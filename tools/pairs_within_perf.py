"""Cost of returning every pair within a threshold instead of the single best match, on a C4-like
job on one GPU: 16 384 queries x 20 000 references of bench.py's C4 generator (seed 200020).

In one session it alternates MultiEngine.best_matches (first minimum) with pairs_within at three
thresholds of p, chosen from a sample of the job's distances so that about 1, 100 and 1 000 pairs
per query are selected, aligned and alignment-free.  It reports pairs/s of every run, the selected
pairs and the bytes of the result.  The device time of the two selection passes per block comes
from a separate profiled pass (torch.profiler, CUDA activity) over the first two device blocks, so
the timed runs carry no tracing.  The card's name and power limit are read in the same call.
Usage: python tools/pairs_within_perf.py [--queries Q] [--refs R] [--rounds N] [--out FILE]"""
from __future__ import annotations

import argparse
import json
import statistics
import subprocess
import sys
import time
from pathlib import Path

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))
sys.path.insert(0, str(ROOT / "tests"))

import numpy as np  # noqa: E402

from synth import coi_like  # noqa: E402
from taxi2_b200.engine import pack_strings  # noqa: E402
from taxi2_b200.multi import MultiEngine  # noqa: E402

PER_ROW = (1, 100, 1000)
KERNELS = ("best_rows_kernel", "within_count_kernel", "within_write_kernel", "DeviceScan")
BYTES_PER_PAIR = 4 + 32 + 16   # index, four metrics, four counts (plus 8 B of row_ptr per query)


def card() -> dict:
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                         capture_output=True, text=True, check=True).stdout.strip()
    name, power, clock = (s.strip() for s in out.split(","))
    return dict(name=name, power_limit=power, max_sm_clock=clock)


def thresholds(multi: MultiEngine, align: bool, r: int) -> dict:
    """Thresholds of p with about 1, 100 and 1 000 selected references per query: quantiles of
    the distances of the first 64 queries (the whole row of each)."""
    eng = multi.engines[0]
    call = eng.align_rect if align else eng.count_rect
    p = call(0, 64, 0, r, want=("metrics",))["metrics"][..., 0]
    p = np.sort(p[~np.isnan(p)])
    per_query = len(p) / 64
    return {f"t{k}": float(p[min(len(p) - 1, int(k / per_query * len(p)))]) for k in PER_ROW}


def kernel_ms(multi: MultiEngine, align: bool, rows: int, ts: dict) -> dict:
    """Device time per launch of the selection kernels over the first `rows` queries (whole device
    blocks), from torch.profiler's CUDA activity records."""
    from torch.profiler import ProfilerActivity, profile

    eng, ny, out = multi.engines[0], multi.ny, {}
    for name, t in (("best", None), *ts.items()):
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            if t is None:
                eng.best_rows(0, rows, 0, ny, 0, align)
            else:
                eng.pairs_within(0, rows, 0, ny, t, 0, align)
        kernels = [e for e in prof.events() if e.device_type.name == "CUDA"]
        per = {}
        for k in KERNELS:
            us = [e.time_range.elapsed_us() for e in kernels if k in e.name]
            if us:
                per[k] = dict(launches=len(us), ms_per_launch=sum(us) / 1e3 / len(us))
        out[name] = dict(rows=rows, kernels=per, kernels_seen=sorted({e.name.split("(")[0][:80] for e in kernels}))
    return out


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--queries", type=int, default=16_384)
    ap.add_argument("--refs", type=int, default=20_000)
    ap.add_argument("--rounds", type=int, default=2, help="aligned rounds; alignment-free runs 4x as many")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()

    import torch

    if not torch.cuda.is_available():
        raise SystemExit("pairs_within_perf needs a CUDA device")
    q, r = args.queries, args.refs
    data, off = pack_strings(coi_like(q + r, seed=200020))
    multi = MultiEngine([0])
    multi.load((data[: off[q]], off[: q + 1]), 0)
    multi.load((data[off[q]:], off[q:] - off[q]), 1)
    pairs = q * r
    record = dict(job=f"{q} queries x {r} references of the C4 generator (seed 200020), one GPU, metric 0 (p)",
                  card=card(), bytes_per_selected_pair=BYTES_PER_PAIR, modes={})
    for align, rounds in ((True, args.rounds), (False, 4 * args.rounds)):
        mode = "aligned" if align else "alignment_free"
        ts = thresholds(multi, align, r)
        # warm-up: a short slice per arm loads the modules and sizes the device and host buffers
        block_rows = (1 << 24 if align else 1 << 27) // r
        eng = multi.engines[0]
        eng.best_rows(0, 64, 0, r, 0, align)
        for t in ts.values():
            eng.pairs_within(0, 64, 0, r, t, 0, align)

        def arms():
            yield "best", lambda: multi.best_matches(0, align)
            for name, t in ts.items():
                yield name, lambda t=t: multi.pairs_within(t, 0, align)

        runs = {name: [] for name, _ in arms()}
        first = {}
        for _ in range(rounds):
            for name, run in arms():
                t0 = time.perf_counter()
                res = run()
                runs[name].append(pairs / (time.perf_counter() - t0))
                first.setdefault(name, res)
        # a query's best match is selected exactly when its value is within the threshold
        best = first["best"]
        for name, t in ts.items():
            res = first[name]
            assert res["row_ptr"][-1] == len(res["index"]), (mode, name)
            rows = np.repeat(np.arange(q), np.diff(res["row_ptr"]))
            hit = np.zeros(q, dtype=bool)
            hit[rows[res["index"] == best["index"][rows]]] = True
            assert np.array_equal(hit, best["metrics"][:, 0] <= t), (mode, name)
        med = {name: statistics.median(v) for name, v in runs.items()}
        selected = {name: int(first[name]["row_ptr"][-1]) for name in ts}
        record["modes"][mode] = dict(
            thresholds=ts, selected_pairs=selected,
            selected_per_query={name: n / q for name, n in selected.items()},
            result_bytes={name: n * BYTES_PER_PAIR + 8 * (q + 1) for name, n in selected.items()},
            pairs_per_s=runs, median_pairs_per_s=med,
            median_vs_best={name: med[name] / med["best"] - 1.0 for name in med if name != "best"},
            kernels=kernel_ms(multi, align, min(q, 2 * block_rows), ts))
        text = json.dumps(record, indent=1)
        if args.out:   # rewritten after each mode
            Path(args.out).parent.mkdir(parents=True, exist_ok=True)
            Path(args.out).write_text(text + "\n")
    multi.close()
    print(text)


if __name__ == "__main__":
    main()
