"""Cost of returning the k closest references per query instead of the single best match, on a
C4-like job on one GPU: 16 384 queries x 20 000 references of bench.py's C4 generator (seed 200020).

In one session it alternates MultiEngine.best_matches (first minimum) with best_matches_k at
k = 1, 10 and 64, aligned and alignment-free, and reports pairs/s of every run.  The selection
kernels' own device time comes from a separate profiled pass (torch.profiler, CUDA activity) over
the first two device blocks of the same job, so the timed runs carry no tracing.  The card's name
and power limit are read in the same call.  Usage: python tools/best_k_perf.py [--queries Q] [--refs R] [--rounds N] [--out FILE]"""
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

KS = (1, 10, 64)
SELECT_KERNELS = ("best_rows_kernel", "best_k_rows_kernel")


def card() -> dict:
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                         capture_output=True, text=True, check=True).stdout.strip()
    name, power, clock = (s.strip() for s in out.split(","))
    return dict(name=name, power_limit=power, max_sm_clock=clock)


def arms():
    yield "best", lambda m, align: m.best_matches(0, align)
    for k in KS:
        yield f"k{k}", lambda m, align, k=k: m.best_matches_k(k, 0, align)


def select_kernel_ms(multi: MultiEngine, align: bool, rows: int) -> dict:
    """Device time per launch of the two selection kernels over the first `rows` queries (whole
    device blocks), from torch.profiler's CUDA activity records."""
    from torch.profiler import ProfilerActivity, profile

    eng, ny, out = multi.engines[0], multi.ny, {}
    for name, k in (("best", None), *((f"k{k}", k) for k in KS)):
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            if k is None:
                eng.best_rows(0, rows, 0, ny, 0, align)
            else:
                eng.best_rows_k(0, rows, 0, ny, k, 0, align)
        kernels = [e for e in prof.events() if e.device_type.name == "CUDA"]
        us = [e.time_range.elapsed_us() for e in kernels if any(n in e.name for n in SELECT_KERNELS)]
        out[name] = dict(rows=rows, launches=len(us), ms_per_launch=sum(us) / 1e3 / max(len(us), 1),
                         kernels_seen=sorted({e.name.split("(")[0] for e in kernels}))
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
        raise SystemExit("best_k_perf needs a CUDA device")
    q, r = args.queries, args.refs
    data, off = pack_strings(coi_like(q + r, seed=200020))
    multi = MultiEngine([0])
    multi.load((data[: off[q]], off[: q + 1]), 0)
    multi.load((data[off[q]:], off[q:] - off[q]), 1)
    pairs = q * r
    record = dict(job=f"{q} queries x {r} references of the C4 generator (seed 200020), one GPU, metric 0 (p)",
                  card=card(), modes={})
    for align, rounds in ((True, args.rounds), (False, 4 * args.rounds)):
        mode = "aligned" if align else "alignment_free"
        # warm-up: a short slice per arm loads the modules and sizes the device buffers
        block_rows = (1 << 24 if align else 1 << 27) // r
        eng = multi.engines[0]
        eng.best_rows(0, 64, 0, r, 0, align)
        for k in KS:
            eng.best_rows_k(0, 64, 0, r, k, 0, align)
        runs = {name: [] for name, _ in arms()}
        first = {}
        for _ in range(rounds):
            for name, run in arms():
                t0 = time.perf_counter()
                res = run(multi, align)
                runs[name].append(pairs / (time.perf_counter() - t0))
                first.setdefault(name, res)
        # every arm selects the same winner; k = 1 is best_matches with a rank axis
        for name in runs:
            if name != "best":
                assert np.array_equal(first[name]["index"][:, 0], first["best"]["index"]), (mode, name)
        assert np.array_equal(first["k1"]["metrics"][:, 0], first["best"]["metrics"], equal_nan=True)
        med = {name: statistics.median(v) for name, v in runs.items()}
        record["modes"][mode] = dict(
            pairs_per_s=runs, median_pairs_per_s=med,
            median_vs_best={name: med[name] / med["best"] - 1.0 for name in med if name != "best"},
            select_kernel=select_kernel_ms(multi, align, min(q, 2 * block_rows)))
        text = json.dumps(record, indent=1)
        if args.out:   # rewritten after each mode
            Path(args.out).parent.mkdir(parents=True, exist_ok=True)
            Path(args.out).write_text(text + "\n")
    multi.close()
    print(text)


if __name__ == "__main__":
    main()
