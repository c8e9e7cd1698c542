"""Cost of single-linkage clusters of one barcode set on one GPU: set 0 x set 0 of coi_like sets,
8 192 sequences aligned and 20 000 alignment-free.  The alignment-free set has coi_like's hierarchy
(50 genera of 20 species, individuals dealt round-robin) with substitutions only: rows of one
length, already aligned, which is the input that mode is for (coi_like's indels shift the frame and
leave no pair within 8 %).

In one session it alternates MultiEngine.best_matches over the same square (the floor: the same
blocks, one row reduction each) with clusters_within at 1, 3 and 8 % p-distance (scale 100) one
threshold per call, and with all three in one call, every arm on the same row tiles.  It also times what a user had to do before:
pairs_within over the square at each threshold, then the components on the host (scipy) -- and
checks that both give the same labels.  It reports pairs/s of every run and their medians.  The
device time per launch of every kernel comes from a separate profiled pass (torch.profiler, CUDA
activity) over the first two device blocks, so the timed runs carry no tracing.  The card's name
and power limit are read in the same call.
Usage: python tools/clusters_perf.py [--aligned N] [--free N] [--rounds R] [--out FILE]"""
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

from scipy.sparse import csr_matrix  # noqa: E402
from scipy.sparse.csgraph import connected_components  # noqa: E402

from synth import ALPHA, COMPOSITION, coi_like  # noqa: E402
from taxi2_b200.multi import MultiEngine  # noqa: E402

PERCENT = (1.0, 3.0, 8.0)


def card() -> dict:
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                         capture_output=True, text=True, check=True).stdout.strip()
    name, power, clock = (s.strip() for s in out.split(","))
    return dict(name=name, power_limit=power, max_sm_clock=clock)


def prealigned(n: int, seed: int, length: int = 650, genera: int = 50, species: int = 20) -> list[bytes]:
    """coi_like's hierarchy without indels: root -> genera (12 % of the sites redrawn) -> species
    (6 %) -> individuals (1 %, and 0.02 % N), dealt round-robin."""
    rng = np.random.default_rng(seed)

    def redraw(seq: np.ndarray, rate: float) -> np.ndarray:
        seq = seq.copy()
        hit = rng.random(len(seq)) < rate
        seq[hit] = ALPHA[rng.choice(4, size=int(hit.sum()), p=COMPOSITION)]
        return seq

    root = ALPHA[rng.choice(4, size=length, p=COMPOSITION)]
    gen = [redraw(root, 0.12) for _ in range(genera)]
    spp = [[redraw(g, 0.06) for _ in range(species)] for g in gen]
    out = []
    for k in range(n):
        ind = redraw(spp[k % genera][(k // genera) % species], 0.01)
        ind[rng.random(length) < 0.0002] = ord("N")
        out.append(ind.tobytes())
    return out


def host_components(res: dict, n: int) -> np.ndarray:
    """Canonical labels (smallest member) of the graph of pairs_within's CSR over n nodes."""
    graph = csr_matrix((np.ones(len(res["index"]), dtype=np.int8), res["index"], res["row_ptr"]), shape=(n, n))
    _, comp = connected_components(graph, directed=False)
    low = np.full(comp.max() + 1, n, dtype=np.int64)
    np.minimum.at(low, comp, np.arange(n))
    return low[comp].astype(np.int32)


def kernel_ms(multi: MultiEngine, align: bool, rows: int) -> dict:
    """Device time per launch of every kernel over the first `rows` rows of the square (whole device
    blocks), from torch.profiler's CUDA activity records."""
    from torch.profiler import ProfilerActivity, profile

    eng, n, out = multi.engines[0], multi.nx, {}
    calls = {"best": lambda: eng.best_rows(0, rows, 0, n, 0, align)}
    for p in PERCENT:
        calls[f"t{p:g}"] = lambda p=p: eng.clusters_within(0, rows, 0, n, p, 0, align, scale=100.0)
    calls["all"] = lambda: eng.clusters_within(0, rows, 0, n, list(PERCENT), 0, align, scale=100.0)
    for name, call in calls.items():
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            call()
        per: dict = {}
        for e in prof.events():
            if e.device_type.name != "CUDA":
                continue
            k = e.name.split("(")[0][:80]
            d = per.setdefault(k, dict(launches=0, ms=0.0))
            d["launches"] += 1
            d["ms"] += e.time_range.elapsed_us() / 1e3
        for d in per.values():
            d["ms_per_launch"] = d["ms"] / d["launches"]
        out[name] = dict(rows=rows, kernels=per)
    return out


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--aligned", type=int, default=8_192)
    ap.add_argument("--free", type=int, default=20_000)
    ap.add_argument("--rounds", type=int, default=3, help="aligned rounds; alignment-free runs 4x as many")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()

    import torch

    if not torch.cuda.is_available():
        raise SystemExit("clusters_perf needs a CUDA device")
    record = dict(job="set 0 x set 0 of coi_like (seed 700; alignment-free: without indels), one GPU, metric 0 (p), "
                      "thresholds in percent (scale 100)",
                  card=card(), thresholds_percent=list(PERCENT), modes={})
    multi = MultiEngine([0])
    text = ""
    for align, n, rounds in ((True, args.aligned, args.rounds), (False, args.free, 4 * args.rounds)):
        mode = "aligned" if align else "alignment_free"
        multi.load(coi_like(n, seed=700) if align else prealigned(n, seed=700), 0)
        pairs = n * n
        eng = multi.engines[0]
        # warm-up: a short slice per arm loads the modules and sizes the device buffers
        eng.best_rows(0, 64, 0, n, 0, align)
        eng.clusters_within(0, 64, 0, n, list(PERCENT), 0, align, scale=100.0)
        eng.pairs_within(0, 64, 0, n, PERCENT[-1], 0, align, scale=100.0, skip_self=True)
        host_components(dict(index=np.zeros(0, np.int32), row_ptr=np.zeros(n + 1, np.int64)), n)

        # every arm runs on the same tiles: row_tiles' default when aligned, and alignment-free the
        # one or two tiles per GPU that clusters_within picks by default
        tile = None if align else max(1, min(-(-n // 2), (1 << 26) // n))

        def arms():
            yield "best", lambda: multi.best_matches(0, align, rows_per_tile=tile)
            for p in PERCENT:
                yield f"t{p:g}", lambda p=p: multi.clusters_within(p, 0, align, scale=100.0, rows_per_tile=tile)
            yield "all", lambda: multi.clusters_within(list(PERCENT), 0, align, scale=100.0, rows_per_tile=tile)
            for p in PERCENT:
                yield f"pairs_host_t{p:g}", lambda p=p: multi.pairs_within(p, 0, align, scale=100.0, skip_self=True,
                                                                           rows_per_tile=tile)

        runs = {name: [] for name, _ in arms()}
        host_s = {name: [] for name in runs if name.startswith("pairs_host")}
        first = {}
        for _ in range(rounds):
            for name, run in arms():
                t0 = time.perf_counter()
                res = run()
                if name.startswith("pairs_host"):
                    t1 = time.perf_counter()
                    res = dict(labels=host_components(res, n)[None, :], selected=int(res["row_ptr"][-1]))
                    host_s[name].append(time.perf_counter() - t1)
                runs[name].append(pairs / (time.perf_counter() - t0))
                first.setdefault(name, res)
        # the device labels equal the host components of the same links, threshold by threshold
        for k, p in enumerate(PERCENT):
            assert np.array_equal(first[f"t{p:g}"]["labels"], first[f"pairs_host_t{p:g}"]["labels"]), (mode, p)
            assert np.array_equal(first["all"]["labels"][k], first[f"t{p:g}"]["labels"][0]), (mode, p)
        med = {name: statistics.median(v) for name, v in runs.items()}
        block_rows = (1 << 24 if align else 1 << 27) // n
        record["modes"][mode] = dict(
            sequences=n, pairs=pairs, rounds=rounds, rows_per_tile=tile or "row_tiles default",
            clusters={f"t{p:g}": int(first["all"]["clusters"][k]) for k, p in enumerate(PERCENT)},
            linked_pairs={f"t{p:g}": first[f"pairs_host_t{p:g}"]["selected"] for p in PERCENT},
            pairs_per_s=runs, median_pairs_per_s=med,
            median_vs_best={name: med[name] / med["best"] - 1.0 for name in med if name != "best"},
            median_host_components_s={name: statistics.median(v) for name, v in host_s.items()},
            kernels=kernel_ms(multi, align, min(n, 2 * block_rows)))
        text = json.dumps(record, indent=1)
        if args.out:   # rewritten after each mode
            Path(args.out).parent.mkdir(parents=True, exist_ok=True)
            Path(args.out).write_text(text + "\n")
    multi.close()
    print(text)


if __name__ == "__main__":
    main()
