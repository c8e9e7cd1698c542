#!/usr/bin/env python
"""bench.py -- benchmarks of the TaxI2 pairwise-distance path on B200.

Headline (default, BASELINE.json metric): aligned pairs/sec & GCUPS, all-pairs ~650 bp COI-like
sequences.  Workload = BASELINE config C3 -- 50 000 synthetic COI-like sequences (seed 650), all
ordered pairs (reference semantics, versus_all.py:746).  One "step" is one TILE_X x TILE_Y tile of
that 50k x 50k pair matrix (global Gotoh alignment with Biopython's first-path tie-breaking + the
four distance metrics per pair).  With N GPUs under torchrun every rank takes its own tile per
step (static tile assignment, weak scaling, no collective on the compute path).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--dump-outputs DIR]
    python bench.py --config C2|C4|C5 [--gpus N] ...      (one process drives N GPUs)

Prints ONE JSON line (rank 0):
  value     device-resident throughput (inputs already in HBM, outputs left in HBM)
  e2e       the same metric through the C-ABI with HOST buffers (uploads + downloads timed)
  roofline  dominant kernel vs the integer-ALU (DP) or HBM (alignment-free) roofline; the kernel
            time is measured live with CUDA events on the launch stream inside the C-ABI
  strong    (C3) one FIXED job -- 8192 x 16384 pairs of the C3 matrix -- sharded over all N GPUs by
            the product path (taxi2_b200/multi.py: one process, one thread per GPU, static LPT
            tiles, every GPU's D2H landing in its slice of one pinned host matrix), gather included
  versus_all (C3) versusAll of the first 8192 sequences as a whole job: all 6.7e7 ORDERED pairs delivered
            into one pinned host matrix from one alignment per unordered pair (mirrored; orientation-
            sensitive pairs re-aligned), checked against the ordinary path on a band of rows
`--impl reference` times the CPU restatement of the reference path (oracle/, "port": Biopython
and the Rust distance crate are not installable here) on all host threads, on the same tiles.
`--dump-outputs DIR` (C3) writes the results of the last timed step (rank 0's tile) as DIR/counts.npy
and DIR/metrics.npy, for comparing two builds output for output (see dump_outputs).
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))
sys.path.insert(0, str(ROOT / "tests"))
sys.dont_write_bytecode = True   # the benchmark leaves the tree as it found it (no __pycache__)

N_SEQ = 50_000
SEQ_LEN = 650
TILE_X = 1536
TILE_Y = 2048
STRONG_X, STRONG_Y = 8192, 16384
SYM_N = 8192               # versusAll as a whole job: all ordered pairs of the first SYM_N sequences
DUMP_PAIRS = 1 << 20       # --dump-outputs: pairs sampled from the last tile (48 MiB; the whole tile is 144 MiB)
OPS_PER_CELL = 13          # SURVEY.md 8d: scalar INT32 ops of the score-only 3-state recurrence
SCORES_TEXT = "match 1, mismatch -1, internal open -8 / extend -1, end open -1 / extend -1"


# ---- inputs -------------------------------------------------------------------------------------
def make_sequences(n: int, seed: int = 650, length: int = SEQ_LEN):
    from synth import coi_like
    from taxi2_b200.engine import pack_strings

    return pack_strings(coi_like(n, length=length, seed=seed))


def make_mixed(n: int):
    """BASELINE C5 geometry: the C3 species tree at 1500 bp, every sequence cut to a uniform
    300-1500 bp."""
    from synth import coi_like
    from taxi2_b200.engine import pack_strings

    rng = np.random.default_rng(5)
    base = coi_like(n, length=1500, seed=5)
    return pack_strings([s[: int(rng.integers(300, 1501))] for s in base])


def make_prealigned(n: int = 9000, columns: int = 618):
    """BASELINE C2 stand-in (the reference's ca9000 file is missing from its checkout): a seeded
    resample of the 120-sequence sample, every row padded with '-' to the common width."""
    from synth import read_tab_sequences
    from taxi2_b200.engine import pack_strings

    _, seqs = read_tab_sequences(ROOT / "tests" / "golden" / "Taxi2test1_120.tab", normalize=False)
    rng = np.random.default_rng(9000)
    rows = []
    for k in rng.integers(0, len(seqs), n):
        s = seqs[int(k)][:columns]
        lead = int(rng.integers(0, columns - len(s) + 1))
        rows.append("-" * lead + s + "-" * (columns - len(s) - lead))
    return pack_strings(rows)


def tile_of(step: int, rank: int, world: int, n: int) -> tuple[int, int]:
    """Static tile assignment: the ordered pair matrix is cut into TILE_X x TILE_Y tiles,
    enumerated row-major; (step, rank) -> tile index step*world + rank."""
    tiles_y = n // TILE_Y
    tiles_x = n // TILE_X
    t = (step * world + rank) % (tiles_x * tiles_y)
    return (t // tiles_y) * TILE_X, (t % tiles_y) * TILE_Y


# ---- clocks, peaks ------------------------------------------------------------------------------
class ClockSampler:
    """nvidia-smi clocks/throttle reasons DURING the timed region (B200_PROFILING.md recipe)."""

    FIELDS = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
              "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
              "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.rows: list[list[str]] = []
        self.proc = None
        self.gpu = gpu_index

    def __enter__(self):
        if self.gpu < 0:
            return self
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={self.FIELDS}", "--format=csv,noheader,nounits", "-lms", "200", "-i", str(self.gpu)],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._pump, daemon=True)
            self.thread.start()
        except OSError:
            self.proc = None
        return self

    def _pump(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def __exit__(self, *exc):
        if self.proc:
            self.proc.terminate()
            try:
                self.proc.wait(timeout=2)
            except subprocess.TimeoutExpired:
                self.proc.kill()

    def summary(self) -> dict:
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            try:
                sm.append(float(r[1])); mx.append(float(r[2]))
            except (ValueError, IndexError):
                continue
            for name, val in zip(names, r[5:9]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        # under load = samples above half the max clock
        load = [s for s in sm if mx and s > 0.5 * max(mx)] or sm
        return dict(sm_mhz=float(np.median(load)) if load else None, sm_max_mhz=max(mx) if mx else None,
                    reasons=sorted(reasons), samples=len(sm))


def measured_peaks() -> dict:
    try:
        return json.loads((ROOT / "MEASURED_PEAKS.json").read_text())
    except (OSError, ValueError):
        return {}


def peak_hbm() -> tuple[float, str]:
    v = measured_peaks().get("hbm_gbs")
    return (float(v), "MEASURED_PEAKS.json hbm_gbs") if v else (6650.0, "fallback of B200_PROFILING.md")


def int32_lanes() -> tuple[float, str]:
    """INT32 issue width, lane-ops/clk/SM: the IADD3 / 2-input VIMNMX rate measured by
    tools/int_peak.cu over >= 50 ms per op (profiles/int_peak_r02.jsonl).  A hardware constant;
    the roofline multiplies it by the SM count and by the SM clock sampled DURING the timed
    region, so the denominator cannot be flattered by a microbenchmark that ran at another clock."""
    path = ROOT / "profiles" / "int_peak_r02.jsonl"
    try:
        best = 0.0
        for line in path.read_text().splitlines():
            rec = json.loads(line)
            if rec.get("op") in ("IADD3", "VIMNMX") and rec.get("threads_per_sm") == 1024:
                best = max(best, float(rec["lane_ops_per_clk_per_sm"]))
        if best > 0:
            return best, f"{path.relative_to(ROOT)} (IADD3/VIMNMX, 1024 threads/SM)"
    except (OSError, ValueError, KeyError):
        pass
    return 128.0, "nominal 128 lanes/clk/SM"


def int_roofline(cells_per_launch: float, launch_s: float, clocks: dict, sms: int, kernel: str, packed: bool) -> dict:
    lanes, lanes_how = int32_lanes()
    mhz = clocks.get("sm_mhz") or measured_peaks().get("sm_max_mhz") or 1965.0
    peak = lanes * sms * mhz * 1e6
    achieved = cells_per_launch * OPS_PER_CELL / launch_s
    traffic = ncu_traffic(kernel)
    out = dict(
        bound="int32_alu", kernel=kernel, achieved=achieved / 1e9, peak=peak / 1e9, unit="Gop/s", frac=achieved / peak,
        # every .U16x2 instruction of the packed kernel advances two cells: against a ceiling of
        # 2 x the scalar issue rate the same number reads half
        frac_packed=(achieved / (2 * peak)) if packed else None,
        traffic=traffic["bytes_per_cell"] * cells_per_launch if traffic else None,
        traffic_source=traffic["source"] if traffic else None,
        how=(f"{OPS_PER_CELL} algorithmic INT32 ops/cell x {cells_per_launch:.4e} cells/launch / {launch_s * 1e3:.2f} ms per launch "
             f"(CUDA events on the launch stream); peak = {lanes:.2f} lane-ops/clk/SM [{lanes_how}] x {sms} SMs x {mhz:.0f} MHz "
             f"(SM clock sampled during the timed region)"),
    )
    return out


def ncu_traffic(kernel: str) -> dict | None:
    """DRAM bytes per DP cell of a kernel from the committed ncu --set full capture (per launch,
    dram__bytes_read.sum + dram__bytes_write.sum / cells of that launch); not re-measured here."""
    try:
        table = json.loads((ROOT / "profiles" / "ncu_traffic.json").read_text())
    except (OSError, ValueError):
        return None
    for name, rec in table.items():
        if kernel.startswith(name):
            return rec
    return None


# ---- CPU baseline (the oracle; bench.py may execute it only here and in --impl reference) --------
def cpu_align_throughput(data, off, seconds: float, pairs_of, threads: int = 0) -> dict:
    """Times the CPU restatement (oracle/) on a bounded sample: `pairs_of(rng, k)` -> (px, py)."""
    import oracle

    rng = np.random.default_rng(1)
    threads = threads or oracle.max_threads()
    lens = np.diff(off)
    pairs = cells = 0
    t0 = time.perf_counter()
    chunk = max(64, 32 * threads)
    while True:
        px, py = pairs_of(rng, chunk)
        oracle.align_count_pairs(data, off, px, py, None, threads)
        pairs += chunk
        cells += int((lens[px] * lens[py]).sum())
        dt = time.perf_counter() - t0
        if dt >= seconds:
            break
    return dict(pairs=pairs, cells=cells, seconds=dt, threads=threads)


def tile_pairs(x0: int, nx: int, y0: int, ny: int):
    def pairs_of(rng, k):
        return (x0 + rng.integers(0, nx, size=k)).astype(np.int32), (y0 + rng.integers(0, ny, size=k)).astype(np.int32)
    return pairs_of


def cpu_count_throughput(data, off, seconds: float) -> dict:
    import oracle

    n = len(off) - 1
    rng = np.random.default_rng(1)
    threads = oracle.max_threads()
    pairs = 0
    t0 = time.perf_counter()
    chunk = 1 << 18
    while True:
        px = rng.integers(0, n, size=chunk).astype(np.int32)
        py = rng.integers(0, n, size=chunk).astype(np.int32)
        oracle.count_pairs(data, off, px, py, threads)
        pairs += chunk
        dt = time.perf_counter() - t0
        if dt >= seconds:
            break
    return dict(pairs=pairs, cells=0, seconds=dt, threads=threads)


# ---- workloads -----------------------------------------------------------------------------------
def workload(config: str, world: int, **kw) -> dict:
    if config == "C3":
        return dict(
            workload=f"C3: all ordered pairs of {N_SEQ} synthetic COI-like sequences (~{SEQ_LEN} bp, seed 650); "
                     f"step = one {TILE_X}x{TILE_Y} tile of the pair matrix per GPU",
            pairs_per_step_per_gpu=TILE_X * TILE_Y, scores=SCORES_TEXT, metrics="p, p-gaps, jc, k2p",
            sharding=f"static tile assignment over {world} GPU(s), no data-path collective",
            l2="256 MiB L2 flush between steps; the per-step traceback arena (2.5 GB) exceeds L2 on its own")
    if config == "C2":
        return dict(
            workload=f"C2: alignment-free (align=False) counts + 4 metrics of all {kw['n']}x{kw['n']} ordered pairs of {kw['n']} pre-aligned "
                     f"rows x 618 columns (seeded resample of Taxi2test1_120.tab padded with '-': the reference's ca9000 file is missing); "
                     f"step = the whole matrix",
            metrics="p, p-gaps, jc, k2p", sharding=f"{world} GPU(s), full-width row tiles, host gather",
            l2="results (3.9 GB per step) exceed L2; the bit planes (2.9 MB) are meant to stay in it")
    if config == "C4":
        return dict(
            workload=f"C4: versusReference best match, {kw['queries']} queries x {kw['refs']} references of the C3 generator (seed 200020): "
                     f"alignment + 4 metrics of every pair, first minimum of p per query, winner's metrics and counts; step = the whole job",
            scores=SCORES_TEXT, metrics="p (main) + p-gaps, jc, k2p of the winner",
            sharding=f"{world} GPU(s) driven by one process: full-width row tiles dealt longest-processing-time-first, winners gathered on the host",
            l2="the traceback arena (2.5 GB per GPU) exceeds L2")
    if config == "C5":
        return dict(
            workload=f"C5 (reduced from 100 000 to {kw['n']} sequences): all ordered pairs of {kw['n']} sequences of 300-1500 bp (C3 species tree), "
                     f"alignment + 4 metrics, rows grouped by kernel geometry; step = the whole matrix in row tiles",
            scores=SCORES_TEXT, metrics="p, p-gaps, jc, k2p",
            sharding=f"{world} GPU(s) driven by one process: full-width row tiles dealt longest-processing-time-first",
            l2="the traceback arena exceeds L2")
    raise ValueError(config)


def ensure_built(local_rank: int) -> None:
    """A fresh checkout has no built artefacts (kept out of history): rank 0 builds, the others wait."""
    needed = [ROOT / "taxi2_b200" / "lib" / "libtaxi2_b200.so", ROOT / "oracle" / "libtaxi_oracle.so"]
    if all(p.exists() for p in needed):
        return
    if local_rank == 0:
        import __graft_entry__

        __graft_entry__.build()
    else:
        deadline = time.time() + 600
        while not all(p.exists() for p in needed) and time.time() < deadline:
            time.sleep(2)
        time.sleep(5)   # let the linker finish writing


# ---- the reference arm ---------------------------------------------------------------------------
def run_reference(args, rank: int, world: int) -> None:
    if rank != 0:
        return
    per_step = 4.0
    if args.config == "C2":
        data, off = make_prealigned(args.nseq or 9000)
        run = lambda k, secs: cpu_count_throughput(data, off, secs)   # noqa: E731
        sample = "random ordered pairs of the C2 rows"
        cfg = workload("C2", world, n=len(off) - 1)
    elif args.config == "C4":
        refs = 20_000
        queries = 4096
        data, off = make_sequences(queries + refs, seed=200020)
        run = lambda k, secs: cpu_align_throughput(data, off, secs, tile_pairs(0, queries, queries, refs))   # noqa: E731
        sample = f"random (query, reference) pairs of the C4 generator (first {queries} queries x {refs} references)"
        cfg = workload("C4", world, queries=args.queries or 200_000, refs=refs)
    elif args.config == "C5":
        n = args.nseq or 16384
        data, off = make_mixed(min(n, 4096))
        run = lambda k, secs: cpu_align_throughput(data, off, secs, tile_pairs(0, len(off) - 1, 0, len(off) - 1))   # noqa: E731
        sample = f"random ordered pairs of the first {len(off) - 1} C5 sequences"
        cfg = workload("C5", world, n=n)
    else:
        n = args.nseq or N_SEQ
        data, off = make_sequences(n)
        # the same tiles the GPU arm aligns at N = 1: step k samples pairs of tile k
        def run(k, secs):
            x0, y0 = tile_of(k, 0, 1, n)
            return cpu_align_throughput(data, off, secs, tile_pairs(x0, TILE_X, y0, TILE_Y))

        sample = f"random ordered pairs inside the {TILE_X}x{TILE_Y} tile of each step (the tiles of the GPU arm at N = 1)"
        cfg = workload("C3", world)
    for k in range(args.warmup):
        run(k, 0.5)
    t0 = time.perf_counter()
    pairs = cells = threads = 0
    for k in range(args.steps):
        r = run(args.warmup + k, per_step)
        pairs += r["pairs"]; cells += r["cells"]; threads = r["threads"]
    dt = time.perf_counter() - t0
    value = pairs / dt
    line = dict(
        impl="reference", metric="aligned_pairs_per_sec", value=value, unit="pairs/s", gcups=cells / dt / 1e9,
        n_gpus=world, steps=args.steps, warmup=args.warmup, ms_per_step=1e3 * dt / args.steps,
        higher_is_better=True, scaling="weak", vs_baseline=None, dtype="f64", data="synthetic", config=cfg,
        cpu_baseline=dict(value=value, unit="pairs/s", cores=threads, kind="port", sample=f"{pairs} {sample}, ~{per_step:.0f} s per step"),
        e2e=dict(value=value, unit="pairs/s", h2d_bytes_per_step=0, d2h_bytes_per_step=0),
        note="CPU restatement of Biopython PairwiseAligner + calculate_distances (oracle/), not the binaries themselves",
    )
    print(json.dumps(line), flush=True)


# ---- C3: the headline ------------------------------------------------------------------------------
def run_c3(args, rank: int, local_rank: int, world: int) -> None:
    import torch
    import torch.distributed as dist

    from taxi2_b200.engine import Engine, PinnedArray

    torch.cuda.set_device(local_rank)
    distributed = world > 1
    host_group = None
    if distributed:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        # stdout carries exactly one JSON line.  This image exports NCCL_DEBUG=VERSION, whose only
        # effect is a "NCCL version ..." line on stdout (NCCL_DEBUG_FILE does not move that one);
        # any other level the caller asked for is kept, with its output sent to stderr.
        if os.environ.get("NCCL_DEBUG", "").upper() == "VERSION":
            del os.environ["NCCL_DEBUG"]
        os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
        host_group = dist.new_group(backend="gloo")   # host-side waiting (no kernel spinning on a GPU)

    n = args.nseq or N_SEQ
    data, off = make_sequences(n)
    eng = Engine(local_rank)
    eng.load((data, off), 0)
    sms = torch.cuda.get_device_properties(local_rank).multi_processor_count

    npairs = TILE_X * TILE_Y
    d_counts = torch.empty((npairs, 4), dtype=torch.int32, device="cuda")
    d_metrics = torch.empty((npairs, 4), dtype=torch.float64, device="cuda")
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")
    lens = np.diff(off)

    def barrier():
        if distributed:
            dist.barrier()
        torch.cuda.synchronize()

    debug = bool(os.environ.get("TAXI_BENCH_DEBUG"))

    def step_device(k: int) -> int:
        x0, y0 = tile_of(k, rank, world, n)
        flush.zero_()
        torch.cuda.synchronize()
        eng.align_rect_device(x0, TILE_X, y0, TILE_Y, 0, d_counts.data_ptr(), d_metrics.data_ptr())
        eng.sync()
        return int(lens[x0:x0 + TILE_X].sum()) * int(lens[y0:y0 + TILE_Y].sum())

    # ---- device-resident throughput ("value") ---------------------------------------------------
    for k in range(args.warmup):
        step_device(k)
    st0 = eng.stats()
    barrier()
    with ClockSampler(local_rank if not os.environ.get("TAXI_NO_SAMPLER") else -1) as clocks:
        t0 = time.perf_counter()
        cells = 0
        for k in range(args.steps):
            cells += step_device(args.warmup + k)
        barrier()
        dt = time.perf_counter() - t0
    st1 = eng.stats()
    kernel_ms = st1["kernel_ms"] - st0["kernel_ms"]
    launches = st1["launches"] - st0["launches"]
    kernel_id = eng.last_kernel
    checksum = int(d_counts.sum().item())
    if args.dump_outputs and rank == 0:
        dump_outputs(Path(args.dump_outputs), d_counts, d_metrics)

    # ---- end to end through the C ABI with host buffers ("e2e") --------------------------------
    eng2 = Engine(local_rank)
    h2d = d2h = 0
    # inputs sit in page-locked host memory: the sequence bytes as a whole, the per-tile offsets
    # in two small pinned scratch arrays that are rewritten every step
    pinned_data = PinnedArray(data.shape, np.uint8)
    pinned_data.array[:] = data
    pinned_xoff = PinnedArray((TILE_X + 1,), np.int64)
    pinned_yoff = PinnedArray((TILE_Y + 1,), np.int64)

    def step_e2e(k: int) -> None:
        nonlocal h2d, d2h
        x0, y0 = tile_of(k, rank, world, n)
        np.subtract(off[x0:x0 + TILE_X + 1], off[x0], out=pinned_xoff.array)
        np.subtract(off[y0:y0 + TILE_Y + 1], off[y0], out=pinned_yoff.array)
        xs = (pinned_data.array[off[x0]:off[x0 + TILE_X]], pinned_xoff.array)
        ys = (pinned_data.array[off[y0]:off[y0 + TILE_Y]], pinned_yoff.array)
        eng2.load(xs, 0)
        eng2.load(ys, 1)
        out = eng2.align_rect(0, TILE_X, 0, TILE_Y, want=("counts", "metrics"), pinned=True)
        h2d = xs[0].nbytes + xs[1].nbytes + ys[0].nbytes + ys[1].nbytes
        d2h = out["counts"].nbytes + out["metrics"].nbytes

    for k in range(args.warmup):   # untimed: buffers reach their steady size
        step_e2e(k)
    barrier()
    t1 = time.perf_counter()
    for k in range(args.steps):
        step_e2e(args.warmup + k)
    barrier()
    dt_e2e = time.perf_counter() - t1
    e2e_launches = eng2.stats()["launches"] * args.steps   # stats are per call: one align launch per step

    # ---- strong scaling: ONE fixed job over all N GPUs through the product path ------------------
    strong = None
    if args.strong and n >= STRONG_Y:
        if rank == 0:
            strong = strong_scaling(data, off, world, debug)
            torch.cuda.set_device(local_rank)
        if distributed:
            dist.barrier(group=host_group)

    # ---- versusAll as a whole: both orientations from one alignment per unordered pair -------------
    versus_all = None
    if args.strong and n >= SYM_N:
        if rank == 0:
            versus_all = versus_all_symmetric(data, off, world)
            torch.cuda.set_device(local_rank)
        if distributed:
            dist.barrier(group=host_group)

    # ---- aggregate over ranks (max time, sum work) ----------------------------------------------
    if distributed:
        t = torch.tensor([dt, dt_e2e, kernel_ms], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dt, dt_e2e, kernel_ms = (float(v) for v in t.tolist())
        w = torch.tensor([cells, launches], dtype=torch.int64, device="cuda")
        dist.all_reduce(w, op=dist.ReduceOp.SUM)
        cells, launches = (int(v) for v in w.tolist())

    if rank == 0:
        pairs_total = npairs * args.steps * world
        value = pairs_total / dt
        gcups = cells / dt / 1e9
        cells_per_launch = cells / max(launches, 1)
        launch_s = kernel_ms / 1e3 / max(launches / world, 1)   # kernel_ms: max over ranks of each rank's sum over its launches
        kernel_name = {16: "gotoh_pair16_kernel<21,0>", 17: "gotoh_pair16_kernel<21,1>"}.get(kernel_id, "gotoh_warp_kernel<21>")
        clk = clocks.summary()
        roof = int_roofline(cells_per_launch, launch_s, clk, sms, kernel_name, kernel_id in (16, 17, 18))
        trace_bytes_per_cell = trace_bytes(kernel_id)
        hbm, hbm_how = peak_hbm()
        roof["hbm"] = dict(achieved=cells_per_launch * trace_bytes_per_cell / launch_s / 1e9, peak=hbm, unit="GB/s",
                           note=f"algorithmic HBM traffic of the same kernel: traceback codes written once ({trace_bytes_per_cell:.3f} B/cell), "
                                f"read back sparsely; peak = {hbm_how}")
        x0, y0 = tile_of(args.warmup, 0, 1, n)
        cpu = cpu_align_throughput(data, off, args.cpu_seconds, tile_pairs(x0, TILE_X, y0, TILE_Y))
        line = dict(
            metric="aligned_pairs_per_sec", value=value, unit="pairs/s", gcups=gcups,
            n_gpus=world, steps=args.steps, warmup=args.warmup, ms_per_step=1e3 * dt / args.steps,
            higher_is_better=True, scaling="weak", vs_baseline=None, dtype="u16x2" if kernel_id in (16, 17, 18) else "int32", data="synthetic",
            config=workload("C3", world),
            roofline=roof,
            cpu_baseline=dict(value=cpu["pairs"] / cpu["seconds"], unit="pairs/s", gcups=cpu["cells"] / cpu["seconds"] / 1e9,
                              cores=cpu["threads"], kind="port",
                              sample=f"{cpu['pairs']} random ordered pairs of the first timed {TILE_X}x{TILE_Y} tile in {cpu['seconds']:.1f} s"),
            e2e=dict(value=npairs * args.steps * world / dt_e2e, unit="pairs/s", h2d_bytes_per_step=h2d, d2h_bytes_per_step=d2h,
                     steps=args.steps),
            strong=strong, versus_all=versus_all,
            gpu_launches=launches + e2e_launches * world, clocks=clk, checksum=checksum,
        )
        print(json.dumps(line), flush=True)
    if distributed:
        dist.destroy_process_group()


def dump_outputs(out_dir: Path, d_counts, d_metrics) -> None:
    """The last timed step's results for a fixed sample of DUMP_PAIRS pairs of its tile (seed 0,
    in row-major pair order; the same inputs every run): counts.npy (DUMP_PAIRS x 4 {same, ts, tv,
    gaps} as float32, exact) and metrics.npy (DUMP_PAIRS x 4 {p, p-gaps, jc, k2p} as float64, NaN =
    undefined)."""
    import torch

    pick = np.sort(np.random.default_rng(0).choice(d_counts.shape[0], DUMP_PAIRS, replace=False))
    idx = torch.from_numpy(pick).to(d_counts.device)
    out_dir.mkdir(parents=True, exist_ok=True)
    np.save(out_dir / "counts.npy", d_counts.index_select(0, idx).float().cpu().numpy())
    np.save(out_dir / "metrics.npy", d_metrics.index_select(0, idx).cpu().numpy())


def trace_bytes(kernel_id: int) -> float:
    """Traceback bytes written per DP cell (Pair16Geom / TraceGeom in the kernels)."""
    return 48.0 / 42.0 if kernel_id in (16, 17, 18) else 24.0 / 21.0


def strong_scaling(data, off, world: int, debug: bool) -> dict:
    """A FIXED job on all `world` GPUs: rows [0, STRONG_X) x columns [0, STRONG_Y) of the C3 pair
    matrix through MultiEngine.align_matrix -- static LPT row tiles, one host thread per GPU, every
    GPU's D2H copy landing in its tiles' slice of one page-locked host matrix.  Timed from the call
    to the last byte in host memory (the gather is inside)."""
    from taxi2_b200.engine import PinnedArray
    from taxi2_b200.multi import MultiEngine

    multi = MultiEngine(list(range(world)))
    try:
        multi.load((data[: off[STRONG_X]], off[: STRONG_X + 1]), 0)
        multi.load((data[: off[STRONG_Y]], off[: STRONG_Y + 1]), 1)
        counts = PinnedArray((STRONG_X, STRONG_Y, 4), np.int32)
        metrics = PinnedArray((STRONG_X, STRONG_Y, 4), np.float64)
        out = dict(counts=counts.array, metrics=metrics.array)
        multi.align_matrix(want=("counts", "metrics"), x_range=(0, 64 * world), out=out)   # warm-up: arenas, occupancy queries
        t0 = time.perf_counter()
        res = multi.align_matrix(want=("counts", "metrics"), out=out)
        dt = time.perf_counter() - t0
        pairs = STRONG_X * STRONG_Y
        return dict(
            job=f"{STRONG_X} x {STRONG_Y} ordered pairs of the C3 matrix, counts + 4 metrics gathered into one pinned host matrix "
                f"({(counts.nbytes + metrics.nbytes) / 1e9:.1f} GB)",
            n_gpus=world, pairs=pairs, seconds=dt, value=pairs / dt, unit="pairs/s", gcups=res["cells"] / dt / 1e9,
            tiles=res["tiles"], kernel_seconds_sum=res["kernel_ms"] / 1e3, gather="host (pinned), inside the timed region; no collective",
            checksum=int(res["counts"][::97, ::89].sum()))
    finally:
        multi.close()


def versus_all_symmetric(data, off, world: int) -> dict:
    """versusAll on the first SYM_N sequences of C3 as a whole job on all `world` GPUs: every ORDERED pair's
    counts and metrics in one page-locked n x n host matrix (versus_all.py:746 aligns (x, y) and (y, x)),
    from ONE alignment per unordered pair -- the kernel notes on the traced path whether the other
    orientation could align differently (a tie between a vertical and a horizontal gap), those pairs
    are re-aligned, the rest mirrored (MultiEngine.align_matrix_symmetric).  `value` counts ordered pairs
    DELIVERED per second; `alignments` is what was actually aligned.  A band of rows is checked
    against the ordinary one-alignment-per-ordered-pair path inside the run."""
    from taxi2_b200.engine import PinnedArray
    from taxi2_b200.multi import MultiEngine

    multi = MultiEngine(list(range(world)))
    try:
        multi.load((data[: off[SYM_N]], off[: SYM_N + 1]), 0)
        counts = PinnedArray((SYM_N, SYM_N, 4), np.int32)
        metrics = PinnedArray((SYM_N, SYM_N, 4), np.float64)
        out = dict(counts=counts.array, metrics=metrics.array)
        band = multi.align_matrix(want=("counts", "metrics"), x_range=(SYM_N // 2, SYM_N // 2 + 64 * world))   # also the warm-up
        runs = []
        for _ in range(2):   # the whole job twice, the faster one reported (both listed): host-side hiccups of a 3 GB gather are not the subject
            t0 = time.perf_counter()
            res = multi.align_matrix_symmetric(want=("counts", "metrics"), out=out)
            runs.append(time.perf_counter() - t0)
        dt = min(runs)
        rows = slice(SYM_N // 2, SYM_N // 2 + 64 * world)
        same = bool(np.array_equal(band["counts"], res["counts"][rows]) and
                    np.array_equal(band["metrics"].view(np.int64), res["metrics"][rows].view(np.int64)))
        pairs = SYM_N * SYM_N
        lens = np.diff(off[: SYM_N + 1])
        return dict(
            job=f"versusAll of {SYM_N} C3 sequences: {pairs} ordered pairs, counts + 4 metrics in one pinned host matrix "
                f"({(counts.nbytes + metrics.nbytes) / 1e9:.1f} GB), one alignment per unordered pair + re-alignment of the orientation-sensitive ones",
            n_gpus=world, ordered_pairs=pairs, seconds=dt, seconds_of_each_run=runs, value=pairs / dt, unit="ordered pairs/s delivered",
            alignments=int(round(res["cells"] / float(lens.mean()) ** 2)), realigned=int(res["redo"]), gcups_computed=res["cells"] / dt / 1e9,
            tiles=res["tiles"], kernel_seconds_sum=res["kernel_ms"] / 1e3,
            identical_to_ordered_path=same, rows_checked=64 * world, checksum=int(res["counts"][::97, ::89].sum()))
    finally:
        multi.close()


# ---- C2 / C4 / C5: one process drives N GPUs ---------------------------------------------------------
def run_config(args) -> None:
    import torch

    from taxi2_b200.engine import PinnedArray
    from taxi2_b200.multi import MultiEngine

    world = args.gpus
    if torch.cuda.device_count() < world:
        raise SystemExit(f"bench.py: --gpus {world} but {torch.cuda.device_count()} CUDA device(s) visible")
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    multi = MultiEngine(list(range(world)))
    cfg = args.config
    hbm, hbm_how = peak_hbm()

    if cfg == "C2":
        data, off = make_prealigned(args.nseq or 9000)
        n = len(off) - 1
        multi.load((data, off), 0)
        pairs = n * n
        # device-resident: one block of rows per GPU, results left in HBM
        tiles = multi.row_tiles(rows_per_tile=-(-n // world))

        def resident(engine, tile, slot):
            engine.count_rect_resident(tile.x0, tile.nx, 0, n)
            return engine.stats()

        def step():
            return [s for _, s in multi.run_tiles(tiles, resident, ordered=False)]

        counts = PinnedArray((n, n, 4), np.int32)
        metrics = PinnedArray((n, n, 4), np.float64)
        out = dict(counts=counts.array, metrics=metrics.array)

        def step_e2e():
            multi.load((data, off), 0)
            return multi.count_matrix(want=("counts", "metrics"), out=out)

        value_pairs, cells = pairs, 0
        kernel = "count_tc_kernel (tcgen05 int8 contraction + fused trim/metric epilogue)"
        h2d, d2h = data.nbytes + off.nbytes, counts.nbytes + metrics.nbytes
        cpu_run = lambda: cpu_count_throughput(data, off, args.cpu_seconds)   # noqa: E731
        cpu_sample = "random ordered pairs of the C2 rows"
        dtype = "u32 bit planes + f64 metrics"
        meta = workload("C2", world, n=n)
    elif cfg == "C4":
        refs = 20_000
        queries = args.queries or 200_000
        data, off = make_sequences(queries + refs, seed=200020)
        qd, qo = data[: off[queries]], off[: queries + 1]
        rd, ro = data[off[queries]:], off[queries:] - off[queries]
        multi.load((qd, qo), 0)
        multi.load((rd, ro), 1)
        pairs = queries * refs
        last = {}

        def step():
            res = multi.best_matches(metric=0, align=True)
            last.update(res)
            return [dict(kernel_ms=res["kernel_ms"], cells=res["cells"], launches=res["launches"])]

        # end to end on a quarter of the queries (the same references): upload of both sets from host
        # memory + alignment + winners back on the host
        e2e_queries = max(1, queries // 4)

        def step_e2e():
            multi.load((data[: off[e2e_queries]], off[: e2e_queries + 1]), 0)
            multi.load((rd, ro), 1)
            return multi.best_matches(metric=0, align=True)

        e2e_pairs = e2e_queries * refs
        value_pairs = pairs
        kernel = "gotoh_pair16_kernel<21,1>"
        h2d, d2h = int(off[e2e_queries]) + rd.nbytes + 8 * (e2e_queries + 1) + ro.nbytes, e2e_queries * (4 + 32 + 16)
        cpu_run = lambda: cpu_align_throughput(data, off, args.cpu_seconds, tile_pairs(0, min(queries, 4096), queries, refs))   # noqa: E731
        cpu_sample = "random (query, reference) pairs of the same sets"
        dtype = "u16x2"
        meta = workload("C4", world, queries=queries, refs=refs)
    else:
        n = args.nseq or 16384
        data, off = make_mixed(n)
        multi.load((data, off), 0)
        pairs = n * n
        tiles = multi.row_tiles()

        def resident(engine, tile, slot):
            engine.align_rect_resident(tile.x0, tile.nx, 0, n, want=("metrics",))
            return engine.stats()

        def step():
            return [s for _, s in multi.run_tiles(tiles, resident, ordered=False)]

        def step_e2e():
            multi.load((data, off), 0)
            total = 0

            def block(engine, tile, slot):
                return engine.align_rect(tile.x0, tile.nx, 0, n, want=("metrics",), pinned=True, slot=slot)["metrics"]

            # the consumer of a task: blocks in row order, each looked at once (dereplicate's threshold test)
            for _, m in multi.run_tiles(tiles, block, depth=2, ordered=True):
                total += int((m[..., 0] <= 0.07).sum())
            return dict(similar=total)

        value_pairs = pairs
        kernel = "gotoh_pair16_kernel<*> (rows grouped by geometry)"
        h2d, d2h = data.nbytes + off.nbytes, pairs * 32
        cpu_run = lambda: cpu_align_throughput(data[: off[min(n, 4096)]], off[: min(n, 4096) + 1], args.cpu_seconds,   # noqa: E731
                                               tile_pairs(0, min(n, 4096), 0, min(n, 4096)))
        cpu_sample = "random ordered pairs of the first 4096 sequences"
        dtype = "u16x2"
        meta = workload("C5", world, n=n)

    # warm-up on the real job is too long for C4/C5: a short slice sizes the arenas instead
    if cfg == "C2":
        for _ in range(args.warmup):
            step()
    else:
        warm_rows = 64 * world
        wt = multi.row_tiles(x_range=(0, min(warm_rows, multi.nx)))
        if cfg == "C4":
            for _ in range(args.warmup):
                for _t, _r in multi.run_tiles(wt, lambda e, t, s: e.best_rows(t.x0, t.nx, 0, multi.ny, 0, True), ordered=False):
                    pass
        else:
            for _ in range(args.warmup):
                for _t, _r in multi.run_tiles(wt, lambda e, t, s: e.align_rect_resident(t.x0, t.nx, 0, multi.ny, want=("metrics",)), ordered=False):
                    pass
    with ClockSampler(0 if not os.environ.get("TAXI_NO_SAMPLER") else -1) as clocks:
        t0 = time.perf_counter()
        stats = []
        for _ in range(args.steps):
            stats += step()
        dt = time.perf_counter() - t0
    kernel_ms = sum(s["kernel_ms"] for s in stats)
    cells = sum(s["cells"] for s in stats)
    launches = sum(s["launches"] for s in stats)
    clk = clocks.summary()

    step_e2e()                       # untimed: pinned staging reaches its steady size
    t1 = time.perf_counter()
    e2e_steps = 1 if cfg != "C2" else args.steps
    for _ in range(e2e_steps):
        extra = step_e2e()
    dt_e2e = time.perf_counter() - t1

    value = value_pairs * args.steps / dt
    if cfg == "C2":
        if multi.engines[0].last_kernel == 8:
            kernel = "count_rect_kernel (popcount)"
        bytes_per_pair = 48.0
        launch_s = kernel_ms / 1e3 / max(launches, 1)
        pairs_per_launch = pairs * args.steps / max(launches, 1)
        lanes, lanes_how = int32_lanes()
        mhz = clk.get("sm_mhz") or 1965.0
        W = (618 + 31) // 32
        roof = dict(bound="hbm", kernel=kernel, achieved=pairs_per_launch * bytes_per_pair / launch_s / 1e9, peak=hbm, unit="GB/s",
                    frac=pairs_per_launch * bytes_per_pair / launch_s / 1e9 / hbm,
                    traffic=(ncu_traffic(kernel) or {}).get("bytes_per_pair", 0) * pairs_per_launch or None,
                    traffic_source=(ncu_traffic(kernel) or {}).get("source"),
                    how=f"{bytes_per_pair:.0f} algorithmic bytes/pair (16 B counts + 32 B metrics written once; the {n * W * 16 / 1e6:.1f} MB of bit planes are "
                        f"re-read from L2) x {pairs_per_launch:.3e} pairs/launch / {launch_s * 1e3:.3f} ms per launch (CUDA events); peak = {hbm_how}",
                    int32=dict(ops_per_pair=12 * W, achieved=pairs_per_launch * 12 * W / launch_s / 1e9, peak=lanes * sms * mhz * 1e6 / 1e9, unit="Gop/s",
                               note=f"SURVEY 8d: ~12 integer ops per 32-column word; peak = {lanes:.2f} lane-ops/clk/SM x {sms} SMs x {mhz:.0f} MHz sampled"))
    else:
        # per-device launch duration: the kernel time summed over devices / launches
        cells_per_launch = cells / max(launches, 1)
        launch_s = kernel_ms / 1e3 / max(launches, 1)
        roof = int_roofline(cells_per_launch, launch_s, clk, sms, kernel, True)
        roof["hbm"] = dict(achieved=cells_per_launch * trace_bytes(17) / launch_s / 1e9, peak=hbm, unit="GB/s",
                           note="algorithmic HBM traffic: traceback codes written once")
    cpu = cpu_run()
    line = dict(
        metric="aligned_pairs_per_sec" if cfg != "C2" else "pairs_per_sec", value=value, unit="pairs/s",
        gcups=cells / dt / 1e9 if cells else None, n_gpus=world, steps=args.steps, warmup=args.warmup, ms_per_step=1e3 * dt / args.steps,
        higher_is_better=True, scaling="strong", vs_baseline=None, dtype=dtype, data="synthetic", config=meta, roofline=roof,
        cpu_baseline=dict(value=cpu["pairs"] / cpu["seconds"], unit="pairs/s", gcups=(cpu["cells"] / cpu["seconds"] / 1e9) if cpu["cells"] else None,
                          cores=cpu["threads"], kind="port", sample=f"{cpu['pairs']} {cpu_sample} in {cpu['seconds']:.1f} s"),
        e2e=dict(value=(e2e_pairs if cfg == "C4" else value_pairs) * e2e_steps / dt_e2e, unit="pairs/s", h2d_bytes_per_step=h2d,
                 d2h_bytes_per_step=d2h, steps=e2e_steps, seconds=dt_e2e,
                 **({"job": f"{e2e_queries} queries x {refs} references (a quarter of the queries)"} if cfg == "C4" else {})),
        gpu_launches=launches, clocks=clk, kernel_seconds_sum=kernel_ms / 1e3,
    )
    if cfg == "C4":
        line["winners_defined"] = int((last["index"] >= 0).sum())
        line["checksum"] = int(last["index"].astype(np.int64).sum())
    if cfg == "C5":
        line["similar_pairs"] = extra["similar"]
    print(json.dumps(line), flush=True)
    multi.close()


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=None)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="taxi2_b200", choices=["taxi2_b200", "reference"])
    ap.add_argument("--config", default="C3", choices=["C2", "C3", "C4", "C5"])
    ap.add_argument("--cpu-seconds", type=float, default=12.0)
    ap.add_argument("--nseq", type=int, default=None, help="C3: sequences generated (default 50000); C2: rows (9000); C5: sequences (16384)")
    ap.add_argument("--queries", type=int, default=None, help="C4: queries (default 200000) against 20000 references")
    ap.add_argument("--no-strong", dest="strong", action="store_false", help="C3: skip the fixed-job strong-scaling sub-record")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="C3: write counts.npy and metrics.npy of the last timed step (a seeded sample of its pairs) to DIR")
    args = ap.parse_args()
    if args.steps is None:
        args.steps = 5 if args.config in ("C3", "C2") else 1
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be at least 1 and --warmup at least 0")
    if args.dump_outputs and (args.config != "C3" or args.impl != "taxi2_b200"):
        ap.error("--dump-outputs is implemented for the C3 workload of taxi2_b200 only")

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    ensure_built(local_rank)

    if args.impl == "reference":
        run_reference(args, rank, world)
        return

    import torch

    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; taxi2_b200 has no CPU path (use --impl reference for the CPU baseline)")
    if args.config == "C3":
        run_c3(args, rank, local_rank, world)
    elif rank == 0:
        run_config(args)


if __name__ == "__main__":
    main()
