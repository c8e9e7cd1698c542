"""The aligner's device-resident outputs, written into memory the caller owns.

`taxi_align_rect_device` and `taxi_align_rect_both_device` store counts and metrics straight into the
caller's tensors (the benchmark's device-resident number is measured that way).  Every other aligned
test reads its results through the library's own device buffers, which are reused from call to call, so
a pair a kernel never writes would come back holding an earlier call's value.  Here every output is a
fresh torch tensor of n + 2 G pairs filled with a sentinel no result can take (score INT32_MIN, which
the range check rules out; counts -7; metrics -7.0), and the call gets `base + G`.  After each call:
- no sentinel is left inside the rectangle (every pair written),
- both guard bands of G pairs are untouched (nothing written outside it),
- a buffer whose output was not requested is untouched (its pointer is passed all the same, through
  the raw ABI, since the Python wrapper derives the flags from the pointers).
Inside the rectangle the results are bit for bit the host form of the same call, scores and counts the
oracle's (the whole rectangle where that is cheap, else a seeded sample), metrics bit for bit
`taxi_metrics_from_counts` of the kernel's own counts.

Cases: every compiled aligner instance in rectangle form (`kernel_geometry.py` picks the row counts),
at 3 x 5 pairs with offsets and, for the packed families, at more warp units than resident warps; the
row-grouped launches; all seven output subsets on one instance of each family; both orientations in
device form (re-aligned pairs, both fallbacks, each output alone); launches queued without a sync;
one device call above 2^24 pairs; the benchmark's own tiles; `taxi_argmin_rows_device`; and the
refusal of misaligned pointers."""
from __future__ import annotations

import ctypes as C
import itertools

import numpy as np
import pytest

import kernel_geometry as K
from taxi2_b200 import _native as N
from test_gpu_align import oracle_batch
from test_gpu_kernel_geometries import DEFAULT, TOP, WIDE, Options, assert_epilogue, tie_set

gpu = pytest.mark.gpu

G = 1024                                   # guard pairs on each side of a rectangle
SENTINEL = {"score": -2**31, "counts": -7, "metrics": -7.0}
KEYS = ("score", "counts", "metrics")
FLAG = {"score": N.OUT_SCORE, "counts": N.OUT_COUNTS, "metrics": N.OUT_METRICS}
SUBSETS = [s for r in (1, 2, 3) for s in itertools.combinations(KEYS, r)]
FULL_CELLS = 3e8                           # the oracle checks the whole rectangle up to this many DP cells ...
SAMPLE = 300                               # ... else this many seeded pairs
LIMIT = 4096                               # highest row count scanned per instance
TAIL_COLS = 33                             # 17 warp units per row, the last one half empty
E_ARG = -1


# -- the plan (no GPU) ------------------------------------------------------------------------------

def _rand(rng, n: int, alphabet: bytes = b"ACGT") -> bytes:
    al = np.frombuffer(alphabet, dtype=np.uint8)
    return al[rng.integers(0, len(al), max(1, n))].tobytes()


def related(rng, n: int, lo: int, hi: int) -> list[bytes]:
    """n sequences with lengths in [lo, hi], the first of length hi: prefixes of one random root with
    10 % of their positions redrawn and a two-base deletion next to a two-base insertion (length kept)."""
    root = _rand(rng, hi)
    out = []
    for k in range(n):
        s = bytearray(root[: hi if k == 0 else int(rng.integers(lo, hi + 1))])
        for i in np.flatnonzero(rng.random(len(s)) < 0.1):
            s[i] = int(b"ACGT"[rng.integers(0, 4)])
        if len(s) > 8:
            at = int(rng.integers(0, len(s) - 4))
            s[at:at + 2] = b""
            at = int(rng.integers(0, len(s)))
            s[at:at] = _rand(rng, 2)
        out.append(bytes(s))
    return out


def _scores_for(family: str, H: int):
    """The first score set under which some row count selects (family, H), and its runs."""
    sets = {"top": (TOP, DEFAULT), "multi": (DEFAULT, WIDE)}.get(family, (DEFAULT,))
    for scores in sets:
        runs = K.selecting_rows(family, H, scores, 1023 if family == "both" else LIMIT)
        if runs:
            return scores, runs
    return None, []


def plan() -> list[dict]:
    """One case per launch: every compiled instance at 3 x 5 pairs ("odd"), the packed ones also at more
    warp units than resident warps ("tail"), and the row-grouped rectangle ("split")."""
    cases = []
    tail_rows = -(-40 * K.SMS // ((TAIL_COLS + 1) // 2))     # 2.5 x the warps of 4 blocks of 4 per SM, and more
    for family, H in K.compiled_instances():
        scores, runs = _scores_for(family, H)
        if scores is None:
            continue
        lo, hi = runs[-1]
        if family == "both":
            lo = max(lo, hi // 2 + 1)                          # the both-orientations kernel wants 2 min > max
        base = dict(family=family, H=H, scores=scores, opts=K.family_options(family, scores))
        cases.append(dict(base, id=f"{K.name(family, H)}-odd", kind="odd", lo=lo, hi=hi, nx=3, ny=5))
        if family in ("top", "bottom", "multi", "both"):
            cases.append(dict(base, id=f"{K.name(family, H)}-tail", kind="tail", lo=max(lo, hi - 64), hi=hi,
                              nx=tail_rows, ny=TAIL_COLS))
    cases.append(dict(id="split-odd", family="split", H=0, scores=DEFAULT, opts={}, kind="split", nx=3, ny=5))
    return cases


PLAN = plan()


def _seed(case) -> int:
    return sum(ord(ch) * (k + 1) for k, ch in enumerate(case["id"])) % 2**32


def case_inputs(case) -> dict:
    """-> xs, ys (None: set 0 serves as both), the rectangle (x0, nx, y0, ny) and the predicted instance."""
    rng = np.random.default_rng(_seed(case))
    nx, ny = case["nx"], case["ny"]
    if case["kind"] == "split":
        rows = [related(rng, 1, L, L)[0] for L in (900, 1200, 1000)]     # both sides of 1 023 bp
        cols = related(rng, ny, 300, 700)
        xs, ys, x0, y0 = [_rand(rng, 500), _rand(rng, 400)] + rows + [_rand(rng, 600)], [_rand(rng, 300)] + cols, 2, 1
    elif case["family"] == "both":
        xs = related(rng, 2 + max(nx, ny), case["lo"], case["hi"])
        xs[0], xs[2] = xs[2], xs[0]                              # the longest inside both ranges
        ys, x0, y0 = None, 2, 1
    else:
        lo, hi = case["lo"], case["hi"]
        rows, cols = related(rng, nx, lo, hi), related(rng, ny, lo, hi)
        xs, ys, x0, y0 = [_rand(rng, lo), _rand(rng, lo)] + rows + [_rand(rng, lo)], [_rand(rng, lo)] + cols + [_rand(rng, lo)] * 2, 2, 1
    yset = xs if ys is None else ys
    la, lb = [len(s) for s in xs[x0:x0 + nx]], [len(s) for s in yset[y0:y0 + ny]]
    form = "both" if case["family"] == "both" else "rect"
    predicted = K.instance(case["scores"], la, lb, form, case["opts"])
    return dict(xs=xs, ys=ys, rect=(x0, nx, y0, ny), predicted=predicted)


def expected_code(case) -> int:
    return 48 if case["family"] == "split" else K.CODE[case["family"]]


def test_plan_covers_every_compiled_instance():
    """Every (family, H) the library compiles has a case, and each case's inputs select it (an instance
    added to the dispatch tables without a case fails here, without a GPU)."""
    planned = {(c["family"], c["H"]) for c in PLAN if c["family"] != "split"}
    assert planned == set(K.compiled_instances()), set(K.compiled_instances()) ^ planned
    for case in PLAN:
        got = case_inputs(case)["predicted"]
        want = ("split", 0, 0) if case["family"] == "split" else (case["family"], case["H"])
        assert got[:len(want)] == want, (case["id"], got)
        if case["kind"] == "tail":
            assert case["nx"] * ((case["ny"] + 1) // 2) > 2 * 16 * K.SMS and case["ny"] % 2 == 1
    assert {c["family"] for c in PLAN} >= {"general", "coop", "top", "bottom", "multi", "both", "split"}


# -- caller-owned buffers -----------------------------------------------------------------------------

class Outputs:
    """One caller-owned device buffer per output, n + 2 G pairs of its sentinel; pair k of the call is
    pair G + k of the buffer."""

    def __init__(self, n: int):
        import torch

        self.n = n
        self.t = {key: torch.full((n + 2 * G,) if key == "score" else (n + 2 * G, 4), SENTINEL[key],
                                  dtype=torch.float64 if key == "metrics" else torch.int32, device="cuda")
                  for key in KEYS}
        torch.cuda.synchronize()   # the library's stream does not wait for torch's: the fill must be done first

    def ptr(self, key: str, at: int = 0) -> int:
        t = self.t[key]
        return t.data_ptr() + (G + at) * t[0].numel() * t.element_size()

    def args(self, at: int = 0) -> list:
        return [C.c_void_p(self.ptr(key, at)) for key in KEYS]

    def check(self, want, where) -> dict:
        """Guard bands and unrequested buffers untouched, no sentinel left among the n pairs -> numpy arrays."""
        out = {}
        for key in KEYS:
            a = self.t[key].cpu().numpy()
            same = (a == SENTINEL[key]).reshape(len(a), -1)      # per pair and element: still the sentinel
            touched = np.flatnonzero(~same.all(axis=1)) - G      # pairs with any element written, call-relative
            if key not in want:
                assert len(touched) == 0, (where, key, "written though not requested, pairs", touched[:8].tolist())
                continue
            outside = touched[(touched < 0) | (touched >= self.n)]
            assert len(outside) == 0, (where, key, "guard band written at pairs", outside[:8].tolist())
            left = np.flatnonzero(same[G:G + self.n].any(axis=1))
            assert len(left) == 0, (where, key, f"{len(left)} of {self.n} pairs left unwritten", left[:8].tolist())
            out[key] = a[G:G + self.n]
        return out


def shaped(res: dict, nx: int, ny: int) -> dict:
    return {k: v.reshape(nx, ny, *v.shape[1:]) for k, v in res.items()}


def align_device(engine, x0, nx, y0, ny, want=KEYS, where=None) -> dict:
    """taxi_align_rect_device through the raw ABI into fresh sentinel buffers, every pointer passed;
    synced and checked -> {key: (nx, ny[, 4]) array} of the requested outputs."""
    out = Outputs(nx * ny)
    flags = sum(FLAG[k] for k in want)
    N.check(engine._lib.taxi_align_rect_device(engine._ctx, x0, nx, y0, ny, flags, *out.args()))
    engine.sync()
    return shaped(out.check(want, where), nx, ny)


def both_device(engine, x0, nx, y0, ny, want=KEYS, where=None) -> tuple[dict, dict]:
    """taxi_align_rect_both_device the same way -> ((x, y) results (nx, ny), (y, x) results (ny, nx))."""
    d, t = Outputs(nx * ny), Outputs(nx * ny)
    flags = sum(FLAG[k] for k in want)
    N.check(engine._lib.taxi_align_rect_both_device(engine._ctx, x0, nx, y0, ny, flags, *d.args(), *t.args()))
    return shaped(d.check(want, (where, "d")), nx, ny), shaped(t.check(want, (where, "t")), ny, nx)


def assert_bits(got: dict, want: dict, where, keys=None):
    for key in keys or got:
        g, w = np.ascontiguousarray(got[key]), np.ascontiguousarray(want[key])
        if key == "metrics":
            g, w = g.view(np.uint64), w.view(np.uint64)
        assert g.shape == w.shape, (where, key, g.shape, w.shape)
        bad = np.argwhere(g != w)
        assert len(bad) == 0, (where, key, len(bad), bad[:4].tolist())


def assert_oracle(got: dict, xs, ys, rect, scores, where, sample: int = SAMPLE):
    """Scores and counts against the oracle over the whole rectangle when that is cheap, else a seeded sample."""
    x0, nx, y0, ny = rect
    ys = xs if ys is None else ys
    cells = sum(map(len, xs[x0:x0 + nx])) * sum(map(len, ys[y0:y0 + ny]))
    if cells <= FULL_CELLS:
        r, c = np.divmod(np.arange(nx * ny), ny)
    else:
        rng = np.random.default_rng(nx * 7919 + ny)
        r, c = rng.integers(0, nx, sample), rng.integers(0, ny, sample)
    want = oracle_batch(xs, ys, (x0 + r).astype(np.int32), (y0 + c).astype(np.int32), scores)
    if "score" in got:
        assert np.array_equal(got["score"][r, c], want["score"]), (where, "score")
    assert np.array_equal(got["counts"][r, c], want["counts"]), (where, "counts")


def load(engine, scores, xs, ys):
    engine.set_scores(scores)
    engine.load(xs, 0)
    if ys is not None:
        engine.load(ys, 1)


# -- a. every compiled instance ----------------------------------------------------------------------

def run_case(engine, case, want=KEYS) -> dict:
    """The case's rectangle in device form (both orientations for the "both" family): kernel, sentinels
    and guard bands, bit for bit the host form, the oracle and the epilogue -> the device results."""
    inp = case_inputs(case)
    xs, ys, rect = inp["xs"], inp["ys"], inp["rect"]
    x0, nx, y0, ny = rect
    where = (case["id"], inp["predicted"])
    with Options(engine, **case["opts"]):
        load(engine, case["scores"], xs, ys)
        if case["family"] == "both":
            got, got_t = both_device(engine, *rect, want=want, where=where)
            assert engine.last_kernel == 20, where
            want_xy, want_yx = engine.align_rect_both(*rect)
            assert_bits(got_t, want_yx, where)
        else:
            got = align_device(engine, *rect, want=want, where=where)
            assert engine.last_kernel == expected_code(case), (where, engine.last_kernel)
            want_xy = engine.align_rect(*rect)
    assert_bits(got, want_xy, where)
    if "counts" in want:
        assert_oracle(got, xs, ys, rect, case["scores"], where)
        if "metrics" in want:
            assert_epilogue(engine, got, where)
    return got


@gpu
@pytest.mark.parametrize("case", PLAN, ids=lambda c: c["id"])
def test_every_instance_in_caller_memory(engine, case):
    run_case(engine, case)


# -- b. output subsets ----------------------------------------------------------------------------------

SUBSET_CASES = [next(c for c in PLAN if c["family"] == f and c["kind"] in ("odd", "split"))
                for f in ("general", "coop", "top", "bottom", "multi", "split")]


@gpu
@pytest.mark.parametrize("case", SUBSET_CASES, ids=lambda c: c["id"])
def test_every_output_subset(engine, case):
    """All seven non-empty subsets of {score, counts, metrics}, every pointer passed: a requested output
    equals the full call's bit for bit, an unrequested buffer keeps its sentinel (Outputs.check)."""
    full = run_case(engine, case)
    inp = case_inputs(case)
    with Options(engine, **case["opts"]):
        load(engine, case["scores"], inp["xs"], inp["ys"])
        for want in SUBSETS:
            got = align_device(engine, *inp["rect"], want=want, where=(case["id"], want))
            assert engine.last_kernel == expected_code(case), (case["id"], want)
            assert_bits(got, full, (case["id"], want), keys=want)


# -- c. both orientations, device form ----------------------------------------------------------------

def both_sets():
    rng = np.random.default_rng(2024)
    from synth import coi_like

    return {
        "ties": (DEFAULT, [s for _ in range(4) for s in tie_set(rng, 8, 100, 160)]),     # many re-aligned pairs
        "coi": (DEFAULT, coi_like(40, length=300, seed=21)),                               # few: the last pair mirrored
        "mixed": (DEFAULT, related(rng, 30, 100, 400)),                                    # lo * 2 <= max_len: two launches
        "top": (TOP, coi_like(30, length=200, seed=22)),                                   # top-aligned: two launches
    }


BOTH = both_sets()
BOTH_RECT = (3, 21, 2, 27)      # odd sizes, offsets; set 0 serves as both


@gpu
@pytest.mark.parametrize("name", list(BOTH))
def test_both_orientations_device_form(engine, name):
    """d_* and t_* in caller memory, bit for bit the host form, the oracle in both orientations, and the
    header's claim taken literally: t_* equals taxi_align_rect_device over the exchanged ranges."""
    scores, xs = BOTH[name]
    x0, nx, y0, ny = BOTH_RECT
    la, lb = [len(s) for s in xs[x0:x0 + nx]], [len(s) for s in xs[y0:y0 + ny]]
    predicted = K.instance(scores, la, lb, "both")
    load(engine, scores, xs, None)
    got, got_t = both_device(engine, *BOTH_RECT, where=name)
    kernel, redo = engine.last_kernel, engine.last_redo
    assert kernel == K.CODE[predicted[0]], (name, predicted, kernel)
    if name in ("ties", "coi"):
        assert predicted[0] == "both", predicted
        assert redo > 0 or name == "coi", (name, redo)     # ties: the re-aligned pairs go through scatter_redo_kernel
    else:
        assert predicted[0] != "both" and redo == 0, (name, predicted, redo)
    want_xy, want_yx = engine.align_rect_both(*BOTH_RECT)
    assert_bits(got, want_xy, (name, "xy"))
    assert_bits(got_t, want_yx, (name, "yx"))
    assert_oracle(got, xs, None, BOTH_RECT, scores, (name, "xy"))
    assert_oracle(got_t, xs, None, (y0, ny, x0, nx), scores, (name, "yx"))
    assert_epilogue(engine, got_t, (name, "yx"))
    assert_bits(got, align_device(engine, *BOTH_RECT), (name, "xy = rect_device"))
    assert_bits(got_t, align_device(engine, y0, ny, x0, nx), (name, "yx = rect_device of the exchanged ranges"))
    for want in (("counts",), ("metrics",), ("score",)):
        d, t = both_device(engine, *BOTH_RECT, want=want, where=(name, want))
        assert_bits(d, got, (name, want, "d"), keys=want)
        assert_bits(t, got_t, (name, want, "t"), keys=want)


# -- d. launches queued without a sync ----------------------------------------------------------------

@gpu
def test_launches_queued_without_a_sync(engine):
    """Three rectangles taking different instances (bottom, row-grouped, general) enqueued back to back
    into disjoint slices of one caller tensor, synced once: each slice equals its own synchronous run."""
    rng = np.random.default_rng(75)
    xs = related(rng, 10, 300, 700) + [related(rng, 1, L, L)[0] for L in (900, 1200, 1000, 1100, 950)]
    ys = related(rng, 9, 300, 700)
    rects = {"bottom": ((0, 9, 0, 7), {}), "split": ((9, 5, 1, 5), {}), "general": ((2, 5, 3, 3), {"force_general": 1})}
    for name, ((x0, nx, y0, ny), opts) in rects.items():
        la, lb = [len(s) for s in xs[x0:x0 + nx]], [len(s) for s in ys[y0:y0 + ny]]
        assert K.instance(DEFAULT, la, lb, "rect", opts)[0] == name
    load(engine, DEFAULT, xs, ys)
    total = sum(r[1] * r[3] for r, _ in rects.values())
    out = Outputs(total)
    at, kernels = 0, {}
    for name, (rect, opts) in rects.items():
        with Options(engine, **opts):
            N.check(engine._lib.taxi_align_rect_device(engine._ctx, *rect, N.OUT_SCORE | N.OUT_COUNTS | N.OUT_METRICS, *out.args(at)))
            kernels[name] = engine.last_kernel
        at += rect[1] * rect[3]
    engine.sync()
    assert kernels == {"bottom": 17, "split": 48, "general": 32}, kernels
    whole = out.check(KEYS, "queued")
    at = 0
    for name, (rect, opts) in rects.items():
        x0, nx, y0, ny = rect
        with Options(engine, **opts):
            alone = align_device(engine, *rect, where=name)
        part = shaped({k: v[at:at + nx * ny] for k, v in whole.items()}, nx, ny)
        assert_bits(part, alone, (name, "queued vs alone"))
        assert_oracle(part, xs, ys, rect, DEFAULT, name)
        at += nx * ny


# -- e. one device call above 2^24 pairs -------------------------------------------------------------

@gpu
def test_one_device_call_above_one_host_block(engine):
    """The device form has no row chunking: 5 000 x 3 400 pairs (> 2^24) in one call equal the host
    form's chunked walk bit for bit, every pair written."""
    rng = np.random.default_rng(224)
    al = np.frombuffer(b"ACGT", dtype=np.uint8)
    xs = [al[rng.integers(0, 4, int(rng.integers(20, 41)))].tobytes() for _ in range(5000)]
    ys = [al[rng.integers(0, 4, int(rng.integers(20, 41)))].tobytes() for _ in range(3400)]
    assert len(xs) * len(ys) > 1 << 24
    load(engine, DEFAULT, xs, ys)
    rect = (0, len(xs), 0, len(ys))
    got = align_device(engine, *rect, where="2^24")
    want = engine.align_rect(*rect)
    assert engine.stats()["launches"] >= 2           # the host form walked it in blocks
    assert_bits(got, want, "2^24")
    assert_oracle(got, xs, ys, rect, DEFAULT, "2^24")


# -- f. the benchmark's workloads ---------------------------------------------------------------------

@gpu
def test_benchmark_tile_through_its_entry_point(engine):
    """One full TILE_X x TILE_Y tile of the benchmark's sequences through Engine.align_rect_device with
    counts and metrics and no score, exactly as bench.py's step_device: the whole tile bit for bit the
    host form, a seeded sample the oracle's; and rows of its mixed-length set, metrics only as in its
    C5 leg, against the counts of the full call."""
    import bench

    data, off = bench.make_sequences(bench.TILE_Y)
    seqs = [data[off[k]:off[k + 1]].tobytes() for k in range(len(off) - 1)]
    engine.set_scores(None)
    engine.load((data, off), 0)
    npairs = bench.TILE_X * bench.TILE_Y
    out = Outputs(npairs)
    engine.align_rect_device(0, bench.TILE_X, 0, bench.TILE_Y, 0, out.ptr("counts"), out.ptr("metrics"))
    engine.sync()
    lens = np.diff(off)
    assert engine.last_kernel == K.CODE[K.instance(DEFAULT, lens[:bench.TILE_X], lens[:bench.TILE_Y], "rect")[0]]
    got = shaped(out.check(("counts", "metrics"), "tile"), bench.TILE_X, bench.TILE_Y)
    want = engine.align_rect(0, bench.TILE_X, 0, bench.TILE_Y, want=("counts", "metrics"))
    assert_bits(got, want, "tile")
    assert_oracle(got, seqs, None, (0, bench.TILE_X, 0, bench.TILE_Y), None, "tile")

    data, off = bench.make_mixed(1024)
    seqs = [data[off[k]:off[k + 1]].tobytes() for k in range(len(off) - 1)]
    engine.load((data, off), 0)
    rect = (100, 64, 0, 1024)
    predicted = K.instance(DEFAULT, [len(s) for s in seqs[100:164]], [len(s) for s in seqs], "rect")
    out = Outputs(64 * 1024)
    engine.align_rect_device(*rect, 0, 0, out.ptr("metrics"))
    engine.sync()
    assert engine.last_kernel == (48 if predicted[0] == "split" else K.CODE[predicted[0]]), predicted
    got = shaped(out.check(("metrics",), "mixed"), 64, 1024)
    full = engine.align_rect(*rect)
    assert_bits(got, full, "mixed", keys=("metrics",))
    assert_epilogue(engine, dict(counts=full["counts"], metrics=got["metrics"]), "mixed")
    assert_oracle(full, seqs, None, rect, None, "mixed")


# -- g. taxi_argmin_rows_device ---------------------------------------------------------------------

def argmin_reference(v: np.ndarray) -> tuple[np.ndarray, np.ndarray]:
    """Per row of v (nx, ny): the first column holding the smallest value that is not NaN (-0.0 and 0.0
    are equal), -1 / NaN for a row without one."""
    nan = np.isnan(v)
    best = np.where(nan, np.inf, v).min(axis=1, initial=np.inf)
    hit = ~nan & (v == best[:, None])
    has = hit.any(axis=1)
    idx = np.where(has, hit.argmax(axis=1), -1).astype(np.int32)
    val = np.where(has, v[np.arange(len(v)), np.maximum(idx, 0)], np.nan)
    return idx, val


POOL = np.array([0.0, -0.0, 0.0625, 0.25, 0.25, 0.5, 1.0, 5e-324, 2.5e-310, np.inf, -np.inf, np.nan, np.nan])


def argmin_matrix(rng, nx: int, ny: int) -> np.ndarray:
    """(nx, ny, 4) values drawn from POOL (exact ties, signed zeros, subnormals, +-inf, NaN), with rows
    of only NaN, of only one value, of NaN and +inf, and of distinct values."""
    m = POOL[rng.integers(0, len(POOL), (nx, ny, 4))]
    if nx:
        m[rng.random(nx) < 0.1] = np.nan
        m[rng.random(nx) < 0.05] = 0.25
        inf_nan = rng.random(nx) < 0.05
        m[inf_nan] = np.where(rng.random((int(inf_nan.sum()), ny, 4)) < 0.5, np.inf, np.nan)
        distinct = rng.random(nx) < 0.1
        m[distinct] = rng.random((int(distinct.sum()), ny, 4))
    return m


def argmin_raw(engine, ptr: int, nx: int, ny: int, metric: int, value: bool = True):
    idx = np.full(max(nx, 1), -5, dtype=np.int32)
    val = np.full(max(nx, 1), -5.0)
    rc = engine._lib.taxi_argmin_rows_device(engine._ctx, C.c_void_p(ptr), nx, ny, metric, C.c_void_p(idx.ctypes.data),
                                             C.c_void_p(val.ctypes.data) if value else None)
    return rc, idx[:nx], val[:nx]


ARGMIN_SHAPES = [(nx, ny) for ny in (1, 31, 32, 33, 1000) for nx in (0, 1, 7, 8, 9)] + [(100_003, 1), (100_003, 33)]


@gpu
@pytest.mark.parametrize("nx,ny", ARGMIN_SHAPES)
def test_argmin_rows_device(engine, nx, ny):
    """First minimum per row against the reference, index and value bit for bit, every metric column;
    nx ~ 1e5 runs 12 501 blocks of eight warps, the last one partial."""
    import torch

    m = argmin_matrix(np.random.default_rng(nx * 1009 + ny), nx, ny)
    d = torch.from_numpy(m.reshape(-1, 4) if nx else np.zeros((1, 4))).cuda()
    torch.cuda.synchronize()
    for metric in range(4):
        rc, idx, val = argmin_raw(engine, d.data_ptr(), nx, ny, metric)
        assert rc == 0, metric
        want_idx, want_val = argmin_reference(m[..., metric]) if nx else (np.zeros(0, np.int32), np.zeros(0))
        assert np.array_equal(idx, want_idx), (metric, np.flatnonzero(idx != want_idx)[:8])
        assert np.array_equal(val.view(np.uint64), want_val.view(np.uint64)), metric
        rc, idx2, _ = argmin_raw(engine, d.data_ptr(), nx, ny, metric, value=False)   # out_value_host = NULL
        assert rc == 0 and np.array_equal(idx2, want_idx), metric


@gpu
def test_argmin_rows_on_aligned_metrics_and_refusals(engine):
    """argmin over the metrics an align_rect_device call left in caller memory; then the refusals:
    metric 4, ny = 0, nx < 0, a null d_metrics."""
    case = next(c for c in PLAN if c["family"] == "bottom" and c["kind"] == "tail")
    inp = case_inputs(case)
    x0, nx, y0, ny = inp["rect"]
    load(engine, case["scores"], inp["xs"], inp["ys"])
    out = Outputs(nx * ny)
    N.check(engine._lib.taxi_align_rect_device(engine._ctx, x0, nx, y0, ny, N.OUT_METRICS, *out.args()))
    engine.sync()
    m = out.check(("metrics",), "argmin")["metrics"].reshape(nx, ny, 4)
    for metric in range(4):
        idx, val = engine.argmin_rows_device(out.ptr("metrics"), nx, ny, metric)
        want_idx, want_val = argmin_reference(m[..., metric])
        assert np.array_equal(idx, want_idx) and np.array_equal(val.view(np.uint64), want_val.view(np.uint64)), metric
    for args in ((out.ptr("metrics"), nx, ny, 4), (out.ptr("metrics"), nx, ny, -1), (out.ptr("metrics"), nx, 0, 0),
                 (out.ptr("metrics"), -1, ny, 0), (0, nx, ny, 0)):
        rc, idx, _ = argmin_raw(engine, *args)
        assert rc == E_ARG, args
        assert (idx == -5).all(), args


# -- h. misaligned pointers refused -----------------------------------------------------------------

@gpu
def test_misaligned_device_pointers_refused(engine):
    """Counts offset by 4 and 8 bytes, metrics by 8 (and score by 2): refused with TAXI_E_ARG by both
    device entry points, argmin_rows_device refusing a d_metrics off by 4.  An empty rectangle is
    probed first: a library without the check returns OK there and launches nothing, and the test
    stops before any launch could see a misaligned pointer."""
    xs = related(np.random.default_rng(3), 8, 40, 60)
    load(engine, DEFAULT, xs, None)
    out, t = Outputs(64), Outputs(64)
    flags = N.OUT_SCORE | N.OUT_COUNTS | N.OUT_METRICS
    entries = {
        "rect": lambda nx, p, q: engine._lib.taxi_align_rect_device(engine._ctx, 1, nx, 0, 5, flags, *p),
        "both (d)": lambda nx, p, q: engine._lib.taxi_align_rect_both_device(engine._ctx, 1, nx, 0, 5, flags, *p, *q),
        "both (t)": lambda nx, p, q: engine._lib.taxi_align_rect_both_device(engine._ctx, 1, nx, 0, 5, flags, *q, *p),
    }
    for (name, call), (key, shift) in itertools.product(entries.items(), (("counts", 4), ("counts", 8), ("metrics", 8), ("score", 2))):
        bad = [C.c_void_p(out.ptr(k) + (shift if k == key else 0)) for k in KEYS]
        rc = call(0, bad, t.args())
        assert rc == E_ARG, (name, key, shift, "an empty rectangle with a misaligned pointer was accepted: "
                                                 "the alignment check is missing or comes after the empty-input return")
        assert call(3, bad, t.args()) == E_ARG, (name, key, shift)
    out.check((), "refused")                              # nothing written anywhere
    t.check((), "refused")
    m = out.ptr("metrics") + 4
    rc, _, _ = argmin_raw(engine, m, 0, 5, 0)
    assert rc == E_ARG, "argmin_rows_device accepted a misaligned d_metrics for nx = 0: the check is missing or comes too late"
    rc, idx, _ = argmin_raw(engine, m, 3, 5, 0)
    assert rc == E_ARG and (idx == -5).all()


@pytest.fixture(scope="module")
def engine():
    from taxi2_b200.engine import Engine

    eng = Engine(0)
    yield eng
    eng.close()
