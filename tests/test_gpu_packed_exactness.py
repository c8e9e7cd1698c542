"""The packed 16-bit kernel at the edges of its exactness proof (`fast16_eligible`, restated in
`packed16_rule.py`): score sets on both sides of every inequality of the restricted recurrence,
lengths at the last packed length of the 16-bit window and one past it, and warp units whose two x
lengths differ by the dead-band budget.  Every result is compared with the oracle -- scores,
counts and gapped strings bit for bit, p / p-gaps bit for bit, JC / K2P within 1e-12 -- and every
check asserts which kernel ran, so that nothing passes on the general kernel by accident."""
from __future__ import annotations

import numpy as np
import pytest

import oracle
import packed16_rule as R
from synth import coi_like, random_pairs

pytestmark = pytest.mark.gpu

REL_TOL = 1e-12
PACKED = (16, 17, 18)
GENERAL = (32, 33)            # 33 = the intra-task form of the general kernel (few pairs spanning several stripes)
VARIANTS = ((0, 0), (0, 1), (1, 0))   # (force_general, force_top): bottom-aligned where eligible, top-aligned, general

SETS = R.score_sets()
ACCEPTED = [s["scores"] for s in SETS if R.restricted_exact(s["scores"])]
REJECTED = [s["scores"] for s in SETS if not R.restricted_exact(s["scores"])]
MUST_REJECT = [s["scores"] for s in SETS if s["accept"] is False]
# last packed length of a square pair up to 150 bp: a few accepted sets with expensive end gaps
# leave no window at all (the top-aligned kernel always spans at least 256 rows)
WINDOW = {s: R.last_packed(s, "square", limit=150) for s in ACCEPTED}
PACKABLE = [s for s in ACCEPTED if WINDOW[s] >= 20]
NEVER_PACKED = REJECTED + [s for s in ACCEPTED if WINDOW[s] == 0]
assert len(PACKABLE) + len(NEVER_PACKED) == len(SETS)


@pytest.fixture(scope="module")
def engine():
    from taxi2_b200.engine import Engine

    eng = Engine(0)
    yield eng
    eng.close()


def assert_metrics_close(got: np.ndarray, want: np.ndarray):
    assert got.shape == want.shape
    nan_g, nan_w = np.isnan(got), np.isnan(want)
    assert np.array_equal(nan_g, nan_w)
    g, w = got[~nan_g], want[~nan_w]
    assert np.all(np.abs(g - w) <= REL_TOL * np.maximum(np.abs(w), 1e-300) + 0.0) or np.allclose(g, w, rtol=REL_TOL, atol=0.0)
    # p and p-gaps are a single IEEE division of exact integers: bit-exact
    assert np.array_equal(got[:, :2][~nan_g[:, :2]], want[:, :2][~nan_w[:, :2]])


def oracle_batch(xs, ys, px, py, scores):
    from taxi2_b200.engine import pack_strings

    data, off = pack_strings(list(xs) + list(ys))
    return oracle.align_count_pairs(data, off, np.asarray(px, dtype=np.int32), np.asarray(py, dtype=np.int32) + len(xs), scores)


def kernel_ok(got: int, predicted: int) -> bool:
    return got in GENERAL if predicted == 32 else got == predicted


class Options:
    """Engine options for one block, restored afterwards."""

    def __init__(self, engine, **opts):
        self.engine, self.opts = engine, opts

    def __enter__(self):
        for k, v in self.opts.items():
            self.engine.set_option(k, v)

    def __exit__(self, *exc):
        defaults = {"force_general": 0, "force_top": 0, "sort_columns": 1}
        for k in self.opts:
            self.engine.set_option(k, defaults[k])


def check_pairs(engine, xs, ys, scores, strings=True, variants=VARIANTS):
    """Pair list (x_k, y_k) through each kernel variant against the oracle; the kernel that ran must
    be the one the restatement predicts.  Returns the kernels seen."""
    n = len(xs)
    px = np.arange(n, dtype=np.int32)
    want = oracle_batch(xs, ys, px, px, scores)
    want_str = [oracle.align(x, y, scores)[:2] for x, y in zip(xs, ys)] if strings else None
    la, lb = [len(x) for x in xs], [len(y) for y in ys]
    seen = []
    for force_general, force_top in variants:
        predicted = R.predict_pairs(scores, la, lb, force_top=bool(force_top), force_general=bool(force_general))
        with Options(engine, force_general=force_general, force_top=force_top):
            engine.set_scores(scores)
            engine.load(xs, 0)
            engine.load(ys, 1)
            got = engine.align_pairs(px, px)
            kernel = engine.last_kernel
            if strings:
                ax, ay, sc = engine.align_strings(px, px)
                assert engine.last_kernel == kernel
        where = (scores, force_general, force_top, kernel)
        assert np.array_equal(got["score"], want["score"]), where
        assert np.array_equal(got["counts"], want["counts"]), where
        assert_metrics_close(got["metrics"], want["metrics"])
        if strings:
            assert np.array_equal(sc, want["score"]), where
            for k in range(n):
                assert (ax[k].decode("latin-1"), ay[k].decode("latin-1")) == want_str[k], (where, k, xs[k][:40], ys[k][:40])
        assert kernel_ok(kernel, predicted), (where, predicted)
        seen.append(kernel)
    return seen


def check_rect(engine, xs, ys, scores, sort_columns=0):
    """Every (x, y) of a rectangle whose rows share one length geometry, against the oracle."""
    px, py = np.divmod(np.arange(len(xs) * len(ys)), len(ys))
    want = oracle_batch(xs, ys, px, py, scores)
    seen = []
    for force_general, force_top in VARIANTS:
        predicted = 32 if force_general else R.predict_rect(scores, max(map(len, xs)), [len(y) for y in ys], force_top=bool(force_top))
        with Options(engine, force_general=force_general, force_top=force_top, sort_columns=sort_columns):
            engine.set_scores(scores)
            engine.load(xs, 0)
            engine.load(ys, 1)
            got = engine.align_rect(0, len(xs), 0, len(ys))
            kernel = engine.last_kernel
        where = (scores, force_general, force_top, kernel)
        assert np.array_equal(got["score"].ravel(), want["score"]), where
        assert np.array_equal(got["counts"].reshape(-1, 4), want["counts"]), where
        assert_metrics_close(got["metrics"].reshape(-1, 4), want["metrics"])
        assert kernel_ok(kernel, predicted), (where, predicted)
        seen.append(kernel)
    return seen


# -- 1. and 2.: the restricted recurrence on every accepted set, the general kernel for the others --

def _fragment(rng, y: bytes, length: int, sub: float = 0.05, at: int | None = None) -> bytes:
    """A slightly mutated piece of y (a long end gap on one or both sides)."""
    al = np.frombuffer(b"ACGT", dtype=np.uint8)
    o = int(rng.integers(0, len(y) - length + 1)) if at is None else at
    s = np.frombuffer(y[o:o + length], dtype=np.uint8).copy()
    hit = rng.random(length) < sub
    s[hit] = al[rng.integers(0, 4, int(hit.sum()))]
    return s.tobytes()


def tie_rich_inputs(rng, top: int = 150):
    """Two-letter and ACGTN pairs of 1-150 bp (indels make x and y differ in length), unrelated
    pairs of independent lengths, and fragments of either sequence in the other (long end gaps);
    no sequence longer than `top`."""
    xs, ys = random_pairs(rng, 40, 1, top - 10, sub=0.3, indel=0.1, alphabet=b"AT")
    x2, y2 = random_pairs(rng, 30, 1, top - 10, sub=0.25, indel=0.08, alphabet=b"ACGTN")
    xs += x2; ys += y2
    xs, ys = [x[:top] for x in xs], [y[:top] for y in ys]
    al = np.frombuffer(b"ACGT", dtype=np.uint8)
    for _ in range(15):
        xs.append(al[rng.integers(0, 4, int(rng.integers(1, top + 1)))].tobytes())
        ys.append(al[rng.integers(0, 4, int(rng.integers(1, top + 1)))].tobytes())
    for k in range(20):
        long = al[rng.integers(0, 4, int(rng.integers(min(60, top), top + 1)))].tobytes()
        short = _fragment(rng, long, int(rng.integers(1, max(2, len(long) // 2))))
        xs.append(short if k % 2 else long)
        ys.append(long if k % 2 else short)
    return xs, ys


@pytest.mark.parametrize("scores", PACKABLE, ids=str)
def test_restricted_recurrence_is_exact(engine, scores):
    rng = np.random.default_rng(abs(hash(scores)) % 2**32)
    xs, ys = tie_rich_inputs(rng, WINDOW[scores])    # within the set's window: every pair runs packed
    seen = check_pairs(engine, xs, ys, scores)
    assert seen[0] in PACKED and seen[2] in GENERAL


@pytest.mark.parametrize("scores", NEVER_PACKED, ids=str)
def test_rejected_sets_run_on_the_general_kernel(engine, scores):
    """Sets the rule rejects (on the edge of a form, Needleman-Wunsch, random) or whose window holds
    no pair (expensive end gaps), in every variant; the
    inputs include the explicit pair on which a rejected edge set has a co-optimal alignment with a
    vertical gap next to a horizontal one (tests/test_packed_proof_premise.py)."""
    rng = np.random.default_rng(abs(hash(scores)) % 2**32)
    xs, ys = random_pairs(rng, 30, 1, 60, sub=0.3, indel=0.1, alphabet=b"AT")
    found = R.witness(scores) if scores in MUST_REJECT and R.is_gotoh(scores) else None
    if found is not None:
        x, y = found[0].encode(), found[1].encode()
        xs += [x, y, x * 3]; ys += [y, x, y * 3]
    seen = check_pairs(engine, xs, ys, scores)
    assert all(k in GENERAL for k in seen)


# -- 3. window edges --------------------------------------------------------------------------------

def _edge_sets():
    """The sets DESIGN.md §3.2 lists plus accepted sets of the generator whose square edge is at most
    4 000 bp, about twenty in all."""
    named = [(1, -1, -8, -1, -1, -1), (2, -1, -3, -2, -1, -1), (3, -2, -6, -2, -3, -2), (5, -4, -10, -4, -4, -4), (0, -1, -3, -1, -2, -1)]
    picked = [s for s in ACCEPTED if s not in named and R.fast16(s, 64, 64) is not None and R.fast16(s, 4000, 4000) is None]
    return named + picked[:: max(1, len(picked) // 15)][:15]


EDGE_SETS = _edge_sets()
SHAPES = {"square": lambda L, s: (L, L), "x_long": lambda L, s: (L, s), "y_long": lambda L, s: (s, L)}


def _bisect_last_packed(engine, scores, shape):
    """Largest L whose one-pair alignment runs packed, found through last_kernel alone; every probe
    also checks the restatement's prediction."""
    probes = {}

    def packed(L):
        rows, cols = SHAPES[shape](L, 1)
        x, y = b"A" * rows, b"C" * cols
        engine.load([x], 0)
        engine.load([y], 1)
        engine.align_pairs([0], [0], want=("score",))
        kernel = engine.last_kernel
        assert kernel_ok(kernel, R.predict_pairs(scores, [rows], [cols])), (scores, shape, L, kernel)
        probes[L] = kernel
        return kernel in PACKED

    engine.set_scores(scores)
    assert packed(1)
    lo, hi = 1, 64
    while packed(hi):
        lo, hi = hi, 2 * hi
        if hi > 1 << 13:
            return None                  # no edge: the window does not grow with this side (an extend score of 0)
    while hi - lo > 1:
        mid = (lo + hi) // 2
        lo, hi = (mid, hi) if packed(mid) else (lo, mid)
    return lo


def _edge_inputs(rng, rows, cols):
    """Inputs that drive the DP to the bottom of the window, of exactly rows x cols."""
    al = np.frombuffer(b"ACGT", dtype=np.uint8)
    at = np.frombuffer(b"AT", dtype=np.uint8)
    xr = al[rng.integers(0, 4, rows)]
    yr = al[rng.integers(0, 4, cols)]                         # ~25 % identity
    xt = at[rng.integers(0, 2, rows)]
    yt = xt[:cols].copy() if cols <= rows else np.concatenate([xt, at[rng.integers(0, 2, cols - rows)]])
    yt[rng.random(cols) < 0.3] = ord("A")
    xs = [b"A" * rows, b"T" * rows, xr.tobytes(), xt.tobytes()]
    ys = [b"C" * cols, b"A" * cols, yr.tobytes(), yt.tobytes()]
    return xs, ys


@pytest.mark.parametrize("scores", EDGE_SETS, ids=str)
def test_window_edges(engine, scores):
    rng = np.random.default_rng(abs(hash(scores)) % 2**32)
    for shape in SHAPES:
        edge = _bisect_last_packed(engine, scores, shape)
        if edge is None:
            assert R.last_packed(scores, shape, limit=1 << 14) == 1 << 14
            continue
        assert edge == R.last_packed(scores, shape, limit=2 * edge + 2), (scores, shape, edge)
        for L in (edge, edge + 1):
            # pair lists: each small side 1..3 in its own launch (the window depends on it)
            for small in ((1, 2, 3) if shape != "square" else (L,)):
                rows, cols = SHAPES[shape](L, small)
                xs, ys = _edge_inputs(rng, rows, cols)
                strings = rows * cols <= 5_000_000
                check_pairs(engine, xs, ys, scores, strings=strings)
            # a rectangle: one row length, columns of different length next to each other in a warp unit
            if shape == "y_long":
                xs = [b"A", b"GT", b"TTA"]
                ys = _edge_inputs(rng, 1, L)[1] + [b"C" * (L // 2), b"G" * 7]
            else:
                xs, ys = _edge_inputs(rng, L, 3 if shape == "x_long" else L)
                ys += [b"C" * max(1, len(ys[0]) // 3), b"T"]
            check_rect(engine, xs, ys, scores)


def test_geometry_transitions(engine):
    """Bottom-aligned: one stripe up to 1 023 rows, several from 1 024 (the border row needs a slot
    of its own).  Top-aligned: one stripe of at most 32 x 32 = 1 024 rows, then the general kernel."""
    rng = np.random.default_rng(1024)
    default, top = (1, -1, -8, -1, -1, -1), (2, -1, -3, -2, -1, -1)
    for L, bottom_kernel, top_kernel in ((1022, 17, 16), (1023, 17, 16), (1024, 18, 16), (1025, 18, 32)):
        xs, ys = _edge_inputs(rng, L, L)
        general = lambda ks: [32 if k in GENERAL else k for k in ks]   # noqa: E731
        assert general(check_pairs(engine, xs, ys, default, strings=False)) == [bottom_kernel, top_kernel, 32]
        assert general(check_pairs(engine, xs, ys, top, strings=L >= 1024, variants=((0, 0),))) == [top_kernel]
        assert general(check_rect(engine, xs, ys + [b"A" * (L // 2)], default)) == [bottom_kernel, top_kernel, 32]


# -- 4. dead band -----------------------------------------------------------------------------------

def _dead_band_pairs(rng, scores, length, d, at_end):
    """Two pairs: a long x (a mutated copy of its y) and a shorter x, d rows shorter, cut from a
    long y of its own -- at the end of y (the longest leading end gap) or at random."""
    al = np.frombuffer(b"ACGT", dtype=np.uint8)
    y1 = al[rng.integers(0, 4, length)].tobytes()
    y2 = al[rng.integers(0, 4, length)].tobytes()
    x1 = _fragment(rng, y1, length, sub=0.03, at=0)
    x2 = _fragment(rng, y2, length - d, sub=0.03, at=(d if at_end else None))
    return [x1, x2], [y1, y2]


@pytest.mark.parametrize("scores,length", [((3, -2, -6, -2, -3, -2), 650), ((1, -1, -8, -1, -1, -1), 1800),
                                           ((1, -1, -8, -1, -1, -1), 1900), ((1, -1, -8, -1, -1, -1), 1950),
                                           ((1, -1, -8, -1, -1, -1), 1981)])
def test_dead_band_budget(engine, scores, length):
    """Two pairs of a list share a warp unit only if their x lengths differ by at most the budget the
    window leaves (127 rows for the first set at 650 bp; the default set in several stripes: 181,
    81, 31 and 0 rows at 1 800 - 1 981 bp).  Differences of budget - 1, budget and budget + 1 (the
    last runs each pair alone), the shorter x a fragment of a long y, in both orders."""
    budget = R.dead_budget(scores, length, length)
    assert budget == {650: 127, 1800: 181, 1900: 81, 1950: 31, 1981: 0}[length]
    rng = np.random.default_rng(length)
    for d in sorted({max(0, budget - 1), budget, budget + 1}):
        la = [length, length - d]
        _, used = R.build_units(la, [length, length], budget)
        assert used == (d if d <= budget else 0)
        for at_end in (True, False):
            xs, ys = _dead_band_pairs(rng, scores, length, d, at_end)
            for order in (slice(None), slice(None, None, -1)):
                seen = check_pairs(engine, xs[order], ys[order], scores, strings=at_end)
                assert seen[0] == (17 if length < 1023 else 18)


# -- 5. both orientations from one alignment ---------------------------------------------------------

# bottom-aligned sets (internal extend == end extend) whose window holds the tie-rich input
BOTTOM_SETS = [s for s in ACCEPTED if s[3] == s[5] and (R.fast16(s, 160, 160) or {}).get("mode") == 1]


@pytest.mark.parametrize("scores", BOTTOM_SETS[:: max(1, len(BOTTOM_SETS) // 8)][:8], ids=str)
def test_both_orientations_against_the_oracle(engine, scores):
    """taxi_align_rect_both derives (y, x) from the alignment of (x, y) unless the traced path chose
    Ix over Iy at equal score; that M-versus-gap ties and choices inside Ix / Iy are orientation
    neutral rests on the restricted recurrence being exact.  Both orientations against the oracle
    directly, on tie-rich two-letter input and on barcodes."""
    rng = np.random.default_rng(abs(hash(scores)) % 2**32)
    cases = [random_pairs(rng, 36, 100, 160, sub=0.3, indel=0.1, alphabet=b"AT")[0]]
    if (f := R.fast16(scores, 650, 650)) is not None and f["mode"] == 1:
        cases.append(coi_like(24, length=650, seed=int(rng.integers(1 << 30))))
    for xs in cases:
        n = len(xs)
        engine.set_scores(scores)
        engine.load(xs, 0)
        xy, yx = engine.align_rect_both(0, n, 0, n)
        assert engine.last_kernel == 20
        redo = engine.last_redo
        px, py = np.divmod(np.arange(n * n), n)
        want = oracle_batch(xs, xs, px, py, scores)
        for got in (xy, yx):            # (y, x) of a square set is (x, y) with the indices exchanged: the oracle's (py, px)
            assert np.array_equal(got["score"].ravel(), want["score"]), scores
            assert np.array_equal(got["counts"].reshape(-1, 4), want["counts"]), scores
            assert_metrics_close(got["metrics"].reshape(-1, 4), want["metrics"])
        counts = want["counts"].reshape(n, n, 4)
        asymmetric = int((counts != np.swapaxes(counts, 0, 1)).any(axis=2).sum())
        assert redo >= asymmetric, (scores, redo, asymmetric)


# -- 6. the general kernel's exact int32 range -------------------------------------------------------

@pytest.mark.parametrize("scores", [(1 << 20, -(1 << 20), -(1 << 20), -(1 << 19), -(1 << 20), -(1 << 18)),
                                    (1000, -4096, -4000, -1000, -3000, -1000),
                                    (3000, -3000, -3000, -3000, -3000, -3000)], ids=str)
def test_general_kernel_int32_edge(engine, scores):
    """(rows + cols + 2) * max|score| < 2^24 keeps every DP value exact after the x64 scaling: at
    the largest admitted lengths the results are the oracle's, one row more is refused."""
    from taxi2_b200._native import E_RANGE, TaxiNativeError

    m = max(abs(s) for s in scores)
    total = ((1 << 24) - 1) // m - 2            # largest rows + cols
    assert (total + 2) * m < 1 << 24 <= (total + 3) * m
    rows = (total + 1) // 2
    cols = total - rows
    rng = np.random.default_rng(m)
    xs, ys = _edge_inputs(rng, rows, cols)
    seen = check_pairs(engine, xs, ys, scores, strings=rows * cols <= 5_000_000, variants=((0, 0), (1, 0)))
    seen += check_rect(engine, xs, ys, scores)
    # the same sum of lengths, all in one sequence (the range check bounds the longest of each side)
    seen += check_pairs(engine, [b"A" * (total - 1), b"AC" * ((total - 1) // 2)], [b"T", b"G"], scores, variants=((0, 0),))
    seen += check_pairs(engine, [b"G", b"T"], [b"C" * (total - 1), b"AC" * ((total - 1) // 2)], scores, variants=((0, 0),))
    assert all(k in GENERAL for k in seen)
    engine.set_scores(scores)
    for x, y in ((b"A" * (rows + 1), b"C" * cols), (b"A" * total, b"C" * 2)):
        engine.load([x], 0)
        engine.load([y], 1)
        with pytest.raises(TaxiNativeError) as err:
            engine.align_pairs([0], [0])
        assert err.value.code == E_RANGE
        with pytest.raises(TaxiNativeError) as err:
            engine.align_rect(0, 1, 0, 1)
        assert err.value.code == E_RANGE
