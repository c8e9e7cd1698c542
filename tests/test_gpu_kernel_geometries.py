"""Every compiled alignment kernel instance against the oracle, at the row counts that select it.

The library compiles one instance of its alignment kernels per geometry (H rows per lane) and picks
one per launch from the score set and the longest row; `kernel_geometry.py` restates that choice.
The case table below is generated from it: for every instance the lowest and the highest row count
that select it (row counts up to GENERAL_LIMIT / PACKED_LIMIT), with y lengths of 1 bp and of the
full window.  Each launch is compared with the oracle -- scores and counts bit for bit, p / p-gaps
bit for bit, JC / K2P within 1e-12, gapped strings for a bounded subset -- and `last_kernel` with
the instance the restatement predicts, so that no case passes on another instance by accident.
The metrics every instance writes are also bit for bit `taxi_metrics_from_counts` of its own counts
(floating-point form, NaN pattern included): each instance inlines its own copy of the epilogue, and
the entry point is the copy test_gpu_metric_arithmetic.py pins against exact references.

The both-orientations kernel (`gotoh_pair16_kernel<H,1,true>`) keeps its tie bits in a word whose
layout depends on H; a missed bit writes a wrong (y, x) result.  Each of its six geometries gets a
square set of tie-rich and of barcode-like families, checked in both orientations against the
oracle, and the re-alignment of the orientation-sensitive pairs is also run on the multi-stripe
packed kernel (a y set longer than one stripe)."""
from __future__ import annotations

import numpy as np
import pytest

import kernel_geometry as K
import oracle
import packed16_rule as R
from poison import poison
from synth import ALPHA, coi_like, random_pairs
from test_gpu_packed_exactness import assert_metrics_close, oracle_batch

pytestmark = pytest.mark.gpu

DEFAULT = (1, -1, -8, -1, -1, -1)
TOP = (2, -1, -3, -2, -1, -1)          # ie != ee: the packed kernel runs top-aligned
NW = (1, -1, -2, -2, -2, -2)           # every open == extend: Needleman-Wunsch order, general kernel only
WIDE = (0, -1, -3, -1, -2, -1)         # 16-bit window up to 3 999 bp: reaches multi-stripe packed H = 16 and 32
GENERAL_LIMIT = 3072                   # highest row count scanned for the general kernel
PACKED_LIMIT = 4000
STRING_CELLS = 2_000_000               # gapped strings from the oracle for pairs up to this many cells
COOP_STRIPES = (2, 11, 12, 13, 25)     # below, at and above the 12 warps of the intra-task kernel, and > 2 x 12


def _case(family, H, scores, rows, note=""):
    return dict(id=f"{K.name(family, H)}-{','.join(map(str, scores))}-{rows}{note}", family=family, H=H,
                scores=scores, rows=rows)


def plan() -> dict:
    """-> {"pairs": [...], "coop": [...], "both": [...]}: one entry per launch the module checks."""
    pairs, coop, both = [], [], []
    for H in K.KH:
        for kind in ("one", "several"):
            runs = K.selecting_rows("general", H, DEFAULT, GENERAL_LIMIT, stripes=kind)
            if not runs:
                continue
            lo, hi = runs[0][0], runs[-1][1]
            pairs += [_case("general", H, DEFAULT, lo), _case("general", H, DEFAULT, hi),
                      _case("general", H, NW, lo), _case("general", H, TOP, hi)]
    for family, sets in (("top", (DEFAULT, TOP)), ("bottom", (DEFAULT,)), ("multi", (DEFAULT, WIDE))):
        for H in {"multi": R.H_MULTI}.get(family, R.H_ONE):
            for scores in sets:
                runs = K.selecting_rows(family, H, scores, PACKED_LIMIT)
                if runs:
                    pairs += [_case(family, H, scores, runs[0][0]), _case(family, H, scores, runs[-1][1])]
    for H in K.COOP_H:
        for stripes in COOP_STRIPES:
            rows = K.coop_rows(H, stripes)
            if rows is not None:
                for scores in (DEFAULT, NW):
                    coop.append(dict(_case("coop", H, scores, rows, f"-s{stripes}"), stripes=stripes))
    for H in R.H_ONE:
        (lo, hi), = K.selecting_rows("both", H, DEFAULT, 1023)
        both.append(dict(id=K.name("both", H), family="both", H=H, scores=DEFAULT, lo=max(lo, hi // 2 + 1), hi=hi))
    return dict(pairs=pairs, coop=coop, both=both)


PLAN = plan()
CASES = PLAN["pairs"] + PLAN["coop"] + PLAN["both"]
# the two-set rectangle whose re-alignment runs on multi-stripe packed, and the symmetric matrix
RECT_X, RECT_Y = (768, 1023), (1100, 1900)
SYMMETRIC = (800, 1000)


def planned_instances() -> set:
    """(family, H) of every planned launch, including the re-alignment of the two-set rectangle."""
    got = {(c["family"], c["H"]) for c in CASES}
    got.add(K.redo_instance(DEFAULT, [RECT_Y[1]], [RECT_X[1]])[:2])
    return got


def _seed(case) -> int:
    return sum(ord(ch) * (k + 1) for k, ch in enumerate(case["id"])) % 2**32


def _rand(rng, n: int, alphabet: bytes = b"ACGT") -> bytes:
    al = np.frombuffer(alphabet, dtype=np.uint8)
    return al[rng.integers(0, len(al), max(1, n))].tobytes()


def _fit(s: bytes, lo: int, hi: int, rng) -> bytes:
    """Cut or pad s (with random bases) to a length in [lo, hi]."""
    if len(s) > hi:
        return s[:hi]
    if len(s) < lo:
        return s + _rand(rng, lo - len(s))
    return s


def pair_inputs(case) -> tuple[list[bytes], list[bytes], dict]:
    """Pair list whose longest x has case["rows"] rows and longest y as many columns: related pairs
    (~10 % substitutions, indels), tie-rich two-letter pairs, 1 bp against the full length either
    way, an all-mismatch pair, a shorter pair, and an odd number of full-length x so that the last
    one shares a warp unit with an x of another length.  -> (xs, ys, engine options)."""
    rng = np.random.default_rng(_seed(case))
    Rw, C, scores = case["rows"], case["rows"], case["scores"]
    xs, ys = random_pairs(rng, 3, Rw, Rw, sub=0.1, indel=0.02, alphabet=b"ACGT")
    x2, y2 = random_pairs(rng, 2, Rw, Rw, sub=0.3, indel=0.1, alphabet=b"AT")
    xs += x2
    ys += y2
    xs += [_rand(rng, Rw), b"A" * Rw, _rand(rng, 1), _rand(rng, max(1, Rw // 3))]
    ys += [_rand(rng, 1), b"C" * C, _rand(rng, C), _rand(rng, max(1, C // 2))]
    opts = K.family_options(case["family"], scores)
    f = R.fast16(scores, Rw, C, 0, bool(opts.get("force_top")))
    d = max(1, Rw // 4) if f is None or f["mode"] == 0 else max(1, min(f["max_dead"], Rw // 4))
    if Rw - d >= 1:
        x, y = random_pairs(rng, 1, Rw - d, Rw - d, sub=0.1, indel=0.02, alphabet=b"ACGT")
        xs += x
        ys += y
    ys = [y[:C] for y in ys]
    return xs, ys, opts


def coop_inputs(case) -> tuple[list[bytes], list[bytes]]:
    """A few long x (one intra-task launch) against short y: mutated fragments of x (long end gaps on
    both sides), a tie-rich two-letter pair, 1 bp, an all-mismatch pair, and a shorter x."""
    rng = np.random.default_rng(_seed(case))
    Rw = case["rows"]
    xs, ys = [], []
    for k in range(3):
        x = _rand(rng, Rw)
        at = int(rng.integers(0, Rw - 300))
        y = bytearray(x[at:at + 300])
        for i in np.flatnonzero(rng.random(len(y)) < 0.1):
            y[i] = int(ALPHA[rng.integers(0, 4)])
        xs.append(x)
        ys.append(bytes(y))
    xs += [_rand(rng, Rw, b"AT"), _rand(rng, Rw), b"A" * Rw, _rand(rng, Rw - 700)]
    ys += [_rand(rng, 250, b"AT"), b"G", b"C" * 200, _rand(rng, 120)]
    return xs, ys


def both_inputs(case, kind: str, n: int) -> list[bytes]:
    """A square set of n sequences with lengths in [lo, hi] (within a factor of 2): "ties" = four
    families of two-letter sequences (tie_set), "coi" = barcode-like families."""
    rng = np.random.default_rng(_seed(case) + (kind == "coi"))
    lo, hi = case["lo"], case["hi"]
    if kind == "coi":
        seqs = coi_like(n, length=(lo + hi) // 2, seed=int(rng.integers(1 << 30)), genera=4, species=3)
        return [_fit(s, lo, hi, rng) for s in seqs]
    return [s for _ in range(4) for s in tie_set(rng, n // 4, lo, hi)]


def tie_set(rng, n: int, lo: int, hi: int) -> list[bytes]:
    """A family of n two-letter sequences: prefixes of lengths in [lo, hi] of one root, 25 % of their
    positions redrawn, indels of 1 - 3 bases at 4 % of the positions, cut or padded back into [lo, hi]."""
    root = _rand(rng, hi, b"AT")
    out = []
    for _ in range(n):
        s = bytearray(root[: int(rng.integers(lo, hi + 1))])
        for i in np.flatnonzero(rng.random(len(s)) < 0.25):
            s[i] = ord("A") if rng.random() < 0.5 else ord("T")
        for _ in range(rng.binomial(len(s), 0.04)):
            at, run = int(rng.integers(0, len(s))), int(rng.integers(1, 4))
            if rng.random() < 0.5:
                del s[at:at + run]
            else:
                s[at:at] = _rand(rng, run, b"AT")
        out.append(_fit(bytes(s), lo, hi, rng))
    return out


# -- GPU ------------------------------------------------------------------------------------------------

@pytest.fixture(scope="module")
def engine():
    from taxi2_b200.engine import Engine

    eng = Engine(0)
    yield eng
    eng.close()


class Options:
    """Engine options for one block, restored to their defaults afterwards."""

    DEFAULTS = {"force_general": 0, "force_top": 0, "no_coop": 0, "sort_columns": 1}

    def __init__(self, engine, **opts):
        self.engine, self.opts = engine, opts

    def __enter__(self):
        for k, v in self.opts.items():
            self.engine.set_option(k, v)

    def __exit__(self, *exc):
        for k in self.opts:
            self.engine.set_option(k, self.DEFAULTS[k])


def assert_same(got: dict, want: dict, where):
    assert np.array_equal(got["score"].ravel(), want["score"].ravel()), where
    assert np.array_equal(got["counts"].reshape(-1, 4), want["counts"].reshape(-1, 4)), where
    assert_metrics_close(got["metrics"].reshape(-1, 4), want["metrics"].reshape(-1, 4))


def assert_epilogue(engine, got: dict, where):
    """The metrics a kernel wrote are bit for bit the floating-point form of taxi_metrics_from_counts
    of the counts it wrote: one contraction or rounding step that differs between the two copies of
    the epilogue moves a value by an ulp, and pairs_within / best-k decide on exact values."""
    counts = got["counts"].reshape(-1, 4)
    want = engine.metrics_from_counts(counts, table=False)
    bits = got["metrics"].reshape(-1, 4).view(np.uint64)
    bad = np.flatnonzero((bits != want.view(np.uint64)).any(axis=1))
    assert len(bad) == 0, (where, counts[bad][:4].tolist(), got["metrics"].reshape(-1, 4)[bad][:4].tolist(), want[bad][:4].tolist())


def run_pairs(engine, xs, ys, scores, opts, family, H, strings=True):
    """Pair list against the oracle; the predicted instance must be (family, H) and must have run."""
    la, lb = [len(x) for x in xs], [len(y) for y in ys]
    predicted = K.instance(scores, la, lb, "pairs", opts)
    assert predicted[:2] == (family, H), predicted
    n = len(xs)
    px = np.arange(n, dtype=np.int32)
    want = oracle_batch(xs, ys, px, px, scores)
    with Options(engine, **opts):
        engine.set_scores(scores)
        poison(engine, n, max(la + lb) + 1)
        engine.load(xs, 0)
        engine.load(ys, 1)
        got = engine.align_pairs(px, px)
        kernel = engine.last_kernel
        where = (K.name(family, H), scores, predicted, kernel)
        assert kernel == K.CODE[family], where
        assert_same(got, want, where)
        assert_epilogue(engine, got, where)
        if strings:
            sub = [k for k in range(n) if la[k] * lb[k] <= STRING_CELLS]
            sub_pred = K.instance(scores, [la[k] for k in sub], [lb[k] for k in sub], "pairs", opts)
            ox, oy, start, off, sc, res = engine.align_strings_raw(px[sub], px[sub], want=("counts", "metrics"))
            assert engine.last_kernel == K.CODE[sub_pred[0]], (where, sub_pred)
            assert np.array_equal(sc, want["score"][sub]), where
            assert np.array_equal(res["counts"], want["counts"][sub]), where
            assert_epilogue(engine, res, (where, "strings"))
            bx, by = ox.tobytes(), oy.tobytes()
            for i, k in enumerate(sub):
                ax, ay = bx[int(start[i]):int(off[i + 1])], by[int(start[i]):int(off[i + 1])]
                assert (ax.decode("latin-1"), ay.decode("latin-1")) == oracle.align(xs[k], ys[k], scores)[:2], (where, k)
    return got, predicted


@pytest.mark.parametrize("case", PLAN["pairs"], ids=lambda c: c["id"])
def test_instance_against_the_oracle(engine, case):
    xs, ys, opts = pair_inputs(case)
    run_pairs(engine, xs, ys, case["scores"], opts, case["family"], case["H"])


@pytest.mark.parametrize("case", PLAN["coop"], ids=lambda c: c["id"])
def test_intra_task_stripe_counts(engine, case):
    """The intra-task kernel hands stripe s of a pair to warp s mod 12: 2 stripes, 11 / 12 / 13 around
    the warp count, and 25 or more (three rounds).  Against the oracle and against the same pairs
    one per warp (no_coop)."""
    xs, ys = coop_inputs(case)
    got, predicted = run_pairs(engine, xs, ys, case["scores"], {"force_general": 1}, "coop", case["H"], strings=False)
    assert predicted[2] == case["stripes"]
    la, lb = [len(x) for x in xs], [len(y) for y in ys]
    assert K.instance(case["scores"], la, lb, "pairs", {"force_general": 1, "no_coop": 1})[0] == "general"
    px = np.arange(len(xs), dtype=np.int32)
    with Options(engine, force_general=1, no_coop=1):
        poison(engine, len(xs), max(la + lb) + 1)
        engine.load(xs, 0)
        engine.load(ys, 1)
        ref = engine.align_pairs(px, px)
        assert engine.last_kernel == 32
    assert np.array_equal(got["score"], ref["score"]) and np.array_equal(got["counts"], ref["counts"])
    assert np.array_equal(got["metrics"], ref["metrics"], equal_nan=True)
    # gapped strings of the first pair, which alone still takes the same intra-task instance
    with Options(engine, force_general=1):
        ax, ay, _ = engine.align_strings(px[:1], px[:1])
        assert engine.last_kernel == 33
    assert (ax[0].decode(), ay[0].decode()) == oracle.align(xs[0], ys[0], case["scores"])[:2]


def check_both(engine, xs, ys, H, tie_rich):
    """align_rect_both of (xs, ys) against the oracle in both orientations -> pairs re-aligned."""
    la, lb = [len(x) for x in xs], [len(y) for y in ys]
    assert K.instance(DEFAULT, la, lb, "both") == ("both", H, 1)
    engine.set_scores(DEFAULT)
    poison(engine, 2 * len(xs) * len(ys), max(la + lb) + 1)     # both halves: (x, y) and the mirrored (y, x)
    engine.load(xs, 0)
    if ys is not xs:
        engine.load(ys, 1)
    xy, yx = engine.align_rect_both(0, len(xs), 0, len(ys))
    assert engine.last_kernel == 20
    redo = engine.last_redo
    nx, ny = len(xs), len(ys)
    px, py = np.divmod(np.arange(nx * ny), ny)
    want_xy = oracle_batch(xs, ys, px, py, DEFAULT)
    qy, qx = np.divmod(np.arange(nx * ny), nx)
    want_yx = want_xy if ys is xs else oracle_batch(ys, xs, qy, qx, DEFAULT)
    assert_same(xy, want_xy, (H, "xy"))
    assert_same(yx, want_yx, (H, "yx"))
    assert_epilogue(engine, xy, (H, "xy"))
    assert_epilogue(engine, yx, (H, "yx"))      # mirrored from the (x, y) pass or re-aligned
    c_xy = want_xy["counts"].reshape(nx, ny, 4)
    c_yx = want_yx["counts"].reshape(ny, nx, 4)
    asymmetric = int((c_xy != np.swapaxes(c_yx, 0, 1)).any(axis=2).sum())
    assert redo >= asymmetric, (H, redo, asymmetric)
    if tie_rich:
        assert asymmetric > 0, H
    return redo


@pytest.mark.parametrize("case", PLAN["both"], ids=lambda c: c["id"])
def test_both_orientations_every_geometry(engine, case):
    n = 32 if case["H"] <= 16 else 24
    for kind in ("ties", "coi"):
        xs = both_inputs(case, kind, n)
        assert case["lo"] <= min(map(len, xs)) and max(map(len, xs)) <= case["hi"]
        check_both(engine, xs, xs, case["H"], tie_rich=kind == "ties")


def rect_inputs():
    rng = np.random.default_rng(1100)
    return tie_set(rng, 12, *RECT_X), tie_set(rng, 12, *RECT_Y)


def test_both_orientations_redo_on_multi_stripe(engine):
    """x rows of one stripe, y columns of 1 100 - 1 900 bp: the re-alignment of the
    orientation-sensitive pairs (rows = their y) runs on the multi-stripe packed kernel."""
    xs, ys = rect_inputs()
    for rows in (min(map(len, ys)), max(map(len, ys))):
        assert K.redo_instance(DEFAULT, [rows], [max(map(len, xs))])[0] == "multi"
    assert check_both(engine, xs, ys, 32, tie_rich=True) > 0


def test_symmetric_matrix_at_h32(engine):
    """MultiEngine.align_matrix_symmetric on one device, 800 - 1 000 bp (H = 32), tiles small enough
    that most of the matrix comes from align_rect_both: bit for bit the matrix of align_rect."""
    from taxi2_b200.multi import MultiEngine

    rng = np.random.default_rng(800)
    seqs = tie_set(rng, 16, *SYMMETRIC) + [_fit(s, *SYMMETRIC, rng) for s in coi_like(16, length=900, seed=9)]
    n = len(seqs)
    assert K.instance(DEFAULT, [SYMMETRIC[1]], [SYMMETRIC[1]], "both")[:2] == ("both", 32)
    engine.set_scores(DEFAULT)
    engine.load(seqs, 0)
    want = engine.align_rect(0, n, 0, n)
    with MultiEngine([0]) as multi:
        multi.load(seqs, 0)
        got = multi.align_matrix_symmetric(block=8)
    assert got["redo"] > 0
    for key in ("score", "counts", "metrics"):
        assert np.array_equal(got[key], want[key], equal_nan=True), key
