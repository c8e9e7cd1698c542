"""GPU parity tests: the CUDA path through the C ABI vs the CPU oracle, bit-exact for scores,
counts and alignment strings; 1e-12 relative for the fp64 metrics (north star tolerance)."""
from __future__ import annotations

import json

import numpy as np
import pytest

import oracle
from conftest import GOLDEN
from synth import coi_like, random_pairs, read_tab_sequences

pytestmark = pytest.mark.gpu

REL_TOL = 1e-12  # JC / K2P: fp64 log/sqrt on device vs glibc

ALIGN = json.loads((GOLDEN / "align_cases.json").read_text())


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
    return oracle.align_count_pairs(data, off, np.asarray(px), np.asarray(py) + len(xs), scores)


def check_pairs(engine, xs, ys, scores, strings=True, expect_fast=None):
    """Both kernels (packed 16-bit fast path where eligible, general int32) against the oracle."""
    n = len(xs)
    px = np.arange(n, dtype=np.int32)
    want = oracle_batch(xs, ys, px, px, scores)
    kernels = set()
    for force_general, force_top in ((0, 0), (0, 1), (1, 0)):
        engine.set_option("force_general", force_general)
        engine.set_option("force_top", force_top)
        try:
            engine.set_scores(scores)
            engine.load(xs, 0)
            engine.load(ys, 1)
            got = engine.align_pairs(px, px)
            kernels.add(engine.last_kernel)
            if force_general:
                assert engine.last_kernel in (32, 33)      # 33 = the intra-task variant (few pairs spanning several stripes)
            assert np.array_equal(got["score"], want["score"])
            assert np.array_equal(got["counts"], want["counts"])
            assert_metrics_close(got["metrics"], want["metrics"])
            if strings:
                ax, ay, sc = engine.align_strings(px, px)
                assert np.array_equal(sc, want["score"])
                for k in range(n):
                    ox, oy, _ = oracle.align(xs[k], ys[k], scores)
                    assert ax[k].decode("latin-1") == ox and ay[k].decode("latin-1") == oy, (force_general, k, xs[k], ys[k])
        finally:
            engine.set_option("force_general", 0)
            engine.set_option("force_top", 0)
    if expect_fast is True:
        assert kernels & {16, 17, 18}, "packed fast path was expected to be eligible"
    if expect_fast is False:
        assert kernels <= {32, 33}


@pytest.mark.parametrize("case", ALIGN["align_tests"] + ALIGN["align_tests_failing"],
                         ids=lambda c: f"{c['x']}-{c['y']}-{c['scores']}")
def test_reference_known_answers(engine, case):
    """tests/test_align.py of the reference, through the CUDA path."""
    engine.set_scores(case["scores"])
    engine.load([case["x"]], 0)
    engine.load([case["y"]], 1)
    ax, ay, sc = engine.align_strings([0], [0])
    got = [ax[0].decode(), ay[0].decode()]
    assert got in case["solutions"]
    ox, oy, oscore = oracle.align(case["x"], case["y"], case["scores"])
    assert got == [ox, oy] and sc[0] == oscore
    if "biopython" in case:
        assert got == case["biopython"]["aligned"] and sc[0] == case["biopython"]["score"]


@pytest.mark.parametrize("scores", [(1, -1, -8, -1, -1, -1), (1, 0, 0, 0, 0, 0), (2, -3, -5, -2, -4, -1),
                                    (1, -1, -1, -1, -2, -2), (10, 0, -10, -6, 0, 0), (1, -1, -8, -1, -3, -2),
                                    (1, 0, 0, -2, -1, 0), (0, 1, -1, 0, 0, 0)])
def test_random_short_pairs(engine, scores):
    rng = np.random.default_rng(hash(scores) % (2**32))
    xs, ys = random_pairs(rng, 300, 1, 70, sub=0.25, indel=0.08)
    check_pairs(engine, xs, ys, scores)


def test_low_complexity_ties(engine):
    """Two-letter alphabets maximise co-optimal paths: stresses the tie-breaking order."""
    rng = np.random.default_rng(7)
    xs, ys = random_pairs(rng, 400, 1, 90, sub=0.3, indel=0.1, alphabet=b"AT")
    for scores in [(1, -1, -8, -1, -1, -1), (1, -1, -2, -1, -1, -1), (1, 0, 0, 0, 0, 0), (1, -1, -1, -1, -1, -1)]:
        check_pairs(engine, xs, ys, scores)


def test_barcode_length_pairs(engine):
    rng = np.random.default_rng(650)
    xs, ys = random_pairs(rng, 64, 560, 700, sub=0.12, indel=0.02)
    check_pairs(engine, xs, ys, (1, -1, -8, -1, -1, -1), expect_fast=True)
    # odd pair count (last warp unit is half empty) and a score set that stays on the general kernel
    check_pairs(engine, xs[:33], ys[:33], (1, -1, -8, -1, -1, -1), expect_fast=True)
    check_pairs(engine, xs[:8], ys[:8], (1, 0, 0, 0, 0, 0), expect_fast=False)


def test_fast_path_score_sets(engine):
    """Score sets that satisfy the fast-path proof obligations, on tie-rich low-complexity input."""
    rng = np.random.default_rng(16)
    xs, ys = random_pairs(rng, 300, 1, 120, sub=0.2, indel=0.06, alphabet=b"ACGTN")
    xs2, ys2 = random_pairs(rng, 300, 1, 120, sub=0.3, indel=0.1, alphabet=b"AT")
    for scores in [(1, -1, -8, -1, -1, -1), (2, -1, -3, -2, -1, -1), (4, -3, -9, -3, -3, -3), (1, -1, -2, -1, -2, -1), (3, -2, -6, -2, -3, -2), (2, -2, -7, -3, -4, -2)]:
        check_pairs(engine, xs, ys, scores, expect_fast=True)
        check_pairs(engine, xs2, ys2, scores, expect_fast=True)
    # match - mismatch > 7 (beyond the one-byte penalty table of round 1): the penalty is applied by an IMAD now
    check_pairs(engine, xs[:60], ys[:60], (5, -4, -10, -4, -4, -4), expect_fast=True)
    short = [k for k in range(len(xs2)) if len(xs2[k]) <= 40 and len(ys2[k]) <= 40]
    check_pairs(engine, [xs2[k] for k in short], [ys2[k] for k in short], (20, -30, -70, -25, -40, -25), expect_fast=True)


def test_mixed_lengths_in_one_warp(engine):
    """Neighbouring pairs of very different lengths share a warp in the packed kernel."""
    rng = np.random.default_rng(99)
    xs, ys = [], []
    for k in range(120):
        lo, hi = (5, 40) if k % 3 == 0 else ((300, 420) if k % 3 == 1 else (600, 700))
        x, y = random_pairs(rng, 1, lo, hi, sub=0.15, indel=0.03)
        xs += x; ys += y
    check_pairs(engine, xs, ys, (1, -1, -8, -1, -1, -1), expect_fast=True)


def _fragments(rng, n, ylen, xlens, sub=0.04):
    """x = a slightly mutated fragment of y cut at a random offset (so y overhangs x on both sides:
    the leading end gap is long), with the given x lengths in turn."""
    al = np.frombuffer(b"ACGT", dtype=np.uint8)
    xs, ys = [], []
    for k in range(n):
        y = al[rng.integers(0, 4, ylen)]
        la = xlens[k % len(xlens)]
        o = int(rng.integers(0, ylen - la + 1)) if la < ylen else 0
        x = y[o:o + la].copy()
        hit = rng.random(len(x)) < sub
        x[hit] = al[rng.integers(0, 4, int(hit.sum()))]
        xs.append(x.tobytes()); ys.append(y.tobytes())
    return xs, ys


def test_fragment_next_to_a_longer_neighbour(engine):
    """The two pairs of a warp unit of the packed kernel with DIFFERENT x lengths, the shorter x a
    fragment of a longer y (a long leading end gap): the shorter pair's surplus row slots are dead
    and must stay inside the dead band however many there are (round-1 advisor finding: they
    decayed below zero, wrapped, and fed the pair's row 0 a nearly free entry point).  Two-pair
    launches force the two lengths into one unit, in both halves."""
    rng = np.random.default_rng(450)
    scores = (1, -1, -8, -1, -1, -1)
    for short, longer in [(450, 490), (450, 520), (450, 560), (450, 600), (300, 650), (200, 640), (90, 650), (5, 600)]:
        xs, ys = _fragments(rng, 2, 650, [short, longer])
        check_pairs(engine, xs, ys, scores, expect_fast=True)
        check_pairs(engine, xs[::-1], ys[::-1], scores, expect_fast=True)
    # a whole list of fragments of every length: units are formed by length, longest first
    xs, ys = _fragments(rng, 90, 650, list(range(40, 651, 7)))
    check_pairs(engine, xs, ys, scores, expect_fast=True)
    xs, ys = _fragments(rng, 31, 1500, [300, 1500, 700, 1100, 1024, 1023, 520])   # several stripes
    check_pairs(engine, xs, ys, scores, strings=False, expect_fast=True)
    # other eligible score sets, short rows-per-lane variants
    for sc in [(2, -1, -3, -2, -1, -1), (1, -1, -2, -1, -2, -1), (3, -2, -6, -2, -3, -2)]:
        xs, ys = _fragments(rng, 40, 250, [30, 250, 90, 200, 140, 60], sub=0.1)
        check_pairs(engine, xs, ys, sc, expect_fast=True)


@pytest.mark.parametrize("ny", [1, 3, 5, 8])
def test_rectangle_rows_of_different_length_odd_width(engine, ny):
    """Rectangles whose width is odd: a warp unit never straddles two rows (rows of different
    length would share it), the last unit of a row holds a single pair."""
    rng = np.random.default_rng(31 + ny)
    xs, ys = _fragments(rng, 14, 650, [450, 560, 300, 650, 520, 90, 600])
    ys = ys[:ny]
    px, py = np.divmod(np.arange(len(xs) * ny), ny)
    want = oracle_batch(xs, ys, px, py, None)
    engine.set_scores(None)
    for force_general, force_top, sort_columns in ((0, 0, 1), (0, 0, 0), (0, 1, 1), (1, 0, 1)):
        engine.set_option("force_general", force_general)
        engine.set_option("force_top", force_top)
        engine.set_option("sort_columns", sort_columns)
        try:
            engine.load(xs, 0)
            engine.load(ys, 1)
            got = engine.align_rect(0, len(xs), 0, ny)
        finally:
            engine.set_option("force_general", 0)
            engine.set_option("force_top", 0)
            engine.set_option("sort_columns", 1)
        assert np.array_equal(got["score"].ravel(), want["score"]), (force_general, force_top, sort_columns)
        assert np.array_equal(got["counts"].reshape(-1, 4), want["counts"])
        assert_metrics_close(got["metrics"].reshape(-1, 4), want["metrics"])


def test_strings_and_metrics_from_one_launch(engine):
    """taxi_align_strings_metrics: gapped strings, scores, counts and metrics of the same alignment
    in one launch, equal to the two separate calls."""
    rng = np.random.default_rng(77)
    xs, ys = random_pairs(rng, 75, 30, 400, sub=0.15, indel=0.04)
    engine.set_scores(None)
    engine.load(xs, 0)
    engine.load(ys, 1)
    px = np.arange(len(xs), dtype=np.int32)
    ox, oy, start, off, score, res = engine.align_strings_raw(px, px, want=("counts", "metrics"))
    sep = engine.align_pairs(px, px)
    ax, ay, sc = engine.align_strings(px, px)
    assert np.array_equal(score, sep["score"]) and np.array_equal(sc, score)
    assert np.array_equal(res["counts"], sep["counts"])
    assert np.array_equal(res["metrics"], sep["metrics"], equal_nan=True)
    bx, by = ox.tobytes(), oy.tobytes()
    for k in range(len(xs)):
        assert bx[int(start[k]):int(off[k + 1])] == ax[k] and by[int(start[k]):int(off[k + 1])] == ay[k]
        c = oracle.count(ax[k].decode(), ay[k].decode()) or (0, 0, 0, 0)
        assert tuple(res["counts"][k]) == tuple(c)


@pytest.mark.parametrize("scores", [(1, -1, -8, -1, -1, -1), (1, 0, 0, 0, 0, 0), (2, -3, -5, -2, -4, -1), (1, -1, -1, -1, -2, -2),
                                    (10, 0, -10, -6, 0, 0), (2, -1, -3, -2, -1, -1), (3, -4, -90, -1, -1, -1)])
def test_emitted_alignments_rescore_to_the_optimum(engine, scores):
    """Independent of the oracle: every gapped pair the CUDA path emits (all three kernel variants),
    re-scored column by column under the six scores with end / internal gap typing, reproduces the
    score the kernel reported, and that score is the optimum of a separate score-only dynamic
    programme (tests/rescore.py).  Pins optimality; only the choice among co-optimal alignments
    rests on the oracle."""
    from rescore import best_score, rescore

    rng = np.random.default_rng(abs(hash(scores)) % (2**32))
    xs, ys = random_pairs(rng, 120, 1, 50, sub=0.3, indel=0.1, alphabet=b"ACGTN")
    xs2, ys2 = random_pairs(rng, 80, 1, 50, sub=0.3, indel=0.1, alphabet=b"AT")
    xs, ys = xs + xs2, ys + ys2
    best = [best_score(x.decode(), y.decode(), scores) for x, y in zip(xs, ys)]
    px = np.arange(len(xs), dtype=np.int32)
    for force_general, force_top in ((0, 0), (0, 1), (1, 0)):
        engine.set_option("force_general", force_general)
        engine.set_option("force_top", force_top)
        try:
            engine.set_scores(scores)
            engine.load(xs, 0)
            engine.load(ys, 1)
            ax, ay, sc = engine.align_strings(px, px)
        finally:
            engine.set_option("force_general", 0)
            engine.set_option("force_top", 0)
        for k in range(len(xs)):
            gx, gy = ax[k].decode(), ay[k].decode()
            assert gx.replace("-", "") == xs[k].decode() and gy.replace("-", "") == ys[k].decode()
            assert rescore(gx, gy, scores) == sc[k] == best[k], (force_general, force_top, xs[k], ys[k])


def test_extra_symbols(engine):
    """IUPAC symbols: up to fifteen distinct symbols (all IUPAC nucleotide codes) stay on the fast
    path, more fall back to the general kernel."""
    rng = np.random.default_rng(5)
    xs, ys = random_pairs(rng, 60, 20, 150, alphabet=b"ACGTNRY")
    check_pairs(engine, xs, ys, (1, -1, -8, -1, -1, -1), expect_fast=True)
    xs, ys = random_pairs(rng, 60, 20, 150, alphabet=b"ACGTNRYKMSW")
    check_pairs(engine, xs, ys, (1, -1, -8, -1, -1, -1), expect_fast=True)
    xs, ys = random_pairs(rng, 80, 20, 700, sub=0.1, indel=0.02, alphabet=b"ACGTNRYKMSWBDHV")
    check_pairs(engine, xs, ys, (1, -1, -8, -1, -1, -1), expect_fast=True)
    xs, ys = random_pairs(rng, 60, 20, 150, alphabet=b"ACGTNRYKMSWBDHVXZ")
    check_pairs(engine, xs, ys, (1, -1, -8, -1, -1, -1), expect_fast=False)


def test_multi_stripe_long_pairs(engine):
    """Lengths above one 32*H stripe: rows cross the stripe-boundary buffer (general kernel and
    the multi-stripe packed kernel)."""
    rng = np.random.default_rng(1500)
    xs, ys = random_pairs(rng, 12, 1100, 1700, sub=0.1, indel=0.02)
    check_pairs(engine, xs, ys, (1, -1, -8, -1, -1, -1), expect_fast=True)
    assert_kernel(engine, xs, ys, (1, -1, -8, -1, -1, -1), 18)
    xs, ys = random_pairs(rng, 3, 2500, 3300, sub=0.1, indel=0.02)
    check_pairs(engine, xs, ys, (2, -1, -3, -2, -1, -1), expect_fast=False)   # beyond the 16-bit window
    # BASELINE config C5 geometry: mixed 300-1500 bp in one launch, neighbours of any length
    xs, ys = random_pairs(rng, 40, 300, 1500, sub=0.1, indel=0.02)
    check_pairs(engine, xs, ys, (1, -1, -8, -1, -1, -1), strings=False, expect_fast=True)
    assert_kernel(engine, xs, ys, (1, -1, -8, -1, -1, -1), 18)


def test_very_long_and_very_lopsided_pairs(engine):
    """The general kernel far beyond the packed kernel's window: a 12 000 x 9 000 bp pair (18
    stripes), a 1 bp sequence against 7 000 bp and the reverse, under Gotoh and NW score sets."""
    rng = np.random.default_rng(12000)
    xs, ys = random_pairs(rng, 1, 11800, 12000, sub=0.08, indel=0.01)
    ys = [ys[0][:9000]]
    long7k = bytes(rng.choice(np.frombuffer(b"ACGT", dtype=np.uint8), 7000))
    xs += [b"G", long7k]
    ys += [long7k, b"T"]
    for scores in [(1, -1, -8, -1, -1, -1), (2, -3, -4, -4, -4, -4)]:
        check_pairs(engine, xs, ys, scores, strings=True, expect_fast=False)


def assert_kernel(engine, xs, ys, scores, kernel):
    engine.set_scores(scores)
    engine.load(xs, 0)
    engine.load(ys, 1)
    engine.align_pairs(np.arange(len(xs), dtype=np.int32), np.arange(len(xs), dtype=np.int32), want=("score",))
    assert engine.last_kernel == kernel


def test_ragged_and_tiny(engine):
    xs = [b"A", b"A", b"ACGT" * 40, b"T", b"ACGTN", b"NNNN", b"A" * 33, b"C" * 129]
    ys = [b"A", b"C", b"G", b"ACGT" * 50, b"NNNNN", b"ACGT", b"A" * 31, b"C" * 64 + b"G" + b"C" * 64]
    for scores in [(1, -1, -8, -1, -1, -1), (1, 0, 0, 0, 0, 0)]:
        check_pairs(engine, xs, ys, scores)


def test_empty_sequence_raises(engine):
    engine.set_scores(None)
    engine.load([b"ACGT", b""], 0)
    engine.load([b"ACGT"], 1)
    with pytest.raises(ValueError):
        engine.align_pairs([1], [0])


def test_sample_120_all_pairs(engine):
    """BASELINE config 1: versusAll on Taxi2test1_120.tab, full ordered N x N product."""
    _, seqs = read_tab_sequences(GOLDEN / "Taxi2test1_120.tab")
    n = len(seqs)
    engine.set_scores(None)
    engine.load(seqs, 0)
    got = engine.align_rect(0, n, 0, n)
    from taxi2_b200.engine import pack_strings

    data, off = pack_strings(seqs)
    px, py = np.divmod(np.arange(n * n, dtype=np.int64), n)
    want = oracle.align_count_pairs(data, off, px.astype(np.int32), py.astype(np.int32))
    assert np.array_equal(got["score"].ravel(), want["score"])
    assert np.array_equal(got["counts"].reshape(-1, 4), want["counts"])
    assert_metrics_close(got["metrics"].reshape(-1, 4), want["metrics"])


def test_coi_rect_vs_oracle(engine):
    seqs = coi_like(96, seed=3)
    engine.set_scores(None)
    engine.load(seqs[:32], 0)
    engine.load(seqs[32:], 1)
    got = engine.align_rect(0, 32, 0, 64)
    px, py = np.divmod(np.arange(32 * 64), 64)
    want = oracle_batch(seqs[:32], seqs[32:], px, py, None)
    assert np.array_equal(got["score"].ravel(), want["score"])
    assert np.array_equal(got["counts"].reshape(-1, 4), want["counts"])
    assert_metrics_close(got["metrics"].reshape(-1, 4), want["metrics"])


def test_prealigned_counts(engine):
    """Alignment-free bit-sliced path vs the oracle's string scan, incl. the reference's metrics.tsv."""
    rows = json.loads((GOLDEN / "metrics_cases.json").read_text())["rows"]
    xs = [r["x"] for r in rows] + ["gg-ccnccta", "---"]
    ys = [r["y"] for r in rows] + ["ggaccaccaa", "nnn"]
    rng = np.random.default_rng(11)
    al = np.frombuffer(b"ACGTacgt-N?RY", dtype=np.uint8)
    for _ in range(300):
        L1, L2 = int(rng.integers(0, 200)), int(rng.integers(0, 200))
        xs.append(al[rng.integers(0, len(al), L1)].tobytes().decode())
        ys.append(al[rng.integers(0, len(al), L2)].tobytes().decode())
    engine.load(xs, 0)
    engine.load(ys, 1)
    px = np.arange(len(xs), dtype=np.int32)
    got = engine.count_pairs(px, px)
    for k in range(len(xs)):
        c = oracle.count(xs[k], ys[k])
        want_c = c if c else (0, 0, 0, 0)
        assert tuple(got["counts"][k]) == tuple(want_c), (k, xs[k], ys[k])
        want_m = np.array(oracle.metrics(want_c))
        assert_metrics_close(got["metrics"][k:k + 1], want_m[None, :])
    rect = engine.count_rect(0, 40, 0, 50)
    for i in range(40):
        for j in range(50):
            c = oracle.count(xs[i], ys[j]) or (0, 0, 0, 0)
            assert tuple(rect["counts"][i, j]) == tuple(c)


def test_alignment_free_on_the_ca200_sample(engine):
    """BASELINE config 2 in its runnable form (SURVEY.md 8d, C2 plan i): the reference's 200-row
    resample, un-aligned (26 distinct lengths, lower case + n), params.pairs.align = False ->
    the raw strings go straight into the counting kernel.  All 40 000 ordered pairs vs the oracle."""
    from synth import read_tab_sequences
    ids, seqs = read_tab_sequences(GOLDEN / "Taxi2test1_ca200.tab", normalize=False)
    assert len(seqs) == 200 and len({len(s) for s in seqs}) > 20
    engine.load(seqs, 0)
    got = engine.count_rect(0, 200, 0, 200)
    text = [s.decode() if isinstance(s, bytes) else s for s in seqs]
    distinct = {}
    for i in range(200):
        for j in range(200):
            key = (text[i], text[j])
            if key not in distinct:
                c = oracle.count(*key) or (0, 0, 0, 0)
                distinct[key] = (tuple(c), np.array(oracle.metrics(c)))
            want_c, want_m = distinct[key]
            assert tuple(got["counts"][i, j]) == want_c, (ids[i], ids[j])
            assert_metrics_close(got["metrics"][i, j][None, :], want_m[None, :])


def test_full_size_tile_properties(engine):
    """BASELINE C3 geometry (650 bp, 384 x 384 ordered pairs = 6.2e10 cells): too large for the CPU
    oracle, so check size-independent properties -- the three kernel variants agree bit for bit,
    the diagonal is exact identity, counts are bounded by the lengths, and a sampled subset matches
    the oracle."""
    seqs = coi_like(384, seed=650)
    n = len(seqs)
    lens = np.array([len(s) for s in seqs])
    results = {}
    for name, opts in (("bottom", (0, 0)), ("top", (0, 1)), ("general", (1, 0))):
        engine.set_option("force_general", opts[0])
        engine.set_option("force_top", opts[1])
        try:
            engine.set_scores(None)
            engine.load(seqs, 0)
            results[name] = engine.align_rect(0, n, 0, n)
            results[name]["kernel"] = engine.last_kernel
        finally:
            engine.set_option("force_general", 0)
            engine.set_option("force_top", 0)
    assert (results["bottom"]["kernel"], results["top"]["kernel"], results["general"]["kernel"]) == (17, 16, 32)
    ref = results["general"]
    for name in ("bottom", "top"):
        assert np.array_equal(results[name]["score"], ref["score"])
        assert np.array_equal(results[name]["counts"], ref["counts"])
        assert np.array_equal(results[name]["metrics"], ref["metrics"], equal_nan=True)
    counts, score = ref["counts"], ref["score"]
    diag = np.arange(n)
    real = np.array([sum(c in b"ACGT" for c in s) for s in seqs])
    assert np.array_equal(counts[diag, diag, 0], real) and not counts[diag, diag, 1:].any()
    assert np.array_equal(score[diag, diag], lens)                      # all matches (N matches N)
    assert np.all(ref["metrics"][diag, diag] == 0.0)
    compared = counts[..., :3].sum(-1)
    assert np.all(compared <= np.minimum(lens[:, None], lens[None, :]))
    assert np.all(counts[..., 3] <= lens[:, None] + lens[None, :])
    assert np.all(score <= np.minimum(lens[:, None], lens[None, :]))
    rng = np.random.default_rng(0)
    px, py = rng.integers(0, n, 200), rng.integers(0, n, 200)
    from taxi2_b200.engine import pack_strings

    data, off = pack_strings(seqs)
    want = oracle.align_count_pairs(data, off, px.astype(np.int32), py.astype(np.int32))
    assert np.array_equal(score[px, py], want["score"]) and np.array_equal(counts[px, py], want["counts"])


def test_mixed_length_rectangle_splits_rows(engine):
    """BASELINE config C5 geometry: 300-1500 bp sequences in one rectangle.  Rows longer than one
    packed stripe go through the general kernel, the others through the packed one, and the
    results land in the usual row-major positions."""
    rng = np.random.default_rng(5)
    xs, _ = random_pairs(rng, 24, 300, 1500, sub=0.1, indel=0.02)
    ys, _ = random_pairs(rng, 10, 300, 1500, sub=0.1, indel=0.02)
    assert max(map(len, xs)) > 1023 and min(map(len, xs)) < 1023
    engine.set_scores(None)
    engine.load(xs, 0)
    engine.load(ys, 1)
    got = engine.align_rect(0, len(xs), 0, len(ys))
    assert engine.last_kernel == 48
    sub = engine.align_rect(3, 11, 2, 7)
    px, py = np.divmod(np.arange(len(xs) * len(ys)), len(ys))
    want = oracle_batch(xs, ys, px, py, None)
    assert np.array_equal(got["score"].ravel(), want["score"])
    assert np.array_equal(got["counts"].reshape(-1, 4), want["counts"])
    assert_metrics_close(got["metrics"].reshape(-1, 4), want["metrics"])
    assert np.array_equal(sub["counts"], got["counts"][3:14, 2:9])
    assert np.array_equal(sub["score"], got["score"][3:14, 2:9])


def test_stripe_boundary_lengths(engine):
    """Lengths on both sides of every geometry threshold (rows per lane x 32, with and without the
    spare border slot of the bottom-aligned variant), all combinations, all kernel variants."""
    rng = np.random.default_rng(1023)
    lengths = [1, 2, 31, 32, 33, 255, 256, 257, 383, 384, 511, 512, 513, 671, 672, 673, 767, 768, 1022, 1023, 1024, 1025, 1343, 1344, 1345]
    base = rng.integers(0, 4, size=1400)
    alpha = np.frombuffer(b"ACGT", dtype=np.uint8)

    def variant(n):
        s = alpha[base[:n]].copy()
        hit = rng.random(n) < 0.08
        s[hit] = alpha[rng.integers(0, 4, size=int(hit.sum()))]
        if n > 40:
            cut = int(rng.integers(5, n - 20))
            s = np.concatenate([s[:cut], s[cut + 3:], alpha[rng.integers(0, 4, size=3)]])   # a 3-base deletion, length kept
        return s.tobytes()

    xs, ys = [], []
    for la in lengths:
        for lb in (1, 33, 672, 1023, 1345, la):
            xs.append(variant(la))
            ys.append(variant(lb))
    check_pairs(engine, xs, ys, (1, -1, -8, -1, -1, -1), strings=False, expect_fast=True)
    # pairs in launch order share warps two by two: also run each boundary length on its own
    for la in (671, 672, 1023, 1024):
        check_pairs(engine, [variant(la)] * 3, [variant(la + d) for d in (-1, 0, 1)], (1, -1, -8, -1, -1, -1), expect_fast=True)


def test_extreme_but_eligible_scores(engine):
    """Large penalties / match bonus and non-default end-gap costs: whichever kernel the host's
    range check picks (the first set overflows the 16-bit window at 300 bp and must fall back),
    the results are the oracle's."""
    rng = np.random.default_rng(77)
    xs, ys = random_pairs(rng, 120, 1, 300, sub=0.2, indel=0.05)
    check_pairs(engine, xs, ys, (7, 0, -60, -9, -30, -9), strings=False, expect_fast=False)
    for scores in [(1, -1, -8, -1, -8, -1), (0, -1, -3, -1, -2, -1)]:
        check_pairs(engine, xs, ys, scores, strings=False, expect_fast=True)
    # cheap end gaps next to expensive mismatches: adjacent opposite gaps can be co-optimal, so the
    # restricted recurrence is not provably exact and the host must keep these on the general kernel
    for scores in [(3, -4, -90, -1, -1, -1), (2, -5, -20, -3, -1, -3)]:
        check_pairs(engine, xs, ys, scores, strings=False, expect_fast=False)
    xs, ys = random_pairs(rng, 120, 1, 60, sub=0.2, indel=0.05)
    check_pairs(engine, xs, ys, (7, 0, -60, -9, -30, -9), expect_fast=True)   # same scores fit at 60 bp


def test_host_rectangle_larger_than_one_device_block(engine):
    """taxi_align_rect / taxi_count_rect walk a rectangle of more than 2^24 pairs in blocks of whole
    rows (the device result buffers are bounded); every block must land in its place."""
    rng = np.random.default_rng(224)
    al = np.frombuffer(b"ACGT", dtype=np.uint8)
    xs = [al[rng.integers(0, 4, int(rng.integers(20, 41)))].tobytes() for _ in range(5000)]
    ys = [al[rng.integers(0, 4, int(rng.integers(20, 41)))].tobytes() for _ in range(3400)]   # 1.7e7 pairs > 2^24
    engine.set_scores(None)
    engine.load(xs, 0)
    engine.load(ys, 1)
    big = engine.align_rect(0, len(xs), 0, len(ys), want=("score", "counts"))
    assert engine.stats()["launches"] >= 2
    for x0 in (0, 4930, 4934, 4999):           # first block, the rows around the block boundary, the last row
        part = engine.align_rect(x0, 1, 0, len(ys), want=("score", "counts"))
        assert np.array_equal(big["score"][x0], part["score"][0])
        assert np.array_equal(big["counts"][x0], part["counts"][0])
    rows = rng.integers(0, len(xs), 40)
    cols = rng.integers(0, len(ys), 40)
    want = oracle_batch(xs, ys, rows.astype(np.int32), cols.astype(np.int32), None)
    assert np.array_equal(big["score"][rows, cols], want["score"])
    assert np.array_equal(big["counts"][rows, cols], want["counts"])
    free = engine.count_rect(0, len(xs), 0, len(ys), want=("counts",))
    for k in range(40):
        c = oracle.count(xs[rows[k]].decode(), ys[cols[k]].decode()) or (0, 0, 0, 0)
        assert tuple(free["counts"][rows[k], cols[k]]) == tuple(c)


def test_alignment_free_long_sequences(engine):
    """Pre-aligned rows far longer than a barcode (9 000 and 40 000 columns): the rectangle kernel
    stages fewer x rows per block instead of refusing."""
    rng = np.random.default_rng(9000)
    al = np.frombuffer(b"ACGT-N", dtype=np.uint8)
    for length, n in ((9000, 20), (40000, 6)):
        base = al[rng.choice(6, length, p=[0.24, 0.24, 0.24, 0.24, 0.03, 0.01])]
        seqs = []
        for _ in range(n):
            s = base.copy()
            hit = rng.random(length) < 0.1
            s[hit] = al[rng.integers(0, 6, int(hit.sum()))]
            seqs.append(s.tobytes())
        engine.load(seqs, 0)
        got = engine.count_rect(0, n, 0, n)
        for i in range(n):
            for j in range(n):
                c = oracle.count(seqs[i].decode(), seqs[j].decode()) or (0, 0, 0, 0)
                assert tuple(got["counts"][i, j]) == tuple(c), (length, i, j)
                assert_metrics_close(got["metrics"][i, j][None, :], np.array(oracle.metrics(c))[None, :])


def _junk_rows(rng, n, lo, hi, alphabet=b"ACGTacgt-N?RY", weights=None):
    al = np.frombuffer(alphabet, dtype=np.uint8)
    p = None if weights is None else np.asarray(weights, dtype=float) / sum(weights)
    return [al[rng.choice(len(al), int(rng.integers(lo, hi + 1)), p=p)].tobytes().decode() for _ in range(n)]


@pytest.mark.parametrize("case", ["ragged", "prealigned", "two_sets", "long"])
def test_tensor_core_counts_equal_popcount_and_oracle(engine, case):
    """The tcgen05 int8 contraction (count_tc.cuh) against the popcount kernel and the oracle's
    string scan: rectangles that are not multiples of the 128 x 128 tile, offsets into the sets,
    two sets of different width, leading / trailing / internal gaps (the trim correction in the
    epilogue), missing symbols, lower case, rows far longer than a barcode."""
    from taxi2_b200.engine import pack_strings

    rng = np.random.default_rng({"ragged": 1, "prealigned": 2, "two_sets": 3, "long": 4}[case])
    if case == "ragged":
        xs = _junk_rows(rng, 300, 0, 400)
        ys = None
    elif case == "prealigned":
        base = _junk_rows(rng, 1, 618, 618, b"ACGT")[0]
        xs = []
        for _ in range(450):
            s = np.frombuffer(base.encode(), dtype=np.uint8).copy()
            hit = rng.random(618) < 0.12
            s[hit] = np.frombuffer(b"ACGT-N", dtype=np.uint8)[rng.choice(6, int(hit.sum()), p=[.22, .22, .22, .22, .09, .03])]
            lead, trail = int(rng.integers(0, 60)), int(rng.integers(0, 60))
            s[:lead] = ord("-"); s[618 - trail:] = ord("-")
            xs.append(s.tobytes().decode())
        ys = None
    elif case == "two_sets":
        xs = _junk_rows(rng, 200, 100, 300, b"ACGT-N", [.23, .23, .23, .23, .06, .02])
        ys = _junk_rows(rng, 333, 250, 700, b"ACGT-N", [.23, .23, .23, .23, .06, .02])
    else:
        xs = _junk_rows(rng, 140, 5000, 5200, b"ACGT-N", [.24, .24, .24, .24, .03, .01])
        ys = None
    engine.load(xs, 0)
    if ys is not None:
        engine.load(ys, 1)
    cols = ys if ys is not None else xs
    nx, ny = len(xs), len(cols)
    results = {}
    for kernel, tile_x in ((1, 64), (2, 64), (2, 128), (3, 64)):   # popcount; tensor cores: two CTAs per SM, one, persistent
        engine.set_option("count_kernel", min(kernel, 2))
        engine.set_option("tc_tile_x", tile_x)
        engine.set_option("tc_persistent", int(kernel == 3))
        try:
            full = engine.count_rect(0, nx, 0, ny)
            assert engine.last_kernel == (8 if kernel == 1 else 9)
            part = engine.count_rect(37, nx - 50, 11, ny - 29)
        finally:
            engine.set_option("count_kernel", 0)
            engine.set_option("tc_tile_x", 128)
            engine.set_option("tc_persistent", 0)
        results[kernel, tile_x] = full
        assert np.array_equal(part["counts"], full["counts"][37:nx - 13, 11:ny - 18])
        assert np.array_equal(part["metrics"], full["metrics"][37:nx - 13, 11:ny - 18], equal_nan=True)
    for key in ((2, 64), (2, 128), (3, 64)):
        assert np.array_equal(results[1, 64]["counts"], results[key]["counts"]), key
        assert np.array_equal(results[1, 64]["metrics"], results[key]["metrics"], equal_nan=True), key
    results[2] = results[2, 64]
    data, off = pack_strings(xs + (ys or []))
    px = rng.integers(0, nx, 3000).astype(np.int32)
    py = rng.integers(0, ny, 3000).astype(np.int32)
    want = oracle.count_pairs(data, off, px, py + (nx if ys is not None else 0))
    assert np.array_equal(results[2]["counts"][px, py], want["counts"])
    assert_metrics_close(results[2]["metrics"][px, py], want["metrics"])


def test_table_form_of_the_metric_epilogue(engine):
    """Rows of at most 1920 columns take JC / K2P from a fixed-point table of ln k (exact integer
    differences) instead of the floating-point formula.  Every (n, ts, tv) combination short rows
    can produce -- including the ones whose logarithm argument is exactly zero, where the
    reference's rounding decides between None and a finite value -- against the oracle and against
    the floating-point form of the same kernels: same NaN pattern, p / p-gaps bit for bit, JC / K2P
    within 1e-12 (measured: 1.4e-13 at worst, tools/metrics_table_check.c)."""
    from taxi2_b200.engine import pack_strings

    rng = np.random.default_rng(31)
    rows = []
    for length in (1, 2, 3, 4, 5, 6, 8, 9, 12, 16, 33, 64):
        base = rng.choice(np.frombuffer(b"ACGT", dtype=np.uint8), length)
        for _ in range(28):
            s = base.copy()
            hit = rng.random(length) < rng.choice([0.0, 0.2, 0.5, 0.9])
            s[hit] = rng.choice(np.frombuffer(b"ACGT-N", dtype=np.uint8), int(hit.sum()))
            rows.append(s.tobytes().decode().ljust(64, "-"))
    engine.load(rows, 0)
    n = len(rows)
    got = {}
    for tables in (1, 0):
        engine.set_option("metric_tables", tables)
        try:
            for kernel in (1, 2):
                engine.set_option("count_kernel", kernel)
                got[tables, kernel] = engine.count_rect(0, n, 0, n)
        finally:
            engine.set_option("count_kernel", 0)
            engine.set_option("metric_tables", 1)
    data, off = pack_strings(rows)
    px, py = np.divmod(np.arange(n * n, dtype=np.int32), n)
    want = oracle.count_pairs(data, off, px.astype(np.int32), py.astype(np.int32))
    for key, res in got.items():
        assert np.array_equal(res["counts"].reshape(-1, 4), want["counts"]), key
        assert_metrics_close(res["metrics"].reshape(-1, 4), want["metrics"])
    assert np.array_equal(got[1, 1]["metrics"], got[1, 2]["metrics"], equal_nan=True)      # both kernels, same arithmetic
    assert np.array_equal(got[0, 1]["metrics"], got[0, 2]["metrics"], equal_nan=True)
    both = ~np.isnan(got[1, 1]["metrics"][..., 2:])
    assert np.array_equal(both, ~np.isnan(got[0, 1]["metrics"][..., 2:])) and both.sum() > 1000
    a, b = got[1, 1]["metrics"][..., 2:][both], got[0, 1]["metrics"][..., 2:][both]
    assert np.all(np.abs(a - b) <= 5e-13 * np.abs(b))
    counts = want["counts"]
    nn, ts, tv = counts[:, :3].sum(axis=1), counts[:, 1], counts[:, 2]
    assert ((nn > 0) & (nn - 2 * ts - tv == 0)).any() and ((nn > 0) & (nn - 2 * tv == 0)).any() and ((nn > 0) & (3 * nn - 4 * (ts + tv) == 0)).any()


def test_metric_formulas_on_every_small_count_tuple(engine):
    """taxi_metrics_from_counts: the epilogue of every kernel on its own.  Every (same, ts, tv) with
    n <= 72 (and a few gap counts), plus random tuples up to 2048 and beyond, through the
    floating-point form and the table form, against the oracle's libm formulas: same None pattern,
    p / p-gaps bit for bit, JC / K2P within 1e-12; zero counts and saturated tuples included."""
    rng = np.random.default_rng(77)
    small = np.array([(n - ts - tv, ts, tv, g) for n in range(0, 73) for ts in range(n + 1) for tv in range(n + 1 - ts)
                      for g in (0, 3)], dtype=np.int32)
    n = rng.integers(1, 2049, 40000)
    ts = (rng.random(40000) * (n + 1)).astype(np.int64)
    tv = (rng.random(40000) * (n - ts + 1)).astype(np.int64)
    big = np.stack([n - ts - tv, ts, tv, rng.integers(0, 50, 40000)], axis=1).astype(np.int32)
    long_rows = big.copy()
    long_rows[:, 0] += 5000                                   # beyond the table: both forms take the floating-point route
    counts = np.concatenate([small, big, long_rows])
    want = np.array([oracle.metrics(c) for c in counts])
    for table in (False, True):
        got = engine.metrics_from_counts(counts, table=table)
        assert_metrics_close(got, want)
    assert np.isnan(want[:, 2]).sum() > 1000 and np.isnan(want[:, 3]).sum() > 1000 and (want[:, 3] > 5).any()


def test_intra_task_kernel_for_few_long_pairs(engine):
    """A handful of pairs spanning many stripes: the stripes of each pair are pipelined over the
    warps of a CTA (gotoh_coop_kernel) instead of one warp running them all.  Same scores, counts
    and alignment strings as the one-pair-per-warp kernel and as the oracle, under a Gotoh and a
    Needleman-Wunsch score set, including pairs with fewer stripes than warps and a 1-column y."""
    rng = np.random.default_rng(4000)
    xs, ys = random_pairs(rng, 5, 2200, 5200, sub=0.1, indel=0.02)
    xs += [bytes(rng.choice(np.frombuffer(b"ACGT", dtype=np.uint8), 3000)), b"ACGTTGCA" * 90, xs[0]]
    ys += [b"G", ys[1], ys[0][:700]]
    px = np.arange(len(xs), dtype=np.int32)
    for scores in [(2, -1, -3, -2, -1, -1), (2, -3, -4, -4, -4, -4)]:
        want = oracle_batch(xs, ys, px, px, scores)
        got = {}
        for no_coop in (0, 1):
            engine.set_option("no_coop", no_coop)
            engine.set_option("force_general", 1)
            try:
                engine.set_scores(scores)
                engine.load(xs, 0)
                engine.load(ys, 1)
                res = engine.align_pairs(px, px)
                assert engine.last_kernel == (32 if no_coop else 33)
                ax, ay, sc = engine.align_strings(px, px)
            finally:
                engine.set_option("no_coop", 0)
                engine.set_option("force_general", 0)
            got[no_coop] = (res, ax, ay, sc)
            assert np.array_equal(res["score"], want["score"]) and np.array_equal(res["counts"], want["counts"])
            assert_metrics_close(res["metrics"], want["metrics"])
            assert np.array_equal(sc, want["score"])
        assert got[0][1] == got[1][1] and got[0][2] == got[1][2]
        for k in (0, 5, 6):
            ox, oy, _ = oracle.align(xs[k], ys[k], scores)
            assert got[0][1][k].decode() == ox and got[0][2][k].decode() == oy


@pytest.mark.parametrize("case", ["coi", "ties", "two_sets", "fallback_mixed", "fallback_scores"])
def test_both_orientations_from_one_alignment(engine, case):
    """versus_all.py:746 aligns (x, y) and (y, x).  taxi_align_rect_both derives the second from the
    first wherever the traced path never had to choose between Ix and Iy at equal score, and
    re-aligns the rest: bit-identical to aligning both ways, on barcodes (few sensitive pairs), on
    two-letter low-complexity input (many), across two different sets, and on inputs that have to
    fall back to two ordinary launches (mixed lengths, Needleman-Wunsch scores)."""
    rng = np.random.default_rng({"coi": 1, "ties": 2, "two_sets": 3, "fallback_mixed": 4, "fallback_scores": 5}[case])
    scores = (1, -1, -8, -1, -1, -1)
    if case == "coi":
        xs = coi_like(300, seed=11); ys = None
    elif case == "ties":
        xs, _ = random_pairs(rng, 150, 100, 160, sub=0.3, indel=0.1, alphabet=b"AT"); ys = None
        scores = (1, -1, -2, -1, -1, -1)
    elif case == "two_sets":
        xs = coi_like(130, seed=12); ys = coi_like(90, length=600, seed=13)
    elif case == "fallback_mixed":
        xs, _ = random_pairs(rng, 60, 100, 1400, sub=0.1, indel=0.02); ys = None
    else:
        xs = coi_like(64, length=200, seed=14); ys = None
        scores = (1, 0, 0, 0, 0, 0)
    engine.set_scores(scores)
    engine.load(xs, 0)
    if ys is not None:
        engine.load(ys, 1)
    nx, ny = len(xs), len(ys if ys is not None else xs)
    xy, yx = engine.align_rect_both(0, nx, 0, ny)
    redo = engine.last_redo
    want_xy = engine.align_rect(0, nx, 0, ny)
    # the other orientation the ordinary way: the sets exchanged
    engine.load(ys if ys is not None else xs, 0)
    engine.load(xs, 1)
    want_yx = engine.align_rect(0, ny, 0, nx)
    for key in ("score", "counts"):
        assert np.array_equal(xy[key], want_xy[key]), key
        assert np.array_equal(yx[key], want_yx[key]), key
    assert np.array_equal(xy["metrics"], want_xy["metrics"], equal_nan=True)
    assert np.array_equal(yx["metrics"], want_yx["metrics"], equal_nan=True)
    asymmetric = int((want_yx["counts"] != np.swapaxes(want_xy["counts"], 0, 1)).any(axis=2).sum())
    if case in ("coi", "two_sets"):
        # a few per cent at most are re-aligned among related barcodes, more between two unrelated families
        assert 0 < redo < (0.05 if case == "coi" else 0.25) * nx * ny and redo >= asymmetric
    if case == "ties":
        assert redo >= asymmetric > 0
    if case.startswith("fallback"):
        assert redo == 0
    # a tile and its mirror written straight into their places of one matrix (strided rows)
    if ys is None and case == "coi":
        engine.load(xs, 0)
        big = {k: np.zeros((nx, nx, *t), dtype=d) for k, t, d in (("counts", (4,), np.int32), ("metrics", (4,), np.float64))}
        r, c0 = slice(10, 110), slice(150, 290)
        engine.align_rect_both(10, 100, 150, 140, want=("counts", "metrics"),
                               out={k: v[r, c0] for k, v in big.items()}, out_t={k: v[c0, r] for k, v in big.items()})
        assert np.array_equal(big["counts"][r, c0], want_xy["counts"][r, c0]) and np.array_equal(big["counts"][c0, r], want_xy["counts"][c0, r])
        assert np.array_equal(big["metrics"][c0, r], want_xy["metrics"][c0, r], equal_nan=True)
        assert not big["counts"][:10].any() and not big["counts"][110:150, :150].any()
