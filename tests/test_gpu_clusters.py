"""Clusters within a distance, linked and united on the device (taxi_clusters_within /
Engine.clusters_within / MultiEngine.clusters_within), against the full metrics matrix of the same
rectangle (align_rect / count_rect, which the rest of the suite checks against the oracle): the
pairs with v not NaN and v * scale <= t, both orientations, go to scipy's connected_components
over all n sequences of set 0, and every component is labelled with its smallest member.  Labels
must match exactly."""
from __future__ import annotations

import numpy as np
import pytest
from scipy.sparse import coo_matrix
from scipy.sparse.csgraph import connected_components

from synth import coi_like

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def eng():
    from taxi2_b200.engine import Engine

    e = Engine(0)
    yield e
    e.close()


def edges(metrics: np.ndarray, t: float, metric: int, x0: int, y0: int, scale: float = 1.0):
    """The links of a rectangle's (nx, ny, 4) metrics at threshold t, as set-0 index pairs."""
    v = metrics[..., metric]
    with np.errstate(invalid="ignore"):
        keep = ~np.isnan(v) & (v * scale <= t)
    r, c = np.nonzero(keep)
    i, j = r + x0, c + y0
    other = i != j
    return i[other], j[other]


def components(n: int, parts) -> np.ndarray:
    """Canonical labels (smallest member) of the graph of n nodes with the edges of every (i, j) part."""
    i = np.concatenate([np.asarray(p[0], dtype=np.int64) for p in parts] + [np.zeros(0, np.int64)])
    j = np.concatenate([np.asarray(p[1], dtype=np.int64) for p in parts] + [np.zeros(0, np.int64)])
    graph = coo_matrix((np.ones(len(i), dtype=np.int8), (i, j)), shape=(n, n))
    _, comp = connected_components(graph, directed=False)
    low = np.full(comp.max() + 1, n, dtype=np.int64)
    np.minimum.at(low, comp, np.arange(n))
    return low[comp].astype(np.int32)


def rect(eng, align: bool, x0: int, nx: int, y0: int, ny: int) -> np.ndarray:
    call = eng.align_rect if align else eng.count_rect
    return call(x0, nx, y0, ny, want=("metrics",))["metrics"]


def small_set(align: bool) -> list[bytes]:
    """76 barcodes of 20 species (3 - 4 individuals each), six exact duplicates, one all-N sequence."""
    length = 650 if align else 600
    seqs = [s[:length] for s in coi_like(69, seed=19, genera=5, species=4)]
    return seqs + seqs[:6] + [b"N" * length]


def load(eng, seqs, refs=None):
    eng.set_scores(None)
    eng.load(seqs, 0)
    if refs is not None:
        eng.load(refs, 1)


@pytest.mark.parametrize("align", [True, False], ids=["align", "free"])
def test_every_metric_and_threshold_against_the_full_square(eng, align):
    seqs = small_set(align)
    load(eng, seqs)
    n = len(seqs)
    full = rect(eng, align, 0, n, 0, n)
    off = ~np.eye(n, dtype=bool)
    for metric in range(4):
        v = full[..., metric][off]
        defined = np.sort(v[~np.isnan(v)])
        edge = float(defined[len(defined) // 20])          # a value that occurs off the diagonal
        below = float(np.nextafter(edge, -np.inf))
        ts = [0.0, edge, below, np.inf, -1.0]
        singles = []
        for t in ts:
            got = eng.clusters_within(0, n, 0, n, t, metric, align)
            assert got.dtype == np.int32 and got.shape == (1, n)
            assert np.array_equal(got[0], components(n, [edges(full, t, metric, 0, 0)])), (metric, t)
            singles.append(got[0])
        # the duplicates join their originals at 0; +inf links every defined pair, the all-N
        # sequence stays alone; a negative threshold links nothing
        assert (singles[0][69:75] == singles[0][:6]).all()
        assert singles[3][n - 1] == n - 1 and len(np.unique(singles[3])) <= len(np.unique(singles[1]))
        assert np.array_equal(singles[4], np.arange(n))
        # all thresholds in one call, in any order: bit for bit one call each
        order = [3, 0, 4, 2, 1]
        many = eng.clusters_within(0, n, 0, n, [ts[k] for k in order], metric, align)
        assert np.array_equal(many, np.stack([singles[k] for k in order])), metric
        # a percentage threshold: scale 100 against 100 * an occurring value
        t100 = 100.0 * edge
        got = eng.clusters_within(0, n, 0, n, t100, metric, align, scale=100.0)
        assert np.array_equal(got[0], components(n, [edges(full, t100, metric, 0, 0, scale=100.0)])), (metric, "scale")


def test_species_structure():
    """coi_like: individuals about 1 % from their species, species about 6 % from their genus.  In
    this set conspecifics are at most 9.4 % apart (p-distance, aligned) and connected at 6 %, other
    species at least 8.3 % apart, so at 7 % the clusters are the species."""
    from taxi2_b200.engine import Engine

    genera, species = 4, 5
    seqs = coi_like(300, seed=61, genera=genera, species=species)
    n = len(seqs)
    k = np.arange(n)
    sp = (k % genera) * species + (k // genera) % species
    first = {}
    want = np.array([first.setdefault(s, i) for i, s in enumerate(sp.tolist())], dtype=np.int32)
    with Engine(0) as e:
        e.load(seqs, 0)
        full = rect(e, True, 0, n, 0, n)
        got = e.clusters_within(0, n, 0, n, [0.07, 0.2], 0, True)
    assert np.array_equal(got[0], components(n, [edges(full, 0.07, 0, 0, 0)]))
    assert np.array_equal(got[0], want)
    assert np.array_equal(got[1], components(n, [edges(full, 0.2, 0, 0, 0)]))
    assert len(np.unique(got[1])) < len(np.unique(got[0]))


@pytest.mark.parametrize("align", [True, False], ids=["align", "free"])
def test_sub_rectangles(eng, align):
    seqs = small_set(align)
    load(eng, seqs)
    n = len(seqs)
    for x0, nx, y0, ny in ((7, 30, 30, 35), (40, 36, 0, 76), (0, 76, 50, 1), (75, 1, 0, 76), (20, 25, 20, 25)):
        full = rect(eng, align, x0, nx, y0, ny)
        for metric, t in ((0, 0.03), (3, 0.1), (1, np.inf)):
            got = eng.clusters_within(x0, nx, y0, ny, t, metric, align)
            assert np.array_equal(got[0], components(n, [edges(full, t, metric, x0, y0)])), (x0, nx, y0, ny, metric, t)


@pytest.mark.parametrize("align", [True, False], ids=["align", "free"])
def test_seed_chaining(eng, align):
    """Two disjoint row ranges, the second seeded with the first's labels, equal one call; so do
    column halves, and a seed with nothing to add comes back unchanged."""
    seqs = small_set(align)
    load(eng, seqs)
    n = len(seqs)
    ts = [0.02, 0.0, 0.06, np.inf]
    whole = eng.clusters_within(0, n, 0, n, ts, 0, align)
    for cut in (1, 30, 75):
        a = eng.clusters_within(0, cut, 0, n, ts, 0, align)
        assert np.array_equal(eng.clusters_within(cut, n - cut, 0, n, ts, 0, align, seed=a), whole), cut
        b = eng.clusters_within(cut, n - cut, 0, n, ts, 0, align)
        assert np.array_equal(eng.clusters_within(0, cut, 0, n, ts, 0, align, seed=b), whole), cut
    left = eng.clusters_within(0, n, 0, 40, ts, 0, align)
    assert np.array_equal(eng.clusters_within(0, n, 40, n - 40, ts, 0, align, seed=left), whole)
    assert np.array_equal(eng.clusters_within(0, n, 0, n, ts, 0, align, seed=whole), whole)
    # nx = 0: the seed, or the singletons
    assert np.array_equal(eng.clusters_within(5, 0, 0, n, ts, 0, align, seed=whole), whole)
    assert np.array_equal(eng.clusters_within(5, 0, 0, n, ts, 0, align), np.tile(np.arange(n, dtype=np.int32), (len(ts), 1)))


@pytest.fixture(scope="module")
def many():
    seqs = coi_like(20_000, seed=44)
    seqs[100:110] = seqs[:10]
    return seqs


def sliced_reference(eng, align: bool, n: int, ts, metric: int, step: int) -> list[np.ndarray]:
    """Components of the whole square at every threshold, the matrix computed and filtered in row slices."""
    parts = [[] for _ in ts]
    for x0 in range(0, n, step):
        nx = min(step, n - x0)
        full = rect(eng, align, x0, nx, 0, n)
        for k, t in enumerate(ts):
            parts[k].append(edges(full, t, metric, x0, 0))
        del full
    return [components(n, p) for p in parts]


@pytest.mark.parametrize("align,n", [(True, 5_000), (False, 20_000)], ids=["align", "free"])
def test_several_device_blocks(eng, many, align, n):
    """n x n is several device blocks (2^24 aligned / 2^27 alignment-free pairs each: 3355 rows of
    5000, 6710 rows of 20 000), and the forests persist across them."""
    seqs = [s if align else s[:600] for s in many[:n]]
    load(eng, seqs)
    rows = (1 << 24 if align else 1 << 27) // n
    assert n > rows
    sample = rect(eng, align, 0, 64, 0, n)[..., 0]
    sample = np.sort(sample[~np.isnan(sample)])
    ts = [0.0, float(sample[len(sample) // 200]), float(sample[len(sample) // 50]), 0.03]
    got = eng.clusters_within(0, n, 0, n, ts, 0, align)
    want = sliced_reference(eng, align, n, ts, 0, 1000)
    for k, t in enumerate(ts):
        assert np.array_equal(got[k], want[k]), t
    assert (got[0][100:110] == np.arange(10)).all()
    # components that cross the block edges
    for k in (1, 2):
        assert (got[k][rows:] < rows).any()


@pytest.mark.parametrize("align", [True, False], ids=["align", "free"])
def test_multi_engine_tiles_equal_one_call(eng, align):
    """Two contexts on device 0, each chaining its tiles through the seed, merged on the host."""
    from taxi2_b200.multi import MultiEngine

    seqs = small_set(align)
    load(eng, seqs)
    n = len(seqs)
    ts = [0.02, 0.0, 0.06, np.inf, -1.0]
    with MultiEngine([0, 0]) as multi:
        multi.load(seqs, 0)
        for metric in (0, 3):
            want = eng.clusters_within(0, n, 0, n, ts, metric, align)
            for rows, col_tiles in ((None, 1), (9, 1), (9, 3), (61, 3), (4, 7)):
                got = multi.clusters_within(ts, metric, align, rows_per_tile=rows, col_tiles=col_tiles)
                assert got["labels"].dtype == np.int32 and got["clusters"].dtype == np.int64
                assert np.array_equal(got["labels"], want), (metric, rows, col_tiles)
                assert np.array_equal(got["clusters"], [len(np.unique(w)) for w in want])
                assert got["tiles"] > 1 or rows is None
        one = multi.clusters_within(0.02, 0, align, scale=1.0)
        assert one["labels"].shape == (1, n)


def test_refusals(eng):
    from taxi2_b200 import _native as N

    seqs = coi_like(6, seed=1)
    load(eng, seqs, seqs)                                # set 1 loaded
    with pytest.raises(N.TaxiNativeError) as err:
        eng.clusters_within(0, 6, 0, 6, 0.1)
    assert err.value.code == N.E_ARG
    load(eng, seqs)
    good = np.arange(6, dtype=np.int32)[None, :]
    for args, kw in (((0, 6, 0, 6, []), {}), ((0, 6, 0, 6, [0.1] * 9), {}), ((0, 6, 0, 6, [0.1, np.nan]), {}),
                     ((0, 6, 0, 6, 0.1), dict(scale=0.0)), ((0, 6, 0, 6, 0.1), dict(scale=-1.0)),
                     ((0, 6, 0, 6, 0.1), dict(scale=np.inf)), ((0, 6, 0, 6, 0.1), dict(scale=np.nan)),
                     ((0, 6, 0, 6, 0.1), dict(metric=4)), ((0, 6, 0, 6, 0.1), dict(metric=-1)),
                     ((0, 6, 0, 0, 0.1), {}), ((0, 7, 0, 6, 0.1), {}), ((0, 6, 3, 4, 0.1), {}),
                     ((0, 6, 0, 6, 0.1), dict(seed=np.array([[0, 2, 2, 3, 4, 5]], np.int32))),     # label above its node
                     ((0, 6, 0, 6, 0.1), dict(seed=np.array([[0, 0, 1, 3, 4, 5]], np.int32))),     # label of a label
                     ((0, 6, 0, 6, 0.1), dict(seed=np.array([[-1, 1, 2, 3, 4, 5]], np.int32))),
                     ((0, 6, 0, 6, [0.1, 0.2]), dict(seed=np.vstack([good, [[0, 1, 2, 3, 4, 6]]]).astype(np.int32)))):
        with pytest.raises(N.TaxiNativeError) as err:
            eng.clusters_within(*args, **kw)
        assert err.value.code == N.E_ARG, (args, kw)
    ts = np.array([0.1], dtype=np.float64)
    out = np.empty((1, 6), dtype=np.int32)
    lib, ctx = eng._lib, eng._ctx
    assert lib.taxi_clusters_within(ctx, 0, 6, 0, 6, 0, 1, None, 1, 1.0, None, out.ctypes.data) == N.E_ARG
    assert lib.taxi_clusters_within(ctx, 0, 6, 0, 6, 0, 1, ts.ctypes.data, 1, 1.0, None, None) == N.E_ARG
    # a refused call leaves the output untouched; ny = 0 is refused with nx = 0 too
    out.fill(-7)
    seed6 = np.zeros((1, 6), dtype=np.int32)
    for x0, nx, y0, ny in ((0, 6, 0, 0), (0, 0, 0, 0), (3, 0, 6, 0)):
        assert lib.taxi_clusters_within(ctx, x0, nx, y0, ny, 0, 1, ts.ctypes.data, 1, 1.0, seed6.ctypes.data,
                                        out.ctypes.data) == N.E_ARG, (x0, nx, y0, ny)
        assert (out == -7).all(), (x0, nx, y0, ny)
    # a seed that is the output array itself is read before it is written
    seed = np.array([[0, 0, 2, 3, 3, 5]], dtype=np.int32)
    want = eng.clusters_within(0, 6, 0, 6, 0.1, seed=seed)
    assert lib.taxi_clusters_within(ctx, 0, 6, 0, 6, 0, 1, ts.ctypes.data, 1, 1.0, seed.ctypes.data, seed.ctypes.data) == 0
    assert np.array_equal(seed, want)
    # the call computes on the context: a held pairs_within result is dropped
    eng.pairs_within(0, 6, 0, 6, 0.5, 0, True)
    eng.clusters_within(0, 6, 0, 6, 0.1)
    assert lib.taxi_pairs_within_fetch(ctx, None, None, None) == N.E_ARG
    # more columns than one device block (2^24 pairs aligned): refused before anything is computed
    big = (1 << 24) + 1
    data = np.full(big, ord("A"), dtype=np.uint8)
    off = np.arange(big + 1, dtype=np.int64)
    from taxi2_b200.engine import Engine

    with Engine(0) as e:
        e.load((data, off), 0)
        kept = np.full((1, big), -7, dtype=np.int32)
        assert e._lib.taxi_clusters_within(e._ctx, 0, 1, 0, big, 0, 1, ts.ctypes.data, 1, 1.0, None, kept.ctypes.data) == N.E_ARG
        assert "device block" in N.load().taxi_last_error().decode()
        assert (kept == -7).all()
