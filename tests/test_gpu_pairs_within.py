"""Pairs within a distance, selected and compacted on the device (taxi_pairs_within /
Engine.pairs_within / MultiEngine.pairs_within), against the full metrics and counts matrix of the
same rectangle (align_rect / count_rect, which the rest of the suite checks against the oracle)
filtered with numpy: v not NaN and v * scale <= threshold, row-major, ascending column within a
row.  row_ptr, index, metrics and counts must match bit for bit."""
from __future__ import annotations

import numpy as np
import pytest

from synth import coi_like

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def eng():
    from taxi2_b200.engine import Engine

    e = Engine(0)
    yield e
    e.close()


def select(full: dict, t: float, metric: int, y0: int = 0, scale: float = 1.0, x0: int | None = None) -> dict:
    """numpy restatement; x0 given: drop the pairs (x0 + r, y0 + c) with x0 + r == y0 + c."""
    v = full["metrics"][..., metric]
    with np.errstate(invalid="ignore"):
        keep = ~np.isnan(v) & (v * scale <= t)
    if x0 is not None:
        r = np.arange(v.shape[0])[:, None] + x0
        c = np.arange(v.shape[1])[None, :] + y0
        keep &= r != c
    rows, cols = np.nonzero(keep)
    row_ptr = np.zeros(v.shape[0] + 1, dtype=np.int64)
    np.cumsum(keep.sum(axis=1), out=row_ptr[1:])
    return dict(row_ptr=row_ptr, index=(cols + y0).astype(np.int32), metrics=full["metrics"][rows, cols],
                counts=full["counts"][rows, cols])


def assert_same(got: dict, want: dict, what=None):
    assert got["row_ptr"].dtype == np.int64 and got["index"].dtype == np.int32, what
    assert np.array_equal(got["row_ptr"], want["row_ptr"]), what
    assert np.array_equal(got["index"], want["index"]), what
    assert got["metrics"].shape == want["metrics"].shape and got["counts"].shape == want["counts"].shape, what
    assert np.array_equal(got["metrics"].view(np.uint64), want["metrics"].view(np.uint64)), what
    assert np.array_equal(got["counts"], want["counts"]), what


def reference(eng, align: bool, x0: int, nx: int, y0: int, ny: int) -> dict:
    call = eng.align_rect if align else eng.count_rect
    return call(x0, nx, y0, ny, want=("counts", "metrics"))


def small_sets(align: bool):
    queries = coi_like(60, seed=19)
    refs = coi_like(45, seed=20)
    length = 650 if align else 600
    queries = [q[:length] for q in queries] + [b"N" * length]                 # a query without any defined distance
    refs = [r[:length] for r in refs]
    refs = refs + refs[:15] + [queries[3], queries[3]] + [b"N" * length] * 3   # exact ties; three undefined columns
    return queries, refs


def load(eng, queries, refs=None):
    eng.set_scores(None)
    eng.load(queries, 0)
    if refs is not None:
        eng.load(refs, 1)


@pytest.mark.parametrize("align", [True, False], ids=["align", "free"])
def test_every_metric_and_threshold_against_the_full_matrix(eng, align):
    queries, refs = small_sets(align)
    load(eng, queries, refs)
    nx, ny = len(queries), len(refs)
    full = reference(eng, align, 0, nx, 0, ny)
    for metric in range(4):
        v = full["metrics"][..., metric]
        defined = np.sort(v[~np.isnan(v)])
        edge = float(defined[len(defined) // 3])          # a value that occurs in the matrix
        below = float(np.nextafter(edge, -np.inf))
        for t in (0.0, edge, below, np.inf, -1.0):
            got = eng.pairs_within(0, nx, 0, ny, t, metric, align)
            assert_same(got, select(full, t, metric), (metric, t))
            assert got["row_ptr"][-1] == got["row_ptr"][-2]   # the undefined query has no pairs
        # the edge pairs are in at `edge` and out just below it
        at_edge = int((v == edge).sum())
        assert at_edge > 0
        n_edge = eng.pairs_within(0, nx, 0, ny, edge, metric, align)["row_ptr"][-1]
        n_below = eng.pairs_within(0, nx, 0, ny, below, metric, align)["row_ptr"][-1]
        assert n_edge - n_below == at_edge
        # +inf selects every defined pair
        assert eng.pairs_within(0, nx, 0, ny, np.inf, metric, align)["row_ptr"][-1] == int((~np.isnan(v)).sum())
        # a percentage threshold: scale 100 against 100 * an occurring value, the tasks' `d * 100 <= similarity`
        t100 = 100.0 * edge
        got = eng.pairs_within(0, nx, 0, ny, t100, metric, align, scale=100.0)
        assert_same(got, select(full, t100, metric, scale=100.0), (metric, "scale"))
    # threshold 0: the duplicated references tie at exactly 0 and are both in
    got = eng.pairs_within(0, nx, 0, ny, 0.0, 0, align)
    row3 = got["index"][got["row_ptr"][3]:got["row_ptr"][4]]
    assert ny - 5 in row3 and ny - 4 in row3


@pytest.mark.parametrize("align", [True, False], ids=["align", "free"])
def test_nothing_selected_fetches_empty_arrays(eng, align):
    queries, refs = small_sets(align)
    load(eng, queries, refs)
    got = eng.pairs_within(0, len(queries), 0, len(refs), -1.0, 2, align)
    assert (got["row_ptr"] == 0).all() and got["row_ptr"].shape == (len(queries) + 1,)
    assert got["index"].shape == (0,) and got["metrics"].shape == (0, 4) and got["counts"].shape == (0, 4)


@pytest.mark.parametrize("align", [True, False], ids=["align", "free"])
def test_offsets(eng, align):
    queries, refs = small_sets(align)
    load(eng, queries, refs)
    x0, nx, y0, ny = 7, 30, 30, 35
    full = reference(eng, align, x0, nx, y0, ny)
    for metric, t in ((0, 0.05), (3, 0.2), (1, np.inf)):
        got = eng.pairs_within(x0, nx, y0, ny, t, metric, align)
        assert_same(got, select(full, t, metric, y0), (metric, t))
        assert ((got["index"] >= y0) & (got["index"] < y0 + ny)).all()


@pytest.mark.parametrize("align", [True, False], ids=["align", "free"])
def test_skip_self_drops_only_the_diagonal(eng, align):
    queries, _ = small_sets(align)
    load(eng, queries)                                    # set 0 serves as both sets
    n = len(queries)
    for x0, nx, y0, ny in ((0, n, 0, n), (5, 20, 12, 30)):
        full = reference(eng, align, x0, nx, y0, ny)
        keep = eng.pairs_within(x0, nx, y0, ny, 0.1, 0, align)
        got = eng.pairs_within(x0, nx, y0, ny, 0.1, 0, align, skip_self=True)
        assert_same(keep, select(full, 0.1, 0, y0))
        assert_same(got, select(full, 0.1, 0, y0, x0=x0))
        # the dropped pairs are exactly the defined diagonal ones inside the rectangle (distance 0)
        diag = [i for i in range(max(x0, y0), min(x0 + nx, y0 + ny)) if i != n - 1]
        assert keep["row_ptr"][-1] - got["row_ptr"][-1] == len(diag) > 0
    load(eng, queries, queries)
    from taxi2_b200 import _native as N

    with pytest.raises(N.TaxiNativeError) as err:
        eng.pairs_within(0, n, 0, n, 0.1, 0, align, skip_self=True)
    assert err.value.code == N.E_ARG


def test_refusals(eng):
    from taxi2_b200 import _native as N
    from taxi2_b200.engine import Engine

    with Engine(0) as fresh:   # nothing computed yet: nothing held
        assert fresh._lib.taxi_pairs_within_fetch(fresh._ctx, None, None, None) == N.E_ARG
    load(eng, coi_like(5, seed=1))
    for args, kw in (((0, 5, 0, 5, 0.1, 4), {}), ((0, 5, 0, 5, np.nan), {}), ((0, 5, 0, 5, 0.1), dict(scale=0.0)),
                     ((0, 5, 0, 5, 0.1), dict(scale=-1.0)), ((0, 5, 0, 5, 0.1), dict(scale=np.inf)),
                     ((0, 5, 0, 5, 0.1), dict(scale=np.nan)), ((0, 5, 0, 0, 0.1), {})):
        with pytest.raises(N.TaxiNativeError) as err:
            eng.pairs_within(*args, **kw)
        assert err.value.code == N.E_ARG, (args, kw)
    # a held result is fetched as often as wanted, and is gone after another call that computes
    got = eng.pairs_within(0, 5, 0, 5, 0.5, 0, True)
    total = int(got["row_ptr"][-1])
    assert total >= 5
    index = np.empty(total, dtype=np.int32)
    assert eng._lib.taxi_pairs_within_fetch(eng._ctx, index.ctypes.data, None, None) == 0
    assert np.array_equal(index, got["index"])
    eng.align_rect(0, 5, 0, 5)
    assert eng._lib.taxi_pairs_within_fetch(eng._ctx, index.ctypes.data, None, None) == N.E_ARG


@pytest.fixture(scope="module")
def wide():
    """C4-width rows: 20 000 barcode references (first the duplicates of a few)."""
    refs = coi_like(20_000, seed=44)
    refs[100:110] = refs[:10]
    return coi_like(7_000, seed=45), refs


@pytest.mark.parametrize("align,nx", [(True, 900), (False, 6_800)], ids=["align", "free"])
def test_several_device_blocks_at_20000_columns(eng, wide, align, nx):
    """nx is larger than one device block (2^24 aligned / 2^27 alignment-free pairs per block, so
    838 / 6710 rows at 20 000 columns).  The first rows, the rows on both sides of the block edge and
    the last rows are compared with the full matrix.  Alignment-free, three rows hold one real base
    followed by gaps: one compared column each, so at threshold 0 nearly every column is selected."""
    queries, refs = wide
    queries = [q if align else q[:600] for q in queries[:nx]]
    refs = refs if align else [r[:600] for r in refs]
    ny = len(refs)
    edge = (1 << 24 if align else 1 << 27) // ny
    assert nx > edge
    if not align:
        first = max(set(r[:1] for r in refs), key=lambda b: sum(r[:1] == b for r in refs))
        for row in (edge - 1, edge, nx - 3):
            queries[row] = first + b"-" * 599
    load(eng, queries, refs)
    t = 0.02 if align else 0.0
    got = eng.pairs_within(0, nx, 0, ny, t, 0, align)
    rp = got["row_ptr"]
    assert rp[0] == 0 and (np.diff(rp) >= 0).all() and rp[-1] == len(got["index"])
    for lo, hi in ((0, 40), (edge - 40, min(nx, edge + 40)), (nx - 20, nx)):
        full = reference(eng, align, lo, hi - lo, 0, ny)
        want = select(full, t, 0)
        part = dict(row_ptr=rp[lo:hi + 1] - rp[lo], index=got["index"][rp[lo]:rp[hi]],
                    metrics=got["metrics"][rp[lo]:rp[hi]], counts=got["counts"][rp[lo]:rp[hi]])
        assert_same(part, want, (lo, hi))
    if not align:
        for row in (edge - 1, edge, nx - 3):
            assert rp[row + 1] - rp[row] > 0.7 * ny, row


@pytest.mark.parametrize("align", [True, False], ids=["align", "free"])
def test_multi_engine_tiles_equal_one_call(eng, align):
    """Two contexts on device 0, row and column tiles assembled on the host (combine_within)."""
    from taxi2_b200.multi import MultiEngine

    queries, refs = small_sets(align)
    load(eng, queries, refs)
    with MultiEngine([0, 0]) as multi:
        multi.load(queries, 0)
        multi.load(refs, 1)
        for metric, t in ((0, 0.05), (3, 0.3), (1, np.inf), (2, -1.0)):
            want = eng.pairs_within(0, len(queries), 0, len(refs), t, metric, align)
            for rows, col_tiles in ((None, 1), (9, 3), (61, 3), (4, 7)):
                got = multi.pairs_within(t, metric, align, rows_per_tile=rows, col_tiles=col_tiles)
                assert_same(got, want, (metric, t, rows, col_tiles))
        # set 0 against itself, the diagonal skipped
        multi.load(queries, 0)
        load(eng, queries)
        want = eng.pairs_within(0, len(queries), 0, len(queries), 0.05, 0, align, skip_self=True)
        got = multi.pairs_within(0.05, 0, align, skip_self=True, rows_per_tile=9, col_tiles=3)
        assert_same(got, want, "skip_self")
