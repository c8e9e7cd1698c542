"""The k closest references per query, selected on the device (taxi_best_rows_k / Engine.best_rows_k /
MultiEngine.best_matches_k), against the full metrics and counts matrix of the same rectangle
(align_rect / count_rect, which the rest of the suite checks against the oracle) sorted with numpy
in the same key order: ascending value, equal values by the smaller column, NaN never ranked.
Index, metrics and counts must match bit for bit."""
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


def select_k(metrics: np.ndarray, counts: np.ndarray, k: int, metric: int, y0: int = 0):
    """numpy restatement: a stable sort puts NaN last and equal values in column order."""
    vals = metrics[..., metric]
    nx, ny = vals.shape
    kk = min(k, ny)
    order = np.argsort(vals, axis=1, kind="stable")[:, :kk]
    rows = np.arange(nx)[:, None]
    defined = ~np.isnan(vals[rows, order])
    index = np.full((nx, k), -1, dtype=np.int32)
    best = np.full((nx, k, 4), np.nan)
    cnt = np.zeros((nx, k, 4), dtype=np.int32)
    index[:, :kk] = np.where(defined, order + y0, -1)
    best[:, :kk] = np.where(defined[..., None], metrics[rows, order], np.nan)
    cnt[:, :kk] = np.where(defined[..., None], counts[rows, order], 0)
    return index, best, cnt


def assert_same(got: dict, want: tuple, what=None):
    index, best, cnt = want
    assert got["index"].shape == index.shape and got["metrics"].shape == best.shape, what
    assert np.array_equal(got["index"], index), what
    assert np.array_equal(got["metrics"].view(np.uint64), best.view(np.uint64)), what
    assert np.array_equal(got["counts"], cnt), what


def reference(eng, align: bool, x0: int, nx: int, y0: int, ny: int) -> dict:
    call = eng.align_rect if align else eng.count_rect
    return call(x0, nx, y0, ny, want=("counts", "metrics"))


def small_sets(align: bool):
    queries = coi_like(60, seed=9)
    refs = coi_like(45, seed=10)
    length = 650 if align else 600
    queries = [q[:length] for q in queries] + [b"N" * length]                 # a query without any defined distance
    refs = [r[:length] for r in refs]
    refs = refs + refs[:15] + [queries[3], queries[3]] + [b"N" * length] * 3   # exact ties; three undefined columns
    return queries, refs


@pytest.mark.parametrize("align", [True, False], ids=["align", "free"])
def test_every_metric_and_k_against_the_full_matrix(eng, align):
    queries, refs = small_sets(align)
    eng.set_scores(None)
    eng.load(queries, 0)
    eng.load(refs, 1)
    nx, ny = len(queries), len(refs)
    full = reference(eng, align, 0, nx, 0, ny)
    defined = ~np.isnan(full["metrics"][..., 0])
    assert not defined[-1].any() and (defined.sum(axis=1) < 64).all()   # fewer than 64 defined values in every row
    for metric in range(4):
        first = eng.best_rows(0, nx, 0, ny, metric, align)
        for k in (1, 2, 10, 64):
            got = eng.best_rows_k(0, nx, 0, ny, k, metric, align)
            assert_same(got, select_k(full["metrics"], full["counts"], k, metric), (metric, k))
            if k == 1:   # the single best match, bit for bit
                assert np.array_equal(got["index"][:, 0], first["index"])
                assert np.array_equal(got["metrics"][:, 0].view(np.uint64), first["metrics"].view(np.uint64))
                assert np.array_equal(got["counts"][:, 0], first["counts"])
    # the duplicated references tie exactly: query 3 has distance 0 to two identical columns, the smaller first
    got = eng.best_rows_k(0, nx, 0, ny, 3, 0, align)
    assert got["index"][3, :2].tolist() == [ny - 5, ny - 4] and (got["metrics"][3, :2, 0] == 0).all()


@pytest.mark.parametrize("align", [True, False], ids=["align", "free"])
def test_k_beyond_the_columns_and_offsets(eng, align):
    queries, refs = small_sets(align)
    eng.set_scores(None)
    eng.load(queries, 0)
    eng.load(refs, 1)
    x0, nx, y0, ny = 7, 30, 30, 20
    full = reference(eng, align, x0, nx, y0, ny)
    for k in (20, 21, 64):
        got = eng.best_rows_k(x0, nx, y0, ny, k, 2, align)
        assert_same(got, select_k(full["metrics"], full["counts"], k, 2, y0), k)
        assert (got["index"][:, ny:] == -1).all()


def test_refusals(eng):
    from taxi2_b200 import _native as N

    eng.load(coi_like(5, seed=1), 0)
    for args in ((0, 5, 0, 5, 0), (0, 5, 0, 5, 65), (0, 5, 0, 0, 3), (0, 5, 0, 5, -1)):
        with pytest.raises(N.TaxiNativeError) as err:
            eng.best_rows_k(*args)
        assert err.value.code == N.E_ARG, args


@pytest.fixture(scope="module")
def wide():
    """C4-width rows: 20 000 barcode references (first the duplicates of a few)."""
    refs = coi_like(20_000, seed=44)
    refs[100:110] = refs[:10]
    return coi_like(7_000, seed=45), refs


@pytest.mark.parametrize("align,nx", [(True, 900), (False, 6_800)], ids=["align", "free"])
def test_several_device_blocks_at_20000_columns(eng, wide, align, nx):
    """nx is larger than one device block (2^24 aligned / 2^27 alignment-free pairs per block, so
    838 / 6710 rows at 20 000 columns); the rows on both sides of the block edge and the first rows
    are compared with the full matrix at k = 64."""
    queries, refs = wide
    queries = [q if align else q[:600] for q in queries[:nx]]
    refs = refs if align else [r[:600] for r in refs]
    eng.set_scores(None)
    eng.load(queries, 0)
    eng.load(refs, 1)
    ny = len(refs)
    edge = (1 << 24 if align else 1 << 27) // ny
    assert nx > edge
    got = eng.best_rows_k(0, nx, 0, ny, 64, 0, align)
    for lo, hi in ((0, 40), (edge - 40, min(nx, edge + 40)), (nx - 20, nx)):
        full = reference(eng, align, lo, hi - lo, 0, ny)
        part = {key: got[key][lo:hi] for key in ("index", "metrics", "counts")}
        assert_same(part, select_k(full["metrics"], full["counts"], 64, 0), (lo, hi))


@pytest.mark.parametrize("align", [True, False], ids=["align", "free"])
def test_multi_engine_column_tiles_equal_one_call(eng, align):
    """Two contexts on device 0, row and column tiles merged on the host (combine_best_k)."""
    from taxi2_b200.multi import MultiEngine

    queries, refs = small_sets(align)
    eng.set_scores(None)
    eng.load(queries, 0)
    eng.load(refs, 1)
    with MultiEngine([0, 0]) as multi:
        multi.load(queries, 0)
        multi.load(refs, 1)
        for metric, k in ((0, 10), (3, 64), (1, 1)):
            want = eng.best_rows_k(0, len(queries), 0, len(refs), k, metric, align)
            for rows, col_tiles in ((None, 1), (9, 3), (61, 5), (4, 64)):
                got = multi.best_matches_k(k, metric, align, rows_per_tile=rows, col_tiles=col_tiles)
                assert_same(got, (want["index"], want["metrics"], want["counts"]), (metric, k, rows, col_tiles))
