"""Host-side merge of per-column-tile k-closest lists (multi.combine_best_k) on CPU: against a
numpy restatement of the selection over the whole row (np.lexsort on (column, value), NaN removed),
for every arrival order of the tiles."""
from __future__ import annotations

import itertools

import numpy as np
import pytest

from taxi2_b200.multi import combine_best_k


def select_k(d: np.ndarray, counts: np.ndarray, lo: int, hi: int, k: int, metric: int):
    """The k smallest (value, column) keys of columns lo..hi of every row, as the device lists them."""
    nx = d.shape[0]
    index = np.full((nx, k), -1, dtype=np.int32)
    best = np.full((nx, k, 4), np.nan)
    cnt = np.zeros((nx, k, 4), dtype=np.int32)
    for i in range(nx):
        cols = np.arange(lo, hi)
        vals = d[i, lo:hi, metric]
        ok = ~np.isnan(vals)
        cols, vals = cols[ok], vals[ok]
        win = cols[np.lexsort((cols, vals))][:k]
        index[i, :len(win)] = win
        best[i, :len(win)] = d[i, win]
        cnt[i, :len(win)] = counts[i, win]
    return index, best, cnt


def matrix(seed: int, nx: int, ny: int, levels: int, nan_share: float):
    rng = np.random.default_rng(seed)
    d = rng.integers(0, levels, (nx, ny, 4)).astype(np.float64) / levels
    d[rng.random((nx, ny)) < nan_share] = np.nan
    d[:3] = np.nan                                                  # rows without a defined value
    d[3:6, 2:] = np.nan                                             # rows with two defined values
    counts = rng.integers(0, 1000, (nx, ny, 4)).astype(np.int32)
    return d, counts


@pytest.mark.parametrize("k", [1, 2, 5, 10, 64])
@pytest.mark.parametrize("levels,nan_share", [(3, 0.2), (40, 0.0), (2, 0.7)])
def test_tiles_merged_in_every_order_equal_one_selection(k, levels, nan_share):
    nx, ny, metric = 60, 41, 1
    d, counts = matrix(k * 100 + levels, nx, ny, levels, nan_share)
    want = select_k(d, counts, 0, ny, k, metric)
    bounds = [0, 7, 8, 23, 41]
    tiles = [select_k(d, counts, bounds[t], bounds[t + 1], k, metric) for t in range(4)]
    for order in itertools.permutations(range(4)):
        index = np.full((nx, k), -1, dtype=np.int32)
        best = np.full((nx, k, 4), np.nan)
        cnt = np.zeros((nx, k, 4), dtype=np.int32)
        for t in order:
            combine_best_k(index, best, cnt, *tiles[t], metric)
        assert np.array_equal(index, want[0]), order
        assert np.array_equal(best, want[1], equal_nan=True), order
        assert np.array_equal(cnt, want[2]), order


def test_undefined_slots_never_displace_defined_ones():
    index = np.array([[4, -1, -1]], dtype=np.int32)
    best = np.full((1, 3, 4), np.nan)
    best[0, 0] = np.inf                                             # a defined value above every finite one
    cnt = np.zeros((1, 3, 4), dtype=np.int32)
    cnt[0, 0] = 7
    new_index = np.array([[-1, -1, -1]], dtype=np.int32)
    combine_best_k(index, best, cnt, new_index, np.full((1, 3, 4), np.nan), np.zeros((1, 3, 4), dtype=np.int32), 0)
    assert index.tolist() == [[4, -1, -1]] and best[0, 0, 0] == np.inf and (cnt[0, 0] == 7).all()
    new_index = np.array([[9, 2, -1]], dtype=np.int32)
    new_best = np.full((1, 3, 4), np.nan)
    new_best[0, :2, 0] = [0.5, np.inf]
    combine_best_k(index, best, cnt, new_index, new_best, np.ones((1, 3, 4), dtype=np.int32), 0)
    assert index.tolist() == [[9, 2, 4]]                          # equal +inf values: the smaller column first
    assert (cnt[0, 2] == 7).all() and (cnt[0, :2] == 1).all()


def test_merge_of_equal_values_keeps_the_smaller_columns():
    """Duplicated references tie exactly: whichever tile arrives first, the smallest columns win."""
    nx, k = 4, 3
    d = np.zeros((nx, 10, 4))
    counts = np.arange(nx * 10 * 4, dtype=np.int32).reshape(nx, 10, 4)
    for order in ([1, 0], [0, 1]):
        index = np.full((nx, k), -1, dtype=np.int32)
        best = np.full((nx, k, 4), np.nan)
        cnt = np.zeros((nx, k, 4), dtype=np.int32)
        parts = [select_k(d, counts, 0, 5, k, 0), select_k(d, counts, 5, 10, k, 0)]
        for t in order:
            combine_best_k(index, best, cnt, *parts[t], 0)
        assert (index == [0, 1, 2]).all()
        assert np.array_equal(cnt, counts[:, :3])
