"""Host-side assembly of per-tile CSR pieces of pairs within a threshold (multi.combine_within) on
CPU: against a numpy restatement of the selection over the whole matrix (row-major, ascending
column within a row), with random tiles including empty ones, in every arrival order; and the C
ABI declares and binds both new entry points."""
from __future__ import annotations

import itertools
import re
from pathlib import Path

import numpy as np
import pytest

from taxi2_b200.multi import combine_within

HEADER = Path(__file__).resolve().parent.parent / "include" / "taxi2_b200.h"


def select(d: np.ndarray, counts: np.ndarray, x0: int, nx: int, y0: int, ny: int, t: float, metric: int, scale: float = 1.0):
    """The CSR of rows x0..x0+nx over columns y0..y0+ny: v not NaN and v * scale <= t, row-major."""
    v = d[x0:x0 + nx, y0:y0 + ny, metric]
    with np.errstate(invalid="ignore"):
        keep = ~np.isnan(v) & (v * scale <= t)
    rows, cols = np.nonzero(keep)             # row-major, ascending column within a row
    row_ptr = np.zeros(nx + 1, dtype=np.int64)
    np.cumsum(keep.sum(axis=1), out=row_ptr[1:])
    return dict(row_ptr=row_ptr, index=(cols + y0).astype(np.int32),
                metrics=d[x0 + rows, y0 + cols], counts=counts[x0 + rows, y0 + cols])


def matrix(seed: int, nx: int, ny: int, levels: int, nan_share: float):
    rng = np.random.default_rng(seed)
    d = rng.integers(0, levels, (nx, ny, 4)).astype(np.float64) / levels
    d[rng.random((nx, ny)) < nan_share] = np.nan
    d[:2] = np.nan                                                  # rows without a defined value
    counts = rng.integers(0, 1000, (nx, ny, 4)).astype(np.int32)
    return d, counts


def assert_same(got: dict, want: dict, what=None):
    assert np.array_equal(got["row_ptr"], want["row_ptr"]), what
    assert np.array_equal(got["index"], want["index"]), what
    assert np.array_equal(got["metrics"].view(np.uint64), want["metrics"].view(np.uint64)), what
    assert np.array_equal(got["counts"], want["counts"]), what


@pytest.mark.parametrize("t", [0.0, 0.3, 0.5, np.inf, -1.0])
@pytest.mark.parametrize("levels,nan_share", [(3, 0.2), (40, 0.0), (2, 0.7)])
def test_tiles_in_every_order_equal_one_selection(t, levels, nan_share):
    nx, ny, metric = 23, 37, 2
    d, counts = matrix(levels * 7 + int(10 * nan_share), nx, ny, levels, nan_share)
    want = select(d, counts, 0, nx, 0, ny, t, metric)
    # irregular tiles: two row bands with different column cuts (one a single column) and a tile without rows
    rects = [(0, 9, 0, 11), (0, 9, 11, 1), (0, 9, 12, 25), (9, 14, 0, 20), (9, 14, 20, 17), (5, 0, 3, 4)]
    tiles = [(x0, n, y0, select(d, counts, x0, n, y0, m, t, metric)) for x0, n, y0, m in rects]
    for order in itertools.permutations(range(len(tiles))):
        got = combine_within([tiles[k] for k in order], nx)
        assert_same(got, want, order)


@pytest.mark.parametrize("seed", range(6))
def test_random_grids_and_scale(seed):
    """Random row and column cuts (a tile may select nothing), tiles shuffled, scale = 100."""
    rng = np.random.default_rng(seed)
    nx, ny = int(rng.integers(1, 40)), int(rng.integers(1, 60))
    d, counts = matrix(100 + seed, nx, ny, 20, 0.1)
    t = float(rng.choice([0.0, 5.0, 35.0, 100.0]))
    want = select(d, counts, 0, nx, 0, ny, t, 0, 100.0)
    xs = np.unique(np.concatenate([[0, nx], rng.integers(0, nx + 1, 3)]))
    ys = np.unique(np.concatenate([[0, ny], rng.integers(0, ny + 1, 4)]))
    tiles = [(int(a), int(b - a), int(c), select(d, counts, a, b - a, c, e - c, t, 0, 100.0))
             for a, b in zip(xs[:-1], xs[1:]) for c, e in zip(ys[:-1], ys[1:])]
    for _ in range(20):
        rng.shuffle(tiles)
        assert_same(combine_within(tiles, nx), want, seed)


def test_full_width_tiles_are_copied_whole():
    d, counts = matrix(5, 30, 12, 5, 0.1)
    want = select(d, counts, 0, 30, 0, 12, 0.4, 1)
    tiles = [(x0, 10, 0, select(d, counts, x0, 10, 0, 12, 0.4, 1)) for x0 in (20, 0, 10)]
    assert_same(combine_within(tiles, 30), want)


def test_nothing_selected():
    d, counts = matrix(6, 8, 9, 4, 0.0)
    tiles = [(0, 8, 0, select(d, counts, 0, 8, 0, 4, -1.0, 0)), (0, 8, 4, select(d, counts, 0, 8, 4, 5, -1.0, 0))]
    got = combine_within(tiles, 8)
    assert (got["row_ptr"] == 0).all() and got["index"].shape == (0,) and got["metrics"].shape == (0, 4)
    assert got["counts"].shape == (0, 4)


def test_abi_declares_and_binds_pairs_within():
    from taxi2_b200 import _native

    text = re.sub(r"/\*.*?\*/", "", HEADER.read_text(), flags=re.S)
    for name in ("taxi_pairs_within", "taxi_pairs_within_fetch"):
        assert re.search(rf"\bint {name}\s*\(", text), name
        assert name in _native.SIGNATURES, name
    lib = _native.load()
    assert hasattr(lib, "taxi_pairs_within") and hasattr(lib, "taxi_pairs_within_fetch")
