"""combine_labels, the host merge of MultiEngine.clusters_within, against scipy's connected
components of the union of both labelings' groups: empty, identity, one component and random
canonical labelings, several rows at once, any merge order, canonical output."""
from __future__ import annotations

import itertools

import numpy as np
import pytest
from scipy.sparse import coo_matrix
from scipy.sparse.csgraph import connected_components

from taxi2_b200.multi import combine_labels


def canonical(groups: np.ndarray) -> np.ndarray:
    """Any group ids of n nodes -> the smallest member index of every node's group."""
    groups = np.asarray(groups)
    first = {}
    for i, g in enumerate(groups.tolist()):
        first.setdefault(g, i)
    return np.array([first[g] for g in groups.tolist()], dtype=np.int32)


def random_labeling(rng, n: int, k: int) -> np.ndarray:
    return canonical(rng.integers(0, max(k, 1), size=n))


def reference(*labelings: np.ndarray) -> np.ndarray:
    """Components of the graph with an edge from every node to its label in every labeling."""
    n = len(labelings[0])
    rows = np.concatenate([np.arange(n)] * len(labelings))
    cols = np.concatenate(labelings).astype(np.int64)
    graph = coo_matrix((np.ones(len(rows), dtype=np.int8), (rows, cols)), shape=(n, n))
    _, comp = connected_components(graph, directed=False)
    return canonical(comp)


def is_canonical(lab: np.ndarray) -> bool:
    idx = np.arange(lab.shape[-1])
    return bool((lab <= idx).all() and (np.take_along_axis(lab, lab.astype(np.int64), axis=-1) == lab).all())


def test_empty():
    out = combine_labels(np.zeros((3, 0), np.int32), np.zeros((3, 0), np.int32))
    assert out.shape == (3, 0) and out.dtype == np.int32
    assert combine_labels(np.zeros(0, np.int32), np.zeros(0, np.int32)).shape == (0,)


def test_identity_and_one_component():
    n = 50
    ident = np.arange(n, dtype=np.int32)
    one = np.zeros(n, dtype=np.int32)
    rng = np.random.default_rng(1)
    lab = random_labeling(rng, n, 7)
    assert np.array_equal(combine_labels(ident, ident), ident)
    assert np.array_equal(combine_labels(ident, lab), lab)
    assert np.array_equal(combine_labels(lab, ident), lab)
    assert np.array_equal(combine_labels(one, lab), one)
    assert np.array_equal(combine_labels(lab, one), one)


@pytest.mark.parametrize("n,k", [(1, 1), (2, 1), (17, 5), (200, 150), (1000, 600), (1000, 30), (3000, 2900)])
def test_random_against_scipy(n, k):
    rng = np.random.default_rng(n * 7 + k)
    for _ in range(5):
        a, b = random_labeling(rng, n, k), random_labeling(rng, n, k)
        out = combine_labels(a, b)
        assert out.dtype == np.int32 and out.shape == (n,)
        assert np.array_equal(out, reference(a, b))
        assert is_canonical(out)


def test_long_chain():
    """Groups of two that overlap by one node across the labelings: one component through n nodes."""
    n = 4001
    a = np.arange(n, dtype=np.int32)
    a[1::2] -= 1                         # {0,1} {2,3} ...
    b = np.arange(n, dtype=np.int32)
    b[2::2] -= 1                         # {0} {1,2} {3,4} ...
    assert np.array_equal(combine_labels(a, b), np.zeros(n, dtype=np.int32))
    # the same from the top end: labels are the minimum, wherever the chain starts
    rev = np.arange(n)[::-1]
    lab_a = canonical(a[rev]); lab_b = canonical(b[rev])
    assert np.array_equal(combine_labels(lab_a, lab_b), np.zeros(n, dtype=np.int32))


def test_rows_are_independent():
    """(m, n) labelings: every threshold row merges on its own."""
    rng = np.random.default_rng(5)
    m, n = 8, 300
    a = np.stack([random_labeling(rng, n, k) for k in (1, 3, 30, 100, 200, 290, 299, 300)])
    b = np.stack([random_labeling(rng, n, k) for k in (300, 250, 150, 80, 40, 10, 2, 1)])
    out = combine_labels(a, b)
    assert out.shape == (m, n) and out.dtype == np.int32
    for t in range(m):
        assert np.array_equal(out[t], reference(a[t], b[t])), t
        assert np.array_equal(out[t], combine_labels(a[t], b[t])), t


def test_any_merge_order():
    rng = np.random.default_rng(9)
    n = 400
    labs = [random_labeling(rng, n, k) for k in (350, 300, 380, 390)]
    want = reference(*labs)
    for order in itertools.permutations(range(len(labs))):
        acc = labs[order[0]]
        for k in order[1:]:
            acc = combine_labels(acc, labs[k])
        assert np.array_equal(acc, want), order
    # commutative and associative
    a, b, c = labs[:3]
    assert np.array_equal(combine_labels(a, b), combine_labels(b, a))
    assert np.array_equal(combine_labels(combine_labels(a, b), c), combine_labels(a, combine_labels(b, c)))


def test_shape_mismatch_is_refused():
    with pytest.raises(ValueError):
        combine_labels(np.zeros(3, np.int32), np.zeros(4, np.int32))
