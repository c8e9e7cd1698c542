"""CPU side of tests/test_gpu_metric_arithmetic.py: the oracle's batch metrics, the ulp and exact-value
helpers of metric_ref.py, and the table-form bound replayed on the CPU (a table rounded from long double
meets it, one rounded from double does not)."""
from __future__ import annotations

import math

import numpy as np

import metric_ref as M
import oracle


def test_batch_metrics_equal_the_per_tuple_oracle():
    rng = np.random.default_rng(1)
    counts = np.concatenate([M.every_tuple(12), M.edges([1, 2, 3, 4, 5, 400, 2048, 2049]),
                             M.random_tuples(rng, 3000, 2**20), np.zeros((1, 4), np.int32)])
    got = oracle.metrics_batch(counts)
    want = np.array([oracle.metrics(c) for c in counts])
    assert np.array_equal(got.view(np.uint64), want.view(np.uint64))
    assert np.isnan(got).any() and not np.isnan(got).all()


def test_ulp_distance():
    x = np.array([1.0, 0.5, 1e-300, 3.0, 0.0, 2.0**-1074])
    assert (M.ulp_distance(x, x) == 0).all()
    assert (M.ulp_distance(np.nextafter(x, np.inf), x) == 1).all()
    assert (M.ulp_distance(x, np.nextafter(x, -np.inf)) == 1).all()
    assert M.ulp_distance(np.array([-0.0]), np.array([0.0]))[0] == 0
    assert M.ulp_distance(np.array([-(2.0**-1074)]), np.array([2.0**-1074]))[0] == 2
    assert M.ulp_distance(np.array([1.0]), np.array([1.0 + 5 * 2.0**-52]))[0] == 5
    assert M.ulp_distance(np.array([1.0]), np.array([1.0 - 5 * 2.0**-53]))[0] == 5


def test_log_ulp_error():
    """glibc's log is within 1 ulp; one step away from it is about 1 ulp more."""
    rng = np.random.default_rng(3)
    x = np.concatenate([rng.random(300) + 1e-300, np.exp(rng.uniform(-700, 700, 300)), [2.0, 0.5, 1.0 + 2.0**-52]])
    for a in x:
        e = M.log_ulp_error(float(a), float(np.log(a)))
        assert e < 1.0
        assert abs(M.log_ulp_error(float(a), float(np.nextafter(np.log(a), np.inf))) - 1.0) <= e + 1e-9
    assert M.log_ulp_error(1.0, 0.0) == 0.0 and M.log_ulp_error(1.0, 1e-300) == math.inf
    # ln 2 rounded up by one ulp of ln 2: the error is one ulp less the rounding error of ln 2
    ln2 = math.log(2.0)
    err = M.log_ulp_error(2.0, math.nextafter(ln2, 1.0))
    assert abs(err + M.log_ulp_error(2.0, ln2) - 1.0) < 1e-9 or abs(err - M.log_ulp_error(2.0, ln2) - 1.0) < 1e-9


def test_edge_families():
    n = 2048
    t = M.edges([n]).astype(np.int64)
    assert (t[:, :3].sum(axis=1) == n).all() and (t >= 0).all()
    d = t[:, 1] + t[:, 2]
    assert set(range(4)) <= set(d.tolist())
    assert {4, 8} <= set((3 * n - 4 * d).tolist())           # 3n - A divisible by 4 for A = 4, 8 at n = 2048
    assert set(range(4)) <= set((n - 2 * t[:, 1] - t[:, 2]).tolist())
    assert {0, 2} <= set((n - 2 * t[:, 2]).tolist())
    assert set(M.edges([2047])[:, :3].sum(axis=1).tolist()) == {2047}
    assert len(M.every_tuple(400)) == sum((k + 1) * (k + 2) // 2 for k in range(401))
    assert len(np.unique(M.every_tuple(30), axis=0)) == len(M.every_tuple(30))
    assert 1900 in M.edge_lengths() and 2**20 in M.edge_lengths() and (M.edge_lengths() <= 2**20).all()


def replay_table(counts, long_double: bool) -> tuple[np.ndarray, np.ndarray]:
    """JC / K2P of metrics_from_counts_table (common.cuh) on the CPU, with the table of taxi_ctx_create
    rounded from long double or, wrongly, from double."""
    k = np.arange(1, 3 * M.LN_TABLE_COLS + 1)
    ln = np.log(k.astype(np.longdouble)) * np.longdouble(2) ** 58 if long_double else np.log(k.astype(np.float64)) * 2.0**58
    tab = np.concatenate([[0], np.rint(ln).astype(np.int64)])
    c = counts.astype(np.int64)
    n, ts, tv = c[:, :3].sum(axis=1), c[:, 1], c[:, 2]
    A, a, b = 3 * n - 4 * (ts + tv), n - 2 * ts - tv, n - 2 * tv
    jc = (tab[A] - tab[3 * n]).astype(np.float64) * (-0.75 * 2.0**-58) + 0.0
    k2p = (2 * tab[a] + tab[b] - 3 * tab[n]).astype(np.float64) * (-0.25 * 2.0**-58) + 0.0
    return jc, k2p


def test_table_bound_on_a_cpu_replay():
    """The bound of test_table_form_against_exact_logarithms, |got - exact| <= 1.5 * 2^-58 + 2 ulp(exact),
    holds for the table as built and fails for one built from the double log."""
    counts = np.concatenate([M.edges(M.edge_lengths()[M.edge_lengths() <= M.LN_TABLE_COLS]),
                             M.random_tuples(np.random.default_rng(9), 20_000, M.LN_TABLE_COLS)]).astype(np.int64)
    n, ts, tv = counts[:, :3].sum(axis=1), counts[:, 1], counts[:, 2]
    counts = counts[(3 * n - 4 * (ts + tv) > 0) & (n - 2 * ts - tv > 0) & (n - 2 * tv > 0)]
    exact = M.table_exact(counts)
    for long_double, fits in ((True, True), (False, False)):
        over = 0
        for got, ex in zip(replay_table(counts, long_double), exact):
            e58, _ = M.table_error(got, ex)
            ulp = np.array([math.ulp(x / 2 ** (M.FRAC + 2)) for x in ex])
            over += int((e58 * 2.0**-58 > 1.5 * 2.0**-58 + 2 * ulp).sum())
        assert (over == 0) == fits, (long_double, over)
