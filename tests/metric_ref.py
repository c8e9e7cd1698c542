"""Exact references for the metric arithmetic: ulp distances on bit patterns, the error of a logarithm
against its value at 160 bits, the exact JC / K2P of the table form, and the count-tuple families at
the edges of the formulas (tests/test_gpu_metric_arithmetic.py, tests/test_metric_arithmetic_host.py)."""
from __future__ import annotations

import math

import numpy as np
from mpmath import mp

FRAC = 128                 # fractional bits of the exact logarithms below (the device table has 58)
LN_TABLE_COLS = 2048       # common.cuh: rows of at most this many compared columns take the table form


def ordered(x: np.ndarray) -> np.ndarray:
    """float64 -> int64 keys in the order of the values, one step per representable double
    (-0.0 and +0.0 share key 0)."""
    k = np.ascontiguousarray(x, dtype=np.float64).view(np.int64)
    return np.where(k < 0, -(k & np.int64(0x7FFFFFFFFFFFFFFF)), k)


def ulp_distance(got: np.ndarray, want: np.ndarray) -> np.ndarray:
    """Number of representable doubles between got and want (finite inputs)."""
    return np.abs(ordered(got) - ordered(want))


def log_ulp_error(x: float, got: float) -> float:
    """|got - ln x| / ulp(ln x), with ln x evaluated at 160 bits; 0 or inf at x = 1 (ln x = 0)."""
    with mp.workprec(160):
        exact = mp.log(mp.mpf(x))
        if exact == 0:
            return 0.0 if got == 0.0 else math.inf
        _, e = mp.frexp(exact)          # |exact| in [2^(e-1), 2^e): ulp = 2^(e-53)
        return float(abs(mp.mpf(got) - exact) / mp.ldexp(1, e - 53))


_LN = []


def ln_fixed(k: np.ndarray) -> list[int]:
    """round(ln k * 2^FRAC) for 1 <= k <= 3 LN_TABLE_COLS, exact integers."""
    if not _LN:
        with mp.workprec(FRAC + 64):
            _LN.extend([0] + [int(mp.nint(mp.ldexp(mp.log(i), FRAC))) for i in range(1, 3 * LN_TABLE_COLS + 1)])
    return [_LN[int(i)] for i in k]


def table_exact(counts: np.ndarray) -> tuple[list[int], list[int]]:
    """Exact -3/4 ln(A / 3n) and -1/4 ln(a^2 b / n^3) of (same, ts, tv, gap) tuples with n <= LN_TABLE_COLS,
    A = 3n - 4d, a = n - 2ts - tv, b = n - 2tv, all positive, as integers in units of 2^-(FRAC + 2)
    (the factor 4 keeps the quarters exact; the table error below 2^-FRAC does not matter here)."""
    c = np.asarray(counts, dtype=np.int64)
    n, ts, tv = c[:, :3].sum(axis=1), c[:, 1], c[:, 2]
    A, a, b = 3 * n - 4 * (ts + tv), n - 2 * ts - tv, n - 2 * tv
    assert (n <= LN_TABLE_COLS).all() and (A > 0).all() and (a > 0).all() and (b > 0).all()
    lA, l3n, la, lb, ln = (ln_fixed(v) for v in (A, 3 * n, a, b, n))
    jc = [-3 * (x - y) for x, y in zip(lA, l3n)]
    k2p = [-(2 * x + y - 3 * z) for x, y, z in zip(la, lb, ln)]
    return jc, k2p


def table_error(got: np.ndarray, exact: list[int]) -> tuple[np.ndarray, np.ndarray]:
    """-> (|got - exact| in units of 2^-58, the same in ulp(exact)), exact from table_exact."""
    scale = FRAC + 2
    err58, errulp = np.empty(len(exact)), np.empty(len(exact))
    for i, (g, x) in enumerate(zip(got.tolist(), exact)):
        gi = math.ldexp(g, scale)
        assert gi == int(gi), g          # got is a multiple of 2^-(FRAC + 2): the difference below is exact
        diff = abs(int(gi) - x)
        err58[i] = diff / 2 ** (scale - 58)
        xf = x / 2**scale                # correctly rounded
        errulp[i] = diff / 2**scale / math.ulp(xf) if xf != 0.0 else (0.0 if diff == 0 else math.inf)
    return err58, errulp


# -- count tuples --------------------------------------------------------------------------------------

def every_tuple(n_max: int) -> np.ndarray:
    """Every (same, ts, tv, 0) with same + ts + tv <= n_max, n = 0 included."""
    out = []
    for n in range(n_max + 1):
        d, tv = np.tril_indices(n + 1)     # every 0 <= tv <= d <= n
        ts = d - tv
        out.append(np.stack([n - ts - tv, ts, tv, np.zeros_like(ts)], axis=1))
    return np.concatenate(out).astype(np.int32)


def edge_lengths() -> np.ndarray:
    """n of the edge families: bands of +-4 around 48 log-spaced lengths up to 2^20, +-2 around every
    power of two, and every n from 1 900 to 2 100 (around the table's 2 048 columns)."""
    c = np.unique(np.round(np.geomspace(4, 2**20, 48)).astype(np.int64))
    n = [c + k for k in range(-4, 5)] + [2 ** np.arange(1, 21) + k for k in range(-2, 3)] + [np.arange(1900, 2101)]
    n = np.unique(np.concatenate(n))
    return n[(n >= 1) & (n <= 2**20)]


def edge_tuples(lengths) -> np.ndarray:
    """(same, ts, tv, gap) at the edges of the formulas for every n in `lengths`:
    d = ts + tv in {0 .. 3} with every ts / tv split; A = 3n - 4d in {1 .. 8} (next to the JC singularity);
    a = n - 2ts - tv in {0 .. 3} (a = 0: the floating-point fallback of the table form); b = n - 2tv in {0 .. 3}."""
    for n in map(int, lengths):
        rows = []
        for d in range(4):
            rows += [(ts, d - ts) for ts in range(d + 1)]
        for A in range(1, 9):
            if (3 * n - A) % 4 == 0 and 0 <= (d := (3 * n - A) // 4) <= n:
                rows += [(ts, d - ts) for ts in {0, 1, d // 2, d - 1, d} if 0 <= ts <= d]
        for a in range(4):
            for tv in {0, 1, 2, 3, (n - a) // 3, n - a - 2, n - a - 1, n - a}:
                if 0 <= tv and (n - a - tv) % 2 == 0 and 0 <= (ts := (n - a - tv) // 2) and ts + tv <= n:
                    rows.append((ts, tv))
        for b in range(4):
            if (n - b) % 2 == 0 and 0 <= (tv := (n - b) // 2) <= n:
                rows += [(ts, tv) for ts in {0, 1, 2, (n - tv) // 2, n - tv} if 0 <= ts <= n - tv]
        yield from ((n - ts - tv, ts, tv) for ts, tv in rows)


def edges(lengths, gaps=(0, 1, 7)) -> np.ndarray:
    """edge_tuples as int32 (n, 4) count tuples, gap counts cycling through `gaps`."""
    t = np.unique(np.array(list(edge_tuples(lengths)), dtype=np.int64), axis=0)
    g = np.resize(np.asarray(gaps, dtype=np.int64), len(t))
    return np.concatenate([t, g[:, None]], axis=1).astype(np.int32)


def random_tuples(rng, count: int, n_max: int) -> np.ndarray:
    """count tuples, n log-uniform in [1, n_max], ts and tv uniform in what is left, gaps up to n / 4."""
    n = np.exp(rng.uniform(0.0, np.log(n_max + 1), count)).astype(np.int64).clip(1, n_max)
    ts = (rng.random(count) * (n + 1)).astype(np.int64)
    tv = (rng.random(count) * (n - ts + 1)).astype(np.int64)
    g = (rng.random(count) * (n // 4 + 1)).astype(np.int64)
    return np.stack([n - ts - tv, ts, tv, g], axis=1).astype(np.int32)
