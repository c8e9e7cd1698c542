"""The metric arithmetic to the last bit.

Every kernel ends in the hand-written fp64 epilogue of common.cuh.  Its primitives are checked here on
the device against the IEEE operations they replace -- through tests/metric_primitives.cu, built by
`__graft_entry__.build()` with the library's code-generation flags -- and both forms of the epilogue are
checked through `taxi_metrics_from_counts`:

* `div_by(a, b, rcp_full(b))` is bit for bit `a / b` for every 0 <= a <= b <= 65 536 and in bands at each
  power of two up to 2^22; `1 - div_by(4p, 3, 1/3)` is bit for bit `1 - 4p/3` for every such p = a / b;
  `sqrt_pos` is bit for bit `sqrt` on every 1 - 2 (tv / n) with n <= 65 536 and on random normals >= 2^-970;
  `count_to_double` is exact on all of [0, 2^31); `log_pos` is within 1 ulp of ln x at 160 bits.
* Floating-point form: p and p-gaps bit for bit the oracle's, JC and K2P within 2 ulp of the oracle's
  libm formula, the oracle's NaN pattern, never -0.0.  The 2 ulp: the argument u (or v) of both sides is
  the same double, since the divisions and the square root are correctly rounded on both; what differs is
  log_pos against glibc's log, each within 1 ulp of ln, so the two logarithms lie within 2 ulp of each other
  and the exact multiply by -0.75 or -0.5 (one rounding on each side, of the same kind) keeps them there.
* Table form (rows of at most 2 048 columns): see test_table_form_against_exact_logarithms.

The worst values measured are printed (pytest -s)."""
from __future__ import annotations

import ctypes as C
import math
from pathlib import Path

import numpy as np
import pytest

import metric_ref as M
import oracle

pytestmark = pytest.mark.gpu

HARNESS = Path(__file__).resolve().parent / "bin" / "libmetric_primitives.so"
FP_ULP = 2                 # JC / K2P of the floating-point form against the oracle (module docstring)
TABLE_REL = 1.4e-13        # table form against the oracle (common.cuh: metrics_from_counts_table)


@pytest.fixture(scope="module")
def prim():
    if not HARNESS.exists():
        pytest.fail(f"{HARNESS} is missing: run `python -c 'import __graft_entry__ as g; g.build()'`")
    lib = C.CDLL(str(HARNESS))
    ull, f64 = C.POINTER(C.c_ulonglong), C.POINTER(C.c_double)
    for name, args in (("mp_div_sweep", [C.c_int, ull, f64]), ("mp_sqrt_sweep", [C.c_int, ull, f64]),
                       ("mp_count_sweep", [ull, f64]), ("mp_apply", [C.c_int, f64, f64, f64, C.c_longlong])):
        getattr(lib, name).argtypes = args
        getattr(lib, name).restype = C.c_int
    return lib


@pytest.fixture(scope="module")
def engine():
    from taxi2_b200.engine import Engine

    eng = Engine(0)
    eng.load([b"ACGT"], 0)          # a context takes count tuples once it holds a sequence set
    yield eng
    eng.close()


def sweep(fn, *args):
    """-> (mismatch count of each check, first offending inputs of each check)."""
    count, first = (C.c_ulonglong * 2)(), (C.c_double * 32)()
    rc = fn(*args, count, first)
    assert rc == 0, f"CUDA error {rc}"
    first = np.array(first).reshape(2, 8, 2)
    return list(count), [first[c][: min(count[c], 8)].tolist() for c in range(2)]


def apply(prim, op: int, a, b=None) -> np.ndarray:
    a = np.ascontiguousarray(a, dtype=np.float64)
    b = None if b is None else np.ascontiguousarray(b, dtype=np.float64)
    out = np.empty_like(a)
    ptr = lambda x: None if x is None else x.ctypes.data_as(C.POINTER(C.c_double))  # noqa: E731
    assert prim.mp_apply(op, ptr(a), ptr(b), ptr(out), len(a)) == 0
    return out


def mismatches(got: np.ndarray, want: np.ndarray) -> np.ndarray:
    return np.flatnonzero(got.view(np.uint64) != want.view(np.uint64))


# -- the primitives ------------------------------------------------------------------------------------

def test_division_every_small_ratio(prim):
    """div_by(a, b, rcp_full(b)) == a / b and 1 - div_by(4p, 3, 1/3) == 1 - 4p/3 (p = a / b), bit for bit,
    for every 0 <= a <= b <= 65 536 (2.1e9 quotients)."""
    count, first = sweep(prim.mp_div_sweep, 65536)
    print(f"\ndivision sweep: {count[0]} quotients and {count[1]} values of u off the IEEE result")
    assert count == [0, 0], first


def test_division_at_powers_of_two(prim):
    """Divisors in bands of +-64 around every power of two up to 2^22 (n + g of the longest pairs), with
    dividends 0, 1, b - 1, b and 60 random ones."""
    rng = np.random.default_rng(22)
    b = np.unique(np.concatenate([2**k + np.arange(-64, 65) for k in range(1, 23)]))
    b = b[b >= 1]
    a = np.concatenate([np.stack([0 * b, 0 * b + 1, b - 1, b], axis=1), (rng.random((len(b), 60)) * (b[:, None] + 1)).astype(np.int64)], axis=1)
    bb = np.repeat(b, a.shape[1]).astype(np.float64)
    a = a.ravel().astype(np.float64)
    bad = mismatches(apply(prim, 0, a, bb), a / bb)
    assert len(bad) == 0, list(zip(a[bad][:8], bb[bad][:8]))
    p = a / bb
    bad = mismatches(apply(prim, 1, p), 1.0 - 4.0 * p / 3.0)
    assert len(bad) == 0, list(zip(a[bad][:8], bb[bad][:8]))


def test_square_root(prim):
    """sqrt_pos(b) == sqrt(b) bit for bit for every b = 1 - 2 (tv / n) > 0 with n <= 65 536 (1.1e9 values),
    formed as metrics_from_counts forms it, and for 10^6 random normals over the whole exponent range from
    2^-970 up.  Below 2^-970 the residual b - g^2 of the final correction is no longer a representable
    double and the result may be 1 ulp off (no metric argument comes near: b >= 1 / n > 2^-31)."""
    count, first = sweep(prim.mp_sqrt_sweep, 65536)
    print(f"\nsquare-root sweep: {count[0]} values off the IEEE result")
    assert count[0] == 0, first[0]
    rng = np.random.default_rng(2)
    bits = (rng.integers(1, 2047, 10**6, dtype=np.uint64) << np.uint64(52)) | rng.integers(0, 2**52, 10**6, dtype=np.uint64)
    x = bits.view(np.float64)
    got, want = apply(prim, 2, x), np.sqrt(x)
    exact = x >= 2.0**-970
    bad = mismatches(got[exact], want[exact])
    assert len(bad) == 0, x[exact][bad][:8].tolist()
    assert M.ulp_distance(got[~exact], want[~exact]).max() <= 1


def test_count_to_double(prim):
    count, first = sweep(prim.mp_count_sweep)
    print(f"\ncount_to_double: {count[0]} of 2^31 counts off (double)k")
    assert count[0] == 0, first[0]


def log_points(rng) -> np.ndarray:
    """About 3e5 arguments of log_pos: the u and (a sample of the) v of every tuple with n <= 400, 1 +- k ulp,
    +-2 000 ulp around the mantissa split of the reduction and around sqrt(2) and sqrt(2)/2, powers of two
    +- 3 ulp over every exponent, the smallest u next to the JC singularity and the rounding residues
    of the K2P argument at n = 2 ts + tv, and random normals."""
    c = M.every_tuple(400).astype(np.float64)
    n, ts, tv = c[:, :3].sum(axis=1), c[:, 1], c[:, 2]
    with np.errstate(divide="ignore", invalid="ignore"):
        p, P, Q = (ts + tv) / n, ts / n, tv / n
        u = 1.0 - 4.0 * p / 3.0
        a, b = 1.0 - 2.0 * P - Q, 1.0 - 2.0 * Q
        v = np.where((a > 0) & (b > 0), a * np.sqrt(np.maximum(b, 0.0)), -1.0)
    u, v = np.unique(u[u > 0]), np.unique(v[v > 0])
    pts = [u, rng.choice(v, 100_000, replace=False)]
    k = np.arange(1, 2001, dtype=np.float64)
    pts += [1.0 + k * 2.0**-52, 1.0 - k * 2.0**-53, [1.0]]
    split = np.array([0x3FF6A09C00000000, 0x3FE6A09C00000000], dtype=np.uint64).view(np.float64)   # hx + 0x95f64 carries into 2^20
    for centre in (*split, math.sqrt(2.0), math.sqrt(0.5)):
        pts.append(centre + np.arange(-2000, 2001) * math.ulp(centre))
    e = np.arange(-1022, 1024, dtype=np.float64)
    pw = np.ldexp(1.0, e.astype(np.int64))
    pts += [pw] + [pw + j * np.ldexp(1.0, (e - 52).astype(np.int64)) for j in (1, 2, 3)] \
        + [pw - j * np.ldexp(1.0, (e - 53).astype(np.int64)) for j in (1, 2, 3)]
    nn = np.unique(np.concatenate([M.edge_lengths(), rng.integers(1, 2**20 + 1, 4000)])).astype(np.float64)
    for A in range(1, 9):
        m = (3 * nn - A) % 4 == 0
        pd = (3 * nn[m] - A) / 4 / nn[m]
        pts.append(1.0 - 4.0 * pd / 3.0)
    r = M.edges(M.edge_lengths()).astype(np.float64)
    r = r[(r[:, 0] + r[:, 1] + r[:, 2] == 2 * r[:, 1] + r[:, 2]) & (r[:, 0] + r[:, 1] + r[:, 2] > 0)]
    rn = r[:, :3].sum(axis=1)
    ra, rb = 1.0 - 2.0 * (r[:, 1] / rn) - r[:, 2] / rn, 1.0 - 2.0 * (r[:, 2] / rn)
    ok = (ra > 0) & (rb > 0)
    pts.append(ra[ok] * np.sqrt(rb[ok]))
    bits = (rng.integers(1, 2047, 50_000, dtype=np.uint64) << np.uint64(52)) | rng.integers(0, 2**52, 50_000, dtype=np.uint64)
    pts += [bits.view(np.float64), rng.random(50_000)]
    x = np.unique(np.concatenate([np.asarray(q, dtype=np.float64) for q in pts]))
    return x[(x >= np.finfo(np.float64).tiny) & np.isfinite(x)]


def test_log_within_one_ulp(prim):
    """log_pos(x) against ln x at 160 bits: below 1 ulp everywhere (fdlibm's bound)."""
    x = log_points(np.random.default_rng(5))
    got = apply(prim, 3, x)
    err = np.array([M.log_ulp_error(a, g) for a, g in zip(x.tolist(), got.tolist())])
    i = int(np.argmax(err))
    print(f"\nlog_pos: {len(x)} arguments, worst error {err[i]:.4f} ulp at x = {x[i]!r}")
    assert len(x) > 250_000
    assert err[i] < 1.0, (x[i], got[i])


# -- both forms through taxi_metrics_from_counts ----------------------------------------------------------

def check_floating_point_form(engine, counts) -> list[int]:
    """-> worst ulp distance of JC and K2P from the oracle."""
    got = engine.metrics_from_counts(counts, table=False)
    want = oracle.metrics_batch(counts)
    assert np.array_equal(np.isnan(got), np.isnan(want))
    for col in (0, 1):
        bad = mismatches(got[:, col].copy(), want[:, col].copy())
        assert len(bad) == 0, (col, counts[bad][:8].tolist())
    assert not (got.view(np.uint64) == np.uint64(1 << 63)).any(), "-0.0"
    worst = []
    for col in (2, 3):
        ok = ~np.isnan(want[:, col])
        dist = M.ulp_distance(got[ok, col], want[ok, col])
        worst.append(int(dist.max(initial=0)))
        assert worst[-1] <= FP_ULP, (col, counts[ok][dist > FP_ULP][:8].tolist())
    return worst


def test_floating_point_form_every_small_tuple(engine):
    """Every (same, ts, tv) with n <= 400 (10.8 M tuples, gap 0), and every (n, d) with gap 1 and 7."""
    small = M.every_tuple(400)
    assert len(small) == 10_827_401
    worst = check_floating_point_form(engine, small)
    gapped = small[small[:, 1] == 0]
    for g in (1, 7):
        gapped[:, 3] = g
        check_floating_point_form(engine, gapped)
    print(f"\nfloating-point form, n <= 400: JC within {worst[0]} ulp, K2P within {worst[1]} ulp of the oracle")


def test_floating_point_form_edges_and_random(engine):
    """The edge families (d <= 3, A = 3n - 4d <= 8, a = n - 2ts - tv <= 3, b = n - 2tv <= 3) for n in bands up
    to 2^20 and every n from 1 900 to 2 100, and 2 M random tuples with log-uniform n up to 2^20."""
    edges = M.edges(M.edge_lengths())
    rand = M.random_tuples(np.random.default_rng(20), 2_000_000, 2**20)
    w_edges = check_floating_point_form(engine, edges)
    w_rand = check_floating_point_form(engine, rand)
    print(f"\nfloating-point form: edges JC {w_edges[0]} / K2P {w_edges[1]} ulp, random JC {w_rand[0]} / K2P {w_rand[1]} ulp")


def test_table_form_against_exact_logarithms(engine):
    """Table form (n <= 2 048) against the exact -3/4 ln(A / 3n) and -1/4 ln(a^2 b / n^3).

    Bound.  Each entry ln k * 2^58 of the table is rounded to an integer (error <= 1/2 unit of 2^-58) from
    logl (error ~2^-64 relative, ln k < 9: below 0.15 units): within 1 unit.  JC takes the difference of 2
    entries, weighted 3/4: 1.5 units; K2P takes 2 ln a + ln b - 3 ln n, 6 entries weighted 1/4: 1.5 units.
    Converting the integer (__ll2double_rn) and the multiply by the exact -3/4 * 2^-58 or -1/4 * 2^-58 round
    once each, 1/2 ulp of the result apiece.  So |got - exact| <= 1.5 * 2^-58 + 2 ulp(exact) for both.  A
    table built from the double log (~500 units per entry) is far outside it.

    The tuples with a = 0 take the floating-point form and are checked against the oracle like it.  On
    top, every value stays within 1.4e-13 relative of the oracle's formula, whose own 1 - x loses about
    1e-16 / x."""
    edges = M.edges(M.edge_lengths())
    counts = np.concatenate([edges[edges[:, :3].sum(axis=1) <= M.LN_TABLE_COLS],
                             M.random_tuples(np.random.default_rng(2048), 300_000, M.LN_TABLE_COLS)])
    got = engine.metrics_from_counts(counts, table=True)
    want = oracle.metrics_batch(counts)
    assert np.array_equal(np.isnan(got), np.isnan(want))
    assert len(mismatches(got[:, :2].copy(), want[:, :2].copy())) == 0
    assert not (got.view(np.uint64) == np.uint64(1 << 63)).any(), "-0.0"
    c = counts.astype(np.int64)
    n, ts, tv = c[:, :3].sum(axis=1), c[:, 1], c[:, 2]
    A, a, b = 3 * n - 4 * (ts + tv), n - 2 * ts - tv, n - 2 * tv
    fallback = (n > 0) & (a == 0) & (b > 0) & ~np.isnan(want[:, 3])
    assert fallback.sum() > 100
    assert M.ulp_distance(got[fallback, 3], want[fallback, 3]).max() <= FP_ULP
    exact_ok = (n > 0) & (A > 0) & (a > 0) & (b > 0)
    ej, ek = M.table_exact(counts[exact_ok])
    report = []
    for col, exact in ((2, ej), (3, ek)):
        g = got[exact_ok, col]
        e58, eulp = M.table_error(g, exact)
        exf = np.array([x / 2 ** (M.FRAC + 2) for x in exact])
        ulp = np.array([math.ulp(x) for x in exf])
        over = e58 * 2.0**-58 > 1.5 * 2.0**-58 + 2 * ulp
        assert not over.any(), (col, counts[exact_ok][over][:8].tolist())
        rel = e58 * 2.0**-58 / np.maximum(exf, 1e-300)
        report.append((e58.max(), eulp.max(), rel.max()))
    for col in (2, 3):
        ok = ~np.isnan(want[:, col]) & (want[:, col] != 0)
        rel = np.abs(got[ok, col] - want[ok, col]) / want[ok, col]
        report.append(rel.max())
        assert rel.max() <= TABLE_REL, (col, counts[ok][rel > TABLE_REL][:8].tolist())
        assert (got[~ok, col][~np.isnan(got[~ok, col])] == 0).all()
    (j58, julp, jrel), (k58, kulp, krel), jo, ko = report
    print(f"\ntable form, {len(counts)} tuples: JC within {j58:.2f} units of 2^-58 / {julp:.2f} ulp / {jrel:.3g} relative of exact, "
          f"K2P within {k58:.2f} / {kulp:.2f} ulp / {krel:.3g}; against the oracle JC {jo:.3g}, K2P {ko:.3g} relative")
