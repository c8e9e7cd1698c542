"""The column sweep of the packed bottom-aligned kernel (`align_two_bottom`) at the edges of its
segments: the fill while lanes start, the steady state that runs without per-step tests, the end
columns of the two pairs of a warp unit and the drain.  Also the y symbols the sweep hands down the
lanes, which lane l0 (the first lane holding a row >= 0) takes from chunks of 32 columns, and the
one-instruction mismatch term of every packed kernel, for every pair of the 16 symbol codes.

Every launch asserts that the bottom-aligned packed kernel ran, and every result is compared with
the oracle: scores, counts and gapped strings bit for bit, metrics within 1e-12."""
from __future__ import annotations

import subprocess
from pathlib import Path

import numpy as np
import pytest

import oracle
from __graft_entry__ import ARCH, NVCC

pytestmark = pytest.mark.gpu

BOTTOM = 17                        # last_kernel of the packed, bottom-aligned, single-stripe kernel
SCORES = (1, -1, -8, -1, -1, -1)   # TaxI2's default; internal extend == end extend: bottom-aligned
ALPHA = np.frombuffer(b"ACGT", dtype=np.uint8)


@pytest.fixture(scope="module")
def engine():
    from taxi2_b200.engine import Engine

    eng = Engine(0)
    eng.set_scores(SCORES)
    yield eng
    eng.close()


def related(rng, nx: int, ny: int, sub: float = 0.1) -> tuple[bytes, bytes]:
    """x of length nx and y of length ny cut from one mutated ancestor (ragged overhangs at both ends)."""
    root = ALPHA[rng.integers(0, 4, max(nx, ny) + 40)]
    x, y = root[:nx].copy(), root[40:40 + ny].copy()
    hit = rng.random(ny) < sub
    y[hit] = ALPHA[rng.integers(0, 4, int(hit.sum()))]
    return x.tobytes(), y.tobytes()


def assert_metrics_close(got: np.ndarray, want: np.ndarray):
    nan_g, nan_w = np.isnan(got), np.isnan(want)
    assert np.array_equal(nan_g, nan_w)
    assert np.allclose(got[~nan_g], want[~nan_w], rtol=1e-12, atol=0.0)


def oracle_batch(xs, ys, px, py):
    from taxi2_b200.engine import pack_strings

    data, off = pack_strings(list(xs) + list(ys))
    return oracle.align_count_pairs(data, off, np.asarray(px, dtype=np.int32), np.asarray(py, dtype=np.int32) + len(xs), SCORES)


def check_units(engine, xs, ys):
    """Align (xs[k], ys[k]) as a pair list; two pairs share a warp unit, so a two-pair list is one unit."""
    n = len(xs)
    px = np.arange(n, dtype=np.int32)
    want = oracle_batch(xs, ys, px, px)
    engine.load(xs, 0)
    engine.load(ys, 1)
    got = engine.align_pairs(px, px)
    assert engine.last_kernel == BOTTOM
    assert np.array_equal(got["score"], want["score"]), [(len(x), len(y)) for x, y in zip(xs, ys)]
    assert np.array_equal(got["counts"], want["counts"])
    assert_metrics_close(got["metrics"], want["metrics"])
    ax, ay, sc = engine.align_strings(px, px)
    assert engine.last_kernel == BOTTOM
    assert np.array_equal(sc, want["score"])
    for k in range(n):
        ox, oy, _ = oracle.align(xs[k], ys[k], SCORES)
        assert ax[k].decode() == ox and ay[k].decode() == oy, (len(xs[k]), len(ys[k]))


# x lengths of a unit and the first live lane l0 they give: one stripe of 32 lanes x 21 rows
# (512..671 rows; row nA sits in the last slot, row 0 in slot 672 - nA - 1)
X_LENGTHS = [(671, 671), (651, 600), (650, 650), (640, 520), (520, 515)]   # l0 = 0, 0, 1, 1, 7


@pytest.mark.parametrize("nx", X_LENGTHS, ids=lambda v: f"x{v[0]}-{v[1]}")
def test_pairs_ending_on_different_columns(engine, nx):
    """The two pairs of a unit end on different columns: a 1 bp y next to a 650 bp one (no steady
    state at all), short y lengths around the fill length (steady state empty or a single step),
    and y lengths one column apart, in both halves of the unit."""
    rng = np.random.default_rng(nx[0] * 1000 + nx[1])
    l0 = (672 - max(nx) - 1) // 21
    fill = 31 - l0
    for ya, yb in [(1, 650), (2, 3), (fill, 650), (fill + 1, 640), (fill + 2, 600), (649, 650), (650, 650), (300, 40)]:
        for first, second in [(ya, yb), (yb, ya)]:
            xa, ya_ = related(rng, nx[0], first)
            xb, yb_ = related(rng, nx[1], second)
            check_units(engine, [xa, xb], [ya_, yb_])


@pytest.mark.parametrize("nx", X_LENGTHS, ids=lambda v: f"x{v[0]}-{v[1]}")
def test_y_lengths_around_chunk_boundaries(engine, nx):
    """y symbols come in chunks of 32 columns: y lengths at multiples of 32 and one either side,
    alone and next to a partner that ends elsewhere."""
    rng = np.random.default_rng(7 + nx[0] + nx[1])
    lengths = [31, 32, 33, 63, 64, 65, 95, 96, 97, 127, 128, 129, 639, 640, 641]
    xs, ys = [], []
    for k, ny in enumerate(lengths):
        for partner in (ny, lengths[(k + 5) % len(lengths)]):
            xa, ya = related(rng, nx[0], ny)
            xb, yb = related(rng, nx[1], partner)
            check_units(engine, [xa, xb], [ya, yb])
            xs += [xa, xb]; ys += [ya, yb]
    check_units(engine, xs, ys)   # many units in one launch


def test_rectangle_columns_of_different_length(engine):
    """The benchmark's shape -- a unit is two neighbouring columns of one rectangle row -- with
    columns of every kind of length next to each other (columns kept in the given order)."""
    rng = np.random.default_rng(650)
    ny = [1, 650, 30, 31, 32, 33, 64, 65, 96, 649, 651, 2, 128, 640, 641]
    root = ALPHA[rng.integers(0, 4, 700)]
    xs = []
    for _ in range(6):
        x = root[:650].copy()
        hit = rng.random(650) < 0.12
        x[hit] = ALPHA[rng.integers(0, 4, int(hit.sum()))]
        xs.append(x.tobytes())
    ys = [related(rng, 650, n)[1] for n in ny]
    engine.load(xs, 0)
    engine.load(ys, 1)
    engine.set_option("sort_columns", 0)
    try:
        got = engine.align_rect(0, len(xs), 0, len(ys))
    finally:
        engine.set_option("sort_columns", 1)
    assert engine.last_kernel == BOTTOM
    px, py = np.divmod(np.arange(len(xs) * len(ys)), len(ys))
    want = oracle_batch(xs, ys, px, py)
    assert np.array_equal(got["score"].ravel(), want["score"])
    assert np.array_equal(got["counts"].reshape(-1, 4), want["counts"])
    assert_metrics_close(got["metrics"].reshape(-1, 4), want["metrics"])


MISMATCH_CHECK = r"""
#include <cstdio>
#include "gotoh_pair16.cuh"
// every (a, b) of pair A in the low half with every (c, d) of pair B in the high half, for H(i-1, j-1)
// values and penalties of the 16-bit window (a half never borrows: the window keeps H above the penalty)
__global__ void check(unsigned long long* bad, unsigned long long* done)
{
    const uint32_t hd[] = {0xFFF3FFF3u, 0x7D007D00u, 0xFFF0FA02u, 0x80008000u, 0xFFFFFFFFu, 0x00200020u};
    const uint32_t d16[] = {16u, 32u, 16u * 2000u, 32767u};
    const uint32_t idx = blockIdx.x * blockDim.x + threadIdx.x;   // a | b << 4 | c << 8 | d << 12
    const uint32_t a = idx & 15u, b = (idx >> 4) & 15u, c = (idx >> 8) & 15u, d = (idx >> 12) & 15u;
    for (uint32_t Hd : hd)
        for (uint32_t D : d16) {
            if ((Hd & 0xFFFFu) < D || (Hd >> 16) < D) continue;
            const uint32_t got = taxi::diag_candidate(Hd, taxi::row_codes(a, c), b | (d << 16), 0u - D);
            const uint32_t lo = (Hd & 0xFFFFu) - (a != b ? D : 0u), hi = (Hd >> 16) - (c != d ? D : 0u);
            atomicAdd(done, 1ULL);
            if (got != (lo | (hi << 16))) atomicAdd(bad, 1ULL);
        }
}
int main()
{
    unsigned long long *dev, host[2] = {0, 0};
    if (cudaMalloc(&dev, 16) != cudaSuccess || cudaMemset(dev, 0, 16) != cudaSuccess) return 2;
    check<<<256, 256>>>(dev, dev + 1);
    if (cudaMemcpy(host, dev, 16, cudaMemcpyDeviceToHost) != cudaSuccess) return 2;
    printf("%llu %llu\n", host[0], host[1]);
    return 0;
}
"""


def test_mismatch_term_for_every_pair_of_codes(tmp_path):
    """diag_candidate() takes the mismatch flag from the packed add of VIADDMNMX.U16x2 on negated
    row codes, which is right only if that add wraps per half instead of saturating: checked on
    the device for all 16 x 16 code pairs in both halves at once (65 536 combinations)."""
    src, exe = tmp_path / "mismatch_check.cu", tmp_path / "mismatch_check"
    src.write_text(MISMATCH_CHECK)
    csrc = Path(__file__).resolve().parent.parent / "taxi2_b200" / "csrc"
    subprocess.run([NVCC, *ARCH, "-O3", "-std=c++17", "-I", str(csrc), "-o", str(exe), str(src)], check=True, capture_output=True)
    out = subprocess.run([str(exe)], check=True, capture_output=True, text=True).stdout.split()
    bad, done = int(out[0]), int(out[1])
    assert done == 65536 * 21   # (H, penalty) combinations inside the window, per code quadruple
    assert bad == 0
