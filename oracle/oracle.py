"""ctypes front-end of oracle/libtaxi_oracle.so (TEST INFRASTRUCTURE ONLY)."""
from __future__ import annotations

import ctypes as C
import subprocess
from pathlib import Path

import numpy as np

_DIR = Path(__file__).parent
_LIB_PATH = _DIR / "libtaxi_oracle.so"
_lib = None

SCORE_KEYS = (  # Scores.defaults order, /root/reference/src/itaxotools/taxi2/align.py:20-27
    "match_score",
    "mismatch_score",
    "internal_open_gap_score",
    "internal_extend_gap_score",
    "end_open_gap_score",
    "end_extend_gap_score",
)
DEFAULT_SCORES = (1, -1, -8, -1, -1, -1)


def build(force: bool = False) -> Path:
    src = _DIR / "taxi_oracle.c"
    if force or not _LIB_PATH.exists() or _LIB_PATH.stat().st_mtime < src.stat().st_mtime:
        subprocess.run(["make", "-C", str(_DIR), "-B", "libtaxi_oracle.so"], check=True, capture_output=True)
    return _LIB_PATH


def _load():
    global _lib
    if _lib is None:
        build()
        lib = C.CDLL(str(_LIB_PATH))
        u8p, i32p, i64p, f64p = (C.POINTER(t) for t in (C.c_uint8, C.c_int32, C.c_int64, C.c_double))
        lib.taxi_oracle_align.argtypes = [C.c_char_p, C.c_int32, C.c_char_p, C.c_int32, f64p,
                                          C.c_char_p, C.c_char_p, i32p, f64p]
        lib.taxi_oracle_align.restype = C.c_int
        lib.taxi_oracle_count.argtypes = [C.c_char_p, C.c_int64, C.c_char_p, C.c_int64, i32p]
        lib.taxi_oracle_count.restype = C.c_int
        lib.taxi_oracle_metrics.argtypes = [i32p, f64p]
        lib.taxi_oracle_metrics.restype = None
        lib.taxi_oracle_metrics_batch.argtypes = [i32p, C.c_int64, f64p]
        lib.taxi_oracle_metrics_batch.restype = None
        lib.taxi_oracle_uses_gotoh.argtypes = [f64p]
        lib.taxi_oracle_uses_gotoh.restype = C.c_int
        lib.taxi_oracle_max_threads.restype = C.c_int
        lib.taxi_oracle_align_count_pairs.argtypes = [u8p, i64p, i32p, i32p, C.c_int64, f64p, C.c_int32,
                                                      i32p, i32p, f64p, i32p]
        lib.taxi_oracle_align_count_pairs.restype = C.c_int
        lib.taxi_oracle_count_pairs.argtypes = [u8p, i64p, i32p, i32p, C.c_int64, C.c_int32, i32p, f64p]
        lib.taxi_oracle_count_pairs.restype = C.c_int
        _lib = lib
    return _lib


def _scores(scores) -> C.Array:
    if scores is None:
        scores = DEFAULT_SCORES
    if isinstance(scores, dict):
        scores = [scores[k] for k in SCORE_KEYS]
    return (C.c_double * 6)(*[float(s) for s in scores])


def uses_gotoh(scores=None) -> bool:
    return bool(_load().taxi_oracle_uses_gotoh(_scores(scores)))


def max_threads() -> int:
    return int(_load().taxi_oracle_max_threads())


def align(x: str | bytes, y: str | bytes, scores=None) -> tuple[str, str, float]:
    """-> (aligned_x, aligned_y, score); raises ValueError on an empty sequence like Biopython."""
    bx = x.encode("latin-1") if isinstance(x, str) else bytes(x)
    by = y.encode("latin-1") if isinstance(y, str) else bytes(y)
    cap = len(bx) + len(by) + 1
    oa, ob = C.create_string_buffer(cap), C.create_string_buffer(cap)
    n, score = C.c_int32(0), C.c_double(0.0)
    rc = _load().taxi_oracle_align(bx, len(bx), by, len(by), _scores(scores), oa, ob, C.byref(n), C.byref(score))
    if rc == -2:
        raise ValueError("sequence has zero length")
    if rc != 0:
        raise RuntimeError(f"taxi_oracle_align failed: {rc}")
    return oa.raw[: n.value].decode("latin-1"), ob.raw[: n.value].decode("latin-1"), score.value


def count(x: str | bytes, y: str | bytes) -> tuple[int, int, int, int] | None:
    """-> (same, transitions, transversions, internal gap columns), or None without overlap."""
    bx = x.encode("latin-1") if isinstance(x, str) else bytes(x)
    by = y.encode("latin-1") if isinstance(y, str) else bytes(y)
    out = (C.c_int32 * 4)()
    ok = _load().taxi_oracle_count(bx, len(bx), by, len(by), out)
    return tuple(out) if ok else None


def metrics(counts) -> tuple[float, float, float, float]:
    """counts -> (p, p-gaps, jc, k2p) with NaN for undefined."""
    cin = (C.c_int32 * 4)(*[int(c) for c in counts])
    out = (C.c_double * 4)()
    _load().taxi_oracle_metrics(cin, out)
    return tuple(out)


def metrics_batch(counts) -> np.ndarray:
    """(n, 4) count tuples -> (n, 4) float64 {p, p-gaps, jc, k2p}: `metrics` of each tuple in one call."""
    counts = np.ascontiguousarray(counts, dtype=np.int32).reshape(-1, 4)
    out = np.empty((len(counts), 4), np.float64)
    _load().taxi_oracle_metrics_batch(counts.ctypes.data_as(C.POINTER(C.c_int32)), len(counts),
                                      out.ctypes.data_as(C.POINTER(C.c_double)))
    return out


def align_count_pairs(seqs: np.ndarray, offsets: np.ndarray, px: np.ndarray, py: np.ndarray,
                      scores=None, threads: int = 0, want_metrics: bool = True):
    """Batch form used by the parity tests and the CPU baseline.

    seqs: uint8 concatenated normalized sequences; offsets: int64[n+1]; px/py: int32 pair lists.
    -> dict(score int32[P], counts int32[P,4], metrics float64[P,4], alnlen int32[P])
    """
    seqs = np.ascontiguousarray(seqs, dtype=np.uint8)
    offsets = np.ascontiguousarray(offsets, dtype=np.int64)
    px = np.ascontiguousarray(px, dtype=np.int32)
    py = np.ascontiguousarray(py, dtype=np.int32)
    P = px.shape[0]
    score = np.zeros(P, np.int32)
    counts = np.zeros((P, 4), np.int32)
    met = np.full((P, 4), np.nan, np.float64)
    alnlen = np.zeros(P, np.int32)
    ptr = lambda a, t: a.ctypes.data_as(C.POINTER(t))  # noqa: E731
    rc = _load().taxi_oracle_align_count_pairs(
        ptr(seqs, C.c_uint8), ptr(offsets, C.c_int64), ptr(px, C.c_int32), ptr(py, C.c_int32), P,
        _scores(scores), threads, ptr(score, C.c_int32), ptr(counts, C.c_int32),
        ptr(met, C.c_double) if want_metrics else None, ptr(alnlen, C.c_int32))
    if rc == -2:
        raise ValueError("sequence has zero length")
    if rc != 0:
        raise RuntimeError(f"taxi_oracle_align_count_pairs failed: {rc}")
    return dict(score=score, counts=counts, metrics=met, alnlen=alnlen)


def count_pairs(seqs: np.ndarray, offsets: np.ndarray, px: np.ndarray, py: np.ndarray, threads: int = 0):
    """Alignment-free batch (align = False): counts int32[P,4] and metrics float64[P,4] of the raw
    strings of every pair, truncated to the shorter one (all-zero counts / NaN without overlap)."""
    seqs = np.ascontiguousarray(seqs, dtype=np.uint8)
    offsets = np.ascontiguousarray(offsets, dtype=np.int64)
    px = np.ascontiguousarray(px, dtype=np.int32)
    py = np.ascontiguousarray(py, dtype=np.int32)
    P = px.shape[0]
    counts = np.zeros((P, 4), np.int32)
    met = np.full((P, 4), np.nan, np.float64)
    ptr = lambda a, t: a.ctypes.data_as(C.POINTER(t))  # noqa: E731
    rc = _load().taxi_oracle_count_pairs(ptr(seqs, C.c_uint8), ptr(offsets, C.c_int64), ptr(px, C.c_int32), ptr(py, C.c_int32),
                                         P, threads, ptr(counts, C.c_int32), ptr(met, C.c_double))
    if rc != 0:
        raise RuntimeError(f"taxi_oracle_count_pairs failed: {rc}")
    return dict(counts=counts, metrics=met)
