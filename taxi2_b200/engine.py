"""Batch engine: one context per GPU over the C ABI.  numpy host buffers in, numpy out.

This is the host-side mirror of the two native calls the reference makes per pair
(/root/reference/src/itaxotools/taxi2/align.py:151-153 and distances.py:323-347), batched.
PyTorch is optional here and only used by callers that want device-resident outputs.
"""
from __future__ import annotations

import ctypes as C
from typing import Iterable, Sequence as Seq

import numpy as np

from . import _native as N

SCORE_KEYS = (
    "match_score",
    "mismatch_score",
    "internal_open_gap_score",
    "internal_extend_gap_score",
    "end_open_gap_score",
    "end_extend_gap_score",
)
DEFAULT_SCORES = (1, -1, -8, -1, -1, -1)
METRIC_LABELS = ("p", "p-gaps", "jc", "k2p")


def scores_vector(scores) -> np.ndarray:
    if scores is None:
        scores = DEFAULT_SCORES
    if isinstance(scores, dict):
        scores = [scores[k] for k in SCORE_KEYS]
    vals = []
    for s in scores:
        if float(s) != int(s):
            raise ValueError(f"taxi2_b200 aligns with integer scores only (got {s!r}); Scores is dict[str, int]")
        vals.append(int(s))
    if len(vals) != 6:
        raise ValueError("expected six scores")
    return np.asarray(vals, dtype=np.int32)


def pack_strings(seqs: Iterable[str | bytes]) -> tuple[np.ndarray, np.ndarray]:
    """list of str/bytes -> (uint8 concatenation, int64 offsets[n+1])"""
    bs = [s.encode("latin-1", "replace") if isinstance(s, str) else bytes(s) for s in seqs]
    off = np.zeros(len(bs) + 1, dtype=np.int64)
    if bs:
        np.cumsum([len(b) for b in bs], out=off[1:])
    data = np.frombuffer(b"".join(bs), dtype=np.uint8) if bs else np.zeros(0, np.uint8)
    return np.ascontiguousarray(data), off


def _p(a: np.ndarray | None):
    return None if a is None else a.ctypes.data_as(C.c_void_p)


class PinnedArray:
    """numpy view of a page-locked host buffer owned by the library (freed with the object)."""

    def __init__(self, shape, dtype):
        self._lib = N.load()
        self.nbytes = int(np.prod(shape)) * np.dtype(dtype).itemsize
        self._ptr = self._lib.taxi_host_alloc(max(self.nbytes, 1))
        if not self._ptr:
            raise MemoryError("taxi_host_alloc failed")
        buf = (C.c_uint8 * max(self.nbytes, 1)).from_address(self._ptr)
        self.array = np.frombuffer(buf, dtype=dtype, count=int(np.prod(shape))).reshape(shape)

    def __del__(self):
        try:
            if getattr(self, "_ptr", None):
                self._lib.taxi_host_free(self._ptr)
                self._ptr = None
        except Exception:
            pass


class Engine:
    """One GPU context.  Not thread-safe; create one per device (one process per GPU)."""

    def __init__(self, device: int = 0, scores=None):
        self._lib = N.load()
        self._ctx = C.c_void_p()
        N.check(self._lib.taxi_ctx_create(int(device), C.byref(self._ctx)))
        self.device = int(device)
        self.n = [0, 0]
        self._string_pool: dict = {}
        self._pinned_pool: dict = {}
        self.set_scores(scores)

    # -- lifecycle ---------------------------------------------------------------------------
    def close(self) -> None:
        if getattr(self, "_ctx", None):
            self._lib.taxi_ctx_destroy(self._ctx)
            self._ctx = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()

    # -- configuration -----------------------------------------------------------------------
    def set_scores(self, scores) -> None:
        v = scores_vector(scores)
        N.check(self._lib.taxi_set_scores(self._ctx, v.ctypes.data_as(C.POINTER(C.c_int32))))
        self.scores = tuple(int(s) for s in v)

    def load(self, seqs, which: int = 0) -> None:
        """Upload a sequence set (list of str/bytes, or (bytes, offsets) arrays). 0 = x/rows, 1 = y/columns."""
        if isinstance(seqs, tuple) and len(seqs) == 2 and isinstance(seqs[0], np.ndarray):
            data, off = seqs
            data = np.ascontiguousarray(data, dtype=np.uint8)
            off = np.ascontiguousarray(off, dtype=np.int64)
        else:
            data, off = pack_strings(seqs)
        N.check(self._lib.taxi_load_sequences(self._ctx, int(which), _p(data), _p(off), len(off) - 1))
        self.n[which] = len(off) - 1
        if which == 0:  # a new row set serves as both until set 1 is loaded again
            self.n[1] = 0
            self._y_is_x = True
        else:
            self._y_is_x = False

    @property
    def ny(self) -> int:
        return self.n[0] if getattr(self, "_y_is_x", True) else self.n[1]

    # -- aligned path ------------------------------------------------------------------------
    def align_rect(self, x0: int, nx: int, y0: int, ny: int, want=("score", "counts", "metrics"), pinned: bool = False,
                   slot: int = 0, out: dict | None = None) -> dict:
        """pinned=True reuses page-locked result buffers owned by the engine: the returned arrays are
        views that the next pinned call with the same `slot` overwrites.  out = {"score" / "counts" /
        "metrics": C-contiguous array of nx*ny entries} makes the library write straight into the
        caller's arrays (e.g. this rectangle's slice of one pinned matrix shared by several GPUs)."""
        npairs = nx * ny
        flags, score, counts, metrics = self._outputs(npairs, want, self._pool(slot) if pinned else None, out)
        N.check(self._lib.taxi_align_rect(self._ctx, x0, nx, y0, ny, flags, _p(score), _p(counts), _p(metrics)))
        return self._result(score, counts, metrics, (nx, ny))

    def align_rect_both(self, x0: int, nx: int, y0: int, ny: int, want=("score", "counts", "metrics"),
                        out: dict | None = None, out_t: dict | None = None) -> tuple[dict, dict]:
        """Both orientations of a rectangle -- (x, y) as (nx, ny, ...) arrays and (y, x) as (ny, nx, ...)
        arrays -- from one alignment per unordered pair plus the re-alignment of the few
        orientation-sensitive ones (taxi_align_rect_both).  Bit-identical to two align_rect calls with
        the sets exchanged.  out / out_t: 2-D views (e.g. a tile and its mirror inside one matrix) whose
        rows may be strided; the last axis must be contiguous."""
        shapes = {"score": ((), np.int32), "counts": ((4,), np.int32), "metrics": ((4,), np.float64)}
        flags = sum(f for k, f in (("score", N.OUT_SCORE), ("counts", N.OUT_COUNTS), ("metrics", N.OUT_METRICS)) if k in want)
        res, res_t, ptr, ptr_t = {}, {}, {}, {}
        ld = {"xy": None, "yx": None}
        for key in ("score", "counts", "metrics"):
            tail, dtype = shapes[key]
            if key not in want:
                ptr[key] = ptr_t[key] = None
                continue
            for which, given, store, ptrs, rows, cols in (("xy", out, res, ptr, nx, ny), ("yx", out_t, res_t, ptr_t, ny, nx)):
                arr = given[key] if given is not None and key in given else np.empty((rows, cols, *tail), dtype=dtype)
                if arr.shape != (rows, cols, *tail) or arr.dtype != np.dtype(dtype):
                    raise ValueError(f"{key}: expected shape {(rows, cols, *tail)} {np.dtype(dtype)}")
                item = arr.dtype.itemsize * (4 if tail else 1)
                if arr.strides[1] != item or (tail and arr.strides[2] != arr.dtype.itemsize) or arr.strides[0] % item:
                    raise ValueError(f"{key}: rows may be strided, pairs within a row must be contiguous")
                stride = arr.strides[0] // item if rows > 1 else cols
                if ld[which] not in (None, stride):
                    raise ValueError("all outputs of one orientation must share their row stride (in pairs)")
                ld[which] = stride
                store[key] = arr
                ptrs[key] = C.c_void_p(arr.ctypes.data)
        N.check(self._lib.taxi_align_rect_both(self._ctx, x0, nx, y0, ny, flags, ptr["score"], ptr["counts"], ptr["metrics"], ld["xy"] or ny,
                                               ptr_t["score"], ptr_t["counts"], ptr_t["metrics"], ld["yx"] or nx))
        return res, res_t

    @property
    def last_redo(self) -> int:
        """Pairs the last both-orientations call had to re-align the other way round."""
        return int(self._lib.taxi_last_redo(self._ctx))

    def align_rect_both_device(self, x0, nx, y0, ny, d_counts=0, d_metrics=0, t_counts=0, t_metrics=0) -> None:
        """Device-resident form (pointers as ints); synchronous."""
        flags = (N.OUT_COUNTS if d_counts else 0) | (N.OUT_METRICS if d_metrics else 0)
        N.check(self._lib.taxi_align_rect_both_device(self._ctx, x0, nx, y0, ny, flags, None, C.c_void_p(d_counts), C.c_void_p(d_metrics),
                                                      None, C.c_void_p(t_counts), C.c_void_p(t_metrics)))

    def align_rect_resident(self, x0: int, nx: int, y0: int, ny: int, want=("counts", "metrics")) -> None:
        """Same work with the results left in the library's device buffers (no download): what a
        caller that reduces on the device needs, and the device-resident leg of bench.py."""
        flags = sum(f for k, f in (("score", N.OUT_SCORE), ("counts", N.OUT_COUNTS), ("metrics", N.OUT_METRICS)) if k in want)
        N.check(self._lib.taxi_align_rect(self._ctx, x0, nx, y0, ny, flags, None, None, None))

    def count_rect_resident(self, x0: int, nx: int, y0: int, ny: int, want=("counts", "metrics")) -> None:
        flags = sum(f for k, f in (("counts", N.OUT_COUNTS), ("metrics", N.OUT_METRICS)) if k in want)
        N.check(self._lib.taxi_count_rect(self._ctx, x0, nx, y0, ny, flags, None, None))

    def _pool(self, slot: int) -> dict:
        return self._pinned_pool.setdefault(int(slot), {})

    def align_pairs(self, px, py, want=("score", "counts", "metrics")) -> dict:
        px = np.ascontiguousarray(px, dtype=np.int32)
        py = np.ascontiguousarray(py, dtype=np.int32)
        flags, score, counts, metrics = self._outputs(len(px), want)
        N.check(self._lib.taxi_align_pairs(self._ctx, _p(px), _p(py), len(px), flags, _p(score), _p(counts), _p(metrics)))
        return self._result(score, counts, metrics, None)

    def align_strings_raw(self, px, py, want=("score",), slot: int | None = None) -> tuple:
        """-> (aln_x, aln_y, start, off, scores[, result dict]): pair k's gapped strings are
        aln_x / aln_y[start[k]:off[k + 1]] (right-aligned in slots of len(x) + len(y) bytes).
        With "counts" / "metrics" in `want` the same launch also fills them (sixth element: the
        dict align_pairs would return), so strings and distances come from ONE alignment.
        slot: the two string arrays are kept and handed out again by the next call with the same
        slot -- a block of barcode pairs is 2.6 KB of strings per pair, and first-touching
        hundreds of fresh megabytes per block costs more than the download itself.  Only for
        callers that are done with a block's strings before they reuse its slot."""
        px = np.ascontiguousarray(px, dtype=np.int32)
        py = np.ascontiguousarray(py, dtype=np.int32)
        n = len(px)
        off = np.zeros(n + 1, dtype=np.int64)
        N.check(self._lib.taxi_alignment_capacity(self._ctx, _p(px), _p(py), n, _p(off)))
        total = int(off[-1])
        if slot is None:
            ox = np.zeros(max(total, 1), dtype=np.uint8)
            oy = np.zeros(max(total, 1), dtype=np.uint8)
        else:
            kept = self._string_pool.setdefault(int(slot), {})
            if "x" not in kept or len(kept["x"]) < total:
                kept["x"] = np.empty(max(total, 1) + total // 8, dtype=np.uint8)
                kept["y"] = np.empty(max(total, 1) + total // 8, dtype=np.uint8)
            ox, oy = kept["x"][: max(total, 1)], kept["y"][: max(total, 1)]
        start = np.zeros(max(n, 1), dtype=np.int64)
        flags, score, counts, metrics = self._outputs(n, tuple(want) + ("score",))
        N.check(self._lib.taxi_align_strings_metrics(self._ctx, _p(px), _p(py), n, _p(off), _p(ox), _p(oy), _p(start),
                                                     flags, _p(score), _p(counts), _p(metrics)))
        if counts is None and metrics is None:
            return ox, oy, start, off, score
        return ox, oy, start, off, score, self._result(score, counts, metrics, None)

    def align_strings(self, px, py) -> tuple[list[bytes], list[bytes], np.ndarray]:
        """-> (aligned x, aligned y, scores) for each pair, Biopython's first alignment."""
        ox, oy, start, off, score = self.align_strings_raw(px, py)
        n = len(score)
        bx, by = ox.tobytes(), oy.tobytes()
        ax = [bx[int(start[k]): int(off[k + 1])] for k in range(n)]
        ay = [by[int(start[k]): int(off[k + 1])] for k in range(n)]
        return ax, ay, score[:n]

    def align_rect_device(self, x0, nx, y0, ny, d_score=0, d_counts=0, d_metrics=0) -> None:
        """Enqueue on the context stream with DEVICE output pointers (ints, e.g. tensor.data_ptr())."""
        flags = (N.OUT_SCORE if d_score else 0) | (N.OUT_COUNTS if d_counts else 0) | (N.OUT_METRICS if d_metrics else 0)
        N.check(self._lib.taxi_align_rect_device(self._ctx, x0, nx, y0, ny, flags,
                                                 C.c_void_p(d_score), C.c_void_p(d_counts), C.c_void_p(d_metrics)))

    # -- alignment-free path -----------------------------------------------------------------
    def count_rect(self, x0: int, nx: int, y0: int, ny: int, want=("counts", "metrics"), pinned: bool = False,
                   slot: int = 0, out: dict | None = None) -> dict:
        flags, _, counts, metrics = self._outputs(nx * ny, want, self._pool(slot) if pinned else None, out)
        N.check(self._lib.taxi_count_rect(self._ctx, x0, nx, y0, ny, flags, _p(counts), _p(metrics)))
        return self._result(None, counts, metrics, (nx, ny))

    def count_pairs(self, px, py, want=("counts", "metrics")) -> dict:
        px = np.ascontiguousarray(px, dtype=np.int32)
        py = np.ascontiguousarray(py, dtype=np.int32)
        flags, _, counts, metrics = self._outputs(len(px), want)
        N.check(self._lib.taxi_count_pairs(self._ctx, _p(px), _p(py), len(px), flags, _p(counts), _p(metrics)))
        return self._result(None, counts, metrics, None)

    def count_rect_device(self, x0, nx, y0, ny, d_counts=0, d_metrics=0) -> None:
        flags = (N.OUT_COUNTS if d_counts else 0) | (N.OUT_METRICS if d_metrics else 0)
        N.check(self._lib.taxi_count_rect_device(self._ctx, x0, nx, y0, ny, flags, C.c_void_p(d_counts), C.c_void_p(d_metrics)))

    def metrics_from_counts(self, counts, table: bool = False) -> np.ndarray:
        """(n, 4) count tuples {same, ts, tv, gaps} -> (n, 4) {p, p-gaps, jc, k2p}, NaN = undefined: the
        epilogue of every kernel on its own (table=True: the fixed-point logarithm table of the
        alignment-free kernels)."""
        counts = np.ascontiguousarray(counts, dtype=np.int32).reshape(-1, 4)
        out = np.empty((len(counts), 4), dtype=np.float64)
        N.check(self._lib.taxi_metrics_from_counts(self._ctx, _p(counts), len(counts), int(bool(table)), _p(out)))
        return out

    def argmin_rows_device(self, d_metrics: int, nx: int, ny: int, metric: int) -> tuple[np.ndarray, np.ndarray]:
        idx = np.zeros(nx, dtype=np.int32)
        val = np.zeros(nx, dtype=np.float64)
        N.check(self._lib.taxi_argmin_rows_device(self._ctx, C.c_void_p(d_metrics), nx, ny, metric, _p(idx), _p(val)))
        return idx, val

    def set_option(self, key: str, value: int) -> None:
        N.check(self._lib.taxi_set_option(self._ctx, key.encode(), int(value)))

    @property
    def last_kernel(self) -> int:
        """32 = general int32 kernel; 16 / 17 / 18 = packed 16-bit kernel (top-aligned / bottom-aligned /
        bottom-aligned in several stripes); 48 = a rectangle whose rows were split into several launches."""
        return int(self._lib.taxi_last_kernel(self._ctx))

    def best_rows(self, x0: int, nx: int, y0: int, ny: int, metric: int = 0, align: bool = True) -> dict:
        """Best match of every row x0..x0+nx over the columns [y0, y0+ny): first minimum of metric
        column `metric` (versus_reference.py:184-188) with all four metrics and the counts of the
        winning pair.  The nx x ny matrix never leaves the device (taxi_best_rows).
        index = -1 where a row has no defined distance."""
        index = np.full(max(nx, 1), -1, dtype=np.int32)[:nx]
        best = np.full((max(nx, 1), 4), np.nan, dtype=np.float64)[:nx]
        counts = np.zeros((max(nx, 1), 4), dtype=np.int32)[:nx]
        N.check(self._lib.taxi_best_rows(self._ctx, x0, nx, y0, ny, int(metric), int(bool(align)), _p(index), _p(best), _p(counts)))
        return dict(index=index, metrics=best, counts=counts)

    def best_rows_k(self, x0: int, nx: int, y0: int, ny: int, k: int, metric: int = 0, align: bool = True) -> dict:
        """The k closest columns of every row x0..x0+nx over [y0, y0+ny), selected on the device
        (taxi_best_rows_k): per row the k smallest (value of metric column `metric`, column index)
        in ascending order, NaN never ranked.  index (nx, k) int32, metrics (nx, k, 4) float64,
        counts (nx, k, 4) int32; slots past a row's defined values hold -1 / NaN / 0.  k = 1 is
        best_rows with a rank axis."""
        k = int(k)
        shape = (nx, max(k, 0))   # the library refuses k outside 1..64
        index = np.full(shape, -1, dtype=np.int32)
        best = np.full((*shape, 4), np.nan, dtype=np.float64)
        counts = np.zeros((*shape, 4), dtype=np.int32)
        N.check(self._lib.taxi_best_rows_k(self._ctx, x0, nx, y0, ny, int(metric), int(bool(align)), k,
                                           _p(index), _p(best), _p(counts)))
        return dict(index=index, metrics=best, counts=counts)

    def pairs_within(self, x0: int, nx: int, y0: int, ny: int, threshold: float, metric: int = 0, align: bool = True,
                     scale: float = 1.0, skip_self: bool = False) -> dict:
        """Every pair of rows x0..x0+nx x columns [y0, y0+ny) whose value v of metric column `metric`
        is not NaN and has v * scale <= threshold, selected and compacted on the device
        (taxi_pairs_within).  CSR in row-major pair order: row_ptr (nx+1,) int64; index (total,)
        int32, the column (an index into set 1), ascending within a row; metrics (total, 4) float64;
        counts (total, 4) int32.  scale=100 with a percentage threshold is the tasks' `d * 100 <=
        similarity`.  skip_self drops the pairs (i, i) of set 0 against itself."""
        row_ptr = np.zeros(max(nx, 0) + 1, dtype=np.int64)
        total = C.c_int64(0)
        N.check(self._lib.taxi_pairs_within(self._ctx, x0, nx, y0, ny, int(metric), int(bool(align)), float(threshold),
                                            float(scale), int(bool(skip_self)), _p(row_ptr), C.byref(total)))
        n = total.value
        index = np.empty(n, dtype=np.int32)
        metrics = np.empty((n, 4), dtype=np.float64)
        counts = np.empty((n, 4), dtype=np.int32)
        N.check(self._lib.taxi_pairs_within_fetch(self._ctx, _p(index), _p(metrics), _p(counts)))
        return dict(row_ptr=row_ptr, index=index, metrics=metrics, counts=counts)

    def clusters_within(self, x0: int, nx: int, y0: int, ny: int, thresholds, metric: int = 0, align: bool = True,
                        scale: float = 1.0, seed: np.ndarray | None = None) -> np.ndarray:
        """Single-linkage clusters of set 0 at one or more thresholds (taxi_clusters_within): x and y
        are linked at threshold t iff the pair (x, y) of rows x0..x0+nx x columns [y0, y0+ny) of set 0
        x set 0 has a value v of metric column `metric` that is not NaN and v * scale <= t (the
        predicate of pairs_within); the pairs (i, i) link nothing.  Returns labels (m, n) int32 for
        the m thresholds (a float or a sequence of up to 8) and the n sequences of set 0: the smallest
        index in each sequence's component.  seed, an earlier result of the same shape, starts the
        components from its labeling, so calls over disjoint row ranges chain."""
        ts = np.ascontiguousarray(np.atleast_1d(np.asarray(thresholds, dtype=np.float64)).ravel())
        labels = np.empty((len(ts), self.n[0]), dtype=np.int32)
        if seed is not None:
            seed = np.ascontiguousarray(seed, dtype=np.int32)
            if seed.shape != labels.shape:
                raise ValueError(f"seed must have shape {labels.shape} (thresholds x sequences of set 0), not {seed.shape}")
        N.check(self._lib.taxi_clusters_within(self._ctx, x0, nx, y0, ny, int(metric), int(bool(align)), _p(ts), len(ts),
                                               float(scale), _p(seed), _p(labels)))
        return labels

    def best_matches(self, metric: int = 0, align: bool = True, rows_per_tile: int | None = None) -> dict:
        """versusReference at scale (BASELINE config C4): best_rows over all of set 0 x all of set 1."""
        return self.best_rows(0, self.n[0], 0, self.ny, metric, align)

    def sync(self) -> None:
        N.check(self._lib.taxi_sync(self._ctx))

    def stats(self) -> dict:
        launches, cells, ms = C.c_int64(0), C.c_int64(0), C.c_double(0.0)
        N.check(self._lib.taxi_last_stats(self._ctx, C.byref(launches), C.byref(cells), C.byref(ms)))
        return dict(launches=launches.value, cells=cells.value, kernel_ms=ms.value)

    # -- helpers -----------------------------------------------------------------------------
    @staticmethod
    def _outputs(n: int, want: Seq[str], pool: dict | None = None, out: dict | None = None):
        def buffer(key, shape, dtype):
            if out is not None and key in out and n > 0:
                given = out[key]
                if given.dtype != np.dtype(dtype) or not given.flags.c_contiguous or given.size != int(np.prod(shape)):
                    raise ValueError(f"out[{key!r}] must be a C-contiguous {np.dtype(dtype)} array of {int(np.prod(shape))} elements")
                return given.reshape(shape)
            if pool is None:
                return np.zeros(shape, dtype=dtype)
            held = pool.get(key)
            if held is None or held.array.shape[0] < shape[0]:
                held = pool[key] = PinnedArray(shape, dtype)
            return held.array[: shape[0]]

        flags = 0
        score = counts = metrics = None
        if "score" in want:
            flags |= N.OUT_SCORE
            score = buffer("score", (max(n, 1),), np.int32)[:n]
        if "counts" in want:
            flags |= N.OUT_COUNTS
            counts = buffer("counts", (max(n, 1), 4), np.int32)[:n]
        if "metrics" in want:
            flags |= N.OUT_METRICS
            metrics = buffer("metrics", (max(n, 1), 4), np.float64)[:n]
        return flags, score, counts, metrics

    @staticmethod
    def _result(score, counts, metrics, shape):
        out = {}
        if score is not None:
            out["score"] = score.reshape(shape) if shape else score
        if counts is not None:
            out["counts"] = counts.reshape(*shape, 4) if shape else counts
        if metrics is not None:
            out["metrics"] = metrics.reshape(*shape, 4) if shape else metrics
        return out


_engines: dict[int, Engine] = {}


def default_engine(device: int = 0) -> Engine:
    """Process-wide engine per device (lazily created; raises without a GPU)."""
    eng = _engines.get(device)
    if eng is None:
        eng = _engines[device] = Engine(device)
    return eng
