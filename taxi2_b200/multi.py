"""Multi-GPU product path: ONE process, one context and one host thread per GPU (SURVEY.md 8e).

Every pair is independent, so the pair matrix shards with no collective on the data path:

* the sequence sets are replicated on every GPU (C3: 32 MB, C4: 143 MB);
* the row-major pair product (pairs.py:23-25, versus_all.py:746) is cut into tiles -- by default
  full-width blocks of rows, so a tile's results are one contiguous slice of the result matrix;
* tiles are dealt to the GPUs statically, longest-processing-time-first by DP cells
  (`sharding.assign_tiles`), each GPU's thread walks its share in row order;
* results are gathered ON THE HOST: every GPU's D2H copy lands directly in its tile's slice of
  one (page-locked) host array, or -- for the best-match row reduction of
  versus_reference.py:184-188 -- only the per-query winners (or k closest references) come back
  and column tiles of one query are combined on the host with the first-index tie-break; the
  pairs within a threshold come back as per-tile CSR pieces, assembled on the host.

ctypes releases the GIL for the duration of a native call, so the threads really run concurrently;
a context is only ever touched by its own thread while a run is in flight.
"""
from __future__ import annotations

import threading
from typing import Callable, Iterable, Iterator

import numpy as np

from . import _native as N
from .engine import Engine, PinnedArray, pack_strings
from .sharding import Tile, assign_tiles, make_tiles


class MultiEngine:
    def __init__(self, devices: Iterable[int] | None = None, scores=None):
        if devices is None:
            count = int(N.load().taxi_device_count())
            if count < 1:
                raise N.TaxiNativeError(N.E_CUDA, "no CUDA device visible (taxi2_b200 has no CPU fallback)")
            devices = range(count)
        self.devices = [int(d) for d in devices]
        if not self.devices:
            raise ValueError("MultiEngine needs at least one device")
        self.engines = [Engine(d, scores) for d in self.devices]
        self.lens: list[np.ndarray | None] = [None, None]

    # -- lifecycle / configuration (broadcast to every context) ------------------------------------
    def close(self) -> None:
        for e in self.engines:
            e.close()

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()

    def _each(self, fn: Callable[[Engine], object]) -> list:
        """fn(engine) on every engine, each on its own thread; re-raises the first failure."""
        if len(self.engines) == 1:
            return [fn(self.engines[0])]
        out: list = [None] * len(self.engines)
        err: list = []

        def run(k):
            try:
                out[k] = fn(self.engines[k])
            except BaseException as e:   # noqa: BLE001 -- re-raised on the caller's thread
                err.append(e)

        threads = [threading.Thread(target=run, args=(k,), daemon=True) for k in range(len(self.engines))]
        for t in threads:
            t.start()
        for t in threads:
            t.join()
        if err:
            raise err[0]
        return out

    def set_scores(self, scores) -> None:
        for e in self.engines:
            e.set_scores(scores)

    def set_option(self, key: str, value: int) -> None:
        for e in self.engines:
            e.set_option(key, value)

    def load(self, seqs, which: int = 0) -> None:
        """Replicate a sequence set on every GPU (packed once on the host, uploaded in parallel)."""
        if isinstance(seqs, tuple) and len(seqs) == 2 and isinstance(seqs[0], np.ndarray):
            data, off = seqs
        else:
            data, off = pack_strings(seqs)
        self._each(lambda e: e.load((data, off), which))
        self.lens[which] = np.diff(np.asarray(off, dtype=np.int64))
        if which == 0:
            self.lens[1] = None

    @property
    def nx(self) -> int:
        return self.engines[0].n[0]

    @property
    def ny(self) -> int:
        return self.engines[0].ny

    def _lens_y(self) -> np.ndarray:
        return self.lens[1] if self.lens[1] is not None else self.lens[0]

    # -- the tile scheduler --------------------------------------------------------------------------
    def row_tiles(self, rows_per_tile: int | None = None, col_tiles: int = 1, x_range: tuple[int, int] | None = None) -> list[Tile]:
        """Tiles of the loaded product: blocks of whole rows (full width unless col_tiles > 1)."""
        lx, ly = self.lens[0], self._lens_y()
        if lx is None:
            raise ValueError("no sequences loaded")
        x0, x1 = x_range if x_range is not None else (0, len(lx))
        nx, ny = x1 - x0, len(ly)
        if rows_per_tile is None:
            # enough tiles for LPT to balance (>= 4 per GPU), each large enough to fill a GPU
            per_gpu_rows = max(1, -(-nx // (4 * len(self.engines))))
            rows_per_tile = max(1, min(per_gpu_rows, max(1, (1 << 22) // max(ny, 1))))
        tile_y = max(1, -(-ny // max(1, col_tiles)))
        tiles = make_tiles(lx[x0:x1], ly, rows_per_tile, tile_y)
        return [Tile(t.index, t.x0 + x0, t.nx, t.y0, t.ny, t.cells) for t in tiles]

    def run_tiles(self, tiles: list[Tile], fn: Callable[[Engine, Tile, int], object], depth: int = 2,
                  ordered: bool = True) -> Iterator[tuple[Tile, object]]:
        """fn(engine, tile, slot) for every tile on the GPU the static LPT plan assigns it to.

        Yields (tile, result) in tile order while the GPUs run ahead: each GPU may hold up to
        `depth` finished tiles the consumer has not taken yet (slot = tile's position modulo
        depth + 1 on its GPU, for double-buffered pinned result buffers), which bounds host memory
        and overlaps the consumer's work (formatting, writing) with the next tiles' compute.
        ordered=False yields tiles as they complete."""
        plan = assign_tiles(tiles, len(self.engines))
        cond = threading.Condition()
        done: dict[int, object] = {}
        failed: list[BaseException] = []
        stop = threading.Event()
        room = [threading.Semaphore(depth) for _ in self.engines]

        def worker(k: int) -> None:
            try:
                for pos, tile in enumerate(plan[k]):
                    while not room[k].acquire(timeout=0.1):
                        if stop.is_set():
                            return
                    if stop.is_set():
                        return
                    res = fn(self.engines[k], tile, pos % (depth + 1))
                    with cond:
                        done[tile.index] = (k, res)
                        cond.notify_all()
            except BaseException as e:   # noqa: BLE001 -- re-raised on the consumer's thread
                with cond:
                    failed.append(e)
                    cond.notify_all()

        threads = [threading.Thread(target=worker, args=(k,), daemon=True) for k in range(len(self.engines))]
        for t in threads:
            t.start()
        try:
            by_index = {t.index: t for t in tiles}
            pending = [t.index for t in tiles]
            while pending:
                with cond:
                    while not failed and not (done if not ordered else pending[0] in done):
                        cond.wait(0.5)
                    if failed:
                        raise failed[0]
                    idx = pending[0] if ordered else next(iter(done))
                    k, res = done.pop(idx)
                pending.remove(idx)
                yield by_index[idx], res
                room[k].release()
        finally:
            stop.set()
            for t in threads:
                t.join()

    # -- whole-matrix products -------------------------------------------------------------------------
    def _matrix(self, mode: str, want, rows_per_tile, pinned: bool, x_range=None, out: dict | None = None) -> dict:
        if rows_per_tile is None and mode == "count":
            # the alignment-free kernel does a row of barcodes in microseconds: one or two tiles per GPU
            rows = (x_range[1] - x_range[0]) if x_range is not None else self.nx
            rows_per_tile = max(1, min(-(-rows // (2 * len(self.engines))), (1 << 26) // max(self.ny, 1)))
        tiles = self.row_tiles(rows_per_tile, 1, x_range)
        x0 = tiles[0].x0 if tiles else 0
        nx, ny = sum(t.nx for t in tiles), self.ny
        shapes = {"score": ((nx, ny), np.int32), "counts": ((nx, ny, 4), np.int32), "metrics": ((nx, ny, 4), np.float64)}
        if mode == "count":
            want = tuple(w for w in want if w != "score")
        holders = {}
        given = out
        out = {}
        for key in want:
            shape, dtype = shapes[key]
            if given is not None and key in given:
                # caller-owned (e.g. one pinned matrix reused between runs): at least nx rows of the right width
                arr = given[key]
                if arr.dtype != np.dtype(dtype) or arr.shape[1:] != shape[1:] or arr.shape[0] < nx or not arr.flags.c_contiguous:
                    raise ValueError(f"out[{key!r}] must be a C-contiguous {np.dtype(dtype)} array of shape >= {shape}")
                out[key] = arr[:nx]
            elif pinned:
                holders[key] = PinnedArray(shape, dtype)
                out[key] = holders[key].array
            else:
                out[key] = np.empty(shape, dtype=dtype)

        def fn(engine: Engine, tile: Tile, slot: int):
            views = {key: out[key][tile.x0 - x0: tile.x0 - x0 + tile.nx] for key in want}
            call = engine.align_rect if mode == "align" else engine.count_rect
            call(tile.x0, tile.nx, 0, ny, want=want, out=views)
            return engine.stats()

        stats = [s for _, s in self.run_tiles(tiles, fn, depth=2, ordered=False)]
        out["_pinned"] = holders   # keeps the page-locked buffers alive as long as the result
        out["kernel_ms"] = sum(s["kernel_ms"] for s in stats)
        out["cells"] = sum(s["cells"] for s in stats)
        out["launches"] = sum(s["launches"] for s in stats)
        out["tiles"] = len(tiles)
        return out

    def align_matrix(self, want=("score", "counts", "metrics"), rows_per_tile: int | None = None, pinned: bool = False,
                     x_range: tuple[int, int] | None = None, out: dict | None = None) -> dict:
        """All ordered pairs set 0 x set 1 (or set 0 x set 0), row-major, gathered on the host:
        every GPU's D2H copy lands in its tiles' slices of one result array per output
        (pinned=True: page-locked arrays owned by the result; out=: the caller's arrays)."""
        return self._matrix("align", want, rows_per_tile, pinned, x_range, out)

    def count_matrix(self, want=("counts", "metrics"), rows_per_tile: int | None = None, pinned: bool = False,
                     x_range: tuple[int, int] | None = None, out: dict | None = None) -> dict:
        """Alignment-free counterpart of align_matrix (params.pairs.align = False)."""
        return self._matrix("count", want, rows_per_tile, pinned, x_range, out)

    # -- versusAll: both orientations from one alignment per unordered pair ---------------------------
    def symmetric_tiles(self, block: int | None = None, max_cols: int | None = None) -> list[Tile]:
        """Tiles of the UPPER triangle of set 0 x set 0 in row-block-major order: per block of rows its
        diagonal square, then rectangles of at most max_cols columns to the right of it.  A
        rectangle (rows r, columns c) yields the results of (r, c) and, mirrored, of (c, r).
        block=None: 2048-row blocks with wide rectangles on one GPU; with several GPUs square tiles,
        small enough that every GPU gets half a dozen of them for the LPT plan to balance."""
        lens = self.lens[0]
        if lens is None:
            raise ValueError("no sequences loaded")
        n = len(lens)
        gpus = len(self.engines)
        if block is None:
            blocks = -(-n // 2048)
            if gpus > 1:
                blocks = max(blocks, int(np.ceil(np.sqrt(12.0 * gpus))) + 1)
            block = -(-n // max(1, blocks))
            if max_cols is None and gpus > 1:
                max_cols = block
        block = max(1, int(block))
        max_cols = max(block, int(max_cols or 4 * block))
        cum = np.concatenate([[0], np.cumsum(lens, dtype=np.int64)])
        tiles: list[Tile] = []
        for x0 in range(0, n, block):
            nx = min(block, n - x0)
            rows = int(cum[x0 + nx] - cum[x0])
            tiles.append(Tile(len(tiles), x0, nx, x0, nx, rows * rows * 3 // 5))
            for y0 in range(x0 + nx, n, max_cols):
                ny = min(max_cols, n - y0)
                tiles.append(Tile(len(tiles), x0, nx, y0, ny, rows * int(cum[y0 + ny] - cum[y0]) * 6 // 5))
        return tiles

    def _diagonal_block(self, engine: Engine, x0: int, n: int, want, out: dict, acc: dict) -> None:
        """A square on the diagonal: its upper-right quarter through the both-orientations call (which
        also fills the lower-left one), the two diagonal quarters recursively; small squares directly."""
        if n <= 192:
            res = engine.align_rect(x0, n, x0, n, want=want)
            for key in want:
                out[key][x0:x0 + n, x0:x0 + n] = res[key]
            _accumulate(acc, engine, redo=False)
            return
        h = n // 2
        engine.align_rect_both(x0, h, x0 + h, n - h, want=want, out={k: out[k][x0:x0 + h, x0 + h:x0 + n] for k in want},
                               out_t={k: out[k][x0 + h:x0 + n, x0:x0 + h] for k in want})
        _accumulate(acc, engine, redo=True)
        self._diagonal_block(engine, x0, h, want, out, acc)
        self._diagonal_block(engine, x0 + h, n - h, want, out, acc)

    def iter_symmetric_rows(self, want=("score", "counts", "metrics"), block: int | None = None, max_cols: int | None = None,
                            pinned: bool = False, out: dict | None = None, on_diagonal=None) -> Iterator[tuple[int, int, dict]]:
        """All ordered pairs of set 0 x set 0 (versus_all.py:746) with ONE alignment per unordered pair:
        the alignment of (y, x) is the transpose of that of (x, y) unless a tie between a vertical and
        a horizontal gap is decided on the traced path; the kernel notices, those few pairs are
        re-aligned the other way round (Engine.align_rect_both).  Bit-identical to align_matrix.

        Yields (x0, nx, out) whenever a block of rows of the full (n, n, ...) result arrays `out` is
        complete (rows x0 .. x0+nx, in order), while the GPUs work ahead on the next tiles.
        on_diagonal(engine, x0, nx): optional per-row-block work that needs a context; runs on the
        GPU thread that owns the block's diagonal tile, its result is out["_extra"][x0]."""
        if self.lens[0] is None or self.lens[1] is not None:
            raise ValueError("iter_symmetric_rows works on set 0 x set 0: load set 0 only")
        n = self.nx
        shapes = {"score": ((n, n), np.int32), "counts": ((n, n, 4), np.int32), "metrics": ((n, n, 4), np.float64)}
        holders, res = {}, {}
        for key in want:
            shape, dtype = shapes[key]
            if out is not None and key in out:
                arr = out[key]
                if arr.dtype != np.dtype(dtype) or arr.shape != shape or not arr.flags.c_contiguous:
                    raise ValueError(f"out[{key!r}] must be a C-contiguous {np.dtype(dtype)} array of shape {shape}")
                res[key] = arr
            elif pinned:
                holders[key] = PinnedArray(shape, dtype)
                res[key] = holders[key].array
            else:
                res[key] = np.empty(shape, dtype=dtype)
        res["_pinned"] = holders
        res["_extra"] = {}
        acc = dict(kernel_ms=0.0, cells=0, launches=0, redo=0)
        lock = threading.Lock()
        tiles = self.symmetric_tiles(block, max_cols)
        last_of_row = {}
        for t in tiles:
            last_of_row[t.x0] = t.index

        def fn(engine: Engine, tile: Tile, slot: int):
            mine = dict(kernel_ms=0.0, cells=0, launches=0, redo=0)
            if tile.y0 == tile.x0:
                self._diagonal_block(engine, tile.x0, tile.nx, want, res, mine)
                if on_diagonal is not None:
                    res["_extra"][tile.x0] = on_diagonal(engine, tile.x0, tile.nx)
            else:
                xs, ys = slice(tile.x0, tile.x0 + tile.nx), slice(tile.y0, tile.y0 + tile.ny)
                engine.align_rect_both(tile.x0, tile.nx, tile.y0, tile.ny, want=want, out={k: res[k][xs, ys] for k in want},
                                       out_t={k: res[k][ys, xs] for k in want})
                _accumulate(mine, engine, redo=True)
            with lock:
                for key, v in mine.items():
                    acc[key] += v
            return None

        for tile, _ in self.run_tiles(tiles, fn, depth=4, ordered=True):
            if last_of_row[tile.x0] == tile.index:
                res.update(acc, tiles=len(tiles))
                yield tile.x0, tile.nx, res

    def align_matrix_symmetric(self, want=("score", "counts", "metrics"), block: int | None = None, max_cols: int | None = None,
                               pinned: bool = False, out: dict | None = None) -> dict:
        """align_matrix for set 0 x set 0 at roughly 0.6 of its cost (iter_symmetric_rows)."""
        res = None
        for _, _, res in self.iter_symmetric_rows(want, block, max_cols, pinned, out):
            pass
        if res is None:
            res = {key: np.empty(shape, dtype=dt) for key, (shape, dt) in
                   {"score": ((0, 0), np.int32), "counts": ((0, 0, 4), np.int32), "metrics": ((0, 0, 4), np.float64)}.items() if key in want}
            res.update(kernel_ms=0.0, cells=0, launches=0, redo=0, tiles=0)
        return res

    def best_matches(self, metric: int = 0, align: bool = True, rows_per_tile: int | None = None, col_tiles: int = 1) -> dict:
        """versusReference at scale (BASELINE config C4): per query of set 0 the FIRST minimum of
        metric column `metric` over all of set 1, with the winner's four metrics and counts.
        Row tiles go to the GPUs by LPT; with col_tiles > 1 a query's references are split too and
        the per-tile winners are combined here: smaller value wins, ties go to the smaller
        reference index (the reference scans references in order and keeps the first minimum)."""
        tiles = self.row_tiles(rows_per_tile, col_tiles)
        nx = self.nx
        index = np.full(nx, -1, dtype=np.int32)
        best = np.full((nx, 4), np.nan, dtype=np.float64)
        counts = np.zeros((nx, 4), dtype=np.int32)

        def fn(engine: Engine, tile: Tile, slot: int):
            res = engine.best_rows(tile.x0, tile.nx, tile.y0, tile.ny, metric, align)
            res["stats"] = engine.stats()
            return res

        kernel_ms = cells = launches = 0
        for tile, res in self.run_tiles(tiles, fn, depth=4, ordered=False):
            rows = slice(tile.x0, tile.x0 + tile.nx)
            combine_best(index[rows], best[rows], counts[rows], res["index"], res["metrics"], res["counts"], metric)
            kernel_ms += res["stats"]["kernel_ms"]; cells += res["stats"]["cells"]; launches += res["stats"]["launches"]
        return dict(index=index, metrics=best, counts=counts, kernel_ms=kernel_ms, cells=cells, launches=launches, tiles=len(tiles))

    def best_matches_k(self, k: int, metric: int = 0, align: bool = True, rows_per_tile: int | None = None,
                       col_tiles: int = 1) -> dict:
        """The k closest references of every query of set 0 over all of set 1 (Engine.best_rows_k):
        index (nx, k), metrics and counts (nx, k, 4), ascending by (value of metric column `metric`,
        reference index).  Tiles are scheduled as in best_matches; with col_tiles > 1 the per-tile
        lists of a query are merged here (combine_best_k), so the result is the same for any tiling,
        tile arrival order and number of GPUs."""
        k = int(k)
        tiles = self.row_tiles(rows_per_tile, col_tiles)
        nx = self.nx
        index = np.full((nx, max(k, 0)), -1, dtype=np.int32)
        best = np.full((nx, max(k, 0), 4), np.nan, dtype=np.float64)
        counts = np.zeros((nx, max(k, 0), 4), dtype=np.int32)

        def fn(engine: Engine, tile: Tile, slot: int):
            res = engine.best_rows_k(tile.x0, tile.nx, tile.y0, tile.ny, k, metric, align)
            res["stats"] = engine.stats()
            return res

        kernel_ms = cells = launches = 0
        for tile, res in self.run_tiles(tiles, fn, depth=4, ordered=False):
            rows = slice(tile.x0, tile.x0 + tile.nx)
            combine_best_k(index[rows], best[rows], counts[rows], res["index"], res["metrics"], res["counts"], metric)
            kernel_ms += res["stats"]["kernel_ms"]; cells += res["stats"]["cells"]; launches += res["stats"]["launches"]
        return dict(index=index, metrics=best, counts=counts, kernel_ms=kernel_ms, cells=cells, launches=launches, tiles=len(tiles))

    def pairs_within(self, threshold: float, metric: int = 0, align: bool = True, scale: float = 1.0, skip_self: bool = False,
                     rows_per_tile: int | None = None, col_tiles: int = 1) -> dict:
        """Every pair of set 0 x set 1 (or set 0 x set 0) whose value of metric column `metric`,
        times `scale`, is at most `threshold` (Engine.pairs_within): one CSR over all of set 0,
        row_ptr (nx+1,), index (total,), metrics and counts (total, 4), row-major with ascending
        reference index within a row.  Tiles are scheduled as in best_matches; the per-tile pieces
        are assembled here (combine_within), so the result is the same for any tiling, tile
        arrival order and number of GPUs."""
        tiles = self.row_tiles(rows_per_tile, col_tiles)

        def fn(engine: Engine, tile: Tile, slot: int):
            res = engine.pairs_within(tile.x0, tile.nx, tile.y0, tile.ny, threshold, metric, align, scale, skip_self)
            res["stats"] = engine.stats()
            return res

        pieces = []
        kernel_ms = cells = launches = 0
        for tile, res in self.run_tiles(tiles, fn, depth=4, ordered=False):
            pieces.append((tile.x0, tile.nx, tile.y0, res))
            kernel_ms += res["stats"]["kernel_ms"]; cells += res["stats"]["cells"]; launches += res["stats"]["launches"]
        out = combine_within(pieces, self.nx)
        out.update(kernel_ms=kernel_ms, cells=cells, launches=launches, tiles=len(tiles))
        return out


def _accumulate(acc: dict, engine, redo: bool) -> None:
    st = engine.stats()
    acc["kernel_ms"] += st["kernel_ms"]; acc["cells"] += st["cells"]; acc["launches"] += st["launches"]
    if redo:
        acc["redo"] += int(getattr(engine, "last_redo", 0))


def combine_best(index, best, counts, new_index, new_best, new_counts, metric: int) -> None:
    """Merge the winners of another column tile into (index, best, counts) in place: a candidate
    replaces the incumbent if it is defined and the incumbent is not, or its value is smaller, or
    equal with a smaller reference index -- i.e. the first minimum in reference order, whatever
    order the tiles arrive in (versus_reference.py:184-188)."""
    cand = new_index >= 0
    have = index >= 0
    nv, ov = new_best[:, metric], best[:, metric]
    with np.errstate(invalid="ignore"):
        take = cand & (~have | (nv < ov) | ((nv == ov) & (new_index < index)))
    index[take] = new_index[take]
    best[take] = new_best[take]
    counts[take] = new_counts[take]


def combine_best_k(index, best, counts, new_index, new_best, new_counts, metric: int) -> None:
    """The k-list counterpart of combine_best: merge another column tile's lists (new_*, (n, k) and
    (n, k, 4), ascending, undefined slots last as the library returns them) into (index, best,
    counts) in place.  Each row keeps the k smallest keys (value of metric column `metric`, reference
    index) of both lists in ascending order; undefined slots (index -1) never displace defined ones and
    are left as -1 / NaN / 0.  The key is a total order over distinct references, so the result does
    not depend on the order of the tiles."""
    k = index.shape[1]
    if k == 0:
        return
    mine, theirs = index[:, 0] >= 0, new_index[:, 0] >= 0
    # a row with nothing defined yet takes the other list as it is (every row of full-width tiles)
    take = theirs & ~mine
    if take.all():
        index[...], best[...], counts[...] = new_index, new_best, new_counts
        return
    index[take] = new_index[take]
    best[take] = new_best[take]
    counts[take] = new_counts[take]
    both = np.flatnonzero(theirs & mine)
    if not len(both):
        return
    idx = np.concatenate([index[both], new_index[both]], axis=1)
    undefined = idx < 0
    val = np.where(undefined, np.inf, np.concatenate([best[both, :, metric], new_best[both, :, metric]], axis=1))
    order = np.lexsort((idx, val, undefined), axis=-1)[:, :k]
    rows = np.arange(len(both))[:, None]
    empty = undefined[rows, order]
    index[both] = np.where(empty, -1, idx[rows, order])
    best[both] = np.where(empty[..., None], np.nan, np.concatenate([best[both], new_best[both]], axis=1)[rows, order])
    counts[both] = np.where(empty[..., None], 0, np.concatenate([counts[both], new_counts[both]], axis=1)[rows, order])


def combine_within(tiles, nx: int) -> dict:
    """Assemble the CSR pieces of taxi_pairs_within calls over tiles of rows 0..nx into one CSR.
    `tiles` holds (x0, nx, y0, piece), piece = dict(row_ptr, index, metrics, counts) of rows x0..x0+nx
    over columns from y0 on, in any order.  A row's segments are placed in ascending y0 (the column
    ranges of one row's tiles are disjoint), so every row lists its pairs in ascending reference
    index and the result is the same for any tiling and arrival order.  Per tile a few numpy
    operations: a tile that holds whole rows is one slice copy, otherwise one scatter."""
    tiles = sorted(tiles, key=lambda t: (t[2], t[0]))
    per_row = np.zeros(nx, dtype=np.int64)
    for x0, n, _, piece in tiles:
        per_row[x0:x0 + n] += np.diff(piece["row_ptr"])
    row_ptr = np.zeros(nx + 1, dtype=np.int64)
    np.cumsum(per_row, out=row_ptr[1:])
    total = int(row_ptr[-1])
    index = np.empty(total, dtype=np.int32)
    metrics = np.empty((total, 4), dtype=np.float64)
    counts = np.empty((total, 4), dtype=np.int32)
    fill = row_ptr[:-1].copy()   # the next free entry of every row
    for x0, n, _, piece in tiles:
        lens = np.diff(piece["row_ptr"])
        if np.array_equal(lens, per_row[x0:x0 + n]):   # the tile holds all of its rows' pairs
            dst = slice(int(row_ptr[x0]), int(row_ptr[x0 + n]))
        else:
            dst = np.repeat(fill[x0:x0 + n] - piece["row_ptr"][:-1], lens) + np.arange(int(piece["row_ptr"][-1]))
        index[dst] = piece["index"]
        metrics[dst] = piece["metrics"]
        counts[dst] = piece["counts"]
        fill[x0:x0 + n] += lens
    return dict(row_ptr=row_ptr, index=index, metrics=metrics, counts=counts)
