"""Which alignment-free counting kernel a call takes, restated in Python (no GPU).

`taxi_count_rect` walks a rectangle in blocks of whole rows (at most COUNT_CHUNK_PAIRS pairs each)
and `enqueue_count` (taxi2_b200/csrc/taxi_abi.cu) picks one of four kernels per block:

    popcount    count_rect_kernel               8   (several launches above 65535 slabs of rows)
    tc128       count_tc_kernel<128>            9   (count_kernel = 2 or the default, tc_tile_x = 128)
    tc64        count_tc_kernel<64>             9   (tc_tile_x = 64)
    persistent  count_tc_persistent_kernel      9   (tc_persistent = 1)
    pairs       count_pairs_kernel              8   (taxi_count_pairs)

It also decides, once per job, whether JC / K2P come from the fixed-point logarithm table: that
depends on the words per row W of the loaded sets, which are padded to whole carry-save groups, so a
set whose longest row has more than 1 920 columns takes the floating-point form.  The constants
below are restated by hand; tests/test_count_dispatch.py parses them from the sources, so a change
there without one here fails."""
from __future__ import annotations

import re
from pathlib import Path

CSRC = Path(__file__).resolve().parent.parent / "taxi2_b200" / "csrc"

TC_TILE = 128                # count_tc.cuh: y columns per tile, bytes of K per k-block
TC_BAND = 12                 # x tiles per band of the CTA order
TC_ROW_SEGMENTS = 8          # operand row = 8 Lp bytes
TC_STAGES = {128: 5, 64: 4}  # TcGeom<TX>::STAGES
TCP_TX = 64                  # persistent form: x rows per tile
TCP_STAGES = 5
COUNT_G = 5                  # count_planes.cuh: words per carry-save group (W is a multiple)
COUNT_SLAB = 64              # x rows staged per popcount block, at most
COUNT_TY = 256               # y columns per popcount block
LN_TABLE_COLS = 2048         # common.cuh
SLAB_BYTES = 64 * 1024       # shared memory a popcount block stages its x rows in
ROW_BYTES_MAX = 200 * 1024   # popcount refusal: W * 16 bytes above this
GRID_Y_MAX = 65535           # popcount slabs per launch; also (nx + 63) / 64 for the tensor cores
TC_MAX_OPERAND_BYTES = 8 << 30
TC_MIN_TILES_PER_SM = 2      # default rule: tensor cores when 128 x 128 tiles >= 2 * SMs
COUNT_CHUNK_PAIRS = 1 << 27  # taxi_count_rect: pairs per device block

CODE = {"popcount": 8, "pairs": 8, "tc128": 9, "tc64": 9, "persistent": 9}


def _cdiv(a: int, b: int) -> int:
    return -(-a // b)


def words(maxlen: int) -> int:
    """W of a set: 32-column words of its longest row, padded to whole carry-save groups (at least one)."""
    return max(1, _cdiv(_cdiv(maxlen, 32), COUNT_G)) * COUNT_G


def padded(maxlen: int) -> int:
    """Lp of a set: the operand row length of the tensor-core kernels, W * 32 padded to TC_TILE."""
    return _cdiv(words(maxlen) * 32, TC_TILE) * TC_TILE


def table_form(x_maxlen: int, y_maxlen: int, metric_tables: int = 1) -> bool:
    """JC / K2P from the logarithm table (else the floating-point form): decided on the smaller W."""
    return bool(metric_tables) and min(words(x_maxlen), words(y_maxlen)) * 32 <= LN_TABLE_COLS


def kblocks(x_maxlen: int, y_maxlen: int) -> int:
    """k-blocks of TC_TILE bytes per tile: 6 Lp over the common operand length."""
    return 6 * min(padded(x_maxlen), padded(y_maxlen)) // TC_TILE


def slab(x_maxlen: int, y_maxlen: int) -> int:
    row_bytes = min(words(x_maxlen), words(y_maxlen)) * 16
    return max(1, min(COUNT_SLAB, SLAB_BYTES // row_bytes))


def operand_bytes(n: int, maxlen: int) -> int:
    return max(n, 1) * TC_ROW_SEGMENTS * padded(maxlen)


class Refused(Exception):
    """The library returns TAXI_E_RANGE."""


def enqueue(nx: int, ny: int, x_set: tuple[int, int], y_set: tuple[int, int], sms: int, count_kernel: int = 0,
            tc_persistent: int = 0, tc_tile_x: int = 128, metric_tables: int = 1) -> dict:
    """One device block of a rectangle (enqueue_count).  x_set / y_set = (sequences, longest row) of
    the loaded sets (y_set = x_set when set 1 is not loaded).  -> dict(kernel, launches, table,
    slab, ntiles, grid, tiles_x, tiles_y, per_cta, kblocks, stages); raises Refused."""
    (xn, xl), (yn, yl) = x_set, y_set
    out = dict(table=table_form(xl, yl, metric_tables), kblocks=kblocks(xl, yl))
    if count_kernel != 1:
        tiles = _cdiv(nx, TC_TILE) * _cdiv(ny, TC_TILE)
        fits = (operand_bytes(xn, xl) <= TC_MAX_OPERAND_BYTES and operand_bytes(yn, yl) <= TC_MAX_OPERAND_BYTES
                and _cdiv(nx, 64) <= GRID_Y_MAX)
        if fits and (count_kernel == 2 or tiles >= TC_MIN_TILES_PER_SM * sms):
            kernel = "persistent" if tc_persistent else ("tc128" if tc_tile_x == 128 else "tc64")
            tx = TCP_TX if tc_persistent else tc_tile_x
            tiles_x, tiles_y = _cdiv(nx, tx), _cdiv(ny, TC_TILE)
            ntiles = tiles_x * tiles_y
            grid = min(ntiles, sms) if tc_persistent else ntiles
            stages = TCP_STAGES if tc_persistent else TC_STAGES[tx]
            return dict(out, kernel=kernel, launches=1, slab=0, ntiles=ntiles, grid=grid, tiles_x=tiles_x, tiles_y=tiles_y,
                        per_cta=_cdiv(ntiles, grid), stages=stages)
        if count_kernel == 2:
            raise Refused("sequences too long for the tensor-core counting kernel")
    if min(words(xl), words(yl)) * 16 > ROW_BYTES_MAX:
        raise Refused("sequences too long for the alignment-free kernel")
    s = slab(xl, yl)
    return dict(out, kernel="popcount", launches=_cdiv(nx, GRID_Y_MAX * s), slab=s, ntiles=0, grid=0, tiles_x=0,
                tiles_y=0, per_cta=0, stages=0)


def count_rect(nx: int, ny: int, x_set, y_set, sms: int, **options) -> dict:
    """taxi_count_rect: the blocks of whole rows, each through `enqueue`.  -> the last block's
    prediction with `launches` summed over the blocks and `blocks` = their number."""
    rows = max(1, min(nx, COUNT_CHUNK_PAIRS // ny))
    launches, blocks, last = 0, 0, None
    for r0 in range(0, nx, rows):
        last = enqueue(min(rows, nx - r0), ny, x_set, y_set, sms, **options)
        launches += last["launches"]
        blocks += 1
    return dict(last, launches=launches, blocks=blocks)


def count_pairs(x_set, y_set, metric_tables: int = 1) -> dict:
    """taxi_count_pairs: one launch of the pair-list kernel."""
    (_, xl), (_, yl) = x_set, y_set
    return dict(kernel="pairs", launches=1, table=table_form(xl, yl, metric_tables))


# ---- the same constants, parsed from the sources ----------------------------------------------------
def _find(pattern: str, text: str, name: str, group: int = 1) -> str:
    m = re.search(pattern, text, re.S)
    assert m, f"{name} not found"
    return m.group(group)


def _product(text: str) -> int:
    a, b = text.split("*")
    return int(a) * int(b)


def parse_constants(csrc: Path = CSRC) -> dict:
    """The constants the restatement depends on, read from the CUDA sources."""
    common = (csrc / "common.cuh").read_text()
    planes = (csrc / "count_planes.cuh").read_text()
    tc = (csrc / "count_tc.cuh").read_text()
    abi = (csrc / "taxi_abi.cu").read_text()
    enq = _find(r"static int enqueue_count\(.*?\n\}\n", abi, "enqueue_count", 0)
    load = _find(r"int taxi_load_sequences\(.*?\n\}\n", abi, "taxi_load_sequences", 0)
    rect = _find(r"int taxi_count_rect\(.*?\n\}\n", abi, "taxi_count_rect", 0)

    def const(text, name):
        return int(_find(rf"constexpr int {name} = (\d+);", text, name))

    out = {name: const(tc, name) for name in ("TC_TILE", "TC_BAND", "TC_ROW_SEGMENTS", "TCP_TX", "TCP_STAGES")}
    out.update({name: const(planes, name) for name in ("COUNT_G", "COUNT_SLAB", "COUNT_TY")})
    out["LN_TABLE_COLS"] = const(common, "LN_TABLE_COLS")
    stages = _find(r"static constexpr int STAGES = TX == 128 \? (\d+) : (\d+);", tc, "TcGeom::STAGES", 0)
    a, b = re.findall(r"\d+", stages.split("?")[1])
    out["TC_STAGES"] = {128: int(a), 64: int(b)}
    m = re.search(r"constexpr size_t kTcMaxOperandBytes = \(size_t\)(\d+) << (\d+);", abi)
    assert m, "kTcMaxOperandBytes not found"
    out["TC_MAX_OPERAND_BYTES"] = int(m.group(1)) << int(m.group(2))
    out["COUNT_CHUNK_PAIRS"] = 1 << int(_find(r"constexpr long long kCountChunkPairs = 1LL << (\d+);", abi, "kCountChunkPairs"))
    out["GRID_Y_MAX"] = int(_find(r"rows_per_launch = (\d+) \* a\.slab;", enq, "rows_per_launch"))
    out["GRID_Y_MAX (tensor cores)"] = int(_find(r"\(a\.nx \+ 63\) / 64 <= (\d+)", enq, "tensor-core row limit"))
    out["TC_MIN_TILES_PER_SM"] = int(_find(r"tiles >= (\d+)LL \* c->sms", enq, "default rule"))
    out["SLAB_BYTES"] = _product(_find(r"std::min<size_t>\(COUNT_SLAB, \((\d+ \* \d+)\) / row_bytes\)", enq, "slab bytes"))
    out["ROW_BYTES_MAX"] = _product(_find(r"if \(row_bytes > (\d+ \* \d+)\) return fail\(TAXI_E_RANGE", enq, "row bytes limit"))
    # the rules themselves, as the restatement reads them
    out["table rule"] = "std::min(X.W, Y.W) * 32 <= LN_TABLE_COLS" in enq
    out["W rule"] = "s.W = std::max(1, ((s.maxlen + 31) / 32 + COUNT_G - 1) / COUNT_G) * COUNT_G;" in load
    out["Lp rule"] = "s.Lp = (s.W * 32 + TC_TILE - 1) / TC_TILE * TC_TILE;" in abi
    out["kblocks rule"] = tc.count("const int kblocks = 6 * blocks_per_L;") == 2 and "std::min(XX.Lp, YY.Lp)" in enq
    out["persistent grid"] = "count_tc_persistent_kernel<<<std::min(ntiles, c->sms)" in enq
    out["chunk rule"] = "std::min<long long>(nx, kCountChunkPairs / ny)" in rect
    return out


def restated_constants() -> dict:
    return {"TC_TILE": TC_TILE, "TC_BAND": TC_BAND, "TC_ROW_SEGMENTS": TC_ROW_SEGMENTS, "TCP_TX": TCP_TX, "TCP_STAGES": TCP_STAGES,
            "COUNT_G": COUNT_G, "COUNT_SLAB": COUNT_SLAB, "COUNT_TY": COUNT_TY, "LN_TABLE_COLS": LN_TABLE_COLS,
            "TC_STAGES": TC_STAGES, "TC_MAX_OPERAND_BYTES": TC_MAX_OPERAND_BYTES, "COUNT_CHUNK_PAIRS": COUNT_CHUNK_PAIRS,
            "GRID_Y_MAX": GRID_Y_MAX, "GRID_Y_MAX (tensor cores)": GRID_Y_MAX, "TC_MIN_TILES_PER_SM": TC_MIN_TILES_PER_SM,
            "SLAB_BYTES": SLAB_BYTES, "ROW_BYTES_MAX": ROW_BYTES_MAX, "table rule": True, "W rule": True, "Lp rule": True,
            "kblocks rule": True, "persistent grid": True, "chunk rule": True}
