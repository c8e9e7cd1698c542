"""The alignment-free dispatch restatement (count_dispatch.py) against the sources it restates (no GPU).

Every constant and rule the restatement uses is parsed from taxi2_b200/csrc; a change there without
the same change in count_dispatch.py fails here, and so would a parser that stopped seeing one (each
constant is altered in a scratch copy of the sources and must be noticed).  The predictions the GPU
module relies on are checked at their edges."""
from __future__ import annotations

import shutil

import pytest

import count_dispatch as D

SMS = 148   # B200


def test_parsed_constants_match_the_restatement():
    assert D.parse_constants() == D.restated_constants()


# (file, text as it is, text altered): one edit per parsed constant or rule
EDITS = [
    ("count_tc.cuh", "constexpr int TC_TILE = 128;", "constexpr int TC_TILE = 256;"),
    ("count_tc.cuh", "constexpr int TC_BAND = 12;", "constexpr int TC_BAND = 16;"),
    ("count_tc.cuh", "constexpr int TC_ROW_SEGMENTS = 8;", "constexpr int TC_ROW_SEGMENTS = 10;"),
    ("count_tc.cuh", "constexpr int TCP_TX = 64;", "constexpr int TCP_TX = 128;"),
    ("count_tc.cuh", "constexpr int TCP_STAGES = 5;", "constexpr int TCP_STAGES = 4;"),
    ("count_tc.cuh", "STAGES = TX == 128 ? 5 : 4;", "STAGES = TX == 128 ? 4 : 4;"),
    ("count_tc.cuh", "STAGES = TX == 128 ? 5 : 4;", "STAGES = TX == 128 ? 5 : 3;"),
    ("count_tc.cuh", "const int kblocks = 6 * blocks_per_L;", "const int kblocks = 8 * blocks_per_L;"),
    ("count_planes.cuh", "constexpr int COUNT_G = 5;", "constexpr int COUNT_G = 4;"),
    ("count_planes.cuh", "constexpr int COUNT_SLAB = 64;", "constexpr int COUNT_SLAB = 32;"),
    ("count_planes.cuh", "constexpr int COUNT_TY = 256;", "constexpr int COUNT_TY = 128;"),
    ("common.cuh", "constexpr int LN_TABLE_COLS = 2048;", "constexpr int LN_TABLE_COLS = 1920;"),
    ("taxi_abi.cu", "kTcMaxOperandBytes = (size_t)8 << 30;", "kTcMaxOperandBytes = (size_t)4 << 30;"),
    ("taxi_abi.cu", "kCountChunkPairs = 1LL << 27;", "kCountChunkPairs = 1LL << 26;"),
    ("taxi_abi.cu", "rows_per_launch = 65535 * a.slab;", "rows_per_launch = 32767 * a.slab;"),
    ("taxi_abi.cu", "(a.nx + 63) / 64 <= 65535", "(a.nx + 63) / 64 <= 32767"),
    ("taxi_abi.cu", "tiles >= 2LL * c->sms", "tiles >= 3LL * c->sms"),
    ("taxi_abi.cu", "(64 * 1024) / row_bytes", "(96 * 1024) / row_bytes"),
    ("taxi_abi.cu", "row_bytes > 200 * 1024", "row_bytes > 100 * 1024"),
    ("taxi_abi.cu", "std::min(X.W, Y.W) * 32 <= LN_TABLE_COLS", "std::min(X.maxlen, Y.maxlen) <= LN_TABLE_COLS"),
    ("taxi_abi.cu", "/ COUNT_G) * COUNT_G;   // whole carry-save groups", ") * 1;   // whole carry-save groups"),
    ("taxi_abi.cu", "count_tc_persistent_kernel<<<std::min(ntiles, c->sms)", "count_tc_persistent_kernel<<<std::min(ntiles, 2 * c->sms)"),
    ("taxi_abi.cu", "std::min<long long>(nx, kCountChunkPairs / ny)", "std::min<long long>(nx, kCountChunkPairs / ny / 2)"),
]


@pytest.mark.parametrize("edit", EDITS, ids=lambda e: e[2])
def test_an_edited_constant_is_noticed(tmp_path, edit):
    name, old, new = edit
    shutil.copytree(D.CSRC, tmp_path / "csrc")
    path = tmp_path / "csrc" / name
    text = path.read_text()
    assert old in text, f"{old!r} no longer in {name}: update EDITS"
    path.write_text(text.replace(old, new, 1))
    try:
        parsed = D.parse_constants(tmp_path / "csrc")
    except AssertionError:
        return   # the parser no longer finds it: noticed as well
    assert parsed != D.restated_constants()


def test_table_threshold_is_1920_columns():
    """W is padded to whole carry-save groups of 5 words (160 columns): the longest row that keeps
    the table form has 1 920 columns, not LN_TABLE_COLS = 2 048; the smaller W of the two sets decides."""
    assert [D.words(n) for n in (0, 1, 160, 161, 1920, 1921, 2048, 2049)] == [5, 5, 5, 10, 60, 65, 65, 65]
    assert D.table_form(1920, 1920) and not D.table_form(1921, 1921) and not D.table_form(2048, 2048)
    assert D.table_form(1920, 2049) and D.table_form(5000, 10)
    assert not D.table_form(100, 100, metric_tables=0)


def test_operand_lengths_and_kblocks():
    """Lp is at least 256 (W >= 5 words): the smallest k loop is 12 blocks, over two passes of the
    5-stage ring plus 2; 384 gives 18.  The common Lp is the smaller of the two sets'."""
    assert [D.padded(n) for n in (0, 160, 161, 320, 321, 1920, 1921)] == [256, 256, 384, 384, 512, 1920, 2176]
    assert D.kblocks(160, 160) == 12 and D.kblocks(300, 300) == 18 and D.kblocks(300, 2049) == 18
    assert D.kblocks(2049, 2049) == 6 * 2176 // 128


def test_default_rule_and_tile_counts():
    x = y = (10000, 300)
    below = D.enqueue(59 * 128, 5 * 128, x, y, SMS)        # 295 tiles = 2 * 148 - 1
    at = D.enqueue(37 * 128, 8 * 128, x, y, SMS)           # 296 tiles
    assert below["kernel"] == "popcount" and at["kernel"] == "tc128"
    assert D.enqueue(1, 1, x, y, SMS, count_kernel=2)["kernel"] == "tc128"
    p = D.enqueue(119 * 64, 5 * 128, x, y, SMS, count_kernel=2, tc_persistent=1)
    assert (p["kernel"], p["ntiles"], p["grid"], p["per_cta"]) == ("persistent", 595, 148, 5)
    t = D.enqueue(25 * 64, 100, x, y, SMS, count_kernel=2, tc_tile_x=64)
    assert (t["kernel"], t["tiles_x"], t["tiles_y"], t["stages"]) == ("tc64", 25, 1, 4)


def test_popcount_split_and_tensor_core_refusal():
    rows = 65535 * 64
    x, y = (rows + 1, 40), (3, 3)
    assert D.count_rect(rows + 1, 3, x, y, SMS)["kernel"] == "popcount"
    assert D.count_rect(rows + 1, 3, x, y, SMS)["launches"] == 2
    assert D.count_rect(rows, 3, x, y, SMS)["kernel"] == "tc128"
    assert D.operand_bytes(rows + 1, 40) <= D.TC_MAX_OPERAND_BYTES   # the refusal is the row limit, not the size
    with pytest.raises(D.Refused):
        D.count_rect(rows + 1, 3, x, y, SMS, count_kernel=2)
    assert D.count_rect(rows, 3, x, y, SMS, count_kernel=1)["launches"] == 1
    # long rows: fewer staged rows per block, so a shorter rectangle already splits
    assert D.slab(9000, 9000) == 64 * 1024 // (D.words(9000) * 16)


def test_device_blocks_of_a_tall_rectangle():
    """taxi_count_rect: blocks of at most 2^27 pairs; each is dispatched on its own rows."""
    r = D.count_rect(70000, 4000, (70000, 300), (4000, 300), SMS)
    assert r["blocks"] == 3 and r["kernel"] == "tc128" and r["launches"] == 3
