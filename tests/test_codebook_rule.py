"""The codebook restatement (codebook.py) against the sources it restates, and its predictions on the
load histories the GPU module replays (no GPU).

Every constant and rule the restatement uses is parsed from taxi2_b200/csrc; a change there without
the same change in codebook.py fails here, and so would a parser that stopped seeing one (each is
altered in a scratch copy of the sources and must be noticed)."""
from __future__ import annotations

import shutil

import pytest

import codebook as B

DEFAULT = (1, -1, -8, -1, -1, -1)


def test_parsed_constants_match_the_restatement():
    assert B.parse_constants() == B.restated_constants()


# (file, text as it is, text altered): one edit per parsed constant or rule
EDITS = [
    ("common.cuh", "constexpr int CODE_SYMBOLS = 15;", "constexpr int CODE_SYMBOLS = 14;"),
    ("common.cuh", "constexpr uint32_t CODE_PADSYM = 15u;", "constexpr uint32_t CODE_PADSYM = 14u;"),
    ("taxi_abi.cu", 'const char* fixed = "ACGTN";', 'const char* fixed = "ACGTU";'),
    ("taxi_abi.cu", "for (int k = 0; k < 5; ++k) c->codebook[", "for (int k = 0; k < 4; ++k) c->codebook["),
    ("taxi_abi.cu", "c->ncodes = 5;", "c->ncodes = 4;"),
    ("taxi_abi.cu", "if (c->ncodes >= CODE_SYMBOLS) c->codebook_ok = false;", "if (c->ncodes > CODE_SYMBOLS) c->codebook_ok = false;"),
    ("taxi_abi.cu", "if (set == 0) c->set[1].loaded = false;", "if (set == 1) c->set[0].loaded = true;"),
    ("taxi_abi.cu", "if (c->force_general || !c->codebook_ok) return false;", "if (c->force_general) return false;"),
    ("taxi_abi.cu", "if (ch == '-') f.has_gap_symbol = 1;", "if (ch == '-') f.has_gap_symbol = 0;"),
    ("taxi_abi.cu", "k < s.total && c->codebook_ok;", "k < s.total;"),
]


@pytest.mark.parametrize("edit", EDITS, ids=lambda e: e[2])
def test_an_edited_constant_is_noticed(tmp_path, edit):
    name, old, new = edit
    shutil.copytree(B.CSRC, tmp_path / "csrc")
    path = tmp_path / "csrc" / name
    text = path.read_text()
    assert old in text, f"{old!r} no longer in {name}: update EDITS"
    path.write_text(text.replace(old, new, 1))
    try:
        parsed = B.parse_constants(tmp_path / "csrc")
    except AssertionError:
        return   # the parser no longer finds it: noticed as well
    assert parsed != B.restated_constants()


def test_set_1_extends_and_set_0_resets():
    c = B.Context().load([b"ACGTRY"], 0)
    assert c.symbols == b"ACGTNRY"
    c.load([b"KRA"], 1)
    assert c.symbols == b"ACGTNRYK" and c.book[ord("R")] == 5       # set 0 keeps the codes of the older book
    c.load([b"M"], 1)
    assert c.symbols == b"ACGTNRYKM"                               # symbols accumulate over set-1 reloads
    assert c.loaded == [True, True]
    c.load([b"S"], 0)
    assert c.symbols == b"ACGTNS" and c.loaded == [True, False]    # reset, set 1 unloaded


def test_overflow_lasts_until_set_0():
    extra = bytes(range(0x80, 0x80 + B.CODE_SYMBOLS - len(B.FIXED)))
    c = B.Context().load([b"ACGT" + extra], 0)
    assert c.ok and len(c.book) == B.CODE_SYMBOLS
    c.load([b"ACGT"], 1)
    assert c.ok
    c.load([b"\x00"], 1)
    assert not c.ok
    c.load([b"ACGT"], 1)
    assert not c.ok
    c.load([b"ACGT"], 0)
    assert c.ok and c.symbols == b"ACGTN"


def test_gap_symbol_follows_the_book():
    c = B.Context().load([b"ACGT"], 0)
    assert not c.has_gap_symbol
    c.load([b"AC-GT"], 1)
    assert c.has_gap_symbol
    c.load([b"ACGT"], 1)
    assert c.has_gap_symbol                                        # no '-' loaded any more, still in the book
    c.load([b"ACGT"], 0)
    assert not c.has_gap_symbol


def test_every_byte_value_in_groups_of_ten_stays_packed():
    """The 251 bytes outside ACGTN in groups of at most ten fit one book each; all 256 do not."""
    others = bytes(b for b in range(256) if b not in B.FIXED)
    assert len(others) == 251
    for k in range(0, len(others), 10):
        c = B.Context().load([others[k:k + 10]], 0)
        assert c.ok
    assert not B.Context().load([bytes(range(256))], 0).ok


@pytest.mark.parametrize("h", B.HISTORIES, ids=lambda h: h["id"])
def test_history_predictions(h):
    c = B.replay([([alphabet], which) for alphabet, which in h["loads"]])
    assert (c.ok, c.has_gap_symbol, len(c.book)) == (h["ok"], h["gap"], h["ncodes"])
    s0, s1 = B.final_sets(h["loads"])
    fresh = B.replay([([s0], 0)] + ([([s1], 1)] if s1 is not None else []))
    # a fresh context overflows only when the final sets themselves hold more than CODE_SYMBOLS symbols
    assert fresh.ok == (len(set(B.FIXED) | set(s0) | set(s1 or b"")) <= B.CODE_SYMBOLS)
    if h["id"] == "overflow-by-set-1-then-plain-set-1":
        assert fresh.ok and not c.ok          # general only because of the history
    # a 100 bp pair list under the default scores: packed bottom-aligned, or general because of the book
    assert B.kernel(c, DEFAULT, [100] * 8, [100] * 8) == (17 if h["ok"] else 32)
    assert B.kernel(fresh, DEFAULT, [100] * 8, [100] * 8) == (17 if fresh.ok else 32)
