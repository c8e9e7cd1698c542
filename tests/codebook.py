"""The symbol codebook of a context, restated in Python (no GPU).

The packed alignment kernel never sees bytes: `taxi_load_sequences` (taxi2_b200/csrc/taxi_abi.cu)
turns every symbol into a 4-bit code from a codebook shared by both sequence sets, and
`fast16_eligible` builds the tables that classify columns and write gapped strings from that book.
The rule:

    - A, C, G, T, N hold the codes 0..4;
    - every other byte takes the next code when it is first seen, set 0 before set 1;
    - there are CODE_SYMBOLS codes in all: the byte that would need one more clears `codebook_ok`,
      and the packed kernel is then refused (the general kernel reads bytes) ...
    - ... until set 0 is loaded again: a set-0 load resets the book (and unloads set 1), a set-1
      load only adds to it, so a book that overflowed stays overflowed over any set-1 reload;
    - `has_gap_symbol` is set when '-' is in the book -- the book, not the sets loaded now.

`Context` replays a history of loads and predicts the book, `codebook_ok` and `has_gap_symbol`;
`kernel` combines that with `kernel_geometry.instance` into the `last_kernel` of a call.  The
constants are restated by hand; tests/test_codebook_rule.py parses them from the sources, so a
change there without one here fails."""
from __future__ import annotations

import re
from pathlib import Path

import kernel_geometry as K

CSRC = Path(__file__).resolve().parent.parent / "taxi2_b200" / "csrc"

CODE_SYMBOLS = 15     # common.cuh: codes 0..14 are symbols
CODE_PADSYM = 15      # common.cuh: the pad code, "matches no symbol"
FIXED = b"ACGTN"      # taxi_load_sequences: the codes every book starts with


def _bytes(seqs) -> bytes:
    return b"".join(s.encode("latin-1") if isinstance(s, str) else bytes(s) for s in seqs)


class Context:
    """The codebook state of one context over a history of `load(seqs, which)` calls."""

    def __init__(self):
        self.book = {b: k for k, b in enumerate(FIXED)}
        self.ok = True
        self.loaded = [False, False]

    def load(self, seqs, which: int) -> "Context":
        if which == 0:
            self.book = {b: k for k, b in enumerate(FIXED)}
            self.ok = True
        if self.ok:
            for b in _bytes(seqs):
                if b not in self.book:
                    if len(self.book) >= CODE_SYMBOLS:
                        self.ok = False
                        break
                    self.book[b] = len(self.book)
        self.loaded[which] = True
        if which == 0:
            self.loaded[1] = False
        return self

    @property
    def has_gap_symbol(self) -> bool:
        return ord("-") in self.book

    @property
    def symbols(self) -> bytes:
        """The book in code order."""
        return bytes(sorted(self.book, key=self.book.get))


def replay(history) -> Context:
    """history: [(seqs, which), ...] -> the Context after those loads."""
    c = Context()
    for seqs, which in history:
        c.load(seqs, which)
    return c


def final_sets(loads):
    """The alphabets a context holds after `loads` = [(alphabet, which), ...]: (set 0, set 1 or None)."""
    s0 = s1 = None
    for alphabet, which in loads:
        if which == 0:
            s0, s1 = alphabet, None
        else:
            s1 = alphabet
    return s0, s1


# Load histories whose outcome tests/test_gpu_symbols.py compares with a fresh context that holds only
# the final sets (each load is a set of sequences over exactly that alphabet), with the prediction
# (codebook_ok, has_gap_symbol, codes in the book) after the last load.
HISTORIES = [
    dict(id="symbol-only-in-set-1", loads=[(b"ACGT", 0), (b"ACGTRY", 1)], ok=True, gap=False, ncodes=7),
    dict(id="set-1-reloaded-three-times-to-15", loads=[(b"ACGTRYKM", 0), (b"ACGTSW", 1), (b"ACGTBD", 1), (b"ACGTHV", 1)],
         ok=True, gap=False, ncodes=15),
    dict(id="15-across-both-sets", loads=[(b"ACGTNRYKMS", 0), (b"ACGTWBDHV", 1)], ok=True, gap=False, ncodes=15),
    dict(id="16th-only-in-set-1", loads=[(b"ACGTNRYKMS", 0), (b"ACGTWBDHVX", 1)], ok=False, gap=False, ncodes=15),
    dict(id="16th-only-in-set-0", loads=[(b"ACGTRYKMSWBDHVX", 0), (b"ACGT", 1)], ok=False, gap=False, ncodes=15),
    # an overflow caused by set 1 lasts over set-1 reloads: the book is only rebuilt by a set-0 load
    dict(id="overflow-by-set-1-then-plain-set-1", loads=[(b"ACGTNRYKMS", 0), (b"ACGTWBDHVX", 1), (b"ACGT", 1)],
         ok=False, gap=False, ncodes=15),
    dict(id="set-0-reloaded-after-overflow", loads=[(b"ACGTNRYKMS", 0), (b"ACGTWBDHVX", 1), (b"ACGTRY", 0), (b"ACGTK", 1)],
         ok=True, gap=False, ncodes=8),
    dict(id="set-1-unloaded-after-overflow", loads=[(b"ACGTNRYKMS", 0), (b"ACGTWBDHVX", 1), (b"ACGT", 1), (b"ACGTR", 0)],
         ok=True, gap=False, ncodes=6),
    # '-' stays in the book after a set-1 reload without it: the packed walk keeps its gap bookkeeping
    dict(id="gap-symbol-kept-by-the-book", loads=[(b"ACGT", 0), (b"ACGT-", 1), (b"ACGTN", 1)], ok=True, gap=True, ncodes=6),
]


def kernel(ctx: Context, scores, la, lb, form: str = "pairs", options: dict | None = None) -> int:
    """`last_kernel` of a call on a context in state `ctx`: the instance kernel_geometry predicts,
    or the general kernel when the book has overflowed (the packed kernel is refused; the general
    kernel is then chosen as under force_general)."""
    o = dict(options or {})
    if not ctx.ok:
        o["force_general"] = 1
    family = K.instance(scores, la, lb, form, o)[0]
    return 48 if family == "split" else K.CODE[family]


# ---- the same constants, parsed from the sources ----------------------------------------------------
def _find(pattern: str, text: str, name: str, group: int = 1) -> str:
    m = re.search(pattern, text, re.S)
    assert m, f"{name} not found"
    return m.group(group)


def parse_constants(csrc: Path = CSRC) -> dict:
    """The constants and rules the restatement depends on, read from the CUDA sources."""
    common = (csrc / "common.cuh").read_text()
    abi = (csrc / "taxi_abi.cu").read_text()
    load = _find(r"int taxi_load_sequences\(.*?\n\}\n", abi, "taxi_load_sequences", 0)
    elig = _find(r"bool fast16_eligible\(.*?\n\}\n", abi, "fast16_eligible", 0)
    out = {
        "CODE_SYMBOLS": int(_find(r"constexpr int CODE_SYMBOLS = (\d+);", common, "CODE_SYMBOLS")),
        "CODE_PADSYM": int(_find(r"constexpr uint32_t CODE_PADSYM = (\d+)u;", common, "CODE_PADSYM")),
        "FIXED": _find(r'const char\* fixed = "([^"]*)";', load, "fixed symbols").encode(),
    }
    nfixed = int(_find(r"for \(int k = 0; k < (\d+); \+\+k\) c->codebook\[\(unsigned char\)fixed\[k\]\]", load, "fixed loop"))
    out["fixed codes"] = nfixed == len(out["FIXED"]) and f"c->ncodes = {nfixed};" in load
    # the rules themselves, as the restatement reads them
    out["reset on set 0"] = "if (set == 0) {" in load and "c->codebook_ok = true;" in load
    out["overflow rule"] = "if (c->ncodes >= CODE_SYMBOLS) c->codebook_ok = false;" in load
    out["first appearance"] = "c->codebook[bytes[k]] = (int16_t)c->ncodes++;" in load
    out["scan stops at overflow"] = "k < s.total && c->codebook_ok;" in load
    out["set 0 unloads set 1"] = "if (set == 0) c->set[1].loaded = false;" in load
    out["refused on overflow"] = "if (c->force_general || !c->codebook_ok) return false;" in elig
    out["gap symbol from the book"] = "if (ch == '-') f.has_gap_symbol = 1;" in elig and "const int k = c->codebook[ch];" in elig
    return out


def restated_constants() -> dict:
    return {"CODE_SYMBOLS": CODE_SYMBOLS, "CODE_PADSYM": CODE_PADSYM, "FIXED": FIXED, "fixed codes": True,
            "reset on set 0": True, "overflow rule": True, "first appearance": True, "scan stops at overflow": True,
            "set 0 unloads set 1": True, "refused on overflow": True, "gap symbol from the book": True}
