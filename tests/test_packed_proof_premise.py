"""The premise of the packed 16-bit kernel's restricted recurrence, checked on the CPU.

The packed kernel drops Biopython's Ix <-> Iy transitions (a vertical gap right next to a horizontal
one).  The host admits a score set only if four families of linear inequalities hold for every
end / internal typing of the two gap runs (`fast16_eligible`, restated in `packed16_rule.py`).
Here, independently of any GPU:

* every set the rule rejects at the edge of one of its forms has an explicit pair and an
  alignment with adjacent opposite gaps that is co-optimal -- the rejection is necessary;
* for every set the rule accepts, no co-optimal alignment of a few hundred tie-rich pairs uses such
  a transition (a two-layer dynamic programme that counts the transition), and the oracle never
  emits one;
* the restatement reproduces the window edges DESIGN.md §3.2 documents."""
from __future__ import annotations

import itertools

import numpy as np
import pytest

import oracle
import packed16_rule as R
from rescore import best_score, best_score_adjacent_gaps, rescore

SETS = R.score_sets()
ACCEPTED = [s["scores"] for s in SETS if R.restricted_exact(s["scores"])]
EDGE_REJECTED = [s for s in SETS if s["accept"] is False and s["kind"] != "nw"]


def adjacent_opposite_gaps(ax: str, ay: str) -> bool:
    cols = ["x" if a == "-" else ("y" if b == "-" else "m") for a, b in zip(ax, ay)]
    return any({p, q} == {"x", "y"} for p, q in zip(cols, cols[1:]))


def test_generator_covers_both_sides_of_every_form():
    """About 150 sets, the same on every run, with a rejected set ON the edge and an accepted set one
    unit inside it for each of the ten distinct linear forms, at two mismatch levels."""
    assert [s["scores"] for s in R.score_sets()] == [s["scores"] for s in SETS]
    assert 140 <= len(SETS) <= 160 and len({s["scores"] for s in SETS}) == len(SETS)
    for side in ("reject", "accept"):
        kinds = [s["kind"] for s in SETS if s["kind"].startswith(side + ":")]
        assert len(kinds) == 20 and len(set(kinds)) == 10, side
    for s in SETS:
        if s["kind"].startswith(("reject:", "accept:")):
            side, family, typing = s["kind"].split(":")
            value = R.margins(s["scores"])[family, int(typing[0]), int(typing[1])]
            edge = 1 if family == "slope" else 0
            assert value == (edge if side == "reject" else edge - 1), s
        if s["accept"] is not None:
            assert R.restricted_exact(s["scores"]) == s["accept"], s
    specials = {s["kind"] for s in SETS}
    assert {"D=0", "match=0", "io==ie", "nw", "default", "top-aligned", "bottom-aligned"} <= specials
    assert 60 <= len(ACCEPTED) <= 100


def test_rule_reduces_to_four_primary_forms():
    """Every form of the rule is the mean of two of 2*io, 2*eo (< mm) and 2*ie, 2*ee (<= mm), so the
    rule is exactly those four; exhaustively over small sets."""
    for match in range(0, 4):
        for mm in range(-6, match + 1):
            for io, ie, eo, ee in itertools.product(range(-6, 1), repeat=4):
                s = (match, mm, io, ie, eo, ee)
                if not R.is_gotoh(s):
                    continue
                primary = 2 * max(io, eo) < mm and 2 * max(ie, ee) <= mm
                assert R.restricted_exact(s) == primary, s


@pytest.mark.parametrize("case", EDGE_REJECTED, ids=lambda s: f"{s['kind']}{s['scores']}")
def test_rejection_at_the_edge_is_necessary(case):
    """A pair whose optimum is reached by an alignment with a vertical gap next to a horizontal one:
    the restricted recurrence cannot produce it, so admitting the set would change the alignment
    chosen (at the edge of a strict form: a tie) or the score (beyond the slope form)."""
    scores = case["scores"]
    found = R.witness(scores)
    assert found is not None, scores
    x, y, ax, ay = found
    assert ax.replace("-", "") == x and ay.replace("-", "") == y and adjacent_opposite_gaps(ax, ay)
    best = best_score(x, y, scores)
    assert rescore(ax, ay, scores) == best
    assert best_score_adjacent_gaps(x, y, scores) == best


def _tie_rich_pairs(rng, n):
    """Short two-letter pairs (every path ties with many others), half of them with matching G
    flanks so that the gap runs inside are internal."""
    al = np.frombuffer(b"AC", dtype=np.uint8)
    out = []
    for k in range(n):
        x = al[rng.integers(0, 2, int(rng.integers(1, 9)))].tobytes().decode()
        y = al[rng.integers(0, 2, int(rng.integers(1, 9)))].tobytes().decode()
        if k % 2:
            x, y = "G" + x + "G", "G" + y + "G"
        out.append((x, y))
    return out


@pytest.mark.parametrize("scores", ACCEPTED, ids=str)
def test_accepted_sets_keep_opposite_gaps_apart(scores):
    rng = np.random.default_rng(abs(hash(scores)) % 2**32)
    pairs = _tie_rich_pairs(rng, 300)
    for x, y in pairs:
        ax, ay, sc = oracle.align(x, y, scores)
        assert not adjacent_opposite_gaps(ax, ay), (x, y, ax, ay)
    for x, y in pairs[:40]:
        assert best_score_adjacent_gaps(x, y, scores) < best_score(x, y, scores), (x, y)


def test_documented_window_edges():
    """The edges of the 16-bit window and the dead-band budgets DESIGN.md §3.2 lists: last packed
    length for a square pair, x long against y = 1 and y long against x = 1, and the largest
    x-length difference two pairs of one warp unit may have."""
    table = {
        (1, -1, -8, -1, -1, -1): (1981, 1981, 3989, 1331),
        (2, -1, -3, -2, -1, -1): (1024, 1024, 3465, None),      # top-aligned: no dead band
        (3, -2, -6, -2, -3, -2): (767, 767, 1976, 127),
        (5, -4, -10, -4, -4, -4): (424, 424, 973, None),         # 650 bp is beyond its window
        (0, -1, -3, -1, -2, -1): (3999, 3999, 4012, 3348),
    }
    for scores, (square, x_long, y_long, budget) in table.items():
        assert R.last_packed(scores, "square", limit=4500) == square, scores
        assert R.last_packed(scores, "x_long", limit=4500) == x_long, scores
        assert R.last_packed(scores, "y_long", limit=4500) == y_long, scores
        f = R.fast16(scores, 650, 650)
        if budget is None:
            assert f is None or f["mode"] == 0
        else:
            assert f["max_dead"] == budget
    default = (1, -1, -8, -1, -1, -1)
    assert [R.dead_budget(default, L, L) for L in (1800, 1900, 1950, 1981)] == [181, 81, 31, 0]
    assert [R.fast16(default, L, L)["mode"] for L in (1022, 1023, 1024)] == [1, 1, 2]
    assert R.fast16(default, 1024, 1024, force_top=True)["mode"] == 0 and R.fast16(default, 1025, 1025, force_top=True) is None
