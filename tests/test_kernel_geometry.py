"""The compiled alignment kernel instances, and that every one of them has a planned GPU case (no GPU).

The instance set is parsed from the dispatch tables of taxi_abi.cu (kernel_geometry.py); an instance
added there without a case in tests/test_gpu_kernel_geometries.py fails here.  The planned inputs
are generated on the CPU, so this module also checks that each case's inputs select the instance
it is meant for."""
from __future__ import annotations

import pytest

import kernel_geometry as K
import test_gpu_kernel_geometries as G

EXPECTED = {
    "general": (4, 8, 12, 16, 21, 24, 32),
    "coop": (21, 24, 32),
    "top": (8, 12, 16, 21, 24, 32),
    "bottom": (8, 12, 16, 21, 24, 32),
    "multi": (16, 21, 24, 32),
    "both": (8, 12, 16, 21, 24, 32),
}
INSTANCES = K.compiled_instances()
SCORE_SETS = (G.DEFAULT, G.TOP, G.NW, G.WIDE)


def test_parsed_instances_match_the_table():
    t = K.parse_tables()
    assert {f: t[f] for f in EXPECTED} == EXPECTED
    assert t["kH"] == EXPECTED["general"]
    assert len(INSTANCES) == 32


@pytest.mark.parametrize("inst", INSTANCES, ids=lambda i: K.name(*i))
def test_instance_is_planned(inst):
    assert inst in G.planned_instances(), f"{K.name(*inst)} has no case in test_gpu_kernel_geometries.py"


def _reachable(family, H) -> bool:
    if family == "coop":
        return any(K.coop_rows(H, s) is not None for s in G.COOP_STRIPES)
    limit = G.GENERAL_LIMIT if family == "general" else G.PACKED_LIMIT
    return any(K.selecting_rows(family, H, s, limit) for s in SCORE_SETS)


def test_no_instance_is_unreachable():
    """Every compiled instance is selected by some row count under one of the score sets the GPU
    module uses; the ones that are not are named."""
    unreachable = [K.name(*i) for i in INSTANCES if not _reachable(*i)]
    assert unreachable == [], f"instances no length selects: {unreachable}"


@pytest.mark.parametrize("case", G.PLAN["pairs"] + G.PLAN["coop"], ids=lambda c: c["id"])
def test_planned_inputs_select_their_instance(case):
    if case["family"] == "coop":
        xs, ys = G.coop_inputs(case)
        opts = {"force_general": 1}
    else:
        xs, ys, opts = G.pair_inputs(case)
    la, lb = [len(x) for x in xs], [len(y) for y in ys]
    assert max(la) == case["rows"]
    got = K.instance(case["scores"], la, lb, "pairs", opts)
    assert got[:2] == (case["family"], case["H"]), got
    if case["family"] == "coop":
        assert got[2] == case["stripes"]
    # the window: each side of it is touched (1 bp and the full length among the y)
    assert min(lb) == 1 and max(lb) >= min(case["rows"], 300)


@pytest.mark.parametrize("case", G.PLAN["both"], ids=lambda c: c["id"])
def test_both_orientation_sets_select_their_instance(case):
    for kind in ("ties", "coi"):
        xs = G.both_inputs(case, kind, 24)
        lens = [len(x) for x in xs]
        assert 2 * min(lens) > max(lens)
        assert K.instance(G.DEFAULT, lens, lens, "both") == ("both", case["H"], 1)


def test_redo_of_the_two_set_rectangle_runs_multi_stripe():
    xs, ys = G.rect_inputs()
    la, lb = [len(x) for x in xs], [len(y) for y in ys]
    assert K.instance(G.DEFAULT, la, lb, "both") == ("both", 32, 1)
    assert min(lb) >= G.RECT_Y[0] > 1023 and max(lb) <= G.RECT_Y[1]
    for rows in (min(lb), max(lb)):
        assert K.redo_instance(G.DEFAULT, [rows], [max(la)])[0] == "multi"


def test_geometry_choices_documented_in_design():
    """DESIGN.md §3.1 / §3.2: the general kernel runs 513 - 640 rows as H = 4 in five stripes (never H = 4
    in one stripe above 128 rows), its multi-stripe H = 16 starts at 2 433 rows; multi-stripe packed
    H = 16 needs a window past 2 303 rows."""
    assert K.selecting_rows("general", 4, G.DEFAULT, 2048, stripes="one") == [(1, 128)]
    assert K.instance(G.DEFAULT, [600], [600], "pairs", {"force_general": 1, "no_coop": 1}) == ("general", 4, 5)
    assert K.selecting_rows("general", 4, G.DEFAULT, 640, stripes="several") == [(513, 640)]
    assert K.selecting_rows("general", 16, G.DEFAULT, 2560, stripes="several")[0][0] == 2433
    assert K.selecting_rows("multi", 16, G.DEFAULT, G.PACKED_LIMIT) == []
    assert K.selecting_rows("multi", 16, G.WIDE, G.PACKED_LIMIT)[0] == (2304, 2559)
