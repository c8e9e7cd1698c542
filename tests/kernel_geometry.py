"""Which compiled alignment kernel instance a launch takes, restated in Python (no GPU).

The library compiles one template instance of its alignment kernels per geometry, H = rows per lane
(one stripe = 32 * H rows), and the host picks one per launch from the score set and the longest row
(`pick_H`, the intra-task choice and `enqueue_align` in taxi2_b200/csrc/taxi_abi.cu; the packed rule
is `packed16_rule.fast16`).  The set of instances is parsed from the dispatch tables of that file, so
it follows the source: an instance added there without a test fails tests/test_kernel_geometry.py.
The restatement assumes at most 15 distinct symbols in the loaded sets (more disable the packed
kernel: the library then runs the general one).

Families and the `last_kernel` code that reports each:
    general  gotoh_warp_kernel<H>           32   (int32, one stripe or several)
    coop     gotoh_coop_kernel<H>           33   (intra-task: the stripes of one pair over 12 warps)
    top      gotoh_pair16_kernel<H,0>       16   (packed, top-aligned)
    bottom   gotoh_pair16_kernel<H,1>       17   (packed, bottom-aligned, one stripe)
    multi    gotoh_pair16_kernel<H,2>       18   (packed, bottom-aligned, several stripes)
    both     gotoh_pair16_kernel<H,1,true>  20   (both orientations of a rectangle from one alignment)"""
from __future__ import annotations

import re
from pathlib import Path

import packed16_rule as R

SOURCE = Path(__file__).resolve().parent.parent / "taxi2_b200" / "csrc" / "taxi_abi.cu"

FAMILIES = ("general", "coop", "top", "bottom", "multi", "both")
CODE = {"general": 32, "coop": 33, "top": 16, "bottom": 17, "multi": 18, "both": 20}
TEMPLATE = {"general": "gotoh_warp_kernel<{H}>", "coop": "gotoh_coop_kernel<{H}>", "top": "gotoh_pair16_kernel<{H},0>",
            "bottom": "gotoh_pair16_kernel<{H},1>", "multi": "gotoh_pair16_kernel<{H},2>", "both": "gotoh_pair16_kernel<{H},1,true>"}

SMS = 148                   # B200
COOP_MIN_ROWS = 2 * 32 * 21
COOP_MAX_STRIPES = 1024     # GOTOH_COOP_MAX_STRIPES
WARPS_PER_BLOCK = 4         # GOTOH_WARPS_PER_BLOCK


def name(family: str, H: int) -> str:
    return TEMPLATE[family].format(H=H)


def _table(text: str, decl: str) -> str:
    m = re.search(re.escape(decl) + r"\s*=\s*\{(.*?)\};", text, re.S)
    assert m, f"{decl} not found in {SOURCE.name}"
    return m.group(1)


def parse_tables(path: Path = SOURCE) -> dict:
    """-> {"kH": (...), "general": (...), "coop": (...), "top": ..., "bottom": ..., "multi": ..., "both": ...}:
    the H of every entry of each dispatch table, in table order."""
    text = path.read_text()
    out = {"kH": tuple(int(v) for v in re.findall(r"\d+", _table(text, "const int kH[]")))}
    general, coop = [], []
    for m in re.finditer(r"\{(\d+), occupancy<(\d+)>, launch_gotoh<(\d+)>, TraceGeom<(\d+)>::HB(?:, launch_coop<(\d+)>)?\}",
                         _table(text, "const Dispatch kDispatch[]")):
        h = {int(v) for v in m.groups() if v is not None}
        assert len(h) == 1, f"kDispatch entry mixes geometries: {m.group(0)}"
        general.append(h.pop())
        if m.group(5):
            coop.append(general[-1])
    out["general"], out["coop"] = tuple(general), tuple(coop)
    for family, decl, mode in (("top", "kDispatch16[]", 0), ("bottom", "kDispatch16b[]", 1), ("multi", "kDispatch16m[]", 2)):
        entries = re.findall(r"P16\((\d+), (\d+)\)", _table(text, "const Dispatch " + decl))
        assert all(int(m) == mode for _, m in entries), f"{decl} holds an entry of another mode: {entries}"
        out[family] = tuple(int(h) for h, _ in entries)
    out["both"] = tuple(int(h) for h in re.findall(r"P16S\((\d+)\)", _table(text, "const Dispatch kDispatch16s[]")))
    return out


def compiled_instances(path: Path = SOURCE) -> list[tuple[str, int]]:
    t = parse_tables(path)
    return [(family, h) for family in FAMILIES for h in t[family]]


_T = parse_tables()
KH = _T["kH"]
assert _T["general"] == KH, "kDispatch and kH list different geometries"
COOP_H = _T["coop"]
assert (_T["top"], _T["bottom"], _T["multi"]) == (R.H_ONE, R.H_ONE, R.H_MULTI), "packed16_rule.H_ONE / H_MULTI are out of date"


def _fewest_slots(rows: int, hs, first: int = 32) -> int:
    """Fewest row slots over whole stripes, ties to the larger H."""
    best, best_slots = first, -1
    for h in hs:
        sl = 32 * h
        slots = -(-rows // sl) * sl
        if best_slots < 0 or slots < best_slots or (slots == best_slots and h > best):
            best, best_slots = h, slots
    return best


def pick_H(max_rows: int) -> int:
    return _fewest_slots(max_rows, KH)


def _enqueue(scores, max_rows: int, max_cols: int, npairs: int, la=None, lb=None, sym: bool = False,
             force_general=False, force_top=False, no_coop=False):
    """enqueue_align: -> (family, H, stripes), or None for a "both orientations" launch the packed
    bottom-aligned one-stripe kernel cannot serve (the caller then falls back)."""
    f = None if force_general else R.fast16(scores, max_rows, max_cols, 0, bool(force_top))
    if f is not None and la is not None:
        _, used = R.build_units(la, lb, max(0, f["max_dead"]))
        if used > 0 and f["mode"] != 0:
            assert R.fast16(scores, max_rows, max_cols, used, bool(force_top)) is not None, "host would report a dead-band error"
    if sym:
        if f is None or f["mode"] != 1 or la is not None:
            return None
        return ("both", f["H"], 1)
    if f is not None:
        H, mode = f["H"], f["mode"]
        stripes = -(-(max_rows + 1) // (32 * H)) if mode == 2 else 1
        return ({0: "top", 1: "bottom", 2: "multi"}[mode], H, stripes)
    H = pick_H(max_rows)
    few = npairs * 4 <= SMS * 3 * WARPS_PER_BLOCK
    if not no_coop and max_rows > COOP_MIN_ROWS and few:
        H = _fewest_slots(max_rows, COOP_H, first=H)
    stripes = -(-max_rows // (32 * H))
    if not no_coop and H in COOP_H and 2 <= stripes <= COOP_MAX_STRIPES and few:
        # the launch also needs npairs <= SMS * (resident CTAs per SM of gotoh_warp_kernel<H>), which is
        # at least SMS: beyond that the occupancy decides, and no prediction is made
        if npairs > SMS:
            raise ValueError(f"{npairs} pairs: whether the intra-task kernel runs depends on the occupancy; set no_coop")
        return ("coop", H, stripes)
    return ("general", H, stripes)


def _rect_split(scores, la, ny: int, mc: int, force_general=False, force_top=False) -> bool:
    """taxi_align_rect_device: rows grouped by packed geometry; more than one group after folding
    the small ones -> several launches (last_kernel 48)."""
    if force_general:
        return False
    bottom = scores[3] == scores[5] and not force_top
    K, M = len(R.H_ONE), len(R.H_MULTI)
    rows = [0] * (K + M)
    for n in la:
        k = 0
        while k < K and 32 * R.H_ONE[k] - (1 if bottom else 0) < n:
            k += 1
        if k == K:
            best = 0
            for m, h in enumerate(R.H_MULTI):
                sl = 32 * h
                slots = -(-(n + 1) // sl) * sl
                if best == 0 or slots <= best:
                    best, k = slots, K + m
        rows[k] += 1
    min_pairs = 8 * SMS * 24
    for k in range(K - 1):
        if rows[k] and rows[k] * ny < min_pairs:
            rows[k + 1] += rows[k]
            rows[k] = 0
    fullest = max(range(K, K + M), key=lambda k: (rows[k], -k))
    for k in range(K, K + M):
        if k != fullest and rows[k] and rows[k] * ny < min_pairs:
            rows[fullest] += rows[k]
            rows[k] = 0
    groups = sum(1 for r in rows if r)
    return groups > 1 and R.fast16(scores, min(max(la), 32 * 32 - 1), mc, 0, bool(force_top)) is not None


def instance(scores, la, lb, form: str = "pairs", options: dict | None = None):
    """Kernel instance of one call -> (family, H, stripes).

    form "pairs": taxi_align_pairs / taxi_align_strings, pair k = (la[k] rows, lb[k] columns);
         "rect":  taxi_align_rect of rows of lengths la x columns of lengths lb (("split", 0, 0) when
                  the rows are spread over several packed geometries);
         "both":  taxi_align_rect_both; without the both-orientations kernel, the instance of its
                  second (swapped) launch, which is what last_kernel reports.
    options: force_general, force_top, no_coop (the engine options of the same name)."""
    o = {k: bool(v) for k, v in {"force_general": 0, "force_top": 0, "no_coop": 0, **(options or {})}.items()}
    la, lb = [int(v) for v in la], [int(v) for v in lb]
    mr, mc = max(la), max(lb)
    if form == "pairs":
        assert len(la) == len(lb)
        return _enqueue(scores, mr, mc, len(la), la, lb, **o)
    npairs = len(la) * len(lb)
    if form == "rect":
        if _rect_split(scores, la, len(lb), mc, o["force_general"], o["force_top"]):
            return ("split", 0, 0)
        return _enqueue(scores, mr, mc, npairs, **o)
    if form == "both":
        got = _enqueue(scores, mr, mc, npairs, sym=True, **o) if 2 * min(la) > mr else None
        return got if got is not None else _enqueue(scores, mc, mr, npairs, **o)
    raise ValueError(form)


def redo_instance(scores, la, lb, options: dict | None = None):
    """The re-alignment of a both-orientations call: the listed pairs as a pair list with the roles
    exchanged (rows = their y lengths la, columns = their x lengths lb)."""
    return instance(scores, la, lb, "pairs", options)


# -- which row counts select an instance --------------------------------------------------------------

def family_options(family: str, scores) -> dict:
    """The options under which a single pair reaches `family`: general runs one pair per warp, the
    top-aligned kernel needs force_top when the set is bottom-aligned (ie == ee)."""
    if family == "general":
        return dict(force_general=1, no_coop=1)
    if family == "coop":
        return dict(force_general=1)
    if family == "top":
        return dict(force_top=int(scores[3] == scores[5]))
    return {}


def selecting_rows(family: str, H: int, scores, limit: int = 4096, cols=None, stripes=None) -> list[tuple[int, int]]:
    """Row counts 1..limit whose one-pair launch (rows x cols, cols=None: square) takes the instance
    (family, H) -> maximal runs [(lo, hi), ...].  stripes: only launches of that many stripes, or
    "one" / "several"."""
    opts = family_options(family, scores)
    runs: list[tuple[int, int]] = []
    for r in range(1, limit + 1):
        c = r if cols is None else cols
        if family == "both":
            got = instance(scores, [r], [c], "both", opts)
        else:
            got = instance(scores, [r], [c], "pairs", opts)
        ok = got[:2] == (family, H)
        if ok and stripes is not None:
            ok = {"one": got[2] == 1, "several": got[2] > 1}.get(stripes, got[2] == stripes)
        if ok:
            if runs and runs[-1][1] == r - 1:
                runs[-1] = (runs[-1][0], r)
            else:
                runs.append((r, r))
    return runs


def coop_rows(H: int, stripes: int, scores=None, limit: int = 40000) -> int | None:
    """Smallest row count whose one-pair launch runs the intra-task kernel <H> in `stripes` stripes."""
    scores = scores or (1, -1, -8, -1, -1, -1)
    for r in range(max(1, (stripes - 1) * 32 * H + 1), min(limit, stripes * 32 * H) + 1):
        if instance(scores, [r], [64], "pairs", dict(force_general=1)) == ("coop", H, stripes):
            return r
    return None
