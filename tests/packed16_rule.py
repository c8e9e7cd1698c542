"""Python restatement of the host rule that admits the packed 16-bit kernel (`fast16_eligible` and
`build_units` in taxi2_b200/csrc/taxi_abi.cu), plus a seeded generator of score sets placed on both
sides of every inequality of the rule.

The restatement only LOCATES inputs (the last packed length, the dead-band budget); whether the
kernel is right there is decided by the oracle.  The GPU tests also assert that it predicts the
kernel the library picked, so a change of the rule in one place and not the other fails loudly.

Score sets are (match, mismatch, internal open, internal extend, end open, end extend)."""
from __future__ import annotations

import numpy as np

# one-stripe geometries (rows per lane) of the packed kernel, and the multi-stripe ones
H_ONE = (8, 12, 16, 21, 24, 32)
H_MULTI = (16, 21, 24, 32)
BIAS = (65535 - 256) // 16 * 16

# the four inequality families of the restricted recurrence; "strict" ones must be < 0, the slope <= 0
FAMILIES = ("a_gt_b", "b_gt_a", "a_eq_b", "slope")
TYPING = ((0, 0), (0, 1), (1, 0), (1, 1))        # (tx, ty): 0 = internal, 1 = end gap


def _cdiv(a: int, b: int) -> int:
    """C++ integer division (truncates toward zero)."""
    q = abs(a) // abs(b)
    return q if (a >= 0) == (b > 0) else -q


def is_gotoh(scores) -> bool:
    _, _, io, ie, eo, ee = scores
    return not (io == ie and eo == ee)


def margins(scores) -> dict:
    """(family, tx, ty) -> left-hand side of the inequality; O / E indexed by typing."""
    _, mm, io, ie, eo, ee = scores
    O, E = (io, eo), (ie, ee)
    out = {}
    for tx, ty in TYPING:
        out["slope", tx, ty] = E[tx] + E[ty] - mm
        out["a_gt_b", tx, ty] = O[tx] + E[ty] - mm
        out["b_gt_a", tx, ty] = O[ty] + E[tx] - mm
        out["a_eq_b", tx, ty] = O[tx] + O[ty] - mm
    return out


def holds(family: str, value: int) -> bool:
    return value <= 0 if family == "slope" else value < 0


def restricted_exact(scores) -> bool:
    """Part one of the rule: no co-optimal path can put a vertical gap next to a horizontal one."""
    match, mm, io, ie, eo, ee = scores
    if not is_gotoh(scores) or match < mm or match < 0 or max(io, ie, eo, ee) > 0:
        return False
    return all(holds(f, v) for (f, _, _), v in margins(scores).items())


def fast16(scores, max_rows: int, max_cols: int, dead_extra: int = 0, force_top: bool = False):
    """-> None (general kernel) or dict(mode, H, max_dead, neg, room); same arithmetic as the host."""
    if not restricted_exact(scores):
        return None
    match, mm, io, ie, eo, ee = scores
    D = match - mm
    bottom = ie == ee and not force_top
    H, mode, R = 0, (1 if bottom else 0), 0
    for h in H_ONE:
        if 32 * h >= max_rows + (1 if bottom else 0):
            H, R = h, 32 * h
            break
    if not H:
        if not bottom:
            return None
        mode = 2
        for h in H_MULTI:
            sl = 32 * h
            slots = (max_rows + 1 + sl - 1) // sl * sl
            if R == 0 or slots < R or (slots == R and h > H):
                R, H = slots, h
    if D > 2000:
        return None
    D16 = 16 * D
    PoX, PeX, PeoX, PeeX = 16 * (match - io), 16 * (match - ie), 16 * (match - eo), 16 * (match - ee)
    PoY, PeY, PeoY, PeeY = -16 * io, -16 * ie, -16 * eo, -16 * ee
    if mode != 0:
        R = max_rows
    C = max_cols
    pen_e = max(PeX, PeeX, PeY, PeeY)
    pen_o = max(PoX, PeoX, PoY, PeoY)
    if pen_o > 3000 or pen_e > 3000:
        return None
    m = min(R, C)
    corner_v = PeoX + R * PeeX
    corner_h = PeoY + C * PeeY
    corner_d = m * D16 + (PeoX + (R - C) * PeeX if R > C else PeoY + (C - R) * PeeY)
    lower = max(corner_v, corner_h, corner_d) + pen_o + pen_e
    dead_step = max(D16, PeX, PeeX, 16)
    dead_fixed = pen_o + pen_e + D16 + 512 + 15
    room = BIAS - lower - 256
    max_dead = (1 << 40) if mode == 0 else _cdiv(room - dead_fixed, dead_step) - H
    neg = ((H if mode == 0 else H + dead_extra) * dead_step + dead_fixed) // 16 * 16
    if neg > room:
        return None
    return dict(mode=mode, H=H, max_dead=max_dead, neg=neg, room=room)


def build_units(la, lb, max_dead: int) -> tuple[list[tuple[int, int]], int]:
    """Pair-list warp units as the host forms them -> (units, largest x-length difference used)."""
    order = sorted(range(len(la)), key=lambda k: (-la[k], -lb[k]))   # stable, like std::stable_sort
    units, used, k = [], 0, 0
    while k < len(order):
        p0 = order[k]
        if k + 1 < len(order) and la[p0] - la[order[k + 1]] <= max_dead:
            p1 = order[k + 1]
            used = max(used, la[p0] - la[p1])
            units.append((p0, p1))
            k += 2
        else:
            units.append((p0, p0))
            k += 1
    return units, used


def predict_pairs(scores, la, lb, force_top: bool = False, force_general: bool = False) -> int:
    """Kernel code a pair-list alignment takes: 16 / 17 / 18 packed, 32 general (33 = its intra-task
    form is not predicted here: callers accept 32 or 33 for 32)."""
    if force_general:
        return 32
    f = fast16(scores, max(la), max(lb), 0, force_top)
    if f is None:
        return 32
    _, used = build_units(la, lb, max(0, f["max_dead"]))
    if used > 0 and f["mode"] != 0:
        assert fast16(scores, max(la), max(lb), used, force_top) is not None, "host would report an internal dead-band error"
    return 16 + f["mode"]


def predict_rect(scores, row_len: int, col_lens, force_top: bool = False) -> int:
    """Kernel code of a rectangle whose rows all have the same length (one geometry: one launch)."""
    f = fast16(scores, row_len, max(col_lens), 0, force_top)
    return 32 if f is None else 16 + f["mode"]


def last_packed(scores, shape: str, force_top: bool = False, small: int = 1, limit: int = 6000) -> int:
    """Largest L packed for one pair of the given shape ("square": L x L, "x_long": L x small,
    "y_long": small x L), scanning every length; 0 if none."""
    last = 0
    for L in range(1, limit + 1):
        rows, cols = {"square": (L, L), "x_long": (L, small), "y_long": (small, L)}[shape]
        if fast16(scores, rows, cols, 0, force_top) is not None:
            last = L
    return last


def dead_budget(scores, max_rows: int, max_cols: int) -> int:
    f = fast16(scores, max_rows, max_cols)
    assert f is not None and f["mode"] != 0
    return f["max_dead"]


# -- score sets ------------------------------------------------------------------------------------

def _base_ok(s) -> bool:
    match, mm, io, ie, eo, ee = s
    return is_gotoh(s) and mm <= match and match >= 0 and max(io, ie, eo, ee) <= 0


def _same_form(a, b) -> bool:
    """Two (family, tx, ty) keys that name the same linear form (a_gt_b at (tx, ty) == b_gt_a at (ty, tx);
    the a_eq_b and slope families are symmetric in tx, ty)."""
    fa, xa, ya = a
    fb, xb, yb = b
    if {fa, fb} == {"a_gt_b", "b_gt_a"}:
        return (xa, ya) == (yb, xb)
    if fa == fb and fa in ("a_eq_b", "slope"):
        return sorted((xa, ya)) == sorted((xb, yb))
    return fa == fb and (xa, ya) == (xb, yb)


def _form_keys(family, tx, ty):
    return [k for k in margins((1, -1, -8, -1, -1, -1)) if _same_form(k, (family, tx, ty))]


def score_sets(seed: int = 2026) -> list[dict]:
    """About 150 integer score sets, deterministic: dict(scores, kind, accept) where `accept` is
    what the rule must decide (None for random sets: whatever it decides is then checked)."""
    rng = np.random.default_rng(seed)
    out: list[dict] = []
    seen: set = set()

    def add(s, kind, accept):
        s = tuple(int(v) for v in s)
        if s in seen:
            return
        seen.add(s)
        if accept is not None:
            assert restricted_exact(s) == accept, (s, kind)
        out.append(dict(scores=s, kind=kind, accept=accept))

    # random small sets: match 0..6, mismatch <= match, gap scores -12..0
    while len(out) < 90:
        match = int(rng.integers(0, 7))
        s = (match, int(rng.integers(-12, match + 1)), *(int(v) for v in rng.integers(-12, 1, 4)))
        if is_gotoh(s):
            add(s, "random", None)

    # both sides of every distinct linear form of the rule, each at two mismatch levels.  The rule
    # reduces to its four "primary" forms (2 io, 2 eo < mm and 2 ie, 2 ee <= mm): every other form
    # is the mean of two primary ones, so it can only reach its edge when a primary form sits on its
    # own edge too.  Those sets are taken with the other forms AT their edges (never beyond), the
    # primary ones with every other form strictly inside.
    O, E = (2, 4), (3, 5)
    forms = []
    for family in FAMILIES:
        for tx, ty in TYPING:
            keys = _form_keys(family, tx, ty)
            if not any(set(keys) == set(f[1]) for f in forms):
                forms.append(((family, tx, ty), keys))
    for (family, tx, ty), keys in forms:
        i, j = {"a_gt_b": (O[tx], E[ty]), "b_gt_a": (O[ty], E[tx]), "a_eq_b": (O[tx], O[ty]), "slope": (E[tx], E[ty])}[family]
        edge = 1 if family == "slope" else 0          # first violating value of the form
        for level in range(2):
            for side, value in (("reject", edge), ("accept", edge - 1)):
                found = None
                for attempt in range(40000):
                    match = int(rng.integers(0, 7))
                    mm = int(rng.integers(-2, match + 1)) if level == 0 else int(rng.integers(-9, -2))
                    s = [match, mm, *(int(v) for v in rng.integers(-12, 1, 4))]
                    if i == j:
                        if (value + mm) % 2:
                            continue
                        s[i] = (value + mm) // 2
                    else:
                        s[j] = value + mm - s[i]
                    s = tuple(s)
                    if not _base_ok(s) or min(s[2:]) < -12 or s in seen:
                        continue
                    mg = margins(s)
                    assert mg[keys[0]] == value
                    strict = attempt < 20000
                    if all(holds(k[0], v) if strict else v <= (1 if k[0] == "slope" else 0)
                           for k, v in mg.items() if k not in keys):
                        found = s
                        break
                assert found is not None, (family, tx, ty, side, level)
                add(found, f"{side}:{family}:{tx}{ty}", side == "accept")

    # special cases
    for s, kind in [
        ((1, 1, -3, -1, -2, -1), "D=0"), ((3, 3, -6, -2, -3, -2), "D=0"), ((0, 0, -2, -1, -1, -1), "D=0 match=0"),
        ((0, -1, -3, -1, -2, -1), "match=0"), ((0, -2, -5, -1, -3, -1), "match=0"), ((0, -1, -4, -2, -4, -1), "match=0"),
        ((1, -1, -8, -1, -1, -1), "default"), ((2, -1, -3, -2, -1, -1), "top-aligned"), ((3, -2, -6, -2, -3, -2), "bottom-aligned"),
        ((1, -1, -2, -2, -3, -1), "io==ie"), ((2, -2, -4, -4, -3, -2), "io==ie"), ((1, -2, -3, -3, -4, -2), "io==ie"),
        ((1, -1, -1, -1, -1, -1), "nw"), ((1, 0, 0, 0, 0, 0), "nw"), ((2, -3, -4, -4, -4, -4), "nw"), ((1, -1, -3, -3, -2, -2), "nw"),
        ((0, -1, -1, -1, -2, -2), "nw"),
    ]:
        add(s, kind, False if kind == "nw" else None)
    return out


def witness(scores, max_run: int = 10):
    """An explicit pair and alignment with a vertical gap next to a horizontal one whose score is
    the optimum, for a score set the rule rejects at the edge of one of its forms: flanks of
    matching G, a core of a x-only A run and a y-only C run (the all-mismatch worst case of the
    rule), in either order, flanks present or not (end / internal typing).  -> (x, y, ax, ay) or None."""
    from rescore import best_score, rescore

    # short runs of any two lengths first, then long runs of equal length (a slope of +1 per column
    # pair only beats the two gap openings after many columns)
    runs = [(a, t - a) for t in range(2, 2 * max_run + 1) for a in range(max(1, t - max_run), min(max_run, t - 1) + 1)]
    for a, b in runs + [(a, a) for a in range(max_run + 1, 4 * max_run)]:
        for left in (0, 1, 2):
            for right in (0, 1, 2):
                L, Rt = "G" * left, "G" * right
                x, y = L + "A" * a + Rt, L + "C" * b + Rt
                best = best_score(x, y, scores)
                for ax, ay in ((L + "A" * a + "-" * b + Rt, L + "-" * a + "C" * b + Rt),
                               (L + "-" * b + "A" * a + Rt, L + "C" * b + "-" * a + Rt)):
                    if rescore(ax, ay, scores) == best:
                        return x, y, ax, ay
    return None
