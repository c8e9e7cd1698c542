"""The alignment kernels on any input bytes: every byte value, '-' inside sequences, and the symbol
codebook across loads, against the oracle.

The general kernel reads bytes.  The packed kernel reads 4-bit symbol codes from a codebook the
context builds as sequences are loaded (codebook.py restates the rule), and classifies columns and
writes gapped strings through tables built from that book (`Fast16::class_lut`, `Fast16::ascii`,
`has_gap_symbol` in fast16_eligible).  A stale code, a missing table entry or a wrong gap column
gives wrong distances without any error, so every check here is bit for bit: score, counts and
p / p-gaps against `oracle.align_count_pairs`, JC / K2P within 1e-12, the metrics bit for bit
`taxi_metrics_from_counts` of the kernel's own counts, gapped strings byte for byte against
`oracle.align`, and `last_kernel` against the instance codebook.py and kernel_geometry.py predict.

- Every byte value: the 251 bytes outside ACGTN in groups of at most ten (one book of at most 15
  codes each, packed), lowercase against uppercase, and all 256 at once (more than 15 symbols: the
  general kernel), as pair lists and rectangles, in the x and the y role, packed bottom-aligned,
  packed top-aligned and general.
- '-' inside sequences on every kernel family: general in one stripe and in several, intra-task,
  packed top / bottom / multi-stripe, a row-grouped rectangle and both orientations, on inputs
  aimed at the gap-column bookkeeping of the packed traceback walk.
- Codebook histories: each compared bit for bit with a fresh context holding only the final sets."""
from __future__ import annotations

import numpy as np
import pytest

import codebook as B
import kernel_geometry as K
import oracle
from synth import random_pairs
from test_gpu_kernel_geometries import Options, assert_epilogue, assert_same, tie_set
from test_gpu_packed_exactness import oracle_batch

pytestmark = pytest.mark.gpu

DEFAULT = (1, -1, -8, -1, -1, -1)
MODES = {"bottom": {}, "top": {"force_top": 1}, "general": {"force_general": 1, "no_coop": 1}}
OTHERS = bytes(b for b in range(256) if b not in B.FIXED)
GROUPS = [OTHERS[k:k + 10] for k in range(0, len(OTHERS), 10)] + [b"acgtn"]


@pytest.fixture(scope="module")
def engine():
    from taxi2_b200.engine import Engine

    eng = Engine(0)
    yield eng
    eng.close()


def _pick(rng, alphabet: bytes, n: int) -> bytes:
    al = np.frombuffer(alphabet, dtype=np.uint8)
    return al[rng.integers(0, len(al), max(1, n))].tobytes()


def symbol_pairs(rng, extra: bytes, n: int = 32, lo: int = 8, hi: int = 120) -> tuple[list[bytes], list[bytes]]:
    """Related pairs over ACGT + extra in which every extra symbol appears in matches, mismatches,
    gap runs, leading and trailing end gaps and at the first and last both-real column."""
    xs, ys = random_pairs(rng, n, lo, hi, sub=0.2, indel=0.05, alphabet=b"ACGT" + extra)
    for s in extra:
        c = bytes([s])
        core = _pick(rng, b"ACGT" + extra, int(rng.integers(20, 40)))
        xs += [c * 3 + core + c * 2, core, c + core + c, core[:10] + c * 6 + core[10:], c * 7]
        ys += [core, c * 4 + core + c * 3, b"A" + core + b"T", core, c * 3 + b"ACGT"]
    return xs, ys


def _strings(engine, xs, ys, px, py, want, scores, where):
    ox, oy, start, off, sc, res = engine.align_strings_raw(px, py, want=("counts", "metrics"))
    assert np.array_equal(sc, want["score"]), where
    assert np.array_equal(res["counts"], want["counts"]), where
    assert_epilogue(engine, res, (where, "strings"))
    bx, by = ox.tobytes(), oy.tobytes()
    for k in range(len(px)):
        ax, ay = bx[int(start[k]):int(off[k + 1])], by[int(start[k]):int(off[k + 1])]
        ex, ey, _ = oracle.align(xs[px[k]], ys[py[k]], scores)
        assert (ax, ay) == (ex.encode("latin-1"), ey.encode("latin-1")), (where, k, xs[px[k]], ys[py[k]])


def check_pairs(engine, xs, ys, scores, opts, kernel, where, strings=True):
    """Pair k = (xs[k], ys[k]) with xs loaded as set 0 and ys as set 1."""
    px = np.arange(len(xs), dtype=np.int32)
    want = oracle_batch(xs, ys, px, px, scores)
    with Options(engine, **opts):
        engine.set_scores(scores)
        engine.load(xs, 0)
        engine.load(ys, 1)
        got = engine.align_pairs(px, px)
        assert engine.last_kernel == kernel, (where, engine.last_kernel)
        assert_same(got, want, where)
        assert_epilogue(engine, got, where)
        if strings:
            _strings(engine, xs, ys, px, px, want, scores, where)
    return got


def check_rect(engine, xs, ys, scores, opts, kernel, where):
    nx, ny = len(xs), len(ys)
    px, py = np.divmod(np.arange(nx * ny, dtype=np.int32), ny)
    want = oracle_batch(xs, ys, px, py, scores)
    with Options(engine, **opts):
        engine.set_scores(scores)
        engine.load(xs, 0)
        engine.load(ys, 1)
        got = engine.align_rect(0, nx, 0, ny)
        assert engine.last_kernel == kernel, (where, engine.last_kernel)
    assert_same(got, want, where)
    assert_epilogue(engine, got, where)
    return got


def predicted(loads, scores, la, lb, form, opts) -> int:
    return B.kernel(B.replay(loads), scores, la, lb, form, opts)


# -- every byte value ---------------------------------------------------------------------------------

@pytest.mark.parametrize("extra", GROUPS, ids=lambda g: "-".join(f"{b:02x}" for b in g[:1] + g[-1:]))
def test_every_byte_value(engine, extra):
    rng = np.random.default_rng(extra[0] * 7 + len(extra))
    xs, ys = symbol_pairs(rng, extra)
    rx, ry = symbol_pairs(rng, extra, n=10, lo=20, hi=90)
    rx, ry = rx[:12], ry[-9:]
    for mode, opts in MODES.items():
        for role, (a, b) in (("x", (xs, ys)), ("y", (ys, xs))):
            la, lb = [len(s) for s in a], [len(s) for s in b]
            kernel = predicted([(a, 0), (b, 1)], DEFAULT, la, lb, "pairs", opts)
            assert kernel == {"bottom": 17, "top": 16, "general": 32}[mode]
            check_pairs(engine, a, b, DEFAULT, opts, kernel, (extra, mode, role, "pairs"))
            ra, rb = (rx, ry) if role == "x" else (ry, rx)
            kernel = predicted([(ra, 0), (rb, 1)], DEFAULT, [len(s) for s in ra], [len(s) for s in rb], "rect", opts)
            check_rect(engine, ra, rb, DEFAULT, opts, kernel, (extra, mode, role, "rect"))


def test_lowercase_against_uppercase(engine):
    """'a' vs 'A' is a mismatch in the score and "same" in the counts (base classes fold case)."""
    rng = np.random.default_rng(97)
    xs, _ = random_pairs(rng, 40, 10, 150, sub=0.0, indel=0.0, alphabet=b"ACGT")
    ys = [bytes(c | 0x20 if rng.random() < 0.4 else c for c in x) for x in xs]
    for mode, opts in MODES.items():
        got = check_pairs(engine, xs, ys, DEFAULT, opts, {"bottom": 17, "top": 16, "general": 32}[mode], ("case", mode))
        # where the gapless alignment is the optimum, its lowercase columns cost a mismatch each in the
        # score and every column counts as "same"
        lower = np.array([sum(c >= 0x61 for c in y) for y in ys])
        diagonal = got["score"] == np.array([len(x) for x in xs]) - 2 * lower
        assert diagonal.sum() >= 30 and (lower[diagonal] > 0).sum() >= 30
        assert np.array_equal(got["counts"][diagonal], np.array([[len(x), 0, 0, 0] for x in xs])[diagonal])


def test_all_256_byte_values_run_general(engine):
    rng = np.random.default_rng(256)
    allb = bytes(range(256))
    xs, ys = random_pairs(rng, 24, 30, 200, sub=0.2, indel=0.05, alphabet=allb)
    xs += [allb, allb[::-1], allb[128:] + allb[:128]]
    ys += [allb, allb, allb[::2]]
    assert not B.replay([(xs, 0), (ys, 1)]).ok
    for mode, opts in MODES.items():
        check_pairs(engine, xs, ys, DEFAULT, opts, 32, ("all 256", mode))
        check_rect(engine, xs[-6:], ys[-5:], DEFAULT, opts, 32, ("all 256", mode, "rect"))


# -- '-' inside sequences -----------------------------------------------------------------------------

def gap_pairs(rng, rows: int) -> tuple[list[bytes], list[bytes]]:
    """Pairs with '-' aimed at the gap-column bookkeeping of the packed walk; the longest x and y
    have `rows` symbols."""
    core = _pick(rng, b"ACGT", 60)
    xs, ys = random_pairs(rng, 12, 8, min(rows, 200), sub=0.15, indel=0.05, alphabet=b"ACGT-")  # '-' next to inserted gaps, '-' vs '-'
    pairs = [
        (b"--" + core + b"---", core),                         # '-' before the first and after the last both-real column
        (core, b"-" + core[5:] + b"--"),
        (b"-A" + core + b"T-", b"G" + core + b"C"),
        (core[:25] + b"-" * 40 + core[25:], core),             # a run of '-' longer than one 32-column chunk
        (core[:25] + b"-" * 70 + core[25:], core[:25] + b"-" * 33 + core[25:]),
        (core[:30] + b"N-N--N" + core[30:], core[:30] + b"-NN-" + core[30:]),   # '-' next to N
        (b"-N-N--N", b"N--N"), (b"----", b"NN"), (b"N", b"-"),                 # no both-real column: NaN metrics
    ]
    # '-' in lane 0 and lane 31 of the walk's 32-cell chunks: a gapless pair walked from its end
    walk = bytearray(_pick(rng, b"ACGT", 100))
    for back in (1, 32, 33, 64, 65, 96):
        walk[-back] = ord("-")
    pairs += [(bytes(walk), bytes(walk)), (bytes(walk), _pick(rng, b"ACGT", 100))]
    for x, y in pairs:
        xs.append(x)
        ys.append(y)
    # one pair of the full size: sets the geometry
    x = bytearray(_pick(rng, b"ACGT", rows))
    for at in rng.integers(0, rows, max(1, rows // 40)):
        x[int(at)] = ord("-")
    y = bytearray(x)
    for at in rng.integers(0, rows, max(1, rows // 10)):
        y[int(at)] = ord("ACGT-"[int(rng.integers(0, 5))])
    xs.append(bytes(x))
    ys.append(bytes(y[:rows]))
    return xs, ys


# (family, H, stripes): the longest row of the selecting run that lies within 2 000 rows, and at least
# 200 (the aimed pairs above are up to 170 columns long)
FAMILIES = [("general", 8, "one"), ("general", 12, "several"), ("top", 8, None), ("top", 32, None),
            ("bottom", 8, None), ("bottom", 32, None), ("multi", 21, None), ("multi", 24, None)]


@pytest.mark.parametrize("family,H,stripes", FAMILIES, ids=lambda v: str(v))
def test_gap_symbol_on_every_family(engine, family, H, stripes):
    runs = K.selecting_rows(family, H, DEFAULT, 2000, stripes=stripes)
    rows = runs[0][1]
    assert rows >= 200, runs
    rng = np.random.default_rng(rows * 31 + H)
    xs, ys = gap_pairs(rng, rows)
    opts = K.family_options(family, DEFAULT)
    la, lb = [len(s) for s in xs], [len(s) for s in ys]
    assert K.instance(DEFAULT, la, lb, "pairs", opts)[:2] == (family, H)
    assert B.replay([(xs, 0), (ys, 1)]).has_gap_symbol
    got = check_pairs(engine, xs, ys, DEFAULT, opts, K.CODE[family], (family, H, rows))
    unreal = [k for k, x in enumerate(xs) if x in (b"-N-N--N", b"----", b"N")]
    assert len(unreal) == 3 and np.isnan(got["metrics"][unreal]).all()   # no both-real column


def test_gap_symbol_intra_task(engine):
    H = K.COOP_H[0]
    rows = K.coop_rows(H, 2)
    rng = np.random.default_rng(33)
    xs, ys = gap_pairs(rng, 200)
    x = bytearray(_pick(rng, b"ACGT", rows))
    for at in rng.integers(0, rows, 40):
        x[int(at)] = ord("-")
    xs.append(bytes(x))
    ys.append(bytes(x[300:500]) + b"-" * 40 + bytes(x[600:700]))
    opts = {"force_general": 1}
    assert K.instance(DEFAULT, [len(s) for s in xs], [len(s) for s in ys], "pairs", opts) == ("coop", H, 2)
    check_pairs(engine, xs, ys, DEFAULT, opts, 33, ("coop", H), strings=False)
    with Options(engine, **opts):
        ax, ay, _ = engine.align_strings([len(xs) - 1], [len(xs) - 1])
        assert engine.last_kernel == 33
    assert (ax[0].decode(), ay[0].decode()) == oracle.align(xs[-1], ys[-1], DEFAULT)[:2]


def test_gap_symbol_row_grouped_rectangle(engine):
    """Rows of one and of several packed stripes in one rectangle: several launches over row lists."""
    rng = np.random.default_rng(48)
    xs = [gap_pairs(rng, n)[0][-1] for n in (150, 400, 900, 1100, 1300)]
    ys = [gap_pairs(rng, n)[1][-1] for n in (120, 200, 260)] + [b"-A-C-", b"N-"]
    kernel = predicted([(xs, 0), (ys, 1)], DEFAULT, [len(s) for s in xs], [len(s) for s in ys], "rect", {})
    assert kernel == 48
    check_rect(engine, xs, ys, DEFAULT, {}, 48, "rect 48")


def _with_gaps(rng, seqs, rate=0.05):
    out = []
    for s in seqs:
        b = bytearray(s)
        for at in np.flatnonzero(rng.random(len(b)) < rate):
            b[at] = ord("-")
        out.append(bytes(b))
    return out


def check_both(engine, xs, ys, where):
    """align_rect_both against the oracle in both orientations and against align_rect of the swapped
    sets in a context of its own -> pairs re-aligned."""
    from taxi2_b200.engine import Engine

    nx, ny = len(xs), len(ys)
    la, lb = [len(s) for s in xs], [len(s) for s in ys]
    kernel = 20 if K.instance(DEFAULT, la, lb, "both")[0] == "both" else None
    engine.set_scores(DEFAULT)
    engine.load(xs, 0)
    engine.load(ys, 1)
    xy, yx = engine.align_rect_both(0, nx, 0, ny)
    assert engine.last_kernel == kernel, where
    redo = engine.last_redo
    px, py = np.divmod(np.arange(nx * ny), ny)
    assert_same(xy, oracle_batch(xs, ys, px, py, DEFAULT), (where, "xy"))
    qy, qx = np.divmod(np.arange(nx * ny), nx)
    assert_same(yx, oracle_batch(ys, xs, qy, qx, DEFAULT), (where, "yx"))
    assert_epilogue(engine, xy, (where, "xy"))
    assert_epilogue(engine, yx, (where, "yx"))
    with Engine(0) as other:
        other.load(ys, 0)
        other.load(xs, 1)
        ref = other.align_rect(0, ny, 0, nx)
    for key in ("score", "counts", "metrics"):
        assert np.array_equal(yx[key], ref[key], equal_nan=True), (where, key)
    return redo


def test_gap_symbol_both_orientations(engine):
    rng = np.random.default_rng(20)
    xs = _with_gaps(rng, tie_set(rng, 16, 100, 150))
    ys = _with_gaps(rng, tie_set(rng, 12, 100, 150))
    xs[0] = b"-" * 60 + xs[0][60:]
    ys[0] = ys[0][:80] + b"-" * 50
    assert check_both(engine, xs, ys, "gaps") > 0


# -- codebook histories -------------------------------------------------------------------------------

def history_sets(loads, seed: int) -> list[list[bytes]]:
    """One set of sequences per load, over exactly that load's alphabet; sets of the same kind are
    related pair by pair (set 1 of the k-th sequence mutates set 0 of the k-th)."""
    rng = np.random.default_rng(seed)
    base = [_pick(rng, b"ACGT", int(rng.integers(40, 130))) for _ in range(20)]
    out = []
    for alphabet, _ in loads:
        seqs = []
        for k, b in enumerate(base):
            s = bytearray(b)
            for at in np.flatnonzero(rng.random(len(s)) < 0.15):
                s[at] = alphabet[int(rng.integers(0, len(alphabet)))]
            if k < len(alphabet):                     # every symbol of the alphabet appears
                s[int(rng.integers(0, len(s)))] = alphabet[k]
            cut = int(rng.integers(0, 6))
            seqs.append(bytes(s[cut:]))
        out.append(seqs)
    return out


def run_history(engine, loads, sets):
    for seqs, (_, which) in zip(sets, loads):
        engine.load(seqs, which)


def results(engine, n0, n1, la, lb, ctx, where):
    """Pair list (i, i), the rectangle and gapped strings, each checked against the predicted kernel."""
    px = np.arange(min(n0, n1), dtype=np.int32)
    out = {}
    out["pairs"] = engine.align_pairs(px, px)
    assert engine.last_kernel == B.kernel(ctx, DEFAULT, [la[i] for i in px], [lb[i] for i in px]), (where, "pairs")
    out["rect"] = engine.align_rect(0, n0, 0, n1)
    assert engine.last_kernel == B.kernel(ctx, DEFAULT, la, lb, "rect"), (where, "rect")
    ox, oy, start, off, sc, res = engine.align_strings_raw(px, px, want=("counts", "metrics"))
    out["strings"] = [(ox[start[k]:off[k + 1]].tobytes(), oy[start[k]:off[k + 1]].tobytes()) for k in range(len(px))]
    out["strings-res"] = dict(res, score=sc)
    return out


def assert_identical(a, b, where):
    for form in ("pairs", "rect", "strings-res"):
        for key in ("score", "counts", "metrics"):
            assert np.array_equal(a[form][key], b[form][key], equal_nan=True), (where, form, key)
    assert a["strings"] == b["strings"], where


@pytest.mark.parametrize("h", B.HISTORIES, ids=lambda h: h["id"])
def test_codebook_history(engine, h):
    from taxi2_b200.engine import Engine

    loads = h["loads"]
    sets = history_sets(loads, sum(map(ord, h["id"])))
    ctx = B.replay([(s, which) for s, (_, which) in zip(sets, loads)])
    assert (ctx.ok, ctx.has_gap_symbol, len(ctx.book)) == (h["ok"], h["gap"], h["ncodes"])
    i0 = max(k for k, (_, w) in enumerate(loads) if w == 0)
    i1 = [k for k, (_, w) in enumerate(loads) if w == 1 and k > i0]
    s0 = sets[i0]
    s1 = sets[i1[-1]] if i1 else s0
    la, lb = [len(s) for s in s0], [len(s) for s in s1]
    engine.set_scores(DEFAULT)
    run_history(engine, loads, sets)
    got = results(engine, len(s0), len(s1), la, lb, ctx, h["id"])
    fresh_loads = [(s0, 0)] + ([(s1, 1)] if i1 else [])
    with Engine(0) as fresh:
        run_history(fresh, [(None, w) for _, w in fresh_loads], [s for s, _ in fresh_loads])
        want = results(fresh, len(s0), len(s1), la, lb, B.replay(fresh_loads), (h["id"], "fresh"))
    assert_identical(got, want, h["id"])
    # and the oracle
    px = np.arange(min(len(s0), len(s1)), dtype=np.int32)
    assert_same(got["pairs"], oracle_batch(s0, s1, px, px, DEFAULT), h["id"])
    for k in range(0, len(px), 3):
        ex, ey, _ = oracle.align(s0[k], s1[k], DEFAULT)
        assert got["strings"][k] == (ex.encode("latin-1"), ey.encode("latin-1")), (h["id"], k)


def test_set_1_only_symbols_as_rows_of_the_realigned_pairs(engine):
    """Symbols only set 1 holds (R, Y: codes the book took after set 0 was encoded) in the pairs
    align_rect_both re-aligns with the roles exchanged, set 1 as rows."""
    rng = np.random.default_rng(1)
    xs = tie_set(rng, 16, 100, 150)
    ys = [bytes(b"RY"[int(rng.integers(0, 2))] if rng.random() < 0.05 else c for c in s) for s in tie_set(rng, 12, 100, 150)]
    ctx = B.replay([(xs, 0), (ys, 1)])
    assert ctx.ok and ctx.book[ord("R")] >= 5 and ord("R") not in B.replay([(xs, 0)]).book
    assert check_both(engine, xs, ys, "set-1 symbols") > 0


def test_gap_symbol_branch_against_a_fresh_context(engine):
    """A book that keeps '-' from an earlier set 1 sends gapless input down the has_gap_symbol branch
    of the packed walk; a fresh context takes the other branch.  Same bits, on the bottom-aligned,
    top-aligned and multi-stripe kernels."""
    from taxi2_b200.engine import Engine

    rng = np.random.default_rng(3)
    xs, ys = random_pairs(rng, 40, 10, 300, sub=0.15, indel=0.05, alphabet=b"ACGTN")
    lx, ly = random_pairs(rng, 4, 1100, 1300, sub=0.1, indel=0.02, alphabet=b"ACGT")
    assert B.replay([(xs, 0), (ys + [b"A-C"], 1), (ys, 1)]).has_gap_symbol
    for (a, b), opts, kernel in (((xs, ys), {}, 17), ((xs, ys), {"force_top": 1}, 16), ((lx, ly), {}, 18)):
        px = np.arange(len(a), dtype=np.int32)
        out = []
        for history in ([(a, 0), (b + [b"A-C"], 1), (b, 1)], [(a, 0), (b, 1)]):
            with Engine(0) as eng, Options(eng, **opts):
                eng.set_scores(DEFAULT)
                run_history(eng, history, [s for s, _ in history])
                got = eng.align_pairs(px, px)
                assert eng.last_kernel == kernel
                ox, oy, start, off, sc, res = eng.align_strings_raw(px, px, want=("counts", "metrics"))
                out.append((got, [(ox[start[k]:off[k + 1]].tobytes(), oy[start[k]:off[k + 1]].tobytes()) for k in range(len(px))], res))
        (g1, s1, r1), (g2, s2, r2) = out
        for key in ("score", "counts", "metrics"):
            assert np.array_equal(g1[key], g2[key], equal_nan=True), (kernel, key)
            assert np.array_equal(r1[key], r2[key], equal_nan=True), (kernel, key)
        assert s1 == s2, kernel
        assert_same(g1, oracle_batch(a, b, px, px, DEFAULT), kernel)


def test_two_contexts_of_one_multi_engine(engine):
    """Both contexts of a MultiEngine replay the same history and agree bit for bit with a fresh one."""
    from taxi2_b200.multi import MultiEngine

    for h in (B.HISTORIES[1], B.HISTORIES[5]):
        loads = h["loads"]
        sets = history_sets(loads, 77)
        ctx = B.replay([(s, which) for s, (_, which) in zip(sets, loads)])
        s0, s1 = sets[0], sets[-1]
        la, lb = [len(s) for s in s0], [len(s) for s in s1]
        with MultiEngine([0, 0]) as multi:
            multi.set_scores(DEFAULT)
            for seqs, (_, which) in zip(sets, loads):
                multi.load(seqs, which)
            got = [results(e, len(s0), len(s1), la, lb, ctx, (h["id"], k)) for k, e in enumerate(multi.engines)]
        engine.set_scores(DEFAULT)
        engine.load(s0, 0)
        engine.load(s1, 1)
        want = results(engine, len(s0), len(s1), la, lb, B.replay([(s0, 0), (s1, 1)]), (h["id"], "fresh"))
        for g in got:
            assert_identical(g, want, h["id"])
