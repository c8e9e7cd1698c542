"""The alignment-free counting kernels against the oracle at the edges of their geometry.

Four kernels fill the alignment-free matrix (count_planes.cuh, count_tc.cuh): the popcount kernel,
the tensor-core kernel with 128- or 64-row tiles and its persistent form; a fifth takes pair lists.
`count_dispatch.py` restates which one a call takes, how many launches it makes and whether JC / K2P
come from the logarithm table.  Every case runs each form that can take it, asserts `last_kernel`
and the launch count the restatement predicts, and checks:
- counts bit for bit against `oracle.count_pairs` (the whole matrix where it is small, else every
  pair of the first and last 128 rows and columns and a seeded sample);
- p / p-gaps bit for bit and JC / K2P within 1e-12 of the oracle;
- the whole matrix bit-identical across the forms, and the pair-list kernel on the checked pairs;
- the metrics bit-identical to `metrics_from_counts` of the same counts in the predicted arithmetic
  form, so that the table decision itself is pinned.

The geometry reached: the persistent kernel with several tiles per CTA (up to 4 SMs + 3 tiles, so
the accumulator ping-pong, its parity and the shared-memory ring phase carried across tiles all
run), bands of 12 x tiles with partial last bands in both tensor-core geometries, k loops of 12 and
18 blocks against 5- and 4-stage rings, row lengths on every 32 / 128 / 160-column boundary, the
table threshold at 1 920 columns, the trim correction far from the row ends, every byte value, the
popcount kernel split over two launches and the tensor-core row limit."""
from __future__ import annotations

import contextlib

import numpy as np
import pytest

import count_dispatch as D
import oracle
from taxi2_b200 import _native as N
from taxi2_b200.engine import pack_strings
from test_gpu_align import assert_metrics_close

pytestmark = pytest.mark.gpu

FORMS = {"popcount": {"count_kernel": 1}, "tc128": {"count_kernel": 2, "tc_tile_x": 128},
         "tc64": {"count_kernel": 2, "tc_tile_x": 64}, "persistent": {"count_kernel": 2, "tc_persistent": 1},
         "default": {}}
DEFAULTS = {"count_kernel": 0, "tc_tile_x": 128, "tc_persistent": 0, "metric_tables": 1}
FULL_LIMIT = 250_000        # pairs: up to here the oracle checks the whole matrix
EDGE = 128                  # else: the first and last EDGE rows and columns ...
SAMPLE = 4000               # ... and this many seeded pairs
SENTINEL = -7

ACGT = np.frombuffer(b"ACGT", dtype=np.uint8)
TRANSITION = np.frombuffer(bytes.maketrans(b"ACGT", b"GTAC"), dtype=np.uint8)
TRANSVERSION = np.frombuffer(bytes.maketrans(b"ACGT", b"CATG"), dtype=np.uint8)

# per form: the largest ntiles / tiles_x / kblocks / tiles per CTA a case ran (printed at the end)
REACHED: dict = {}


@pytest.fixture(scope="module")
def engine():
    import torch
    from taxi2_b200.engine import Engine

    eng = Engine(0)
    eng.sms = torch.cuda.get_device_properties(0).multi_processor_count
    yield eng
    eng.close()
    print("\ngeometry reached (form: ntiles, tiles_x, kblocks, tiles per CTA):")
    for form, r in sorted(REACHED.items()):
        print(f"  {form}: {r['ntiles']}, {r['tiles_x']}, {r['kblocks']}, {r['per_cta']}")


@contextlib.contextmanager
def _options(engine, **opts):
    try:
        for key, value in opts.items():
            engine.set_option(key, value)
        yield
    finally:
        for key, value in DEFAULTS.items():
            engine.set_option(key, value)


def _array(rows):
    return rows if isinstance(rows, tuple) else pack_strings(rows)


class Sets:
    """The loaded x set and y set (None: set 0 serves as both), with the concatenation the oracle reads."""

    def __init__(self, engine, xs, ys=None):
        xd, xo = _array(xs)
        engine.load((xd, xo), 0)
        self.x_set = (len(xo) - 1, int(np.diff(xo).max(initial=0)))
        if ys is None:
            self.y_set, self.yoff = self.x_set, 0
            self.data, self.off = xd, xo
        else:
            yd, yo = _array(ys)
            engine.load((yd, yo), 1)
            self.y_set, self.yoff = (len(yo) - 1, int(np.diff(yo).max(initial=0))), len(xo) - 1
            self.data = np.concatenate([xd, yd])
            self.off = np.concatenate([xo, yo[1:] + xo[-1]])

    def oracle(self, rows, cols):
        return oracle.count_pairs(self.data, self.off, np.asarray(rows, np.int32), (self.yoff + np.asarray(cols)).astype(np.int32))


def _record(pred):
    if pred["kernel"] != "popcount":
        r = REACHED.setdefault(pred["kernel"], dict(ntiles=0, tiles_x=0, kblocks=0, per_cta=0))
        for key in r:
            r[key] = max(r[key], pred[key])


def _count_device(engine, x0, nx, y0, ny, want):
    """count_rect_device into fresh buffers filled with SENTINEL (no count or metric takes that
    value), so that a pair no CTA writes shows instead of an earlier launch's result.
    -> (result, launches)"""
    import torch

    bufs = {key: torch.full((nx * ny, 4), SENTINEL, dtype=dtype, device="cuda")
            for key, dtype in (("counts", torch.int32), ("metrics", torch.float64)) if key in want}
    torch.cuda.synchronize()   # the library's stream does not wait for torch's: the fill must be done first
    before = engine.stats()["launches"]
    engine.count_rect_device(x0, nx, y0, ny, *(bufs[k].data_ptr() if k in bufs else 0 for k in ("counts", "metrics")))
    engine.sync()
    return {k: v.cpu().numpy().reshape(nx, ny, 4) for k, v in bufs.items()}, engine.stats()["launches"] - before


def run_forms(engine, S, x0, nx, y0, ny, forms=tuple(FORMS), metric_tables=1, want=("counts", "metrics")):
    """One device block of the rectangle on each form; asserts the kernel and the launches the
    restatement predicts.  -> ({form: result}, {form: prediction})"""
    out, preds = {}, {}
    for form in forms:
        opts = FORMS[form]
        pred = D.enqueue(nx, ny, S.x_set, S.y_set, engine.sms, metric_tables=metric_tables, **opts)
        with _options(engine, metric_tables=metric_tables, **opts):
            res, launches = _count_device(engine, x0, nx, y0, ny, want)
            got = (engine.last_kernel, launches)
        assert got == (D.CODE[pred["kernel"]], pred["launches"]), (form, pred)
        assert form == "default" or pred["kernel"] == form, (form, pred)
        _record(pred)
        out[form], preds[form] = res, pred
    return out, preds


def _checked_pairs(rng, nx, ny):
    if nx * ny <= FULL_LIMIT:
        r, c = np.divmod(np.arange(nx * ny), ny)
        return r, c
    rows = np.unique(np.concatenate([np.arange(min(EDGE, nx)), np.arange(max(nx - EDGE, 0), nx)]))
    cols = np.unique(np.concatenate([np.arange(min(EDGE, ny)), np.arange(max(ny - EDGE, 0), ny)]))
    a = np.stack(np.meshgrid(rows, np.arange(ny), indexing="ij"), -1).reshape(-1, 2)
    b = np.stack(np.meshgrid(np.arange(nx), cols, indexing="ij"), -1).reshape(-1, 2)
    s = np.stack([rng.integers(0, nx, SAMPLE), rng.integers(0, ny, SAMPLE)], -1)
    p = np.concatenate([a, b, s])
    return p[:, 0], p[:, 1]


def check(engine, S, x0, nx, y0, ny, results, preds, rng, metric_tables=1):
    forms = list(results)
    ref = results[forms[0]]
    for form in forms[1:]:
        assert np.array_equal(results[form]["counts"], ref["counts"]), form
        assert np.array_equal(results[form]["metrics"], ref["metrics"], equal_nan=True), form
    table = preds[forms[0]]["table"]
    assert all(p["table"] == table for p in preds.values())
    pinned = engine.metrics_from_counts(ref["counts"].reshape(-1, 4), table=table)
    assert np.array_equal(ref["metrics"].reshape(-1, 4), pinned, equal_nan=True), "metrics not in the predicted arithmetic form"
    r, c = _checked_pairs(rng, nx, ny)
    want = S.oracle(x0 + r, y0 + c)
    assert np.array_equal(ref["counts"][r, c], want["counts"])
    assert_metrics_close(ref["metrics"][r, c], want["metrics"])
    with _options(engine, metric_tables=metric_tables):
        pairs = engine.count_pairs(x0 + r, y0 + c)
        assert (engine.last_kernel, engine.stats()["launches"]) == (D.CODE["pairs"], 1)
    assert np.array_equal(pairs["counts"], ref["counts"][r, c])
    assert np.array_equal(pairs["metrics"], ref["metrics"][r, c], equal_nan=True)


def run_and_check(engine, S, x0, nx, y0, ny, rng, forms=tuple(FORMS), metric_tables=1):
    results, preds = run_forms(engine, S, x0, nx, y0, ny, forms, metric_tables)
    check(engine, S, x0, nx, y0, ny, results, preds, rng, metric_tables)
    return results, preds


def _rows(rng, n, lo, hi, sub=0.1, gaps=0.04, missing=0.02, ends=40, base=None):
    """Rows of one family (pre-aligned look): a common base with substitutions, '-' and N inside,
    runs of '-' at both ends, lengths in [lo, hi]."""
    if base is None:
        base = ACGT[rng.integers(0, 4, hi)]
    out = []
    for _ in range(n):
        L = int(rng.integers(lo, hi + 1))
        s = base[:L].copy()
        u = rng.random(L)
        hit = u < sub
        s[hit] = ACGT[rng.integers(0, 4, int(hit.sum()))]
        s[(u >= sub) & (u < sub + gaps)] = ord("-")
        s[(u >= sub + gaps) & (u < sub + gaps + missing)] = ord("N")
        lead, trail = (int(v) for v in rng.integers(0, ends + 1, 2))
        s[:lead] = ord("-")
        s[max(L - trail, 0):] = ord("-")
        out.append(s.tobytes())
    return out


# ---- many tiles per persistent CTA --------------------------------------------------------------------
def _split(tiles: int) -> tuple[int, int]:
    """tiles = tiles_x * tiles_y with a few y tiles where the count allows."""
    ty = next(d for d in (5, 4, 3, 2, 1) if tiles % d == 0)
    return tiles // ty, ty


@pytest.mark.parametrize("maxlen", [160, 320], ids=["Lp256", "Lp384"])
@pytest.mark.parametrize("target", ["sms+1", "2sms", "2sms+1", "4sms+3"])
def test_many_tiles_per_persistent_cta(engine, target, maxlen):
    """The persistent kernel's grid is min(tiles, SMs): past SMs tiles a CTA walks several, carrying
    the accumulator set (it & 1), the acc_empty parity and the ring phase kbg from tile to tile.
    k loops of 12 and 18 blocks are not multiples of the 5 stages, so the phase shifts every tile."""
    sms = engine.sms
    tiles = {"sms+1": sms + 1, "2sms": 2 * sms, "2sms+1": 2 * sms + 1, "4sms+3": 4 * sms + 3}[target]
    tx, ty = _split(tiles)
    nx, ny = tx * D.TCP_TX - 17, ty * D.TC_TILE - 51
    rng = np.random.default_rng(tiles * 1000 + maxlen)
    S = Sets(engine, _rows(rng, nx, maxlen - 60, maxlen), _rows(rng, ny, maxlen - 60, maxlen))
    _, preds = run_and_check(engine, S, 0, nx, 0, ny, rng)
    p = preds["persistent"]
    assert p["ntiles"] == tiles and p["grid"] == min(tiles, sms)
    assert p["kblocks"] == (12 if maxlen == 160 else 18) and p["kblocks"] % p["stages"] != 0
    if target == "4sms+3":
        assert p["per_cta"] >= 3 and p["tiles_x"] % D.TC_BAND != 0      # and a partial last band


# ---- bands of the CTA order ---------------------------------------------------------------------------
BAND_NX, BAND_NY = 25 * 128 + 40, 560


@pytest.fixture(scope="module")
def band_sets(engine):
    rng = np.random.default_rng(12)
    return _rows(rng, BAND_NX, 200, 300), _rows(rng, BAND_NY, 150, 330)


@pytest.mark.parametrize("several_y", [False, True], ids=["one_y_tile", "four_y_tiles"])
@pytest.mark.parametrize("tiles_x", [12, 13, 24, 25])
@pytest.mark.parametrize("tx", [128, 64])
def test_bands(engine, band_sets, tx, tiles_x, several_y):
    """tile_origin / band_rows map a CTA to its tile in bands of 12 x tiles, column by column; 13 and
    25 tiles leave a last band of one tile.  The rectangles with several y tiles end on the sets' last
    row and column, so the TMA boxes of the last tiles reach past the sets."""
    S = Sets(engine, *band_sets)
    nx = (tiles_x - 1) * tx + (tx if tiles_x % 2 == 0 else 5)
    ny = 3 * D.TC_TILE + 40 if several_y else 100
    x0, y0 = (BAND_NX - nx, BAND_NY - ny) if several_y else (3, 1)
    rng = np.random.default_rng(tx * 100 + tiles_x)
    _, preds = run_and_check(engine, S, x0, nx, y0, ny, rng)
    p = preds["tc128" if tx == 128 else "tc64"]
    assert p["tiles_x"] == tiles_x and p["tiles_y"] == (4 if several_y else 1)


# ---- row lengths --------------------------------------------------------------------------------------
BOUNDARY_LENGTHS = (0, 1, 31, 32, 33, 127, 128, 129, 159, 160, 161, 255, 256, 257, 1919, 1920, 1921, 2048, 2049)


def test_row_lengths_around_every_boundary(engine):
    """Rows on both sides of every word (32), operand tile (128) and carry-save group (160 columns)
    boundary, mixed in one set, and up to the table threshold and past 2 048."""
    rng = np.random.default_rng(33)
    base = ACGT[rng.integers(0, 4, 2049)]
    rows = []
    for L in BOUNDARY_LENGTHS:
        rows += _rows(rng, 5, L, L, ends=min(L // 3, 70), base=base)
    rng.shuffle(rows)
    S = Sets(engine, rows)
    _, preds = run_and_check(engine, S, 0, len(rows), 0, len(rows), rng)
    assert not preds["popcount"]["table"] and preds["tc128"]["kblocks"] == 6 * D.padded(2049) // 128


@pytest.mark.parametrize("order", ["narrow_x", "wide_x"])
def test_sets_of_different_width(engine, order):
    """Two sets whose W and Lp differ (segment offsets with LpX != LpY; the k loop runs over the
    smaller Lp, the popcount kernel over the smaller W), in both roles."""
    rng = np.random.default_rng(7 if order == "narrow_x" else 8)
    base = ACGT[rng.integers(0, 4, 1100)]
    narrow = _rows(rng, 300, 100, 300, base=base)      # W 10, Lp 384
    wide = _rows(rng, 260, 250, 1100, base=base)       # W 35, Lp 1152
    xs, ys = (narrow, wide) if order == "narrow_x" else (wide, narrow)
    S = Sets(engine, xs, ys)
    assert D.padded(S.x_set[1]) != D.padded(S.y_set[1])
    run_and_check(engine, S, 0, len(xs), 0, len(ys), rng)


# ---- the table threshold ------------------------------------------------------------------------------
def _mutant(rng, base, ts, tv):
    """base with exactly ts transitions and tv transversions at random columns."""
    s = base.copy()
    pos = rng.permutation(len(base))
    s[pos[:ts]] = TRANSITION[s[pos[:ts]]]
    s[pos[ts:ts + tv]] = TRANSVERSION[s[pos[ts:ts + tv]]]
    return s


def _threshold_rows(rng, base, L, n=36):
    """Rows of L columns, all real: base[:L] itself, mutants whose tuple against it sits on or next
    to an exactly-zero logarithm argument (3n = 4d, n = 2 tv, n = 2 ts + tv, and the last two at
    once), random mutants, and a few one column shorter."""
    base = base[:L]
    tuples = []
    for e in (-1, 0, 1):
        tuples += [(3 * L // 4 - L // 4 + e, L // 4),           # 3n = 4d at e = 0
                   (L // 8, L // 2 + e),                          # n = 2 tv
                   ((L - L // 3) // 2 + e, L // 3),               # n = 2 ts + tv
                   ((L - L // 2) // 2 + e, L // 2)]               # both
    rows = [base] + [_mutant(rng, base, ts, tv) for ts, tv in tuples if ts >= 0 and tv >= 0 and ts + tv <= L]
    while len(rows) < n - 3:
        ts, tv = (int(v) for v in rng.integers(0, L // 2, 2))
        rows.append(_mutant(rng, base, ts, tv))
    rows += [r[:L - 1] for r in rows[1:4]]
    return [r.tobytes() for r in rows]


@pytest.mark.parametrize("metric_tables", [1, 0])
@pytest.mark.parametrize("longest", [1920, 1921, 2048, 2049, "1920x2049", "2049x1920"])
def test_table_threshold(engine, longest, metric_tables):
    """The table form is chosen from the smaller W of the two sets: up to 1 920 columns (W = 60), not
    2 048; n reaches the top of the table, and the tuples next to the exactly-zero logarithm
    arguments run through it.  With metric_tables = 0 every set takes the floating-point form."""
    rng = np.random.default_rng([metric_tables, *str(longest).encode()])
    base = ACGT[rng.integers(0, 4, 2049)]
    if isinstance(longest, int):
        S = Sets(engine, _threshold_rows(rng, base, longest))
        expect = metric_tables == 1 and longest <= 1920
    else:
        a, b = (int(v) for v in longest.split("x"))
        S = Sets(engine, _threshold_rows(rng, base, a), _threshold_rows(rng, base, b))
        expect = metric_tables == 1
    nx, ny = S.x_set[0], S.y_set[0]
    results, preds = run_and_check(engine, S, 0, nx, 0, ny, rng, metric_tables=metric_tables)
    assert preds["popcount"]["table"] == expect
    n = results["popcount"]["counts"][..., :3].sum(-1)
    assert n.max() >= min(S.x_set[1], S.y_set[1]) - 1


# ---- the trim correction ------------------------------------------------------------------------------
def _trim_rows(rng):
    """Pairs whose first / last both-real column lies far from the row ends, with gap columns on
    the far side of it (counted by the contraction and removed by gaps_outside_trim)."""
    L = 2000
    rows = []
    # one both-real column, in the last word; x real at both ends with '-' between, y real everywhere but its ends
    x = np.full(L, ord("-"), np.uint8); x[[0, 1990, L - 1]] = ACGT[rng.integers(0, 4, 3)]
    y = ACGT[rng.integers(0, 4, L)]; y[[0, L - 1]] = ord("N")
    rows += [x, y]
    # leading gaps of x over many words while y is real there, and the mirror
    for start, end in ((700, L), (0, 1300), (33, 1967), (700, 701)):
        x = ACGT[rng.integers(0, 4, L)]
        x[:start] = ord("-"); x[end:] = ord("-")
        x[rng.random(L) < 0.02] = ord("-")
        x[[max(start - 200, 0)]] = ord("A")      # real outside the window: the gaps next to it lie inside x's span
        rows.append(x)
    # x real only in the first half and y only in the second: no both-real column, no gap column
    rows.append(np.concatenate([ACGT[rng.integers(0, 4, L // 2)], np.full(L // 2, ord("-"), np.uint8)]))
    rows.append(np.concatenate([np.full(L // 2, ord("-"), np.uint8), ACGT[rng.integers(0, 4, L // 2)]]))
    # interleaved: real where the other has '-', gap columns everywhere, n = 0
    a = np.where(np.arange(L) % 2 == 0, ord("A"), ord("-")).astype(np.uint8)
    rows += [a, np.where(np.arange(L) % 2 == 1, ord("C"), ord("-")).astype(np.uint8)]
    # gap and both-real columns at bit 0 and bit 31 of words
    for first, last in ((32 * 5, 32 * 50 + 31), (32 * 5 + 31, 32 * 50), (32 * 7, 32 * 7), (32 * 7 + 31, 32 * 8)):
        x = np.full(L, ord("-"), np.uint8)
        x[first:last + 1] = ACGT[rng.integers(0, 4, last + 1 - first)]
        x[[0, L - 1]] = ord("G")
        for w in range(0, L // 32, 3):
            x[32 * w + rng.choice([0, 31])] = ord("-") if rng.random() < 0.5 else ord("T")
        rows.append(x)
    # all-gap, all-N and empty rows
    rows += [np.full(L, ord("-"), np.uint8), np.full(L, ord("N"), np.uint8), np.zeros(0, np.uint8),
             np.full(300, ord("-"), np.uint8)]
    # short rows of the same families, so one set also takes the table form
    return [r.tobytes() for r in rows]


@pytest.mark.parametrize("width", [2000, 320])
def test_trim_correction(engine, width):
    """Every constructed row against every other: both-real spans of one column, starting many words
    in, bounded at bit 0 / bit 31; n = 0 with gap columns; all-gap, all-N and empty rows."""
    rng = np.random.default_rng(width)
    rows = [r[:width] for r in _trim_rows(rng)]
    rows += _rows(rng, 20, width // 2, width, gaps=0.2, ends=width // 3)
    S = Sets(engine, rows)
    results, _ = run_and_check(engine, S, 0, len(rows), 0, len(rows), rng)
    c = results["popcount"]["counts"]
    n = c[..., :3].sum(-1)
    assert (n == 1).any() and ((n > 0) & (c[..., 3] > 0)).any()


# ---- every byte value ---------------------------------------------------------------------------------
def test_every_byte_value(engine):
    """base_class folds case with c & 0xDF; every one of the 256 byte values, in the x role and in the
    y role, against A / C / G / T in both cases, '-' and N, must classify as the oracle's switch does."""
    rng = np.random.default_rng(256)
    every = np.arange(256, dtype=np.uint8)
    rows = [np.roll(every, k) for k in range(0, 256, 37)] + [rng.permutation(every) for _ in range(6)]
    al = np.frombuffer(b"ACGTacgt-N", dtype=np.uint8)
    rows += [al[rng.integers(0, len(al), 256)] for _ in range(24)]
    rows += [np.full(256, v, np.uint8) for v in b"AaCcGgTt-N"]
    S = Sets(engine, [r.tobytes() for r in rows])
    run_and_check(engine, S, 0, len(rows), 0, len(rows), rng)
    # and in two sets, so x and y roles read different planes
    S = Sets(engine, [r.tobytes() for r in rows[:13]], [r.tobytes() for r in rows[13:]])
    run_and_check(engine, S, 0, 13, 0, len(rows) - 13, rng)


# ---- dispatch threshold and outputs -------------------------------------------------------------------
@pytest.mark.parametrize("extra", [-1, 0])
def test_default_dispatch_threshold(engine, extra):
    """The default takes the tensor cores from 2 * SMs tiles of 128 x 128 on, the popcount kernel below."""
    tiles = 2 * engine.sms + extra
    rng = np.random.default_rng(tiles)
    nx, ny = tiles * D.TC_TILE - 3, 90
    S = Sets(engine, _rows(rng, nx, 60, 150), _rows(rng, ny, 60, 150))
    _, preds = run_and_check(engine, S, 0, nx, 0, ny, rng, forms=("default", "popcount"))
    assert preds["default"]["kernel"] == ("popcount" if extra < 0 else "tc128")


def test_outputs(engine):
    """Counts only and metrics only on every form equal the halves of a full run (the kernels skip
    different branches of store_pair, and the tensor-core kernels skip the table staging without
    metrics); the same through taxi_count_rect's host buffers; one pair on the tensor cores."""
    rng = np.random.default_rng(48)
    S = Sets(engine, _rows(rng, 400, 100, 300), _rows(rng, 300, 100, 300))
    full, preds = run_and_check(engine, S, 5, 390, 7, 290, rng)
    counts, _ = run_forms(engine, S, 5, 390, 7, 290, want=("counts",))
    metrics, _ = run_forms(engine, S, 5, 390, 7, 290, want=("metrics",))
    for form in FORMS:
        assert "metrics" not in counts[form] and "counts" not in metrics[form]
        assert np.array_equal(counts[form]["counts"], full[form]["counts"]), form
        assert np.array_equal(metrics[form]["metrics"], full[form]["metrics"], equal_nan=True), form
    for form in FORMS:   # the host path: taxi_count_rect downloads each device block
        pred = D.count_rect(390, 290, S.x_set, S.y_set, engine.sms, **FORMS[form])
        with _options(engine, **FORMS[form]):
            got = engine.count_rect(5, 390, 7, 290)
            assert (engine.last_kernel, engine.stats()["launches"]) == (D.CODE[pred["kernel"]], pred["launches"])
        assert np.array_equal(got["counts"], full[form]["counts"]), form
        assert np.array_equal(got["metrics"], full[form]["metrics"], equal_nan=True), form
    run_and_check(engine, S, 399, 1, 299, 1, rng, forms=("tc128", "tc64", "persistent", "popcount"))
    assert preds["tc128"]["table"]


# ---- the popcount launch split and the tensor-core row limit ------------------------------------------
def test_popcount_split_and_tensor_core_row_limit(engine):
    """65535 * 64 + 1 rows against 3 columns: the default runs the popcount kernel (the tensor-core
    kernel refuses more than 65535 64-row tiles) in two launches, the second writing at its own
    offset; 65535 * 64 rows run on the tensor cores, and forcing them one row further is refused."""
    rng = np.random.default_rng(65535)
    limit = 65535 * 64
    n = limit + 1
    lens = rng.integers(32, 41, n)
    off = np.zeros(n + 1, np.int64)
    np.cumsum(lens, out=off[1:])
    data = ACGT[rng.integers(0, 4, int(off[-1]), dtype=np.uint8)]
    data[rng.integers(0, 32, len(data), dtype=np.uint8) == 0] = ord("-")
    ys = [b"A", b"CG", b"GT-"]
    S = Sets(engine, (data, off), ys)
    assert S.x_set[1] <= 40 and D.slab(S.x_set[1], S.y_set[1]) == 64

    big, preds = run_forms(engine, S, 0, n, 0, 3, forms=("default",))
    assert preds["default"]["kernel"] == "popcount" and preds["default"]["launches"] == 2
    rows = np.concatenate([np.arange(64), np.arange(limit - 64, n), rng.integers(0, n, 3000)])
    r, c = np.repeat(rows, 3), np.tile(np.arange(3), len(rows))
    want = S.oracle(r, c)
    assert np.array_equal(big["default"]["counts"][r, c], want["counts"])
    assert_metrics_close(big["default"]["metrics"][r, c], want["metrics"])
    pinned = engine.metrics_from_counts(big["default"]["counts"].reshape(-1, 4), table=preds["default"]["table"])
    assert np.array_equal(big["default"]["metrics"].reshape(-1, 4), pinned, equal_nan=True)
    for x0 in (limit - 1, limit):   # the last row of the first launch and the row of the second
        one, _ = _count_device(engine, x0, 1, 0, 3, ("counts", "metrics"))
        assert np.array_equal(one["counts"][0], big["default"]["counts"][x0])
        assert np.array_equal(one["metrics"][0], big["default"]["metrics"][x0], equal_nan=True)

    tc, preds = run_forms(engine, S, 0, limit, 0, 3, forms=("default",))
    assert preds["default"]["kernel"] == "tc128"
    assert np.array_equal(tc["default"]["counts"], big["default"]["counts"][:limit])
    assert np.array_equal(tc["default"]["metrics"], big["default"]["metrics"][:limit], equal_nan=True)
    del big, tc

    with pytest.raises(D.Refused):
        D.count_rect(n, 3, S.x_set, S.y_set, engine.sms, count_kernel=2)
    with _options(engine, count_kernel=2), pytest.raises(N.TaxiNativeError) as err:
        engine.count_rect(0, n, 0, 3)
    assert err.value.code == N.E_RANGE
