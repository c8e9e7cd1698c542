"""Native batch formatter / aggregator (host C++, no GPU) against the Python handlers it replaces:
same bytes in the files, same fp64 aggregates, for several float formats incl. NaN / masked values."""
from __future__ import annotations

from math import inf, isnan

from pathlib import Path

import numpy as np
import pytest

from taxi2_b200 import fastwrite as fw
from taxi2_b200.distances import Distance, DistanceHandler, DistanceMetric
from taxi2_b200.sequences import Sequence

METRICS = [DistanceMetric.Uncorrected(), DistanceMetric.UncorrectedWithGaps(), DistanceMetric.JukesCantor(), DistanceMetric.Kimura2P()]


def make_block(nx, ny, seed=0):
    rng = np.random.default_rng(seed)
    m = rng.random((nx, ny, 4))
    m[rng.random((nx, ny, 4)) < 0.1] = np.nan
    # values that sit exactly on decimal rounding ties in binary (0.03125 -> "0.0312", 0.5, 0.125 ...)
    m[0, 0] = [0.03125, 0.5, 0.125, 0.09375]
    m[0, 1 % ny] = [0.0, 1.0, 2.5, 1e-7]
    undefined = (rng.random((nx, ny)) < 0.1).astype(np.uint8)
    undefined[0, 0] = undefined[0, 1 % ny] = 0
    xs = [Sequence(f"x{i}", None, {"voucher": f"v{i}", "organism": None if i % 3 == 0 else f"Genus{i % 2} sp{i % 5}"}) for i in range(nx)]
    ys = [Sequence(f"y{j}", None, {"voucher": f"w{j}", "organism": f"Genus{j % 2} sp{j % 4}"}) for j in range(ny)]
    return m, undefined, xs, ys


def value(m, undefined, i, j, c, scale):
    v = m[i, j, c]
    return None if (undefined[i, j] or isnan(v)) else v * scale


@pytest.mark.parametrize("spec,scale,missing", [("{:.4f}", 1.0, "NA"), ("{:f}", 100.0, "nan"), ("{:.2e}", 1.0, "NA"), ("{:.0f}", 100.0, "-")])
def test_linear_and_matrix_rows_match_the_python_handlers(tmp_path, spec, scale, missing):
    nx, ny = 7, 5
    m, undefined, xs, ys = make_block(nx, ny)
    fmt = fw.printf_format(spec)
    cols = [0, 1, 2, 3]
    # Python handlers (the reference's writer logic)
    want_linear, want_matrix = tmp_path / "want.linear", tmp_path / "want.matrix"
    with DistanceHandler.Linear.WithExtras(want_linear, "w", missing=missing, formatter=spec) as lin, \
            DistanceHandler.Matrix(want_matrix, "w", missing=missing, formatter=spec) as mat:
        for i in range(nx):
            for j in range(ny):
                for c, metric in zip(cols, METRICS):
                    d = Distance(metric, xs[i], ys[j], value(m, undefined, i, j, c, scale))
                    lin.write(d)
                    if c == 2:
                        mat.write(d)
    # native: header in Python, rows from the library, in two blocks with a row offset
    got_linear, got_matrix = tmp_path / "got.linear", tmp_path / "got.matrix"
    fill = lambda s: [missing if v is None else v for v in s.extras.values()]  # noqa: E731
    xt = fw.StringTable(["\t".join([s.id, *fill(s)]) for s in xs])
    yt = fw.StringTable(["\t".join([s.id, *fill(s)]) for s in ys])
    xid = fw.StringTable([s.id for s in xs])
    got_linear.write_text("\t".join(["seqid (query)", "voucher (query)", "organism (query)", "seqid (reference)", "voucher (reference)",
                                     "organism (reference)", "p", "p-gaps", "jc", "k2p"]) + "\n")
    got_matrix.write_text("\t".join(["", *(s.id for s in ys)]) + "\n")
    for x0, rows in ((0, 3), (3, 4)):
        blk, und = m[x0:x0 + rows], np.ascontiguousarray(undefined[x0:x0 + rows])
        fw.format_pairs(got_linear, [fw.SEG_X[0], fw.SEG_Y[0], fw.SEG_SCORES], [xt], [yt], x0, rows, ny, blk, und, cols, scale, fmt, missing, threads=3)
        fw.format_matrix(got_matrix, xid, x0, rows, ny, blk, und, 2, scale, fmt, missing, threads=2)
    assert got_linear.read_bytes() == want_linear.read_bytes()
    assert got_matrix.read_bytes() == want_matrix.read_bytes()


def test_unsupported_format_specs_fall_back():
    assert fw.printf_format("{:.4f}") == "%.4f" and fw.printf_format("{:f}") == "%f" and fw.printf_format("{:.3e}") == "%.3e"
    assert fw.printf_format("{:>10.4f}") is None and fw.printf_format("{:.2%}") is None and fw.printf_format("{}") is None


def test_subset_aggregation_matches_the_reference_order_and_sums():
    nx, ny = 9, 8
    m, undefined, xs, ys = make_block(nx, ny, seed=3)
    names = {}
    ident = lambda name: names.setdefault(name, len(names))  # noqa: E731
    xsub = np.array([ident(s.extras["organism"]) for s in xs], dtype=np.int32)
    ysub = np.array([ident(s.extras["organism"]) for s in ys], dtype=np.int32)
    state = fw.NativeSubsetState(len(names))
    for x0, rows in ((0, 4), (4, 5)):
        state.add_block(m[x0:x0 + rows], np.ascontiguousarray(undefined[x0:x0 + rows]), x0, rows, ny, 1, 100.0, xsub, ysub)
    want = {}
    for i in range(nx):
        for j in range(ny):
            a = want.setdefault((int(xsub[i]), int(ysub[j])), [0.0, inf, 0.0, 0])
            v = value(m, undefined, i, j, 1, 100.0)
            if v is not None:
                a[0] += v; a[1] = min(a[1], v); a[2] = max(a[2], v); a[3] += 1
    got = list(state.items())
    assert [k for k, _ in got] == list(want)                       # insertion order of the reference's dict
    for (key, (mn, mx, mean, n)) in got:
        s = want[key]
        assert n == s[3]
        if n:
            assert (mn, mx, mean) == (s[1], s[2], s[0] / s[3])      # bit-identical fp64


def test_comparison_type_column(tmp_path):
    nx, ny = 4, 4
    m, undefined, xs, ys = make_block(nx, ny, seed=5)
    genus = np.array([0, 0, 1, -1], dtype=np.int32)
    species = np.array([0, 1, 2, -1], dtype=np.int32)
    xid = fw.StringTable([s.id for s in xs])
    yid = fw.StringTable([s.id for s in ys])
    for g, s in ((genus, species), (None, species), (genus, None), (None, None)):
        out = tmp_path / "types.tsv"
        out.write_text("")
        fw.format_pairs(out, [fw.SEG_X[0], fw.SEG_Y[0], fw.SEG_COMPARISON], [xid], [yid], 0, nx, ny, m, None, [0], 1.0, "%.4f", "NA",
                        xgenus=g, xspecies=s, ygenus=g, yspecies=s, threads=1)
        rows = [line.split("\t") for line in out.read_text().splitlines()]
        for r, (i, j) in zip(rows, ((i, j) for i in range(nx) for j in range(ny))):
            sg = None if g is None else bool(g[i] == g[j])
            ss = None if s is None else bool(s[i] == s[j])
            want = {(None, None): "no info", (None, True): "intra-species", (None, False): "inter-species",
                    (False, None): "inter-genus", (False, True): "inter-genus", (False, False): "inter-genus",
                    (True, None): "intra-genus", (True, True): "intra-species", (True, False): "inter-species"}[(sg, ss)]
            assert r == [xs[i].id, ys[j].id, want]


def test_aligned_pair_records_match_the_python_handler(tmp_path):
    """taxi_format_aligned_pairs against SequencePairHandler.Formatted (and the reference's own
    fixture tests/test_pairs/simple.formatted): same bytes, across two blocks and several threads."""
    from taxi2_b200.pairs import SequencePair, SequencePairHandler

    rng = np.random.default_rng(8)
    nx, ny = 5, 4
    xs = [Sequence(f"x{i}", None) for i in range(nx)]
    ys = [Sequence(f"id {j}", None) for j in range(ny)]
    al = np.frombuffer(b"ACGTN-", dtype=np.uint8)
    pairs, slots = [], []
    for i in range(nx):
        for j in range(ny):
            length = int(rng.integers(1, 40))
            ax = al[rng.integers(0, 6, length)].tobytes()
            ay = al[rng.integers(0, 6, length)].tobytes()
            pairs.append((ax, ay))
            slots.append(length + int(rng.integers(0, 9)))          # right-aligned in a larger slot
    off = np.concatenate([[0], np.cumsum(slots)]).astype(np.int64)
    start = np.array([off[k + 1] - len(pairs[k][0]) for k in range(len(pairs))], dtype=np.int64)
    ox = np.full(int(off[-1]), ord("?"), dtype=np.uint8)
    oy = np.full(int(off[-1]), ord("?"), dtype=np.uint8)
    for k, (ax, ay) in enumerate(pairs):
        ox[start[k]:off[k + 1]] = np.frombuffer(ax, dtype=np.uint8)
        oy[start[k]:off[k + 1]] = np.frombuffer(ay, dtype=np.uint8)
    want = tmp_path / "want.txt"
    with SequencePairHandler.Formatted(want, "w") as file:
        for k, (ax, ay) in enumerate(pairs):
            file.write(SequencePair(Sequence(xs[k // ny].id, ax.decode()), Sequence(ys[k % ny].id, ay.decode())))
    got = tmp_path / "got.txt"
    got.write_bytes(b"")
    xid, yid = fw.StringTable([s.id for s in xs]), fw.StringTable([s.id for s in ys])
    first = True
    for x0, rows in ((0, 2), (2, 3)):
        lo, hi = x0 * ny, (x0 + rows) * ny
        # a block's arrays start at its own first pair, like a fresh align_strings_raw call
        boff = off[lo:hi + 1] - off[lo]
        bstart = start[lo:hi] - off[lo]
        fw.format_aligned_pairs(got, first, xid, yid, x0, rows, ny, ox[off[lo]:off[hi]].copy(), oy[off[lo]:off[hi]].copy(),
                                np.ascontiguousarray(bstart), np.ascontiguousarray(boff), threads=3)
        first = False
    assert got.read_bytes() == want.read_bytes()
    # the reference's fixture, through the same entry point
    fixture = [("id1", "id2", b"ATC-", b"ATG-"), ("id1", "id3", b"ATC-", b"-TAA"), ("id2", "id3", b"ATG-", b"-TAA")]
    out = tmp_path / "fixture.txt"
    out.write_bytes(b"")
    for k, (idx, idy, ax, ay) in enumerate(fixture):
        fw.format_aligned_pairs(out, k == 0, fw.StringTable([idx]), fw.StringTable([idy]), 0, 1, 1, np.frombuffer(ax, dtype=np.uint8).copy(),
                                np.frombuffer(ay, dtype=np.uint8).copy(), np.zeros(1, dtype=np.int64), np.array([0, 4], dtype=np.int64))
    assert out.read_bytes() == (Path(__file__).parent / "golden" / "pairs_simple.formatted").read_bytes()


def test_aligned_pair_records_on_every_byte_value(tmp_path):
    """Gapped strings over every byte 0x01-0xFF (ASCII ids): the library writes the UTF-8 text of
    the latin-1 symbols, byte for byte what SequencePairHandler.Formatted writes for the decoded str
    (0xC9 'É' -> C3 89), with one pattern character per symbol; ASCII records stay as they are."""
    from taxi2_b200.pairs import SequencePair, SequencePairHandler

    rng = np.random.default_rng(255)
    every = np.arange(1, 256, dtype=np.uint8)
    pairs = [(every.tobytes(), every.tobytes()), (every.tobytes(), every[::-1].tobytes()),
             (b"AC\xc9GT-", b"AC\xc9G-T"), (b"ACGT", b"AC-T")]
    for _ in range(6):
        n = int(rng.integers(1, 300))
        pairs.append((every[rng.integers(0, 255, n)].tobytes(), every[rng.integers(0, 255, n)].tobytes()))
    ny = 2
    nx = len(pairs) // ny
    slots = [len(ax) + int(rng.integers(0, 5)) for ax, _ in pairs]
    off = np.concatenate([[0], np.cumsum(slots)]).astype(np.int64)
    start = np.array([off[k + 1] - len(pairs[k][0]) for k in range(len(pairs))], dtype=np.int64)
    ox = np.zeros(int(off[-1]), dtype=np.uint8)
    oy = np.zeros(int(off[-1]), dtype=np.uint8)
    for k, (ax, ay) in enumerate(pairs):
        ox[start[k]:off[k + 1]] = np.frombuffer(ax, dtype=np.uint8)
        oy[start[k]:off[k + 1]] = np.frombuffer(ay, dtype=np.uint8)
    xids, yids = [f"x{i}" for i in range(nx)], [f"y{j}" for j in range(ny)]
    want = tmp_path / "want.txt"
    with SequencePairHandler.Formatted(want, "w") as file:
        for k, (ax, ay) in enumerate(pairs):
            file.write(SequencePair(Sequence(xids[k // ny], ax.decode("latin-1")), Sequence(yids[k % ny], ay.decode("latin-1"))))
    got = tmp_path / "got.txt"
    got.write_bytes(b"")
    fw.format_aligned_pairs(got, True, fw.StringTable(xids), fw.StringTable(yids), 0, nx, ny, ox, oy, start, off, threads=2)
    assert got.read_bytes() == want.read_bytes()
    assert b"\nx1 / y0\nAC\xc3\x89GT-\n||||--\nAC\xc3\x89G-T\n\nx1 / y1\nACGT\n||-|\nAC-T\n" in got.read_bytes()


@pytest.mark.parametrize("spec", ["{:.4f}", "{:.0f}", "{:.2f}", "{:.9f}", "{:f}"])
def test_fixed_point_fast_path_equals_python_format(tmp_path, spec):
    """The integer-arithmetic formatter behind "%.Nf" (host_format.cpp: append_fixed) against
    Python's own format over magnitudes from subnormal to 1e15, exact decimal ties (0.125, 2.5,
    0.00005 ...), values a hair on either side of a tie, negative values and negative zero."""
    from taxi2_b200 import fastwrite

    rng = np.random.default_rng(len(spec))
    vals = [0.0, -0.0, 0.5, 1.5, 2.5, 0.125, 0.375, 0.00005, 0.00015, 0.99995, 0.999949999999, 1e-300, 5e-324, 123456789.987654321,
            9.999999999e14, 0.1, 0.2, 0.3, 1 / 3, 2 / 3, 0.07, 0.0625, 0.03125, 1e15 + 0.5, 4503599627370497.0, 1e22]
    for k in range(1, 40):
        base = k / 20000.0            # multiples of 0.00005: ties of "{:.4f}" when exactly representable
        vals += [base, np.nextafter(base, 1.0), np.nextafter(base, 0.0)]
    vals += list(rng.random(20000)) + list(rng.random(5000) * 10.0 ** rng.integers(-12, 14, 5000)) + list(-rng.random(2000))
    vals = np.array(vals, dtype=np.float64)
    n = len(vals)
    m = np.zeros((1, n, 4))
    m[0, :, 2] = vals
    ids = fastwrite.StringTable(["row"])
    path = tmp_path / "m.tsv"
    path.write_bytes(b"")
    fastwrite.format_matrix(path, ids, 0, 1, n, m, None, 2, 1.0, fastwrite.printf_format(spec), "NA")
    got = path.read_text().rstrip("\n").split("\t")[1:]
    want = [spec.format(v) for v in vals]
    assert got == want


@pytest.mark.parametrize("template", ["{mean} ({min}-{max})", "[{mean}|{min}|{max}]", "{mean}"])
def test_subset_statistics_files_native_rows_equal_the_python_rows(tmp_path, monkeypatch, template):
    """subsets/*/linear/{pairs,identity}.tsv and matricial/<metric>.tsv (versus_all.py:143-249): the
    library's row writers against the Python string assembly of the same arrays -- keys in
    first-seen order, a subset that is None ("?"), keys without any defined distance ("NA"),
    several runs of equal first subset, values on decimal rounding ties.  A statistics template
    that is not the three fields in order keeps the Python rows."""
    from types import SimpleNamespace

    from taxi2_b200.tasks.versus_all import SubsetAggregation

    rng = np.random.default_rng(12)
    names = ["Alpha beta", None, "Gamma", "Delta epsilon zeta", "Eta"]
    nsub = len(names)
    labels = ["p-distance", "k2p"]
    states = []
    order = rng.permutation(nsub * nsub)[: nsub * nsub - 3]          # three keys never seen
    for _ in labels:
        st = fw.NativeSubsetState(nsub)
        st.first_seen[order] = np.arange(len(order))
        st.count[order] = rng.integers(0, 4, len(order))
        seen = order[st.count[order] > 0]
        st.sum[seen] = np.round(rng.random(len(seen)) * 3, 5)
        st.min[seen] = np.round(rng.random(len(seen)), 5)
        st.max[seen] = np.round(rng.random(len(seen)) + 1, 4) + 0.00005
        states.append(st)
    agg = SubsetAggregation.__new__(SubsetAggregation)
    agg.native = (names, labels, states)
    fmt = SimpleNamespace(float="{:.4f}", stats_template=template)
    agg.write_arrays(tmp_path / "native", fmt)
    monkeypatch.setattr(fw, "printf_format", lambda spec: None)      # the Python rows of the same method
    agg.write_arrays(tmp_path / "python", fmt)
    files = sorted(p.relative_to(tmp_path / "python") for p in (tmp_path / "python").rglob("*.tsv"))
    assert [str(f) for f in files] == ["linear/identity.tsv", "linear/pairs.tsv", "matricial/k2p.tsv", "matricial/p-distance.tsv"]
    for rel in files:
        assert (tmp_path / "native" / rel).read_bytes() == (tmp_path / "python" / rel).read_bytes(), rel
    assert b"NA" in (tmp_path / "native" / "linear" / "pairs.tsv").read_bytes() and b"?" in (tmp_path / "native" / "matricial" / "k2p.tsv").read_bytes()
