"""Task-level parity on the GPU: every output file of VersusAll / VersusReference byte-for-byte
against the per-pair restatement of the reference pipeline (tests/ref_pipeline.py, oracle-backed).
The reference itself pins no task output (its only task test is an xfail stub), so this is the
strongest check available: same order, same None/NA quirks, same aggregates, same formatting."""
from __future__ import annotations

from pathlib import Path

import pytest

import ref_pipeline
from conftest import GOLDEN
from taxi2_b200.distances import DistanceMetric
from taxi2_b200.partitions import Partition, PartitionHandler
from taxi2_b200.sequences import Sequence, SequenceHandler, Sequences
from taxi2_b200.tasks import VersusAll, VersusReference

pytestmark = pytest.mark.gpu

SILENT = lambda *a: None  # noqa: E731


def load(name):
    path = GOLDEN / name
    seqs = Sequences.fromPath(path, SequenceHandler.Tabfile, idHeader="seqid", seqHeader="sequence")
    species = Partition.fromPath(path, PartitionHandler.Tabfile, idHeader="seqid", subHeader="organism")
    genera = Partition.fromPath(path, PartitionHandler.Tabfile, idHeader="seqid", subHeader="organism",
                                filter=PartitionHandler.subset_first_word)
    return seqs, species, genera


def assert_same_tree(got: Path, want: Path):
    files_got = sorted(p.relative_to(got) for p in got.rglob("*") if p.is_file())
    files_want = sorted(p.relative_to(want) for p in want.rglob("*") if p.is_file())
    assert files_got == files_want
    for rel in files_want:
        assert (got / rel).read_bytes() == (want / rel).read_bytes(), rel


@pytest.mark.parametrize("native", [True, False])
@pytest.mark.parametrize("align,write,multiply", [(True, True, False), (True, False, True), (False, False, False)])
def test_versus_all_outputs(tmp_path, align, write, multiply, native):
    seqs, species, genera = load("Taxi2test1_10.tab")
    # a duplicated record and a pair of different records with equal sequences exercise the x != y quirk
    records = list(seqs)
    records.append(records[3])
    records.append(Sequence("twin", records[5].seq, records[5].extras))
    task = VersusAll()
    task.work_dir = tmp_path / "got"
    task.progress_handler = SILENT
    task.input.sequences = Sequences(records)
    task.input.species, task.input.genera = species, genera
    task.params.pairs.align, task.params.pairs.write = align, write
    task.params.format.percentage_multiply = multiply
    task.native_writers = native   # batch formatter vs the per-value Python handlers: same bytes
    results = task.start()
    assert results.output_directory == task.work_dir and results.seconds_taken > 0
    want = tmp_path / "want"
    ref_pipeline.versus_all(records, want, species, genera, align=align, multiply=multiply)
    if align and not write:
        (want / "align" / "aligned_pairs.txt").unlink()
        (want / "align").rmdir()
    assert_same_tree(task.work_dir, want)


@pytest.mark.parametrize("write,block_pairs", [(True, None), (False, None), (False, 600)])
def test_versus_all_on_the_50_sequence_sample(tmp_path, monkeypatch, write, block_pairs):
    """The reference's Taxi2test1_50.tab as shipped (2 500 ordered pairs, 416-618 bp, species and
    genera from the organism column): all output files, aligned pairs included, byte for byte.
    Without the aligned-pairs file the task aligns each unordered pair once and mirrors the result
    (MultiEngine.iter_symmetric_rows), in one block and in blocks of 12 rows."""
    from taxi2_b200.tasks import common

    if block_pairs:
        monkeypatch.setattr(common, "MAX_BLOCK_PAIRS", block_pairs)
    seqs, species, genera = load("Taxi2test1_50.tab")
    task = VersusAll()
    task.work_dir = tmp_path / "got"
    task.progress_handler = SILENT
    task.input.sequences = seqs
    task.input.species, task.input.genera = species, genera
    task.params.pairs.write = write
    task.start()
    ref_pipeline.versus_all(list(seqs), tmp_path / "want", species, genera)
    if not write:
        (tmp_path / "want" / "align" / "aligned_pairs.txt").unlink()
        (tmp_path / "want" / "align").rmdir()
    assert_same_tree(task.work_dir, tmp_path / "want")


@pytest.mark.parametrize("fmt", ["{:.4f}", "{:.2e}", "{:>9.3f}"])
def test_versus_all_without_partitions_and_metric_subset(tmp_path, fmt):
    seqs, _, _ = load("Taxi2test1_10.tab")
    task = VersusAll()
    task.work_dir = tmp_path / "got"
    task.progress_handler = SILENT
    task.input.sequences = seqs
    task.params.distances.metrics = [DistanceMetric.Kimura2P(), DistanceMetric.Uncorrected()]
    task.params.format.float = fmt      # the last one is not a plain spec: Python handlers take over
    task.start()
    ref_pipeline.versus_all(list(seqs), tmp_path / "want", metrics=[DistanceMetric.Kimura2P(), DistanceMetric.Uncorrected()], fmt=fmt)
    assert_same_tree(task.work_dir, tmp_path / "want")


def test_versus_all_sequences_without_extras(tmp_path):
    records = [Sequence(f"s{k}", seq) for k, seq in enumerate(["ACGTACGTAC", "ACGTTCGTAC", "ACG-ACGNAC", "TTGTACGAAC"])]
    task = VersusAll()
    task.work_dir = tmp_path / "got"
    task.progress_handler = SILENT
    task.input.sequences = Sequences(records)
    task.start()
    ref_pipeline.versus_all(records, tmp_path / "want")
    assert_same_tree(task.work_dir, tmp_path / "want")


@pytest.mark.parametrize("native", [True, False])
@pytest.mark.parametrize("align,multiply,main", [(True, False, "p"), (True, True, "k2p"), (False, False, "p-gaps")])
def test_versus_reference_outputs(tmp_path, align, multiply, main, native):
    seqs, _, _ = load("Taxi2test1_50.tab")
    records = list(seqs)
    data, reference = records[:12], records[12:40]
    task = VersusReference()
    task.work_dir = tmp_path / "got"
    task.progress_handler = SILENT
    task.input.data, task.input.reference = Sequences(data), Sequences(reference)
    task.params.pairs.align = align
    task.params.distances.metric = DistanceMetric.fromLabel(main)
    task.params.format.percentage_multiply = multiply
    task.native_writers = native
    task.start()
    ref_pipeline.versus_reference(data, reference, tmp_path / "want", align=align, metric=DistanceMetric.fromLabel(main), multiply=multiply)
    assert_same_tree(task.work_dir, tmp_path / "want")


def with_accented_letters(records):
    """A few sequences carrying letters outside ASCII ('É', 'ü'), as a UTF-8 input file can hold."""
    out = list(records)
    for k, (at, letters) in enumerate(((5, "É"), (40, "üü"), (90, "ÉüÉ"))):
        s = out[k]
        out[k] = Sequence(s.id, s.seq[:at] + letters + s.seq[at:], s.extras)
    return out


@pytest.mark.parametrize("native", [True, False])
def test_aligned_pairs_with_letters_outside_ascii(tmp_path, native):
    """VersusAll and VersusReference with aligned pairs on sequences with 'É' / 'ü': the native and
    the Python writers and the restated reference pipeline write the same bytes -- the UTF-8 text of
    the aligned strings."""
    seqs, species, genera = load("Taxi2test1_10.tab")
    records = with_accented_letters(seqs)
    task = VersusAll()
    task.work_dir = tmp_path / "got"
    task.progress_handler = SILENT
    task.input.sequences = Sequences(records)
    task.input.species, task.input.genera = species, genera
    task.native_writers = native
    task.start()
    ref_pipeline.versus_all(records, tmp_path / "want", species, genera)
    assert "É".encode("utf-8") in (task.work_dir / "align" / "aligned_pairs.txt").read_bytes()
    assert_same_tree(task.work_dir, tmp_path / "want")

    data, reference = records[:4], records[3:]
    task = VersusReference()
    task.work_dir = tmp_path / "got_ref"
    task.progress_handler = SILENT
    task.input.data, task.input.reference = Sequences(data), Sequences(reference)
    task.native_writers = native
    task.start()
    ref_pipeline.versus_reference(data, reference, tmp_path / "want_ref", align=True, metric=DistanceMetric.fromLabel("p"))
    assert_same_tree(task.work_dir, tmp_path / "want_ref")


def test_versus_reference_raises_without_any_defined_distance(tmp_path):
    task = VersusReference()
    task.work_dir = tmp_path / "got"
    task.progress_handler = SILENT
    task.input.data = Sequences([Sequence("q", "NNNN")])
    task.input.reference = Sequences([Sequence("r", "ACGT")])
    with pytest.raises(ValueError):
        task.start()


# ---- dereplicate / decontaminate -------------------------------------------------------------------
from taxi2_b200.files import FileFormat  # noqa: E402
from taxi2_b200.tasks import Decontaminate, Decontaminate2, Dereplicate  # noqa: E402


def near_duplicates():
    """The 50-sample plus truncated / mutated copies so that the greedy walk excludes things
    in the middle of rows (the order-observable part of the reference)."""
    seqs, _, _ = load("Taxi2test1_50.tab")
    records = list(seqs)[:24]
    extra = []
    for k, s in enumerate(records[:10]):
        cut = s.seq[: len(s.seq) - 7 * (k + 1)]
        extra.append(Sequence(f"short{k}", cut, s.extras))
        extra.append(Sequence(f"long{k}", s.seq + "acgtacgt"[: k + 1], s.extras))
    records[5:5] = extra[:8]
    records += extra[8:]
    records.append(Sequence("tiny", "acgt", {"specimen_voucher": "v", "organism": "o"}))
    return records


@pytest.mark.parametrize("align,write,multiply,fasta", [(True, True, False, False), (True, False, True, True), (False, False, False, False)])
def test_dereplicate_outputs(tmp_path, align, write, multiply, fasta):
    records = near_duplicates()
    task = Dereplicate()
    task.work_dir = tmp_path / "got"
    task.progress_handler = SILENT
    task.input = Sequences(records)
    task.output_format = FileFormat.Fasta if fasta else FileFormat.Tabfile
    task.rows_per_block = 7   # several device blocks: exclusions made in one block shrink the next
    task.params.pairs.align, task.params.pairs.write = align, write
    task.params.format.percentage_multiply = multiply
    task.params.thresholds.similarity = 7.0 if multiply else 0.07
    task.start()
    excluded = ref_pipeline.dereplicate(records, tmp_path / "want", similarity=task.params.thresholds.similarity, align=align,
                                        multiply=multiply, fasta=fasta)
    if align and not write:
        (tmp_path / "want" / "aligned_pairs.txt").unlink()
    assert task.excluded == excluded and len(excluded) >= 10
    assert_same_tree(task.work_dir, tmp_path / "want")


@pytest.mark.parametrize("native", [True, False])
@pytest.mark.parametrize("align,multiply,fasta", [(True, False, False), (True, True, True), (False, False, False)])
def test_decontaminate_outputs(tmp_path, align, multiply, fasta, native):
    seqs, _, _ = load("Taxi2test1_50.tab")
    records = list(seqs)
    data, outgroup, ingroup = records[:14], records[14:30], records[30:46]
    data.append(Sequence("allN", "nnnnnnnn", records[0].extras))
    task = Decontaminate()
    task.work_dir = tmp_path / "got1"
    task.native_writers = native   # block path vs per-pair path: same bytes
    task.progress_handler = SILENT
    task.input, task.outgroup = Sequences(data), Sequences(outgroup)
    task.output_format = FileFormat.Fasta if fasta else FileFormat.Tabfile
    task.params.pairs.align = align
    task.params.format.percentage_multiply = multiply
    task.params.thresholds.similarity = 12.0 if multiply else 0.12
    task.start()
    ref_pipeline.decontaminate(data, outgroup, tmp_path / "want1", similarity=task.params.thresholds.similarity, align=align,
                               multiply=multiply, fasta=fasta)
    assert_same_tree(task.work_dir, tmp_path / "want1")

    task2 = Decontaminate2()
    task2.work_dir = tmp_path / "got2"
    task2.native_writers = native
    task2.progress_handler = SILENT
    task2.input, task2.outgroup, task2.ingroup = Sequences(data), Sequences(outgroup), Sequences(ingroup)
    task2.output_format = FileFormat.Fasta if fasta else FileFormat.Tabfile
    task2.params.pairs.align = align
    task2.params.format.percentage_multiply = multiply
    task2.params.weights.outgroup, task2.params.weights.ingroup = 1.0, 1.5
    task2.start()
    ref_pipeline.decontaminate2(data, outgroup, ingroup, tmp_path / "want2", w_out=1.0, w_in=1.5, align=align, multiply=multiply, fasta=fasta)
    assert_same_tree(task2.work_dir, tmp_path / "want2")
