"""`process` from a BAM alone: junction extraction with anchor extents, the regtools-layout BED12 writer, the `junctions` and
`processBam` commands and spl_process_bam_extract (one ingest: extract, filter, count).

The CPU tests run the host layers for real and answer the GPU calls with the restatements (oracle/junction_oracle.py for the
extraction, the C oracle for the count); the GPU tests hold the kernels to the same restatements."""
import os

import numpy as np
import pytest

from common import load_golden
from oracle import c_oracle, junction_oracle
from spliser_b200 import Records, api
from test_cli_cpu import OracleContext

HAND_READS = [("C", 100, 0, "20M100N20M"), ("C", 100, 16, "20M100N20M"), ("C", 113, 0, "7M100N20M"), ("C", 100, 0, "20M100N7M"),
              ("C", 100, 0, "20M60N20M"), ("C", 100, 0, "20M600000N20M"), ("C", 300, 0, "5M2D4M90N3M1I6M"), ("C", 500, 0, "10M80N6M80N10M"),
              ("C", 700, 0, "10M80N8M80N10M"), ("C", 900, 0, "4S7M100N20M"), ("C", 100, 99, "20M100N20M"), ("C", 100, 147, "20M100N20M")]
HAND_ROWS = [(0, 119, 219, 4, "?"), (0, 310, 400, 1, "?"), (0, 709, 789, 1, "?"), (0, 797, 877, 1, "?")]

# extents with known answers: (reads, extraction kwargs, [(left, right, score, start, end)])
EXTENT_CASES = [
    ("two reads of different overhang", [("C", 100, 0, "20M100N20M"), ("C", 105, 0, "15M100N30M")], {}, [(119, 219, 2, 99, 249)]),
    ("a D inside a stretch, an I that adds nothing, soft clips", [("C", 300, 0, "3S5M2D4M90N3M1I6M2S")], {}, [(310, 400, 1, 299, 409)]),
    ("two junctions sharing the middle stretch", [("C", 500, 0, "10M80N12M80N10M")], {}, [(509, 589, 1, 499, 601), (601, 681, 1, 589, 691)]),
    ("a 0N splits the stretch", [("C", 700, 0, "10M0N10M80N10M")], {}, [(719, 799, 1, 709, 809)]),
    ("a 0N is a junction of its own without the intron bound", [("C", 700, 0, "10M0N10M80N10M")], dict(min_intron=0),
     [(709, 709, 1, 699, 719), (719, 799, 1, 709, 809)]),
    ("a 0M adds nothing", [("C", 900, 0, "10M80N0M10M"), ("C", 890, 0, "20M80N0M9M2M")], {}, [(909, 989, 2, 889, 1000)]),
]


def _rows(j):
    return sorted(zip(j.chrom.tolist(), j.left.tolist(), j.right.tolist(), j.score.tolist(), [chr(x) for x in j.strand.tolist()]))


def _full(j):
    return list(zip(j.chrom.tolist(), j.left.tolist(), j.right.tolist(), j.score.tolist(), j.strand.tolist(), j.start.tolist(), j.end.tolist()))


class ExtractOracleContext(OracleContext):
    """Answers the extraction calls like spliser_b200.Context, from the restatement and the C oracle."""

    def extract_junctions_bam(self, bam_path, chrom_names, flags=0, min_anchor=8, min_intron=70, max_intron=500000):
        rec = Records.from_bam(bam_path, chrom_names)
        return junction_oracle.extract(rec, len(chrom_names), flags & 3, min_anchor, min_intron, max_intron)

    def process_bam_extract(self, bam_path, chrom_names, flags=0, min_anchor=8, min_intron=70, max_intron=500000, qchrom="All",
                            gene_bounds=None, window_max_intron=0):
        rec = Records.from_bam(bam_path, chrom_names)
        j = junction_oracle.extract(rec, len(chrom_names), flags & 3, min_anchor, min_intron, max_intron)
        j = junction_oracle.filter_rows(j, chrom_names, qchrom, gene_bounds, window_max_intron)
        return j, api.SiteTable(**c_oracle.process(rec, len(chrom_names), j, flags))


def _write_bam(tmp, reads, name="x.bam"):
    refs = sorted({r[0] for r in reads}) or ["C"]
    bam = os.path.join(tmp, name)
    Records.from_reads(refs, reads).write_bam(bam, refs)
    return bam


def _bam_only_equals_two_steps(cli, ctx, d, bam, stranded, stype, cryptic, bounds=(8, 70, 500000), **kw):
    """processBam's TSV == junctions + process -b on the same BAM; returns the number of BED rows."""
    a, m, M = bounds
    bed = str(d / "j.bed")
    cli.junctions(bam, bed, minAnchor=a, minIntron=m, maxIntron=M, isStranded=stranded, strandedType=stype, ctx=ctx)
    cli.process(bam, bed, str(d / "two"), isStranded=stranded, strandedType=stype, isbeta2Cryptic=cryptic, ctx=ctx, **kw)
    cli.processBam(bam, str(d / "one"), isStranded=stranded, strandedType=stype, isbeta2Cryptic=cryptic, minAnchor=a, minIntron=m,
                   maxIntron=M, ctx=ctx, **kw)
    two, one = open(str(d / "two.SpliSER.tsv")).read(), open(str(d / "one.SpliSER.tsv")).read()
    assert one == two, (stranded, stype, cryptic, bounds, kw)
    return sum(1 for _ in open(bed))


MODES = ((False, None), (True, "fr"), (True, "rf"))


# ---------------------------------------------------------------------------------------------------------- CPU
def test_restatement_reproduces_the_hand_made_filter_case(built_library):
    rec = Records.from_reads(["C"], HAND_READS)
    assert _rows(junction_oracle.extract(rec, 1, 0)) == HAND_ROWS
    got = _rows(junction_oracle.extract(rec, 1, 1 | 2))
    assert (0, 119, 219, 1, "+") in got and (0, 119, 219, 3, "-") in got, got


def test_restatement_reproduces_the_synthetic_truth_tables(built_library):
    from spliser_b200 import synth
    for stranded, paired, seed in ((False, False, 5), (True, True, 6)):
        w = synth.generate(synth.config_small(20_000, seed=seed, stranded=stranded, paired=paired))
        got = junction_oracle.extract(w.records, len(w.chroms), w.flags & 3)
        assert _rows(got) == _rows(w.junctions)
        assert np.all(got.start <= got.left - 8) and np.all(got.end >= got.right + 8)


def test_restatement_extents_on_hand_made_cases(built_library):
    for name, reads, kw, want in EXTENT_CASES:
        j = junction_oracle.extract(Records.from_reads(["C"], reads), 1, 0, **kw)
        assert [(l, r, s, a, b) for _, l, r, s, _, a, b in _full(j)] == want, name


def test_bed_writer_bytes_and_round_trip(tmp_path, built_library):
    from spliser_b200.bed import parse_bed12, write_junctions_bed
    rng = np.random.default_rng(20261021)
    chroms = ["chr1", "chrUn_KI270302v1", "HLA-A*01:01:01:01", "chrEBV", "C"]
    for k, n in enumerate((0, 1, 700)):
        left = rng.integers(0, 2 ** 28, n)
        right = left + rng.integers(0, 500_000, n)
        a, b = rng.integers(0, 300, n), rng.integers(0, 300, n)
        junc = api.Junctions(rng.integers(0, len(chroms), n), left, right, rng.integers(1, 2 ** 40, n),
                             rng.choice(np.frombuffer(b"+-?", np.uint8), n), np.maximum(left - a, 0), right + b)
        p = str(tmp_path / ("w%d.bed" % k))
        write_junctions_bed(p, chroms, junc)
        text = open(p).read()
        assert text == junction_oracle.bed_text(chroms, junc)
        assert n < 2 or "\tJUNC00000002\t" in text
        names, back, sstr = parse_bed12(text)
        assert [(names[c], l, r, s, chr(t)) for c, l, r, s, t in zip(back.chrom.tolist(), back.left.tolist(), back.right.tolist(),
                                                                    back.score.tolist(), back.strand.tolist())] == \
            [(chroms[c], l, r, s, chr(t)) for c, l, r, s, t in zip(junc.chrom.tolist(), junc.left.tolist(), junc.right.tolist(),
                                                                   junc.score.tolist(), junc.strand.tolist())]
        assert list(sstr) == [chr(t) for t in junc.strand.tolist()]
    with pytest.raises(ValueError):                        # extents inside the junction
        write_junctions_bed(str(tmp_path / "bad.bed"), ["C"], api.Junctions([0], [10], [20], [1], [63], [11], [25]))


def test_process_bam_equals_junctions_then_process_on_cpu(tmp_path, built_library):
    from spliser_b200 import cli
    cases = load_golden("appendix_a.json.gz")["process"] + load_golden("process_fuzz.json.gz")[::9]
    ctx = ExtractOracleContext()
    rows = 0
    for k, case in enumerate(cases):
        d = tmp_path / ("p%d" % k)
        d.mkdir()
        bam = _write_bam(str(d), [tuple(r) for r in case["reads"]])
        for stranded, stype in MODES:
            for cryptic in (False, True):
                for bounds in ((8, 70, 500000), (1, 1, 500000)):
                    rows += _bam_only_equals_two_steps(cli, ctx, d, bam, stranded, stype, cryptic, bounds)
    assert rows > 200


def test_process_bam_with_annotation_chromosome_and_gene_window_on_cpu(tmp_path, built_library):
    """-A, -c (also naming a chromosome the BAM does not have) and -g ... -m on the annotated golden cases."""
    from spliser_b200 import cli
    cases = [c for c in load_golden("appendix_a.json.gz")["process"] + load_golden("process_fuzz.json.gz") if c.get("gff")]
    assert cases
    ctx = ExtractOracleContext()
    for k, case in enumerate(cases[:40]):
        d = tmp_path / ("a%d" % k)
        d.mkdir()
        reads = [tuple(r) for r in case["reads"]]
        bam = _write_bam(str(d), reads)
        gff = str(d / "a.gff")
        open(gff, "w").write(case["gff"])
        stranded, stype = case["stranded"], case["stype"]
        chrom = reads[0][0] if reads else "C"
        for kw in (dict(annotationFile=gff), dict(annotationFile=gff, qChrom=chrom), dict(qChrom="NOPE"),
                   dict(annotationFile=gff, qChrom=case.get("qchrom", "All"), qGene=case.get("qgene", "All"),
                        maxIntronSize=case.get("max_intron", 0))):
            if kw.get("qGene", "All") != "All":
                try:
                    cli.processBam(bam, str(d / "probe"), ctx=ctx, **kw)
                except AttributeError:                # -g gene absent from the annotation: both commands raise it (S:283)
                    with pytest.raises(AttributeError):
                        cli.process(bam, str(d / "j.bed"), str(d / "x"), ctx=ctx, **kw)
                    continue
            for bounds in ((8, 70, 500000), (1, 1, 500000)):
                _bam_only_equals_two_steps(cli, ctx, d, bam, stranded, stype, case["cryptic"], bounds, **kw)
        assert open(str(d / "one.SpliSER.tsv")).read().count("\n") >= 1


def test_new_subcommands_parse_like_regtools_and_process(built_library, monkeypatch):
    from spliser_b200 import cli
    seen = {}
    monkeypatch.setattr(cli, "junctions", lambda **kw: seen.update(kw))
    monkeypatch.setattr(cli, "processBam", lambda **kw: seen.update(kw))
    cli.main(["junctions", "-B", "x.bam", "-o", "x.bed"])
    assert seen == dict(inBAM="x.bam", outBed="x.bed", minAnchor=8, minIntron=70, maxIntron=500000, isStranded=False, strandedType=None)
    seen.clear()
    cli.main(["junctions", "-B", "x.bam", "-o", "x.bed", "-a", "6", "-m", "50", "-M", "1000", "--isStranded", "-s", "rf"])
    assert seen == dict(inBAM="x.bam", outBed="x.bed", minAnchor=6, minIntron=50, maxIntron=1000, isStranded=True, strandedType="rf")
    seen.clear()
    cli.main(["processBam", "-B", "x.bam", "-o", "out"])
    assert seen == dict(inBAM="x.bam", outputPath="out", annotationFile=None, aType="gene", qChrom="All", qGene="All", maxIntronSize=0,
                        isStranded=False, strandedType=None, isbeta2Cryptic=False, minAnchor=8, minIntron=70, maxIntron=500000)
    seen.clear()
    cli.main(["processBam", "-B", "x.bam", "-o", "out", "-A", "g.gff", "-t", "mRNA", "-c", "C", "-g", "G1", "-m", "5000", "--isStranded",
              "-s", "fr", "--beta2Cryptic", "--minAnchor", "4", "--minIntron", "20", "--maxIntron", "9000"])
    assert seen == dict(inBAM="x.bam", outputPath="out", annotationFile="g.gff", aType="mRNA", qChrom="C", qGene="G1", maxIntronSize=5000,
                        isStranded=True, strandedType="fr", isbeta2Cryptic=True, minAnchor=4, minIntron=20, maxIntron=9000)
    for argv in (["processBam", "-B", "x.bam", "-o", "out", "-g", "G1"],          # --gene requires --annotationFile (S:1350-1353)
                 ["processBam", "-B", "x.bam", "-o", "out", "--isStranded"],       # --isStranded requires -s (S:1354-1355)
                 ["junctions", "-B", "x.bam", "-o", "x.bed", "--isStranded"],
                 ["processBam", "-B", "x.bam"], ["junctions", "-o", "x.bed"]):
        with pytest.raises(SystemExit):
            cli.main(argv)


def test_reference_names_in_header_order(tmp_path, built_library):
    names = ["chr%d" % i for i in range(4000, 0, -1)] + ["HLA-A*01:01:01:01"]
    bam = str(tmp_path / "h.bam")
    Records.from_reads(names, [(names[-1], 10, 0, "10M")]).write_bam(bam, names)
    assert api.bam_reference_names(bam) == names
    with pytest.raises(IOError):
        api.bam_reference_names(str(tmp_path / "missing.bam"))


# ---------------------------------------------------------------------------------------------------------- GPU
def _extents_equal(ctx, tmp_path, rec, chroms, flags, tag, **kw):
    want = junction_oracle.extract(rec, len(chroms), flags & 3, **kw)
    got = ctx.extract_junctions_records(rec, len(chroms), flags & 3, **kw)
    assert _full(got) == _full(want), tag
    bam = str(tmp_path / ("%s.bam" % tag))
    rec.write_bam(bam, chroms)
    assert _full(ctx.extract_junctions_bam(bam, chroms, flags & 3, **kw)) == _full(want), tag
    return want


@pytest.mark.gpu
def test_extents_of_the_kernel_equal_the_restatement(ctx, tmp_path):
    from oracle import fuzzgen
    from spliser_b200 import synth
    for stranded, paired, seed in ((False, False, 5), (True, True, 6)):
        w = synth.generate(synth.config_small(120_000, seed=seed, stranded=stranded, paired=paired))
        got = _extents_equal(ctx, tmp_path, w.records, w.chroms, w.flags, "small%d" % seed)
        assert _rows(got) == _rows(w.junctions)                # the five columns the kernel always returned
    w = synth.generate_long_reads(synth.config_long_reads(12_000))
    for flags in (0, 1):
        _extents_equal(ctx, tmp_path, w.records, w.chroms, flags, "long%d" % flags)
        _extents_equal(ctx, tmp_path, w.records, w.chroms, flags, "long_all%d" % flags, min_anchor=0, min_intron=0)
    rows = 0
    for seed in range(960000, 960200):
        case = fuzzgen.gen_long_case(seed, dirty=(seed % 4 == 1))
        chroms = sorted({r[0] for r in case["reads"]}) or ["C"]
        rec = Records.from_reads(chroms, [tuple(r) for r in case["reads"]])
        for flags, kw in ((0, {}), (3, dict(min_anchor=1, min_intron=1))):
            want = junction_oracle.extract(rec, len(chroms), flags, **kw)
            assert _full(ctx.extract_junctions_records(rec, len(chroms), flags, **kw)) == _full(want), seed
            rows += len(want)
    assert rows > 1000
    for name, reads, kw, want in EXTENT_CASES:
        j = ctx.extract_junctions_records(Records.from_reads(["C"], reads), 1, 0, **kw)
        assert [(l, r, s, a, b) for _, l, r, s, _, a, b in _full(j)] == want, name
    assert _rows(ctx.extract_junctions_records(Records.from_reads(["C"], HAND_READS), 1, 0)) == HAND_ROWS


def _two_step(ctx, bam, chroms, flags, qchrom="All", gene_bounds=None, window=0):
    j = ctx.extract_junctions_bam(bam, chroms, flags & 3)
    j = junction_oracle.filter_rows(j, chroms, qchrom, gene_bounds, window)
    return j, ctx.process_bam(bam, chroms, j, flags)


@pytest.mark.gpu
@pytest.mark.parametrize("host_bam", [False, True])
def test_process_bam_extract_equals_extract_then_process(ctx, tmp_path, monkeypatch, host_bam):
    from spliser_b200 import synth
    if host_bam:
        monkeypatch.setenv("SPLISER_HOST_BAM", "1")
    for stranded, paired, seed in ((False, False, 5), (True, True, 6)):
        w = synth.generate(synth.config_small(120_000, seed=seed, stranded=stranded, paired=paired))
        bam = str(tmp_path / ("e%d.bam" % seed))
        w.records.write_bam(bam, w.chroms, w.chrom_len)
        mid = int(np.median(w.junctions.left))
        for flags in ((w.flags & 3), (w.flags & 3) | 4):
            for qchrom, bounds, win in (("All", None, 0), (w.chroms[0], None, 0), ("All", (mid, mid + 20000), 5000),
                                        (w.chroms[-1], (mid, mid + 20000), 0), ("NOPE", None, 0)):
                jw, tw = _two_step(ctx, bam, w.chroms, flags, qchrom, bounds, win)
                j, t = ctx.process_bam_extract(bam, w.chroms, flags, qchrom=qchrom, gene_bounds=bounds, window_max_intron=win)
                st = ctx.stats()
                assert st["bam_on_device"] == (0.0 if host_bam else 1.0)
                assert _full(j) == _full(jw), (qchrom, bounds)
                assert c_oracle.diff_tables(c_oracle.table_dict(t), c_oracle.table_dict(tw)) is None, (flags, qchrom, bounds)
                want = c_oracle.process(w.records, len(w.chroms), j, flags, threads=8)
                assert c_oracle.diff_tables(c_oracle.table_dict(t), want) is None, (flags, qchrom, bounds)
                assert (len(j) > 0) == (qchrom != "NOPE")


@pytest.mark.gpu
def test_process_bam_extract_ingests_once(ctx, tmp_path):
    from spliser_b200 import synth
    w = synth.generate(synth.config_small(400_000, seed=7, stranded=True, paired=True))
    bam = str(tmp_path / "once.bam")
    w.records.write_bam(bam, w.chroms, w.chrom_len)
    j, _ = ctx.process_bam_extract(bam, w.chroms, w.flags)
    one = ctx.stats()
    ctx.process_bam(bam, w.chroms, j, w.flags)
    ref = ctx.stats()
    assert one["bam_on_device"] == 1.0 and ref["bam_on_device"] == 1.0
    # beyond spl_process: the extraction's copy of the chunk table (48 B per 1024 records of a chromosome) and its segment list;
    # a second ingest would add the whole file image again
    chunk_table = 48 * (len(w.records) // 1024 + len(w.chroms) + 1)
    assert one["h2d_bytes"] <= ref["h2d_bytes"] + 21 * len(j) + chunk_table, (one["h2d_bytes"], ref["h2d_bytes"])
    assert one["h2d_bytes"] - ref["h2d_bytes"] < os.path.getsize(bam) / 4
    assert one["ms_extract"] > 0 and one["n_junctions"] >= len(j)


@pytest.mark.gpu
def test_header_with_4000_references(ctx, tmp_path):
    """More than 2,048 references used to fail with 'too many chromosomes for the packed key'."""
    names = ["ctg%04d" % i for i in range(4000)]
    reads = []
    for c in names[-3:]:
        reads += [(c, 1000, 0, "20M300N30M"), (c, 1005, 16, "15M300N10M5I20M"), (c, 5000, 0, "10M100N10M80N12M")]
    rec = Records.from_reads(names, reads)
    bam = str(tmp_path / "many.bam")
    rec.write_bam(bam, names, [100_000] * 4000)
    want = junction_oracle.extract(rec, 4000, 0)
    assert len(want) == 9
    assert _full(ctx.extract_junctions_records(rec, 4000, 0)) == _full(want)
    assert _full(ctx.extract_junctions_bam(bam, names, 0)) == _full(want)
    j, t = ctx.process_bam_extract(bam, names, 0)
    assert _full(j) == _full(want)
    assert c_oracle.diff_tables(c_oracle.table_dict(t), c_oracle.process(rec, 4000, want, 0)) is None


@pytest.mark.gpu
def test_hot_queue_overflow_through_process_bam_extract(tmp_path):
    """A fresh context whose first pass overflows the hot-item queue (the long-read sample, every N kept) repeats it with room."""
    import spliser_b200
    from spliser_b200 import synth
    w = synth.generate_long_reads(synth.config_long_reads(12_000))
    bam = str(tmp_path / "long.bam")
    w.records.write_bam(bam, w.chroms, w.chrom_len)
    kw = dict(min_anchor=0, min_intron=0)
    want_j = junction_oracle.extract(w.records, len(w.chroms), 1, **kw)
    with spliser_b200.Context(0) as fresh:
        j, t = fresh.process_bam_extract(bam, w.chroms, 1, **kw)
        hot = fresh.stats()["n_hot_items"]
    assert _full(j) == _full(want_j)
    assert hot > max(2 ** 18, len(w.records.cigar) // 16 + 2 ** 16), hot
    assert c_oracle.diff_tables(c_oracle.table_dict(t), c_oracle.process(w.records, len(w.chroms), want_j, 1, threads=8)) is None


@pytest.mark.gpu
def test_cli_process_bam_equals_junctions_then_process_on_gpu(ctx, tmp_path):
    from oracle import c4_shape
    from spliser_b200 import cli
    for k, case in enumerate(load_golden("appendix_a.json.gz")["process"]):
        d = tmp_path / ("p%d" % k)
        d.mkdir()
        bam = _write_bam(str(d), [tuple(r) for r in case["reads"]])
        for stranded, stype in MODES:
            for cryptic in (False, True):
                _bam_only_equals_two_steps(cli, ctx, d, bam, stranded, stype, cryptic, (1, 1, 500000))
    chroms, chrom_len, samples = c4_shape.build_samples()
    for i, (title, rec, _) in enumerate(samples[:2]):
        d = tmp_path / ("c4_%d" % i)
        d.mkdir()
        bam = str(d / "s.bam")
        rec.write_bam(bam, chroms, chrom_len)
        assert _bam_only_equals_two_steps(cli, ctx, d, bam, True, "rf", False) > 1000
        assert _bam_only_equals_two_steps(cli, ctx, d, bam, False, None, True) > 1000
