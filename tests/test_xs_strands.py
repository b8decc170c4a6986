"""Junction strands from the aligner's XS tag (SPL_FLAG_XS_STRAND): the aux walk of both BAM readers, extraction with a per-record
strand column, and `junctions` / `processBam --strandFromXS`.

The CPU tests hold the host reader to the restatement of the rule (tests/xs_oracle.py) and run the commands with the extraction
and count answered by the restatements; the GPU tests hold the device ingest and the kernels to the same restatements."""
import ctypes as C
import os

import numpy as np
import pytest

from common import load_golden
from oracle import c_oracle, junction_oracle
from spliser_b200 import Records, api
from test_bam_only_process import ExtractOracleContext
from xs_oracle import encode_aux, extract, star_aux, xs_of_aux

XS = api.FLAG_XS_STRAND
_MD = ("MD", "Z", "12A3XSA+7")                 # the bytes XSA+ inside a Z value are not a field


def _crafted():
    """(name, aux bytes) of hand-made aux blocks."""
    every = [("Ac", "A", "x"), ("cc", "c", -5), ("CC", "C", 200), ("ss", "s", -3000), ("SS", "S", 60000), ("ii", "i", -7),
             ("II", "I", 4000000000), ("ff", "f", 1.5), ("ZZ", "Z", "hello"), ("HH", "H", "1AE301")]
    arrays = [("B" + s, "B", (s, [1, 2, 3])) for s in "cCsSiIf"]
    cases = [
        ("no aux", b""),
        ("XS first", encode_aux([("XS", "A", "+"), ("NH", "i", 1)])),
        ("XS last", encode_aux([("NH", "i", 1), ("HI", "i", 1), ("XS", "A", "-")])),
        ("XS absent", encode_aux([("NH", "i", 1), _MD])),
        ("after every type", encode_aux(every + [("XS", "A", "-")])),
        ("after every B subtype", encode_aux(arrays + [("XS", "A", "+")])),
        ("empty B arrays", encode_aux([("Bz", "B", ("i", [])), ("XS", "A", "-")])),
        ("XS:Z:+", encode_aux([("XS", "Z", "+")])),
        ("XS:i", encode_aux([("XS", "i", 43)])),
        ("XS:A:.", encode_aux([("XS", "A", ".")])),
        ("two XS, + first", encode_aux([("XS", "A", "+"), ("XS", "A", "-")])),
        ("two XS, Z first", encode_aux([("XS", "Z", "-"), ("XS", "A", "-")])),
        ("lowercase xs", encode_aux([("xs", "A", "+")])),
        ("XSA+ inside MD:Z", encode_aux([_MD])),
        ("XSA+ inside MD:Z, then XS", encode_aux([_MD, ("XS", "A", "-")])),
        ("unknown type before XS", b"QQq\x01" + encode_aux([("XS", "A", "+")])),
        ("unknown type after XS", encode_aux([("XS", "A", "+")]) + b"QQq\x01"),
        ("B count past the record", b"BBBI\xff\xff\x00\x00" + encode_aux([("XS", "A", "+")])),
        ("unterminated Z", b"MDZ12A3"),
        ("unterminated Z after XS", encode_aux([("XS", "A", "-")]) + b"MDZ12A3"),
        ("XS:A without its value", b"NHi\x01\x00\x00\x00XSA"),
        ("two stray bytes", encode_aux([("NH", "i", 1)]) + b"XS"),
        ("truncated i", b"NHi\x01\x00"),
    ]
    return cases


def _fuzz(seed, n):
    """Random aux blocks: valid fields with XS anywhere, then truncated, with bytes flipped or replaced by noise."""
    rng = np.random.default_rng(seed)
    kinds = [("A", lambda: chr(rng.choice(list(b"+-.?x")))), ("c", lambda: int(rng.integers(-128, 128))),
             ("C", lambda: int(rng.integers(0, 256))), ("s", lambda: int(rng.integers(-2 ** 15, 2 ** 15))),
             ("S", lambda: int(rng.integers(0, 2 ** 16))), ("i", lambda: int(rng.integers(-2 ** 31, 2 ** 31))),
             ("I", lambda: int(rng.integers(0, 2 ** 32))), ("f", lambda: float(rng.random())),
             ("Z", lambda: "".join(chr(c) for c in rng.choice(list(b"XSA+-0123456789ACGT^"), rng.integers(0, 12)))),
             ("H", lambda: "AB" * int(rng.integers(0, 4))),
             ("B", lambda: (str(rng.choice(list("cCsSiIf"))), [int(x) for x in rng.integers(0, 100, rng.integers(0, 5))]))]
    out = []
    for _ in range(n):
        fields = []
        for _ in range(rng.integers(0, 7)):
            ty, val = kinds[rng.integers(0, len(kinds))]
            tag = rng.choice(["XS", "NH", "MD", "xs", "XA", "SX"], p=[0.3, 0.2, 0.2, 0.1, 0.1, 0.1])
            fields.append((str(tag), ty, val()))
        blob = bytearray(encode_aux(fields))
        mode = rng.integers(0, 4)
        if mode == 1 and blob:
            blob = blob[:rng.integers(0, len(blob))]
        elif mode == 2 and blob:
            blob[rng.integers(0, len(blob))] = int(rng.integers(0, 256))
        elif mode == 3:
            blob += bytes(rng.integers(0, 256, rng.integers(0, 9), dtype=np.uint8))
        out.append(bytes(blob))
    return out


def _one_intron_each(blobs):
    """One record per blob, record i with its own junction (l = 1019 + 1000 i): the table's strand column reads back each
    record's XS."""
    reads = [("C", 1000 + 1000 * i, 0, "20M100N20M") for i in range(len(blobs))]
    return Records.from_reads(["C"], reads)


def _rows(j):
    return list(zip(j.chrom.tolist(), j.left.tolist(), j.right.tolist(), j.score.tolist(), [chr(x) for x in j.strand.tolist()],
                    j.start.tolist(), j.end.tolist()))


# ---------------------------------------------------------------------------------------------------------- CPU
@pytest.mark.parametrize("with_seq", [False, True])
def test_host_reader_xs_equals_the_restatement(tmp_path, built_library, with_seq):
    names = [n for n, _ in _crafted()]
    blobs = [b for _, b in _crafted()] + _fuzz(20261021 + with_seq, 3000)
    rec = _one_intron_each(blobs)
    bam = str(tmp_path / "aux.bam")
    rec.write_bam(bam, ["C"], with_seq=with_seq, aux=blobs)
    back = Records.from_bam(bam, ["C"], xs=True)
    assert len(back) == len(blobs)
    np.testing.assert_array_equal(back.pos, rec.pos)
    want = [xs_of_aux(b) for b in blobs]
    got = [chr(x) for x in back.xs.tolist()]
    for k, name in enumerate(names):
        assert got[k] == want[k], name
    assert got == want
    assert set(want) == {"+", "-", "?"}
    assert Records.from_bam(bam, ["C"]).xs is None          # the plain reader does not walk the tags


def test_restatement_of_the_rule_on_named_cases(built_library):
    want = {"no aux": "?", "XS first": "+", "XS last": "-", "XS absent": "?", "after every type": "-", "after every B subtype": "+",
            "empty B arrays": "-", "XS:Z:+": "?", "XS:i": "?", "XS:A:.": "?", "two XS, + first": "+", "two XS, Z first": "?",
            "lowercase xs": "?", "XSA+ inside MD:Z": "?", "XSA+ inside MD:Z, then XS": "-", "unknown type before XS": "?",
            "unknown type after XS": "+", "B count past the record": "?", "unterminated Z": "?", "unterminated Z after XS": "-",
            "XS:A without its value": "?", "two stray bytes": "?", "truncated i": "?"}
    assert {n: xs_of_aux(b) for n, b in _crafted()} == want


HAND = [("C", 100, 0, "20M100N20M", "+"), ("C", 100, 16, "20M100N20M", "+"), ("C", 105, 0, "15M100N30M", "-"),
        ("C", 90, 0, "30M100N10M", "?"), ("C", 100, 0, "20M60N20M", "+")]
HAND_ROWS = [(0, 119, 219, 1, "?", 89, 229), (0, 119, 219, 2, "+", 99, 239), (0, 119, 219, 1, "-", 104, 249)]


def test_restatement_of_hand_made_extraction(built_library):
    rec = Records.from_reads(["C"], HAND)
    for flags in (0, 1, 3):                                  # the FLAG does not touch XS strands
        assert _rows(extract(rec, 1, flags, xs=rec.xs)) == HAND_ROWS
    assert [r[4] for r in _rows(extract(rec, 1, 0))] == ["?"]


def _tagged(reads, seed):
    """The reads with an XS strand each ('+', '-' or '?') and the aux blocks that carry it ('?': no tag, or XS:A:.)."""
    rng = np.random.default_rng(seed)
    out, aux = [], []
    for r in reads:
        s = str(rng.choice(["+", "-", "?", "?"]))
        fields = [("NH", "i", 1), _MD]
        if s != "?":
            fields.insert(int(rng.integers(0, 3)), ("XS", "A", s))
        elif rng.random() < 0.3:
            fields.append(("XS", "A", "."))
        out.append(tuple(r[:4]) + (s,))
        aux.append(encode_aux(fields))
    return out, aux


class XsOracleContext(ExtractOracleContext):
    """ExtractOracleContext that honours FLAG_XS_STRAND."""

    def extract_junctions_bam(self, bam_path, chrom_names, flags=0, min_anchor=8, min_intron=70, max_intron=500000):
        rec = Records.from_bam(bam_path, chrom_names, xs=True)
        return extract(rec, len(chrom_names), flags & 3, min_anchor, min_intron, max_intron, xs=rec.xs if flags & XS else None)

    def process_bam_extract(self, bam_path, chrom_names, flags=0, min_anchor=8, min_intron=70, max_intron=500000, qchrom="All",
                            gene_bounds=None, window_max_intron=0):
        rec = Records.from_bam(bam_path, chrom_names, xs=True)
        j = extract(rec, len(chrom_names), flags & 3, min_anchor, min_intron, max_intron, xs=rec.xs if flags & XS else None)
        j = junction_oracle.filter_rows(j, chrom_names, qchrom, gene_bounds, window_max_intron)
        return j, api.SiteTable(**c_oracle.process(rec, len(chrom_names), j, flags & ~XS))


def _xs_one_equals_two(cli, ctx, d, bam, stranded, stype, cryptic, bounds=(8, 70, 500000)):
    """processBam --strandFromXS == junctions --strandFromXS + process -b; returns the BED12's strand column."""
    a, m, M = bounds
    bed = str(d / "j.bed")
    cli.junctions(bam, bed, minAnchor=a, minIntron=m, maxIntron=M, strandFromXS=True, ctx=ctx)
    cli.process(bam, bed, str(d / "two"), isStranded=stranded, strandedType=stype, isbeta2Cryptic=cryptic, ctx=ctx)
    cli.processBam(bam, str(d / "one"), isStranded=stranded, strandedType=stype, isbeta2Cryptic=cryptic, minAnchor=a, minIntron=m,
                   maxIntron=M, strandFromXS=True, ctx=ctx)
    two, one = open(str(d / "two.SpliSER.tsv")).read(), open(str(d / "one.SpliSER.tsv")).read()
    assert one == two, (stranded, stype, cryptic, bounds)
    return [line.split("\t")[5] for line in open(bed)]


def test_process_bam_xs_equals_junctions_xs_then_process_on_cpu(tmp_path, built_library):
    from spliser_b200 import cli
    cases = load_golden("appendix_a.json.gz")["process"] + load_golden("process_fuzz.json.gz")[::9]
    ctx = XsOracleContext()
    strands = []
    for k, case in enumerate(cases):
        d = tmp_path / ("p%d" % k)
        d.mkdir()
        reads, aux = _tagged([tuple(r) for r in case["reads"]], 7000 + k)
        refs = sorted({r[0] for r in reads}) or ["C"]
        bam = str(d / "x.bam")
        Records.from_reads(refs, reads).write_bam(bam, refs, aux=aux)
        for stranded, stype in ((False, None), (True, "rf")):
            for bounds in ((8, 70, 500000), (1, 1, 500000)):
                strands += _xs_one_equals_two(cli, ctx, d, bam, stranded, stype, k % 2 == 1, bounds)
    assert {"+", "-", "?"} <= set(strands) and len(strands) > 200


def test_strand_from_xs_argument_parsing(built_library, monkeypatch):
    from spliser_b200 import cli
    seen = {}
    monkeypatch.setattr(cli, "junctions", lambda **kw: seen.update(kw))
    monkeypatch.setattr(cli, "processBam", lambda **kw: seen.update(kw))
    cli.main(["junctions", "-B", "x.bam", "-o", "x.bed", "--strandFromXS"])
    assert seen == dict(inBAM="x.bam", outBed="x.bed", minAnchor=8, minIntron=70, maxIntron=500000, isStranded=False, strandedType=None,
                        strandFromXS=True)
    seen.clear()
    cli.main(["processBam", "-B", "x.bam", "-o", "out", "--strandFromXS", "--isStranded", "-s", "rf"])
    assert seen["strandFromXS"] is True and seen["isStranded"] is True and seen["strandedType"] == "rf"
    seen.clear()
    cli.main(["processBam", "-B", "x.bam", "-o", "out"])
    assert "strandFromXS" not in seen                        # without the flag the call is what it always was
    with pytest.raises(SystemExit):                          # two strand sources for one table
        cli.main(["junctions", "-B", "x.bam", "-o", "x.bed", "--strandFromXS", "--isStranded", "-s", "fr"])


def test_records_xs_validation(built_library):
    with pytest.raises(ValueError):
        Records.from_reads(["C"], [("C", 1, 0, "5M", "+"), ("C", 2, 0, "5M")])
    with pytest.raises(ValueError):
        Records([1], [0], [0, 1], [80], [0], [0, 1], xs=[43, 45])


# ---------------------------------------------------------------------------------------------------------- GPU
def _tagged_sample(tmp_path, seed, stranded, n=120_000, name=None):
    from spliser_b200 import synth
    w = synth.generate(synth.config_small(n, seed=seed, stranded=stranded, paired=stranded))
    xs, aux = star_aux(w.records, seed)
    bam = str(tmp_path / (name or "xs%d.bam" % seed))
    w.records.write_bam(bam, w.chroms, w.chrom_len, aux=aux)
    rec = Records(w.records.pos, w.records.flag, w.records.cig_off, w.records.cigar, w.records.seg_chrom, w.records.seg_off, xs=xs)
    return w, rec, bam, aux


@pytest.mark.gpu
@pytest.mark.parametrize("host_bam", [False, True])
def test_device_xs_equals_host_xs_per_record(ctx, tmp_path, monkeypatch, host_bam):
    if host_bam:
        monkeypatch.setenv("SPLISER_HOST_BAM", "1")
    for with_seq in (False, True):
        blobs = [b for _, b in _crafted()] + _fuzz(31 + with_seq, 3000)
        rec = _one_intron_each(blobs)
        bam = str(tmp_path / ("d%d.bam" % with_seq))
        rec.write_bam(bam, ["C"], with_seq=with_seq, aux=blobs)
        j = ctx.extract_junctions_bam(bam, ["C"], XS)
        assert ctx.stats()["bam_on_device"] == (0.0 if host_bam else 1.0)
        assert j.left.tolist() == [1019 + 1000 * i for i in range(len(blobs))]
        assert [chr(x) for x in j.strand.tolist()] == [xs_of_aux(b) for b in blobs]
        host = Records.from_bam(bam, ["C"], xs=True)
        np.testing.assert_array_equal(j.strand, host.xs)


@pytest.mark.gpu
def test_xs_extraction_equals_the_restatement(ctx, tmp_path):
    from oracle import fuzzgen
    rng = np.random.default_rng(5150)
    rows = 0
    for seed in range(970000, 970200):
        case = fuzzgen.gen_long_case(seed, dirty=(seed % 4 == 1))
        chroms = sorted({r[0] for r in case["reads"]}) or ["C"]
        base = Records.from_reads(chroms, [tuple(r) for r in case["reads"]])
        xs = rng.choice(np.frombuffer(b"+-?", np.uint8), len(base))
        rec = Records(base.pos, base.flag, base.cig_off, base.cigar, base.seg_chrom, base.seg_off, xs=xs)
        for flags, kw in ((XS, {}), (XS | 3, dict(min_anchor=1, min_intron=1))):
            want = extract(rec, len(chroms), flags & 3, xs=xs, **kw)
            assert _rows(ctx.extract_junctions_records(rec, len(chroms), flags, **kw)) == _rows(want), seed
            rows += len(want)
        if seed % 10 == 0:                                   # the BAM path, XS written as tags
            bam = str(tmp_path / ("f%d.bam" % seed))
            rec.write_bam(bam, chroms, aux=[encode_aux([("XS", "A", chr(s))]) if s != ord("?") else b"" for s in xs.tolist()])
            assert _rows(ctx.extract_junctions_bam(bam, chroms, XS, min_anchor=1, min_intron=1)) == \
                _rows(extract(rec, len(chroms), 0, min_anchor=1, min_intron=1, xs=xs)), seed
    assert rows > 1000
    hand = Records.from_reads(["C"], HAND)
    assert _rows(ctx.extract_junctions_records(hand, 1, XS)) == HAND_ROWS
    untagged = Records.from_reads(["C"], [r[:4] for r in HAND])
    with pytest.raises(ValueError):                          # no strand column to read
        ctx.extract_junctions_records(untagged, 1, XS)
    v, h = untagged.view(), C.c_void_p()
    assert ctx._lib.spl_extract_junctions_records(ctx._h, C.byref(v), 1, 8, 70, 500000, XS, C.byref(h)) == -1     # SPL_ERR_ARG
    for stranded, seed in ((False, 5), (True, 6)):
        w, rec, bam, _ = _tagged_sample(tmp_path, seed, stranded)
        want = extract(rec, len(w.chroms), 0, xs=rec.xs)
        assert {"+", "-", "?"} <= {chr(s) for s in want.strand.tolist()}
        assert _rows(ctx.extract_junctions_records(rec, len(w.chroms), XS)) == _rows(want)
        assert _rows(ctx.extract_junctions_records(rec, len(w.chroms), XS | 3)) == _rows(want)
        assert _rows(ctx.extract_junctions_bam(bam, w.chroms, XS)) == _rows(want)


@pytest.mark.gpu
@pytest.mark.parametrize("host_bam", [False, True])
def test_process_bam_extract_xs_equals_extract_then_process(ctx, tmp_path, monkeypatch, host_bam):
    if host_bam:
        monkeypatch.setenv("SPLISER_HOST_BAM", "1")
    for stranded, seed in ((False, 5), (True, 6)):
        w, rec, bam, _ = _tagged_sample(tmp_path, seed, stranded)
        mid = int(np.median(w.junctions.left))
        for count_flags in (0, 3, 4):
            for qchrom, bounds, win in (("All", None, 0), (w.chroms[0], None, 0), ("All", (mid, mid + 20000), 5000)):
                jw = ctx.extract_junctions_bam(bam, w.chroms, XS)
                jw = junction_oracle.filter_rows(jw, w.chroms, qchrom, bounds, win)
                tw = ctx.process_bam(bam, w.chroms, jw, count_flags)
                j, t = ctx.process_bam_extract(bam, w.chroms, count_flags | XS, qchrom=qchrom, gene_bounds=bounds, window_max_intron=win)
                assert ctx.stats()["bam_on_device"] == (0.0 if host_bam else 1.0)
                assert _rows(j) == _rows(jw), (count_flags, qchrom, bounds)
                want_j = junction_oracle.filter_rows(extract(rec, len(w.chroms), 0, xs=rec.xs), w.chroms, qchrom, bounds, win)
                assert _rows(j) == _rows(want_j)
                assert c_oracle.diff_tables(c_oracle.table_dict(t), c_oracle.table_dict(tw)) is None, (count_flags, qchrom)
                want = c_oracle.process(w.records, len(w.chroms), j, count_flags, threads=8)
                assert c_oracle.diff_tables(c_oracle.table_dict(t), want) is None, (count_flags, qchrom, bounds)
                assert len(j) > 0


@pytest.mark.gpu
def test_cli_process_bam_xs_equals_junctions_xs_then_process_on_gpu(ctx, tmp_path):
    from spliser_b200 import cli
    _, _, bam, _ = _tagged_sample(tmp_path, 8, True)
    for stranded, stype in ((False, None), (True, "rf")):
        d = tmp_path / ("c%d" % stranded)
        d.mkdir()
        strands = _xs_one_equals_two(cli, ctx, d, bam, stranded, stype, False)
        assert {"+", "-", "?"} <= set(strands) and len(strands) > 500


@pytest.mark.gpu
def test_process_bam_extract_xs_ingests_once(ctx, tmp_path):
    w, _, bam, _ = _tagged_sample(tmp_path, 7, True, n=400_000)
    j, _ = ctx.process_bam_extract(bam, w.chroms, w.flags | XS)
    one = ctx.stats()
    ctx.process_bam(bam, w.chroms, j, w.flags)
    ref = ctx.stats()
    assert one["bam_on_device"] == 1.0 and ref["bam_on_device"] == 1.0
    chunk_table = 48 * (len(w.records) // 1024 + len(w.chroms) + 1)
    assert one["h2d_bytes"] <= ref["h2d_bytes"] + 21 * len(j) + chunk_table, (one["h2d_bytes"], ref["h2d_bytes"])
    assert one["h2d_bytes"] - ref["h2d_bytes"] < os.path.getsize(bam) / 4


@pytest.mark.gpu
def test_default_extraction_ignores_the_tags(ctx, tmp_path):
    w, _, tagged, _ = _tagged_sample(tmp_path, 9, True)
    plain = str(tmp_path / "plain.bam")
    w.records.write_bam(plain, w.chroms, w.chrom_len)
    for flags in (0, 1, 3):
        assert _rows(ctx.extract_junctions_bam(tagged, w.chroms, flags)) == _rows(ctx.extract_junctions_bam(plain, w.chroms, flags))
    ja, ta = ctx.process_bam_extract(tagged, w.chroms, w.flags)
    jb, tb = ctx.process_bam_extract(plain, w.chroms, w.flags)
    assert _rows(ja) == _rows(jb)
    assert c_oracle.diff_tables(c_oracle.table_dict(ta), c_oracle.table_dict(tb)) is None
