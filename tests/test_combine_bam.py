"""`combineBam` and the device-resident samples behind it (Context.load_bam -> DeviceSample): every BAM of a multi-sample run is
ingested once, its records stay in GPU memory for the extraction + count and for the re-count of the sites the sample lacks.

The CPU tests run the host layers for real with stand-in contexts whose load_bam returns a host-side stand-in sample answered
by the restatements (oracle/junction_oracle.py for the extraction, the C oracle for the counts): combineBam must write exactly
what `processBam` per sample followed by `combine` / `combineShallow` writes.  The GPU tests hold the resident calls to the
path calls (spl_process_bam_extract, spl_recount) and to the C oracle."""
import hashlib
import os

import numpy as np
import pytest

from oracle import c4_shape, c_oracle, junction_oracle
from spliser_b200 import Records, api
from test_bam_only_process import ExtractOracleContext, _full

SHALLOW = c4_shape.SIX.shallow


# ---------------------------------------------------------------------------------------------------------- fixtures
class HostSample:
    """Stand-in DeviceSample: the BAM's records on the host under the header's reference order, mapped to a caller's chromosome
    list by name (first index of a repeated name) as spl_sample_* does."""

    def __init__(self, owner, path, xs):
        self.owner, self.path = owner, path
        self.refs = api.bam_reference_names(path)
        self.rec = Records.from_bam(path, self.refs, xs=xs)
        self.closed = False

    def _records(self, chrom_names):
        index = {}
        for i, c in enumerate(chrom_names):
            index.setdefault(c, i)
        m = np.array([index.get(r, -1) for r in self.refs] + [-1], np.int32)
        r = self.rec
        return Records(r.pos, r.flag, r.cig_off, r.cigar, m[r.seg_chrom], r.seg_off, xs=r.xs)

    def process_extract(self, chrom_names, flags=0, min_anchor=8, min_intron=70, max_intron=500000, qchrom="All", gene_bounds=None,
                        window_max_intron=0):
        assert not self.closed
        rec = self._records(chrom_names)
        j = junction_oracle.extract(rec, len(chrom_names), flags & 3, min_anchor, min_intron, max_intron)
        j = junction_oracle.filter_rows(j, chrom_names, qchrom, gene_bounds, window_max_intron)
        return j, api.SiteTable(**c_oracle.process(rec, len(chrom_names), j, flags))

    def recount(self, chrom_names, gaps, flags):
        assert not self.closed
        self.owner.sample_recounts.append(self.path)
        return c_oracle.recount(self._records(chrom_names), len(chrom_names), gaps, flags)

    def close(self):
        self.closed = True

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()


class ResidentOracleContext(ExtractOracleContext):
    """ExtractOracleContext with load_bam; the BAMs named in `refuse` raise SampleMemoryError, as a full device would."""

    def __init__(self, refuse=()):
        self.refuse = set(refuse)
        self.samples, self.path_extracts, self.path_recounts, self.sample_recounts = [], [], [], []

    def load_bam(self, bam_path, xs=False):
        if os.path.basename(bam_path) in self.refuse:
            raise api.SampleMemoryError("stand-in: %s does not fit" % bam_path)
        s = HostSample(self, bam_path, xs)
        self.samples.append(s)
        return s

    def process_bam_extract(self, bam_path, *a, **kw):
        self.path_extracts.append(bam_path)
        return super().process_bam_extract(bam_path, *a, **kw)

    def recount_bam(self, bam_path, chrom_names, gaps, flags):
        self.path_recounts.append(bam_path)
        return super().recount_bam(bam_path, chrom_names, gaps, flags)


@pytest.fixture(scope="module")
def memo_extract():
    """The Python extraction restatement is slow on c4's 200k-record samples and every comparison asks it the same questions
    twice (combineBam and processBam): answer repeats from a cache keyed by the records' bytes."""
    mp = pytest.MonkeyPatch()
    plain, memo = junction_oracle.extract, {}

    def extract(rec, n_chrom, flags=0, min_anchor=8, min_intron=70, max_intron=500000):
        h = hashlib.sha1()
        for a in (rec.pos, rec.flag, rec.cig_off, rec.cigar, rec.seg_chrom, rec.seg_off):
            h.update(np.ascontiguousarray(a).tobytes())
        key = (h.digest(), n_chrom, flags, min_anchor, min_intron, max_intron)
        if key not in memo:
            memo[key] = plain(rec, n_chrom, flags, min_anchor, min_intron, max_intron)
        return memo[key]
    mp.setattr(junction_oracle, "extract", extract)
    yield
    mp.undo()


def _write_c4(d, shape=c4_shape.SIX):
    """BAMs of c4_shape's samples and a GFF of its genome -> (titles, bam paths, gff path)."""
    from oracle.c2_annotated import gff_lines
    chroms, chrom_len, samples = c4_shape.build_samples(shape)
    os.makedirs(d, exist_ok=True)
    bams = []
    for i, (title, rec, _) in enumerate(samples):
        bams.append(os.path.join(d, "s%d.bam" % i))
        rec.write_bam(bams[-1], chroms, chrom_len)
    gff = os.path.join(d, "genes.gff")
    with open(gff, "w") as fh:
        fh.write("##gff-version 3\n" + "".join(gff_lines(chroms, chrom_len)))
    return [s[0] for s in samples], bams, gff


@pytest.fixture(scope="module")
def c4_files(tmp_path_factory, built_library):
    return _write_c4(str(tmp_path_factory.mktemp("c4")))


def _busy_gene(cli, ctx, d, bam, gff):
    """The gene with the most sites in a sample's annotated table: what -g names in the tests."""
    from collections import Counter
    out = os.path.join(d, "probe")
    cli.processBam(bam, out, annotationFile=gff, ctx=ctx)
    lines = open(out + ".SpliSER.tsv").read().splitlines()
    col = lines[0].split("\t").index("Gene")
    gene, n = Counter(x.split("\t")[col] for x in lines[1:] if x.split("\t")[col] != "NA").most_common(1)[0]
    assert n >= 4
    return gene


def _samples_file(d, titles, bams, tag):
    tsvs = [os.path.join(d, "%s%d.SpliSER.tsv" % (tag, i)) for i in range(len(bams))]
    sf = os.path.join(d, "%s_samples.tsv" % tag)
    with open(sf, "w") as fh:
        fh.writelines("%s\t%s\t%s\n" % x for x in zip(titles, tsvs, bams))
    return sf, tsvs


def _reference(cli, ctx, d, titles, bams, annotation=None, gene="All", stranded=False, stype=None, cryptic=False, xs=False,
               shallow=False):
    """processBam per sample, then combine / combineShallow over its files -> (per-sample TSV texts, combined text)."""
    sf, tsvs = _samples_file(d, titles, bams, "ref")
    texts = []
    for bam, tsv in zip(bams, tsvs):
        cli.processBam(bam, tsv[:-len(".SpliSER.tsv")], annotationFile=annotation, isStranded=stranded, strandedType=stype,
                       isbeta2Cryptic=cryptic, ctx=ctx, **(dict(strandFromXS=True) if xs else {}))
        texts.append(open(tsv).read())
    out = os.path.join(d, "ref")
    st = dict(strandedType=stype) if stype else {}
    if shallow:
        cli.combineShallow(sf, out, qGene=gene, isStranded=stranded, minSamples=SHALLOW[0], minReads=SHALLOW[1], minSSE=SHALLOW[2],
                           isbeta2Cryptic=cryptic, ctx=ctx, **st)
    else:
        cli.combine(sf, out, qGene=gene, isStranded=stranded, isbeta2Cryptic=cryptic, ctx=ctx, **st)
    return texts, open(out + ".combined.tsv").read()


def _combine_bam(cli, d, titles, bams, tag, annotation=None, gene="All", stranded=False, stype=None, cryptic=False, xs=False,
                 shallow=False, **kw):
    sf, tsvs = _samples_file(d, titles, bams, tag)
    out = os.path.join(d, tag)
    cli.combineBam(sf, out, annotationFile=annotation, qGene=gene, isStranded=stranded, strandedType=stype, isbeta2Cryptic=cryptic,
                   strandFromXS=xs, shallow=shallow, minSamples=SHALLOW[0], minReads=SHALLOW[1], minSSE=SHALLOW[2], **kw)
    return [open(t).read() for t in tsvs], open(out + ".combined.tsv").read()


CASES = {
    "unstranded": dict(),
    "rf": dict(stranded=True, stype="rf"),
    "unstranded_cryptic": dict(cryptic=True),
    "rf_cryptic": dict(stranded=True, stype="rf", cryptic=True),
    "annotated_gene": dict(stranded=True, stype="rf", annotated=True),
    "shallow": dict(stranded=True, stype="rf", shallow=True),
}


# ---------------------------------------------------------------------------------------------------------- CPU
@pytest.mark.parametrize("case", sorted(CASES))
def test_combine_bam_equals_process_bam_then_combine_on_cpu(tmp_path, c4_files, memo_extract, case):
    from spliser_b200 import cli
    titles, bams, gff = c4_files
    kw = dict(CASES[case])
    d = str(tmp_path)
    if kw.pop("annotated", False):
        kw["annotation"] = gff
        kw["gene"] = _busy_gene(cli, ExtractOracleContext(), d, bams[0], gff)
    ref_tsvs, ref_combined = _reference(cli, ExtractOracleContext(), d, titles, bams, **kw)
    made = []

    def factory(device):
        made.append(ResidentOracleContext())
        return made[-1]
    tsvs, combined = _combine_bam(cli, d, titles, bams, "one", context_factory=factory, **kw)
    assert tsvs == ref_tsvs
    assert combined == ref_combined
    assert combined.count("\n") > (4 if "gene" in kw else 1000)
    c, = made
    assert len(c.samples) == 6 and not c.path_extracts and not c.path_recounts
    assert all(s.closed for s in c.samples)
    assert len(c.sample_recounts) >= 1                     # every re-count came from a resident sample


def test_combine_bam_over_three_contexts_and_refused_samples_on_cpu(tmp_path, c4_files, memo_extract):
    from spliser_b200 import cli
    titles, bams, _ = c4_files
    d = str(tmp_path)
    kw = dict(stranded=True, stype="rf")
    ref_tsvs, ref_combined = _reference(cli, ExtractOracleContext(), d, titles, bams, **kw)
    for refuse in ((), ("s1.bam", "s4.bam"), tuple("s%d.bam" % i for i in range(6))):
        made = {}

        def factory(device):
            made[device] = ResidentOracleContext(refuse)
            return made[device]
        tag = "r%d" % len(refuse)
        tsvs, combined = _combine_bam(cli, d, titles, bams, tag, devices=[0, 1, 2], context_factory=factory, **kw)
        assert tsvs == ref_tsvs and combined == ref_combined, refuse
        assert sorted(made) == [0, 1, 2]
        for rank, c in made.items():                       # the same samples on the same rank in both phases
            mine = {bams[k] for k in range(rank, 6, 3)}
            assert {s.path for s in c.samples} == {b for b in mine if os.path.basename(b) not in refuse}
            assert set(c.path_extracts) == {b for b in mine if os.path.basename(b) in refuse}
            assert set(c.path_recounts) <= set(c.path_extracts) and set(c.sample_recounts) <= mine
            assert all(s.closed for s in c.samples)


def test_combine_bam_command_line(tmp_path, built_library, monkeypatch):
    from spliser_b200 import cli
    seen = {}
    monkeypatch.setattr(cli, "combineBam", lambda **kw: seen.update(kw))
    cli.main(["combineBam", "-S", "s.tsv", "-o", "out"])
    assert seen == dict(samplesFile="s.tsv", outputPath="out", annotationFile=None, aType="gene", qGene="All", isStranded=False,
                        strandedType=None, isbeta2Cryptic=False, minAnchor=8, minIntron=70, maxIntron=500000, strandFromXS=False,
                        shallow=False, minSamples=0, minReads=10, minSSE=0.0, devices=[0])
    seen.clear()
    cli.main(["combineBam", "-S", "s.tsv", "-o", "out", "-A", "g.gff", "-t", "mRNA", "-g", "G1", "--isStranded", "-s", "rf",
              "--beta2Cryptic", "--minAnchor", "4", "--minIntron", "20", "--maxIntron", "9000", "--strandFromXS", "--shallow",
              "-m", "3", "-r", "12", "-e", "0.25", "--gpus", "3"])
    assert seen == dict(samplesFile="s.tsv", outputPath="out", annotationFile="g.gff", aType="mRNA", qGene="G1", isStranded=True,
                        strandedType="rf", isbeta2Cryptic=True, minAnchor=4, minIntron=20, maxIntron=9000, strandFromXS=True,
                        shallow=True, minSamples=3, minReads=12, minSSE=0.25, devices=[0, 1, 2])
    for argv in (["combineBam", "-S", "s.tsv", "-o", "out", "--isStranded"],            # --isStranded requires -s
                 ["combineBam", "-S", "s.tsv", "-o", "out", "-g", "G1"],                # -g requires -A
                 ["combineBam", "-o", "out"], ["combineBam", "-S", "s.tsv"]):
        with pytest.raises(SystemExit):
            cli.main(argv)


def test_malformed_samples_file_raises_in_combine_mode_and_is_skipped_in_shallow_mode(tmp_path, c4_files, memo_extract):
    from spliser_b200 import cli
    titles, bams, _ = c4_files
    d = str(tmp_path)
    sf, tsvs = _samples_file(d, titles[:2], bams[:2], "m")
    with open(sf, "a") as fh:
        fh.write("only\ttwo\n")
    with pytest.raises(Exception, match="exactly 3 tab-separated columns"):
        cli.combineBam(sf, os.path.join(d, "m"), context_factory=lambda dev: ResidentOracleContext())
    assert not any(os.path.exists(t) for t in tsvs)        # refused before any sample was processed
    cli.combineBam(sf, os.path.join(d, "m"), shallow=True, context_factory=lambda dev: ResidentOracleContext())
    assert all(os.path.exists(t) for t in tsvs)
    ref = os.path.join(d, "m_ref")
    cli.combineShallow(sf, ref, minSamples=0, minReads=10, minSSE=0.0, ctx=ExtractOracleContext())
    assert open(os.path.join(d, "m.combined.tsv")).read() == open(ref + ".combined.tsv").read()


# ---------------------------------------------------------------------------------------------------------- GPU
def _split(w, n, seed):
    """n samples of one synthetic workload: every record goes to one sample."""
    owner = np.random.default_rng(seed).integers(0, n, len(w.records))
    return [c4_shape._subset(w.records, owner == k) for k in range(n)]


def _gap_cases(ctx, cli, d, bams, flags_stranded, stype):
    """Gap lists of a real merge of the samples' processBam tables: [(bam, header-local chromosome list, GapTable)]."""
    from spliser_b200.hosttext import CombineMerge
    tsvs = []
    for i, bam in enumerate(bams):
        out = os.path.join(d, "g%d" % i)
        cli.processBam(bam, out, isStranded=flags_stranded, strandedType=stype, ctx=ctx)
        tsvs.append(out + ".SpliSER.tsv")
    cases = []
    with CombineMerge() as cm:
        cm.add_samples(["t%d" % i for i in range(len(bams))], tsvs)
        regions = cm.region_names()
        cm.merge(list(range(len(regions))), "All", flags_stranded)
        for k, bam in enumerate(bams):
            g = cm.gaps(k)
            if not len(g):
                continue
            # a chromosome list that reorders the header's names, drops those without gaps and adds one the BAM lacks
            used = sorted(set(g.chrom.tolist()), reverse=True)
            names = ["chrNOPE"] + [regions[r] for r in used]
            remap = np.full(len(regions), -1, np.int32)
            remap[used] = np.arange(1, len(used) + 1, dtype=np.int32)
            g.chrom = np.ascontiguousarray(remap[g.chrom])
            cases.append((bam, names, g))
    assert cases
    return cases


@pytest.mark.gpu
@pytest.mark.parametrize("host_bam", [False, True])
def test_resident_sample_equals_the_path_calls(ctx, tmp_path, monkeypatch, host_bam):
    from spliser_b200 import cli, synth
    if host_bam:
        monkeypatch.setenv("SPLISER_HOST_BAM", "1")
    for stranded, paired, seed in ((False, False, 5), (True, True, 6)):
        w = synth.generate(synth.config_small(120_000, seed=seed, stranded=stranded, paired=paired))
        bam = str(tmp_path / ("e%d.bam" % seed))
        w.records.write_bam(bam, w.chroms, w.chrom_len)
        mid = int(np.median(w.junctions.left))
        with ctx.load_bam(bam) as s:
            st = ctx.stats()
            assert st["bam_on_device"] == (0.0 if host_bam else 1.0)
            assert s.n_records == len(w.records) and s.device_bytes >= 10 * len(w.records) + 4 * len(w.records.cigar)
            for flags in ((w.flags & 3), (w.flags & 3) | 4):
                for qchrom, bounds, win in (("All", None, 0), (w.chroms[0], None, 0), ("All", (mid, mid + 20000), 5000),
                                            (w.chroms[-1], (mid, mid + 20000), 0), ("NOPE", None, 0)):
                    jw, tw = ctx.process_bam_extract(bam, w.chroms, flags, qchrom=qchrom, gene_bounds=bounds, window_max_intron=win)
                    j, t = s.process_extract(w.chroms, flags, qchrom=qchrom, gene_bounds=bounds, window_max_intron=win)
                    assert _full(j) == _full(jw), (qchrom, bounds)
                    assert c_oracle.diff_tables(c_oracle.table_dict(t), c_oracle.table_dict(tw)) is None, (flags, qchrom, bounds)
                    assert (len(j) > 0) == (qchrom != "NOPE")
            # the caller's list may order the names differently from the header and leave some out
            rev = list(reversed(w.chroms))[:-1] + ["chrNOPE"]
            jw, tw = ctx.process_bam_extract(bam, rev, w.flags & 3)
            j, t = s.process_extract(rev, w.flags & 3)
            assert _full(j) == _full(jw) and c_oracle.diff_tables(c_oracle.table_dict(t), c_oracle.table_dict(tw)) is None
        # re-count: gap lists of a real merge of three samples of the workload
        d = str(tmp_path / ("m%d" % seed))
        os.makedirs(d)
        bams = []
        for k, r in enumerate(_split(w, 3, seed)):
            bams.append(os.path.join(d, "s%d.bam" % k))
            r.write_bam(bams[-1], w.chroms, w.chrom_len)
        flags = api.mode_flags(stranded, "rf" if stranded else None, combine=True)
        for bam, names, g in _gap_cases(ctx, cli, d, bams, stranded, "rf" if stranded else None):
            want = c_oracle.recount(Records.from_bam(bam, names), len(names), g, flags)
            path = ctx.recount_bam(bam, names, g, flags)
            with ctx.load_bam(bam) as s:
                got = s.recount(names, g, flags)
            for a, b, c in zip(got, path, want):
                assert np.array_equal(a, b) and np.array_equal(a, c)


@pytest.mark.gpu
@pytest.mark.parametrize("host_bam", [False, True])
def test_resident_sample_with_xs_strands(ctx, tmp_path, monkeypatch, host_bam):
    from test_xs_strands import _tagged_sample
    if host_bam:
        monkeypatch.setenv("SPLISER_HOST_BAM", "1")
    for stranded, seed in ((False, 41), (True, 42)):
        w, rec, bam, _ = _tagged_sample(tmp_path, seed, stranded)
        flags = (w.flags & 3) | api.FLAG_XS_STRAND
        jw, tw = ctx.process_bam_extract(bam, w.chroms, flags)
        with ctx.load_bam(bam, xs=True) as s:
            j, t = s.process_extract(w.chroms, flags)
        assert _full(j) == _full(jw) and len(j) > 0
        assert set(j.strand.tolist()) >= {ord("+"), ord("-")}
        assert c_oracle.diff_tables(c_oracle.table_dict(t), c_oracle.table_dict(tw)) is None
        with ctx.load_bam(bam) as s:                       # loaded without the XS column: the flag has nothing to read
            with pytest.raises(api.SpliserError):
                s.process_extract(w.chroms, flags)
            j2, _ = s.process_extract(w.chroms, w.flags & 3)
            assert len(j2) > 0                             # and the context carries on


@pytest.mark.gpu
def test_interleaved_resident_samples_give_what_each_gives_alone(ctx, tmp_path):
    """The context's scratch (inflate buffers, extraction and counting memory) must never overwrite resident records."""
    from spliser_b200 import cli, synth
    w = synth.generate(synth.config_small(300_000, seed=11, stranded=True, paired=True))
    d = str(tmp_path)
    bams = []
    for k, r in enumerate(_split(w, 5, 11)):
        bams.append(os.path.join(d, "s%d.bam" % k))
        r.write_bam(bams[-1], w.chroms, w.chrom_len)
    flags = w.flags & 3
    gaps = {bam: (names, g) for bam, names, g in _gap_cases(ctx, cli, d, bams, True, "rf" if flags & 2 else "fr")}
    cflags = api.mode_flags(True, "rf" if flags & 2 else "fr", combine=True)
    alone = {}
    for bam in bams:
        j, t = ctx.process_bam_extract(bam, w.chroms, flags)
        names, g = gaps.get(bam, ([w.chroms[0]], api.GapTable.from_tuples([])))
        alone[bam] = (_full(j), c_oracle.table_dict(t), ctx.recount_bam(bam, names, g, cflags))

    def check(s, bam, what):
        if what == "process":
            j, t = s.process_extract(w.chroms, flags)
            assert _full(j) == alone[bam][0] and c_oracle.diff_tables(c_oracle.table_dict(t), alone[bam][1]) is None, bam
        else:
            names, g = gaps.get(bam, ([w.chroms[0]], api.GapTable.from_tuples([])))
            for a, b in zip(s.recount(names, g, cflags), alone[bam][2]):
                assert np.array_equal(a, b), bam
    a, b = ctx.load_bam(bams[0]), ctx.load_bam(bams[1])
    for s, bam, what in ((b, bams[1], "process"), (a, bams[0], "process"), (a, bams[0], "recount"), (b, bams[1], "recount")):
        check(s, bam, what)
    more = [a, b] + [ctx.load_bam(x) for x in bams[2:]]
    order = [4, 0, 3, 1, 2]
    for i in order:
        check(more[i], bams[i], "process")
    ctx.process_bam_extract(bams[2], w.chroms, flags)      # a path call in between re-uses the ingest scratch
    for i in reversed(order):
        check(more[i], bams[i], "recount")
        check(more[i], bams[i], "process")
    for s in more:
        s.close()


@pytest.mark.gpu
def test_resident_sample_ingests_once(ctx, tmp_path):
    from spliser_b200 import synth
    w = synth.generate(synth.config_small(400_000, seed=7, stranded=True, paired=True))
    bam = str(tmp_path / "once.bam")
    w.records.write_bam(bam, w.chroms, w.chrom_len, with_seq=True)     # sequencer-shaped: a records-only file is a few bytes per read
    size = os.path.getsize(bam)
    with ctx.load_bam(bam) as s:
        load = ctx.stats()
        j, t = s.process_extract(w.chroms, w.flags)
        proc = ctx.stats()
        g = api.GapTable.from_tuples([(int(t.chrom[i]), int(t.pos[i]), t.strand_str(i), list(t.partners(i)), t.competitors(i))
                                      for i in range(0, len(t), 7)])
        flags = api.mode_flags(True, "rf" if w.flags & 2 else "fr", combine=True)
        got = s.recount(w.chroms, g, flags)
        rec = ctx.stats()
    assert load["bam_on_device"] == 1.0
    # the file image and its member table (24 B per BGZF member of at most 64 KiB inflated)
    assert size <= load["h2d_bytes"] <= size * 1.01
    # then only the junction table (21 B per row) and the chunk tables (48 B per 1024 records of a chromosome) of the extraction
    # and the count, and the re-count's gap table: no second file image
    chunk_table = 48 * (len(w.records) // 1024 + len(w.chroms) + 1)
    assert proc["h2d_bytes"] <= 21 * len(j) + 2 * chunk_table, proc["h2d_bytes"]
    assert rec["h2d_bytes"] < 0.01 * size, rec["h2d_bytes"]
    want = ctx.recount_bam(bam, w.chroms, g, flags)
    assert all(np.array_equal(a, b) for a, b in zip(got, want))


@pytest.mark.gpu
def test_freeing_keeps_resident_bytes_constant(ctx, tmp_path):
    import spliser_b200
    from spliser_b200 import synth
    w = synth.generate(synth.config_small(120_000, seed=5))
    bam = str(tmp_path / "f.bam")
    w.records.write_bam(bam, w.chroms, w.chrom_len)
    jw, tw = ctx.process_bam_extract(bam, w.chroms, 0)
    sizes = []
    for _ in range(20):
        s = ctx.load_bam(bam)
        sizes.append(s.device_bytes)
        s.close()
    assert len(set(sizes)) == 1 and sizes[0] > 0
    with ctx.load_bam(bam) as s:
        j, t = s.process_extract(w.chroms, 0)
        assert _full(j) == _full(jw) and c_oracle.diff_tables(c_oracle.table_dict(t), c_oracle.table_dict(tw)) is None
        with spliser_b200.Context(0) as other:             # a sample belongs to the context that loaded it
            with pytest.raises(api.SpliserError, match="another context"):
                other._extract_and_count(other._lib.spl_sample_process_extract, s._h, w.chroms, 0, 8, 70, 500000, "All", None, 0)
    j, t = ctx.process_bam_extract(bam, w.chroms, 0)
    assert _full(j) == _full(jw)


class _CountingContext:
    """Context factory for the CLI tests: records which samples load_bam refused."""

    def __init__(self):
        self.refused = []

    def __call__(self, device):
        import spliser_b200
        owner = self

        class Ctx(spliser_b200.Context):
            def load_bam(self, bam_path, xs=False):
                try:
                    return super().load_bam(bam_path, xs)
                except api.SampleMemoryError:
                    owner.refused.append(os.path.basename(bam_path))
                    raise
        return Ctx(device)


@pytest.mark.gpu
def test_cli_combine_bam_equals_process_bam_then_combine_on_gpu(ctx, tmp_path, monkeypatch):
    import ctypes
    from spliser_b200 import cli
    titles, bams, gff = _write_c4(str(tmp_path / "in"))
    n_dev = ctypes.c_int(0)
    ctypes.CDLL("libcuda.so.1").cuDeviceGetCount(ctypes.byref(n_dev))
    three = [0, 1, 2] if n_dev.value >= 3 else [0, 0, 0]
    with ctx.load_bam(bams[0]) as s:
        one = s.device_bytes
    gene = _busy_gene(cli, ctx, str(tmp_path), bams[0], gff)
    for kw in (dict(stranded=True, stype="rf"), dict(cryptic=True, annotation=gff, gene=gene, stranded=True, stype="rf"),
               dict(stranded=True, stype="rf", shallow=True), dict()):
        d = str(tmp_path / ("k%d" % len(os.listdir(str(tmp_path)))))
        os.makedirs(d)
        ref = _reference(cli, ctx, d, titles, bams, **kw)
        assert ref[1].count("\n") > (4 if "gene" in kw else 1000)
        runs = [("one", [0], None, 0), ("three", three, None, 0), ("budget0", [0], "0", 6),
                ("budget3", [0], str(int(3.5 * one) >> 20), 3)]
        for tag, devices, budget, n_refused in runs:
            if budget is None:
                monkeypatch.delenv("SPLISER_SAMPLE_BUDGET_MB", raising=False)
            else:
                monkeypatch.setenv("SPLISER_SAMPLE_BUDGET_MB", budget)
            counting = _CountingContext()
            got = _combine_bam(cli, d, titles, bams, tag, devices=devices, context_factory=counting, **kw)
            assert got == ref, (kw, tag)
            assert len(counting.refused) == n_refused, (tag, counting.refused)
        monkeypatch.delenv("SPLISER_SAMPLE_BUDGET_MB", raising=False)


@pytest.mark.gpu
def test_cli_combine_bam_with_48_samples(ctx, tmp_path):
    from spliser_b200 import cli
    titles, bams, _ = _write_c4(str(tmp_path / "in"), c4_shape.FORTY_EIGHT)
    d = str(tmp_path)
    kw = dict(stranded=True, stype="rf")
    ref = _reference(cli, ctx, d, titles, bams, **kw)
    assert _combine_bam(cli, d, titles, bams, "b48", devices=[0], **kw) == ref
    ref = _reference(cli, ctx, d, titles, bams, shallow=True, **kw)
    assert _combine_bam(cli, d, titles, bams, "b48s", devices=[0], shallow=True, **kw) == ref
