"""The read filter at BAM ingest (include/spliser_b200.h, spl_read_filter): samtools view -q / -F / -f applied where a BAM
becomes records, on the device ingest and on the host reader.

Its defining property: a command run with the filter on x.bam gives byte for byte what the same command gives without a
filter on x.bam with the dropped records removed.  The smaller BAM is written here from the kept subset (spl_write_bam_mapq),
so no samtools is needed.  The CPU tests hold the host reader to a numpy restatement of the rule and run the commands with
stand-in contexts fed from that reader; the GPU tests run the commands on both ingest routes."""
import dataclasses
import os

import numpy as np
import pytest

from spliser_b200 import ReadFilter, Records, api
from test_strand_inference import VotingContext, gff_of, xs_aux, xs_column

MAPQS = np.array([0, 1, 3, 60, 255], np.uint8)
ODD_BITS = (0x4, 0x200, 0x800, 0x400)


# ---------------------------------------------------------------------------------------------------------- fixtures
def keeps(flag, mapq, f: ReadFilter):
    """The rule, restated: MAPQ >= q, no bit of F, every bit of f."""
    flag = flag.astype(np.uint32)
    return (mapq >= f.min_mapq) & ((flag & f.exclude_flags) == 0) & ((flag & f.require_flags) == f.require_flags)


def subset(rec: Records, mask):
    """The records of `mask`, segments and CIGAR offsets rebuilt (empty segments dropped)."""
    idx = np.flatnonzero(mask)
    off = rec.cig_off.astype(np.int64)
    n_op = (off[1:] - off[:-1])[idx]
    cig = np.concatenate([rec.cigar[off[i]:off[i + 1]] for i in idx]) if len(idx) else np.zeros(0, np.uint32)
    seg_of = np.searchsorted(rec.seg_off, np.arange(len(rec)), side="right") - 1
    counts = np.bincount(seg_of[idx], minlength=len(rec.seg_chrom))
    keep_seg = counts > 0
    seg_off = np.concatenate([[0], np.cumsum(counts[keep_seg])])
    return Records(rec.pos[idx], rec.flag[idx], np.concatenate([[0], np.cumsum(n_op)]), cig, rec.seg_chrom[keep_seg],
                   seg_off if keep_seg.any() else [0], xs=None if rec.xs is None else rec.xs[idx])


def _aux_subset(aux, idx):
    off, blob = aux
    parts = [blob[off[i]:off[i + 1]] for i in idx]
    new = np.zeros(len(idx) + 1, np.int64)
    new[1:] = np.cumsum([len(p) for p in parts])
    return new, (np.concatenate(parts) if parts else np.zeros(0, np.uint8))


def odd_library(seed, n=8000):
    """A small paired, stranded synth library with a realistic MAPQ / FLAG mix: frac_odd_flag raised, MAPQ from
    {0, 1, 3, 60, 255}, and some unmapped (0x4), QC-fail (0x200), supplementary (0x800) and duplicate (0x400) bits.  Its XS
    column is that of an rf aligner.  -> (workload, Records with xs, mapq)"""
    from spliser_b200 import synth
    cfg = dataclasses.replace(synth.config_small(n, seed=seed, stranded=True, paired=True), frac_odd_flag=0.15)
    w = synth.generate(cfg)
    r = w.records
    rng = np.random.default_rng(seed)
    flag = r.flag.copy()
    for bit in ODD_BITS:
        flag[rng.random(len(r)) < 0.06] |= bit
    rec = Records(r.pos, flag, r.cig_off, r.cigar, r.seg_chrom, r.seg_off)
    rec.xs = xs_column(rec)
    return w, rec, MAPQS[rng.integers(0, len(MAPQS), len(rec))]


def write_pair(d, name, w, rec, mapq, f: ReadFilter, xs=True):
    """x.bam and the same BAM with the records f drops removed -> (full path, pre-filtered path, kept mask)."""
    aux = xs_aux(rec.xs) if xs else None
    full = os.path.join(d, name + ".bam")
    rec.write_bam(full, w.chroms, w.chrom_len, aux=aux, mapq=mapq)
    m = keeps(rec.flag, mapq, f)
    pre = os.path.join(d, name + ".pre.bam")
    idx = np.flatnonzero(m)
    subset(rec, m).write_bam(pre, w.chroms, w.chrom_len, aux=_aux_subset(aux, idx) if xs else None, mapq=mapq[idx])
    return full, pre, m


SETTINGS = [ReadFilter(1), ReadFilter(255), ReadFilter(0, 0x904), ReadFilter(0, 0x4), ReadFilter(0, 0, 0x2),
            ReadFilter(10, 0x904), ReadFilter(3, 0x400, 0x40), ReadFilter(0, 0x2, 0x2)]
FILTER = ReadFilter(10, 0x904)                      # the usual samtools view -q 10 -F 0x904


@pytest.fixture(scope="module")
def odd(built_library):
    return odd_library(23)


def _same_records(a: Records, b: Records):
    for name in ("pos", "flag", "cig_off", "cigar", "seg_chrom", "seg_off"):
        assert np.array_equal(getattr(a, name), getattr(b, name)), name
    assert (a.xs is None) == (b.xs is None) and (a.xs is None or np.array_equal(a.xs, b.xs))


# ---------------------------------------------------------------------------------------------------------- CPU: the reader
def test_filtered_reader_equals_a_numpy_subset(tmp_path, odd):
    w, rec, mapq = odd
    bam = str(tmp_path / "x.bam")
    rec.write_bam(bam, w.chroms, w.chrom_len, aux=xs_aux(rec.xs), mapq=mapq)
    # every chromosome, and all but the last: records of an unknown reference are the keep rule's, never counted as dropped
    for chroms in (list(w.chroms), list(w.chroms)[:-1]):
        known = np.repeat(np.isin(rec.seg_chrom, np.arange(len(chroms))), np.diff(rec.seg_off))
        base = subset(rec, known)
        for f in SETTINGS:
            m = keeps(rec.flag, mapq, f)
            for xs in (False, True):
                got = api.read_bam(bam, chroms, xs=xs, read_filter=f)
                want = subset(rec, m & known)
                if not xs:
                    want.xs = None
                _same_records(got, want)
                assert got.filter_counts == (int((m & known).sum()), int((~m & known).sum())), f
        # no filter, and a filter that keeps everything, read every kept record
        _same_records(api.read_bam(bam, chroms, xs=True, read_filter=ReadFilter()), base)
        _same_records(Records.from_bam(bam, chroms, xs=True), base)
    assert not keeps(rec.flag, mapq, ReadFilter(0, 0x2, 0x2)).any()        # overlapping F and f keep nothing
    assert 0 < keeps(rec.flag, mapq, FILTER).mean() < 0.9


def test_mapq_writer_with_255_writes_the_plain_writers_bytes(tmp_path, odd):
    w, rec, _ = odd
    full = np.full(len(rec), 255, np.uint8)
    for with_seq in (False, True):
        for aux in (None, xs_aux(rec.xs)):
            a, b = str(tmp_path / "a.bam"), str(tmp_path / "b.bam")
            rec.write_bam(a, w.chroms, w.chrom_len, with_seq=with_seq, aux=aux)
            rec.write_bam(b, w.chroms, w.chrom_len, with_seq=with_seq, aux=aux, mapq=full)
            assert open(a, "rb").read() == open(b, "rb").read(), (with_seq, aux is None)


def test_read_filter_values_are_checked(tmp_path, odd):
    for bad in (dict(min_mapq=-1), dict(min_mapq=256), dict(exclude_flags=0x10000), dict(require_flags=-1)):
        with pytest.raises(ValueError):
            ReadFilter(**bad)
    assert ReadFilter().is_none and not ReadFilter(0, 0, 1).is_none
    from spliser_b200 import _lib as L
    import ctypes as C
    lib = L.load()
    w, rec, mapq = odd
    bam = str(tmp_path / "x.bam")
    rec.write_bam(bam, w.chroms, w.chrom_len, mapq=mapq)
    names = (C.c_char_p * len(w.chroms))(*[c.encode() for c in w.chroms])
    h, err = C.c_void_p(), C.create_string_buffer(256)
    for raw in ((256, 0, 0), (-1, 0, 0), (0, 0x10000, 0), (0, 0, 0x10000)):
        assert lib.spl_read_bam_filtered(bam.encode(), len(w.chroms), names, 0, C.byref(L.ReadFilterC(*raw)), 0, C.byref(h), err, 256) == -1
        assert b"read filter" in err.value


# ---------------------------------------------------------------------------------------------------------- CPU: arguments
COMMAND_ARGS = {
    "process": ["-B", "x.bam", "-b", "x.bed", "-o", "o"],
    "combine": ["-S", "s.tsv", "-o", "o"],
    "combineShallow": ["-S", "s.tsv", "-o", "o"],
    "junctions": ["-B", "x.bam", "-o", "x.bed"],
    "processBam": ["-B", "x.bam", "-o", "o"],
    "combineBam": ["-S", "s.tsv", "-o", "o"],
    "inferStrandedness": ["-B", "x.bam"],
}


def _parsed(monkeypatch, argv):
    from spliser_b200 import cli
    got = {}
    for name in COMMAND_ARGS:
        monkeypatch.setattr(cli, name, lambda _n=name, **kw: got.update(kw, command=_n))
    cli.main(argv)
    return got


@pytest.mark.parametrize("command", sorted(COMMAND_ARGS))
def test_every_command_takes_the_filter_options(monkeypatch, built_library, command):
    base = [command] + COMMAND_ARGS[command]
    got = _parsed(monkeypatch, base + ["--minMAPQ", "10", "--excludeFlags", "0x904", "--requireFlags", "2"])
    assert got["command"] == command and got["read_filter"] == ReadFilter(10, 0x904, 2)
    assert _parsed(monkeypatch, base + ["--excludeFlags", "2308"])["read_filter"] == ReadFilter(0, 0x904)
    assert "read_filter" not in _parsed(monkeypatch, base)                  # no filter: the commands see what they saw before
    assert "read_filter" not in _parsed(monkeypatch, base + ["--minMAPQ", "0", "--excludeFlags", "0"])


@pytest.mark.parametrize("bad", [["--minMAPQ", "256"], ["--minMAPQ", "-1"], ["--excludeFlags", "0x10000"],
                                 ["--requireFlags", "-4"], ["--excludeFlags", "0xZZ"], ["-q", "10"], ["-F", "4"]])
def test_bad_filter_options_are_parser_errors(monkeypatch, built_library, bad):
    with pytest.raises(SystemExit) as e:
        _parsed(monkeypatch, ["processBam", "-B", "x.bam", "-o", "o"] + bad)
    assert e.value.code == 2


# ---------------------------------------------------------------------------------------------------------- CPU: the commands
class FilteringContext(VotingContext):
    """VotingContext (restatements behind every call) whose reads go through spl_read_bam_filtered under the filter set on it,
    as a context's host-reader fallback does."""

    active = [None, (0, 0)]                         # the filter of the context in use, and its last counts (one thread)

    def set_read_filter(self, f):
        self.rf = None if f.is_none else f
        FilteringContext.active[0] = self.rf

    def last_read_filter(self):
        return FilteringContext.active[1]


@pytest.fixture
def filtered_reads(monkeypatch):
    """Records.from_bam under the active stand-in's filter."""
    plain = Records.from_bam.__func__

    def from_bam(cls, path, chrom_names, threads=0, xs=False, read_filter=None):
        f = read_filter or FilteringContext.active[0]
        r = plain(cls, path, chrom_names, threads, xs, f)
        if f is not None:
            FilteringContext.active[1] = r.filter_counts
        return r
    monkeypatch.setattr(Records, "from_bam", classmethod(from_bam))
    FilteringContext.active[:] = [None, (0, 0)]
    yield
    FilteringContext.active[:] = [None, (0, 0)]


@pytest.fixture(scope="module")
def odd_bams(tmp_path_factory, built_library):
    """Three samples (full BAM, pre-filtered BAM) under FILTER, and a GFF of their genes."""
    d = str(tmp_path_factory.mktemp("odd"))
    out, first = [], None
    for i, seed in enumerate((31, 32, 33)):
        w, rec, mapq = odd_library(seed, 6000)
        full, pre, m = write_pair(d, "s%d" % i, w, rec, mapq, FILTER)
        out.append((full, pre, int(m.sum())))
        first = first or w
    gff = os.path.join(d, "genes.gff")
    gff_of(first, gff)                              # the genes of sample 0, which the single-sample tests read
    return d, out, gff


def _text(path):
    return open(path).read()


def test_process_bam_and_infer_strandedness_with_stand_ins(tmp_path, odd_bams, filtered_reads, capsys):
    from spliser_b200 import cli
    _, bams, gff = odd_bams
    full, pre, n_kept = bams[0]
    for kw in (dict(), dict(isStranded=True, strandedType="rf"), dict(annotationFile=gff), dict(isStranded=True, strandedType="auto")):
        cli.processBam(full, str(tmp_path / "f"), ctx=FilteringContext(), read_filter=FILTER, **kw)
        out = capsys.readouterr().out
        assert "Read filter %s:\tkept %d\tdropped " % (full, n_kept) in out
        cli.processBam(pre, str(tmp_path / "p"), ctx=VotingContext(), **kw)
        assert "Read filter" not in capsys.readouterr().out
        assert _text(tmp_path / "f.SpliSER.tsv") == _text(tmp_path / "p.SpliSER.tsv"), kw
    for g in (None, gff):
        a = cli.inferStrandedness(full, g, ctx=FilteringContext(), read_filter=FILTER)
        b = cli.inferStrandedness(pre, g, ctx=VotingContext())
        assert a == b


@pytest.mark.parametrize("refuse", [(), ("s1.bam",)])
def test_combine_bam_with_stand_ins(tmp_path, odd_bams, filtered_reads, refuse, capsys):
    from spliser_b200 import cli
    _, bams, gff = odd_bams
    d = str(tmp_path)
    texts = {}
    for tag, col in (("f", 0), ("p", 1)):
        sf = os.path.join(d, tag + ".txt")
        with open(sf, "w") as fh:
            fh.writelines("T%d\t%s\t%s\n" % (i, os.path.join(d, "%s%d.SpliSER.tsv" % (tag, i)), b[col]) for i, b in enumerate(bams))
        for mode, kw in (("plain", dict(isStranded=True, strandedType="rf")), ("auto", dict(isStranded=True, strandedType="auto")),
                         ("shallow", dict(shallow=True, minReads=2, annotationFile=gff))):
            rf = dict(read_filter=FILTER) if tag == "f" else {}
            ref = tuple(os.path.basename(bams[1][col]) for _ in refuse)
            cli.combineBam(sf, os.path.join(d, tag + mode), context_factory=lambda dev: (FilteringContext if rf else VotingContext)(ref),
                           **kw, **rf)
            out = capsys.readouterr().out
            if rf:
                for full, _, n_kept in bams:
                    assert out.count("Read filter %s:\tkept %d\t" % (full, n_kept)) == 1, (mode, out)
            texts[tag, mode] = [_text(os.path.join(d, "%s%d.SpliSER.tsv" % (tag, i))) for i in range(3)] + \
                [_text(os.path.join(d, tag + mode + ".combined.tsv"))]
    for mode in ("plain", "auto", "shallow"):
        assert texts["f", mode] == texts["p", mode], mode


def test_combine_with_stand_ins(tmp_path, odd_bams, filtered_reads):
    from spliser_b200 import cli
    _, bams, _ = odd_bams
    d = str(tmp_path)
    tsvs = []
    for i, (_, pre, _) in enumerate(bams):                 # the sample tables of the pre-filtered BAMs, for both runs
        cli.processBam(pre, os.path.join(d, "t%d" % i), ctx=VotingContext(), isStranded=True, strandedType="rf")
        tsvs.append(os.path.join(d, "t%d.SpliSER.tsv" % i))
    got = {}
    for tag, col in (("f", 0), ("p", 1)):
        sf = os.path.join(d, tag + ".txt")
        with open(sf, "w") as fh:
            fh.writelines("T%d\t%s\t%s\n" % (i, t, b[col]) for i, (t, b) in enumerate(zip(tsvs, bams)))
        rf = dict(read_filter=FILTER) if tag == "f" else {}
        cli.combine(sf, os.path.join(d, tag), isStranded=True, strandedType="rf", ctx=FilteringContext() if rf else VotingContext(), **rf)
        cli.combineShallow(sf, os.path.join(d, tag + "s"), isStranded=True, strandedType="rf", minReads=2,
                           ctx=FilteringContext() if rf else VotingContext(), **rf)
        got[tag] = (_text(os.path.join(d, tag + ".combined.tsv")), _text(os.path.join(d, tag + "s.combined.tsv")))
    assert got["f"] == got["p"]


# ---------------------------------------------------------------------------------------------------------- GPU
ROUTES = ("device", "host")


@pytest.fixture
def route(request, monkeypatch):
    if request.param == "host":
        monkeypatch.setenv("SPLISER_HOST_BAM", "1")
    else:
        monkeypatch.delenv("SPLISER_HOST_BAM", raising=False)
    return request.param


@pytest.fixture(scope="module")
def gpu_bams(tmp_path_factory, built_library):
    """Three larger samples under FILTER: (dir, [(full, pre, kept)], gff, (workload, Records, mapq) of sample 0)."""
    d = str(tmp_path_factory.mktemp("gpu_odd"))
    out, first = [], None
    for i, seed in enumerate((41, 42, 43)):
        w, rec, mapq = odd_library(seed, 30_000)
        full, pre, m = write_pair(d, "g%d" % i, w, rec, mapq, FILTER)
        out.append((full, pre, int(m.sum())))
        first = first or (w, rec, mapq)
    gff = os.path.join(d, "genes.gff")
    gff_of(first[0], gff)
    return d, out, gff, first


@pytest.mark.gpu
@pytest.mark.parametrize("route", ROUTES, indirect=True)
def test_single_bam_commands_on_gpu(tmp_path, gpu_bams, route, capsys):
    from spliser_b200 import cli
    _, bams, gff, _ = gpu_bams
    full, pre, n_kept = bams[0]
    d = str(tmp_path)
    for xs in (False, True):
        cli.junctions(full, os.path.join(d, "f.bed"), strandFromXS=xs, read_filter=FILTER)
        assert "Read filter %s:\tkept %d\tdropped " % (full, n_kept) in capsys.readouterr().out
        cli.junctions(pre, os.path.join(d, "p.bed"), strandFromXS=xs)
        assert "Read filter" not in capsys.readouterr().out
        assert _text(os.path.join(d, "f.bed")) == _text(os.path.join(d, "p.bed")), xs
    bed = os.path.join(d, "p.bed")
    for kw in (dict(), dict(isStranded=True, strandedType="rf", annotationFile=gff)):
        cli.process(full, bed, os.path.join(d, "f"), read_filter=FILTER, **kw)
        cli.process(pre, bed, os.path.join(d, "p"), **kw)
        assert _text(os.path.join(d, "f.SpliSER.tsv")) == _text(os.path.join(d, "p.SpliSER.tsv")), kw
    for kw in (dict(), dict(strandFromXS=True), dict(isStranded=True, strandedType="auto"),
               dict(isStranded=True, strandedType="auto", annotationFile=gff)):
        cli.processBam(full, os.path.join(d, "f"), read_filter=FILTER, **kw)
        cli.processBam(pre, os.path.join(d, "p"), **kw)
        assert _text(os.path.join(d, "f.SpliSER.tsv")) == _text(os.path.join(d, "p.SpliSER.tsv")), kw
    for g in (None, gff):
        assert cli.inferStrandedness(full, g, read_filter=FILTER) == cli.inferStrandedness(pre, g)


@pytest.mark.gpu
@pytest.mark.parametrize("route", ROUTES, indirect=True)
@pytest.mark.parametrize("budget", [None, "0"])
def test_multi_sample_commands_on_gpu(tmp_path, gpu_bams, route, budget, monkeypatch):
    from spliser_b200 import cli
    if budget is not None:
        monkeypatch.setenv("SPLISER_SAMPLE_BUDGET_MB", budget)     # every combineBam sample takes the path route
    _, bams, gff, _ = gpu_bams
    d = str(tmp_path)
    got = {}
    for tag, col in (("p", 1), ("f", 0)):                  # "p" first: its combineBam writes the tables both combine runs read
        rf = dict(read_filter=FILTER) if tag == "f" else {}
        sf = os.path.join(d, tag + ".txt")
        with open(sf, "w") as fh:
            fh.writelines("T%d\t%s\t%s\n" % (i, os.path.join(d, "%s%d.SpliSER.tsv" % (tag, i)), b[col]) for i, b in enumerate(bams))
        res = []
        for kw in (dict(isStranded=True, strandedType="rf"), dict(isStranded=True, strandedType="auto", strandFromXS=True),
                   dict(shallow=True, minReads=2, annotationFile=gff)):
            cli.combineBam(sf, os.path.join(d, tag + "cb"), **kw, **rf)
            res.append([_text(os.path.join(d, "%s%d.SpliSER.tsv" % (tag, i))) for i in range(3)] + [_text(os.path.join(d, tag + "cb.combined.tsv"))])
        # combine / combineShallow: the same (pre-filtered) sample tables, the re-count from the full or pre-filtered BAMs
        sf2 = os.path.join(d, tag + "2.txt")
        with open(sf2, "w") as fh:
            fh.writelines("T%d\t%s\t%s\n" % (i, os.path.join(d, "p%d.SpliSER.tsv" % i), b[col]) for i, b in enumerate(bams))
        cli.combine(sf2, os.path.join(d, tag + "c"), isStranded=True, strandedType="rf", **rf)
        cli.combineShallow(sf2, os.path.join(d, tag + "s"), isStranded=True, strandedType="rf", minReads=2, **rf)
        res.append([_text(os.path.join(d, tag + "c.combined.tsv")), _text(os.path.join(d, tag + "s.combined.tsv"))])
        got[tag] = res
    for a, b in zip(got["f"], got["p"]):
        assert a == b


@pytest.mark.gpu
def test_counts_and_routes_agree_on_gpu(gpu_bams, monkeypatch):
    _, bams, _, (w, rec, mapq) = gpu_bams
    full = bams[0][0]
    chroms = list(w.chroms)
    with api.Context(0) as c:
        for f in SETTINGS:
            m = keeps(rec.flag, mapq, f)
            want = (int(m.sum()), int((~m).sum()))
            c.set_read_filter(f)
            seen = []
            for host in ("0", "1"):
                monkeypatch.setenv("SPLISER_HOST_BAM", host)
                j, t = c.process_bam_extract(full, chroms, api.FLAG_XS_STRAND | 1 | 2)
                assert c.stats()["bam_on_device"] == (1.0 if host == "0" else 0.0)
                assert c.last_read_filter() == want, (f, host)
                v = c.infer_strand_bam(full, chroms)
                assert c.last_read_filter() == want
                with c.load_bam(full, xs=True) as s:
                    assert s.n_records == want[0] and c.last_read_filter() == want
                    sj, st = s.process_extract(chroms, api.FLAG_XS_STRAND | 1 | 2)
                    sv = s.infer_strand(chroms)
                seen.append((j, t, v, sj, st, sv))
            # the device ingest and the host reader give the same records: every result computed from them is the same
            for got in seen[1:] + [seen[0][3:] * 2]:
                for a, b in zip(seen[0], got):
                    if isinstance(a, api.Junctions):
                        assert all(np.array_equal(getattr(a, k), getattr(b, k)) for k in ("chrom", "left", "right", "score", "strand"))
                    elif isinstance(a, api.SiteTable):
                        assert all(np.array_equal(getattr(a, k), getattr(b, k)) for k in ("pos", "alpha", "beta1", "beta2simple", "beta2cryptic"))
                    else:
                        assert a == b
        c.set_read_filter()
        c.extract_junctions_bam(full, chroms)
        assert c.last_read_filter() == (len(rec), 0)


@pytest.mark.gpu
def test_filter_mismatches_are_refused_on_gpu(gpu_bams):
    _, bams, _, (w, rec, mapq) = gpu_bams
    full = bams[0][0]
    chroms = list(w.chroms)
    small = Records.from_bam(full, chroms)
    j = api.Junctions([0], [1000], [2000], [1], [ord("+")])
    with api.Context(0) as c:
        c.set_read_filter(FILTER)
        s = c.load_bam(full)
        assert s.read_filter == FILTER
        want = s.process_extract(chroms)[1].alpha
        gaps = [(0, 1000, "+", [2000], [])]
        for other in (ReadFilter(11, 0x904), None):
            c.set_read_filter(other or ReadFilter())
            for call in (lambda: s.process_extract(chroms), lambda: s.recount(chroms, gaps, 8), lambda: s.infer_strand(chroms, None)):
                with pytest.raises(api.SpliserError, match="read filter"):
                    call()
        c.set_read_filter(FILTER)
        assert np.array_equal(s.process_extract(chroms)[1].alpha, want)
        s.recount(chroms, gaps, 8)
        s.close()
        calls = (lambda: c.process_records(small, len(chroms), j, 0),
                 lambda: c.process_packed(api.PackedRecords.from_records(small), len(chroms), j, 0),
                 lambda: c.process_compact(api.CompactRecords.from_records(small), len(chroms), j, 0),
                 lambda: c.recount_records(small, len(chroms), gaps, 8),
                 lambda: c.extract_junctions_records(small, len(chroms)),
                 lambda: c.infer_strand_records(Records(small.pos, small.flag, small.cig_off, small.cigar, small.seg_chrom, small.seg_off,
                                                        xs=np.full(len(small), ord("+"), np.uint8)), len(chroms)),
                 lambda: c.resident_load(small, len(chroms), j, 0))
        for call in calls:
            with pytest.raises(api.SpliserError, match="no MAPQ"):
                call()
        c.set_read_filter()
        for call in calls:
            call()
