"""Library strandedness from the BAM: the vote rule (tests/strand_oracle.py restates it), the host gene index, library_type's
thresholds, spl_infer_strand* on the GPU, and `inferStrandedness` / `processBam -s auto` / `combineBam -s auto`.

On the CPU the commands run with stand-in contexts whose votes come from the restatement (and whose extraction and counts come
from the oracles, as in test_combine_bam); `-s auto` must write exactly what the explicit flags of the verdict write."""
import ctypes as C
import os

import numpy as np
import pytest

import strand_oracle
from spliser_b200 import Records, api
from spliser_b200.api import GeneStrands, StrandVotes
from test_combine_bam import HostSample, ResidentOracleContext, memo_extract  # noqa: F401  (fixture)

AGREE, OPP, NONE = "agree", "opp", "none"


# ---------------------------------------------------------------------------------------------------------- fixtures
def _genes(chroms, rows):
    """GeneStrands over chroms from (chrom, left, right, strand char) rows; chromosomes may be left out at the end."""
    offs, left, right, strand = [0], [], [], []
    for c in chroms:
        mine = [r for r in rows if r[0] == c]
        left += [r[1] for r in mine]; right += [r[2] for r in mine]; strand += [ord(r[3]) for r in mine]
        offs.append(len(left))
    return GeneStrands(offs, left, right, strand)


CHROMS = ["C1", "C2", "C3"]
GENES = [("C1", 100, 200, "+"),                          # GFF 101..200
         ("C1", 300, 500, "-"), ("C1", 400, 600, "+"),   # both strands over 401..500
         ("C1", 700, 800, "."), ("C1", 750, 900, "+"),   # a '.' gene ignored
         ("C1", 1000, 1100, "+"), ("C1", 1500, 1600, "-"),
         ("C1", 2000, 1990, "-"),                        # end < start: an empty span
         ("C2", 10, 20, "+")]
# C3 has no entry in the view at all (a caller chromosome beyond the annotation)
GENE_VIEW = _genes(CHROMS[:2], GENES)

# (chrom, POS, FLAG, CIGAR, XS, vote from the genes, vote from XS); None = not a kept record
CRAFTED = [
    ("C1", 91, 0, "10M", "+", NONE, AGREE),              # ends at base left = 100: just before the gene
    ("C1", 92, 0, "10M", "-", AGREE, OPP),               # ends at base left + 1 = 101: the gene's first base
    ("C1", 200, 0, "10M", "?", AGREE, NONE),             # starts at base right = 200: its last base
    ("C1", 201, 0, "10M", "+", NONE, AGREE),             # starts at right + 1
    ("C1", 451, 0, "20M", "+", NONE, AGREE),             # genes of both strands
    ("C1", 301, 0, "20M", "-", OPP, OPP),                # '-' only: fr '+' read is opposite
    ("C1", 710, 0, "20M", "?", NONE, NONE),              # a '.' gene only
    ("C1", 760, 0, "20M", "+", AGREE, AGREE),            # '.' and '+': the '+' one counts
    ("C1", 1050, 0, "20M450N20M", "+", NONE, AGREE),     # the N reaches into the '-' gene
    ("C1", 1050, 0, "20M400N20M", "+", AGREE, AGREE),    # it stops short of it
    ("C1", 1050, 0, "5S20M40D3I", "+", AGREE, AGREE),
    ("C1", 150, 0, "10S", "-", AGREE, OPP),              # S only: L = 1
    ("C1", 150, 16, "5I", "-", OPP, AGREE),              # I only, reverse
    ("C1", 1985, 0, "30M", "-", NONE, OPP),              # over the empty gene
    ("C1", 150, 99, "10M", "+", AGREE, AGREE),           # first mate forward: fr '+'
    ("C1", 150, 147, "10M", "+", AGREE, AGREE),          # second mate reverse: fr '+'
    ("C1", 150, 83, "10M", "+", OPP, OPP),               # first mate reverse: fr '-'
    ("C1", 150, 163, "10M", "-", OPP, AGREE),            # second mate forward: fr '-'
    ("C1", 150, 16 | 1024, "10M", "?", OPP, NONE),       # single-end reverse, duplicate: no FLAG filter
    ("C1", 150, 4, "*", "+", None, None),                # no CIGAR operator
    ("C2", 5, 0, "10M", "+", AGREE, AGREE),              # overlaps C2's gene
    ("C2", 50, 0, "10M", "+", NONE, AGREE),              # C2 beyond its genes
    ("C3", 150, 0, "10M", "-", NONE, OPP),               # C3: no genes in the view
    ("CX", 150, 0, "10M", "+", None, None),              # not a caller chromosome
]


def _crafted_records():
    reads = sorted(CRAFTED, key=lambda r: ["C1", "C2", "C3", "CX"].index(r[0]))
    return reads, Records.from_reads(CHROMS, [r[:5] for r in reads])


def _tiny_bam(path):
    """The crafted records as a BAM with XS tags (CX a header reference too): far fewer than 100 votes."""
    reads, _ = _crafted_records()
    rec = Records.from_reads(CHROMS + ["CX"], [r[:5] for r in reads])
    rec.write_bam(path, CHROMS + ["CX"], aux=xs_aux(rec.xs))
    return path


def _expected(reads, col):
    v = [r[col] for r in reads]
    return StrandVotes(v.count(AGREE), v.count(OPP), v.count(NONE))


def flipped(rec, sel):
    """The records with the fr / rf read strand of `sel` turned over: mate bits swapped when paired, bit 16 flipped when single-end.
    POS does not change, so a sorted file stays sorted."""
    f = rec.flag.copy()
    paired = (f & 1) != 0
    sw = sel & paired
    m = f[sw]
    f[sw] = (m & ~np.uint16(192)) | ((m & 64) << 1) | ((m & 128) >> 1)
    f[sel & ~paired] ^= 16
    return Records(rec.pos, f, rec.cig_off, rec.cigar, rec.seg_chrom, rec.seg_off, xs=rec.xs)


def single_end(rec):
    """A paired library as single-end with the same fr read strands: second mates turned over, pairing bits cleared."""
    f = rec.flag.copy()
    f[(f & 128) != 0] ^= 16
    f &= ~np.uint16(1 | 2 | 8 | 32 | 64 | 128)
    return Records(rec.pos, f, rec.cig_off, rec.cigar, rec.seg_chrom, rec.seg_off, xs=rec.xs)


def xs_column(rec):
    """XS as an aligner writes it for a dUTP (rf) library: the transcript strand of every spliced record, '?' elsewhere."""
    off = rec.cig_off.astype(np.int64)
    spliced = np.zeros(len(rec), bool)
    spliced[np.searchsorted(off, np.flatnonzero((rec.cigar & 15) == 3), side="right") - 1] = True
    plus = ~strand_oracle.fr_plus(rec.flag)
    return np.where(spliced, np.where(plus, ord("+"), ord("-")), ord("?")).astype(np.uint8)


def xs_aux(xs):
    """One XS:A field for every record with a strand, nothing for the others."""
    has = xs != ord("?")
    off = np.zeros(len(xs) + 1, np.int64)
    off[1:] = np.cumsum(np.where(has, 4, 0))
    blob = np.zeros(int(off[-1]), np.uint8).reshape(-1, 4) if off[-1] else np.zeros((0, 4), np.uint8)
    blob[:, 0], blob[:, 1], blob[:, 2], blob[:, 3] = ord("X"), ord("S"), ord("A"), xs[has]
    return off, blob.reshape(-1)


def gff_of(w, path):
    """A gene around every junction of the workload, on the junction's (transcript's) strand."""
    j = w.junctions
    with open(path, "w") as fh:
        for i in range(len(j)):
            fh.write("%s\tsynthetic\tgene\t%d\t%d\t.\t%s\t.\tID=J%06d\n" % (w.chroms[int(j.chrom[i])], max(1, int(j.left[i]) - 150),
                                                                        int(j.right[i]) + 150, chr(int(j.strand[i])), i))


FORMS = ("rf", "fr", "unstranded")


def forms(rec, seed):
    """The library as generated (dUTP: rf), as fr, and unstranded (a seeded half of the records turned over)."""
    half = np.random.default_rng(seed).random(len(rec)) < 0.5
    return {"rf": rec, "fr": flipped(rec, np.ones(len(rec), bool)), "unstranded": flipped(rec, half)}


def _small(seed, n=20_000):
    """config_small paired and stranded (so the junctions carry the transcript strands), with its XS column."""
    from spliser_b200 import synth
    w = synth.generate(synth.config_small(n, seed=seed, stranded=True, paired=True))
    r = w.records
    return w, Records(r.pos, r.flag, r.cig_off, r.cigar, r.seg_chrom, r.seg_off, xs=xs_column(r))


# ---------------------------------------------------------------------------------------------------------- CPU: the rule
def test_restatement_on_crafted_records():
    reads, rec = _crafted_records()
    assert strand_oracle.votes(rec, len(CHROMS), GENE_VIEW) == _expected(reads, 5)
    assert strand_oracle.votes(rec, len(CHROMS), None) == _expected(reads, 6)


def test_library_type_thresholds():
    lt = api.library_type
    assert lt(StrandVotes(99, 0, 5)) is None and lt(StrandVotes(100, 0, 0)) == "fr"
    assert lt(StrandVotes(0, 99, 0)) is None and lt(StrandVotes(0, 100, 0)) == "rf"
    assert lt(StrandVotes(80, 20, 7)) == "fr" and lt(StrandVotes(79, 21, 0)) is None
    assert lt(StrandVotes(20, 80, 0)) == "rf" and lt(StrandVotes(21, 79, 0)) is None
    assert lt(StrandVotes(35, 65, 0)) == "unstranded" and lt(StrandVotes(34, 66, 0)) is None
    assert lt(StrandVotes(65, 35, 0)) == "unstranded" and lt(StrandVotes(66, 34, 0)) is None
    assert lt(StrandVotes(800, 200, 0)) == "fr" and lt(StrandVotes(7, 13, 10 ** 6)) is None


def _index_masks(genes, n_chrom, chrom, start, length):
    from spliser_b200 import _lib as L
    lib = L.load()
    chrom, start, length = (np.ascontiguousarray(a, dt) for a, dt in ((chrom, np.int32), (start, np.int64), (length, np.int64)))
    out = np.zeros(len(chrom), np.uint8)
    err = C.create_string_buffer(256)
    rc = lib.spl_debug_gene_strand_mask(n_chrom, C.byref(genes.view()), len(chrom), chrom.ctypes.data_as(L.c_i32p),
                                        start.ctypes.data_as(L.c_i64p), length.ctypes.data_as(L.c_i64p), out.ctypes.data_as(L.c_u8p), err, 256)
    assert rc == 0, err.value
    return out


def test_host_gene_index_equals_a_scan_of_every_gene(built_library):
    rng = np.random.default_rng(3)
    for trial in range(40):
        n_chrom = int(rng.integers(1, 5))
        rows = []
        for c in range(int(rng.integers(0, n_chrom + 1))):      # later chromosomes may be beyond the view
            G = int(rng.integers(0, 60 if trial % 4 else 3000))
            left = rng.integers(0, 20_000, G)
            length = np.where(rng.random(G) < 0.1, rng.integers(-5, 1, G), rng.integers(1, 3000 if trial % 3 else 19_000, G))
            st = rng.choice(list("+-.?"), G, p=[0.42, 0.42, 0.1, 0.06])
            rows += [("c%d" % c, int(a), int(a + b), s) for a, b, s in zip(left, length, st)]
        names = ["c%d" % c for c in range(n_chrom)]
        view_chroms = names[:len({r[0] for r in rows})] if rows else []
        genes = _genes(view_chroms, rows)
        Q = 2000
        chrom = rng.integers(0, n_chrom, Q)
        start = rng.integers(-100, 21_000, Q)
        length = np.where(rng.random(Q) < 0.2, 1, rng.integers(1, 5000, Q))
        got = _index_masks(genes, n_chrom, chrom, start, length)
        want = np.zeros(Q, np.uint8)
        for c in range(n_chrom):
            sel = np.flatnonzero(chrom == c)
            want[sel] = strand_oracle.gene_mask(genes, c, start[sel], length[sel])
        assert np.array_equal(got, want), trial


def test_gene_strands_of_an_annotation(tmp_path, built_library):
    from spliser_b200.genes import load_annotation
    gff = tmp_path / "g.gff"
    gff.write_text("A\tx\tgene\t11\t20\t.\t+\t.\tID=a1\nB\tx\tgene\t5\t9\t.\t.\t.\tID=b1\nA\tx\tgene\t3\t30\t.\t-\t.\tID=a2\n"
                   "A\tx\texon\t3\t30\t.\t-\t.\tID=e\nB\tx\tgene\t1\t2\t.\t+ \t.\tID=b2\n")
    g = api.gene_strands(load_annotation(str(gff)), ["B", "Z", "A", "A"])
    assert g.chrom_off.tolist() == [0, 2, 2, 4, 4]            # a repeated name: the genes go to its first index
    assert g.left.tolist() == [0, 4, 2, 10] and g.right.tolist() == [2, 9, 30, 20]      # each chromosome's genes by left
    assert g.strand.tolist() == [0, 0, ord("-"), ord("+")]      # '+ ' and '.' are not exactly '+' or '-'


# ---------------------------------------------------------------------------------------------------------- CPU: the commands
class VotingSample(HostSample):
    def infer_strand(self, chrom_names, genes=None):
        assert not self.closed
        if genes is None:
            assert self.rec.xs is not None, "the XS source needs a sample loaded with xs=True"
        self.owner.sample_votes.append(self.path)
        return strand_oracle.votes(self._records(chrom_names), len(chrom_names), genes)


class VotingContext(ResidentOracleContext):
    """ResidentOracleContext whose votes come from the restatement."""

    def __init__(self, refuse=()):
        super().__init__(refuse)
        self.sample_votes, self.path_votes = [], []

    def load_bam(self, bam_path, xs=False):
        if os.path.basename(bam_path) in self.refuse:
            raise api.SampleMemoryError("stand-in: %s does not fit" % bam_path)
        s = VotingSample(self, bam_path, xs)
        self.samples.append(s)
        return s

    def infer_strand_bam(self, bam_path, chrom_names, genes=None):
        self.path_votes.append(bam_path)
        return strand_oracle.votes(Records.from_bam(bam_path, chrom_names, xs=genes is None), len(chrom_names), genes)


@pytest.fixture(scope="module")
def small_bams(tmp_path_factory, built_library):
    """The three forms of one small rf library as BAMs with XS tags, and a GFF of its junctions."""
    d = tmp_path_factory.mktemp("forms")
    w, rec = _small(17)
    gff = str(d / "genes.gff")
    gff_of(w, gff)
    bams = {}
    for name, r in forms(rec, 17).items():
        bams[name] = str(d / ("%s.bam" % name))
        r.write_bam(bams[name], w.chroms, w.chrom_len, aux=xs_aux(r.xs))
    return w, bams, gff


def _tsv(path):
    with open(path) as fh:
        return fh.read()


@pytest.mark.parametrize("annotated", [False, True])
def test_process_bam_auto_writes_what_the_verdict_flags_write(tmp_path, small_bams, annotated):
    from spliser_b200 import cli
    w, bams, gff = small_bams
    ann = dict(annotationFile=gff) if annotated else {}
    for form, explicit in (("rf", dict(isStranded=True, strandedType="rf")), ("fr", dict(isStranded=True, strandedType="fr")),
                           ("unstranded", dict())):
        ref = str(tmp_path / ("ref_" + form))
        cli.processBam(bams[form], ref, ctx=ResidentOracleContext(), **explicit, **ann)
        for refuse in ((), (form + ".bam",)):
            c = VotingContext(refuse)
            out = str(tmp_path / ("auto_%s_%d" % (form, len(refuse))))
            cli.processBam(bams[form], out, isStranded=True, strandedType="auto", ctx=c, **ann)
            assert _tsv(out + ".SpliSER.tsv") == _tsv(ref + ".SpliSER.tsv"), (form, refuse)
            if refuse:                                     # does not fit: votes and count from the path, two ingests
                assert c.path_votes == [bams[form]] and c.path_extracts == [bams[form]] and not c.samples
            else:                                          # one load: votes and count from the resident sample
                assert c.sample_votes == [bams[form]] and not c.path_extracts and c.samples[0].closed
                assert (c.samples[0].rec.xs is not None) == (not annotated)


def test_process_bam_auto_with_a_gene_query_votes_over_every_gene(tmp_path, small_bams, capsys):
    from spliser_b200 import cli
    from spliser_b200.genes import load_annotation
    w, bams, gff = small_bams
    gene = load_annotation(gff).columns.name(0)
    ref, out = str(tmp_path / "ref"), str(tmp_path / "auto")
    cli.processBam(bams["rf"], ref, qGene=gene, maxIntronSize=5000, annotationFile=gff, isStranded=True, strandedType="rf",
                   ctx=ResidentOracleContext())
    capsys.readouterr()
    cli.processBam(bams["rf"], out, qGene=gene, maxIntronSize=5000, annotationFile=gff, isStranded=True, strandedType="auto",
                   ctx=VotingContext())
    assert _tsv(out + ".SpliSER.tsv") == _tsv(ref + ".SpliSER.tsv")
    text = capsys.readouterr().out
    want = strand_oracle.votes(Records.from_bam(bams["rf"], api.bam_reference_names(bams["rf"])), len(w.chroms),
                               api.gene_strands(load_annotation(gff), w.chroms))
    assert "agree with fr %d\topposite %d\tno vote %d" % (want.agree_fr, want.opposite, want.no_vote) in text
    assert want.agree_fr + want.opposite > 1000          # far more than the query gene's reads
    assert "Library type:\t\t\trf: --isStranded -s rf" in text


def test_undecided_runs_write_nothing(tmp_path, small_bams, built_library):
    from spliser_b200 import cli
    tiny = _tiny_bam(str(tmp_path / "tiny.bam"))
    w, bams, gff = small_bams
    out = str(tmp_path / "o")
    with pytest.raises(cli.StrandednessError, match="undecided"):
        cli.processBam(tiny, out, isStranded=True, strandedType="auto", ctx=VotingContext())
    # 70 / 30: between the thresholds
    r = Records.from_bam(bams["rf"], w.chroms, xs=True)
    mixed = flipped(r, np.random.default_rng(5).random(len(r)) < 0.3)
    mbam = str(tmp_path / "mixed.bam")
    mixed.write_bam(mbam, w.chroms, w.chrom_len, aux=xs_aux(mixed.xs))
    with pytest.raises(cli.StrandednessError, match="undecided"):
        cli.processBam(mbam, out, isStranded=True, strandedType="auto", ctx=VotingContext())
    sf = str(tmp_path / "s.tsv")
    with open(sf, "w") as fh:
        fh.write("a\t%s_a.SpliSER.tsv\t%s\nb\t%s_b.SpliSER.tsv\t%s\n" % (out, tiny, out, mbam))
    with pytest.raises(cli.StrandednessError, match="undecided"):
        cli.combineBam(sf, out, isStranded=True, strandedType="auto", context_factory=lambda d: VotingContext())
    assert not [f for f in os.listdir(str(tmp_path)) if f.startswith("o")]


def test_combine_bam_auto_pools_the_votes(tmp_path, small_bams, memo_extract):
    from spliser_b200 import cli
    from test_combine_bam import _combine_bam, _split
    w, bams, gff = small_bams
    d = str(tmp_path)
    parts = {}
    for form in ("rf", "fr"):
        w_form = type("W", (), {"records": Records.from_bam(bams[form], w.chroms)})()
        for k, s in enumerate(_split(w_form, 4, 9)):
            parts[form, k] = s
    titles = ["t%d" % k for k in range(4)]
    for form in ("rf", "fr"):
        paths = []
        for k in range(4):
            paths.append(os.path.join(d, "%s%d.bam" % (form, k)))
            parts[form, k].write_bam(paths[-1], w.chroms, w.chrom_len)
        ref = _combine_bam(cli, d, titles, paths, "ref" + form, annotation=gff, stranded=True, stype=form,
                           context_factory=lambda dev: ResidentOracleContext())
        made = []

        def factory(dev):
            made.append(VotingContext(("%s1.bam" % form,)))
            return made[-1]
        got = _combine_bam(cli, d, titles, paths, "auto" + form, annotation=gff, stranded=True, stype="auto", devices=[0, 1],
                           context_factory=factory)
        assert got == ref, form
        assert sum(len(c.sample_votes) for c in made) == 3 and sum(len(c.path_votes) for c in made) == 1
    # one sample of the other protocol among ten: the pooled votes say rf, the sample says fr -- refused, nothing written
    mix = []
    for k in range(10):
        form = "fr" if k == 1 else "rf"
        part = _split(type("W", (), {"records": Records.from_bam(bams[form], w.chroms)})(), 10, 4)[k]
        mix.append(os.path.join(d, "m%d.bam" % k))
        part.write_bam(mix[-1], w.chroms, w.chrom_len)
    with pytest.raises(cli.StrandednessError, match=r"pooled library type rf: t1 is fr \(agree with fr \d+, opposite \d+, no vote \d+\)$"):
        _combine_bam(cli, d, ["t%d" % k for k in range(10)], mix, "mix", annotation=gff, stranded=True, stype="auto",
                     context_factory=lambda dev: VotingContext())
    assert [f for f in os.listdir(d) if f.startswith("mix")] == ["mix_samples.tsv"]


def test_infer_strandedness_prints_the_verdict(tmp_path, small_bams, capsys, monkeypatch):
    from spliser_b200 import cli
    w, bams, gff = small_bams
    monkeypatch.setattr(api, "Context", lambda device=0: VotingContext())
    for form in FORMS:
        for ann in (None, gff):
            verdict, votes = cli.inferStrandedness(bams[form], annotationFile=ann)
            assert verdict == form
            text = capsys.readouterr().out
            assert "Thresholds:\t\t\tat least 100 votes; fr when f >= 0.8, rf when f <= 0.2, unstranded when 0.35 <= f <= 0.65" in text
            flags = {"rf": "rf: --isStranded -s rf", "fr": "fr: --isStranded -s fr", "unstranded": "unstranded: no --isStranded"}
            assert "Library type:\t\t\t" + flags[form] in text
            assert "f = agree / (agree + opposite):\t%.4f" % (votes.agree_fr / (votes.agree_fr + votes.opposite)) in text
    cli.main(["inferStrandedness", "-B", bams["rf"]])
    assert "Library type:\t\t\trf" in capsys.readouterr().out
    tiny = _tiny_bam(str(tmp_path / "tiny.bam"))
    with pytest.raises(SystemExit):
        cli.main(["inferStrandedness", "-B", tiny])
    assert "Library type:\t\t\tundecided" in capsys.readouterr().out


def test_command_line_passes_auto_on(monkeypatch, built_library):
    from spliser_b200 import cli
    seen = {}
    for name in ("processBam", "combineBam", "inferStrandedness"):
        monkeypatch.setattr(cli, name, lambda name=name, **kw: seen.update(kw, _cmd=name))
    cli.main(["processBam", "-B", "x.bam", "-o", "out", "--isStranded", "-s", "auto"])
    assert seen.pop("_cmd") == "processBam" and seen["isStranded"] and seen["strandedType"] == "auto"
    assert "strandFromXS" not in seen
    seen.clear()
    cli.main(["combineBam", "-S", "s.tsv", "-o", "out", "--isStranded", "-s", "auto"])
    assert seen.pop("_cmd") == "combineBam" and seen["strandedType"] == "auto" and seen["devices"] == [0]
    seen.clear()
    cli.main(["inferStrandedness", "-B", "x.bam", "-A", "g.gff"])
    assert seen == dict(_cmd="inferStrandedness", inBAM="x.bam", annotationFile="g.gff")
    with pytest.raises(SystemExit):
        cli.main(["inferStrandedness", "-A", "g.gff"])
    # process keeps check_strand's UnboundLocalError for a type that is neither fr nor rf
    with pytest.raises(UnboundLocalError):
        api.mode_flags(True, "auto")


def test_process_bam_auto_without_is_stranded_runs_unstranded(tmp_path, small_bams):
    from spliser_b200 import cli
    w, bams, gff = small_bams
    a, b = str(tmp_path / "a"), str(tmp_path / "b")
    cli.processBam(bams["rf"], a, strandedType="auto", ctx=ResidentOracleContext())
    cli.processBam(bams["rf"], b, ctx=ResidentOracleContext())
    assert _tsv(a + ".SpliSER.tsv") == _tsv(b + ".SpliSER.tsv")


# ---------------------------------------------------------------------------------------------------------- GPU
@pytest.mark.gpu
def test_device_votes_on_crafted_records(ctx):
    reads, rec = _crafted_records()
    assert ctx.infer_strand_records(rec, len(CHROMS), GENE_VIEW) == _expected(reads, 5)
    assert ctx.infer_strand_records(rec, len(CHROMS)) == _expected(reads, 6)
    assert ctx.stats()["ms_strand_votes"] > 0


def _bam_votes(ctx, monkeypatch, bam, chroms, genes):
    """spl_infer_strand through the device ingest and the host reader, and spl_sample_infer_strand: all must agree."""
    got = [ctx.infer_strand_bam(bam, chroms, genes)]
    assert ctx.stats()["bam_on_device"] == 1.0
    with ctx.load_bam(bam, xs=genes is None) as s:
        got.append(s.infer_strand(chroms, genes))
    monkeypatch.setenv("SPLISER_HOST_BAM", "1")
    got.append(ctx.infer_strand_bam(bam, chroms, genes))
    assert ctx.stats()["bam_on_device"] == 0.0
    monkeypatch.delenv("SPLISER_HOST_BAM")
    assert got[0] == got[1] == got[2], got
    return got[0]


@pytest.mark.gpu
@pytest.mark.parametrize("paired", [True, False])
def test_device_votes_on_synthetic_libraries(ctx, tmp_path, monkeypatch, paired):
    from spliser_b200.genes import load_annotation
    w, rec = _small(23, 120_000)
    if not paired:
        rec = single_end(rec)
    gff = str(tmp_path / "g.gff")
    gff_of(w, gff)
    genes = api.gene_strands(load_annotation(gff), w.chroms)
    for form, r in forms(rec, 29).items():
        for src in (genes, None):
            want = strand_oracle.votes(r, len(w.chroms), src)
            assert ctx.infer_strand_records(r, len(w.chroms), src) == want, (form, src is None)
            assert api.library_type(want) == form, (form, want)
            bam = str(tmp_path / ("%s.bam" % form))
            r.write_bam(bam, w.chroms, w.chrom_len, aux=xs_aux(r.xs))
            # the caller's list may reorder the header's names and add one the file lacks
            names = ["chrNOPE"] + list(reversed(w.chroms))
            g2 = api.gene_strands(load_annotation(gff), names) if src is not None else None
            assert _bam_votes(ctx, monkeypatch, bam, names, g2) == want, (form, src is None)


@pytest.mark.gpu
def test_device_votes_on_long_reads(ctx, tmp_path, monkeypatch):
    from spliser_b200 import synth
    w = synth.generate_long_reads(synth.config_long_reads())
    r = w.records
    rec = Records(r.pos, r.flag, r.cig_off, r.cigar, r.seg_chrom, r.seg_off, xs=xs_column(r))
    assert int(np.diff(rec.cig_off.astype(np.int64)).max()) > 100
    gff = str(tmp_path / "g.gff")
    gff_of(w, gff)
    from spliser_b200.genes import load_annotation
    genes = api.gene_strands(load_annotation(gff), w.chroms)
    bam = str(tmp_path / "long.bam")
    rec.write_bam(bam, w.chroms, w.chrom_len, aux=xs_aux(rec.xs))
    for src in (genes, None):
        want = strand_oracle.votes(rec, len(w.chroms), src)
        assert want.agree_fr + want.opposite > 1000
        assert ctx.infer_strand_records(rec, len(w.chroms), src) == want
        assert _bam_votes(ctx, monkeypatch, bam, w.chroms, src) == want


@pytest.mark.gpu
def test_sample_without_xs_refuses_the_xs_source(ctx, small_bams):
    w, bams, gff = small_bams
    with ctx.load_bam(bams["rf"]) as s:
        with pytest.raises(api.SpliserError, match="SPL_FLAG_XS_STRAND"):
            s.infer_strand(w.chroms)
        from spliser_b200.genes import load_annotation
        assert api.library_type(s.infer_strand(w.chroms, api.gene_strands(load_annotation(gff), w.chroms))) == "rf"


@pytest.mark.gpu
def test_cli_auto_on_gpu_equals_the_explicit_flags(ctx, tmp_path, monkeypatch):
    from spliser_b200 import cli
    from test_combine_bam import _combine_bam
    d = str(tmp_path)
    w, rec = _small(31, 120_000)
    gff = os.path.join(d, "g.gff")
    gff_of(w, gff)
    bams = {}
    for form, r in forms(rec, 31).items():
        bams[form] = os.path.join(d, form + ".bam")
        r.write_bam(bams[form], w.chroms, w.chrom_len, aux=xs_aux(r.xs))
    explicit = {"rf": dict(isStranded=True, strandedType="rf"), "fr": dict(isStranded=True, strandedType="fr"), "unstranded": {}}
    for form in FORMS:
        for ann in ({}, dict(annotationFile=gff)):
            ref, out = os.path.join(d, "ref"), os.path.join(d, "auto")
            cli.processBam(bams[form], ref, ctx=ctx, **explicit[form], **ann)
            cli.processBam(bams[form], out, isStranded=True, strandedType="auto", ctx=ctx, **ann)
            assert _tsv(out + ".SpliSER.tsv") == _tsv(ref + ".SpliSER.tsv"), (form, ann)
    # combineBam: three resident samples and one refused by the budget
    r = rec
    titles = ["t%d" % k for k in range(4)]
    from test_combine_bam import _split
    paths = []
    for k, s in enumerate(_split(type("W", (), {"records": r})(), 4, 3)):
        paths.append(os.path.join(d, "c%d.bam" % k))
        s.write_bam(paths[-1], w.chroms, w.chrom_len)
    with ctx.load_bam(paths[0]) as s:
        one = s.device_bytes
    ref = _combine_bam(cli, d, titles, paths, "cref", annotation=gff, stranded=True, stype="rf", devices=[0])
    monkeypatch.setenv("SPLISER_SAMPLE_BUDGET_MB", str(int(3.5 * one) >> 20))
    got = _combine_bam(cli, d, titles, paths, "cauto", annotation=gff, stranded=True, stype="auto", devices=[0])
    monkeypatch.delenv("SPLISER_SAMPLE_BUDGET_MB")
    assert got == ref
