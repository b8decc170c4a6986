"""Several samples in one BAM told apart by an aux tag: the tag group table (include/spliser_b200.h, spl_tag_groups), the split of
one ingest into resident group samples (Context.load_bam_groups) and `combineGroups`.

The defining property: group g's sample holds exactly the kept records whose value maps to g, in BAM order, and every call on it
answers as the same call on a sample loaded from a BAM of just those records.  The CPU tests hold the host reader's group column
to a Python restatement of the value rule and run `combineGroups` with stand-in contexts against `combineBam` over one BAM per
group; the GPU tests hold the split's samples to load_bam of the group BAMs, on the device ingest and on the host reader."""
import os
import struct

import numpy as np
import pytest

from spliser_b200 import ReadFilter, Records, api
from test_read_filter import FILTER, _aux_subset, keeps, odd_library, subset
from test_strand_inference import VotingContext, VotingSample, gff_of
from xs_oracle import encode_aux

BARCODES = ["AAACCTGAGC-1", "AAACCTGCAT-1", "AAAGATGGTC-1", "AACTCAGTCC-1", "AAGGAGCGTA-1", "ACACCGGCAC-1", "ACGATACGTT-1",
            "AGCTCTCCAT-1"]
CLUSTERS = {b: "c%d" % (i % 3) for i, b in enumerate(BARCODES[:6])}        # the last two barcodes are in no cluster


# ---------------------------------------------------------------------------------------------------------- the rule, restated
_SIZE = {"A": 1, "c": 1, "C": 1, "s": 2, "S": 2, "i": 4, "I": 4, "f": 4}
_INT = {"c": "<b", "C": "<B", "s": "<h", "S": "<H", "i": "<i", "I": "<I"}


def field_end(b, p):
    """aux_field_end, restated: the end of the field at p, or None when it is malformed."""
    if len(b) - p < 3:
        return None
    ty, q = chr(b[p + 2]), p + 3
    if ty in _SIZE:
        e = q + _SIZE[ty]
    elif ty in "ZH":
        k = b.find(b"\0", q)
        if k < 0:
            return None
        e = k + 1
    elif ty == "B":
        if len(b) - q < 5:
            return None
        cnt = struct.unpack_from("<I", b, q + 1)[0]
        es = 1 if chr(b[q]) in "cC" else 2 if chr(b[q]) in "sS" else 4
        e = q + 5 + cnt * es
    else:
        return None
    return e if e <= len(b) else None


def tag_value(b, tag):
    """The value of the first field with `tag` (bytes), or None: no field, a type without a value, a malformed field before it."""
    p = 0
    while len(b) - p >= 3:
        e = field_end(b, p)
        if e is None:
            return None
        if b[p:p + 2] == tag:
            ty = chr(b[p + 2])
            if ty == "Z":
                return bytes(b[p + 3:e - 1])
            if ty == "A":
                return bytes(b[p + 3:p + 4])
            if ty in _INT:
                return str(struct.unpack_from(_INT[ty], b, p + 3)[0]).encode()
            return None
        p = e
    return None


def restated_groups(aux, table: api.TagGroups):
    """The group of every record: a group, -1 no value, -2 value in no group."""
    off, blob = aux
    raw = blob.tobytes()
    lut = dict(zip(table.values, table.groups.tolist()))
    out = np.empty(len(off) - 1, np.int32)
    for i in range(len(out)):
        v = tag_value(raw[off[i]:off[i + 1]], table.tag)
        out[i] = -1 if v is None else lut.get(v, -2)
    return out


# ---------------------------------------------------------------------------------------------------------- fixtures
def aux_blocks(rec, seed):
    """Aux fields for every record: STAR-like fields around CB:Z, RG:Z and HP in several integer types, and the odd cases --
    no CB, a barcode in no cluster, a repeated CB (the first one counts), CB after a malformed field, CB as f and B."""
    rng = np.random.default_rng(seed)
    parts = []
    for i in range(len(rec)):
        xs = chr(rec.xs[i])
        bc = BARCODES[rng.integers(0, len(BARCODES))]
        hp_ty = "iCsc"[rng.integers(0, 4)]
        hp = int(rng.integers(1, 3))
        fields = [("NH", "i", 1), ("HI", "C", 1), ("AS", "i", int(rng.integers(50, 150))), ("nM", "C", 0)]
        if xs in "+-":
            fields.append(("XS", "A", xs))
        kind = rng.random()
        if kind < 0.06:
            pass                                                    # no CB
        elif kind < 0.10:
            fields += [("CB", "Z", bc), ("CB", "Z", BARCODES[-1])]  # the first one counts
        elif kind < 0.12:
            fields.append(("CB", "f", 1.5))
        elif kind < 0.14:
            fields.append(("CB", "B", ("c", [1, 2, 3])))
        else:
            fields.append(("CB", "Z", bc))
        fields += [("UB", "Z", "ACGTACGTAC"), ("RG", "Z", "lib%d" % rng.integers(1, 4))]
        if hp_ty == "c" and rng.random() < 0.2:
            hp = -3
        if rng.random() < 0.9:
            fields.append(("HP", hp_ty, hp))
        b = encode_aux(fields)
        if rng.random() < 0.03:                                     # a malformed field before a CB: no value
            b += b"ZZQ" + encode_aux([("CB", "Z", bc)])
        parts.append(b)
    off = np.zeros(len(parts) + 1, np.int64)
    off[1:] = np.cumsum([len(p) for p in parts])
    return off, np.frombuffer(b"".join(parts), np.uint8).copy()


def tables():
    titles = []
    for b in BARCODES[:6]:
        if CLUSTERS[b] not in titles:
            titles.append(CLUSTERS[b])
    cb = api.TagGroups("CB", BARCODES[:6] + ["TTTTTTTTTT-1"], [titles.index(CLUSTERS[b]) for b in BARCODES[:6]] + [len(titles)],
                       len(titles) + 1)                        # + a group whose one value no record has
    rg = api.TagGroups("RG", ["lib1", "lib2"], [1, 0], 2)                                                      # lib3: in no group
    hp = api.TagGroups("HP", ["1", "2", "-3"], [0, 1, 1], 2)
    return {"CB": cb, "RG": rg, "HP": hp}


def write_groups(d, name, w, rec, aux, mapq, table):
    """The BAM and one BAM per group of `table` (the records the rule puts there, with their aux and MAPQ)."""
    full = os.path.join(d, name + ".bam")
    rec.write_bam(full, w.chroms, w.chrom_len, aux=aux, mapq=mapq)
    grp = restated_groups(aux, table)
    per = []
    for g in range(table.n_groups):
        idx = np.flatnonzero(grp == g)
        p = os.path.join(d, "%s.g%d.bam" % (name, g))
        subset(rec, grp == g).write_bam(p, w.chroms, w.chrom_len, aux=_aux_subset(aux, idx), mapq=mapq[idx])
        per.append(p)
    return full, per, grp


@pytest.fixture(scope="module")
def lib(built_library):
    w, rec, mapq = odd_library(51, 6000)
    return w, rec, mapq, aux_blocks(rec, 51)


def _same_records(a: Records, b: Records):
    for name in ("pos", "flag", "cig_off", "cigar", "seg_chrom", "seg_off"):
        assert np.array_equal(getattr(a, name), getattr(b, name)), name


# ---------------------------------------------------------------------------------------------------------- CPU: the reader
def test_reader_groups_equal_the_restated_rule(tmp_path, lib):
    w, rec, mapq, aux = lib
    bam = str(tmp_path / "x.bam")
    rec.write_bam(bam, w.chroms, w.chrom_len, aux=aux, mapq=mapq)
    for name, table in tables().items():
        want = restated_groups(aux, table)
        for f in (None, FILTER):
            m = np.ones(len(rec), bool) if f is None else keeps(rec.flag, mapq, f)
            got = api.read_bam(bam, list(w.chroms), xs=True, read_filter=f, groups=table)
            _same_records(got, subset(rec, m))
            assert np.array_equal(got.group, want[m]), (name, f)
            assert np.array_equal(got.xs, rec.xs[m])
        classes = np.bincount(want + 2, minlength=table.n_groups + 2)
        assert classes.sum() == len(rec) and (classes[2:] > 0).sum() >= 2, name
    cb = restated_groups(aux, tables()["CB"])
    assert (cb == -1).sum() > 0 and (cb == -2).sum() > 0 and not (cb == 3).any()       # no value, no group, the empty group


CRAFTED_TABLE = (["1", "-3", "X", "4294967295", "-32768"], [0, 1, 2, 3, 1], 4)
# (aux fields, value, group under CRAFTED_TABLE): every type, the extremes of the integer types, repeats in both orders
CRAFTED = [([("HP", "i", 1)], b"1", 0), ([("HP", "C", 1)], b"1", 0), ([("HP", "s", 1)], b"1", 0), ([("HP", "S", 1)], b"1", 0),
           ([("HP", "I", 1)], b"1", 0), ([("HP", "c", -3)], b"-3", 1), ([("HP", "s", -32768)], b"-32768", 1),
           ([("HP", "i", -3)], b"-3", 1), ([("HP", "I", 4294967295)], b"4294967295", 3), ([("HP", "i", -2147483648)], b"-2147483648", -2),
           ([("HP", "A", "X")], b"X", 2), ([("HP", "Z", "X")], b"X", 2), ([("HP", "Z", "1")], b"1", 0), ([("HP", "Z", "")], b"", -2),
           ([("HP", "f", 1.0)], None, -1), ([("HP", "H", "1A")], None, -1), ([("HP", "B", ("i", [1]))], None, -1),
           ([("XS", "A", "+")], None, -1), ([], None, -1), ([("HP", "i", 1), ("HP", "i", 2)], b"1", 0),
           ([("HP", "i", 2), ("HP", "i", 1)], b"2", -2), ([("HP", "c", -3), ("HP", "A", "X")], b"-3", 1),
           ([("HP", "A", "X"), ("HP", "c", -3)], b"X", 2), ([("NH", "i", 1), ("HP", "C", 255)], b"255", -2),
           ([("RG", "Z", "a"), ("XS", "A", "-"), ("HP", "S", 65535)], b"65535", -2)]
CRAFTED_RAW = [(b"NHQ" + encode_aux([("HP", "i", 1)]), None, -1),                        # a malformed field before the tag
               (encode_aux([("HP", "c", -3)]) + b"ZZQ", b"-3", 1),                       # ... after it: the tag already decided
               (encode_aux([("HP", "i", 1)])[:-1], None, -1)]                            # a value cut short by the record's end


def crafted_bam(path):
    """One record per crafted aux block, POS 100, 200, ... on chr1 -> (aux blocks, expected groups)."""
    blocks = [encode_aux(f) for f, _, _ in CRAFTED] + [b for b, _, _ in CRAFTED_RAW]
    want = np.array([g for _, _, g in CRAFTED] + [g for _, _, g in CRAFTED_RAW], np.int32)
    n = len(blocks)
    rec = Records(100 * np.arange(1, n + 1), np.zeros(n, np.uint16), np.arange(n + 1), np.full(n, 50 << 4, np.uint32), [0], [0, n])
    off = np.r_[0, np.cumsum([len(b) for b in blocks])].astype(np.int64)
    rec.write_bam(path, ["chr1"], [1_000_000], aux=(off, np.frombuffer(b"".join(blocks), np.uint8)))
    return rec, blocks, want


def test_the_rule_on_crafted_fields(tmp_path, built_library):
    """The restatement against hand-written answers, then the library's host reader against both on a BAM of those fields."""
    t = api.TagGroups("HP", *CRAFTED_TABLE)
    for fields, value, _ in CRAFTED:
        assert tag_value(encode_aux(fields), t.tag) == value, fields
    for raw, value, _ in CRAFTED_RAW:
        assert tag_value(raw, t.tag) == value, raw
    rec, blocks, want = crafted_bam(str(tmp_path / "c.bam"))
    lut = dict(zip(t.values, t.groups.tolist()))
    assert [(-1 if tag_value(b, t.tag) is None else lut.get(tag_value(b, t.tag), -2)) for b in blocks] == want.tolist()
    got = api.read_bam(str(tmp_path / "c.bam"), ["chr1"], groups=t)
    _same_records(got, rec)
    assert got.group.tolist() == want.tolist()


def test_tables_that_break_the_rule_are_refused(tmp_path, lib):
    w, rec, mapq, aux = lib
    bam = str(tmp_path / "x.bam")
    rec.write_bam(bam, w.chroms, w.chrom_len, aux=aux, mapq=mapq)
    bad = [api.TagGroups("1B", ["a"], [0], 1), api.TagGroups("C_", ["a"], [0], 1), api.TagGroups("CB", ["a"], [0], 0),
           api.TagGroups("CB", ["a"], [0], 65536), api.TagGroups("CB", ["a", "b", "a"], [0, 1, 0], 2),
           api.TagGroups("CB", ["a"], [1], 1), api.TagGroups("CB", ["a"], [-1], 1), api.TagGroups("CB", [""], [0], 1),
           api.TagGroups("CB", ["a\tb"], [0], 1), api.TagGroups("CB", [b"a\0b"], [0], 1), api.TagGroups("CB", ["a\nb"], [0], 1),
           api.TagGroups("CB", ["x" * 256], [0], 1)]
    for t in bad:
        with pytest.raises(ValueError):
            api.read_bam(bam, list(w.chroms), groups=t)
    ok = api.read_bam(bam, list(w.chroms), groups=api.TagGroups("CB", ["x" * 255], [0], 65535))
    assert set(np.unique(ok.group).tolist()) <= {-1, -2}


# ---------------------------------------------------------------------------------------------------------- CPU: the groups file
def test_groups_file_parsing(tmp_path):
    from spliser_b200 import cli
    p = tmp_path / "g.tsv"
    p.write_text("AAAC-1\tT cells\nAAAG-1\tB\nAACT-1\tT cells\n")
    assert cli.read_groups_file(str(p)) == (["AAAC-1", "AAAG-1", "AACT-1"], [0, 1, 0], ["T cells", "B"])
    for text, line in (("a\tA\nb\n", 2), ("a\tA\tx\n", 1), ("a\tA\na\tB\n", 2), ("a\tx/y\n", 1), ("a\tx\0y\n", 1), ("\tA\n", 1),
                       ("a\t\n", 1), ("a\tA\n" + "x" * 256 + "\tB\n", 2), ("a\0b\tA\n", 1), ("a\tA\n" + "\u00e9" * 128 + "\tB\n", 2)):
        p.write_text(text)
        with pytest.raises(cli.GroupsFileError, match="line %d" % line):
            cli.read_groups_file(str(p))


def test_groups_file_errors_are_parser_errors(tmp_path, monkeypatch, capsys, built_library):
    from spliser_b200 import cli
    p = tmp_path / "g.tsv"
    p.write_text("a\tA\na\tB\n")
    with pytest.raises(SystemExit) as e:
        cli.main(["combineGroups", "-B", "x.bam", "--tag", "CB", "-G", str(p), "-o", str(tmp_path / "o")])
    assert e.value.code == 2 and "line 2" in capsys.readouterr().err
    for tag in ("C", "1B", "CBX"):
        with pytest.raises(SystemExit):
            cli.main(["combineGroups", "-B", "x.bam", "--tag", tag, "-G", str(p), "-o", str(tmp_path / "o")])


# ---------------------------------------------------------------------------------------------------------- CPU: the command
class GroupHostSample(VotingSample):
    """A stand-in group sample: the group's records of the host reader, under the BAM's full header."""

    def __init__(self, owner, path, refs, rec):
        self.owner, self.path, self.refs, self.rec, self.closed = owner, path, refs, rec, False


class GroupingContext(VotingContext):
    """VotingContext with load_bam_groups, answered by the host reader's group column (spl_read_bam_groups)."""

    def load_bam_groups(self, bam_path, groups, xs=False):
        refs = api.bam_reference_names(bam_path)
        r = api.read_bam(bam_path, refs, xs=xs, groups=groups)
        self.kept = len(r)
        samples = []
        for g in range(groups.n_groups):
            s = subset(r, r.group == g)
            if xs:
                s.xs = r.xs[r.group == g]
            samples.append(GroupHostSample(self, bam_path, refs, s))
        counts = [int((r.group == g).sum()) for g in range(groups.n_groups)]
        return api.GroupedSamples(samples, counts, int((r.group == -1).sum()), int((r.group == -2).sum()))

    def last_read_filter(self):
        return self.kept, 0


def _groups_file(d, table, titles):
    p = os.path.join(d, "groups.tsv")
    with open(p, "w") as fh:
        fh.writelines("%s\t%s\n" % (v.decode(), titles[g]) for v, g in zip(table.values, table.groups.tolist()))
    return p


def _texts(paths):
    return [open(p).read() for p in paths]


@pytest.fixture(scope="module")
def cb_bams(tmp_path_factory, lib):
    w, rec, mapq, aux = lib
    d = str(tmp_path_factory.mktemp("cb"))
    table = tables()["CB"]
    titles = ["c0", "c1", "c2", "empty"]
    full, per, grp = write_groups(d, "x", w, rec, aux, mapq, table)
    gff = os.path.join(d, "genes.gff")
    gff_of(w, gff)
    return d, table, titles, full, per, grp, gff


CLI_MODES = {"rf": dict(isStranded=True, strandedType="rf"), "auto": dict(isStranded=True, strandedType="auto"),
             "shallow": dict(shallow=True, minSamples=1, minReads=2, minSSE=0.1, annotationFile=None),
             "xs": dict(strandFromXS=True)}


def _reference(d, tag, per, titles, factory=None, **kw):
    sf = os.path.join(d, tag + ".samples.tsv")
    tsvs = [os.path.join(d, "%s.%s.SpliSER.tsv" % (tag, t)) for t in titles]
    with open(sf, "w") as fh:
        fh.writelines("%s\t%s\t%s\n" % x for x in zip(titles, tsvs, per))
    from spliser_b200 import cli
    cli.combineBam(sf, os.path.join(d, tag), context_factory=factory, **kw)
    return _texts(tsvs + [os.path.join(d, tag + ".combined.tsv")])


def _groups_run(d, tag, full, gf, titles, factory=None, **kw):
    from spliser_b200 import cli
    out = os.path.join(d, tag)
    cli.combineGroups(full, "CB", gf, out, context_factory=factory, **kw)
    return _texts(["%s.%s.SpliSER.tsv" % (out, t) for t in titles] + [out + ".combined.tsv"])


@pytest.mark.parametrize("mode", sorted(CLI_MODES))
def test_combine_groups_with_stand_ins(tmp_path, cb_bams, mode, capsys):
    d0, table, titles, full, per, grp, gff = cb_bams
    d = str(tmp_path)
    kw = dict(CLI_MODES[mode])
    if mode == "shallow":
        kw["annotationFile"] = gff
    gf = _groups_file(d, table, titles)
    want = _reference(d, "ref", per, titles, lambda dev: VotingContext(), **kw)
    capsys.readouterr()
    lines = {}
    for n in (1, 3):
        got = _groups_run(d, "g%d" % n, full, gf, titles, lambda dev: GroupingContext(), devices=list(range(n)), **kw)
        assert got == want, (mode, n)
        lines[n] = [x for x in capsys.readouterr().out.splitlines() if x.startswith("Records per group")]
    assert lines[1] == lines[3] and len(lines[1]) == 1
    counts = np.bincount(grp + 2, minlength=len(titles) + 2)
    assert lines[1][0] == "Records per group (CB):\t%s\tno value %d\tvalue in no group %d" % (
        "\t".join("%s %d" % (t, counts[g + 2]) for g, t in enumerate(titles)), counts[1], counts[0])
    assert "empty" in titles and counts[2 + titles.index("empty")] == 0


def test_combine_groups_auto_refuses_disagreeing_groups(tmp_path, lib, built_library):
    """-s auto pools the groups' votes and refuses a run whose groups disagree: group 0 is the library as it is, group 1 the same
    reads with every strand flipped (an fr library), nothing written."""
    from spliser_b200 import cli
    w, rec, mapq, aux = lib
    both = Records(np.concatenate([rec.pos, rec.pos]), np.concatenate([rec.flag, rec.flag ^ 16]),
                   np.concatenate([rec.cig_off[:-1], rec.cig_off + rec.cig_off[-1]]), np.concatenate([rec.cigar, rec.cigar]),
                   [0], [0, 2 * len(rec)])
    chrom_all = np.concatenate([np.repeat(rec.seg_chrom, np.diff(rec.seg_off))] * 2)
    order = np.lexsort((np.arange(len(both)), both.pos, chrom_all))
    chrom = chrom_all[order]
    off = both.cig_off.astype(np.int64)
    cig = np.concatenate([both.cigar[off[i]:off[i + 1]] for i in order])
    n_op = (off[1:] - off[:-1])[order]
    seg = np.flatnonzero(np.r_[True, chrom[1:] != chrom[:-1]])
    mixed = Records(both.pos[order], both.flag[order], np.r_[0, np.cumsum(n_op)], cig, chrom[seg], np.r_[seg, len(order)])
    hp = np.repeat([1, 2], len(rec))[order]
    parts = [encode_aux([("HP", "i", int(h))]) for h in hp]
    off2 = np.r_[0, np.cumsum([len(p) for p in parts])]
    bam = str(tmp_path / "m.bam")
    mixed.write_bam(bam, w.chroms, w.chrom_len, aux=(off2, np.frombuffer(b"".join(parts), np.uint8)))
    gff = str(tmp_path / "genes.gff")
    gff_of(w, gff)
    gf = tmp_path / "g.tsv"
    gf.write_text("1\tas_is\n2\tflipped\n")
    with pytest.raises(cli.StrandednessError, match="flipped|as_is"):
        cli.combineGroups(bam, "HP", str(gf), str(tmp_path / "o"), annotationFile=gff, isStranded=True, strandedType="auto",
                          context_factory=lambda dev: GroupingContext())
    assert not os.path.exists(str(tmp_path / "o.combined.tsv"))


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
def gpu_lib(tmp_path_factory, built_library):
    w, rec, mapq = odd_library(61, 40_000)
    aux = aux_blocks(rec, 61)
    d = str(tmp_path_factory.mktemp("gpu_cb"))
    table = tables()["CB"]
    titles = ["c0", "c1", "c2", "empty"]
    full, per, grp = write_groups(d, "x", w, rec, aux, mapq, table)
    gff = os.path.join(d, "genes.gff")
    gff_of(w, gff)
    return d, w, table, titles, full, per, grp, gff


def _gaps(rec, chroms, n=300, seed=3):
    rng = np.random.default_rng(seed)
    seg = rng.integers(0, len(rec.seg_chrom), n)
    pos = rec.pos[np.minimum(rec.seg_off[seg] + rng.integers(0, 50, n), len(rec) - 1)] + rng.integers(0, 200, n)
    out = []
    for k in range(n):
        out.append((int(rec.seg_chrom[seg[k]]), int(pos[k]), "+-"[k % 2], [int(pos[k]) + 500], [int(pos[k]) - 300]))
    out.sort(key=lambda g: (g[0], g[1]))
    return out


def _calls(s, chroms, genes, gaps, xs):
    j, t = s.process_extract(chroms, api.FLAG_XS_STRAND if xs else 0)
    j2, t2 = s.process_extract(chroms, api.mode_flags(True, "rf"))
    b1, b2 = s.recount(chroms, gaps, api.mode_flags(True, "rf", combine=True))
    v = [s.infer_strand(chroms, genes)] + ([s.infer_strand(chroms, None)] if xs else [])
    return [j.chrom, j.left, j.right, j.strand, t.alpha, t.beta1, t.beta2simple, t.sse, j2.left, t2.beta1, b1, b2, v]


def _same(a, b):
    assert len(a) == len(b)
    for x, y in zip(a, b):
        if isinstance(x, np.ndarray):
            assert np.array_equal(x, y)
        else:
            assert x == y


@pytest.mark.gpu
@pytest.mark.parametrize("route", ROUTES, indirect=True)
@pytest.mark.parametrize("xs", [False, True])
def test_split_samples_answer_as_group_bams_on_gpu(gpu_lib, route, xs):
    from spliser_b200.genes import load_annotation
    d, w, table, titles, full, per, grp, gff = gpu_lib
    chroms = list(w.chroms)
    genes = api.gene_strands(load_annotation(gff, "All"), chroms)
    base = Records.from_bam(full, chroms)
    gaps = _gaps(base, chroms)
    with api.Context(0) as ctx:
        with ctx.load_bam_groups(full, table, xs=xs) as split:
            assert split.counts == [int((grp == g).sum()) for g in range(table.n_groups)]
            assert (split.no_value, split.unmatched) == (int((grp == -1).sum()), int((grp == -2).sum()))
            assert ctx.stats()["bam_on_device"] == (1.0 if route == "device" else 0.0)
            assert sum(split.counts) + split.no_value + split.unmatched == ctx.last_read_filter()[0]
            for g, s in enumerate(split.samples):
                assert s.n_records == split.counts[g]
                with ctx.load_bam(per[g], xs=xs) as ref:
                    a, b = s.records(), ref.records()
                    _same_records(a, b)                                 # the same columns, in the same (BAM) order
                    assert (a.xs is None) == (not xs) and (a.xs is None or np.array_equal(a.xs, b.xs))
                    _same(_calls(s, chroms, genes, gaps, xs), _calls(ref, chroms, genes, gaps, xs))
        # under a read filter: the same split of the kept records
        ctx.set_read_filter(FILTER)
        with ctx.load_bam_groups(full, table, xs=xs) as split:
            kept = ctx.last_read_filter()[0]
            assert sum(split.counts) + split.no_value + split.unmatched == kept


@pytest.mark.gpu
def test_combine_groups_equals_process_bam_and_combine_bam_on_gpu(tmp_path, gpu_lib):
    d0, w, table, titles, full, per, grp, gff = gpu_lib
    d = str(tmp_path)
    gf = _groups_file(d, table, titles)
    import torch
    n_dev = torch.cuda.device_count()
    modes = [dict(), dict(annotationFile=gff, qGene="busy"), dict(isStranded=True, strandedType="rf"),
             dict(isStranded=True, strandedType="auto"), dict(strandFromXS=True),
             dict(shallow=True, minSamples=1, minReads=2, minSSE=0.1), dict(read_filter=FILTER)]
    from spliser_b200 import cli
    from test_combine_bam import _busy_gene
    with api.Context(0) as c:
        gene = _busy_gene(cli, c, d, per[0], gff)
    for i, kw in enumerate(modes):
        kw = dict(kw)
        if "qGene" in kw:
            kw["qGene"] = gene
        want = _reference(d, "ref%d" % i, per, titles, **kw)
        got = _groups_run(d, "grp%d" % i, full, gf, titles, **kw)
        assert got == want, kw
    if n_dev >= 2:
        assert _groups_run(d, "two", full, gf, titles, devices=[0, 1]) == _reference(d, "ref_two", per, titles, devices=[0, 1])


def _keyed_bam(path, n, n_chrom, n_values, seed):
    """n records on n_chrom chromosomes (sorted by chromosome, then POS), every one with a CB:Z value drawn from n_values, and a
    FLAG and CIGAR length that change from record to record so that any reordering shows -> (Records, chrom, value)."""
    rng = np.random.default_rng(seed)
    chrom = np.sort(rng.integers(0, n_chrom, n)).astype(np.int32)
    pos = np.empty(n, np.int32)
    seg = np.flatnonzero(np.r_[True, chrom[1:] != chrom[:-1]])
    bounds = np.r_[seg, n]
    for k in range(len(seg)):
        pos[bounds[k]:bounds[k + 1]] = np.sort(rng.integers(1, 50_000_000, bounds[k + 1] - bounds[k]))
    i = np.arange(n)
    rec = Records(pos, ((i & 1) * 16).astype(np.uint16), np.arange(n + 1, dtype=np.uint32),
                  (((20 + i % 200) << 4)).astype(np.uint32), chrom[seg], bounds)
    val = rng.integers(0, n_values, n)
    fields = np.frombuffer(b"".join(b"CBZv%05d\0" % v for v in range(n_values)), np.uint8).reshape(n_values, 10)
    rec.write_bam(path, ["chr%d" % c for c in range(n_chrom)], [60_000_000] * n_chrom,
                  aux=(np.arange(n + 1, dtype=np.int64) * 10, fields[val].ravel()))       # every field: CB Z v00000 NUL
    return rec, chrom, val


def _check_group(sample, rec, chrom, sel):
    """The sample holds exactly the selected records, in BAM order, with their chromosome segments."""
    got = sample.records()
    idx = np.flatnonzero(sel)
    c = chrom[idx]
    seg = np.flatnonzero(np.r_[True, c[1:] != c[:-1]]) if len(idx) else np.zeros(0, np.int64)
    assert np.array_equal(got.pos, rec.pos[idx]) and np.array_equal(got.flag, rec.flag[idx])
    assert np.array_equal(got.cigar, rec.cigar[idx]) and np.array_equal(got.cig_off, np.arange(len(idx) + 1))
    assert np.array_equal(got.seg_chrom, c[seg]) and np.array_equal(got.seg_off, np.r_[seg, len(idx)] if len(idx) else [0])


@pytest.mark.gpu
def test_a_thousand_groups_on_gpu(tmp_path, built_library):
    """4M records, random values of 1000 groups (and 50 values in none): the two-pass sort.  Per-group counts equal numpy's, and
    each group's records, copied back, are the group's records in BAM order."""
    n, G = 4_000_000, 1000
    bam = str(tmp_path / "k.bam")
    rec, chrom, val = _keyed_bam(bam, n, 1, G + 50, 7)
    table = api.TagGroups("CB", [("v%05d" % v) for v in range(G)], list(range(G)), G)
    with api.Context(0) as ctx:
        with ctx.load_bam_groups(bam, table) as split:
            want = np.bincount(val, minlength=G + 50)
            assert split.counts == want[:G].tolist() and split.unmatched == int(want[G:].sum()) and split.no_value == 0
            for g in (0, 1, 3, 255, 256, 257, 511, 700, 999):
                _check_group(split.samples[g], rec, chrom, val == g)


@pytest.mark.gpu
def test_more_segments_than_one_bam_has_on_gpu(tmp_path, built_library):
    """A group restarts a segment on every chromosome it has records on: 30 chromosomes x 3000 groups give 90,000 segments, more
    than the 65,536 + 3000 a split first makes room for.  Every group still comes out whole."""
    n, R, G = 2_000_000, 30, 3000
    bam = str(tmp_path / "m.bam")
    rec, chrom, val = _keyed_bam(bam, n, R, G, 11)
    table = api.TagGroups("CB", [("v%05d" % v) for v in range(G)], list(range(G)), G)
    segs = len(np.unique(chrom.astype(np.int64) * G + val))
    assert segs > (1 << 16) + G
    with api.Context(0) as ctx:
        with ctx.load_bam_groups(bam, table) as split:
            assert split.counts == np.bincount(val, minlength=G).tolist()
            for g in (0, 1, 1500, 2999):
                _check_group(split.samples[g], rec, chrom, val == g)
            j, t = split.samples[5].process_extract(["chr%d" % c for c in range(R)])
            assert len(t) == 0                                          # unspliced records: no sites, and the call runs


@pytest.mark.gpu
@pytest.mark.parametrize("route", ROUTES, indirect=True)
def test_crafted_fields_on_gpu(tmp_path, route):
    t = api.TagGroups("HP", *CRAFTED_TABLE)
    rec, blocks, want = crafted_bam(str(tmp_path / "c.bam"))
    with api.Context(0) as ctx:
        with ctx.load_bam_groups(str(tmp_path / "c.bam"), t) as split:
            assert split.counts == [int((want == g).sum()) for g in range(t.n_groups)]
            assert (split.no_value, split.unmatched) == (int((want == -1).sum()), int((want == -2).sum()))
            for g in range(t.n_groups):
                _check_group(split.samples[g], rec, np.zeros(len(rec), np.int32), want == g)


@pytest.mark.gpu
def test_shared_allocation_is_freed_on_gpu(gpu_lib, monkeypatch):
    d, w, table, titles, full, per, grp, gff = gpu_lib
    chroms = list(w.chroms)
    with api.Context(0) as ctx:
        split = ctx.load_bam_groups(full, table)
        want = [s.process_extract(chroms)[1].beta1.copy() for s in split.samples]
        total = sum(s.device_bytes for s in split.samples)
        for g in (1, 3):                                                # interleaved: the others keep answering
            split.samples[g].close()
        for g in (0, 2):
            assert np.array_equal(split.samples[g].process_extract(chroms)[1].beta1, want[g])
        split.close()
        monkeypatch.setenv("SPLISER_SAMPLE_BUDGET_MB", str(total // (1 << 20) + 1))
        sums = set()
        for _ in range(20):
            with ctx.load_bam_groups(full, table) as s:
                sums.add(sum(x.device_bytes for x in s.samples))
        assert sums == {total}
        monkeypatch.setenv("SPLISER_SAMPLE_BUDGET_MB", str(max(0, total // (1 << 20) - 1)))
        with pytest.raises(api.SampleMemoryError, match="bytes"):
            ctx.load_bam_groups(full, table)


@pytest.mark.gpu
def test_combine_groups_refuses_a_split_that_does_not_fit_on_gpu(tmp_path, gpu_lib, monkeypatch, capsys):
    from spliser_b200 import cli
    d, w, table, titles, full, per, grp, gff = gpu_lib
    gf = _groups_file(str(tmp_path), table, titles)
    monkeypatch.setenv("SPLISER_SAMPLE_BUDGET_MB", "0")
    with pytest.raises(SystemExit):
        cli.main(["combineGroups", "-B", full, "--tag", "CB", "-G", gf, "-o", str(tmp_path / "o")])
    assert "--gpus" in capsys.readouterr().err
