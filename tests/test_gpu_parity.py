"""GPU parity tests proper: the CUDA path through the C ABI against (a) the committed golden
vectors produced by the unmodified reference and (b) the oracle on fresh seeded inputs.
Integer counts must be identical; float64 SSE / beta2Cryptic_weighted are compared bit-for-bit
(0 ulp: IEEE division, no FMA contraction -- tighter than the 1 ulp north_star allows)."""
import pytest

from common import (case_flags, first_diff, gpu_process_rows, load_golden, oracle_process_rows, strip_gene)

pytestmark = pytest.mark.gpu


def test_appendix_a_known_answers(ctx):
    g = load_golden("appendix_a.json.gz")
    for case in g["process"]:
        if "qgene" in case:      # locus filter needs the annotation: covered by the CLI test
            continue
        got = gpu_process_rows(ctx, case)
        d = first_diff(got, strip_gene(case["rows"]))
        assert d is None, "%s: %s" % (case["name"], d)


def test_golden_process_fuzz(ctx):
    cases = load_golden("process_fuzz.json.gz")
    assert len(cases) >= 300
    bad = []
    for case in cases:
        d = first_diff(gpu_process_rows(ctx, case), strip_gene(case["rows"]))
        if d:
            bad.append((case["seed"], d))
    assert not bad, "%d/%d cases differ; first: seed %s %s" % (len(bad), len(cases), bad[0][0], bad[0][1])


def test_golden_process_via_bam(ctx, tmp_path):
    cases = load_golden("process_fuzz.json.gz")[:60]
    for case in cases:
        d = first_diff(gpu_process_rows(ctx, case, via_bam=str(tmp_path)), strip_gene(case["rows"]))
        assert d is None, "seed %s: %s" % (case["seed"], d)


def test_golden_combine_recount(ctx):
    from spliser_b200 import Records
    cases = load_golden("combine_fuzz.json.gz") + load_golden("appendix_a.json.gz")["combine"]
    n = 0
    for case in cases:
        flags = case_flags(case) | 8
        by_sample = {}
        for gap in case["gaps"]:
            by_sample.setdefault(gap["sample"], []).append(gap)
        for s, gaps in by_sample.items():
            reads = [tuple(r) for r in case["samples"][s]["reads"]]
            rec = Records.from_reads(["C"], reads)
            arg = [(0 if g["chrom"] == "C" else -1, g["pos"], g["strand"], g["partners"], g["competitors"]) for g in gaps]
            b1, b2 = ctx.recount_records(rec, 1, arg, flags)
            for g, x, y in zip(gaps, b1, b2):
                n += 1
                assert (int(x), int(y)) == (g["beta1"], g["beta2s"]), (case.get("seed", case.get("name")), g, int(x), int(y))
    assert n > 300


@pytest.mark.parametrize("seed0", [900000, 910000])
def test_live_fuzz_vs_oracle(ctx, seed0):
    from oracle import fuzzgen
    bad = []
    for seed in range(seed0, seed0 + 150):
        case = fuzzgen.gen_case(seed, n_chrom=1 + (seed % 3 == 0), dirty=(seed % 4 == 1), max_reads=60)
        d = first_diff(gpu_process_rows(ctx, case), oracle_process_rows(case))
        if d:
            bad.append((seed, d))
    assert not bad, "%d cases differ; first: seed %s %s" % (len(bad), bad[0][0], bad[0][1])


def test_empty_and_ragged_inputs(ctx):
    import numpy as np
    from spliser_b200 import Junctions, Records
    empty_j = Junctions(np.zeros(0, np.int32), np.zeros(0, np.int32), np.zeros(0, np.int32), np.zeros(0, np.int64), np.zeros(0, np.uint8))
    # no junctions, no reads
    t = ctx.process_records(Records.from_reads([], []), 0, empty_j, 0)
    assert len(t) == 0
    # reads but no junctions
    t = ctx.process_records(Records.from_reads(["C"], [("C", 10, 0, "50M")]), 1, empty_j, 0)
    assert len(t) == 0
    # junctions but no reads; reads on a chromosome without junctions; reads without CIGAR
    j = Junctions([0, 0], [100, 100], [200, 300], [5, 3], [ord("+"), ord("+")])
    t = ctx.process_records(Records.from_reads(["C", "D"], [("D", 90, 0, "30M"), ("Z", 5, 0, "10M"), ("C", 95, 0, "*")]), 2, j, 0)
    assert list(t.pos) == [100, 200, 300] and list(t.alpha) == [8, 5, 3] and int(t.beta1.sum()) == 0
    assert [float(x) for x in t.sse] == [1.0, 0.625, 1.0]      # site 200: junction (100,300) flanks it -> beta2Simple 3 (S:594-599)
    assert list(t.beta2simple) == [0, 3, 0]


@pytest.mark.parametrize("stranded,paired,n", [(False, False, 150_000), (True, True, 400_000)])
def test_synthetic_workload_vs_c_oracle(ctx, stranded, paired, n):
    """Config-shaped synthetic sample (sizes the C oracle finishes in seconds), every output column."""
    from oracle import c_oracle
    from spliser_b200 import synth
    w = synth.generate(synth.config_small(n, seed=21 + stranded, stranded=stranded, paired=paired))
    for flags in (w.flags, w.flags | 4, w.flags | 8):
        want = c_oracle.process(w.records, len(w.chroms), w.junctions, flags, threads=8)
        got = c_oracle.table_dict(ctx.process_records(w.records, len(w.chroms), w.junctions, flags))
        assert c_oracle.diff_tables(got, want) is None, (flags, c_oracle.diff_tables(got, want))
    assert int(want["beta1"].sum()) > 0 and int(want["beta2simple"].sum()) > 0


def test_c1_shaped_workload_vs_c_oracle(ctx):
    """BASELINE configs[0] shape at reduced depth (400k of the 2M records), unstranded."""
    from oracle import c_oracle
    from spliser_b200 import synth
    cfg = synth.config_c1()
    cfg.n_records = 400_000
    w = synth.generate(cfg)
    want = c_oracle.process(w.records, len(w.chroms), w.junctions, w.flags, threads=8)
    got = c_oracle.table_dict(ctx.process_records(w.records, len(w.chroms), w.junctions, w.flags))
    assert c_oracle.diff_tables(got, want) is None, c_oracle.diff_tables(got, want)


def test_full_configs0_equals_the_unmodified_reference(ctx, tmp_path):
    """BASELINE configs[0] at its full size (2M records, 28.6k junctions, 56k sites, unstranded): the unmodified reference
    ran this workload in the authoring container (oracle/time_reference.py) and left a digest of its own per-site result
    (tests/golden/c1_full_reference.json).  The CUDA path must reproduce it from the record arrays and from a BAM file."""
    import json
    import os
    from common import GOLDEN
    from oracle import c_oracle, time_reference
    from spliser_b200 import synth
    gold = json.load(open(os.path.join(GOLDEN, "c1_full_reference.json")))
    w = synth.generate(synth.config_c1())
    got = c_oracle.table_dict(ctx.process_records(w.records, len(w.chroms), w.junctions, w.flags))
    assert len(got["pos"]) == gold["sites"]
    assert {k: int(got[k].sum()) for k in ("alpha", "beta1", "beta2simple")} == gold["sums"]
    assert time_reference.digest_of_table(got) == gold["digest"]
    full = json.load(open(os.path.join(GOLDEN, "reference_digests.json")))["shapes"]["c1_full"]["digest"]
    assert time_reference.full_digest_of_table(got) == full                # every column, Partners / Competitors included
    bam = str(tmp_path / "c1.bam")
    w.records.write_bam(bam, w.chroms, w.chrom_len)
    via_bam = c_oracle.table_dict(ctx.process_bam(bam, w.chroms, w.junctions, w.flags))
    assert time_reference.digest_of_table(via_bam) == gold["digest"]


def test_resident_path_equals_process_path(ctx):
    from oracle import c_oracle
    from spliser_b200 import synth
    w = synth.generate(synth.config_small(120_000, seed=33, stranded=True, paired=True))
    a = c_oracle.table_dict(ctx.process_records(w.records, len(w.chroms), w.junctions, w.flags | 4))
    ctx.resident_load(w.records, len(w.chroms), w.junctions, w.flags | 4)
    st = ctx.resident_count(3)                 # idempotent: counters are re-zeroed every pass
    b = c_oracle.table_dict(ctx.resident_fetch())
    assert c_oracle.diff_tables(a, b) is None
    assert st["n_aligned"] == len(w.records) and st["ms_total"] > 0


def test_stabbing_variant_equals_difference_array_variant(ctx):
    """north_star: the stabbing count (block-vs-site, TMA-staged site tiles) is checked against the difference-array /
    prefix-scan formulation.  Both variants must give the oracle's table: fuzz cases (every branch), a stranded synthetic
    sample through process, the resident path and a combine re-count."""
    from oracle import c_oracle, fuzzgen
    from spliser_b200 import synth
    import os
    small = os.environ.get("SPLISER_SANITIZE_SMALL") == "1"           # under compute-sanitizer: the same kernels on less data
    w = synth.generate(synth.config_small(6_000 if small else 150_000, seed=35, stranded=True, paired=True))
    want = c_oracle.process(w.records, len(w.chroms), w.junctions, w.flags | 4, threads=8)
    cases = [fuzzgen.gen_case(seed, n_chrom=1 + (seed % 2), dirty=(seed % 4 == 1), max_reads=60) for seed in range(930000, 930008 if small else 930040)]
    try:
        for variant in ("stab", "fused"):
            ctx.set_variant(variant)
            for case in cases:
                d = first_diff(gpu_process_rows(ctx, case), oracle_process_rows(case))
                assert d is None, (variant, case["seed"], d)
            got = c_oracle.table_dict(ctx.process_records(w.records, len(w.chroms), w.junctions, w.flags | 4))
            assert c_oracle.diff_tables(got, want) is None, (variant, c_oracle.diff_tables(got, want))
            ctx.resident_load(w.records, len(w.chroms), w.junctions, w.flags | 4)
            ctx.resident_count(2)
            got = c_oracle.table_dict(ctx.resident_fetch())
            assert c_oracle.diff_tables(got, want) is None, (variant, "resident", c_oracle.diff_tables(got, want))
    finally:
        ctx.set_variant("fused")


@pytest.mark.parametrize("parts", [1, 3])
def test_packed_view_equals_plain_view(ctx, monkeypatch, parts):
    """spl_process_packed (POS, three flag bits, operator count, sparse CIGAR index; offsets and SAM flag bits rebuilt on the
    device) gives the table of spl_process_records: a stranded paired synthetic sample incl. odd flags, one slab and three."""
    from oracle import c_oracle, fuzzgen
    from spliser_b200 import PackedRecords, Records, synth
    from spliser_b200.bed import parse_bed12
    w = synth.generate(synth.config_small(150_000, seed=77, stranded=True, paired=True))
    want = c_oracle.process(w.records, len(w.chroms), w.junctions, w.flags | 4, threads=8)
    monkeypatch.setenv("SPLISER_SPLIT_MIN_RECORDS", "1000" if parts > 1 else "1000000000")
    monkeypatch.setenv("SPLISER_SPLIT_PARTS", str(parts))
    pk = PackedRecords.from_records(w.records)
    got = c_oracle.table_dict(ctx.process_packed(pk, len(w.chroms), w.junctions, w.flags | 4))
    assert ctx.stats()["n_parts"] == float(parts)
    assert c_oracle.diff_tables(got, want) is None, c_oracle.diff_tables(got, want)
    monkeypatch.delenv("SPLISER_SPLIT_MIN_RECORDS"); monkeypatch.delenv("SPLISER_SPLIT_PARTS")
    for seed in range(940000, 940030):                       # every flag combination / CIGAR shape of the fuzz generator
        case = fuzzgen.gen_case(seed, n_chrom=1 + (seed % 2), dirty=(seed % 4 == 1), max_reads=60)
        chroms, junc, _ = parse_bed12(case["bed"].splitlines(True))
        rec = Records.from_reads(chroms, [tuple(r) for r in case["reads"]])
        a = c_oracle.table_dict(ctx.process_records(rec, len(chroms), junc, case_flags(case)))
        b = c_oracle.table_dict(ctx.process_packed(PackedRecords.from_records(rec), len(chroms), junc, case_flags(case)))
        assert c_oracle.diff_tables(a, b) is None, (seed, c_oracle.diff_tables(a, b))


@pytest.mark.parametrize("parts", [1, 3])
def test_compact_view_equals_plain_view(ctx, monkeypatch, parts):
    """spl_process_compact (16-bit POS offsets per stride, operator count in a byte, 16-bit operators with a 32-bit stream for
    records with a long one; every stride unpacked on the device from its own anchors) gives the table of spl_process_records:
    a stranded paired sample in one slab and three, a GRCh38-shaped tile (wide strides, introns of 4096 bases and more),
    shuffled records (every stride wide) and the fuzz generator's flag / CIGAR shapes incl. empty inputs."""
    import numpy as np
    from oracle import c_oracle, fuzzgen
    from spliser_b200 import CompactRecords, Records, synth
    from spliser_b200.bed import parse_bed12
    import os
    small = os.environ.get("SPLISER_SANITIZE_SMALL") == "1"           # under compute-sanitizer: the same kernels on less data
    w = synth.generate(synth.config_small(8_000 if small else 150_000, seed=77, stranded=True, paired=True))
    want = c_oracle.process(w.records, len(w.chroms), w.junctions, w.flags | 4, threads=8)
    monkeypatch.setenv("SPLISER_SPLIT_MIN_RECORDS", "1000" if parts > 1 else "1000000000")
    monkeypatch.setenv("SPLISER_SPLIT_PARTS", str(parts))
    ck = CompactRecords.from_records(w.records)
    assert small or ck.wire_bytes < 10 * len(w.records)
    got = c_oracle.table_dict(ctx.process_compact(ck, len(w.chroms), w.junctions, w.flags | 4))
    assert ctx.stats()["n_parts"] == float(parts)
    assert c_oracle.diff_tables(got, want) is None, c_oracle.diff_tables(got, want)
    w3 = synth.generate(synth.config_c3_tile(20_000 if small else 200_000, tile=1))
    ck3 = CompactRecords.from_records(w3.records)
    assert len(ck3.cigar32) > 0 and len(ck3.pos_wide) > 0 and len(ck3.cigar16) > 0
    a = c_oracle.table_dict(ctx.process_records(w3.records, len(w3.chroms), w3.junctions, w3.flags | 4))
    b = c_oracle.table_dict(ctx.process_compact(ck3, len(w3.chroms), w3.junctions, w3.flags | 4))
    assert c_oracle.diff_tables(a, b) is None, c_oracle.diff_tables(a, b)
    monkeypatch.delenv("SPLISER_SPLIT_MIN_RECORDS"); monkeypatch.delenv("SPLISER_SPLIT_PARTS")
    # shuffled inside the segments: positions of a stride span the chromosome
    r = w.records
    rng = np.random.default_rng(3)
    order = np.concatenate([int(r.seg_off[s]) + rng.permutation(int(r.seg_off[s + 1] - r.seg_off[s])) for s in range(len(r.seg_chrom))])
    nop = np.diff(r.cig_off.astype(np.int64))[order]
    off = np.concatenate([[0], np.cumsum(nop)])
    src = np.repeat(r.cig_off[:-1].astype(np.int64)[order], nop) + (np.arange(int(off[-1])) - np.repeat(off[:-1], nop))
    sh = Records(r.pos[order], r.flag[order], off, r.cigar[src], r.seg_chrom, r.seg_off)
    b = c_oracle.table_dict(ctx.process_compact(CompactRecords.from_records(sh), len(w.chroms), w.junctions, w.flags | 4))
    assert c_oracle.diff_tables(b, want) is None, c_oracle.diff_tables(b, want)
    for seed in range(940000, 940006 if small else 940030):   # every flag combination / CIGAR shape of the fuzz generator
        case = fuzzgen.gen_case(seed, n_chrom=1 + (seed % 2), dirty=(seed % 4 == 1), max_reads=60)
        chroms, junc, _ = parse_bed12(case["bed"].splitlines(True))
        rec = Records.from_reads(chroms, [tuple(r) for r in case["reads"]])
        a = c_oracle.table_dict(ctx.process_records(rec, len(chroms), junc, case_flags(case)))
        b = c_oracle.table_dict(ctx.process_compact(CompactRecords.from_records(rec), len(chroms), junc, case_flags(case)))
        assert c_oracle.diff_tables(a, b) is None, (seed, c_oracle.diff_tables(a, b))
    empty = Records.from_reads(["A"], [])
    t = ctx.process_compact(CompactRecords.from_records(empty), len(w.chroms), w.junctions, w.flags)
    assert int(t.beta1.sum()) == 0 and np.array_equal(t.alpha, got["alpha"])
    from spliser_b200 import Junctions
    none = ctx.process_compact(ck, len(w.chroms), Junctions([], [], [], [], []), w.flags)
    assert len(none) == 0
    # a view whose per-record operator counts disagree with a stride's index is refused (by the device, which is what trusts
    # them), and the context works afterwards
    from spliser_b200 import SpliserError
    bad = CompactRecords.from_records(w.records)
    bad.n_op8 = bad.n_op8.copy()
    bad.n_op8[len(bad) // 2] += 3
    with pytest.raises(SpliserError):
        ctx.process_compact(bad, len(w.chroms), w.junctions, w.flags | 4)
    again = c_oracle.table_dict(ctx.process_compact(ck, len(w.chroms), w.junctions, w.flags | 4))
    assert c_oracle.diff_tables(again, want) is None


def test_shuffled_records_give_identical_counts(ctx):
    """Any record order inside a chromosome segment is exact (the sorted-input fast paths have fallbacks)."""
    import numpy as np
    from oracle import c_oracle
    from spliser_b200 import Records, synth
    w = synth.generate(synth.config_small(60_000, seed=44))
    r = w.records
    rng = np.random.default_rng(1)
    pos, flag, ops = [], [], []
    off = [0]
    for s in range(len(r.seg_chrom)):
        idx = np.arange(int(r.seg_off[s]), int(r.seg_off[s + 1]))
        rng.shuffle(idx)
        for i in idx:
            pos.append(r.pos[i]); flag.append(r.flag[i])
            ops.extend(r.cigar[int(r.cig_off[i]):int(r.cig_off[i + 1])])
            off.append(len(ops))
    sh = Records(pos, flag, off, ops, r.seg_chrom, r.seg_off)
    a = c_oracle.table_dict(ctx.process_records(r, len(w.chroms), w.junctions, 4))
    b = c_oracle.table_dict(ctx.process_records(sh, len(w.chroms), w.junctions, 4))
    assert c_oracle.diff_tables(a, b) is None


def test_tiles_concatenate_to_the_untiled_result(built_library):
    """Genomic-tile sharding: each tile context counts only the sites it owns; owned slices concatenate
    to the single-context result (SURVEY.md 8(e), run sequentially on one GPU)."""
    import numpy as np
    import spliser_b200
    from spliser_b200 import synth
    w = synth.generate(synth.config_small(80_000, seed=55, stranded=True, paired=True))
    with spliser_b200.Context(0) as full:
        ref = full.process_records(w.records, len(w.chroms), w.junctions, w.flags)
    S = len(ref)
    n_tiles = 3
    b1 = np.zeros(S, np.int64); b2 = np.zeros(S, np.int64); sse = np.zeros(S)
    for ti in range(n_tiles):
        with spliser_b200.Context(0, tile=(ti, n_tiles)) as c:
            t = c.process_records(w.records, len(w.chroms), w.junctions, w.flags)
        lo, hi = S * ti // n_tiles, S * (ti + 1) // n_tiles
        b1[lo:hi], b2[lo:hi], sse[lo:hi] = t.beta1[lo:hi], t.beta2simple[lo:hi], t.sse[lo:hi]
    assert np.array_equal(b1, ref.beta1) and np.array_equal(b2, ref.beta2simple) and np.array_equal(sse, ref.sse)


@pytest.mark.parametrize("shape", ["c3_tile", "c5_dense_locus", "c2_stranded"])
def test_config_shaped_workloads_vs_c_oracle(ctx, shape):
    """The other BASELINE.json configs at depths the C oracle finishes in seconds:
    configs[2] (one GRCh38-scale tile: long introns up to 500 kb), configs[4] (dense alternative-splicing locus,
    --beta2Cryptic) and configs[1] (TAIR10 contigs, stranded rf).  The unmodified reference ran the same three workloads in
    the authoring container (oracle/time_reference.py --shapes): the digest of its whole table (every column, Partners and
    Competitors included, floats by their bits) is in tests/golden/reference_digests.json and must be reproduced too."""
    import json
    import os
    from common import GOLDEN
    from oracle import c_oracle, time_reference
    from spliser_b200 import synth
    w, flags = time_reference.shape_workload(shape)
    flags_extra = flags & 4
    want = c_oracle.process(w.records, len(w.chroms), w.junctions, flags, threads=8)
    got = c_oracle.table_dict(ctx.process_records(w.records, len(w.chroms), w.junctions, flags))
    assert c_oracle.diff_tables(got, want) is None, c_oracle.diff_tables(got, want)
    assert int(want["beta1"].sum()) > 0 and int(want["beta2simple"].sum()) > 0
    if flags_extra:
        assert int(want["beta2cryptic"].sum()) > 0
    gold = json.load(open(os.path.join(GOLDEN, "reference_digests.json")))["shapes"][shape]
    assert gold["records"] == len(w.records) and gold["sites"] == len(got["pos"])
    assert time_reference.full_digest_of_table(got) == gold["digest"]


def test_host_and_device_graph_builders_agree(ctx, monkeypatch):
    """Clean regime: the site table / competing-site graph is built on the device (sort / unique / group-by,
    graph_build.cu); SPLISER_HOST_GRAPH=1 forces the host builder (site_graph.cpp).  Every output column and
    both CSR structures must be identical, stranded and unstranded."""
    from oracle import c_oracle
    from spliser_b200 import synth
    for stranded in (True, False):
        w = synth.generate(synth.config_small(100_000, seed=77 + stranded, stranded=stranded, paired=stranded))
        monkeypatch.delenv("SPLISER_HOST_GRAPH", raising=False)
        dev = c_oracle.table_dict(ctx.process_records(w.records, len(w.chroms), w.junctions, w.flags | 4))
        assert ctx.stats()["graph_on_device"] == 1.0
        monkeypatch.setenv("SPLISER_HOST_GRAPH", "1")
        host = c_oracle.table_dict(ctx.process_records(w.records, len(w.chroms), w.junctions, w.flags | 4))
        assert ctx.stats()["graph_on_device"] == 0.0
        monkeypatch.delenv("SPLISER_HOST_GRAPH", raising=False)
        assert c_oracle.diff_tables(dev, host) is None, c_oracle.diff_tables(dev, host)
        assert len(dev["pos"]) > 1000 and len(dev["comp_pos"]) > 0


def test_cooperative_and_per_phase_graph_builds_agree(ctx, tmp_path):
    """K1 runs as ONE cooperative kernel (k_gb_coop); SPLISER_K1_LAUNCHES=1 selects the launch-per-phase build it replaced (the
    choice is taken once per process, hence the child process).  Both must give the same table in every column -- stranded and
    unstranded, a table with hub sites (many partners per site: the general per-site loops) and a one-junction table."""
    import json
    import os
    import subprocess
    import sys
    import textwrap
    ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    script = tmp_path / "k1.py"
    script.write_text(textwrap.dedent('''
        import hashlib, json, sys
        sys.path.insert(0, %r)
        import numpy as np
        import spliser_b200
        from spliser_b200 import Junctions, synth
        from oracle import c_oracle
        out = {}
        with spliser_b200.Context(0) as ctx:
            for name, stranded in (("s", True), ("u", False)):
                w = synth.generate(synth.config_small(150_000, seed=501 + stranded, stranded=stranded, paired=stranded))
                j = w.junctions
                cases = {"full": j, "one": Junctions(j.chrom[:1], j.left[:1], j.right[:1], j.score[:1], j.strand[:1])}
                # hubs: every 7th junction gets the left end of its predecessor on the same chromosome
                left = j.left.copy()
                for i in range(7, len(left), 7):
                    if j.chrom[i] == j.chrom[i - 1] and left[i - 1] < j.right[i]: left[i] = left[i - 1]
                cases["hubs"] = Junctions(j.chrom, left, j.right, j.score, j.strand)
                for cname, jj in cases.items():
                    t = c_oracle.table_dict(ctx.process_records(w.records, len(w.chroms), jj, w.flags | 4))
                    assert ctx.stats()["graph_on_device"] == 1.0
                    d = c_oracle.diff_tables(t, c_oracle.process(w.records, len(w.chroms), jj, w.flags | 4, threads=8))
                    assert d is None, (name, cname, d)
                    h = hashlib.sha256()
                    for k in sorted(t):
                        h.update(k.encode()); h.update(np.ascontiguousarray(t[k]).tobytes())
                    out[name + "/" + cname] = [h.hexdigest(), int(len(t["pos"])), int(len(t["comp_pos"]))]
        print("DIGESTS " + json.dumps(out))
    ''' % ROOT))
    got = {}
    for mode in ("0", "1"):
        env = dict(os.environ, SPLISER_K1_LAUNCHES=mode)
        res = subprocess.run([sys.executable, str(script)], capture_output=True, text=True, timeout=600, env=env)
        assert res.returncode == 0, res.stdout[-1500:] + res.stderr[-1500:]
        got[mode] = json.loads([l for l in res.stdout.splitlines() if l.startswith("DIGESTS ")][-1][8:])
    assert got["0"] == got["1"], (got["0"], got["1"])
    assert got["0"]["s/hubs"][1] > 1000 and got["0"]["s/hubs"][2] > got["0"]["s/full"][2]      # hubs make competitors


def test_c4_shaped_recount_vs_c_oracle(ctx):
    """BASELINE configs[3] shape at reduced size: K samples of one genome (own reads, own junction subset); every site
    of the merged table that a sample lacks is re-counted in that sample's reads with the partner / competitor
    positions accumulated from the lower-indexed samples (S:869-904), strand '' when no earlier sample had it."""
    import numpy as np
    from oracle import c_oracle
    from spliser_b200 import Junctions, Records, api, synth
    K = 4
    w = synth.generate(synth.config_small(240_000, seed=91, stranded=True, paired=True))
    rng = np.random.default_rng(5)
    r, j = w.records, w.junctions
    n_chrom = len(w.chroms)
    samples = []
    for k in range(K):
        keep_j = rng.random(len(j)) < 0.85
        jk = Junctions(j.chrom[keep_j], j.left[keep_j], j.right[keep_j], j.score[keep_j], j.strand[keep_j])
        pos, flag, ops, off, seg_off = [], [], [], [0], [0]
        for s in range(len(r.seg_chrom)):
            for i in range(int(r.seg_off[s]) + k, int(r.seg_off[s + 1]), K):
                pos.append(r.pos[i]); flag.append(r.flag[i])
                ops.extend(r.cigar[int(r.cig_off[i]):int(r.cig_off[i + 1])])
                off.append(len(ops))
            seg_off.append(len(pos))
        rk = Records(pos, flag, off, ops, r.seg_chrom, seg_off)
        tk = api.build_site_table(n_chrom, jk, w.flags)
        table = {}
        for i in range(len(tk)):
            table[(int(tk.chrom[i]), int(tk.pos[i]), tk.strand_str(i))] = (sorted(tk.partners(i)), tk.competitors(i))
        samples.append((rk, table))
    union = sorted(set().union(*[set(t) for _, t in samples]))
    total = 0
    for k in range(K):
        rk, tab = samples[k]
        gaps = []
        for key in union:
            if key in tab:
                continue
            P, C, strand = set(), set(), ""
            for jx in range(k):
                if key in samples[jx][1]:
                    p, c = samples[jx][1][key]
                    P |= set(p); C |= set(c); strand = key[2]
            gaps.append((key[0], key[1], strand, sorted(P), sorted(C)))
        assert gaps
        want1, want2 = c_oracle.recount(rk, n_chrom, gaps, w.flags | 8, threads=8)
        got1, got2 = ctx.recount_records(rk, n_chrom, gaps, w.flags | 8)
        assert np.array_equal(got1, want1) and np.array_equal(got2, want2), (k, int(np.sum(got1 != want1)), int(np.sum(got2 != want2)))
        total += int(want1.sum()) + int(want2.sum())
    assert total > 0


def _subset(r, keep):
    """Records restricted to a boolean mask (vectorised; segments keep their chromosome)."""
    import numpy as np
    from spliser_b200 import Records
    ncig = np.diff(r.cig_off.astype(np.int64))
    op_keep = np.repeat(keep, ncig)
    off = np.zeros(int(keep.sum()) + 1, np.uint32)
    np.cumsum(ncig[keep], out=off[1:])
    csum = np.concatenate([[0], np.cumsum(keep)])
    seg_off = csum[r.seg_off]
    return Records(r.pos[keep], r.flag[keep], off, r.cigar[op_keep], r.seg_chrom, seg_off)


def test_full_size_configs1_properties(ctx):
    """BASELINE configs[1] at its full size (40M records, stranded rf): (0) the whole table equals the C oracle's, and
    size-independent properties:
    (1) counts are additive over any split of the reads once the junction-table-only part is removed,
    (2) genomic tiles concatenate to the untiled result, (3) passes over the resident layout are idempotent,
    (4) alpha equals the junction scores summed per site."""
    import os
    import tempfile
    import numpy as np
    import spliser_b200
    from spliser_b200 import Records, synth
    n = int(os.environ.get("SPLISER_FULLSIZE_READS", "40000000"))
    cache = os.environ.get("SPLISER_BENCH_CACHE", os.path.join(tempfile.gettempdir(), "spliser_bench_cache"))
    w = synth.generate(synth.config_c2(n), cache_dir=cache)
    r, j, nc = w.records, w.junctions, len(w.chroms)
    full = ctx.process_records(r, nc, j, w.flags)
    S = len(full)
    assert S > 100_000 and int(full.beta1.sum()) > 0 and int(full.beta2simple.sum()) > 0
    # (0) the whole table against the C oracle (the reference's algorithm, pinned to its golden vectors) at the full size, every
    # column, floats bit for bit -- through the plain view and through the compact view
    from oracle import c_oracle
    from spliser_b200 import CompactRecords
    want = c_oracle.process(r, nc, j, w.flags, threads=os.cpu_count() or 8)
    d = c_oracle.diff_tables(c_oracle.table_dict(full), want)
    assert d is None, d
    d = c_oracle.diff_tables(c_oracle.table_dict(ctx.process_compact(CompactRecords.from_records(r), nc, j, w.flags)), want)
    assert d is None, d
    del want
    # (4)
    assert int(full.alpha.sum()) == 2 * int(j.score.sum())
    # (1) linearity
    rng = np.random.default_rng(11)
    keep = rng.random(len(r)) < 0.5
    a = ctx.process_records(_subset(r, keep), nc, j, w.flags)
    b = ctx.process_records(_subset(r, ~keep), nc, j, w.flags)
    none = ctx.process_records(Records(np.zeros(0, np.int32), np.zeros(0, np.uint16), np.zeros(1, np.uint32), np.zeros(0, np.uint32),
                                       np.zeros(0, np.int32), np.zeros(1, np.int64)), nc, j, w.flags)
    assert np.array_equal(a.pos, full.pos) and np.array_equal(none.pos, full.pos)
    assert int(none.beta1.sum()) == 0
    assert np.array_equal(a.beta1 + b.beta1, full.beta1)
    assert np.array_equal(a.beta2simple + b.beta2simple - none.beta2simple, full.beta2simple)
    assert np.array_equal(a.alpha, full.alpha) and np.array_equal(a.partner_cnt, full.partner_cnt)
    # (3) idempotence of the resident passes
    ctx.resident_load(r, nc, j, w.flags)
    ctx.resident_count(3)
    res = ctx.resident_fetch()
    for k in ("beta1", "beta2simple", "sse", "alpha", "beta2cryptic"):
        assert np.array_equal(getattr(res, k), getattr(full, k)), k
    # (2) tiles
    n_tiles = 4
    b1 = np.zeros(S, np.int64); b2 = np.zeros(S, np.int64)
    for ti in range(n_tiles):
        with spliser_b200.Context(0, tile=(ti, n_tiles)) as c:
            t = c.process_records(r, nc, j, w.flags)
            lo, hi = S * ti // n_tiles, S * (ti + 1) // n_tiles
            b1[lo:hi], b2[lo:hi] = t.beta1[lo:hi], t.beta2simple[lo:hi]
    assert np.array_equal(b1, full.beta1) and np.array_equal(b2, full.beta2simple)


def test_configs2_tile_at_scale_vs_c_oracle(ctx):
    """A GRCh38-scale tile of BASELINE configs[2] with 25M records (introns up to 500 kb): the rows of the first chromosome
    segment against the C oracle run on that segment's records and junction rows (every column a read can change), and the
    whole table's alpha against the junction scores."""
    import os
    import tempfile
    import numpy as np
    from oracle import c_oracle
    from spliser_b200 import Junctions, Records, synth
    n = int(os.environ.get("SPLISER_C3_TILE_READS", "25000000"))
    cache = os.environ.get("SPLISER_BENCH_CACHE", os.path.join(tempfile.gettempdir(), "spliser_bench_cache"))
    w = synth.generate(synth.config_c3_tile(n, tile=0), cache_dir=cache)
    r, j, nc = w.records, w.junctions, len(w.chroms)
    t = ctx.process_records(r, nc, j, w.flags)
    assert int(t.alpha.sum()) == 2 * int(j.score.sum()) and int(t.beta1.sum()) > 0
    k = int(r.seg_off[1] - r.seg_off[0])
    c0 = int(r.seg_chrom[0])
    rec = Records(r.pos[:k], r.flag[:k], r.cig_off[:k + 1], r.cigar[:int(r.cig_off[k])], [c0], [0, k])
    keep = j.chrom == c0
    sub = Junctions(j.chrom[keep], j.left[keep], j.right[keep], j.score[keep], j.strand[keep])
    want = c_oracle.process(rec, nc, sub, w.flags, threads=os.cpu_count() or 8)
    rows = np.nonzero(np.asarray(t.chrom) == c0)[0]
    assert len(rows) == len(want["pos"]) > 1000
    got = c_oracle.table_dict(t)
    for col in ("pos", "strand", "alpha", "beta1", "beta2simple", "beta2cryptic"):
        assert np.array_equal(np.asarray(got[col])[rows], np.asarray(want[col])), col
    assert np.array_equal(np.asarray(got["sse"])[rows].view(np.int64), np.asarray(want["sse"]).view(np.int64))


def test_bam_ingest_on_the_device(ctx, tmp_path, monkeypatch):
    """spl_process / spl_recount from a BAM file: BGZF inflate and BAM record parsing run on the GPU (bam_gpu.cu; record
    boundaries are speculated per BGZF member and verified as one chain).  Results must equal the records path and the
    host reader, with references in a different order than the caller's chromosome index and an unknown reference."""
    import numpy as np
    from oracle import c_oracle
    from spliser_b200 import Junctions, Records, synth
    w = synth.generate(synth.config_small(150_000, seed=61, stranded=True, paired=True))
    r, j = w.records, w.junctions
    # BAM reference order: [ZZ (unknown to the caller), T1, T2]; caller chrom_index: [T2, T1]
    bam = str(tmp_path / "s.bam")
    extra = Records.from_reads(["ZZ"], [("ZZ", 100 + 3 * i, 0, "20M100N20M") for i in range(500)])
    pos = np.concatenate([extra.pos, r.pos]); flag = np.concatenate([extra.flag, r.flag])
    cig = np.concatenate([extra.cigar, r.cigar])
    off = np.concatenate([extra.cig_off, r.cig_off[1:] + extra.cig_off[-1]])
    seg_chrom = np.concatenate([[0], r.seg_chrom + 1]); seg_off = np.concatenate([[0], r.seg_off + len(extra)])
    Records(pos, flag, off, cig, seg_chrom, seg_off).write_bam(bam, ["ZZ"] + list(w.chroms))
    caller = [w.chroms[1], w.chroms[0]]
    remap = np.array([1, 0], np.int32)
    jj = Junctions(remap[j.chrom], j.left, j.right, j.score, j.strand)
    order = [int(np.nonzero(r.seg_chrom == c)[0][0]) for c in (0, 1)]     # records path input in BAM order, caller indices
    rec_caller = Records(r.pos, r.flag, r.cig_off, r.cigar, remap[r.seg_chrom], r.seg_off)
    want = c_oracle.table_dict(ctx.process_records(rec_caller, 2, jj, w.flags | 4))
    monkeypatch.delenv("SPLISER_HOST_BAM", raising=False)
    got = c_oracle.table_dict(ctx.process_bam(bam, caller, jj, w.flags | 4))
    st = ctx.stats()
    assert st["bam_on_device"] == 1.0 and st["n_aligned"] == len(r), st
    assert c_oracle.diff_tables(got, want) is None, c_oracle.diff_tables(got, want)
    monkeypatch.setenv("SPLISER_HOST_BAM", "1")
    host = c_oracle.table_dict(ctx.process_bam(bam, caller, jj, w.flags | 4))
    assert ctx.stats()["bam_on_device"] == 0.0
    assert c_oracle.diff_tables(host, want) is None
    monkeypatch.delenv("SPLISER_HOST_BAM", raising=False)
    # the re-count entry point takes the same route
    t = ctx.process_records(rec_caller, 2, jj, w.flags)
    gaps = [(int(t.chrom[i]), int(t.pos[i]), t.strand_str(i), sorted(t.partners(i)), t.competitors(i)) for i in range(0, len(t), 7)]
    a1, a2 = ctx.recount_records(rec_caller, 2, gaps, w.flags | 8)
    b1, b2 = ctx.recount_bam(bam, caller, gaps, w.flags | 8)
    assert ctx.stats()["bam_on_device"] == 1.0
    assert np.array_equal(a1, b1) and np.array_equal(a2, b2) and int(a1.sum()) > 0
    assert len(order) == 2
    # a sequencer-shaped file (read names, SEQ, QUAL: members of mostly literals, records far longer than their CIGAR)
    seq_bam = str(tmp_path / "seq.bam")
    rec_caller.write_bam(seq_bam, caller, with_seq=True)
    import os
    assert os.path.getsize(seq_bam) > 5 * os.path.getsize(bam)
    got = c_oracle.table_dict(ctx.process_bam(seq_bam, caller, jj, w.flags | 4))
    assert ctx.stats()["bam_on_device"] == 1.0
    assert c_oracle.diff_tables(got, want) is None, c_oracle.diff_tables(got, want)


@pytest.mark.parametrize("shape,parts", [("small", 2), ("small", 3), ("c2", 3)])
def test_split_upload_equals_single_upload(ctx, monkeypatch, shape, parts):
    """A big host upload is cut into up to three parts (at chunk granularity, inside a chromosome if need be) so that the
    expansion of one part overlaps the copy of the next; the counting kernels then run once per part into the same
    counters.  SPLISER_SPLIT_MIN_RECORDS forces / forbids the cut, SPLISER_SPLIT_PARTS picks the number of parts."""
    from oracle import c_oracle
    from spliser_b200 import synth
    w = synth.generate(synth.config_small(150_000, seed=71, stranded=True, paired=True) if shape == "small" else synth.config_c2(400_000))
    monkeypatch.setenv("SPLISER_SPLIT_MIN_RECORDS", "1000000000")
    one = c_oracle.table_dict(ctx.process_records(w.records, len(w.chroms), w.junctions, w.flags | 4))
    assert ctx.stats()["n_parts"] == 1.0
    monkeypatch.setenv("SPLISER_SPLIT_MIN_RECORDS", "1000")
    monkeypatch.setenv("SPLISER_SPLIT_PARTS", str(parts))
    two = c_oracle.table_dict(ctx.process_records(w.records, len(w.chroms), w.junctions, w.flags | 4))
    st = ctx.stats()
    assert st["n_parts"] == float(parts) and st["n_aligned"] == len(w.records)
    monkeypatch.delenv("SPLISER_SPLIT_MIN_RECORDS", raising=False)
    monkeypatch.delenv("SPLISER_SPLIT_PARTS", raising=False)
    assert c_oracle.diff_tables(one, two) is None, c_oracle.diff_tables(one, two)
    want = c_oracle.process(w.records, len(w.chroms), w.junctions, w.flags | 4, threads=8)
    assert c_oracle.diff_tables(two, want) is None


def test_bam_ingest_records_longer_than_a_bgzf_member(ctx, tmp_path):
    """A BAM record of ~160 KB (40,000 CIGAR operators) spans three BGZF members, so some members contain no record
    start at all: the chain verification has to skip them, and the device path must still agree with the records path."""
    import numpy as np
    from oracle import c_oracle
    from spliser_b200 import Junctions, Records
    rng = np.random.default_rng(9)
    reads = []
    for i in range(3000):
        p = 1000 + 7 * i
        reads.append(("C", p, 16 * int(rng.integers(0, 2)), "30M%dN40M" % (200 + 10 * (i % 5))))
    long_cigar = "".join("3M1I" for _ in range(20000))                 # 40,000 operators, 60 kb on the reference
    reads.insert(1500, ("C", 1000 + 7 * 1500, 0, long_cigar))
    reads.insert(1501, ("C", 1000 + 7 * 1500, 0, "50M"))
    rec = Records.from_reads(["C"], reads)
    bam = str(tmp_path / "long.bam")
    rec.write_bam(bam, ["C"])
    lefts = sorted({1000 + 7 * i + 29 for i in range(0, 3000, 3)})
    j = Junctions(np.zeros(len(lefts), np.int32), np.array(lefts, np.int32), np.array([l + 200 for l in lefts], np.int32),
                  np.ones(len(lefts), np.int64), np.full(len(lefts), ord("?"), np.uint8))
    want = c_oracle.table_dict(ctx.process_records(rec, 1, j, 0))
    got = c_oracle.table_dict(ctx.process_bam(bam, ["C"], j, 0))
    assert ctx.stats()["bam_on_device"] == 1.0
    assert c_oracle.diff_tables(got, want) is None, c_oracle.diff_tables(got, want)
    assert int(want["beta1"].sum()) > 0


def test_tile_sharded_process_with_record_slices(built_library):
    """One sample sharded by genomic tile the way N GPUs would do it (here sequentially on one): every tile context gets
    only the records spliser_b200.dist.tile_records cuts for it and counts only the sites it owns; the owned slices
    concatenate to the single-context result (SURVEY.md 8(e): no exchange step)."""
    import numpy as np
    import spliser_b200
    from spliser_b200 import api, dist, synth
    w = synth.generate(synth.config_c3_tile(200_000, tile=1))
    nc = len(w.chroms)
    with spliser_b200.Context(0) as full_ctx:
        ref = full_ctx.process_records(w.records, nc, w.junctions, w.flags | 4)
        ref = {k: np.array(getattr(ref, k)) for k in ("beta1", "beta2simple", "beta2cryptic", "sse", "alpha", "pos")}
    table = api.build_site_table(nc, w.junctions, w.flags)
    S = len(table)
    assert np.array_equal(table.pos, ref["pos"])
    span = dist.max_reference_span(w.records)
    n_tiles = 4
    got = {k: np.zeros(S, ref[k].dtype) for k in ("beta1", "beta2simple", "beta2cryptic", "sse")}
    for t in range(n_tiles):
        rec_t = dist.tile_records(w.records, table, nc, t, n_tiles, max_span=span)
        assert 0 < len(rec_t) < len(w.records)
        with spliser_b200.Context(0, tile=(t, n_tiles)) as c:
            part = c.process_records(rec_t, nc, w.junctions, w.flags | 4)
            lo, hi = dist.tile_of(t, n_tiles, S)
            for k in got:
                got[k][lo:hi] = getattr(part, k)[lo:hi]
    for k in got:
        assert np.array_equal(got[k], ref[k]), k


@pytest.mark.parametrize("shape,n_tiles", [("c3_tile", 4), ("c2", 3)])
def test_tiles_with_their_own_graph_concatenate_to_the_untiled_table(built_library, shape, n_tiles):
    """Tile sharding with the site table + competing-site graph built per tile from the junction rows dist.tile_junctions keeps
    (what bench.py --gpus N runs): read-balanced cuts, per-segment span bounds, every column of the concatenated owned rows
    equal to the single-context table AND to the C oracle's."""
    import numpy as np
    import spliser_b200
    from oracle import c_oracle
    from spliser_b200 import api, dist, synth
    w = synth.generate(synth.config_c3_tile(300_000, tile=1) if shape == "c3_tile" else synth.config_c2(400_000))
    nc = len(w.chroms)
    flags = w.flags | 4
    with spliser_b200.Context(0) as full_ctx:
        whole = c_oracle.table_dict(full_ctx.process_records(w.records, nc, w.junctions, flags))
        whole = {k: np.array(v) for k, v in whole.items()}
    table = api.build_site_table(nc, w.junctions, w.flags)
    cuts = dist.balanced_tiles(w.records, table, nc, n_tiles)
    spans = dist.segment_max_spans(w.records)
    parts = []
    for t in range(n_tiles):
        lo, hi = cuts[t], cuts[t + 1]
        rows, junc_t, local = dist.tile_junctions(w.junctions, table, nc, (lo, hi), w.flags)
        rec_t = dist.tile_records(w.records, table, nc, t, n_tiles, site_range=(lo, hi), seg_spans=spans)
        with spliser_b200.Context(0) as c:
            c.set_tile_sites(*local)
            parts.append(dist.owned_part(c.process_records(rec_t, nc, junc_t, flags), local, rows))
    cat = dist.concat_parts(parts, whole)
    assert c_oracle.diff_tables(cat, whole) is None, c_oracle.diff_tables(cat, whole)
    want = c_oracle.process(w.records, nc, w.junctions, flags, threads=8)
    assert c_oracle.diff_tables(cat, want) is None, c_oracle.diff_tables(cat, want)


def test_dirty_strand_regime_at_scale_equals_the_unmodified_reference(ctx):
    """configs[1] shape (500k records, stranded rf) with '?' in every 12th BED row (regtools writes '?' for junctions without an
    XS tag): SURVEY.md 8(a)'s dirty regime -- a '?' row joins whichever same-position site the reference's bisection lands on,
    partner links cross strands, '?' sites never match a read -- at 144k sites, against the whole-table digest of the
    unmodified reference (tests/golden/reference_digests.json) and the C oracle."""
    test_config_shaped_workloads_vs_c_oracle(ctx, "c2_dirty_strands")


def test_full_configs4_equals_the_unmodified_reference(ctx):
    """BASELINE configs[4] at its full size (1M records on the dense alternative-splicing locus, 7.7k sites, --beta2Cryptic: the
    legacy weighted competing-site mode): whole-table digest of the unmodified reference (34 s of its Python for this
    workload; tests/golden/reference_digests.json) and the C oracle."""
    test_config_shaped_workloads_vs_c_oracle(ctx, "c5_full")



def test_junction_extraction_from_the_alignments(ctx, tmp_path):
    """SURVEY 8(f) row 3: the junction table from the records themselves (the `regtools junctions extract` pre-step).  regtools is
    not in the reference tree, so its rules are restated (parity unpinned); here the kernel is pinned to what is known: the
    synthetic generator's own table (anchors >= 8 on both sides, score = supporting records, strand of the gene / '?'), a
    numpy restatement on the same records, hand-made records for every filter, and process on the extracted table."""
    import numpy as np
    from oracle import c_oracle
    from spliser_b200 import Records, synth

    def as_rows(j):
        return sorted(zip(j.chrom.tolist(), j.left.tolist(), j.right.tolist(), j.score.tolist(), [chr(x) for x in j.strand.tolist()]))

    for stranded, paired, seed in ((False, False, 5), (True, True, 6)):
        w = synth.generate(synth.config_small(120_000, seed=seed, stranded=stranded, paired=paired))
        got = ctx.extract_junctions_records(w.records, len(w.chroms), w.flags & 3)
        assert as_rows(got) == as_rows(w.junctions)
        assert [tuple(x) for x in zip(got.chrom.tolist(), got.left.tolist(), got.right.tolist())] == sorted(zip(got.chrom.tolist(), got.left.tolist(), got.right.tolist()))
        # the same through a BAM file, and `process` on the extracted table equals `process` on the generator's table
        bam = str(tmp_path / ("j%d.bam" % seed))
        w.records.write_bam(bam, w.chroms, w.chrom_len)
        assert as_rows(ctx.extract_junctions_bam(bam, w.chroms, w.flags & 3)) == as_rows(w.junctions)
        a = c_oracle.table_dict(ctx.process_records(w.records, len(w.chroms), got, w.flags))
        b = c_oracle.process(w.records, len(w.chroms), w.junctions, w.flags, threads=8)
        for k in ("pos", "alpha", "beta1", "beta2simple", "sse"):
            assert np.array_equal(np.asarray(a[k]), np.asarray(b[k])), k
    # every filter, by hand: anchors (incl. a D inside the stretch and an I that does not count), intron bounds, two junctions in
    # one read sharing the middle stretch, a soft clip that is no anchor, strands from the flags
    reads = [("C", 100, 0, "20M100N20M"), ("C", 100, 16, "20M100N20M"), ("C", 113, 0, "7M100N20M"), ("C", 100, 0, "20M100N7M"),
             ("C", 100, 0, "20M60N20M"), ("C", 100, 0, "20M600000N20M"), ("C", 300, 0, "5M2D4M90N3M1I6M"), ("C", 500, 0, "10M80N6M80N10M"),
             ("C", 700, 0, "10M80N8M80N10M"), ("C", 900, 0, "4S7M100N20M"), ("C", 100, 99, "20M100N20M"), ("C", 100, 147, "20M100N20M")]
    rec = Records.from_reads(["C"], reads)
    got = as_rows(ctx.extract_junctions_records(rec, 1, 0))
    assert got == [(0, 119, 219, 4, "?"), (0, 310, 400, 1, "?"), (0, 709, 789, 1, "?"), (0, 797, 877, 1, "?")], got
    got = as_rows(ctx.extract_junctions_records(rec, 1, 1 | 2))          # --isStranded -s rf
    assert (0, 119, 219, 1, "+") in got and (0, 119, 219, 3, "-") in got, got       # flags 0, 99, 147 read '-' under rf, flag 16 '+' (S:374-406)


def test_bench_dump_outputs_equal_the_reference_arms(tmp_path):
    """`bench.py --dump-outputs DIR` on the CUDA arm writes the table of its last timed resident pass: column for column the
    reference arm's (the C oracle's) for the same arguments."""
    import numpy as np
    from test_dist_cpu import _bench_dump
    ours = _bench_dump(tmp_path, "ours", "--no-bam", "--no-variants", "--no-cpu-baseline")
    ref = _bench_dump(tmp_path, "reference", "--impl", "reference")
    assert sorted(ours) == sorted(ref)
    for k in ref:
        assert ours[k].dtype == np.float64 and np.array_equal(ours[k], ref[k], equal_nan=True), k
    assert len(ref["pos"]) > 500 and ref["sse"].any()
