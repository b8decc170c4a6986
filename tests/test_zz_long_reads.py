"""Long-read and unusual CIGAR shapes against the oracles, on every counting path.

Two inputs feed these tests:
  * oracle.fuzzgen.gen_long_case: small cases (10-40 grid sites, 10-60 junction rows) whose reads walk 5-40 exons with small
    I / D inside the blocks, leading and trailing N / D, zero-length M / N / D, back-to-back N N / N D, clips, flags 256 / 2048,
    junction rows on both strands at one position and hub sites;
  * synth.generate_long_reads: a long-read sample (1-10 kb reads, ~100-255 operators, unspliced reads of 4096 bp and more).
They reach the kernels' special cases that short reads never do: CIGAR words read from global memory when a chunk's operators
do not fit the stage (FC_CIG), hot items of reads with more junctions / blocks than the registers keep (ReadWalk in hot_item,
ReadGlobal in k_junc_complex), pair-site lists longer than CXD_T, hot-queue overflow and the repeated pass, M operators longer
than FC_WALK, zero-length operators, N / D before anything advanced, more than two N among the first operators.  The shape
guards below check from the inputs alone that every one of these is reached, so that a later generator change cannot quietly
stop reaching them.

The unmodified reference is not in the tree, so its answers on these shapes are not pinned.  What the GPU is compared with is
the two independent restatements of checkBam (oracle/spliser_oracle.py and oracle/spliser_oracle.c), which are checked against
each other here first: two restatements that agree are the best evidence available for these shapes.

Collects after the other GPU modules, so that its first run on a B200 cannot stop them under `pytest -x`.
"""
import functools
import os

import numpy as np
import pytest

from common import case_flags, first_diff, gpu_process_rows, oracle_process_rows

SMALL = os.environ.get("SPLISER_SANITIZE_SMALL") == "1"        # under compute-sanitizer: the same kernels on less data
N_CASES = 24 if SMALL else 200
SEED0 = 950000
FC_RECS, FC_CIG, FC_MAXJ, FC_MAXB, CXD_T, FC_WALK = 1024, 4096, 4, 6, 4, 256      # count_fused.cu / device_types.h / kernels.cu
OP_M, OP_N, OP_D, OP_EQ, OP_X = 0, 3, 2, 7, 8
MODES = (1, 3, 0, 1 | 4)                                        # stranded fr, stranded rf, unstranded, fr with --beta2Cryptic


# ---------------------------------------------------------------------------------------------- inputs
def _case(seed):
    from oracle import fuzzgen
    return fuzzgen.gen_long_case(seed, dirty=(seed % 4 == 1))


def _case_inputs(case):
    from spliser_b200 import Records
    from spliser_b200.bed import parse_bed12
    chroms, junc, _ = parse_bed12(case["bed"].splitlines(True))
    return chroms, junc, Records.from_reads(chroms, [tuple(r) for r in case["reads"]])


@functools.lru_cache(maxsize=None)
def _cases():
    return [_case(s) for s in range(SEED0, SEED0 + N_CASES)]


@functools.lru_cache(maxsize=None)
def _case_rows():
    return [oracle_process_rows(c) for c in _cases()]


@functools.lru_cache(maxsize=None)
def _sample(n_records=None):
    from spliser_b200 import synth
    return synth.generate_long_reads(synth.config_long_reads(n_records or (2_000 if SMALL else 12_000)))


@functools.lru_cache(maxsize=None)
def _sample_want(flags, n_records=None):
    from oracle import c_oracle
    w = _sample(n_records)
    return c_oracle.process(w.records, len(w.chroms), w.junctions, flags, threads=8)


def _rows_of(chroms, d):
    """c_oracle / SiteTable dict -> rows in the layout of oracle_process_rows."""
    rows = []
    for i in range(len(d["pos"])):
        p0, p1, c0, c1 = (int(d["partner_off"][i]), int(d["partner_off"][i + 1]), int(d["comp_off"][i]), int(d["comp_off"][i + 1]))
        b = int(d["strand"][i])
        rows.append(dict(chrom=chroms[int(d["chrom"][i])], pos=int(d["pos"][i]), strand=chr(b) if b else "", alpha=int(d["alpha"][i]),
                         beta1=int(d["beta1"][i]), beta2s=int(d["beta2simple"][i]), beta2c=int(d["beta2cryptic"][i]),
                         beta2w=float(d["beta2weighted"][i]).hex(), sse=float(d["sse"][i]).hex(),
                         partners=[[int(p), int(c)] for p, c in zip(d["partner_pos"][p0:p1], d["partner_cnt"][p0:p1])],
                         competitors=[int(c) for c in d["comp_pos"][c0:c1]]))
    return rows


def _ops(rec, i):
    c = rec.cigar[int(rec.cig_off[i]):int(rec.cig_off[i + 1])]
    return c & 15, (c >> 4).astype(np.int64)


# ---------------------------------------------------------------------------------------------- shape guards
def _shape_stats(rec, n_chrom, junc, flags):
    """What the records and the site table make the kernels do (see the module docstring)."""
    from spliser_b200 import api
    t = api.build_site_table(n_chrom, junc, flags)
    first = {}
    for i in range(len(t)):
        first.setdefault((int(t.chrom[i]), int(t.pos[i])), i)
    hot = np.zeros(len(t), bool)                  # first site at its position, and a partner of it has competitors
    for i in range(len(t)):
        if t.comp_off[i + 1] > t.comp_off[i]:
            for p in t.partner_pos[t.partner_off[i]:t.partner_off[i + 1]]:
                j = first.get((int(t.chrom[i]), int(p)))
                if j is not None:
                    hot[j] = True
    # pair sites of a (junction, side): sites t with the anchored end among P_t and the other end among C_t
    pair_sites = {}
    for i in range(len(t)):
        ci, P, C = int(t.chrom[i]), set(t.partners(i)), set(t.competitors(i))
        for a in P:
            for o in C:
                pair_sites[(ci, a, o)] = pair_sites.get((ci, a, o), 0) + 1
    st = dict(chunks=0, big_chunks=0, long_hot_reads=0, zero_len=0, lead_nd=0, many_n_first5=0, long_m=0, max_pair_sites=0,
              max_ops=0, reads=len(rec), n_sites=len(t))
    off = rec.cig_off.astype(np.int64)
    for s in range(len(rec.seg_chrom)):
        a, b = int(rec.seg_off[s]), int(rec.seg_off[s + 1])
        ci = int(rec.seg_chrom[s])
        for lo in range(a, b, FC_RECS):
            hi = min(lo + FC_RECS, b)
            st["chunks"] += 1
            st["big_chunks"] += ((int(off[hi]) - (int(off[lo]) & ~3) + 3) & ~3) > FC_CIG
        for i in range(a, b):
            op, ln = _ops(rec, i)
            st["max_ops"] = max(st["max_ops"], len(op))
            adv = np.isin(op, (OP_M, OP_N, OP_D, OP_EQ, OP_X))
            isM = np.isin(op, (OP_M, OP_EQ, OP_X))
            isN = op == OP_N
            st["zero_len"] += int((adv & (ln == 0)).sum())
            st["long_m"] += int((isM & (ln > FC_WALK)).sum())
            k = np.nonzero(adv)[0]
            st["lead_nd"] += bool(len(k) and op[k[0]] in (OP_N, OP_D))
            st["many_n_first5"] += int(isN[:5].sum()) > 2
            start = int(rec.pos[i]) + np.concatenate([[0], np.cumsum(np.where(adv, ln, 0))[:-1]])
            ends = [(ci, int(x)) for j in np.nonzero(isN)[0] for x in (start[j] - 1, start[j] + ln[j] - 1)]
            if (isN.sum() > FC_MAXJ or isM.sum() > FC_MAXB) and any(e in first and hot[first[e]] for e in ends):
                st["long_hot_reads"] += 1
            for j in np.nonzero(isN)[0]:
                l, r = int(start[j] - 1), int(start[j] + ln[j] - 1)
                st["max_pair_sites"] = max(st["max_pair_sites"], pair_sites.get((ci, l, r), 0), pair_sites.get((ci, r, l), 0))
    return st


def test_long_case_shapes_reach_the_special_paths():
    """gen_long_case reaches, summed over the seeds: reads past FC_MAXJ / FC_MAXB with a junction end on a hot site, zero-length
    operators, N / D before anything advanced, more than two N among the first five operators, M longer than FC_WALK, (junction,
    side) pairs with more than CXD_T pair sites; its chunks are staged (the long-read sample covers the global-memory CIGAR)."""
    tot = {}
    for case in _cases()[:60]:
        chroms, junc, rec = _case_inputs(case)
        st = _shape_stats(rec, len(chroms), junc, case_flags(case))
        for k, v in st.items():
            tot[k] = max(tot.get(k, 0), v) if k.startswith("max_") else tot.get(k, 0) + v
    assert tot["big_chunks"] == 0
    assert tot["long_hot_reads"] >= 200, tot
    assert tot["zero_len"] >= 50 and tot["lead_nd"] >= 20 and tot["many_n_first5"] >= 20, tot
    assert tot["long_m"] >= 1 and tot["max_pair_sites"] > CXD_T, tot


def test_long_read_sample_shapes_reach_the_special_paths():
    """The long-read sample: most 1024-record chunks hold more CIGAR words than a stage (FM_GLOBAL_CIG), thousands of reads past
    FC_MAXJ / FC_MAXB end a junction on a hot site, M operators over FC_WALK and of 4096 bp or more (the compact view's 32-bit
    stream) are common, no record has more operators than the compact view carries, and the hot items the fused kernel queues
    exceed the queue's initial capacity (max(2^18, n_cigar / 16 + 2^16): the first pass overflows)."""
    w = _sample()
    rec = w.records
    st = _shape_stats(rec, len(w.chroms), w.junctions, 1)
    assert st["big_chunks"] >= 0.9 * st["chunks"], st
    assert st["long_hot_reads"] >= 0.5 * len(rec), st
    assert st["long_m"] >= len(rec) and st["max_ops"] <= 255, st
    op, ln = rec.cigar & 15, rec.cigar >> 4
    assert int(((op == OP_M) & (ln >= 4096)).sum()) >= 0.02 * len(rec)
    nN = np.add.reduceat((op == OP_N).astype(np.int64), rec.cig_off[:-1].astype(np.int64))
    assert np.median(nN) >= 10 and np.percentile(nN, 95) >= 30
    if not SMALL:
        assert _hot_items_bound(w) > _hot_cap0(rec), (_hot_items_bound(w), _hot_cap0(rec))


def _hot_cap0(rec):
    return max(2 ** 18, len(rec.cigar) // 16 + 2 ** 16)


def _hot_items_bound(w):
    """Lower bound of the fused kernel's hot items: junction ends of the reads on a hot site (each queues at least one item)."""
    from spliser_b200 import api
    rec = w.records
    t = api.build_site_table(len(w.chroms), w.junctions, 1)
    keys = t.chrom.astype(np.int64) << 32 | t.pos.astype(np.int64)
    first = np.concatenate([[True], keys[1:] != keys[:-1]])
    has_c = np.diff(t.comp_off) > 0
    part_keys = np.repeat(t.chrom.astype(np.int64), np.diff(t.partner_off)) << 32 | t.partner_pos.astype(np.int64)
    hot_keys = np.unique(part_keys[np.repeat(has_c, np.diff(t.partner_off))])
    hot_keys = np.intersect1d(hot_keys, keys[first])
    op, ln = (rec.cigar & 15).astype(np.int64), (rec.cigar >> 4).astype(np.int64)
    adv = np.where(np.isin(op, (OP_M, OP_N, OP_D, OP_EQ, OP_X)), ln, 0)
    nop = np.diff(rec.cig_off.astype(np.int64))
    rid = np.repeat(np.arange(len(rec)), nop)
    cs = np.cumsum(adv) - adv
    start = rec.pos.astype(np.int64)[rid] + cs - cs[rec.cig_off[:-1].astype(np.int64)][rid]
    chrom = np.repeat(np.repeat(rec.seg_chrom.astype(np.int64), np.diff(rec.seg_off)), nop)
    n = op == OP_N
    ends = np.concatenate([chrom[n] << 32 | (start[n] - 1), chrom[n] << 32 | (start[n] + ln[n] - 1)])
    return int(np.isin(ends, hot_keys).sum())


def test_compact_view_takes_255_operators_and_refuses_256():
    from spliser_b200 import CompactRecords, Records
    for n in (255, 254):
        cig = "".join("%dM%dI" % (5 + q % 7, 1 + q % 3) for q in range(n // 2)) + ("5000M" if n % 2 else "")
        rec = Records.from_reads(["C"], [("C", 100, 0, "10M"), ("C", 120, 16, cig), ("C", 130, 0, "3M0N4D2M")])
        assert int(np.diff(rec.cig_off.astype(np.int64)).max()) == n
        back = CompactRecords.from_records(rec).to_records()
        for k in ("pos", "flag", "cig_off", "cigar", "seg_chrom", "seg_off"):
            assert np.array_equal(getattr(back, k), getattr(rec, k)), (n, k)
    rec = Records.from_reads(["C"], [("C", 100, 0, "10M"), ("C", 120, 0, "2M1I" * 128)])
    with pytest.raises(ValueError):
        CompactRecords.from_records(rec)


# ---------------------------------------------------------------------------------------------- oracle vs oracle
def test_c_oracle_equals_python_oracle_on_long_cases():
    """Every column of every row; every final branch of checkBam (S:519-559) fires on these cases."""
    from oracle import c_oracle, spliser_oracle as O
    before = dict(O.BRANCH_HITS)
    _case_rows.cache_clear()
    for case, want in zip(_cases(), _case_rows()):
        chroms, junc, rec = _case_inputs(case)
        got = _rows_of(chroms, c_oracle.process(rec, len(chroms), junc, case_flags(case)))
        d = first_diff(got, want)
        assert d is None, (case["seed"], d)
    assert len(_cases()) >= (24 if SMALL else 200)
    for k, v in O.BRANCH_HITS.items():
        assert v > before[k], (k, before, O.BRANCH_HITS)


def test_c_oracle_equals_python_oracle_on_a_long_read_slice():
    """A few hundred consecutive reads of the long-read sample with the junction rows they reach, every flag mode."""
    from oracle import c_oracle, spliser_oracle as O
    from spliser_b200 import Junctions, Records
    w = _sample()
    r, j = w.records, w.junctions
    a, n = int(r.seg_off[0]) + 400, 250
    rec = Records(r.pos[a:a + n], r.flag[a:a + n], r.cig_off[a:a + n + 1] - r.cig_off[a], r.cigar[int(r.cig_off[a]):int(r.cig_off[a + n])],
                  [int(r.seg_chrom[0])], [0, n])
    lo = int(rec.pos.min()) - 1
    hi = max(int(rec.pos[i]) + int(np.where(np.isin(_ops(rec, i)[0], (OP_M, OP_N, OP_D)), _ops(rec, i)[1], 0).sum()) for i in range(n))
    keep = (j.chrom == int(r.seg_chrom[0])) & (j.left >= lo) & (j.right <= hi)
    sub = Junctions(j.chrom[keep], j.left[keep], j.right[keep], j.score[keep], j.strand[keep])
    assert 100 <= len(sub) <= 1500
    letters = "MIDNSHP=X"
    reads = [(int(rec.pos[i]), int(rec.flag[i]), [(int(x), letters[o]) for o, x in zip(*_ops(rec, i))]) for i in range(n)]
    junc = [(int(c), int(x), int(y), int(s), chr(int(t))) for c, x, y, s, t in zip(sub.chrom, sub.left, sub.right, sub.score, sub.strand)]
    rbc = [[] for _ in w.chroms]
    rbc[int(r.seg_chrom[0])] = reads
    for flags in MODES:
        want = O.rows_from_sites(w.chroms, O.process(len(w.chroms), junc, rbc, flags))
        got = _rows_of(w.chroms, c_oracle.process(rec, len(w.chroms), sub, flags))
        assert first_diff(got, want) is None, (flags, first_diff(got, want))
        assert sum(x["beta1"] for x in want) > 0 and sum(x["beta2s"] for x in want) > 0


# ---------------------------------------------------------------------------------------------- GPU
@pytest.mark.gpu
@pytest.mark.parametrize("variant", ["fused", "stab"])
def test_long_cases_vs_python_oracle(ctx, variant):
    bad = []
    try:
        ctx.set_variant(variant)
        for case, want in zip(_cases(), _case_rows()):
            d = first_diff(gpu_process_rows(ctx, case), want)
            if d:
                bad.append((case["seed"], d))
    finally:
        ctx.set_variant("fused")
    assert not bad, "%d/%d cases differ; first: seed %s %s" % (len(bad), len(_cases()), bad[0][0], bad[0][1])


@pytest.mark.gpu
def test_long_cases_via_bam_vs_python_oracle(ctx, tmp_path):
    for case, want in list(zip(_cases(), _case_rows()))[:60]:
        d = first_diff(gpu_process_rows(ctx, case, via_bam=str(tmp_path)), want)
        assert d is None, (case["seed"], d)


def _check(got_table, flags, what):
    from oracle import c_oracle
    want = _sample_want(flags)
    d = c_oracle.diff_tables(c_oracle.table_dict(got_table), want)
    assert d is None, (what, flags, d)


@pytest.mark.gpu
@pytest.mark.parametrize("variant", ["fused", "stab"])
def test_long_read_sample_process_records(ctx, variant):
    w = _sample()
    try:
        ctx.set_variant(variant)
        for flags in MODES:
            _check(ctx.process_records(w.records, len(w.chroms), w.junctions, flags), flags, variant)
    finally:
        ctx.set_variant("fused")
    want = _sample_want(1)
    assert int(want["beta1"].sum()) > 0 and int(want["beta2simple"].sum()) > 0 and int(_sample_want(1 | 4)["beta2cryptic"].sum()) > 0


@pytest.mark.gpu
def test_long_read_sample_resident_packed_compact_split(ctx, monkeypatch):
    from spliser_b200 import CompactRecords, PackedRecords
    w = _sample()
    nc = len(w.chroms)
    for flags in MODES:
        ctx.resident_load(w.records, nc, w.junctions, flags)
        ctx.resident_count(2)
        _check(ctx.resident_fetch(), flags, "resident")
    pk = PackedRecords.from_records(w.records)
    ck = CompactRecords.from_records(w.records)
    assert len(ck.cigar32) > 0 and len(ck.cigar16) > 0
    for flags in MODES:
        _check(ctx.process_packed(pk, nc, w.junctions, flags), flags, "packed")
        _check(ctx.process_compact(ck, nc, w.junctions, flags), flags, "compact")
    monkeypatch.setenv("SPLISER_SPLIT_MIN_RECORDS", "1000")
    monkeypatch.setenv("SPLISER_SPLIT_PARTS", "3")
    for flags in (1 | 4, 3):
        _check(ctx.process_records(w.records, nc, w.junctions, flags), flags, "split")
        assert ctx.stats()["n_parts"] == 3.0
        _check(ctx.process_compact(ck, nc, w.junctions, flags), flags, "split compact")


@pytest.mark.gpu
def test_long_read_sample_from_a_sequencer_shaped_bam(ctx, tmp_path, monkeypatch):
    w = _sample()
    bam = str(tmp_path / "long.bam")
    w.records.write_bam(bam, w.chroms, w.chrom_len, with_seq=True)
    for flags in (1 | 4, 3):
        monkeypatch.delenv("SPLISER_HOST_BAM", raising=False)
        _check(ctx.process_bam(bam, w.chroms, w.junctions, flags), flags, "bam on the device")
        assert ctx.stats()["bam_on_device"] == 1.0
        monkeypatch.setenv("SPLISER_HOST_BAM", "1")
        _check(ctx.process_bam(bam, w.chroms, w.junctions, flags), flags, "bam on the host")
        assert ctx.stats()["bam_on_device"] == 0.0
    monkeypatch.delenv("SPLISER_HOST_BAM", raising=False)


@pytest.mark.gpu
def test_long_read_sample_recount(ctx):
    """combine's re-count (S:899-904) at every 5th site of the table, with its Partners / Competitors."""
    from oracle import c_oracle
    from spliser_b200 import api
    w = _sample()
    nc = len(w.chroms)
    for flags in MODES:
        t = api.build_site_table(nc, w.junctions, flags)
        gaps = [(int(t.chrom[i]), int(t.pos[i]), t.strand_str(i), sorted(t.partners(i)), t.competitors(i)) for i in range(0, len(t), 5)]
        want1, want2 = c_oracle.recount(w.records, nc, gaps, flags | 8, threads=8)
        got1, got2 = ctx.recount_records(w.records, nc, gaps, flags | 8)
        assert np.array_equal(got1, want1) and np.array_equal(got2, want2), (flags, int(np.sum(got1 != want1)), int(np.sum(got2 != want2)))
        assert int(want1.sum()) > 0 and int(want2.sum()) > 0


@pytest.mark.gpu
def test_long_read_sample_in_four_tiles(built_library):
    """Read-balanced tiles with their own junction rows: reads several kb long cross the cuts; the owned rows concatenate to the
    oracle's table."""
    import spliser_b200
    from oracle import c_oracle
    from spliser_b200 import api, dist
    w = _sample()
    nc = len(w.chroms)
    for flags in (1 | 4, 0):
        want = _sample_want(flags)
        table = api.build_site_table(nc, w.junctions, flags)
        cuts = dist.balanced_tiles(w.records, table, nc, 4)
        spans = dist.segment_max_spans(w.records)
        parts = []
        for t in range(4):
            lo, hi = cuts[t], cuts[t + 1]
            rows, junc_t, local = dist.tile_junctions(w.junctions, table, nc, (lo, hi), flags)
            rec_t = dist.tile_records(w.records, table, nc, t, 4, site_range=(lo, hi), seg_spans=spans)
            with spliser_b200.Context(0) as c:
                c.set_tile_sites(*local)
                parts.append(dist.owned_part(c.process_records(rec_t, nc, junc_t, flags), local, rows))
        cat = dist.concat_parts(parts, want)
        assert c_oracle.diff_tables(cat, want) is None, (flags, c_oracle.diff_tables(cat, want))


@pytest.fixture
def fresh_ctx(built_library):
    """A context of its own: the session context's hot queue may have grown already, and a grown queue never overflows."""
    import spliser_b200
    c = spliser_b200.Context(0)
    yield c
    c.close()


@pytest.mark.gpu
def test_hot_queue_overflow_repeats_the_process_pass(fresh_ctx):
    """More hot (record, operator, side) items than the queue's initial capacity: the pass is repeated with a grown queue and
    the table is the oracle's; a second call on the grown queue gives the same table."""
    w = _sample(12_000)
    cap0 = _hot_cap0(w.records)
    for attempt in range(2):
        t = fresh_ctx.process_records(w.records, len(w.chroms), w.junctions, 1 | 4)
        n = fresh_ctx.stats()["n_hot_items"]
        assert n > cap0, (attempt, n, cap0)
        print("process call %d: n_hot_items %d, initial capacity %d" % (attempt, n, cap0))
        from oracle import c_oracle
        d = c_oracle.diff_tables(c_oracle.table_dict(t), _sample_want(1 | 4, 12_000))
        assert d is None, (attempt, d)


@pytest.mark.gpu
def test_hot_queue_overflow_repeats_the_resident_pass(fresh_ctx):
    """The same overflow on the resident path, whose retry loop is separate code."""
    from oracle import c_oracle
    w = _sample(12_000)
    cap0 = _hot_cap0(w.records)
    fresh_ctx.resident_load(w.records, len(w.chroms), w.junctions, 3)
    for attempt in range(2):
        st = fresh_ctx.resident_count(2)
        assert st["n_hot_items"] > cap0, (attempt, st["n_hot_items"], cap0)
        print("resident pass %d: n_hot_items %d, initial capacity %d" % (attempt, st["n_hot_items"], cap0))
        d = c_oracle.diff_tables(c_oracle.table_dict(fresh_ctx.resident_fetch()), _sample_want(3, 12_000))
        assert d is None, (attempt, d)
