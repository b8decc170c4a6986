"""SpliSER-compatible command line: `process` and `combine` with the reference's flags and byte-identical
.SpliSER.tsv / .combined.tsv output, the counting done by libspliser_b200.so on the GPU.

    python -m spliser_b200.cli process -B x.bam -b x.bed -o out [-A genes.gff] [-c chr] [-g gene -m 500000]
                                       [--isStranded -s rf|fr] [--beta2Cryptic]
    python -m spliser_b200.cli combine -S samples.tsv -o out [-g gene] [--isStranded -s rf|fr] [--beta2Cryptic]

Without regtools (not a reference command; regtools' option letters):
    python -m spliser_b200.cli junctions -B x.bam -o x.bed [-a 8] [-m 70] [-M 500000] [--isStranded -s rf|fr | --strandFromXS]
    python -m spliser_b200.cli processBam -B x.bam -o out [process's -A -t -c -g -m --isStranded -s rf|fr|auto --beta2Cryptic]
                                          [--minAnchor 8] [--minIntron 70] [--maxIntron 500000] [--strandFromXS]
    python -m spliser_b200.cli combineBam -S samples.tsv -o out [-A genes.gff] [-t gene] [-g gene] [--isStranded -s rf|fr|auto]
                                          [--beta2Cryptic] [--minAnchor 8] [--minIntron 70] [--maxIntron 500000] [--strandFromXS]
                                          [--shallow [-m 0] [-r 10] [-e 0.0]] [--gpus N]
    python -m spliser_b200.cli inferStrandedness -B x.bam [-A genes.gff]
    python -m spliser_b200.cli combineGroups -B x.bam --tag CB -G groups.tsv -o out [combineBam's -A -t -g --isStranded -s
                                          --beta2Cryptic --minAnchor --minIntron --maxIntron --strandFromXS --shallow -m -r -e --gpus]
Every command that reads a BAM also takes [--minMAPQ N] [--excludeFlags F] [--requireFlags F], samtools view's -q / -F / -f
applied as the BAM is ingested (flags in decimal or 0x hex; include/spliser_b200.h, spl_read_filter, states the rule).
`junctions` writes the junction BED12 that `regtools junctions extract` would feed `process` with; `processBam` is
`junctions` followed by `process -b` in one call that reads the BAM once, and writes the same .SpliSER.tsv.  --strandFromXS
takes the junction strands from the aligner's XS tag, as regtools does for unstranded libraries; processBam still counts
with --isStranded -s.  `combineBam` is `processBam` for every sample of a samples file (writing its column 2) followed by
`combine` (`combineShallow` with --shallow), with every BAM read once: the records stay in GPU memory for the re-count.
`inferStrandedness` tells which of --isStranded -s fr, -s rf or an unstranded run fits the library (one vote per record,
against the annotation's genes or the XS tag); `processBam` and `combineBam` take --isStranded -s auto to infer it over the
same ingest and run with its verdict.  `combineGroups` is `combineBam` over the groups of one BAM that an aux tag tells apart
(read groups, cell-barcode clusters, haplotypes), split on the GPU from one ingest instead of one BAM per group.

What stays in Python is what the reference does in text: BED12 parsing and its filters (S:255-288), the
annotation and gene lookup (S:50-173), the TSV writers (S:641-664, S:722-740) and the lock-step merge of
`combine` (S:742-917).  The body of `process` (S:710-717) is one spl_process call; every checkBam call of
`combine` (S:903) goes into one batched spl_recount call per sample.
"""
from __future__ import annotations

import argparse
import functools
import sys
import timeit

import numpy as np

from . import api
from .bed import StrandColumn, parse_bed12, write_junctions_bed
from .dist import samples_of
from .genes import load_annotation
from .hosttext import CombineMerge, write_process_tsv as _native_write_process_tsv

VERSION = "v0.1.8 (spliser_b200)"


# ------------------------------------------------------------------------------------------------ read filter
def _with_filter(ctx, read_filter):
    """ctx under the command's read filter (api.ReadFilter, or None: the context is left as it is)."""
    if read_filter is not None:
        ctx.set_read_filter(read_filter)
    return ctx


def _report_filter(ctx, bam, read_filter):
    """With a read filter, the one line per BAM: the records its ingest kept and the records the filter dropped."""
    if read_filter is not None:
        kept, dropped = ctx.last_read_filter()
        print("Read filter {}:\tkept {}\tdropped {}".format(bam, kept, dropped))


# ------------------------------------------------------------------------------------------------ process
def _append_bed_chroms(annotation, bed_chroms, junc):
    """Chromosome index of a BED12 parsed on its own -> the reference's index: the annotation's names first (S:90-92), then
    the BED's names not among them in their order of first appearance (S:265-268); the junction table is renumbered."""
    chroms = list(annotation.chrom_index)
    at = {c: i for i, c in enumerate(chroms)}
    remap = np.zeros(max(1, len(bed_chroms)), dtype=np.int32)
    for i, c in enumerate(bed_chroms):
        if c not in at:
            at[c] = len(chroms)
            chroms.append(c)
        remap[i] = at[c]
    return chroms, api.Junctions(remap[junc.chrom], junc.left, junc.right, junc.score, junc.strand)


def process_table(ctx, bam_path, bed_lines, *, annotation=None, qchrom="All", qgene="All", max_intron=0,
                  is_stranded=False, stranded_type=None, beta2_cryptic=False, records=None, parsed_bed=None):
    """Steps 1-3 of process() (S:710-717).  Returns (chrom_index, SiteTable, strand strings per junction row).
    parsed_bed: (chroms, Junctions, strand column) of the same BED12 already parsed WITHOUT an annotation (process() does
    that while the annotation loads); only valid without -g, whose window needs the gene first."""
    chrom_index = list(annotation.chrom_index) if annotation is not None else []
    bounds = None
    if qgene != "All":
        q = annotation.query_gene if annotation is not None else None
        if q is None:                           # S:283: QUERY_gene is None -> AttributeError in the reference
            raise AttributeError("'NoneType' object has no attribute 'getLeftPos'")
        bounds = (q.left, q.right)
    if parsed_bed is not None and bounds is None:
        chroms, junc, sstr = parsed_bed
        if annotation is not None:
            chroms, junc = _append_bed_chroms(annotation, chroms, junc)
    else:
        chroms, junc, sstr = parse_bed12(bed_lines, chrom_index, qchrom, bounds, int(max_intron))
    flags = api.mode_flags(is_stranded, stranded_type, beta2_cryptic)
    if records is not None:
        table = ctx.process_records(records, len(chroms), junc, flags)
    else:
        table = ctx.process_bam(bam_path, chroms, junc, flags)
    return chroms, table, sstr


def write_process_tsv(path, chroms, table, sstr, *, annotation=None, is_stranded=False, beta2_cryptic=False):
    """outputBedFile (S:641-664) with the Gene column of S:313-329: native (csrc/host_text.cpp), one call for the table."""
    _native_write_process_tsv(path, chroms, table, sstr, annotation=annotation, is_stranded=is_stranded,
                              beta2_cryptic=beta2_cryptic)


def process(inBAM, inBed, outputPath, qGene="All", qChrom="All", maxIntronSize=0, annotationFile=None, aType="gene",
            isStranded=False, strandedType=None, isbeta2Cryptic=False, ctx=None, read_filter=None):
    print("Processing")
    print("Stranded Analysis {}".format(strandedType) if isStranded else "Unstranded Analysis")
    parsed_bed = None
    if annotationFile is not None and qGene == "All":
        # without -g the annotation and the BED12 do not depend on each other: both parse at the same time (native code,
        # the GIL is released) and the BED's chromosome numbers are appended to the annotation's afterwards.  The
        # annotation is loaded on this thread, so its errors still come first, as in the reference (S:703-711).
        from concurrent.futures import ThreadPoolExecutor

        def bed_alone():
            with open(inBed) as fh:
                return parse_bed12(fh, None, qChrom, None, 0)
        with ThreadPoolExecutor(max_workers=1) as pool:
            fut = pool.submit(bed_alone)
            annotation = load_annotation(annotationFile, qGene)
            parsed_bed = fut.result()
    else:
        annotation = load_annotation(annotationFile, qGene) if annotationFile is not None else None
    own = ctx is None
    ctx = ctx or api.Context(0)
    try:
        _with_filter(ctx, read_filter)
        with open(inBed) as fh:
            chroms, table, sstr = process_table(ctx, inBAM, fh, annotation=annotation, qchrom=qChrom, qgene=qGene,
                                                max_intron=maxIntronSize, is_stranded=isStranded, stranded_type=strandedType,
                                                beta2_cryptic=isbeta2Cryptic, parsed_bed=parsed_bed)
        _report_filter(ctx, inBAM, read_filter)
    finally:
        if own:
            ctx.close()
    print("Sites:\t\t\t" + str(len(table)))
    write_process_tsv(outputPath + ".SpliSER.tsv", chroms, table, sstr, annotation=annotation, is_stranded=isStranded,
                      beta2_cryptic=isbeta2Cryptic)


# ------------------------------------------------------------------------------------------------ without regtools
def junctions(inBAM, outBed, minAnchor=8, minIntron=70, maxIntron=500000, isStranded=False, strandedType=None, strandFromXS=False,
              ctx=None, read_filter=None):
    """The `regtools junctions extract -a -m -M` step on the GPU: the junction table of every header reference, written as
    BED12 in regtools' layout (chromStart / chromEnd from the longest anchors).  Strands: with strandFromXS the record's XS tag
    ('?' without one; include/spliser_b200.h, SPL_FLAG_XS_STRAND), else '?' unstranded, else the strand check_strand derives
    from the FLAG (S:374-406)."""
    chroms = api.bam_reference_names(inBAM)
    flags = api.FLAG_XS_STRAND if strandFromXS else api.mode_flags(isStranded, strandedType)
    own = ctx is None
    ctx = ctx or api.Context(0)
    try:
        junc = _with_filter(ctx, read_filter).extract_junctions_bam(inBAM, chroms, flags, minAnchor, minIntron, maxIntron)
        _report_filter(ctx, inBAM, read_filter)
    finally:
        if own:
            ctx.close()
    print("Junctions:\t\t" + str(len(junc)))
    write_junctions_bed(outBed, chroms, junc)


def _strand_column(junc):
    """Column 6 of the BED12 `junctions` writes for these rows, as parse_bed12 would return it."""
    texts, lut = [], np.zeros(256, dtype=np.int32)
    for b in dict.fromkeys(junc.strand.tolist()):            # distinct bytes in first-appearance order
        lut[b] = len(texts)
        texts.append(chr(b) if b else "")
    return StrandColumn(texts, lut[junc.strand])


def processBam(inBAM, outputPath, qGene="All", qChrom="All", maxIntronSize=0, annotationFile=None, aType="gene", isStranded=False,
               strandedType=None, isbeta2Cryptic=False, minAnchor=8, minIntron=70, maxIntron=500000, strandFromXS=False, ctx=None,
               read_filter=None):
    """`junctions` + `process -b` in one GPU call that ingests the BAM once (spl_process_bam_extract).  The chromosome list is
    the annotation's names, then the header's references not among them in header order: the relative order `process` gets
    from a BED12 written by `junctions`, so the .SpliSER.tsv is the same byte for byte.  strandFromXS: the table's strands come
    from the XS tag (`junctions --strandFromXS`); the count still follows isStranded / strandedType.

    isStranded with strandedType 'auto': the library type is inferred first (inferStrandedness: votes from every gene of the
    annotation, or from the XS tag without one) over the same ingest -- the BAM is loaded into GPU memory once, voted on and
    counted from there (a BAM the device cannot hold is read twice: votes, then the count) -- and the run is the one the verdict's
    flags give.  An undecided verdict raises StrandednessError before anything is written."""
    print("Processing")
    auto = isStranded and strandedType == "auto"
    if not auto:
        print("Stranded Analysis {}".format(strandedType) if isStranded else "Unstranded Analysis")
    annotation = load_annotation(annotationFile, qGene) if annotationFile is not None else None
    bounds = None
    if qGene != "All":
        q = annotation.query_gene if annotation is not None else None
        if q is None:                           # S:283, as in process
            raise AttributeError("'NoneType' object has no attribute 'getLeftPos'")
        bounds = (q.left, q.right)
    own = ctx is None
    ctx = ctx or api.Context(0)
    sample = None
    try:
        _with_filter(ctx, read_filter)
        extract = functools.partial(ctx.process_bam_extract, inBAM)
        if auto:
            chroms = _chrom_list(annotation, inBAM)
            genes = None
            if annotationFile is not None:
                genes = api.gene_strands(annotation if qGene == "All" else load_annotation(annotationFile, "All"), chroms)
            try:
                sample = ctx.load_bam(inBAM, xs=genes is None or strandFromXS)
                extract = sample.process_extract
                votes = sample.infer_strand(chroms, genes)
            except api.SampleMemoryError:
                votes = ctx.infer_strand_bam(inBAM, chroms, genes)
            _report_filter(ctx, inBAM, read_filter)
            isStranded, strandedType = _verdict_flags(votes, inBAM)
            print("Stranded Analysis {}".format(strandedType) if isStranded else "Unstranded Analysis")
        _process_bam_sample(extract, inBAM, outputPath + ".SpliSER.tsv", annotation, bounds, qChrom, maxIntronSize, isStranded,
                            strandedType, isbeta2Cryptic, minAnchor, minIntron, maxIntron, strandFromXS)
        if not auto:
            _report_filter(ctx, inBAM, read_filter)
    finally:
        if sample is not None:
            sample.close()
        if own:
            ctx.close()


def _chrom_list(annotation, inBAM):
    """processBam's chromosome list: the annotation's names, then the header's references not among them in header order."""
    chroms = list(annotation.chrom_index) if annotation is not None else []
    known = set(chroms)
    return chroms + [c for c in api.bam_reference_names(inBAM) if c not in known]


def _process_bam_sample(extract, inBAM, tsv_path, annotation, bounds, qChrom, maxIntronSize, isStranded, strandedType, isbeta2Cryptic,
                        minAnchor, minIntron, maxIntron, strandFromXS, chroms=None):
    """processBam after the annotation load.  extract(chrom_names, flags, min_anchor, min_intron, max_intron, qchrom=, gene_bounds=,
    window_max_intron=) answers like Context.process_bam_extract of this BAM (or DeviceSample.process_extract of it loaded).
    chroms: _chrom_list(annotation, inBAM) when the caller has it already."""
    chroms = _chrom_list(annotation, inBAM) if chroms is None else chroms
    flags = api.mode_flags(isStranded, strandedType, isbeta2Cryptic) | (api.FLAG_XS_STRAND if strandFromXS else 0)
    junc, table = extract(chroms, flags, minAnchor, minIntron, maxIntron, qchrom=qChrom, gene_bounds=bounds,
                          window_max_intron=int(maxIntronSize))
    print("Sites:\t\t\t" + str(len(table)))
    write_process_tsv(tsv_path, chroms, table, _strand_column(junc), annotation=annotation, is_stranded=isStranded,
                      beta2_cryptic=isbeta2Cryptic)


# ------------------------------------------------------------------------------------------------ library strandedness
class StrandednessError(ValueError):
    """-s auto could not settle the library type: too few votes, a share between the thresholds, or samples that disagree."""


_FLAGS_OF = {"fr": "--isStranded -s fr", "rf": "--isStranded -s rf", "unstranded": "no --isStranded (unstranded)"}


def _strand_report(votes):
    """The lines every command that infers prints: the counts, f, the thresholds and the verdict as the flags to pass."""
    v = votes.agree_fr + votes.opposite
    verdict = api.library_type(votes)
    return verdict, [
        "Strand votes (one per record):\tagree with fr {}\topposite {}\tno vote {}".format(votes.agree_fr, votes.opposite, votes.no_vote),
        "f = agree / (agree + opposite):\t" + ("{:.4f}".format(votes.agree_fr / v) if v else "n/a"),
        "Thresholds:\t\t\tat least {} votes; fr when f >= {}, rf when f <= {}, unstranded when {} <= f <= {}".format(
            api.MIN_VOTES, api.FR_MIN, api.RF_MAX, *api.UNSTRANDED_RANGE),
        "Library type:\t\t\t" + (verdict + ": " + _FLAGS_OF[verdict] if verdict else "undecided")]


def _verdict_flags(votes, what):
    """Prints the report; (isStranded, strandedType) of the verdict, or StrandednessError when it is undecided."""
    verdict, lines = _strand_report(votes)
    print("\n".join(lines))
    if verdict is None:
        raise StrandednessError("the library type of %s is undecided: pass --isStranded -s fr|rf, or nothing for an unstranded run"
                                % what)
    return (False, None) if verdict == "unstranded" else (True, verdict)


def inferStrandedness(inBAM, annotationFile=None, ctx=None, read_filter=None):
    """The library's protocol from the BAM (one vote per record; include/spliser_b200.h, spl_gene_strands, states the rule): the
    reference strand from every gene of the annotation, or from the aligner's XS tag without one.  Prints the counts, f, the
    thresholds and the verdict as the flags to pass; returns (verdict, StrandVotes) and raises StrandednessError when it is
    undecided."""
    chroms = api.bam_reference_names(inBAM)
    genes = api.gene_strands(load_annotation(annotationFile, "All"), chroms) if annotationFile is not None else None
    own = ctx is None
    ctx = ctx or api.Context(0)
    try:
        votes = _with_filter(ctx, read_filter).infer_strand_bam(inBAM, chroms, genes)
        _report_filter(ctx, inBAM, read_filter)
    finally:
        if own:
            ctx.close()
    _verdict_flags(votes, inBAM)
    return api.library_type(votes), votes


# ------------------------------------------------------------------------------------------------ combine
def _chrom_order(runs_per_file):
    """Region order across files: the reference builds a before/after graph and sorts it topologically
    (S:761-789, Graph in Gene_Site_Iter_Graph_v0_1_8.py:358-396).  runs_per_file: for every sample file the consecutive
    distinct regions of its rows (all the reference's scan looks at)."""
    all_chroms, before_list, after_list = [], [], []
    for runs in runs_per_file:
        before = "-1"
        for chrom in runs:
            if chrom != before:
                before_list.append(before)
                after_list.append(chrom)
                before = chrom
                if chrom not in all_chroms:
                    all_chroms.insert(0, chrom)
    if not all_chroms:
        print("No genomic regions found - EXITING")
        sys.exit()
    all_chroms.insert(0, "-1")
    graph = {}
    for b, a in zip(before_list, after_list):
        lst = graph.setdefault(b, [])
        if a not in lst:
            lst.append(a)
    visited = [False] * len(all_chroms)
    stack = []

    def visit(region):
        visited[all_chroms.index(region)] = True
        for nxt in graph.get(region, []):
            if not visited[all_chroms.index(nxt)]:
                visit(nxt)
        stack.insert(0, region)

    sys.setrecursionlimit(max(sys.getrecursionlimit(), len(all_chroms) + 1000))
    for i, region in enumerate(all_chroms):
        if not visited[i]:
            visit(region)
    return stack[1:]


def _recount_sample(ctx, cm, k, regions, recount):
    """Every S:903 call of sample k in one recount(ctx, k, chrom_names, gaps) -> (beta1, beta2simple) call (one spl_recount);
    returns False when the sample has no gaps."""
    gaps = cm.gaps(k)
    if not len(gaps):
        return False
    uniq, first = np.unique(gaps.chrom, return_index=True)
    local = uniq[np.argsort(first)]                 # the sample's gap regions in first-appearance order
    names = [regions[r] for r in local]
    remap = np.full(len(regions), -1, dtype=np.int32)
    remap[local] = np.arange(len(local), dtype=np.int32)
    gaps.chrom = np.ascontiguousarray(remap[gaps.chrom])
    b1, b2 = recount(ctx, k, names, gaps)
    cm.set_recount(k, b1, b2)
    return True


def _read_samples_file(samplesFile, shallow):
    """(titles, tsv paths, BAM paths) of a samples file: a line without exactly three columns raises in `combine` and is
    skipped by `combineShallow` (S:930-935)."""
    titles, bed_paths, bam_paths = [], [], []
    with open(samplesFile) as fh:
        for line in fh:
            values = line.split("\t")
            if len(values) == 3:
                titles.append(values[0]); bed_paths.append(values[1]); bam_paths.append(values[2].rstrip())
            elif not shallow:
                print(str(titles), str(bed_paths), str(bam_paths))
                raise Exception("Samples File contains lines that do not have exactly 3 tab-separated columns")
    return titles, bed_paths, bam_paths


def _on_ranks(n_ranks, work):
    """work(rank) for every rank, each on a host thread of its own (the calling thread when there is one rank)."""
    if n_ranks == 1:
        work(0)
        return
    from concurrent.futures import ThreadPoolExecutor
    with ThreadPoolExecutor(max_workers=n_ranks) as pool:
        list(pool.map(work, range(n_ranks)))


def _merge_recount_write(titles, tsv_paths, outputPath, qGene, isStranded, isbeta2Cryptic, shallow, n_ranks, rank_ctx, recount):
    """The merge of `combine` (or combineShallow's, shallow = (minSamples, minReads, minSSE)) over the sample tables in
    samples-file order, the re-count of every sample's gaps, the .combined.tsv.  The re-count shards by sample: rank r takes
    dist.samples_of(r, n_ranks, n) on a host thread of its own (the calling thread when n_ranks == 1) with the context
    rank_ctx(r), asked for once the rank meets its first sample with gaps; recount(ctx, k, chrom_names, gaps) -> (beta1,
    beta2simple) counts sample k."""
    n = len(titles)
    with CombineMerge() as cm:
        cm.add_samples(titles, tsv_paths)
        regions = cm.region_names()
        order = _chrom_order([[regions[r] for r in cm.sample_runs(k)] for k in range(n)])
        region_id = {name: i for i, name in enumerate(regions)}
        if shallow is None:
            cm.merge([region_id[name] for name in order], qGene, isStranded)
        else:
            cm.merge_shallow([region_id[name] for name in order], qGene, isStranded, *shallow)

        def rank_work(rank):
            ctx = None
            for k in samples_of(rank, n_ranks, n):
                if cm.n_gaps(k):
                    ctx = ctx or rank_ctx(rank)
                    _recount_sample(ctx, cm, k, regions, recount)
        _on_ranks(n_ranks, rank_work)
        cm.write(outputPath + ".combined.tsv", isbeta2Cryptic)
        filled = cm.n_filled()
    print("Filled in Beta read counts for {} Sites not detected in some samples".format(filled))


def combineShallow(samplesFile, outputPath, qGene="All", isStranded=False, minSamples=0, minReads=10, minSSE=0.0, strandedType=None,
                   isbeta2Cryptic=False, ctx=None, records_by_bam=None, devices=None, context_factory=None, read_filter=None):
    """combineShallow (S:920-1167): `combine` for many shallow samples.  The same lock-step merge and the same re-count of the
    sites a sample lacks (checkBam at S:1145 -> one spl_recount call per sample), with three filters on which positions are
    kept at all -- a position needs at least `minSamples` samples showing it with alpha + beta1 + beta2Simple >= `minReads`
    and SSE >= `minSSE` (S:1066-1084, S:1108) -- and, with -g, only the rows of that gene loaded from every table
    (S:947-956).  The quirks of the reference's loop are kept (csrc/host_text.cpp, merge_impl): the count runs over the rows
    of both strands of a position, and a dropped position moves every sample on whose current row has that position number,
    whatever its region or strand (S:1158-1160).  Unlike `combine`, a samples-file line without exactly three columns is
    skipped silently (S:930-935)."""
    return combine(samplesFile, outputPath, qGene, isStranded, strandedType, isbeta2Cryptic, ctx, records_by_bam, devices,
                   context_factory, _shallow=(minSamples, minReads, minSSE), read_filter=read_filter)


def combine(samplesFile, outputPath, qGene="All", isStranded=False, strandedType="fr", isbeta2Cryptic=False, ctx=None,
            records_by_bam=None, devices=None, context_factory=None, _shallow=None, read_filter=None):
    """combine (S:742-917).  The native merge driver (csrc/host_text.cpp) parses the sample tables and replays the
    lock-step merge, collecting per sample the sites it lacks together with the partner / competitor / strand context
    gathered from lower-indexed samples only (the reference's order dependence, SURVEY.md F7); one spl_recount call
    per sample fills them; the driver then writes the rows.

    The re-count shards by sample (SURVEY.md 8(e)): with `devices` = several CUDA ordinals, one context per device runs on
    its own host thread and takes the samples dist.samples_of(rank, n_devices, n_samples); a sample's result depends on
    nothing but its own BAM and gap list, so the host only collects the count arrays.  `ctx` (one existing context) takes
    precedence; `context_factory(device)` replaces api.Context (tests).  read_filter (api.ReadFilter) applies to every
    context the re-count uses."""
    print("Combining samples...")
    titles, bed_paths, bam_paths = _read_samples_file(samplesFile, _shallow is not None)
    flags = api.mode_flags(isStranded, strandedType, False, combine=True)

    def recount(c, k, names, gaps):
        if records_by_bam is not None:
            return c.recount_records(records_by_bam(bam_paths[k], names), len(names), gaps, flags)
        got = c.recount_bam(bam_paths[k], names, gaps, flags)
        _report_filter(c, bam_paths[k], read_filter)
        return got
    make = context_factory or api.Context
    devs = [0] if not devices else list(devices)
    n_ranks = 1 if ctx is not None else len(devs)
    made = []

    def rank_ctx(rank):                             # one context per device, made when its rank first needs it
        if ctx is not None:
            return _with_filter(ctx, read_filter)
        made.append(make(devs[rank]))
        return _with_filter(made[-1], read_filter)
    try:
        _merge_recount_write(titles, bed_paths, outputPath, qGene, isStranded, isbeta2Cryptic, _shallow, n_ranks, rank_ctx, recount)
    finally:
        for c in made:
            c.close()


def combineBam(samplesFile, outputPath, annotationFile=None, aType="gene", qGene="All", isStranded=False, strandedType=None,
               isbeta2Cryptic=False, minAnchor=8, minIntron=70, maxIntron=500000, strandFromXS=False, shallow=False, minSamples=0,
               minReads=10, minSSE=0.0, devices=None, context_factory=None, read_filter=None):
    """`processBam` for every sample of a samples file, then `combine` (or, with shallow, `combineShallow -m -r -e`) over them,
    reading every BAM once.  Column 2 of the samples file is where the sample's .SpliSER.tsv is written: the file `processBam -B
    <column 3>` writes with the same -A / --isStranded -s / --beta2Cryptic / --minAnchor --minIntron --maxIntron / --strandFromXS
    and without -c / -g.  The .combined.tsv is the one `combine -g qGene` (`combineShallow`) writes from those files.

    One context per device in `devices` (context_factory(device) replaces api.Context), each on a host thread of its own with the
    samples dist.samples_of(rank, n_devices, n_samples) in both GPU phases: a sample is loaded into its rank's GPU memory
    (Context.load_bam), its table extracted and counted from there, and after the merge its gaps are re-counted from there.  A
    sample the device cannot hold (SampleMemoryError) takes the path route -- process_bam_extract, then recount_bam -- with the
    same output.

    isStranded with strandedType 'auto': every rank loads its samples and votes on each (inferStrandedness's rule) before any
    extraction; the verdict is taken on the pooled votes and is refused (StrandednessError, nothing written) when it is undecided
    or when a sample's own decided verdict differs from it.  The run is then the one the verdict's flags give.

    read_filter (api.ReadFilter) applies to every rank's context: the samples are loaded, voted on and counted under it."""
    print("Combining samples from their BAMs...")
    titles, tsv_paths, bam_paths = _read_samples_file(samplesFile, shallow)
    annotation = load_annotation(annotationFile, "All") if annotationFile is not None else None

    def load(rank, c, k, xs):
        try:
            s = c.load_bam(bam_paths[k], xs=xs)
        except api.SampleMemoryError:
            return None
        _report_filter(c, bam_paths[k], read_filter)
        return s
    _combine_resident(titles, tsv_paths, bam_paths, outputPath, annotation, qGene, isStranded, strandedType, isbeta2Cryptic, minAnchor,
                      minIntron, maxIntron, strandFromXS, shallow, minSamples, minReads, minSSE, devices, context_factory, read_filter, load)


def _combine_resident(titles, tsv_paths, bam_paths, outputPath, annotation, qGene, isStranded, strandedType, isbeta2Cryptic, minAnchor,
                      minIntron, maxIntron, strandFromXS, shallow, minSamples, minReads, minSSE, devices, context_factory, read_filter,
                      load):
    """combineBam's orchestration over samples that are held in GPU memory: load(rank, ctx, k, xs) -> the DeviceSample of sample
    k on that rank's context, or None for the path route (process_bam_extract / recount_bam on bam_paths[k]).  The samples of
    rank r are dist.samples_of(r, n_ranks, n), asked for in order on the rank's host thread."""
    n = len(titles)
    make = context_factory or api.Context
    devs = [0] if not devices else list(devices)
    n_ranks = len(devs)
    ctxs = [None] * n_ranks
    resident = [None] * n                           # DeviceSample, or None: the path route
    auto = isStranded and strandedType == "auto"
    votes = [None] * n
    flags = None if auto else api.mode_flags(isStranded, strandedType, False, combine=True)
    chrom_lists = {}

    def chroms_of(k):                               # the header is read once per BAM (combineGroups: one BAM for every sample)
        if bam_paths[k] not in chrom_lists:
            chrom_lists[bam_paths[k]] = _chrom_list(annotation, bam_paths[k])
        return chrom_lists[bam_paths[k]]

    def extract(rank, k):
        c = ctxs[rank]
        ex = resident[k].process_extract if resident[k] is not None else functools.partial(c.process_bam_extract, bam_paths[k])
        _process_bam_sample(ex, bam_paths[k], tsv_paths[k], annotation, None, "All", 0, isStranded, strandedType, isbeta2Cryptic,
                            minAnchor, minIntron, maxIntron, strandFromXS, chroms_of(k))

    def process_rank(rank):
        mine = samples_of(rank, n_ranks, n)
        if not mine:
            return
        ctxs[rank] = c = _with_filter(make(devs[rank]), read_filter)
        for k in mine:
            genes = None
            if auto:
                chroms = chroms_of(k)
                genes = api.gene_strands(annotation, chroms) if annotation is not None else None
            resident[k] = load(rank, c, k, strandFromXS or (auto and annotation is None))
            if not auto:
                extract(rank, k)
            elif resident[k] is not None:
                votes[k] = resident[k].infer_strand(chroms, genes)
            else:
                votes[k] = c.infer_strand_bam(bam_paths[k], chroms, genes)
            if resident[k] is None:                 # the path route's first ingest of the BAM
                _report_filter(c, bam_paths[k], read_filter)

    def extract_rank(rank):
        for k in samples_of(rank, n_ranks, n):
            extract(rank, k)

    def recount(c, k, names, gaps):
        s, resident[k] = resident[k], None
        if s is None:
            return c.recount_bam(bam_paths[k], names, gaps, flags)     # the same BAM and filter again: no second report
        with s:
            return s.recount(names, gaps, flags)
    try:
        _on_ranks(n_ranks, process_rank)
        if auto:
            # with -s auto every sample is loaded and voted on first; the extraction then runs with the pooled verdict's flags
            isStranded, strandedType = _pooled_verdict(titles, votes)
            flags = api.mode_flags(isStranded, strandedType, False, combine=True)
            _on_ranks(n_ranks, extract_rank)
        _merge_recount_write(titles, tsv_paths, outputPath, qGene, isStranded, isbeta2Cryptic,
                             (minSamples, minReads, minSSE) if shallow else None, n_ranks, lambda rank: ctxs[rank], recount)
    finally:
        for s in resident:
            if s is not None:
                s.close()
        for c in ctxs:
            if c is not None:
                c.close()


def _pooled_verdict(titles, votes):
    """combineBam -s auto: the verdict on the votes of all samples together; StrandednessError when it is undecided or when a
    sample's own decided verdict differs from it (the error names those samples and their counts)."""
    pooled = api.StrandVotes(*(sum(getattr(v, f) for v in votes) for f in ("agree_fr", "opposite", "no_vote")))
    verdict = api.library_type(pooled)
    odd = [(t, v, api.library_type(v)) for t, v in zip(titles, votes) if api.library_type(v) not in (None, verdict)]
    if odd and verdict is not None:
        print("\n".join(_strand_report(pooled)[1]))
        raise StrandednessError("samples disagree with the pooled library type %s: %s" % (verdict, "; ".join(
            "%s is %s (agree with fr %d, opposite %d, no vote %d)" % (t, lt, v.agree_fr, v.opposite, v.no_vote) for t, v, lt in odd)))
    return _verdict_flags(pooled, "the pooled samples")


# ------------------------------------------------------------------------------------------------ samples told apart by a tag
class GroupsFileError(ValueError):
    """A groups file (value <TAB> title per line) that cannot be read; the message names the line."""


def _tag_value(x):
    if len(x) != 2 or not (x[0].isascii() and x[0].isalpha()) or not (x[1].isascii() and x[1].isalnum()):
        raise argparse.ArgumentTypeError("a tag is two characters, [A-Za-z][A-Za-z0-9], got %r" % x)
    return x


def read_groups_file(path):
    """(values, group of every value, titles) of a groups file: lines `value <TAB> title`; many values may share a title (a
    barcode -> cluster table).  The group order is the order in which titles first appear.  GroupsFileError names the line
    that has not exactly two non-empty columns, has a value the library refuses (more than 255 bytes, NUL; TAB and newline cannot
    occur), repeats a value, or has a title with '/', TAB or NUL."""
    values, groups, titles, at, seen = [], [], [], {}, {}
    with open(path, encoding="utf-8", newline="") as fh:
        for ln, line in enumerate(fh, 1):
            cols = line.rstrip("\r\n").split("\t")
            if len(cols) != 2 or not cols[0] or not cols[1]:
                raise GroupsFileError("%s line %d: not two tab-separated columns (value <TAB> title)" % (path, ln))
            value, title = cols
            if len(value.encode()) > 255 or "\0" in value:
                raise GroupsFileError("%s line %d: value %r is longer than 255 bytes or contains NUL" % (path, ln, value))
            if "/" in title or "\0" in title:
                raise GroupsFileError("%s line %d: title %r contains '/', TAB or NUL" % (path, ln, title))
            if value in seen:
                raise GroupsFileError("%s line %d: value %r repeats line %d" % (path, ln, value, seen[value]))
            seen[value] = ln
            if title not in at:
                at[title] = len(titles)
                titles.append(title)
            values.append(value)
            groups.append(at[title])
    if not titles:
        raise GroupsFileError("%s: no groups" % path)
    return values, groups, titles


def _rank_table(tag, values, groups, mine):
    """The tag group table of the groups `mine` (global indices, in order): their values, renumbered 0 .. len(mine) - 1."""
    local = {g: i for i, g in enumerate(mine)}
    keep = [(v, local[g]) for v, g in zip(values, groups) if g in local]
    return api.TagGroups(tag, [v for v, _ in keep], [g for _, g in keep], len(mine))


def combineGroups(inBAM, tag, groupsFile, outputPath, annotationFile=None, aType="gene", qGene="All", isStranded=False,
                  strandedType=None, isbeta2Cryptic=False, minAnchor=8, minIntron=70, maxIntron=500000, strandFromXS=False,
                  shallow=False, minSamples=0, minReads=10, minSSE=0.0, devices=None, context_factory=None, read_filter=None):
    """The groups of one BAM told apart by an aux tag (read groups RG, cell-barcode clusters CB, haplotypes HP) as the samples of
    combineBam: the BAM is ingested once per rank and split on the GPU (Context.load_bam_groups; include/spliser_b200.h,
    spl_tag_groups, states the rule).  out.<title>.SpliSER.tsv is what processBam writes on a BAM of that group's records, and
    out.combined.tsv what combineBam writes over those BAMs in group order, the order in which titles first appear in the groups
    file.  With several devices rank r splits off the groups dist.samples_of(r, n_ranks, n_groups) only.  A split that does not
    fit raises SampleMemoryError naming the bytes it needs; there is no path route for a group."""
    print("Combining the groups of one BAM...")
    values, groups, titles = read_groups_file(groupsFile)
    n = len(titles)
    tsv_paths = ["%s.%s.SpliSER.tsv" % (outputPath, t) for t in titles]
    annotation = load_annotation(annotationFile, "All") if annotationFile is not None else None
    n_ranks = len(devices) if devices else 1
    splits, counts, no_value, kept = {}, [0] * n, [0], [0, 0]

    def load(rank, c, k, xs):
        if rank not in splits:
            mine = samples_of(rank, n_ranks, n)
            splits[rank] = (mine, c.load_bam_groups(inBAM, _rank_table(tag, values, groups, mine), xs=xs))
            got = splits[rank][1]
            for g, cnt in zip(mine, got.counts):
                counts[g] = cnt
            no_value[0] = got.no_value
            kept[:] = c.last_read_filter()
        mine, got = splits[rank]
        return got.samples[mine.index(k)]
    try:
        _combine_resident(titles, tsv_paths, [inBAM] * n, outputPath, annotation, qGene, isStranded, strandedType, isbeta2Cryptic,
                          minAnchor, minIntron, maxIntron, strandFromXS, shallow, minSamples, minReads, minSSE, devices, context_factory,
                          read_filter, load)
    finally:
        for _, got in splits.values():
            got.close()
    print("Records per group ({}):\t{}\tno value {}\tvalue in no group {}".format(
        tag, "\t".join("%s %d" % x for x in zip(titles, counts)), no_value[0], kept[0] - sum(counts) - no_value[0]))
    if read_filter is not None:
        print("Read filter {}:\tkept {}\tdropped {}".format(inBAM, *kept))


# ------------------------------------------------------------------------------------------------ main
def _mapq_value(x):
    v = int(x, 0)
    if not 0 <= v <= 255:
        raise argparse.ArgumentTypeError("MAPQ must be in 0..255, got %s" % x)
    return v


def _flag_value(x):
    v = int(x, 0)
    if not 0 <= v <= 0xFFFF:
        raise argparse.ArgumentTypeError("FLAG bits must be in 0..0xFFFF, got %s" % x)
    return v


def _add_read_filter_options(p):
    """samtools view's -q / -F / -f under long names only (the short letters stay free for the reference's options)."""
    p.add_argument("--minMAPQ", dest="minMAPQ", default=0, type=_mapq_value, metavar="N",
                   help="keep records with MAPQ >= N (samtools -q; 255, unavailable, passes)")
    p.add_argument("--excludeFlags", dest="excludeFlags", default=0, type=_flag_value, metavar="F",
                   help="drop records with any of these FLAG bits (samtools -F), e.g. 0x904")
    p.add_argument("--requireFlags", dest="requireFlags", default=0, type=_flag_value, metavar="F",
                   help="keep records with all of these FLAG bits (samtools -f), e.g. 0x2")


READ_COMMANDS = ("process", "combine", "combineShallow", "junctions", "processBam", "combineBam", "inferStrandedness", "combineGroups")


def main(argv=None):
    print("\nSpliSER " + VERSION + "\n")
    start = timeit.default_timer()
    parser = argparse.ArgumentParser(description="SpliSER - Splice Site Strength Estimates from RNA-seq (B200 counting path)")
    sub = parser.add_subparsers(dest="command")
    p = sub.add_parser("process")
    p.add_argument("-B", "--BAMFile", dest="inBAM", required=True)
    p.add_argument("-b", "--bedFile", dest="inBed", required=True)
    p.add_argument("-o", "--outputPath", dest="outputPath", required=True)
    p.add_argument("-A", "--annotationFile", dest="annotationFile", required=False)
    p.add_argument("-t", "--annotationType", dest="aType", nargs="?", default="gene", type=str)
    p.add_argument("-c", "--chromosome", dest="qChrom", nargs="?", default="All", type=str)
    p.add_argument("-g", "--gene", dest="qGene", nargs="?", default="All", type=str)
    p.add_argument("-m", "--maxIntronSize", dest="maxIntronSize", nargs="?", default=0, type=int)
    p.add_argument("--isStranded", dest="isStranded", default=False, action="store_true")
    p.add_argument("-s", "--strandedType", dest="strandedType", nargs="?", type=str)
    p.add_argument("--beta2Cryptic", dest="isbeta2Cryptic", default=False, action="store_true")
    c = sub.add_parser("combine")
    c.add_argument("-S", "--samplesFile", dest="samplesFile", required=True)
    c.add_argument("-o", "--outputPath", dest="outputPath", required=True)
    c.add_argument("-g", "--gene", dest="qGene", nargs="?", default="All", type=str)
    c.add_argument("--isStranded", dest="isStranded", default=False, action="store_true")
    c.add_argument("-s", "--strandedType", dest="strandedType", nargs="?", default="fr", type=str)
    c.add_argument("--beta2Cryptic", dest="isbeta2Cryptic", default=False, action="store_true")
    c.add_argument("--gpus", dest="n_gpus", nargs="?", default=1, type=int,
                   help="re-count the samples on this many GPUs (sharded by sample; not a reference option)")
    cs = sub.add_parser("combineShallow")
    cs.add_argument("-S", "--samplesFile", dest="samplesFile", required=True)
    cs.add_argument("-g", "--gene", dest="qGene", nargs="?", default="All", type=str)
    cs.add_argument("-o", "--outputPath", dest="outputPath", required=True)
    cs.add_argument("--isStranded", dest="isStranded", default=False, action="store_true")
    cs.add_argument("-m", "--minSamples", dest="minSamples", nargs="?", default=0, type=int)
    cs.add_argument("-r", "--minReads", dest="minReads", nargs="?", default=10, type=int)
    cs.add_argument("-e", "--minSSE", dest="minSSE", nargs="?", default=0.00, type=float)
    cs.add_argument("-s", "--strandedType", dest="strandedType", nargs="?", type=str)
    cs.add_argument("--beta2Cryptic", dest="isbeta2Cryptic", default=False, action="store_true")
    cs.add_argument("--gpus", dest="n_gpus", nargs="?", default=1, type=int,
                    help="re-count the samples on this many GPUs (sharded by sample; not a reference option)")
    j = sub.add_parser("junctions", help="junction BED12 from the BAM alone (the regtools junctions extract step)")
    j.add_argument("-B", "--BAMFile", dest="inBAM", required=True)
    j.add_argument("-o", "--output", dest="outBed", required=True)
    j.add_argument("-a", "--minAnchor", dest="minAnchor", default=8, type=int)
    j.add_argument("-m", "--minIntron", dest="minIntron", default=70, type=int)
    j.add_argument("-M", "--maxIntron", dest="maxIntron", default=500000, type=int)
    j.add_argument("--isStranded", dest="isStranded", default=False, action="store_true")
    j.add_argument("-s", "--strandedType", dest="strandedType", nargs="?", type=str)
    j.add_argument("--strandFromXS", dest="strandFromXS", default=argparse.SUPPRESS, action="store_true",
                   help="junction strands from the aligner's XS tag ('?' without one), as regtools writes them")
    pb = sub.add_parser("processBam", help="process without a BED12: junctions extracted from the BAM in the same pass")
    pb.add_argument("-B", "--BAMFile", dest="inBAM", required=True)
    pb.add_argument("-o", "--outputPath", dest="outputPath", required=True)
    pb.add_argument("-A", "--annotationFile", dest="annotationFile", required=False)
    pb.add_argument("-t", "--annotationType", dest="aType", nargs="?", default="gene", type=str)
    pb.add_argument("-c", "--chromosome", dest="qChrom", nargs="?", default="All", type=str)
    pb.add_argument("-g", "--gene", dest="qGene", nargs="?", default="All", type=str)
    pb.add_argument("-m", "--maxIntronSize", dest="maxIntronSize", nargs="?", default=0, type=int)
    pb.add_argument("--isStranded", dest="isStranded", default=False, action="store_true")
    pb.add_argument("-s", "--strandedType", dest="strandedType", nargs="?", type=str)
    pb.add_argument("--beta2Cryptic", dest="isbeta2Cryptic", default=False, action="store_true")
    pb.add_argument("--minAnchor", dest="minAnchor", default=8, type=int)
    pb.add_argument("--minIntron", dest="minIntron", default=70, type=int)
    pb.add_argument("--maxIntron", dest="maxIntron", default=500000, type=int)
    pb.add_argument("--strandFromXS", dest="strandFromXS", default=argparse.SUPPRESS, action="store_true",
                    help="junction strands from the aligner's XS tag; the count still follows --isStranded -s")
    cb = sub.add_parser("combineBam", help="processBam for every sample, then combine, reading every BAM once")
    cb.add_argument("-S", "--samplesFile", dest="samplesFile", required=True,
                    help="title <TAB> .SpliSER.tsv to write <TAB> BAM, one sample per line (combine's samples file)")
    cb.add_argument("-o", "--outputPath", dest="outputPath", required=True)
    cb.add_argument("-A", "--annotationFile", dest="annotationFile", required=False)
    cb.add_argument("-t", "--annotationType", dest="aType", nargs="?", default="gene", type=str)
    cb.add_argument("-g", "--gene", dest="qGene", nargs="?", default="All", type=str)
    cb.add_argument("--isStranded", dest="isStranded", default=False, action="store_true")
    cb.add_argument("-s", "--strandedType", dest="strandedType", nargs="?", type=str)
    cb.add_argument("--beta2Cryptic", dest="isbeta2Cryptic", default=False, action="store_true")
    cb.add_argument("--minAnchor", dest="minAnchor", default=8, type=int)
    cb.add_argument("--minIntron", dest="minIntron", default=70, type=int)
    cb.add_argument("--maxIntron", dest="maxIntron", default=500000, type=int)
    cb.add_argument("--strandFromXS", dest="strandFromXS", default=False, action="store_true",
                    help="junction strands from the aligner's XS tag; the count still follows --isStranded -s")
    cb.add_argument("--shallow", dest="shallow", default=False, action="store_true", help="merge as combineShallow")
    cb.add_argument("-m", "--minSamples", dest="minSamples", nargs="?", default=0, type=int)
    cb.add_argument("-r", "--minReads", dest="minReads", nargs="?", default=10, type=int)
    cb.add_argument("-e", "--minSSE", dest="minSSE", nargs="?", default=0.00, type=float)
    cb.add_argument("--gpus", dest="n_gpus", nargs="?", default=1, type=int,
                    help="hold and count the samples on this many GPUs (sharded by sample)")
    cg = sub.add_parser("combineGroups", help="combineBam over the groups of one BAM told apart by an aux tag, with one ingest")
    cg.add_argument("-B", "--BAMFile", dest="inBAM", required=True)
    cg.add_argument("--tag", dest="tag", required=True, type=_tag_value, help="the aux tag that tells the groups apart, e.g. RG, CB, HP")
    cg.add_argument("-G", "--groupsFile", dest="groupsFile", required=True,
                    help="value <TAB> title per line; values that share a title form one group, in the order titles first appear")
    cg.add_argument("-o", "--outputPath", dest="outputPath", required=True)
    cg.add_argument("-A", "--annotationFile", dest="annotationFile", required=False)
    cg.add_argument("-t", "--annotationType", dest="aType", nargs="?", default="gene", type=str)
    cg.add_argument("-g", "--gene", dest="qGene", nargs="?", default="All", type=str)
    cg.add_argument("--isStranded", dest="isStranded", default=False, action="store_true")
    cg.add_argument("-s", "--strandedType", dest="strandedType", nargs="?", type=str)
    cg.add_argument("--beta2Cryptic", dest="isbeta2Cryptic", default=False, action="store_true")
    cg.add_argument("--minAnchor", dest="minAnchor", default=8, type=int)
    cg.add_argument("--minIntron", dest="minIntron", default=70, type=int)
    cg.add_argument("--maxIntron", dest="maxIntron", default=500000, type=int)
    cg.add_argument("--strandFromXS", dest="strandFromXS", default=False, action="store_true",
                    help="junction strands from the aligner's XS tag; the count still follows --isStranded -s")
    cg.add_argument("--shallow", dest="shallow", default=False, action="store_true", help="merge as combineShallow")
    cg.add_argument("-m", "--minSamples", dest="minSamples", nargs="?", default=0, type=int)
    cg.add_argument("-r", "--minReads", dest="minReads", nargs="?", default=10, type=int)
    cg.add_argument("-e", "--minSSE", dest="minSSE", nargs="?", default=0.00, type=float)
    cg.add_argument("--gpus", dest="n_gpus", nargs="?", default=1, type=int,
                    help="split and count the groups on this many GPUs (sharded by group; each GPU ingests the BAM once)")
    inf = sub.add_parser("inferStrandedness", help="the library type (--isStranded -s fr|rf, or unstranded) from the BAM")
    inf.add_argument("-B", "--BAMFile", dest="inBAM", required=True)
    inf.add_argument("-A", "--annotationFile", dest="annotationFile", required=False,
                     help="reference strands from the genes of this GFF / GTF (default: from the aligner's XS tag)")
    for name, sp in sub.choices.items():
        if name in READ_COMMANDS:
            _add_read_filter_options(sp)
    kwargs = vars(parser.parse_args(argv))          # --strandFromXS is only passed on when given (SUPPRESS)
    command = kwargs.pop("command")
    if command in READ_COMMANDS:
        rf = api.ReadFilter(kwargs.pop("minMAPQ"), kwargs.pop("excludeFlags"), kwargs.pop("requireFlags"))
        if not rf.is_none:
            kwargs["read_filter"] = rf
    if command in ("combine", "combineShallow", "combineBam", "combineGroups"):
        kwargs["devices"] = list(range(max(1, kwargs.pop("n_gpus") or 1)))
    if command in ("process", "processBam") and kwargs.get("qGene") != "All" and (kwargs.get("annotationFile") is None or kwargs.get("maxIntronSize") is None):
        parser.error("--gene requires --annotationFile and --maxIntronSize")                      # S:1350-1353
    elif command in ("combineBam", "combineGroups") and kwargs.get("qGene") != "All" and kwargs.get("annotationFile") is None:
        parser.error("--gene requires --annotationFile (the Gene column comes from it)")
    elif command in ("process", "combine", "combineShallow", "junctions", "processBam", "combineBam", "combineGroups") and kwargs.get("isStranded") and kwargs.get("strandedType") is None:
        parser.error("--isStranded requires parameter --strandedType/-s as fr or rf")            # S:1354-1355
    elif command == "junctions" and kwargs.get("strandFromXS") and kwargs.get("isStranded"):
        parser.error("--strandFromXS and --isStranded name two strand sources for the junction table")
    elif command == "process":
        process(**kwargs)
    elif command == "combine":
        combine(**kwargs)
    elif command == "combineShallow":
        combineShallow(**kwargs)
    elif command == "junctions":
        junctions(**kwargs)
    elif command in ("processBam", "combineBam", "inferStrandedness", "combineGroups"):
        try:
            {"processBam": processBam, "combineBam": combineBam, "inferStrandedness": inferStrandedness,
             "combineGroups": combineGroups}[command](**kwargs)
        except (StrandednessError, GroupsFileError) as e:
            parser.error(str(e))
        except api.SampleMemoryError as e:
            if command != "combineGroups":
                raise
            parser.error("the groups do not fit in GPU memory: %s" % e)
    else:
        parser.error("command must be process, combine, combineShallow, junctions, processBam, combineBam or inferStrandedness "
                     "(output is unchanged Python in the reference)")
    print("Total runtime (s): \t" + str(timeit.default_timer() - start))


if __name__ == "__main__":
    main()
