"""SpliSER-compatible command line: `process` and `combine` with the reference's flags and byte-identical
.SpliSER.tsv / .combined.tsv output, the counting done by libspliser_b200.so on the GPU.

    python -m spliser_b200.cli process -B x.bam -b x.bed -o out [-A genes.gff] [-c chr] [-g gene -m 500000]
                                       [--isStranded -s rf|fr] [--beta2Cryptic]
    python -m spliser_b200.cli combine -S samples.tsv -o out [-g gene] [--isStranded -s rf|fr] [--beta2Cryptic]

Without regtools (not a reference command; regtools' option letters):
    python -m spliser_b200.cli junctions -B x.bam -o x.bed [-a 8] [-m 70] [-M 500000] [--isStranded -s rf|fr | --strandFromXS]
    python -m spliser_b200.cli processBam -B x.bam -o out [process's -A -t -c -g -m --isStranded -s --beta2Cryptic]
                                          [--minAnchor 8] [--minIntron 70] [--maxIntron 500000] [--strandFromXS]
`junctions` writes the junction BED12 that `regtools junctions extract` would feed `process` with; `processBam` is
`junctions` followed by `process -b` in one call that reads the BAM once, and writes the same .SpliSER.tsv.  --strandFromXS
takes the junction strands from the aligner's XS tag, as regtools does for unstranded libraries; processBam still counts
with --isStranded -s.

What stays in Python is what the reference does in text: BED12 parsing and its filters (S:255-288), the
annotation and gene lookup (S:50-173), the TSV writers (S:641-664, S:722-740) and the lock-step merge of
`combine` (S:742-917).  The body of `process` (S:710-717) is one spl_process call; every checkBam call of
`combine` (S:903) goes into one batched spl_recount call per sample.
"""
from __future__ import annotations

import argparse
import sys
import timeit

import numpy as np

from . import api
from .bed import StrandColumn, parse_bed12, write_junctions_bed
from .dist import samples_of
from .genes import load_annotation
from .hosttext import CombineMerge, write_process_tsv as _native_write_process_tsv

VERSION = "v0.1.8 (spliser_b200)"


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
            isStranded=False, strandedType=None, isbeta2Cryptic=False, ctx=None):
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
        with open(inBed) as fh:
            chroms, table, sstr = process_table(ctx, inBAM, fh, annotation=annotation, qchrom=qChrom, qgene=qGene,
                                                max_intron=maxIntronSize, is_stranded=isStranded, stranded_type=strandedType,
                                                beta2_cryptic=isbeta2Cryptic, parsed_bed=parsed_bed)
    finally:
        if own:
            ctx.close()
    print("Sites:\t\t\t" + str(len(table)))
    write_process_tsv(outputPath + ".SpliSER.tsv", chroms, table, sstr, annotation=annotation, is_stranded=isStranded,
                      beta2_cryptic=isbeta2Cryptic)


# ------------------------------------------------------------------------------------------------ without regtools
def junctions(inBAM, outBed, minAnchor=8, minIntron=70, maxIntron=500000, isStranded=False, strandedType=None, strandFromXS=False,
              ctx=None):
    """The `regtools junctions extract -a -m -M` step on the GPU: the junction table of every header reference, written as
    BED12 in regtools' layout (chromStart / chromEnd from the longest anchors).  Strands: with strandFromXS the record's XS tag
    ('?' without one; include/spliser_b200.h, SPL_FLAG_XS_STRAND), else '?' unstranded, else the strand check_strand derives
    from the FLAG (S:374-406)."""
    chroms = api.bam_reference_names(inBAM)
    flags = api.FLAG_XS_STRAND if strandFromXS else api.mode_flags(isStranded, strandedType)
    own = ctx is None
    ctx = ctx or api.Context(0)
    try:
        junc = ctx.extract_junctions_bam(inBAM, chroms, flags, minAnchor, minIntron, maxIntron)
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
               strandedType=None, isbeta2Cryptic=False, minAnchor=8, minIntron=70, maxIntron=500000, strandFromXS=False, ctx=None):
    """`junctions` + `process -b` in one GPU call that ingests the BAM once (spl_process_bam_extract).  The chromosome list is
    the annotation's names, then the header's references not among them in header order: the relative order `process` gets
    from a BED12 written by `junctions`, so the .SpliSER.tsv is the same byte for byte.  strandFromXS: the table's strands come
    from the XS tag (`junctions --strandFromXS`); the count still follows isStranded / strandedType."""
    print("Processing")
    print("Stranded Analysis {}".format(strandedType) if isStranded else "Unstranded Analysis")
    annotation = load_annotation(annotationFile, qGene) if annotationFile is not None else None
    bounds = None
    if qGene != "All":
        q = annotation.query_gene if annotation is not None else None
        if q is None:                           # S:283, as in process
            raise AttributeError("'NoneType' object has no attribute 'getLeftPos'")
        bounds = (q.left, q.right)
    chroms = list(annotation.chrom_index) if annotation is not None else []
    known = set(chroms)
    chroms += [c for c in api.bam_reference_names(inBAM) if c not in known]
    flags = api.mode_flags(isStranded, strandedType, isbeta2Cryptic) | (api.FLAG_XS_STRAND if strandFromXS else 0)
    own = ctx is None
    ctx = ctx or api.Context(0)
    try:
        junc, table = ctx.process_bam_extract(inBAM, chroms, flags, minAnchor, minIntron, maxIntron, qchrom=qChrom, gene_bounds=bounds,
                                              window_max_intron=int(maxIntronSize))
    finally:
        if own:
            ctx.close()
    print("Sites:\t\t\t" + str(len(table)))
    write_process_tsv(outputPath + ".SpliSER.tsv", chroms, table, _strand_column(junc), annotation=annotation, is_stranded=isStranded,
                      beta2_cryptic=isbeta2Cryptic)


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


def _recount_sample(ctx, cm, k, regions, bam_path, flags, records_by_bam):
    """Every S:903 call of sample k in one spl_recount call; returns False when the sample has no gaps."""
    gaps = cm.gaps(k)
    if not len(gaps):
        return False
    uniq, first = np.unique(gaps.chrom, return_index=True)
    local = uniq[np.argsort(first)]                 # the sample's gap regions in first-appearance order
    names = [regions[r] for r in local]
    remap = np.full(len(regions), -1, dtype=np.int32)
    remap[local] = np.arange(len(local), dtype=np.int32)
    gaps.chrom = np.ascontiguousarray(remap[gaps.chrom])
    if records_by_bam is not None:
        b1, b2 = ctx.recount_records(records_by_bam(bam_path, names), len(names), gaps, flags)
    else:
        b1, b2 = ctx.recount_bam(bam_path, names, gaps, flags)
    cm.set_recount(k, b1, b2)
    return True


def combineShallow(samplesFile, outputPath, qGene="All", isStranded=False, minSamples=0, minReads=10, minSSE=0.0, strandedType=None,
                   isbeta2Cryptic=False, ctx=None, records_by_bam=None, devices=None, context_factory=None):
    """combineShallow (S:920-1167): `combine` for many shallow samples.  The same lock-step merge and the same re-count of the
    sites a sample lacks (checkBam at S:1145 -> one spl_recount call per sample), with three filters on which positions are
    kept at all -- a position needs at least `minSamples` samples showing it with alpha + beta1 + beta2Simple >= `minReads`
    and SSE >= `minSSE` (S:1066-1084, S:1108) -- and, with -g, only the rows of that gene loaded from every table
    (S:947-956).  The quirks of the reference's loop are kept (csrc/host_text.cpp, merge_impl): the count runs over the rows
    of both strands of a position, and a dropped position moves every sample on whose current row has that position number,
    whatever its region or strand (S:1158-1160).  Unlike `combine`, a samples-file line without exactly three columns is
    skipped silently (S:930-935)."""
    return combine(samplesFile, outputPath, qGene, isStranded, strandedType, isbeta2Cryptic, ctx, records_by_bam, devices,
                   context_factory, _shallow=(minSamples, minReads, minSSE))


def combine(samplesFile, outputPath, qGene="All", isStranded=False, strandedType="fr", isbeta2Cryptic=False, ctx=None,
            records_by_bam=None, devices=None, context_factory=None, _shallow=None):
    """combine (S:742-917).  The native merge driver (csrc/host_text.cpp) parses the sample tables and replays the
    lock-step merge, collecting per sample the sites it lacks together with the partner / competitor / strand context
    gathered from lower-indexed samples only (the reference's order dependence, SURVEY.md F7); one spl_recount call
    per sample fills them; the driver then writes the rows.

    The re-count shards by sample (SURVEY.md 8(e)): with `devices` = several CUDA ordinals, one context per device runs on
    its own host thread and takes the samples dist.samples_of(rank, n_devices, n_samples); a sample's result depends on
    nothing but its own BAM and gap list, so the host only collects the count arrays.  `ctx` (one existing context) takes
    precedence; `context_factory(device)` replaces api.Context (tests)."""
    print("Combining samples...")
    titles, bed_paths, bam_paths = [], [], []
    with open(samplesFile) as fh:
        for line in fh:
            values = line.split("\t")
            if len(values) == 3:
                titles.append(values[0]); bed_paths.append(values[1]); bam_paths.append(values[2].rstrip())
            elif _shallow is None:
                print(str(titles), str(bed_paths), str(bam_paths))
                raise Exception("Samples File contains lines that do not have exactly 3 tab-separated columns")
    n = len(titles)
    flags = api.mode_flags(isStranded, strandedType, False, combine=True)
    with CombineMerge() as cm:
        cm.add_samples(titles, bed_paths)
        regions = cm.region_names()
        order = _chrom_order([[regions[r] for r in cm.sample_runs(k)] for k in range(n)])
        region_id = {name: i for i, name in enumerate(regions)}
        if _shallow is None:
            cm.merge([region_id[name] for name in order], qGene, isStranded)
        else:
            cm.merge_shallow([region_id[name] for name in order], qGene, isStranded, *_shallow)
        make = context_factory or api.Context
        devs = [0] if not devices else list(devices)
        if ctx is not None or len(devs) == 1:
            own = None
            try:
                for k in range(n):
                    if ctx is None and cm.n_gaps(k):
                        ctx = own = make(devs[0])
                    if cm.n_gaps(k):
                        _recount_sample(ctx, cm, k, regions, bam_paths[k], flags, records_by_bam)
            finally:
                if own is not None:
                    own.close()
        else:
            from concurrent.futures import ThreadPoolExecutor

            def rank_work(rank):                    # one context per device, samples dealt round-robin
                mine = [k for k in samples_of(rank, len(devs), n) if cm.n_gaps(k)]
                if not mine:
                    return 0
                c = make(devs[rank])
                try:
                    for k in mine:
                        _recount_sample(c, cm, k, regions, bam_paths[k], flags, records_by_bam)
                finally:
                    c.close()
                return len(mine)
            with ThreadPoolExecutor(max_workers=len(devs)) as pool:
                list(pool.map(rank_work, range(len(devs))))
        cm.write(outputPath + ".combined.tsv", isbeta2Cryptic)
        filled = cm.n_filled()
    print("Filled in Beta read counts for {} Sites not detected in some samples".format(filled))


# ------------------------------------------------------------------------------------------------ main
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
    kwargs = vars(parser.parse_args(argv))          # --strandFromXS is only passed on when given (SUPPRESS)
    command = kwargs.pop("command")
    if command in ("combine", "combineShallow"):
        kwargs["devices"] = list(range(max(1, kwargs.pop("n_gpus") or 1)))
    if command in ("process", "processBam") and kwargs.get("qGene") != "All" and (kwargs.get("annotationFile") is None or kwargs.get("maxIntronSize") is None):
        parser.error("--gene requires --annotationFile and --maxIntronSize")                      # S:1350-1353
    elif command in ("process", "combine", "combineShallow", "junctions", "processBam") and kwargs.get("isStranded") and kwargs.get("strandedType") is None:
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
    elif command == "processBam":
        processBam(**kwargs)
    else:
        parser.error("command must be process, combine, combineShallow, junctions or processBam (output is unchanged Python in the reference)")
    print("Total runtime (s): \t" + str(timeit.default_timer() - start))


if __name__ == "__main__":
    main()
