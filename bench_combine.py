"""bench.py --workload c4: BASELINE configs[3] -- `combine` of 48 samples (6 conditions x 8 replicates) with the re-count of
the sites a sample lacks (SpliSER_v0_1_8.py:742-917), sample-sharded over the GPUs of the box.

Every sample of a C1-like genome has its own reads (>= 1M records) and its own junction subset (a condition drops a share
of the junctions, a replicate a few more), so the merged table has gaps in every sample.  The 48 samples are first run
through `process` (BAM + BED12 -> .SpliSER.tsv, timed per sample), then `combine` is timed as a whole: native merge of the
48 tables, one spl_recount(bam) per sample on the device that owns the sample (dist.samples_of), native writer.  One process
drives every device (one context per device, one host thread each); under torchrun rank 0 alone runs.  The reference's own
figure for this stage on the small 48-sample golden workload (tests/golden/c4_48_samples_reference.json) is printed beside it.
"""
from __future__ import annotations

import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
N_COND, N_REP = 6, 8
CONTIGS = (("Chr1", 30427671), ("Chr2", 19698289), ("Chr3", 23459830), ("Chr4", 18585056), ("Chr5", 26975502))


def _subset(r, keep):
    from spliser_b200 import Records
    ncig = np.diff(r.cig_off.astype(np.int64))
    off = np.zeros(int(keep.sum()) + 1, np.uint32)
    np.cumsum(ncig[keep], out=off[1:])
    csum = np.concatenate([[0], np.cumsum(keep)])
    return Records(r.pos[keep], r.flag[keep], off, r.cigar[np.repeat(keep, ncig)], r.seg_chrom, csum[r.seg_off])


def _bed12(chroms, j, anchor=8):
    c, l, r, sc, st = j.chrom.tolist(), j.left.tolist(), j.right.tolist(), j.score.tolist(), j.strand.tolist()
    return "".join("%s\t%d\t%d\tJ%d\t%d\t%s\t%d\t%d\t255,0,0\t2\t%d,%d\t0,%d\n" % (chroms[c[i]], l[i] - anchor, r[i] + anchor, i, sc[i], chr(st[i]),
                                                                                  l[i] - anchor, r[i] + anchor, anchor, anchor, r[i] - l[i] + anchor)
                   for i in range(len(l)))


def build_samples(cache, reads_per_sample):
    """-> (chroms, [(title, bam, bed)]); files are kept in `cache`."""
    from spliser_b200 import Junctions, synth
    n_s = N_COND * N_REP
    tag = os.path.join(cache, "c4_%d" % reads_per_sample)
    meta = tag + ".json"
    chroms = [c for c, _ in CONTIGS]
    if os.path.exists(meta):
        return chroms, [tuple(x) for x in json.load(open(meta))["samples"]]
    os.makedirs(cache, exist_ok=True)
    cfg = synth.SynthConfig(name="c4bench", seed=20260004, contigs=CONTIGS, n_records=n_s * reads_per_sample, read_len=100, paired=True,
                            stranded=True, genes_per_mb=165.0, per_contig_rng=True)
    w = synth.generate(cfg)
    rng = np.random.default_rng(cfg.seed)
    r, j = w.records, w.junctions
    owner = rng.integers(0, n_s, len(r))                       # every record belongs to one sample
    cond_drop = rng.random((N_COND, len(j))) < 0.05
    samples = []
    for c in range(N_COND):
        for rep in range(N_REP):
            k = c * N_REP + rep
            keep_j = ~cond_drop[c] & (j.score >= 2 * n_s) | (~cond_drop[c] & (rng.random(len(j)) >= 0.5))     # a replicate loses weakly supported junctions
            score = np.maximum(1, (j.score[keep_j] + k) // n_s)
            jk = Junctions(j.chrom[keep_j], j.left[keep_j], j.right[keep_j], score, j.strand[keep_j])
            bam, bed = "%s_s%02d.bam" % (tag, k), "%s_s%02d.bed" % (tag, k)
            _subset(r, owner == k).write_bam(bam, chroms, [n for _, n in CONTIGS])
            with open(bed, "w") as fh:
                fh.write(_bed12(chroms, jk))
            samples.append(("cond%d_rep%d" % (c + 1, rep + 1), bam, bed))
    json.dump({"samples": samples}, open(meta, "w"))
    return chroms, samples


def run(args, rank, world, local, emit):
    if rank != 0:
        return
    sys.path.insert(0, ROOT)
    import spliser_b200
    from spliser_b200 import cli
    from bench import CACHE
    reads = args.reads or 1_000_000
    n_dev = max(1, args.gpus)
    t0 = time.perf_counter()
    chroms, samples = build_samples(CACHE, reads)
    t_build = time.perf_counter() - t0
    out_dir = os.path.join(CACHE, "c4_out_%d" % reads)
    os.makedirs(out_dir, exist_ok=True)
    # ---- process every sample (device 0): BAM + BED12 -> .SpliSER.tsv
    lines, t_proc = [], []
    with spliser_b200.Context(0) as ctx:
        for i, (title, bam, bed) in enumerate(samples):
            outp = os.path.join(out_dir, "s%02d" % i)
            a = time.perf_counter()
            cli.process(bam, bed, outp, isStranded=True, strandedType="rf", ctx=ctx)
            t_proc.append(time.perf_counter() - a)
            lines.append("%s\t%s\t%s\n" % (title, outp + ".SpliSER.tsv", bam))
    sf = os.path.join(out_dir, "samples.tsv")
    with open(sf, "w") as fh:
        fh.writelines(lines)
    # ---- combine: merge + re-count (sample-sharded over the devices) + write
    outc = os.path.join(out_dir, "combined")
    devices = list(range(n_dev))
    times = []
    for it in range(1 + args.steps):                                 # first run = warm-up (contexts, page cache)
        a = time.perf_counter()
        cli.combine(sf, outc, isStranded=True, strandedType="rf", devices=devices)
        if it:
            times.append(time.perf_counter() - a)
    rows = sum(1 for _ in open(outc + ".combined.tsv")) - 1
    total_reads = reads * len(samples)
    step = float(np.mean(times))
    ref = None
    try:
        g = json.load(open(os.path.join(ROOT, "tests", "golden", "c4_48_samples_reference.json")))
        ref = {"workload": g["workload"], "combined_rows": g["combined_rows"], "recounted_gaps": g["recounted_gaps"], "reference_seconds": g.get("reference_seconds"),
               "note": "the unmodified reference on the small 48-sample golden workload (authoring container); not the workload timed here"}
    except (OSError, ValueError, KeyError):
        pass
    emit(json.dumps({
        "metric": "aligned reads/s re-read by combine (configs[3])", "value": total_reads / step, "unit": "reads/s", "n_gpus": n_dev,
        "steps": len(times), "warmup": 1, "ms_per_step": 1e3 * step, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
        "dtype": "u32", "data": "synthetic",
        "config": {"workload": "configs[3]: combine of 48 samples (6 conditions x 8 replicates, %d records each, C1-like five-chromosome genome, stranded rf) with the "
                               "re-count of the sites a sample lacks, samples sharded over %d GPU(s) (one context per device in one process)" % (reads, n_dev),
                   "combined_rows": rows, "samples": len(samples), "timing": "host wall clock around cli.combine: native merge of 48 .SpliSER.tsv, 48 x spl_recount(bam) "
                   "(device BAM ingest + fused counting kernel in combine mode), native writer"},
        "process_per_sample_ms": {"mean": 1e3 * float(np.mean(t_proc[1:])), "max": 1e3 * float(np.max(t_proc[1:]))},
        "build_inputs_s": round(t_build, 1),
        "reference": ref,
        "e2e": {"value": total_reads / step, "unit": "reads/s", "h2d_bytes_per_step": int(sum(os.path.getsize(s[1]) for s in samples)), "d2h_bytes_per_step": 0},
        "gpu_launches": None}))
