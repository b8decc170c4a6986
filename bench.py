#!/usr/bin/env python
"""Benchmark of the SpliSER counting path (BASELINE.json metric: aligned reads/s to per-site SSE).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload c2|c3|c1|small|c4]
    torchrun --nproc-per-node N ... bench.py --gpus N ...          (one rank per GPU)

One "step" = one pass of the hot path over one sample: alignment records + junction table -> per-site alpha, beta1,
beta2Simple, beta2Cryptic, SSE (what `process` does per sample, SpliSER_v0_1_8.py:710-717).

  N = 1   workload = BASELINE.json configs[1] (full A. thaliana genome, 40M 150 bp PE records, --isStranded -s rf).
  N > 1   ONE sample sharded over the GPUs by genomic tile (north_star; SURVEY 8(e)): workload = configs[2] (GRCh38
          contig lengths, 200M 150 bp PE records); every rank receives the records of its read-balanced tile (reads that
          reach across a tile edge go to both tiles) and counts the sites it owns; no data-path collective.  `--scaling weak`
          runs one sample per GPU instead (replicas).

  value     reads/s of the WHOLE per-sample path with the record arrays and the junction table resident in HBM: site table
            + competing-site graph (K1), counters zeroed, fused counting kernel, prefix scan + beta2 gather + SSE.  CUDA events
            on the library's stream around K passes, every kernel of the path inside; max over ranks.
  e2e       the same through the C ABI from pinned host arrays (spl_process_records): H2D of records and junction table, the
            path above, D2H of the result table, host wall clock.
  roofline  the slowest kernel of the timed path (k_count_fused): SURVEY 8(d) algorithmic bytes of the read SoA / its
            CUDA-event time vs the measured HBM peak.
  parity    the table e2e returned is compared with the oracle's C port of the reference on the SAME full workload
            (every column, floats bit for bit); that oracle run is also the cpu_baseline.

  --dump-outputs DIR   after the timed steps, the site table the last timed step computed (rank 0's; --impl reference:
            the oracle's table of its last step) goes to DIR/<column>.npy as float64, so that two builds run with the same
            arguments (seeded, identical inputs) can be compared output for output.
"""
from __future__ import annotations

import argparse
import hashlib
import json
import os
import subprocess
import sys
import tempfile
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "aligned reads/s to per-site SSE"
CACHE = os.environ.get("SPLISER_BENCH_CACHE", os.path.join(tempfile.gettempdir(), "spliser_bench_cache"))


def workload_config(name, reads, rank=0):
    from spliser_b200 import synth
    if name == "c2":
        cfg = synth.config_c2(reads or 40_000_000)
        desc = "configs[1]: full A. thaliana genome (TAIR10 contig lengths), %d 150 bp PE records, --isStranded -s rf" % cfg.n_records
    elif name == "c3":
        cfg = synth.config_c3_full(reads or 200_000_000)
        desc = "configs[2]: GRCh38 primary contig lengths, %d 150 bp PE records, introns up to 500 kb, --isStranded -s rf" % cfg.n_records
    elif name == "c1":
        cfg = synth.config_c1()
        if reads:
            cfg.n_records = reads
        desc = "configs[0]: Chr1-sized contig, %d 100 bp SE records, unstranded" % cfg.n_records
    elif name == "small":
        cfg = synth.config_small(reads or 200_000, seed=3, stranded=True, paired=True)
        desc = "small test workload, %d records" % cfg.n_records
    else:
        raise SystemExit("unknown workload %s" % name)
    cfg.seed += 7919 * rank
    return cfg, desc


def generate_once(cfg, ranks):
    """Rank 0 builds the workload into the cache; the other ranks of the node load it from there."""
    from spliser_b200 import synth
    if ranks.rank == 0:
        w = synth.generate(cfg, cache_dir=CACHE)
    ranks.barrier()
    if ranks.rank != 0:
        w = synth.generate(cfg, cache_dir=CACHE)
    return w


def first_segment(w):
    """Records of the first chromosome segment + its junctions (the bounded sample of the reference arm on big workloads)."""
    from spliser_b200 import Junctions, Records
    r, j = w.records, w.junctions
    n = int(r.seg_off[1] - r.seg_off[0]) if len(r.seg_chrom) else 0
    c0 = int(r.seg_chrom[0])
    rec = Records(r.pos[:n], r.flag[:n], r.cig_off[:n + 1], r.cigar[:int(r.cig_off[n])], [c0], [0, n])
    keep = j.chrom == c0
    return rec, Junctions(j.chrom[keep], j.left[keep], j.right[keep], j.score[keep], j.strand[keep])


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, device):
        self.rows, self.proc = [], None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(device), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits",
                                          "-lms", "50"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._pump, daemon=True)
            self.thread.start()
        except OSError:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.rows.append((time.time(), line.strip()))

    def window(self, t0, t1):
        sm, mx, reasons = [], 0.0, set()
        rows = [r for t, r in self.rows if t0 - 0.05 <= t <= t1 + 0.15] or [r for _, r in self.rows[-3:]]
        for r in rows:
            f = [x.strip() for x in r.split(",")]
            try:
                sm.append(float(f[0])); mx = max(mx, float(f[1]))
            except (ValueError, IndexError):
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": mx or None, "reasons": sorted(reasons), "samples": len(sm)}

    def stop(self):
        if self.proc:
            self.proc.terminate()


def measured_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        return float(json.load(open(p))["hbm_gbs"]), "MEASURED_PEAKS.json hbm_gbs (of measured)"
    return 6650.0, "B200_PROFILING.md fallback 6.65 TB/s (of fallback)"


def traffic_from_profile(kernel):
    p = os.path.join(ROOT, "profiles", "traffic.json")
    try:
        d = json.load(open(p))
        return d.get("step_dram_bytes") if kernel == "step" else d.get(kernel + "_dram_bytes_per_launch")
    except (ValueError, OSError):
        return None


def python_reference_note():
    """The unmodified (Python) reference cannot run on the GPU box; oracle/time_reference.py timed it in the authoring
    container on configs[0] and recorded how much faster the C port timed here is (profiles/r1_reference_python_c1.json)."""
    p = os.path.join(ROOT, "profiles", "r1_reference_python_c1.json")
    try:
        d = json.load(open(p))
        return {"reads_per_s": d["reference_reads_per_s"], "cores": 1, "workload": "configs[0], authoring container, samtools fork replaced by an in-process indexed store (its time excluded)",
                "c_port_over_python_reference_1_thread": d["c_port_over_reference"]["threads_1"], "source": "profiles/r1_reference_python_c1.json"}
    except (OSError, ValueError, KeyError):
        return None


def soa_counts(r):
    """What SURVEY 8(d) counts in the read SoA: M/=/X blocks, N operators, spliced reads."""
    op = r.cigar & 15
    is_m = (op == 0) | (op == 7) | (op == 8)
    is_n = op == 3
    b_m, b_n = int(is_m.sum()), int(is_n.sum())
    csum = np.concatenate([[0], np.cumsum(is_n, dtype=np.int64)])
    per_rec = csum[r.cig_off[1:].astype(np.int64)] - csum[r.cig_off[:-1].astype(np.int64)]
    return b_m, b_n, int((per_rec > 0).sum())


def table_digest(t):
    """sha256 over every column of a result table (dict of arrays or SiteTable), floats bit for bit."""
    from oracle import c_oracle
    d = t if isinstance(t, dict) else c_oracle.table_dict(t)
    h = hashlib.sha256()
    for k in c_oracle.TABLE_FIELDS:
        h.update(np.ascontiguousarray(d[k]).tobytes())
    return h.hexdigest()[:32]


DUMP_BYTES = 64_000_000
DUMP_SEED = 20261020


def dump_outputs(out_dir, t, limit=DUMP_BYTES):
    """Every column of a result table (dict of arrays or SiteTable) -> out_dir/<column>.npy, float64 (exact for the integer
    columns).  When the columns come to more than `limit` bytes, each keeps the same fixed share of its entries: a seeded
    sample that depends only on the array's length, so columns of one length keep the same rows and two runs with the same
    inputs keep the same entries."""
    from oracle import c_oracle
    d = t if isinstance(t, dict) else c_oracle.table_dict(t)
    cols = {k: np.asarray(d[k]) for k in c_oracle.TABLE_FIELDS}
    keep = min(1.0, (limit - 128 * len(cols)) / max(1, sum(8 * len(a) for a in cols.values())))     # 128 B: the header of a 1-D .npy
    os.makedirs(out_dir, exist_ok=True)
    rows = {}
    for k, a in cols.items():
        if keep < 1.0:
            n = len(a)
            if n not in rows:
                rows[n] = np.sort(np.random.default_rng([DUMP_SEED, n]).choice(n, int(n * keep), replace=False))
            a = a[rows[n]]
        np.save(os.path.join(out_dir, k + ".npy"), a.astype(np.float64))


def synthetic_gff(w, path):
    """A gene every ~4 kb on both strands (seeded): only the Gene column of the TSV depends on it."""
    rng = np.random.default_rng(20260099)
    with open(path, "w") as fh:
        for c, n in zip(w.chroms, w.chrom_len):
            k = max(1, int(n) // 4000)
            starts = np.sort(rng.integers(1, max(2, int(n) - 6000), size=k))
            lens = rng.integers(500, 6000, size=k)
            strand = rng.integers(0, 2, size=k)
            fh.writelines("%s\tsynthetic\tgene\t%d\t%d\t.\t%s\t.\tID=%s_G%06d;Name=n%d\n" % (c, a, a + b, "+-"[d], c, i, i)
                          for i, (a, b, d) in enumerate(zip(starts.tolist(), lens.tolist(), strand.tolist())))


def cli_process_run(ctx, w, bam, args, reads):
    """`spliser_b200.cli.process` on files, timed as a whole and per stage (host wall clock)."""
    from spliser_b200 import cli
    from spliser_b200.genes import load_annotation
    stem = os.path.join(CACHE, "bench_%s_%d" % (args.workload, len(w.records)))
    bed, gff, outp = stem + ".bed", stem + ".gff", stem + ".out"
    if not os.path.exists(bed):
        open(bed + ".tmp", "w").write(w.bed12_text())
        os.replace(bed + ".tmp", bed)
    if not os.path.exists(gff):
        synthetic_gff(w, gff + ".tmp")
        os.replace(gff + ".tmp", gff)
    stranded = bool(w.flags & 1)
    kw = dict(annotationFile=gff, isStranded=stranded, strandedType="rf" if stranded else None, ctx=ctx)
    cli.process(bam, bed, outp, **kw)                               # warm-up (page cache, allocations)
    ts = []
    for _ in range(max(1, args.e2e_steps)):
        a = time.perf_counter()
        cli.process(bam, bed, outp, **kw)
        ts.append(time.perf_counter() - a)
    a = time.perf_counter()
    ann = load_annotation(gff)
    b = time.perf_counter()
    with open(bed) as fh:
        chroms, table, sstr = cli.process_table(ctx, bam, fh, annotation=ann, is_stranded=stranded, stranded_type=kw["strandedType"])
    c = time.perf_counter()
    ms_count = ctx.stats()["ms_total"]
    cli.write_process_tsv(outp + ".SpliSER.tsv", chroms, table, sstr, annotation=ann, is_stranded=stranded)
    d = time.perf_counter()
    n_rows = sum(1 for _ in open(outp + ".SpliSER.tsv")) - 1
    step = float(np.mean(ts))
    return {"value": reads / step, "unit": "reads/s", "ms_per_step": 1e3 * step, "rows_written": n_rows, "tsv_bytes": os.path.getsize(outp + ".SpliSER.tsv"),
            "genes": sum(len(g) for g in ann.genes),
            "breakdown_ms": {"annotation": round(1e3 * (b - a), 2), "bed_parse+spl_process": round(1e3 * (c - b), 2), "of_which_spl_process": round(ms_count, 2),
                             "gene_column+tsv_writer": round(1e3 * (d - c), 2)},
            "note": "cli.process(BAM, BED12, GFF) -> .SpliSER.tsv: annotation and BED12 parse (native), spl_process(bam) on the device, "
                    "Gene column + TSV writer (native); byte-identical output is pinned by tests/test_cli_*.py"}


def emit(line):
    """The ONE JSON line goes to the real stdout; everything else a library prints (NCCL banner, warnings) was
    redirected to stderr at start-up."""
    os.write(_REAL_STDOUT, (line + "\n").encode())


_REAL_STDOUT = 1


def reference_arm(args, ncores):
    """The reference's algorithm on the host cores: oracle/spliser_oracle.c (C port, OpenMP over sites).  configs[1] runs in
    full every step; configs[2] is bounded to its first chromosome so that K + W steps end within minutes."""
    from oracle import c_oracle
    from spliser_b200 import synth
    strong = args.gpus > 1 and args.scaling == "strong"
    cfg, desc = workload_config(args.workload, args.reads)
    w = synth.generate(cfg, cache_dir=CACHE)
    if args.workload == "c3" and not args.reference_full:
        rec, junc = first_segment(w)
        sample = "first chromosome of the workload (%s: %d records, %d junctions) per step" % (w.chroms[int(rec.seg_chrom[0])], len(rec), len(junc))
    else:
        rec, junc = w.records, w.junctions
        sample = "the full workload (%d records, %d junctions) per step" % (len(rec), len(junc))
    times = []
    for i in range(args.warmup + args.steps):
        t0 = time.perf_counter()
        res = c_oracle.process(rec, len(w.chroms), junc, w.flags, threads=ncores)
        if i >= args.warmup:
            times.append(time.perf_counter() - t0)
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, res)
    tot = float(sum(times))
    val = len(rec) * len(times) / tot
    if strong:
        desc += " -- ONE sample sharded by genomic tile over %d GPUs" % args.gpus
    emit(json.dumps({
        "impl": "reference", "metric": METRIC, "value": val, "unit": "reads/s", "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * tot / len(times), "higher_is_better": True, "scaling": "strong" if strong else "weak",
        "vs_baseline": None, "dtype": "int64", "data": "synthetic",
        "config": {"workload": desc, "note": "the reference is single-threaded Python + one samtools fork per site and cannot run on this box (no samtools / HTSeq); this arm times the "
                                             "oracle's C port of its algorithm (per-site read fetch + per-CIGAR-op state machine, S:408-639) with OpenMP over sites on every host core"},
        "cpu_baseline": {"value": val, "unit": "reads/s", "cores": ncores, "kind": "port", "sample": sample, "python_reference": python_reference_note()},
        "e2e": {"value": val, "unit": "reads/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0}))


def main():
    global _REAL_STDOUT
    sys.stdout.flush()
    _REAL_STDOUT = os.dup(1)
    os.dup2(2, 1)                      # fd 1 -> stderr for the rest of the process (C libraries included)
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default=None, help="c2 (default at N = 1), c3 (default at N > 1), c1, small, c4 (combine of 48 samples)")
    ap.add_argument("--reads", type=int, default=0, help="records of the sample (default: the named config's size)")
    ap.add_argument("--e2e-steps", type=int, default=3)
    ap.add_argument("--no-cpu-baseline", action="store_true", help="skip the oracle run (parity check + cpu_baseline)")
    ap.add_argument("--no-bam", action="store_true", help="skip the from-a-BAM-file and CLI measurements")
    ap.add_argument("--no-variants", action="store_true", help="skip the stabbing-variant comparison pass")
    ap.add_argument("--reference-full", action="store_true", help="reference arm: the full workload every step even on configs[2]")
    ap.add_argument("--profile", action="store_true", help="resident passes only (for ncu): no e2e, no CPU baseline")
    ap.add_argument("--scaling", default="strong", choices=["weak", "strong"],
                    help="N > 1: strong (default) = ONE sample sharded over the GPUs by genomic tile; weak = one sample per GPU (replicas)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the site table of the last timed step to DIR/<column>.npy (float64, at most 64 MB, a seeded sample above that)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.warmup < 3:
        args.warmup = 3

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    ncores = os.cpu_count() or 1
    if args.workload is None:
        args.workload = "c2" if max(world, args.gpus) == 1 else "c3"
    if args.workload == "c4":
        if args.dump_outputs:
            ap.error("--dump-outputs: the combine workload (c4) writes .combined.tsv files, not a site table")
        import bench_combine
        return bench_combine.run(args, rank, world, local, emit)

    if args.impl == "reference":
        if rank == 0:
            reference_arm(args, ncores)
        return

    # ------------------------------------------------------------------ our arm
    import spliser_b200
    from spliser_b200 import api, dist, synth
    from spliser_b200.api import Records, pinned_empty
    from spliser_b200.dist import Ranks, bind_to_device_node, host_topology
    topo = host_topology(local)
    topo["bound_to_gpu_node"] = bind_to_device_node(topo) if os.environ.get("SPLISER_NUMA_BIND", "1") == "1" else False
    topo.pop("_bind", None)
    ranks = Ranks("nccl" if world > 1 else None)
    strong = args.scaling == "strong" and world > 1
    cfg, desc = workload_config(args.workload, args.reads, 0 if (strong or world == 1) else rank)
    w = generate_once(cfg, ranks) if (strong or world == 1) else synth.generate(cfg, cache_dir=CACHE)
    n_chrom = len(w.chroms)
    n_sample = len(w.records)
    full_records = w.records
    tile = None
    if strong:
        # the same sample on every rank; rank r keeps the records of its read-balanced genomic tile and owns that slice of the site table
        table0 = api.build_site_table(n_chrom, w.junctions, w.flags)
        cuts = dist.balanced_tiles(full_records, table0, n_chrom, world)
        tile = (cuts[rank], cuts[rank + 1])
        w.records = dist.tile_records(full_records, table0, n_chrom, rank, world, site_range=tile, seg_spans=dist.segment_max_spans(full_records))
        # ... and builds its own site table + graph from the junction rows its sites and their partners touch (BED order kept)
        full_junctions = w.junctions
        rows_kept, w.junctions, tile_local = dist.tile_junctions(full_junctions, table0, n_chrom, tile, w.flags)
        desc += " -- ONE sample sharded by genomic tile over %d GPUs" % world
        ctx = spliser_b200.Context(local)
        ctx.set_tile_sites(*tile_local)
    else:
        ctx = spliser_b200.Context(local)
    barrier, max_over_ranks, sum_over_ranks = ranks.barrier, ranks.max, ranks.sum

    sampler = ClockSampler(local)
    # ---- resident: records + junction table in HBM -> SSE in HBM, the whole per-sample path timed
    ctx.resident_load(w.records, n_chrom, w.junctions, w.flags)
    t_load = time.time()
    ctx.resident_count(args.warmup)
    barrier()
    st = ctx.resident_count(args.steps)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, ctx.resident_fetch())
    barrier()
    ms_total = max_over_ranks(st["ms_total"])
    reads_rank = st["n_aligned"]
    reads_all = float(n_sample) if strong else sum_over_ranks(reads_rank)      # strong: the sample counts once, edge duplicates do not
    value = reads_all * args.steps / (ms_total * 1e-3)
    S, E = st["n_sites"], st["n_edges"]
    peak, peak_src = measured_peak()
    kernel_ms = {"site_table+graph (K1)": st["ms_graph_dev"] / args.steps, "k_count_fused": st["ms_beta1"] / args.steps,
                 "k_hot_items": st["ms_spliced"] / args.steps, "memset+scan+beta2+SSE (K5)": st["ms_final"] / args.steps}
    b_m, b_n, r_spl = soa_counts(w.records)
    # SURVEY 8(d): bytes = 9 B_M + 8 B_N + 8 R_spl + 5 S (site table) for the counting kernel; + 12 E + 20 S for the whole path
    k_bytes = 9.0 * b_m + 8.0 * b_n + 8.0 * r_spl + 5.0 * S
    path_bytes = k_bytes + 12.0 * E + 20.0 * S
    rec_bytes = 10.0 * len(w.records) + 4.0 * len(w.records.cigar)
    k_ms = kernel_ms["k_count_fused"]
    k_gbs = k_bytes / (k_ms * 1e-3) / 1e9 if k_ms > 0 else 0.0
    path_ms = st["ms_total"] / args.steps

    if args.profile:
        emit(json.dumps({"profile_run": True, "ms_per_step": ms_total / args.steps, "kernel_ms": kernel_ms, "launches_per_step": st["launches"]}))
        sampler.stop()
        ctx.close()
        ranks.close()
        return

    # ---- the north_star cross-check: the stabbing variant's counting pass over its pre-digested layout (N = 1 only)
    variants = None
    if world == 1 and not args.no_variants:
        try:
            ctx.set_variant("stab")
            ctx.resident_load(w.records, n_chrom, w.junctions, w.flags)
            ctx.resident_count(args.warmup)
            sv = ctx.resident_count(args.steps)
            load_ms = ctx.stats()["ms_expand"]
            stab_table = ctx.resident_fetch()
            variants = {"stab": {"ms_count_pass": sv["ms_total"] / args.steps, "ms_layout_kernels_at_load": load_ms,
                                 "ms_k_beta1_stab": sv["ms_beta1"] / args.steps, "ms_junction_kernels": sv["ms_spliced"] / args.steps,
                                 "digest": table_digest(stab_table),
                                 "note": "block-vs-site stabbing over a bin-partitioned block stream (TMA-staged site tiles): its counting pass needs the layout "
                                         "kernels first (expansion, bin partition, junction grouping), so the per-sample path is their sum"},
                        "fused": {"ms_per_sample_path": path_ms}}
            del stab_table
        finally:
            ctx.set_variant("fused")

    # ---- e2e through the C ABI from pinned host arrays
    r = w.records
    pinned = {}
    for k in ("pos", "flag", "cig_off", "cigar"):
        a = getattr(r, k)
        b = pinned_empty(len(a), a.dtype)
        b[:] = a
        pinned[k] = b
    pr = Records(pinned["pos"], pinned["flag"], pinned["cig_off"], pinned["cigar"], r.seg_chrom, r.seg_off)
    pk = api.PackedRecords.from_records(pr, alloc=pinned_empty)      # the packed host layout (17 B per record), page-locked; shares nothing with pr but the segments
    pk.cigar = pr.cigar                                              # (the CIGAR array is the same in both layouts)
    try:
        ck = api.CompactRecords.from_records(pr, alloc=pinned_empty)  # the compact host layout (about 9 B per record), page-locked
    except ValueError:                                               # a record with more than 255 operators: the packed view is the fallback
        ck = None

    def timed_calls(fn):
        fn()                                                         # warm-up (allocations)
        barrier()
        ts, st_, tab = [], None, None
        for _ in range(max(1, args.e2e_steps)):
            tab = None                   # the previous sample's result is released before the next call (its pinned arena is reused)
            barrier()
            a = time.perf_counter()
            tab = fn()
            ts.append(time.perf_counter() - a)
            st_ = ctx.stats()
        return max_over_ranks(float(np.mean(ts))), st_, tab

    plain_step, plain_stats, table = timed_calls(lambda: ctx.process_records(pr, n_chrom, w.junctions, w.flags))
    plain_digest = table_digest(table)
    table = None
    packed_step, packed_stats, table = timed_calls(lambda: ctx.process_packed(pk, n_chrom, w.junctions, w.flags))
    packed_digest = table_digest(table)
    if ck is not None:
        table = None
        e2e_step, stats, table = timed_calls(lambda: ctx.process_compact(ck, n_chrom, w.junctions, w.flags))
    else:
        e2e_step, stats = packed_step, packed_stats
    e2e_val = reads_all / e2e_step
    clocks = sampler.window(t_load, time.time())
    clocks["window"] = "warm-up + timed passes + e2e calls"
    if variants is not None:
        variants["fused"]["digest"] = table_digest(table)
        variants["identical"] = variants["fused"]["digest"] == variants["stab"]["digest"]

    out = {
        "metric": METRIC, "value": value, "unit": "reads/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": ms_total / args.steps, "higher_is_better": True, "scaling": "strong" if strong else "weak", "vs_baseline": None,
        "dtype": "u32", "data": "synthetic",
        "config": {"workload": desc, "records_per_gpu": int(reads_rank), "sites": len(table0) if strong else int(S),
                   "junction_rows": len(full_junctions) if strong else len(w.junctions),
                   "tile_sites": list(tile) if tile else None,
                   "tile_graph": {"junction_rows_of_the_sample": len(full_junctions), "junction_rows_of_this_tile": len(w.junctions),
                                  "sites_of_this_tile_table": int(S), "owned_slice_of_it": list(tile_local),
                                  "note": "every rank builds the site table + competing-site graph of ITS tile from the junction rows that touch "
                                          "its sites or their partners (dist.tile_junctions); owned rows are identical to the full table's"} if tile else None,
                   "l2": "no flush needed: every pass streams %.0f MB of records, larger than the 126 MB L2" % (rec_bytes / 1e6),
                   "host": topo,
                   "timing": "CUDA events on the library's stream around %d passes; max over ranks" % args.steps,
                   "value_scope": "records + junction table resident in HBM -> per-site table in HBM, every per-sample kernel inside the timed region: site table + "
                                  "competing-site graph build (K1, %s), counter memset, fused counting kernel, prefix scan + beta2 gather + SSE; only the copies "
                                  "are outside (they are inside e2e)" % ("rebuilt every pass" if st.get("graph_timed") else "NOT rebuilt: host-built graph")},
        "clocks": clocks,
        "e2e": {"value": e2e_val, "unit": "reads/s", "h2d_bytes_per_step": int(stats["h2d_bytes"]), "d2h_bytes_per_step": int(stats["d2h_bytes"]),
                "ms_per_step": 1e3 * e2e_step, "parts": int(stats["n_parts"]),
                "breakdown_ms": {k: round(stats[k], 3) for k in ("ms_total", "ms_graph", "ms_upload", "ms_count")},
                "graph_on_device": bool(stats["graph_on_device"]),
                "entry_point": "spl_process_compact" if ck is not None else "spl_process_packed",
                "bytes_per_record_on_the_wire": round(float(stats["h2d_bytes"]) / max(1, len(r)), 2),
                "note": "host wall clock around spl_process_compact (POS as 16-bit offsets per stride of 1024 records, operator count in a byte, 16-bit CIGAR operators "
                        "with a 32-bit stream for records with a long one): junction table -> site table + graph (device), pinned H2D of the records in slabs with the "
                        "unpack + counting kernels of a slab under the copy of the next, finalize, D2H of the table",
                "packed_view": {"ms_per_step": 1e3 * packed_step, "h2d_bytes_per_step": int(packed_stats["h2d_bytes"]), "identical_table": packed_digest == table_digest(table),
                                "note": "the same through spl_process_packed (17 B per record: POS i32, three flag bits, operator count u16, CIGAR words)"},
                "plain_view": {"ms_per_step": 1e3 * plain_step, "h2d_bytes_per_step": int(plain_stats["h2d_bytes"]), "identical_table": plain_digest == table_digest(table),
                               "note": "the same through spl_process_records (20 B per record: POS i32, FLAG u16, cig_off u32, CIGAR words)"}},
        "gpu_launches": int(round(st["launches"] * args.steps)),
        "launches_per_step": st["launches"],
        "roofline": {"bound": "hbm", "kernel": "k_count_fused", "achieved": k_gbs, "peak": peak, "unit": "GB/s",
                     "frac": k_gbs / peak, "traffic": traffic_from_profile("k_count_fused"), "algorithmic_bytes_per_launch": k_bytes,
                     "ms_per_launch": k_ms, "peak_source": peak_src,
                     "bytes_definition": "SURVEY 8(d): 9 B per M/=/X block + 8 B per N + 8 B per spliced read + 5 B per site; the kernel streams the more compact "
                                         "record layout (10 B per record + 4 B per CIGAR operator = %.0f MB per launch)" % (rec_bytes / 1e6),
                     "record_bytes_per_launch": rec_bytes, "achieved_on_record_bytes_gbs": rec_bytes / (k_ms * 1e-3) / 1e9 if k_ms > 0 else 0.0},
        "roofline_path": {"algorithmic_bytes_per_step": path_bytes, "ms_per_step": path_ms, "traffic": traffic_from_profile("step") if world == 1 and args.workload == "c2" else None,
                          "achieved_gbs": path_bytes / (path_ms * 1e-3) / 1e9, "frac": path_bytes / (path_ms * 1e-3) / 1e9 / peak,
                          "kernel_ms": kernel_ms},
        "kernel_path": {"n_mblocks": b_m, "n_junction_ops": b_n, "n_spliced_reads": r_spl, "n_edges": int(E), "n_cigar_ops": int(len(w.records.cigar))},
        "variants": variants,
        "checksum": {k: int(getattr(table, k)[slice(*tile_local) if strong else slice(None)].sum()) for k in ("beta1", "beta2simple", "alpha")},
    }

    # ---- parity inside the measurement + CPU baseline on the SAME workload
    if strong:
        # the owned slices of every rank concatenate to the table one GPU computes for the whole sample
        part = dist.owned_part(table, tile_local, rows_kept)
        np.savez(os.path.join(CACHE, "tile_%d_of_%d.npz" % (rank, world)), **part)
        barrier()
        if rank == 0:
            from oracle import c_oracle
            parts = [dict(np.load(os.path.join(CACHE, "tile_%d_of_%d.npz" % (q, world)))) for q in range(world)]
            ctx.set_tile_sites(-1, -1)
            whole = ctx.process_records(full_records, n_chrom, full_junctions, w.flags)
            cat = dist.concat_parts(parts, c_oracle.table_dict(whole))
            d = c_oracle.diff_tables(cat, c_oracle.table_dict(whole))
            out["parity_checked"] = d is None
            out["parity"] = {"against": "the untiled single-GPU table of the same sample (rank 0): the owned rows of the %d per-tile tables (each built from the tile's own "
                                        "junction rows), concatenated, every column incl. Partners / PartnerCounts / CompetitorPos" % world,
                             "tiles_digest": table_digest(cat), "single_gpu_digest": table_digest(whole), "first_difference": d}
            table = whole
            # the same sample, untiled, on ONE GPU through the same timed path: the denominator of the strong-scaling efficiency
            ctx.resident_load(full_records, n_chrom, full_junctions, w.flags)
            ctx.resident_count(args.warmup)
            s1 = ctx.resident_count(args.steps)
            v1 = n_sample * args.steps / (s1["ms_total"] * 1e-3)
            out["strong_scaling"] = {"value_1gpu_same_workload": v1, "ms_per_step_1gpu": s1["ms_total"] / args.steps, "speedup": value / v1,
                                     "efficiency": value / v1 / world,
                                     "kernel_ms_1gpu": {"site_table+graph (K1)": s1["ms_graph_dev"] / args.steps, "k_count_fused": s1["ms_beta1"] / args.steps,
                                                        "k_hot_items": s1["ms_spliced"] / args.steps, "memset+scan+beta2+SSE (K5)": s1["ms_final"] / args.steps},
                                     "note": "rank 0 times the untiled sample (all records, all junction rows) on its GPU after the tiled measurement"}
        sent = sum_over_ranks(float(len(w.records)))
        if rank == 0:
            out["parity"]["records_sent"] = int(sent)
            out["parity"]["edge_duplication"] = sent / n_sample - 1.0
    if rank == 0 and not args.no_cpu_baseline:
        from oracle import c_oracle
        if args.workload == "c3":
            # bounded: the first chromosome of the sample (its sites are the first rows of the table)
            rec_s, junc_s = first_segment(Workload_like(full_records, full_junctions if strong else w.junctions))
            sample = "first chromosome of the sample (%d records, %d junctions)" % (len(rec_s), len(junc_s))
            t0 = time.perf_counter()
            want = c_oracle.process(rec_s, n_chrom, junc_s, w.flags, threads=ncores)
            dt = time.perf_counter() - t0
            ns = len(want["pos"])
            got = c_oracle.table_dict(table)
            sub_ok = all(np.array_equal(np.asarray(got[k][:ns]).view(np.int64) if np.asarray(got[k]).dtype.kind == "f" else np.asarray(got[k][:ns]),
                                        np.asarray(want[k]).view(np.int64) if np.asarray(want[k]).dtype.kind == "f" else np.asarray(want[k]))
                         for k in ("pos", "alpha", "beta1", "beta2simple", "beta2cryptic", "sse"))
            out.setdefault("parity", {})["oracle_subset"] = {"against": "oracle/spliser_oracle.c on " + sample + ": the first %d rows of the table" % ns, "identical": bool(sub_ok)}
            out["parity_checked"] = bool(out.get("parity_checked", True) and sub_ok)
            out["cpu_baseline"] = {"value": len(rec_s) / dt, "unit": "reads/s", "cores": ncores, "kind": "port", "sample": sample, "python_reference": python_reference_note()}
        else:
            t0 = time.perf_counter()
            want = c_oracle.process(full_records, n_chrom, w.junctions, w.flags, threads=ncores)
            dt = time.perf_counter() - t0
            diff = c_oracle.diff_tables(c_oracle.table_dict(table), want)
            out["parity_checked"] = diff is None
            out["parity"] = {"against": "oracle/spliser_oracle.c (C port of the reference, pinned to the reference's golden vectors) on the same full workload, every column, floats bit for bit",
                             "table_digest": table_digest(table), "oracle_digest": table_digest(want), "first_difference": diff}
            out["cpu_baseline"] = {"value": n_sample / dt, "unit": "reads/s", "cores": ncores, "kind": "port",
                                   "sample": "the full workload, once (%d records, %d junctions, %.1f s): C port of the reference algorithm, OpenMP over sites" % (n_sample, len(w.junctions), dt),
                                   "python_reference": python_reference_note()}
    elif rank == 0:
        out["cpu_baseline"] = None

    # ---- the same call from a BAM FILE (spl_process): BGZF inflate + record parse on the device vs the host reader
    if world == 1 and not args.no_bam:
        try:
            bam = os.path.join(CACHE, "bench_%s_%d.bam" % (args.workload, len(r)))
            if not os.path.exists(bam):
                os.makedirs(CACHE, exist_ok=True)
                r.write_bam(bam + ".tmp", w.chroms, w.chrom_len)
                os.replace(bam + ".tmp", bam)
            table = None
            ctx.process_bam(bam, w.chroms, w.junctions, w.flags)       # warm-up (allocations, page cache)
            tb = []
            table_b = None
            for _ in range(max(1, args.e2e_steps)):
                table_b = None                    # release the previous result first (its pinned arena is reused)
                a = time.perf_counter()
                table_b = ctx.process_bam(bam, w.chroms, w.junctions, w.flags)
                tb.append(time.perf_counter() - a)
                sb = ctx.stats()
            os.environ["SPLISER_HOST_BAM"] = "1"
            a = time.perf_counter()
            th = ctx.process_bam(bam, w.chroms, w.junctions, w.flags)
            host_s = time.perf_counter() - a
            sh = ctx.stats()
            del os.environ["SPLISER_HOST_BAM"]
            out["bam_e2e"] = {"value": reads_rank / float(np.mean(tb)), "unit": "reads/s", "ms_per_step": 1e3 * float(np.mean(tb)),
                              "bam_bytes": os.path.getsize(bam), "bam_on_device": bool(sb["bam_on_device"]), "ms_ingest": round(sb["ms_decode"], 3),
                              "host_reader": {"ms_per_step": 1e3 * host_s, "ms_decode": round(sh["ms_decode"], 3), "threads": ncores},
                              "identical_to_host_reader": bool(np.array_equal(th.beta1, table_b.beta1) and np.array_equal(th.beta2simple, table_b.beta2simple)
                                                                and np.array_equal(th.sse, table_b.sse)),
                              "note": "spl_process(bam_path): file image -> pinned -> H2D, BGZF inflate + BAM parse on the device, then the same path as e2e; "
                                      "synthetic BAM without SEQ/QUAL (records only), so the file is much smaller than a sequencer's"}
        except Exception as ex:                                      # never lose the main line over the extra measurement
            out["bam_e2e"] = {"error": repr(ex)}
        # ---- the same from a sequencer-shaped BAM (read names, SEQ, QUAL): the first 8M records of the sample
        try:
            n_seq = min(len(r), 8_000_000)
            sub = Records(r.pos[:n_seq], r.flag[:n_seq], r.cig_off[:n_seq + 1], r.cigar[:int(r.cig_off[n_seq])],
                          *_cut_segments(r, n_seq))
            seq_bam = os.path.join(CACHE, "bench_%s_%d_seq.bam" % (args.workload, n_seq))
            if not os.path.exists(seq_bam):
                sub.write_bam(seq_bam + ".tmp", w.chroms, w.chrom_len, with_seq=True)
                os.replace(seq_bam + ".tmp", seq_bam)
            op = sub.cigar & 15
            qop = np.where((op == 0) | (op == 1) | (op == 4) | (op == 7) | (op == 8), sub.cigar >> 4, 0).astype(np.int64)
            qs = np.concatenate([[0], np.cumsum(qop)])
            qlen = qs[sub.cig_off[1:].astype(np.int64)] - qs[sub.cig_off[:-1].astype(np.int64)]
            inflated = int((36 + 11 + 4 * np.diff(sub.cig_off.astype(np.int64)) + (qlen + 1) // 2 + qlen).sum())
            ctx.process_bam(seq_bam, w.chroms, w.junctions, w.flags)
            ts = []
            for _ in range(max(1, args.e2e_steps)):
                a = time.perf_counter()
                ts_table = ctx.process_bam(seq_bam, w.chroms, w.junctions, w.flags)
                ts.append(time.perf_counter() - a)
                ss = ctx.stats()
                del ts_table
            want_seq = ctx.process_records(sub, n_chrom, w.junctions, w.flags)
            got_seq = ctx.process_bam(seq_bam, w.chroms, w.junctions, w.flags)
            out["bam_e2e_seq"] = {"records": n_seq, "value": n_seq / float(np.mean(ts)), "unit": "reads/s", "ms_per_step": 1e3 * float(np.mean(ts)),
                                  "bam_bytes": os.path.getsize(seq_bam), "inflated_bytes": inflated, "ms_ingest": round(ss["ms_decode"], 3),
                                  "bam_on_device": bool(ss["bam_on_device"]),
                                  "inflated_gb_per_s_of_ingest": inflated / (ss["ms_decode"] * 1e-3) / 1e9 if ss["ms_decode"] > 0 else None,
                                  "identical_to_records_path": bool(np.array_equal(want_seq.beta1, got_seq.beta1) and np.array_equal(want_seq.beta2simple, got_seq.beta2simple)
                                                                    and np.array_equal(want_seq.sse, got_seq.sse)),
                                  "note": "a sequencer-shaped file: read names, SEQ and QUAL of the CIGAR's query length (seeded pseudo-random bases, slowly changing "
                                          "qualities), so the BGZF members are mostly literals and the inflated stream is ~8 x the records-only file's per record"}
            del want_seq, got_seq
        except Exception as ex:
            out["bam_e2e_seq"] = {"error": repr(ex)}
        # ---- the whole `process` command: BAM + BED12 + GFF files -> .SpliSER.tsv on disk (what a SpliSER user runs)
        try:
            out["cli_e2e"] = cli_process_run(ctx, w, bam, args, reads_rank)
        except Exception as ex:
            out["cli_e2e"] = {"error": repr(ex)}
    sampler.stop()
    if rank == 0:
        emit(json.dumps(out))
    ctx.close()
    ranks.close()


def _cut_segments(r, n):
    """(seg_chrom, seg_off) of the first n records of r."""
    k = int(np.searchsorted(np.asarray(r.seg_off), n, side="left"))
    off = [int(x) for x in r.seg_off[:k]] + [n]
    return [int(c) for c in r.seg_chrom[:len(off) - 1]], off


class Workload_like:
    def __init__(self, records, junctions):
        self.records, self.junctions = records, junctions


if __name__ == "__main__":
    main()
