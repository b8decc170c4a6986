"""What inferring the library type costs, on the configs[1] BAM (synth.config_c2: 40M records, seed 20260002; the file bench.py's
bam_e2e reads), in two copies: as written (annotation source, genes of bench.synthetic_gff) and with an XS:A tag on every spliced
record (XS source, the transcript strand a dUTP library's aligner writes).

  (a) k_strand_votes alone: CUDA events around the kernel (SPL_STAT_MS_STRAND_VOTES), on a resident sample (DeviceSample.infer_strand)
      and through the path call with its ingest (Context.infer_strand_bam), both sources
  (b) processBam --isStranded -s rf against -s auto on the XS copy without -A: host clock around the whole command, 2 warm-up
      rounds, then alternating timed rounds; the two .SpliSER.tsv files must be the same bytes

Records the GPU name and power limit of the run.

    python profiles/tools/strand_votes.py [--records 40000000] [--steps 5] [--out profiles/strand_votes_c2.json]
"""
import argparse
import contextlib
import io
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
import spliser_b200  # noqa: E402
from spliser_b200 import api, cli, synth  # noqa: E402
from spliser_b200.genes import load_annotation  # noqa: E402

CACHE = os.environ.get("SPLISER_BENCH_CACHE", os.path.join(tempfile.gettempdir(), "spliser_bench_cache"))


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
    if q.returncode != 0 or not q.stdout.strip():
        raise RuntimeError("no GPU visible to nvidia-smi: this measurement needs the B200")
    name, power, clk = [x.strip() for x in q.stdout.strip().splitlines()[0].split(",")]
    return {"name": name, "power_limit": power, "max_sm_clock": clk}


def xs_aux(rec):
    """(aux offsets, aux bytes) with XS:A:<rf strand> on every spliced record (the synthetic FLAGs are dUTP-style)."""
    off = rec.cig_off.astype(np.int64)
    spliced = np.zeros(len(rec), bool)
    spliced[np.searchsorted(off, np.flatnonzero((rec.cigar & 15) == 3), side="right") - 1] = True
    f = rec.flag.astype(np.int64)
    fr_plus = (((f & 64) != 0) | ((f & 1) == 0)) != ((f & 16) != 0)
    aux_off = np.zeros(len(rec) + 1, np.int64)
    aux_off[1:] = np.cumsum(np.where(spliced, 4, 0))
    blob = np.zeros((int(spliced.sum()), 4), np.uint8)
    blob[:, 0], blob[:, 1], blob[:, 2] = ord("X"), ord("S"), ord("A")
    blob[:, 3] = np.where(fr_plus[spliced], ord("-"), ord("+"))
    return aux_off, blob.reshape(-1)


def summary(xs):
    return {"mean": float(np.mean(xs)), "min": float(np.min(xs)), "max": float(np.max(xs)), "n": len(xs)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--records", type=int, default=40_000_000)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "strand_votes_c2.json"))
    args = ap.parse_args()
    gpu = gpu_info()
    sys.path.insert(0, ROOT)
    import bench
    cfg = synth.config_c2(args.records)
    w = synth.generate(cfg, cache_dir=CACHE)
    os.makedirs(CACHE, exist_ok=True)
    bam = os.path.join(CACHE, "bam_only_%s_%d.bam" % (cfg.key(), len(w.records)))
    if not os.path.exists(bam):
        w.records.write_bam(bam + ".tmp", w.chroms, w.chrom_len)
        os.replace(bam + ".tmp", bam)
    bam_xs = os.path.join(CACHE, "strand_votes_xs_%s_%d.bam" % (cfg.key(), len(w.records)))
    if not os.path.exists(bam_xs):
        w.records.write_bam(bam_xs + ".tmp", w.chroms, w.chrom_len, aux=xs_aux(w.records))
        os.replace(bam_xs + ".tmp", bam_xs)
    gff = os.path.join(CACHE, "strand_votes_%s.gff" % cfg.key())
    bench.synthetic_gff(w, gff)
    chroms = w.chroms
    genes = api.gene_strands(load_annotation(gff), chroms)
    out_dir = tempfile.mkdtemp(prefix="strand_votes_")
    res = {"what": "library-type inference on configs[1] (synth.config_c2, %d records, seed %d)" % (len(w.records), cfg.seed),
           "gpu": gpu, "records": len(w.records), "genes": int(len(genes.left)),
           "bam_bytes": os.path.getsize(bam), "bam_xs_bytes": os.path.getsize(bam_xs)}
    with spliser_b200.Context(0) as ctx:
        # (a) the kernel: resident samples, then the path call
        for src, path, g in (("annotation", bam, genes), ("xs", bam_xs, None)):
            with ctx.load_bam(path, xs=g is None) as s:
                for _ in range(args.warmup):
                    s.infer_strand(chroms, g)
                ev, wall = [], []
                for _ in range(args.steps):
                    t0 = time.perf_counter()
                    v = s.infer_strand(chroms, g)
                    wall.append(1e3 * (time.perf_counter() - t0))
                    ev.append(ctx.stats()["ms_strand_votes"])
            path_ev, path_wall = [], []
            for _ in range(max(2, args.steps // 2)):
                t0 = time.perf_counter()
                pv = ctx.infer_strand_bam(path, chroms, g)
                path_wall.append(1e3 * (time.perf_counter() - t0))
                path_ev.append(ctx.stats()["ms_strand_votes"])
            assert pv == v, (pv, v)
            res["a_" + src] = {"votes": v.__dict__, "verdict": api.library_type(v),
                               "resident_kernel_ms": summary(ev), "resident_call_ms": summary(wall),
                               "path_kernel_ms": summary(path_ev), "path_call_ms": summary(path_wall)}
        # (b) processBam -s rf against -s auto (XS copy, no annotation)
        def run(stype, tag):
            with contextlib.redirect_stdout(io.StringIO()):
                t0 = time.perf_counter()
                cli.processBam(bam_xs, os.path.join(out_dir, tag), isStranded=True, strandedType=stype, ctx=ctx)
                return 1e3 * (time.perf_counter() - t0)
        for _ in range(args.warmup):
            run("rf", "rf")
            run("auto", "auto")
        t_rf, t_auto = [], []
        for _ in range(args.steps):
            t_rf.append(run("rf", "rf"))
            t_auto.append(run("auto", "auto"))
        with open(os.path.join(out_dir, "rf.SpliSER.tsv"), "rb") as a, open(os.path.join(out_dir, "auto.SpliSER.tsv"), "rb") as b:
            identical = a.read() == b.read()
        res["b_process_bam"] = {"rf_ms": summary(t_rf), "auto_ms": summary(t_auto),
                                "auto_minus_rf_ms_mean": float(np.mean(t_auto) - np.mean(t_rf)), "identical_tsv": identical,
                                "how": "host clock around cli.processBam on one context, %d warm-up rounds, %d alternating timed rounds"
                                       % (args.warmup, args.steps)}
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as fh:
        json.dump(res, fh, indent=1)
    print(json.dumps(res))
    if not identical:
        sys.exit("processBam -s auto and -s rf differ")


if __name__ == "__main__":
    main()
