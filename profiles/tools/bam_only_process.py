"""`process` from a BAM alone, timed on the configs[1] BAM (synth.config_c2: 40M records, seed 20260002; the file bench.py's
bam_e2e reads):

  (a) extract_junctions_bam + process_bam   -- two ingests of the file
  (b) process_bam_extract                   -- one ingest: extract, filter, count on the same device-resident records
  (c) CUDA events around the extraction kernels (anchor-extent walk included, and alone), from the library's stats

Host clock around calls that end in a device synchronise, after warm-up; (a) and (b) alternate.  Checks that (a) and (b)
return the same junction table (extents included) and the same site table.  Records the GPU name and power limit of the run.

    python profiles/tools/bam_only_process.py [--records 40000000] [--steps 10] [--out profiles/bam_only_process_c2.json]
"""
import argparse
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
from spliser_b200 import synth  # noqa: E402

CACHE = os.environ.get("SPLISER_BENCH_CACHE", os.path.join(tempfile.gettempdir(), "spliser_bench_cache"))
TABLE = ("chrom", "pos", "strand", "first_line", "alpha", "beta1", "beta2simple", "beta2cryptic", "beta2weighted", "sse",
         "partner_off", "partner_pos", "partner_cnt", "comp_off", "comp_pos")
JUNC = ("chrom", "left", "right", "score", "strand", "start", "end")


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
    if q.returncode != 0 or not q.stdout.strip():
        raise RuntimeError("no GPU visible to nvidia-smi: this measurement needs the B200")
    name, power, clk = [x.strip() for x in q.stdout.strip().splitlines()[0].split(",")]
    return {"name": name, "power_limit": power, "max_sm_clock": clk}


def same(a, b, fields):
    return all(np.array_equal(np.asarray(getattr(a, k)), np.asarray(getattr(b, k))) for k in fields)


def stats_of(s):
    return {k: round(s[k], 4) for k in ("ms_total", "ms_decode", "ms_extract", "ms_extents", "n_junctions", "h2d_bytes", "bam_on_device")}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--records", type=int, default=40_000_000)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "bam_only_process_c2.json"))
    args = ap.parse_args()
    gpu = gpu_info()
    cfg = synth.config_c2(args.records)
    w = synth.generate(cfg, cache_dir=CACHE)
    bam = os.path.join(CACHE, "bam_only_%s_%d.bam" % (cfg.key(), len(w.records)))
    if not os.path.exists(bam):
        os.makedirs(CACHE, exist_ok=True)
        w.records.write_bam(bam + ".tmp", w.chroms, w.chrom_len)
        os.replace(bam + ".tmp", bam)
    chroms, flags = w.chroms, w.flags

    with spliser_b200.Context(0) as ctx:
        def two_ingests():
            j = ctx.extract_junctions_bam(bam, chroms, flags & 3)
            s_ex = ctx.stats()
            t = ctx.process_bam(bam, chroms, j, flags)
            return j, t, s_ex, ctx.stats()

        def one_ingest():
            j, t = ctx.process_bam_extract(bam, chroms, flags)
            return j, t, ctx.stats()

        for _ in range(args.warmup):
            two_ingests()
            one_ingest()
        ta, tb, st_a, st_b = [], [], [], []
        ja = tbl_a = jb = tbl_b = None
        for _ in range(args.steps):
            ja = tbl_a = None
            t0 = time.perf_counter()
            ja, tbl_a, s_ex, s_pr = two_ingests()
            ta.append(time.perf_counter() - t0)
            st_a.append((s_ex, s_pr))
            jb = tbl_b = None
            t0 = time.perf_counter()
            jb, tbl_b, s = one_ingest()
            tb.append(time.perf_counter() - t0)
            st_b.append(s)
        identical = same(ja, jb, JUNC) and same(tbl_a, tbl_b, TABLE)
        ms_ex = [s["ms_extract"] for s in st_b] + [s[0]["ms_extract"] for s in st_a]
        ms_xt = [s["ms_extents"] for s in st_b] + [s[0]["ms_extents"] for s in st_a]
        res = {
            "what": "process from a BAM alone on configs[1] (synth.config_c2, %d records, seed %d): (a) extract_junctions_bam + "
                    "process_bam, two ingests; (b) process_bam_extract, one ingest; host clock around calls ending in a device "
                    "synchronise, %d warm-up rounds, %d alternating timed rounds; (c) CUDA events around the extraction kernels"
                    % (len(w.records), cfg.seed, args.warmup, args.steps),
            "gpu": gpu,
            "bam_bytes": os.path.getsize(bam),
            "records": len(w.records), "junctions": len(jb), "sites": len(tbl_b),
            "a_two_ingests_ms": {"mean": 1e3 * float(np.mean(ta)), "min": 1e3 * float(np.min(ta)), "max": 1e3 * float(np.max(ta))},
            "b_one_ingest_ms": {"mean": 1e3 * float(np.mean(tb)), "min": 1e3 * float(np.min(tb)), "max": 1e3 * float(np.max(tb))},
            "saved_ms_mean": 1e3 * float(np.mean(ta) - np.mean(tb)),
            "c_extraction_kernels_ms": {"mean": float(np.mean(ms_ex)), "min": float(np.min(ms_ex)), "max": float(np.max(ms_ex))},
            "c_extent_walk_ms": {"mean": float(np.mean(ms_xt)), "min": float(np.min(ms_xt)), "max": float(np.max(ms_xt))},
            "a_stats_last": {"extract": stats_of(st_a[-1][0]), "process": stats_of(st_a[-1][1])},
            "b_stats_last": stats_of(st_b[-1]),
            "identical_tables": bool(identical),
        }
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as fh:
        json.dump(res, fh, indent=1)
    print(json.dumps(res))
    if not identical:
        sys.exit("(a) and (b) differ")


if __name__ == "__main__":
    main()
