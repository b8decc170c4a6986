"""The read filter at ingest (samtools view -q 10 -F 0x904 done by the ingest itself), timed on a BAM of bench size: the
configs[1] records (synth.config_c2: 40M records, seed 20260002, the records bench.py's bam_e2e reads) with a realistic MAPQ /
FLAG mix added -- MAPQ drawn from {0 (5 %), 1 (3 %), 3 (7 %), 60 (25 %), 255 (60 %)}, secondary (0x100, 4 %), supplementary
(0x800, 1 %), duplicate (0x400, 8 %) and QC-fail (0x200, 0.5 %) bits.

  (a) processBam without a filter
  (b) processBam --minMAPQ 10 --excludeFlags 0x904

Host clock around cli.processBam on one context (the call ends in a device synchronise), SPL_STAT_MS_DECODE (the ingest, host
wall ms until the records are on the device) from the library's stats; (a) and (b) alternate after warm-up.  Checks the kept /
dropped counts against a numpy restatement of the rule.  Records the GPU name and power limit of the run.

    python profiles/tools/read_filter.py [--records 40000000] [--steps 5] [--out profiles/read_filter_c2.json]
"""
import argparse
import contextlib
import io
import json
import os
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "profiles", "tools"))
import spliser_b200  # noqa: E402
from spliser_b200 import cli, synth  # noqa: E402
from bam_only_process import CACHE, gpu_info  # noqa: E402

FILTER = spliser_b200.ReadFilter(10, 0x904)
MAPQ_MIX = ((0, 0.05), (1, 0.03), (3, 0.07), (60, 0.25), (255, 0.60))
FLAG_MIX = ((0x100, 0.04), (0x800, 0.01), (0x400, 0.08), (0x200, 0.005))


def realistic_mix(rec, seed):
    rng = np.random.default_rng(seed)
    mapq = rng.choice([q for q, _ in MAPQ_MIX], len(rec), p=[p for _, p in MAPQ_MIX]).astype(np.uint8)
    flag = rec.flag.copy()
    for bit, p in FLAG_MIX:
        flag[rng.random(len(rec)) < p] |= bit
    return flag, mapq


def spread(xs):
    return {"mean": float(np.mean(xs)), "min": float(np.min(xs)), "max": float(np.max(xs))}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--records", type=int, default=40_000_000)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=1)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "read_filter_c2.json"))
    args = ap.parse_args()
    gpu = gpu_info()
    cfg = synth.config_c2(args.records)
    w = synth.generate(cfg, cache_dir=CACHE)
    r = w.records
    flag, mapq = realistic_mix(r, cfg.seed)
    bam = os.path.join(CACHE, "read_filter_%s_%d.bam" % (cfg.key(), len(r)))
    if not os.path.exists(bam):
        os.makedirs(CACHE, exist_ok=True)
        spliser_b200.Records(r.pos, flag, r.cig_off, r.cigar, r.seg_chrom, r.seg_off).write_bam(bam + ".tmp", w.chroms, w.chrom_len,
                                                                                                 mapq=mapq)
        os.replace(bam + ".tmp", bam)
    f32 = flag.astype(np.uint32)
    m = (mapq >= FILTER.min_mapq) & ((f32 & FILTER.exclude_flags) == 0)
    want = (int(m.sum()), int((~m).sum()))

    out_dir = tempfile.mkdtemp(prefix="read_filter_")
    with spliser_b200.Context(0) as ctx:
        def run(rf):
            ctx.set_read_filter(rf or spliser_b200.ReadFilter())
            t0 = time.perf_counter()
            with contextlib.redirect_stdout(io.StringIO()):
                cli.processBam(bam, os.path.join(out_dir, "x"), ctx=ctx, read_filter=rf)
            dt = time.perf_counter() - t0
            s = ctx.stats()
            return dt, s["ms_decode"], s["bam_on_device"], ctx.last_read_filter()

        for _ in range(args.warmup):
            run(None)
            run(FILTER)
        wall = {"a": [], "b": []}
        dec = {"a": [], "b": []}
        counts, on_dev = {}, set()
        for _ in range(args.steps):
            for key, rf in (("a", None), ("b", FILTER)):
                dt, ms, dev, cnt = run(rf)
                wall[key].append(1e3 * dt)
                dec[key].append(ms)
                counts[key] = cnt
                on_dev.add(dev)
    res = {
        "what": "processBam on configs[1]'s records (synth.config_c2, %d records, seed %d) with a realistic MAPQ / FLAG mix: (a) no "
                "filter, (b) --minMAPQ 10 --excludeFlags 0x904; host clock around cli.processBam on one context and "
                "SPL_STAT_MS_DECODE (ingest), %d warm-up rounds, %d alternating timed rounds" % (len(r), cfg.seed, args.warmup, args.steps),
        "gpu": gpu,
        "bam_bytes": os.path.getsize(bam),
        "mapq_mix": dict((str(q), p) for q, p in MAPQ_MIX), "flag_mix": dict((hex(b), p) for b, p in FLAG_MIX),
        "records": len(r),
        "a_no_filter": {"processBam_ms": spread(wall["a"]), "ingest_ms": spread(dec["a"]), "kept_dropped": list(counts["a"])},
        "b_q10_F0x904": {"processBam_ms": spread(wall["b"]), "ingest_ms": spread(dec["b"]), "kept_dropped": list(counts["b"])},
        "expected_kept_dropped_b": list(want),
        "ingest_on_device": sorted(on_dev),
        "counts_match": counts["b"] == want and counts["a"] == (len(r), 0),
    }
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as fh:
        json.dump(res, fh, indent=1)
    print(json.dumps(res))
    if not res["counts_match"]:
        sys.exit("kept / dropped counts differ from the restatement")


if __name__ == "__main__":
    main()
