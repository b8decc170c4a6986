"""Samples told apart by an aux tag (combineGroups), timed on a sequencer-shaped BAM of bench size: configs[1]'s records
(synth.config_c2: 40M records, seed 20260002) written with SEQ / QUAL and a CB:Z cell barcode per record (4000 barcodes drawn
uniformly; the aux column is built with numpy in write_bam's (offsets, blob) form).  Barcode b belongs to group b % G.

  (1) ingest: Context.load_bam (no lookup) against Context.load_bam_groups at G = 16 and G = 1000 (lookup + split), host clock
      around the call (it ends in a device synchronise) and SPL_STAT_MS_DECODE, alternated after warm-up
  (2) the k_group_* kernels and k_bam_fill (with and without the lookup): torch.profiler with CUDA activities, in a run of its
      own, one load_bam and one split per G
  (3) combineGroups at G = 16 against combineBam over the 16 pre-split group BAMs (written from the same records), host clock,
      alternated; the outputs are compared byte for byte
  (4) where each command's time goes: a fresh context's first split against its second (and the first of 16 load_bam calls on
      the group BAMs), and cProfile of one run of each command by the Python calls into the library and the writers

Checks the per-group counts against numpy.  Records the GPU name and power limit of the run.

    python profiles/tools/tag_groups.py [--records 40000000] [--steps 3] [--out profiles/tag_groups_c2.json]
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
from spliser_b200 import api, cli, synth  # noqa: E402
from bam_only_process import CACHE, gpu_info  # noqa: E402

N_BARCODES = 4000


def spread(xs):
    return {"mean": float(np.mean(xs)), "min": float(np.min(xs)), "max": float(np.max(xs)), "n": len(xs)}


def subset(r, idx):
    off = r.cig_off.astype(np.int64)
    n_op = off[idx + 1] - off[idx]
    starts = np.repeat(off[idx], n_op)
    within = np.arange(int(n_op.sum())) - np.repeat(np.cumsum(n_op) - n_op, n_op)
    chrom = np.repeat(r.seg_chrom, np.diff(r.seg_off))[idx]
    seg = np.flatnonzero(np.r_[True, chrom[1:] != chrom[:-1]]) if len(idx) else np.zeros(0, np.int64)
    return spliser_b200.Records(r.pos[idx], r.flag[idx], np.r_[0, np.cumsum(n_op)], r.cigar[starts + within], chrom[seg],
                                np.r_[seg, len(idx)] if len(idx) else [0])


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--records", type=int, default=40_000_000)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=1)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "tag_groups_c2.json"))
    args = ap.parse_args()
    gpu = gpu_info()
    cfg = synth.config_c2(args.records)
    w = synth.generate(cfg, cache_dir=CACHE)
    r = w.records
    rng = np.random.default_rng(cfg.seed)
    bc = rng.integers(0, N_BARCODES, len(r))
    names = [b"%010d-1" % b for b in range(N_BARCODES)]
    fields = np.frombuffer(b"".join(b"CBZ" + n + b"\0" for n in names), np.uint8).reshape(N_BARCODES, 16)
    os.makedirs(CACHE, exist_ok=True)
    bam = os.path.join(CACHE, "tag_groups_%s_%d.bam" % (cfg.key(), len(r)))
    t0 = time.perf_counter()
    if not os.path.exists(bam):
        r.write_bam(bam + ".tmp", w.chroms, w.chrom_len, with_seq=True,
                    aux=(np.arange(len(r) + 1, dtype=np.int64) * 16, fields[bc].ravel()))
        os.replace(bam + ".tmp", bam)
    write_s = time.perf_counter() - t0
    tables = {G: api.TagGroups("CB", names, [b % G for b in range(N_BARCODES)], G) for G in (16, 1000)}
    want = {G: np.bincount(bc % G, minlength=G).tolist() for G in tables}
    res = {"what": "combineGroups on configs[1]'s records (synth.config_c2, %d records, seed %d), sequencer-shaped BAM with a CB:Z "
                   "barcode per record (%d barcodes, barcode b in group b %% G)" % (len(r), cfg.seed, N_BARCODES),
           "gpu": gpu, "bam_bytes": os.path.getsize(bam), "records": len(r), "bam_write_s": write_s}

    # (1) ingest with and without the lookup + split
    with spliser_b200.Context(0) as ctx:
        def plain():
            t = time.perf_counter()
            with ctx.load_bam(bam):
                dt = time.perf_counter() - t
            return 1e3 * dt, ctx.stats()["ms_decode"]

        def split(G):
            t = time.perf_counter()
            s = ctx.load_bam_groups(bam, tables[G])
            dt = time.perf_counter() - t
            st = ctx.stats()
            ok = s.counts == want[G] and s.no_value == 0 and s.unmatched == 0
            held = sum(x.device_bytes for x in s.samples)
            s.close()
            return 1e3 * dt, st["ms_decode"], ok, held, st["bam_on_device"]
        for _ in range(args.warmup):
            plain(); split(16); split(1000)
        t = {"load_bam": ([], []), 16: ([], []), 1000: ([], [])}
        ok, held, dev = True, {}, set()
        for _ in range(args.steps):
            a, b = plain()
            t["load_bam"][0].append(a); t["load_bam"][1].append(b)
            for G in (16, 1000):
                a, b, good, h, d = split(G)
                t[G][0].append(a); t[G][1].append(b)
                ok &= good; held[G] = h; dev.add(d)
        res["ingest"] = {"load_bam_ms": spread(t["load_bam"][0]), "load_bam_decode_ms": spread(t["load_bam"][1])}
        for G in (16, 1000):
            res["ingest"]["load_bam_groups_%d_ms" % G] = spread(t[G][0])
            res["ingest"]["load_bam_groups_%d_decode_ms" % G] = spread(t[G][1])
            res["ingest"]["split_bytes_%d" % G] = held[G]
        res["ingest"]["on_device"] = sorted(dev)
        res["counts_match"] = ok

    # (2) kernels, in a run of their own
    import re

    import torch
    from torch.profiler import ProfilerActivity, profile
    kern = {}
    with spliser_b200.Context(0) as ctx:
        runs = {"load_bam": lambda: ctx.load_bam(bam).close()}
        for G in (16, 1000):
            runs["groups_%d" % G] = (lambda G=G: ctx.load_bam_groups(bam, tables[G]).close())
        for key, fn in runs.items():
            fn()
            with profile(activities=[ProfilerActivity.CUDA]) as prof:
                fn()
                torch.cuda.synchronize()
            rows = {}
            for e in prof.key_averages():
                m = re.search(r"(k_group_\w+|k_bam_fill)(<[^>(]*>)?", e.key)
                if m:
                    dt = getattr(e, "device_time_total", None) or getattr(e, "cuda_time_total", 0)
                    rows[m.group(0)] = rows.get(m.group(0), 0.0) + dt / 1e3
            kern[key] = {k: round(v, 4) for k, v in sorted(rows.items())}
            kern[key]["k_group_total_ms"] = round(sum(v for k, v in rows.items() if k.startswith("k_group_")), 4)
    res["kernels_ms"] = kern

    # (3) combineGroups against combineBam over the pre-split BAMs, G = 16
    d = tempfile.mkdtemp(prefix="tag_groups_")
    G = 16
    titles = ["g%02d" % g for g in range(G)]
    gf = os.path.join(d, "groups.tsv")
    with open(gf, "w") as fh:
        fh.writelines("%s\t%s\n" % (names[b].decode(), titles[b % G]) for b in range(N_BARCODES))
    per = []
    for g in range(G):
        idx = np.flatnonzero(bc % G == g)
        p = os.path.join(CACHE, "tag_groups_%s_%d.g%d_of_%d.bam" % (cfg.key(), len(r), g, G))
        if not os.path.exists(p):
            sub = subset(r, idx)
            sub.write_bam(p + ".tmp", w.chroms, w.chrom_len, with_seq=True, aux=(np.arange(len(idx) + 1, dtype=np.int64) * 16,
                                                                                 fields[bc[idx]].ravel()))
            os.replace(p + ".tmp", p)
        per.append(p)
    sf = os.path.join(d, "samples.tsv")
    with open(sf, "w") as fh:
        fh.writelines("%s\t%s\t%s\n" % (t, os.path.join(d, "b.%s.SpliSER.tsv" % t), p) for t, p in zip(titles, per))

    def run_groups():
        t = time.perf_counter()
        with contextlib.redirect_stdout(io.StringIO()):
            cli.combineGroups(bam, "CB", gf, os.path.join(d, "g"))
        return 1e3 * (time.perf_counter() - t)

    def run_bam():
        t = time.perf_counter()
        with contextlib.redirect_stdout(io.StringIO()):
            cli.combineBam(sf, os.path.join(d, "b"))
        return 1e3 * (time.perf_counter() - t)
    for _ in range(args.warmup):
        run_groups(); run_bam()
    wg, wb = [], []
    for _ in range(args.steps):
        wg.append(run_groups()); wb.append(run_bam())
    same = all(open(os.path.join(d, "g.%s.SpliSER.tsv" % t)).read() == open(os.path.join(d, "b.%s.SpliSER.tsv" % t)).read()
               for t in titles) and open(os.path.join(d, "g.combined.tsv")).read() == open(os.path.join(d, "b.combined.tsv")).read()
    res["cli_16_groups"] = {"combineGroups_ms": spread(wg), "combineBam_presplit_ms": spread(wb), "outputs_identical": same,
                            "note": "host clock around each CLI call, which makes its own context: combineGroups stages one %d-byte file "
                                    "(page-locked image and inflate buffers of that size allocated by the fresh context), combineBam "
                                    "16 files of about 1/16 of it" % os.path.getsize(bam)}

    # (4) where the time of each command goes: a fresh context's first ingest against its second, and a profile of one run of each
    # command by the Python calls it makes (cumulative seconds; every library call ends in a device synchronise)
    def clock(fn):
        t = time.perf_counter()
        out = fn()
        return 1e3 * (time.perf_counter() - t), out
    fresh = {}
    fresh["context_ms"], ctx = clock(lambda: spliser_b200.Context(0))
    fresh["first_load_bam_groups_ms"], s = clock(lambda: ctx.load_bam_groups(bam, tables[16]))
    s.close()
    fresh["second_load_bam_groups_ms"], s = clock(lambda: ctx.load_bam_groups(bam, tables[16]))
    s.close()
    fresh["close_ms"], _ = clock(ctx.close)
    fresh["bam_context_ms"], ctx = clock(lambda: spliser_b200.Context(0))
    loads = []
    for p in per:
        dt, s = clock(lambda p=p: ctx.load_bam(p))
        loads.append(dt)
        s.close()
    fresh["bam_first_load_ms"], fresh["bam_16_loads_ms"] = loads[0], sum(loads)
    fresh["bam_close_ms"], _ = clock(ctx.close)
    res["fresh_context"] = fresh

    import cProfile
    import pstats
    wanted = {("api.py", "__init__"), ("api.py", "close"), ("api.py", "load_bam_groups"), ("api.py", "load_bam"),
              ("api.py", "process_extract"), ("api.py", "recount"), ("api.py", "infer_strand"), ("cli.py", "_merge_recount_write"),
              ("cli.py", "write_process_tsv"), ("cli.py", "read_groups_file"), ("cli.py", "combineGroups"), ("cli.py", "combineBam")}
    prof_s = {}
    for name, fn in (("combineGroups", run_groups), ("combineBam", run_bam)):
        pr = cProfile.Profile()
        pr.enable()
        fn()
        pr.disable()
        rows = {}
        for (fname, line, func), (cc, nc, tt, ct, _) in pstats.Stats(pr).stats.items():
            key = (os.path.basename(fname), func)
            if key in wanted and "spliser_b200" in fname:
                k = "%s:%d:%s" % (key[0], line, func)
                rows[k] = {"calls": rows.get(k, {}).get("calls", 0) + nc, "cum_s": round(rows.get(k, {}).get("cum_s", 0) + ct, 4)}
        prof_s[name] = dict(sorted(rows.items(), key=lambda kv: -kv[1]["cum_s"]))
    res["cli_profile"] = prof_s
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as fh:
        json.dump(res, fh, indent=1)
    print(json.dumps(res))
    if not (ok and same):
        sys.exit("counts or outputs differ")


if __name__ == "__main__":
    main()
