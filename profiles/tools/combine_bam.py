"""A multi-sample run from BAMs alone, timed on the 48-sample configs[3] workload of bench_combine.build_samples and on a
sequencer-shaped variant of it (the same records rewritten with spl_write_bam_seq: read names, SEQ and QUAL, so the ingest costs
what it costs on a real file):

  (a) processBam for every sample, then combine   -- every BAM is ingested twice (extraction + count, then the re-count)
  (b) combineBam                                   -- every BAM is ingested once and kept in GPU memory for the re-count

each at 1 GPU and at every visible GPU (one context per GPU, samples dealt by dist.samples_of in both).  Contexts are made once
per configuration and warmed up on one sample; (a) and (b) alternate.  Host clock around calls that end in a device synchronise.
Reports wall time per phase and summed per call kind (ingest, holding a sample, extraction + count, re-count), H2D bytes per
sample (spl_last_stats, plus the file image a path re-count's device ingest copies, which its stats leave out), resident bytes
per sample and in all, samples that fell back to the path route, and the
GPU name and power limit read in the same run.  Checks that (a) and (b) write the same bytes.

    python profiles/tools/combine_bam.py [--reads-per-sample 1000000] [--repeats 2] [--out profiles/combine_bam_c4_48.json]
"""
import argparse
import json
import os
import shutil
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
import bench_combine  # noqa: E402
import spliser_b200  # noqa: E402
from spliser_b200 import Records, api, cli  # noqa: E402

CACHE = os.environ.get("SPLISER_BENCH_CACHE", os.path.join(tempfile.gettempdir(), "spliser_bench_cache"))


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
    if q.returncode != 0 or not q.stdout.strip():
        raise RuntimeError("no GPU visible to nvidia-smi: this measurement needs the B200")
    rows = [[x.strip() for x in line.split(",")] for line in q.stdout.strip().splitlines()]
    return {"name": rows[0][0], "power_limit": rows[0][1], "max_sm_clock": rows[0][2], "n_visible": len(rows)}


class Metered(spliser_b200.Context):
    """A context that adds up what crossed PCIe per sample and what stayed resident."""

    def __init__(self, device, log):
        super().__init__(device)
        self.log = log

    def _note(self, bam, key, value):
        self.log.setdefault(os.path.basename(bam), {}).setdefault(key, 0)
        self.log[os.path.basename(bam)][key] += value

    def load_bam(self, bam_path, xs=False):
        try:
            s = super().load_bam(bam_path, xs)
        except api.SampleMemoryError:
            self._note(bam_path, "fell_back", 1)
            raise
        st = self.stats()
        self._note(bam_path, "h2d_bytes", st["h2d_bytes"])
        self._note(bam_path, "load_ingest_s", st["ms_decode"] / 1e3)
        self._note(bam_path, "load_hold_s", (st["ms_total"] - st["ms_decode"]) / 1e3)      # allocation + copy into the sample
        self._note(bam_path, "resident_bytes", s.device_bytes)
        ctx, process_extract, recount = self, s.process_extract, s.recount

        def pe(*a, **kw):
            t0 = time.perf_counter()
            r = process_extract(*a, **kw)
            ctx._note(bam_path, "extract_count_s", time.perf_counter() - t0)
            ctx._note(bam_path, "h2d_bytes", ctx.stats()["h2d_bytes"])
            return r

        def rc(*a, **kw):
            t0 = time.perf_counter()
            r = recount(*a, **kw)
            ctx._note(bam_path, "recount_s", time.perf_counter() - t0)
            ctx._note(bam_path, "h2d_bytes", ctx.stats()["h2d_bytes"])
            return r
        s.process_extract, s.recount = pe, rc
        return s

    def process_bam_extract(self, bam_path, *a, **kw):
        t0 = time.perf_counter()
        r = super().process_bam_extract(bam_path, *a, **kw)
        self._note(bam_path, "extract_count_s", time.perf_counter() - t0)
        self._note(bam_path, "h2d_bytes", self.stats()["h2d_bytes"])
        return r

    def recount_bam(self, bam_path, *a, **kw):
        t0 = time.perf_counter()
        r = super().recount_bam(bam_path, *a, **kw)
        self._note(bam_path, "recount_s", time.perf_counter() - t0)
        st = self.stats()
        # spl_recount's stats leave out the file image its device ingest copied: add it
        self._note(bam_path, "h2d_bytes", st["h2d_bytes"] + (os.path.getsize(bam_path) if st["bam_on_device"] else 0))
        return r


def samples_file(d, samples, tag):
    sf = os.path.join(d, tag + "_samples.tsv")
    with open(sf, "w") as fh:
        for k, (title, bam, _) in enumerate(samples):
            fh.write("%s\t%s\t%s\n" % (title, os.path.join(d, "%s%02d.SpliSER.tsv" % (tag, k)), bam))
    return sf


def run_a(d, samples, ctxs):
    """processBam per sample (rank r takes samples_of(r)), then combine on the same contexts."""
    sf = samples_file(d, samples, "a")
    lines = [line.rstrip("\n").split("\t") for line in open(sf)]
    t0 = time.perf_counter()

    def rank(r):
        for k in cli.samples_of(r, len(ctxs), len(lines)):
            cli.processBam(lines[k][2], lines[k][1][:-len(".SpliSER.tsv")], isStranded=True, strandedType="rf", ctx=ctxs[r])
    cli._on_ranks(len(ctxs), rank)
    t1 = time.perf_counter()
    if len(ctxs) == 1:
        cli.combine(sf, os.path.join(d, "a"), isStranded=True, strandedType="rf", ctx=ctxs[0])
    else:
        pool = list(ctxs)
        cli.combine(sf, os.path.join(d, "a"), isStranded=True, strandedType="rf", devices=list(range(len(ctxs))),
                    context_factory=lambda dev: _Borrowed(pool[dev]))
    t2 = time.perf_counter()
    return {"phase1_process_s": t1 - t0, "phase2_combine_s": t2 - t1, "total_s": t2 - t0}


class _Borrowed:
    """An existing context handed to combine's per-rank factory; combine closes what it gets, the owner closes it later."""

    def __init__(self, c):
        self.c = c

    def __getattr__(self, k):
        return getattr(self.c, k)

    def close(self):
        pass


def run_b(d, samples, ctxs):
    sf = samples_file(d, samples, "b")
    stamp = {}
    inner = cli._merge_recount_write

    def timed(*a, **kw):
        stamp["merge"] = time.perf_counter()
        return inner(*a, **kw)
    cli._merge_recount_write = timed
    try:
        pool = list(ctxs)
        t0 = time.perf_counter()
        cli.combineBam(sf, os.path.join(d, "b"), isStranded=True, strandedType="rf", devices=list(range(len(ctxs))),
                       context_factory=lambda dev: _Borrowed(pool[dev]))
        t2 = time.perf_counter()
    finally:
        cli._merge_recount_write = inner
    return {"phase1_load_process_s": stamp["merge"] - t0, "phase2_merge_recount_write_s": t2 - stamp["merge"], "total_s": t2 - t0}


def same_outputs(d, n):
    for k in range(n):
        if open(os.path.join(d, "a%02d.SpliSER.tsv" % k), "rb").read() != open(os.path.join(d, "b%02d.SpliSER.tsv" % k), "rb").read():
            return False
    return open(os.path.join(d, "a.combined.tsv"), "rb").read() == open(os.path.join(d, "b.combined.tsv"), "rb").read()


def seq_variant(chroms, samples):
    out = []
    lens = [n for _, n in bench_combine.CONTIGS]
    for title, bam, bed in samples:
        seq = bam[:-4] + "_seq.bam"
        if not os.path.exists(seq):
            Records.from_bam(bam, chroms).write_bam(seq, chroms, lens, with_seq=True)
        out.append((title, seq, bed))
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reads-per-sample", type=int, default=1_000_000)
    ap.add_argument("--repeats", type=int, default=2)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "combine_bam_c4_48.json"))
    args = ap.parse_args()
    gpu = gpu_info()
    chroms, plain = bench_combine.build_samples(CACHE, args.reads_per_sample)
    variants = {"records_only": plain, "sequencer_shaped": seq_variant(chroms, plain)}
    doc = {"tool": "profiles/tools/combine_bam.py", "gpu": gpu, "reads_per_sample": args.reads_per_sample, "n_samples": len(plain),
           "workload": "bench_combine.build_samples: 48 samples (6 conditions x 8 replicates), stranded rf", "runs": []}
    for vname, samples in variants.items():
        file_bytes = {os.path.basename(b): os.path.getsize(b) for _, b, _ in samples}
        for n_gpu in sorted({1, gpu["n_visible"]}):
            log = {}
            ctxs = [Metered(dev, log) for dev in range(n_gpu)]
            try:
                for c in ctxs:                                 # warm-up: module load, first allocations, one of each call
                    with c.load_bam(samples[0][1]) as s:
                        s.process_extract(chroms, api.FLAG_STRANDED | api.FLAG_RF)
                    c.process_bam_extract(samples[0][1], chroms, api.FLAG_STRANDED | api.FLAG_RF)
                for rep in range(args.repeats):
                    for arm, fn in (("a_processBam_then_combine", run_a), ("b_combineBam", run_b)):
                        d = tempfile.mkdtemp(prefix="combine_bam_")
                        log.clear()
                        try:
                            t = fn(d, samples, ctxs)
                            per = list(log.values())
                            t.update(variant=vname, n_gpus=n_gpu, arm=arm, repeat=rep,
                                     h2d_bytes_per_sample_mean=sum(x.get("h2d_bytes", 0) for x in per) / len(samples),
                                     file_bytes_per_sample_mean=sum(file_bytes.values()) / len(samples),
                                     resident_bytes_per_sample_mean=sum(x.get("resident_bytes", 0) for x in per) / len(samples),
                                     resident_bytes_total=sum(x.get("resident_bytes", 0) for x in per),
                                     fell_back=sum(x.get("fell_back", 0) for x in per),
                                     **{k + "_sum": sum(x.get(k, 0) for x in per)
                                        for k in ("load_ingest_s", "load_hold_s", "extract_count_s", "recount_s")})
                            if arm.startswith("a"):
                                keep_a = d
                            else:
                                for k in range(len(samples)):
                                    shutil.copy(os.path.join(keep_a, "a%02d.SpliSER.tsv" % k), d)
                                shutil.copy(os.path.join(keep_a, "a.combined.tsv"), d)
                                t["same_bytes_as_a"] = same_outputs(d, len(samples))
                                shutil.rmtree(keep_a, ignore_errors=True)
                                shutil.rmtree(d, ignore_errors=True)
                            doc["runs"].append(t)
                            print(json.dumps(t), flush=True)
                        except BaseException:
                            shutil.rmtree(d, ignore_errors=True)
                            raise
            finally:
                for c in ctxs:
                    c.close()
    os.makedirs(os.path.dirname(args.out), exist_ok=True)
    with open(args.out, "w") as fh:
        json.dump(doc, fh, indent=1)
        fh.write("\n")
    print("wrote", args.out)


if __name__ == "__main__":
    main()
