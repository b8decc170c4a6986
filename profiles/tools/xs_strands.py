"""Cost of taking junction strands from the XS tag (SPL_FLAG_XS_STRAND) on a sequencer-shaped file.

The input is the shape of `bam_ingest_profile.py N seq` (synth.config_c2 records with read names, SEQ and QUAL; 8M records by
default) plus STAR-like aux fields on every record: NH:i HI:i AS:i nM:i NM:i MD:Z, and XS:A on spliced records.  The XS strand
is the dUTP (rf) strand of the record's FLAG, dropped for about 10 % and flipped for about 2 % of the spliced records (seeded).

extract_junctions_bam runs without and with the XS bit, alternating, after one warm-up pass of each.  Per call the library's
stats give the ingest time (ms_decode: host wall clock around the device BGZF inflate + record parse, which ends in a stream
synchronise; the XS aux walk runs inside it) and the CUDA-event time of the extraction kernels (ms_extract).  Checks that both
tables hold the same supporting-record total and that the XS table has every strand.  Records the GPU name and power limit.

    python profiles/tools/xs_strands.py [--records 8000000] [--steps 7] [--out profiles/xs_strands_seq8M.json]
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
import spliser_b200  # noqa: E402
from spliser_b200 import api, synth  # noqa: E402

CACHE = os.environ.get("SPLISER_BENCH_CACHE", os.path.join(tempfile.gettempdir(), "spliser_bench_cache"))


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
    if q.returncode != 0 or not q.stdout.strip():
        raise RuntimeError("no GPU visible to nvidia-smi: this measurement needs the B200")
    name, power, clk = [x.strip() for x in q.stdout.strip().splitlines()[0].split(",")]
    return {"name": name, "power_limit": power, "max_sm_clock": clk}


def star_aux(rec, seed):
    """(aux offsets [n + 1], aux bytes, XS column) of STAR-like tags for the records, built column-wise."""
    n = len(rec)
    rng = np.random.default_rng(seed)
    off = rec.cig_off.astype(np.int64)
    ops, lens = rec.cigar & 15, (rec.cigar >> 4).astype(np.int64)
    owner = np.repeat(np.arange(n), np.diff(off))
    m = np.bincount(owner, weights=np.where(np.isin(ops, (0, 7, 8)), lens, 0), minlength=n).astype(np.int64)
    spliced = np.bincount(owner, weights=(ops == 3), minlength=n) > 0
    flag = rec.flag.astype(np.int64)
    first = ((flag & 64) != 0) | ((flag & 1) == 0)
    plus = first != ((flag & 16) != 0)
    plus = ~plus                                                  # dUTP: rf
    u = rng.random(n)
    has_xs = spliced & (u >= 0.10)
    plus = np.where(u < 0.12, ~plus, plus)                        # about 2 % of the tagged ones flipped
    xs = np.where(has_xs, np.where(plus, ord("+"), ord("-")), ord("?")).astype(np.uint8)
    digits = np.maximum(1, np.floor(np.log10(np.maximum(m, 1))).astype(np.int64) + 1)
    length = 35 + 3 + digits + 1 + 4 * has_xs
    W = int(length.max()) if n else 0
    a = np.zeros((n, W), np.uint8)
    for k, (tag, val) in enumerate((("NH", 1), ("HI", 1), ("AS", None), ("nM", 0), ("NM", 0))):
        v = (2 * m - 2) if val is None else np.full(n, val, np.int64)
        c = 7 * k
        a[:, c], a[:, c + 1], a[:, c + 2] = ord(tag[0]), ord(tag[1]), ord("i")
        a[:, c + 3:c + 7] = v.astype("<i4").view(np.uint8).reshape(n, 4)
    a[:, 35], a[:, 36], a[:, 37] = ord("M"), ord("D"), ord("Z")
    rows = np.arange(n)
    for d in range(1, int(digits.max()) + 1 if n else 1):
        sel = rows[digits == d]
        for q in range(d):                                        # most significant digit first
            a[sel, 38 + q] = ord("0") + (m[sel] // 10 ** (d - 1 - q)) % 10
        c = 38 + d + 1                                            # after the NUL
        tx = sel[has_xs[sel]]
        a[tx, c], a[tx, c + 1], a[tx, c + 2], a[tx, c + 3] = ord("X"), ord("S"), ord("A"), xs[tx]
    mask = np.arange(W)[None, :] < length[:, None]
    aux_off = np.zeros(n + 1, np.int64)
    aux_off[1:] = np.cumsum(length)
    return aux_off, a[mask], xs


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--records", type=int, default=8_000_000)
    ap.add_argument("--steps", type=int, default=7)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "xs_strands_seq8M.json"))
    args = ap.parse_args()
    gpu = gpu_info()
    cfg = synth.config_c2(args.records)
    w = synth.generate(cfg, cache_dir=CACHE)
    bam = os.path.join(CACHE, "xs_seq_%s_%d.bam" % (cfg.key(), len(w.records)))
    aux_off, aux, xs = star_aux(w.records, cfg.seed)
    if not os.path.exists(bam):
        os.makedirs(CACHE, exist_ok=True)
        w.records.write_bam(bam + ".tmp", w.chroms, w.chrom_len, with_seq=True, aux=(aux_off, aux))
        os.replace(bam + ".tmp", bam)
    modes = (("default", 0), ("xs", api.FLAG_XS_STRAND))
    runs = {name: [] for name, _ in modes}
    tables = {}
    with spliser_b200.Context(0) as ctx:
        for name, flags in modes:                                 # warm-up
            ctx.extract_junctions_bam(bam, w.chroms, flags)
        for _ in range(args.steps):
            for name, flags in modes:
                tables[name] = ctx.extract_junctions_bam(bam, w.chroms, flags)
                s = ctx.stats()
                if s["bam_on_device"] != 1.0:
                    sys.exit("the device ingest fell back to the host reader")
                runs[name].append({"ingest_ms": s["ms_decode"], "extract_kernels_ms": s["ms_extract"], "total_ms": s["ms_total"]})

    def summary(v):
        return {"mean": float(np.mean(v)), "min": float(np.min(v)), "max": float(np.max(v))}
    res = {
        "what": "extract_junctions_bam on a sequencer-shaped file with STAR-like aux (synth.config_c2, %d records, seed %d; "
                "read names, SEQ, QUAL; NH HI AS nM NM MD on every record, XS:A on %d of %d spliced records), without and with "
                "SPL_FLAG_XS_STRAND, one warm-up pass each, then %d alternating timed passes; device BGZF ingest"
                % (len(w.records), cfg.seed, int((xs != ord("?")).sum()), int(len(xs)), args.steps),
        "gpu": gpu,
        "bam_bytes": os.path.getsize(bam),
        "aux_bytes": int(len(aux)),
        "records": len(w.records),
    }
    for name, _ in modes:
        res[name] = {k: summary([r[k] for r in runs[name]]) for k in ("ingest_ms", "extract_kernels_ms", "total_ms")}
        res[name]["junctions"] = len(tables[name])
    res["xs_minus_default_ingest_ms_mean"] = res["xs"]["ingest_ms"]["mean"] - res["default"]["ingest_ms"]["mean"]
    res["xs_minus_default_extract_kernels_ms_mean"] = res["xs"]["extract_kernels_ms"]["mean"] - res["default"]["extract_kernels_ms"]["mean"]
    st = {chr(c): int(k) for c, k in zip(*np.unique(tables["xs"].strand, return_counts=True))}
    res["xs_table_rows_by_strand"] = st
    ok = int(tables["xs"].score.sum()) == int(tables["default"].score.sum()) and set(st) == {"+", "-", "?"}
    res["checks_pass"] = bool(ok)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as fh:
        json.dump(res, fh, indent=1)
    print(json.dumps(res))
    if not ok:
        sys.exit("the XS table does not hold the same supporting records")


if __name__ == "__main__":
    main()
