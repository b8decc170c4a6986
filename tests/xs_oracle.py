"""Pure-Python restatement of the XS-tag strand rule (SPL_FLAG_XS_STRAND, include/spliser_b200.h) and of junction extraction
with strands from a per-record XS column, plus the aux-field encoder the tests write BAM files with.  Test infrastructure
only; the extraction itself is oracle/junction_oracle.py's, run once per strand."""
from __future__ import annotations

import struct

import numpy as np

from oracle import junction_oracle

_FIXED = {"A": 1, "c": 1, "C": 1, "s": 2, "S": 2, "i": 4, "I": 4, "f": 4}
_PACK = {"c": "<b", "C": "<B", "s": "<h", "S": "<H", "i": "<i", "I": "<I", "f": "<f"}


def encode_aux(fields) -> bytes:
    """Bytes of aux fields (tag, type, value) in order: A takes a one-character str, c C s S i I f a number, Z and H a str,
    B a (subtype, list of numbers) pair."""
    out = bytearray()
    for tag, ty, val in fields:
        out += tag.encode() + ty.encode()
        if ty == "A":
            out += val.encode()
        elif ty in _PACK:
            out += struct.pack(_PACK[ty], val)
        elif ty in "ZH":
            out += val.encode() + b"\0"
        elif ty == "B":
            sub, items = val
            out += sub.encode() + struct.pack("<I", len(items))
            for x in items:
                out += struct.pack(_PACK[sub], x)
        else:
            raise ValueError("unknown aux type %r" % ty)
    return bytes(out)


def xs_of_aux(blob: bytes) -> str:
    """Strand of a record whose aux block is `blob`: the first field tagged XS decides (XS:A:+ '+', XS:A:- '-', anything else
    '?'); '?' without one, or when an unknown type or a field that runs past the end comes first."""
    p, n = 0, len(blob)
    while n - p >= 3:
        tag, ty, v = blob[p:p + 2], chr(blob[p + 2]), p + 3
        if ty in _FIXED:
            end = v + _FIXED[ty]
        elif ty in "ZH":
            nul = blob.find(b"\0", v)
            if nul < 0:
                return "?"
            end = nul + 1
        elif ty == "B":
            if n - v < 5:
                return "?"
            sub = chr(blob[v])
            es = 1 if sub in "cC" else 2 if sub in "sS" else 4
            end = v + 5 + struct.unpack_from("<I", blob, v + 1)[0] * es
        else:
            return "?"
        if end > n:
            return "?"
        if tag == b"XS":
            return chr(blob[v]) if ty == "A" and blob[v:v + 1] in (b"+", b"-") else "?"
        p = end
    return "?"


def _subset(records, keep):
    """The records with keep[r], in order, with the chromosome segments recounted."""
    from spliser_b200.api import Records
    idx = np.flatnonzero(keep)
    off = records.cig_off.astype(np.int64)
    cig = [records.cigar[off[r]:off[r + 1]] for r in idx]
    cig_off = np.zeros(len(idx) + 1, np.int64)
    cig_off[1:] = np.cumsum([len(c) for c in cig])
    seg_off = np.searchsorted(idx, records.seg_off)
    return Records(records.pos[idx], records.flag[idx], cig_off, np.concatenate(cig) if cig else np.zeros(0, np.uint32),
                   records.seg_chrom, seg_off)


def extract(records, n_chrom, flags=0, min_anchor=8, min_intron=70, max_intron=500000, xs=None):
    """junction_oracle.extract; with xs (one '+', '-' or '?' byte per record) every junction of a record takes its xs strand
    (any other byte counts as '?') and `flags` does not touch the strands."""
    if xs is None:
        return junction_oracle.extract(records, n_chrom, flags, min_anchor, min_intron, max_intron)
    from spliser_b200.api import Junctions
    xs = np.asarray(xs, np.uint8)
    xs = np.where((xs == ord("+")) | (xs == ord("-")), xs, ord("?")).astype(np.uint8)
    parts = []
    for rank, s in enumerate(b"?+-"):
        j = junction_oracle.extract(_subset(records, xs == s), n_chrom, 0, min_anchor, min_intron, max_intron)
        parts.append((j, rank, s))
    cols = {k: np.concatenate([getattr(j, k) for j, _, _ in parts]) for k in ("chrom", "left", "right", "score", "start", "end")}
    rank = np.concatenate([np.full(len(j), r) for j, r, _ in parts])
    strand = np.concatenate([np.full(len(j), s, np.uint8) for j, _, s in parts])
    o = np.lexsort((rank, cols["right"], cols["left"], cols["chrom"]))
    return Junctions(cols["chrom"][o], cols["left"][o], cols["right"][o], cols["score"][o], strand[o], cols["start"][o], cols["end"][o])


def star_aux(records, seed, drop=0.10, flip=0.02):
    """XS column and STAR-like aux bytes for records whose FLAG is dUTP-style (rf): a spliced record's XS is the rf strand of
    its FLAG, dropped (no tag) for about `drop` of them and flipped for about `flip`; every record carries NH HI AS nM NM MD."""
    rng = np.random.default_rng(seed)
    n = len(records)
    off = records.cig_off.astype(np.int64)
    ops = records.cigar & 15
    spliced = np.zeros(n, bool)
    has_n = np.flatnonzero(ops == 3)
    spliced[np.searchsorted(off, has_n, side="right") - 1] = True
    u = rng.random(n)
    xs = np.full(n, ord("?"), np.uint8)
    aux = []
    flg = records.flag.tolist()
    for r in range(n):
        m = int(sum(int(v) >> 4 for v in records.cigar[off[r]:off[r + 1]] if (v & 15) in (0, 7, 8)))
        fields = [("NH", "i", 1), ("HI", "i", 1), ("AS", "i", 2 * m - 2), ("nM", "i", 0), ("NM", "i", 0), ("MD", "Z", str(m))]
        if spliced[r] and u[r] >= drop:
            s = chr(junction_oracle._strand(flg[r], 3))
            if u[r] < drop + flip:
                s = "+" if s == "-" else "-"
            fields.append(("XS", "A", s))
            xs[r] = ord(s)
        aux.append(encode_aux(fields))
    return xs, aux
