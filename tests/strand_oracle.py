"""Numpy restatement of the library-strandedness vote (include/spliser_b200.h, spl_gene_strands, states the rule): one vote per
kept record, its fr read strand against the reference strand of the genes that overlap it (brute force over every gene) or of its
XS tag.  What the tests hold spl_infer_strand* and the host gene index to, and what the CPU stand-ins answer votes with."""
import numpy as np

from spliser_b200.api import GeneStrands, StrandVotes

REF_OPS = (0, 2, 3, 7, 8)                 # M D N = X


def spans(records):
    """(POS - 1, L, operators) per record: L = the M D N = X lengths summed, 1 when that sum is 0."""
    off = records.cig_off.astype(np.int64)
    n = len(records)
    nop = np.diff(off)
    owner = np.repeat(np.arange(n), nop)
    lens = np.where(np.isin(records.cigar & 15, REF_OPS), (records.cigar >> 4).astype(np.int64), 0)
    L = np.zeros(n, np.int64)
    np.add.at(L, owner, lens)
    L[L == 0] = 1
    return records.pos.astype(np.int64) - 1, L, nop


def record_chrom(records, n_chrom):
    """Caller chromosome of every record from the segments; -1 when the segment's is unknown."""
    c = np.repeat(records.seg_chrom.astype(np.int64), np.diff(records.seg_off))
    return np.where((c >= 0) & (c < n_chrom), c, -1)


def fr_plus(flag):
    """check_strand's read strand under fr is '+' (S:374-406)."""
    f = flag.astype(np.int64)
    first = ((f & 64) != 0) | ((f & 1) == 0)
    return first != ((f & 16) != 0)


def gene_mask(genes: GeneStrands, c, p, L):
    """Bit 0 '+', bit 1 '-' over the genes of caller chromosome c overlapping each span (p = POS - 1, L), by a scan of every
    gene: POS - 1 < right and POS - 1 + L > left, strands '+' / '-' only, empty spans (right <= left) ignored."""
    out = np.zeros(len(p), np.uint8)
    if c >= genes.n_chrom or not len(p):
        return out
    a, b = int(genes.chrom_off[c]), int(genes.chrom_off[c + 1])
    left, right, st = genes.left[a:b].astype(np.int64), genes.right[a:b].astype(np.int64), genes.strand[a:b]
    keep = ((st == ord("+")) | (st == ord("-"))) & (right > left)
    left, right, plus = left[keep], right[keep], st[keep] == ord("+")
    if not len(left):
        return out
    step = max(1, 4_000_000 // len(left))
    for i in range(0, len(p), step):
        pp, ll = p[i:i + step, None], L[i:i + step, None]
        ov = (pp < right[None, :]) & (pp + ll > left[None, :])
        out[i:i + step] = (ov & plus[None, :]).any(1) | ((ov & ~plus[None, :]).any(1) << 1)
    return out


def votes(records, n_chrom, genes: GeneStrands = None) -> StrandVotes:
    """The three counters; genes=None takes the reference strand from records.xs."""
    p, L, nop = spans(records)
    chrom = record_chrom(records, n_chrom)
    kept = (chrom >= 0) & (nop > 0)
    ref = np.zeros(len(records), np.uint8)
    if genes is None:
        ref = np.where(records.xs == ord("+"), 1, np.where(records.xs == ord("-"), 2, 0)).astype(np.uint8)
    else:
        for c in np.unique(chrom[kept]):
            sel = np.flatnonzero(kept & (chrom == c))
            ref[sel] = gene_mask(genes, int(c), p[sel], L[sel])
    voted = kept & ((ref == 1) | (ref == 2))
    agree = voted & ((ref == 1) == fr_plus(records.flag))
    return StrandVotes(int(agree.sum()), int(voted.sum() - agree.sum()), int(kept.sum() - voted.sum()))
