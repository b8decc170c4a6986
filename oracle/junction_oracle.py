"""Pure-Python restatement of the junction extraction (`k_je_*` in spliser_b200/csrc/graph_build.cu) with anchor extents, and of
the two row filters `process` applies to a BED12 (-c, S:269; -g window, S:279-288).  Test infrastructure only.

A record supports the junction (l, r) of one of its N operators when min_intron <= length(N) <= max_intron and the aligned
stretches on both sides (M/=/X/D bases since the previous N or the read start, up to the next N or the read end; I, S, H and P
add nothing) are at least min_anchor long.  l is the position before the N, r = l + length(N).  Per junction: score = the
supporting records, start = l - the longest left stretch, end = r + the longest right stretch among them.  Strand: '?', or with
FLAG_STRANDED the strand check_strand derives from the FLAG (S:374-406).  Rows are sorted by (chromosome, l, r, strand) with
'?' < '+' < '-'."""
from __future__ import annotations

import numpy as np

_ADV = (0, 2, 7, 8)                          # M D = X: advance the reference and lengthen the stretch
_STRAND_ORDER = {ord("?"): 0, ord("+"): 1, ord("-"): 2}


def _strand(flag, flags):
    if not flags & 1:
        return ord("?")
    first = bool(flag & 64) or not (flag & 1)
    plus = first != bool(flag & 16)
    if flags & 2:
        plus = not plus
    return ord("+") if plus else ord("-")


def extract(records, n_chrom, flags=0, min_anchor=8, min_intron=70, max_intron=500000):
    """records: api.Records -> api.Junctions with start / end."""
    from spliser_b200.api import Junctions
    rows = {}                                # (chrom, l, r, strand) -> [score, max_left, max_right]
    pos, flg = records.pos.tolist(), records.flag.tolist()
    off, cig = records.cig_off.tolist(), records.cigar.tolist()
    seg_off = records.seg_off.tolist()
    for s, chrom in enumerate(records.seg_chrom.tolist()):
        if chrom < 0 or chrom >= n_chrom:
            continue
        for r in range(seg_off[s], seg_off[s + 1]):
            st = _strand(flg[r], flags)
            cur, left, pl, plen, pleft = pos[r], 0, 0, -1, 0
            ops = cig[off[r]:off[r + 1]] + [3]    # a virtual N closes the last stretch
            last = len(ops) - 1
            for k, v in enumerate(ops):
                op, ln = v & 15, v >> 4
                if op == 3:
                    if plen >= 0 and min_intron <= plen <= max_intron and pleft >= min_anchor and left >= min_anchor:
                        row = rows.setdefault((chrom, pl, pl + plen, st), [0, 0, 0])
                        row[0] += 1
                        row[1] = max(row[1], pleft)
                        row[2] = max(row[2], left)
                    pl, plen, pleft, left = cur - 1, (ln if k < last else -1), left, 0
                    cur += ln
                elif op in _ADV:
                    left += ln
                    cur += ln
    keys = sorted(rows, key=lambda k: (k[0], k[1], k[2], _STRAND_ORDER[k[3]]))
    val = [rows[k] for k in keys]
    return Junctions(np.array([k[0] for k in keys], np.int32), np.array([k[1] for k in keys], np.int32),
                     np.array([k[2] for k in keys], np.int32), np.array([v[0] for v in val], np.int64),
                     np.array([k[3] for k in keys], np.uint8),
                     np.array([k[1] - v[1] for k, v in zip(keys, val)], np.int32),
                     np.array([k[2] + v[2] for k, v in zip(keys, val)], np.int32))


def filter_rows(junc, chroms, qchrom="All", gene_bounds=None, max_intron=0):
    """The rows of `junc` that `process` keeps of a BED12 holding them: -c (S:269) and the -g window (S:279-288)."""
    from spliser_b200.api import Junctions
    keep = np.ones(len(junc), bool)
    if qchrom != "All":
        keep &= np.array([chroms[c] == qchrom for c in junc.chrom.tolist()], bool)
    if gene_bounds is not None:
        gl, gr = gene_bounds
        lf, rt = junc.left.astype(np.int64), junc.right.astype(np.int64)
        keep &= ((lf + max_intron >= gl) & (lf <= gr)) | ((rt - max_intron <= gr) & (rt >= gl))
    return Junctions(junc.chrom[keep], junc.left[keep], junc.right[keep], junc.score[keep], junc.strand[keep],
                     None if junc.start is None else junc.start[keep], None if junc.end is None else junc.end[keep])


def bed_text(chroms, junc):
    """The bytes spl_write_junctions_bed writes for `junc` (regtools' BED12 layout)."""
    out = []
    for i in range(len(junc)):
        s, e = int(junc.start[i]), int(junc.end[i])
        a, b = int(junc.left[i]) - s, e - int(junc.right[i])
        st = int(junc.strand[i])
        out.append("%s\t%d\t%d\tJUNC%08d\t%d\t%s\t%d\t%d\t255,0,0\t2\t%d,%d\t0,%d\n" % (
            chroms[int(junc.chrom[i])], s, e, i + 1, int(junc.score[i]), chr(st) if st else "", s, e, a, b, e - s - b))
    return "".join(out)
