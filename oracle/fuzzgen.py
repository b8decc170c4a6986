"""TEST INFRASTRUCTURE ONLY -- seeded random case generator shared by oracle/make_golden.py
(reference vs oracle, authoring container) and the parity tests (CUDA vs oracle, GPU box).

The generator follows SURVEY.md Appendix B: a handful of site positions on a coarse grid,
junction lines with random scores/strands, and reads made of 1-4 mapped blocks whose ends
snap to site positions most of the time, separated by N / D / I / short-N operators, with
optional soft clips and the SAM flag combinations that exercise check_strand
(SpliSER_v0_1_8.py:374-406).
"""
from __future__ import annotations

import random

from .ref_runner import bed_line  # pure string helper, no reference needed

FLAGS = (0, 16, 99, 147, 83, 163, 1, 65, 129, 256, 1040, 81, 161, 97, 145)


def gen_case(seed, *, n_chrom=1, dirty=False, max_reads=39, grid_lo=100, grid_hi=1000):
    rng = random.Random(seed)
    chroms = ["C%d" % i for i in range(n_chrom)] if n_chrom > 1 else ["C"]
    stranded = rng.random() < 0.6
    stype = rng.choice(["fr", "rf"]) if stranded else None
    cryptic = rng.random() < 0.5
    bed, reads = [], []
    strand_choices = ["+", "-", "?"] if dirty else ["+", "-"]
    for chrom in chroms:
        nsite = rng.randint(4, 9)
        grid = sorted(rng.sample(range(grid_lo, grid_hi, 10), nsite))
        njl = rng.randint(2, 8)
        for _ in range(njl):
            l, r = sorted(rng.sample(grid, 2))
            if stranded:
                strand = rng.choice(strand_choices)
            else:
                strand = rng.choice(["+", "-", "?", "."])
            bed.append(bed_line(chrom, l, r, rng.randint(1, 8), strand))
        if rng.random() < 0.15:
            bed.append("track name=junctions\n")          # non-12-column line is skipped (S:259)
        nreads = rng.randint(5, max_reads)
        for _ in range(nreads):
            reads.append((chrom,) + _gen_read(rng, grid))
    reads.sort(key=lambda x: (chroms.index(x[0]), x[1]))  # coordinate-sorted like a real BAM
    return dict(seed=seed, chroms=chroms, bed="".join(bed), reads=reads, stranded=stranded,
                stype=stype, cryptic=cryptic)


def _gen_read(rng, grid):
    """Builds a read right-to-left from a chain of reference boundaries so that block ends land
    exactly on the site conventions: a block ending at site l covers up to l (next op starts at
    l+1); an N ending at r (last intron base) is followed by a block starting at r+1."""
    nblk = rng.choice([1, 1, 1, 2, 2, 3, 4])
    lo, hi = grid[0] - 40, grid[-1] + 40
    pos = rng.randint(lo, hi)
    # optionally snap the start so that the first block begins right after an acceptor-style site
    if rng.random() < 0.3:
        pos = rng.choice(grid) + rng.choice([1, 1, 0, 2, -1])
    cur = pos
    ops = []
    if rng.random() < 0.15:
        ops.append("%dS" % rng.randint(1, 9))
    for b in range(nblk):
        # block end: 70 % snapped so that the block's last base is a grid site (or site+1: covers it)
        if rng.random() < 0.7:
            cands = [g for g in grid if g >= cur]
            if cands:
                end = rng.choice(cands[:3]) + rng.choice([0, 0, 0, 1, 2, -1])  # last base of block
                blen = max(1, end - cur + 1)
            else:
                blen = rng.randint(1, 60)
        else:
            blen = rng.randint(1, 80)
        kind = rng.choice(["M", "M", "M", "M", "=", "X"])
        ops.append("%d%s" % (blen, kind))
        cur += blen
        if b == nblk - 1:
            break
        sep = rng.random()
        if sep < 0.55:                       # N, 80 % snapped: last intron base on a grid site
            if rng.random() < 0.8:
                cands = [g for g in grid if g >= cur]
                if cands:
                    r = rng.choice(cands[:4])
                    nlen = max(1, r - cur + 1)
                else:
                    nlen = rng.randint(1, 120)
            else:
                nlen = rng.randint(1, 150)
            ops.append("%dN" % nlen)
            cur += nlen
            if rng.random() < 0.08:          # back-to-back N / D after N
                extra = rng.randint(1, 30)
                ops.append("%d%s" % (extra, rng.choice(["N", "D"])))
                cur += extra
        elif sep < 0.72:
            d = rng.randint(1, 12)
            ops.append("%dD" % d)
            cur += d
        elif sep < 0.88:
            ops.append("%dI" % rng.randint(1, 5))
        else:
            n = rng.randint(1, 15)           # short N
            ops.append("%dN" % n)
            cur += n
    if rng.random() < 0.15:
        ops.append("%dS" % rng.randint(1, 9))
    if rng.random() < 0.03:
        ops.append("3H")
    flag = rng.choice(FLAGS)
    cigar = "".join(ops)
    if rng.random() < 0.02:
        cigar = "*"
    return (max(1, pos), flag, cigar)


LONG_FLAGS = FLAGS + (2048, 2064, 272)


def gen_long_case(seed, *, dirty=False, max_long=14, max_short=20):
    """Long-read shapes in the dict layout of gen_case: reads that walk 5-40 exons whose ends snap to a site grid (junction
    ends land on hot anchors), small I / D every 5-60 bp inside the blocks, leading and trailing N or D, zero-length M / N / D,
    back-to-back N N and N D, soft and hard clips, and the flags of gen_case plus 256 and 2048.  Junction rows often come on
    both strands at the same positions (two sites per position), and some grid sites are hubs with six or more partners, so
    one (junction, side) is a partner/competitor pair for five sites or more.  Short gen_case reads are mixed in."""
    rng = random.Random(seed)
    n_chrom = rng.choice([1, 1, 2])
    chroms = ["C%d" % i for i in range(n_chrom)] if n_chrom > 1 else ["C"]
    stranded = rng.random() < 0.6
    stype = rng.choice(["fr", "rf"]) if stranded else None
    cryptic = rng.random() < 0.5
    bed, reads = [], []
    strands = ["+", "-", "?"] if dirty else ["+", "-"]
    for chrom in chroms:
        nsite = rng.randint(10, 40)
        grid, p = [], rng.randint(200, 400)
        for _ in range(nsite):
            grid.append(p)
            p += rng.randint(12, 90)
        rows = []
        for _ in range(rng.randint(10, 60)):
            a = rng.randrange(len(grid) - 1)
            b = min(len(grid) - 1, a + rng.randint(1, 4))
            rows.append((grid[a], grid[b]))
        if rng.random() < 0.5:                                       # a hub: one site partnered with six or more others
            h = rng.randrange(len(grid))
            others = [g for g in grid if g != grid[h]]
            for o in rng.sample(others, min(len(others), rng.randint(6, 9))):
                rows.append((min(o, grid[h]), max(o, grid[h])))
        for l, r in rows:
            st = rng.choice(strands) if stranded else rng.choice(["+", "-", "?", "."])
            bed.append(bed_line(chrom, l, r, rng.randint(1, 8), st))
            if rng.random() < 0.3:                                   # the same junction on the other strand
                bed.append(bed_line(chrom, l, r, rng.randint(1, 8), {"+": "-", "-": "+"}.get(st, "+")))
        for _ in range(rng.randint(1, max_long)):
            reads.append((chrom,) + _gen_long_read(rng, grid))
        for _ in range(rng.randint(0, max_short)):
            reads.append((chrom,) + _gen_read(rng, grid))
    rng.shuffle(bed)
    reads.sort(key=lambda x: (chroms.index(x[0]), x[1]))
    return dict(seed=seed, chroms=chroms, bed="".join(bed), reads=reads, stranded=stranded, stype=stype, cryptic=cryptic)


def _block_ops(rng, blen, ops, split):
    """A mapped block of reference length blen (>= 1): M / = / X pieces of 5-60 bp split by small I or D (or one piece)."""
    if not split:
        ops.append("%d%s" % (blen, rng.choice("MMMM=X")))
        return
    rem = blen
    while rem > 0:
        m = min(rem, rng.randint(5, 60))
        ops.append("%d%s" % (m, rng.choice("MMMM=X")))
        rem -= m
        if rem > 1 and rng.random() < 0.4:
            d = min(rng.randint(1, 3), rem - 1)
            ops.append("%dD" % d)
            rem -= d
        elif rem > 0 and rng.random() < 0.4:
            ops.append("%dI" % rng.randint(1, 4))
        if rng.random() < 0.03:
            ops.append("0%s" % rng.choice("MND"))


def _gen_long_read(rng, grid):
    """One read across 5-40 exons: a block ends on a grid site (its last base, 75 %), the N that follows ends on a grid site
    (its last base, 85 %) so that the next block starts right after it."""
    ops = []
    if rng.random() < 0.1:
        ops.append("%dH" % rng.randint(1, 20))
    if rng.random() < 0.3:
        ops.append("%dS" % rng.randint(1, 40))
    start = rng.choice(grid) + rng.choice([1, 1, 1, 0, -5, -20])
    cur = start
    split = rng.random() < 0.7                                       # else unsplit blocks: often more than two N in five operators
    if rng.random() < 0.25:                                          # leading N / D: nothing advanced before it
        n = rng.choice([0, 1, 7, 30])
        ops.append("%d%s" % (n, rng.choice("ND")))
        cur += n
    nblk = rng.randint(5, 40)
    for b in range(nblk):
        cands = [g for g in grid if g >= cur]
        if cands and rng.random() < 0.75:
            end = rng.choice(cands[:3])
            blen = max(1, end - cur + 1)
        else:
            blen = rng.randint(1, 70)
        _block_ops(rng, blen, ops, split)
        cur += blen
        if b == nblk - 1:
            break
        sep = rng.random()
        cands = [g for g in grid if g > cur]
        if sep < 0.7 and cands:
            r = rng.choice(cands[:4]) if rng.random() < 0.85 else cur + rng.randint(0, 40)
            n = r - cur + 1
            ops.append("%dN" % n)
            cur += n
            if rng.random() < 0.1:                                   # back-to-back N N / N D
                e = rng.randint(0, 25)
                ops.append("%d%s" % (e, rng.choice("ND")))
                cur += e
        elif sep < 0.78:
            ops.append("0N")                                         # zero-length N: both ends on one position
        elif sep < 0.88:
            d = rng.randint(1, 15)
            ops.append("%dD" % d)
            cur += d
        else:
            n = rng.randint(1, 15)
            ops.append("%dN" % n)
            cur += n
    if rng.random() < 0.2:                                           # trailing N / D
        ops.append("%d%s" % (rng.choice([0, 1, 9, 40]), rng.choice("ND")))
    if rng.random() < 0.3:
        ops.append("%dS" % rng.randint(1, 40))
    if rng.random() < 0.1:
        ops.append("%dH" % rng.randint(1, 20))
    return (max(1, start), rng.choice(LONG_FLAGS), "".join(ops))


def gen_combine_case(seed):
    """Two or three samples over one shared site universe; each sample sees a random subset of
    the junction lines, so the combined table has gaps that need a re-count (S:899-904)."""
    rng = random.Random(seed)
    stranded = rng.random() < 0.5
    stype = rng.choice(["fr", "rf"])
    nsite = rng.randint(5, 9)
    grid = sorted(rng.sample(range(100, 1000, 10), nsite))
    universe = []
    for _ in range(rng.randint(4, 9)):
        l, r = sorted(rng.sample(grid, 2))
        universe.append((l, r, rng.choice(["+", "-"])))
    samples = []
    for s in range(rng.randint(2, 3)):
        keep = [j for j in universe if rng.random() < 0.6] or [universe[0]]
        bed = "".join(bed_line("C", l, r, rng.randint(1, 8), st) for l, r, st in keep)
        reads = sorted((("C",) + _gen_read(rng, grid) for _ in range(rng.randint(5, 30))),
                       key=lambda x: x[1])
        samples.append(dict(title="S%d" % s, bed=bed, reads=reads))
    return dict(seed=seed, samples=samples, stranded=stranded, stype=stype)


def gen_combine_wide_case(seed):
    """`combine` beyond the single-region cases: 2-5 samples over 1-3 regions (a sample may lack a whole region, which
    exercises the region order of S:761-789), a GFF so that the Gene column is filled and `-g` can filter the merged
    rows (S:908), `--beta2Cryptic` on about half the cases (beta2_weighted goes through str(float), S:734), overlapping
    genes on both strands."""
    rng = random.Random(seed)
    stranded = rng.random() < 0.5
    stype = rng.choice(["fr", "rf"])
    cryptic = rng.random() < 0.5
    chroms = ["K%d" % i for i in range(rng.randint(1, 3))]
    gff, grids, universe, genes = [], {}, {}, []
    for c in chroms:
        nsite = rng.randint(5, 9)
        grids[c] = sorted(rng.sample(range(100, 1000, 10), nsite))
        universe[c] = []
        for _ in range(rng.randint(4, 9)):
            l, r = sorted(rng.sample(grids[c], 2))
            universe[c].append((l, r, rng.choice(["+", "-"])))
        cut = rng.randrange(300, 800, 10)
        spans = [(90, cut + rng.choice([0, 0, 60])), (cut, 1010)]
        if rng.random() < 0.3:
            spans.append((rng.randrange(100, 500, 10), rng.randrange(510, 1000, 10)))
        for k, (a, b) in enumerate(spans):
            name = "%s_g%d" % (c, k)
            genes.append(name)
            gff.append("%s\tx\tgene\t%d\t%d\t.\t%s\t.\tID=%s;Name=n%d\n" % (c, a, b, rng.choice(["+", "-"]), name, k))
    samples = []
    for s in range(rng.randint(2, 5)):
        present = [c for c in chroms if rng.random() < 0.8] or [chroms[0]]
        bed, reads = [], []
        for c in present:
            keep = [j for j in universe[c] if rng.random() < 0.6] or [universe[c][0]]
            bed.extend(bed_line(c, l, r, rng.randint(1, 8), st) for l, r, st in keep)
        for c in chroms:
            reads.extend(sorted(((c,) + _gen_read(rng, grids[c]) for _ in range(rng.randint(5, 30))), key=lambda x: x[1]))
        samples.append(dict(title="W%d" % s, bed="".join(bed), reads=reads))
    qgene = rng.choice(genes) if rng.random() < 0.3 else "All"
    return dict(seed=seed, chroms=chroms, samples=samples, stranded=stranded, stype=stype, cryptic=cryptic,
                gff="".join(gff), qgene=qgene)
