"""Seeded synthetic RNA-seq workloads of the shapes BASELINE.json names (SURVEY.md 8(d)).

Everything is vectorised numpy: gene models -> transcripts (with alternative 5'/3' sites and
skipped exons so that competitor / flanking / mutually-exclusive reads exist) -> fragments ->
reads as BAM-style records (POS, FLAG, CIGAR ops) sorted by coordinate, plus the regtools-style
junction table (every junction with a read whose two anchors are >= 8 bp, score = read count).
No file is read: the generator must run on the GPU box, where /root/reference does not exist.
"""
from __future__ import annotations

import hashlib
import os
from dataclasses import asdict, dataclass, field

import numpy as np

from .api import Junctions, Records

OP_M, OP_I, OP_D, OP_N, OP_S = 0, 1, 2, 3, 4

TAIR10 = (("Chr1", 30427671), ("Chr2", 19698289), ("Chr3", 23459830), ("Chr4", 18585056),
          ("Chr5", 26975502), ("ChrC", 154478), ("ChrM", 366924))
GRCH38 = (("chr1", 248956422), ("chr2", 242193529), ("chr3", 198295559), ("chr4", 190214555),
          ("chr5", 181538259), ("chr6", 170805979), ("chr7", 159345973), ("chr8", 145138636),
          ("chr9", 138394717), ("chr10", 133797422), ("chr11", 135086622), ("chr12", 133275309),
          ("chr13", 114364328), ("chr14", 107043718), ("chr15", 101991189), ("chr16", 90338345),
          ("chr17", 83257441), ("chr18", 80373285), ("chr19", 58617616), ("chr20", 64444167),
          ("chr21", 46709983), ("chr22", 50818468), ("chrX", 156040895), ("chrY", 57227415))


@dataclass
class SynthConfig:
    name: str = "c1"
    seed: int = 20260001
    contigs: tuple = (("Chr1", 30427671),)
    n_records: int = 2_000_000
    read_len: int = 100
    paired: bool = False
    stranded: bool = False            # BED strand column: gene strand if True, '?' otherwise
    genes_per_mb: float = 165.0
    exon_median: float = 150.0
    intron_median: float = 100.0
    intron_min: int = 70
    intron_max: int = 6000
    mean_exons: float = 5.0
    frac_alt_site: float = 0.20       # genes with an alternative 5'/3' splice site isoform
    frac_exon_skip: float = 0.05      # genes with an exon-skipping isoform
    frac_retained: float = 0.02       # reads drawn from unspliced pre-mRNA (cover splice sites -> beta1)
    frac_indel: float = 0.01
    frac_softclip: float = 0.01
    frac_odd_flag: float = 0.005      # secondary / duplicate bits added (the reference filters nothing, S:422)
    fragment_mean: int = 300
    min_anchor: int = 8
    organelle_share: float = 0.0      # share of reads on contigs shorter than 1 Mb
    extra_isoforms: int = 0           # per multi-exon gene: isoforms with random exon skipping / shifted boundaries (dense loci)
    per_contig_rng: bool = False      # every contig draws from its own generator (seed, contig index): contigs can be built in parallel

    def key(self) -> str:
        return hashlib.sha1(repr(sorted(asdict(self).items())).encode()).hexdigest()[:16]


def config_c1() -> SynthConfig:
    return SynthConfig()


def config_c2(n_records=40_000_000) -> SynthConfig:
    return SynthConfig(name="c2", seed=20260002, contigs=TAIR10, n_records=n_records, read_len=150, paired=True,
                       stranded=True, genes_per_mb=240.0, organelle_share=0.02)


def config_c3_tile(n_records=25_000_000, tile=0, n_tiles=8) -> SynthConfig:
    """One genomic tile of the GRCh38-scale config: contigs dealt round-robin to tiles."""
    contigs = tuple(c for i, c in enumerate(GRCH38) if i % n_tiles == tile)
    return SynthConfig(name="c3t%d" % tile, seed=20260003 + 100 * tile, contigs=contigs, n_records=n_records, read_len=150,
                       paired=True, stranded=True, genes_per_mb=9.0, exon_median=140.0, intron_median=1500.0,
                       intron_min=70, intron_max=500_000, mean_exons=9.0)


def config_c3_full(n_records=200_000_000) -> SynthConfig:
    """BASELINE configs[2]: GRCh38 primary contig lengths, 150 bp PE records, ~400k junctions, introns up to 500 kb."""
    return SynthConfig(name="c3full", seed=20260003, contigs=GRCH38, n_records=n_records, read_len=150, paired=True,
                       stranded=True, genes_per_mb=9.0, exon_median=140.0, intron_median=1500.0, intron_min=70,
                       intron_max=500_000, mean_exons=9.0, per_contig_rng=True)


def config_c5() -> SynthConfig:
    return SynthConfig(name="c5", seed=20260005, contigs=(("L1", 2_000_000),), n_records=1_000_000, read_len=100,
                       genes_per_mb=1.0, mean_exons=400.0, exon_median=120.0, intron_median=900.0, intron_max=20000,
                       frac_alt_site=1.0, frac_exon_skip=1.0, extra_isoforms=12)


def config_small(n_records=20000, seed=1, stranded=False, paired=False) -> SynthConfig:
    return SynthConfig(name="small", seed=seed, contigs=(("T1", 400_000), ("T2", 250_000)), n_records=n_records,
                       read_len=75, paired=paired, stranded=stranded, genes_per_mb=120.0, organelle_share=0.0)


@dataclass
class Workload:
    cfg: SynthConfig
    chroms: list
    chrom_len: list
    records: Records
    junctions: Junctions
    junction_strand_str: list = field(default_factory=list)

    @property
    def flags(self) -> int:
        return (1 | 2) if self.cfg.stranded else 0      # --isStranded -s rf for the dUTP-style flags below

    def bed12_text(self) -> str:
        j = self.junctions
        a = self.cfg.min_anchor
        out = []
        for i in range(len(j)):
            l, r = int(j.left[i]), int(j.right[i])
            s, e = l - a, r + a
            out.append("\t".join(map(str, [self.chroms[int(j.chrom[i])], s, e, "JUNC%08d" % i, int(j.score[i]),
                                           chr(int(j.strand[i])), s, e, "255,0,0", 2, "%d,%d" % (a, a),
                                           "0,%d" % (r - l + a)])) + "\n")
        return "".join(out)


# --------------------------------------------------------------------------------------------------
def _gene_models(rng, cfg, clen):
    """Returns transcripts of one contig as flat exon arrays:
    t_off [T+1] into exon arrays, ex_start, ex_len (1-based inclusive start), t_strand [T], t_gene [T], gene span."""
    n_genes = max(1, int(clen / 1e6 * cfg.genes_per_mb))
    n_ex = 1 + rng.geometric(1.0 / cfg.mean_exons, size=n_genes)
    n_ex = np.minimum(n_ex, 2000)
    tot = int(n_ex.sum())
    ex_len = np.maximum(30, rng.lognormal(np.log(cfg.exon_median), 0.6, size=tot)).astype(np.int64)
    in_len = np.clip(rng.lognormal(np.log(cfg.intron_median), 0.9, size=tot), cfg.intron_min, cfg.intron_max).astype(np.int64)
    g_off = np.zeros(n_genes + 1, np.int64)
    np.cumsum(n_ex, out=g_off[1:])
    first = np.zeros(tot, bool)
    first[g_off[:-1]] = True
    in_len[first] = 0                                   # "intron before exon": none before the first exon of a gene
    span = np.add.reduceat(ex_len + in_len, g_off[:-1])
    gap_total = clen - int(span.sum()) - 2000
    if gap_total < n_genes:                             # too dense for this contig: thin the gene list
        keep = max(1, int(n_genes * (clen - 2000) / (span.sum() + n_genes * 200.0)))
        return _gene_models_subset(rng, cfg, clen, keep, n_ex, ex_len, in_len, g_off)
    gaps = rng.dirichlet(np.ones(n_genes + 1)) * gap_total
    g_start = 1000 + np.floor(np.cumsum(gaps[:-1])).astype(np.int64) + np.concatenate(([0], np.cumsum(span)[:-1]))
    return _finish_models(rng, cfg, n_genes, n_ex, ex_len, in_len, g_off, g_start)


def _gene_models_subset(rng, cfg, clen, keep, n_ex, ex_len, in_len, g_off):
    n_ex = n_ex[:keep]
    tot = int(n_ex.sum())
    ex_len, in_len = ex_len[:tot], in_len[:tot]
    g_off = g_off[:keep + 1]
    span = np.add.reduceat(ex_len + in_len, g_off[:-1])
    scale = min(1.0, (clen - 2000 - keep * 50) / float(span.sum()))
    if scale < 1.0:
        in_len = np.maximum((in_len * scale).astype(np.int64), np.where(in_len > 0, cfg.intron_min, 0))
        span = np.add.reduceat(ex_len + in_len, g_off[:-1])
    gap_total = max(keep, clen - int(span.sum()) - 2000)
    gaps = rng.dirichlet(np.ones(keep + 1)) * gap_total
    g_start = 1000 + np.floor(np.cumsum(gaps[:-1])).astype(np.int64) + np.concatenate(([0], np.cumsum(span)[:-1]))
    return _finish_models(rng, cfg, keep, n_ex, ex_len, in_len, g_off, g_start)


def _finish_models(rng, cfg, n_genes, n_ex, ex_len, in_len, g_off, g_start):
    tot = len(ex_len)
    gene_of = np.repeat(np.arange(n_genes), n_ex)
    c = np.cumsum(ex_len + in_len)
    gene_base = np.concatenate(([0], c[g_off[1:-1] - 1]))      # cumulative length before each gene
    within = c - np.repeat(gene_base, n_ex)                    # offset of each exon's last base inside its gene
    ex_end = np.repeat(g_start, n_ex) + within - 1          # inclusive end
    ex_start = ex_end - ex_len + 1
    strand = rng.integers(0, 2, size=n_genes)               # 0 '+', 1 '-'
    # canonical transcripts
    t_off = [g_off.copy()]
    exs, exl, tstr, tgene = [ex_start], [ex_len], [strand], [np.arange(n_genes)]
    base = tot
    # alternative splice site isoform: move one internal exon boundary inwards by 5..60 bp
    multi = np.nonzero(n_ex >= 3)[0]
    pick = multi[rng.random(len(multi)) < cfg.frac_alt_site]
    if len(pick):
        counts = n_ex[pick]
        idx = np.concatenate([np.arange(g_off[g], g_off[g + 1]) for g in pick])
        a_start, a_len = ex_start[idx].copy(), ex_len[idx].copy()
        off = np.zeros(len(pick) + 1, np.int64)
        np.cumsum(counts, out=off[1:])
        which = off[:-1] + 1 + (rng.random(len(pick)) * (counts - 2)).astype(np.int64)   # an internal exon
        shift = rng.integers(5, 61, size=len(pick))
        shift = np.minimum(shift, a_len[which] - 20)
        ok = shift > 0
        side = rng.random(len(pick)) < 0.5
        # donor side: shorten the exon's end; acceptor side: move the exon's start right
        sel = which[ok & side]
        a_len[sel] -= shift[ok & side]
        sel = which[ok & ~side]
        a_start[sel] += shift[ok & ~side]
        a_len[sel] -= shift[ok & ~side]
        exs.append(a_start); exl.append(a_len); tstr.append(strand[pick]); tgene.append(pick)
        t_off.append(base + off)
        base += len(idx)
    # exon skipping isoform: drop one internal exon
    pick = multi[rng.random(len(multi)) < cfg.frac_exon_skip]
    if len(pick):
        counts = n_ex[pick]
        idx = np.concatenate([np.arange(g_off[g], g_off[g + 1]) for g in pick])
        off = np.zeros(len(pick) + 1, np.int64)
        np.cumsum(counts, out=off[1:])
        drop = off[:-1] + 1 + (rng.random(len(pick)) * (counts - 2)).astype(np.int64)
        keepm = np.ones(len(idx), bool)
        keepm[drop] = False
        exs.append(ex_start[idx][keepm]); exl.append(ex_len[idx][keepm]); tstr.append(strand[pick]); tgene.append(pick)
        off2 = off - np.arange(len(pick) + 1)
        t_off.append(base + off2)
        base += int(keepm.sum())
    # dense alternative combinations (configs[4]): several isoforms per gene, each skipping a random subset of the
    # internal exons and moving some exon boundaries
    if cfg.extra_isoforms:
        for gidx in multi:
            e0, e1 = int(g_off[gidx]), int(g_off[gidx + 1])
            for _ in range(cfg.extra_isoforms):
                keep = rng.random(e1 - e0) > 0.3
                keep[0] = keep[-1] = True
                st = ex_start[e0:e1][keep].copy()
                ln = ex_len[e0:e1][keep].copy()
                sh = rng.integers(0, 40, size=len(st)) * (rng.random(len(st)) < 0.25)
                sh = np.minimum(sh, ln - 20) * (ln > 40)
                side = rng.random(len(st)) < 0.5
                st = st + np.where(side, 0, sh)
                ln = ln - sh
                exs.append(st); exl.append(ln); tstr.append(strand[gidx:gidx + 1]); tgene.append(np.array([gidx]))
                t_off.append(np.array([base, base + len(st)], dtype=np.int64))
                base += len(st)
    ex_start_all = np.concatenate(exs)
    ex_len_all = np.concatenate(exl)
    offs = [t_off[0]] + [o[1:] for o in t_off[1:]]
    t_off_all = np.concatenate(offs)
    t_strand = np.concatenate(tstr)
    t_gene = np.concatenate(tgene)
    g_end = ex_end[g_off[1:] - 1]
    return dict(t_off=t_off_all, ex_start=ex_start_all, ex_len=ex_len_all, t_strand=t_strand, t_gene=t_gene,
                g_start=g_start, g_end=g_end, g_strand=strand)


def _reads_for_contig(rng, cfg, m, n_rec):
    """-> pos, flag, ncig, ops(list of arrays per slot) for n_rec records on one contig."""
    L = cfg.read_len
    t_off, ex_start, ex_len = m["t_off"], m["ex_start"], m["ex_len"]
    T = len(t_off) - 1
    t_len = np.add.reduceat(ex_len, t_off[:-1])
    glob = np.zeros(len(ex_len) + 1, np.int64)
    np.cumsum(ex_len, out=glob[1:])
    n_frag = n_rec // 2 if cfg.paired else n_rec
    n_ret = int(round(n_frag * cfg.frac_retained))
    n_spl = n_frag - n_ret
    # expression: lognormal per gene, isoforms share it
    g_expr = rng.lognormal(0.0, 1.6, size=len(m["g_start"]))
    usable = t_len >= L
    w = g_expr[m["t_gene"]] * np.maximum(t_len - L + 1, 0) * usable
    if w.sum() <= 0:
        w = usable.astype(float) + 1e-9
    cdf = np.cumsum(w / w.sum())
    tsel = np.minimum(np.searchsorted(cdf, rng.random(n_spl), side="right"), T - 1)
    frag_len = np.clip(rng.normal(cfg.fragment_mean, 40, size=n_spl).astype(np.int64), L, None) if cfg.paired else np.full(n_spl, L)
    frag_len = np.minimum(frag_len, t_len[tsel])
    f_start = (rng.random(n_spl) * (t_len[tsel] - frag_len + 1)).astype(np.int64)          # transcript coordinate
    if cfg.paired:
        x = np.concatenate([f_start, f_start + frag_len - L])
        tt = np.concatenate([tsel, tsel])
        mate = np.concatenate([np.zeros(n_spl, np.int8), np.ones(n_spl, np.int8)])       # 0 = left mate, 1 = right mate
    else:
        x, tt, mate = f_start, tsel, np.zeros(n_spl, np.int8)
    gx = glob[t_off[tt]] + x                                                              # global exon-space coordinate
    e0 = np.searchsorted(glob, gx, side="right") - 1
    e1 = np.searchsorted(glob, gx + L - 1, side="right") - 1
    nblk = (e1 - e0 + 1).astype(np.int64)
    pos = ex_start[e0] + (gx - glob[e0])
    kmax = int(nblk.max()) if len(nblk) else 1
    n = len(gx)
    # op slots: block0, N0, block1, N1, ...
    ops = np.zeros((n, 2 * kmax - 1), np.uint32)
    remaining = np.full(n, L, np.int64)
    cur_e = e0.copy()
    first_len = np.minimum(remaining, glob[e0 + 1] - gx)
    ops[:, 0] = (first_len.astype(np.uint32) << 4) | OP_M
    remaining -= first_len
    for k in range(1, kmax):
        act = nblk > k
        if not act.any():
            break
        nxt = cur_e + 1
        nlen = np.where(act, ex_start[np.minimum(nxt, len(ex_start) - 1)] - (ex_start[cur_e] + ex_len[cur_e]), 0)
        blen = np.where(act, np.minimum(remaining, ex_len[np.minimum(nxt, len(ex_len) - 1)]), 0)
        ops[:, 2 * k - 1] = np.where(act, (nlen.astype(np.uint32) << 4) | OP_N, 0)
        ops[:, 2 * k] = np.where(act, (blen.astype(np.uint32) << 4) | OP_M, 0)
        remaining -= blen
        cur_e = np.where(act, nxt, cur_e)
    strand = m["t_strand"][tt]
    # retained-intron / pre-mRNA reads: one block anywhere inside a gene's genomic span
    if n_ret:
        gw = g_expr * np.maximum(m["g_end"] - m["g_start"] + 1 - L, 0)
        if gw.sum() <= 0:
            gw = np.ones_like(gw)
        gsel = np.minimum(np.searchsorted(np.cumsum(gw / gw.sum()), rng.random(n_ret), side="right"), len(gw) - 1)
        glen = m["g_end"][gsel] - m["g_start"][gsel] + 1
        fl = np.minimum(np.clip(rng.normal(cfg.fragment_mean, 40, size=n_ret).astype(np.int64), L, None), np.maximum(glen, L)) if cfg.paired else np.full(n_ret, L)
        rs = m["g_start"][gsel] + (rng.random(n_ret) * np.maximum(glen - fl + 1, 1)).astype(np.int64)
        if cfg.paired:
            rpos = np.concatenate([rs, rs + fl - L])
            rmate = np.concatenate([np.zeros(n_ret, np.int8), np.ones(n_ret, np.int8)])
            rstrand = np.concatenate([m["g_strand"][gsel]] * 2)
        else:
            rpos, rmate, rstrand = rs, np.zeros(n_ret, np.int8), m["g_strand"][gsel]
        rops = np.zeros((len(rpos), ops.shape[1]), np.uint32)
        rops[:, 0] = (np.uint32(L) << 4) | OP_M
        pos = np.concatenate([pos, rpos]); ops = np.concatenate([ops, rops])
        mate = np.concatenate([mate, rmate]); strand = np.concatenate([strand, rstrand])
    n = len(pos)
    # flags
    if cfg.paired:
        # dUTP / rf: '+' gene -> left mate is read 2 forward (163), right mate read 1 reverse (83);
        #            '-' gene -> left mate is read 1 forward (99), right mate read 2 reverse (147)
        flag = np.where(strand == 0, np.where(mate == 0, 163, 83), np.where(mate == 0, 99, 147)).astype(np.uint16)
    else:
        flag = np.where(rng.random(n) < 0.5, 0, 16).astype(np.uint16)
    odd = rng.random(n) < cfg.frac_odd_flag
    flag[odd] |= np.where(rng.random(int(odd.sum())) < 0.5, 256, 1024).astype(np.uint16)
    return pos.astype(np.int64), flag, ops, strand.astype(np.int8)


def _add_indels_softclips(rng, cfg, pos, ops):
    """Rewrites a small share of reads: split the first block with 1I / 2D, or soft-clip its start."""
    n, w = ops.shape
    extra = np.zeros((n, 2), np.uint32)                     # up to two ops inserted after slot 0
    pre = np.zeros(n, np.uint32)                            # optional leading soft clip
    first = (ops[:, 0] >> 4).astype(np.int64)
    r = rng.random(n)
    indel = (r < cfg.frac_indel) & (first >= 24)
    k = int(indel.sum())
    if k:
        cut = 8 + (rng.random(k) * (first[indel] - 16)).astype(np.int64)
        is_ins = rng.random(k) < 0.5
        a = cut
        b = first[indel] - cut - np.where(is_ins, 1, 0)     # an insertion consumes one read base
        ops[indel, 0] = (a.astype(np.uint32) << 4) | OP_M
        e = np.zeros((k, 2), np.uint32)
        e[:, 0] = np.where(is_ins, (1 << 4) | OP_I, (2 << 4) | OP_D)
        e[:, 1] = (b.astype(np.uint32) << 4) | OP_M
        extra[indel] = e
    clip = (r >= cfg.frac_indel) & (r < cfg.frac_indel + cfg.frac_softclip) & (first >= 20)
    k = int(clip.sum())
    if k:
        c = rng.integers(1, 9, size=k)
        pre[clip] = (c.astype(np.uint32) << 4) | OP_S
        ops[clip, 0] = ((first[clip] - c).astype(np.uint32) << 4) | OP_M
        pos = pos.copy()
        pos[clip] += c
    full = np.concatenate([pre[:, None], ops[:, :1], extra, ops[:, 1:]], axis=1)
    return pos, full


def _contig(cfg, rng, clen, n_rec):
    """Records + junction table of one contig."""
    m = _gene_models(rng, cfg, int(clen))
    pos, flag, ops, strand = _reads_for_contig(rng, cfg, m, int(n_rec))
    pos, ops = _add_indels_softclips(rng, cfg, pos, ops)
    order = np.argsort(pos, kind="stable")
    pos, flag, ops, strand = pos[order], flag[order], ops[order], strand[order]
    out = dict(jl=None, jr=None, js=None, jst=None)
    # junction table from the reads themselves (regtools-style anchors)
    w = ops.shape[1]
    is_n = (ops & 15) == OP_N
    is_n &= ops > 0
    adv = np.where(np.isin(ops & 15, (OP_M, OP_D, OP_N)) & (ops > 0), ops >> 4, 0).astype(np.int64)
    start_of_op = pos[:, None] + np.cumsum(adv, axis=1) - adv
    rr, cc = np.nonzero(is_n)
    if len(rr):
        left = start_of_op[rr, cc] - 1
        right = left + (ops[rr, cc] >> 4).astype(np.int64)
        pc = np.maximum(cc - 1, 0)
        nc = np.minimum(cc + 1, w - 1)
        # nearest non-empty op on each side is an M block by construction
        prev_m = (ops[rr, pc] >> 4) * ((ops[rr, pc] & 15) == OP_M)
        for back in (2, 3):
            pc2 = np.maximum(cc - back, 0)
            prev_m = np.where(prev_m == 0, (ops[rr, pc2] >> 4) * ((ops[rr, pc2] & 15) == OP_M) * (ops[rr, pc2] > 0), prev_m)
        next_m = (ops[rr, nc] >> 4) * ((ops[rr, nc] & 15) == OP_M)
        good = (prev_m >= cfg.min_anchor) & (next_m >= cfg.min_anchor)
        key = left[good] * (1 << 31) + right[good]
        uk, first_idx, cnt = np.unique(key, return_index=True, return_counts=True)
        out["jl"] = (uk >> 31).astype(np.int32); out["jr"] = (uk & ((1 << 31) - 1)).astype(np.int32)
        out["js"] = cnt.astype(np.int64)
        st = strand[rr][good][first_idx]
        out["jst"] = np.where(st == 0, ord("+"), ord("-")).astype(np.uint8) if cfg.stranded else np.full(len(uk), ord("?"), np.uint8)
    out["pos"] = pos.astype(np.int32); out["flag"] = flag
    out["ncig"] = (ops > 0).sum(axis=1).astype(np.int64)
    out["flat"] = ops[ops > 0]                                  # row-major: per-read op order is preserved
    return out


def _contig_job(args):
    cfg, ci, clen, n = args
    return _contig(cfg, np.random.default_rng([cfg.seed, ci]), clen, n)


def _contigs_parallel(cfg, todo, workers):
    """Contigs of a per_contig_rng config, built by a pool of processes (the result does not depend on the pool size)."""
    jobs = [(cfg, ci, clen, n) for ci, clen, n in todo]
    workers = max(1, min(int(workers or 1), len(jobs)))
    if workers == 1:
        return [_contig_job(j) for j in jobs]
    import multiprocessing as mp
    with mp.get_context("fork").Pool(workers) as pool:
        return pool.map(_contig_job, jobs, chunksize=1)


def generate(cfg: SynthConfig, cache_dir=None, workers=None) -> Workload:
    """Builds (or loads from the .npz cache) the workload for `cfg`.  workers: processes for per_contig_rng configs
    (default: half the cores)."""
    if workers is None:
        workers = max(1, (os.cpu_count() or 2) // 2)
    if cache_dir:
        path = os.path.join(cache_dir, "spliser_synth_%s_%s.npz" % (cfg.name, cfg.key()))
        if os.path.exists(path):
            z = np.load(path, allow_pickle=False)
            rec = Records(z["pos"], z["flag"], z["cig_off"], z["cigar"], z["seg_chrom"], z["seg_off"])
            j = Junctions(z["j_chrom"], z["j_left"], z["j_right"], z["j_score"], z["j_strand"])
            return Workload(cfg, [c for c, _ in cfg.contigs], [l for _, l in cfg.contigs], rec, j)
    rng = np.random.default_rng(cfg.seed)
    lens = np.array([l for _, l in cfg.contigs], float)
    small = lens < 1e6
    share = np.where(small, 0.0, lens)
    share = share / share.sum() * (1.0 - (cfg.organelle_share if small.any() else 0.0)) if share.sum() > 0 else np.ones_like(lens) / len(lens)
    if small.any() and share.sum() > 0:
        share = share + np.where(small, cfg.organelle_share / small.sum(), 0.0)
    n_per = np.floor(share * cfg.n_records).astype(np.int64)
    if cfg.paired:
        n_per -= n_per % 2
    n_per[int(np.argmax(n_per))] += cfg.n_records - int(n_per.sum())
    P, F, O, C = [], [], [], []
    seg_chrom, seg_off = [], [0]
    jc, jl, jr, js, jst = [], [], [], [], []
    total = 0
    todo = [(ci, int(clen), int(n_per[ci])) for ci, (cname, clen) in enumerate(cfg.contigs) if n_per[ci] > 0]
    if cfg.per_contig_rng:
        results = _contigs_parallel(cfg, todo, workers)
    else:
        results = (_contig(cfg, rng, clen, n) for ci, clen, n in todo)
    for (ci, clen, n), res in zip(todo, results):
        if res["jl"] is not None:
            jl.append(res["jl"]); jr.append(res["jr"]); js.append(res["js"]); jst.append(res["jst"])
            jc.append(np.full(len(res["jl"]), len(seg_chrom), np.int32))
        P.append(res["pos"]); F.append(res["flag"]); O.append(res["ncig"]); C.append(res["flat"])
        seg_chrom.append(ci)
        total += len(res["pos"])
        seg_off.append(total)
    pos = np.concatenate(P) if P else np.zeros(0, np.int32)
    flag = np.concatenate(F) if F else np.zeros(0, np.uint16)
    ncig = np.concatenate(O) if O else np.zeros(0, np.int64)
    cig_off = np.zeros(len(pos) + 1, np.uint32)
    np.cumsum(ncig, out=cig_off[1:])
    cigar = np.concatenate(C) if C else np.zeros(0, np.uint32)
    # chromosome index = position in cfg.contigs (every contig is listed, reads or not)
    chroms = [c for c, _ in cfg.contigs]
    rec = Records(pos, flag, cig_off, cigar, np.array(seg_chrom, np.int32), np.array(seg_off, np.int64))
    if jc:
        seg_to_chrom = np.array(seg_chrom, np.int32)
        j = Junctions(seg_to_chrom[np.concatenate(jc)], np.concatenate(jl), np.concatenate(jr), np.concatenate(js), np.concatenate(jst))
    else:
        j = Junctions(np.zeros(0, np.int32), np.zeros(0, np.int32), np.zeros(0, np.int32), np.zeros(0, np.int64), np.zeros(0, np.uint8))
    if cache_dir:
        os.makedirs(cache_dir, exist_ok=True)
        tmp = path + ".tmp.%d.npz" % os.getpid()
        np.savez(tmp, pos=rec.pos, flag=rec.flag, cig_off=rec.cig_off, cigar=rec.cigar, seg_chrom=rec.seg_chrom,
                 seg_off=rec.seg_off, j_chrom=j.chrom, j_left=j.left, j_right=j.right, j_score=j.score, j_strand=j.strand)
        os.replace(tmp, path)
    return Workload(cfg, chroms, [l for _, l in cfg.contigs], rec, j)


def config_long_reads(n_records=12_000, seed=20260011) -> SynthConfig:
    """Long-read RNA-seq (Iso-Seq / ONT shaped) for generate_long_reads: ~25 exons per gene, every gene with alternative sites,
    skipped exons and extra isoforms (most junction ends have competitors), reads of 1-10 kb, 5 % unspliced pre-mRNA reads."""
    return SynthConfig(name="long", seed=seed, contigs=(("L1", 1_500_000), ("L2", 1_000_000), ("L3", 1_000_000)), n_records=n_records,
                       read_len=10_000, stranded=True, genes_per_mb=25.0, exon_median=220.0, intron_median=600.0, intron_min=70,
                       intron_max=20_000, mean_exons=25.0, frac_alt_site=1.0, frac_exon_skip=1.0, extra_isoforms=3, frac_retained=0.05,
                       frac_softclip=0.2, frac_odd_flag=0.03)


LONG_MAX_OPS = 255          # operators per record: what CompactRecords can carry


def _long_block(rng, ops, blen):
    """One exon's stretch of a read: unsplit (so exons over FC_WALK bases stay one M) or split by small I / D every 10-120 bp."""
    if rng.random() < 0.4 or len(ops) > LONG_MAX_OPS - 24:
        ops.append((blen << 4) | OP_M)
        return
    rem = blen
    while rem > 0:
        m = min(rem, int(rng.integers(10, 121)))
        if len(ops) > LONG_MAX_OPS - 24:
            m = rem
        ops.append((m << 4) | OP_M)
        rem -= m
        if rem > 2 and rng.random() < 0.5:
            d = int(rng.integers(1, 3))
            ops.append((d << 4) | OP_D)
            rem -= d
        elif rem > 0:
            ops.append((int(rng.integers(1, 4)) << 4) | OP_I)


def _long_reads_for_contig(rng, cfg, m, n_rec):
    """-> pos, flag, per-record operator lists, junction (left, right) -> (count, strand) of one contig."""
    t_off, ex_start, ex_len = m["t_off"], m["ex_start"], m["ex_len"]
    t_len = np.add.reduceat(ex_len, t_off[:-1])
    g_expr = rng.lognormal(0.0, 1.0, size=len(m["g_start"]))
    w = g_expr[m["t_gene"]] * np.maximum(t_len - 999, 0)
    cdf = np.cumsum(w / w.sum())
    pos, flag, reads, junc = [], [], [], {}
    for _ in range(n_rec):
        ops = []
        if rng.random() < cfg.frac_softclip:
            ops.append((int(rng.integers(5, 60)) << 4) | OP_S)
        if rng.random() < cfg.frac_retained:                   # unspliced pre-mRNA: one block of 4096 bp or more
            g = int(rng.integers(0, len(m["g_start"])))
            L = int(rng.integers(4096, cfg.read_len + 1))
            p = int(m["g_start"][g]) + int(rng.integers(0, max(1, int(m["g_end"][g] - m["g_start"][g]) - L // 2)))
            ops.append((L << 4) | OP_M)
            strand = int(m["g_strand"][g])
        else:
            t = min(int(np.searchsorted(cdf, rng.random(), side="right")), len(t_len) - 1)
            L = min(int(rng.integers(1000, cfg.read_len + 1)), int(t_len[t]))
            x = int(rng.integers(0, int(t_len[t]) - L + 1))       # transcript coordinate of the first base
            e, e1 = int(t_off[t]), int(t_off[t + 1])
            while x >= ex_len[e]:
                x -= int(ex_len[e]); e += 1
            p = int(ex_start[e]) + x
            cur, rem = p, L
            while rem > 0 and e < e1 and len(ops) <= LONG_MAX_OPS - 3:
                blen = min(rem, int(ex_start[e] + ex_len[e]) - cur)
                _long_block(rng, ops, blen)
                rem -= blen; cur += blen; e += 1
                if rem > 0 and e < e1 and len(ops) <= LONG_MAX_OPS - 3:      # room for N, a block and a clip
                    n = int(ex_start[e]) - cur
                    ops.append((n << 4) | OP_N)
                    key = (cur - 1, cur + n - 1)                 # last exon base, last intron base (S:482-483)
                    junc[key] = (junc.get(key, (0, 0))[0] + 1, int(m["t_strand"][t]))
                    cur += n
            strand = int(m["t_strand"][t])
        if rng.random() < cfg.frac_softclip:
            ops.append((int(rng.integers(5, 60)) << 4) | OP_S)
        f = 16 if strand else 0                                  # single-end, sense reads map like fr; 30 % antisense (cDNA)
        if rng.random() < 0.3:
            f ^= 16
        if rng.random() < cfg.frac_odd_flag:
            f |= int(rng.choice([256, 2048]))
        pos.append(p); flag.append(f); reads.append(ops)
    return pos, flag, reads, junc


def generate_long_reads(cfg: SynthConfig) -> Workload:
    """A long-read sample on the gene models of _gene_models: reads of 1-10 kb along transcripts (5-40 junctions, ~100-255
    operators each), unspliced reads of 4096 bp and more, and the junction table of every N in the reads (score = reads,
    strand = transcript's).  cfg.read_len is the longest read."""
    rng = np.random.default_rng(cfg.seed)
    lens = np.array([l for _, l in cfg.contigs], float)
    n_per = np.floor(lens / lens.sum() * cfg.n_records).astype(np.int64)
    n_per[0] += cfg.n_records - int(n_per.sum())
    P, F, O, C, jc, jl, jr, js, jst, seg_off = [], [], [], [], [], [], [], [], [], [0]
    for ci, (_, clen) in enumerate(cfg.contigs):
        m = _gene_models(rng, cfg, int(clen))
        pos, flag, reads, junc = _long_reads_for_contig(rng, cfg, m, int(n_per[ci]))
        order = np.argsort(np.array(pos), kind="stable")
        P.append(np.array(pos, np.int32)[order]); F.append(np.array(flag, np.uint16)[order])
        O.extend(len(reads[i]) for i in order); C.extend(op for i in order for op in reads[i])
        seg_off.append(seg_off[-1] + len(pos))
        for (l, r), (cnt, st) in sorted(junc.items()):
            jc.append(ci); jl.append(l); jr.append(r); js.append(cnt); jst.append(ord("-") if st else ord("+"))
    cig_off = np.zeros(sum(len(p) for p in P) + 1, np.uint32)
    np.cumsum(O, out=cig_off[1:])
    rec = Records(np.concatenate(P), np.concatenate(F), cig_off, np.array(C, np.uint32), np.arange(len(cfg.contigs), dtype=np.int32),
                  np.array(seg_off, np.int64))
    return Workload(cfg, [c for c, _ in cfg.contigs], [l for _, l in cfg.contigs], rec, Junctions(jc, jl, jr, js, jst))


def reads_as_tuples(w: Workload):
    """(chrom_name, pos, flag, cigar_string) per record -- for text-based consumers on small workloads."""
    rec = w.records
    out = []
    letters = "MIDNSHP=X"
    for s in range(len(rec.seg_chrom)):
        cname = w.chroms[int(rec.seg_chrom[s])]
        for i in range(int(rec.seg_off[s]), int(rec.seg_off[s + 1])):
            ops = rec.cigar[int(rec.cig_off[i]):int(rec.cig_off[i + 1])]
            out.append((cname, int(rec.pos[i]), int(rec.flag[i]), "".join("%d%s" % (o >> 4, letters[o & 15]) for o in ops)))
    return out
