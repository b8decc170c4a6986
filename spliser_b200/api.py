"""Host-side API over the C ABI: numpy in, numpy out.

The names mirror the reference's stages: `Context.process_*` is the body of `process`
(SpliSER_v0_1_8.py:710-717: findAlphaCounts -> findCompetitorPos -> processSites) and
`Context.recount_*` is the `checkBam` call `combine` makes for a site missing from a sample
(S:899-904).  Everything that counts runs on the GPU behind libspliser_b200.so.
"""
from __future__ import annotations

import ctypes as C
import re
from dataclasses import dataclass

import numpy as np

from . import _lib as L

FLAG_STRANDED, FLAG_RF, FLAG_CRYPTIC, FLAG_COMBINE = 1, 2, 4, 8
FLAG_XS_STRAND = 16          # junction extraction: strands from the XS tag (include/spliser_b200.h states the rule)

_CIG = re.compile(r"(\d+)([MIDNSHP=X])")
_OPS = {c: i for i, c in enumerate("MIDNSHP=X")}


def mode_flags(is_stranded=False, stranded_type=None, beta2_cryptic=False, combine=False) -> int:
    """CLI switches (S:1314-1316) -> ABI flags.  Mirrors check_strand's UnboundLocalError (S:378-406)
    for a stranded run whose type is neither 'fr' nor 'rf'."""
    f = 0
    if is_stranded:
        if stranded_type not in ("fr", "rf"):
            raise UnboundLocalError("cannot access local variable 'readStrand': strandedType must be 'fr' or 'rf'")
        f |= FLAG_STRANDED | (FLAG_RF if stranded_type == "rf" else 0)
    if beta2_cryptic:
        f |= FLAG_CRYPTIC
    if combine:
        f |= FLAG_COMBINE
    return f


def encode_cigar(cigar: str):
    if cigar == "*" or not cigar:
        return []
    return [(int(n) << 4) | _OPS[op] for n, op in _CIG.findall(cigar)]


def _ptr(a, ty):
    return a.ctypes.data_as(ty)


@dataclass
class Junctions:
    """Junction table in BED-line order after the text filters (S:259-288).  start / end: the BED12 chromStart / chromEnd of
    every row (left - its longest left anchor, right + its longest right anchor) when the table was extracted from the
    alignments, else None."""
    chrom: np.ndarray
    left: np.ndarray
    right: np.ndarray
    score: np.ndarray
    strand: np.ndarray
    start: np.ndarray = None
    end: np.ndarray = None

    def __post_init__(self):
        self.chrom = np.ascontiguousarray(self.chrom, dtype=np.int32)
        self.left = np.ascontiguousarray(self.left, dtype=np.int32)
        self.right = np.ascontiguousarray(self.right, dtype=np.int32)
        self.score = np.ascontiguousarray(self.score, dtype=np.int64)
        self.strand = np.ascontiguousarray(self.strand, dtype=np.uint8)
        n = len(self.chrom)
        if not (len(self.left) == len(self.right) == len(self.score) == len(self.strand) == n):
            raise ValueError("junction arrays differ in length")
        if (self.start is None) != (self.end is None):
            raise ValueError("start and end come together")
        if self.start is not None:
            self.start = np.ascontiguousarray(self.start, dtype=np.int32)
            self.end = np.ascontiguousarray(self.end, dtype=np.int32)
            if not (len(self.start) == len(self.end) == n):
                raise ValueError("junction arrays differ in length")

    def __len__(self):
        return len(self.chrom)

    def args(self):
        return (C.c_int64(len(self)), _ptr(self.chrom, L.c_i32p), _ptr(self.left, L.c_i32p), _ptr(self.right, L.c_i32p),
                _ptr(self.score, L.c_i64p), _ptr(self.strand, L.c_u8p))


class Records:
    """Alignment records as flat arrays grouped in chromosome segments (spl_records_view).  xs: optional strand of every record
    from its XS tag (uint8 '+', '-' or '?'), what extraction with FLAG_XS_STRAND reads."""

    def __init__(self, pos, flag, cig_off, cigar, seg_chrom, seg_off, _owner=None, xs=None):
        self.pos = np.ascontiguousarray(pos, dtype=np.int32)
        self.flag = np.ascontiguousarray(flag, dtype=np.uint16)
        self.cig_off = np.ascontiguousarray(cig_off, dtype=np.uint32)
        self.cigar = np.ascontiguousarray(cigar, dtype=np.uint32)
        self.seg_chrom = np.ascontiguousarray(seg_chrom, dtype=np.int32)
        self.seg_off = np.ascontiguousarray(seg_off, dtype=np.int64)
        self._owner = _owner
        self.xs = None if xs is None else np.ascontiguousarray(xs, dtype=np.uint8)
        if len(self.cig_off) != len(self.pos) + 1 or len(self.flag) != len(self.pos):
            raise ValueError("record arrays differ in length")
        if self.xs is not None and len(self.xs) != len(self.pos):
            raise ValueError("xs must have one entry per record")
        if len(self.seg_off) != len(self.seg_chrom) + 1:
            raise ValueError("seg_off must have n_seg+1 entries")

    def __len__(self):
        return len(self.pos)

    def view(self) -> L.RecordsView:
        v = L.RecordsView()
        v.n_rec = len(self.pos)
        v.n_cigar = len(self.cigar)
        v.pos = _ptr(self.pos, L.c_i32p)
        v.flag = _ptr(self.flag, L.c_u16p)
        v.cig_off = _ptr(self.cig_off, L.c_u32p)
        v.cigar = _ptr(self.cigar, L.c_u32p)
        v.n_seg = len(self.seg_chrom)
        v.seg_chrom = _ptr(self.seg_chrom, L.c_i32p)
        v.seg_off = _ptr(self.seg_off, L.c_i64p)
        return v

    @classmethod
    def from_reads(cls, chrom_names, reads):
        """reads: iterable of (chrom_name, pos1, flag, cigar_string[, xs]) in file order, xs = '+', '-' or '?' (the strand of
        the read's XS tag; given for every read or for none).  Reads on unknown chromosomes become segments with chromosome -1
        (skipped by the library)."""
        index = {c: i for i, c in enumerate(chrom_names)}
        pos, flag, off, cig, seg_chrom, seg_off, xs = [], [], [0], [], [], [], []
        cur = None
        for r in reads:
            chrom, p, f, cg = r[:4]
            if len(r) > 4:
                xs.append(ord(r[4]))
            ci = index.get(chrom, -1)
            if ci != cur:
                seg_chrom.append(ci)
                seg_off.append(len(pos))
                cur = ci
            pos.append(p)
            flag.append(f)
            cig.extend(encode_cigar(cg))
            off.append(len(cig))
        seg_off.append(len(pos))
        if not seg_chrom:
            seg_off = [0]
        if xs and len(xs) != len(pos):
            raise ValueError("an xs strand for every read or for none")
        return cls(pos, flag, off, cig, seg_chrom, seg_off, xs=xs if xs else None)

    @classmethod
    def from_bam(cls, path, chrom_names, threads=0, xs=False):
        """xs: also read every record's strand from its XS tag (Records.xs)."""
        lib = L.load()
        names = (C.c_char_p * max(1, len(chrom_names)))(*[c.encode() for c in chrom_names])
        h = C.c_void_p()
        err = C.create_string_buffer(512)
        rc = (lib.spl_read_bam_xs if xs else lib.spl_read_bam)(str(path).encode(), len(chrom_names), names, threads, C.byref(h), err, 512)
        if rc != 0:
            raise IOError("spl_read_bam(%s): %s" % (path, err.value.decode()))
        try:
            v = lib.spl_records_get(h).contents
            n, nc, ns = v.n_rec, v.n_cigar, v.n_seg

            def arr(p, cnt, dt):
                return np.ctypeslib.as_array(p, shape=(cnt,)).astype(dt, copy=True) if cnt else np.zeros(0, dt)
            out = cls(arr(v.pos, n, np.int32), arr(v.flag, n, np.uint16),
                      np.ctypeslib.as_array(v.cig_off, shape=(n + 1,)).astype(np.uint32, copy=True),
                      arr(v.cigar, nc, np.uint32), arr(v.seg_chrom, ns, np.int32),
                      np.ctypeslib.as_array(v.seg_off, shape=(ns + 1,)).astype(np.int64, copy=True),
                      xs=arr(lib.spl_records_xs(h), n, np.uint8) if xs else None)
        finally:
            lib.spl_records_free(h)
        return out

    def write_bam(self, path, ref_names, ref_len=None, threads=0, with_seq=False, aux=None):
        """with_seq: read names, SEQ and QUAL of the CIGAR's query length are written too (a sequencer-shaped file).
        aux: raw aux bytes per record, a list of bytes (see encode_aux) or (offsets[n_rec + 1], uint8 blob)."""
        lib = L.load()
        names = (C.c_char_p * max(1, len(ref_names)))(*[c.encode() for c in ref_names])
        rl = None
        if ref_len is not None:
            rl = np.ascontiguousarray(ref_len, dtype=np.int32)
        v = self.view()
        rlp = _ptr(rl, L.c_i32p) if rl is not None else None
        if aux is None:
            rc = (lib.spl_write_bam_seq if with_seq else lib.spl_write_bam)(str(path).encode(), len(ref_names), names, rlp, C.byref(v), threads)
        else:
            if isinstance(aux, tuple):
                off, blob = aux
            else:
                off = np.zeros(len(aux) + 1, np.int64)
                off[1:] = np.cumsum([len(a) for a in aux])
                blob = np.frombuffer(b"".join(aux), np.uint8)
            off = np.ascontiguousarray(off, dtype=np.int64)
            blob = np.ascontiguousarray(blob, dtype=np.uint8)
            if len(off) != len(self) + 1 or (len(off) and (off[0] != 0 or off[-1] != len(blob) or np.any(np.diff(off) < 0))):
                raise ValueError("aux offsets must run from 0 to len(blob), one record each")
            rc = lib.spl_write_bam_aux(str(path).encode(), len(ref_names), names, rlp, C.byref(v), _ptr(off, L.c_i64p),
                                       _ptr(blob, L.c_u8p) if len(blob) else C.cast(C.c_char_p(b""), L.c_u8p), int(with_seq), threads)
        if rc != 0:
            raise IOError("spl_write_bam(%s) failed with %d" % (path, rc))


PACKED_INDEX_STRIDE = 1024


class PackedRecords:
    """The packed host layout of spl_process_packed (spl_packed_view): POS, three flag bits, operator count and a sparse
    CIGAR index -- 17 bytes per record on the wire instead of 20.  `alloc` = a function (n, dtype) -> array, e.g.
    api.pinned_empty for page-locked columns."""

    def __init__(self, pos, flag8, n_op, cigar, cig_index, seg_chrom, seg_off):
        self.pos = np.ascontiguousarray(pos, dtype=np.int32)
        self.flag8 = np.ascontiguousarray(flag8, dtype=np.uint8)
        self.n_op = np.ascontiguousarray(n_op, dtype=np.uint16)
        self.cigar = np.ascontiguousarray(cigar, dtype=np.uint32)
        self.cig_index = np.ascontiguousarray(cig_index, dtype=np.uint32)
        self.seg_chrom = np.ascontiguousarray(seg_chrom, dtype=np.int32)
        self.seg_off = np.ascontiguousarray(seg_off, dtype=np.int64)

    def __len__(self):
        return len(self.pos)

    @classmethod
    def from_records(cls, r: "Records", alloc=None):
        nop = np.diff(r.cig_off.astype(np.int64))
        if len(nop) and int(nop.max()) > 65535:
            raise ValueError("a record has more than 65535 CIGAR operators: use the plain Records view")
        f = r.flag
        flag8 = ((f & 1) | (((f >> 4) & 1) << 1) | (((f >> 6) & 1) << 2)).astype(np.uint8)
        index = np.concatenate([r.cig_off[::PACKED_INDEX_STRIDE], r.cig_off[-1:]]).astype(np.uint32)
        cols = dict(pos=r.pos, flag8=flag8, n_op=nop.astype(np.uint16), cigar=r.cigar, cig_index=index)
        if alloc is not None:
            for k, a in list(cols.items()):
                b = alloc(len(a), a.dtype)
                b[:] = a
                cols[k] = b
        return cls(cols["pos"], cols["flag8"], cols["n_op"], cols["cigar"], cols["cig_index"], r.seg_chrom, r.seg_off)

    def view(self) -> L.PackedView:
        v = L.PackedView()
        v.n_rec = len(self.pos)
        v.n_cigar = len(self.cigar)
        v.pos = _ptr(self.pos, L.c_i32p)
        v.flag8 = _ptr(self.flag8, L.c_u8p)
        v.n_op = _ptr(self.n_op, L.c_u16p)
        v.cigar = _ptr(self.cigar, L.c_u32p)
        v.cig_index = _ptr(self.cig_index, L.c_u32p)
        v.n_seg = len(self.seg_chrom)
        v.seg_chrom = _ptr(self.seg_chrom, L.c_i32p)
        v.seg_off = _ptr(self.seg_off, L.c_i64p)
        return v


class CompactRecords:
    """The compact host layout of spl_process_compact (spl_compact_view), about 9 bytes per record on the wire: POS as a 16-bit
    offset from the lowest POS of the record's stride of PACKED_INDEX_STRIDE records (strides spanning more than 65535 bp keep
    their 32-bit positions in pos_wide), operator count in a byte, operators in 16 bits unless the record has one of length
    >= 4096 (then all of its operators are BAM-encoded in the 32-bit stream).  `alloc` as in PackedRecords."""
    COLS = (("pos16", np.uint16), ("flag8", np.uint8), ("n_op8", np.uint8), ("cigar16", np.uint16), ("cigar32", np.uint32),
            ("pos_base", np.int32), ("pos_wide", np.int32), ("idx16", np.uint32), ("idx32", np.uint32))

    def __init__(self, cols, seg_chrom, seg_off):
        for k, dt in self.COLS:
            setattr(self, k, np.ascontiguousarray(cols[k], dtype=dt))
        self.seg_chrom = np.ascontiguousarray(seg_chrom, dtype=np.int32)
        self.seg_off = np.ascontiguousarray(seg_off, dtype=np.int64)

    def __len__(self):
        return len(self.pos16)

    @property
    def wire_bytes(self):
        return sum(getattr(self, k).nbytes for k, _ in self.COLS)

    @classmethod
    def from_records(cls, r: "Records", alloc=None):
        K = PACKED_INDEX_STRIDE
        R = len(r)
        off = r.cig_off.astype(np.int64)
        nop = np.diff(off)
        if R and int(nop.max()) > 255:
            raise ValueError("a record has more than 255 CIGAR operators: use the packed or the plain Records view")
        # records with an operator of 4096 bases or more keep 32-bit operators
        long_op = (r.cigar >> 4) >= 4096
        csum = np.concatenate([[0], np.cumsum(long_op, dtype=np.int64)])
        rec_long = (csum[off[1:]] - csum[off[:-1]]) > 0
        op_long = np.repeat(rec_long, nop)
        c32 = r.cigar[op_long]
        c16 = r.cigar[~op_long].astype(np.uint16)
        f = r.flag
        flag8 = ((f & 1) | (((f >> 4) & 1) << 1) | (((f >> 6) & 1) << 2) | (rec_long.astype(np.uint16) << 3)).astype(np.uint8)
        nS = np.concatenate([[0], np.cumsum(np.where(rec_long, 0, nop), dtype=np.int64)])
        nL = np.concatenate([[0], np.cumsum(np.where(rec_long, nop, 0), dtype=np.int64)])
        NS = (R + K - 1) // K
        starts = np.minimum(np.arange(NS + 1, dtype=np.int64) * K, R)
        idx16, idx32 = nS[starts].astype(np.uint32), nL[starts].astype(np.uint32)
        # positions: per stride the lowest POS and 16-bit offsets, or the stride's 32-bit positions when it spans too much
        pos = r.pos.astype(np.int64)
        pad = NS * K - R
        if NS:
            lo = np.minimum.reduceat(pos, starts[:-1]) if R else np.zeros(0, np.int64)
            hi = np.maximum.reduceat(pos, starts[:-1]) if R else np.zeros(0, np.int64)
        else:
            lo = hi = np.zeros(0, np.int64)
        wide = ((hi - lo) > 65535) | (lo < 0)
        w_id = np.cumsum(wide) - 1
        pos_base = np.where(wide, -(w_id + 1), lo).astype(np.int32)
        stride_of = np.arange(R, dtype=np.int64) // K
        pos16 = np.where(wide[stride_of], 0, pos - lo[stride_of]).astype(np.uint16) if R else np.zeros(0, np.uint16)
        pos_wide = np.zeros(int(wide.sum()) * K, np.int32)
        if wide.any():
            padded = np.concatenate([r.pos, np.zeros(pad, np.int32)]).reshape(NS, K)
            pos_wide = np.ascontiguousarray(padded[wide]).reshape(-1)
        cols = dict(pos16=pos16, flag8=flag8, n_op8=nop.astype(np.uint8), cigar16=c16, cigar32=c32, pos_base=pos_base, pos_wide=pos_wide,
                    idx16=idx16, idx32=idx32)
        if alloc is not None:
            for k, a in list(cols.items()):
                b = alloc(len(a), a.dtype)
                b[:] = a
                cols[k] = b
        return cls(cols, r.seg_chrom, r.seg_off)

    def to_records(self) -> "Records":
        """The plain view again (numpy restatement of what k_unpack_compact does on the device; used by the CPU tests)."""
        K = PACKED_INDEX_STRIDE
        R = len(self)
        nop = self.n_op8.astype(np.int64)
        rec_long = (self.flag8 & 8) != 0
        off = np.concatenate([[0], np.cumsum(nop)])
        op_long = np.repeat(rec_long, nop)
        cigar = np.zeros(int(off[-1]), np.uint32)
        cigar[op_long] = self.cigar32
        cigar[~op_long] = self.cigar16.astype(np.uint32)
        stride_of = np.arange(R, dtype=np.int64) // K
        base = self.pos_base.astype(np.int64)[stride_of] if R else np.zeros(0, np.int64)
        pos = base + self.pos16.astype(np.int64)
        w = base < 0
        if w.any():
            pos[w] = self.pos_wide[(-(base[w] + 1)) * K + (np.arange(R)[w] % K)]
        f = self.flag8.astype(np.uint16)
        flag = ((f & 1) | ((f & 2) << 3) | ((f & 4) << 4)).astype(np.uint16)
        return Records(pos.astype(np.int32), flag, off.astype(np.uint32), cigar, self.seg_chrom, self.seg_off)

    def view(self) -> L.CompactView:
        v = L.CompactView()
        v.n_rec = len(self.pos16)
        v.n16, v.n32 = len(self.cigar16), len(self.cigar32)
        v.n_cigar = v.n16 + v.n32
        v.n_wide = len(self.pos_wide) // PACKED_INDEX_STRIDE
        v.pos16 = _ptr(self.pos16, L.c_u16p); v.flag8 = _ptr(self.flag8, L.c_u8p); v.n_op8 = _ptr(self.n_op8, L.c_u8p)
        v.cigar16 = _ptr(self.cigar16, L.c_u16p); v.cigar32 = _ptr(self.cigar32, L.c_u32p)
        v.pos_base = _ptr(self.pos_base, L.c_i32p); v.pos_wide = _ptr(self.pos_wide, L.c_i32p)
        v.idx16 = _ptr(self.idx16, L.c_u32p); v.idx32 = _ptr(self.idx32, L.c_u32p)
        v.n_seg = len(self.seg_chrom)
        v.seg_chrom = _ptr(self.seg_chrom, L.c_i32p)
        v.seg_off = _ptr(self.seg_off, L.c_i64p)
        return v


@dataclass
class GapTable:
    """The (site, sample) gaps of one sample for `combine`'s re-count (S:899-904) in the argument layout of
    spl_recount: position, chromosome index, strand byte (0 = ''), partner / competitor positions as CSR.
    Iterating yields the tuples (chrom_idx, pos, strand_str, partners, competitors)."""
    chrom: np.ndarray
    pos: np.ndarray
    strand: np.ndarray
    p_off: np.ndarray
    p_pos: np.ndarray
    c_off: np.ndarray
    c_pos: np.ndarray

    def __post_init__(self):
        self.chrom = np.ascontiguousarray(self.chrom, dtype=np.int32)
        self.pos = np.ascontiguousarray(self.pos, dtype=np.int32)
        self.strand = np.ascontiguousarray(self.strand, dtype=np.uint8)
        self.p_off = np.ascontiguousarray(self.p_off, dtype=np.int64)
        self.p_pos = np.ascontiguousarray(self.p_pos, dtype=np.int32)
        self.c_off = np.ascontiguousarray(self.c_off, dtype=np.int64)
        self.c_pos = np.ascontiguousarray(self.c_pos, dtype=np.int32)
        n = len(self.pos)
        if not (len(self.chrom) == len(self.strand) == n and len(self.p_off) == len(self.c_off) == n + 1):
            raise ValueError("gap arrays differ in length")

    def __len__(self):
        return len(self.pos)

    def __iter__(self):
        for i in range(len(self.pos)):
            b = int(self.strand[i])
            yield (int(self.chrom[i]), int(self.pos[i]), chr(b) if b else "",
                   [int(x) for x in self.p_pos[self.p_off[i]:self.p_off[i + 1]]],
                   [int(x) for x in self.c_pos[self.c_off[i]:self.c_off[i + 1]]])

    @classmethod
    def from_tuples(cls, gaps):
        n = len(gaps)
        p_off = np.zeros(n + 1, dtype=np.int64)
        c_off = np.zeros(n + 1, dtype=np.int64)
        pp, cp = [], []
        for i, g in enumerate(gaps):
            pp.extend(g[3])
            cp.extend(g[4])
            p_off[i + 1] = len(pp)
            c_off[i + 1] = len(cp)
        return cls(np.array([g[0] for g in gaps], dtype=np.int32), np.array([g[1] for g in gaps], dtype=np.int32),
                   np.array([(ord(g[2][0]) if g[2] else 0) for g in gaps], dtype=np.uint8),
                   p_off, np.array(pp, dtype=np.int32), c_off, np.array(cp, dtype=np.int32))


@dataclass
class SiteTable:
    """Per-site results in the reference's output order (outputBedFile, S:645-663)."""
    chrom: np.ndarray
    pos: np.ndarray
    strand: np.ndarray       # raw byte
    alpha: np.ndarray
    beta1: np.ndarray
    beta2simple: np.ndarray
    beta2cryptic: np.ndarray
    beta2weighted: np.ndarray
    sse: np.ndarray
    first_line: np.ndarray
    partner_off: np.ndarray
    partner_pos: np.ndarray
    partner_cnt: np.ndarray
    comp_off: np.ndarray
    comp_pos: np.ndarray

    def __len__(self):
        return len(self.pos)

    def partners(self, i):
        a, b = self.partner_off[i], self.partner_off[i + 1]
        return {int(p): int(c) for p, c in zip(self.partner_pos[a:b], self.partner_cnt[a:b])}

    def competitors(self, i):
        a, b = self.comp_off[i], self.comp_off[i + 1]
        return [int(c) for c in self.comp_pos[a:b]]

    def strand_str(self, i):
        b = int(self.strand[i])
        return chr(b) if b else ""


class _ResultOwner:
    """Owns one spl_result handle."""

    def __init__(self, lib, h):
        self._lib, self._h = lib, h

    def __del__(self):
        h, self._h = self._h, None
        if h:
            try:
                self._lib.spl_result_free(h)
            except Exception:
                pass


class SpliserError(RuntimeError):
    pass


class Context:
    """One spl_ctx = one GPU (one process per GPU)."""

    def __init__(self, device=0, tile=None, threads=0):
        self._lib = L.load()
        self._h = C.c_void_p()
        dev = (C.c_int32 * 1)(device)
        rc = self._lib.spl_create(C.byref(self._h), dev, 1)
        if rc != 0:
            msg = self._lib.spl_last_error(self._h).decode() if self._h else "spl_create failed"
            if self._h:
                self._lib.spl_destroy(self._h)
                self._h = C.c_void_p()
            raise SpliserError("spl_create: %s (code %d)" % (msg, rc))
        if tile is not None:
            self._check(self._lib.spl_set_tile(self._h, int(tile[0]), int(tile[1])), "spl_set_tile")
        if threads:
            self._lib.spl_set_threads(self._h, int(threads))

    def close(self):
        if getattr(self, "_h", None):
            self._lib.spl_destroy(self._h)
            self._h = C.c_void_p()

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _check(self, rc, what):
        if rc != 0:
            raise SpliserError("%s: %s (code %d)" % (what, self._lib.spl_last_error(self._h).decode(), rc))

    def set_tile_sites(self, site_lo, site_hi):
        """Owned range [site_lo, site_hi) of global site indices for the following calls (tiles balanced by read count,
        spliser_b200.dist.balanced_tiles); (-1, -1) = no tiling."""
        self._check(self._lib.spl_set_tile_sites(self._h, int(site_lo), int(site_hi)), "spl_set_tile_sites")

    def set_variant(self, variant):
        """'fused' (product path: difference arrays straight from the records) or 'stab' (block-vs-site stabbing over a
        bin-partitioned block stream; the cross-check)."""
        v = {"fused": 0, "stab": 1}[variant] if isinstance(variant, str) else int(variant)
        self._check(self._lib.spl_set_variant(self._h, v), "spl_set_variant")

    def stats(self):
        buf = (C.c_double * L.SPL_NSTATS)()
        self._lib.spl_last_stats(self._h, buf)
        return dict(zip(L.STAT_NAMES, list(buf)))

    # ---- process -----------------------------------------------------------------------------
    def _take(self, h) -> SiteTable:
        """SiteTable whose arrays are zero-copy views of the library-owned result; the result is freed
        (spl_result_free) when the last array that refers to it is garbage-collected."""
        lib = self._lib
        owner = _ResultOwner(lib, h)
        n = lib.spl_result_n_sites(h)

        def arr(fn, cnt, ct, dt):
            if cnt == 0:
                return np.zeros(0, dt)
            buf = (ct * cnt).from_address(C.addressof(fn(h).contents))
            buf._owner = owner                     # numpy keeps `buf` as the base object, `buf` keeps the result alive
            return np.frombuffer(buf, dtype=dt)
        poff = arr(lib.spl_result_partner_off, n + 1, C.c_int64, np.int64)
        coff = arr(lib.spl_result_comp_off, n + 1, C.c_int64, np.int64)
        ne, nc = int(poff[-1]), int(coff[-1])
        return SiteTable(
            chrom=arr(lib.spl_result_chrom, n, C.c_int32, np.int32), pos=arr(lib.spl_result_pos, n, C.c_int32, np.int32),
            strand=arr(lib.spl_result_strand, n, C.c_uint8, np.uint8), alpha=arr(lib.spl_result_alpha, n, C.c_int64, np.int64),
            beta1=arr(lib.spl_result_beta1, n, C.c_int64, np.int64), beta2simple=arr(lib.spl_result_beta2simple, n, C.c_int64, np.int64),
            beta2cryptic=arr(lib.spl_result_beta2cryptic, n, C.c_int64, np.int64),
            beta2weighted=arr(lib.spl_result_beta2weighted, n, C.c_double, np.float64), sse=arr(lib.spl_result_sse, n, C.c_double, np.float64),
            first_line=arr(lib.spl_result_first_line, n, C.c_int64, np.int64),
            partner_off=poff, partner_pos=arr(lib.spl_result_partner_pos, ne, C.c_int32, np.int32),
            partner_cnt=arr(lib.spl_result_partner_cnt, ne, C.c_int64, np.int64),
            comp_off=coff, comp_pos=arr(lib.spl_result_comp_pos, nc, C.c_int32, np.int32))

    def process_records(self, records: Records, n_chrom: int, junctions: Junctions, flags: int) -> SiteTable:
        v = records.view()
        h = C.c_void_p()
        rc = self._lib.spl_process_records(self._h, C.byref(v), n_chrom, *junctions.args(), flags, C.byref(h))
        self._check(rc, "spl_process_records")
        return self._take(h)

    def process_packed(self, records: "PackedRecords", n_chrom: int, junctions: Junctions, flags: int) -> SiteTable:
        v = records.view()
        h = C.c_void_p()
        rc = self._lib.spl_process_packed(self._h, C.byref(v), n_chrom, *junctions.args(), flags, C.byref(h))
        self._check(rc, "spl_process_packed")
        return self._take(h)

    def process_compact(self, records: "CompactRecords", n_chrom: int, junctions: Junctions, flags: int) -> SiteTable:
        v = records.view()
        h = C.c_void_p()
        rc = self._lib.spl_process_compact(self._h, C.byref(v), n_chrom, *junctions.args(), flags, C.byref(h))
        self._check(rc, "spl_process_compact")
        return self._take(h)

    def process_bam(self, bam_path, chrom_names, junctions: Junctions, flags: int) -> SiteTable:
        names = (C.c_char_p * max(1, len(chrom_names)))(*[c.encode() for c in chrom_names])
        h = C.c_void_p()
        rc = self._lib.spl_process(self._h, str(bam_path).encode(), len(chrom_names), names, *junctions.args(), flags, C.byref(h))
        self._check(rc, "spl_process")
        return self._take(h)

    # ---- junction extraction (the regtools pre-step, README.md:41) ---------------------------------
    def _take_junctions(self, h) -> Junctions:
        lib = self._lib
        try:
            n = lib.spl_junctions_n(h)

            def arr(fn, dt):
                return np.ctypeslib.as_array(fn(h), shape=(n,)).astype(dt, copy=True) if n else np.zeros(0, dt)
            return Junctions(arr(lib.spl_junctions_chrom, np.int32), arr(lib.spl_junctions_left, np.int32), arr(lib.spl_junctions_right, np.int32),
                             arr(lib.spl_junctions_score, np.int64), arr(lib.spl_junctions_strand, np.uint8),
                             arr(lib.spl_junctions_start, np.int32), arr(lib.spl_junctions_end, np.int32))
        finally:
            lib.spl_junctions_free(h)

    def extract_junctions_records(self, records: Records, n_chrom: int, flags: int = 0, min_anchor=8, min_intron=70, max_intron=500000) -> Junctions:
        """Junction table (left, right, score, strand) from the alignments: what `regtools junctions extract -a 8 -m 70 -M 500000`
        feeds the reference with.  flags: FLAG_XS_STRAND takes the strands from records.xs, FLAG_STRANDED (| FLAG_RF) gives
        '+' / '-' strands from the FLAG, else '?'."""
        v = records.view()
        h = C.c_void_p()
        if flags & FLAG_XS_STRAND:
            if records.xs is None:
                raise ValueError("FLAG_XS_STRAND needs records.xs (Records.from_bam(..., xs=True) or from_reads with an xs column)")
            rc = self._lib.spl_extract_junctions_records_xs(self._h, C.byref(v), _ptr(records.xs, L.c_u8p), n_chrom, min_anchor, min_intron,
                                                            max_intron, flags, C.byref(h))
        else:
            rc = self._lib.spl_extract_junctions_records(self._h, C.byref(v), n_chrom, min_anchor, min_intron, max_intron, flags, C.byref(h))
        self._check(rc, "spl_extract_junctions_records")
        return self._take_junctions(h)

    def extract_junctions_bam(self, bam_path, chrom_names, flags: int = 0, min_anchor=8, min_intron=70, max_intron=500000) -> Junctions:
        names = (C.c_char_p * max(1, len(chrom_names)))(*[c.encode() for c in chrom_names])
        h = C.c_void_p()
        rc = self._lib.spl_extract_junctions(self._h, str(bam_path).encode(), len(chrom_names), names, min_anchor, min_intron, max_intron, flags, C.byref(h))
        self._check(rc, "spl_extract_junctions")
        return self._take_junctions(h)

    def process_bam_extract(self, bam_path, chrom_names, flags: int = 0, min_anchor=8, min_intron=70, max_intron=500000,
                            qchrom="All", gene_bounds=None, window_max_intron=0):
        """`process` without a BED12 file: the BAM is ingested once, its junction table extracted (as extract_junctions_bam),
        filtered like a BED12 of it (-c qchrom, -g window gene_bounds = (leftPos, rightPos) widened by window_max_intron,
        S:269, S:279-288) and counted against the same device-resident records.  Returns (Junctions after the filters, in the
        order they were counted -- first_line indexes them; SiteTable)."""
        names = (C.c_char_p * max(1, len(chrom_names)))(*[c.encode() for c in chrom_names])
        o = L.ExtractOpts(int(min_anchor), int(min_intron), int(max_intron), None if qchrom == "All" else str(qchrom).encode(),
                          int(gene_bounds is not None), *(int(x) for x in (gene_bounds or (0, 0))), int(window_max_intron))
        hj, hr = C.c_void_p(), C.c_void_p()
        rc = self._lib.spl_process_bam_extract(self._h, str(bam_path).encode(), len(chrom_names), names, C.byref(o), flags,
                                               C.byref(hj), C.byref(hr))
        self._check(rc, "spl_process_bam_extract")
        return self._take_junctions(hj), self._take(hr)

    # ---- combine re-count ----------------------------------------------------------------------
    @staticmethod
    def _gap_args(gaps):
        """gaps: GapTable, or a list of (chrom_idx, pos, strand_str, partner_positions, competitor_positions)."""
        g = gaps if isinstance(gaps, GapTable) else GapTable.from_tuples(gaps)
        args = (C.c_int64(len(g)), _ptr(g.chrom, L.c_i32p), _ptr(g.pos, L.c_i32p), _ptr(g.strand, L.c_u8p),
                _ptr(g.p_off, L.c_i64p), _ptr(g.p_pos, L.c_i32p), _ptr(g.c_off, L.c_i64p), _ptr(g.c_pos, L.c_i32p))
        return g, args

    def recount_records(self, records: Records, n_chrom: int, gaps, flags: int):
        keep, args = self._gap_args(gaps)
        b1 = np.zeros(len(gaps), dtype=np.int64)
        b2 = np.zeros(len(gaps), dtype=np.int64)
        v = records.view()
        rc = self._lib.spl_recount_records(self._h, C.byref(v), n_chrom, *args, flags, _ptr(b1, L.c_i64p), _ptr(b2, L.c_i64p))
        self._check(rc, "spl_recount_records")
        return b1, b2

    def recount_bam(self, bam_path, chrom_names, gaps, flags: int):
        keep, args = self._gap_args(gaps)
        b1 = np.zeros(len(gaps), dtype=np.int64)
        b2 = np.zeros(len(gaps), dtype=np.int64)
        names = (C.c_char_p * max(1, len(chrom_names)))(*[c.encode() for c in chrom_names])
        rc = self._lib.spl_recount(self._h, str(bam_path).encode(), len(chrom_names), names, *args, flags,
                                   _ptr(b1, L.c_i64p), _ptr(b2, L.c_i64p))
        self._check(rc, "spl_recount")
        return b1, b2

    # ---- resident (benchmark) path -------------------------------------------------------------
    def resident_load(self, records: Records, n_chrom: int, junctions: Junctions, flags: int):
        v = records.view()
        self._check(self._lib.spl_resident_load(self._h, C.byref(v), n_chrom, *junctions.args(), flags), "spl_resident_load")

    def resident_count(self, iters=1):
        buf = (C.c_double * L.SPL_NSTATS)()
        self._check(self._lib.spl_resident_count(self._h, iters, buf), "spl_resident_count")
        return dict(zip(L.STAT_NAMES, list(buf)))

    def resident_fetch(self) -> SiteTable:
        h = C.c_void_p()
        self._check(self._lib.spl_resident_fetch(self._h, C.byref(h)), "spl_resident_fetch")
        return self._take(h)


def bam_reference_names(path):
    """Reference names of a BAM header in header order (host only)."""
    lib = L.load()
    n, need = C.c_int64(), C.c_int64()
    err = C.create_string_buffer(512)
    cap = 1 << 16
    while True:
        buf = C.create_string_buffer(cap)
        rc = lib.spl_bam_reference_names(str(path).encode(), buf, cap, C.byref(n), C.byref(need), err, 512)
        if rc != 0:
            raise IOError("spl_bam_reference_names(%s): %s" % (path, err.value.decode()))
        if need.value <= cap:
            break
        cap = need.value
    return [x.decode() for x in buf.raw[:need.value].split(b"\0")[:n.value]]


def build_site_table(n_chrom: int, junctions: Junctions, flags: int) -> SiteTable:
    """Host-only site table (findAlphaCounts + findCompetitorPos, S:289-372): alpha, Partners, Competitors.
    beta / SSE columns are zero -- they need the alignments and the GPU."""
    lib = L.load()
    h = C.c_void_p()
    err = C.create_string_buffer(512)
    rc = lib.spl_build_site_table(n_chrom, *junctions.args(), flags, C.byref(h), err, 512)
    if rc != 0:
        raise SpliserError("spl_build_site_table: %s (code %d)" % (err.value.decode(), rc))
    return Context._take(_LibOnly(lib), h)


class _LibOnly:
    def __init__(self, lib):
        self._lib = lib


def pinned_empty(n, dtype):
    """numpy array over page-locked memory from spl_host_alloc (full-speed host->device copies)."""
    lib = L.load()
    dt = np.dtype(dtype)
    nbytes = max(1, int(n) * dt.itemsize)
    p = lib.spl_host_alloc(nbytes)
    if not p:
        raise SpliserError("spl_host_alloc(%d) failed (no CUDA device?)" % nbytes)
    buf = (C.c_uint8 * nbytes).from_address(p)
    a = np.frombuffer(buf, dtype=dt, count=int(n))
    _PINNED[id(buf)] = (buf, p)
    return a


_PINNED = {}
