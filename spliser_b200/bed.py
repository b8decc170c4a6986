"""BED12 junction file -> junction table (the text half of findAlphaCounts, SpliSER_v0_1_8.py:255-288), and the BED12 of a
junction table extracted from the alignments (what `regtools junctions extract` writes).

Text handling, not counting, so it sits on the host side of the counting ABI; the per-line work is native
(spl_bed_parse in csrc/host_text.cpp): the 12-column test (S:259), the chromosome index in first-appearance order
(S:265-268, appended to whatever the annotation already registered, S:90-92), the -c filter (S:269) and the -g window
filter (S:279-288).
"""
from __future__ import annotations

import ctypes as C

import numpy as np

from . import _lib as L
from .api import Junctions


class StrandColumn:
    """Column 6 of every kept BED row as (distinct texts, id per row); reads like the list of texts.  The Gene column
    and the TSV print the full text verbatim, while the counting ABI only carries its first byte."""

    def __init__(self, texts, ids):
        self.texts = list(texts)
        self.ids = np.ascontiguousarray(ids, dtype=np.int32)

    def __len__(self):
        return len(self.ids)

    def __getitem__(self, i):
        if isinstance(i, slice):
            return [self.texts[k] for k in self.ids[i]]
        return self.texts[int(self.ids[i])]

    def __iter__(self):
        t = self.texts
        return (t[k] for k in self.ids.tolist())

    def __eq__(self, other):
        return list(self) == list(other)


def _bytes_of(lines) -> bytes:
    """File image as the reference's text-mode iteration sees it (universal newlines)."""
    if isinstance(lines, str):
        return lines.encode()
    if not isinstance(lines, bytes):
        raw = getattr(lines, "buffer", None)         # open text file: take the bytes underneath, no decode + encode
        if raw is not None and hasattr(raw, "read") and lines.tell() == 0:
            lines = raw.read()
        elif hasattr(lines, "read"):
            data = lines.read()
            return data if isinstance(data, bytes) else data.encode()
        else:
            return "".join((x if x.endswith("\n") else x + "\n") for x in map(str, lines)).encode()
    if b"\r" in lines:
        lines = lines.replace(b"\r\n", b"\n").replace(b"\r", b"\n")
    return lines


def parse_bed12(lines, chrom_index=None, qchrom="All", qgene_bounds=None, max_intron=0):
    """Returns (chrom_index, Junctions, strand column).

    lines: an open text file, the file's text, or an iterable of lines.
    chrom_index: list of names already registered by the annotation (a copy with the BED's names appended is returned).
    qgene_bounds: (leftPos, rightPos) of the query gene when -g is used, else None."""
    from .hosttext import StrTable
    lib = L.load()
    raw = _bytes_of(lines)
    tab = StrTable(list(chrom_index)) if chrom_index else None
    gl, gr = (int(qgene_bounds[0]), int(qgene_bounds[1])) if qgene_bounds is not None else (0, 0)
    h = C.c_void_p()
    err = C.create_string_buffer(256)
    rc = lib.spl_bed_parse(raw, len(raw), tab.ref() if tab is not None else None,
                           None if qchrom == "All" else str(qchrom).encode(), int(qgene_bounds is not None), gl, gr,
                           int(max_intron), C.byref(h), err, 256)
    if rc != 0:
        raise (OverflowError if rc == -5 else ValueError)(err.value.decode())
    try:
        n = lib.spl_bed_n_junctions(h)

        def arr(fn, dt):
            return np.ctypeslib.as_array(fn(h), shape=(n,)).astype(dt, copy=True) if n else np.zeros(0, dt)

        def names(count, get):
            ln = C.c_int64()
            return [C.string_at(get(h, i, C.byref(ln)), ln.value).decode() for i in range(count)]
        junc = Junctions(arr(lib.spl_bed_chrom, np.int32), arr(lib.spl_bed_left, np.int32), arr(lib.spl_bed_right, np.int32),
                         arr(lib.spl_bed_score, np.int64), arr(lib.spl_bed_strand, np.uint8))
        sstr = StrandColumn(names(lib.spl_bed_n_strand_texts(h), lib.spl_bed_strand_text), arr(lib.spl_bed_strand_id, np.int32))
        chroms = names(lib.spl_bed_n_chrom(h), lib.spl_bed_chrom_name)
    finally:
        lib.spl_bed_free(h)
    return chroms, junc, sstr


def write_junctions_bed(path, chroms, junc: Junctions):
    """The BED12 of an extracted junction table in regtools' layout (spl_write_junctions_bed): chromStart / chromEnd from the
    anchor extents junc.start / junc.end, names JUNC00000001, ... in row order.  parse_bed12 of the file gives back
    (chrom, left, right, score, strand).  Byte parity with regtools itself is not pinned."""
    from .hosttext import StrTable
    if junc.start is None:
        raise ValueError("the junction table has no anchor extents (start / end)")
    lib = L.load()
    tab = StrTable(list(chroms))
    err = C.create_string_buffer(256)
    p32 = lambda a: a.ctypes.data_as(L.c_i32p)  # noqa: E731
    rc = lib.spl_write_junctions_bed(str(path).encode(), len(junc), p32(junc.chrom), p32(junc.left), p32(junc.right), p32(junc.start),
                                     p32(junc.end), junc.score.ctypes.data_as(L.c_i64p), junc.strand.ctypes.data_as(L.c_u8p), tab.ref(),
                                     err, 256)
    if rc != 0:
        raise (ValueError if rc == -1 else IOError)(err.value.decode())
