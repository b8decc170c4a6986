"""ctypes binding of libspliser_b200.so (include/spliser_b200.h).  Fails loudly when the library is
missing or a symbol is absent -- there is no Python or CPU fallback for the counting path."""
from __future__ import annotations

import ctypes as C
import os

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "libspliser_b200.so")

SPL_FLAG_STRANDED = 1
SPL_FLAG_RF = 2
SPL_FLAG_CRYPTIC = 4
SPL_FLAG_COMBINE = 8
SPL_FLAG_XS_STRAND = 16

SPL_NSTATS = 32
STAT_NAMES = ("ms_total", "ms_beta1", "ms_spliced", "ms_final", "n_mblocks_a", "n_mblocks_b", "n_junc_ops",
              "n_spliced", "n_sites", "n_edges", "n_aligned", "launches", "ms_expand", "ms_decode",
              "h2d_bytes", "d2h_bytes", "ms_graph", "ms_upload", "ms_count", "n_distinct_junc", "n_simple_junc", "n_complex_junc", "graph_on_device", "bam_on_device", "n_parts", "ms_graph_dev", "graph_timed", "n_hot_items", "ms_extract", "ms_extents", "n_junctions", "r31")

c_i32p = C.POINTER(C.c_int32)
c_i64p = C.POINTER(C.c_int64)
c_u8p = C.POINTER(C.c_uint8)
c_u16p = C.POINTER(C.c_uint16)
c_u32p = C.POINTER(C.c_uint32)
c_f64p = C.POINTER(C.c_double)
c_strp = C.POINTER(C.c_char_p)


class RecordsView(C.Structure):
    _fields_ = [("n_rec", C.c_int64), ("n_cigar", C.c_int64), ("pos", c_i32p), ("flag", c_u16p),
                ("cig_off", c_u32p), ("cigar", c_u32p), ("n_seg", C.c_int32), ("seg_chrom", c_i32p),
                ("seg_off", c_i64p)]


class PackedView(C.Structure):
    _fields_ = [("n_rec", C.c_int64), ("n_cigar", C.c_int64), ("pos", c_i32p), ("flag8", c_u8p), ("n_op", c_u16p),
                ("cigar", c_u32p), ("cig_index", c_u32p), ("n_seg", C.c_int32), ("seg_chrom", c_i32p), ("seg_off", c_i64p)]


class CompactView(C.Structure):
    _fields_ = [("n_rec", C.c_int64), ("n_cigar", C.c_int64), ("n16", C.c_int64), ("n32", C.c_int64), ("n_wide", C.c_int64),
                ("pos16", c_u16p), ("flag8", c_u8p), ("n_op8", c_u8p), ("cigar16", c_u16p), ("cigar32", c_u32p),
                ("pos_base", c_i32p), ("pos_wide", c_i32p), ("idx16", c_u32p), ("idx32", c_u32p),
                ("n_seg", C.c_int32), ("seg_chrom", c_i32p), ("seg_off", c_i64p)]


class StrTab(C.Structure):
    _fields_ = [("n", C.c_int64), ("blob", C.c_char_p), ("off", c_i64p)]


class ExtractOpts(C.Structure):
    _fields_ = [("min_anchor", C.c_int32), ("min_intron", C.c_int32), ("max_intron", C.c_int32), ("qchrom", C.c_char_p),
                ("use_gene_window", C.c_int32), ("gene_left", C.c_int64), ("gene_right", C.c_int64), ("window_max_intron", C.c_int64)]


class SiteColumns(C.Structure):
    _fields_ = [("n_sites", C.c_int64), ("chrom", c_i32p), ("pos", c_i32p), ("first_line", c_i64p),
                ("alpha", c_i64p), ("beta1", c_i64p), ("beta2simple", c_i64p), ("beta2cryptic", c_i64p),
                ("beta2weighted", c_f64p), ("sse", c_f64p), ("partner_off", c_i64p), ("partner_pos", c_i32p),
                ("partner_cnt", c_i64p), ("comp_off", c_i64p), ("comp_pos", c_i32p)]


_JUNC = [C.c_int64, c_i32p, c_i32p, c_i32p, c_i64p, c_u8p]
_GAPS = [C.c_int64, c_i32p, c_i32p, c_u8p, c_i64p, c_i32p, c_i64p, c_i32p]

# every symbol declared in include/spliser_b200.h: name -> (restype, argtypes)
SIGNATURES = {
    "spl_version": (C.c_char_p, []),
    "spl_kernel_launches": (C.c_ulonglong, []),
    "spl_create": (C.c_int, [C.POINTER(C.c_void_p), c_i32p, C.c_int]),
    "spl_destroy": (None, [C.c_void_p]),
    "spl_last_error": (C.c_char_p, [C.c_void_p]),
    "spl_set_tile": (C.c_int, [C.c_void_p, C.c_int, C.c_int]),
    "spl_set_tile_sites": (C.c_int, [C.c_void_p, C.c_int64, C.c_int64]),
    "spl_set_threads": (C.c_int, [C.c_void_p, C.c_int]),
    "spl_set_variant": (C.c_int, [C.c_void_p, C.c_int]),
    "spl_last_stats": (C.c_int, [C.c_void_p, c_f64p]),
    "spl_process": (C.c_int, [C.c_void_p, C.c_char_p, C.c_int32, c_strp] + _JUNC + [C.c_uint32, C.POINTER(C.c_void_p)]),
    "spl_process_records": (C.c_int, [C.c_void_p, C.POINTER(RecordsView), C.c_int32] + _JUNC + [C.c_uint32, C.POINTER(C.c_void_p)]),
    "spl_process_packed": (C.c_int, [C.c_void_p, C.POINTER(PackedView), C.c_int32] + _JUNC + [C.c_uint32, C.POINTER(C.c_void_p)]),
    "spl_process_compact": (C.c_int, [C.c_void_p, C.POINTER(CompactView), C.c_int32] + _JUNC + [C.c_uint32, C.POINTER(C.c_void_p)]),
    "spl_extract_junctions": (C.c_int, [C.c_void_p, C.c_char_p, C.c_int32, c_strp, C.c_int32, C.c_int32, C.c_int32, C.c_uint32, C.POINTER(C.c_void_p)]),
    "spl_extract_junctions_records": (C.c_int, [C.c_void_p, C.POINTER(RecordsView), C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_uint32, C.POINTER(C.c_void_p)]),
    "spl_extract_junctions_records_xs": (C.c_int, [C.c_void_p, C.POINTER(RecordsView), c_u8p, C.c_int32, C.c_int32, C.c_int32, C.c_int32,
                                                   C.c_uint32, C.POINTER(C.c_void_p)]),
    "spl_junctions_n": (C.c_int64, [C.c_void_p]),
    "spl_junctions_chrom": (c_i32p, [C.c_void_p]),
    "spl_junctions_left": (c_i32p, [C.c_void_p]),
    "spl_junctions_right": (c_i32p, [C.c_void_p]),
    "spl_junctions_score": (c_i64p, [C.c_void_p]),
    "spl_junctions_strand": (c_u8p, [C.c_void_p]),
    "spl_junctions_start": (c_i32p, [C.c_void_p]),
    "spl_junctions_end": (c_i32p, [C.c_void_p]),
    "spl_junctions_free": (None, [C.c_void_p]),
    "spl_process_bam_extract": (C.c_int, [C.c_void_p, C.c_char_p, C.c_int32, c_strp, C.POINTER(ExtractOpts), C.c_uint32,
                                          C.POINTER(C.c_void_p), C.POINTER(C.c_void_p)]),
    "spl_bam_reference_names": (C.c_int, [C.c_char_p, C.c_char_p, C.c_int64, c_i64p, c_i64p, C.c_char_p, C.c_int]),
    "spl_write_junctions_bed": (C.c_int, [C.c_char_p, C.c_int64, c_i32p, c_i32p, c_i32p, c_i32p, c_i32p, c_i64p, c_u8p,
                                          C.POINTER(StrTab), C.c_char_p, C.c_int]),
    "spl_recount": (C.c_int, [C.c_void_p, C.c_char_p, C.c_int32, c_strp] + _GAPS + [C.c_uint32, c_i64p, c_i64p]),
    "spl_recount_records": (C.c_int, [C.c_void_p, C.POINTER(RecordsView), C.c_int32] + _GAPS + [C.c_uint32, c_i64p, c_i64p]),
    "spl_build_site_table": (C.c_int, [C.c_int32] + _JUNC + [C.c_uint32, C.POINTER(C.c_void_p), C.c_char_p, C.c_int]),
    "spl_result_n_sites": (C.c_int64, [C.c_void_p]),
    "spl_result_chrom": (c_i32p, [C.c_void_p]),
    "spl_result_pos": (c_i32p, [C.c_void_p]),
    "spl_result_strand": (c_u8p, [C.c_void_p]),
    "spl_result_alpha": (c_i64p, [C.c_void_p]),
    "spl_result_beta1": (c_i64p, [C.c_void_p]),
    "spl_result_beta2simple": (c_i64p, [C.c_void_p]),
    "spl_result_beta2cryptic": (c_i64p, [C.c_void_p]),
    "spl_result_beta2weighted": (c_f64p, [C.c_void_p]),
    "spl_result_sse": (c_f64p, [C.c_void_p]),
    "spl_result_first_line": (c_i64p, [C.c_void_p]),
    "spl_result_partner_off": (c_i64p, [C.c_void_p]),
    "spl_result_partner_pos": (c_i32p, [C.c_void_p]),
    "spl_result_partner_cnt": (c_i64p, [C.c_void_p]),
    "spl_result_comp_off": (c_i64p, [C.c_void_p]),
    "spl_result_comp_pos": (c_i32p, [C.c_void_p]),
    "spl_result_free": (None, [C.c_void_p]),
    "spl_resident_load": (C.c_int, [C.c_void_p, C.POINTER(RecordsView), C.c_int32] + _JUNC + [C.c_uint32]),
    "spl_resident_count": (C.c_int, [C.c_void_p, C.c_int, c_f64p]),
    "spl_resident_fetch": (C.c_int, [C.c_void_p, C.POINTER(C.c_void_p)]),
    "spl_write_bam": (C.c_int, [C.c_char_p, C.c_int32, c_strp, c_i32p, C.POINTER(RecordsView), C.c_int]),
    "spl_write_bam_seq": (C.c_int, [C.c_char_p, C.c_int32, c_strp, c_i32p, C.POINTER(RecordsView), C.c_int]),
    "spl_write_bam_aux": (C.c_int, [C.c_char_p, C.c_int32, c_strp, c_i32p, C.POINTER(RecordsView), c_i64p, c_u8p, C.c_int, C.c_int]),
    "spl_read_bam": (C.c_int, [C.c_char_p, C.c_int32, c_strp, C.c_int, C.POINTER(C.c_void_p), C.c_char_p, C.c_int]),
    "spl_read_bam_xs": (C.c_int, [C.c_char_p, C.c_int32, c_strp, C.c_int, C.POINTER(C.c_void_p), C.c_char_p, C.c_int]),
    "spl_records_get": (C.POINTER(RecordsView), [C.c_void_p]),
    "spl_records_xs": (c_u8p, [C.c_void_p]),
    "spl_records_free": (None, [C.c_void_p]),
    "spl_debug_inflate": (C.c_int, [c_u8p, C.c_uint32, c_u8p, C.c_uint32, c_u32p]),
    "spl_bed_parse": (C.c_int, [C.c_char_p, C.c_int64, C.POINTER(StrTab), C.c_char_p, C.c_int, C.c_int64, C.c_int64, C.c_int64,
                                C.POINTER(C.c_void_p), C.c_char_p, C.c_int]),
    "spl_bed_free": (None, [C.c_void_p]),
    "spl_bed_n_junctions": (C.c_int64, [C.c_void_p]),
    "spl_bed_chrom": (c_i32p, [C.c_void_p]),
    "spl_bed_left": (c_i32p, [C.c_void_p]),
    "spl_bed_right": (c_i32p, [C.c_void_p]),
    "spl_bed_score": (c_i64p, [C.c_void_p]),
    "spl_bed_strand": (c_u8p, [C.c_void_p]),
    "spl_bed_strand_id": (c_i32p, [C.c_void_p]),
    "spl_bed_n_chrom": (C.c_int64, [C.c_void_p]),
    "spl_bed_chrom_name": (C.c_void_p, [C.c_void_p, C.c_int64, c_i64p]),
    "spl_bed_n_strand_texts": (C.c_int64, [C.c_void_p]),
    "spl_bed_strand_text": (C.c_void_p, [C.c_void_p, C.c_int64, c_i64p]),
    "spl_genes_parse": (C.c_int, [C.c_char_p, C.c_int64, C.c_char_p, C.POINTER(C.c_void_p), C.c_char_p, C.c_int]),
    "spl_genes_free": (None, [C.c_void_p]),
    "spl_genes_n": (C.c_int64, [C.c_void_p]),
    "spl_genes_n_chrom": (C.c_int64, [C.c_void_p]),
    "spl_genes_chrom_name": (C.c_void_p, [C.c_void_p, C.c_int64, c_i64p]),
    "spl_genes_chrom_off": (c_i64p, [C.c_void_p]),
    "spl_genes_left": (c_i32p, [C.c_void_p]),
    "spl_genes_right": (c_i32p, [C.c_void_p]),
    "spl_genes_strand_id": (c_i32p, [C.c_void_p]),
    "spl_genes_n_strand_texts": (C.c_int64, [C.c_void_p]),
    "spl_genes_strand_text": (C.c_void_p, [C.c_void_p, C.c_int64, c_i64p]),
    "spl_genes_names": (C.c_void_p, [C.c_void_p]),
    "spl_genes_name_off": (c_i64p, [C.c_void_p]),
    "spl_genes_query": (C.c_int64, [C.c_void_p]),
    "spl_gene_search": (C.c_int, [C.c_int64, c_i32p, c_i32p, c_i32p, C.c_int64, c_i32p, c_i32p, C.c_int32, C.c_int32, C.c_int, c_i32p]),
    "spl_write_process_tsv": (C.c_int, [C.c_char_p, C.POINTER(SiteColumns), C.POINTER(StrTab), C.POINTER(StrTab), c_i32p,
                                        C.POINTER(StrTab), c_i32p, C.c_int, C.c_char_p, C.c_int]),
    "spl_combine_create": (C.c_int, [C.POINTER(C.c_void_p)]),
    "spl_combine_destroy": (None, [C.c_void_p]),
    "spl_combine_last_error": (C.c_char_p, [C.c_void_p]),
    "spl_combine_set_threads": (C.c_int, [C.c_void_p, C.c_int]),
    "spl_combine_add_sample": (C.c_int, [C.c_void_p, C.c_char_p, C.c_char_p]),
    "spl_combine_add_samples": (C.c_int, [C.c_void_p, C.c_int64, c_strp, c_strp, C.c_int]),
    "spl_combine_n_samples": (C.c_int64, [C.c_void_p]),
    "spl_combine_n_regions": (C.c_int64, [C.c_void_p]),
    "spl_combine_region_name": (C.c_char_p, [C.c_void_p, C.c_int64]),
    "spl_combine_sample_rows": (C.c_int64, [C.c_void_p, C.c_int64]),
    "spl_combine_sample_runs": (C.c_int64, [C.c_void_p, C.c_int64, C.POINTER(c_i32p)]),
    "spl_combine_merge": (C.c_int, [C.c_void_p, C.c_int64, c_i32p, C.c_char_p, C.c_int]),
    "spl_combine_merge_shallow": (C.c_int, [C.c_void_p, C.c_int64, c_i32p, C.c_char_p, C.c_int, C.c_int64, C.c_int64, C.c_double]),
    "spl_combine_n_sites": (C.c_int64, [C.c_void_p]),
    "spl_combine_n_filled": (C.c_int64, [C.c_void_p]),
    "spl_combine_gaps": (C.c_int64, [C.c_void_p, C.c_int64, C.POINTER(c_i32p), C.POINTER(c_i32p), C.POINTER(c_u8p),
                                     C.POINTER(c_i64p), C.POINTER(c_i32p), C.POINTER(c_i64p), C.POINTER(c_i32p)]),
    "spl_combine_set_recount": (C.c_int, [C.c_void_p, C.c_int64, C.c_int64, c_i64p, c_i64p]),
    "spl_combine_write": (C.c_int, [C.c_void_p, C.c_char_p, C.c_int]),
    "spl_host_alloc": (C.c_void_p, [C.c_size_t]),
    "spl_host_free": (None, [C.c_void_p]),
}

_lib = None


class SpliserLibraryError(RuntimeError):
    pass


def load():
    """Loads the shared library and binds every declared symbol; raises if anything is missing."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise SpliserLibraryError(
            "%s not found: build it with `python -m spliser_b200.build` (nvcc, sm_100a). "
            "spliser_b200 has no CPU fallback." % LIB_PATH)
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        try:
            fn = getattr(lib, name)
        except AttributeError as e:
            raise SpliserLibraryError("libspliser_b200.so does not export %s" % name) from e
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib
