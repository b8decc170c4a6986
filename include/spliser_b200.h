/* spliser_b200.h -- C ABI of libspliser_b200.so
 *
 * Drop-in boundary for the counting path of SpliSER v0.1.8 (`process`, and the re-count that
 * `combine` performs for sites missing from a sample).  The reference has no FFI of its own;
 * this seam replaces, inside /root/reference/SpliSER_v0_1_8.py ("S:"):
 *
 *   spl_process*   <- S:710-717  findAlphaCounts (S:227-362, after the BED text filters of
 *                     S:255-288), findCompetitorPos (S:364-372), processSites (S:681-692) with
 *                     checkBam (S:408-559), findBeta2Counts (S:581-623), calculateSSE (S:626-639)
 *   spl_recount*   <- S:903 (and S:1145)  checkBam for a (site, sample) gap in combine mode
 *
 * Plain pointers and sizes only; no torch / C++ types.  All functions return 0 on success or a
 * negative spl_status; the message is available from spl_last_error().  Nothing here ever calls
 * exit() or throws across the boundary.  A context is not thread-safe: one call at a time per
 * spl_ctx (the reference is single-threaded with module-global state, S:23-47); different
 * contexts may be used concurrently.  There is NO CPU fallback: every entry point that counts
 * fails with SPL_ERR_CUDA when no sm_100 device is usable.
 *
 * Conventions
 *   positions   1-based int32, the reference's site convention (S:274-276, S:482-483)
 *   strands     one raw byte per junction/site: the first byte of BED column 6 ('+', '-', '?', ...);
 *               0 means the empty strand '' of combine's makeSingleSpliceSite (S:855)
 *   chromosomes int32 index into the caller's chrom_index order (S:23, S:90, S:265)
 *   counts      int64 at the ABI (device counters are u32 per launch, widened on the device)
 *   ownership   inputs are borrowed for the duration of the call; spl_result is library-owned
 *               until spl_result_free; spl_recount* outputs are caller-allocated
 */
#ifndef SPLISER_B200_H
#define SPLISER_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct spl_ctx spl_ctx;
typedef struct spl_result spl_result;

typedef enum spl_status {
    SPL_OK = 0,
    SPL_ERR_ARG = -1,      /* bad argument (null pointer, negative size, unsorted input ...) */
    SPL_ERR_CUDA = -2,     /* CUDA runtime / no usable device / kernel failure */
    SPL_ERR_IO = -3,       /* BAM file cannot be opened / is truncated / is not BGZF-BAM */
    SPL_ERR_NOMEM = -4,
    SPL_ERR_RANGE = -5     /* input exceeds a 32-bit device index (e.g. > 2^32 CIGAR ops per call) */
} spl_status;

/* flags for spl_process* / spl_recount* (S:1314-1316; COMBINE mirrors sys.argv[1] at S:531) */
#define SPL_FLAG_STRANDED 1u   /* --isStranded */
#define SPL_FLAG_RF       2u   /* -s rf (else fr); only read when STRANDED */
#define SPL_FLAG_CRYPTIC  4u   /* --beta2Cryptic: SSE includes beta2Cryptic_weighted (S:633-635) */
#define SPL_FLAG_COMBINE  8u   /* checkBam runs under `combine`: flanking reads add beta2Simple (S:531-532) */
/* Junction extraction only (spl_extract_junctions, spl_extract_junctions_records_xs, spl_process_bam_extract): the table's
 * strands come from the aligner's XS tag, as `regtools junctions extract` takes them for unstranded libraries; STRANDED / RF
 * then do not touch the table (spl_process_bam_extract still counts with them).  The rule, one strand per record:
 *   - walk the aux fields in order from the end of QUAL to the end of the record, sizing each by its type: A c C 1 byte,
 *     s S 2, i I f 4, Z H up to and including the NUL, B a subtype byte, a u32 count and count x the subtype's size
 *     (1 for c C, 2 for s S, 4 otherwise);
 *   - the FIRST field tagged exactly XS decides: XS:A:+ gives '+', XS:A:- gives '-', any other type or character '?'
 *     (later XS fields are ignored, as htslib's bam_aux_get does);
 *   - '?' also when there is no XS field, or when an unknown type byte or a field running past the end of the record (a Z
 *     without its NUL does) comes before it.  A malformed aux block is not an error.
 * Every junction a record supports takes that record's strand.  Deviation: regtools writes other XS:A characters (such as
 * '.') through unchanged; here they are '?'. */
#define SPL_FLAG_XS_STRAND 16u

/* ---- context ------------------------------------------------------------------------------- */
/* device_ids: CUDA ordinals this context drives (one process per GPU: pass exactly one).
 * tile_index / tile_count (spl_set_tile) select the genomic tile this context owns when a job
 * is sharded over several processes: the context then counts only sites whose global index
 * (reference list order) falls in its tile and zero-fills the rest. */
int  spl_create(spl_ctx** out, const int* device_ids, int n_devices);
void spl_destroy(spl_ctx* ctx);
const char* spl_last_error(const spl_ctx* ctx);   /* NUL-terminated, valid until next call on ctx */
int  spl_set_tile(spl_ctx* ctx, int tile_index, int tile_count);
/* The same with an explicit owned range [site_lo, site_hi) of global site indices (reference list order), for tiles
 * balanced by read count rather than by site count (SURVEY 8(e)); (-1, -1) returns to spl_set_tile's equal slices. */
int  spl_set_tile_sites(spl_ctx* ctx, int64_t site_lo, int64_t site_hi);
int  spl_set_threads(spl_ctx* ctx, int n_host_threads);   /* BGZF inflate / record parse workers */
/* Counting variant of the following calls on this context.  Both give identical results (tests hold them to each other
 * and to the reference); FUSED is the product path, STAB the cross-check north_star asks for:
 *   SPL_VARIANT_FUSED  one kernel walks the records' CIGARs and range-adds into difference arrays over the site
 *                      table (S:469, S:507 as +1/-1 at two lower_bound indices), prefix scan in the finalize kernel
 *   SPL_VARIANT_STAB   records are first expanded into a bin-partitioned block stream; a block-vs-site stabbing
 *                      kernel with TMA-staged site tiles counts coverage, junctions are handled per distinct junction */
#define SPL_VARIANT_FUSED 0
#define SPL_VARIANT_STAB  1
int  spl_set_variant(spl_ctx* ctx, int variant);
const char* spl_version(void);
unsigned long long spl_kernel_launches(void);   /* kernels this library has launched in this process so far (every launch is counted) */

/* ---- process (S:710-717) ------------------------------------------------------------------- */
/* Junction table = BED12 lines in file order AFTER the 12-column / -c / -g filters (S:259-288):
 * j_left = int(col1)+blockSizes[0], j_right = int(col2)-blockSizes[1], j_score = int(col4),
 * j_strand = first byte of col5 (S:272-277).  chrom_names[i] is chrom_index[i]. */
int spl_process(spl_ctx* ctx, const char* bam_path,
                int32_t n_chrom, const char* const* chrom_names,
                int64_t n_junc, const int32_t* j_chrom, const int32_t* j_left, const int32_t* j_right,
                const int64_t* j_score, const uint8_t* j_strand,
                uint32_t flags, spl_result** out);

/* Same, with the alignment records already decoded into host arrays (what `samtools view`
 * would print, S:429-437: FLAG, POS, CIGAR).  Records are grouped in segments of one chromosome
 * each (a coordinate-sorted BAM has one segment per reference); coordinate-sorted input is
 * fastest, but any record order inside a segment gives the same counts. */
typedef struct spl_records_view {
    int64_t n_rec;
    int64_t n_cigar;              /* == cig_off[n_rec]; must be < 2^32 */
    const int32_t*  pos;          /* [n_rec]   1-based leftmost position (SAM POS) */
    const uint16_t* flag;         /* [n_rec]   SAM FLAG */
    const uint32_t* cig_off;      /* [n_rec+1] offsets into cigar[] */
    const uint32_t* cigar;        /* [n_cigar] BAM-encoded: len<<4 | op, op indexes "MIDNSHP=X" */
    int32_t n_seg;
    const int32_t*  seg_chrom;    /* [n_seg]   chrom_index of the segment; < 0 = not a known chromosome (skipped) */
    const int64_t*  seg_off;      /* [n_seg+1] records [seg_off[k], seg_off[k+1]) form segment k */
} spl_records_view;

int spl_process_records(spl_ctx* ctx, const spl_records_view* rec,
                        int32_t n_chrom,
                        int64_t n_junc, const int32_t* j_chrom, const int32_t* j_left, const int32_t* j_right,
                        const int64_t* j_score, const uint8_t* j_strand,
                        uint32_t flags, spl_result** out);

/* The same from a packed host layout: 17 bytes per record instead of 20 cross PCIe (the copy is what bounds the call).
 * Per record POS, the three flag bits check_strand reads (S:374-406) and the operator count; a sparse index gives the CIGAR
 * offset of every SPL_PACKED_INDEX_STRIDE-th record (what a decoder knows as it appends), the per-record offsets are
 * rebuilt on the device.  Records with more than 65535 operators (BAM's own n_cigar_op limit) need the plain view. */
#define SPL_PACKED_INDEX_STRIDE 1024
typedef struct spl_packed_view {
    int64_t n_rec;
    int64_t n_cigar;
    const int32_t*  pos;          /* [n_rec]   1-based leftmost position (SAM POS) */
    const uint8_t*  flag8;        /* [n_rec]   bit 0 = FLAG & 0x1 (paired), bit 1 = FLAG & 0x10 (reverse), bit 2 = FLAG & 0x40 (first in pair) */
    const uint16_t* n_op;         /* [n_rec]   CIGAR operators of the record */
    const uint32_t* cigar;        /* [n_cigar] BAM-encoded operators of all records, back to back */
    const uint32_t* cig_index;    /* [n_rec / STRIDE + 1] offset into cigar[] of record k * STRIDE */
    int32_t n_seg;
    const int32_t*  seg_chrom;    /* as in spl_records_view */
    const int64_t*  seg_off;
} spl_packed_view;

int spl_process_packed(spl_ctx* ctx, const spl_packed_view* rec,
                       int32_t n_chrom,
                       int64_t n_junc, const int32_t* j_chrom, const int32_t* j_left, const int32_t* j_right,
                       const int64_t* j_score, const uint8_t* j_strand,
                       uint32_t flags, spl_result** out);

/* The same from a compact host layout: about 9 bytes per record cross PCIe.  Records are taken in strides of
 * SPL_PACKED_INDEX_STRIDE (the last one may be short).  POS travels as a 16-bit offset from pos_base[stride] (the lowest POS of
 * the stride); a stride whose positions span more than 65535 has pos_base = -(w + 1) and its POS values, 32-bit, in
 * pos_wide[w * STRIDE ..].  A record's operators are 16-bit words (op | len << 4) in cigar16 when every length is below 4096,
 * else BAM-encoded 32-bit words in cigar32 (flag8 bit 3 says which); idx16 / idx32 give the offset of every stride's first
 * record in the two streams, so that a decoder appends to both as it goes and the device unpacks every stride on its own.
 * Records with more than 255 operators need the plain or the packed view. */
typedef struct spl_compact_view {
    int64_t n_rec;
    int64_t n_cigar;              /* operators of all records (n16 + n32); must be < 2^32 */
    int64_t n16, n32;             /* words in cigar16 / cigar32 */
    int64_t n_wide;               /* strides listed in pos_wide */
    const uint16_t* pos16;        /* [n_rec]   POS - pos_base[r / STRIDE] (anything for records of a wide stride) */
    const uint8_t*  flag8;        /* [n_rec]   bits 0-2 as in spl_packed_view; bit 3: the operators are in cigar32 */
    const uint8_t*  n_op8;        /* [n_rec]   CIGAR operators of the record */
    const uint16_t* cigar16;      /* [n16] */
    const uint32_t* cigar32;      /* [n32] */
    const int32_t*  pos_base;     /* [ceil(n_rec / STRIDE)] */
    const int32_t*  pos_wide;     /* [n_wide * STRIDE] */
    const uint32_t* idx16;        /* [ceil(n_rec / STRIDE) + 1] */
    const uint32_t* idx32;        /* [ceil(n_rec / STRIDE) + 1] */
    int32_t n_seg;
    const int32_t*  seg_chrom;    /* as in spl_records_view */
    const int64_t*  seg_off;
} spl_compact_view;

int spl_process_compact(spl_ctx* ctx, const spl_compact_view* rec,
                        int32_t n_chrom,
                        int64_t n_junc, const int32_t* j_chrom, const int32_t* j_left, const int32_t* j_right,
                        const int64_t* j_score, const uint8_t* j_strand,
                        uint32_t flags, spl_result** out);

/* ---- combine re-count (S:899-904) ---------------------------------------------------------- */
/* One call per sample.  For gap site i: position s_pos[i] on chromosome s_chrom[i] with strand
 * byte s_strand[i] (0 = ''), partner positions p_pos[p_off[i] .. p_off[i+1]) (keys of
 * PartnerCounts, S:417-419) and competitor positions c_pos[c_off[i] .. c_off[i+1]).
 * SPL_FLAG_COMBINE is implied.  Writes beta1_out[i], beta2simple_out[i]. */
int spl_recount(spl_ctx* ctx, const char* bam_path, int32_t n_chrom, const char* const* chrom_names,
                int64_t n_sites, const int32_t* s_chrom, const int32_t* s_pos, const uint8_t* s_strand,
                const int64_t* p_off, const int32_t* p_pos, const int64_t* c_off, const int32_t* c_pos,
                uint32_t flags, int64_t* beta1_out, int64_t* beta2simple_out);
int spl_recount_records(spl_ctx* ctx, const spl_records_view* rec,
                        int32_t n_chrom,
                        int64_t n_sites, const int32_t* s_chrom, const int32_t* s_pos, const uint8_t* s_strand,
                        const int64_t* p_off, const int32_t* p_pos, const int64_t* c_off, const int32_t* c_pos,
                        uint32_t flags, int64_t* beta1_out, int64_t* beta2simple_out);

/* Host-only half of findAlphaCounts + findCompetitorPos (S:289-372): the site table in output order,
 * alpha, PartnerCounts and CompetitorPos from the junction table alone.  beta1 / beta2* / SSE are
 * zero: they need the alignments and therefore the GPU.  Useful for tools that only need the site
 * universe, and for testing the host logic on a machine without a GPU. */
int spl_build_site_table(int32_t n_chrom,
                         int64_t n_junc, const int32_t* j_chrom, const int32_t* j_left, const int32_t* j_right,
                         const int64_t* j_score, const uint8_t* j_strand,
                         uint32_t flags, spl_result** out, char* err, int err_len);

/* ---- junction extraction (SURVEY 8(f) row 3) -------------------------------------------------
 * The junction table `process` needs, from the alignments themselves: replaces the `regtools junctions extract` pre-step
 * of the reference's workflow (README.md:41) -- alpha is then the count of the same records the beta terms are counted
 * from (S:274-277 reads it from the BED12 score column).  A record supports the junction (l, r) of one of its N operators
 * when min_intron <= length(N) <= max_intron and the aligned stretches on both sides of the N (M/=/X/D operators up to the
 * neighbouring N or the end of the read) are at least min_anchor long; regtools' defaults are 8 / 70 / 500000.  regtools is
 * not part of the reference tree: these rules are restated from its documentation (parity unpinned; the tests pin the
 * kernel to synthetic samples whose generator knows the table).  Strand: with SPL_FLAG_XS_STRAND the record's XS tag (rule
 * above), else with SPL_FLAG_STRANDED the strand check_strand derives from the FLAG ('+' / '-'), else '?'.  Rows are sorted by
 * (chromosome, l, r, strand) with '?' < '+' < '-'.  spl_extract_junctions_records has no tags to read: SPL_FLAG_XS_STRAND is
 * SPL_ERR_ARG there; spl_extract_junctions_records_xs takes the strands from xs[n_rec] ('+', '-' or '?' per record, e.g.
 * spl_records_xs) when the flag is set. */
typedef struct spl_junctions spl_junctions;
int spl_extract_junctions(spl_ctx* ctx, const char* bam_path, int32_t n_chrom, const char* const* chrom_names,
                          int32_t min_anchor, int32_t min_intron, int32_t max_intron, uint32_t flags, spl_junctions** out);
int spl_extract_junctions_records(spl_ctx* ctx, const spl_records_view* rec, int32_t n_chrom,
                                  int32_t min_anchor, int32_t min_intron, int32_t max_intron, uint32_t flags, spl_junctions** out);
int spl_extract_junctions_records_xs(spl_ctx* ctx, const spl_records_view* rec, const uint8_t* xs, int32_t n_chrom,
                                     int32_t min_anchor, int32_t min_intron, int32_t max_intron, uint32_t flags, spl_junctions** out);
int64_t        spl_junctions_n(const spl_junctions* j);
const int32_t* spl_junctions_chrom(const spl_junctions* j);
const int32_t* spl_junctions_left(const spl_junctions* j);      /* j_left / j_right / j_score / j_strand of spl_process */
const int32_t* spl_junctions_right(const spl_junctions* j);
const int64_t* spl_junctions_score(const spl_junctions* j);
const uint8_t* spl_junctions_strand(const spl_junctions* j);
/* Anchor extents, what a BED12 of the table carries in chromStart / chromEnd: start = left - the longest flanking stretch in
 * front of the junction among its supporting records, end = right + the longest one behind it (stretches as above: M/=/X/D
 * since the previous N or the read start, up to the next N or the read end).  blockSizes = (left - start, end - right), so
 * that spl_bed_parse gives back left = chromStart + blockSizes[0] and right = chromEnd - blockSizes[1] (S:275-276). */
const int32_t* spl_junctions_start(const spl_junctions* j);
const int32_t* spl_junctions_end(const spl_junctions* j);
void spl_junctions_free(spl_junctions* j);

/* `process` without a BED12 file (the regtools step and process in one call): ingest the BAM once (on the device, or the host
 * reader as the fallback, as spl_process chooses), extract its junction table (min_anchor / min_intron / max_intron as
 * above; strands from SPL_FLAG_XS_STRAND, else SPL_FLAG_STRANDED / SPL_FLAG_RF), keep the rows `process` would keep of a BED12 holding that table
 * -- -c (S:269) and the -g window (S:279-288), the same filter code as spl_bed_parse -- and count those rows against the same
 * device-resident records as spl_process_records would.  *rows_out is the table after the filters in the order it was
 * counted (spl_result_first_line indexes it); free it with spl_junctions_free.  Writing *rows_out with
 * spl_write_junctions_bed and running spl_process on that file gives the same result. */
typedef struct spl_extract_opts {
    int32_t min_anchor, min_intron, max_intron;   /* regtools -a / -m / -M (8 / 70 / 500000) */
    const char* qchrom;                           /* -c: keep the rows of this chromosome name only; NULL = "All" */
    int32_t use_gene_window;                      /* -g: keep rows with a site in [gene_left - window_max_intron, gene_right + window_max_intron] */
    int64_t gene_left, gene_right, window_max_intron;
} spl_extract_opts;
int spl_process_bam_extract(spl_ctx* ctx, const char* bam_path, int32_t n_chrom, const char* const* chrom_names,
                            const spl_extract_opts* opts, uint32_t flags, spl_junctions** rows_out, spl_result** out);

/* Reference names of a BAM header in header order (host only, no GPU): written NUL-terminated back to back into
 * names[0 .. cap) when *bytes (the space they need) <= cap; *n_ref and *bytes are always set. */
int spl_bam_reference_names(const char* path, char* names, int64_t cap, int64_t* n_ref, int64_t* bytes, char* err, int err_len);

/* ---- result accessors ---------------------------------------------------------------------- */
/* Sites are in the reference's output order: chrom_index order, then the per-chromosome list
 * order of site2D_array (position ascending; '+' before '-' in a stranded run, G:123-136). */
int64_t        spl_result_n_sites(const spl_result* r);
const int32_t* spl_result_chrom(const spl_result* r);
const int32_t* spl_result_pos(const spl_result* r);
const uint8_t* spl_result_strand(const spl_result* r);
const int64_t* spl_result_alpha(const spl_result* r);
const int64_t* spl_result_beta1(const spl_result* r);
const int64_t* spl_result_beta2simple(const spl_result* r);
const int64_t* spl_result_beta2cryptic(const spl_result* r);
const double*  spl_result_beta2weighted(const spl_result* r);
const double*  spl_result_sse(const spl_result* r);
/* index of the BED line (into the junction table passed in) that created each site: the caller
 * assigns the Gene column with that line's strand (S:313) */
const int64_t* spl_result_first_line(const spl_result* r);
/* PartnerCounts in insertion order (TSV "Partners" column, S:662) and sorted CompetitorPos
 * (TSV "Competitors" column, S:663) as CSR over sites */
const int64_t* spl_result_partner_off(const spl_result* r);
const int32_t* spl_result_partner_pos(const spl_result* r);
const int64_t* spl_result_partner_cnt(const spl_result* r);
const int64_t* spl_result_comp_off(const spl_result* r);
const int32_t* spl_result_comp_pos(const spl_result* r);
void spl_result_free(spl_result* r);

/* ---- resident (benchmark) path -------------------------------------------------------------
 * Roofline measurements need the read SoA already in HBM when the timed region starts:
 *   spl_resident_load   uploads records + junction table, builds the site graph and expands
 *                       the records into the structure-of-arrays the counting kernels stream
 *   spl_resident_count  runs the per-sample path `iters` times on the context's stream, timed with CUDA
 *                       events on that stream; results stay in HBM.  Fused variant: site table + graph from
 *                       the resident junction table, counters zeroed, counting kernel over the resident
 *                       records, prefix scan + beta2 gather + SSE -- everything spl_process_records
 *                       launches for a sample except the copies.  Stabbing variant: the counting pass
 *                       over the layout spl_resident_load prepared.
 *   spl_resident_fetch  copies the last results to the host as an spl_result
 * stats_out (may be NULL) receives SPL_NSTATS doubles, see SPL_STAT_* below. */
int spl_resident_load(spl_ctx* ctx, const spl_records_view* rec,
                      int32_t n_chrom,
                      int64_t n_junc, const int32_t* j_chrom, const int32_t* j_left, const int32_t* j_right,
                      const int64_t* j_score, const uint8_t* j_strand, uint32_t flags);
int spl_resident_count(spl_ctx* ctx, int iters, double* stats_out);
int spl_resident_fetch(spl_ctx* ctx, spl_result** out);

#define SPL_STAT_MS_TOTAL      0   /* CUDA-event ms for all `iters` passes                      */
#define SPL_STAT_MS_BETA1      1   /* summed ms of the beta1 stabbing kernel                    */
#define SPL_STAT_MS_SPLICED    2   /* summed ms of the spliced-read kernel                      */
#define SPL_STAT_MS_FINAL      3   /* summed ms of alpha reduce + scan + beta2 gather + SSE     */
#define SPL_STAT_N_MBLOCKS_A   4   /* M/=/X blocks of unspliced reads                           */
#define SPL_STAT_N_MBLOCKS_B   5   /* M/=/X blocks of spliced reads                             */
#define SPL_STAT_N_JUNC_OPS    6   /* N operators                                               */
#define SPL_STAT_N_SPLICED     7   /* reads with >= 1 N operator                                */
#define SPL_STAT_N_SITES       8
#define SPL_STAT_N_EDGES       9   /* directed site->partner entries                            */
#define SPL_STAT_N_ALIGNED    10   /* records with >= 1 CIGAR op ("aligned reads")              */
#define SPL_STAT_LAUNCHES     11   /* kernels launched per pass (counted at the launch sites)   */
#define SPL_STAT_MS_EXPAND    12   /* ms of the record -> SoA expansion at load time            */
#define SPL_NSTATS            32

/* per-call statistics of the last spl_process* / spl_recount* call (same indices; MS_* are
 * host wall-clock of the stages; extra indices below) */
#define SPL_STAT_MS_DECODE    13   /* BAM inflate + parse (host wall ms)                        */
#define SPL_STAT_H2D_BYTES    14
#define SPL_STAT_D2H_BYTES    15
#define SPL_STAT_MS_GRAPH     16   /* host: site table + competing-site graph construction          */
#define SPL_STAT_MS_UPLOAD    17   /* host wall ms until records are uploaded and expanded           */
#define SPL_STAT_MS_COUNT     18   /* host wall ms of the counting pass + result download            */
#define SPL_STAT_N_DISTINCT_J 19   /* distinct (chromosome, l, r, class) junctions of the sample     */
#define SPL_STAT_N_SIMPLE_J   20   /* junction instances of block-N-block reads (aggregated path)    */
#define SPL_STAT_N_COMPLEX_J  21   /* junction instances handled per read                            */
#define SPL_STAT_BAM_DEVICE   23   /* 1 = BGZF inflate + BAM record parse ran on the device, 0 = host reader (fallback)  */
#define SPL_STAT_N_PARTS      24   /* parts the record upload was cut into (1 or 2; 2 = expansion overlapped with the copy)  */
#define SPL_STAT_GRAPH_DEVICE 22   /* 1 = site table + graph built on the device (clean regime), 0 = host emulation */
#define SPL_STAT_MS_GRAPH_DEV 25   /* spl_resident_count: summed CUDA-event ms of the site table + graph build inside the timed passes */
#define SPL_STAT_N_HOT_ITEMS  27   /* junction ends on hot sites queued for the exception kernel in the last pass (fused variant) */
#define SPL_STAT_GRAPH_TIMED  26   /* spl_resident_count: 1 = every pass rebuilt the site table + graph (fused variant, clean regime) */
#define SPL_STAT_MS_EXTRACT   28   /* junction extraction: CUDA-event ms of its kernels (anchor extents included)           */
#define SPL_STAT_MS_EXTENTS   29   /* junction extraction: CUDA-event ms of the anchor-extent walk alone                    */
#define SPL_STAT_N_JUNCTIONS  30   /* junction extraction: rows extracted (before the -c / -g filters of spl_process_bam_extract) */
int spl_last_stats(const spl_ctx* ctx, double* stats_out);

/* ---- host text layer (no GPU): Gene column, .SpliSER.tsv writer, combine merge driver ------------
 * What surrounds the counting call in the reference's CLI, done natively because per-row Python
 * string work costs seconds where the counting costs milliseconds.  Byte-identical output. */
typedef struct spl_strtab {          /* n strings: string i = blob[off[i] .. off[i+1]) (no terminators) */
    int64_t n;
    const char* blob;
    const int64_t* off;              /* [n+1] */
} spl_strtab;

typedef struct spl_site_columns {    /* the arrays of an spl_result (or any table in the same layout) */
    int64_t n_sites;
    const int32_t* chrom;  const int32_t* pos;  const int64_t* first_line;
    const int64_t* alpha;  const int64_t* beta1;  const int64_t* beta2simple;  const int64_t* beta2cryptic;
    const double* beta2weighted;  const double* sse;
    const int64_t* partner_off;  const int32_t* partner_pos;  const int64_t* partner_cnt;
    const int64_t* comp_off;  const int32_t* comp_pos;
} spl_site_columns;

/* The text half of findAlphaCounts (S:255-288) for a whole BED12 file image: lines with exactly 12
 * tab-separated fields (S:259), chromosome index in first-appearance order appended to chrom_index
 * (what the annotation registered, S:90-92, S:265-268; may be NULL), -c filter (qchrom, NULL = "All",
 * S:269), site positions and score (S:274-277), -g window (S:279-288) when use_gene_window != 0.
 * The result carries the junction table in the layout of spl_process, the id of every kept row's
 * column-6 text (for spl_write_process_tsv) and the two string lists.  A field int() would reject
 * fails the call (SPL_ERR_ARG; the reference raises ValueError). */
typedef struct spl_bed spl_bed;
int spl_bed_parse(const char* text, int64_t len, const spl_strtab* chrom_index, const char* qchrom,
                  int use_gene_window, int64_t gene_left, int64_t gene_right, int64_t max_intron,
                  spl_bed** out, char* err, int err_len);
void spl_bed_free(spl_bed* b);
int64_t spl_bed_n_junctions(const spl_bed* b);
const int32_t* spl_bed_chrom(const spl_bed* b);
const int32_t* spl_bed_left(const spl_bed* b);
const int32_t* spl_bed_right(const spl_bed* b);
const int64_t* spl_bed_score(const spl_bed* b);
const uint8_t* spl_bed_strand(const spl_bed* b);
const int32_t* spl_bed_strand_id(const spl_bed* b);
int64_t spl_bed_n_chrom(const spl_bed* b);
const char* spl_bed_chrom_name(const spl_bed* b, int64_t i, int64_t* len);
int64_t spl_bed_n_strand_texts(const spl_bed* b);
const char* spl_bed_strand_text(const spl_bed* b, int64_t i, int64_t* len);

/* createGenes (S:50-116) for a whole GFF / GTF file image, without HTSeq: feature lines of type "gene" give
 * leftPos = start - 1, rightPos = end, the strand column and, as name, the value of the first attribute
 * (README.md:64).  Chromosomes in first-appearance order among the gene lines (S:90-92); genes grouped by
 * chromosome (spl_genes_chrom_off), each list in insort order by leftPos (S:95).  With qgene != NULL only
 * the genes of that name are kept (file order) and spl_genes_query is the last of them (QUERY_gene). */
typedef struct spl_genes spl_genes;
int spl_genes_parse(const char* text, int64_t len, const char* qgene, spl_genes** out, char* err, int err_len);
void spl_genes_free(spl_genes* g);
int64_t spl_genes_n(const spl_genes* g);
int64_t spl_genes_n_chrom(const spl_genes* g);
const char* spl_genes_chrom_name(const spl_genes* g, int64_t i, int64_t* len);
const int64_t* spl_genes_chrom_off(const spl_genes* g);
const int32_t* spl_genes_left(const spl_genes* g);
const int32_t* spl_genes_right(const spl_genes* g);
const int32_t* spl_genes_strand_id(const spl_genes* g);
int64_t spl_genes_n_strand_texts(const spl_genes* g);
const char* spl_genes_strand_text(const spl_genes* g, int64_t i, int64_t* len);
const char* spl_genes_names(const spl_genes* g);          /* blob of all names, see spl_genes_name_off */
const int64_t* spl_genes_name_off(const spl_genes* g);    /* [n + 1] */
int64_t spl_genes_query(const spl_genes* g);              /* flat index of QUERY_gene, -1 = none */

/* binary_gene_search (S:118-173) for n positions against the genes of ONE chromosome in list order
 * (insort by leftPos, S:95), control flow kept: overlapping genes make the bisection order-dependent
 * and the last-ditch window (S:162-169) never looks at the last gene.  Strands are compared as ids
 * of the caller's string table (equal id <=> equal text); plus_id / minus_id are the ids of "+" / "-".
 * out_idx[i] = index into the gene list, or -1 ("NA"). */
int spl_gene_search(int64_t n_genes, const int32_t* g_left, const int32_t* g_right, const int32_t* g_strand,
                    int64_t n, const int32_t* pos, const int32_t* strand, int32_t plus_id, int32_t minus_id,
                    int is_stranded, int32_t* out_idx);

/* outputBedFile (S:641-664).  strand_texts = the distinct BED column-6 texts, line_strand[j] = id of
 * junction row j's text (the Strand column prints the text of the row that created the site:
 * first_line); site_gene[i] indexes gene_names, < 0 (or site_gene == NULL) prints "NA". */
/* The BED12 of a junction table in the layout `regtools junctions extract` writes (its documentation; byte parity with
 * regtools is not pinned), one line per row in table order:
 *   chrom  start  end  JUNC%08d  score  strand  start  end  255,0,0  2  a,b  0,end-start-b
 * with a = left - start, b = end - right; names are numbered from 1; chrom_names[chrom[i]] names row i's chromosome; a strand
 * byte 0 writes an empty column. */
int spl_write_junctions_bed(const char* path, int64_t n, const int32_t* chrom, const int32_t* left, const int32_t* right,
                            const int32_t* start, const int32_t* end, const int64_t* score, const uint8_t* strand,
                            const spl_strtab* chrom_names, char* err, int err_len);

int spl_write_process_tsv(const char* path, const spl_site_columns* table, const spl_strtab* chrom_names,
                          const spl_strtab* strand_texts, const int32_t* line_strand,
                          const spl_strtab* gene_names, const int32_t* site_gene, int cryptic,
                          char* err, int err_len);

/* combine (S:742-917) around the re-count: parse every sample's .SpliSER.tsv, replay the lock-step
 * merge (S:791-917; a gap of sample k sees the partners / competitors / strand gathered from the
 * samples before k only), hand out each sample's gap list in the argument layout of spl_recount
 * (s_chrom = region ids of spl_combine_region_name), take the counts back, write the .combined.tsv
 * (outputCombinedLines, S:722-740).  The region order (S:761-789) is the caller's: it gets the run
 * of consecutive distinct regions of every file from spl_combine_sample_runs. */
typedef struct spl_combine spl_combine;
int  spl_combine_create(spl_combine** out);
void spl_combine_destroy(spl_combine* c);
const char* spl_combine_last_error(const spl_combine* c);
int  spl_combine_set_threads(spl_combine* c, int n_threads);    /* parsing / formatting workers; 0 = all hardware threads */
int  spl_combine_add_sample(spl_combine* c, const char* title, const char* tsv_path);
/* n samples in samples-file order, parsed concurrently (n_threads 0 = the context's setting) */
int  spl_combine_add_samples(spl_combine* c, int64_t n, const char* const* titles, const char* const* tsv_paths,
                             int n_threads);
int64_t spl_combine_n_samples(const spl_combine* c);
int64_t spl_combine_n_regions(const spl_combine* c);
const char* spl_combine_region_name(const spl_combine* c, int64_t region);
int64_t spl_combine_sample_rows(const spl_combine* c, int64_t sample);
int64_t spl_combine_sample_runs(const spl_combine* c, int64_t sample, const int32_t** runs);
int  spl_combine_merge(spl_combine* c, int64_t n_order, const int32_t* region_order,
                       const char* qgene /* NULL = "All" */, int is_stranded);
/* combineShallow (SpliSER_v0_1_8.py:920-1167): the same merge with the -m/--minSamples, -r/--minReads, -e/--minSSE filters
 * (S:1066-1084, S:1108, S:1154-1160) and, with -g, only that gene's rows loaded (S:947-956); everything after the merge
 * (spl_combine_gaps, spl_recount, spl_combine_set_recount, spl_combine_write) is shared with combine */
int  spl_combine_merge_shallow(spl_combine* c, int64_t n_order, const int32_t* region_order,
                               const char* qgene /* NULL = "All" */, int is_stranded,
                               int64_t min_samples, int64_t min_reads, double min_sse);
int64_t spl_combine_n_sites(const spl_combine* c);     /* merged sites that will be written */
int64_t spl_combine_n_filled(const spl_combine* c);    /* "Filled in Beta read counts for N Sites" (S:917) */
int64_t spl_combine_gaps(const spl_combine* c, int64_t sample, const int32_t** s_region, const int32_t** s_pos,
                         const uint8_t** s_strand, const int64_t** p_off, const int32_t** p_pos,
                         const int64_t** c_off, const int32_t** c_pos);
int  spl_combine_set_recount(spl_combine* c, int64_t sample, int64_t n_gaps, const int64_t* beta1,
                             const int64_t* beta2simple);
int  spl_combine_write(spl_combine* c, const char* path, int cryptic);

/* ---- BAM utilities (used by tests / benchmarks to make synthetic inputs) -------------------- */
/* Writes a coordinate-sorted BAM (BGZF, no index needed by this library) from record arrays;
 * ref_len may be NULL (lengths written as 2^29).  SEQ/QUAL are omitted ('*'). */
int spl_write_bam(const char* path, int32_t n_ref, const char* const* ref_names, const int32_t* ref_len,
                  const spl_records_view* rec /* seg_chrom indexes ref_names */, int n_threads);
/* The same with read names, SEQ and QUAL of the CIGAR's query length (seeded pseudo-random bases, quality strings that change
 * slowly): a sequencer-shaped file -- members of mostly literals, about 10 x the inflated bytes -- for the ingest benchmark. */
int spl_write_bam_seq(const char* path, int32_t n_ref, const char* const* ref_names, const int32_t* ref_len,
                      const spl_records_view* rec, int n_threads);
/* spl_write_bam (with_seq = 0) or spl_write_bam_seq (with_seq != 0) with aux fields: record i (record order of the view) ends
 * with the raw bytes aux[aux_off[i] .. aux_off[i + 1]), written as given (aux_off has n_rec + 1 entries). */
int spl_write_bam_aux(const char* path, int32_t n_ref, const char* const* ref_names, const int32_t* ref_len,
                      const spl_records_view* rec, const int64_t* aux_off, const uint8_t* aux, int with_seq, int n_threads);
/* Decodes a BAM into library-owned record arrays (host only; no GPU needed).  chrom_names maps
 * BAM reference names to caller chromosome indices; records on other references are dropped. */
typedef struct spl_records spl_records;
int spl_read_bam(const char* path, int32_t n_chrom, const char* const* chrom_names, int n_threads,
                 spl_records** out, char* err, int err_len);
/* The same, and the strand of every kept record from its XS tag (SPL_FLAG_XS_STRAND's rule): spl_records_xs. */
int spl_read_bam_xs(const char* path, int32_t n_chrom, const char* const* chrom_names, int n_threads,
                    spl_records** out, char* err, int err_len);
const spl_records_view* spl_records_get(const spl_records* r);
const uint8_t* spl_records_xs(const spl_records* r);      /* [n_rec] '+', '-' or '?'; NULL for a handle of spl_read_bam */
void spl_records_free(spl_records* r);

/* Test hook: the raw-DEFLATE decoder the device runs on every BGZF member (csrc/inflate.h), compiled for the host.
 * Returns 0 and *out_len on success, a positive decoder error code on corrupt input, -1 on NULL arguments. */
int spl_debug_inflate(const uint8_t* src, uint32_t n, uint8_t* dst, uint32_t cap, uint32_t* out_len);

/* Page-locked host memory for callers that want full-speed host->device copies of their record
 * arrays (numpy arrays can be built over it).  Needs a CUDA device. */
void* spl_host_alloc(size_t bytes);
void  spl_host_free(void* p);

#ifdef __cplusplus
}
#endif
#endif /* SPLISER_B200_H */
