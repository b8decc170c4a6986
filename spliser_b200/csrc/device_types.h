// Device-side data layout shared by kernels.cu and pipeline.cu.  See DESIGN.md "Data layout in HBM".
#pragma once
#include <atomic>
#include <cstdint>

#include <vector_types.h>

namespace spl {

// every kernel launch of the library is counted (bench.py reports the launches inside its timed region)
extern std::atomic<unsigned long long> g_kernel_launches;
#define SPL_LAUNCH (++::spl::g_kernel_launches)

#ifndef SPL_BIN_SHIFT
#define SPL_BIN_SHIFT 6
#endif
#ifndef SPL_SB_SHIFT
#define SPL_SB_SHIFT 6
#endif
constexpr int BIN_SHIFT = SPL_BIN_SHIFT;   // 64 bp genomic bins of the block partition (stream C)
constexpr int SB_SHIFT = SPL_SB_SHIFT;     // 64 bp bins of the direct-address site index

// One work tile = up to CHUNK_READS consecutive records of one chromosome.  The expansion kernels
// fill the bases/counts; the bin partition and the junction grouping walk the SoA chunk by chunk.
struct Chunk {
    int32_t  chrom;
    uint32_t rec_lo, rec_hi;            // [rec_lo, rec_hi) records (host-filled)
    uint32_t a_cnt, b_cnt, s_cnt, j_cnt;     // totals (expand pass 1)
    uint32_t a_base, b_base, s_base, j_base; // exclusive scan of the totals
    int32_t  a_lo, a_hi;                // min block start / max (block end - 2) over A blocks (empty: lo > hi)
    int32_t  s_lo, s_hi;                // min / max position any lookup of the chunk's spliced reads can ask for
};

// Work item of the fused counting kernel (count_fused.cu): up to FC_RECS consecutive records of one chromosome.
// The host fills chrom / rec_lo / rec_hi; k_chunk_bounds adds the CIGAR range and the chromosome's site / bin ranges.
constexpr int FC_RECS = 1024;
struct FChunk {
    int32_t  chrom;
    uint32_t rec_lo, rec_hi;            // records [rec_lo, rec_hi)
    uint32_t c_lo, c_hi;                // their CIGAR words [c_lo, c_hi)
    int32_t  s0, s1;                    // site index range of the chromosome
    int32_t  sb_g0, sb_nb;              // direct-address bin index of the chromosome: first entry, number of bins (sentinel at sb_nb)
    int32_t  pad[3];
};
static_assert(sizeof(FChunk) == 48, "FChunk is loaded as three 128-bit words");

struct DevGraph {
    int32_t n_chrom, n_sites, n_edges;
    int32_t own_lo, own_hi;             // site index range this context owns (tile sharding)
    int32_t pt_is_pc;                   // 1: Partners entry a <-> PartnerCounts entry a (clean regime; pt_off == pc_off)
    const int32_t* cs_off;              // [n_chrom+1]
    const int32_t* site_pos;            // [n_sites + 8], tail padded with INT32_MAX
    const uint8_t* site_cls;            // [n_sites]
    const uint8_t* site_hot;            // [n_sites + 32] 1 = some site in the reverse-partner list anchored here has competitors
    // direct-address index of the site table: for chromosome c and bin b = pos >> SB_SHIFT,
    // sb_off[sb_base[c] + b] = first global site index with position >= b << SB_SHIFT (one sentinel per chromosome)
    const int32_t* sb_base;             // [n_chrom+1]
    const int32_t* sb_off;              // [sb_base[n_chrom] + 64]
    const int32_t *pt_off, *pt_site;    // Partners (site indices)
    const int32_t *pc_off, *pc_pos;     // PartnerCounts keys
    const int32_t *cp_off, *cp_pos;     // CompetitorPos (sorted)
    const int32_t *rp_off, *rp_site;    // reverse partner index, anchored at first site of a position
    const int32_t *inc_off, *inc_line;  // alpha reduction segments
    const int32_t *einc_beg, *einc_end, *einc_line;   // PartnerCounts reduction segments [einc_beg[e], einc_end[e])
    const int64_t* j_score;             // junction scores (device copy)
};

struct DevRecords {
    uint32_t n_rec;
    const int32_t*  pos;                // 1-based
    const uint16_t* flag;
    const uint32_t* cig_off;            // [n_rec+1]
    const uint32_t* cigar;              // BAM-encoded ops
};

// Structure-of-arrays the counting kernels stream.  Positions are < 2^31, so bit 31 of the second
// word of every element carries the read's strand class (0 = '+' / unstranded, 1 = '-'):
//   blocks     (start, end | class<<31)            [start, end) of one M/=/X operator
//   junctions  (l | firstN<<31, r | class<<31)     l = last base before the N, r = last base of the N;
//                                                  firstN marks an N that starts at POS (l = POS - 1: nothing before it
//                                                  moved the position, zero-length operators included)
// Blocks of unspliced reads (stream A, sorted by start) come first, blocks of spliced reads (stream B,
// contiguous per read) follow in the same arrays.
struct DevSoA {
    uint32_t nA, nB, nS, nJ;
    int32_t* m_start; uint32_t* m_endk;                 // [nA + nB] (+ padding); B stream starts at index bB
    uint32_t bB;                                        // first element of stream B (multiple of 4)
    uint32_t* sr_boff; uint32_t* sr_joff;               // [nS+1] per spliced read: offsets into stream B / junctions
    uint32_t* jn_l; uint32_t* jn_rk;                    // [nJ]
    uint32_t* jn_read;                                  // [nJ] owning spliced read | simple<<31
    int32_t*  ji_a0; int32_t* ji_end;                   // [nJ] first block start / last block end of the owning read (simple reads)
};
constexpr uint32_t POS_MASK = 0x7fffffffu;

// Bin-partitioned copy of all M blocks (stream C): blocks grouped by (chromosome, start >> BIN_SHIFT), order
// inside a bin arbitrary.  K3 streams it in fixed tiles; every warp then sees a tiny genomic window whatever
// the record order or the intron lengths were.  Each chromosome is padded to a multiple of K3_TILE with
// never-matching elements so that tiles do not straddle chromosomes.
constexpr int K3_TILE = 2048;           // blocks per tile / pipeline stage (16 KB)
// Junction groups: every distinct (chromosome, l, r, class) junction of the sample with its multiplicity,
// built once at load time (open-addressing table, one power-of-two sub-table per chromosome, then compacted).
// A "simple" instance belongs to a read that is exactly block-N-block (no other N, no D, no I-split): for those
// the exception logic only needs the read's first block start and last block end, kept grouped per junction.
struct DevJunc {
    // load-time table
    uint32_t  n_slots;
    uint32_t* chrom_jn;           // [n_chrom]   junction instances per chromosome
    uint32_t* tab_base;           // [n_chrom+1] first slot of each chromosome's sub-table
    unsigned long long* key;      // [n_slots]   ~(l | rk << 32), 0 = empty
    uint32_t* s_all; uint32_t* s_simple;        // [n_slots] instance counts
    uint32_t* s_used; uint32_t* s_off;          // [n_slots+1] scans: dense id, offset of the group's simple instances
    uint32_t* s_coff;             // [n_slots+1] scan: offset of the group's complex instances
    uint32_t* s_cursor; uint32_t* s_ccur;       // [n_slots] scatter cursors (simple / complex)
    uint32_t* slot_of;            // [nJ] slot of each instance
    uint32_t* overflow;           // [1] a sub-table filled up (never with the sizes chosen; checked anyway); follows cx_n
    uint32_t* scan_tmp;           // block sums of the scans
    // dense distinct-junction table
    uint32_t  D;
    uint32_t* dj_l; uint32_t* dj_rk; int32_t* dj_chrom;
    uint32_t* dj_all; uint32_t* dj_simple; uint32_t* dj_off;
    int32_t*  gi_a0; int32_t* gi_end;           // simple instances grouped by junction
    uint32_t  n_complex;
    uint32_t* dj_coff;            // [D] offset of the junction's complex instances in cx_j
    uint32_t* cx_j; uint32_t* cx_n;             // complex instances grouped by junction: global junction index; cx_n: scratch word before `overflow`
    uint4*    cx_rng;             // [n_complex] the owning read of each complex instance: junctions [x, y), blocks [z, w) (absolute indices)
    // per (sample, site table): filled by k_junc_lookup after the graph is on the device
    uint32_t* hot_l; uint32_t* hot_r;           // [D] anchor + 1 of a hot endpoint, 0 otherwise
    uint32_t* sp_x0; uint32_t* sp_x1;           // [D] offsets into cnt.span of the junction's +n / -n (sp_x1 = ~0: no site strictly inside)
    uint32_t* cx_pack;                          // [flat hot complex instances * 24] packed reads (k_junc_pack), sized after k_junc_lookup
    uint32_t* prep;                             // [8] [2] simple work-list length, [4..5] one u64: complex descriptors << 40 | flat instances
    unsigned long long* wl;       // hot units: chunk << 32 | junction << 1 | side
    uint32_t* cxd_base; uint32_t* cxd_ds;       // [2 D] per pass: descriptors of hot (junction, side) with complex instances: first flat index, d << 1 | side
    uint32_t* cxd_nt; int32_t* cxd_t;           // [2 D], [2 D * CXD_T] sites the (junction, side) is a partner/competitor pair for
};

constexpr int CXD_T = 4;          // pair sites kept inline per descriptor

struct Tile { uint32_t e0; int32_t w_lo, w_hi; int32_t pad; };   // first element, site index window [w_lo, w_hi)
struct DevBins {
    uint32_t* chrom_ext;        // [n_chrom]   largest block start seen (atomicMax)
    uint32_t* chrom_tot;        // [n_chrom]   blocks on the chromosome
    uint32_t* chrom_jn;         // [n_chrom]   junction instances on the chromosome
    uint32_t* tab_base;         // [n_chrom+1] junction sub-table layout (see DevJunc)
    uint32_t* chrom_bin_base;   // [n_chrom+1] first bin of each chromosome
    uint32_t* chrom_tile_base;  // [n_chrom+1] first tile of each chromosome
    uint32_t* max_len;          // [1]         longest block
    uint32_t* bin_off;          // [total_bins+1] counts, then exclusive offsets
    uint32_t* bin_cursor;       // [total_bins]
    uint32_t* scan_tmp;         // block sums of the scan
    int32_t*  c_start; uint32_t* c_endk;   // [nC]
    Tile*     tiles;            // [n_tiles]
    uint32_t  total_bins, n_tiles, nC;
    int32_t   n_chrom;
};

// Per-pass counters, one contiguous u32 buffer (zeroed by one memset per pass).
// diff: four difference arrays in site-index space, interleaved per site (one 16-byte element per site):
//   word 4*s + k      reads of strand class k whose M/=/X block covers site s and s+1 (S:469)
//   word 4*s + 2 + k  reads of strand class k whose N strictly spans site s (S:507-512)
// An operator that stabs the site index range [lo, hi) adds +1 at lo and -1 at hi; k_finalize takes the prefix sums.
struct DevCounters {
    uint32_t* diff;    // [(S+1) * 4]
    uint32_t* dir;     // [S * 4]   same four kinds, counted directly per site (fused kernel, groups with a narrow site window)
    uint32_t* cov;     // [2][S]   direct coverage counts by read strand class (stabbing variant K3 only; zero otherwise)
    uint32_t* covx;    // [S] covering reads that are beta1-type (moved from beta1 to beta2Simple)
    uint32_t* spanx;   // [S] spanning reads that are flanking (removed from the mutually-exclusive count)
    uint32_t* flank;   // [S] flanking reads (counted as beta2Simple in combine mode only)
    uint32_t* dc;      // [E] PartnerBeta2DoubleCounts increments seen in the BAM
    uint32_t* work;    // [16] work-item counters: [0] K3 tiles, [8 + p] chunks of upload part p (fused kernel)
};

struct DevOutputs {
    int64_t* alpha; int64_t* pc_cnt;    // [S], [E]
    int64_t* beta1; int64_t* beta2s; int64_t* beta2c;
    double* beta2w; double* sse;
    int64_t* dc_tot; uint8_t* dc_present;   // [E] scratch of the beta2 gather
    uint32_t* span_blk;                 // [4 per block] block sums of the four difference arrays
};

constexpr int CHUNK_READS = 4096;       // records per chunk
constexpr int EXPAND_THREADS = 512;     // one record per thread and round
constexpr int FIN_THREADS = 256;        // sites per block of the difference-array scan (one site per thread: the beta2 gather wants that)

constexpr uint32_t FLAG_STRANDED = 1u, FLAG_RF = 2u, FLAG_CRYPTIC = 4u, FLAG_COMBINE = 8u;
#ifdef SPL_DEBUG_HOOKS
constexpr uint32_t FLAG_DEBUG_SKIP_EXC = 0x10000u;   // kernel timing experiments only: compiled in with -DSPL_DEBUG_HOOKS, never in the shipped library
#else
constexpr uint32_t FLAG_DEBUG_SKIP_EXC = 0u;
#endif

struct KernelTimes { float beta1_ms, spliced_ms, final_ms; };

// launchers (kernels.cu); all asynchronous on `stream`
void launch_expand_count(const DevRecords& rec, Chunk* chunks, int n_chunks, uint32_t flags, DevBins bins, void* stream);
void launch_chunk_scan(Chunk* chunks, int n_chunks, uint32_t* totals8, DevBins bins, void* stream);
void launch_bin_partition(const Chunk* chunks, int n_chunks, DevSoA soa, DevBins bins, void* stream);
void launch_tile_hints(DevBins bins, DevGraph g, void* stream);
void launch_expand_scatter(const DevRecords& rec, const Chunk* chunks, int n_chunks, DevSoA soa, uint32_t flags, void* stream);
void launch_beta1(DevBins bins, DevGraph g, DevCounters cnt, void* stream);
void launch_jtab_layout(DevBins bins, int attempt, uint32_t* totals8, void* stream);
void launch_junction_groups_a(const Chunk* chunks, int n_chunks, DevSoA soa, DevJunc jg, uint32_t* totals4, void* stream);
void launch_junction_groups_b(DevSoA soa, DevJunc jg, int n_chrom, uint32_t* totals4, void* stream);
void launch_junction_prepare(DevJunc jg, DevGraph g, uint32_t flags, void* stream);
void launch_junction_pack(DevSoA soa, DevJunc jg, void* stream);
void launch_junctions(DevSoA soa, DevJunc jg, DevGraph g, DevCounters cnt, uint32_t flags, void* stream);
void launch_finalize(DevGraph g, DevCounters cnt, DevOutputs out, uint32_t flags, void* stream);
int  kernel_launch_count_per_pass();
void launch_exscan_u32(uint32_t* a, uint32_t n, uint32_t* tmp, uint32_t* total_out, void* stream);
uint32_t exscan_tmp_words(uint32_t n);
// fused difference-array variant (count_fused.cu)
void launch_chunk_bounds(FChunk* chunks, uint32_t lo, uint32_t hi, const uint32_t* cig_off, DevGraph g, void* stream);
void launch_count_fused(const DevRecords& rec, const FChunk* chunks, uint32_t lo, uint32_t hi, DevGraph g, DevCounters cnt,
                        uint32_t* work, uint32_t flags, uint4* hotq, uint32_t* hot_n, uint32_t hot_cap, void* stream);
void launch_hot_items(const DevRecords& rec, DevGraph g, DevCounters cnt, uint32_t flags, const uint4* hotq, const uint32_t* hot_n,
                      uint32_t hot_cap, void* stream);
uint32_t unpack_desc_words(uint32_t n_rec);
void launch_unpack_records(const uint16_t* n_op, const uint8_t* flag8, uint32_t r0, uint32_t r1, uint32_t cig_base, uint32_t* cig_off,
                           uint16_t* flag16, unsigned long long* desc, uint32_t* ticket, uint32_t epoch, void* stream);
void launch_unpack_compact(const uint16_t* pos16, const uint8_t* flag8, const uint8_t* n_op8, const uint16_t* c16, const uint32_t* c32,
                           const int32_t* pos_base, const int32_t* pos_wide, const uint32_t* idx16, const uint32_t* idx32, uint32_t r0,
                           uint32_t r1, int32_t* pos, uint16_t* flag16, uint32_t* cig_off, uint32_t* cigar, uint32_t* bad, void* stream);
int  sm_count_current_device();

}  // namespace spl
