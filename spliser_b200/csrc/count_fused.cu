// Fused counting kernel: alignment records resident in HBM -> per-site counters, one pass, nothing materialised.
//
// Replaces processSites -> checkBam per site (SpliSER_v0_1_8.py:681-692, :408-559) by one traversal of the records.
// This is the difference-array / prefix-scan formulation of the stabbing count: every advancing CIGAR operator [cur, cur+len)
// of type M/=/X (S:457-459, :469) or N (S:480-483, :507-512) stabs the sites with position in [cur, cur+len-2], i.e. the
// contiguous site index range [lb(cur), lb(cur+len-1)) of the sorted site table.  The range gets +1 / -1 in the class's
// difference array (cnt.diff, cov words for M, span words for N); k_finalize takes the prefix sums.  The stabbing
// variant (k_beta1_stab in kernels.cu, streaming a bin-partitioned copy of the blocks) is kept for the cross-check.
//
// Layout of the kernel: persistent CTAs (2 per SM), one producer warp + 15 consumer warps (512 threads: with 64 registers each, two CTAs fill the register file).
//   producer  claims chunks of <= FC_RECS records from a global counter and stages their pos / flag / cig_off / CIGAR
//             slices into a 3-stage shared-memory ring with 1-D TMA bulk copies (cp.async.bulk + mbarrier);
//   consumers one record per lane.  A lane walks its CIGAR from shared memory and carries the site index of its
//             current reference position along (one lookup through the direct-address bin index per read or long
//             jump, short walks over the L1-resident site table otherwise).  Lanes run their operators in lock step, so
//             that equal (index, class, kind) targets of neighbouring lanes -- coordinate-sorted reads hit the same
//             few sites -- merge into one RED per run.
//   A junction endpoint that sits on a "hot" site (an anchor whose reverse-partner list has competitors) may make
//   compSplicing true for some site (S:494-501): the (record, operator, side) goes to the warp's shared-memory list and
//   is classified after the warp's records of the chunk, all lanes busy, from the CIGAR still staged (S:503-557).
#include <cuda_runtime.h>

#include <climits>
#include <cstdint>
#include <mutex>

#include "../../include/spliser_b200.h"
#include "dev_helpers.cuh"
#include "device_types.h"

namespace spl {

namespace {

constexpr int FC_STAGES = 3;
#ifndef SPL_FC_CWARPS
#define SPL_FC_CWARPS 15
#endif
constexpr int FC_CWARPS = SPL_FC_CWARPS;
constexpr int FC_CONSUMERS = FC_CWARPS * 32;
constexpr int FC_THREADS = FC_CONSUMERS + 32;
constexpr int FC_RPAD = 16;                 // slack for the 16-byte alignment of the staged record slices
constexpr int FC_CIG = 4096;                // staged CIGAR words per stage (a chunk with more reads them from global memory)
constexpr int FC_LIST = 160;                // hot items per warp list
constexpr int FC_BATCH = 2;                 // chunks a producer claims per atomic
constexpr int FC_WALK = 256;                // operators longer than this jump through the bin index instead of walking
constexpr int FC_MAXJ = 4, FC_MAXB = 6;     // junctions / blocks of a read kept in registers by the exception path

constexpr uint32_t FM_DONE = 1u, FM_GLOBAL_CIG = 2u;

struct FStage {
    int32_t  pos[FC_RECS + FC_RPAD];
    uint32_t off[FC_RECS + FC_RPAD];
    uint32_t cig[FC_CIG + 8];
    uint16_t flag[FC_RECS + FC_RPAD];
};
static_assert(sizeof(FStage) % 16 == 0 && ((FC_RECS + FC_RPAD) * 4) % 16 == 0 && ((FC_CIG + 8) * 4) % 16 == 0, "TMA destinations are 16-byte aligned");

struct FMeta {
    uint32_t flags, n_rec, skip, cig_base;  // skip: staged index of the chunk's first record; cig_base: absolute index of staged word 0
    uint32_t rec_lo;                        // absolute index of the chunk's first record
    int32_t  chrom, s0, s1, sb_g0, sb_nb;
};

struct FSmem {
    uint4 lut[32];                      // operator table, entry 2 * code + strand class: {advance mask, field of the warp's sum, counted mask, is N}
                                        // (first member: 512-byte aligned, so that an entry's address is base | code << 5 | class << 4)
    FStage st[FC_STAGES];
    unsigned long long list[FC_CWARPS][FC_LIST];
    uint32_t lother[FC_CWARPS][FC_LIST];  // the junction's other end (position) of every list entry
    FMeta meta[FC_STAGES];
    uint32_t next_group[FC_STAGES];     // next record of the staged chunk (the consumer warps take 32 at a time)
    uint64_t full[FC_STAGES], empty[FC_STAGES];
};

struct FArgs {
    DevRecords rec;
    const FChunk* chunks;
    uint32_t chunk_lo, chunk_hi;
    DevGraph g;
    DevCounters cnt;
    uint32_t* work;
    uint32_t mode;
    uint4* hotq;             // global queue of hot (record, operator, side) items: {anchor, record, operator | side << 31, position of the junction's other end}
    uint32_t* hot_n;         // [0] items written (may exceed hot_cap: the excess was dropped and the pass must be repeated with room)
    uint32_t hot_cap;
};

// +n on word `key` of the difference arrays for every run of neighbouring lanes with the same key (v: the lane takes part)
__device__ __forceinline__ void run_add(uint32_t* base, uint32_t key, bool v, bool neg, int lane) {
    const uint32_t kk = v ? key : 0xffffffffu;
    const uint32_t prev = __shfl_up_sync(0xffffffffu, kk, 1);
    const bool head = lane == 0 || kk != prev;
    const uint32_t heads = __ballot_sync(0xffffffffu, head);
    if (head && v) {
        const uint32_t after = heads & ~((2u << lane) - 1u);           // heads above this lane
        const uint32_t n = (uint32_t)((after ? __ffs(after) - 1 : 32) - lane);
        atomicAdd(base + key, neg ? 0u - n : n);
    }
}

// plain RED for lanes with distinct addresses (the compiler wraps atomicAdd in a warp-aggregation sequence of a dozen instructions)
__device__ __forceinline__ void red_add64(unsigned long long* p, unsigned long long v) {
    asm volatile("red.global.add.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}

// the staged (or, for oversized chunks, global) CIGAR words of a chunk
template <bool STAGED>
struct CigSrc {
    const uint32_t* p;       // STAGED: stage array, indexed by (absolute index - base); else the global array
    uint32_t base;
    __device__ __forceinline__ uint32_t operator()(uint32_t c) const { return STAGED ? p[c - base] : __ldg(p + c); }
};

// first site index >= the caller's lower bound `from` with position >= pos, through the chromosome's bin index
__device__ __forceinline__ int bin_lower(const DevGraph& g, const FMeta& m, int32_t pos, int from) {
    int i = __ldg(g.sb_off + m.sb_g0 + min(max(pos, 0) >> SB_SHIFT, m.sb_nb));
    i = max(i, from);
    while (i < m.s1 && __ldg(g.site_pos + i) < pos) ++i;
    return i;
}

// ---- exception path -----------------------------------------------------------------------------
struct ReadRegs {            // a read with <= FC_MAXJ junctions and <= FC_MAXB blocks
    uint32_t jlv[FC_MAXJ], jrv[FC_MAXJ];
    int32_t bsv[FC_MAXB]; uint32_t bev[FC_MAXB];
    uint32_t nj, nb, jrel;
    __device__ __forceinline__ uint32_t jl(uint32_t x) const { return jlv[x]; }
    __device__ __forceinline__ uint32_t jr(uint32_t x) const { return jrv[x]; }
    __device__ __forceinline__ int32_t bs(uint32_t x) const { return bsv[x]; }
    __device__ __forceinline__ uint32_t be(uint32_t x) const { return bev[x]; }
};
template <bool STAGED>
struct ReadWalk {            // any read: every access walks the CIGAR again (long reads only)
    CigSrc<STAGED> cw;
    uint32_t c0, nop;
    int32_t pos;
    uint32_t nj, nb, jrel;
    // x-th operator of the wanted kind (N or mapped): start position, end position, "it starts at POS"
    __device__ __forceinline__ void find(bool want_n, uint32_t x, int32_t& a, int32_t& b, bool& at_pos) const {
        int32_t cur = pos; uint32_t cnt = 0;
        a = b = 0; at_pos = false;
        for (uint32_t q = 0; q < nop; ++q) {
            const uint32_t w = cw(c0 + q), op = w & 15u;
            const int32_t len = (int32_t)(w >> 4);
            const bool isM = op == 0u || op == 7u || op == 8u, isN = op == 3u;
            if ((want_n && isN) || (!want_n && isM)) {
                if (cnt == x) { a = cur; b = cur + len; at_pos = cur == pos; return; }
                ++cnt;
            }
            if (isM || isN || op == 2u) cur += len;
        }
    }
    __device__ __forceinline__ uint32_t jl(uint32_t x) const { int32_t a, b; bool s; find(true, x, a, b, s); return (uint32_t)(a - 1) | (s ? 0x80000000u : 0u); }
    __device__ __forceinline__ uint32_t jr(uint32_t x) const { int32_t a, b; bool s; find(true, x, a, b, s); return (uint32_t)(b - 1); }
    __device__ __forceinline__ int32_t bs(uint32_t x) const { int32_t a, b; bool s; find(false, x, a, b, s); return a; }
    __device__ __forceinline__ uint32_t be(uint32_t x) const { int32_t a, b; bool s; find(false, x, a, b, s); return (uint32_t)b; }
};

// one hot (record, operator, side): find the sites the junction is a partner/competitor pair for and classify the read there
// (S:494-557).  Runs in k_hot_items, one thread per queued item, from the record arrays in global memory.
__device__ __forceinline__ void hot_item(const DevRecords& rec, const DevGraph& g, const DevCounters& cnt, uint32_t mode, uint4 it) {
    const int anchor = (int)it.x;
    const uint32_t ri = it.y, side = it.z >> 31, j = it.z & 0x7fffffffu;
    // the junction: the anchored end sits on the anchor's position, the item carries the other one.  Most items end here: the
    // anchor is hot because SOME junction through it is a partner/competitor pair for a site -- this one only if its other end
    // is a competitor of a site of the anchor's reverse-partner list (graph lookups only, no record is touched)
    const int32_t ap = __ldg(g.site_pos + anchor), other = (int32_t)it.w;
    const int32_t jl = side == 0u ? ap : other, jr = side == 0u ? other : ap;
    const int q0 = g.rp_off[anchor], q1 = g.rp_off[anchor + 1];
    int first = -1;
    for (int q = q0; q < q1 && first < 0; ++q)
        if (k4_pair_site(g, q, (int)side, jl, jr) >= 0) first = q;
    if (first < 0) return;
    const int32_t pos = __ldg(rec.pos + ri);
    const uint32_t c0 = __ldg(rec.cig_off + ri), nop = __ldg(rec.cig_off + ri + 1) - c0;
    const uint32_t k = read_class(__ldg(rec.flag + ri), mode);
    const bool combine = (mode & FLAG_COMBINE) != 0;
    const CigSrc<false> cw{rec.cigar, 0u};
    ReadRegs rr;
    rr.nj = rr.nb = rr.jrel = 0;
    int32_t cur = pos;
    for (uint32_t q = 0; q < nop; ++q) {
        const uint32_t w = cw(c0 + q), op = w & 15u;
        const int32_t len = (int32_t)(w >> 4);
        if (op == 0u || op == 7u || op == 8u) {
            if (rr.nb < (uint32_t)FC_MAXB) { rr.bsv[rr.nb] = cur; rr.bev[rr.nb] = (uint32_t)(cur + len); }
            ++rr.nb; cur += len;
        } else if (op == 3u) {
            if (q == j) rr.jrel = rr.nj;
            if (rr.nj < (uint32_t)FC_MAXJ) { rr.jlv[rr.nj] = (uint32_t)(cur - 1) | (cur == pos ? 0x80000000u : 0u); rr.jrv[rr.nj] = (uint32_t)(cur + len - 1); }
            ++rr.nj; cur += len;
        } else if (op == 2u) {
            cur += len;
        }
    }
    if (rr.nj <= (uint32_t)FC_MAXJ && rr.nb <= (uint32_t)FC_MAXB) {
        for (int q = first; q < q1; ++q) {
            const int t = k4_pair_site(g, q, (int)side, jl, jr);
            if (t >= 0) k4_classify(rr, g, cnt, t, k, combine, 1u);
        }
    } else {
        const ReadWalk<false> rw{cw, c0, nop, pos, rr.nj, rr.nb, rr.jrel};
        for (int q = first; q < q1; ++q) {
            const int t = k4_pair_site(g, q, (int)side, jl, jr);
            if (t >= 0) k4_classify(rw, g, cnt, t, k, combine, 1u);
        }
    }
}

__global__ void __launch_bounds__(256) k_hot_items(DevRecords rec, DevGraph g, DevCounters cnt, uint32_t mode, const uint4* __restrict__ hotq,
                                                   const uint32_t* __restrict__ hot_n, uint32_t hot_cap) {
    const uint32_t n = min(*hot_n, hot_cap);
    for (uint32_t x = blockIdx.x * blockDim.x + threadIdx.x; x < n; x += gridDim.x * blockDim.x) hot_item(rec, g, cnt, mode, hotq[x]);
}

// the warp's list goes to the global queue: one reservation per flush
__device__ __forceinline__ void flush_list(const unsigned long long* list, const uint32_t* lother, uint32_t list_n, uint32_t rec_lo, const FArgs& A, int lane) {
    __syncwarp();
    uint32_t base = 0;
    if (lane == 0) base = atomicAdd(A.hot_n, list_n);
    base = __shfl_sync(0xffffffffu, base, 0);
    for (uint32_t x = (uint32_t)lane; x < list_n; x += 32) {
        const unsigned long long it = list[x];
        const uint32_t lo = (uint32_t)it;
        if (base + x < A.hot_cap) A.hotq[base + x] = make_uint4((uint32_t)(it >> 32), rec_lo + (lo >> 21), (lo & 0xfffffu) | (((lo >> 20) & 1u) << 31), lother[x]);
    }
    __syncwarp();
}

// hot endpoints of this step go to the warp's list: hl / hr = anchor + 1 of the junction's left / right end (0: not hot);
// pl / pr = the junction's l / r (each entry carries the end that is NOT on its anchor)
__device__ __forceinline__ void push_hot(unsigned long long* list, uint32_t* lother, uint32_t& list_n, uint32_t hl, uint32_t hr, int32_t pl, int32_t pr,
                                         uint32_t i, uint32_t j, int lane) {
    const uint32_t pm_l = __ballot_sync(0xffffffffu, hl != 0u), pm_r = __ballot_sync(0xffffffffu, hr != 0u);
    if (pm_l | pm_r) {
        const uint32_t lt = (1u << lane) - 1u;
        const uint32_t tag = (i << 21) | (j & 0xfffffu);
        if (hl) { const uint32_t x = list_n + __popc(pm_l & lt); list[x] = ((unsigned long long)(hl - 1u) << 32) | tag; lother[x] = (uint32_t)pr; }
        if (hr) { const uint32_t x = list_n + __popc(pm_l) + __popc(pm_r & lt); list[x] = ((unsigned long long)(hr - 1u) << 32) | tag | (1u << 20); lother[x] = (uint32_t)pl; }
        list_n += (uint32_t)(__popc(pm_l) + __popc(pm_r));
    }
}

// ---- the records of one staged chunk ---------------------------------------------------------------
// Groups of 32 consecutive records are handed out dynamically (shared-memory counter of the stage): a warp that is held up
// does not hold the stage.  Per group, two ways to the same counts:
//   stab   the group's reads are coordinate-sorted neighbours, so their first FC_SLOTS operators cover a window of a few
//          sites.  The window's site range is found once per warp; every site is then tested against each lane's operators
//          from registers ((uint32)(p - start) < len - 1, S:469 / S:507) and the per-kind, per-class hits of the warp are
//          summed with one redux.sync -> direct counts (cnt.dir), one RED per (warp, site, kind).  A hot site also checks
//          the lanes' junction ends against its position.
//   chain  wide windows (long introns next to dense sites, unsorted input) and operators beyond the first FC_SLOTS: the lane
//          carries the site index of its reference position along its CIGAR and adds +1 / -1 at the two ends of the stabbed
//          index range in the difference arrays (cnt.diff), runs of equal targets in neighbouring lanes merged.
constexpr int FC_SLOTS = 5;
#ifndef SPL_FC_STAB_MAX
#define SPL_FC_STAB_MAX 16
#endif
constexpr int FC_STAB_MAX = SPL_FC_STAB_MAX;
static_assert(FC_STAB_MAX < 32, "the anchor loop masks the window's sites with (1 << nw) - 1");

template <bool STAGED>
__device__ __forceinline__ void consume(const FStage& st, const FMeta& m, unsigned long long* list, uint32_t* lother, uint32_t* next_group, uint32_t lut_base, const FArgs& A) {
    const int lane = threadIdx.x & 31;
    const DevGraph& g = A.g;
    const CigSrc<STAGED> cw{STAGED ? st.cig : A.rec.cigar, STAGED ? m.cig_base : 0u};
    const int32_t* __restrict__ sp = g.site_pos;
    const uint8_t* __restrict__ hot = g.site_hot;
    const int s0 = m.s0, s1 = m.s1, own_lo = g.own_lo, own_hi = g.own_hi;
    uint32_t list_n = 0;                                             // warp-uniform
    for (;;) {
        // a group pushes at most 4 entries per lane on the stab path (two junctions in FC_SLOTS operators)
        if (list_n > (uint32_t)(FC_LIST - 128)) { flush_list(list, lother, list_n, m.rec_lo, A, lane); list_n = 0; }
        // every lane takes a record number from the stage's counter: ptxas turns the warp's 32 increments of one address into a single
        // ATOMS of +32 and hands the lanes consecutive numbers (nothing below needs more than "each record exactly once")
        const uint32_t i = atomicAdd(next_group, 1u);
        const bool live = i < m.n_rec;
        if (!__any_sync(0xffffffffu, live)) break;
        int32_t pos = 0;
        uint32_t nop = 0, k = 0;
        // ---- the first FC_SLOTS operators in registers: operator j covers [b[j], b[j+1]); a site at p is stabbed by it
        // (covered, S:469 / strictly inside the junction, S:507) iff (uint32)(p - b[j]) < len1[j] with len1 = length - 1 for
        // M/=/X/N operators and 0 otherwise; wf[j] is the operator's field of the warp's sum (cov / span x strand class)
        int32_t b[FC_SLOTS + 1];
        uint32_t len1[FC_SLOTS], wf[FC_SLOTS];
        uint32_t tN = 0;                                             // bit j: operator j is N (S:480-483)
        uint32_t zl = 0;                                             // bit 31: a zero-length M / N (left to the chain path, like more than two N)
        {
            uint32_t c0 = 0;
            if (live) {
                pos = st.pos[m.skip + i];
                c0 = st.off[m.skip + i];
                nop = st.off[m.skip + i + 1] - c0;
                k = read_class(st.flag[m.skip + i], A.mode);
            }
            b[0] = pos;
            const uint32_t lut_k = lut_base | (k << 4);             // shared-memory address of this strand class's entries
#pragma unroll
            for (int j = 0; j < FC_SLOTS; ++j) {                     // (no test against the group's longest read: nearly every group has one with FC_SLOTS operators)
                const uint32_t cwd = (uint32_t)j < nop ? cw(c0 + j) : 5u;      // filler: a zero-length H (no progression)
                uint4 e;                                             // what the operator code means (S:457-464, :480-483), looked up instead of computed
                asm("ld.shared.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(e.x), "=r"(e.y), "=r"(e.z), "=r"(e.w) : "r"(lut_k | ((cwd << 5) & 0x1e0u)));
                const uint32_t len = cwd >> 4;
                b[j + 1] = b[j] + (int32_t)(len & e.x);
                len1[j] = (len - 1u) & e.z;                          // length 1 stabs nothing; length 0 sets bit 31 (-> chain path)
                zl |= len1[j];
                wf[j] = e.y;
                tN += e.w << j;
            }
        }
        const bool odd = (zl >> 31) != 0u || __popc(tN) > 2;
        const bool has = live && nop != 0u;
        const int32_t wlo = __reduce_min_sync(0xffffffffu, has ? pos - 1 : INT_MAX);
        const int32_t whi = __reduce_max_sync(0xffffffffu, has ? b[FC_SLOTS] - 1 : INT_MIN);
        if (wlo > whi) continue;                                     // nothing aligned in this group
        // ---- the window's sites: one coalesced load of the 32 sites from the window's bin on, the rest by ballot
        const int ib = max(__ldg(g.sb_off + m.sb_g0 + min(max(wlo, 0) >> SB_SHIFT, m.sb_nb)), s0);
        const int32_t v = ib + lane < s1 ? __ldg(sp + ib + lane) : INT_MAX;
        const uint32_t hotv = ib + lane < s1 ? (uint32_t)__ldg(hot + ib + lane) : 0u;
        const int d = __popc(__ballot_sync(0xffffffffu, v < wlo));   // loaded sites in front of the window
        const int nw = __popc(__ballot_sync(0xffffffffu, v >= wlo && v <= whi));
        const uint32_t hotmask = __ballot_sync(0xffffffffu, hotv != 0u);
        const bool wide = __any_sync(0xffffffffu, odd) || d + nw >= 32 || nw > FC_STAB_MAX;
        uint32_t j0 = 0;                                             // first operator left to the chain path
        bool act = has;
        int32_t cur = pos;
        if (!wide) {
            uint32_t mine = 0;                                       // lane q keeps the warp's sums for the q-th site of the window
#pragma unroll 2
            for (int q = 0; q < nw; ++q) {                           // warp-uniform
                const int32_t p = __shfl_sync(0xffffffffu, v, d + q);
                uint32_t c = 0;                                      // the operators are disjoint: at most one of them is hit
#pragma unroll
                for (int j = 0; j < FC_SLOTS; ++j)
                    asm("{\n\t.reg .pred hit;\n\tsetp.lt.u32 hit, %1, %2;\n\t@hit add.u32 %0, %0, %3;\n\t}" : "+r"(c) : "r"((uint32_t)(p - b[j])), "r"(len1[j]), "r"(wf[j]));
                c = __reduce_add_sync(0xffffffffu, c);
                if (lane == q) mine = c;
            }
            // anchors in the window: junction ends of the lanes that sit on them (S:494-501)
            for (uint32_t hs = (hotmask >> d) & ((1u << nw) - 1u); hs; hs &= hs - 1u) {      // warp-uniform; nw <= FC_STAB_MAX < 32
                const int q = __ffs(hs) - 1;
                const int32_t p1 = __shfl_sync(0xffffffffu, v, d + q) + 1;
                const int s = ib + d + q;
                uint32_t hl = 0, hr = 0, jl = 0, jr = 0;
                int32_t ol = 0, orr = 0;                              // the other end of the junction whose left / right end sits here
#pragma unroll
                for (int j = 0; j < FC_SLOTS; ++j) {
                    if ((tN >> j) & 1u) {
                        if (p1 == b[j]) { hl = (uint32_t)s + 1u; jl = (uint32_t)j; ol = b[j + 1] - 1; }        // l = start - 1 (S:482)
                        if (p1 == b[j + 1]) { hr = (uint32_t)s + 1u; jr = (uint32_t)j; orr = b[j] - 1; }       // r = end - 1 (S:483)
                    }
                }
                // one list entry carries one operator index: the two ends of a lane at this site belong to different operators
                if (__any_sync(0xffffffffu, (hl | hr) != 0u)) {
                    push_hot(list, lother, list_n, hl, 0u, 0, ol, i, jl, lane);
                    push_hot(list, lother, list_n, 0u, hr, orr, 0, i, jr, lane);
                }
            }
            // one lane per site of the window adds the warp's sums to the direct counters: two 64-bit REDs, each the two strand
            // classes of a kind (the 32-bit halves cannot carry into each other: a counter never exceeds the record count)
            const int sm_ = ib + d + lane;
            if (mine && lane < nw && sm_ >= own_lo && sm_ < own_hi) {
                unsigned long long* dst = reinterpret_cast<unsigned long long*>(A.cnt.dir + 4 * sm_);
                if (mine & 0xffffu) red_add64(dst, (unsigned long long)(mine & 0xffu) | ((unsigned long long)((mine >> 8) & 0xffu) << 32));
                if (mine >> 16) red_add64(dst + 1, (unsigned long long)((mine >> 16) & 0xffu) | ((unsigned long long)(mine >> 24) << 32));
            }
            j0 = FC_SLOTS;
            act = live && nop > (uint32_t)FC_SLOTS;
            cur = b[FC_SLOTS];
        }
        if (!__any_sync(0xffffffffu, act)) continue;
        // ---- chain path: operators [j0, nop) of the active lanes in lock step
        const uint32_t c0 = live ? st.off[m.skip + i] : 0u;
        const uint32_t rem = act ? nop - j0 : 0u;
        const uint32_t maxrem = __reduce_max_sync(0xffffffffu, rem);
        int idx = act ? bin_lower(g, m, cur, s0) : s0;               // first site with position >= cur, carried along the read
        for (uint32_t t = 0; t < maxrem; ++t) {
            if (list_n > (uint32_t)(FC_LIST - 64)) { flush_list(list, lother, list_n, m.rec_lo, A, lane); list_n = 0; }
            const uint32_t j = j0 + t;
            const uint32_t w = t < rem ? cw(c0 + j) : 5u;
            const uint32_t op = w & 15u;
            const int32_t len = (int32_t)(w >> 4);
            const bool isM = (0x181u >> op) & 1u;
            const bool isN = op == 3u;
            const bool adv = (0x18du >> op) & 1u;
            int ie = idx, inx = idx;
            bool v = false;
            uint32_t key_lo = 0, key_hi = 0, hl = 0, hr = 0;
            if (adv && len > 0) {
                const int32_t e = cur + len - 1;                      // last base of the operator
                if (len > FC_WALK) ie = bin_lower(g, m, e, idx);
                while (ie < s1 && __ldg(sp + ie) < e) ++ie;           // first site with position >= e
                inx = ie;
                while (inx < s1 && __ldg(sp + inx) == e) ++inx;       // first site with position > e = lb(cur + len)
                if (isM || isN) {
                    // stabbed positions [cur, e - 1]: covered by the block (a <= t, b >= t + 2, S:469) or strictly inside the
                    // junction (l < t < r with l = cur - 1, r = e; S:507)
                    const int lo = max(idx, own_lo), hi = min(ie, own_hi);
                    v = lo < hi;
                    const uint32_t kind = (isN ? 2u : 0u) + k;
                    key_lo = 4u * (uint32_t)lo + kind; key_hi = 4u * (uint32_t)hi + kind;
                }
            }
            if (isN) {                                                // hot endpoints: l = cur - 1, r = cur + len - 1
                const int32_t l = cur - 1;
                int a = idx;
                while (a > s0 && __ldg(sp + a - 1) == l) --a;         // first site at position l, if any
                if (a < idx && __ldg(hot + a)) hl = (uint32_t)a + 1u;
                if (len > 0) { if (ie < s1 && __ldg(sp + ie) == l + len && __ldg(hot + ie)) hr = (uint32_t)ie + 1u; }
                else hr = hl;                                         // zero-length N: both ends on the same position
            }
            if (__any_sync(0xffffffffu, v)) {
                run_add(A.cnt.diff, key_lo, v, false, lane);
                run_add(A.cnt.diff, key_hi, v, true, lane);
            }
            push_hot(list, lother, list_n, hl, hr, cur - 1, cur + len - 1, i, j, lane);
            if (adv) { cur += len; idx = inx; }
        }
    }
    if (list_n) flush_list(list, lother, list_n, m.rec_lo, A, lane);
}

__global__ void __launch_bounds__(FC_THREADS, 2) k_count_fused(const __grid_constant__ FArgs A) {
    extern __shared__ __align__(1024) uint8_t smem_raw[];
    FSmem& sm = *reinterpret_cast<FSmem*>(smem_raw);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    if (threadIdx.x == 0) {
        if (smem_u32(sm.lut) & 511u) __trap();                       // the table's addressing relies on it
        for (int s = 0; s < FC_STAGES; ++s) { mbar_init(&sm.full[s], 1); mbar_init(&sm.empty[s], FC_CONSUMERS); }
    }
    if (threadIdx.x < 32) {
        // entry 2 * code + class: M = X stab sites with the coverage field of the class (S:457-459, :469), N with the span field
        // (S:480-483, :507), D only advances (S:460-462), I S H P (and the unassigned codes) do nothing
        const uint32_t op = threadIdx.x >> 1, k = threadIdx.x & 1u;
        const bool isM = op == 0u || op == 7u || op == 8u, isN = op == 3u, adv = isM || isN || op == 2u;
        const uint32_t incM = 1u << (8u * k);                        // byte fields of the redux word: cov class 0 / 1, span class 0 / 1
        sm.lut[threadIdx.x] = make_uint4(adv ? 0xffffffffu : 0u, isM ? incM : (isN ? incM << 16 : 0u), (isM || isN) ? 0xffffffffu : 0u, isN ? 1u : 0u);
    }
    const uint32_t lut_base = smem_u32(sm.lut);
    __syncthreads();
    if (warp == FC_CWARPS) {
        // ===== producer =====
        if (lane != 0) return;
        uint32_t it = 0;
        const uint32_t n_chunks = A.chunk_hi - A.chunk_lo;
        const uint4* cq = reinterpret_cast<const uint4*>(A.chunks + A.chunk_lo);
        uint32_t nbase = atomicAdd(A.work, (uint32_t)FC_BATCH);
        uint4 nq[FC_BATCH][3];
#pragma unroll
        for (int b = 0; b < FC_BATCH; ++b) {
            const uint32_t c = min(nbase + b, n_chunks - 1u);
#pragma unroll
            for (int q = 0; q < 3; ++q) nq[b][q] = __ldg(cq + 3u * c + q);
        }
        for (;;) {
            const uint32_t base = nbase;
            if (base >= n_chunks) break;
            uint4 cur[FC_BATCH][3];
#pragma unroll
            for (int b = 0; b < FC_BATCH; ++b)
#pragma unroll
                for (int q = 0; q < 3; ++q) cur[b][q] = nq[b][q];
            // the next claim and its descriptors are in flight while this batch is staged
            nbase = atomicAdd(A.work, (uint32_t)FC_BATCH);
#pragma unroll
            for (int b = 0; b < FC_BATCH; ++b) {
                const uint32_t c = min(nbase + b, n_chunks - 1u);
#pragma unroll
                for (int q = 0; q < 3; ++q) nq[b][q] = __ldg(cq + 3u * c + q);
            }
#pragma unroll
            for (int b = 0; b < FC_BATCH; ++b) {
                if (base + b >= n_chunks) continue;
                const uint4 q0 = cur[b][0], q1 = cur[b][1], q2 = cur[b][2];
                const int32_t chrom = (int32_t)q0.x;
                const uint32_t rec_lo = q0.y, rec_hi = q0.z, c_lo = q0.w, c_hi = q1.x;
                const int32_t s0 = (int32_t)q1.y, s1 = (int32_t)q1.z, sb_g0 = (int32_t)q1.w, sb_nb = (int32_t)q2.x;
                if (rec_hi <= rec_lo || s1 <= s0 || c_hi <= c_lo) continue;      // nothing to count on a chromosome without sites
                const uint32_t a0 = rec_lo & ~7u, nr = (rec_hi - a0 + 7u) & ~7u, noff = (rec_hi - a0 + 1u + 3u) & ~3u;
                const uint32_t ca = c_lo & ~3u, nw = (c_hi - ca + 3u) & ~3u;
                const bool staged = nw <= (uint32_t)FC_CIG;
                const uint32_t stage = it % FC_STAGES, parity = (it / FC_STAGES) & 1u;
                mbar_wait_backoff(&sm.empty[stage], parity ^ 1u);
                FMeta& m = sm.meta[stage];
                m.flags = staged ? 0u : FM_GLOBAL_CIG; m.n_rec = rec_hi - rec_lo; m.skip = rec_lo - a0; m.cig_base = ca;
                m.rec_lo = rec_lo; m.chrom = chrom; m.s0 = s0; m.s1 = s1; m.sb_g0 = sb_g0; m.sb_nb = sb_nb;
                sm.next_group[stage] = 0u;
                FStage& st = sm.st[stage];
                mbar_expect_tx(&sm.full[stage], nr * 4u + noff * 4u + nr * 2u + (staged ? nw * 4u : 0u));
                bulk_g2s(st.pos, A.rec.pos + a0, nr * 4u, &sm.full[stage]);
                bulk_g2s(st.off, A.rec.cig_off + a0, noff * 4u, &sm.full[stage]);
                bulk_g2s(st.flag, A.rec.flag + a0, nr * 2u, &sm.full[stage]);
                if (staged) bulk_g2s(st.cig, A.rec.cigar + ca, nw * 4u, &sm.full[stage]);
                ++it;
            }
        }
        const uint32_t stage = it % FC_STAGES, parity = (it / FC_STAGES) & 1u;
        mbar_wait_backoff(&sm.empty[stage], parity ^ 1u);
        sm.meta[stage].flags = FM_DONE;
        mbar_arrive(&sm.full[stage]);
        return;
    }
    // ===== consumers =====
    for (uint32_t it = 0;; ++it) {
        const uint32_t stage = it % FC_STAGES, parity = (it / FC_STAGES) & 1u;
        mbar_wait(&sm.full[stage], parity);
        const FMeta m = sm.meta[stage];
        if (m.flags & FM_DONE) break;
        if (m.flags & FM_GLOBAL_CIG) consume<false>(sm.st[stage], m, sm.list[warp], sm.lother[warp], &sm.next_group[stage], lut_base, A);
        else consume<true>(sm.st[stage], m, sm.list[warp], sm.lother[warp], &sm.next_group[stage], lut_base, A);
        // every consumer thread releases the stage itself: its reads of the stage (and of the stage's meta data) are ordered
        // before the producer's next copy by its own arrive (release) / the producer's wait (acquire)
        mbar_arrive(&sm.empty[stage]);
    }
}

// CIGAR range and chromosome site / bin ranges of every chunk (runs once the site table is on the device)
__global__ void k_chunk_bounds(FChunk* chunks, uint32_t lo, uint32_t hi, const uint32_t* __restrict__ cig_off, DevGraph g) {
    const uint32_t i = lo + blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= hi) return;
    FChunk c = chunks[i];
    c.c_lo = cig_off[c.rec_lo]; c.c_hi = cig_off[c.rec_hi];
    if (c.chrom >= 0 && c.chrom < g.n_chrom && g.n_sites > 0) {
        c.s0 = g.cs_off[c.chrom]; c.s1 = g.cs_off[c.chrom + 1];
        c.sb_g0 = g.sb_base[c.chrom]; c.sb_nb = g.sb_base[c.chrom + 1] - c.sb_g0 - 1;
    } else {
        c.s0 = c.s1 = 0; c.sb_g0 = 0; c.sb_nb = 0;
    }
    chunks[i] = c;
}

// ---- packed host layout -> the arrays the counting kernel stages (spl_process_packed) -------------------------------
// Per record the packed view carries POS, three flag bits and the operator count; the CIGAR offsets are rebuilt here by a
// single-pass exclusive scan (decoupled look-back: tiles take tickets, publish epoch | flag | value in one 64-bit word), and
// the flag bits are put back where check_strand expects them (S:374-406).
constexpr int UP_THREADS = 256, UP_ITEMS = 8, UP_TILE = UP_THREADS * UP_ITEMS;
__global__ void __launch_bounds__(UP_THREADS)
k_unpack_records(const uint16_t* __restrict__ n_op, const uint8_t* __restrict__ flag8, uint32_t r0, uint32_t r1, uint32_t cig_base,
                 uint32_t* __restrict__ cig_off, uint16_t* __restrict__ flag16, unsigned long long* __restrict__ desc,
                 uint32_t* __restrict__ ticket, uint32_t epoch) {
    __shared__ uint32_t s_tile, s_prev, wsum[UP_THREADS / 32];
    if (threadIdx.x == 0) s_tile = atomicAdd(ticket, 1u);
    __syncthreads();
    const uint32_t t = s_tile;
    const uint32_t base = r0 + t * UP_TILE + threadIdx.x * UP_ITEMS;
    uint32_t v[UP_ITEMS], sum = 0;
#pragma unroll
    for (int q = 0; q < UP_ITEMS; ++q) {
        v[q] = 0;
        if (base + q < r1) {
            v[q] = n_op[base + q];
            const uint32_t f = flag8[base + q];
            flag16[base + q] = (uint16_t)((f & 1u) | ((f & 2u) << 3) | ((f & 4u) << 4));      // 0x1 paired, 0x10 reverse, 0x40 first in pair
        }
        sum += v[q];
    }
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    uint32_t inc = sum;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) { const uint32_t x = __shfl_up_sync(0xffffffffu, inc, o); if (lane >= o) inc += x; }
    if (lane == 31) wsum[warp] = inc;
    __syncthreads();
    uint32_t wbase = 0, total = 0;
#pragma unroll
    for (int w = 0; w < UP_THREADS / 32; ++w) { if (w < warp) wbase += wsum[w]; total += wsum[w]; }
    if (threadIdx.x == 0) {
        const unsigned long long tag = (unsigned long long)epoch << 34;
        volatile unsigned long long* d = desc;
        uint32_t prev = 0;
        if (t == 0) {
            d[0] = tag | (2ull << 32) | total;
        } else {
            d[t] = tag | (1ull << 32) | total;
            for (uint32_t p = t - 1;;) {
                const unsigned long long w = d[p];
                if ((w >> 34) != epoch || ((w >> 32) & 3ull) == 0ull) continue;          // not published yet
                prev += (uint32_t)w;
                if (((w >> 32) & 3ull) == 2ull) break;
                --p;
            }
            d[t] = tag | (2ull << 32) | (prev + total);
        }
        s_prev = prev;
        if (t == gridDim.x - 1) *ticket = 0u;                           // every ticket of this launch has been handed out
    }
    __syncthreads();
    uint32_t run = cig_base + s_prev + wbase + inc - sum;
#pragma unroll
    for (int q = 0; q < UP_ITEMS; ++q) {
        if (base + q < r1) cig_off[base + q] = run;
        run += v[q];
        if (base + q + 1 == r1) cig_off[r1] = run;                      // the slab's end offset (the next slab writes the same value)
    }
}

// ---- compact host layout -> the same arrays (spl_process_compact) ----------------------------------------------------
// 9 B per record on the wire instead of 17: POS as a 16-bit offset from the lowest POS of the record's stride of
// SPL_PACKED_INDEX_STRIDE records (strides wider than 65535 bp keep 32-bit positions in a side array), operator count in a byte,
// CIGAR operators in 16 bits (op | len << 4, len < 4096) unless the record has a longer operator (then its operators are in the
// 32-bit stream, BAM-encoded).  Per stride the view carries the offsets of its first record in both operator streams, so every
// stride unpacks on its own: one CTA per stride, four consecutive records per thread, block-local scans of the two operator
// counts.  A 16-bit operator zero-extends to the BAM encoding.
constexpr int UC_THREADS = 256, UC_PER = 4;
static_assert(UC_THREADS * UC_PER == SPL_PACKED_INDEX_STRIDE, "one CTA unpacks one stride");
struct CompactDev {
    const uint16_t* pos16; const uint8_t* flag8; const uint8_t* n_op8;
    const uint16_t* c16; const uint32_t* c32;
    const int32_t* pos_base; const int32_t* pos_wide; const uint32_t* idx16; const uint32_t* idx32;
};
__global__ void __launch_bounds__(UC_THREADS)
k_unpack_compact(CompactDev v, uint32_t stride0, uint32_t r_end, int32_t* __restrict__ pos, uint16_t* __restrict__ flag16,
                 uint32_t* __restrict__ cig_off, uint32_t* __restrict__ cigar, uint32_t* __restrict__ bad) {
    __shared__ uint32_t wS[UC_THREADS / 32], wL[UC_THREADS / 32];
    const uint32_t k = stride0 + blockIdx.x;
    const uint32_t rb = k * (uint32_t)SPL_PACKED_INDEX_STRIDE + threadIdx.x * UC_PER;
    uint32_t n[UC_PER], f[UC_PER], sS = 0, sL = 0;
#pragma unroll
    for (int q = 0; q < UC_PER; ++q) {
        n[q] = 0; f[q] = 0;
        if (rb + q < r_end) { n[q] = v.n_op8[rb + q]; f[q] = v.flag8[rb + q]; }
        if (f[q] & 8u) sL += n[q]; else sS += n[q];
    }
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    uint32_t iS = sS, iL = sL;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const uint32_t a = __shfl_up_sync(0xffffffffu, iS, o), b = __shfl_up_sync(0xffffffffu, iL, o);
        if (lane >= o) { iS += a; iL += b; }
    }
    if (lane == 31) { wS[warp] = iS; wL[warp] = iL; }
    __syncthreads();
    uint32_t bS = v.idx16[k] + iS - sS, bL = v.idx32[k] + iL - sL;       // this thread's first operator in either stream
    uint32_t tS = 0, tL = 0;
#pragma unroll
    for (int w = 0; w < UC_THREADS / 32; ++w) { if (w < warp) { bS += wS[w]; bL += wL[w]; } tS += wS[w]; tL += wL[w]; }
    // the per-record counts must add up to what the stride's anchors say, or the offsets below would leave the streams: such a
    // stride is unpacked as records without operators and the call fails (the host reads the flag after the pass)
    if (tS != v.idx16[k + 1] - v.idx16[k] || tL != v.idx32[k + 1] - v.idx32[k]) {
        if (threadIdx.x == 0) atomicOr(bad, 1u);
        const uint32_t o = v.idx16[k] + v.idx32[k];
#pragma unroll
        for (int q = 0; q < UC_PER; ++q) {
            const uint32_t r = rb + q;
            if (r >= r_end) break;
            cig_off[r] = o; pos[r] = 0; flag16[r] = 0;
            if (r + 1 == r_end) cig_off[r_end] = o;
        }
        return;
    }
    uint32_t out = bS + bL;                                                // operators of all records before this one
    const int32_t base = v.pos_base[k];
#pragma unroll
    for (int q = 0; q < UC_PER; ++q) {
        const uint32_t r = rb + q;
        if (r >= r_end) break;
        cig_off[r] = out;
        pos[r] = base >= 0 ? base + (int32_t)v.pos16[r] : v.pos_wide[(size_t)(-(base + 1)) * SPL_PACKED_INDEX_STRIDE + (r - k * (uint32_t)SPL_PACKED_INDEX_STRIDE)];
        flag16[r] = (uint16_t)((f[q] & 1u) | ((f[q] & 2u) << 3) | ((f[q] & 4u) << 4));          // 0x1 paired, 0x10 reverse, 0x40 first in pair
        if (f[q] & 8u) { for (uint32_t j = 0; j < n[q]; ++j) cigar[out + j] = v.c32[bL + j]; bL += n[q]; }
        else           { for (uint32_t j = 0; j < n[q]; ++j) cigar[out + j] = (uint32_t)v.c16[bS + j]; bS += n[q]; }
        out += n[q];
        if (r + 1 == r_end) cig_off[r_end] = out;                           // the slab's end offset (the next slab writes the same value)
    }
}

int fused_grid() {
    static std::mutex mu;
    static int grid_of[64] = {0};
    int dev = 0;
    cudaGetDevice(&dev);
    std::lock_guard<std::mutex> lock(mu);
    if (dev >= 0 && dev < 64 && grid_of[dev]) return grid_of[dev];
    cudaFuncSetAttribute((const void*)k_count_fused, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(FSmem));
    int per_sm = 1;
    cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, (const void*)k_count_fused, FC_THREADS, sizeof(FSmem));
    if (per_sm < 1) per_sm = 1;
    const int grid = sm_count_current_device() * per_sm;     // one resident CTA per slot: a multiple of the SM count
    if (dev >= 0 && dev < 64) grid_of[dev] = grid;
    return grid;
}

}  // namespace

void launch_chunk_bounds(FChunk* chunks, uint32_t lo, uint32_t hi, const uint32_t* cig_off, DevGraph g, void* stream) {
    if (hi > lo) { SPL_LAUNCH; k_chunk_bounds<<<(hi - lo + 255) / 256, 256, 0, (cudaStream_t)stream>>>(chunks, lo, hi, cig_off, g); }
}

// `work` points at a zeroed u32 (the chunk counter of this launch); hot items are appended to hotq (hot_n counts them)
void launch_count_fused(const DevRecords& rec, const FChunk* chunks, uint32_t lo, uint32_t hi, DevGraph g, DevCounters cnt,
                        uint32_t* work, uint32_t flags, uint4* hotq, uint32_t* hot_n, uint32_t hot_cap, void* stream) {
    if (hi <= lo || g.n_sites <= 0) return;
    FArgs a{rec, chunks, lo, hi, g, cnt, work, flags, hotq, hot_n, hot_cap};
    const int grid = (int)min((uint32_t)fused_grid(), (hi - lo + (uint32_t)FC_BATCH - 1u) / (uint32_t)FC_BATCH);
    { SPL_LAUNCH; k_count_fused<<<grid, FC_THREADS, sizeof(FSmem), (cudaStream_t)stream>>>(a); }
}

// records [r0, r1) of a packed upload: cig_off[r0 .. r1] (cig_base = offset of record r0) and flag[r0 .. r1)
uint32_t unpack_desc_words(uint32_t n_rec) { return (n_rec + UP_TILE - 1) / UP_TILE + 8; }
void launch_unpack_records(const uint16_t* n_op, const uint8_t* flag8, uint32_t r0, uint32_t r1, uint32_t cig_base, uint32_t* cig_off,
                           uint16_t* flag16, unsigned long long* desc, uint32_t* ticket, uint32_t epoch, void* stream) {
    if (r1 <= r0) return;
    { SPL_LAUNCH; k_unpack_records<<<(r1 - r0 + UP_TILE - 1) / UP_TILE, UP_THREADS, 0, (cudaStream_t)stream>>>(n_op, flag8, r0, r1, cig_base, cig_off, flag16, desc, ticket, epoch); }
}

// strides [stride0, ...) up to record r_end of a compact upload: pos / flag / cig_off[.. r_end] / cigar of those records
void launch_unpack_compact(const uint16_t* pos16, const uint8_t* flag8, const uint8_t* n_op8, const uint16_t* c16, const uint32_t* c32,
                           const int32_t* pos_base, const int32_t* pos_wide, const uint32_t* idx16, const uint32_t* idx32, uint32_t r0,
                           uint32_t r1, int32_t* pos, uint16_t* flag16, uint32_t* cig_off, uint32_t* cigar, uint32_t* bad, void* stream) {
    if (r1 <= r0) return;
    const CompactDev v{pos16, flag8, n_op8, c16, c32, pos_base, pos_wide, idx16, idx32};
    const uint32_t s0 = r0 / SPL_PACKED_INDEX_STRIDE, s1 = (r1 + SPL_PACKED_INDEX_STRIDE - 1) / SPL_PACKED_INDEX_STRIDE;
    { SPL_LAUNCH; k_unpack_compact<<<s1 - s0, UC_THREADS, 0, (cudaStream_t)stream>>>(v, s0, r1, pos, flag16, cig_off, cigar, bad); }
}

// the queued hot items of every slab, after the counting kernels: one thread per item
void launch_hot_items(const DevRecords& rec, DevGraph g, DevCounters cnt, uint32_t flags, const uint4* hotq, const uint32_t* hot_n,
                      uint32_t hot_cap, void* stream) {
    if (g.n_sites <= 0 || hot_cap == 0) return;
    { SPL_LAUNCH; k_hot_items<<<sm_count_current_device() * 8, 256, 0, (cudaStream_t)stream>>>(rec, g, cnt, flags, hotq, hot_n, hot_cap); }
}

}  // namespace spl
