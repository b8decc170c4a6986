// Device helpers shared by the counting kernels (kernels.cu: stabbing variant; count_fused.cu: fused difference-array
// variant): mbarrier / 1-D TMA wrappers, searches over the sorted site table, check_strand, and the per-read exception
// logic of checkBam (SpliSER_v0_1_8.py:494-557).
#pragma once
#include <cuda_runtime.h>

#include <climits>
#include <cstdint>

#include "device_types.h"

namespace spl {

// ------------------------------------------------------------------------------------------------
// mbarrier + 1-D TMA bulk copy (cp.async.bulk, SASS: UBLKCP / SYNCS)
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
// 1-D TMA bulk copy global -> shared, completion signalled on the mbarrier (SASS: UBLKCP)
__device__ __forceinline__ void bulk_g2s(void* dst, const void* src, uint32_t bytes, uint64_t* bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                     smem_u32(dst)),
                 "l"(src), "r"(bytes), "r"(smem_u32(bar))
                 : "memory");
}
// consumer-side wait: try_wait with a suspend-time hint parks the warp in hardware until the phase flips (or the hint
// expires), instead of spinning through issue slots the other resident warps need
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
    asm volatile(
        "{\n"
        ".reg .pred P1;\n"
        "LAB_WAIT:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 P1, [%0], %1, %2;\n"
        "@P1 bra DONE;\n"
        "bra LAB_WAIT;\n"
        "DONE:\n"
        "}\n" ::"r"(smem_u32(bar)),
        "r"(parity), "r"(20000u)
        : "memory");
}
// producer-side wait: the single producer lane would otherwise spin on the empty barrier for most of the
// kernel and steal issue slots from the consumers of the co-resident CTAs
__device__ __forceinline__ void mbar_wait_backoff(uint64_t* bar, uint32_t parity, uint32_t ns = 5000) {
    const uint32_t addr = smem_u32(bar);
    for (;;) {
        uint32_t done;
        asm volatile(
            "{\n"
            ".reg .pred P1;\n"
            "mbarrier.try_wait.parity.shared::cta.b64 P1, [%1], %2, %3;\n"     // suspend-time hint: the thread sleeps in hardware
            "selp.u32 %0, 1, 0, P1;\n"
            "}\n"
            : "=r"(done) : "r"(addr), "r"(parity), "r"(ns * 4u) : "memory");
        if (done) return;
    }
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}

__device__ __forceinline__ int4 ldg_stream(const int4* p) {   // streaming 128-bit load, no L1 allocation
    int4 r;
    asm volatile("ld.global.nc.L1::no_allocate.v4.s32 {%0,%1,%2,%3}, [%4];" : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w) : "l"(p));
    return r;
}
__device__ __forceinline__ uint32_t ldg_stream_u32(const uint32_t* p) {
    uint32_t r;
    asm volatile("ld.global.nc.L1::no_allocate.u32 %0, [%1];" : "=r"(r) : "l"(p));
    return r;
}

// ------------------------------------------------------------------------------------------------
// searches
// ------------------------------------------------------------------------------------------------
// first index in [lo, hi) with a[idx] >= key
__device__ __forceinline__ int lower_bound_i32(const int32_t* a, int lo, int hi, int32_t key) {
    while (lo < hi) {
        const int mid = (lo + hi) >> 1;
        if (a[mid] < key) lo = mid + 1; else hi = mid;
    }
    return lo;
}
// first index in [lo, hi) with a[idx] > key
__device__ __forceinline__ int upper_bound_i32(const int32_t* a, int lo, int hi, int32_t key) {
    while (lo < hi) {
        const int mid = (lo + hi) >> 1;
        if (a[mid] <= key) lo = mid + 1; else hi = mid;
    }
    return lo;
}

// lower_bound(key_lo) and upper_bound(key_hi) over the same sorted range [lo, hi) in one branch-free loop:
// the two dependent-load chains overlap, and with warp-uniform arguments the trip count is uniform
__device__ __forceinline__ void bound_pair_i32(const int32_t* a, int lo, int hi, int32_t key_lo, int32_t key_hi, int& i0, int& i1) {
    int n = hi - lo;
    if (n <= 0) { i0 = i1 = lo; return; }
    const int32_t* b0 = a + lo;
    const int32_t* b1 = a + lo;
    while (n > 1) {
        const int half = n >> 1;
        const int32_t v0 = b0[half - 1], v1 = b1[half - 1];
        b0 = (v0 < key_lo) ? b0 + half : b0;
        b1 = (v1 <= key_hi) ? b1 + half : b1;
        n -= half;
    }
    i0 = (int)(b0 - a) + (b0[0] < key_lo ? 1 : 0);
    i1 = (int)(b1 - a) + (b1[0] <= key_hi ? 1 : 0);
}

// first site index of chromosome `chrom` with position >= pos, through the direct-address bin index
__device__ __forceinline__ int site_lower(const DevGraph& g, int chrom, int32_t pos) {
    const int g0 = g.sb_base[chrom], nb = g.sb_base[chrom + 1] - g0 - 1;
    const int s1 = g.cs_off[chrom + 1];
    int i = g.sb_off[g0 + min(max(pos, 0) >> SB_SHIFT, nb)];
    while (i < s1 && g.site_pos[i] < pos) ++i;
    return i;
}

// ------------------------------------------------------------------------------------------------
// check_strand (S:374-406)
// ------------------------------------------------------------------------------------------------
// strand class bit of a read: 0 = '+', 1 = '-' under check_strand; always 0 when unstranded
__device__ __forceinline__ uint32_t read_class(uint32_t flag, uint32_t mode) {
    if (!(mode & FLAG_STRANDED)) return 0u;
    const bool first = (flag & 64u) || !(flag & 1u);
    const bool rev = (flag & 16u) != 0;
    bool plus = first != rev;               // fr
    if (mode & FLAG_RF) plus = !plus;
    return plus ? 0u : 1u;
}

// does a read of class k match a site of class c?  (CLS_ANY matches class 0 only because every
// read of an unstranded run is class 0)
__device__ __forceinline__ bool strand_ok(uint32_t site_cls, uint32_t k) {
    return (site_cls == 0u && k == 0u) || (site_cls == 1u && k == 0u) || (site_cls == 2u && k == 1u);
}

// ------------------------------------------------------------------------------------------------
// compSplicing exceptions (S:494-557) for one read at one site
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ bool in_list(const int32_t* a, int lo, int hi, int32_t key) {
    for (int i = lo; i < hi; ++i)
        if (a[i] == key) return true;
    return false;
}
__device__ __forceinline__ bool in_sorted(const int32_t* a, int lo, int hi, int32_t key) {
    const int i = lower_bound_i32(a, lo, hi, key);
    return i < hi && a[i] == key;
}

// is junction (l, r) a partner/competitor pair for site t?  (S:494-501)
__device__ __forceinline__ bool pc_pair(const DevGraph& g, int t, int32_t l, int32_t r) {
    const int p0 = g.pc_off[t], p1 = g.pc_off[t + 1], c0 = g.cp_off[t], c1 = g.cp_off[t + 1];
    return (in_list(g.pc_pos, p0, p1, l) && in_sorted(g.cp_pos, c0, c1, r)) ||
           (in_sorted(g.cp_pos, c0, c1, l) && in_list(g.pc_pos, p0, p1, r));
}

// +w on a counter, aggregated over the lanes of the warp that are here with the same address (the instances a warp handles
// mostly belong to one junction, so they hit the same few sites: one RED per warp and address instead of one per read)
__device__ __forceinline__ void agg_add(uint32_t* p, uint32_t w) {
    const unsigned active = __activemask();
    const unsigned peers = __match_any_sync(active, (unsigned long long)(uintptr_t)p);
    const uint32_t total = __reduce_add_sync(peers, w);
    if ((int)(threadIdx.x & 31u) == __ffs(peers) - 1) atomicAdd(p, total);
}

// The read makes compSplicing true for site t through its junction number rd.jrel, unless an earlier junction of the read
// already did: classify the read at t (S:503-557, first match wins); every counter moves by w.  Rd: nj, nb, jrel, jl(x) (bit 31: the N is the read's
// N starts at POS -> l = POS - 1), jr(x), bs(x), be(x) (block start / end; callers may leave flag bits in bit 31).
template <class Rd>
__device__ __forceinline__ void k4_classify(const Rd& rd, const DevGraph& g, const DevCounters& cnt, int t, uint32_t k, bool combine,
                                            uint32_t w = 1u /* identical reads this one stands for */) {
    bool earlier = false;
    for (uint32_t x = 0; x < rd.jrel && !earlier; ++x)
        earlier = pc_pair(g, t, (int32_t)(rd.jl(x) & POS_MASK), (int32_t)(rd.jr(x) & POS_MASK));
    if (earlier) return;
    const int32_t tp = g.site_pos[t];
    const bool ok = strand_ok(g.site_cls[t], k);
    bool alpha = false; int32_t partner_used = 0; int kstar = -1;
    for (uint32_t x = 0; x < rd.nj; ++x) {
        const uint32_t lraw = rd.jl(x);
        const int32_t ll = (int32_t)(lraw & POS_MASK), rr = (int32_t)(rd.jr(x) & POS_MASK);
        if (ll == tp && (lraw >> 31)) return;                    // POS > t: the read is skipped (S:435), a zero-length N's r = l too
        if (ll == tp) { alpha = true; partner_used = rr; }
        if (rr == tp) { alpha = true; partner_used = ll; }
        if (ll < tp && tp < rr) kstar = (int)x;
    }
    if (alpha) {                                                   // S:519-527
        for (int e = g.pc_off[t]; e < g.pc_off[t + 1]; ++e) {
            const int32_t pp = g.pc_pos[e];
            if (pp == partner_used) continue;
            bool in_read = false;
            for (uint32_t x = 0; x < rd.nj && !in_read; ++x)
                in_read = (int32_t)(rd.jl(x) & POS_MASK) == pp || (int32_t)(rd.jr(x) & POS_MASK) == pp;
            if (in_read) agg_add(cnt.dc + e, w);
        }
    } else if (kstar >= 0) {
        if (kstar >= (int)rd.jrel) {                               // compSplicing already true at k*: flanking (S:503-505)
            if (ok) agg_add(cnt.spanx + t, w);
            if (combine) agg_add(cnt.flank + t, w);
        }
    } else if (ok) {
        bool covers = false;
        for (uint32_t b = 0; b < rd.nb && !covers; ++b)
            covers = rd.bs(b) <= tp && (int32_t)(rd.be(b) & POS_MASK) >= tp + 2;
        if (covers) {                                              // beta1-type, S:544-552
            agg_add(cnt.covx + t, w);
            for (int e = g.pc_off[t]; e < g.pc_off[t + 1]; ++e) {
                const int32_t pp = g.pc_pos[e];
                bool in_read = false;
                for (uint32_t x = 0; x < rd.nj && !in_read; ++x)
                    in_read = (int32_t)(rd.jl(x) & POS_MASK) == pp || (int32_t)(rd.jr(x) & POS_MASK) == pp;
                if (in_read) agg_add(cnt.dc + e, w);
            }
        }
    }
}

// Is junction (l, r), whose endpoint (side 0 = l, 1 = r) sits on `anchor`, a partner/competitor pair for the q-th site
// of the anchor's reverse-partner list?  Every t of that list has the anchored endpoint in P_t by construction, so
// (l, r) is a pair for t (S:494-501) iff the OTHER endpoint is in C_t.  Returns t or -1.
__device__ __forceinline__ int k4_pair_site(const DevGraph& g, int q, int side, int32_t l, int32_t r) {
    const int t = g.rp_site[q];
    if (t < g.own_lo || t >= g.own_hi) return -1;
    const int c0 = g.cp_off[t], c1 = g.cp_off[t + 1];
    if (c0 == c1 || !in_sorted(g.cp_pos, c0, c1, side == 0 ? r : l)) return -1;
    // side 1 finds (r in P_t, l in C_t); if (l in P_t, r in C_t) holds as well, side 0 already handled t
    if (side == 1 && in_sorted(g.cp_pos, c0, c1, r) && in_list(g.pc_pos, g.pc_off[t], g.pc_off[t + 1], l)) return -1;
    return t;
}

}  // namespace spl
