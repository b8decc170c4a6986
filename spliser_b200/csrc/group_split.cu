// Stable partition of one ingest's records by tag group (group_split.h).
//
//   k_group_hist<FIRST>     per tile of 4096 records: histogram of one 8-bit digit of the group id (digit-major, so that one
//                           scan per digit orders the tiles); the first pass skips records without a group and counts them
//   k_group_scan            one block per digit: exclusive scan over the tiles, and the digit's total
//   k_group_scatter<FIRST>  per tile: every record's rank among the records of its digit before it in the tile (warp match +
//                           per-warp counts), so the pass is stable; writes the 16-bit key and the record index
//   k_group_cigsum / k_group_scan / k_group_cigscan   exclusive scan of the sorted records' CIGAR lengths
//   k_group_bounds          the first sorted record and operator of every group, and the (group, chromosome) segments
//   k_group_gather<XS>      the columns of every kept record into its group's slice; k_group_term: cig_off[n] of every group
// The first pass reads the ingest's int32 group column and drops the records with a negative group; a second pass over the
// high byte runs only when there are more than 256 groups.  Scratch: 6 B per record for each key / index buffer pair, 4 B per
// record for the CIGAR offsets, 1 KiB per 4096 records for the histograms -- O(records), whatever the number of groups.
#include <cuda_runtime.h>

#include <algorithm>
#include <cstdint>
#include <string>
#include <vector>

#include "device_types.h"
#include "group_split.h"

namespace spl {

namespace {

constexpr int GT = 256;                // threads per block
constexpr int GI = 16;                 // records per thread and tile
constexpr uint32_t TILE = GT * GI;

// exclusive scan of one value per thread over a block of GT threads; *total receives the sum
__device__ __forceinline__ uint32_t block_excl_scan(uint32_t v, uint32_t* s_warp, uint32_t* total) {
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    uint32_t x = v;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) { const uint32_t y = __shfl_up_sync(0xffffffffu, x, d); if (lane >= d) x += y; }
    if (lane == 31) s_warp[w] = x;
    __syncthreads();
    uint32_t before = 0, all = 0;
#pragma unroll
    for (int k = 0; k < GT / 32; ++k) { const uint32_t t = s_warp[k]; if (k < w) before += t; all += t; }
    __syncthreads();                                                    // s_warp may be re-used by the caller
    *total = all;
    return before + x - v;
}

template <bool FIRST>
__device__ __forceinline__ bool load_key(const int32_t* __restrict__ grp, const uint16_t* __restrict__ keys, uint64_t i, uint64_t n, uint32_t& key) {
    if (i >= n) return false;
    if (FIRST) { const int32_t g = grp[i]; key = (uint32_t)g; return g >= 0; }
    key = keys[i];
    return true;
}

template <bool FIRST>
__global__ void __launch_bounds__(GT) k_group_hist(const int32_t* __restrict__ grp, const uint16_t* __restrict__ keys, uint64_t n, int shift,
                                                   uint32_t* __restrict__ hist, uint32_t n_tiles, unsigned long long* __restrict__ neg) {
    __shared__ uint32_t s_h[256];
    __shared__ uint32_t s_neg[2];
    const uint32_t tile = blockIdx.x;
    s_h[threadIdx.x] = 0;
    if (threadIdx.x < 2) s_neg[threadIdx.x] = 0;
    __syncthreads();
    uint32_t nv = 0, ng = 0;
    for (int r = 0; r < GI; ++r) {
        const uint64_t i = (uint64_t)tile * TILE + (uint32_t)r * GT + threadIdx.x;
        uint32_t key = 0;
        if (load_key<FIRST>(grp, keys, i, n, key)) atomicAdd(&s_h[(key >> shift) & 255u], 1u);
        else if (FIRST && i < n) { if ((int32_t)key == -1) ++nv; else ++ng; }
    }
    if (FIRST) {
        nv = __reduce_add_sync(0xffffffffu, nv); ng = __reduce_add_sync(0xffffffffu, ng);
        if ((threadIdx.x & 31) == 0 && (nv | ng)) { atomicAdd(&s_neg[0], nv); atomicAdd(&s_neg[1], ng); }
    }
    __syncthreads();
    hist[(size_t)threadIdx.x * n_tiles + tile] = s_h[threadIdx.x];
    if (FIRST && threadIdx.x < 2 && s_neg[threadIdx.x]) atomicAdd(&neg[threadIdx.x], (unsigned long long)s_neg[threadIdx.x]);
}

// block b: exclusive scan of a[b * n .. b * n + n) in place, tot[b] = its sum
__global__ void __launch_bounds__(GT) k_group_scan(uint32_t* __restrict__ a, uint32_t n, uint32_t* __restrict__ tot) {
    __shared__ uint32_t s_warp[GT / 32];
    uint32_t* row = a + (size_t)blockIdx.x * n;
    uint32_t carry = 0;
    for (uint32_t c0 = 0; c0 < n; c0 += GT) {
        const uint32_t i = c0 + threadIdx.x;
        const uint32_t v = i < n ? row[i] : 0u;
        uint32_t all;
        const uint32_t ex = block_excl_scan(v, s_warp, &all);
        if (i < n) row[i] = carry + ex;
        carry += all;
    }
    if (threadIdx.x == 0) tot[blockIdx.x] = carry;
}

template <bool FIRST>
__global__ void __launch_bounds__(GT) k_group_scatter(const int32_t* __restrict__ grp, const uint16_t* __restrict__ keys_in,
                                                      const uint32_t* __restrict__ idx_in, uint64_t n, int shift,
                                                      const uint32_t* __restrict__ hist, uint32_t n_tiles, const uint32_t* __restrict__ tot,
                                                      uint16_t* __restrict__ keys_out, uint32_t* __restrict__ idx_out) {
    __shared__ uint32_t s_run[256];                                     // next output slot of every digit in this tile
    __shared__ uint32_t s_cnt[GT / 32][256];                            // records of every digit in every warp, this round
    __shared__ uint32_t s_off[GT / 32][256];                            // the warp's first output slot of every digit, this round
    __shared__ uint32_t s_warp[GT / 32];
    const uint32_t tile = blockIdx.x, d_me = threadIdx.x;
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    {
        uint32_t all;
        const uint32_t base = block_excl_scan(tot[d_me], s_warp, &all);
        s_run[d_me] = base + hist[(size_t)d_me * n_tiles + tile];
    }
#pragma unroll
    for (int k = 0; k < GT / 32; ++k) s_cnt[k][d_me] = 0;
    __syncthreads();
    for (int r = 0; r < GI; ++r) {
        const uint64_t i = (uint64_t)tile * TILE + (uint32_t)r * GT + threadIdx.x;
        uint32_t key = 0;
        const bool live = load_key<FIRST>(grp, keys_in, i, n, key);
        const uint32_t d = (key >> shift) & 255u;
        const uint32_t peers = __match_any_sync(0xffffffffu, live ? d : 256u + (uint32_t)lane);
        const uint32_t rank = __popc(peers & ((1u << lane) - 1u));
        if (live && rank == 0) s_cnt[w][d] = __popc(peers);
        __syncthreads();
        {
            uint32_t run = s_run[d_me];
#pragma unroll
            for (int k = 0; k < GT / 32; ++k) { s_off[k][d_me] = run; run += s_cnt[k][d_me]; s_cnt[k][d_me] = 0; }
            s_run[d_me] = run;
        }
        __syncthreads();
        if (live) {
            const uint32_t o = s_off[w][d] + rank;
            keys_out[o] = (uint16_t)key;
            idx_out[o] = FIRST ? (uint32_t)i : idx_in[i];
        }
    }
}

__device__ __forceinline__ uint32_t cig_len(const uint32_t* __restrict__ cig_off, uint32_t s) { return cig_off[s + 1] - cig_off[s]; }

// per tile: the sum of the sorted records' CIGAR lengths
__global__ void __launch_bounds__(GT) k_group_cigsum(const uint32_t* __restrict__ idx, uint64_t n, const uint32_t* __restrict__ cig_off,
                                                     uint32_t* __restrict__ part) {
    __shared__ uint32_t s_warp[GT / 32];
    uint32_t v = 0;
    for (int r = 0; r < GI; ++r) {
        const uint64_t i = (uint64_t)blockIdx.x * TILE + (uint32_t)r * GT + threadIdx.x;
        if (i < n) v += cig_len(cig_off, idx[i]);
    }
    uint32_t all;
    block_excl_scan(v, s_warp, &all);
    if (threadIdx.x == 0) part[blockIdx.x] = all;
}

// coff[i] = CIGAR operators of the sorted records before i; coff[n] = all of them
__global__ void __launch_bounds__(GT) k_group_cigscan(const uint32_t* __restrict__ idx, uint64_t n, const uint32_t* __restrict__ cig_off,
                                                      const uint32_t* __restrict__ part, uint32_t* __restrict__ coff) {
    __shared__ uint32_t s_warp[GT / 32];
    uint32_t carry = part[blockIdx.x];
    for (int r = 0; r < GI; ++r) {
        const uint64_t i = (uint64_t)blockIdx.x * TILE + (uint32_t)r * GT + threadIdx.x;
        const uint32_t v = i < n ? cig_len(cig_off, idx[i]) : 0u;
        uint32_t all;
        const uint32_t ex = block_excl_scan(v, s_warp, &all);
        if (i < n) coff[i] = carry + ex;
        if (i + 1 == n) coff[n] = carry + ex + v;
        carry += all;
    }
}

__global__ void k_group_bounds(const uint16_t* __restrict__ keys, const uint32_t* __restrict__ idx, const int32_t* __restrict__ chrom,
                               const uint32_t* __restrict__ coff, uint64_t n, uint32_t* __restrict__ g_start, uint32_t* __restrict__ g_cig,
                               uint32_t* __restrict__ n_seg, uint32_t* __restrict__ seg_first, int32_t* __restrict__ seg_chrom, uint32_t cap) {
    const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const uint32_t k = keys[i];
    const bool new_group = i == 0 || keys[i - 1] != k;
    if (new_group) { g_start[k] = (uint32_t)i; g_cig[k] = coff[i]; }
    const int32_t c = chrom[idx[i]];
    if (new_group || c != chrom[idx[i - 1]]) {
        const uint32_t s = atomicAdd(n_seg, 1u);
        if (s < cap) { seg_first[s] = (uint32_t)i; seg_chrom[s] = c; }
    }
}

template <bool XS>
__global__ void __launch_bounds__(GT) k_group_gather(const uint16_t* __restrict__ keys, const uint32_t* __restrict__ idx,
                                                     const uint32_t* __restrict__ coff, uint64_t n, DevRecordArrays in,
                                                     const GroupCols* __restrict__ cols, char* __restrict__ base) {
    const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const GroupCols c = cols[keys[i]];
    const uint32_t s = idx[i], l = (uint32_t)i - c.start, c0 = coff[i] - c.cig0;
    reinterpret_cast<int32_t*>(base + c.pos)[l] = in.pos[s];
    reinterpret_cast<uint16_t*>(base + c.flag)[l] = in.flag[s];
    reinterpret_cast<uint32_t*>(base + c.off)[l] = c0;
    if (XS) reinterpret_cast<uint8_t*>(base + c.xs)[l] = in.xs[s];
    uint32_t* cig = reinterpret_cast<uint32_t*>(base + c.cig) + c0;
    const uint32_t a = in.cig_off[s], b = in.cig_off[s + 1];
    for (uint32_t q = a; q < b; ++q) cig[q - a] = in.cigar[q];
}

__global__ void k_group_term(const GroupCols* __restrict__ cols, uint32_t n_groups, char* __restrict__ base) {
    const uint32_t g = blockIdx.x * blockDim.x + threadIdx.x;
    if (g < n_groups) reinterpret_cast<uint32_t*>(base + cols[g].off)[cols[g].n] = cols[g].nc;
}

}  // namespace

#define GS_CU(call)                                                                     \
    do {                                                                                \
        cudaError_t _e = (call);                                                        \
        if (_e != cudaSuccess) { err = std::string(#call) + ": " + cudaGetErrorString(_e); return -1; } \
    } while (0)

int group_sort(GroupSplitMem& m, const DevRecordArrays& in, const int32_t* grp, uint64_t n, int32_t n_groups, cudaStream_t st, GroupSort& out, std::string& err) {
    const uint32_t G = (uint32_t)n_groups;
    out = GroupSort{};
    out.n_rec.assign(G, 0); out.n_cig.assign(G, 0);
    out.seg_chrom.assign(G, {}); out.seg_off.assign(G, std::vector<int64_t>(1, 0));
    out.g_start.assign(G, 0); out.g_cig.assign(G, 0);
    if (n >= (uint64_t)UINT32_MAX - 16) { err = "more than 2^32 records"; return -1; }
    const uint32_t n_tiles = (uint32_t)std::max<uint64_t>(1, (n + TILE - 1) / TILE);
    const bool two = G > 256;
    // scratch: two key/index buffer pairs (one when a single pass suffices), CIGAR offsets, histograms, counters, bounds
    size_t off = 0;
    auto take = [&](size_t bytes) { off = (off + 255) & ~(size_t)255; const size_t o = off; off += bytes; return o; };
    const size_t o_k0 = take((n + 4) * 2), o_i0 = take((n + 4) * 4), o_k1 = two ? take((n + 4) * 2) : 0, o_i1 = two ? take((n + 4) * 4) : 0,
                 o_co = take((n + 4) * 4), o_h = take((size_t)256 * n_tiles * 4), o_t = take(256 * 4 + 16), o_neg = take(16),
                 o_gs = take((size_t)G * 4), o_gc = take((size_t)G * 4), o_ns = take(16);
    if (m.sort.reserve(off + 256) != cudaSuccess) { cudaGetLastError(); err = "not enough device memory for the sort scratch"; return 1; }
    // segment boundaries: a group restarts a segment on every chromosome it has records on, so a sorted BAM with R references
    // in use gives up to R x G of them.  The first try holds as many as a BAM's own segments plus one per group; when the count
    // says more, the buffer takes exactly that many (at most one per record) and the boundaries are found again.
    uint32_t cap = (uint32_t)std::min<uint64_t>(n + 1, (uint64_t)BAMGPU_MAX_SEG + G);
    auto seg_buf = [&](uint32_t c) { return m.seg.reserve((size_t)c * 8 + 512) == cudaSuccess; };
    if (!seg_buf(cap)) { cudaGetLastError(); err = "not enough device memory for the segment boundaries"; return 1; }
    char* b = (char*)m.sort.p;
    uint16_t* k0 = (uint16_t*)(b + o_k0); uint32_t* i0 = (uint32_t*)(b + o_i0);
    uint16_t* k1 = (uint16_t*)(b + o_k1); uint32_t* i1 = (uint32_t*)(b + o_i1);
    uint32_t* coff = (uint32_t*)(b + o_co); uint32_t* hist = (uint32_t*)(b + o_h); uint32_t* tot = (uint32_t*)(b + o_t);
    unsigned long long* neg = (unsigned long long*)(b + o_neg);
    uint32_t* gst = (uint32_t*)(b + o_gs); uint32_t* gcg = (uint32_t*)(b + o_gc); uint32_t* ns = (uint32_t*)(b + o_ns);
    uint32_t* sf = (uint32_t*)m.seg.p; int32_t* scd = (int32_t*)((char*)m.seg.p + (((size_t)cap * 4 + 255) & ~(size_t)255));
    GS_CU(cudaMemsetAsync(neg, 0, 16, st));
    GS_CU(cudaMemsetAsync(ns, 0, 16, st));
    GS_CU(cudaMemsetAsync(gst, 0xff, (size_t)G * 4, st));
    // ---- pass 1: the low byte, records without a group dropped
    { SPL_LAUNCH; k_group_hist<true><<<n_tiles, GT, 0, st>>>(grp, nullptr, n, 0, hist, n_tiles, neg); }
    { SPL_LAUNCH; k_group_scan<<<256, GT, 0, st>>>(hist, n_tiles, tot); }
    { SPL_LAUNCH; k_group_scatter<true><<<n_tiles, GT, 0, st>>>(grp, nullptr, nullptr, n, 0, hist, n_tiles, tot, two ? k1 : k0, two ? i1 : i0); }
    GS_CU(cudaGetLastError());
    unsigned long long h_neg[2] = {0, 0};
    GS_CU(cudaMemcpyAsync(h_neg, neg, 16, cudaMemcpyDeviceToHost, st));
    GS_CU(cudaStreamSynchronize(st));
    out.no_value = h_neg[0]; out.no_group = h_neg[1];
    const uint64_t nk = n - h_neg[0] - h_neg[1];
    out.n_kept = nk;
    const uint32_t kt = (uint32_t)std::max<uint64_t>(1, (nk + TILE - 1) / TILE);
    // ---- pass 2: the high byte, stable over pass 1's order
    if (two) {
        { SPL_LAUNCH; k_group_hist<false><<<kt, GT, 0, st>>>(nullptr, k1, nk, 8, hist, kt, nullptr); }
        { SPL_LAUNCH; k_group_scan<<<256, GT, 0, st>>>(hist, kt, tot); }
        { SPL_LAUNCH; k_group_scatter<false><<<kt, GT, 0, st>>>(nullptr, k1, i1, nk, 8, hist, kt, tot, k0, i0); }
    }
    // ---- CIGAR offsets of the sorted records, group starts, segments
    { SPL_LAUNCH; k_group_cigsum<<<kt, GT, 0, st>>>(i0, nk, in.cig_off, hist); }
    { SPL_LAUNCH; k_group_scan<<<1, GT, 0, st>>>(hist, kt, tot); }
    { SPL_LAUNCH; k_group_cigscan<<<kt, GT, 0, st>>>(i0, nk, in.cig_off, hist, coff); }
    if (nk == 0) GS_CU(cudaMemsetAsync(coff, 0, 4, st));
    if (nk) { SPL_LAUNCH; k_group_bounds<<<(unsigned)((nk + GT - 1) / GT), GT, 0, st>>>(k0, i0, in.chrom, coff, nk, gst, gcg, ns, sf, scd, cap); }
    GS_CU(cudaGetLastError());
    uint32_t h_ns = 0, h_ctot = 0;
    GS_CU(cudaMemcpyAsync(&h_ns, ns, 4, cudaMemcpyDeviceToHost, st));
    GS_CU(cudaMemcpyAsync(&h_ctot, coff + nk, 4, cudaMemcpyDeviceToHost, st));
    GS_CU(cudaMemcpyAsync(out.g_start.data(), gst, (size_t)G * 4, cudaMemcpyDeviceToHost, st));
    GS_CU(cudaMemcpyAsync(out.g_cig.data(), gcg, (size_t)G * 4, cudaMemcpyDeviceToHost, st));
    GS_CU(cudaStreamSynchronize(st));
    if (h_ns > cap) {
        cap = h_ns;
        if (!seg_buf(cap)) { cudaGetLastError(); err = "not enough device memory for the segment boundaries"; return 1; }
        sf = (uint32_t*)m.seg.p; scd = (int32_t*)((char*)m.seg.p + (((size_t)cap * 4 + 255) & ~(size_t)255));
        GS_CU(cudaMemsetAsync(ns, 0, 4, st));
        { SPL_LAUNCH; k_group_bounds<<<(unsigned)((nk + GT - 1) / GT), GT, 0, st>>>(k0, i0, in.chrom, coff, nk, gst, gcg, ns, sf, scd, cap); }
        GS_CU(cudaGetLastError());
        GS_CU(cudaMemcpyAsync(&h_ns, ns, 4, cudaMemcpyDeviceToHost, st));
        GS_CU(cudaStreamSynchronize(st));
        if (h_ns > cap) { err = "segment count changed between two passes"; return -1; }
    }
    std::vector<uint32_t> sf_h(h_ns), first(h_ns);
    std::vector<int32_t> sc_h(h_ns), sc(h_ns);
    if (h_ns) {
        GS_CU(cudaMemcpyAsync(sf_h.data(), sf, (size_t)h_ns * 4, cudaMemcpyDeviceToHost, st));
        GS_CU(cudaMemcpyAsync(sc_h.data(), scd, (size_t)h_ns * 4, cudaMemcpyDeviceToHost, st));
        GS_CU(cudaStreamSynchronize(st));
    }
    {
        std::vector<uint32_t> order(h_ns);
        for (uint32_t k = 0; k < h_ns; ++k) order[k] = k;
        std::sort(order.begin(), order.end(), [&](uint32_t a, uint32_t c) { return sf_h[a] < sf_h[c]; });
        for (uint32_t k = 0; k < h_ns; ++k) { first[k] = sf_h[order[k]]; sc[k] = sc_h[order[k]]; }
    }
    // per group: records and operators from the starts of the next non-empty group, segments from the sorted boundaries
    std::vector<uint32_t> nonempty;
    for (uint32_t g = 0; g < G; ++g) if (out.g_start[g] != UINT32_MAX) nonempty.push_back(g);
    size_t s = 0;
    for (size_t q = 0; q < nonempty.size(); ++q) {
        const uint32_t g = nonempty[q];
        const uint64_t r0 = out.g_start[g], r1 = q + 1 < nonempty.size() ? out.g_start[nonempty[q + 1]] : nk;
        const uint64_t c1 = q + 1 < nonempty.size() ? out.g_cig[nonempty[q + 1]] : h_ctot;
        out.n_rec[g] = (int64_t)(r1 - r0); out.n_cig[g] = (int64_t)(c1 - out.g_cig[g]);
        auto& so = out.seg_off[g];
        so.clear();
        while (s < first.size() && first[s] < r1) { out.seg_chrom[g].push_back(sc[s]); so.push_back((int64_t)(first[s] - r0)); ++s; }
        so.push_back((int64_t)(r1 - r0));
    }
    for (uint32_t g = 0; g < G; ++g) if (out.g_start[g] == UINT32_MAX) out.g_start[g] = 0;
    out.keys = k0; out.idx = i0; out.coff = coff;
    return 0;
}

int group_gather(GroupSplitMem& m, const DevRecordArrays& in, const GroupSort& gs, const std::vector<GroupCols>& cols, char* base,
                 cudaStream_t st, std::string& err) {
    const uint32_t G = (uint32_t)cols.size();
    if (m.tab.reserve((size_t)G * sizeof(GroupCols) + 256) != cudaSuccess) { cudaGetLastError(); err = "not enough device memory for the group table"; return 1; }
    GroupCols* d_cols = (GroupCols*)m.tab.p;
    GS_CU(cudaMemcpyAsync(d_cols, cols.data(), (size_t)G * sizeof(GroupCols), cudaMemcpyHostToDevice, st));
    const uint64_t n = gs.n_kept;
    if (n) {
        const unsigned nb = (unsigned)((n + GT - 1) / GT);
        if (in.xs) { SPL_LAUNCH; k_group_gather<true><<<nb, GT, 0, st>>>(gs.keys, gs.idx, gs.coff, n, in, d_cols, base); }
        else { SPL_LAUNCH; k_group_gather<false><<<nb, GT, 0, st>>>(gs.keys, gs.idx, gs.coff, n, in, d_cols, base); }
    }
    { SPL_LAUNCH; k_group_term<<<(G + GT - 1) / GT, GT, 0, st>>>(d_cols, G, base); }
    GS_CU(cudaGetLastError());
    return 0;
}

}  // namespace spl
