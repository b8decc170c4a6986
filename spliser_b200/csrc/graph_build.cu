// K1 on the device: site table + competing-site graph from the junction table (clean regime).
//
// Replaces the structural half of findAlphaCounts (SpliSER_v0_1_8.py:289-355: binary_site_search, insort, addPartner,
// addPartnerCount) and findCompetitorPos (S:364-372) by sort / unique / group-by passes over the junction rows:
//   A  endpoint keys (chrom, pos, strand bit | row id) -> radix sort -> unique = sites in the reference's list order
//      (chrom_index order, position ascending, '+' before '-' per Site.__lt__, G:123-136); the first row of a run
//      gives the displayed strand and the Gene lookup line (first-seen semantics, S:296-345)
//   B  directed (site, partner | row) keys -> radix sort -> unique = PartnerCounts entries with their row segments
//   C  (site, first row | entry) -> radix sort = Partners / PartnerCounts in first-appearance order (G:243-262)
//   D  (site, partner-of-partner position) candidates -> radix sort -> unique = CompetitorPos (G:264-266)
//   E  reverse-partner index + hot flags, direct-address bin index of the site table
// The radix sort is a plain stable LSD sort (8-bit digits; per-tile histogram, scan, ranked scatter) written here;
// tables are a few 10^5..10^6 keys, so launch count matters more than bandwidth.
// The dirty regime ('?' strands in a stranded run, l == r rows) keeps the sequential host emulation (site_graph.cpp).
#include <cuda_runtime.h>

#include <climits>
#include <cstdint>
#include <algorithm>
#include <atomic>
#include <cstdio>
#include <cstdlib>
#include <string>
#include <vector>

#include "device_types.h"
#include "graph_build.h"

namespace spl {

namespace {

// Stable LSD radix sort, RS_BITS-bit digits: the site keys of a 30 Mb genome are 29 bits wide (3 passes of 10 instead of 4 of 8),
// GRCh38's 34 bits (4 instead of 5); every pass is three small launches, so the pass count is the cost.
constexpr int RS_THREADS = 256, RS_ITEMS = 8, RS_TILE = RS_THREADS * RS_ITEMS;
constexpr int RS_BITS = 10, RS_BINS = 1 << RS_BITS, RS_BPT = RS_BINS / RS_THREADS;      // digits a thread looks after

__global__ void __launch_bounds__(RS_THREADS)
k_rs_hist(const uint64_t* __restrict__ in, uint32_t n, int shift, uint32_t mask, uint32_t* __restrict__ hist, uint32_t n_tiles) {
    __shared__ uint32_t h[RS_BINS];
#pragma unroll
    for (int q = 0; q < RS_BPT; ++q) h[q * RS_THREADS + threadIdx.x] = 0;
    __syncthreads();
    const uint32_t base = blockIdx.x * RS_TILE;
#pragma unroll
    for (int r = 0; r < RS_ITEMS; ++r) {
        const uint32_t i = base + r * RS_THREADS + threadIdx.x;
        if (i < n) atomicAdd(&h[(uint32_t)(in[i] >> shift) & mask], 1u);
    }
    __syncthreads();
#pragma unroll
    for (int q = 0; q < RS_BPT; ++q) {                               // digit-major: one scan gives every (digit, tile) offset
        const uint32_t d = q * RS_THREADS + threadIdx.x;
        hist[d * n_tiles + blockIdx.x] = h[d];
    }
}

// stable ranked scatter: element order inside a tile is (round, warp, lane) = index order
__global__ void __launch_bounds__(RS_THREADS)
k_rs_scatter(const uint64_t* __restrict__ in, uint64_t* __restrict__ out, uint32_t n, int shift, uint32_t mask,
             const uint32_t* __restrict__ offs, uint32_t n_tiles) {
    __shared__ uint32_t wc[RS_THREADS / 32][RS_BINS];
    __shared__ uint32_t base[RS_BINS];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
    for (int q = 0; q < RS_BPT; ++q) {
        const uint32_t d = q * RS_THREADS + threadIdx.x;
        base[d] = offs[d * n_tiles + blockIdx.x];
#pragma unroll
        for (int w = 0; w < RS_THREADS / 32; ++w) wc[w][d] = 0;
    }
    __syncthreads();
    const uint32_t t0 = blockIdx.x * RS_TILE;
    for (int r = 0; r < RS_ITEMS; ++r) {
        const uint32_t i = t0 + r * RS_THREADS + threadIdx.x;
        const bool live = i < n;
        const uint64_t key = live ? in[i] : 0ull;
        const uint32_t d = live ? ((uint32_t)(key >> shift) & mask) : (uint32_t)RS_BINS;   // dead lanes form their own group
        const uint32_t peers = __match_any_sync(0xffffffffu, d);
        const uint32_t below = __popc(peers & ((1u << lane) - 1u));
        if (live && below == 0) wc[warp][d] = (uint32_t)__popc(peers);
        __syncthreads();
        uint32_t pre = 0;
        if (live) {
            for (int w = 0; w < warp; ++w) pre += wc[w][d];
            out[base[d] + pre + below] = key;
        }
        __syncthreads();
        // only the digits this round touched have counts: the thread that wrote a count (first lane of its group in its warp)
        // adds it to the digit's base and clears it -- no sweep over all RS_BINS digits per round
        if (live && below == 0) { atomicAdd(&base[d], wc[warp][d]); wc[warp][d] = 0; }
        __syncthreads();
    }
}

// ---- single-pass exclusive scan (decoupled look-back): one launch, no host-known length needed ------------------
// Tiles take tickets from a counter (so every predecessor of a running tile is running or done) and publish
// (epoch | flag | value) in one 64-bit word; a new epoch per call makes the words of earlier calls read as "not yet".
constexpr int LB_THREADS = 512, LB_ITEMS = 16, LB_TILE = LB_THREADS * LB_ITEMS;   // big tiles: the tables are 10^5 - 10^6 elements, and a
                                                                               // tile's look-back costs one L2 round trip per 32 predecessors
constexpr unsigned long long LB_AGG = 1ull, LB_PREFIX = 2ull;

__global__ void __launch_bounds__(LB_THREADS)
k_scan_lb(uint32_t* __restrict__ a, uint32_t n_host, const uint32_t* __restrict__ n_dev, unsigned long long* __restrict__ desc,
          uint32_t* __restrict__ ticket, uint32_t epoch, uint32_t* __restrict__ total_out, uint32_t* __restrict__ total_out2) {
    __shared__ uint32_t s_tile, s_prev, wsum[LB_THREADS / 32];
    const uint32_t n = n_dev ? min(*n_dev, n_host) : n_host;
    if (threadIdx.x == 0) s_tile = atomicAdd(ticket, 1u);
    __syncthreads();
    const uint32_t t = s_tile;
    const uint32_t base = t * LB_TILE + threadIdx.x * LB_ITEMS;
    uint32_t v[LB_ITEMS], sum = 0;
#pragma unroll
    for (int q = 0; q < LB_ITEMS; ++q) { v[q] = base + q < n ? a[base + q] : 0u; sum += v[q]; }
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    uint32_t inc = sum;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) { const uint32_t x = __shfl_up_sync(0xffffffffu, inc, o); if (lane >= o) inc += x; }
    if (lane == 31) wsum[warp] = inc;
    __syncthreads();
    uint32_t wbase = 0, total = 0;
#pragma unroll
    for (int w = 0; w < LB_THREADS / 32; ++w) { if (w < warp) wbase += wsum[w]; total += wsum[w]; }
    if (warp == 0) {
        // look-back by one warp: 32 predecessors per round; the nearest one that already knows its inclusive prefix ends the walk
        const unsigned long long tag = (unsigned long long)epoch << 34;
        volatile unsigned long long* d = desc;
        uint32_t prev = 0;
        if (t == 0) {
            if (lane == 0) d[0] = tag | (LB_PREFIX << 32) | total;
        } else {
            if (lane == 0) d[t] = tag | (LB_AGG << 32) | total;
            int64_t hi = (int64_t)t - 1;                                // lane 0 looks at tile hi, lane 1 at hi - 1, ...
            for (;;) {
                const int64_t p = hi - lane;
                unsigned long long w = 0;
                bool ready = true;
                if (p >= 0) {
                    w = d[p];
                    ready = (w >> 34) == epoch && ((w >> 32) & 3ull) != 0ull;
                }
                if (!__all_sync(0xffffffffu, ready)) continue;          // somebody has not published yet: look again
                const uint32_t is_prefix = __ballot_sync(0xffffffffu, p >= 0 && ((w >> 32) & 3ull) == LB_PREFIX);
                const int stop = is_prefix ? __ffs(is_prefix) - 1 : 31; // nearest tile with an inclusive prefix
                prev += __reduce_add_sync(0xffffffffu, (p >= 0 && lane <= stop) ? (uint32_t)w : 0u);
                if (is_prefix || hi - 32 < 0) break;
                hi -= 32;
            }
            if (lane == 0) d[t] = tag | (LB_PREFIX << 32) | (prev + total);
        }
        if (lane == 0) {
            s_prev = prev;
            if (t == gridDim.x - 1) {                                   // every ticket of this launch has been handed out
                *ticket = 0u;
                if (total_out) *total_out = prev + total;
                if (total_out2) *total_out2 = prev + total;
            }
        }
    }
    __syncthreads();
    uint32_t run = s_prev + wbase + inc - sum;
#pragma unroll
    for (int q = 0; q < LB_ITEMS; ++q) { if (base + q < n) a[base + q] = run; run += v[q]; }
}

// ---- the same scan with ONE grid-wide rendezvous instead of a look-back chain ------------------------------------------
// The tables of this path are 10^5 - 10^6 elements: a few hundred tiles, all resident at once.  Every tile publishes its sum,
// waits until all have (arrive counter), and adds up the sums of the tiles in front of it -- the latency of one global
// round trip instead of one per 32 predecessors.  Only launched when the grid fits the device (the launcher checks); the
// look-back kernel above takes the larger inputs.  gb[0] = arrive, gb[1] = depart (the last tile to leave zeroes both),
// gb[8 + t] = sum of tile t.
constexpr int GS_THREADS = 512, GS_ITEMS = 8, GS_TILE = GS_THREADS * GS_ITEMS, GS_MAX_TILES = 1024;
constexpr int SC_EXTRA = 16 + (8 + GS_MAX_TILES) / 2 + 8;              // 64-bit words behind the descriptors: ticket at +8, gb at +16

__global__ void __launch_bounds__(GS_THREADS)
k_scan_gb(uint32_t* __restrict__ a, uint32_t n_host, const uint32_t* __restrict__ n_dev, uint32_t* __restrict__ gb,
          uint32_t* __restrict__ total_out, uint32_t* __restrict__ total_out2) {
    __shared__ uint32_t wsum[GS_THREADS / 32], wpre[GS_THREADS / 32], s_prev;
    const uint32_t n = n_dev ? min(*n_dev, n_host) : n_host;
    const uint32_t t = blockIdx.x, tiles = gridDim.x;
    const uint32_t base = t * GS_TILE + threadIdx.x * GS_ITEMS;
    uint32_t v[GS_ITEMS], sum = 0;
    if (base + GS_ITEMS <= n) {                                         // two 16-byte loads (the arrays are 256-byte aligned)
        const uint4 x = *reinterpret_cast<const uint4*>(a + base), y = *reinterpret_cast<const uint4*>(a + base + 4);
        v[0] = x.x; v[1] = x.y; v[2] = x.z; v[3] = x.w; v[4] = y.x; v[5] = y.y; v[6] = y.z; v[7] = y.w;
    } else {
#pragma unroll
        for (int q = 0; q < GS_ITEMS; ++q) v[q] = base + q < n ? a[base + q] : 0u;
    }
#pragma unroll
    for (int q = 0; q < GS_ITEMS; ++q) sum += v[q];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    uint32_t inc = sum;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) { const uint32_t x = __shfl_up_sync(0xffffffffu, inc, o); if (lane >= o) inc += x; }
    if (lane == 31) wsum[warp] = inc;
    __syncthreads();
    uint32_t wbase = 0, total = 0;
#pragma unroll
    for (int w = 0; w < GS_THREADS / 32; ++w) { if (w < warp) wbase += wsum[w]; total += wsum[w]; }
    volatile uint32_t* vg = gb;
    if (threadIdx.x == 0) {
        vg[8 + t] = total;
        __threadfence();
        atomicAdd(gb, 1u);
        while (vg[0] < tiles) { }                                       // every tile of the grid is resident (launcher), so this ends
        __threadfence();
    }
    __syncthreads();
    // sums of the tiles in front: GS_THREADS threads, at most GS_MAX_TILES / GS_THREADS values each
    uint32_t part = 0;
    for (uint32_t x = threadIdx.x; x < t; x += GS_THREADS) part += vg[8 + x];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) part += __shfl_down_sync(0xffffffffu, part, o);
    if (lane == 0) wpre[warp] = part;
    __syncthreads();
    if (threadIdx.x == 0) {
        uint32_t prev = 0;
#pragma unroll
        for (int w = 0; w < GS_THREADS / 32; ++w) prev += wpre[w];
        s_prev = prev;
        if (t == tiles - 1) {
            if (total_out) *total_out = prev + total;
            if (total_out2) *total_out2 = prev + total;
        }
        __threadfence();
        if (atomicAdd(gb + 1, 1u) == tiles - 1) { vg[0] = 0u; vg[1] = 0u; }   // the last one out: nobody reads the sums any more
    }
    __syncthreads();
    uint32_t run = s_prev + wbase + inc - sum;
    if (base + GS_ITEMS <= n) {
        uint4 x, y;
        x.x = run; run += v[0]; x.y = run; run += v[1]; x.z = run; run += v[2]; x.w = run; run += v[3];
        y.x = run; run += v[4]; y.y = run; run += v[5]; y.z = run; run += v[6]; y.w = run;
        *reinterpret_cast<uint4*>(a + base) = x; *reinterpret_cast<uint4*>(a + base + 4) = y;
    } else {
#pragma unroll
        for (int q = 0; q < GS_ITEMS; ++q) { if (base + q < n) a[base + q] = run; run += v[q]; }
    }
}

// tiles of k_scan_gb that are resident at once on the current device (the rendezvous needs all of them)
int scan_gb_capacity() {
    static std::atomic<int> cap_of[64];
    int dev = 0;
    cudaGetDevice(&dev);
    if (dev < 0 || dev >= 64) return 0;
    int c = cap_of[dev].load();
    if (c) return c;
    int per_sm = 0, sms = 0;
    cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, (const void*)k_scan_gb, GS_THREADS, 0);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    c = std::max(1, std::min(GS_MAX_TILES, per_sm * sms / 2));          // half of it: other streams may hold SMs (upload-time kernels)
    cap_of[dev].store(c);
    return c;
}

struct Scanner {
    unsigned long long* desc;     // [max tiles], zeroed once
    uint32_t* ticket;             // [1], zero between launches
    uint32_t* epoch;              // host counter
    cudaStream_t st;
    uint32_t* gb;                 // [8 + GS_MAX_TILES] rendezvous words + tile sums of k_scan_gb, zeroed once
    // exclusive scan of a[0..n) in place; n = min(n_host, *n_dev) when n_dev is given; the total goes to total_out (and total_out2)
    void scan(uint32_t* a, uint32_t n_host, const uint32_t* n_dev, uint32_t* total_out, uint32_t* total_out2 = nullptr) const {
        const uint32_t tiles = (n_host + LB_TILE - 1) / LB_TILE;
        if (tiles == 0) { if (total_out) cudaMemsetAsync(total_out, 0, 4, st); if (total_out2) cudaMemsetAsync(total_out2, 0, 4, st); return; }
        const uint32_t gtiles = (n_host + GS_TILE - 1) / GS_TILE;
        if (gb && (int)gtiles <= scan_gb_capacity()) {
            { SPL_LAUNCH; k_scan_gb<<<gtiles, GS_THREADS, 0, st>>>(a, n_host, n_dev, gb, total_out, total_out2); }
            return;
        }
        *epoch = (*epoch + 1u) & 0x3fffffffu;
        if (*epoch == 0u) *epoch = 1u;
        { SPL_LAUNCH; k_scan_lb<<<tiles, LB_THREADS, 0, st>>>(a, n_host, n_dev, desc, ticket, *epoch, total_out, total_out2); }
    }
};

struct Sorter {
    uint32_t* hist;      // [RS_BINS * max_tiles + 1]
    Scanner sc;
    uint32_t* total;     // [1] scratch
    cudaStream_t st;
    // stable sort of a[0..n) on bits [lo, hi); b is the ping-pong buffer; returns the buffer that holds the result
    uint64_t* sort(uint64_t* a, uint64_t* b, uint32_t n, int lo, int hi) const {
        if (n < 2) return a;
        const uint32_t n_tiles = (n + RS_TILE - 1) / RS_TILE;
        // equal digit widths (34 bits = 4 x 9 rather than 10 + 10 + 10 + 4): the histogram of a narrow digit is cheaper to scan
        const int passes = (hi - lo + RS_BITS - 1) / RS_BITS, step = (hi - lo + passes - 1) / passes;
        for (int shift = lo; shift < hi; shift += step) {
            const int width = hi - shift < step ? hi - shift : step;
            const uint32_t mask = (1u << width) - 1u;
            { SPL_LAUNCH; k_rs_hist<<<n_tiles, RS_THREADS, 0, st>>>(a, n, shift, mask, hist, n_tiles); }
            sc.scan(hist, (mask + 1u) * n_tiles, nullptr, total);
            { SPL_LAUNCH; k_rs_scatter<<<n_tiles, RS_THREADS, 0, st>>>(a, b, n, shift, mask, hist, n_tiles); }
            uint64_t* t = a; a = b; b = t;
        }
        return a;
    }
};

__host__ __device__ inline int bits_for_u64(uint64_t v) { int b = 1; while (b < 64 && (v >> b)) ++b; return b; }

// ---- phase A: endpoints -> sites ----------------------------------------------------------------
__global__ void k_gb_keys_a(const int32_t* __restrict__ jc, const int32_t* __restrict__ jl, const int32_t* __restrict__ jr,
                            const uint8_t* __restrict__ js, uint32_t J, int stranded, int pb, int vb, uint64_t* __restrict__ keys) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= J) return;
    const uint64_t sb = (stranded && js[i] == '-') ? 1u : 0u;
    const uint64_t c = (uint64_t)(uint32_t)jc[i] << (pb + 1);
    keys[2 * i] = ((c | ((uint64_t)(uint32_t)jl[i] << 1) | sb) << vb) | (uint64_t)(2 * i);
    keys[2 * i + 1] = ((c | ((uint64_t)(uint32_t)jr[i] << 1) | sb) << vb) | (uint64_t)(2 * i + 1);
}

// flag[e] = 1 when sorted element e starts a new run of (key >> low)
__global__ void k_gb_heads(const uint64_t* __restrict__ k, uint32_t n, int low, uint32_t* __restrict__ flag) {
    const uint32_t e = blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= n) return;
    flag[e] = (e == 0 || (k[e] >> low) != (k[e - 1] >> low)) ? 1u : 0u;
}

__global__ void k_gb_sites(const uint64_t* __restrict__ k, const uint32_t* __restrict__ ex, uint32_t n, int vb, int pb, int stranded,
                           const uint8_t* __restrict__ js, GraphDev g, uint32_t* __restrict__ site_of, uint32_t* __restrict__ inc_eid,
                           uint32_t* __restrict__ counts) {
    const uint32_t e = blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= n) return;
    const uint64_t key = k[e] >> vb;
    const bool head = e == 0 || key != (k[e - 1] >> vb);
    const uint32_t idx = ex[e] - (head ? 0u : 1u);
    const uint32_t eid = (uint32_t)(k[e] & ((1ull << vb) - 1ull));
    site_of[eid] = idx;
    inc_eid[e] = eid;                                                  // endpoint 2 * row + side; its junction partner is eid ^ 1
    g.inc_line[e] = (int32_t)(eid >> 1);
    if (head) {
        const uint32_t line = eid >> 1;
        const int32_t chrom = (int32_t)(key >> (pb + 1));
        const uint8_t st = js[line];
        g.site_chrom[idx] = chrom;
        g.site_pos[idx] = (int32_t)((key >> 1) & ((1ull << pb) - 1ull));
        g.site_strand[idx] = st;                                       // first-seen strand (stable sort keeps row order)
        g.first_line[idx] = (int64_t)line;
        g.site_cls[idx] = !stranded ? 0 : st == '+' ? 1 : st == '-' ? 2 : 3;
        g.inc_off[idx] = (int32_t)e;
    }
    if (e == n - 1) {
        g.inc_off[idx + 1] = (int32_t)n;
        counts[7] = idx + 2u;                                          // S + 1: length of the per-site scans that also want their total
        for (int q = 0; q < 64; ++q) g.site_pos[idx + 1 + q] = INT_MAX;   // tail padding (never matches)
    }
}

// per-chromosome site ranges (the table is sorted by chromosome, so cs_off[c] is a lower bound) and the layout of the
// direct-address bin index, one CTA: the searches run side by side, only the running sum over the chromosomes is serial
__global__ void __launch_bounds__(256) k_gb_chroms(GraphDev g, int n_chrom, uint32_t* __restrict__ counts) {
    const int S = (int)counts[0];
    // one warp per chromosome: 32 probes per round narrow [lo, hi) by a factor of 33 (four dependent loads for a million sites
    // instead of twenty)
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, n_warps = blockDim.x >> 5;
    for (int c = warp; c <= n_chrom; c += n_warps) {
        int lo = 0, hi = S;                                             // first site with chromosome >= c lies in [lo, hi]
        while (hi - lo > 0) {
            const int step = (hi - lo + 32) / 33;                       // probes at lo + (lane + 1) * step - 1
            const int at = min(lo + (lane + 1) * step - 1, hi - 1);
            const bool ge = g.site_chrom[at] >= c;
            const uint32_t bal = __ballot_sync(0xffffffffu, ge);
            if (bal == 0u) { lo = min(lo + 32 * step, hi); if (lo + 0 >= hi) break; continue; }
            const int first = __ffs(bal) - 1;                           // first probe that is already >= c
            hi = min(lo + (first + 1) * step - 1, hi - 1);
            lo = first ? min(lo + first * step, hi) : lo;
            if (step == 1) { lo = hi; break; }
        }
        if (lane == 0) g.cs_off[c] = lo;
    }
    __syncthreads();
    for (int c = threadIdx.x; c < n_chrom; c += blockDim.x) {
        const int32_t s0 = g.cs_off[c], s1 = g.cs_off[c + 1];
        g.sb_base[c] = (s1 > s0 ? (max(g.site_pos[s1 - 1], 0) >> SB_SHIFT) + 1 : 0) + 1;     // bins + sentinel (turned into offsets below)
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        int32_t nb = 0;
        for (int c = 0; c < n_chrom; ++c) { const int32_t v = g.sb_base[c]; g.sb_base[c] = nb; nb += v; }
        g.sb_base[n_chrom] = nb;
        counts[1] = (uint32_t)nb;
    }
}

// direct-address bin index: sb_off[sb_base[c] + b] = first site of chromosome c with position >= b << SB_SHIFT.  A thread owns
// eight consecutive entries (one 32-byte store): one binary search for the first, a forward walk over the site table for the
// rest -- consecutive bins mostly share their site, and a GRCh38-scale index has 5e7 entries.
constexpr int SBF_RUN = 8;
__global__ void __launch_bounds__(256) k_gb_sb_fill(GraphDev g, int n_chrom, const uint32_t* __restrict__ counts) {
    const uint32_t S = counts[0], n_entries = counts[1];
    const uint32_t n_runs = (n_entries + 64u + SBF_RUN - 1) / SBF_RUN;
    for (uint32_t r = blockIdx.x * blockDim.x + threadIdx.x; r < n_runs; r += gridDim.x * blockDim.x) {
        const uint32_t i0 = r * SBF_RUN;
        int32_t out[SBF_RUN];
        int c = -1, s0 = 0, s1 = 0, cur = 0;
        int32_t nb = 0, cb = 0;
#pragma unroll
        for (int q = 0; q < SBF_RUN; ++q) {
            const uint32_t i = i0 + q;
            if (i >= n_entries) { out[q] = (int32_t)S; continue; }
            if (c < 0 || (int32_t)i >= g.sb_base[c + 1]) {              // (re)locate the chromosome of this entry
                int lo = 0, hi = n_chrom;                               // last chromosome with sb_base <= i
                while (hi - lo > 1) { const int mid = (lo + hi) >> 1; if ((uint32_t)g.sb_base[mid] <= i) lo = mid; else hi = mid; }
                c = lo; cb = g.sb_base[c]; nb = g.sb_base[c + 1] - cb - 1;
                s0 = g.cs_off[c]; s1 = g.cs_off[c + 1];
                const int32_t key = ((int32_t)i - cb) << SB_SHIFT;
                int a = s0, e = s1;
                while (a < e) { const int mid = (a + e) >> 1; if (g.site_pos[mid] < key) a = mid + 1; else e = mid; }
                cur = a;
            }
            const int32_t bq = (int32_t)i - cb;
            if (bq >= nb) { out[q] = s1; continue; }                    // the chromosome's sentinel
            const int32_t key = bq << SB_SHIFT;
            while (cur < s1 && g.site_pos[cur] < key) ++cur;
            out[q] = cur;
        }
        int4* dst = reinterpret_cast<int4*>(g.sb_off + i0);            // the array is allocated in whole runs
        dst[0] = make_int4(out[0], out[1], out[2], out[3]);
        dst[1] = make_int4(out[4], out[5], out[6], out[7]);
    }
}

// ---- phase B: Partners / PartnerCounts of every site, straight from its incident endpoints ----------------
// The endpoints of a site are already grouped and in row order (phase A); the junction partner of endpoint e is e ^ 1.
// A site's distinct partners in first-appearance order (G:243-262) are found by one thread per site: degrees are small
// (a splice site has a handful of partners), so the quadratic scan over the incident list stays in L1.
__device__ __forceinline__ uint32_t partner_of(const uint32_t* __restrict__ site_of, const uint32_t* __restrict__ inc_eid, uint32_t k) {
    return site_of[inc_eid[k] ^ 1u];
}
__global__ void k_gb_pt_count(GraphDev g, const uint32_t* __restrict__ counts, const uint32_t* __restrict__ site_of,
                              const uint32_t* __restrict__ inc_eid, uint32_t* __restrict__ npt) {
    const uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= counts[0]) return;
    const uint32_t o = (uint32_t)g.inc_off[t], d = (uint32_t)g.inc_off[t + 1] - o;
    uint32_t u = 0;
    for (uint32_t i = 0; i < d; ++i) {
        const uint32_t p = partner_of(site_of, inc_eid, o + i);
        bool first = true;
        for (uint32_t q = 0; q < i && first; ++q) first = partner_of(site_of, inc_eid, o + q) != p;
        u += first;
    }
    npt[t] = u;
}
// entries of site t: partner site, partner position, and the rows whose score adds to the entry (S:353-355), grouped
__global__ void k_gb_pt_fill(GraphDev g, uint32_t* __restrict__ counts, const uint32_t* __restrict__ site_of,
                             const uint32_t* __restrict__ inc_eid, const uint32_t* __restrict__ pt_off_u, uint32_t* __restrict__ e_src) {
    const uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
    const uint32_t S = counts[0];
    if (t > S) return;
    g.pt_off[t] = (int32_t)pt_off_u[t];
    g.pt_off64[t] = (int64_t)pt_off_u[t];
    if (t == S) return;
    const uint32_t o = (uint32_t)g.inc_off[t], d = (uint32_t)g.inc_off[t + 1] - o;
    uint32_t x = pt_off_u[t], w = o;
    for (uint32_t i = 0; i < d; ++i) {
        const uint32_t p = partner_of(site_of, inc_eid, o + i);
        bool first = true;
        for (uint32_t q = 0; q < i && first; ++q) first = partner_of(site_of, inc_eid, o + q) != p;
        if (!first) continue;
        g.pt_site[x] = (int32_t)p;
        g.pc_pos[x] = g.site_pos[p];
        g.einc_beg[x] = (int32_t)w;
        for (uint32_t q = i; q < d; ++q)
            if (partner_of(site_of, inc_eid, o + q) == p) g.einc_line[w++] = (int32_t)(inc_eid[o + q] >> 1);
        g.einc_end[x] = (int32_t)w;
        e_src[x] = t;
        ++x;
    }
}

// ---- phase D: competitors (S:364-372): sorted distinct positions of the partners' partners, own position excluded ---
// One thread per site, selection by repeated minimum: every round finds the smallest candidate above the last one written.
__device__ __forceinline__ int32_t next_competitor(const GraphDev& g, const int32_t* __restrict__ pt_off, uint32_t t, int32_t tp, int32_t last) {
    int32_t best = INT_MAX;
    for (int a = pt_off[t]; a < pt_off[t + 1]; ++a) {
        const int p = g.pt_site[a];
        for (int q = pt_off[p]; q < pt_off[p + 1]; ++q) {
            const int32_t c = g.pc_pos[q];                                // position of the partner's partner
            if (c != tp && c > last && c < best) best = c;
        }
    }
    return best;
}
__global__ void k_gb_cp_count(GraphDev g, const uint32_t* __restrict__ counts, uint32_t* __restrict__ ncp) {
    const uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= counts[0]) return;
    const int32_t tp = g.site_pos[t];
    uint32_t u = 0;
    for (int32_t last = INT_MIN;;) {
        last = next_competitor(g, g.pt_off, t, tp, last);
        if (last == INT_MAX) break;
        ++u;
    }
    ncp[t] = u;
}
__global__ void k_gb_cp_fill(GraphDev g, uint32_t* __restrict__ counts, const uint32_t* __restrict__ cp_off_u, uint32_t cap) {
    const uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
    const uint32_t S = counts[0];
    if (t > S) return;
    g.cp_off[t] = (int32_t)cp_off_u[t];
    g.cp_off64[t] = (int64_t)cp_off_u[t];
    if (t == S) { if (cp_off_u[S] > cap) counts[6] = 1u; return; }          // the competitor array is too small: the host re-runs with room
    const int32_t tp = g.site_pos[t];
    uint32_t x = cp_off_u[t];
    for (int32_t last = INT_MIN;;) {
        last = next_competitor(g, g.pt_off, t, tp, last);
        if (last == INT_MAX) break;
        if (x < cap) g.cp_pos[x] = last;
        ++x;
    }
}

// ---- phase E: reverse-partner index ---------------------------------------------------------------
// the list hangs off the FIRST site index sharing (chromosome, position) with the partner; the clean regime has at
// most two sites per position ('+' then '-')
__device__ __forceinline__ uint32_t anchor_of(const GraphDev& g, uint32_t p) {
    return (p > 0 && g.site_pos[p - 1] == g.site_pos[p] && g.site_chrom[p - 1] == g.site_chrom[p]) ? p - 1 : p;
}
__global__ void k_gb_rp_count(GraphDev g, const uint32_t* __restrict__ counts, uint32_t* __restrict__ rp_cnt) {
    const uint32_t x = blockIdx.x * blockDim.x + threadIdx.x;
    if (x >= counts[2]) return;
    atomicAdd(rp_cnt + anchor_of(g, (uint32_t)g.pt_site[x]), 1u);
}
__global__ void k_gb_rp_fill(GraphDev g, const uint32_t* __restrict__ counts, const uint32_t* __restrict__ e_src, const uint32_t* __restrict__ rp_off_u,
                             uint32_t* __restrict__ rp_cur) {
    const uint32_t x = blockIdx.x * blockDim.x + threadIdx.x;
    if (x <= counts[0]) g.rp_off[x] = (int32_t)rp_off_u[x];
    if (x >= counts[2]) return;
    const uint32_t a = anchor_of(g, (uint32_t)g.pt_site[x]);
    const uint32_t t = e_src[x];
    g.rp_site[rp_off_u[a] + atomicAdd(rp_cur + a, 1u)] = (int32_t)t;      // order inside a list does not matter: only counted
    if (g.cp_off[t + 1] > g.cp_off[t]) g.site_hot[a] = 1;
}

inline uint32_t cdiv(uint32_t a, uint32_t b) { return (a + b - 1) / b; }

struct Carve {
    size_t off = 0;
    template <class T> size_t take(size_t n) {
        off = (off + 255) & ~(size_t)255;
        const size_t o = off;
        off += n * sizeof(T);
        return o;
    }
};

// ---- K1 as ONE persistent cooperative kernel -----------------------------------------------------------------------
// The launches above are 3 - 17 us each for tables of 10^5 - 10^6 keys: two dozen of them have a floor of ~0.2 ms whatever the
// size of the table (DESIGN section 9).  Here one CTA per SM walks through the same phases, separated by grid-wide barriers
// (14 of them) instead of kernel boundaries; every CTA owns one contiguous slice of the keys and, later, of the sites (a warp
// one run of the slice's keys in the sort, a thread one run of the slice's sites in the per-site phases: no block-wide
// synchronisation inside the loops, the warps hide each other's latency):
//   keys -> 3 x [histogram | B | per-digit scan over the CTAs | B | digit bases, ranked scatter | B]
//        -> heads counted | B | site indices, site columns | B | (last CTA: chromosome ranges + bin layout)
//        -> Partners counted | B | Partners filled, reverse-partner counts | B | competitors counted | B
//        -> competitors filled, reverse partners filled, hot flags.
// The bin index (up to 5e7 entries on GRCh38) keeps its own wide launch behind it.  Launched with
// cudaLaunchCooperativeKernel (co-residency guaranteed by the driver); the launch-per-phase path above stays as the fallback
// (SPLISER_K1_LAUNCHES=1, or a device without cooperative launch) and the two are held to the same table by the tests.
constexpr int CO_THREADS = 512, CO_WARPS = CO_THREADS / 32, CO_MAX_G = CO_THREADS, CO_STAMPS = 24, CO_KB = 4, CO_WL = RS_BINS / 2;
static_assert(RS_BINS == 2 * CO_THREADS, "digit prefix: two digits per thread");
constexpr size_t CO_SMEM = ((size_t)CO_WARPS * RS_BINS + 32 + 2 * CO_MAX_G) * sizeof(uint32_t);

struct CoopArgs {
    const int32_t *jc, *jl, *jr;
    const uint8_t* js;
    uint32_t J;
    int stranded, pb, vb, lo, hi, n_chrom;
    uint64_t *ka, *kb;
    uint32_t *hist;                  // [RS_BINS * G], digit-major
    uint32_t *dtot;                  // [RS_BINS]
    uint32_t *parts;                 // [4][CO_MAX_G] per-CTA sums: heads, Partners entries, competitors, reverse partners
    uint32_t *bar;                   // [0] arrive (monotonic inside a launch), [1] depart; zero between launches
    uint32_t *cnt;                   // the d_cnt words of the launch-per-phase path
    uint32_t *stamps;                // [CO_STAMPS] globaltimer (ns, low word) of CTA 0 after every barrier, or null
    uint32_t *site_of, *inc_eid, *e_src, *ncp, *rp_cnt, *rp_cur, *loc_rp;
    uint32_t cap;
    GraphDev g;
};

__device__ __forceinline__ void co_grid_sync(uint32_t* bar, uint32_t& target) {
    __syncthreads();
    if (threadIdx.x == 0) {
        target += gridDim.x;
        __threadfence();
        atomicAdd(bar, 1u);
        while (*(volatile uint32_t*)bar < target) { }
        __threadfence();
    }
    __syncthreads();
}

__device__ __forceinline__ void co_stamp(uint32_t* stamps, int k) {
    if (stamps && k < CO_STAMPS && blockIdx.x == 0 && threadIdx.x == 0) {
        unsigned long long t;
        asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
        stamps[k] = (uint32_t)t;
    }
}

// exclusive prefix of one value per thread over the CTA; total = sum over the CTA (two __syncthreads: s_w is free again after it)
__device__ __forceinline__ uint32_t co_block_excl(uint32_t v, uint32_t* s_w, uint32_t& total) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    uint32_t inc = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) { const uint32_t x = __shfl_up_sync(0xffffffffu, inc, o); if (lane >= o) inc += x; }
    if (lane == 31) s_w[warp] = inc;
    __syncthreads();
    uint32_t wbase = 0, tot = 0;
#pragma unroll
    for (int w = 0; w < CO_WARPS; ++w) { const uint32_t x = s_w[w]; if (w < warp) wbase += x; tot += x; }
    __syncthreads();
    total = tot;
    return wbase + inc - v;
}

// exclusive prefix of v over the lanes of the warp; total = the warp's sum
__device__ __forceinline__ uint32_t co_warp_excl(uint32_t v, uint32_t& total) {
    const int lane = threadIdx.x & 31;
    uint32_t inc = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) { const uint32_t x = __shfl_up_sync(0xffffffffu, inc, o); if (lane >= o) inc += x; }
    total = __shfl_sync(0xffffffffu, inc, 31);
    return inc - v;
}
// exclusive prefix of one (warp-uniform) value per warp over the warps of the CTA; total = the CTA's sum
__device__ __forceinline__ uint32_t co_warps_excl(uint32_t wtotal, uint32_t* s_w, uint32_t& total) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    if (lane == 0) s_w[warp] = wtotal;
    __syncthreads();
    uint32_t wbase = 0, tot = 0;
#pragma unroll
    for (int w = 0; w < CO_WARPS; ++w) { const uint32_t x = s_w[w]; if (w < warp) wbase += x; tot += x; }
    __syncthreads();
    total = tot;
    return wbase;
}

// after a barrier: s_pre[c] = sum of part[0..c) for every CTA c, total = sum of all; returns this CTA's prefix
__device__ __forceinline__ uint32_t co_parts_prefix(const uint32_t* part, uint32_t* s_pre, uint32_t* s_w, uint32_t& total) {
    const uint32_t v = threadIdx.x < gridDim.x ? __ldcg(part + threadIdx.x) : 0u;
    const uint32_t ex = co_block_excl(v, s_w, total);
    if (threadIdx.x < gridDim.x) s_pre[threadIdx.x] = ex;
    __syncthreads();
    return s_pre[blockIdx.x];
}

__device__ __forceinline__ uint32_t co_partner(const CoopArgs& a, uint32_t k) { return a.site_of[a.inc_eid[k] ^ 1u]; }

// the general per-site loops (any degree), as in k_gb_pt_count / k_gb_pt_fill / k_gb_cp_count
__device__ __forceinline__ uint32_t co_pt_count_site(const CoopArgs& a, uint32_t o, uint32_t d) {
    uint32_t u = 0;
    for (uint32_t i = 0; i < d; ++i) {
        const uint32_t p = co_partner(a, o + i);
        bool first = true;
        for (uint32_t q = 0; q < i && first; ++q) first = co_partner(a, o + q) != p;
        u += first;
    }
    return u;
}
__device__ __forceinline__ uint32_t co_pt_fill_site(const CoopArgs& a, const GraphDev& g, uint32_t t, uint32_t o, uint32_t d, uint32_t x) {
    uint32_t w = o;
    for (uint32_t i = 0; i < d; ++i) {
        const uint32_t p = co_partner(a, o + i);
        bool first = true;
        for (uint32_t q = 0; q < i && first; ++q) first = co_partner(a, o + q) != p;
        if (!first) continue;
        g.pt_site[x] = (int32_t)p;
        g.pc_pos[x] = g.site_pos[p];
        g.einc_beg[x] = (int32_t)w;
        for (uint32_t q = i; q < d; ++q)
            if (co_partner(a, o + q) == p) g.einc_line[w++] = (int32_t)(a.inc_eid[o + q] >> 1);
        g.einc_end[x] = (int32_t)w;
        a.e_src[x] = t;
        atomicAdd(a.rp_cnt + anchor_of(g, p), 1u);
        ++x;
    }
    return x;
}
__device__ __forceinline__ uint32_t co_cp_count_site(const GraphDev& g, uint32_t t) {
    const int32_t tp = g.site_pos[t];
    uint32_t u = 0;
    for (int32_t last = INT_MIN;;) {
        last = next_competitor(g, g.pt_off, t, tp, last);
        if (last == INT_MAX) break;
        ++u;
    }
    return u;
}

__global__ void __launch_bounds__(CO_THREADS, 2) k_gb_coop(const CoopArgs a) {
    extern __shared__ __align__(16) uint32_t co_sm[];
    uint32_t (*wc)[RS_BINS] = reinterpret_cast<uint32_t (*)[RS_BINS]>(co_sm);      // [CO_WARPS][RS_BINS]: counts, then bases, per warp
    uint32_t* s_w = co_sm + CO_WARPS * RS_BINS;                                    // [32]
    uint32_t* s_pre = s_w + 32;                                                    // [CO_MAX_G]
    uint32_t* s_pre2 = s_pre + CO_MAX_G;                                           // [CO_MAX_G]
    const uint32_t G = gridDim.x, c = blockIdx.x, tid = threadIdx.x;
    const int lane = tid & 31, warp = tid >> 5;
    const uint32_t J = a.J, n2 = 2u * J;
    const GraphDev& g = a.g;
    const int vb = a.vb, pb = a.pb;
    uint32_t target = 0;
    int stamp = 0;
    co_stamp(a.stamps, stamp++);

    // ---- scratch that the later phases add into; endpoint keys of this CTA's slice
    for (uint32_t i = c * CO_THREADS + tid; i < n2 + 64u; i += G * CO_THREADS) g.site_hot[i] = 0;
    for (uint32_t i = c * CO_THREADS + tid; i < n2 + 4u; i += G * CO_THREADS) { a.rp_cnt[i] = 0u; a.rp_cur[i] = 0u; }
    if (c == 0 && tid == 0) a.cnt[6] = 0u;
    if (c == 0) for (int ch = tid; ch <= a.n_chrom; ch += CO_THREADS) g.sb_base[ch] = 1;      // a chromosome without sites: its sentinel bin
    const uint32_t K = (n2 + G - 1) / G;                                           // keys per CTA
    const uint32_t k0 = min(c * K, n2), k1 = min(k0 + K, n2);
    const uint32_t Kw = (K + CO_WARPS - 1) / CO_WARPS;                             // ... per warp: [w0, w1), in index order over the warps
    const uint32_t w0 = min(k0 + (uint32_t)warp * Kw, k1), w1 = min(w0 + Kw, k1);
    for (uint32_t e = w0 + lane; e < w1; e += 32) {
        const uint32_t i = e >> 1;
        const uint64_t sb = (a.stranded && a.js[i] == '-') ? 1u : 0u;
        const uint64_t ch = (uint64_t)(uint32_t)a.jc[i] << (pb + 1);
        const uint32_t pos = (uint32_t)((e & 1u) ? a.jr[i] : a.jl[i]);
        a.ka[e] = ((ch | ((uint64_t)pos << 1) | sb) << vb) | (uint64_t)e;
    }
    __syncwarp();

    // ---- stable LSD radix sort.  Every warp ranks its own run of keys: counts per (warp, digit) in shared memory, the CTA's
    // sums go through the grid-wide digit scan, come back as the CTA's bases, and are turned into per-warp bases in place.
    uint64_t* in = a.ka;
    uint64_t* out = a.kb;
    {
        const int passes = (a.hi - a.lo + RS_BITS - 1) / RS_BITS, step = (a.hi - a.lo + passes - 1) / passes;
        for (int shift = a.lo; shift < a.hi; shift += step) {
            const int width = a.hi - shift < step ? a.hi - shift : step;
            const uint32_t nb = 1u << width, mask = nb - 1u;
            for (uint32_t i = tid; i < (uint32_t)(CO_WARPS * RS_BINS); i += CO_THREADS) co_sm[i] = 0u;
            __syncthreads();
            for (uint32_t eb = w0; eb < w1; eb += 32 * CO_KB) {                    // CO_KB loads in flight per lane, then the counts
                uint64_t kr[CO_KB];
#pragma unroll
                for (int q = 0; q < CO_KB; ++q) { const uint32_t e = eb + q * 32 + lane; kr[q] = e < w1 ? in[e] : 0ull; }
#pragma unroll
                for (int q = 0; q < CO_KB; ++q) if (eb + q * 32 + lane < w1) atomicAdd(&wc[warp][(uint32_t)(kr[q] >> shift) & mask], 1u);
            }
            __syncthreads();
            for (uint32_t d = tid; d < nb; d += CO_THREADS) {
                uint32_t h = 0;
#pragma unroll
                for (int w = 0; w < CO_WARPS; ++w) h += wc[w][d];
                a.hist[d * G + c] = h;
            }
            co_grid_sync(a.bar, target);
            co_stamp(a.stamps, stamp++);
            // one warp per digit: exclusive scan of the digit's counts over the CTAs, digit total
            for (uint32_t d = c + G * (uint32_t)warp; d < nb; d += G * CO_WARPS) {
                uint32_t v[CO_MAX_G / 32];
#pragma unroll
                for (int q = 0; q < CO_MAX_G / 32; ++q) { const uint32_t x = q * 32 + lane; v[q] = x < G ? a.hist[d * G + x] : 0u; }
                uint32_t run = 0;
#pragma unroll
                for (int q = 0; q < CO_MAX_G / 32; ++q) {
                    if ((uint32_t)(q * 32) >= G) break;
                    const uint32_t x = q * 32 + lane;
                    uint32_t inc = v[q];
#pragma unroll
                    for (int o = 1; o < 32; o <<= 1) { const uint32_t y = __shfl_up_sync(0xffffffffu, inc, o); if (lane >= o) inc += y; }
                    if (x < G) a.hist[d * G + x] = run + inc - v[q];
                    run += __shfl_sync(0xffffffffu, inc, 31);
                }
                if (lane == 0) a.dtot[d] = run;
            }
            co_grid_sync(a.bar, target);
            co_stamp(a.stamps, stamp++);
            {   // base of digit d for this CTA = keys with a smaller digit + keys with digit d in the CTAs in front; then per warp
                const uint32_t d0 = 2u * tid;
                const uint32_t v0 = d0 < nb ? a.dtot[d0] : 0u, v1 = d0 + 1u < nb ? a.dtot[d0 + 1u] : 0u;
                const uint32_t h0 = d0 < nb ? a.hist[d0 * G + c] : 0u, h1 = d0 + 1u < nb ? a.hist[(d0 + 1u) * G + c] : 0u;
                uint32_t tot;
                const uint32_t ex = co_block_excl(v0 + v1, s_w, tot);
                if (d0 < nb) {
                    uint32_t b = ex + h0;
#pragma unroll
                    for (int w = 0; w < CO_WARPS; ++w) { const uint32_t t = wc[w][d0]; wc[w][d0] = b; b += t; }
                }
                if (d0 + 1u < nb) {
                    uint32_t b = ex + v0 + h1;
#pragma unroll
                    for (int w = 0; w < CO_WARPS; ++w) { const uint32_t t = wc[w][d0 + 1u]; wc[w][d0 + 1u] = b; b += t; }
                }
            }
            __syncthreads();
            for (uint32_t eb = w0; eb < w1; eb += 32 * CO_KB) {                    // element order = (warp, round, lane) = index order
                uint64_t kr[CO_KB];
#pragma unroll
                for (int q = 0; q < CO_KB; ++q) { const uint32_t e = eb + q * 32 + lane; kr[q] = e < w1 ? in[e] : 0ull; }
#pragma unroll
                for (int q = 0; q < CO_KB; ++q) {
                    if (eb + q * 32 >= w1) break;                                   // warp-uniform
                    const bool live = eb + q * 32 + lane < w1;
                    const uint64_t key = kr[q];
                    const uint32_t d = live ? ((uint32_t)(key >> shift) & mask) : (uint32_t)RS_BINS;   // dead lanes form their own group
                    const uint32_t peers = __match_any_sync(0xffffffffu, d);
                    const uint32_t below = __popc(peers & ((1u << lane) - 1u));
                    uint32_t at = 0;
                    if (live) at = wc[warp][d];
                    __syncwarp();
                    if (live) {
                        out[at + below] = key;
                        if (below == 0) wc[warp][d] = at + (uint32_t)__popc(peers);
                    }
                    __syncwarp();
                }
            }
            co_grid_sync(a.bar, target);
            co_stamp(a.stamps, stamp++);
            uint64_t* t = in; in = out; out = t;
        }
    }
    const uint64_t* sk = in;

    // ---- sites: heads of the runs of equal (chromosome, position, strand bit).  The warp keeps its run [w0, w1) of the sorted keys,
    // lane-consecutive (coalesced loads and stores); heads are ranked by ballot inside the warp, over the warps by their totals
    const uint32_t full = 0xffffffffu, lt_mask = (1u << lane) - 1u;
    uint32_t heads_in_front;                                                        // ... of this warp's first key, inside the CTA
    {
        uint32_t h = 0;
        for (uint32_t eb = w0; eb < w1; eb += 32 * CO_KB) {
            uint64_t kr[CO_KB], kp[CO_KB];
#pragma unroll
            for (int q = 0; q < CO_KB; ++q) {
                const uint32_t e = eb + q * 32 + lane;
                kr[q] = e < w1 ? sk[e] : 0ull; kp[q] = (e < w1 && e > 0) ? sk[e - 1] : 0ull;
            }
#pragma unroll
            for (int q = 0; q < CO_KB; ++q) {
                const uint32_t e = eb + q * 32 + lane;
                h += __popc(__ballot_sync(full, e < w1 && (e == 0 || (kr[q] >> vb) != (kp[q] >> vb))));
            }
        }
        uint32_t tot;
        heads_in_front = co_warps_excl(h, s_w, tot);
        if (tid == 0) a.parts[0 * CO_MAX_G + c] = tot;
    }
    co_grid_sync(a.bar, target);
    co_stamp(a.stamps, stamp++);
    uint32_t S;
    {
        uint32_t run = co_parts_prefix(a.parts + 0 * CO_MAX_G, s_pre, s_w, S) + heads_in_front;   // heads in front of the round
        for (uint32_t eb = w0; eb < w1; eb += 32 * CO_KB) {
            uint64_t kr[CO_KB], kp[CO_KB];
            uint8_t sr[CO_KB];
#pragma unroll
            for (int q = 0; q < CO_KB; ++q) {
                const uint32_t e = eb + q * 32 + lane;
                kr[q] = e < w1 ? sk[e] : 0ull; kp[q] = (e < w1 && e > 0) ? sk[e - 1] : 0ull;
            }
#pragma unroll
            for (int q = 0; q < CO_KB; ++q) sr[q] = eb + q * 32 + lane < w1 ? a.js[(uint32_t)(kr[q] & ((1ull << vb) - 1ull)) >> 1] : (uint8_t)0;
#pragma unroll
            for (int q = 0; q < CO_KB; ++q) {
                if (eb + q * 32 >= w1) break;                                       // warp-uniform
                const uint32_t e = eb + q * 32 + lane;
                const bool live = e < w1;
                const uint64_t kk = kr[q];
                const uint64_t key = kk >> vb;
                const bool head = live && (e == 0 || key != (kp[q] >> vb));
                const uint32_t hb = __ballot_sync(full, head);
                if (live) {
                    const uint32_t idx = run + __popc(hb & lt_mask) + (head ? 1u : 0u) - 1u;
                    const uint32_t eid = (uint32_t)(kk & ((1ull << vb) - 1ull));
                    a.site_of[eid] = idx;
                    a.inc_eid[e] = eid;                                             // endpoint 2 * row + side; its junction partner is eid ^ 1
                    g.inc_line[e] = (int32_t)(eid >> 1);
                    if (head) {
                        const uint32_t line = eid >> 1;
                        const uint8_t st = sr[q];
                        // chromosome ranges of the table and the bin count of every chromosome, where the chromosome changes
                        const int ccur = (int)(key >> (pb + 1)), cprev = e == 0 ? -1 : (int)((kp[q] >> vb) >> (pb + 1));
                        if (ccur != cprev) {
                            for (int ch = cprev + 1; ch <= ccur; ++ch) g.cs_off[ch] = (int32_t)idx;
                            if (cprev >= 0) g.sb_base[cprev] = (int32_t)((((kp[q] >> vb) >> 1) & ((1ull << pb) - 1ull)) >> SB_SHIFT) + 2;   // bins + sentinel
                        }
                        g.site_chrom[idx] = (int32_t)(key >> (pb + 1));
                        g.site_pos[idx] = (int32_t)((key >> 1) & ((1ull << pb) - 1ull));
                        g.site_strand[idx] = st;                                    // first-seen strand (stable sort keeps row order)
                        g.first_line[idx] = (int64_t)line;
                        g.site_cls[idx] = !a.stranded ? 0 : st == '+' ? 1 : st == '-' ? 2 : 3;
                        g.inc_off[idx] = (int32_t)e;
                    }
                    if (e == n2 - 1u) {                                             // the last key closes the last chromosome with sites
                        const int ccur = (int)(key >> (pb + 1));
                        for (int ch = ccur + 1; ch <= a.n_chrom; ++ch) g.cs_off[ch] = (int32_t)S;
                        g.sb_base[ccur] = (int32_t)(((key >> 1) & ((1ull << pb) - 1ull)) >> SB_SHIFT) + 2;
                    }
                }
                run += __popc(hb);
            }
        }
        if (c == 0 && tid < 64) g.site_pos[S + tid] = INT_MAX;                     // tail padding (never matches)
        if (c == 0 && tid == 0) { g.inc_off[S] = (int32_t)n2; a.cnt[0] = S; a.cnt[7] = S + 1u; }
    }
    co_grid_sync(a.bar, target);
    co_stamp(a.stamps, stamp++);

    // ---- layout of the bin index: running sum of the chromosomes' bin counts, one warp of the last CTA (only k_gb_sb_fill reads it)
    if (c == G - 1 && warp == 0) {
        uint32_t nbins = 0;
        for (int cb0 = 0; cb0 < a.n_chrom; cb0 += 32) {
            const int ch = cb0 + lane;
            const uint32_t v = ch < a.n_chrom ? (uint32_t)g.sb_base[ch] : 0u;
            uint32_t wt;
            const uint32_t ex = co_warp_excl(v, wt);
            if (ch < a.n_chrom) g.sb_base[ch] = (int32_t)(nbins + ex);
            nbins += wt;
        }
        if (lane == 0) { g.sb_base[a.n_chrom] = (int32_t)nbins; a.cnt[1] = nbins; }
    }

    // ---- per-site phases: CTA c owns the sites [s0, s1), warp w the run [t0, t1) of them, lane-consecutive
    // Every loop below takes CO_KB rounds of 32 sites (or entries) at a time and loads level by level -- all of a level's loads are in
    // flight together.  Sites of degree one (nearly all of them) take the short way, the others the general loops of the
    // launch-per-phase kernels.
    const uint32_t Ks = max((S + G - 1) / G, 1u);
    const uint32_t s0 = min(c * Ks, S), s1 = min(s0 + Ks, S);
    const uint32_t Kws = (Ks + CO_WARPS - 1) / CO_WARPS;
    const uint32_t t0 = min(s0 + (uint32_t)warp * Kws, s1), t1 = min(t0 + Kws, s1);
    // sites that need the general loops go to the warp's list (the sort's counters are free now) and are taken 32 at a time: a warp
    // pays the long dependent chains once per 32 such sites, not once per round that holds one
    uint32_t* wl = co_sm + (uint32_t)warp * RS_BINS;                                // [CO_WL] (site, offset) pairs
    uint32_t ln = 0;                                                                // entries in the list (warp-uniform)
    uint32_t pt_front;                                                              // Partners entries in front of site t0, inside the CTA
    {
        uint32_t run = 0;
        auto drain = [&]() {
            __syncwarp();
            for (uint32_t i0 = 0; i0 < ln; i0 += 32) {
                uint32_t u = 0;
                if (i0 + lane < ln) {
                    const uint32_t t = wl[2u * (i0 + lane)];
                    const uint32_t o = (uint32_t)g.inc_off[t];
                    u = co_pt_count_site(a, o, (uint32_t)g.inc_off[t + 1] - o);
                    a.ncp[t] = u;
                }
                run += __reduce_add_sync(full, u);
            }
            __syncwarp();
            ln = 0;
        };
        for (uint32_t tb = t0; tb < t1; tb += 32 * CO_KB) {
            uint32_t io[CO_KB], io1[CO_KB];
#pragma unroll
            for (int q = 0; q < CO_KB; ++q) {
                const uint32_t t = tb + q * 32 + lane;
                io[q] = t < t1 ? (uint32_t)g.inc_off[t] : 0u; io1[q] = t < t1 ? (uint32_t)g.inc_off[t + 1] : 0u;
            }
#pragma unroll
            for (int q = 0; q < CO_KB; ++q) {
                const uint32_t t = tb + q * 32 + lane;
                const uint32_t d = io1[q] - io[q];
                const bool one = t < t1 && d == 1u, gen = t < t1 && d != 1u;
                if (one) a.ncp[t] = 1u;                                             // ncp: scratch until the competitors
                run += __popc(__ballot_sync(full, one));
                const uint32_t gm = __ballot_sync(full, gen);
                if (gm) {
                    if (ln + 32u > (uint32_t)CO_WL) drain();
                    if (gen) wl[2u * (ln + __popc(gm & lt_mask))] = t;
                    ln += __popc(gm);
                }
            }
        }
        drain();
        uint32_t tot;
        pt_front = co_warps_excl(run, s_w, tot);
        if (tid == 0) a.parts[1 * CO_MAX_G + c] = tot;
    }
    co_grid_sync(a.bar, target);
    co_stamp(a.stamps, stamp++);
    uint32_t E;
    {
        uint32_t xrun = co_parts_prefix(a.parts + 1 * CO_MAX_G, s_pre, s_w, E) + pt_front;
        auto drain = [&]() {
            __syncwarp();
            for (uint32_t i = lane; i < ln; i += 32) {
                const uint32_t t = wl[2u * i], x = wl[2u * i + 1u];
                const uint32_t o = (uint32_t)g.inc_off[t];
                co_pt_fill_site(a, g, t, o, (uint32_t)g.inc_off[t + 1] - o, x);
            }
            __syncwarp();
            ln = 0;
        };
        for (uint32_t tb = t0; tb < t1; tb += 32 * CO_KB) {
            uint32_t io[CO_KB], io1[CO_KB], uu[CO_KB], eid[CO_KB], pp[CO_KB];
            int32_t pos[CO_KB], posm[CO_KB], chr[CO_KB], chrm[CO_KB];
#pragma unroll
            for (int q = 0; q < CO_KB; ++q) {
                const uint32_t t = tb + q * 32 + lane;
                io[q] = t < t1 ? (uint32_t)g.inc_off[t] : 0u; io1[q] = t < t1 ? (uint32_t)g.inc_off[t + 1] : 0u; uu[q] = t < t1 ? a.ncp[t] : 0u;
            }
#pragma unroll
            for (int q = 0; q < CO_KB; ++q) eid[q] = tb + q * 32 + lane < t1 ? a.inc_eid[io[q]] : 0u;
#pragma unroll
            for (int q = 0; q < CO_KB; ++q) pp[q] = tb + q * 32 + lane < t1 ? a.site_of[eid[q] ^ 1u] : 0u;
#pragma unroll
            for (int q = 0; q < CO_KB; ++q) {
                const bool lv = tb + q * 32 + lane < t1 && io1[q] - io[q] == 1u;
                pos[q] = lv ? g.site_pos[pp[q]] : 0; chr[q] = lv ? g.site_chrom[pp[q]] : 0;
                posm[q] = lv && pp[q] > 0 ? g.site_pos[pp[q] - 1] : -1; chrm[q] = lv && pp[q] > 0 ? g.site_chrom[pp[q] - 1] : -1;
            }
#pragma unroll
            for (int q = 0; q < CO_KB; ++q) {
                if (tb + q * 32 >= t1) break;                                       // warp-uniform
                const uint32_t t = tb + q * 32 + lane;
                uint32_t wt;
                const uint32_t x = xrun + co_warp_excl(uu[q], wt);
                xrun += wt;
                const uint32_t o = io[q], d = io1[q] - o;
                const bool live = t < t1, gen = live && d != 1u;
                if (live) { g.pt_off[t] = (int32_t)x; g.pt_off64[t] = (int64_t)x; }
                if (live && !gen) {
                    g.pt_site[x] = (int32_t)pp[q];
                    g.pc_pos[x] = pos[q];
                    g.einc_beg[x] = (int32_t)o;
                    g.einc_line[o] = (int32_t)(eid[q] >> 1);
                    g.einc_end[x] = (int32_t)(o + 1u);
                    a.e_src[x] = t;
                    atomicAdd(a.rp_cnt + ((pp[q] > 0 && posm[q] == pos[q] && chrm[q] == chr[q]) ? pp[q] - 1u : pp[q]), 1u);
                }
                const uint32_t gm = __ballot_sync(full, gen);
                if (gm) {
                    if (ln + 32u > (uint32_t)CO_WL) drain();
                    if (gen) { const uint32_t i = ln + __popc(gm & lt_mask); wl[2u * i] = t; wl[2u * i + 1u] = x; }
                    ln += __popc(gm);
                }
            }
        }
        drain();
        if (c == 0 && tid == 0) { g.pt_off[S] = (int32_t)E; g.pt_off64[S] = (int64_t)E; a.cnt[2] = E; }
    }
    co_grid_sync(a.bar, target);
    co_stamp(a.stamps, stamp++);
    uint32_t cp_front;
    {   // competitors counted; the reverse-partner counts of the own sites are final since the barrier
        uint32_t run = 0, run2 = 0;
        auto drain = [&]() {
            __syncwarp();
            for (uint32_t i0 = 0; i0 < ln; i0 += 32) {
                uint32_t u = 0;
                if (i0 + lane < ln) {
                    const uint32_t t = wl[2u * (i0 + lane)];
                    u = co_cp_count_site(g, t);
                    a.ncp[t] = u;
                }
                run += __reduce_add_sync(full, u);
            }
            __syncwarp();
            ln = 0;
        };
        for (uint32_t tb = t0; tb < t1; tb += 32 * CO_KB) {
            uint32_t xo[CO_KB], xo1[CO_KB], pp[CO_KB], po0[CO_KB], po1[CO_KB], rc[CO_KB];
#pragma unroll
            for (int q = 0; q < CO_KB; ++q) {
                const uint32_t t = tb + q * 32 + lane;
                xo[q] = t < t1 ? (uint32_t)g.pt_off[t] : 0u; xo1[q] = t < t1 ? (uint32_t)g.pt_off[t + 1] : 0u; rc[q] = t < t1 ? a.rp_cnt[t] : 0u;
            }
#pragma unroll
            for (int q = 0; q < CO_KB; ++q) pp[q] = tb + q * 32 + lane < t1 ? (uint32_t)g.pt_site[xo[q]] : 0u;
#pragma unroll
            for (int q = 0; q < CO_KB; ++q) {
                const bool lv = tb + q * 32 + lane < t1;
                po0[q] = lv ? (uint32_t)g.pt_off[pp[q]] : 0u; po1[q] = lv ? (uint32_t)g.pt_off[pp[q] + 1u] : 0u;
            }
#pragma unroll
            for (int q = 0; q < CO_KB; ++q) {
                if (tb + q * 32 >= t1) break;                                       // warp-uniform
                const uint32_t t = tb + q * 32 + lane;
                // one partner whose only partner is this site: nobody competes
                const bool live = t < t1, none = live && xo1[q] - xo[q] == 1u && po1[q] - po0[q] == 1u, gen = live && !none;
                if (none) a.ncp[t] = 0u;
                uint32_t wt2;
                const uint32_t ex2 = co_warp_excl(rc[q], wt2);
                if (live) a.loc_rp[t] = run2 + ex2;                                 // inside the warp for now
                run2 += wt2;
                const uint32_t gm = __ballot_sync(full, gen);
                if (gm) {
                    if (ln + 32u > (uint32_t)CO_WL) drain();
                    if (gen) wl[2u * (ln + __popc(gm & lt_mask))] = t;
                    ln += __popc(gm);
                }
            }
        }
        drain();
        uint32_t tot, tot2;
        cp_front = co_warps_excl(run, s_w, tot);
        const uint32_t rp_front = co_warps_excl(run2, s_w, tot2);
        for (uint32_t t = t0 + lane; t < t1; t += 32) a.loc_rp[t] += rp_front;      // read by other CTAs after the barrier
        if (tid == 0) { a.parts[2 * CO_MAX_G + c] = tot; a.parts[3 * CO_MAX_G + c] = tot2; }
    }
    co_grid_sync(a.bar, target);
    co_stamp(a.stamps, stamp++);
    {
        uint32_t C, RP;
        uint32_t xrun = co_parts_prefix(a.parts + 2 * CO_MAX_G, s_pre, s_w, C) + cp_front;
        const uint32_t rpb = co_parts_prefix(a.parts + 3 * CO_MAX_G, s_pre2, s_w, RP);
        auto drain = [&]() {
            __syncwarp();
            for (uint32_t i = lane; i < ln; i += 32) {
                const uint32_t t = wl[2u * i];
                uint32_t x = wl[2u * i + 1u];
                const int32_t tp = g.site_pos[t];
                for (int32_t last = INT_MIN;;) {
                    last = next_competitor(g, g.pt_off, t, tp, last);
                    if (last == INT_MAX) break;
                    if (x < a.cap) g.cp_pos[x] = last;
                    ++x;
                }
            }
            __syncwarp();
            ln = 0;
        };
        for (uint32_t tb = t0; tb < t1; tb += 32 * CO_KB) {
            uint32_t nc[CO_KB], lr[CO_KB];
#pragma unroll
            for (int q = 0; q < CO_KB; ++q) {
                const uint32_t t = tb + q * 32 + lane;
                nc[q] = t < t1 ? a.ncp[t] : 0u; lr[q] = t < t1 ? a.loc_rp[t] : 0u;
            }
#pragma unroll
            for (int q = 0; q < CO_KB; ++q) {
                if (tb + q * 32 >= t1) break;                                       // warp-uniform
                const uint32_t t = tb + q * 32 + lane;
                uint32_t wt;
                const uint32_t x = xrun + co_warp_excl(nc[q], wt);
                xrun += wt;
                const bool live = t < t1, gen = live && nc[q] != 0u;
                if (live) {
                    g.cp_off[t] = (int32_t)x;
                    g.cp_off64[t] = (int64_t)x;
                    g.rp_off[t] = (int32_t)(rpb + lr[q]);
                }
                const uint32_t gm = __ballot_sync(full, gen);
                if (gm) {
                    if (ln + 32u > (uint32_t)CO_WL) drain();
                    if (gen) { const uint32_t i = ln + __popc(gm & lt_mask); wl[2u * i] = t; wl[2u * i + 1u] = x; }
                    ln += __popc(gm);
                }
            }
        }
        drain();
        if (c == 0 && tid == 0) {
            g.cp_off[S] = (int32_t)C; g.cp_off64[S] = (int64_t)C; g.rp_off[S] = (int32_t)RP;
            a.cnt[4] = C; a.cnt[5] = RP;
            if (C > a.cap) a.cnt[6] = 1u;                                          // the host re-runs with room
        }
        // reverse-partner lists + hot flags, one thread per Partners entry; the offset of a site owned by another CTA is its
        // prefix inside that CTA (written before the barrier) + that CTA's base
        const uint32_t stride = G * CO_THREADS;
        for (uint32_t eb = c * CO_THREADS + tid; eb < E; eb += CO_KB * stride) {
            uint32_t pp[CO_KB], ts[CO_KB], an[CO_KB], nc[CO_KB], lr[CO_KB], at[CO_KB];
            int32_t pos[CO_KB], posm[CO_KB], chr[CO_KB], chrm[CO_KB];
#pragma unroll
            for (int q = 0; q < CO_KB; ++q) {
                const uint32_t e = eb + q * stride;
                pp[q] = e < E ? (uint32_t)g.pt_site[e] : 0u; ts[q] = e < E ? a.e_src[e] : 0u;
            }
#pragma unroll
            for (int q = 0; q < CO_KB; ++q) {
                const bool lv = eb + q * stride < E;
                pos[q] = lv ? g.site_pos[pp[q]] : 0; chr[q] = lv ? g.site_chrom[pp[q]] : 0;
                posm[q] = lv && pp[q] > 0 ? g.site_pos[pp[q] - 1] : -1; chrm[q] = lv && pp[q] > 0 ? g.site_chrom[pp[q] - 1] : -1;
                nc[q] = lv ? a.ncp[ts[q]] : 0u;
            }
#pragma unroll
            for (int q = 0; q < CO_KB; ++q) {
                const bool lv = eb + q * stride < E;
                an[q] = (pp[q] > 0 && posm[q] == pos[q] && chrm[q] == chr[q]) ? pp[q] - 1u : pp[q];
                lr[q] = lv ? a.loc_rp[an[q]] : 0u;
                at[q] = lv ? atomicAdd(a.rp_cur + an[q], 1u) : 0u;
            }
#pragma unroll
            for (int q = 0; q < CO_KB; ++q) {
                if (eb + q * stride >= E) break;
                g.rp_site[s_pre2[an[q] / Ks] + lr[q] + at[q]] = (int32_t)ts[q];     // order inside a list does not matter: only counted
                if (nc[q] > 0u) g.site_hot[an[q]] = 1;
            }
        }
    }
    co_stamp(a.stamps, stamp++);
    __syncthreads();
    if (tid == 0) {
        __threadfence();
        if (atomicAdd(a.bar + 1, 1u) == G - 1) { a.bar[0] = 0u; a.bar[1] = 0u; }  // the last CTA out: nobody waits on the words any more
    }
}

// CTAs of k_gb_coop on the current device (one per SM), 0 when the device cannot run it
static std::atomic<int> grid_of[64];
void coop_disable() {
    int dev = 0;
    cudaGetDevice(&dev);
    if (dev >= 0 && dev < 64) grid_of[dev].store(-1);
}
int coop_grid() {
    int dev = 0;
    cudaGetDevice(&dev);
    if (dev < 0 || dev >= 64) return 0;
    int gsz = grid_of[dev].load();
    if (gsz) return gsz > 0 ? gsz : 0;
    int coop = 0, sms = 0, per_sm = 0;
    cudaDeviceGetAttribute(&coop, cudaDevAttrCooperativeLaunch, dev);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    if (coop && cudaFuncSetAttribute((const void*)k_gb_coop, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)CO_SMEM) == cudaSuccess)
        cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, (const void*)k_gb_coop, CO_THREADS, CO_SMEM);
    cudaGetLastError();
    // one CTA per SM: measured against two on configs[1] (474k keys): 91 vs 96 us -- the barriers (3 - 4 us each with 148 arrivals,
    // more with 296) weigh more than the extra warps bring; SPLISER_K1_CTAS_PER_SM=2 for experiments
    int want = 1;
    if (const char* f = std::getenv("SPLISER_K1_CTAS_PER_SM")) want = std::max(1, atoi(f));
    gsz = (coop && per_sm >= 1 && sms >= 1) ? std::min(sms * std::min(per_sm, want), CO_MAX_G) : -1;
    if (const char* f = std::getenv("SPLISER_K1_LAUNCHES")) if (f[0] == '1') gsz = -1;
    grid_of[dev].store(gsz);
    return gsz > 0 ? gsz : 0;
}


// ---- junction extraction from the alignments (SURVEY 8(f) row 3; replaces the `regtools junctions extract` pre-step,
// README.md:41): every N operator with min_intron <= length <= max_intron whose two flanking aligned stretches (M/=/X/D up to
// the neighbouring N or the end of the read) are >= min_anchor long supports the junction (chromosome, l, r, strand); the
// score of a junction is the number of supporting records (what findAlphaCounts reads as alpha, S:274-277).  regtools is
// neither in the reference tree nor in this image: its defaults (-a 8 -m 70 -M 500000) are restated from its documentation.
struct JeSeg { const int64_t* seg_off; const int32_t* seg_chrom; int32_t n_seg; };

__device__ __forceinline__ int je_chrom_of(const JeSeg& sg, uint32_t r) {
    int lo = 0, hi = sg.n_seg;                                          // last segment with seg_off <= r
    while (hi - lo > 1) { const int mid = (lo + hi) >> 1; if (sg.seg_off[mid] <= (int64_t)r) lo = mid; else hi = mid; }
    return sg.seg_chrom[lo];
}

// Pass JE_COUNT: count the supporting N operators of every record and the largest l among them (sizes the position field of
// the key); JE_EMIT: write their keys at the scanned offsets; JE_EXTENT: find each one's row in the sorted unique keys
// (lower_bound; the table is small and stays in L2) and raise the row's longest left / right flanking stretch -- the anchor
// extents a BED12 writes as chromStart = l - max_left, chromEnd = r + max_right.
enum : int { JE_COUNT = 0, JE_EMIT = 1, JE_EXTENT = 2 };
struct JeOut {
    uint32_t* cnt;                  // [R] supporting N operators per record (JE_COUNT writes, JE_EMIT reads its scan)
    uint32_t* max_l;                // JE_COUNT: atomicMax of l over the supporting N operators
    uint64_t* keys;                 // JE_EMIT
    const uint64_t* ukeys;          // JE_EXTENT: unique keys, ascending
    uint32_t n_u;
    uint32_t* ext_l;                // JE_EXTENT: [n_u] atomicMax of the left / right stretch
    uint32_t* ext_r;
};
// XS: every junction of record r takes the strand xs[r] ('+', '-', else '?') instead of the one `mode` derives from the FLAG
template <int PASS, bool XS>
__global__ void __launch_bounds__(256) k_je_walk(DevRecords rec, JeSeg sg, uint32_t mode, int32_t min_anchor, int32_t min_intron, int32_t max_intron,
                                                 int pb, JeOut o, const uint8_t* __restrict__ xs) {
    const uint32_t r = blockIdx.x * blockDim.x + threadIdx.x;
    const bool live = r < rec.n_rec;                                    // every lane reaches the warp reduction of JE_COUNT
    const int chrom = live ? je_chrom_of(sg, r) : -1;
    uint32_t n = 0, w = (PASS == JE_EMIT && live) ? o.cnt[r] : 0u, top = 0;
    if (chrom >= 0) {
        const uint32_t c0 = rec.cig_off[r], c1 = rec.cig_off[r + 1];
        const uint32_t flag = rec.flag[r];
        uint32_t strand = 0;                                            // 0 '?', 1 '+', 2 '-'
        if (XS) {
            const uint8_t x = xs[r];
            strand = x == '+' ? 1u : x == '-' ? 2u : 0u;
        } else if (mode & FLAG_STRANDED) {
            const bool first = (flag & 64u) || !(flag & 1u), rev = (flag & 16u) != 0;
            bool plus = first != rev;
            if (mode & FLAG_RF) plus = !plus;
            strand = plus ? 1u : 2u;
        }
        int32_t cur = rec.pos[r];
        int32_t left = 0;                                               // aligned stretch in front of the pending N
        int32_t pl = 0, plen = -1;                                      // pending junction: l, length (-1: none)
        int32_t pleft = 0;
        for (uint32_t k = c0; k <= c1; ++k) {
            const uint32_t v = k < c1 ? rec.cigar[k] : 3u;              // a virtual N closes the last stretch
            const uint32_t op = v & 15u;
            const int32_t len = (int32_t)(v >> 4);
            if (op == 3u) {
                if (plen >= 0 && plen >= min_intron && plen <= max_intron && pleft >= min_anchor && left >= min_anchor) {
                    if (PASS == JE_COUNT) top = max(top, (uint32_t)pl);
                    if (PASS != JE_COUNT) {
                        const uint64_t key = ((((uint64_t)(uint32_t)chrom << pb | (uint64_t)(uint32_t)pl) << 20 | (uint64_t)(uint32_t)plen) << 2) | strand;
                        if (PASS == JE_EMIT) o.keys[w] = key;
                        if (PASS == JE_EXTENT) {
                            uint32_t lo = 0, hi = o.n_u;                // first unique key >= key: the key is there
                            while (lo < hi) { const uint32_t mid = (lo + hi) >> 1; if (o.ukeys[mid] < key) lo = mid + 1; else hi = mid; }
                            atomicMax(o.ext_l + lo, (uint32_t)pleft);
                            atomicMax(o.ext_r + lo, (uint32_t)left);
                        }
                    }
                    ++w; ++n;
                }
                pl = cur - 1; plen = k < c1 ? len : -1; pleft = left; left = 0;
                cur += len;
            } else if (op == 0u || op == 7u || op == 8u || op == 2u) {
                left += len; cur += len;
            }
        }
    }
    if (PASS == JE_COUNT) {
        if (live) o.cnt[r] = n;
        top = __reduce_max_sync(0xffffffffu, top);                      // one atomic per warp
        if ((threadIdx.x & 31u) == 0 && top) atomicMax(o.max_l, top);
    }
}

__global__ void k_je_heads(const uint64_t* __restrict__ k, uint32_t n, uint32_t* __restrict__ flag) {
    const uint32_t e = blockIdx.x * blockDim.x + threadIdx.x;
    if (e < n) flag[e] = (e == 0 || k[e] != k[e - 1]) ? 1u : 0u;
}
__global__ void k_je_out(const uint64_t* __restrict__ k, const uint32_t* __restrict__ ex, uint32_t n, int pb, int32_t* __restrict__ o_chrom,
                         int32_t* __restrict__ o_left, int32_t* __restrict__ o_right, uint8_t* __restrict__ o_strand, unsigned long long* __restrict__ o_score,
                         uint64_t* __restrict__ o_key) {
    const uint32_t e = blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= n) return;
    const bool head = e == 0 || k[e] != k[e - 1];
    const uint32_t idx = ex[e] - (head ? 0u : 1u);
    atomicAdd(o_score + idx, 1ull);
    if (head) {
        const uint64_t key = k[e];
        o_key[idx] = key;
        const uint32_t st = (uint32_t)(key & 3u);
        const int32_t plen = (int32_t)((key >> 2) & 0xfffffu);
        const int32_t l = (int32_t)((key >> 22) & ((1ull << pb) - 1ull));
        o_chrom[idx] = (int32_t)(key >> (22 + pb));
        o_left[idx] = l; o_right[idx] = l + plen;
        o_strand[idx] = st == 1u ? (uint8_t)'+' : st == 2u ? (uint8_t)'-' : (uint8_t)'?';
    }
}

}  // namespace

bool graph_build_fits(int64_t J, int32_t n_chrom, int32_t max_pos) {
    if (J <= 0 || J >= ((int64_t)1 << 27)) return false;
    const int pb = bits_for_u64((uint64_t)(max_pos > 0 ? max_pos : 1)), cb = bits_for_u64((uint64_t)(n_chrom > 1 ? n_chrom - 1 : 1));
    const int vb = bits_for_u64((uint64_t)(2 * J - 1)), lb = bits_for_u64((uint64_t)(J - 1));
    const int sb = bits_for_u64((uint64_t)(2 * J));                     // S <= 2J (S itself is a sentinel value), E <= 2J
    return cb + pb + 1 + vb <= 64 && 2 * sb + lb <= 64 && sb + lb + vb <= 64 && pb + sb + 1 <= 64;
}

#define GB_CU(call)                                                                     \
    do {                                                                                \
        cudaError_t _e = (call);                                                        \
        if (_e != cudaSuccess) { err = std::string(#call) + ": " + cudaGetErrorString(_e); return false; } \
    } while (0)

bool graph_build_device(GraphBuildMem& m, const int32_t* j_chrom, const int32_t* j_left, const int32_t* j_right, const uint8_t* j_strand,
                        const int64_t* j_score, int64_t n_junc, int32_t n_chrom, int32_t max_pos, bool stranded, void* stream,
                        int phase, GraphDev& g, GraphCounts& counts, std::string& err) {
    cudaStream_t st = (cudaStream_t)stream;
    const uint32_t J = (uint32_t)n_junc, n2 = 2 * J;
    const int pb = bits_for_u64((uint64_t)(max_pos > 0 ? max_pos : 1)), cb = bits_for_u64((uint64_t)(n_chrom > 1 ? n_chrom - 1 : 1));
    const int vb = bits_for_u64((uint64_t)(n2 - 1));

    if (phase == 0) {
        // exact size of the direct-address bin index: per chromosome, bins up to its highest site position + a sentinel
        std::vector<int32_t> cmax((size_t)n_chrom, -1);
        for (int64_t i = 0; i < n_junc; ++i) {
            int32_t& v = cmax[(size_t)j_chrom[i]];
            v = std::max(v, std::max(j_left[i], j_right[i]));
        }
        uint64_t nb = 0;
        for (int32_t c = 0; c < n_chrom; ++c) nb += (cmax[(size_t)c] >= 0 ? (uint64_t)(cmax[(size_t)c] >> SB_SHIFT) + 1u : 0u) + 1u;
        if (nb >= ((uint64_t)1 << 31)) { err = "graph build: bin index exceeds 2^31 entries"; return false; }
        m.nb_host = (uint32_t)nb;
        if (m.cap_c < 8u * (size_t)n2 + 1024u) m.cap_c = 8u * (size_t)n2 + 1024u;
    }

    // ---- final arrays (bounded by J), competitor array (capacity, checked on the device) and bin index
    Carve f;
    const size_t o_cs = f.take<int32_t>((size_t)n_chrom + 1), o_sbb = f.take<int32_t>((size_t)n_chrom + 1);
    const size_t o_chrom = f.take<int32_t>(n2 + 1), o_pos = f.take<int32_t>(n2 + 72), o_strand = f.take<uint8_t>(n2 + 8), o_cls = f.take<uint8_t>(n2 + 8);
    const size_t o_hot = f.take<uint8_t>(n2 + 72), o_fl = f.take<int64_t>(n2 + 1);
    const size_t o_pto = f.take<int32_t>(n2 + 2), o_pts = f.take<int32_t>(n2 + 1), o_pcp = f.take<int32_t>(n2 + 1);
    const size_t o_cpo = f.take<int32_t>(n2 + 2), o_rpo = f.take<int32_t>(n2 + 2), o_rps = f.take<int32_t>(n2 + 1);
    const size_t o_ino = f.take<int32_t>(n2 + 2), o_inl = f.take<int32_t>(n2 + 1);
    const size_t o_eib = f.take<int32_t>(n2 + 1), o_eie = f.take<int32_t>(n2 + 1), o_eil = f.take<int32_t>(n2 + 1);
    const size_t o_js = f.take<int64_t>((size_t)J + 1);
    const size_t o_pto64 = f.take<int64_t>(n2 + 2), o_cpo64 = f.take<int64_t>(n2 + 2);
    const size_t o_jc = f.take<int32_t>(J), o_jl = f.take<int32_t>(J), o_jr = f.take<int32_t>(J), o_jst = f.take<uint8_t>((size_t)J + 8);
    GB_CU(m.fin.reserve(f.off + 256));
    Carve x;
    const size_t x_cp = x.take<int32_t>(m.cap_c + 1), x_sb = x.take<int32_t>((size_t)m.nb_host + 64 + 16);
    GB_CU(m.fin2.reserve(x.off + 256));
    char* fb = (char*)m.fin.p;
    g = GraphDev{};
    g.cs_off = (int32_t*)(fb + o_cs); g.sb_base = (int32_t*)(fb + o_sbb);
    g.site_chrom = (int32_t*)(fb + o_chrom); g.site_pos = (int32_t*)(fb + o_pos); g.site_strand = (uint8_t*)(fb + o_strand);
    g.site_cls = (uint8_t*)(fb + o_cls); g.site_hot = (uint8_t*)(fb + o_hot); g.first_line = (int64_t*)(fb + o_fl);
    g.pt_off = (int32_t*)(fb + o_pto); g.pt_site = (int32_t*)(fb + o_pts); g.pc_pos = (int32_t*)(fb + o_pcp);
    g.cp_off = (int32_t*)(fb + o_cpo); g.rp_off = (int32_t*)(fb + o_rpo); g.rp_site = (int32_t*)(fb + o_rps);
    g.inc_off = (int32_t*)(fb + o_ino); g.inc_line = (int32_t*)(fb + o_inl);
    g.einc_beg = (int32_t*)(fb + o_eib); g.einc_end = (int32_t*)(fb + o_eie); g.einc_line = (int32_t*)(fb + o_eil);
    g.j_score = (int64_t*)(fb + o_js); g.pt_off64 = (int64_t*)(fb + o_pto64); g.cp_off64 = (int64_t*)(fb + o_cpo64);
    g.cp_pos = (int32_t*)((char*)m.fin2.p + x_cp); g.sb_off = (int32_t*)((char*)m.fin2.p + x_sb);
    int32_t* d_jc = (int32_t*)(fb + o_jc); int32_t* d_jl = (int32_t*)(fb + o_jl); int32_t* d_jr = (int32_t*)(fb + o_jr);
    uint8_t* d_js = (uint8_t*)(fb + o_jst);

    const uint32_t max_tiles = cdiv(n2, RS_TILE) + 1;
    const uint32_t lb_tiles = cdiv(std::max((uint32_t)RS_BINS * max_tiles, n2 + 2u), LB_TILE) + 2;
    Carve w;
    const size_t w_ka = w.take<uint64_t>(n2 + 2), w_kb = w.take<uint64_t>(n2 + 2), w_flag = w.take<uint32_t>(n2 + 2);
    const size_t w_hist = w.take<uint32_t>((size_t)RS_BINS * (size_t)max_tiles + 2);
    const size_t w_cnt = w.take<uint32_t>(16), w_site_of = w.take<uint32_t>(n2 + 2), w_eid = w.take<uint32_t>(n2 + 2);
    const size_t w_esrc = w.take<uint32_t>(n2 + 2), w_npt = w.take<uint32_t>(n2 + 4), w_ncp = w.take<uint32_t>(n2 + 4);
    const size_t w_c1 = w.take<uint32_t>(n2 + 4), w_c2 = w.take<uint32_t>(n2 + 4);
    const size_t w_desc = w.take<unsigned long long>(lb_tiles + SC_EXTRA);  // descriptors, then the ticket word and the rendezvous words
    const int coop_g = coop_grid();                                         // scratch of the one-kernel build (k_gb_coop)
    const size_t w_chist = w.take<uint32_t>((size_t)RS_BINS * (size_t)std::max(coop_g, 1)), w_dtot = w.take<uint32_t>(RS_BINS);
    const size_t w_parts = w.take<uint32_t>(4 * CO_MAX_G), w_bar = w.take<uint32_t>(16);
    const size_t w_l3 = w.take<uint32_t>(n2 + 4), w_stamps = w.take<uint32_t>(CO_STAMPS);
    const bool fresh = m.work.cap < w.off + 256;
    GB_CU(m.work.reserve(w.off + 256));
    char* wb = (char*)m.work.p;
    uint64_t* ka = (uint64_t*)(wb + w_ka); uint64_t* kb = (uint64_t*)(wb + w_kb);
    uint32_t* flag = (uint32_t*)(wb + w_flag);
    uint32_t* d_cnt = (uint32_t*)(wb + w_cnt);     // [0] S, [1] bin entries, [2] E, [4] C, [5] scratch, [6] competitor overflow, [7] S + 1
    uint32_t* site_of = (uint32_t*)(wb + w_site_of); uint32_t* inc_eid = (uint32_t*)(wb + w_eid);
    uint32_t* e_src = (uint32_t*)(wb + w_esrc);
    uint32_t* npt = (uint32_t*)(wb + w_npt); uint32_t* ncp = (uint32_t*)(wb + w_ncp);
    uint32_t* c1 = (uint32_t*)(wb + w_c1); uint32_t* c2 = (uint32_t*)(wb + w_c2);
    unsigned long long* desc = (unsigned long long*)(wb + w_desc);
    const Scanner sc{desc, (uint32_t*)(desc + lb_tiles + 8), &m.scan_epoch, st, (uint32_t*)(desc + lb_tiles + 16)};
    const Sorter sorter{(uint32_t*)(wb + w_hist), sc, d_cnt + 5, st};

    // ---- junction table to the device (phase 0: queued before the caller starts the big record upload, which
    // would otherwise sit in front of it on the host->device copy engine)
    if (phase == 0) {
        GB_CU(cudaMemcpyAsync(d_jc, j_chrom, (size_t)J * 4, cudaMemcpyHostToDevice, st));
        GB_CU(cudaMemcpyAsync(d_jl, j_left, (size_t)J * 4, cudaMemcpyHostToDevice, st));
        GB_CU(cudaMemcpyAsync(d_jr, j_right, (size_t)J * 4, cudaMemcpyHostToDevice, st));
        GB_CU(cudaMemcpyAsync(d_js, j_strand, (size_t)J, cudaMemcpyHostToDevice, st));
        GB_CU(cudaMemcpyAsync((void*)g.j_score, j_score, (size_t)J * 8, cudaMemcpyHostToDevice, st));
        counts.h2d_bytes = (double)J * 21.0;
        GB_CU(cudaMemsetAsync(d_cnt, 0, 64, st));
        m.scan_epoch = 0;
        GB_CU(cudaMemsetAsync(desc, 0, ((size_t)lb_tiles + SC_EXTRA) * sizeof(unsigned long long), st));     // descriptors + ticket + rendezvous words
        GB_CU(cudaMemsetAsync(wb + w_bar, 0, 64, st));                     // barrier words of k_gb_coop (it leaves them zero)
        m.ready = true;
        return true;
    }
    if (fresh || !m.ready) { err = "graph build: phase 1 without phase 0"; return false; }

    bool coop_done = false;
    if (coop_g > 0) {
        CoopArgs ca{};
        ca.jc = d_jc; ca.jl = d_jl; ca.jr = d_jr; ca.js = d_js;
        ca.J = J; ca.stranded = stranded ? 1 : 0; ca.pb = pb; ca.vb = vb; ca.lo = vb; ca.hi = vb + 1 + pb + cb; ca.n_chrom = n_chrom;
        ca.ka = ka; ca.kb = kb;
        ca.hist = (uint32_t*)(wb + w_chist); ca.dtot = (uint32_t*)(wb + w_dtot); ca.parts = (uint32_t*)(wb + w_parts);
        ca.bar = (uint32_t*)(wb + w_bar); ca.cnt = d_cnt;
        ca.site_of = site_of; ca.inc_eid = inc_eid; ca.e_src = e_src; ca.ncp = ncp; ca.rp_cnt = c1; ca.rp_cur = c2;
        ca.loc_rp = (uint32_t*)(wb + w_l3);
        static const bool want_stamps = std::getenv("SPLISER_K1_STAMPS") != nullptr;      // phase timeline of CTA 0 (diagnostics)
        ca.stamps = want_stamps ? (uint32_t*)(wb + w_stamps) : nullptr;
        ca.cap = (uint32_t)std::min<size_t>(m.cap_c, 0xffffffffu);
        ca.g = g;
        void* params[] = {(void*)&ca};
        // a launch the device refuses (the grid does not fit at once: instrumented builds, a partitioned device) is not an error of
        // the build: this device takes the launch-per-phase kernels from now on
        const cudaError_t le = cudaLaunchCooperativeKernel((const void*)k_gb_coop, dim3((unsigned)coop_g), dim3(CO_THREADS), params, CO_SMEM, st);
        if (le == cudaSuccess) { SPL_LAUNCH; coop_done = true; }
        else { cudaGetLastError(); coop_disable(); }
        if (coop_done) {
            { SPL_LAUNCH; k_gb_sb_fill<<<148 * 8, 256, 0, st>>>(g, n_chrom, d_cnt); }
            GB_CU(cudaGetLastError());
            if (want_stamps && phase == 1) {
                uint32_t h[CO_STAMPS] = {0};
                GB_CU(cudaMemsetAsync(wb + w_stamps, 0, sizeof(h), st));
                SPL_LAUNCH;
                GB_CU(cudaLaunchCooperativeKernel((const void*)k_gb_coop, dim3((unsigned)coop_g), dim3(CO_THREADS), params, CO_SMEM, st));
                GB_CU(cudaMemcpyAsync(h, wb + w_stamps, sizeof(h), cudaMemcpyDeviceToHost, st));
                GB_CU(cudaStreamSynchronize(st));
                fprintf(stderr, "[k1 stamps, us since kernel start, grid %d]", coop_g);
                for (int q = 1; q < CO_STAMPS && h[q]; ++q) fprintf(stderr, " %.1f", (double)(uint32_t)(h[q] - h[0]) * 1e-3);
                fprintf(stderr, "\n");
            }
        }
    }
    if (!coop_done) {
    // ---- A: sites
    GB_CU(cudaMemsetAsync(d_cnt + 6, 0, 4, st));
    { SPL_LAUNCH; k_gb_keys_a<<<cdiv(J, 256), 256, 0, st>>>(d_jc, d_jl, d_jr, d_js, J, stranded ? 1 : 0, pb, vb, ka); }
    uint64_t* sa = sorter.sort(ka, kb, n2, vb, vb + 1 + pb + cb);
    { SPL_LAUNCH; k_gb_heads<<<cdiv(n2, 256), 256, 0, st>>>(sa, n2, vb, flag); }
    sc.scan(flag, n2, nullptr, d_cnt + 0);
    GB_CU(cudaMemsetAsync(g.site_hot, 0, (size_t)n2 + 64, st));
    { SPL_LAUNCH; k_gb_sites<<<cdiv(n2, 256), 256, 0, st>>>(sa, flag, n2, vb, pb, stranded ? 1 : 0, d_js, g, site_of, inc_eid, d_cnt); }
    { SPL_LAUNCH; k_gb_chroms<<<1, 256, 0, st>>>(g, n_chrom, d_cnt); }

    // ---- B: Partners / PartnerCounts entries per site
    GB_CU(cudaMemsetAsync(npt, 0, (size_t)((char*)(c2 + n2 + 4) - (char*)npt), st));   // npt, ncp, rp_cnt, rp_cur: adjacent in the carve
    { SPL_LAUNCH; k_gb_pt_count<<<cdiv(n2, 128), 128, 0, st>>>(g, d_cnt, site_of, inc_eid, npt); }
    sc.scan(npt, n2 + 2, d_cnt + 7, d_cnt + 2);
    { SPL_LAUNCH; k_gb_pt_fill<<<cdiv(n2 + 1, 128), 128, 0, st>>>(g, d_cnt, site_of, inc_eid, npt, e_src); }

    // ---- D: competitors
    { SPL_LAUNCH; k_gb_cp_count<<<cdiv(n2, 128), 128, 0, st>>>(g, d_cnt, ncp); }
    sc.scan(ncp, n2 + 2, d_cnt + 7, d_cnt + 4);
    { SPL_LAUNCH; k_gb_cp_fill<<<cdiv(n2 + 1, 128), 128, 0, st>>>(g, d_cnt, ncp, (uint32_t)std::min<size_t>(m.cap_c, 0xffffffffu)); }

    // ---- E: reverse partners, hot flags, bin index
    { SPL_LAUNCH; k_gb_rp_count<<<cdiv(n2, 256), 256, 0, st>>>(g, d_cnt, c1); }
    sc.scan(c1, n2 + 2, d_cnt + 7, d_cnt + 5);
    { SPL_LAUNCH; k_gb_rp_fill<<<cdiv(n2 + 2, 256), 256, 0, st>>>(g, d_cnt, e_src, c1, c2); }
    { SPL_LAUNCH; k_gb_sb_fill<<<148 * 8, 256, 0, st>>>(g, n_chrom, d_cnt); }
    GB_CU(cudaGetLastError());
    }
    if (phase == 2) return true;                                           // timed rebuild of a table whose sizes are known

    GB_CU(cudaMemcpyAsync(m.h_cnt, d_cnt, 64, cudaMemcpyDeviceToHost, st));
    GB_CU(cudaStreamSynchronize(st));
    const uint32_t S = m.h_cnt[0], NB = m.h_cnt[1], E = m.h_cnt[2], C = m.h_cnt[4];
    if (S == 0 || S > n2) { err = "graph build: bad site count"; return false; }
    if (E == 0 || E > n2) { err = "graph build: bad edge count"; return false; }
    if (NB != m.nb_host) { err = "graph build: bin index size mismatch"; return false; }
    if (m.h_cnt[6]) {                                                      // more competitors than the array holds: once more with room
        if ((size_t)C <= m.cap_c) { err = "graph build: inconsistent competitor overflow"; return false; }
        m.cap_c = (size_t)C + 1024;
        return graph_build_device(m, j_chrom, j_left, j_right, j_strand, j_score, n_junc, n_chrom, max_pos, stranded, stream, phase, g, counts, err);
    }
    counts.S = S; counts.E = E; counts.NB = NB; counts.C = C;
    return true;
}

// Junction table of the device-resident records, sorted by (chromosome, l, r, strand), with each row's anchor extents.
// Synchronises the stream (sizes).
bool junction_extract_device(JuncExtractMem& m, const DevRecords& rec, const int64_t* h_seg_off, const int32_t* h_seg_chrom, int32_t n_seg,
                             int32_t n_chrom, uint32_t mode, const uint8_t* xs, int32_t min_anchor, int32_t min_intron, int32_t max_intron,
                             void* stream, std::vector<int32_t>& chrom, std::vector<int32_t>& left, std::vector<int32_t>& right,
                             std::vector<int64_t>& score, std::vector<uint8_t>& strand, std::vector<int32_t>& start, std::vector<int32_t>& end,
                             std::string& err) {
    cudaStream_t st = (cudaStream_t)stream;
    chrom.clear(); left.clear(); right.clear(); score.clear(); strand.clear(); start.clear(); end.clear();
    const uint32_t R = rec.n_rec;
    if (R == 0 || n_seg == 0) return true;
    if (max_intron >= (1 << 20)) { err = "junction extraction: max_intron must be below 2^20"; return false; }
    const int cb = bits_for_u64((uint64_t)(n_chrom > 1 ? n_chrom - 1 : 1));
    Carve a;
    const size_t a_so = a.take<int64_t>((size_t)n_seg + 1), a_sc = a.take<int32_t>((size_t)n_seg + 1), a_cnt = a.take<uint32_t>((size_t)R + 4);
    const uint32_t lb_tiles0 = cdiv(R + 2u, LB_TILE) + 2;
    const size_t a_desc = a.take<unsigned long long>(lb_tiles0 + SC_EXTRA), a_tot = a.take<uint32_t>(16);
    GB_CU(m.a.reserve(a.off + 256));
    char* ab = (char*)m.a.p;
    GB_CU(cudaMemcpyAsync(ab + a_so, h_seg_off, ((size_t)n_seg + 1) * 8, cudaMemcpyHostToDevice, st));
    GB_CU(cudaMemcpyAsync(ab + a_sc, h_seg_chrom, (size_t)n_seg * 4, cudaMemcpyHostToDevice, st));
    GB_CU(cudaMemsetAsync(ab + a_desc, 0, ((size_t)lb_tiles0 + SC_EXTRA) * 8, st));
    GB_CU(cudaMemsetAsync(ab + a_tot, 0, 64, st));
    const JeSeg sg{(const int64_t*)(ab + a_so), (const int32_t*)(ab + a_sc), n_seg};
    uint32_t* cnt = (uint32_t*)(ab + a_cnt);
    uint32_t* d_tot = (uint32_t*)(ab + a_tot);                          // [0] keys, [1] unique keys, [3] largest l, [5] sorter scratch
    uint32_t epoch = 0;
    unsigned long long* desc0 = (unsigned long long*)(ab + a_desc);
    const Scanner sc0{desc0, (uint32_t*)(desc0 + lb_tiles0 + 8), &epoch, st, (uint32_t*)(desc0 + lb_tiles0 + 16)};
    JeOut jo{};
    jo.cnt = cnt; jo.max_l = d_tot + 3;
    for (auto& e : m.ev) if (!e) GB_CU(cudaEventCreate(&e));
    m.ms_kernels = m.ms_extent = 0;
    GB_CU(cudaEventRecord(m.ev[0], st));
    if (xs) { SPL_LAUNCH; k_je_walk<JE_COUNT, true><<<cdiv(R, 256), 256, 0, st>>>(rec, sg, mode, min_anchor, min_intron, max_intron, 0, jo, xs); }
    else { SPL_LAUNCH; k_je_walk<JE_COUNT, false><<<cdiv(R, 256), 256, 0, st>>>(rec, sg, mode, min_anchor, min_intron, max_intron, 0, jo, nullptr); }
    sc0.scan(cnt, R, nullptr, d_tot);
    GB_CU(cudaEventRecord(m.ev[1], st));
    uint32_t h_tot[4] = {0, 0, 0, 0};
    GB_CU(cudaMemcpyAsync(h_tot, d_tot, 16, cudaMemcpyDeviceToHost, st));
    GB_CU(cudaStreamSynchronize(st));
    const uint32_t n = h_tot[0];
    GB_CU(cudaEventElapsedTime(&m.ms_kernels, m.ev[0], m.ev[1]));
    if (n == 0) return true;
    // the position field holds the largest l of the data (a real genome needs at most 28 bits), so headers with thousands of
    // references still fit the 64-bit key
    const int pb = bits_for_u64((uint64_t)std::max<uint32_t>(h_tot[3], 1u));
    if (cb + pb + 22 > 64) { err = "junction extraction: too many chromosomes for the packed key"; return false; }
    const uint32_t max_tiles = cdiv(n, RS_TILE) + 1;
    const uint32_t lb_tiles = cdiv(std::max((uint32_t)RS_BINS * max_tiles, n + 2u), LB_TILE) + 2;
    Carve b;
    const size_t b_ka = b.take<uint64_t>((size_t)n + 2), b_kb = b.take<uint64_t>((size_t)n + 2), b_flag = b.take<uint32_t>((size_t)n + 2);
    const size_t b_hist = b.take<uint32_t>((size_t)RS_BINS * (size_t)max_tiles + 2), b_desc = b.take<unsigned long long>(lb_tiles + SC_EXTRA);
    const size_t b_oc = b.take<int32_t>((size_t)n + 1), b_ol = b.take<int32_t>((size_t)n + 1), b_or = b.take<int32_t>((size_t)n + 1),
                 b_os = b.take<uint8_t>((size_t)n + 8), b_sc = b.take<unsigned long long>((size_t)n + 1);
    const size_t b_uk = b.take<uint64_t>((size_t)n + 1), b_xl = b.take<uint32_t>((size_t)n + 1), b_xr = b.take<uint32_t>((size_t)n + 1);
    GB_CU(m.b.reserve(b.off + 256));
    char* bb = (char*)m.b.p;
    uint64_t* ka = (uint64_t*)(bb + b_ka); uint64_t* kb = (uint64_t*)(bb + b_kb);
    uint32_t* flag = (uint32_t*)(bb + b_flag);
    unsigned long long* desc = (unsigned long long*)(bb + b_desc);
    GB_CU(cudaMemsetAsync(desc, 0, ((size_t)lb_tiles + SC_EXTRA) * 8, st));
    GB_CU(cudaMemsetAsync(bb + b_sc, 0, ((size_t)n + 1) * 8, st));
    uint32_t epoch2 = 0;
    const Scanner sc{desc, (uint32_t*)(desc + lb_tiles + 8), &epoch2, st, (uint32_t*)(desc + lb_tiles + 16)};
    const Sorter sorter{(uint32_t*)(bb + b_hist), sc, d_tot + 5, st};
    jo.keys = ka;
    GB_CU(cudaEventRecord(m.ev[2], st));
    if (xs) { SPL_LAUNCH; k_je_walk<JE_EMIT, true><<<cdiv(R, 256), 256, 0, st>>>(rec, sg, mode, min_anchor, min_intron, max_intron, pb, jo, xs); }
    else { SPL_LAUNCH; k_je_walk<JE_EMIT, false><<<cdiv(R, 256), 256, 0, st>>>(rec, sg, mode, min_anchor, min_intron, max_intron, pb, jo, nullptr); }
    uint64_t* sk = sorter.sort(ka, kb, n, 0, 22 + pb + cb);
    { SPL_LAUNCH; k_je_heads<<<cdiv(n, 256), 256, 0, st>>>(sk, n, flag); }
    sc.scan(flag, n, nullptr, d_tot + 1);
    uint64_t* ukey = (uint64_t*)(bb + b_uk);
    { SPL_LAUNCH; k_je_out<<<cdiv(n, 256), 256, 0, st>>>(sk, flag, n, pb, (int32_t*)(bb + b_oc), (int32_t*)(bb + b_ol), (int32_t*)(bb + b_or),
                                                       (uint8_t*)(bb + b_os), (unsigned long long*)(bb + b_sc), ukey); }
    GB_CU(cudaGetLastError());
    GB_CU(cudaEventRecord(m.ev[3], st));
    uint32_t h_u = 0;
    GB_CU(cudaMemcpyAsync(&h_u, d_tot + 1, 4, cudaMemcpyDeviceToHost, st));
    GB_CU(cudaStreamSynchronize(st));
    const size_t U = h_u;
    // anchor extents of the U rows
    GB_CU(cudaMemsetAsync(bb + b_xl, 0, U * 4, st));
    GB_CU(cudaMemsetAsync(bb + b_xr, 0, U * 4, st));
    jo.ukeys = ukey; jo.n_u = (uint32_t)U; jo.ext_l = (uint32_t*)(bb + b_xl); jo.ext_r = (uint32_t*)(bb + b_xr);
    GB_CU(cudaEventRecord(m.ev[4], st));
    if (xs) { SPL_LAUNCH; k_je_walk<JE_EXTENT, true><<<cdiv(R, 256), 256, 0, st>>>(rec, sg, mode, min_anchor, min_intron, max_intron, pb, jo, xs); }
    else { SPL_LAUNCH; k_je_walk<JE_EXTENT, false><<<cdiv(R, 256), 256, 0, st>>>(rec, sg, mode, min_anchor, min_intron, max_intron, pb, jo, nullptr); }
    GB_CU(cudaGetLastError());
    GB_CU(cudaEventRecord(m.ev[5], st));
    chrom.resize(U); left.resize(U); right.resize(U); strand.resize(U); score.resize(U); start.resize(U); end.resize(U);
    std::vector<uint32_t> xl(U), xr(U);
    GB_CU(cudaMemcpyAsync(chrom.data(), bb + b_oc, U * 4, cudaMemcpyDeviceToHost, st));
    GB_CU(cudaMemcpyAsync(left.data(), bb + b_ol, U * 4, cudaMemcpyDeviceToHost, st));
    GB_CU(cudaMemcpyAsync(right.data(), bb + b_or, U * 4, cudaMemcpyDeviceToHost, st));
    GB_CU(cudaMemcpyAsync(strand.data(), bb + b_os, U, cudaMemcpyDeviceToHost, st));
    GB_CU(cudaMemcpyAsync(score.data(), bb + b_sc, U * 8, cudaMemcpyDeviceToHost, st));
    GB_CU(cudaMemcpyAsync(xl.data(), bb + b_xl, U * 4, cudaMemcpyDeviceToHost, st));
    GB_CU(cudaMemcpyAsync(xr.data(), bb + b_xr, U * 4, cudaMemcpyDeviceToHost, st));
    GB_CU(cudaStreamSynchronize(st));
    float ms_b = 0;
    GB_CU(cudaEventElapsedTime(&ms_b, m.ev[2], m.ev[3]));
    GB_CU(cudaEventElapsedTime(&m.ms_extent, m.ev[4], m.ev[5]));
    m.ms_kernels += ms_b + m.ms_extent;
    for (size_t i = 0; i < U; ++i) {
        start[i] = left[i] - (int32_t)xl[i];
        end[i] = right[i] + (int32_t)xr[i];
    }
    return true;
}

}  // namespace spl
