// Hand-written sm_100a kernels for the SpliSER counting path.
//
//   K0  expand_count / chunk_scan / expand_scatter : BAM-style records -> SoA
//   K1  alpha reduce (extra blocks of k_span_blocksum): junction scores -> alpha[site], PartnerCounts[edge]   (SpliSER_v0_1_8.py:341,:353-355)
//   K3  beta1_stab     : M-block vs site stabbing count                        (S:454-477)
//   K4  spliced        : N-span range adds + compSplicing exceptions           (S:480-557)
//   K5  span_blocksum / finalize : prefix scan, beta2 gather (S:581-623), SSE (S:626-639)
//
// Nothing here is a dense contraction, so no tensor-core path: the kernels are HBM streaming
// (K3) or L2/latency bound graph lookups (K4, K5).  Site tiles are staged into shared memory with
// a 1-D TMA bulk copy (cp.async.bulk + mbarrier), blocks are loaded 128 bits at a time, matches
// are aggregated per warp with redux.sync before a single RED per (warp, site).
#include <mutex>
#include <cuda_runtime.h>
#include <climits>
#include <cstdint>

#include "device_types.h"
#include "dev_helpers.cuh"

namespace spl {

std::atomic<unsigned long long> g_kernel_launches{0};

struct Cnt4 { uint32_t a, b, s, j; };

// ------------------------------------------------------------------------------------------------
// K0: record expansion (BAM-style records -> SoA).  One CTA per chunk, one record per thread and
// round; the per-round exclusive scan keeps the output in record order, which is what makes the
// A stream sorted by start and the chunk windows tight.
// ------------------------------------------------------------------------------------------------
struct ReadShape {
    uint32_t nM, nN;        // mapped (M,=,X) ops and N ops
    int32_t  lo, hi;        // min block start, max (block end - 2) over M ops  (lo > hi when none)
    int32_t  qlo, qhi;      // min / max position a site lookup of this read may ask for
    int32_t  smax, lmax;    // largest block start, longest block
};

__device__ __forceinline__ ReadShape read_shape(const DevRecords& rec, uint32_t i) {
    ReadShape s;
    s.nM = s.nN = 0;
    s.lo = INT_MAX; s.hi = INT_MIN; s.qlo = INT_MAX; s.qhi = INT_MIN; s.smax = 0; s.lmax = 0;
    int32_t cur = rec.pos[i];
    const uint32_t c0 = rec.cig_off[i], c1 = rec.cig_off[i + 1];
    for (uint32_t k = c0; k < c1; ++k) {
        const uint32_t v = rec.cigar[k];
        const uint32_t op = v & 15u;
        const int32_t len = (int32_t)(v >> 4);
        if (op == 0u || op == 7u || op == 8u) {           // M = X : mapped + advance (S:457-459)
            s.nM++;
            s.lo = min(s.lo, cur);
            s.hi = max(s.hi, cur + len - 2);
            s.qlo = min(s.qlo, cur);
            s.qhi = max(s.qhi, cur + len);
            s.smax = max(s.smax, cur); s.lmax = max(s.lmax, len);
            cur += len;
        } else if (op == 3u) {                            // N : advance, junction (S:480-483)
            s.nN++;
            s.qlo = min(s.qlo, cur - 1);
            s.qhi = max(s.qhi, cur + len);
            cur += len;
        } else if (op == 2u) {                            // D : advance only (S:460-462)
            cur += len;
        }                                                 // I S H P : no progression (S:463-464)
    }
    return s;
}

// block-wide exclusive scan of four counters; returns the exclusive prefix and the block total
__device__ __forceinline__ Cnt4 block_exscan4(Cnt4 v, Cnt4& total, Cnt4* warp_tot /* [33] shared */) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    Cnt4 inc = v;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        const uint32_t a = __shfl_up_sync(0xffffffffu, inc.a, d), b = __shfl_up_sync(0xffffffffu, inc.b, d);
        const uint32_t s = __shfl_up_sync(0xffffffffu, inc.s, d), j = __shfl_up_sync(0xffffffffu, inc.j, d);
        if (lane >= d) { inc.a += a; inc.b += b; inc.s += s; inc.j += j; }
    }
    __syncthreads();                                      // previous use of warp_tot is over
    if (lane == 31) warp_tot[warp] = inc;
    __syncthreads();
    if (warp == 0) {
        const int nw = blockDim.x >> 5;
        Cnt4 w = lane < nw ? warp_tot[lane] : Cnt4{0, 0, 0, 0};
        Cnt4 wi = w;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            const uint32_t a = __shfl_up_sync(0xffffffffu, wi.a, d), b = __shfl_up_sync(0xffffffffu, wi.b, d);
            const uint32_t s = __shfl_up_sync(0xffffffffu, wi.s, d), j = __shfl_up_sync(0xffffffffu, wi.j, d);
            if (lane >= d) { wi.a += a; wi.b += b; wi.s += s; wi.j += j; }
        }
        if (lane < nw) warp_tot[lane] = Cnt4{wi.a - w.a, wi.b - w.b, wi.s - w.s, wi.j - w.j};   // exclusive
        if (lane == nw - 1) warp_tot[32] = wi;                                                  // total
    }
    __syncthreads();
    const Cnt4 base = warp_tot[warp];
    total = warp_tot[32];
    return Cnt4{base.a + inc.a - v.a, base.b + inc.b - v.b, base.s + inc.s - v.s, base.j + inc.j - v.j};
}

__global__ void __launch_bounds__(EXPAND_THREADS) k_expand_count(DevRecords rec, Chunk* chunks, uint32_t mode, DevBins bins) {
    Chunk& ck = chunks[blockIdx.x];
    Cnt4 c{0, 0, 0, 0};
    int32_t alo = INT_MAX, ahi = INT_MIN, slo = INT_MAX, shi = INT_MIN, smax = 0, lmax = 0;
    for (uint32_t i = ck.rec_lo + threadIdx.x; i < ck.rec_hi; i += EXPAND_THREADS) {
        const ReadShape s = read_shape(rec, i);
        smax = max(smax, s.smax); lmax = max(lmax, s.lmax);
        if (s.nN == 0) {
            c.a += s.nM;
            alo = min(alo, s.lo); ahi = max(ahi, s.hi);
        } else {
            c.b += s.nM; c.s += 1; c.j += s.nN;
            slo = min(slo, s.qlo); shi = max(shi, s.qhi);
        }
    }
    __shared__ Cnt4 wt[33];
    __shared__ int32_t red[6][EXPAND_THREADS / 32];
    Cnt4 total;
    (void)block_exscan4(c, total, wt);
    alo = __reduce_min_sync(0xffffffffu, alo); ahi = __reduce_max_sync(0xffffffffu, ahi);
    slo = __reduce_min_sync(0xffffffffu, slo); shi = __reduce_max_sync(0xffffffffu, shi);
    smax = __reduce_max_sync(0xffffffffu, smax); lmax = __reduce_max_sync(0xffffffffu, lmax);
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    if (lane == 0) { red[0][warp] = alo; red[1][warp] = ahi; red[2][warp] = slo; red[3][warp] = shi; red[4][warp] = smax; red[5][warp] = lmax; }
    __syncthreads();
    if (threadIdx.x == 0) {
        for (int w = 1; w < EXPAND_THREADS / 32; ++w) {
            alo = min(alo, red[0][w]); ahi = max(ahi, red[1][w]);
            slo = min(slo, red[2][w]); shi = max(shi, red[3][w]);
            smax = max(smax, red[4][w]); lmax = max(lmax, red[5][w]);
        }
        ck.a_cnt = total.a; ck.b_cnt = total.b; ck.s_cnt = total.s; ck.j_cnt = total.j;
        ck.a_lo = alo; ck.a_hi = ahi; ck.s_lo = slo; ck.s_hi = shi;
        if (total.a + total.b) {
            atomicMax(bins.chrom_ext + ck.chrom, (uint32_t)smax);
            atomicAdd(bins.chrom_tot + ck.chrom, total.a + total.b);
            atomicMax(bins.max_len, (uint32_t)lmax);
        }
        if (total.j) atomicAdd(bins.chrom_jn + ck.chrom, total.j);
    }
}

// bin / tile layout of stream C from the per-chromosome extents and block totals (tiny: one thread)
__global__ void k_bin_layout(DevBins bins, uint32_t* totals8) {
    if (blockIdx.x || threadIdx.x) return;
    uint32_t nb = 0, nt = 0;
    for (int c = 0; c < bins.n_chrom; ++c) {
        bins.chrom_bin_base[c] = nb; bins.chrom_tile_base[c] = nt;
        if (bins.chrom_tot[c]) {
            nb += (bins.chrom_ext[c] >> BIN_SHIFT) + 1;
            nt += (bins.chrom_tot[c] + K3_TILE - 1) / K3_TILE;
        }
    }
    bins.chrom_bin_base[bins.n_chrom] = nb; bins.chrom_tile_base[bins.n_chrom] = nt;
    totals8[4] = nb; totals8[5] = nt; totals8[6] = nt * K3_TILE; totals8[7] = bins.max_len[0];
}

// junction sub-tables, one power-of-two table per chromosome.  attempt 0 sizes them for the usual case (distinct
// junctions are a tiny fraction of the N operators: instances / 8, at least 1024 slots); if a probe sequence gets long
// the insert kernel raises the overflow flag and the host retries with attempt 1: >= 2 x instances, which cannot fill.
__global__ void k_jtab_layout(DevBins bins, int attempt, uint32_t* totals8) {
    if (blockIdx.x || threadIdx.x) return;
    uint32_t ns = 0;
    for (int c = 0; c < bins.n_chrom; ++c) {
        bins.tab_base[c] = ns;
        if (bins.chrom_jn[c]) {
            const uint32_t jn = bins.chrom_jn[c];
            const uint32_t want = (attempt > 0 || jn <= 4096u) ? 2u * jn : max(8192u, jn >> 3);
            uint32_t t = 64;
            while (t < want) t <<= 1;
            ns += t;
        }
    }
    bins.tab_base[bins.n_chrom] = ns;
    totals8[8] = ns;
}

// exclusive scan of the per-chunk totals; single CTA (n_chunks is R / 4096: at most ~1e5)
__global__ void __launch_bounds__(1024) k_chunk_scan(Chunk* chunks, int n_chunks, uint32_t* totals4) {
    __shared__ Cnt4 wt[33];
    __shared__ Cnt4 carry;
    if (threadIdx.x == 0) carry = Cnt4{0, 0, 0, 0};
    __syncthreads();
    for (int base = 0; base < n_chunks; base += 1024) {
        const int i = base + (int)threadIdx.x;
        Cnt4 v{0, 0, 0, 0};
        if (i < n_chunks) v = Cnt4{chunks[i].a_cnt, chunks[i].b_cnt, chunks[i].s_cnt, chunks[i].j_cnt};
        Cnt4 total;
        const Cnt4 ex = block_exscan4(v, total, wt);
        const Cnt4 c = carry;
        if (i < n_chunks) {
            chunks[i].a_base = c.a + ex.a; chunks[i].b_base = c.b + ex.b;
            chunks[i].s_base = c.s + ex.s; chunks[i].j_base = c.j + ex.j;
        }
        __syncthreads();
        if (threadIdx.x == 0) carry = Cnt4{c.a + total.a, c.b + total.b, c.s + total.s, c.j + total.j};
        __syncthreads();
    }
    if (threadIdx.x == 0) {
        totals4[0] = carry.a; totals4[1] = carry.b; totals4[2] = carry.s; totals4[3] = carry.j;
    }
}

__global__ void __launch_bounds__(EXPAND_THREADS)
k_expand_scatter(DevRecords rec, const Chunk* chunks, DevSoA soa, uint32_t mode) {
    const Chunk ck = chunks[blockIdx.x];
    __shared__ Cnt4 wt[33];
    Cnt4 run{ck.a_base, soa.bB + ck.b_base, ck.s_base, ck.j_base};       // running output cursors of the chunk
    for (uint32_t base = ck.rec_lo; base < ck.rec_hi; base += EXPAND_THREADS) {   // uniform trip count
        const uint32_t i = base + threadIdx.x;
        const bool live = i < ck.rec_hi;
        uint32_t nM = 0, nN = 0, c0 = 0, c1 = 0;
        if (live) {
            c0 = rec.cig_off[i]; c1 = rec.cig_off[i + 1];
            for (uint32_t k = c0; k < c1; ++k) {
                const uint32_t op = rec.cigar[k] & 15u;
                nM += (op == 0u || op == 7u || op == 8u);
                nN += (op == 3u);
            }
        }
        const bool spliced = nN != 0;
        Cnt4 v{spliced ? 0u : nM, spliced ? nM : 0u, spliced ? 1u : 0u, nN};
        Cnt4 total;
        const Cnt4 ex = block_exscan4(v, total, wt);
        if (live) {
            uint32_t im = spliced ? run.b + ex.b : run.a + ex.a;              // block cursor (A or B stream)
            uint32_t ij = run.j + ex.j;
            const uint32_t kbit = read_class(rec.flag[i], mode) << 31;
            if (spliced) { soa.sr_boff[run.s + ex.s] = im - soa.bB; soa.sr_joff[run.s + ex.s] = ij; }
            int32_t cur = rec.pos[i];
            bool last_n = false;
            int32_t a0 = 0;
            uint32_t nD = 0, first_m = 1;
            const uint32_t ij_first = ij;
            for (uint32_t kk = c0; kk < c1; ++kk) {
                const uint32_t w = rec.cigar[kk];
                const uint32_t op = w & 15u;
                const int32_t len = (int32_t)(w >> 4);
                if (op == 0u || op == 7u || op == 8u) {
                    if (first_m) { a0 = cur; first_m = 0; }
                    soa.m_start[im] = cur; soa.m_endk[im] = (uint32_t)(cur + len) | kbit; ++im;
                    cur += len; last_n = false;
                } else if (op == 3u) {
                    soa.jn_l[ij] = (uint32_t)(cur - 1) | (cur == rec.pos[i] ? 0x80000000u : 0u);    // S:482; the N starts at POS (POS <= t filter, S:435)
                    soa.jn_rk[ij] = (uint32_t)(cur + len - 1) | kbit;                   // S:483
                    ++ij;
                    cur += len; last_n = true;
                } else if (op == 2u) {
                    cur += len; ++nD;
                }
            }
            if (spliced) {
                // "simple" read: exactly block - N - block (the aggregated exception path needs only a0 and the end)
                const bool simple = nN == 1u && nM == 2u && nD == 0u && !last_n && !(soa.jn_l[ij_first] >> 31);
                const uint32_t tag = (run.s + ex.s) | (simple ? 0x80000000u : 0u);
                for (uint32_t jj = ij_first; jj < ij; ++jj) { soa.jn_read[jj] = tag; soa.ji_a0[jj] = a0; soa.ji_end[jj] = cur; }
            }
        }
        run.a += total.a; run.b += total.b; run.s += total.s; run.j += total.j;
    }
    if (blockIdx.x == gridDim.x - 1 && threadIdx.x == 0) {   // CSR sentinels
        soa.sr_boff[ck.s_base + ck.s_cnt] = ck.b_base + ck.b_cnt;
        soa.sr_joff[ck.s_base + ck.s_cnt] = ck.j_base + ck.j_cnt;
    }
}

// ------------------------------------------------------------------------------------------------
// K0d: bin partition of all M blocks (stream C).  Count and scatter traverse the record-ordered
// streams chunk by chunk; per-CTA shared-memory histograms (bins relative to the chunk's first
// bin) keep the global atomics down to one per (chunk, bin).
// ------------------------------------------------------------------------------------------------
constexpr int BIN_HIST = 2048;          // 512 kb of chunk span handled in shared memory

__global__ void k_bin_pad(DevBins bins) {        // pad every chromosome to a whole number of tiles
    const int c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= bins.n_chrom || !bins.chrom_tot[c]) return;
    const uint32_t pad = (K3_TILE - bins.chrom_tot[c] % K3_TILE) % K3_TILE;
    if (pad) atomicAdd(bins.bin_off + bins.chrom_bin_base[c + 1] - 1, pad);
}

template <bool SCATTER>
__global__ void __launch_bounds__(256) k_bin_pass(const Chunk* __restrict__ chunks, DevSoA soa, DevBins bins) {
    const Chunk ck = chunks[blockIdx.x >> 1];
    const bool bstream = blockIdx.x & 1;
    const uint32_t n = bstream ? ck.b_cnt : ck.a_cnt;
    if (n == 0) return;
    const uint32_t e0 = bstream ? soa.bB + ck.b_base : ck.a_base;
    const uint32_t gbase = bins.chrom_bin_base[ck.chrom];
    const int bin0 = max(bstream ? ck.s_lo : ck.a_lo, 0) >> BIN_SHIFT;
    __shared__ uint32_t hist[BIN_HIST];
    __shared__ uint32_t base[SCATTER ? BIN_HIST : 1];
    for (int i = threadIdx.x; i < BIN_HIST; i += 256) hist[i] = 0;
    __syncthreads();
    for (uint32_t e = e0 + threadIdx.x; e < e0 + n; e += 256) {
        const int rel = (max(soa.m_start[e], 0) >> BIN_SHIFT) - bin0;
        if (rel >= 0 && rel < BIN_HIST) atomicAdd(&hist[rel], 1u);
        else if (!SCATTER) atomicAdd(bins.bin_off + gbase + bin0 + rel, 1u);
    }
    __syncthreads();
    if constexpr (!SCATTER) {
        for (int i = threadIdx.x; i < BIN_HIST; i += 256)
            if (hist[i]) atomicAdd(bins.bin_off + gbase + bin0 + i, hist[i]);
        return;
    } else {
        for (int i = threadIdx.x; i < BIN_HIST; i += 256) {
            base[i] = hist[i] ? atomicAdd(bins.bin_cursor + gbase + bin0 + i, hist[i]) : 0u;
            hist[i] = 0;
        }
        __syncthreads();
        for (uint32_t e = e0 + threadIdx.x; e < e0 + n; e += 256) {
            const int32_t st = soa.m_start[e];
            const int rel = (max(st, 0) >> BIN_SHIFT) - bin0;
            uint32_t slot;
            if (rel >= 0 && rel < BIN_HIST) slot = base[rel] + atomicAdd(&hist[rel], 1u);
            else slot = atomicAdd(bins.bin_cursor + gbase + bin0 + rel, 1u);
            const uint32_t ek = soa.m_endk[e];
            bins.c_start[slot] = st;
            // stream C carries (start, len1 | class<<31) with len1 = end - 1 - start: site p is covered (S:469) iff
            // (uint32)(p - start) < len1; blocks of one base have len1 = 0 and never match
            bins.c_endk[slot] = (uint32_t)max((int32_t)(ek & POS_MASK) - 1 - st, 0) | (ek & 0x80000000u);
        }
    }
}

// the slots that pad a chromosome to a whole number of tiles: never-matching elements placed at the chromosome's
// largest block start, so that they do not widen the site window of the warp that holds them
__global__ void __launch_bounds__(256) k_bin_fill_pad(DevBins bins) {
    const int c = blockIdx.x;
    if (!bins.chrom_tot[c]) return;
    const uint32_t pad = (K3_TILE - bins.chrom_tot[c] % K3_TILE) % K3_TILE;
    const uint32_t end = bins.bin_off[bins.chrom_bin_base[c + 1]];
    for (uint32_t i = threadIdx.x; i < pad; i += 256) {
        bins.c_start[end - pad + i] = (int32_t)bins.chrom_ext[c];
        bins.c_endk[end - pad + i] = 0u;
    }
}

// generic exclusive scan of a u32 array (in place), a[n] receives the total
constexpr int SCAN_TILE = 4096;
__global__ void __launch_bounds__(256) k_scan_blocksum(const uint32_t* a, uint32_t n, uint32_t* sums) {
    __shared__ uint32_t red[8];
    uint32_t s = 0;
    const uint32_t b0 = blockIdx.x * SCAN_TILE;
    for (uint32_t i = b0 + threadIdx.x; i < min(b0 + SCAN_TILE, n); i += 256) s += a[i];
    s = __reduce_add_sync(0xffffffffu, s);
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = s;
    __syncthreads();
    if (threadIdx.x == 0) { for (int w = 1; w < 8; ++w) s += red[w]; sums[blockIdx.x] = s; }
}
__global__ void __launch_bounds__(1024) k_scan_sums(uint32_t* sums, uint32_t nblk, uint32_t* total_out) {
    __shared__ uint32_t wt[32];
    __shared__ uint32_t carry;
    if (threadIdx.x == 0) carry = 0;
    __syncthreads();
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    for (uint32_t base = 0; base < nblk; base += 1024) {
        const uint32_t i = base + threadIdx.x;
        const uint32_t v = i < nblk ? sums[i] : 0;
        uint32_t a = v;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) { const uint32_t x = __shfl_up_sync(0xffffffffu, a, d); if (lane >= d) a += x; }
        if (lane == 31) wt[warp] = a;
        __syncthreads();
        if (warp == 0) {
            const uint32_t w = wt[lane]; uint32_t b = w;
#pragma unroll
            for (int d = 1; d < 32; d <<= 1) { const uint32_t x = __shfl_up_sync(0xffffffffu, b, d); if (lane >= d) b += x; }
            wt[lane] = b - w;
        }
        __syncthreads();
        const uint32_t e = carry + wt[warp] + a - v;
        if (i < nblk) sums[i] = e;
        __syncthreads();
        if (threadIdx.x == 1023) carry = e + v;
        __syncthreads();
    }
    if (threadIdx.x == 0) *total_out = carry;
}
__global__ void __launch_bounds__(256) k_scan_apply(uint32_t* a, uint32_t n, const uint32_t* sums, uint32_t* copy) {
    __shared__ uint32_t wt[8];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const uint32_t b0 = blockIdx.x * SCAN_TILE + threadIdx.x * 16;      // 16 consecutive items per thread
    uint32_t v[16], t = 0;
#pragma unroll
    for (int q = 0; q < 16; ++q) { v[q] = (b0 + q < n) ? a[b0 + q] : 0u; t += v[q]; }
    uint32_t inc = t;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) { const uint32_t x = __shfl_up_sync(0xffffffffu, inc, d); if (lane >= d) inc += x; }
    if (lane == 31) wt[warp] = inc;
    __syncthreads();
    uint32_t run = sums[blockIdx.x] + inc - t;
    for (int w = 0; w < warp; ++w) run += wt[w];
#pragma unroll
    for (int q = 0; q < 16; ++q) {
        if (b0 + q < n) { a[b0 + q] = run; if (copy) copy[b0 + q] = run; }
        run += v[q];
    }
}

// per-tile site windows of stream C
__global__ void k_tile_hints(DevBins bins, DevGraph g) {
    const uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= bins.n_tiles) return;
    int lo = 0, hi = bins.n_chrom;                              // last chromosome with tile_base <= t
    while (hi - lo > 1) { const int mid = (lo + hi) >> 1; if (bins.chrom_tile_base[mid] <= t) lo = mid; else hi = mid; }
    const int c = lo;
    const uint32_t cb0 = bins.chrom_bin_base[c], cb1 = bins.chrom_bin_base[c + 1];
    const uint32_t e0 = bins.bin_off[cb0] + (t - bins.chrom_tile_base[c]) * K3_TILE, e1 = e0 + K3_TILE;
    auto bin_of = [&](uint32_t e) {                             // last bin of the chromosome with offset <= e
        uint32_t l = cb0, h = cb1;
        while (h - l > 1) { const uint32_t mid = (l + h) >> 1; if (bins.bin_off[mid] <= e) l = mid; else h = mid; }
        return l;
    };
    const uint32_t b0 = bin_of(e0), b1 = bin_of(e1 - 1);
    const int32_t plo = (int32_t)((b0 - cb0) << BIN_SHIFT);
    const int64_t phi64 = (int64_t)(((uint64_t)(b1 - cb0 + 1)) << BIN_SHIFT) + (int64_t)bins.max_len[0];
    const int32_t phi = (int32_t)min(phi64, (int64_t)INT_MAX - 1);
    const int s0 = g.cs_off[c], s1 = g.cs_off[c + 1];
    const int w_lo = lower_bound_i32(g.site_pos, s0, s1, plo);
    const int w_hi = upper_bound_i32(g.site_pos, w_lo, s1, phi);
    Tile tl;
    tl.e0 = e0; tl.w_lo = max(w_lo, g.own_lo); tl.w_hi = min(w_hi, g.own_hi); tl.pad = 0;
    bins.tiles[t] = tl;
}

// ------------------------------------------------------------------------------------------------
// K0e: junction groups.  Every N operator of the sample is inserted into an open-addressing table
// (one sub-table per chromosome, keys compared exactly); the table is then compacted into the dense
// distinct-junction arrays, and the simple instances are grouped per junction.
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ unsigned long long jkey(uint32_t lraw, uint32_t rraw) {
    return ~((unsigned long long)(lraw & POS_MASK) | ((unsigned long long)rraw << 32));    // never 0
}

__global__ void __launch_bounds__(256) k_jg_insert(const Chunk* __restrict__ chunks, DevSoA soa, DevJunc jg) {
    const Chunk ck = chunks[blockIdx.x];
    if (ck.j_cnt == 0) return;
    const uint32_t t0 = jg.tab_base[ck.chrom], tmask = jg.tab_base[ck.chrom + 1] - t0 - 1;
    const int lane = threadIdx.x & 31;
    for (uint32_t jb = ck.j_base; jb < ck.j_base + ck.j_cnt; jb += 256) {
        const uint32_t j = jb + threadIdx.x;
        const bool live = j < ck.j_base + ck.j_cnt;
        const unsigned long long key = live ? jkey(soa.jn_l[j], soa.jn_rk[j]) : 0ull;
        const bool simple = live && (soa.jn_read[j] >> 31);
        // neighbouring reads carry the same junction: one table access per distinct key of the warp
        const uint32_t peers = __match_any_sync(0xffffffffu, key);
        const uint32_t simple_peers = __ballot_sync(0xffffffffu, simple) & peers;
        uint32_t slot = 0;
        if (live && (int)(__ffs(peers) - 1) == lane) {
            uint32_t h = (uint32_t)((key * 0x9E3779B97F4A7C15ull) >> 32) & tmask;
            uint32_t probes = 0;
            for (;;) {
                const unsigned long long old = atomicCAS(jg.key + t0 + h, 0ull, key);
                if (old == 0ull || old == key) break;
                h = (h + 1) & tmask;
                if (++probes > min(tmask, 512u)) { atomicExch(jg.overflow, 1u); break; }      // the host re-sizes the table and retries
            }
            slot = t0 + h;
            atomicAdd(jg.s_all + slot, (uint32_t)__popc(peers));
            if (simple_peers) atomicAdd(jg.s_simple + slot, (uint32_t)__popc(simple_peers));
        }
        slot = __shfl_sync(0xffffffffu, slot, live ? (__ffs(peers) - 1) : 0);
        if (live) jg.slot_of[j] = slot;
    }
}

__global__ void k_jg_used(DevJunc jg) {
    const uint32_t s = blockIdx.x * blockDim.x + threadIdx.x;
    if (s < jg.n_slots) { jg.s_used[s] = jg.key[s] != 0ull; jg.s_off[s] = jg.s_simple[s]; jg.s_coff[s] = jg.s_all[s] - jg.s_simple[s]; }
    if (s == jg.n_slots) { jg.s_used[s] = 0; jg.s_off[s] = 0; jg.s_coff[s] = 0; }
}

__global__ void k_jg_compact(DevJunc jg, int n_chrom) {
    const uint32_t s = blockIdx.x * blockDim.x + threadIdx.x;
    if (s >= jg.n_slots || jg.key[s] == 0ull) return;
    const uint32_t d = jg.s_used[s];
    const unsigned long long key = ~jg.key[s];
    int lo = 0, hi = n_chrom;                                     // last chromosome with tab_base <= s
    while (hi - lo > 1) { const int mid = (lo + hi) >> 1; if (jg.tab_base[mid] <= s) lo = mid; else hi = mid; }
    jg.dj_l[d] = (uint32_t)(key & POS_MASK); jg.dj_rk[d] = (uint32_t)(key >> 32); jg.dj_chrom[d] = lo;
    jg.dj_all[d] = jg.s_all[s]; jg.dj_simple[d] = jg.s_simple[s]; jg.dj_off[d] = jg.s_off[s]; jg.dj_coff[d] = jg.s_coff[s];
}

__global__ void __launch_bounds__(256) k_jg_scatter(DevSoA soa, DevJunc jg) {
    const uint32_t j = blockIdx.x * blockDim.x + threadIdx.x;
    const bool live = j < soa.nJ;
    bool cx = false;
    uint32_t slot = 0;
    if (live) {
        slot = jg.slot_of[j];
        cx = !(soa.jn_read[j] >> 31);
    }
    // neighbouring reads carry the same junction: one cursor atomic per distinct (slot, kind) of the warp
    const uint32_t peers = __match_any_sync(0xffffffffu, live ? ((slot << 1) | (cx ? 1u : 0u)) : 0xffffffffu);
    const int lane = threadIdx.x & 31;
    const int leader = __ffs(peers) - 1;
    uint32_t base = 0;
    if (live && lane == leader) base = atomicAdd((cx ? jg.s_ccur : jg.s_cursor) + slot, (uint32_t)__popc(peers));
    base = __shfl_sync(0xffffffffu, base, leader);
    if (live) {
        const uint32_t rank = base + (uint32_t)__popc(peers & ((1u << lane) - 1u));
        if (cx) {
            const uint32_t ri = soa.jn_read[j] & POS_MASK;
            jg.cx_j[jg.s_coff[slot] + rank] = j;
            jg.cx_rng[jg.s_coff[slot] + rank] = make_uint4(soa.sr_joff[ri], soa.sr_joff[ri + 1], soa.bB + soa.sr_boff[ri], soa.bB + soa.sr_boff[ri + 1]);
        }
        else { const uint32_t p = jg.s_off[slot] + rank; jg.gi_a0[p] = soa.ji_a0[j]; jg.gi_end[p] = soa.ji_end[j]; }
    }
}

// ------------------------------------------------------------------------------------------------
// K1: alpha and PartnerCounts as segmented reductions of the junction scores
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ void alpha_reduce_item(const DevGraph& g, const DevOutputs& out, int i) {
    if (i < g.n_sites) {
        int64_t a = 0;
        for (int k = g.inc_off[i]; k < g.inc_off[i + 1]; ++k) a += g.j_score[g.inc_line[k]];
        out.alpha[i] = a;
    } else if (i < g.n_sites + g.n_edges) {
        const int e = i - g.n_sites;
        int64_t a = 0;
        for (int k = g.einc_beg[e]; k < g.einc_end[e]; ++k) a += g.j_score[g.einc_line[k]];
        out.pc_cnt[e] = a;
    }
}

// ------------------------------------------------------------------------------------------------
// Persistent, warp-specialised streaming kernels (K3, K4).
//
// grid = SMs x resident CTAs; every CTA has one producer warp and eight consumer warps.  The producer
// (one elected lane) pulls work items from a global atomic counter (dynamic scheduling: chunks differ
// a lot in cost), and for each piece of an item issues 1-D TMA bulk copies (cp.async.bulk) of the
// SoA slices and of the chunk's site window into a ring of shared-memory stages, completion tracked
// by mbarriers (full/empty pair per stage).  The consumers never touch HBM for streamed data: DRAM
// latency is hidden by the ring, not by occupancy.
// ------------------------------------------------------------------------------------------------
constexpr int PS_STAGES = 3;
constexpr int PS_CONSUMERS = 256;                  // 8 consumer warps
constexpr int PS_THREADS = PS_CONSUMERS + 32;      // + 1 producer warp
#ifndef SPL_K3_SITES
#define SPL_K3_SITES 504
#endif
constexpr int K3_SITES = SPL_K3_SITES;             // staged site positions per stage (2 KB; a tile's window is a few dozen sites)

struct StageMeta {
    uint32_t e0, e1;        // valid global element range of the item
    uint32_t p0, n;         // global index of staged element 0 (multiple of 4), staged element count
    int32_t  w_lo, w_hi;    // site window (global indices, already clamped to the owned range)
    int32_t  al;            // global site index of staged site 0
    uint32_t flags;         // PS_DONE | PS_GLOBAL_SITES
    int32_t  chunk;
    int32_t  sb_g0;         // global sb_off index of the chromosome's bin 0
    int32_t  sb_nb;         // bins of the chromosome (the sentinel sits at index sb_nb)
    int32_t  sb_al;         // global sb_off index of staged bin entry 0
};
constexpr uint32_t PS_DONE = 1u, PS_GLOBAL_SITES = 2u;

__device__ __forceinline__ void consumer_sync() { asm volatile("bar.sync 1, %0;" ::"n"(PS_CONSUMERS) : "memory"); }

struct K3Stage {
    int32_t  start[K3_TILE];
    uint32_t endk[K3_TILE];
    int32_t  sites[K3_SITES + 8];
};
struct K3Smem {
    K3Stage st[PS_STAGES];
    StageMeta meta[PS_STAGES];
    uint64_t full[PS_STAGES], empty[PS_STAGES];
};

// ------------------------------------------------------------------------------------------------
// K3: beta1 stabbing count over both block streams (A: unspliced reads, sorted; B: spliced reads).
// Each consumer warp narrows the staged site window to [min start, max end-2] of the 256 blocks it
// holds with two redux.sync and a warp-uniform binary search (broadcast LDS, no bank conflicts).
// Short narrowed ranges (the common case: 0-3 sites) are tested against the lane's blocks from
// registers and summed across the warp with one redux.sync per site -> one RED per (warp, site,
// class); long ranges (sparse coverage, displaced blocks of spliced reads) use a per-lane search.
// ------------------------------------------------------------------------------------------------
#ifndef SPL_K3_BATCH
#define SPL_K3_BATCH 4
#endif
constexpr int K3_BATCH = SPL_K3_BATCH;     // tiles a producer claims per atomic
constexpr int K3_GROUPS = 2;     // int4 groups (4 blocks each) per thread: a warp owns 256 consecutive elements of the tile
#ifndef SPL_K3_DENSE
#define SPL_K3_DENSE 12
#endif
constexpr int K3_DENSE = SPL_K3_DENSE;     // narrowed ranges longer than this use the per-lane search path
static_assert(K3_TILE == PS_CONSUMERS * K3_GROUPS * 4, "one pass of the consumer warps covers a tile");

__device__ __forceinline__ void k3_consume(const K3Stage& stg, const StageMeta& m, const int32_t* __restrict__ sp,
                                           const DevGraph& g, const DevCounters& cnt) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int4* gs = reinterpret_cast<const int4*>(stg.start);
    const uint4* gw = reinterpret_cast<const uint4*>(stg.endk);
    int a[K3_GROUPS * 4];
    uint32_t len[K3_GROUPS * 4], inc[K3_GROUPS * 4];
    int lo = INT_MAX, hi = INT_MIN;
#pragma unroll
    for (int u = 0; u < K3_GROUPS; ++u) {
        const int gi = (warp * K3_GROUPS + u) * 32 + lane;
        const int4 st = gs[gi];
        const uint4 w = gw[gi];
        const int sv[4] = {st.x, st.y, st.z, st.w};
        const uint32_t wv[4] = {w.x, w.y, w.z, w.w};
#pragma unroll
        for (int q = 0; q < 4; ++q) {
            const int e = u * 4 + q;
            a[e] = sv[q];
            len[e] = wv[q] & POS_MASK;                       // stabbed positions: start <= p < start + len
            inc[e] = 1u + (wv[q] >> 31) * 0xffffu;           // class 0 counts in the low half-word, class 1 in the high one
            lo = min(lo, sv[q]);
            hi = max(hi, sv[q] + (int)len[e]);
        }
    }
    const int wlo = __reduce_min_sync(0xffffffffu, lo), whi = __reduce_max_sync(0xffffffffu, hi) - 1;
    if (wlo > whi) return;
    int i0, i1;
    if (m.w_hi - m.w_lo <= 32) {                                     // usual case: one site per lane, two ballots
        const int sidx = m.w_lo + lane;
        const int sv = sidx < m.w_hi ? sp[sidx] : INT_MAX;
        i0 = m.w_lo + __popc(__ballot_sync(0xffffffffu, sv < wlo));
        i1 = m.w_lo + __popc(__ballot_sync(0xffffffffu, sv <= whi));
    } else {
        bound_pair_i32(sp, m.w_lo, m.w_hi, wlo, whi, i0, i1);
    }
    if (i0 >= i1) return;
    if (i1 - i0 <= K3_DENSE) {
        for (int s = i0; s < i1; ++s) {                           // warp-uniform loop
            const int p = sp[s];
            uint32_t c = 0;
#pragma unroll
            for (int e = 0; e < K3_GROUPS * 4; ++e)
                c += ((uint32_t)(p - a[e]) < len[e]) ? inc[e] : 0u;
            c = __reduce_add_sync(0xffffffffu, c);
            if (lane == 0 && c) {
                if (c & 0xffffu) atomicAdd(cnt.cov + s, c & 0xffffu);
                if (c >> 16) atomicAdd(cnt.cov + g.n_sites + s, c >> 16);
            }
        }
    } else {                                                       // wide window: per-lane search
#pragma unroll
        for (int e = 0; e < K3_GROUPS * 4; ++e) {
            if (!len[e]) continue;
            const uint32_t k = inc[e] >> 16;
            const int b = a[e] + (int)len[e] - 1;
            for (int s = lower_bound_i32(sp, i0, i1, a[e]); s < i1 && sp[s] <= b; ++s)
                atomicAdd(cnt.cov + k * g.n_sites + s, 1u);
        }
    }
}

__global__ void __launch_bounds__(PS_THREADS)
k_beta1_stab(DevBins bins, DevGraph g, DevCounters cnt) {
    extern __shared__ __align__(128) uint8_t smem_raw[];
    K3Smem& sm = *reinterpret_cast<K3Smem*>(smem_raw);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    if (threadIdx.x == 0) {
        for (int s = 0; s < PS_STAGES; ++s) { mbar_init(&sm.full[s], 1); mbar_init(&sm.empty[s], PS_CONSUMERS); }
    }
    __syncthreads();
    if (warp == PS_CONSUMERS / 32) {
        // ===== producer =====
        if (lane != 0) return;
        uint32_t it = 0;
        // tiles are claimed K3_BATCH at a time: the round trips of the claim (atomic) and of the descriptor loads are paid once
        // per batch, after the copies of the current batch are in flight
        uint32_t nbase = atomicAdd(cnt.work + 0, (uint32_t)K3_BATCH);
        Tile ntl[K3_BATCH];
#pragma unroll
        for (int b = 0; b < K3_BATCH; ++b) ntl[b] = bins.tiles[min(nbase + b, bins.n_tiles - 1u)];
        for (;;) {
            const uint32_t base = nbase;
            if (base >= bins.n_tiles) break;
            Tile tls[K3_BATCH];
#pragma unroll
            for (int b = 0; b < K3_BATCH; ++b) tls[b] = ntl[b];
#pragma unroll
            for (int b = 0; b < K3_BATCH; ++b) {
                const Tile tl = tls[b];
                if (base + b >= bins.n_tiles || tl.w_lo >= tl.w_hi) continue;     // past the end / zone-map prune: no (owned) site near this tile's bins
                const int site_n = tl.w_hi - tl.w_lo;
                const bool staged = site_n <= K3_SITES;
                const int al = tl.w_lo & ~3;
                const uint32_t nst = staged ? (uint32_t)(((tl.w_hi + 3) & ~3) - al) : 0u;
                const uint32_t stage = it % PS_STAGES, parity = (it / PS_STAGES) & 1u;
                mbar_wait_backoff(&sm.empty[stage], parity ^ 1u);
                StageMeta& m = sm.meta[stage];
                m.e0 = tl.e0; m.e1 = tl.e0 + K3_TILE; m.p0 = tl.e0; m.n = K3_TILE; m.w_lo = tl.w_lo; m.w_hi = tl.w_hi; m.al = al;
                m.flags = staged ? 0u : PS_GLOBAL_SITES; m.chunk = (int32_t)(base + b);
                mbar_expect_tx(&sm.full[stage], K3_TILE * 8u + nst * 4u);
                bulk_g2s(sm.st[stage].start, bins.c_start + tl.e0, K3_TILE * 4u, &sm.full[stage]);
                bulk_g2s(sm.st[stage].endk, bins.c_endk + tl.e0, K3_TILE * 4u, &sm.full[stage]);
                if (nst) bulk_g2s(sm.st[stage].sites, g.site_pos + al, nst * 4u, &sm.full[stage]);
                ++it;
            }
            nbase = atomicAdd(cnt.work + 0, (uint32_t)K3_BATCH);
#pragma unroll
            for (int b = 0; b < K3_BATCH; ++b) ntl[b] = bins.tiles[min(nbase + b, bins.n_tiles - 1u)];
        }
        const uint32_t stage = it % PS_STAGES, parity = (it / PS_STAGES) & 1u;
        mbar_wait_backoff(&sm.empty[stage], parity ^ 1u);
        sm.meta[stage].flags = PS_DONE;
        mbar_arrive(&sm.full[stage]);
        return;
    }
    // ===== consumers =====
    for (uint32_t it = 0;; ++it) {
        const uint32_t stage = it % PS_STAGES, parity = (it / PS_STAGES) & 1u;
        mbar_wait(&sm.full[stage], parity);
        const StageMeta m = sm.meta[stage];
        if (m.flags & PS_DONE) break;
        if (m.flags & PS_GLOBAL_SITES) k3_consume(sm.st[stage], m, g.site_pos, g, cnt);
        else k3_consume(sm.st[stage], m, sm.st[stage].sites - m.al, g, cnt);
        mbar_arrive(&sm.empty[stage]);       // every consumer thread releases the stage itself (release / acquire with the producer's wait)
    }
}

// Two views of the read that owns a complex junction instance: straight from the record-ordered SoA (three dependent
// DRAM round trips per item) or from the packed record k_junc_pack wrote at load time (one coalesced 96-byte load).
struct ReadGlobal {
    const DevSoA& soa;
    uint32_t j0, b0, nj, nb, jrel;
    __device__ __forceinline__ uint32_t jl(uint32_t x) const { return soa.jn_l[j0 + x]; }
    __device__ __forceinline__ uint32_t jr(uint32_t x) const { return soa.jn_rk[j0 + x]; }
    __device__ __forceinline__ int32_t bs(uint32_t x) const { return soa.m_start[b0 + x]; }
    __device__ __forceinline__ uint32_t be(uint32_t x) const { return soa.m_endk[b0 + x]; }
};
constexpr int CXP_WORDS = 24, CXP_MAXJ = 4, CXP_MAXB = 6;     // packed record: header, 4 junctions, 6 blocks, descriptor, class
struct ReadPacked {
    const uint32_t* w;
    uint32_t nj, nb, jrel;
    __device__ __forceinline__ uint32_t jl(uint32_t x) const { return w[1 + 2 * x]; }
    __device__ __forceinline__ uint32_t jr(uint32_t x) const { return w[2 + 2 * x]; }
    __device__ __forceinline__ int32_t bs(uint32_t x) const { return (int32_t)w[9 + 2 * x]; }
    __device__ __forceinline__ uint32_t be(uint32_t x) const { return w[10 + 2 * x]; }
};

// ------------------------------------------------------------------------------------------------
// K4: junction kernels over the DISTINCT junctions of the sample.
//   k_junc_lookup   (load time) one thread per distinct junction: site lookups through the bin index, offsets of its
//                   span range add, hot flags of its endpoints, pair sites, work lists
//   k_junc_span     span range add weighted by the junction's multiplicity (S:507-512)
//   k_junc_simple   one warp per hot (junction, endpoint): the junction's simple instances are classified at
//                   every exception site in aggregate -- flanking ones by the count alone, covering ones by a
//                   coalesced pass over the group's (first block start, read end) arrays
//   k_junc_complex  one thread per complex instance (several N, D or I splits) of a hot junction: the general
//                   per-read logic (k4_exceptions)
// ------------------------------------------------------------------------------------------------
constexpr uint32_t JS_CHUNK = 2048;

__global__ void __launch_bounds__(256) k_junc_lookup(DevJunc jg, DevGraph g, uint32_t mode) {
    const uint32_t d = blockIdx.x * blockDim.x + threadIdx.x;
    const bool live = d < jg.D;
    uint32_t hl = 0, hr = 0;
    if (live) {
        const int32_t l = (int32_t)jg.dj_l[d], r = (int32_t)(jg.dj_rk[d] & POS_MASK);
        const uint32_t k = jg.dj_rk[d] >> 31;
        const int c = jg.dj_chrom[d], s1 = g.cs_off[c + 1];
        const int il = site_lower(g, c, l);
        int iu = il;
        while (iu < s1 && g.site_pos[iu] == l) ++iu;                   // upper_bound(l)
        int ir = il;
        if (r > l) { ir = max(site_lower(g, c, r), iu); }
        const int x0 = max(iu, g.own_lo), x1 = min(ir, g.own_hi);     // sites strictly inside (l, r)
        jg.sp_x0[d] = 4u * (uint32_t)max(x0, 0) + 2u + k;                  // word of cnt.diff where k_junc_span adds +n / -n (S:507-512)
        jg.sp_x1[d] = x0 < x1 ? 4u * (uint32_t)x1 + 2u + k : 0xffffffffu;
        if (!(mode & FLAG_DEBUG_SKIP_EXC)) {
            if (il < s1 && g.site_pos[il] == l && g.site_hot[il]) hl = (uint32_t)il + 1u;
            if (ir < s1 && g.site_pos[ir] == r && g.site_hot[ir]) hr = (uint32_t)ir + 1u;
        }
        jg.hot_l[d] = hl; jg.hot_r[d] = hr;
    }
    // Reservations are aggregated per warp (one atomic per warp and list instead of one per hot junction).
    const int lane = threadIdx.x & 31;
    const uint32_t lt = (1u << lane) - 1u;
    const uint32_t sides = (hl ? 1u : 0u) + (hr ? 1u : 0u);
    // complex instances of a hot (junction, side): one descriptor reserves a range of the flat per-pass index space;
    // the 64-bit counter carries (descriptors << 40 | instances), so descriptor order == flat index order
    {
        const uint32_t nc = (live && sides) ? jg.dj_all[d] - jg.dj_simple[d] : 0u;
        const uint32_t nd = nc ? sides : 0u, ni = nc * sides;
        uint32_t pd = nd, pi = ni;                                     // inclusive warp scans
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const uint32_t a = __shfl_up_sync(0xffffffffu, pd, o), b = __shfl_up_sync(0xffffffffu, pi, o);
            if (lane >= o) { pd += a; pi += b; }
        }
        const uint32_t td = __shfl_sync(0xffffffffu, pd, 31), ti = __shfl_sync(0xffffffffu, pi, 31);
        if (td) {                                                      // warp-uniform
            unsigned long long old = 0;
            if (lane == 0) old = atomicAdd(reinterpret_cast<unsigned long long*>(jg.prep + 4), ((unsigned long long)td << 40) | ti);
            old = __shfl_sync(0xffffffffu, old, 0);
            uint32_t slot = (uint32_t)(old >> 40) + pd - nd, base = (uint32_t)(old & ((1ull << 40) - 1ull)) + pi - ni;
            if (nc) {
                for (int side = 0; side < 2; ++side) {
                    if (!(side == 0 ? hl : hr)) continue;
                    jg.cxd_base[slot] = base; jg.cxd_ds[slot] = (d << 1) | (uint32_t)side;
                    // the sites this (junction, side) is a partner/competitor pair for depend on the junction alone:
                    // found once here, not once per instance (CXD_T inline slots; more -> the instances walk the list)
                    const int anchor = (int)((side == 0 ? hl : hr) - 1u);
                    const int32_t jl = (int32_t)jg.dj_l[d], jr = (int32_t)(jg.dj_rk[d] & POS_MASK);
                    uint32_t nt = 0;
                    for (int q = g.rp_off[anchor]; q < g.rp_off[anchor + 1]; ++q) {
                        const int t = k4_pair_site(g, q, side, jl, jr);
                        if (t < 0) continue;
                        if (nt < (uint32_t)CXD_T) jg.cxd_t[slot * CXD_T + nt] = t;
                        ++nt;
                    }
                    jg.cxd_nt[slot] = nt;
                    ++slot; base += nc;
                }
            }
        }
    }
    // work list of hot (junction, side, chunk of simple instances) units; big groups are split so that one warp
    // never walks more than JS_CHUNK instances
    {
        const uint32_t ns = (live && sides) ? jg.dj_simple[d] : 0u;
        const uint32_t nch = (ns + JS_CHUNK - 1) / JS_CHUNK;
        const uint32_t nu = nch * sides;
        uint32_t pu = nu;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) { const uint32_t a = __shfl_up_sync(0xffffffffu, pu, o); if (lane >= o) pu += a; }
        const uint32_t tu = __shfl_sync(0xffffffffu, pu, 31);
        if (tu) {
            uint32_t base = 0;
            if (lane == 0) base = atomicAdd(jg.prep + 2, tu);
            base = __shfl_sync(0xffffffffu, base, 0);
            uint32_t p = base + pu - nu;
            if (nu) {
                for (int side = 0; side < 2; ++side) {
                    if (!(side == 0 ? hl : hr)) continue;
                    for (uint32_t c = 0; c < nch; ++c) jg.wl[p++] = ((unsigned long long)c << 32) | (d << 1) | (uint32_t)side;
                }
            }
        }
    }
    (void)lt;
}



// per pass: the span difference array gets +-multiplicity of every distinct junction at the offsets found at load time
__global__ void __launch_bounds__(256) k_junc_span(DevJunc jg, DevCounters cnt) {
    const uint32_t d = blockIdx.x * blockDim.x + threadIdx.x;
    if (d >= jg.D) return;
    const uint32_t x1 = jg.sp_x1[d];
    if (x1 == 0xffffffffu) return;
    const uint32_t n = jg.dj_all[d];
    atomicAdd(cnt.diff + jg.sp_x0[d], n);
    atomicAdd(cnt.diff + x1, 0u - n);
}

__global__ void __launch_bounds__(256) k_junc_simple(DevJunc jg, DevGraph g, DevCounters cnt, uint32_t mode) {
    const bool combine = (mode & FLAG_COMBINE) != 0;
    const int lane = threadIdx.x & 31;
    const uint32_t n_items = jg.prep[2];
    for (uint32_t item = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5); item < n_items; item += gridDim.x * (blockDim.x >> 5)) {
        const unsigned long long w64 = jg.wl[item];
        const uint32_t w = (uint32_t)w64, chunk = (uint32_t)(w64 >> 32);
        const uint32_t d = w >> 1;
        const int side = (int)(w & 1u);
        const uint32_t ns_all = jg.dj_simple[d];
        const uint32_t i0 = chunk * JS_CHUNK, i1 = min(ns_all, i0 + JS_CHUNK);
        const uint32_t ns = i1 - i0;
        const int32_t l = (int32_t)jg.dj_l[d], r = (int32_t)(jg.dj_rk[d] & POS_MASK);
        const uint32_t k = jg.dj_rk[d] >> 31;
        const int anchor = (int)((side == 0 ? jg.hot_l[d] : jg.hot_r[d]) - 1u);
        const int32_t other = side == 0 ? r : l;
        const uint32_t off = jg.dj_off[d] + i0;
        for (int q = g.rp_off[anchor]; q < g.rp_off[anchor + 1]; ++q) {     // warp-uniform loop
            const int t = g.rp_site[q];
            if (t < g.own_lo || t >= g.own_hi) continue;
            const int c0 = g.cp_off[t], c1 = g.cp_off[t + 1];
            if (c0 == c1 || !in_sorted(g.cp_pos, c0, c1, other)) continue;
            if (side == 1 && in_sorted(g.cp_pos, c0, c1, r) && in_list(g.pc_pos, g.pc_off[t], g.pc_off[t + 1], l)) continue;
            const int32_t tp = g.site_pos[t];
            const bool ok = strand_ok(g.site_cls[t], k);
            if (l < tp && tp < r) {                                    // flanking for every simple instance (S:503-505)
                if (lane == 0) {
                    if (ok) atomicAdd(cnt.spanx + t, ns);
                    if (combine) atomicAdd(cnt.flank + t, ns);
                }
            } else if (ok && tp != l && tp != r) {                     // beta1-type for the instances whose block covers t
                uint32_t c = 0;
                if (tp < l) { for (uint32_t i = lane; i < ns; i += 32) c += jg.gi_a0[off + i] <= tp; }
                else        { for (uint32_t i = lane; i < ns; i += 32) c += jg.gi_end[off + i] >= tp + 2; }
                c = __reduce_add_sync(0xffffffffu, c);
                if (c && lane == 0) {
                    atomicAdd(cnt.covx + t, c);
                    for (int e = g.pc_off[t]; e < g.pc_off[t + 1]; ++e)    // S:546-551: partners of t among the read's splice sites
                        if (g.pc_pos[e] == l || g.pc_pos[e] == r) atomicAdd(cnt.dc + e, c);
                }
            }
        }
    }
}

// flat index of a hot complex instance -> its descriptor: lane 0 of the warp searches, the others step forward (the warp's 32
// consecutive flat indices mostly share a descriptor)
__device__ __forceinline__ uint32_t cx_descriptor(const DevJunc& jg, uint32_t n_desc, uint32_t i) {
    const int lane = threadIdx.x & 31;
    uint32_t lo = 0;
    if (lane == 0) {
        uint32_t hi = n_desc;                                          // last descriptor with base <= i
        while (hi - lo > 1) { const uint32_t mid = (lo + hi) >> 1; if (jg.cxd_base[mid] <= i) lo = mid; else hi = mid; }
    }
    lo = __shfl_sync(__activemask(), lo, 0);
    while (lo + 1 < n_desc && jg.cxd_base[lo + 1] <= i) ++lo;
    return lo;
}

// load time: one packed record per hot complex instance, in flat-index order, so that the per-pass kernel reads its
// read's junctions and blocks with one coalesced load instead of chasing them through the SoA
__global__ void __launch_bounds__(256) k_junc_pack(DevSoA soa, DevJunc jg) {
    const unsigned long long w64 = *reinterpret_cast<const unsigned long long*>(jg.prep + 4);
    const uint32_t n_desc = (uint32_t)(w64 >> 40), n = (uint32_t)(w64 & ((1ull << 40) - 1ull));
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        const uint32_t lo = cx_descriptor(jg, n_desc, i);
        const uint32_t d = jg.cxd_ds[lo] >> 1;
        const uint32_t p = jg.dj_coff[d] + (i - jg.cxd_base[lo]);
        const uint32_t j = jg.cx_j[p];
        const uint4 rr = jg.cx_rng[p];                                 // the owning read: junctions [x, y), blocks [z, w)
        const uint32_t nj = rr.y - rr.x, nb = rr.w - rr.z;
        uint32_t* o = jg.cx_pack + (size_t)i * CXP_WORDS;
        for (int q = 0; q < CXP_WORDS; ++q) o[q] = 0u;                // the reader loads whole records
        if (nj > (uint32_t)CXP_MAXJ || nb > (uint32_t)CXP_MAXB) { o[0] = 0xffffffffu; o[21] = lo; continue; }    // walked through the SoA instead
        o[0] = nj | (nb << 8) | ((j - rr.x) << 16);
        for (uint32_t x = 0; x < nj; ++x) { o[1 + 2 * x] = soa.jn_l[rr.x + x]; o[2 + 2 * x] = soa.jn_rk[rr.x + x]; }
        for (uint32_t b = 0; b < nb; ++b) { o[9 + 2 * b] = (uint32_t)soa.m_start[rr.z + b]; o[10 + 2 * b] = soa.m_endk[rr.z + b]; }
        o[21] = lo;
    }
}

// per pass: the general per-read state machine for the complex instances of hot junctions
__global__ void __launch_bounds__(256) k_junc_complex(DevSoA soa, DevJunc jg, DevGraph g, DevCounters cnt, uint32_t mode) {
    const bool combine = (mode & FLAG_COMBINE) != 0;
    const unsigned long long w64 = *reinterpret_cast<const unsigned long long*>(jg.prep + 4);
    const uint32_t n = (uint32_t)(w64 & ((1ull << 40) - 1ull));
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        uint32_t w[CXP_WORDS];
        const uint4* src = reinterpret_cast<const uint4*>(jg.cx_pack + (size_t)i * CXP_WORDS);
#pragma unroll
        for (int q = 0; q < CXP_WORDS / 4; ++q) { const uint4 v = src[q]; w[4 * q] = v.x; w[4 * q + 1] = v.y; w[4 * q + 2] = v.z; w[4 * q + 3] = v.w; }
        const uint32_t lo = w[21];
        const uint32_t nt = jg.cxd_nt[lo];
        if (nt == 0) continue;
        const uint32_t ds = jg.cxd_ds[lo], d = ds >> 1;
        const int side = (int)(ds & 1u);
        const uint32_t k = jg.dj_rk[d] >> 31;
        if (w[0] != 0xffffffffu) {
            const ReadPacked rd{w, w[0] & 0xffu, (w[0] >> 8) & 0xffu, w[0] >> 16};
            if (nt <= (uint32_t)CXD_T) {
                for (uint32_t x = 0; x < nt; ++x) k4_classify(rd, g, cnt, jg.cxd_t[lo * CXD_T + x], k, combine);
            } else {
                const int anchor = (int)((side == 0 ? jg.hot_l[d] : jg.hot_r[d]) - 1u);
                const int32_t jl = (int32_t)jg.dj_l[d], jr = (int32_t)(jg.dj_rk[d] & POS_MASK);
                for (int q = g.rp_off[anchor]; q < g.rp_off[anchor + 1]; ++q) {
                    const int t = k4_pair_site(g, q, side, jl, jr);
                    if (t >= 0) k4_classify(rd, g, cnt, t, k, combine);
                }
            }
        } else {                                                       // long read: more junctions / blocks than a packed record holds
            const uint32_t p = jg.dj_coff[d] + (i - jg.cxd_base[lo]);
            const uint32_t j = jg.cx_j[p];
            const uint4 rr = jg.cx_rng[p];
            const ReadGlobal rd{soa, rr.x, rr.z, rr.y - rr.x, rr.w - rr.z, j - rr.x};
            const int anchor = (int)((side == 0 ? jg.hot_l[d] : jg.hot_r[d]) - 1u);
            const int32_t jl = (int32_t)jg.dj_l[d], jr = (int32_t)(jg.dj_rk[d] & POS_MASK);
            for (int q = g.rp_off[anchor]; q < g.rp_off[anchor + 1]; ++q) {
                const int t = k4_pair_site(g, q, side, jl, jr);
                if (t >= 0) k4_classify(rd, g, cnt, t, k, combine);
            }
        }
    }
}

// ------------------------------------------------------------------------------------------------
// K5: prefix scan of the four difference arrays + beta2 gather + SSE
// ------------------------------------------------------------------------------------------------
// blocks [0, nblk): per-block sums of the difference arrays; blocks beyond: alpha / PartnerCounts reduction (K1), which
// only has to be done before k_finalize and shares this launch
__global__ void __launch_bounds__(FIN_THREADS) k_span_blocksum(DevCounters cnt, int S, uint32_t* blk, int nblk, int blk0, DevGraph g, DevOutputs out) {
    if ((int)blockIdx.x >= nblk) {
        alpha_reduce_item(g, out, ((int)blockIdx.x - nblk) * FIN_THREADS + (int)threadIdx.x);
        return;
    }
    __shared__ uint32_t red[4][FIN_THREADS / 32];
    const int bx = (int)blockIdx.x + blk0;                 // only the blocks that hold owned sites (tile sharding)
    const int i = bx * FIN_THREADS + (int)threadIdx.x;
    uint4 v = make_uint4(0, 0, 0, 0);
    if (i < S) v = reinterpret_cast<const uint4*>(cnt.diff)[i];
    v.x = __reduce_add_sync(0xffffffffu, v.x); v.y = __reduce_add_sync(0xffffffffu, v.y);
    v.z = __reduce_add_sync(0xffffffffu, v.z); v.w = __reduce_add_sync(0xffffffffu, v.w);
    if ((threadIdx.x & 31) == 0) { const int w = threadIdx.x >> 5; red[0][w] = v.x; red[1][w] = v.y; red[2][w] = v.z; red[3][w] = v.w; }
    __syncthreads();
    if (threadIdx.x < 4) {
        uint32_t s = 0;
        for (int w = 0; w < FIN_THREADS / 32; ++w) s += red[threadIdx.x][w];
        blk[4 * bx + threadIdx.x] = s;
    }
}

__global__ void __launch_bounds__(FIN_THREADS)
k_finalize(DevGraph g, DevCounters cnt, DevOutputs out, uint32_t mode, int blk0) {
    const int S = g.n_sites;
    __shared__ uint32_t wt[4][FIN_THREADS / 32];
    __shared__ uint32_t pre[4][FIN_THREADS / 32];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int bx = (int)blockIdx.x + blk0;                 // blocks before blk0 hold no owned site: their sums are zero
    const int t = bx * FIN_THREADS + (int)threadIdx.x;     // one site per thread
    uint4 d = make_uint4(0, 0, 0, 0);
    if (t < S) d = reinterpret_cast<const uint4*>(cnt.diff)[t];
    uint32_t a[4] = {d.x, d.y, d.z, d.w};
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
#pragma unroll
        for (int c = 0; c < 4; ++c) { const uint32_t x = __shfl_up_sync(0xffffffffu, a[c], o); if (lane >= o) a[c] += x; }
    }
    if (lane == 31) { wt[0][warp] = a[0]; wt[1][warp] = a[1]; wt[2][warp] = a[2]; wt[3][warp] = a[3]; }
    // prefix over the preceding blocks' sums (k_span_blocksum): a few thousand values, summed by the block itself
    uint32_t p[4] = {0, 0, 0, 0};
    for (int b = blk0 + (int)threadIdx.x; b < bx; b += FIN_THREADS) {
        const uint4 s = reinterpret_cast<const uint4*>(out.span_blk)[b];
        p[0] += s.x; p[1] += s.y; p[2] += s.z; p[3] += s.w;
    }
#pragma unroll
    for (int c = 0; c < 4; ++c) p[c] = __reduce_add_sync(0xffffffffu, p[c]);
    if (lane == 0) { pre[0][warp] = p[0]; pre[1][warp] = p[1]; pre[2][warp] = p[2]; pre[3][warp] = p[3]; }
    __syncthreads();
    uint32_t run[4];                                        // inclusive prefix at site t
#pragma unroll
    for (int c = 0; c < 4; ++c) {
        uint32_t r = a[c];
        for (int w = 0; w < FIN_THREADS / 32; ++w) r += pre[c][w];
        for (int w = 0; w < warp; ++w) r += wt[c][w];
        run[c] = r;
    }
    if (t >= S) return;
    {   // + the direct counts of the same four kinds
        const uint4 dd = reinterpret_cast<const uint4*>(cnt.dir)[t];
        run[0] += dd.x; run[1] += dd.y; run[2] += dd.z; run[3] += dd.w;
    }

    const bool stranded = (mode & FLAG_STRANDED) != 0, cryptic = (mode & FLAG_CRYPTIC) != 0, combine = (mode & FLAG_COMBINE) != 0;
    const bool owned = t >= g.own_lo && t < g.own_hi;
    const uint32_t c = g.site_cls[t];
    uint32_t cov = 0, span = 0;
    if (!stranded || c == 1u) { cov = run[0] + cnt.cov[t]; span = run[2]; }
    else if (c == 2u) { cov = run[1] + cnt.cov[S + t]; span = run[3]; }
    const uint32_t covx = cnt.covx[t], spanx = cnt.spanx[t];
    int64_t b1 = (int64_t)cov - (int64_t)covx;
    int64_t b2 = (int64_t)covx + (int64_t)span - (int64_t)spanx + (combine ? (int64_t)cnt.flank[t] : 0);
    if (!owned || c == 4u) { b1 = 0; b2 = 0; }
    // ---- findBeta2Counts, S:581-623
    const int32_t tp = g.site_pos[t];
    const int64_t alpha_t = out.alpha[t];
    const int e_lo = g.pc_off[t], e_hi = g.pc_off[t + 1];
    int64_t b2c = 0;
    double b2w = 0.0;
    if (g.pt_is_pc) {
        // clean regime: Partners and PartnerCounts entries correspond one to one (a partner object per position), so the
        // double-count bookkeeping of S:592-611 stays in registers
        for (int x = g.pt_off[t]; x < g.pt_off[t + 1]; ++x) {
            const int pp_site = g.pt_site[x];
            const int32_t pp = g.pc_pos[x];
            int64_t tab = 0; bool hit = false;
            for (int y = g.pc_off[pp_site]; y < g.pc_off[pp_site + 1]; ++y) {      // S:592-599
                const int32_t cpos = g.pc_pos[y];
                if ((pp > tp && cpos < tp) || (pp < tp && cpos > tp)) { tab += out.pc_cnt[y]; hit = true; }
            }
            b2 += tab;
            const uint32_t dcv = cnt.dc[x];
            const int64_t pcount = out.pc_cnt[x];
            int64_t v = out.alpha[pp_site] - pcount;                       // S:606
            if (hit || dcv) { v -= (int64_t)dcv + tab; if (v < 0) v = 0; }       // subIntNoNeg, S:608-611
            b2c += v;
            const double wgt = alpha_t > 0 ? __ddiv_rn((double)pcount, (double)alpha_t) : 0.0;   // S:615
            b2w = __dadd_rn(b2w, __dmul_rn((double)v, wgt));               // mul then add, no FMA (S:617-619)
        }
    } else {
        for (int e = e_lo; e < e_hi; ++e) { out.dc_tot[e] = cnt.dc[e]; out.dc_present[e] = cnt.dc[e] != 0; }
        for (int x = g.pt_off[t]; x < g.pt_off[t + 1]; ++x) {
            const int pp_site = g.pt_site[x];
            const int32_t pp = g.site_pos[pp_site];
            int et = e_lo;
            while (et < e_hi && g.pc_pos[et] != pp) ++et;                  // PartnerCounts[pSite.getPos()], S:604
            int64_t tab = 0; bool hit = false;
            for (int y = g.pc_off[pp_site]; y < g.pc_off[pp_site + 1]; ++y) {  // S:592-599
                const int32_t cpos = g.pc_pos[y];
                if ((pp > tp && cpos < tp) || (pp < tp && cpos > tp)) { tab += out.pc_cnt[y]; hit = true; }
            }
            b2 += tab;
            if (et < e_hi) {
                if (hit) { out.dc_tot[et] += tab; out.dc_present[et] = 1; }
                const int64_t pcount = out.pc_cnt[et];
                int64_t v = out.alpha[pp_site] - pcount;                   // S:606
                if (out.dc_present[et]) { v -= out.dc_tot[et]; if (v < 0) v = 0; }   // subIntNoNeg, S:608-611
                b2c += v;
                const double wgt = alpha_t > 0 ? __ddiv_rn((double)pcount, (double)alpha_t) : 0.0;   // S:615
                b2w = __dadd_rn(b2w, __dmul_rn((double)v, wgt));           // mul then add, no FMA (S:617-619)
            }
        }
    }
    // ---- calculateSSE, S:626-639
    double sse = 0.0;
    if (cryptic) {
        const double betas = __dadd_rn((double)(b1 + b2), b2w);
        const double den = __dadd_rn((double)alpha_t, betas);
        if (den > 0.0) sse = __ddiv_rn((double)alpha_t, den);
    } else {
        const int64_t den = alpha_t + b1 + b2;
        if (den > 0) sse = __ddiv_rn((double)alpha_t, (double)den);
    }
    if (!owned) { b1 = 0; b2 = 0; b2c = 0; b2w = 0.0; sse = 0.0; }     // another tile's site: zero-filled (include/spliser_b200.h)
    out.beta1[t] = b1; out.beta2s[t] = b2; out.beta2c[t] = b2c; out.beta2w[t] = b2w; out.sse[t] = sse;
}

// ------------------------------------------------------------------------------------------------
// launchers
// ------------------------------------------------------------------------------------------------
// in-place exclusive scan of a[0..n); the total goes to *total_out (device).  tmp needs n / SCAN_TILE + 3 words.
void launch_exscan_u32(uint32_t* a, uint32_t n, uint32_t* tmp, uint32_t* total_out, void* stream) {
    cudaStream_t st = (cudaStream_t)stream;
    if (n == 0) { cudaMemsetAsync(total_out, 0, 4, st); return; }
    const uint32_t nblk = (n + SCAN_TILE - 1) / SCAN_TILE;
    { SPL_LAUNCH; k_scan_blocksum<<<nblk, 256, 0, st>>>(a, n, tmp); }
    { SPL_LAUNCH; k_scan_sums<<<1, 1024, 0, st>>>(tmp, nblk, total_out); }
    { SPL_LAUNCH; k_scan_apply<<<nblk, 256, 0, st>>>(a, n, tmp, nullptr); }
}
uint32_t exscan_tmp_words(uint32_t n) { return n / SCAN_TILE + 4; }
void launch_expand_count(const DevRecords& rec, Chunk* chunks, int n_chunks, uint32_t flags, DevBins bins, void* stream) {
    if (n_chunks > 0) { SPL_LAUNCH; k_expand_count<<<n_chunks, EXPAND_THREADS, 0, (cudaStream_t)stream>>>(rec, chunks, flags, bins); }
}
void launch_chunk_scan(Chunk* chunks, int n_chunks, uint32_t* totals8, DevBins bins, void* stream) {
    { SPL_LAUNCH; k_chunk_scan<<<1, 1024, 0, (cudaStream_t)stream>>>(chunks, n_chunks, totals8); }
    { SPL_LAUNCH; k_bin_layout<<<1, 32, 0, (cudaStream_t)stream>>>(bins, totals8); }
}
void launch_bin_partition(const Chunk* chunks, int n_chunks, DevSoA soa, DevBins bins, void* stream) {
    cudaStream_t st = (cudaStream_t)stream;
    if (n_chunks <= 0 || bins.total_bins == 0) return;
    cudaMemsetAsync(bins.bin_off, 0, ((size_t)bins.total_bins + 1) * 4, st);
    { SPL_LAUNCH; k_bin_pad<<<(bins.n_chrom + 127) / 128, 128, 0, st>>>(bins); }
    { SPL_LAUNCH; k_bin_pass<false><<<2 * n_chunks, 256, 0, st>>>(chunks, soa, bins); }
    const uint32_t n = bins.total_bins + 1;                              // the extra slot receives the total
    const uint32_t nblk = (n + SCAN_TILE - 1) / SCAN_TILE;
    { SPL_LAUNCH; k_scan_blocksum<<<nblk, 256, 0, st>>>(bins.bin_off, n, bins.scan_tmp); }
    { SPL_LAUNCH; k_scan_sums<<<1, 1024, 0, st>>>(bins.scan_tmp, nblk, bins.scan_tmp + nblk); }
    { SPL_LAUNCH; k_scan_apply<<<nblk, 256, 0, st>>>(bins.bin_off, n, bins.scan_tmp, bins.bin_cursor); }
    { SPL_LAUNCH; k_bin_pass<true><<<2 * n_chunks, 256, 0, st>>>(chunks, soa, bins); }
    { SPL_LAUNCH; k_bin_fill_pad<<<bins.n_chrom, 256, 0, st>>>(bins); }
}
void launch_tile_hints(DevBins bins, DevGraph g, void* stream) {
    if (bins.n_tiles) { SPL_LAUNCH; k_tile_hints<<<(bins.n_tiles + 127) / 128, 128, 0, (cudaStream_t)stream>>>(bins, g); }
}
void launch_expand_scatter(const DevRecords& rec, const Chunk* chunks, int n_chunks, DevSoA soa, uint32_t flags, void* stream) {
    if (n_chunks > 0) { SPL_LAUNCH; k_expand_scatter<<<n_chunks, EXPAND_THREADS, 0, (cudaStream_t)stream>>>(rec, chunks, soa, flags); }
}
// SM count of the CURRENT device (one process may drive several devices, one context each)
int sm_count_current_device() {
    static std::mutex mu;
    static int sms_of[64] = {0};
    int dev = 0;
    cudaGetDevice(&dev);
    std::lock_guard<std::mutex> lock(mu);
    if (dev >= 0 && dev < 64 && sms_of[dev]) return sms_of[dev];
    int sms = 0;
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    if (sms < 1) sms = 1;
    if (dev >= 0 && dev < 64) sms_of[dev] = sms;
    return sms;
}
// Grid of the persistent K3 kernel on the CURRENT device: the dynamic shared-memory attribute and the SM count belong to a
// device, and one process may drive several (one context per device, e.g. the sample-sharded re-count of `combine`).
static int beta1_grid() {
    static std::mutex mu;
    static int grid_of[64] = {0};
    int dev = 0;
    cudaGetDevice(&dev);
    std::lock_guard<std::mutex> lock(mu);
    if (dev >= 0 && dev < 64 && grid_of[dev]) return grid_of[dev];
    int sms = 0;
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    cudaFuncSetAttribute((const void*)k_beta1_stab, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(K3Smem));
    int per_sm = 1;
    cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, (const void*)k_beta1_stab, PS_THREADS, sizeof(K3Smem));
    if (per_sm < 1) per_sm = 1;
    const int grid = sms * per_sm;           // one resident CTA per slot: a multiple of the SM count
    if (dev >= 0 && dev < 64) grid_of[dev] = grid;
    return grid;
}
void launch_beta1(DevBins bins, DevGraph g, DevCounters cnt, void* stream) {
    if (bins.n_tiles == 0 || g.n_sites <= 0) return;
    { SPL_LAUNCH; k_beta1_stab<<<beta1_grid(), PS_THREADS, sizeof(K3Smem), (cudaStream_t)stream>>>(bins, g, cnt); }
}
// phase A: table insert + scans; totals3[0] = distinct junctions, [1] = simple instances (read by the host to size
// the dense arrays).  phase B: compaction + grouping; totals3[2] = complex instances, [3] = overflow flag.
void launch_junction_groups_a(const Chunk* chunks, int n_chunks, DevSoA soa, DevJunc jg, uint32_t* totals4, void* stream) {
    cudaStream_t st = (cudaStream_t)stream;
    cudaMemsetAsync(totals4, 0, 16, st);
    if (n_chunks <= 0 || jg.n_slots == 0 || soa.nJ == 0) return;
    cudaMemsetAsync(jg.key, 0, (size_t)jg.n_slots * 8, st);
    cudaMemsetAsync(jg.s_all, 0, (size_t)jg.n_slots * 4, st);
    cudaMemsetAsync(jg.s_simple, 0, (size_t)jg.n_slots * 4, st);
    cudaMemsetAsync(jg.s_cursor, 0, (size_t)jg.n_slots * 4, st);
    cudaMemsetAsync(jg.s_ccur, 0, (size_t)jg.n_slots * 4, st);
    cudaMemsetAsync(jg.cx_n, 0, 8, st);                                  // cx_n and overflow are adjacent
    { SPL_LAUNCH; k_jg_insert<<<n_chunks, 256, 0, st>>>(chunks, soa, jg); }
    const uint32_t n = jg.n_slots + 1;
    { SPL_LAUNCH; k_jg_used<<<(n + 255) / 256, 256, 0, st>>>(jg); }
    const uint32_t nblk = (n + SCAN_TILE - 1) / SCAN_TILE;
    { SPL_LAUNCH; k_scan_blocksum<<<nblk, 256, 0, st>>>(jg.s_used, n, jg.scan_tmp); }
    { SPL_LAUNCH; k_scan_sums<<<1, 1024, 0, st>>>(jg.scan_tmp, nblk, jg.scan_tmp + nblk); }
    { SPL_LAUNCH; k_scan_apply<<<nblk, 256, 0, st>>>(jg.s_used, n, jg.scan_tmp, nullptr); }
    { SPL_LAUNCH; k_scan_blocksum<<<nblk, 256, 0, st>>>(jg.s_off, n, jg.scan_tmp); }
    { SPL_LAUNCH; k_scan_sums<<<1, 1024, 0, st>>>(jg.scan_tmp, nblk, jg.scan_tmp + nblk); }
    { SPL_LAUNCH; k_scan_apply<<<nblk, 256, 0, st>>>(jg.s_off, n, jg.scan_tmp, nullptr); }
    { SPL_LAUNCH; k_scan_blocksum<<<nblk, 256, 0, st>>>(jg.s_coff, n, jg.scan_tmp); }
    { SPL_LAUNCH; k_scan_sums<<<1, 1024, 0, st>>>(jg.scan_tmp, nblk, jg.scan_tmp + nblk); }
    { SPL_LAUNCH; k_scan_apply<<<nblk, 256, 0, st>>>(jg.s_coff, n, jg.scan_tmp, nullptr); }
    cudaMemcpyAsync(totals4 + 2, jg.s_coff + jg.n_slots, 4, cudaMemcpyDeviceToDevice, st);
    cudaMemcpyAsync(totals4, jg.s_used + jg.n_slots, 4, cudaMemcpyDeviceToDevice, st);
    cudaMemcpyAsync(totals4 + 1, jg.s_off + jg.n_slots, 4, cudaMemcpyDeviceToDevice, st);
    cudaMemcpyAsync(totals4 + 3, jg.overflow, 4, cudaMemcpyDeviceToDevice, st);
}
void launch_jtab_layout(DevBins bins, int attempt, uint32_t* totals8, void* stream) {
    { SPL_LAUNCH; k_jtab_layout<<<1, 32, 0, (cudaStream_t)stream>>>(bins, attempt, totals8); }
}
void launch_junction_groups_b(DevSoA soa, DevJunc jg, int n_chrom, uint32_t* totals4, void* stream) {
    cudaStream_t st = (cudaStream_t)stream;
    if (jg.n_slots == 0 || soa.nJ == 0) return;
    { SPL_LAUNCH; k_jg_compact<<<(jg.n_slots + 255) / 256, 256, 0, st>>>(jg, n_chrom); }
    { SPL_LAUNCH; k_jg_scatter<<<(soa.nJ + 255) / 256, 256, 0, st>>>(soa, jg); }
    cudaMemcpyAsync(totals4 + 3, jg.overflow, 4, cudaMemcpyDeviceToDevice, st);
}
void launch_junctions(DevSoA soa, DevJunc jg, DevGraph g, DevCounters cnt, uint32_t flags, void* stream) {
    cudaStream_t st = (cudaStream_t)stream;
    if (jg.D == 0 || g.n_sites <= 0) return;
    { SPL_LAUNCH; k_junc_span<<<(jg.D + 255) / 256, 256, 0, st>>>(jg, cnt); }
    const int sms = sm_count_current_device();
    { SPL_LAUNCH; k_junc_simple<<<sms * 8, 256, 0, st>>>(jg, g, cnt, flags); }
    if (jg.n_complex && jg.cx_pack) { SPL_LAUNCH; k_junc_complex<<<sms * 8, 256, 0, st>>>(soa, jg, g, cnt, flags); }
}
// load time (after the site table is on the device): per distinct junction, the site lookups, hot flags, pair sites and the
// work lists of the exception kernels -- all functions of (sample junctions x site table), like the tile hints
void launch_junction_prepare(DevJunc jg, DevGraph g, uint32_t flags, void* stream) {
    cudaStream_t st = (cudaStream_t)stream;
    if (jg.D == 0 || g.n_sites <= 0) return;
    cudaMemsetAsync(jg.prep, 0, 32, st);
    { SPL_LAUNCH; k_junc_lookup<<<(jg.D + 255) / 256, 256, 0, st>>>(jg, g, flags); }
}
void launch_junction_pack(DevSoA soa, DevJunc jg, void* stream) {
    if (jg.D == 0 || jg.n_complex == 0 || !jg.cx_pack) return;
    const int sms = sm_count_current_device();
    { SPL_LAUNCH; k_junc_pack<<<sms * 8, 256, 0, (cudaStream_t)stream>>>(soa, jg); }
}
void launch_finalize(DevGraph g, DevCounters cnt, DevOutputs out, uint32_t flags, void* stream) {
    if (g.n_sites <= 0) return;
    // only the blocks of FIN_THREADS sites that hold sites this context owns (all of them without tile sharding)
    const int lo = min(max(g.own_lo, 0), g.n_sites), hi = min(max(g.own_hi, lo), g.n_sites);
    const int blk0 = lo / FIN_THREADS, nblk = hi > lo ? (hi - 1) / FIN_THREADS - blk0 + 1 : 0;
    const int nalpha = (g.n_sites + g.n_edges + FIN_THREADS - 1) / FIN_THREADS;
    { SPL_LAUNCH; k_span_blocksum<<<nblk + nalpha, FIN_THREADS, 0, (cudaStream_t)stream>>>(cnt, g.n_sites, out.span_blk, nblk, blk0, g, out); }
    if (nblk) { SPL_LAUNCH; k_finalize<<<nblk, FIN_THREADS, 0, (cudaStream_t)stream>>>(g, cnt, out, flags, blk0); }
}
int kernel_launch_count_per_pass() { return 6; }   // stabbing variant: beta1_stab, junc_span, junc_simple, junc_complex, span_blocksum (+ alpha reduce), finalize

}  // namespace spl
