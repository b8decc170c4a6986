// Library strandedness: one vote per record (rule: include/spliser_b200.h, spl_gene_strands).  The host indexes the genes; the
// kernel reads each record once where the ingest left it and adds its vote to three block-reduced 64-bit counters.
#include <cuda_runtime.h>

#include <algorithm>
#include <cstdio>

#include "strand_votes.h"

namespace spl {

std::string build_gene_index(const spl_gene_strands* g, int32_t n_chrom, GeneIndexHost& h) {
    h = GeneIndexHost{};
    if (n_chrom < 0) return "negative chromosome count";
    if (!g) return "gene view is NULL";
    if (g->n_chrom < 0 || g->n_chrom > n_chrom) return "gene view covers more chromosomes than the call";
    if (g->n_chrom > 0 && !g->chrom_off) return "chrom_off is NULL";
    const int64_t G = g->n_chrom > 0 ? g->chrom_off[g->n_chrom] : 0;
    if (g->n_chrom > 0 && g->chrom_off[0] != 0) return "chrom_off[0] must be 0";
    for (int32_t c = 0; c < g->n_chrom; ++c)
        if (g->chrom_off[c + 1] < g->chrom_off[c]) return "chrom_off must be monotone";
    if (G > 0 && (!g->left || !g->right || !g->strand)) return "NULL gene array";
    if (G >= (int64_t)INT32_MAX / 4) return "too many genes";
    h.bnd_off.assign((size_t)n_chrom + 1, 0);
    std::vector<uint8_t> mask;
    std::vector<int32_t> b, dp, dm;
    for (int32_t c = 0; c < n_chrom; ++c) {
        b.clear();
        const int64_t g0 = c < g->n_chrom ? g->chrom_off[c] : 0, g1 = c < g->n_chrom ? g->chrom_off[c + 1] : 0;
        auto valid = [&](int64_t k) { return (g->strand[k] == '+' || g->strand[k] == '-') && g->right[k] > g->left[k]; };
        for (int64_t k = g0; k < g1; ++k)
            if (valid(k)) { b.push_back(g->left[k]); b.push_back(g->right[k]); }
        std::sort(b.begin(), b.end());
        b.erase(std::unique(b.begin(), b.end()), b.end());
        // every gene covers the elementary intervals [lower_bound(left), lower_bound(right)): difference counts per strand
        dp.assign(b.size() + 1, 0); dm.assign(b.size() + 1, 0);
        for (int64_t k = g0; k < g1; ++k) {
            if (!valid(k)) continue;
            const size_t a = (size_t)(std::lower_bound(b.begin(), b.end(), g->left[k]) - b.begin());
            const size_t e = (size_t)(std::lower_bound(b.begin(), b.end(), g->right[k]) - b.begin());
            std::vector<int32_t>& d = g->strand[k] == '+' ? dp : dm;
            ++d[a]; --d[e];
        }
        int32_t sp = 0, sm = 0;
        for (size_t k = 0; k < b.size(); ++k) {
            sp += dp[k]; sm += dm[k];
            mask.push_back((uint8_t)((sp > 0 ? 1 : 0) | (sm > 0 ? 2 : 0)));
        }
        h.bnd.insert(h.bnd.end(), b.begin(), b.end());
        h.bnd_off[(size_t)c + 1] = (int32_t)h.bnd.size();
    }
    h.m = (uint32_t)mask.size();
    h.levels = 1;
    while (h.m >> h.levels) ++h.levels;                     // levels j with 2^j <= m
    h.table.assign((size_t)h.levels * h.m, 0);
    std::copy(mask.begin(), mask.end(), h.table.begin());
    for (int32_t j = 1; j < h.levels; ++j) {
        const size_t half = (size_t)1 << (j - 1), span = (size_t)1 << j;
        uint8_t* t = h.table.data() + (size_t)j * h.m;
        const uint8_t* s = t - h.m;
        for (size_t i = 0; i + span <= h.m; ++i) t[i] = s[i] | s[i + half];
    }
    return "";
}

namespace {

constexpr int SV_THREADS = 256;
constexpr uint32_t REF_OPS = (1u << 0) | (1u << 2) | (1u << 3) | (1u << 7) | (1u << 8);   // M D N = X move along the reference

// One block per chunk (FC_RECS records of one chromosome), one record per thread and round.  ANNOT: the reference strand from
// the gene index over the record's span (its CIGAR walked for L); else from the XS column.
template <bool ANNOT>
__global__ void __launch_bounds__(SV_THREADS) k_strand_votes(DevRecords rec, const uint8_t* __restrict__ xs,
                                                             const FChunk* __restrict__ chunks, GeneIndexDev gi,
                                                             unsigned long long* __restrict__ counts) {
    const int32_t chrom = chunks[blockIdx.x].chrom;
    const uint32_t r0 = chunks[blockIdx.x].rec_lo, r1 = chunks[blockIdx.x].rec_hi;
    int32_t b0 = 0, b1 = 0;
    if (ANNOT && chrom < gi.n_chrom) { b0 = gi.bnd_off[chrom]; b1 = gi.bnd_off[chrom + 1]; }
    uint32_t agree = 0, opposite = 0, none = 0;
    for (uint32_t r = r0 + threadIdx.x; r < r1; r += SV_THREADS) {
        const uint32_t c0 = __ldg(rec.cig_off + r), c1 = __ldg(rec.cig_off + r + 1);
        if (c1 == c0) continue;                                 // no CIGAR operator: not a kept record
        const uint32_t f = __ldg(rec.flag + r);
        const bool first = (f & 64u) || !(f & 1u);
        const bool fr_plus = first != ((f & 16u) != 0);
        uint32_t ref;                                           // bit 0 '+', bit 1 '-'
        if (ANNOT) {
            int64_t L = 0;
            for (uint32_t k = c0; k < c1; ++k) {
                const uint32_t op = __ldg(rec.cigar + k);
                if ((REF_OPS >> (op & 15u)) & 1u) L += op >> 4;
            }
            if (L == 0) L = 1;
            const int64_t p = (int64_t)__ldg(rec.pos + r) - 1;
            ref = gene_strand_mask(gi.bnd, gi.table, gi.m, b0, b1, p, p + L);
        } else {
            const uint8_t x = __ldg(xs + r);
            ref = x == '+' ? 1u : (x == '-' ? 2u : 0u);
        }
        if (ref == 1u || ref == 2u) {
            if ((ref == 1u) == fr_plus) ++agree; else ++opposite;
        } else {
            ++none;
        }
    }
    agree = __reduce_add_sync(0xffffffffu, agree);
    opposite = __reduce_add_sync(0xffffffffu, opposite);
    none = __reduce_add_sync(0xffffffffu, none);
    __shared__ uint32_t part[3][SV_THREADS / 32];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    if (lane == 0) { part[0][warp] = agree; part[1][warp] = opposite; part[2][warp] = none; }
    __syncthreads();
    if (threadIdx.x < 3) {
        unsigned long long s = 0;
        for (int w = 0; w < SV_THREADS / 32; ++w) s += part[threadIdx.x][w];
        if (s) atomicAdd(counts + threadIdx.x, s);
    }
}

}  // namespace

void launch_strand_votes(const DevRecords& rec, const uint8_t* xs, const FChunk* chunks, uint32_t n_chunks, const GeneIndexDev* gi,
                         unsigned long long* counts, void* stream) {
    if (!n_chunks) return;
    cudaStream_t s = (cudaStream_t)stream;
    SPL_LAUNCH;
    if (gi) k_strand_votes<true><<<n_chunks, SV_THREADS, 0, s>>>(rec, nullptr, chunks, *gi, counts);
    else k_strand_votes<false><<<n_chunks, SV_THREADS, 0, s>>>(rec, xs, chunks, GeneIndexDev{}, counts);
}

}  // namespace spl

extern "C" int spl_debug_gene_strand_mask(int32_t n_chrom, const spl_gene_strands* genes, int64_t n, const int32_t* chrom,
                                          const int64_t* start, const int64_t* len, uint8_t* mask_out, char* err, int err_len) {
    auto fail = [&](const std::string& why) {
        if (err && err_len > 0) snprintf(err, (size_t)err_len, "%s", why.c_str());
        return (int)SPL_ERR_ARG;
    };
    spl::GeneIndexHost h;
    const std::string e = spl::build_gene_index(genes, n_chrom, h);
    if (!e.empty()) return fail(e);
    if (n < 0 || (n > 0 && (!chrom || !start || !len || !mask_out))) return fail("bad query arrays");
    for (int64_t i = 0; i < n; ++i) {
        if (chrom[i] < 0 || chrom[i] >= n_chrom) return fail("query chromosome out of range");
        if (len[i] <= 0) return fail("query length must be positive");
        mask_out[i] = (uint8_t)spl::gene_strand_mask(h.bnd.data(), h.table.data(), h.m, h.bnd_off[(size_t)chrom[i]],
                                                     h.bnd_off[(size_t)chrom[i] + 1], start[i], start[i] + len[i]);
    }
    return SPL_OK;
}
