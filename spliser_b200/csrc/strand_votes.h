// Library strandedness: the gene-strand index and the vote kernel (strand_votes.cu).  The rule is stated in
// include/spliser_b200.h at spl_gene_strands.
#pragma once
#include <cstdint>
#include <string>
#include <vector>

#include "../../include/spliser_b200.h"
#include "device_types.h"

namespace spl {

// Per caller chromosome c the sorted distinct gene boundaries bnd[bnd_off[c] .. bnd_off[c + 1]); entry k of them also indexes
// the elementary interval [bnd[k], bnd[k + 1]) and its strand mask (bit 0 '+', bit 1 '-'; the chromosome's last entry is 0).
// table[j * m + i] = OR of the masks i .. i + 2^j - 1 (sparse table over all m entries; level 0 is the masks).
struct GeneIndexHost {
    std::vector<int32_t> bnd, bnd_off;
    std::vector<uint8_t> table;
    uint32_t m = 0;
    int32_t levels = 0;
};

struct GeneIndexDev {
    const int32_t* bnd;
    const int32_t* bnd_off;       // [n_chrom + 1]
    const uint8_t* table;         // [levels * m]
    uint32_t m;
    int32_t n_chrom;
};

// "" or the reason the view is malformed.  n_chrom: the caller's chromosome count (the view may cover fewer).
std::string build_gene_index(const spl_gene_strands* g, int32_t n_chrom, GeneIndexHost& out);

// Range-OR of the masks of the elementary intervals of one chromosome's boundaries bnd[b0 .. b1) that meet [p, q) (p < q).
__host__ __device__ inline uint32_t gene_strand_mask(const int32_t* bnd, const uint8_t* table, uint32_t m, int32_t b0, int32_t b1,
                                                     int64_t p, int64_t q) {
    const int32_t nb = b1 - b0;
    if (nb < 2) return 0;
    const int32_t* B = bnd + b0;
    int32_t lo = 0, hi = nb;                      // upper_bound(B, p)
    while (lo < hi) { const int32_t mid = (lo + hi) >> 1; if ((int64_t)B[mid] <= p) lo = mid + 1; else hi = mid; }
    int32_t k_lo = lo - 1;
    lo = 0; hi = nb;                              // lower_bound(B, q)
    while (lo < hi) { const int32_t mid = (lo + hi) >> 1; if ((int64_t)B[mid] < q) lo = mid + 1; else hi = mid; }
    int32_t k_hi = lo - 1;
    if (k_lo < 0) k_lo = 0;
    if (k_hi > nb - 2) k_hi = nb - 2;
    if (k_lo > k_hi) return 0;
    const uint32_t len = (uint32_t)(k_hi - k_lo + 1);
#ifdef __CUDA_ARCH__
    const int j = 31 - __clz(len);
#else
    int j = 0;
    while ((2u << j) <= len) ++j;
#endif
    return (uint32_t)table[(size_t)j * m + (size_t)(b0 + k_lo)] | (uint32_t)table[(size_t)j * m + (size_t)(b0 + k_hi - (1 << j) + 1)];
}

// counts[3] (u64, zeroed by the caller) += the votes of the records of chunks [0, n_chunks) (SPL_VOTE_* order).  gi == NULL: the
// XS source, from xs[]; otherwise the annotation source.
void launch_strand_votes(const DevRecords& rec, const uint8_t* xs, const FChunk* chunks, uint32_t n_chunks, const GeneIndexDev* gi,
                         unsigned long long* counts, void* stream);

}  // namespace spl
