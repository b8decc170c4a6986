// Device-side construction of the site table and competing-site graph (graph_build.cu).
#pragma once
#include <cuda_runtime.h>

#include <cstdint>
#include <string>
#include <vector>

namespace spl {

struct GbBuf {                       // grow-only device allocation
    void* p = nullptr;
    size_t cap = 0;
    cudaError_t reserve(size_t bytes) {
        if (bytes <= cap) return cudaSuccess;
        if (p) cudaFree(p);
        p = nullptr; cap = 0;
        const size_t want = bytes + bytes / 8 + 4096;
        cudaError_t e = cudaMalloc(&p, want);
        if (e == cudaSuccess) cap = want;
        return e;
    }
    void release() { if (p) cudaFree(p); p = nullptr; cap = 0; }
};

struct GraphBuildMem {
    GbBuf fin, fin2, work, work2;    // final arrays (sized by J / by C and the bin count), workspaces
    uint32_t* h_cnt = nullptr;       // pinned, 16 words
    uint32_t scan_epoch = 0;         // look-back scans: a new epoch per launch
    uint32_t nb_host = 0;            // entries of the direct-address bin index (exact, from the junction table)
    size_t cap_c = 0;                // capacity of the competitor array (checked on the device; grown and re-run when too small)
    bool ready = false;              // phase 0 has run on these buffers
};

// writable view of the arrays DevGraph points at, plus what only the host-facing result needs
struct GraphDev {
    int32_t *cs_off, *sb_base, *sb_off;
    int32_t *site_chrom, *site_pos;
    uint8_t *site_strand, *site_cls, *site_hot;
    int64_t *first_line;
    int32_t *pt_off, *pt_site, *pc_pos;
    int32_t *cp_off, *cp_pos;
    int32_t *rp_off, *rp_site;
    int32_t *inc_off, *inc_line;
    int32_t *einc_beg, *einc_end, *einc_line;
    int64_t *j_score;
    int64_t *pt_off64, *cp_off64;    // offsets widened for the ABI
};

struct GraphCounts { uint32_t S = 0, E = 0, C = 0, NB = 0; double h2d_bytes = 0; };

// do the packed sort keys fit in 64 bits for a table of J rows?
bool graph_build_fits(int64_t J, int32_t n_chrom, int32_t max_pos);

// clean-regime build on `stream`.  Phase 1 synchronises the stream ONCE, at the end, to read the table sizes; phase 2 runs
// the same kernels without any host synchronisation (timed rebuild of a table whose sizes are known).  false + err on failure.
bool graph_build_device(GraphBuildMem& m, const int32_t* j_chrom, const int32_t* j_left, const int32_t* j_right, const uint8_t* j_strand,
                        const int64_t* j_score, int64_t n_junc, int32_t n_chrom, int32_t max_pos, bool stranded, void* stream,
                        int phase /* 0: allocate + upload the junction table, 1: build + read sizes, 2: build only */, GraphDev& g, GraphCounts& counts, std::string& err);

// junction extraction from device-resident records (graph_build.cu, shares its sort / scan kernels); start / end: the rows'
// BED12 chromStart / chromEnd (l - longest left anchor, r + longest right anchor).  xs: NULL (strands from `mode`: FLAG_STRANDED /
// FLAG_RF) or a device column of one strand byte per record ('+', '-', '?'), which then gives every junction of the record its strand
struct JuncExtractMem {
    GbBuf a, b;
    cudaEvent_t ev[6] = {};          // bracket the three kernel stretches between the host reads of the sizes
    float ms_kernels = 0, ms_extent = 0;   // CUDA-event ms of the last call: all extraction kernels / the extents walk alone
    void release() {
        a.release(); b.release();
        for (auto& e : ev) if (e) { cudaEventDestroy(e); e = nullptr; }
    }
};
struct DevRecords;
bool junction_extract_device(JuncExtractMem& m, const DevRecords& rec, const int64_t* h_seg_off, const int32_t* h_seg_chrom, int32_t n_seg,
                             int32_t n_chrom, uint32_t mode, const uint8_t* xs, int32_t min_anchor, int32_t min_intron, int32_t max_intron, void* stream,
                             std::vector<int32_t>& chrom, std::vector<int32_t>& left, std::vector<int32_t>& right, std::vector<int64_t>& score,
                             std::vector<uint8_t>& strand, std::vector<int32_t>& start, std::vector<int32_t>& end, std::string& err);

}  // namespace spl
