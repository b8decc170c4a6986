// BAM ingest on the device (bam_gpu.cu) + the host-side scan that prepares it (bam_io.cpp).
#pragma once
#include <cuda_runtime.h>

#include <cstdint>
#include <string>
#include <vector>

#include "graph_build.h"   // GbBuf

namespace spl {

struct BgzfMember {          // one BGZF member with payload
    uint64_t coff;           // offset of the raw DEFLATE stream in the file
    uint32_t clen, isize;    // compressed / inflated size
    uint64_t uoff;           // offset of its output in the inflated stream
};

struct DevRecordArrays {     // what DevRecords points at, plus the chromosome of every record
    int32_t* pos = nullptr;
    uint16_t* flag = nullptr;
    uint32_t* cig_off = nullptr;
    uint32_t* cigar = nullptr;
    int32_t* chrom = nullptr;
    uint8_t* xs = nullptr;   // strand of every record from its XS tag ('+', '-', '?'; bam_aux.h), only when the ingest was asked for it
};

struct BamGpuMem { GbBuf comp, unc, tab, rec, list; };

struct BamGpuCounts {
    uint64_t n_rec = 0, n_cigar = 0;
    std::vector<int32_t> seg_chrom;
    std::vector<int64_t> seg_off;
    double h2d_bytes = 0;
};

constexpr uint32_t BAMGPU_MAX_SEG = 1u << 16;
enum : int { BAMGPU_OK = 0, BAMGPU_FALLBACK = 1, BAMGPU_ERROR = 2 };

// Host: BGZF member table of a whole file image + BAM header (names -> caller chromosome indices).
// first_record = offset of the first alignment record in the inflated stream; ref_names (may be NULL) receives the header's
// reference names in header order.  Returns "" or an error.
std::string bam_scan(const uint8_t* file, size_t fsz, int32_t n_chrom, const char* const* chrom_names, std::vector<BgzfMember>& members,
                     uint64_t& total_u, uint64_t& first_record, int32_t& n_ref, std::vector<int32_t>& refmap,
                     std::vector<std::string>* ref_names = nullptr);

// Device: inflate + parse.  BAMGPU_FALLBACK (err says why) = use the host reader instead; nothing was counted yet.
int bam_gpu_ingest(BamGpuMem& mem, const uint8_t* file_pinned, size_t fsz, const std::vector<BgzfMember>& members, uint64_t total_u,
                   uint64_t first_record, int32_t n_ref, const std::vector<int32_t>& refmap, void* stream,
                   bool comp_uploaded /* mem.comp already holds the file image (copy queued on `stream`) */,
                   bool want_xs /* fill out.xs */, DevRecordArrays& out, BamGpuCounts& cnt, std::string& err);

}  // namespace spl
