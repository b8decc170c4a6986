// The read filter of both BAM readers (host reader bam_io.cpp, device ingest bam_gpu.cu), so that the two cannot disagree.
// The rule is stated in include/spliser_b200.h (spl_read_filter); it applies to records the keep rule already keeps.
#pragma once
#include <cstdint>

#ifdef __CUDACC__
#define SPL_RF_HD __host__ __device__ __forceinline__
#else
#define SPL_RF_HD inline
#endif

namespace spl {

// {0, 0, 0} keeps every record: the value of "no filter"
struct ReadFilter { uint32_t min_mapq = 0, exclude = 0, require = 0; };

SPL_RF_HD bool read_filter_keeps(const ReadFilter& f, uint32_t mapq, uint32_t flag) {
    return mapq >= f.min_mapq && (flag & f.exclude) == 0u && (flag & f.require) == f.require;
}

SPL_RF_HD bool read_filter_none(const ReadFilter& f) { return f.min_mapq == 0 && f.exclude == 0 && f.require == 0; }

}  // namespace spl
