// Minimal BGZF / BAM reader and writer over zlib (htslib is not available in this image).
// The reader produces exactly the fields the reference's checkBam consumes from `samtools view`
// (FLAG, POS, CIGAR; SpliSER_v0_1_8.py:429-437) as flat arrays grouped into chromosome segments.
#pragma once
#include <cstdint>
#include <string>
#include <vector>

#include "../../include/spliser_b200.h"

namespace spl {

struct BamRecords {
    std::vector<int32_t> pos;        // 1-based
    std::vector<uint16_t> flag;
    std::vector<uint32_t> cig_off;   // n+1
    std::vector<uint32_t> cigar;
    std::vector<uint8_t> xs;         // read_bam(want_xs): strand of every record from its XS tag ('+', '-', '?'; bam_aux.h)
    std::vector<int32_t> seg_chrom;
    std::vector<int64_t> seg_off;    // n_seg+1
    int64_t n_total = 0;             // records in the file
    int64_t n_skipped = 0;           // unmapped / unknown reference / no CIGAR
    spl_records_view view() const;
};

// Returns "" or an error message.  chrom_names maps BAM reference names to caller indices.
std::string read_bam(const char* path, int32_t n_chrom, const char* const* chrom_names, int n_threads, BamRecords& out,
                     bool want_xs = false);

std::string write_bam(const char* path, int32_t n_ref, const char* const* ref_names, const int32_t* ref_len,
                      const spl_records_view* rec, int n_threads, bool with_seq = false,
                      const int64_t* aux_off = nullptr /* [n_rec + 1], or NULL */, const uint8_t* aux = nullptr /* raw aux bytes */);

}  // namespace spl
