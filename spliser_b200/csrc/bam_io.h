// Minimal BGZF / BAM reader and writer over zlib (htslib is not available in this image).
// The reader produces exactly the fields the reference's checkBam consumes from `samtools view`
// (FLAG, POS, CIGAR; SpliSER_v0_1_8.py:429-437) as flat arrays grouped into chromosome segments.
#pragma once
#include <cstdint>
#include <string>
#include <vector>

#include "../../include/spliser_b200.h"
#include "read_filter.h"
#include "tag_groups.h"

namespace spl {

struct BamRecords {
    std::vector<int32_t> pos;        // 1-based
    std::vector<uint16_t> flag;
    std::vector<uint32_t> cig_off;   // n+1
    std::vector<uint32_t> cigar;
    std::vector<uint8_t> xs;         // read_bam(want_xs): strand of every record from its XS tag ('+', '-', '?'; bam_aux.h)
    std::vector<int32_t> grp;        // read_bam(tags): tag group of every record (tag_groups.h)
    std::vector<int32_t> seg_chrom;
    std::vector<int64_t> seg_off;    // n_seg+1
    int64_t n_total = 0;             // records in the file
    int64_t n_skipped = 0;           // unmapped / unknown reference / no CIGAR
    int64_t n_filtered = 0;          // kept by the rule above, dropped by the read filter
    spl_records_view view() const;
};

// The caller's chromosome index of every header reference: the index of the same name in chrom_names (the first one when a
// name repeats there), else -1.  Every reader and the device-resident samples map references with this one rule.
std::vector<int32_t> map_references(const std::vector<std::string>& ref_names, int32_t n_chrom, const char* const* chrom_names);

// The ABI's filter checked (MAPQ 0..255, flags <= 0xFFFF) and converted; false with the reason in err.
bool read_filter_from(const spl_read_filter& f, ReadFilter& out, std::string& err);

// A tag group table (spl_tag_groups) checked and laid out for tag_group_of: the open-addressing table and the values on the host.
struct TagTableHost {
    uint8_t t0 = 0, t1 = 0;
    int32_t n_groups = 0;
    uint32_t mask = 0;
    std::vector<uint32_t> slot, off;
    std::vector<uint8_t> blob;
    std::vector<int32_t> group;
    TagTableView view() const;       // over the host vectors
};
// O(n_values); "" or the reason the table breaks the rule (include/spliser_b200.h)
std::string build_tag_table(const spl_tag_groups* g, TagTableHost& out);

// Returns "" or an error message.  chrom_names maps BAM reference names to caller indices.  header_order != NULL: chrom_names
// is ignored, every record keeps its header reference index (seg_chrom) and *header_order receives the reference names.
// rf: the read filter, applied after the keep rule (and after a CG-tag CIGAR replaced the placeholder).
std::string read_bam(const char* path, int32_t n_chrom, const char* const* chrom_names, int n_threads, BamRecords& out,
                     bool want_xs = false, std::vector<std::string>* header_order = nullptr, const ReadFilter& rf = ReadFilter{},
                     const TagTableView* tags = nullptr /* fill out.grp */);

// A spl_records handle that owns r (has_xs: r.xs holds one strand byte per record)
spl_records* records_handle(BamRecords&& r, bool has_xs);

std::string write_bam(const char* path, int32_t n_ref, const char* const* ref_names, const int32_t* ref_len,
                      const spl_records_view* rec, int n_threads, bool with_seq = false,
                      const int64_t* aux_off = nullptr /* [n_rec + 1], or NULL */, const uint8_t* aux = nullptr /* raw aux bytes */,
                      const uint8_t* mapq = nullptr /* [n_rec], or NULL = 255 */);

}  // namespace spl
