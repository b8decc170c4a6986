// Split of one ingest's records into the samples of a tag group table (group_split.cu; the rule is stated in
// include/spliser_b200.h, spl_tag_groups): a stable partition by group, the records of no group dropped.
#pragma once
#include <cuda_runtime.h>

#include <cstdint>
#include <string>
#include <vector>

#include "bam_gpu.h"
#include "graph_build.h"   // GbBuf

namespace spl {

// the host reader's upload, the sort scratch, the segment boundaries, the per-group table: all released after each split
struct GroupSplitMem {
    GbBuf in, sort, seg, tab;
    void release() { in.release(); sort.release(); seg.release(); tab.release(); }
};

// The sorted order and what each group needs, from group_sort
struct GroupSort {
    uint64_t n_kept = 0;                     // records with a group
    uint64_t no_value = 0, no_group = 0;
    std::vector<int64_t> n_rec, n_cig;       // per group
    std::vector<std::vector<int32_t>> seg_chrom;   // per group: the chromosome (the ingest's chrom column) of every segment
    std::vector<std::vector<int64_t>> seg_off;     // per group: [n_seg + 1], from 0
    // device, inside GroupSplitMem::sort: the sorted group of every kept record, its index in the ingest, its CIGAR offset
    // among the sorted records
    const uint16_t* keys = nullptr;
    const uint32_t* idx = nullptr;
    const uint32_t* coff = nullptr;
    std::vector<uint32_t> g_start, g_cig;    // first sorted record / CIGAR operator of every group
};

// Where group g's columns go: byte offsets from the base of the split's allocation
struct GroupCols { uint64_t pos, flag, off, cig, xs; uint32_t start, cig0, n, nc; };

// Sorts the n records of `in` (grp[n], in.chrom and in.cig_off with its n-th entry set) by group: an LSD radix sort over the
// 16-bit group id with the record index as payload, one 8-bit pass when n_groups <= 256, two otherwise.  Memory is O(n).
int group_sort(GroupSplitMem& m, const DevRecordArrays& in, const int32_t* grp, uint64_t n, int32_t n_groups, cudaStream_t st, GroupSort& out,
               std::string& err);

// Writes every kept record's POS, FLAG, CIGAR offset (from 0 within its group), CIGAR operators and, when in.xs is set, XS
// strand into base + cols[g] of its group g; cig_off[n] = the group's operator count for every group.
int group_gather(GroupSplitMem& m, const DevRecordArrays& in, const GroupSort& gs, const std::vector<GroupCols>& cols, char* base,
                 cudaStream_t st, std::string& err);

}  // namespace spl
