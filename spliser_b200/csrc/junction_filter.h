// The two row filters findAlphaCounts applies to a junction table (S:269, S:279-288), shared by the BED12 parser
// (spl_bed_parse, host_text.cpp) and spl_process_bam_extract (pipeline.cu), which applies them to the table it extracted
// from the alignments.  Host only.
#pragma once
#include <string_view>

namespace spl {

struct JunctionFilter {
    const char* qchrom;                            // -c: only rows of this chromosome (NULL = "All")
    bool window;                                   // -g: only rows with a site inside the gene, widened by -m
    long long gene_left, gene_right, max_intron;

    bool chrom_kept(std::string_view chrom) const { return !qchrom || chrom == std::string_view(qchrom); }   // S:269
    bool window_kept(long long left, long long right) const {                                                // S:279-288
        if (!window) return true;
        const bool lin = (left + max_intron >= gene_left) && (left <= gene_right);
        const bool rin = (right - max_intron <= gene_right) && (right >= gene_left);
        return lin || rin;
    }
};

}  // namespace spl
