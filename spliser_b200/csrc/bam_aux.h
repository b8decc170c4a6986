// Walk of a BAM record's aux fields (SAM spec 4.2.4), shared by the host reader (bam_io.cpp: CG and XS tags) and the device
// ingest (bam_gpu.cu: XS tag), so that the two cannot disagree on where a field ends.  The XS rule is stated in
// include/spliser_b200.h (SPL_FLAG_XS_STRAND).  Byte loads only: a field is never read past `end`.
#pragma once
#include <cstddef>
#include <cstdint>

#ifdef __CUDACC__
#define SPL_AUX_HD __host__ __device__ __forceinline__
#else
#define SPL_AUX_HD inline
#endif

namespace spl {

// End of the aux field starting at f (two tag bytes, a type byte, the value), or nullptr when the field is malformed: fewer
// than three bytes left, an unknown type byte, or a value that runs past `end` (a Z / H without its NUL does).
// B arrays: subtype byte, u32 count, count x 1 (c C) / 2 (s S) / 4 (any other subtype) bytes.
SPL_AUX_HD const uint8_t* aux_field_end(const uint8_t* f, const uint8_t* end) {
    if (end - f < 3) return nullptr;
    const uint8_t* p = f + 3;
    const size_t left = (size_t)(end - p);
    size_t sz;
    switch (f[2]) {
        case 'A': case 'c': case 'C': sz = 1; break;
        case 's': case 'S': sz = 2; break;
        case 'i': case 'I': case 'f': sz = 4; break;
        case 'Z': case 'H': {
            size_t k = 0;
            while (k < left && p[k]) ++k;
            if (k == left) return nullptr;
            sz = k + 1;
            break;
        }
        case 'B': {
            if (left < 5) return nullptr;
            const uint8_t sub = p[0];
            const uint64_t cnt = (uint64_t)p[1] | ((uint64_t)p[2] << 8) | ((uint64_t)p[3] << 16) | ((uint64_t)p[4] << 24);
            const uint64_t es = (sub == 'c' || sub == 'C') ? 1 : (sub == 's' || sub == 'S') ? 2 : 4;
            if (cnt * es > (uint64_t)(left - 5)) return nullptr;
            sz = 5 + (size_t)(cnt * es);
            break;
        }
        default: return nullptr;
    }
    return sz <= left ? p + sz : nullptr;
}

// Strand of a record from its aux block [p, end): the first field tagged XS decides -- XS:A:+ gives '+', XS:A:- gives '-',
// any other type or character '?'.  No XS field, or a malformed field before it (aux_field_end), gives '?'.
SPL_AUX_HD uint8_t aux_xs_strand(const uint8_t* p, const uint8_t* end) {
    while (end - p >= 3) {
        const uint8_t* nx = aux_field_end(p, end);
        if (!nx) return '?';
        if (p[0] == 'X' && p[1] == 'S') return (p[2] == 'A' && (p[3] == '+' || p[3] == '-')) ? p[3] : (uint8_t)'?';
        p = nx;
    }
    return '?';
}

}  // namespace spl
