// Tag group lookup, shared by the host reader (bam_io.cpp) and the device ingest (bam_gpu.cu: k_bam_fill<XS, true>), so that
// the two cannot disagree on a record's group.  The rule is stated in include/spliser_b200.h (spl_tag_groups): the first aux
// field with the table's tag decides; Z gives the bytes before its NUL, A its one character, c C s S i I the decimal text of the
// integer; any other type, no such field, or a malformed field before it (aux_field_end) gives no value.  The value is hashed
// (FNV-1a, 32 bits) and looked up in an open-addressing table with linear probing that the host builds once per table.
#pragma once
#include <cstddef>
#include <cstdint>

#include "bam_aux.h"

#ifdef __CUDACC__
#define SPL_TG_HD __host__ __device__ __forceinline__
#else
#define SPL_TG_HD inline
#endif

namespace spl {

constexpr int32_t TAG_NO_VALUE = -1;   // no field with the tag, a type without a value, or a malformed field before it
constexpr int32_t TAG_NO_GROUP = -2;   // a value that is in none of the table's groups
constexpr uint32_t TAG_MAX_VALUE = 255;

// The table as both routes read it: slot[h & mask] = 1 + value index, 0 = empty.  Values are blob[off[v] .. off[v + 1]).
struct TagTableView {
    uint8_t t0 = 0, t1 = 0;            // the two tag characters
    uint32_t mask = 0;                 // slots - 1 (a power of two, at least twice the values)
    const uint32_t* slot = nullptr;
    const uint32_t* off = nullptr;     // [n_values + 1]
    const uint8_t* blob = nullptr;
    const int32_t* group = nullptr;    // [n_values]
};

SPL_TG_HD uint32_t tag_hash(const uint8_t* p, uint32_t n) {
    uint32_t h = 2166136261u;
    for (uint32_t k = 0; k < n; ++k) h = (h ^ p[k]) * 16777619u;
    return h;
}

// Group of the value p[0 .. n): the probe ends at the first empty slot
SPL_TG_HD int32_t tag_lookup(const TagTableView& t, const uint8_t* p, uint32_t n) {
    for (uint32_t s = tag_hash(p, n) & t.mask;; s = (s + 1) & t.mask) {
        const uint32_t e = t.slot[s];
        if (e == 0) return TAG_NO_GROUP;
        const uint32_t v = e - 1, o = t.off[v];
        if (t.off[v + 1] - o != n) continue;
        uint32_t k = 0;
        while (k < n && t.blob[o + k] == p[k]) ++k;
        if (k == n) return t.group[v];
    }
}

// Decimal text of x into buf (at most 11 bytes: "-2147483648"); returns its length
SPL_TG_HD uint32_t tag_decimal(int64_t x, uint8_t* buf) {
    uint8_t tmp[12];
    uint32_t n = 0;
    const bool neg = x < 0;
    uint64_t u = neg ? (uint64_t)(-x) : (uint64_t)x;
    do { tmp[n++] = (uint8_t)('0' + u % 10u); u /= 10u; } while (u);
    uint32_t m = 0;
    if (neg) buf[m++] = '-';
    while (n) buf[m++] = tmp[--n];
    return m;
}

// Group of a record from its aux block [p, end): a group index, TAG_NO_VALUE or TAG_NO_GROUP
SPL_TG_HD int32_t tag_group_of(const TagTableView& t, const uint8_t* p, const uint8_t* end) {
    while (end - p >= 3) {
        const uint8_t* nx = aux_field_end(p, end);
        if (!nx) return TAG_NO_VALUE;
        if (p[0] == t.t0 && p[1] == t.t1) {
            const uint8_t* v = p + 3;
            int64_t x;
            switch (p[2]) {
                case 'Z': return tag_lookup(t, v, (uint32_t)(nx - v - 1));   // the bytes before the NUL
                case 'A': return tag_lookup(t, v, 1);
                case 'c': x = (int8_t)v[0]; break;
                case 'C': x = v[0]; break;
                case 's': x = (int16_t)(uint16_t)(v[0] | (v[1] << 8)); break;
                case 'S': x = (uint16_t)(v[0] | (v[1] << 8)); break;
                case 'i': x = (int32_t)((uint32_t)v[0] | ((uint32_t)v[1] << 8) | ((uint32_t)v[2] << 16) | ((uint32_t)v[3] << 24)); break;
                case 'I': x = (int64_t)((uint32_t)v[0] | ((uint32_t)v[1] << 8) | ((uint32_t)v[2] << 16) | ((uint32_t)v[3] << 24)); break;
                default: return TAG_NO_VALUE;                                // f, H, B
            }
            uint8_t buf[12];
            return tag_lookup(t, buf, tag_decimal(x, buf));
        }
        p = nx;
    }
    return TAG_NO_VALUE;
}

}  // namespace spl
