// BAM ingest on the device (SURVEY.md 8(f) row 1): BGZF members are inflated by the GPU and the BAM records are parsed
// straight into the record arrays the expansion kernels read -- the decoded records never exist on the host.
//
//   k_bgzf_inflate     one warp per BGZF member (<= 64 KiB each, independent DEFLATE streams): the warp runs the decoder of
//                      inflate.h (Huffman tables in shared memory, symbol decode uniform across the lanes, LZ77 match bytes
//                      split between the lanes); tens of thousands of members decode concurrently
//   k_bam_first        per member: the first offset at which a plausible chain of BAM records starts (records are NOT
//                      aligned to members in general: htsjdk and this library's own writer cut members every 0xff00 bytes)
//   k_bam_walk<false>  per member: walks the record chain from that offset to the member's end, counting records and
//                      CIGAR operators and reporting where the walk lands
//   (host)             the landing offsets are chained from the header's end: member s is accepted iff the walk of the
//                      previous accepted member lands exactly on its candidate.  If every link holds, the chain is the
//                      true record chain by induction -- the speculation in k_bam_first is verified, never trusted.
//                      Any broken link (or a feature this path does not parse: CG-tag long CIGARs) -> the caller falls
//                      back to the host reader (bam_io.cpp).
//   k_bam_fill         one warp per accepted member: the kept records (offsets listed by the counting walk) are written out
//                      round-robin by the lanes: POS, FLAG, chromosome and CIGAR (k_bam_fill<true>: and the XS strand, from
//                      a walk of the record's aux fields by the same lane)
//   k_bam_segments     chromosome boundaries of the record arrays (a coordinate-sorted BAM has one segment per reference)
// Kept records follow the host reader: mapped to a caller chromosome and with at least one CIGAR operator (bam_io.cpp).
#include <cuda_runtime.h>

#include <algorithm>
#include <cstdint>
#include <cstring>
#include <string>
#include <vector>

#include "bam_aux.h"
#include "bam_gpu.h"
#include "device_types.h"
#include "inflate.h"

namespace spl {

namespace {

constexpr int INF_WARPS = 8;

__global__ void __launch_bounds__(INF_WARPS * 32)
k_bgzf_inflate(const uint8_t* __restrict__ comp, const BgzfMember* __restrict__ mem, uint32_t n_mem, uint8_t* __restrict__ out, uint32_t* __restrict__ err) {
    __shared__ InflateTables tabs[INF_WARPS];
    const uint32_t m = blockIdx.x * INF_WARPS + (threadIdx.x >> 5);
    if (m >= n_mem) return;                                              // whole warps leave together
    const BgzfMember b = mem[m];
    uint32_t produced = 0;
    const int rc = inflate_member(comp + b.coff, b.clen, out + b.uoff, b.isize, &produced, tabs[threadIdx.x >> 5], WarpLanes());
    if ((threadIdx.x & 31) == 0 && (rc != INF_OK || produced != b.isize)) atomicMax(err, 1u + m);
}

// unaligned little-endian 32-bit load from two aligned words (the inflated stream is 256-byte aligned and padded)
__device__ __forceinline__ uint32_t ld32u(const uint8_t* __restrict__ u, uint64_t o) {
    const uint32_t* w = reinterpret_cast<const uint32_t*>(u + (o & ~3ull));
    return __funnelshift_r(w[0], w[1], (uint32_t)(o & 3ull) * 8u);
}

// fixed part of a BAM record at offset o, read as 9 aligned words
struct RecHdr { uint32_t bs, l_name, n_cig, flag; int32_t refid, pos, l_seq, next_ref, next_pos; };
__device__ __forceinline__ RecHdr read_hdr(const uint8_t* __restrict__ u, uint64_t o) {
    const uint32_t* w = reinterpret_cast<const uint32_t*>(u + (o & ~3ull));
    const uint32_t sh = (uint32_t)(o & 3ull) * 8u;
    uint32_t a[9];
#pragma unroll
    for (int i = 0; i < 9; ++i) a[i] = w[i];
    RecHdr h;
    h.bs = __funnelshift_r(a[0], a[1], sh);
    h.refid = (int32_t)__funnelshift_r(a[1], a[2], sh);
    h.pos = (int32_t)__funnelshift_r(a[2], a[3], sh);
    h.l_name = __funnelshift_r(a[3], a[4], sh) & 0xffu;
    const uint32_t cf = __funnelshift_r(a[4], a[5], sh);
    h.n_cig = cf & 0xffffu; h.flag = cf >> 16;
    h.l_seq = (int32_t)__funnelshift_r(a[5], a[6], sh);
    h.next_ref = (int32_t)__funnelshift_r(a[6], a[7], sh);
    h.next_pos = (int32_t)__funnelshift_r(a[7], a[8], sh);
    return h;
}

// Could a BAM record start at offset o?  Necessary conditions only: a true record always passes.
__device__ __forceinline__ bool plausible(const uint8_t* __restrict__ u, uint64_t o, uint64_t total, int32_t n_ref, uint64_t* next, RecHdr* out = nullptr) {
    if (o + 36 > total) return false;
    const RecHdr h = read_hdr(u, o);
    if (h.bs < 32u || h.bs > (1u << 30)) return false;
    if (h.refid < -1 || h.refid >= n_ref || h.next_ref < -1 || h.next_ref >= n_ref) return false;
    if (h.pos < -1 || h.next_pos < -1 || h.l_name < 1u || h.l_seq < 0) return false;
    const uint64_t need = 32ull + h.l_name + 4ull * h.n_cig + ((uint64_t)h.l_seq + 1) / 2 + (uint64_t)h.l_seq;
    if (need > h.bs || o + 4 + h.bs > total) return false;
    if (u[o + 36 + h.l_name - 1] != 0) return false;                   // read name is NUL-terminated
    *next = o + 4 + h.bs;
    if (out) *out = h;
    return true;
}

// first[m] = smallest offset in member m's byte range from which three plausible records chain (or the stream ends)
__global__ void __launch_bounds__(256) k_bam_first(const uint8_t* __restrict__ u, const BgzfMember* __restrict__ mem, uint32_t n_mem,
                                                   uint64_t total, int32_t n_ref, uint64_t first0, uint64_t* __restrict__ first) {
    const uint32_t m = blockIdx.x * 8 + (threadIdx.x >> 5);
    const int lane = threadIdx.x & 31;
    if (m >= n_mem) return;
    const uint64_t lo = mem[m].uoff, hi = lo + mem[m].isize;
    if (first0 >= hi) { if (lane == 0) first[m] = ~0ull; return; }      // header-only member
    if (first0 >= lo) { if (lane == 0) first[m] = first0; return; }     // the member holding the header's end: known exactly
    uint64_t found = ~0ull;
    for (uint64_t base = lo; base < hi && found == ~0ull; base += 32) {
        const uint64_t o = base + lane;
        bool ok = false;
        if (o < hi) {
            uint64_t a, b, c;
            ok = plausible(u, o, total, n_ref, &a) && (a == total || (plausible(u, a, total, n_ref, &b) && (b == total || plausible(u, b, total, n_ref, &c))));
        }
        const uint32_t bal = __ballot_sync(0xffffffffu, ok);
        if (bal) found = base + (uint64_t)(__ffs(bal) - 1);
    }
    if (lane == 0) first[m] = found;
}

struct WalkOut { uint64_t land; uint32_t n_rec, n_cig, flags, pad; };
constexpr uint32_t WALK_BAD = 1u, WALK_LONG_CIGAR = 2u;

// slot of member m's first kept-record offset in the scratch list: a record is at least 36 bytes, so the records that
// START inside a member of isize bytes number at most isize / 32 + 1
__device__ __forceinline__ uint64_t list_base(const BgzfMember& b, uint32_t m) { return (b.uoff >> 5) + m; }

template <bool FILL>
__global__ void __launch_bounds__(128) k_bam_walk(const uint8_t* __restrict__ u, const BgzfMember* __restrict__ mem, uint32_t n_mem, uint64_t total,
                                                  int32_t n_ref, const int32_t* __restrict__ refmap, const uint64_t* __restrict__ first,
                                                  WalkOut* __restrict__ wo, const uint64_t* __restrict__ rec_base, const uint64_t* __restrict__ cig_base,
                                                  DevRecordArrays out, uint32_t* __restrict__ kept) {
    const uint32_t m = blockIdx.x * blockDim.x + threadIdx.x;
    if (m >= n_mem) return;
    uint64_t o = first[m];
    if (FILL) { if (rec_base[m] == ~0ull) return; }                      // member not on the verified chain
    if (o == ~0ull) { if (!FILL) wo[m] = WalkOut{~0ull, 0, 0, 0, 0}; return; }
    const uint64_t limit = mem[m].uoff + mem[m].isize;
    uint32_t n_rec = 0, n_cig_tot = 0, flags = 0;
    uint64_t ri = FILL ? rec_base[m] : 0, ci = FILL ? cig_base[m] : 0;
    while (o < limit) {
        uint64_t nx;
        RecHdr h;
        if (!plausible(u, o, total, n_ref, &nx, &h)) { flags |= WALK_BAD; break; }
        const uint64_t cig = o + 36 + h.l_name;
        // CIGARs of more than 65535 operators live in a CG tag (SAM spec 4.2.2): left to the host reader
        if (h.n_cig == 2 && ld32u(u, cig) == (((uint32_t)h.l_seq << 4) | 4u) && (ld32u(u, cig + 4) & 15u) == 3u) flags |= WALK_LONG_CIGAR;
        const int32_t chrom = h.refid >= 0 ? refmap[h.refid] : -1;
        if (chrom >= 0 && h.n_cig > 0) {
            if (!FILL && kept) kept[list_base(mem[m], m) + n_rec] = (uint32_t)(o - mem[m].uoff);   // may exceed isize-1 never: o < limit
            if (FILL) {
                out.pos[ri] = h.pos + 1;
                out.flag[ri] = (uint16_t)h.flag;
                out.chrom[ri] = chrom;
                out.cig_off[ri] = (uint32_t)ci;
                for (uint32_t k = 0; k < h.n_cig; ++k) out.cigar[ci + k] = ld32u(u, cig + 4ull * k);
            }
            ++n_rec; n_cig_tot += h.n_cig; ++ri; ci += h.n_cig;
        }
        o = nx;
    }
    if (!FILL) wo[m] = WalkOut{o, n_rec, n_cig_tot, flags, 0};
}

// second pass, one WARP per accepted member: the lanes take the kept records of the member round-robin from the offset list
// the counting walk left, so neighbouring lanes write neighbouring records (the per-thread walk wrote with a stride of
// ~1,000 records between lanes)
template <bool XS>
__global__ void __launch_bounds__(256) k_bam_fill(const uint8_t* __restrict__ u, const BgzfMember* __restrict__ mem, uint32_t n_mem,
                                                  const int32_t* __restrict__ refmap, const WalkOut* __restrict__ wo,
                                                  const uint64_t* __restrict__ rec_base, const uint64_t* __restrict__ cig_base,
                                                  const uint32_t* __restrict__ kept, DevRecordArrays out) {
    const uint32_t m = blockIdx.x * 8 + (threadIdx.x >> 5);
    const int lane = threadIdx.x & 31;
    if (m >= n_mem || rec_base[m] == ~0ull) return;
    const BgzfMember b = mem[m];
    const uint32_t n = wo[m].n_rec;
    const uint64_t lb = list_base(b, m), r0 = rec_base[m];
    uint64_t ci = cig_base[m];
    for (uint32_t k0 = 0; k0 < n; k0 += 32) {                           // warp-uniform
        const uint32_t k = k0 + lane;
        const bool live = k < n;
        uint64_t o = 0;
        RecHdr h{};
        if (live) { o = b.uoff + kept[lb + k]; h = read_hdr(u, o); }
        const uint32_t nc = live ? h.n_cig : 0u;
        uint32_t pre = nc;                                             // inclusive scan of the CIGAR lengths
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) { const uint32_t x = __shfl_up_sync(0xffffffffu, pre, d); if (lane >= d) pre += x; }
        const uint32_t tot = __shfl_sync(0xffffffffu, pre, 31);
        if (live) {
            const uint64_t c0 = ci + pre - nc, ri = r0 + k;
            out.pos[ri] = h.pos + 1;
            out.flag[ri] = (uint16_t)h.flag;
            out.chrom[ri] = refmap[h.refid];
            out.cig_off[ri] = (uint32_t)c0;
            const uint64_t cig = o + 36 + h.l_name;
            for (uint32_t q = 0; q < nc; ++q) out.cigar[c0 + q] = ld32u(u, cig + 4ull * q);
            if (XS) {                                                  // aux fields: from the end of QUAL to the end of the record
                const uint64_t aux = cig + 4ull * nc + ((uint64_t)h.l_seq + 1) / 2 + (uint64_t)h.l_seq;
                out.xs[ri] = aux_xs_strand(u + aux, u + o + 4 + h.bs);  // aux <= the record end: the counting walk checked it
            }
        }
        ci += tot;
    }
}

// boundaries of the chromosome segments: seg[k] = (first record, chromosome)
__global__ void k_bam_segments(const int32_t* __restrict__ chrom, uint64_t n, uint32_t* __restrict__ n_seg, uint64_t* __restrict__ seg_first,
                               int32_t* __restrict__ seg_chrom, uint32_t cap) {
    const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    if (i == 0 || chrom[i] != chrom[i - 1]) {
        const uint32_t k = atomicAdd(n_seg, 1u);
        if (k < cap) { seg_first[k] = i; seg_chrom[k] = chrom[i]; }
    }
}

__global__ void k_set_u32(uint32_t* p, uint32_t v) { *p = v; }

}  // namespace

#define BG_CU(call)                                                                     \
    do {                                                                                \
        cudaError_t _e = (call);                                                        \
        if (_e != cudaSuccess) { err = std::string(#call) + ": " + cudaGetErrorString(_e); return BAMGPU_ERROR; } \
    } while (0)

int bam_gpu_ingest(BamGpuMem& mem, const uint8_t* file_pinned, size_t fsz, const std::vector<BgzfMember>& members, uint64_t total_u,
                   uint64_t first_record, int32_t n_ref, const std::vector<int32_t>& refmap, void* stream, bool comp_uploaded,
                   bool want_xs, DevRecordArrays& out, BamGpuCounts& cnt, std::string& err) {
    cudaStream_t st = (cudaStream_t)stream;
    const uint32_t n_mem = (uint32_t)members.size();
    cnt = BamGpuCounts{};
    if (n_mem == 0 || first_record >= total_u) { out = DevRecordArrays{}; return BAMGPU_OK; }
    // ---- compressed file + member table to the device, inflate
    // not enough device memory for the file image + the inflated stream: the host reader streams the file instead
    if (mem.comp.reserve(fsz + 64) != cudaSuccess ||
        mem.unc.reserve(total_u + 256) != cudaSuccess ||                // the aligned-word reads of the parser run a few bytes past the end
        mem.tab.reserve((size_t)n_mem * (sizeof(BgzfMember) + 8 + sizeof(WalkOut) + 16) + ((size_t)n_ref + 1) * 4 + 4096) != cudaSuccess ||
        mem.list.reserve(((size_t)(total_u >> 5) + n_mem + 8) * 4) != cudaSuccess) {
        cudaGetLastError();
        mem.comp.release(); mem.unc.release();
        err = "not enough device memory for the inflated BAM";
        return BAMGPU_FALLBACK;
    }
    char* tb = (char*)mem.tab.p;
    BgzfMember* d_mem = (BgzfMember*)tb; tb += (size_t)n_mem * sizeof(BgzfMember);
    uint64_t* d_first = (uint64_t*)tb; tb += (size_t)n_mem * 8;
    WalkOut* d_wo = (WalkOut*)tb; tb += (size_t)n_mem * sizeof(WalkOut);
    uint64_t* d_rbase = (uint64_t*)tb; tb += (size_t)n_mem * 8;
    uint64_t* d_cbase = (uint64_t*)tb; tb += (size_t)n_mem * 8;
    int32_t* d_refmap = (int32_t*)tb; tb += ((size_t)n_ref + 1) * 4;
    uint32_t* d_err = (uint32_t*)(((uintptr_t)tb + 15) & ~(uintptr_t)15);
    if (!comp_uploaded) BG_CU(cudaMemcpyAsync(mem.comp.p, file_pinned, fsz, cudaMemcpyHostToDevice, st));
    BG_CU(cudaMemcpyAsync(d_mem, members.data(), (size_t)n_mem * sizeof(BgzfMember), cudaMemcpyHostToDevice, st));
    if (n_ref > 0) BG_CU(cudaMemcpyAsync(d_refmap, refmap.data(), (size_t)n_ref * 4, cudaMemcpyHostToDevice, st));
    BG_CU(cudaMemsetAsync(d_err, 0, 16, st));
    cnt.h2d_bytes = (double)fsz + (double)n_mem * sizeof(BgzfMember);
    const uint8_t* d_u = (const uint8_t*)mem.unc.p;
    uint32_t* d_kept = (uint32_t*)mem.list.p;
    BG_CU(cudaMemsetAsync((uint8_t*)mem.unc.p + total_u, 0, 256, st));     // the parser's aligned-word reads run a few bytes past the end
    { SPL_LAUNCH; k_bgzf_inflate<<<(n_mem + INF_WARPS - 1) / INF_WARPS, INF_WARPS * 32, 0, st>>>((const uint8_t*)mem.comp.p, d_mem, n_mem, (uint8_t*)mem.unc.p, d_err); }
    // ---- speculative record starts + counting walk
    { SPL_LAUNCH; k_bam_first<<<(n_mem + 7) / 8, 256, 0, st>>>(d_u, d_mem, n_mem, total_u, n_ref, first_record, d_first); }
    { SPL_LAUNCH; k_bam_walk<false><<<(n_mem + 127) / 128, 128, 0, st>>>(d_u, d_mem, n_mem, total_u, n_ref, d_refmap, d_first, d_wo, nullptr, nullptr, DevRecordArrays{}, d_kept); }
    BG_CU(cudaGetLastError());
    std::vector<uint64_t> h_first(n_mem);
    std::vector<WalkOut> h_wo(n_mem);
    uint32_t h_err[4] = {0, 0, 0, 0};
    BG_CU(cudaMemcpyAsync(h_first.data(), d_first, (size_t)n_mem * 8, cudaMemcpyDeviceToHost, st));
    BG_CU(cudaMemcpyAsync(h_wo.data(), d_wo, (size_t)n_mem * sizeof(WalkOut), cudaMemcpyDeviceToHost, st));
    BG_CU(cudaMemcpyAsync(h_err, d_err, 16, cudaMemcpyDeviceToHost, st));
    BG_CU(cudaStreamSynchronize(st));
    if (h_err[0]) { err = "BGZF inflate failed on the device (member " + std::to_string(h_err[0] - 1) + ")"; return BAMGPU_FALLBACK; }
    // ---- verify the chain: each accepted member's walk must land exactly on the next accepted member's candidate
    std::vector<uint64_t> rbase(n_mem, ~0ull), cbase(n_mem, ~0ull);
    uint64_t expect = first_record, nrec = 0, ncig = 0;
    uint32_t m = 0;
    while (expect < total_u) {
        while (m < n_mem && members[m].uoff + members[m].isize <= expect) ++m;      // member that holds `expect`
        if (m >= n_mem) { err = "record chain leaves the file"; return BAMGPU_FALLBACK; }
        if (h_first[m] != expect) { err = "record boundary speculation failed"; return BAMGPU_FALLBACK; }
        if (h_wo[m].flags & WALK_BAD) { err = "implausible BAM record"; return BAMGPU_FALLBACK; }
        if (h_wo[m].flags & WALK_LONG_CIGAR) { err = "CG-tag CIGAR"; return BAMGPU_FALLBACK; }
        rbase[m] = nrec; cbase[m] = ncig;
        nrec += h_wo[m].n_rec; ncig += h_wo[m].n_cig;
        expect = h_wo[m].land;
        ++m;
    }
    if (expect != total_u) { err = "truncated BAM (partial record at end of file)"; return BAMGPU_FALLBACK; }
    if (nrec >= (uint64_t)UINT32_MAX - 16 || ncig >= (uint64_t)UINT32_MAX - 16) { err = "more than 2^32 records or CIGAR operators"; return BAMGPU_FALLBACK; }
    cnt.n_rec = nrec; cnt.n_cigar = ncig;
    // ---- record arrays
    {
        size_t off = 0;
        auto take = [&](size_t bytes) { off = (off + 255) & ~(size_t)255; const size_t o = off; off += bytes; return o; };
        const size_t o_pos = take((nrec + 4) * 4), o_flag = take((nrec + 4) * 2), o_off = take((nrec + 4) * 4), o_cig = take((ncig + 4) * 4),
                     o_chr = take((nrec + 4) * 4), o_sf = take(BAMGPU_MAX_SEG * 8), o_sc = take(BAMGPU_MAX_SEG * 4), o_ns = take(16),
                     o_xs = want_xs ? take(nrec + 4) : 0;
        if (mem.rec.reserve(off + 256) != cudaSuccess) { cudaGetLastError(); err = "not enough device memory for the record arrays"; return BAMGPU_FALLBACK; }
        char* rb = (char*)mem.rec.p;
        out.pos = (int32_t*)(rb + o_pos); out.flag = (uint16_t*)(rb + o_flag); out.cig_off = (uint32_t*)(rb + o_off);
        out.cigar = (uint32_t*)(rb + o_cig); out.chrom = (int32_t*)(rb + o_chr);
        out.xs = want_xs ? (uint8_t*)(rb + o_xs) : nullptr;
        uint64_t* d_sf = (uint64_t*)(rb + o_sf); int32_t* d_sc = (int32_t*)(rb + o_sc); uint32_t* d_ns = (uint32_t*)(rb + o_ns);
        BG_CU(cudaMemcpyAsync(d_rbase, rbase.data(), (size_t)n_mem * 8, cudaMemcpyHostToDevice, st));
        BG_CU(cudaMemcpyAsync(d_cbase, cbase.data(), (size_t)n_mem * 8, cudaMemcpyHostToDevice, st));
        BG_CU(cudaMemsetAsync(d_ns, 0, 16, st));
        if (want_xs) { SPL_LAUNCH; k_bam_fill<true><<<(n_mem + 7) / 8, 256, 0, st>>>(d_u, d_mem, n_mem, d_refmap, d_wo, d_rbase, d_cbase, d_kept, out); }
        else { SPL_LAUNCH; k_bam_fill<false><<<(n_mem + 7) / 8, 256, 0, st>>>(d_u, d_mem, n_mem, d_refmap, d_wo, d_rbase, d_cbase, d_kept, out); }
        { SPL_LAUNCH; k_set_u32<<<1, 1, 0, st>>>(out.cig_off + nrec, (uint32_t)ncig); }
        if (nrec) { SPL_LAUNCH; k_bam_segments<<<(unsigned)((nrec + 255) / 256), 256, 0, st>>>(out.chrom, nrec, d_ns, d_sf, d_sc, BAMGPU_MAX_SEG); }
        BG_CU(cudaGetLastError());
        uint32_t h_ns = 0;
        BG_CU(cudaMemcpyAsync(&h_ns, d_ns, 4, cudaMemcpyDeviceToHost, st));
        BG_CU(cudaStreamSynchronize(st));
        if (h_ns > BAMGPU_MAX_SEG) { err = "too many chromosome segments (unsorted BAM?)"; return BAMGPU_FALLBACK; }
        std::vector<uint64_t> sf(h_ns);
        std::vector<int32_t> sc(h_ns);
        if (h_ns) {
            BG_CU(cudaMemcpyAsync(sf.data(), d_sf, (size_t)h_ns * 8, cudaMemcpyDeviceToHost, st));
            BG_CU(cudaMemcpyAsync(sc.data(), d_sc, (size_t)h_ns * 4, cudaMemcpyDeviceToHost, st));
            BG_CU(cudaStreamSynchronize(st));
        }
        std::vector<uint32_t> order(h_ns);
        for (uint32_t k = 0; k < h_ns; ++k) order[k] = k;
        std::sort(order.begin(), order.end(), [&](uint32_t a, uint32_t b) { return sf[a] < sf[b]; });
        cnt.seg_chrom.clear(); cnt.seg_off.clear();
        for (uint32_t k : order) { cnt.seg_chrom.push_back(sc[k]); cnt.seg_off.push_back((int64_t)sf[k]); }
        cnt.seg_off.push_back((int64_t)nrec);
        if (cnt.seg_chrom.empty()) cnt.seg_off.assign(1, 0);
    }
    return BAMGPU_OK;
}

}  // namespace spl

// host build of the same decoder the device runs (unit tests compare it with zlib without a GPU)
extern "C" int spl_debug_inflate(const uint8_t* src, uint32_t n, uint8_t* dst, uint32_t cap, uint32_t* out_len) {
    if (!src || !dst || !out_len) return -1;
    static thread_local spl::InflateTables t;
    return spl::inflate_member(src, n, dst, cap, out_len, t, spl::OneLane());
}
