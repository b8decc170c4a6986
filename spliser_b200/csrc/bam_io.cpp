// BGZF / BAM reader and writer over zlib.  Replaces, for this path, the `samtools view` subprocess
// of SpliSER_v0_1_8.py:422 (one fork per splice site) by one streaming pass over the file.
#include "bam_io.h"
#include "bam_aux.h"
#include "bam_gpu.h"

#include <fcntl.h>
#include <sys/mman.h>
#include <sys/stat.h>
#include <unistd.h>
#include <zlib.h>

#include <algorithm>
#include <atomic>
#include <cstdio>
#include <cstring>
#include <thread>
#include <unordered_map>

namespace spl {

spl_records_view BamRecords::view() const {
    spl_records_view v{};
    v.n_rec = (int64_t)pos.size();
    v.n_cigar = (int64_t)cigar.size();
    v.pos = pos.data(); v.flag = flag.data(); v.cig_off = cig_off.data(); v.cigar = cigar.data();
    v.n_seg = (int32_t)seg_chrom.size();
    v.seg_chrom = seg_chrom.data(); v.seg_off = seg_off.data();
    return v;
}

namespace {

inline uint16_t rd16(const uint8_t* p) { return (uint16_t)(p[0] | (p[1] << 8)); }
inline uint32_t rd32(const uint8_t* p) { return (uint32_t)p[0] | ((uint32_t)p[1] << 8) | ((uint32_t)p[2] << 16) | ((uint32_t)p[3] << 24); }
inline int32_t rdi32(const uint8_t* p) { return (int32_t)rd32(p); }

struct BgzfBlock { size_t coff; uint32_t clen; uint32_t isize; size_t uoff; uint32_t crc = 0; };

int worker_count(int n) {
    if (n > 0) return n;
    unsigned h = std::thread::hardware_concurrency();
    return (int)std::max(1u, std::min(h ? h : 4u, 32u));
}

bool inflate_block(const uint8_t* src, uint32_t clen, uint8_t* dst, uint32_t isize) {
    z_stream zs;
    memset(&zs, 0, sizeof zs);
    if (inflateInit2(&zs, -15) != Z_OK) return false;
    zs.next_in = const_cast<Bytef*>(src); zs.avail_in = clen;
    zs.next_out = dst; zs.avail_out = isize;
    const int rc = inflate(&zs, Z_FINISH);
    const bool ok = (rc == Z_STREAM_END) && zs.total_out == isize;
    inflateEnd(&zs);
    return ok;
}

// aux walk: find CG:B,I (real CIGAR of reads with > 65535 operators)
bool find_cg(const uint8_t* p, const uint8_t* end, const uint8_t*& data, uint32_t& n) {
    while (end - p >= 3) {
        const uint8_t* nx = aux_field_end(p, end);
        if (!nx) return false;
        if (p[0] == 'C' && p[1] == 'G' && p[2] == 'B' && p[3] == 'I') { data = p + 8; n = rd32(p + 4); return true; }
        p = nx;
    }
    return false;
}

}  // namespace

std::string read_bam(const char* path, int32_t n_chrom, const char* const* chrom_names, int n_threads, BamRecords& out, bool want_xs) {
    out = BamRecords();
    const int fd = open(path, O_RDONLY);
    if (fd < 0) return std::string("cannot open BAM file ") + path;
    struct stat st;
    if (fstat(fd, &st) != 0 || st.st_size < 28) { close(fd); return std::string("BAM file too small: ") + path; }
    const size_t fsz = (size_t)st.st_size;
    const uint8_t* file = (const uint8_t*)mmap(nullptr, fsz, PROT_READ, MAP_PRIVATE, fd, 0);
    close(fd);
    if (file == MAP_FAILED) return std::string("mmap failed for ") + path;
    madvise((void*)file, fsz, MADV_SEQUENTIAL);
    struct Unmap { const uint8_t* p; size_t n; ~Unmap() { munmap((void*)p, n); } } unmap{file, fsz};

    // ---- BGZF block index ------------------------------------------------------------------------
    std::vector<BgzfBlock> blocks;
    size_t off = 0, utotal = 0;
    while (off + 18 <= fsz) {
        const uint8_t* h = file + off;
        if (h[0] != 0x1f || h[1] != 0x8b || h[2] != 8 || !(h[3] & 4)) return "not a BGZF file (bad gzip member header)";
        const uint32_t xlen = rd16(h + 10);
        if (off + 12 + xlen > fsz) return "truncated BGZF header";
        uint32_t bsize = 0;
        bool have = false;
        for (uint32_t x = 0; x + 4 <= xlen;) {
            const uint8_t* e = h + 12 + x;
            const uint32_t slen = rd16(e + 2);
            if (e[0] == 'B' && e[1] == 'C' && slen == 2 && x + 6 <= xlen) { bsize = rd16(e + 4); have = true; }
            x += 4 + slen;
        }
        if (!have) return "BGZF member without BC subfield";
        const size_t total = (size_t)bsize + 1;
        if (off + total > fsz || total < 12 + xlen + 8) return "truncated BGZF block";
        BgzfBlock b;
        b.coff = off + 12 + xlen;
        b.clen = (uint32_t)(total - 12 - xlen - 8);
        b.isize = rd32(file + off + total - 4);
        if (b.isize > 65536u) return "BGZF member claims more than 64 KiB of data (ISIZE)";     // the format's bound; bam_scan enforces the same
        b.crc = rd32(file + off + total - 8);
        b.uoff = utotal;
        utotal += b.isize;
        if (b.isize) blocks.push_back(b);
        off += total;
    }
    if (off != fsz) return "trailing garbage after last BGZF block";

    const int nthr = worker_count(n_threads);
    const size_t SLAB = (size_t)256 << 20;
    std::vector<uint8_t> buf;          // carry-over bytes + inflated slab
    size_t carry = 0;
    std::vector<int32_t> refmap;
    bool header_done = false;
    int32_t cur_chrom = INT32_MIN;
    out.cig_off.push_back(0);

    size_t bi = 0;
    while (bi < blocks.size()) {
        size_t bj = bi, ubytes = 0;
        while (bj < blocks.size() && (ubytes == 0 || ubytes + blocks[bj].isize <= SLAB)) ubytes += blocks[bj++].isize;
        buf.resize(carry + ubytes);
        const size_t ubase = blocks[bi].uoff;
        std::atomic<size_t> next(bi);
        std::atomic<bool> bad(false);
        auto work = [&]() {
            for (;;) {
                const size_t k = next.fetch_add(1);
                if (k >= bj) break;
                const BgzfBlock& b = blocks[k];
                uint8_t* dst = buf.data() + carry + (b.uoff - ubase);
                if (!inflate_block(file + b.coff, b.clen, dst, b.isize)) bad = true;
                else if ((uint32_t)crc32(crc32(0L, Z_NULL, 0), dst, b.isize) != b.crc) bad = true;     // htslib checks it too: a damaged member that still inflates to ISIZE bytes must not be counted
            }
        };
        std::vector<std::thread> pool;
        const int nt = (int)std::min<size_t>((size_t)nthr, bj - bi);
        for (int t = 1; t < nt; ++t) pool.emplace_back(work);
        work();
        for (auto& t : pool) t.join();
        if (bad) return "BGZF inflate failed (corrupt block or CRC32 mismatch)";
        bi = bj;

        const uint8_t* p = buf.data();
        const uint8_t* end = p + buf.size();
        if (!header_done) {
            if (end - p < 12 || memcmp(p, "BAM\1", 4) != 0) return "not a BAM file (bad magic)";
            const int64_t l_text = rdi32(p + 4);
            if (l_text < 0 || p + 8 + l_text + 4 > end) return "BAM header larger than the first 256 MB slab";
            const uint8_t* q = p + 8 + l_text;
            const int32_t n_ref = rdi32(q);
            q += 4;
            std::unordered_map<std::string, int32_t> names;
            for (int32_t c = 0; c < n_chrom; ++c)
                if (chrom_names && chrom_names[c]) names.emplace(chrom_names[c], c);
            refmap.assign((size_t)std::max(n_ref, 0), -1);
            for (int32_t r = 0; r < n_ref; ++r) {
                if (q + 4 > end) return "truncated BAM reference list";
                const int32_t l_name = rdi32(q);
                if (l_name < 1 || q + 4 + l_name + 4 > end) return "truncated BAM reference list";
                std::string nm((const char*)q + 4, (size_t)l_name - 1);
                auto it = names.find(nm);
                if (it != names.end()) refmap[(size_t)r] = it->second;
                q += 4 + l_name + 4;
            }
            p = q;
            header_done = true;
        }
        while (end - p >= 4) {
            const uint32_t bs = rd32(p);
            if (bs < 32) return "corrupt BAM record (block_size < 32)";
            if ((size_t)(end - p) < 4 + (size_t)bs) break;
            const uint8_t* r = p + 4;
            const int32_t refid = rdi32(r), pos0 = rdi32(r + 4);
            const uint32_t l_name = r[8];
            uint32_t n_cig = rd16(r + 12);
            const uint16_t flag = rd16(r + 14);
            const int32_t l_seq = rdi32(r + 16);
            const uint8_t* cig = r + 32 + l_name;
            if (32 + (size_t)l_name + (size_t)n_cig * 4 > bs) return "corrupt BAM record (CIGAR overruns record)";
            out.n_total++;
            p += 4 + bs;
            // end of QUAL = start of the aux fields (l_seq < 0 or past the record: no aux block)
            const uint8_t* aux = l_seq >= 0 ? cig + 4 * (size_t)n_cig + ((size_t)l_seq + 1) / 2 + (size_t)l_seq : nullptr;
            if (aux && aux > r + bs) aux = nullptr;
            if (n_cig == 2 && l_seq >= 0 && rd32(cig) == (((uint32_t)l_seq << 4) | 4u) && (rd32(cig + 4) & 15u) == 3u) {
                const uint8_t* cg = nullptr;
                uint32_t n = 0;
                if (aux && find_cg(aux, r + bs, cg, n)) { cig = cg; n_cig = n; }
            }
            const int32_t chrom = (refid >= 0 && (size_t)refid < refmap.size()) ? refmap[(size_t)refid] : -1;
            if (chrom < 0 || n_cig == 0) { out.n_skipped++; continue; }
            if (chrom != cur_chrom) {
                out.seg_chrom.push_back(chrom);
                out.seg_off.push_back((int64_t)out.pos.size());
                cur_chrom = chrom;
            }
            out.pos.push_back(pos0 + 1);
            out.flag.push_back(flag);
            if (want_xs) out.xs.push_back(aux ? aux_xs_strand(aux, r + bs) : (uint8_t)'?');
            const size_t c0 = out.cigar.size();
            out.cigar.resize(c0 + n_cig);
            memcpy(out.cigar.data() + c0, cig, (size_t)n_cig * 4);   // BAM is little-endian, so is every host we build for
            if (out.cigar.size() >= (size_t)UINT32_MAX) return "more than 2^32 CIGAR operators in one BAM";
            out.cig_off.push_back((uint32_t)out.cigar.size());
        }
        carry = (size_t)(end - p);
        if (carry) memmove(buf.data(), p, carry);
        buf.resize(carry);
    }
    if (!header_done) return "empty BAM file";
    if (carry) return "truncated BAM (partial record at end of file)";
    out.seg_off.push_back((int64_t)out.pos.size());
    if (out.seg_chrom.empty()) out.seg_off.assign(1, 0);
    return "";
}

// ---- scan for the device ingest path (bam_gpu.cu) -----------------------------------------------
std::string bam_scan(const uint8_t* file, size_t fsz, int32_t n_chrom, const char* const* chrom_names, std::vector<BgzfMember>& members,
                     uint64_t& total_u, uint64_t& first_record, int32_t& n_ref, std::vector<int32_t>& refmap,
                     std::vector<std::string>* ref_names) {
    members.clear();
    if (ref_names) ref_names->clear();
    size_t off = 0;
    uint64_t utotal = 0;
    while (off + 18 <= fsz) {
        const uint8_t* h = file + off;
        if (h[0] != 0x1f || h[1] != 0x8b || h[2] != 8 || !(h[3] & 4)) return "not a BGZF file (bad gzip member header)";
        const uint32_t xlen = rd16(h + 10);
        if (off + 12 + xlen > fsz) return "truncated BGZF header";
        uint32_t bsize = 0;
        bool have = false;
        for (uint32_t x = 0; x + 4 <= xlen;) {
            const uint8_t* e = h + 12 + x;
            const uint32_t slen = rd16(e + 2);
            if (e[0] == 'B' && e[1] == 'C' && slen == 2 && x + 6 <= xlen) { bsize = rd16(e + 4); have = true; }
            x += 4 + slen;
        }
        if (!have) return "BGZF member without BC subfield";
        const size_t total = (size_t)bsize + 1;
        if (off + total > fsz || total < 12 + xlen + 8) return "truncated BGZF block";
        BgzfMember b;
        b.coff = off + 12 + xlen;
        b.clen = (uint32_t)(total - 12 - xlen - 8);
        b.isize = rd32(file + off + total - 4);
        b.uoff = utotal;
        if (b.isize > 65536) return "BGZF member larger than 64 KiB";
        utotal += b.isize;
        if (b.isize) members.push_back(b);
        off += total;
    }
    if (off != fsz) return "trailing garbage after last BGZF block";
    total_u = utotal;
    // ---- header: inflate leading members on the host until it is complete
    std::vector<uint8_t> hb;
    size_t mi = 0;
    auto need = [&](size_t bytes) -> bool {
        while (hb.size() < bytes && mi < members.size()) {
            const BgzfMember& b = members[mi++];
            const size_t o = hb.size();
            hb.resize(o + b.isize);
            if (!inflate_block(file + b.coff, b.clen, hb.data() + o, b.isize)) return false;
        }
        return hb.size() >= bytes;
    };
    if (!need(12) || memcmp(hb.data(), "BAM\1", 4) != 0) return "not a BAM file (bad magic)";
    const int64_t l_text = rdi32(hb.data() + 4);
    if (l_text < 0 || !need(8 + (size_t)l_text + 4)) return "truncated BAM header";
    size_t q = 8 + (size_t)l_text;
    n_ref = rdi32(hb.data() + q);
    q += 4;
    if (n_ref < 0) return "corrupt BAM header (n_ref < 0)";
    std::unordered_map<std::string, int32_t> names;
    for (int32_t c = 0; c < n_chrom; ++c)
        if (chrom_names && chrom_names[c]) names.emplace(chrom_names[c], c);
    refmap.assign((size_t)n_ref, -1);
    for (int32_t r = 0; r < n_ref; ++r) {
        if (!need(q + 4)) return "truncated BAM reference list";
        const int32_t l_name = rdi32(hb.data() + q);
        if (l_name < 1 || !need(q + 4 + (size_t)l_name + 4)) return "truncated BAM reference list";
        std::string nm((const char*)hb.data() + q + 4, (size_t)l_name - 1);
        auto it = names.find(nm);
        if (it != names.end()) refmap[(size_t)r] = it->second;
        if (ref_names) ref_names->push_back(std::move(nm));
        q += 4 + (size_t)l_name + 4;
    }
    first_record = q;
    return "";
}

// ---- writer -------------------------------------------------------------------------------------
namespace {

inline void wr16(std::vector<uint8_t>& v, uint16_t x) { v.push_back((uint8_t)x); v.push_back((uint8_t)(x >> 8)); }
inline void wr32(std::vector<uint8_t>& v, uint32_t x) { for (int i = 0; i < 4; ++i) v.push_back((uint8_t)(x >> (8 * i))); }

int reg2bin(int64_t beg, int64_t end) {
    --end;
    if (beg >> 14 == end >> 14) return (int)(((1 << 15) - 1) / 7 + (beg >> 14));
    if (beg >> 17 == end >> 17) return (int)(((1 << 12) - 1) / 7 + (beg >> 17));
    if (beg >> 20 == end >> 20) return (int)(((1 << 9) - 1) / 7 + (beg >> 20));
    if (beg >> 23 == end >> 23) return (int)(((1 << 6) - 1) / 7 + (beg >> 23));
    if (beg >> 26 == end >> 26) return (int)(((1 << 3) - 1) / 7 + (beg >> 26));
    return 0;
}

bool deflate_block(const uint8_t* src, uint32_t n, std::vector<uint8_t>& dst) {
    dst.resize(18 + compressBound(n) + 8);
    z_stream zs;
    memset(&zs, 0, sizeof zs);
    if (deflateInit2(&zs, 1, Z_DEFLATED, -15, 8, Z_DEFAULT_STRATEGY) != Z_OK) return false;
    zs.next_in = const_cast<Bytef*>(src); zs.avail_in = n;
    zs.next_out = dst.data() + 18; zs.avail_out = (uInt)(dst.size() - 18 - 8);
    const int rc = deflate(&zs, Z_FINISH);
    const size_t clen = zs.total_out;
    deflateEnd(&zs);
    if (rc != Z_STREAM_END) return false;
    const size_t total = 18 + clen + 8;
    if (total > 65536) return false;
    static const uint8_t hdr[12] = {0x1f, 0x8b, 8, 4, 0, 0, 0, 0, 0, 0xff, 6, 0};
    memcpy(dst.data(), hdr, 12);
    dst[12] = 'B'; dst[13] = 'C'; dst[14] = 2; dst[15] = 0;
    dst[16] = (uint8_t)((total - 1) & 0xff); dst[17] = (uint8_t)((total - 1) >> 8);
    const uint32_t crc = (uint32_t)crc32(crc32(0L, Z_NULL, 0), src, n);
    uint8_t* t = dst.data() + 18 + clen;
    for (int i = 0; i < 4; ++i) t[i] = (uint8_t)(crc >> (8 * i));
    for (int i = 0; i < 4; ++i) t[4 + i] = (uint8_t)(n >> (8 * i));
    dst.resize(total);
    return true;
}

}  // namespace

std::string write_bam(const char* path, int32_t n_ref, const char* const* ref_names, const int32_t* ref_len,
                      const spl_records_view* rec, int n_threads, bool with_seq, const int64_t* aux_off, const uint8_t* aux) {
    if (!path || !rec || n_ref < 0 || (aux_off && !aux)) return "bad argument";
    std::vector<uint8_t> u;
    u.reserve((size_t)rec->n_rec * (with_seq ? 300 : 40) + (size_t)rec->n_cigar * 4 + 4096);
    u.insert(u.end(), {'B', 'A', 'M', 1});
    std::string text = "@HD\tVN:1.6\tSO:coordinate\n";
    for (int32_t r = 0; r < n_ref; ++r)
        text += std::string("@SQ\tSN:") + ref_names[r] + "\tLN:" + std::to_string(ref_len ? ref_len[r] : (1 << 29)) + "\n";
    wr32(u, (uint32_t)text.size());
    u.insert(u.end(), text.begin(), text.end());
    wr32(u, (uint32_t)n_ref);
    for (int32_t r = 0; r < n_ref; ++r) {
        const size_t l = strlen(ref_names[r]) + 1;
        wr32(u, (uint32_t)l);
        u.insert(u.end(), ref_names[r], ref_names[r] + l);
        wr32(u, (uint32_t)(ref_len ? ref_len[r] : (1 << 29)));
    }
    for (int32_t s = 0; s < rec->n_seg; ++s) {
        const int32_t ref = rec->seg_chrom[s];
        if (ref >= n_ref) return "segment reference index out of range";
        for (int64_t i = rec->seg_off[s]; i < rec->seg_off[s + 1]; ++i) {
            const uint32_t c0 = rec->cig_off[i], c1 = rec->cig_off[i + 1];
            uint32_t n_cig = c1 - c0;
            if (n_cig > 65535) return "write_bam: more than 65535 CIGAR operators (CG tag not written)";
            int64_t reflen = 0;
            for (uint32_t k = c0; k < c1; ++k) {
                const uint32_t op = rec->cigar[k] & 15u;
                if (op == 0 || op == 2 || op == 3 || op == 7 || op == 8) reflen += rec->cigar[k] >> 4;
            }
            const int32_t pos0 = rec->pos[i] - 1;
            const int64_t a0 = aux_off ? aux_off[i] : 0, a1 = aux_off ? aux_off[i + 1] : 0;
            if (a1 < a0 || a1 - a0 > (1 << 24)) return "write_bam: bad aux offsets";
            const uint32_t n_aux = (uint32_t)(a1 - a0);
            if (!with_seq) {
                wr32(u, 32 + 2 + n_cig * 4 + n_aux);
                wr32(u, (uint32_t)ref);
                wr32(u, (uint32_t)pos0);
                u.push_back(2);                       // l_read_name
                u.push_back(255);                     // mapq
                wr16(u, (uint16_t)reg2bin(pos0, pos0 + (reflen ? reflen : 1)));
                wr16(u, (uint16_t)n_cig);
                wr16(u, rec->flag[i]);
                wr32(u, 0);                           // l_seq
                wr32(u, (uint32_t)-1); wr32(u, (uint32_t)-1); wr32(u, 0);   // next_refID, next_pos, tlen
                u.push_back('r'); u.push_back(0);
                for (uint32_t k = c0; k < c1; ++k) wr32(u, rec->cigar[k]);
                u.insert(u.end(), aux + a0, aux + a1);
                continue;
            }
            // a sequencer-shaped record: read name, SEQ and QUAL of the CIGAR's query length (seeded pseudo-random bases and
            // qualities: the member then consists mostly of literals, like a real file; the counting path reads none of it)
            uint32_t qlen = 0;
            for (uint32_t k = c0; k < c1; ++k) {
                const uint32_t op = rec->cigar[k] & 15u;
                if (op == 0 || op == 1 || op == 4 || op == 7 || op == 8) qlen += rec->cigar[k] >> 4;
            }
            char name[16];
            const int ln = snprintf(name, sizeof name, "r%09lld", (long long)(i % 1000000000LL)) + 1;
            wr32(u, 32 + (uint32_t)ln + n_cig * 4 + (qlen + 1) / 2 + qlen + n_aux);
            wr32(u, (uint32_t)ref);
            wr32(u, (uint32_t)pos0);
            u.push_back((uint8_t)ln);
            u.push_back(255);
            wr16(u, (uint16_t)reg2bin(pos0, pos0 + (reflen ? reflen : 1)));
            wr16(u, (uint16_t)n_cig);
            wr16(u, rec->flag[i]);
            wr32(u, qlen);
            wr32(u, (uint32_t)-1); wr32(u, (uint32_t)-1); wr32(u, 0);
            u.insert(u.end(), name, name + ln);
            for (uint32_t k = c0; k < c1; ++k) wr32(u, rec->cigar[k]);
            uint64_t x = 0x9e3779b97f4a7c15ull * (uint64_t)(i + 1);
            auto rnd = [&x]() { x ^= x << 13; x ^= x >> 7; x ^= x << 17; return x; };
            static const uint8_t base4[4] = {1, 2, 4, 8};          // A C G T in the 4-bit encoding
            for (uint32_t q = 0; q < (qlen + 1) / 2; ++q) { const uint64_t v = rnd(); u.push_back((uint8_t)((base4[v & 3] << 4) | base4[(v >> 2) & 3])); }
            uint32_t ql = 30;
            for (uint32_t q = 0; q < qlen; ++q) {                   // a slow random walk around Q30, like a quality string
                const uint64_t v = rnd();
                if ((v & 7) == 0) ql = 2 + (uint32_t)((v >> 8) % 39);
                u.push_back((uint8_t)ql);
            }
            u.insert(u.end(), aux + a0, aux + a1);
        }
    }
    const size_t PIECE = 0xff00;
    const size_t nblk = (u.size() + PIECE - 1) / PIECE;
    std::vector<std::vector<uint8_t>> comp(nblk);
    std::atomic<size_t> next(0);
    std::atomic<bool> bad(false);
    auto work = [&]() {
        for (;;) {
            const size_t k = next.fetch_add(1);
            if (k >= nblk) break;
            const size_t o = k * PIECE;
            if (!deflate_block(u.data() + o, (uint32_t)std::min(PIECE, u.size() - o), comp[k])) bad = true;
        }
    };
    std::vector<std::thread> pool;
    const int nt = (int)std::min<size_t>((size_t)worker_count(n_threads), std::max<size_t>(nblk, 1));
    for (int t = 1; t < nt; ++t) pool.emplace_back(work);
    work();
    for (auto& t : pool) t.join();
    if (bad) return "deflate failed";
    FILE* f = fopen(path, "wb");
    if (!f) return std::string("cannot create ") + path;
    for (auto& c : comp)
        if (fwrite(c.data(), 1, c.size(), f) != c.size()) { fclose(f); return "short write"; }
    static const uint8_t eof[28] = {0x1f, 0x8b, 8, 4, 0, 0, 0, 0, 0, 0xff, 6, 0, 'B', 'C', 2, 0, 0x1b, 0, 3, 0, 0, 0, 0, 0, 0, 0, 0, 0};
    fwrite(eof, 1, 28, f);
    if (fclose(f) != 0) return "close failed";
    return "";
}

}  // namespace spl

// ---- C ABI for the BAM utilities ------------------------------------------------------------------
struct spl_records {
    spl::BamRecords r;
    spl_records_view v;
    bool has_xs = false;    // read by spl_read_bam_xs: r.xs holds one strand byte per record
};

extern "C" {

int spl_write_bam_seq(const char* path, int32_t n_ref, const char* const* ref_names, const int32_t* ref_len,
                      const spl_records_view* rec, int n_threads) {
    const std::string e = spl::write_bam(path, n_ref, ref_names, ref_len, rec, n_threads, true);
    if (!e.empty()) { fprintf(stderr, "spl_write_bam_seq: %s\n", e.c_str()); return SPL_ERR_IO; }
    return SPL_OK;
}

int spl_write_bam_aux(const char* path, int32_t n_ref, const char* const* ref_names, const int32_t* ref_len, const spl_records_view* rec,
                      const int64_t* aux_off, const uint8_t* aux, int with_seq, int n_threads) {
    if (!aux_off) return SPL_ERR_ARG;
    const std::string e = spl::write_bam(path, n_ref, ref_names, ref_len, rec, n_threads, with_seq != 0, aux_off, aux);
    if (!e.empty()) { fprintf(stderr, "spl_write_bam_aux: %s\n", e.c_str()); return SPL_ERR_IO; }
    return SPL_OK;
}

int spl_write_bam(const char* path, int32_t n_ref, const char* const* ref_names, const int32_t* ref_len,
                  const spl_records_view* rec, int n_threads) {
    const std::string e = spl::write_bam(path, n_ref, ref_names, ref_len, rec, n_threads);
    if (!e.empty()) { fprintf(stderr, "spl_write_bam: %s\n", e.c_str()); return SPL_ERR_IO; }
    return SPL_OK;
}

namespace {
int read_bam_handle(const char* path, int32_t n_chrom, const char* const* chrom_names, int n_threads, bool want_xs, spl_records** out,
                    char* err, int err_len) {
    if (!out || !path) return SPL_ERR_ARG;
    *out = nullptr;
    spl_records* h = new (std::nothrow) spl_records();
    if (!h) return SPL_ERR_NOMEM;
    const std::string e = spl::read_bam(path, n_chrom, chrom_names, n_threads, h->r, want_xs);
    if (!e.empty()) {
        if (err && err_len > 0) snprintf(err, (size_t)err_len, "%s", e.c_str());
        delete h;
        return SPL_ERR_IO;
    }
    h->v = h->r.view();
    h->has_xs = want_xs;
    *out = h;
    return SPL_OK;
}
}  // namespace

int spl_read_bam(const char* path, int32_t n_chrom, const char* const* chrom_names, int n_threads, spl_records** out,
                 char* err, int err_len) {
    return read_bam_handle(path, n_chrom, chrom_names, n_threads, false, out, err, err_len);
}

int spl_read_bam_xs(const char* path, int32_t n_chrom, const char* const* chrom_names, int n_threads, spl_records** out,
                    char* err, int err_len) {
    return read_bam_handle(path, n_chrom, chrom_names, n_threads, true, out, err, err_len);
}

const spl_records_view* spl_records_get(const spl_records* r) { return r ? &r->v : nullptr; }
const uint8_t* spl_records_xs(const spl_records* r) { return r && r->has_xs ? r->r.xs.data() : nullptr; }

int spl_bam_reference_names(const char* path, char* names, int64_t cap, int64_t* n_ref, int64_t* bytes, char* err, int err_len) {
    if (!path || !n_ref || !bytes || cap < 0 || (cap > 0 && !names)) return SPL_ERR_ARG;
    auto fail = [&](const std::string& e) {
        if (err && err_len > 0) snprintf(err, (size_t)err_len, "%s", e.c_str());
        return SPL_ERR_IO;
    };
    const int fd = open(path, O_RDONLY);
    if (fd < 0) return fail(std::string("cannot open BAM file ") + path);
    struct stat st;
    if (fstat(fd, &st) != 0 || st.st_size < 28) { close(fd); return fail(std::string("BAM file too small: ") + path); }
    const size_t fsz = (size_t)st.st_size;
    const uint8_t* file = (const uint8_t*)mmap(nullptr, fsz, PROT_READ, MAP_PRIVATE, fd, 0);
    close(fd);
    if (file == MAP_FAILED) return fail(std::string("mmap failed for ") + path);
    std::vector<spl::BgzfMember> members;
    std::vector<int32_t> refmap;
    std::vector<std::string> ref;
    uint64_t total_u = 0, first_record = 0;
    int32_t nr = 0;
    const std::string e = spl::bam_scan(file, fsz, 0, nullptr, members, total_u, first_record, nr, refmap, &ref);
    munmap((void*)file, fsz);
    if (!e.empty()) return fail(e);
    int64_t need = 0;
    for (const auto& s : ref) need += (int64_t)s.size() + 1;
    *n_ref = (int64_t)ref.size();
    *bytes = need;
    if (cap >= need) {
        char* p = names;
        for (const auto& s : ref) { memcpy(p, s.c_str(), s.size() + 1); p += s.size() + 1; }
    }
    return SPL_OK;
}
void spl_records_free(spl_records* r) { delete r; }

}  // extern "C"
