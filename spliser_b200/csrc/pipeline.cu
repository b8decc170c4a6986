// Context, device memory management, kernel orchestration and the C ABI of libspliser_b200.so.
// See include/spliser_b200.h for the contract of every entry point.
#include <cuda_runtime.h>

#include <algorithm>
#include <chrono>
#include <climits>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <functional>
#include <fcntl.h>
#include <sys/stat.h>
#include <unistd.h>
#include <atomic>
#include <memory>
#include <mutex>
#include <string>
#include <thread>
#include <vector>

#include "../../include/spliser_b200.h"
#include "bam_gpu.h"
#include "bam_io.h"
#include "device_types.h"
#include "graph_build.h"
#include "group_split.h"
#include "junction_filter.h"
#include "site_graph.h"
#include "strand_votes.h"

using namespace spl;

namespace {

double now_ms() {
    using namespace std::chrono;
    return duration<double, std::milli>(steady_clock::now().time_since_epoch()).count();
}

struct DevBuf {
    void* p = nullptr;
    size_t cap = 0;
    cudaError_t reserve(size_t bytes) {
        if (bytes <= cap) return cudaSuccess;
        if (p) cudaFree(p);
        p = nullptr; cap = 0;
        size_t want = bytes + bytes / 8 + 4096;
        cudaError_t e = cudaMalloc(&p, want);
        if (e != cudaSuccess) { cudaGetLastError(); want = bytes; e = cudaMalloc(&p, want); }
        if (e == cudaSuccess) cap = want;
        return e;
    }
    void release() { if (p) cudaFree(p); p = nullptr; cap = 0; }
};

// carve sub-arrays out of one allocation
struct Carver {
    size_t off = 0;
    template <class T> size_t take(size_t n) {
        off = (off + 255) & ~(size_t)255;
        const size_t o = off;
        off += n * sizeof(T);
        return o;
    }
};

}  // namespace

// Result arrays live in ONE host allocation (page-locked when a device is present, so the D2H copies run at
// full PCIe speed); freed arenas are kept in a small pool because pinning tens of MB costs milliseconds.
struct spl_result {
    int64_t n = 0, E = 0, C = 0;
    void* arena = nullptr;
    size_t bytes = 0;
    bool pinned = false;
    int32_t *chrom = nullptr, *pos = nullptr;
    uint8_t* strand = nullptr;
    int64_t *alpha = nullptr, *beta1 = nullptr, *beta2s = nullptr, *beta2c = nullptr, *first_line = nullptr;
    double *beta2w = nullptr, *sse = nullptr;
    int64_t *pc_off = nullptr, *pc_cnt = nullptr, *cp_off = nullptr;
    int32_t *pc_pos = nullptr, *cp_pos = nullptr;
};

namespace {
struct Arena { void* p; size_t bytes; bool pinned; };
std::mutex g_pool_mu;
std::vector<Arena> g_pool;

Arena arena_get(size_t bytes, bool pinned) {
    {
        std::lock_guard<std::mutex> lk(g_pool_mu);
        size_t best = g_pool.size();
        for (size_t i = 0; i < g_pool.size(); ++i)
            if (g_pool[i].pinned == pinned && g_pool[i].bytes >= bytes && (best == g_pool.size() || g_pool[i].bytes < g_pool[best].bytes)) best = i;
        if (best < g_pool.size()) { Arena a = g_pool[best]; g_pool.erase(g_pool.begin() + (ptrdiff_t)best); return a; }
    }
    Arena a{nullptr, bytes + bytes / 8 + 4096, pinned};
    if (pinned) {
        if (cudaHostAlloc(&a.p, a.bytes, cudaHostAllocDefault) != cudaSuccess) { cudaGetLastError(); a.p = nullptr; }
    } else {
        a.p = malloc(a.bytes);
    }
    return a;
}
void arena_put(Arena a) {
    if (!a.p) return;
    {
        std::lock_guard<std::mutex> lk(g_pool_mu);
        if (g_pool.size() < 4) { g_pool.push_back(a); return; }
    }
    if (a.pinned) cudaFreeHost(a.p); else free(a.p);
}

spl_result* result_alloc(size_t S, size_t E, size_t C, bool pinned) {
    Carver c;
    const size_t o_chrom = c.take<int32_t>(S + 1), o_pos = c.take<int32_t>(S + 1), o_strand = c.take<uint8_t>(S + 1);
    const size_t o_alpha = c.take<int64_t>(S + 1), o_b1 = c.take<int64_t>(S + 1), o_b2s = c.take<int64_t>(S + 1), o_b2c = c.take<int64_t>(S + 1);
    const size_t o_fl = c.take<int64_t>(S + 1), o_b2w = c.take<double>(S + 1), o_sse = c.take<double>(S + 1);
    const size_t o_pco = c.take<int64_t>(S + 2), o_pcc = c.take<int64_t>(E + 1), o_cpo = c.take<int64_t>(S + 2);
    const size_t o_pcp = c.take<int32_t>(E + 1), o_cpp = c.take<int32_t>(C + 1);
    Arena a = arena_get(c.off + 256, pinned);
    if (!a.p) return nullptr;
    spl_result* r = new (std::nothrow) spl_result();
    if (!r) { arena_put(a); return nullptr; }
    char* b = (char*)a.p;
    r->n = (int64_t)S; r->E = (int64_t)E; r->C = (int64_t)C;
    r->arena = a.p; r->bytes = a.bytes; r->pinned = a.pinned;
    r->chrom = (int32_t*)(b + o_chrom); r->pos = (int32_t*)(b + o_pos); r->strand = (uint8_t*)(b + o_strand);
    r->alpha = (int64_t*)(b + o_alpha); r->beta1 = (int64_t*)(b + o_b1); r->beta2s = (int64_t*)(b + o_b2s); r->beta2c = (int64_t*)(b + o_b2c);
    r->first_line = (int64_t*)(b + o_fl); r->beta2w = (double*)(b + o_b2w); r->sse = (double*)(b + o_sse);
    r->pc_off = (int64_t*)(b + o_pco); r->pc_cnt = (int64_t*)(b + o_pcc); r->cp_off = (int64_t*)(b + o_cpo);
    r->pc_pos = (int32_t*)(b + o_pcp); r->cp_pos = (int32_t*)(b + o_cpp);
    r->pc_off[0] = 0; r->cp_off[0] = 0;
    if (S == 0) { r->pc_off[1] = 0; r->cp_off[1] = 0; }
    return r;
}
void result_from_host_graph(spl_result* r, const SiteGraph& h) {
    const size_t S = (size_t)h.n_sites, E = h.pc_pos.size(), Cn = h.cp_pos.size();
    if (S) {
        memcpy(r->chrom, h.chrom.data(), S * 4); memcpy(r->pos, h.pos.data(), S * 4); memcpy(r->strand, h.strand.data(), S);
        memcpy(r->first_line, h.first_line.data(), S * 8);
        memcpy(r->pc_off, h.pc_off.data(), (S + 1) * 8); memcpy(r->cp_off, h.cp_off.data(), (S + 1) * 8);
    }
    if (E) memcpy(r->pc_pos, h.pc_pos.data(), E * 4);
    if (Cn) memcpy(r->cp_pos, h.cp_pos.data(), Cn * 4);
}
}  // namespace

// Everything derived from one contiguous run of records.  A big upload is cut into up to three parts so that the expansion
// of one part overlaps the host->device copy of the next; the counting kernels then run once per part into the same
// counters (every part has its own bins / tiles / junction tables; a chromosome or a junction may appear in several
// parts -- counts are additive).
constexpr int MAX_PARTS = 3;
struct Part {
    DevBuf d_rec, d_chunks, d_soa, d_tot, d_lay, d_bins, d_jtab, d_jdense, d_cxpack;
    uint32_t* h_tot = nullptr;      // pinned totals read back during the expansion
    void* h_chunks = nullptr;       // pinned staging of the chunk table
    size_t h_chunks_bytes = 0;
    cudaEvent_t ev_up = nullptr;    // the part's records (and chunk table) have arrived
    cudaEvent_t ev_e0 = nullptr, ev_e1 = nullptr;   // bracket the part's load-time kernels (read after the call's final sync)
    bool timed = false;
    DevBins bins{};
    DevJunc jg{};
    DevRecords rec{};
    DevSoA soa{};
    Chunk* chunks = nullptr;
    int n_chunks = 0;
    void release() {
        d_rec.release(); d_chunks.release(); d_soa.release(); d_tot.release(); d_lay.release(); d_bins.release();
        d_jtab.release(); d_jdense.release(); d_cxpack.release();
    }
};

// Fused variant: the records of a call live in ONE device allocation (absolute record / CIGAR indices); the upload is cut
// into slabs so that the counting kernel of one slab runs under the copy of the next.
constexpr int MAX_FPARTS = 8;
struct FPart {
    uint32_t chunk_lo = 0, chunk_hi = 0;
    cudaEvent_t ev_up = nullptr;
    // packed / compact uploads: the slab's unpack kernel.  It is launched by the first counting pass, right in front of the slab's
    // counting kernel -- queued at upload time it would sit in the stream behind the LAST slab's copy together with everything
    // that follows it, and no counting would overlap the upload
    std::function<void(cudaStream_t)> unpack;
};

struct spl_ctx {
    int device = 0;
    cudaStream_t stream = nullptr;
    std::string err;
    int n_threads = 0;
    int tile_index = 0, tile_count = 1;
    int64_t tile_lo = -1, tile_hi = -1;   // explicit owned site range (spl_set_tile_sites); -1: equal slices by tile_index / tile_count
    int variant = SPL_VARIANT_FUSED;
    int loaded_variant = SPL_VARIANT_FUSED;
    double stats[SPL_NSTATS] = {0};
    ReadFilter rf;                  // spl_set_read_filter; {0, 0, 0} = none
    int64_t rf_counts[2] = {0, 0};  // kept / dropped by the filter in the last ingest (spl_last_read_filter)
    bool from_bam = false;          // the records of the current call came from an ingest under rf (see refuse_records)

    // fused variant (count_fused.cu)
    DevBuf d_cpk;                                        // the columns of a compact upload (spl_process_compact)
    DevBuf d_frec, d_fchunks, d_hotq, d_fpk, d_unpack;   // d_fpk: packed columns (n_op, flag8) of spl_process_packed; d_unpack: scan descriptors + ticket
    DevBuf d_xs;                    // XS strand column of host records for the extraction (SPL_FLAG_XS_STRAND)
    DevBuf d_votes;                 // strand votes: the three counters and the gene-strand index (spl_infer_strand*)
    uint32_t unpack_epoch = 0;
    uint32_t hot_cap = 0;           // items the global hot queue holds; a pass that needs more is repeated with room
    uint32_t* h_hot = nullptr;      // pinned: hot item count of the last pass
    void* h_fchunks = nullptr;
    size_t h_fchunks_bytes = 0;
    DevRecords frec{};
    FChunk* fchunks = nullptr;
    uint32_t n_fchunks = 0;
    FPart fpart[MAX_FPARTS];
    int n_fparts = 0;

    // device memory
    DevBuf d_graph, d_cnt, d_out;
    Part part[MAX_PARTS];           // record-derived state (see Part)
    int n_parts = 1;
    cudaStream_t copy_stream = nullptr;   // record uploads (so that a part's expansion overlaps the next part's copy)
    std::vector<cudaEvent_t> events;
    // device-side graph build (clean regime)
    cudaStream_t stream2 = nullptr;
    cudaEvent_t ev_graph = nullptr;
    GraphBuildMem gbm;
    JuncExtractMem jem;
    GraphDev gdev{};
    GraphCounts gcnt;
    bool graph_on_device = false;
    void* h_stage = nullptr;        // pinned staging of the host-built graph
    size_t h_stage_bytes = 0;
    // device-side BAM ingest
    BamGpuMem bgm;
    GroupSplitMem gsm;              // tag group split: the host reader's upload, the sort scratch, the tables (spl_sample_load_bam_groups;
                                    // released when the split returns, so that the context holds none of it between calls)
    DevRecordArrays dev_rec{};
    bool rec_on_device = false;     // the next load takes its records from dev_rec (no host arrays, no upload)
    spl_result* pending = nullptr;  // result whose structure arrays are already on their way to the host (device-built graph)
    void* h_file = nullptr;         // pinned image of the BAM file
    size_t h_file_bytes = 0;

    // junction table of the last clean-regime load (resident on the device): spl_resident_count rebuilds the site table
    // and graph from it in every timed iteration, so that the timed region covers every per-sample kernel
    int64_t res_n_junc = 0;
    int32_t res_n_chrom = 0, res_max_pos = 0;
    bool res_stranded = false, res_clean = false;

    // state of the last load
    SiteGraph hg;                   // host graph (structure) of the last load
    DevGraph g{};
    DevCounters cnt{};
    DevOutputs out{};
    size_t cnt_bytes = 0;
    uint32_t flags = 0;
    bool loaded = false;
    int64_t n_aligned = 0;
    int32_t n_chrom_loaded = 0;

    int fail(int code, const char* fmt, ...) {
        char buf[512];
        va_list ap;
        va_start(ap, fmt);
        vsnprintf(buf, sizeof buf, fmt, ap);
        va_end(ap);
        err = buf;
        return code;
    }
};

#define CU(call)                                                                                   \
    do {                                                                                           \
        cudaError_t _e = (call);                                                                   \
        if (_e != cudaSuccess)                                                                     \
            return ctx->fail(SPL_ERR_CUDA, "%s failed: %s (%s:%d)", #call, cudaGetErrorString(_e), __FILE__, __LINE__); \
    } while (0)

namespace {

template <class T> std::vector<int32_t> to_i32(const std::vector<T>& v) {
    std::vector<int32_t> r(v.size());
    for (size_t i = 0; i < v.size(); ++i) r[i] = (int32_t)v[i];
    return r;
}

int alloc_counters_outputs(spl_ctx* ctx, size_t S, size_t E);

// site index range this context owns (tile sharding of one sample)
void owned_range(const spl_ctx* ctx, int64_t S, int32_t& lo, int32_t& hi) {
    if (ctx->tile_lo >= 0) {
        lo = (int32_t)std::min<int64_t>(ctx->tile_lo, S); hi = (int32_t)std::min<int64_t>(std::max(ctx->tile_hi, ctx->tile_lo), S);
        return;
    }
    const int64_t tc = std::max(1, ctx->tile_count), ti = std::min<int64_t>(std::max(0, ctx->tile_index), tc - 1);
    lo = (int32_t)(S * ti / tc); hi = (int32_t)(S * (ti + 1) / tc);
}

int upload_graph(spl_ctx* ctx, const int64_t* j_score, int64_t n_junc) {
    const SiteGraph& h = ctx->hg;
    const size_t S = (size_t)h.n_sites, E = h.pc_pos.size();
    if (h.pt_site.size() >= (size_t)INT_MAX || h.inc_line.size() >= (size_t)INT_MAX || h.cp_pos.size() >= (size_t)INT_MAX)
        return ctx->fail(SPL_ERR_RANGE, "site graph exceeds 2^31 entries");
    Carver c;
    const size_t o_cs = c.take<int32_t>((size_t)h.n_chrom + 1), o_pos = c.take<int32_t>(S + 64), o_cls = c.take<uint8_t>(S + 8);
    const size_t o_hot = c.take<uint8_t>(S + 64);
    // direct-address bin index of the site table
    std::vector<int32_t> sb_base((size_t)h.n_chrom + 1, 0), sb_off;
    for (int32_t ch = 0; ch < h.n_chrom; ++ch) {
        const int64_t s0 = h.cs_off[(size_t)ch], s1 = h.cs_off[(size_t)ch + 1];
        const int64_t nb = s1 > s0 ? (int64_t)(std::max(h.pos[(size_t)s1 - 1], 0) >> SB_SHIFT) + 1 : 0;
        sb_base[(size_t)ch] = (int32_t)sb_off.size();
        int64_t i = s0;
        for (int64_t b = 0; b < nb; ++b) {
            while (i < s1 && h.pos[(size_t)i] < (int32_t)(b << SB_SHIFT)) ++i;
            sb_off.push_back((int32_t)i);
        }
        sb_off.push_back((int32_t)s1);                                 // sentinel: positions beyond the last bin
    }
    sb_base[(size_t)h.n_chrom] = (int32_t)sb_off.size();
    sb_off.resize(sb_off.size() + 64, (int32_t)S);
    const size_t o_sbb = c.take<int32_t>(sb_base.size()), o_sbo = c.take<int32_t>(sb_off.size());
    const size_t o_pto = c.take<int32_t>(S + 1), o_pts = c.take<int32_t>(h.pt_site.size() + 1);
    const size_t o_pco = c.take<int32_t>(S + 1), o_pcp = c.take<int32_t>(E + 1);
    const size_t o_cpo = c.take<int32_t>(S + 1), o_cpp = c.take<int32_t>(h.cp_pos.size() + 1);
    const size_t o_rpo = c.take<int32_t>(S + 1), o_rps = c.take<int32_t>(h.rp_site.size() + 1);
    const size_t o_ino = c.take<int32_t>(S + 1), o_inl = c.take<int32_t>(h.inc_line.size() + 1);
    const size_t o_eio = c.take<int32_t>(E + 1), o_eil = c.take<int32_t>(h.einc_line.size() + 1);
    const size_t o_js = c.take<int64_t>((size_t)n_junc + 1);
    const size_t total = c.off + 256;
    CU(ctx->d_graph.reserve(total));
    if (ctx->h_stage_bytes < total) {                                   // pinned staging, kept across calls
        if (ctx->h_stage) cudaFreeHost(ctx->h_stage);
        ctx->h_stage = nullptr; ctx->h_stage_bytes = 0;
        CU(cudaHostAlloc(&ctx->h_stage, total + total / 4, cudaHostAllocDefault));
        ctx->h_stage_bytes = total + total / 4;
    }
    uint8_t* stage = (uint8_t*)ctx->h_stage;
    auto put = [&](size_t off, const void* src, size_t bytes) { if (bytes) memcpy(stage + off, src, bytes); };
    auto put32 = [&](size_t off, const std::vector<int64_t>& v, size_t expect) {
        std::vector<int32_t> t = to_i32(v);
        t.resize(expect, t.empty() ? 0 : t.back());
        put(off, t.data(), t.size() * 4);
    };
    memset(stage, 0, total);
    put32(o_cs, h.cs_off, (size_t)h.n_chrom + 1);
    {
        std::vector<int32_t> p(h.pos);
        p.resize(S + 64, INT_MAX);
        put(o_pos, p.data(), p.size() * 4);
    }
    put(o_cls, h.cls.data(), S);
    put(o_sbb, sb_base.data(), sb_base.size() * 4);
    put(o_sbo, sb_off.data(), sb_off.size() * 4);
    {   // hot[anchor] = some site of the reverse-partner list anchored here has competitors
        std::vector<uint8_t> hot(S + 64, 0);
        for (size_t a = 0; a < S; ++a)
            for (int64_t q = h.rp_off[a]; q < h.rp_off[a + 1] && !hot[a]; ++q) {
                const size_t t = (size_t)h.rp_site[(size_t)q];
                hot[a] = h.cp_off[t + 1] > h.cp_off[t];
            }
        put(o_hot, hot.data(), hot.size());
    }
    put32(o_pto, h.pt_off, S + 1); put(o_pts, h.pt_site.data(), h.pt_site.size() * 4);
    put32(o_pco, h.pc_off, S + 1); put(o_pcp, h.pc_pos.data(), E * 4);
    put32(o_cpo, h.cp_off, S + 1); put(o_cpp, h.cp_pos.data(), h.cp_pos.size() * 4);
    put32(o_rpo, h.rp_off, S + 1); put(o_rps, h.rp_site.data(), h.rp_site.size() * 4);
    put32(o_ino, h.inc_off, S + 1); put(o_inl, h.inc_line.data(), h.inc_line.size() * 4);
    put32(o_eio, h.einc_off, E + 1); put(o_eil, h.einc_line.data(), h.einc_line.size() * 4);
    if (n_junc) put(o_js, j_score, (size_t)n_junc * 8);
    CU(cudaMemcpyAsync(ctx->d_graph.p, stage, total, cudaMemcpyHostToDevice, ctx->stream));
    CU(cudaStreamSynchronize(ctx->stream));   // the staging buffer is reused by the next call
    ctx->stats[SPL_STAT_H2D_BYTES] += (double)total;
    char* b = (char*)ctx->d_graph.p;
    DevGraph& g = ctx->g;
    g.n_chrom = h.n_chrom; g.n_sites = (int32_t)S; g.n_edges = (int32_t)E;
    owned_range(ctx, (int64_t)S, g.own_lo, g.own_hi);
    g.pt_is_pc = (!h.dirty_regime && h.gap_index.empty() && h.pt_site.size() == h.pc_pos.size() && h.pt_off == h.pc_off) ? 1 : 0;
    g.cs_off = (const int32_t*)(b + o_cs); g.site_pos = (const int32_t*)(b + o_pos); g.site_cls = (const uint8_t*)(b + o_cls);
    g.site_hot = (const uint8_t*)(b + o_hot);
    g.sb_base = (const int32_t*)(b + o_sbb); g.sb_off = (const int32_t*)(b + o_sbo);
    g.pt_off = (const int32_t*)(b + o_pto); g.pt_site = (const int32_t*)(b + o_pts);
    g.pc_off = (const int32_t*)(b + o_pco); g.pc_pos = (const int32_t*)(b + o_pcp);
    g.cp_off = (const int32_t*)(b + o_cpo); g.cp_pos = (const int32_t*)(b + o_cpp);
    g.rp_off = (const int32_t*)(b + o_rpo); g.rp_site = (const int32_t*)(b + o_rps);
    g.inc_off = (const int32_t*)(b + o_ino); g.inc_line = (const int32_t*)(b + o_inl);
    g.einc_beg = (const int32_t*)(b + o_eio); g.einc_end = g.einc_beg + 1; g.einc_line = (const int32_t*)(b + o_eil);
    g.j_score = (const int64_t*)(b + o_js);

    ctx->graph_on_device = false;
    return alloc_counters_outputs(ctx, S, E);
}

int alloc_counters_outputs(spl_ctx* ctx, size_t S, size_t E) {
    // counters + outputs
    Carver cc;
    const size_t c_diff = cc.take<uint32_t>(4 * (S + 1) + 4), c_dir = cc.take<uint32_t>(4 * (S + 1) + 4), c_cov = cc.take<uint32_t>(2 * S + 2);
    const size_t c_covx = cc.take<uint32_t>(S + 1), c_spanx = cc.take<uint32_t>(S + 1), c_flank = cc.take<uint32_t>(S + 1);
    const size_t c_dc = cc.take<uint32_t>(E + 1), c_work = cc.take<uint32_t>(32);
    ctx->cnt_bytes = cc.off + 256;
    CU(ctx->d_cnt.reserve(ctx->cnt_bytes));
    char* cb = (char*)ctx->d_cnt.p;
    ctx->cnt.diff = (uint32_t*)(cb + c_diff); ctx->cnt.dir = (uint32_t*)(cb + c_dir); ctx->cnt.cov = (uint32_t*)(cb + c_cov);
    ctx->cnt.covx = (uint32_t*)(cb + c_covx); ctx->cnt.spanx = (uint32_t*)(cb + c_spanx);
    ctx->cnt.flank = (uint32_t*)(cb + c_flank); ctx->cnt.dc = (uint32_t*)(cb + c_dc); ctx->cnt.work = (uint32_t*)(cb + c_work);
    Carver oc;
    const size_t nblk = (S + FIN_THREADS - 1) / FIN_THREADS + 1;
    const size_t o_al = oc.take<int64_t>(S + 1), o_pc = oc.take<int64_t>(E + 1), o_b1 = oc.take<int64_t>(S + 1),
                 o_b2 = oc.take<int64_t>(S + 1), o_b2c = oc.take<int64_t>(S + 1), o_b2w = oc.take<double>(S + 1),
                 o_sse = oc.take<double>(S + 1), o_dct = oc.take<int64_t>(E + 1), o_dcp = oc.take<uint8_t>(E + 1),
                 o_blk = oc.take<uint32_t>(4 * nblk + 4);
    CU(ctx->d_out.reserve(oc.off + 256));
    char* ob = (char*)ctx->d_out.p;
    DevOutputs& o = ctx->out;
    o.alpha = (int64_t*)(ob + o_al); o.pc_cnt = (int64_t*)(ob + o_pc); o.beta1 = (int64_t*)(ob + o_b1);
    o.beta2s = (int64_t*)(ob + o_b2); o.beta2c = (int64_t*)(ob + o_b2c); o.beta2w = (double*)(ob + o_b2w);
    o.sse = (double*)(ob + o_sse); o.dc_tot = (int64_t*)(ob + o_dct); o.dc_present = (uint8_t*)(ob + o_dcp);
    o.span_blk = (uint32_t*)(ob + o_blk);
    // a tile context finalizes only the sites it owns; the others read back as zeros
    if (ctx->tile_count > 1 || ctx->tile_lo >= 0) CU(cudaMemsetAsync(ctx->d_out.p, 0, oc.off + 256, ctx->stream));
    return SPL_OK;
}

int check_view(spl_ctx* ctx, const spl_records_view* v, int32_t n_chrom) {
    if (!v) return ctx->fail(SPL_ERR_ARG, "records view is NULL");
    if (v->n_rec < 0 || v->n_cigar < 0 || v->n_seg < 0) return ctx->fail(SPL_ERR_ARG, "negative size in records view");
    const bool dev = ctx->rec_on_device;
    if (!dev && v->n_rec > 0 && (!v->pos || !v->flag || !v->cig_off)) return ctx->fail(SPL_ERR_ARG, "NULL record array");
    if (!dev && v->n_cigar > 0 && !v->cigar) return ctx->fail(SPL_ERR_ARG, "NULL cigar array");
    if (v->n_seg > 0 && (!v->seg_chrom || !v->seg_off)) return ctx->fail(SPL_ERR_ARG, "NULL segment array");
    if (v->n_rec >= (int64_t)UINT32_MAX - 16 || v->n_cigar >= (int64_t)UINT32_MAX - 16)
        return ctx->fail(SPL_ERR_RANGE, "more than 2^32 records or CIGAR operators in one call");
    int64_t prev = 0;
    for (int32_t k = 0; k < v->n_seg; ++k) {
        if (v->seg_off[k] != prev || v->seg_off[k + 1] < prev) return ctx->fail(SPL_ERR_ARG, "segment offsets must start at 0 and be monotone");
        prev = v->seg_off[k + 1];
        if (v->seg_chrom[k] >= n_chrom) return ctx->fail(SPL_ERR_ARG, "segment chromosome index out of range");
    }
    if (v->n_seg > 0 && prev != v->n_rec) return ctx->fail(SPL_ERR_ARG, "segments do not cover all records");
    if (v->n_seg == 0 && v->n_rec != 0) return ctx->fail(SPL_ERR_ARG, "records without segments");
    if (!dev && v->n_rec > 0 && (int64_t)v->cig_off[v->n_rec] != v->n_cigar) return ctx->fail(SPL_ERR_ARG, "cig_off[n_rec] != n_cigar");
    return SPL_OK;
}

// enqueue the upload of records [r0, r1) on the copy stream (asynchronous when the caller's arrays are
// page-locked); record / CIGAR indices inside the part are relative to its first record, CIGAR offsets stay absolute
int upload_records(spl_ctx* ctx, Part& P, const spl_records_view* v, int64_t r0, int64_t r1, int32_t n_chrom) {
    ctx->n_chrom_loaded = n_chrom;
    const bool dev = ctx->rec_on_device;
    std::vector<Chunk> hc;
    for (int32_t k = 0; k < v->n_seg; ++k) {                            // the part's share of every chromosome segment
        if (v->seg_chrom[k] < 0) continue;
        const int64_t a = std::max(v->seg_off[k], r0), b = std::min(v->seg_off[k + 1], r1);
        for (int64_t lo = a; lo < b; lo += CHUNK_READS) {
            Chunk c{};
            c.chrom = v->seg_chrom[k];
            c.rec_lo = (uint32_t)(lo - r0);
            c.rec_hi = (uint32_t)(std::min<int64_t>(lo + CHUNK_READS, b) - r0);
            hc.push_back(c);
        }
    }
    P.n_chunks = (int)hc.size();
    const size_t R = (size_t)(r1 - r0);
    const size_t c0 = (dev || R == 0) ? 0 : (size_t)v->cig_off[r0], c1 = dev ? (size_t)v->n_cigar : (R == 0 ? 0 : (size_t)v->cig_off[r1]);
    const size_t NC = c1 - c0;
    Carver c;
    const size_t o_pos = c.take<int32_t>(R + 4), o_flag = c.take<uint16_t>(R + 4), o_off = c.take<uint32_t>(R + 4),
                 o_cig = c.take<uint32_t>(NC + 4);
    if (!dev) CU(P.d_rec.reserve(c.off + 256));
    char* rb = (char*)P.d_rec.p;
    // the chunk table travels from a page-locked staging buffer on the same stream as the records, in front of them (a
    // pageable copy on the compute stream would queue behind every big copy already submitted and hold the kernels back)
    CU(P.d_chunks.reserve((hc.size() + 1) * sizeof(Chunk)));
    P.chunks = (Chunk*)P.d_chunks.p;
    cudaStream_t cs = dev ? ctx->stream : ctx->copy_stream;
    if (!hc.empty()) {
        const size_t bytes = hc.size() * sizeof(Chunk);
        if (P.h_chunks_bytes < bytes) {
            if (P.h_chunks) cudaFreeHost(P.h_chunks);
            P.h_chunks = nullptr; P.h_chunks_bytes = 0;
            CU(cudaHostAlloc(&P.h_chunks, bytes + bytes / 4 + 4096, cudaHostAllocDefault));
            P.h_chunks_bytes = bytes + bytes / 4 + 4096;
        }
        memcpy(P.h_chunks, hc.data(), bytes);
        CU(cudaMemcpyAsync(P.chunks, P.h_chunks, bytes, cudaMemcpyHostToDevice, cs));
    }
    if (dev) {                                                         // parsed on the device from the BAM (bam_gpu.cu)
        P.rec.n_rec = (uint32_t)R;
        P.rec.pos = ctx->dev_rec.pos; P.rec.flag = ctx->dev_rec.flag;
        P.rec.cig_off = ctx->dev_rec.cig_off; P.rec.cigar = ctx->dev_rec.cigar;
        CU(cudaEventRecord(P.ev_up, ctx->stream));
        return SPL_OK;
    }
    if (R) {
        CU(cudaMemcpyAsync(rb + o_pos, v->pos + r0, R * 4, cudaMemcpyHostToDevice, cs));
        CU(cudaMemcpyAsync(rb + o_flag, v->flag + r0, R * 2, cudaMemcpyHostToDevice, cs));
        CU(cudaMemcpyAsync(rb + o_off, v->cig_off + r0, (R + 1) * 4, cudaMemcpyHostToDevice, cs));
        if (NC) CU(cudaMemcpyAsync(rb + o_cig, v->cigar + c0, NC * 4, cudaMemcpyHostToDevice, cs));
    }
    CU(cudaEventRecord(P.ev_up, cs));
    ctx->stats[SPL_STAT_H2D_BYTES] += (double)(R * 10 + 4 + NC * 4 + hc.size() * sizeof(Chunk));
    P.rec.n_rec = (uint32_t)R;
    P.rec.pos = (const int32_t*)(rb + o_pos); P.rec.flag = (const uint16_t*)(rb + o_flag);
    P.rec.cig_off = (const uint32_t*)(rb + o_off);
    P.rec.cigar = (const uint32_t*)(rb + o_cig) - c0;                  // indexed with the absolute offsets of cig_off
    return SPL_OK;
}

// run the expansion kernels, leave the SoA + chunk table on the device
int expand_records(spl_ctx* ctx, Part& P, const spl_records_view* v, int64_t r0, int64_t r1, uint32_t flags) {
    CU(cudaStreamWaitEvent(ctx->stream, P.ev_up, 0));
    CU(P.d_tot.reserve(256));
    CU(cudaMemsetAsync(P.d_tot.p, 0, 256, ctx->stream));
    // per-chromosome layout arrays of the bin-partitioned stream
    DevBins& bins = P.bins;
    bins = DevBins{};
    const size_t nchr = (size_t)std::max(ctx->n_chrom_loaded, 1);
    {
        Carver lc;
        const size_t o_ext = lc.take<uint32_t>(nchr + 1), o_tot = lc.take<uint32_t>(nchr + 1), o_bb = lc.take<uint32_t>(nchr + 2),
                     o_tb = lc.take<uint32_t>(nchr + 2), o_ml = lc.take<uint32_t>(4), o_cj = lc.take<uint32_t>(nchr + 1),
                     o_jt = lc.take<uint32_t>(nchr + 2);
        CU(P.d_lay.reserve(lc.off + 256));
        CU(cudaMemsetAsync(P.d_lay.p, 0, lc.off + 256, ctx->stream));
        char* lb = (char*)P.d_lay.p;
        bins.chrom_ext = (uint32_t*)(lb + o_ext); bins.chrom_tot = (uint32_t*)(lb + o_tot);
        bins.chrom_bin_base = (uint32_t*)(lb + o_bb); bins.chrom_tile_base = (uint32_t*)(lb + o_tb);
        bins.max_len = (uint32_t*)(lb + o_ml);
        bins.chrom_jn = (uint32_t*)(lb + o_cj); bins.tab_base = (uint32_t*)(lb + o_jt);
        bins.n_chrom = ctx->n_chrom_loaded;
    }
    CU(cudaEventRecord(P.ev_e0, ctx->stream));
    launch_expand_count(P.rec, P.chunks, P.n_chunks, flags, bins, ctx->stream);
    launch_chunk_scan(P.chunks, P.n_chunks, (uint32_t*)P.d_tot.p, bins, ctx->stream);
    if (P.n_chunks) launch_jtab_layout(bins, 0, (uint32_t*)P.d_tot.p, ctx->stream);       // sizes of the junction sub-tables ride on the same read-back
    CU(cudaGetLastError());
    CU(cudaMemcpyAsync(P.h_tot, P.d_tot.p, 40, cudaMemcpyDeviceToHost, ctx->stream));
    CU(cudaStreamSynchronize(ctx->stream));   // also makes `hc` (pageable) safe to drop
    const size_t nA = P.h_tot[0], nB = P.h_tot[1], nS = P.h_tot[2], nJ = P.h_tot[3];
    const size_t total_bins = P.n_chunks ? P.h_tot[4] : 0, n_tiles = P.n_chunks ? P.h_tot[5] : 0;
    const size_t nC = n_tiles * (size_t)K3_TILE;
    if (nC >= (size_t)UINT32_MAX - 64) return ctx->fail(SPL_ERR_RANGE, "more than 2^32 mapped blocks in one call");
    Carver s;
    const size_t bB = (nA + 3) & ~(size_t)3;                      // stream B starts on a 128-bit boundary
    if (bB + nB >= (size_t)UINT32_MAX - 64) return ctx->fail(SPL_ERR_RANGE, "more than 2^32 mapped blocks in one call");
    const size_t o_ms = s.take<int32_t>(bB + nB + 32), o_me = s.take<uint32_t>(bB + nB + 32);
    const size_t o_sb = s.take<uint32_t>(nS + 16), o_sj = s.take<uint32_t>(nS + 16);
    const size_t o_jl = s.take<uint32_t>(nJ + 16), o_jr = s.take<uint32_t>(nJ + 16), o_jq = s.take<uint32_t>(nJ + 16);
    const size_t o_ja = s.take<int32_t>(nJ + 16), o_je = s.take<int32_t>(nJ + 16);
    CU(P.d_soa.reserve(s.off + 256));
    char* sb = (char*)P.d_soa.p;
    DevSoA& soa = P.soa;
    soa.nA = (uint32_t)nA; soa.nB = (uint32_t)nB; soa.nS = (uint32_t)nS; soa.nJ = (uint32_t)nJ;
    soa.m_start = (int32_t*)(sb + o_ms); soa.m_endk = (uint32_t*)(sb + o_me); soa.bB = (uint32_t)bB;
    soa.sr_boff = (uint32_t*)(sb + o_sb); soa.sr_joff = (uint32_t*)(sb + o_sj);
    soa.jn_l = (uint32_t*)(sb + o_jl); soa.jn_rk = (uint32_t*)(sb + o_jr); soa.jn_read = (uint32_t*)(sb + o_jq);
    soa.ji_a0 = (int32_t*)(sb + o_ja); soa.ji_end = (int32_t*)(sb + o_je);
    {
        Carver bc;
        const size_t nscan = (total_bins + 1 + 4095) / 4096 + 8;
        const size_t o_bo = bc.take<uint32_t>(total_bins + 8), o_bcur = bc.take<uint32_t>(total_bins + 8), o_tmp = bc.take<uint32_t>(nscan + 8),
                     o_cs = bc.take<int32_t>(nC + 32), o_ce = bc.take<uint32_t>(nC + 32), o_tl = bc.take<Tile>(n_tiles + 1);
        CU(P.d_bins.reserve(bc.off + 256));
        char* bb = (char*)P.d_bins.p;
        bins.bin_off = (uint32_t*)(bb + o_bo); bins.bin_cursor = (uint32_t*)(bb + o_bcur); bins.scan_tmp = (uint32_t*)(bb + o_tmp);
        bins.c_start = (int32_t*)(bb + o_cs); bins.c_endk = (uint32_t*)(bb + o_ce); bins.tiles = (Tile*)(bb + o_tl);
        bins.total_bins = (uint32_t)total_bins; bins.n_tiles = (uint32_t)n_tiles; bins.nC = (uint32_t)nC;
    }
    launch_expand_scatter(P.rec, P.chunks, P.n_chunks, soa, flags, ctx->stream);
    launch_bin_partition(P.chunks, P.n_chunks, soa, bins, ctx->stream);
    CU(cudaGetLastError());
    // ---- junction groups: table -> (sync: distinct count) -> dense arrays + grouped simple instances
    DevJunc& jg = P.jg;
    jg = DevJunc{};
    uint32_t* d_jtot = (uint32_t*)P.d_tot.p + 12;
    for (int attempt = 0;; ++attempt) {
        size_t n_slots = 0;
        if (P.n_chunks) {
            if (attempt > 0) {                                          // a crowded sub-table: re-size for the worst case
                launch_jtab_layout(bins, attempt, (uint32_t*)P.d_tot.p, ctx->stream);
                CU(cudaMemcpyAsync(P.h_tot + 8, (uint32_t*)P.d_tot.p + 8, 4, cudaMemcpyDeviceToHost, ctx->stream));
                CU(cudaStreamSynchronize(ctx->stream));
            }
            n_slots = P.h_tot[8];
        }
        Carver jc;
        const size_t nscan = (n_slots + 1 + 4095) / 4096 + 8;
        const size_t o_key = jc.take<unsigned long long>(n_slots + 2), o_sa = jc.take<uint32_t>(n_slots + 2),
                     o_ss = jc.take<uint32_t>(n_slots + 2), o_su = jc.take<uint32_t>(n_slots + 2), o_so = jc.take<uint32_t>(n_slots + 2),
                     o_sc = jc.take<uint32_t>(n_slots + 2), o_sl = jc.take<uint32_t>(nJ + 2), o_cn = jc.take<uint32_t>(4),
                     o_co = jc.take<uint32_t>(n_slots + 2), o_cc = jc.take<uint32_t>(n_slots + 2),
                     o_tmp = jc.take<uint32_t>(2 * nscan + 8);
        CU(P.d_jtab.reserve(jc.off + 256));
        char* jb = (char*)P.d_jtab.p;
        jg.n_slots = (uint32_t)n_slots; jg.chrom_jn = bins.chrom_jn; jg.tab_base = bins.tab_base;
        jg.key = (unsigned long long*)(jb + o_key); jg.s_all = (uint32_t*)(jb + o_sa); jg.s_simple = (uint32_t*)(jb + o_ss);
        jg.s_used = (uint32_t*)(jb + o_su); jg.s_off = (uint32_t*)(jb + o_so); jg.s_cursor = (uint32_t*)(jb + o_sc);
        jg.slot_of = (uint32_t*)(jb + o_sl); jg.cx_n = (uint32_t*)(jb + o_cn); jg.overflow = jg.cx_n + 1;
        jg.scan_tmp = (uint32_t*)(jb + o_tmp);
        jg.s_coff = (uint32_t*)(jb + o_co); jg.s_ccur = (uint32_t*)(jb + o_cc);
        launch_junction_groups_a(P.chunks, P.n_chunks, soa, jg, d_jtot, ctx->stream);
        CU(cudaGetLastError());
        CU(cudaMemcpyAsync(P.h_tot + 12, d_jtot, 16, cudaMemcpyDeviceToHost, ctx->stream));
        CU(cudaStreamSynchronize(ctx->stream));
        if (!P.h_tot[15]) break;                                    // no sub-table got crowded
        if (attempt >= 1) return ctx->fail(SPL_ERR_CUDA, "junction table overflow (internal sizing error)");
    }
    const size_t D = P.h_tot[12], n_simple = P.h_tot[13], n_complex = P.h_tot[14];
    {
        Carver dc;
        const size_t o_l = dc.take<uint32_t>(D + 2), o_rk = dc.take<uint32_t>(D + 2), o_ch = dc.take<int32_t>(D + 2),
                     o_al = dc.take<uint32_t>(D + 2), o_si = dc.take<uint32_t>(D + 2), o_of = dc.take<uint32_t>(D + 2), o_cf = dc.take<uint32_t>(D + 2),
                     o_a0 = dc.take<int32_t>(n_simple + 2), o_en = dc.take<int32_t>(n_simple + 2),
                     o_cj = dc.take<uint32_t>(n_complex + 2),
                     o_hl = dc.take<uint32_t>(D + 2), o_hr = dc.take<uint32_t>(D + 2),
                     o_wl = dc.take<unsigned long long>(2 * D + 2 * (n_simple / 2048 + 1) + 8),
                     o_xb = dc.take<uint32_t>(2 * D + 2), o_xd = dc.take<uint32_t>(2 * D + 2),
                     o_xn = dc.take<uint32_t>(2 * D + 2), o_xt = dc.take<int32_t>((2 * D + 2) * CXD_T), o_cr = dc.take<uint4>(n_complex + 2),
                     o_s0 = dc.take<uint32_t>(D + 2), o_s1 = dc.take<uint32_t>(D + 2), o_pr = dc.take<uint32_t>(8);
        CU(P.d_jdense.reserve(dc.off + 256));
        char* db = (char*)P.d_jdense.p;
        jg.D = (uint32_t)D;
        jg.dj_l = (uint32_t*)(db + o_l); jg.dj_rk = (uint32_t*)(db + o_rk); jg.dj_chrom = (int32_t*)(db + o_ch);
        jg.dj_all = (uint32_t*)(db + o_al); jg.dj_simple = (uint32_t*)(db + o_si); jg.dj_off = (uint32_t*)(db + o_of);
        jg.dj_coff = (uint32_t*)(db + o_cf);
        jg.gi_a0 = (int32_t*)(db + o_a0); jg.gi_end = (int32_t*)(db + o_en);
        jg.cx_j = (uint32_t*)(db + o_cj);
        jg.hot_l = (uint32_t*)(db + o_hl); jg.hot_r = (uint32_t*)(db + o_hr); jg.wl = (unsigned long long*)(db + o_wl);
        jg.cxd_base = (uint32_t*)(db + o_xb); jg.cxd_ds = (uint32_t*)(db + o_xd);
        jg.cxd_nt = (uint32_t*)(db + o_xn); jg.cxd_t = (int32_t*)(db + o_xt); jg.cx_rng = (uint4*)(db + o_cr);
        jg.sp_x0 = (uint32_t*)(db + o_s0); jg.sp_x1 = (uint32_t*)(db + o_s1); jg.prep = (uint32_t*)(db + o_pr);
        jg.n_complex = (uint32_t)n_complex;
    }
    launch_junction_groups_b(soa, jg, ctx->n_chrom_loaded, d_jtot, ctx->stream);
    CU(cudaGetLastError());
    CU(cudaEventRecord(P.ev_e1, ctx->stream));                         // no host sync here: the caller's next sync covers it
    P.timed = true;
    ctx->stats[SPL_STAT_N_DISTINCT_J] += (double)D; ctx->stats[SPL_STAT_N_SIMPLE_J] += (double)n_simple;
    ctx->stats[SPL_STAT_N_COMPLEX_J] += (double)jg.n_complex;
    ctx->stats[SPL_STAT_N_MBLOCKS_A] += (double)nA; ctx->stats[SPL_STAT_N_MBLOCKS_B] += (double)nB;
    ctx->stats[SPL_STAT_N_SPLICED] += (double)nS; ctx->stats[SPL_STAT_N_JUNC_OPS] += (double)nJ;
    int64_t aligned = 0;
    for (int32_t k = 0; k < v->n_seg; ++k)
        if (v->seg_chrom[k] >= 0) aligned += std::max<int64_t>(0, std::min(v->seg_off[k + 1], r1) - std::max(v->seg_off[k], r0));
    ctx->n_aligned += aligned;
    ctx->stats[SPL_STAT_N_ALIGNED] += (double)aligned;
    return SPL_OK;
}

int upload_and_expand(spl_ctx* ctx, const spl_records_view* v, uint32_t flags, int32_t n_chrom) {
    ctx->n_parts = 1;
    ctx->n_aligned = 0;
    int rc = upload_records(ctx, ctx->part[0], v, 0, v->n_rec, n_chrom);
    if (rc) return rc;
    return expand_records(ctx, ctx->part[0], v, 0, v->n_rec, flags);
}

// Fused variant: chunk table + records to the device.  The records of the call go into one allocation; a big host upload is
// cut into up to MAX_FPARTS slabs (at chunk granularity) on the copy stream, each followed by an event: the counting
// kernel of a slab runs while the next one is still on the wire.  Records parsed on the device (bam_gpu.cu) are adopted.
int fused_upload(spl_ctx* ctx, const spl_records_view* v, int32_t n_chrom, bool split_ok) {
    ctx->n_chrom_loaded = n_chrom;
    for (auto& P : ctx->fpart) P.unpack = nullptr;                    // nothing left over from an earlier call
    const bool dev = ctx->rec_on_device;
    std::vector<FChunk> hc;
    int64_t aligned = 0;
    for (int32_t k = 0; k < v->n_seg; ++k) {
        if (v->seg_chrom[k] < 0) continue;
        const int64_t a = v->seg_off[k], b = v->seg_off[k + 1];
        aligned += b - a;
        for (int64_t lo = a; lo < b; lo += FC_RECS) {
            FChunk c{};
            c.chrom = v->seg_chrom[k];
            c.rec_lo = (uint32_t)lo;
            c.rec_hi = (uint32_t)std::min<int64_t>(lo + FC_RECS, b);
            hc.push_back(c);
        }
    }
    ctx->n_aligned = aligned;
    ctx->stats[SPL_STAT_N_ALIGNED] = (double)aligned;
    ctx->n_fchunks = (uint32_t)hc.size();
    const size_t R = (size_t)v->n_rec, NC = (size_t)v->n_cigar;
    cudaStream_t cs = dev ? ctx->stream : ctx->copy_stream;
    // the chunk table travels from a page-locked staging buffer on the same stream as the records, in front of them
    CU(ctx->d_fchunks.reserve((hc.size() + 1) * sizeof(FChunk)));
    ctx->fchunks = (FChunk*)ctx->d_fchunks.p;
    if (!hc.empty()) {
        const size_t bytes = hc.size() * sizeof(FChunk);
        if (ctx->h_fchunks_bytes < bytes) {
            if (ctx->h_fchunks) cudaFreeHost(ctx->h_fchunks);
            ctx->h_fchunks = nullptr; ctx->h_fchunks_bytes = 0;
            CU(cudaHostAlloc(&ctx->h_fchunks, bytes + bytes / 4 + 4096, cudaHostAllocDefault));
            ctx->h_fchunks_bytes = bytes + bytes / 4 + 4096;
        }
        memcpy(ctx->h_fchunks, hc.data(), bytes);
        CU(cudaMemcpyAsync(ctx->fchunks, ctx->h_fchunks, bytes, cudaMemcpyHostToDevice, cs));
        ctx->stats[SPL_STAT_H2D_BYTES] += (double)bytes;
    }
    {   // global queue of hot items (count_fused.cu): sized for the usual share, grown when a pass overflows it
        const uint64_t want = std::max<uint64_t>(1u << 18, (uint64_t)v->n_cigar / 16 + (1u << 16));
        if (ctx->hot_cap < want) {
            CU(ctx->d_hotq.reserve((size_t)want * 16));
            ctx->hot_cap = (uint32_t)std::min<uint64_t>(want, 0xfffffff0u);
        }
        *ctx->h_hot = 0;
    }
    ctx->n_fparts = 1;
    ctx->fpart[0].chunk_lo = 0; ctx->fpart[0].chunk_hi = ctx->n_fchunks;
    if (dev) {
        ctx->frec.n_rec = (uint32_t)R;
        ctx->frec.pos = ctx->dev_rec.pos; ctx->frec.flag = ctx->dev_rec.flag;
        ctx->frec.cig_off = ctx->dev_rec.cig_off; ctx->frec.cigar = ctx->dev_rec.cigar;
        CU(cudaEventRecord(ctx->fpart[0].ev_up, ctx->stream));
        return SPL_OK;
    }
    Carver c;
    const size_t o_pos = c.take<int32_t>(R + 32), o_flag = c.take<uint16_t>(R + 32), o_off = c.take<uint32_t>(R + 40),
                 o_cig = c.take<uint32_t>(NC + 32);
    CU(ctx->d_frec.reserve(c.off + 256));
    char* rb = (char*)ctx->d_frec.p;
    ctx->frec.n_rec = (uint32_t)R;
    ctx->frec.pos = (const int32_t*)(rb + o_pos); ctx->frec.flag = (const uint16_t*)(rb + o_flag);
    ctx->frec.cig_off = (const uint32_t*)(rb + o_off); ctx->frec.cigar = (const uint32_t*)(rb + o_cig);
    // slabs
    int want = 1;
    {
        int64_t min_rec = 2000000;
        int max_parts = MAX_FPARTS;
        if (const char* f = std::getenv("SPLISER_SPLIT_MIN_RECORDS")) min_rec = std::max<int64_t>(1, atoll(f));
        if (const char* f = std::getenv("SPLISER_SPLIT_PARTS")) max_parts = std::max(1, std::min(MAX_FPARTS, atoi(f)));
        if (split_ok) want = (int)std::max<int64_t>(1, std::min<int64_t>(max_parts, (int64_t)R / min_rec));
        want = (int)std::min<size_t>((size_t)want, std::max<size_t>(1, hc.size()));
    }
    ctx->n_fparts = want;
    size_t r_prev = 0;
    for (int p = 0; p < want; ++p) {
        const uint32_t k0 = (uint32_t)(hc.size() * (size_t)p / (size_t)want), k1 = (uint32_t)(hc.size() * (size_t)(p + 1) / (size_t)want);
        ctx->fpart[p].chunk_lo = k0; ctx->fpart[p].chunk_hi = k1;
        const size_t r0 = r_prev, r1 = (p == want - 1 || k1 >= hc.size()) ? R : (size_t)hc[k1].rec_lo;
        r_prev = r1;
        if (r1 > r0) {
            const size_t c0 = (size_t)v->cig_off[r0], c1 = (size_t)v->cig_off[r1];
            CU(cudaMemcpyAsync(rb + o_pos + r0 * 4, v->pos + r0, (r1 - r0) * 4, cudaMemcpyHostToDevice, cs));
            CU(cudaMemcpyAsync(rb + o_flag + r0 * 2, v->flag + r0, (r1 - r0) * 2, cudaMemcpyHostToDevice, cs));
            CU(cudaMemcpyAsync(rb + o_off + r0 * 4, v->cig_off + r0, (r1 - r0 + 1) * 4, cudaMemcpyHostToDevice, cs));
            if (c1 > c0) CU(cudaMemcpyAsync(rb + o_cig + c0 * 4, v->cigar + c0, (c1 - c0) * 4, cudaMemcpyHostToDevice, cs));
            ctx->stats[SPL_STAT_H2D_BYTES] += (double)((r1 - r0) * 10 + 4 + (c1 - c0) * 4);
        }
        CU(cudaEventRecord(ctx->fpart[p].ev_up, cs));
    }
    return SPL_OK;
}

// The same for the packed host layout (spl_packed_view: POS, three flag bits, operator count; 17 B per record instead of 20):
// slabs are cut at multiples of SPL_PACKED_INDEX_STRIDE records, where the view's sparse CIGAR index gives the offsets; the
// CIGAR offsets of every record and the SAM flag bits are rebuilt on the device (k_unpack_records) as each slab arrives.
int fused_upload_packed(spl_ctx* ctx, const spl_packed_view* v, int32_t n_chrom, bool split_ok) {
    ctx->n_chrom_loaded = n_chrom;
    for (auto& P : ctx->fpart) P.unpack = nullptr;                    // nothing left over from an earlier call
    std::vector<FChunk> hc;
    int64_t aligned = 0;
    for (int32_t k = 0; k < v->n_seg; ++k) {
        if (v->seg_chrom[k] < 0) continue;
        const int64_t a = v->seg_off[k], b = v->seg_off[k + 1];
        aligned += b - a;
        for (int64_t lo = a; lo < b; lo += FC_RECS) {
            FChunk c{};
            c.chrom = v->seg_chrom[k];
            c.rec_lo = (uint32_t)lo;
            c.rec_hi = (uint32_t)std::min<int64_t>(lo + FC_RECS, b);
            hc.push_back(c);
        }
    }
    ctx->n_aligned = aligned;
    ctx->stats[SPL_STAT_N_ALIGNED] = (double)aligned;
    ctx->n_fchunks = (uint32_t)hc.size();
    const size_t R = (size_t)v->n_rec, NC = (size_t)v->n_cigar;
    cudaStream_t cs = ctx->copy_stream;
    CU(ctx->d_fchunks.reserve((hc.size() + 1) * sizeof(FChunk)));
    ctx->fchunks = (FChunk*)ctx->d_fchunks.p;
    if (!hc.empty()) {
        const size_t bytes = hc.size() * sizeof(FChunk);
        if (ctx->h_fchunks_bytes < bytes) {
            if (ctx->h_fchunks) cudaFreeHost(ctx->h_fchunks);
            ctx->h_fchunks = nullptr; ctx->h_fchunks_bytes = 0;
            CU(cudaHostAlloc(&ctx->h_fchunks, bytes + bytes / 4 + 4096, cudaHostAllocDefault));
            ctx->h_fchunks_bytes = bytes + bytes / 4 + 4096;
        }
        memcpy(ctx->h_fchunks, hc.data(), bytes);
        CU(cudaMemcpyAsync(ctx->fchunks, ctx->h_fchunks, bytes, cudaMemcpyHostToDevice, cs));
        ctx->stats[SPL_STAT_H2D_BYTES] += (double)bytes;
    }
    {
        const uint64_t want = std::max<uint64_t>(1u << 18, (uint64_t)v->n_cigar / 16 + (1u << 16));
        if (ctx->hot_cap < want) {
            CU(ctx->d_hotq.reserve((size_t)want * 16));
            ctx->hot_cap = (uint32_t)std::min<uint64_t>(want, 0xfffffff0u);
        }
        *ctx->h_hot = 0;
    }
    Carver c;
    const size_t o_pos = c.take<int32_t>(R + 32), o_flag = c.take<uint16_t>(R + 32), o_off = c.take<uint32_t>(R + 40),
                 o_cig = c.take<uint32_t>(NC + 32);
    CU(ctx->d_frec.reserve(c.off + 256));
    char* rb = (char*)ctx->d_frec.p;
    ctx->frec.n_rec = (uint32_t)R;
    ctx->frec.pos = (const int32_t*)(rb + o_pos); ctx->frec.flag = (const uint16_t*)(rb + o_flag);
    ctx->frec.cig_off = (const uint32_t*)(rb + o_off); ctx->frec.cigar = (const uint32_t*)(rb + o_cig);
    Carver pc;
    const size_t p_nop = pc.take<uint16_t>(R + 32), p_f8 = pc.take<uint8_t>(R + 32);
    CU(ctx->d_fpk.reserve(pc.off + 256));
    char* pb = (char*)ctx->d_fpk.p;
    const size_t dwords = unpack_desc_words((uint32_t)R);
    if (ctx->d_unpack.cap < (dwords + 8) * 8) {
        CU(ctx->d_unpack.reserve((dwords + 8) * 8));
        CU(cudaMemsetAsync(ctx->d_unpack.p, 0, ctx->d_unpack.cap, ctx->stream));
        ctx->unpack_epoch = 0;
    }
    uint32_t* ticket = (uint32_t*)ctx->d_unpack.p;                    // fixed place: calls of different sizes share it (it is zero between launches)
    unsigned long long* desc = (unsigned long long*)ctx->d_unpack.p + 2;
    // slabs: cut at multiples of the index stride; a chunk belongs to the slab that holds its last record
    const size_t K = SPL_PACKED_INDEX_STRIDE;
    int want = 1;
    {
        int64_t min_rec = 2000000;
        int max_parts = MAX_FPARTS;
        if (const char* f = std::getenv("SPLISER_SPLIT_MIN_RECORDS")) min_rec = std::max<int64_t>(1, atoll(f));
        if (const char* f = std::getenv("SPLISER_SPLIT_PARTS")) max_parts = std::max(1, std::min(MAX_FPARTS, atoi(f)));
        if (split_ok) want = (int)std::max<int64_t>(1, std::min<int64_t>(max_parts, (int64_t)R / min_rec));
        want = (int)std::min<size_t>((size_t)want, std::max<size_t>(1, R / K));
    }
    ctx->n_fparts = want;
    size_t r0 = 0;
    uint32_t k0 = 0;
    for (int p = 0; p < want; ++p) {
        size_t r1 = (p == want - 1) ? R : (R * (size_t)(p + 1) / (size_t)want) / K * K;
        if (r1 < r0) r1 = r0;
        uint32_t k1 = k0;
        while (k1 < hc.size() && hc[k1].rec_hi <= r1) ++k1;
        ctx->fpart[p].chunk_lo = k0; ctx->fpart[p].chunk_hi = k1;
        k0 = k1;
        const size_t c0 = (size_t)v->cig_index[r0 / K], c1 = r1 == R ? NC : (size_t)v->cig_index[r1 / K];
        if (r1 > r0) {
            CU(cudaMemcpyAsync(rb + o_pos + r0 * 4, v->pos + r0, (r1 - r0) * 4, cudaMemcpyHostToDevice, cs));
            CU(cudaMemcpyAsync(pb + p_nop + r0 * 2, v->n_op + r0, (r1 - r0) * 2, cudaMemcpyHostToDevice, cs));
            CU(cudaMemcpyAsync(pb + p_f8 + r0, v->flag8 + r0, (r1 - r0), cudaMemcpyHostToDevice, cs));
            if (c1 > c0) CU(cudaMemcpyAsync(rb + o_cig + c0 * 4, v->cigar + c0, (c1 - c0) * 4, cudaMemcpyHostToDevice, cs));
            ctx->stats[SPL_STAT_H2D_BYTES] += (double)((r1 - r0) * 7 + (c1 - c0) * 4);
        }
        CU(cudaEventRecord(ctx->fpart[p].ev_up, cs));
        ctx->fpart[p].unpack = nullptr;
        if (r1 > r0) {
            ctx->unpack_epoch = (ctx->unpack_epoch + 1u) & 0x3fffffffu;
            if (ctx->unpack_epoch == 0u) ctx->unpack_epoch = 1u;
            const uint32_t epoch = ctx->unpack_epoch;
            ctx->fpart[p].unpack = [=](cudaStream_t st) {
                launch_unpack_records((const uint16_t*)(pb + p_nop), (const uint8_t*)(pb + p_f8), (uint32_t)r0, (uint32_t)r1, (uint32_t)c0,
                                      (uint32_t*)(rb + o_off), (uint16_t*)(rb + o_flag), desc, ticket, epoch, st);
            };
        }
        r0 = r1;
    }
    ctx->fpart[want - 1].chunk_hi = (uint32_t)hc.size();
    return SPL_OK;
}

// The same for the compact host layout (spl_compact_view, about 9 B per record): every stride of SPL_PACKED_INDEX_STRIDE records
// carries its own anchors (lowest POS, offsets into the 16-bit and the 32-bit operator streams), so a slab is unpacked by one
// kernel (k_unpack_compact, one CTA per stride) as soon as it has arrived, under the copy of the next slab.
int fused_upload_compact(spl_ctx* ctx, const spl_compact_view* v, int32_t n_chrom, bool split_ok) {
    ctx->n_chrom_loaded = n_chrom;
    for (auto& P : ctx->fpart) P.unpack = nullptr;                    // nothing left over from an earlier call
    std::vector<FChunk> hc;
    int64_t aligned = 0;
    for (int32_t k = 0; k < v->n_seg; ++k) {
        if (v->seg_chrom[k] < 0) continue;
        const int64_t a = v->seg_off[k], b = v->seg_off[k + 1];
        aligned += b - a;
        for (int64_t lo = a; lo < b; lo += FC_RECS) {
            FChunk c{};
            c.chrom = v->seg_chrom[k];
            c.rec_lo = (uint32_t)lo;
            c.rec_hi = (uint32_t)std::min<int64_t>(lo + FC_RECS, b);
            hc.push_back(c);
        }
    }
    ctx->n_aligned = aligned;
    ctx->stats[SPL_STAT_N_ALIGNED] = (double)aligned;
    ctx->n_fchunks = (uint32_t)hc.size();
    const size_t R = (size_t)v->n_rec, NC = (size_t)v->n_cigar, K = SPL_PACKED_INDEX_STRIDE;
    const size_t NS = (R + K - 1) / K, N16 = (size_t)v->n16, N32 = (size_t)v->n32, NW = (size_t)v->n_wide;
    cudaStream_t cs = ctx->copy_stream;
    CU(ctx->d_fchunks.reserve((hc.size() + 1) * sizeof(FChunk)));
    ctx->fchunks = (FChunk*)ctx->d_fchunks.p;
    if (!hc.empty()) {
        const size_t bytes = hc.size() * sizeof(FChunk);
        if (ctx->h_fchunks_bytes < bytes) {
            if (ctx->h_fchunks) cudaFreeHost(ctx->h_fchunks);
            ctx->h_fchunks = nullptr; ctx->h_fchunks_bytes = 0;
            CU(cudaHostAlloc(&ctx->h_fchunks, bytes + bytes / 4 + 4096, cudaHostAllocDefault));
            ctx->h_fchunks_bytes = bytes + bytes / 4 + 4096;
        }
        memcpy(ctx->h_fchunks, hc.data(), bytes);
        CU(cudaMemcpyAsync(ctx->fchunks, ctx->h_fchunks, bytes, cudaMemcpyHostToDevice, cs));
        ctx->stats[SPL_STAT_H2D_BYTES] += (double)bytes;
    }
    {
        const uint64_t want = std::max<uint64_t>(1u << 18, (uint64_t)v->n_cigar / 16 + (1u << 16));
        if (ctx->hot_cap < want) {
            CU(ctx->d_hotq.reserve((size_t)want * 16));
            ctx->hot_cap = (uint32_t)std::min<uint64_t>(want, 0xfffffff0u);
        }
        *ctx->h_hot = 0;
    }
    Carver c;
    const size_t o_pos = c.take<int32_t>(R + 32), o_flag = c.take<uint16_t>(R + 32), o_off = c.take<uint32_t>(R + 40),
                 o_cig = c.take<uint32_t>(NC + 32);
    CU(ctx->d_frec.reserve(c.off + 256));
    char* rb = (char*)ctx->d_frec.p;
    ctx->frec.n_rec = (uint32_t)R;
    ctx->frec.pos = (const int32_t*)(rb + o_pos); ctx->frec.flag = (const uint16_t*)(rb + o_flag);
    ctx->frec.cig_off = (const uint32_t*)(rb + o_off); ctx->frec.cigar = (const uint32_t*)(rb + o_cig);
    Carver pc;
    const size_t p_p16 = pc.take<uint16_t>(R + 32), p_f8 = pc.take<uint8_t>(R + 32), p_n8 = pc.take<uint8_t>(R + 32),
                 p_c16 = pc.take<uint16_t>(N16 + 32), p_c32 = pc.take<uint32_t>(N32 + 32), p_base = pc.take<int32_t>(NS + 8),
                 p_i16 = pc.take<uint32_t>(NS + 8), p_i32 = pc.take<uint32_t>(NS + 8), p_wide = pc.take<int32_t>(NW * K + 32);
    CU(ctx->d_cpk.reserve(pc.off + 256));
    char* pb = (char*)ctx->d_cpk.p;
    if (R > 0) {
        // the per-stride anchors (12 B per 1024 records) and the wide strides' positions go first
        CU(cudaMemcpyAsync(pb + p_base, v->pos_base, NS * 4, cudaMemcpyHostToDevice, cs));
        CU(cudaMemcpyAsync(pb + p_i16, v->idx16, (NS + 1) * 4, cudaMemcpyHostToDevice, cs));
        CU(cudaMemcpyAsync(pb + p_i32, v->idx32, (NS + 1) * 4, cudaMemcpyHostToDevice, cs));
        if (NW) CU(cudaMemcpyAsync(pb + p_wide, v->pos_wide, NW * K * 4, cudaMemcpyHostToDevice, cs));
        ctx->stats[SPL_STAT_H2D_BYTES] += (double)(NS * 12 + 8 + NW * K * 4);
    }
    int want = 1;
    {
        int64_t min_rec = 2000000;
        int max_parts = MAX_FPARTS;
        if (const char* f = std::getenv("SPLISER_SPLIT_MIN_RECORDS")) min_rec = std::max<int64_t>(1, atoll(f));
        if (const char* f = std::getenv("SPLISER_SPLIT_PARTS")) max_parts = std::max(1, std::min(MAX_FPARTS, atoi(f)));
        if (split_ok) want = (int)std::max<int64_t>(1, std::min<int64_t>(max_parts, (int64_t)R / min_rec));
        want = (int)std::min<size_t>((size_t)want, std::max<size_t>(1, R / K));
    }
    ctx->n_fparts = want;
    size_t r0 = 0;
    uint32_t k0 = 0;
    for (int p = 0; p < want; ++p) {
        // slabs of decreasing size (cumulative share 1 - (1 - (p + 1) / n)^2): what stays exposed after the last copy is the unpack
        // and the counting of the last slab, so that one is small
        const double rest = 1.0 - (double)(p + 1) / (double)want;
        size_t r1 = (p == want - 1) ? R : (size_t)((double)R * (1.0 - rest * rest)) / K * K;
        if (r1 < r0) r1 = r0;
        uint32_t k1 = k0;
        while (k1 < hc.size() && hc[k1].rec_hi <= r1) ++k1;
        ctx->fpart[p].chunk_lo = k0; ctx->fpart[p].chunk_hi = k1;
        k0 = k1;
        if (r1 > r0) {
            const size_t s0 = r0 / K, s1 = (r1 + K - 1) / K;
            const size_t a16 = v->idx16[s0], b16 = v->idx16[s1], a32 = v->idx32[s0], b32 = v->idx32[s1];
            CU(cudaMemcpyAsync(pb + p_p16 + r0 * 2, v->pos16 + r0, (r1 - r0) * 2, cudaMemcpyHostToDevice, cs));
            CU(cudaMemcpyAsync(pb + p_f8 + r0, v->flag8 + r0, (r1 - r0), cudaMemcpyHostToDevice, cs));
            CU(cudaMemcpyAsync(pb + p_n8 + r0, v->n_op8 + r0, (r1 - r0), cudaMemcpyHostToDevice, cs));
            if (b16 > a16) CU(cudaMemcpyAsync(pb + p_c16 + a16 * 2, v->cigar16 + a16, (b16 - a16) * 2, cudaMemcpyHostToDevice, cs));
            if (b32 > a32) CU(cudaMemcpyAsync(pb + p_c32 + a32 * 4, v->cigar32 + a32, (b32 - a32) * 4, cudaMemcpyHostToDevice, cs));
            ctx->stats[SPL_STAT_H2D_BYTES] += (double)((r1 - r0) * 4 + (b16 - a16) * 2 + (b32 - a32) * 4);
        }
        CU(cudaEventRecord(ctx->fpart[p].ev_up, cs));
        ctx->fpart[p].unpack = nullptr;
        if (r1 > r0) {
            ctx->fpart[p].unpack = [=](cudaStream_t st) {
                launch_unpack_compact((const uint16_t*)(pb + p_p16), (const uint8_t*)(pb + p_f8), (const uint8_t*)(pb + p_n8),
                                      (const uint16_t*)(pb + p_c16), (const uint32_t*)(pb + p_c32), (const int32_t*)(pb + p_base),
                                      (const int32_t*)(pb + p_wide), (const uint32_t*)(pb + p_i16), (const uint32_t*)(pb + p_i32),
                                      (uint32_t)r0, (uint32_t)r1, (int32_t*)(rb + o_pos), (uint16_t*)(rb + o_flag), (uint32_t*)(rb + o_off),
                                      (uint32_t*)(rb + o_cig), ctx->cnt.work + 25, st);
            };
        }
        r0 = r1;
    }
    ctx->fpart[want - 1].chunk_hi = (uint32_t)hc.size();
    return SPL_OK;
}

// fused variant: one pass = counters zeroed, one counting kernel per slab (as soon as the slab has arrived), finalize
int fused_count_pass(spl_ctx* ctx, cudaEvent_t* ev /* 5 or NULL */) {
    if (ev) CU(cudaEventRecord(ev[0], ctx->stream));
    if (ctx->g.n_sites > 0) CU(cudaMemsetAsync(ctx->d_cnt.p, 0, ctx->cnt_bytes, ctx->stream));
    if (ev) CU(cudaEventRecord(ev[1], ctx->stream));
    uint32_t* hot_n = ctx->cnt.work + 24;
    for (int p = 0; p < ctx->n_fparts; ++p) {
        FPart& P = ctx->fpart[p];
        CU(cudaStreamWaitEvent(ctx->stream, P.ev_up, 0));
        if (P.unpack) { if (ctx->g.n_sites > 0) P.unpack(ctx->stream); P.unpack = nullptr; }   // once: a repeated pass finds the arrays in place (no sites: nothing reads them)
        launch_chunk_bounds(ctx->fchunks, P.chunk_lo, P.chunk_hi, ctx->frec.cig_off, ctx->g, ctx->stream);
        launch_count_fused(ctx->frec, ctx->fchunks, P.chunk_lo, P.chunk_hi, ctx->g, ctx->cnt, ctx->cnt.work + 8 + p, ctx->flags,
                           (uint4*)ctx->d_hotq.p, hot_n, ctx->hot_cap, ctx->stream);
    }
    if (ev) CU(cudaEventRecord(ev[2], ctx->stream));
    if (ctx->n_fchunks) launch_hot_items(ctx->frec, ctx->g, ctx->cnt, ctx->flags, (const uint4*)ctx->d_hotq.p, hot_n, ctx->hot_cap, ctx->stream);
    if (ctx->g.n_sites > 0) CU(cudaMemcpyAsync(ctx->h_hot, hot_n, 8, cudaMemcpyDeviceToHost, ctx->stream));   // + the unpack kernels' verdict
    if (ev) CU(cudaEventRecord(ev[3], ctx->stream));
    launch_finalize(ctx->g, ctx->cnt, ctx->out, ctx->flags, ctx->stream);
    if (ev) CU(cudaEventRecord(ev[4], ctx->stream));
    CU(cudaGetLastError());
    return SPL_OK;
}

// one counting pass over the resident SoA; events (if given) bracket the three kernel groups
int count_pass(spl_ctx* ctx, cudaEvent_t* ev /* 5 or NULL */) {
    if (ctx->loaded_variant == SPL_VARIANT_FUSED) return fused_count_pass(ctx, ev);
    if (ev) CU(cudaEventRecord(ev[0], ctx->stream));
    if (ctx->g.n_sites > 0) CU(cudaMemsetAsync(ctx->d_cnt.p, 0, ctx->cnt_bytes, ctx->stream));
    if (ev) CU(cudaEventRecord(ev[1], ctx->stream));
    for (int p = 0; p < ctx->n_parts; ++p) {
        if (p && ctx->g.n_sites > 0) CU(cudaMemsetAsync(ctx->cnt.work, 0, 32, ctx->stream));      // tile counter of the previous part
        launch_beta1(ctx->part[p].bins, ctx->g, ctx->cnt, ctx->stream);
    }
    if (ev) CU(cudaEventRecord(ev[2], ctx->stream));
    for (int p = 0; p < ctx->n_parts; ++p) {
        launch_junctions(ctx->part[p].soa, ctx->part[p].jg, ctx->g, ctx->cnt, ctx->flags, ctx->stream);
    }
    if (ev) CU(cudaEventRecord(ev[3], ctx->stream));
    launch_finalize(ctx->g, ctx->cnt, ctx->out, ctx->flags, ctx->stream);
    if (ev) CU(cudaEventRecord(ev[4], ctx->stream));
    CU(cudaGetLastError());
    return SPL_OK;
}

// after a stream sync that follows a fused pass: did the hot queue hold every item?  If not, it is grown and the caller
// repeats the pass (counters are re-zeroed by the pass itself).
int hot_queue_overflow(spl_ctx* ctx, bool* again) {
    *again = false;
    if (ctx->loaded_variant != SPL_VARIANT_FUSED || ctx->g.n_sites <= 0) return SPL_OK;
    const uint32_t n = *ctx->h_hot;
    ctx->stats[SPL_STAT_N_HOT_ITEMS] = (double)n;
    if (ctx->h_hot[1]) { ctx->h_hot[1] = 0; return ctx->fail(SPL_ERR_ARG, "compact view: the operator counts of a stride disagree with its index"); }
    if (n <= ctx->hot_cap) return SPL_OK;
    const uint64_t want = (uint64_t)n + (n >> 3) + 1024;
    if (want >= 0xfffffff0ull) return ctx->fail(SPL_ERR_RANGE, "more than 2^32 hot junction items in one call");
    CU(ctx->d_hotq.reserve((size_t)want * 16));
    ctx->hot_cap = (uint32_t)want;
    *again = true;
    return SPL_OK;
}

int fetch(spl_ctx* ctx, spl_result** out_r) {
    const bool dev = ctx->graph_on_device;
    const SiteGraph& h = ctx->hg;
    const size_t S = dev ? ctx->gcnt.S : (size_t)h.n_sites, E = dev ? ctx->gcnt.E : h.pc_pos.size(), Cn = dev ? ctx->gcnt.C : h.cp_pos.size();
    const bool pre = dev && ctx->pending && (size_t)ctx->pending->n == S && (size_t)ctx->pending->E == E && (size_t)ctx->pending->C == Cn;
    spl_result* r = pre ? ctx->pending : result_alloc(S, E, Cn, true);
    if (pre) ctx->pending = nullptr;
    if (!r) return ctx->fail(SPL_ERR_NOMEM, "cannot allocate the result (%zu sites)", S);
    std::unique_ptr<spl_result, void (*)(spl_result*)> guard(r, spl_result_free);
    cudaStream_t st = ctx->stream;
    double bytes = 0;
    if (S) {
        CU(cudaMemcpyAsync(r->alpha, ctx->out.alpha, S * 8, cudaMemcpyDeviceToHost, st));
        CU(cudaMemcpyAsync(r->beta1, ctx->out.beta1, S * 8, cudaMemcpyDeviceToHost, st));
        CU(cudaMemcpyAsync(r->beta2s, ctx->out.beta2s, S * 8, cudaMemcpyDeviceToHost, st));
        CU(cudaMemcpyAsync(r->beta2c, ctx->out.beta2c, S * 8, cudaMemcpyDeviceToHost, st));
        CU(cudaMemcpyAsync(r->beta2w, ctx->out.beta2w, S * 8, cudaMemcpyDeviceToHost, st));
        CU(cudaMemcpyAsync(r->sse, ctx->out.sse, S * 8, cudaMemcpyDeviceToHost, st));
        if (E) CU(cudaMemcpyAsync(r->pc_cnt, ctx->out.pc_cnt, E * 8, cudaMemcpyDeviceToHost, st));
        bytes += (double)(S * 48 + E * 8);
        if (pre) {                                                     // structure arrays were sent during the load
            CU(cudaStreamSynchronize(ctx->stream2));
        } else if (dev) {                                              // the structure lives on the device too
            const GraphDev& d = ctx->gdev;
            CU(cudaMemcpyAsync(r->chrom, d.site_chrom, S * 4, cudaMemcpyDeviceToHost, st));
            CU(cudaMemcpyAsync(r->pos, d.site_pos, S * 4, cudaMemcpyDeviceToHost, st));
            CU(cudaMemcpyAsync(r->strand, d.site_strand, S, cudaMemcpyDeviceToHost, st));
            CU(cudaMemcpyAsync(r->first_line, d.first_line, S * 8, cudaMemcpyDeviceToHost, st));
            CU(cudaMemcpyAsync(r->pc_off, d.pt_off64, (S + 1) * 8, cudaMemcpyDeviceToHost, st));
            CU(cudaMemcpyAsync(r->cp_off, d.cp_off64, (S + 1) * 8, cudaMemcpyDeviceToHost, st));
            if (E) CU(cudaMemcpyAsync(r->pc_pos, d.pc_pos, E * 4, cudaMemcpyDeviceToHost, st));
            if (Cn) CU(cudaMemcpyAsync(r->cp_pos, d.cp_pos, Cn * 4, cudaMemcpyDeviceToHost, st));
            bytes += (double)(S * 33 + 16 + E * 4 + Cn * 4);
        } else {
            result_from_host_graph(r, h);
        }
        CU(cudaStreamSynchronize(st));
    }
    ctx->stats[SPL_STAT_D2H_BYTES] += bytes;
    *out_r = guard.release();
    return SPL_OK;
}

void reset_stats(spl_ctx* ctx) { std::fill(ctx->stats, ctx->stats + SPL_NSTATS, 0.0); }

// an entry point is about to return an error: nothing may still be reading the caller's (borrowed) arrays
int drain_on_error(spl_ctx* ctx, int rc) {
    if (rc && ctx->stream) {
        cudaStreamSynchronize(ctx->copy_stream);
        cudaStreamSynchronize(ctx->stream2);
        cudaStreamSynchronize(ctx->stream);
        cudaGetLastError();
    }
    return rc;
}

// CUDA-event time of the load-time kernels; call after a stream sync that follows the load
void collect_expand_ms(spl_ctx* ctx) {
    for (int p = 0; p < MAX_PARTS; ++p) {
        Part& P = ctx->part[p];
        if (!P.timed) continue;
        P.timed = false;
        float ms = 0;
        if (cudaEventElapsedTime(&ms, P.ev_e0, P.ev_e1) == cudaSuccess) ctx->stats[SPL_STAT_MS_EXPAND] += ms;
        else cudaGetLastError();
    }
}

// Everything that depends on (sample x site table): site windows of the chunks / tiles, and per distinct junction the site
// lookups, hot flags, pair sites and exception work lists; then one packed record per hot complex instance (its count is
// only known now, hence the one read-back).
int prepare_parts(spl_ctx* ctx) {
    for (int p = 0; p < ctx->n_parts; ++p) {
        Part& P = ctx->part[p];
        launch_tile_hints(P.bins, ctx->g, ctx->stream);
        P.jg.cx_pack = nullptr;
        launch_junction_prepare(P.jg, ctx->g, ctx->flags, ctx->stream);
        P.h_tot[20] = P.h_tot[21] = 0;
        if (P.jg.D && P.jg.n_complex && ctx->g.n_sites > 0)
            CU(cudaMemcpyAsync(P.h_tot + 20, P.jg.prep + 4, 8, cudaMemcpyDeviceToHost, ctx->stream));
    }
    CU(cudaGetLastError());
    CU(cudaStreamSynchronize(ctx->stream));
    for (int p = 0; p < ctx->n_parts; ++p) {
        Part& P = ctx->part[p];
        const unsigned long long w = (unsigned long long)P.h_tot[20] | ((unsigned long long)P.h_tot[21] << 32);
        const size_t n_flat = (size_t)(w & ((1ull << 40) - 1ull));
        if (!n_flat) continue;
        CU(P.d_cxpack.reserve(n_flat * 24 * sizeof(uint32_t) + 256));
        P.jg.cx_pack = (uint32_t*)P.d_cxpack.p;
        launch_junction_pack(P.soa, P.jg, ctx->stream);
    }
    CU(cudaGetLastError());
    return SPL_OK;
}

// DevGraph view of a device-built graph
void adopt_device_graph(spl_ctx* ctx) {
    const GraphDev& d = ctx->gdev;
    DevGraph& g = ctx->g;
    const size_t S = ctx->gcnt.S;
    g.n_chrom = ctx->n_chrom_loaded; g.n_sites = (int32_t)S; g.n_edges = (int32_t)ctx->gcnt.E;
    owned_range(ctx, (int64_t)S, g.own_lo, g.own_hi);
    g.pt_is_pc = 1;
    g.cs_off = d.cs_off; g.site_pos = d.site_pos; g.site_cls = d.site_cls; g.site_hot = d.site_hot;
    g.sb_base = d.sb_base; g.sb_off = d.sb_off;
    g.pt_off = d.pt_off; g.pt_site = d.pt_site; g.pc_off = d.pt_off; g.pc_pos = d.pc_pos;     // clean regime: one PartnerCounts key per partner
    g.cp_off = d.cp_off; g.cp_pos = d.cp_pos; g.rp_off = d.rp_off; g.rp_site = d.rp_site;
    g.inc_off = d.inc_off; g.inc_line = d.inc_line;
    g.einc_beg = d.einc_beg; g.einc_end = d.einc_end; g.einc_line = d.einc_line;
    g.j_score = d.j_score;
}

int load_common(spl_ctx* ctx, const spl_records_view* rec, int32_t n_chrom, int64_t n_junc, const int32_t* j_chrom,
                const int32_t* j_left, const int32_t* j_right, const int64_t* j_score, const uint8_t* j_strand, uint32_t flags,
                bool split_ok, const spl_packed_view* packed = nullptr, const spl_compact_view* compact = nullptr) {
    ctx->loaded = false;
    if (ctx->pending) { cudaStreamSynchronize(ctx->stream2); spl_result_free(ctx->pending); ctx->pending = nullptr; }
    int rc = check_view(ctx, rec, n_chrom);
    if (rc) return rc;
    if (n_junc < 0) return ctx->fail(SPL_ERR_ARG, "negative size");
    if (n_junc > 0 && (!j_chrom || !j_left || !j_right || !j_strand)) return ctx->fail(SPL_ERR_ARG, "null junction array");
    if (n_junc > 0 && !j_score) return ctx->fail(SPL_ERR_ARG, "NULL j_score");
    CU(cudaSetDevice(ctx->device));
    reset_stats(ctx);
    flags &= 0xfu;
#ifdef SPL_DEBUG_HOOKS
    if (const char* dbg = std::getenv("SPLISER_DEBUG_SKIP_EXC"))
        if (dbg[0] == '1') flags |= FLAG_DEBUG_SKIP_EXC;
#endif
    ctx->flags = flags;
    const bool fused = ctx->variant == SPL_VARIANT_FUSED;
    ctx->loaded_variant = ctx->variant;
    const bool stranded = (flags & SPL_FLAG_STRANDED) != 0;
    const double tg0 = now_ms();
    // which regime?  (SURVEY 8(a): a '?' strand in a stranded run or a degenerate row makes the outcome depend on
    // the reference's bisection path -> sequential host emulation; everything else is sort/unique on the device)
    bool clean = n_junc > 0;
    int32_t max_pos = 1;
    for (int64_t i = 0; i < n_junc; ++i) {
        if (j_chrom[i] < 0 || j_chrom[i] >= n_chrom) return ctx->fail(SPL_ERR_ARG, "junction chromosome index out of range");
        const uint8_t st = j_strand[i];
        if ((stranded && st != '+' && st != '-') || j_left[i] == j_right[i] || j_left[i] < 0 || j_right[i] < 0) clean = false;
        max_pos = std::max(max_pos, std::max(j_left[i], j_right[i]));
    }
    if (const char* f = std::getenv("SPLISER_FORCE_EMULATION")) if (f[0] == '1') clean = false;
    if (const char* f = std::getenv("SPLISER_HOST_GRAPH")) if (f[0] == '1') clean = false;
    if (clean && !graph_build_fits(n_junc, n_chrom, max_pos)) clean = false;
    ctx->res_clean = clean; ctx->res_n_junc = n_junc; ctx->res_n_chrom = n_chrom; ctx->res_max_pos = max_pos; ctx->res_stranded = stranded;

    // the records start travelling first; the graph is built meanwhile (device: second stream, host: a thread)
    if (clean) {
        std::string e;
        if (!graph_build_device(ctx->gbm, j_chrom, j_left, j_right, j_strand, j_score, n_junc, n_chrom, max_pos, stranded, ctx->stream2,
                                0, ctx->gdev, ctx->gcnt, e))
            return ctx->fail(SPL_ERR_CUDA, "%s", e.c_str());
    }
    // A big host upload is cut into up to three parts of decreasing size (55 / 30 / 15 % of the records, at chunk
    // granularity, inside a chromosome if need be): the expansion of each part runs while the next one is still on the
    // wire, and only the last, smallest part's expansion stays exposed.
    int64_t cuts[MAX_PARTS + 1] = {0, rec->n_rec, rec->n_rec, rec->n_rec};
    ctx->n_parts = 1;
    {
        int64_t min_rec = 4000000;
        int want_parts = MAX_PARTS;
        if (const char* f = std::getenv("SPLISER_SPLIT_MIN_RECORDS")) min_rec = atoll(f);
        if (const char* f = std::getenv("SPLISER_SPLIT_PARTS")) want_parts = std::max(1, std::min(MAX_PARTS, atoi(f)));
        if (split_ok && !ctx->rec_on_device && want_parts > 1 && rec->n_rec >= min_rec && rec->n_rec >= 4 * (int64_t)CHUNK_READS) {
            const double frac2[] = {0.80}, frac3[] = {0.55, 0.85};
            const double* fr = want_parts == 2 ? frac2 : frac3;
            ctx->n_parts = want_parts;
            for (int p = 1; p < want_parts; ++p) {
                int64_t c = (int64_t)(fr[p - 1] * (double)rec->n_rec) / CHUNK_READS * CHUNK_READS;
                cuts[p] = std::max(cuts[p - 1] + CHUNK_READS, std::min(c, rec->n_rec - CHUNK_READS));
            }
            cuts[want_parts] = rec->n_rec;
        }
    }
    ctx->n_aligned = 0;
    cudaEvent_t dbg[6] = {nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};
    const bool dbg_on = std::getenv("SPLISER_TIMING") != nullptr;
    if (dbg_on) { for (auto& e : dbg) cudaEventCreate(&e); cudaEventRecord(dbg[0], ctx->copy_stream); }
    if (fused) {
        ctx->n_parts = 0;
        rc = compact ? fused_upload_compact(ctx, compact, n_chrom, split_ok)
                     : packed ? fused_upload_packed(ctx, packed, n_chrom, split_ok) : fused_upload(ctx, rec, n_chrom, split_ok);
        if (rc) return rc;
    }
    for (int p = 0; p < ctx->n_parts; ++p) {
        rc = upload_records(ctx, ctx->part[p], rec, cuts[p], cuts[p + 1], n_chrom);
        if (rc) return rc;
        if (dbg_on && p == 0) cudaEventRecord(dbg[1], ctx->copy_stream);
    }
    if (dbg_on) cudaEventRecord(dbg[2], ctx->copy_stream);
    const bool timing = std::getenv("SPLISER_TIMING") != nullptr;
    if (timing) fprintf(stderr, "[load] +%.2f ms uploads queued (%d part(s))\n", now_ms() - tg0, ctx->n_parts);
    auto expand_all = [&]() -> int {
        for (int p = 0; p < ctx->n_parts; ++p) {
            if (timing) fprintf(stderr, "[load] +%.2f ms expand part %d starts\n", now_ms() - tg0, p);
            if (dbg_on && p == 0) { cudaStreamWaitEvent(ctx->stream, ctx->part[0].ev_up, 0); cudaEventRecord(dbg[3], ctx->stream); }
            const int r = expand_records(ctx, ctx->part[p], rec, cuts[p], cuts[p + 1], flags);
            if (r) return r;
            if (dbg_on && p == 0) cudaEventRecord(dbg[4], ctx->stream);
            if (timing) fprintf(stderr, "[load] +%.2f ms expand part %d done\n", now_ms() - tg0, p);
            if (dbg_on && p == ctx->n_parts - 1) {
                cudaDeviceSynchronize();
                float a = 0, b = 0, c = 0, d = 0;
                cudaEventElapsedTime(&a, dbg[0], dbg[1]); cudaEventElapsedTime(&b, dbg[0], dbg[2]);
                cudaEventElapsedTime(&c, dbg[0], dbg[3]); cudaEventElapsedTime(&d, dbg[0], dbg[4]);
                fprintf(stderr, "[load] device timeline: copies A done %.2f, copies B done %.2f, kernels A start %.2f, kernels A end %.2f ms\n", a, b, c, d);
                for (auto& e : dbg) cudaEventDestroy(e);
            }
        }
        return SPL_OK;
    };
    if (clean) {
        std::string e;
        if (!graph_build_device(ctx->gbm, j_chrom, j_left, j_right, j_strand, j_score, n_junc, n_chrom, max_pos, stranded, ctx->stream2,
                                1, ctx->gdev, ctx->gcnt, e))
            return ctx->fail(SPL_ERR_CUDA, "%s", e.c_str());
        CU(cudaEventRecord(ctx->ev_graph, ctx->stream2));
        ctx->graph_on_device = true;
        if (split_ok) {
            // one-shot call: the site table / CSR structure goes back to the host now, under the record upload (PCIe is
            // full duplex), so that the final fetch only moves the per-site results
            const GraphDev& d = ctx->gdev;
            const size_t S = ctx->gcnt.S, E = ctx->gcnt.E, Cn = ctx->gcnt.C;
            spl_result* r = result_alloc(S, E, Cn, true);
            if (r) {
                cudaStream_t s2 = ctx->stream2;
                ctx->pending = r;
                CU(cudaMemcpyAsync(r->chrom, d.site_chrom, S * 4, cudaMemcpyDeviceToHost, s2));
                CU(cudaMemcpyAsync(r->pos, d.site_pos, S * 4, cudaMemcpyDeviceToHost, s2));
                CU(cudaMemcpyAsync(r->strand, d.site_strand, S, cudaMemcpyDeviceToHost, s2));
                CU(cudaMemcpyAsync(r->first_line, d.first_line, S * 8, cudaMemcpyDeviceToHost, s2));
                CU(cudaMemcpyAsync(r->pc_off, d.pt_off64, (S + 1) * 8, cudaMemcpyDeviceToHost, s2));
                CU(cudaMemcpyAsync(r->cp_off, d.cp_off64, (S + 1) * 8, cudaMemcpyDeviceToHost, s2));
                if (E) CU(cudaMemcpyAsync(r->pc_pos, d.pc_pos, E * 4, cudaMemcpyDeviceToHost, s2));
                if (Cn) CU(cudaMemcpyAsync(r->cp_pos, d.cp_pos, Cn * 4, cudaMemcpyDeviceToHost, s2));
                ctx->stats[SPL_STAT_D2H_BYTES] += (double)(S * 33 + 16 + E * 4 + Cn * 4);
            }
        }
        ctx->stats[SPL_STAT_H2D_BYTES] += ctx->gcnt.h2d_bytes;
        adopt_device_graph(ctx);
        rc = alloc_counters_outputs(ctx, ctx->gcnt.S, ctx->gcnt.E);
        if (rc) return rc;
        ctx->stats[SPL_STAT_MS_GRAPH] = now_ms() - tg0;
        rc = expand_all();
        ctx->stats[SPL_STAT_MS_UPLOAD] = now_ms() - tg0;
        if (rc) return rc;
        CU(cudaStreamWaitEvent(ctx->stream, ctx->ev_graph, 0));
        ctx->stats[SPL_STAT_N_SITES] = (double)ctx->gcnt.S;
        ctx->stats[SPL_STAT_N_EDGES] = (double)ctx->gcnt.E;
    } else {
        std::string e;
        double graph_ms = 0;
        std::thread builder([&]() {
            e = build_site_graph(n_chrom, n_junc, j_chrom, j_left, j_right, j_strand, stranded, ctx->hg);
            graph_ms = now_ms() - tg0;
        });
        rc = expand_all();
        ctx->stats[SPL_STAT_MS_UPLOAD] = now_ms() - tg0;
        builder.join();
        if (rc) return rc;
        if (!e.empty()) return ctx->fail(SPL_ERR_ARG, "%s", e.c_str());
        const double tu0 = now_ms();
        rc = upload_graph(ctx, j_score, n_junc);
        if (rc) return rc;
        ctx->stats[SPL_STAT_MS_GRAPH] = graph_ms + (now_ms() - tu0);
        ctx->stats[SPL_STAT_N_SITES] = (double)ctx->hg.n_sites;
        ctx->stats[SPL_STAT_N_EDGES] = (double)ctx->hg.pc_pos.size();
    }
    if (!fused) { const int prc = prepare_parts(ctx); if (prc) return prc; }
    CU(cudaGetLastError());
    ctx->stats[SPL_STAT_LAUNCHES] = fused ? (double)(2 * ctx->n_fparts + 2) : (double)kernel_launch_count_per_pass();
    ctx->stats[SPL_STAT_GRAPH_DEVICE] = ctx->graph_on_device ? 1.0 : 0.0;
    ctx->stats[SPL_STAT_N_PARTS] = (double)(fused ? ctx->n_fparts : ctx->n_parts);
    ctx->loaded = true;
    return SPL_OK;
}

// BAM file -> record arrays on the device.  SPL_OK: ctx->dev_rec / `cnt` are filled and `view` describes them
// (array pointers NULL, ctx->rec_on_device must be set by the caller around the load).  *fallback = true: use the host reader.
// want_xs: ctx->dev_rec.xs receives the XS strand of every record as well.  header_order != NULL: chrom_names is ignored, every
// record keeps its header reference index (no reference is dropped) and *header_order receives the reference names.
int ingest_bam_device(spl_ctx* ctx, const char* path, int32_t n_chrom, const char* const* chrom_names, BamGpuCounts& cnt,
                      spl_records_view& view, bool* fallback, bool want_xs = false, std::vector<std::string>* header_order = nullptr,
                      const TagTableHost* tags = nullptr) {
    *fallback = false;
    if (const char* f = std::getenv("SPLISER_HOST_BAM")) if (f[0] == '1') { *fallback = true; return SPL_OK; }
    const int fd = open(path, O_RDONLY);
    if (fd < 0) return ctx->fail(SPL_ERR_IO, "cannot open BAM file %s", path);
    struct stat st;
    if (fstat(fd, &st) != 0 || st.st_size < 28) { close(fd); return ctx->fail(SPL_ERR_IO, "BAM file too small: %s", path); }
    const size_t fsz = (size_t)st.st_size;
    if (ctx->h_file_bytes < fsz) {
        if (ctx->h_file) cudaFreeHost(ctx->h_file);
        ctx->h_file = nullptr; ctx->h_file_bytes = 0;
        if (cudaHostAlloc(&ctx->h_file, fsz + fsz / 8 + 4096, cudaHostAllocDefault) != cudaSuccess) {
            cudaGetLastError(); close(fd);
            *fallback = true;                                           // not enough page-locked memory: the host reader streams
            return SPL_OK;
        }
        ctx->h_file_bytes = fsz + fsz / 8 + 4096;
    }
    // page cache -> page-locked image in slabs (a few threads per slab); a slab starts travelling to the device as soon as it is
    // in place, under the read of the next one; the host walks the BGZF member headers after the last slab
    bool uploaded = ctx->bgm.comp.reserve(fsz + 64) == cudaSuccess;
    if (!uploaded) cudaGetLastError();
    {
        const size_t SLAB = (size_t)64 << 20;
        const int nt = (int)std::min<size_t>(8, std::max<size_t>(1, std::min(fsz, SLAB) >> 23));
        std::atomic<bool> bad(false);
        for (size_t s0 = 0; s0 < fsz; s0 += SLAB) {
            const size_t s1 = std::min(fsz, s0 + SLAB), len = s1 - s0;
            auto rd = [&](int t) {
                size_t lo = s0 + len * (size_t)t / (size_t)nt;
                const size_t hi = s0 + len * (size_t)(t + 1) / (size_t)nt;
                while (lo < hi) {
                    const ssize_t k = pread(fd, (char*)ctx->h_file + lo, hi - lo, (off_t)lo);
                    if (k <= 0) { bad = true; return; }
                    lo += (size_t)k;
                }
            };
            std::vector<std::thread> pool;
            for (int t = 1; t < nt; ++t) pool.emplace_back(rd, t);
            rd(0);
            for (auto& t : pool) t.join();
            if (bad) break;
            if (uploaded && cudaMemcpyAsync((char*)ctx->bgm.comp.p + s0, (const char*)ctx->h_file + s0, len, cudaMemcpyHostToDevice, ctx->stream) != cudaSuccess) {
                close(fd);
                cudaStreamSynchronize(ctx->stream);
                return ctx->fail(SPL_ERR_CUDA, "copy of the BAM image failed: %s", cudaGetErrorString(cudaGetLastError()));
            }
        }
        close(fd);
        if (bad) { cudaStreamSynchronize(ctx->stream); return ctx->fail(SPL_ERR_IO, "read error on %s", path); }
    }
    std::vector<BgzfMember> members;
    std::vector<int32_t> refmap;
    uint64_t total_u = 0, first_record = 0;
    int32_t n_ref = 0;
    std::string e = bam_scan((const uint8_t*)ctx->h_file, fsz, n_chrom, chrom_names, members, total_u, first_record, n_ref, refmap,
                             header_order);
    if (!e.empty()) { cudaStreamSynchronize(ctx->stream); return ctx->fail(SPL_ERR_IO, "%s", e.c_str()); }
    if (header_order) for (int32_t r = 0; r < n_ref; ++r) refmap[(size_t)r] = r;
    TagTableView d_tags;                                               // the tag group table in device memory
    if (tags) {
        const size_t b_slot = tags->slot.size() * 4, b_off = tags->off.size() * 4, b_grp = tags->group.size() * 4;
        const size_t o_off = (b_slot + 255) & ~(size_t)255, o_grp = (o_off + b_off + 255) & ~(size_t)255, o_blob = (o_grp + b_grp + 255) & ~(size_t)255;
        if (ctx->bgm.tags.reserve(o_blob + tags->blob.size() + 16) != cudaSuccess) {
            cudaGetLastError(); cudaStreamSynchronize(ctx->stream);
            return ctx->fail(SPL_ERR_NOMEM, "not enough device memory for the tag group table");
        }
        char* tb = (char*)ctx->bgm.tags.p;
        CU(cudaMemcpyAsync(tb, tags->slot.data(), b_slot, cudaMemcpyHostToDevice, ctx->stream));
        CU(cudaMemcpyAsync(tb + o_off, tags->off.data(), b_off, cudaMemcpyHostToDevice, ctx->stream));
        CU(cudaMemcpyAsync(tb + o_grp, tags->group.data(), b_grp, cudaMemcpyHostToDevice, ctx->stream));
        CU(cudaMemcpyAsync(tb + o_blob, tags->blob.data(), tags->blob.size(), cudaMemcpyHostToDevice, ctx->stream));
        d_tags = tags->view();
        d_tags.slot = (const uint32_t*)tb; d_tags.off = (const uint32_t*)(tb + o_off);
        d_tags.group = (const int32_t*)(tb + o_grp); d_tags.blob = (const uint8_t*)(tb + o_blob);
    }
    const int rc = bam_gpu_ingest(ctx->bgm, (const uint8_t*)ctx->h_file, fsz, members, total_u, first_record, n_ref, refmap, ctx->stream,
                                  uploaded, want_xs, ctx->rf, tags ? &d_tags : nullptr, ctx->dev_rec, cnt, e);
    if (rc != BAMGPU_OK) cudaStreamSynchronize(ctx->stream);           // the pinned image may be re-used by the fallback / next call
    if (rc == BAMGPU_ERROR) return ctx->fail(SPL_ERR_CUDA, "%s", e.c_str());
    if (rc == BAMGPU_FALLBACK) { *fallback = true; return SPL_OK; }
    ctx->rf_counts[0] = (int64_t)cnt.n_rec; ctx->rf_counts[1] = (int64_t)cnt.n_dropped;
    view = spl_records_view{};
    view.n_rec = (int64_t)cnt.n_rec; view.n_cigar = (int64_t)cnt.n_cigar;
    view.n_seg = (int32_t)cnt.seg_chrom.size();
    view.seg_chrom = cnt.seg_chrom.data(); view.seg_off = cnt.seg_off.data();
    return SPL_OK;
}

// The host reader under the context's read filter: the fallback of every ingest above
std::string read_bam_ctx(spl_ctx* ctx, const char* path, int32_t n_chrom, const char* const* chrom_names, BamRecords& recs, bool want_xs = false,
                         std::vector<std::string>* header_order = nullptr, const TagTableView* tags = nullptr) {
    std::string e = read_bam(path, n_chrom, chrom_names, ctx->n_threads, recs, want_xs, header_order, ctx->rf, tags);
    if (e.empty()) { ctx->rf_counts[0] = (int64_t)recs.pos.size(); ctx->rf_counts[1] = recs.n_filtered; }
    return e;
}

// Host record arrays carry no MAPQ: a record-array entry point refuses to run while a read filter is set, unless its records
// came from an ingest that applied it (the path entry points and the resident samples call these routines themselves)
int refuse_records(spl_ctx* ctx, const char* fn) {
    if (ctx->from_bam || read_filter_none(ctx->rf)) return SPL_OK;
    return ctx->fail(SPL_ERR_ARG, "%s: host record arrays carry no MAPQ, so the context's read filter cannot be applied; "
                     "remove it (spl_set_read_filter(ctx, NULL)) or pass the BAM path", fn);
}

// marks the records of one call as ingested under the context's filter
struct FromBam {
    spl_ctx* ctx;
    bool saved;
    explicit FromBam(spl_ctx* c) : ctx(c), saved(c->from_bam) { ctx->from_bam = true; }
    ~FromBam() { ctx->from_bam = saved; }
};

}  // namespace

// ------------------------------------------------------------------------------------------------
// C ABI
// ------------------------------------------------------------------------------------------------
extern "C" {

const char* spl_version(void) { return "spliser_b200 0.1.0 (SpliSER v0.1.8 counting path, sm_100a)"; }

int spl_create(spl_ctx** out, const int* device_ids, int n_devices) {
    if (!out) return SPL_ERR_ARG;
    *out = nullptr;
    spl_ctx* ctx = new (std::nothrow) spl_ctx();
    if (!ctx) return SPL_ERR_NOMEM;
    *out = ctx;   // returned even on failure so that spl_last_error() can be read; caller destroys it
    if (n_devices != 1 || !device_ids)
        return ctx->fail(SPL_ERR_ARG, "this build drives exactly one GPU per context (one process per GPU); got n_devices=%d", n_devices);
    int count = 0;
    cudaError_t e = cudaGetDeviceCount(&count);
    if (e != cudaSuccess || count == 0) {
        cudaGetLastError();
        return ctx->fail(SPL_ERR_CUDA, "no CUDA device available (%s); libspliser_b200 has no CPU fallback",
                         e == cudaSuccess ? "device count is 0" : cudaGetErrorString(e));
    }
    if (device_ids[0] < 0 || device_ids[0] >= count) return ctx->fail(SPL_ERR_ARG, "device %d out of range (%d devices)", device_ids[0], count);
    ctx->device = device_ids[0];
    CU(cudaSetDevice(ctx->device));
    cudaDeviceProp prop;
    CU(cudaGetDeviceProperties(&prop, ctx->device));
    if (prop.major != 10)
        return ctx->fail(SPL_ERR_CUDA, "device %d is sm_%d%d; this library carries sm_100a code only", ctx->device, prop.major, prop.minor);
    CU(cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking));
    CU(cudaStreamCreateWithFlags(&ctx->stream2, cudaStreamNonBlocking));
    CU(cudaEventCreateWithFlags(&ctx->ev_graph, cudaEventDisableTiming));
    CU(cudaStreamCreateWithFlags(&ctx->copy_stream, cudaStreamNonBlocking));
    for (int p = 0; p < MAX_PARTS; ++p) {
        CU(cudaHostAlloc((void**)&ctx->part[p].h_tot, 256, cudaHostAllocDefault));
        CU(cudaEventCreateWithFlags(&ctx->part[p].ev_up, cudaEventDisableTiming));
        CU(cudaEventCreate(&ctx->part[p].ev_e0)); CU(cudaEventCreate(&ctx->part[p].ev_e1));
    }
    for (int p = 0; p < MAX_FPARTS; ++p) CU(cudaEventCreateWithFlags(&ctx->fpart[p].ev_up, cudaEventDisableTiming));
    CU(cudaHostAlloc((void**)&ctx->h_hot, 64, cudaHostAllocDefault));
    *ctx->h_hot = 0;
    CU(cudaHostAlloc((void**)&ctx->gbm.h_cnt, 256, cudaHostAllocDefault));
    return SPL_OK;
}

void spl_destroy(spl_ctx* ctx) {
    if (!ctx) return;
    if (ctx->stream) {
        cudaSetDevice(ctx->device);
        cudaStreamSynchronize(ctx->stream);
        for (cudaEvent_t e : ctx->events) cudaEventDestroy(e);
        ctx->d_graph.release(); ctx->d_cnt.release(); ctx->d_out.release();
        for (int p = 0; p < MAX_PARTS; ++p) {
            ctx->part[p].release();
            if (ctx->part[p].h_tot) cudaFreeHost(ctx->part[p].h_tot);
            if (ctx->part[p].h_chunks) cudaFreeHost(ctx->part[p].h_chunks);
            if (ctx->part[p].ev_up) cudaEventDestroy(ctx->part[p].ev_up);
            if (ctx->part[p].ev_e0) cudaEventDestroy(ctx->part[p].ev_e0);
            if (ctx->part[p].ev_e1) cudaEventDestroy(ctx->part[p].ev_e1);
        }
        if (ctx->copy_stream) { cudaStreamSynchronize(ctx->copy_stream); cudaStreamDestroy(ctx->copy_stream); }
        ctx->d_frec.release(); ctx->d_fchunks.release(); ctx->d_hotq.release(); ctx->d_fpk.release(); ctx->d_unpack.release(); ctx->d_cpk.release();
        ctx->d_xs.release(); ctx->d_votes.release();
        if (ctx->h_hot) cudaFreeHost(ctx->h_hot);
        if (ctx->h_fchunks) cudaFreeHost(ctx->h_fchunks);
        for (int p = 0; p < MAX_FPARTS; ++p) if (ctx->fpart[p].ev_up) cudaEventDestroy(ctx->fpart[p].ev_up);
        if (ctx->gbm.h_cnt) cudaFreeHost(ctx->gbm.h_cnt);
        if (ctx->pending) { spl_result_free(ctx->pending); ctx->pending = nullptr; }
        if (ctx->h_stage) cudaFreeHost(ctx->h_stage);
        if (ctx->h_file) cudaFreeHost(ctx->h_file);
        ctx->bgm.comp.release(); ctx->bgm.unc.release(); ctx->bgm.tab.release(); ctx->bgm.rec.release(); ctx->bgm.list.release();
        ctx->bgm.tags.release(); ctx->gsm.release();
        ctx->gbm.fin.release(); ctx->gbm.fin2.release(); ctx->gbm.work.release(); ctx->gbm.work2.release();
        ctx->jem.release();
        if (ctx->stream2) { cudaStreamSynchronize(ctx->stream2); cudaStreamDestroy(ctx->stream2); }
        if (ctx->ev_graph) cudaEventDestroy(ctx->ev_graph);
        cudaStreamDestroy(ctx->stream);
    }
    delete ctx;
}

const char* spl_last_error(const spl_ctx* ctx) { return ctx ? ctx->err.c_str() : "NULL context"; }

int spl_set_tile(spl_ctx* ctx, int tile_index, int tile_count) {
    if (!ctx) return SPL_ERR_ARG;
    if (tile_count < 1 || tile_index < 0 || tile_index >= tile_count) return ctx->fail(SPL_ERR_ARG, "bad tile %d/%d", tile_index, tile_count);
    ctx->tile_index = tile_index; ctx->tile_count = tile_count;
    ctx->tile_lo = ctx->tile_hi = -1;
    return SPL_OK;
}

int spl_set_tile_sites(spl_ctx* ctx, int64_t site_lo, int64_t site_hi) {
    if (!ctx) return SPL_ERR_ARG;
    if (site_lo < 0 && site_hi < 0) { ctx->tile_lo = ctx->tile_hi = -1; return SPL_OK; }
    if (site_lo < 0 || site_hi < site_lo) return ctx->fail(SPL_ERR_ARG, "bad owned site range [%lld, %lld)", (long long)site_lo, (long long)site_hi);
    ctx->tile_lo = site_lo; ctx->tile_hi = site_hi;
    return SPL_OK;
}

int spl_set_variant(spl_ctx* ctx, int variant) {
    if (!ctx) return SPL_ERR_ARG;
    if (variant != SPL_VARIANT_FUSED && variant != SPL_VARIANT_STAB) return ctx->fail(SPL_ERR_ARG, "unknown variant %d", variant);
    ctx->variant = variant;
    ctx->loaded = false;
    return SPL_OK;
}

unsigned long long spl_kernel_launches(void) { return g_kernel_launches.load(); }

int spl_set_threads(spl_ctx* ctx, int n) {
    if (!ctx) return SPL_ERR_ARG;
    ctx->n_threads = n < 0 ? 0 : n;
    return SPL_OK;
}

int spl_set_read_filter(spl_ctx* ctx, const spl_read_filter* filter) {
    if (!ctx) return SPL_ERR_ARG;
    ReadFilter rf;
    std::string e;
    if (filter && !read_filter_from(*filter, rf, e)) return ctx->fail(SPL_ERR_ARG, "%s", e.c_str());
    ctx->rf = rf;
    return SPL_OK;
}

int spl_last_read_filter(const spl_ctx* ctx, int64_t counts[2]) {
    if (!ctx || !counts) return SPL_ERR_ARG;
    counts[0] = ctx->rf_counts[0]; counts[1] = ctx->rf_counts[1];
    return SPL_OK;
}

int spl_last_stats(const spl_ctx* ctx, double* stats_out) {
    if (!ctx || !stats_out) return SPL_ERR_ARG;
    memcpy(stats_out, ctx->stats, sizeof ctx->stats);
    return SPL_OK;
}

int spl_process_records(spl_ctx* ctx, const spl_records_view* rec, int32_t n_chrom, int64_t n_junc, const int32_t* j_chrom,
                        const int32_t* j_left, const int32_t* j_right, const int64_t* j_score, const uint8_t* j_strand,
                        uint32_t flags, spl_result** out) {
    if (!ctx) return SPL_ERR_ARG;
    if (!out) return ctx->fail(SPL_ERR_ARG, "out is NULL");
    *out = nullptr;
    if (!ctx->stream) return ctx->fail(SPL_ERR_CUDA, "context has no CUDA device; libspliser_b200 has no CPU fallback");
    if (const int rr = refuse_records(ctx, "spl_process_records")) return rr;
    const double t0 = now_ms();
    int rc = load_common(ctx, rec, n_chrom, n_junc, j_chrom, j_left, j_right, j_score, j_strand, flags, true);
    if (rc) return drain_on_error(ctx, rc);
    const double tc0 = now_ms();
    for (;;) {
        rc = count_pass(ctx, nullptr);
        if (rc) return drain_on_error(ctx, rc);
        rc = drain_on_error(ctx, fetch(ctx, out));
        if (rc) return rc;
        bool again = false;
        rc = hot_queue_overflow(ctx, &again);
        if (rc) { spl_result_free(*out); *out = nullptr; return rc; }
        if (!again) break;
        spl_result_free(*out); *out = nullptr;
    }
    collect_expand_ms(ctx);
    ctx->stats[SPL_STAT_MS_COUNT] = now_ms() - tc0;
    ctx->stats[SPL_STAT_MS_TOTAL] = now_ms() - t0;
    return rc;
}

int spl_process_packed(spl_ctx* ctx, const spl_packed_view* pv, int32_t n_chrom, int64_t n_junc, const int32_t* j_chrom,
                       const int32_t* j_left, const int32_t* j_right, const int64_t* j_score, const uint8_t* j_strand,
                       uint32_t flags, spl_result** out) {
    if (!ctx) return SPL_ERR_ARG;
    if (!out) return ctx->fail(SPL_ERR_ARG, "out is NULL");
    *out = nullptr;
    if (!ctx->stream) return ctx->fail(SPL_ERR_CUDA, "context has no CUDA device; libspliser_b200 has no CPU fallback");
    if (!pv) return ctx->fail(SPL_ERR_ARG, "packed view is NULL");
    if (const int rr = refuse_records(ctx, "spl_process_packed")) return rr;
    if (ctx->variant != SPL_VARIANT_FUSED) return ctx->fail(SPL_ERR_ARG, "the packed view is read by the fused variant only");
    if (pv->n_rec > 0 && (!pv->pos || !pv->flag8 || !pv->n_op || !pv->cig_index)) return ctx->fail(SPL_ERR_ARG, "NULL packed array");
    if (pv->n_cigar > 0 && !pv->cigar) return ctx->fail(SPL_ERR_ARG, "NULL cigar array");
    // the segment / size checks are those of the plain view (arrays are not dereferenced there for device-resident records)
    spl_records_view shell{};
    shell.n_rec = pv->n_rec; shell.n_cigar = pv->n_cigar; shell.n_seg = pv->n_seg; shell.seg_chrom = pv->seg_chrom; shell.seg_off = pv->seg_off;
    const double t0 = now_ms();
    ctx->rec_on_device = true;                                         // check_view: no host record arrays to look at
    int rc = load_common(ctx, &shell, n_chrom, n_junc, j_chrom, j_left, j_right, j_score, j_strand, flags, true, pv);
    ctx->rec_on_device = false;
    if (rc) return drain_on_error(ctx, rc);
    const double tc0 = now_ms();
    for (;;) {
        rc = count_pass(ctx, nullptr);
        if (rc) return drain_on_error(ctx, rc);
        rc = drain_on_error(ctx, fetch(ctx, out));
        if (rc) return rc;
        bool again = false;
        rc = hot_queue_overflow(ctx, &again);
        if (rc) { spl_result_free(*out); *out = nullptr; return rc; }
        if (!again) break;
        spl_result_free(*out); *out = nullptr;
    }
    ctx->stats[SPL_STAT_MS_COUNT] = now_ms() - tc0;
    ctx->stats[SPL_STAT_MS_TOTAL] = now_ms() - t0;
    return rc;
}

int spl_process_compact(spl_ctx* ctx, const spl_compact_view* cv, int32_t n_chrom, int64_t n_junc, const int32_t* j_chrom,
                        const int32_t* j_left, const int32_t* j_right, const int64_t* j_score, const uint8_t* j_strand,
                        uint32_t flags, spl_result** out) {
    if (!ctx) return SPL_ERR_ARG;
    if (!out) return ctx->fail(SPL_ERR_ARG, "out is NULL");
    *out = nullptr;
    if (!ctx->stream) return ctx->fail(SPL_ERR_CUDA, "context has no CUDA device; libspliser_b200 has no CPU fallback");
    if (!cv) return ctx->fail(SPL_ERR_ARG, "compact view is NULL");
    if (const int rr = refuse_records(ctx, "spl_process_compact")) return rr;
    if (ctx->variant != SPL_VARIANT_FUSED) return ctx->fail(SPL_ERR_ARG, "the compact view is read by the fused variant only");
    if (cv->n_rec < 0 || cv->n16 < 0 || cv->n32 < 0 || cv->n_wide < 0 || cv->n16 + cv->n32 != cv->n_cigar)
        return ctx->fail(SPL_ERR_ARG, "compact view: inconsistent sizes");
    if (cv->n_rec > 0 && (!cv->pos16 || !cv->flag8 || !cv->n_op8 || !cv->pos_base || !cv->idx16 || !cv->idx32))
        return ctx->fail(SPL_ERR_ARG, "NULL compact array");
    if ((cv->n16 > 0 && !cv->cigar16) || (cv->n32 > 0 && !cv->cigar32) || (cv->n_wide > 0 && !cv->pos_wide))
        return ctx->fail(SPL_ERR_ARG, "NULL compact array");
    {   // the anchors are what the device trusts: check them here (12 B per 1024 records)
        const int64_t K = SPL_PACKED_INDEX_STRIDE, NS = (cv->n_rec + K - 1) / K;
        if (cv->n_rec > 0 && (cv->idx16[0] != 0 || cv->idx32[0] != 0 || (int64_t)cv->idx16[NS] != cv->n16 || (int64_t)cv->idx32[NS] != cv->n32))
            return ctx->fail(SPL_ERR_ARG, "compact view: operator index does not span the streams");
        for (int64_t k = 0; k < NS; ++k) {
            if (cv->idx16[k + 1] < cv->idx16[k] || cv->idx32[k + 1] < cv->idx32[k]) return ctx->fail(SPL_ERR_ARG, "compact view: operator index not monotonic");
            if ((uint64_t)(cv->idx16[k + 1] - cv->idx16[k]) + (cv->idx32[k + 1] - cv->idx32[k]) > 255u * (uint64_t)K)
                return ctx->fail(SPL_ERR_ARG, "compact view: a stride claims more operators than its records can hold");
            if (cv->pos_base[k] < 0 && -(int64_t)cv->pos_base[k] - 1 >= cv->n_wide) return ctx->fail(SPL_ERR_ARG, "compact view: wide stride out of range");
        }
    }
    spl_records_view shell{};
    shell.n_rec = cv->n_rec; shell.n_cigar = cv->n_cigar; shell.n_seg = cv->n_seg; shell.seg_chrom = cv->seg_chrom; shell.seg_off = cv->seg_off;
    const double t0 = now_ms();
    ctx->rec_on_device = true;                                         // check_view: no host record arrays to look at
    bool timeline = std::getenv("SPLISER_TIMING") != nullptr;
    cudaEvent_t te[3] = {nullptr, nullptr, nullptr};
    if (timeline) { for (auto& e : te) cudaEventCreate(&e); cudaEventRecord(te[0], ctx->copy_stream); }
    int rc = load_common(ctx, &shell, n_chrom, n_junc, j_chrom, j_left, j_right, j_score, j_strand, flags, true, nullptr, cv);
    ctx->rec_on_device = false;
    if (rc) return drain_on_error(ctx, rc);
    if (timeline) cudaEventRecord(te[2], ctx->copy_stream);            // behind the last slab's copy
    const double tc0 = now_ms();
    for (;;) {
        rc = count_pass(ctx, nullptr);
        if (rc) return drain_on_error(ctx, rc);
        if (timeline) cudaEventRecord(te[1], ctx->stream);
        rc = drain_on_error(ctx, fetch(ctx, out));
        if (rc) return rc;
        if (timeline) {
            float a = 0, b = 0;
            cudaEventElapsedTime(&a, te[0], te[2]); cudaEventElapsedTime(&b, te[0], te[1]);
            fprintf(stderr, "[compact] host: load returned +%.2f ms, fetch done +%.2f ms; device: last slab arrived +%.2f ms, finalize done +%.2f ms\n",
                    tc0 - t0, now_ms() - t0, a, b);
            for (auto& e : te) cudaEventDestroy(e);
            timeline = false;
        }
        bool again = false;
        rc = hot_queue_overflow(ctx, &again);
        if (rc) { spl_result_free(*out); *out = nullptr; return rc; }
        if (!again) break;
        spl_result_free(*out); *out = nullptr;
    }
    ctx->stats[SPL_STAT_MS_COUNT] = now_ms() - tc0;
    ctx->stats[SPL_STAT_MS_TOTAL] = now_ms() - t0;
    return rc;
}

int spl_process(spl_ctx* ctx, const char* bam_path, int32_t n_chrom, const char* const* chrom_names, int64_t n_junc,
                const int32_t* j_chrom, const int32_t* j_left, const int32_t* j_right, const int64_t* j_score,
                const uint8_t* j_strand, uint32_t flags, spl_result** out) {
    if (!ctx) return SPL_ERR_ARG;
    if (!out) return ctx->fail(SPL_ERR_ARG, "out is NULL");
    *out = nullptr;
    if (!ctx->stream) return ctx->fail(SPL_ERR_CUDA, "context has no CUDA device; libspliser_b200 has no CPU fallback");
    if (!bam_path) return ctx->fail(SPL_ERR_ARG, "bam_path is NULL");
    const double t0 = now_ms();
    CU(cudaSetDevice(ctx->device));
    FromBam from_bam(ctx);
    {   // BGZF inflate + record parse on the device; the host reader is the fallback for what that path does not cover
        BamGpuCounts cnt;
        spl_records_view dv{};
        bool fallback = false;
        int rc = ingest_bam_device(ctx, bam_path, n_chrom, chrom_names, cnt, dv, &fallback);
        if (rc) return rc;
        if (!fallback) {
            const double t1 = now_ms();
            ctx->rec_on_device = true;
            rc = spl_process_records(ctx, &dv, n_chrom, n_junc, j_chrom, j_left, j_right, j_score, j_strand, flags, out);
            ctx->rec_on_device = false;
            ctx->stats[SPL_STAT_MS_DECODE] = t1 - t0;
            ctx->stats[SPL_STAT_H2D_BYTES] += cnt.h2d_bytes;
            ctx->stats[SPL_STAT_BAM_DEVICE] = 1.0;
            ctx->stats[SPL_STAT_MS_TOTAL] = now_ms() - t0;
            return rc;
        }
    }
    BamRecords recs;
    std::string e = read_bam_ctx(ctx, bam_path, n_chrom, chrom_names, recs);
    if (!e.empty()) return ctx->fail(SPL_ERR_IO, "%s", e.c_str());
    const double t1 = now_ms();
    spl_records_view v = recs.view();
    int rc = spl_process_records(ctx, &v, n_chrom, n_junc, j_chrom, j_left, j_right, j_score, j_strand, flags, out);
    ctx->stats[SPL_STAT_MS_DECODE] = t1 - t0;
    ctx->stats[SPL_STAT_MS_TOTAL] = now_ms() - t0;
    return rc;
}

struct spl_junctions {
    std::vector<int32_t> chrom, left, right;
    std::vector<int64_t> score;
    std::vector<uint8_t> strand;
    std::vector<int32_t> start, end;    // BED12 chromStart / chromEnd: left - longest left anchor, right + longest right anchor
};

namespace {
// xs: the host records' XS strand column (SPL_FLAG_XS_STRAND without records on the device; the device ingest fills ctx->dev_rec.xs)
int extract_common(spl_ctx* ctx, const spl_records_view* rec, const uint8_t* xs, int32_t n_chrom, int32_t min_anchor, int32_t min_intron,
                   int32_t max_intron, uint32_t flags, spl_junctions** out) {
    if (min_anchor < 0 || min_intron < 0 || max_intron < min_intron) return ctx->fail(SPL_ERR_ARG, "bad anchor / intron bounds");
    ctx->loaded = false;
    int rc = check_view(ctx, rec, n_chrom);
    if (rc) return rc;
    CU(cudaSetDevice(ctx->device));
    reset_stats(ctx);
    rc = fused_upload(ctx, rec, n_chrom, false);
    if (rc) return drain_on_error(ctx, rc);
    CU(cudaStreamWaitEvent(ctx->stream, ctx->fpart[0].ev_up, 0));
    const uint8_t* d_xs = nullptr;
    if ((flags & SPL_FLAG_XS_STRAND) && rec->n_rec > 0) {
        if (ctx->rec_on_device) {
            d_xs = ctx->dev_rec.xs;
        } else if (xs) {                                                   // 1 B per record, once
            CU(ctx->d_xs.reserve((size_t)rec->n_rec + 16));
            CU(cudaMemcpyAsync(ctx->d_xs.p, xs, (size_t)rec->n_rec, cudaMemcpyHostToDevice, ctx->stream));
            ctx->stats[SPL_STAT_H2D_BYTES] += (double)rec->n_rec;
            d_xs = (const uint8_t*)ctx->d_xs.p;
        }
        if (!d_xs) return drain_on_error(ctx, ctx->fail(SPL_ERR_ARG, "SPL_FLAG_XS_STRAND without an XS strand column"));
    }
    std::unique_ptr<spl_junctions> j(new (std::nothrow) spl_junctions());
    if (!j) return ctx->fail(SPL_ERR_NOMEM, "out of memory");
    std::string e;
    if (!junction_extract_device(ctx->jem, ctx->frec, rec->seg_off, rec->seg_chrom, rec->n_seg, n_chrom, flags & 3u, d_xs, min_anchor,
                                 min_intron, max_intron, ctx->stream, j->chrom, j->left, j->right, j->score, j->strand, j->start, j->end, e))
        return drain_on_error(ctx, ctx->fail(SPL_ERR_CUDA, "%s", e.c_str()));
    ctx->stats[SPL_STAT_MS_EXTRACT] = ctx->jem.ms_kernels;
    ctx->stats[SPL_STAT_MS_EXTENTS] = ctx->jem.ms_extent;
    ctx->stats[SPL_STAT_N_JUNCTIONS] = (double)j->chrom.size();
    *out = j.release();
    return SPL_OK;
}

// spl_process_bam_extract after the ingest: junction table of the records, the -c / -g row filters, then the count over the
// same records, which extract_common left on the device (ctx->frec) -- they cross PCIe at most once.  SPL_FLAG_XS_STRAND only
// chooses the table's strands: the count runs with the remaining flags.
int extract_and_count(spl_ctx* ctx, const spl_records_view* rec, const uint8_t* xs, int32_t n_chrom, const char* const* chrom_names,
                      const spl_extract_opts* o, uint32_t flags, spl_junctions** rows_out, spl_result** out) {
    spl_junctions* got = nullptr;
    int rc = extract_common(ctx, rec, xs, n_chrom, o->min_anchor, o->min_intron, o->max_intron, flags, &got);
    if (rc) return rc;
    std::unique_ptr<spl_junctions> all(got);
    double keep[SPL_NSTATS];
    memcpy(keep, ctx->stats, sizeof keep);
    std::unique_ptr<spl_junctions> j(new (std::nothrow) spl_junctions());
    if (!j) return ctx->fail(SPL_ERR_NOMEM, "out of memory");
    const JunctionFilter f{o->qchrom, o->use_gene_window != 0, o->gene_left, o->gene_right, o->window_max_intron};
    for (size_t i = 0; i < all->chrom.size(); ++i) {
        const int32_t c = all->chrom[i];
        if (!f.chrom_kept(chrom_names[c]) || !f.window_kept(all->left[i], all->right[i])) continue;
        j->chrom.push_back(c); j->left.push_back(all->left[i]); j->right.push_back(all->right[i]);
        j->score.push_back(all->score[i]); j->strand.push_back(all->strand[i]);
        j->start.push_back(all->start[i]); j->end.push_back(all->end[i]);
    }
    // the count reads the records where the extraction left them: device-parsed records are ctx->dev_rec already, records of
    // the host reader are in the extraction's upload (ctx->d_frec)
    const DevRecordArrays saved = ctx->dev_rec;
    const bool saved_dev = ctx->rec_on_device;
    ctx->dev_rec.pos = const_cast<int32_t*>(ctx->frec.pos); ctx->dev_rec.flag = const_cast<uint16_t*>(ctx->frec.flag);
    ctx->dev_rec.cig_off = const_cast<uint32_t*>(ctx->frec.cig_off); ctx->dev_rec.cigar = const_cast<uint32_t*>(ctx->frec.cigar);
    spl_records_view dv{};
    dv.n_rec = rec->n_rec; dv.n_cigar = rec->n_cigar; dv.n_seg = rec->n_seg; dv.seg_chrom = rec->seg_chrom; dv.seg_off = rec->seg_off;
    ctx->rec_on_device = true;
    rc = spl_process_records(ctx, &dv, n_chrom, (int64_t)j->chrom.size(), j->chrom.data(), j->left.data(), j->right.data(),
                             j->score.data(), j->strand.data(), flags & ~SPL_FLAG_XS_STRAND, out);
    ctx->rec_on_device = saved_dev;
    ctx->dev_rec = saved;
    if (rc) return rc;
    ctx->stats[SPL_STAT_H2D_BYTES] += keep[SPL_STAT_H2D_BYTES];
    for (int k : {SPL_STAT_MS_EXTRACT, SPL_STAT_MS_EXTENTS, SPL_STAT_N_JUNCTIONS}) ctx->stats[k] = keep[k];
    *rows_out = j.release();
    return SPL_OK;
}
}  // namespace

int spl_extract_junctions_records(spl_ctx* ctx, const spl_records_view* rec, int32_t n_chrom, int32_t min_anchor, int32_t min_intron,
                                  int32_t max_intron, uint32_t flags, spl_junctions** out) {
    if (!ctx) return SPL_ERR_ARG;
    if (!out) return ctx->fail(SPL_ERR_ARG, "out is NULL");
    *out = nullptr;
    if (!ctx->stream) return ctx->fail(SPL_ERR_CUDA, "context has no CUDA device; libspliser_b200 has no CPU fallback");
    if (flags & SPL_FLAG_XS_STRAND) return ctx->fail(SPL_ERR_ARG, "SPL_FLAG_XS_STRAND needs the strand column of spl_extract_junctions_records_xs");
    if (const int rr = refuse_records(ctx, "spl_extract_junctions_records")) return rr;
    return extract_common(ctx, rec, nullptr, n_chrom, min_anchor, min_intron, max_intron, flags, out);
}

int spl_extract_junctions_records_xs(spl_ctx* ctx, const spl_records_view* rec, const uint8_t* xs, int32_t n_chrom, int32_t min_anchor,
                                     int32_t min_intron, int32_t max_intron, uint32_t flags, spl_junctions** out) {
    if (!ctx) return SPL_ERR_ARG;
    if (!out) return ctx->fail(SPL_ERR_ARG, "out is NULL");
    *out = nullptr;
    if (!ctx->stream) return ctx->fail(SPL_ERR_CUDA, "context has no CUDA device; libspliser_b200 has no CPU fallback");
    if (!xs && rec && rec->n_rec > 0) return ctx->fail(SPL_ERR_ARG, "xs is NULL");
    if (const int rr = refuse_records(ctx, "spl_extract_junctions_records_xs")) return rr;
    return extract_common(ctx, rec, xs, n_chrom, min_anchor, min_intron, max_intron, flags, out);
}

int spl_extract_junctions(spl_ctx* ctx, const char* bam_path, int32_t n_chrom, const char* const* chrom_names, int32_t min_anchor,
                          int32_t min_intron, int32_t max_intron, uint32_t flags, spl_junctions** out) {
    if (!ctx) return SPL_ERR_ARG;
    if (!out) return ctx->fail(SPL_ERR_ARG, "out is NULL");
    *out = nullptr;
    if (!ctx->stream) return ctx->fail(SPL_ERR_CUDA, "context has no CUDA device; libspliser_b200 has no CPU fallback");
    if (!bam_path) return ctx->fail(SPL_ERR_ARG, "bam_path is NULL");
    const double t0 = now_ms();
    CU(cudaSetDevice(ctx->device));
    {
        BamGpuCounts cnt;
        spl_records_view dv{};
        bool fallback = false;
        int rc = ingest_bam_device(ctx, bam_path, n_chrom, chrom_names, cnt, dv, &fallback, (flags & SPL_FLAG_XS_STRAND) != 0);
        if (rc) return rc;
        if (!fallback) {
            const double t1 = now_ms();
            ctx->rec_on_device = true;
            rc = extract_common(ctx, &dv, nullptr, n_chrom, min_anchor, min_intron, max_intron, flags, out);
            ctx->rec_on_device = false;
            ctx->stats[SPL_STAT_MS_DECODE] = t1 - t0;
            ctx->stats[SPL_STAT_H2D_BYTES] += cnt.h2d_bytes;
            ctx->stats[SPL_STAT_BAM_DEVICE] = 1.0;
            ctx->stats[SPL_STAT_MS_TOTAL] = now_ms() - t0;
            return rc;
        }
    }
    BamRecords recs;
    std::string e = read_bam_ctx(ctx, bam_path, n_chrom, chrom_names, recs, (flags & SPL_FLAG_XS_STRAND) != 0);
    if (!e.empty()) return ctx->fail(SPL_ERR_IO, "%s", e.c_str());
    const double t1 = now_ms();
    spl_records_view v = recs.view();
    const int rc = extract_common(ctx, &v, recs.xs.data(), n_chrom, min_anchor, min_intron, max_intron, flags, out);
    ctx->stats[SPL_STAT_MS_DECODE] = t1 - t0;
    ctx->stats[SPL_STAT_MS_TOTAL] = now_ms() - t0;
    return rc;
}

int64_t spl_junctions_n(const spl_junctions* j) { return j ? (int64_t)j->chrom.size() : 0; }
const int32_t* spl_junctions_chrom(const spl_junctions* j) { return j->chrom.data(); }
const int32_t* spl_junctions_left(const spl_junctions* j) { return j->left.data(); }
const int32_t* spl_junctions_right(const spl_junctions* j) { return j->right.data(); }
const int64_t* spl_junctions_score(const spl_junctions* j) { return j->score.data(); }
const uint8_t* spl_junctions_strand(const spl_junctions* j) { return j->strand.data(); }
const int32_t* spl_junctions_start(const spl_junctions* j) { return j->start.data(); }
const int32_t* spl_junctions_end(const spl_junctions* j) { return j->end.data(); }

int spl_process_bam_extract(spl_ctx* ctx, const char* bam_path, int32_t n_chrom, const char* const* chrom_names, const spl_extract_opts* opts,
                            uint32_t flags, spl_junctions** rows_out, spl_result** out) {
    if (!ctx) return SPL_ERR_ARG;
    if (!out || !rows_out) return ctx->fail(SPL_ERR_ARG, "out is NULL");
    *out = nullptr; *rows_out = nullptr;
    if (!ctx->stream) return ctx->fail(SPL_ERR_CUDA, "context has no CUDA device; libspliser_b200 has no CPU fallback");
    if (!bam_path || !opts) return ctx->fail(SPL_ERR_ARG, "bam_path or opts is NULL");
    if (n_chrom < 0 || (n_chrom > 0 && !chrom_names)) return ctx->fail(SPL_ERR_ARG, "chrom_names is NULL");
    for (int32_t c = 0; c < n_chrom; ++c) if (!chrom_names[c]) return ctx->fail(SPL_ERR_ARG, "chromosome name %d is NULL", c);
    const double t0 = now_ms();
    CU(cudaSetDevice(ctx->device));
    FromBam from_bam(ctx);
    {   // ingest exactly as spl_process chooses: BGZF inflate + record parse on the device, the host reader as the fallback
        BamGpuCounts cnt;
        spl_records_view dv{};
        bool fallback = false;
        int rc = ingest_bam_device(ctx, bam_path, n_chrom, chrom_names, cnt, dv, &fallback, (flags & SPL_FLAG_XS_STRAND) != 0);
        if (rc) return rc;
        if (!fallback) {
            const double t1 = now_ms();
            ctx->rec_on_device = true;
            rc = extract_and_count(ctx, &dv, nullptr, n_chrom, chrom_names, opts, flags, rows_out, out);
            ctx->rec_on_device = false;
            ctx->stats[SPL_STAT_MS_DECODE] = t1 - t0;
            ctx->stats[SPL_STAT_H2D_BYTES] += cnt.h2d_bytes;
            ctx->stats[SPL_STAT_BAM_DEVICE] = 1.0;
            ctx->stats[SPL_STAT_MS_TOTAL] = now_ms() - t0;
            return rc;
        }
    }
    BamRecords recs;
    std::string e = read_bam_ctx(ctx, bam_path, n_chrom, chrom_names, recs, (flags & SPL_FLAG_XS_STRAND) != 0);
    if (!e.empty()) return ctx->fail(SPL_ERR_IO, "%s", e.c_str());
    const double t1 = now_ms();
    spl_records_view v = recs.view();
    const int rc = extract_and_count(ctx, &v, recs.xs.data(), n_chrom, chrom_names, opts, flags, rows_out, out);
    ctx->stats[SPL_STAT_MS_DECODE] = t1 - t0;
    ctx->stats[SPL_STAT_MS_TOTAL] = now_ms() - t0;
    return rc;
}
void spl_junctions_free(spl_junctions* j) { delete j; }

int spl_recount_records(spl_ctx* ctx, const spl_records_view* rec, int32_t n_chrom, int64_t n_sites, const int32_t* s_chrom,
                        const int32_t* s_pos, const uint8_t* s_strand, const int64_t* p_off, const int32_t* p_pos,
                        const int64_t* c_off, const int32_t* c_pos, uint32_t flags, int64_t* beta1_out, int64_t* beta2simple_out) {
    if (!ctx) return SPL_ERR_ARG;
    if (!ctx->stream) return ctx->fail(SPL_ERR_CUDA, "context has no CUDA device; libspliser_b200 has no CPU fallback");
    if (n_sites > 0 && (!beta1_out || !beta2simple_out)) return ctx->fail(SPL_ERR_ARG, "NULL output array");
    if (const int rr = refuse_records(ctx, "spl_recount_records")) return rr;
    ctx->loaded = false;
    int rc = check_view(ctx, rec, n_chrom);
    if (rc) return rc;
    CU(cudaSetDevice(ctx->device));
    reset_stats(ctx);
    const double t0 = now_ms();
    flags |= SPL_FLAG_COMBINE;
    flags &= ~SPL_FLAG_CRYPTIC;
    std::string e = build_recount_graph(n_chrom, n_sites, s_chrom, s_pos, s_strand, p_off, p_pos, c_off, c_pos,
                                        (flags & SPL_FLAG_STRANDED) != 0, ctx->hg);
    if (!e.empty()) return ctx->fail(SPL_ERR_ARG, "%s", e.c_str());
    ctx->flags = flags;
    const int save_ti = ctx->tile_index, save_tc = ctx->tile_count;
    const int64_t save_lo = ctx->tile_lo, save_hi = ctx->tile_hi;
    ctx->tile_index = 0; ctx->tile_count = 1; ctx->tile_lo = ctx->tile_hi = -1;   // a re-count is sharded by sample, never by tile
    rc = upload_graph(ctx, nullptr, 0);
    ctx->tile_index = save_ti; ctx->tile_count = save_tc; ctx->tile_lo = save_lo; ctx->tile_hi = save_hi;
    if (rc) return rc;
    ctx->loaded_variant = ctx->variant;
    if (ctx->variant == SPL_VARIANT_FUSED) {
        rc = fused_upload(ctx, rec, n_chrom, false);
        if (rc) return drain_on_error(ctx, rc);
    } else {
        rc = upload_and_expand(ctx, rec, flags, n_chrom);
        if (rc) return drain_on_error(ctx, rc);
        const int prc = prepare_parts(ctx);
        if (prc) return drain_on_error(ctx, prc);
    }
    const size_t S = (size_t)ctx->hg.n_sites;
    std::vector<int64_t> b1(S), b2(S);
    for (;;) {
        rc = count_pass(ctx, nullptr);
        if (rc) return drain_on_error(ctx, rc);
        if (S) {
            CU(cudaMemcpyAsync(b1.data(), ctx->out.beta1, S * 8, cudaMemcpyDeviceToHost, ctx->stream));
            CU(cudaMemcpyAsync(b2.data(), ctx->out.beta2s, S * 8, cudaMemcpyDeviceToHost, ctx->stream));
        }
        CU(cudaStreamSynchronize(ctx->stream));
        bool again = false;
        rc = hot_queue_overflow(ctx, &again);
        if (rc) return rc;
        if (!again) break;
    }
    collect_expand_ms(ctx);
    for (int64_t i = 0; i < n_sites; ++i) { beta1_out[i] = 0; beta2simple_out[i] = 0; }
    for (size_t k = 0; k < S; ++k) {
        const int64_t gi = ctx->hg.gap_index[k];
        if (gi >= 0) { beta1_out[gi] = b1[k]; beta2simple_out[gi] = b2[k]; }
    }
    ctx->stats[SPL_STAT_D2H_BYTES] += (double)(S * 16);
    ctx->stats[SPL_STAT_N_SITES] = (double)n_sites;
    ctx->stats[SPL_STAT_MS_TOTAL] = now_ms() - t0;
    return SPL_OK;
}

int spl_recount(spl_ctx* ctx, const char* bam_path, int32_t n_chrom, const char* const* chrom_names, int64_t n_sites,
                const int32_t* s_chrom, const int32_t* s_pos, const uint8_t* s_strand, const int64_t* p_off, const int32_t* p_pos,
                const int64_t* c_off, const int32_t* c_pos, uint32_t flags, int64_t* beta1_out, int64_t* beta2simple_out) {
    if (!ctx) return SPL_ERR_ARG;
    if (!ctx->stream) return ctx->fail(SPL_ERR_CUDA, "context has no CUDA device; libspliser_b200 has no CPU fallback");
    if (!bam_path) return ctx->fail(SPL_ERR_ARG, "bam_path is NULL");
    const double t0 = now_ms();
    CU(cudaSetDevice(ctx->device));
    FromBam from_bam(ctx);
    {
        BamGpuCounts cnt;
        spl_records_view dv{};
        bool fallback = false;
        int rc = ingest_bam_device(ctx, bam_path, n_chrom, chrom_names, cnt, dv, &fallback);
        if (rc) return rc;
        if (!fallback) {
            const double t1 = now_ms();
            ctx->rec_on_device = true;
            rc = spl_recount_records(ctx, &dv, n_chrom, n_sites, s_chrom, s_pos, s_strand, p_off, p_pos, c_off, c_pos, flags,
                                     beta1_out, beta2simple_out);
            ctx->rec_on_device = false;
            ctx->stats[SPL_STAT_MS_DECODE] = t1 - t0;
            ctx->stats[SPL_STAT_BAM_DEVICE] = 1.0;
            ctx->stats[SPL_STAT_MS_TOTAL] = now_ms() - t0;
            return rc;
        }
    }
    BamRecords recs;
    std::string e = read_bam_ctx(ctx, bam_path, n_chrom, chrom_names, recs);
    if (!e.empty()) return ctx->fail(SPL_ERR_IO, "%s", e.c_str());
    const double t1 = now_ms();
    spl_records_view v = recs.view();
    int rc = spl_recount_records(ctx, &v, n_chrom, n_sites, s_chrom, s_pos, s_strand, p_off, p_pos, c_off, c_pos, flags,
                                 beta1_out, beta2simple_out);
    ctx->stats[SPL_STAT_MS_DECODE] = t1 - t0;
    ctx->stats[SPL_STAT_MS_TOTAL] = now_ms() - t0;
    return rc;
}

// ---- device-resident samples ----------------------------------------------------------------------------------------------
namespace {
std::atomic<int64_t> g_resident_bytes(0);          // what the samples of this process hold (SPLISER_SAMPLE_BUDGET_MB caps it)

// One device allocation of resident samples: a sample of spl_sample_load_bam owns one, the group samples of one
// spl_sample_load_bam_groups share one.  The last owner frees it and returns its bytes to the residency count.
struct SampleBlock {
    void* p = nullptr;
    size_t bytes = 0;
    int device = 0;
    SampleBlock(void* p_, size_t b, int d) : p(p_), bytes(b), device(d) {}
    ~SampleBlock() {
        if (!p) return;
        cudaSetDevice(device);
        cudaFree(p);
        g_resident_bytes -= (int64_t)bytes;
    }
};
}  // namespace

struct spl_sample {
    const spl_ctx* ctx = nullptr;         // the context that loaded it (compared, never dereferenced)
    int device = 0;
    std::shared_ptr<SampleBlock> mem;     // the device allocation that holds every column (shared by the samples of one split)
    size_t bytes = 0;                     // the sample's own slice of it
    DevRecordArrays rec{};                // pos / flag / cig_off / cigar (/ xs) inside mem; no per-record chromosome
    int64_t n_rec = 0, n_cigar = 0;
    std::vector<std::string> ref_names;   // the header's references, in header order
    ReadFilter rf;                        // the read filter the records were ingested under
    std::vector<int32_t> seg_ref;         // header reference index of every segment
    std::vector<int64_t> seg_off;         // [n_seg + 1]
};

namespace {
constexpr size_t SAMPLE_HEADROOM = (size_t)1 << 30;

// Takes `bytes` of device memory for a sample under the residency policy of spl_sample_load_bam; SPL_ERR_NOMEM holds nothing.
int sample_reserve(spl_ctx* ctx, size_t bytes, void** p) {
    *p = nullptr;
    const int64_t b = (int64_t)bytes;
    const int64_t held = g_resident_bytes.fetch_add(b) + b;
    auto refuse = [&](int code, const char* why) {
        g_resident_bytes -= b;
        return ctx->fail(code, "a resident sample of %zu bytes is not held: %s", bytes, why);
    };
    if (const char* cap = std::getenv("SPLISER_SAMPLE_BUDGET_MB"))
        if (held > std::max<int64_t>(0, atoll(cap)) * ((int64_t)1 << 20)) return refuse(SPL_ERR_NOMEM, "over SPLISER_SAMPLE_BUDGET_MB");
    size_t free_b = 0, total_b = 0;
    if (cudaMemGetInfo(&free_b, &total_b) != cudaSuccess) { cudaGetLastError(); return refuse(SPL_ERR_CUDA, "cudaMemGetInfo failed"); }
    if (free_b < 2 * bytes + SAMPLE_HEADROOM) return refuse(SPL_ERR_NOMEM, "it would leave the context less free device memory than its headroom");
    if (cudaMalloc(p, bytes) != cudaSuccess) { cudaGetLastError(); *p = nullptr; return refuse(SPL_ERR_NOMEM, "cudaMalloc failed"); }
    return SPL_OK;
}

int check_sample(spl_ctx* ctx, const spl_sample* s, int32_t n_chrom, const char* const* chrom_names) {
    if (!s) return ctx->fail(SPL_ERR_ARG, "sample is NULL");
    if (s->ctx != ctx) return ctx->fail(SPL_ERR_ARG, "the sample was loaded by another context");
    if (s->rf.min_mapq != ctx->rf.min_mapq || s->rf.exclude != ctx->rf.exclude || s->rf.require != ctx->rf.require)
        return ctx->fail(SPL_ERR_ARG, "the sample was loaded under read filter (min MAPQ %u, exclude 0x%x, require 0x%x) and the context's is "
                         "now (min MAPQ %u, exclude 0x%x, require 0x%x): load the sample again, or set its filter back",
                         s->rf.min_mapq, s->rf.exclude, s->rf.require, ctx->rf.min_mapq, ctx->rf.exclude, ctx->rf.require);
    if (n_chrom < 0 || (n_chrom > 0 && !chrom_names)) return ctx->fail(SPL_ERR_ARG, "chrom_names is NULL");
    for (int32_t c = 0; c < n_chrom; ++c) if (!chrom_names[c]) return ctx->fail(SPL_ERR_ARG, "chromosome name %d is NULL", c);
    return SPL_OK;
}

// The sample's segments under the caller's chromosome list, by the rule the readers map references with (map_references): a
// reference that is not in the list becomes -1 and its records are skipped.  `seg_chrom` must outlive the view.
spl_records_view sample_view(const spl_sample* s, int32_t n_chrom, const char* const* chrom_names, std::vector<int32_t>& seg_chrom) {
    const std::vector<int32_t> refmap = map_references(s->ref_names, n_chrom, chrom_names);
    seg_chrom.resize(s->seg_ref.size());
    for (size_t k = 0; k < seg_chrom.size(); ++k) seg_chrom[k] = refmap[(size_t)s->seg_ref[k]];
    spl_records_view v{};
    v.n_rec = s->n_rec; v.n_cigar = s->n_cigar;
    v.n_seg = (int32_t)seg_chrom.size(); v.seg_chrom = seg_chrom.data(); v.seg_off = s->seg_off.data();
    return v;
}

// ctx->dev_rec is the sample's columns for the duration of one call (records on the device, no upload)
struct SampleBinding {
    spl_ctx* ctx;
    DevRecordArrays saved;
    bool saved_dev;
    FromBam from_bam;                     // the sample's records were ingested under its filter, which check_sample matched
    SampleBinding(spl_ctx* c, const spl_sample* s) : ctx(c), saved(c->dev_rec), saved_dev(c->rec_on_device), from_bam(c) {
        ctx->dev_rec = s->rec;
        ctx->rec_on_device = true;
    }
    ~SampleBinding() { ctx->dev_rec = saved; ctx->rec_on_device = saved_dev; }
};
}  // namespace

int spl_sample_load_bam(spl_ctx* ctx, const char* bam_path, uint32_t flags, spl_sample** out) {
    if (!ctx) return SPL_ERR_ARG;
    if (!out) return ctx->fail(SPL_ERR_ARG, "out is NULL");
    *out = nullptr;
    if (!ctx->stream) return ctx->fail(SPL_ERR_CUDA, "context has no CUDA device; libspliser_b200 has no CPU fallback");
    if (!bam_path) return ctx->fail(SPL_ERR_ARG, "bam_path is NULL");
    if (flags & ~SPL_FLAG_XS_STRAND) return ctx->fail(SPL_ERR_ARG, "spl_sample_load_bam takes SPL_FLAG_XS_STRAND only");
    const bool want_xs = (flags & SPL_FLAG_XS_STRAND) != 0;
    const double t0 = now_ms();
    CU(cudaSetDevice(ctx->device));
    reset_stats(ctx);
    std::unique_ptr<spl_sample> s(new (std::nothrow) spl_sample());
    if (!s) return ctx->fail(SPL_ERR_NOMEM, "out of memory");
    s->ctx = ctx;
    s->device = ctx->device;
    s->rf = ctx->rf;
    // ingest exactly as spl_process chooses, every reference kept in header order
    BamGpuCounts cnt;
    spl_records_view dv{};
    bool fallback = false;
    int rc = ingest_bam_device(ctx, bam_path, 0, nullptr, cnt, dv, &fallback, want_xs, &s->ref_names);
    if (rc) return rc;
    BamRecords recs;
    if (fallback) {
        std::string e = read_bam_ctx(ctx, bam_path, 0, nullptr, recs, want_xs, &s->ref_names);
        if (!e.empty()) return ctx->fail(SPL_ERR_IO, "%s", e.c_str());
        s->n_rec = (int64_t)recs.pos.size(); s->n_cigar = (int64_t)recs.cigar.size();
        s->seg_ref = recs.seg_chrom; s->seg_off = recs.seg_off;
    } else {
        s->n_rec = (int64_t)cnt.n_rec; s->n_cigar = (int64_t)cnt.n_cigar;
        s->seg_ref = cnt.seg_chrom; s->seg_off = cnt.seg_off;
    }
    if (s->seg_off.empty()) s->seg_off.assign(1, 0);
    const double t1 = now_ms();
    const size_t n = (size_t)s->n_rec, nc = (size_t)s->n_cigar;
    Carver c;
    const size_t o_pos = c.take<int32_t>(n + 4), o_flag = c.take<uint16_t>(n + 4), o_off = c.take<uint32_t>(n + 4),
                 o_cig = c.take<uint32_t>(nc + 4), o_xs = want_xs ? c.take<uint8_t>(n + 4) : 0;
    void* mp = nullptr;
    rc = sample_reserve(ctx, c.off, &mp);
    if (rc) return rc;
    s->mem = std::make_shared<SampleBlock>(mp, c.off, ctx->device);
    s->bytes = c.off;
    char* m = (char*)mp;
    s->rec.pos = (int32_t*)(m + o_pos); s->rec.flag = (uint16_t*)(m + o_flag);
    s->rec.cig_off = (uint32_t*)(m + o_off); s->rec.cigar = (uint32_t*)(m + o_cig);
    s->rec.xs = want_xs ? (uint8_t*)(m + o_xs) : nullptr;
    // device ingest: one copy out of the context's scratch (which the next ingest re-uses); host reader: the upload itself
    const cudaMemcpyKind kind = fallback ? cudaMemcpyHostToDevice : cudaMemcpyDeviceToDevice;
    const DevRecordArrays& src = ctx->dev_rec;
    cudaError_t ce = cudaSuccess;
    auto copy = [&](void* dst, const void* from, size_t bytes) {
        if (bytes && ce == cudaSuccess) ce = cudaMemcpyAsync(dst, from, bytes, kind, ctx->stream);
    };
    if (n) {
        copy(s->rec.pos, fallback ? (const void*)recs.pos.data() : src.pos, n * 4);
        copy(s->rec.flag, fallback ? (const void*)recs.flag.data() : src.flag, n * 2);
        copy(s->rec.cig_off, fallback ? (const void*)recs.cig_off.data() : src.cig_off, (n + 1) * 4);
        copy(s->rec.cigar, fallback ? (const void*)recs.cigar.data() : src.cigar, nc * 4);
        if (want_xs) copy(s->rec.xs, fallback ? (const void*)recs.xs.data() : src.xs, n);
    } else if (cudaMemsetAsync(s->rec.cig_off, 0, 4, ctx->stream) != cudaSuccess) {
        ce = cudaGetLastError();
    }
    if (ce == cudaSuccess) ce = cudaStreamSynchronize(ctx->stream);
    if (ce != cudaSuccess) {
        cudaStreamSynchronize(ctx->stream);
        cudaGetLastError();
        spl_sample_free(s.release());
        return ctx->fail(SPL_ERR_CUDA, "copy of the sample's records failed: %s", cudaGetErrorString(ce));
    }
    ctx->stats[SPL_STAT_H2D_BYTES] = fallback ? (double)(n * 10 + 4 + nc * 4 + (want_xs ? n : 0)) : cnt.h2d_bytes;
    ctx->stats[SPL_STAT_BAM_DEVICE] = fallback ? 0.0 : 1.0;
    ctx->stats[SPL_STAT_MS_DECODE] = t1 - t0;
    ctx->stats[SPL_STAT_MS_TOTAL] = now_ms() - t0;
    *out = s.release();
    return SPL_OK;
}

int spl_sample_load_bam_groups(spl_ctx* ctx, const char* bam_path, uint32_t flags, const spl_tag_groups* groups, spl_sample** out,
                               int64_t* counts) {
    if (!ctx) return SPL_ERR_ARG;
    if (!out || !counts) return ctx->fail(SPL_ERR_ARG, "out / counts is NULL");
    if (!ctx->stream) return ctx->fail(SPL_ERR_CUDA, "context has no CUDA device; libspliser_b200 has no CPU fallback");
    if (!bam_path) return ctx->fail(SPL_ERR_ARG, "bam_path is NULL");
    if (flags & ~SPL_FLAG_XS_STRAND) return ctx->fail(SPL_ERR_ARG, "spl_sample_load_bam_groups takes SPL_FLAG_XS_STRAND only");
    TagTableHost tags;
    {
        const std::string e = build_tag_table(groups, tags);
        if (!e.empty()) return ctx->fail(SPL_ERR_ARG, "tag group table: %s", e.c_str());
    }
    const uint32_t G = (uint32_t)tags.n_groups;
    for (uint32_t g = 0; g < G; ++g) out[g] = nullptr;
    const bool want_xs = (flags & SPL_FLAG_XS_STRAND) != 0;
    const double t0 = now_ms();
    CU(cudaSetDevice(ctx->device));
    reset_stats(ctx);
    struct ReleaseScratch {                                            // on every return: cudaFree waits for the stream's work
        GroupSplitMem& m;
        ~ReleaseScratch() { m.release(); }
    } release_scratch{ctx->gsm};
    // ---- one ingest, every reference kept in header order, the group of every record found as it is parsed
    std::vector<std::string> ref_names;
    BamGpuCounts cnt;
    spl_records_view dv{};
    bool fallback = false;
    int rc = ingest_bam_device(ctx, bam_path, 0, nullptr, cnt, dv, &fallback, want_xs, &ref_names, &tags);
    if (rc) return rc;
    DevRecordArrays in{};
    const int32_t* grp = cnt.grp;
    uint64_t n = 0;
    double h2d = cnt.h2d_bytes;
    if (!fallback) {
        in = ctx->dev_rec;
        n = cnt.n_rec;
    } else {                                                           // the host reader's records and groups, uploaded once
        BamRecords recs;
        const TagTableView tv = tags.view();
        std::string e = read_bam_ctx(ctx, bam_path, 0, nullptr, recs, want_xs, &ref_names, &tv);
        if (!e.empty()) return ctx->fail(SPL_ERR_IO, "%s", e.c_str());
        n = recs.pos.size();
        const size_t nc = recs.cigar.size();
        std::vector<int32_t> chrom(n);
        for (size_t k = 0; k + 1 < recs.seg_off.size(); ++k)
            std::fill(chrom.begin() + recs.seg_off[k], chrom.begin() + recs.seg_off[k + 1], recs.seg_chrom[k]);
        Carver c;
        const size_t o_pos = c.take<int32_t>(n + 4), o_flag = c.take<uint16_t>(n + 4), o_off = c.take<uint32_t>(n + 4),
                     o_cig = c.take<uint32_t>(nc + 4), o_chr = c.take<int32_t>(n + 4), o_grp = c.take<int32_t>(n + 4),
                     o_xs = want_xs ? c.take<uint8_t>(n + 4) : 0;
        if (ctx->gsm.in.reserve(c.off + 256) != cudaSuccess) {
            cudaGetLastError();
            return ctx->fail(SPL_ERR_NOMEM, "the split of %s is not held: no device memory for the records (%zu bytes); use more GPUs", bam_path, c.off);
        }
        char* b = (char*)ctx->gsm.in.p;
        in.pos = (int32_t*)(b + o_pos); in.flag = (uint16_t*)(b + o_flag); in.cig_off = (uint32_t*)(b + o_off);
        in.cigar = (uint32_t*)(b + o_cig); in.chrom = (int32_t*)(b + o_chr);
        int32_t* d_grp = (int32_t*)(b + o_grp);
        grp = d_grp;
        in.xs = want_xs ? (uint8_t*)(b + o_xs) : nullptr;
        if (n) {
            CU(cudaMemcpyAsync(in.pos, recs.pos.data(), n * 4, cudaMemcpyHostToDevice, ctx->stream));
            CU(cudaMemcpyAsync(in.flag, recs.flag.data(), n * 2, cudaMemcpyHostToDevice, ctx->stream));
            CU(cudaMemcpyAsync(in.cigar, recs.cigar.data(), nc * 4, cudaMemcpyHostToDevice, ctx->stream));
            CU(cudaMemcpyAsync(in.chrom, chrom.data(), n * 4, cudaMemcpyHostToDevice, ctx->stream));
            CU(cudaMemcpyAsync(d_grp, recs.grp.data(), n * 4, cudaMemcpyHostToDevice, ctx->stream));
            if (want_xs) CU(cudaMemcpyAsync(in.xs, recs.xs.data(), n, cudaMemcpyHostToDevice, ctx->stream));
        }
        CU(cudaMemcpyAsync(in.cig_off, recs.cig_off.data(), (n + 1) * 4, cudaMemcpyHostToDevice, ctx->stream));
        CU(cudaStreamSynchronize(ctx->stream));                         // recs is freed at the end of this scope
        h2d = (double)(n * 18 + 4 + nc * 4 + (want_xs ? n : 0));
    }
    const double t1 = now_ms();
    // ---- stable sort by group, then one allocation with every group's columns in a slice of its own
    GroupSort gs;
    std::string e;
    rc = group_sort(ctx->gsm, in, grp, n, (int32_t)G, ctx->stream, gs, e);
    if (rc < 0) { cudaStreamSynchronize(ctx->stream); return ctx->fail(SPL_ERR_CUDA, "%s", e.c_str()); }
    if (rc > 0) { cudaStreamSynchronize(ctx->stream); return ctx->fail(SPL_ERR_NOMEM, "the split of %s is not held: %s; use more GPUs", bam_path, e.c_str()); }
    std::vector<GroupCols> cols(G);
    std::vector<size_t> slice0(G + 1);
    Carver c;
    for (uint32_t g = 0; g < G; ++g) {
        const size_t ng = (size_t)gs.n_rec[g], ncg = (size_t)gs.n_cig[g];
        c.off = (c.off + 255) & ~(size_t)255;
        slice0[g] = c.off;
        GroupCols& q = cols[g];
        q.pos = c.take<int32_t>(ng + 4); q.flag = c.take<uint16_t>(ng + 4); q.off = c.take<uint32_t>(ng + 4);
        q.cig = c.take<uint32_t>(ncg + 4); q.xs = want_xs ? c.take<uint8_t>(ng + 4) : 0;
        q.start = gs.g_start[g]; q.cig0 = gs.g_cig[g]; q.n = (uint32_t)ng; q.nc = (uint32_t)ncg;
    }
    c.off = (c.off + 255) & ~(size_t)255;
    slice0[G] = c.off;
    void* mp = nullptr;
    rc = sample_reserve(ctx, c.off, &mp);
    if (rc == SPL_ERR_NOMEM) {
        const std::string why = spl_last_error(ctx);
        return ctx->fail(SPL_ERR_NOMEM, "the split of %s needs %zu bytes of device memory for the kept records of its groups, which are "
                         "not held (%s); use more GPUs (--gpus) so that each holds fewer groups", bam_path, c.off, why.c_str());
    }
    if (rc) return rc;
    auto block = std::make_shared<SampleBlock>(mp, c.off, ctx->device);
    rc = group_gather(ctx->gsm, in, gs, cols, (char*)mp, ctx->stream, e);
    cudaError_t ce = cudaStreamSynchronize(ctx->stream);
    if (rc || ce != cudaSuccess) {
        cudaGetLastError();
        return ctx->fail(SPL_ERR_CUDA, "the split of %s failed: %s", bam_path, rc ? e.c_str() : cudaGetErrorString(ce));
    }
    std::vector<std::unique_ptr<spl_sample>> made(G);
    for (uint32_t g = 0; g < G; ++g) {
        made[g].reset(new (std::nothrow) spl_sample());
        if (!made[g]) return ctx->fail(SPL_ERR_NOMEM, "out of memory");
        spl_sample& s = *made[g];
        char* m = (char*)mp;
        s.ctx = ctx; s.device = ctx->device; s.rf = ctx->rf;
        s.mem = block; s.bytes = slice0[g + 1] - slice0[g];
        s.rec.pos = (int32_t*)(m + cols[g].pos); s.rec.flag = (uint16_t*)(m + cols[g].flag);
        s.rec.cig_off = (uint32_t*)(m + cols[g].off); s.rec.cigar = (uint32_t*)(m + cols[g].cig);
        s.rec.xs = want_xs ? (uint8_t*)(m + cols[g].xs) : nullptr;
        s.n_rec = gs.n_rec[g]; s.n_cigar = gs.n_cig[g];
        s.ref_names = ref_names;
        s.seg_ref = gs.seg_chrom[g]; s.seg_off = gs.seg_off[g];
    }
    for (uint32_t g = 0; g < G; ++g) { counts[g] = gs.n_rec[g]; out[g] = made[g].release(); }
    counts[G] = (int64_t)gs.no_value; counts[G + 1] = (int64_t)gs.no_group;
    ctx->stats[SPL_STAT_H2D_BYTES] = h2d;
    ctx->stats[SPL_STAT_BAM_DEVICE] = fallback ? 0.0 : 1.0;
    ctx->stats[SPL_STAT_MS_DECODE] = t1 - t0;
    ctx->stats[SPL_STAT_MS_TOTAL] = now_ms() - t0;
    return SPL_OK;
}

int spl_sample_fetch_records(spl_ctx* ctx, const spl_sample* s, spl_records** out) {
    if (!ctx) return SPL_ERR_ARG;
    if (!out) return ctx->fail(SPL_ERR_ARG, "out is NULL");
    *out = nullptr;
    if (!ctx->stream) return ctx->fail(SPL_ERR_CUDA, "context has no CUDA device; libspliser_b200 has no CPU fallback");
    if (!s) return ctx->fail(SPL_ERR_ARG, "sample is NULL");
    if (s->ctx != ctx) return ctx->fail(SPL_ERR_ARG, "the sample was loaded by another context");
    CU(cudaSetDevice(ctx->device));
    const size_t n = (size_t)s->n_rec, nc = (size_t)s->n_cigar;
    BamRecords r;
    r.pos.resize(n); r.flag.resize(n); r.cig_off.resize(n + 1); r.cigar.resize(nc);
    if (s->rec.xs) r.xs.resize(n);
    if (n) {
        CU(cudaMemcpyAsync(r.pos.data(), s->rec.pos, n * 4, cudaMemcpyDeviceToHost, ctx->stream));
        CU(cudaMemcpyAsync(r.flag.data(), s->rec.flag, n * 2, cudaMemcpyDeviceToHost, ctx->stream));
        if (s->rec.xs) CU(cudaMemcpyAsync(r.xs.data(), s->rec.xs, n, cudaMemcpyDeviceToHost, ctx->stream));
    }
    if (nc) CU(cudaMemcpyAsync(r.cigar.data(), s->rec.cigar, nc * 4, cudaMemcpyDeviceToHost, ctx->stream));
    CU(cudaMemcpyAsync(r.cig_off.data(), s->rec.cig_off, (n + 1) * 4, cudaMemcpyDeviceToHost, ctx->stream));
    CU(cudaStreamSynchronize(ctx->stream));
    r.seg_chrom = s->seg_ref; r.seg_off = s->seg_off;
    const bool xs = s->rec.xs != nullptr;
    *out = records_handle(std::move(r), xs);
    return *out ? SPL_OK : ctx->fail(SPL_ERR_NOMEM, "out of memory");
}

int spl_sample_process_extract(spl_ctx* ctx, const spl_sample* s, int32_t n_chrom, const char* const* chrom_names,
                               const spl_extract_opts* opts, uint32_t flags, spl_junctions** rows_out, spl_result** out) {
    if (!ctx) return SPL_ERR_ARG;
    if (!out || !rows_out) return ctx->fail(SPL_ERR_ARG, "out is NULL");
    *out = nullptr; *rows_out = nullptr;
    if (!ctx->stream) return ctx->fail(SPL_ERR_CUDA, "context has no CUDA device; libspliser_b200 has no CPU fallback");
    if (!opts) return ctx->fail(SPL_ERR_ARG, "opts is NULL");
    int rc = check_sample(ctx, s, n_chrom, chrom_names);
    if (rc) return rc;
    const double t0 = now_ms();
    CU(cudaSetDevice(ctx->device));
    std::vector<int32_t> seg_chrom;
    const spl_records_view dv = sample_view(s, n_chrom, chrom_names, seg_chrom);
    {
        SampleBinding bind(ctx, s);
        rc = extract_and_count(ctx, &dv, nullptr, n_chrom, chrom_names, opts, flags, rows_out, out);
    }
    ctx->stats[SPL_STAT_MS_TOTAL] = now_ms() - t0;
    return rc;
}

int spl_sample_recount(spl_ctx* ctx, const spl_sample* s, int32_t n_chrom, const char* const* chrom_names, int64_t n_sites,
                       const int32_t* s_chrom, const int32_t* s_pos, const uint8_t* s_strand, const int64_t* p_off, const int32_t* p_pos,
                       const int64_t* c_off, const int32_t* c_pos, uint32_t flags, int64_t* beta1_out, int64_t* beta2simple_out) {
    if (!ctx) return SPL_ERR_ARG;
    if (!ctx->stream) return ctx->fail(SPL_ERR_CUDA, "context has no CUDA device; libspliser_b200 has no CPU fallback");
    int rc = check_sample(ctx, s, n_chrom, chrom_names);
    if (rc) return rc;
    CU(cudaSetDevice(ctx->device));
    std::vector<int32_t> seg_chrom;
    const spl_records_view dv = sample_view(s, n_chrom, chrom_names, seg_chrom);
    SampleBinding bind(ctx, s);
    return spl_recount_records(ctx, &dv, n_chrom, n_sites, s_chrom, s_pos, s_strand, p_off, p_pos, c_off, c_pos, flags, beta1_out,
                               beta2simple_out);
}

namespace {
// The one routine behind spl_infer_strand*: the records are where fused_upload finds them (host arrays, or ctx->dev_rec when
// ctx->rec_on_device); xs = the host records' XS column (XS source with host records).  Only the three counters come back.
int infer_common(spl_ctx* ctx, const spl_records_view* rec, const uint8_t* xs, int32_t n_chrom, const spl_gene_strands* genes,
                 int64_t counts[3]) {
    if (!counts) return ctx->fail(SPL_ERR_ARG, "counts is NULL");
    ctx->loaded = false;
    int rc = check_view(ctx, rec, n_chrom);
    if (rc) return rc;
    GeneIndexHost gh;
    if (genes) {
        const std::string e = build_gene_index(genes, n_chrom, gh);
        if (!e.empty()) return ctx->fail(SPL_ERR_ARG, "%s", e.c_str());
    } else if (rec->n_rec > 0 && !(ctx->rec_on_device ? (const uint8_t*)ctx->dev_rec.xs : xs)) {
        return ctx->fail(SPL_ERR_ARG, "the XS source needs the records' XS strand column");
    }
    CU(cudaSetDevice(ctx->device));
    reset_stats(ctx);
    while (ctx->events.size() < 2) {
        cudaEvent_t e;
        CU(cudaEventCreate(&e));
        ctx->events.push_back(e);
    }
    rc = fused_upload(ctx, rec, n_chrom, false);
    if (rc) return drain_on_error(ctx, rc);
    CU(cudaStreamWaitEvent(ctx->stream, ctx->fpart[0].ev_up, 0));
    const uint8_t* d_xs = ctx->rec_on_device ? ctx->dev_rec.xs : nullptr;
    if (!genes && !ctx->rec_on_device && rec->n_rec > 0) {             // 1 B per record, once
        CU(ctx->d_xs.reserve((size_t)rec->n_rec + 16));
        CU(cudaMemcpyAsync(ctx->d_xs.p, xs, (size_t)rec->n_rec, cudaMemcpyHostToDevice, ctx->stream));
        ctx->stats[SPL_STAT_H2D_BYTES] += (double)rec->n_rec;
        d_xs = (const uint8_t*)ctx->d_xs.p;
    }
    Carver c;
    const size_t o_cnt = c.take<unsigned long long>(4), o_bnd = c.take<int32_t>(gh.bnd.size() + 1),
                 o_off = c.take<int32_t>(gh.bnd_off.size() + 1), o_tab = c.take<uint8_t>(gh.table.size() + 1);
    CU(ctx->d_votes.reserve(c.off + 256));
    char* vb = (char*)ctx->d_votes.p;
    unsigned long long* d_cnt = (unsigned long long*)(vb + o_cnt);
    CU(cudaMemsetAsync(d_cnt, 0, 3 * sizeof(unsigned long long), ctx->stream));
    GeneIndexDev gd{(const int32_t*)(vb + o_bnd), (const int32_t*)(vb + o_off), (const uint8_t*)(vb + o_tab), gh.m, n_chrom};
    if (genes) {
        if (!gh.bnd.empty()) CU(cudaMemcpyAsync(vb + o_bnd, gh.bnd.data(), gh.bnd.size() * 4, cudaMemcpyHostToDevice, ctx->stream));
        CU(cudaMemcpyAsync(vb + o_off, gh.bnd_off.data(), gh.bnd_off.size() * 4, cudaMemcpyHostToDevice, ctx->stream));
        if (!gh.table.empty()) CU(cudaMemcpyAsync(vb + o_tab, gh.table.data(), gh.table.size(), cudaMemcpyHostToDevice, ctx->stream));
        ctx->stats[SPL_STAT_H2D_BYTES] += (double)(gh.bnd.size() * 4 + gh.bnd_off.size() * 4 + gh.table.size());
    }
    CU(cudaEventRecord(ctx->events[0], ctx->stream));
    launch_strand_votes(ctx->frec, d_xs, ctx->fchunks, ctx->n_fchunks, genes ? &gd : nullptr, d_cnt, ctx->stream);
    CU(cudaGetLastError());
    CU(cudaEventRecord(ctx->events[1], ctx->stream));
    unsigned long long h_cnt[3] = {0, 0, 0};
    CU(cudaMemcpyAsync(h_cnt, d_cnt, sizeof h_cnt, cudaMemcpyDeviceToHost, ctx->stream));
    CU(cudaStreamSynchronize(ctx->stream));
    float ms = 0.f;
    CU(cudaEventElapsedTime(&ms, ctx->events[0], ctx->events[1]));
    ctx->stats[SPL_STAT_MS_STRAND_VOTES] = ms;
    ctx->stats[SPL_STAT_D2H_BYTES] += (double)sizeof h_cnt;
    for (int k = 0; k < 3; ++k) counts[k] = (int64_t)h_cnt[k];
    return SPL_OK;
}
}  // namespace

int spl_infer_strand_records(spl_ctx* ctx, const spl_records_view* rec, const uint8_t* xs, int32_t n_chrom,
                             const spl_gene_strands* genes, int64_t counts[3]) {
    if (!ctx) return SPL_ERR_ARG;
    if (!ctx->stream) return ctx->fail(SPL_ERR_CUDA, "context has no CUDA device; libspliser_b200 has no CPU fallback");
    if (const int rr = refuse_records(ctx, "spl_infer_strand_records")) return rr;
    const double t0 = now_ms();
    const int rc = infer_common(ctx, rec, xs, n_chrom, genes, counts);
    ctx->stats[SPL_STAT_MS_TOTAL] = now_ms() - t0;
    return rc;
}

int spl_infer_strand(spl_ctx* ctx, const char* bam_path, int32_t n_chrom, const char* const* chrom_names,
                     const spl_gene_strands* genes, int64_t counts[3]) {
    if (!ctx) return SPL_ERR_ARG;
    if (!ctx->stream) return ctx->fail(SPL_ERR_CUDA, "context has no CUDA device; libspliser_b200 has no CPU fallback");
    if (!bam_path) return ctx->fail(SPL_ERR_ARG, "bam_path is NULL");
    if (n_chrom < 0 || (n_chrom > 0 && !chrom_names)) return ctx->fail(SPL_ERR_ARG, "chrom_names is NULL");
    for (int32_t c = 0; c < n_chrom; ++c) if (!chrom_names[c]) return ctx->fail(SPL_ERR_ARG, "chromosome name %d is NULL", c);
    const bool want_xs = genes == nullptr;
    const double t0 = now_ms();
    CU(cudaSetDevice(ctx->device));
    {   // ingest as spl_extract_junctions chooses: on the device, the host reader as the fallback
        BamGpuCounts cnt;
        spl_records_view dv{};
        bool fallback = false;
        int rc = ingest_bam_device(ctx, bam_path, n_chrom, chrom_names, cnt, dv, &fallback, want_xs);
        if (rc) return rc;
        if (!fallback) {
            const double t1 = now_ms();
            ctx->rec_on_device = true;
            rc = infer_common(ctx, &dv, nullptr, n_chrom, genes, counts);
            ctx->rec_on_device = false;
            ctx->stats[SPL_STAT_MS_DECODE] = t1 - t0;
            ctx->stats[SPL_STAT_H2D_BYTES] += cnt.h2d_bytes;
            ctx->stats[SPL_STAT_BAM_DEVICE] = 1.0;
            ctx->stats[SPL_STAT_MS_TOTAL] = now_ms() - t0;
            return rc;
        }
    }
    BamRecords recs;
    std::string e = read_bam_ctx(ctx, bam_path, n_chrom, chrom_names, recs, want_xs);
    if (!e.empty()) return ctx->fail(SPL_ERR_IO, "%s", e.c_str());
    const double t1 = now_ms();
    spl_records_view v = recs.view();
    const int rc = infer_common(ctx, &v, recs.xs.data(), n_chrom, genes, counts);
    ctx->stats[SPL_STAT_MS_DECODE] = t1 - t0;
    ctx->stats[SPL_STAT_MS_TOTAL] = now_ms() - t0;
    return rc;
}

int spl_sample_infer_strand(spl_ctx* ctx, const spl_sample* s, int32_t n_chrom, const char* const* chrom_names,
                            const spl_gene_strands* genes, int64_t counts[3]) {
    if (!ctx) return SPL_ERR_ARG;
    if (!ctx->stream) return ctx->fail(SPL_ERR_CUDA, "context has no CUDA device; libspliser_b200 has no CPU fallback");
    int rc = check_sample(ctx, s, n_chrom, chrom_names);
    if (rc) return rc;
    if (!genes && !s->rec.xs) return ctx->fail(SPL_ERR_ARG, "the XS source needs a sample loaded with SPL_FLAG_XS_STRAND");
    const double t0 = now_ms();
    CU(cudaSetDevice(ctx->device));
    std::vector<int32_t> seg_chrom;
    const spl_records_view dv = sample_view(s, n_chrom, chrom_names, seg_chrom);
    {
        SampleBinding bind(ctx, s);
        rc = infer_common(ctx, &dv, nullptr, n_chrom, genes, counts);
    }
    ctx->stats[SPL_STAT_MS_TOTAL] = now_ms() - t0;
    return rc;
}

int64_t spl_sample_n_records(const spl_sample* s) { return s ? s->n_rec : 0; }
int64_t spl_sample_device_bytes(const spl_sample* s) { return s ? (int64_t)s->bytes : 0; }

void spl_sample_free(spl_sample* s) {
    delete s;                             // the last sample of an allocation frees it (SampleBlock)
}

int spl_resident_load(spl_ctx* ctx, const spl_records_view* rec, int32_t n_chrom, int64_t n_junc, const int32_t* j_chrom,
                      const int32_t* j_left, const int32_t* j_right, const int64_t* j_score, const uint8_t* j_strand, uint32_t flags) {
    if (!ctx) return SPL_ERR_ARG;
    if (!ctx->stream) return ctx->fail(SPL_ERR_CUDA, "context has no CUDA device; libspliser_b200 has no CPU fallback");
    if (const int rr = refuse_records(ctx, "spl_resident_load")) return rr;
    int rc = load_common(ctx, rec, n_chrom, n_junc, j_chrom, j_left, j_right, j_score, j_strand, flags, false);
    if (rc) return drain_on_error(ctx, rc);
    CU(cudaStreamSynchronize(ctx->stream));
    collect_expand_ms(ctx);
    // stabbing variant: the raw records are not needed once expanded
    for (int p = 0; p < MAX_PARTS; ++p) ctx->part[p].d_rec.release();
    return SPL_OK;
}

int spl_resident_count(spl_ctx* ctx, int iters, double* stats_out) {
    if (!ctx) return SPL_ERR_ARG;
    if (!ctx->loaded) return ctx->fail(SPL_ERR_ARG, "spl_resident_count without a successful spl_resident_load");
    if (iters < 1) return ctx->fail(SPL_ERR_ARG, "iters must be >= 1");
    CU(cudaSetDevice(ctx->device));
    while (ctx->events.size() < (size_t)iters * 6) {
        cudaEvent_t e;
        CU(cudaEventCreate(&e));
        ctx->events.push_back(e);
    }
    // Fused variant, clean regime: the whole per-sample path is inside the timed region -- site table + graph from the
    // resident junction table (K1), counters zeroed, counting kernel, prefix scan + beta2 gather + SSE.  (The stabbing
    // variant times its counting pass over the layout prepared at load time; the dirty regime keeps its host-built graph.)
    const bool regraph = ctx->loaded_variant == SPL_VARIANT_FUSED && ctx->res_clean && ctx->graph_on_device;
    for (int attempt = 0;; ++attempt) {
    const unsigned long long launches0 = g_kernel_launches.load();
    for (int it = 0; it < iters; ++it) {
        cudaEvent_t* ev = ctx->events.data() + (size_t)it * 6;
        CU(cudaEventRecord(ev[5], ctx->stream));
        if (regraph) {
            std::string e;
            if (!graph_build_device(ctx->gbm, nullptr, nullptr, nullptr, nullptr, nullptr, ctx->res_n_junc, ctx->res_n_chrom, ctx->res_max_pos,
                                    ctx->res_stranded, ctx->stream, 2, ctx->gdev, ctx->gcnt, e))
                return ctx->fail(SPL_ERR_CUDA, "%s", e.c_str());
            adopt_device_graph(ctx);
            int rc = alloc_counters_outputs(ctx, ctx->gcnt.S, ctx->gcnt.E);
            if (rc) return rc;
        }
        int rc = count_pass(ctx, ev);
        if (rc) return rc;
    }
    CU(cudaStreamSynchronize(ctx->stream));
    {
        bool again = false;
        const int orc = hot_queue_overflow(ctx, &again);
        if (orc) return orc;
        if (again && attempt < 4) continue;
    }
    float total = 0, b1 = 0, sp = 0, fin = 0, gr = 0;
    CU(cudaEventElapsedTime(&total, ctx->events[5], ctx->events[(size_t)(iters - 1) * 6 + 4]));
    for (int it = 0; it < iters; ++it) {
        cudaEvent_t* ev = ctx->events.data() + (size_t)it * 6;
        float a, b, c, d, g0;
        CU(cudaEventElapsedTime(&a, ev[0], ev[1])); CU(cudaEventElapsedTime(&b, ev[1], ev[2]));
        CU(cudaEventElapsedTime(&c, ev[2], ev[3])); CU(cudaEventElapsedTime(&d, ev[3], ev[4]));
        CU(cudaEventElapsedTime(&g0, ev[5], ev[0]));
        b1 += b; sp += c; fin += a + d; gr += g0;
    }
    ctx->stats[SPL_STAT_MS_TOTAL] = total; ctx->stats[SPL_STAT_MS_BETA1] = b1;
    ctx->stats[SPL_STAT_MS_SPLICED] = sp; ctx->stats[SPL_STAT_MS_FINAL] = fin;
    ctx->stats[SPL_STAT_MS_GRAPH_DEV] = gr;
    ctx->stats[SPL_STAT_GRAPH_TIMED] = regraph ? 1.0 : 0.0;
    ctx->stats[SPL_STAT_LAUNCHES] = (double)(g_kernel_launches.load() - launches0) / (double)iters;   // kernels launched per timed pass (counted)
    break;
    }
    if (stats_out) memcpy(stats_out, ctx->stats, sizeof ctx->stats);
    return SPL_OK;
}

int spl_resident_fetch(spl_ctx* ctx, spl_result** out) {
    if (!ctx) return SPL_ERR_ARG;
    if (!out) return ctx->fail(SPL_ERR_ARG, "out is NULL");
    *out = nullptr;
    if (!ctx->loaded) return ctx->fail(SPL_ERR_ARG, "nothing loaded");
    CU(cudaSetDevice(ctx->device));
    return fetch(ctx, out);
}

int spl_build_site_table(int32_t n_chrom, int64_t n_junc, const int32_t* j_chrom, const int32_t* j_left, const int32_t* j_right,
                         const int64_t* j_score, const uint8_t* j_strand, uint32_t flags, spl_result** out, char* err, int err_len) {
    if (!out) return SPL_ERR_ARG;
    *out = nullptr;
    SiteGraph h;
    std::string e = (n_junc > 0 && !j_score) ? std::string("NULL j_score")
                                              : build_site_graph(n_chrom, n_junc, j_chrom, j_left, j_right, j_strand,
                                                                 (flags & SPL_FLAG_STRANDED) != 0, h);
    if (!e.empty()) {
        if (err && err_len > 0) snprintf(err, (size_t)err_len, "%s", e.c_str());
        return SPL_ERR_ARG;
    }
    const size_t S = (size_t)h.n_sites, E = h.pc_pos.size();
    spl_result* r = result_alloc(S, E, h.cp_pos.size(), false);
    if (!r) {
        if (err && err_len > 0) snprintf(err, (size_t)err_len, "out of memory");
        return SPL_ERR_NOMEM;
    }
    result_from_host_graph(r, h);
    for (size_t t = 0; t < S; ++t) {
        r->alpha[t] = 0; r->beta1[t] = 0; r->beta2s[t] = 0; r->beta2c[t] = 0; r->beta2w[t] = 0.0; r->sse[t] = 0.0;
        for (int64_t k = h.inc_off[t]; k < h.inc_off[t + 1]; ++k) r->alpha[t] += j_score[h.inc_line[(size_t)k]];
    }
    for (size_t x = 0; x < E; ++x) {
        r->pc_cnt[x] = 0;
        for (int64_t k = h.einc_off[x]; k < h.einc_off[x + 1]; ++k) r->pc_cnt[x] += j_score[h.einc_line[(size_t)k]];
    }
    *out = r;
    return SPL_OK;
}

int64_t spl_result_n_sites(const spl_result* r) { return r ? r->n : 0; }
const int32_t* spl_result_chrom(const spl_result* r) { return r->chrom; }
const int32_t* spl_result_pos(const spl_result* r) { return r->pos; }
const uint8_t* spl_result_strand(const spl_result* r) { return r->strand; }
const int64_t* spl_result_alpha(const spl_result* r) { return r->alpha; }
const int64_t* spl_result_beta1(const spl_result* r) { return r->beta1; }
const int64_t* spl_result_beta2simple(const spl_result* r) { return r->beta2s; }
const int64_t* spl_result_beta2cryptic(const spl_result* r) { return r->beta2c; }
const double* spl_result_beta2weighted(const spl_result* r) { return r->beta2w; }
const double* spl_result_sse(const spl_result* r) { return r->sse; }
const int64_t* spl_result_first_line(const spl_result* r) { return r->first_line; }
const int64_t* spl_result_partner_off(const spl_result* r) { return r->pc_off; }
const int32_t* spl_result_partner_pos(const spl_result* r) { return r->pc_pos; }
const int64_t* spl_result_partner_cnt(const spl_result* r) { return r->pc_cnt; }
const int64_t* spl_result_comp_off(const spl_result* r) { return r->cp_off; }
const int32_t* spl_result_comp_pos(const spl_result* r) { return r->cp_pos; }
void spl_result_free(spl_result* r) {
    if (!r) return;
    arena_put(Arena{r->arena, r->bytes, r->pinned});
    delete r;
}

void* spl_host_alloc(size_t bytes) {
    void* p = nullptr;
    if (cudaHostAlloc(&p, bytes ? bytes : 1, cudaHostAllocDefault) != cudaSuccess) { cudaGetLastError(); return nullptr; }
    return p;
}
void spl_host_free(void* p) { if (p) cudaFreeHost(p); }

}  // extern "C"
