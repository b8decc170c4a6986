// host_text.cpp -- the text side of the CLI, native: Gene column lookup, the .SpliSER.tsv writer and the `combine`
// merge driver (SURVEY 8(f) rows 2 and 4).  Host only, no CUDA: once the counting takes tens of milliseconds the
// per-row Python string work around it (seconds) is what a user waits for.
//
// Restates, inside /root/reference/SpliSER_v0_1_8.py ("S:"): binary_gene_search (S:118-173), outputBedFile (S:641-664),
// outputCombinedLines (S:722-740) and the lock-step merge of combine (S:791-917) with its order dependence (a gap of
// sample k sees the partners / competitors / strand collected from the samples before k only, SURVEY F7).  Output is
// byte-identical to the reference's: Python's str(int), "{:.3f}" / "{:.5f}" (correctly rounded, like glibc printf),
// str(float) (shortest round-trip digits, exponent form outside 1e-4 <= |v| < 1e16), str(dict), str(list).
#include <algorithm>
#include <atomic>
#include <charconv>
#include <cerrno>
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <limits>
#include <mutex>
#include <condition_variable>
#include <exception>
#include <string>
#include <string_view>
#include <system_error>
#include <thread>
#include <unordered_map>
#include <vector>

#include "../../include/spliser_b200.h"
#include "junction_filter.h"

namespace {

void set_err(char* err, int err_len, const char* fmt, ...) {
    if (!err || err_len <= 0) return;
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(err, (size_t)err_len, fmt, ap);
    va_end(ap);
}

// ---- buffered text output -----------------------------------------------------------------------------------------
struct Out {
    FILE* f = nullptr;                 // sink: a file ...
    std::string* mem = nullptr;        // ... or a string (the parallel formatters of spl_combine_write)
    std::vector<char> buf;
    size_t n = 0;
    bool bad = false;
    explicit Out(FILE* fp) : f(fp), buf(1 << 20) {}
    explicit Out(std::string* m) : mem(m), buf(1 << 16) {}
    void flush() {
        if (n && f && fwrite(buf.data(), 1, n, f) != n) bad = true;
        if (n && mem) mem->append(buf.data(), n);
        n = 0;
    }
    char* room(size_t need) {
        if (n + need > buf.size()) flush();
        if (need > buf.size()) buf.resize(need);
        return buf.data() + n;
    }
    void put(const char* s, size_t len) {
        memcpy(room(len), s, len);
        n += len;
    }
    void put(std::string_view s) { put(s.data(), s.size()); }
    void ch(char c) { *room(1) = c; n += 1; }
    void i64(long long v) {                                   // str(int)
        char* p = room(24);
        auto r = std::to_chars(p, p + 24, v);
        n += (size_t)(r.ptr - p);
    }
    void fixed(double v, int prec) {                          // "{0:.<prec>f}".format(v): correctly rounded like printf
        char* p = room(400);
        if (v - v != 0.0) { n += (size_t)snprintf(p, 400, "%.*f", prec, v); return; }     // inf / nan spelled by printf
        auto r = std::to_chars(p, p + 400, v, std::chars_format::fixed, prec);
        n += (size_t)(r.ptr - p);
    }
    void pyfloat(double v) {                                  // str(float)
        char* p = room(40);
        if (v != v) { memcpy(p, "nan", 3); n += 3; return; }
        if (v == 0.0) { size_t k = std::signbit(v) ? 4 : 3; memcpy(p, std::signbit(v) ? "-0.0" : "0.0", k); n += k; return; }
        if (v - v != 0.0) { size_t k = v < 0 ? 4 : 3; memcpy(p, v < 0 ? "-inf" : "inf", k); n += k; return; }
        char t[40];
        auto r = std::to_chars(t, t + 40, v, std::chars_format::scientific);   // shortest round trip: [-]d[.ddd]e[+-]XX
        size_t len = (size_t)(r.ptr - t);
        size_t epos = 0;
        while (epos < len && t[epos] != 'e') ++epos;
        int e10 = atoi(std::string(t + epos + 1, len - epos - 1).c_str());
        if (e10 < -4 || e10 >= 16) { memcpy(p, t, len); n += len; return; }    // float_repr_style 'r': exponent form
        char* q = p;
        size_t i = 0;
        if (t[0] == '-') { *q++ = '-'; i = 1; }
        char dig[24];
        int nd = 0;
        for (; i < epos; ++i) if (t[i] != '.') dig[nd++] = t[i];
        int decpt = e10 + 1;
        if (decpt <= 0) {
            *q++ = '0'; *q++ = '.';
            for (int z = 0; z < -decpt; ++z) *q++ = '0';
            memcpy(q, dig, (size_t)nd); q += nd;
        } else if (decpt >= nd) {
            memcpy(q, dig, (size_t)nd); q += nd;
            for (int z = 0; z < decpt - nd; ++z) *q++ = '0';
            *q++ = '.'; *q++ = '0';
        } else {
            memcpy(q, dig, (size_t)decpt); q += decpt;
            *q++ = '.';
            memcpy(q, dig + decpt, (size_t)(nd - decpt)); q += nd - decpt;
        }
        n += (size_t)(q - p);
    }
};

inline std::string_view tab_get(const spl_strtab* t, int64_t i) {
    return std::string_view(t->blob + t->off[i], (size_t)(t->off[i + 1] - t->off[i]));
}

inline long long floordiv2(long long a) { return a >= 0 ? a / 2 : -((-a + 1) / 2); }

// runs `work` on nt threads (the caller's included); a thread that cannot be started just means fewer workers
template <class F> void run_parallel(int nt, F& work) {
    std::vector<std::thread> pool;
    for (int t = 1; t < nt; ++t) {
        try { pool.emplace_back([&work]() { work(); }); } catch (const std::system_error&) { break; }
    }
    work();
    for (auto& th : pool) th.join();
}

int worker_count(int requested, size_t jobs) {
    if (requested <= 0) {                              // SPLISER_HOST_THREADS bounds the text layer's workers (default: all cores)
        const char* env = getenv("SPLISER_HOST_THREADS");
        if (env && atoi(env) > 0) requested = atoi(env);
    }
    int n = requested > 0 ? requested : (int)std::thread::hardware_concurrency();
    if (n < 1) n = 1;
    if (n > 64) n = 64;
    return (int)std::min<size_t>((size_t)n, std::max<size_t>(jobs, 1));
}

// Formats [0, total) in blocks of `block` items on up to `threads` workers (0 = every hardware thread) and writes the
// blocks to `f` in order.  fmt(lo, hi, out) appends the text of items [lo, hi).
template <class F> bool write_blocks(FILE* f, size_t total, size_t block, int threads, F fmt) {
    const size_t n_blocks = (total + block - 1) / block;
    if (n_blocks == 0) return true;
    const int nt = worker_count(threads, n_blocks);
    if (nt <= 1 || n_blocks == 1) {                                       // nothing to overlap
        std::string text;
        for (size_t j = 0; j < n_blocks; ++j) {
            text.clear();
            Out o(&text);
            fmt(j * block, std::min(total, (j + 1) * block), o);
            o.flush();
            if (fwrite(text.data(), 1, text.size(), f) != text.size()) return false;
        }
        return true;
    }
    // The workers format blocks in index order of claim; the calling thread writes block j as soon as it is ready, while the
    // later blocks are still being formatted.  A worker does not start block j before block j - window has been written,
    // which bounds the text held in memory to `window` blocks whatever the size of the table.
    const size_t window = (size_t)nt * 3;
    std::vector<std::string> slot(window);
    std::vector<char> ready(n_blocks, 0);
    std::mutex mu;
    std::condition_variable cv_ready, cv_room;
    size_t written = 0, next = 0;
    bool failed = false;
    std::exception_ptr worker_error;
    auto work = [&]() {
        for (;;) {
            size_t j;
            {
                std::unique_lock<std::mutex> lk(mu);
                if (failed || next >= n_blocks) return;
                j = next++;
                cv_room.wait(lk, [&] { return failed || j < written + window; });
                if (failed) return;
            }
            std::string& text = slot[j % window];
            try {
                text.clear();
                Out o(&text);
                fmt(j * block, std::min(total, (j + 1) * block), o);
                o.flush();
            } catch (...) {
                std::lock_guard<std::mutex> lk(mu);
                if (!worker_error) worker_error = std::current_exception();
                failed = true;
                cv_ready.notify_all(); cv_room.notify_all();
                return;
            }
            {
                std::lock_guard<std::mutex> lk(mu);
                ready[j] = 1;
            }
            cv_ready.notify_all();
        }
    };
    std::vector<std::thread> pool;
    for (int t = 0; t < nt; ++t) {
        try { pool.emplace_back(work); } catch (const std::system_error&) { break; }
    }
    bool ok = true;
    if (pool.empty()) {                                                   // no thread could be started: format here
        std::lock_guard<std::mutex> lk(mu);
        failed = true;
        ok = false;
    }
    for (size_t j = 0; ok && j < n_blocks; ++j) {
        {
            std::unique_lock<std::mutex> lk(mu);
            cv_ready.wait(lk, [&] { return failed || ready[j]; });
            if (failed) { ok = false; break; }
        }
        const std::string& text = slot[j % window];
        if (fwrite(text.data(), 1, text.size(), f) != text.size()) ok = false;
        {
            std::lock_guard<std::mutex> lk(mu);
            written = j + 1;
            if (!ok) failed = true;
        }
        cv_room.notify_all();
    }
    {
        std::lock_guard<std::mutex> lk(mu);
        if (!ok) failed = true;
    }
    cv_room.notify_all(); cv_ready.notify_all();
    for (auto& th : pool) th.join();
    if (worker_error) std::rethrow_exception(worker_error);
    if (pool.empty()) {                                                   // sequential fallback, from the start
        std::string text;
        for (size_t j = 0; j < n_blocks; ++j) {
            text.clear();
            Out o(&text);
            fmt(j * block, std::min(total, (j + 1) * block), o);
            o.flush();
            if (fwrite(text.data(), 1, text.size(), f) != text.size()) return false;
        }
        return true;
    }
    return ok;
}

}  // namespace

// ======================================================================================================= gene lookup
extern "C" int spl_gene_search(int64_t n_genes, const int32_t* g_left, const int32_t* g_right, const int32_t* g_strand,
                               int64_t n, const int32_t* pos, const int32_t* strand, int32_t plus_id, int32_t minus_id,
                               int is_stranded, int32_t* out_idx) {
    if (n_genes < 0 || n < 0 || (n_genes && (!g_left || !g_right || !g_strand)) || (n && (!pos || !strand || !out_idx)))
        return SPL_ERR_ARG;
    const long long length = n_genes;
    auto search = [&](int64_t lo, int64_t hi) {
    for (int64_t s = lo; s < hi; ++s) {
        if (length == 0) { out_idx[s] = -1; continue; }
        const long long p = pos[s];
        const int32_t st = strand[s];
        const bool any_strand = !is_stranded || (st != plus_id && st != minus_id);
        auto strand_ok = [&](long long k) { return st == g_strand[k] || any_strand; };
        long long idx = length / 2, past_max = length, past_min = 0, last_idx = -1, new_idx = idx;
        bool stuck = false, found = false;
        while (!stuck && !found) {                                          // S:142-160
            const long long gl = g_left[idx], gr = g_right[idx];
            if (p >= gl && p <= gr && strand_ok(idx)) { found = true; break; }
            else if (p >= gr) { new_idx = idx + floordiv2(past_max - idx); past_min = idx; }
            else if (p <= gl) { new_idx = idx - floordiv2(idx - past_min); past_max = idx; if (idx == 1) new_idx = 0; }
            if (idx != last_idx) { last_idx = idx; idx = new_idx; }
            else stuck = true;
        }
        if (!found && stuck) {                                              // S:162-169: the window moves with idx
            for (int i = -3; i < 3; ++i) {
                const long long k = idx + i;
                if (k >= 0 && k < length - 1 && p >= g_left[k] && p <= g_right[k] && strand_ok(k)) {
                    found = true; stuck = false; idx = k;
                }
            }
        }
        out_idx[s] = (found && !stuck) ? (int32_t)idx : -1;
    }
    };
    // the sites are independent: blocks of them on every core
    const int64_t block = 8192;
    const int64_t n_blocks = (n + block - 1) / block;
    if (n_blocks <= 1) { search(0, n); return SPL_OK; }
    std::atomic<int64_t> next{0};
    auto work = [&]() {
        for (int64_t b; (b = next.fetch_add(1)) < n_blocks;) search(b * block, std::min(n, (b + 1) * block));
    };
    try {
        run_parallel(worker_count(0, (size_t)n_blocks), work);
    } catch (const std::exception&) {
        return SPL_ERR_NOMEM;
    }
    return SPL_OK;
}

// ================================================================================================== .SpliSER.tsv writer
namespace {
const char PROCESS_HEADER[] =
    "Region\tSite\tStrand\tGene\tSSE\talpha_count\tbeta1_count\tbeta2Simple_count\tbeta2Cryptic_count\t"
    "beta2Cryptic_weighted\tPartners\tCompetitors\n";
const char COMBINE_HEADER[] =
    "Sample\tRegion\tSite\tStrand\tGene\tSSE\talpha_count\tbeta1_count\tbeta2Simple_count\tbeta2Cryptic_count\t"
    "beta2_weighted\tPartners\tCompetitors\n";
}

extern "C" int spl_write_process_tsv(const char* path, const spl_site_columns* t, const spl_strtab* chrom_names,
                                     const spl_strtab* strand_texts, const int32_t* line_strand,
                                     const spl_strtab* gene_names, const int32_t* site_gene, int cryptic,
                                     char* err, int err_len) {
    if (!path || !t || !chrom_names || !strand_texts || (t->n_sites && !line_strand)) {
        set_err(err, err_len, "spl_write_process_tsv: null argument");
        return SPL_ERR_ARG;
    }
    for (int64_t i = 0; i < t->n_sites; ++i) {
        const int32_t ci = t->chrom[i];
        const int32_t sid = line_strand[t->first_line[i]];
        if (ci < 0 || ci >= chrom_names->n || sid < 0 || sid >= strand_texts->n ||
            (site_gene && gene_names && site_gene[i] >= gene_names->n)) {
            set_err(err, err_len, "spl_write_process_tsv: site %lld refers to a name outside its table", (long long)i);
            return SPL_ERR_ARG;
        }
    }
    FILE* f = fopen(path, "w");
    if (!f) { set_err(err, err_len, "cannot open %s: %s", path, strerror(errno)); return SPL_ERR_IO; }
    bool ok = fwrite(PROCESS_HEADER, 1, sizeof(PROCESS_HEADER) - 1, f) == sizeof(PROCESS_HEADER) - 1;
    auto rows = [&](size_t lo, size_t hi, Out& o) {
        for (size_t i = lo; i < hi; ++i) {
            o.put(tab_get(chrom_names, t->chrom[i])); o.ch('\t');
            o.i64(t->pos[i]); o.ch('\t');
            o.put(tab_get(strand_texts, line_strand[t->first_line[i]])); o.ch('\t');
            if (site_gene && gene_names && site_gene[i] >= 0) o.put(tab_get(gene_names, site_gene[i]));
            else o.put("NA", 2);
            o.ch('\t');
            o.fixed(t->sse[i], 3); o.ch('\t');
            o.i64(t->alpha[i]); o.ch('\t');
            o.i64(t->beta1[i]); o.ch('\t');
            o.i64(t->beta2simple[i]); o.ch('\t');
            if (cryptic) {
                o.i64(t->beta2cryptic[i]); o.ch('\t');
                o.fixed(t->beta2weighted[i], 5); o.ch('\t');
            } else {
                o.put("NA\tNA\t", 6);
            }
            o.ch('{');                                                       // str(dict): PartnerCounts, S:662
            for (int64_t e = t->partner_off[i]; e < t->partner_off[i + 1]; ++e) {
                if (e > t->partner_off[i]) o.put(", ", 2);
                o.i64(t->partner_pos[e]); o.put(": ", 2); o.i64(t->partner_cnt[e]);
            }
            o.put("}\t[", 3);                                                // str(list): CompetitorPos, S:663
            for (int64_t e = t->comp_off[i]; e < t->comp_off[i + 1]; ++e) {
                if (e > t->comp_off[i]) o.put(", ", 2);
                o.i64(t->comp_pos[e]);
            }
            o.put("]\n", 2);
        }
    };
    try {
        ok = ok && write_blocks(f, (size_t)t->n_sites, 16384, 0, rows);
    } catch (const std::exception& e) {
        fclose(f);
        set_err(err, err_len, "spl_write_process_tsv: %s", e.what());
        return SPL_ERR_NOMEM;
    }
    if (fclose(f) != 0 || !ok) { set_err(err, err_len, "write to %s failed", path); return SPL_ERR_IO; }
    return SPL_OK;
}

// ======================================================================================================= combine merge
namespace {

struct Interner {
    std::unordered_map<std::string, int32_t> map;
    std::vector<std::string> names;
    int32_t last = -1;                                 // consecutive rows mostly repeat the region / strand / gene
    int32_t id(std::string_view s) {
        if (last >= 0 && names[(size_t)last] == s) return last;
        if (names.size() <= 8) {                       // a handful of strands / regions: no hashing
            for (size_t k = 0; k < names.size(); ++k)
                if (names[k] == s) return last = (int32_t)k;
        }
        auto it = map.find(std::string(s));
        if (it != map.end()) return last = it->second;
        int32_t k = (int32_t)names.size();
        names.emplace_back(s);
        map.emplace(names.back(), k);
        return last = k;
    }
};

struct Sample {
    std::string title;
    // one entry per data row of the .SpliSER.tsv, file order
    std::vector<int32_t> region, pos, strand, gene;
    std::vector<int64_t> alpha, beta1, beta2s, beta2c;
    std::vector<double> beta2w;
    std::vector<double> sse;                           // column 4 as float(text); NaN when it is not a number (only combineShallow reads it)
    std::vector<uint8_t> has_cryptic;                  // column 8 != "NA"
    std::vector<int64_t> p_off, c_off;                 // CSR of the Partners / Competitors columns
    std::vector<int32_t> p_key, c_key;
    std::vector<int64_t> p_cnt;
    std::vector<int32_t> runs;                         // consecutive distinct regions (for the region order, S:761-789)
    // gaps of this sample in the argument layout of spl_recount
    std::vector<int32_t> g_region, g_pos;
    std::vector<uint8_t> g_strand;
    std::vector<int64_t> gp_off{0}, gc_off{0};
    std::vector<int32_t> gp_pos, gc_pos;
    std::vector<int64_t> r_beta1, r_beta2s;            // re-count results handed back by the caller
    bool have_recount = false;
};

struct Merged {
    int32_t region, pos, gene;
    int64_t cell;                                      // first of n_samples entries in `cells`
    int64_t part_off, comp_off;                        // final unions in `u_part` / `u_comp`
};

}  // namespace

struct spl_combine {
    Interner regions, strands, genes;
    std::vector<Sample> samples;
    std::vector<Merged> merged;
    std::vector<int64_t> cells;                        // per (merged site, sample): row index, or -(gap id)-2, or -1 = not emitted
    std::vector<int32_t> u_part, u_comp;
    std::vector<int64_t> u_part_end, u_comp_end;
    int64_t n_filled = 0;
    int n_threads = 0;                                 // 0 = every hardware thread
    bool merged_done = false;
    std::string err;
};

namespace {

// int(text) for the plain decimal forms a .SpliSER.tsv holds
bool parse_i64(std::string_view s, int64_t* out) {
    while (!s.empty() && (s.front() == ' ')) s.remove_prefix(1);
    while (!s.empty() && (s.back() == ' ')) s.remove_suffix(1);
    if (!s.empty() && s.front() == '+') s.remove_prefix(1);
    if (s.empty()) return false;
    long long v = 0;
    auto r = std::from_chars(s.data(), s.data() + s.size(), v);
    if (r.ec != std::errc() || r.ptr != s.data() + s.size()) return false;
    *out = v;
    return true;
}

bool parse_f64(std::string_view s, double* out) {
    std::string z(s);
    char* end = nullptr;
    errno = 0;
    double v = strtod(z.c_str(), &end);
    if (end == z.c_str()) return false;
    while (*end == ' ') ++end;
    if (*end) return false;
    *out = v;
    return true;
}

// "{200: 5, 300: 3}" -> keys / counts;  "[200, 300]" -> keys
bool parse_partners(std::string_view s, std::vector<int32_t>& key, std::vector<int64_t>& cnt) {
    while (!s.empty() && s.front() == ' ') s.remove_prefix(1);
    while (!s.empty() && s.back() == ' ') s.remove_suffix(1);
    if (s.size() < 2 || s.front() != '{' || s.back() != '}') return false;
    s = s.substr(1, s.size() - 2);
    if (s.find_first_not_of(' ') == std::string_view::npos) return true;
    size_t first = key.size();
    while (true) {
        size_t comma = s.find(',');
        std::string_view item = s.substr(0, comma);
        size_t colon = item.find(':');
        if (colon == std::string_view::npos) return false;
        int64_t k, c;
        if (!parse_i64(item.substr(0, colon), &k) || !parse_i64(item.substr(colon + 1), &c)) return false;
        bool dup = false;                                  // a dict keeps the first position of a repeated key, the last value
        for (size_t e = first; e < key.size(); ++e) if (key[e] == (int32_t)k) { cnt[e] = c; dup = true; }
        if (!dup) { key.push_back((int32_t)k); cnt.push_back(c); }
        if (comma == std::string_view::npos) break;
        s.remove_prefix(comma + 1);
    }
    return true;
}

bool parse_competitors(std::string_view s, std::vector<int32_t>& key) {
    while (!s.empty() && s.front() == ' ') s.remove_prefix(1);
    while (!s.empty() && s.back() == ' ') s.remove_suffix(1);
    if (s.size() < 2 || s.front() != '[' || s.back() != ']') return false;
    s = s.substr(1, s.size() - 2);
    if (s.find_first_not_of(' ') == std::string_view::npos) return true;
    while (true) {
        size_t comma = s.find(',');
        int64_t k;
        if (!parse_i64(s.substr(0, comma), &k)) return false;
        key.push_back((int32_t)k);
        if (comma == std::string_view::npos) break;
        s.remove_prefix(comma + 1);
    }
    return true;
}

bool read_file(const char* path, std::string& data) {
    FILE* f = fopen(path, "rb");
    if (!f) return false;
    char chunk[1 << 16];
    size_t k;
    while ((k = fread(chunk, 1, sizeof chunk, f)) > 0) data.append(chunk, k);
    bool ok = !ferror(f);
    fclose(f);
    return ok;
}

inline bool is_py_space(char c) { return c == ' ' || c == '\t' || c == '\n' || c == '\r' || c == '\v' || c == '\f'; }

}  // namespace

extern "C" int spl_combine_create(spl_combine** out) {
    if (!out) return SPL_ERR_ARG;
    *out = new (std::nothrow) spl_combine();
    return *out ? SPL_OK : SPL_ERR_NOMEM;
}

extern "C" void spl_combine_destroy(spl_combine* c) { delete c; }

extern "C" int spl_combine_set_threads(spl_combine* c, int n_threads) {
    if (!c || n_threads < 0) return SPL_ERR_ARG;
    c->n_threads = n_threads;
    return SPL_OK;
}

extern "C" const char* spl_combine_last_error(const spl_combine* c) { return c ? c->err.c_str() : "null spl_combine"; }

// One sample = one row of the samples file (S:750-759): its title and its .SpliSER.tsv.  The header line is skipped
// (S:799-800); every other line is rstrip()ped and split on tabs (S:836) and must have the twelve columns of S:643.
// Region / strand / gene ids are local to the sample here (samples parse concurrently); spl_combine_add_samples
// renumbers them into the shared tables in sample order.
namespace {
struct LocalTables { Interner regions, strands, genes; };

int parse_sample(const char* title, const char* tsv_path, Sample& s, LocalTables& lt, std::string& err) {
    std::string data;
    if (!read_file(tsv_path, data)) { err = std::string("cannot read ") + tsv_path; return SPL_ERR_IO; }
    s.title = title;
    s.p_off.push_back(0);
    s.c_off.push_back(0);
    size_t at = 0, line_no = 0;
    int32_t last_region = -1;
    try {
        while (at < data.size()) {
            const char* nlp = (const char*)memchr(data.data() + at, '\n', data.size() - at);
            size_t end = nlp ? (size_t)(nlp - data.data()) : data.size();
            std::string_view line(data.data() + at, end - at);
            at = nlp ? end + 1 : data.size();
            if (line_no++ == 0) continue;
            while (!line.empty() && is_py_space(line.back())) line.remove_suffix(1);
            std::string_view col[12];
            int nc = 0;
            {                                                       // further columns are ignored (vals[11] is the 12th)
                const char* q = line.data();
                const char* const e = q + line.size();
                const char* field = q;
                for (; q < e && nc < 12; ++q)
                    if (*q == '\t') { col[nc++] = std::string_view(field, (size_t)(q - field)); field = q + 1; }
                if (nc < 12) col[nc++] = std::string_view(field, (size_t)(e - field));
            }
            if (nc < 12) {
                err = std::string(tsv_path) + ": line " + std::to_string(line_no) + " has fewer than 12 tab-separated columns";
                return SPL_ERR_ARG;
            }
            int64_t pos, a, b1, b2, bc = 0;
            double bw = 0.0;
            bool ok = parse_i64(col[1], &pos) && parse_i64(col[5], &a) && parse_i64(col[6], &b1) && parse_i64(col[7], &b2);
            const bool has_c = col[8] != "NA";
            if (ok && has_c) ok = parse_i64(col[8], &bc) && parse_f64(col[9], &bw);
            ok = ok && parse_partners(col[10], s.p_key, s.p_cnt) && parse_competitors(col[11], s.c_key);
            if (!ok) {
                err = std::string(tsv_path) + ": line " + std::to_string(line_no) + " is not a .SpliSER.tsv row";
                return SPL_ERR_ARG;
            }
            const int32_t rid = lt.regions.id(col[0]);
            if (rid != last_region) { s.runs.push_back(rid); last_region = rid; }
            s.region.push_back(rid);
            s.pos.push_back((int32_t)pos);
            s.strand.push_back(lt.strands.id(col[2]));
            s.gene.push_back(lt.genes.id(col[3]));
            s.alpha.push_back(a); s.beta1.push_back(b1); s.beta2s.push_back(b2); s.beta2c.push_back(bc);
            s.beta2w.push_back(bw);
            {
                double sse = 0.0;
                s.sse.push_back(parse_f64(col[4], &sse) ? sse : std::numeric_limits<double>::quiet_NaN());
            }
            s.has_cryptic.push_back(has_c ? 1 : 0);
            s.p_off.push_back((int64_t)s.p_key.size());
            s.c_off.push_back((int64_t)s.c_key.size());
        }
    } catch (const std::bad_alloc&) {
        err = "out of memory";
        return SPL_ERR_NOMEM;
    }
    return SPL_OK;
}

}  // namespace

extern "C" int spl_combine_add_samples(spl_combine* c, int64_t n, const char* const* titles, const char* const* tsv_paths,
                                       int n_threads) {
    if (!c || n < 0 || (n && (!titles || !tsv_paths))) return SPL_ERR_ARG;
    if (c->merged_done) { c->err = "spl_combine_add_samples after spl_combine_merge"; return SPL_ERR_ARG; }
    for (int64_t k = 0; k < n; ++k)
        if (!titles[k] || !tsv_paths[k]) { c->err = "spl_combine_add_samples: null title or path"; return SPL_ERR_ARG; }
    std::vector<Sample> parsed((size_t)n);
    std::vector<LocalTables> local((size_t)n);
    std::vector<std::string> errs((size_t)n);
    std::vector<int> rcs((size_t)n, SPL_OK);
    std::atomic<int64_t> next{0};
    auto work = [&]() {
        for (int64_t k; (k = next.fetch_add(1)) < n;)
            rcs[(size_t)k] = parse_sample(titles[k], tsv_paths[k], parsed[(size_t)k], local[(size_t)k], errs[(size_t)k]);
    };
    const int nt = worker_count(n_threads > 0 ? n_threads : c->n_threads, (size_t)n);
    try {
        run_parallel(nt, work);
        for (int64_t k = 0; k < n; ++k)
            if (rcs[(size_t)k] != SPL_OK) { c->err = errs[(size_t)k]; return rcs[(size_t)k]; }   // the first failing sample, in file order
        for (int64_t k = 0; k < n; ++k) {                       // local ids -> shared ids, first appearance in sample order
            Sample& s = parsed[(size_t)k];
            LocalTables& lt = local[(size_t)k];
            std::vector<int32_t> rmap, smap, gmap;
            for (auto& nm : lt.regions.names) rmap.push_back(c->regions.id(nm));
            for (auto& nm : lt.strands.names) smap.push_back(c->strands.id(nm));
            for (auto& nm : lt.genes.names) gmap.push_back(c->genes.id(nm));
            for (auto& v : s.region) v = rmap[(size_t)v];
            for (auto& v : s.runs) v = rmap[(size_t)v];
            for (auto& v : s.strand) v = smap[(size_t)v];
            for (auto& v : s.gene) v = gmap[(size_t)v];
            c->samples.push_back(std::move(s));
        }
    } catch (const std::exception& e) {
        c->err = std::string("spl_combine_add_samples: ") + e.what();
        return SPL_ERR_NOMEM;
    }
    return SPL_OK;
}

extern "C" int spl_combine_add_sample(spl_combine* c, const char* title, const char* tsv_path) {
    return spl_combine_add_samples(c, 1, &title, &tsv_path, 1);
}

extern "C" int64_t spl_combine_n_samples(const spl_combine* c) { return c ? (int64_t)c->samples.size() : 0; }
extern "C" int64_t spl_combine_n_regions(const spl_combine* c) { return c ? (int64_t)c->regions.names.size() : 0; }
extern "C" const char* spl_combine_region_name(const spl_combine* c, int64_t i) {
    return (c && i >= 0 && i < (int64_t)c->regions.names.size()) ? c->regions.names[(size_t)i].c_str() : nullptr;
}
extern "C" int64_t spl_combine_sample_rows(const spl_combine* c, int64_t sample) {
    return (c && sample >= 0 && sample < (int64_t)c->samples.size()) ? (int64_t)c->samples[(size_t)sample].pos.size() : -1;
}
extern "C" int64_t spl_combine_sample_runs(const spl_combine* c, int64_t sample, const int32_t** runs) {
    if (!c || sample < 0 || sample >= (int64_t)c->samples.size()) return -1;
    const Sample& s = c->samples[(size_t)sample];
    if (runs) *runs = s.runs.data();
    return (int64_t)s.runs.size();
}

// The lock-step merge of `combine` (S:791-917) and, with `sh`, of `combineShallow` (S:977-1167).
// region_order = chromsInOrder (S:761-789 / S:960-988) as region ids; qgene NULL = "All".
// combineShallow differs in four places, each marked SHALLOW below: with -g only the rows of that gene are loaded at all
// (S:947-956), a '+' row takes over a tied position only from a row of another strand (S:1066), a position is kept only
// if at least minSamples samples show it with >= minReads reads and SSE >= minSSE -- counted over the rows of BOTH strands
// at that position, in sample order, restarting whenever the lowest position changes hands (S:1066-1084, S:1108) -- and a
// position that fails makes every sample whose current row has that position NUMBER move on, whatever the row's region or
// strand (S:1158-1160).
namespace {
struct ShallowOpts { int64_t min_samples, min_reads; double min_sse; };

int merge_impl(spl_combine* c, int64_t n_order, const int32_t* region_order, const char* qgene, int is_stranded, const ShallowOpts* sh) {
    if (!c || n_order <= 0 || !region_order) { if (c) c->err = "spl_combine_merge: empty region order"; return SPL_ERR_ARG; }
    if (c->merged_done) { c->err = "spl_combine_merge called twice"; return SPL_ERR_ARG; }
    const size_t n = c->samples.size();
    if (n == 0) { c->err = "spl_combine_merge: no samples"; return SPL_ERR_ARG; }
    const int32_t NONE = -2, INITIAL = -3;                 // chroms[idx] = None (iterator done) / '' (nothing read yet)
    const int32_t plus_id = c->strands.map.count("+") ? c->strands.map["+"] : -9;
    int32_t qgene_id = -1;
    bool all_genes = (qgene == nullptr);
    if (!all_genes) { auto it = c->genes.map.find(qgene); qgene_id = it == c->genes.map.end() ? -9 : it->second; }
    std::vector<int64_t> cur(n, -1), nrows(n), fpos(n, -1);          // fpos: position in rows[k] when filtered
    std::vector<int32_t> chroms(n, INITIAL);
    std::vector<char> go(n, 1), done(n, 0);
    for (size_t k = 0; k < n; ++k) nrows[k] = (int64_t)c->samples[k].pos.size();
    // SHALLOW with -g: the merge only ever sees the rows of that gene (S:947-956)
    const bool filtered = sh && !all_genes;
    std::vector<std::vector<int64_t>> rows;
    if (filtered) {
        rows.resize(n);
        for (size_t k = 0; k < n; ++k)
            for (int64_t r = 0; r < nrows[k]; ++r)
                if (c->samples[k].gene[(size_t)r] == qgene_id) rows[k].push_back(r);
    }
    if (sh)
        for (size_t k = 0; k < n; ++k)
            for (size_t r = 0; r < c->samples[k].sse.size(); ++r)
                if (c->samples[k].sse[r] != c->samples[k].sse[r] && (!filtered || c->samples[k].gene[r] == qgene_id)) {
                    c->err = "combineShallow: sample " + c->samples[k].title + ", data row " + std::to_string(r + 1) + ": the SSE column is not a number";
                    return SPL_ERR_ARG;
                }
    int64_t pos_counter = 0;
    int64_t order_at = 0;
    int32_t current = region_order[0];
    int64_t lowest = -1;
    int32_t lowest_strand = -1;
    size_t n_done = 0;
    std::vector<int32_t> part, comp;
    try {
        while (n_done < n) {
            int32_t assoc_gene = -1;                                              // ""
            pos_counter = 0;                                                      // S:1014
            for (size_t k = 0; k < n; ++k) {                                      // S:827-855 / S:1016-1084
                if (done[k]) continue;
                Sample& s = c->samples[k];
                if (go[k]) {
                    bool got;
                    if (filtered) { got = fpos[k] + 1 < (int64_t)rows[k].size(); if (got) cur[k] = rows[k][(size_t)++fpos[k]]; }
                    else { got = cur[k] + 1 < nrows[k]; if (got) ++cur[k]; }
                    if (got) { chroms[k] = s.region[(size_t)cur[k]]; go[k] = 0; }
                    else { done[k] = 1; ++n_done; chroms[k] = NONE; }
                }
                if (chroms[k] == current && chroms[k] >= 0) {
                    const int64_t p = s.pos[(size_t)cur[k]];
                    const int32_t st = s.strand[(size_t)cur[k]];
                    // S:847; SHALLOW (S:1066): only a '+' row of ANOTHER strand than the current holder takes a tie
                    const bool tie = is_stranded && p == lowest && st == plus_id && (!sh || st != lowest_strand);
                    const bool pass = sh && (s.alpha[(size_t)cur[k]] + s.beta1[(size_t)cur[k]] + s.beta2s[(size_t)cur[k]] >= sh->min_reads) &&
                                      (s.sse[(size_t)cur[k]] >= sh->min_sse);
                    if (p < lowest || lowest == -1 || tie) {
                        lowest = p; lowest_strand = st; assoc_gene = s.gene[(size_t)cur[k]];
                        pos_counter = pass ? 1 : 0;                                       // S:1071-1077
                    } else if (p == lowest && pass) {
                        ++pos_counter;                                                    // S:1079-1084
                    }
                }
            }
            if (n_done < n) {
                bool any_here = false;
                for (size_t k = 0; k < n; ++k) if (chroms[k] == current && chroms[k] >= 0) any_here = true;
                if (!any_here) {                                                  // S:857-866
                    if (++order_at >= n_order) {
                        c->err = "spl_combine_merge: rows remain on a region that is not in the region order";
                        return SPL_ERR_ARG;
                    }
                    current = region_order[order_at];
                } else if (sh && pos_counter < sh->min_samples) {                // SHALLOW, S:1154-1160: the position is dropped
                    for (size_t k = 0; k < n; ++k)
                        if (!done[k] && cur[k] >= 0 && c->samples[k].pos[(size_t)cur[k]] == lowest) go[k] = 1;
                } else {
                    const bool emit = all_genes || (assoc_gene == qgene_id);
                    Merged m;
                    m.region = current; m.pos = (int32_t)lowest; m.gene = assoc_gene;
                    m.cell = emit ? (int64_t)c->cells.size() : -1;
                    if (emit) c->cells.resize(c->cells.size() + n, -1);
                    part.clear(); comp.clear();
                    int32_t strand_now = -1;                                      // ''
                    bool filled_gap = false;
                    for (size_t k = 0; k < n; ++k) {                              // S:868-904
                        Sample& s = c->samples[k];
                        const int64_t r = cur[k];
                        const bool has = !done[k] && r >= 0 && s.region[(size_t)r] == current && s.pos[(size_t)r] == lowest &&
                                         (!is_stranded || s.strand[(size_t)r] == lowest_strand);
                        if (has) {
                            go[k] = 1;
                            strand_now = s.strand[(size_t)r];
                            if (emit) c->cells[(size_t)m.cell + k] = r;
                            for (int64_t e = s.p_off[(size_t)r]; e < s.p_off[(size_t)r + 1]; ++e) {          // S:889-892
                                bool seen = false;
                                for (int32_t q : part) if (q == s.p_key[(size_t)e]) { seen = true; break; }
                                if (!seen) part.push_back(s.p_key[(size_t)e]);
                            }
                            for (int64_t e = s.c_off[(size_t)r]; e < s.c_off[(size_t)r + 1]; ++e) {          // S:894-897
                                const int32_t v = s.c_key[(size_t)e];
                                size_t at = 0;
                                while (at < comp.size() && comp[at] < v) ++at;
                                if (at == comp.size() || comp[at] != v) comp.insert(comp.begin() + (long)at, v);
                            }
                        } else if (emit) {                                        // S:899-904: a gap of sample k
                            filled_gap = true;
                            c->cells[(size_t)m.cell + k] = -(int64_t)s.g_pos.size() - 2;
                            s.g_region.push_back(current);
                            s.g_pos.push_back((int32_t)lowest);
                            const std::string* sn = strand_now >= 0 ? &c->strands.names[(size_t)strand_now] : nullptr;
                            s.g_strand.push_back((sn && !sn->empty()) ? (uint8_t)(*sn)[0] : 0);
                            s.gp_pos.insert(s.gp_pos.end(), part.begin(), part.end());
                            s.gc_pos.insert(s.gc_pos.end(), comp.begin(), comp.end());
                            s.gp_off.push_back((int64_t)s.gp_pos.size());
                            s.gc_off.push_back((int64_t)s.gc_pos.size());
                        }
                    }
                    if (emit) {
                        m.part_off = (int64_t)c->u_part.size();
                        m.comp_off = (int64_t)c->u_comp.size();
                        c->u_part.insert(c->u_part.end(), part.begin(), part.end());
                        c->u_comp.insert(c->u_comp.end(), comp.begin(), comp.end());
                        c->u_part_end.push_back((int64_t)c->u_part.size());
                        c->u_comp_end.push_back((int64_t)c->u_comp.size());
                        c->merged.push_back(m);
                        if (filled_gap) ++c->n_filled;
                    }
                }
            }
            lowest = -1;
        }
    } catch (const std::bad_alloc&) {
        c->err = "out of memory";
        return SPL_ERR_NOMEM;
    }
    c->merged_done = true;
    return SPL_OK;
}
}  // namespace

extern "C" int spl_combine_merge(spl_combine* c, int64_t n_order, const int32_t* region_order, const char* qgene, int is_stranded) {
    return merge_impl(c, n_order, region_order, qgene, is_stranded, nullptr);
}

extern "C" int spl_combine_merge_shallow(spl_combine* c, int64_t n_order, const int32_t* region_order, const char* qgene, int is_stranded,
                                         int64_t min_samples, int64_t min_reads, double min_sse) {
    const ShallowOpts sh{min_samples, min_reads, min_sse};
    return merge_impl(c, n_order, region_order, qgene, is_stranded, &sh);
}

extern "C" int64_t spl_combine_n_sites(const spl_combine* c) { return c ? (int64_t)c->merged.size() : 0; }
extern "C" int64_t spl_combine_n_filled(const spl_combine* c) { return c ? c->n_filled : 0; }

extern "C" int64_t spl_combine_gaps(const spl_combine* c, int64_t sample, const int32_t** s_region, const int32_t** s_pos,
                                    const uint8_t** s_strand, const int64_t** p_off, const int32_t** p_pos,
                                    const int64_t** c_off, const int32_t** c_pos) {
    if (!c || !c->merged_done || sample < 0 || sample >= (int64_t)c->samples.size()) return -1;
    const Sample& s = c->samples[(size_t)sample];
    if (s_region) *s_region = s.g_region.data();
    if (s_pos) *s_pos = s.g_pos.data();
    if (s_strand) *s_strand = s.g_strand.data();
    if (p_off) *p_off = s.gp_off.data();
    if (p_pos) *p_pos = s.gp_pos.data();
    if (c_off) *c_off = s.gc_off.data();
    if (c_pos) *c_pos = s.gc_pos.data();
    return (int64_t)s.g_pos.size();
}

extern "C" int spl_combine_set_recount(spl_combine* c, int64_t sample, int64_t n_gaps, const int64_t* beta1,
                                       const int64_t* beta2simple) {
    if (!c || !c->merged_done || sample < 0 || sample >= (int64_t)c->samples.size()) return SPL_ERR_ARG;
    Sample& s = c->samples[(size_t)sample];
    if (n_gaps != (int64_t)s.g_pos.size() || (n_gaps && (!beta1 || !beta2simple))) {
        c->err = "spl_combine_set_recount: gap count differs from spl_combine_gaps";
        return SPL_ERR_ARG;
    }
    s.r_beta1.assign(beta1, beta1 + n_gaps);
    s.r_beta2s.assign(beta2simple, beta2simple + n_gaps);
    s.have_recount = true;
    return SPL_OK;
}

// outputCombinedLines for every merged site (S:722-740, called at S:912-915).  Blocks of merged sites are formatted
// concurrently into memory and written in order.
namespace {
void format_merged_site(const spl_combine* c, size_t mi, int cryptic, Out& o) {
    const size_t n = c->samples.size();
    const Merged& m = c->merged[mi];
    const int64_t* cell = &c->cells[(size_t)m.cell];
    int32_t strand_final = -1;                          // Site.setStrand by every sample that has the site (S:873)
    for (size_t k = 0; k < n; ++k)
        if (cell[k] >= 0) strand_final = c->samples[k].strand[(size_t)cell[k]];
    const int32_t* part = c->u_part.data() + m.part_off;
    const size_t n_part = (size_t)(c->u_part_end[mi] - m.part_off);
    const int32_t* comp = c->u_comp.data() + m.comp_off;
    const size_t n_comp = (size_t)(c->u_comp_end[mi] - m.comp_off);
    for (size_t k = 0; k < n; ++k) {
        const Sample& s = c->samples[k];
        long long alpha = 0, beta1 = 0, beta2s = 0, beta2c = 0;
        double beta2w = 0.0, sse = 0.0;
        const int64_t r = cell[k];
        bool cryptic_row = false;
        if (r >= 0) {
            alpha = s.alpha[(size_t)r]; beta1 = s.beta1[(size_t)r]; beta2s = s.beta2s[(size_t)r];
            if (s.has_cryptic[(size_t)r]) { beta2c = s.beta2c[(size_t)r]; beta2w = s.beta2w[(size_t)r]; cryptic_row = true; }
            if (cryptic) {                              // calculateSSE (S:626-639)
                double betas = (double)(beta1 + beta2s) + beta2w;
                double den = (double)alpha + betas;
                sse = den > 0.0 ? (double)alpha / den : 0.0;
            } else {
                long long den = alpha + beta1 + beta2s;
                sse = den > 0 ? (double)alpha / (double)den : 0.0;
            }
        } else if (r <= -2) {
            const size_t g = (size_t)(-r - 2);
            beta1 = s.r_beta1[g]; beta2s = s.r_beta2s[g];
        }
        o.put(s.title); o.ch('\t');
        o.put(c->regions.names[(size_t)m.region]); o.ch('\t');
        o.i64(m.pos); o.ch('\t');
        if (strand_final >= 0) o.put(c->strands.names[(size_t)strand_final]);
        o.ch('\t');
        if (m.gene >= 0) o.put(c->genes.names[(size_t)m.gene]);
        o.ch('\t');
        o.fixed(sse, 3); o.ch('\t');
        o.i64(alpha); o.ch('\t'); o.i64(beta1); o.ch('\t'); o.i64(beta2s); o.ch('\t');
        if (cryptic) { o.i64(beta2c); o.ch('\t'); o.pyfloat(cryptic_row ? beta2w : 0.0); o.ch('\t'); }
        else o.put("NA\tNA\t", 6);
        o.ch('{');
        for (size_t e = 0; e < n_part; ++e) {
            long long cnt = 0;
            if (r >= 0)
                for (int64_t q = s.p_off[(size_t)r]; q < s.p_off[(size_t)r + 1]; ++q)
                    if (s.p_key[(size_t)q] == part[e]) { cnt = s.p_cnt[(size_t)q]; break; }
            if (e) o.put(", ", 2);
            o.i64(part[e]); o.put(": ", 2); o.i64(cnt);
        }
        o.put("}\t[", 3);
        for (size_t e = 0; e < n_comp; ++e) {
            if (e) o.put(", ", 2);
            o.i64(comp[e]);
        }
        o.put("]\n", 2);
    }
}
}  // namespace

extern "C" int spl_combine_write(spl_combine* c, const char* path, int cryptic) {
    if (!c || !path) return SPL_ERR_ARG;
    if (!c->merged_done) { c->err = "spl_combine_write before spl_combine_merge"; return SPL_ERR_ARG; }
    const size_t n = c->samples.size();
    for (size_t k = 0; k < n; ++k)
        if (!c->samples[k].g_pos.empty() && !c->samples[k].have_recount) {
            c->err = "spl_combine_write: sample " + std::to_string(k) + " has gaps without re-count results";
            return SPL_ERR_ARG;
        }
    FILE* f = fopen(path, "w");
    if (!f) { c->err = std::string("cannot open ") + path + ": " + strerror(errno); return SPL_ERR_IO; }
    bool bad = fwrite(COMBINE_HEADER, 1, sizeof(COMBINE_HEADER) - 1, f) != sizeof(COMBINE_HEADER) - 1;
    const size_t block = std::max<size_t>(64, 65536 / std::max<size_t>(n, 1));        // merged sites per formatting job
    try {
        bad = bad || !write_blocks(f, c->merged.size(), block, c->n_threads, [&](size_t lo, size_t hi, Out& o) {
            for (size_t mi = lo; mi < hi; ++mi) format_merged_site(c, mi, cryptic, o);
        });
    } catch (const std::exception& e) {
        fclose(f);
        c->err = std::string("spl_combine_write: ") + e.what();
        return SPL_ERR_NOMEM;
    }
    if (fclose(f) != 0 || bad) { c->err = std::string("write to ") + path + " failed"; return SPL_ERR_IO; }
    return SPL_OK;
}

// ===================================================================================================== BED12 junctions
// The text half of findAlphaCounts (S:255-288): lines with exactly 12 tab-separated fields (S:259), chromosome index in
// first-appearance order appended to what the annotation registered (S:90-92, S:265-268), -c filter (S:269), left /
// right site positions and score (S:274-277), -g window (S:279-288).
struct spl_bed {
    std::vector<int32_t> chrom, left, right, strand_id;
    std::vector<int64_t> score;
    std::vector<uint8_t> strand;
    Interner chroms, strand_texts;
};

namespace {
// int(text): optional surrounding blanks, optional sign, decimal digits
bool bed_int(std::string_view s, long long* out) {
    while (!s.empty() && is_py_space(s.front())) s.remove_prefix(1);
    while (!s.empty() && is_py_space(s.back())) s.remove_suffix(1);
    if (!s.empty() && s.front() == '+') { s.remove_prefix(1); if (!s.empty() && s.front() == '-') return false; }
    if (s.empty()) return false;
    auto r = std::from_chars(s.data(), s.data() + s.size(), *out);
    return r.ec == std::errc() && r.ptr == s.data() + s.size();
}
}  // namespace

namespace {
using BedFilter = spl::JunctionFilter;

// Parses the lines of text[lo, hi) (hi at a line boundary) into `b` with ids local to `b`; returns SPL_OK or the error
// of the first bad line (err_line = its 1-based number inside the piece).  n_lines = lines seen.
int bed_parse_piece(const char* text, int64_t lo, int64_t hi, const BedFilter& f, spl_bed* b, int64_t* n_lines,
                    int64_t* err_line, const char** err_msg) {
    // the line count is kept in a local and stored once per return path: the pieces' counters sit next to each other in
    // one cache line, so a store per line from every worker would bounce that line between the cores
    int64_t at = lo, line_no = 0;
    *n_lines = 0;
    while (at < hi) {
        // one pass over the line: fields end at tabs, the line at '\n' (its text stays out of the last field)
        const char* p = text + at;
        const char* const e = text + hi;
        const char* field = p;
        std::string_view col[12];
        int nc = 0;
        for (; p < e && *p != '\n'; ++p) {
            if (*p == '\t') {
                if (nc < 12) col[nc] = std::string_view(field, (size_t)(p - field));
                ++nc;
                field = p + 1;
            }
        }
        if (nc < 12) col[nc] = std::string_view(field, (size_t)(p - field));
        ++nc;
        at = p < e ? (p - text) + 1 : hi;
        ++line_no;
        if (nc != 12) continue;                                          // S:259
        const int32_t ci = b->chroms.id(col[0]);                         // registered before the -c test (S:265-269)
        if (!f.chrom_kept(col[0])) continue;
        std::string_view sizes = col[10];
        size_t comma = sizes.find(',');
        if (comma == std::string_view::npos) { *n_lines = line_no; *err_line = line_no; *err_msg = "blockSizes needs two values"; return SPL_ERR_ARG; }
        std::string_view second = sizes.substr(comma + 1);
        second = second.substr(0, second.find(','));
        long long start, stop, a0, a1, score;
        if (!bed_int(col[1], &start) || !bed_int(col[2], &stop) || !bed_int(sizes.substr(0, comma), &a0) ||
            !bed_int(second, &a1) || !bed_int(col[4], &score)) {
            *n_lines = line_no; *err_line = line_no; *err_msg = "invalid literal for int()";
            return SPL_ERR_ARG;
        }
        const long long left = start + a0, right = stop - a1;            // S:275-276
        if (!f.window_kept(left, right)) continue;
        if (left < INT32_MIN || left > INT32_MAX || right < INT32_MIN || right > INT32_MAX) {
            *n_lines = line_no; *err_line = line_no; *err_msg = "position outside 32 bits";
            return SPL_ERR_RANGE;
        }
        b->chrom.push_back(ci);
        b->left.push_back((int32_t)left);
        b->right.push_back((int32_t)right);
        b->score.push_back(score);
        b->strand.push_back(col[5].empty() ? 0 : (uint8_t)col[5][0]);
        b->strand_id.push_back(b->strand_texts.id(col[5]));
    }
    *n_lines = line_no;
    return SPL_OK;
}
}  // namespace

// The file image is cut into pieces at line ends; the pieces parse concurrently with ids local to the piece and are
// appended in file order, which renumbers chromosomes and strand texts by first appearance exactly as one pass would.
extern "C" int spl_bed_parse(const char* text, int64_t len, const spl_strtab* chrom_index, const char* qchrom,
                             int use_gene_window, int64_t gene_left, int64_t gene_right, int64_t max_intron,
                             spl_bed** out, char* err, int err_len) {
    if (!out || len < 0 || (len && !text)) { set_err(err, err_len, "spl_bed_parse: null argument"); return SPL_ERR_ARG; }
    spl_bed* b = new (std::nothrow) spl_bed();
    if (!b) return SPL_ERR_NOMEM;
    const BedFilter f{qchrom, use_gene_window != 0, gene_left, gene_right, max_intron};
    try {
        if (chrom_index)
            for (int64_t i = 0; i < chrom_index->n; ++i) b->chroms.id(tab_get(chrom_index, i));
        const int nt = worker_count(0, (size_t)(len / (1 << 20)) + 1);       // about 1 MB of text per piece and worker
        std::vector<int64_t> cut{0};
        for (int k = 1; k < nt; ++k) {
            int64_t c = std::max(cut.back(), len * k / nt);
            const char* nl = c < len ? (const char*)memchr(text + c, '\n', (size_t)(len - c)) : nullptr;
            cut.push_back(nl ? (nl - text) + 1 : len);
        }
        cut.push_back(len);
        const size_t np = cut.size() - 1;
        std::vector<spl_bed> piece(np);
        std::vector<int> rc(np, SPL_OK);
        std::vector<int64_t> lines(np, 0), bad_line(np, 0);
        std::vector<const char*> msg(np, "");
        std::atomic<size_t> next{0};
        auto work = [&]() {
            for (size_t k; (k = next.fetch_add(1)) < np;) {
                try { rc[k] = bed_parse_piece(text, cut[k], cut[k + 1], f, &piece[k], &lines[k], &bad_line[k], &msg[k]); }
                catch (const std::bad_alloc&) { rc[k] = SPL_ERR_NOMEM; msg[k] = "out of memory"; }
            }
        };
        run_parallel((int)std::min<size_t>((size_t)nt, np), work);
        int64_t line0 = 0;
        for (size_t k = 0; k < np; ++k) {                                    // the first bad line in file order decides
            if (rc[k] != SPL_OK) {
                if (rc[k] == SPL_ERR_NOMEM) set_err(err, err_len, "out of memory");
                else set_err(err, err_len, "BED line %lld: %s", (long long)(line0 + bad_line[k]), msg[k]);
                const int code = rc[k];
                delete b;
                return code;
            }
            line0 += lines[k];
        }
        size_t total = 0;
        for (auto& pc : piece) total += pc.chrom.size();
        b->chrom.reserve(total); b->left.reserve(total); b->right.reserve(total);
        b->score.reserve(total); b->strand.reserve(total); b->strand_id.reserve(total);
        for (auto& pc : piece) {
            std::vector<int32_t> cmap, smap;
            for (auto& nm : pc.chroms.names) cmap.push_back(b->chroms.id(nm));
            for (auto& nm : pc.strand_texts.names) smap.push_back(b->strand_texts.id(nm));
            for (int32_t v : pc.chrom) b->chrom.push_back(cmap[(size_t)v]);
            for (int32_t v : pc.strand_id) b->strand_id.push_back(smap[(size_t)v]);
            b->left.insert(b->left.end(), pc.left.begin(), pc.left.end());
            b->right.insert(b->right.end(), pc.right.begin(), pc.right.end());
            b->score.insert(b->score.end(), pc.score.begin(), pc.score.end());
            b->strand.insert(b->strand.end(), pc.strand.begin(), pc.strand.end());
        }
    } catch (const std::exception&) {
        delete b;
        set_err(err, err_len, "out of memory");
        return SPL_ERR_NOMEM;
    }
    *out = b;
    return SPL_OK;
}

extern "C" void spl_bed_free(spl_bed* b) { delete b; }
extern "C" int64_t spl_bed_n_junctions(const spl_bed* b) { return b ? (int64_t)b->chrom.size() : 0; }
extern "C" const int32_t* spl_bed_chrom(const spl_bed* b) { return b->chrom.data(); }
extern "C" const int32_t* spl_bed_left(const spl_bed* b) { return b->left.data(); }
extern "C" const int32_t* spl_bed_right(const spl_bed* b) { return b->right.data(); }
extern "C" const int64_t* spl_bed_score(const spl_bed* b) { return b->score.data(); }
extern "C" const uint8_t* spl_bed_strand(const spl_bed* b) { return b->strand.data(); }
extern "C" const int32_t* spl_bed_strand_id(const spl_bed* b) { return b->strand_id.data(); }
extern "C" int64_t spl_bed_n_chrom(const spl_bed* b) { return b ? (int64_t)b->chroms.names.size() : 0; }
extern "C" const char* spl_bed_chrom_name(const spl_bed* b, int64_t i, int64_t* len) {
    if (!b || i < 0 || i >= (int64_t)b->chroms.names.size()) return nullptr;
    if (len) *len = (int64_t)b->chroms.names[(size_t)i].size();
    return b->chroms.names[(size_t)i].data();
}
extern "C" int64_t spl_bed_n_strand_texts(const spl_bed* b) { return b ? (int64_t)b->strand_texts.names.size() : 0; }
extern "C" const char* spl_bed_strand_text(const spl_bed* b, int64_t i, int64_t* len) {
    if (!b || i < 0 || i >= (int64_t)b->strand_texts.names.size()) return nullptr;
    if (len) *len = (int64_t)b->strand_texts.names[(size_t)i].size();
    return b->strand_texts.names[(size_t)i].data();
}

// The BED12 that `regtools junctions extract` writes, one line per row in table order:
//   chrom  start  end  JUNC%08d  score  strand  start  end  255,0,0  2  a,b  0,end-start-b
// with a = left - start and b = end - right the longest anchors, so that spl_bed_parse gives back left = start + a and
// right = end - b (S:275-276).  The layout follows regtools' documentation; byte parity with regtools is not pinned.
extern "C" int spl_write_junctions_bed(const char* path, int64_t n, const int32_t* chrom, const int32_t* left, const int32_t* right,
                                       const int32_t* start, const int32_t* end, const int64_t* score, const uint8_t* strand,
                                       const spl_strtab* chrom_names, char* err, int err_len) {
    if (!path || n < 0 || !chrom_names || (n > 0 && (!chrom || !left || !right || !start || !end || !score || !strand))) {
        set_err(err, err_len, "spl_write_junctions_bed: null argument");
        return SPL_ERR_ARG;
    }
    for (int64_t i = 0; i < n; ++i)
        if (chrom[i] < 0 || chrom[i] >= chrom_names->n || start[i] > left[i] || end[i] < right[i]) {
            set_err(err, err_len, "spl_write_junctions_bed: row %lld: chromosome out of range or anchor extents inside the junction", (long long)i);
            return SPL_ERR_ARG;
        }
    FILE* f = fopen(path, "w");
    if (!f) { set_err(err, err_len, "cannot open %s: %s", path, strerror(errno)); return SPL_ERR_IO; }
    bool bad = false;
    {
        Out o(f);
        char name[32];
        for (int64_t i = 0; i < n; ++i) {
            const long long s = start[i], e = end[i], a = left[i] - s, b = e - right[i];
            o.put(tab_get(chrom_names, chrom[i])); o.ch('\t');
            o.i64(s); o.ch('\t'); o.i64(e); o.ch('\t');
            o.put(name, (size_t)snprintf(name, sizeof name, "JUNC%08lld", (long long)(i + 1))); o.ch('\t');
            o.i64(score[i]); o.ch('\t');
            if (strand[i]) o.ch((char)strand[i]);
            o.ch('\t');
            o.i64(s); o.ch('\t'); o.i64(e); o.put("\t255,0,0\t2\t");
            o.i64(a); o.ch(','); o.i64(b); o.put("\t0,"); o.i64(e - s - b); o.ch('\n');
        }
        o.flush();
        bad = o.bad;
    }
    if (fclose(f) != 0 || bad) { set_err(err, err_len, "write to %s failed", path); return SPL_ERR_IO; }
    return SPL_OK;
}

// ========================================================================================================== annotation
// createGenes (S:50-116) without HTSeq: every feature line whose type column is "gene" becomes a Gene with
// leftPos = GFF start - 1, rightPos = GFF end (HTSeq's iv.start / iv.end), its strand column and, as name, the value of
// its first attribute (README.md:64).  Chromosomes are indexed by first appearance among the gene lines (S:90-92).
// Without a query gene every chromosome's list is in insort order (S:95: bisect.insort by leftPos = stable sort by
// leftPos); with one, only the genes of that name are kept, in file order, and the last of them is QUERY_gene (S:97-101).
struct spl_genes {
    Interner chroms, strand_texts;
    std::vector<int64_t> chrom_off;                    // [n_chrom + 1] into the arrays below (grouped by chromosome)
    std::vector<int32_t> left, right, strand_id;
    std::vector<int64_t> name_off{0};
    std::string names;
    int64_t query = -1;                                // flat index of QUERY_gene, -1 = none
};

namespace {
struct GeneRow { int32_t chrom, left, right, strand; int64_t name_at, name_len, order; };

std::string_view py_strip(std::string_view s) {
    while (!s.empty() && is_py_space(s.front())) s.remove_prefix(1);
    while (!s.empty() && is_py_space(s.back())) s.remove_suffix(1);
    return s;
}

// Value of the first attribute, the way HTSeq.GFF_Reader names a feature (parse_GFF_attribute_string, restated from its
// published source; HTSeq is not in this image, so: parity unpinned): the attribute column is cut at the first ';' that is
// not inside double quotes; the piece must look like  \s* key [\s=]+ value  with a key free of blanks and '='; the value runs to
// the end of the piece (trailing blanks included) and loses one pair of enclosing double quotes.  "ID=AT1G01010;..." ->
// AT1G01010 (GFF3), 'gene_id "X"; ...' -> X (GTF), 'gene_id "A=B"' -> A=B, "ID= X" -> X.  An empty first piece names the
// feature "_unnamed_"; a piece without a separator (HTSeq raises there) keeps the whole piece.
std::string_view first_attribute(std::string_view col9) {
    static const char unnamed[] = "_unnamed_";
    size_t cut = col9.size();
    bool in_quote = false;
    for (size_t i = 0; i < col9.size(); ++i) {
        if (col9[i] == '"') in_quote = !in_quote;
        else if (!in_quote && col9[i] == ';') { cut = i; break; }
    }
    std::string_view piece = col9.substr(0, cut);
    size_t a = 0;
    while (a < piece.size() && is_py_space(piece[a])) ++a;
    if (a == piece.size()) return std::string_view(unnamed, 9);
    size_t k = a;
    while (k < piece.size() && !is_py_space(piece[k]) && piece[k] != '=') ++k;          // the key
    size_t v = k;
    while (v < piece.size() && (is_py_space(piece[v]) || piece[v] == '=')) ++v;          // [\s=]+
    if (k == a || v == k) return py_strip(piece);                                        // no key or no separator
    std::string_view val = piece.substr(v);
    if (val.size() >= 2 && val.front() == '"' && val.back() == '"') { val.remove_prefix(1); val.remove_suffix(1); }
    return val;
}
}  // namespace

extern "C" int spl_genes_parse(const char* text, int64_t len, const char* qgene, spl_genes** out, char* err, int err_len) {
    if (!out || len < 0 || (len && !text)) { set_err(err, err_len, "spl_genes_parse: null argument"); return SPL_ERR_ARG; }
    spl_genes* g = new (std::nothrow) spl_genes();
    if (!g) return SPL_ERR_NOMEM;
    try {
        const std::string_view q = qgene ? std::string_view(qgene) : std::string_view();
        std::vector<GeneRow> rows;
        int64_t at = 0, line_no = 0, last_match = -1;
        while (at < len) {
            const char* nl = (const char*)memchr(text + at, '\n', (size_t)(len - at));
            const int64_t end = nl ? (nl - text) : len;
            std::string_view line(text + at, (size_t)(end - at));
            at = nl ? end + 1 : len;
            ++line_no;
            if (!line.empty() && line.back() == '\r') line.remove_suffix(1);   // universal newlines, as Python's text mode reads the file
            if (line.empty() || line.front() == '#') continue;
            std::string_view col[9];
            int nc = 0;
            {
                const char* p = line.data();
                const char* const e = p + line.size();
                const char* field = p;
                for (; p < e && nc < 9; ++p)
                    if (*p == '\t') { col[nc++] = std::string_view(field, (size_t)(p - field)); field = p + 1; }
                if (nc < 9) col[nc++] = std::string_view(field, (size_t)(e - field));
            }
            if (nc < 9 || col[2] != "gene") continue;
            long long start, stop;
            if (!bed_int(col[3], &start) || !bed_int(col[4], &stop)) {
                set_err(err, err_len, "annotation line %lld: invalid literal for int()", (long long)line_no);
                delete g;
                return SPL_ERR_ARG;
            }
            if (start - 1 < INT32_MIN || start - 1 > INT32_MAX || stop < INT32_MIN || stop > INT32_MAX) {
                set_err(err, err_len, "annotation line %lld: position outside 32 bits", (long long)line_no);
                delete g;
                return SPL_ERR_RANGE;
            }
            const std::string_view name = first_attribute(col[8]);
            const int32_t ci = g->chroms.id(col[0]);             // registered for every gene line, kept or not (S:90-92)
            if (qgene && name != q) continue;
            if (qgene) last_match = (int64_t)rows.size();
            rows.push_back(GeneRow{ci, (int32_t)(start - 1), (int32_t)stop, g->strand_texts.id(col[6]),
                                   (int64_t)(name.data() - text), (int64_t)name.size(), (int64_t)rows.size()});
        }
        // group by chromosome; inside one: insort order (stable by leftPos) without a query gene, file order with one
        std::stable_sort(rows.begin(), rows.end(), [&](const GeneRow& a, const GeneRow& b) {
            if (a.chrom != b.chrom) return a.chrom < b.chrom;
            return !qgene && a.left < b.left;
        });
        const size_t nc = g->chroms.names.size();
        g->chrom_off.assign(nc + 1, 0);
        for (const GeneRow& r : rows) g->chrom_off[(size_t)r.chrom + 1]++;
        for (size_t c = 0; c < nc; ++c) g->chrom_off[c + 1] += g->chrom_off[c];
        for (size_t i = 0; i < rows.size(); ++i) {
            const GeneRow& r = rows[i];
            g->left.push_back(r.left); g->right.push_back(r.right); g->strand_id.push_back(r.strand);
            g->names.append(text + r.name_at, (size_t)r.name_len);
            g->name_off.push_back((int64_t)g->names.size());
            if (r.order == last_match) g->query = (int64_t)i;
        }
    } catch (const std::exception&) {
        delete g;
        set_err(err, err_len, "out of memory");
        return SPL_ERR_NOMEM;
    }
    *out = g;
    return SPL_OK;
}

extern "C" void spl_genes_free(spl_genes* g) { delete g; }
extern "C" int64_t spl_genes_n(const spl_genes* g) { return g ? (int64_t)g->left.size() : 0; }
extern "C" int64_t spl_genes_n_chrom(const spl_genes* g) { return g ? (int64_t)g->chroms.names.size() : 0; }
extern "C" const char* spl_genes_chrom_name(const spl_genes* g, int64_t i, int64_t* len) {
    if (!g || i < 0 || i >= (int64_t)g->chroms.names.size()) return nullptr;
    if (len) *len = (int64_t)g->chroms.names[(size_t)i].size();
    return g->chroms.names[(size_t)i].data();
}
extern "C" const int64_t* spl_genes_chrom_off(const spl_genes* g) { return g->chrom_off.data(); }
extern "C" const int32_t* spl_genes_left(const spl_genes* g) { return g->left.data(); }
extern "C" const int32_t* spl_genes_right(const spl_genes* g) { return g->right.data(); }
extern "C" const int32_t* spl_genes_strand_id(const spl_genes* g) { return g->strand_id.data(); }
extern "C" int64_t spl_genes_n_strand_texts(const spl_genes* g) { return g ? (int64_t)g->strand_texts.names.size() : 0; }
extern "C" const char* spl_genes_strand_text(const spl_genes* g, int64_t i, int64_t* len) {
    if (!g || i < 0 || i >= (int64_t)g->strand_texts.names.size()) return nullptr;
    if (len) *len = (int64_t)g->strand_texts.names[(size_t)i].size();
    return g->strand_texts.names[(size_t)i].data();
}
extern "C" const char* spl_genes_names(const spl_genes* g) { return g->names.data(); }
extern "C" const int64_t* spl_genes_name_off(const spl_genes* g) { return g->name_off.data(); }
extern "C" int64_t spl_genes_query(const spl_genes* g) { return g ? g->query : -1; }
