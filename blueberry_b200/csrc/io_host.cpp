// io_host.cpp - libbbkio.so: the significances writer of include/bbk_io.h (host only).
#include <algorithm>
#include <atomic>
#include <charconv>
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstring>
#include <string>
#include <thread>
#include <vector>
#include <zlib.h>

#include "../../include/bbk.h"
#include "../../include/bbk_io.h"

namespace {

thread_local char g_err[512] = "";
void set_error(const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
}

inline char* put_int(char* o, long long v) {
    if (v < 0) { *o++ = '-'; }
    unsigned long long u = v < 0 ? 0ull - (unsigned long long)v : (unsigned long long)v;
    char tmp[24];
    int k = 0;
    do { tmp[k++] = (char)('0' + u % 10); u /= 10; } while (u);
    while (k) *o++ = tmp[--k];
    return o;
}

// Python / numpy float64 str: shortest round-trip digits; positional when the decimal point position is in (-4, 16]
int format_double(double x, char* out) {
    char* o = out;
    if (x != x) { memcpy(o, "nan", 3); return 3; }
    if (x < 0 || (x == 0 && std::signbit(x))) { *o++ = '-'; x = -x; }
    if (x == 0) { memcpy(o, "0.0", 3); return (int)(o - out) + 3; }
    if (x > 1.7976931348623157e308) { memcpy(o, "inf", 3); return (int)(o - out) + 3; }
    char sci[40];
    auto r = std::to_chars(sci, sci + sizeof(sci), x, std::chars_format::scientific);     // d[.ddd]e[+-]XX, shortest
    char digits[24];
    int nd = 0;
    const char* s = sci;
    for (; s < r.ptr && *s != 'e'; ++s) if (*s != '.') digits[nd++] = *s;
    int e10 = 0;
    {
        ++s;                                     // 'e'
        bool neg = *s == '-';
        ++s;
        for (; s < r.ptr; ++s) e10 = e10 * 10 + (*s - '0');
        if (neg) e10 = -e10;
    }
    const int decpt = e10 + 1;                   // digits * 10^(decpt - nd)
    if (decpt > -4 && decpt <= 16) {
        if (decpt <= 0) {
            *o++ = '0'; *o++ = '.';
            for (int i = 0; i < -decpt; ++i) *o++ = '0';
            memcpy(o, digits, nd); o += nd;
        } else if (decpt >= nd) {
            memcpy(o, digits, nd); o += nd;
            for (int i = nd; i < decpt; ++i) *o++ = '0';
            *o++ = '.'; *o++ = '0';
        } else {
            memcpy(o, digits, decpt); o += decpt;
            *o++ = '.';
            memcpy(o, digits + decpt, nd - decpt); o += nd - decpt;
        }
    } else {
        *o++ = digits[0];
        if (nd > 1) { *o++ = '.'; memcpy(o, digits + 1, nd - 1); o += nd - 1; }
        *o++ = 'e';
        int e = decpt - 1;
        *o++ = e < 0 ? '-' : '+';
        if (e < 0) e = -e;
        if (e < 10) *o++ = '0';
        o = put_int(o, e);
    }
    return (int)(o - out);
}

struct Job {
    const char* const* names;
    const size_t* name_len;
    const int32_t *chr1, *chr2;
    const int64_t *mid1, *mid2, *count;
    const double *p, *q;
};

// rows [lo, hi) -> text -> one gzip member appended to `out`; returns rows kept, or -1
long long format_and_deflate(const Job& J, long long lo, long long hi, bool header, int level, std::string& text, std::string& out) {
    text.clear();
    if (header) text += "chr1\tfragmentMid1\tchr2\tfragmentMid2\tcontactCount\tp-value\tq-value\n";
    long long kept = 0;
    char line[2 * 100 + 160];          // two names of at most 100 bytes (checked by the caller) + 3 integers + 2 doubles + separators
    for (long long i = lo; i < hi; ++i) {
        const double pv = J.p[i];
        if (!(pv <= 1.0)) continue;
        const int a = J.chr1 ? J.chr1[i] : 0, b = J.chr2 ? J.chr2[i] : 0;
        char* o = line;
        memcpy(o, J.names[a], J.name_len[a]); o += J.name_len[a]; *o++ = '\t';
        o = put_int(o, J.mid1[i]); *o++ = '\t';
        memcpy(o, J.names[b], J.name_len[b]); o += J.name_len[b]; *o++ = '\t';
        o = put_int(o, J.mid2[i]); *o++ = '\t';
        o = put_int(o, J.count[i]); *o++ = '\t';
        o += format_double(pv, o); *o++ = '\t';
        if (J.q) o += format_double(J.q[i], o); else { *o++ = '-'; *o++ = '1'; }
        *o++ = '\n';
        text.append(line, (size_t)(o - line));
        kept += 1;
    }
    z_stream zs;
    memset(&zs, 0, sizeof(zs));
    if (deflateInit2(&zs, level, Z_DEFLATED, 15 + 16, 8, Z_DEFAULT_STRATEGY) != Z_OK) return -1;
    const size_t bound = deflateBound(&zs, (uLong)text.size()) + 64;
    const size_t at = out.size();
    out.resize(at + bound);
    zs.next_in = (Bytef*)text.data();
    zs.avail_in = (uInt)text.size();
    zs.next_out = (Bytef*)&out[at];
    zs.avail_out = (uInt)bound;
    const int rc = deflate(&zs, Z_FINISH);
    const size_t produced = bound - zs.avail_out;
    deflateEnd(&zs);
    if (rc != Z_STREAM_END) return -1;
    out.resize(at + produced);
    return kept;
}

}  // namespace

extern "C" void bbkio_last_error(char* buf, size_t len) {
    if (!buf || !len) return;
    strncpy(buf, g_err, len - 1);
    buf[len - 1] = 0;
}

extern "C" int bbkio_format_double(double x, char* buf) { return format_double(x, buf); }

extern "C" int bbkio_write_significances(const char* path, const char* const* chrom_names, int32_t n_chrom, const int32_t* chr1,
                                         const int64_t* mid1, const int32_t* chr2, const int64_t* mid2, const int64_t* count,
                                         const double* p, const double* q, int64_t n, int32_t threads, int32_t level,
                                         int64_t* rows_written) {
    if (!path || !chrom_names || n_chrom <= 0 || n < 0 || (n > 0 && (!mid1 || !mid2 || !count || !p)) || ((chr1 == nullptr) != (chr2 == nullptr))) {
        set_error("bbkio_write_significances: bad arguments");
        return BBKIO_E_INVALID;
    }
    if (level < 1 || level > 9) level = 1;
    std::vector<size_t> name_len(n_chrom);
    for (int c = 0; c < n_chrom; ++c) {
        if (!chrom_names[c] || strlen(chrom_names[c]) > 100) { set_error("bbkio_write_significances: bad chromosome name %d", c); return BBKIO_E_INVALID; }
        name_len[c] = strlen(chrom_names[c]);
    }
    if (chr1) {
        for (int64_t i = 0; i < n; ++i)
            if (chr1[i] < 0 || chr1[i] >= n_chrom || chr2[i] < 0 || chr2[i] >= n_chrom) {
                set_error("bbkio_write_significances: chromosome id out of range at row %lld", (long long)i);
                return BBKIO_E_INVALID;
            }
    }
    int T = threads > 0 ? threads : (int)std::thread::hardware_concurrency();
    if (T < 1) T = 1;
    const long long block = 1 << 17;                                  // rows per gzip member (~6 MB of text)
    const long long n_blocks = n == 0 ? 1 : (n + block - 1) / block;
    if (T > n_blocks) T = (int)n_blocks;
    FILE* fh = fopen(path, "wb");
    if (!fh) { set_error("bbkio_write_significances: cannot open %s", path); return BBKIO_E_IO; }
    Job J = {chrom_names, name_len.data(), chr1, chr2, mid1, mid2, count, p, q};
    std::vector<std::string> text(T), out(T);
    std::vector<long long> kept(T);
    long long total = 0;
    int rc = BBKIO_OK;
    for (long long wave = 0; wave < n_blocks && rc == BBKIO_OK; wave += T) {
        const int live = (int)((n_blocks - wave) < T ? (n_blocks - wave) : T);
        std::vector<std::thread> pool;
        for (int t = 0; t < live; ++t) {
            pool.emplace_back([&, t]() {
                const long long b = wave + t, lo = b * block, hi = (lo + block < n) ? lo + block : n;
                out[t].clear();
                kept[t] = format_and_deflate(J, lo, hi, b == 0, level, text[t], out[t]);
            });
        }
        for (auto& th : pool) th.join();
        for (int t = 0; t < live; ++t) {
            if (kept[t] < 0) { set_error("bbkio_write_significances: zlib failed"); rc = BBKIO_E_ZLIB; break; }
            if (fwrite(out[t].data(), 1, out[t].size(), fh) != out[t].size()) { set_error("bbkio_write_significances: short write to %s", path); rc = BBKIO_E_IO; break; }
            total += kept[t];
        }
    }
    if (fclose(fh) != 0 && rc == BBKIO_OK) { set_error("bbkio_write_significances: close failed on %s", path); rc = BBKIO_E_IO; }
    if (rows_written) *rows_written = total;
    return rc;
}

// =====================================================================================================================
// reader: the interactions file (fithic.py:243-247)
// =====================================================================================================================
#include <condition_variable>
#include <deque>
#include <mutex>
#include <unordered_map>

struct BbkioTable {
    std::vector<std::string> names;
    std::vector<int32_t> chr1, chr2;
    std::vector<int64_t> mid1, mid2, count;
};

namespace {

struct Block {                       // whole lines of text + the (1-based) number of its first line
    std::string text;
    long long first_line = 0;
    long long index = 0;
};

struct Parsed {
    std::vector<int32_t> chr1, chr2;                 // block-local name ids
    std::vector<int64_t> mid1, mid2, count;
    std::vector<std::string> names;                  // block-local names in order of first appearance
    std::string error;
};

inline bool is_space(char c) { return c == ' ' || c == '\t' || c == '\r' || c == '\v' || c == '\f'; }

// Python's int() on a field: optional sign, decimal digits (underscore separators and other exotica are not accepted)
inline bool parse_int(const char* b, const char* e, int64_t* out) {
    if (b == e) return false;
    bool neg = false;
    if (*b == '+' || *b == '-') { neg = *b == '-'; ++b; }
    if (b == e || e - b > 18) return false;
    int64_t v = 0;
    for (; b < e; ++b) {
        if (*b < '0' || *b > '9') return false;
        v = v * 10 + (*b - '0');
    }
    *out = neg ? -v : v;
    return true;
}

void parse_block(const Block& B, Parsed& P) {
    std::unordered_map<std::string, int32_t> ids;
    const char* p = B.text.data();
    const char* end = p + B.text.size();
    long long line_no = B.first_line;
    auto name_id = [&](const char* b, const char* e) {
        std::string s(b, e);
        auto it = ids.find(s);
        if (it != ids.end()) return it->second;
        int32_t id = (int32_t)P.names.size();
        ids.emplace(s, id);
        P.names.push_back(std::move(s));
        return id;
    };
    const size_t guess = B.text.size() / 28 + 16;
    P.chr1.reserve(guess); P.chr2.reserve(guess); P.mid1.reserve(guess); P.mid2.reserve(guess); P.count.reserve(guess);
    while (p < end) {
        const char* eol = (const char*)memchr(p, '\n', (size_t)(end - p));
        if (!eol) eol = end;
        const char* tb[6];
        const char* te[6];
        int nf = 0;
        const char* q = p;
        while (q < eol) {
            while (q < eol && is_space(*q)) ++q;
            if (q == eol) break;
            const char* b = q;
            while (q < eol && !is_space(*q)) ++q;
            if (nf < 6) { tb[nf] = b; te[nf] = q; }
            ++nf;
        }
        if (nf != 5) {
            char msg[160];
            snprintf(msg, sizeof(msg), nf < 5 ? "line %lld: not enough values to unpack (expected 5, got %d)"
                                               : "line %lld: too many values to unpack (expected 5)", line_no, nf);
            P.error = msg;
            return;
        }
        int64_t m1, m2, c;
        if (!parse_int(tb[1], te[1], &m1) || !parse_int(tb[3], te[3], &m2) || !parse_int(tb[4], te[4], &c)) {
            char msg[160];
            snprintf(msg, sizeof(msg), "line %lld: invalid literal for int() with base 10", line_no);
            P.error = msg;
            return;
        }
        P.chr1.push_back(name_id(tb[0], te[0]));
        P.chr2.push_back(name_id(tb[2], te[2]));
        P.mid1.push_back(m1); P.mid2.push_back(m2); P.count.push_back(c);
        p = eol + 1;
        ++line_no;
    }
}

}  // namespace

extern "C" int bbkio_read_interactions(const char* path, int32_t threads, BbkioTable** out) {
    if (!path || !out) { set_error("bbkio_read_interactions: bad arguments"); return BBKIO_E_INVALID; }
    *out = nullptr;
    gzFile gz = gzopen(path, "rb");                  // reads plain text too; continues over concatenated members
    if (!gz) { set_error("bbkio_read_interactions: cannot open %s", path); return BBKIO_E_IO; }
    gzbuffer(gz, 1 << 20);
    int T = threads > 0 ? threads : (int)std::thread::hardware_concurrency();
    if (T < 1) T = 1;
    std::mutex mu;
    std::condition_variable cv_work, cv_space;
    std::deque<Block> queue;
    bool done = false, failed = false;
    std::vector<Parsed> results;                     // indexed by block
    std::mutex res_mu;
    std::string first_error;
    long long first_error_block = -1;
    auto worker = [&]() {
        for (;;) {
            Block B;
            {
                std::unique_lock<std::mutex> lk(mu);
                cv_work.wait(lk, [&] { return !queue.empty() || done; });
                if (queue.empty()) return;
                B = std::move(queue.front());
                queue.pop_front();
            }
            cv_space.notify_one();
            Parsed P;
            parse_block(B, P);
            std::lock_guard<std::mutex> lk(res_mu);
            if (!P.error.empty() && (first_error_block < 0 || B.index < first_error_block)) { first_error_block = B.index; first_error = P.error; failed = true; }
            if ((long long)results.size() <= B.index) results.resize(B.index + 1);
            results[B.index] = std::move(P);
        }
    };
    std::vector<std::thread> pool;
    for (int t = 0; t < T; ++t) pool.emplace_back(worker);
    const size_t CHUNK = 8u << 20;
    std::string carry;
    long long line_no = 1, index = 0;
    int io_rc = BBKIO_OK;
    std::vector<char> buf(CHUNK);
    for (;;) {
        int got = gzread(gz, buf.data(), (unsigned)CHUNK);
        if (got < 0) { int e; set_error("bbkio_read_interactions: %s", gzerror(gz, &e)); io_rc = BBKIO_E_ZLIB; break; }
        const bool last = got == 0;
        Block B;
        if (!last) {
            // cut at the last newline; the rest waits for the next chunk
            int cut = got;
            while (cut > 0 && buf[cut - 1] != '\n') --cut;
            B.text = std::move(carry);
            B.text.append(buf.data(), (size_t)cut);
            carry.assign(buf.data() + cut, (size_t)(got - cut));
            if (cut == 0) { carry = std::move(B.text) + carry; continue; }       // no newline in this chunk yet
        } else {
            if (carry.empty()) break;
            B.text = std::move(carry);                                       // last line without a newline
            carry.clear();
        }
        B.first_line = line_no;
        B.index = index++;
        for (char ch : B.text) line_no += ch == '\n';
        if (last && (B.text.empty() || B.text.back() != '\n')) line_no += 1;
        {
            std::unique_lock<std::mutex> lk(mu);
            cv_space.wait(lk, [&] { return (int)queue.size() < 2 * T; });
            queue.push_back(std::move(B));
        }
        cv_work.notify_one();
        if (last) break;
        { std::lock_guard<std::mutex> lk(res_mu); if (failed) break; }
    }
    { std::lock_guard<std::mutex> lk(mu); done = true; }
    cv_work.notify_all();
    for (auto& th : pool) th.join();
    gzclose(gz);
    if (io_rc != BBKIO_OK) return io_rc;
    if (failed) { set_error("bbkio_read_interactions: %s", first_error.c_str()); return BBKIO_E_PARSE; }
    // stitch: global name ids in order of first appearance over the blocks
    BbkioTable* Tb = new BbkioTable();
    std::unordered_map<std::string, int32_t> gids;
    size_t total = 0;
    for (auto& P : results) total += P.mid1.size();
    Tb->chr1.resize(total); Tb->chr2.resize(total); Tb->mid1.resize(total); Tb->mid2.resize(total); Tb->count.resize(total);
    std::vector<size_t> offs(results.size() + 1, 0);
    std::vector<std::vector<int32_t>> luts(results.size());
    for (size_t b = 0; b < results.size(); ++b) {
        offs[b + 1] = offs[b] + results[b].mid1.size();
        // first appearance inside a block is not by row for chr2 before chr1 of the same row: keep the row order exact
        auto& P = results[b];
        luts[b].assign(P.names.size(), -1);
        for (size_t i = 0; i < P.chr1.size(); ++i) {
            for (int32_t loc : {P.chr1[i], P.chr2[i]}) {
                if (luts[b][loc] >= 0) continue;
                auto it = gids.find(P.names[loc]);
                if (it == gids.end()) { int32_t id = (int32_t)Tb->names.size(); gids.emplace(P.names[loc], id); Tb->names.push_back(P.names[loc]); luts[b][loc] = id; }
                else luts[b][loc] = it->second;
            }
            bool all = true;
            for (int32_t v : luts[b]) all = all && v >= 0;
            if (all) break;
        }
    }
    std::vector<std::thread> copy_pool;
    std::atomic<size_t> next(0);
    for (int t = 0; t < T; ++t) {
        copy_pool.emplace_back([&]() {
            for (;;) {
                size_t b = next.fetch_add(1);
                if (b >= results.size()) return;
                auto& P = results[b];
                const size_t o = offs[b], m = P.mid1.size();
                for (size_t i = 0; i < m; ++i) { Tb->chr1[o + i] = luts[b][P.chr1[i]]; Tb->chr2[o + i] = luts[b][P.chr2[i]]; }
                if (m) {
                    memcpy(&Tb->mid1[o], P.mid1.data(), m * sizeof(int64_t));
                    memcpy(&Tb->mid2[o], P.mid2.data(), m * sizeof(int64_t));
                    memcpy(&Tb->count[o], P.count.data(), m * sizeof(int64_t));
                }
                Parsed().chr1.swap(P.chr1); Parsed().mid1.swap(P.mid1); Parsed().mid2.swap(P.mid2); Parsed().count.swap(P.count); Parsed().chr2.swap(P.chr2);
            }
        });
    }
    for (auto& th : copy_pool) th.join();
    *out = Tb;
    return BBKIO_OK;
}

extern "C" int64_t bbkio_table_rows(const BbkioTable* t) { return t ? (int64_t)t->mid1.size() : 0; }
extern "C" int32_t bbkio_table_n_chrom(const BbkioTable* t) { return t ? (int32_t)t->names.size() : 0; }
extern "C" const char* bbkio_table_chrom_name(const BbkioTable* t, int32_t id) {
    return (t && id >= 0 && id < (int32_t)t->names.size()) ? t->names[id].c_str() : nullptr;
}
extern "C" int bbkio_table_copy(const BbkioTable* t, int32_t* chr1, int64_t* mid1, int32_t* chr2, int64_t* mid2, int64_t* count) {
    if (!t) { set_error("bbkio_table_copy: null table"); return BBKIO_E_INVALID; }
    const size_t n = t->mid1.size();
    if (chr1 && n) memcpy(chr1, t->chr1.data(), n * sizeof(int32_t));
    if (chr2 && n) memcpy(chr2, t->chr2.data(), n * sizeof(int32_t));
    if (mid1 && n) memcpy(mid1, t->mid1.data(), n * sizeof(int64_t));
    if (mid2 && n) memcpy(mid2, t->mid2.data(), n * sizeof(int64_t));
    if (count && n) memcpy(count, t->count.data(), n * sizeof(int64_t));
    return BBKIO_OK;
}
extern "C" void bbkio_table_free(BbkioTable* t) { delete t; }

// ---- bbkio_unpack_scores: the packed p / q columns of a pass (bbk_pack_scores) back into dense columns -------------------
static int unpack_scores_impl(const uint32_t* codes, const void* chunks_v, const double* values_p, const double* values_q,
                              int64_t m, double* p, double* q, uint8_t* keep, int32_t threads) {
    if (m < 0 || (m > 0 && (!codes || !chunks_v || !p))) { set_error("bbkio_unpack_scores: null pointer / negative size"); return BBKIO_E_INVALID; }
    if (m == 0) return BBKIO_OK;
    struct Chunk { uint64_t base_p, base_q; uint32_t n_p, n_q; };
    static_assert(sizeof(Chunk) == 24, "chunk records are 24 bytes");
    const Chunk* chunks = static_cast<const Chunk*>(chunks_v);
    const int64_t CH = 4096;
    const int64_t n_chunks = (m + CH - 1) / CH;
    int nt = threads > 0 ? threads : (int)std::thread::hardware_concurrency();
    if (nt < 1) nt = 1;
    if ((int64_t)nt > n_chunks) nt = (int)n_chunks;
    uint64_t qnan_bits = 0x7ff8000000000000ull;
    double qnan;
    memcpy(&qnan, &qnan_bits, 8);
    std::atomic<int> bad(0);
    auto work = [&](int t) {
        const int64_t lo = n_chunks * t / nt, hi = n_chunks * (t + 1) / nt;
        for (int64_t c = lo; c < hi; ++c) {
            const double* vp = values_p ? values_p + chunks[c].base_p : nullptr;
            const double* vq = values_q ? values_q + chunks[c].base_q : nullptr;
            const int64_t r0 = c * CH, r1 = std::min(m, r0 + CH);
            uint32_t ip = 0, iq = 0;
            for (int64_t r = r0; r < r1; r += 16) {
                uint32_t w = codes[r >> 4];
                const int64_t e = std::min<int64_t>(r + 16, r1);
                for (int64_t i = r; i < e; ++i, w >>= 2) {
                    const uint32_t cd = w & 3u;
                    if (cd == 0u) { p[i] = 1.0; if (q) q[i] = 1.0; if (keep) keep[i] = 1; }
                    else if (cd == 1u) { p[i] = qnan; if (q) q[i] = qnan; if (keep) keep[i] = 0; }
                    else {
                        if (!vp) { bad = 1; return; }
                        p[i] = vp[ip++];
                        if (keep) keep[i] = p[i] <= 1.0 ? 1 : 0;
                        if (cd == 3u) { if (!vq) { bad = 1; return; } const double v = vq[iq++]; if (q) q[i] = v; }
                        else if (q) q[i] = 1.0;
                    }
                }
            }
            if (ip != chunks[c].n_p || iq != chunks[c].n_q) { bad = 1; return; }
        }
    };
    std::vector<std::thread> pool;
    for (int t = 1; t < nt; ++t) pool.emplace_back(work, t);
    work(0);
    for (auto& th : pool) th.join();
    if (bad) { set_error("bbkio_unpack_scores: the code words and the chunk table disagree (or a value list is missing)"); return BBKIO_E_INVALID; }
    return BBKIO_OK;
}

extern "C" int bbkio_unpack_scores(const uint32_t* codes, const void* chunks_v, const double* values_p, const double* values_q,
                                   int64_t m, double* p, double* q, int32_t threads) {
    return unpack_scores_impl(codes, chunks_v, values_p, values_q, m, p, q, nullptr, threads);
}

extern "C" int bbkio_unpack_scores_keep(const uint32_t* codes, const void* chunks_v, const double* values_p, const double* values_q,
                                        int64_t m, double* p, double* q, uint8_t* keep, int32_t threads) {
    return unpack_scores_impl(codes, chunks_v, values_p, values_q, m, p, q, keep, threads);
}

// ---- bbkio_copy_bytes: a large host copy by all cores (numpy columns into pinned staging memory and back) ---------------
extern "C" int bbkio_copy_bytes(void* dst, const void* src, size_t n, int32_t threads) {
    if (n == 0) return BBKIO_OK;
    if (!dst || !src) { set_error("bbkio_copy_bytes: null pointer"); return BBKIO_E_INVALID; }
    int nt = threads > 0 ? threads : (int)std::thread::hardware_concurrency();
    if (nt < 1) nt = 1;
    const size_t min_piece = (size_t)4 << 20;
    if ((size_t)nt > n / min_piece) nt = (int)std::max<size_t>(1, n / min_piece);
    auto work = [&](int t) {
        const size_t lo = n / nt * t, hi = t == nt - 1 ? n : n / nt * (t + 1);
        memcpy(static_cast<char*>(dst) + lo, static_cast<const char*>(src) + lo, hi - lo);
    };
    std::vector<std::thread> pool;
    for (int t = 1; t < nt; ++t) pool.emplace_back(work, t);
    work(0);
    for (auto& th : pool) th.join();
    return BBKIO_OK;
}

// ---- bbkio_pack_records / bbkio_check_records: the packed contact records of a pass (format: bbk.h, BbkRecHeader) ------
namespace {

static_assert(sizeof(BbkRecHeader) == 32, "the record header is 32 bytes");
static_assert(sizeof(BbkRecChunk) == 64, "a chunk record is 64 bytes");
constexpr int64_t RC = BBK_REC_CHUNK;
constexpr int REC_MAX_BITS[3] = {32, 33, 32};

int64_t rec_chunks(int64_t rows) { return rows <= 0 ? 0 : (rows + RC - 1) / RC; }
uint64_t rec_payload(int64_t n, const uint8_t* bits) {
    return BBK_REC_COL_BYTES(n, bits[0]) + BBK_REC_COL_BYTES(n, bits[1]) + BBK_REC_COL_BYTES(n, bits[2]);
}

// exact division and divisibility by a fixed d > 0: d = odd << k, and odd * inv == 1 (mod 2^64)
struct ExactDiv {
    uint64_t inv = 1, lim = ~0ull;
    int k = 0;
    explicit ExactDiv(uint64_t d) {
        while (!(d & 1)) { d >>= 1; ++k; }
        uint64_t x = d;                                     // Newton: 3 -> 6 -> 12 -> 24 -> 48 -> 96 correct bits
        for (int i = 0; i < 5; ++i) x *= 2 - d * x;
        inv = x;
        lim = ~0ull / d;
    }
    bool divides(uint64_t x) const { return !(x & ((1ull << k) - 1)) && (x >> k) * inv <= lim; }
    uint64_t div(uint64_t x) const { return (x >> k) * inv; }
};

uint64_t gcd64(uint64_t a, uint64_t b) {
    while (b) { const uint64_t t = a % b; a = b; b = t; }
    return a;
}

struct RecSource {
    const int32_t* const* mid1;
    const int32_t* const* mid2;
    const int32_t* const* count;
    std::vector<int64_t> starts, sizes;       // the pass layout: shard i at starts[i], a multiple of 4
    // rows [r0, r1) of the layout into local columns (padding rows are zeros)
    void load(int64_t r0, int64_t r1, int32_t* m1, int32_t* m2, int32_t* ct) const {
        const int64_t n = r1 - r0;
        memset(m1, 0, n * 4); memset(m2, 0, n * 4); memset(ct, 0, n * 4);
        size_t i = std::upper_bound(starts.begin(), starts.end(), r0) - starts.begin();
        i = i ? i - 1 : 0;
        for (; i < starts.size() && starts[i] < r1; ++i) {
            const int64_t a = std::max(r0, starts[i]), b = std::min(r1, starts[i] + sizes[i]);
            if (b <= a) continue;
            const int64_t o = a - starts[i];
            memcpy(m1 + (a - r0), mid1[i] + o, (b - a) * 4);
            memcpy(m2 + (a - r0), mid2[i] + o, (b - a) * 4);
            memcpy(ct + (a - r0), count[i] + o, (b - a) * 4);
        }
    }
};

inline int64_t rec_value(int j, const int32_t* m1, const int32_t* m2, const int32_t* ct, int64_t i) {
    return j == 0 ? (int64_t)m1[i] : j == 1 ? (int64_t)m2[i] - (int64_t)m1[i] : (int64_t)ct[i];
}

// phase 1: base, step, bits of the chunk's three columns
void rec_stats(const int32_t* m1, const int32_t* m2, const int32_t* ct, int64_t n, BbkRecChunk& C) {
    for (int j = 0; j < 3; ++j) {
        const int64_t v0 = rec_value(j, m1, m2, ct, 0);
        int64_t mn = v0, mx = v0;
        uint64_t g = 0;                                  // gcd of |v - v0| over the chunk = gcd of v - min
        ExactDiv dv(1);
        for (int64_t i = 0; i < n; ++i) {
            const int64_t v = rec_value(j, m1, m2, ct, i);
            mn = std::min(mn, v); mx = std::max(mx, v);
            const uint64_t d = v >= v0 ? (uint64_t)(v - v0) : (uint64_t)(v0 - v);
            if (g == 1 || d == 0) continue;
            if (g == 0 || !dv.divides(d)) { g = gcd64(g, d); dv = ExactDiv(g); }
        }
        const uint64_t step = g ? g : 1, span = dv.div((uint64_t)(mx - mn));
        C.base[j] = mn;
        C.step[j] = step;
        C.bits[j] = (uint8_t)(span ? 64 - __builtin_clzll(span) : 0);
    }
}

// phase 2: u = (v - base) / step, bits[j] bits each, into the column blocks from `dst`
void rec_encode(const int32_t* m1, const int32_t* m2, const int32_t* ct, int64_t n, const BbkRecChunk& C, uint8_t* dst) {
    for (int j = 0; j < 3; ++j) {
        const int b = C.bits[j];
        const uint64_t bytes = BBK_REC_COL_BYTES(n, b);
        uint64_t* w = reinterpret_cast<uint64_t*>(dst);
        memset(dst, 0, bytes);
        dst += bytes;
        if (!b) continue;
        const ExactDiv dv(C.step[j]);
        const int64_t base = C.base[j];
        uint64_t acc = 0;
        int fill = 0;
        size_t k = 0;
        for (int64_t i = 0; i < n; ++i) {
            const uint64_t u = dv.div((uint64_t)(rec_value(j, m1, m2, ct, i) - base));
            acc |= u << fill;
            fill += b;
            if (fill >= 64) {
                w[k++] = acc;
                fill -= 64;
                acc = fill ? u >> (b - fill) : 0;
            }
        }
        if (fill) w[k] = acc;
    }
}

template <class F>
void rec_parallel(int64_t n_chunks, int threads, F&& f) {
    int nt = threads > 0 ? threads : (int)std::thread::hardware_concurrency();
    if (nt < 1) nt = 1;
    if ((int64_t)nt > n_chunks) nt = (int)std::max<int64_t>(1, n_chunks);
    auto work = [&](int t) {
        std::vector<int32_t> buf(3 * RC);
        const int64_t lo = n_chunks * t / nt, hi = n_chunks * (t + 1) / nt;
        for (int64_t c = lo; c < hi; ++c) f(c, buf.data(), buf.data() + RC, buf.data() + 2 * RC);
    };
    std::vector<std::thread> pool;
    for (int t = 1; t < nt; ++t) pool.emplace_back(work, t);
    work(0);
    for (auto& th : pool) th.join();
}

}  // namespace

extern "C" uint64_t bbkio_pack_records_bound(int64_t rows) {
    const int64_t nc = rec_chunks(rows);
    uint64_t total = sizeof(BbkRecHeader) + (uint64_t)nc * sizeof(BbkRecChunk);
    if (nc) {
        const uint8_t worst[3] = {32, 33, 32};
        total += (uint64_t)(nc - 1) * rec_payload(RC, worst) + rec_payload(rows - (nc - 1) * RC, worst);
    }
    return total;
}

extern "C" int bbkio_pack_records(const int32_t* const* mid1, const int32_t* const* mid2, const int32_t* const* count,
                                  const int64_t* sizes, int32_t n_shards, void* out, uint64_t capacity, uint64_t* bytes,
                                  int32_t threads) {
    if (n_shards < 0 || (n_shards > 0 && (!sizes || !mid1 || !mid2 || !count)) || !out || !bytes) {
        set_error("bbkio_pack_records: bad arguments");
        return BBKIO_E_INVALID;
    }
    RecSource S{mid1, mid2, count, {}, {}};
    int64_t rows = 0;
    for (int i = 0; i < n_shards; ++i) {
        if (sizes[i] < 0 || (sizes[i] > 0 && (!mid1[i] || !mid2[i] || !count[i]))) {
            set_error("bbkio_pack_records: shard %d: negative size or null column", i);
            return BBKIO_E_INVALID;
        }
        S.starts.push_back(rows);
        S.sizes.push_back(sizes[i]);
        rows += (sizes[i] + 3) & ~(int64_t)3;
    }
    const int64_t nc = rec_chunks(rows);
    const uint64_t head = sizeof(BbkRecHeader) + (uint64_t)nc * sizeof(BbkRecChunk);
    if (capacity < head) { set_error("bbkio_pack_records: capacity %llu below the %llu bytes of the tables", (unsigned long long)capacity, (unsigned long long)head); return BBKIO_E_INVALID; }
    BbkRecChunk* table = reinterpret_cast<BbkRecChunk*>(static_cast<uint8_t*>(out) + sizeof(BbkRecHeader));
    // phase 1: every chunk's frame of reference (all cores)
    rec_parallel(nc, threads, [&](int64_t c, int32_t* m1, int32_t* m2, int32_t* ct) {
        const int64_t r0 = c * RC, r1 = std::min(rows, r0 + RC);
        S.load(r0, r1, m1, m2, ct);
        BbkRecChunk C;
        memset(&C, 0, sizeof(C));
        rec_stats(m1, m2, ct, r1 - r0, C);
        table[c] = C;
    });
    // offsets in chunk order: the bytes do not depend on the thread count
    uint64_t at = head;
    for (int64_t c = 0; c < nc; ++c) {
        table[c].offset = at;
        at += rec_payload(std::min(RC, rows - c * RC), table[c].bits);
    }
    *bytes = at;
    if (at > capacity) {
        set_error("bbkio_pack_records: %llu bytes needed, capacity %llu", (unsigned long long)at, (unsigned long long)capacity);
        return BBKIO_E_INVALID;
    }
    // phase 2: the bits (all cores)
    rec_parallel(nc, threads, [&](int64_t c, int32_t* m1, int32_t* m2, int32_t* ct) {
        const int64_t r0 = c * RC, r1 = std::min(rows, r0 + RC);
        S.load(r0, r1, m1, m2, ct);
        rec_encode(m1, m2, ct, r1 - r0, table[c], static_cast<uint8_t*>(out) + table[c].offset);
    });
    BbkRecHeader H;
    memset(&H, 0, sizeof(H));
    H.magic = BBK_REC_MAGIC;
    H.version = BBK_REC_VERSION;
    H.rows = rows;
    H.bytes = at;
    memcpy(out, &H, sizeof(H));
    return BBKIO_OK;
}

extern "C" int bbkio_check_records(const void* buf, uint64_t bytes, int64_t rows) {
    if (!buf || rows < 0) { set_error("bbkio_check_records: bad arguments"); return BBKIO_E_INVALID; }
    if (bytes < sizeof(BbkRecHeader)) { set_error("bbkio_check_records: %llu bytes, shorter than the header", (unsigned long long)bytes); return BBKIO_E_INVALID; }
    BbkRecHeader H;
    memcpy(&H, buf, sizeof(H));
    if (H.magic != BBK_REC_MAGIC || H.version != BBK_REC_VERSION) { set_error("bbkio_check_records: not a packed record buffer (magic / version)"); return BBKIO_E_INVALID; }
    if (H.rows != rows) { set_error("bbkio_check_records: %lld rows, expected %lld", (long long)H.rows, (long long)rows); return BBKIO_E_INVALID; }
    if (H.bytes > bytes) { set_error("bbkio_check_records: the buffer says %llu bytes, only %llu given", (unsigned long long)H.bytes, (unsigned long long)bytes); return BBKIO_E_INVALID; }
    const int64_t nc = rec_chunks(rows);
    if ((uint64_t)nc > H.bytes / sizeof(BbkRecChunk)) { set_error("bbkio_check_records: the chunk table runs past the end"); return BBKIO_E_INVALID; }
    const uint64_t head = sizeof(BbkRecHeader) + (uint64_t)nc * sizeof(BbkRecChunk);
    if (head > H.bytes) { set_error("bbkio_check_records: the chunk table runs past the end"); return BBKIO_E_INVALID; }
    const uint8_t* p = static_cast<const uint8_t*>(buf) + sizeof(BbkRecHeader);
    uint64_t end = head;
    for (int64_t c = 0; c < nc; ++c) {
        BbkRecChunk C;
        memcpy(&C, p + c * sizeof(BbkRecChunk), sizeof(C));
        for (int j = 0; j < 3; ++j)
            if (C.bits[j] > REC_MAX_BITS[j]) { set_error("bbkio_check_records: chunk %lld column %d: %d bits", (long long)c, j, (int)C.bits[j]); return BBKIO_E_INVALID; }
        if (C.offset < end || (C.offset & 15)) { set_error("bbkio_check_records: chunk %lld: offset out of order or misaligned", (long long)c); return BBKIO_E_INVALID; }
        const uint64_t need = rec_payload(std::min(RC, rows - c * RC), C.bits);
        if (C.offset > H.bytes || need > H.bytes - C.offset) { set_error("bbkio_check_records: chunk %lld: payload past the end", (long long)c); return BBKIO_E_INVALID; }
        end = C.offset + need;
    }
    return BBKIO_OK;
}
