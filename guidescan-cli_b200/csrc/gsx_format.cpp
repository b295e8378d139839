// gsx_format.cpp -- host text output: reproduces the reference's CSV / SAM writers byte for byte
// (include/genomics/printer.hpp:18-360) from the result arrays of gsx_enumerate, plus the whole-file driver that
// mirrors do_enumerate_cmd (src/guidescan.cxx:181-258).  Text formatting stays on the host (SURVEY.md section 2).
#include "../../include/gsx.h"
#include "gsx_host.h"
#include "gsx_core.h"
#include "gsx_sites.h"
#include <algorithm>
#include <cstdio>
#include <cstdlib>
#include <chrono>
#include <cstring>
#include <condition_variable>
#include <deque>
#include <map>
#include <memory>
#include <mutex>
#include <string>
#include <thread>
#include <vector>

using namespace gsx;

int gsx_set_error(int code, const std::string& msg);      // gsx_api.cpp

namespace {
thread_local std::string t_err;

inline void put_u64(std::string& s, uint64_t v) {
    char t[24]; int n = 24;
    do { t[--n] = (char)('0' + v % 10); v /= 10; } while (v);
    s.append(t + n, 24 - n);
}
inline void put_float(std::string& s, float f) { char t[64]; int n = snprintf(t, sizeof t, "%f", (double)f); s.append(t, n); }   // std::to_string(float)
// 16 hex digits of a little-endian int64 (printer.hpp:18-88: byte by byte from the low one, high nibble first), four bytes at a time
// in one 64-bit word: bytes spread to 16-bit lanes, nibbles split and swapped into output order, '0'..'9' / 'a'..'f' added without a
// table or a branch.  (A guide at 4 mismatches has hundreds of these; this loop is what the host spends its time in on SAM output.)
inline uint64_t hex8_of_u32(uint32_t x) {
    uint64_t t = x;
    t = (t | (t << 16)) & 0x0000FFFF0000FFFFull;
    t = (t | (t << 8)) & 0x00FF00FF00FF00FFull;                                   // byte i in the low half of 16-bit lane i
    const uint64_t n = ((t >> 4) & 0x000F000F000F000Full) | ((t & 0x000F000F000F000Full) << 8);      // lane: [high nibble][low nibble] in memory order
    const uint64_t alpha = ((n + 0x0606060606060606ull) >> 4) & 0x0101010101010101ull;                 // 1 where the nibble is 10..15
    return n + 0x3030303030303030ull + alpha * 39u;                                // '0' + n, + ('a' - '0' - 10) for letters
}
inline char* put_hex_le64_at(char* w, uint64_t v) {
    const uint64_t lo = hex8_of_u32((uint32_t)v), hi = hex8_of_u32((uint32_t)(v >> 32));
    memcpy(w, &lo, 8); memcpy(w + 8, &hi, 8);                                      // (little-endian host: lane 0 is the first character)
    return w + 16;
}
std::string revcomp(const std::string& x) { std::string r(x.size(), 'N'); for (size_t i = 0; i < x.size(); i++) r[i] = complement_char(x[x.size() - 1 - i]); return r; }

// The results of a call lie in one part per device (gsx_host.h HostArrays), each with its own guide and hit numbering.  The
// formatter reads the parts in place: the merged arrays of the public view are only built when a caller asks for them
// (gsx_result_view_get) -- for a multi-GPU SAM job that concatenation was a second copy of gigabytes per batch.
struct GuideAt {
    const gsx::HostArrays* P; size_t gl; uint64_t b; uint32_t n;      // the part, the guide's number in it, its first hit there, its hit count
};
inline GuideAt guide_at(const gsx_result* r, size_t g) {
    size_t pi = 0;
    if (r->parts.size() > 1) pi = (size_t)(std::upper_bound(r->part_g0.begin(), r->part_g0.end(), g) - r->part_g0.begin()) - 1;
    const HostArrays& P = r->parts[pi];
    const size_t gl = g - r->part_g0[pi];
    return {&P, gl, P.hoff[gl], P.n_hits_of[gl]};
}

struct Base5x4 { uint8_t d[625][4]; constexpr Base5x4() : d() { for (int v = 0; v < 625; v++) { int x = v; for (int j = 0; j < 4; j++) { d[v][j] = (uint8_t)(x % 5); x /= 5; } } } };
static constexpr Base5x4 kBase5{};                                                          // the four base-5 digits of 0 .. 624, lowest first

// match.sequence of hit hl (numbered within the part) of guide g, complemented as printed (= gsx_result_match_sequence,
// printer.hpp:232,264), table-driven: the character selects of gsx_core.h decode_match mispredict on every other character on a host core
inline size_t match_sequence_at(const gsx_result* r, const HostArrays& P, size_t g, uint64_t hl, char* out) {
    static const char UPC[8] = {'T', 'G', 'C', 'A', 'N', '?', '?', '?'};                    // complement of the guide's own symbol
    static const char LOWC[8] = {0, 't', 'g', 'c', 'a', '?', '?', '?'};                      // digit 1..4 = a,c,g,t -> complement
    static const char PAMC[8] = {'T', 'G', 'C', 'N', 'A', '?', '?', '?'};                    // PAM digit A,C,G,N,T -> complement
    static const char WIDEC[16] = {'?', '.', 'T', 'G', 'C', 'N', 'A', 't', 'g', 'c', 'a', '?', '?', '?', '?', '?'};
    const uint32_t len = P.mlen[hl];
    if (r->wide) {
        uint64_t hi = P.key_hi[hl], lo = P.key_lo[hl];
        for (uint32_t i = 0; i < len; i++) { out[i] = WIDEC[hi >> 60]; hi = (hi << 4) | (lo >> 60); lo <<= 4; }
        return len;
    }
    const GuideRec& gr = r->guides[g];
    const uint32_t qlen = gr.qlen;
    // base-5 digits, last character in the lowest digit: a chain of 27 dependent divisions by 5 is the slowest thing in a CSV row, so
    // the key is cut in two halves that divide independently, four digits (a division by 625 and a table of their digits) at a time
    uint8_t dg[32];
    {
        const uint64_t k = P.key_lo[hl];
        uint64_t lo = k % 244140625ull, hi = k / 244140625ull;                               // 5^12: digits len-12 .. len-1 | the rest
        for (int c = 0; c < 3; c++) {
            const uint32_t a = (uint32_t)(lo % 625u), b = (uint32_t)(hi % 625u); lo /= 625u; hi /= 625u;
            memcpy(dg + 4 * c, kBase5.d[a], 4); memcpy(dg + 12 + 4 * c, kBase5.d[b], 4);
        }
        memcpy(dg + 24, kBase5.d[hi % 625u], 4); memcpy(dg + 28, kBase5.d[(hi / 625u) % 625u], 4);      // (a narrow key has at most 27 digits)
    }
    for (uint32_t i = 0; i < len; i++) {                                                     // dg[j] = digit of character len - 1 - j
        const uint32_t d = dg[len - 1u - i];
        const char proto = d ? LOWC[d] : UPC[gr.q[i < kMaxQ ? i : 0] & 7u];
        out[i] = i < qlen ? proto : PAMC[d];
    }
    return len;
}

// decimal digits, two at a time from a 200-byte table (positions have up to ten digits; this and the match string are what a CSV row costs)
struct Digits2 { char d[200]; constexpr Digits2() : d() { for (int i = 0; i < 100; i++) { d[2 * i] = (char)('0' + i / 10); d[2 * i + 1] = (char)('0' + i % 10); } } };
static constexpr Digits2 kDigits2{};
inline char* put_u64_at(char* w, uint64_t v) {
    if (v < 10) { *w = (char)('0' + v); return w + 1; }
    char t[24]; int n = 24;
    while (v >= 100) { const uint64_t q = v / 100; const uint32_t r = (uint32_t)(v - q * 100); v = q; n -= 2; memcpy(t + n, kDigits2.d + 2 * r, 2); }
    if (v >= 10) { n -= 2; memcpy(t + n, kDigits2.d + 2 * v, 2); } else t[--n] = (char)('0' + v);
    memcpy(w, t + n, 24 - n); return w + (24 - n);
}

// One CSV row per counted hit (printer.hpp:244-300).  Rows are assembled in a local buffer and appended once: at millions of
// rows per second per thread the per-field std::string appends were the cost.
void format_csv_guide(const gsx_index* ix, const gsx_result* r, const gsx_guide_row& row, size_t g, const gsx_params* p, bool complete, std::string& out) {
    const GuideAt at = guide_at(r, g);
    const HostArrays& P = *at.P;
    if (P.dropped[at.gl]) return;                                                            // process.hpp:68-70: nothing is printed
    std::string prefix(row.id); prefix += ",";
    if (p->start) { prefix += row.pam; prefix += row.seq; } else { prefix += row.seq; prefix += row.pam; }
    const uint64_t b = at.b; const uint32_t n = at.n;
    if (n == 0) {                                                                            // printer.hpp:190-199
        out += prefix; out += ",NA,NA,NA,0";
        if (complete) out += ",NA,NA,NA";
        out += ",1.0\n";
        return;
    }
    prefix += ",";
    char sp[64]; int spn = snprintf(sp, sizeof sp, "%f", (double)P.specificity[at.gl]);
    constexpr size_t kLine = 1024;
    char line[kLine];
    const bool fits = prefix.size() + 400 < kLine;                                           // (chromosome names are checked per row)
    if (fits) memcpy(line, prefix.data(), prefix.size());
    for (uint64_t h = b; h < b + n; h++) {
        if (!P.counted[h]) continue;
        const std::string& chr = ix->host.chr_names[P.chr[h]];
        if (fits && chr.size() < 256) {
            char* w = line + prefix.size();
            memcpy(w, chr.data(), chr.size()); w += chr.size(); *w++ = ',';
            w = put_u64_at(w, P.pos1[h]); *w++ = ','; *w++ = (char)P.strand[h]; *w++ = ','; w = put_u64_at(w, P.distance[h]);
            if (complete) {
                *w++ = ','; w += match_sequence_at(r, P, g, h, w);
                *w++ = ','; w = put_u64_at(w, P.rna[h]); *w++ = ','; w = put_u64_at(w, P.dna[h]);
            }
            *w++ = ','; memcpy(w, sp, spn); w += spn; *w++ = '\n';
            out.append(line, (size_t)(w - line));
            continue;
        }
        out += prefix;
        out += chr; out += ","; put_u64(out, P.pos1[h]); out += ",";
        out.push_back((char)P.strand[h]); out += ","; put_u64(out, P.distance[h]);
        if (complete) {
            char ms[64]; const size_t ml = match_sequence_at(r, P, g, h, ms);
            out += ","; out.append(ms, ml); out += ","; put_u64(out, P.rna[h]); out += ","; put_u64(out, P.dna[h]);
        }
        out += ","; out.append(sp, spn); out += "\n";
    }
}

void format_sam_guide(const gsx_index* ix, const gsx_result* r, const gsx_guide_row& row, size_t g, const gsx_params* p, bool complete, std::string& out) {
    const GuideAt at = guide_at(r, g);
    const HostArrays& P = *at.P;
    if (P.dropped[at.gl]) return;
    const uint64_t b = at.b; const uint32_t n = at.n, n_dist = r->n_dist;
    if (n == 0) return;
    uint32_t n0 = 0;
    for (uint64_t h = b; h < b + n && P.distance[h] == 0; h++) n0++;
    if (!n0) return;                                                                         // rows exist only for 0-mismatch alignments
    std::string sequence = p->start ? std::string(row.pam) + row.seq : std::string(row.seq) + row.pam;
    std::string seq_out = row.sense_positive ? sequence : revcomp(sequence);
    const uint32_t* cbd = P.cbd + at.gl * n_dist;
    // the row up to the of:H: list, and behind it; the list itself (off_target_fields, printer.hpp:115-170) is written straight into
    // the output buffer: 16 hex digits per counted hit plus a (distance, delimiter) pair per distance -- kilobytes per guide at m = 4
    size_t hex_len = 0;
    if (complete) { size_t cnt = 0; for (uint64_t h = b; h < b + n; h++) cnt += P.counted[h] ? 1 : 0; hex_len = (cnt + 2 * (size_t)n_dist) * 16; }
    char sp[64]; int spn = snprintf(sp, sizeof sp, "%f", (double)P.specificity[at.gl]);
    const int64_t delim = -((int64_t)ix->host.genome_length + 1);
    for (uint64_t h0 = b; h0 < b + n0; h0++) {
        out += row.id; out += "\t"; out += row.sense_positive ? "0" : "16"; out += "\t";
        if (P.chr[h0] >= 0) { out += ix->host.chr_names[P.chr[h0]]; out += "\t"; put_u64(out, P.pos1[h0]); }
        else out += "\t0";                                                                   // sentinel coordinates: chr "" offset 0
        out += "\t100\t"; put_u64(out, sequence.size()); out += "M\t*\t0\t0\t"; out += seq_out; out += "\t*";
        for (uint32_t d = 0; d < n_dist; d++) { out += "\tk"; put_u64(out, d); out += ":i:"; put_u64(out, cbd[d]); }
        if (complete) {
            out += "\tof:H:";
            const size_t at0 = out.size();
            out.resize(at0 + hex_len);
            char* w = &out[at0];
            uint64_t h = b;
            for (uint32_t d = 0; d < n_dist; d++) {
                for (uint32_t j = 0; j < cbd[d]; j++, h++) if (P.counted[h]) w = put_hex_le64_at(w, (uint64_t)P.abs_pos[h]);
                w = put_hex_le64_at(w, d); w = put_hex_le64_at(w, (uint64_t)delim);
            }
        }
        out += "\tsp:f:"; out.append(sp, spn); out += "\n";
    }
}

int ret_buf(const std::string& s, char** buf, size_t* len) {
    char* b = (char*)malloc(s.size() + 1);
    if (!b) { t_err = "out of memory"; return GSX_ERR_NOMEM; }
    memcpy(b, s.data(), s.size()); b[s.size()] = 0;
    *buf = b; *len = s.size();
    return GSX_OK;
}

// guides CSV (reference src/genomics/kmer.cxx:9-25 on fast-cpp-csv-parser with trim_chars<' ','\t'>, no quoting):
// the header must name all six columns (any order); position is parsed but unused downstream.
// The file is read whole and parsed in place by several host threads (fields trimmed and NUL-terminated inside the buffer):
// at a few million guides per second of GPU throughput a getline / std::string reader is what a job would wait for.
struct GuideTable {
    std::vector<char> buf;
    std::vector<const char*> id, seq, pam; std::vector<uint8_t> positive;
    size_t size() const { return id.size(); }
};

std::string trim(const std::string& s) {
    size_t b = 0, e = s.size();
    while (b < e && (s[b] == ' ' || s[b] == '\t')) b++;
    while (e > b && (s[e - 1] == ' ' || s[e - 1] == '\t' || s[e - 1] == '\r')) e--;
    return s.substr(b, e - b);
}

bool read_guides_csv(const char* path, GuideTable& t, std::string& err) {
    FILE* f = fopen(path, "rb");
    if (!f) { err = std::string("cannot open kmers file ") + path; return false; }
    {
        std::vector<char>& b = t.buf; size_t have = 0; b.resize(1 << 20);
        for (;;) { if (have == b.size()) b.resize(b.size() * 2); size_t got = fread(b.data() + have, 1, b.size() - have, f); if (!got) break; have += got; }
        b.resize(have + 1); b[have] = 0;
    }
    fclose(f);
    char* const base = t.buf.data(); const size_t total = t.buf.size() - 1;
    static const char* want[6] = {"id", "sequence", "pam", "chromosome", "position", "sense"};
    int col_of[6] = {-1, -1, -1, -1, -1, -1}; int ncol = 0;
    if (total == 0) { err = "empty kmers file"; return false; }
    size_t body = 0;
    {
        const char* nl = (const char*)memchr(base, '\n', total);
        size_t l = nl ? (size_t)(nl - base) : total; body = nl ? l + 1 : total;
        std::string h(base, l); while (!h.empty() && (h.back() == '\n' || h.back() == '\r')) h.pop_back();
        size_t b = 0;
        for (;;) {
            size_t e = h.find(',', b); std::string name = trim(h.substr(b, e == std::string::npos ? std::string::npos : e - b));
            bool known = false;
            for (int k = 0; k < 6; k++) if (name == want[k]) { col_of[k] = ncol; known = true; }
            if (!known) { err = "Extra column \"" + name + "\" in header of kmers file"; return false; }
            ncol++;
            if (e == std::string::npos) break;
            b = e + 1;
        }
        for (int k = 0; k < 6; k++) if (col_of[k] < 0) { err = std::string("Missing column \"") + want[k] + "\" in header of kmers file"; return false; }
    }
    // body: pieces cut at line starts, one host thread each
    const size_t len = total - body;
    const size_t nt = std::max<size_t>(1, std::min<size_t>({(size_t)16, len / (1 << 20), (size_t)std::max(1u, std::thread::hardware_concurrency())}));
    struct Piece { std::vector<const char*> id, seq, pam; std::vector<uint8_t> positive; bool bad = false; std::string bad_line; };
    std::vector<Piece> pieces(nt);
    std::vector<size_t> cut(nt + 1, total);
    cut[0] = body;
    for (size_t k = 1; k < nt; k++) {
        size_t at = body + len * k / nt;
        if (at < cut[k - 1]) at = cut[k - 1];
        const char* nl = at < total ? (const char*)memchr(base + at, '\n', total - at) : nullptr;
        cut[k] = nl ? (size_t)(nl - base) + 1 : total;
    }
    auto work = [&](size_t k) {
        Piece& P = pieces[k];
        const size_t approx = (cut[k + 1] - cut[k]) / 40 + 16;
        P.id.reserve(approx); P.seq.reserve(approx); P.pam.reserve(approx); P.positive.reserve(approx);
        char* fb[32]; char* fe[32];
        for (size_t at = cut[k]; at < cut[k + 1];) {
            char* line = base + at;
            char* nl = (char*)memchr(line, '\n', cut[k + 1] - at);
            char* end = nl ? nl : base + cut[k + 1];
            at = (size_t)(end - base) + (nl ? 1 : 0);
            while (end > line && (end[-1] == '\n' || end[-1] == '\r')) end--;
            if (end == line) continue;
            int nf = 0; char* b = line; bool too_many = false;
            for (;;) {
                char* e = (char*)memchr(b, ',', (size_t)(end - b));
                if (nf < 32) { fb[nf] = b; fe[nf] = e ? e : end; } else too_many = true;
                nf++;
                if (!e) break;
                b = e + 1;
            }
            if (nf != ncol || too_many) { P.bad = true; P.bad_line.assign(line, end); return; }
            const int need[4] = {col_of[0], col_of[1], col_of[2], col_of[5]};
            const char* out[4];
            for (int q = 0; q < 4; q++) {                                                     // trim_chars<' ', '\t'>, then terminate in place
                char* x = fb[need[q]]; char* y = fe[need[q]];
                while (x < y && (*x == ' ' || *x == '\t')) x++;
                while (y > x && (y[-1] == ' ' || y[-1] == '\t' || y[-1] == '\r')) y--;
                *y = 0; out[q] = x;
            }
            P.id.push_back(out[0]); P.seq.push_back(out[1]); P.pam.push_back(out[2]);
            P.positive.push_back(out[3][0] == '+' && out[3][1] == 0);
        }
    };
    if (nt == 1) work(0);
    else { std::vector<std::thread> th; for (size_t k = 0; k < nt; k++) th.emplace_back(work, k); for (auto& x : th) x.join(); }
    size_t n = 0;
    for (const Piece& P : pieces) { if (P.bad) { err = "wrong number of columns in kmers file line: " + P.bad_line; return false; } n += P.id.size(); }
    t.id.reserve(n); t.seq.reserve(n); t.pam.reserve(n); t.positive.reserve(n);
    for (const Piece& P : pieces) {
        t.id.insert(t.id.end(), P.id.begin(), P.id.end()); t.seq.insert(t.seq.end(), P.seq.begin(), P.seq.end());
        t.pam.insert(t.pam.end(), P.pam.begin(), P.pam.end()); t.positive.insert(t.positive.end(), P.positive.begin(), P.positive.end());
    }
    return true;
}
}  // namespace

extern "C" int gsx_format_header(const gsx_index* ix, int format_sam, int complete, char** buf, size_t* len) {
    if (!ix || !buf || !len) return GSX_ERR_ARG;
    std::string s;
    if (format_sam) {                                                                        // printer.hpp:173-179
        s += "@HD\tVN:1.0\tSO:unknown\n@PG\tID:Guidescan\tVN:2.0.0\n";
        for (size_t i = 0; i < ix->host.chr_names.size(); i++) { s += "@SQ\tSN:" + ix->host.chr_names[i] + "\tLN:"; put_u64(s, ix->host.chr_lens[i]); s += "\n"; }
    } else {                                                                                 // printer.hpp:181-187
        s += "id,sequence,match_chrm,match_position,match_strand,match_distance";
        if (complete) s += ",match_sequence,rna_bulges,dna_bulges";
        s += ",specificity\n";
    }
    return ret_buf(s, buf, len);
}

// Output buffers of the formatter slices, recycled between batches: a multi-GPU SAM job formats gigabytes per batch, and fresh
// allocations of that size are page faults on every 4 KB of them (32 formatter threads fighting over one address-space lock: the
// 8-GPU run of configs[4] spent more time there than in the search).  A buffer handed back keeps its capacity.
namespace {
struct StringPool {
    std::mutex mu; std::vector<std::string> free_;
    std::string get() { std::lock_guard<std::mutex> g(mu); if (free_.empty()) return std::string(); std::string s = std::move(free_.back()); free_.pop_back(); return s; }
    void put(std::string&& s) { s.clear(); std::lock_guard<std::mutex> g(mu); if (free_.size() < 128 && s.capacity() <= (512u << 20)) free_.push_back(std::move(s)); }
};
StringPool& string_pool() { static StringPool p; return p; }
}  // namespace

// guides are independent: slices are formatted on host threads into their own buffers, in guide order
static void format_rows_parts(const gsx_index* ix, const gsx_result* r, const gsx_guide_row* rows, size_t g0, size_t g1,
                              const gsx_params* p, int format_sam, int complete, std::vector<std::string>& parts) {
    size_t n = g1 - g0;
    // slices of about equal numbers of ROWS (a guide with bulges has thousands of hits, a plain one about ten), cut at guides
    const std::vector<uint64_t>& first_hit = r->first_hit;                                   // (n_guides + 1 entries)
    const uint64_t h0 = n ? first_hit[g0] : 0, h1 = n ? first_hit[g1] : 0;
    // (with several devices every device job has a host thread that must stay responsive -- it launches that device's kernels between
    // read-backs -- so those cores are left to them)
    unsigned hw = std::max(1u, std::thread::hardware_concurrency());
    if (ix->dev.size() > 1 && hw > 2 * ix->dev.size() + 2) hw -= (unsigned)ix->dev.size() + 1;
    unsigned nt = (unsigned)std::min<size_t>(hw, std::max<size_t>({(size_t)1, n / 2048, (size_t)((h1 - h0) / 32768)}));
    if (const char* e = getenv("GSX_FORMAT_THREADS")) if (*e) nt = (unsigned)std::max(1, atoi(e));      // tests
    if (nt > n) nt = (unsigned)std::max<size_t>(1, n);
    std::vector<size_t> cut(nt + 1, g1);
    cut[0] = g0;
    for (unsigned t = 1; t < nt; t++) {
        const uint64_t target = h0 + (h1 - h0) * t / nt + (uint64_t)n * t / nt;               // rows + guides: guides without hits still cost a row
        size_t lo = cut[t - 1], hi = g1;                                                     // first guide whose (first_hit + index) reaches the target
        while (lo < hi) { const size_t mid = lo + (hi - lo) / 2; if (first_hit[mid] + (mid - g0) < target) lo = mid + 1; else hi = mid; }
        cut[t] = lo;
    }
    for (std::string& old : parts) string_pool().put(std::move(old));
    parts.clear(); parts.resize(nt);
    for (unsigned t = 0; t < nt; t++) parts[t] = string_pool().get();
    auto work = [&](unsigned t) {
        size_t a = cut[t], b = cut[t + 1];
        std::string& o = parts[t];
        size_t hits = (b > a) ? (size_t)(first_hit[b] - first_hit[a]) : 0;
        // (SAM complete: 16 hex digits per hit in the of:H: list, a few hundred bytes of row around it)
        o.reserve(format_sam ? (b - a) * 320 + (complete ? hits * 17 : 0) : hits * 112 + (b - a) * 64);
        for (size_t g = a; g < b; g++) {
            if (format_sam) format_sam_guide(ix, r, rows[g - g0], g, p, complete != 0, o);
            else format_csv_guide(ix, r, rows[g - g0], g, p, complete != 0, o);
        }
    };
    if (nt == 1) work(0);
    else { std::vector<std::thread> th; for (unsigned t = 0; t < nt; t++) th.emplace_back(work, t); for (auto& x : th) x.join(); }
}

extern "C" int gsx_format_rows(const gsx_index* ix, const gsx_result* r, const gsx_guide_row* rows, size_t g0, size_t g1,
                               const gsx_params* p, int format_sam, int complete, char** buf, size_t* len) {
    if (!ix || !r || !rows || !p || !buf || !len || g1 > r->view.n_guides || g0 > g1) return GSX_ERR_ARG;
    std::vector<std::string> parts;
    format_rows_parts(ix, r, rows, g0, g1, p, format_sam, complete, parts);
    size_t tot = 0; for (auto& s : parts) tot += s.size();
    char* b = (char*)malloc(tot + 1);
    if (!b) return GSX_ERR_NOMEM;
    size_t o = 0; for (auto& s : parts) { memcpy(b + o, s.data(), s.size()); o += s.size(); }
    b[tot] = 0; *buf = b; *len = tot;
    for (std::string& s : parts) string_pool().put(std::move(s));
    return GSX_OK;
}

// ---- guides CSV as an ABI object (what genomics::kmer_producer is to the reference, src/genomics/kmer.cxx:9-25) -------------
struct gsx_guide_table { GuideTable t; };

extern "C" int gsx_guides_csv_open(const char* path, gsx_guide_table** out, size_t* n_guides) {
    if (!path || !out) return gsx_set_error(GSX_ERR_ARG, "null argument");
    *out = nullptr;
    gsx_guide_table* g = new gsx_guide_table(); std::string err;
    if (!read_guides_csv(path, g->t, err)) { delete g; return gsx_set_error(GSX_ERR_IO, err); }
    if (n_guides) *n_guides = g->t.size();
    *out = g;
    return GSX_OK;
}
extern "C" int gsx_guides_csv_row(const gsx_guide_table* g, size_t i, gsx_guide_row* row) {
    if (!g || !row || i >= g->t.size()) return gsx_set_error(GSX_ERR_ARG, "row out of range");
    row->id = g->t.id[i]; row->seq = g->t.seq[i]; row->pam = g->t.pam[i]; row->sense_positive = (int)g->t.positive[i];
    return GSX_OK;
}
extern "C" void gsx_guides_csv_close(gsx_guide_table* g) { delete g; }

// ---- output file ---------------------------------------------------------------------------------------------------------
// The formatting workers leave one buffer per slice; how those reach the file is a property of the file system more than of this
// code.  Measured on the GPU box's /tmp with 1.09 GB of CSV (profiles/r02f_session_3100mb_files_skew.jsonl): ONE sequential write(2)
// stream 2.02 GB/s, every slice at its own offset on its own thread (pwrite) 1.60 GB/s -- buffered writes to one inode serialise and
// the threads only add contention --, slices copied into a shared mapping of the extended file 1.12 GB/s; tmpfs takes 2.5 GB/s in
// every mode and /dev/null 3.2 M guides/s, i.e. the formatter keeps up with the GPU and the file system is what a file-to-file job
// waits for.  GSX_OUT_MODE = "write" (default) | "pwrite" | "mmap".
#include <fcntl.h>
#include <sys/mman.h>
#include <sys/stat.h>
#include <unistd.h>
namespace {
struct OutFile {
    int fd = -1; uint64_t size = 0; int mode = 0;       // 0 write, 1 pwrite, 2 mmap
    bool open(const char* path) {
        fd = ::open(path, O_RDWR | O_CREAT | O_TRUNC, 0644);
        if (fd < 0) { fd = ::open(path, O_WRONLY | O_CREAT | O_TRUNC, 0644); if (fd < 0) return false; }
        struct stat st;
        const bool regular = fstat(fd, &st) == 0 && S_ISREG(st.st_mode);
        const char* e = getenv("GSX_OUT_MODE");
        mode = !regular ? 0 : (e && !strcmp(e, "pwrite")) ? 1 : (e && !strcmp(e, "mmap")) ? 2 : 0;
        return true;
    }
    static bool write_all(int fd, const char* p, size_t n) {
        while (n) { ssize_t w = ::write(fd, p, n); if (w < 0) return false; p += w; n -= (size_t)w; }
        return true;
    }
    static bool pwrite_all(int fd, const char* p, size_t n, uint64_t off) {
        while (n) { ssize_t w = ::pwrite(fd, p, n, (off_t)off); if (w < 0) return false; p += w; n -= (size_t)w; off += (uint64_t)w; }
        return true;
    }
    // appends the parts in order; in the threaded modes the copies run on up to parts.size() threads
    bool append(const std::vector<std::string>& parts) {
        uint64_t total = 0; for (const std::string& s : parts) total += s.size();
        if (!total) return true;
        if (mode == 1) {
            std::vector<std::thread> th; std::vector<char> ok(parts.size(), 1); uint64_t off = size; size_t k = 0;
            for (const std::string& s : parts) {
                if (!s.empty()) th.emplace_back([this, off, &s, &ok, k] { ok[k] = pwrite_all(fd, s.data(), s.size(), off) ? 1 : 0; });
                off += s.size(); k++;
            }
            for (auto& t : th) t.join();
            for (char c : ok) if (!c) return false;
            size += total;
            return true;
        }
        if (mode == 2) {
            const uint64_t page = (uint64_t)sysconf(_SC_PAGESIZE), map_off = size & ~(page - 1), len = size + total - map_off;
            if (ftruncate(fd, (off_t)(size + total)) == 0) {
                void* m = mmap(nullptr, (size_t)len, PROT_READ | PROT_WRITE, MAP_SHARED, fd, (off_t)map_off);
                if (m != MAP_FAILED) {
                    char* dst = (char*)m + (size - map_off);
                    std::vector<std::thread> th; uint64_t off = 0;
                    for (const std::string& s : parts) { if (!s.empty()) th.emplace_back([dst, off, &s] { memcpy(dst + off, s.data(), s.size()); }); off += s.size(); }
                    for (auto& t : th) t.join();
                    munmap(m, (size_t)len);
                    size += total;
                    return true;
                }
                if (ftruncate(fd, (off_t)size) != 0) return false;
            }
            mode = 0;                                                         // (not extendable / not mappable after all: sequential writes from here)
            if (lseek(fd, (off_t)size, SEEK_SET) < 0) return false;
        }
        for (const std::string& s : parts) if (!s.empty() && !write_all(fd, s.data(), s.size())) return false;
        size += total;
        return true;
    }
    bool close_file() { const bool ok = fd < 0 || ::close(fd) == 0; fd = -1; return ok; }
};
}  // namespace

// test hook (not part of the ABI in include/gsx.h): `rounds` appends of the given parts through the output writer above
extern "C" int gsx_internal_write_parts(const char* path, const char* const* parts, const size_t* lens, size_t n_parts, size_t rounds) {
    OutFile out;
    if (!out.open(path)) return GSX_ERR_IO;
    std::vector<std::string> v;
    for (size_t i = 0; i < n_parts; i++) v.emplace_back(parts[i], lens[i]);
    bool ok = true;
    for (size_t r = 0; r < rounds && ok; r++) ok = out.append(v);
    return out.close_file() && ok ? GSX_OK : GSX_ERR_IO;
}

// test hook (not part of the ABI): the formatter alone, as the whole-file driver runs it -- `rounds` passes over the rows of a result
// into pooled buffers, nothing concatenated or written; seconds and bytes of the last pass
extern "C" int gsx_internal_format_rate(const gsx_index* ix, const gsx_result* r, const gsx_guide_row* rows, size_t n, const gsx_params* p,
                                        int format_sam, int complete, size_t rounds, double* seconds, size_t* bytes) {
    if (!ix || !r || !rows || !p || !seconds || !bytes) return GSX_ERR_ARG;
    for (size_t k = 0; k < rounds; k++) {
        std::vector<std::string> parts;
        const auto t0 = std::chrono::steady_clock::now();
        format_rows_parts(ix, r, rows, 0, n, p, format_sam, complete, parts);
        *seconds = std::chrono::duration<double>(std::chrono::steady_clock::now() - t0).count();
        *bytes = 0; for (auto& x : parts) *bytes += x.size();
        for (std::string& x : parts) string_pool().put(std::move(x));
    }
    return GSX_OK;
}

// ---- whole-file driver -------------------------------------------------------------------------------------------------------
// The guides come from a batch source: the parsed guides CSV (gsx_enumerate_file) or the PAM sites of a genome (gsx_enumerate_genome).
// A batch owns what its rows point to that the source does not keep (`arena`); it lives until the formatter has released it.
namespace {
struct GuideBatch {
    std::vector<gsx_guide> g; std::vector<gsx_guide_row> rows;
    std::string arena;
};
struct BatchSource {
    virtual ~BatchSource() = default;
    // the next at most `max` guides in output order into b; false when there are none left.  Throws gsx::SiteError.
    virtual bool next(size_t max, GuideBatch& b) = 0;
    virtual std::string timing() const { return std::string(); }        // appended to the GSX_FILE_TIMING line
};

struct TableSource : BatchSource {
    const GuideTable& t; size_t at = 0;
    explicit TableSource(const GuideTable& tt) : t(tt) {}
    bool next(size_t max, GuideBatch& b) override {
        const size_t b1 = std::min(t.size(), at + max);
        if (at >= b1) return false;
        b.g.resize(b1 - at); b.rows.resize(b1 - at);
        for (size_t i = at; i < b1; i++) { b.g[i - at] = {t.seq[i], t.pam[i]}; b.rows[i - at] = {t.id[i], t.seq[i], t.pam[i], (int)t.positive[i]}; }
        at = b1;
        return true;
    }
};

// Guides per call: the per-device default (or GSX_FILE_BATCH) times the index's devices, fewer with bulges.  n: the guides of the whole
// job when they are known in advance (n_known: a CSV), which lets a short job use smaller batches.
size_t file_batch_guides(const gsx_index* ix, const gsx_params* p, uint32_t qlen, bool n_known, size_t n) {
    // a batch large enough for the slice-major kernels, small enough that its hits fit the arenas: a guide with bulges has
    // thousands of edited forms and about ten hits per form
    const char* e = getenv("GSX_FILE_BATCH");
    size_t batch_guides = e && *e ? (size_t)atoll(e) : 200000;                                 // per device
    if (p->rna_bulges || p->dna_bulges) {
        const uint64_t forms = std::max<uint64_t>(1, bulge_variant_count(std::min<uint32_t>(qlen, 31), p->rna_bulges, p->dna_bulges));
        batch_guides = (size_t)std::min<uint64_t>(batch_guides, std::max<uint64_t>(64, (4u << 20) / forms));
    }
    batch_guides *= (size_t)std::max(1, gsx_index_n_devices(ix));                             // (guides are sharded over the index's devices)
    // a file of only a few such batches: smaller ones, so that formatting and writing batch k still overlap the search of batch
    // k+1 (not below 50 k guides per device: the slice-major kernels lose a fifth of their rate there)
    if (n_known && !(e && *e) && !(p->rna_bulges || p->dna_bulges) && n < 4 * batch_guides)
        batch_guides = std::max<size_t>((n + 3) / 4, (size_t)50000 * (size_t)std::max(1, gsx_index_n_devices(ix)));
    return batch_guides ? batch_guides : 1;
}

// Four things overlap: the GPU enumerates batch k+1 while the host packs the guides of batch k+2 (two-slot gsx_enumerate_start /
// _wait), a formatter thread turns batch k into text on the host cores, and a writer thread copies the text of batch k-1 into the
// output file on several threads; batches go out in file order.  The reference's counterpart is N worker threads behind one
// mutex-guarded ofstream (process.hpp:119-126).
int run_file_job(const gsx_index* ix, BatchSource& src, const char* out_path, const gsx_params* p, int format_sam, int complete,
                 size_t batch_guides, size_t* n_guides, gsx_counters* counters) {
    OutFile out;
    if (!out.open(out_path)) { fprintf(stderr, "gsx: cannot write %s\n", out_path); return gsx_set_error(GSX_ERR_IO, std::string("cannot write ") + out_path); }
    {
        char* buf = nullptr; size_t len = 0;
        gsx_format_header(ix, format_sam, complete, &buf, &len);
        std::vector<std::string> hdr(1, std::string(buf, len)); free(buf);
        if (!out.append(hdr)) { out.close_file(); return gsx_set_error(GSX_ERR_IO, std::string("cannot write ") + out_path); }
    }
    gsx_params pp = *p; pp.sam_scoring = format_sam ? 1 : 0;
    size_t n = 0;                                                                              // guides submitted
    struct Item { gsx_result* r; std::unique_ptr<GuideBatch> b; };
    struct Text { std::vector<std::string> parts; };
    std::mutex mu; std::condition_variable cv;
    std::deque<Item> queue; bool done = false; int wrc = GSX_OK;
    std::deque<Text> wqueue; bool fdone = false;
    gsx_counters total{};
    // GSX_FILE_TIMING=1: where the wall time of the job went (stderr): busy seconds of the formatter and the writer, and how long the
    // submitting thread waited for a finished call and for room in the formatter's queue
    const bool timing = getenv("GSX_FILE_TIMING") != nullptr;
    double s_format = 0, s_free = 0, s_write = 0, s_wait_call = 0, s_wait_queue = 0, s_fwait_writer = 0;
    auto now = [] { return std::chrono::steady_clock::now(); };
    auto since = [](std::chrono::steady_clock::time_point t) { return std::chrono::duration<double>(std::chrono::steady_clock::now() - t).count(); };
    const auto t_job = now();
    std::thread writer([&] {
        for (;;) {
            Text tx;
            { std::unique_lock<std::mutex> lk(mu); cv.wait(lk, [&] { return !wqueue.empty() || fdone; }); if (wqueue.empty()) return; tx = std::move(wqueue.front()); }
            const auto tw = now();
            if (wrc == GSX_OK && !out.append(tx.parts)) wrc = GSX_ERR_IO;
            s_write += since(tw);
            for (std::string& sp : tx.parts) string_pool().put(std::move(sp));
            { std::lock_guard<std::mutex> lk(mu); wqueue.pop_front(); }                // (popped after the work: the formatter stays at most two batches ahead)
            cv.notify_all();
        }
    });
    std::thread formatter([&] {
        for (;;) {
            Item it;
            { std::unique_lock<std::mutex> lk(mu); cv.wait(lk, [&] { return !queue.empty() || done; }); if (queue.empty()) break; it = std::move(queue.front()); }
            Text tx;
            const auto tf = now();
            if (wrc == GSX_OK) {
                format_rows_parts(ix, it.r, it.b->rows.data(), 0, it.b->rows.size(), &pp, format_sam, complete, tx.parts);
                gsx_counters c; gsx_result_counters(it.r, &c);
                total.nodes += c.nodes; total.lookups += c.lookups; total.matches += c.matches; total.hits += c.hits; total.lf_steps += c.lf_steps; total.spills += c.spills; total.launches += c.launches;
                total.ms_search += c.ms_search; total.ms_arrange += c.ms_arrange; total.ms_locate += c.ms_locate; total.ms_score += c.ms_score;
                total.ms_total_device += c.ms_total_device; total.ms_h2d += c.ms_h2d; total.ms_d2h += c.ms_d2h; total.ms_sweep += c.ms_sweep; total.seeds += c.seeds; total.ms_prepare += c.ms_prepare; total.ms_wall += c.ms_wall; total.sectors += c.sectors; total.edited_guides += c.edited_guides;
            }
            s_format += since(tf);
            const auto tr = now();
            gsx_result_free(it.r);
            it.b.reset();
            s_free += since(tr);
            {
                std::unique_lock<std::mutex> lk(mu);
                queue.pop_front();                                                     // (popped after the work: the producer stays at most two batches ahead)
                cv.notify_all();
                const auto tq = now();
                cv.wait(lk, [&] { return wqueue.size() < 2; });
                s_fwait_writer += since(tq);
                wqueue.push_back(std::move(tx));
            }
            cv.notify_all();
        }
        { std::lock_guard<std::mutex> lk(mu); fdone = true; }
        cv.notify_all();
    });
    int rc = GSX_OK; std::string rc_msg;
    // only the per-hit arrays the formatter reads come back from the devices (format_sam_guide: 18 of the 39 bytes per hit,
    // format_csv_guide: 22, 12 in succinct mode)
    const uint32_t want = format_sam ? (kWantDistance | kWantCounted | kWantAbsPos | kWantChr | kWantPos1)
                                     : (kWantDistance | kWantCounted | kWantChr | kWantPos1 | kWantStrand | (complete ? kWantBulges | kWantMatchString : 0u));
    // two batches in flight: the guides of batch k+1 are taken from the source (and its small uploads issued) while batch k runs on the
    // device
    struct Slot { std::unique_ptr<GuideBatch> b; gsx_pending* pd = nullptr; };
    Slot slots[2]; int n_pending = 0, head = 0;
    auto finish_one = [&]() {
        Slot& sl = slots[head]; head ^= 1; n_pending--;
        gsx_result* r = nullptr;
        const auto tc = now();
        const int rc1 = gsx_enumerate_wait(sl.pd, &r); sl.pd = nullptr;
        s_wait_call += since(tc);
        if (rc1) { if (rc == GSX_OK) { rc = rc1; rc_msg = gsx_last_error(); } sl.b.reset(); return; }
        if (rc != GSX_OK) { gsx_result_free(r); sl.b.reset(); return; }
        std::unique_lock<std::mutex> lk(mu);
        const auto tq = now();
        cv.wait(lk, [&] { return queue.size() < 2; });
        s_wait_queue += since(tq);
        queue.push_back({r, std::move(sl.b)});
        lk.unlock(); cv.notify_all();
    };
    while (rc == GSX_OK) {
        if (n_pending == 2) finish_one();
        if (rc != GSX_OK) break;
        Slot& sl = slots[(head + n_pending) & 1];
        sl.b.reset(new GuideBatch());
        try {
            if (!src.next(batch_guides, *sl.b)) { sl.b.reset(); break; }
        } catch (const gsx::SiteError& f) { rc = f.code; rc_msg = f.msg; sl.b.reset(); break; }
        catch (const std::bad_alloc&) { rc = GSX_ERR_NOMEM; rc_msg = "out of host memory"; sl.b.reset(); break; }
        n += sl.b->g.size();
        const int rc1 = gsx_internal_enumerate_start_want(ix, sl.b->g.data(), sl.b->g.size(), &pp, want, &sl.pd);
        if (rc1) { rc = rc1; rc_msg = gsx_last_error(); sl.b.reset(); break; }
        n_pending++;
    }
    while (n_pending) finish_one();
    { std::lock_guard<std::mutex> lk(mu); done = true; }
    cv.notify_all();
    formatter.join(); writer.join();
    if (timing)
        fprintf(stderr, "gsx file job: %.3f s wall, %zu guides in batches of %zu; formatter busy %.3f s (+ %.3f s releasing results, %.3f s waiting for the writer), "
                "writer busy %.3f s; submitter waited %.3f s for calls and %.3f s for the formatter; calls: device %.3f s, d2h %.3f s, h2d %.3f s, prepare %.3f s, call walls %.3f s%s\n",
                since(t_job), n, batch_guides, s_format, s_free, s_fwait_writer, s_write, s_wait_call, s_wait_queue, total.ms_total_device / 1e3, total.ms_d2h / 1e3,
                total.ms_h2d / 1e3, total.ms_prepare / 1e3, total.ms_wall / 1e3, src.timing().c_str());
    if (!out.close_file() && wrc == GSX_OK) wrc = GSX_ERR_IO;
    if (rc) return gsx_set_error(rc, rc_msg);
    if (wrc) return gsx_set_error(wrc, std::string("cannot write ") + out_path);
    if (n_guides) *n_guides = n;
    if (counters) *counters = total;
    return GSX_OK;
}
}  // namespace

extern "C" int gsx_enumerate_file(const gsx_index* ix, const char* kmers_csv, const char* out_path, const gsx_params* p,
                                  int format_sam, int complete, size_t batch_guides, size_t* n_guides, gsx_counters* counters) {
    if (!ix || !kmers_csv || !out_path || !p) return GSX_ERR_ARG;
    GuideTable t; std::string err;
    if (!read_guides_csv(kmers_csv, t, err)) { fprintf(stderr, "gsx: %s\n", err.c_str()); return gsx_set_error(GSX_ERR_IO, err); }
    if (batch_guides == 0) batch_guides = file_batch_guides(ix, p, t.size() ? (uint32_t)std::min<size_t>(strlen(t.seq[0]), 31) : 20, true, t.size());
    TableSource src(t);
    return run_file_job(ix, src, out_path, p, format_sam, complete, batch_guides, n_guides, counters);
}

// ---- genome in, guides enumerated: gsx_generate_kmers -> (BED selection) -> gsx_enumerate_file without the CSV in between --------
namespace {
// The sites of one chromosome at a time from the producer (gsx_sites.h), turned into rows by the generator's own row logic; a
// batch may span chromosomes, so its strings are copied into the batch's arena.
struct GenomeSource : BatchSource {
    gsx::FastaReader rd; gsx::SiteScanner S;
    const std::string pam, prefix; const uint64_t min_len;
    const std::map<std::string, std::vector<std::pair<uint64_t, uint64_t>>>* regions;      // null: every site
    std::string name, seq; std::vector<gsx::StartRange> ranges;
    size_t list = 0, at = 0; bool have_chr = false;
    GenomeSource(FILE* in, const std::string& pam_, uint32_t k, bool start, int device, const std::string& prefix_, uint64_t min_len_,
                 const std::map<std::string, std::vector<std::pair<uint64_t, uint64_t>>>* regions_)
        : rd(in), S(pam_, k, start, device), pam(pam_), prefix(prefix_), min_len(min_len_), regions(regions_) {}
    bool load() {                                                                              // the next chromosome with sites to offer
        for (;;) {
            if (!rd.next(name, &seq, nullptr)) return false;
            if (seq.size() < min_len || seq.empty()) continue;
            if (regions) {
                const auto it = regions->find(name);
                ranges = it == regions->end() ? std::vector<gsx::StartRange>() : gsx::merge_regions(it->second, S.k());
                if (ranges.empty()) continue;
            }
            S.scan(seq, regions ? &ranges : nullptr);
            list = 0; at = 0; have_chr = true;
            return true;
        }
    }
    bool next(size_t max, GuideBatch& b) override {
        std::vector<size_t> off; std::vector<uint8_t> fwd;                                     // id at off[i], k-mer behind it
        while (off.size() < max) {
            if (!have_chr || list == S.n_lists()) { have_chr = false; seq.clear(); if (!load()) break; continue; }
            const std::vector<uint32_t>& v = S.sites(list);
            if (at == v.size()) { list++; at = 0; continue; }
            const bool f = S.forward(list);
            const size_t m = std::min(v.size() - at, max - off.size());
            for (size_t q = at; q < at + m; q++) {
                char num[16]; const int nl = (int)(put_u64_at(num, S.pos1(list, v[q])) - num);
                off.push_back(b.arena.size()); fwd.push_back(f);
                gsx::append_site_id(b.arena, prefix, name, num, nl, f); b.arena += '\0';
                gsx::append_site_kmer(b.arena, seq, S.kmer_start(list, v[q]), S.k(), f); b.arena += '\0';
            }
            at += m;
        }
        if (off.empty()) return false;
        b.g.resize(off.size()); b.rows.resize(off.size());
        for (size_t i = 0; i < off.size(); i++) {
            const char* id = b.arena.data() + off[i]; const char* kmer = id + strlen(id) + 1;
            b.g[i] = {kmer, pam.c_str()}; b.rows[i] = {id, kmer, pam.c_str(), (int)fwd[i]};
        }
        return true;
    }
    std::string timing() const override {
        char t[160]; snprintf(t, sizeof t, "; PAM scan %.3f s over %zu chromosome(s) (+ %.3f s waiting for the device)", S.seconds, S.chromosomes, S.wait_seconds);
        return t;
    }
};

// BED intervals (0-based, half-open) per chromosome, checked against the index's chromosome table
bool read_bed(const char* path, const std::map<std::string, uint64_t>& chr_len, std::map<std::string, std::vector<std::pair<uint64_t, uint64_t>>>& out,
              int& code, std::string& err) {
    FILE* f = fopen(path, "rb");
    if (!f) { code = GSX_ERR_IO; err = std::string("cannot open regions file ") + path; return false; }
    std::string line; char chunk[1 << 16]; size_t lineno = 0; bool ok = true;
    auto parse_u64 = [](const std::string& s, uint64_t& v) {
        if (s.empty() || s.size() > 19) return false;
        v = 0; for (char c : s) { if (c < '0' || c > '9') return false; v = v * 10 + (uint64_t)(c - '0'); }
        return true;
    };
    auto handle = [&](std::string l) {
        lineno++;
        while (!l.empty() && (l.back() == '\n' || l.back() == '\r')) l.pop_back();
        std::vector<std::string> w;
        for (size_t b = 0; b < l.size();) {
            while (b < l.size() && (l[b] == ' ' || l[b] == '\t')) b++;
            size_t e = b; while (e < l.size() && l[e] != ' ' && l[e] != '\t') e++;
            if (e > b) w.push_back(l.substr(b, e - b));
            b = e;
        }
        if (w.empty() || l[0] == '#' || l.compare(0, 5, "track") == 0 || l.compare(0, 7, "browser") == 0) return true;
        code = GSX_ERR_ARG;
        const std::string where = std::string("regions file ") + path + " line " + std::to_string(lineno);
        uint64_t s = 0, e = 0;
        if (w.size() < 3 || !parse_u64(w[1], s) || !parse_u64(w[2], e)) { err = where + ": expected \"chrom start end\""; return false; }
        const auto it = chr_len.find(w[0]);
        if (it == chr_len.end()) { err = where + ": chromosome \"" + w[0] + "\" is not in the index"; return false; }
        if (s > e) { err = where + ": start " + w[1] + " is past end " + w[2]; return false; }
        if (e > it->second) { err = where + ": end " + w[2] + " is past the end of " + w[0] + " (" + std::to_string(it->second) + " bases)"; return false; }
        out[w[0]].emplace_back(s, e);
        return true;
    };
    while (ok && fgets(chunk, sizeof chunk, f)) {
        line += chunk;
        if (line.back() == '\n') { ok = handle(line); line.clear(); }
    }
    if (ok && !line.empty()) ok = handle(line);
    fclose(f);
    return ok;
}
}  // namespace

extern "C" int gsx_enumerate_genome(const gsx_index* ix, const char* fasta_path, const char* pam_c, uint32_t k, uint64_t min_chr_length,
                                    const char* prefix_c, const char* regions_bed, const char* out_path, const gsx_params* p,
                                    int format_sam, int complete, size_t batch_guides, size_t* n_guides, gsx_counters* counters) {
    if (!ix || !fasta_path || !pam_c || !out_path || !p) return gsx_set_error(GSX_ERR_ARG, "null argument");
    if (n_guides) *n_guides = 0;
    // everything is checked before the first device work: options, then the FASTA against the index, then the regions
    const std::string pam(pam_c), prefix(prefix_c ? prefix_c : "");
    if (k < 1 || k > 32) return gsx_set_error(GSX_ERR_ARG, "kmer_length " + std::to_string(k) + " is outside 1..32");
    if (pam.empty() || pam.size() > 8) return gsx_set_error(GSX_ERR_ARG, "PAM \"" + pam + "\" must have 1..8 characters");
    for (char c : pam)
        if (!(c == 'A' || c == 'C' || c == 'G' || c == 'T' || c == 'N'))
            return gsx_set_error(GSX_ERR_ARG, "PAM \"" + pam + "\" has the character '" + std::string(1, c) + "': PAM characters must be A, C, G, T or N");
    std::string longest = pam;
    for (uint32_t i = 0; i < p->n_alt_pams; i++) if (p->alt_pams && p->alt_pams[i] && strlen(p->alt_pams[i]) > longest.size()) longest = p->alt_pams[i];
    if (k + longest.size() + p->dna_bulges > 32)
        return gsx_set_error(GSX_ERR_ARG, "k-mer length " + std::to_string(k) + " + PAM \"" + longest + "\" + " + std::to_string(p->dna_bulges) +
                                              " DNA bulge(s) is longer than 32 characters");
    if (ix->dev.empty()) return gsx_set_error(GSX_ERR_NO_DEVICE, "index is not resident on any device");
    std::map<std::string, uint64_t> chr_len;
    for (size_t i = 0; i < ix->host.chr_names.size(); i++) chr_len[ix->host.chr_names[i]] = ix->host.chr_lens[i];
    FILE* in = fopen(fasta_path, "rb");
    if (!in) return gsx_set_error(GSX_ERR_IO, std::string("cannot open ") + fasta_path);
    {
        gsx::FastaReader rd(in);
        std::string name; uint64_t len = 0;
        while (rd.next(name, nullptr, &len)) {
            if (len < min_chr_length || len == 0) continue;
            const auto it = chr_len.find(name);
            if (it == chr_len.end()) { fclose(in); return gsx_set_error(GSX_ERR_ARG, "FASTA record \"" + name + "\" (" + std::to_string(len) + " bases) is not a chromosome of the index"); }
            if (it->second != len) {
                fclose(in);
                return gsx_set_error(GSX_ERR_ARG, "FASTA record \"" + name + "\" has " + std::to_string(len) + " bases, the index's chromosome of that name " +
                                                      std::to_string(it->second) + ": index and FASTA are of different assemblies");
            }
        }
        rewind(in);
    }
    std::map<std::string, std::vector<std::pair<uint64_t, uint64_t>>> regions;
    if (regions_bed) {
        int code = GSX_OK; std::string err;
        if (!read_bed(regions_bed, chr_len, regions, code, err)) { fclose(in); return gsx_set_error(code, err); }
    }
    if (batch_guides == 0) batch_guides = file_batch_guides(ix, p, k, false, 0);
    int rc;
    try {
        GenomeSource src(in, pam, k, p->start != 0, ix->dev[0].device, prefix, min_chr_length, regions_bed ? &regions : nullptr);
        rc = run_file_job(ix, src, out_path, p, format_sam, complete, batch_guides, n_guides, counters);
    } catch (const gsx::SiteError& f) { rc = gsx_set_error(f.code, f.msg); }
    catch (const std::bad_alloc&) { rc = gsx_set_error(GSX_ERR_NOMEM, "out of host memory"); }
    fclose(in);
    return rc;
}
