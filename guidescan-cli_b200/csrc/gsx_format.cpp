// gsx_format.cpp -- host text output: reproduces the reference's CSV / SAM writers byte for byte
// (include/genomics/printer.hpp:18-360) from the result arrays of gsx_enumerate, plus the whole-file driver that
// mirrors do_enumerate_cmd (src/guidescan.cxx:181-258).  Text formatting stays on the host (SURVEY.md section 2).
#include "../../include/gsx.h"
#include "gsx_host.h"
#include "gsx_core.h"
#include "gsx_sites.h"
#include "gsx_decode.h"
#include "gsx_iupac.h"
#include <algorithm>
#include <atomic>
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
// complement of a SAM SEQ character: IUPAC class letters to their partners (R<->Y, K<->M, B<->V, D<->H; S, W kept), as
// Bio.Seq.reverse_complement does; every other character as complement_char
static char seq_complement(char c) { return iupac_is_class(c) ? iupac_complement(c) : complement_char(c); }
static std::string seq_revcomp(const std::string& x) { std::string r(x.size(), 'N'); for (size_t i = 0; i < x.size(); i++) r[i] = seq_complement(x[x.size() - 1 - i]); return r; }

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
    std::string seq_out = row.sense_positive ? sequence : seq_revcomp(sequence);
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

namespace {
std::string csv_header(bool complete) {                                                     // printer.hpp:181-187
    std::string s = "id,sequence,match_chrm,match_position,match_strand,match_distance";
    if (complete) s += ",match_sequence,rna_bulges,dna_bulges";
    return s + ",specificity\n";
}
}  // namespace

extern "C" int gsx_format_header(const gsx_index* ix, int format_sam, int complete, char** buf, size_t* len) {
    if (!ix || !buf || !len) return GSX_ERR_ARG;
    std::string s;
    if (format_sam) {                                                                        // printer.hpp:173-179
        s += "@HD\tVN:1.0\tSO:unknown\n@PG\tID:Guidescan\tVN:2.0.0\n";
        for (size_t i = 0; i < ix->host.chr_names.size(); i++) { s += "@SQ\tSN:" + ix->host.chr_names[i] + "\tLN:"; put_u64(s, ix->host.chr_lens[i]); s += "\n"; }
    } else s = csv_header(complete != 0);
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
    for (char c : pam) {
        if (!iupac_pam_char(c))
            return gsx_set_error(GSX_ERR_ARG, "PAM \"" + pam + "\" has the character '" + std::string(1, c) +
                                                  "': PAM characters must be A, C, G, T, N or an IUPAC class letter (R, Y, S, W, K, M, B, D, H, V)");
        // the generated guides carry the pattern as their PAM column: without class semantics they could never match
        if (iupac_is_class(c) && !p->iupac_pams)
            return gsx_set_error(GSX_ERR_ARG, "PAM \"" + pam + "\" has the class letter '" + std::string(1, c) + "': it needs iupac_pams (--iupac-pam)");
    }
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

// ---- SAM complete database in, off-target rows out (gsx_decode_database) -------------------------------------------------------
// A host thread reads the SAM in batches of whole lines and splits the records; the of:H: lists go to the device inside the batch's
// own text (gsx_decode.cu), the rows come back as arrays, and a formatter and a writer thread turn them into CSV behind the reader,
// in record order -- the structure of run_file_job.
namespace {
struct DecodeRec {
    const char* id; const char* sp; uint32_t id_len, sp_len;
    uint32_t seq_at, seq_len;              // the guide's sequence in the batch's `seqs`
    uint64_t at;                           // byte offset of the record in the file
};
struct DecodeBatch {
    gsx::PinnedBuf text_buf; const char* text = nullptr; size_t len = 0; uint64_t file_off = 0;
    std::vector<DecodeRec> recs; std::string seqs;
    std::vector<uint64_t> rec_hex; std::vector<uint32_t> rec_entry; std::vector<gsx::DecodeGuide> guides;
    gsx::DecodeRows rows;
    void clear() { recs.clear(); seqs.clear(); rec_hex.clear(); rec_entry.assign(1, 0); guides.clear(); len = 0; }
};

gsx::SiteError decode_error(const std::string& msg) { return gsx::SiteError{GSX_ERR_ARG, msg}; }
std::string quoted(const char* p, size_t n) { return "\"" + std::string(p, std::min<size_t>(n, 200)) + "\""; }

// the SAM in batches of whole lines, about `bytes` each (a longer line makes its batch longer)
struct SamReader {
    FILE* f; uint64_t off = 0; std::string carry; bool eof = false;
    explicit SamReader(FILE* ff) : f(ff) {}
    bool next(size_t bytes, DecodeBatch& b) {
        b.clear(); b.file_off = off;
        size_t cap = std::max(bytes, 2 * carry.size() + 1);
        char* t = (char*)b.text_buf.need(cap); cap = b.text_buf.cap;
        memcpy(t, carry.data(), carry.size());
        size_t have = carry.size(); carry.clear();
        for (;;) {
            while (!eof && have < cap) { const size_t got = fread(t + have, 1, cap - have, f); if (!got) eof = true; have += got; }
            const char* nl = have ? (const char*)memrchr(t, '\n', have) : nullptr;
            if (nl || eof) {
                const size_t keep = nl && !eof ? (size_t)(nl - t) + 1 : have;
                carry.assign(t + keep, have - keep); b.len = keep;
                break;
            }
            std::string whole(t, have);                                                     // one line longer than the batch
            t = (char*)b.text_buf.need(2 * cap); cap = b.text_buf.cap; memcpy(t, whole.data(), have);
        }
        b.text = t; off += b.len;
        return b.len > 0;
    }
};

// one record's fields: QNAME, FLAG, RNAME, POS, SEQ and the two tags the decode reads
struct SamFields {
    const char* f[11]; uint32_t n[11]; int nf = 0;
    const char* of = nullptr; size_t of_len = 0; const char* sp = nullptr; size_t sp_len = 0;
    void split(const char* p, const char* end) {
        nf = 0; of = sp = nullptr;
        for (;;) {
            const char* tab = (const char*)memchr(p, '\t', (size_t)(end - p));
            const char* e = tab ? tab : end;
            if (nf < 11) { f[nf] = p; n[nf] = (uint32_t)(e - p); }
            else if (e - p >= 5 && !memcmp(p, "of:H:", 5)) { of = p + 5; of_len = (size_t)(e - p) - 5; }
            else if (e - p >= 5 && !memcmp(p, "sp:f:", 5)) { sp = p + 5; sp_len = (size_t)(e - p) - 5; }
            nf++;
            if (!tab) break;
            p = tab + 1;
        }
    }
    bool number(int i, uint64_t& v) const {
        if (!n[i] || n[i] > 19) return false;
        v = 0; for (uint32_t k = 0; k < n[i]; k++) { const char c = f[i][k]; if (c < '0' || c > '9') return false; v = v * 10 + (uint64_t)(c - '0'); }
        return true;
    }
};

int64_t hex_le64(const char* p) {                                                           // 16 digits, low byte first (printer.hpp:18-88)
    uint64_t v = 0;
    for (int b = 0; b < 8; b++) {
        int d[2];
        for (int k = 0; k < 2; k++) { const char c = p[2 * b + k], l = (char)(c | 32); d[k] = c >= '0' && c <= '9' ? c - '0' : (l >= 'a' && l <= 'f' ? l - 'a' + 10 : -1); }
        if (d[0] < 0 || d[1] < 0) return 0;
        v |= (uint64_t)(d[0] * 16 + d[1]) << (8 * b);
    }
    return (int64_t)v;
}

// Records of a batch: which are decoded, with their guides.  Consecutive records of one QNAME are one guide: the first is decoded, the
// others must carry the same list.
struct DecodeSplitter {
    uint32_t pam_len; const std::map<std::string, std::vector<std::pair<uint64_t, uint64_t>>>* regions;
    std::map<std::string, std::vector<gsx::StartRange>> ranges; uint32_t ranges_k = 0;      // the regions as site starts for sites of ranges_k bases
    std::string prev_id, prev_of; const char* pid = nullptr; size_t pid_len = 0; const char* pof = nullptr; size_t pof_len = 0; bool have_prev = false;
    size_t records = 0;

    bool selected(const SamFields& F, uint32_t L) {
        if (!regions) return true;
        uint64_t pos = 0;
        if (!F.number(3, pos) || pos == 0) return false;                                     // (a sentinel record, or POS 0)
        if (L != ranges_k) {
            ranges.clear(); ranges_k = L;
            for (const auto& kv : *regions) ranges[kv.first] = gsx::merge_regions(kv.second, L);
        }
        const auto it = ranges.find(std::string(F.f[2], F.n[2]));
        if (it == ranges.end()) return false;
        const uint64_t a = pos - 1;                                                          // the site is [POS - 1, POS - 1 + L)
        const std::vector<gsx::StartRange>& v = it->second;
        const auto r = std::upper_bound(v.begin(), v.end(), a, [](uint64_t x, const gsx::StartRange& s) { return x < s.first; });
        return r != v.begin() && a <= (r - 1)->second;
    }

    void split(DecodeBatch& b) {
        SamFields F;
        for (size_t at = 0; at < b.len;) {
            const char* line = b.text + at;
            const char* nl = (const char*)memchr(line, '\n', b.len - at);
            const char* end = nl ? nl : b.text + b.len;
            const uint64_t where = b.file_off + at;
            at = (size_t)(end - b.text) + (nl ? 1 : 0);
            if (end > line && end[-1] == '\r') end--;
            if (end == line || line[0] == '@') continue;
            records++;
            F.split(line, end);
            auto rec = [&] { return "record " + quoted(F.f[0], F.n[0]) + " at byte " + std::to_string(where); };
            if (F.nf < 11) throw decode_error(rec() + " has " + std::to_string(F.nf) + " tab-separated fields, a SAM record at least 11");
            if (!F.of) throw decode_error(rec() + " has no of:H: tag: a database written with --mode succinct lists no off-targets; write it with --mode complete");
            if (!F.sp) throw decode_error(rec() + " has no sp:f: tag");
            if (F.of_len < 32 || F.of_len % 16) throw decode_error(rec() + ": its of:H: value has " + std::to_string(F.of_len) + " hex digits, not a whole list of 16-digit values (truncated?)");
            if (have_prev && F.n[0] == pid_len && !memcmp(F.f[0], pid, pid_len)) {           // another perfect match of the same guide
                if (F.of_len != pof_len || memcmp(F.of, pof, pof_len)) throw decode_error(rec() + ": its of:H: list differs from the previous record of the same QNAME");
                continue;
            }
            have_prev = true; pid = F.f[0]; pid_len = F.n[0]; pof = F.of; pof_len = F.of_len;
            uint64_t flag = 0;
            if (!F.number(1, flag)) throw decode_error(rec() + ": FLAG " + quoted(F.f[1], F.n[1]) + " is not a number");
            const uint32_t L = F.n[9];
            if (L <= pam_len || L - pam_len > (uint32_t)kMaxQ)
                throw decode_error(rec() + ": SEQ has " + std::to_string(L) + " bases; with a PAM column of " + std::to_string(pam_len) + " the protospacer must have 1.." + std::to_string(kMaxQ));
            if (!selected(F, L)) continue;
            gsx::DecodeGuide g{};
            const char* s = F.f[9];
            for (uint32_t i = 0; i < L; i++) g.seq[i] = (flag & 16) ? seq_complement(s[L - 1 - i]) : s[i];
            g.qlen = (uint8_t)(L - pam_len); g.plen = (uint8_t)pam_len;
            b.recs.push_back({F.f[0], F.sp, F.n[0], (uint32_t)F.sp_len, (uint32_t)b.seqs.size(), L, where});
            b.seqs.append(g.seq, L);
            b.guides.push_back(g);
            b.rec_hex.push_back((uint64_t)(F.of - b.text));
            b.rec_entry.push_back(b.rec_entry.back() + (uint32_t)(F.of_len / 16));
        }
        if (have_prev) {                                                                     // the next batch compares with a copy
            prev_id.assign(pid, pid_len); prev_of.assign(pof, pof_len);
            pid = prev_id.data(); pof = prev_of.data();
        }
    }
};

// the rows of records [r0, r1) of a decoded batch, as format_csv_guide prints them (+ the CFD column)
void format_decoded(const DecodeBatch& b, size_t r0, size_t r1, const std::vector<std::string>& chr_names, bool complete, bool with_cfd, std::string& o) {
    const gsx::DecodeRows& R = b.rows;
    std::vector<char> line;
    for (size_t r = r0; r < r1; r++) {
        const DecodeRec& c = b.recs[r];
        const uint32_t h0 = R.rec_row[r], h1 = R.rec_row[r + 1];
        if (h0 == h1) continue;
        const size_t need = c.id_len + c.seq_len + c.sp_len + 2 * (kMaxQ + kMaxPamLen) + 96;
        size_t prefix = c.id_len + 1 + c.seq_len + 1;
        if (line.size() < need) line.resize(need + 256);
        char* l = line.data();
        memcpy(l, c.id, c.id_len); l[c.id_len] = ','; memcpy(l + c.id_len + 1, b.seqs.data() + c.seq_at, c.seq_len); l[prefix - 1] = ',';
        for (uint32_t h = h0; h < h1; h++) {
            const std::string& chr = chr_names[R.chr[h]];
            if (line.size() < need + chr.size()) { line.resize(need + chr.size() + 256); l = line.data(); }
            char* w = l + prefix;
            memcpy(w, chr.data(), chr.size()); w += chr.size(); *w++ = ',';
            w = put_u64_at(w, R.pos1[h]); *w++ = ','; *w++ = (char)R.strand[h]; *w++ = ','; w = put_u64_at(w, R.distance[h]);
            if (complete) {
                *w++ = ','; memcpy(w, R.match + (size_t)h * R.stride, c.seq_len); w += c.seq_len;
                memcpy(w, ",0,0", 4); w += 4;
            }
            *w++ = ','; memcpy(w, c.sp, c.sp_len); w += c.sp_len;
            if (with_cfd) { *w++ = ','; w += snprintf(w, 32, "%.9g", (double)R.cfd[h]); }
            *w++ = '\n';
            o.append(l, (size_t)(w - l));
        }
    }
}
}  // namespace

extern "C" int gsx_decode_database(const char* sam_path, const char* fasta_path, const char* out_path, uint32_t pam_length,
                                   const char* const* alt_pams, uint32_t n_alt_pams, int complete, int with_cfd, const char* regions_bed,
                                   int device, size_t* n_guides, size_t* n_rows) {
    if (!sam_path || !fasta_path || !out_path || (n_alt_pams && !alt_pams)) return gsx_set_error(GSX_ERR_ARG, "null argument");
    if (n_guides) *n_guides = 0;
    if (n_rows) *n_rows = 0;
    // everything is checked before the first device work: options, the SAM's header and first list against the FASTA, the regions
    if (pam_length < 1 || pam_length > (uint32_t)kMaxPamLen) return gsx_set_error(GSX_ERR_ARG, "pam_length " + std::to_string(pam_length) + " is outside 1.." + std::to_string(kMaxPamLen));
    if (n_alt_pams > (uint32_t)kMaxPams - 1) return gsx_set_error(GSX_ERR_ARG, std::to_string(n_alt_pams) + " alternative PAMs: at most " + std::to_string(kMaxPams - 1));
    gsx::DecodePams pams{};
    pams.n = n_alt_pams;
    for (uint32_t i = 0; i < n_alt_pams; i++) {
        const std::string a = alt_pams[i] ? alt_pams[i] : "";
        if (a.size() != pam_length) return gsx_set_error(GSX_ERR_ARG, "alternative PAM \"" + a + "\" has " + std::to_string(a.size()) + " characters, the PAM column " + std::to_string(pam_length));
        for (char c : a)
            if (!iupac_pam_char(c))
                return gsx_set_error(GSX_ERR_ARG, "alternative PAM \"" + a + "\" has the character '" + std::string(1, c) +
                                                      "': PAM characters must be A, C, G, T, N or an IUPAC class letter (R, Y, S, W, K, M, B, D, H, V)");
        memcpy(pams.p[i], a.data(), a.size());
    }
    if (device < 0) return gsx_set_error(GSX_ERR_ARG, "device " + std::to_string(device) + " is not a device ordinal");
    FILE* in = fopen(sam_path, "rb");
    if (!in) return gsx_set_error(GSX_ERR_IO, std::string("cannot open ") + sam_path);
    struct Closer { FILE* f; ~Closer() { fclose(f); } } closer{in};
    // the header's @SQ lines and the first record
    std::vector<std::pair<std::string, uint64_t>> sq;
    std::string first; uint64_t first_at = 0;
    {
        char* lp = nullptr; size_t lcap = 0; ssize_t n; uint64_t at = 0;
        while ((n = getline(&lp, &lcap, in)) > 0) {
            std::string l(lp, (size_t)n);
            while (!l.empty() && (l.back() == '\n' || l.back() == '\r')) l.pop_back();
            if (l.empty()) { at += (uint64_t)n; continue; }
            if (l[0] != '@') { first = l; first_at = at; break; }
            if (l.compare(0, 4, "@SQ\t") == 0) {
                std::string sn; uint64_t ln = 0; bool have_ln = false;
                for (size_t b = 4; b <= l.size();) {
                    size_t e = l.find('\t', b); if (e == std::string::npos) e = l.size();
                    if (l.compare(b, 3, "SN:") == 0) sn = l.substr(b + 3, e - b - 3);
                    if (l.compare(b, 3, "LN:") == 0) { ln = strtoull(l.c_str() + b + 3, nullptr, 10); have_ln = true; }
                    b = e + 1;
                }
                if (sn.empty() || !have_ln) { free(lp); return gsx_set_error(GSX_ERR_ARG, "header line at byte " + std::to_string(at) + " of " + sam_path + " is an @SQ line without SN or LN"); }
                sq.emplace_back(sn, ln);
            }
            at += (uint64_t)n;
        }
        free(lp);
        rewind(in);
    }
    gsx::HostIndex gi; std::vector<uint8_t> genome; std::string err;
    const auto t_fasta = std::chrono::steady_clock::now();
    if (!gsx::read_fasta(fasta_path, genome, gi, err)) return gsx_set_error(GSX_ERR_IO, err);
    const double s_fasta = std::chrono::duration<double>(std::chrono::steady_clock::now() - t_fasta).count();
    if (genome.size() != gi.genome_length) return gsx_set_error(GSX_ERR_ARG, std::string("FASTA ") + fasta_path + " has white space inside its sequence lines");
    if (!sq.empty()) {
        for (size_t i = 0; i < std::max(sq.size(), gi.chr_names.size()); i++) {
            if (i < sq.size() && i < gi.chr_names.size() && sq[i].first == gi.chr_names[i] && sq[i].second == gi.chr_lens[i]) continue;
            const std::string s = i < sq.size() ? "\"" + sq[i].first + "\" of " + std::to_string(sq[i].second) + " bases" : "nothing";
            const std::string fa = i < gi.chr_names.size() ? "\"" + gi.chr_names[i] + "\" of " + std::to_string(gi.chr_lens[i]) + " bases" : "nothing";
            return gsx_set_error(GSX_ERR_ARG, "@SQ line " + std::to_string(i + 1) + " of the database names " + s + ", FASTA record " + std::to_string(i + 1) +
                                                  " is " + fa + ": the database was not computed on this assembly");
        }
    }
    const int64_t delim = -((int64_t)gi.genome_length + 1);
    if (!first.empty()) {
        SamFields F; F.split(first.data(), first.data() + first.size());
        const std::string rec = "record " + quoted(F.f[0], F.n[0]) + " at byte " + std::to_string(first_at);
        if (!F.of) return gsx_set_error(GSX_ERR_ARG, rec + " has no of:H: tag: a database written with --mode succinct lists no off-targets; write it with --mode complete");
        if (F.of_len < 32 || F.of_len % 16) return gsx_set_error(GSX_ERR_ARG, rec + ": its of:H: value has " + std::to_string(F.of_len) + " hex digits, not a whole list of 16-digit values (truncated?)");
        const int64_t d = hex_le64(F.of + F.of_len - 16);
        if (d != delim)
            return gsx_set_error(GSX_ERR_ARG, rec + ": its of:H: list ends with " + std::to_string(d) + ", the delimiter of a genome of " + std::to_string(gi.genome_length) +
                                                  " bases is " + std::to_string(delim) + ": the database was not computed on this assembly");
    }
    std::map<std::string, uint64_t> chr_len;
    for (size_t i = 0; i < gi.chr_names.size(); i++) chr_len[gi.chr_names[i]] = gi.chr_lens[i];
    std::map<std::string, std::vector<std::pair<uint64_t, uint64_t>>> regions;
    if (regions_bed) {
        int code = GSX_OK;
        if (!read_bed(regions_bed, chr_len, regions, code, err)) return gsx_set_error(code, err);
    }
    const int have = gsx_device_count();
    if (have <= 0) return gsx_set_error(GSX_ERR_NO_DEVICE, "no CUDA device available (this library has no CPU path)");
    if (device >= have) return gsx_set_error(GSX_ERR_ARG, "device " + std::to_string(device) + " is out of range (" + std::to_string(have) + " device(s))");

    OutFile out;
    if (!out.open(out_path)) return gsx_set_error(GSX_ERR_IO, std::string("cannot write ") + out_path);
    {
        std::string h = csv_header(complete != 0);
        if (with_cfd) { h.pop_back(); h += ",cfd\n"; }
        if (!out.append(std::vector<std::string>(1, h))) { out.close_file(); return gsx_set_error(GSX_ERR_IO, std::string("cannot write ") + out_path); }
    }
    const char* eb = getenv("GSX_DECODE_BATCH_BYTES");                                      // (tests: batches of a few records)
    const size_t batch_bytes = eb && *eb && atoll(eb) > 0 ? (size_t)atoll(eb) : ((size_t)128 << 20);
    const bool timing = getenv("GSX_FILE_TIMING") != nullptr;
    auto now = [] { return std::chrono::steady_clock::now(); };
    auto since = [](std::chrono::steady_clock::time_point t) { return std::chrono::duration<double>(std::chrono::steady_clock::now() - t).count(); };
    const auto t_job = now();
    double s_upload = 0, s_read = 0, s_device = 0, ms_device = 0, s_format = 0, s_write = 0;
    size_t n_batches = 0, guides = 0, rows = 0, sam_bytes = 0;

    // reader (this thread) -> device (this thread) -> formatter -> writer; at most two batches wait between two stages
    std::mutex mu; std::condition_variable cv;
    std::deque<std::unique_ptr<DecodeBatch>> fqueue, spare; std::deque<std::vector<std::string>> wqueue;
    bool rdone = false, fdone = false, failed = false; int wrc = GSX_OK;
    std::atomic<bool> format_nomem{false};
    std::thread writer([&] {
        for (;;) {
            std::vector<std::string> parts;
            { std::unique_lock<std::mutex> lk(mu); cv.wait(lk, [&] { return !wqueue.empty() || fdone; }); if (wqueue.empty()) return; parts = std::move(wqueue.front()); }
            const auto tw = now();
            if (wrc == GSX_OK && !out.append(parts)) wrc = GSX_ERR_IO;
            s_write += since(tw);
            for (std::string& p : parts) string_pool().put(std::move(p));
            { std::lock_guard<std::mutex> lk(mu); wqueue.pop_front(); }
            cv.notify_all();
        }
    });
    std::thread formatter([&] {
        const unsigned hw = std::max(1u, std::thread::hardware_concurrency());
        for (;;) {
            std::unique_ptr<DecodeBatch> b; bool skip;
            {
                std::unique_lock<std::mutex> lk(mu);
                cv.wait(lk, [&] { return !fqueue.empty() || rdone; });
                if (fqueue.empty()) break;
                b = std::move(fqueue.front()); fqueue.pop_front(); skip = failed;
            }
            cv.notify_all();
            if (skip) { std::lock_guard<std::mutex> lk(mu); spare.push_back(std::move(b)); continue; }
            const auto tf = now();
            // slices of about equal numbers of rows, cut at records
            const size_t nr = b->recs.size(), total = b->rows.n_rows;
            const unsigned nt = (unsigned)std::max<size_t>(1, std::min<size_t>({(size_t)hw, nr, total / 32768 + 1}));
            std::vector<size_t> cut(nt + 1, nr); cut[0] = 0;
            for (unsigned t = 1; t < nt; t++) cut[t] = (size_t)(std::lower_bound(b->rows.rec_row, b->rows.rec_row + nr, (uint32_t)(total * t / nt)) - b->rows.rec_row);
            std::vector<std::string> parts(nt);
            auto work = [&](unsigned t) {
                parts[t] = string_pool().get();
                const size_t a = std::min(cut[t], nr), e = std::max(a, std::min(cut[t + 1], nr));
                parts[t].reserve((size_t)(b->rows.rec_row[e] - b->rows.rec_row[a]) * 120);
                try { format_decoded(*b, a, e, gi.chr_names, complete != 0, with_cfd != 0, parts[t]); }
                catch (const std::bad_alloc&) { format_nomem = true; parts[t].clear(); }
            };
            if (nt == 1) work(0);
            else { std::vector<std::thread> th; for (unsigned t = 0; t < nt; t++) th.emplace_back(work, t); for (auto& x : th) x.join(); }
            s_format += since(tf);
            std::unique_lock<std::mutex> lk(mu);
            spare.push_back(std::move(b));
            cv.wait(lk, [&] { return wqueue.size() < 2; });
            wqueue.push_back(std::move(parts));
            lk.unlock(); cv.notify_all();
        }
        { std::lock_guard<std::mutex> lk(mu); fdone = true; }
        cv.notify_all();
    });

    int rc = GSX_OK; std::string rc_msg;
    try {
        const auto tu = now();
        std::vector<gsx::Chrom> chroms; uint64_t start = 0;
        for (uint64_t l : gi.chr_lens) { chroms.push_back({start, l}); start += l; }
        gsx::DecodeDevice dev(device, genome.data(), gi.genome_length, chroms, pams);
        s_upload = since(tu);
        SamReader reader(in);
        DecodeSplitter splitter{pam_length, regions_bed ? &regions : nullptr};
        for (;;) {
            std::unique_ptr<DecodeBatch> b;
            {
                std::unique_lock<std::mutex> lk(mu);
                cv.wait(lk, [&] { return fqueue.size() < 2; });
                if (!spare.empty()) { b = std::move(spare.front()); spare.pop_front(); }
            }
            if (!b) b.reset(new DecodeBatch());
            const auto tr = now();
            if (!reader.next(batch_bytes, *b)) break;
            splitter.split(*b);
            s_read += since(tr);
            sam_bytes += b->len;
            if (b->recs.empty()) { std::lock_guard<std::mutex> lk(mu); spare.push_back(std::move(b)); continue; }      // (keeps its pinned text)
            const auto td = now();
            dev.run({b->text, b->len, b->rec_hex.data(), b->rec_entry.data(), b->guides.data(), (uint32_t)b->recs.size()}, b->rows);
            s_device += since(td); ms_device += b->rows.ms; n_batches++;
            if (b->rows.err_code) {
                const gsx::DecodeRows& R = b->rows;
                const size_t r = (size_t)(std::upper_bound(b->rec_entry.begin(), b->rec_entry.end(), R.err_entry) - b->rec_entry.begin()) - 1;
                const DecodeRec& c = b->recs[r];
                const std::string rec = "record " + quoted(c.id, c.id_len) + " at byte " + std::to_string(c.at);
                const uint32_t t = R.err_entry - b->rec_entry[r];
                std::string what;
                if (R.err_code == gsx::kDecodeBadHex) what = "value " + std::to_string(t) + " of its of:H: list is not 16 hex digits";
                else if (R.err_code == gsx::kDecodeBadGroup) what = "its of:H: list is not a run of groups [positions] d " + std::to_string(delim) + " for d = 0, 1, ... (at value " + std::to_string(t) + ")";
                else {
                    const int64_t abs = R.err_value; const gsx::DecodeGuide& g = b->guides[r];
                    uint32_t pos1 = 0; uint8_t sc = '+';
                    const int chr = gsx::resolve_abs(chroms.data(), (uint32_t)chroms.size(), abs, g.qlen, g.plen, &pos1, &sc);
                    const std::string site = "off-target " + std::to_string(abs) + (chr >= 0 ? " (" + gi.chr_names[chr] + ":" + std::to_string(pos1) + ":" + (char)sc + ")" : "");
                    if (R.err_code == gsx::kDecodeOutside) what = site + " does not lie inside one chromosome of the genome";
                    else if (R.err_code == gsx::kDecodeDistance)
                        what = site + " has " + std::to_string(R.err_found) + " mismatches to the guide but is listed at distance " + std::to_string(R.err_listed) + ": the database was written with bulges, or "
                               "on another genome";
                    else what = site + " carries neither the guide's PAM column nor an alternative PAM: the database was written with bulges, with other PAMs (-a), or "
                           "on another genome";
                }
                throw decode_error(rec + ": " + what);
            }
            guides += b->recs.size(); rows += b->rows.n_rows;
            {
                std::lock_guard<std::mutex> lk(mu);
                fqueue.push_back(std::move(b));
            }
            cv.notify_all();
        }
    } catch (const gsx::SiteError& f) { rc = f.code; rc_msg = f.msg; }
    catch (const std::bad_alloc&) { rc = GSX_ERR_NOMEM; rc_msg = "out of host memory"; }
    catch (const std::exception& x) { rc = GSX_ERR_INTERNAL; rc_msg = std::string("decode: ") + x.what(); }
    { std::lock_guard<std::mutex> lk(mu); rdone = true; failed = rc != GSX_OK; }
    cv.notify_all();
    formatter.join(); writer.join();
    if (timing)
        fprintf(stderr, "gsx decode: %.3f s wall, %zu SAM bytes, %zu guides decoded, %zu rows, %zu batch(es); FASTA read %.3f s (before the wall); genome upload %.3f s; read/split %.3f s; "
                "device %.3f s (events %.3f ms, %.3f ms per batch); format %.3f s; write %.3f s\n",
                since(t_job), sam_bytes, guides, rows, n_batches, s_fasta, s_upload, s_read, s_device, ms_device, n_batches ? ms_device / n_batches : 0.0, s_format, s_write);
    if (!out.close_file() && wrc == GSX_OK) wrc = GSX_ERR_IO;
    if (rc) return gsx_set_error(rc, rc_msg);
    if (format_nomem) return gsx_set_error(GSX_ERR_NOMEM, "out of host memory formatting the rows");
    if (wrc) return gsx_set_error(wrc, std::string("cannot write ") + out_path);
    if (n_guides) *n_guides = guides;
    if (n_rows) *n_rows = rows;
    return GSX_OK;
}
