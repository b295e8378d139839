// gsx_index.cpp -- host side of the GPU index: reading the reference's index files and laying them out for HBM.
//
// Input format = what the reference's `guidescan index` stores with sdsl::store_to_file
// (reference src/guidescan.cxx:167-175): csa_wt<wt_huff<>,64,8192>::serialize (sdsl csa_wt.hpp:372-382) =
// wt_pc::serialize (wt_pc.hpp:656-671) + SA samples + ISA samples + byte_alphabet.  Field layout verified
// against real files: SURVEY.md App. B.
#include "gsx_host.h"
#include "gsx_core.h"
#include <algorithm>
#include <cctype>
#include <cstdio>
#include <cstring>
#include <fstream>
#include <functional>
#include <sstream>
#include <thread>

namespace gsx {

static inline int sym_code(uint8_t c) { return c == 'A' ? 0 : c == 'C' ? 1 : c == 'G' ? 2 : c == 'T' ? 3 : -1; }

StrandBuilder::StrandBuilder(HostStrand* o, uint64_t n_rows) : out(o), n(n_rows) {
    memset(run, 0, sizeof run);
    memset(&cur, 0, sizeof cur);
    out->n = n;
    out->blocks.clear(); out->blocks.reserve(n / 64 + 1);
    out->exc_rows.clear(); out->exc_lf.clear(); out->n_rows.clear(); out->exc_sym.clear();
}

void StrandBuilder::push(uint8_t sym) {
    uint32_t r = (uint32_t)(row & 63);
    if (r == 0) {
        memset(&cur, 0, sizeof cur);
        cur.cnt[0] = (uint32_t)run['A']; cur.cnt[1] = (uint32_t)run['C']; cur.cnt[2] = (uint32_t)run['G']; cur.cnt[3] = (uint32_t)run['T'];
    }
    int code = sym_code(sym);
    if (code < 0) {
        out->exc_rows.push_back((uint32_t)row);
        out->exc_sym.push_back(sym); exc_rank.push_back(run[sym]);
        if (sym == 'N') out->n_rows.push_back((uint32_t)row);
        code = 0;
    }
    cur.hi |= (uint64_t)(code >> 1) << r;
    cur.lo |= (uint64_t)(code & 1) << r;
    run[sym]++;
    row++;
    if ((row & 63) == 0) out->blocks.push_back(cur);
}

void StrandBuilder::finish() {
    if (row & 63) out->blocks.push_back(cur);
    else {      // n is a multiple of 64: one more checkpoint-only block for lookups at i == n
        memset(&cur, 0, sizeof cur);
        cur.cnt[0] = (uint32_t)run['A']; cur.cnt[1] = (uint32_t)run['C']; cur.cnt[2] = (uint32_t)run['G']; cur.cnt[3] = (uint32_t)run['T'];
        out->blocks.push_back(cur);
    }
    uint64_t Cb[257]; uint64_t acc = 0;
    for (int c = 0; c < 256; c++) { Cb[c] = acc; acc += run[c]; }
    out->C[0] = (uint32_t)Cb['A']; out->C[1] = (uint32_t)Cb['C']; out->C[2] = (uint32_t)Cb['G']; out->C[3] = (uint32_t)Cb['T'];
    out->C[4] = (uint32_t)Cb['N'];
    out->exc_lf.resize(out->exc_rows.size());
    for (size_t i = 0; i < out->exc_rows.size(); i++) out->exc_lf[i] = (uint32_t)(Cb[out->exc_sym[i]] + exc_rank[i]);
}

// ---- sdsl file reader ------------------------------------------------------------------------------------
namespace {
struct Reader {
    FILE* f = nullptr; std::string err; uint64_t file_bytes = 0;
    bool u64(uint64_t& v) { return fread(&v, 8, 1, f) == 1; }
    bool u8(uint8_t& v) { return fread(&v, 1, 1, f) == 1; }
    // int_vector<w>: u64 size in bits, [u8 width if w == 0], ceil(bits/64) words  (sdsl int_vector.hpp:593-609,1563-1595)
    bool int_vector(int w, uint64_t& bits, uint8_t& width, std::vector<uint64_t>* data) {
        if (!u64(bits)) return false;
        width = (uint8_t)w;
        if (w == 0 && !u8(width)) return false;
        uint64_t words = (bits + 63) / 64;
        // (a vector longer than what is left of the file is a corrupt or truncated file, not an allocation request)
        const off_t at = ftello(f);
        if (at < 0 || (uint64_t)at > file_bytes || words > (file_bytes - (uint64_t)at) / 8) return false;
        if (data) { data->resize(words); return words == 0 || fread(data->data(), 8, words, f) == words; }
        return fseeko(f, (off_t)(words * 8), SEEK_CUR) == 0;
    }
    // select_support_mcl (select_support_mcl.hpp:425-493): skipped, the hot path never selects
    bool skip_select() {
        uint64_t arg_cnt; if (!u64(arg_cnt)) return false;
        if (!arg_cnt) return true;
        uint64_t bits; uint8_t w;
        if (!int_vector(0, bits, w, nullptr)) return false;     // superblock
        if (!int_vector(1, bits, w, nullptr)) return false;     // mini_or_long
        uint64_t sb = (arg_cnt + 4095) >> 12;
        for (uint64_t i = 0; i < sb; i++) if (!int_vector(0, bits, w, nullptr)) return false;
        return true;
    }
};
struct WtNode { uint64_t bv_pos, bv_pos_rank; uint16_t parent, child[2]; };
}  // namespace

bool load_sdsl_strand(const std::string& path, HostStrand& out, std::string& err) {
    Reader r; r.f = fopen(path.c_str(), "rb");
    if (!r.f) { err = "cannot open " + path; return false; }
    if (fseeko(r.f, 0, SEEK_END) == 0) { const off_t e = ftello(r.f); r.file_bytes = e > 0 ? (uint64_t)e : 0; }
    fseeko(r.f, 0, SEEK_SET);
    auto fail = [&](const char* what) { err = std::string("malformed index file ") + path + " (" + what + ")"; fclose(r.f); return false; };
    uint64_t size, sigma, bits; uint8_t w;
    if (!r.u64(size) || !r.u64(sigma)) return fail("header");
    if (size == 0 || size > 0xFFFFFFFFull) return fail("size out of range for 32-bit rows");
    std::vector<uint64_t> bv;
    if (!r.int_vector(1, bits, w, &bv)) return fail("wavelet tree bit vector");
    uint64_t skipped;
    if (!r.int_vector(64, skipped, w, nullptr)) return fail("rank support");
    if (!r.skip_select() || !r.skip_select()) return fail("select support");
    uint64_t n_nodes; if (!r.u64(n_nodes) || n_nodes == 0 || n_nodes > 1024) return fail("tree size");
    std::vector<WtNode> nodes(n_nodes);
    for (auto& nd : nodes) {                                   // wt_helper.hpp:109-126
        if (fread(&nd.bv_pos, 8, 1, r.f) != 1 || fread(&nd.bv_pos_rank, 8, 1, r.f) != 1 || fread(&nd.parent, 2, 1, r.f) != 1 ||
            fread(nd.child, 2, 2, r.f) != 2) return fail("tree nodes");
    }
    if (fseeko(r.f, 256 * 2 + 256 * 8, SEEK_CUR) != 0) return fail("c_to_leaf/path");
    std::vector<uint64_t> sa_words; uint64_t sa_bits; uint8_t sa_w;
    if (!r.int_vector(0, sa_bits, sa_w, &sa_words)) return fail("sa samples");
    fclose(r.f);
    if (sa_w == 0 || sa_w > 32) { err = "SA sample width unsupported in " + path; return false; }

    for (size_t v = 0; v < n_nodes; v++) {                       // breadth-first layout: children come after their parent
        const WtNode& nd = nodes[v];
        const bool leaf = nd.child[0] == 0xFFFF;
        if (leaf ? nd.child[1] != 0xFFFF : (nd.child[0] <= v || nd.child[1] <= v || nd.child[0] >= n_nodes || nd.child[1] >= n_nodes || nd.bv_pos > bits))
            { err = "malformed index file " + path + " (tree)"; return false; }
    }
    // BWT recovery: walk the tree for every row with one read cursor per inner node (children receive their elements in order,
    // so no rank is needed along the way).  Row ranges are independent once the cursors at a range start are known: the rows
    // before r that pass a node are counted down from the root with ranks over the bit vector (ones before each 512-bit block
    // are summed here; the file's own rank directory is not trusted with it).  One host thread per range.
    const uint64_t* bvp = bv.data();
    std::vector<uint64_t> ones512(bv.size() / 8 + 2, 0);
    for (size_t w = 0; w < bv.size(); w++) { if ((w & 7) == 0) ones512[w / 8 + 1] = ones512[w / 8]; ones512[w / 8 + 1] += (uint64_t)__builtin_popcountll(bvp[w]); }
    auto rank1 = [&](uint64_t pos) {                           // ones in bits [0, pos)
        uint64_t r = ones512[pos >> 9];
        for (uint64_t w = (pos >> 9) * 8; w < (pos >> 6); w++) r += (uint64_t)__builtin_popcountll(bvp[w]);
        if (pos & 63) r += (uint64_t)__builtin_popcountll(bvp[pos >> 6] & (~0ull >> (64 - (pos & 63))));
        return r;
    };
    const uint64_t n_blocks = size / 64 + 1;
    out.n = size; out.blocks.assign(n_blocks, OccBlock{});
    out.exc_rows.clear(); out.exc_lf.clear(); out.n_rows.clear(); out.exc_sym.clear();
    const char* knob = getenv("GSX_LOAD_THREADS");               // tests: several ranges on a small index
    const unsigned T = knob && atoi(knob) > 0 ? (unsigned)atoi(knob)
                     : (unsigned)std::max<uint64_t>(1, std::min<uint64_t>(std::max(1u, std::thread::hardware_concurrency()), size / (1u << 20) + 1));
    struct Range { uint64_t run[256]; std::vector<uint32_t> exc_rows, n_rows; std::vector<uint8_t> exc_sym; std::vector<uint64_t> exc_rank; bool ok = true; };
    std::vector<Range> ranges(T);
    auto decode = [&](unsigned t) {
        Range& R = ranges[t];
        const uint64_t r0 = (size / 64) * t / T * 64, r1 = t + 1 == T ? size : (size / 64) * (t + 1) / T * 64;
        std::vector<uint64_t> passing(n_nodes, 0), cursor(n_nodes, 0);
        memset(R.run, 0, sizeof R.run);
        passing[0] = r0;
        for (size_t v = 0; v < n_nodes; v++) {
            const WtNode& nd = nodes[v];
            if (nd.child[0] == 0xFFFF) { R.run[(uint8_t)nd.bv_pos_rank] = passing[v]; continue; }
            if (nd.bv_pos + passing[v] > bits) { R.ok = false; return; }
            const uint64_t ones = rank1(nd.bv_pos + passing[v]) - rank1(nd.bv_pos);
            passing[nd.child[1]] = ones; passing[nd.child[0]] = passing[v] - ones;
            cursor[v] = nd.bv_pos + passing[v];
        }
        OccBlock cur{};
        for (uint64_t row = r0; row < r1; row++) {
            const uint32_t r = (uint32_t)(row & 63);
            if (r == 0) {
                cur = OccBlock{};
                cur.cnt[0] = (uint32_t)R.run['A']; cur.cnt[1] = (uint32_t)R.run['C']; cur.cnt[2] = (uint32_t)R.run['G']; cur.cnt[3] = (uint32_t)R.run['T'];
            }
            uint32_t v = 0;
            while (nodes[v].child[0] != 0xFFFF) {
                const uint64_t p = cursor[v]++;
                if (p >= bits) { R.ok = false; return; }
                v = nodes[v].child[(bvp[p >> 6] >> (p & 63)) & 1];
            }
            const uint8_t sym = (uint8_t)nodes[v].bv_pos_rank;
            int code = sym_code(sym);
            if (code < 0) {
                R.exc_rows.push_back((uint32_t)row); R.exc_sym.push_back(sym); R.exc_rank.push_back(R.run[sym]);
                if (sym == 'N') R.n_rows.push_back((uint32_t)row);
                code = 0;
            }
            cur.hi |= (uint64_t)(code >> 1) << r; cur.lo |= (uint64_t)(code & 1) << r;
            R.run[sym]++;
            if (r == 63 || row + 1 == size) out.blocks[row >> 6] = cur;
        }
    };
    {
        std::vector<std::thread> pool;
        for (unsigned t = 1; t < T; t++) pool.emplace_back(decode, t);
        decode(0);
        for (auto& th : pool) th.join();
    }
    for (const Range& R : ranges) if (!R.ok) { err = "malformed index file " + path + " (wavelet tree bits)"; return false; }
    const uint64_t* total = ranges[T - 1].run;                  // a range starts from the counts before it, so the last one ends on the totals
    if (size % 64 == 0) {                                      // one more checkpoint-only block for lookups at i == n
        OccBlock& last = out.blocks[n_blocks - 1];
        last.cnt[0] = (uint32_t)total['A']; last.cnt[1] = (uint32_t)total['C']; last.cnt[2] = (uint32_t)total['G']; last.cnt[3] = (uint32_t)total['T'];
    }
    uint64_t Cb[257], acc = 0;
    for (int c = 0; c < 256; c++) { Cb[c] = acc; acc += total[c]; }
    out.C[0] = (uint32_t)Cb['A']; out.C[1] = (uint32_t)Cb['C']; out.C[2] = (uint32_t)Cb['G']; out.C[3] = (uint32_t)Cb['T']; out.C[4] = (uint32_t)Cb['N'];
    for (const Range& R : ranges) {
        out.exc_rows.insert(out.exc_rows.end(), R.exc_rows.begin(), R.exc_rows.end());
        out.n_rows.insert(out.n_rows.end(), R.n_rows.begin(), R.n_rows.end());
        out.exc_sym.insert(out.exc_sym.end(), R.exc_sym.begin(), R.exc_sym.end());
        for (size_t i = 0; i < R.exc_rows.size(); i++) out.exc_lf.push_back((uint32_t)(Cb[R.exc_sym[i]] + R.exc_rank[i]));
    }
    // SA samples: entry k = SA[64 k], bit-packed little-endian (csa_sampling_strategy.hpp:85-111)
    uint64_t n_samples = sa_bits / sa_w;
    if (n_samples < (size + 63) / 64) { err = "too few SA samples in " + path; return false; }
    out.sa_shift = 6;
    out.sa_samples.resize(n_samples);
    const uint64_t mask = sa_w == 64 ? ~0ull : ((1ull << sa_w) - 1);
    for (uint64_t k = 0; k < n_samples; k++) {
        uint64_t bitpos = k * sa_w, wd = bitpos >> 6, sh = bitpos & 63;
        uint64_t v = sa_words[wd] >> sh;
        if (sh + sa_w > 64) v |= sa_words[wd + 1] << (64 - sh);
        out.sa_samples[k] = (uint32_t)(v & mask);
    }
    return true;
}

DevStrand host_view(const HostStrand& h) {
    DevStrand d{};
    d.blocks = h.blocks.data(); d.sa_samples = h.sa_samples.data(); d.exc_rows = h.exc_rows.data(); d.exc_lf = h.exc_lf.data();
    d.n_rows = h.n_rows.data(); d.n = (uint32_t)h.n; d.n_exc = (uint32_t)h.exc_rows.size(); d.n_nrows = (uint32_t)h.n_rows.size();
    d.sa_shift = h.sa_shift; for (int c = 0; c < 5; c++) d.C[c] = h.C[c];
    d.exc_lo = h.exc_rows.empty() ? 0xFFFFFFFFu : h.exc_rows.front(); d.exc_hi = h.exc_rows.empty() ? 0u : h.exc_rows.back();
    d.blk_shift = 5;
    return d;
}

bool load_genome_structure(const std::string& path, HostIndex& ix, std::string& err) {
    std::ifstream fs(path);
    if (!fs) { err = "No genome structure file " + path + " located."; return false; }
    ix.chr_names.clear(); ix.chr_lens.clear(); ix.genome_length = 0;
    while (fs) {
        std::string name, len;
        std::getline(fs, name); std::getline(fs, len);
        if (name.empty() || len.empty()) break;
        char* endp = nullptr; const long long v = strtoll(len.c_str(), &endp, 10);
        if (endp == len.c_str() || v < 0) { err = "malformed genome structure file " + path + " (length \"" + len + "\")"; return false; }
        ix.chr_names.push_back(name); ix.chr_lens.push_back((uint64_t)v);
        ix.genome_length += ix.chr_lens.back();
    }
    return true;
}

bool read_fasta(const std::string& path, std::vector<uint8_t>& seq, HostIndex& ix, std::string& err) {
    std::ifstream is(path);
    if (!is) { err = "ERROR: FASTA file \"" + path + "\" does not exist."; return false; }
    ix.chr_names.clear(); ix.chr_lens.clear(); seq.clear();
    std::string line;
    while (std::getline(is, line)) {
        if (!line.empty() && line[0] == '>') {
            std::string name = line.substr(1);
            size_t b = 0; while (b < name.size() && isspace((unsigned char)name[b])) b++;
            size_t e = name.size(); while (e > b && isspace((unsigned char)name[e - 1])) e--;
            name = name.substr(b, e - b);
            size_t sp = name.find(' ');
            if (sp != std::string::npos) name = name.substr(0, sp);
            ix.chr_names.push_back(name); ix.chr_lens.push_back(0);
            continue;
        }
        if (!ix.chr_lens.empty()) ix.chr_lens.back() += line.size();        // raw line length, as the reference counts it
        size_t b = 0; while (b < line.size() && isspace((unsigned char)line[b])) b++;
        size_t e = line.size(); while (e > b && isspace((unsigned char)line[e - 1])) e--;
        for (size_t i = b; i < e; i++) seq.push_back((uint8_t)toupper((unsigned char)line[i]));
    }
    ix.genome_length = 0;
    for (auto l : ix.chr_lens) ix.genome_length += l;
    return true;
}

std::vector<uint64_t> ftab_combos(uint32_t n_pos, uint32_t M) {
    std::vector<uint64_t> out;
    if (n_pos > 16) n_pos = 16;
    std::vector<uint32_t> pos;
    // subsets of positions in increasing order, each with 3^j substitution choices
    struct Rec { static void go(uint32_t start, uint32_t n_pos, uint32_t M, std::vector<uint32_t>& pos, std::vector<uint64_t>& out) {
        const uint32_t j = (uint32_t)pos.size();
        uint32_t n_sub = 1; for (uint32_t t = 0; t < j; t++) n_sub *= 3;
        for (uint32_t code = 0; code < n_sub; code++) {
            uint64_t w = j; uint32_t c = code;
            for (uint32_t t = 0; t < j; t++) { uint32_t sub = 1 + c % 3; c /= 3; w |= (uint64_t)(pos[t] | (sub << 4)) << (3 + 6 * t); }
            out.push_back(w);
        }
        if (j == M) return;
        for (uint32_t p = start; p < n_pos; p++) { pos.push_back(p); go(p + 1, n_pos, M, pos, out); pos.pop_back(); }
    } };
    Rec::go(0, n_pos, M, pos, out);
    // by number of substitutions: the 32 combos a warp handles in one table step then share their remaining budget, and
    // a step whose combos have none left only looks at the exact ending
    std::stable_sort(out.begin(), out.end(), [](uint64_t x, uint64_t y) { return (x & 7u) < (y & 7u); });
    return out;
}

std::vector<uint32_t> build_exc_map(const HostStrand& h) {
    std::vector<uint32_t> map((h.blocks.size() + 31) / 32 + 1, 0u);
    for (uint32_t row : h.exc_rows) { const uint32_t b = row >> 6; map[b >> 5] |= 1u << (b & 31u); }
    return map;
}

// every op list (gsx_core.h variant_op) with at most R RNA bulges and D DNA bulges for a guide of qlen characters, in the
// canonical order (by level; the DNA bulges of a level, in sequence, before its skip); the empty list comes last of its
// branch like everything else, order is irrelevant.  R + D <= 4.
std::vector<uint32_t> bulge_variants(uint32_t qlen, uint32_t R, uint32_t D) {
    std::vector<uint32_t> out;
    struct Rec { static void go(uint32_t lvl, uint32_t qlen, uint32_t r, uint32_t d, uint32_t desc, uint32_t nops, std::vector<uint32_t>& out) {
        if (lvl > qlen) { out.push_back(desc); return; }
        if (d && nops < 4) for (uint32_t sym = 0; sym < 4; sym++) go(lvl, qlen, r, d - 1, desc | (variant_op(lvl, 1, sym) << (8 * nops)), nops + 1, out);
        if (lvl < qlen && r && nops < 4) go(lvl + 1, qlen, r - 1, d, desc | (variant_op(lvl, 0, 0) << (8 * nops)), nops + 1, out);
        go(lvl + 1, qlen, r, d, desc, nops, out);
    } };
    if (R + D <= 4 && qlen >= 1 && qlen < 32) Rec::go(1, qlen, R, D, 0, 0, out);
    return out;
}
uint64_t bulge_variant_count(uint32_t qlen, uint32_t R, uint32_t D) {
    // skips: subsets of positions 1 .. qlen-1 of size <= R; inserts: sequences of <= D (slot, symbol) with slots non-decreasing
    // = multisets of slots (qlen of them) times 4^k
    auto choose = [](uint64_t n, uint64_t k) { if (k > n) return (uint64_t)0; uint64_t v = 1; for (uint64_t i = 0; i < k; i++) v = v * (n - i) / (i + 1); return v; };
    uint64_t skips = 0, ins = 0;
    for (uint32_t k = 0; k <= R; k++) skips += choose(qlen ? qlen - 1 : 0, k);
    for (uint32_t k = 0; k <= D; k++) ins += choose(qlen + k - 1, k) << (2 * k);
    return skips * ins;
}

void sweep_make_plan(uint32_t L, uint32_t sb, uint32_t M, SweepPlan& plan, std::vector<uint32_t>& xtab) {
    memset(&plan, 0, sizeof plan);
    plan.L = L; plan.sb = sb; plan.M = M;
    const uint32_t n_pos = L - sb;                          // characters 0 .. n_pos-1 lie outside the slice
    // every xor value with at most M substituted characters, grouped by their number
    std::vector<std::vector<uint32_t>> by_count(M + 1);
    std::vector<uint32_t> pos;
    for (uint32_t j = 0; j <= M && j <= n_pos; j++) {
        pos.assign(j, 0); for (uint32_t t = 0; t < j; t++) pos[t] = t;
        for (;;) {
            uint32_t n_sub = 1; for (uint32_t t = 0; t < j; t++) n_sub *= 3;
            for (uint32_t code = 0; code < n_sub; code++) {
                uint32_t m = 0, c = code;
                for (uint32_t t = 0; t < j; t++) { m |= (1u + c % 3u) << (2u * pos[t]); c /= 3u; }
                by_count[j].push_back(m | (j << 28));
            }
            int t = (int)j - 1;
            while (t >= 0 && pos[t] == n_pos - j + t) t--;
            if (t < 0) break;
            pos[t]++; for (uint32_t u = t + 1; u < j; u++) pos[u] = pos[u - 1] + 1;
        }
    }
    xtab.clear();
    for (uint32_t B = 0; B <= M; B++) {
        plan.xoff[1][B] = (uint32_t)xtab.size(); xtab.insert(xtab.end(), by_count[B].begin(), by_count[B].end());
        plan.xcnt[1][B] = (uint32_t)xtab.size() - plan.xoff[1][B];
    }
    for (uint32_t B = 0; B <= M; B++) {
        plan.xoff[0][B] = (uint32_t)xtab.size();
        for (uint32_t j = 0; j < B; j++) xtab.insert(xtab.end(), by_count[j].begin(), by_count[j].end());
        plan.xcnt[0][B] = (uint32_t)xtab.size() - plan.xoff[0][B];
    }
    for (uint32_t z = 0; z < 2; z++)
        for (uint32_t B = 0; B <= M; B++)
            for (uint32_t t = 0; t < plan.xcnt[z][B]; t++) if ((xtab[plan.xoff[z][B] + t] & 15u) == 0u) plan.xlines[z][B]++;
}

void split_make_plan(uint32_t L, uint32_t sb, uint32_t M, uint32_t qlen, uint32_t plen, uint32_t pampack, uint32_t half, SplitPlan& plan,
                     std::vector<uint32_t>& xtab) {
    memset(&plan, 0, sizeof plan);
    xtab.clear();
    const uint32_t n_pos = L - sb, top_mask = (1u << (2u * sb)) - 1u;
    for (uint32_t f = 0; f < 2; f++) {
        uint32_t cost, cap, exact, freec;
        split_classes(f, L, qlen, plen, pampack, half, cost, cap, exact, freec);
        plan.cost_top[f] = (cost >> (2u * n_pos)) & top_mask;
        plan.cap_top[f] = (cap >> (2u * n_pos)) & top_mask;
        plan.exact_top[f] = (exact >> (2u * n_pos)) & top_mask;
        for (uint32_t c = 0; c < 2; c++)
            for (uint32_t B = 0; B <= M; B++) {
                plan.xoff[f][c][B] = (uint32_t)xtab.size();
                // every xor value over characters 0 .. n_pos-1 with at most B substitutions that cost budget, at most c of them capped
                std::function<void(uint32_t, uint32_t, uint32_t, uint32_t)> walk = [&](uint32_t k, uint32_t x, uint32_t used, uint32_t capped) {
                    if (k == n_pos) { xtab.push_back(x | (used << 28)); return; }
                    const uint32_t bit = 1u << (2u * k);
                    if (exact & bit) { walk(k + 1, x, used, capped); return; }
                    if (freec & bit) { for (uint32_t s = 0; s < 4; s++) walk(k + 1, x | (s << (2u * k)), used, capped); return; }
                    walk(k + 1, x, used, capped);
                    const uint32_t cp = (cap & bit) ? 1u : 0u;
                    if (used < B && capped + cp <= c)
                        for (uint32_t s = 1; s < 4; s++) walk(k + 1, x | (s << (2u * k)), used + 1u, capped + cp);
                };
                walk(0, 0, 0, 0);
                plan.xcnt[f][c][B] = (uint32_t)xtab.size() - plan.xoff[f][c][B];
            }
    }
}

// ---- native cache format (<prefix>.gsx): a flat dump of the HBM layout ----------------------------------------
namespace {
const char kMagic[8] = {'G', 'S', 'X', 'I', 'D', 'X', '0', '2'};
template <class T> bool wr(FILE* f, const std::vector<T>& v) { uint64_t n = v.size(); return fwrite(&n, 8, 1, f) == 1 && (n == 0 || fwrite(v.data(), sizeof(T), n, f) == n); }
// (a section longer than what is left of the file is a corrupt header, not an allocation request)
template <class T> bool rd(FILE* f, std::vector<T>& v) {
    uint64_t n; if (fread(&n, 8, 1, f) != 1) return false;
    const off_t at = ftello(f); if (at < 0 || fseeko(f, 0, SEEK_END) != 0) return false;
    const off_t end = ftello(f); if (fseeko(f, at, SEEK_SET) != 0) return false;
    if (n > (uint64_t)(end - at) / sizeof(T)) return false;
    v.resize(n); return n == 0 || fread(v.data(), sizeof(T), n, f) == n;
}
}  // namespace

bool save_gsx(const std::string& prefix, const HostIndex& ix, std::string& err) {
    FILE* f = fopen((prefix + ".gsx").c_str(), "wb");
    if (!f) { err = "cannot write " + prefix + ".gsx"; return false; }
    bool ok = fwrite(kMagic, 8, 1, f) == 1;
    for (int s = 0; s < 2 && ok; s++) {
        const HostStrand& h = ix.st[s];
        ok = fwrite(&h.n, 8, 1, f) == 1 && fwrite(&h.sa_shift, 4, 1, f) == 1 && fwrite(h.C, 4, 5, f) == 5 && wr(f, h.blocks) &&
             wr(f, h.sa_samples) && wr(f, h.exc_rows) && wr(f, h.exc_lf) && wr(f, h.n_rows) && wr(f, h.exc_sym);
    }
    fclose(f);
    if (!ok) { err = "short write to " + prefix + ".gsx"; return false; }
    std::ofstream gs(prefix + ".gs");                                     // seq_io.cxx:112-122
    for (size_t i = 0; i < ix.chr_names.size(); i++) gs << ix.chr_names[i] << "\n" << ix.chr_lens[i] << "\n";
    return true;
}

bool load_gsx(const std::string& prefix, HostIndex& ix, std::string& err) {
    FILE* f = fopen((prefix + ".gsx").c_str(), "rb");
    if (!f) { err = "cannot open " + prefix + ".gsx"; return false; }
    char magic[8]; bool ok = fread(magic, 8, 1, f) == 1 && memcmp(magic, kMagic, 8) == 0;
    for (int s = 0; s < 2 && ok; s++) {
        HostStrand& h = ix.st[s];
        ok = fread(&h.n, 8, 1, f) == 1 && fread(&h.sa_shift, 4, 1, f) == 1 && fread(h.C, 4, 5, f) == 5 && rd(f, h.blocks) &&
             rd(f, h.sa_samples) && rd(f, h.exc_rows) && rd(f, h.exc_lf) && rd(f, h.n_rows) && rd(f, h.exc_sym);
    }
    fclose(f);
    // section sizes must agree with the row count: the kernels index these arrays by row without further checks
    for (int s = 0; s < 2 && ok; s++) {
        const HostStrand& h = ix.st[s];
        ok = h.n >= 1 && h.n <= 0xFFFFFFFFull && h.sa_shift <= 12 && h.blocks.size() == h.n / 64 + 1 &&
             h.sa_samples.size() == ((h.n - 1) >> h.sa_shift) + 1 && h.exc_lf.size() == h.exc_rows.size() && h.exc_sym.size() == h.exc_rows.size() &&
             h.n_rows.size() <= h.exc_rows.size() && !h.exc_rows.empty();
        for (size_t i = 0; ok && i < h.exc_rows.size(); i++) ok = h.exc_rows[i] < h.n && h.exc_lf[i] < h.n && (i == 0 || h.exc_rows[i] > h.exc_rows[i - 1]);
        for (size_t i = 0; ok && i < h.n_rows.size(); i++) ok = h.n_rows[i] < h.n;
    }
    if (ok) ok = ix.st[0].n == ix.st[1].n;
    if (!ok) { err = "malformed " + prefix + ".gsx"; return false; }
    if (!load_genome_structure(prefix + ".gs", ix, err)) return false;
    if (ix.genome_length + 1 != ix.st[0].n) { err = prefix + ".gs does not describe the genome of " + prefix + ".gsx"; return false; }
    return true;
}

}  // namespace gsx
