// gsx_kmers.cu -- genome-wide guide generation on the GPU (SURVEY.md section 8(f)-2): what the reference's
// scripts/generate_kmers.py does in Python (reference scripts/generate_kmers.py:55-136), as a PAM scan kernel + ordered
// compaction per chromosome, with the CSV rows formatted on the host.  Output is byte-identical to the script's stdout.
// The scan and the compaction form one site producer (gsx::SiteScanner, gsx_sites.h) with two consumers: gsx_generate_kmers, which
// writes the CSV, and gsx_enumerate_genome (gsx_format.cpp), which feeds the sites to the search without the CSV in between.
//
// Semantics restated (not copied) from the script:
//   * chromosome = first word of the FASTA header; sequence upper-cased; records shorter than min_chr_length are skipped
//   * the PAM pattern's N's are expanded one at a time, first N first, in the order A,C,T,G, breadth first -- e.g. NGG gives
//     AGG, CGG, TGG, GGG (generate_kmers.py:55-68); the "-" strand uses the reverse complements of the same list.  IUPAC class
//     letters (R, Y, ..., V) expand the same way into their members, in the same order (NRG: AAG, AGG, CAG, CGG, TAG, ...)
//   * for each concrete PAM, every (overlapping) occurrence i: PAM at the end (default): "+" k-mer = chr[i-k, i), position
//     i-k; "-" k-mer = revcomp(chr[i+|pam|, i+|pam|+k)), position i.  PAM at the start (--start): "+" k-mer =
//     chr[i+|pam|, i+|pam|+k), position i; "-" k-mer = revcomp(chr[i-k, i)), position i-k (generate_kmers.py:70-100)
//   * dropped: negative position, k-mer running off the chromosome, any base outside ACGT (generate_kmers.py:96-117)
//   * row: id = prefix + chr:pos1:sense, sequence, pam PATTERN, chr, pos1 (1-based), sense; per chromosome all "+" rows by
//     concrete PAM then position, then all "-" rows; duplicates are kept (generate_kmers.py:119-136)
#include "../../include/gsx.h"
#include "gsx_host.h"
#include "gsx_sites.h"
#include "gsx_iupac.h"
#include <cub/cub.cuh>
#include <thrust/iterator/counting_iterator.h>
#include <cuda_runtime.h>
#include <algorithm>
#include <chrono>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <deque>
#include <mutex>
#include <string>
#include <thread>
#include <vector>

int gsx_set_error(int code, const std::string& msg);      // gsx_api.cpp

namespace {

// flags[i] = 1 iff a k-mer is generated for PAM occurrence i
//   kmer_off: offset of the k-mer relative to i (may be negative); the reported position is i + pos_off
//   kRegions: the k-mer must also start inside one of the n_ranges sorted, disjoint [lo, hi] ranges (a binary search per
//   candidate; without regions the kernel is the plain scan)
template <bool kRegions>
__global__ void kmer_scan_kernel(const unsigned char* __restrict__ chr, uint32_t len, uint64_t pam_packed, uint32_t plen,
                                 int32_t kmer_off, uint32_t k, const uint2* __restrict__ ranges, uint32_t n_ranges,
                                 unsigned char* __restrict__ flags) {
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < len; i += gridDim.x * blockDim.x) {
        bool ok = i + plen <= len;
        for (uint32_t j = 0; ok && j < plen; j++) ok = chr[i + j] == (unsigned char)(pam_packed >> (8 * j));
        const int64_t a = (int64_t)i + kmer_off;
        ok = ok && a >= 0 && a + k <= len;
        if (kRegions && ok) {
            uint32_t lo = 0, hi = n_ranges;                                                   // ranges with .x <= a: [0, lo)
            while (lo < hi) { const uint32_t mid = (lo + hi) / 2; if (ranges[mid].x <= (uint32_t)a) lo = mid + 1; else hi = mid; }
            ok = lo > 0 && (uint32_t)a <= ranges[lo - 1].y;
        }
        for (uint32_t j = 0; ok && j < k; j++) { const unsigned char c = chr[a + j]; ok = c == 'A' || c == 'C' || c == 'G' || c == 'T'; }
        flags[i] = ok ? 1 : 0;
    }
}
__global__ void upper_kernel(unsigned char* s, uint32_t len) {
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < len; i += gridDim.x * blockDim.x) { unsigned char c = s[i]; if (c >= 'a' && c <= 'z') s[i] = c - 32; }
}

#define KCK(x) do { cudaError_t e_ = (x); if (e_ != cudaSuccess) throw gsx::SiteError{GSX_ERR_CUDA, std::string(#x ": ") + cudaGetErrorString(e_)}; } while (0)

// (IUPAC class letters expand into their members the same way: gsx_iupac.h)
std::vector<std::string> expand_pam(const std::string& pam) { return gsx::iupac_expand(pam); }

struct DeviceScratch {
    unsigned char* chr = nullptr; unsigned char* flags = nullptr; uint32_t* pos = nullptr; uint32_t* count = nullptr; void* tmp = nullptr;
    uint2* ranges = nullptr;
    size_t cap = 0, tmp_bytes = 0, ranges_cap = 0;
    ~DeviceScratch() { cudaFree(chr); cudaFree(flags); cudaFree(pos); cudaFree(count); cudaFree(tmp); cudaFree(ranges); }
    void reserve(size_t len) {
        if (len <= cap) return;
        cudaFree(chr); cudaFree(flags); cudaFree(pos); cudaFree(tmp); chr = flags = nullptr; pos = nullptr; tmp = nullptr;
        cap = len + len / 4 + 1024;
        KCK(cudaMalloc(&chr, cap)); KCK(cudaMalloc(&flags, cap)); KCK(cudaMalloc(&pos, cap * 4));
        if (!count) KCK(cudaMalloc(&count, 4));
        tmp_bytes = 0;
        thrust::counting_iterator<uint32_t> it(0);
        KCK(cub::DeviceSelect::Flagged(nullptr, tmp_bytes, it, flags, pos, count, (int)cap));
        KCK(cudaMalloc(&tmp, tmp_bytes));
    }
    void reserve_ranges(size_t n) {
        if (n <= ranges_cap) return;
        cudaFree(ranges); ranges = nullptr;
        ranges_cap = n + n / 2 + 16;
        KCK(cudaMalloc(&ranges, ranges_cap * sizeof(uint2)));
    }
};

}  // namespace

namespace gsx {

bool FastaReader::read_line() {
    line_.clear();
    char chunk[1 << 16];
    while (fgets(chunk, sizeof chunk, f_)) {
        line_ += chunk;
        if (line_.back() == '\n') return true;
    }
    return !line_.empty();
}

bool FastaReader::next(std::string& name, std::string* seq, uint64_t* len) {
    while (!have_header_) {
        if (!read_line()) return false;
        have_header_ = !line_.empty() && line_[0] == '>';
    }
    {
        const std::string& l = line_;
        size_t b = 1; while (b < l.size() && isspace((unsigned char)l[b])) b++;
        size_t e = b; while (e < l.size() && !isspace((unsigned char)l[e])) e++;
        name = l.substr(b, e - b);
    }
    have_header_ = false;
    if (seq) seq->clear();
    uint64_t n = 0;
    while (read_line()) {
        const std::string& l = line_;
        if (!l.empty() && l[0] == '>') { have_header_ = true; break; }
        size_t e = l.size(); while (e && isspace((unsigned char)l[e - 1])) e--;
        bool inner = false; for (size_t q = 0; q < e; q++) if (isspace((unsigned char)l[q])) { inner = true; break; }
        if (!inner) { if (seq) seq->append(l, 0, e); n += e; }                             // the usual line: one block
        else for (size_t q = 0; q < e; q++) if (!isspace((unsigned char)l[q])) { if (seq) *seq += l[q]; n++; }
    }
    if (len) *len = n;
    return true;
}

std::vector<StartRange> merge_regions(std::vector<std::pair<uint64_t, uint64_t>> iv, uint32_t k) {
    std::vector<StartRange> out;
    std::sort(iv.begin(), iv.end());
    for (const auto& x : iv) {
        if (x.second < x.first + k) continue;                                                // shorter than a k-mer
        const uint32_t lo = (uint32_t)x.first, hi = (uint32_t)(x.second - k);
        if (!out.empty() && (uint64_t)lo <= (uint64_t)out.back().second + 1) out.back().second = std::max(out.back().second, hi);
        else out.emplace_back(lo, hi);
    }
    return out;
}

struct SiteScanner::Impl { DeviceScratch D; };

SiteScanner::SiteScanner(const std::string& pam, uint32_t k, bool start, int device)
    : d_(new Impl()), k_(k), plen_((uint32_t)pam.size()), start_(start), device_(device) {
    pams_ = expand_pam(pam);
    n_pams_ = pams_.size();
    for (size_t q = 0; q < n_pams_; q++) { std::string r(pams_[q].rbegin(), pams_[q].rend()); for (auto& c : r) c = site_comp(c); pams_.push_back(r); }
    sites_.resize(2 * n_pams_);
}
SiteScanner::~SiteScanner() { if (d_) cudaSetDevice(device_); }      // (the scratch is freed on the device it lives on)

void SiteScanner::scan(std::string& seq, const std::vector<StartRange>* ranges) {
    for (auto& s : sites_) s.clear();
    if (ranges && ranges->empty()) return;
    if (seq.size() >= (1ull << 32) - 64) throw SiteError{GSX_ERR_ARG, "chromosome longer than 2^32 bases"};
    const uint32_t len = (uint32_t)seq.size();
    if (!len) return;
    const auto t_wait = std::chrono::steady_clock::now();
    std::unique_lock<std::mutex> turn = device_turn(device_);
    const auto t0 = std::chrono::steady_clock::now();
    wait_seconds += std::chrono::duration<double>(t0 - t_wait).count();
    DeviceScratch& D = d_->D;
    KCK(cudaSetDevice(device_));
    D.reserve(len);
    if (ranges) {
        static_assert(sizeof(StartRange) == sizeof(uint2), "ranges are uploaded as uint2");
        D.reserve_ranges(ranges->size());
        KCK(cudaMemcpy(D.ranges, ranges->data(), ranges->size() * sizeof(uint2), cudaMemcpyHostToDevice));
    }
    KCK(cudaMemcpy(D.chr, seq.data(), len, cudaMemcpyHostToDevice));
    const int blocks = (int)std::min<uint64_t>((len + 255) / 256, 148 * 16);
    upper_kernel<<<blocks, 256>>>(D.chr, len);
    KCK(cudaMemcpy(&seq[0], D.chr, len, cudaMemcpyDeviceToHost));                         // the rows print the upper-cased bases
    for (size_t l = 0; l < sites_.size(); l++) {
        const std::string& p = pams_[l];
        uint64_t packed = 0; for (uint32_t j = 0; j < plen_; j++) packed |= (uint64_t)(unsigned char)p[j] << (8 * j);
        if (ranges) kmer_scan_kernel<true><<<blocks, 256>>>(D.chr, len, packed, plen_, kmer_off(l), k_, D.ranges, (uint32_t)ranges->size(), D.flags);
        else kmer_scan_kernel<false><<<blocks, 256>>>(D.chr, len, packed, plen_, kmer_off(l), k_, nullptr, 0, D.flags);
        thrust::counting_iterator<uint32_t> it(0);
        size_t tb = D.tmp_bytes;
        KCK(cub::DeviceSelect::Flagged(D.tmp, tb, it, D.flags, D.pos, D.count, (int)len));
        uint32_t n = 0; KCK(cudaMemcpy(&n, D.count, 4, cudaMemcpyDeviceToHost));
        sites_[l].resize(n);
        if (n) KCK(cudaMemcpy(sites_[l].data(), D.pos, (size_t)n * 4, cudaMemcpyDeviceToHost));
    }
    chromosomes++;
    seconds += std::chrono::duration<double>(std::chrono::steady_clock::now() - t0).count();
}

}  // namespace gsx

extern "C" int gsx_generate_kmers(const char* fasta_path, const char* out_csv_path, const char* pam_c, uint32_t k, uint64_t min_chr_length,
                                  const char* prefix_c, int start, int device, uint64_t* n_kmers) {
    if (!fasta_path || !out_csv_path || !pam_c) return gsx_set_error(GSX_ERR_ARG, "null argument");
    const std::string pam(pam_c), prefix(prefix_c ? prefix_c : "");
    if (pam.empty() || pam.size() > 8 || k == 0 || k > 64) return gsx_set_error(GSX_ERR_ARG, "PAM must have 1..8 characters and the k-mer 1..64");
    for (char c : pam) if (!gsx::iupac_pam_char(c)) return gsx_set_error(GSX_ERR_ARG, "PAM characters must be A, C, G, T, N or an IUPAC class letter (R, Y, S, W, K, M, B, D, H, V)");
    int have = 0;
    if (cudaGetDeviceCount(&have) != cudaSuccess || have <= 0) return gsx_set_error(GSX_ERR_NO_DEVICE, "no CUDA device available (this library has no CPU path)");
    if (device < 0 || device >= have) return gsx_set_error(GSX_ERR_ARG, "device ordinal out of range");
    FILE* in = fopen(fasta_path, "rb");
    if (!in) return gsx_set_error(GSX_ERR_IO, std::string("cannot open ") + fasta_path);
    FILE* out = fopen(out_csv_path, "wb");
    if (!out) { fclose(in); return gsx_set_error(GSX_ERR_IO, std::string("cannot write ") + out_csv_path); }
    uint64_t total = 0;
    int rc = GSX_OK;
    try {
        KCK(cudaSetDevice(device));
        gsx::SiteScanner S(pam, k, start != 0, device);
        std::string buf; buf.reserve(1 << 22);
        fputs("id,sequence,pam,chromosome,position,sense\n", out);
        size_t rows_per_thread = 16384;                                                      // (tests lower it to reach the threaded writer on small inputs)
        if (const char* e = getenv("GSX_KMERS_ROWS_PER_THREAD")) if (*e && atoll(e) > 0) rows_per_thread = (size_t)atoll(e);

        auto process = [&](const std::string& name, std::string& seq) {
            if (seq.size() < min_chr_length || seq.empty()) return;
            S.scan(seq, nullptr);
            for (size_t l = 0; l < S.n_lists(); l++) {
                const std::vector<uint32_t>& hpos = S.sites(l);
                const bool fwd = S.forward(l);
                const size_t n = hpos.size();
                // rows of sites [lo, hi) appended to o (find_kmers + the print loop of the script)
                auto format_rows = [&](size_t lo, size_t hi, std::string& o, bool flush) {
                    for (size_t q = lo; q < hi; q++) {
                        char num[16]; const int nl = snprintf(num, sizeof num, "%u", S.pos1(l, hpos[q]));
                        gsx::append_site_id(o, prefix, name, num, nl, fwd); o += ',';
                        gsx::append_site_kmer(o, seq, S.kmer_start(l, hpos[q]), k, fwd);
                        o += ','; o += pam; o += ','; o += name; o += ','; o.append(num, nl); o += ','; o += fwd ? '+' : '-'; o += '\n';
                        if (flush && o.size() > (1u << 22) - 256) { fwrite(o.data(), 1, o.size(), out); o.clear(); }
                    }
                };
                const size_t nt = std::min<size_t>(std::max(1u, std::thread::hardware_concurrency()), n / rows_per_thread);
                if (nt < 2) format_rows(0, n, buf, true);
                else {
                    // many rows (a whole chromosome of PAM sites): slices on host threads, written in order behind what is buffered
                    fwrite(buf.data(), 1, buf.size(), out); buf.clear();
                    std::vector<std::string> parts(nt); std::vector<std::thread> th;
                    const size_t row_bytes = 2 * (prefix.size() + name.size()) + 2 * 11 + k + pam.size() + 16;
                    for (size_t t = 0; t < nt; t++)
                        th.emplace_back([&, t] { const size_t lo = (size_t)n * t / nt, hi = (size_t)n * (t + 1) / nt; parts[t].reserve((hi - lo) * row_bytes); format_rows(lo, hi, parts[t], false); });
                    for (auto& x : th) x.join();
                    for (const std::string& o : parts) fwrite(o.data(), 1, o.size(), out);
                }
                total += n;
            }
        };

        gsx::FastaReader rd(in);
        std::string name, seq;
        while (rd.next(name, &seq, nullptr)) process(name, seq);
        fwrite(buf.data(), 1, buf.size(), out);
    } catch (const gsx::SiteError& f) { rc = gsx_set_error(f.code, f.msg); }
    catch (const std::bad_alloc&) { rc = gsx_set_error(GSX_ERR_NOMEM, "out of host memory"); }
    fclose(in); fclose(out);
    if (n_kmers) *n_kmers = total;
    return rc;
}
