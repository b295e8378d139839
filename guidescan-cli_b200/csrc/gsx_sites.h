// gsx_sites.h -- the PAM site producer of gsx_kmers.cu and the generator's row logic, shared by its two consumers: the guides-CSV
// writer gsx_generate_kmers and the fused genome driver gsx_enumerate_genome (gsx_format.cpp).
#ifndef GSX_SITES_H
#define GSX_SITES_H
#include <cstdint>
#include <cstdio>
#include <memory>
#include <string>
#include <utility>
#include <vector>

namespace gsx {

struct SiteError { int code; std::string msg; };       // thrown by the producer and the FASTA reader

// FASTA records one at a time: name = first word of the header, sequence = the lines joined without white space (generate_kmers.py
// reads records the same way through Biopython).  Lines before the first header are ignored.
class FastaReader {
public:
    explicit FastaReader(FILE* f) : f_(f) {}
    // the next record; seq == nullptr: only its length is counted (*len)
    bool next(std::string& name, std::string* seq, uint64_t* len);
private:
    bool read_line();
    FILE* f_; std::string line_; bool have_header_ = false;
};

// Allowed first bases of a k-mer on the + strand, [lo, hi] inclusive: sorted, disjoint (merge_regions)
using StartRange = std::pair<uint32_t, uint32_t>;
// BED intervals [s, e) of one chromosome -> the k-mer starts whose k bases lie inside one of them
std::vector<StartRange> merge_regions(std::vector<std::pair<uint64_t, uint64_t>> intervals, uint32_t k);

// Per chromosome, the PAM occurrences whose k-mer the generator emits, as one ordered list per sense and concrete PAM: the PAM
// pattern's N's expanded as generate_kmers.py does (first N first, A, C, T, G), the "-" strand through their reverse complements.
// Runs on one device and takes that device's turn (gsx_host.h device_turn) for the upload and the scan, so that it never streams a
// chromosome under a search on the same device.
class SiteScanner {
public:
    SiteScanner(const std::string& pam, uint32_t k, bool start, int device);
    ~SiteScanner();
    // upper-cases seq (on the device, copied back: the rows print upper-case bases) and fills sites(); ranges == nullptr: every site,
    // else only those whose k-mer starts inside a range (an empty list selects nothing and skips the device)
    void scan(std::string& seq, const std::vector<StartRange>* ranges);
    size_t n_lists() const { return 2 * n_pams_; }
    bool forward(size_t list) const { return list < n_pams_; }          // lists [0, n_pams): "+" by concrete PAM; then "-"
    const std::vector<uint32_t>& sites(size_t list) const { return sites_[list]; }
    // first base of the k-mer of site i on the + strand, and the 1-based position the row reports
    uint32_t kmer_start(size_t list, uint32_t i) const { return (uint32_t)((int64_t)i + kmer_off(list)); }
    uint32_t pos1(size_t list, uint32_t i) const { return kmer_start(list, i) + 1u - (before(list) ? 0u : plen_); }
    uint32_t k() const { return k_; }
    double seconds = 0, wait_seconds = 0;     // spent scanning (upload to last site list back), and waiting for the device's turn
    size_t chromosomes = 0;
private:
    bool before(size_t list) const { return forward(list) == !start_; }      // the k-mer lies in front of the PAM occurrence
    int32_t kmer_off(size_t list) const { return before(list) ? -(int32_t)k_ : (int32_t)plen_; }
    struct Impl; std::unique_ptr<Impl> d_;
    uint32_t k_, plen_; bool start_; size_t n_pams_; int device_;
    std::vector<std::string> pams_;            // forward concrete PAMs, then their reverse complements
    std::vector<std::vector<uint32_t>> sites_;
};

inline char site_comp(char c) { return c == 'A' ? 'T' : c == 'T' ? 'A' : c == 'C' ? 'G' : c == 'G' ? 'C' : 0; }
// the row's id, prefix + chr:pos1:sense, and its k-mer (reverse-complemented on "-") -- generate_kmers.py:119-136
inline void append_site_id(std::string& o, const std::string& prefix, const std::string& name, const char* num, int nl, bool fwd) {
    o += prefix; o += name; o += ':'; o.append(num, nl); o += ':'; o += fwd ? '+' : '-';
}
inline void append_site_kmer(std::string& o, const std::string& seq, uint32_t a, uint32_t k, bool fwd) {
    if (fwd) o.append(seq, a, k);
    else for (uint32_t j = 0; j < k; j++) o += site_comp(seq[a + k - 1 - j]);
}

}  // namespace gsx
#endif
