// gsx_host.h -- host-side structures behind the C ABI (include/gsx.h).
#ifndef GSX_HOST_H
#define GSX_HOST_H
#include "gsx_types.h"
#include "gsx_kernels.h"
#include <map>
#include <mutex>
#include <string>
#include <vector>
#include <cstdint>

namespace gsx {

struct HostStrand {
    uint64_t n = 0;                       // rows = text length + 1
    std::vector<OccBlock> blocks;         // n/64 + 1
    std::vector<uint32_t> sa_samples;
    uint32_t sa_shift = 6;
    std::vector<uint32_t> exc_rows, exc_lf, n_rows;
    std::vector<uint8_t> exc_sym;         // BWT byte of each exception row (0 = sentinel)
    uint32_t C[5] = {0, 0, 0, 0, 0};
};

struct HostIndex {
    HostStrand st[2];
    std::vector<std::string> chr_names;
    std::vector<uint64_t> chr_lens;
    uint64_t genome_length = 0;
};

// Builds blocks / exception tables / C from a BWT given as bytes (0 = sentinel).  `next` yields row i's symbol.
struct StrandBuilder {
    HostStrand* out;
    uint64_t n, row = 0;
    uint64_t run[256];
    std::vector<uint64_t> exc_rank;
    OccBlock cur;
    explicit StrandBuilder(HostStrand* o, uint64_t n_rows);
    void push(uint8_t sym);
    void finish();
};

bool load_sdsl_strand(const std::string& path, HostStrand& out, std::string& err);       // SURVEY.md App. B
bool load_genome_structure(const std::string& path, HostIndex& ix, std::string& err);    // seq_io.cxx:124-144
bool read_fasta(const std::string& path, std::vector<uint8_t>& seq, HostIndex& ix, std::string& err);   // seq_io.cxx:57-63,74-110
bool save_gsx(const std::string& prefix, const HostIndex& ix, std::string& err);
bool load_gsx(const std::string& prefix, HostIndex& ix, std::string& err);
DevStrand host_view(const HostStrand& h);                          // the host arrays behind the kernels' own index arithmetic (gsx_core.h)
// the reference's own format back out (gsx_sdsl_write.cpp): <prefix>.forward / .reverse / .gs, byte for byte what `guidescan index` writes
bool save_sdsl_index(const std::string& prefix, const HostIndex& ix, std::string& err);
bool save_sdsl_strand(const std::string& path, const HostStrand& h, unsigned threads, std::string& err);
// parts of it on their own, for tests/sdsl_write_check.cpp
bool sdsl_write_wavelet_tree(const std::string& path, const HostStrand& h, unsigned threads, std::string& err);
bool sdsl_write_bit_vector_supports(const std::string& path, const std::vector<uint64_t>& words, uint64_t n_bits, std::string& err);

// the device arrays of one strand index, each with its size in bytes (the replicas on further devices are peer copies)
//   exc_map: one bit per 64-row block holding an exception row (SearchArgs::exc_map)
#define GSX_STRAND_ARRAYS(X) X(blocks) X(lines) X(sum0) X(sum1) X(sum2) X(ftab) X(sa) X(exc_rows) X(exc_lf) X(n_rows) X(exc_map)
struct DeviceStrand {
    DevStrand d{};
#define GSX_DECL(name) void* name = nullptr; size_t name##_bytes = 0;
    GSX_STRAND_ARRAYS(GSX_DECL)
#undef GSX_DECL
};
struct DeviceIndex {
    int device = 0;
    int sm_count = 148;
    int alias_of = -1;            // >= 0: this slot names a device that an earlier slot already holds; it shares that slot's arrays
    DeviceStrand st[2];
    Chrom* chroms = nullptr;
    uint64_t bytes = 0;
};

// a device's turn (gsx_api.cpp): held by a call from its first search launch to its last result copy, and by the PAM scan of the
// genome driver (gsx_sites.h) from its chromosome upload to its last site list; an empty lock when GSX_DEVICE_LOCK=0
std::unique_lock<std::mutex> device_turn(int device);

// GPU suffix sorting (gsx_build.cu): text (bytes, no sentinel) -> HostStrand with samples every 2^sa_shift rows
bool build_strand_gpu(int device, const uint8_t* text, uint64_t len, uint32_t sa_shift, HostStrand& out, std::string& err);

}  // namespace gsx

struct gsx_index {
    gsx::HostIndex host;
    std::vector<gsx::DeviceIndex> dev;
    std::vector<gsx::Chrom> chroms;
    // seconds spent by gsx_index_open / gsx_index_build: [0] reading + converting the files (or suffix sorting), [1] upload and
    // derived arrays (jump table, look-ahead lines, summaries) on the first device, [2] replication to the other devices
    double open_seconds[3] = {0, 0, 0};
    // matches per guide that earlier calls needed, per option set (gsx_api.cpp: first size of the match arena); the one mutable
    // part of an otherwise immutable handle
    mutable std::mutex learn_mu; mutable std::map<uint64_t, double> learned_matches_per_guide;
};

#include "../../include/gsx.h"
#include <new>
namespace gsx {
// size-bucketed recycling of device (device >= 0) and pinned host (device == -1) allocations: cudaMalloc /
// cudaHostAlloc cost milliseconds each, far more than the kernels of a small batch
void* pool_get(int device, size_t bytes);
void pool_put(int device, void* p, size_t bytes);
void pool_trim(int device);

struct HostArrays {             // one device batch worth of results (pinned host memory)
    size_t n_guides = 0, n_hits = 0;
    uint8_t* dropped = nullptr; uint32_t* n_hits_of = nullptr; uint32_t* hoff = nullptr; float* specificity = nullptr; uint8_t* perfect = nullptr;
    uint32_t* cbd = nullptr;
    int64_t* abs_pos = nullptr; uint32_t* sa_row = nullptr; int32_t* chr = nullptr; uint32_t* pos1 = nullptr; uint8_t* strand = nullptr;
    uint8_t* distance = nullptr; uint8_t* rna = nullptr; uint8_t* dna = nullptr; uint8_t* index_id = nullptr; float* cfd = nullptr;
    uint8_t* counted = nullptr;
    uint64_t* key_lo = nullptr; uint64_t* key_hi = nullptr; uint8_t* mlen = nullptr;      // match string of each hit: sort key (key_hi: wide keys only) and length
    std::vector<std::pair<void*, size_t>> owned;
    template <class T> T* alloc(size_t n) {
        size_t bytes = (n ? n : 1) * sizeof(T);
        void* p = pool_get(-1, bytes);               // pinned host memory, recycled between calls
        if (!p) throw std::bad_alloc();
        owned.emplace_back(p, bytes); return (T*)p;
    }
    void release() { for (auto& q : owned) pool_put(-1, q.first, q.second); owned.clear(); }
};

}  // namespace gsx

namespace gsx {
struct Prepared {
    std::vector<GuideRec> recs;
    PamSet pamsets[kMaxPamSets];
    uint32_t max_pams = 1;
    bool wide = false;
    // fast-path description (search_fast_kernel): valid when fast_ok
    bool fast_ok = false;
    std::vector<uint64_t> gq;      // per guide: 2-bit symbols in consumption order | qlen << 58
    uint32_t pampack = 0, plen = 0, min_qlen = 0;      // (first PAM of the list)
    uint32_t n_fast_pams = 0, pampacks[kMaxPams] = {0}, plens[kMaxPams] = {0};      // every PAM of the (single) PAM set: one search pass each
    uint32_t pammask = 0, pammasks[kMaxPams] = {0};    // members of the class characters of pampack / pampacks (0: A/C/G/T/N only)
    // bulges on the specialised kernels: every guide is replaced by its edited guides (gsx_core.h variant_rewrite); valid when
    // the batch would be a fast-path batch without its bulges and the edited guides are few enough
    bool variant_ok = false;
    uint32_t max_qlen = 0;
};

// what the search plan reads from a device index (DeviceIndex)
struct IndexShape {
    bool plain = true;              // no BWT row outside A/C/G/T but the sentinel, on either strand (n_exc == 1, n_nrows == 0)
    bool lines = false;             // look-ahead lines
    bool exc_map = false;           // exception-block bitmaps on both strands
    uint32_t ftab_L[2] = {0, 0};    // jump-table depth per strand
    bool sum0 = false;              // pattern summaries on both strands
    uint64_t rows = 0;              // rows of the forward strand
    int sm_count = 0;
};

// How a device job searches its n guides (gsx_api.cpp plan_search): the path, the kernel variants, the slice widths, the first
// arena sizes and every GSX_* knob of the search.  A pure function of the batch, the parameters, the index's shape and the
// environment.
struct SearchPlan {
    bool use_fast = false;          // search_fast_kernel; otherwise the general search_kernel
    bool exc = false;               // ... over an index with N (search_fast_kernel<..., EXC>)
    bool use_variants = false;      // bulges as edited guides, `chunk` edited guides per launch
    bool late_guides = false;       // the guide records go up on the second stream under the first search
    int variant_general[2] = {0, 0}, variant_fast = 1;     // occupancy variants of the tree search: general narrow / wide, fast
    int search_warps = 0, threshold_warps = 0;              // grids of the main search and of the threshold pass (<= 0: unknown variant)
    bool fuse_pams = false;         // every alternative PAM in one pass
    uint32_t search_sb = 0, threshold_sb = 0;               // slice characters of the sweep, 0 = no sweep
    bool combos = false, threshold_combos = false;          // jump-table combos (search_fast_kernel without a sweep)
    bool split = false; uint32_t split_sb = 0; int split_ctas = 6;       // two-part sweep (sweep_split_kernel)
    uint32_t load_mode = 2, pin_width = 0;
    size_t expand_roots = 0;        // general kernel with fewer tasks than its grid keeps busy: roots expanded to this many nodes
    uint32_t chunk = 0; bool fmask = false;                 // edited guides per launch; the sweep skips substituted insertions
    uint32_t edited_qmin = 0, edited_qmax = 0;              // lengths of the edited guides
    uint64_t queue_cap = 0, chunk_queue_cap = 0;            // seed queue: batch (and threshold pass), edited-guide chunk
    double match_per_guide = 0;     // main search's match arena per guide, before what earlier calls needed
    uint64_t match_cap_set = 0;     // GSX_MATCH_CAP
    uint64_t chunk_match_cap = 0, edited_match_cap = 0;     // match arenas of one edited-guide chunk and of the whole batch
    uint32_t spill_cap = 0;         // spill stack entries per warp of the main search
    // GSX_ORDER (0 warp per guide, 1 CTA per guide, 2 radix sort), GSX_SPEC_WARP, GSX_SWEEP_VARIANT; INT_MIN when not set: by
    // matches per guide, hits per guide, and mismatches and guide lengths
    int order_mode = 0, spec_warp = 0, sweep_variant_set = 0;
    bool order_probe = true;        // measure the largest matches per guide for the automatic ordering
    // the sweep's slice characters where a batch is large enough (0 = no sweep), for launches whose batch is known per chunk
    uint32_t ftab_L = 0, sweep_width = 0, sweep_min = 0;

    // slice characters of a sweep over ng guides no shorter than min_qlen with M mismatches, 0 = no sweep
    uint32_t sweep_sb(uint32_t ng, uint32_t min_qlen, uint32_t M) const;
    // sweep kernel variant for guide lengths qmin .. qmax, M mismatches and this PAM (2 where sweep_lean_kernel has no layout)
    int sweep_variant(uint32_t M, uint32_t qmin, uint32_t qmax, uint32_t plen, uint32_t pampack) const;
};
SearchPlan plan_search(const Prepared& prep, const gsx_params& p, const IndexShape& ix, uint32_t n);

// every way to substitute at most M of the first n_pos characters (k-mer jump table enumeration, gsx_core.h)
std::vector<uint64_t> ftab_combos(uint32_t n_pos, uint32_t M);
// slice-major enumeration plan (gsx_core.h sweep_pattern): the xor table of every way to substitute at most M of the
// characters outside the slice, listed per pass and budget
void sweep_make_plan(uint32_t L, uint32_t sb, uint32_t M, SweepPlan& plan, std::vector<uint32_t>& xtab);
// the same for the two-part enumeration of guides of qlen characters and a PAM of plen (gsx_types.h SplitPlan, gsx_core.h split_classes)
void split_make_plan(uint32_t L, uint32_t sb, uint32_t M, uint32_t qlen, uint32_t plen, uint32_t pampack, uint32_t half, SplitPlan& plan,
                     std::vector<uint32_t>& xtab);
// one bit per 64-row block that holds a row whose BWT symbol is not A/C/G/T (gsx_core.h exc_before)
std::vector<uint32_t> build_exc_map(const HostStrand& h);
// bulges as edited guides (gsx_core.h variant_op): every op list within the budgets; their number
std::vector<uint32_t> bulge_variants(uint32_t qlen, uint32_t R, uint32_t D);
uint64_t bulge_variant_count(uint32_t qlen, uint32_t R, uint32_t D);
}  // namespace gsx

struct gsx_result {
    using HostArrays = gsx::HostArrays; using GuideRec = gsx::GuideRec;
    std::vector<HostArrays> parts;          // in guide order
    std::vector<size_t> part_g0, part_h0;
    // merged view (only materialised when there is more than one part, and only when gsx_result_view_get asks for it)
    bool merged = false; std::mutex merge_mu;
    std::vector<uint8_t> dropped, perfect, strand, distance, rna, dna, index_id, counted;
    std::vector<uint64_t> first_hit; std::vector<uint32_t> n_hits_of, cbd, sa_row, pos1; std::vector<float> specificity, cfd;
    std::vector<int64_t> abs_pos; std::vector<int32_t> chr;
    std::vector<GuideRec> guides;
    gsx_result_view view{};
    gsx_counters counters{};
    uint32_t n_dist = 0; bool wide = false;
};


// per-hit result arrays a caller inside the library wants on the host (gsx_internal_enumerate_start_want): the whole-file driver
// formats SAM from 18 of the 39 bytes per hit and CSV from 22, and at hundreds of hits per guide the result copy is a third of a
// call.  The public calls copy everything (kWantAll); an array that was not wanted is a null pointer in HostArrays.
enum : uint32_t { kWantAbsPos = 1u, kWantSaRow = 2u, kWantChr = 4u, kWantPos1 = 8u, kWantStrand = 16u, kWantDistance = 32u, kWantBulges = 64u,
                  kWantIndexId = 128u, kWantCfd = 256u, kWantCounted = 512u, kWantMatchString = 1024u, kWantAll = 0xFFFFFFFFu };
extern "C" int gsx_internal_enumerate_start_want(const gsx_index* ix, const gsx_guide* guides, size_t n_guides, const gsx_params* p, uint32_t want, gsx_pending** out);

// internal entry points shared with the host-side unit-test harness (tests/host_core_check.cpp)
int gsx_prepare_guides(const gsx_guide* guides, size_t n, const gsx_params* p, gsx::Prepared& out);
void gsx_build_view(gsx_result* r);

#endif
