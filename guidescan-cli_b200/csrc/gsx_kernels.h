// gsx_kernels.h -- launch interface between the C-ABI host code and the CUDA kernels.
#ifndef GSX_KERNELS_H
#define GSX_KERNELS_H
#include "gsx_types.h"
#include <cuda_runtime.h>

namespace gsx {

enum : uint32_t {
    GSX_KERR_MATCH_OVERFLOW = 1,   // match arena too small: host retries with a larger one
    GSX_KERR_SPILL_OVERFLOW = 2,   // a warp's global spill stack is full: host retries with a larger one
    GSX_KERR_WATCHDOG = 4,         // iteration cap hit (never expected)
    GSX_KERR_QUEUE_OVERFLOW = 8,   // seed queue of the sweep kernel too small: host retries with a larger one
    GSX_KERR_REANCHOR = 16         // a form-1 match of a two-part search has no interval in the other index (never expected)
};

// level-L node that survived the sweep kernel's filter: the DFS kernel continues from it
struct alignas(16) SeedNode { uint32_t sp, ep, idx, tlm; };      // idx: table index of its pattern (gives the string key)

struct SearchArgs {
    DevStrand st[2];
    const GuideRec* guides;
    const PamSet* pamsets;             // kMaxPamSets entries
    SearchParams p;
    const uint8_t* skip;               // per guide: 1 = do not search (dropped by the threshold pass); may be null
    MatchRec* matches;
    uint32_t* match_count;
    uint32_t* guide_nmatch;            // per guide
    unsigned long long* guide_count;   // per guide, counting pass only
    uint32_t* task_counter;
    uint32_t* spill;                   // warps_total * spill_cap * node_words u32
    unsigned long long* stats;         // [0] nodes [1] lookups [2] spilled nodes [3] LF steps [7] lookups of search_fast_kernel alone
    uint32_t* error_flag;
    uint32_t max_iters;
    uint32_t max_pams;
    // fast path only (search_fast_kernel): one PAM for all guides, ACGT-only guides, sentinel-only exception tables
    const uint64_t* gq;                // per guide: 2-bit symbol codes in consumption order | qlen << 58
    uint32_t pampack;                  // 3 bits per PAM character in consumption order (4 = N wildcard, 5 = never matches, 6 = class)
    uint32_t plen;
    uint32_t pin_width;                // packed-block loads of intervals at least this wide ask L2 to keep the line (evict_last)
    const uint64_t* combos;            // k-mer jump table enumeration: substitution combos over characters 2 .. ftab_L - 1
    uint32_t n_combos;
    const Node* gseeds;                // general kernel, if set: the tasks are these nodes (roots expanded a few levels on the host
    uint32_t n_gseeds;                 // so that a small batch still gives every warp work), not (guide, strand) roots
    const SeedNode* seeds;             // if set: the tasks are these level-L nodes (written by sweep_kernel), not (guide, strand) roots
    const uint32_t* n_seeds;           // device word: number of seeds written (may exceed seed_cap if the queue overflowed)
    uint32_t seed_cap;
    // several alternative PAMs in one pass (gsx_core.h fused_pam_ok): pampack above is then the filter PAM; 0 = off
    uint32_t n_fused;
    uint32_t fused_pams[kMaxPams];
    // genomes with N / IUPAC characters on the specialised tree search (search_fast_kernel<..., EXC>): one bit per 64-row block
    // that holds a row whose BWT symbol is not A/C/G/T (occ(A) is corrected from the exception table only there); 0 = off
    uint32_t exc;
    const uint32_t* exc_map[2];
    // edited guides (bulges): per guide, the must-match positions as an index mask (gsx_core.h variant_forced_mask); the sweep
    // skips the patterns that substitute them; nullptr = off
    const uint32_t* fmask;
    // IUPAC class characters (code 6 of pampack / fused_pams): 4 bits per PAM character, the members (A=1, C=2, G=4, T=8) of a class
    // character and 0 for every other one -- all zero for an A/C/G/T/N PAM list
    uint32_t pammask;
    uint32_t fused_masks[kMaxPams];
};

constexpr int kSweepXtabShared = 4352;          // words of shared memory the sweep kernels keep for the xor table (17 KB)
struct SweepArgs {
    DevStrand st[2];
    const uint64_t* gq;                // as SearchArgs::gq
    const uint8_t* skip;
    uint32_t n_guides;
    SweepPlan plan;
    const uint32_t* xtab;              // gsx_core.h sweep_pattern
    uint32_t n_xtab;
    uint32_t* gtab;                    // n_guides * 20 words: per-guide constants, written by launch_sweep_guides
    uint32_t M, plen, pampack;
    uint32_t parts;                    // (unused: cutting the work units was measured and did not pay)
    uint32_t load_mode;                // cache policy of the summary loads: 0 ld.global.nc, 1 + L1::no_allocate, 2 ld.global.cg
    SeedNode* queue; uint32_t queue_cap;
    uint32_t* queue_count; uint32_t* item_counter; uint32_t* error_flag;
    unsigned long long* stats;         // [0] nodes [1] lookups (reference unit) [5] summary sectors loaded
    const uint32_t* fmask;             // as SearchArgs::fmask (nullptr = off)
    // two-part enumeration (sweep_split_kernel): gtab holds 2 * n_guides rows, form 0 (gq) then form 1 (gq2); seeds of form 1 go to queue2
    const uint64_t* gq2;
    SeedNode* queue2; uint32_t* queue2_count;
    SplitPlan split;
};

// the form-1 matches of a two-part search (sweep_split_kernel) -> the records the distal-first search emits for the same alignments
struct ReanchorArgs {
    DevStrand st[2];
    const MatchRec* in; const uint32_t* n_in; uint32_t in_cap;     // form-1 matches (task = guide * 2 + the index they were found in)
    const uint64_t* gq; const uint64_t* gq2;
    uint32_t pampack, plen;
    MatchRec* out; uint32_t* out_count; uint32_t out_cap;
    uint32_t* guide_nmatch; uint32_t* error_flag;
    unsigned long long* stats;         // [7] += jump-table and occurrence lookups
};

struct LocateArgs {
    DevStrand st[2];
    const MatchRec* matches;
    const GuideRec* guides;
    const PamSet* pamsets;
    const Chrom* chroms;
    const uint32_t* hit_match;
    const uint32_t* hit_row;
    uint32_t n_hits, n_chr, wide;
    uint64_t genome_length;
    int64_t* abs_pos; int32_t* chr; uint32_t* pos1; uint8_t* strand; uint8_t* distance; uint8_t* dna; uint8_t* rna;
    uint8_t* index_id; float* cfd; uint8_t* flags;
    // the match string of the hit, as the host decodes it (gsx_core.h decode_match): its sort key and its length -- so that the result
    // carries 9 (17 with bulges) bytes per hit instead of the 32-byte match record and an index into the arena
    uint64_t* key_lo; uint64_t* key_hi; uint8_t* mlen;      // key_hi: wide keys only (else nullptr)
    unsigned long long* stats;
};

struct SpecArgs {
    const uint32_t* guide_hoff;        // n_guides + 1
    const uint32_t* count_by_distance;
    const int32_t* chr; const float* cfd; const uint8_t* flags;
    uint8_t* counted; float* specificity; uint8_t* perfect;
    uint32_t n_guides, n_dist, sam_rule;
    int64_t max_off_targets;
    uint32_t warp_per_guide;           // 1: one warp per guide (batches averaging more than 64 hits per guide), 0: one thread per guide
};

cudaError_t upload_cfd_tables();
// packed 32-byte blocks (src) -> 128-byte lines with look-ahead planes t1..t6 (dst must hold n_blocks * 128 bytes)
// k-mer jump table of depth L for one strand; tab and tmp must each hold 4^L entries of 8 bytes; result ends up in tab
cudaError_t launch_build_ftab(const DevStrand& st, uint32_t L, void* tab, void* tmp, cudaStream_t s);
// (tail: optional scratch of n_blocks * 32 bytes receiving the planes t7, t8)
cudaError_t launch_build_lookahead(const DevStrand& src, unsigned char* lines, unsigned char* tail, uint32_t n_blocks, cudaStream_t s);
// jump table + look-ahead lines -> pattern summaries of the sweep kernel (sum0, sum1: 32 bytes per table entry each)
cudaError_t launch_build_summary(const void* tab, const unsigned char* lines, const unsigned char* tail, unsigned char* sum0, unsigned char* sum1,
                                 unsigned char* sum2, uint64_t n_entries, cudaStream_t s);      // sum2: 16 bytes per entry, with tail only
int search_grid_warps(bool wide, int variant, int sm_count);
cudaError_t launch_search(const SearchArgs& a, bool wide, int variant, int sm_count, cudaStream_t s, int* warps_total);
int search_fast_grid_warps(int variant, int sm_count);
cudaError_t launch_search_fast(const SearchArgs& a, int variant, int sm_count, cudaStream_t s);
cudaError_t launch_sweep_guides(const SweepArgs& a, cudaStream_t s);      // per-guide filter masks (before launch_sweep)
cudaError_t launch_sweep(const SweepArgs& a, int variant, int sm_count, cudaStream_t s);
// two-part enumeration: PAM-first queries of the guides (gsx_core.h split_query), the sweep over both forms, the re-anchoring
cudaError_t launch_split_queries(const uint64_t* gq, uint32_t n, uint32_t pampack, uint32_t plen, uint64_t* gq2, cudaStream_t s);
constexpr int kSplitXtabShared = 1024;          // words of shared memory sweep_split_kernel keeps for its xor table
cudaError_t launch_sweep_split(const SweepArgs& a, int ctas_per_sm, int sm_count, cudaStream_t s);
cudaError_t launch_reanchor(const ReanchorArgs& r, cudaStream_t s);
// bulges as edited guides (gsx_core.h variant_rewrite)
cudaError_t launch_variant_expand(const GuideRec* guides, uint32_t n_seg, uint32_t n_v, const uint32_t* seg, const uint32_t* descs,
                                  const uint32_t* doff, uint64_t* vq, uint32_t* vdesc, uint32_t* vguide, uint32_t* vfmask, cudaStream_t s);
cudaError_t launch_variant_rewrite(const MatchRec* vm, uint32_t n_vm, const GuideRec* guides, const uint32_t* vdesc, const uint32_t* vguide,
                                   MatchRec* out, uint32_t out_cap, uint32_t* out_count, uint32_t* guide_nmatch, uint32_t* error_flag, cudaStream_t s);
// ordering of batches with thousands of matches per guide (gsx_arrange.cu): three stable radix-sort passes instead of the
// per-guide rank sort; same outputs as launch_order.  scratch: order_sorted_scratch_bytes(n_matches) bytes
size_t order_sorted_scratch_bytes(uint32_t n_matches);
cudaError_t launch_order_sorted(const MatchRec* m, uint32_t n_matches, const uint32_t* moff, uint32_t n_guides, uint32_t n_dist,
                                uint32_t* sorted, uint32_t* sorted_off, uint32_t* nhits, uint32_t* cbd, void* scratch, size_t scratch_bytes, cudaStream_t s);
cudaError_t launch_scan(const uint32_t* in, uint32_t* out, uint32_t n, cudaStream_t s);
cudaError_t launch_scatter(const MatchRec* m, uint32_t n, const uint32_t* moff, uint32_t* cursor, uint32_t* by_guide, cudaStream_t s);
cudaError_t launch_order(const MatchRec* m, const uint32_t* moff, const uint32_t* by_guide, uint32_t n_guides, uint32_t n_dist,
                         uint32_t* sorted, uint32_t* sorted_off, uint32_t* nhits, uint32_t* cbd, bool many_per_guide, cudaStream_t s);
cudaError_t launch_expand(const MatchRec* m, const uint32_t* moff, const uint32_t* sorted, const uint32_t* sorted_off, const uint32_t* hoff,
                          uint32_t n_guides, uint32_t n_sorted, uint32_t* hit_match, uint32_t* hit_row, uint32_t* hit_guide, cudaStream_t s);
cudaError_t launch_locate_score(const LocateArgs& a, cudaStream_t s);
cudaError_t launch_specificity(const SpecArgs& a, cudaStream_t s);
cudaError_t launch_threshold(const unsigned long long* gc, uint8_t* dropped, uint32_t n, cudaStream_t s);
// small read-backs that must not queue on the copy engine: stores into pinned host memory
cudaError_t launch_publish(const uint32_t* src, uint32_t n_words, uint32_t* host_dst, cudaStream_t s);
// host_dst[0] = 64-bit sum, host_dst[1] = maximum of the n counts; scratch: 2 zeroed words, done: 1 zeroed word
cudaError_t launch_total_u32(const uint32_t* in, uint32_t n, unsigned long long* scratch, unsigned int* done, unsigned long long* host_dst, cudaStream_t s);
cudaError_t launch_checksum(const void* p, size_t bytes, unsigned long long seed, unsigned long long* out, cudaStream_t s);      // *out += digest
cudaError_t launch_rank_query(const DevStrand& st, const uint32_t* rows, const uint8_t* syms, uint32_t n, uint32_t* out, cudaStream_t s);
cudaError_t launch_locate_query(const DevStrand& st, const uint32_t* rows, uint32_t n, uint32_t* out, cudaStream_t s);

}  // namespace gsx
#endif
