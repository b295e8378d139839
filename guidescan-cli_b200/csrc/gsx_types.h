// gsx_types.h -- data layout shared by host code and CUDA kernels.
//
// GPU index layout (per strand index; replaces sdsl::csa_wt<wt_huff<>,64,8192>, reference src/guidescan.cxx:24-27):
//   * OccBlock[n/64 + 1]: one 32-byte sector per 64 BWT rows = 4 x u32 occurrence checkpoints (A,C,G,T before the
//     block) + the 64 rows' 2-bit symbols as two bit planes.  One occurrence lookup = ONE aligned 32 B load
//     (LDG.E.256), against 4-6 dependent cache lines in wt_pc::rank (sdsl wt_pc.hpp:360-384).
//   * rows whose BWT symbol is not A/C/G/T ('$' sentinel row, genome N / IUPAC) are stored as code 0 in the planes
//     and listed in a sorted exception table; occ(A) is corrected from it, so rank stays exact.
//   * SA samples: SA[row] for every row that is a multiple of 2^sa_shift (reference density: 64 rows).
//   * optional look-ahead lines: a B200 L1 miss always pulls the whole 128-byte line from L2/DRAM
//     (profiles/r01e_gather_width_ncu.csv).  Wide SA intervals (top of the search tree) use the packed blocks, where
//     one line covers 256 rows and both interval ends usually share it; for narrow intervals (all rows inside one
//     64-row block, the deep random-access part of the tree) a second array gives each block its own line:
//     bytes 0..31 the OccBlock, bytes 32..127 the 2-bit symbols t1..t6 of the same rows,
//     t_j(r) = BWT[LF^j(r)] = text[SA[r] - 1 - j] -- the next six characters a backward search from row r would
//     consume.  The search prunes children that cannot survive them, at no extra DRAM traffic.
#ifndef GSX_TYPES_H
#define GSX_TYPES_H
#include <stdint.h>
#include <stddef.h>

#if defined(__CUDACC__)
#define GSX_HD __host__ __device__ __forceinline__
#else
#define GSX_HD inline
#endif

namespace gsx {

constexpr int kMaxQ = 32;          // protospacer length limit
constexpr int kMaxPamLen = 8;
constexpr int kMaxPams = 8;        // alt PAMs + the guide's own
constexpr int kMaxPamSets = 16;    // distinct (pam column value) groups per call
constexpr int kMaxDist = 8;        // mismatches <= 7

// symbol codes: 0..3 = A,C,G,T ; 4 = N ; 5 = anything else (never matches) ; 6 = an IUPAC class letter of a PAM (R, Y, ..., V:
// gsx_iupac.h), whose members come from a parallel mask (PamSet::cmask, the pammask words of the kernels)
enum : uint8_t { SYM_A = 0, SYM_C = 1, SYM_G = 2, SYM_T = 3, SYM_N = 4, SYM_X = 5, SYM_CLS = 6 };

struct alignas(32) OccBlock {
    uint32_t cnt[4];   // occurrences of A,C,G,T in BWT[0, 64*b)
    uint64_t hi;       // bit j = high bit of the 2-bit code of row 64*b + j
    uint64_t lo;       // bit j = low bit
};

struct DevStrand {
    const OccBlock* blocks;
    const uint32_t* sa_samples;    // SA[k << sa_shift]
    const uint32_t* exc_rows;      // sorted rows whose BWT symbol is not ACGT
    const uint32_t* exc_lf;        // LF target of each exception row
    const uint32_t* n_rows;        // sorted rows whose BWT symbol is 'N'
    uint32_t n;                    // number of rows = genome length + 1
    uint32_t n_exc;
    uint32_t n_nrows;
    uint32_t sa_shift;
    uint32_t C[5];                 // C[A],C[C],C[G],C[T],C[N]: rows whose suffix starts with a smaller symbol
    uint32_t exc_lo, exc_hi;       // first / last exception row (fast reject)
    uint32_t blk_shift;            // log2 of the byte stride between OccBlocks in `blocks` (5 = packed)
    const void* ftab;              // optional k-mer jump table: 4^ftab_L FtabEntry {sp, width} (gsx_core.h), nullptr if absent
    uint32_t ftab_L;
    const unsigned char* lines;    // optional second copy, one 128-byte line per 64 rows: OccBlock + six look-ahead symbol
                                   // planes (see build_lookahead_kernel); nullptr if absent
    const unsigned char* sum0;     // optional pattern summaries of the sweep kernel, 32 bytes per jump-table entry (same index):
    const unsigned char* sum2;     //   (sum2[e], 16 bytes: the two further symbols t7, t8 of rows sp .. sp+31 as 32-bit plane pairs -- for a
                                   //   20-nt guide at L = 14 these are the two fixed PAM characters; read only by the few survivors)
    const unsigned char* sum1;     //   sum0[e] = header + the seven look-ahead symbols t0..t6 of rows sp .. sp+15 of the entry's
                                   //   interval as 16-bit plane pairs, sum1[e] = the same for rows sp+16 .. sp+31 (gsx_core.h
                                   //   summary_eval).  t_j = the character a backward search from that row consumes j steps ahead
                                   //   (as in `lines`).  One 32-byte load indexed by the pattern itself replaces the table entry
                                   //   + look-ahead line reads; nullptr if absent (see build_summary_kernel)
};

GSX_HD const OccBlock* block_ptr(const DevStrand& st, uint32_t b) {
    return reinterpret_cast<const OccBlock*>(reinterpret_cast<const char*>(st.blocks) + ((size_t)b << st.blk_shift));
}

struct GuideRec {                  // 80 bytes
    uint8_t q[kMaxQ];              // symbol code consumed at level l (consumption order)
    char    seq[kMaxQ];            // k.sequence as given (for CFD)
    uint8_t qlen;
    uint8_t pamset;
    uint8_t seqlen;
    uint8_t pad[13];
};

struct PamSet {
    uint8_t n_pams;
    uint8_t plen[kMaxPams];
    uint8_t sym[kMaxPams][kMaxPamLen];   // consumption order; SYM_N = wildcard
    uint8_t kpam_len;                    // length of the guide's own pam column (coordinates use it: structures.cxx:36,41)
    uint8_t pad[6];
    uint8_t cmask[kMaxPams][kMaxPamLen]; // members of a SYM_CLS character (A=1, C=2, G=4, T=8); 0 for every other character
};

struct SearchParams {
    uint32_t M, R, D;              // max mismatches / RNA bulges / DNA bulges (max_bulge_size is 1)
    uint32_t counting;             // 1 = threshold prefilter pass: only add interval widths per guide
    uint32_t n_tasks;              // 2 * n_guides  (task = guide * 2 + strand)
    uint32_t match_cap;
    uint32_t spill_cap;            // nodes per warp in the global spill stack
};

// one emitted SA interval (= reference `match`, structures.hpp:33-43)
struct alignas(8) MatchRec {
    uint64_t key_hi;               // string sort key (wide form: 4 bits per character, left aligned; narrow: 0)
    uint64_t key_lo;               // narrow form: base-5 path number
    uint32_t task;                 // guide * 2 + strand
    uint32_t sp;
    uint32_t width;                // ep - sp + 1
    uint32_t info;                 // mm | dna << 8 | rna << 16 | len << 24
};

struct Chrom { uint64_t start; uint64_t length; };

// slice-major enumeration plan of the sweep kernel (gsx_core.h)
struct SweepPlan {
    uint32_t L, sb, M;
    // xoff[z][B] = start, in the xor table, of the patterns of pass z (0: patterns that keep some budget, 1: patterns that
    // use the budget up) under budget B; xcnt[z][B] = their number
    uint32_t xoff[2][kMaxDist + 1];
    uint32_t xcnt[2][kMaxDist + 1];
    uint32_t xlines[2][kMaxDist + 1];   // how many of those patterns leave the first two characters alone (each opens a jump-table line: work counter)
};

// two-part enumeration of the sweep (sweep_split_kernel, gsx_core.h split_query): every alignment with at most 3 mismatches has at
// most one of them among the guide's ten PAM-distal characters (form 0: the guide read distal-first, as sweep_lean_kernel reads it)
// or at most one among the ten PAM-proximal ones (form 1: the guide read PAM-first, searched in the other strand's index).  Per form
// and table character a class: costs budget, never substituted, free (all four symbols at no cost), or costs budget and counts
// against the cap of one substitution over the form's capped half.
constexpr uint32_t kSplitMaxM = 3;
struct SplitPlan {
    // the slice characters (2 bits each, the low bit set) of each form that cost budget / count against the cap / are never substituted
    uint32_t cost_top[2], cap_top[2], exact_top[2];
    // xoff[f][c][B]: start, in the xor table, of the patterns of form f over the characters outside the slice with at most c (0 or 1)
    // substitutions left under the cap and budget B; xcnt: their number.  Entry = xor value | budget used << 28 (sweep_pattern)
    uint32_t xoff[2][2][kSplitMaxM + 1], xcnt[2][2][kSplitMaxM + 1];
};

// node meta word
constexpr uint32_t META_LVL_MASK = 63u;           // bits 0..5   guide positions + PAM characters consumed
constexpr uint32_t META_MM_SHIFT = 6;             // bits 6..8
constexpr uint32_t META_PAM_SHIFT = 9;            // bits 9..11
constexpr uint32_t META_DNA_SHIFT = 12;           // bits 12..14
constexpr uint32_t META_RNA_SHIFT = 15;           // bits 15..17
constexpr uint32_t META_STATE_SHIFT = 18;         // bits 18..19  0 none 1 dna 2 rna
constexpr uint32_t META_CURR_SHIFT = 20;          // bit 20

struct Node {
    uint32_t sp, ep;
    uint64_t key_lo, key_hi;
    uint32_t meta;
    uint32_t task;
};

}  // namespace gsx
#endif
