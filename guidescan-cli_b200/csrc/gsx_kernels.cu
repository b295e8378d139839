// gsx_kernels.cu -- sm_100a kernels of the off-target enumeration path.
//
//   search_kernel   backtracking backward search (reference include/genomics/index.hpp:125-398), all guides, both
//                   strand indexes.  Persistent grid; every WARP is an independent worker with its own search stack
//                   (a ring buffer in shared memory, spilling to global memory), one search-tree node per lane per
//                   iteration, children compacted onto the stack with ballot/popc.  Each occurrence lookup is one
//                   32-byte LDG.E.256 of an OccBlock; a node needs the blocks of rows sp and ep+1 (one load if both
//                   fall into the same block).  HBM-random-access bound: no tensor cores, no TMA (32 B gathers).
//   arrange_*       group the emitted SA intervals per guide, order them as the reference's std::set does,
//                   drop duplicates, expand to SA rows (reference include/genomics/process.hpp:100-115).
//   locate_score    LF walk to an SA sample per hit (sdsl csa_wt.hpp:333-346), absolute coordinate, chromosome
//                   resolution (src/genomics/structures.cxx:7-52), CFD (include/genomics/printer.hpp:98-113).
//   specificity     per-guide float32 reduction in reference order (printer.hpp:244-300 / 115-170).
#include "gsx_kernels.h"
#include "gsx_core.h"
#include "cfd_tables.h"
#include <cuda_runtime.h>

namespace gsx {

__constant__ double c_cfd_mm[4 * 4 * 20];
__constant__ double c_cfd_pam[4 * 4];

__constant__ uint64_t c_pow5[32];

cudaError_t upload_cfd_tables() {
    cudaError_t e = cudaMemcpyToSymbol(c_cfd_mm, GSX_CFD_MM, sizeof(c_cfd_mm));
    if (e != cudaSuccess) return e;
    uint64_t p5[32]; p5[0] = 1; for (int i = 1; i < 32; i++) p5[i] = p5[i - 1] * 5ull;      // 5^27 < 2^63
    e = cudaMemcpyToSymbol(c_pow5, p5, sizeof(p5));
    if (e != cudaSuccess) return e;
    return cudaMemcpyToSymbol(c_cfd_pam, GSX_CFD_PAM, sizeof(c_cfd_pam));
}

// ---------------------------------------------------------------------------------------------------------
// search
// ---------------------------------------------------------------------------------------------------------
struct Blk { uint32_t c0, c1, c2, c3; uint64_t hi, lo; };

__device__ __forceinline__ Blk ld_block(const OccBlock* p) {
    Blk b; uint32_t h0, h1, l0, l1;
    asm volatile("ld.global.nc.v8.b32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
                 : "=r"(b.c0), "=r"(b.c1), "=r"(b.c2), "=r"(b.c3), "=r"(h0), "=r"(h1), "=r"(l0), "=r"(l1)
                 : "l"(p));
    b.hi = ((uint64_t)h1 << 32) | h0; b.lo = ((uint64_t)l1 << 32) | l0;
    return b;
}

__device__ __forceinline__ Blk ld_block_hint(const void* p, uint64_t policy) {
    Blk b; uint32_t h0, h1, l0, l1;
    asm volatile("ld.global.nc.L2::cache_hint.v8.b32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8], %9;"
                 : "=r"(b.c0), "=r"(b.c1), "=r"(b.c2), "=r"(b.c3), "=r"(h0), "=r"(h1), "=r"(l0), "=r"(l1)
                 : "l"(p), "l"(policy));
    b.hi = ((uint64_t)h1 << 32) | h0; b.lo = ((uint64_t)l1 << 32) | l0;
    return b;
}

template <bool WIDE, int CAP>
struct WarpRing {
    uint32_t* sp; uint32_t* ep; uint32_t* meta; uint32_t* task; uint64_t* klo; uint64_t* khi;
    __device__ __forceinline__ void store(uint32_t slot, const Node& n) {
        slot &= (CAP - 1);
        sp[slot] = n.sp; ep[slot] = n.ep; meta[slot] = n.meta; task[slot] = n.task; klo[slot] = n.key_lo;
        if (WIDE) khi[slot] = n.key_hi;
    }
    __device__ __forceinline__ void load(uint32_t slot, Node& n) const {
        slot &= (CAP - 1);
        n.sp = sp[slot]; n.ep = ep[slot]; n.meta = meta[slot]; n.task = task[slot]; n.key_lo = klo[slot];
        n.key_hi = WIDE ? khi[slot] : 0ull;
    }
};

template <bool WIDE> __host__ __device__ constexpr int node_words() { return WIDE ? 8 : 6; }

// global spill area of one warp: SoA, `cap` nodes
template <bool WIDE>
struct SpillView {
    uint32_t* base; uint32_t cap;
    __device__ __forceinline__ void store(uint32_t i, const Node& n) {
        base[i] = n.sp; base[cap + i] = n.ep; base[2 * cap + i] = n.meta; base[3 * cap + i] = n.task;
        reinterpret_cast<uint64_t*>(base + 4 * (size_t)cap)[i] = n.key_lo;
        if (WIDE) reinterpret_cast<uint64_t*>(base + 6 * (size_t)cap)[i] = n.key_hi;
    }
    __device__ __forceinline__ void load(uint32_t i, Node& n) const {
        n.sp = base[i]; n.ep = base[cap + i]; n.meta = base[2 * cap + i]; n.task = base[3 * cap + i];
        n.key_lo = reinterpret_cast<const uint64_t*>(base + 4 * (size_t)cap)[i];
        n.key_hi = WIDE ? reinterpret_cast<const uint64_t*>(base + 6 * (size_t)cap)[i] : 0ull;
    }
};

template <bool WIDE, int WARPS, int CAP, int MINB>
__global__ void __launch_bounds__(WARPS * 32, MINB) search_kernel(SearchArgs a) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    __shared__ PamSet s_pams[kMaxPamSets];
    __shared__ DevStrand s_st[2];       // indexed per lane by strand: kept out of the (statically indexed) param bank
    for (int i = threadIdx.x; i < (int)(sizeof(PamSet) * kMaxPamSets / 4); i += blockDim.x)
        reinterpret_cast<uint32_t*>(s_pams)[i] = reinterpret_cast<const uint32_t*>(a.pamsets)[i];
    if (threadIdx.x == 0) { s_st[0] = a.st[0]; s_st[1] = a.st[1]; }
    __syncthreads();

    const uint32_t lane = threadIdx.x & 31u, warp = threadIdx.x >> 5;
    const uint32_t lt_mask = (1u << lane) - 1u;
    const uint32_t FULL = 0xffffffffu;
    constexpr int WORDS = node_words<WIDE>();

    WarpRing<WIDE, CAP> ring;
    {
        unsigned char* base = smem_raw + (size_t)warp * CAP * WORDS * 4;
        ring.klo = reinterpret_cast<uint64_t*>(base); base += CAP * 8;
        ring.khi = reinterpret_cast<uint64_t*>(base); if (WIDE) base += CAP * 8;
        ring.sp = reinterpret_cast<uint32_t*>(base); base += CAP * 4;
        ring.ep = reinterpret_cast<uint32_t*>(base); base += CAP * 4;
        ring.meta = reinterpret_cast<uint32_t*>(base); base += CAP * 4;
        ring.task = reinterpret_cast<uint32_t*>(base);
    }
    const uint32_t gwarp = blockIdx.x * WARPS + warp;
    SpillView<WIDE> spill;
    spill.cap = a.p.spill_cap;
    spill.base = a.spill + (size_t)gwarp * a.p.spill_cap * WORDS;

    uint32_t head = 0, count = 0, spill_count = 0;      // warp-uniform
    bool tasks_remain = true;                           // warp-uniform
    bool has = false;
    Node nd; nd.sp = nd.ep = nd.meta = nd.task = 0; nd.key_lo = nd.key_hi = 0;
    unsigned long long n_nodes = 0, n_lookups = 0, n_spilled = 0;
    const bool any_n = (a.st[0].n_nrows | a.st[1].n_nrows) != 0;
    uint32_t iters = 0;

    for (;;) {
        if (++iters > a.max_iters) { if (lane == 0) atomicOr(a.error_flag, GSX_KERR_WATCHDOG); break; }
        // ---- 1. give idle lanes a node ------------------------------------------------------------------
        uint32_t need_mask = __ballot_sync(FULL, !has);
        uint32_t n_need = __popc(need_mask);
        if (n_need) {
            if (count < n_need && spill_count > 0) {                 // bring back the most recently spilled chunk
                uint32_t take = spill_count < 64u ? spill_count : 64u;
                for (uint32_t j = lane; j < take; j += 32) {
                    Node t; spill.load(spill_count - take + j, t);
                    ring.store(head + count + j, t);
                }
                __syncwarp();
                count += take; spill_count -= take;
            }
            if (count < n_need && tasks_remain && a.gseeds) {        // tasks = pre-expanded nodes, 32 at a time (count < 32 <= CAP - 32)
                uint32_t t = 0;
                if (lane == 0) t = atomicAdd(a.task_counter, 32u);
                t = __shfl_sync(FULL, t, 0);
                if (t >= a.n_gseeds) tasks_remain = false;
                else {
                    const uint32_t i = t + lane;
                    const bool ok = i < a.n_gseeds && !(a.skip && a.skip[a.gseeds[i].task >> 1]);
                    const uint32_t m = __ballot_sync(FULL, ok);
                    if (ok) ring.store(head + count + __popc(m & lt_mask), a.gseeds[i]);
                    __syncwarp();
                    count += __popc(m);
                }
            } else if (count < n_need && tasks_remain) {             // start one more (guide, strand) task
                uint32_t t = 0;
                if (lane == 0) t = atomicAdd(a.task_counter, 1u);
                t = __shfl_sync(FULL, t, 0);
                if (t >= a.p.n_tasks) tasks_remain = false;
                else if (!(a.skip && a.skip[t >> 1])) {
                    if (lane == 0) {
                        Node r; r.sp = 0; r.ep = s_st[t & 1u].n - 1; r.meta = 0; r.task = t; r.key_lo = r.key_hi = 0;
                        ring.store(head + count, r);
                    }
                    __syncwarp();
                    count += 1;
                }
            }
            uint32_t take = count < n_need ? count : n_need;
            uint32_t rank = __popc(need_mask & lt_mask);
            if (!has && rank < take) { ring.load(head + count - 1 - rank, nd); has = true; }
            __syncwarp();
            count -= take;
        }
        uint32_t act = __ballot_sync(FULL, has);
        if (act == 0) {
            if (count == 0 && spill_count == 0 && !tasks_remain) break;
            continue;
        }
        // ---- 2. occurrence lookups -----------------------------------------------------------------------
        uint32_t os[4] = {0, 0, 0, 0}, oe[4] = {0, 0, 0, 0};
        const uint32_t strand = nd.task & 1u;
        const DevStrand& st = s_st[strand];
        if (has) {
            uint32_t bs = nd.sp >> 6, be = (nd.ep + 1u) >> 6;
            Blk B0 = ld_block(block_ptr(st, bs));
            Blk B1 = B0;
            if (be != bs) B1 = ld_block(block_ptr(st, be));
            n_nodes++; n_lookups += (be != bs) ? 2 : 1;
            uint32_t c0[4] = {B0.c0, B0.c1, B0.c2, B0.c3};
            block_occ(st, c0, B0.hi, B0.lo, nd.sp, os);
            uint32_t c1[4] = {B1.c0, B1.c1, B1.c2, B1.c3};
            block_occ(st, c1, B1.hi, B1.lo, nd.ep + 1u, oe);
        }
        // ---- 3. children ---------------------------------------------------------------------------------
        ExpandCtx cx;
        const GuideRec* g = a.guides + (nd.task >> 1);
        cx.st = &st; cx.g = g; cx.ps = &s_pams[has ? g->pamset : 0]; cx.M = a.p.M; cx.R = a.p.R; cx.D = a.p.D;
        Node keep; bool has_keep = false;
        keep = nd;
#pragma unroll
        for (int cand = 0; cand < CAND_END; cand++) {
            if (!WIDE && cand > CAND_FORK) break;
            if (cand == CAND_LITN && !any_n) continue;
            if (cand == CAND_FORK && a.max_pams <= 1) continue;
            Node ch; bool emit = false;
            bool valid = has && make_child<WIDE>(cand, nd, cx, os, oe, ch, emit);
            // finished alignments -> match arena (or per-guide width counter in the threshold pass)
            uint32_t emask = __ballot_sync(FULL, valid && emit);
            if (emask) {
                if (a.p.counting) {
                    if (valid && emit) atomicAdd(a.guide_count + (ch.task >> 1), (unsigned long long)(ch.ep - ch.sp + 1));
                } else {
                    uint32_t base = 0;
                    int leader = __ffs(emask) - 1;
                    if ((int)lane == leader) base = atomicAdd(a.match_count, (uint32_t)__popc(emask));
                    base = __shfl_sync(FULL, base, leader);
                    if (valid && emit) {
                        uint32_t slot = base + __popc(emask & lt_mask);
                        if (slot < a.p.match_cap) {
                            MatchRec m; fill_match(m, ch, WIDE);
                            a.matches[slot] = m;
                            atomicAdd(a.guide_nmatch + (ch.task >> 1), 1u);
                        } else atomicOr(a.error_flag, GSX_KERR_MATCH_OVERFLOW);
                    }
                }
            }
            bool push = valid && !emit;
            if (push && !has_keep) { keep = ch; has_keep = true; push = false; }     // continue depth-first in registers
            uint32_t pmask = __ballot_sync(FULL, push);
            if (pmask) {
                uint32_t np = __popc(pmask);
                if (count + np > (uint32_t)CAP) {                                     // spill the 64 oldest nodes
                    if (spill_count + 64u > spill.cap) {
                        if (lane == 0) atomicOr(a.error_flag, GSX_KERR_SPILL_OVERFLOW);
                    } else {
                        for (uint32_t j = lane; j < 64u; j += 32) { Node t; ring.load(head + j, t); spill.store(spill_count + j, t); }
                        spill_count += 64u; n_spilled += (lane == 0) ? 64 : 0;
                    }
                    __syncwarp();
                    head = (head + 64u) & (CAP - 1); count -= 64u;
                }
                if (push) ring.store(head + count + __popc(pmask & lt_mask), ch);
                __syncwarp();
                count += np;
            }
        }
        has = has_keep;
        nd = keep;
    }
    // ---- statistics ----------------------------------------------------------------------------------------
    for (int o = 16; o; o >>= 1) {
        n_nodes += __shfl_xor_sync(FULL, n_nodes, o);
        n_lookups += __shfl_xor_sync(FULL, n_lookups, o);
        n_spilled += __shfl_xor_sync(FULL, n_spilled, o);
    }
    if (lane == 0) {
        atomicAdd(a.stats + 0, n_nodes); atomicAdd(a.stats + 1, n_lookups); atomicAdd(a.stats + 2, n_spilled);
    }
}

template <bool WIDE, int WARPS, int CAP, int MINB>
static cudaError_t launch_search_t(const SearchArgs& a, int sm_count, cudaStream_t s) {
    size_t smem = (size_t)WARPS * CAP * node_words<WIDE>() * 4;
    int blocks = sm_count * MINB;
    auto k = search_kernel<WIDE, WARPS, CAP, MINB>;
    cudaError_t e = cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
    k<<<blocks, WARPS * 32, smem, s>>>(a);
    return cudaGetLastError();
}

// variant -> (warps per CTA, ring capacity, CTAs per SM); the CTA count per SM is enforced through __launch_bounds__
#define GSX_SEARCH_VARIANTS(X) \
    X(false, 0, 8, 256, 3) /* 768 thr/SM, 144 KB smem */ \
    X(false, 1, 8, 256, 4) /* 1024 thr/SM (<= 64 regs) */ \
    X(false, 2, 8, 128, 6) /* 1536 thr/SM (<= 40 regs) */ \
    X(false, 3, 8, 512, 2) /* 512 thr/SM, deep rings */ \
    X(false, 4, 4, 256, 8) /* 1024 thr/SM in 4-warp CTAs */ \
    X(true, 0, 8, 256, 2)  /* 512 thr/SM, 128 KB smem */ \
    X(true, 1, 8, 128, 4)  /* 1024 thr/SM */

cudaError_t launch_search(const SearchArgs& a, bool wide, int variant, int sm_count, cudaStream_t s, int* warps_total) {
#define X(W, V, WARPS, CAP, MINB) \
    if (wide == W && variant == V) { if (warps_total) *warps_total = sm_count * MINB * WARPS; return launch_search_t<W, WARPS, CAP, MINB>(a, sm_count, s); }
    GSX_SEARCH_VARIANTS(X)
#undef X
    return cudaErrorInvalidValue;
}

int search_grid_warps(bool wide, int variant, int sm_count) {
#define X(W, V, WARPS, CAP, MINB) if (wide == W && variant == V) return sm_count * MINB * WARPS;
    GSX_SEARCH_VARIANTS(X)
#undef X
    return -1;
}

// ---------------------------------------------------------------------------------------------------------
// k-mer jump table: one backward-search expansion per entry and level.  Entry e of level d (e = sum c_i 4^i over the d
// consumed characters) has the children e + s * 4^d: the last consumed character is the most significant digit, which
// keeps sp monotone in the index (gsx_core.h)
// ---------------------------------------------------------------------------------------------------------
__global__ void ftab_expand_kernel(DevStrand st, const FtabEntry* __restrict__ cur, FtabEntry* __restrict__ nxt, uint32_t n_cur) {
    for (uint32_t e = blockIdx.x * blockDim.x + threadIdx.x; e < n_cur; e += gridDim.x * blockDim.x) {
        const FtabEntry t = cur[e];
        uint32_t os[4] = {0, 0, 0, 0}, oe[4] = {0, 0, 0, 0};
        if (t.width) {
            const uint32_t e1 = t.sp + t.width;
            Blk B0 = ld_block(block_ptr(st, t.sp >> 6));
            uint32_t c0[4] = {B0.c0, B0.c1, B0.c2, B0.c3};
            block_occ(st, c0, B0.hi, B0.lo, t.sp, os);
            Blk B1 = ld_block(block_ptr(st, e1 >> 6));
            uint32_t c1[4] = {B1.c0, B1.c1, B1.c2, B1.c3};
            block_occ(st, c1, B1.hi, B1.lo, e1, oe);
        }
        for (int s = 0; s < 4; s++)
            reinterpret_cast<uint2*>(nxt)[(size_t)e + (size_t)s * n_cur] = make_uint2(st.C[s] + os[s], oe[s] - os[s]);
    }
}
__global__ void ftab_root_kernel(FtabEntry* t, uint32_t n) { if (threadIdx.x == 0 && blockIdx.x == 0) { t[0].sp = 0; t[0].width = n; } }

cudaError_t launch_build_ftab(const DevStrand& st, uint32_t L, void* tab, void* tmp, cudaStream_t s) {
    // ping-pong so that level L lands in `tab`
    FtabEntry* a = (FtabEntry*)((L & 1) ? tmp : tab);
    FtabEntry* b = (FtabEntry*)((L & 1) ? tab : tmp);
    ftab_root_kernel<<<1, 32, 0, s>>>(a, st.n);
    uint32_t n_cur = 1;
    for (uint32_t d = 0; d < L; d++) {
        long blocks = ((long)n_cur + 255) / 256; if (blocks > 148 * 16) blocks = 148 * 16;
        ftab_expand_kernel<<<(int)blocks, 256, 0, s>>>(st, a, b, n_cur);
        FtabEntry* t = a; a = b; b = t;
        n_cur *= 4;
    }
    return cudaGetLastError();
}

// ---------------------------------------------------------------------------------------------------------
// look-ahead planes: t_j(r) = BWT[LF^j(r)], j = 1..6, stored behind each OccBlock in its own 128-byte line
// (optionally also j = 7, 8 into `tail`, a scratch array the pattern summaries are built from)
// ---------------------------------------------------------------------------------------------------------
__global__ void build_lookahead_kernel(DevStrand st, unsigned char* __restrict__ lines, unsigned char* __restrict__ tail, uint32_t n_blocks) {
    const uint32_t lane = threadIdx.x & 31;
    const uint64_t warp = (blockIdx.x * (uint64_t)blockDim.x + threadIdx.x) >> 5, n_warps = ((uint64_t)gridDim.x * blockDim.x) >> 5;
    for (uint64_t hb = warp; hb < 2ull * n_blocks; hb += n_warps) {          // one warp per half block (32 rows)
        const uint32_t b = (uint32_t)(hb >> 1), half = (uint32_t)(hb & 1);
        unsigned char* line = lines + (size_t)b * 128;
        if (half == 0 && lane < 8) reinterpret_cast<uint32_t*>(line)[lane] = reinterpret_cast<const uint32_t*>(block_ptr(st, b))[lane];
        const uint64_t row64 = (uint64_t)b * 64 + half * 32 + lane;
        const bool valid = row64 < st.n;
        uint32_t cur = valid ? (uint32_t)row64 : 0u;
        uint32_t steps = 0;
        for (int j = 1; j <= (tail ? 8 : 6); j++) {
            uint32_t sym = 0;
            if (valid) {
                bool exc = false;
                if (st.n_exc && cur >= st.exc_lo && cur <= st.exc_hi) {
                    uint32_t k = lower_bound_u32(st.exc_rows, st.n_exc, cur);
                    if (k < st.n_exc && st.exc_rows[k] == cur) { cur = st.exc_lf[k]; exc = true; }
                }
                if (!exc) {
                    Blk B = ld_block(block_ptr(st, cur >> 6));
                    uint32_t c[4] = {B.c0, B.c1, B.c2, B.c3}, o[4];
                    block_occ(st, c, B.hi, B.lo, cur, o);
                    uint32_t s0 = block_sym(B.hi, B.lo, cur);
                    cur = st.C[s0] + o[s0];
                }
                const OccBlock* nb = block_ptr(st, cur >> 6);
                sym = block_sym(nb->hi, nb->lo, cur);                   // exception rows read as code 0
            }
            const uint32_t mh = __ballot_sync(0xffffffffu, valid && (sym & 2u)), ml = __ballot_sync(0xffffffffu, valid && (sym & 1u));
            if (lane == 0) {                                             // t7, t8 go to their own array (32 bytes per block)
                uint32_t* p = reinterpret_cast<uint32_t*>(j <= 6 ? line + 32 + 16 * (j - 1) : tail + (size_t)b * 32 + 16 * (j - 7));
                p[half] = mh; p[2 + half] = ml;                          // hi plane = words 0,1 ; lo plane = words 2,3
            }
        }
        (void)steps;
    }
}

// pattern summaries of the sweep kernel (DevStrand::sum0/sum1): one thread per jump-table entry gathers the rows of its
// interval from the look-ahead lines (at most two lines for the <= 32 rows it keeps)
struct DevPlane {
    const unsigned char* lines; const unsigned char* tail;
    __device__ __forceinline__ uint64_t operator()(uint32_t b, uint32_t j, bool hi) const {
        if (j >= 7u) return __ldg(reinterpret_cast<const uint64_t*>(tail + ((size_t)b << 5)) + 2 * (j - 7) + (hi ? 0 : 1));
        const uint64_t* line = reinterpret_cast<const uint64_t*>(lines + ((size_t)b << 7));
        return __ldg(j == 0 ? line + (hi ? 2 : 3) : line + 4 + 2 * (j - 1) + (hi ? 0 : 1));
    }
};
__global__ void build_summary_kernel(const FtabEntry* __restrict__ tab, const unsigned char* __restrict__ lines, const unsigned char* __restrict__ tail,
                                     unsigned char* __restrict__ sum0, unsigned char* __restrict__ sum1, unsigned char* __restrict__ sum2, uint64_t n_entries) {
    DevPlane plane; plane.lines = lines; plane.tail = tail;
    for (uint64_t e = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x; e < n_entries; e += (uint64_t)gridDim.x * blockDim.x) {
        const FtabEntry t = tab[e];
        uint32_t s0[8], s1[8], s2[4];
        summary_build(plane, tail != nullptr, t.sp, t.width, s0, s1, s2);
        uint4* d0 = reinterpret_cast<uint4*>(sum0 + e * 32); uint4* d1 = reinterpret_cast<uint4*>(sum1 + e * 32);
        d0[0] = make_uint4(s0[0], s0[1], s0[2], s0[3]); d0[1] = make_uint4(s0[4], s0[5], s0[6], s0[7]);
        d1[0] = make_uint4(s1[0], s1[1], s1[2], s1[3]); d1[1] = make_uint4(s1[4], s1[5], s1[6], s1[7]);
        if (tail) *reinterpret_cast<uint4*>(sum2 + e * 16) = make_uint4(s2[0], s2[1], s2[2], s2[3]);
    }
}
cudaError_t launch_build_summary(const void* tab, const unsigned char* lines, const unsigned char* tail, unsigned char* sum0, unsigned char* sum1,
                                 unsigned char* sum2, uint64_t n_entries, cudaStream_t s) {
    build_summary_kernel<<<148 * 16, 256, 0, s>>>((const FtabEntry*)tab, lines, tail, sum0, sum1, sum2, n_entries);
    return cudaGetLastError();
}

cudaError_t launch_build_lookahead(const DevStrand& src, unsigned char* lines, unsigned char* tail, uint32_t n_blocks, cudaStream_t s) {
    build_lookahead_kernel<<<148 * 16, 256, 0, s>>>(src, lines, tail, n_blocks);
    return cudaGetLastError();
}

// ---------------------------------------------------------------------------------------------------------
// search, fast path: the same search specialised for what the headline workload is -- no bulges, one PAM pattern shared
// by all guides, ACGT-only guides, an index whose only non-ACGT BWT row is the sentinel.  Same tree, same matches, same
// keys as search_kernel; fewer instructions per node:
//   * node = 5 words (sp, ep, 64-bit key, task | mismatches << 24 | level << 27); the guide's packed symbols stay in a
//     register of the lane while it follows one path and are re-read only when the lane pops another guide's node
//   * strand-dependent constants (block base, C[], sentinel row) are selected from the parameter bank, no shared copy
//   * all four children are evaluated branch-free; siblings are compacted with two ballots (push count bit 0 / bit 1)
// ---------------------------------------------------------------------------------------------------------
template <int WARPS, int CAP, int MINB, bool LOOK, bool FUSED = false, bool EXC = false>
__global__ void __launch_bounds__(WARPS * 32, MINB) search_fast_kernel(SearchArgs a) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const uint32_t lane = threadIdx.x & 31u, warp = threadIdx.x >> 5;
    const uint32_t lt_mask = (1u << lane) - 1u;
    const uint32_t FULL = 0xffffffffu;
    uint64_t* r_key = reinterpret_cast<uint64_t*>(smem_raw + (size_t)warp * CAP * 20);
    uint32_t* r_sp = reinterpret_cast<uint32_t*>(r_key + CAP);
    uint32_t* r_ep = r_sp + CAP;
    uint32_t* r_tlm = r_ep + CAP;
    const uint32_t gwarp = blockIdx.x * WARPS + warp;
    const uint32_t scap = a.p.spill_cap;
    uint32_t* s_base = a.spill + (size_t)gwarp * scap * 6;          // sp | ep | tlm | key (u64)
    uint64_t* s_key = reinterpret_cast<uint64_t*>(s_base + 4 * (size_t)scap);

    uint32_t head = 0, count = 0, spill_count = 0;
    bool tasks_remain = true, has = false;
    uint32_t sp = 0, ep = 0, tlm = 0; uint64_t key = 0, q = 0;
    // k-mer jump table phase of the warp's current task (all warp-uniform)
    uint32_t cur_task = 0xFFFFFFFFu, cursor = 0, task_gidx = 0; uint64_t task_q = 0;
    unsigned long long n_nodes = 0, n_lookups = 0, n_spilled = 0;     // accumulated by lane 0 only
    const uint32_t M = a.p.M, plen = a.plen;
    uint32_t n_seeds = 0;
    if (a.seeds) { n_seeds = *a.n_seeds; if (n_seeds > a.seed_cap) n_seeds = a.seed_cap; }
    uint32_t iters = 0;
    uint64_t pol_keep, pol_stream;
    asm volatile("createpolicy.fractional.L2::evict_last.b64 %0, 1.0;" : "=l"(pol_keep));
    asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(pol_stream));

    for (;;) {
        if (++iters > a.max_iters) { if (lane == 0) atomicOr(a.error_flag, GSX_KERR_WATCHDOG); break; }
        uint32_t need_mask = __ballot_sync(FULL, !has);
        if (need_mask) {
            uint32_t n_need = __popc(need_mask);
            if (count < n_need && spill_count > 0) {
                uint32_t take = spill_count < 64u ? spill_count : 64u;
                for (uint32_t j = lane; j < take; j += 32) {
                    uint32_t i = spill_count - take + j, slot = (head + count + j) & (CAP - 1);
                    r_sp[slot] = s_base[i]; r_ep[slot] = s_base[scap + i]; r_tlm[slot] = s_base[2 * scap + i]; r_key[slot] = s_key[i];
                }
                __syncwarp();
                count += take; spill_count -= take;
            }
            if (count < n_need && tasks_remain && a.seeds) {
                // tasks are the level-L nodes the sweep kernel let through, 32 at a time (count < 32 <= CAP - 32: room)
                uint32_t t = 0;
                if (lane == 0) t = atomicAdd(a.task_counter, 32u);
                t = __shfl_sync(FULL, t, 0);
                if (t >= n_seeds) tasks_remain = false;
                else {
                    const uint32_t i = t + lane;
                    if (i < n_seeds) {
                        const SeedNode sn = a.seeds[i];
                        const uint32_t slot = (head + count + lane) & (CAP - 1);
                        r_sp[slot] = sn.sp; r_ep[slot] = sn.ep; r_tlm[slot] = sn.tlm;
                        r_key[slot] = ftab_key(sn.idx, __ldg(a.gq + ((sn.tlm & 0xFFFFFFu) >> 1)), sn.tlm >> 27);
                    }
                    __syncwarp();
                    count += (n_seeds - t < 32u) ? (n_seeds - t) : 32u;
                }
            } else if (count < n_need && cur_task == 0xFFFFFFFFu && tasks_remain) {
                uint32_t t = 0;
                if (lane == 0) t = atomicAdd(a.task_counter, 1u);
                t = __shfl_sync(FULL, t, 0);
                if (t >= a.p.n_tasks) tasks_remain = false;
                else if (!(a.skip && a.skip[t >> 1])) {
                    const uint64_t tq = __ldg(a.gq + (t >> 1));
                    const uint32_t L = (t & 1u) ? a.st[1].ftab_L : a.st[0].ftab_L;
                    if (L && (uint32_t)(tq >> 58) >= L && a.n_combos) {
                        // start the task from the k-mer jump table: exact index of its first L characters
                        cur_task = t; cursor = 0; task_q = tq;
                        task_gidx = ftab_exact_index(tq, L);
                    } else {
                        if (lane == 0) {
                            uint32_t slot = (head + count) & (CAP - 1);
                            r_sp[slot] = 0; r_ep[slot] = ((t & 1u) ? a.st[1].n : a.st[0].n) - 1u; r_tlm[slot] = t; r_key[slot] = 0;
                        }
                        __syncwarp();
                        count += 1;
                    }
                }
            }
            if (count < n_need && cur_task != 0xFFFFFFFFu) {
                // one table step: lane = one substitution combo over characters 2 .. L-1 = one 128-byte line of 16
                // beginnings; every beginning within the remaining budget whose interval is non-empty becomes a level-L node
                const bool s1t = (cur_task & 1u) != 0;
                const uint32_t L = s1t ? a.st[1].ftab_L : a.st[0].ftab_L;
                const FtabEntry* tab = reinterpret_cast<const FtabEntry*>(s1t ? a.st[1].ftab : a.st[0].ftab);
                const uint32_t ci = cursor + lane;
                const bool hasc = ci < a.n_combos;
                uint32_t idx = 0, j = 0; uint64_t kbase = 0;
                if (hasc) ftab_apply(__ldg(a.combos + ci), task_q, L, task_gidx, c_pow5, idx, kbase, j);
                const uint32_t budget = M - j;                       // combos hold at most M substitutions
                const uint32_t e0 = (uint32_t)task_q & 15u;
                {
                    const uint32_t lines_mask = __ballot_sync(FULL, hasc);
                    if (lane == 0) n_lookups += __popc(lines_mask);
                }
#pragma unroll 1
                for (uint32_t i = 0; i < 16; i++) {
                    const uint32_t e = (e0 + i) & 15u;               // the exact beginning first: it is valid for every combo
                    uint64_t k2 = kbase;
                    const uint32_t extra = ftab_beginning(e, task_q, L, c_pow5, k2);
                    const bool ok = hasc && extra <= budget;
                    FtabEntry t; t.sp = 0; t.width = 0;
                    if (ok) { const uint2 v = __ldg(reinterpret_cast<const uint2*>(tab + ((idx & ~15u) | e))); t.sp = v.x; t.width = v.y; }
                    const bool push = ok && t.width != 0;
                    const uint32_t pmask = __ballot_sync(FULL, push);
                    if (pmask) {
                        const uint32_t np = __popc(pmask);
                        if (count + np > (uint32_t)CAP) {
                            if (spill_count + 32u > scap) { if (lane == 0) atomicOr(a.error_flag, GSX_KERR_SPILL_OVERFLOW); }
                            else {
                                const uint32_t slot = (head + lane) & (CAP - 1), si = spill_count + lane;
                                s_base[si] = r_sp[slot]; s_base[scap + si] = r_ep[slot]; s_base[2 * scap + si] = r_tlm[slot]; s_key[si] = r_key[slot];
                                spill_count += 32u; if (lane == 0) n_spilled += 32;
                            }
                            __syncwarp();
                            head = (head + 32u) & (CAP - 1); count -= 32u;
                        }
                        if (push) {
                            const uint32_t w = (head + count + __popc(pmask & lt_mask)) & (CAP - 1);
                            r_sp[w] = t.sp; r_ep[w] = t.sp + t.width - 1u; r_key[w] = k2;
                            r_tlm[w] = cur_task | ((j + extra) << 24) | (L << 27);
                        }
                        __syncwarp();
                        count += np;
                    }
                    if (!__any_sync(FULL, hasc && budget != 0u)) break;      // no budget left anywhere: only the exact beginning counts
                }
                cursor += 32u;
                if (cursor >= a.n_combos) cur_task = 0xFFFFFFFFu;
            }
            uint32_t take = count < n_need ? count : n_need;
            uint32_t rank = __popc(need_mask & lt_mask);
            if (!has && rank < take) {
                uint32_t slot = (head + count - 1 - rank) & (CAP - 1);
                sp = r_sp[slot]; ep = r_ep[slot]; tlm = r_tlm[slot]; key = r_key[slot];
                q = __ldg(a.gq + ((tlm & 0xFFFFFFu) >> 1));
                has = true;
            }
            __syncwarp();
            count -= take;
        }
        const uint32_t act = __ballot_sync(FULL, has);
        if (act == 0) {
            if (count == 0 && spill_count == 0 && !tasks_remain && cur_task == 0xFFFFFFFFu) break;
            continue;
        }
        // ---- occurrence lookups -----------------------------------------------------------------------------
        const bool s1 = (tlm & 1u) != 0;
        uint32_t os0 = 0, os1 = 0, os2 = 0, os3 = 0, oe0 = 0, oe1 = 0, oe2 = 0, oe3 = 0;
        bool two = false;
        uint64_t phi[7] = {0, 0, 0, 0, 0, 0, 0}, plo[7] = {0, 0, 0, 0, 0, 0, 0};      // look-ahead planes (LOOK only)
        bool narrow = false; uint32_t vm = 15u;
        const uint32_t lvl = tlm >> 27, mm = (tlm >> 24) & 7u, qlen = (uint32_t)(q >> 58);
        if (has) {
            const OccBlock* blocks = s1 ? a.st[1].blocks : a.st[0].blocks;
            const uint32_t dollar = s1 ? a.st[1].exc_lo : a.st[0].exc_lo;
            const uint32_t e1 = ep + 1u, bs = sp >> 6, be = e1 >> 6;
            two = be != bs;
            Blk B0, B1;
            if (LOOK && be - bs <= 1u) {
                // all rows of the interval sit in one block or in two adjacent ones: read the block's own 128-byte line
                // (OccBlock + as many look-ahead planes as the remaining levels can use -- same line, so no further DRAM
                // traffic) and find the children that can still reach the final level; streaming in L2
                narrow = true;
                const unsigned char* lines = s1 ? a.st[1].lines : a.st[0].lines;
                const uint32_t left = qlen + plen - lvl;
                uint32_t r_lo = sp, r_hi = two ? 63u : ep;            // rows of the current part (low 6 bits matter)
                vm = 0;
#pragma unroll 1
                for (uint32_t part = 0; part < (two ? 2u : 1u); part++) {
                    const unsigned char* line = lines + ((size_t)(bs + part) << 7);
                    const Blk B = ld_block_hint(line, pol_stream);
                    if (part == 0) B0 = B;
                    B1 = B;
                    if (part == 1) { if ((e1 & 63u) == 0u) break; r_lo = 0; r_hi = ep; }   // ep is the last row of block bs
                    if (left > 1) { Blk P = ld_block_hint(line + 32, pol_stream);
                                    phi[1] = ((uint64_t)P.c1 << 32) | P.c0; plo[1] = ((uint64_t)P.c3 << 32) | P.c2; phi[2] = P.hi; plo[2] = P.lo; }
                    if (left > 3) { Blk P = ld_block_hint(line + 64, pol_stream);
                                    phi[3] = ((uint64_t)P.c1 << 32) | P.c0; plo[3] = ((uint64_t)P.c3 << 32) | P.c2; phi[4] = P.hi; plo[4] = P.lo; }
                    if (left > 5) { Blk P = ld_block_hint(line + 96, pol_stream);
                                    phi[5] = ((uint64_t)P.c1 << 32) | P.c0; plo[5] = ((uint64_t)P.c3 << 32) | P.c2; phi[6] = P.hi; plo[6] = P.lo; }
                    phi[0] = B.hi; plo[0] = B.lo;
                    vm |= viable_children(phi, plo, r_lo, r_hi, lvl, qlen, qlen + plen, q, a.pampack, M - mm);
                }
            } else {
                // packed blocks: 256 rows per line; the top of the tree is shared by all guides -> keep it in L2
                const uint64_t pol = (ep - sp >= a.pin_width) ? pol_keep : pol_stream;
                B0 = ld_block_hint(blocks + bs, pol);
                B1 = B0;
                if (two) B1 = ld_block_hint(blocks + be, pol);
            }
            {
                uint32_t r = sp & 63u; uint64_t mask = r ? (~0ull >> (64 - r)) : 0ull;
                uint64_t hi = B0.hi & mask, lo = B0.lo & mask;
                uint32_t t = __popcll(hi & lo), g = __popcll(hi) - t, c = __popcll(lo) - t;
                uint32_t aa = r - t - g - c - ((dollar >= sp - r && dollar < sp) ? 1u : 0u);
                if constexpr (EXC) aa = r - t - g - c - exc_before(s1 ? a.exc_map[1] : a.exc_map[0], s1 ? a.st[1].exc_rows : a.st[0].exc_rows, s1 ? a.st[1].n_exc : a.st[0].n_exc, sp);
                os0 = B0.c0 + aa; os1 = B0.c1 + c; os2 = B0.c2 + g; os3 = B0.c3 + t;
            }
            {
                uint32_t r = e1 & 63u; uint64_t mask = r ? (~0ull >> (64 - r)) : 0ull;
                uint64_t hi = B1.hi & mask, lo = B1.lo & mask;
                uint32_t t = __popcll(hi & lo), g = __popcll(hi) - t, c = __popcll(lo) - t;
                uint32_t aa = r - t - g - c - ((dollar >= e1 - r && dollar < e1) ? 1u : 0u);
                if constexpr (EXC) aa = r - t - g - c - exc_before(s1 ? a.exc_map[1] : a.exc_map[0], s1 ? a.st[1].exc_rows : a.st[0].exc_rows, s1 ? a.st[1].n_exc : a.st[0].n_exc, e1);
                oe0 = B1.c0 + aa; oe1 = B1.c1 + c; oe2 = B1.c2 + g; oe3 = B1.c3 + t;
            }
        }
        if (lane == 0) { n_nodes += __popc(act); }
        {
            uint32_t two_mask = __ballot_sync(FULL, has && two);
            if (lane == 0) n_lookups += __popc(act) + __popc(two_mask);
        }
        // ---- children (branch-free) ---------------------------------------------------------------------------
        const bool in_proto = lvl < qlen;
        const uint32_t c = in_proto ? ((uint32_t)(q >> (2u * lvl)) & 3u) : ((a.pampack >> (3u * (lvl - qlen))) & 7u);
        // symbols other than c that may be consumed: all four within the mismatch budget or under a PAM wildcard, the members of a
        // class PAM character (code 6, whose members are in pammask), none otherwise
        const uint32_t allow = in_proto ? (mm < M ? 15u : 0u) : (c == 4u ? 15u : ((a.pammask >> (4u * (lvl - qlen))) & 15u));
        const bool final_lvl = (lvl + 1u == qlen + plen);
        const uint32_t w0 = oe0 - os0, w1 = oe1 - os1, w2 = oe2 - os2, w3 = oe3 - os3;
        bool v0 = has && w0 && (c == 0u || (allow & 1u)), v1 = has && w1 && (c == 1u || (allow & 2u));
        bool v2 = has && w2 && (c == 2u || (allow & 4u)), v3 = has && w3 && (c == 3u || (allow & 8u));
        if (LOOK && narrow) {        // drop children that cannot survive the next (up to) seven characters
            v0 = v0 && (vm & 1u); v1 = v1 && (vm & 2u); v2 = v2 && (vm & 4u); v3 = v3 && (vm & 8u);
        }
        const uint32_t C0 = s1 ? a.st[1].C[0] : a.st[0].C[0], C1 = s1 ? a.st[1].C[1] : a.st[0].C[1];
        const uint32_t C2 = s1 ? a.st[1].C[2] : a.st[0].C[2], C3 = s1 ? a.st[1].C[3] : a.st[0].C[3];
        const uint64_t key5 = key * 5ull;
        const uint32_t tlm1 = tlm + (1u << 27);
        const uint32_t mis = in_proto ? (1u << 24) : 0u;                 // a protospacer child other than c costs one mismatch
        // child s: sp' = Cs + os_s, ep' = sp' + w_s - 1, key' = key5 + digit_s, tlm' = tlm1 + (s != c ? mis : 0)
#define GSX_CH_SP(s) (C##s + os##s)
#define GSX_CH_DIGIT(s) (in_proto ? (c == (s) ? 0u : 1u + (s)) : ((s) < 3 ? (uint32_t)(s) : 4u))
#define GSX_CH_TLM(s) (tlm1 + (c == (s) ? 0u : mis))
        // ---- finished alignments (rare) ---------------------------------------------------------------------------
        if (__any_sync(FULL, final_lvl && (v0 || v1 || v2 || v3))) {
#define GSX_EMIT(s)                                                                                                   \
            {                                                                                                         \
                const bool e = final_lvl && v##s && (!FUSED || fused_pam_ok(key5 + GSX_CH_DIGIT(s), plen, a.fused_pams, a.n_fused, a.fused_masks)); \
                const uint32_t emask = __ballot_sync(FULL, e);                                                         \
                if (emask) {                                                                                          \
                    if (a.p.counting) {                                                                               \
                        if (e) atomicAdd(a.guide_count + ((tlm & 0xFFFFFFu) >> 1), (unsigned long long)w##s);          \
                    } else {                                                                                          \
                        uint32_t base = 0; const int leader = __ffs(emask) - 1;                                       \
                        if ((int)lane == leader) base = atomicAdd(a.match_count, (uint32_t)__popc(emask));            \
                        base = __shfl_sync(FULL, base, leader);                                                       \
                        if (e) {                                                                                      \
                            const uint32_t slot = base + __popc(emask & lt_mask);                                     \
                            if (slot < a.p.match_cap) {                                                               \
                                MatchRec m; m.key_hi = 0; m.key_lo = key5 + GSX_CH_DIGIT(s); m.task = tlm & 0xFFFFFFu;  \
                                m.sp = GSX_CH_SP(s); m.width = w##s;                                                   \
                                m.info = ((GSX_CH_TLM(s) >> 24) & 7u) | ((lvl + 1u) << 24);                            \
                                a.matches[slot] = m;                                                                  \
                                atomicAdd(a.guide_nmatch + ((tlm & 0xFFFFFFu) >> 1), 1u);                              \
                            } else atomicOr(a.error_flag, GSX_KERR_MATCH_OVERFLOW);                                   \
                        }                                                                                             \
                    }                                                                                                 \
                }                                                                                                     \
            }
            GSX_EMIT(0) GSX_EMIT(1) GSX_EMIT(2) GSX_EMIT(3)
#undef GSX_EMIT
        }
        // ---- genome N under a PAM wildcard (EXC only): the reference's PAM stage tries the literal character first, so a
        //      pattern N also consumes a genome N (index.hpp:139-150); that child lives in the N range of the index ----------
        if constexpr (EXC) {
            const uint32_t nn = s1 ? a.st[1].n_nrows : a.st[0].n_nrows;
            const bool litn = has && !in_proto && c == 4u && nn != 0u;
            if (__any_sync(FULL, litn)) {
                uint32_t o_s = 0, wN = 0;
                if (litn) {
                    const uint32_t* nr = s1 ? a.st[1].n_rows : a.st[0].n_rows;
                    o_s = lower_bound_u32(nr, nn, sp); wN = lower_bound_u32(nr, nn, ep + 1u) - o_s;
                }
                const bool vN = litn && wN != 0u;
                const uint32_t spN = (s1 ? a.st[1].C[4] : a.st[0].C[4]) + o_s;
                const bool eN = vN && final_lvl && (!FUSED || fused_pam_ok(key5 + 3u, plen, a.fused_pams, a.n_fused, a.fused_masks));
                const uint32_t emask = __ballot_sync(FULL, eN);
                if (emask) {
                    if (a.p.counting) { if (eN) atomicAdd(a.guide_count + ((tlm & 0xFFFFFFu) >> 1), (unsigned long long)wN); }
                    else {
                        uint32_t base = 0; const int leader = __ffs(emask) - 1;
                        if ((int)lane == leader) base = atomicAdd(a.match_count, (uint32_t)__popc(emask));
                        base = __shfl_sync(FULL, base, leader);
                        if (eN) {
                            const uint32_t slot = base + __popc(emask & lt_mask);
                            if (slot < a.p.match_cap) {
                                MatchRec m; m.key_hi = 0; m.key_lo = key5 + 3u; m.task = tlm & 0xFFFFFFu; m.sp = spN; m.width = wN;
                                m.info = ((tlm >> 24) & 7u) | ((lvl + 1u) << 24);
                                a.matches[slot] = m;
                                atomicAdd(a.guide_nmatch + ((tlm & 0xFFFFFFu) >> 1), 1u);
                            } else atomicOr(a.error_flag, GSX_KERR_MATCH_OVERFLOW);
                        }
                    }
                }
                const bool pN = vN && !final_lvl;
                const uint32_t pmask = __ballot_sync(FULL, pN);
                if (pmask) {
                    const uint32_t np = __popc(pmask);
                    while (count + np > (uint32_t)CAP) {
                        if (spill_count + 32u > scap) { if (lane == 0) atomicOr(a.error_flag, GSX_KERR_SPILL_OVERFLOW); }
                        else {
                            const uint32_t slot = (head + lane) & (CAP - 1), i = spill_count + lane;
                            s_base[i] = r_sp[slot]; s_base[scap + i] = r_ep[slot]; s_base[2 * scap + i] = r_tlm[slot]; s_key[i] = r_key[slot];
                            spill_count += 32u; if (lane == 0) n_spilled += 32;
                        }
                        __syncwarp();
                        head = (head + 32u) & (CAP - 1); count -= 32u;
                    }
                    if (pN) {
                        const uint32_t w = (head + count + __popc(pmask & lt_mask)) & (CAP - 1);
                        r_sp[w] = spN; r_ep[w] = spN + wN - 1u; r_tlm[w] = tlm1; r_key[w] = key5 + 3u;
                    }
                    __syncwarp();
                    count += np;
                }
            }
        }
        // ---- keep one child in registers, push the siblings ---------------------------------------------------------
        const uint32_t nvalid = final_lvl ? 0u : ((uint32_t)v0 + (uint32_t)v1 + (uint32_t)v2 + (uint32_t)v3);
        const uint32_t pushes = nvalid ? nvalid - 1u : 0u;
        const uint32_t b0 = __ballot_sync(FULL, pushes & 1u), b1 = __ballot_sync(FULL, pushes & 2u);
        const uint32_t total = __popc(b0) + 2u * __popc(b1);
        if (total) {
            while (count + total > (uint32_t)CAP) {                       // spill the 32 oldest nodes (total can reach 96)
                if (spill_count + 32u > scap) { if (lane == 0) atomicOr(a.error_flag, GSX_KERR_SPILL_OVERFLOW); }
                else {
                    const uint32_t slot = (head + lane) & (CAP - 1), i = spill_count + lane;
                    s_base[i] = r_sp[slot]; s_base[scap + i] = r_ep[slot]; s_base[2 * scap + i] = r_tlm[slot]; s_key[i] = r_key[slot];
                    spill_count += 32u; if (lane == 0) n_spilled += 32;
                }
                __syncwarp();
                head = (head + 32u) & (CAP - 1); count -= 32u;
            }
        }
        uint32_t slot = head + count + __popc(b0 & lt_mask) + 2u * __popc(b1 & lt_mask);
        bool kept = false;
        uint32_t nsp = sp, nep = ep, ntlm = tlm; uint64_t nkey = key;
#define GSX_CHILD(s)                                                                                                  \
        if (v##s && !final_lvl) {                                                                                     \
            const uint32_t csp = GSX_CH_SP(s), cep = csp + w##s - 1u, ctlm = GSX_CH_TLM(s);                             \
            const uint64_t ckey = key5 + GSX_CH_DIGIT(s);                                                              \
            if (!kept) { kept = true; nsp = csp; nep = cep; ntlm = ctlm; nkey = ckey; }                                 \
            else { const uint32_t w = slot & (CAP - 1); r_sp[w] = csp; r_ep[w] = cep; r_tlm[w] = ctlm; r_key[w] = ckey; slot++; } \
        }
        GSX_CHILD(0) GSX_CHILD(1) GSX_CHILD(2) GSX_CHILD(3)
#undef GSX_CHILD
#undef GSX_CH_SP
#undef GSX_CH_DIGIT
#undef GSX_CH_TLM
        if (total) { __syncwarp(); count += total; }
        has = kept; sp = nsp; ep = nep; tlm = ntlm; key = nkey;
    }
    if (lane == 0) { atomicAdd(a.stats + 0, n_nodes); atomicAdd(a.stats + 1, n_lookups); atomicAdd(a.stats + 2, n_spilled); atomicAdd(a.stats + 7, n_lookups); }
}

template <int WARPS, int CAP, int MINB, bool LOOK, bool FUSED = false, bool EXC = false>
static cudaError_t launch_fast_t(const SearchArgs& a, int sm_count, cudaStream_t s) {
    size_t smem = (size_t)WARPS * CAP * 20;
    auto k = search_fast_kernel<WARPS, CAP, MINB, LOOK, FUSED, EXC>;
    cudaError_t e = cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
    k<<<sm_count * MINB, WARPS * 32, smem, s>>>(a);
    return cudaGetLastError();
}

#define GSX_FAST_VARIANTS(X) \
    X(0, 8, 256, 4) /* 1024 thr/SM, 160 KB smem */ \
    X(1, 8, 256, 3) /* 768 thr/SM */ \
    X(2, 8, 128, 6) /* 1536 thr/SM */ \
    X(3, 8, 128, 8) /* 2048 thr/SM (<= 32 regs) */ \
    X(4, 8, 256, 5) /* 1280 thr/SM, 200 KB smem */

cudaError_t launch_search_fast(const SearchArgs& a, int variant, int sm_count, cudaStream_t s) {
    const bool look = a.st[0].lines != nullptr && a.st[1].lines != nullptr;
    if (a.n_fused || a.exc) {         // several PAMs in one pass / genome with N: the default occupancy variant only
        if (variant != 1 || (a.n_fused && a.p.counting) || (a.exc && (!a.exc_map[0] || !a.exc_map[1]))) return cudaErrorInvalidValue;
        if (a.exc) {
            if (a.n_fused) return look ? launch_fast_t<8, 256, 3, true, true, true>(a, sm_count, s) : launch_fast_t<8, 256, 3, false, true, true>(a, sm_count, s);
            return look ? launch_fast_t<8, 256, 3, true, false, true>(a, sm_count, s) : launch_fast_t<8, 256, 3, false, false, true>(a, sm_count, s);
        }
        return look ? launch_fast_t<8, 256, 3, true, true>(a, sm_count, s) : launch_fast_t<8, 256, 3, false, true>(a, sm_count, s);
    }
#define X(V, WARPS, CAP, MINB) if (variant == V) return look ? launch_fast_t<WARPS, CAP, MINB, true>(a, sm_count, s) : launch_fast_t<WARPS, CAP, MINB, false>(a, sm_count, s);
    GSX_FAST_VARIANTS(X)
#undef X
    return cudaErrorInvalidValue;
}
int search_fast_grid_warps(int variant, int sm_count) {
#define X(V, WARPS, CAP, MINB) if (variant == V) return sm_count * MINB * WARPS;
    GSX_FAST_VARIANTS(X)
#undef X
    return -1;
}

// ---------------------------------------------------------------------------------------------------------
// search, slice-major front end (large batches on the fast path).  After the jump table and the look-ahead planes, what is
// left of the search is one question per candidate pattern -- "does any row of this 14-mer's interval continue with the
// guide's next characters and a PAM?" -- asked ~10.7 k times per guide and strand (3.1 Gb, m = 3) and answered by one
// 32-byte pattern summary each (DevStrand::sum0; gsx_core.h summary_eval*).  Guide by guide those reads are uniformly
// scattered over 17 GB: every one a DRAM line fetch and a TLB miss.  But a batch of 50-200 k guides wants every summary
// line several times.  The sweep kernel therefore turns the loops inside out: the grid walks the index slice by slice
// (a slice = all patterns sharing their last `sb` consumed characters = a contiguous 1/4^sb of the table and of the
// summaries, L2-resident), and inside a slice it visits every guide of the batch and tests that guide's patterns that
// fall into the slice (xor table of substitution choices, gsx_core.h sweep_pattern).  Survivors (~1 %) go to a queue;
// search_fast_kernel continues from them (a.seeds).
// Work unit = (strand, slice, block of 32 guides), handed out slice-major through one counter, so that all warps work on
// the same few slices at any time.  Inside a unit: (1) one lane-parallel step for the guides whose only pattern in the
// slice is the unsubstituted one, (2) the guides with budget left one at a time, all 32 lanes on the same guide -- its
// filter masks in registers, the xor table read with unit stride from shared memory, two summary loads in flight per lane.
// ---------------------------------------------------------------------------------------------------------
static inline int grid_for_n(uint32_t n, int threads, int cap) { long b = ((long)n + threads - 1) / threads; if (b < 1) b = 1; if (b > cap) b = cap; return (int)b; }

struct DevSummaryLoader {
    const unsigned char* sum0; const unsigned char* sum1;
    __device__ __forceinline__ void operator()(uint32_t stage, uint32_t idx, uint32_t w[8]) const {
        asm volatile("ld.global.nc.v8.b32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"                                       // LDG.E.256
                     : "=r"(w[0]), "=r"(w[1]), "=r"(w[2]), "=r"(w[3]), "=r"(w[4]), "=r"(w[5]), "=r"(w[6]), "=r"(w[7])
                     : "l"((stage ? sum1 : sum0) + ((size_t)idx << 5)));
    }
};
__device__ __forceinline__ void load_tail(const unsigned char* sum2, uint32_t idx, uint32_t t[4]) {
    const uint4 v = __ldg(reinterpret_cast<const uint4*>(sum2 + ((size_t)idx << 4)));
    t[0] = v.x; t[1] = v.y; t[2] = v.z; t[3] = v.w;
}

struct SweepStats { uint32_t nodes, lookups, sectors; };  // nodes, lookups: per lane; sectors (32-byte summary loads issued): warp-uniform

// per-warp buffer of nodes whose first 16 rows are dead but which have more (gsx_core.h summary_eval, stage 1): 64 records
// in shared memory
//   idx    table index of the pattern (sp, ep are read from the jump table if the node survives)
//   codes  plane codes of its guide
//   tlm    task | mismatches << 24 | remaining budget << 27
struct ContBuf {
    uint32_t* idx; uint32_t* codes; uint32_t* tlm; uint32_t* codes2;
    uint32_t count;                                                  // warp-uniform
};

__device__ __forceinline__ void cont_push(ContBuf& cb, uint32_t lane, bool want, uint32_t idx, uint32_t codes, uint32_t codes2, uint32_t tlm) {
    const uint32_t m = __ballot_sync(0xffffffffu, want);
    if (want) {
        const uint32_t slot = cb.count + __popc(m & ((1u << lane) - 1u));
        cb.idx[slot] = idx; cb.codes[slot] = codes; cb.tlm[slot] = tlm; cb.codes2[slot] = codes2;
    }
    cb.count += __popc(m);
    __syncwarp();
}

// surviving level-L node -> seed queue; sp / ep come from the jump table (only survivors ever read it)
__device__ __forceinline__ void sweep_emit(const SweepArgs& a, uint32_t lane, bool emit, uint32_t idx, uint32_t tlm, SweepStats& st) {
    const uint32_t emask = __ballot_sync(0xffffffffu, emit);
    if (!emask) return;
    uint32_t qbase = 0; const int leader = __ffs(emask) - 1;
    if ((int)lane == leader) qbase = atomicAdd(a.queue_count, (uint32_t)__popc(emask));
    qbase = __shfl_sync(0xffffffffu, qbase, leader);
    if (emit) {
        const uint32_t slot = qbase + __popc(emask & ((1u << lane) - 1u));
        if (slot < a.queue_cap) {
            const FtabEntry* tab = reinterpret_cast<const FtabEntry*>((tlm & 1u) ? a.st[1].ftab : a.st[0].ftab);
            const uint2 e = __ldg(reinterpret_cast<const uint2*>(tab + idx));
            SeedNode sn; sn.sp = e.x; sn.ep = e.x + e.y - 1u; sn.idx = idx; sn.tlm = (tlm & 0x07FFFFFFu) | (a.plan.L << 27);
            a.queue[slot] = sn;
        } else atomicOr(a.error_flag, GSX_KERR_QUEUE_OVERFLOW);
    }
}

// drain up to 32 parked nodes: rows 16..31 of their intervals, all lanes busy
template <int NB>
__device__ __forceinline__ void cont_process(const SweepArgs& a, ContBuf& cb, uint32_t lane, SweepStats& st) {
    const uint32_t n = cb.count < 32u ? cb.count : 32u;
    const bool mine = lane < n;
    uint32_t idx = 0, codes = 0, codes2 = 0x77u, tlm = 0; uint32_t u[NB];
#pragma unroll
    for (int r = 0; r < NB; r++) u[r] = 0;
    if (mine) { const uint32_t slot = cb.count - n + lane; idx = cb.idx[slot]; codes = cb.codes[slot]; tlm = cb.tlm[slot]; codes2 = cb.codes2[slot]; }
    __syncwarp();
    cb.count -= n; st.sectors += n;
    if (mine) {
        DevSummaryLoader ld; ld.sum0 = nullptr; ld.sum1 = (tlm & 1u) ? a.st[1].sum1 : a.st[0].sum1;
        summary_eval<NB>(ld, 1u, idx, codes, (tlm >> 27) & 7u, u);
        const unsigned char* sum2 = (tlm & 1u) ? a.st[1].sum2 : a.st[0].sum2;
        if (u[0] && sum2 && sweep_has_tail(codes2)) { uint32_t t[4]; load_tail(sum2, idx, t); summary_tail<NB>(t, 1u, codes2, u); }
    }
    sweep_emit(a, lane, mine && u[0] != 0u, idx, tlm, st);
}

// per-guide constants of the sweep (20 words): written once per call by sweep_guides_kernel, copied to shared memory by
// each work unit, read back by whichever lanes end up working on that guide's patterns
//   [0..6] A, [7..13] X, [14] pflags (gsx_core.h summary_masks)   [15] low 2(L-sb) bits of the packed guide
//   [16] plane codes of levels L .. L+6   [17] of levels L+7, L+8
constexpr int CB_SLOTS = 64;          // parked nodes per warp: drained below 32 before every step, which adds at most 32
constexpr int XT_SMEM = kSweepXtabShared;
constexpr int GT_WORDS = 20, GT_QLOW = 15, GT_CODES = 16, GT_CODES2 = 17, GT_FMASK = 18, GT_SHAPE = 19;      // [18] must-match positions of an edited guide (index mask)

__global__ void sweep_guides_kernel(SweepArgs a, uint32_t* __restrict__ gtab) {
    for (uint32_t g = blockIdx.x * blockDim.x + threadIdx.x; g < a.n_guides; g += gridDim.x * blockDim.x) {
        const uint64_t q = a.gq[g];
        uint32_t t[GT_WORDS];
        const uint32_t codes = sweep_codes(q, a.plan.L, a.plen, a.pampack);
        summary_masks(codes, t);
        t[GT_QLOW] = (uint32_t)q & ((1u << (2u * (a.plan.L - a.plan.sb))) - 1u);
        t[GT_CODES] = codes; t[GT_CODES2] = sweep_codes2(q, a.plan.L, a.plen, a.pampack); t[GT_FMASK] = a.fmask ? a.fmask[g] : 0u; t[GT_SHAPE] = (uint32_t)sweep_shape_of(codes);
        uint4* dst = reinterpret_cast<uint4*>(gtab + (size_t)g * GT_WORDS);
        for (int k = 0; k < GT_WORDS / 4; k++) dst[k] = make_uint4(t[4 * k], t[4 * k + 1], t[4 * k + 2], t[4 * k + 3]);
    }
}

__device__ __forceinline__ void sweep_load(const unsigned char* sum0, uint32_t idx, uint32_t w[8], uint32_t mode = 0) {
    if (mode == 1)
        asm volatile("ld.global.nc.L1::no_allocate.v8.b32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
                     : "=r"(w[0]), "=r"(w[1]), "=r"(w[2]), "=r"(w[3]), "=r"(w[4]), "=r"(w[5]), "=r"(w[6]), "=r"(w[7])
                     : "l"(sum0 + ((size_t)idx << 5)));
    else if (mode == 2)
        asm volatile("ld.global.cg.v8.b32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
                     : "=r"(w[0]), "=r"(w[1]), "=r"(w[2]), "=r"(w[3]), "=r"(w[4]), "=r"(w[5]), "=r"(w[6]), "=r"(w[7])
                     : "l"(sum0 + ((size_t)idx << 5)));
    else
        asm volatile("ld.global.nc.v8.b32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"                                       // LDG.E.256
                     : "=r"(w[0]), "=r"(w[1]), "=r"(w[2]), "=r"(w[3]), "=r"(w[4]), "=r"(w[5]), "=r"(w[6]), "=r"(w[7])
                     : "l"(sum0 + ((size_t)idx << 5)));
}
// one pattern of one guide against its summary sector; EXACT = no budget left (one row mask)
template <bool EXACT, int NB>
__device__ __forceinline__ void sweep_judge(const uint32_t w[8], const unsigned char* sum2, uint32_t idx, uint32_t qlow, const uint32_t gm[15],
                                            uint32_t codes2, uint32_t budget, bool& emit, bool& park, SweepStats& st) {
    uint32_t alive;
    const bool tail = sum2 && sweep_has_tail(codes2) && !(w[0] & SUM_WIDE32);
    if (EXACT) {
        alive = summary_eval_exact(w, gm);
        if (alive && tail) { uint32_t t[4], v[1] = {alive}; load_tail(sum2, idx, t); summary_tail<1>(t, 0u, codes2, v); alive = v[0]; }
    } else {
        uint32_t u[NB]; summary_eval_masks<NB>(w, gm, budget, u);
        if (u[0] && tail) { uint32_t t[4]; load_tail(sum2, idx, t); summary_tail<NB>(t, 0u, codes2, u); }
        alive = u[0];
    }
    if (((idx ^ qlow) & 15u) == 0u) st.lookups++;                             // one table line per 16 beginnings
    if (w[0] & 0xFFFFu) {
        st.nodes++; st.lookups += (w[0] & SUM_TWO_BLOCKS) ? 2u : 1u;
        emit = alive != 0u || (w[0] & SUM_WIDE32) != 0u;                      // (more than 32 rows: not summarised, the tree search takes it)
        park = !emit && (w[0] & SUM_WIDE16) != 0u;
    }
}

// all patterns of ONE guide (lane `o` of the unit) in one pass, 32 per step: the guide's masks sit in registers, the xor
// table (shared memory when it fits) is read with unit stride, nothing is looked up per lane but the summary sector itself.
// (Two summary loads in flight per lane were tried and lost to register pressure: profiles/r01x_*.)
template <bool ZERO, int NB, bool FORCED = false>
__device__ __forceinline__ void sweep_run(const SweepArgs& a, const SweepPlan& pl, ContBuf& cb, const uint32_t* sg, const uint32_t* xtab, uint32_t lane,
                                          uint32_t strand, uint32_t hi_bits, uint32_t guide, uint32_t o, uint32_t B, SweepStats& st) {
    const uint32_t M = a.M, n = pl.xcnt[ZERO ? 1 : 0][B];
    if (n == 0u) return;
    const uint32_t* xt = xtab + pl.xoff[ZERO ? 1 : 0][B];
    const unsigned char* sum0 = strand ? a.st[1].sum0 : a.st[0].sum0;
    const uint4* gp = reinterpret_cast<const uint4*>(sg + o * GT_WORDS);       // same address in every lane: broadcast
    const uint4 g0 = gp[0], g1 = gp[1], g2 = gp[2], g3 = gp[3];
    const uint32_t gm[15] = {g0.x, g0.y, g0.z, g0.w, g1.x, g1.y, g1.z, g1.w, g2.x, g2.y, g2.z, g2.w, g3.x, g3.y, g3.z};
    const uint32_t qlow = g3.w, codes = sg[o * GT_WORDS + GT_CODES], codes2 = sg[o * GT_WORDS + GT_CODES2];
    const unsigned char* sum2 = strand ? a.st[1].sum2 : a.st[0].sum2;
    const uint32_t tl = (guide << 1) | strand;
    uint32_t fm = 0;
    if constexpr (FORCED) fm = sg[o * GT_WORDS + GT_FMASK] & 0x0FFFFFFFu;      // patterns that substitute a must-match position are skipped
    if constexpr (!FORCED) st.sectors += n;
    for (uint32_t base = 0; base < n; base += 32u) {
        while (cb.count >= 32u) cont_process<NB>(a, cb, lane, st);
        const uint32_t t = base + lane;
        bool emit = false, park = false; uint32_t idx = 0, mm = M;
        bool live = t < n;
        if constexpr (FORCED) { if (live && (xt[t] & fm)) live = false; st.sectors += __popc(__ballot_sync(0xffffffffu, live)); }
        if (live) {
            const uint32_t xw = xt[t];
            idx = hi_bits | (qlow ^ (xw & 0x0FFFFFFFu));
            if (!ZERO) mm = M - B + (xw >> 28);                               // (pass 1 always ends at M)
            uint32_t w[8];
            sweep_load(sum0, idx, w, a.load_mode);
            sweep_judge<ZERO, NB>(w, sum2, idx, qlow, gm, codes2, M - mm, emit, park, st);
        }
        const uint32_t tlm = tl | (mm << 24) | ((M - mm) << 27);
        sweep_emit(a, lane, emit, idx, tlm, st);
        cont_push(cb, lane, park, idx, codes, codes2, tlm);
    }
}

template <int WARPS, int MINB, int NB, bool FORCED = false>
__global__ void __launch_bounds__(WARPS * 32, MINB) sweep_kernel(SweepArgs a) {
    __shared__ SweepPlan s_plan;
    __shared__ uint32_t s_c32[WARPS][4][CB_SLOTS];
    __shared__ __align__(16) uint32_t s_g[WARPS][33 * GT_WORDS];
    __shared__ uint32_t s_xtab[XT_SMEM];                  // the xor table, when it fits (it does for up to 3 mismatches)
    for (int i = threadIdx.x; i < (int)(sizeof(SweepPlan) / 4); i += blockDim.x)
        reinterpret_cast<uint32_t*>(&s_plan)[i] = reinterpret_cast<const uint32_t*>(&a.plan)[i];
    const bool xt_shared = a.n_xtab <= (uint32_t)XT_SMEM;
    if (xt_shared) for (uint32_t i = threadIdx.x; i < a.n_xtab; i += blockDim.x) s_xtab[i] = a.xtab[i];
    const uint32_t* xtab = xt_shared ? s_xtab : a.xtab;
    __syncthreads();
    const uint32_t lane = threadIdx.x & 31u, warp = threadIdx.x >> 5, FULL = 0xffffffffu;
    ContBuf cb;
    cb.idx = s_c32[warp][0]; cb.codes = s_c32[warp][1]; cb.tlm = s_c32[warp][2]; cb.codes2 = s_c32[warp][3]; cb.count = 0;
    uint32_t* sg = s_g[warp];
    const uint32_t L = s_plan.L, sb = s_plan.sb, M = a.M;
    const uint32_t n_slices = 1u << (2u * sb), n_gb = (a.n_guides + 31u) >> 5;
    const uint64_t items_per_strand = (uint64_t)n_slices * n_gb, n_items = 2ull * items_per_strand;
    SweepStats st = {0, 0, 0};
    for (;;) {
        uint32_t item = 0;
        if (lane == 0) item = atomicAdd(a.item_counter, 1u);
        item = __shfl_sync(FULL, item, 0);
        if ((uint64_t)item >= n_items) break;
        const uint32_t strand = (uint64_t)item >= items_per_strand ? 1u : 0u;
        const uint32_t rem = item - (strand ? (uint32_t)items_per_strand : 0u);
        const uint32_t beta = rem / n_gb, gb = rem - beta * n_gb;
        const uint32_t g = gb * 32u + lane;
        const bool valid = g < a.n_guides && !(a.skip && a.skip[g]);
        int B = -1;
        __syncwarp();
        if (valid) {                                                           // this guide's row of the table -> shared memory
            const uint4* src = reinterpret_cast<const uint4*>(a.gtab + (size_t)g * GT_WORDS);
            uint4* dst = reinterpret_cast<uint4*>(sg + lane * GT_WORDS);
            const uint4 v0 = __ldg(src), v1 = __ldg(src + 1), v2 = __ldg(src + 2), v3 = __ldg(src + 3), v4 = __ldg(src + 4);
            dst[0] = v0; dst[1] = v1; dst[2] = v2; dst[3] = v3; dst[4] = v4;
            const uint32_t h = sweep_slice_distance(__ldg(a.gq + g), L, sb, beta);
            if (h <= M) B = (int)(M - h);
            if constexpr (FORCED) {      // the slice substitutes a must-match position of this (edited) guide: nothing to do here
                const uint32_t top = (uint32_t)(__ldg(a.gq + g) >> (2u * (L - sb))) & ((1u << (2u * sb)) - 1u);
                if ((top ^ beta) & (v4.z >> (2u * (L - sb)))) B = -1;
            }
        }
        __syncwarp();
        const uint32_t hi_bits = beta << (2u * (L - sb));
        // (1) guides whose only pattern in this slice is the unsubstituted one (budget 0), and the unsubstituted pattern of
        //     the guides with budget 1: one pattern per lane, each lane with its own guide's masks
        {
            // (the previous unit may have left up to 63 parked nodes and this step can park 32 more: make room first -- batches
            // of near-identical guides, e.g. the edited forms of one guide, park in every lane at once)
            while (cb.count >= 32u) cont_process<NB>(a, cb, lane, st);
            bool emit = false, park = false; uint32_t idx = 0, codes = 0, codes2 = 0x77u;
            st.sectors += __popc(__ballot_sync(FULL, B == 0 || B == 1));
            if (B == 0 || B == 1) {
                const uint4* gp = reinterpret_cast<const uint4*>(sg + lane * GT_WORDS);
                const uint4 g0 = gp[0], g1 = gp[1], g2 = gp[2], g3 = gp[3];
                const uint32_t gm[15] = {g0.x, g0.y, g0.z, g0.w, g1.x, g1.y, g1.z, g1.w, g2.x, g2.y, g2.z, g2.w, g3.x, g3.y, g3.z};
                codes = sg[lane * GT_WORDS + GT_CODES]; codes2 = sg[lane * GT_WORDS + GT_CODES2];
                idx = hi_bits | g3.w;
                uint32_t w[8];
                sweep_load(strand ? a.st[1].sum0 : a.st[0].sum0, idx, w);
                sweep_judge<false, NB>(w, strand ? a.st[1].sum2 : a.st[0].sum2, idx, g3.w, gm, codes2, (uint32_t)B, emit, park, st);
            }
            const uint32_t tlm = ((g << 1) | strand) | ((M - (uint32_t)(B > 0 ? B : 0)) << 24) | ((uint32_t)(B > 0 ? B : 0) << 27);
            sweep_emit(a, lane, emit, idx, tlm, st);
            cont_push(cb, lane, park, idx, codes, codes2, tlm);
        }
        // (2) guides with budget left after the slice characters, one at a time: first the patterns that use the budget up
        //     (most of them, cheapest arithmetic), then -- from budget 2 on -- the ones that keep some
        uint32_t todo = __ballot_sync(FULL, B >= 1);
        while (todo) {
            const uint32_t o = (uint32_t)__ffs(todo) - 1u; todo &= todo - 1u;
            const uint32_t Bo = (uint32_t)__shfl_sync(FULL, B, o);
            sweep_run<true, NB, FORCED>(a, s_plan, cb, sg, xtab, lane, strand, hi_bits, gb * 32u + o, o, Bo, st);
            if (Bo >= 2u) sweep_run<false, NB, FORCED>(a, s_plan, cb, sg, xtab, lane, strand, hi_bits, gb * 32u + o, o, Bo, st);
        }
    }
    while (cb.count) cont_process<NB>(a, cb, lane, st);
    unsigned long long n_nodes = st.nodes, n_lookups = st.lookups;
    for (int o = 16; o; o >>= 1) { n_nodes += __shfl_xor_sync(FULL, n_nodes, o); n_lookups += __shfl_xor_sync(FULL, n_lookups, o); }
    if (lane == 0) { atomicAdd(a.stats + 0, n_nodes); atomicAdd(a.stats + 1, n_lookups); atomicAdd(a.stats + 5, (unsigned long long)st.sectors); }
}

// ---------------------------------------------------------------------------------------------------------
// sweep_lean_kernel: the same enumeration as sweep_kernel with the inner loops rewritten around what ncu showed on the 3.1 Gb
// workload (profiles/r01ac_sweep_kernel_*): 188 warp instructions per 32 patterns, the whole register file at 50 % occupancy,
// one summary load in flight per lane.  Here
//   * the loops are compiled per PLANE LAYOUT (gsx_core.h sweep_shape_of): which planes count is a template constant, so a
//     pattern without budget costs one LOP3 per used plane (acc |= w ^ X); the guide's seven X words are the same in every
//     lane of a run and end up in uniform registers.  A run picks its loop by the guide's layout (the edited guides of a bulge
//     search mix 19, 20 and 21 characters);
//   * the patterns that use the budget up (nine tenths) are taken 64 per iteration: both summary sectors of a lane are
//     requested before the first is looked at;
//   * nodes with more than 16 rows whose first 16 are dead are parked as ONE word (the table index; everything else is the
//     run's) and drained 32 at a time by the same compiled loop body over sum1 -- no general evaluator, no per-record codes;
//   * loads are predicated instead of branched around, the xor table is always in shared memory (the host sends batches whose
//     table does not fit to sweep_kernel), per-guide constants come straight from the global table (no staging copy), the
//     unsubstituted-pattern step tests "at most one mismatch" with two masks instead of four and reads its second sector
//     in place;
//   * 20 KB of shared memory per 256 threads instead of 47 and 38-55 registers: five or six CTAs per SM fit.
// Same seeds, same counters as sweep_kernel (the tests run both).
// ---------------------------------------------------------------------------------------------------------
constexpr int PK_SLOTS = 96;           // parked nodes per warp: drained below 32 at the top of an iteration, which adds at most 64

// predicated 32-byte summary load (L2 only): lanes without a pattern keep w = 0, i.e. an empty node.  (Letting those lanes load table
// entry 0 instead -- no predicate, no zeroing, nine instructions fewer per load -- was measured and lost 1-2 %: the idle lanes' extra
// sector costs more than the instructions, profiles/r02l_session_3100mb_variant13.jsonl.)
__device__ __forceinline__ void lean_load(const unsigned char* sum, uint32_t idx, bool live, uint32_t w[8]) {
    w[0] = 0u;
#pragma unroll
    for (int j = 1; j < 8; j++) w[j] = 0u;
    asm volatile("{\n\t.reg .pred p;\n\tsetp.ne.u32 p, %9, 0;\n\t@p ld.global.cg.v8.b32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];\n\t}"
                 : "+r"(w[0]), "+r"(w[1]), "+r"(w[2]), "+r"(w[3]), "+r"(w[4]), "+r"(w[5]), "+r"(w[6]), "+r"(w[7])
                 : "l"(sum + ((size_t)idx << 5)), "r"((uint32_t)live));
}

struct LeanRun {                       // warp-uniform: one guide in one slice of one strand
    const unsigned char* sum0; const unsigned char* sum1; const unsigned char* sum2;
    const FtabEntry* tab;
    uint32_t qh;                       // table index of the unsubstituted pattern: slice characters | the guide's other characters
    uint32_t X[7];                     // gsx_core.h summary_masks
    uint32_t codes2, tl, fm;
};
struct LeanStats { uint32_t nodes, two, lines, sectors; };      // nodes, two (nodes over two 64-row blocks): per lane; lines, sectors: warp-uniform
// nodes with more than 16 rows whose first 16 are dead, waiting for a look at rows 16..31 (sum1): two words each -- table index |
// remaining budget << 28, and the task (guide * 2 + strand; everything else is in the guide's row of the guide table).  The buffer
// lives as long as the warp: it is drained 32 at a time, all lanes busy, whichever guides and slices the nodes came from.
struct ParkBuf { uint32_t* idx; uint32_t* tl; uint32_t count; };      // count: warp-uniform

// surviving level-L node -> seed queue (as sweep_emit)
__device__ __forceinline__ void lean_emit(const SweepArgs& a, uint32_t lane, bool emit, uint32_t idx, uint32_t tlm, const FtabEntry* tab) {
    const uint32_t emask = __ballot_sync(0xffffffffu, emit);
    if (!emask) return;
    uint32_t qbase = 0; const int leader = __ffs(emask) - 1;
    if ((int)lane == leader) qbase = atomicAdd(a.queue_count, (uint32_t)__popc(emask));
    qbase = __shfl_sync(0xffffffffu, qbase, leader);
    if (emit) {
        const uint32_t slot = qbase + __popc(emask & ((1u << lane) - 1u));
        if (slot < a.queue_cap) {
            const uint2 e = __ldg(reinterpret_cast<const uint2*>(tab + idx));
            SeedNode sn; sn.sp = e.x; sn.ep = e.x + e.y - 1u; sn.idx = idx; sn.tlm = (tlm & 0x07FFFFFFu) | (a.plan.L << 27);
            a.queue[slot] = sn;
        } else atomicOr(a.error_flag, GSX_KERR_QUEUE_OVERFLOW);
    }
}
__device__ __forceinline__ void lean_park(ParkBuf& pk, uint32_t lane, bool park, uint32_t word, uint32_t tl) {
    const uint32_t m = __ballot_sync(0xffffffffu, park);
    if (!m) return;
    if (park) { const uint32_t slot = pk.count + __popc(m & ((1u << lane) - 1u)); pk.idx[slot] = word; pk.tl[slot] = tl; }
    pk.count += __popc(m);
    __syncwarp();
}
// one judged first sector: counters, then nothing (empty node / no row left), the seed queue, or the parking buffer
__device__ __forceinline__ void lean_settle(const SweepArgs& a, ParkBuf& pk, uint32_t lane, uint32_t w0, uint32_t alive, uint32_t idx, uint32_t budget,
                                            uint32_t tl, const FtabEntry* tab, LeanStats& st) {
    // (w0 == 0 for lanes without a pattern and for empty table entries; the flags are only ever set on non-empty ones)
    const bool emit = (alive | (w0 & SUM_WIDE32)) != 0u;                             // (more than 32 rows: not summarised, the tree search takes it)
    const bool park = !emit && (w0 & SUM_WIDE16) != 0u;
    st.nodes += (w0 & 0xFFFFu) ? 1u : 0u;
    st.two += (w0 & SUM_TWO_BLOCKS) ? 1u : 0u;
    lean_emit(a, lane, emit, idx, tl | ((a.M - budget) << 24) | (budget << 27), tab);
    lean_park(pk, lane, park, idx | (budget << 28), tl);
}
// one pattern of one guide -- its row of the guide table, any plane layout -- against one summary sector: rows still alive after
// the seven planes and, where the guide has them, the two levels behind (sum2).  EXACT: no budget left.  PROTO: the guide's planes
// are all protospacer levels or wildcards (gsx_core.h summary_eval_proto).
template <int NBX, bool EXACT, bool PROTO = false>
__device__ __forceinline__ uint32_t lean_row_eval(const uint32_t* __restrict__ row, const unsigned char* sum, const unsigned char* sum2, uint32_t idx,
                                                  uint32_t budget, uint32_t half, bool live, uint32_t& w0) {
    const uint4* gp = reinterpret_cast<const uint4*>(row);
    const uint4 g0 = __ldg(gp), g1 = __ldg(gp + 1), g2 = __ldg(gp + 2), g3 = __ldg(gp + 3);
    const uint32_t gm[15] = {g0.x, g0.y, g0.z, g0.w, g1.x, g1.y, g1.z, g1.w, g2.x, g2.y, g2.z, g2.w, g3.x, g3.y, g3.z};
    const uint32_t codes2 = __ldg(row + GT_CODES2);
    uint32_t w[8];
    lean_load(sum, idx, live, w);
    w0 = w[0];
    const bool tail = sum2 && sweep_has_tail(codes2) && !(w0 & SUM_WIDE32);
    if (EXACT) {
        uint32_t v[1] = {summary_eval_exact(w, gm)};
        if (v[0] && tail) { uint32_t t[4]; load_tail(sum2, idx, t); summary_tail<1>(t, half, codes2, v); }
        return v[0];
    }
    uint32_t u[NBX];
    if (PROTO) summary_eval_proto<NBX>(w, gm, budget, u); else summary_eval_masks<NBX>(w, gm, budget, u);
    if (u[0] && tail) { uint32_t t[4]; load_tail(sum2, idx, t); summary_tail<NBX>(t, half, codes2, u); }
    return u[0];
}
// up to 32 parked nodes: rows 16..31 of their intervals, each lane with its own node's guide
template <int NB>
__device__ __forceinline__ void lean_drain(const SweepArgs& a, ParkBuf& pk, uint32_t lane, LeanStats& st) {
    const uint32_t n = pk.count < 32u ? pk.count : 32u;
    const bool mine = lane < n;
    uint32_t word = 0, tl = 0;
    if (mine) { word = pk.idx[pk.count - n + lane]; tl = pk.tl[pk.count - n + lane]; }
    __syncwarp();
    pk.count -= n; st.sectors += n;
    const uint32_t idx = word & 0x0FFFFFFFu, budget = word >> 28;
    const bool s1 = (tl & 1u) != 0u;
    uint32_t alive = 0, w0;
    if (mine) alive = lean_row_eval<NB, false>(a.gtab + (size_t)(tl >> 1) * GT_WORDS, s1 ? a.st[1].sum1 : a.st[0].sum1, s1 ? a.st[1].sum2 : a.st[0].sum2,
                                               idx, budget, 1u, true, w0);
    lean_emit(a, lane, alive != 0u, idx, tl | ((a.M - budget) << 24) | (budget << 27), reinterpret_cast<const FtabEntry*>(s1 ? a.st[1].ftab : a.st[0].ftab));
}

// the patterns of pass 1 (exactly B substitutions outside the slice: no budget left), 64 per iteration
template <uint32_t USED, int NB, bool FORCED>
__device__ __forceinline__ void lean_exact_pass(const SweepArgs& a, ParkBuf& pk, const uint32_t* xt, uint32_t n, uint32_t n_lines, uint32_t lane,
                                                const LeanRun& r, LeanStats& st) {
    const uint32_t tl_m = r.tl | (a.M << 24);
    if (n == 0u) return;
    const bool tail = r.sum2 != nullptr && sweep_has_tail(r.codes2);
    if constexpr (!FORCED) { st.sectors += n; st.lines += n_lines; }
    for (uint32_t base = 0; base < n; base += 64u) {
        while (pk.count >= 32u) lean_drain<NB>(a, pk, lane, st);
        const bool two = base + 32u < n;                                             // warp-uniform: a second 32 patterns in this iteration
        const uint32_t t0 = base + lane, t1 = t0 + 32u;
        bool live0 = t0 < n, live1 = t1 < n;
        const uint32_t x0 = xt[t0], x1 = xt[t1];                                     // (the shared table has 64 readable words behind its end)
        if constexpr (FORCED) {                                                      // patterns that substitute a must-match position are skipped
            live0 = live0 && !(x0 & r.fm); live1 = live1 && !(x1 & r.fm);
            const uint32_t b0 = __ballot_sync(0xffffffffu, live0), b1 = __ballot_sync(0xffffffffu, live1);
            st.sectors += __popc(b0) + __popc(b1);
            st.lines += __popc(__ballot_sync(0xffffffffu, live0 && (x0 & 15u) == 0u)) + __popc(__ballot_sync(0xffffffffu, live1 && (x1 & 15u) == 0u));
        }
        const uint32_t idx0 = r.qh ^ (x0 & 0x0FFFFFFFu), idx1 = r.qh ^ (x1 & 0x0FFFFFFFu);
        uint32_t w0[8], w1[8];
        lean_load(r.sum0, idx0, live0, w0);
        lean_load(r.sum0, idx1, live1, w1);                                    // (no lane has a pattern there when there is no second 32)
        uint32_t al0 = summary_exact_shape<USED>(w0, r.X), al1 = two ? summary_exact_shape<USED>(w1, r.X) : 0u;
        if (!two) w1[0] = 0u;
        if (al0 && tail && !(w0[0] & SUM_WIDE32)) { uint32_t t[4], v[1] = {al0}; load_tail(r.sum2, idx0, t); summary_tail<1>(t, 0u, r.codes2, v); al0 = v[0]; }
        if (al1 && tail && !(w1[0] & SUM_WIDE32)) { uint32_t t[4], v[1] = {al1}; load_tail(r.sum2, idx1, t); summary_tail<1>(t, 0u, r.codes2, v); al1 = v[0]; }
        // (w[0] == 0 for lanes without a pattern and for empty table entries; the flags are only ever set on non-empty ones)
        const bool emit0 = (al0 | (w0[0] & SUM_WIDE32)) != 0u, emit1 = (al1 | (w1[0] & SUM_WIDE32)) != 0u;      // (more than 32 rows: the tree search takes it)
        const bool park0 = !emit0 && (w0[0] & SUM_WIDE16) != 0u, park1 = !emit1 && (w1[0] & SUM_WIDE16) != 0u;
        st.nodes += ((w0[0] & 0xFFFFu) ? 1u : 0u) + ((w1[0] & 0xFFFFu) ? 1u : 0u);
        st.two += ((w0[0] & SUM_TWO_BLOCKS) ? 1u : 0u) + ((w1[0] & SUM_TWO_BLOCKS) ? 1u : 0u);
        if (__any_sync(0xffffffffu, emit0 || emit1)) { lean_emit(a, lane, emit0, idx0, tl_m, r.tab); lean_emit(a, lane, emit1, idx1, tl_m, r.tab); }
        const uint32_t m0 = __ballot_sync(0xffffffffu, park0), m1 = __ballot_sync(0xffffffffu, park1);
        if (m0 | m1) {
            const uint32_t lt = (1u << lane) - 1u;
            if (park0) { const uint32_t slot = pk.count + __popc(m0 & lt); pk.idx[slot] = idx0; pk.tl[slot] = r.tl; }
            if (park1) { const uint32_t slot = pk.count + __popc(m0) + __popc(m1 & lt); pk.idx[slot] = idx1; pk.tl[slot] = r.tl; }
            pk.count += __popc(m0) + __popc(m1);
            __syncwarp();
        }
    }
}
// the patterns of pass 0 (fewer than B substitutions outside the slice: budget left), 32 per iteration
template <uint32_t PROTO, uint32_t PAM, int NB, bool FORCED>
__device__ __forceinline__ void lean_budget_pass(const SweepArgs& a, ParkBuf& pk, const uint32_t* xt, uint32_t n, uint32_t n_lines, uint32_t lane,
                                                 const LeanRun& r, uint32_t B, LeanStats& st) {
    if (n == 0u) return;
    const bool tail = r.sum2 != nullptr && sweep_has_tail(r.codes2);
    if constexpr (!FORCED) { st.sectors += n; st.lines += n_lines; }
    for (uint32_t base = 0; base < n; base += 32u) {
        while (pk.count >= 32u) lean_drain<NB>(a, pk, lane, st);
        const uint32_t t = base + lane;
        bool live = t < n;
        const uint32_t xw = xt[t];
        if constexpr (FORCED) {
            live = live && !(xw & r.fm);
            st.sectors += __popc(__ballot_sync(0xffffffffu, live)); st.lines += __popc(__ballot_sync(0xffffffffu, live && (xw & 15u) == 0u));
        }
        const uint32_t idx = r.qh ^ (xw & 0x0FFFFFFFu), budget = B - (xw >> 28);
        uint32_t w[8];
        lean_load(r.sum0, idx, live, w);
        uint32_t u[NB];
        summary_masks_shape<PROTO, PAM, NB>(w, r.X, budget, u);
        if (u[0] && tail && !(w[0] & SUM_WIDE32)) { uint32_t tt[4]; load_tail(r.sum2, idx, tt); summary_tail<NB>(tt, 0u, r.codes2, u); }
        lean_settle(a, pk, lane, w[0], u[0], idx, budget, r.tl, r.tab, st);
    }
}
template <int SHAPE, int NB, bool FORCED>
__device__ __forceinline__ void lean_run(const SweepArgs& a, const SweepPlan& pl, ParkBuf& pk, const uint32_t* xtab, uint32_t lane, const LeanRun& r,
                                         uint32_t B, LeanStats& st) {
    constexpr uint32_t PROTO = SHAPE == 0 ? 0x3Fu : SHAPE == 1 ? 0x7Fu : 0x1Fu, PAM = SHAPE == 2 ? 0x40u : 0u;
    lean_exact_pass<PROTO | PAM, NB, FORCED>(a, pk, xtab + pl.xoff[1][B], pl.xcnt[1][B], pl.xlines[1][B], lane, r, st);
    lean_budget_pass<PROTO, PAM, NB, FORCED>(a, pk, xtab + pl.xoff[0][B], pl.xcnt[0][B], pl.xlines[0][B], lane, r, B, st);
}

// XTG: the xor table is too long for shared memory (4 mismatches: 15.8 k words) and is read from global memory (unit stride,
// the same few KB by every warp: L1 hits); the host pads it with 64 readable words
template <int WARPS, int MINB, int NB, bool FORCED = false, bool XTG = false>
__global__ void __launch_bounds__(WARPS * 32, MINB) sweep_lean_kernel(SweepArgs a) {
    __shared__ SweepPlan s_plan;
    __shared__ uint32_t s_park[WARPS][2][PK_SLOTS];
    __shared__ uint32_t s_rank[WARPS][32];
    __shared__ uint32_t s_xtab_[XTG ? 1 : XT_SMEM];
    for (int i = threadIdx.x; i < (int)(sizeof(SweepPlan) / 4); i += blockDim.x)
        reinterpret_cast<uint32_t*>(&s_plan)[i] = reinterpret_cast<const uint32_t*>(&a.plan)[i];
    if constexpr (!XTG) for (uint32_t i = threadIdx.x; i < (uint32_t)XT_SMEM; i += blockDim.x) s_xtab_[i] = i < a.n_xtab ? a.xtab[i] : 0u;
    const uint32_t* const s_xtab = XTG ? a.xtab : s_xtab_;
    __syncthreads();
    const uint32_t lane = threadIdx.x & 31u, warp = threadIdx.x >> 5, FULL = 0xffffffffu;
    ParkBuf pk; pk.idx = s_park[warp][0]; pk.tl = s_park[warp][1]; pk.count = 0;
    const uint32_t L = s_plan.L, sb = s_plan.sb, M = a.M;
    const uint32_t np1 = s_plan.xcnt[1][1], np1_magic = np1 ? 0xFFFFFFFFu / np1 + 1u : 0u;      // f / np1 = umulhi(f, magic) for the small f used here
    const uint32_t n_slices = 1u << (2u * sb), n_gb = (a.n_guides + 31u) >> 5;
    const uint32_t items_per_strand = n_slices * n_gb, n_items = 2u * items_per_strand;      // (the host keeps this below 2^32)
    LeanStats st = {0, 0, 0, 0};
    for (;;) {
        uint32_t item = 0;
        if (lane == 0) item = atomicAdd(a.item_counter, 1u);
        item = __shfl_sync(FULL, item, 0);
        if (item >= n_items) break;
        const uint32_t strand = item >= items_per_strand ? 1u : 0u;
        const uint32_t rem = item - (strand ? items_per_strand : 0u);
        const uint32_t beta = rem / n_gb, gb = rem - beta * n_gb;
        const uint32_t g = gb * 32u + lane;
        const bool valid = g < a.n_guides && !(a.skip && a.skip[g]);
        const unsigned char* sum0 = strand ? a.st[1].sum0 : a.st[0].sum0;
        const unsigned char* sum1 = strand ? a.st[1].sum1 : a.st[0].sum1;
        const unsigned char* sum2 = strand ? a.st[1].sum2 : a.st[0].sum2;
        const FtabEntry* tab = reinterpret_cast<const FtabEntry*>(strand ? a.st[1].ftab : a.st[0].ftab);
        const uint32_t hi_bits = beta << (2u * (L - sb));
        int B = -1;
        if (valid) {
            const uint64_t q = __ldg(a.gq + g);
            const uint32_t h = sweep_slice_distance(q, L, sb, beta);
            if (h <= M) B = (int)(M - h);
            if constexpr (FORCED) {      // the slice substitutes a must-match position of this (edited) guide: nothing to do here
                const uint32_t top = (uint32_t)(q >> (2u * (L - sb))) & ((1u << (2u * sb)) - 1u);
                if ((top ^ beta) & (__ldg(a.gtab + (size_t)g * GT_WORDS + GT_FMASK) >> (2u * (L - sb)))) B = -1;
            }
        }
        // (1) guides whose only pattern in this slice is the unsubstituted one (budget 0), and the unsubstituted pattern of the guides
        //     with budget 1: one pattern per lane, each lane with its own guide's masks (any plane layout); a node with more than 16
        //     rows whose first 16 are dead reads its second sector right here
        {
            const bool mine = B == 0 || B == 1;
            const uint32_t mmask = __ballot_sync(FULL, mine);
            st.sectors += __popc(mmask); st.lines += __popc(mmask);                  // (the unsubstituted pattern opens its table line)
            uint32_t idx = 0, alive = 0, w0 = 0;
            bool more = false;
            if (mine) {
                idx = hi_bits | __ldg(a.gtab + (size_t)g * GT_WORDS + GT_QLOW);
                alive = lean_row_eval<2, false>(a.gtab + (size_t)g * GT_WORDS, sum0, sum2, idx, (uint32_t)B, 0u, true, w0);
                more = alive == 0u && !(w0 & SUM_WIDE32) && (w0 & SUM_WIDE16);
            }
            const uint32_t moremask = __ballot_sync(FULL, more);
            if (moremask) {
                st.sectors += __popc(moremask);
                uint32_t w1;
                if (more) alive = lean_row_eval<2, false>(a.gtab + (size_t)g * GT_WORDS, sum1, sum2, idx, (uint32_t)B, 1u, true, w1);
            }
            st.nodes += (w0 & 0xFFFFu) ? 1u : 0u;
            st.two += (w0 & SUM_TWO_BLOCKS) ? 1u : 0u;
            const uint32_t Bp = (uint32_t)(B > 0 ? B : 0);
            lean_emit(a, lane, (alive | (w0 & SUM_WIDE32)) != 0u, idx, ((g << 1) | strand) | ((M - Bp) << 24) | (Bp << 27), tab);
        }
        // (2) guides with budget 1: their patterns with exactly one substitution outside the slice, all of them as ONE list, 32 per
        //     step, each lane with its own guide's masks.  (There are about three such guides per unit with 27 patterns each: a run per
        //     guide costs more in set-up than in patterns -- 90 % of the runs of the first version of this kernel were these.)
        {
            const uint32_t todo1 = __ballot_sync(FULL, B == 1);
            if (todo1 && np1) {
                if (B == 1) s_rank[warp][__popc(todo1 & ((1u << lane) - 1u))] = lane;
                __syncwarp();
                const uint32_t total = (uint32_t)__popc(todo1) * np1;
                const uint32_t* xt1 = s_xtab + s_plan.xoff[1][1];
                for (uint32_t f0 = 0; f0 < total; f0 += 32u) {
                    while (pk.count >= 32u) lean_drain<NB>(a, pk, lane, st);
                    const uint32_t f = f0 + lane;
                    bool live = f < total;
                    const uint32_t k = live ? __umulhi(f, np1_magic) : 0u, t = live ? f - k * np1 : 0u;
                    const uint32_t go = gb * 32u + s_rank[warp][k];
                    const uint32_t* row = a.gtab + (size_t)go * GT_WORDS;
                    const uint32_t xw = xt1[t];
                    if constexpr (FORCED) live = live && !(xw & (__ldg(row + GT_FMASK) & 0x0FFFFFFFu));
                    st.sectors += __popc(__ballot_sync(FULL, live)); st.lines += __popc(__ballot_sync(FULL, live && (xw & 15u) == 0u));
                    const uint32_t idx = hi_bits | (__ldg(row + GT_QLOW) ^ (xw & 0x0FFFFFFFu));
                    uint32_t w0;
                    const uint32_t alive = lean_row_eval<1, true>(row, sum0, sum2, idx, 0u, 0u, live, w0);
                    lean_settle(a, pk, lane, w0, alive, idx, 0u, (go << 1) | strand, tab, st);
                }
                __syncwarp();
            }
        }
        // (3) guides with more budget left after the slice characters, one at a time, all lanes on that guide's patterns
        uint32_t todo = __ballot_sync(FULL, B >= 2);
        while (todo) {
            const uint32_t o = (uint32_t)__ffs(todo) - 1u; todo &= todo - 1u;
            const uint32_t Bo = (uint32_t)__shfl_sync(FULL, B, o), go = gb * 32u + o;
            const uint4* gp = reinterpret_cast<const uint4*>(a.gtab + (size_t)go * GT_WORDS);      // same address in every lane: one transaction
            const uint4 g1 = __ldg(gp + 1), g2 = __ldg(gp + 2), g3 = __ldg(gp + 3), g4 = __ldg(gp + 4);
            LeanRun r;
            r.sum0 = sum0; r.sum1 = sum1; r.sum2 = sum2; r.tab = tab; r.qh = hi_bits | g3.w;
            r.X[0] = g1.w; r.X[1] = g2.x; r.X[2] = g2.y; r.X[3] = g2.z; r.X[4] = g2.w; r.X[5] = g3.x; r.X[6] = g3.y;
            r.codes2 = g4.y; r.fm = g4.z & 0x0FFFFFFFu; r.tl = (go << 1) | strand;
            const uint32_t shape = g4.w;
            if (shape == 0u) lean_run<0, NB, FORCED>(a, s_plan, pk, s_xtab, lane, r, Bo, st);
            else if (shape == 1u) lean_run<1, NB, FORCED>(a, s_plan, pk, s_xtab, lane, r, Bo, st);
            else lean_run<2, NB, FORCED>(a, s_plan, pk, s_xtab, lane, r, Bo, st);
        }
    }
    while (pk.count) lean_drain<NB>(a, pk, lane, st);
    unsigned long long n_nodes = st.nodes, n_two = st.two;
    for (int o = 16; o; o >>= 1) { n_nodes += __shfl_xor_sync(FULL, n_nodes, o); n_two += __shfl_xor_sync(FULL, n_two, o); }
    if (lane == 0) { atomicAdd(a.stats + 0, n_nodes); atomicAdd(a.stats + 1, n_nodes + n_two + st.lines); atomicAdd(a.stats + 5, (unsigned long long)st.sectors); }
}

// ---------------------------------------------------------------------------------------------------------
// sweep_split_kernel: the two-part enumeration (gsx_types.h SplitPlan).  An alignment with at most 3 mismatches has at most one of
// them among the guide's ten PAM-distal characters -- form 0, the guide read distal-first as above, capped to one substitution over
// those ten: 2 185 patterns per guide and strand at L = 14 -- or at most one among the ten PAM-proximal ones -- form 1, the same
// site read PAM-first in the other strand's index: the PAM's concrete characters fixed, its wildcard free, one substitution over the
// proximal half: 496 patterns.  Together a quarter of the 10 690 patterns of the plain enumeration.  A work unit = (index i, slice,
// 32 guides) runs form 0 of task (g, i) and form 1 of task (g, 1 - i), both against index i's slice.  With a few patterns per guide
// in a slice, the unit's patterns of both forms are ONE flat (guide, pattern) list, each lane judging its pattern with its own
// guide's row of the guide table (rows n .. 2n-1: form 1).  Seeds of form 1 go to a queue of their own: search_fast_kernel
// finishes them with the PAM-first query, and reanchor_kernel turns their matches into the records of the distal-first search.
// ---------------------------------------------------------------------------------------------------------
__device__ __forceinline__ void split_emit(const SweepArgs& a, uint32_t lane, bool emit, bool form1, uint32_t idx, uint32_t tlm, const FtabEntry* tab) {
#pragma unroll
    for (int f = 0; f < 2; f++) {
        const bool e = emit && (form1 == (f == 1));
        const uint32_t emask = __ballot_sync(0xffffffffu, e);
        if (!emask) continue;
        uint32_t* cnt = f ? a.queue2_count : a.queue_count;
        SeedNode* queue = f ? a.queue2 : a.queue;
        uint32_t qbase = 0; const int leader = __ffs(emask) - 1;
        if ((int)lane == leader) qbase = atomicAdd(cnt, (uint32_t)__popc(emask));
        qbase = __shfl_sync(0xffffffffu, qbase, leader);
        if (e) {
            const uint32_t slot = qbase + __popc(emask & ((1u << lane) - 1u));
            if (slot < a.queue_cap) {
                const uint2 v = __ldg(reinterpret_cast<const uint2*>(tab + idx));
                SeedNode sn; sn.sp = v.x; sn.ep = v.x + v.y - 1u; sn.idx = idx; sn.tlm = (tlm & 0x07FFFFFFu) | (a.plan.L << 27);
                queue[slot] = sn;
            } else atomicOr(a.error_flag, GSX_KERR_QUEUE_OVERFLOW);
        }
    }
}
// up to 32 parked nodes of either form: rows 16..31 of their intervals (as lean_drain)
template <int NB, bool PROTO>
__device__ __forceinline__ void split_drain(const SweepArgs& a, ParkBuf& pk, uint32_t lane, LeanStats& st) {
    const uint32_t n = pk.count < 32u ? pk.count : 32u;
    const bool mine = lane < n;
    uint32_t word = 0, tl = 0;
    if (mine) { word = pk.idx[pk.count - n + lane]; tl = pk.tl[pk.count - n + lane]; }
    __syncwarp();
    pk.count -= n; st.sectors += n;
    const uint32_t idx = word & 0x0FFFFFFFu, budget = word >> 28, row = tl >> 1;
    const bool s1 = (tl & 1u) != 0u, form1 = row >= a.n_guides;
    uint32_t alive = 0, w0;
    if (mine) alive = lean_row_eval<NB, false, PROTO>(a.gtab + (size_t)row * GT_WORDS, s1 ? a.st[1].sum1 : a.st[0].sum1,
                                                      s1 ? a.st[1].sum2 : a.st[0].sum2, idx, budget, 1u, true, w0);
    const uint32_t g = row - (form1 ? a.n_guides : 0u);
    split_emit(a, lane, alive != 0u, form1, idx, ((g << 1) | (tl & 1u)) | ((a.M - budget) << 24) | (budget << 27),
               reinterpret_cast<const FtabEntry*>(s1 ? a.st[1].ftab : a.st[0].ftab));
}

// PROTO: the rows of both forms have only protospacer and wildcard planes (20-nt guides at jump-table depth 13 or 14): judged with
// summary_eval_proto, half the instructions of the general filter
template <int WARPS, int MINB, int NB, bool PROTO>
__global__ void __launch_bounds__(WARPS * 32, MINB) sweep_split_kernel(SweepArgs a) {
    __shared__ SplitPlan s_sp;
    __shared__ uint32_t s_park[WARPS][2][PK_SLOTS];
    __shared__ uint32_t s_off[WARPS][32], s_n0[WARPS][32], s_l0[WARPS][32], s_l1[WARPS][32];
    __shared__ uint32_t s_xtab[kSplitXtabShared];
    for (int i = threadIdx.x; i < (int)(sizeof(SplitPlan) / 4); i += blockDim.x)
        reinterpret_cast<uint32_t*>(&s_sp)[i] = reinterpret_cast<const uint32_t*>(&a.split)[i];
    for (uint32_t i = threadIdx.x; i < (uint32_t)kSplitXtabShared; i += blockDim.x) s_xtab[i] = i < a.n_xtab ? a.xtab[i] : 0u;
    __syncthreads();
    const uint32_t lane = threadIdx.x & 31u, warp = threadIdx.x >> 5, FULL = 0xffffffffu;
    ParkBuf pk; pk.idx = s_park[warp][0]; pk.tl = s_park[warp][1]; pk.count = 0;
    const uint32_t L = a.plan.L, sb = a.plan.sb, M = a.M, n = a.n_guides;
    const uint32_t low = 2u * (L - sb), top_mask = (1u << (2u * sb)) - 1u;
    const uint32_t n_slices = 1u << (2u * sb), n_gb = (n + 31u) >> 5;
    const uint32_t items_per_strand = n_slices * n_gb, n_items = 2u * items_per_strand;      // (the host keeps this below 2^32)
    LeanStats st = {0, 0, 0, 0};
    for (;;) {
        uint32_t item = 0;
        if (lane == 0) item = atomicAdd(a.item_counter, 1u);
        item = __shfl_sync(FULL, item, 0);
        if (item >= n_items) break;
        const uint32_t strand = item >= items_per_strand ? 1u : 0u;
        const uint32_t rem = item - (strand ? items_per_strand : 0u);
        const uint32_t beta = rem / n_gb, gb = rem - beta * n_gb;
        const uint32_t g = gb * 32u + lane;
        const bool valid = g < n && !(a.skip && a.skip[g]);
        // this lane's guide: how many patterns of each form fall into the slice, and which list of the xor table they are
        uint32_t cnt0 = 0, cnt1 = 0, l0 = 0, l1 = 0;
        if (valid) {
#pragma unroll
            for (uint32_t f = 0; f < 2u; f++) {
                const uint64_t q = __ldg((f ? a.gq2 : a.gq) + g);
                const uint32_t x = ((uint32_t)(q >> low) & top_mask) ^ beta, d = (x | (x >> 1)) & 0x55555555u;
                const uint32_t h = __popc(d & s_sp.cost_top[f]), cp = __popc(d & s_sp.cap_top[f]);
                if (!(d & s_sp.exact_top[f]) && h <= M && cp <= 1u) {
                    const uint32_t Bf = M - h, c = 1u - cp;
                    const uint32_t w = s_sp.xoff[f][c][Bf] | (Bf << 16), k = s_sp.xcnt[f][c][Bf];
                    if (f) { cnt1 = k; l1 = w; } else { cnt0 = k; l0 = w; }
                }
            }
        }
        const uint32_t mine = cnt0 + cnt1;
        uint32_t incl = mine;
#pragma unroll
        for (uint32_t o = 1; o < 32u; o <<= 1) { const uint32_t v = __shfl_up_sync(FULL, incl, o); if (lane >= o) incl += v; }
        const uint32_t total = __shfl_sync(FULL, incl, 31);
        if (total == 0u) continue;
        __syncwarp();
        s_off[warp][lane] = incl - mine; s_n0[warp][lane] = cnt0; s_l0[warp][lane] = l0; s_l1[warp][lane] = l1;
        __syncwarp();
        st.sectors += total;
        const unsigned char* sum0 = strand ? a.st[1].sum0 : a.st[0].sum0;
        const unsigned char* sum2 = strand ? a.st[1].sum2 : a.st[0].sum2;
        const FtabEntry* tab = reinterpret_cast<const FtabEntry*>(strand ? a.st[1].ftab : a.st[0].ftab);
        const uint32_t hi_bits = beta << low;
        for (uint32_t f0 = 0; f0 < total; f0 += 32u) {
            while (pk.count >= 32u) split_drain<NB, PROTO>(a, pk, lane, st);
            const uint32_t fi = f0 + lane;
            const bool live = fi < total;
            uint32_t k = 0;                                                           // the lane whose list holds pattern fi: last k with off[k] <= fi
#pragma unroll
            for (uint32_t step = 16; step; step >>= 1) if (s_off[warp][k + step] <= fi) k += step;
            uint32_t t = fi - s_off[warp][k];
            const uint32_t n0 = s_n0[warp][k];
            const bool form1 = t >= n0;
            if (form1) t -= n0;
            const uint32_t lw = form1 ? s_l1[warp][k] : s_l0[warp][k];
            const uint32_t xw = live ? s_xtab[(lw & 0xFFFFu) + t] : 0u;
            const uint32_t go = gb * 32u + k, row = live ? go + (form1 ? n : 0u) : 0u;
            const uint32_t* rowp = a.gtab + (size_t)row * GT_WORDS;
            const uint32_t idx = hi_bits | (__ldg(rowp + GT_QLOW) ^ (xw & 0x0FFFFFFFu));
            const uint32_t budget = live ? (lw >> 16) - (xw >> 28) : 0u;
            st.lines += __popc(__ballot_sync(FULL, live && (xw & 15u) == 0u));
            uint32_t w0;
            const uint32_t alive = lean_row_eval<NB, false, PROTO>(rowp, sum0, sum2, idx, budget, 0u, live, w0);
            // (w0 == 0 for lanes without a pattern and for empty table entries; the flags are only ever set on non-empty ones)
            const bool emit = (alive | (w0 & SUM_WIDE32)) != 0u;                     // (more than 32 rows: not summarised, the tree search takes it)
            const bool park = !emit && (w0 & SUM_WIDE16) != 0u;
            st.nodes += (w0 & 0xFFFFu) ? 1u : 0u;
            st.two += (w0 & SUM_TWO_BLOCKS) ? 1u : 0u;
            split_emit(a, lane, emit, form1, idx, ((go << 1) | strand) | ((M - budget) << 24) | (budget << 27), tab);
            lean_park(pk, lane, park, idx | (budget << 28), (row << 1) | strand);
        }
    }
    while (pk.count) split_drain<NB, PROTO>(a, pk, lane, st);
    unsigned long long n_nodes = st.nodes, n_two = st.two;
    for (int o = 16; o; o >>= 1) { n_nodes += __shfl_xor_sync(FULL, n_nodes, o); n_two += __shfl_xor_sync(FULL, n_two, o); }
    if (lane == 0) { atomicAdd(a.stats + 0, n_nodes); atomicAdd(a.stats + 1, n_nodes + n_two + st.lines); atomicAdd(a.stats + 5, (unsigned long long)st.sectors); }
}

__global__ void split_queries_kernel(const uint64_t* __restrict__ gq, uint32_t n, uint32_t pampack, uint32_t plen, uint64_t* __restrict__ gq2) {
    for (uint32_t g = blockIdx.x * blockDim.x + threadIdx.x; g < n; g += gridDim.x * blockDim.x) gq2[g] = split_query(gq[g], pampack, plen);
}

// one form-1 match: back to the distal-first consumed string of the same site; dropped when it has fewer than two mismatches among the
// guide's first ten characters (form 0 found it); else its interval in the other index by an exact backward search (jump table, then
// one occurrence lookup per interval end and character) and the record the distal-first search emits for it
__global__ void reanchor_kernel(ReanchorArgs r) {
    const uint32_t n_in = min(*r.n_in, r.in_cap);
    unsigned long long lookups = 0;
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n_in; i += gridDim.x * blockDim.x) {
        const MatchRec m = r.in[i];
        const uint32_t g = m.task >> 1, s = (m.task & 1u) ^ 1u;
        const uint64_t q = __ldg(r.gq + g), q2 = __ldg(r.gq2 + g);
        const uint32_t qlen = (uint32_t)(q >> 58), T = qlen + r.plen, half = qlen / 2u;
        uint32_t u[kMaxQ];
        if (split_unfold(m.key_lo, q2, T, q, half, u) < 2u) continue;
        uint32_t mm;
        const uint64_t key = split_key(u, q, r.plen, mm);
        const DevStrand& st = r.st[s];
        const uint32_t L = st.ftab_L;
        uint32_t e = 0;
        for (uint32_t j = 0; j < L; j++) e |= u[j] << (2u * j);
        const uint2 v = __ldg(reinterpret_cast<const uint2*>(reinterpret_cast<const FtabEntry*>(st.ftab) + e));
        uint32_t sp = v.x, e1 = v.x + v.y;
        lookups += 1u + 2u * (T - L);
        for (uint32_t j = L; j < T && sp < e1; j++) {
            const OccBlock* b0 = block_ptr(st, sp >> 6); const OccBlock* b1 = block_ptr(st, e1 >> 6);
            uint32_t os[4], oe[4];
            block_occ(st, b0->cnt, b0->hi, b0->lo, sp, os); block_occ(st, b1->cnt, b1->hi, b1->lo, e1, oe);
            sp = st.C[u[j]] + os[u[j]]; e1 = st.C[u[j]] + oe[u[j]];
        }
        if (e1 - sp != m.width || sp >= e1) { atomicOr(r.error_flag, GSX_KERR_REANCHOR); continue; }
        const uint32_t slot = atomicAdd(r.out_count, 1u);
        if (slot < r.out_cap) {
            MatchRec o; o.key_hi = 0; o.key_lo = key; o.task = (g << 1) | s; o.sp = sp; o.width = m.width; o.info = mm | (T << 24);
            r.out[slot] = o;
            atomicAdd(r.guide_nmatch + g, 1u);
        } else atomicOr(r.error_flag, GSX_KERR_MATCH_OVERFLOW);
    }
    if (lookups) atomicAdd(r.stats + 7, lookups);
}

cudaError_t launch_split_queries(const uint64_t* gq, uint32_t n, uint32_t pampack, uint32_t plen, uint64_t* gq2, cudaStream_t s) {
    split_queries_kernel<<<grid_for_n(n, 256, 148 * 8), 256, 0, s>>>(gq, n, pampack, plen, gq2);
    return cudaGetLastError();
}
cudaError_t launch_sweep_split(const SweepArgs& a, int ctas_per_sm, int sm_count, cudaStream_t s) {
    if (a.M > kSplitMaxM || a.n_xtab > (uint32_t)kSplitXtabShared) return cudaErrorInvalidValue;
    const dim3 block(8 * 32);
    // both forms' plane layouts (20-nt guides; form 1 reads all 23 characters as protospacer): protospacer and wildcard planes only?
    const int shape0 = sweep_shape_of(sweep_codes((uint64_t)20 << 58, a.plan.L, a.plen, a.pampack));
    const int shape1 = sweep_shape_of(sweep_codes((uint64_t)(20 + a.plen) << 58, a.plan.L, 0, 0));
    const bool proto = (shape0 == 0 || shape0 == 1) && (shape1 == 0 || shape1 == 1);
#define GSX_SPLIT_LAUNCH(C)                                                                                      \
    case C: if (proto) sweep_split_kernel<8, C, 4, true><<<sm_count * C, block, 0, s>>>(a);                   \
            else sweep_split_kernel<8, C, 4, false><<<sm_count * C, block, 0, s>>>(a); break;
    switch (ctas_per_sm) {
    GSX_SPLIT_LAUNCH(4) GSX_SPLIT_LAUNCH(5) GSX_SPLIT_LAUNCH(6) GSX_SPLIT_LAUNCH(8)
    default: return cudaErrorInvalidValue;
    }
#undef GSX_SPLIT_LAUNCH
    return cudaGetLastError();
}
cudaError_t launch_reanchor(const ReanchorArgs& r, cudaStream_t s) {
    reanchor_kernel<<<148 * 4, 256, 0, s>>>(r);
    return cudaGetLastError();
}

cudaError_t launch_sweep_guides(const SweepArgs& a, cudaStream_t s) {
    sweep_guides_kernel<<<grid_for_n(a.n_guides, 256, 148 * 8), 256, 0, s>>>(a, a.gtab);
    return cudaGetLastError();
}

template <int WARPS, int MINB>
static cudaError_t launch_sweep_t(const SweepArgs& a, int sm_count, cudaStream_t s) {
    // NB = number of budget masks of the row filter: at most 3 mismatches (the default) or at most 4
    if (a.M <= 3) sweep_kernel<WARPS, MINB, 4><<<sm_count * MINB, WARPS * 32, 0, s>>>(a);
    else if (a.M <= 4) sweep_kernel<WARPS, MINB, 5><<<sm_count * MINB, WARPS * 32, 0, s>>>(a);
    else return cudaErrorInvalidValue;
    return cudaGetLastError();
}
template <int MINB>
static cudaError_t launch_sweep_lean_t(const SweepArgs& a, int sm_count, cudaStream_t s) {
    const bool shared_xt = a.n_xtab + 64u <= (uint32_t)XT_SMEM;                     // (else: a.xtab holds 64 readable words behind the table)
    const dim3 grid(sm_count * MINB), block(8 * 32);
    if (a.M <= 3 && shared_xt) {
        if (a.fmask) sweep_lean_kernel<8, MINB, 4, true, false><<<grid, block, 0, s>>>(a); else sweep_lean_kernel<8, MINB, 4, false, false><<<grid, block, 0, s>>>(a);
    } else if (a.M <= 4) {
        if (a.fmask) sweep_lean_kernel<8, MINB, 5, true, true><<<grid, block, 0, s>>>(a); else sweep_lean_kernel<8, MINB, 5, false, true><<<grid, block, 0, s>>>(a);
    } else return cudaErrorInvalidValue;
    return cudaGetLastError();
}
cudaError_t launch_sweep(const SweepArgs& a, int variant, int sm_count, cudaStream_t s) {
    switch (variant) {
    case 10: return launch_sweep_lean_t<4>(a, sm_count, s);   // lean loops, 1024 thr/SM
    case 11: return launch_sweep_lean_t<5>(a, sm_count, s);   // 1280 thr/SM
    case 12: return launch_sweep_lean_t<6>(a, sm_count, s);   // 1536 thr/SM
    case 0: return launch_sweep_t<8, 3>(a, sm_count, s);      // 768 thr/SM
    case 1: return launch_sweep_t<8, 2>(a, sm_count, s);      // 512 thr/SM
    case 2:                                                   // 1024 thr/SM
        if (a.fmask) {                                        // edited guides with their must-match positions: the default variant only
            if (a.M <= 3) sweep_kernel<8, 4, 4, true><<<sm_count * 4, 8 * 32, 0, s>>>(a);
            else if (a.M <= 4) sweep_kernel<8, 4, 5, true><<<sm_count * 4, 8 * 32, 0, s>>>(a);
            else return cudaErrorInvalidValue;
            return cudaGetLastError();
        }
        return launch_sweep_t<8, 4>(a, sm_count, s);
    case 3: return launch_sweep_t<8, 6>(a, sm_count, s);      // 1536 thr/SM
    case 4: return launch_sweep_t<8, 8>(a, sm_count, s);      // 2048 thr/SM
    case 5: return launch_sweep_t<8, 5>(a, sm_count, s);      // 1280 thr/SM
    }
    return cudaErrorInvalidValue;
}

// ---------------------------------------------------------------------------------------------------------
// bulges as edited guides (gsx_core.h variant_rewrite): a bulge batch is searched as a mismatch-only batch holding every
// edited form of every guide -- which puts it on the sweep / jump-table kernels above instead of the general tree walk --
// and its matches are rewritten into the guides' own (wide-key) matches afterwards.
// ---------------------------------------------------------------------------------------------------------
// one thread per edited guide v of the chunk: which guide, which op list; the packed edited guide for the search kernels
//   seg[3 * i ..]: {first edited guide of segment i within the chunk, its guide, index of its first op list among the guide's};
//   a segment = a run of op lists of one guide (a guide whose edited forms exceed a chunk spans several);
//   seg[3 * n_seg] = number of edited guides of the chunk;  doff[qlen]: start of the op lists for guides of that length
__global__ void variant_expand_kernel(const GuideRec* __restrict__ guides, uint32_t n_seg, const uint32_t* __restrict__ seg,
                                      const uint32_t* __restrict__ descs, const uint32_t* __restrict__ doff,
                                      uint64_t* __restrict__ vq, uint32_t* __restrict__ vdesc, uint32_t* __restrict__ vguide, uint32_t* __restrict__ vfmask) {
    const uint32_t n_v = seg[3u * n_seg];
    for (uint32_t v = blockIdx.x * blockDim.x + threadIdx.x; v < n_v; v += gridDim.x * blockDim.x) {
        uint32_t lo = 0, hi = n_seg;                                 // last segment starting at or before v
        while (hi - lo > 1u) { const uint32_t mid = (lo + hi) >> 1; if (seg[3u * mid] <= v) lo = mid; else hi = mid; }
        const uint32_t gi = seg[3u * lo + 1u];
        const GuideRec& g = guides[gi];
        const uint32_t desc = descs[doff[g.qlen] + seg[3u * lo + 2u] + (v - seg[3u * lo])];
        vq[v] = variant_pack(g.q, g.qlen, desc); vdesc[v] = desc; vguide[v] = gi;
        if (vfmask) vfmask[v] = variant_forced_mask(g.qlen, desc);
    }
}
cudaError_t launch_variant_expand(const GuideRec* guides, uint32_t n_seg, uint32_t n_v, const uint32_t* seg, const uint32_t* descs,
                                  const uint32_t* doff, uint64_t* vq, uint32_t* vdesc, uint32_t* vguide, uint32_t* vfmask, cudaStream_t s) {
    if (!n_v) return cudaSuccess;
    long b = ((long)n_v + 255) / 256; if (b > 148 * 8) b = 148 * 8;
    variant_expand_kernel<<<(int)b, 256, 0, s>>>(guides, n_seg, seg, descs, doff, vq, vdesc, vguide, vfmask);
    return cudaGetLastError();
}

// matches of the edited guides -> matches of the guides (appended to `out`); alignments that substituted an inserted
// character are dropped
__global__ void variant_rewrite_kernel(const MatchRec* __restrict__ vm, uint32_t n_vm, const GuideRec* __restrict__ guides,
                                       const uint32_t* __restrict__ vdesc, const uint32_t* __restrict__ vguide,
                                       MatchRec* __restrict__ out, uint32_t out_cap, uint32_t* out_count, uint32_t* guide_nmatch, uint32_t* error_flag) {
    const uint32_t lane = threadIdx.x & 31u;
    const uint32_t n_round = (n_vm + 31u) & ~31u;
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n_round; i += gridDim.x * blockDim.x) {
        MatchRec o; bool ok = false; uint32_t g = 0;
        if (i < n_vm) {
            const MatchRec m = vm[i];
            const uint32_t v = m.task >> 1;
            g = vguide[v];
            ok = variant_rewrite(m, guides[g], vdesc[v], (g << 1) | (m.task & 1u), o);
        }
        const uint32_t mask = __ballot_sync(0xffffffffu, ok);
        if (!mask) continue;
        uint32_t base = 0; const int leader = __ffs(mask) - 1;
        if ((int)lane == leader) base = atomicAdd(out_count, (uint32_t)__popc(mask));
        base = __shfl_sync(0xffffffffu, base, leader);
        if (ok) {
            const uint32_t slot = base + __popc(mask & ((1u << lane) - 1u));
            if (slot < out_cap) { out[slot] = o; atomicAdd(guide_nmatch + g, 1u); }
            else atomicOr(error_flag, GSX_KERR_MATCH_OVERFLOW);
        }
    }
}
cudaError_t launch_variant_rewrite(const MatchRec* vm, uint32_t n_vm, const GuideRec* guides, const uint32_t* vdesc, const uint32_t* vguide,
                                   MatchRec* out, uint32_t out_cap, uint32_t* out_count, uint32_t* guide_nmatch, uint32_t* error_flag, cudaStream_t s) {
    if (!n_vm) return cudaSuccess;
    long b = ((long)n_vm + 255) / 256; if (b > 148 * 8) b = 148 * 8;
    variant_rewrite_kernel<<<(int)b, 256, 0, s>>>(vm, n_vm, guides, vdesc, vguide, out, out_cap, out_count, guide_nmatch, error_flag);
    return cudaGetLastError();
}

// ---------------------------------------------------------------------------------------------------------
// arrange: group by guide, order, de-duplicate, expand
// ---------------------------------------------------------------------------------------------------------
// exclusive scan of in[0..n) into out[0..n], out[n] = total; one block
__global__ void scan_u32_kernel(const uint32_t* in, uint32_t* out, uint32_t n) {
    __shared__ uint32_t s_warp[32];
    __shared__ uint32_t s_carry;
    if (threadIdx.x == 0) s_carry = 0;
    __syncthreads();
    const uint32_t lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = blockDim.x >> 5;
    for (uint32_t base = 0; base < n; base += blockDim.x) {
        uint32_t i = base + threadIdx.x;
        uint32_t v = i < n ? in[i] : 0, x = v;
        for (int o = 1; o < 32; o <<= 1) { uint32_t y = __shfl_up_sync(0xffffffffu, x, o); if (lane >= (uint32_t)o) x += y; }
        if (lane == 31) s_warp[warp] = x;
        __syncthreads();
        if (warp == 0) {
            uint32_t w = lane < nw ? s_warp[lane] : 0, z = w;
            for (int o = 1; o < 32; o <<= 1) { uint32_t y = __shfl_up_sync(0xffffffffu, z, o); if (lane >= (uint32_t)o) z += y; }
            s_warp[lane] = z - w;
        }
        __syncthreads();
        uint32_t carry = s_carry;
        if (i < n) out[i] = carry + s_warp[warp] + x - v;
        __syncthreads();
        if (threadIdx.x == blockDim.x - 1) s_carry = carry + s_warp[warp] + x;
        __syncthreads();
    }
    if (threadIdx.x == 0) out[n] = s_carry;
}

__global__ void scatter_matches_kernel(const MatchRec* matches, uint32_t n_matches, const uint32_t* guide_moff,
                                       uint32_t* cursor, uint32_t* by_guide) {
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n_matches; i += gridDim.x * blockDim.x) {
        uint32_t g = matches[i].task >> 1;
        by_guide[guide_moff[g] + atomicAdd(cursor + g, 1u)] = i;
    }
}

// one warp per guide: rank sort of its matches (typically ~10), duplicates (same bucket and string) die
__global__ void order_matches_kernel(const MatchRec* matches, const uint32_t* guide_moff, const uint32_t* by_guide,
                                     uint32_t n_guides, uint32_t n_dist, uint32_t* sorted, uint32_t* sorted_off,
                                     uint32_t* guide_nhits, uint32_t* count_by_distance) {
    const uint32_t lane = threadIdx.x & 31;
    const uint32_t wid = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, nw = (gridDim.x * blockDim.x) >> 5;
    for (uint32_t g = wid; g < n_guides; g += nw) {
        const uint32_t b = guide_moff[g], s = guide_moff[g + 1] - b;
        for (uint32_t i = lane; i < s; i += 32) {
            const uint32_t mi = by_guide[b + i];
            const MatchRec x = matches[mi];
            uint32_t rank = 0; bool dup = false;
            for (uint32_t j = 0; j < s; j++) {
                const uint32_t mj = by_guide[b + j];
                if (mj == mi) continue;
                int c = match_cmp(matches[mj], x);
                if (c < 0) rank++;
                else if (c == 0) { if (mj < mi) { rank++; dup = true; } }
            }
            sorted[b + rank] = dup ? (mi | 0x80000000u) : mi;
        }
        __syncwarp();
        // hit offsets in sorted order
        uint32_t running = 0;
        for (uint32_t base = 0; base < s; base += 32) {
            uint32_t i = base + lane;
            uint32_t w = 0, d = 0;
            if (i < s) { uint32_t e = sorted[b + i]; if (!(e & 0x80000000u)) { w = matches[e].width; d = matches[e].info & 0xffu; } }
            uint32_t x = w;
            for (int o = 1; o < 32; o <<= 1) { uint32_t y = __shfl_up_sync(0xffffffffu, x, o); if (lane >= (uint32_t)o) x += y; }
            if (i < s) sorted_off[b + i] = running + x - w;
            if (w && d < n_dist) atomicAdd(count_by_distance + (size_t)g * n_dist + d, w);
            running += __shfl_sync(0xffffffffu, x, 31);
        }
        if (lane == 0) guide_nhits[g] = running;
        __syncwarp();
    }
}

// the same for guides with thousands of matches (bulges): one CTA per guide, the O(s^2) rank sort spread over all its
// threads, then warp 0 lays out the hit offsets
__global__ void order_matches_cta_kernel(const MatchRec* matches, const uint32_t* guide_moff, const uint32_t* by_guide,
                                         uint32_t n_guides, uint32_t n_dist, uint32_t* sorted, uint32_t* sorted_off,
                                         uint32_t* guide_nhits, uint32_t* count_by_distance) {
    const uint32_t lane = threadIdx.x & 31;
    for (uint32_t g = blockIdx.x; g < n_guides; g += gridDim.x) {
        const uint32_t b = guide_moff[g], s = guide_moff[g + 1] - b;
        for (uint32_t i = threadIdx.x; i < s; i += blockDim.x) {
            const uint32_t mi = by_guide[b + i];
            const MatchRec x = matches[mi];
            uint32_t rank = 0; bool dup = false;
            for (uint32_t j = 0; j < s; j++) {
                const uint32_t mj = by_guide[b + j];
                if (mj == mi) continue;
                int c = match_cmp(matches[mj], x);
                if (c < 0) rank++;
                else if (c == 0) { if (mj < mi) { rank++; dup = true; } }
            }
            sorted[b + rank] = dup ? (mi | 0x80000000u) : mi;
        }
        __syncthreads();
        if (threadIdx.x < 32) {
            uint32_t running = 0;
            for (uint32_t base = 0; base < s; base += 32) {
                uint32_t i = base + lane;
                uint32_t w = 0, d = 0;
                if (i < s) { uint32_t e = sorted[b + i]; if (!(e & 0x80000000u)) { w = matches[e].width; d = matches[e].info & 0xffu; } }
                uint32_t x = w;
                for (int o = 1; o < 32; o <<= 1) { uint32_t y = __shfl_up_sync(0xffffffffu, x, o); if (lane >= (uint32_t)o) x += y; }
                if (i < s) sorted_off[b + i] = running + x - w;
                if (w && d < n_dist) atomicAdd(count_by_distance + (size_t)g * n_dist + d, w);
                running += __shfl_sync(0xffffffffu, x, 31);
            }
            if (lane == 0) guide_nhits[g] = running;
        }
        __syncthreads();
    }
}

// one warp per sorted match: write its rows
__global__ void expand_hits_kernel(const MatchRec* matches, const uint32_t* guide_moff, const uint32_t* sorted,
                                   const uint32_t* sorted_off, const uint32_t* guide_hoff, uint32_t n_guides,
                                   uint32_t n_sorted, uint32_t* hit_match, uint32_t* hit_row, uint32_t* hit_guide) {
    const uint32_t lane = threadIdx.x & 31;
    const uint32_t wid = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, nw = (gridDim.x * blockDim.x) >> 5;
    for (uint32_t i = wid; i < n_sorted; i += nw) {
        uint32_t e = sorted[i];
        if (e & 0x80000000u) continue;
        const uint32_t g = matches[e].task >> 1;
        const uint32_t base = guide_hoff[g] + sorted_off[i];
        const uint32_t sp = matches[e].sp, w = matches[e].width;
        for (uint32_t r = lane; r < w; r += 32) { hit_match[base + r] = e; hit_row[base + r] = sp + r; hit_guide[base + r] = g; }
    }
}

// ---------------------------------------------------------------------------------------------------------
// locate + coordinates + CFD, one thread per hit
// ---------------------------------------------------------------------------------------------------------
struct DevBlockLoader {
    __device__ __forceinline__ void operator()(const OccBlock* p, uint32_t c[4], uint64_t& hi, uint64_t& lo) const {
        Blk B = ld_block(p); c[0] = B.c0; c[1] = B.c1; c[2] = B.c2; c[3] = B.c3; hi = B.hi; lo = B.lo;
    }
};
__device__ __forceinline__ uint32_t locate_row(const DevStrand& st, uint32_t row, uint32_t* steps) {
    return locate_row_t(st, row, steps, DevBlockLoader());
}

__global__ void locate_score_kernel(LocateArgs a) {
    __shared__ DevStrand s_st[2];
    if (threadIdx.x == 0) { s_st[0] = a.st[0]; s_st[1] = a.st[1]; }
    __syncthreads();
    uint32_t steps = 0;
    for (uint32_t h = blockIdx.x * blockDim.x + threadIdx.x; h < a.n_hits; h += gridDim.x * blockDim.x) {
        const MatchRec m = a.matches[a.hit_match[h]];
        uint32_t sa = locate_row(s_st[m.task & 1u], a.hit_row[h], &steps);
        score_hit(a, h, m, sa, c_cfd_mm, c_cfd_pam);
    }
    for (int o = 16; o; o >>= 1) steps += __shfl_xor_sync(0xffffffffu, steps, o);
    if ((threadIdx.x & 31) == 0 && steps) atomicAdd(a.stats + 3, (unsigned long long)steps);
}

// one thread per guide: float32 running sum in the reference's output order (batches with a dozen hits per guide)
__global__ void specificity_kernel(SpecArgs a) {
    for (uint32_t g = blockIdx.x * blockDim.x + threadIdx.x; g < a.n_guides; g += gridDim.x * blockDim.x) guide_specificity(a, g);
}
// One WARP per guide, for batches with hundreds or thousands of hits per guide (bulges: 14 k; repeat-family and low-complexity
// guides): the per-thread form walks its hits one dependent load at a time (8.7 ms for 512 bulge guides, a third of the device time on
// the skew stressor).  Here the lanes fetch 32 consecutive hits at once; which of them the reference's loop visits before its
// max_off_targets cut (printer.hpp:129 / :259) is a prefix count (ballot); the float32 additions then happen in hit order, one lane's
// value after the other, so the sum has the reference's rounding (same statement as gsx_core.h guide_specificity, checked against it
// by the golden tests in both forms).
__global__ void specificity_warp_kernel(SpecArgs a) {
    const uint32_t lane = threadIdx.x & 31u, FULL = 0xffffffffu;
    const uint32_t warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, n_warps = (gridDim.x * blockDim.x) >> 5;
    for (uint32_t g = warp; g < a.n_guides; g += n_warps) {
        const uint32_t b = a.guide_hoff[g], n = a.guide_hoff[g + 1] - b;
        float cfd_sum = 0.0f; bool perfect = false;
        uint32_t i = 0;
        for (uint32_t d = 0; d < a.n_dist; d++) {
            const uint32_t cnt = a.count_by_distance[(size_t)g * a.n_dist + d];
            long long n_off = 0;                                                  // resolved hits of this distance so far (SAM rule)
            bool cut = false;                                                     // the reference's loop has hit its `break`
            for (uint32_t j0 = 0; j0 < cnt && !cut; j0 += 32u) {
                const uint32_t j = j0 + lane;
                const bool in = j < cnt;
                const uint32_t h = b + i + j;
                uint8_t fl = 0; int32_t chr = -1; float c = 0.0f;
                if (in) { fl = a.flags[h]; chr = a.chr[h]; c = a.cfd[h]; }
                const bool resolved = in && chr >= 0;
                const uint32_t rmask = __ballot_sync(FULL, resolved);
                // visited: the loop reaches hit j (every hit before the cut is looked at, resolved or not)
                bool visited = in;
                if (a.max_off_targets != -1) {
                    if (a.sam_rule) visited = in && n_off + (long long)__popc(rmask & ((1u << lane) - 1u)) < (long long)a.max_off_targets;
                    else visited = in && (long long)j < (long long)a.max_off_targets;
                }
                const uint32_t vmask = __ballot_sync(FULL, visited);
                if (__ballot_sync(FULL, visited && (fl & 1))) perfect = true;
                const bool add = visited && resolved;
                uint32_t amask = __ballot_sync(FULL, add);
                if (add) a.counted[h] = 1;
                n_off += __popc(amask);
                // the additions, in hit order (every lane keeps the same running sum)
                while (amask) {
                    const int src = __ffs(amask) - 1; amask &= amask - 1u;
                    cfd_sum += __shfl_sync(FULL, c, src);
                }
                if (vmask != __ballot_sync(FULL, in)) cut = true;                 // some hit of this chunk was not visited: the loop has broken
            }
            i += cnt;
        }
        float spec = 0.0f;
        if (n == 0 && !a.sam_rule) spec = 1.0f;                                   // NA row, printer.hpp:190-199
        else { if (!perfect) cfd_sum += 1.0f; if (cfd_sum > 0.0f) spec = 1.0f / cfd_sum; }
        if (lane == 0) { a.specificity[g] = spec; a.perfect[g] = perfect ? 1 : 0; }
    }
}

__global__ void threshold_kernel(const unsigned long long* guide_count, uint8_t* dropped, uint32_t n_guides) {
    for (uint32_t g = blockIdx.x * blockDim.x + threadIdx.x; g < n_guides; g += gridDim.x * blockDim.x)
        dropped[g] = guide_count[g] > 1ull ? 1 : 0;                               // process.hpp:68,70
}

// primitive queries for parity tests
__global__ void rank_query_kernel(DevStrand st, const uint32_t* rows, const uint8_t* syms, uint32_t n, uint32_t* out) {
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        uint32_t row = rows[i], s = syms[i], r = 0;
        if (s < 4) {
            Blk B = ld_block(block_ptr(st, row >> 6));
            uint32_t c[4] = {B.c0, B.c1, B.c2, B.c3}, o[4];
            block_occ(st, c, B.hi, B.lo, row, o);
            r = o[s];
        } else if (s == SYM_N) r = rank_n(st, row);
        out[i] = r;
    }
}
__global__ void locate_query_kernel(DevStrand st, const uint32_t* rows, uint32_t n, uint32_t* out) {
    uint32_t steps = 0;
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) out[i] = locate_row(st, rows[i], &steps);
}

// ---------------------------------------------------------------------------------------------------------
// host-side launchers
// ---------------------------------------------------------------------------------------------------------
static inline int grid_for(uint32_t n, int threads, int cap) { long b = ((long)n + threads - 1) / threads; if (b < 1) b = 1; if (b > cap) b = cap; return (int)b; }

cudaError_t launch_scan(const uint32_t* in, uint32_t* out, uint32_t n, cudaStream_t s) {
    scan_u32_kernel<<<1, 1024, 0, s>>>(in, out, n); return cudaGetLastError();
}
cudaError_t launch_scatter(const MatchRec* m, uint32_t n, const uint32_t* moff, uint32_t* cursor, uint32_t* by_guide, cudaStream_t s) {
    if (!n) return cudaSuccess;
    scatter_matches_kernel<<<grid_for(n, 256, 148 * 8), 256, 0, s>>>(m, n, moff, cursor, by_guide); return cudaGetLastError();
}
cudaError_t launch_order(const MatchRec* m, const uint32_t* moff, const uint32_t* by_guide, uint32_t n_guides, uint32_t n_dist,
                         uint32_t* sorted, uint32_t* sorted_off, uint32_t* nhits, uint32_t* cbd, bool many_per_guide, cudaStream_t s) {
    if (many_per_guide) order_matches_cta_kernel<<<grid_for(n_guides, 1, 148 * 8), 256, 0, s>>>(m, moff, by_guide, n_guides, n_dist, sorted, sorted_off, nhits, cbd);
    else order_matches_kernel<<<grid_for(n_guides * 32u, 256, 148 * 8), 256, 0, s>>>(m, moff, by_guide, n_guides, n_dist, sorted, sorted_off, nhits, cbd);
    return cudaGetLastError();
}
cudaError_t launch_expand(const MatchRec* m, const uint32_t* moff, const uint32_t* sorted, const uint32_t* sorted_off, const uint32_t* hoff,
                          uint32_t n_guides, uint32_t n_sorted, uint32_t* hit_match, uint32_t* hit_row, uint32_t* hit_guide, cudaStream_t s) {
    if (!n_sorted) return cudaSuccess;
    expand_hits_kernel<<<grid_for(n_sorted * 32u, 256, 148 * 8), 256, 0, s>>>(m, moff, sorted, sorted_off, hoff, n_guides, n_sorted, hit_match, hit_row, hit_guide);
    return cudaGetLastError();
}
cudaError_t launch_locate_score(const LocateArgs& a, cudaStream_t s) {
    if (!a.n_hits) return cudaSuccess;
    locate_score_kernel<<<grid_for(a.n_hits, 128, 148 * 16), 128, 0, s>>>(a); return cudaGetLastError();
}
cudaError_t launch_specificity(const SpecArgs& a, cudaStream_t s) {
    if (a.warp_per_guide) specificity_warp_kernel<<<grid_for(a.n_guides * 32u, 128, 148 * 16), 128, 0, s>>>(a);
    else specificity_kernel<<<grid_for(a.n_guides, 128, 148 * 8), 128, 0, s>>>(a);
    return cudaGetLastError();
}
cudaError_t launch_threshold(const unsigned long long* gc, uint8_t* dropped, uint32_t n, cudaStream_t s) {
    threshold_kernel<<<grid_for(n, 256, 148 * 4), 256, 0, s>>>(gc, dropped, n); return cudaGetLastError();
}
// Small mid-pipeline read-backs (error flags and counts after a search launch, the hit total before the result arrays are
// sized) go through a kernel that stores into pinned host memory instead of a cudaMemcpy: a copy would queue on the copy engine
// behind the bulk result transfer of the PREVIOUS call when calls are pipelined (gsx_enumerate_start) -- measured: 12 ms of
// waiting per 200 k-guide batch with two batches in flight.
__global__ void publish_kernel(const uint32_t* __restrict__ src, uint32_t n, volatile uint32_t* dst) {
    if (threadIdx.x < n) dst[threadIdx.x] = src[threadIdx.x];
}
cudaError_t launch_publish(const uint32_t* src, uint32_t n_words, uint32_t* host_dst, cudaStream_t s) {
    publish_kernel<<<1, 32, 0, s>>>(src, n_words < 32u ? n_words : 32u, host_dst);
    return cudaGetLastError();
}
// 64-bit total and maximum of n 32-bit counts, stored into pinned host memory (dst[0], dst[1]); scratch[0..1] and *done must be zero
__global__ void total_u32_kernel(const uint32_t* __restrict__ in, uint32_t n, unsigned long long* scratch, unsigned int* done, volatile unsigned long long* dst) {
    unsigned long long acc = 0; uint32_t mx = 0;
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) { const uint32_t v = in[i]; acc += v; mx = v > mx ? v : mx; }
    for (int o = 16; o; o >>= 1) { acc += __shfl_xor_sync(0xffffffffu, acc, o); const uint32_t t = __shfl_xor_sync(0xffffffffu, mx, o); mx = t > mx ? t : mx; }
    if ((threadIdx.x & 31) == 0 && acc) { atomicAdd(scratch, acc); atomicMax(scratch + 1, (unsigned long long)mx); }
    __syncthreads();
    if (threadIdx.x == 0) {
        __threadfence();
        if (atomicAdd(done, 1u) == gridDim.x - 1) { __threadfence(); dst[0] = atomicAdd(scratch, 0ull); dst[1] = atomicAdd(scratch + 1, 0ull); }      // last block out publishes
    }
}
cudaError_t launch_total_u32(const uint32_t* in, uint32_t n, unsigned long long* scratch, unsigned int* done, unsigned long long* host_dst, cudaStream_t s) {
    const int blocks = (int)((n + 1023u) / 1024u < 1u ? 1u : ((n + 1023u) / 1024u > 296u ? 296u : (n + 1023u) / 1024u));
    total_u32_kernel<<<blocks, 256, 0, s>>>(in, n, scratch, done, host_dst);
    return cudaGetLastError();
}
// order-independent 64-bit digest of a device array (4-byte words, each mixed with its position): equal arrays <=> equal digests
// for all practical purposes; used to check that the index replicas on several devices are byte-identical
__global__ void checksum_kernel(const uint32_t* __restrict__ p, size_t n_words, unsigned long long seed, unsigned long long* out) {
    unsigned long long acc = 0;
    for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < n_words; i += (size_t)gridDim.x * blockDim.x) {
        unsigned long long x = (unsigned long long)p[i] + (i + 1) * 0x9E3779B97F4A7C15ull + seed;
        x ^= x >> 31; x *= 0xBF58476D1CE4E5B9ull; x ^= x >> 29; x *= 0x94D049BB133111EBull; x ^= x >> 32;
        acc += x;
    }
    for (int o = 16; o; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
    if ((threadIdx.x & 31) == 0) atomicAdd(out, acc);
}
cudaError_t launch_checksum(const void* p, size_t bytes, unsigned long long seed, unsigned long long* out, cudaStream_t s) {
    if (bytes < 4) return cudaSuccess;
    checksum_kernel<<<148 * 8, 256, 0, s>>>(reinterpret_cast<const uint32_t*>(p), bytes / 4, seed, out);
    return cudaGetLastError();
}
cudaError_t launch_rank_query(const DevStrand& st, const uint32_t* rows, const uint8_t* syms, uint32_t n, uint32_t* out, cudaStream_t s) {
    rank_query_kernel<<<grid_for(n, 256, 148 * 8), 256, 0, s>>>(st, rows, syms, n, out); return cudaGetLastError();
}
cudaError_t launch_locate_query(const DevStrand& st, const uint32_t* rows, uint32_t n, uint32_t* out, cudaStream_t s) {
    locate_query_kernel<<<grid_for(n, 128, 148 * 16), 128, 0, s>>>(st, rows, n, out); return cudaGetLastError();
}

}  // namespace gsx
