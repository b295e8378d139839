// gsx_core.h -- per-node arithmetic of the search, shared verbatim by the CUDA kernels and by the host-side
// unit tests of this arithmetic (tests/host_core_check.cpp).  Nothing here is a CPU fallback of the product: the
// product only ever calls these from device code.
//
// Semantics follow the reference's three recursions in include/genomics/index.hpp (125-170 PAM / wildcard
// stage, 182-248 mismatch-only, 250-375 bulge-aware); the traversal ORDER differs (children are explored in
// parallel), the set of emitted (string, sp, ep, mismatches, dna, rna) tuples does not.
#ifndef GSX_CORE_H
#define GSX_CORE_H
#include "gsx_types.h"
#include "gsx_kernels.h"

namespace gsx {

GSX_HD uint32_t popc64(uint64_t v) {
#if defined(__CUDA_ARCH__)
    return (uint32_t)__popcll(v);
#else
    return (uint32_t)__builtin_popcountll(v);
#endif
}

GSX_HD uint32_t lower_bound_u32(const uint32_t* a, uint32_t n, uint32_t v) {   // first index with a[idx] >= v
    uint32_t lo = 0, hi = n;
    while (lo < hi) {
        uint32_t mid = (lo + hi) >> 1;
        if (a[mid] < v) lo = mid + 1; else hi = mid;
    }
    return lo;
}

// number of exception rows in [start, i)
GSX_HD uint32_t exc_in(const DevStrand& st, uint32_t start, uint32_t i) {
    if (i <= st.exc_lo || start > st.exc_hi) return 0;
    if (st.n_exc == 1) return 1;        // exc_lo == exc_hi lies in [start, i)
    return lower_bound_u32(st.exc_rows, st.n_exc, i) - lower_bound_u32(st.exc_rows, st.n_exc, start);
}

// the same count for the block of row i, [i - (i & 63), i), behind a one-bit-per-block map of the blocks that hold any exception
// row (search_fast_kernel<..., EXC>: on a genome with N almost every block of the A/C/G/T ranges is clean, so the table is
// searched for a few lookups only)
GSX_HD uint32_t exc_before(const uint32_t* map, const uint32_t* rows, uint32_t n_exc, uint32_t i) {
    const uint32_t b = i >> 6, r = i & 63u;
    if (r == 0u || !((map[b >> 5] >> (b & 31u)) & 1u)) return 0u;
    return lower_bound_u32(rows, n_exc, i) - lower_bound_u32(rows, n_exc, i - r);
}

// occurrences of 'N' in BWT[0, i)
GSX_HD uint32_t rank_n(const DevStrand& st, uint32_t i) { return lower_bound_u32(st.n_rows, st.n_nrows, i); }

// occ(c, i) for c = A,C,G,T from the block that holds row i  (= csa.rank_bwt(i, c), sdsl csa_wt.hpp:270-273)
GSX_HD void block_occ(const DevStrand& st, const uint32_t cnt[4], uint64_t bhi, uint64_t blo, uint32_t i, uint32_t o[4]) {
    uint32_t r = i & 63u;
    uint64_t mask = r ? (~0ull >> (64 - r)) : 0ull;
    uint64_t hi = bhi & mask, lo = blo & mask;
    uint32_t t = popc64(hi & lo);
    uint32_t g = popc64(hi) - t;
    uint32_t c = popc64(lo) - t;
    uint32_t a = r - t - g - c;                   // rows below r with code 0, exceptions included ...
    if (st.n_exc) a -= exc_in(st, i - r, i);      // ... and removed here
    o[0] = cnt[0] + a; o[1] = cnt[1] + c; o[2] = cnt[2] + g; o[3] = cnt[3] + t;
}

// BWT symbol code of a non-exception row
GSX_HD uint32_t block_sym(uint64_t bhi, uint64_t blo, uint32_t row) {
    uint32_t r = row & 63u;
    return (uint32_t)(((bhi >> r) & 1ull) << 1 | ((blo >> r) & 1ull));
}

// ---- string sort keys --------------------------------------------------------------------------------
// The reference orders the matches of one guide/strand/mismatch bucket by std::string comparison of the consumed
// characters (structures.hpp:43); in ASCII '.' < 'A' < 'C' < 'G' < 'N' < 'T' < 'a' < 'c' < 'g' < 't'.
//   narrow key (no bulges, qlen + plen <= 27): base-5 number, one digit per character. Protospacer position:
//     0 = the guide's own (upper-case) character, 1..4 = lower-case a,c,g,t. PAM position: A,C,G,N,T = 0..4.
//   wide key (bulges): 4 bits per character, '.'=1 A=2 C=3 G=4 N=5 T=6 a=7 c=8 g=9 t=10, left aligned in 128 bits.
GSX_HD uint32_t wide_upper_digit(uint32_t s) { return s < 3 ? 2 + s : (s == 3 ? 6u : 5u); }   // s: 0..3 ACGT, 4 N

template <bool WIDE>
GSX_HD void key_append(Node& n, uint32_t digit) {
    if (WIDE) {
        n.key_hi = (n.key_hi << 4) | (n.key_lo >> 60);
        n.key_lo = (n.key_lo << 4) | digit;
    } else {
        n.key_lo = n.key_lo * 5ull + digit;
    }
}

GSX_HD void key_left_align(uint64_t& hi, uint64_t& lo, uint32_t len) {   // wide key: shift left by 4*(32-len) bits
    uint32_t sh = 4u * (32u - len);
    if (sh == 0) return;
    if (sh >= 64) { hi = sh == 64 ? lo : (lo << (sh - 64)); lo = 0; }
    else { hi = (hi << sh) | (lo >> (64 - sh)); lo <<= sh; }
}

struct ExpandCtx {
    const DevStrand* st;
    const GuideRec* g;
    const PamSet* ps;
    uint32_t M, R, D;
};

// candidate children of one node
enum : int {
    CAND_SYM0 = 0,        // 0..3: consume genome symbol A,C,G,T (exact / mismatch / PAM character)
    CAND_LITN = 4,        // consume a literal genome 'N' (query character or PAM pattern character is N)
    CAND_FORK = 5,        // same node for the next alternative PAM
    CAND_DNA0 = 6,        // 6..9: DNA bulge consuming A,C,G,T            (bulge kernels only)
    CAND_RNA = 10,        // RNA bulge                                    (bulge kernels only)
    CAND_SELF = 11,       // emit the node itself (bulge kernels, guide without PAM)
    CAND_END = 12
};

GSX_HD uint32_t meta_lvl(uint32_t m) { return m & META_LVL_MASK; }
GSX_HD uint32_t meta_mm(uint32_t m) { return (m >> META_MM_SHIFT) & 7u; }
GSX_HD uint32_t meta_pam(uint32_t m) { return (m >> META_PAM_SHIFT) & 7u; }
GSX_HD uint32_t meta_dna(uint32_t m) { return (m >> META_DNA_SHIFT) & 7u; }
GSX_HD uint32_t meta_rna(uint32_t m) { return (m >> META_RNA_SHIFT) & 7u; }
GSX_HD uint32_t meta_state(uint32_t m) { return (m >> META_STATE_SHIFT) & 3u; }
GSX_HD uint32_t meta_curr(uint32_t m) { return (m >> META_CURR_SHIFT) & 1u; }
GSX_HD uint32_t meta_make(uint32_t lvl, uint32_t mm, uint32_t pam, uint32_t dna, uint32_t rna, uint32_t state, uint32_t curr) {
    return lvl | (mm << META_MM_SHIFT) | (pam << META_PAM_SHIFT) | (dna << META_DNA_SHIFT) | (rna << META_RNA_SHIFT) |
           (state << META_STATE_SHIFT) | (curr << META_CURR_SHIFT);
}

// Evaluates candidate `cand` of node `nd`.  os / oe = occ(A,C,G,T) at nd.sp and at nd.ep + 1.
// Returns false if the candidate does not exist; otherwise fills `ch` and sets `emit` when the child is a
// finished alignment (it is then reported as a match and never expanded).
template <bool WIDE>
GSX_HD bool make_child(int cand, const Node& nd, const ExpandCtx& cx, const uint32_t os[4], const uint32_t oe[4],
                       Node& ch, bool& emit) {
    const uint32_t meta = nd.meta;
    const uint32_t lvl = meta_lvl(meta), mm = meta_mm(meta), pam = meta_pam(meta);
    const uint32_t dna = meta_dna(meta), rna = meta_rna(meta), state = meta_state(meta), curr = meta_curr(meta);
    const uint32_t qlen = cx.g->qlen;
    const bool in_proto = lvl < qlen;
    emit = false;
    ch = nd;

    if (cand < 4 || cand == CAND_LITN) {
        uint32_t s = (uint32_t)cand;                 // 0..3, or 4 for N
        uint32_t nmm = mm, digit;
        if (in_proto) {
            uint32_t c = cx.g->q[lvl];
            bool exact = c == s;
            if (cand == CAND_LITN) { if (!exact) return false; }
            else if (!exact) { if (mm >= cx.M) return false; nmm = mm + 1; }        // index.hpp:226, 331
            digit = WIDE ? (exact ? wide_upper_digit(s) : 7u + s) : (exact ? 0u : 1u + s);
        } else {
            uint32_t j = lvl - qlen;
            if (j >= cx.ps->plen[pam]) return false;
            uint32_t pc = cx.ps->sym[pam][j];
            if (cand == CAND_LITN) { if (pc != SYM_N) return false; }
            else if (!(pc == s || pc == SYM_N || (pc == SYM_CLS && ((cx.ps->cmask[pam][j] >> s) & 1u)))) return false;   // index.hpp:151-168 with mismatches = 0
                                                                                    // (a class: its members only, never a literal N)
            digit = WIDE ? wide_upper_digit(s) : (s < 3 ? s : (s == 3 ? 4u : 3u));
        }
        uint32_t o_s, o_e;
        if (cand == CAND_LITN) {
            if (cx.st->n_nrows == 0) return false;
            o_s = rank_n(*cx.st, nd.sp); o_e = rank_n(*cx.st, nd.ep + 1);
        } else { o_s = os[s]; o_e = oe[s]; }
        uint32_t within = o_e - o_s;
        if (within == 0) return false;
        ch.sp = cx.st->C[s] + o_s;
        ch.ep = ch.sp + within - 1;
        key_append<WIDE>(ch, digit);
        uint32_t nl = lvl + 1;
        uint32_t npam = nl <= qlen ? 0u : pam;
        ch.meta = meta_make(nl, nmm, npam, dna, rna, in_proto ? 0u : state, curr);   // state -> none, curr kept (index.hpp:319-320)
        emit = (nl == qlen + cx.ps->plen[npam]) && !(WIDE && nl == qlen);
        return true;
    }
    if (cand == CAND_FORK) {
        if (lvl != qlen || pam + 1 >= cx.ps->n_pams) return false;                  // for (pam : pams) index.hpp:210-212
        ch.meta = meta_make(lvl, mm, pam + 1, dna, rna, state, curr);
        return true;
    }
    if (!WIDE) return false;
    if (cand >= CAND_DNA0 && cand < CAND_DNA0 + 4) {                                // index.hpp:265-296
        if (lvl > qlen) return false;
        uint32_t d_state = state, d_curr = curr, d_dna = dna;
        if (cx.D > dna) { if (state != 1u || d_curr == 1u) { d_state = 1; d_curr = 0; d_dna = dna + 1; } }
        if (!(d_state == 1u && d_curr < 1u && lvl != 0)) return false;              // position != query.length() - 1
        d_curr += 1;
        uint32_t s = (uint32_t)(cand - CAND_DNA0);
        uint32_t within = oe[s] - os[s];
        if (within == 0) return false;
        ch.sp = cx.st->C[s] + os[s];
        ch.ep = ch.sp + within - 1;
        key_append<WIDE>(ch, 7u + s);
        ch.meta = meta_make(lvl, mm, pam, d_dna, rna, d_state, d_curr);
        return true;
    }
    if (cand == CAND_RNA) {                                                         // index.hpp:352-368
        if (!in_proto) return false;
        uint32_t r_state = state, r_curr = curr, r_rna = rna;
        if (cx.R > rna) { if (state != 2u || r_curr == 1u) { r_state = 2; r_curr = 0; r_rna = rna + 1; } }
        if (!(r_state == 2u && r_curr < 1u && lvl != 0)) return false;
        r_curr += 1;
        key_append<WIDE>(ch, 1u);
        ch.meta = meta_make(lvl + 1, mm, 0, dna, r_rna, r_state, r_curr);
        return true;
    }
    if (cand == CAND_SELF) {
        if (lvl != qlen || cx.ps->plen[pam] != 0) return false;                     // empty PAM: emit at position < 0
        emit = true;
        return true;
    }
    return false;
}

GSX_HD uint32_t string_len(uint32_t meta) { return meta_lvl(meta) + meta_dna(meta); }

GSX_HD void fill_match(MatchRec& m, const Node& ch, bool wide) {
    uint32_t len = string_len(ch.meta);
    uint64_t hi = ch.key_hi, lo = ch.key_lo;
    if (wide) key_left_align(hi, lo, len); else hi = 0;
    m.key_hi = hi; m.key_lo = lo; m.task = ch.task; m.sp = ch.sp; m.width = ch.ep - ch.sp + 1;
    m.info = meta_mm(ch.meta) | (meta_dna(ch.meta) << 8) | (meta_rna(ch.meta) << 16) | (len << 24);
}

// ---- bulges as edited guides -----------------------------------------------------------------------------------------
// With max_bulge_size = 1 (hard-wired by the reference, process.hpp:82-87) the bulge-aware recursion (index.hpp:250-375)
// reduces to: walk the guide in consumption order; before position lvl >= 1 (and once more after the last position, before
// the PAM) any number of DNA bulges may consume one arbitrary genome character each, written in lower case, at no mismatch
// cost; position lvl >= 1 may be skipped without consuming anything (RNA bulge, written '.'); every such step needs budget
// (dna < D, rna < R), nothing else -- `state` / `curr_bulge_size` only ever matter for bulges longer than one.
// Hence: alignments of the guide with bulges = union, over every op list within the budgets, of the MISMATCH-ONLY
// alignments of an edited guide (skipped positions removed, inserted positions holding a concrete character that must
// match exactly).  The edited guides run through the specialised kernels like any other guide; variant_rewrite turns
// their matches back into the reference's strings.  Different op lists can spell the same string (then with the same
// counts and the same interval): the collector's de-duplication on the string takes care of it, as std::set does.
//   op byte (up to four per variant, first op in the low byte, 0 = none): lvl | kind << 5 | sym << 6
//     kind 0 = RNA bulge: guide position lvl is skipped;  kind 1 = DNA bulge: genome symbol sym consumed before position lvl
//   ops are ordered by lvl, DNA bulges of a level before its skip.
GSX_HD uint32_t variant_op(uint32_t lvl, uint32_t kind, uint32_t sym) { return lvl | (kind << 5) | (sym << 6); }

// the edited guide: 2-bit symbols in consumption order | length << 58; q = the guide's own symbols (all < 4)
GSX_HD uint64_t variant_pack(const uint8_t* q, uint32_t qlen, uint32_t desc) {
    uint64_t v = 0; uint32_t n = 0;
    for (uint32_t lvl = 0; lvl <= qlen; lvl++) {
        while ((desc & 0xFFu) && (desc & 31u) == lvl && (desc & 32u)) { v |= (uint64_t)((desc >> 6) & 3u) << (2u * n); n++; desc >>= 8; }
        if (lvl == qlen) break;
        if ((desc & 0xFFu) && (desc & 31u) == lvl) { desc >>= 8; continue; }              // skipped
        v |= (uint64_t)(q[lvl] & 3u) << (2u * n); n++;
    }
    return v | ((uint64_t)n << 58);
}

// inserted (must-match) positions of the edited guide as a mask over the 2-bit fields of a jump-table index: bits 2f, 2f+1 set
// for every inserted position f < 16.  A pattern that substitutes such a position can only lead to alignments variant_rewrite
// drops, so the sweep may skip it (sweep_kernel<..., FORCED>).
GSX_HD uint32_t variant_forced_mask(uint32_t qlen, uint32_t desc) {
    uint32_t m = 0, n = 0;
    for (uint32_t lvl = 0; lvl <= qlen; lvl++) {
        while ((desc & 0xFFu) && (desc & 31u) == lvl && (desc & 32u)) { if (n < 16u) m |= 3u << (2u * n); n++; desc >>= 8; }
        if (lvl == qlen) break;
        if ((desc & 0xFFu) && (desc & 31u) == lvl) { desc >>= 8; continue; }
        n++;
    }
    return m;
}
// does table index idx keep the guide's own characters at the forced positions?  (the patterns the sweep still has to visit)
GSX_HD bool forced_kept(uint32_t idx, uint64_t q, uint32_t fmask) { return ((idx ^ (uint32_t)q) & fmask) == 0u; }

// match of an edited guide (narrow key over its own characters) -> match of the guide itself (wide key, bulge counts);
// false if an inserted position was matched by substitution (that alignment belongs to the variant holding the other symbol)
GSX_HD bool variant_rewrite(const MatchRec& in, const GuideRec& g, uint32_t desc, uint32_t real_task, MatchRec& out) {
    const uint32_t vlen = in.info >> 24;
    uint8_t dg[40];
    { uint64_t k = in.key_lo; for (uint32_t i = vlen; i-- > 0;) { dg[i] = (uint8_t)(k % 5ull); k /= 5ull; } }
    Node acc; acc.key_lo = acc.key_hi = 0;
    uint32_t vl = 0, len = 0, dna = 0, rna = 0;
    const uint32_t qlen = g.qlen;
    for (uint32_t lvl = 0; lvl <= qlen; lvl++) {
        while ((desc & 0xFFu) && (desc & 31u) == lvl && (desc & 32u)) {
            if (dg[vl] != 0) return false;
            key_append<true>(acc, 7u + ((desc >> 6) & 3u)); vl++; len++; dna++; desc >>= 8;
        }
        if (lvl == qlen) break;
        if ((desc & 0xFFu) && (desc & 31u) == lvl) { key_append<true>(acc, 1u); len++; rna++; desc >>= 8; continue; }
        const uint32_t d = dg[vl++];
        key_append<true>(acc, d == 0 ? wide_upper_digit(g.q[lvl]) : 6u + d); len++;
    }
    for (; vl < vlen; vl++) { const uint32_t d = dg[vl]; key_append<true>(acc, d < 3u ? 2u + d : (d == 3u ? 5u : 6u)); len++; }   // PAM: A,C,G,N,T
    key_left_align(acc.key_hi, acc.key_lo, len);
    out.key_hi = acc.key_hi; out.key_lo = acc.key_lo; out.task = real_task; out.sp = in.sp; out.width = in.width;
    out.info = (in.info & 0xffu) | (dna << 8) | (rna << 16) | (len << 24);
    return true;
}

// ---- decoding a match back into the reference's match.sequence ---------------------------------------------
GSX_HD char sym_char(uint32_t s) { return s == 0 ? 'A' : s == 1 ? 'C' : s == 2 ? 'G' : s == 3 ? 'T' : s == 4 ? 'N' : '?'; }
GSX_HD char complement_char(char c) {                                               // sequences.cxx:14-28
    switch (c) {
    case 'A': return 'T'; case 'T': return 'A'; case 'C': return 'G'; case 'G': return 'C';
    case 'a': return 't'; case 't': return 'a'; case 'c': return 'g'; case 'g': return 'c';
    default: return c;
    }
}

// out receives match.sequence (the consumed characters, pre-complement); returns its length (<= 32)
GSX_HD uint32_t decode_match(const MatchRec& m, const GuideRec& g, bool wide, char* out) {
    uint32_t len = m.info >> 24;
    if (wide) {
        uint64_t hi = m.key_hi, lo = m.key_lo;
        for (uint32_t i = 0; i < len; i++) {
            uint32_t d = (uint32_t)(hi >> 60);
            hi = (hi << 4) | (lo >> 60); lo <<= 4;
            out[i] = d == 1 ? '.' : d == 2 ? 'A' : d == 3 ? 'C' : d == 4 ? 'G' : d == 5 ? 'N' : d == 6 ? 'T'
                   : d == 7 ? 'a' : d == 8 ? 'c' : d == 9 ? 'g' : d == 10 ? 't' : '?';
        }
    } else {
        uint64_t k = m.key_lo;
        for (uint32_t ii = 0; ii < len; ii++) {
            uint32_t i = len - 1 - ii;
            uint32_t d = (uint32_t)(k % 5ull); k /= 5ull;
            if (i < g.qlen) out[i] = d == 0 ? sym_char(g.q[i]) : (d == 1 ? 'a' : d == 2 ? 'c' : d == 3 ? 'g' : 't');
            else out[i] = d == 0 ? 'A' : d == 1 ? 'C' : d == 2 ? 'G' : d == 3 ? 'N' : 'T';
        }
    }
    return len;
}

GSX_HD int cfd_base(char c) { return c == 'A' ? 0 : c == 'C' ? 1 : c == 'G' ? 2 : c == 'T' ? 3 : -1; }
GSX_HD char upper_char(char c) { return (c >= 'a' && c <= 'z') ? (char)(c - 32) : c; }

// calculate_cfd (printer.hpp:98-113) on match_sequence = complement(match.sequence).
// mmtab[4][4][20] / pamtab[4][4]: flat double tables (missing key => 0.0).
GSX_HD float cfd_score(const char* sgrna, uint32_t sglen, const char* match_seq, uint32_t mlen,
                       const double* mmtab, const double* pamtab) {
    uint32_t plen = mlen < 20 ? 0 : (mlen - 20 < 3 ? mlen - 20 : 3);
    if (sglen != 20 || plen != 3) return 1.0f;
    float cfd = 1.0f;
    for (int i = 0; i < 20; i++) {
        char a = sgrna[i], b = match_seq[i];
        if (a != b) {
            int r = a == 'U' ? 3 : cfd_base(a);
            int d = cfd_base(upper_char(complement_char(b)));
            double v = (r >= 0 && d >= 0) ? mmtab[(r * 4 + d) * 20 + i] : 0.0;
            cfd = (float)((double)cfd * v);
        }
    }
    int p1 = cfd_base(match_seq[21]), p2 = cfd_base(match_seq[22]);
    double pv = (p1 >= 0 && p2 >= 0) ? pamtab[p1 * 4 + p2] : 0.0;
    cfd = (float)((double)cfd * pv);
    return cfd;
}

// resolve_absolute (structures.cxx:7-52). chroms: cumulative starts + lengths, zero-length chromosomes can never
// hold a position.  Returns chromosome index or -1 (sentinel).
GSX_HD int resolve_abs(const Chrom* chroms, uint32_t n_chr, int64_t abs, uint32_t seq_len, uint32_t pam_len,
                       uint32_t* pos1, uint8_t* strand) {
    *strand = '+';
    if (abs < 0) { abs = -abs; *strand = '-'; }
    // last chromosome with start <= abs and length > 0 containing abs
    uint32_t lo = 0, hi = n_chr;
    while (lo < hi) { uint32_t mid = (lo + hi) >> 1; if (chroms[mid].start + chroms[mid].length <= (uint64_t)abs) lo = mid + 1; else hi = mid; }
    if (lo >= n_chr) return -1;
    int64_t off = abs - (int64_t)chroms[lo].start;
    int64_t start, end;
    if (*strand == '+') { end = off + 1; start = end - (int64_t)seq_len - (int64_t)pam_len + 1; }
    else { start = off + 1; end = start + (int64_t)seq_len + (int64_t)pam_len - 1; }
    if (start < 0 || end > (int64_t)chroms[lo].length) return -1;
    *pos1 = (uint32_t)start;
    return (int)lo;
}

// csa[row]: LF walk to the next sampled row, then sample + steps (mod n) -- sdsl csa_wt.hpp:333-346,
// suffix_array_helper.hpp:337-349.  `ld` loads one OccBlock (LDG.E.256 on the device).
template <class LoadBlk>
GSX_HD uint32_t locate_row_t(const DevStrand& st, uint32_t row, uint32_t* steps, LoadBlk ld) {
    uint32_t off = 0;
    const uint32_t smask = (1u << st.sa_shift) - 1u;
    while (row & smask) {
        bool is_exc = false;
        if (st.n_exc && row >= st.exc_lo && row <= st.exc_hi) {
            uint32_t j = lower_bound_u32(st.exc_rows, st.n_exc, row);
            if (j < st.n_exc && st.exc_rows[j] == row) { row = st.exc_lf[j]; is_exc = true; }
        }
        if (!is_exc) {
            uint32_t c[4], o[4]; uint64_t hi, lo;
            ld(block_ptr(st, row >> 6), c, hi, lo);
            block_occ(st, c, hi, lo, row, o);
            uint32_t s = block_sym(hi, lo, row);
            row = st.C[s] + o[s];
        }
        off++;
    }
    *steps += off;
    uint64_t v = (uint64_t)st.sa_samples[row >> st.sa_shift] + off;
    return (uint32_t)(v >= st.n ? v - st.n : v);
}

// one located hit: absolute coordinate (process.hpp:104,111), chromosome (structures.cxx:7-52), CFD (printer.hpp:98-113)
GSX_HD void score_hit(const LocateArgs& a, uint32_t h, const MatchRec& m, uint32_t sa, const double* mmtab, const double* pamtab) {
    const uint32_t strand = m.task & 1u;
    const GuideRec& g = a.guides[m.task >> 1];
    const PamSet& ps = a.pamsets[g.pamset];
    int64_t abs = strand == 0 ? -(int64_t)sa : (int64_t)a.genome_length - ((int64_t)sa + 1);
    uint32_t pos1 = 0; uint8_t sc = '+';
    int chr = resolve_abs(a.chroms, a.n_chr, abs, g.seqlen, ps.kpam_len, &pos1, &sc);
    char ms[kMaxQ + kMaxPamLen + 8];
    uint32_t len = decode_match(m, g, a.wide != 0, ms);
    for (uint32_t i = 0; i < len; i++) ms[i] = complement_char(ms[i]);            // match_sequence, printer.hpp:264
    float cfd = cfd_score(g.seq, g.seqlen, ms, len, mmtab, pamtab);
    uint32_t mm = m.info & 0xffu;
    bool perfect = mm == 0 && len >= 23 && ms[21] == 'G' && ms[22] == 'G';        // printer.hpp:276
    a.abs_pos[h] = abs; a.chr[h] = chr; a.pos1[h] = pos1; a.strand[h] = sc;
    a.distance[h] = (uint8_t)mm; a.dna[h] = (uint8_t)((m.info >> 8) & 0xffu); a.rna[h] = (uint8_t)((m.info >> 16) & 0xffu);
    a.index_id[h] = (uint8_t)strand; a.cfd[h] = cfd; a.flags[h] = perfect ? 1 : 0;
    a.key_lo[h] = m.key_lo; a.mlen[h] = (uint8_t)len;
    if (a.key_hi) a.key_hi[h] = m.key_hi;
}

// per-guide float32 reduction in the reference's output order (printer.hpp:244-300 CSV rule / 115-170 SAM rule)
GSX_HD void guide_specificity(const SpecArgs& a, uint32_t g) {
    const uint32_t b = a.guide_hoff[g], n = a.guide_hoff[g + 1] - b;
    float cfd_sum = 0.0f; bool perfect = false;
    uint32_t i = 0;
    for (uint32_t d = 0; d < a.n_dist; d++) {
        const uint32_t cnt = a.count_by_distance[(size_t)g * a.n_dist + d];
        int64_t n_off = 0;
        for (uint32_t j = 0; j < cnt; j++) {
            const uint32_t h = b + i + j;
            if (a.sam_rule) { if (a.max_off_targets != -1 && n_off >= a.max_off_targets) break; }       // printer.hpp:129
            else { if (a.max_off_targets != -1 && (int64_t)j >= a.max_off_targets) break; }              // printer.hpp:259
            if (a.flags[h] & 1) perfect = true;
            if (a.chr[h] < 0) continue;
            cfd_sum += a.cfd[h];
            a.counted[h] = 1;
            n_off++;
        }
        i += cnt;
    }
    float spec = 0.0f;
    if (n == 0 && !a.sam_rule) spec = 1.0f;                                       // NA row, printer.hpp:190-199
    else { if (!perfect) cfd_sum += 1.0f; if (cfd_sum > 0.0f) spec = 1.0f / cfd_sum; }
    a.specificity[g] = spec; a.perfect[g] = perfect ? 1 : 0;
}

// ---- look-ahead pruning (blk_shift = 7 indexes, specialised search kernel) --------------------------------------
// hi[j], lo[j]: bit planes of t_j for the 64 rows of one block, t_0 being the BWT symbol itself.  A backward search
// sitting on row r at level lvl will consume t_0(r), t_1(r), ... against the query characters of levels lvl, lvl+1, ...
// Returns a 4-bit mask: bit s is set iff some row of [sp, ep] (all in this block) with t_0 = s can consume its next
// J = min(7, total - lvl) characters with at most `budget` further protospacer mismatches and every fixed PAM
// character matched.  A child whose bit is clear can never reach the final level, so it is not expanded: the set of
// emitted matches is unchanged.  Planes hold arbitrary symbols where the true one is not A/C/G/T or lies before the
// text start; that can only set bits spuriously (no pruning), never clear one that should be set, because such a
// path cannot be continued by an A/C/G/T query character in the first place.  A class PAM character (code 6) counts as a wildcard
// here: its members always survive, a non-member is only pruned later (the child itself is tested against the class), so the mask
// stays a superset of the exact one at no extra registers on the tree search's hot loop.
GSX_HD uint32_t viable_children(const uint64_t hi[7], const uint64_t lo[7], uint32_t sp, uint32_t ep, uint32_t lvl,
                                uint32_t qlen, uint32_t total, uint64_t q, uint32_t pampack, uint32_t budget) {
    const uint32_t r0 = sp & 63u, r1 = ep & 63u;
    uint64_t rows = (r1 == 63u ? ~0ull : ((1ull << (r1 + 1u)) - 1ull)) & ~((1ull << r0) - 1ull);
    uint64_t c0 = 0, c1 = 0, c2 = 0, dead = 0;          // bit-sliced per-row mismatch counter (0..7)
    const uint32_t left = total - lvl;
#if defined(__CUDA_ARCH__)
#pragma unroll
#endif
    for (uint32_t j = 0; j < 7; j++) {
        if (j < left) {
            const uint32_t L = lvl + j;
            uint32_t sym; bool proto = L < qlen, wild = false, kill = false;
            if (proto) sym = (uint32_t)(q >> (2u * L)) & 3u;
            else { uint32_t pc = (pampack >> (3u * (L - qlen))) & 7u; sym = pc & 3u; wild = pc == 4u || pc == 6u; kill = pc == 5u || pc == 7u; }
            const uint64_t eq = ~(hi[j] ^ ((sym & 2u) ? ~0ull : 0ull)) & ~(lo[j] ^ ((sym & 1u) ? ~0ull : 0ull));
            if (proto) {
                const uint64_t mis = ~eq;
                const uint64_t k0 = c0 & mis; c0 ^= mis;
                const uint64_t k1 = c1 & k0; c1 ^= k0;
                c2 ^= k1;
            } else if (kill) dead = ~0ull;
            else if (!wild) dead |= ~eq;
        }
    }
    const uint64_t B0 = (budget & 1u) ? ~0ull : 0ull, B1 = (budget & 2u) ? ~0ull : 0ull, B2 = (budget & 4u) ? ~0ull : 0ull;
    const uint64_t gt = (c2 & ~B2) | (~(c2 ^ B2) & ((c1 & ~B1) | (~(c1 ^ B1) & (c0 & ~B0))));
    const uint64_t alive = rows & ~dead & ~gt;
    const uint64_t h0 = hi[0], l0 = lo[0];
    return ((alive & ~h0 & ~l0) ? 1u : 0u) | ((alive & ~h0 & l0) ? 2u : 0u) | ((alive & h0 & ~l0) ? 4u : 0u) | ((alive & h0 & l0) ? 8u : 0u);
}

// ---- the row filter of the sweep kernel --------------------------------------------------------------------------------
// The sweep kernel never walks the interval of a level-L pattern: it reads the pattern's SUMMARY (DevStrand::sum0/sum1, indexed
// like the jump table) -- the next seven characters of every row of the interval as bit planes -- and tests all rows at once.
//   codes: per guide, 4 bits per plane j = 0..6 of what a row must show at level L + j: 0..3 = that symbol in the
//          protospacer (anything else costs one mismatch), 8..11 = that symbol in the PAM (anything else kills the row),
//          12 = PAM wildcard, 13 = kills every row, 7 = no such level.  A class PAM character (pampack code 6) is a wildcard here:
//          the sweep only chooses seeds and the tree search behind it tests the class exactly, so this keeps a superset of the
//          seeds and the compiled plane layouts (shape 0 covers NRG, NNGRRT and --start TTTV at 20 nt).
//   u[r]:  rows with at most budget - r mismatches so far (r = 0 .. NB-1, NB > budget); u[0] = rows still alive.
//   One 32-byte sector holds all seven levels for 16 rows (sum0: rows 0..15 of the interval, sum1: rows 16..31), so a single
//          load settles nine nodes out of ten; lanes whose node has more than 16 rows and found nothing among the first 16
//          park it in a per-warp buffer that is drained 32 at a time, all lanes busy.
GSX_HD uint32_t sweep_codes(uint64_t q, uint32_t L, uint32_t plen, uint32_t pampack) {
    const uint32_t qlen = (uint32_t)(q >> 58);
    uint32_t codes = 0;
    for (uint32_t j = 0; j < 7u; j++) {
        const uint32_t Lv = L + j;
        uint32_t c;
        if (Lv < qlen) c = (uint32_t)(q >> (2u * Lv)) & 3u;
        else if (Lv < qlen + plen) { c = (pampack >> (3u * (Lv - qlen))) & 7u; c = c == 6u ? 4u : c > 4u ? 5u : c; c |= 8u; }     // bit 3: PAM level
        else c = 7u;
        codes |= c << (4u * j);
    }
    return codes;
}
// the same for the two levels behind them (L + 7, L + 8): 4 bits each
GSX_HD uint32_t sweep_codes2(uint64_t q, uint32_t L, uint32_t plen, uint32_t pampack) {
    const uint32_t qlen = (uint32_t)(q >> 58);
    uint32_t codes = 0;
    for (uint32_t j = 0; j < 2u; j++) {
        const uint32_t Lv = L + 7u + j;
        uint32_t c;
        if (Lv < qlen) c = (uint32_t)(q >> (2u * Lv)) & 3u;
        else if (Lv < qlen + plen) { c = (pampack >> (3u * (Lv - qlen))) & 7u; c = c == 6u ? 4u : c > 4u ? 5u : c; c |= 8u; }
        else c = 7u;
        codes |= c << (4u * j);
    }
    return codes;
}
GSX_HD bool sweep_has_tail(uint32_t codes2) { return (codes2 & 15u) != 7u; }
enum : uint32_t { SUM_WIDE16 = 1u << 16, SUM_WIDE32 = 1u << 17, SUM_TWO_BLOCKS = 1u << 18 };

// One summary sector = header word + seven plane words.  header: bits 0..15 = valid rows (bit i = row i of the sector's 16
// rows), SUM_WIDE16 = the interval has more than 16 rows (rows 16..31 are in sum1), SUM_WIDE32 = more than 32 rows (not
// summarised: such a node goes to the tree search unexamined), SUM_TWO_BLOCKS = it straddles two 64-row blocks (statistics
// only).  plane word j: bits 0..15 = high bit of the 2-bit symbol t_j of each row, bits 16..31 = its low bit.
// summary_eval: u[r] = rows with at most budget - r mismatches after all seven levels; returns the header.
template <int NB, class LoadSummary>
GSX_HD uint32_t summary_eval(LoadSummary ld, uint32_t stage, uint32_t idx, uint32_t codes, uint32_t budget, uint32_t u[NB]) {
    uint32_t w[8];
    ld(stage, idx, w);
    const uint32_t valid = w[0] & 0xFFFFu;
#if defined(__CUDA_ARCH__)
#pragma unroll
#endif
    for (int r = 0; r < NB; r++) u[r] = budget >= (uint32_t)r ? valid : 0u;
#if defined(__CUDA_ARCH__)
#pragma unroll
#endif
    for (uint32_t j = 0; j < 7u; j++) {
        const uint32_t c = (codes >> (4u * j)) & 15u;
        if (c == 7u || c == 12u) continue;                                       // no such level / PAM wildcard
        const uint32_t x = w[1u + j] ^ (((c & 2u) ? 0xFFFFu : 0u) | ((c & 1u) ? 0xFFFF0000u : 0u));
        uint32_t eq = ~(x | (x >> 16)) & 0xFFFFu;                                // rows whose symbol is the wanted one
        if (c < 4u) {                                                            // protospacer: a differing row loses one unit of budget
#if defined(__CUDA_ARCH__)
#pragma unroll
#endif
            for (int r = 0; r + 1 < NB; r++) u[r] = (u[r] & eq) | u[r + 1];
            u[NB - 1] &= eq;
        } else {
            if (c == 13u) eq = 0u;                                               // PAM character that can never match
#if defined(__CUDA_ARCH__)
#pragma unroll
#endif
            for (int r = 0; r < NB; r++) u[r] &= eq;
        }
    }
    return w[0];
}
// The same evaluation with the per-guide part hoisted out (what the sweep kernel runs): per plane j two masks such that
// y_j = (w_j & A_j) ^ X_j has a set bit in either half exactly for the rows that differ from the wanted symbol
// (wildcard / absent level: A = X = 0; never-matching PAM character: A = 0, X = ~0); pflags bit j = plane j is a
// protospacer level (a differing row loses one unit of budget instead of dying).
//   gm[0..6] = A, gm[7..13] = X, gm[14] = pflags
GSX_HD void summary_masks(uint32_t codes, uint32_t gm[15]) {
    uint32_t pflags = 0;
    for (uint32_t j = 0; j < 7u; j++) {
        const uint32_t c = (codes >> (4u * j)) & 15u;
        uint32_t A = ~0u, X = ((c & 2u) ? 0xFFFFu : 0u) | ((c & 1u) ? 0xFFFF0000u : 0u);
        if (c == 7u || c == 12u) { A = 0u; X = 0u; }
        else if (c == 13u) { A = 0u; X = ~0u; }
        else if (c < 4u) pflags |= 1u << j;
        gm[j] = A; gm[7u + j] = X;
    }
    gm[14] = pflags;
}
// The plane layouts the lean sweep loops (sweep_lean_kernel) are compiled for: which of the seven planes hold a protospacer level
// and which a concrete PAM character; every other plane is a wildcard or lies behind the guide's last level.  They cover 19-21 nt
// guides with an NGG-type PAM at L = 14 (plain guides and the edited forms of a bulge search) and every guide whose seven planes
// are all protospacer (smaller genomes: L <= 13).  -1: some other layout (the general loops of sweep_kernel handle it).
//   shape 0: 111111.  (20 nt at L = 14: six protospacer levels, the PAM wildcard)      shape 1: 1111111  (seven protospacer levels)
//   shape 2: 11111.P  (19 nt at L = 14: five protospacer levels, the wildcard, the first concrete PAM character)
constexpr int kSweepShapes = 3;
GSX_HD uint32_t sweep_shape_proto(int s) { return s == 0 ? 0x3Fu : s == 1 ? 0x7Fu : 0x1Fu; }
GSX_HD uint32_t sweep_shape_pam(int s) { return s == 2 ? 0x40u : 0u; }
GSX_HD int sweep_shape_of(uint32_t codes) {
    uint32_t proto = 0, pam = 0;
    for (uint32_t j = 0; j < 7u; j++) {
        const uint32_t c = (codes >> (4u * j)) & 15u;
        if (c < 4u) proto |= 1u << j;
        else if (c >= 8u && c < 12u) pam |= 1u << j;
        else if (c != 7u && c != 12u) return -1;                                  // a PAM character that can never match
    }
    for (int s = 0; s < kSweepShapes; s++) if (sweep_shape_proto(s) == proto && sweep_shape_pam(s) == pam) return s;
    return -1;
}
// The evaluation with the plane layout as a compile-time constant (sweep_lean_kernel): X = gm + 7 of summary_masks; no "A" words,
// unused planes cost nothing.  Equal to summary_eval_exact / summary_eval_masks for every guide of that layout (tests/host_core_check).
template <uint32_t USED>
GSX_HD uint32_t summary_exact_shape(const uint32_t w[8], const uint32_t X[7]) {
    uint32_t acc = 0;
#if defined(__CUDA_ARCH__)
#pragma unroll
#endif
    for (int j = 0; j < 7; j++) if (USED & (1u << j)) acc |= w[1 + j] ^ X[j];
    return w[0] & ~(acc | (acc >> 16)) & 0xFFFFu;
}
template <uint32_t PROTO, uint32_t PAM, int NB>
GSX_HD void summary_masks_shape(const uint32_t w[8], const uint32_t X[7], uint32_t budget, uint32_t u[NB]) {
    const uint32_t valid = w[0] & 0xFFFFu;
#if defined(__CUDA_ARCH__)
#pragma unroll
#endif
    for (int r = 0; r < NB; r++) u[r] = budget >= (uint32_t)r ? valid : 0u;
#if defined(__CUDA_ARCH__)
#pragma unroll
#endif
    for (int j = 0; j < 7; j++) {
        if (!((PROTO | PAM) & (1u << j))) continue;
        const uint32_t y = w[1 + j] ^ X[j];
        const uint32_t eq = ~(y | (y >> 16));
        if (PROTO & (1u << j)) {
#if defined(__CUDA_ARCH__)
#pragma unroll
#endif
            for (int r = 0; r + 1 < NB; r++) u[r] = (u[r] & eq) | u[r + 1];
            u[NB - 1] &= eq;
        } else {
#if defined(__CUDA_ARCH__)
#pragma unroll
#endif
            for (int r = 0; r < NB; r++) u[r] &= eq;
        }
    }
}
// no budget left: every differing row dies, whatever the level
GSX_HD uint32_t summary_eval_exact(const uint32_t w[8], const uint32_t gm[15]) {
    uint32_t acc = 0;
#if defined(__CUDA_ARCH__)
#pragma unroll
#endif
    for (uint32_t j = 0; j < 7u; j++) acc |= (w[1u + j] & gm[j]) ^ gm[7u + j];
    return w[0] & 0xFFFFu & ~(acc | (acc >> 16));
}
template <int NB>
GSX_HD void summary_eval_masks(const uint32_t w[8], const uint32_t gm[15], uint32_t budget, uint32_t u[NB]) {
    const uint32_t valid = w[0] & 0xFFFFu;
#if defined(__CUDA_ARCH__)
#pragma unroll
#endif
    for (int r = 0; r < NB; r++) u[r] = budget >= (uint32_t)r ? valid : 0u;
#if defined(__CUDA_ARCH__)
#pragma unroll
#endif
    for (uint32_t j = 0; j < 7u; j++) {
        const uint32_t y = (w[1u + j] & gm[j]) ^ gm[7u + j];
        const uint32_t eq = ~(y | (y >> 16));
        if ((gm[14] >> j) & 1u) {
#if defined(__CUDA_ARCH__)
#pragma unroll
#endif
            for (int r = 0; r + 1 < NB; r++) u[r] = (u[r] & eq) | u[r + 1];
            u[NB - 1] &= eq;
        } else {
#if defined(__CUDA_ARCH__)
#pragma unroll
#endif
            for (int r = 0; r < NB; r++) u[r] &= eq;
        }
    }
}
// The same for guides whose seven planes are all protospacer levels or wildcards / absent levels (no concrete PAM character among them:
// sweep_shape_of 0 or 1): every plane is stepped as a protospacer level.  A wildcard plane has A = X = 0, so every row matches it and
// the step u[r] = u[r] | u[r+1] leaves the nested masks (u[r+1] within u[r]) as they are.  No per-plane flag: about half the
// instructions of summary_eval_masks.  Equal to it for every such guide (tests/sweep_proto_check.cpp).
template <int NB>
GSX_HD void summary_eval_proto(const uint32_t w[8], const uint32_t gm[15], uint32_t budget, uint32_t u[NB]) {
    const uint32_t valid = w[0] & 0xFFFFu;
#if defined(__CUDA_ARCH__)
#pragma unroll
#endif
    for (int r = 0; r < NB; r++) u[r] = budget >= (uint32_t)r ? valid : 0u;
#if defined(__CUDA_ARCH__)
#pragma unroll
#endif
    for (uint32_t j = 0; j < 7u; j++) {
        const uint32_t y = (w[1u + j] & gm[j]) ^ gm[7u + j];
        const uint32_t eq = ~(y | (y >> 16));
#if defined(__CUDA_ARCH__)
#pragma unroll
#endif
        for (int r = 0; r + 1 < NB; r++) u[r] = (u[r] & eq) | u[r + 1];
        u[NB - 1] &= eq;
    }
}

// levels L + 7 and L + 8 for the rows that survived the first seven: t = sum2[e] = {hi7, lo7, hi8, lo8} over rows 0..31,
// half = which 16 of them the masks u[] describe
template <int NB>
GSX_HD void summary_tail(const uint32_t t[4], uint32_t half, uint32_t codes2, uint32_t u[NB]) {
#if defined(__CUDA_ARCH__)
#pragma unroll
#endif
    for (uint32_t j = 0; j < 2u; j++) {
        const uint32_t c = (codes2 >> (4u * j)) & 15u;
        if (c == 7u || c == 12u) continue;
        const uint32_t hi = (t[2u * j] >> (16u * half)) & 0xFFFFu, lo = (t[2u * j + 1u] >> (16u * half)) & 0xFFFFu;
        uint32_t eq = ~((hi ^ ((c & 2u) ? 0xFFFFu : 0u)) | (lo ^ ((c & 1u) ? 0xFFFFu : 0u))) & 0xFFFFu;
        if (c < 4u) {
#if defined(__CUDA_ARCH__)
#pragma unroll
#endif
            for (int r = 0; r + 1 < NB; r++) u[r] = (u[r] & eq) | u[r + 1];
            u[NB - 1] &= eq;
        } else {
            if (c == 13u) eq = 0u;
#if defined(__CUDA_ARCH__)
#pragma unroll
#endif
            for (int r = 0; r < NB; r++) u[r] &= eq;
        }
    }
}

// whole-node form (reference semantics for the tests): can any row of the pattern's interval still reach the final level?
template <int NB, class LoadSummary>
GSX_HD bool summary_viable(LoadSummary ld, uint32_t idx, uint32_t codes, uint32_t codes2, uint32_t budget) {
    uint32_t u[NB], t[8];
    const uint32_t head = summary_eval<NB>(ld, 0u, idx, codes, budget, u);
    if (head & SUM_WIDE32) return true;
    const bool tail = sweep_has_tail(codes2);
    if (tail) ld(2u, idx, t);
    if (u[0] && tail) summary_tail<NB>(t, 0u, codes2, u);
    if (u[0]) return true;
    if (!(head & SUM_WIDE16)) return false;
    summary_eval<NB>(ld, 1u, idx, codes, budget, u);
    if (u[0] && tail) summary_tail<NB>(t, 1u, codes2, u);
    return u[0] != 0u;
}
// builds the summary sectors of one table entry from the look-ahead planes; plane(b, j, hi) = 64-bit plane of t_j
// (hi or lo half of the 2-bit symbol) of 64-row block b, j = 0..6 (and 7, 8 with_tail)
template <class Plane>
GSX_HD void summary_build(Plane plane, bool with_tail, uint32_t sp, uint32_t width, uint32_t s0[8], uint32_t s1[8], uint32_t s2[4]) {
    for (int i = 0; i < 8; i++) s0[i] = s1[i] = 0u;
    for (int i = 0; i < 4; i++) s2[i] = 0u;
    if (width == 0u) return;
    const uint32_t e1 = sp + width;
    const uint32_t flags = (((e1 >> 6) != (sp >> 6)) ? SUM_TWO_BLOCKS : 0u) | (width > 16u ? SUM_WIDE16 : 0u) | (width > 32u ? SUM_WIDE32 : 0u);
    if (width > 32u) { s0[0] = 0xFFFFu | flags; return; }
    const uint32_t valid = width == 32u ? ~0u : ((1u << width) - 1u);
    const uint32_t b = sp >> 6, r0 = sp & 63u, nA = (64u - r0) < width ? (64u - r0) : width;      // rows taken from block b
    s0[0] = (valid & 0xFFFFu) | flags; s1[0] = (valid >> 16) | flags;
    for (uint32_t j = 0; j < 7u; j++) {
        uint32_t v[2];
        for (uint32_t h = 0; h < 2u; h++) {
            uint64_t bits = plane(b, j, h == 0u) >> r0;
            if (nA < width) bits |= plane(b + 1u, j, h == 0u) << nA;
            v[h] = (uint32_t)bits & valid;                                       // v[0] = high bits, v[1] = low bits of rows 0..31
        }
        s0[1u + j] = (v[0] & 0xFFFFu) | (v[1] << 16);
        s1[1u + j] = (v[0] >> 16) | (v[1] & 0xFFFF0000u);
    }
    if (with_tail)
        for (uint32_t j = 7; j < 9u; j++)
            for (uint32_t h = 0; h < 2u; h++) {
                uint64_t bits = plane(b, j, h == 0u) >> r0;
                if (nA < width) bits |= plane(b + 1u, j, h == 0u) << nA;
                s2[2u * (j - 7u) + h] = (uint32_t)bits & valid;
            }
}

// ---- k-mer jump table (specialised search kernels) ------------------------------------------------------------------
// ftab[s][e] = SA interval of the L-character pattern whose consumed characters c_0 .. c_{L-1} give the index
// e = sum c_i * 4^i.  The LAST consumed character is the first character of the pattern in text order, so e is the
// lexicographic rank of the pattern among all L-mers and sp is non-decreasing in e: a contiguous range of table entries
// covers a contiguous range of BWT rows (the slice-major kernel relies on it).  With the 2-bit codes of a guide packed
// at bits 2i of q, the guide's own entry is simply q & (4^L - 1).  The 16 patterns that differ only in their first two
// consumed characters share one 128-byte line.
// Instead of walking the top L levels of the tree, the kernels enumerate every pattern within the mismatch budget of
// the guide's first L characters and start the tree search from the surviving level-L intervals.  Same nodes at level L,
// same keys, as the level-by-level search.
struct FtabEntry { uint32_t sp, width; };

GSX_HD uint32_t ftab_exact_index(uint64_t q, uint32_t L) { return L >= 16 ? (uint32_t)q : (uint32_t)q & ((1u << (2u * L)) - 1u); }

// DFS kernel enumeration: one "combo" per choice of substituted positions among characters 2 .. L-1, times the 16
// beginnings (characters 0 and 1).
// combo word: bits 0..2 = number of substitutions j, then j fields of 6 bits: p (4 bits, character p + 2) | sub << 4
// (sub = 1..3: the substituted symbol is (c + sub) & 3)
GSX_HD void ftab_apply(uint64_t combo, uint64_t q, uint32_t L, uint32_t gidx, const uint64_t* pow5,
                       uint32_t& idx, uint64_t& key, uint32_t& j) {
    j = (uint32_t)(combo & 7u); idx = gidx; key = 0;
    for (uint32_t t = 0; t < j; t++) {
        const uint32_t f = (uint32_t)(combo >> (3u + 6u * t)) & 63u, p = (f & 15u) + 2u, sub = f >> 4;
        const uint32_t c = (uint32_t)(q >> (2u * p)) & 3u, s2 = (c + sub) & 3u;
        idx += (s2 - c) << (2u * p);                                            // (mod 2^32: a smaller symbol subtracts)
        key += (uint64_t)(1u + s2) * pow5[L - 1u - p];
    }
}
// beginning e (0..15) of a combo: e & 3 = symbol of character 0, e >> 2 = symbol of character 1; returns the extra
// mismatches and adds their key digits
GSX_HD uint32_t ftab_beginning(uint32_t e, uint64_t q, uint32_t L, const uint64_t* pow5, uint64_t& key) {
    const uint32_t s0 = e & 3u, s1 = e >> 2;
    const uint32_t c0 = (uint32_t)q & 3u, c1 = (uint32_t)(q >> 2) & 3u;
    uint32_t extra = 0;
    if (s0 != c0) { extra++; key += (uint64_t)(1u + s0) * pow5[L - 1u]; }
    if (s1 != c1) { extra++; key += (uint64_t)(1u + s1) * pow5[L - 2u]; }
    return extra;
}

// narrow string key (base 5, first consumed character most significant) of the L-character pattern with table index idx
GSX_HD uint64_t ftab_key(uint32_t idx, uint64_t q, uint32_t L) {
    uint64_t key = 0;
    for (uint32_t i = 0; i < L; i++) {
        const uint32_t c = (idx >> (2u * i)) & 3u, g = (uint32_t)(q >> (2u * i)) & 3u;
        key = key * 5ull + (c == g ? 0u : 1u + c);
    }
    return key;
}

// ---- slice-major enumeration (sweep kernel) ----------------------------------------------------------------------
// A slice fixes the last `sb` consumed characters of the pattern (the top 2*sb bits of the table index): its table
// entries and the BWT rows they point to are both contiguous and small enough to stay in L2 while every guide of the
// batch visits them.  For one guide and one slice with h substitutions inside the slice characters, the patterns are
// listed in an xor table built on the host (sweep_make_plan): entry = xor value over characters 0 .. L-sb-1 (2 bits per
// character; symbol' = symbol ^ x, x = 1..3) | number of substituted characters << 28.  Pass 1 lists the patterns that use
// the budget B = M - h up (exactly B substitutions) -- nine tenths of all patterns at m = 3, and the cheapest to test
// (one row mask); pass 0 the patterns that keep some budget (fewer than B).
// substitutions between the guide's slice characters and slice beta
GSX_HD uint32_t sweep_slice_distance(uint64_t q, uint32_t L, uint32_t sb, uint32_t beta) {
    const uint32_t top = (uint32_t)(q >> (2u * (L - sb))) & ((1u << (2u * sb)) - 1u);
    const uint32_t x = top ^ beta;
    return popc64((uint64_t)((x | (x >> 1)) & 0x55555555u));
}
// pattern t of (guide q, slice beta, budget B) in pass `zero`: table index; `used` = substitutions outside the slice characters
GSX_HD uint32_t sweep_pattern(const SweepPlan& pl, const uint32_t* xtab, uint32_t zero, uint64_t q, uint32_t beta, uint32_t B, uint32_t t, uint32_t& used) {
    const uint32_t w = xtab[pl.xoff[zero][B] + t];
    used = w >> 28;
    const uint32_t low_bits = 2u * (pl.L - pl.sb);
    return (beta << low_bits) | (((uint32_t)q & ((1u << low_bits) - 1u)) ^ (w & 0x0FFFFFFFu));
}

// ---- two-part enumeration (sweep_split_kernel) ------------------------------------------------------------------------------
// The strand indexes are over a text and its reverse complement, so the alignment a backward search of the consumed string
// u_0 .. u_{T-1} finds in one index is the one a backward search of c_k = complement(u_{T-1-k}) finds in the other: the same
// site read PAM-first.  split_query turns a distal-first query (q: protospacer, then pampack) into that PAM-first form: the PAM's
// characters complemented in reverse order (a wildcard becomes A: the plan lets that character take all four symbols), then the
// protospacer complemented from its PAM-proximal end.  The narrow key of such a match has T digits, all of the protospacer kind.
GSX_HD uint64_t split_query(uint64_t q, uint32_t pampack, uint32_t plen) {
    const uint32_t qlen = (uint32_t)(q >> 58), T = qlen + plen;
    uint64_t v = (uint64_t)T << 58;
    for (uint32_t k = 0; k < T; k++) {
        uint32_t c;
        if (k < plen) { const uint32_t pc = (pampack >> (3u * (plen - 1u - k))) & 7u; c = pc < 4u ? 3u - pc : 0u; }
        else c = 3u - ((uint32_t)(q >> (2u * (qlen - 1u - (k - plen)))) & 3u);
        v |= (uint64_t)c << (2u * k);
    }
    return v;
}
// A form-1 match (key over the PAM-first characters, found with query q2) as the distal-first consumed string u[0 .. T-1] (2-bit
// codes) of the same site; returns the mismatches of u among the first `head` protospacer characters of q
GSX_HD uint32_t split_unfold(uint64_t key, uint64_t q2, uint32_t T, uint64_t q, uint32_t head, uint32_t u[kMaxQ]) {
    for (uint32_t k = T; k-- > 0;) {
        const uint32_t d = (uint32_t)(key % 5ull); key /= 5ull;
        const uint32_t c = d == 0u ? ((uint32_t)(q2 >> (2u * k)) & 3u) : d - 1u;
        u[T - 1u - k] = 3u - c;
    }
    uint32_t mm = 0;
    for (uint32_t j = 0; j < head; j++) mm += u[j] != (((uint32_t)(q >> (2u * j))) & 3u) ? 1u : 0u;
    return mm;
}
// the narrow key and the mismatches the distal-first search gives the consumed string u (protospacer digits against q, then PAM digits)
GSX_HD uint64_t split_key(const uint32_t* u, uint64_t q, uint32_t plen, uint32_t& mm) {
    const uint32_t qlen = (uint32_t)(q >> 58);
    uint64_t key = 0; mm = 0;
    for (uint32_t j = 0; j < qlen + plen; j++) {
        uint32_t d;
        if (j < qlen) { d = u[j] == ((uint32_t)(q >> (2u * j)) & 3u) ? 0u : 1u + u[j]; mm += d ? 1u : 0u; }
        else d = u[j] < 3u ? u[j] : 4u;
        key = key * 5ull + d;
    }
    return key;
}
// table characters (2 bits each, low bit set) of form 0 / 1 by class; the split is after the guide's first `half` characters
//   form 0 (distal-first, qlen characters then the PAM): characters 0 .. half-1 capped, the rest cost budget
//   form 1 (PAM-first): the PAM's concrete characters never substituted, its wildcards free, the next qlen - half characters capped
GSX_HD void split_classes(uint32_t form, uint32_t L, uint32_t qlen, uint32_t plen, uint32_t pampack, uint32_t half,
                          uint32_t& cost, uint32_t& cap, uint32_t& exact, uint32_t& freec) {
    cost = cap = exact = freec = 0;
    for (uint32_t k = 0; k < L && k < 16u; k++) {
        const uint32_t bit = 1u << (2u * k);
        if (form == 0u) { cost |= bit; if (k < half) cap |= bit; continue; }
        if (k < plen) { if (((pampack >> (3u * (plen - 1u - k))) & 7u) == 4u) freec |= bit; else exact |= bit; continue; }
        cost |= bit;
        if (k < plen + (qlen - half)) cap |= bit;
    }
}

// ---- several alternative PAMs in one pass (specialised kernels, optional) ----------------------------------------------
// The reference searches the PAMs of a guide one after the other into the same std::set (process.hpp:51-56, index.hpp:210-212),
// so the result is the union of the per-PAM match sets.  One pass finds the same union: search with the FILTER PAM -- the
// common character where all PAMs agree, the wildcard where they differ -- and keep a finished alignment only if the PAM
// characters it consumed spell one of the real PAMs.  (Counting passes keep one pass per PAM: the reference's threshold
// counter counts a site once per PAM it satisfies.)
//   packs[k]: 3 bits per PAM character in consumption order (0..3 symbol, 4 = N wildcard, 5 = never matches, 6 = class); equal
//   lengths.  masks[k] (nullptr: no class anywhere): 4 bits per character, the members of a class character.  Two classes at one
//   position are the same character only with the same members (NRG + NYG filter on the wildcard); *out_mask = the filter's masks.
GSX_HD uint32_t fused_filter_pampack(const uint32_t* packs, uint32_t n, uint32_t plen, const uint32_t* masks = nullptr,
                                     uint32_t* out_mask = nullptr) {
    uint32_t out = 0, omask = 0;
    for (uint32_t j = 0; j < plen; j++) {
        const uint32_t c0 = (packs[0] >> (3u * j)) & 7u, m0 = masks ? (masks[0] >> (4u * j)) & 15u : 0u;
        bool same = true;
        for (uint32_t k = 1; k < n; k++) same = same && (((packs[k] >> (3u * j)) & 7u) == c0) && (!masks || ((masks[k] >> (4u * j)) & 15u) == m0);
        out |= (same ? c0 : 4u) << (3u * j);
        if (same) omask |= m0 << (4u * j);
    }
    if (out_mask) *out_mask = omask;
    return out;
}
// key: narrow string key whose last plen digits are the consumed PAM characters (A,C,G,N,T = 0..4, gsx_core.h key_append)
// (masks as in fused_filter_pampack: a class character accepts the digits of its members, never N's)
GSX_HD bool fused_pam_ok(uint64_t key, uint32_t plen, const uint32_t* packs, uint32_t n, const uint32_t* masks = nullptr) {
    uint32_t dg[kMaxPamLen];
    for (uint32_t j = plen; j-- > 0;) { dg[j] = (uint32_t)(key % 5ull); key /= 5ull; }
    for (uint32_t k = 0; k < n; k++) {
        bool ok = true;
        for (uint32_t j = 0; j < plen; j++) {
            const uint32_t pc = (packs[k] >> (3u * j)) & 7u;
            const uint32_t cm = (pc == 6u && masks) ? (masks[k] >> (4u * j)) & 15u : 0u;
            const uint32_t sbit = dg[j] == 3u ? 0u : 1u << (dg[j] < 3u ? dg[j] : 3u);       // digit A,C,G,N,T -> member bit (N: none)
            ok = ok && (pc == 4u || (pc < 4u && dg[j] == (pc < 3u ? pc : 4u)) || (cm & sbit) != 0u);
        }
        if (ok) return true;
    }
    return false;
}

// ordering of the matches of one guide: bucket (mismatches) ascending, forward index before reverse index, string order
GSX_HD int match_cmp(const MatchRec& x, const MatchRec& y) {
    uint32_t bx = ((x.info & 0xffu) << 1) | (x.task & 1u), by = ((y.info & 0xffu) << 1) | (y.task & 1u);
    if (bx != by) return bx < by ? -1 : 1;
    if (x.key_hi != y.key_hi) return x.key_hi < y.key_hi ? -1 : 1;
    if (x.key_lo != y.key_lo) return x.key_lo < y.key_lo ? -1 : 1;
    return 0;
}

}  // namespace gsx
#endif
