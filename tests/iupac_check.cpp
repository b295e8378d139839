// iupac_check -- IUPAC class letters in PAMs on the host: the letter tables (gsx_iupac.h), the device arithmetic that tests a class
// character (gsx_core.h make_child, viable_children, fused_filter_pampack / fused_pam_ok) against brute force, the PAM bytes
// gsx_prepare_guides packs, and the search path plan_search picks for class batches.  Prints the generator's expansions for
// tests/test_iupac_host.py to compare with the Python restatement.  No index, no GPU.
#include "../guidescan-cli_b200/csrc/gsx_host.h"
#include "../guidescan-cli_b200/csrc/gsx_core.h"
#include "../guidescan-cli_b200/csrc/gsx_iupac.h"
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <random>
#include <string>
#include <vector>

using namespace gsx;

static int failures = 0;
#define CHECK(cond) do { if (!(cond)) { fprintf(stderr, "FAILED %s (line %d)\n", #cond, __LINE__); failures++; } } while (0)

static const char* kClasses = "RYSWKMBDHV";

// does PAM code pc (mask cm for code 6) accept consumed symbol s (0..3) / a literal N (s = 4)?
static bool accepts(uint32_t pc, uint32_t cm, uint32_t s) {
    if (pc == 4u) return true;
    if (s == 4u) return false;
    if (pc < 4u) return pc == s;
    if (pc == 6u) return (cm >> s) & 1u;
    return false;
}

static void tables() {
    const char* members[10] = {"AG", "CT", "CG", "AT", "GT", "AC", "CGT", "AGT", "ACT", "ACG"};
    const char* partner = "RYSWKMBDHV";
    const char* comp = "YRSWMKVHDB";
    for (int i = 0; i < 10; i++) {
        uint32_t m = 0; for (const char* p = members[i]; *p; p++) m |= iupac_base_bit(*p);
        CHECK(iupac_mask(kClasses[i]) == m);
        CHECK(iupac_is_class(kClasses[i]));
        CHECK(iupac_complement(partner[i]) == comp[i]);
        CHECK(iupac_complement(iupac_complement(kClasses[i])) == kClasses[i]);
        // the complement's members are the complements of the members
        uint32_t cm = 0; for (const char* p = members[i]; *p; p++) cm |= iupac_base_bit(complement_char(*p));
        CHECK(iupac_mask(iupac_complement(kClasses[i])) == cm);
    }
    CHECK(iupac_mask('A') == 1 && iupac_mask('C') == 2 && iupac_mask('G') == 4 && iupac_mask('T') == 8 && iupac_mask('N') == 15);
    for (char c : std::string("ACGTN")) { CHECK(!iupac_is_class(c)); CHECK(iupac_pam_char(c)); }
    for (char c : std::string("acgtnryXZU.-*")) { CHECK(iupac_mask(c) == 0); CHECK(!iupac_pam_char(c)); CHECK(!iupac_is_class(c)); }
    CHECK(iupac_complement('N') == 'N' && iupac_complement('A') == 'T' && iupac_complement('G') == 'C');
    // a class never accepts a genome N; N accepts it
    CHECK(!iupac_pam_fits('R', 'N') && iupac_pam_fits('N', 'N') && iupac_pam_fits('R', 'G') && !iupac_pam_fits('R', 'C') && iupac_pam_fits('A', 'A'));
    // complement_char keeps the reference's behaviour: class letters unchanged
    for (int i = 0; i < 10; i++) CHECK(complement_char(kClasses[i]) == kClasses[i]);
}

static void expansions() {
    const char* pats[] = {"NGG", "NAG", "NNG", "TTTN", "NNNNGATT", "ACGT", "N", "NRG", "NNGRRT", "TTTV", "NRRH", "NNNNRYAC", "NNAGAAW", "NYN", "BDHV"};
    for (const char* p : pats) {
        printf("expand %s:", p);
        for (auto& s : iupac_expand(p)) printf(" %s", s.c_str());
        printf("\n");
        printf("classes %s:", p);
        for (auto& s : iupac_expand_classes(p)) printf(" %s", s.c_str());
        printf("\n");
    }
}

// random PAM lists of code 0..6 characters: fused_pam_ok against the definition, the filter PAM as a superset of the list
static void fused(std::mt19937_64& rng) {
    for (int it = 0; it < 20000; it++) {
        const uint32_t plen = 1 + rng() % 5, n = 1 + rng() % kMaxPams;
        uint32_t packs[kMaxPams] = {0}, masks[kMaxPams] = {0};
        for (uint32_t k = 0; k < n; k++)
            for (uint32_t j = 0; j < plen; j++) {
                uint32_t pc = rng() % 7;
                if (pc == 5u && rng() % 4) pc = 6u;
                packs[k] |= pc << (3 * j);
                if (pc == 6u) { const char c = kClasses[rng() % 10]; masks[k] |= iupac_mask(c) << (4 * j); }
            }
        if (rng() % 3 == 0) for (uint32_t k = 1; k < n; k++) { packs[k] = packs[0]; masks[k] = masks[0]; }
        uint32_t fmask = 0;
        const uint32_t filt = fused_filter_pampack(packs, n, plen, masks, &fmask);
        for (int t = 0; t < 64; t++) {
            uint32_t dg[kMaxPamLen]; uint64_t key = rng() % 1000;          // (digits above the PAM's are ignored)
            for (uint32_t j = 0; j < plen; j++) { dg[j] = rng() % 5; key = key * 5 + dg[j]; }
            bool want = false;
            for (uint32_t k = 0; k < n && !want; k++) {
                bool ok = true;
                for (uint32_t j = 0; j < plen; j++) {
                    const uint32_t s = dg[j] == 3u ? 4u : dg[j] == 4u ? 3u : dg[j];       // digit A,C,G,N,T -> symbol (4 = N)
                    ok = ok && accepts((packs[k] >> (3 * j)) & 7u, (masks[k] >> (4 * j)) & 15u, s);
                }
                want = ok;
            }
            CHECK(fused_pam_ok(key, plen, packs, n, masks) == want);
            if (want) CHECK(fused_pam_ok(key, plen, &filt, 1, &fmask));
            bool no_class = true;
            for (uint32_t k = 0; k < n; k++) no_class = no_class && masks[k] == 0;
            if (no_class) CHECK(fused_pam_ok(key, plen, packs, n) == want);
        }
    }
    // NRG + NYG (consumption order as a 3-character PAM): the class position becomes the wildcard, never one of the two classes
    const uint32_t p2[2] = {4u | (6u << 3) | (2u << 6), 4u | (6u << 3) | (2u << 6)}, m2[2] = {5u << 4, 10u << 4};
    uint32_t fm = 99;
    const uint32_t f2 = fused_filter_pampack(p2, 2, 3, m2, &fm);
    CHECK(((f2 >> 3) & 7u) == 4u && fm == 0u);
    const uint32_t m3[2] = {5u << 4, 5u << 4};
    const uint32_t f3 = fused_filter_pampack(p2, 2, 3, m3, &fm);
    CHECK(f3 == p2[0] && fm == m3[0]);
    // an A/C/G/T/N list: the same filter with and without masks
    const uint32_t pa[2] = {4u | (2u << 3) | (2u << 6), 4u | (0u << 3) | (2u << 6)}, ma[2] = {0, 0};
    CHECK(fused_filter_pampack(pa, 2, 3, ma, &fm) == fused_filter_pampack(pa, 2, 3) && fm == 0u);
}

// viable_children: exact brute force (class exact) is a subset of the result; treating the class as a wildcard gives it exactly
static void viable(std::mt19937_64& rng) {
    for (int it = 0; it < 20000; it++) {
        uint64_t hi[7], lo[7];
        for (int j = 0; j < 7; j++) { hi[j] = rng(); lo[j] = rng(); }
        const uint32_t qlen = 1 + rng() % 24, plen = 1 + rng() % 6, total = qlen + plen;
        uint64_t q = (uint64_t)qlen << 58; for (uint32_t l = 0; l < qlen && l < 29; l++) q |= (uint64_t)(rng() & 3) << (2 * l);
        uint32_t pampack = 0, pammask = 0;
        for (uint32_t j = 0; j < plen; j++) {
            const uint32_t r = rng() % 10, pc = r < 4 ? r : r < 6 ? 4u : r == 6 ? 5u : 6u;
            pampack |= pc << (3 * j);
            if (pc == 6u) pammask |= iupac_mask(kClasses[rng() % 10]) << (4 * j);
        }
        const uint32_t lvl = rng() % total, budget = rng() % 4;
        uint32_t sp = rng() & 63, ep = rng() & 63; if (sp > ep) std::swap(sp, ep);
        const uint32_t got = viable_children(hi, lo, sp, ep, lvl, qlen, total, q, pampack, budget);
        uint32_t exact = 0, wild = 0;
        for (uint32_t r = sp; r <= ep; r++) {
            uint32_t mm = 0; bool dead_e = false, dead_w = false;
            for (uint32_t j = 0; j < 7 && lvl + j < total; j++) {
                const uint32_t s = (uint32_t)(((hi[j] >> r) & 1) << 1 | ((lo[j] >> r) & 1)), L = lvl + j;
                if (L < qlen) { mm += s != ((q >> (2 * L)) & 3u) ? 1u : 0u; continue; }
                const uint32_t pc = (pampack >> (3 * (L - qlen))) & 7u, cm = (pammask >> (4 * (L - qlen))) & 15u;
                dead_e = dead_e || !accepts(pc, cm, s);
                dead_w = dead_w || !accepts(pc == 6u ? 4u : pc, 0u, s);
            }
            const uint32_t s0 = (uint32_t)(((hi[0] >> r) & 1) << 1 | ((lo[0] >> r) & 1));
            if (mm <= budget && !dead_e) exact |= 1u << s0;
            if (mm <= budget && !dead_w) wild |= 1u << s0;
        }
        CHECK((exact & ~got) == 0u);
        CHECK(got == wild);
        if (!pammask) CHECK(got == exact);
    }
}

// make_child on a PAM level: the children of every code against the definition (literal N only under N)
static void children() {
    static const uint32_t nrows[4] = {3, 9, 17, 40};
    DevStrand st{}; st.n_rows = nrows; st.n_nrows = 4; st.n = 64; for (int c = 0; c < 5; c++) st.C[c] = 10u * c;
    GuideRec g{}; g.qlen = 4; for (int l = 0; l < 4; l++) g.q[l] = (uint8_t)l;
    for (uint32_t pc = 0; pc < 7; pc++)
        for (int ci = -1; ci < 10; ci++) {
            if ((pc == 6u) != (ci >= 0)) continue;
            PamSet ps{}; ps.n_pams = 1; ps.plen[0] = 2; ps.sym[0][0] = (uint8_t)pc; ps.sym[0][1] = SYM_N; ps.kpam_len = 2;
            if (pc == 6u) ps.cmask[0][0] = (uint8_t)iupac_mask(kClasses[ci]);
            ExpandCtx cx{&st, &g, &ps, 3, 0, 0};
            Node nd{}; nd.sp = 0; nd.ep = 50; nd.meta = meta_make(4, 1, 0, 0, 0, 0, 0);
            const uint32_t os[4] = {0, 0, 0, 0}, oe[4] = {2, 3, 4, 5};
            for (int cand = 0; cand <= CAND_LITN; cand++) {
                Node ch; bool emit;
                const bool got = make_child<false>(cand, nd, cx, os, oe, ch, emit);
                CHECK(got == accepts(pc, ps.cmask[0][0], (uint32_t)cand));
                if (got) { CHECK(meta_mm(ch.meta) == 1u); CHECK(!emit); }
            }
        }
}

struct Prep {
    gsx_params p; Prepared prep; std::vector<std::string> seqs; std::vector<const char*> alt;
    int run(const char* pam, std::vector<const char*> alts, bool iupac, bool start, size_t n = 16, uint32_t qlen = 20) {
        std::mt19937_64 rng(7);
        seqs.clear(); for (size_t i = 0; i < n; i++) { std::string s(qlen, 'A'); for (auto& c : s) c = "ACGT"[rng() & 3]; seqs.push_back(s); }
        gsx_params_default(&p); p.iupac_pams = iupac ? 1 : 0; p.start = start ? 1 : 0;
        alt = alts; p.alt_pams = alt.data(); p.n_alt_pams = (uint32_t)alt.size();
        std::vector<gsx_guide> g(n); for (size_t i = 0; i < n; i++) g[i] = {seqs[i].c_str(), pam};
        prep = Prepared();
        return gsx_prepare_guides(g.data(), n, &p, prep);
    }
};

static uint8_t old_sym(char c) { return c == 'A' ? SYM_A : c == 'C' ? SYM_C : c == 'G' ? SYM_G : c == 'T' ? SYM_T : c == 'N' ? SYM_N : SYM_X; }

// the PAM bytes of A/C/G/T/N lists: what the packing gave before class letters existed, with the option on or off
static void packing() {
    struct L { const char* pam; std::vector<const char*> alts; bool start; };
    const std::vector<L> lists = {{"NGG", {}, false}, {"NGG", {"NAG"}, false}, {"TTTN", {}, true}, {"NNG", {}, false}, {"NAG", {}, false},
                                  {"TTG", {}, false}, {"NGG", {"NAG", "NGA", "NNGRRT"}, false}, {"NNNNGATT", {}, false}};
    for (const L& l : lists) {
        Prep a, b;
        CHECK(a.run(l.pam, l.alts, false, l.start) == 0);
        CHECK(b.run(l.pam, l.alts, true, l.start) == 0);
        const bool has_class = l.alts.size() == 3;
        if (!has_class) CHECK(memcmp(a.prep.pamsets, b.prep.pamsets, sizeof a.prep.pamsets) == 0);
        const PamSet& ps = a.prep.pamsets[0];
        std::vector<std::string> pams; for (auto x : l.alts) pams.push_back(x); pams.push_back(l.pam);
        CHECK(ps.n_pams == pams.size());
        for (size_t k = 0; k < pams.size(); k++) {
            uint32_t pack = 0;
            for (size_t j = 0; j < pams[k].size(); j++) {
                const uint8_t want = l.start ? old_sym(pams[k][pams[k].size() - 1 - j]) : old_sym(complement_char(pams[k][j]));
                CHECK(ps.sym[k][j] == want);
                CHECK(ps.cmask[k][j] == 0);
                pack |= (uint32_t)want << (3 * j);
            }
            if (a.prep.fast_ok && pams[0].size() == pams[k].size()) { CHECK(a.prep.pampacks[k] == pack); CHECK(a.prep.pammasks[k] == 0u); }
        }
        CHECK(a.prep.pammask == 0u);
    }
    // NRG in the default orientation: consumption order comp(G), comp(R), comp(N) read from the PAM's 5' end = N, Y, C
    Prep c;
    CHECK(c.run("NRG", {}, true, false) == 0);
    CHECK(c.prep.pamsets[0].sym[0][0] == SYM_N && c.prep.pamsets[0].sym[0][1] == SYM_CLS && c.prep.pamsets[0].sym[0][2] == SYM_C);
    CHECK(c.prep.pamsets[0].cmask[0][1] == 10u);                                // Y = {C, T}
    CHECK(c.prep.pampack == (4u | (6u << 3) | (1u << 6)) && c.prep.pammask == (10u << 4));
    CHECK(c.run("NRG", {}, false, false) == 0);                                 // without the option: never matches, as before
    CHECK(c.prep.pamsets[0].sym[0][1] == SYM_X && c.prep.pamsets[0].cmask[0][1] == 0u);
    CHECK(c.run("TTTV", {}, true, true) == 0);                                  // --start: consumption order V, T, T, T, no complement
    CHECK(c.prep.pamsets[0].sym[0][0] == SYM_CLS && c.prep.pamsets[0].cmask[0][0] == 7u && c.prep.pamsets[0].sym[0][1] == SYM_T);
    // one class PAM is one PamSet entry: NRRH (12 concrete PAMs) fits where its expansion would not
    CHECK(c.run("NRRH", {"NGG"}, true, false) == 0);
    CHECK(c.prep.pamsets[0].n_pams == 2);
    CHECK(c.run("NGG", {"NAG", "NGA", "NCG", "NTG", "AGG", "CGG", "TGG", "GGG"}, true, false) != 0);     // (9 PAMs: the limit holds)
}

// a class batch takes the path of its concrete expansion: fast kernel, lean sweep, never the general kernel or the two-part sweep
static void paths() {
    IndexShape ix; ix.plain = true; ix.lines = true; ix.exc_map = true; ix.ftab_L[0] = ix.ftab_L[1] = 14; ix.sum0 = true;
    ix.rows = 3100000001ull; ix.sm_count = 148;
    IndexShape ixn = ix; ixn.plain = false;
    struct C { const char* pam; std::vector<const char*> alts; bool start; const char* cpam; std::vector<const char*> calts; };
    const std::vector<C> cases = {{"NRG", {}, false, "NAG", {"NGG"}}, {"NNGRRT", {}, false, "NNGAAT", {"NNGAGT", "NNGGAT", "NNGGGT"}},
                                  {"TTTV", {}, true, "TTTA", {"TTTC", "TTTG"}}, {"NGG", {"NRG"}, false, "NGG", {"NAG", "NGG"}}};
    for (const C& c : cases)
        for (const IndexShape* x : {&ix, &ixn}) {
            Prep a, b;
            CHECK(a.run(c.pam, c.alts, true, c.start, 20000) == 0);
            CHECK(b.run(c.cpam, c.calts, false, c.start, 20000) == 0);
            const SearchPlan pa = plan_search(a.prep, a.p, *x, 20000), pb = plan_search(b.prep, b.p, *x, 20000);
            CHECK(pa.use_fast && pa.use_fast == pb.use_fast && pa.exc == pb.exc && pa.search_sb == pb.search_sb && pa.search_sb != 0);
            CHECK(!pa.split);
            CHECK(pa.sweep_variant(3, a.prep.min_qlen, a.prep.max_qlen, a.prep.plen, a.prep.pampack) == 12);
            // the arena estimate counts |class| / 4 of the sites: the same as the expansion's
            CHECK(std::abs(pa.match_per_guide - pb.match_per_guide) < 1e-6 * pb.match_per_guide);
        }
    // bulges: edited guides for the class batch as for its expansion
    Prep a; a.run("NRG", {}, true, false, 20000);
    a.p.rna_bulges = a.p.dna_bulges = 1;
    std::vector<gsx_guide> g(a.seqs.size()); for (size_t i = 0; i < g.size(); i++) g[i] = {a.seqs[i].c_str(), "NRG"};
    Prepared pr; CHECK(gsx_prepare_guides(g.data(), g.size(), &a.p, pr) == 0);
    CHECK(plan_search(pr, a.p, ixn, 20000).use_variants);
}

int main() {
    std::mt19937_64 rng(20261022);
    tables();
    expansions();
    fused(rng);
    viable(rng);
    children();
    packing();
    paths();
    if (failures) { fprintf(stderr, "%d check(s) failed\n", failures); return 1; }
    printf("iupac selftest ok\n");
    return 0;
}
