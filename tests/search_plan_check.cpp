// search_plan_check -- the path, variants and widths plan_search (gsx_api.cpp) chooses for synthetic batches and index shapes,
// through the product's own guide packing (gsx_prepare_guides).  Each case names the condition of the device job that decides
// it.  No index, no GPU.
#include "../guidescan-cli_b200/csrc/gsx_host.h"
#include <climits>
#include <cstdio>
#include <cstdlib>
#include <random>
#include <string>
#include <vector>

using namespace gsx;

static int failures = 0;
#define CHECK(cond) do { if (!(cond)) { fprintf(stderr, "%s: FAILED %s (line %d)\n", name, #cond, __LINE__); failures++; } } while (0)

struct Batch {
    std::vector<std::string> seqs; std::string pam; std::vector<const char*> alt;
    gsx_params p; Prepared prep;
    Batch(size_t n, uint32_t qlen, const char* pam_, uint32_t m) : pam(pam_) {
        std::mt19937_64 rng(20261020);
        for (size_t i = 0; i < n; i++) { std::string s(qlen, 'A'); for (auto& c : s) c = "ACGT"[rng() & 3]; seqs.push_back(s); }
        gsx_params_default(&p); p.mismatches = m;
    }
    SearchPlan plan(const IndexShape& ix) {
        std::vector<gsx_guide> g(seqs.size());
        for (size_t i = 0; i < seqs.size(); i++) g[i] = {seqs[i].c_str(), pam.c_str()};
        p.alt_pams = alt.data(); p.n_alt_pams = (uint32_t)alt.size();
        prep = Prepared();
        if (gsx_prepare_guides(g.data(), g.size(), &p, prep) != 0) { fprintf(stderr, "gsx_prepare_guides failed\n"); exit(1); }
        return plan_search(prep, p, ix, (uint32_t)seqs.size());
    }
    int variant(const SearchPlan& pl, uint32_t M) const { return pl.sweep_variant(M, prep.min_qlen, prep.max_qlen, prep.plen, prep.pampack); }
};

static IndexShape plain_index(uint32_t ftab_L) {
    IndexShape x;
    x.plain = true; x.lines = true; x.exc_map = true; x.ftab_L[0] = x.ftab_L[1] = ftab_L; x.sum0 = true;
    x.rows = 3100000001ull; x.sm_count = 148;            // (a B200)
    return x;
}

int main() {
    const IndexShape ix14 = plain_index(14);
    {   const char* name = "200k NGG 20-mers, m = 3, ftab_L 14: two-part sweep";
        Batch b(200000, 20, "NGG", 3); const SearchPlan pl = b.plan(ix14);
        CHECK(pl.use_fast && !pl.exc && !pl.use_variants && pl.late_guides);
        CHECK(pl.search_sb == 5);                        // 40 * 4^(14 - sb) <= 12 MB
        CHECK(pl.split && pl.split_sb == 4 && pl.split_ctas == 6);        // one character less than the plain sweep's slices
        CHECK(!pl.combos && !pl.fuse_pams && pl.expand_roots == 0);
        CHECK(pl.queue_cap == 200000ull * 256);
        CHECK(pl.spill_cap == 2048);
        CHECK(pl.order_mode == INT_MIN && pl.order_probe && pl.spec_warp == INT_MIN && pl.sweep_variant_set == INT_MIN);
    }
    {   const char* name = "GSX_SPLIT=0: lean sweep variant 12";
        setenv("GSX_SPLIT", "0", 1);
        Batch b(200000, 20, "NGG", 3); const SearchPlan pl = b.plan(ix14);
        unsetenv("GSX_SPLIT");
        CHECK(!pl.split && pl.search_sb == 5 && b.variant(pl, 3) == 12);
    }
    {   const char* name = "m = 4: no split (m > kSplitMaxM), lean variant 11";
        Batch b(200000, 20, "NGG", 4); const SearchPlan pl = b.plan(ix14);
        CHECK(!pl.split && pl.search_sb == 5 && b.variant(pl, 4) == 11);
        CHECK(pl.queue_cap == 200000ull * 1024);
    }
    {   const char* name = "ftab_L 12: no split (12 < plen + 10), sb 3";
        Batch b(200000, 20, "NGG", 3); const SearchPlan pl = b.plan(plain_index(12));
        CHECK(!pl.split && pl.search_sb == 3);
    }
    {   const char* name = "ftab_L 13: split";
        Batch b(200000, 20, "NGG", 3); const SearchPlan pl = b.plan(plain_index(13));
        CHECK(pl.split && pl.search_sb == 4 && pl.split_sb == 3);
    }
    {   const char* name = "threshold 2: no split, threshold pass with its own sb";
        Batch b(200000, 20, "NGG", 3); b.p.threshold = 2; const SearchPlan pl = b.plan(ix14);
        CHECK(!pl.split && pl.search_sb == 5 && pl.threshold_sb == 5 && !pl.threshold_combos);
    }
    {   const char* name = "NGG + NAG: fused PAMs, no split";
        Batch b(200000, 20, "NGG", 3); b.alt.push_back("NAG"); const SearchPlan pl = b.plan(ix14);
        CHECK(pl.fuse_pams && !pl.split && pl.search_sb == 5);
    }
    {   const char* name = "NAG alone: split";
        Batch b(200000, 20, "NAG", 3); CHECK(b.plan(ix14).split);
    }
    {   const char* name = "TTG: no split (first PAM character not the wildcard)";
        Batch b(200000, 20, "TTG", 3); CHECK(!b.plan(ix14).split);
    }
    {   const char* name = "NNG: no split (second PAM character not concrete)";
        Batch b(200000, 20, "NNG", 3); CHECK(!b.plan(ix14).split);
    }
    {   const char* name = "--start, TTTN: no split";
        Batch b(200000, 20, "TTTN", 3); b.p.start = 1; const SearchPlan pl = b.plan(ix14);
        CHECK(!pl.split && pl.search_sb == 5);
    }
    {   const char* name = "19-nt guides: lean sweep, no split";
        Batch b(200000, 19, "NGG", 3); const SearchPlan pl = b.plan(ix14);
        CHECK(!pl.split && pl.search_sb == 5 && b.variant(pl, 3) == 12);
    }
    {   const char* name = "8191 guides: no sweep (< GSX_SWEEP_MIN), combos";
        Batch b(8191, 20, "NGG", 3); const SearchPlan pl = b.plan(ix14);
        CHECK(pl.use_fast && pl.search_sb == 0 && pl.combos && !pl.split);
    }
    {   const char* name = "a guide containing N, 100 guides: general kernel, roots expanded";
        Batch b(100, 20, "NGG", 3); b.seqs[7][3] = 'N'; const SearchPlan pl = b.plan(ix14);
        const int gw = search_grid_warps(false, 0, 148);
        CHECK(!pl.use_fast && pl.search_sb == 0 && !pl.split && pl.expand_roots == (size_t)8 * gw && pl.search_warps == gw);
    }
    {   const char* name = "R = D = 1: edited guides, chunk 262144, fmask";
        Batch b(1000, 20, "NGG", 3); b.p.rna_bulges = b.p.dna_bulges = 1; const SearchPlan pl = b.plan(ix14);
        CHECK(pl.use_fast && pl.use_variants && !pl.late_guides && pl.chunk == 262144 && pl.fmask);
        CHECK(pl.search_sb == 0 && !pl.split && pl.combos && pl.edited_qmin == 19 && pl.edited_qmax == 21);
        CHECK(pl.sweep_sb(262144, 19, 3) == 5 && pl.sweep_variant(3, 19, 21, 3, b.prep.pampack) == 11);
        CHECK(pl.chunk_queue_cap == 262144ull * 256 && pl.chunk_match_cap == 262144ull * 48);
        CHECK(pl.edited_match_cap == 1000ull * bulge_variants(20, 1, 1).size() * 12);
    }
    {   const char* name = "index with N, lines and exc_map: fast path with exc, no split";
        IndexShape x = ix14; x.plain = false;
        Batch b(200000, 20, "NGG", 3); const SearchPlan pl = b.plan(x);
        CHECK(pl.use_fast && pl.exc && !pl.split && pl.search_sb == 5);
    }
    {   const char* name = "index with N, no exc_map: general kernel";
        IndexShape x = ix14; x.plain = false; x.exc_map = false;
        Batch b(200000, 20, "NGG", 3); CHECK(!b.plan(x).use_fast);
    }
    {   const char* name = "GSX_FORCE_GENERAL=1: general kernel";
        setenv("GSX_FORCE_GENERAL", "1", 1);
        Batch b(200000, 20, "NGG", 3); const SearchPlan pl = b.plan(ix14);
        unsetenv("GSX_FORCE_GENERAL");
        CHECK(!pl.use_fast && !pl.split && pl.search_sb == 0 && pl.expand_roots == 0);
    }
    if (failures) return 1;
    printf("search plan selftest ok\n");
    return 0;
}
