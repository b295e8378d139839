// split_plan_check -- the two-part enumeration of the sweep (gsx_types.h SplitPlan, gsx_core.h split_*) restated on the host
// through the product's own plan builder and helpers, for 20-nt guides with an NGG-type PAM at jump-table depth 14:
//   * the patterns each form reaches, walked slice by slice as sweep_split_kernel walks them (slice masks + xor table), are
//     distinct and number 2 185 + 496 per guide and strand;
//   * every alignment with at most 3 mismatches is reached by exactly one form: form 0 when at most one mismatch lies among the
//     guide's ten distal characters, form 1 (the same site read PAM-first) otherwise -- the re-anchoring drops form-1 matches with
//     fewer than two there, so nothing is found twice;
//   * split_unfold / split_key give back the distal-first string and the narrow key of the plain search.
// Prints patterns and sectors per guide and strand.  No index, no GPU.
#include "../guidescan-cli_b200/csrc/gsx_host.h"
#include "../guidescan-cli_b200/csrc/gsx_core.h"
#include <cstdio>
#include <map>
#include <random>

using namespace gsx;

static uint32_t pack_idx(const uint32_t* c, uint32_t L) { uint32_t e = 0; for (uint32_t j = 0; j < L; j++) e |= c[j] << (2u * j); return e; }

int main() {
    const uint32_t L = 14, M = 3, qlen = 20, plen = 3, half = 10, T = qlen + plen;
    const uint32_t pampack = 4u | (1u << 3) | (1u << 6);        // N C C: an NGG PAM in the consumption order of the distal-first query
    std::mt19937_64 rng(20261020);
    for (uint32_t sb : {3u, 4u, 5u}) {
        SplitPlan pl; std::vector<uint32_t> xt;
        split_make_plan(L, sb, M, qlen, plen, pampack, half, pl, xt);
        const uint32_t low = 2u * (L - sb), top_mask = (1u << (2u * sb)) - 1u, low_mask = (1u << low) - 1u;
        uint64_t n_pat[2] = {0, 0}, n_guides = 0, n_sites = 0;
        for (int gi = 0; gi < 24; gi++) {
            uint64_t q = (uint64_t)qlen << 58;
            for (uint32_t j = 0; j < qlen; j++) q |= (uint64_t)(rng() & 3u) << (2u * j);
            const uint64_t q2 = split_query(q, pampack, plen);
            std::map<uint32_t, uint32_t> reach[2];                  // table index -> mismatches of its table characters
            for (uint32_t f = 0; f < 2; f++) {
                const uint64_t qq = f ? q2 : q;
                for (uint32_t beta = 0; beta <= top_mask; beta++) {
                    const uint32_t x = ((uint32_t)(qq >> low) & top_mask) ^ beta, d = (x | (x >> 1)) & 0x55555555u;
                    const uint32_t h = __builtin_popcount(d & pl.cost_top[f]), cp = __builtin_popcount(d & pl.cap_top[f]);
                    if ((d & pl.exact_top[f]) || h > M || cp > 1u) continue;
                    const uint32_t c = 1u - cp, B = M - h;
                    for (uint32_t t = 0; t < pl.xcnt[f][c][B]; t++) {
                        const uint32_t xw = xt[pl.xoff[f][c][B] + t];
                        const uint32_t idx = (beta << low) | (((uint32_t)qq & low_mask) ^ (xw & 0x0FFFFFFFu));
                        if (!reach[f].emplace(idx, h + (xw >> 28)).second) { fprintf(stderr, "form %u reaches pattern %u twice\n", f, idx); return 3; }
                    }
                }
                n_pat[f] += reach[f].size();
            }
            n_guides++;
            // random sites within 3 mismatches (concrete PAM characters matched, the wildcard anything)
            for (int it = 0; it < 20000; it++) {
                uint32_t u[kMaxQ], c[kMaxQ];
                for (uint32_t j = 0; j < qlen; j++) u[j] = (uint32_t)(q >> (2u * j)) & 3u;
                const uint32_t k = (uint32_t)(rng() % (M + 1u));
                for (uint32_t s = 0; s < k; s++) { const uint32_t p = (uint32_t)(rng() % qlen); u[p] = (u[p] + 1u + (uint32_t)(rng() % 3u)) & 3u; }
                for (uint32_t j = 0; j < plen; j++) { const uint32_t pc = (pampack >> (3u * j)) & 7u; u[qlen + j] = pc < 4u ? pc : (uint32_t)(rng() & 3u); }
                for (uint32_t j = 0; j < T; j++) c[j] = 3u - u[T - 1u - j];
                uint32_t dmm = 0, mm0 = 0, mm1 = 0;
                for (uint32_t j = 0; j < qlen; j++) if (u[j] != ((uint32_t)(q >> (2u * j)) & 3u)) { dmm += j < half ? 1u : 0u; mm0 += j < L ? 1u : 0u; }
                for (uint32_t j = plen; j < L; j++) mm1 += c[j] != ((uint32_t)(q2 >> (2u * j)) & 3u) ? 1u : 0u;
                const auto a = reach[0].find(pack_idx(u, L)), b = reach[1].find(pack_idx(c, L));
                const bool in0 = a != reach[0].end() && a->second == mm0, in1 = b != reach[1].end() && b->second == mm1;
                if (dmm <= 1u && !in0) { fprintf(stderr, "form 0 misses a site with %u distal mismatches\n", dmm); return 3; }
                if (dmm >= 2u && (in0 || !in1)) { fprintf(stderr, "site with %u distal mismatches: form 0 %d form 1 %d\n", dmm, (int)in0, (int)in1); return 3; }
                // the form-1 match of the site as the plain search records it
                uint64_t key1 = 0;
                for (uint32_t j = 0; j < T; j++) key1 = key1 * 5ull + (c[j] == (((uint32_t)(q2 >> (2u * j))) & 3u) ? 0u : 1u + c[j]);
                uint32_t v[kMaxQ];
                if (split_unfold(key1, q2, T, q, half, v) != dmm) { fprintf(stderr, "split_unfold: distal mismatches differ\n"); return 3; }
                uint64_t key0 = 0; uint32_t mmw = 0;
                for (uint32_t j = 0; j < T; j++) {
                    if (v[j] != u[j]) { fprintf(stderr, "split_unfold: character %u differs\n", j); return 3; }
                    const uint32_t dg = j < qlen ? (u[j] == (((uint32_t)(q >> (2u * j))) & 3u) ? 0u : 1u + u[j]) : (u[j] < 3u ? u[j] : 4u);
                    mmw += (j < qlen && dg) ? 1u : 0u;
                    key0 = key0 * 5ull + dg;
                }
                uint32_t mmk;
                if (split_key(v, q, plen, mmk) != key0 || mmk != mmw) { fprintf(stderr, "split_key differs from the plain key\n"); return 3; }
                n_sites++;
            }
        }
        const double per0 = (double)n_pat[0] / n_guides, per1 = (double)n_pat[1] / n_guides;
        printf("sb %u: patterns per guide and strand %.1f (form 0 %.1f, form 1 %.1f), xor table %zu words, %llu sites checked\n",
               sb, per0 + per1, per0, per1, xt.size(), (unsigned long long)n_sites);
    }
    // the plain enumeration for comparison: every pattern within 3 substitutions of the 14 table characters
    uint64_t plain = 0, c = 1;
    for (uint32_t j = 0; j <= M; j++) { plain += c; c = c * 3u * (L - j) / (j + 1u); }
    printf("plain sweep: patterns per guide and strand %llu\n", (unsigned long long)plain);
    printf("split selftest ok\n");
    return 0;
}
