// sweep_proto_check -- gsx_core.h summary_eval_proto (the filter of the two-part sweep for guides whose seven summary planes are
// protospacer levels or wildcards) against the general summary_eval_masks, on random summary sectors, for every plane layout made of
// protospacer levels (codes 0..3), absent levels (7) and PAM wildcards (12), and every budget.  No index, no GPU.
#include "../guidescan-cli_b200/csrc/gsx_host.h"
#include "../guidescan-cli_b200/csrc/gsx_core.h"
#include <cstdio>
#include <random>

using namespace gsx;

int main() {
    constexpr int NB = 4;
    std::mt19937_64 rng(20261023);
    uint64_t n = 0;
    for (int it = 0; it < 400000; it++) {
        uint32_t codes = 0;
        for (uint32_t j = 0; j < 7u; j++) {
            const uint32_t k = (uint32_t)(rng() % 6u);
            const uint32_t c = k < 4u ? k : k == 4u ? 7u : 12u;
            codes |= c << (4u * j);
        }
        uint32_t gm[15];
        summary_masks(codes, gm);
        uint32_t w[8];
        // header: a random number of valid rows (sometimes all 16, sometimes none)
        const uint32_t rows = (uint32_t)(rng() % 18u);
        w[0] = rows >= 16u ? 0xFFFFu : (1u << rows) - 1u;
        // planes: random, or near the guide's own symbols so that rows survive
        const bool near = (rng() & 1u) != 0u;
        for (uint32_t j = 0; j < 7u; j++) {
            uint32_t v = (uint32_t)rng();
            if (near) v = gm[7u + j] ^ ((uint32_t)rng() & (uint32_t)rng() & (uint32_t)rng());
            w[1u + j] = v;
        }
        for (uint32_t budget = 0; budget < (uint32_t)NB; budget++) {
            uint32_t a[NB], b[NB];
            summary_eval_masks<NB>(w, gm, budget, a);
            summary_eval_proto<NB>(w, gm, budget, b);
            for (int r = 0; r < NB; r++)
                if ((a[r] & 0xFFFFu) != (b[r] & 0xFFFFu)) {
                    fprintf(stderr, "summary_eval_proto differs: codes %07x budget %u mask %d: %04x vs %04x\n", codes, budget, r, a[r] & 0xFFFFu, b[r] & 0xFFFFu);
                    return 3;
                }
            n++;
        }
    }
    // the layouts the two-part sweep compiles it for: form 0 and form 1 of 20-nt guides with NGG at depth 13 and 14
    const uint32_t pampack = 4u | (1u << 3) | (1u << 6);
    for (uint32_t L : {13u, 14u}) {
        const int s0 = sweep_shape_of(sweep_codes((uint64_t)20 << 58, L, 3, pampack)), s1 = sweep_shape_of(sweep_codes((uint64_t)23 << 58, L, 0, 0));
        if (!((s0 == 0 || s0 == 1) && s1 == 1)) { fprintf(stderr, "L %u: layouts %d / %d are not protospacer-and-wildcard only\n", L, s0, s1); return 3; }
    }
    printf("%llu evaluations equal\nproto selftest ok\n", (unsigned long long)n);
    return 0;
}
