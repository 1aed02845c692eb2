// CPU-only harness for the host hierarchy builder of the multigrid preconditioner (lkb_mg.cu: mg_hierarchy): reads cases
// "<dim> <nx> <ny> <nz>" followed by 7 coefficients as "re im" pairs from stdin, and prints "case <status> <levels>", one
// line per level "nx ny nz  c0  cm0 cp0 e0  cm1 cp1 e1  cm2 cp2 e2  lmax" (complex values as "re im") and then the coarsest
// inverse, column-major, one "re im" per line.  It links liblkb.so and makes no CUDA call, so it runs without a GPU
// (tests/test_multigrid_host.py).
#include <cstdio>
#include "lkb_internal.h"
int main() {
    int dim;
    long long n[3];
    while (scanf("%d %lld %lld %lld", &dim, &n[0], &n[1], &n[2]) == 4) {
        lkb::cd coef[7];
        for (auto& c : coef) {
            double re = 0, im = 0;
            if (scanf("%lf %lf", &re, &im) != 2) return 1;
            c = lkb::cd(re, im);
        }
        const int64_t n64[3] = {n[0], n[1], n[2]};
        std::vector<lkb::MgHostLevel> lv;
        std::vector<lkb::cd> inv;
        const int e = lkb::mg_hierarchy(dim, n64, coef, lv, inv);
        printf("case %d %zu %zu\n", e, lv.size(), inv.size());
        auto pc = [](lkb::cd v) { printf(" %.17g %.17g", v.real(), v.imag()); };
        for (const auto& L : lv) {
            printf("%lld %lld %lld", (long long)L.n[0], (long long)L.n[1], (long long)L.n[2]);
            pc(L.c0);
            for (int d = 0; d < 3; ++d) { pc(L.cm[d]); pc(L.cp[d]); pc(L.e[d]); }
            printf(" %.17g\n", L.lmax);
        }
        for (const auto& v : inv) printf("%.17g %.17g\n", v.real(), v.imag());
    }
    return 0;
}
