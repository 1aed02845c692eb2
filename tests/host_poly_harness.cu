// CPU-only harness for the root construction of the GMRES-polynomial preconditioner (lkb_poly.cu: gmres_poly_roots): reads
// cases "<kind> <k>" followed by the (k+1) x k Hessenberg matrix column-major as "re im" pairs from stdin, and prints
// "case <status> <count>" and the roots as "re im" lines.  It links liblkb.so and makes no CUDA call, so it runs without a
// GPU (tests/test_poly_host.py).  argv[1]: the LAPACK provider (scipy's OpenBLAS).
#include <cstdio>
#include "lkb_internal.h"
int main(int argc, char** argv) {
    if (argc < 2 || lkb_set_lapack(argv[1], "scipy_", "_")) { printf("open failed: %s\n", lkb_last_error()); return 1; }
    char kc;
    int k;
    while (scanf(" %c %d", &kc, &k) == 2) {
        const int kind = kc == 's' ? LKB_S : kc == 'd' ? LKB_D : kc == 'c' ? LKB_C : LKB_Z;
        std::vector<lkb::cd> H((size_t)(k + 1) * k);
        for (auto& h : H) {
            double re = 0, im = 0;
            if (scanf("%lf %lf", &re, &im) != 2) return 1;
            h = lkb::cd(re, im);
        }
        std::vector<lkb::cd> roots;
        const int e = lkb::gmres_poly_roots(kind, H.data(), k + 1, k, roots);
        printf("case %d %zu\n", e, roots.size());
        for (const auto& r : roots) printf("%.17g %.17g\n", r.real(), r.imag());
    }
    return 0;
}
