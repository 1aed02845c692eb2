// host_expm_mock.cu -- TEST INFRASTRUCTURE: runs the product's Krylov-exponential shells (lkb_expm.cu: kexpm_vec, kexpm_mat,
// krylov_exptA -- the restated stdlib expm, the error estimates, the on-demand growth of the work basis, the breakdown exits) WITHOUT
// a GPU.  lkb_expm.cu is included verbatim; the C-ABI entry points it calls are implemented on host memory: block Arnoldi steps and
// the unpivoted QR by the C oracle, the pivoting QR by a callback into the Python oracle (oracle.qr_with_pivoting).
// tests/test_host_shells_mock.py compares the C++ shells with the Python oracle shells.  Nothing here is part of the product.
#include <complex>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <vector>
#include "../include/lkb.h"
#include "lkb_internal.h"

#include "lkb_expm.cu"        // the product's host shells, verbatim

#include "host_mock_common.inc"

extern "C" {
#define ORACLE_QR(sfx, R) int lko_qr_##sfx(int64_t n, void* Q, int64_t ldq, int p, void* Rm, int ldr, R tol, uint64_t* seed, int64_t row0);
ORACLE_QR(s, float) ORACLE_QR(d, double) ORACLE_QR(c, float) ORACLE_QR(z, double)
#undef ORACLE_QR
}

namespace {
typedef int (*qr_pivoting_cb)(int kind, int64_t n, int p, void* Q, int64_t ld, void* R, int ldr, int32_t* perm, double tol, int32_t* info);
qr_pivoting_cb g_qr_pivoting = nullptr;
}

extern "C" {

void mock_set_qr_pivoting(qr_pivoting_cb cb) { g_qr_pivoting = cb; }

int lkb_arnoldi(lkb_op_t A, lkb_basis_t X, void* H, int ldh, int32_t* info, int32_t kstart, int32_t kend, double tol, int32_t transpose,
                int32_t blksize) {
    const int p = blksize > 0 ? blksize : 1;
    const int kdim = (X->ncols - p) / p;
    if (kstart <= 0) kstart = 1;
    if (kend <= 0) kend = kdim;
    if (kstart > kend || kend > kdim || ldh < (kend + 1) * p) { set_error("mock arnoldi: inconsistent sizes"); return LKB_ERR_ARG; }
    if (tol < 0) tol = atol_of(X->kind);
    switch (X->kind) {
        case KS: *info = lko_arnoldi_s(A->user, X->n, X->d, X->ld, H, ldh, kdim, kstart, kend, (float)tol, transpose, p, &g_oracle_seed); break;
        case KD: *info = lko_arnoldi_d(A->user, X->n, X->d, X->ld, H, ldh, kdim, kstart, kend, tol, transpose, p, &g_oracle_seed); break;
        case KC: *info = lko_arnoldi_c(A->user, X->n, X->d, X->ld, H, ldh, kdim, kstart, kend, (float)tol, transpose, p, &g_oracle_seed); break;
        default: *info = lko_arnoldi_z(A->user, X->n, X->d, X->ld, H, ldh, kdim, kstart, kend, tol, transpose, p, &g_oracle_seed); break;
    }
    for (int k = kstart; k <= kend; ++k) for (int i = 0; i < p; ++i) { if (transpose) A->n_rmatvec++; else A->n_matvec++; }
    return 0;
}
int lkb_basis_axpby(const void* alpha, lkb_basis_t X, int xcol0, const void* beta, lkb_basis_t Y, int ycol0, int ncols) {
    if (!X || !Y || xcol0 + ncols > X->ncols || ycol0 + ncols > Y->ncols || X->n != Y->n || X->kind != Y->kind) return LKB_ERR_ARG;
    const bool sp = (Y->kind == KS || Y->kind == KC), cplx = kind_cplx(Y->kind);
    auto ld = [&](const void* p) { return sp ? Scalar{((const float*)p)[0], cplx ? ((const float*)p)[1] : 0.0}
                                             : Scalar{((const double*)p)[0], cplx ? ((const double*)p)[1] : 0.0}; };
    for (int q = 0; q < ncols; ++q) launch_axpby(Y->kind, nullptr, ld(alpha), col_ptr(X, xcol0 + q), ld(beta), col_ptr(Y, ycol0 + q), Y->n, 0);
    return 0;
}
int lkb_basis_col(lkb_basis_t b, int i0, lkb_vec_t* view) {
    if (!b || i0 < 0 || i0 >= b->ncols) return LKB_ERR_ARG;
    if (alloc_fails()) return LKB_ERR_ALLOC;
    *view = new lkb_vec_s{b->ctx, b->kind, b->n, b->n_global, b->row0, col_ptr(b, i0), false};
    g_live[LIVE_VECS]++;
    return 0;
}
int lkb_vec_destroy(lkb_vec_t v) { if (!v) return LKB_ERR_ARG; if (v->owns) free(v->d); delete v; g_live[LIVE_VECS]--; return 0; }
int lkb_vec_zero(lkb_vec_t v) { memset(v->d, 0, (size_t)v->n * kind_size(v->kind)); return 0; }
// y = X(:, :j) coef
int lkb_basis_lincomb(lkb_basis_t X, int j, const void* coef, lkb_vec_t y) {
    if (!X || !y || j < 0 || j > X->ncols || X->n != y->n || X->kind != y->kind) return LKB_ERR_ARG;
    dispatch(X->kind, [&](auto* tag) {
        typedef typename std::remove_pointer<decltype(tag)>::type E;
        const E* x = (const E*)X->d; const E* c = (const E*)coef; E* out = (E*)y->d;
        for (int64_t r = 0; r < X->n; ++r) {
            std::complex<double> acc = 0;
            for (int i = 0; i < j; ++i) acc += std::complex<double>(x[r + X->ld * i]) * std::complex<double>(c[i]);
            if constexpr (std::is_floating_point<E>::value) out[r] = (E)acc.real();
            else out[r] = E((typename E::value_type)acc.real(), (typename E::value_type)acc.imag());
        }
    });
    return 0;
}
// initialize_krylov_subspace(X, X0): zero X, X(:p0) = X0, orthonormalize_basis(X(:p0)) = unpivoted QR with R discarded
int lkb_initialize_krylov_subspace(lkb_basis_t X, lkb_basis_t X0, int x0col0, int p0) {
    lkb_basis_zero(X, 0, X->ncols);
    if (!X0) return 0;
    const size_t es = kind_size(X->kind);
    for (int q = 0; q < p0; ++q) memcpy(col_ptr(X, q), col_ptr(X0, x0col0 + q), (size_t)X->n * es);
    std::vector<char> R((size_t)p0 * p0 * es, 0);
    uint64_t seed = 4242;
    switch (X->kind) {
        case KS: lko_qr_s(X->n, X->d, X->ld, p0, R.data(), p0, (float)atol_of(KS), &seed, 0); break;
        case KD: lko_qr_d(X->n, X->d, X->ld, p0, R.data(), p0, atol_of(KD), &seed, 0); break;
        case KC: lko_qr_c(X->n, X->d, X->ld, p0, R.data(), p0, (float)atol_of(KC), &seed, 0); break;
        default: lko_qr_z(X->n, X->d, X->ld, p0, R.data(), p0, atol_of(KZ), &seed, 0); break;
    }
    return 0;
}
int lkb_qr_pivoting(lkb_basis_t Q, int col0, int p, void* R, int ldr, int32_t* perm, double tol, int32_t* info) {
    if (!g_qr_pivoting) { set_error("mock: no pivoting-QR callback"); return LKB_ERR_ARG; }
    return g_qr_pivoting(Q->kind, Q->n, p, col_ptr(Q, col0), Q->ld, R, ldr, perm, tol, info);
}

}  // extern "C"
