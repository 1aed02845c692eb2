// host_shells_mock.cu -- TEST INFRASTRUCTURE: runs the product's host shells (lkb_eig.cu: eigs, eighs, svds, krylov_schur --
// their control flow, LAPACK calls, sorting, restarts, post-processing, write_intermediate side effects) WITHOUT a GPU.
//
// The translation unit lkb_eig.cu is included verbatim.  Everything it reaches on the device side is replaced here:
//   * the CUDA runtime calls it makes directly are redirected to host equivalents by macros ("device" memory = host memory);
//   * the internal step API (arnoldi / lanczos / bidiag enqueue-fetch-collect, basis GEMM, vector helpers, allocation) is
//     implemented on the CPU -- the Krylov steps by the C oracle (oracle/liblk_oracle.so), so that the Hessenberg / tridiagonal /
//     bidiagonal columns the shells see are exactly those the Python oracle shells see.
// tests/test_host_shells_mock.py then requires the C++ shells and the Python oracle shells to agree.  Nothing here is part of
// the product: the library never contains this file, and the GPU parity tests remain the check of the real device path.
#include <complex>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <map>
#include <vector>
#include "../include/lkb.h"
#include "lkb_internal.h"

// ---- CUDA runtime calls made directly by lkb_eig.cu -> host ----------------------------------------------------------------
cudaError_t mock_malloc_host(void** p, size_t n);      // (host_mock_common.inc: counted, can be made to fail)
cudaError_t mock_free_host(void* p);
static cudaError_t mock_memcpy2d(void* dst, size_t dpitch, const void* src, size_t spitch, size_t width, size_t height) {
    for (size_t r = 0; r < height; ++r) memcpy((char*)dst + r * dpitch, (const char*)src + r * spitch, width);
    return cudaSuccess;
}
#define cudaMallocHost(p, n) mock_malloc_host((void**)(p), (n))
#define cudaFreeHost(p) mock_free_host(p)
#define cudaEventCreateWithFlags(e, f) (*(e) = (cudaEvent_t)(uintptr_t)1, cudaSuccess)
#define cudaEventDestroy(e) ((void)(e), cudaSuccess)
#define cudaEventRecord(e, s) ((void)(e), (void)(s), cudaSuccess)
#define cudaEventSynchronize(e) ((void)(e), cudaSuccess)
#define cudaStreamSynchronize(s) ((void)(s), cudaSuccess)
#define cudaMemcpyAsync(d, s, n, k, st) (memmove((d), (s), (n)), (void)(st), cudaSuccess)
#define cudaMemcpy2DAsync(d, dp, s, sp, w, h, k, st) mock_memcpy2d((d), (dp), (s), (sp), (w), (h))

#include "lkb_eig.cu"        // the product's host shells, verbatim

#include "host_mock_common.inc"

cudaError_t mock_malloc_host(void** p, size_t n) {
    *p = alloc_fails() ? nullptr : calloc(1, n ? n : 1);
    if (!*p) return cudaErrorMemoryAllocation;
    g_live[LIVE_PINNED]++;
    return cudaSuccess;
}
cudaError_t mock_free_host(void* p) { free(p); g_live[LIVE_PINNED]--; return cudaSuccess; }

namespace {
std::vector<char> g_col;          // the H / T / B column of the step enqueued last (one step is in flight at a time)
int g_info = 0;
void stash_column(const void* H, int ldh, int col, size_t es) {
    g_col.assign((size_t)ldh * es, 0);
    memcpy(g_col.data(), (const char*)H + (size_t)ldh * col * es, (size_t)ldh * es);
}
}  // namespace

namespace lkb {

// Y(:, q) = sum_i X(:, i) Z(i, q)
void launch_basis_gemm(int kind, cudaStream_t, const void* X, int64_t ldx, int k, const void* Z, int ldz, int p, void* Y, int64_t ldy,
                       int64_t n, int) {
    dispatch(kind, [&](auto* tag) {
        typedef typename std::remove_pointer<decltype(tag)>::type E;
        const E* x = (const E*)X; const E* z = (const E*)Z; E* y = (E*)Y;
        for (int q = 0; q < p; ++q)
            for (int64_t r = 0; r < n; ++r) {
                std::complex<double> acc = 0;
                for (int i = 0; i < k; ++i) acc += std::complex<double>(x[r + ldx * i]) * std::complex<double>(z[i + (int64_t)ldz * q]);
                if constexpr (std::is_floating_point<E>::value) y[r + ldy * q] = (E)acc.real();
                else y[r + ldy * q] = E((typename E::value_type)acc.real(), (typename E::value_type)acc.imag());
            }
    });
}

// ---- Krylov steps: one step of the C oracle on the host copy of the basis; the new column travels through g_col -----------------
int arnoldi_enqueue(lkb_op_s* A, lkb_basis_s* X, int kstart, int kend, double tol, bool tr) {
    if (kstart != kend) { set_error("mock: one step at a time"); return LKB_ERR_ARG; }
    const int kdim = X->ncols - 1, ldh = kdim + 1; const size_t es = kind_size(X->kind);
    std::vector<char> H((size_t)ldh * kdim * es, 0);
    switch (X->kind) {
        case KS: g_info = lko_arnoldi_s(A->user, X->n, X->d, X->ld, H.data(), ldh, kdim, kstart, kend, (float)tol, tr, 1, &g_oracle_seed); break;
        case KD: g_info = lko_arnoldi_d(A->user, X->n, X->d, X->ld, H.data(), ldh, kdim, kstart, kend, tol, tr, 1, &g_oracle_seed); break;
        case KC: g_info = lko_arnoldi_c(A->user, X->n, X->d, X->ld, H.data(), ldh, kdim, kstart, kend, (float)tol, tr, 1, &g_oracle_seed); break;
        default: g_info = lko_arnoldi_z(A->user, X->n, X->d, X->ld, H.data(), ldh, kdim, kstart, kend, tol, tr, 1, &g_oracle_seed); break;
    }
    stash_column(H.data(), ldh, kstart - 1, es);
    return 0;
}
static void fetch_into(void* slot, int ld, size_t es) {
    memcpy(slot, g_col.data(), (size_t)ld * es);
    memcpy((char*)slot + (size_t)ld * es, &g_info, sizeof(int));
}
static void collect_from(const void* slot, void* M, int ld, int k, size_t es, int32_t* info) {
    memcpy((char*)M + (size_t)ld * (k - 1) * es, slot, (size_t)std::min(ld, k + 1) * es);       // rows 0..k of column k
    int v; memcpy(&v, (const char*)slot + (size_t)ld * es, sizeof(int)); *info = v;
}
int arnoldi_collect(lkb_op_s* A, lkb_basis_s* X, void* H, int ldh, int32_t* info, int kstart, int, bool tr, const void* slot) {
    if (ldh != X->ncols) { set_error("mock: ldh"); return LKB_ERR_ARG; }
    collect_from(slot, H, ldh, kstart, kind_size(X->kind), info);
    if (tr) A->n_rmatvec++; else A->n_matvec++;
    return 0;
}
int lanczos_enqueue(lkb_op_s* A, lkb_basis_s* X, int kstart, int kend, double tol) {
    if (kstart != kend) { set_error("mock: one step at a time"); return LKB_ERR_ARG; }
    const int kdim = X->ncols - 1, ldt = kdim + 1; const size_t es = kind_size(X->kind);
    std::vector<char> T((size_t)ldt * kdim * es, 0);
    switch (X->kind) {
        case KS: g_info = lko_lanczos_s(A->user, X->n, X->d, X->ld, T.data(), ldt, kdim, kstart, kend, (float)tol); break;
        case KD: g_info = lko_lanczos_d(A->user, X->n, X->d, X->ld, T.data(), ldt, kdim, kstart, kend, tol); break;
        case KC: g_info = lko_lanczos_c(A->user, X->n, X->d, X->ld, T.data(), ldt, kdim, kstart, kend, (float)tol); break;
        default: g_info = lko_lanczos_z(A->user, X->n, X->d, X->ld, T.data(), ldt, kdim, kstart, kend, tol); break;
    }
    stash_column(T.data(), ldt, kstart - 1, es);
    return 0;
}
int krylov_fetch_async(lkb_ctx_s*, int kind, int ld, int, int, void* slot) { fetch_into(slot, ld, kind_size(kind)); return 0; }
int lanczos_collect(lkb_op_s* A, lkb_basis_s* X, void* T, int ldt, int32_t* info, int kstart, int, const void* slot) {
    collect_from(slot, T, ldt, kstart, kind_size(X->kind), info);
    A->n_matvec++;
    return 0;
}
static lkb_basis_s* g_V = nullptr;     // bidiag_collect does not receive V: remembered from bidiag_enqueue
int bidiag_enqueue(lkb_op_s* A, lkb_basis_s* U, lkb_basis_s* V, int kstart, int kend, double tol) {
    if (kstart != kend) { set_error("mock: one step at a time"); return LKB_ERR_ARG; }
    const int kdim = U->ncols - 1, ldb = kdim + 1; const size_t es = kind_size(U->kind);
    std::vector<char> B((size_t)ldb * kdim * es, 0);
    g_V = V;
    switch (U->kind) {
        case KS: g_info = lko_bidiag_s(A->user, U->n, V->n, U->d, U->ld, V->d, V->ld, B.data(), ldb, kdim, kstart, kend, (float)tol); break;
        case KD: g_info = lko_bidiag_d(A->user, U->n, V->n, U->d, U->ld, V->d, V->ld, B.data(), ldb, kdim, kstart, kend, tol); break;
        case KC: g_info = lko_bidiag_c(A->user, U->n, V->n, U->d, U->ld, V->d, V->ld, B.data(), ldb, kdim, kstart, kend, (float)tol); break;
        default: g_info = lko_bidiag_z(A->user, U->n, V->n, U->d, U->ld, V->d, V->ld, B.data(), ldb, kdim, kstart, kend, tol); break;
    }
    stash_column(B.data(), ldb, kstart - 1, es);
    return 0;
}
int bidiag_collect(lkb_op_s* A, lkb_basis_s* U, void* B, int ldb, int32_t* info, int kstart, int, const void* slot) {
    collect_from(slot, B, ldb, kstart, kind_size(U->kind), info);
    A->n_matvec++; A->n_rmatvec++;
    return 0;
}

}  // namespace lkb
