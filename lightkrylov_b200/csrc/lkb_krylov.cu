// lkb_krylov.cu -- the Krylov step loops (arnoldi / lanczos / bidiagonalization), the Gram-Schmidt
// entry points and qr_no_pivoting, enqueued on the context stream and captured as CUDA graphs.
//
// Host control flow mirrors the reference's step loops
//   src/Krylov/arnoldi.fypp:34-73, lanczos.fypp:22-41 + 46-64, golub_kahan.fypp:26-61,
//   gram_schmidt.fypp:12-200, qr.fypp:116-167
// but every O(n) operation is one of the fused kernels and every O(kdim) scalar decision
// (H column = c1 + c2, beta = ||w||, breakdown test) happens on the device, so a whole
// kstart..kend factorisation is a single graph launch with one host sync at the end.
#include <stdio.h>
#include <string.h>
#include <vector>
#include "../../include/lkb.h"
#include "lkb_internal.h"

using namespace lkb;

namespace lkb {

int dot_reduce(lkb_ctx_s* c, int kind, const void* V, int64_t ld, int j, const void* w, int64_t n, void* out, const int* flags) {
    prof_launch(c, PC_DOT, 1, [&] { launch_multidot(kind, c->stream, V, ld, j, w, n, c->partial, out, c->counter, flags, c->sms, c->p2p_arg()); });
    LKB_TRY(check_launch(c, "multidot"));
    return allreduce_w(c, out, (size_t)(j + 1) * (kind_cplx(kind) ? 2 : 1));
}
int axpy_sub(lkb_ctx_s* c, int kind, const void* V, int64_t ld, int j, const void* coef, void* w, int64_t n, bool want_norm,
             const int* flags) {
    prof_launch(c, PC_AXPY, 1, [&] {
        launch_multiaxpy(kind, c->stream, V, ld, j, coef, w, n, want_norm, c->partial, c->nrm2, c->counter, flags, c->sms, c->p2p_arg());
    });
    LKB_TRY(check_launch(c, "multiaxpy"));
    return want_norm ? allreduce_w(c, c->nrm2, 1) : 0;
}

int dgs_enqueue(lkb_ctx_s* c, int kind, const void* V, int64_t ld, int j, void* w, int64_t n, int* flags,
                bool want_norm, bool want_gsinfo, const FinArgs* fin) {
    if (j <= 0) {
        if (want_norm) return norm2_enqueue(c, kind, w, n, flags);
        return 0;
    }
    LKB_TRY(ensure_ws(c, j + 1));
    // serpentine sweeps: pass-1 dot, fused middle and final update walk the rows in alternating directions, and the
    // first direction alternates with the step index (the previous step's final update ended where this one starts)
    const int d0 = (c->serpentine && fin) ? (fin->kstep & 1) : 0;
    const int d1 = (c->serpentine && fin) ? 1 - d0 : 0;
    // pass 1 coefficients
    { SweepDir sd(d0); LKB_TRY(dot_reduce(c, kind, V, ld, j, w, n, c->c1, flags)); }
    // pass-1 update fused with the pass-2 coefficients (V read once for both) when the shape allows
    bool fused = false;
    if (c->fused && axpy_dot_supported(kind, V, ld, j, w, n)) {
        prof_begin(c, PC_FUSED);
        { SweepDir sd(d1); fused = launch_axpy_dot(kind, c->stream, V, ld, j, c->c1, w, n, c->partial, c->c2, c->counter, flags, c->sms, c->p2p_arg()); }
        prof_end(c, PC_FUSED, fused ? 1 : 0);       // (not launched only when the driver rejected the tensor map)
        LKB_TRY(check_launch(c, "axpy_dot"));
    }
    if (fused) {
        LKB_TRY(allreduce_w(c, c->c2, (size_t)(j + 1) * (kind_cplx(kind) ? 2 : 1)));
    } else {
        LKB_TRY(axpy_sub(c, kind, V, ld, j, c->c1, w, n, false, flags));
        LKB_TRY(dot_reduce(c, kind, V, ld, j, w, n, c->c2, flags));
    }
    if (want_gsinfo)
        prof_launch(c, PC_OTHER, 1, [&] {
            launch_gsinfo(c->stream, (char*)c->c2.get() + (size_t)j * (kind_cplx(kind) ? 16 : 8), kind_cplx(kind), atol_of(kind), c->flags);
        });
    if (fin) {
        // pass-2 update + predicted-norm normalisation + H/T/B column + (optional) halo push in ONE kernel
        SweepDir sd(d0);
        prof_launch(c, PC_AXPY, 1, [&] {
            launch_multiaxpy_fin(kind, c->stream, V, ld, j, fin->with_c1 ? c->c1.get() : nullptr, c->c2, w, n, c->partial, c->nrm2, c->counter,
                                 fin->hcol, fin->tol, atol_of(kind), c->inv, flags, fin->kstep, fin->mode, c->sms, c->p2p_arg(), fin->hp);
        });
        return check_launch(c, "multiaxpy_fin");
    }
    return axpy_sub(c, kind, V, ld, j, c->c2, w, n, want_norm, flags);
}

// Orthogonalisation + normalisation + column update of ONE Krylov step (everything after the matvec):
//   CGS2 of w against V(:, 0:j), beta = ||w||, column of H / T / B, breakdown decision, w /= beta.
// mode 0 arnoldi (hcol(0:j) = c1 + c2), 1 lanczos, 2 bidiag (only hcol(j) = beta is written).
// Default: the final pass is k_multiaxpy_fin (3 kernels + 1 empty launch per step, 2 reductions).  Where fin_usable
// rules it out: the round-1 sequence (multi-axpy with norm, allreduce, k_update, k_scale_dev).
int step_tail_enqueue(lkb_ctx_s* c, int kind, const void* V, int64_t ld, int j, void* w, int64_t n, int mode, double tol,
                      int kstep, void* hcol, const HaloP2P* hp) {
    if (fin_usable(c, j)) {
        const FinArgs fa{mode, tol, kstep, hcol, mode == 0, hp};
        LKB_TRY(dgs_enqueue(c, kind, V, ld, j, w, n, c->flags, false, false, &fa));
    } else {
        LKB_TRY(dgs_enqueue(c, kind, V, ld, j, w, n, c->flags, true, false));
        prof_launch(c, PC_OTHER, 1, [&] {
            launch_update(kind, c->stream, mode == 0 ? c->c1.get() : nullptr, mode == 0 ? c->c2.get() : nullptr, j, c->nrm2, hcol, tol,
                          atol_of(kind), c->inv, c->flags, kstep, mode);
        });
    }
    prof_launch(c, PC_OTHER, 1, [&] { launch_scale_dev(kind, c->stream, w, n, c->inv, c->flags, kstep, c->sms, hp); });
    return check_launch(c, "step tail");
}

int capture_graph(lkb_ctx_s* c, const char* what, const std::function<int()>& body, GraphExec* ge) {
    const int64_t l0 = c->launches;
    cudaError_t e = cudaStreamBeginCapture(c->stream, cudaStreamCaptureModeThreadLocal);
    if (e != cudaSuccess) { set_error("%sgraph capture failed: %s", what, cudaGetErrorString(e)); return LKB_ERR_CUDA; }
    c->capturing = true;
    int r = body();
    c->capturing = false;
    cudaGraph_t g = nullptr;
    e = cudaStreamEndCapture(c->stream, &g);
    ge->launches = c->launches - l0;
    c->launches = l0;
    if (r == 0 && e != cudaSuccess) { set_error("%sgraph capture failed: %s", what, cudaGetErrorString(e)); r = LKB_ERR_CUDA; }
    if (r == 0 && cudaGraphInstantiate(ge->exec.out(), g, 0) != cudaSuccess) { set_error("%sgraph instantiate failed", what); r = LKB_ERR_CUDA; }
    if (g) cudaGraphDestroy(g);
    return r;
}

// Run `body` (which only enqueues work on c->stream) either directly or through a cached CUDA graph.
static int run_maybe_graph(lkb_ctx_s* c, bool allow_graph, const std::string& key, const std::function<int()>& body) {
    if (!(c->graphs && allow_graph) || c->profile) return body();
    auto it = c->graph_cache.find(key);
    if (it == c->graph_cache.end()) {
        GraphExec ge;
        LKB_TRY(capture_graph(c, "", body, &ge));
        if (c->graph_cache.size() > 4096) c->graph_cache.clear();   // bound the cache
        it = c->graph_cache.emplace(key, std::move(ge)).first;
    }
    LKB_CUDA(cudaGraphLaunch(it->second.exec, c->stream));
    c->launches += it->second.launches;
    return 0;
}

static std::string make_key(const char* tag, const lkb_op_s* A, const lkb_basis_s* X, const lkb_basis_s* Y,
                            int kstart, int kend, double tol, int trans) {
    char buf[256];
    snprintf(buf, sizeof(buf), "%s:%llu:%llu:%llu:%d:%d:%a:%d", tag, (unsigned long long)A->uid,
             (unsigned long long)X->uid, (unsigned long long)(Y ? Y->uid : 0), kstart, kend, tol, trans);
    return std::string(buf);
}

static void host_store(int kind, void* H, int64_t idx, const void* src, int64_t sidx) {
    const size_t es = kind_size(kind);
    memcpy((char*)H + (size_t)idx * es, (const char*)src + (size_t)sidx * es, es);
}
static double host_abs(int kind, const void* p) {
    switch (kind) {
        case KS: return fabs((double)*(const float*)p);
        case KD: return fabs(*(const double*)p);
        case KC: return hypot((double)((const float*)p)[0], (double)((const float*)p)[1]);
        default: return hypot(((const double*)p)[0], ((const double*)p)[1]);
    }
}

int fetch_coeffs(lkb_ctx_s* c, int kind, int j, bool two, std::vector<Scalar>& out, double* nrm2, int* flags) {
    const size_t wsz = kind_cplx(kind) ? 16 : 8;
    LKB_TRY(ensure_hstage(c, 2 * (size_t)(j + 1) * 16 + 4096));
    char* hs = (char*)c->hstage;
    if (j > 0) {
        LKB_CUDA(cudaMemcpyAsync(hs, c->c1, (size_t)j * wsz, cudaMemcpyDeviceToHost, c->stream));
        if (two) LKB_CUDA(cudaMemcpyAsync(hs + (size_t)j * wsz, c->c2, (size_t)j * wsz, cudaMemcpyDeviceToHost, c->stream));
    }
    char* tail = hs + 2 * (size_t)j * wsz;
    LKB_CUDA(cudaMemcpyAsync(tail, c->nrm2, 16, cudaMemcpyDeviceToHost, c->stream));
    LKB_CUDA(cudaMemcpyAsync(tail + 16, c->flags, F_COUNT * sizeof(int), cudaMemcpyDeviceToHost, c->stream));
    LKB_CUDA(cudaStreamSynchronize(c->stream));
    out.assign(j, Scalar{0, 0});
    for (int i = 0; i < j; ++i) {
        const double* a = (const double*)(hs + (size_t)i * wsz);
        out[i].re = a[0]; if (kind_cplx(kind)) out[i].im = a[1];
        if (two) {
            const double* b = (const double*)(hs + (size_t)(j + i) * wsz);
            out[i].re += b[0]; if (kind_cplx(kind)) out[i].im += b[1];
        }
    }
    if (nrm2) *nrm2 = *(const double*)tail;
    if (flags) memcpy(flags, tail + 16, F_COUNT * sizeof(int));
    return 0;
}
// upload host coefficients (kind elements, length len) as W type into c->coefd, scaled by sgn
static int upload_coef(lkb_ctx_s* c, int kind, const void* coef, int len, double sgn) {
    const size_t wsz = kind_cplx(kind) ? 16 : 8;
    LKB_TRY(ensure_hstage(c, (size_t)len * 16 + 4096));
    LKB_TRY(ensure_coefd(c, std::max((size_t)len * 16, (size_t)4096)));
    LKB_CUDA(cudaStreamSynchronize(c->stream));   // hstage may still be in flight
    for (int i = 0; i < len; ++i) {
        const cd s = load_kind(kind, coef, i);
        double* d = (double*)((char*)c->hstage + (size_t)i * wsz);
        d[0] = sgn * s.real(); if (kind_cplx(kind)) d[1] = sgn * s.imag();
    }
    LKB_CUDA(cudaMemcpyAsync(c->coefd, c->hstage, (size_t)len * wsz, cudaMemcpyHostToDevice, c->stream));
    return 0;
}

static int reset_flags(lkb_ctx_s* c) {
    LKB_CUDA(cudaMemsetAsync(c->flags, 0, F_COUNT * sizeof(int), c->stream));
    return 0;
}

// ---- the frame shared by arnoldi (p = 1), lanczos and bidiagonalization -------------------------------------------------
// X (U for bidiag) holds kdim + 1 columns; the device H / T / B has leading dimension kdim + 1.
// Enqueue `steps` kstart..kend after the shared prologue, directly or through the graph cached under (tag, A, X, Y, ...).
static int krylov_run(const char* tag, lkb_op_s* A, const lkb_basis_s* X, const lkb_basis_s* Y, int kstart, int kend, double tol,
                      bool tr, const std::function<int()>& steps) {
    lkb_ctx_s* c = X->ctx;
    LKB_TRY(ensure_Hd(c, (size_t)X->ncols * (X->ncols - 1) * kind_size(X->kind)));
    LKB_TRY(ensure_ws(c, kend + 1));
    auto body = [&]() -> int {
        LKB_TRY(reset_flags(c));
        PdlScope pdl(c->pdl && !c->profile);      // the kernels of the step loop overlap their heads with the predecessors' tails
        return steps();
    };
    return run_maybe_graph(c, op_capturable(A), make_key(tag, A, X, Y, kstart, kend, tol, tr), body);
}
// The synchronous entry points: enqueue, copy the new columns and the flags to the staging buffer, wait, collect from it.
static int krylov_sync(const lkb_basis_s* X, int kstart, int kend, const std::function<int()>& enqueue,
                       const std::function<int(const void*)>& collect) {
    lkb_ctx_s* c = X->ctx;
    LKB_TRY(ensure_hstage(c, (size_t)X->ncols * (kend - kstart + 1) * kind_size(X->kind) + 4096));
    LKB_TRY(enqueue());
    LKB_TRY(krylov_fetch_async(c, X->kind, X->ncols, kstart, kend, c->hstage));
    LKB_CUDA(cudaStreamSynchronize(c->stream));
    return collect(c->hstage);
}
// The flags krylov_fetch_async staged behind the ncol columns; a NaN norm is an error with message `nan_msg`.
static int staged_flags(const lkb_basis_s* X, int ncol, const void* host, int* hf, const char* nan_msg) {
    memcpy(hf, (const char*)host + (size_t)X->ncols * ncol * kind_size(X->kind), F_COUNT * sizeof(int));
    if (hf[F_NAN]) { set_error("%s", nan_msg); return LKB_ERR_NAN; }
    return 0;
}

// is_orthonormal (src/Krylov/utilities.fypp:90-98): mnorm(Gram(X) - I, "Fro") > rtol_sp (hard-wired, all kinds) => not orthonormal
static int check_orthonormal(lkb_basis_s* X, int j, bool* ok) {
    lkb_ctx_s* c = X->ctx;
    *ok = true;
    std::vector<Scalar> col;
    double fro2 = 0.0;                                         // squared Frobenius norm of G - I, column by column
    const double lim2 = 1e-3 * 1e-3;                           // rtol_sp = sqrt(atol_sp) = 1e-3
    for (int q = 0; q < j && fro2 <= lim2; ++q) {
        LKB_TRY(ensure_ws(c, j + 1));
        LKB_TRY(dot_reduce(c, X->kind, X->d, X->ld, j, col_ptr(X, q), X->n, c->c1, nullptr));
        LKB_TRY(fetch_coeffs(c, X->kind, j, false, col, nullptr, nullptr));
        for (int i = 0; i < j; ++i) {
            const double re = col[i].re - (i == q ? 1.0 : 0.0);
            fro2 += re * re + col[i].im * col[i].im;
        }
    }
    *ok = !(fro2 > lim2);
    return 0;
}

}  // namespace lkb

extern "C" {

int lkb_basis_innerprod(lkb_basis_t X, int j, lkb_basis_t W, int wcol0, int p, void* out, int ldout) {
    if (!X || !W || !out || j < 0 || j > X->ncols || wcol0 < 0 || wcol0 + p > W->ncols || X->n != W->n || X->kind != W->kind)
        { set_error("innerprod: bad arguments"); return LKB_ERR_ARG; }
    lkb_ctx_s* c = X->ctx;
    std::vector<Scalar> col;
    for (int q = 0; q < p; ++q) {
        LKB_TRY(ensure_ws(c, j + 1));
        LKB_TRY(dot_reduce(c, X->kind, X->d, X->ld, j, col_ptr(W, wcol0 + q), X->n, c->c1, nullptr));
        LKB_TRY(fetch_coeffs(c, X->kind, j, false, col, nullptr, nullptr));
        for (int i = 0; i < j; ++i)
            store_kind(X->kind, out, (size_t)i + (size_t)ldout * q, cd(col[i].re, col[i].im));
    }
    return 0;
}

int lkb_basis_lincomb_sub(lkb_basis_t X, int j, const void* coef, int ldcoef, lkb_basis_t W, int wcol0, int p) {
    if (!X || !W || !coef || j < 0 || j > X->ncols || wcol0 < 0 || wcol0 + p > W->ncols || X->n != W->n || X->kind != W->kind)
        { set_error("lincomb_sub: bad arguments"); return LKB_ERR_ARG; }
    lkb_ctx_s* c = X->ctx;
    for (int q = 0; q < p; ++q) {
        LKB_TRY(upload_coef(c, X->kind, (const char*)coef + (size_t)ldcoef * q * kind_size(X->kind), j, 1.0));
        LKB_TRY(axpy_sub(c, X->kind, X->d, X->ld, j, c->coefd, col_ptr(W, wcol0 + q), X->n, false, nullptr));
    }
    return 0;
}

int lkb_basis_lincomb(lkb_basis_t X, int j, const void* coef, lkb_vec_t y) {
    if (!X || !y || !coef || j < 0 || j > X->ncols || X->n != y->n || X->kind != y->kind)
        { set_error("lincomb: bad arguments"); return LKB_ERR_ARG; }
    lkb_ctx_s* c = X->ctx;
    LKB_TRY(upload_coef(c, X->kind, coef, j, -1.0));
    LKB_TRY(lkb_vec_zero(y));
    return axpy_sub(c, X->kind, X->d, X->ld, j, c->coefd, y->d, X->n, false, nullptr);
}

static int gs_common(lkb_basis_t X, int j, lkb_basis_t W, int wcol0, int p, int32_t chk, void* beta, int ldbeta,
                     int32_t* info, bool two_pass) {
    if (!X || !W || !info || j < 0 || j > X->ncols || wcol0 < 0 || wcol0 + p > W->ncols || X->n != W->n || X->kind != W->kind)
        { set_error("gram_schmidt: bad arguments"); return LKB_ERR_ARG; }
    if (beta && ldbeta < j) { set_error("gram_schmidt: beta has the wrong shape (assert_shape)"); return LKB_ERR_ARG; }
    lkb_ctx_s* c = X->ctx;
    *info = 0;
    if (chk) {
        bool ok = true;
        LKB_TRY(check_orthonormal(X, j, &ok));
        if (!ok) { set_error("Input basis not orthonormal."); return LKB_ERR_ARG; }
    }
    std::vector<Scalar> col;
    int hf[F_COUNT];
    for (int q = 0; q < p; ++q) {
        void* w = col_ptr(W, wcol0 + q);
        LKB_TRY(reset_flags(c));
        if (two_pass) {
            LKB_TRY(dgs_enqueue(c, X->kind, X->d, X->ld, j, w, X->n, c->flags, false, true));
        } else {
            LKB_TRY(ensure_ws(c, j + 1));
            LKB_TRY(dot_reduce(c, X->kind, X->d, X->ld, j, w, X->n, c->c1, nullptr));
            prof_launch(c, PC_OTHER, 1, [&] {
                launch_gsinfo(c->stream, (char*)c->c1.get() + (size_t)j * (kind_cplx(X->kind) ? 16 : 8), 0, atol_of(X->kind), c->flags);
            });
            LKB_TRY(axpy_sub(c, X->kind, X->d, X->ld, j, c->c1, w, X->n, false, nullptr));
        }
        LKB_TRY(fetch_coeffs(c, X->kind, j, two_pass, col, nullptr, hf));
        if (hf[F_GSINFO]) *info = q + 1;
        if (beta)
            for (int i = 0; i < j; ++i)
                store_kind(X->kind, beta, (size_t)i + (size_t)ldbeta * q, cd(col[i].re, col[i].im));
    }
    return 0;
}
int lkb_dgs_step(lkb_basis_t X, int j, lkb_basis_t W, int wcol0, int p, int32_t chk, void* beta, int ldbeta, int32_t* info) {
    return gs_common(X, j, W, wcol0, p, chk, beta, ldbeta, info, true);
}
int lkb_orthogonalize_against_basis(lkb_basis_t X, int j, lkb_basis_t W, int wcol0, int p, int32_t chk, void* beta,
                                    int ldbeta, int32_t* info) {
    return gs_common(X, j, W, wcol0, p, chk, beta, ldbeta, info, false);
}

// qr_no_pivoting: src/Krylov/qr.fypp:116-167 (literal info semantics: the DGS calls reuse `info`)
int lkb_qr(lkb_basis_t Q, int col0, int p, void* R, int ldr, double tol, int32_t* info) {
    if (!Q || !R || !info || col0 < 0 || col0 + p > Q->ncols || ldr < p) { set_error("qr: bad arguments"); return LKB_ERR_ARG; }
    lkb_ctx_s* c = Q->ctx;
    const int kind = Q->kind;
    const size_t es = kind_size(kind);
    if (tol < 0) tol = atol_of(kind);
    *info = 0;
    bool flag = false;
    for (int jj = 0; jj < p; ++jj) for (int i = 0; i < p; ++i) memset((char*)R + ((size_t)i + (size_t)ldr * jj) * es, 0, es);
    std::vector<Scalar> col;
    int hf[F_COUNT];
    for (int j = 0; j < p; ++j) {
        void* q = col_ptr(Q, col0 + j);
        double nrm2 = 0;
        LKB_TRY(reset_flags(c));
        LKB_TRY(dgs_enqueue(c, kind, col_ptr(Q, col0), Q->ld, j, q, Q->n, c->flags, true, true));
        LKB_TRY(fetch_coeffs(c, kind, j, true, col, &nrm2, hf));
        if (j > 0) {
            *info = hf[F_GSINFO] ? 1 : 0;
            for (int i = 0; i < j; ++i) store_kind(kind, R, (size_t)i + (size_t)ldr * j, cd(col[i].re, col[i].im));
        }
        double beta = sqrt(fabs(nrm2));
        if (beta != beta) { set_error("|beta| = NaN detected! Abort"); return LKB_ERR_NAN; }
        if (beta < tol) {
            if (!flag) { flag = true; *info = j + 1; }
            prof_launch(c, PC_OTHER, 1, [&] { launch_fill(kind, c->stream, q, Q->n, Q->row0, LKB_DIST_NORMAL, next_seed(c), c->sms); });
            LKB_TRY(reset_flags(c));
            LKB_TRY(dgs_enqueue(c, kind, col_ptr(Q, col0), Q->ld, j, q, Q->n, c->flags, true, true));
            LKB_TRY(fetch_coeffs(c, kind, j, true, col, &nrm2, hf));
            if (j > 0) *info = hf[F_GSINFO] ? 1 : 0;
            beta = sqrt(fabs(nrm2));
        } else {
            store_kind(kind, R, (size_t)j + (size_t)ldr * j, beta);
        }
        prof_launch(c, PC_OTHER, 1, [&] { launch_scal(kind, c->stream, Scalar{1.0 / beta, 0.0}, q, Q->n, c->sms); });
        LKB_TRY(check_launch(c, "qr scal"));
    }
    return 0;
}

// qr_with_pivoting: src/Krylov/qr.fypp:32-107 (+ swap_columns :174-201), interface BaseKrylov.fypp:395-417.
// Greedy column pivoting on the down-dated squared norms Rii.  Literal details kept: Rii (SQUARED norms) is compared with
// `tol` unsquared; the down-date is Rii(i) - R(j,i)**2, a complex square for the complex kinds; `info = j` set before the
// refill of a cancelled column is overwritten by the Gram-Schmidt call that follows; a Gram-Schmidt step against the empty
// section Q(:0) is a no-op with info = 0.  perm is 1-based, as the reference returns it.
int lkb_qr_pivoting(lkb_basis_t Q, int col0, int p, void* R, int ldr, int32_t* perm, double tol, int32_t* info) {
    if (!Q || !R || !perm || !info || col0 < 0 || p < 1 || col0 + p > Q->ncols || ldr < p) { set_error("qr_pivoting: bad arguments"); return LKB_ERR_ARG; }
    lkb_ctx_s* c = Q->ctx;
    const int kind = Q->kind;
    const size_t es = kind_size(kind);
    const bool sp = (kind == KS || kind == KC), cplx = kind_cplx(kind);
    if (tol < 0) tol = atol_of(kind);
    *info = 0;
    auto Rat = [&](int i, int j) { return (char*)R + ((size_t)i + (size_t)ldr * j) * es; };
    auto qcol = [&](int i) { return col_ptr(Q, col0 + i); };
    auto round_kind = [&](Scalar s) { if (sp) { s.re = (double)(float)s.re; s.im = (double)(float)s.im; } if (!cplx) s.im = 0.0; return s; };
    for (int j = 0; j < p; ++j) for (int i = 0; i < p; ++i) memset(Rat(i, j), 0, es);
    std::vector<Scalar> Rii(p, Scalar{0, 0}), col;
    int hf[F_COUNT];
    for (int i = 0; i < p; ++i) {
        perm[i] = i + 1;
        LKB_TRY(vec_dot_sync(c, kind, qcol(i), qcol(i), Q->n, &Rii[i]));
        Rii[i] = round_kind(Rii[i]);
    }
    DevBuf tmp(c);
    // Q(i) <- rand ; double_gram_schmidt_step(Q(i), Q(:i-1)) ; returns the step's info and the norm afterwards
    auto refill = [&](int i, int32_t* ginfo, double* beta) -> int {
        prof_launch(c, PC_OTHER, 1, [&] { launch_fill(kind, c->stream, qcol(i), Q->n, Q->row0, LKB_DIST_NORMAL, next_seed(c), c->sms); });
        double nrm2 = 0;
        LKB_TRY(reset_flags(c));
        LKB_TRY(dgs_enqueue(c, kind, qcol(0), Q->ld, i, qcol(i), Q->n, c->flags, true, true));
        LKB_TRY(fetch_coeffs(c, kind, i, true, col, &nrm2, hf));
        *ginfo = (i > 0 && hf[F_GSINFO]) ? 1 : 0;
        *beta = sqrt(fabs(nrm2));
        return 0;
    };
    for (int j = 0; j < p; ++j) {
        int idx = 0; double best = -1.0;                                    // maxloc(abs(Rii)): first maximum
        for (int i = 0; i < p; ++i) { const double a = hypot(Rii[i].re, Rii[i].im); if (a > best) { best = a; idx = i; } }
        if (best < tol) {                                                   // rank exhausted: random orthonormal completion (:55-66)
            for (int i = j; i < p; ++i) {
                int32_t g = 0; double beta = 0;
                LKB_TRY(refill(i, &g, &beta));
                prof_launch(c, PC_OTHER, 1, [&] { launch_scal(kind, c->stream, Scalar{1.0 / beta, 0.0}, qcol(i), Q->n, c->sms); });
                LKB_TRY(check_launch(c, "qr_pivoting completion"));
            }
            *info = j + 1;
            break;
        }
        // swap_columns(Q, R, Rii, perm, j, idx)
        if (idx != j) {
            const size_t bytes = (size_t)Q->n * es;
            if (!tmp.p && bytes) LKB_TRY(tmp.alloc(bytes));
            if (bytes) {
                LKB_CUDA(cudaMemcpyAsync(tmp.p, qcol(j), bytes, cudaMemcpyDeviceToDevice, c->stream));
                LKB_CUDA(cudaMemcpyAsync(qcol(j), qcol(idx), bytes, cudaMemcpyDeviceToDevice, c->stream));
                LKB_CUDA(cudaMemcpyAsync(qcol(idx), tmp.p, bytes, cudaMemcpyDeviceToDevice, c->stream));
            }
            std::swap(Rii[j], Rii[idx]);
            std::swap(perm[j], perm[idx]);
            char t[16];
            for (int r = 0; r < j; ++r) { memcpy(t, Rat(r, j), es); memcpy(Rat(r, j), Rat(r, idx), es); memcpy(Rat(r, idx), t, es); }
        }
        double beta = 0;
        LKB_TRY(vec_norm_sync(c, kind, qcol(j), Q->n, &beta));
        if (beta != beta) { set_error("|beta| = NaN detected! Abort"); return LKB_ERR_NAN; }
        if (beta < tol) {                                                   // cancelled column (:80-87)
            int32_t g = 0;
            LKB_TRY(refill(j, &g, &beta));
            *info = g;                                                      // `info = j` is overwritten by the DGS call
        } else {
            store_kind(kind, R, (size_t)j + (size_t)ldr * j, beta);
        }
        prof_launch(c, PC_OTHER, 1, [&] { launch_scal(kind, c->stream, Scalar{1.0 / beta, 0.0}, qcol(j), Q->n, c->sms); });
        for (int i = j + 1; i < p; ++i) {                                   // orthogonalise the trailing columns (:93-97)
            Scalar b{0, 0};
            LKB_TRY(vec_dot_sync(c, kind, qcol(j), qcol(i), Q->n, &b));
            b = round_kind(b);
            prof_launch(c, PC_OTHER, 1, [&] { launch_axpby(kind, c->stream, Scalar{-b.re, -b.im}, qcol(j), Scalar{1.0, 0.0}, qcol(i), Q->n, c->sms); });
            store_kind(kind, R, (size_t)j + (size_t)ldr * i, cd(b.re, b.im));
            Rii[i] = round_kind(Scalar{Rii[i].re - (b.re * b.re - b.im * b.im), Rii[i].im - 2.0 * b.re * b.im});
        }
        LKB_TRY(check_launch(c, "qr_pivoting"));
        Rii[j] = Scalar{0, 0};
    }
    LKB_CUDA(cudaStreamSynchronize(c->stream));
    return 0;
}

// orthonormalize_basis (src/Krylov/utilities.fypp:70-81): in-place QR of X(:, col0 : col0 + p), R discarded
int lkb_orthonormalize_basis(lkb_basis_t X, int col0, int p, int32_t* info) {
    if (!X || !info || p < 1) { set_error("orthonormalize_basis: bad arguments"); return LKB_ERR_ARG; }
    std::vector<char> R((size_t)p * p * kind_size(X->kind));
    return lkb_qr(X, col0, p, R.data(), p, -1.0, info);
}
// initialize_krylov_subspace(X [, X0]) (src/Krylov/utilities.fypp:32-46): zero X; X(:p) = X0; orthonormalise X(:p)
int lkb_initialize_krylov_subspace(lkb_basis_t X, lkb_basis_t X0, int x0col0, int p0) {
    if (!X) { set_error("initialize_krylov_subspace: null basis"); return LKB_ERR_ARG; }
    LKB_TRY(lkb_basis_zero(X, 0, X->ncols));
    if (X0) {
        if (p0 < 1 || p0 > X->ncols) { set_error("initialize_krylov_subspace: size(X0) = %d does not fit", p0); return LKB_ERR_ARG; }
        const double one[2] = {1.0, 0.0}, zero[2] = {0.0, 0.0};
        const float onef[2] = {1.f, 0.f}, zerof[2] = {0.f, 0.f};
        const bool sp = (X->kind == KS || X->kind == KC);
        LKB_TRY(lkb_basis_axpby(sp ? (const void*)onef : (const void*)one, X0, x0col0, sp ? (const void*)zerof : (const void*)zero, X, 0, p0));
        int32_t info = 0;
        LKB_TRY(lkb_orthonormalize_basis(X, 0, p0, &info));
    }
    return 0;
}
// initialize_random_orthonormal_basis (utilities.fypp:52-62)
int lkb_initialize_random_orthonormal_basis(lkb_basis_t X, int col0, int p) {
    LKB_TRY(lkb_basis_rand(X, col0, p, 0));
    int32_t info = 0;
    return lkb_orthonormalize_basis(X, col0, p, &info);
}

// ------------------------------------------------------------------------------------------
// arnoldi
// ------------------------------------------------------------------------------------------
static int arnoldi_block(lkb_op_t A, lkb_basis_t X, void* H, int ldh, int32_t* info, int kstart, int kend,
                         double tol, bool trans, int p);

int lkb_arnoldi(lkb_op_t A, lkb_basis_t X, void* H, int ldh, int32_t* info, int32_t kstart, int32_t kend,
                double tol, int32_t transpose, int32_t blksize) {
    if (!A || !X || !H || !info) { set_error("arnoldi: null argument"); return LKB_ERR_ARG; }
    const int p = blksize > 0 ? blksize : 1;
    const int kdim = (X->ncols - p) / p;
    if (kstart <= 0) kstart = 1;
    if (kend <= 0) kend = kdim;
    if (kstart > kend || kend > kdim || ldh < (kend + 1) * p || A->kind != X->kind || A->m != X->n || A->n != X->n)
        { set_error("arnoldi: inconsistent sizes (kdim=%d kstart=%d kend=%d ldh=%d)", kdim, kstart, kend, ldh); return LKB_ERR_ARG; }
    if (tol < 0) tol = atol_of(X->kind);
    *info = 0;
    if (p > 1) return arnoldi_block(A, X, H, ldh, info, kstart, kend, tol, transpose != 0, p);

    const bool tr = transpose != 0;
    return krylov_sync(X, kstart, kend, [&] { return arnoldi_enqueue(A, X, kstart, kend, tol, tr); },
                       [&](const void* hs) { return arnoldi_collect(A, X, H, ldh, info, kstart, kend, tr, hs); });
}

}  // extern "C"

namespace lkb {
// The three phases of a p = 1 arnoldi call, exposed so that eigs can overlap the host geev of
// step k with the device work of step k+1 (SURVEY 8f rank 3).
int arnoldi_enqueue(lkb_op_s* A, lkb_basis_s* X, int kstart, int kend, double tol, bool tr) {
    lkb_ctx_s* c = X->ctx;
    const size_t es = kind_size(X->kind);
    return krylov_run("arn", A, X, nullptr, kstart, kend, tol, tr, [&]() -> int {
        bool pushed = false;       // X(k-1)'s boundary rows already sit in the neighbours' halo buffers
        for (int k = kstart; k <= kend; ++k) {
            void* w = col_ptr(X, k);
            LKB_TRY(op_apply_enqueue(A, col_ptr(X, k - 1), w, tr, c->flags, pushed));
            // the kernel that finishes X(k) also pushes its halo rows for the next step's matvec
            const HaloP2P* hp = (k < kend) ? op_halo_desc(A, k) : nullptr;
            LKB_TRY(step_tail_enqueue(c, X->kind, X->d, X->ld, k, w, X->n, 0, tol, k, (char*)c->Hd.get() + (size_t)X->ncols * (k - 1) * es, hp));
            pushed = hp != nullptr;
        }
        return 0;
    });
}
// after the stream reached the fetch: scatter the columns into the caller's H, set info, refill on breakdown
int arnoldi_collect(lkb_op_s* A, lkb_basis_s* X, void* H, int ldh, int32_t* info, int kstart, int kend, bool tr,
                    const void* host) {
    lkb_ctx_s* c = X->ctx;
    const int kind = X->kind;
    const int ldhd = X->ncols;
    const char* hs = (const char*)host;
    int hf[F_COUNT];
    LKB_TRY(staged_flags(X, kend - kstart + 1, host, hf, "|beta| = NaN detected! Abort"));
    const int kdone = hf[F_STOP] ? hf[F_INFO] : kend;
    for (int k = kstart; k <= kdone; ++k)
        for (int i = 0; i <= k; ++i)
            host_store(kind, H, (int64_t)i + (int64_t)ldh * (k - 1), hs, (int64_t)i + (int64_t)ldhd * (k - kstart));
    if (tr) A->n_rmatvec += kdone - kstart + 1; else A->n_matvec += kdone - kstart + 1;
    *info = 0;
    if (hf[F_STOP]) {
        *info = hf[F_INFO];
        if (hf[F_REFILL]) {
            // qr.fypp:153-158 : the numerically-zero vector is replaced by a normalised random one
            void* w = col_ptr(X, kdone);
            prof_launch(c, PC_OTHER, 1, [&] { launch_fill(kind, c->stream, w, X->n, X->row0, LKB_DIST_NORMAL, next_seed(c), c->sms); });
            double nrm = 0;
            LKB_TRY(vec_norm_sync(c, kind, w, X->n, &nrm));
            prof_launch(c, PC_OTHER, 1, [&] { launch_scal(kind, c->stream, Scalar{1.0 / nrm, 0.0}, w, X->n, c->sms); });
            LKB_TRY(check_launch(c, "refill"));
        }
    }
    return 0;
}
}  // namespace lkb

extern "C" {

// Block Arnoldi (blksize > 1), host-driven: arnoldi.fypp:36-71 with the per-column passes of
// DGS_basis_against_basis (columns of Y are independent within a pass) and qr_no_pivoting.
static int arnoldi_block(lkb_op_t A, lkb_basis_t X, void* H, int ldh, int32_t* info, int kstart, int kend,
                         double tol, bool trans, int p) {
    lkb_ctx_s* c = X->ctx;
    const int kind = X->kind;
    const size_t es = kind_size(kind);
    std::vector<Scalar> col;
    std::vector<char> R((size_t)p * p * es);
    int hf[F_COUNT];
    for (int k = kstart; k <= kend; ++k) {
        const int kpm = (k - 1) * p, kp = kpm + p;
        for (int i = 0; i < p; ++i) {
            LKB_TRY(op_apply_enqueue(A, col_ptr(X, kpm + i), col_ptr(X, kp + i), trans, nullptr));
            if (trans) A->n_rmatvec++; else A->n_matvec++;
        }
        for (int i = 0; i < p; i += 2) {
            LKB_TRY(reset_flags(c));
            if (i + 1 < p) {
                // two block columns per sweep of the basis (k_multidot2 / k_multiaxpy2): c laid out [2][kp+1]
                const int jp = kp + 1;
                const size_t wsz = kind_cplx(kind) ? 16 : 8;
                const size_t nd = (size_t)2 * jp * (kind_cplx(kind) ? 2 : 1);
                LKB_TRY(ensure_ws(c, 2 * jp));
                void* w0 = col_ptr(X, kp + i); void* w1 = col_ptr(X, kp + i + 1);
                for (int pass = 0; pass < 2; ++pass) {
                    void* cb = pass == 0 ? c->c1 : c->c2;
                    prof_begin(c, PC_DOT);
                    launch_multidot2(kind, c->stream, X->d, X->ld, kp, w0, w1, X->n, c->partial, cb, c->counter, nullptr, c->sms, c->p2p_arg());
                    prof_end(c, PC_DOT, 1);
                    LKB_TRY(allreduce_w(c, cb, nd));
                    prof_begin(c, PC_AXPY);
                    launch_multiaxpy2(kind, c->stream, X->d, X->ld, kp, cb, w0, w1, X->n, nullptr, c->sms);
                    prof_end(c, PC_AXPY, 1);
                    LKB_TRY(check_launch(c, "block gram-schmidt"));
                }
                LKB_TRY(ensure_hstage(c, 4 * (size_t)jp * 16 + 4096));
                char* hs = (char*)c->hstage;
                LKB_CUDA(cudaMemcpyAsync(hs, c->c1, 2 * (size_t)jp * wsz, cudaMemcpyDeviceToHost, c->stream));
                LKB_CUDA(cudaMemcpyAsync(hs + 2 * (size_t)jp * wsz, c->c2, 2 * (size_t)jp * wsz, cudaMemcpyDeviceToHost, c->stream));
                LKB_CUDA(cudaStreamSynchronize(c->stream));
                for (int q = 0; q < 2; ++q)
                    for (int r = 0; r < kp; ++r) {
                        const double* a = (const double*)(hs + ((size_t)q * jp + r) * wsz);
                        const double* b = (const double*)(hs + (2 * (size_t)jp + (size_t)q * jp + r) * wsz);
                        store_kind(kind, H, (size_t)r + (size_t)ldh * (kpm + i + q), cd(a[0] + b[0], kind_cplx(kind) ? a[1] + b[1] : 0.0));
                    }
                continue;
            }
            LKB_TRY(dgs_enqueue(c, kind, X->d, X->ld, kp, col_ptr(X, kp + i), X->n, c->flags, false, true));
            LKB_TRY(fetch_coeffs(c, kind, kp, true, col, nullptr, hf));
            for (int r = 0; r < kp; ++r)
                store_kind(kind, H, (size_t)r + (size_t)ldh * (kpm + i), cd(col[r].re, col[r].im));
        }
        int32_t qinfo = 0;
        LKB_TRY(lkb_qr(X, kp, p, R.data(), p, -1.0, &qinfo));
        double beta = 1e300;
        for (int jj = 0; jj < p; ++jj)
            for (int i = 0; i < p; ++i) {
                memcpy((char*)H + ((size_t)(kp + i) + (size_t)ldh * (kpm + jj)) * es, &R[((size_t)i + (size_t)p * jj) * es], es);
                if (i == jj) beta = std::min(beta, host_abs(kind, &R[((size_t)i + (size_t)p * jj) * es]));
            }
        if (beta < tol) { *info = kp; break; }
    }
    return 0;
}

// ------------------------------------------------------------------------------------------
// lanczos : src/Krylov/lanczos.fypp:7-64
// ------------------------------------------------------------------------------------------
int lkb_lanczos(lkb_op_t A, lkb_basis_t X, void* T, int ldt, int32_t* info, int32_t kstart, int32_t kend, double tol) {
    if (!A || !X || !T || !info) { set_error("lanczos: null argument"); return LKB_ERR_ARG; }
    const int kdim = X->ncols - 1;
    if (kstart <= 0) kstart = 1;
    if (kend <= 0) kend = kdim;
    if (kstart > kend || kend > kdim || ldt < kend + 1 || A->kind != X->kind || A->m != X->n || A->n != X->n)
        { set_error("lanczos: inconsistent sizes"); return LKB_ERR_ARG; }
    if (tol < 0) tol = atol_of(X->kind);
    *info = 0;
    return krylov_sync(X, kstart, kend, [&] { return lanczos_enqueue(A, X, kstart, kend, tol); },
                       [&](const void* hs) { return lanczos_collect(A, X, T, ldt, info, kstart, kend, hs); });
}

}  // extern "C"

namespace lkb {
// The three phases of lanczos / bidiagonalization (as for arnoldi): eighs and svds overlap the host syev / gesdd of
// step k with the device work of a speculative step k+1 (SURVEY 8f rank 3).
int lanczos_enqueue(lkb_op_s* A, lkb_basis_s* X, int kstart, int kend, double tol) {
    lkb_ctx_s* c = X->ctx;
    const int kind = X->kind;
    const size_t es = kind_size(kind);
    return krylov_run("lan", A, X, nullptr, kstart, kend, tol, false, [&]() -> int {
        bool pushed = false;
        for (int k = kstart; k <= kend; ++k) {
            void* w = col_ptr(X, k);
            char* tcol = (char*)c->Hd.get() + (size_t)X->ncols * (k - 1) * es;
            LKB_TRY(op_apply_enqueue(A, col_ptr(X, k - 1), w, false, c->flags, pushed));
            for (int i = (k - 1 > 1 ? k - 1 : 1); i <= k; ++i) {        // update_tridiag_matrix :57-59
                void* xi = col_ptr(X, i - 1);
                LKB_TRY(dot_reduce(c, kind, xi, X->ld, 1, w, X->n, c->tmpw, c->flags));
                prof_launch(c, PC_OTHER, 2, [&] {
                    launch_narrow(kind, c->stream, c->tmpw, tcol + (size_t)(i - 1) * es, 1, c->flags);
                    launch_axpy_dev(kind, c->stream, c->tmpw, -1.0, xi, w, X->n, c->flags, c->sms);
                });
            }
            const HaloP2P* hp = (k < kend) ? op_halo_desc(A, k) : nullptr;
            LKB_TRY(step_tail_enqueue(c, kind, X->d, X->ld, k, w, X->n, 1, tol, k, tcol, hp));
            pushed = hp != nullptr;
        }
        return 0;
    });
}
// D2H of the freshly written columns of the device-side H / T / B (leading dimension ldd) + flags, no sync
int krylov_fetch_async(lkb_ctx_s* c, int kind, int ldd, int kstart, int kend, void* host) {
    const size_t es = kind_size(kind);
    const int ncol = kend - kstart + 1;
    char* hs = (char*)host;
    LKB_CUDA(cudaMemcpyAsync(hs, (char*)c->Hd.get() + (size_t)ldd * (kstart - 1) * es, (size_t)ldd * ncol * es, cudaMemcpyDeviceToHost, c->stream));
    LKB_CUDA(cudaMemcpyAsync(hs + (size_t)ldd * ncol * es, c->flags, F_COUNT * sizeof(int), cudaMemcpyDeviceToHost, c->stream));
    return 0;
}
int lanczos_collect(lkb_op_s* A, lkb_basis_s* X, void* T, int ldt, int32_t* info, int kstart, int kend, const void* host) {
    const int kind = X->kind;
    const int ldtd = X->ncols;
    const char* hs = (const char*)host;
    int hf[F_COUNT];
    LKB_TRY(staged_flags(X, kend - kstart + 1, host, hf, "lanczos: NaN norm"));
    const int kdone = hf[F_STOP] ? hf[F_INFO] : kend;
    for (int k = kstart; k <= kdone; ++k)
        for (int i = (k - 1 > 1 ? k - 1 : 1); i <= k + 1; ++i)
            host_store(kind, T, (int64_t)(i - 1) + (int64_t)ldt * (k - 1), hs, (int64_t)(i - 1) + (int64_t)ldtd * (k - kstart));
    A->n_matvec += kdone - kstart + 1;
    *info = hf[F_STOP] ? hf[F_INFO] : 0;
    return 0;
}
}  // namespace lkb

extern "C" {

// ------------------------------------------------------------------------------------------
// bidiagonalization : src/Krylov/golub_kahan.fypp:7-64.   A is m x n; U has m rows, V has n rows.
// Stage tags on the device: 2k-1 = alpha stage of step k, 2k = beta stage.
// ------------------------------------------------------------------------------------------
int lkb_bidiag(lkb_op_t A, lkb_basis_t U, lkb_basis_t V, void* B, int ldb, int32_t* info, int32_t kstart, int32_t kend, double tol) {
    if (!A || !U || !V || !B || !info) { set_error("bidiag: null argument"); return LKB_ERR_ARG; }
    const int kdim = U->ncols - 1;
    if (kstart <= 0) kstart = 1;
    if (kend <= 0) kend = kdim;
    if (kstart > kend || kend > kdim || V->ncols < kend || ldb < kend + 1 || A->kind != U->kind || A->kind != V->kind ||
        A->m != U->n || A->n != V->n) { set_error("bidiag: inconsistent sizes"); return LKB_ERR_ARG; }
    if (tol < 0) tol = atol_of(U->kind);
    *info = 0;
    return krylov_sync(U, kstart, kend, [&] { return bidiag_enqueue(A, U, V, kstart, kend, tol); },
                       [&](const void* hs) { return bidiag_collect(A, U, B, ldb, info, kstart, kend, hs); });
}

}  // extern "C"

namespace lkb {
int bidiag_enqueue(lkb_op_s* A, lkb_basis_s* U, lkb_basis_s* V, int kstart, int kend, double tol) {
    lkb_ctx_s* c = U->ctx;
    const int kind = U->kind;
    const size_t es = kind_size(kind);
    return krylov_run("bid", A, U, V, kstart, kend, tol, false, [&]() -> int {
        for (int k = kstart; k <= kend; ++k) {
            char* bcol = (char*)c->Hd.get() + (size_t)U->ncols * (k - 1) * es;
            void* vk = col_ptr(V, k - 1);
            LKB_TRY(op_apply_enqueue(A, col_ptr(U, k - 1), vk, true, c->flags));
            LKB_TRY(step_tail_enqueue(c, kind, V->d, V->ld, k - 1, vk, V->n, 2, tol, 2 * k - 1, bcol, nullptr));
            void* uk1 = col_ptr(U, k);
            LKB_TRY(op_apply_enqueue(A, vk, uk1, false, c->flags));
            LKB_TRY(step_tail_enqueue(c, kind, U->d, U->ld, k, uk1, U->n, 2, tol, 2 * k, bcol, nullptr));
        }
        return 0;
    });
}
int bidiag_collect(lkb_op_s* A, lkb_basis_s* U, void* B, int ldb, int32_t* info, int kstart, int kend, const void* host) {
    const int kind = U->kind;
    const int ldbd = U->ncols;
    const char* hs = (const char*)host;
    int hf[F_COUNT];
    LKB_TRY(staged_flags(U, kend - kstart + 1, host, hf, "bidiag: NaN norm"));
    const int stage = hf[F_STOP] ? hf[F_INFO] : 2 * kend;
    const int kdone = (stage + 1) / 2;
    for (int k = kstart; k <= kdone; ++k) {
        host_store(kind, B, (int64_t)(k - 1) + (int64_t)ldb * (k - 1), hs, (int64_t)(k - 1) + (int64_t)ldbd * (k - kstart));
        if (2 * k <= stage)
            host_store(kind, B, (int64_t)k + (int64_t)ldb * (k - 1), hs, (int64_t)k + (int64_t)ldbd * (k - kstart));
    }
    A->n_rmatvec += kdone - kstart + 1;
    A->n_matvec += (stage / 2) - kstart + 1;
    *info = hf[F_STOP] ? kdone : 0;
    return 0;
}
}  // namespace lkb
