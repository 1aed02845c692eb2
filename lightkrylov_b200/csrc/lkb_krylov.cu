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

int dgs_enqueue(lkb_ctx_s* c, int kind, const void* V, int64_t ld, int j, void* w, int64_t n, int* flags,
                bool want_norm, bool want_gsinfo, const FinArgs* fin) {
    if (j <= 0) {
        if (want_norm) return norm2_enqueue(c, kind, w, n, flags);
        return 0;
    }
    LKB_TRY(ensure_ws(c, j + 1));
    const size_t nd = (size_t)(j + 1) * (kind_cplx(kind) ? 2 : 1);
    const size_t wsz = kind_cplx(kind) ? 16 : 8;
    // serpentine sweeps: pass-1 dot, fused middle and final update walk the rows in alternating directions, and the
    // first direction alternates with the step index (the previous step's final update ended where this one starts)
    const int d0 = (c->serpentine && fin) ? (fin->kstep & 1) : 0;
    const int d1 = (c->serpentine && fin) ? 1 - d0 : 0;
    // pass 1 coefficients
    prof_begin(c, PC_DOT);
    { SweepDir sd(d0); launch_multidot(kind, c->stream, V, ld, j, w, n, c->partial, c->c1, c->counter, flags, c->sms, c->p2p_arg()); }
    prof_end(c, PC_DOT, 1);
    LKB_TRY(check_launch(c, "multidot"));
    LKB_TRY(allreduce_w(c, c->c1, nd));
    // pass-1 update fused with the pass-2 coefficients (V read once for both) when the shape allows
    bool fused = false;
    if (c->fused) {
        prof_begin(c, PC_FUSED);
        { SweepDir sd(d1); fused = launch_axpy_dot(kind, c->stream, V, ld, j, c->c1, w, n, c->partial, c->c2, c->counter, flags, c->sms, c->p2p_arg()); }
        prof_end(c, PC_FUSED, fused ? 1 : 0);
        if (!fused && c->profile && !c->capturing) { cudaEventDestroy(c->prof_evs.back().a); cudaEventDestroy(c->prof_evs.back().b); c->prof_evs.pop_back(); }
        LKB_TRY(check_launch(c, "axpy_dot"));
    }
    if (!fused) {
        prof_begin(c, PC_AXPY);
        launch_multiaxpy(kind, c->stream, V, ld, j, c->c1, w, n, false, c->partial, c->nrm2, c->counter, flags, c->sms, c->p2p_arg());
        prof_end(c, PC_AXPY, 1);
        prof_begin(c, PC_DOT);
        launch_multidot(kind, c->stream, V, ld, j, w, n, c->partial, c->c2, c->counter, flags, c->sms, c->p2p_arg());
        prof_end(c, PC_DOT, 1);
        LKB_TRY(check_launch(c, "multidot"));
    }
    LKB_TRY(allreduce_w(c, c->c2, nd));
    if (want_gsinfo) {
        launch_gsinfo(c->stream, (char*)c->c2.get() + (size_t)j * wsz, kind_cplx(kind), atol_of(kind), c->flags);
        c->launches++;
    }
    if (fin) {
        // pass-2 update + predicted-norm normalisation + H/T/B column + (optional) halo push in ONE kernel
        prof_begin(c, PC_AXPY);
        SweepDir sd(d0);
        launch_multiaxpy_fin(kind, c->stream, V, ld, j, fin->with_c1 ? c->c1.get() : nullptr, c->c2, w, n, c->partial, c->nrm2, c->counter,
                             fin->hcol, fin->tol, atol_of(kind), c->inv, flags, fin->kstep, fin->mode, c->sms, c->p2p_arg(), fin->hp);
        prof_end(c, PC_AXPY, 1);
        return check_launch(c, "multiaxpy_fin");
    }
    prof_begin(c, PC_AXPY);
    launch_multiaxpy(kind, c->stream, V, ld, j, c->c2, w, n, want_norm, c->partial, c->nrm2, c->counter, flags, c->sms, c->p2p_arg());
    prof_end(c, PC_AXPY, 1);
    LKB_TRY(check_launch(c, "multiaxpy"));
    if (want_norm) LKB_TRY(allreduce_w(c, c->nrm2, 1));
    return 0;
}

// Orthogonalisation + normalisation + column update of ONE Krylov step (everything after the matvec):
//   CGS2 of w against V(:, 0:j), beta = ||w||, column of H / T / B, breakdown decision, w /= beta.
// mode 0 arnoldi (hcol(0:j) = c1 + c2), 1 lanczos, 2 bidiag (only hcol(j) = beta is written).
// Default: the final pass is k_multiaxpy_fin (3 kernels + 1 empty launch per step, 2 reductions).  Falls back to
// the round-1 sequence (multi-axpy with norm, allreduce, k_update, k_scale_dev) for j = 0, when the reductions
// go through ncclAllReduce (the predicted norm must not be summed over ranks), or with option "fin" = 0.
int step_tail_enqueue(lkb_ctx_s* c, int kind, const void* V, int64_t ld, int j, void* w, int64_t n, int mode, double tol,
                      int kstep, void* hcol, const HaloP2P* hp) {
    const bool fin_ok = c->fin && j > 0 && (c->world == 1 || c->p2p_active);
    if (fin_ok) {
        FinArgs fa; fa.mode = mode; fa.tol = tol; fa.kstep = kstep; fa.hcol = hcol; fa.with_c1 = (mode == 0); fa.hp = hp;
        LKB_TRY(dgs_enqueue(c, kind, V, ld, j, w, n, c->flags, false, false, &fa));
    } else {
        LKB_TRY(dgs_enqueue(c, kind, V, ld, j, w, n, c->flags, true, false));
        prof_begin(c, PC_OTHER);
        launch_update(kind, c->stream, mode == 0 ? c->c1.get() : nullptr, mode == 0 ? c->c2.get() : nullptr, j, c->nrm2, hcol, tol,
                      atol_of(kind), c->inv, c->flags, kstep, mode);
        prof_end(c, PC_OTHER, 1);
    }
    prof_begin(c, PC_OTHER);
    launch_scale_dev(kind, c->stream, w, n, c->inv, c->flags, kstep, c->sms, hp);
    prof_end(c, PC_OTHER, 1);
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

// Read c1 + c2 (first j entries) and, optionally, nrm2 to the host (one sync).
static int fetch_coeffs(lkb_ctx_s* c, int kind, int j, bool two, std::vector<Scalar>& out, double* nrm2, int* flags) {
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

// is_orthonormal (src/Krylov/utilities.fypp:90-98): mnorm(Gram(X) - I, "Fro") > rtol_sp (hard-wired, all kinds) => not orthonormal
static int check_orthonormal(lkb_basis_s* X, int j, bool* ok) {
    lkb_ctx_s* c = X->ctx;
    *ok = true;
    std::vector<Scalar> col;
    double fro2 = 0.0;                                         // squared Frobenius norm of G - I, column by column
    const double lim2 = 1e-3 * 1e-3;                           // rtol_sp = sqrt(atol_sp) = 1e-3
    for (int q = 0; q < j && fro2 <= lim2; ++q) {
        LKB_TRY(ensure_ws(c, j + 1));
        launch_multidot(X->kind, c->stream, X->d, X->ld, j, col_ptr(X, q), X->n, c->partial, c->c1, c->counter, nullptr, c->sms, c->p2p_arg());
        c->launches++;
        LKB_TRY(check_launch(c, "gram"));
        LKB_TRY(allreduce_w(c, c->c1, (size_t)(j + 1) * (kind_cplx(X->kind) ? 2 : 1)));
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
        prof_begin(c, PC_DOT);
        launch_multidot(X->kind, c->stream, X->d, X->ld, j, col_ptr(W, wcol0 + q), X->n, c->partial, c->c1, c->counter, nullptr, c->sms, c->p2p_arg());
        prof_end(c, PC_DOT, 1);
        LKB_TRY(check_launch(c, "innerprod"));
        LKB_TRY(allreduce_w(c, c->c1, (size_t)(j + 1) * (kind_cplx(X->kind) ? 2 : 1)));
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
        prof_begin(c, PC_AXPY);
        launch_multiaxpy(X->kind, c->stream, X->d, X->ld, j, c->coefd, col_ptr(W, wcol0 + q), X->n, false, c->partial, c->nrm2, c->counter, nullptr, c->sms, c->p2p_arg());
        prof_end(c, PC_AXPY, 1);
        LKB_TRY(check_launch(c, "lincomb_sub"));
    }
    return 0;
}

int lkb_basis_lincomb(lkb_basis_t X, int j, const void* coef, lkb_vec_t y) {
    if (!X || !y || !coef || j < 0 || j > X->ncols || X->n != y->n || X->kind != y->kind)
        { set_error("lincomb: bad arguments"); return LKB_ERR_ARG; }
    lkb_ctx_s* c = X->ctx;
    LKB_TRY(upload_coef(c, X->kind, coef, j, -1.0));
    LKB_TRY(lkb_vec_zero(y));
    prof_begin(c, PC_AXPY);
    launch_multiaxpy(X->kind, c->stream, X->d, X->ld, j, c->coefd, y->d, X->n, false, c->partial, c->nrm2, c->counter, nullptr, c->sms, c->p2p_arg());
    prof_end(c, PC_AXPY, 1);
    return check_launch(c, "lincomb");
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
            prof_begin(c, PC_DOT);
            launch_multidot(X->kind, c->stream, X->d, X->ld, j, w, X->n, c->partial, c->c1, c->counter, nullptr, c->sms, c->p2p_arg());
            prof_end(c, PC_DOT, 1);
            LKB_TRY(allreduce_w(c, c->c1, (size_t)(j + 1) * (kind_cplx(X->kind) ? 2 : 1)));
            launch_gsinfo(c->stream, (char*)c->c1.get() + (size_t)j * (kind_cplx(X->kind) ? 16 : 8), 0, atol_of(X->kind), c->flags);
            prof_begin(c, PC_AXPY);
            launch_multiaxpy(X->kind, c->stream, X->d, X->ld, j, c->c1, w, X->n, false, c->partial, c->nrm2, c->counter, nullptr, c->sms, c->p2p_arg());
            prof_end(c, PC_AXPY, 1);
            LKB_TRY(check_launch(c, "orthogonalize"));
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
            launch_fill(kind, c->stream, q, Q->n, Q->row0, LKB_DIST_NORMAL, next_seed(c), c->sms);
            c->launches++;
            LKB_TRY(reset_flags(c));
            LKB_TRY(dgs_enqueue(c, kind, col_ptr(Q, col0), Q->ld, j, q, Q->n, c->flags, true, true));
            LKB_TRY(fetch_coeffs(c, kind, j, true, col, &nrm2, hf));
            if (j > 0) *info = hf[F_GSINFO] ? 1 : 0;
            beta = sqrt(fabs(nrm2));
        } else {
            store_kind(kind, R, (size_t)j + (size_t)ldr * j, beta);
        }
        launch_scal(kind, c->stream, Scalar{1.0 / beta, 0.0}, q, Q->n, c->sms);
        c->launches++;
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
        launch_fill(kind, c->stream, qcol(i), Q->n, Q->row0, LKB_DIST_NORMAL, next_seed(c), c->sms);
        c->launches++;
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
                launch_scal(kind, c->stream, Scalar{1.0 / beta, 0.0}, qcol(i), Q->n, c->sms);
                c->launches++;
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
        launch_scal(kind, c->stream, Scalar{1.0 / beta, 0.0}, qcol(j), Q->n, c->sms);
        c->launches++;
        for (int i = j + 1; i < p; ++i) {                                   // orthogonalise the trailing columns (:93-97)
            Scalar b{0, 0};
            LKB_TRY(vec_dot_sync(c, kind, qcol(j), qcol(i), Q->n, &b));
            b = round_kind(b);
            launch_axpby(kind, c->stream, Scalar{-b.re, -b.im}, qcol(j), Scalar{1.0, 0.0}, qcol(i), Q->n, c->sms);
            c->launches++;
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
    lkb_ctx_s* c = X->ctx;
    const int kind = X->kind;
    const size_t es = kind_size(kind);
    if (tol < 0) tol = atol_of(kind);
    *info = 0;
    if (p > 1) return arnoldi_block(A, X, H, ldh, info, kstart, kend, tol, transpose != 0, p);

    const bool tr = transpose != 0;
    LKB_TRY(ensure_hstage(c, (size_t)(kdim + 1) * (kend - kstart + 1) * es + 4096));
    LKB_TRY(arnoldi_enqueue(A, X, kstart, kend, tol, tr));
    LKB_TRY(arnoldi_fetch_async(X, kstart, kend, c->hstage));
    LKB_CUDA(cudaStreamSynchronize(c->stream));
    return arnoldi_collect(A, X, H, ldh, info, kstart, kend, tr, c->hstage);
}

}  // extern "C"

namespace lkb {
// The three phases of a p = 1 arnoldi call, exposed so that eigs can overlap the host geev of
// step k with the device work of step k+1 (SURVEY 8f rank 3).
int arnoldi_enqueue(lkb_op_s* A, lkb_basis_s* X, int kstart, int kend, double tol, bool tr) {
    lkb_ctx_s* c = X->ctx;
    const int kind = X->kind;
    const size_t es = kind_size(kind);
    const int kdim = X->ncols - 1;
    const int ldhd = kdim + 1;
    LKB_TRY(ensure_Hd(c, (size_t)ldhd * kdim * es));
    LKB_TRY(ensure_ws(c, kend + 1));
    auto body = [&]() -> int {
        LKB_TRY(reset_flags(c));
        PdlScope pdl(c->pdl && !c->profile);      // the kernels of the step loop overlap their heads with the predecessors' tails
        bool pushed = false;       // X(k-1)'s boundary rows already sit in the neighbours' halo buffers
        for (int k = kstart; k <= kend; ++k) {
            void* w = col_ptr(X, k);
            LKB_TRY(op_apply_enqueue(A, col_ptr(X, k - 1), w, tr, c->flags, pushed));
            // the kernel that finishes X(k) also pushes its halo rows for the next step's matvec
            const HaloP2P* hp = (k < kend) ? op_halo_desc(A) : nullptr;
            LKB_TRY(step_tail_enqueue(c, kind, X->d, X->ld, k, w, X->n, 0, tol, k, (char*)c->Hd.get() + (size_t)ldhd * (k - 1) * es, hp));
            pushed = hp != nullptr;
        }
        return 0;
    };
    return run_maybe_graph(c, op_capturable(A), make_key("arn", A, X, nullptr, kstart, kend, tol, tr), body);
}
// D2H of the freshly written Hessenberg columns + flags into `host` (pinned), no sync
int arnoldi_fetch_async(lkb_basis_s* X, int kstart, int kend, void* host) {
    return krylov_fetch_async(X->ctx, X->kind, X->ncols, kstart, kend, host);
}
// after the stream reached the fetch: scatter the columns into the caller's H, set info, refill on breakdown
int arnoldi_collect(lkb_op_s* A, lkb_basis_s* X, void* H, int ldh, int32_t* info, int kstart, int kend, bool tr,
                    const void* host) {
    lkb_ctx_s* c = X->ctx;
    const int kind = X->kind;
    const size_t es = kind_size(kind);
    const int ldhd = X->ncols;
    const int ncol = kend - kstart + 1;
    const char* hs = (const char*)host;
    int hf[F_COUNT];
    memcpy(hf, hs + (size_t)ldhd * ncol * es, sizeof(hf));
    if (hf[F_NAN]) { set_error("|beta| = NaN detected! Abort"); return LKB_ERR_NAN; }
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
            launch_fill(kind, c->stream, w, X->n, X->row0, LKB_DIST_NORMAL, next_seed(c), c->sms);
            c->launches++;
            double nrm = 0;
            LKB_TRY(vec_norm_sync(c, kind, w, X->n, &nrm));
            launch_scal(kind, c->stream, Scalar{1.0 / nrm, 0.0}, w, X->n, c->sms);
            c->launches++;
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
    lkb_ctx_s* c = X->ctx;
    if (tol < 0) tol = atol_of(X->kind);
    *info = 0;
    LKB_TRY(ensure_hstage(c, (size_t)(kdim + 1) * (kend - kstart + 1) * kind_size(X->kind) + 4096));
    LKB_TRY(lanczos_enqueue(A, X, kstart, kend, tol));
    LKB_TRY(krylov_fetch_async(X->ctx, X->kind, kdim + 1, kstart, kend, c->hstage));
    LKB_CUDA(cudaStreamSynchronize(c->stream));
    return lanczos_collect(A, X, T, ldt, info, kstart, kend, c->hstage);
}

}  // extern "C"

namespace lkb {
// The three phases of lanczos / bidiagonalization (as for arnoldi): eighs and svds overlap the host syev / gesdd of
// step k with the device work of a speculative step k+1 (SURVEY 8f rank 3).
int lanczos_enqueue(lkb_op_s* A, lkb_basis_s* X, int kstart, int kend, double tol) {
    lkb_ctx_s* c = X->ctx;
    const int kind = X->kind;
    const size_t es = kind_size(kind);
    const int kdim = X->ncols - 1;
    const int ldtd = kdim + 1;
    LKB_TRY(ensure_Hd(c, (size_t)ldtd * kdim * es));
    LKB_TRY(ensure_ws(c, kend + 1));
    const size_t ndw = 2 * (size_t)(kind_cplx(kind) ? 2 : 1);
    auto body = [&]() -> int {
        LKB_TRY(reset_flags(c));
        PdlScope pdl(c->pdl && !c->profile);
        bool pushed = false;
        for (int k = kstart; k <= kend; ++k) {
            void* w = col_ptr(X, k);
            char* tcol = (char*)c->Hd.get() + (size_t)ldtd * (k - 1) * es;
            LKB_TRY(op_apply_enqueue(A, col_ptr(X, k - 1), w, false, c->flags, pushed));
            for (int i = (k - 1 > 1 ? k - 1 : 1); i <= k; ++i) {        // update_tridiag_matrix :57-59
                void* xi = col_ptr(X, i - 1);
                prof_begin(c, PC_DOT);
                launch_multidot(kind, c->stream, xi, X->ld, 1, w, X->n, c->partial, c->tmpw, c->counter, c->flags, c->sms, c->p2p_arg());
                prof_end(c, PC_DOT, 1);
                LKB_TRY(allreduce_w(c, c->tmpw, ndw));
                prof_begin(c, PC_OTHER);
                launch_narrow(kind, c->stream, c->tmpw, tcol + (size_t)(i - 1) * es, 1, c->flags);
                launch_axpy_dev(kind, c->stream, c->tmpw, -1.0, xi, w, X->n, c->flags, c->sms);
                prof_end(c, PC_OTHER, 2);
            }
            const HaloP2P* hp = (k < kend) ? op_halo_desc(A) : nullptr;
            LKB_TRY(step_tail_enqueue(c, kind, X->d, X->ld, k, w, X->n, 1, tol, k, tcol, hp));
            pushed = hp != nullptr;
        }
        return 0;
    };
    return run_maybe_graph(c, op_capturable(A), make_key("lan", A, X, nullptr, kstart, kend, tol, 0), body);
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
    const size_t es = kind_size(kind);
    const int ldtd = X->ncols;
    const int ncol = kend - kstart + 1;
    const char* hs = (const char*)host;
    int hf[F_COUNT];
    memcpy(hf, hs + (size_t)ldtd * ncol * es, sizeof(hf));
    if (hf[F_NAN]) { set_error("lanczos: NaN norm"); return LKB_ERR_NAN; }
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
    lkb_ctx_s* c = U->ctx;
    if (tol < 0) tol = atol_of(U->kind);
    *info = 0;
    LKB_TRY(ensure_hstage(c, (size_t)(kdim + 1) * (kend - kstart + 1) * kind_size(U->kind) + 4096));
    LKB_TRY(bidiag_enqueue(A, U, V, kstart, kend, tol));
    LKB_TRY(krylov_fetch_async(c, U->kind, kdim + 1, kstart, kend, c->hstage));
    LKB_CUDA(cudaStreamSynchronize(c->stream));
    return bidiag_collect(A, U, B, ldb, info, kstart, kend, c->hstage);
}

}  // extern "C"

namespace lkb {
int bidiag_enqueue(lkb_op_s* A, lkb_basis_s* U, lkb_basis_s* V, int kstart, int kend, double tol) {
    lkb_ctx_s* c = U->ctx;
    const int kind = U->kind;
    const size_t es = kind_size(kind);
    const int kdim = U->ncols - 1;
    const int ldbd = kdim + 1;
    LKB_TRY(ensure_Hd(c, (size_t)ldbd * kdim * es));
    LKB_TRY(ensure_ws(c, kend + 1));
    auto body = [&]() -> int {
        LKB_TRY(reset_flags(c));
        PdlScope pdl(c->pdl && !c->profile);
        for (int k = kstart; k <= kend; ++k) {
            char* bcol = (char*)c->Hd.get() + (size_t)ldbd * (k - 1) * es;
            void* vk = col_ptr(V, k - 1);
            LKB_TRY(op_apply_enqueue(A, col_ptr(U, k - 1), vk, true, c->flags));
            LKB_TRY(step_tail_enqueue(c, kind, V->d, V->ld, k - 1, vk, V->n, 2, tol, 2 * k - 1, bcol, nullptr));
            void* uk1 = col_ptr(U, k);
            LKB_TRY(op_apply_enqueue(A, vk, uk1, false, c->flags));
            LKB_TRY(step_tail_enqueue(c, kind, U->d, U->ld, k, uk1, U->n, 2, tol, 2 * k, bcol, nullptr));
        }
        return 0;
    };
    return run_maybe_graph(c, op_capturable(A), make_key("bid", A, U, V, kstart, kend, tol, 0), body);
}
int bidiag_collect(lkb_op_s* A, lkb_basis_s* U, void* B, int ldb, int32_t* info, int kstart, int kend, const void* host) {
    const int kind = U->kind;
    const size_t es = kind_size(kind);
    const int ldbd = U->ncols;
    const int ncol = kend - kstart + 1;
    const char* hs = (const char*)host;
    int hf[F_COUNT];
    memcpy(hf, hs + (size_t)ldbd * ncol * es, sizeof(hf));
    if (hf[F_NAN]) { set_error("bidiag: NaN norm"); return LKB_ERR_NAN; }
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
