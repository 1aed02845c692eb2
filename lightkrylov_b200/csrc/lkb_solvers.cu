// lkb_solvers.cu -- host shells of the iterative solvers around the device Krylov step.
//
//   gmres : src/IterativeSolvers/GMRES/gmres.fypp:65-255 (+ Givens, submodule_utility_functions.fypp:169-204)
//   cg    : src/IterativeSolvers/CG/CG.fypp:61-196
// The k x k / k-vector algebra (Givens rotations, back substitution) stays on the host exactly as
// in the reference; every O(n) operation is a device kernel.
#include <math.h>
#include <string.h>
#include <complex>
#include <vector>
#include "../../include/lkb.h"
#include "lkb_internal.h"

using namespace lkb;

namespace {

// LAPACK 3.10 la_lartg (real): c = |f|/d, r = sign(d, f), s = g/r
void lartg(double f, double g, double& c, double& s, double& r) {
    if (g == 0.0) { c = 1.0; s = 0.0; r = f; return; }
    if (f == 0.0) { c = 0.0; s = g > 0 ? 1.0 : -1.0; r = fabs(g); return; }
    const double d = hypot(f, g);
    c = fabs(f) / d; r = copysign(d, f); s = g / r;
}
// apply_givens_rotation (h has k+1 entries; c, s have k)
void givens_real(cd* h, cd* c, cd* s, int k) {
    for (int j = 0; j < k - 1; ++j) {                       // lasr('L','V','F')
        const double t = h[j + 1].real();
        h[j + 1] = c[j].real() * t - s[j].real() * h[j].real();
        h[j] = s[j].real() * t + c[j].real() * h[j].real();
    }
    double cc, ss, r;
    lartg(h[k - 1].real(), h[k].real(), cc, ss, r);
    c[k - 1] = cc; s[k - 1] = ss; h[k - 1] = r; h[k] = 0.0;
}
void givens_cplx(cd* h, cd* c, cd* s, int k) {             // hand-rolled unnormalised-conjugate form
    for (int i = 0; i < k - 1; ++i) {
        const cd t = c[i] * h[i] + s[i] * h[i + 1];
        h[i + 1] = -s[i] * h[i] + c[i] * h[i + 1];
        h[i] = t;
    }
    const double nrm = sqrt(std::norm(h[k - 1]) + std::norm(h[k]));
    c[k - 1] = h[k - 1] / nrm; s[k - 1] = h[k] / nrm;
    h[k - 1] = c[k - 1] * h[k - 1] + s[k - 1] * h[k];
    h[k] = 0.0;
}
// element helpers (round through the kind's precision, as the reference stores H / e / c / s in `kind`)
cd round_kind(int kind, cd v) {
    if (kind == KS || kind == KC) return cd((double)(float)v.real(), (double)(float)v.imag());
    return v;
}
void push_res(double* res, int32_t cap, int32_t* len, double v) {
    if (res && *len < cap) res[*len] = v;
    (*len)++;
}
// Waits for the stream when it leaves scope, before the owners declared ahead of it release what the device loop still uses
struct StreamSync {
    cudaStream_t s;
    ~StreamSync() { cudaStreamSynchronize(s); }
};

}  // namespace

extern "C" {

// flexible = fgmres (GMRES/fgmres.fypp:65-260): the preconditioned vectors Z(k) are stored and the update is
// dx = Z(:k) y, so the preconditioner may change from one inner step to the next.
// M: the right preconditioner as an operator (gmres only): it is enqueued inside the device cycle like A.
static int gmres_impl(lkb_op_t A, lkb_vec_t b, lkb_vec_t x, int32_t* info, double rtol, double atol, int32_t transpose,
                      lkb_gmres_io* io, lkb_precond_fn precond, void* puser, bool flexible = false, lkb_op_t M = nullptr) {
    if (!A || !b || !x || !info) { set_error("gmres: null argument"); return LKB_ERR_ARG; }
    if (b->n != x->n || b->kind != A->kind || x->kind != A->kind || A->m != b->n || A->n != b->n)
        { set_error("gmres: size/kind mismatch"); return LKB_ERR_ARG; }
    if (M && (M->kind != A->kind || M->m != b->n || M->n != b->n)) { set_error("gmres: preconditioner size/kind mismatch"); return LKB_ERR_ARG; }
    lkb_ctx_s* c = b->ctx;
    const int kind = b->kind;
    const bool cplx = kind_cplx(kind);
    const bool trans = transpose != 0;
    lkb_gmres_io local; memset(&local, 0, sizeof(local));
    if (!io) io = &local;
    const int kdim = io->kdim > 0 ? io->kdim : 30;
    const int maxiter = io->maxiter > 0 ? io->maxiter : 10;
    if (rtol < 0) rtol = rtol_of(kind);
    if (atol < 0) atol = atol_of(kind);
    io->n_iter = io->n_inner = io->n_outer = io->converged = 0; io->res_len = 0;

    double bnorm = 0;
    LKB_TRY(vec_norm_sync(c, kind, b->d, b->n, &bnorm));
    const double tol = atol + rtol * bnorm;

    BasisOwner V, Z;
    VecOwner dx, wrk;
    LKB_TRY(lkb_basis_create(c, kind, b->n, b->n_global, b->row0, kdim + 1, V.out()));
    LKB_TRY(lkb_vec_create(c, kind, b->n, b->n_global, b->row0, dx.out()));
    if ((precond || M) && !flexible) LKB_TRY(lkb_vec_create(c, kind, b->n, b->n_global, b->row0, wrk.out()));
    if (flexible) LKB_TRY(lkb_basis_create(c, kind, b->n, b->n_global, b->row0, kdim, Z.out()));
    std::vector<cd> H((size_t)(kdim + 1) * kdim), e(kdim + 1), cs(kdim), sn(kdim), y(kdim);
    const Scalar one{1, 0}, mone{-1, 0};
    int hf[F_COUNT];
    auto apply_precond = [&](void* v, int iter, double cur, double target) -> int {
        int r = precond(puser, v, b->n, iter, cur, target, (void*)c->stream);
        if (r != 0) { set_error("preconditioner callback returned %d", r); return LKB_ERR_ARG; }
        return 0;
    };

    auto residual_into_v1 = [&](bool skip_if_zero) -> int {
        // V(1) = b - A x   (gmres.fypp:134-143, 205-214)
        double xn = 1.0;
        if (skip_if_zero) LKB_TRY(vec_norm_sync(c, kind, x->d, x->n, &xn));
        if (xn != 0.0) {
            if (trans) A->n_rmatvec++; else A->n_matvec++;
            LKB_TRY(op_apply_enqueue(A, x->d, col_ptr(V, 0), trans, nullptr));
        }
        launch_axpby(kind, c->stream, one, b->d, mone, col_ptr(V, 0), b->n, c->sms);   // sub(b); chsgn()
        c->launches++;
        return check_launch(c, "gmres residual");
    };

    // Without a preconditioner callback the whole inner cycle runs on the device (graph-captured once per call)
    const bool device_cycle = !precond && !flexible;
    // released in reverse order: the stream is synchronised, then the graph and these buffers go, then the work space above
    DevBuf gH(c), ge(c), gres(c);
    GraphExec cycle;
    StreamSync sync{c->stream};
    auto enqueue_cycle = [&]() -> int {
        char* gcs = (char*)ge.p + (size_t)(kdim + 1) * 16; char* gsn = gcs + (size_t)kdim * 16;
        const bool fin_ok = c->fin && (c->world == 1 || c->p2p_active);
        PdlScope pdl(c->pdl && !c->profile);
        bool pushed = false;
        for (int kk = 1; kk <= kdim; ++kk) {
            void* w = col_ptr(V, kk);
            const void* src = col_ptr(V, kk - 1);
            if (M) { LKB_TRY(op_apply_enqueue(M, src, wrk->d, false, c->flags)); src = wrk->d; }   // wrk = M V(k)  (gmres.fypp:155)
            LKB_TRY(op_apply_enqueue(A, src, w, trans, c->flags, pushed));
            // the fused halo push of V(k+1) is right only when V(k+1) is A's next input; with M in between that input is
            // wrk, and op_apply_enqueue(A, wrk, ...) exchanges its halo itself
            const HaloP2P* hp = (kk < kdim && !M) ? op_halo_desc(A) : nullptr;
            if (fin_ok) {     // final pass normalises with the predicted norm (mode 4: k_gmres_update does the column)
                FinArgs fa; fa.mode = 4; fa.tol = tol; fa.kstep = kk; fa.hcol = nullptr; fa.with_c1 = false; fa.hp = hp;
                LKB_TRY(dgs_enqueue(c, kind, V->d, V->ld, kk, w, b->n, c->flags, false, false, &fa));
            } else {
                LKB_TRY(dgs_enqueue(c, kind, V->d, V->ld, kk, w, b->n, c->flags, true, false));
            }
            pushed = fin_ok && hp != nullptr;
            prof_begin(c, PC_OTHER);
            launch_gmres_update(kind, c->stream, c->c1, c->c2, kk, c->nrm2, gH.p, kdim + 1, ge.p, gcs, gsn, tol, c->inv, c->flags, (double*)gres.p);
            launch_scale_dev(kind, c->stream, w, b->n, c->inv, c->flags, kk, c->sms, fin_ok ? hp : nullptr);
            prof_end(c, PC_OTHER, 2);
            LKB_TRY(check_launch(c, "gmres update"));
        }
        return 0;
    };
    if (device_cycle) {
        LKB_TRY(gH.alloc((size_t)(kdim + 1) * kdim * 16));
        LKB_TRY(ge.alloc((size_t)(3 * kdim + 2) * 16));
        LKB_TRY(gres.alloc((size_t)(kdim + 2) * 8));
        LKB_TRY(ensure_ws(c, kdim + 1));
        if (c->graphs && !c->profile && op_capturable(A) && (!M || op_capturable(M)))
            LKB_TRY(capture_graph(c, "gmres: ", enqueue_cycle, &cycle));
    }
    while (!io->converged && io->n_outer <= maxiter) {
        std::fill(H.begin(), H.end(), cd(0));
        LKB_TRY(lkb_basis_zero(V, 0, kdim + 1));
        LKB_TRY(residual_into_v1(true));
        std::fill(e.begin(), e.end(), cd(0));
        double beta = 0;
        LKB_TRY(vec_norm_sync(c, kind, col_ptr(V, 0), b->n, &beta));
        e[0] = round_kind(kind, beta);
        launch_scal(kind, c->stream, Scalar{1.0 / beta, 0}, col_ptr(V, 0), b->n, c->sms); c->launches++;
        std::fill(cs.begin(), cs.end(), cd(0)); std::fill(sn.begin(), sn.end(), cd(0));
        if (io->n_outer == 0) push_res(io->res, io->res_cap, &io->res_len, fabs(beta));
        int k = 1;
        if (device_cycle) {
            // ---- whole restart cycle on the device: one CUDA graph, one host sync (k_gmres_update) ----
            const size_t hbytes = (size_t)(kdim + 1) * kdim * 16;
            LKB_CUDA(cudaMemsetAsync(gH.p, 0, hbytes, c->stream));
            LKB_CUDA(cudaMemsetAsync(ge.p, 0, (size_t)(3 * kdim + 2) * 16, c->stream));   // e, cs, sn
            const double e0[2] = {e[0].real(), 0.0};
            LKB_CUDA(cudaMemcpyAsync(ge.p, e0, 16, cudaMemcpyHostToDevice, c->stream));
            LKB_CUDA(cudaMemsetAsync(c->flags, 0, F_COUNT * sizeof(int), c->stream));
            if (cycle.exec) { LKB_CUDA(cudaGraphLaunch(cycle.exec, c->stream)); c->launches += cycle.launches; }
            else LKB_TRY(enqueue_cycle());
            LKB_TRY(ensure_hstage(c, hbytes + (size_t)(kdim + 2) * 24 + 64 + 4096));
            char* hs = (char*)c->hstage;
            cudaMemcpyAsync(hs, gH.p, hbytes, cudaMemcpyDeviceToHost, c->stream);
            cudaMemcpyAsync(hs + hbytes, ge.p, (size_t)(kdim + 1) * 16, cudaMemcpyDeviceToHost, c->stream);
            cudaMemcpyAsync(hs + hbytes + (size_t)(kdim + 1) * 16, gres.p, (size_t)(kdim + 1) * 8, cudaMemcpyDeviceToHost, c->stream);
            char* hflags = hs + hbytes + (size_t)(kdim + 1) * 24;      // (fetch_flags would stage at offset 0 and clobber H)
            cudaMemcpyAsync(hflags, c->flags, F_COUNT * sizeof(int), cudaMemcpyDeviceToHost, c->stream);
            LKB_CUDA(cudaStreamSynchronize(c->stream));
            memcpy(hf, hflags, sizeof(hf));
            const int kdone = hf[F_STOP] ? hf[F_INFO] : kdim;
            const double* Hh = (const double*)hs; const double* eh = (const double*)(hs + hbytes);
            const double* rh = (const double*)(hs + hbytes + (size_t)(kdim + 1) * 16);
            for (size_t t = 0; t < (size_t)(kdim + 1) * kdim; ++t) H[t] = cd(Hh[2 * t], Hh[2 * t + 1]);
            for (int i = 0; i <= kdim; ++i) e[i] = cd(eh[2 * i], eh[2 * i + 1]);
            for (int i = 1; i <= kdone; ++i) { io->n_iter++; io->n_inner++; push_res(io->res, io->res_cap, &io->res_len, rh[i]); }
            if (trans) A->n_rmatvec += kdone; else A->n_matvec += kdone;
            if (M) M->n_matvec += kdone;
            if (hf[F_STOP]) io->converged = 1;
            k = hf[F_STOP] ? kdone : kdim + 1;
        } else
        for (k = 1; k <= kdim; ++k) {
            void* w = col_ptr(V, k);
            if (trans) A->n_rmatvec++; else A->n_matvec++;
            const void* src = col_ptr(V, k - 1);
            if (flexible) {     // copy(Z(k), V(k)) ; preconditioner%apply(Z(k), k, beta, tol)   (fgmres.fypp:160-161)
                launch_axpby(kind, c->stream, one, col_ptr(V, k - 1), Scalar{0, 0}, col_ptr(Z, k - 1), b->n, c->sms); c->launches++;
                if (precond) LKB_TRY(apply_precond(col_ptr(Z, k - 1), k, beta, tol));
                src = col_ptr(Z, k - 1);
            } else if (precond) {      // wrk = V(k) ; preconditioner%apply(wrk, k, beta, tol)   (gmres.fypp:155)
                launch_axpby(kind, c->stream, one, col_ptr(V, k - 1), Scalar{0, 0}, wrk->d, b->n, c->sms); c->launches++;
                LKB_TRY(apply_precond(wrk->d, k, beta, tol));
                src = wrk->d;
            }
            LKB_TRY(op_apply_enqueue(A, src, w, trans, nullptr));
            LKB_CUDA(cudaMemsetAsync(c->flags, 0, F_COUNT * sizeof(int), c->stream));
            LKB_TRY(dgs_enqueue(c, kind, V->d, V->ld, k, w, b->n, c->flags, true, false));
            // H(:k, k) = c1 + c2 ; H(k+1, k) = ||V(k+1)||
            {
                const size_t wsz = cplx ? 16 : 8;
                LKB_TRY(ensure_hstage(c, 2 * (size_t)(k + 1) * 16 + 4096));
                char* hs = (char*)c->hstage;
                cudaMemcpyAsync(hs, c->c1, (size_t)k * wsz, cudaMemcpyDeviceToHost, c->stream);
                cudaMemcpyAsync(hs + (size_t)k * wsz, c->c2, (size_t)k * wsz, cudaMemcpyDeviceToHost, c->stream);
                cudaMemcpyAsync(hs + 2 * (size_t)k * wsz, c->nrm2, 16, cudaMemcpyDeviceToHost, c->stream);
                LKB_CUDA(cudaStreamSynchronize(c->stream));
                for (int i = 0; i < k; ++i) {
                    const double* a = (const double*)(hs + (size_t)i * wsz);
                    const double* bb = (const double*)(hs + (size_t)(k + i) * wsz);
                    H[i + (size_t)(kdim + 1) * (k - 1)] = round_kind(kind, cd(a[0] + bb[0], cplx ? a[1] + bb[1] : 0.0));
                }
                const double hk = sqrt(fabs(*(const double*)(hs + 2 * (size_t)k * wsz)));
                H[k + (size_t)(kdim + 1) * (k - 1)] = round_kind(kind, hk);
                if (hk > tol) { launch_scal(kind, c->stream, Scalar{1.0 / hk, 0}, w, b->n, c->sms); c->launches++; }
            }
            cd* hcol = &H[(size_t)(kdim + 1) * (k - 1)];
            if (cplx) givens_cplx(hcol, cs.data(), sn.data(), k); else givens_real(hcol, cs.data(), sn.data(), k);
            for (int i = 0; i <= k; ++i) hcol[i] = round_kind(kind, hcol[i]);
            e[k] = round_kind(kind, -sn[k - 1] * e[k - 1]);
            e[k - 1] = round_kind(kind, cs[k - 1] * e[k - 1]);
            beta = std::abs(e[k]);
            io->n_iter++; io->n_inner++;
            push_res(io->res, io->res_cap, &io->res_len, fabs(beta));
            if (fabs(beta) < tol) { io->converged = 1; break; }
        }
        k = k < kdim ? k : kdim;
        // trtrs('u','n','n'): back substitution on H(:k,:k) y = e(:k)
        for (int i = k - 1; i >= 0; --i) {
            cd s = e[i];
            for (int j = i + 1; j < k; ++j) s -= H[i + (size_t)(kdim + 1) * j] * y[j];
            y[i] = s / H[i + (size_t)(kdim + 1) * i];
        }
        {   // dx = V(:k) y ; x += dx
            std::vector<char> yk((size_t)k * kind_size(kind));
            for (int i = 0; i < k; ++i) store_kind(kind, yk.data(), i, y[i]);
            LKB_TRY(lkb_basis_lincomb(flexible ? Z : V, k, yk.data(), dx));         // fgmres: dx = Z(:k) y (fgmres.fypp:207)
            if (precond && !flexible) LKB_TRY(apply_precond(dx->d, -1, -1.0, -1.0)); // preconditioner%apply(dx)  (gmres.fypp:202)
            const void* upd = dx->d;
            if (M) { M->n_matvec++; LKB_TRY(op_apply_enqueue(M, dx->d, wrk->d, false, nullptr)); upd = wrk->d; }   // dx <- M dx
            launch_axpby(kind, c->stream, one, upd, one, x->d, x->n, c->sms); c->launches++;
        }
        LKB_TRY(residual_into_v1(false));
        LKB_TRY(vec_norm_sync(c, kind, col_ptr(V, 0), b->n, &beta));
        if (fabs(beta) > 0.0) { launch_scal(kind, c->stream, Scalar{1.0 / beta, 0}, col_ptr(V, 0), b->n, c->sms); c->launches++; }
        io->n_iter++; io->n_outer++;
        push_res(io->res, io->res_cap, &io->res_len, fabs(beta));
        if (fabs(beta) < tol) { io->converged = 1; break; }
    }
    *info = io->converged ? io->n_iter : -io->n_iter;
    io->info = *info;
    return 0;
}

int lkb_gmres(lkb_op_t A, lkb_vec_t b, lkb_vec_t x, int32_t* info, double rtol, double atol, int32_t transpose,
              lkb_gmres_io* io) {
    return gmres_impl(A, b, x, info, rtol, atol, transpose, io, nullptr, nullptr);
}
int lkb_gmres_precond(lkb_op_t A, lkb_vec_t b, lkb_vec_t x, int32_t* info, double rtol, double atol, int32_t transpose,
                      lkb_gmres_io* io, lkb_precond_fn precond, void* user) {
    return gmres_impl(A, b, x, info, rtol, atol, transpose, io, precond, user);
}
int lkb_fgmres(lkb_op_t A, lkb_vec_t b, lkb_vec_t x, int32_t* info, double rtol, double atol, int32_t transpose,
               lkb_gmres_io* io, lkb_precond_fn precond, void* user) {
    return gmres_impl(A, b, x, info, rtol, atol, transpose, io, precond, user, true);
}
int lkb_gmres_precond_op(lkb_op_t A, lkb_vec_t b, lkb_vec_t x, int32_t* info, double rtol, double atol, int32_t transpose,
                         lkb_gmres_io* io, lkb_op_t M) {
    if (!M) { set_error("gmres_precond_op: null preconditioner"); return LKB_ERR_ARG; }
    return gmres_impl(A, b, x, info, rtol, atol, transpose, io, nullptr, nullptr, false, M);
}

// The preconditioner is a host callback (precond: host-driven loop below) or an operator M (device-resident loop).
static int cg_impl(lkb_op_t A, lkb_vec_t b, lkb_vec_t x, int32_t* info, double rtol, double atol, lkb_cg_io* io,
                   lkb_precond_fn precond, void* puser, lkb_op_t M = nullptr) {
    if (!A || !b || !x || !info) { set_error("cg: null argument"); return LKB_ERR_ARG; }
    if (b->n != x->n || b->kind != A->kind || x->kind != A->kind || A->m != b->n || A->n != b->n)
        { set_error("cg: size/kind mismatch"); return LKB_ERR_ARG; }
    if (M && (M->kind != A->kind || M->m != b->n || M->n != b->n)) { set_error("cg: preconditioner size/kind mismatch"); return LKB_ERR_ARG; }
    // a diagonal M is fused into k_cg_update / k_cg_direction; any other M is applied to r and reduced by a multi-dot
    const int mode = !M ? CG_PLAIN : (M->type == OP_DIAG ? CG_DIAG : CG_NORED);
    lkb_ctx_s* c = b->ctx;
    const int kind = b->kind;
    lkb_cg_io local; memset(&local, 0, sizeof(local));
    if (!io) io = &local;
    const int maxiter = io->maxiter > 0 ? io->maxiter : 100;
    if (rtol < 0) rtol = rtol_of(kind);
    if (atol < 0) atol = atol_of(kind);
    io->n_iter = 0; io->converged = 0; io->res_len = 0;
    double bnorm = 0;
    LKB_TRY(vec_norm_sync(c, kind, b->d, b->n, &bnorm));
    const double tol = atol + rtol * bnorm;
    VecOwner r, p, Ap, z;
    LKB_TRY(lkb_vec_create(c, kind, b->n, b->n_global, b->row0, r.out()));
    LKB_TRY(lkb_vec_create(c, kind, b->n, b->n_global, b->row0, p.out()));
    LKB_TRY(lkb_vec_create(c, kind, b->n, b->n_global, b->row0, Ap.out()));
    if (precond || mode == CG_NORED) LKB_TRY(lkb_vec_create(c, kind, b->n, b->n_global, b->row0, z.out()));
    // z = r ; preconditioner%apply(z)   (CG.fypp:113-114, 137)
    auto make_z = [&]() -> int {
        launch_axpby(kind, c->stream, Scalar{1, 0}, r->d, Scalar{0, 0}, z->d, b->n, c->sms); c->launches++;
        int pr = precond(puser, z->d, b->n, -1, -1.0, -1.0, (void*)c->stream);
        if (pr != 0) { set_error("preconditioner callback returned %d", pr); return LKB_ERR_ARG; }
        return 0;
    };
    const Scalar one{1, 0}, mone{-1, 0}, zero{0, 0};
    double xn = 0;
    LKB_TRY(vec_norm_sync(c, kind, x->d, x->n, &xn));
    if (xn > 0) { A->n_matvec++; LKB_TRY(op_apply_enqueue(A, x->d, r->d, false, nullptr)); }
    launch_axpby(kind, c->stream, one, b->d, mone, r->d, b->n, c->sms); c->launches++;      // r = b - A x
    Scalar rr_old;
    if (precond) {
        LKB_TRY(make_z());
        launch_axpby(kind, c->stream, one, z->d, zero, p->d, b->n, c->sms); c->launches++;  // p = z
        LKB_TRY(vec_dot_sync(c, kind, r->d, z->d, b->n, &rr_old));
    } else if (M) {
        // z = M r ; p = z ; rz = r^H z   (a diagonal M writes z straight into p: the loop never stores z)
        M->n_matvec++;
        void* z0 = mode == CG_DIAG ? p->d : z->d;
        LKB_TRY(op_apply_enqueue(M, r->d, z0, false, nullptr));
        if (mode == CG_NORED) { launch_axpby(kind, c->stream, one, z->d, zero, p->d, b->n, c->sms); c->launches++; }
        LKB_TRY(vec_dot_sync(c, kind, r->d, z0, b->n, &rr_old));
    } else {
        launch_axpby(kind, c->stream, one, r->d, zero, p->d, b->n, c->sms); c->launches++;  // p = r
        LKB_TRY(vec_dot_sync(c, kind, r->d, r->d, b->n, &rr_old));
    }
    push_res(io->res, io->res_cap, &io->res_len, sqrt(hypot(rr_old.re, rr_old.im)));
    if (!precond) {
        // ---- device-resident iteration: alpha, beta and the convergence test stay on the GPU; chunks of
        // CH iterations run as one CUDA graph, the host reads the flags between chunks (kernels_vec.cu) ----
        const int CH = 16;
        const size_t wsz = kind_cplx(kind) ? 16 : 8;
        DevBuf scal(c), res_hist(c);
        GraphExec chunk;
        StreamSync sync{c->stream};
        LKB_TRY(scal.alloc(64));
        LKB_TRY(res_hist.alloc((size_t)(maxiter + 2) * sizeof(double)));
        LKB_TRY(ensure_ws(c, 2));
        cudaMemsetAsync(scal.p, 0, 64, c->stream);
        cudaMemcpyAsync(scal.p, c->tmpw, wsz, cudaMemcpyDeviceToDevice, c->stream);     // r_dot_r_old (just reduced)
        cudaMemsetAsync(c->flags, 0, F_COUNT * sizeof(int), c->stream);
        const size_t ndw = 2 * (size_t)(kind_cplx(kind) ? 2 : 1);
        auto one_iteration = [&]() -> int {
            LKB_TRY(op_apply_enqueue(A, p->d, Ap->d, false, c->flags));
            prof_begin(c, PC_DOT);
            launch_multidot(kind, c->stream, p->d, b->n, 1, Ap->d, b->n, c->partial, c->tmpw, c->counter, c->flags, c->sms, c->p2p_arg());
            prof_end(c, PC_DOT, 1);
            LKB_TRY(allreduce_w(c, c->tmpw, ndw));
            prof_begin(c, PC_OTHER);
            launch_cg_update(kind, c->stream, scal.p, c->tmpw, p->d, Ap->d, x->d, r->d, b->n, c->partial, c->nrm2, c->counter,
                             c->flags, c->sms, c->p2p_arg(), mode, mode == CG_DIAG ? M->diag.get() : nullptr);
            prof_end(c, PC_OTHER, 1);
            const void* rr_new = c->nrm2;
            if (mode == CG_NORED) {         // z = M r ; rz = r^H z (multi-dot, j = 1: c2[0])
                LKB_TRY(op_apply_enqueue(M, r->d, z->d, false, c->flags));
                prof_begin(c, PC_DOT);
                launch_multidot(kind, c->stream, r->d, b->n, 1, z->d, b->n, c->partial, c->c2, c->counter, c->flags, c->sms, c->p2p_arg());
                prof_end(c, PC_DOT, 1);
                LKB_TRY(allreduce_w(c, c->c2, ndw));
                rr_new = c->c2;
            } else {
                LKB_TRY(allreduce_w(c, c->nrm2, mode == CG_DIAG && kind_cplx(kind) ? 2 : 1));
            }
            prof_begin(c, PC_OTHER);
            launch_cg_check(kind, c->stream, scal.p, rr_new, tol, maxiter, (double*)res_hist.p, c->flags);
            launch_cg_direction(kind, c->stream, scal.p, mode == CG_NORED ? z->d : r->d, p->d, b->n, c->flags, c->sms,
                                mode == CG_DIAG ? M->diag.get() : nullptr);
            prof_end(c, PC_OTHER, 2);
            return check_launch(c, "cg iteration");
        };
        auto one_chunk = [&]() -> int {
            for (int q = 0; q < CH; ++q) LKB_TRY(one_iteration());
            return 0;
        };
        if (c->graphs && !c->profile && op_capturable(A) && (!M || op_capturable(M)))
            LKB_TRY(capture_graph(c, "cg: ", one_chunk, &chunk));
        int hf[F_COUNT] = {0};
        while (true) {
            if (chunk.exec) { LKB_CUDA(cudaGraphLaunch(chunk.exec, c->stream)); c->launches += chunk.launches; }
            else LKB_TRY(one_chunk());
            LKB_TRY(fetch_flags(c, hf));
            if (hf[F_STOP]) break;
        }
        io->n_iter = hf[5]; io->converged = hf[6];
        A->n_matvec += io->n_iter;
        if (M) M->n_matvec += io->n_iter;
        std::vector<double> hist((size_t)io->n_iter + 1);
        LKB_CUDA(cudaMemcpy(hist.data(), res_hist.p, hist.size() * sizeof(double), cudaMemcpyDeviceToHost));
        for (int i = 1; i <= io->n_iter; ++i) push_res(io->res, io->res_cap, &io->res_len, hist[i]);
        *info = io->converged ? io->n_iter : -io->n_iter;
        io->info = *info;
        return check_launch(c, "cg");
    }
    for (int it = 1; it <= maxiter; ++it) {
        A->n_matvec++;
        LKB_TRY(op_apply_enqueue(A, p->d, Ap->d, false, nullptr));
        Scalar pAp;
        LKB_TRY(vec_dot_sync(c, kind, p->d, Ap->d, b->n, &pAp));
        const cd alpha = round_kind(kind, cd(rr_old.re, rr_old.im) / cd(pAp.re, pAp.im));
        launch_axpby(kind, c->stream, to_scalar(alpha), p->d, one, x->d, b->n, c->sms);      // x += alpha p
        launch_axpby(kind, c->stream, to_scalar(-alpha), Ap->d, one, r->d, b->n, c->sms);    // r -= alpha Ap
        c->launches += 2;
        Scalar rr_new;
        LKB_TRY(make_z()); LKB_TRY(vec_dot_sync(c, kind, r->d, z->d, b->n, &rr_new));
        const double residual = sqrt(hypot(rr_new.re, rr_new.im));
        io->n_iter++;
        push_res(io->res, io->res_cap, &io->res_len, residual);
        if (residual < tol) { io->converged = 1; break; }
        const cd beta = round_kind(kind, cd(rr_new.re, rr_new.im) / cd(rr_old.re, rr_old.im));
        launch_axpby(kind, c->stream, one, z->d, to_scalar(beta), p->d, b->n, c->sms);       // p = z + beta p
        c->launches++;
        rr_old = rr_new;
    }
    *info = io->converged ? io->n_iter : -io->n_iter;
    io->info = *info;
    return check_launch(c, "cg");
}

int lkb_cg(lkb_op_t A, lkb_vec_t b, lkb_vec_t x, int32_t* info, double rtol, double atol, lkb_cg_io* io) {
    return cg_impl(A, b, x, info, rtol, atol, io, nullptr, nullptr);
}
int lkb_cg_precond(lkb_op_t A, lkb_vec_t b, lkb_vec_t x, int32_t* info, double rtol, double atol, lkb_cg_io* io,
                   lkb_precond_fn precond, void* user) {
    return cg_impl(A, b, x, info, rtol, atol, io, precond, user);
}
int lkb_cg_precond_op(lkb_op_t A, lkb_vec_t b, lkb_vec_t x, int32_t* info, double rtol, double atol, lkb_cg_io* io,
                      lkb_op_t M) {
    if (!M) { set_error("cg_precond_op: null preconditioner"); return LKB_ERR_ARG; }
    return cg_impl(A, b, x, info, rtol, atol, io, nullptr, nullptr, M);
}

}  // extern "C"
