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
typedef std::complex<double> cd;

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
Scalar to_scalar(cd v) { return Scalar{v.real(), v.imag()}; }
void store_kind(int kind, cd v, void* p) {
    switch (kind) {
        case KS: *(float*)p = (float)v.real(); break;
        case KD: *(double*)p = v.real(); break;
        case KC: ((float*)p)[0] = (float)v.real(); ((float*)p)[1] = (float)v.imag(); break;
        default: ((double*)p)[0] = v.real(); ((double*)p)[1] = v.imag(); break;
    }
}
void push_res(double* res, int32_t cap, int32_t* len, double v) {
    if (res && *len < cap) res[*len] = v;
    (*len)++;
}

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

    lkb_basis_t V = nullptr, Z = nullptr;
    lkb_vec_t dx = nullptr, wrk = nullptr;
    {
        int ra = lkb_basis_create(c, kind, b->n, b->n_global, b->row0, kdim + 1, &V);
        if (!ra) ra = lkb_vec_create(c, kind, b->n, b->n_global, b->row0, &dx);
        if (!ra && (precond || M) && !flexible) ra = lkb_vec_create(c, kind, b->n, b->n_global, b->row0, &wrk);
        if (!ra && flexible) ra = lkb_basis_create(c, kind, b->n, b->n_global, b->row0, kdim, &Z);
        if (ra) {      // release whatever was allocated before the failure
            if (V) lkb_basis_destroy(V); if (dx) lkb_vec_destroy(dx); if (wrk) lkb_vec_destroy(wrk); if (Z) lkb_basis_destroy(Z);
            return ra;
        }
    }
    std::vector<cd> H((size_t)(kdim + 1) * kdim), e(kdim + 1), cs(kdim), sn(kdim), y(kdim);
    std::vector<Scalar> col;
    const Scalar one{1, 0}, mone{-1, 0};
    int hf[F_COUNT];
    int rc = 0;
    auto cleanup = [&](int r) { lkb_basis_destroy(V); lkb_vec_destroy(dx); if (wrk) lkb_vec_destroy(wrk); if (Z) lkb_basis_destroy(Z); return r; };
    auto apply_precond = [&](void* v, int iter, double cur, double target) -> int {
        int r = precond(puser, v, b->n, iter, cur, target, (void*)c->stream);
        if (r != 0) { set_error("preconditioner callback returned %d", r); return LKB_ERR_ARG; }
        return 0;
    };
#define GM_TRY(call) do { rc = (call); if (rc) return cleanup(rc); } while (0)

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
    void* gH = nullptr; void* ge = nullptr; double* gres = nullptr;
    cudaGraphExec_t cycle_exec = nullptr; int64_t cycle_launches = 0;
    auto cleanup_dev = [&]() { cudaStreamSynchronize(c->stream); if (cycle_exec) cudaGraphExecDestroy(cycle_exec); dev_free(c, gH); dev_free(c, ge); dev_free(c, gres); };
    auto enqueue_cycle = [&]() -> int {
        char* gcs = (char*)ge + (size_t)(kdim + 1) * 16; char* gsn = gcs + (size_t)kdim * 16;
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
            launch_gmres_update(kind, c->stream, c->c1, c->c2, kk, c->nrm2, gH, kdim + 1, ge, gcs, gsn, tol, c->inv, c->flags, gres);
            launch_scale_dev(kind, c->stream, w, b->n, c->inv, c->flags, kk, c->sms, fin_ok ? hp : nullptr);
            prof_end(c, PC_OTHER, 2);
            LKB_TRY(check_launch(c, "gmres update"));
        }
        return 0;
    };
    if (device_cycle) {
        if (dev_alloc(c, &gH, (size_t)(kdim + 1) * kdim * 16) != 0 || dev_alloc(c, &ge, (size_t)(3 * kdim + 2) * 16) != 0 ||
            dev_alloc(c, (void**)&gres, (size_t)(kdim + 2) * 8) != 0) { cleanup_dev(); return cleanup(LKB_ERR_ALLOC); }
        rc = ensure_ws(c, kdim + 1);
        if (rc) { cleanup_dev(); return cleanup(rc); }
        if (c->graphs && !c->profile && (A->type != 9 || A->capturable) && (!M || M->type != 9 || M->capturable)) {
            const int64_t l0 = c->launches;
            int r2 = cudaStreamBeginCapture(c->stream, cudaStreamCaptureModeThreadLocal) == cudaSuccess ? 0 : LKB_ERR_CUDA;
            if (r2 == 0) {
                c->capturing = true; r2 = enqueue_cycle(); c->capturing = false;
                cudaGraph_t g = nullptr;
                cudaError_t ce = cudaStreamEndCapture(c->stream, &g);
                if (r2 == 0 && ce != cudaSuccess) { set_error("gmres: graph capture failed: %s", cudaGetErrorString(ce)); r2 = LKB_ERR_CUDA; }
                if (r2 == 0 && cudaGraphInstantiate(&cycle_exec, g, 0) != cudaSuccess) { set_error("gmres: graph instantiate failed"); r2 = LKB_ERR_CUDA; }
                if (g) cudaGraphDestroy(g);
            }
            cycle_launches = c->launches - l0; c->launches = l0;
            if (r2) { cleanup_dev(); return cleanup(r2); }
        }
    }
#undef GM_TRY
#define GM_TRY(call) do { rc = (call); if (rc) { cleanup_dev(); return cleanup(rc); } } while (0)
    while (!io->converged && io->n_outer <= maxiter) {
        std::fill(H.begin(), H.end(), cd(0));
        GM_TRY(lkb_basis_zero(V, 0, kdim + 1));
        GM_TRY(residual_into_v1(true));
        std::fill(e.begin(), e.end(), cd(0));
        double beta = 0;
        GM_TRY(vec_norm_sync(c, kind, col_ptr(V, 0), b->n, &beta));
        e[0] = round_kind(kind, beta);
        launch_scal(kind, c->stream, Scalar{1.0 / beta, 0}, col_ptr(V, 0), b->n, c->sms); c->launches++;
        std::fill(cs.begin(), cs.end(), cd(0)); std::fill(sn.begin(), sn.end(), cd(0));
        if (io->n_outer == 0) push_res(io->res, io->res_cap, &io->res_len, fabs(beta));
        int k = 1;
        if (device_cycle) {
            // ---- whole restart cycle on the device: one CUDA graph, one host sync (k_gmres_update) ----
            const size_t hbytes = (size_t)(kdim + 1) * kdim * 16;
            GM_TRY(cudaMemsetAsync(gH, 0, hbytes, c->stream) == cudaSuccess ? 0 : LKB_ERR_CUDA);
            GM_TRY(cudaMemsetAsync(ge, 0, (size_t)(3 * kdim + 2) * 16, c->stream) == cudaSuccess ? 0 : LKB_ERR_CUDA);   // e, cs, sn
            const double e0[2] = {e[0].real(), 0.0};
            GM_TRY(cudaMemcpyAsync(ge, e0, 16, cudaMemcpyHostToDevice, c->stream) == cudaSuccess ? 0 : LKB_ERR_CUDA);
            GM_TRY(cudaMemsetAsync(c->flags, 0, F_COUNT * sizeof(int), c->stream) == cudaSuccess ? 0 : LKB_ERR_CUDA);
            if (cycle_exec) { GM_TRY(cudaGraphLaunch(cycle_exec, c->stream) == cudaSuccess ? 0 : LKB_ERR_CUDA); c->launches += cycle_launches; }
            else GM_TRY(enqueue_cycle());
            GM_TRY(ensure_hstage(c, hbytes + (size_t)(kdim + 2) * 24 + 64 + 4096));
            char* hs = (char*)c->hstage;
            cudaMemcpyAsync(hs, gH, hbytes, cudaMemcpyDeviceToHost, c->stream);
            cudaMemcpyAsync(hs + hbytes, ge, (size_t)(kdim + 1) * 16, cudaMemcpyDeviceToHost, c->stream);
            cudaMemcpyAsync(hs + hbytes + (size_t)(kdim + 1) * 16, gres, (size_t)(kdim + 1) * 8, cudaMemcpyDeviceToHost, c->stream);
            char* hflags = hs + hbytes + (size_t)(kdim + 1) * 24;      // (fetch_flags would stage at offset 0 and clobber H)
            cudaMemcpyAsync(hflags, c->flags, F_COUNT * sizeof(int), cudaMemcpyDeviceToHost, c->stream);
            GM_TRY(cudaStreamSynchronize(c->stream) == cudaSuccess ? 0 : LKB_ERR_CUDA);
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
                if (precond) GM_TRY(apply_precond(col_ptr(Z, k - 1), k, beta, tol));
                src = col_ptr(Z, k - 1);
            } else if (precond) {      // wrk = V(k) ; preconditioner%apply(wrk, k, beta, tol)   (gmres.fypp:155)
                launch_axpby(kind, c->stream, one, col_ptr(V, k - 1), Scalar{0, 0}, wrk->d, b->n, c->sms); c->launches++;
                GM_TRY(apply_precond(wrk->d, k, beta, tol));
                src = wrk->d;
            }
            GM_TRY(op_apply_enqueue(A, src, w, trans, nullptr));
            GM_TRY(cudaMemsetAsync(c->flags, 0, F_COUNT * sizeof(int), c->stream) == cudaSuccess ? 0 : LKB_ERR_CUDA);
            GM_TRY(dgs_enqueue(c, kind, V->d, V->ld, k, w, b->n, c->flags, true, false));
            // H(:k, k) = c1 + c2 ; H(k+1, k) = ||V(k+1)||
            {
                const size_t wsz = cplx ? 16 : 8;
                GM_TRY(ensure_hstage(c, 2 * (size_t)(k + 1) * 16 + 4096));
                char* hs = (char*)c->hstage;
                cudaMemcpyAsync(hs, c->c1, (size_t)k * wsz, cudaMemcpyDeviceToHost, c->stream);
                cudaMemcpyAsync(hs + (size_t)k * wsz, c->c2, (size_t)k * wsz, cudaMemcpyDeviceToHost, c->stream);
                cudaMemcpyAsync(hs + 2 * (size_t)k * wsz, c->nrm2, 16, cudaMemcpyDeviceToHost, c->stream);
                GM_TRY(cudaStreamSynchronize(c->stream) == cudaSuccess ? 0 : LKB_ERR_CUDA);
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
            for (int i = 0; i < k; ++i) store_kind(kind, y[i], &yk[(size_t)i * kind_size(kind)]);
            GM_TRY(lkb_basis_lincomb(flexible ? Z : V, k, yk.data(), dx));         // fgmres: dx = Z(:k) y (fgmres.fypp:207)
            if (precond && !flexible) GM_TRY(apply_precond(dx->d, -1, -1.0, -1.0)); // preconditioner%apply(dx)  (gmres.fypp:202)
            const void* upd = dx->d;
            if (M) { M->n_matvec++; GM_TRY(op_apply_enqueue(M, dx->d, wrk->d, false, nullptr)); upd = wrk->d; }   // dx <- M dx
            launch_axpby(kind, c->stream, one, upd, one, x->d, x->n, c->sms); c->launches++;
        }
        GM_TRY(residual_into_v1(false));
        GM_TRY(vec_norm_sync(c, kind, col_ptr(V, 0), b->n, &beta));
        if (fabs(beta) > 0.0) { launch_scal(kind, c->stream, Scalar{1.0 / beta, 0}, col_ptr(V, 0), b->n, c->sms); c->launches++; }
        io->n_iter++; io->n_outer++;
        push_res(io->res, io->res_cap, &io->res_len, fabs(beta));
        if (fabs(beta) < tol) { io->converged = 1; break; }
    }
#undef GM_TRY
    (void)col;
    cleanup_dev();
    *info = io->converged ? io->n_iter : -io->n_iter;
    io->info = *info;
    return cleanup(0);
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
    const int mode = !M ? CG_PLAIN : (M->type == 4 ? CG_DIAG : CG_NORED);
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
    lkb_vec_t r = nullptr, p = nullptr, Ap = nullptr, z = nullptr;
    {
        int ra = lkb_vec_create(c, kind, b->n, b->n_global, b->row0, &r);
        if (!ra) ra = lkb_vec_create(c, kind, b->n, b->n_global, b->row0, &p);
        if (!ra) ra = lkb_vec_create(c, kind, b->n, b->n_global, b->row0, &Ap);
        if (!ra && (precond || mode == CG_NORED)) ra = lkb_vec_create(c, kind, b->n, b->n_global, b->row0, &z);
        if (ra) {
            if (r) lkb_vec_destroy(r); if (p) lkb_vec_destroy(p); if (Ap) lkb_vec_destroy(Ap); if (z) lkb_vec_destroy(z);
            return ra;
        }
    }
    int rc = 0;
    auto cleanup = [&](int rr) { lkb_vec_destroy(r); lkb_vec_destroy(p); lkb_vec_destroy(Ap); if (z) lkb_vec_destroy(z); return rr; };
    // z = r ; preconditioner%apply(z)   (CG.fypp:113-114, 137)
    auto make_z = [&]() -> int {
        launch_axpby(kind, c->stream, Scalar{1, 0}, r->d, Scalar{0, 0}, z->d, b->n, c->sms); c->launches++;
        int pr = precond(puser, z->d, b->n, -1, -1.0, -1.0, (void*)c->stream);
        if (pr != 0) { set_error("preconditioner callback returned %d", pr); return LKB_ERR_ARG; }
        return 0;
    };
#define CG_TRY(call) do { rc = (call); if (rc) return cleanup(rc); } while (0)
    const Scalar one{1, 0}, mone{-1, 0}, zero{0, 0};
    double xn = 0;
    CG_TRY(vec_norm_sync(c, kind, x->d, x->n, &xn));
    if (xn > 0) { A->n_matvec++; CG_TRY(op_apply_enqueue(A, x->d, r->d, false, nullptr)); }
    launch_axpby(kind, c->stream, one, b->d, mone, r->d, b->n, c->sms); c->launches++;      // r = b - A x
    Scalar rr_old;
    if (precond) {
        CG_TRY(make_z());
        launch_axpby(kind, c->stream, one, z->d, zero, p->d, b->n, c->sms); c->launches++;  // p = z
        CG_TRY(vec_dot_sync(c, kind, r->d, z->d, b->n, &rr_old));
    } else if (M) {
        // z = M r ; p = z ; rz = r^H z   (a diagonal M writes z straight into p: the loop never stores z)
        M->n_matvec++;
        void* z0 = mode == CG_DIAG ? p->d : z->d;
        CG_TRY(op_apply_enqueue(M, r->d, z0, false, nullptr));
        if (mode == CG_NORED) { launch_axpby(kind, c->stream, one, z->d, zero, p->d, b->n, c->sms); c->launches++; }
        CG_TRY(vec_dot_sync(c, kind, r->d, z0, b->n, &rr_old));
    } else {
        launch_axpby(kind, c->stream, one, r->d, zero, p->d, b->n, c->sms); c->launches++;  // p = r
        CG_TRY(vec_dot_sync(c, kind, r->d, r->d, b->n, &rr_old));
    }
    push_res(io->res, io->res_cap, &io->res_len, sqrt(hypot(rr_old.re, rr_old.im)));
    if (!precond) {
        // ---- device-resident iteration: alpha, beta and the convergence test stay on the GPU; chunks of
        // CH iterations run as one CUDA graph, the host reads the flags between chunks (kernels_vec.cu) ----
        const int CH = 16;
        const size_t wsz = kind_cplx(kind) ? 16 : 8;
        void* scal = nullptr; double* res_hist = nullptr;
        auto cleanup2 = [&](int rr) { cudaStreamSynchronize(c->stream); dev_free(c, scal); dev_free(c, res_hist); return cleanup(rr); };
        if (dev_alloc(c, &scal, 64) != 0 || dev_alloc(c, (void**)&res_hist, (size_t)(maxiter + 2) * sizeof(double)) != 0)
            return cleanup2(LKB_ERR_ALLOC);
#undef CG_TRY
#define CG_TRY(call) do { rc = (call); if (rc) return cleanup2(rc); } while (0)
        CG_TRY(ensure_ws(c, 2));
        cudaMemsetAsync(scal, 0, 64, c->stream);
        cudaMemcpyAsync(scal, c->tmpw, wsz, cudaMemcpyDeviceToDevice, c->stream);     // r_dot_r_old (just reduced)
        cudaMemsetAsync(c->flags, 0, F_COUNT * sizeof(int), c->stream);
        const size_t ndw = 2 * (size_t)(kind_cplx(kind) ? 2 : 1);
        auto one_iteration = [&]() -> int {
            LKB_TRY(op_apply_enqueue(A, p->d, Ap->d, false, c->flags));
            prof_begin(c, PC_DOT);
            launch_multidot(kind, c->stream, p->d, b->n, 1, Ap->d, b->n, c->partial, c->tmpw, c->counter, c->flags, c->sms, c->p2p_arg());
            prof_end(c, PC_DOT, 1);
            LKB_TRY(allreduce_w(c, c->tmpw, ndw));
            prof_begin(c, PC_OTHER);
            launch_cg_update(kind, c->stream, scal, c->tmpw, p->d, Ap->d, x->d, r->d, b->n, c->partial, c->nrm2, c->counter,
                             c->flags, c->sms, c->p2p_arg(), mode, mode == CG_DIAG ? M->diag : nullptr);
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
            launch_cg_check(kind, c->stream, scal, rr_new, tol, maxiter, res_hist, c->flags);
            launch_cg_direction(kind, c->stream, scal, mode == CG_NORED ? z->d : r->d, p->d, b->n, c->flags, c->sms,
                                mode == CG_DIAG ? M->diag : nullptr);
            prof_end(c, PC_OTHER, 2);
            return check_launch(c, "cg iteration");
        };
        cudaGraphExec_t exec = nullptr;
        int64_t graph_launches = 0;
        const bool use_graph = c->graphs && !c->profile && (A->type != 9 || A->capturable) && (!M || M->type != 9 || M->capturable);
        if (use_graph) {
            const int64_t l0 = c->launches;
            CG_TRY(cudaStreamBeginCapture(c->stream, cudaStreamCaptureModeThreadLocal) == cudaSuccess ? 0 : LKB_ERR_CUDA);
            c->capturing = true;
            int r2 = 0;
            for (int q = 0; q < CH && r2 == 0; ++q) r2 = one_iteration();
            c->capturing = false;
            cudaGraph_t g = nullptr;
            cudaError_t e = cudaStreamEndCapture(c->stream, &g);
            if (r2 == 0 && e != cudaSuccess) { set_error("cg: graph capture failed: %s", cudaGetErrorString(e)); r2 = LKB_ERR_CUDA; }
            if (r2 == 0 && cudaGraphInstantiate(&exec, g, 0) != cudaSuccess) { set_error("cg: graph instantiate failed"); r2 = LKB_ERR_CUDA; }
            if (g) cudaGraphDestroy(g);
            graph_launches = c->launches - l0; c->launches = l0;
            CG_TRY(r2);
        }
        int hf[F_COUNT] = {0};
        while (true) {
            if (exec) { CG_TRY(cudaGraphLaunch(exec, c->stream) == cudaSuccess ? 0 : LKB_ERR_CUDA); c->launches += graph_launches; }
            else for (int q = 0; q < CH; ++q) CG_TRY(one_iteration());
            CG_TRY(fetch_flags(c, hf));
            if (hf[F_STOP]) break;
        }
        if (exec) cudaGraphExecDestroy(exec);
        io->n_iter = hf[5]; io->converged = hf[6];
        A->n_matvec += io->n_iter;
        if (M) M->n_matvec += io->n_iter;
        std::vector<double> hist((size_t)io->n_iter + 1);
        CG_TRY(cudaMemcpy(hist.data(), res_hist, hist.size() * sizeof(double), cudaMemcpyDeviceToHost) == cudaSuccess ? 0 : LKB_ERR_CUDA);
        for (int i = 1; i <= io->n_iter; ++i) push_res(io->res, io->res_cap, &io->res_len, hist[i]);
        *info = io->converged ? io->n_iter : -io->n_iter;
        io->info = *info;
        return cleanup2(check_launch(c, "cg"));
    }
#undef CG_TRY
#define CG_TRY(call) do { rc = (call); if (rc) return cleanup(rc); } while (0)
    for (int it = 1; it <= maxiter; ++it) {
        A->n_matvec++;
        CG_TRY(op_apply_enqueue(A, p->d, Ap->d, false, nullptr));
        Scalar pAp;
        CG_TRY(vec_dot_sync(c, kind, p->d, Ap->d, b->n, &pAp));
        const cd alpha = round_kind(kind, cd(rr_old.re, rr_old.im) / cd(pAp.re, pAp.im));
        launch_axpby(kind, c->stream, to_scalar(alpha), p->d, one, x->d, b->n, c->sms);      // x += alpha p
        launch_axpby(kind, c->stream, to_scalar(-alpha), Ap->d, one, r->d, b->n, c->sms);    // r -= alpha Ap
        c->launches += 2;
        Scalar rr_new;
        CG_TRY(make_z()); CG_TRY(vec_dot_sync(c, kind, r->d, z->d, b->n, &rr_new));
        const double residual = sqrt(hypot(rr_new.re, rr_new.im));
        io->n_iter++;
        push_res(io->res, io->res_cap, &io->res_len, residual);
        if (residual < tol) { io->converged = 1; break; }
        const cd beta = round_kind(kind, cd(rr_new.re, rr_new.im) / cd(rr_old.re, rr_old.im));
        launch_axpby(kind, c->stream, one, z->d, to_scalar(beta), p->d, b->n, c->sms);       // p = z + beta p
        c->launches++;
        rr_old = rr_new;
    }
#undef CG_TRY
    *info = io->converged ? io->n_iter : -io->n_iter;
    io->info = *info;
    return cleanup(check_launch(c, "cg"));
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
