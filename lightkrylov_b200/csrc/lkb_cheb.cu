// lkb_cheb.cu -- Chebyshev polynomial preconditioner: M r = z_m, the result of m Chebyshev iterations (Saad, Iterative
// Methods for Sparse Linear Systems, Alg. 12.1, true-residual form) on the Jacobi-scaled system D^-1 A z = D^-1 r from
// z_0 = 0, D = diag(A), on the interval [a, b] = [lmin, lmax]:
//     theta = (b + a) / 2, delta = (b - a) / 2, sigma = theta / delta, rho_0 = 1 / sigma
//     d_0 = D^-1 r / theta ;  z_1 = d_0
//     k = 1 .. m-1:  s_k = D^-1 (r - A z_k) ;  rho_k = 1 / (2 sigma - rho_{k-1})
//                    d_k = rho_k rho_{k-1} d_{k-1} + (2 rho_k / delta) s_k ;  z_{k+1} = z_k + d_k
// A fixed linear operator built from m - 1 applications of A and a diagonal scaling: no inner products, so no reductions.
// On a stencil every step is one kernel: the stencil kernel with the update as its store epilogue (kernels_ops.cu:
// ChebStep); on any other operator a step is A's matvec and k_cheb_update (kernels_vec.cu).
#include <math.h>
#include <algorithm>
#include "../../include/lkb.h"
#include "lkb_internal.h"

using namespace lkb;

namespace lkb {
// z_j (j >= 2) of a stencil operator's steps lives in y when m - j is even, else in cheb_z: the last step writes y, and no
// step reads and writes the same buffer (the stencil's neighbours read z_k while z_{k+1} is written)
static void* stencil_z(lkb_op_s* M, void* y, int j) { return ((M->cheb_m - j) % 2 == 0) ? y : M->cheb_z.get(); }

void cheb_coefficients(int m, double a, double b, std::vector<double>& ca, std::vector<double>& cb) {
    const double theta = (b + a) / 2, delta = (b - a) / 2, sigma = theta / delta;
    ca.assign(m, 0.0); cb.assign(m, 0.0);
    cb[0] = 1.0 / theta;
    double rho = 1.0 / sigma;
    for (int k = 1; k < m; ++k) {
        const double rho_k = 1.0 / (2.0 * sigma - rho);
        ca[k] = rho_k * rho;
        cb[k] = 2.0 * rho_k / delta;
        rho = rho_k;
    }
}

int cheb_apply_enqueue(lkb_op_s* M, const void* r, void* y, bool trans, const int* flags) {
    lkb_op_s* A = M->base;
    lkb_ctx_s* c = M->ctx;
    const int m = M->cheb_m;
    const Scalar invd = M->cheb_invd;       // k_cheb_update conjugates it for trans; the fused step takes conj(D)^-1 itself
    const void* invd_vec = A->type == OP_STENCIL ? nullptr : M->diag.get();
    // z_1 = D^-1 r / theta: the output when m = 1 (on a stencil with m > 1 the first fused step forms it on the fly)
    if (m == 1 || A->type != OP_STENCIL) {
        prof_launch(c, PC_OTHER, 1, [&] {
            launch_cheb_update(M->kind, c->stream, r, invd_vec, invd, nullptr, nullptr, nullptr, y, M->m, 0.0, M->cheb_b[0], trans,
                               true, flags, c->sms);
        });
        LKB_TRY(check_launch(c, "chebyshev"));
    }
    for (int k = 1; k < m; ++k) {
        const bool last = k == m - 1;
        if (A->type == OP_STENCIL) {
            const void* zk = k == 1 ? r : stencil_z(M, y, k);
            const ChebArgs ca{r, M->cheb_d.get(), trans ? Scalar{invd.re, -invd.im} : invd, M->cheb_a[k], M->cheb_b[k], M->cheb_b[0],
                              k == 1, last};
            int nl = 0;
            prof_begin(c, PC_MATVEC);
            const int e = stencil_halo_exchange(A, zk, flags, false, &nl);
            if (e == 0) launch_stencil_cheb(A->kind, c->stream, A->st, zk, stencil_z(M, y, k + 1), trans, flags, ca);
            prof_end(c, PC_MATVEC, e == 0 ? nl + 1 : nl);
            LKB_TRY(e);
            LKB_TRY(check_launch(c, "chebyshev step"));
        } else {
            // t = A z_k (z lives in y), then d, z updated; d_0 = z_1, so the first step reads d from y
            LKB_TRY(op_apply_enqueue(A, y, M->cheb_t, trans, flags));
            prof_launch(c, PC_OTHER, 1, [&] {
                launch_cheb_update(M->kind, c->stream, r, invd_vec, invd, M->cheb_t, k == 1 ? y : M->cheb_d.get(),
                                   last ? nullptr : M->cheb_d.get(), y, M->m, M->cheb_a[k], M->cheb_b[k], trans, false, flags, c->sms);
            });
            LKB_TRY(check_launch(c, "chebyshev update"));
        }
    }
    return 0;
}
}  // namespace lkb

extern "C" {
// Creation: D^-1 through the Jacobi set-up (k_jacobi; the scalar 1 / c0 for a stencil), the Gershgorin bound when lmax <= 0
// (host for a stencil or a diagonal operator, k_gershgorin otherwise), the coefficients on the host in double, the work
// vectors.  Collective only for a row-sharded CSR with lmax <= 0: the bound is a max over the ranks.
int lkb_op_chebyshev_create(lkb_op_t A, int32_t degree, double lmin, double lmax, lkb_op_t* M) {
    if (!A || !M) { set_error("chebyshev_create: null argument"); return LKB_ERR_ARG; }
    if (degree < 1) { set_error("chebyshev_create: degree %d < 1", (int)degree); return LKB_ERR_ARG; }
    lkb_ctx_s* c = A->ctx;
    JacobiSrc src; int64_t n_global = 0;
    LKB_TRY(jacobi_source(A, "chebyshev_create", &src, &n_global));
    cudaSetDevice(c->dev);
    OpOwner op(new lkb_op_s());
    op->ctx = c; op->type = OP_CHEB; op->kind = A->kind; op->m = op->n = A->m; op->uid = next_uid();
    op->cheb_m = degree;
    const bool want_bound = !(lmax > 0.0);
    const bool collective = want_bound && A->type == OP_CSR && A->dist && c->world > 1;
    unsigned long long bad = ~0ULL;
    double bound = 0.0;
    int err = 0;       // a local failure; with `collective` it is reported only after the ranks agreed
    if (A->type == OP_STENCIL) {
        const Scalar c0 = A->st.coef[0];
        const double q = c0.re * c0.re + c0.im * c0.im;
        if (!(q > 0.0) || !isfinite(q)) bad = (unsigned long long)src.row0;
        else op->cheb_invd = Scalar{c0.re / q, -c0.im / q};
        double sum = 0.0;
        for (int k = 0; k < (A->st.dim == 2 ? 5 : 7); ++k) sum += hypot(A->st.coef[k].re, A->st.coef[k].im);
        bound = sum / sqrt(q);
    } else {
        err = cuda_alloc(op->diag, std::max<size_t>((size_t)A->m * kind_size(A->kind), 16));
        if (err == 0) err = jacobi_build(c, A->kind, src, op->diag, &bad, (want_bound && A->type != OP_DIAG) ? &bound : nullptr);
        if (A->type == OP_DIAG) bound = 1.0;     // D^-1 A = I
    }
    if (collective) {
        // every rank contributes (bound, failed); the max over the ranks is the global bound and whether any rank failed
        NcclApi* api = nccl_api();
        double v[2] = {bound, (err != 0 || bad != ~0ULL) ? 1.0 : 0.0};
        if (!api) return LKB_ERR_NCCL;
        LKB_TRY(ensure_ws(c, 2));
        LKB_CUDA(cudaMemcpyAsync(c->tmpw, v, sizeof(v), cudaMemcpyHostToDevice, c->stream));
        if (api->AllReduce(c->tmpw, c->tmpw, 2, /*ncclFloat64*/ 8, /*ncclMax*/ 2, c->comm, c->stream) != 0) {
            set_error("chebyshev_create: all-reduce of the Gershgorin bound failed"); return LKB_ERR_NCCL;
        }
        LKB_CUDA(cudaMemcpyAsync(v, c->tmpw, sizeof(v), cudaMemcpyDeviceToHost, c->stream));
        LKB_CUDA(cudaStreamSynchronize(c->stream));
        if (v[1] != 0.0 && err == 0 && bad == ~0ULL) { set_error("chebyshev_create: the set-up failed on another rank"); return LKB_ERR_ARG; }
        bound = v[0];
    }
    LKB_TRY(err);
    if (bad != ~0ULL) { set_error("chebyshev_create: the diagonal entry of global row %llu is zero or not finite", bad); return LKB_ERR_ARG; }
    const double b = want_bound ? bound : lmax;
    const double a = lmin > 0.0 ? lmin : b / 100.0;
    if (!(a < b) || !isfinite(b)) { set_error("chebyshev_create: lmin = %g is not below lmax = %g", a, b); return LKB_ERR_ARG; }
    cheb_coefficients(degree, a, b, op->cheb_a, op->cheb_b);
    const size_t bytes = std::max<size_t>((size_t)A->m * kind_size(A->kind), 16);
    if (degree >= 3) LKB_TRY(cuda_alloc(op->cheb_d, bytes));
    if (degree >= 3 && A->type == OP_STENCIL) LKB_TRY(cuda_alloc(op->cheb_z, bytes));
    if (degree >= 2 && A->type != OP_STENCIL) LKB_TRY(cuda_alloc(op->cheb_t, bytes));
    op->base = A;
    A->users++;
    *M = op.release();
    return 0;
}
}  // extern "C"
