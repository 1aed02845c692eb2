// lkb_poly.cu -- GMRES-polynomial preconditioner (Loe & Morgan, "Toward efficient polynomial preconditioning for GMRES",
// Numer. Linear Algebra Appl. 2022; Trilinos Belos GmresPoly).  With nonzero roots theta_1 .. theta_d,
//     pi(z) = prod_i (1 - z / theta_i),   p(z) = (1 - pi(z)) / z   (degree d - 1),   M = p(A),   A M = I - pi(A).
// M r by the product recurrence, in the order the roots are stored:
//     y = r ; z = 0
//     root theta (real kinds: real theta; complex kinds: any):  z += y / theta ;  y <- y - A (y / theta)
//     pair (theta, conj theta) of a real kind, a = Re theta, q = |theta|^2:
//                                t = A y ;  w = (2a/q) y - t/q ;  z += w ;  y <- y - A w
// with the last factor's y update skipped: d - 1 applications of A and no inner products.  A last single root's z update
// is folded into the launch before it.  On a stencil every application of A is one launch of the stencil kernel with the
// PolyStep store epilogue (kernels_ops.cu); on any other operator it is A's matvec and k_poly_update (kernels_vec.cu).
// lkb_op_gmres_poly_create takes the roots from a short Arnoldi run: the harmonic Ritz values, with extra copies of the
// outlying ones and in modified Leja order (gmres_poly_roots).
#include <math.h>
#include <algorithm>
#include <complex>
#include <vector>
#include "../../include/lkb.h"
#include "lkb_internal.h"

using namespace lkb;

namespace lkb {
namespace {

constexpr int POLY_MAX_ROOTS = 256, POLY_MAX_DEGREE = 128;

// A must map its vectors onto vectors of the same layout: the recurrence applies it to its own output
int poly_square(const lkb_op_s* A, const char* what) {
    if (A->m != A->n) {
        set_error("%s: A is not square (%lld x %lld local rows / columns)", what, (long long)A->m, (long long)A->n);
        return LKB_ERR_ARG;
    }
    if (A->type == OP_CSR && A->dist) {
        const int r = A->ctx->rank;
        if (A->row_off[r] != A->col_off[r] || A->row_cnt[r] != A->col_cnt[r] || A->m_global != A->n_global) {
            set_error("%s: A is not square (row-sharded CSR whose row slab [%lld,+%lld) differs from its column slab "
                      "[%lld,+%lld) on rank %d)", what, (long long)A->row_off[r], (long long)A->row_cnt[r],
                      (long long)A->col_off[r], (long long)A->col_cnt[r], r);
            return LKB_ERR_ARG;
        }
    }
    return 0;
}

// global index of this rank's first row and the global length of A's vectors (a callback's vectors start at row 0)
void poly_layout(const lkb_op_s* A, int64_t* row0, int64_t* n_global) {
    *row0 = 0; *n_global = A->m;
    if (A->type == OP_STENCIL) {
        const int64_t plane = A->st.dim == 2 ? A->st.nx : A->st.nx * A->st.ny;
        *row0 = A->slow0 * plane; *n_global = A->nslow_global * plane;
    } else if (A->type == OP_CSR && A->dist) {
        *row0 = A->row_off[A->ctx->rank]; *n_global = A->m_global;
    } else if (A->type == OP_DIAG) {
        *row0 = A->diag_row0; *n_global = A->diag_n_global;
    } else if (A->type == OP_CHEB || A->type == OP_POLY) {
        poly_layout(A->base, row0, n_global);
    }
}

// The steps of one application (lkb_internal.h: PolyStepPlan) and the number of work vectors they use.  y lives in r
// and then in the work vectors; every step's output goes to a work vector that none of its operands occupies, so no fused
// stencil step writes the buffer it reads its stencil input from.  On the generic path a step without an output still
// needs a work vector for A x.
int poly_plan(const std::vector<Scalar>& roots, bool cplx, bool stencil, std::vector<PolyStepPlan>& plan) {
    struct Factor { bool pair; cd th; };
    std::vector<Factor> F;
    for (size_t i = 0; i < roots.size(); ++i) {
        const cd th(roots[i].re, roots[i].im);
        F.push_back({!cplx && th.imag() != 0.0, th});
        if (F.back().pair) ++i;
    }
    bool used[3] = {false, false, false};
    int nslots = 0;
    auto take = [&]() {
        for (int s = 0; s < 3; ++s)
            if (!used[s]) { used[s] = true; nslots = std::max(nslots, s + 1); return s; }
        return (int)POLY_NONE;      // not reached: at most y, w and the new y are live
    };
    auto release = [&](int s) { if (s >= 0) used[s] = false; };
    bool acc_seen = false;
    auto step = [&](int x, int dst, int v, bool matvec, bool out, cd a0, cd a1, cd a2, bool acc, cd b0, cd b1, cd b2) {
        PolyStepPlan p;
        p.x = x; p.dst = dst; p.v = v; p.matvec = matvec; p.out = out;
        p.acc = acc ? (acc_seen ? 2 : 1) : 0;
        acc_seen = acc_seen || acc;
        const cd a[3] = {a0, a1, a2}, b[3] = {b0, b1, b2};
        for (int i = 0; i < 3; ++i) { p.a[i] = to_scalar(a[i]); p.b[i] = to_scalar(b[i]); }
        plan.push_back(p);
    };
    const cd O = 0.0, I = 1.0;
    int y = POLY_R;
    const size_t nf = F.size();
    for (size_t f = 0; f < nf; ++f) {
        const bool last = f + 1 == nf;
        const bool fold = f + 2 == nf && !F[nf - 1].pair;       // a last single root: its z update joins this factor's last launch
        const cd il = fold ? I / F[nf - 1].th : O;
        if (!F[f].pair) {
            const cd it = I / F[f].th;
            if (last) {                                         // the only root: z = r / theta, no A
                step(y, POLY_NONE, POLY_NONE, false, false, O, O, O, true, it, O, O);
            } else if (fold) {                                  // z += y/theta + (y - A y/theta)/theta_d
                const int d = stencil ? (int)POLY_NONE : take();
                step(y, d, POLY_NONE, true, false, O, O, O, true, it + il, -it * il, O);
                release(d);
                break;
            } else {                                            // z += y/theta ; y <- y - A y/theta
                const int d = take();
                step(y, d, POLY_NONE, true, true, I, -it, O, true, it, O, O);
                release(y); y = d;
            }
        } else {
            const double q = std::norm(F[f].th);
            const cd c0 = 2.0 * F[f].th.real() / q, c1 = -1.0 / q;
            if (last) {                                         // z += (2a/q) y - A y/q
                const int d = stencil ? (int)POLY_NONE : take();
                step(y, d, POLY_NONE, true, false, O, O, O, true, c0, c1, O);
                release(d);
            } else {
                const int w = take();                           // w = (2a/q) y - A y/q ; z += w
                step(y, w, POLY_NONE, true, true, c0, c1, O, true, c0, c1, O);
                if (fold) {                                     // z += (y - A w)/theta_d
                    const int d = stencil ? (int)POLY_NONE : take();
                    step(w, d, y, true, false, O, O, O, true, O, -il, il);
                    release(d);
                    break;
                }
                const int d = take();                           // y <- y - A w
                step(w, d, y, true, true, O, -I, I, false, O, O, O);
                release(y); release(w); y = d;
            }
        }
    }
    return nslots;
}

// The polynomial operator on A from roots in application order, after the checks of lkb_op_poly_create
int poly_make(lkb_op_s* A, const std::vector<cd>& roots, const char* what, lkb_op_t* M) {
    lkb_ctx_s* c = A->ctx;
    LKB_TRY(poly_square(A, what));
    const int n = (int)roots.size();
    if (n < 1 || n > POLY_MAX_ROOTS) { set_error("%s: %d roots (1 .. %d)", what, n, POLY_MAX_ROOTS); return LKB_ERR_ARG; }
    const bool cplx = kind_cplx(A->kind);
    for (int i = 0; i < n; ++i) {
        const cd th = roots[i];
        if (!std::isfinite(th.real()) || !std::isfinite(th.imag()) || th == 0.0) {
            set_error("%s: root %d = (%g, %g) is zero or not finite", what, i, th.real(), th.imag());
            return LKB_ERR_ARG;
        }
    }
    if (!cplx)
        for (int i = 0; i < n; ++i) {
            if (roots[i].imag() == 0.0) continue;
            if (i + 1 >= n || roots[i + 1] != std::conj(roots[i])) {
                set_error("%s: complex root %d = (%g, %g) of a real operator is not immediately followed by its conjugate",
                          what, i, roots[i].real(), roots[i].imag());
                return LKB_ERR_ARG;
            }
            ++i;
        }
    cudaSetDevice(c->dev);
    OpOwner op(new lkb_op_s());
    op->ctx = c; op->type = OP_POLY; op->kind = A->kind; op->m = op->n = A->m; op->uid = next_uid();
    for (const cd& th : roots) op->poly_roots.push_back(to_scalar(th));
    const int nslots = poly_plan(op->poly_roots, cplx, A->type == OP_STENCIL, op->poly_plan);
    for (int s = 0; s < nslots; ++s) LKB_TRY(cuda_alloc(op->poly_w[s], std::max<size_t>((size_t)A->m * kind_size(A->kind), 16)));
    op->base = A;
    A->users++;
    *M = op.release();
    return 0;
}

}  // namespace

int poly_apply_enqueue(lkb_op_s* M, const void* r, void* y, bool trans, const int* flags) {
    lkb_op_s* A = M->base;
    lkb_ctx_s* c = M->ctx;
    auto buf = [&](int id) -> void* { return id == POLY_R ? const_cast<void*>(r) : id == POLY_NONE ? nullptr : M->poly_w[id].get(); };
    for (const PolyStepPlan& p : M->poly_plan) {
        PolyArgs pa;
        pa.v = buf(p.v); pa.acc = p.acc ? y : nullptr; pa.acc_read = p.acc == 2;
        for (int i = 0; i < 3; ++i) {          // M^H = conj(p)(A^H): every coefficient conjugated
            pa.a[i] = Scalar{p.a[i].re, trans ? -p.a[i].im : p.a[i].im};
            pa.b[i] = Scalar{p.b[i].re, trans ? -p.b[i].im : p.b[i].im};
        }
        const void* x = buf(p.x);
        if (!p.matvec) {
            prof_launch(c, PC_OTHER, 1, [&] { launch_poly_update(M->kind, c->stream, x, nullptr, nullptr, M->m, pa, flags, c->sms); });
            LKB_TRY(check_launch(c, "polynomial update"));
        } else if (A->type == OP_STENCIL) {
            int nl = 0;
            prof_begin(c, PC_MATVEC);
            const int e = stencil_halo_exchange(A, x, flags, false, &nl);
            if (e == 0) launch_stencil_poly(A->kind, c->stream, A->st, x, p.out ? buf(p.dst) : nullptr, trans, flags, pa);
            prof_end(c, PC_MATVEC, e == 0 ? nl + 1 : nl);
            LKB_TRY(e);
            LKB_TRY(check_launch(c, "polynomial step"));
        } else {
            void* t = buf(p.dst);
            LKB_TRY(op_apply_enqueue(A, x, t, trans, flags));
            prof_launch(c, PC_OTHER, 1, [&] {
                launch_poly_update(M->kind, c->stream, x, t, p.out ? t : nullptr, M->m, pa, flags, c->sms);
            });
            LKB_TRY(check_launch(c, "polynomial update"));
        }
    }
    return 0;
}

int gmres_poly_roots(int kind, const cd* H, int ldh, int k, std::vector<cd>& roots) {
    roots.clear();
    const bool cplx = kind_cplx(kind);
    if (k < 1 || ldh < k + 1) { set_error("gmres_poly_roots: k = %d, ldh = %d", k, ldh); return LKB_ERR_ARG; }
    // f = H_k^-H e_k: Gaussian elimination with partial pivoting on H_k^H
    std::vector<cd> L((size_t)k * k), f(k, 0.0);
    for (int j = 0; j < k; ++j)
        for (int i = 0; i < k; ++i) L[i + (size_t)k * j] = std::conj(H[j + (size_t)ldh * i]);
    f[k - 1] = 1.0;
    for (int j = 0; j < k; ++j) {
        int p = j;
        for (int i = j + 1; i < k; ++i)
            if (std::abs(L[i + (size_t)k * j]) > std::abs(L[p + (size_t)k * j])) p = i;
        const double piv = std::abs(L[p + (size_t)k * j]);
        if (!(piv > 0.0) || !std::isfinite(piv)) {
            set_error("gmres_poly_roots: the %d x %d Hessenberg matrix H_k is singular", k, k);
            return LKB_ERR_ARG;
        }
        if (p != j) {
            for (int q = j; q < k; ++q) std::swap(L[j + (size_t)k * q], L[p + (size_t)k * q]);
            std::swap(f[j], f[p]);
        }
        for (int i = j + 1; i < k; ++i) {
            const cd m = L[i + (size_t)k * j] / L[j + (size_t)k * j];
            if (m == 0.0) continue;
            for (int q = j + 1; q < k; ++q) L[i + (size_t)k * q] -= m * L[j + (size_t)k * q];
            f[i] -= m * f[j];
        }
    }
    for (int i = k - 1; i >= 0; --i) {
        cd s = f[i];
        for (int q = i + 1; q < k; ++q) s -= L[i + (size_t)k * q] * f[q];
        f[i] = s / L[i + (size_t)k * i];
    }
    // harmonic Ritz values: eig(H_k + |h_{k+1,k}|^2 f e_k^T)
    const double h2 = std::norm(H[k + (size_t)ldh * (k - 1)]);
    std::vector<cd> G((size_t)k * k);
    for (int j = 0; j < k; ++j)
        for (int i = 0; i < k; ++i) G[i + (size_t)k * j] = H[i + (size_t)ldh * j] + (j == k - 1 ? h2 * f[i] : 0.0);
    std::vector<cd> th;
    LKB_TRY(host_eig_double(cplx, k, G, k, th));
    for (int i = 0; i < k; ++i)
        if (!std::isfinite(th[i].real()) || !std::isfinite(th[i].imag()) || th[i] == 0.0) {
            set_error("gmres_poly_roots: harmonic Ritz value %d = (%g, %g) is zero or not finite", i, th[i].real(), th[i].imag());
            return LKB_ERR_ARG;
        }
    // stability: ceil((log10 pof_i - 4) / 14) extra copies of a root at which the other factors' product pof_i > 1e4
    // (real kinds: a pair's conjugate gets the copies of its im > 0 member; geev returns it right after)
    std::vector<cd> ext(th);
    for (int i = 0; i < k; ++i) {
        double lp = 0.0;
        for (int j = 0; j < k; ++j)
            if (j != i) lp += std::log10(std::abs(1.0 - th[i] / th[j]));
        const int extra = lp > 4.0 ? (int)std::ceil((lp - 4.0) / 14.0) : 0;
        const bool pair = !cplx && th[i].imag() > 0.0;
        for (int e = 0; e < extra; ++e) {
            ext.push_back(th[i]);
            if (pair) ext.push_back(th[i + 1]);
        }
        if (pair) ++i;
    }
    // modified Leja order: the largest modulus first, then the root maximising sum_j log|theta - theta_j| over the roots
    // placed so far; ties to the lowest index.  Real kinds: a pair is placed as a whole, im > 0 first.
    const int n = (int)ext.size();
    std::vector<char> placed(n, 0);
    auto candidate = [&](int j) { return !placed[j] && (cplx || ext[j].imag() >= 0.0); };
    auto place = [&](int j) {
        roots.push_back(ext[j]); placed[j] = 1;
        if (!cplx && ext[j].imag() > 0.0) { roots.push_back(ext[j + 1]); placed[j + 1] = 1; }
    };
    int best = -1;
    for (int j = 0; j < n; ++j)
        if (candidate(j) && (best < 0 || std::abs(ext[j]) > std::abs(ext[best]))) best = j;
    place(best);
    while ((int)roots.size() < n) {
        best = -1;
        double bs = 0.0;
        for (int j = 0; j < n; ++j) {
            if (!candidate(j)) continue;
            double s = 0.0;
            for (const cd& p : roots) s += std::log(std::abs(ext[j] - p));
            if (best < 0 || s > bs) { best = j; bs = s; }
        }
        place(best);
    }
    return 0;
}
}  // namespace lkb

extern "C" {
int lkb_op_poly_create(lkb_op_t A, int32_t nroots, const double* roots, lkb_op_t* M) {
    if (!A || !M || (nroots > 0 && !roots)) { set_error("poly_create: null argument"); return LKB_ERR_ARG; }
    if (nroots < 1 || nroots > POLY_MAX_ROOTS) { set_error("poly_create: %d roots (1 .. %d)", (int)nroots, POLY_MAX_ROOTS); return LKB_ERR_ARG; }
    std::vector<cd> th(nroots);
    for (int i = 0; i < nroots; ++i) th[i] = cd(roots[2 * i], roots[2 * i + 1]);
    return poly_make(A, th, "poly_create", M);
}

// Collective (the Arnoldi run is).  The start vector is the seeded normal fill of lkb_vec_fill_random, normalised: the
// same global vector at any sharding.  The context's `rand` stream is left where it was, also when the Arnoldi run breaks
// down and refills a column.  Rank 0's roots are authoritative (bcast_host).
int lkb_op_gmres_poly_create(lkb_op_t A, int32_t degree, uint64_t seed, lkb_op_t* M) {
    if (!A || !M) { set_error("gmres_poly_create: null argument"); return LKB_ERR_ARG; }
    if (degree < 1 || degree > POLY_MAX_DEGREE) { set_error("gmres_poly_create: degree %d (1 .. %d)", (int)degree, POLY_MAX_DEGREE); return LKB_ERR_ARG; }
    LKB_TRY(poly_square(A, "gmres_poly_create"));
    lkb_ctx_s* c = A->ctx;
    cudaSetDevice(c->dev);
    int64_t row0 = 0, n_global = 0;
    poly_layout(A, &row0, &n_global);
    const int ldh = degree + 1;
    std::vector<char> H((size_t)ldh * degree * kind_size(A->kind), 0);
    int32_t info = 0;
    {
        BasisOwner X;
        LKB_TRY(lkb_basis_create(c, A->kind, A->m, n_global, row0, degree + 1, X.out()));
        VecOwner v0;
        LKB_TRY(lkb_basis_col(X, 0, v0.out()));
        LKB_TRY(lkb_vec_fill_random(v0, LKB_DIST_NORMAL, seed));
        double nrm = 0.0;
        LKB_TRY(lkb_vec_norm(v0, &nrm));
        if (!(nrm > 0.0) || !std::isfinite(nrm)) { set_error("gmres_poly_create: start vector norm %g", nrm); return LKB_ERR_ARG; }
        prof_launch(c, PC_OTHER, 1, [&] { launch_scal(A->kind, c->stream, Scalar{1.0 / nrm, 0.0}, v0->d, v0->n, c->sms); });
        LKB_TRY(check_launch(c, "scal"));
        const uint64_t seed_calls = c->seed_calls;
        const int e = lkb_arnoldi(A, X, H.data(), ldh, &info, 1, degree, -1.0, 0, 1);
        c->seed_calls = seed_calls;
        LKB_TRY(e);
    }
    const int k = info > 0 && info < degree ? info : degree;
    std::vector<cd> Hd((size_t)ldh * k);
    for (int j = 0; j < k; ++j)
        for (int i = 0; i <= std::min(j + 1, k); ++i) Hd[i + (size_t)ldh * j] = load_kind(A->kind, H.data(), i + (size_t)ldh * j);
    std::vector<cd> roots;
    double head[2] = {0.0, 0.0};                        // rank 0's status and root count
    head[0] = gmres_poly_roots(A->kind, Hd.data(), ldh, k, roots);
    head[1] = (double)roots.size();
    LKB_TRY(bcast_host(c, head, sizeof(head)));
    if (head[0] != 0.0) {
        if (c->rank != 0) set_error("gmres_poly_create: the roots failed on rank 0");
        return (int)head[0];
    }
    roots.resize((size_t)head[1]);
    LKB_TRY(bcast_host(c, roots.data(), roots.size() * sizeof(cd)));
    return poly_make(A, roots, "gmres_poly_create", M);
}

int lkb_op_poly_roots(lkb_op_t M, int32_t cap, int32_t* nroots, double* roots) {
    if (!M || !nroots) { set_error("poly_roots: null argument"); return LKB_ERR_ARG; }
    if (M->type != OP_POLY) { set_error("poly_roots: not a polynomial operator (type %d)", M->type); return LKB_ERR_ARG; }
    const int n = (int)M->poly_roots.size();
    *nroots = n;
    if (cap < n || (n > 0 && !roots)) { set_error("poly_roots: %d roots do not fit cap = %d", n, (int)cap); return LKB_ERR_ARG; }
    for (int i = 0; i < n; ++i) { roots[2 * i] = M->poly_roots[i].re; roots[2 * i + 1] = M->poly_roots[i].im; }
    return 0;
}
}  // extern "C"
