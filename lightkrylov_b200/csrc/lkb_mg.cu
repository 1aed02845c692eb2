// lkb_mg.cu -- geometric multigrid preconditioner for the 5- and 7-point stencils (Trottenberg, Oosterlee & Schueller,
// Multigrid, 2001): M r is one V-cycle from a zero initial guess.
//
// Level 0 is A.  Write A = rho I + sum_d T_d, T_d = tri(c-d, -(c-d + c+d), c+d) along axis d, rho = c0 + sum_d (c-d + c+d).
// Every axis is coarsened at once, n -> n / 2 with coarse point c at fine point 2c+1; P is the tensor product of the 1-D
// linear interpolations (fine 2c+1 takes coarse c, fine 2c and 2c+2 half of it, coarse points outside the grid are zero)
// and R = 2^-dim P^T.  The coarse operator takes the Galerkin product along each axis, T_d' = 1/2 P_d^T T_d P_d, with rho
// unchanged: T_d' is tridiagonal with constant off-diagonals and a constant diagonal except its last entry, which differs
// once a level on the way had an even size along d (a vertex-centred grid of even size has no nested uniform coarse grid).
// So every level is a 5- / 7-point stencil plus at most dim centre corrections e_d on its last rows, which the fused kernels
// carry (kernels_ops.cu: MgStep).  Coarsening stops at the first level with <= 512 unknowns or an axis below 2 points; that
// level is inverted densely on the host in double and applied with k_dense.
//
// Smoother on level ell: Chebyshev of degree m in D^-1 A (lkb_cheb.cu's recurrence; Adams, Brezina, Hu & Tuminaro,
// J. Comput. Phys. 188, 2003) on [b / (2 dim), b], b the Gershgorin bound of the level's D^-1 A.  Pre-smoothing starts from
// 0, post-smoothing from the corrected x with d_0 = D^-1 (b - A x) / theta:
//     V(ell, b) = A_L^-1 b                                                  ell = L
//               : x = S(b, 0) ;  x += P V(ell + 1, R (b - A x)) ;  x = S(b, x)
// M^H is the same cycle on A_ell^H with conj(D) and (A_L^-1)^H (P and R are real); with the same polynomial before and
// after, M is Hermitian for Hermitian A, and positive definite when b >= lambda_max.
#include <math.h>
#include <algorithm>
#include <complex>
#include <vector>
#include "../../include/lkb.h"
#include "lkb_internal.h"

using namespace lkb;

namespace lkb {
namespace {

constexpr int64_t MG_COARSE_MAX = 512;       // unknowns of the coarsest level (its dense inverse is formed on the host)

// a 1-D tridiagonal operator tri(lo, dg, up) of size n whose last diagonal entry is dgl
struct Tri { int64_t n; cd lo, up, dg, dgl; };
cd tri_at(const Tri& T, int64_t p, int64_t q) {
    if (q == p - 1) return T.lo;
    if (q == p + 1) return T.up;
    if (q == p) return p == T.n - 1 ? T.dgl : T.dg;
    return 0.0;
}
// (1/2 P^T T P)_ij: P's column c holds fine 2c, 2c+1, 2c+2 with weights 1/2, 1, 1/2 (those inside the grid)
cd galerkin(const Tri& T, int64_t i, int64_t j) {
    static const double w[3] = {0.5, 1.0, 0.5};
    cd s = 0.0;
    for (int a = 0; a < 3 && 2 * i + a < T.n; ++a)
        for (int b = 0; b < 3 && 2 * j + b < T.n; ++b) s += w[a] * tri_at(T, 2 * i + a, 2 * j + b) * w[b];
    return 0.5 * s;
}
// T' = 1/2 P^T T P, checked to be tridiagonal with constant off-diagonals and a diagonal constant but for its last entry
int coarsen(const Tri& T, Tri& C, int level, int axis) {
    C.n = T.n / 2;
    C.dg = galerkin(T, 0, 0); C.dgl = galerkin(T, C.n - 1, C.n - 1);
    C.lo = C.n > 1 ? galerkin(T, 1, 0) : cd(0.0); C.up = C.n > 1 ? galerkin(T, 0, 1) : cd(0.0);
    for (int64_t i = 0; i < C.n; ++i) {
        bool ok = i == C.n - 1 || galerkin(T, i, i) == C.dg;
        if (i > 0) ok = ok && galerkin(T, i, i - 1) == C.lo;
        if (i + 1 < C.n) ok = ok && galerkin(T, i, i + 1) == C.up;
        if (i + 2 < C.n) ok = ok && galerkin(T, i, i + 2) == 0.0;
        if (!ok) {
            set_error("multigrid_create: the coarse operator of level %d along axis %d is not a constant-coefficient "
                      "tridiagonal at row %lld", level + 1, axis, (long long)i);
            return LKB_ERR_ARG;
        }
    }
    return 0;
}
}  // namespace

int mg_hierarchy(int dim, const int64_t* n0, const cd* coef, std::vector<MgHostLevel>& lv, std::vector<cd>& inv) {
    lv.clear(); inv.clear();
    Tri T[3];
    cd rho = coef[0];
    for (int d = 0; d < dim; ++d) {
        const cd cm = coef[1 + 2 * d], cp = coef[2 + 2 * d];
        T[d] = Tri{n0[d], cm, cp, -(cm + cp), -(cm + cp)};
        rho += cm + cp;
    }
    int64_t N = 0;
    for (int level = 0;; ++level) {
        MgHostLevel L = {};
        L.c0 = level == 0 ? coef[0] : rho;
        N = 1;
        int64_t nmin = T[0].n;
        for (int d = 0; d < 3; ++d) {
            L.n[d] = d < dim ? T[d].n : 1;
            if (d >= dim) continue;
            if (level > 0) L.c0 += T[d].dg;
            L.cm[d] = T[d].lo; L.cp[d] = T[d].up; L.e[d] = T[d].dgl - T[d].dg;
            N *= T[d].n; nmin = std::min(nmin, T[d].n);
        }
        // Gershgorin bound of D^-1 A over the row types: along each axis the first row, an interior one and the last
        // (whichever exist), which differ in the neighbours they have and, for the last, in the centre
        L.lmax = 0.0;
        int ncomb = 1;
        for (int d = 0; d < dim; ++d) ncomb *= 3;
        for (int comb = 0; comb < ncomb; ++comb) {
            cd centre = L.c0;
            double off = 0.0;
            bool exists = true;
            for (int d = 0, cc = comb; d < dim; ++d, cc /= 3) {
                const int pos = cc % 3;                        // 0 first, 1 interior, 2 last
                const int64_t i = pos == 0 ? 0 : pos == 1 ? 1 : L.n[d] - 1;
                if ((pos == 1 && L.n[d] < 3) || (pos == 2 && L.n[d] < 2)) { exists = false; break; }
                if (i > 0) off += std::abs(L.cm[d]);
                if (i < L.n[d] - 1) off += std::abs(L.cp[d]); else centre += L.e[d];
            }
            if (!exists) continue;
            const double ac = std::abs(centre);
            if (!(ac > 0.0) || !std::isfinite(ac)) {
                set_error("multigrid_create: a centre coefficient of level %d (grid %lld x %lld x %lld) is zero or not finite",
                          level, (long long)L.n[0], (long long)L.n[1], (long long)L.n[2]);
                return LKB_ERR_ARG;
            }
            L.lmax = std::max(L.lmax, (ac + off) / ac);
        }
        lv.push_back(L);
        if (N <= MG_COARSE_MAX || nmin < 2) break;
        for (int d = 0; d < dim; ++d) {
            Tri C;
            LKB_TRY(coarsen(T[d], C, level, d));
            T[d] = C;
        }
    }
    const MgHostLevel& L = lv.back();
    if (N > MG_COARSE_MAX) {
        set_error("multigrid_create: the coarsest grid %lld x %lld x %lld (level %d, an axis below 2 points) has %lld > %lld "
                  "unknowns", (long long)L.n[0], (long long)L.n[1], (long long)L.n[2], (int)lv.size() - 1, (long long)N,
                  (long long)MG_COARSE_MAX);
        return LKB_ERR_ARG;
    }
    // the coarsest operator, row-major, then Gauss-Jordan with partial pivoting on [A | I]
    std::vector<cd> a((size_t)N * N, 0.0), x((size_t)N * N, 0.0);
    const int64_t stride[3] = {1, L.n[0], L.n[0] * L.n[1]};
    for (int64_t p = 0; p < N; ++p) {
        const int64_t idx[3] = {p % L.n[0], (p / L.n[0]) % L.n[1], p / (L.n[0] * L.n[1])};
        cd centre = L.c0;
        for (int d = 0; d < dim; ++d) {
            if (idx[d] > 0) a[(size_t)p * N + p - stride[d]] = L.cm[d];
            if (idx[d] < L.n[d] - 1) a[(size_t)p * N + p + stride[d]] = L.cp[d]; else centre += L.e[d];
        }
        a[(size_t)p * N + p] = centre;
        x[(size_t)p * N + p] = 1.0;
    }
    for (int64_t k = 0; k < N; ++k) {
        int64_t piv = k;
        for (int64_t r = k + 1; r < N; ++r)
            if (std::abs(a[(size_t)r * N + k]) > std::abs(a[(size_t)piv * N + k])) piv = r;
        const double ap = std::abs(a[(size_t)piv * N + k]);
        if (!(ap > 0.0) || !std::isfinite(ap)) {
            set_error("multigrid_create: the coarsest operator (level %d, %lld unknowns) is singular", (int)lv.size() - 1, (long long)N);
            return LKB_ERR_ARG;
        }
        if (piv != k)
            for (int64_t c = 0; c < N; ++c) { std::swap(a[(size_t)k * N + c], a[(size_t)piv * N + c]); std::swap(x[(size_t)k * N + c], x[(size_t)piv * N + c]); }
        const cd s = 1.0 / a[(size_t)k * N + k];
        for (int64_t c = 0; c < N; ++c) { a[(size_t)k * N + c] *= s; x[(size_t)k * N + c] *= s; }
        for (int64_t r = 0; r < N; ++r) {
            const cd f = a[(size_t)r * N + k];
            if (r == k || f == 0.0) continue;
            for (int64_t c = k; c < N; ++c) a[(size_t)r * N + c] -= f * a[(size_t)k * N + c];
            for (int64_t c = 0; c < N; ++c) x[(size_t)r * N + c] -= f * x[(size_t)k * N + c];
        }
    }
    inv.assign((size_t)N * N, 0.0);
    for (int64_t i = 0; i < N; ++i)
        for (int64_t j = 0; j < N; ++j) inv[(size_t)i + (size_t)N * j] = x[(size_t)i * N + j];
    return 0;
}

namespace {
// one fused smoothing step on level L (kernels_ops.cu: MgStep); for M^H with A_ell^H and conj(D)
int mg_step(lkb_op_s* M, const MgLevel& L, const void* x, void* y, bool trans, const int* flags, int mode, const void* r,
            const void* d_in, void* d_out, double alpha, double beta) {
    lkb_ctx_s* c = M->ctx;
    MgArgs ma;
    ma.r = r; ma.d_in = d_in; ma.d_out = d_out;
    for (int q = 0; q < 8; ++q) {
        ma.invd[q] = Scalar{L.invd[q].re, trans ? -L.invd[q].im : L.invd[q].im};
        ma.ecor[q] = Scalar{L.ecor[q].re, trans ? -L.ecor[q].im : L.ecor[q].im};
    }
    ma.alpha = alpha; ma.beta = beta; ma.b0 = L.b0; ma.mode = mode;
    prof_launch(c, PC_MATVEC, 1, [&] { launch_stencil_mg(M->kind, c->stream, L.st, x, y, trans, flags, ma); });
    return check_launch(c, "multigrid smoothing step");
}

// y = V(ell, b)
int vcycle(lkb_op_s* M, size_t ell, const void* b, void* y, bool trans, const int* flags) {
    lkb_ctx_s* c = M->ctx;
    MgLevel& L = M->mg[ell];
    if (ell + 1 == M->mg.size()) {
        const int64_t n = L.st.nx * L.st.ny * L.st.nz;
        prof_launch(c, PC_OTHER, 1, [&] { launch_dense(M->kind, c->stream, n, n, M->mg_inv, b, y, trans, flags); });
        return check_launch(c, "multigrid coarsest solve");
    }
    const int m = M->mg_m;
    // pre-smoothing from 0: z_1 .. z_m, z_j in xa when m - j is even (z_m = xa), else in xb
    auto z = [&](int j) -> void* { return (m - j) % 2 == 0 ? L.xa.get() : L.xb.get(); };
    int k0 = 1;
    if (!L.edges && m >= 2) {          // D is constant: the first step forms z_1 from b on the fly
        LKB_TRY(mg_step(M, L, b, z(2), trans, flags, MG_FIRST_R, b, nullptr, m > 2 ? L.d.get() : nullptr, L.ca[1], L.cb[1]));
        k0 = 2;
    } else {
        LKB_TRY(mg_step(M, L, b, z(1), trans, flags, MG_SCALE, b, nullptr, nullptr, 0.0, 0.0));
    }
    for (int k = k0; k < m; ++k)       // d_0 = z_1
        LKB_TRY(mg_step(M, L, z(k), z(k + 1), trans, flags, MG_STEP, b, k == 1 ? z(1) : L.d.get(),
                        k == m - 1 ? nullptr : L.d.get(), L.ca[k], L.cb[k]));
    // coarse-grid correction
    Scalar ecor[8];
    for (int q = 0; q < 8; ++q) ecor[q] = Scalar{L.ecor[q].re, trans ? -L.ecor[q].im : L.ecor[q].im};
    MgLevel& C = M->mg[ell + 1];
    prof_launch(c, PC_OTHER, 1, [&] {
        launch_mg_restrict(M->kind, c->stream, L.st, ecor, L.xa, b, C.b, trans, flags, c->sms);
    });
    LKB_TRY(check_launch(c, "multigrid restriction"));
    LKB_TRY(vcycle(M, ell + 1, C.b, C.e, trans, flags));
    prof_launch(c, PC_OTHER, 1, [&] { launch_mg_prolong(M->kind, c->stream, L.st, C.e, L.xa, flags, c->sms); });
    LKB_TRY(check_launch(c, "multigrid prolongation"));
    // post-smoothing from xa: o_1 .. o_m, o_j in y when m - j is even (o_m = y), else in xb
    auto o = [&](int j) -> void* { return (m - j) % 2 == 0 ? y : L.xb.get(); };
    LKB_TRY(mg_step(M, L, L.xa, o(1), trans, flags, MG_STEP, b, nullptr, m > 1 ? L.d.get() : nullptr, 0.0, L.b0));
    for (int j = 2; j <= m; ++j)
        LKB_TRY(mg_step(M, L, o(j - 1), o(j), trans, flags, MG_STEP, b, L.d, j == m ? nullptr : L.d.get(), L.ca[j - 1], L.cb[j - 1]));
    return 0;
}
}  // namespace

int mg_apply_enqueue(lkb_op_s* M, const void* r, void* y, bool trans, const int* flags) {
    return vcycle(M, 0, r, y, trans, flags);
}
}  // namespace lkb

extern "C" {
int lkb_op_multigrid_create(lkb_op_t A, int32_t degree, lkb_op_t* M) {
    if (!A || !M) { set_error("multigrid_create: null argument"); return LKB_ERR_ARG; }
    if (A->type != OP_STENCIL) {
        set_error("multigrid_create: A is not a 5- or 7-point stencil (operator type %d); the Chebyshev or GMRES-polynomial "
                  "preconditioner serves other operators", A->type);
        return LKB_ERR_ARG;
    }
    if (degree < 1) { set_error("multigrid_create: degree %d < 1", (int)degree); return LKB_ERR_ARG; }
    const StencilArgs& st = A->st;
    const int dim = st.dim;
    const int64_t nslow = dim == 2 ? st.ny : st.nz;
    if (nslow != A->nslow_global) {
        set_error("multigrid_create: A is row-sharded (this rank holds %lld of its %lld %s); multigrid needs the whole grid "
                  "on one GPU", (long long)nslow, (long long)A->nslow_global, dim == 2 ? "rows" : "planes");
        return LKB_ERR_ARG;
    }
    const int64_t n0[3] = {st.nx, st.ny, st.nz};
    cd coef[7];
    for (int q = 0; q < 7; ++q) coef[q] = cd(st.coef[q].re, st.coef[q].im);
    std::vector<MgHostLevel> hl;
    std::vector<cd> inv;
    LKB_TRY(mg_hierarchy(dim, n0, coef, hl, inv));
    lkb_ctx_s* c = A->ctx;
    cudaSetDevice(c->dev);
    OpOwner op(new lkb_op_s());
    op->ctx = c; op->type = OP_MG; op->kind = A->kind; op->m = op->n = A->m; op->uid = next_uid();
    op->mg_m = degree;
    const size_t es = kind_size(A->kind);
    op->mg.resize(hl.size());
    for (size_t ell = 0; ell < hl.size(); ++ell) {
        const MgHostLevel& H = hl[ell];
        MgLevel& L = op->mg[ell];
        L.st.nx = H.n[0]; L.st.ny = H.n[1]; L.st.nz = H.n[2]; L.st.dim = dim;
        L.st.halo_lo = L.st.halo_hi = nullptr;
        L.st.coef[0] = to_scalar(H.c0);
        for (int d = 0; d < 3; ++d) { L.st.coef[1 + 2 * d] = to_scalar(H.cm[d]); L.st.coef[2 + 2 * d] = to_scalar(H.cp[d]); }
        for (int q = 0; q < 8; ++q) {
            cd e = 0.0;
            for (int d = 0; d < dim; ++d)
                if (q >> d & 1) e += H.e[d];
            L.ecor[q] = to_scalar(e);
            L.invd[q] = to_scalar(1.0 / (H.c0 + e));
            L.edges = L.edges || e != 0.0;
        }
        const size_t bytes = std::max<size_t>((size_t)(H.n[0] * H.n[1] * H.n[2]) * es, 16);
        if (ell > 0) { LKB_TRY(cuda_alloc(L.b, bytes)); LKB_TRY(cuda_alloc(L.e, bytes)); }
        if (ell + 1 == hl.size()) continue;
        cheb_coefficients(degree, H.lmax / (2 * dim), H.lmax, L.ca, L.cb);
        L.b0 = L.cb[0];
        LKB_TRY(cuda_alloc(L.xa, bytes));
        if (degree >= 2) { LKB_TRY(cuda_alloc(L.xb, bytes)); LKB_TRY(cuda_alloc(L.d, bytes)); }
    }
    const size_t ni = inv.size();
    std::vector<char> hinv(ni * es);
    for (size_t q = 0; q < ni; ++q) store_kind(A->kind, hinv.data(), q, inv[q]);
    LKB_TRY(cuda_alloc(op->mg_inv, std::max<size_t>(ni * es, 16)));
    LKB_CUDA(cudaMemcpyAsync(op->mg_inv, hinv.data(), ni * es, cudaMemcpyHostToDevice, c->stream));
    LKB_CUDA(cudaStreamSynchronize(c->stream));
    op->base = A;
    A->users++;
    *M = op.release();
    return 0;
}
}  // extern "C"
