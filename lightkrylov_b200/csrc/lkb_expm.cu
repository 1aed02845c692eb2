// lkb_expm.cu -- further callers of the Arnoldi step (SURVEY 8f rank 4) and the on-disk formats of the spectral solvers.
//
//   kexpm_vec          src/Expm/ExpmLib.fypp:128-232      c = exp(tau A) b by Arnoldi + dense expm of the small matrix
//   write_results      src/IterativeSolvers/IterativeSolvers.fypp:882-924   text table of intermediate Ritz values
//   save_eigenspectrum src/IterativeSolvers/IterativeSolvers.fypp:941-960   .npy (real array k x 2 or k x 3, Fortran order)
//
// The dense `expm` of the reference is stdlib_linalg's (fortran-lang/stdlib, unpinned in fpm.toml:25; absent from the
// tree): Pade approximant of order 10 with scaling and squaring (Moler & Van Loan method 3 / Golub & Van Loan
// Alg. 11.3.1, the algorithm stdlib documents for `expm`).  It is restated below on the host in complex double.
#include <math.h>
#include <stdio.h>
#include <string.h>
#include <algorithm>
#include <complex>
#include <numeric>
#include <string>
#include <vector>
#include "../../include/lkb.h"
#include "lkb_internal.h"

using namespace lkb;

namespace {

// C = A B (n x n, column-major)
void matmul(int n, const std::vector<cd>& A, const std::vector<cd>& B, std::vector<cd>& C) {
    C.assign((size_t)n * n, cd(0));
    for (int j = 0; j < n; ++j)
        for (int l = 0; l < n; ++l) {
            const cd b = B[l + (size_t)n * j];
            if (b == cd(0)) continue;
            for (int i = 0; i < n; ++i) C[i + (size_t)n * j] += A[i + (size_t)n * l] * b;
        }
}
// solve D X = E in place of E (LU with partial pivoting, as gesv)
bool solve(int n, std::vector<cd> D, std::vector<cd>& E) {
    for (int c = 0; c < n; ++c) {
        int piv = c; double best = std::abs(D[c + (size_t)n * c]);
        for (int i = c + 1; i < n; ++i) if (std::abs(D[i + (size_t)n * c]) > best) { best = std::abs(D[i + (size_t)n * c]); piv = i; }
        if (best == 0.0) return false;
        if (piv != c)
            for (int j = 0; j < n; ++j) { std::swap(D[c + (size_t)n * j], D[piv + (size_t)n * j]); std::swap(E[c + (size_t)n * j], E[piv + (size_t)n * j]); }
        const cd inv = cd(1) / D[c + (size_t)n * c];
        for (int i = c + 1; i < n; ++i) {
            const cd f = D[i + (size_t)n * c] * inv;
            if (f == cd(0)) continue;
            for (int j = c; j < n; ++j) D[i + (size_t)n * j] -= f * D[c + (size_t)n * j];
            for (int j = 0; j < n; ++j) E[i + (size_t)n * j] -= f * E[c + (size_t)n * j];
        }
    }
    for (int j = 0; j < n; ++j)
        for (int i = n - 1; i >= 0; --i) {
            cd s = E[i + (size_t)n * j];
            for (int l = i + 1; l < n; ++l) s -= D[i + (size_t)n * l] * E[l + (size_t)n * j];
            E[i + (size_t)n * j] = s / D[i + (size_t)n * i];
        }
    return true;
}
// E = exp(A): Pade order q = 10, scaling and squaring
bool dense_expm(int n, const std::vector<cd>& Ain, std::vector<cd>& E) {
    const int q = 10;
    double nrm = 0.0;                                   // infinity norm
    for (int i = 0; i < n; ++i) { double s = 0; for (int j = 0; j < n; ++j) s += std::abs(Ain[i + (size_t)n * j]); nrm = std::max(nrm, s); }
    int ee = 0;
    if (nrm > 0.0) { int ex; frexp(nrm, &ex); ee = std::max(0, ex + 1); }     // max(0, 1 + exponent(norm))
    std::vector<cd> A(Ain);
    const double sc = ldexp(1.0, -ee);
    for (auto& v : A) v *= sc;
    std::vector<cd> X(A), D((size_t)n * n, cd(0)), T;
    E.assign((size_t)n * n, cd(0));
    double c = 0.5;
    for (int i = 0; i < n; ++i) { E[i + (size_t)n * i] = 1.0; D[i + (size_t)n * i] = 1.0; }
    for (size_t t = 0; t < A.size(); ++t) { E[t] += c * A[t]; D[t] -= c * A[t]; }
    bool pos = true;
    for (int k = 2; k <= q; ++k) {
        c = c * (double)(q - k + 1) / (double)(k * (2 * q - k + 1));
        matmul(n, A, X, T); X.swap(T);
        for (size_t t = 0; t < X.size(); ++t) { E[t] += c * X[t]; D[t] += (pos ? c : -c) * X[t]; }
        pos = !pos;
    }
    if (!solve(n, D, E)) return false;
    for (int s = 0; s < ee; ++s) { matmul(n, E, E, T); E.swap(T); }
    return true;
}

// Fortran edit descriptor E16.9: 0.ddddddddd E+ee right-justified in 16 columns
std::string fortran_e16_9(double v) {
    char buf[64];
    if (v != v) return std::string("             NaN");
    if (isinf(v)) return std::string(v > 0 ? "        Infinity" : "       -Infinity");
    if (v == 0.0) { snprintf(buf, sizeof(buf), "%16s", "0.000000000E+00"); return buf; }
    const double a = fabs(v);
    int e = (int)floor(log10(a)) + 1;
    double m = a / pow(10.0, e);
    long long digits = llround(m * 1e9);
    if (digits >= 1000000000LL) { digits = 100000000LL; e += 1; }
    if (digits < 100000000LL) { digits *= 10; e -= 1; }          // log10 rounding at powers of ten
    char body[40];
    if (abs(e) <= 99) snprintf(body, sizeof(body), "%s0.%09lldE%c%02d", v < 0 ? "-" : "", digits, e < 0 ? '-' : '+', abs(e));
    else snprintf(body, sizeof(body), "%s0.%09lld%c%03d", v < 0 ? "-" : "", digits, e < 0 ? '-' : '+', abs(e));
    snprintf(buf, sizeof(buf), "%16s", body);
    return buf;
}

}  // namespace

extern "C" {

// kexpm_vec(c, A, b, tau, tol, info, trans, kdim)       src/Expm/ExpmLib.fypp:128-232
//   info = kp (dimension used) when the error estimate |E(kp,1) beta| <= tol, -1 otherwise; kdim <= 0 = kmax = 100.
int lkb_kexpm_vec(lkb_vec_t cvec, lkb_op_t A, lkb_vec_t b, double tau, double tol, int32_t* info, int32_t trans, int32_t kdim) {
    if (!cvec || !A || !b || !info || cvec->n != b->n || cvec->kind != b->kind || A->kind != b->kind || A->m != b->n || A->n != b->n)
        { set_error("kexpm_vec: bad arguments"); return LKB_ERR_ARG; }
    lkb_ctx_s* c = b->ctx;
    const int kind = b->kind;
    const size_t es = kind_size(kind);
    const int nk = kdim > 0 ? kdim : 100;
    *info = 0;
    double beta = 0.0;
    LKB_TRY(vec_norm_sync(c, kind, b->d, b->n, &beta));
    if (beta == 0.0) {                                  // input is zero => output is zero (:180-184)
        LKB_TRY(lkb_vec_zero(cvec));
        *info = 1;
        return 0;
    }
    BasisOwner X;
    LKB_TRY(lkb_basis_create(c, kind, b->n, b->n_global, b->row0, nk + 1, X.out()));
    prof_launch(c, PC_OTHER, 1, [&] { launch_axpby(kind, c->stream, Scalar{1.0 / beta, 0.0}, b->d, Scalar{0, 0}, X->d, b->n, c->sms); });   // X(1) = b / beta
    LKB_TRY(check_launch(c, "kexpm start"));
    const int ldh = nk + 1;
    std::vector<char> H((size_t)ldh * (nk + 1) * es, 0);          // (nk+1) x (nk+1) as in the reference (:170)
    std::vector<cd> Hk, E;
    double err_est = 0.0;
    int kp = 1;
    for (int k = 1; k <= nk; ++k) {
        kp = k + 1;
        int32_t ainfo = 0;
        LKB_TRY(lkb_arnoldi(A, X, H.data(), ldh, &ainfo, k, k, -1.0, trans, 1));
        const bool breakdown = (ainfo == k);
        if (breakdown) kp = k;                                     // do not consider the extended matrix (:199-203)
        Hk.assign((size_t)kp * kp, cd(0));
        for (int j = 0; j < kp; ++j)
            for (int i = 0; i < kp; ++i) Hk[i + (size_t)kp * j] = tau * load_kind(kind, H.data(), (size_t)i + (size_t)ldh * j);
        if (!dense_expm(kp, Hk, E)) { set_error("kexpm_vec: singular Pade denominator"); return LKB_ERR_LAPACK; }
        // |E(kp,1) beta| (:213).  The reference writes merge(0, abs(E(kp,1)*beta), info == k), but `info` was overwritten with -2
        // three lines earlier when the breakdown was detected (:201), so the estimate is NOT zeroed on breakdown: the loop goes
        // on with the refilled vector and stops two steps later, where E(kp,1) is exactly zero (H(k+1,k) = 0 decouples the
        // blocks).  Reproduced literally: info = k + 2 after a breakdown at step k unless |E(k,1) beta| <= tol already.
        err_est = std::abs(E[(size_t)(kp - 1)] * beta);
        LKB_TRY(bcast_host(c, &err_est, sizeof(double)));
        if (err_est <= tol || k == nk) {
            // c = beta * X(:kp) E(:kp,1)   (:209-210; the reference forms it every step, only the last one survives)
            std::vector<char> coef((size_t)kp * es);
            for (int i = 0; i < kp; ++i) store_kind(kind, coef.data(), i, beta * E[(size_t)i]);
            LKB_TRY(lkb_basis_lincomb(X, kp, coef.data(), cvec));
            if (err_est <= tol) break;
        }
    }
    LKB_TRY(lkb_sync(c));
    *info = (err_est <= tol) ? kp : -1;
    return 0;
}

// kexpm_mat(C, A, B, tau, tol, info, trans, kdim)       src/Expm/ExpmLib.fypp:234-362
//   C(:, :p) = exp(tau A) B(:, :p) by block Arnoldi with blksize p = size(B).  B = Q R by the pivoting QR (qr.fypp:32-107),
//   the columns of R are permuted back (:295); each block step exponentiates the extended block-Hessenberg matrix and
//   estimates the error by norm(matmul(E(kp+1:kpp, :p), R), 2) -- stdlib's `norm` of a rank-2 array is the 2-norm over ALL
//   elements (Frobenius).  Literal details: the loop runs up to nk = kdim*p BLOCK steps (:279, :300); on Arnoldi breakdown
//   kpp = kp, the section E(kp+1:kpp, :) is empty, the estimate is 0 and the loop exits.  The reference allocates all
//   p*(nk+1) basis vectors and the (p(nk+1))^2 matrices H and E up front (:281-289) -- 903 vectors for p = 3 and the default
//   kdim; here the basis and H start with room for 8 block steps and double on demand (new columns are zero, as zero_basis
//   leaves them), so the memory follows the steps actually taken.
//   info = kpp (dimension used) when err_est <= tol, -1 otherwise; kdim <= 0 = kmax = 100.  The reference forms
//   C = (X E(:, :p)) R every step; only the last one survives, so it is formed once, as X (E(:, :p) R).
int lkb_kexpm_mat(lkb_basis_t Cb, lkb_op_t A, lkb_basis_t B, int p, double tau, double tol, int32_t* info, int32_t trans, int32_t kdim) {
    if (!Cb || !A || !B || !info || p < 1 || B->ncols < p || Cb->ncols < p || Cb->n != B->n || Cb->kind != B->kind ||
        A->kind != B->kind || A->m != B->n || A->n != B->n) { set_error("kexpm_mat: bad arguments"); return LKB_ERR_ARG; }
    lkb_ctx_s* c = B->ctx;
    const int kind = B->kind;
    const size_t es = kind_size(kind);
    const int nsteps = kdim > 0 ? kdim : 100;
    const int nk = nsteps * p;
    *info = 0;
    BasisOwner Xwrk, X;
    LKB_TRY(lkb_basis_create(c, kind, B->n, B->n_global, B->row0, p, Xwrk.out()));
    const double one_d[2] = {1.0, 0.0}, zero_d[2] = {0.0, 0.0};
    const float one_f[2] = {1.f, 0.f}, zero_f[2] = {0.f, 0.f};
    const bool sp = (kind == KS || kind == KC);
    LKB_TRY(lkb_basis_axpby(sp ? (const void*)one_f : (const void*)one_d, B, 0, sp ? (const void*)zero_f : (const void*)zero_d, Xwrk, 0, p));
    // B = Q R P^T : pivoting QR, then permcols(R, invperm(perm))   (:295)
    std::vector<char> Rp((size_t)p * p * es, 0);
    std::vector<int32_t> perm(p, 0), invp(p, 0);
    int32_t qinfo = 0;
    LKB_TRY(lkb_qr_pivoting(Xwrk, 0, p, Rp.data(), p, perm.data(), -1.0, &qinfo));
    for (int i = 0; i < p; ++i) invp[perm[i] - 1] = i;
    std::vector<cd> R((size_t)p * p);
    double fro2 = 0.0;
    for (int q = 0; q < p; ++q)
        for (int i = 0; i < p; ++i) {
            R[i + (size_t)p * q] = load_kind(kind, Rp.data(), (size_t)i + (size_t)p * invp[q]);
            fro2 += std::norm(R[i + (size_t)p * q]);
        }
    double err_est = 0.0;
    int kpp = p;
    if (fro2 == 0.0) {                                             // input is zero => output is zero (:297-300)
        LKB_TRY(lkb_basis_zero(Cb, 0, p));
    } else {
        int cap = std::min(nk, 8);                                 // block steps the basis / H currently have room for
        LKB_TRY(lkb_basis_create(c, kind, B->n, B->n_global, B->row0, p * (cap + 1), X.out()));
        LKB_TRY(lkb_initialize_krylov_subspace(X, Xwrk, 0, p));
        int ldh = p * (cap + 1);
        std::vector<char> H((size_t)ldh * ldh * es, 0);
        std::vector<cd> Hk, E, M;
        std::vector<char> coef;
        const void* one = sp ? (const void*)one_f : (const void*)one_d;
        const void* zero = sp ? (const void*)zero_f : (const void*)zero_d;
        for (int k = 1; k <= nk; ++k) {
            if (k > cap) {                                         // double the room: copy the basis and re-lay H
                const int cap2 = std::min(nk, 2 * cap), ld2 = p * (cap2 + 1);
                BasisOwner X2;
                LKB_TRY(lkb_basis_create(c, kind, B->n, B->n_global, B->row0, p * (cap2 + 1), X2.out()));
                LKB_TRY(lkb_basis_axpby(one, X, 0, zero, X2, 0, p * (cap + 1)));
                std::swap(X, X2);                                  // the old basis goes with X2
                std::vector<char> H2((size_t)ld2 * ld2 * es, 0);
                for (int j = 0; j < ldh; ++j) memcpy(&H2[(size_t)j * ld2 * es], &H[(size_t)j * ldh * es], (size_t)ldh * es);
                H.swap(H2);
                ldh = ld2; cap = cap2;
            }
            const int kp = k * p;
            kpp = kp + p;
            int32_t ainfo = 0;
            LKB_TRY(lkb_arnoldi(A, X, H.data(), ldh, &ainfo, k, k, -1.0, trans, p));
            if (ainfo == kp) kpp = kp;                             // breakdown: do not consider the extended matrix (:314-318)
            Hk.assign((size_t)kpp * kpp, cd(0));
            for (int j = 0; j < kpp; ++j)
                for (int i = 0; i < kpp; ++i) Hk[i + (size_t)kpp * j] = tau * load_kind(kind, H.data(), (size_t)i + (size_t)ldh * j);
            if (!dense_expm(kpp, Hk, E)) { set_error("kexpm_mat: singular Pade denominator"); return LKB_ERR_LAPACK; }
            // M = E(:kpp, :p) R ; err_est = || M(kp+1:kpp, :) ||_F   (:338-346; the section is empty after a breakdown)
            M.assign((size_t)kpp * p, cd(0));
            for (int q = 0; q < p; ++q)
                for (int l = 0; l < p; ++l) {
                    const cd r = R[l + (size_t)p * q];
                    if (r == cd(0)) continue;
                    for (int i = 0; i < kpp; ++i) M[i + (size_t)kpp * q] += E[i + (size_t)kpp * l] * r;
                }
            double e2 = 0.0;
            for (int q = 0; q < p; ++q) for (int i = kp; i < kpp; ++i) e2 += std::norm(M[i + (size_t)kpp * q]);
            err_est = sqrt(e2);
            LKB_TRY(bcast_host(c, &err_est, sizeof(double)));
            if (err_est <= tol || k == nk) {
                coef.resize((size_t)kpp * es);
                for (int q = 0; q < p; ++q) {
                    for (int i = 0; i < kpp; ++i) store_kind(kind, coef.data(), i, M[i + (size_t)kpp * q]);
                    VecOwner cq;
                    LKB_TRY(lkb_basis_col(Cb, q, cq.out()));
                    LKB_TRY(lkb_basis_lincomb(X, kpp, coef.data(), cq));
                }
                if (err_est <= tol) break;
            }
        }
    }
    LKB_TRY(lkb_sync(c));
    *info = (err_est <= tol) ? kpp : -1;
    return 0;
}

// krylov_exptA(vec_out, A, vec_in, tau, info, trans)    src/Expm/ExpmLib.fypp:364-392: the wrapper that conforms to the
// abstract_exptA interface (AbstractLinops.fypp:105-123): kexpm_vec with tol = atol_kind and kdim = 30.
int lkb_krylov_expta(lkb_vec_t vec_out, lkb_op_t A, lkb_vec_t vec_in, double tau, int32_t* info, int32_t trans) {
    if (!vec_in) { set_error("krylov_exptA: bad arguments"); return LKB_ERR_ARG; }
    return lkb_kexpm_vec(vec_out, A, vec_in, tau, atol_of(vec_in->kind), info, trans, 30);
}

// write_results(filename, vals, res, tol)                IterativeSolvers.fypp:882-924
//   vals: k reals (is_complex = 0) or k (re, im) pairs; res is sorted ascending IN PLACE, as the reference does.
int lkb_write_results(const char* filename, int32_t is_complex, const double* vals, double* res, int32_t k, double tol) {
    if (!filename || !vals || !res || k < 0) { set_error("write_results: bad arguments"); return LKB_ERR_ARG; }
    std::vector<int> idx(k);
    std::iota(idx.begin(), idx.end(), 0);
    std::stable_sort(idx.begin(), idx.end(), [&](int a, int b) { return res[a] < res[b]; });       // sort_index(res, indices)
    std::vector<double> sorted(k);
    for (int i = 0; i < k; ++i) sorted[i] = res[idx[i]];
    for (int i = 0; i < k; ++i) res[i] = sorted[i];
    FILE* f = fopen(filename, "w");
    if (!f) { set_error("write_results: cannot open %s", filename); return LKB_ERR_ARG; }
    if (is_complex) fprintf(f, "%6s%18s%18s%18s%18s%6s\n", "Iter", "Re", "Im", "modulus", "residual", "conv");
    else fprintf(f, "%6s%18s%18s%6s\n", "Iter", "value", "residual", "conv");
    for (int i = 0; i < k; ++i) {
        const int s = idx[i];
        if (is_complex) {
            const double re = vals[2 * s], im = vals[2 * s + 1];
            fprintf(f, "%6d  %s  %s  %s  %s  %4s\n", k, fortran_e16_9(re).c_str(), fortran_e16_9(im).c_str(),
                    fortran_e16_9(sqrt(re * re + im * im)).c_str(), fortran_e16_9(res[i]).c_str(), res[i] < tol ? "T" : "F");
        } else {
            fprintf(f, "%6d  %s  %s  %4s\n", k, fortran_e16_9(vals[s]).c_str(), fortran_e16_9(res[i]).c_str(), res[i] < tol ? "T" : "F");
        }
    }
    fclose(f);
    return 0;
}

// save_eigenspectrum(lambda, residuals, fname)           IterativeSolvers.fypp:941-960  (stdlib save_npy)
//   array(k, 3) = (Re, Im, residual) for complex lambda, array(k, 2) = (lambda, residual) for real; Fortran order,
//   '<f8' (single_precision = 0) or '<f4'.
int lkb_save_eigenspectrum(const char* fname, int32_t is_complex, int32_t single_precision, const double* lambda,
                           const double* residuals, int32_t k) {
    if (!fname || !lambda || !residuals || k < 0) { set_error("save_eigenspectrum: bad arguments"); return LKB_ERR_ARG; }
    const int ncol = is_complex ? 3 : 2;
    char dict[256];
    snprintf(dict, sizeof(dict), "{'descr': '%s', 'fortran_order': True, 'shape': (%d, %d), }", single_precision ? "<f4" : "<f8", k, ncol);
    std::string header(dict);
    const size_t pre = 6 + 2 + 2;                                  // magic, version, header length (NPY 1.0)
    size_t total = pre + header.size() + 1;
    const size_t pad = (64 - total % 64) % 64;
    header.append(pad, ' ');
    header.push_back('\n');
    FILE* f = fopen(fname, "wb");
    if (!f) { set_error("save_eigenspectrum: cannot open %s", fname); return LKB_ERR_ARG; }
    const unsigned char magic[8] = {0x93, 'N', 'U', 'M', 'P', 'Y', 1, 0};
    const unsigned short hlen = (unsigned short)header.size();
    fwrite(magic, 1, 8, f); fwrite(&hlen, 2, 1, f); fwrite(header.data(), 1, header.size(), f);
    auto put = [&](double v) { if (single_precision) { const float x = (float)v; fwrite(&x, 4, 1, f); } else fwrite(&v, 8, 1, f); };
    if (is_complex) {
        for (int i = 0; i < k; ++i) put(lambda[2 * i]);
        for (int i = 0; i < k; ++i) put(lambda[2 * i + 1]);
    } else {
        for (int i = 0; i < k; ++i) put(lambda[i]);
    }
    for (int i = 0; i < k; ++i) put(residuals[i]);
    fclose(f);
    return 0;
}

}  // extern "C"
