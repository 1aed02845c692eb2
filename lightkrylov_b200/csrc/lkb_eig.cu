// lkb_eig.cu -- eigs / eighs / svds / krylov_schur: host shells around the device Krylov step.
//
//   eigs         src/IterativeSolvers/IterativeSolvers.fypp:972-1143
//   krylov_schur src/Krylov/BaseKrylov.fypp:782-834
//   eighs        src/IterativeSolvers/EIGHS/eighs.fypp:29-126
//   svds         src/IterativeSolvers/SVDS/svd_solvers.fypp:28-121
//   eig/ordschur src/Utilities/submodule_utility_functions.fypp:55-117
//
// The k x k algebra (k <= kdim) stays on the host as in the reference, which gets it from
// stdlib_linalg_lapack (geev, gees, trsen, syev/heev, gesdd; fortran-lang/stdlib, version unpinned
// in fpm.toml:25).  Here a Fortran-ABI LAPACK is resolved at run time with dlopen
// (lkb_set_lapack) and called IN THE PRECISION OF THE KIND, as stdlib's eig / schur / eigh / svd dispatch
// (sgeev / cgeev ... for rsp / csp, dgeev / zgeev ... for rdp / cdp); the surrounding bookkeeping (residuals,
// sorting) is done on the returned values in double.  All O(n) work (basis update X Z, Ritz-vector assembly)
// is the tall-skinny device GEMM in kernels_gemm.cu.
#include <dlfcn.h>
#include <math.h>
#include <stdlib.h>
#include <string.h>
#include <algorithm>
#include <complex>
#include <numeric>
#include <string>
#include <vector>
#include "../../include/lkb.h"
#include "lkb_internal.h"

using namespace lkb;
typedef int lint;   // LP64 LAPACK

namespace {

// One table per precision: the reference calls the LAPACK routines OF THE KIND (stdlib eig / schur / eigh / svd dispatch to
// sgeev / cgeev ... for rsp / csp and dgeev / zgeev ... for rdp / cdp), so the fp32 kinds run the s / c routines here too.
template <typename R> struct LaP {
    typedef std::complex<R> C;
    void (*geev)(const char*, const char*, const lint*, R*, const lint*, R*, R*, R*, const lint*, R*, const lint*, R*,
                 const lint*, lint*, size_t, size_t) = nullptr;
    void (*cgeev)(const char*, const char*, const lint*, C*, const lint*, C*, C*, const lint*, C*, const lint*, C*,
                  const lint*, R*, lint*, size_t, size_t) = nullptr;
    void (*gees)(const char*, const char*, void*, const lint*, R*, const lint*, lint*, R*, R*, R*, const lint*, R*,
                 const lint*, lint*, lint*, size_t, size_t) = nullptr;
    void (*cgees)(const char*, const char*, void*, const lint*, C*, const lint*, lint*, C*, C*, const lint*, C*,
                  const lint*, R*, lint*, lint*, size_t, size_t) = nullptr;
    void (*trsen)(const char*, const char*, const lint*, const lint*, R*, const lint*, R*, const lint*, R*, R*, lint*,
                  R*, R*, R*, const lint*, lint*, const lint*, lint*, size_t, size_t) = nullptr;
    void (*ctrsen)(const char*, const char*, const lint*, const lint*, C*, const lint*, C*, const lint*, C*, lint*, R*,
                   R*, C*, const lint*, lint*, size_t, size_t) = nullptr;
    void (*syev)(const char*, const char*, const lint*, R*, const lint*, R*, R*, const lint*, lint*, size_t, size_t) = nullptr;
    void (*heev)(const char*, const char*, const lint*, C*, const lint*, R*, C*, const lint*, R*, lint*, size_t, size_t) = nullptr;
    void (*gesdd)(const char*, const lint*, const lint*, R*, const lint*, R*, R*, const lint*, R*, const lint*, R*,
                  const lint*, lint*, lint*, size_t) = nullptr;
    void (*cgesdd)(const char*, const lint*, const lint*, C*, const lint*, R*, C*, const lint*, C*, const lint*, C*,
                   const lint*, R*, lint*, lint*, size_t) = nullptr;
};
struct Lapack {
    void* h = nullptr;
    LaP<double> d;
    LaP<float> s;
};
Lapack g_la;
template <typename R> const LaP<R>& la_of();
template <> const LaP<double>& la_of<double>() { return g_la.d; }
template <> const LaP<float>& la_of<float>() { return g_la.s; }

int lapack_open(const char* path, const char* prefix, const char* suffix) {
    void* h = dlopen(path, RTLD_NOW | RTLD_LOCAL);
    if (!h) { set_error("cannot dlopen LAPACK provider %s: %s", path, dlerror()); return LKB_ERR_LAPACK; }
    Lapack la; la.h = h;
    auto sym = [&](const char* name) -> void* {
        std::string s = std::string(prefix ? prefix : "") + name + (suffix ? suffix : "");
        return dlsym(h, s.c_str());
    };
#define LA(field, name) *(void**)(&la.field) = sym(name); if (!la.field) { set_error("LAPACK provider %s lacks %s%s%s", path, prefix ? prefix : "", name, suffix ? suffix : ""); dlclose(h); return LKB_ERR_LAPACK; }
    LA(d.geev, "dgeev") LA(d.cgeev, "zgeev") LA(d.gees, "dgees") LA(d.cgees, "zgees") LA(d.trsen, "dtrsen") LA(d.ctrsen, "ztrsen")
    LA(d.syev, "dsyev") LA(d.heev, "zheev") LA(d.gesdd, "dgesdd") LA(d.cgesdd, "zgesdd")
    LA(s.geev, "sgeev") LA(s.cgeev, "cgeev") LA(s.gees, "sgees") LA(s.cgees, "cgees") LA(s.trsen, "strsen") LA(s.ctrsen, "ctrsen")
    LA(s.syev, "ssyev") LA(s.heev, "cheev") LA(s.gesdd, "sgesdd") LA(s.cgesdd, "cgesdd")
#undef LA
    g_la = la;
    return 0;
}
int lapack_ready() {
    if (g_la.h) return 0;
    if (const char* env = getenv("LKB_LAPACK_LIB")) {
        const char* pre = getenv("LKB_LAPACK_PREFIX"); const char* suf = getenv("LKB_LAPACK_SUFFIX");
        if (lapack_open(env, pre ? pre : "", suf ? suf : "_") == 0) return 0;
    }
    for (const char* p : {"liblapack.so.3", "libopenblas.so.0", "libopenblas.so", "liblapack.so"})
        if (lapack_open(p, "", "_") == 0) return 0;
    set_error("no host LAPACK provider: call lkb_set_lapack(path, prefix, suffix) or set LKB_LAPACK_LIB");
    return LKB_ERR_LAPACK;
}

// eig(A(:k,:k)) -> vals (complex), vecs in LAPACK layout: for real kinds the REAL-pair convention
// (column i = Re, i+1 = Im of the pair), stored in the real parts of `vecs`.  R = precision of the kind.
template <typename R>
int host_eig_t(bool cplx, int k, const std::vector<cd>& A, int lda, std::vector<cd>& vals, std::vector<cd>& vecs) {
    typedef std::complex<R> C;
    const LaP<R>& la = la_of<R>();
    vals.assign(k, cd(0)); vecs.assign((size_t)k * k, cd(0));
    lint n = k, ldvl = 1, ldvr = k, info = 0;
    if (cplx) {
        std::vector<C> a((size_t)k * k), w(k), vr((size_t)k * k), work(std::max(1, 4 * k)); std::vector<R> rwork(2 * k);
        for (int j = 0; j < k; ++j) for (int i = 0; i < k; ++i) a[i + (size_t)k * j] = C(A[i + (size_t)lda * j]);
        C vl; lint lwork = (lint)work.size();
        la.cgeev("N", "V", &n, a.data(), &n, w.data(), &vl, &ldvl, vr.data(), &ldvr, work.data(), &lwork, rwork.data(), &info, 1, 1);
        for (int i = 0; i < k; ++i) vals[i] = cd(w[i]);
        for (size_t t = 0; t < vr.size(); ++t) vecs[t] = cd(vr[t]);
    } else {
        std::vector<R> a((size_t)k * k), wr(k), wi(k), vr((size_t)k * k), work(std::max(1, 8 * k));
        for (int j = 0; j < k; ++j) for (int i = 0; i < k; ++i) a[i + (size_t)k * j] = (R)A[i + (size_t)lda * j].real();
        R vl; lint lwork = (lint)work.size();
        la.geev("N", "V", &n, a.data(), &n, wr.data(), wi.data(), &vl, &ldvl, vr.data(), &ldvr, work.data(), &lwork, &info, 1, 1);
        for (int i = 0; i < k; ++i) vals[i] = cd(wr[i], wi[i]);
        for (size_t t = 0; t < vr.size(); ++t) vecs[t] = cd(vr[t], 0.0);
    }
    if (info != 0) { set_error("GEEV failed, info = %d", (int)info); return LKB_ERR_LAPACK; }
    return 0;
}
int host_eig(int kind, int k, const std::vector<cd>& A, int lda, std::vector<cd>& vals, std::vector<cd>& vecs) {
    LKB_TRY(lapack_ready());
    return (kind == KS || kind == KC) ? host_eig_t<float>(kind_cplx(kind), k, A, lda, vals, vecs)
                                      : host_eig_t<double>(kind_cplx(kind), k, A, lda, vals, vecs);
}

// schur(H) + median selector + ordschur (BaseKrylov.fypp:806-814, IterativeSolvers.fypp:1136-1141): T, Z (k x k) and the
// number of selected eigenvalues, in the precision of the kind.  H given as k x k complex doubles.
template <typename R>
int host_schur_select_t(bool cplx, int k, const std::vector<cd>& Hk, std::vector<cd>& Tc, std::vector<cd>& Zc, int32_t* nkeep) {
    typedef std::complex<R> C;
    const LaP<R>& la = la_of<R>();
    lint n = k, sdim = 0, info = 0, m = 0;
    std::vector<lint> sel(k, 0);
    std::vector<R> av(k);
    R s_ = 0, sep = 0;
    auto select = [&]() {
        std::vector<R> srt(av); std::sort(srt.begin(), srt.end());
        const R med = (k % 2) ? srt[k / 2] : (R)0.5 * (srt[k / 2 - 1] + srt[k / 2]);
        int cnt = 0; for (int i = 0; i < k; ++i) { sel[i] = av[i] > med; cnt += sel[i]; }
        *nkeep = cnt;
    };
    Tc.assign((size_t)k * k, cd(0)); Zc.assign((size_t)k * k, cd(0));
    if (cplx) {
        std::vector<C> T((size_t)k * k), Z((size_t)k * k), ev(k), work(std::max(1, 4 * k)); std::vector<R> rwork(k);
        for (size_t t = 0; t < T.size(); ++t) T[t] = C(Hk[t]);
        lint lwork = (lint)work.size(); lint bwork = 0;
        la.cgees("V", "N", nullptr, &n, T.data(), &n, &sdim, ev.data(), Z.data(), &n, work.data(), &lwork, rwork.data(), &bwork, &info, 1, 1);
        if (info != 0) { set_error("GEES failed, info = %d", (int)info); return LKB_ERR_LAPACK; }
        for (int i = 0; i < k; ++i) av[i] = std::abs(ev[i]);
        select();
        std::vector<C> w(k), wk(std::max(1, k)); lint lw = (lint)wk.size();
        la.ctrsen("N", "V", sel.data(), &n, T.data(), &n, Z.data(), &n, w.data(), &m, &s_, &sep, wk.data(), &lw, &info, 1, 1);
        if (info != 0) { set_error("TRSEN failed, info = %d", (int)info); return LKB_ERR_LAPACK; }
        for (size_t t = 0; t < T.size(); ++t) { Tc[t] = cd(T[t]); Zc[t] = cd(Z[t]); }
    } else {
        std::vector<R> T((size_t)k * k), Z((size_t)k * k), wr(k), wi(k), work(std::max(1, 8 * k));
        for (size_t t = 0; t < T.size(); ++t) T[t] = (R)Hk[t].real();
        lint lwork = (lint)work.size(); lint bwork = 0;
        la.gees("V", "N", nullptr, &n, T.data(), &n, &sdim, wr.data(), wi.data(), Z.data(), &n, work.data(), &lwork, &bwork, &info, 1, 1);
        if (info != 0) { set_error("GEES failed, info = %d", (int)info); return LKB_ERR_LAPACK; }
        for (int i = 0; i < k; ++i) av[i] = std::abs(C(wr[i], wi[i]));
        select();
        std::vector<R> wk(std::max(1, k)); lint lw = (lint)wk.size(); std::vector<lint> iwork(std::max(1, k)); lint liw = 1;
        la.trsen("N", "V", sel.data(), &n, T.data(), &n, Z.data(), &n, wr.data(), wi.data(), &m, &s_, &sep, wk.data(), &lw, iwork.data(), &liw, &info, 1, 1);
        if (info != 0) { set_error("TRSEN failed, info = %d", (int)info); return LKB_ERR_LAPACK; }
        for (size_t t = 0; t < T.size(); ++t) { Tc[t] = cd(T[t], 0.0); Zc[t] = cd(Z[t], 0.0); }
    }
    return 0;
}

// eigh(A(:k,:k)) on the lower triangle (syev / heev): eigenvalues ascending, eigenvectors as k x k (ld k)
template <typename R>
int host_eigh_t(bool cplx, int k, const std::vector<cd>& Ak, double* ev, std::vector<cd>& vk) {
    typedef std::complex<R> C;
    const LaP<R>& la = la_of<R>();
    lint n = k, linf = 0;
    std::vector<R> w(k);
    vk.assign((size_t)k * k, cd(0));
    if (cplx) {
        std::vector<C> a((size_t)k * k), work(std::max(1, 4 * k)); std::vector<R> rwork(std::max(1, 3 * k));
        for (size_t t = 0; t < a.size(); ++t) a[t] = C(Ak[t]);
        lint lwork = (lint)work.size();
        la.heev("V", "L", &n, a.data(), &n, w.data(), work.data(), &lwork, rwork.data(), &linf, 1, 1);
        for (size_t t = 0; t < a.size(); ++t) vk[t] = cd(a[t]);
    } else {
        std::vector<R> a((size_t)k * k), work(std::max(1, 8 * k));
        for (size_t t = 0; t < a.size(); ++t) a[t] = (R)Ak[t].real();
        lint lwork = (lint)work.size();
        la.syev("V", "L", &n, a.data(), &n, w.data(), work.data(), &lwork, &linf, 1, 1);
        for (size_t t = 0; t < a.size(); ++t) vk[t] = cd(a[t], 0.0);
    }
    if (linf != 0) { set_error("SYEV/HEEV failed, info = %d", (int)linf); return LKB_ERR_LAPACK; }
    for (int i = 0; i < k; ++i) ev[i] = (double)w[i];
    return 0;
}

// svd(A(:k,:k)) by gesdd: singular values, U and V = hermitian(VT) as k x k (ld k)
template <typename R>
int host_svd_t(bool cplx, int k, const std::vector<cd>& Ak, double* sv, std::vector<cd>& uk, std::vector<cd>& vk) {
    typedef std::complex<R> C;
    const LaP<R>& la = la_of<R>();
    lint n = k, linf = 0;
    std::vector<lint> iwork(8 * k);
    std::vector<R> s(k);
    uk.assign((size_t)k * k, cd(0)); vk.assign((size_t)k * k, cd(0));
    if (cplx) {
        std::vector<C> a((size_t)k * k), u((size_t)k * k), vt((size_t)k * k), work(std::max(1, 4 * k * k + 8 * k));
        std::vector<R> rwork(std::max(1, 8 * k * k + 8 * k));
        for (size_t t = 0; t < a.size(); ++t) a[t] = C(Ak[t]);
        lint lwork = (lint)work.size();
        la.cgesdd("A", &n, &n, a.data(), &n, s.data(), u.data(), &n, vt.data(), &n, work.data(), &lwork, rwork.data(), iwork.data(), &linf, 1);
        for (int j = 0; j < k; ++j) for (int i = 0; i < k; ++i) {
            uk[i + (size_t)k * j] = cd(u[i + (size_t)k * j]);
            vk[i + (size_t)k * j] = std::conj(cd(vt[j + (size_t)k * i]));      // V = hermitian(VT)
        }
    } else {
        std::vector<R> a((size_t)k * k), u((size_t)k * k), vt((size_t)k * k), work(std::max(1, 8 * k * k + 16 * k));
        for (size_t t = 0; t < a.size(); ++t) a[t] = (R)Ak[t].real();
        lint lwork = (lint)work.size();
        la.gesdd("A", &n, &n, a.data(), &n, s.data(), u.data(), &n, vt.data(), &n, work.data(), &lwork, iwork.data(), &linf, 1);
        for (int j = 0; j < k; ++j) for (int i = 0; i < k; ++i) {
            uk[i + (size_t)k * j] = cd(u[i + (size_t)k * j], 0.0);
            vk[i + (size_t)k * j] = cd(vt[j + (size_t)k * i], 0.0);
        }
    }
    if (linf != 0) { set_error("GESDD failed, info = %d", (int)linf); return LKB_ERR_LAPACK; }
    for (int i = 0; i < k; ++i) sv[i] = (double)s[i];
    return 0;
}

// stdlib sort_index(array, index, reverse=.true.): "non-increasing values in stable order" -- stdlib reverses the array,
// merge-sorts it (stable, ascending) and reverses again, so ties keep their ORIGINAL order: a conjugate pair stays (+, -) as
// LAPACK returns it and the eigenvector columns keep the (Re, Im) layout.  Pinned by the reference's own test, which compares
// eigvals with the analytic spectrum elementwise in the order (a + iw, a - iw) (test/TestIterativeSolvers.fypp:176-186).
std::vector<int> sort_index_reverse(const std::vector<double>& key) {
    std::vector<int> idx(key.size());
    std::iota(idx.begin(), idx.end(), 0);
    std::stable_sort(idx.begin(), idx.end(), [&](int a, int b) { return key[a] > key[b]; });
    return idx;
}

// Y(:, 0:p) = Xw(:, 0:k) Zc(0:k, 0:p) on the device; Zc given on the host as complex doubles
int device_combine(lkb_basis_s* Xw, int k, const std::vector<cd>& Zc, int ldz, int p, void* Yd, int64_t ldy) {
    lkb_ctx_s* c = Xw->ctx;
    const int kind = Xw->kind;
    const size_t es = kind_size(kind);
    LKB_TRY(ensure_hstage(c, (size_t)k * p * es + 4096));
    LKB_TRY(ensure_coefd(c, std::max((size_t)k * p * es, (size_t)4096)));
    LKB_CUDA(cudaStreamSynchronize(c->stream));
    for (int q = 0; q < p; ++q) for (int i = 0; i < k; ++i) store_kind(kind, c->hstage, (size_t)i + (size_t)k * q, Zc[i + (size_t)ldz * q]);
    LKB_CUDA(cudaMemcpyAsync(c->coefd, c->hstage, (size_t)k * p * es, cudaMemcpyHostToDevice, c->stream));
    prof_launch(c, PC_OTHER, 1, [&] { launch_basis_gemm(kind, c->stream, Xw->d, Xw->ld, k, c->coefd, k, p, Yd, ldy, Xw->n, c->sms); });
    return check_launch(c, "basis_gemm");
}

// Two pinned host slots + events for the "collect step k, enqueue step k+1 speculatively, then run the host LAPACK
// of step k" pipeline shared by eigs / eighs / svds.  A speculative step's copy into a slot may still be in flight when
// the solver returns: the destructor waits for the stream before it frees the slots.
struct StepSlots {
    cudaStream_t stream;
    void* slot[2] = {nullptr, nullptr};
    cudaEvent_t ev[2] = {nullptr, nullptr};
    explicit StepSlots(cudaStream_t s) : stream(s) {}
    StepSlots(const StepSlots&) = delete;
    StepSlots& operator=(const StepSlots&) = delete;
    ~StepSlots() {
        cudaStreamSynchronize(stream);
        for (int q = 0; q < 2; ++q) { if (slot[q]) cudaFreeHost(slot[q]); if (ev[q]) cudaEventDestroy(ev[q]); }
    }
    int init(size_t bytes) {
        for (int q = 0; q < 2; ++q)
            if (cudaMallocHost(&slot[q], bytes) != cudaSuccess || cudaEventCreateWithFlags(&ev[q], cudaEventDisableTiming) != cudaSuccess) {
                set_error("pinned staging allocation failed"); return LKB_ERR_ALLOC;
            }
        return 0;
    }
};

int start_vector(lkb_basis_s* Xw, lkb_vec_t x0) {
    lkb_ctx_s* c = Xw->ctx;
    const int kind = Xw->kind;
    LKB_TRY(lkb_basis_zero(Xw, 0, Xw->ncols));
    if (x0) {
        if (x0->n != Xw->n || x0->kind != kind) { set_error("x0: size/kind mismatch"); return LKB_ERR_ARG; }
        prof_launch(c, PC_OTHER, 1, [&] { launch_axpby(kind, c->stream, Scalar{1, 0}, x0->d, Scalar{0, 0}, Xw->d, Xw->n, c->sms); });   // copy(Xwrk(1), x0)
    } else {
        prof_launch(c, PC_OTHER, 1, [&] { launch_fill(kind, c->stream, Xw->d, Xw->n, Xw->row0, LKB_DIST_NORMAL, next_seed(c), c->sms); });   // rand(.true.)
    }
    double nrm = 0;
    LKB_TRY(vec_norm_sync(c, kind, Xw->d, Xw->n, &nrm));
    prof_launch(c, PC_OTHER, 1, [&] { launch_scal(kind, c->stream, Scalar{1.0 / nrm, 0}, Xw->d, Xw->n, c->sms); });
    return check_launch(c, "start vector");
}

}  // namespace

extern "C" {

int lkb_set_lapack(const char* path, const char* prefix, const char* suffix) {
    if (!path) return LKB_ERR_ARG;
    return lapack_open(path, prefix ? prefix : "", suffix ? suffix : "_");
}

// krylov_schur(n, X, H, median_selector): BaseKrylov.fypp:782-834 + IterativeSolvers.fypp:1136-1141
int lkb_krylov_schur(lkb_basis_t X, void* H, int ldh, int kdim, int32_t* nkeep) {
    if (!X || !H || !nkeep || kdim < 1 || X->ncols < kdim + 1 || ldh < kdim + 1) { set_error("krylov_schur: bad arguments"); return LKB_ERR_ARG; }
    LKB_TRY(lapack_ready());
    lkb_ctx_s* c = X->ctx;
    const int kind = X->kind;
    const bool cplx = kind_cplx(kind);
    const size_t es = kind_size(kind);
    const int k = kdim;
    const bool sp = (kind == KS || kind == KC);
    std::vector<cd> Hk((size_t)k * k), Zc, Tc;
    for (int j = 0; j < k; ++j) for (int i = 0; i < k; ++i) Hk[i + (size_t)k * j] = load_kind(kind, H, (size_t)i + (size_t)ldh * j);
    LKB_TRY(sp ? host_schur_select_t<float>(cplx, k, Hk, Tc, Zc, nkeep) : host_schur_select_t<double>(cplx, k, Hk, Tc, Zc, nkeep));
    {   // rank 0's Schur data is authoritative (see bcast_host)
        LKB_TRY(bcast_host(c, Zc.data(), Zc.size() * sizeof(cd)));
        LKB_TRY(bcast_host(c, Tc.data(), Tc.size() * sizeof(cd)));
        int32_t nk0 = *nkeep;
        LKB_TRY(bcast_host(c, &nk0, sizeof(nk0)));
        *nkeep = nk0;
    }
    const int nk = *nkeep;
    // basis: X(:n) <- X(:kdim) Z(:, :n) ; X(n+1) <- X(kdim+1) ; X(n+2:) = 0
    if (nk > 0) {
        // The update is row-local, so it is done in place one row chunk at a time through a bounded
        // staging buffer (<= 1 GB) instead of a second n x nk basis (C3: 64 GB at n = 134M).
        LKB_TRY(ensure_hstage(c, (size_t)k * nk * es + 4096));
        LKB_TRY(ensure_coefd(c, std::max((size_t)k * nk * es, (size_t)4096)));
        LKB_CUDA(cudaStreamSynchronize(c->stream));
        for (int q = 0; q < nk; ++q) for (int i = 0; i < k; ++i) store_kind(kind, c->hstage, (size_t)i + (size_t)k * q, Zc[i + (size_t)k * q]);
        LKB_CUDA(cudaMemcpyAsync(c->coefd, c->hstage, (size_t)k * nk * es, cudaMemcpyHostToDevice, c->stream));
        int64_t chunk = (int64_t)(((size_t)1 << 30) / ((size_t)nk * es));
        chunk = std::max<int64_t>(4096, (chunk / 4096) * 4096);
        chunk = std::min<int64_t>(chunk, ((X->n + 4095) / 4096) * 4096);
        DevBuf tmp(c);
        LKB_TRY(tmp.alloc((size_t)chunk * nk * es));
        int r = 0;
        for (int64_t r0 = 0; r0 < X->n && r == 0; r0 += chunk) {
            const int64_t rows = std::min<int64_t>(chunk, X->n - r0);
            prof_launch(c, PC_OTHER, 1, [&] { launch_basis_gemm(kind, c->stream, (char*)X->d + (size_t)r0 * es, X->ld, k, c->coefd, k, nk, tmp.p, chunk, rows, c->sms); });
            r = check_launch(c, "basis_gemm");
            if (r == 0 && cudaMemcpy2DAsync((char*)X->d + (size_t)r0 * es, (size_t)X->ld * es, tmp.p, (size_t)chunk * es,
                                            (size_t)rows * es, nk, cudaMemcpyDeviceToDevice, c->stream) != cudaSuccess) r = LKB_ERR_CUDA;
        }
        cudaStreamSynchronize(c->stream);
        if (r) return r;
    }
    LKB_CUDA(cudaMemcpyAsync(col_ptr(X, nk), col_ptr(X, k), (size_t)X->n * es, cudaMemcpyDeviceToDevice, c->stream));
    if (nk + 1 < X->ncols) LKB_TRY(lkb_basis_zero(X, nk + 1, X->ncols - nk - 1));
    // Hessenberg: H(:k,:) = T ; b = H(k+1,:) Z ; H(n+1,:) = b ; H(n+2:,:) = 0 ; H(:, n+1:) = 0
    std::vector<cd> b(k, cd(0));
    for (int j = 0; j < k; ++j) for (int i = 0; i < k; ++i) b[j] += load_kind(kind, H, (size_t)k + (size_t)ldh * i) * Zc[i + (size_t)k * j];
    for (int j = 0; j < k; ++j) for (int i = 0; i < k; ++i) store_kind(kind, H, (size_t)i + (size_t)ldh * j, Tc[i + (size_t)k * j]);
    for (int j = 0; j < k; ++j) store_kind(kind, H, (size_t)nk + (size_t)ldh * j, b[j]);
    for (int j = 0; j < k; ++j) for (int i = nk + 1; i < k + 1; ++i) store_kind(kind, H, (size_t)i + (size_t)ldh * j, cd(0));
    for (int j = nk; j < k; ++j) for (int i = 0; i < k + 1; ++i) store_kind(kind, H, (size_t)i + (size_t)ldh * j, cd(0));
    return 0;
}

int lkb_eigs(lkb_op_t A, lkb_basis_t X, int nev, double* eigvals, double* residuals, int32_t* info, lkb_vec_t x0,
             int32_t kdim, double tolerance, int32_t transpose) {
    if (!A || !X || !eigvals || !residuals || !info || nev < 1 || X->ncols < nev) { set_error("eigs: bad arguments"); return LKB_ERR_ARG; }
    LKB_TRY(lapack_ready());
    lkb_ctx_s* c = X->ctx;
    const int kind = X->kind;
    const bool cplx = kind_cplx(kind);
    const size_t es = kind_size(kind);
    const int kd = kdim > 0 ? kdim : 4 * nev;
    const double tol = tolerance >= 0 ? tolerance : rtol_of(kind);
    BasisOwner Xw;
    LKB_TRY(lkb_basis_create(c, kind, X->n, X->n_global, X->row0, kd + 1, Xw.out()));
    LKB_TRY(start_vector(Xw, x0));
    const int ldh = kd + 1;
    std::vector<char> H((size_t)ldh * kd * es, 0);
    std::vector<cd> vals, vecs, Hc((size_t)kd * kd);
    std::vector<double> res(kd, 0.0);
    int kstart = 1, conv = 0, niter = 0, k = 1;
    auto load_Hc = [&](int kk) {
        for (int j = 0; j < kk; ++j) for (int i = 0; i < kk; ++i) Hc[i + (size_t)kd * j] = load_kind(kind, H.data(), (size_t)i + (size_t)ldh * j);
    };
    // Host/device overlap (SURVEY 8f rank 3): the per-step geev of the reference
    // (IterativeSolvers.fypp:1062-1066) costs up to ~14 ms at k = 128, longer than a device step at C2
    // size.  Step k+1 is therefore enqueued speculatively BEFORE the host decomposes H_k; Xwrk and H
    // are internal work arrays and the post-processing only reads their first k columns, so a
    // speculative step that turns out to be unnecessary (convergence at k) is simply discarded.
    const bool tr = transpose != 0;
    const double atolk = atol_of(kind);
    StepSlots ss(c->stream);
    if (ss.init((size_t)ldh * es + 256)) { set_error("eigs: pinned staging allocation failed"); return LKB_ERR_ALLOC; }
    auto enqueue_step = [&](int kk) -> int {
        LKB_TRY(arnoldi_enqueue(A, Xw, kk, kk, atolk, tr));
        LKB_TRY(krylov_fetch_async(c, kind, Xw->ncols, kk, kk, ss.slot[kk & 1]));
        LKB_CUDA(cudaEventRecord(ss.ev[kk & 1], c->stream));
        return 0;
    };
    int restarts = 0;
    while (conv < nev) {
        int inflight = 0;                              // highest step already enqueued
        for (k = kstart; k <= kd; ++k) {
            int32_t ainfo = 0;
            if (inflight < k) { LKB_TRY(enqueue_step(k)); inflight = k; }
            LKB_CUDA(cudaEventSynchronize(ss.ev[k & 1]));
            LKB_TRY(arnoldi_collect(A, Xw, H.data(), ldh, &ainfo, k, k, tr, ss.slot[k & 1]));
            if (ainfo == 0 && k < kd) { LKB_TRY(enqueue_step(k + 1)); inflight = k + 1; }   // speculative
            load_Hc(k);
            LKB_TRY(host_eig(kind, k, Hc, kd, vals, vecs));
            const cd beta = load_kind(kind, H.data(), (size_t)k + (size_t)ldh * (k - 1));
            std::fill(res.begin(), res.end(), 0.0);
            for (int i = 0; i < k; ++i) {
                double alpha;
                if (cplx) alpha = std::abs(vecs[(k - 1) + (size_t)k * i]);
                else if (vals[i].imag() > 0) alpha = hypot(vecs[(k - 1) + (size_t)k * i].real(), vecs[(k - 1) + (size_t)k * (i + 1)].real());
                else if (vals[i].imag() < 0) alpha = hypot(vecs[(k - 1) + (size_t)k * (i - 1)].real(), vecs[(k - 1) + (size_t)k * i].real());
                else alpha = fabs(vecs[(k - 1) + (size_t)k * i].real());
                res[i] = std::abs(beta) * alpha;
            }
            niter++;
            LKB_TRY(bcast_host(c, res.data(), (size_t)k * sizeof(double)));
            conv = 0; for (int i = 0; i < k; ++i) conv += res[i] < tol;
            if (c->write_intermediate) {                          // write_results_c(eigs_output, ...)  (:1091)
                // LITERAL side effect: write_results sorts its `res` argument IN PLACE (`call sort_index(res, indices)`, intent(inout),
                // IterativeSolvers.fypp:907), so with write_intermediate (the reference's DEFAULT for eigs) residuals_wrk(:k) is left
                // in ascending order and the residuals returned at the end are entries of that sorted table.  The reference does this
                // on the I/O rank only (its other ranks keep the unsorted table); here every rank applies the same sort.
                std::vector<double> rr(res.begin(), res.begin() + k);
                if (c->rank == 0) {
                    std::vector<double> vv(2 * (size_t)k);
                    for (int i = 0; i < k; ++i) { vv[2 * i] = vals[i].real(); vv[2 * i + 1] = vals[i].imag(); }
                    (void)lkb_write_results("eigs_output.txt", 1, vv.data(), rr.data(), k, tol);   // rr is sorted even if the file cannot be written;
                                                                                                  // an I/O failure on one rank must not desynchronise the ranks
                } else {
                    std::stable_sort(rr.begin(), rr.end());
                }
                std::copy(rr.begin(), rr.end(), res.begin());
            }
            if (conv >= nev) {
                // a speculative step k+1 may still be running: it is discarded (never collected, so the
                // operator's matvec counter does not include it); the sync below waits for it
                break;
            }
        }
        // LITERAL control flow (IterativeSolvers.fypp:1088-1099): `exit arnoldi_factorization` leaves only the inner loop, so the
        // reference runs krylov_schur once more AFTER convergence, before `do while (conv < nev)` is re-evaluated, and then
        // post-processes the restarted H and basis while `res` still holds the pre-restart residuals.  Reproduced as is.
        const int converged_at = conv >= nev ? k : 0;
        if (converged_at && converged_at < kd) {
            // a speculative step k+1 wrote X(k+2); in the reference the columns beyond k+1 are still zero at this point
            LKB_CUDA(cudaStreamSynchronize(c->stream));
            LKB_TRY(lkb_basis_zero(Xw, converged_at + 1, kd - converged_at));
        }
        // Krylov-Schur restart (IterativeSolvers.fypp:1096-1100); note the loop index is kd+1 here unless converged
        int32_t nk = 0;
        LKB_TRY(lkb_krylov_schur(Xw, H.data(), ldh, kd, &nk));
        kstart = nk + 1;
        k = converged_at ? converged_at : kd + 1;
        if (++restarts > 2000) { set_error("eigs: no convergence after 2000 Krylov-Schur restarts"); return LKB_ERR_ARG; }
    }
    LKB_CUDA(cudaStreamSynchronize(c->stream));
    // post-process (:1108-1132)
    k = std::min(k, kd);
    load_Hc(k);
    LKB_TRY(host_eig(kind, k, Hc, kd, vals, vecs));
    LKB_TRY(bcast_host(c, vals.data(), vals.size() * sizeof(cd)));
    LKB_TRY(bcast_host(c, vecs.data(), vecs.size() * sizeof(cd)));
    std::vector<double> av(kd, 0.0);
    for (int i = 0; i < k; ++i) av[i] = std::abs(vals[i]);
    std::vector<int> idx = sort_index_reverse(av);
    std::vector<cd> Y((size_t)k * nev, cd(0));
    for (int i = 0; i < nev; ++i) {
        const int s = idx[i];
        cd v = s < k ? vals[s] : cd(0);
        eigvals[2 * i] = v.real(); eigvals[2 * i + 1] = v.imag();
        residuals[i] = res[s];
        if (s < k) for (int j = 0; j < k; ++j) Y[j + (size_t)k * i] = vecs[j + (size_t)k * s];
    }
    LKB_TRY(device_combine(Xw, k, Y, k, nev, X->d, X->ld));
    LKB_TRY(lkb_sync(c));
    *info = niter;
    return 0;
}

int lkb_eighs(lkb_op_t A, lkb_basis_t X, int nev, double* eigvals, double* residuals, int32_t* info, lkb_vec_t x0,
              int32_t kdim, double tolerance) {
    if (!A || !X || !eigvals || !residuals || !info || nev < 1 || X->ncols < nev) { set_error("eighs: bad arguments"); return LKB_ERR_ARG; }
    LKB_TRY(lapack_ready());
    lkb_ctx_s* c = X->ctx;
    const int kind = X->kind;
    const bool cplx = kind_cplx(kind);
    const size_t es = kind_size(kind);
    const int kd = kdim > 0 ? kdim : 4 * nev;
    const double tol = tolerance >= 0 ? tolerance : rtol_of(kind);
    BasisOwner Xw;
    LKB_TRY(lkb_basis_create(c, kind, X->n, X->n_global, X->row0, kd + 1, Xw.out()));
    LKB_TRY(start_vector(Xw, x0));
    const int ldt = kd + 1;
    std::vector<char> T((size_t)ldt * kd * es, 0);
    std::vector<double> ev(kd, 0.0), res(kd, 0.0);
    std::vector<cd> vecs((size_t)kd * kd, cd(0)), Tk, vk;
    const bool sp = (kind == KS || kind == KC);
    int k = 1, conv = 0;
    // Host/device overlap as in eigs: step k+1 is enqueued speculatively before the host runs syev / heev on T_k
    // (eighs.fypp:84-100); Xwrk and T are internal work arrays, a speculative step past convergence is discarded.
    StepSlots ss(c->stream);
    LKB_TRY(ss.init((size_t)ldt * es + 256));
    const double atolk = atol_of(kind);
    auto enqueue_step = [&](int kk) -> int {
        LKB_TRY(lanczos_enqueue(A, Xw, kk, kk, atolk));
        LKB_TRY(krylov_fetch_async(c, kind, ldt, kk, kk, ss.slot[kk & 1]));
        LKB_CUDA(cudaEventRecord(ss.ev[kk & 1], c->stream));
        return 0;
    };
    int inflight = 0;
    for (k = 1; k <= kd; ++k) {
        int32_t linfo = 0;
        if (inflight < k) { LKB_TRY(enqueue_step(k)); inflight = k; }
        LKB_CUDA(cudaEventSynchronize(ss.ev[k & 1]));
        LKB_TRY(lanczos_collect(A, Xw, T.data(), ldt, &linfo, k, k, ss.slot[k & 1]));
        if (linfo == 0 && k < kd) { LKB_TRY(enqueue_step(k + 1)); inflight = k + 1; }      // speculative
        std::fill(ev.begin(), ev.end(), 0.0); std::fill(vecs.begin(), vecs.end(), cd(0));
        Tk.assign((size_t)k * k, cd(0));
        for (int j = 0; j < k; ++j) for (int i = 0; i < k; ++i) Tk[i + (size_t)k * j] = load_kind(kind, T.data(), (size_t)i + (size_t)ldt * j);
        LKB_TRY(sp ? host_eigh_t<float>(cplx, k, Tk, ev.data(), vk) : host_eigh_t<double>(cplx, k, Tk, ev.data(), vk));
        for (int j = 0; j < k; ++j) for (int i = 0; i < k; ++i) vecs[i + (size_t)kd * j] = vk[i + (size_t)k * j];
        const cd beta = load_kind(kind, T.data(), (size_t)k + (size_t)ldt * (k - 1));
        std::fill(res.begin(), res.end(), 0.0);
        for (int i = 0; i < k; ++i) res[i] = std::abs(beta * vecs[(k - 1) + (size_t)kd * i]);
        LKB_TRY(bcast_host(c, res.data(), (size_t)k * sizeof(double)));
        conv = 0; for (int i = 0; i < k; ++i) conv += res[i] < tol;
        if (c->write_intermediate) {                              // write_results_r(eighs_output, ...)  (eighs.fypp:99)
            std::vector<double> rr(res.begin(), res.begin() + k); // sorts the residual table in place, see lkb_eigs
            if (c->rank == 0) (void)lkb_write_results("eighs_output.txt", 0, ev.data(), rr.data(), k, tol);
            else std::stable_sort(rr.begin(), rr.end());
            std::copy(rr.begin(), rr.end(), res.begin());
        }
        if (conv >= nev) break;
    }
    LKB_CUDA(cudaStreamSynchronize(c->stream));     // a discarded speculative step may still run
    LKB_TRY(bcast_host(c, ev.data(), ev.size() * sizeof(double)));
    LKB_TRY(bcast_host(c, vecs.data(), vecs.size() * sizeof(cd)));
    std::vector<int> idx = sort_index_reverse(ev);        // over all kdim_ entries, zero padding included (eighs.fypp:106-107)
    k = std::min(k, kd);
    std::vector<cd> Y((size_t)k * nev, cd(0));
    for (int i = 0; i < nev; ++i) {
        const int s = idx[i];
        eigvals[i] = ev[s]; residuals[i] = res[s];
        for (int j = 0; j < k; ++j) Y[j + (size_t)k * i] = vecs[j + (size_t)kd * s];
    }
    LKB_TRY(device_combine(Xw, k, Y, k, nev, X->d, X->ld));
    LKB_TRY(lkb_sync(c));
    *info = k;
    return 0;
}

int lkb_svds(lkb_op_t A, lkb_basis_t U, double* S, lkb_basis_t V, int nsv, double* residuals, int32_t* info,
             lkb_vec_t u0, int32_t kdim, double tolerance) {
    if (!A || !U || !V || !S || !residuals || !info || nsv < 1 || U->ncols < nsv || V->ncols < nsv) { set_error("svds: bad arguments"); return LKB_ERR_ARG; }
    LKB_TRY(lapack_ready());
    lkb_ctx_s* c = U->ctx;
    const int kind = U->kind;
    const bool cplx = kind_cplx(kind);
    const size_t es = kind_size(kind);
    const int kd = kdim > 0 ? kdim : 4 * nsv;
    const double tol = tolerance >= 0 ? tolerance : rtol_of(kind);
    BasisOwner Uw, Vw;
    LKB_TRY(lkb_basis_create(c, kind, U->n, U->n_global, U->row0, kd + 1, Uw.out()));
    LKB_TRY(lkb_basis_create(c, kind, V->n, V->n_global, V->row0, kd + 1, Vw.out()));
    LKB_TRY(start_vector(Uw, u0));
    const int ldb = kd + 1;
    std::vector<char> B((size_t)ldb * kd * es, 0);
    std::vector<double> sv(kd, 0.0), res(kd, 0.0);
    std::vector<cd> umat((size_t)kd * kd), vmat((size_t)kd * kd), Bk, uk, vk;
    const bool sp = (kind == KS || kind == KC);
    *info = 0;
    int k = 1, conv = 0;
    // speculative step k+1 overlapped with the host gesdd of B_k (svd_solvers.fypp:85-101), as in eigs / eighs
    StepSlots ss(c->stream);
    LKB_TRY(ss.init((size_t)ldb * es + 256));
    auto enqueue_step = [&](int kk) -> int {
        LKB_TRY(bidiag_enqueue(A, Uw, Vw, kk, kk, tol));                    // tol = solver tolerance (svd_solvers.fypp:82)
        LKB_TRY(krylov_fetch_async(c, kind, ldb, kk, kk, ss.slot[kk & 1]));
        LKB_CUDA(cudaEventRecord(ss.ev[kk & 1], c->stream));
        return 0;
    };
    int inflight = 0;
    for (k = 1; k <= kd; ++k) {
        int32_t binfo = 0;
        if (inflight < k) { LKB_TRY(enqueue_step(k)); inflight = k; }
        LKB_CUDA(cudaEventSynchronize(ss.ev[k & 1]));
        LKB_TRY(bidiag_collect(A, Uw, B.data(), ldb, &binfo, k, k, ss.slot[k & 1]));
        if (binfo == 0 && k < kd) { LKB_TRY(enqueue_step(k + 1)); inflight = k + 1; }      // speculative
        std::fill(sv.begin(), sv.end(), 0.0);
        std::fill(umat.begin(), umat.end(), cd(0)); std::fill(vmat.begin(), vmat.end(), cd(0));
        Bk.assign((size_t)k * k, cd(0));
        for (int j = 0; j < k; ++j) for (int i = 0; i < k; ++i) Bk[i + (size_t)k * j] = load_kind(kind, B.data(), (size_t)i + (size_t)ldb * j);
        LKB_TRY(sp ? host_svd_t<float>(cplx, k, Bk, sv.data(), uk, vk) : host_svd_t<double>(cplx, k, Bk, sv.data(), uk, vk));
        for (int j = 0; j < k; ++j) for (int i = 0; i < k; ++i) {
            umat[i + (size_t)kd * j] = uk[i + (size_t)k * j];
            vmat[i + (size_t)kd * j] = vk[i + (size_t)k * j];
        }
        const cd beta = load_kind(kind, B.data(), (size_t)k + (size_t)ldb * (k - 1));
        std::fill(res.begin(), res.end(), 0.0);
        for (int i = 0; i < k; ++i) res[i] = std::abs(beta * vmat[(k - 1) + (size_t)kd * i]);
        LKB_TRY(bcast_host(c, res.data(), (size_t)k * sizeof(double)));
        conv = 0; for (int i = 0; i < k; ++i) conv += res[i] < tol;
        if (c->write_intermediate) {                              // write_results_r(svds_output, ...)  (svd_solvers.fypp:100)
            std::vector<double> rr(res.begin(), res.begin() + k); // sorts the residual table in place, see lkb_eigs
            if (c->rank == 0) (void)lkb_write_results("svds_output.txt", 0, sv.data(), rr.data(), k, tol);
            else std::stable_sort(rr.begin(), rr.end());
            std::copy(rr.begin(), rr.end(), res.begin());
        }
        if (conv >= nsv) break;
    }
    LKB_CUDA(cudaStreamSynchronize(c->stream));
    LKB_TRY(bcast_host(c, sv.data(), sv.size() * sizeof(double)));
    LKB_TRY(bcast_host(c, umat.data(), umat.size() * sizeof(cd)));
    LKB_TRY(bcast_host(c, vmat.data(), vmat.size() * sizeof(cd)));
    for (int i = 0; i < nsv; ++i) { S[i] = sv[i]; residuals[i] = res[i]; }
    k = std::min(k, kd);
    *info = k;
    std::vector<cd> Yu((size_t)k * nsv), Yv((size_t)k * nsv);
    for (int i = 0; i < nsv; ++i) for (int j = 0; j < k; ++j) {
        Yu[j + (size_t)k * i] = umat[j + (size_t)kd * i];
        Yv[j + (size_t)k * i] = vmat[j + (size_t)kd * i];
    }
    LKB_TRY(device_combine(Uw, k, Yu, k, nsv, U->d, U->ld));
    LKB_TRY(device_combine(Vw, k, Yv, k, nsv, V->d, V->ld));
    LKB_TRY(lkb_sync(c));
    return 0;
}

}  // extern "C"
