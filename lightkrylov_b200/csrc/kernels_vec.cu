// kernels_vec.cu -- single-vector TBPs of the device abstract_vector (axpby, scal, rand, ...)
// and the O(kdim) scalar kernels that keep the Hessenberg / tridiagonal / bidiagonal update and
// the breakdown decision on the device, so a whole factorisation can run as one CUDA graph.
//
// Reference semantics: src/AbstractTypes/AbstractVectors.fypp:295-381 (deferred TBPs),
// :424-460 (norm/sub/chsgn), src/Krylov/qr.fypp:137-164, arnoldi.fypp:59-71,
// lanczos.fypp:29-40, golub_kahan.fypp:37-59.
#include "lkb_kernels.h"
#include "lkb_rng.h"
#include "lkb_p2p.cuh"
#include "lkb_step.cuh"
#include "lkb_reduce.cuh"

namespace lkb {

static inline int ew_grid(int64_t npk, int sms) {
    int64_t nb = (npk + 255) / 256;
    if (nb < 1) nb = 1;
    if (nb > (int64_t)sms * 8) nb = (int64_t)sms * 8;
    return (int)nb;
}

// y = alpha*x + beta*y ; beta == 0 => overwrite without reading y (copy semantics,
// AbstractVectors.fypp:717-723: `copy` is axpby(1, from, 0) on an intent(out) target).
template <int K, bool BETA0>
__global__ void __launch_bounds__(256)
k_axpby(typename Tr<K>::E alpha, const typename Tr<K>::E* __restrict__ x, typename Tr<K>::E beta,
        typename Tr<K>::E* __restrict__ y, int64_t n)
{
    using E = typename Tr<K>::E;
    constexpr int EPP = Tr<K>::EPP;
    using P = Pack<E, EPP>;
    const int64_t npk = n / EPP;
    for (int64_t pk = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; pk < npk; pk += (int64_t)gridDim.x * blockDim.x) {
        const P xv = ld_pack_nc<P>(x + pk * EPP);
        P yv;
        if (!BETA0) yv = ld_pack<P>(y + pk * EPP);
#pragma unroll
        for (int e = 0; e < EPP; ++e) {
            E r = mul_v(alpha, xv.v[e]);
            if (!BETA0) r = add_v(r, mul_v(beta, yv.v[e]));
            yv.v[e] = r;
        }
        st_pack(y + pk * EPP, yv);
    }
    if (blockIdx.x == 0 && threadIdx.x == 0)
        for (int64_t t = npk * EPP; t < n; ++t) {
            E r = mul_v(alpha, x[t]);
            if (!BETA0) r = add_v(r, mul_v(beta, y[t]));
            y[t] = r;
        }
}

// y += sgn * (*alpha) * x, alpha on the device in W precision
template <int K>
__global__ void __launch_bounds__(256)
k_axpy_dev(const typename Tr<K>::W* __restrict__ alpha_dev, double sgn, const typename Tr<K>::E* __restrict__ x,
           typename Tr<K>::E* __restrict__ y, int64_t n, const int* __restrict__ flags)
{
    using E = typename Tr<K>::E;
    constexpr int EPP = Tr<K>::EPP;
    using P = Pack<E, EPP>;
    if (flags && flags[F_STOP]) return;
    E alpha; narrow(*alpha_dev, alpha);
    alpha = rscale(alpha, (typename Tr<K>::Rl)sgn);
    const int64_t npk = n / EPP;
    for (int64_t pk = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; pk < npk; pk += (int64_t)gridDim.x * blockDim.x) {
        const P xv = ld_pack_nc<P>(x + pk * EPP);
        P yv = ld_pack<P>(y + pk * EPP);
#pragma unroll
        for (int e = 0; e < EPP; ++e) fmacc(yv.v[e], xv.v[e], alpha);
        st_pack(y + pk * EPP, yv);
    }
    if (blockIdx.x == 0 && threadIdx.x == 0)
        for (int64_t t = npk * EPP; t < n; ++t) { E a = y[t]; fmacc(a, x[t], alpha); y[t] = a; }
}

template <int K>
__global__ void __launch_bounds__(256)
k_scal(typename Tr<K>::E alpha, typename Tr<K>::E* __restrict__ x, int64_t n)
{
    using E = typename Tr<K>::E;
    constexpr int EPP = Tr<K>::EPP;
    using P = Pack<E, EPP>;
    const int64_t npk = n / EPP;
    for (int64_t pk = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; pk < npk; pk += (int64_t)gridDim.x * blockDim.x) {
        P xv = ld_pack<P>(x + pk * EPP);
#pragma unroll
        for (int e = 0; e < EPP; ++e) xv.v[e] = mul_v(xv.v[e], alpha);
        st_pack(x + pk * EPP, xv);
    }
    if (blockIdx.x == 0 && threadIdx.x == 0)
        for (int64_t t = npk * EPP; t < n; ++t) x[t] = mul_v(x[t], alpha);
}

// x *= *inv (real scalar on the device).  Gate: !scaled && (!stop || info == kstep) && !refill.
// flags[F_SCALED] is raised by k_multiaxpy_fin when it already normalised the vector (the usual case): this
// kernel is then an empty launch.  With a P2P halo descriptor (hp.he > 0, multi-GPU stencil inside a Krylov
// loop) the finished boundary rows are also stored into the neighbours' halo buffers and the epoch is
// published, exactly as k_multiaxpy_fin does on its fast path -- whichever kernel finishes the vector pushes.
template <int K>
__global__ void __launch_bounds__(256)
k_scale_dev(typename Tr<K>::E* __restrict__ x, int64_t n, const double* __restrict__ inv_dev,
            const int* __restrict__ flags, int kstep, const HaloP2P hp)
{
    using E = typename Tr<K>::E;
    using Rl = typename Tr<K>::Rl;
    constexpr int EPP = Tr<K>::EPP;
    using P = Pack<E, EPP>;
    pdl_wait();
    pdl_trigger();
    if (flags) {
        if (flags[F_SCALED]) return;
        if (flags[F_STOP] && flags[F_INFO] != kstep) return;
        if (flags[F_REFILL]) return;
    }
    const Rl inv = (Rl)(*inv_dev);
    const bool push = hp.he > 0;
    if (inv == (Rl)1 && !push) return;
    const unsigned ep = push ? *hp.epoch + 1u : 0u;
    const size_t par = (size_t)(ep & 1u) * 2 * hp.side_bytes;
    E* push_lo = (push && hp.lo_region) ? reinterpret_cast<E*>(hp.lo_region + hp.data_off + par + hp.side_bytes) : nullptr;
    E* push_hi = (push && hp.hi_region) ? reinterpret_cast<E*>(hp.hi_region + hp.data_off + par) : nullptr;
    const int64_t hi0 = n - hp.he;
    const int64_t npk = n / EPP;
    for (int64_t pk = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; pk < npk; pk += (int64_t)gridDim.x * blockDim.x) {
        const int64_t off = pk * EPP;
        P xv = ld_pack<P>(x + off);
#pragma unroll
        for (int e = 0; e < EPP; ++e) xv.v[e] = rscale(xv.v[e], inv);
        st_pack(x + off, xv);
        if (push_lo && off < hp.he) {
#pragma unroll
            for (int e = 0; e < EPP; ++e) if (off + e < hp.he) push_lo[off + e] = xv.v[e];
        }
        if (push_hi && off + EPP > hi0) {
#pragma unroll
            for (int e = 0; e < EPP; ++e) if (off + e >= hi0) push_hi[off + e - hi0] = xv.v[e];
        }
    }
    if (blockIdx.x == 0 && threadIdx.x == 0)
        for (int64_t t = npk * EPP; t < n; ++t) {
            const E a = rscale(x[t], inv);
            x[t] = a;
            if (push_lo && t < hp.he) push_lo[t] = a;
            if (push_hi && t >= hi0) push_hi[t - hi0] = a;
        }
    if (!push) return;
    __shared__ bool is_last;
    __threadfence_system();
    __syncthreads();
    if (threadIdx.x == 0) is_last = (atomicAdd(hp.ticket, 1u) == gridDim.x - 1u);
    __syncthreads();
    if (is_last && threadIdx.x == 0) {
        __threadfence_system();
        if (hp.lo_region) st_volatile_u32(reinterpret_cast<unsigned*>(hp.lo_region + 128), ep);
        if (hp.hi_region) st_volatile_u32(reinterpret_cast<unsigned*>(hp.hi_region), ep);
        *hp.ticket = 0u;
        *hp.epoch = ep;
    }
}

template <int K>
__global__ void __launch_bounds__(256)
k_copy_gated(const typename Tr<K>::E* __restrict__ src, typename Tr<K>::E* __restrict__ dst, int64_t n, const int* __restrict__ flags)
{
    if (flags && flags[F_STOP]) return;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) dst[i] = src[i];
}

template <int K>
__global__ void __launch_bounds__(256)
k_fill(typename Tr<K>::E* __restrict__ x, int64_t n, int64_t row0, int dist, uint64_t seed_mixed)
{
    using E = typename Tr<K>::E;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        const uint64_t g = (uint64_t)(row0 + i);
        Scalar s;
        s.re = dist == 0 ? rng_normal(seed_mixed, g, 0) : rng_uniform(seed_mixed, g, 0);
        s.im = 0.0;
        if (Tr<K>::cplx) s.im = dist == 0 ? rng_normal(seed_mixed, g, 1) : rng_uniform(seed_mixed, g, 1);
        E v; from_scalar(s, v);
        x[i] = v;
    }
}

// Column update of H / T / B after the second CGS pass; one CTA.  (Only on the paths that do not end in
// k_multiaxpy_fin: j = 0, NCCL allreduce, host-driven loops.)
//   hcol[0..j) = c1 + c2 (if c1),  beta = sqrt(|nrm2|),  hcol[j] = beta (or 0), inv = 1/beta
template <int K>
__global__ void k_update(const typename Tr<K>::W* __restrict__ c1, const typename Tr<K>::W* __restrict__ c2, int j,
                         const typename Tr<K>::W* __restrict__ nrm2, typename Tr<K>::E* __restrict__ hcol,
                         double tol, double atol, double* __restrict__ inv_dev, int* __restrict__ flags,
                         int kstep, int mode)
{
    using E = typename Tr<K>::E;
    using W = typename Tr<K>::W;
    if (flags[F_STOP]) return;
    if (c1 && hcol)
        for (int i = threadIdx.x; i < j; i += blockDim.x) {
            W a = c1[i];
            if (c2) wadd(a, c2[i]);
            narrow(a, hcol[i]);
        }
    if (threadIdx.x == 0) {
        flags[F_SCALED] = 0;                  // the k_scale_dev that follows does the scaling
        step_decide<K>(sqrt(fabs(wreal(nrm2[0]))), hcol, j, tol, atol, inv_dev, flags, kstep, mode);
    }
}

__global__ void k_gsinfo(const double* __restrict__ ww, double atol, int* __restrict__ flags) {
    if (flags[F_STOP]) return;
    flags[F_GSINFO] = (sqrt(fabs(ww[0])) < atol) ? 1 : 0;
}

template <int K>
__global__ void k_narrow(const typename Tr<K>::W* src, typename Tr<K>::E* dst, int n, const int* flags) {
    if (flags && flags[F_STOP]) return;
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) narrow(src[i], dst[i]);
}

// ------------------------------------------------------------------------------------------
// Conjugate gradient on the device (CG/CG.fypp:123-171).  One iteration =
//   matvec ; pAp = p^H Ap (multi-dot) ; k_cg_update ; k_cg_check ; k_cg_direction
// with alpha / beta / the residual test kept in device scalars, so a chunk of iterations is one CUDA
// graph and the host only looks at the flags between chunks.  Iterations enqueued after the one that
// converged are no-ops (every kernel returns on flags[F_STOP]) => n_iter, x and the residual history
// are exactly those of the reference's sequential loop.
//   scal[0] = r_dot_r_old, scal[1] = beta ; flags[5] = iteration counter, flags[6] = converged
LKB_DI double2 wdiv(double2 a, double2 b) {
    const double d = b.x * b.x + b.y * b.y;
    return make_double2((a.x * b.x + a.y * b.y) / d, (a.y * b.x - a.x * b.y) / d);
}
LKB_DI double2 as_w2(double a) { return make_double2(a, 0.0); }
LKB_DI double2 as_w2(double2 a) { return a; }
LKB_DI void from_w2(double2 a, double& o) { o = a.x; }
LKB_DI void from_w2(double2 a, double2& o) { o = a; }

// Preconditioned CG (CG.fypp:113-116, 137: z = M r, rz = r^H z, p = z + beta p) runs in the same kernels, selected at
// compile time by MODE:
//   CG_PLAIN  no preconditioner: nrm2 = r^H r (the unpreconditioned loop; its code is unchanged by the other modes)
//   CG_DIAG   M = diag(d): nrm2 = sum conj(r_i) (d_i r_i) in W (complex for c / z, d need not be real), and
//             k_cg_direction forms p = d o r + beta p.  z is never stored: the mode reads d twice per iteration.
//   CG_NORED  any other M: only x and r are updated; the caller applies M to r and reduces r^H z with a multi-dot.

// One W per CTA: all threads of the LAST CTA call this after the ticket; the total is returned in thread 0
// (fixed order, as reduce_scalar_last).
template <typename W>
LKB_DI W reduce_w_last(const W* __restrict__ partial, int nb)
{
    __shared__ W s_red[32];
    const int tid = threadIdx.x, nt = blockDim.x;
    W a = zero_v(W());
    for (int b = tid; b < nb; b += nt) wadd(a, ldcg_w(&partial[b]));
    a = warp_sum(a);
    __syncthreads();
    if ((tid & 31) == 0) s_red[tid >> 5] = a;
    __syncthreads();
    W t = zero_v(W());
    if (tid == 0)
        for (int q = 0; q < (nt + 31) / 32; ++q) wadd(t, s_red[q]);
    return t;
}

// x += alpha p ; r -= alpha Ap ; nrm2 = r_new^H r_new (CG_DIAG: r_new^H d o r_new)   with alpha = rr_old / pAp  (device scalars)
template <int K, int MODE>
__global__ void __launch_bounds__(256, 2)
k_cg_update(const typename Tr<K>::W* __restrict__ scal, const typename Tr<K>::W* __restrict__ pAp,
            const typename Tr<K>::E* __restrict__ p, const typename Tr<K>::E* __restrict__ Ap,
            typename Tr<K>::E* __restrict__ x, typename Tr<K>::E* __restrict__ r, int64_t n,
            double* __restrict__ partial, typename Tr<K>::W* __restrict__ nrm2_out,
            unsigned* __restrict__ counter, const int* __restrict__ flags, const P2P p2p,
            const typename Tr<K>::E* __restrict__ d)
{
    using E = typename Tr<K>::E;
    using W = typename Tr<K>::W;
    constexpr int EPP = Tr<K>::EPP;
    using P = Pack<E, EPP>;
    if (flags[F_STOP]) return;
    W aw; from_w2(wdiv(as_w2(scal[0]), as_w2(pAp[0])), aw);
    E alpha; narrow(aw, alpha);
    const int64_t npk = n / EPP;
    double nrm = 0.0;
    W rz = zero_v(W());
    for (int64_t pk = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; pk < npk; pk += (int64_t)gridDim.x * blockDim.x) {
        const P pv = ld_pack_nc<P>(p + pk * EPP), av = ld_pack_nc<P>(Ap + pk * EPP);
        P xv = ld_pack<P>(x + pk * EPP), rv = ld_pack<P>(r + pk * EPP);
        P dv;
        if constexpr (MODE == CG_DIAG) dv = ld_pack_nc<P>(d + pk * EPP);
#pragma unroll
        for (int e = 0; e < EPP; ++e) {
            fmacc(xv.v[e], pv.v[e], alpha);
            fnma(rv.v[e], av.v[e], alpha);
            if constexpr (MODE == CG_PLAIN) nrm += abs2_w(rv.v[e]);
            if constexpr (MODE == CG_DIAG) fma_conj(rz, widen(rv.v[e]), widen(mul_v(dv.v[e], rv.v[e])));
        }
        st_pack(x + pk * EPP, xv);
        st_pack(r + pk * EPP, rv);
    }
    if (blockIdx.x == 0 && threadIdx.x == 0)
        for (int64_t t = npk * EPP; t < n; ++t) {
            E xv = x[t], rv = r[t];
            fmacc(xv, p[t], alpha); fnma(rv, Ap[t], alpha);
            x[t] = xv; r[t] = rv;
            if constexpr (MODE == CG_PLAIN) nrm += abs2_w(rv);
            if constexpr (MODE == CG_DIAG) fma_conj(rz, widen(rv), widen(mul_v(d[t], rv)));
        }
    if constexpr (MODE == CG_NORED) return;
    if constexpr (MODE == CG_DIAG) {
        __shared__ W smw[8];
        __shared__ bool is_last_w;
        W* pw = reinterpret_cast<W*>(partial);
        const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
        const W a = warp_sum(rz);
        if (lane == 0) smw[wid] = a;
        __syncthreads();
        if (threadIdx.x == 0) {
            W t = smw[0];
            for (int q = 1; q < (int)(blockDim.x >> 5); ++q) wadd(t, smw[q]);
            pw[blockIdx.x] = t;
            __threadfence();
            is_last_w = (atomicAdd(counter, 1u) == gridDim.x - 1u);
        }
        __syncthreads();
        if (is_last_w) {
            __threadfence();
            const W t = reduce_w_last<W>(pw, (int)gridDim.x);
            if (threadIdx.x == 0) { nrm2_out[0] = t; *counter = 0u; }
            __syncthreads();
            if (p2p.world > 1) p2p_allreduce_cta<W>(p2p, nrm2_out, 1);
        }
        return;
    }
    __shared__ double sm[8];
    __shared__ bool is_last;
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    const double a = warp_sum(nrm);
    if (lane == 0) sm[wid] = a;
    __syncthreads();
    if (threadIdx.x == 0) {
        double t = sm[0];
        for (int q = 1; q < (int)(blockDim.x >> 5); ++q) t += sm[q];
        partial[blockIdx.x] = t;
        __threadfence();
        is_last = (atomicAdd(counter, 1u) == gridDim.x - 1u);
    }
    __syncthreads();
    if (is_last) {
        __threadfence();
        const double t = reduce_scalar_last(partial, (int)gridDim.x);
        if (threadIdx.x == 0) {
            W o = zero_v(W());
            *reinterpret_cast<double*>(&o) = t;
            nrm2_out[0] = o;
            *counter = 0u;
        }
        __syncthreads();
        if (p2p.world > 1) p2p_allreduce_cta<W>(p2p, nrm2_out, 1);
    }
}

// residual = sqrt(|rr_new|) ; history ; convergence / maxiter stop ; beta = rr_new / rr_old ; rr_old <- rr_new
template <int K>
__global__ void k_cg_check(typename Tr<K>::W* __restrict__ scal, const typename Tr<K>::W* __restrict__ rr_new,
                           double tol, int maxiter, double* __restrict__ res_hist, int* __restrict__ flags)
{
    using W = typename Tr<K>::W;
    if (flags[F_STOP]) return;
    const double2 rn = as_w2(rr_new[0]), ro = as_w2(scal[0]);
    const double residual = sqrt(sqrt(rn.x * rn.x + rn.y * rn.y));
    const int it = ++flags[5];
    res_hist[it] = residual;
    if (residual < tol) { flags[F_STOP] = 1; flags[F_INFO] = it; flags[6] = 1; return; }
    W b; from_w2(wdiv(rn, ro), b);
    scal[1] = b;
    scal[0] = rr_new[0];
    if (it >= maxiter) { flags[F_STOP] = 1; flags[F_INFO] = it; }
}

// p = r + beta p  (beta = scal[1] on the device);  CG_DIAG: p = d o r + beta p  (r is then the residual, d o r = z)
template <int K, int MODE>
__global__ void __launch_bounds__(256)
k_cg_direction(const typename Tr<K>::W* __restrict__ scal, const typename Tr<K>::E* __restrict__ r,
               typename Tr<K>::E* __restrict__ p, int64_t n, const int* __restrict__ flags,
               const typename Tr<K>::E* __restrict__ d)
{
    using E = typename Tr<K>::E;
    constexpr int EPP = Tr<K>::EPP;
    using P = Pack<E, EPP>;
    if (flags[F_STOP]) return;
    E beta; narrow(scal[1], beta);
    const int64_t npk = n / EPP;
    for (int64_t pk = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; pk < npk; pk += (int64_t)gridDim.x * blockDim.x) {
        P rv = ld_pack_nc<P>(r + pk * EPP);
        if constexpr (MODE == CG_DIAG) {
            const P dv = ld_pack_nc<P>(d + pk * EPP);
#pragma unroll
            for (int e = 0; e < EPP; ++e) rv.v[e] = mul_v(dv.v[e], rv.v[e]);
        }
        P pv = ld_pack<P>(p + pk * EPP);
#pragma unroll
        for (int e = 0; e < EPP; ++e) pv.v[e] = add_v(rv.v[e], mul_v(beta, pv.v[e]));
        st_pack(p + pk * EPP, pv);
    }
    if (blockIdx.x == 0 && threadIdx.x == 0)
        for (int64_t t = npk * EPP; t < n; ++t) {
            E z = r[t];
            if constexpr (MODE == CG_DIAG) z = mul_v(d[t], z);
            p[t] = add_v(z, mul_v(beta, p[t]));
        }
}

// y = d o x (matvec of a diagonal operator) or conj(d) o x (rmatvec).  y may be x: every pack is read once, by the
// thread that then writes it, so the streaming read-only loads stay valid in place.
template <int K, bool CONJ>
__global__ void __launch_bounds__(256)
k_diag(const typename Tr<K>::E* __restrict__ d, const typename Tr<K>::E* x, typename Tr<K>::E* y, int64_t n,
       const int* __restrict__ flags)
{
    using E = typename Tr<K>::E;
    constexpr int EPP = Tr<K>::EPP;
    using P = Pack<E, EPP>;
    if (flags && flags[F_STOP]) return;
    const int64_t npk = n / EPP;
    for (int64_t pk = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; pk < npk; pk += (int64_t)gridDim.x * blockDim.x) {
        const P dv = ld_pack_nc<P>(d + pk * EPP);
        P xv = ld_pack_nc<P>(x + pk * EPP);
#pragma unroll
        for (int e = 0; e < EPP; ++e) xv.v[e] = mul_v(CONJ ? conj_v(dv.v[e]) : dv.v[e], xv.v[e]);
        st_pack(y + pk * EPP, xv);
    }
    if (blockIdx.x == 0 && threadIdx.x == 0)
        for (int64_t t = npk * EPP; t < n; ++t) y[t] = mul_v(CONJ ? conj_v(d[t]) : d[t], x[t]);
}

// One step of the Chebyshev preconditioner on an operator without a fused step (lkb_cheb.cu), after t = A z_k:
//     s = invd o (r - t) ;  d <- alpha d_in + beta s ;  z <- z + d      (d_out: nullptr on the last step)
// init: t, d_in and z read as zero, so z = beta invd o r = z_1 (beta = 1 / theta).  invd is the vector D^-1 (conj: conj(D)^-1),
// or the scalar invd_s when it is nullptr.  d_in may be z (first step: d_0 = z_1) and d_out may be d_in: every pack is read
// by the thread that then writes it, as in k_diag.
template <int K>
__global__ void __launch_bounds__(256)
k_cheb_update(const typename Tr<K>::E* __restrict__ r, const typename Tr<K>::E* __restrict__ invd, typename Tr<K>::E invd_s,
              const typename Tr<K>::E* __restrict__ t, const typename Tr<K>::E* d_in, typename Tr<K>::E* d_out,
              typename Tr<K>::E* z, int64_t n, typename Tr<K>::Rl alpha, typename Tr<K>::Rl beta, bool conj, bool init,
              const int* __restrict__ flags)
{
    using E = typename Tr<K>::E;
    using Rl = typename Tr<K>::Rl;
    constexpr int EPP = Tr<K>::EPP;
    using P = Pack<E, EPP>;
    if (flags && flags[F_STOP]) return;
    auto step = [&](E rv, E iv, E tv, E dv) -> E {
        const E s = mul_v(conj ? conj_v(iv) : iv, add_v(rv, rscale(tv, (Rl)-1)));
        return add_v(rscale(dv, alpha), rscale(s, beta));
    };
    const int64_t npk = n / EPP;
    for (int64_t pk = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; pk < npk; pk += (int64_t)gridDim.x * blockDim.x) {
        const int64_t o = pk * EPP;
        const P rv = ld_pack_nc<P>(r + o);
        P iv, tv, dv, zv;
#pragma unroll
        for (int e = 0; e < EPP; ++e) { iv.v[e] = invd_s; tv.v[e] = dv.v[e] = zv.v[e] = zero_v(E()); }
        if (invd) iv = ld_pack_nc<P>(invd + o);
        if (!init) { tv = ld_pack_nc<P>(t + o); dv = ld_pack_nc<P>(d_in + o); zv = ld_pack_nc<P>(z + o); }
#pragma unroll
        for (int e = 0; e < EPP; ++e) {
            dv.v[e] = step(rv.v[e], iv.v[e], tv.v[e], dv.v[e]);
            zv.v[e] = add_v(zv.v[e], dv.v[e]);
        }
        if (d_out) st_pack(d_out + o, dv);
        st_pack(z + o, zv);
    }
    if (blockIdx.x == 0 && threadIdx.x == 0)
        for (int64_t i = npk * EPP; i < n; ++i) {
            const E zv = init ? zero_v(E()) : z[i];
            const E dv = step(r[i], invd ? invd[i] : invd_s, init ? zero_v(E()) : t[i], init ? zero_v(E()) : d_in[i]);
            if (d_out) d_out[i] = dv;
            z[i] = add_v(zv, dv);
        }
}

// One step of the GMRES-polynomial preconditioner on an operator without a fused step (lkb_poly.cu), after t = A x
// (poly_comb, lkb_types.cuh):  out = a . (x, t, v) ;  acc = [acc] + b . (x, t, v).  t and v may be nullptr (read as zero:
// t for the degree-1 polynomial, v outside a root pair's second half), out and acc may be nullptr (absent).  out may be t
// or v (the step's result replaces its own operand): every pack is read by the thread that then writes it, as in k_diag.
template <int K>
__global__ void __launch_bounds__(256)
k_poly_update(const typename Tr<K>::E* __restrict__ x, const typename Tr<K>::E* t, const typename Tr<K>::E* v,
              typename Tr<K>::E* out, typename Tr<K>::E* __restrict__ acc, int64_t n, const PolyCoef<typename Tr<K>::E> c,
              int acc_read, const int* __restrict__ flags)
{
    using E = typename Tr<K>::E;
    constexpr int EPP = Tr<K>::EPP;
    using P = Pack<E, EPP>;
    if (flags && flags[F_STOP]) return;
    const int64_t npk = n / EPP;
    for (int64_t pk = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; pk < npk; pk += (int64_t)gridDim.x * blockDim.x) {
        const int64_t o = pk * EPP;
        const P xv = ld_pack_nc<P>(x + o);
        P tv, vv, av;
#pragma unroll
        for (int e = 0; e < EPP; ++e) tv.v[e] = vv.v[e] = av.v[e] = zero_v(E());
        if (t) tv = ld_pack_nc<P>(t + o);
        if (v) vv = ld_pack_nc<P>(v + o);
        if (acc && acc_read) av = ld_pack_nc<P>(acc + o);
        if (out) {
            P ov;
#pragma unroll
            for (int e = 0; e < EPP; ++e) ov.v[e] = poly_comb(xv.v[e], tv.v[e], vv.v[e], c.a[0], c.a[1], c.a[2]);
            st_pack(out + o, ov);
        }
        if (acc) {
#pragma unroll
            for (int e = 0; e < EPP; ++e) av.v[e] = add_v(av.v[e], poly_comb(xv.v[e], tv.v[e], vv.v[e], c.b[0], c.b[1], c.b[2]));
            st_pack(acc + o, av);
        }
    }
    if (blockIdx.x == 0 && threadIdx.x == 0)
        for (int64_t i = npk * EPP; i < n; ++i) {
            const E tv = t ? t[i] : zero_v(E()), vv = v ? v[i] : zero_v(E());
            const E av = (acc && acc_read) ? acc[i] : zero_v(E());
            if (out) out[i] = poly_comb(x[i], tv, vv, c.a[0], c.a[1], c.a[2]);
            if (acc) acc[i] = add_v(av, poly_comb(x[i], tv, vv, c.b[0], c.b[1], c.b[2]));
        }
}

// ------------------------------------------------------------------------------------------
// GMRES column update on the device (gmres.fypp:167-194 + submodule_utility_functions.fypp:169-204): after the
// CGS2 kernels of inner step k this single CTA forms H(:k,k) = c1 + c2 and H(k+1,k) = ||w||, decides the
// scaling (`abs(H(k+1,k)) > tol`), applies the stored Givens rotations to the new column, generates the new
// rotation, updates the right-hand side e, appends |e(k+1)| to the residual history and raises the stop flag
// when it drops below tol.  With it a whole restart cycle is one CUDA graph; inner steps enqueued after the
// converged one are no-ops.  H / e / c / s live on the device as double2 (real kinds use .x), rounded through
// the kind's precision at the same points as the host shell.
LKB_DI double2 rnd_kind(double2 v, bool single) {
    return single ? make_double2((double)(float)v.x, (double)(float)v.y) : v;
}
LKB_DI double2 cmul2(double2 a, double2 b) { return make_double2(a.x * b.x - a.y * b.y, a.x * b.y + a.y * b.x); }
template <int K>
__global__ void k_gmres_update(const typename Tr<K>::W* __restrict__ c1, const typename Tr<K>::W* __restrict__ c2, int k,
                               const typename Tr<K>::W* __restrict__ nrm2, double2* __restrict__ H, int ldh,
                               double2* __restrict__ e, double2* __restrict__ cs, double2* __restrict__ sn, double tol,
                               double* __restrict__ inv_dev, int* __restrict__ flags, double* __restrict__ res_hist)
{
    constexpr bool cplx = Tr<K>::cplx;
    constexpr bool single = (K == KS || K == KC);
    if (flags[F_STOP]) return;
    extern __shared__ double2 gh[];                       // h(0..k)
    for (int i = threadIdx.x; i < k; i += blockDim.x) {
        double2 a = as_w2(c1[i]); const double2 b = as_w2(c2[i]);
        a.x += b.x; a.y += b.y;
        if (!cplx) a.y = 0.0;
        gh[i] = rnd_kind(a, single);
    }
    __syncthreads();
    if (threadIdx.x != 0) return;
    const double beta = sqrt(fabs(wreal(nrm2[0])));
    gh[k] = rnd_kind(make_double2(beta, 0.0), single);
    *inv_dev = beta > tol ? 1.0 / beta : 1.0;
    if (!cplx) {
        for (int j = 0; j < k - 1; ++j) {                  // lasr('L','V','F')
            const double t = gh[j + 1].x;
            gh[j + 1].x = cs[j].x * t - sn[j].x * gh[j].x;
            gh[j].x = sn[j].x * t + cs[j].x * gh[j].x;
        }
        const double f = gh[k - 1].x, g = gh[k].x;         // LAPACK 3.10 lartg
        double cc, ss, r;
        if (g == 0.0) { cc = 1.0; ss = 0.0; r = f; }
        else if (f == 0.0) { cc = 0.0; ss = g > 0 ? 1.0 : -1.0; r = fabs(g); }
        else { const double d = hypot(f, g); cc = fabs(f) / d; r = copysign(d, f); ss = g / r; }
        cs[k - 1] = make_double2(cc, 0.0); sn[k - 1] = make_double2(ss, 0.0);
        gh[k - 1] = make_double2(r, 0.0); gh[k] = make_double2(0.0, 0.0);
    } else {
        for (int i = 0; i < k - 1; ++i) {
            const double2 a = cmul2(cs[i], gh[i]), b = cmul2(sn[i], gh[i + 1]);
            const double2 t = make_double2(a.x + b.x, a.y + b.y);
            const double2 p = cmul2(sn[i], gh[i]), q = cmul2(cs[i], gh[i + 1]);
            gh[i + 1] = make_double2(q.x - p.x, q.y - p.y);
            gh[i] = t;
        }
        const double nrm = sqrt(gh[k - 1].x * gh[k - 1].x + gh[k - 1].y * gh[k - 1].y + gh[k].x * gh[k].x + gh[k].y * gh[k].y);
        cs[k - 1] = make_double2(gh[k - 1].x / nrm, gh[k - 1].y / nrm);
        sn[k - 1] = make_double2(gh[k].x / nrm, gh[k].y / nrm);
        const double2 a = cmul2(cs[k - 1], gh[k - 1]), b = cmul2(sn[k - 1], gh[k]);
        gh[k - 1] = make_double2(a.x + b.x, a.y + b.y);
        gh[k] = make_double2(0.0, 0.0);
    }
    for (int i = 0; i <= k; ++i) H[i + (size_t)ldh * (k - 1)] = rnd_kind(gh[i], single);
    const double2 ek = e[k - 1];
    const double2 m = cmul2(sn[k - 1], ek);
    e[k] = rnd_kind(make_double2(-m.x, -m.y), single);
    e[k - 1] = rnd_kind(cmul2(cs[k - 1], ek), single);
    const double res = sqrt(e[k].x * e[k].x + e[k].y * e[k].y);
    res_hist[k] = res;
    flags[5] = k;
    if (res < tol) { flags[F_STOP] = 1; flags[F_INFO] = k; }
}

// ------------------------------------------------------------------------------------------
#define LKB_DISPATCH(kind, ...)                                \
    switch (kind) {                                            \
        case KS: { constexpr int K = KS; __VA_ARGS__; } break; \
        case KD: { constexpr int K = KD; __VA_ARGS__; } break; \
        case KC: { constexpr int K = KC; __VA_ARGS__; } break; \
        default: { constexpr int K = KZ; __VA_ARGS__; } break; \
    }

void launch_axpby(int kind, cudaStream_t s, Scalar alpha, const void* x, Scalar beta, void* y, int64_t n, int sms) {
    const bool b0 = (beta.re == 0.0 && beta.im == 0.0);
    LKB_DISPATCH(kind, {
        using E = typename Tr<K>::E;
        E a, b; from_scalar(alpha, a); from_scalar(beta, b);
        const int g = ew_grid(n / Tr<K>::EPP, sms);
        if (b0) k_axpby<K, true><<<g, 256, 0, s>>>(a, (const E*)x, b, (E*)y, n);
        else    k_axpby<K, false><<<g, 256, 0, s>>>(a, (const E*)x, b, (E*)y, n);
    });
}
void launch_axpy_dev(int kind, cudaStream_t s, const void* alpha_dev, double sgn, const void* x, void* y, int64_t n,
                     const int* flags, int sms) {
    LKB_DISPATCH(kind, {
        using E = typename Tr<K>::E; using W = typename Tr<K>::W;
        k_axpy_dev<K><<<ew_grid(n / Tr<K>::EPP, sms), 256, 0, s>>>((const W*)alpha_dev, sgn, (const E*)x, (E*)y, n, flags);
    });
}
void launch_scal(int kind, cudaStream_t s, Scalar alpha, void* x, int64_t n, int sms) {
    LKB_DISPATCH(kind, {
        using E = typename Tr<K>::E;
        E a; from_scalar(alpha, a);
        k_scal<K><<<ew_grid(n / Tr<K>::EPP, sms), 256, 0, s>>>(a, (E*)x, n);
    });
}
void launch_scale_dev(int kind, cudaStream_t s, void* x, int64_t n, const void* inv_dev, const int* flags, int kstep, int sms,
                      const HaloP2P* hp) {
    const HaloP2P h = hp ? *hp : HaloP2P();
    LKB_DISPATCH(kind, {
        using E = typename Tr<K>::E;
        launch_ex(k_scale_dev<K>, (unsigned)ew_grid(n / Tr<K>::EPP, sms), 256, 0, s, pdl_take(16), (E*)x, n, (const double*)inv_dev, flags, kstep, h);
    });
}
void launch_copy_gated(int kind, cudaStream_t s, const void* src, void* dst, int64_t n, const int* flags, int sms) {
    LKB_DISPATCH(kind, {
        using E = typename Tr<K>::E;
        k_copy_gated<K><<<ew_grid(n, sms), 256, 0, s>>>((const E*)src, (E*)dst, n, flags);
    });
}
void launch_fill(int kind, cudaStream_t s, void* x, int64_t n, int64_t row0, int dist, uint64_t seed, int sms) {
    LKB_DISPATCH(kind, {
        using E = typename Tr<K>::E;
        k_fill<K><<<ew_grid(n, sms), 256, 0, s>>>((E*)x, n, row0, dist, mix64(seed));
    });
}
void launch_update(int kind, cudaStream_t s, const void* c1, const void* c2, int j, const void* nrm2, void* hcol,
                   double tol, double atol, void* inv_dev, int* flags, int kstep, int mode) {
    LKB_DISPATCH(kind, {
        using E = typename Tr<K>::E; using W = typename Tr<K>::W;
        k_update<K><<<1, 128, 0, s>>>((const W*)c1, (const W*)c2, j, (const W*)nrm2, (E*)hcol, tol, atol,
                                      (double*)inv_dev, flags, kstep, mode);
    });
}
void launch_cg_update(int kind, cudaStream_t s, const void* scal, const void* pAp, const void* p, const void* Ap, void* x,
                      void* r, int64_t n, void* partial, void* nrm2_out, unsigned* counter, const int* flags, int sms,
                      const P2P* p2p, int mode, const void* d) {
    const P2P pp = p2p ? *p2p : P2P();
    LKB_DISPATCH(kind, {
        using E = typename Tr<K>::E; using W = typename Tr<K>::W;
        int64_t nb = (n / Tr<K>::EPP + 255) / 256; if (nb < 1) nb = 1; if (nb > 4 * (int64_t)sms) nb = 4 * (int64_t)sms;
        if (nb > MAX_ROWBLOCKS) nb = MAX_ROWBLOCKS;
        auto kern = mode == CG_DIAG ? k_cg_update<K, CG_DIAG> : mode == CG_NORED ? k_cg_update<K, CG_NORED> : k_cg_update<K, CG_PLAIN>;
        kern<<<(int)nb, 256, 0, s>>>((const W*)scal, (const W*)pAp, (const E*)p, (const E*)Ap, (E*)x, (E*)r, n,
                                     (double*)partial, (W*)nrm2_out, counter, flags, pp, (const E*)d);
    });
}
void launch_cg_check(int kind, cudaStream_t s, void* scal, const void* rr_new, double tol, int maxiter, double* res_hist, int* flags) {
    LKB_DISPATCH(kind, { using W = typename Tr<K>::W; k_cg_check<K><<<1, 1, 0, s>>>((W*)scal, (const W*)rr_new, tol, maxiter, res_hist, flags); });
}
void launch_cg_direction(int kind, cudaStream_t s, const void* scal, const void* r, void* p, int64_t n, const int* flags, int sms,
                         const void* d) {
    LKB_DISPATCH(kind, {
        using E = typename Tr<K>::E; using W = typename Tr<K>::W;
        auto kern = d ? k_cg_direction<K, CG_DIAG> : k_cg_direction<K, CG_PLAIN>;
        kern<<<ew_grid(n / Tr<K>::EPP, sms), 256, 0, s>>>((const W*)scal, (const E*)r, (E*)p, n, flags, (const E*)d);
    });
}
void launch_diag(int kind, cudaStream_t s, const void* d, const void* x, void* y, int64_t n, bool conj, const int* flags, int sms) {
    LKB_DISPATCH(kind, {
        using E = typename Tr<K>::E;
        auto kern = conj ? k_diag<K, true> : k_diag<K, false>;
        kern<<<ew_grid(n / Tr<K>::EPP, sms), 256, 0, s>>>((const E*)d, (const E*)x, (E*)y, n, flags);
    });
}
void launch_cheb_update(int kind, cudaStream_t s, const void* r, const void* invd, Scalar invd_s, const void* t, const void* d_in,
                        void* d_out, void* z, int64_t n, double alpha, double beta, bool conj, bool init, const int* flags, int sms) {
    LKB_DISPATCH(kind, {
        using E = typename Tr<K>::E; using Rl = typename Tr<K>::Rl;
        E is; from_scalar(invd_s, is);
        k_cheb_update<K><<<ew_grid(n / Tr<K>::EPP, sms), 256, 0, s>>>((const E*)r, (const E*)invd, is, (const E*)t, (const E*)d_in,
                                                                       (E*)d_out, (E*)z, n, (Rl)alpha, (Rl)beta, conj, init, flags);
    });
}
void launch_poly_update(int kind, cudaStream_t s, const void* x, const void* t, void* out, int64_t n, const PolyArgs& pa,
                        const int* flags, int sms) {
    LKB_DISPATCH(kind, {
        using E = typename Tr<K>::E;
        PolyCoef<E> c;
        for (int i = 0; i < 3; ++i) { from_scalar(pa.a[i], c.a[i]); from_scalar(pa.b[i], c.b[i]); }
        k_poly_update<K><<<ew_grid(n / Tr<K>::EPP, sms), 256, 0, s>>>((const E*)x, (const E*)t, (const E*)pa.v, (E*)out,
                                                                       (E*)pa.acc, n, c, pa.acc_read ? 1 : 0, flags);
    });
}
void launch_gmres_update(int kind, cudaStream_t s, const void* c1, const void* c2, int k, const void* nrm2, void* H, int ldh,
                         void* e, void* cs, void* sn, double tol, void* inv_dev, int* flags, double* res_hist) {
    LKB_DISPATCH(kind, {
        using W = typename Tr<K>::W;
        k_gmres_update<K><<<1, 128, (size_t)(k + 1) * sizeof(double2), s>>>((const W*)c1, (const W*)c2, k, (const W*)nrm2, (double2*)H, ldh,
                                                                             (double2*)e, (double2*)cs, (double2*)sn, tol, (double*)inv_dev, flags, res_hist);
    });
}
void launch_gsinfo(cudaStream_t s, const void* ww, int, double atol, int* flags) {
    k_gsinfo<<<1, 1, 0, s>>>((const double*)ww, atol, flags);
}
void launch_narrow(int kind, cudaStream_t s, const void* src, void* dst, int n, const int* flags) {
    LKB_DISPATCH(kind, {
        using E = typename Tr<K>::E; using W = typename Tr<K>::W;
        k_narrow<K><<<1, 256, 0, s>>>((const W*)src, (E*)dst, n, flags);
    });
}

}  // namespace lkb
