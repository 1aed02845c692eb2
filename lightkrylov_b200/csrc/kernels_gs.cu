// kernels_gs.cu -- the two HBM-bound kernels of one classical Gram-Schmidt pass.
//
// They replace, on a contiguous column-major device basis,
//   innerprod(X(:j), y)            = j separate dot sweeps   (AbstractVectors.fypp:659-675)
//   y%norm() zero check            = one more sweep           (gram_schmidt.fypp:127)
//   linear_combination + y%sub     = j axpbys on a temporary  (gram_schmidt.fypp:141-146)
// by ONE multi-dot (reads V once, w once) and ONE multi-axpy (reads V once, w once, writes w once).
// Algorithmic bytes per pass: 2*j*n*s (+3*n*s for w).  No tensor cores: AI ~ 0.25 flop/B.
#include <stdlib.h>
#include "lkb_kernels.h"
#include "lkb_p2p.cuh"
#include "lkb_step.cuh"
#include "lkb_reduce.cuh"

namespace lkb {

// ------------------------------------------------------------------------------------------
// multi-dot.  Persistent grid of 2 CTAs per SM; every CTA owns a contiguous row range and walks
// it in tiles of MD_THREADS*PT packs.  Per tile the w packs are loaded ONCE into registers and
// stay there while the CTA sweeps all j basis columns in chunks of MD_CB: V and w are each read
// exactly once from HBM ((j+1)*n*s bytes per launch).  Every thread keeps MD_CB accumulators
// and issues independent 128-bit loads; at the end of a (tile, chunk) the warp folds its
// MD_CB x 32 partial sums with a transposing butterfly (16 shuffles instead of 80) and adds
// them to its private row of shared-memory accumulators.
// Stage 1: fixed-order sum over the CTA's warps -> one partial row per CTA.  Stage 2: the last
// CTA to retire (atomic ticket) folds the partial rows in fixed order => run-to-run deterministic.
// ------------------------------------------------------------------------------------------
template <typename T> LKB_DI T shfl_xor_t(T v, int m);
template <> LKB_DI float shfl_xor_t<float>(float v, int m) { return __shfl_xor_sync(0xffffffffu, v, m); }
template <> LKB_DI double shfl_xor_t<double>(double v, int m) { return __shfl_xor_sync(0xffffffffu, v, m); }
template <> LKB_DI float2 shfl_xor_t<float2>(float2 v, int m) {
    return make_float2(__shfl_xor_sync(0xffffffffu, v.x, m), __shfl_xor_sync(0xffffffffu, v.y, m));
}
template <> LKB_DI double2 shfl_xor_t<double2>(double2 v, int m) {
    return make_double2(__shfl_xor_sync(0xffffffffu, v.x, m), __shfl_xor_sync(0xffffffffu, v.y, m));
}

// Transposing warp reduction of 16 per-lane values: afterwards acc[0] of lane l holds the warp
// total of value index ((l>>4)&1)*8 + ((l>>3)&1)*4 + ((l>>2)&1)*2 + ((l>>1)&1).  Fixed order.
template <typename E> LKB_DI void warp_fold16(E (&acc)[16], int lane) {
#pragma unroll
    for (int half = 8, bit = 16; half >= 1; half >>= 1, bit >>= 1) {
        const bool up = (lane & bit) != 0;
#pragma unroll
        for (int i = 0; i < half; ++i) {
            const E send = up ? acc[i] : acc[i + half];
            const E keep = up ? acc[i + half] : acc[i];
            acc[i] = add_v(keep, shfl_xor_t<E>(send, bit));
        }
    }
    acc[0] = add_v(acc[0], shfl_xor_t<E>(acc[0], 1));
}

// One tile of MD_THREADS*PT packs starting at pack `tb`: the PT packs of w of this thread are loaded once and stay in
// registers while all j columns are swept in chunks of 16.  FULL: every pack of the tile lies below `p1`.
template <int K, int PT, bool FULL>
LKB_DI void md_tile(const typename Tr<K>::E* __restrict__ V, int64_t ld, int j, int nchunk,
                    const typename Tr<K>::E* __restrict__ w, int64_t tb, int64_t p1,
                    typename Tr<K>::W* __restrict__ myacc, typename Tr<K>::E& accw, int lane, int fold_idx,
                    bool keep = false, uint64_t pol = 0)
{
    using E = typename Tr<K>::E;
    constexpr int EPP = Tr<K>::EPP;
    constexpr int CB = MD_CB;
    using P = Pack<E, EPP>;
    const int64_t base = tb + threadIdx.x;
    P wv[PT];
#pragma unroll
    for (int q = 0; q < PT; ++q) {
        const int64_t pk = base + (int64_t)q * MD_THREADS;
        if (FULL || pk < p1) wv[q] = ld_pack_nc_w<P>(w + pk * EPP, keep, pol);
        else {
#pragma unroll
            for (int e = 0; e < EPP; ++e) wv[q].v[e] = zero_v(E());
        }
#pragma unroll
        for (int e = 0; e < EPP; ++e) fma_conj(accw, wv[q].v[e], wv[q].v[e]);
    }
    for (int c = 0; c < nchunk; ++c) {
        const int c0 = c * CB;
        const int ncv = min(CB, j - c0);
        const E* vb = V + (int64_t)c0 * ld;
        E acc[CB];
#pragma unroll
        for (int i = 0; i < CB; ++i) acc[i] = zero_v(E());
        if (FULL && ncv == CB) {
#pragma unroll
            for (int q = 0; q < PT; ++q) {
                const int64_t off = (base + (int64_t)q * MD_THREADS) * EPP;
                P v[CB];
#pragma unroll
                for (int i = 0; i < CB; ++i) v[i] = ld_pack_nc<P>(vb + (int64_t)i * ld + off);
#pragma unroll
                for (int i = 0; i < CB; ++i)
#pragma unroll
                    for (int e = 0; e < EPP; ++e) fma_conj(acc[i], v[i].v[e], wv[q].v[e]);
            }
        } else {
#pragma unroll
            for (int q = 0; q < PT; ++q) {
                const int64_t pk = base + (int64_t)q * MD_THREADS;
                if (FULL || pk < p1) {
                    const int64_t off = pk * EPP;
#pragma unroll
                    for (int i = 0; i < CB; ++i) {
                        if (i < ncv) {
                            const P v = ld_pack_nc<P>(vb + (int64_t)i * ld + off);
#pragma unroll
                            for (int e = 0; e < EPP; ++e) fma_conj(acc[i], v.v[e], wv[q].v[e]);
                        }
                    }
                }
            }
        }
        warp_fold16<E>(acc, lane);
        if ((lane & 1) == 0 && fold_idx < ncv) wadd(myacc[c0 + fold_idx], widen(acc[0]));
    }
}

template <int K>
__global__ void __launch_bounds__(MD_THREADS, 2)
k_multidot(const typename Tr<K>::E* __restrict__ V, int64_t ld, int j,
           const typename Tr<K>::E* __restrict__ w, int64_t n,
           typename Tr<K>::W* __restrict__ partial, typename Tr<K>::W* __restrict__ out,
           unsigned* __restrict__ counter, const int* __restrict__ flags, const P2P p2p, const int desc)
{
    using E = typename Tr<K>::E;
    using W = typename Tr<K>::W;
    constexpr int EPP = Tr<K>::EPP;
    constexpr int CB = MD_CB;
    constexpr int NW = MD_THREADS / 32;
    static_assert(CB == 16, "warp_fold16 assumes 16 columns per chunk");

    extern __shared__ __align__(16) unsigned char smem_raw[];
    W* sacc = reinterpret_cast<W*>(smem_raw);   // [NW][jp]
    const int jp = j + 1;
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    for (int i = threadIdx.x; i < NW * jp; i += MD_THREADS) sacc[i] = zero_v(W());
    pdl_wait();                                  // w (and the stop flag) come from the predecessor
    pdl_trigger();
    if (flags && flags[F_STOP]) return;
    __syncthreads();
    W* myacc = sacc + wid * jp;
    const int fold_idx = ((lane >> 4) & 1) * 8 + ((lane >> 3) & 1) * 4 + ((lane >> 2) & 1) * 2 + ((lane >> 1) & 1);
    ktime_cta(p2p, 0);

    // Row walk = one global sweep (lkb_kernels.h "serpentine sweeps"): `nfull` rounds of big tiles (4 packs per thread:
    // one warp fold per 64 loads), round r covering the band [r, r + 1) * gridDim.x * 1024 packs with one tile per CTA,
    // then the remainder region split over the CTAs in 32-pack groups (balanced to within ONE group = 512 B for any n)
    // and walked in 1-pack tiles, only the final < 256 packs of a CTA taking the masked path.  desc = the same tiles in
    // the opposite order.  (Round 1 split whole tiles and shrank ALL tiles to 1 pack per thread at 1/8 of C2 per GPU to
    // stay balanced; a first round-2 version kept 4-pack tiles and masked the remainder -- 13 % of a CTA's rows there --
    // which was slower still.)
    const bool keep = (desc & 2) != 0;            // w is small: keep it L2-resident (lkb_types.cuh)
    const uint64_t pol = keep ? pol_evict_last() : 0ULL;
    const bool down = (desc & 1) != 0;
    const int64_t npk = n / EPP;
    constexpr int64_t BIG = 4 * MD_THREADS;
    const int64_t nfull = npk / (BIG * gridDim.x);
    const int64_t rem0 = nfull * BIG * gridDim.x;
    const int64_t rgroups = (npk - rem0 + 31) / 32;
    const int64_t q0 = rem0 + (((int64_t)blockIdx.x * rgroups) / gridDim.x) * 32;
    const int64_t q1 = min(npk, rem0 + ((((int64_t)blockIdx.x + 1) * rgroups) / gridDim.x) * 32);
    const int nchunk = (j + CB - 1) / CB;
    E accw = zero_v(E());
    auto remainder = [&]() {
        int64_t tb = q0;
        for (; tb + MD_THREADS <= q1; tb += MD_THREADS) md_tile<K, 1, true>(V, ld, j, nchunk, w, tb, q1, myacc, accw, lane, fold_idx, keep, pol);
        if (tb < q1) md_tile<K, 1, false>(V, ld, j, nchunk, w, tb, q1, myacc, accw, lane, fold_idx, keep, pol);
    };
    if (!down) {
        for (int64_t r = 0; r < nfull; ++r)
            md_tile<K, 4, true>(V, ld, j, nchunk, w, (r * gridDim.x + blockIdx.x) * BIG, npk, myacc, accw, lane, fold_idx, keep, pol);
        remainder();
    } else {
        remainder();
        for (int64_t r = nfull - 1; r >= 0; --r)
            md_tile<K, 4, true>(V, ld, j, nchunk, w, (r * gridDim.x + blockIdx.x) * BIG, npk, myacc, accw, lane, fold_idx, keep, pol);
    }
    // ragged tail (n not a multiple of the pack width): one thread of CTA 0
    __syncwarp();
    if (blockIdx.x == 0 && threadIdx.x == 0) {
        for (int64_t r = npk * EPP; r < n; ++r) {
            const E wt = w[r];
            for (int i = 0; i < j; ++i) {
                E a = zero_v(E());
                fma_conj(a, V[(int64_t)i * ld + r], wt);
                wadd(myacc[i], widen(a));
            }
            fma_conj(accw, wt, wt);
        }
    }
    {
        W a = warp_sum(widen(accw));
        if (lane == 0) wadd(myacc[j], a);
    }
    // ---- stage 1: fixed-order sum over the warps of this CTA ----
    __syncthreads();
    ktime_cta(p2p, 1);
    for (int i = threadIdx.x; i < jp; i += MD_THREADS) {
        W a = sacc[i];
#pragma unroll
        for (int q = 1; q < NW; ++q) wadd(a, sacc[q * jp + i]);
        partial[(int64_t)blockIdx.x * jp + i] = a;
    }
    // ---- stage 2: two-level tree over the partial rows (lkb_reduce.cuh) ----
    ktime_cta(p2p, 2);
    if (reduce_rows_tree<W>(partial, jp, out, counter)) {
        ktime_last(p2p, 1);
        if (p2p.world > 1) p2p_allreduce_cta<W>(p2p, out, jp);
        ktime_last(p2p, 2);
        ktime_accumulate_wait(p2p, 0);
    }
}


// ------------------------------------------------------------------------------------------
// Block (blksize > 1) Gram-Schmidt: two right-hand sides per sweep of V.
//   innerprod_matrix / linear_combination_matrix (AbstractVectors.fypp:605-643, 677-695) loop over the p
//   columns of Y, re-reading X for each; here a pair of columns shares one read of every V pack, so a
//   block step with p = 2 moves the same bytes as a single-vector step.  Same tile walk, transposing fold
//   and deterministic two-stage reduction as k_multidot; out / partial are laid out [2][j+1].
template <int K, int PT, int MINB>
__global__ void __launch_bounds__(MD_THREADS, MINB)
k_multidot2(const typename Tr<K>::E* __restrict__ V, int64_t ld, int j,
            const typename Tr<K>::E* __restrict__ w0, const typename Tr<K>::E* __restrict__ w1, int64_t n,
            typename Tr<K>::W* __restrict__ partial, typename Tr<K>::W* __restrict__ out,
            unsigned* __restrict__ counter, const int* __restrict__ flags, const P2P p2p)
{
    using E = typename Tr<K>::E;
    using W = typename Tr<K>::W;
    constexpr int EPP = Tr<K>::EPP;
    constexpr int CB = MD_CB, NW = MD_THREADS / 32;
    using P = Pack<E, EPP>;
    if (flags && flags[F_STOP]) return;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    W* sacc = reinterpret_cast<W*>(smem_raw);   // [NW][2][jp]
    const int jp = j + 1;
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    for (int i = threadIdx.x; i < NW * 2 * jp; i += MD_THREADS) sacc[i] = zero_v(W());
    __syncthreads();
    W* myacc = sacc + (size_t)wid * 2 * jp;
    const int fold_idx = ((lane >> 4) & 1) * 8 + ((lane >> 3) & 1) * 4 + ((lane >> 2) & 1) * 2 + ((lane >> 1) & 1);
    const int64_t npk = n / EPP;
    constexpr int64_t TILE = (int64_t)MD_THREADS * PT;
    const int64_t ntiles = (npk + TILE - 1) / TILE;
    const int64_t tper = (ntiles + gridDim.x - 1) / gridDim.x;
    const int64_t t0 = (int64_t)blockIdx.x * tper, t1 = min(ntiles, t0 + tper);
    const int nchunk = (j + CB - 1) / CB;
    E aw0 = zero_v(E()), aw1 = zero_v(E());
    for (int64_t t = t0; t < t1; ++t) {
        const int64_t base = t * TILE + threadIdx.x;
        P u0[PT], u1[PT];
#pragma unroll
        for (int q = 0; q < PT; ++q) {
            const int64_t pk = base + (int64_t)q * MD_THREADS;
            if (pk < npk) { u0[q] = ld_pack_nc<P>(w0 + pk * EPP); u1[q] = ld_pack_nc<P>(w1 + pk * EPP); }
            else {
#pragma unroll
                for (int e = 0; e < EPP; ++e) { u0[q].v[e] = zero_v(E()); u1[q].v[e] = zero_v(E()); }
            }
#pragma unroll
            for (int e = 0; e < EPP; ++e) { fma_conj(aw0, u0[q].v[e], u0[q].v[e]); fma_conj(aw1, u1[q].v[e], u1[q].v[e]); }
        }
        for (int c = 0; c < nchunk; ++c) {
            const int c0 = c * CB;
            const int ncv = min(CB, j - c0);
            const E* vb = V + (int64_t)c0 * ld;
            E a0[CB], a1[CB];
#pragma unroll
            for (int i = 0; i < CB; ++i) { a0[i] = zero_v(E()); a1[i] = zero_v(E()); }
#pragma unroll
            for (int q = 0; q < PT; ++q) {
                const int64_t pk = base + (int64_t)q * MD_THREADS;
                if (pk < npk) {
                    const int64_t off = pk * EPP;
#pragma unroll
                    for (int i = 0; i < CB; ++i) {
                        if (i < ncv) {
                            const P v = ld_pack_nc<P>(vb + (int64_t)i * ld + off);
#pragma unroll
                            for (int e = 0; e < EPP; ++e) { fma_conj(a0[i], v.v[e], u0[q].v[e]); fma_conj(a1[i], v.v[e], u1[q].v[e]); }
                        }
                    }
                }
            }
            warp_fold16<E>(a0, lane);
            warp_fold16<E>(a1, lane);
            if ((lane & 1) == 0 && fold_idx < ncv) {
                wadd(myacc[c0 + fold_idx], widen(a0[0]));
                wadd(myacc[jp + c0 + fold_idx], widen(a1[0]));
            }
        }
    }
    __syncwarp();
    if (blockIdx.x == 0 && threadIdx.x == 0) {
        for (int64_t r = npk * EPP; r < n; ++r) {
            const E x0 = w0[r], x1 = w1[r];
            for (int i = 0; i < j; ++i) {
                E b0 = zero_v(E()), b1 = zero_v(E());
                fma_conj(b0, V[(int64_t)i * ld + r], x0); fma_conj(b1, V[(int64_t)i * ld + r], x1);
                wadd(myacc[i], widen(b0)); wadd(myacc[jp + i], widen(b1));
            }
            fma_conj(aw0, x0, x0); fma_conj(aw1, x1, x1);
        }
    }
    {
        const W b0 = warp_sum(widen(aw0)), b1 = warp_sum(widen(aw1));
        if (lane == 0) { wadd(myacc[j], b0); wadd(myacc[jp + j], b1); }
    }
    __syncthreads();
    for (int i = threadIdx.x; i < 2 * jp; i += MD_THREADS) {
        W a = sacc[i];
#pragma unroll
        for (int q = 1; q < NW; ++q) wadd(a, sacc[(size_t)q * 2 * jp + i]);
        partial[(int64_t)blockIdx.x * 2 * jp + i] = a;
    }
    if (reduce_rows_tree<W>(partial, 2 * jp, out, counter))
        if (p2p.world > 1) p2p_allreduce_cta<W>(p2p, out, 2 * jp);
}

// W_q -= V c_q for q = 0, 1 with one read of every V pack; c laid out [2][j+1] (W type).
template <int K>
__global__ void __launch_bounds__(256, 2)
k_multiaxpy2(const typename Tr<K>::E* __restrict__ V, int64_t ld, int j, const typename Tr<K>::W* __restrict__ c,
             typename Tr<K>::E* __restrict__ w0, typename Tr<K>::E* __restrict__ w1, int64_t n, const int* __restrict__ flags)
{
    using E = typename Tr<K>::E;
    constexpr int EPP = Tr<K>::EPP;
    using P = Pack<E, EPP>;
    if (flags && flags[F_STOP]) return;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    E* cs = reinterpret_cast<E*>(smem_raw);      // [2][j]
    for (int i = threadIdx.x; i < j; i += blockDim.x) { narrow(c[i], cs[i]); narrow(c[(j + 1) + i], cs[j + i]); }
    __syncthreads();
    const int64_t npk = n / EPP;
    for (int64_t pk = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; pk < npk; pk += (int64_t)gridDim.x * blockDim.x) {
        const int64_t off = pk * EPP;
        P a0 = ld_pack<P>(w0 + off), a1 = ld_pack<P>(w1 + off);
        const E* vp = V + off;
        int i = 0;
        for (; i + 8 <= j; i += 8) {
            P v[8];
#pragma unroll
            for (int u = 0; u < 8; ++u) v[u] = ld_pack_nc<P>(vp + (int64_t)(i + u) * ld);
#pragma unroll
            for (int u = 0; u < 8; ++u)
#pragma unroll
                for (int e = 0; e < EPP; ++e) { fnma(a0.v[e], v[u].v[e], cs[i + u]); fnma(a1.v[e], v[u].v[e], cs[j + i + u]); }
        }
        for (; i < j; ++i) {
            const P v = ld_pack_nc<P>(vp + (int64_t)i * ld);
#pragma unroll
            for (int e = 0; e < EPP; ++e) { fnma(a0.v[e], v.v[e], cs[i]); fnma(a1.v[e], v.v[e], cs[j + i]); }
        }
        st_pack(w0 + off, a0); st_pack(w1 + off, a1);
    }
    if (blockIdx.x == 0 && threadIdx.x == 0)
        for (int64_t t = npk * EPP; t < n; ++t) {
            E a0 = w0[t], a1 = w1[t];
            for (int i = 0; i < j; ++i) { fnma(a0, V[(int64_t)i * ld + t], cs[i]); fnma(a1, V[(int64_t)i * ld + t], cs[j + i]); }
            w0[t] = a0; w1[t] = a1;
        }
}

// ------------------------------------------------------------------------------------------
// dot of two vectors (the `dot` TBP, CG's p^H Ap, Lanczos' 3-term coefficients): the j = 1 case of the
// multi-dot contract -- out[0] = x^H y, out[1] = y^H y -- as a plain grid-stride kernel with 4 + 4
// independent 128-bit loads in flight per thread (the chunked multi-dot keeps only 1 of its 16 column
// slots busy for j = 1 and ran at 2.4 TB/s).  Same deterministic two-stage reduction + p2p allreduce.
template <int K>
__global__ void __launch_bounds__(256, 4)
k_dot2(const typename Tr<K>::E* __restrict__ x, const typename Tr<K>::E* __restrict__ y, int64_t n,
       typename Tr<K>::W* __restrict__ partial, typename Tr<K>::W* __restrict__ out,
       unsigned* __restrict__ counter, const int* __restrict__ flags, const P2P p2p)
{
    using E = typename Tr<K>::E;
    using W = typename Tr<K>::W;
    constexpr int EPP = Tr<K>::EPP;
    constexpr int U = 4;
    using P = Pack<E, EPP>;
    pdl_wait();
    pdl_trigger();
    if (flags && flags[F_STOP]) return;
    const int64_t npk = n / EPP;
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    E axy = zero_v(E()), ayy = zero_v(E());
    int64_t pk = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    for (; pk + (U - 1) * stride < npk; pk += U * stride) {
        P xv[U], yv[U];
#pragma unroll
        for (int u = 0; u < U; ++u) { xv[u] = ld_pack_nc<P>(x + (pk + u * stride) * EPP); yv[u] = ld_pack_nc<P>(y + (pk + u * stride) * EPP); }
#pragma unroll
        for (int u = 0; u < U; ++u)
#pragma unroll
            for (int e = 0; e < EPP; ++e) { fma_conj(axy, xv[u].v[e], yv[u].v[e]); fma_conj(ayy, yv[u].v[e], yv[u].v[e]); }
    }
    for (; pk < npk; pk += stride) {
        const P xv = ld_pack_nc<P>(x + pk * EPP), yv = ld_pack_nc<P>(y + pk * EPP);
#pragma unroll
        for (int e = 0; e < EPP; ++e) { fma_conj(axy, xv.v[e], yv.v[e]); fma_conj(ayy, yv.v[e], yv.v[e]); }
    }
    if (blockIdx.x == 0 && threadIdx.x == 0)
        for (int64_t t = npk * EPP; t < n; ++t) { fma_conj(axy, x[t], y[t]); fma_conj(ayy, y[t], y[t]); }
    __shared__ W sm[8][2];
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    const W a = warp_sum(widen(axy)), b = warp_sum(widen(ayy));
    if (lane == 0) { sm[wid][0] = a; sm[wid][1] = b; }
    __syncthreads();
    if (threadIdx.x < 2) {
        W t = sm[0][threadIdx.x];
        for (int q = 1; q < 8; ++q) wadd(t, sm[q][threadIdx.x]);
        partial[(int64_t)blockIdx.x * 2 + threadIdx.x] = t;
    }
    if (reduce_rows_tree<W>(partial, 2, out, counter))
        if (p2p.world > 1) p2p_allreduce_cta<W>(p2p, out, 2);
}

// ------------------------------------------------------------------------------------------
// multi-axpy:  w -= V(:, 0:j) c.  One 16-byte pack of w per thread per iteration, the j basis
// packs streamed with UA independent 128-bit loads in flight; c broadcast from shared memory.
// Optional epilogue: ||w_new||^2 with the same two-stage deterministic reduction (this is the
// norm the reference recomputes in the next pass' zero check / in qr_no_pivoting).
// ------------------------------------------------------------------------------------------
template <int K, bool NORM>
__global__ void __launch_bounds__(256, 2)
k_multiaxpy(const typename Tr<K>::E* __restrict__ V, int64_t ld, int j,
            const typename Tr<K>::W* __restrict__ c, typename Tr<K>::E* __restrict__ w, int64_t n,
            double* __restrict__ partial, typename Tr<K>::W* __restrict__ nrm2_out,
            unsigned* __restrict__ counter, const int* __restrict__ flags, const P2P p2p)
{
    using E = typename Tr<K>::E;
    using W = typename Tr<K>::W;
    constexpr int EPP = Tr<K>::EPP;
    constexpr int UA = 8;
    using P = Pack<E, EPP>;
    pdl_wait();
    pdl_trigger();
    if (flags && flags[F_STOP]) return;

    extern __shared__ __align__(16) unsigned char smem_raw[];
    E* cs = reinterpret_cast<E*>(smem_raw);
    for (int i = threadIdx.x; i < j; i += blockDim.x) narrow(c[i], cs[i]);
    __syncthreads();

    const int64_t npk = n / EPP;
    double nrm = 0.0;
    for (int64_t pk = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; pk < npk; pk += (int64_t)gridDim.x * blockDim.x) {
        const int64_t off = pk * EPP;
        P a = ld_pack<P>(w + off);
        const E* vp = V + off;
        int i = 0;
        for (; i + UA <= j; i += UA) {
            P v[UA];
#pragma unroll
            for (int u = 0; u < UA; ++u) v[u] = ld_pack_nc<P>(vp + (int64_t)(i + u) * ld);
#pragma unroll
            for (int u = 0; u < UA; ++u) {
                const E ci = cs[i + u];
#pragma unroll
                for (int e = 0; e < EPP; ++e) fnma(a.v[e], v[u].v[e], ci);
            }
        }
        for (; i < j; ++i) {
            const P v = ld_pack_nc<P>(vp + (int64_t)i * ld);
            const E ci = cs[i];
#pragma unroll
            for (int e = 0; e < EPP; ++e) fnma(a.v[e], v.v[e], ci);
        }
        st_pack(w + off, a);
        if (NORM)
#pragma unroll
            for (int e = 0; e < EPP; ++e) nrm += abs2_w(a.v[e]);
    }
    if (blockIdx.x == 0 && threadIdx.x == 0) {
        for (int64_t t = npk * EPP; t < n; ++t) {
            E a = w[t];
            for (int i = 0; i < j; ++i) fnma(a, V[(int64_t)i * ld + t], cs[i]);
            w[t] = a;
            if (NORM) nrm += abs2_w(a);
        }
    }
    if (NORM) {
        __shared__ double sm[8];
        __shared__ bool is_last;
        const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
        double a = warp_sum(nrm);
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
                *reinterpret_cast<double*>(&o) = t;   // real part
                nrm2_out[0] = o;
                *counter = 0u;
            }
            __syncthreads();
            if (p2p.world > 1) p2p_allreduce_cta<W>(p2p, nrm2_out, 1);
        }
    }
}


// ------------------------------------------------------------------------------------------
// Final multi-axpy of a CGS2 step fused with the normalisation of the new basis vector and with the
// Hessenberg / tridiagonal / bidiagonal column update (round 2):
//     w'' = w' - V c2 ;  beta = ||w''|| ;  v_{k+1} = w'' / beta ;  H(1:k,k) = c1 + c2 ; H(k+1,k) = beta.
// The reference computes beta with one more sweep (qr_no_pivoting: `beta = Q(j)%norm()`, qr.fypp:137) and
// scales with another (`Q(j)%scal(one/beta)`, :164).  Here beta is known BEFORE the update from quantities the
// second pass already produced: V is orthonormal and c2 = V^H w', so
//     ||w' - V c2||^2 = ||w'||^2 - ||c2||^2         (Pythagoras; ||w'||^2 = c2[j] rides along with c2).
// Relative error of the right-hand side: eps * (1 + r) / (1 - r) + O(||V^H V - I||) * r with r = ||c2||^2 /
// ||w'||^2; in CGS2 r is O(eps^2 kappa^2), so the prediction is as accurate as a computed norm.  When r > 1e-2
// (pass 1 left more than 10 % of w' inside span(V): severe cancellation, i.e. at or next to a breakdown) every
// CTA takes the exact path instead: plain update, exact ||w''||^2 by the two-stage reduction (+ the in-kernel
// allreduce), and the separate k_scale_dev sweep that follows in the stream does the scaling (it returns at
// once when flags[F_SCALED] is set).  The decision is a pure function of (c2, ww), identical on every CTA and,
// after the allreduce of c2, on every rank.  Saves per step: one n*s read + n*s write sweep, one reduction with
// its cross-GPU synchronisation point, and the 1-CTA update kernel.
// ------------------------------------------------------------------------------------------
struct FinParams {
    const void* c1;      // pass-1 coefficients (W type) or nullptr (lanczos / bidiag: only the norm entry is stored)
    void* hcol;          // column of H / T / B on the device (E type) or nullptr (mode 4)
    double tol, atol;
    double* inv_dev;
    int* flags;
    int kstep, mode;     // mode 0 arnoldi, 1 lanczos, 2 bidiag, 4 gmres (norm + scaling only; k_gmres_update follows)
};

template <int K>
__global__ void __launch_bounds__(256, 2)
k_multiaxpy_fin(const typename Tr<K>::E* __restrict__ V, int64_t ld, int j,
                const typename Tr<K>::W* __restrict__ c, typename Tr<K>::E* __restrict__ w, int64_t n,
                double* __restrict__ partial, typename Tr<K>::W* __restrict__ nrm2_out,
                unsigned* __restrict__ counter, const FinParams fp, const P2P p2p, const HaloP2P hp, const int desc_mode)
{
    using E = typename Tr<K>::E;
    using W = typename Tr<K>::W;
    using Rl = typename Tr<K>::Rl;
    constexpr int EPP = Tr<K>::EPP;
    constexpr int UA = 8;
    using P = Pack<E, EPP>;
    pdl_wait();                                  // c2 / w' / flags come from the predecessor
    pdl_trigger();
    if (fp.flags[F_STOP]) return;

    extern __shared__ __align__(16) unsigned char smem_raw[];
    E* cs = reinterpret_cast<E*>(smem_raw);
    __shared__ double sm[8];
    __shared__ double s_s2;
    __shared__ bool is_last;
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    // ---- prologue: coefficients to shared memory, ||c2||^2 in a fixed order (identical on every CTA) ----
    double s2p = 0.0;
    for (int i = threadIdx.x; i < j; i += blockDim.x) {
        const W ci = c[i];
        narrow(ci, cs[i]);
        if constexpr (Tr<K>::cplx) s2p += ci.x * ci.x + ci.y * ci.y; else s2p += ci * ci;
    }
    s2p = warp_sum(s2p);
    if (lane == 0) sm[wid] = s2p;
    __syncthreads();
    if (threadIdx.x == 0) {
        double t = sm[0];
        for (int q = 1; q < (int)(blockDim.x >> 5); ++q) t += sm[q];
        s_s2 = t;
    }
    __syncthreads();
    const double s2 = s_s2;
    const double ww = wreal(c[j]);
    const bool exact = !(s2 <= 1e-2 * ww);                 // also true for NaN input
    const double pred = ww - s2;
    const double beta_p = sqrt(fabs(pred));
    const Rl inv = exact ? (Rl)1 : (Rl)fin_inv(fp.mode, beta_p, fp.tol, fp.atol);
    const bool do_scale = !exact && inv != (Rl)1;
    // P2P halo push of the finished vector (fast path only; the exact path pushes from k_scale_dev)
    const bool push = hp.he > 0 && !exact;
    const unsigned ep = push ? *hp.epoch + 1u : 0u;
    const size_t par = (size_t)(ep & 1u) * 2 * hp.side_bytes;
    E* push_lo = (push && hp.lo_region) ? reinterpret_cast<E*>(hp.lo_region + hp.data_off + par + hp.side_bytes) : nullptr;
    E* push_hi = (push && hp.hi_region) ? reinterpret_cast<E*>(hp.hi_region + hp.data_off + par) : nullptr;
    const int64_t hi0 = n - hp.he;
    ktime_cta(p2p, 0);

    const bool keep = (desc_mode & 2) != 0;
    const uint64_t pol = keep ? pol_evict_last() : 0ULL;
    const int desc = desc_mode & 1;
    // Row walk = one global sweep in time (lkb_kernels.h "serpentine sweeps").  The grid is two waves of CTAs (the second
    // wave is picked up by whichever SMs finish first: dynamic balance); the CTAs of the first wave (low blockIdx) stride
    // over the half of the rows the sweep visits first, those of the second wave over the other half.
    const int64_t npk = n / EPP;
    double nrm = 0.0;
    int64_t h0 = 0, h1 = npk;
    int idx = (int)blockIdx.x, cnt = (int)gridDim.x;
    if (gridDim.x >= 2) {
        const int half = ((int)gridDim.x + 1) / 2;
        const bool second = (int)blockIdx.x >= half;
        const int64_t mid = min(npk, ((npk / 2) + 31) / 32 * 32);
        const bool upper = (second != (desc != 0));             // which half of the rows this CTA strides over
        h0 = upper ? mid : 0; h1 = upper ? npk : mid;
        idx = second ? (int)blockIdx.x - half : (int)blockIdx.x;
        cnt = second ? (int)gridDim.x - half : half;
    }
    const int64_t stride1 = (int64_t)cnt * blockDim.x;
    const int64_t first1 = h0 + (int64_t)idx * blockDim.x + threadIdx.x;
    const int64_t nit1 = first1 < h1 ? (h1 - first1 + stride1 - 1) / stride1 : 0;
    for (int64_t it = 0; it < nit1; ++it) {
        const int64_t pk = first1 + (desc ? nit1 - 1 - it : it) * stride1;
        const int64_t off = pk * EPP;
        P a = ld_pack_w<P>(w + off, keep, pol);
        const E* vp = V + off;
        int i = 0;
        for (; i + UA <= j; i += UA) {
            P v[UA];
#pragma unroll
            for (int u = 0; u < UA; ++u) v[u] = ld_pack_nc<P>(vp + (int64_t)(i + u) * ld);
#pragma unroll
            for (int u = 0; u < UA; ++u) {
                const E ci = cs[i + u];
#pragma unroll
                for (int e = 0; e < EPP; ++e) fnma(a.v[e], v[u].v[e], ci);
            }
        }
        for (; i < j; ++i) {
            const P v = ld_pack_nc<P>(vp + (int64_t)i * ld);
            const E ci = cs[i];
#pragma unroll
            for (int e = 0; e < EPP; ++e) fnma(a.v[e], v.v[e], ci);
        }
        if (exact) {
#pragma unroll
            for (int e = 0; e < EPP; ++e) nrm += abs2_w(a.v[e]);
        } else if (do_scale) {
#pragma unroll
            for (int e = 0; e < EPP; ++e) a.v[e] = rscale(a.v[e], inv);
        }
        st_pack_w(w + off, a, keep, pol);
        if (push_lo && off < hp.he) {
#pragma unroll
            for (int e = 0; e < EPP; ++e) if (off + e < hp.he) push_lo[off + e] = a.v[e];
        }
        if (push_hi && off + EPP > hi0) {
#pragma unroll
            for (int e = 0; e < EPP; ++e) if (off + e >= hi0) push_hi[off + e - hi0] = a.v[e];
        }
    }
    if (blockIdx.x == 0 && threadIdx.x == 0) {
        for (int64_t t = npk * EPP; t < n; ++t) {
            E a = w[t];
            for (int i = 0; i < j; ++i) fnma(a, V[(int64_t)i * ld + t], cs[i]);
            if (exact) nrm += abs2_w(a); else if (do_scale) a = rscale(a, inv);
            w[t] = a;
            if (push_lo && t < hp.he) push_lo[t] = a;
            if (push_hi && t >= hi0) push_hi[t - hi0] = a;
        }
    }
    // ---- ticket: the last CTA to finish finalises the step ----
    __syncthreads();
    ktime_cta(p2p, 1);
    if (exact) {
        const double a = warp_sum(nrm);
        __syncthreads();
        if (lane == 0) sm[wid] = a;
        __syncthreads();
        if (threadIdx.x == 0) {
            double t = sm[0];
            for (int q = 1; q < (int)(blockDim.x >> 5); ++q) t += sm[q];
            partial[blockIdx.x] = t;
        }
    }
    if (push) __threadfence_system();
    __threadfence();
    __syncthreads();
    if (threadIdx.x == 0) is_last = (atomicAdd(counter, 1u) == gridDim.x - 1u);
    __syncthreads();
    if (!is_last) return;
    __threadfence();
    __shared__ double s_val;
    if (exact) {
        const double t = reduce_scalar_last(partial, (int)gridDim.x);
        if (threadIdx.x == 0) { W o = zero_v(W()); *reinterpret_cast<double*>(&o) = t; nrm2_out[0] = o; }
        __syncthreads();
        if (p2p.world > 1) p2p_allreduce_cta<W>(p2p, nrm2_out, 1);
        __syncthreads();
        if (threadIdx.x == 0) s_val = wreal(nrm2_out[0]);
    } else if (threadIdx.x == 0) {
        W o = zero_v(W()); *reinterpret_cast<double*>(&o) = pred; nrm2_out[0] = o;
        s_val = pred;
    }
    __syncthreads();
    if (fp.mode != 4) {
        E* hcol = reinterpret_cast<E*>(fp.hcol);
        const W* c1 = reinterpret_cast<const W*>(fp.c1);
        if (c1 && hcol)
            for (int i = threadIdx.x; i < j; i += blockDim.x) { W a = c1[i]; wadd(a, c[i]); narrow(a, hcol[i]); }
        if (threadIdx.x == 0)
            step_decide<K>(sqrt(fabs(s_val)), hcol, j, fp.tol, fp.atol, fp.inv_dev, fp.flags, fp.kstep, fp.mode);
    }
    ktime_last(p2p, 1);
    if (threadIdx.x == 0) {
        fp.flags[F_SCALED] = exact ? 0 : 1;
        *counter = 0u;
        if (push) {
            // all CTAs of this rank have stored (and fenced) their boundary rows: publish the epoch to the
            // neighbours; the NEXT stencil kernel waits for theirs (k_stencil*: halo_wait), not this kernel
            __threadfence_system();
            if (hp.lo_region) st_volatile_u32(reinterpret_cast<unsigned*>(hp.lo_region + 128), ep);
            if (hp.hi_region) st_volatile_u32(reinterpret_cast<unsigned*>(hp.hi_region), ep);
            *hp.epoch = ep;
        }
    }
}

// ------------------------------------------------------------------------------------------
// Dynamic shared memory of each launcher, and the attribute it runs with (SmemAttrOnce): launches that fit the fixed
// value keep it, larger ones raise it up to the device's limit.
template <int K> static size_t multidot_smem(int j) { return (size_t)(MD_THREADS / 32) * (size_t)(j + 1) * sizeof(typename Tr<K>::W); }
template <int K> static size_t multidot2_smem(int j) { return (size_t)(MD_THREADS / 32) * 2 * (size_t)(j + 1) * sizeof(typename Tr<K>::W); }
template <int K> static size_t multiaxpy_smem(int j) { return (size_t)(j > 0 ? j : 1) * sizeof(typename Tr<K>::E); }
template <int K> static const SmemAttrOnce& multidot_attr() { static const SmemAttrOnce a((const void*)k_multidot<K>, 160 * 1024); return a; }
template <int K> static const SmemAttrOnce& multidot2_attr() { static const SmemAttrOnce a((const void*)k_multidot2<K, 1, 2>, 100 * 1024); return a; }
template <int K, bool NORM> static const SmemAttrOnce& multiaxpy_attr() { static const SmemAttrOnce a((const void*)k_multiaxpy<K, NORM>, 0); return a; }
template <int K> static const SmemAttrOnce& multiaxpy_fin_attr() { static const SmemAttrOnce a((const void*)k_multiaxpy_fin<K>, 0); return a; }

template <int K> static bool multidot_fits_t(int j, SmemFit* f) {
    const size_t w = (MD_THREADS / 32) * sizeof(typename Tr<K>::W);
    return smem_fit(multidot_attr<K>(), multidot_smem<K>(j), w, w, f);
}
template <int K> static bool multidot2_fits_t(int j, SmemFit* f) {
    const size_t w = (MD_THREADS / 32) * 2 * sizeof(typename Tr<K>::W);
    return smem_fit(multidot2_attr<K>(), multidot2_smem<K>(j), w, w, f);
}
template <int K> static bool multiaxpy_fits_t(int j, bool fin, SmemFit* f) {
    // k_multiaxpy<K, true> holds the norm's reduction in static shared memory: its (lower) limit stands for both variants
    const SmemAttrOnce& a = fin ? multiaxpy_fin_attr<K>() : multiaxpy_attr<K, true>();
    return smem_fit(a, multiaxpy_smem<K>(j), sizeof(typename Tr<K>::E), 0, f);
}
template <int K>
static void multidot_t(cudaStream_t s, const void* V, int64_t ld, int j, const void* w, int64_t n,
                       void* partial, void* out, unsigned* counter, const int* flags, int sms, const P2P* p2p) {
    using E = typename Tr<K>::E; using W = typename Tr<K>::W;
    if (j == 1) {      // two-vector dot: dedicated streaming kernel
        const int64_t npk1 = n / Tr<K>::EPP;
        int64_t nb1 = (npk1 + 256 * 4 - 1) / (256 * 4);
        if (nb1 < 1) nb1 = 1;
        if (nb1 > 4 * (int64_t)sms) nb1 = 4 * (int64_t)sms;
        if (nb1 > RT_MAXROWS) nb1 = RT_MAXROWS;
        launch_ex(k_dot2<K>, (unsigned)nb1, 256, 0, s, pdl_take(2), (const E*)V, (const E*)w, n, (W*)partial, (W*)out, counter, flags, p2p ? *p2p : P2P());
        return;
    }
    const int64_t npk = n / Tr<K>::EPP;
    const P2P pp = p2p ? *p2p : P2P();
    // grid: fixed function of the problem size (2 resident CTAs per SM), never of timing.  The kernel balances the
    // rows over the CTAs in 32-pack groups, so the tile size only has to fit a CTA's share: 4 packs of w per
    // thread whenever a CTA owns at least ~one such tile, smaller tiles for small vectors.
    const int64_t ngroups = (npk + 31) / 32;
    int64_t nb = 2 * (int64_t)sms;
    if (nb > ngroups) nb = ngroups;
    if (nb < 1) nb = 1;
    if (nb > RT_MAXROWS) nb = RT_MAXROWS;
    const size_t sh = multidot_smem<K>(j);
    multidot_attr<K>().ensure(sh);
    launch_ex(k_multidot<K>, (unsigned)nb, MD_THREADS, sh, s, pdl_take(2), (const E*)V, ld, j, (const E*)w, n, (W*)partial, (W*)out, counter, flags, pp,
              sweep_dir() | (((size_t)n * sizeof(E) <= W_KEEP_BYTES) ? 2 : 0));
}
void launch_multidot(int kind, cudaStream_t s, const void* V, int64_t ld, int j, const void* w, int64_t n,
                     void* partial, void* out, unsigned* counter, const int* flags, int sms, const P2P* p2p) {
    switch (kind) {
        case KS: multidot_t<KS>(s, V, ld, j, w, n, partial, out, counter, flags, sms, p2p); break;
        case KD: multidot_t<KD>(s, V, ld, j, w, n, partial, out, counter, flags, sms, p2p); break;
        case KC: multidot_t<KC>(s, V, ld, j, w, n, partial, out, counter, flags, sms, p2p); break;
        default: multidot_t<KZ>(s, V, ld, j, w, n, partial, out, counter, flags, sms, p2p); break;
    }
}

template <int K>
static void multiaxpy_t(cudaStream_t s, const void* V, int64_t ld, int j, const void* c, void* w, int64_t n,
                        bool want_norm, void* partial, void* nrm2_out, unsigned* counter, const int* flags, int sms,
                        const P2P* p2p) {
    using E = typename Tr<K>::E; using W = typename Tr<K>::W;
    const P2P pp = p2p ? *p2p : P2P();
    const int64_t npk = n / Tr<K>::EPP;
    int64_t nb = (npk + 255) / 256;
    if (nb < 1) nb = 1;
    if (nb > 2 * sms * 2) nb = 2 * sms * 2;
    if (nb > MAX_ROWBLOCKS) nb = MAX_ROWBLOCKS;
    const size_t sh = multiaxpy_smem<K>(j);
    const bool pdl = pdl_take(8);
    if (want_norm) multiaxpy_attr<K, true>().ensure(sh);
    else multiaxpy_attr<K, false>().ensure(sh);
    if (want_norm)
        launch_ex(k_multiaxpy<K, true>, (unsigned)nb, 256, sh, s, pdl, (const E*)V, ld, j, (const W*)c, (E*)w, n, (double*)partial, (W*)nrm2_out, counter, flags, pp);
    else
        launch_ex(k_multiaxpy<K, false>, (unsigned)nb, 256, sh, s, pdl, (const E*)V, ld, j, (const W*)c, (E*)w, n, (double*)partial, (W*)nrm2_out, counter, flags, pp);
}
void launch_multiaxpy(int kind, cudaStream_t s, const void* V, int64_t ld, int j, const void* c, void* w, int64_t n,
                      bool want_norm, void* partial, void* nrm2_out, unsigned* counter, const int* flags, int sms,
                      const P2P* p2p) {
    switch (kind) {
        case KS: multiaxpy_t<KS>(s, V, ld, j, c, w, n, want_norm, partial, nrm2_out, counter, flags, sms, p2p); break;
        case KD: multiaxpy_t<KD>(s, V, ld, j, c, w, n, want_norm, partial, nrm2_out, counter, flags, sms, p2p); break;
        case KC: multiaxpy_t<KC>(s, V, ld, j, c, w, n, want_norm, partial, nrm2_out, counter, flags, sms, p2p); break;
        default: multiaxpy_t<KZ>(s, V, ld, j, c, w, n, want_norm, partial, nrm2_out, counter, flags, sms, p2p); break;
    }
}

template <int K>
static void multiaxpy_fin_t(cudaStream_t s, const void* V, int64_t ld, int j, const void* c1, const void* c2, void* w, int64_t n,
                            void* partial, void* nrm2_out, unsigned* counter, void* hcol, double tol, double atol,
                            void* inv_dev, int* flags, int kstep, int mode, int sms, const P2P* p2p, const HaloP2P* hp) {
    using E = typename Tr<K>::E; using W = typename Tr<K>::W;
    const int64_t npk = n / Tr<K>::EPP;
    int64_t nb = (npk + 255) / 256;
    if (nb < 1) nb = 1;
    if (nb > 2 * sms * 2) nb = 2 * sms * 2;
    if (nb > MAX_ROWBLOCKS) nb = MAX_ROWBLOCKS;
    const size_t sh = multiaxpy_smem<K>(j);
    multiaxpy_fin_attr<K>().ensure(sh);
    FinParams fp;
    fp.c1 = c1; fp.hcol = hcol; fp.tol = tol; fp.atol = atol; fp.inv_dev = (double*)inv_dev; fp.flags = flags;
    fp.kstep = kstep; fp.mode = mode;
    launch_ex(k_multiaxpy_fin<K>, (unsigned)nb, 256, sh, s, pdl_take(8), (const E*)V, ld, j, (const W*)c2, (E*)w, n, (double*)partial,
              (W*)nrm2_out, counter, fp, p2p ? *p2p : P2P(), hp ? *hp : HaloP2P(),
              sweep_dir() | (((size_t)n * sizeof(E) <= W_KEEP_BYTES) ? 2 : 0));
}
void launch_multiaxpy_fin(int kind, cudaStream_t s, const void* V, int64_t ld, int j, const void* c1, const void* c2, void* w,
                          int64_t n, void* partial, void* nrm2_out, unsigned* counter, void* hcol, double tol, double atol,
                          void* inv_dev, int* flags, int kstep, int mode, int sms, const P2P* p2p, const HaloP2P* hp) {
    switch (kind) {
        case KS: multiaxpy_fin_t<KS>(s, V, ld, j, c1, c2, w, n, partial, nrm2_out, counter, hcol, tol, atol, inv_dev, flags, kstep, mode, sms, p2p, hp); break;
        case KD: multiaxpy_fin_t<KD>(s, V, ld, j, c1, c2, w, n, partial, nrm2_out, counter, hcol, tol, atol, inv_dev, flags, kstep, mode, sms, p2p, hp); break;
        case KC: multiaxpy_fin_t<KC>(s, V, ld, j, c1, c2, w, n, partial, nrm2_out, counter, hcol, tol, atol, inv_dev, flags, kstep, mode, sms, p2p, hp); break;
        default: multiaxpy_fin_t<KZ>(s, V, ld, j, c1, c2, w, n, partial, nrm2_out, counter, hcol, tol, atol, inv_dev, flags, kstep, mode, sms, p2p, hp); break;
    }
}

template <int K>
static void multidot2_t(cudaStream_t s, const void* V, int64_t ld, int j, const void* w0, const void* w1, int64_t n,
                        void* partial, void* out, unsigned* counter, const int* flags, int sms, const P2P* p2p) {
    using E = typename Tr<K>::E; using W = typename Tr<K>::W;
    const int64_t npk = n / Tr<K>::EPP;
    // 2 CTAs per SM, one pack of each w per thread (110 registers).  The round-1 shape (1 CTA per SM, 2 packs per thread, 158
    // registers) ran block Arnoldi on the C2 operator at 233 vectors/s (blksize 2) against 287 now (gpurun_out/r02_blk.log).
    const int64_t ntiles = (npk + (int64_t)MD_THREADS - 1) / (int64_t)MD_THREADS;
    int64_t nb = 2 * (int64_t)sms;
    if (nb > ntiles) nb = ntiles;
    if (nb < 1) nb = 1;
    const size_t sh = multidot2_smem<K>(j);
    multidot2_attr<K>().ensure(sh);
    k_multidot2<K, 1, 2><<<(int)nb, MD_THREADS, sh, s>>>((const E*)V, ld, j, (const E*)w0, (const E*)w1, n, (W*)partial, (W*)out,
                                                         counter, flags, p2p ? *p2p : P2P());
}
void launch_multidot2(int kind, cudaStream_t s, const void* V, int64_t ld, int j, const void* w0, const void* w1, int64_t n,
                      void* partial, void* out, unsigned* counter, const int* flags, int sms, const P2P* p2p) {
    switch (kind) {
        case KS: multidot2_t<KS>(s, V, ld, j, w0, w1, n, partial, out, counter, flags, sms, p2p); break;
        case KD: multidot2_t<KD>(s, V, ld, j, w0, w1, n, partial, out, counter, flags, sms, p2p); break;
        case KC: multidot2_t<KC>(s, V, ld, j, w0, w1, n, partial, out, counter, flags, sms, p2p); break;
        default: multidot2_t<KZ>(s, V, ld, j, w0, w1, n, partial, out, counter, flags, sms, p2p); break;
    }
}
template <int K>
static void multiaxpy2_t(cudaStream_t s, const void* V, int64_t ld, int j, const void* c, void* w0, void* w1, int64_t n,
                         const int* flags, int sms) {
    using E = typename Tr<K>::E; using W = typename Tr<K>::W;
    int64_t nb = (n / Tr<K>::EPP + 255) / 256;
    if (nb < 1) nb = 1;
    if (nb > 4 * (int64_t)sms) nb = 4 * (int64_t)sms;
    const size_t sh = (size_t)2 * (j > 0 ? j : 1) * sizeof(E);
    static const SmemAttrOnce attr((const void*)k_multiaxpy2<K>, 160 * 1024);
    attr.ensure(sh);
    k_multiaxpy2<K><<<(int)nb, 256, sh, s>>>((const E*)V, ld, j, (const W*)c, (E*)w0, (E*)w1, n, flags);
}
void launch_multiaxpy2(int kind, cudaStream_t s, const void* V, int64_t ld, int j, const void* c, void* w0, void* w1,
                       int64_t n, const int* flags, int sms) {
    switch (kind) {
        case KS: multiaxpy2_t<KS>(s, V, ld, j, c, w0, w1, n, flags, sms); break;
        case KD: multiaxpy2_t<KD>(s, V, ld, j, c, w0, w1, n, flags, sms); break;
        case KC: multiaxpy2_t<KC>(s, V, ld, j, c, w0, w1, n, flags, sms); break;
        default: multiaxpy2_t<KZ>(s, V, ld, j, c, w0, w1, n, flags, sms); break;
    }
}

bool multidot_fits(int kind, int j, SmemFit* f) {
    if (j == 1) { if (f) *f = SmemFit{0, 0, 1}; return true; }     // k_dot2: no dynamic shared memory
    switch (kind) {
        case KS: return multidot_fits_t<KS>(j, f);
        case KD: return multidot_fits_t<KD>(j, f);
        case KC: return multidot_fits_t<KC>(j, f);
        default: return multidot_fits_t<KZ>(j, f);
    }
}
bool multidot2_fits(int kind, int j, SmemFit* f) {
    switch (kind) {
        case KS: return multidot2_fits_t<KS>(j, f);
        case KD: return multidot2_fits_t<KD>(j, f);
        case KC: return multidot2_fits_t<KC>(j, f);
        default: return multidot2_fits_t<KZ>(j, f);
    }
}
bool multiaxpy_fits(int kind, int j, bool fin, SmemFit* f) {
    switch (kind) {
        case KS: return multiaxpy_fits_t<KS>(j, fin, f);
        case KD: return multiaxpy_fits_t<KD>(j, fin, f);
        case KC: return multiaxpy_fits_t<KC>(j, fin, f);
        default: return multiaxpy_fits_t<KZ>(j, fin, f);
    }
}

}  // namespace lkb
