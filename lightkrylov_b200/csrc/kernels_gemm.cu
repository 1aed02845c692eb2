// kernels_gemm.cu -- tall-skinny basis update  Y(:, 0:p) = X(:, 0:k) Z(0:k, 0:p).
//
// This is the only dense contraction adjacent to the hot path: the Krylov-Schur restart
// X(:n) <- X(:kdim) Z(:, :n)  (src/Krylov/BaseKrylov.fypp:816-824) and the Ritz-vector assembly
// X(i) = sum_j y(j,i) Xwrk(j) (IterativeSolvers.fypp:1127-1132, eighs.fypp:116-123,
// svd_solvers.fypp:113-119), which the reference performs as k*p separate axpby sweeps.
// Row-local (no collective).  Each thread owns one 16-byte pack of rows and PB output columns in
// registers; X is streamed once per group of PB outputs with 128-bit loads, Z is broadcast from
// shared memory.  PB = 16 (real) / 8 (complex) keeps the fp64 FMA rate needed at full HBM speed below the
// B200 fp64 pipe, so this stays HBM-bound without tensor cores (a DMMA variant is a later row).
#include "lkb_kernels.h"

namespace lkb {

template <int K, int PB>
__global__ void __launch_bounds__(256)
k_basis_gemm(const typename Tr<K>::E* __restrict__ X, int64_t ldx, int k,
             const typename Tr<K>::E* __restrict__ Z, int ldz, int p,
             typename Tr<K>::E* __restrict__ Y, int64_t ldy, int64_t n)
{
    using E = typename Tr<K>::E;
    constexpr int EPP = Tr<K>::EPP;
    using P = Pack<E, EPP>;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    E* zs = reinterpret_cast<E*>(smem_raw);            // [k][PB]
    const int p0 = blockIdx.y * PB;
    const int np = min(PB, p - p0);
    for (int t = threadIdx.x; t < k * PB; t += blockDim.x) {
        const int i = t / PB, q = t % PB;
        zs[t] = q < np ? Z[i + (int64_t)ldz * (p0 + q)] : zero_v(E());
    }
    __syncthreads();
    const int64_t npk = n / EPP;
    for (int64_t pk = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; pk < npk; pk += (int64_t)gridDim.x * blockDim.x) {
        const int64_t off = pk * EPP;
        P acc[PB];
#pragma unroll
        for (int q = 0; q < PB; ++q)
#pragma unroll
            for (int e = 0; e < EPP; ++e) acc[q].v[e] = zero_v(E());
        int i = 0;
        for (; i + 4 <= k; i += 4) {
            P v[4];
#pragma unroll
            for (int u = 0; u < 4; ++u) v[u] = ld_pack_nc<P>(X + (int64_t)(i + u) * ldx + off);
#pragma unroll
            for (int u = 0; u < 4; ++u)
#pragma unroll
                for (int q = 0; q < PB; ++q) {
                    const E z = zs[(i + u) * PB + q];
#pragma unroll
                    for (int e = 0; e < EPP; ++e) fmacc(acc[q].v[e], v[u].v[e], z);
                }
        }
        for (; i < k; ++i) {
            const P v = ld_pack_nc<P>(X + (int64_t)i * ldx + off);
#pragma unroll
            for (int q = 0; q < PB; ++q) {
                const E z = zs[i * PB + q];
#pragma unroll
                for (int e = 0; e < EPP; ++e) fmacc(acc[q].v[e], v.v[e], z);
            }
        }
#pragma unroll
        for (int q = 0; q < PB; ++q)
            if (q < np) st_pack(Y + (int64_t)(p0 + q) * ldy + off, acc[q]);
    }
    if (blockIdx.x == 0 && threadIdx.x == 0)
        for (int64_t r = npk * EPP; r < n; ++r)
            for (int q = 0; q < np; ++q) {
                E a = zero_v(E());
                for (int i = 0; i < k; ++i) fmacc(a, X[(int64_t)i * ldx + r], zs[i * PB + q]);
                Y[(int64_t)(p0 + q) * ldy + r] = a;
            }
}

// ------------------------------------------------------------------------------------------
// fp64 tensor-core variant (rdp): Y(256-row tile, 0:pb) = X(tile, 0:k) Z(0:k, 0:pb) with mma.sync.m8n8k4.f64 (DMMA).
// The contraction is compute-bound on B200 (2*k flop per 8 bytes of X: k = 128 needs 32 flop/B against a ridge of
// ~6), so the point of the tensor-core form is not the flop rate -- DMMA and DFMA peak are the same on B200 -- but
// operand reuse: one A fragment (8 rows x 4 k) is used for all pb/8 column tiles and one B fragment (4 k x 8 cols)
// for 4 row tiles, ~20x fewer shared-memory operand loads per flop than the FMA kernel's broadcast of Z, so a
// single sweep of X produces up to 64 output columns (the FMA kernel: 16, i.e. X re-read 4x for p = 64).
//   CTA = 8 warps = 256 rows; warp = 32 rows x 64 columns = 4 x 8 accumulator tiles (64 doubles per lane pair).
//   X is streamed column-slice by column-slice (8 k-columns x 256 rows = 16 KB) through a 3-stage cp.async ring
//   ([kk][row], row stride 260: conflict-free 64-bit fragment loads); Z sits in shared memory as [kk][col],
//   stride 68.  Rows past n are zero-filled by cp.async (src-size 0) and never stored.
// ------------------------------------------------------------------------------------------
enum { GM_ROWS = 256, GM_KS = 8, GM_XS = GM_ROWS + 4, GM_PB = 64, GM_ZS = GM_PB + 4, GM_STAGES = 3 };

LKB_DI void dmma_m8n8k4(double& c0, double& c1, double a, double b) {
    asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0, %1}, {%2}, {%3}, {%0, %1};"
                 : "+d"(c0), "+d"(c1) : "d"(a), "d"(b));
}
LKB_DI void cp_async16_zfill(void* smem_dst, const void* gsrc, bool valid) {
    const uint32_t d = (uint32_t)__cvta_generic_to_shared(smem_dst);
    const int sz = valid ? 16 : 0;
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(d), "l"(gsrc), "r"(sz) : "memory");
}

__global__ void __launch_bounds__(256, 1)
k_basis_gemm_dmma(const double* __restrict__ X, int64_t ldx, int k, const double* __restrict__ Z, int ldz, int p,
                  double* __restrict__ Y, int64_t ldy, int64_t n)
{
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int kpad = (k + GM_KS - 1) / GM_KS * GM_KS;
    double* zs = reinterpret_cast<double*>(smem_raw);                 // [kpad][GM_ZS]
    double* xs = zs + (size_t)kpad * GM_ZS;                            // [GM_STAGES][GM_KS][GM_XS]
    const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
    const int p0 = blockIdx.y * GM_PB;
    const int np = min((int)GM_PB, p - p0);
    const int64_t r0 = (int64_t)blockIdx.x * GM_ROWS;
    // Z block -> shared memory, zero padded in both directions
    for (int t = tid; t < kpad * GM_PB; t += 256) {
        const int kk = t / GM_PB, q = t % GM_PB;
        zs[kk * GM_ZS + q] = (kk < k && q < np) ? Z[kk + (int64_t)ldz * (p0 + q)] : 0.0;
    }
    // cp.async of one k-slice: 8 columns x 256 rows, 16 bytes (2 rows) per request, 4 requests per thread
    auto issue = [&](int slice) {
        double* dst = xs + (size_t)(slice % GM_STAGES) * GM_KS * GM_XS;
        const int kk0 = slice * GM_KS;
#pragma unroll
        for (int q = 0; q < (GM_KS * GM_ROWS / 2) / 256; ++q) {
            const int t = tid + q * 256;
            const int kk = t / (GM_ROWS / 2), rp = t % (GM_ROWS / 2);
            const int64_t row = r0 + 2 * rp;
            const int col = min(kk0 + kk, k - 1);                      // columns past k meet zero rows of Z
            cp_async16_zfill(dst + kk * GM_XS + 2 * rp, X + (int64_t)col * ldx + min(row, n - 1) / 2 * 2, row < n);
        }
        asm volatile("cp.async.commit_group;" ::: "memory");
    };
    const int nslice = kpad / GM_KS;
    issue(0);
    if (nslice > 1) issue(1); else asm volatile("cp.async.commit_group;" ::: "memory");

    double acc[4][8][2];
#pragma unroll
    for (int mt = 0; mt < 4; ++mt)
#pragma unroll
        for (int nt = 0; nt < 8; ++nt) { acc[mt][nt][0] = 0.0; acc[mt][nt][1] = 0.0; }
    const int arow = wid * 32 + (lane >> 2);        // + 8 * mt
    const int akk = lane & 3;
    const int ntiles = (np + 7) / 8;

    for (int s = 0; s < nslice; ++s) {
        asm volatile("cp.async.wait_group 1;" ::: "memory");
        __syncthreads();                             // slice s has landed for every thread; slice s-1's buffer is free
        if (s + 2 < nslice) issue(s + 2); else asm volatile("cp.async.commit_group;" ::: "memory");
        const double* xt = xs + (size_t)(s % GM_STAGES) * GM_KS * GM_XS;
        const double* zt = zs + (size_t)s * GM_KS * GM_ZS;
#pragma unroll
        for (int h = 0; h < GM_KS / 4; ++h) {
            double a[4];
#pragma unroll
            for (int mt = 0; mt < 4; ++mt) a[mt] = xt[(h * 4 + akk) * GM_XS + arow + 8 * mt];
#pragma unroll
            for (int nt = 0; nt < 8; ++nt) {
                if (nt < ntiles) {
                    const double b = zt[(h * 4 + akk) * GM_ZS + nt * 8 + (lane >> 2)];
#pragma unroll
                    for (int mt = 0; mt < 4; ++mt) dmma_m8n8k4(acc[mt][nt][0], acc[mt][nt][1], a[mt], b);
                }
            }
        }
    }
    // C fragment: row = lane / 4, columns 2 * (lane % 4) + {0, 1}
#pragma unroll
    for (int mt = 0; mt < 4; ++mt) {
        const int64_t row = r0 + wid * 32 + 8 * mt + (lane >> 2);
        if (row < n) {
#pragma unroll
            for (int nt = 0; nt < 8; ++nt) {
                const int c0 = nt * 8 + 2 * (lane & 3);
                if (c0 < np) Y[(int64_t)(p0 + c0) * ldy + row] = acc[mt][nt][0];
                if (c0 + 1 < np) Y[(int64_t)(p0 + c0 + 1) * ldy + row] = acc[mt][nt][1];
            }
        }
    }
}

static bool gemm_dmma(cudaStream_t s, const void* X, int64_t ldx, int k, const void* Z, int ldz, int p, void* Y, int64_t ldy, int64_t n) {
    if (k < 1 || p < 1 || n < 1) return false;
    if (((uintptr_t)X & 15) || (ldx % 2)) return false;                 // 16-byte cp.async
    const int kpad = (k + GM_KS - 1) / GM_KS * GM_KS;
    const size_t sh = ((size_t)kpad * GM_ZS + (size_t)GM_STAGES * GM_KS * GM_XS) * sizeof(double);
    if (sh > 220 * 1024) return false;                                   // k > ~380: FMA kernel
    static const SmemAttrOnce attr((const void*)k_basis_gemm_dmma, 224 * 1024);
    attr.ensure();
    dim3 grid((unsigned)((n + GM_ROWS - 1) / GM_ROWS), (unsigned)((p + GM_PB - 1) / GM_PB));
    k_basis_gemm_dmma<<<grid, 256, sh, s>>>((const double*)X, ldx, k, (const double*)Z, ldz, p, (double*)Y, ldy, n);
    return true;
}

template <int K> static constexpr int gemm_pb() { return Tr<K>::cplx ? 8 : 16; }
template <int K> static const SmemAttrOnce& gemm_attr() {
    static const SmemAttrOnce a((const void*)k_basis_gemm<K, gemm_pb<K>()>, 160 * 1024);
    return a;
}
template <int K> static bool gemm_fits_t(int k, SmemFit* f) {
    const size_t per = (size_t)gemm_pb<K>() * sizeof(typename Tr<K>::E);
    return smem_fit(gemm_attr<K>(), (size_t)k * per, per, 0, f);
}
bool basis_gemm_fits(int kind, int k, SmemFit* f) {
    switch (kind) {
        case KS: return gemm_fits_t<KS>(k, f);
        case KD: return gemm_fits_t<KD>(k, f);
        case KC: return gemm_fits_t<KC>(k, f);
        default: return gemm_fits_t<KZ>(k, f);
    }
}

template <int K>
static void gemm_t(cudaStream_t s, const void* X, int64_t ldx, int k, const void* Z, int ldz, int p, void* Y,
                   int64_t ldy, int64_t n, int sms) {
    using E = typename Tr<K>::E;
    // output columns per sweep of X: 16 for the real kinds (2 * 16 FMA per 16-byte pack = 26 TFLOP/s fp64 at
    // full HBM speed, ~70 % of the B200 fp64 pipe), 8 for the complex kinds (4 FMA per complex multiply-add)
    constexpr int PB = gemm_pb<K>();
    const int64_t npk = n / Tr<K>::EPP;
    int64_t nb = (npk + 255) / 256;
    if (nb < 1) nb = 1;
    if (nb > 4 * (int64_t)sms) nb = 4 * (int64_t)sms;
    dim3 grid((unsigned)nb, (unsigned)((p + PB - 1) / PB));
    const size_t sh = (size_t)k * PB * sizeof(E);
    gemm_attr<K>().ensure(sh);
    k_basis_gemm<K, PB><<<grid, 256, sh, s>>>((const E*)X, ldx, k, (const E*)Z, ldz, p, (E*)Y, ldy, n);
}
void launch_basis_gemm(int kind, cudaStream_t s, const void* X, int64_t ldx, int k, const void* Z, int ldz, int p,
                       void* Y, int64_t ldy, int64_t n, int sms) {
    SmemFit f;
    if (!basis_gemm_fits(kind, k, &f)) { refuse_launch("basis_gemm", "k", k, f); return; }
    if (kind == KD && p >= 8 && gemm_dmma(s, X, ldx, k, Z, ldz, p, Y, ldy, n)) return;      // fp64 tensor cores
    switch (kind) {
        case KS: gemm_t<KS>(s, X, ldx, k, Z, ldz, p, Y, ldy, n, sms); break;
        case KD: gemm_t<KD>(s, X, ldx, k, Z, ldz, p, Y, ldy, n, sms); break;
        case KC: gemm_t<KC>(s, X, ldx, k, Z, ldz, p, Y, ldy, n, sms); break;
        default: gemm_t<KZ>(s, X, ldx, k, Z, ldz, p, Y, ldy, n, sms); break;
    }
}

}  // namespace lkb
