// kernels_fused.cu -- pass-1 multi-axpy fused with the pass-2 multi-dot of one CGS2 step.
//
// CGS2 (gram_schmidt.fypp:12-57) is   c1 = V^H w ; w' = w - V c1 ; c2 = V^H w' ; w'' = w' - V c2.
// The two middle operations touch the same rows of V: for a tile of rows, w'[tile] needs only
// V[tile, :] and c1, and the tile's contribution to c2 needs only V[tile, :] and w'[tile].  Holding
// the V tile in shared memory between the two phases removes one of the four sweeps over V per
// step: 3*j*n*s bytes instead of 4*j*n*s.  The arithmetic is the reference's (same c1, w', c2),
// only the summation order differs.
//
// Data movement: one TMA 2-D tensor map over V(:, 0:j) (column-major, box = TP packs of rows x 16
// columns, out-of-range rows/columns zero-filled by the hardware, no HBM traffic for them); a
// ring of 3..8 shared-memory stages (as many <= 64 KB tiles as fit in ~220 KB) filled by
// cp.async.bulk.tensor (one elected thread), completion on mbarriers.  One CTA per SM (persistent).
//   phase A  warp q owns columns 16q..16q+15, lanes own row packs: partial row sums -> smem
//   combine  w'[tile] = w[tile] - sum over warps (fixed order); stored to HBM and to smem; w'.w'
//   phase B  per-lane accumulators acc[16] += conj(V[tile, col]) * w'[tile]  (persist over tiles)
// End: one transposing warp fold per warp, one partial row per CTA, last CTA folds the rows in fixed
// order (same deterministic two-stage scheme as k_multidot).
#include <cuda.h>
#include "lkb_kernels.h"
#include "lkb_p2p.cuh"
#include "lkb_reduce.cuh"

namespace lkb {

LKB_DI uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
LKB_DI void mbar_init(uint32_t bar, int count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count));
}
LKB_DI void fence_barrier_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
LKB_DI void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
LKB_DI void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
LKB_DI void mbar_wait(uint32_t bar, uint32_t parity) {
    uint32_t done;
    do {
        asm volatile(
            "{\n\t.reg .pred p;\n\t"
            "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
            "selp.u32 %0, 1, 0, p;\n\t}"
            : "=r"(done) : "r"(bar), "r"(parity) : "memory");
    } while (!done);
}
LKB_DI void mbar_arrive(uint32_t bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
LKB_DI void consumer_sync() { asm volatile("bar.sync 1, 256;" ::: "memory"); }   // the 8 consumer warps only
LKB_DI void bulk_load_1d(uint32_t dst, const void* src, uint32_t bytes, uint32_t bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 ::"r"(dst), "l"(src), "r"(bytes), "r"(bar) : "memory");
}
LKB_DI void bulk_load_1d_hint(uint32_t dst, const void* src, uint32_t bytes, uint32_t bar, uint64_t pol) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint [%0], [%1], %2, [%3], %4;"
                 ::"r"(dst), "l"(src), "r"(bytes), "r"(bar), "l"(pol) : "memory");
}
LKB_DI void tma_load_2d(uint32_t dst, const CUtensorMap* map, int c0, int c1, uint32_t bar) {
    asm volatile(
        "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];"
        ::"r"(dst), "l"(map), "r"(c0), "r"(c1), "r"(bar) : "memory");
}

template <typename T> LKB_DI T shfl_xor_f(T v, int m);
template <> LKB_DI float shfl_xor_f<float>(float v, int m) { return __shfl_xor_sync(0xffffffffu, v, m); }
template <> LKB_DI double shfl_xor_f<double>(double v, int m) { return __shfl_xor_sync(0xffffffffu, v, m); }
template <> LKB_DI float2 shfl_xor_f<float2>(float2 v, int m) {
    return make_float2(__shfl_xor_sync(0xffffffffu, v.x, m), __shfl_xor_sync(0xffffffffu, v.y, m));
}
template <> LKB_DI double2 shfl_xor_f<double2>(double2 v, int m) {
    return make_double2(__shfl_xor_sync(0xffffffffu, v.x, m), __shfl_xor_sync(0xffffffffu, v.y, m));
}
template <typename E> LKB_DI void warp_fold16_f(E (&acc)[16], int lane) {
#pragma unroll
    for (int half = 8, bit = 16; half >= 1; half >>= 1, bit >>= 1) {
        const bool up = (lane & bit) != 0;
#pragma unroll
        for (int i = 0; i < half; ++i) {
            const E send = up ? acc[i] : acc[i + half];
            const E keep = up ? acc[i + half] : acc[i];
            acc[i] = add_v(keep, shfl_xor_f<E>(send, bit));
        }
    }
    acc[0] = add_v(acc[0], shfl_xor_f<E>(acc[0], 1));
}

enum { FZ_THREADS = 288, FZ_NW = 8, FZ_MAXSTAGES = 8, FZ_CB = 16 };   // 8 consumer warps + 1 TMA producer warp

template <int K>
__global__ void __launch_bounds__(FZ_THREADS, 1)
k_axpy_dot(const __grid_constant__ CUtensorMap tmap, int j, int tp, int nst, int elt_per_pack,
           const typename Tr<K>::W* __restrict__ c1, typename Tr<K>::E* __restrict__ w, int64_t n,
           typename Tr<K>::W* __restrict__ partial, typename Tr<K>::W* __restrict__ out,
           unsigned* __restrict__ counter, const int* __restrict__ flags, const P2P p2p, const int desc_mode)
{
    using E = typename Tr<K>::E;
    using W = typename Tr<K>::W;
    constexpr int EPP = Tr<K>::EPP;
    using P = Pack<E, EPP>;
    const int desc = desc_mode & 1;
    const bool keep = (desc_mode & 2) != 0;       // w is small: keep it L2-resident (lkb_types.cuh)
    const uint64_t pol = keep ? pol_evict_last() : 0ULL;

    extern __shared__ __align__(1024) unsigned char smem[];
    const int jp = j + 1;
    const int jc = (j + FZ_CB - 1) & ~(FZ_CB - 1);
    const int nchunk = jc / FZ_CB;
    const uint32_t stage_bytes = (uint32_t)jc * (uint32_t)tp * 16u;
    P* part = reinterpret_cast<P*>(smem + (size_t)nst * stage_bytes);         // [nchunk][tp]
    P* wnew = part + (size_t)FZ_NW * tp;                                       // [tp]
    P* wst = wnew + tp;                                                        // [nst][tp]  w tiles (bulk copies)
    uint64_t* bars = reinterpret_cast<uint64_t*>(wst + (size_t)nst * tp);      // full[nst], empty[nst]
    uint64_t* ebars = bars + nst;
    __shared__ double sww[FZ_NW + 1];

    const int tid = threadIdx.x, lane = tid & 31, wv = tid >> 5;
    const int64_t npk = n / EPP;
    const int64_t ntiles = (npk + tp - 1) / tp;
    // tiles are dealt round-robin (one global sweep over the rows, lkb_kernels.h "serpentine sweeps"), balanced to within
    // one tile; desc walks the same deal from the top
    const int nmine = (int)(((int64_t)blockIdx.x < ntiles) ? (ntiles - blockIdx.x + gridDim.x - 1) / gridDim.x : 0);
    auto tile_of = [&](int it) -> int64_t {
        const int64_t t = (int64_t)it * gridDim.x + blockIdx.x;
        return desc ? ntiles - 1 - t : t;
    };

    ktime_cta(p2p, 0);
    if (tid == 0) {
        for (int s = 0; s < nst; ++s) { mbar_init(smem_u32(&bars[s]), 1); mbar_init(smem_u32(&ebars[s]), FZ_NW); }
        fence_barrier_init();
    }
    __syncthreads();

    // Work split of the 8 consumer warps: chunk q = 16 columns, row slice = every rs-th group of 32 packs.
    // With few columns (nchunk < 8) the warps share a chunk and split the tile's rows instead of idling.
    const int msteps = tp / 32;
    const int rs = min(msteps, FZ_NW / nchunk);
    const bool worker = wv < nchunk * rs;
    const int q = worker ? wv % nchunk : 0;
    const int slice = worker ? wv / nchunk : 0;
    E c1r[FZ_CB], acc[FZ_CB];
#pragma unroll
    for (int i = 0; i < FZ_CB; ++i) { c1r[i] = zero_v(E()); acc[i] = zero_v(E()); }
    double wwacc = 0.0;

    if (wv == FZ_NW) {
        // ---- producer warp: one elected lane streams tiles through the ring (one 2-D TMA box of
        // tp packs x jc columns plus one 1-D bulk copy of the w packs per tile) ----
        // The first ring-full of tiles is issued BEFORE griddepcontrol.wait: V(:, 0:j) is not written by anyone in
        // this step and w was completed by the predecessor's predecessor (the matvec; the predecessor -- the pass-1
        // multi-dot -- only reads it), see lkb_types.cuh.  With a programmatic launch the ring (~200 KB per SM)
        // therefore fills while the multi-dot's last CTAs, its reduction tree and its NVLink allreduce still run.
        auto issue = [&](int it) {
            const int s = it % nst;
            const uint32_t bar = smem_u32(&bars[s]);
            const int64_t pk0 = tile_of(it) * tp;
            const uint32_t wbytes = (uint32_t)min((int64_t)tp, npk - pk0) * 16u;
            mbar_expect_tx(bar, stage_bytes + wbytes);
            tma_load_2d(smem_u32(smem + (size_t)s * stage_bytes), &tmap, (int)pk0 * elt_per_pack, 0, bar);
            if (keep) bulk_load_1d_hint(smem_u32(wst + (size_t)s * tp), w + pk0 * EPP, wbytes, bar, pol);
            else bulk_load_1d(smem_u32(wst + (size_t)s * tp), w + pk0 * EPP, wbytes, bar);
        };
        const int pre = min(nmine, nst);
        if (lane == 0)
            for (int it = 0; it < pre; ++it) issue(it);
        pdl_wait();
        pdl_trigger();
        const bool stop = flags && flags[F_STOP];
        if (lane == 0) {
            if (stop) {
                // breakdown raised by an earlier step: nobody consumes the tiles, but a CTA must not retire with
                // bulk copies in flight
                for (int it = 0; it < pre; ++it) mbar_wait(smem_u32(&bars[it]), 0u);
            } else {
                for (int it = pre; it < nmine; ++it) {
                    mbar_wait(smem_u32(&ebars[it % nst]), (uint32_t)((it / nst - 1) & 1));
                    issue(it);
                }
            }
        }
        if (stop) return;
    } else {
    pdl_wait();                                  // c1 and the stop flag come from the predecessor
    pdl_trigger();
    if (flags && flags[F_STOP]) return;
    // this warp's 16 coefficients of pass 1 and its 16 accumulators of pass 2
#pragma unroll
    for (int i = 0; i < FZ_CB; ++i) {
        const int col = q * FZ_CB + i;
        c1r[i] = zero_v(E());
        if (col < j) narrow(c1[col], c1r[i]);
        acc[i] = zero_v(E());
    }
    for (int it = 0; it < nmine; ++it) {
        const int s = it % nst;
        const uint32_t parity = (uint32_t)((it / nst) & 1);
        const P* tile = reinterpret_cast<const P*>(smem + (size_t)s * stage_bytes);
        // this tile's packs of w arrive with the V tile (1-D bulk copy on the same mbarrier)
        const bool own = tid < tp;
        const int64_t pk = tile_of(it) * tp + tid;
        const bool inb = own && pk < npk;

        mbar_wait(smem_u32(&bars[s]), parity);

        // ---- phase A: partial row sums over this warp's 16 columns ----
        if (worker) {
            for (int m = slice; m < msteps; m += rs) {
                const int r = m * 32 + lane;
                P ra;
#pragma unroll
                for (int e = 0; e < EPP; ++e) ra.v[e] = zero_v(E());
#pragma unroll
                for (int i = 0; i < FZ_CB; ++i) {
                    const P v = tile[(size_t)(q * FZ_CB + i) * tp + r];
#pragma unroll
                    for (int e = 0; e < EPP; ++e) fmacc(ra.v[e], v.v[e], c1r[i]);
                }
                part[(size_t)q * tp + r] = ra;
            }
        }
        consumer_sync();

        // ---- combine: w' = w - sum over warps (fixed order) ----
        if (own) {
            P wp;
#pragma unroll
            for (int e = 0; e < EPP; ++e) wp.v[e] = zero_v(E());
            if (inb) wp = wst[(size_t)s * tp + tid];
            P sum = part[tid];
            for (int qq = 1; qq < nchunk; ++qq) {
                const P t = part[(size_t)qq * tp + tid];
#pragma unroll
                for (int e = 0; e < EPP; ++e) sum.v[e] = add_v(sum.v[e], t.v[e]);
            }
            if (inb) {
#pragma unroll
                for (int e = 0; e < EPP; ++e) {
                    wp.v[e] = add_v(wp.v[e], rscale(sum.v[e], (typename Tr<K>::Rl)(-1)));
                    wwacc += abs2_w(wp.v[e]);
                }
                st_pack_w(w + pk * EPP, wp, keep, pol);
            }
            wnew[tid] = wp;
        }
        consumer_sync();

        // ---- phase B: c2 partials, accumulators persist across tiles ----
        if (worker) {
            for (int m = slice; m < msteps; m += rs) {
                const int r = m * 32 + lane;
                const P wn = wnew[r];
#pragma unroll
                for (int i = 0; i < FZ_CB; ++i) {
                    const P v = tile[(size_t)(q * FZ_CB + i) * tp + r];
#pragma unroll
                    for (int e = 0; e < EPP; ++e) fma_conj(acc[i], v.v[e], wn.v[e]);
                }
            }
        }
        // this warp is done with the stage: release it to the producer
        __syncwarp();
        if (lane == 0) mbar_arrive(smem_u32(&ebars[s]));
    }
    }   // consumer warps

    // ---- stage 1: one partial row per CTA; the rs row-slice warps of a chunk are summed in fixed order ----
    const int fold_idx = ((lane >> 4) & 1) * 8 + ((lane >> 3) & 1) * 4 + ((lane >> 2) & 1) * 2 + ((lane >> 1) & 1);
    __syncthreads();                                   // the ring is drained: reuse `part` as [rs][jc] W scratch
    ktime_cta(p2p, 1);
    W* fold = reinterpret_cast<W*>(part);
    if (worker) {
        warp_fold16_f<E>(acc, lane);
        if ((lane & 1) == 0) fold[(size_t)slice * jc + q * FZ_CB + fold_idx] = widen(acc[0]);
    }
    {
        const double a = warp_sum(wwacc);
        if (lane == 0) sww[wv] = a;
    }
    __syncthreads();
    for (int col = tid; col < j; col += FZ_THREADS) {
        W a = fold[col];
        for (int sl = 1; sl < rs; ++sl) wadd(a, fold[(size_t)sl * jc + col]);
        partial[(int64_t)blockIdx.x * jp + col] = a;
    }
    if (tid == 0) {
        double t = sww[0];
        for (int q = 1; q < FZ_NW; ++q) t += sww[q];     // the producer warp's slot is always zero
        W o = zero_v(W());
        *reinterpret_cast<double*>(&o) = t;
        partial[(int64_t)blockIdx.x * jp + j] = o;
    }
    // ---- stage 2: two-level tree over the partial rows (lkb_reduce.cuh) ----
    ktime_cta(p2p, 2);
    if (reduce_rows_tree<W>(partial, jp, out, counter)) {
        ktime_last(p2p, 1);
        if (p2p.world > 1) p2p_allreduce_cta<W>(p2p, out, jp);
        ktime_last(p2p, 2);
        ktime_accumulate_wait(p2p, 1);
    }
}

// ------------------------------------------------------------------------------------------
typedef CUresult (*PFN_tmapEncodeTiled)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                        const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                        CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
static PFN_tmapEncodeTiled get_encode() {
    static PFN_tmapEncodeTiled fn = nullptr;
    static bool tried = false;
    if (!tried) {
        tried = true;
        void* p = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess &&
            q == cudaDriverEntryPointSuccess)
            fn = (PFN_tmapEncodeTiled)p;
    }
    return fn;
}

template <int K>
static bool axpy_dot_ok(const void* V, int64_t ld, int j, const void* w, int64_t n) {
    constexpr int EPP = Tr<K>::EPP;
    const size_t es = sizeof(typename Tr<K>::E);
    const int eltsz = (K == KS) ? 4 : 8;                           // tensor described in 4- or 8-byte words
    if (j < 1 || j > FZ_NW * FZ_CB) return false;                 // one 16-column chunk per warp
    if (n % EPP != 0 || n < 32 * EPP) return false;
    if (((uintptr_t)V & 15) || ((uintptr_t)w & 15) || ((size_t)ld * es) % 16) return false;
    return get_encode() && (int64_t)n * (int64_t)es / eltsz < ((int64_t)1 << 31);
}

template <int K>
static bool axpy_dot_t(cudaStream_t s, const void* V, int64_t ld, int j, const void* c1, void* w, int64_t n,
                       void* partial, void* out, unsigned* counter, const int* flags, int sms, const P2P* p2p) {
    using E = typename Tr<K>::E; using W = typename Tr<K>::W;
    constexpr int EPP = Tr<K>::EPP;
    const size_t es = sizeof(E);
    const int jc = (j + FZ_CB - 1) & ~(FZ_CB - 1);
    // rows per tile: stage = jc * tp * 16 B <= 64 KB; few columns -> taller tiles, so the per-tile
    // synchronisation cost (~1500 clk) stays small against the tile's HBM time (TMA box rows <= 256 words)
    const int tp = jc > 64 ? 32 : ((jc > 32 || K == KS) ? 64 : 128);
    const int eltsz = (K == KS) ? 4 : 8;                           // tensor described in 4- or 8-byte words
    const int elt_per_pack = 16 / eltsz;
    CUtensorMap tmap;
    cuuint64_t gdim[2] = {(cuuint64_t)((size_t)n * es / eltsz), (cuuint64_t)j};
    cuuint64_t gstr[1] = {(cuuint64_t)((size_t)ld * es)};
    cuuint32_t box[2] = {(cuuint32_t)(tp * elt_per_pack), (cuuint32_t)jc};   // one box = the whole tile
    cuuint32_t estr[2] = {1, 1};
    CUresult r = get_encode()(&tmap, eltsz == 4 ? CU_TENSOR_MAP_DATA_TYPE_UINT32 : CU_TENSOR_MAP_DATA_TYPE_UINT64, 2,
                              const_cast<void*>(V), gdim, gstr, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                              CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) return false;
    // as many stages as fit: the ring must keep >= ~100 KB in flight per SM to cover the ~2 us loaded
    // TMA latency at 23 B/clk/SM (measured: 3 x 40 KB stages ran latency-bound at 5.0 TB/s).  Any j <= 128 leaves room
    // for at least 3 stages of <= 66 KB.
    const size_t budget = 222 * 1024;
    const size_t fixed = (size_t)(FZ_NW + 1) * tp * 16 + 128;
    int nst = (int)((budget - fixed) / ((size_t)jc * tp * 16 + (size_t)tp * 16 + 16));
    if (nst > FZ_MAXSTAGES) nst = FZ_MAXSTAGES;
    const size_t sh = (size_t)nst * jc * tp * 16 + (size_t)(FZ_NW + 1 + nst) * tp * 16 + 16 * nst + 64;
    static const SmemAttrOnce attr((const void*)k_axpy_dot<K>, 224 * 1024);
    attr.ensure();
    const int64_t ntiles = (n / EPP + tp - 1) / tp;
    int64_t nb = sms;
    if (nb > ntiles) nb = ntiles;
    if (nb > RT_MAXROWS) nb = RT_MAXROWS;
    launch_ex(k_axpy_dot<K>, (unsigned)nb, FZ_THREADS, sh, s, pdl_take(4), tmap, j, tp, nst, elt_per_pack, (const W*)c1, (E*)w, n, (W*)partial, (W*)out, counter, flags, p2p ? *p2p : P2P(),
              sweep_dir() | (((size_t)n * sizeof(E) <= W_KEEP_BYTES) ? 2 : 0));
    return true;
}

bool axpy_dot_supported(int kind, const void* V, int64_t ld, int j, const void* w, int64_t n) {
    switch (kind) {
        case KS: return axpy_dot_ok<KS>(V, ld, j, w, n);
        case KD: return axpy_dot_ok<KD>(V, ld, j, w, n);
        case KC: return axpy_dot_ok<KC>(V, ld, j, w, n);
        default: return axpy_dot_ok<KZ>(V, ld, j, w, n);
    }
}
bool launch_axpy_dot(int kind, cudaStream_t s, const void* V, int64_t ld, int j, const void* c1, void* w, int64_t n,
                     void* partial, void* out, unsigned* counter, const int* flags, int sms, const P2P* p2p) {
    switch (kind) {
        case KS: return axpy_dot_t<KS>(s, V, ld, j, c1, w, n, partial, out, counter, flags, sms, p2p);
        case KD: return axpy_dot_t<KD>(s, V, ld, j, c1, w, n, partial, out, counter, flags, sms, p2p);
        case KC: return axpy_dot_t<KC>(s, V, ld, j, c1, w, n, partial, out, counter, flags, sms, p2p);
        default: return axpy_dot_t<KZ>(s, V, ld, j, c1, w, n, partial, out, counter, flags, sms, p2p);
    }
}

}  // namespace lkb
