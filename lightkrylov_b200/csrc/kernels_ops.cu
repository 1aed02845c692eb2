// kernels_ops.cu -- abstract_linop extensions: matrix-free 5-/7-point stencils and CSR SpMV.
//
// Reference contract: src/AbstractTypes/AbstractLinops.fypp:58-87 (matvec / rmatvec, vec_out is
// intent(out)).  Stencil index convention: p = i + nx*(j + ny*k); coef = (center,-x,+x,-y,+y,-z,+z),
// homogeneous Dirichlet outside the global grid.  The slowest axis (y in 2-D, z in 3-D) is the
// row-sharded one: the neighbouring slab's boundary row / plane arrives in halo_lo / halo_hi.
#include <algorithm>
#include <type_traits>
#include "lkb_kernels.h"
#include "lkb_p2p.cuh"

namespace lkb {

template <typename E> struct Coef7 { E c[7]; };

template <typename E, int PW> struct PackOps {
    using P = Pack<E, PW>;
    // Pack is alignas(16), so sizeof(P) == 16 even for a partial pack (PW elements < 16 bytes: rows whose length is not a
    // multiple of the pack width): only a FULL pack may be moved with one 128-bit access
    static constexpr bool FULL = (PW * sizeof(E) == 16);
    static LKB_DI P ld(const E* p) {
        if constexpr (FULL) return ld_pack_l1<P>(p);
        else { P r;
#pragma unroll
            for (int e = 0; e < PW; ++e) r.v[e] = __ldg(p + e);
            return r; }
    }
    // halo data written by a peer GPU during this kernel's lifetime: bypass L1 (ld.global.cg)
    static LKB_DI P ld_cg(const E* p) {
        if constexpr (FULL) { int4 r = __ldcg(reinterpret_cast<const int4*>(p)); return *reinterpret_cast<P*>(&r); }
        else { P r;
#pragma unroll
            for (int e = 0; e < PW; ++e) r.v[e] = __ldcg(p + e);
            return r; }
    }
    // row-local operands of the Chebyshev epilogue (r, d): streamed, no L1 allocation
    static LKB_DI P ld_nc(const E* p) {
        if constexpr (FULL) return ld_pack_nc<P>(p);
        else { P r;
#pragma unroll
            for (int e = 0; e < PW; ++e) r.v[e] = p[e];
            return r; }
    }
    static LKB_DI void st(E* p, const P& v) {
        if constexpr (FULL) st_pack(p, v);
        else {
#pragma unroll
            for (int e = 0; e < PW; ++e) p[e] = v.v[e];
        }
    }
    // the matvec output is the work vector w of the step that follows: small slices are stored with L2 evict_last (lkb_types.cuh)
    static LKB_DI void st_w(E* p, const P& v, bool keep, uint64_t pol) {
        if constexpr (FULL) st_pack_w(p, v, keep, pol);
        else st(p, v);
    }
    static LKB_DI P zero() { P r;
#pragma unroll
        for (int e = 0; e < PW; ++e) r.v[e] = zero_v(E());
        return r; }
};


// Store epilogues of the two stencil kernels, chosen at compile time.  StorePlain: y = A x (the matvec).  ChebStep: one
// step k of the Chebyshev preconditioner (lkb_cheb.cu) on the matvec's output t = (A x)_i and its input x_i = (z_k)_i,
//     s = invd (r_i - t) ;  d_i <- alpha d_i + beta s ;  y_i = z_{k+1} = z_k + d_i
// with x = z_k, or on the first step x = r itself (z_1 = d_0 = b0 invd r, so z_1 and A z_1 are b0 invd times x and A x).
// The last step stores only y.  HBM traffic per step: x, r, d read, d, y written (first step: r read, d, y written).
struct StorePlain {};
template <typename E> struct ChebStep {
    const E* r; E* d;
    E invd;                                     // D^-1: the scalar 1 / c0 (conjugated for the rmatvec)
    double alpha, beta, b0;                     // step coefficients (lkb_cheb.cu), rounded to the kind in the kernel
    int first, last;
};
template <typename E, int PW, typename Rl>
LKB_DI void cheb_store(const ChebStep<E>& c, E* y, int64_t q, const Pack<E, PW>& t, const Pack<E, PW>& x) {
    using PO = PackOps<E, PW>;
    using P = Pack<E, PW>;
    const Rl alpha = (Rl)c.alpha, beta = (Rl)c.beta, b0 = (Rl)c.b0;
    const P rv = c.first ? x : PO::ld_nc(c.r + q);
    P dv, zn;
    if (!c.first) dv = PO::ld_nc(c.d + q);
#pragma unroll
    for (int e = 0; e < PW; ++e) {
        const E zk = c.first ? rscale(mul_v(c.invd, x.v[e]), b0) : x.v[e];
        const E tk = c.first ? rscale(mul_v(c.invd, t.v[e]), b0) : t.v[e];
        const E s = mul_v(c.invd, add_v(rv.v[e], rscale(tk, (Rl)-1)));
        dv.v[e] = add_v(rscale(c.first ? zk : dv.v[e], alpha), rscale(s, beta));
        zn.v[e] = add_v(zk, dv.v[e]);
    }
    if (!c.last) PO::st(c.d + q, dv);
    PO::st(y + q, zn);
}
// PolyStep: one step of the GMRES-polynomial preconditioner (lkb_poly.cu) on t = (A x)_i and x_i:
//     y_i = a . (x, t, v)_i  (y may be nullptr: no output) ;  acc_i = [acc_i] + b . (x, t, v)_i  (acc may be nullptr)
// v (nullptr: zero) is the held y of a root pair's second half.  HBM traffic: x read, then at most one of (y written,
// v read) plus acc read and written: at most 4 n s per step.
template <typename E> struct PolyStep {
    const E* v; E* acc;
    PolyCoef<E> c;
    int acc_read;                               // 0: acc is written, 1: accumulated
};
template <typename E, int PW>
LKB_DI void poly_store(const PolyStep<E>& c, E* y, int64_t q, const Pack<E, PW>& t, const Pack<E, PW>& x) {
    using PO = PackOps<E, PW>;
    using P = Pack<E, PW>;
    P vv = PO::zero(), a = PO::zero(), o;
    if (c.v) vv = PO::ld_nc(c.v + q);
    if (c.acc_read) a = PO::ld_nc(c.acc + q);
#pragma unroll
    for (int e = 0; e < PW; ++e) {
        o.v[e] = poly_comb(x.v[e], t.v[e], vv.v[e], c.c.a[0], c.c.a[1], c.c.a[2]);
        a.v[e] = add_v(a.v[e], poly_comb(x.v[e], t.v[e], vv.v[e], c.c.b[0], c.c.b[1], c.c.b[2]));
    }
    if (y) PO::st(y + q, o);
    if (c.acc) PO::st(c.acc + q, a);
}
// MgStep: one Chebyshev smoothing step on a level of the multigrid preconditioner (lkb_mg.cu), on t = (A x)_i and x_i.  A
// coarse level's centre is c0 + ecor[mask] on the points that sit on the last index of the axes in mask (bit 0 x, 1 y, 2 z):
// t gains ecor[mask] x_i there, and D^-1 there is invd[mask] (ecor[0] = 0, invd[0] = 1 / c0).  Modes:
//   MG_SCALE    y = b0 D^-1 x: z_1 of a smoothing from zero (t is not used)
//   MG_FIRST_R  ChebStep's first step on x = r, valid only where D is constant (a level without edge corrections)
//   MG_STEP     s = D^-1 (r - t) ; d = alpha d_in + beta s ; y = x + d.  With d_in nullptr, d = beta s and d_in is not
//               read (the first post-smoothing step, from a nonzero guess: stale memory must not enter as 0 * NaN).
// d goes to d_out unless that is nullptr.  HBM traffic per step as ChebStep's.  (The modes: lkb_kernels.h.)
template <typename E> struct MgStep {
    const E* r; const E* d_in; E* d_out;
    E invd[8], ecor[8];
    double alpha, beta, b0;
    int mode;
};
// a[mk] by selects: a dynamic index into a kernel parameter would copy the whole array to local memory
template <typename E> LKB_DI E pick8(const E (&a)[8], int mk) {
    E v = a[0];
#pragma unroll
    for (int q = 1; q < 8; ++q) if (mk == q) v = a[q];
    return v;
}
// myz: the y / z mask bits of this row; xlast: the pack element on the last x index (outside 0 .. PW-1: none)
template <typename E, int PW, typename Rl>
LKB_DI void mg_store(const MgStep<E>& c, E* y, int64_t q, const Pack<E, PW>& t, const Pack<E, PW>& x, int myz, int64_t xlast) {
    using PO = PackOps<E, PW>;
    using P = Pack<E, PW>;
    const Rl alpha = (Rl)c.alpha, beta = (Rl)c.beta, b0 = (Rl)c.b0;
    P zn;
    if (c.mode == MG_SCALE) {
#pragma unroll
        for (int e = 0; e < PW; ++e) zn.v[e] = rscale(mul_v(pick8(c.invd, myz | (e == xlast ? 1 : 0)), x.v[e]), b0);
        PO::st(y + q, zn);
        return;
    }
    const P rv = c.mode == MG_FIRST_R ? x : PO::ld_nc(c.r + q);
    P dv = PO::zero();
    if (c.mode == MG_STEP && c.d_in) dv = PO::ld_nc(c.d_in + q);
#pragma unroll
    for (int e = 0; e < PW; ++e) {
        const int mk = myz | (e == xlast ? 1 : 0);
        const E iv = mk ? pick8(c.invd, mk) : c.invd[0];
        E tk = t.v[e], zk = x.v[e];
        if (mk) fmacc(tk, x.v[e], pick8(c.ecor, mk));
        if (c.mode == MG_FIRST_R) { zk = rscale(mul_v(iv, x.v[e]), b0); tk = rscale(mul_v(iv, tk), b0); dv.v[e] = zk; }
        const E s = mul_v(iv, add_v(rv.v[e], rscale(tk, (Rl)-1)));
        dv.v[e] = add_v(rscale(dv.v[e], alpha), rscale(s, beta));
        zn.v[e] = add_v(zk, dv.v[e]);
    }
    if (c.d_out) PO::st(c.d_out + q, dv);
    PO::st(y + q, zn);
}

// Both stencil kernels take one CTA per (column block, row block[, plane]) of a 1-D grid, column block fastest
// (consecutive CTAs stream consecutive segments of the same grid rows).  The row blocks (2-D) / planes (3-D) are rotated
// by one so that the CTAs that read the inter-GPU halos (first / last row block in 2-D, first / last plane in 3-D) are
// scheduled LAST: the slab interior is computed while the neighbours' halo rows are still in flight (SURVEY 8e:
// "overlapped with the interior update").  halo_wait: the halo-reading CTAs wait until the neighbours published the
// epoch the local counter says (k_halo_push has already waited, so this is one load; after a push fused into
// k_multiaxpy_fin / k_scale_dev nobody has waited yet and this is where the exchange is synchronised).
// Both kernels take the same argument list; in 2-D, nz is 1 and the z coefficients are unused.
enum { ST_RY = 8 };           // grid rows per CTA
LKB_DI void halo_wait(const unsigned* halo_epoch, const unsigned* flag_lo, const unsigned* flag_hi, bool need_lo, bool need_hi) {
    if (!halo_epoch || !(need_lo || need_hi)) return;      // uniform over the CTA
    if (threadIdx.x == 0) {
        const unsigned ep = *halo_epoch;
        if (need_lo && flag_lo) spin_until(flag_lo, ep);
        if (need_hi && flag_hi) spin_until(flag_hi, ep);
        __threadfence_system();
    }
    __syncthreads();
}

// ------------------------------------------------------------------------------------------
// 3-D 7-point stencil: register y-march (2.5-D blocking).  One CTA = blockDim.x threads side by side along x
// (blockDim.x * PW points of one grid row of plane k), marching ST_RY rows in y: the south / centre / north packs of a
// column live in registers, so every x element of the plane is loaded from HBM once per CTA (+2 halo rows per ST_RY
// rows, served by L2 because the neighbouring CTA streams them at the same time).  The x-halo (west / east neighbour of
// a pack) comes from L1 (the neighbouring thread loaded that line), the z-neighbours from L2 (the CTAs of planes k-1 /
// k+1 stream them) or, at the slab edges, from the inter-GPU halo planes halo_lo / halo_hi.
// HBM traffic ~ (2 + 2/ST_RY) * n * s.
// Why this kernel (B200, fp64, 384^3, profiles/stencil_ab.py -> profiles/r02_stencil_ab.txt): 5.15 TB/s, against
// 2.9-3.7 TB/s for the 2-D kernel's shared-memory staging extended by the planes k-1 / k+1 (3 * ST_RY + 2 staged rows
// per CTA cut the occupancy) and 3.95 TB/s for a z-march with the planes in registers (y-neighbours re-read through L1;
// a deeper plane prefetch thrashed L1).  A z-march with the plane staged in shared memory (two block barriers per
// plane, round 1) reached 2.8 TB/s.
// ------------------------------------------------------------------------------------------
template <int K, int PW, class EPI = StorePlain>
__global__ void __launch_bounds__(256)
k_stencil(const typename Tr<K>::E* __restrict__ x, typename Tr<K>::E* __restrict__ y,
          int64_t nx, int64_t ny, int64_t nz, Coef7<typename Tr<K>::E> cf,
          const typename Tr<K>::E* __restrict__ halo_lo, const typename Tr<K>::E* __restrict__ halo_hi,
          const unsigned* __restrict__ halo_epoch, int64_t halo_parity_stride, const unsigned* __restrict__ flag_lo,
          const unsigned* __restrict__ flag_hi, int64_t ncb, const int* __restrict__ flags, const int keep_w, const EPI epi)
{
    using E = typename Tr<K>::E;
    using PO = PackOps<E, PW>;
    const bool keep = keep_w != 0;
    const uint64_t pol = keep ? pol_evict_last() : 0ULL;
    pdl_wait();            // x, the stop flag and the halo epoch come from the predecessor
    pdl_trigger();
    if (flags && flags[F_STOP]) return;
    if (halo_epoch) {      // double-buffered p2p halos: pick the parity of the current epoch
        const int64_t off = (int64_t)(*halo_epoch & 1u) * halo_parity_stride;
        if (halo_lo) halo_lo += off;
        if (halo_hi) halo_hi += off;
    }
    using P = typename PO::P;
    const int64_t npk_row = nx / PW;
    const int64_t nyb = (ny + ST_RY - 1) / ST_RY;
    const int64_t bid = blockIdx.x;
    const int64_t cb = bid % ncb, rg = bid / ncb;
    const int64_t rb = rg % nyb, k = (rg / nyb + 1) % nz;
    const int64_t ip = cb * blockDim.x + threadIdx.x;
    const bool active = ip < npk_row;                 // idle lanes march the row's last pack and store nothing
    const int64_t i0 = (active ? ip : npk_row - 1) * PW;
    const int64_t j0 = rb * ST_RY;
    const int64_t j1 = min(ny, j0 + ST_RY);
    halo_wait(halo_epoch, flag_lo, flag_hi, halo_lo && k == 0, halo_hi && k == nz - 1);
    const int64_t plane = nx * ny;
    const E* xk = x + k * plane;

    auto getrow = [&](int64_t j) -> P {
        if (j < 0 || j >= ny) return PO::zero();
        return PO::ld(xk + j * nx + i0);
    };
    P south = getrow(j0 - 1), center = getrow(j0);
    for (int64_t j = j0; j < j1; ++j) {
        const P north = getrow(j + 1);
        const int64_t p = j * nx + i0;
        const E west = i0 > 0 ? __ldg(xk + p - 1) : zero_v(E());
        const E east = (i0 + PW < nx) ? __ldg(xk + p + PW) : zero_v(E());
        const P down = (k > 0) ? PO::ld(xk + p - plane) : (halo_lo ? PO::ld_cg(halo_lo + p) : PO::zero());
        const P up = (k < nz - 1) ? PO::ld(xk + p + plane) : (halo_hi ? PO::ld_cg(halo_hi + p) : PO::zero());
        P out;
#pragma unroll
        for (int e = 0; e < PW; ++e) {
            E s = mul_v(cf.c[0], center.v[e]);
            fmacc(s, (e > 0 ? center.v[e > 0 ? e - 1 : 0] : west), cf.c[1]);
            fmacc(s, (e < PW - 1 ? center.v[e < PW - 1 ? e + 1 : 0] : east), cf.c[2]);
            fmacc(s, south.v[e], cf.c[3]);
            fmacc(s, north.v[e], cf.c[4]);
            fmacc(s, down.v[e], cf.c[5]);
            fmacc(s, up.v[e], cf.c[6]);
            out.v[e] = s;
        }
        if constexpr (std::is_same_v<EPI, StorePlain>) {
            if (active) PO::st_w(y + k * plane + p, out, keep, pol);
        } else if constexpr (std::is_same_v<EPI, PolyStep<E>>) {
            if (active) poly_store<E, PW>(epi, y, k * plane + p, out, center);
        } else if constexpr (std::is_same_v<EPI, MgStep<E>>) {
            if (active) mg_store<E, PW, typename Tr<K>::Rl>(epi, y, k * plane + p, out, center,
                                                             (j == ny - 1 ? 2 : 0) | (k == nz - 1 ? 4 : 0), nx - 1 - i0);
        } else {
            if (active) cheb_store<E, PW, typename Tr<K>::Rl>(epi, y, k * plane + p, out, center);
        }
        south = center; center = north;
    }
}

// ------------------------------------------------------------------------------------------
// 2-D 5-point stencil: shared-memory halo staging.  One CTA = ST_TX packs in x by ST_RY rows in y.  The CTA first
// issues ALL its loads -- the (ST_RY+2) x ST_TX tile including the y-halo rows (from the neighbouring rows, from the
// inter-GPU halo buffers at slab edges, or zero at the Dirichlet boundary) -- as cp.async copies straight into shared
// memory (ST_RY+2 requests in flight per thread, no register staging), waits once, and then computes the ST_RY output
// rows from shared memory: north / south / west / east neighbours are shared-memory reads, only the west/east scalar
// of the tile's edge columns comes from global memory.  Every x element is fetched from L2/HBM once per CTA.
// Why this kernel (B200, fp64, 4096^2, profiles/stencil_ab.py -> profiles/r02_stencil_ab.txt): 5.85 TB/s, against
// 4.85 TB/s for a register y-march like the 3-D kernel's and 5.81 TB/s for the same staging with 4 rows per CTA.
// ------------------------------------------------------------------------------------------
enum { ST_TX = 128 };

template <int BYTES> LKB_DI void cp_async(void* smem_dst, const void* gsrc) {
    const uint32_t d = (uint32_t)__cvta_generic_to_shared(smem_dst);
    if constexpr (BYTES == 16) asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(d), "l"(gsrc) : "memory");
    else if constexpr (BYTES == 8) asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"(d), "l"(gsrc) : "memory");
    else asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"(d), "l"(gsrc) : "memory");
}
LKB_DI void cp_async_wait_all() { asm volatile("cp.async.commit_group;\n\tcp.async.wait_group 0;" ::: "memory"); }

template <int K, int PW, class EPI = StorePlain>
__global__ void __launch_bounds__(ST_TX)
k_stencil_smem(const typename Tr<K>::E* __restrict__ x, typename Tr<K>::E* __restrict__ y,
               int64_t nx, int64_t ny, int64_t nz, Coef7<typename Tr<K>::E> cf,
               const typename Tr<K>::E* __restrict__ halo_lo, const typename Tr<K>::E* __restrict__ halo_hi,
               const unsigned* __restrict__ halo_epoch, int64_t halo_parity_stride, const unsigned* __restrict__ flag_lo,
               const unsigned* __restrict__ flag_hi, int64_t ncb, const int* __restrict__ flags, const int keep_w, const EPI epi)
{
    using E = typename Tr<K>::E;
    using P = Pack<E, PW>;
    constexpr int PB = PW * (int)sizeof(E);       // payload bytes (Pack is padded to 16 B)
    const bool keep = keep_w != 0;
    const uint64_t pol = keep ? pol_evict_last() : 0ULL;
    pdl_wait();
    pdl_trigger();
    if (flags && flags[F_STOP]) return;
    if (halo_epoch) {
        const int64_t off = (int64_t)(*halo_epoch & 1u) * halo_parity_stride;
        if (halo_lo) halo_lo += off;
        if (halo_hi) halo_hi += off;
    }
    extern __shared__ __align__(16) unsigned char st_smem[];
    P* tile = reinterpret_cast<P*>(st_smem);                       // [(ST_RY+2)][ST_TX]
    const int tx = threadIdx.x;
    const int64_t npk_row = nx / PW;
    const int64_t nyb = (ny + ST_RY - 1) / ST_RY;
    const int64_t bid = blockIdx.x;
    const int64_t cb = bid % ncb, rb = (bid / ncb + 1) % nyb;
    const int64_t ip = cb * ST_TX + tx;
    const bool active = ip < npk_row;
    const int64_t i0 = ip * PW;
    const int64_t j0 = rb * ST_RY;
    halo_wait(halo_epoch, flag_lo, flag_hi, halo_lo && j0 == 0, halo_hi && j0 + ST_RY >= ny);
    P zero;
#pragma unroll
    for (int e = 0; e < PW; ++e) zero.v[e] = zero_v(E());

    if (active) {
        // ---- issue every load of the tile ----
#pragma unroll
        for (int r = 0; r < ST_RY + 2; ++r) {
            const int64_t j = j0 - 1 + r;
            const E* src = nullptr;
            if (j >= 0 && j < ny) src = x + j * nx + i0;
            else if (j < 0 && halo_lo) src = halo_lo + i0;
            else if (j == ny && halo_hi) src = halo_hi + i0;
            if (src && j <= ny) cp_async<PB>(&tile[r * ST_TX + tx], src);
            else tile[r * ST_TX + tx] = zero;
        }
    }
    cp_async_wait_all();
    __syncthreads();
    if (!active) return;
    // ---- compute ST_RY rows out of shared memory ----
#pragma unroll
    for (int r = 0; r < ST_RY; ++r) {
        const int64_t j = j0 + r;
        if (j >= ny) break;
        const int64_t p = j * nx + i0;
        const P center = tile[(r + 1) * ST_TX + tx], south = tile[r * ST_TX + tx], north = tile[(r + 2) * ST_TX + tx];
        E west, east;
        if (tx > 0) west = tile[(r + 1) * ST_TX + tx - 1].v[PW - 1];
        else west = i0 > 0 ? __ldg(x + p - 1) : zero_v(E());
        if (tx < ST_TX - 1 && ip + 1 < npk_row) east = tile[(r + 1) * ST_TX + tx + 1].v[0];
        else east = (i0 + PW < nx) ? __ldg(x + p + PW) : zero_v(E());
        P out;
#pragma unroll
        for (int e = 0; e < PW; ++e) {
            E sacc = mul_v(cf.c[0], center.v[e]);
            fmacc(sacc, (e > 0 ? center.v[e > 0 ? e - 1 : 0] : west), cf.c[1]);
            fmacc(sacc, (e < PW - 1 ? center.v[e < PW - 1 ? e + 1 : 0] : east), cf.c[2]);
            fmacc(sacc, south.v[e], cf.c[3]);
            fmacc(sacc, north.v[e], cf.c[4]);
            out.v[e] = sacc;
        }
        if constexpr (std::is_same_v<EPI, StorePlain>) PackOps<E, PW>::st_w(y + p, out, keep, pol);
        else if constexpr (std::is_same_v<EPI, PolyStep<E>>) poly_store<E, PW>(epi, y, p, out, center);
        else if constexpr (std::is_same_v<EPI, MgStep<E>>)
            mg_store<E, PW, typename Tr<K>::Rl>(epi, y, p, out, center, j == ny - 1 ? 2 : 0, nx - 1 - i0);
        else cheb_store<E, PW, typename Tr<K>::Rl>(epi, y, p, out, center);
    }
}

template <typename E> static Coef7<E> stencil_coef(const StencilArgs& a, bool trans) {
    Coef7<E> cf;
    Scalar c[7];
    for (int q = 0; q < 7; ++q) c[q] = a.coef[q];
    if (trans) {  // A^H of a constant-coefficient stencil: swap +/- neighbours, conjugate
        Scalar t;
        t = c[1]; c[1] = c[2]; c[2] = t; t = c[3]; c[3] = c[4]; c[4] = t; t = c[5]; c[5] = c[6]; c[6] = t;
        for (int q = 0; q < 7; ++q) c[q].im = -c[q].im;
    }
    for (int q = 0; q < 7; ++q) from_scalar(c[q], cf.c[q]);
    return cf;
}

template <int K, int PW, int DIM, class EPI>
static void stencil_launch(cudaStream_t s, const StencilArgs& a, const void* x, void* y, bool trans, const int* flags, const EPI& epi) {
    using E = typename Tr<K>::E;
    const Coef7<E> cf = stencil_coef<E>(a, trans);
    const int64_t npk_row = a.nx / PW;
    const int64_t nyb = (a.ny + ST_RY - 1) / ST_RY;
    const int keep_w = ((size_t)a.nx * (size_t)a.ny * (size_t)a.nz * sizeof(E) <= W_KEEP_BYTES) ? 1 : 0;
    auto launch = [&](auto kern, int64_t ncb, unsigned block, size_t smem) {
        const unsigned grid = (unsigned)(nyb * a.nz * ncb);
        launch_ex(kern, grid, block, smem, s, pdl_take(1), (const E*)x, (E*)y, a.nx, a.ny, a.nz, cf,
                  (const E*)a.halo_lo, (const E*)a.halo_hi, a.halo_epoch, a.halo_parity_stride, a.flag_lo, a.flag_hi, ncb, flags, keep_w, epi);
    };
    if constexpr (DIM == 2) {
        static const SmemAttrOnce once((const void*)k_stencil_smem<K, PW, EPI>, 96 * 1024);
        once.ensure();
        launch(k_stencil_smem<K, PW, EPI>, (npk_row + ST_TX - 1) / ST_TX, ST_TX, (size_t)(ST_RY + 2) * ST_TX * sizeof(Pack<E, PW>));
    } else {
        // CTA width: the narrowest multiple of 32 threads that covers a grid row with the same number of CTAs as 256-wide
        // ones would (384^3: 192 packs per row -> 192 threads, no idle lanes; a 256-wide CTA left 25 % of its threads idle:
        // 4.28 TB/s at 384^3 against 5.17 TB/s at 512^3)
        const int64_t ncb = (npk_row + 255) / 256;
        launch(k_stencil<K, PW, EPI>, ncb, (unsigned)std::min<int64_t>(256, ((npk_row + ncb - 1) / ncb + 31) / 32 * 32), 0);
    }
}

template <int K, class EPI>
static void stencil_t(cudaStream_t s, const StencilArgs& a, const void* x, void* y, bool trans, const int* flags, const EPI& epi) {
    constexpr int EPP = Tr<K>::EPP;
    const bool vec = (a.nx % EPP == 0);
    if (a.dim == 2) {
        if (vec) stencil_launch<K, EPP, 2>(s, a, x, y, trans, flags, epi);
        else stencil_launch<K, 1, 2>(s, a, x, y, trans, flags, epi);
    } else {
        if (vec) stencil_launch<K, EPP, 3>(s, a, x, y, trans, flags, epi);
        else stencil_launch<K, 1, 3>(s, a, x, y, trans, flags, epi);
    }
}
void launch_stencil(int kind, cudaStream_t s, const StencilArgs& a, const void* x, void* y, bool trans,
                    const int* flags, int) {
    switch (kind) {
        case KS: stencil_t<KS>(s, a, x, y, trans, flags, StorePlain()); break;
        case KD: stencil_t<KD>(s, a, x, y, trans, flags, StorePlain()); break;
        case KC: stencil_t<KC>(s, a, x, y, trans, flags, StorePlain()); break;
        default: stencil_t<KZ>(s, a, x, y, trans, flags, StorePlain()); break;
    }
}
// One fused Chebyshev step (ChebStep above): y = z_{k+1} from x = z_k (first step: x = r)
template <int K>
static void stencil_cheb_t(cudaStream_t s, const StencilArgs& a, const void* x, void* y, bool trans, const int* flags,
                           const ChebArgs& ca) {
    using E = typename Tr<K>::E;
    ChebStep<E> epi;
    epi.r = (const E*)ca.r; epi.d = (E*)ca.d;
    from_scalar(ca.invd, epi.invd);
    epi.alpha = ca.alpha; epi.beta = ca.beta; epi.b0 = ca.b0;
    epi.first = ca.first ? 1 : 0; epi.last = ca.last ? 1 : 0;
    stencil_t<K>(s, a, x, y, trans, flags, epi);
}
void launch_stencil_cheb(int kind, cudaStream_t s, const StencilArgs& a, const void* x, void* y, bool trans, const int* flags,
                         const ChebArgs& ca) {
    switch (kind) {
        case KS: stencil_cheb_t<KS>(s, a, x, y, trans, flags, ca); break;
        case KD: stencil_cheb_t<KD>(s, a, x, y, trans, flags, ca); break;
        case KC: stencil_cheb_t<KC>(s, a, x, y, trans, flags, ca); break;
        default: stencil_cheb_t<KZ>(s, a, x, y, trans, flags, ca); break;
    }
}
// One fused polynomial step (PolyStep above): y = out (nullptr: none), acc updated, from the stencil input x
template <int K>
static void stencil_poly_t(cudaStream_t s, const StencilArgs& a, const void* x, void* y, bool trans, const int* flags,
                           const PolyArgs& pa) {
    using E = typename Tr<K>::E;
    PolyStep<E> epi;
    epi.v = (const E*)pa.v; epi.acc = (E*)pa.acc;
    for (int i = 0; i < 3; ++i) { from_scalar(pa.a[i], epi.c.a[i]); from_scalar(pa.b[i], epi.c.b[i]); }
    epi.acc_read = pa.acc_read ? 1 : 0;
    stencil_t<K>(s, a, x, y, trans, flags, epi);
}
void launch_stencil_poly(int kind, cudaStream_t s, const StencilArgs& a, const void* x, void* y, bool trans, const int* flags,
                         const PolyArgs& pa) {
    switch (kind) {
        case KS: stencil_poly_t<KS>(s, a, x, y, trans, flags, pa); break;
        case KD: stencil_poly_t<KD>(s, a, x, y, trans, flags, pa); break;
        case KC: stencil_poly_t<KC>(s, a, x, y, trans, flags, pa); break;
        default: stencil_poly_t<KZ>(s, a, x, y, trans, flags, pa); break;
    }
}
// One fused multigrid smoothing step (MgStep above)
template <int K>
static void stencil_mg_t(cudaStream_t s, const StencilArgs& a, const void* x, void* y, bool trans, const int* flags,
                         const MgArgs& ma) {
    using E = typename Tr<K>::E;
    MgStep<E> epi;
    epi.r = (const E*)ma.r; epi.d_in = (const E*)ma.d_in; epi.d_out = (E*)ma.d_out;
    for (int q = 0; q < 8; ++q) { from_scalar(ma.invd[q], epi.invd[q]); from_scalar(ma.ecor[q], epi.ecor[q]); }
    epi.alpha = ma.alpha; epi.beta = ma.beta; epi.b0 = ma.b0; epi.mode = ma.mode;
    stencil_t<K>(s, a, x, y, trans, flags, epi);
}
void launch_stencil_mg(int kind, cudaStream_t s, const StencilArgs& a, const void* x, void* y, bool trans, const int* flags,
                       const MgArgs& ma) {
    switch (kind) {
        case KS: stencil_mg_t<KS>(s, a, x, y, trans, flags, ma); break;
        case KD: stencil_mg_t<KD>(s, a, x, y, trans, flags, ma); break;
        case KC: stencil_mg_t<KC>(s, a, x, y, trans, flags, ma); break;
        default: stencil_mg_t<KZ>(s, a, x, y, trans, flags, ma); break;
    }
}

// ------------------------------------------------------------------------------------------
// Grid transfers of the multigrid preconditioner (lkb_mg.cu).  Every axis n -> n / 2, coarse point c at fine point 2c+1;
// 1-D interpolation P: fine 2c+1 takes coarse c, fine 2c and 2c+2 take half of it, coarse points outside the grid are zero.
// k_mg_restrict: bc = 2^-dim P^T (b - A x), one thread per coarse point, which gathers the residuals of the fine points
// 2c .. 2c+2 along each axis (weights 1/2, 1, 1/2; 2c+2 may lie past the grid).  A residual is formed where it is used, from
// x through L1 (a fine point on an even index serves two coarse points): b and x are read from HBM once and the fine
// residual is never stored.  The centre of the fine level is c0 + ecor[mask] as in MgStep, ecor[mask] the sum of the
// per-axis corrections ed.c[d] = ecor[1 << d].
template <typename E> struct Edge3 { E c[3]; };
template <int K>
__global__ void __launch_bounds__(256, 1)
k_mg_restrict(const typename Tr<K>::E* __restrict__ x, const typename Tr<K>::E* __restrict__ b, typename Tr<K>::E* __restrict__ bc,
              int64_t nx, int64_t ny, int64_t nz, bool three, Coef7<typename Tr<K>::E> cf, Edge3<typename Tr<K>::E> ed,
              const int* __restrict__ flags)
{
    using E = typename Tr<K>::E;
    using Rl = typename Tr<K>::Rl;
    if (flags && flags[F_STOP]) return;
    const int64_t cx = nx / 2, cy = ny / 2, cz = three ? nz / 2 : 1;
    const int64_t ncoarse = cx * cy * cz;
    auto res = [&](int64_t i, int64_t j, int64_t k) -> E {
        const int64_t p = i + nx * (j + ny * k);
        const E xc = __ldg(x + p);
        E s = mul_v(cf.c[0], xc);
        if (i > 0) fmacc(s, __ldg(x + p - 1), cf.c[1]);
        if (i < nx - 1) fmacc(s, __ldg(x + p + 1), cf.c[2]); else fmacc(s, xc, ed.c[0]);
        if (j > 0) fmacc(s, __ldg(x + p - nx), cf.c[3]);
        if (j < ny - 1) fmacc(s, __ldg(x + p + nx), cf.c[4]); else fmacc(s, xc, ed.c[1]);
        if (three) {
            if (k > 0) fmacc(s, __ldg(x + p - nx * ny), cf.c[5]);
            if (k < nz - 1) fmacc(s, __ldg(x + p + nx * ny), cf.c[6]); else fmacc(s, xc, ed.c[2]);
        }
        return add_v(__ldg(b + p), rscale(s, (Rl)-1));
    };
    for (int64_t q = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; q < ncoarse; q += (int64_t)gridDim.x * blockDim.x) {
        const int64_t ic = q % cx, jc = (q / cx) % cy, kc = q / (cx * cy);
        E acc = zero_v(E());
#pragma unroll 1
        for (int dz = 0; dz < (three ? 3 : 1); ++dz) {
            const int64_t k = three ? 2 * kc + dz : 0;
            if (k >= nz) break;
            const Rl wz = (three && dz != 1) ? (Rl)0.5 : (Rl)1;
            for (int dy = 0; dy < 3; ++dy) {
                const int64_t j = 2 * jc + dy;
                if (j >= ny) break;
                const Rl wyz = dy == 1 ? wz : wz * (Rl)0.5;
                for (int dx = 0; dx < 3; ++dx) {
                    const int64_t i = 2 * ic + dx;
                    if (i >= nx) break;
                    acc = add_v(acc, rscale(res(i, j, k), dx == 1 ? wyz : wyz * (Rl)0.5));
                }
            }
        }
        bc[q] = rscale(acc, three ? (Rl)0.125 : (Rl)0.25);
    }
}
// k_mg_prolong: x += P e on the fine grid, one thread per fine point; e is the coarse vector (cached in L1 / L2)
template <int K>
__global__ void __launch_bounds__(256)
k_mg_prolong(typename Tr<K>::E* __restrict__ x, const typename Tr<K>::E* __restrict__ e, int64_t nx, int64_t ny, int64_t nz,
             bool three, const int* __restrict__ flags)
{
    using E = typename Tr<K>::E;
    using Rl = typename Tr<K>::Rl;
    if (flags && flags[F_STOP]) return;
    const int64_t cx = nx / 2, cy = ny / 2, cz = three ? nz / 2 : 1;
    const int64_t n = nx * ny * nz;
    // the coarse points of fine index i along an axis of nc coarse points: c0 (weight w0) and c0 + 1 (weight w1); a weight is
    // zero where the point is outside the coarse grid or not a neighbour
    auto axis = [](int64_t i, int64_t nc, int64_t& c0, Rl& w0, Rl& w1) {
        if (i & 1) { c0 = i >> 1; w0 = (Rl)1; w1 = (Rl)0; return; }
        c0 = (i >> 1) - 1;
        w0 = i > 0 ? (Rl)0.5 : (Rl)0;
        w1 = (i >> 1) < nc ? (Rl)0.5 : (Rl)0;
    };
    for (int64_t p = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; p < n; p += (int64_t)gridDim.x * blockDim.x) {
        const int64_t i = p % nx, j = (p / nx) % ny, k = p / (nx * ny);
        int64_t ci, cj, ck = 0;
        Rl wi[2], wj[2], wk[2] = {(Rl)1, (Rl)0};
        axis(i, cx, ci, wi[0], wi[1]); axis(j, cy, cj, wj[0], wj[1]);
        if (three) axis(k, cz, ck, wk[0], wk[1]);
        E acc = zero_v(E());
#pragma unroll
        for (int a = 0; a < 2; ++a)
#pragma unroll
            for (int bb = 0; bb < 2; ++bb)
#pragma unroll
                for (int c = 0; c < 2; ++c) {
                    const Rl w = wi[c] * wj[bb] * wk[a];
                    if (w != (Rl)0) acc = add_v(acc, rscale(__ldg(e + (ci + c) + cx * ((cj + bb) + cy * (ck + a))), w));
                }
        x[p] = add_v(x[p], acc);
    }
}
template <int K>
static void mg_transfer_t(cudaStream_t s, const StencilArgs& a, const Scalar* ecor, const void* x, const void* b, void* out,
                          bool trans, bool restrict_, const int* flags, int sms) {
    using E = typename Tr<K>::E;
    const bool three = a.dim == 3;
    const int64_t work = restrict_ ? (a.nx / 2) * (a.ny / 2) * (three ? a.nz / 2 : 1) : a.nx * a.ny * a.nz;
    int64_t nb = (work + 255) / 256;
    if (nb < 1) nb = 1;
    if (nb > (int64_t)sms * 32) nb = (int64_t)sms * 32;
    if (restrict_) {
        Edge3<E> ed;
        for (int d = 0; d < 3; ++d) from_scalar(ecor[1 << d], ed.c[d]);
        k_mg_restrict<K><<<(int)nb, 256, 0, s>>>((const E*)x, (const E*)b, (E*)out, a.nx, a.ny, a.nz, three, stencil_coef<E>(a, trans),
                                                  ed, flags);
    } else {
        k_mg_prolong<K><<<(int)nb, 256, 0, s>>>((E*)out, (const E*)x, a.nx, a.ny, a.nz, three, flags);
    }
}
void launch_mg_restrict(int kind, cudaStream_t s, const StencilArgs& a, const Scalar* ecor, const void* x, const void* b, void* bc,
                        bool trans, const int* flags, int sms) {
    switch (kind) {
        case KS: mg_transfer_t<KS>(s, a, ecor, x, b, bc, trans, true, flags, sms); break;
        case KD: mg_transfer_t<KD>(s, a, ecor, x, b, bc, trans, true, flags, sms); break;
        case KC: mg_transfer_t<KC>(s, a, ecor, x, b, bc, trans, true, flags, sms); break;
        default: mg_transfer_t<KZ>(s, a, ecor, x, b, bc, trans, true, flags, sms); break;
    }
}
void launch_mg_prolong(int kind, cudaStream_t s, const StencilArgs& a, const void* e, void* x, const int* flags, int sms) {
    switch (kind) {
        case KS: mg_transfer_t<KS>(s, a, nullptr, e, nullptr, x, false, false, flags, sms); break;
        case KD: mg_transfer_t<KD>(s, a, nullptr, e, nullptr, x, false, false, flags, sms); break;
        case KC: mg_transfer_t<KC>(s, a, nullptr, e, nullptr, x, false, false, flags, sms); break;
        default: mg_transfer_t<KZ>(s, a, nullptr, e, nullptr, x, false, false, flags, sms); break;
    }
}

// ------------------------------------------------------------------------------------------
// Halo exchange over NVLink peer memory, fused with its synchronisation: replaces the
// ncclSend/ncclRecv group in front of the stencil.  Every CTA copies a slice of the boundary rows
// straight into the neighbours' (CUDA-IPC mapped) halo buffers; the last CTA to finish raises this
// rank's epoch flag in both neighbours and waits for theirs, so when the kernel retires the local
// halo buffers of the current parity are complete.  Buffers alternate by epoch parity: a neighbour
// can push for matvec m+1 only after it saw my push for matvec m, i.e. after I finished matvec m-1,
// the last reader of that parity.
template <int K>
__global__ void __launch_bounds__(256)
k_halo_push(HaloP2P h, const typename Tr<K>::E* __restrict__ x, int64_t n_loc, const int* __restrict__ flags)
{
    using E = typename Tr<K>::E;
    if (flags && flags[F_STOP]) return;
    __shared__ bool is_last;
    const unsigned ep = *h.epoch + 1u;
    const size_t par = (size_t)(ep & 1u) * 2 * h.side_bytes;
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    const int64_t t0 = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (h.lo_region) {      // my first row/plane -> lower neighbour's halo_hi (side 1)
        E* dst = reinterpret_cast<E*>(h.lo_region + h.data_off + par + h.side_bytes);
        for (int64_t i = t0; i < h.he; i += stride) dst[i] = x[i];
    }
    if (h.hi_region) {      // my last row/plane -> upper neighbour's halo_lo (side 0)
        E* dst = reinterpret_cast<E*>(h.hi_region + h.data_off + par);
        const E* src = x + (n_loc - h.he);
        for (int64_t i = t0; i < h.he; i += stride) dst[i] = src[i];
    }
    __threadfence_system();
    __syncthreads();
    if (threadIdx.x == 0) is_last = (atomicAdd(h.ticket, 1u) == gridDim.x - 1u);
    __syncthreads();
    if (is_last && threadIdx.x == 0) {
        __threadfence_system();
        if (h.lo_region) st_volatile_u32(reinterpret_cast<unsigned*>(h.lo_region + 128), ep);   // "upper neighbour pushed"
        if (h.hi_region) st_volatile_u32(reinterpret_cast<unsigned*>(h.hi_region), ep);         // "lower neighbour pushed"
        if (h.lo_region) spin_until(reinterpret_cast<const unsigned*>(h.my_region), ep);
        if (h.hi_region) spin_until(reinterpret_cast<const unsigned*>(h.my_region + 128), ep);
        __threadfence_system();
        *h.ticket = 0u;
        *h.epoch = ep;
    }
}
void launch_halo_push(int kind, cudaStream_t s, const HaloP2P& h, const void* x, int64_t n_loc, const int* flags) {
    int nb = (int)((h.he + 2047) / 2048);
    if (nb < 1) nb = 1;
    if (nb > 64) nb = 64;
    switch (kind) {
        case KS: k_halo_push<KS><<<nb, 256, 0, s>>>(h, (const float*)x, n_loc, flags); break;
        case KD: k_halo_push<KD><<<nb, 256, 0, s>>>(h, (const double*)x, n_loc, flags); break;
        case KC: k_halo_push<KC><<<nb, 256, 0, s>>>(h, (const float2*)x, n_loc, flags); break;
        default: k_halo_push<KZ><<<nb, 256, 0, s>>>(h, (const double2*)x, n_loc, flags); break;
    }
}

// ------------------------------------------------------------------------------------------
// CSR SpMV.  LPR lanes cooperate on one row (LPR = 32: warp-per-row; LPR < 32: vector-per-row
// for short rows).  Fixed shuffle tree => deterministic.  rmatvec uses an explicit transposed
// copy built at operator creation (no atomics), with conj_vals for A^H.
// ------------------------------------------------------------------------------------------
template <int K, int LPR>
__global__ void __launch_bounds__(256)
k_csr(int64_t m, const int64_t* __restrict__ rowptr, const int32_t* __restrict__ col,
      const typename Tr<K>::E* __restrict__ val, const typename Tr<K>::E* __restrict__ x,
      typename Tr<K>::E* __restrict__ y, bool conj_vals, const int* __restrict__ flags)
{
    using E = typename Tr<K>::E;
    if (flags && flags[F_STOP]) return;
    const int sub = threadIdx.x % LPR;
    const int64_t rows_per_cta = 256 / LPR;
    for (int64_t row = (int64_t)blockIdx.x * rows_per_cta + threadIdx.x / LPR; row < m;
         row += (int64_t)gridDim.x * rows_per_cta) {
        const int64_t q0 = rowptr[row], q1 = rowptr[row + 1];
        E acc = zero_v(E());
        for (int64_t q = q0 + sub; q < q1; q += LPR) {
            E a = __ldg(val + q);
            if (conj_vals) a = conj_v(a);
            fmacc(acc, a, __ldg(x + __ldg(col + q)));
        }
        typename Tr<K>::W wv = widen(acc);
#pragma unroll
        for (int o = LPR / 2; o > 0; o >>= 1) {
            if constexpr (Tr<K>::cplx) {
                wv.x += __shfl_down_sync(0xffffffffu, wv.x, o, LPR);
                wv.y += __shfl_down_sync(0xffffffffu, wv.y, o, LPR);
            } else {
                wv += __shfl_down_sync(0xffffffffu, wv, o, LPR);
            }
        }
        if (sub == 0) { E r; narrow(wv, r); y[row] = r; }
    }
}

template <int K>
static void csr_t(cudaStream_t s, int64_t m, const int64_t* rowptr, const int32_t* col, const void* val,
                  const void* x, void* y, bool conj_vals, const int* flags, int sms, int lpr) {
    using E = typename Tr<K>::E;
    auto grid = [&](int L) { int64_t nb = (m * L + 255) / 256; if (nb < 1) nb = 1; if (nb > (int64_t)sms * 16) nb = (int64_t)sms * 16; return (int)nb; };
    if (lpr >= 32)      k_csr<K, 32><<<grid(32), 256, 0, s>>>(m, rowptr, col, (const E*)val, (const E*)x, (E*)y, conj_vals, flags);
    else if (lpr >= 16) k_csr<K, 16><<<grid(16), 256, 0, s>>>(m, rowptr, col, (const E*)val, (const E*)x, (E*)y, conj_vals, flags);
    else if (lpr >= 8)  k_csr<K, 8><<<grid(8), 256, 0, s>>>(m, rowptr, col, (const E*)val, (const E*)x, (E*)y, conj_vals, flags);
    else                k_csr<K, 4><<<grid(4), 256, 0, s>>>(m, rowptr, col, (const E*)val, (const E*)x, (E*)y, conj_vals, flags);
}
// lanes per row are chosen by the caller from the average row length and passed in `sms >> 16`
void launch_csr(int kind, cudaStream_t s, int64_t m, const int64_t* rowptr, const int32_t* col, const void* val,
                const void* x, void* y, bool conj_vals, const int* flags, int sms_lpr) {
    const int sms = sms_lpr & 0xffff, lpr = sms_lpr >> 16;
    switch (kind) {
        case KS: csr_t<KS>(s, m, rowptr, col, val, x, y, conj_vals, flags, sms, lpr); break;
        case KD: csr_t<KD>(s, m, rowptr, col, val, x, y, conj_vals, flags, sms, lpr); break;
        case KC: csr_t<KC>(s, m, rowptr, col, val, x, y, conj_vals, flags, sms, lpr); break;
        default: csr_t<KZ>(s, m, rowptr, col, val, x, y, conj_vals, flags, sms, lpr); break;
    }
}

// ------------------------------------------------------------------------------------------
// L2-blocked CSR SpMV (layout: lkb_csr.cu).  One launch per column block; thread-per-row (a row has ~nnz/nb entries
// in a block: 1-3 for C5), consecutive threads read consecutive table entries and nearly consecutive values.
// The x gathers of a block all fall into one L2-resident slice and carry an L2 evict_last policy; the streamed
// operands (table, col, val) carry evict_normal.
// Why this kernel (B200, full-size C5 matrix, 48 MB slices, matvec ms per sweep, profiles/spmv_ab.py): 16.4 ms
// (profiles/r02_spmv_ab3_persistL2.jsonl), bandwidth-bound on its actual traffic (ncu: DRAM 6.9 GB per block at
// 5.3 TB/s, of which ~3 GB are x-gather sectors that missed L2; profiles/r02_ncu_summary.md).  Measured slower:
//   the same kernel with evict_first streams                              17.2 ms  (profiles/r02_spmv_ab2.jsonl)
//   CSR-stream: coalesced col / val runs per CTA, products staged in      19.5 ms  (profiles/r02_spmv_ab2.jsonl)
//     shared memory; latency-bound at 64 registers, 4 CTAs / SM
//   warp-pipelined CSR-stream (cp.async-staged col / val, no barrier)     20.7 ms  (profiles/r02_spmv_ab4_warp_pipelined.jsonl)
// All stream forms land at 19-21 ms whatever hides the col / val latency: the L2 gather rate (~100 G sectors/s), not the
// streams, is what they wait for.  A persisting-L2 set-aside (64 / 79 MB) changed none of them by more than 2 %.
LKB_DI uint64_t l2_policy_evict_normal() { uint64_t p; asm volatile("createpolicy.fractional.L2::evict_normal.b64 %0, 1.0;" : "=l"(p)); return p; }
template <typename T> LKB_DI T ld_hint(const T* p, uint64_t pol);
template <> LKB_DI float ld_hint<float>(const float* p, uint64_t pol) {
    float v; asm volatile("ld.global.nc.L2::cache_hint.f32 %0, [%1], %2;" : "=f"(v) : "l"(p), "l"(pol)); return v; }
template <> LKB_DI double ld_hint<double>(const double* p, uint64_t pol) {
    double v; asm volatile("ld.global.nc.L2::cache_hint.f64 %0, [%1], %2;" : "=d"(v) : "l"(p), "l"(pol)); return v; }
template <> LKB_DI float2 ld_hint<float2>(const float2* p, uint64_t pol) {
    float2 v; asm volatile("ld.global.nc.L2::cache_hint.v2.f32 {%0, %1}, [%2], %3;" : "=f"(v.x), "=f"(v.y) : "l"(p), "l"(pol)); return v; }
template <> LKB_DI double2 ld_hint<double2>(const double2* p, uint64_t pol) {
    double2 v; asm volatile("ld.global.nc.L2::cache_hint.v2.f64 {%0, %1}, [%2], %3;" : "=d"(v.x), "=d"(v.y) : "l"(p), "l"(pol)); return v; }
template <> LKB_DI int32_t ld_hint<int32_t>(const int32_t* p, uint64_t pol) {
    int32_t v; asm volatile("ld.global.nc.L2::cache_hint.s32 %0, [%1], %2;" : "=r"(v) : "l"(p), "l"(pol)); return v; }
template <> LKB_DI uint32_t ld_hint<uint32_t>(const uint32_t* p, uint64_t pol) {
    uint32_t v; asm volatile("ld.global.nc.L2::cache_hint.u32 %0, [%1], %2;" : "=r"(v) : "l"(p), "l"(pol)); return v; }

template <int K>
__global__ void __launch_bounds__(256)
k_csr_blocked(int64_t rows, const uint32_t* __restrict__ tab, const int32_t* __restrict__ col,
              const typename Tr<K>::E* __restrict__ val, const typename Tr<K>::E* __restrict__ x,
              typename Tr<K>::E* __restrict__ y, bool conj_vals, bool first, const int* __restrict__ flags)
{
    using E = typename Tr<K>::E;
    if (flags && flags[F_STOP]) return;
    const uint64_t keep = pol_evict_last(), stream = l2_policy_evict_normal();
    for (int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; r < rows; r += (int64_t)gridDim.x * blockDim.x) {
        const uint32_t q0 = ld_hint<uint32_t>(tab + r, stream), q1 = ld_hint<uint32_t>(tab + r + 1, stream);
        if (q0 == q1 && !first) continue;                       // nothing in this block for row r
        E acc = first ? zero_v(E()) : y[r];
        for (uint32_t q = q0; q < q1; ++q) {
            E a = ld_hint<E>(val + q, stream);
            if (conj_vals) a = conj_v(a);
            fmacc(acc, a, ld_hint<E>(x + ld_hint<int32_t>(col + q, stream), keep));
        }
        y[r] = acc;
    }
}
void launch_csr_blocked(int kind, cudaStream_t s, const CsrBlocked& b, const void* x, void* y, bool conj_vals, const int* flags, int sms) {
    int64_t nb = (b.rows + 255) / 256;
    if (nb < 1) nb = 1;
    if (nb > (int64_t)sms * 16) nb = (int64_t)sms * 16;
    for (int blk = 0; blk < b.nb; ++blk) {
        const uint32_t* tab = b.tab + (size_t)blk * (b.rows + 1);
        switch (kind) {
            case KS: k_csr_blocked<KS><<<(int)nb, 256, 0, s>>>(b.rows, tab, b.col, (const float*)b.val, (const float*)x, (float*)y, conj_vals, blk == 0, flags); break;
            case KD: k_csr_blocked<KD><<<(int)nb, 256, 0, s>>>(b.rows, tab, b.col, (const double*)b.val, (const double*)x, (double*)y, conj_vals, blk == 0, flags); break;
            case KC: k_csr_blocked<KC><<<(int)nb, 256, 0, s>>>(b.rows, tab, b.col, (const float2*)b.val, (const float2*)x, (float2*)y, conj_vals, blk == 0, flags); break;
            default: k_csr_blocked<KZ><<<(int)nb, 256, 0, s>>>(b.rows, tab, b.col, (const double2*)b.val, (const double2*)x, (double2*)y, conj_vals, blk == 0, flags); break;
        }
    }
}

// ------------------------------------------------------------------------------------------
// Jacobi preconditioner (set-up, once per operator): d_r = 1 / A_rr, the diagonal found the way each operator stores it.
//   stencil       the centre coefficient on every row
//   csr           the sum of the row's entries at column col0 + r (duplicates summed, as k_csr sums them)
//   blocked csr   the same, scanning only the column block that holds col0 + r (tab gives the row's range in it)
//   dense         a[r + rows * r]
//   diagonal      the operator's own d
// The diagonal is formed in W precision and inverted there; a zero or non-finite entry lowers *bad_row to its global row.
LKB_DI bool finite_nonzero(double a) { return isfinite(a) && a != 0.0; }
LKB_DI bool finite_nonzero(double2 a) { return isfinite(a.x) && isfinite(a.y) && (a.x != 0.0 || a.y != 0.0); }
LKB_DI double recip_w(double a) { return 1.0 / a; }
LKB_DI double2 recip_w(double2 a) { const double q = a.x * a.x + a.y * a.y; return make_double2(a.x / q, -a.y / q); }

template <int K, int MODE>
__global__ void __launch_bounds__(256)
k_jacobi(const JacobiSrc src, typename Tr<K>::E* __restrict__ d, unsigned long long* __restrict__ bad_row)
{
    using E = typename Tr<K>::E;
    using W = typename Tr<K>::W;
    const E* val = (const E*)src.val;
    for (int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; r < src.rows; r += (int64_t)gridDim.x * blockDim.x) {
        W a = zero_v(W());
        if constexpr (MODE == JAC_STENCIL) {
            E c; from_scalar(src.c0, c); a = widen(c);
        } else if constexpr (MODE == JAC_CSR) {
            const int64_t cr = src.col0 + r;
            for (int64_t q = src.rowptr[r]; q < src.rowptr[r + 1]; ++q)
                if (src.col[q] == cr) wadd(a, widen(val[q]));
        } else if constexpr (MODE == JAC_CSR_BLOCKED) {
            const int64_t cr = src.col0 + r;
            const uint32_t* tab = src.blk.tab + (size_t)(cr / src.blk.cw) * (src.rows + 1);
            const E* bval = (const E*)src.blk.val;
            for (uint32_t q = tab[r]; q < tab[r + 1]; ++q)
                if (src.blk.col[q] == cr) wadd(a, widen(bval[q]));
        } else if constexpr (MODE == JAC_DENSE) {
            a = widen(((const E*)src.a)[r * (src.rows + 1)]);
        } else {
            a = widen(((const E*)src.a)[r]);
        }
        if (finite_nonzero(a)) narrow(recip_w(a), d[r]);
        else atomicMin(bad_row, (unsigned long long)(src.row0 + r));
    }
}
template <int K>
static void jacobi_t(cudaStream_t s, const JacobiSrc& src, void* d, unsigned long long* bad, int sms) {
    using E = typename Tr<K>::E;
    int64_t nb = (src.rows + 255) / 256;
    if (nb < 1) nb = 1;
    if (nb > (int64_t)sms * 16) nb = (int64_t)sms * 16;
    switch (src.mode) {
        case JAC_STENCIL: k_jacobi<K, JAC_STENCIL><<<(int)nb, 256, 0, s>>>(src, (E*)d, bad); break;
        case JAC_CSR: k_jacobi<K, JAC_CSR><<<(int)nb, 256, 0, s>>>(src, (E*)d, bad); break;
        case JAC_CSR_BLOCKED: k_jacobi<K, JAC_CSR_BLOCKED><<<(int)nb, 256, 0, s>>>(src, (E*)d, bad); break;
        case JAC_DENSE: k_jacobi<K, JAC_DENSE><<<(int)nb, 256, 0, s>>>(src, (E*)d, bad); break;
        default: k_jacobi<K, JAC_DIAG><<<(int)nb, 256, 0, s>>>(src, (E*)d, bad); break;
    }
}
void launch_jacobi(int kind, cudaStream_t s, const JacobiSrc& src, void* d, unsigned long long* bad_row, int sms) {
    switch (kind) {
        case KS: jacobi_t<KS>(s, src, d, bad_row, sms); break;
        case KD: jacobi_t<KD>(s, src, d, bad_row, sms); break;
        case KC: jacobi_t<KC>(s, src, d, bad_row, sms); break;
        default: jacobi_t<KZ>(s, src, d, bad_row, sms); break;
    }
}

// Gershgorin bound of D^-1 A (Chebyshev preconditioner set-up, once per operator): max over the rows of
// sum_c |a_rc| / |a_rr|, each a_rc the sum of the row's entries at column c (duplicates summed, as the SpMV sums them), in
// double.  The max of non-negative doubles is exact in any order, so one atomicMax on their bit patterns per warp gives a
// deterministic result.  Rows whose diagonal entry is zero or not finite are skipped: k_jacobi reports them.
LKB_DI double abs_w(double a) { return fabs(a); }
LKB_DI double abs_w(double2 a) { return hypot(a.x, a.y); }
LKB_DI double2 w2(double a) { return make_double2(a, 0.0); }
LKB_DI double2 w2(double2 a) { return a; }
// sum over the distinct columns of entries [q0, q1) of |sum of the entries at that column|; dg = the entry sum at column cr
template <typename E, typename Q>
LKB_DI double row_abs_sum(const int32_t* col, const E* val, Q q0, Q q1, int64_t cr, double2& dg) {
    bool sorted = true;
    for (Q q = q0 + 1; q < q1; ++q) sorted = sorted && col[q - 1] <= col[q];
    double sum = 0.0;
    for (Q q = q0; q < q1;) {
        const int32_t cq = col[q];
        auto a = widen(val[q]);
        Q next = q + 1;
        if (sorted) {
            for (; next < q1 && col[next] == cq; ++next) wadd(a, widen(val[next]));
        } else {
            bool seen = false;
            for (Q p = q0; p < q && !seen; ++p) seen = col[p] == cq;
            if (seen) { q = next; continue; }
            for (Q p = next; p < q1; ++p) if (col[p] == cq) wadd(a, widen(val[p]));
        }
        sum += abs_w(a);
        if (cq == cr) dg = w2(a);
        q = next;
    }
    return sum;
}
template <int K, int MODE>
__global__ void __launch_bounds__(256)
k_gershgorin(const JacobiSrc src, unsigned long long* __restrict__ bound_bits)
{
    using E = typename Tr<K>::E;
    double best = 0.0;
    for (int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; r < src.rows; r += (int64_t)gridDim.x * blockDim.x) {
        const int64_t cr = src.col0 + r;
        double2 dg = make_double2(0.0, 0.0);
        double sum = 0.0;
        if constexpr (MODE == JAC_CSR) {
            sum = row_abs_sum((const int32_t*)src.col, (const E*)src.val, src.rowptr[r], src.rowptr[r + 1], cr, dg);
        } else if constexpr (MODE == JAC_CSR_BLOCKED) {
            for (int b = 0; b < src.blk.nb; ++b) {
                const uint32_t* tab = src.blk.tab + (size_t)b * (src.rows + 1);
                sum += row_abs_sum((const int32_t*)src.blk.col, (const E*)src.blk.val, tab[r], tab[r + 1], cr, dg);
            }
        } else {      // dense, column-major rows x rows
            const E* a = (const E*)src.a;
            for (int64_t c = 0; c < src.rows; ++c) sum += abs_w(widen(a[r + src.rows * c]));
            dg = w2(widen(a[r * (src.rows + 1)]));
        }
        const double ad = hypot(dg.x, dg.y);
        if (isfinite(ad) && ad != 0.0) best = fmax(best, sum / ad);
    }
    unsigned long long bits = (unsigned long long)__double_as_longlong(best);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) bits = max(bits, __shfl_xor_sync(0xffffffffu, bits, o));
    if ((threadIdx.x & 31) == 0) atomicMax(bound_bits, bits);
}
template <int K>
static void gershgorin_t(cudaStream_t s, const JacobiSrc& src, unsigned long long* bound_bits, int sms) {
    int64_t nb = (src.rows + 255) / 256;
    if (nb < 1) nb = 1;
    if (nb > (int64_t)sms * 16) nb = (int64_t)sms * 16;
    switch (src.mode) {
        case JAC_CSR: k_gershgorin<K, JAC_CSR><<<(int)nb, 256, 0, s>>>(src, bound_bits); break;
        case JAC_CSR_BLOCKED: k_gershgorin<K, JAC_CSR_BLOCKED><<<(int)nb, 256, 0, s>>>(src, bound_bits); break;
        default: k_gershgorin<K, JAC_DENSE><<<(int)nb, 256, 0, s>>>(src, bound_bits); break;
    }
}
void launch_gershgorin(int kind, cudaStream_t s, const JacobiSrc& src, unsigned long long* bound_bits, int sms) {
    switch (kind) {
        case KS: gershgorin_t<KS>(s, src, bound_bits, sms); break;
        case KD: gershgorin_t<KD>(s, src, bound_bits, sms); break;
        case KC: gershgorin_t<KC>(s, src, bound_bits, sms); break;
        default: gershgorin_t<KZ>(s, src, bound_bits, sms); break;
    }
}

// ------------------------------------------------------------------------------------------
// dense_linop (AbstractLinops.fypp:608-671, gemv): only the n = 128 plumbing config uses it.
template <int K>
__global__ void k_dense(int64_t m, int64_t n, const typename Tr<K>::E* __restrict__ a,
                        const typename Tr<K>::E* __restrict__ x, typename Tr<K>::E* __restrict__ y, bool trans,
                        const int* __restrict__ flags)
{
    using E = typename Tr<K>::E;
    if (flags && flags[F_STOP]) return;
    if (!trans) {
        for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < m; i += (int64_t)gridDim.x * blockDim.x) {
            E s = zero_v(E());
            for (int64_t j = 0; j < n; ++j) fmacc(s, a[i + m * j], x[j]);
            y[i] = s;
        }
    } else {
        // one warp per output column
        const int lane = threadIdx.x & 31;
        for (int64_t j = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5; j < n; j += ((int64_t)gridDim.x * blockDim.x) >> 5) {
            E s = zero_v(E());
            for (int64_t i = lane; i < m; i += 32) fma_conj(s, a[i + m * j], x[i]);
            typename Tr<K>::W wv = warp_sum(widen(s));
            if (lane == 0) { E r; narrow(wv, r); y[j] = r; }
        }
    }
}
void launch_dense(int kind, cudaStream_t s, int64_t m, int64_t n, const void* a, const void* x, void* y, bool trans,
                  const int* flags) {
    const int64_t work = trans ? n * 32 : m;
    int nb = (int)((work + 127) / 128); if (nb < 1) nb = 1; if (nb > 4096) nb = 4096;
    switch (kind) {
        case KS: k_dense<KS><<<nb, 128, 0, s>>>(m, n, (const float*)a, (const float*)x, (float*)y, trans, flags); break;
        case KD: k_dense<KD><<<nb, 128, 0, s>>>(m, n, (const double*)a, (const double*)x, (double*)y, trans, flags); break;
        case KC: k_dense<KC><<<nb, 128, 0, s>>>(m, n, (const float2*)a, (const float2*)x, (float2*)y, trans, flags); break;
        default: k_dense<KZ><<<nb, 128, 0, s>>>(m, n, (const double2*)a, (const double2*)x, (double2*)y, trans, flags); break;
    }
}

}  // namespace lkb
