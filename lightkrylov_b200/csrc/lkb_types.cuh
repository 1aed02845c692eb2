// lkb_types.cuh -- element traits for the four LightKrylov kinds (rsp, rdp, csp, cdp).
//
// The reference instantiates every routine over (rsp, rdp, csp, cdp) with fypp
// (/root/reference/include/common.fypp:19-46).  Here the same four kinds are one template
// parameter K; every kernel moves data in 16-byte packs (128-bit loads/stores) holding
// EPP elements of kind K.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace lkb {

enum Kind : int { KS = 0, KD = 1, KC = 2, KZ = 3 };

template <int K> struct Tr;
template <> struct Tr<KS> { using E = float;   using Rl = float;  using W = double;  static constexpr int EPP = 4; static constexpr bool cplx = false; };
template <> struct Tr<KD> { using E = double;  using Rl = double; using W = double;  static constexpr int EPP = 2; static constexpr bool cplx = false; };
template <> struct Tr<KC> { using E = float2;  using Rl = float;  using W = double2; static constexpr int EPP = 2; static constexpr bool cplx = true; };
template <> struct Tr<KZ> { using E = double2; using Rl = double; using W = double2; static constexpr int EPP = 1; static constexpr bool cplx = true; };

static inline size_t kind_size(int k) { return k == KS ? 4 : (k == KZ ? 16 : 8); }
static inline int kind_epp(int k) { return k == KS ? 4 : (k == KZ ? 1 : 2); }
static inline bool kind_cplx(int k) { return k >= KC; }

#define LKB_DI __device__ __forceinline__

// Programmatic dependent launch (PDL): a kernel launched with cudaLaunchAttributeProgrammaticStreamSerialization may
// start while its predecessor in the stream is still draining.  pdl_wait() blocks until every predecessor grid has
// COMPLETED and its memory is visible (no-op for a normally launched kernel); pdl_trigger() lets the runtime launch
// this kernel's own dependent once all CTAs have executed it.  Every PDL-aware kernel here runs
//     [work that touches nothing the predecessor writes]  pdl_wait();  pdl_trigger();  [everything else]
// so a dependent's pre-wait code only ever runs once the predecessor's predecessor is complete.
#if defined(__CUDACC__)
LKB_DI void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
LKB_DI void pdl_trigger() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }
#endif
#define LKB_HDI __host__ __device__ __forceinline__

// ---- scalar algebra, overloaded on the element type ---------------------------------------
LKB_HDI float   zero_v(float)   { return 0.f; }
LKB_HDI double  zero_v(double)  { return 0.0; }
LKB_HDI float2  zero_v(float2)  { return make_float2(0.f, 0.f); }
LKB_HDI double2 zero_v(double2) { return make_double2(0.0, 0.0); }

// a += conj(v) * w     (dot(self, vec) conjugates self: AbstractVectors.fypp:548-551)
LKB_DI void fma_conj(float& a, float v, float w)    { a = fmaf(v, w, a); }
LKB_DI void fma_conj(double& a, double v, double w) { a = fma(v, w, a); }
LKB_DI void fma_conj(float2& a, float2 v, float2 w) {
    a.x = fmaf(v.x, w.x, a.x); a.x = fmaf(v.y, w.y, a.x);
    a.y = fmaf(v.x, w.y, a.y); a.y = fmaf(-v.y, w.x, a.y);
}
LKB_DI void fma_conj(double2& a, double2 v, double2 w) {
    a.x = fma(v.x, w.x, a.x); a.x = fma(v.y, w.y, a.x);
    a.y = fma(v.x, w.y, a.y); a.y = fma(-v.y, w.x, a.y);
}
// a -= v * c
LKB_DI void fnma(float& a, float v, float c)    { a = fmaf(-v, c, a); }
LKB_DI void fnma(double& a, double v, double c) { a = fma(-v, c, a); }
LKB_DI void fnma(float2& a, float2 v, float2 c) {
    a.x = fmaf(-v.x, c.x, a.x); a.x = fmaf(v.y, c.y, a.x);
    a.y = fmaf(-v.x, c.y, a.y); a.y = fmaf(-v.y, c.x, a.y);
}
LKB_DI void fnma(double2& a, double2 v, double2 c) {
    a.x = fma(-v.x, c.x, a.x); a.x = fma(v.y, c.y, a.x);
    a.y = fma(-v.x, c.y, a.y); a.y = fma(-v.y, c.x, a.y);
}
// a += v * c
LKB_DI void fmacc(float& a, float v, float c)    { a = fmaf(v, c, a); }
LKB_DI void fmacc(double& a, double v, double c) { a = fma(v, c, a); }
LKB_DI void fmacc(float2& a, float2 v, float2 c) {
    a.x = fmaf(v.x, c.x, a.x); a.x = fmaf(-v.y, c.y, a.x);
    a.y = fmaf(v.x, c.y, a.y); a.y = fmaf(v.y, c.x, a.y);
}
LKB_DI void fmacc(double2& a, double2 v, double2 c) {
    a.x = fma(v.x, c.x, a.x); a.x = fma(-v.y, c.y, a.x);
    a.y = fma(v.x, c.y, a.y); a.y = fma(v.y, c.x, a.y);
}
LKB_HDI float   mul_v(float a, float b)   { return a * b; }
LKB_HDI double  mul_v(double a, double b) { return a * b; }
LKB_HDI float2  mul_v(float2 a, float2 b)   { return make_float2(a.x * b.x - a.y * b.y, a.x * b.y + a.y * b.x); }
LKB_HDI double2 mul_v(double2 a, double2 b) { return make_double2(a.x * b.x - a.y * b.y, a.x * b.y + a.y * b.x); }
LKB_HDI float   add_v(float a, float b)   { return a + b; }
LKB_HDI double  add_v(double a, double b) { return a + b; }
LKB_HDI float2  add_v(float2 a, float2 b)   { return make_float2(a.x + b.x, a.y + b.y); }
LKB_HDI double2 add_v(double2 a, double2 b) { return make_double2(a.x + b.x, a.y + b.y); }
LKB_HDI float   conj_v(float a)   { return a; }
LKB_HDI double  conj_v(double a)  { return a; }
LKB_HDI float2  conj_v(float2 a)  { return make_float2(a.x, -a.y); }
LKB_HDI double2 conj_v(double2 a) { return make_double2(a.x, -a.y); }
LKB_HDI float   rscale(float a, float r)    { return a * r; }
LKB_HDI double  rscale(double a, double r)  { return a * r; }
LKB_HDI float2  rscale(float2 a, float r)   { return make_float2(a.x * r, a.y * r); }
LKB_HDI double2 rscale(double2 a, double r) { return make_double2(a.x * r, a.y * r); }
LKB_HDI double abs2_w(float a)   { return (double)a * (double)a; }
LKB_HDI double abs2_w(double a)  { return a * a; }
LKB_HDI double abs2_w(float2 a)  { return (double)a.x * a.x + (double)a.y * a.y; }
LKB_HDI double abs2_w(double2 a) { return a.x * a.x + a.y * a.y; }
LKB_HDI bool is_zero_v(float a)   { return a == 0.f; }
LKB_HDI bool is_zero_v(double a)  { return a == 0.0; }
LKB_HDI bool is_zero_v(float2 a)  { return a.x == 0.f && a.y == 0.f; }
LKB_HDI bool is_zero_v(double2 a) { return a.x == 0.0 && a.y == 0.0; }

// One step of the GMRES-polynomial preconditioner (lkb_poly.cu) on the matvec input x, its image t = (A x)_i and a held
// vector v:  out = a0 x + a1 t + a2 v ;  acc = [acc] + b0 x + b1 t + b2 v.  Shared by the fused stencil epilogue
// (kernels_ops.cu) and k_poly_update (kernels_vec.cu), so both paths round alike.
template <typename E> struct PolyCoef { E a[3], b[3]; };
template <typename E> LKB_DI E poly_comb(E x, E t, E v, E c0, E c1, E c2) {
    E s = mul_v(c0, x);
    fmacc(s, t, c1);
    fmacc(s, v, c2);
    return s;
}

// widen element -> reduction type W, and narrow back
LKB_HDI double  widen(float a)   { return (double)a; }
LKB_HDI double  widen(double a)  { return a; }
LKB_HDI double2 widen(float2 a)  { return make_double2(a.x, a.y); }
LKB_HDI double2 widen(double2 a) { return a; }
LKB_HDI void narrow(double a, float& o)   { o = (float)a; }
LKB_HDI void narrow(double a, double& o)  { o = a; }
LKB_HDI void narrow(double2 a, float2& o)  { o = make_float2((float)a.x, (float)a.y); }
LKB_HDI void narrow(double2 a, double2& o) { o = a; }
LKB_HDI void wadd(double& a, double b)   { a += b; }
LKB_HDI void wadd(double2& a, double2 b) { a.x += b.x; a.y += b.y; }
LKB_HDI double wreal(double a)  { return a; }
LKB_HDI double wreal(double2 a) { return a.x; }

// host scalar container used across the C ABI: always {re, im} in double
struct Scalar { double re, im; };
LKB_HDI void from_scalar(Scalar s, float& o)   { o = (float)s.re; }
LKB_HDI void from_scalar(Scalar s, double& o)  { o = s.re; }
LKB_HDI void from_scalar(Scalar s, float2& o)  { o = make_float2((float)s.re, (float)s.im); }
LKB_HDI void from_scalar(Scalar s, double2& o) { o = make_double2(s.re, s.im); }

// ---- 16-byte packs ---------------------------------------------------------------------------
template <typename E, int EPP> struct alignas(16) Pack { E v[EPP]; };

// Streaming 128-bit loads.  Every Gram-Schmidt / vector kernel reads each byte exactly once, so an L1 line allocated
// for it is pure overhead: with L1::no_allocate the multi-dot / multi-axpy kernels run 4-5 % faster at the per-GPU
// share of N = 8 (measured round 2, profiles/r02_pdl3.sh: 1828 -> 1917 Arnoldi steps/s at 4096 x 512) and no longer
// depend on the SM's L1 / shared-memory carve-out (a max-shared carve-out cost the allocating version 11 %).
// ld_pack_l1 keeps the allocating read-only path for the stencils, whose x-neighbours are re-read through L1.
template <typename P> LKB_DI P ld_pack_l1(const void* p) {   // read-only path with L1 allocation (LDG.E.128.CONSTANT)
    int4 r = __ldg(reinterpret_cast<const int4*>(p));
    return *reinterpret_cast<P*>(&r);
}
template <typename P> LKB_DI P ld_pack_nc(const void* p) {   // read-only streaming path, no L1 allocation
#ifdef LKB_L1_ALLOC
    return ld_pack_l1<P>(p);
#else
    int4 r;
    // (an additional L2::256B prefetch-size hint was measured neutral: 1917 vs 1909 steps/s at 4096 x 512, profiles/r02_l2hint.sh)
    asm volatile("ld.global.nc.L1::no_allocate.v4.s32 {%0, %1, %2, %3}, [%4];" : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w) : "l"(p));
    return *reinterpret_cast<P*>(&r);
#endif
}
template <typename P> LKB_DI P ld_pack(const void* p) {      // coherent streaming load (the vector is rewritten by this kernel)
#ifdef LKB_L1_ALLOC
    int4 r = *reinterpret_cast<const int4*>(p);
#else
    int4 r;
    asm volatile("ld.global.L1::no_allocate.v4.s32 {%0, %1, %2, %3}, [%4];" : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w) : "l"(p) : "memory");
#endif
    return *reinterpret_cast<P*>(&r);
}
// Accesses of the WORK VECTOR w of a Krylov step.  When a GPU's slice of w is small (<= W_KEEP_BYTES = 48 MB: the
// 1/4 and 1/8 shares of C2) every access of w carries an L2 evict_last policy, so w survives the j columns of V that
// stream through L2 between its uses (matvec writes it, the multi-dot, the fused kernel and the final axpy read it):
// 4096 x 512 1917 -> 1943 steps/s (+1.4 %, the fused kernel +5 %).  At full size (134 MB per vector > L2) the hint costs
// 0.9 %, hence the size switch (profiles/r02_l2hint.sh with the -DLKB_W_EVICT_LAST experiment build, round 2; A/B of the
// threshold in profiles/r02_wkeep_result.txt).
constexpr size_t W_KEEP_BYTES = (size_t)48 << 20;
LKB_DI uint64_t pol_evict_last() { uint64_t p; asm volatile("createpolicy.fractional.L2::evict_last.b64 %0, 1.0;" : "=l"(p)); return p; }
template <typename P> LKB_DI P ld_pack_w(const void* p, bool keep, uint64_t pol) {          // coherent (w is rewritten by the kernel)
    if (!keep) return ld_pack<P>(p);
    int4 r;
    asm volatile("ld.global.L1::no_allocate.L2::cache_hint.v4.s32 {%0, %1, %2, %3}, [%4], %5;" : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w) : "l"(p), "l"(pol) : "memory");
    return *reinterpret_cast<P*>(&r);
}
template <typename P> LKB_DI P ld_pack_nc_w(const void* p, bool keep, uint64_t pol) {       // read-only
    if (!keep) return ld_pack_nc<P>(p);
    int4 r;
    asm volatile("ld.global.nc.L1::no_allocate.L2::cache_hint.v4.s32 {%0, %1, %2, %3}, [%4], %5;" : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w) : "l"(p), "l"(pol));
    return *reinterpret_cast<P*>(&r);
}
template <typename P> LKB_DI void st_pack_w(void* p, const P& v, bool keep, uint64_t pol) {
    if (!keep) { *reinterpret_cast<int4*>(p) = *reinterpret_cast<const int4*>(&v); return; }
    const int4 r = *reinterpret_cast<const int4*>(&v);
    asm volatile("st.global.L2::cache_hint.v4.s32 [%0], {%1, %2, %3, %4}, %5;" :: "l"(p), "r"(r.x), "r"(r.y), "r"(r.z), "r"(r.w), "l"(pol) : "memory");
}
template <typename P> LKB_DI void st_pack(void* p, const P& v) {
    *reinterpret_cast<int4*>(p) = *reinterpret_cast<const int4*>(&v);
}

LKB_DI double warp_sum(double a) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) a += __shfl_down_sync(0xffffffffu, a, o);
    return a;
}
LKB_DI double2 warp_sum(double2 a) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        a.x += __shfl_down_sync(0xffffffffu, a.x, o);
        a.y += __shfl_down_sync(0xffffffffu, a.y, o);
    }
    return a;
}

}  // namespace lkb
