// lkb_kernels.h -- host-callable launchers of the sm_100a kernels (kind-dispatched).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include "lkb_types.cuh"

namespace lkb {

// Device-side control block shared by all kernels of one Krylov process.
//   flags[0] stop      set when a breakdown was detected; kernels of later steps return at once
//   flags[1] info      step index (1-based) at which stop was raised
//   flags[2] refill    the new vector was numerically zero (< atol): host must rand-refill it
//   flags[3] nan       a norm evaluated to NaN (reference: stop_error, qr.fypp:139-145)
//   flags[4] gs_info   info of the last orthogonalize_against_basis pass (zero-vector check)
//   flags[5], flags[6] iteration counter / converged (device-resident cg and gmres cycles)
//   flags[7] scaled    k_multiaxpy_fin already normalised the new vector: the k_scale_dev that follows is a no-op
enum { F_STOP = 0, F_INFO = 1, F_REFILL = 2, F_NAN = 3, F_GSINFO = 4, F_SCALED = 7, F_COUNT = 8 };

enum { MD_CB = 16 };           // basis columns per multi-dot CTA
enum { MD_THREADS = 256 };
enum { MAX_ROWBLOCKS = 1024 }; // upper bound on stage-1 partial rows

// In-kernel allreduce over NVLink peer memory (one process per GPU, buffers mapped with CUDA IPC).
// Region layout per rank: flags[world] (one per 128 B line) | data[2][world][P2P_SLOT] (16-byte words).
enum { P2P_MAXW = 8, P2P_SLOT = 1040, P2P_FLAG_BYTES = 128 * P2P_MAXW };
struct P2P {
    int world = 1, rank = 0;
    unsigned* epoch = nullptr;          // device-side collective counter (identical on all ranks)
    char* peer[P2P_MAXW] = {nullptr};   // peer[r] = rank r's region as mapped in this process
    // in-kernel timeline (lkb_debug_ktime): [cta][4] = {start, main loop done, ticket taken, -} then
    // [4*MAX_ROWBLOCKS + {0,1,2}] = {stage-2 start, stage-2 done, allreduce done} of the last CTA (%globaltimer ns)
    unsigned long long* dbg = nullptr;
};
enum { KT_WORDS = 4 * 1024 + 16 };
static inline size_t p2p_region_bytes() { return (size_t)P2P_FLAG_BYTES + 2 * (size_t)P2P_MAXW * P2P_SLOT * 16; }

// cudaFuncAttributeMaxDynamicSharedMemorySize is a PER-DEVICE attribute: set it once for every device a kernel is
// launched on (a process may hold contexts on several GPUs), not once per process.
struct SmemAttrOnce {
    const void* fn; int bytes; mutable unsigned long long done = 0ULL;      // bit d = set on device d
    SmemAttrOnce(const void* f, int b) : fn(f), bytes(b) {}
    void ensure() const {
        int dev = 0;
        cudaGetDevice(&dev);
        const unsigned long long bit = 1ULL << (dev & 63);
        if (!(done & bit)) { cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes); done |= bit; }
    }
};

// ---- programmatic dependent launch (PDL) of the step-loop kernels ------------------------------------------
// The Krylov step loops chain 5 kernels per step whose tails (two-stage reduction, in-kernel allreduce) leave the GPU
// idle for 5-15 us; with PDL the next kernel's CTAs are scheduled as SMs drain, run their prologue (k_axpy_dot: fill
// the TMA ring) and block in griddepcontrol.wait until the predecessor has completed.  Host side: a per-thread state
// armed by the step loop (PdlScope); the launchers of PDL-aware kernels ask pdl_take().  State 1 = "armed": the next
// aware launch is a normal one (its predecessor in the stream is not one of our kernels: memset, NCCL, user
// callback), afterwards the chain is on.  pdl_rearm() after anything that is not a kernel of this library.
int& pdl_state();
// Kernel classes launched programmatically (bits: 1 matvec, 2 multi-dot, 4 fused axpy+dot, 8 multi-axpy, 16 scale): only
// the TMA kernel.  Measured on B200 (profiles/r02_pdl2.sh .. r02_pdl4.sh): a programmatically launched kernel inherits the
// predecessor's L1 / shared-memory carve-out, which costs the LDG-based multi-dot / multi-axpy kernels up to 11 %
// (4096 x 512: all classes 1729 steps/s, none 1870, fused only 1876); the TMA kernel is carve-out neutral and gains from
// filling its ring during the multi-dot's tail (reduction tree + NVLink allreduce).
constexpr int PDL_CLASSES = 4;
// cls: the class bit of the launching kernel
inline bool pdl_take(int cls = 0xff) { int& s = pdl_state(); if (s == 2) return (PDL_CLASSES & cls) != 0; if (s == 1) s = 2; return false; }
inline void pdl_rearm() { int& s = pdl_state(); if (s == 2) s = 1; }
struct PdlScope {
    int prev;
    explicit PdlScope(bool on) : prev(pdl_state()) { pdl_state() = on ? 1 : 0; }
    ~PdlScope() { pdl_state() = prev; }
};
// ---- serpentine sweeps (L2 reuse between consecutive kernels of a step) ---------------------------------------------
// The three Gram-Schmidt kernels of a step each stream V(:, 0:j) once.  All of them walk the rows as ONE global sweep
// (at any time every CTA works inside the same narrow band of rows), and consecutive kernels sweep in opposite
// directions: a kernel starts on the rows its predecessor read last, which are still L2-resident (126 MB L2: ~10 % of
// a kernel's bytes at the per-GPU share of N = 8, ~1 % at N = 1).  The direction is a pure function of the step index
// (dgs_enqueue), so results stay bitwise reproducible (graphs on / off, one-shot vs step-by-step, any launch timing).
int& sweep_dir();     // 0 ascending, 1 descending: read by launch_multidot / launch_axpy_dot / launch_multiaxpy_fin
struct SweepDir {
    int prev;
    explicit SweepDir(int d) : prev(sweep_dir()) { sweep_dir() = d; }
    ~SweepDir() { sweep_dir() = prev; }
};
template <typename... KArgs, typename... Args>
inline cudaError_t launch_ex(void (*kern)(KArgs...), unsigned grid, unsigned block, size_t smem, cudaStream_t s, bool pdl, Args&&... args) {
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(grid, 1, 1); cfg.blockDim = dim3(block, 1, 1); cfg.dynamicSmemBytes = smem; cfg.stream = s;
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    at[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = at; cfg.numAttrs = pdl ? 1u : 0u;
    return cudaLaunchKernelEx(&cfg, kern, static_cast<KArgs>(args)...);
}

struct StencilArgs {
    int64_t nx, ny, nz;        // local slab: nx fastest; the slowest axis is the sharded one
    Scalar coef[7];            // center, -x, +x, -y, +y, -z, +z
    const void* halo_lo;       // previous slab's last row/plane (nullptr = Dirichlet boundary)
    const void* halo_hi;       // next slab's first row/plane
    int dim;                   // 2 or 3
    // p2p halo exchange: halo_lo / halo_hi point at parity 0 of double-buffered regions; the kernel adds
    // (epoch & 1) * halo_parity_stride elements, epoch being the device counter of the push kernel
    const unsigned* halo_epoch = nullptr;
    int64_t halo_parity_stride = 0;
    // flags the neighbours raise in this rank's halo region ("lower / upper neighbour pushed epoch e"): the CTAs
    // that read a halo wait on them (see halo_wait in kernels_ops.cu)
    const unsigned* flag_lo = nullptr;
    const unsigned* flag_hi = nullptr;
};
// P2P halo push (kernels_ops.cu): my first / last `he` elements of x go straight into the neighbours' halo
// buffers over NVLink; the last CTA signals the neighbours and waits for their pushes.
struct HaloP2P {
    char* my_region = nullptr;      // flags[2] (128 B apart) then data[parity][side][he]
    char* lo_region = nullptr;      // rank-1's region (mapped), nullptr at the domain boundary
    char* hi_region = nullptr;      // rank+1's region
    unsigned* epoch = nullptr;      // device counter of pushes (same sequence on every rank)
    unsigned* ticket = nullptr;
    int64_t he = 0;                 // halo elements
    size_t data_off = 256, side_bytes = 0;   // layout
};
void launch_halo_push(int kind, cudaStream_t s, const HaloP2P& h, const void* x, int64_t n_loc, const int* flags);

// c[0..j) = V(:, 0:j)^H w, c[j] = w^H w.  Two-stage deterministic reduction; the last CTA to
// finish folds the stage-1 partials in fixed order into out[0..j].
void launch_multidot(int kind, cudaStream_t s, const void* V, int64_t ld, int j, const void* w, int64_t n,
                     void* partial, void* out, unsigned* counter, const int* flags, int sms, const P2P* p2p = nullptr);
// w -= V(:, 0:j) c ; optionally nrm2_out[0] = ||w_new||^2 (same two-stage scheme).
void launch_multiaxpy(int kind, cudaStream_t s, const void* V, int64_t ld, int j, const void* c, void* w, int64_t n,
                      bool want_norm, void* partial, void* nrm2_out, unsigned* counter, const int* flags, int sms,
                      const P2P* p2p = nullptr);
// Block Gram-Schmidt, two right-hand sides per sweep of V: out / c are laid out [2][j+1] (W type)
void launch_multidot2(int kind, cudaStream_t s, const void* V, int64_t ld, int j, const void* w0, const void* w1, int64_t n,
                      void* partial, void* out, unsigned* counter, const int* flags, int sms, const P2P* p2p = nullptr);
void launch_multiaxpy2(int kind, cudaStream_t s, const void* V, int64_t ld, int j, const void* c, void* w0, void* w1,
                       int64_t n, const int* flags, int sms);
// Fused pass-1 multi-axpy + pass-2 multi-dot (TMA + mbarrier pipeline, kernels_fused.cu):
//   w -= V c1 ; out[0..j) = V^H w_new ; out[j] = w_new^H w_new.   axpy_dot_supported is false when the shape is not
//   supported (j > 128, ragged n, unaligned, no tensor-map encoder) -- the caller then runs the two separate kernels.
//   launch_axpy_dot returns false, without launching, only when the driver rejects the tensor map: the same fallback.
bool axpy_dot_supported(int kind, const void* V, int64_t ld, int j, const void* w, int64_t n);
bool launch_axpy_dot(int kind, cudaStream_t s, const void* V, int64_t ld, int j, const void* c1, void* w, int64_t n,
                     void* partial, void* out, unsigned* counter, const int* flags, int sms, const P2P* p2p = nullptr);
// y = alpha*x + beta*y  (beta == 0: y is overwritten without being read)
void launch_axpby(int kind, cudaStream_t s, Scalar alpha, const void* x, Scalar beta, void* y, int64_t n, int sms);
// y = sgn * (*alpha_dev) * x + y   with alpha on the device (W type)
void launch_axpy_dev(int kind, cudaStream_t s, const void* alpha_dev, double sgn, const void* x, void* y, int64_t n,
                     const int* flags, int sms);
void launch_scal(int kind, cudaStream_t s, Scalar alpha, void* x, int64_t n, int sms);
// x *= *inv_dev (real, device); runs when !stop or info == kstep, and never when refill is set
void launch_scale_dev(int kind, cudaStream_t s, void* x, int64_t n, const void* inv_dev, const int* flags, int kstep, int sms,
                      const HaloP2P* hp = nullptr);
// Final CGS2 update fused with the normalisation (predicted norm), the H/T/B column update and, optionally, the
// P2P halo push of the finished vector (kernels_gs.cu: k_multiaxpy_fin).  mode: 0 arnoldi, 1 lanczos, 2 bidiag,
// 4 gmres (no column update).  c2 has j+1 entries, c2[j] = ||w'||^2.
void launch_multiaxpy_fin(int kind, cudaStream_t s, const void* V, int64_t ld, int j, const void* c1, const void* c2, void* w,
                          int64_t n, void* partial, void* nrm2_out, unsigned* counter, void* hcol, double tol, double atol,
                          void* inv_dev, int* flags, int kstep, int mode, int sms, const P2P* p2p, const HaloP2P* hp);
// dst = src unless flags[F_STOP] (E type, length n)
void launch_copy_gated(int kind, cudaStream_t s, const void* src, void* dst, int64_t n, const int* flags, int sms);
void launch_fill(int kind, cudaStream_t s, void* x, int64_t n, int64_t row0, int dist, uint64_t seed, int sms);

// device-resident CG iteration (kernels_vec.cu): see k_cg_update / k_cg_check / k_cg_direction.
// mode: CG_PLAIN (no preconditioner), CG_DIAG (M = diag(d) fused into both vector kernels), CG_NORED (any other M:
// k_cg_update skips its reduction, the caller applies M and reduces r^H z)
enum { CG_PLAIN = 0, CG_DIAG = 1, CG_NORED = 2 };
void launch_cg_update(int kind, cudaStream_t s, const void* scal, const void* pAp, const void* p, const void* Ap, void* x,
                      void* r, int64_t n, void* partial, void* nrm2_out, unsigned* counter, const int* flags, int sms,
                      const P2P* p2p, int mode = CG_PLAIN, const void* d = nullptr);
void launch_cg_check(int kind, cudaStream_t s, void* scal, const void* rr_new, double tol, int maxiter, double* res_hist, int* flags);
// p = r + beta p, or with d != nullptr p = d o r + beta p
void launch_cg_direction(int kind, cudaStream_t s, const void* scal, const void* r, void* p, int64_t n, const int* flags, int sms,
                         const void* d = nullptr);
// diagonal operator: y = d o x (conj: y = conj(d) o x); y may alias x
void launch_diag(int kind, cudaStream_t s, const void* d, const void* x, void* y, int64_t n, bool conj, const int* flags, int sms);

// GMRES column update + Givens + convergence flag on the device (H / e / cs / sn are double2 arrays)
void launch_gmres_update(int kind, cudaStream_t s, const void* c1, const void* c2, int k, const void* nrm2, void* H, int ldh,
                         void* e, void* cs, void* sn, double tol, void* inv_dev, int* flags, double* res_hist);

// Hessenberg / tridiagonal / bidiagonal column update (one tiny CTA).
//   mode 0 arnoldi (qr_no_pivoting p=1 + breakdown test), 1 lanczos (< tol), 2 bidiag (<= tol), 3 plain norm
void launch_update(int kind, cudaStream_t s, const void* c1, const void* c2, int j, const void* nrm2, void* hcol,
                   double tol, double atol, void* inv_dev, int* flags, int kstep, int mode);
// gs_info: flags[F_GSINFO] = (sqrt(|ww|) < atol)
void launch_gsinfo(cudaStream_t s, const void* ww, int is_cplx, double atol, int* flags);
// dst (E type) = src (W type) narrowed, length n
void launch_narrow(int kind, cudaStream_t s, const void* src, void* dst, int n, const int* flags);

// L2-blocked CSR (lkb_csr.cu): non-zeros sorted by column block; tab[b * (rows + 1) + r] = first entry of (block b, row r)
struct CsrBlocked {
    int nb = 0; int64_t cw = 0, rows = 0, nnz = 0;
    uint32_t* tab = nullptr; int32_t* col = nullptr; void* val = nullptr;
};
// y = A x over the blocked layout: one sweep per column block, y accumulated across the blocks
void launch_csr_blocked(int kind, cudaStream_t s, const CsrBlocked& b, const void* x, void* y, bool conj_vals, const int* flags, int sms);
// Jacobi preconditioner d = diag(A)^-1 built on the device (kernels_ops.cu: k_jacobi, one instantiation per operator type).
// Rows whose diagonal entry is zero or not finite leave d unwritten and lower *bad_row (initialised to ~0) to their global row.
enum { JAC_STENCIL = 0, JAC_CSR = 1, JAC_CSR_BLOCKED = 2, JAC_DENSE = 3, JAC_DIAG = 4 };
struct JacobiSrc {
    int mode = JAC_STENCIL;
    int64_t rows = 0, row0 = 0;       // local rows; global index of the first (error message only)
    Scalar c0 = {0, 0};               // stencil: the centre coefficient
    const int64_t* rowptr = nullptr; const int32_t* col = nullptr; const void* val = nullptr;   // plain csr
    CsrBlocked blk;                   // L2-blocked csr
    int64_t col0 = 0;                 // csr: the diagonal of local row r is at column col0 + r (row-sharded: global index)
    const void* a = nullptr;          // dense (column-major rows x rows) or the diagonal operator's d
};
void launch_jacobi(int kind, cudaStream_t s, const JacobiSrc& src, void* d, unsigned long long* bad_row, int sms);
void launch_stencil(int kind, cudaStream_t s, const StencilArgs& a, const void* x, void* y, bool trans,
                    const int* flags, int sms);
// CSR SpMV y = A x (vector-per-row); conj_vals: use conj(A) values (for the explicit-transpose rmatvec)
void launch_csr(int kind, cudaStream_t s, int64_t m, const int64_t* rowptr, const int32_t* col, const void* val,
                const void* x, void* y, bool conj_vals, const int* flags, int sms);
// dense column-major m x n operator (plumbing config: n = 128): y = A x or y = A^H x
void launch_dense(int kind, cudaStream_t s, int64_t m, int64_t n, const void* a, const void* x, void* y, bool trans,
                  const int* flags);
// Y(:, 0:p) = X(:, 0:k) Z(0:k, 0:p)   tall-skinny basis update (Z on device, E type, ldz)
void launch_basis_gemm(int kind, cudaStream_t s, const void* X, int64_t ldx, int k, const void* Z, int ldz, int p,
                       void* Y, int64_t ldy, int64_t n, int sms);

}  // namespace lkb
