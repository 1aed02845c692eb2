// lkb_internal.h -- host-side objects behind the opaque C handles.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <complex>
#include <functional>
#include <map>
#include <string>
#include <tuple>
#include <utility>
#include <vector>
#include "../../include/lkb.h"
#include "lkb_kernels.h"

namespace lkb {

void set_error(const char* fmt, ...);

// ---- NCCL, resolved at run time with dlopen (no link-time dependency) ----------------------
struct NcclId { char internal[128]; };
struct NcclApi {
    void* handle = nullptr;
    int (*GetUniqueId)(void*) = nullptr;
    int (*CommInitRank)(void**, int, /*ncclUniqueId by value*/ NcclId, int) = nullptr;
    int (*CommDestroy)(void*) = nullptr;
    int (*AllReduce)(const void*, void*, size_t, int, int, void*, cudaStream_t) = nullptr;
    int (*Broadcast)(const void*, void*, size_t, int, int, void*, cudaStream_t) = nullptr;
    int (*AllGather)(const void*, void*, size_t, int, void*, cudaStream_t) = nullptr;
    int (*Reduce)(const void*, void*, size_t, int, int, int, void*, cudaStream_t) = nullptr;
    int (*Send)(const void*, size_t, int, int, void*, cudaStream_t) = nullptr;
    int (*Recv)(void*, size_t, int, int, void*, cudaStream_t) = nullptr;
    int (*GroupStart)() = nullptr;
    int (*GroupEnd)() = nullptr;
    const char* (*GetErrorString)(int) = nullptr;
};
NcclApi* nccl_api();   // nullptr (+ error set) when libnccl cannot be loaded

enum ProfClass { PC_MATVEC = 0, PC_DOT = 1, PC_AXPY = 2, PC_OTHER = 3, PC_FUSED = 4, PC_COUNT = 8 };
// lkb_op_s::type.  The values are printed by lkb_op_jacobi_create's error message.
enum OpType { OP_DENSE = 0, OP_STENCIL = 1, OP_CSR = 3, OP_DIAG = 4, OP_CALLBACK = 9 };

// ---- owners: every raw CUDA resource and every solver work object has exactly one, and goes with it ------------------
// Members and locals are released in reverse order of declaration.  (The host-shell test mocks replace lkb_basis_destroy,
// lkb_vec_destroy and dev_free.)
template <class T, auto Release> class Owner {
  public:
    Owner() = default;
    explicit Owner(T p) : p_(p) {}
    Owner(Owner&& o) noexcept : p_(o.release()) {}
    Owner& operator=(Owner&& o) noexcept { reset(o.release()); return *this; }
    Owner(const Owner&) = delete;
    Owner& operator=(const Owner&) = delete;
    ~Owner() { reset(); }
    void reset(T p = nullptr) { T old = p_; p_ = p; if (old) Release(old); }
    T release() { T p = p_; p_ = nullptr; return p; }   // hand the resource to a caller, or back to one on failure
    T* out() { return &p_; }                   // for the create call that fills an empty owner
    T get() const { return p_; }
    operator T() const { return p_; }
    T operator->() const { return p_; }
  private:
    T p_ = nullptr;
};
int comm_destroy(void* comm);                  // ncclCommDestroy through nccl_api()
template <class T> using CudaPtr = Owner<T*, cudaFree>;     // cudaMalloc memory (operator and context buffers)
typedef Owner<void*, cudaFreeHost> PinnedPtr;
typedef Owner<void*, cudaIpcCloseMemHandle> IpcMap;         // a peer's region mapped with cudaIpcOpenMemHandle
typedef Owner<cudaStream_t, cudaStreamDestroy> StreamOwner;
typedef Owner<void*, comm_destroy> CommOwner;
typedef Owner<lkb_basis_t, lkb_basis_destroy> BasisOwner;
typedef Owner<lkb_vec_t, lkb_vec_destroy> VecOwner;
typedef Owner<lkb_op_t, lkb_op_destroy> OpOwner;           // an operator until its creator hands it out
// an instantiated CUDA graph and the kernel launches one replay stands for
struct GraphExec { Owner<cudaGraphExec_t, cudaGraphExecDestroy> exec; int64_t launches = 0; };
// the arrays an L2-blocked CsrBlocked views
struct CsrBlockedMem { CudaPtr<uint32_t> tab; CudaPtr<int32_t> col; CudaPtr<void> val; };
}  // namespace lkb

struct lkb_ctx_s {
    int dev = 0, sms = 148;
    int rank = 0, world = 1;
    // The owners below go in reverse order: cached graphs, the communicator, the peer mappings, the buffers, the stream.
    lkb::StreamOwner stream;
    // device workspace
    lkb::CudaPtr<void> partial; size_t partial_bytes = 0;
    lkb::CudaPtr<void> c1, c2, tmpw; size_t cbuf_len = 0;   // W elements
    lkb::CudaPtr<void> nrm2;       // one W
    lkb::CudaPtr<double> inv;      // one double
    lkb::CudaPtr<int> flags;       // F_COUNT ints
    lkb::CudaPtr<unsigned> counter;
    lkb::CudaPtr<void> Hd; size_t Hd_bytes = 0;
    // coefd and hstage are views of the two owners below.  (The host-shell test mocks point them at host memory that they
    // allocate and free themselves, and leave the owners empty.)
    void* coefd = nullptr; size_t coefd_bytes = 0;
    void* hstage = nullptr; size_t hstage_bytes = 0;     // pinned host staging
    lkb::CudaPtr<void> coefd_mem;
    lkb::PinnedPtr hstage_mem;
    uint64_t seed = 0x1234abcdULL, seed_calls = 0;
    bool graphs = true;
    bool fused = true;
    bool fin = true;            // final CGS2 pass fused with normalisation + column update (k_multiaxpy_fin)
    bool serpentine = true;     // consecutive Gram-Schmidt kernels of a step sweep the rows in opposite directions (lkb_kernels.h)
    bool pdl = true;            // programmatic dependent launch of the step-loop kernels (lkb_kernels.h: PdlScope)
    int csr_slice_kb = 48 * 1024, csr_block_min_kb = 96 * 1024;   // L2 blocking of CSR operators (lkb_csr.cu)
    bool write_intermediate = false;   // eigs / eighs / svds rewrite <solver>_output.txt every step (rank 0)
    bool fused_halo = true;     // P2P halo push fused into the kernel that finishes the next matvec input
    // in-kernel NVLink allreduce (CUDA IPC peer buffers); falls back to NCCL when not attached
    bool p2p_active = false;
    lkb::P2P p2p;               // kernel view of the four owners below
    lkb::CudaPtr<void> p2p_region;
    lkb::CudaPtr<unsigned> p2p_epoch;
    lkb::CudaPtr<unsigned long long> ktime;      // lkb_debug_ktime
    lkb::IpcMap peer_map[lkb::P2P_MAXW];
    lkb::CommOwner comm;
    const lkb::P2P* p2p_arg() const { return (p2p_active || p2p.dbg) ? &p2p : nullptr; }
    bool capturing = false;
    bool profile = false;
    int64_t launches = 0;
    double prof_ms[lkb::PC_COUNT] = {0, 0, 0, 0, 0, 0, 0, 0};
    int64_t prof_n[lkb::PC_COUNT] = {0, 0, 0, 0, 0, 0, 0, 0};
    struct ProfEv { int cls; cudaEvent_t a, b; };
    std::vector<ProfEv> prof_evs;
    std::map<std::string, lkb::GraphExec> graph_cache;
};

struct lkb_vec_s {
    lkb_ctx_s* ctx; int kind; int64_t n, n_global, row0; void* d; bool owns;
};
struct lkb_basis_s {
    lkb_ctx_s* ctx; int kind; int64_t n, n_global, row0, ld; int ncols; void* d; uint64_t uid;
    bool owns = true;          // false: lkb_basis_view of a column range of another basis
};
struct lkb_op_s {
    lkb_ctx_s* ctx; int type; int kind;           // type: lkb::OpType
    int64_t m, n;                                 // local rows of the output / input vectors
    int64_t n_matvec = 0, n_rmatvec = 0;
    // stencil
    lkb::StencilArgs st; int64_t slow0 = 0, nslow_global = 0;
    lkb::CudaPtr<void> halo_lo, halo_hi; int64_t halo_elems = 0;
    // P2P halo exchange: hp views this rank's halo region, its counters and the neighbours' regions mapped into this process
    lkb::HaloP2P hp; bool hp_active = false;
    lkb::CudaPtr<void> hp_region; lkb::CudaPtr<unsigned> hp_ctr; lkb::IpcMap hp_lo_map, hp_hi_map;
    // csr (+ explicit transpose for rmatvec)
    lkb::CudaPtr<int64_t> rowptr; lkb::CudaPtr<int32_t> col; lkb::CudaPtr<void> val; int lpr = 8;
    lkb::CudaPtr<int64_t> t_rowptr; lkb::CudaPtr<int32_t> t_col; lkb::CudaPtr<void> t_val; int t_lpr = 8;
    lkb::CsrBlocked blk, t_blk;                   // L2-blocked layouts (nb > 0: they replace the plain arrays above)
    lkb::CsrBlockedMem blk_mem, t_blk_mem;
    // row-sharded csr: full-length gather / scatter buffers and every rank's (offset, count) of the column and row spaces
    bool dist = false; int64_t m_global = 0, n_global = 0;
    lkb::CudaPtr<void> x_full, y_full, y_red;
    std::vector<int64_t> col_off, col_cnt, row_off, row_cnt;
    // dense
    lkb::CudaPtr<void> a;
    // diagonal: y = d o x, d laid out like the vectors it applies to (global index of the first row, global length)
    lkb::CudaPtr<void> diag; int64_t diag_row0 = 0, diag_n_global = 0;
    // callback
    int (*fn)(void*, const void*, void*, int32_t, void*) = nullptr; void* user = nullptr; bool capturable = false;
    uint64_t uid = 0;
};

// ---- internal helpers shared by lkb_core / lkb_krylov / lkb_solvers --------------------------
namespace lkb {
#define LKB_CUDA(call) do { cudaError_t e_ = (call); if (e_ != cudaSuccess) { \
    lkb::set_error("%s:%d: %s -> %s", __FILE__, __LINE__, #call, cudaGetErrorString(e_)); return LKB_ERR_CUDA; } } while (0)
#define LKB_TRY(call) do { int r_ = (call); if (r_ != 0) return r_; } while (0)

int dev_alloc(lkb_ctx_s* c, void** p, size_t bytes);   // stream-ordered, pooled (vectors, bases, solver work space)
void dev_free(lkb_ctx_s* c, void* p);
// Fill an owner with `bytes` of cudaMalloc memory (of pinned host memory for a PinnedPtr).  A failure clears the runtime's
// last error, so that it is not reported again by the next launch check.
template <class T, auto Release> int cuda_alloc(Owner<T, Release>& o, size_t bytes) {
    constexpr bool host = Release == cudaFreeHost;
    void* p = nullptr;
    const cudaError_t e = host ? cudaMallocHost(&p, bytes) : cudaMalloc(&p, bytes);
    if (e != cudaSuccess) {
        cudaGetLastError();
        set_error("%s(%zu) failed: %s", host ? "cudaMallocHost" : "cudaMalloc", bytes, cudaGetErrorString(e));
        return LKB_ERR_ALLOC;
    }
    o.reset((T)p);
    return 0;
}
int ensure_ws(lkb_ctx_s* c, int jp);                 // grow partial / c1 / c2 for jp = j+1 coefficients
int ensure_hstage(lkb_ctx_s* c, size_t bytes);
int ensure_Hd(lkb_ctx_s* c, size_t bytes);
int ensure_coefd(lkb_ctx_s* c, size_t bytes);
int allreduce_w(lkb_ctx_s* c, void* buf, size_t ndoubles);
// make rank 0's copy of a small HOST array authoritative on every rank (k x k host-LAPACK results)
int bcast_host(lkb_ctx_s* c, void* host_buf, size_t bytes);   // in-place sum over ranks (no-op when world == 1)
int check_launch(lkb_ctx_s* c, const char* what);
// The profile bracket: prof_end counts the launches in c->launches and, with lkb_set_profile, times them under class
// `cls`.  Every kernel launch of the library goes through it exactly once (graph replays add their recorded count).
void prof_begin(lkb_ctx_s* c, int cls);
void prof_end(lkb_ctx_s* c, int cls, int nlaunch);
template <class F> void prof_launch(lkb_ctx_s* c, int cls, int nlaunch, F&& launch) { prof_begin(c, cls); launch(); prof_end(c, cls, nlaunch); }
int prof_collect(lkb_ctx_s* c);
inline void* col_ptr(const lkb_basis_s* b, int i) { return (char*)b->d + (size_t)i * (size_t)b->ld * kind_size(b->kind); }
inline double atol_of(int kind) { return (kind == KS || kind == KC) ? 1e-6 : 1e-15; }   // Constants.f90:18-37
inline double rtol_of(int kind) { return (kind == KS || kind == KC) ? 1e-3 : 3.1622776601683795e-08; }
// enqueue y = A x (trans: y = A^H x) on the context stream, including halo exchange
// halo_prepushed: x's boundary rows were already stored into the neighbours' halo buffers by the kernel that
// finished x (k_multiaxpy_fin / k_scale_dev with a HaloP2P descriptor): skip the k_halo_push kernel.
int op_apply_enqueue(lkb_op_s* A, const void* x, void* y, bool trans, const int* flags, bool halo_prepushed = false);
// The final CGS2 pass of a step against V(:, 0:j) may be k_multiaxpy_fin, which normalises with the predicted norm: not for
// j = 0, not with option "fin" = 0, and not when the reductions go through ncclAllReduce (the predicted norm must not be
// summed over ranks).
inline bool fin_usable(const lkb_ctx_s* c, int j) { return c->fin && j > 0 && (c->world == 1 || c->p2p_active); }
// descriptor for a fused halo push of this operator's next input vector by the final pass of a step against V(:, 0:j), or
// nullptr (single GPU / NCCL halos / not a stencil / no k_multiaxpy_fin)
const lkb::HaloP2P* op_halo_desc(const lkb_op_s* A, int j);
// final-pass description of a CGS2 step that ends in k_multiaxpy_fin (see step_tail_enqueue)
struct FinArgs { int mode; double tol; int kstep; void* hcol; bool with_c1; const lkb::HaloP2P* hp; };
// multi-dot out(0:j) = V(:, 0:j)^H w, out(j) = w^H w, summed over the ranks
int dot_reduce(lkb_ctx_s* c, int kind, const void* V, int64_t ld, int j, const void* w, int64_t n, void* out, const int* flags);
// multi-axpy w -= V(:, 0:j) coef; with want_norm, nrm2 = ||w||^2 summed over the ranks
int axpy_sub(lkb_ctx_s* c, int kind, const void* V, int64_t ld, int j, const void* coef, void* w, int64_t n, bool want_norm,
             const int* flags);
// enqueue one double Gram-Schmidt step of w against V(:, 0:j); leaves c1, c2 (and nrm2 if asked) in the workspace
int dgs_enqueue(lkb_ctx_s* c, int kind, const void* V, int64_t ld, int j, void* w, int64_t n, int* flags,
                bool want_norm, bool want_gsinfo, const FinArgs* fin = nullptr);
// Read c1 + c2 (first j entries; only c1 unless `two`) and, optionally, nrm2 and the flags to the host (one sync)
int fetch_coeffs(lkb_ctx_s* c, int kind, int j, bool two, std::vector<Scalar>& out, double* nrm2, int* flags);
int step_tail_enqueue(lkb_ctx_s* c, int kind, const void* V, int64_t ld, int j, void* w, int64_t n, int mode, double tol,
                      int kstep, void* hcol, const lkb::HaloP2P* hp);
int norm2_enqueue(lkb_ctx_s* c, int kind, const void* w, int64_t n, const int* flags);  // nrm2 <- ||w||^2
int vec_norm_sync(lkb_ctx_s* c, int kind, const void* w, int64_t n, double* out);
int vec_dot_sync(lkb_ctx_s* c, int kind, const void* x, const void* y, int64_t n, Scalar* out);
int fetch_flags(lkb_ctx_s* c, int* host_flags);
uint64_t next_seed(lkb_ctx_s* c);
// CSR set-up (lkb_csr.cu): host arrays -> device + validation + explicit transpose; or finish arrays already on the device
int csr_build(lkb_ctx_s* c, lkb_op_s* op, int kind, int64_t rows, int64_t ncols_index, const int64_t* rowptr,
              const int32_t* col, const void* val);
int csr_finish_device(lkb_ctx_s* c, lkb_op_s* op, int kind, int64_t rows, int64_t ncols_index);
uint64_t next_uid();
void invalidate_graphs(lkb_ctx_s* c, uint64_t uid);   // uid == 0: all
int arnoldi_enqueue(lkb_op_s* A, lkb_basis_s* X, int kstart, int kend, double tol, bool tr);
int arnoldi_collect(lkb_op_s* A, lkb_basis_s* X, void* H, int ldh, int32_t* info, int kstart, int kend, bool tr,
                    const void* pinned_host);
int krylov_fetch_async(lkb_ctx_s* c, int kind, int ldd, int kstart, int kend, void* pinned_host);
int lanczos_enqueue(lkb_op_s* A, lkb_basis_s* X, int kstart, int kend, double tol);
int lanczos_collect(lkb_op_s* A, lkb_basis_s* X, void* T, int ldt, int32_t* info, int kstart, int kend, const void* pinned_host);
int bidiag_enqueue(lkb_op_s* A, lkb_basis_s* U, lkb_basis_s* V, int kstart, int kend, double tol);
int bidiag_collect(lkb_op_s* A, lkb_basis_s* U, void* B, int ldb, int32_t* info, int kstart, int kend, const void* pinned_host);
// a callback operator may be captured into a CUDA graph only when its creator declared it capturable
inline bool op_capturable(const lkb_op_s* A) { return A->type != OP_CALLBACK || A->capturable; }

// One element of a host array of `kind` as a complex double, and back (the single precisions round on the way in)
typedef std::complex<double> cd;
inline cd load_kind(int kind, const void* base, size_t idx) {
    switch (kind) {
        case KS: return cd(((const float*)base)[idx], 0.0);
        case KD: return cd(((const double*)base)[idx], 0.0);
        case KC: return cd(((const float*)base)[2 * idx], ((const float*)base)[2 * idx + 1]);
        default: return cd(((const double*)base)[2 * idx], ((const double*)base)[2 * idx + 1]);
    }
}
inline void store_kind(int kind, void* base, size_t idx, cd v) {
    switch (kind) {
        case KS: ((float*)base)[idx] = (float)v.real(); break;
        case KD: ((double*)base)[idx] = v.real(); break;
        case KC: ((float*)base)[2 * idx] = (float)v.real(); ((float*)base)[2 * idx + 1] = (float)v.imag(); break;
        default: ((double*)base)[2 * idx] = v.real(); ((double*)base)[2 * idx + 1] = v.imag(); break;
    }
}
inline Scalar to_scalar(cd v) { return Scalar{v.real(), v.imag()}; }

// a dev_alloc buffer
struct DevBuf {
    lkb_ctx_s* c; void* p = nullptr;
    explicit DevBuf(lkb_ctx_s* ctx) : c(ctx) {}
    DevBuf(const DevBuf&) = delete;
    DevBuf& operator=(const DevBuf&) = delete;
    ~DevBuf() { dev_free(c, p); }
    int alloc(size_t bytes) { return dev_alloc(c, &p, bytes); }
};
// Run `body` (which only enqueues work on c->stream) under stream capture with c->capturing set, and instantiate the graph.
// The launches the body counted go to g->launches, not to c->launches.  `what` prefixes the error messages ("gmres: ").
int capture_graph(lkb_ctx_s* c, const char* what, const std::function<int()>& body, GraphExec* g);
}  // namespace lkb
