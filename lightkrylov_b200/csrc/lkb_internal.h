// lkb_internal.h -- host-side objects behind the opaque C handles.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <map>
#include <string>
#include <tuple>
#include <vector>
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

}  // namespace lkb

struct lkb_ctx_s {
    int dev = 0, sms = 148;
    int rank = 0, world = 1;
    void* comm = nullptr;
    cudaStream_t stream = nullptr;
    // device workspace
    void* partial = nullptr; size_t partial_bytes = 0;
    void* c1 = nullptr; void* c2 = nullptr; void* tmpw = nullptr; size_t cbuf_len = 0;   // W elements
    void* nrm2 = nullptr;       // one W
    double* inv = nullptr;      // one double
    int* flags = nullptr;       // F_COUNT ints
    unsigned* counter = nullptr;
    void* Hd = nullptr; size_t Hd_bytes = 0;
    void* coefd = nullptr; size_t coefd_bytes = 0;
    // pinned host staging
    void* hstage = nullptr; size_t hstage_bytes = 0;
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
    lkb::P2P p2p;
    void* p2p_region = nullptr;
    const lkb::P2P* p2p_arg() const { return (p2p_active || p2p.dbg) ? &p2p : nullptr; }
    bool capturing = false;
    bool profile = false;
    int64_t launches = 0;
    double prof_ms[lkb::PC_COUNT] = {0, 0, 0, 0, 0, 0, 0, 0};
    int64_t prof_n[lkb::PC_COUNT] = {0, 0, 0, 0, 0, 0, 0, 0};
    struct ProfEv { int cls; cudaEvent_t a, b; };
    std::vector<ProfEv> prof_evs;
    struct GraphEntry { cudaGraphExec_t exec; int64_t launches; };
    std::map<std::string, GraphEntry> graph_cache;
};

struct lkb_vec_s {
    lkb_ctx_s* ctx; int kind; int64_t n, n_global, row0; void* d; bool owns;
};
struct lkb_basis_s {
    lkb_ctx_s* ctx; int kind; int64_t n, n_global, row0, ld; int ncols; void* d; uint64_t uid;
    bool owns = true;          // false: lkb_basis_view of a column range of another basis
};
struct lkb_op_s {
    lkb_ctx_s* ctx; int type; int kind;           // type: 0 dense, 1 stencil, 3 csr, 4 diagonal, 9 callback
    int64_t m, n;                                 // local rows of the output / input vectors
    int64_t n_matvec = 0, n_rmatvec = 0;
    // stencil
    lkb::StencilArgs st; int64_t slow0 = 0, nslow_global = 0;
    void* halo_lo = nullptr; void* halo_hi = nullptr; int64_t halo_elems = 0;
    lkb::HaloP2P hp; bool hp_active = false; void* hp_lo_map = nullptr; void* hp_hi_map = nullptr;
    // csr (+ explicit transpose for rmatvec)
    int64_t* rowptr = nullptr; int32_t* col = nullptr; void* val = nullptr; int lpr = 8;
    int64_t* t_rowptr = nullptr; int32_t* t_col = nullptr; void* t_val = nullptr; int t_lpr = 8;
    lkb::CsrBlocked blk, t_blk;                   // L2-blocked layouts (nb > 0: they replace the plain arrays above)
    // row-sharded csr: full-length gather / scatter buffers and every rank's (offset, count) of the column and row spaces
    bool dist = false; int64_t m_global = 0, n_global = 0;
    void* x_full = nullptr; void* y_full = nullptr; void* y_red = nullptr;
    std::vector<int64_t> col_off, col_cnt, row_off, row_cnt;
    // dense
    void* a = nullptr;
    // diagonal: y = d o x, d laid out like the vectors it applies to (global index of the first row, global length)
    void* diag = nullptr; int64_t diag_row0 = 0, diag_n_global = 0;
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
int ensure_ws(lkb_ctx_s* c, int jp);                 // grow partial / c1 / c2 for jp = j+1 coefficients
int ensure_hstage(lkb_ctx_s* c, size_t bytes);
int ensure_Hd(lkb_ctx_s* c, size_t bytes);
int ensure_coefd(lkb_ctx_s* c, size_t bytes);
int allreduce_w(lkb_ctx_s* c, void* buf, size_t ndoubles);
// make rank 0's copy of a small HOST array authoritative on every rank (k x k host-LAPACK results)
int bcast_host(lkb_ctx_s* c, void* host_buf, size_t bytes);   // in-place sum over ranks (no-op when world == 1)
int check_launch(lkb_ctx_s* c, const char* what);
void prof_begin(lkb_ctx_s* c, int cls);
void prof_end(lkb_ctx_s* c, int cls, int nlaunch);
int prof_collect(lkb_ctx_s* c);
inline void* col_ptr(const lkb_basis_s* b, int i) { return (char*)b->d + (size_t)i * (size_t)b->ld * kind_size(b->kind); }
inline double atol_of(int kind) { return (kind == KS || kind == KC) ? 1e-6 : 1e-15; }   // Constants.f90:18-37
inline double rtol_of(int kind) { return (kind == KS || kind == KC) ? 1e-3 : 3.1622776601683795e-08; }
// enqueue y = A x (trans: y = A^H x) on the context stream, including halo exchange
// halo_prepushed: x's boundary rows were already stored into the neighbours' halo buffers by the kernel that
// finished x (k_multiaxpy_fin / k_scale_dev with a HaloP2P descriptor): skip the k_halo_push kernel.
int op_apply_enqueue(lkb_op_s* A, const void* x, void* y, bool trans, const int* flags, bool halo_prepushed = false);
// descriptor for a fused halo push of this operator's next input vector, or nullptr (single GPU / NCCL halos / not a stencil)
const lkb::HaloP2P* op_halo_desc(const lkb_op_s* A);
// final-pass description of a CGS2 step that ends in k_multiaxpy_fin (see step_tail_enqueue)
struct FinArgs { int mode; double tol; int kstep; void* hcol; bool with_c1; const lkb::HaloP2P* hp; };
// enqueue one double Gram-Schmidt step of w against V(:, 0:j); leaves c1, c2 (and nrm2 if asked) in the workspace
int dgs_enqueue(lkb_ctx_s* c, int kind, const void* V, int64_t ld, int j, void* w, int64_t n, int* flags,
                bool want_norm, bool want_gsinfo, const FinArgs* fin = nullptr);
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
int arnoldi_fetch_async(lkb_basis_s* X, int kstart, int kend, void* pinned_host);
int arnoldi_collect(lkb_op_s* A, lkb_basis_s* X, void* H, int ldh, int32_t* info, int kstart, int kend, bool tr,
                    const void* pinned_host);
int krylov_fetch_async(lkb_ctx_s* c, int kind, int ldd, int kstart, int kend, void* pinned_host);
int lanczos_enqueue(lkb_op_s* A, lkb_basis_s* X, int kstart, int kend, double tol);
int lanczos_collect(lkb_op_s* A, lkb_basis_s* X, void* T, int ldt, int32_t* info, int kstart, int kend, const void* pinned_host);
int bidiag_enqueue(lkb_op_s* A, lkb_basis_s* U, lkb_basis_s* V, int kstart, int kend, double tol);
int bidiag_collect(lkb_op_s* A, lkb_basis_s* U, void* B, int ldb, int32_t* info, int kstart, int kend, const void* pinned_host);
}  // namespace lkb
