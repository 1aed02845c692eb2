/* lkb.h -- C ABI of the B200-native Krylov-factorisation hot path (liblkb.so).
 *
 * The reference (nekStab/LightKrylov) is pure Fortran and has NO existing FFI: its plugin
 * boundary is the pair of abstract types `abstract_vector_{rsp,rdp,csp,cdp}` /
 * `abstract_linop_*` plus the generic procedures `arnoldi`, `lanczos`, `bidiagonalization`,
 * `double_gram_schmidt_step`, `gmres`, `cg`, ...  The entry points below are exactly what a thin
 * ISO_C_BINDING shim (fortran/lightkrylov_cuda.f90, INTEGRATION.md) binds to so that device-
 * resident extensions of those types run this library.  Every declaration cites the reference
 * interface it replaces (paths relative to the reference tree).
 *
 * Conventions
 *   - plain pointers and sizes only; no torch / C++ types.
 *   - kind: LKB_S/D/C/Z = rsp/rdp/csp/cdp.  Scalars cross the ABI as `const void*` pointing to one
 *     element of that kind (float, double, float[2], double[2]); real results as double.
 *   - Fortran `integer` <-> int32_t, `logical` <-> int32_t (0/1), indices are 1-based where the
 *     reference's are (kstart, kend, info); sizes of device data are int64_t.
 *   - all calls are synchronous w.r.t. host-visible results and must come from one host thread
 *     per context (the reference is serial and not thread-safe).
 *   - return value: 0 = ok, <0 = fatal (CUDA/NCCL failure, bad argument, NaN norm); the Fortran
 *     shim maps a non-zero return to `stop_error` (src/Utilities/Logger.f90:290-298).
 *     `info` out-arguments follow the reference (SURVEY.md 8b): 0 ok, >0 benign.
 *   - there is NO CPU fallback: without a CUDA device every entry point fails with LKB_ERR_CUDA.
 */
#ifndef LKB_H
#define LKB_H
#include <stdint.h>
#ifdef __cplusplus
extern "C" {
#endif

enum { LKB_S = 0, LKB_D = 1, LKB_C = 2, LKB_Z = 3 };
enum { LKB_OK = 0, LKB_ERR_CUDA = -1, LKB_ERR_ARG = -2, LKB_ERR_NCCL = -3, LKB_ERR_NAN = -4,
       LKB_ERR_LAPACK = -5, LKB_ERR_ALLOC = -6 };
enum { LKB_DIST_NORMAL = 0, LKB_DIST_UNIFORM = 1 };

typedef struct lkb_ctx_s*   lkb_ctx_t;
typedef struct lkb_vec_s*   lkb_vec_t;     /* device abstract_vector */
typedef struct lkb_basis_s* lkb_basis_t;   /* contiguous column-major array of abstract_vectors */
typedef struct lkb_op_s*    lkb_op_t;      /* device abstract_linop */

/* ---- context -----------------------------------------------------------------------------
 * One context per process per GPU.  Replaces comm_setup/comm_close (Logger.f90:245-288): the
 * reference's only parallel hook is MPI init for logging; global reductions were the user's job
 * inside `dot`.  Here the context owns the stream, workspaces and (optionally) the NCCL
 * communicator used to all-reduce partial inner products across the row-sharded ranks. */
int lkb_init(int device, lkb_ctx_t* ctx);
int lkb_nccl_unique_id(void* id128);                       /* rank 0 creates, caller broadcasts */
int lkb_init_dist(int device, int rank, int world, const void* id128, lkb_ctx_t* ctx);
int lkb_finalize(lkb_ctx_t ctx);
int lkb_sync(lkb_ctx_t ctx);
void* lkb_stream(lkb_ctx_t ctx);                           /* cudaStream_t of the context */
const char* lkb_last_error(void);
int lkb_set_seed(lkb_ctx_t ctx, uint64_t seed);            /* seed of the `rand` TBP stream */
int lkb_set_graphs(lkb_ctx_t ctx, int enable);             /* CUDA-graph capture of step loops (default on) */
int lkb_set_option(lkb_ctx_t ctx, const char* name, int value); /* "graphs", "fused" (fused CGS2 kernel), "p2p" */
/* In-kernel NVLink allreduce (all ranks on one NVSwitch box): each rank exports a CUDA-IPC handle
 * (64 bytes) of its exchange buffer, the caller all-gathers the handles (rank order) and attaches.
 * Afterwards the (j+1)-coefficient reductions happen inside the multi-dot / fused / multi-axpy
 * kernels over peer memory instead of separate ncclAllReduce launches.  Optional: without it the
 * NCCL path is used.  lkb_set_option(ctx, "p2p", 0/1) toggles it. */
int lkb_p2p_export(lkb_ctx_t ctx, void* handle64);
int lkb_p2p_attach(lkb_ctx_t ctx, const void* handles_world_x_64);
int lkb_rank(lkb_ctx_t ctx); int lkb_world(lkb_ctx_t ctx);

/* ---- abstract_vector TBPs : src/AbstractTypes/AbstractVectors.fypp:295-381, 424-460 ------
 * n_local rows live on this GPU and are rows [row0, row0+n_local) of an n_global-row vector. */
int lkb_vec_create(lkb_ctx_t ctx, int kind, int64_t n_local, int64_t n_global, int64_t row0, lkb_vec_t* v);
int lkb_vec_wrap(lkb_ctx_t ctx, int kind, int64_t n_local, int64_t n_global, int64_t row0, void* devptr, lkb_vec_t* v);
int lkb_vec_clone(lkb_vec_t src, lkb_vec_t* dst);          /* allocate(source=) / defined assignment */
int lkb_vec_destroy(lkb_vec_t v);
int lkb_vec_zero(lkb_vec_t v);                             /* :304-308 */
int lkb_vec_rand(lkb_vec_t v, int32_t ifnorm);             /* :310-321 (normal deviates; honours ifnorm) */
int lkb_vec_fill_random(lkb_vec_t v, int dist, uint64_t seed);  /* seeded, sharding-independent */
int lkb_vec_scal(lkb_vec_t v, const void* alpha);          /* :323-332 */
int lkb_vec_axpby(const void* alpha, lkb_vec_t x, const void* beta, lkb_vec_t self); /* :334-348 self = alpha*x + beta*self */
int lkb_vec_dot(lkb_vec_t self, lkb_vec_t vec, void* out); /* :350-361 out = self^H vec (conj on self) */
int lkb_vec_norm(lkb_vec_t v, double* out);                /* :424-432 sqrt(abs(dot(v,v))) */
int64_t lkb_vec_size(lkb_vec_t v);                         /* :363-379 get_size (global) */
int64_t lkb_vec_local_size(lkb_vec_t v);
void* lkb_vec_ptr(lkb_vec_t v);                            /* raw device pointer */
int lkb_vec_put(lkb_vec_t v, const void* host);            /* TestUtils.fypp:391-441 put_data */
int lkb_vec_get(lkb_vec_t v, void* host);                  /* get_data */

/* ---- basis = X(:) : the contiguous column-major device array that replaces arrays of
 * polymorphic vectors (AbstractVectors.fypp:571-730 operate on `X(:)`). */
int lkb_basis_create(lkb_ctx_t ctx, int kind, int64_t n_local, int64_t n_global, int64_t row0, int ncols, lkb_basis_t* b);
int lkb_basis_destroy(lkb_basis_t b);
int lkb_basis_col(lkb_basis_t b, int i0, lkb_vec_t* view); /* non-owning view of column i0 (0-based) */
int lkb_basis_zero(lkb_basis_t b, int col0, int ncols);    /* zero_basis :711-715 */
/* non-owning view of columns [col0, col0+ncols): the array section X(k1:k2); release with lkb_basis_destroy */
int lkb_basis_view(lkb_basis_t b, int col0, int ncols, lkb_basis_t* view);
/* axpby_basis :697-709  Y(:, ycol0+q) = alpha X(:, xcol0+q) + beta Y(:, ycol0+q), q < ncols; beta == 0 is `copy` :717-723 */
int lkb_basis_axpby(const void* alpha, lkb_basis_t X, int xcol0, const void* beta, lkb_basis_t Y, int ycol0, int ncols);
int lkb_basis_rand(lkb_basis_t b, int col0, int ncols, int32_t ifnorm);   /* rand_basis :725-730 */
/* src/Krylov/utilities.fypp:32-81 (interfaces BaseKrylov.fypp:490-600): block-Arnoldi start helpers */
int lkb_orthonormalize_basis(lkb_basis_t X, int col0, int p, int32_t* info);
int lkb_initialize_krylov_subspace(lkb_basis_t X, lkb_basis_t X0 /* may be NULL */, int x0col0, int p0);
int lkb_initialize_random_orthonormal_basis(lkb_basis_t X, int col0, int p);
int lkb_basis_put(lkb_basis_t b, int col0, int ncols, const void* host, int64_t ldhost);
int lkb_basis_get(lkb_basis_t b, int col0, int ncols, void* host, int64_t ldhost);
int lkb_basis_ncols(lkb_basis_t b);
int64_t lkb_basis_ld(lkb_basis_t b);
/* innerprod(X(:j), W(:p)) -> out (j x p, ld ldout)              AbstractVectors.fypp:659-695 */
int lkb_basis_innerprod(lkb_basis_t X, int j, lkb_basis_t W, int wcol0, int p, void* out, int ldout);
/* W(:, q) -= X(:j) coef(:, q)   = linear_combination + sub      AbstractVectors.fypp:571-643 */
int lkb_basis_lincomb_sub(lkb_basis_t X, int j, const void* coef, int ldcoef, lkb_basis_t W, int wcol0, int p);
/* y = X(:j) coef   (linear_combination into an existing vector) */
int lkb_basis_lincomb(lkb_basis_t X, int j, const void* coef, lkb_vec_t y);
/* double_gram_schmidt_step(Y(:p), X(:j), info, if_chk_orthonormal, beta)
 *   src/Krylov/gram_schmidt.fypp:12-105, interface BaseKrylov.fypp:634-712.  beta may be NULL. */
int lkb_dgs_step(lkb_basis_t X, int j, lkb_basis_t W, int wcol0, int p, int32_t if_chk_orthonormal,
                 void* beta, int ldbeta, int32_t* info);
/* orthogonalize_against_basis (one pass)  gram_schmidt.fypp:113-200, BaseKrylov.fypp:601-629 */
int lkb_orthogonalize_against_basis(lkb_basis_t X, int j, lkb_basis_t W, int wcol0, int p,
                                    int32_t if_chk_orthonormal, void* beta, int ldbeta, int32_t* info);
/* qr(Q(:p), R, info, tol)  no pivoting   src/Krylov/qr.fypp:116-167, BaseKrylov.fypp:395-417 */
int lkb_qr(lkb_basis_t Q, int col0, int p, void* R, int ldr, double tol, int32_t* info);
/* qr(Q(:p), R, perm, info, tol)  with column pivoting   src/Krylov/qr.fypp:32-107 (+ swap_columns :174-201), BaseKrylov.fypp:395-417.
 * In place on columns [col0, col0+p): A(:, perm) = Q R.  perm (p entries) is 1-based as the reference returns it.  info = j > 0:
 * numerical rank j-1, the remaining columns are a random orthonormal completion and their R entries are zero. */
int lkb_qr_pivoting(lkb_basis_t Q, int col0, int p, void* R, int ldr, int32_t* perm, double tol, int32_t* info);

/* ---- abstract_linop : src/AbstractTypes/AbstractLinops.fypp:58-87, 204-256, 391-461 ----- */
/* coef = (center, -x, +x, -y, +y[, -z, +z]) of kind `kind`; (nx, ny[, nz]) is the GLOBAL grid,
 * the slowest axis is sharded: this rank owns `nslow_local` rows/planes starting at `slow0`. */
int lkb_op_stencil5_create(lkb_ctx_t ctx, int kind, int64_t nx, int64_t ny, const void* coef5,
                           int64_t slow0, int64_t nslow_local, lkb_op_t* A);
int lkb_op_stencil7_create(lkb_ctx_t ctx, int kind, int64_t nx, int64_t ny, int64_t nz, const void* coef7,
                           int64_t slow0, int64_t nslow_local, lkb_op_t* A);
int lkb_op_csr_create(lkb_ctx_t ctx, int kind, int64_t m, int64_t n, const int64_t* rowptr, const int32_t* col,
                      const void* val, lkb_op_t* A);
/* The same operator from CSR arrays that already live on this GPU (cudaMalloc'ed device pointers).  adopt != 0: the
 * library takes ownership of the three arrays (freed by lkb_op_destroy; on failure they stay with the caller),
 * adopt == 0: they are copied.  (rowptr, col) are validated on the device: rowptr[0] == 0, non-decreasing,
 * 0 <= col < n, else LKB_ERR_ARG.  The explicit transpose for rmatvec is built on the device. */
int lkb_op_csr_create_device(lkb_ctx_t ctx, int kind, int64_t m, int64_t n, int64_t* rowptr_dev, int32_t* col_dev,
                             void* val_dev, int32_t adopt, lkb_op_t* A);
/* Row-sharded CSR (collective): this rank owns rows [row0, row0+m_local) with GLOBAL column indices; vectors of
 * the column space are sharded as [col0, col0+n_local).  matvec gathers x over the ranks, rmatvec reduces the
 * partial A_loc^H u_loc onto the owners (NCCL over NVLink). */
int lkb_op_csr_create_dist(lkb_ctx_t ctx, int kind, int64_t m_global, int64_t n_global, int64_t row0, int64_t m_local,
                           int64_t col0, int64_t n_local, const int64_t* rowptr_local, const int32_t* col_global,
                           const void* val, lkb_op_t* A);
/* The same from local CSR arrays that already live on this GPU (cudaMalloc'ed, e.g. lkb_csr_random_device); the library
 * takes ownership (adopt must be non-zero; on failure the arrays stay with the caller).  Lets BASELINE config 5
 * (1.6e9 non-zeros) be built row-sharded without ever touching the host. */
int lkb_op_csr_create_dist_device(lkb_ctx_t ctx, int kind, int64_t m_global, int64_t n_global, int64_t row0, int64_t m_local,
                                  int64_t col0, int64_t n_local, int64_t* rowptr_dev, int32_t* col_dev, void* val_dev,
                                  int32_t adopt, lkb_op_t* A);
int lkb_op_dense_create(lkb_ctx_t ctx, int kind, int64_t m, int64_t n, const void* a_colmajor, lkb_op_t* A);
/* user-supplied device matvec (a Fortran/C extension of abstract_linop): fn launches on `stream` */
typedef int (*lkb_matvec_fn)(void* user, const void* x_dev, void* y_dev, int32_t trans, void* stream);
int lkb_op_callback_create(lkb_ctx_t ctx, int kind, int64_t m_local, int64_t n_local, lkb_matvec_fn fn,
                           void* user, int32_t capturable, lkb_op_t* A);
/* diagonal operator M = diag(d): matvec y = d o x, rmatvec y = conj(d) o x, in place allowed (x may be y).  The values
 * are copied at creation; M has d's layout (n_local, n_global, row0) and needs no communication at N > 1. */
int lkb_op_diag_create(lkb_vec_t d, lkb_op_t* M);
/* Jacobi preconditioner M = diag(A)^-1 as a diagonal operator, built on the device.  A: stencil, CSR (plain, L2-blocked,
 * or row-sharded with equal row and column slabs on this rank), dense or diagonal.  LKB_ERR_ARG for a callback or non-square
 * A, and for a zero or non-finite diagonal entry (lkb_last_error names its global row). */
int lkb_op_jacobi_create(lkb_op_t A, lkb_op_t* M);
/* Chebyshev polynomial preconditioner M of degree m >= 1, built on A: M r = z_m, the result of m Chebyshev iterations
 * (Saad, Iterative Methods, Alg. 12.1, true-residual form) on D^-1 A z = D^-1 r from z_0 = 0, D = diag(A), on [a, b] =
 * [lmin, lmax].  With theta = (b + a)/2, delta = (b - a)/2, sigma = theta/delta, rho_0 = 1/sigma:
 *     d_0 = D^-1 r / theta ;  z_1 = d_0 ;  for k = 1 .. m-1:  s_k = D^-1 (r - A z_k) ;  rho_k = 1 / (2 sigma - rho_{k-1}) ;
 *     d_k = rho_k rho_{k-1} d_{k-1} + (2 rho_k / delta) s_k ;  z_{k+1} = z_k + d_k.
 * m - 1 applications of A and no inner products; m = 1 is D^-1 / theta.  lkb_op_rmatvec applies M^H (A's rmatvec,
 * conj(D)^-1).  lmax <= 0 selects the Gershgorin bound max_r sum_c |a_rc / a_rr| of D^-1 A (never below its spectral
 * radius; 2 for the 5- and 7-point Laplacians); lmin <= 0 selects lmax / 100.  lmin >= lmax (after the defaults) is
 * LKB_ERR_ARG.  For Hermitian A with a positive diagonal and 0 < lmin < lmax, lmax >= lambda_max(D^-1 A), M is Hermitian
 * positive definite, so CG may use it; an explicit lmax below the spectrum can make M indefinite and break PCG.
 * A: stencil (every step is one fused stencil kernel), CSR (plain, L2-blocked, or row-sharded with equal row and column
 * slabs), dense or diagonal; LKB_ERR_ARG for a callback or non-square A and for a zero or non-finite diagonal entry (the
 * message names its global row).  Collective when A is a row-sharded CSR and lmax <= 0 (the bound is a max over the ranks).
 * M keeps a pointer to A: lkb_op_destroy(A) returns LKB_ERR_ARG while M is alive.  M's work vectors are allocated here;
 * M's matvec counter counts applications of M, A's counters are not touched. */
int lkb_op_chebyshev_create(lkb_op_t A, int32_t degree, double lmin, double lmax, lkb_op_t* M);
/* GMRES-polynomial preconditioner M = p(A) (Loe & Morgan, Numer. Linear Algebra Appl. 2022; Trilinos Belos GmresPoly).
 * With nonzero roots theta_1 .. theta_d, pi(z) = prod_i (1 - z/theta_i) and p(z) = (1 - pi(z))/z (degree d - 1), so
 * A M = I - pi(A).  M r by the product recurrence, in the order the roots are stored:
 *     y = r ; z = 0
 *     root theta (real kinds: real theta; complex kinds: any):  z += y/theta ;  y <- y - A (y/theta)
 *     pair (theta, conj theta), real kinds only, a = Re theta, q = |theta|^2:
 *                                   t = A y ;  w = (2a/q) y - t/q ;  z += w ;  y <- y - A w
 *     return z                      (the last factor's y update is skipped)
 * d - 1 applications of A and no inner products; d = 1 is r / theta_1.  lkb_op_rmatvec applies M^H = conj(p)(A^H): the
 * same recurrence with conj(theta_i) and A's rmatvec.  M needs neither spectral bounds nor diag(A), so A may be any square
 * operator, callbacks included; on a stencil every application of A is one fused stencil kernel.  M is not Hermitian
 * positive definite in general: it is meant for gmres.  M keeps a pointer to A: lkb_op_destroy(A) returns LKB_ERR_ARG
 * while M is alive.  M's work vectors (at most three) are allocated here; M's matvec counter counts applications of M,
 * A's counters are not touched.  M may be captured into a CUDA graph when A may.
 * roots: nroots (re, im) pairs, applied in the given order.  LKB_ERR_ARG for nroots outside 1 .. 256, a zero or non-finite
 * root, in a real kind a root with im != 0 not immediately followed by its exact conjugate (the message names its index),
 * and a non-square A. */
int lkb_op_poly_create(lkb_op_t A, int32_t nroots, const double* roots, lkb_op_t* M);
/* The GMRES polynomial of A of the given degree (1 .. 128), collective: `degree` Arnoldi steps (lkb_arnoldi, p = 1,
 * default tol; A's matvec counter grows by the steps taken) from the normalised lkb_vec_fill_random(normal, seed) vector,
 * which is the same at any sharding and leaves the context's rand stream alone.  The roots are the harmonic Ritz values,
 * the eigenvalues of H_k + |h_{k+1,k}|^2 f e_k^T with f = H_k^-H e_k (k = degree, or the step of a breakdown), computed in
 * double; a root at which pof = prod_{j != i} |1 - theta_i/theta_j| exceeds 1e4 gets ceil((log10 pof - 4)/14) extra copies
 * (in a real kind its conjugate as many); they are applied in modified Leja order (the largest modulus first, then the
 * root maximising sum_j log|theta - theta_j| over those already placed, ties to the lowest index; in a real kind a pair
 * is placed im > 0 first, its conjugate right after).  Rank 0's roots are used on every rank.  LKB_ERR_ARG for a degree
 * out of range, a singular H_k or a zero / non-finite root; LKB_ERR_LAPACK without a host LAPACK (see lkb_set_lapack). */
int lkb_op_gmres_poly_create(lkb_op_t A, int32_t degree, uint64_t seed, lkb_op_t* M);
/* The roots of a polynomial operator in application order: *nroots of them as (re, im) pairs.  LKB_ERR_ARG when M is
 * not a polynomial operator or cap < *nroots (*nroots is still set).  Feed them to lkb_op_poly_create to rebuild M. */
int lkb_op_poly_roots(lkb_op_t M, int32_t cap, int32_t* nroots, double* roots);
/* Geometric multigrid preconditioner M of a 5- or 7-point stencil A: M r is one V-cycle from a zero initial guess on a
 * hierarchy built from A (Trottenberg, Oosterlee & Schueller, Multigrid, 2001).
 *   Level 0 is A: grid (nx, ny[, nz]), coefficients (c0, c-x, c+x, c-y, c+y[, c-z, c+z]).  Write A = rho I + sum_d T_d with
 *   T_d = tri(c-d, -(c-d + c+d), c+d) acting along axis d and rho = c0 + sum_d (c-d + c+d).
 *   Coarsening: every axis at once, n -> n_c = floor(n/2), coarse point i at fine point 2i+1.  P_d is 1-D linear
 *   interpolation (fine 2i+1 takes coarse i, fine 2i and 2i+2 half of it, coarse points outside the grid are zero), P the
 *   tensor product of the P_d, and R = 2^-dim P^T, boundaries included.
 *   Coarse operators: T_d' = 1/2 P_d^T T_d P_d along each axis, rho unchanged.  T_d' has constant off-diagonals and a
 *   constant diagonal except its last entry, so every level is a 5- / 7-point stencil whose centre at (i, j, k) is
 *   c0 + sum_d [i_d = n_d - 1] e_d.  The hierarchy is built on the host in double (complex for the complex kinds).
 *   Coarsening stops at the first level with <= 512 unknowns or an axis below 2 points; that level's operator is
 *   inverted densely on the host in double with partial pivoting, stored in the kind, and applied as a dense matvec.
 *   Smoother on level l: Chebyshev of degree m (`degree`) in D_l^-1 A_l with lkb_op_chebyshev_create's recurrence on
 *   [b_l / (2 dim), b_l], b_l the Gershgorin bound of D_l^-1 A_l.  Pre-smoothing starts from 0; post-smoothing starts from
 *   the corrected x with d_0 = D^-1 (b - A x) / theta, z_1 = x + d_0, and continues as before.
 *   V-cycle:  V(l, b) = A_L^-1 b if l = L, else  x = S(b, 0) ;  x += P V(l+1, R (b - A_l x)) ;  x = S(b, x).
 * lkb_op_rmatvec applies M^H: the same cycle on A_l^H with conj(D) and (A_L^-1)^H.  M is Hermitian for Hermitian A, and
 * positive definite as well when b_l >= lambda_max on every level (always, with the Gershgorin bound), so CG may use it.
 * On each level but the coarsest one application costs: pre-smoothing m launches (m - 1 when m >= 2 and the level has no
 * edge correction), one restriction (k_mg_restrict), one prolongation (k_mg_prolong) and m post-smoothing launches; plus
 * one launch for the coarsest solve.  Every smoothing step is one fused stencil kernel.  All buffers are allocated here;
 * M may be captured into a CUDA graph.  M keeps a pointer to A: lkb_op_destroy(A) returns LKB_ERR_ARG while M is alive.
 * M's matvec counter counts applications of M, A's counters are not touched.
 * LKB_ERR_ARG for an A that is not a stencil (use the Chebyshev or GMRES-polynomial preconditioner), a row-sharded stencil
 * whose slab is not the whole grid, degree < 1, a zero or non-finite centre on any level (the message names the level), a
 * coarsest level above 512 unknowns (the message names the grid) and a singular coarsest matrix. */
int lkb_op_multigrid_create(lkb_op_t A, int32_t degree, lkb_op_t* M);
/* LKB_ERR_ARG, and A stays, while a Chebyshev, GMRES-polynomial or multigrid preconditioner built on A is alive */
int lkb_op_destroy(lkb_op_t A);
int lkb_op_matvec(lkb_op_t A, lkb_vec_t x, lkb_vec_t y);    /* apply_matvec  :391-407 (bumps counter) */
int lkb_op_rmatvec(lkb_op_t A, lkb_vec_t x, lkb_vec_t y);   /* apply_rmatvec :409-424 */
int lkb_op_counters(lkb_op_t A, int64_t* n_matvec, int64_t* n_rmatvec);
int lkb_op_reset_counters(lkb_op_t A);

/* ---- Krylov processes : src/Krylov ------------------------------------------------------- */
/* arnoldi(A, X, H, info, kstart, kend, tol, transpose, blksize)
 *   src/Krylov/arnoldi.fypp:8-76, contract BaseKrylov.fypp:60-155.
 *   X has (kdim+1)*blksize columns; H is HOST (kdim+1)p x kdim*p column-major with ld ldh, inout:
 *   only columns kstart..kend are written.  kstart/kend 1-based; pass 0 for "absent"
 *   (kstart = 1, kend = kdim); tol < 0 = absent (atol_kind). */
int lkb_arnoldi(lkb_op_t A, lkb_basis_t X, void* H, int ldh, int32_t* info,
                int32_t kstart, int32_t kend, double tol, int32_t transpose, int32_t blksize);
/* lanczos(A, X, T, info, kstart, kend, tol)   src/Krylov/lanczos.fypp:7-64, BaseKrylov.fypp:157-237 */
int lkb_lanczos(lkb_op_t A, lkb_basis_t X, void* T, int ldt, int32_t* info,
                int32_t kstart, int32_t kend, double tol);
/* bidiagonalization(A, U, V, B, info, kstart, kend, tol)  golub_kahan.fypp:7-64, BaseKrylov.fypp:239-333 */
int lkb_bidiag(lkb_op_t A, lkb_basis_t U, lkb_basis_t V, void* B, int ldb, int32_t* info,
               int32_t kstart, int32_t kend, double tol);
/* krylov_schur(n, X, H, select)  BaseKrylov.fypp:782-834 with the median selector of eigs */
int lkb_krylov_schur(lkb_basis_t X, void* H, int ldh, int kdim, int32_t* nkeep);

/* ---- solvers (host shells around the device step) ---------------------------------------- */
typedef struct {            /* gmres_dp_opts / gmres_dp_metadata : IterativeSolvers.fypp:140-188 */
    int32_t kdim;           /* default 30 */
    int32_t maxiter;        /* default 10 */
    int32_t n_iter, n_inner, n_outer, converged, info;   /* metadata out */
    double* res; int32_t res_cap, res_len;               /* optional residual history (caller-owned) */
} lkb_gmres_io;
/* gmres(A, b, x, info, rtol, atol, preconditioner, options, transpose, meta)  gmres.fypp:65-255
 * rtol/atol < 0 = absent.  lkb_gmres_precond adds the optional right preconditioner. */
int lkb_gmres(lkb_op_t A, lkb_vec_t b, lkb_vec_t x, int32_t* info, double rtol, double atol,
              int32_t transpose, lkb_gmres_io* io);
/* abstract_precond_*: `apply(vec, iter, current_residual, target_residual)` (IterativeSolvers.fypp:73-107).
 * The callback transforms vec_dev in place with work launched on `stream`; iter / residuals are -1 when the
 * reference passes them as absent (`preconditioner%apply(dx)`, `preconditioner%apply(z)`). */
typedef int (*lkb_precond_fn)(void* user, void* vec_dev, int64_t n_local, int32_t iter, double current_residual,
                              double target_residual, void* stream);
int lkb_gmres_precond(lkb_op_t A, lkb_vec_t b, lkb_vec_t x, int32_t* info, double rtol, double atol,
                      int32_t transpose, lkb_gmres_io* io, lkb_precond_fn precond, void* user);
/* right preconditioner given as an operator M (wrk = M V(k), w = A wrk; dx <- M dx): the restart cycle stays one device
 * graph with one host sync.  M's matvec counter counts its applications. */
int lkb_gmres_precond_op(lkb_op_t A, lkb_vec_t b, lkb_vec_t x, int32_t* info, double rtol, double atol,
                         int32_t transpose, lkb_gmres_io* io, lkb_op_t M);
/* fgmres(A, b, x, info, rtol, atol, preconditioner, options, transpose, meta)  GMRES/fgmres.fypp:65-260:
 * flexible GMRES, the preconditioned vectors Z(k) are stored; options / metadata as gmres. */
int lkb_fgmres(lkb_op_t A, lkb_vec_t b, lkb_vec_t x, int32_t* info, double rtol, double atol,
               int32_t transpose, lkb_gmres_io* io, lkb_precond_fn precond, void* user);
typedef struct {            /* cg_dp_opts / cg_dp_metadata : IterativeSolvers.fypp:467-507 */
    int32_t maxiter;        /* default 100 */
    int32_t n_iter, converged, info;
    double* res; int32_t res_cap, res_len;
} lkb_cg_io;
/* cg(A, b, x, info, rtol, atol, preconditioner, options, meta)  CG/CG.fypp:61-196 */
int lkb_cg(lkb_op_t A, lkb_vec_t b, lkb_vec_t x, int32_t* info, double rtol, double atol, lkb_cg_io* io);
int lkb_cg_precond(lkb_op_t A, lkb_vec_t b, lkb_vec_t x, int32_t* info, double rtol, double atol, lkb_cg_io* io,
                   lkb_precond_fn precond, void* user);
/* preconditioner given as an operator M (z = M r): the iteration stays on the device (chunks of 16 iterations, one graph
 * each when A and M are capturable).  A diagonal M (lkb_op_diag_create / lkb_op_jacobi_create) is fused into the CG vector
 * kernels.  Residual = sqrt(|r^H z|); M's matvec counter grows by n_iter + 1. */
int lkb_cg_precond_op(lkb_op_t A, lkb_vec_t b, lkb_vec_t x, int32_t* info, double rtol, double atol,
                      lkb_cg_io* io, lkb_op_t M);
/* eigs(A, X, eigvals, residuals, info, x0, kdim, tolerance, transpose)  IterativeSolvers.fypp:972-1143
 *   X: nev columns (out); eigvals: nev complex (double[2] each); residuals: nev doubles.
 *   x0 may be NULL (random start); kdim <= 0 = 4*nev; tolerance < 0 = rtol_kind. */
int lkb_eigs(lkb_op_t A, lkb_basis_t X, int nev, double* eigvals, double* residuals, int32_t* info,
             lkb_vec_t x0, int32_t kdim, double tolerance, int32_t transpose);
/* eighs(A, X, eigvals, residuals, info, x0, kdim, tolerance)  EIGHS/eighs.fypp:29-126 */
int lkb_eighs(lkb_op_t A, lkb_basis_t X, int nev, double* eigvals, double* residuals, int32_t* info,
              lkb_vec_t x0, int32_t kdim, double tolerance);
/* svds(A, U, S, V, residuals, info, u0, kdim, tolerance)  SVDS/svd_solvers.fypp:28-121 */
int lkb_svds(lkb_op_t A, lkb_basis_t U, double* S, lkb_basis_t V, int nsv, double* residuals, int32_t* info,
             lkb_vec_t u0, int32_t kdim, double tolerance);
/* kexpm_vec(c, A, b, tau, tol, info, trans, kdim)  src/Expm/ExpmLib.fypp:128-232: c = exp(tau A) b by Arnoldi + dense expm of
 * the (k+1) x (k+1) extended Hessenberg matrix (stdlib_linalg `expm`: Pade 10 + scaling and squaring, restated on the host).
 * info = dimension used when |E(kp,1) beta| <= tol, -1 when not converged within kdim (<= 0: 100) steps. */
int lkb_kexpm_vec(lkb_vec_t c, lkb_op_t A, lkb_vec_t b, double tau, double tol, int32_t* info, int32_t trans, int32_t kdim);
/* kexpm_mat(C, A, B, tau, tol, info, trans, kdim)  src/Expm/ExpmLib.fypp:234-362: C(:, :p) = exp(tau A) B(:, :p) by block Arnoldi with
 * blksize p = size(B) (pivoting QR of B, dense expm of the extended block-Hessenberg matrix per block step, error estimate
 * ||E(kp+1:kpp, :p) R||_F).  info = dimension used when the estimate is <= tol, -1 when not converged within kdim*p block steps
 * (kdim <= 0: 100) -- the reference's loop bound.  The work basis starts with room for 8 block steps and doubles on demand
 * (the reference allocates all p*(kdim*p + 1) vectors up front). */
int lkb_kexpm_mat(lkb_basis_t C, lkb_op_t A, lkb_basis_t B, int p, double tau, double tol, int32_t* info, int32_t trans, int32_t kdim);
/* krylov_exptA(vec_out, A, vec_in, tau, info, trans)  src/Expm/ExpmLib.fypp:364-392: kexpm_vec with tol = atol_kind, kdim = 30
 * (the procedure the reference plugs into abstract_exptA_linop, AbstractLinops.fypp:105-123). */
int lkb_krylov_expta(lkb_vec_t vec_out, lkb_op_t A, lkb_vec_t vec_in, double tau, int32_t* info, int32_t trans);
/* on-disk formats of the spectral solvers (IterativeSolvers.fypp:882-963).  write_results: the text table the reference
 * rewrites every step as eigs_output.txt / eighs_output.txt / svds_output.txt ('(I6,4(2X,E16.9),2X,L4)'); vals = k reals or
 * k (re, im) pairs, res is sorted ascending in place as the reference does.  save_eigenspectrum: NPY 1.0, Fortran order,
 * k x 3 (Re, Im, residual) or k x 2 (value, residual), '<f8' or '<f4'.  lkb_set_option(ctx, "write_intermediate", 1) makes
 * eigs / eighs / svds write their table every step (rank 0 only); default off (the reference: on for eigs only). */
int lkb_write_results(const char* filename, int32_t is_complex, const double* vals, double* res, int32_t k, double tol);
int lkb_save_eigenspectrum(const char* fname, int32_t is_complex, int32_t single_precision, const double* lambda,
                           const double* residuals, int32_t k);
/* host LAPACK provider for the k x k algebra of eigs/eighs/svds/krylov_schur ({s,d,c,z}geev, gees, trsen,
 * {s,d}syev / {c,z}heev, gesdd -- each kind runs the routines of its own precision, as the reference does): a shared
 * library exporting Fortran-ABI LAPACK, symbol = prefix + name + suffix (e.g. scipy's bundled OpenBLAS: prefix
 * "scipy_", suffix "_").  The reference gets these from stdlib_linalg_lapack (submodule_utility_functions.fypp:55-117). */
int lkb_set_lapack(const char* path, const char* prefix, const char* suffix);

/* ---- measurement helpers ----------------------------------------------------------------- */
/* Synthetic CSR matrix of BASELINE config 5 generated ON THE DEVICE (SURVEY.md 8d: `per_row` column indices per row
 * drawn uniformly, sorted, values N(0,1)[+ i N(0,1)]), rows [row0, row0 + m_local) of the global matrix, counter RNG
 * keyed on (seed, global row, slot) -- the oracle regenerates the identical matrix on the host.  The three arrays are
 * cudaMalloc'ed; hand them to lkb_op_csr_create_device(adopt = 1) or release them with lkb_dev_free. */
int lkb_csr_random_device(lkb_ctx_t ctx, int kind, int64_t m_local, int64_t row0, int64_t n, int32_t per_row, uint64_t seed,
                          int64_t** rowptr_dev, int32_t** col_dev, void** val_dev);
int lkb_dev_free(void* devptr);
/* per-kernel-class device time (ms) accumulated since lkb_set_profile(ctx, 1), measured with CUDA
 * events on the context stream (graphs are bypassed while profiling).  8 slots:
 * [0] matvec, [1] multi-dot, [2] multi-axpy, [3] other, [4] fused axpy+dot, [5..7] reserved */
int lkb_set_profile(lkb_ctx_t ctx, int enable);
int lkb_get_profile(lkb_ctx_t ctx, double* ms8, int64_t* launches8);
int64_t lkb_kernel_launches(lkb_ctx_t ctx);               /* kernels launched since context creation */
/* in-kernel timeline of the last reduction kernel launched (k_multidot / k_axpy_dot): per CTA {start, main loop done,
 * ticket taken, -} in %globaltimer ns, then at word 4096 {stage-2 start, stage-2 done, allreduce done} of the last CTA.
 * Used by profiles/ktime_probe.py to split a launch into ramp-up / streaming / reduction tail. */
int lkb_debug_ktime(lkb_ctx_t ctx, int enable);
int lkb_debug_ktime_read(lkb_ctx_t ctx, uint64_t* out, int nwords);

#ifdef __cplusplus
}
#endif
#endif /* LKB_H */
