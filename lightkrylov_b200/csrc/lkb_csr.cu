// lkb_csr.cu -- CSR operator set-up on the device: validation of the user's arrays, the explicit transpose that
// makes `rmatvec` a gather (no atomics, deterministic), and a seeded synthetic generator for BASELINE config C5.
//
// Reference contract: `abstract_linop_*` with `matvec` / `rmatvec` (src/AbstractTypes/AbstractLinops.fypp:58-87);
// a user's CSR type would store (rowptr, col, val) and loop over rows.  Everything here is SET-UP (once per
// operator): the hot path is k_csr in kernels_ops.cu.
//
// Transpose = stable LSD radix sort of the nnz by column (CUB DeviceRadixSort on (col, original position) pairs,
// library code, set-up only).  Stability keeps the entries of one column in ascending row order, so the
// summation order of A^H u -- and hence the result -- is a fixed function of the matrix, identical to the host
// counting sort of round 1.  1.6e9 nnz (C5 at BASELINE size) transpose in well under a second; the round-1 host
// build needed minutes and ~70 GB of host memory.
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <algorithm>
#include <cub/device/device_radix_sort.cuh>
#include "../../include/lkb.h"
#include "lkb_internal.h"
#include "lkb_rng.h"

using namespace lkb;

namespace {

// err[0]: 1 = rowptr[0] != 0, 2 = rowptr decreasing, 3 = column index out of range, 4 = rowptr[rows] != nnz
__global__ void k_csr_validate(int64_t rows, int64_t ncols, int64_t nnz, const int64_t* __restrict__ rowptr,
                               const int32_t* __restrict__ col, int* __restrict__ err)
{
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    const int64_t t0 = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t0 == 0) {
        if (rowptr[0] != 0) atomicMax(err, 1);
        if (rowptr[rows] != nnz) atomicMax(err, 4);
    }
    for (int64_t i = t0; i < rows; i += stride)
        if (rowptr[i + 1] < rowptr[i]) atomicMax(err, 2);
    for (int64_t q = t0; q < nnz; q += stride) {
        const int32_t cq = col[q];
        if (cq < 0 || (int64_t)cq >= ncols) atomicMax(err, 3);
    }
}

__global__ void k_iota_u32(uint32_t* __restrict__ p, int64_t n) {
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) p[i] = (uint32_t)i;
}

// t_rowptr from the sorted column keys: position d starts every column in (key[d-1], key[d]]
__global__ void k_csr_trowptr(int64_t nnz, int64_t ncols, const uint32_t* __restrict__ keys, int64_t* __restrict__ trp) {
    for (int64_t d = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; d <= nnz; d += (int64_t)gridDim.x * blockDim.x) {
        const int64_t prev = d == 0 ? -1 : (int64_t)keys[d - 1];
        const int64_t cur = d == nnz ? ncols : (int64_t)keys[d];
        for (int64_t cidx = prev + 1; cidx <= cur; ++cidx) trp[cidx] = d;
    }
}

// t_col[d] = row of original entry perm[d] (binary search in rowptr), t_val[d] = val[perm[d]]
template <typename E>
__global__ void k_csr_tfill(int64_t nnz, int64_t rows, const int64_t* __restrict__ rowptr, const uint32_t* __restrict__ perm,
                            const E* __restrict__ val, int32_t* __restrict__ tcol, E* __restrict__ tval) {
    for (int64_t d = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; d < nnz; d += (int64_t)gridDim.x * blockDim.x) {
        const int64_t q = (int64_t)perm[d];
        int64_t lo = 0, hi = rows;                    // largest i with rowptr[i] <= q
        while (hi - lo > 1) {
            const int64_t mid = (lo + hi) >> 1;
            if (rowptr[mid] <= q) lo = mid; else hi = mid;
        }
        tcol[d] = (int32_t)lo;
        tval[d] = val[q];
    }
}

// Synthetic C5 matrix (SURVEY 8d): `per_row` column indices per row drawn uniformly from [0, n) with the counter RNG
// of lkb_rng.h, sorted within the row (duplicate columns are kept as separate entries = "duplicates summed"),
// values N(0,1) (+ i N(0,1)) keyed on the position in the sorted row.  The oracle builds the identical matrix
// from its own copy of the generator: col = floor(u(seed, q) * n), val = normal(seed + 1, q), q = row * per_row + slot.
template <typename E, bool CPLX>
__global__ void k_csr_random(int64_t m_local, int64_t row0, int64_t n, int per_row, uint64_t seed_col, uint64_t seed_val,
                             int64_t* __restrict__ rowptr, int32_t* __restrict__ col, E* __restrict__ val)
{
    constexpr int MAXPR = 64;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i <= m_local; i += (int64_t)gridDim.x * blockDim.x) {
        rowptr[i] = i * per_row;
        if (i == m_local) break;
        int32_t cbuf[MAXPR];
        const uint64_t g0 = (uint64_t)(row0 + i) * (uint64_t)per_row;
        for (int s = 0; s < per_row; ++s) {
            int32_t cv = (int32_t)floor(rng_uniform(seed_col, g0 + s, 0) * (double)n);
            if (cv >= n) cv = (int32_t)(n - 1);
            int t = s;                                  // insertion sort (per_row <= 64)
            while (t > 0 && cbuf[t - 1] > cv) { cbuf[t] = cbuf[t - 1]; --t; }
            cbuf[t] = cv;
        }
        for (int s = 0; s < per_row; ++s) {
            const int64_t q = i * per_row + s;
            col[q] = cbuf[s];
            Scalar sc;
            sc.re = rng_normal(seed_val, g0 + s, 0);
            sc.im = CPLX ? rng_normal(seed_val, g0 + s, 1) : 0.0;
            E v; from_scalar(sc, v);
            val[q] = v;
        }
    }
}

// ---- L2-blocked layout (column blocks) ---------------------------------------------------------------------
// A random sparse matrix gathers x with no locality: once x no longer fits in L2 every gather is a DRAM sector
// (and a TLB miss).  Measured on C5 at BASELINE size (x = 640 MB): 0.97 TB/s algorithmic for matvec, against
// 2.85 TB/s at 1/10 scale where x (64 MB) still half-fits.  The remedy is the classic one: cut the COLUMN space
// into blocks whose slice of x stays L2 resident (default 48 MB, LKB_CSR_SLICE_MB) and sweep the matrix block by
// block; y is accumulated across the blocks (read-modify-write per block, the price of the blocking).
// Layout: the non-zeros stably sorted by column block (one 1-pass CUB radix sort on a <= 8-bit key), so inside a
// block they are still ordered by row and by their original position in the row; tab[b * (rows + 1) + r] is the
// position of the first entry of (block b, row r) -- a per-block CSR row pointer into the blocked arrays.
// The summation order of every row is a fixed function of the matrix => deterministic, no atomics.
__global__ void k_blk_keys(int64_t nnz, int64_t cw, const int32_t* __restrict__ col, uint8_t* __restrict__ keys, uint32_t* __restrict__ iota) {
    for (int64_t q = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; q < nnz; q += (int64_t)gridDim.x * blockDim.x) {
        keys[q] = (uint8_t)((int64_t)col[q] / cw);
        iota[q] = (uint32_t)q;
    }
}
template <typename E>
__global__ void k_blk_gather(int64_t nnz, int64_t rows, const int64_t* __restrict__ rowptr, const uint32_t* __restrict__ perm,
                             const int32_t* __restrict__ col, const E* __restrict__ val, int32_t* __restrict__ bcol,
                             E* __restrict__ bval, uint32_t* __restrict__ brow) {
    for (int64_t d = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; d < nnz; d += (int64_t)gridDim.x * blockDim.x) {
        const int64_t q = (int64_t)perm[d];
        int64_t lo = 0, hi = rows;                    // largest i with rowptr[i] <= q
        while (hi - lo > 1) {
            const int64_t mid = (lo + hi) >> 1;
            if (rowptr[mid] <= q) lo = mid; else hi = mid;
        }
        brow[d] = (uint32_t)lo;
        bcol[d] = col[q];
        bval[d] = val[q];
    }
}
// tab[key] = first position whose (block, row) key is >= key, key = block * (rows + 1) + row
__global__ void k_blk_table(int64_t nnz, int64_t rows, int nb, const uint8_t* __restrict__ bkey, const uint32_t* __restrict__ brow,
                            uint32_t* __restrict__ tab) {
    const int64_t nkeys = (int64_t)nb * (rows + 1);
    for (int64_t d = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; d <= nnz; d += (int64_t)gridDim.x * blockDim.x) {
        const int64_t prev = d == 0 ? -1 : (int64_t)bkey[d - 1] * (rows + 1) + (int64_t)brow[d - 1];
        const int64_t cur = d == nnz ? nkeys - 1 : (int64_t)bkey[d] * (rows + 1) + (int64_t)brow[d];
        for (int64_t key = prev + 1; key <= cur; ++key) tab[key] = (uint32_t)d;
    }
}

int grid_for(int64_t n, int sms) {
    int64_t nb = (n + 255) / 256;
    if (nb < 1) nb = 1;
    if (nb > (int64_t)sms * 32) nb = (int64_t)sms * 32;
    return (int)nb;
}

int pick_lpr(int64_t nnz, int64_t rows) {
    const double avg = rows > 0 ? (double)nnz / (double)rows : 0.0;
    return avg >= 48 ? 32 : (avg >= 24 ? 16 : (avg >= 10 ? 8 : 4));
}

}  // namespace

namespace lkb {

void csr_block_device(lkb_ctx_s* c, int kind, int64_t rows, int64_t ncols, int64_t nnz, CudaPtr<int64_t>& rowptr, CudaPtr<int32_t>& col,
                      CudaPtr<void>& val, CsrBlocked* blk, CsrBlockedMem* mem);

// Validate (rowptr, col) ON THE DEVICE and build the explicit transpose.  `rows` = local rows, `ncols_index` =
// size of the column index space (global n for a row-sharded operator).  op->rowptr / col / val must already
// point at device arrays owned by the operator.  Nothing can fail once the L2 blocking may have released them.
int csr_finish_device(lkb_ctx_s* c, lkb_op_s* op, int kind, int64_t rows, int64_t ncols_index) {
    const size_t es = kind_size(kind);
    int64_t nnz = 0;
    LKB_CUDA(cudaMemcpy(&nnz, op->rowptr.get() + rows, sizeof(int64_t), cudaMemcpyDeviceToHost));
    if (nnz < 0 || nnz >= (int64_t)0xffffffffLL) { set_error("csr: nnz = %lld is outside [0, 2^32-1)", (long long)nnz); return LKB_ERR_ARG; }
    if (rows > 2147483647LL || ncols_index > 2147483647LL) { set_error("csr: more than 2^31-1 rows / columns per rank"); return LKB_ERR_ARG; }
    // ---- validation: rowptr[0] == 0, rowptr non-decreasing, 0 <= col < ncols_index (ADVICE r01: an out-of-range
    // index, e.g. 1-based Fortran indices, must be an LKB_ERR_ARG, not heap corruption) ----
    CudaPtr<int> derr;
    LKB_TRY(cuda_alloc(derr, sizeof(int)));
    LKB_CUDA(cudaMemsetAsync(derr, 0, sizeof(int), c->stream));
    k_csr_validate<<<grid_for(std::max(rows, nnz), c->sms), 256, 0, c->stream>>>(rows, ncols_index, nnz, op->rowptr, op->col, derr);
    int herr = 0;
    LKB_CUDA(cudaMemcpyAsync(&herr, derr, sizeof(int), cudaMemcpyDeviceToHost, c->stream));
    LKB_CUDA(cudaStreamSynchronize(c->stream));
    if (herr) {
        static const char* what[] = {"", "rowptr[0] != 0", "rowptr is not non-decreasing", "column index out of range (indices are 0-based)",
                                     "rowptr[rows] != nnz"};
        set_error("csr: invalid matrix: %s", what[herr]);
        return LKB_ERR_ARG;
    }
    op->lpr = pick_lpr(nnz, rows); op->t_lpr = pick_lpr(nnz, ncols_index);
    // ---- transpose: stable radix sort of (col, position) ----
    const int64_t nn = std::max<int64_t>(nnz, 1);
    CudaPtr<uint32_t> keys_out, perm_in, perm_out; CudaPtr<void> tmp;
    LKB_TRY(cuda_alloc(keys_out, nn * sizeof(uint32_t)));
    LKB_TRY(cuda_alloc(perm_in, nn * sizeof(uint32_t)));
    LKB_TRY(cuda_alloc(perm_out, nn * sizeof(uint32_t)));
    k_iota_u32<<<grid_for(nnz, c->sms), 256, 0, c->stream>>>(perm_in, nnz);
    int end_bit = 1;
    while (end_bit < 32 && ((int64_t)1 << end_bit) < ncols_index) ++end_bit;
    size_t tmp_bytes = 0;
    LKB_CUDA(cub::DeviceRadixSort::SortPairs(nullptr, tmp_bytes, (const uint32_t*)op->col.get(), keys_out.get(), perm_in.get(), perm_out.get(), nnz, 0, end_bit, c->stream));
    LKB_TRY(cuda_alloc(tmp, std::max<size_t>(tmp_bytes, 16)));
    LKB_CUDA(cub::DeviceRadixSort::SortPairs(tmp, tmp_bytes, (const uint32_t*)op->col.get(), keys_out.get(), perm_in.get(), perm_out.get(), nnz, 0, end_bit, c->stream));
    LKB_TRY(cuda_alloc(op->t_rowptr, (ncols_index + 1) * sizeof(int64_t)));
    LKB_TRY(cuda_alloc(op->t_col, nn * sizeof(int32_t)));
    LKB_TRY(cuda_alloc(op->t_val, nn * es));
    k_csr_trowptr<<<grid_for(nnz + 1, c->sms), 256, 0, c->stream>>>(nnz, ncols_index, keys_out, op->t_rowptr);
    const int g = grid_for(nnz, c->sms);
    switch (kind) {
        case KS: k_csr_tfill<float><<<g, 256, 0, c->stream>>>(nnz, rows, op->rowptr, perm_out, (const float*)op->val.get(), op->t_col, (float*)op->t_val.get()); break;
        case KD: k_csr_tfill<double><<<g, 256, 0, c->stream>>>(nnz, rows, op->rowptr, perm_out, (const double*)op->val.get(), op->t_col, (double*)op->t_val.get()); break;
        case KC: k_csr_tfill<float2><<<g, 256, 0, c->stream>>>(nnz, rows, op->rowptr, perm_out, (const float2*)op->val.get(), op->t_col, (float2*)op->t_val.get()); break;
        default: k_csr_tfill<double2><<<g, 256, 0, c->stream>>>(nnz, rows, op->rowptr, perm_out, (const double2*)op->val.get(), op->t_col, (double2*)op->t_val.get()); break;
    }
    LKB_CUDA(cudaGetLastError());
    LKB_CUDA(cudaStreamSynchronize(c->stream));
    keys_out.reset(); perm_in.reset(); perm_out.reset(); tmp.reset();
    // L2 blocking when the gathered vector exceeds L2 (no-op otherwise).  Row-sharded operator: only the forward
    // orientation (it gathers from the full-length x_full; the transposed one gathers from this rank's slab of u)
    csr_block_device(c, kind, rows, ncols_index, nnz, op->rowptr, op->col, op->val, &op->blk, &op->blk_mem);
    if (!op->dist) csr_block_device(c, kind, ncols_index, rows, nnz, op->t_rowptr, op->t_col, op->t_val, &op->t_blk, &op->t_blk_mem);
    return 0;
}

// The L2-blocked copy of a CSR matrix in nb column blocks of width cw.  On success it replaces the plain arrays (they are
// released) and blk views mem.
static int csr_blocked_copy(lkb_ctx_s* c, int kind, int64_t rows, int64_t nnz, int nb, int64_t cw, CudaPtr<int64_t>& rowptr,
                            CudaPtr<int32_t>& col, CudaPtr<void>& val, CsrBlocked* blk, CsrBlockedMem* mem) {
    const size_t es = kind_size(kind);
    CudaPtr<uint8_t> keys, keys_out; CudaPtr<uint32_t> iota, perm, brow; CudaPtr<void> tmp;
    CsrBlockedMem b;
    LKB_TRY(cuda_alloc(keys, nnz)); LKB_TRY(cuda_alloc(keys_out, nnz));
    LKB_TRY(cuda_alloc(iota, nnz * sizeof(uint32_t))); LKB_TRY(cuda_alloc(perm, nnz * sizeof(uint32_t)));
    k_blk_keys<<<grid_for(nnz, c->sms), 256, 0, c->stream>>>(nnz, cw, col, keys, iota);
    int end_bit = 1; while ((1 << end_bit) < nb) ++end_bit;
    size_t tmp_bytes = 0;
    LKB_CUDA(cub::DeviceRadixSort::SortPairs(nullptr, tmp_bytes, keys.get(), keys_out.get(), iota.get(), perm.get(), nnz, 0, end_bit, c->stream));
    LKB_TRY(cuda_alloc(tmp, std::max<size_t>(tmp_bytes, 16)));
    LKB_CUDA(cub::DeviceRadixSort::SortPairs(tmp, tmp_bytes, keys.get(), keys_out.get(), iota.get(), perm.get(), nnz, 0, end_bit, c->stream));
    LKB_CUDA(cudaStreamSynchronize(c->stream));
    keys.reset(); iota.reset(); tmp.reset();
    LKB_TRY(cuda_alloc(brow, nnz * sizeof(uint32_t)));
    LKB_TRY(cuda_alloc(b.col, nnz * sizeof(int32_t)));
    LKB_TRY(cuda_alloc(b.val, nnz * es));
    const int g = grid_for(nnz, c->sms);
    switch (kind) {
        case KS: k_blk_gather<float><<<g, 256, 0, c->stream>>>(nnz, rows, rowptr, perm, col, (const float*)val.get(), b.col, (float*)b.val.get(), brow); break;
        case KD: k_blk_gather<double><<<g, 256, 0, c->stream>>>(nnz, rows, rowptr, perm, col, (const double*)val.get(), b.col, (double*)b.val.get(), brow); break;
        case KC: k_blk_gather<float2><<<g, 256, 0, c->stream>>>(nnz, rows, rowptr, perm, col, (const float2*)val.get(), b.col, (float2*)b.val.get(), brow); break;
        default: k_blk_gather<double2><<<g, 256, 0, c->stream>>>(nnz, rows, rowptr, perm, col, (const double2*)val.get(), b.col, (double2*)b.val.get(), brow); break;
    }
    LKB_CUDA(cudaGetLastError());
    LKB_CUDA(cudaStreamSynchronize(c->stream));
    perm.reset();
    LKB_TRY(cuda_alloc(b.tab, (size_t)nb * (rows + 1) * sizeof(uint32_t)));
    k_blk_table<<<grid_for(nnz + 1, c->sms), 256, 0, c->stream>>>(nnz, rows, nb, keys_out, brow, b.tab);
    LKB_CUDA(cudaGetLastError());
    LKB_CUDA(cudaStreamSynchronize(c->stream));
    rowptr.reset(); col.reset(); val.reset();
    blk->nb = nb; blk->cw = cw; blk->rows = rows; blk->nnz = nnz; blk->tab = b.tab; blk->col = b.col; blk->val = b.val;
    *mem = std::move(b);
    return 0;
}

// Build the L2-blocked copy of a CSR matrix (rows x ncols, nnz entries) when the gathered vector is too large for L2.
// blk.nb == 0 afterwards: not blocked.  A failure here (in practice: not enough memory for the second copy) is not fatal:
// the plain arrays are only released after everything else succeeded, so the matrix simply stays unblocked.
void csr_block_device(lkb_ctx_s* c, int kind, int64_t rows, int64_t ncols, int64_t nnz, CudaPtr<int64_t>& rowptr, CudaPtr<int32_t>& col,
                      CudaPtr<void>& val, CsrBlocked* blk, CsrBlockedMem* mem) {
    blk->nb = 0;
    const size_t es = kind_size(kind);
    // slice / threshold: lkb_set_option(ctx, "csr_slice_kb" | "csr_block_min_kb", v); defaults 48 MB / 96 MB
    const int64_t slice_b = (int64_t)c->csr_slice_kb * 1024, min_b = (int64_t)c->csr_block_min_kb * 1024;
    if (slice_b <= 0 || (int64_t)ncols * (int64_t)es < min_b) return;                 // x (nearly) fits in L2: plain CSR
    if (nnz < 1) return;
    int64_t cw = (slice_b / (int64_t)es + 1023) / 1024 * 1024;
    int nb = (int)((ncols + cw - 1) / cw);
    if (nb > 255) { nb = 255; cw = ((ncols + nb - 1) / nb + 1023) / 1024 * 1024; nb = (int)((ncols + cw - 1) / cw); }
    if (nb < 2) return;
    if ((int64_t)nb * (rows + 1) >= (int64_t)1 << 40) return;
    if (csr_blocked_copy(c, kind, rows, nnz, nb, cw, rowptr, col, val, blk, mem) != 0) cudaGetLastError();
}

// host arrays -> device copies owned by the operator, then the common device set-up
int csr_build(lkb_ctx_s* c, lkb_op_s* op, int kind, int64_t rows, int64_t ncols_index, const int64_t* rowptr,
              const int32_t* col, const void* val) {
    if (!rowptr) { set_error("csr: rowptr is null"); return LKB_ERR_ARG; }
    const int64_t nnz = rowptr[rows];
    if (nnz < 0) { set_error("csr: rowptr[rows] = %lld < 0", (long long)nnz); return LKB_ERR_ARG; }
    if (nnz > 0 && (!col || !val)) { set_error("csr: col / val are null with nnz = %lld", (long long)nnz); return LKB_ERR_ARG; }
    const size_t es = kind_size(kind);
    LKB_TRY(cuda_alloc(op->rowptr, (rows + 1) * sizeof(int64_t)));
    LKB_TRY(cuda_alloc(op->col, std::max<int64_t>(nnz, 1) * sizeof(int32_t)));
    LKB_TRY(cuda_alloc(op->val, std::max<int64_t>(nnz, 1) * es));
    LKB_CUDA(cudaMemcpy(op->rowptr, rowptr, (rows + 1) * sizeof(int64_t), cudaMemcpyHostToDevice));
    if (nnz > 0) {
        LKB_CUDA(cudaMemcpy(op->col, col, nnz * sizeof(int32_t), cudaMemcpyHostToDevice));
        LKB_CUDA(cudaMemcpy(op->val, val, nnz * es, cudaMemcpyHostToDevice));
    }
    return csr_finish_device(c, op, kind, rows, ncols_index);
}

}  // namespace lkb

extern "C" {

int lkb_op_csr_create(lkb_ctx_t c, int kind, int64_t m, int64_t n, const int64_t* rowptr, const int32_t* col,
                      const void* val, lkb_op_t* A) {
    if (!c || !A || !rowptr || m < 1 || n < 1 || kind < 0 || kind > 3) { set_error("csr_create: bad arguments"); return LKB_ERR_ARG; }
    if (c->world > 1) { set_error("lkb_op_csr_create is single-rank; use lkb_op_csr_create_dist for a row-sharded matrix"); return LKB_ERR_ARG; }
    cudaSetDevice(c->dev);
    OpOwner op(new lkb_op_s());
    op->ctx = c; op->type = OP_CSR; op->kind = kind; op->m = m; op->n = n; op->uid = next_uid();
    LKB_TRY(csr_build(c, op, kind, m, n, rowptr, col, val));
    *A = op.release();
    return 0;
}

int lkb_op_csr_create_device(lkb_ctx_t c, int kind, int64_t m, int64_t n, int64_t* rowptr_dev, int32_t* col_dev,
                             void* val_dev, int32_t adopt, lkb_op_t* A) {
    if (!c || !A || !rowptr_dev || !col_dev || !val_dev || m < 1 || n < 1 || kind < 0 || kind > 3) { set_error("csr_create_device: bad arguments"); return LKB_ERR_ARG; }
    if (c->world > 1) { set_error("lkb_op_csr_create_device is single-rank"); return LKB_ERR_ARG; }
    cudaSetDevice(c->dev);
    OpOwner op(new lkb_op_s());
    op->ctx = c; op->type = OP_CSR; op->kind = kind; op->m = m; op->n = n; op->uid = next_uid();
    if (adopt) {
        op->rowptr.reset(rowptr_dev); op->col.reset(col_dev); op->val.reset(val_dev);
    } else {
        int64_t nnz = 0;            // (a negative nnz is rejected by csr_finish_device)
        LKB_CUDA(cudaMemcpy(&nnz, rowptr_dev + m, sizeof(int64_t), cudaMemcpyDeviceToHost));
        const size_t es = kind_size(kind);
        const int64_t nn = std::max<int64_t>(nnz, 1);
        LKB_TRY(cuda_alloc(op->rowptr, (m + 1) * sizeof(int64_t)));
        LKB_TRY(cuda_alloc(op->col, nn * sizeof(int32_t)));
        LKB_TRY(cuda_alloc(op->val, nn * es));
        LKB_CUDA(cudaMemcpy(op->rowptr, rowptr_dev, (m + 1) * sizeof(int64_t), cudaMemcpyDeviceToDevice));
        if (nnz > 0) {
            LKB_CUDA(cudaMemcpy(op->col, col_dev, nnz * sizeof(int32_t), cudaMemcpyDeviceToDevice));
            LKB_CUDA(cudaMemcpy(op->val, val_dev, nnz * es, cudaMemcpyDeviceToDevice));
        }
    }
    if (int r = csr_finish_device(c, op, kind, m, n)) {
        if (adopt) { op->rowptr.release(); op->col.release(); op->val.release(); }    // the caller keeps ownership on failure
        return r;
    }
    *A = op.release();
    return 0;
}

int lkb_csr_random_device(lkb_ctx_t c, int kind, int64_t m_local, int64_t row0, int64_t n, int32_t per_row, uint64_t seed,
                          int64_t** rowptr_dev, int32_t** col_dev, void** val_dev) {
    if (!c || !rowptr_dev || !col_dev || !val_dev || m_local < 1 || n < 1 || n > 2147483647LL || per_row < 1 || per_row > 64 ||
        kind < 0 || kind > 3) { set_error("csr_random: bad arguments (1 <= per_row <= 64)"); return LKB_ERR_ARG; }
    cudaSetDevice(c->dev);
    const int64_t nnz = m_local * per_row;
    const size_t es = kind_size(kind);
    CudaPtr<int64_t> rp; CudaPtr<int32_t> ci; CudaPtr<void> va;
    LKB_TRY(cuda_alloc(rp, (m_local + 1) * sizeof(int64_t)));
    LKB_TRY(cuda_alloc(ci, nnz * sizeof(int32_t)));
    LKB_TRY(cuda_alloc(va, nnz * es));
    const uint64_t sc = mix64(seed), sv = mix64(seed + 1);
    const int g = grid_for(m_local + 1, c->sms);
    switch (kind) {
        case KS: k_csr_random<float, false><<<g, 256, 0, c->stream>>>(m_local, row0, n, per_row, sc, sv, rp, ci, (float*)va.get()); break;
        case KD: k_csr_random<double, false><<<g, 256, 0, c->stream>>>(m_local, row0, n, per_row, sc, sv, rp, ci, (double*)va.get()); break;
        case KC: k_csr_random<float2, true><<<g, 256, 0, c->stream>>>(m_local, row0, n, per_row, sc, sv, rp, ci, (float2*)va.get()); break;
        default: k_csr_random<double2, true><<<g, 256, 0, c->stream>>>(m_local, row0, n, per_row, sc, sv, rp, ci, (double2*)va.get()); break;
    }
    LKB_TRY(check_launch(c, "csr_random"));
    LKB_CUDA(cudaStreamSynchronize(c->stream));
    *rowptr_dev = rp.release(); *col_dev = ci.release(); *val_dev = va.release();
    return 0;
}

int lkb_dev_free(void* devptr) {
    if (devptr) cudaFree(devptr);
    return 0;
}

}  // extern "C"
