"""Test problems of the preconditioner tests (tests/test_gpu_precond.py, tests/mgpu_precond_worker.py) and of
profiles/precond_ab.py: a variable-coefficient diffusion matrix whose diagonal varies over four orders of magnitude, the
case a Jacobi preconditioner is for."""
import numpy as np


def varcoef_spd_csr(dims, seed, dtype=np.float64):
    """3-D 7-point diffusion on an nx x ny x nz grid (row i + nx*(j + ny*k)), cell coefficient 10^(4u-2) with u uniform
    from `seed`, harmonic-mean face coefficients, Dirichlet boundary faces (the cell's own coefficient on the diagonal).
    Real kinds: symmetric positive definite.  Complex kinds: Hermitian, each off-diagonal pair rotated by a seeded phase,
    the diagonal 5 % above the row's off-diagonal sum (strictly diagonally dominant, so positive definite).
    Returns (rowptr int64, col int32, val dtype, diag dtype)."""
    import scipy.sparse as sp
    nx, ny, nz = dims
    n = nx * ny * nz
    cplx = np.issubdtype(np.dtype(dtype), np.complexfloating)
    rng = np.random.default_rng(seed)
    k = 10.0 ** (4.0 * rng.random(n) - 2.0)
    idx = np.arange(n).reshape(nz, ny, nx)
    rows, cols, vals = [], [], []
    offsum = np.zeros(n); bnd = np.zeros(n)
    for axis in (2, 1, 0):
        m = idx.shape[axis]
        a = idx.take(range(0, m - 1), axis=axis).ravel(); b = idx.take(range(1, m), axis=axis).ravel()
        f = 2.0 * k[a] * k[b] / (k[a] + k[b])
        v = -f * np.exp(1j * rng.uniform(-np.pi, np.pi, f.size)) if cplx else -f
        rows += [a, b]; cols += [b, a]; vals += [v, np.conj(v)]
        np.add.at(offsum, a, f); np.add.at(offsum, b, f)
        for face in (idx.take([0], axis=axis).ravel(), idx.take([m - 1], axis=axis).ravel()):
            np.add.at(bnd, face, k[face])
    diag = (1.05 if cplx else 1.0) * offsum + bnd
    rows.append(np.arange(n)); cols.append(np.arange(n)); vals.append(diag.astype(np.complex128) if cplx else diag)
    S = sp.coo_matrix((np.concatenate(vals), (np.concatenate(rows), np.concatenate(cols))), shape=(n, n)).tocsr()
    S.sum_duplicates(); S.sort_indices()
    return (S.indptr.astype(np.int64), S.indices.astype(np.int32), S.data.astype(dtype), diag.astype(dtype))
