"""Host reference of the Chebyshev preconditioner (include/lkb.h: lkb_op_chebyshev_create) and the matrices its tests use
(tests/test_chebyshev_host.py, tests/test_gpu_chebyshev.py, tests/mgpu_chebyshev_worker.py, profiles/chebyshev_ab.py)."""
import numpy as np


def coefficients(m, a, b):
    """theta and the (alpha_k, beta_k) = (rho_k rho_{k-1}, 2 rho_k / delta) of steps k = 1 .. m-1, in double."""
    theta, delta = (b + a) / 2.0, (b - a) / 2.0
    sigma = theta / delta
    rho, steps = 1.0 / sigma, []
    for _ in range(1, m):
        rho_k = 1.0 / (2.0 * sigma - rho)
        steps.append((rho_k * rho, 2.0 * rho_k / delta))
        rho = rho_k
    return theta, steps


def chebyshev_apply(op, invd, r, m, a, b, trans=False):
    """M r (trans: M^H r) by the recurrence of lkb_op_chebyshev_create, in the precision of r.  op: an oracle.Op (applied with
    Op.apply), or the 1-D array d of a diagonal operator (a plain elementwise product).  invd: D^-1, a scalar or a vector."""
    if isinstance(op, np.ndarray):
        apply = (lambda x: np.conj(op) * x) if trans else (lambda x: op * x)
    else:
        apply = lambda x: op.apply(x, trans)                                      # noqa: E731
    iv = np.conj(invd) if trans else invd
    theta, steps = coefficients(m, a, b)
    z = (iv * r) * r.real.dtype.type(1.0 / theta)
    d = z
    for alpha, beta in steps:
        s = iv * (r - apply(z))
        d = d * r.real.dtype.type(alpha) + s * r.real.dtype.type(beta)
        z = z + d
    return z


def chebyshev_closed_form(A, m, a, b):
    """M = D^{-1/2} (I - R_m(B)) B^{-1} D^{-1/2}, B = D^{-1/2} A D^{-1/2}, R_m(l) = T_m((theta - l)/delta) / T_m(sigma), for a
    dense Hermitian A with a positive diagonal (eigendecomposition of B, in double)."""
    from numpy.polynomial import chebyshev as ch
    dh = 1.0 / np.sqrt(np.diag(A).real)
    B = dh[:, None] * A * dh[None, :]
    lam, Q = np.linalg.eigh(B)
    theta, delta = (b + a) / 2.0, (b - a) / 2.0
    Tm = ch.Chebyshev.basis(m)
    f = (1.0 - Tm((theta - lam) / delta) / Tm(theta / delta)) / lam
    return dh[:, None] * ((Q * f) @ Q.conj().T) * dh[None, :]


def gershgorin(S):
    """max_r sum_c |a_rc / a_rr| of a scipy sparse or dense matrix (duplicates summed)."""
    import scipy.sparse as sp
    S = sp.csr_matrix(S, copy=True)
    S = S.astype(np.complex128 if np.iscomplexobj(S.data) else np.float64)      # in double, as the library computes it
    S.sum_duplicates()
    rows = np.abs(S).sum(axis=1).A.ravel()
    return float(np.max(rows / np.abs(S.diagonal())))


def stencil_csr(dims, coef, dtype=None):
    """The 5- (dims = (nx, ny)) or 7-point stencil operator of lkb_op_stencil{5,7}_create as a scipy CSR matrix: row
    p = i + nx (j + ny k), coef = (centre, -x, +x, -y, +y, -z, +z), homogeneous Dirichlet outside the grid.  dtype: that
    of coef by default."""
    import scipy.sparse as sp
    dtype = np.asarray(coef).dtype if dtype is None else dtype
    dims = tuple(dims) + (1,) * (3 - len(dims))
    nx, ny, nz = dims
    n = nx * ny * nz
    idx = np.arange(n).reshape(nz, ny, nx)
    rows, cols, vals = [idx.ravel()], [idx.ravel()], [np.full(n, coef[0])]
    for q, (axis, off) in enumerate([(2, -1), (2, 1), (1, -1), (1, 1), (0, -1), (0, 1)], start=1):
        if q >= len(coef):
            break
        m = idx.shape[axis]
        keep = range(1, m) if off < 0 else range(0, m - 1)
        src = idx.take(keep, axis=axis).ravel()
        dst = idx.take([k + off for k in keep], axis=axis).ravel()
        rows.append(src); cols.append(dst); vals.append(np.full(src.size, coef[q]))
    S = sp.coo_matrix((np.concatenate(vals).astype(dtype), (np.concatenate(rows), np.concatenate(cols))), shape=(n, n)).tocsr()
    S.sort_indices()
    return S
