"""Host reference of the multigrid preconditioner (include/lkb.h: lkb_op_multigrid_create), in complex double with scipy
(tests/test_multigrid_host.py, tests/test_gpu_multigrid.py, profiles/multigrid_ab.py)."""
import numpy as np
import scipy.sparse as sp

from chebyshev_cases import coefficients, stencil_csr

CAP = 512                        # largest coarsest level (dense inverse)


def interp1(n):
    """1-D linear interpolation: coarse i <-> fine 2i+1, nc = n // 2, coarse points outside the grid are zero."""
    nc = n // 2
    rows, cols, vals = [], [], []
    for i in range(nc):
        for f, w in ((2 * i, 0.5), (2 * i + 1, 1.0), (2 * i + 2, 0.5)):
            if f < n:
                rows.append(f); cols.append(i); vals.append(w)
    return sp.csr_matrix((vals, (rows, cols)), shape=(n, nc))


def _tri(n, cm, cp):
    return sp.diags([np.full(n - 1, cm), np.full(n, -(cm + cp)), np.full(n - 1, cp)], [-1, 0, 1], shape=(n, n),
                    dtype=complex).tocsr()


def _tensor(Ps):
    P = Ps[0]
    for P1 in Ps[1:]:
        P = sp.kron(P1, P).tocsr()                   # x fastest
    return P


def level_matrix(dims, c0, cm, cp, e):
    """The stencil of a level with its centre corrections: c0 + sum_d [i_d = n_d - 1] e_d on the diagonal."""
    dim = len(dims)
    coef = [c0] + [v for d in range(dim) for v in (cm[d], cp[d])]
    A = stencil_csr(dims, np.array(coef, dtype=complex))
    idx = np.indices(dims[::-1]).reshape(dim, -1)[::-1]           # idx[d] = the index along axis d (x fastest)
    corr = sum(np.where(idx[d] == dims[d] - 1, e[d], 0.0) for d in range(dim))
    return (A + sp.diags(corr)).tocsr()


def hierarchy(dims, coef, assemble=True):
    """The levels as dicts: dims, c0, cm, cp, e (per axis), T (1-D operators), A, lmax (Gershgorin bound of D^-1 A), P and R
    (to the next level) or inv (the coarsest level).  Built by the Galerkin product along each axis, as the library does.
    assemble=False: A, lmax, P and R only on the coarsest level (for grids too large to assemble on the host)."""
    dims = tuple(int(n) for n in dims)
    dim = len(dims)
    coef = np.asarray(coef, dtype=complex)
    Ts = [_tri(dims[d], coef[1 + 2 * d], coef[2 + 2 * d]) for d in range(dim)]
    rho = coef[0] + sum(coef[1 + 2 * d] + coef[2 + 2 * d] for d in range(dim))
    levels = []
    while True:
        n = tuple(T.shape[0] for T in Ts)
        first = not levels
        dg = [T.diagonal() for T in Ts]
        c0 = coef[0] if first else rho + sum(dg[d][0] for d in range(dim))
        cm = [coef[1 + 2 * d] if first else (Ts[d][1, 0] if n[d] > 1 else 0.0) for d in range(dim)]
        cp = [coef[2 + 2 * d] if first else (Ts[d][0, 1] if n[d] > 1 else 0.0) for d in range(dim)]
        e = [dg[d][-1] - dg[d][0] for d in range(dim)]
        lv = dict(dims=n, c0=c0, cm=cm, cp=cp, e=e, T=Ts)
        levels.append(lv)
        last = int(np.prod(n)) <= CAP or min(n) < 2
        if assemble or last:
            lv["A"] = level_matrix(n, c0, cm, cp, e)
            lv["lmax"] = float(np.max(abs(lv["A"]).sum(axis=1).A.ravel() / abs(lv["A"].diagonal())))
        if last:
            break
        Ps = [interp1(m) for m in n]
        if assemble:
            lv["P"] = _tensor(Ps)
            lv["R"] = (lv["P"].T / 2 ** dim).tocsr()
        Ts = [(P1.T @ T @ P1 / 2).tocsr() for P1, T in zip(Ps, Ts)]
    if levels[-1]["A"].shape[0] > CAP:
        raise ValueError("coarsest level too large")
    levels[-1]["inv"] = np.linalg.inv(levels[-1]["A"].toarray())
    return levels


def _cheb(A, invd, b, x, m, lo, hi):
    theta, steps = coefficients(m, lo, hi)
    z = invd * b / theta if x is None else x + invd * (b - A @ x) / theta
    d = z if x is None else z - x
    for al, be in steps:
        d = al * d + be * (invd * (b - A @ z))
        z = z + d
    return z


def vcycle(levels, b, m=2, trans=False, ell=0):
    """M b (trans: M^H b), one V-cycle, in complex double."""
    lv = levels[ell]
    if "inv" in lv:
        return (lv["inv"].conj().T if trans else lv["inv"]) @ b
    A = lv["A"].conj().T.tocsr() if trans else lv["A"]
    invd = 1.0 / A.diagonal()
    hi = lv["lmax"]
    lo = hi / (2 * len(lv["dims"]))
    x = _cheb(A, invd, b, None, m, lo, hi)
    x = x + lv["P"] @ vcycle(levels, lv["R"] @ (b - A @ x), m, trans, ell + 1)
    return _cheb(A, invd, b, x, m, lo, hi)


def launches(levels, m):
    """Kernel launches of one application: per level above the coarsest, pre-smoothing (m - 1 when m >= 2 and the level has
    no centre correction, else m), restriction, prolongation and m post-smoothing steps; one coarsest solve."""
    total = 1
    for lv in levels[:-1]:
        edges = any(e != 0 for e in lv["e"])
        total += (m - 1 if m >= 2 and not edges else m) + 2 + m
    return total
