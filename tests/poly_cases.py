"""Host reference of the GMRES-polynomial preconditioner (include/lkb.h: lkb_op_poly_create, lkb_op_gmres_poly_create):
the product recurrence, the closed form, and the root construction (harmonic Ritz values, extra copies, modified Leja
order).  Used by tests/test_poly_host.py, tests/test_gpu_poly.py, tests/mgpu_poly_worker.py and profiles/gmres_poly_ab.py."""
import math

import numpy as np


def factors(roots, cplx):
    """The roots as factors: ("root", theta) or, in a real kind, ("pair", theta) for theta followed by its conjugate."""
    roots = np.asarray(roots, dtype=np.complex128)
    out, i = [], 0
    while i < roots.size:
        if not cplx and roots[i].imag != 0.0:
            assert i + 1 < roots.size and roots[i + 1] == np.conj(roots[i]), (i, roots)
            out.append(("pair", roots[i])); i += 2
        else:
            out.append(("root", roots[i])); i += 1
    return out


def poly_apply(op, roots, r, trans=False):
    """M r (trans: M^H r) by the product recurrence of lkb_op_poly_create, in the precision of r.  op: an oracle.Op
    (Op.apply), a callable x -> A x (trans: A^H x), or the 1-D array d of a diagonal operator."""
    if isinstance(op, np.ndarray):
        apply = (lambda x: np.conj(op) * x) if trans else (lambda x: op * x)
    elif hasattr(op, "apply"):
        apply = lambda x: op.apply(x, trans)                                      # noqa: E731
    else:
        apply = op
    cplx = np.iscomplexobj(r)
    dt, rt = r.dtype.type, r.real.dtype.type
    th = np.conj(np.asarray(roots, dtype=np.complex128)) if trans else np.asarray(roots, dtype=np.complex128)
    fs = factors(th, cplx)
    y, z = r.copy(), np.zeros_like(r)
    for i, (kind, t) in enumerate(fs):
        last = i + 1 == len(fs)
        if kind == "root":
            it = dt(1.0 / t) if cplx else rt((1.0 / t).real)
            z = z + y * it
            if not last:
                y = y - apply(y * it)
        else:
            q = abs(t) ** 2
            c0, c1 = rt(2.0 * t.real / q), rt(1.0 / q)
            w = y * c0 - apply(y) * c1
            z = z + w
            if not last:
                y = y - apply(w)
    return z


def poly_closed_form(A, roots):
    """p(A) = A^-1 (I - prod_i (I - A / theta_i)) for a small dense A, in double (complex)."""
    A = np.asarray(A, dtype=np.complex128)
    n = A.shape[0]
    P = np.eye(n, dtype=np.complex128)
    for t in np.asarray(roots, dtype=np.complex128):
        P = P @ (np.eye(n) - A / t)
    return np.linalg.solve(A, np.eye(n) - P)


def harmonic_ritz(H, k, cplx):
    """Eigenvalues of H_k + |h_{k+1,k}|^2 f e_k^T, f = H_k^-H e_k, in double; for a real H in LAPACK's order (a complex
    pair adjacent, im > 0 first)."""
    import scipy.linalg as sla
    H = np.asarray(H, dtype=np.complex128 if cplx else np.float64)
    Hk = H[:k, :k]
    e = np.zeros(k, dtype=H.dtype); e[-1] = 1.0
    f = np.linalg.solve(Hk.conj().T, e)
    G = Hk.copy()
    G[:, -1] += abs(H[k, k - 1]) ** 2 * f
    return sla.eigvals(G)


def extra_copies(th, cplx):
    """ceil((log10 pof_i - 4) / 14) for log10 pof_i = sum_{j != i} log10|1 - theta_i / theta_j| > 4, else 0; in a real kind
    a pair's conjugate takes the count of its im > 0 member."""
    th = [complex(t) for t in th]
    k, out, i = len(th), [0] * len(th), 0
    while i < k:
        lp = sum(math.log10(abs(1.0 - th[i] / th[j])) for j in range(k) if j != i)
        out[i] = math.ceil((lp - 4.0) / 14.0) if lp > 4.0 else 0
        if not cplx and th[i].imag > 0.0:
            out[i + 1] = out[i]; i += 1
        i += 1
    return out


def extend(th, cplx):
    """The roots followed by their extra copies (a real kind's pairs copied as pairs), as lkb_poly.cu builds the list."""
    th = [complex(t) for t in th]
    ext, ex, i = list(th), extra_copies(th, cplx), 0
    while i < len(th):
        pair = not cplx and th[i].imag > 0.0
        for _ in range(ex[i]):
            ext.append(th[i])
            if pair:
                ext.append(th[i + 1])
        i += 2 if pair else 1
    return ext


def leja(ext, cplx):
    """Modified Leja order: the largest modulus first, then the root maximising sum_j log|theta - theta_j| over those
    placed (in placement order, math.log as the library's libm log); ties to the lowest index.  Real kinds: a pair is placed
    im > 0 first, its conjugate right after."""
    n = len(ext)
    placed, order = [False] * n, []
    cand = lambda j: not placed[j] and (cplx or ext[j].imag >= 0.0)          # noqa: E731

    def place(j):
        order.append(ext[j]); placed[j] = True
        if not cplx and ext[j].imag > 0.0:
            order.append(ext[j + 1]); placed[j + 1] = True
    best = None
    for j in range(n):
        if cand(j) and (best is None or abs(ext[j]) > abs(ext[best])):
            best = j
    place(best)
    while len(order) < n:
        best, bs = None, 0.0
        for j in range(n):
            if not cand(j):
                continue
            s = 0.0
            for p in order:
                d = abs(ext[j] - p)
                s += math.log(d) if d > 0.0 else -math.inf
            if best is None or s > bs:
                best, bs = j, s
        place(best)
    return np.array(order, dtype=np.complex128)


def gmres_poly_roots(H, k, cplx):
    """The roots lkb_op_gmres_poly_create applies, from the (k+1) x k Arnoldi Hessenberg matrix H."""
    return leja(extend(harmonic_ritz(H, k, cplx), cplx), cplx)


def hessenberg_case(eigs, seed, cplx=False, hk1=0.3):
    """A (k+1) x k upper Hessenberg matrix whose H_k is similar to diag(eigs) (real kinds: eigs closed under conjugation)."""
    import scipy.linalg as sla
    rng = np.random.default_rng(seed)
    eigs = np.asarray(eigs, dtype=np.complex128)
    k = eigs.size
    X = rng.standard_normal((k, k)) + (1j * rng.standard_normal((k, k)) if cplx else 0)
    if cplx:
        D = np.diag(eigs)
    else:                          # real block diagonal with 2 x 2 blocks [[a, b], [-b, a]] for the pairs
        D = np.zeros((k, k)); i = 0
        while i < k:
            if eigs[i].imag != 0.0:
                a, b = eigs[i].real, eigs[i].imag
                D[i:i + 2, i:i + 2] = [[a, b], [-b, a]]; i += 2
            else:
                D[i, i] = eigs[i].real; i += 1
    Hk = sla.hessenberg(X @ D @ np.linalg.inv(X))
    H = np.zeros((k + 1, k), dtype=np.complex128 if cplx else np.float64)
    H[:k] = Hk
    H[k, k - 1] = hk1
    return H


def convdiff_coef(dim, peclet):
    """Centred convection-diffusion stencil with unit diffusion and cell Peclet number Pe = c h / 2 along every axis:
    (centre, -x, +x, -y, +y[, -z, +z]) = (2 dim, -1 - Pe, -1 + Pe, ...).  Pe > 1: the spectrum of the real operator is
    complex."""
    lo, hi = -1.0 - peclet, -1.0 + peclet
    return (2.0 * dim,) + (lo, hi) * dim
