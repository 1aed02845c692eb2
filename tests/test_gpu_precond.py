"""Operator preconditioners on the device: the diagonal operator, the Jacobi preconditioner built from each operator type,
and preconditioned CG / GMRES that keep their iteration on the device, against the CPU oracle with the same
preconditioner applied on the host (tolerances: helpers.tol_for, 1e-10 fp64 / 1e-4 fp32)."""
import os
import socket
import subprocess
import sys

import numpy as np
import pytest

from helpers import CONVDIFF7, LAPLACE7, rel_normwise, tol_for
from precond_cases import varcoef_spd_csr

pytestmark = pytest.mark.gpu
KINDS = ["s", "d", "c", "z"]
TYPESTR = {"s": "<f4", "d": "<f8", "c": "<c8", "z": "<c16"}
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def lk():
    import lightkrylov_b200 as lk
    return lk


@pytest.fixture(scope="module")
def ctx(lk):
    c = lk.Context(0)
    yield c
    c.close()


class _DevArray:
    def __init__(self, ptr, n, typestr):
        self.__cuda_array_interface__ = {"shape": (n,), "typestr": typestr, "data": (ptr, False), "version": 3}


def _torch_diag_callback(ctx, kind, dh, calls=None):
    """Today's callback path: z *= d with torch on the library's stream."""
    import torch
    dd = torch.from_numpy(np.ascontiguousarray(dh)).cuda()
    ext = torch.cuda.ExternalStream(ctx.stream)

    def precond(ptr, nloc, it, cur, tgt, stream):
        if calls is not None:
            calls.append(it)
        with torch.cuda.stream(ext):
            torch.as_tensor(_DevArray(ptr, nloc, TYPESTR[kind]), device="cuda").mul_(dd)
        return 0
    return precond


def _wrap(lk, ctx, kind, n, ptr):
    import ctypes as C
    h = C.c_void_p()
    from lightkrylov_b200._lib import check
    check(ctx.lib.lkb_vec_wrap(ctx.h, lk.KINDS[kind], n, n, 0, ptr, C.byref(h)), "vec_wrap")
    return lk.Vector(ctx, kind, n, _handle=h)


def _csr_with_duplicate_diagonal(rng, m, dt, zero_row=None):
    """5 random columns per row plus the diagonal entered twice (the SpMV sums duplicates, so Jacobi must too)."""
    rows, cols, vals = [], [], []
    cplx = np.issubdtype(dt, np.complexfloating)
    for i in range(m):
        c = list(rng.integers(0, m, 5)) + [i, i]
        v = list(rng.standard_normal(7) + (1j * rng.standard_normal(7) if cplx else 0))
        v[5] += 3.0; v[6] += 1.5
        if i == zero_row:                                   # no entry on the diagonal at all
            keep = [t for t in range(7) if c[t] != i]
            c, v = [c[t] for t in keep], [v[t] for t in keep]
        o = np.argsort(c, kind="stable")
        rows += [i] * len(c); cols += [c[t] for t in o]; vals += [v[t] for t in o]
    rp = np.zeros(m + 1, dtype=np.int64); np.add.at(rp, np.array(rows) + 1, 1); rp = np.cumsum(rp)
    ci = np.array(cols, dtype=np.int32); va = np.array(vals).astype(dt)
    diag = np.zeros(m, dtype=np.complex128 if cplx else np.float64)
    hit = ci == np.array(rows)
    np.add.at(diag, np.array(rows)[hit], va[hit].astype(diag.dtype))
    return rp, ci, va, diag


# ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("kind", KINDS)
def test_diag_operator_matvec_rmatvec(lk, ctx, oracle, kind):
    dt = lk.DTYPES[kind]; n = 100003                        # odd length: packs and the scalar tail
    dh = oracle.fill(n, kind, "normal", 61); xh = oracle.fill(n, kind, "normal", 62)
    dv = lk.Vector(ctx, kind, n).put(dh)
    M = lk.LinOp.diag(dv)
    dv.put(np.zeros(n, dtype=dt))                           # the values were copied at creation
    x = lk.Vector(ctx, kind, n).put(xh); y = lk.Vector(ctx, kind, n)
    M.matvec(x, y)
    assert rel_normwise(y.get(), dh * xh) < tol_for(kind)
    M.rmatvec(x, y)
    assert rel_normwise(y.get(), np.conj(dh) * xh) < tol_for(kind)
    M.matvec(x, x)                                          # in place
    assert rel_normwise(x.get(), dh * xh) < tol_for(kind)
    x.put(xh); M.rmatvec(x, x)
    assert rel_normwise(x.get(), np.conj(dh) * xh) < tol_for(kind)
    assert M.counters() == (2, 2)
    M.reset_counter()
    assert M.counters() == (0, 0)


@pytest.mark.parametrize("kind", KINDS)
def test_jacobi_diagonal_vs_numpy(lk, ctx, oracle, kind):
    dt = lk.DTYPES[kind]; tol = tol_for(kind)
    cf = (1.0 + 0.25j) if kind in ("c", "z") else 1.0        # complex centre coefficient for the complex kinds

    def check(A, diag):
        M = lk.LinOp.jacobi(A)
        n = A.m
        xh = oracle.fill(n, kind, "normal", 71)
        x = lk.Vector(ctx, kind, n).put(xh); y = lk.Vector(ctx, kind, n)
        M.matvec(x, y)
        assert rel_normwise(y.get(), xh / np.asarray(diag, dtype=np.complex128 if kind in "cz" else np.float64)) < tol
        return M

    c5 = np.array(CONVDIFF7[:5], dtype=np.complex128) * np.array([cf, 1, 1, 1, 1])
    c7 = np.array(CONVDIFF7, dtype=np.complex128) * np.array([cf, 1, 1, 1, 1, 1, 1])
    if kind in ("s", "d"):
        c5, c7 = c5.real, c7.real
    A5 = lk.LinOp.stencil5(ctx, kind, 64, 37, c5); check(A5, np.full(64 * 37, c5[0]))
    A7 = lk.LinOp.stencil7(ctx, kind, 20, 16, 13, c7); check(A7, np.full(20 * 16 * 13, c7[0]))
    rng = np.random.default_rng(7)
    m = 20011
    rp, ci, va, diag = _csr_with_duplicate_diagonal(rng, m, dt)
    check(lk.LinOp.csr(ctx, m, m, rp, ci, va), diag)                    # plain layout
    for slice_kb in (8, 64):                                            # L2-blocked layout, forced
        ctx.set_option("csr_slice_kb", slice_kb); ctx.set_option("csr_block_min_kb", 0)
        try:
            check(lk.LinOp.csr(ctx, m, m, rp, ci, va), diag)
        finally:
            ctx.set_option("csr_slice_kb", 48 * 1024); ctx.set_option("csr_block_min_kb", 96 * 1024)
    Ad = (rng.standard_normal((128, 128)) + (1j * rng.standard_normal((128, 128)) if kind in "cz" else 0)).astype(dt)
    check(lk.LinOp.dense(ctx, np.asfortranarray(Ad)), np.diag(Ad))
    dh = (0.5 + oracle.fill(4099, kind, "uniform", 72)).astype(dt)
    Md = check(lk.LinOp.diag(lk.Vector(ctx, kind, 4099).put(dh)), dh)
    check(Md, 1.0 / dh.astype(np.complex128 if kind in "cz" else np.float64))   # Jacobi of a Jacobi: d again
    # rejected with LKB_ERR_ARG (-2)
    rp0, ci0, va0, _ = _csr_with_duplicate_diagonal(np.random.default_rng(8), 3001, dt, zero_row=1234)
    with pytest.raises(lk.LkbError, match=r"code -2: .*global row 1234 is zero or not finite"):
        lk.LinOp.jacobi(lk.LinOp.csr(ctx, 3001, 3001, rp0, ci0, va0))
    cb = lk.LinOp.callback(ctx, kind, 100, 100, lambda x, y, t, s: 0)
    with pytest.raises(lk.LkbError, match=r"code -2: .*callback"):
        lk.LinOp.jacobi(cb)
    with pytest.raises(lk.LkbError, match=r"code -2: .*not square"):
        lk.LinOp.jacobi(lk.LinOp.dense(ctx, np.asfortranarray(Ad[:, :64])))


def _cg_problems(lk, ctx, oracle, kind):
    """(name, device A, oracle A, host diagonal of A) for the variable-coefficient CSR and the C4 Laplacian."""
    dt = lk.DTYPES[kind]
    dims = (16, 14, 12); n = int(np.prod(dims))
    rp, ci, va, diag = varcoef_spd_csr(dims, 5, dt)
    yield "varcoef_csr", lk.LinOp.csr(ctx, n, n, rp, ci, va), oracle.Op.csr(n, n, rp, ci, va), diag
    dims = (20, 16, 12); n = int(np.prod(dims))
    yield "laplace7", lk.LinOp.stencil7(ctx, kind, *dims, LAPLACE7), oracle.Op.stencil(kind, dims, LAPLACE7), np.full(n, 6.0, dtype=dt)


@pytest.mark.parametrize("kind", KINDS)
def test_pcg_device_jacobi_vs_oracle(lk, ctx, oracle, kind):
    dt = lk.DTYPES[kind]; tol = tol_for(kind); maxiter = 3000
    for name, A, Ao, diag in _cg_problems(lk, ctx, oracle, kind):
        n = A.m
        dinv = (1.0 / diag.astype(np.complex128 if kind in "cz" else np.float64)).astype(dt)
        bh = oracle.fill(n, kind, "uniform", 45)
        b = lk.Vector(ctx, kind, n).put(bh)
        M = lk.LinOp.jacobi(A)
        runs = {}
        for graphs in (True, False):
            ctx.set_graphs(graphs)
            M.reset_counter()
            x = lk.Vector(ctx, kind, n)
            info, meta = lk.cg(A, b, x, maxiter=maxiter, preconditioner=M)
            runs[graphs] = (info, meta, x.get())
            assert M.counters() == (meta["n_iter"] + 1, 0), name
        ctx.set_graphs(True)
        info, meta, xg = runs[True]
        assert runs[False][0] == info and runs[False][1]["res"] == meta["res"], name        # bitwise, graphs on / off
        assert np.array_equal(runs[False][2], xg), name

        def precond_host(v):
            v *= dinv
        xo = np.zeros(n, dtype=dt)
        oinfo, ometa = oracle.cg(Ao, bh, xo, maxiter=maxiter, precond=precond_host)
        assert info == oinfo > 0, (name, info, oinfo)
        assert meta["n_iter"] == ometa["n_iter"]
        assert rel_normwise(np.array(meta["res"]), np.array(ometa["res"])) < tol, name
        assert np.linalg.norm(xg - xo) / np.linalg.norm(xo) < tol, name
        # the host-driven callback path with the same diagonal
        xc = lk.Vector(ctx, kind, n)
        cinfo, cmeta = lk.cg(A, b, xc, maxiter=maxiter, preconditioner=_torch_diag_callback(ctx, kind, dinv))
        assert cinfo == info and cmeta["n_iter"] == meta["n_iter"], name
        assert rel_normwise(np.array(cmeta["res"]), np.array(meta["res"])) < tol, name
        if name == "varcoef_csr":                                                           # Jacobi pays off here
            xu = lk.Vector(ctx, kind, n)
            uinfo, umeta = lk.cg(A, b, xu, maxiter=maxiter)
            assert umeta["n_iter"] > meta["n_iter"], (umeta["n_iter"], meta["n_iter"])


def test_pcg_general_operator_preconditioner_vs_oracle(lk, ctx, oracle):
    """M = an SPD stencil operator (applied to r, then a multi-dot), and M = a capturable callback operator that enqueues
    the same stencil: both against the oracle with M applied on the host, and bitwise equal to each other."""
    dims = (20, 16, 12); n = int(np.prod(dims))
    # first-order Neumann polynomial of A = 6 (I - N/6): M = (I + N/6) / 6, SPD (N's eigenvalues lie in (-6, 6)); 32 iterations
    # instead of 68.  (A stencil that does not approximate A^-1, e.g. (1, -0.1, ...), squares the condition number: 129
    # iterations whose tail amplifies rounding so much that two correct host restatements, differing only in the order of
    # their dot-product sums, already differ by 1.4e-9 normwise -- such a case cannot check a 1e-10 parity.)
    mc = (1.0 / 6.0,) + (1.0 / 36.0,) * 6
    A = lk.LinOp.stencil7(ctx, "d", *dims, LAPLACE7); Ao = oracle.Op.stencil("d", dims, LAPLACE7)
    S = lk.LinOp.stencil7(ctx, "d", *dims, mc); So = oracle.Op.stencil("d", dims, mc)

    def cb(xp, yp, trans, stream):
        S.matvec(_wrap(lk, ctx, "d", n, xp), _wrap(lk, ctx, "d", n, yp))
        return 0
    Mcb = lk.LinOp.callback(ctx, "d", n, n, cb, capturable=True)
    bh = oracle.fill(n, "d", "uniform", 45)
    b = lk.Vector(ctx, "d", n).put(bh)

    def precond_host(v):
        v[:] = So.apply(v)
    xo = np.zeros(n); oinfo, ometa = oracle.cg(Ao, bh, xo, maxiter=2000, precond=precond_host)
    out = []
    for M in (S, Mcb):
        M.reset_counter()
        x = lk.Vector(ctx, "d", n)
        info, meta = lk.cg(A, b, x, maxiter=2000, preconditioner=M)
        assert info == oinfo > 0
        assert rel_normwise(np.array(meta["res"]), np.array(ometa["res"])) < 1e-10
        assert np.linalg.norm(x.get() - xo) / np.linalg.norm(xo) < 1e-10
        assert M.counters()[0] == info + 1
        out.append((meta["res"], x.get()))
    assert out[0][0] == out[1][0] and np.array_equal(out[0][1], out[1][1])


@pytest.mark.parametrize("kind", ["d", "z"])
@pytest.mark.parametrize("trans", [False, True])
def test_gmres_device_precond_vs_oracle(lk, ctx, oracle, kind, trans):
    dt = lk.DTYPES[kind]; tol = tol_for(kind)
    dims = (20, 16, 12); n = int(np.prod(dims))
    A = lk.LinOp.stencil7(ctx, kind, *dims, CONVDIFF7); Ao = oracle.Op.stencil(kind, dims, CONVDIFF7)
    u = oracle.fill(n, kind, "uniform", 99)
    # complex kinds: a genuinely complex M with phases within +-0.25 rad (uniformly random phases up to 45 degrees make
    # M A indefinite enough that neither the oracle nor the device converges in 30 restarts)
    dh = (0.2 + u) if kind == "d" else (0.2 + u.real) * np.exp(0.5j * (u.imag - 0.5))
    M = lk.LinOp.diag(lk.Vector(ctx, kind, n).put(dh))
    bh = oracle.fill(n, kind, "uniform", 45)
    b = lk.Vector(ctx, kind, n).put(bh)
    runs = {}
    for graphs in (True, False):
        ctx.set_graphs(graphs)
        M.reset_counter()
        x = lk.Vector(ctx, kind, n)
        info, meta = lk.gmres(A, b, x, kdim=20, maxiter=30, transpose=trans, preconditioner=M)
        runs[graphs] = (info, meta, x.get())
        assert M.counters() == (meta["n_inner"] + meta["n_outer"], 0)
    ctx.set_graphs(True)
    info, meta, xg = runs[True]
    assert runs[False][0] == info and runs[False][1]["res"] == meta["res"] and np.array_equal(runs[False][2], xg)

    def precond_host(v):
        v *= dh
    xo = np.zeros(n, dtype=dt)
    oinfo, ometa = oracle.gmres(Ao, bh, xo, kdim=20, maxiter=30, trans=trans, precond=precond_host)
    assert info == oinfo > 0 and meta["n_outer"] == ometa["n_outer"]
    assert rel_normwise(np.array(meta["res"]), np.array(ometa["res"])) < tol
    assert np.linalg.norm(xg - xo) / np.linalg.norm(xo) < tol
    xc = lk.Vector(ctx, kind, n)
    cinfo, cmeta = lk.gmres(A, b, xc, kdim=20, maxiter=30, transpose=trans, preconditioner=_torch_diag_callback(ctx, kind, dh))
    assert cinfo == info and cmeta["n_outer"] == meta["n_outer"]
    assert rel_normwise(np.array(cmeta["res"]), np.array(meta["res"])) < tol
    with pytest.raises(TypeError):
        lk.fgmres(A, b, xc, preconditioner=M)


def _ngpus():
    import torch
    return torch.cuda.device_count() if torch.cuda.is_available() else 0


@pytest.mark.parametrize("world", [2, 4, 8])
def test_sharded_precond_vs_oracle(world):
    if _ngpus() < world:
        pytest.skip(f"needs {world} GPUs")
    s = socket.socket(); s.bind(("127.0.0.1", 0)); port = s.getsockname()[1]; s.close()
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={world}",
           "--master-addr", "127.0.0.1", "--master-port", str(port), os.path.join(ROOT, "tests", "mgpu_precond_worker.py")]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0 and f"MGPU_PRECOND_OK world={world}" in r.stdout, r.stdout[-2000:] + r.stderr[-4000:]
