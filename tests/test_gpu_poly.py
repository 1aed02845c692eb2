"""The GMRES-polynomial preconditioner on the device (include/lkb.h: lkb_op_poly_create, lkb_op_gmres_poly_create) against
the host reference of tests/poly_cases.py, and GMRES with it against the CPU oracle with that reference as the
preconditioner (tolerances: helpers.tol_for, 1e-10 fp64 / 1e-4 fp32, normwise)."""
import os
import socket
import subprocess
import sys

import numpy as np
import pytest

from chebyshev_cases import stencil_csr
from helpers import CONVDIFF7, LAPLACE7, rel_normwise, tol_for
from poly_cases import convdiff_coef, gmres_poly_roots, poly_apply

pytestmark = pytest.mark.gpu
KINDS = ["s", "d", "c", "z"]
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def lk():
    import lightkrylov_b200 as lk
    return lk


@pytest.fixture(scope="module")
def ctx(lk):
    lk.set_lapack_from_scipy()                    # the builder's host eigenvalue problem
    c = lk.Context(0)
    yield c
    c.close()


def _wrap(lk, ctx, kind, n, ptr):
    import ctypes as C
    h = C.c_void_p()
    from lightkrylov_b200._lib import check
    check(ctx.lib.lkb_vec_wrap(ctx.h, lk.KINDS[kind], n, n, 0, ptr, C.byref(h)), "vec_wrap")
    return lk.Vector(ctx, kind, n, _handle=h)


def _callback(lk, ctx, kind, S, capturable=True):
    """A callback operator that enqueues S's matvec / rmatvec on the library's stream."""
    n = S.m

    def cb(xp, yp, trans, stream):
        (S.rmatvec if trans else S.matvec)(_wrap(lk, ctx, kind, n, xp), _wrap(lk, ctx, kind, n, yp))
        return 0
    return lk.LinOp.callback(ctx, kind, n, n, cb, capturable=capturable)


def _coef(kind, coef):
    c = np.array(coef, dtype=np.complex128)
    if kind in "cz":
        c[0] *= 1.0 + 0.25j
    return c if kind in "cz" else c.real


def _roots(kind, scale, d):
    """Test roots around `scale`: d = 1, 2 (a pair in the real kinds), 5 (a pair last) and 6 (a pair given im < 0 first,
    a real root last)."""
    base = {1: [1.0], 2: [0.9 + 0.3j, 0.9 - 0.3j], 5: [1.5, 0.6, 1.2, 0.8 + 0.4j, 0.8 - 0.4j],
            6: [0.75 - 0.2j, 0.75 + 0.2j, 1.7, 1.1 + 0.35j, 1.1 - 0.35j, 1.3]}[d]
    th = np.array(base, dtype=np.complex128) * scale
    return th * np.exp(0.3j) if kind in "cz" else th


def _csr_nonsym(oracle, kind, m, per_row, seed, scale, shift):
    """shift I + scale R with R the random matrix of oracle.csr_random, as sorted CSR arrays (rowptr, col, val)."""
    import scipy.sparse as sp
    rp, ci, va = oracle.csr_random(kind, m, m, per_row, seed)
    S = (sp.csr_matrix((va * scale, ci, rp), shape=(m, m)) + shift * sp.identity(m, dtype=va.dtype)).tocsr()
    S.sum_duplicates(); S.sort_indices()
    return S.indptr.astype(np.int64), S.indices.astype(np.int32), S.data.astype(va.dtype)


def _operators(lk, ctx, oracle, kind):
    """(name, device A, host reference operator, the scale of A's spectrum)."""
    dt = lk.DTYPES[kind]
    c5 = _coef(kind, CONVDIFF7[:5]); c7 = _coef(kind, CONVDIFF7)
    epp = {"s": 4, "d": 2, "c": 2, "z": 1}[kind]
    for name, dims, cf in (("stencil2d", (16 * epp, 23), c5), ("stencil2d_ragged", (16 * epp + 1, 23), c5),
                           ("stencil3d", (20, 16, 13), c7)):
        A = (lk.LinOp.stencil5 if len(dims) == 2 else lk.LinOp.stencil7)(ctx, kind, *dims, cf)
        yield name, A, oracle.Op.stencil(kind, dims, cf), abs(cf[0])
    m = 5003
    rp, ci, va = _csr_nonsym(oracle, kind, m, 6, 11, 0.3, 8.0)
    yield "csr", lk.LinOp.csr(ctx, m, m, rp, ci, va), oracle.Op.csr(m, m, rp, ci, va), 8.0
    ctx.set_option("csr_slice_kb", 8); ctx.set_option("csr_block_min_kb", 0)
    try:
        Ab = lk.LinOp.csr(ctx, m, m, rp, ci, va)
    finally:
        ctx.set_option("csr_slice_kb", 48 * 1024); ctx.set_option("csr_block_min_kb", 96 * 1024)
    yield "csr_blocked", Ab, oracle.Op.csr(m, m, rp, ci, va), 8.0
    rng = np.random.default_rng(5)
    Ad = ((rng.standard_normal((96, 96)) + (1j * rng.standard_normal((96, 96)) if kind in "cz" else 0)) + 40 * np.eye(96)).astype(dt)
    yield "dense", lk.LinOp.dense(ctx, np.asfortranarray(Ad)), oracle.Op.dense(np.asfortranarray(Ad)), 40.0
    dh = (0.5 + oracle.fill(4099, kind, "uniform", 72)).astype(dt)
    yield "diag", lk.LinOp.diag(lk.Vector(ctx, kind, 4099).put(dh)), dh, 1.0
    S = lk.LinOp.stencil7(ctx, kind, 20, 16, 13, c7)
    yield "callback", _callback(lk, ctx, kind, S), oracle.Op.stencil(kind, (20, 16, 13), c7), abs(c7[0])


@pytest.mark.parametrize("kind", KINDS)
def test_apply_and_adjoint_vs_reference(lk, ctx, oracle, kind):
    tol = tol_for(kind)
    for name, A, Ao, scale in _operators(lk, ctx, oracle, kind):
        n = A.m
        rh = oracle.fill(n, kind, "normal", 81)
        r = lk.Vector(ctx, kind, n).put(rh); y = lk.Vector(ctx, kind, n)
        for d in (1, 2, 5, 6):
            th = _roots(kind, scale, d)
            M = lk.LinOp.polynomial(A, th)
            assert np.array_equal(M.poly_roots(), th)
            A.reset_counter()
            M.matvec(r, y)
            assert rel_normwise(y.get(), poly_apply(Ao, th, rh)) < tol, (name, d, "M")
            M.rmatvec(r, y)
            assert rel_normwise(y.get(), poly_apply(Ao, th, rh, trans=True)) < tol, (name, d, "M^H")
            assert M.counters() == (1, 1) and A.counters() == (0, 0), name
            assert np.array_equal(r.get(), rh), name                                  # r is read only


@pytest.mark.parametrize("kind", ["d", "z"])
def test_fused_stencil_path_equals_generic_path(lk, ctx, oracle, kind):
    """The same matrix as a stencil (fused steps) and as CSR (matvec + k_poly_update)."""
    dt = lk.DTYPES[kind]
    for dims, cf in (((64, 37), _coef(kind, CONVDIFF7[:5])), ((20, 16, 13), _coef(kind, CONVDIFF7))):
        As = (lk.LinOp.stencil5 if len(dims) == 2 else lk.LinOp.stencil7)(ctx, kind, *dims, cf)
        S = stencil_csr(dims, cf, dt)
        Ac = lk.LinOp.csr(ctx, S.shape[0], S.shape[0], S.indptr, S.indices, S.data)
        rh = oracle.fill(As.m, kind, "normal", 82)
        r = lk.Vector(ctx, kind, As.m).put(rh); ys = lk.Vector(ctx, kind, As.m); yc = lk.Vector(ctx, kind, As.m)
        for d in (1, 2, 5, 6):
            th = _roots(kind, abs(cf[0]), d)
            for trans in (False, True):
                Ms, Mc = lk.LinOp.polynomial(As, th), lk.LinOp.polynomial(Ac, th)
                (Ms.rmatvec if trans else Ms.matvec)(r, ys); (Mc.rmatvec if trans else Mc.matvec)(r, yc)
                assert rel_normwise(ys.get(), yc.get()) < 1e-13, (dims, d, trans)


@pytest.mark.parametrize("kind", ["d", "z"])
def test_builder_roots_vs_reference(lk, ctx, oracle, kind):
    """The builder's roots against the reference from the H that lk.arnoldi returns for the same seeded, normalised start
    vector; two builds are identical; A's matvec counter grows by the steps; the rand stream is left alone."""
    dims = (40, 36)
    cf = _coef(kind, convdiff_coef(2, 1.5))
    A = lk.LinOp.stencil5(ctx, kind, *dims, cf)
    n = A.m
    for degree in (4, 10):
        v0 = lk.Vector(ctx, kind, n).fill_random("normal", 77)
        x0 = v0.get(); x0 = x0 / np.linalg.norm(x0)
        X = lk.Basis(ctx, kind, n, degree + 1).put(x0)
        H = np.zeros((degree + 1, degree), dtype=lk.DTYPES[kind], order="F")
        assert lk.arnoldi(A, X, H) == 0
        ref = gmres_poly_roots(H, degree, kind in "cz")
        ctx.set_seed(5)
        probe = lk.Vector(ctx, kind, n)
        A.reset_counter()
        M = lk.LinOp.gmres_poly(A, degree, seed=77)
        assert A.counters() == (degree, 0)
        got = M.poly_roots()
        assert got.size == ref.size and np.abs(got - ref).max() <= 1e-10 * np.abs(ref).max(), (degree, got, ref)
        assert np.array_equal(lk.LinOp.gmres_poly(A, degree, seed=77).poly_roots(), got)
        ctx.lib.lkb_vec_rand(probe.h, 0); after = probe.get()
        ctx.set_seed(5); ctx.lib.lkb_vec_rand(probe.h, 0)
        assert np.array_equal(probe.get(), after)                 # the builds did not advance the rand stream


def test_builder_breakdown_on_diagonal_operator(lk, ctx):
    dh = np.tile([0.5, 2.0, 3.5], 1000)
    A = lk.LinOp.diag(lk.Vector(ctx, "d", dh.size).put(dh))
    M = lk.LinOp.gmres_poly(A, 8, seed=3)
    got = M.poly_roots()
    assert got.size == 3 and np.all(got.imag == 0), got
    assert np.allclose(np.sort(got.real), [0.5, 2.0, 3.5], rtol=1e-10, atol=0), got
    assert got[0].real == 3.5 or abs(got[0].real - 3.5) < 1e-10                  # largest modulus first


def _gmres_problems(lk, ctx, oracle, kind):
    """(name, device A, host A): a convection-dominated 3-D stencil (cell Peclet 1.5: complex spectrum, so conjugate pairs
    in a real kind), a shifted indefinite 2-D Laplacian, a complex shifted Laplacian, a random nonsymmetric CSR."""
    if kind == "d":
        dims, cf = (24, 20, 16), convdiff_coef(3, 1.5)
        yield "convdiff3d", lk.LinOp.stencil7(ctx, kind, *dims, cf), oracle.Op.stencil(kind, dims, cf)
        # shift 0.2 puts four of the Laplacian's eigenvalues below zero.  A harder case (24 x 20, shift 0.3: 161 inner
        # steps) amplifies the rounding differences between the device and the oracle to 1e-10 in the residual history,
        # so it cannot check a 1e-10 parity; this one converges in about 20 steps and keeps them near 1e-15.
        dims, shift = (20, 18), 0.2
        lam = np.add.outer(2.0 - 2.0 * np.cos(np.pi * np.arange(1, dims[0] + 1) / (dims[0] + 1)),
                           2.0 - 2.0 * np.cos(np.pi * np.arange(1, dims[1] + 1) / (dims[1] + 1))) - shift
        assert lam.min() < 0.0 < lam.max() and (lam < 0.0).sum() == 4
        cf = (4.0 - shift, -1.0, -1.0, -1.0, -1.0)
        yield "shifted2d", lk.LinOp.stencil5(ctx, kind, *dims, cf), oracle.Op.stencil(kind, dims, cf)
        m = 4000
        rp, ci, va = _csr_nonsym(oracle, kind, m, 7, 21, 0.5, 1.5)
        yield "csr", lk.LinOp.csr(ctx, m, m, rp, ci, va), oracle.Op.csr(m, m, rp, ci, va)
    else:
        dims, cf = (48, 40), np.array((4.0 - 0.4j, -1.0, -1.0, -1.0, -1.0))
        yield "complex_shifted2d", lk.LinOp.stencil5(ctx, kind, *dims, cf), oracle.Op.stencil(kind, dims, cf)


@pytest.mark.parametrize("kind", ["d", "z"])
def test_gmres_poly_vs_oracle(lk, ctx, oracle, kind):
    dt = lk.DTYPES[kind]; tol = tol_for(kind)
    kdim, maxiter = 20, 40
    for name, A, Ao in _gmres_problems(lk, ctx, oracle, kind):
        n = A.m
        bh = oracle.fill(n, kind, "uniform", 45)
        bv = lk.Vector(ctx, kind, n).put(bh)
        xu = lk.Vector(ctx, kind, n)
        _, umeta = lk.gmres(A, bv, xu, kdim=kdim, maxiter=maxiter)
        M = lk.LinOp.gmres_poly(A, 10, seed=1)
        th = M.poly_roots()
        runs = {}
        for graphs in (True, False, True):
            ctx.set_graphs(graphs)
            M.reset_counter(); A.reset_counter()
            x = lk.Vector(ctx, kind, n)
            info, meta = lk.gmres(A, bv, x, kdim=kdim, maxiter=maxiter, preconditioner=M)
            assert M.counters() == (meta["n_inner"] + meta["n_outer"], 0), name
            if graphs in runs:                                                        # run to run
                assert runs[graphs][0] == info and runs[graphs][1]["res"] == meta["res"], name
                assert np.array_equal(runs[graphs][2], x.get()), name
            runs[graphs] = (info, meta, x.get())
        ctx.set_graphs(True)
        info, meta, xg = runs[True]
        assert runs[False][0] == info and runs[False][1]["res"] == meta["res"], name        # bitwise, graphs on / off
        assert np.array_equal(runs[False][2], xg), name
        xo = np.zeros(n, dtype=dt)

        def precond_host(v):
            v[:] = poly_apply(Ao, th, v.copy())
        oinfo, ometa = oracle.gmres(Ao, bh, xo, kdim=kdim, maxiter=maxiter, precond=precond_host)
        assert info == oinfo and meta["n_inner"] == ometa["n_inner"] and meta["n_outer"] == ometa["n_outer"], \
            (name, info, oinfo, meta["n_inner"], ometa["n_inner"])
        assert rel_normwise(np.array(meta["res"]), np.array(ometa["res"])) < tol, name
        assert np.linalg.norm(xg - xo) / np.linalg.norm(xo) < tol, name
        assert meta["n_inner"] < umeta["n_inner"], (name, meta["n_inner"], umeta["n_inner"])


def test_launches_and_counters(lk, ctx):
    """max(d - 1, 1) fused launches per application on a stencil; (d - 1) (A's launches + 1) on a plain CSR, 1 for
    d = 1.  M's counter counts applications of M, A's counters stay."""
    A = lk.LinOp.stencil7(ctx, "d", 20, 16, 12, CONVDIFF7)
    S = stencil_csr((20, 16, 12), CONVDIFF7)
    Ac = lk.LinOp.csr(ctx, S.shape[0], S.shape[0], S.indptr, S.indices, S.data)
    r = lk.Vector(ctx, "d", A.m).fill_random("uniform", 3); y = lk.Vector(ctx, "d", A.m)
    for Aop, per in ((A, lambda d: max(d - 1, 1)), (Ac, lambda d: 2 * (d - 1) if d > 1 else 1)):
        for d in (1, 2, 5, 6):
            M = lk.LinOp.polynomial(Aop, _roots("d", 6.0, d))
            Aop.reset_counter()
            l0 = ctx.kernel_launches
            M.matvec(r, y)
            assert ctx.kernel_launches - l0 == per(d), (d,)
            M.rmatvec(r, y); M.matvec(r, y)
            assert M.counters() == (2, 1) and Aop.counters() == (0, 0)


def test_callback_operator(lk, ctx, oracle):
    """A capturable callback A reaches the stencil's GMRES result; a non-capturable one still solves (without a graph)."""
    dims, cf = (24, 20, 16), convdiff_coef(3, 1.5)
    A = lk.LinOp.stencil7(ctx, "d", *dims, cf)
    n = A.m
    bh = oracle.fill(n, "d", "uniform", 46)
    b = lk.Vector(ctx, "d", n).put(bh)
    th = lk.LinOp.gmres_poly(A, 8, seed=2).poly_roots()
    x = lk.Vector(ctx, "d", n)
    info, meta = lk.gmres(A, b, x, kdim=20, maxiter=40, preconditioner=lk.LinOp.polynomial(A, th))
    assert info > 0
    for capturable in (True, False):
        Acb = _callback(lk, ctx, "d", A, capturable=capturable)
        Mcb = lk.LinOp.polynomial(Acb, th)
        assert np.array_equal(lk.LinOp.gmres_poly(Acb, 8, seed=2).poly_roots(), th)   # the same Arnoldi run
        xc = lk.Vector(ctx, "d", n)
        cinfo, cmeta = lk.gmres(Acb, b, xc, kdim=20, maxiter=40, preconditioner=Mcb)
        assert cinfo == info and cmeta["n_inner"] == meta["n_inner"], capturable
        assert rel_normwise(np.array(cmeta["res"]), np.array(meta["res"])) < 1e-10, capturable
        assert Mcb.counters()[0] == cmeta["n_inner"] + cmeta["n_outer"]


def test_error_paths(lk, ctx):
    A = lk.LinOp.stencil7(ctx, "d", 8, 8, 8, LAPLACE7)
    with pytest.raises(lk.LkbError, match=r"code -2: .*0 roots"):
        lk.LinOp.polynomial(A, [])
    with pytest.raises(lk.LkbError, match=r"code -2: .*257 roots"):
        lk.LinOp.polynomial(A, np.ones(257))
    with pytest.raises(lk.LkbError, match=r"code -2: .*root 1 .* zero or not finite"):
        lk.LinOp.polynomial(A, [1.0, 0.0])
    with pytest.raises(lk.LkbError, match=r"code -2: .*root 2 .* zero or not finite"):
        lk.LinOp.polynomial(A, [1.0, 2.0, np.inf])
    with pytest.raises(lk.LkbError, match=r"code -2: .*complex root 1 .*not immediately followed by its conjugate"):
        lk.LinOp.polynomial(A, [1.0, 1 + 1j, 2.0, 1 - 1j])
    with pytest.raises(lk.LkbError, match=r"code -2: .*complex root 0 .*not immediately followed by its conjugate"):
        lk.LinOp.polynomial(A, [1 + 1j, 1 - 1.0000001j])
    rng = np.random.default_rng(1)
    Ar = lk.LinOp.dense(ctx, np.asfortranarray(rng.standard_normal((64, 32))))
    with pytest.raises(lk.LkbError, match=r"code -2: .*not square"):
        lk.LinOp.polynomial(Ar, [1.0])
    with pytest.raises(lk.LkbError, match=r"code -2: .*not square"):
        lk.LinOp.gmres_poly(Ar, 4)
    with pytest.raises(lk.LkbError, match=r"code -2: .*degree 0"):
        lk.LinOp.gmres_poly(A, 0)
    with pytest.raises(lk.LkbError, match=r"code -2: .*degree 129"):
        lk.LinOp.gmres_poly(A, 129)
    with pytest.raises(lk.LkbError, match=r"code -2: .*not a polynomial operator"):
        A.poly_roots()
    Az = lk.LinOp.stencil7(ctx, "z", 8, 8, 8, LAPLACE7)
    lk.LinOp.polynomial(Az, [1 + 1j, 2.0 - 0.5j])                                   # any complex roots in a complex kind
    M = lk.LinOp.polynomial(A, [6.0, 3.0])
    M2 = lk.LinOp.gmres_poly(A, 3)
    assert ctx.lib.lkb_op_destroy(A.h) == -2
    assert "Chebyshev" in ctx.lib.lkb_last_error().decode()
    x = lk.Vector(ctx, "d", A.m).fill_random("uniform", 4); y = lk.Vector(ctx, "d", A.m)
    M.matvec(x, y)                                                           # A is still there
    assert ctx.lib.lkb_op_destroy(M.h) == 0
    M.h = None
    assert ctx.lib.lkb_op_destroy(A.h) == -2                                 # M2 still holds it
    assert ctx.lib.lkb_op_destroy(M2.h) == 0
    M2.h = None
    assert ctx.lib.lkb_op_destroy(A.h) == 0
    A.h = None


def _ngpus():
    import torch
    return torch.cuda.device_count() if torch.cuda.is_available() else 0


@pytest.mark.parametrize("world", [2, 4])
def test_sharded_poly(world):
    if _ngpus() < world:
        pytest.skip(f"needs {world} GPUs")
    s = socket.socket(); s.bind(("127.0.0.1", 0)); port = s.getsockname()[1]; s.close()
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={world}",
           "--master-addr", "127.0.0.1", "--master-port", str(port), os.path.join(ROOT, "tests", "mgpu_poly_worker.py")]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=900)
    assert r.returncode == 0 and f"MGPU_POLY_OK world={world}" in r.stdout, r.stdout[-2000:] + r.stderr[-4000:]
