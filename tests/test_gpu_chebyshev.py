"""The Chebyshev preconditioner on the device (include/lkb.h: lkb_op_chebyshev_create) against the host reference of
tests/chebyshev_cases.py, and Chebyshev-preconditioned CG / GMRES against the CPU oracle with that reference as the
preconditioner (tolerances: helpers.tol_for, 1e-10 fp64 / 1e-4 fp32, normwise)."""
import os
import socket
import subprocess
import sys

import numpy as np
import pytest

from chebyshev_cases import chebyshev_apply, gershgorin, stencil_csr
from helpers import CONVDIFF7, LAPLACE7, rel_normwise, tol_for
from precond_cases import varcoef_spd_csr

pytestmark = pytest.mark.gpu
KINDS = ["s", "d", "c", "z"]
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


def _cdt(kind):
    return np.complex128 if kind in "cz" else np.float64


def _stencil_coef(kind, coef):
    """CONVDIFF-like coefficients; the complex kinds get a complex centre, so D^-1 and conj(D)^-1 differ."""
    c = np.array(coef, dtype=np.complex128)
    if kind in "cz":
        c[0] *= 1.0 + 0.25j
    return c if kind in "cz" else c.real


def _csr_case(kind, m, seed):
    """7 entries per row including a dominant diagonal, one duplicated column per row, unsorted columns."""
    rng = np.random.default_rng(seed)
    rows, cols, vals = [], [], []
    for i in range(m):
        c = list(rng.integers(0, m, 4)) + [i]
        c.append(c[0])
        v = rng.standard_normal(6) + (1j * rng.standard_normal(6) if kind in "cz" else 0)
        v[4] = 8.0 + (2.0j if kind in "cz" else 0)
        rows += [i] * 6; cols += c; vals += list(v)
    import scipy.sparse as sp
    S = sp.coo_matrix((np.array(vals), (rows, cols)), shape=(m, m)).tocsr()
    rp = np.zeros(m + 1, dtype=np.int64); np.add.at(rp, np.array(rows) + 1, 1); rp = np.cumsum(rp)
    return rp, np.array(cols, dtype=np.int32), np.array(vals).astype(np.dtype({"s": "f4", "d": "f8", "c": "c8", "z": "c16"}[kind])), S


def _operators(lk, ctx, oracle, kind):
    """(name, device A, host reference operator, D^-1 in the kind, Gershgorin bound of the assembled matrix)."""
    dt = lk.DTYPES[kind]
    inv = lambda dg: (1.0 / np.asarray(dg, dtype=_cdt(kind))).astype(dt)            # noqa: E731
    c5 = _stencil_coef(kind, CONVDIFF7[:5]); c7 = _stencil_coef(kind, CONVDIFF7)
    epp = {"s": 4, "d": 2, "c": 2, "z": 1}[kind]
    for name, dims, cf in (("stencil2d", (16 * epp, 23), c5), ("stencil2d_ragged", (16 * epp + 1, 23), c5),
                           ("stencil3d", (20, 16, 13), c7)):
        A = (lk.LinOp.stencil5 if len(dims) == 2 else lk.LinOp.stencil7)(ctx, kind, *dims, cf)
        yield name, A, oracle.Op.stencil(kind, dims, cf), inv(cf[0]), gershgorin(stencil_csr(dims, cf))
    m = 5003
    rp, ci, va, S = _csr_case(kind, m, 11)
    dg = S.diagonal()
    yield "csr", lk.LinOp.csr(ctx, m, m, rp, ci, va), oracle.Op.csr(m, m, rp, ci, va), inv(dg), gershgorin(S)
    ctx.set_option("csr_slice_kb", 8); ctx.set_option("csr_block_min_kb", 0)
    try:
        Ab = lk.LinOp.csr(ctx, m, m, rp, ci, va)
    finally:
        ctx.set_option("csr_slice_kb", 48 * 1024); ctx.set_option("csr_block_min_kb", 96 * 1024)
    yield "csr_blocked", Ab, oracle.Op.csr(m, m, rp, ci, va), inv(dg), gershgorin(S)
    rng = np.random.default_rng(5)
    Ad = (rng.standard_normal((96, 96)) + (1j * rng.standard_normal((96, 96)) if kind in "cz" else 0)) + 40 * np.eye(96)
    Ad = Ad.astype(dt)
    yield "dense", lk.LinOp.dense(ctx, np.asfortranarray(Ad)), oracle.Op.dense(np.asfortranarray(Ad)), inv(np.diag(Ad)), gershgorin(Ad)
    dh = (0.5 + oracle.fill(4099, kind, "uniform", 72)).astype(dt)
    yield "diag", lk.LinOp.diag(lk.Vector(ctx, kind, 4099).put(dh)), dh, inv(dh), 1.0


@pytest.mark.parametrize("kind", KINDS)
def test_apply_and_adjoint_vs_reference(lk, ctx, oracle, kind):
    tol = tol_for(kind)
    for name, A, Ao, invd, b in _operators(lk, ctx, oracle, kind):
        n = A.m
        rh = oracle.fill(n, kind, "normal", 81)
        r = lk.Vector(ctx, kind, n).put(rh); y = lk.Vector(ctx, kind, n)
        for m in (1, 2, 3, 8):
            M = lk.LinOp.chebyshev(A, m)
            A.reset_counter()
            M.matvec(r, y)
            ref = chebyshev_apply(Ao, invd, rh, m, b / 100.0, b)
            assert rel_normwise(y.get(), ref) < tol, (name, m, "M")
            M.rmatvec(r, y)
            ref = chebyshev_apply(Ao, invd, rh, m, b / 100.0, b, trans=True)
            assert rel_normwise(y.get(), ref) < tol, (name, m, "M^H")
            assert M.counters() == (1, 1) and A.counters() == (0, 0), name
            assert np.array_equal(r.get(), rh), name                                  # r is read only


@pytest.mark.parametrize("kind", ["d", "z"])
def test_fused_stencil_path_equals_generic_path(lk, ctx, oracle, kind):
    """The same matrix as a stencil (fused steps) and as CSR (matvec + k_cheb_update)."""
    dt = lk.DTYPES[kind]
    for dims, cf in (((64, 37), _stencil_coef(kind, CONVDIFF7[:5])), ((20, 16, 13), _stencil_coef(kind, CONVDIFF7))):
        As = (lk.LinOp.stencil5 if len(dims) == 2 else lk.LinOp.stencil7)(ctx, kind, *dims, cf)
        S = stencil_csr(dims, cf, dt)
        Ac = lk.LinOp.csr(ctx, S.shape[0], S.shape[0], S.indptr, S.indices, S.data)
        rh = oracle.fill(As.m, kind, "normal", 82)
        r = lk.Vector(ctx, kind, As.m).put(rh); ys = lk.Vector(ctx, kind, As.m); yc = lk.Vector(ctx, kind, As.m)
        for m in (1, 2, 3, 8):
            for trans in (False, True):
                Ms, Mc = lk.LinOp.chebyshev(As, m), lk.LinOp.chebyshev(Ac, m)
                (Ms.rmatvec if trans else Ms.matvec)(r, ys); (Mc.rmatvec if trans else Mc.matvec)(r, yc)
                assert rel_normwise(ys.get(), yc.get()) < 1e-13, (dims, m, trans)


def test_default_bounds(lk, ctx, oracle):
    """lmax <= 0 is the Gershgorin bound (numpy's, passed explicitly); lmin <= 0 is lmax / 100."""
    rp, ci, va, S = _csr_case("d", 3001, 12)
    b = gershgorin(S)
    for A, exact in ((lk.LinOp.stencil7(ctx, "d", 20, 16, 13, LAPLACE7), True), (lk.LinOp.csr(ctx, 3001, 3001, rp, ci, va), False)):
        bnd = 2.0 if exact else b
        rh = oracle.fill(A.m, "d", "normal", 83)
        r = lk.Vector(ctx, "d", A.m).put(rh)
        out = []
        for lmin, lmax in ((None, None), (None, bnd), (bnd / 100.0, bnd), (bnd / 100.0, None)):
            y = lk.Vector(ctx, "d", A.m)
            lk.LinOp.chebyshev(A, 4, lmin=lmin, lmax=lmax).matvec(r, y)
            out.append(y.get())
        for o in out[1:]:
            if exact:
                assert np.array_equal(o, out[0])
            else:            # the device sums |a_rc| in row order, numpy in its own: the bounds may differ in the last bit
                assert rel_normwise(o, out[0]) < 1e-14
        assert np.array_equal(out[1], out[2])


def _pcg_problems(lk, ctx, oracle, kind):
    dt = lk.DTYPES[kind]
    dims = (64, 64, 64)
    yield "laplace7_64", lk.LinOp.stencil7(ctx, kind, *dims, LAPLACE7), oracle.Op.stencil(kind, dims, LAPLACE7), dt(1.0 / 6.0), 2.0
    dims = (16, 14, 12); n = int(np.prod(dims))
    rp, ci, va, diag = varcoef_spd_csr(dims, 5, dt)
    import scipy.sparse as sp
    b = gershgorin(sp.csr_matrix((va, ci, rp), shape=(n, n)))
    yield "varcoef_csr", lk.LinOp.csr(ctx, n, n, rp, ci, va), oracle.Op.csr(n, n, rp, ci, va), \
        (1.0 / diag.astype(_cdt(kind))).astype(dt), b


@pytest.mark.parametrize("kind", ["s", "d", "z"])
def test_pcg_chebyshev_vs_oracle(lk, ctx, oracle, kind):
    dt = lk.DTYPES[kind]; tol = tol_for(kind); maxiter = 3000
    for name, A, Ao, invd, b in _pcg_problems(lk, ctx, oracle, kind):
        n = A.m
        bh = oracle.fill(n, kind, "uniform", 45)
        bv = lk.Vector(ctx, kind, n).put(bh)
        xu = lk.Vector(ctx, kind, n)
        _, umeta = lk.cg(A, bv, xu, maxiter=maxiter)
        for m in ((4, 8) if name == "laplace7_64" else (4,)):
            M = lk.LinOp.chebyshev(A, m)
            runs = {}
            for graphs in (True, False, True):
                ctx.set_graphs(graphs)
                M.reset_counter(); A.reset_counter()
                x = lk.Vector(ctx, kind, n)
                info, meta = lk.cg(A, bv, x, maxiter=maxiter, preconditioner=M)
                assert M.counters() == (meta["n_iter"] + 1, 0) and A.counters()[0] == meta["n_iter"], name
                if graphs in runs:                                                    # run to run
                    assert runs[graphs][0] == info and np.array_equal(runs[graphs][2], x.get()), name
                runs[graphs] = (info, meta, x.get())
            ctx.set_graphs(True)
            info, meta, xg = runs[True]
            assert runs[False][0] == info and runs[False][1]["res"] == meta["res"], name     # bitwise, graphs on / off
            assert np.array_equal(runs[False][2], xg), name
            xo = np.zeros(n, dtype=dt)

            def precond_host(v):
                v[:] = chebyshev_apply(Ao, invd, v.copy(), m, b / 100.0, b)
            oinfo, ometa = oracle.cg(Ao, bh, xo, maxiter=maxiter, precond=precond_host)
            assert info == oinfo > 0 and meta["n_iter"] == ometa["n_iter"], (name, m, info, oinfo)
            assert rel_normwise(np.array(meta["res"]), np.array(ometa["res"])) < tol, (name, m)
            assert np.linalg.norm(xg - xo) / np.linalg.norm(xo) < tol, (name, m)
            assert meta["n_iter"] < umeta["n_iter"], (name, m, meta["n_iter"], umeta["n_iter"])


@pytest.mark.parametrize("kind", ["d", "z"])
def test_gmres_chebyshev_vs_oracle(lk, ctx, oracle, kind):
    dt = lk.DTYPES[kind]; tol = tol_for(kind)
    dims = (20, 16, 12); n = int(np.prod(dims))
    A = lk.LinOp.stencil7(ctx, kind, *dims, CONVDIFF7); Ao = oracle.Op.stencil(kind, dims, CONVDIFF7)
    b = gershgorin(stencil_csr(dims, CONVDIFF7))
    M = lk.LinOp.chebyshev(A, 4)
    bh = oracle.fill(n, kind, "uniform", 45)
    bv = lk.Vector(ctx, kind, n).put(bh)
    x = lk.Vector(ctx, kind, n)
    info, meta = lk.gmres(A, bv, x, kdim=20, maxiter=30, preconditioner=M)
    assert M.counters() == (meta["n_inner"] + meta["n_outer"], 0)
    xo = np.zeros(n, dtype=dt)

    def precond_host(v):
        v[:] = chebyshev_apply(Ao, dt(1.0 / 6.0), v.copy(), 4, b / 100.0, b)
    oinfo, ometa = oracle.gmres(Ao, bh, xo, kdim=20, maxiter=30, precond=precond_host)
    assert info == oinfo > 0 and meta["n_outer"] == ometa["n_outer"] and meta["n_inner"] == ometa["n_inner"]
    assert rel_normwise(np.array(meta["res"]), np.array(ometa["res"])) < tol
    assert np.linalg.norm(x.get() - xo) / np.linalg.norm(xo) < tol


def test_launches_per_application(lk, ctx, oracle):
    """m - 1 fused launches on a stencil (1 for m = 1); 1 + (m - 1) (matvec + update) on a plain CSR; and in CG one
    application of M per iteration on top of the CG_NORED launches."""
    A = lk.LinOp.stencil7(ctx, "d", 20, 16, 12, LAPLACE7)
    S = stencil_csr((20, 16, 12), LAPLACE7)
    Ac = lk.LinOp.csr(ctx, S.shape[0], S.shape[0], S.indptr, S.indices, S.data)
    r = lk.Vector(ctx, "d", A.m).fill_random("uniform", 3); y = lk.Vector(ctx, "d", A.m)
    for Aop, per in ((A, lambda m: max(m - 1, 1)), (Ac, lambda m: 1 + 2 * (m - 1))):
        for m in (1, 2, 5):
            M = lk.LinOp.chebyshev(Aop, m)
            l0 = ctx.kernel_launches
            M.matvec(r, y)
            assert ctx.kernel_launches - l0 == per(m), (m,)
        counts = {}
        for m in (2, 5):
            M = lk.LinOp.chebyshev(Aop, m)
            x = lk.Vector(ctx, "d", A.m)
            l0 = ctx.kernel_launches
            info, meta = lk.cg(Aop, r, x, rtol=1e-300, atol=0.0, maxiter=32, preconditioner=M)   # two full chunks of 16
            assert meta["n_iter"] == 32 and info == -32
            counts[m] = ctx.kernel_launches - l0
        assert counts[5] - counts[2] == 33 * (per(5) - per(2))              # the first application + 32 iterations


def test_error_paths(lk, ctx):
    A = lk.LinOp.stencil7(ctx, "d", 8, 8, 8, LAPLACE7)
    with pytest.raises(lk.LkbError, match=r"code -2: .*degree 0 < 1"):
        lk.LinOp.chebyshev(A, 0)
    with pytest.raises(lk.LkbError, match=r"code -2: .*lmin = 2 is not below lmax = 2"):
        lk.LinOp.chebyshev(A, 3, lmin=2.0)                                    # at the Gershgorin default
    with pytest.raises(lk.LkbError, match=r"code -2: .*lmin = 3 is not below lmax = 1"):
        lk.LinOp.chebyshev(A, 3, lmin=3.0, lmax=1.0)
    with pytest.raises(lk.LkbError, match=r"code -2: .*callback"):
        lk.LinOp.chebyshev(lk.LinOp.callback(ctx, "d", 100, 100, lambda x, y, t, s: 0), 3)
    rng = np.random.default_rng(1)
    with pytest.raises(lk.LkbError, match=r"code -2: .*not square"):
        lk.LinOp.chebyshev(lk.LinOp.dense(ctx, np.asfortranarray(rng.standard_normal((64, 32)))), 3)
    rp, ci, va, S = _csr_case("d", 3001, 13)
    keep = ~((np.repeat(np.arange(3001), np.diff(rp)) == 1234) & (ci == 1234))     # row 1234 without its diagonal
    rows = np.repeat(np.arange(3001), np.diff(rp))[keep]
    rp0 = np.concatenate([[0], np.cumsum(np.bincount(rows, minlength=3001))]).astype(np.int64)
    with pytest.raises(lk.LkbError, match=r"code -2: .*global row 1234 is zero or not finite"):
        lk.LinOp.chebyshev(lk.LinOp.csr(ctx, 3001, 3001, rp0, ci[keep], va[keep]), 3)
    with pytest.raises(lk.LkbError, match=r"code -2: .*global row 0 is zero or not finite"):
        lk.LinOp.chebyshev(lk.LinOp.stencil5(ctx, "d", 16, 16, (0.0, -1.0, -1.0, -1.0, -1.0)), 3)
    M = lk.LinOp.chebyshev(A, 3)
    assert ctx.lib.lkb_op_destroy(A.h) == -2
    assert "Chebyshev" in ctx.lib.lkb_last_error().decode()
    x = lk.Vector(ctx, "d", A.m).fill_random("uniform", 4); y = lk.Vector(ctx, "d", A.m)
    M.matvec(x, y)                                                           # A is still there
    assert ctx.lib.lkb_op_destroy(M.h) == 0
    M.h = None
    assert ctx.lib.lkb_op_destroy(A.h) == 0
    A.h = None


def _ngpus():
    import torch
    return torch.cuda.device_count() if torch.cuda.is_available() else 0


@pytest.mark.parametrize("world", [2, 4])
def test_sharded_chebyshev(world):
    if _ngpus() < world:
        pytest.skip(f"needs {world} GPUs")
    s = socket.socket(); s.bind(("127.0.0.1", 0)); port = s.getsockname()[1]; s.close()
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={world}",
           "--master-addr", "127.0.0.1", "--master-port", str(port), os.path.join(ROOT, "tests", "mgpu_chebyshev_worker.py")]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=900)
    assert r.returncode == 0 and f"MGPU_CHEBYSHEV_OK world={world}" in r.stdout, r.stdout[-2000:] + r.stderr[-4000:]
