"""The multigrid preconditioner on the device (include/lkb.h: lkb_op_multigrid_create) against the host reference V-cycle
of tests/mg_cases.py, and multigrid-preconditioned CG / GMRES against the CPU oracle with that reference as the
preconditioner (tolerances: helpers.tol_for, 1e-10 fp64 / 1e-4 fp32, normwise)."""
import numpy as np
import pytest

from helpers import CONVDIFF7, LAPLACE7, POISSON5, rel_normwise, tol_for
from mg_cases import hierarchy, launches, vcycle

pytestmark = pytest.mark.gpu
KINDS = ["s", "d", "c", "z"]


@pytest.fixture(scope="module")
def lk():
    import lightkrylov_b200 as lk
    return lk


@pytest.fixture(scope="module")
def ctx(lk):
    c = lk.Context(0)
    yield c
    c.close()


def _coef(kind, name, dim):
    """POISSON / LAPLACE, CONVDIFF7, or CONVDIFF7 with a complex centre (complex kinds only)."""
    base = {"poisson": POISSON5 if dim == 2 else LAPLACE7, "convdiff": CONVDIFF7[:2 * dim + 1],
            "ccentre": CONVDIFF7[:2 * dim + 1]}[name]
    c = np.array(base, dtype=np.complex128)
    if name == "ccentre":
        c[0] *= 1.0 + 0.25j
    return c if kind in "cz" else c.real


def _stencil(lk, ctx, kind, dims, cf):
    return (lk.LinOp.stencil5 if len(dims) == 2 else lk.LinOp.stencil7)(ctx, kind, *dims, cf)


def _cases(kind):
    epp = {"s": 4, "d": 2, "c": 2, "z": 1}[kind]
    grids = [(64 * epp, 48), (64 * epp + 1, 47), (63, 64), (40, 33, 34), (33, 32, 31)]     # even, ragged, odd; 2-D, 3-D
    names = ["poisson", "convdiff"] + (["ccentre"] if kind in "cz" else [])
    for dims in grids:
        for name in names:
            yield dims, name


@pytest.mark.parametrize("kind", KINDS)
def test_apply_and_adjoint_vs_reference(lk, ctx, oracle, kind):
    tol = tol_for(kind)
    dt = lk.DTYPES[kind]
    for dims, name in _cases(kind):
        cf = _coef(kind, name, len(dims))
        A = _stencil(lk, ctx, kind, dims, cf)
        lev = hierarchy(dims, cf)
        assert len(lev) >= 2, dims
        rh = oracle.fill(A.m, kind, "normal", 91)
        r = lk.Vector(ctx, kind, A.m).put(rh); y = lk.Vector(ctx, kind, A.m)
        for m in (1, 2, 3):
            M = lk.LinOp.multigrid(A, m)
            A.reset_counter()
            for trans in (False, True):
                (M.rmatvec if trans else M.matvec)(r, y)
                ref = vcycle(lev, rh.astype(np.complex128), m, trans)
                ref = ref if kind in "cz" else ref.real
                assert rel_normwise(y.get(), ref.astype(dt)) < tol, (dims, name, m, trans)
            assert M.counters() == (1, 1) and A.counters() == (0, 0)
            assert np.array_equal(r.get(), rh)                                          # r is read only


@pytest.mark.parametrize("kind", ["d", "z"])
def test_adjoint_identity(lk, ctx, oracle, kind):
    """<x, M y> = <M^H x, y> on the device, for a non-Hermitian operator."""
    for dims in ((130, 97), (24, 21, 26)):
        cf = _coef(kind, "ccentre" if kind == "z" else "convdiff", len(dims))
        A = _stencil(lk, ctx, kind, dims, cf)
        M = lk.LinOp.multigrid(A)
        xh, yh = oracle.fill(A.m, kind, "normal", 92), oracle.fill(A.m, kind, "normal", 93)
        x = lk.Vector(ctx, kind, A.m).put(xh); y = lk.Vector(ctx, kind, A.m).put(yh)
        My = lk.Vector(ctx, kind, A.m); MHx = lk.Vector(ctx, kind, A.m)
        M.matvec(y, My); M.rmatvec(x, MHx)
        lhs, rhs = np.vdot(xh, My.get()), np.vdot(MHx.get(), yh)
        assert abs(lhs - rhs) <= 1e-12 * np.linalg.norm(xh) * np.linalg.norm(My.get()), (dims, lhs, rhs)


@pytest.mark.parametrize("kind", ["s", "d", "z"])
def test_pcg_multigrid_vs_oracle(lk, ctx, oracle, kind):
    dt = lk.DTYPES[kind]; tol = tol_for(kind)
    for dims, cf in (((96, 80), POISSON5), ((32, 31, 30), LAPLACE7)):
        n = int(np.prod(dims))
        A = _stencil(lk, ctx, kind, dims, cf)
        Ao = oracle.Op.stencil(kind, dims, cf)
        lev = hierarchy(dims, cf)
        bh = oracle.fill(n, kind, "uniform", 45)
        bv = lk.Vector(ctx, kind, n).put(bh)
        M = lk.LinOp.multigrid(A, 2)
        runs = {}
        for graphs in (True, False, True):
            ctx.set_graphs(graphs)
            M.reset_counter(); A.reset_counter()
            x = lk.Vector(ctx, kind, n)
            info, meta = lk.cg(A, bv, x, maxiter=200, preconditioner=M)
            assert M.counters() == (meta["n_iter"] + 1, 0) and A.counters()[0] == meta["n_iter"]
            if graphs in runs:
                assert runs[graphs][0] == info and np.array_equal(runs[graphs][2], x.get())
            runs[graphs] = (info, meta, x.get())
        ctx.set_graphs(True)
        info, meta, xg = runs[True]
        assert runs[False][0] == info and runs[False][1]["res"] == meta["res"]            # bitwise, graphs on / off
        assert np.array_equal(runs[False][2], xg)
        xo = np.zeros(n, dtype=dt)

        def precond_host(v):
            z = vcycle(lev, v.astype(np.complex128), 2)
            v[:] = (z if kind in "cz" else z.real).astype(dt)
        oinfo, ometa = oracle.cg(Ao, bh, xo, maxiter=200, precond=precond_host)
        assert info == oinfo > 0 and meta["n_iter"] == ometa["n_iter"], (dims, info, oinfo)
        assert meta["n_iter"] <= 12, meta["n_iter"]
        assert rel_normwise(np.array(meta["res"]), np.array(ometa["res"])) < tol
        assert np.linalg.norm(xg - xo) / np.linalg.norm(xo) < tol


@pytest.mark.parametrize("kind", ["d", "z"])
def test_gmres_multigrid_vs_oracle(lk, ctx, oracle, kind):
    dt = lk.DTYPES[kind]; tol = tol_for(kind)
    dims = (34, 32, 30); n = int(np.prod(dims))
    A = lk.LinOp.stencil7(ctx, kind, *dims, CONVDIFF7); Ao = oracle.Op.stencil(kind, dims, CONVDIFF7)
    lev = hierarchy(dims, CONVDIFF7)
    M = lk.LinOp.multigrid(A, 2)
    bh = oracle.fill(n, kind, "uniform", 45)
    bv = lk.Vector(ctx, kind, n).put(bh)
    x = lk.Vector(ctx, kind, n)
    info, meta = lk.gmres(A, bv, x, kdim=20, maxiter=10, preconditioner=M)
    assert M.counters() == (meta["n_inner"] + meta["n_outer"], 0)
    xo = np.zeros(n, dtype=dt)

    def precond_host(v):
        z = vcycle(lev, v.astype(np.complex128), 2)
        v[:] = (z if kind == "z" else z.real).astype(dt)
    oinfo, ometa = oracle.gmres(Ao, bh, xo, kdim=20, maxiter=10, precond=precond_host)
    assert info == oinfo > 0 and meta["n_outer"] == ometa["n_outer"] and meta["n_inner"] == ometa["n_inner"]
    assert rel_normwise(np.array(meta["res"]), np.array(ometa["res"])) < tol
    assert np.linalg.norm(x.get() - xo) / np.linalg.norm(xo) < tol


def test_full_size_fp64(lk, ctx):
    """PCG on 4096^2 (C2) and 384^3 (C4) in <= 12 iterations at the default tolerance; gmres(kdim=50, maxiter=10) on C2."""
    for dims, cf in (((4096, 4096), POISSON5), ((384, 384, 384), LAPLACE7)):
        A = _stencil(lk, ctx, "d", dims, cf)
        M = lk.LinOp.multigrid(A, 2)
        b = lk.Vector(ctx, "d", A.m).fill_random("uniform", 7)
        x = lk.Vector(ctx, "d", A.m)
        info, meta = lk.cg(A, b, x, preconditioner=M)
        assert meta["converged"] and meta["n_iter"] <= 12, (dims, info, meta["n_iter"])
        if len(dims) == 2:
            x = lk.Vector(ctx, "d", A.m)
            info, meta = lk.gmres(A, b, x, kdim=50, maxiter=10, preconditioner=M)
            assert meta["converged"] and info > 0, (info, meta["n_inner"])
        del M, A


def test_launches_per_application(lk, ctx):
    for dims, cf in (((256, 200), POISSON5), ((255, 63), POISSON5), ((40, 33, 34), LAPLACE7)):
        A = _stencil(lk, ctx, "d", dims, cf)
        lev = hierarchy(dims, cf)
        r = lk.Vector(ctx, "d", A.m).fill_random("uniform", 3); y = lk.Vector(ctx, "d", A.m)
        for m in (1, 2, 3):
            M = lk.LinOp.multigrid(A, m)
            l0 = ctx.kernel_launches
            M.matvec(r, y)
            assert ctx.kernel_launches - l0 == launches(lev, m), (dims, m)
            l0 = ctx.kernel_launches
            M.rmatvec(r, y)
            assert ctx.kernel_launches - l0 == launches(lev, m), (dims, m)


def test_coarsest_only(lk, ctx, oracle):
    """A grid of <= 512 unknowns is its own coarsest level: M = A^-1."""
    A = lk.LinOp.stencil5(ctx, "d", 20, 25, CONVDIFF7[:5])
    M = lk.LinOp.multigrid(A)
    rh = oracle.fill(A.m, "d", "normal", 94)
    r = lk.Vector(ctx, "d", A.m).put(rh); y = lk.Vector(ctx, "d", A.m); Ay = lk.Vector(ctx, "d", A.m)
    M.matvec(r, y); A.matvec(y, Ay)
    assert rel_normwise(Ay.get(), rh) < 1e-12


def test_error_paths(lk, ctx):
    A = lk.LinOp.stencil7(ctx, "d", 16, 16, 16, LAPLACE7)
    with pytest.raises(lk.LkbError, match=r"code -2: .*degree 0 < 1"):
        lk.LinOp.multigrid(A, 0)
    with pytest.raises(lk.LkbError, match=r"code -2: .*not a 5- or 7-point stencil.*Chebyshev or GMRES-polynomial"):
        lk.LinOp.multigrid(lk.LinOp.dense(ctx, np.asfortranarray(np.eye(64))))
    with pytest.raises(lk.LkbError, match=r"code -2: .*centre coefficient of level 0"):
        lk.LinOp.multigrid(lk.LinOp.stencil5(ctx, "d", 64, 64, (0.0, -1.0, -1.0, -1.0, -1.0)))
    # rho = c0 + sum (c- + c+) = -1 and each axis adds 1/2 to the coarse centre: the centre of level 1 is zero
    with pytest.raises(lk.LkbError, match=r"code -2: .*centre coefficient of level 1"):
        lk.LinOp.multigrid(lk.LinOp.stencil5(ctx, "d", 64, 63, (3.0, -1.0, -1.0, -1.0, -1.0)))
    with pytest.raises(lk.LkbError, match=r"code -2: .*coarsest grid 1 x 2048 x 1 .* > 512 unknowns"):
        lk.LinOp.multigrid(lk.LinOp.stencil5(ctx, "d", 2, 4096, POISSON5))
    with pytest.raises(lk.LkbError, match=r"code -2: .*coarsest operator .* is singular"):
        lk.LinOp.multigrid(lk.LinOp.stencil5(ctx, "d", 2, 16, (1.0, 1.0, 1.0, 0.0, 0.0)))     # blocks [[1, 1], [1, 1]]
    M = lk.LinOp.multigrid(A, 2)
    assert ctx.lib.lkb_op_destroy(A.h) == -2
    assert "multigrid" in ctx.lib.lkb_last_error().decode()
    x = lk.Vector(ctx, "d", A.m).fill_random("uniform", 4); y = lk.Vector(ctx, "d", A.m)
    M.matvec(x, y)                                                               # A is still there
    assert ctx.lib.lkb_op_destroy(M.h) == 0
    M.h = None
    assert ctx.lib.lkb_op_destroy(A.h) == 0
    A.h = None
