"""Launch accounting: every kernel launch of the library is counted once, in lkb_kernel_launches and under one class of the
profile.  With profiling on (graphs off), the launches the profile lists over all its classes must add up to the growth of
the launch counter, for every entry point that enqueues kernels."""
import numpy as np
import pytest

from helpers import POISSON5

pytestmark = pytest.mark.gpu
DIMS = (64, 48)                                   # a small 2-D stencil
N = DIMS[0] * DIMS[1]
CONVDIFF5 = (4.0, -1.3, -0.7, -1.2, -0.8)         # nonsymmetric, for arnoldi / bidiagonalization / gmres / eigs
CLASSES = ("matvec", "multidot", "fused_axpy_dot", "multiaxpy", "other")


@pytest.fixture(scope="module")
def lk():
    import lightkrylov_b200 as lk
    lk.set_lapack_from_scipy()
    return lk


@pytest.fixture(scope="module")
def ctx(lk):
    c = lk.Context(0)
    yield c
    c.close()


def profiled(ctx, run):
    """Run `run()` with profiling on; returns (growth of the launch counter, {class: launches})."""
    ctx.set_profile(True)
    try:
        l0 = ctx.kernel_launches
        run()
        prof = ctx.get_profile()
        return ctx.kernel_launches - l0, {k: n for k, (_, n) in prof.items()}
    finally:
        ctx.set_profile(False)


def basis(lk, ctx, kind, ncols, seed, orthonormal=False, n=N):
    rng = np.random.default_rng(seed)
    a = rng.standard_normal((n, ncols))
    if kind == "z":
        a = a + 1j * rng.standard_normal((n, ncols))
    a = np.linalg.qr(a)[0] if orthonormal else a / np.linalg.norm(a, axis=0)
    return lk.Basis(ctx, kind, n, ncols).put(np.asfortranarray(a))


def vector(lk, ctx, kind, seed, n=N):
    return lk.Vector(ctx, kind, n).put(basis(lk, ctx, kind, 1, seed, n=n).get()[:, 0])


def hmat(kind, rows, cols):
    return np.zeros((rows, cols), dtype=np.complex128 if kind == "z" else np.float64, order="F")


def entry_points(lk, ctx, kind):
    A = lk.LinOp.stencil5(ctx, kind, *DIMS, CONVDIFF5)
    S = lk.LinOp.stencil5(ctx, kind, *DIMS, POISSON5)           # Hermitian positive definite, for lanczos and cg
    kdim = 12

    def arnoldi(p):
        X = basis(lk, ctx, kind, p * (kdim + 1), 1, orthonormal=True)
        return lambda: lk.arnoldi(A, X, hmat(kind, p * (kdim + 1), p * kdim), blksize=p)

    def lanczos():
        X = basis(lk, ctx, kind, kdim + 1, 2)
        lk.lanczos(S, X, hmat(kind, kdim + 1, kdim))

    def bidiag():
        U, V = basis(lk, ctx, kind, kdim + 1, 3), lk.Basis(ctx, kind, N, kdim)
        lk.bidiagonalization(A, U, V, hmat(kind, kdim + 1, kdim))

    def gram_schmidt(fn):
        X, W = basis(lk, ctx, kind, 8, 4, orthonormal=True), basis(lk, ctx, kind, 3, 5)
        return lambda: fn(W, 0, 3, X, 8)

    def qr(fn):
        Q = basis(lk, ctx, kind, 6, 6)
        Q.axpby(1.0, Q, 0.0, xcol0=0, ycol0=5, ncols=1)             # a dependent column: the refill path
        return lambda: fn(Q)

    def solve(solver, op, **kw):
        b, x = vector(lk, ctx, kind, 7), lk.Vector(ctx, kind, N)
        return lambda: solver(op, b, x, **kw)

    def eigs():             # on a smaller grid, with a loose tolerance: a few Krylov-Schur restarts
        dims = (16, 12); n = dims[0] * dims[1]
        B = lk.LinOp.stencil5(ctx, kind, *dims, CONVDIFF5)
        lk.eigs(B, lk.Basis(ctx, kind, n, 2), 2, x0=vector(lk, ctx, kind, 8, n), kdim=32, tolerance=1e-4)

    def kexpm():
        lk.kexpm(lk.Vector(ctx, kind, N), S, vector(lk, ctx, kind, 9), 0.1, 1e-10)

    M = lk.LinOp.stencil5(ctx, kind, *DIMS, (1.0, 0.1, 0.1, 0.1, 0.1))
    return {
        "arnoldi_p1": arnoldi(1),
        "arnoldi_p2": arnoldi(2),
        "lanczos": lanczos,
        "bidiagonalization": bidiag,
        "double_gram_schmidt_step": gram_schmidt(lk.double_gram_schmidt_step),
        "orthogonalize_against_basis": gram_schmidt(lk.orthogonalize_against_basis),
        "qr": qr(lk.qr),
        "qr_pivoting": qr(lk.qr_pivoting),
        "gmres": solve(lk.gmres, A, kdim=20, maxiter=5),
        "cg": solve(lk.cg, S, maxiter=60),
        "cg_jacobi": solve(lk.cg, S, maxiter=60, preconditioner=lk.LinOp.jacobi(S)),
        "cg_stencil": solve(lk.cg, S, maxiter=60, preconditioner=M),
        "eigs": eigs,
        "kexpm": kexpm,
    }


@pytest.mark.parametrize("kind", ["d", "z"])
def test_profile_adds_up_to_the_launch_counter(lk, ctx, kind):
    for name, run in entry_points(lk, ctx, kind).items():
        launches, prof = profiled(ctx, run)
        assert launches > 0, name
        assert sum(prof.values()) == launches, (name, launches, prof)


@pytest.mark.parametrize("kind", ["d", "z"])
def test_arnoldi_step_is_one_launch_per_class(lk, ctx, kind):
    """A p = 1 Arnoldi step: the matvec, the pass-1 multi-dot, the fused pass-1 update + pass-2 dot, the final pass and the
    gated scaling."""
    kdim = 12
    A = lk.LinOp.stencil5(ctx, kind, *DIMS, CONVDIFF5)
    X = basis(lk, ctx, kind, kdim + 1, 1, orthonormal=True)
    launches, prof = profiled(ctx, lambda: lk.arnoldi(A, X, hmat(kind, kdim + 1, kdim)))
    assert prof == {k: kdim for k in CLASSES} and launches == 5 * kdim, prof


@pytest.mark.parametrize("kind", ["d", "z"])
def test_orthogonalize_against_basis_counts_its_gsinfo(lk, ctx, kind):
    """One pass per column: multi-dot, the zero-vector check (k_gsinfo) and multi-axpy."""
    X, W = basis(lk, ctx, kind, 8, 4, orthonormal=True), basis(lk, ctx, kind, 3, 5)
    launches, prof = profiled(ctx, lambda: lk.orthogonalize_against_basis(W, 0, 3, X, 8, if_chk_orthonormal=False))
    assert prof == {"matvec": 0, "multidot": 3, "fused_axpy_dot": 0, "multiaxpy": 3, "other": 3} and launches == 9, prof
