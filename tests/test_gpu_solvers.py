"""GPU parity of the solver shells built on the device Krylov step: eigs (+ Krylov-Schur),
eighs, svds -- the reference's known-answer tests (test/TestIterativeSolvers.fypp) run through
the C ABI, plus entrywise comparison with the numpy/scipy oracle shells on identical inputs."""
import numpy as np
import pytest

from helpers import CONVDIFF7, LAPLACE7, POISSON5, randn, random_csr, rel_normwise, tol_for

pytestmark = pytest.mark.gpu
N = 128


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


def _toeplitz(n, sub, diag, sup, dtype=np.float64):
    A = np.zeros((n, n), dtype=dtype); i = np.arange(n)
    A[i, i] = diag; A[i[1:], i[:-1]] = sub; A[i[:-1], i[1:]] = sup
    return np.asfortranarray(A)


def _match(a, b):
    return np.abs(a[:, None] - b[None, :]).min(axis=1).max()


def test_eigs_known_answer_full(lk, ctx, oracle):
    """TestIterativeSolvers.fypp:134-197 (nev = n = 128, kdim at its default 4*nev = 512 > n as in the reference's test: the
    literal post-convergence krylov_schur then retains all n Ritz values, see tests/test_oracle_pins.py)."""
    a, b = 1.0, 0.5
    Ah = _toeplitz(N, -b, a, b)
    x0h = np.random.default_rng(20).standard_normal(N)
    A = lk.LinOp.dense(ctx, Ah); X = lk.Basis(ctx, "d", N, N)
    x0 = lk.Vector(ctx, "d", N).put(x0h)
    ev, res, info = lk.eigs(A, X, N, x0=x0)
    true = a + 2j * b * np.cos(np.arange(1, N + 1) * np.pi / (N + 1))
    assert _match(ev, true) < lk.RTOL["d"] and _match(true, ev) < lk.RTOL["d"]
    evo, reso, Xo, infoo = oracle.eigs(oracle.Op.dense(Ah), N, N, x0h)
    assert info == infoo
    assert _match(ev, evo) < 1e-10
    # the reference's literal assertion: ELEMENTWISE against (a + iw_1, a - iw_1, a + iw_2, ...) -- pins the tie order of
    # sort_index(abs, reverse=.true.) (stable: a conjugate pair stays (+, -)) and with it the (Re, Im) column layout
    tref = np.zeros(N, dtype=np.complex128)
    for k in range(1, N // 2 + 1):
        tref[2 * k - 2] = a + 2j * b * np.cos(k * np.pi / (N + 1)); tref[2 * k - 1] = np.conj(tref[2 * k - 2])
    assert np.max(np.abs(ev - tref) / np.abs(tref)) < lk.RTOL["d"]
    assert np.max(np.abs(evo - tref) / np.abs(tref)) < lk.RTOL["d"]
    Xg = X.get()
    v = Xg[:, 0] + 1j * Xg[:, 1]
    assert ev[0].imag > 0 and np.linalg.norm(Ah @ v - ev[0] * v) < 1e-6 * np.linalg.norm(v)


@pytest.mark.parametrize("kind", ["d", "z", "s"])
def test_eigs_krylov_schur_vs_oracle(lk, ctx, oracle, kind):
    """TestIterativeSolvers.fypp:161-209: nev = 8, kdim = 32, restarts; same niter, Ritz values to 1e-10."""
    dt = lk.DTYPES[kind]; a, b, nev = 1.0, 0.5, 8
    Ah = _toeplitz(N, -b, a, b, dt)
    x0h = randn(np.random.default_rng(21), N, dt)
    A = lk.LinOp.dense(ctx, Ah); X = lk.Basis(ctx, kind, N, nev)
    ev, res, info = lk.eigs(A, X, nev, x0=lk.Vector(ctx, kind, N).put(x0h), kdim=4 * nev)
    evo, reso, Xo, infoo = oracle.eigs(oracle.Op.dense(Ah), N, nev, x0h, kdim=4 * nev)
    tol = 1e-10 if kind in "dz" else 1e-4
    if kind in "dz":
        assert info == infoo
    assert _match(ev, evo) < tol * np.abs(evo).max()
    true = a + 2j * b * np.cos(np.arange(1, N + 1) * np.pi / (N + 1))
    lead = true[np.argsort(-np.abs(true))][:nev]
    assert _match(ev, lead) < (1e-6 if kind in "dz" else 1e-3)
    # eigenvectors: A v = lambda v through the real-pair convention / directly for complex kinds
    Xg = X.get().astype(np.complex128)
    Ac = Ah.astype(np.complex128)
    i = 0
    while i < nev:
        if kind in "cz" or ev[i].imag == 0:
            v, lam = Xg[:, i], ev[i]; i += 1
        elif i + 1 < nev:
            v = Xg[:, i] + 1j * Xg[:, i + 1] if ev[i].imag > 0 else Xg[:, i + 1] + 1j * Xg[:, i]
            lam = ev[i] if ev[i].imag > 0 else ev[i + 1]; i += 2
        else:
            break
        # fp32: the solver stops at Ritz residual < rtol_sp = 1e-3, so eigenpairs are only that accurate
        assert np.linalg.norm(Ac @ v - lam * v) < (1e-6 if kind in "dz" else 1e-2) * np.linalg.norm(v)


def test_krylov_schur_restart_relation(lk, ctx, oracle):
    """TestKrylov.fypp:298-347 on the device: A X_n = X_{n+1} H(:n+1,:n), orthonormal; vs oracle."""
    rng = np.random.default_rng(22); kdim = 32
    Ah = randn(rng, (N, N), np.float64) / np.sqrt(N)
    x0 = randn(rng, N, np.float64); oracle.normalize(x0)
    A = lk.LinOp.dense(ctx, Ah)
    X = lk.Basis(ctx, "d", N, kdim + 1).put(x0); H = np.zeros((kdim + 1, kdim), order="F")
    assert lk.arnoldi(A, X, H) == 0
    nk = lk.krylov_schur(X, H, kdim)
    Xo = np.zeros((N, kdim + 1), order="F"); Xo[:, 0] = x0; Ho = np.zeros_like(H)
    oracle.arnoldi(oracle.Op.dense(Ah), Xo, Ho); nko = oracle.krylov_schur(Xo, Ho)
    assert nk == nko and 0 < nk < kdim
    Xg = X.get()
    assert np.abs(Ah @ Xg[:, :nk] - Xg[:, :nk + 1] @ H[:nk + 1, :nk]).max() < lk.RTOL["d"]
    assert np.abs(Xg[:, :nk + 1].T @ Xg[:, :nk + 1] - np.eye(nk + 1)).max() < 1e-12
    assert not Xg[:, nk + 1:].any() and not H[nk + 1:, :].any() and not H[:, nk:].any()
    # the reordered real Schur form is not unique (2x2 block standardisation, swap order), so compare the
    # invariants: the retained Ritz values and the residual row norm
    assert _match(np.linalg.eigvals(H[:nk, :nk]), np.linalg.eigvals(Ho[:nk, :nk])) < 1e-10
    assert abs(np.linalg.norm(H[nk, :nk]) - np.linalg.norm(Ho[nk, :nk])) < 1e-10
    # resume the factorisation from the restarted state (the way eigs does)
    assert lk.arnoldi(A, X, H, kstart=nk + 1, kend=kdim) == 0
    Xg = X.get()
    assert np.abs(Ah @ Xg[:, :kdim] - Xg @ H).max() < lk.RTOL["d"]


@pytest.mark.parametrize("kind", ["d", "s", "z"])
def test_eighs_known_answer_and_oracle(lk, ctx, oracle, kind):
    """TestIterativeSolvers.fypp:254-307."""
    dt = lk.DTYPES[kind]; a, b, nev = 2.0, -1.0, 8
    Ah = _toeplitz(N, b, a, b, dt)
    x0h = randn(np.random.default_rng(23), N, dt)
    A = lk.LinOp.dense(ctx, Ah); X = lk.Basis(ctx, kind, N, nev)
    ev, res, info = lk.eighs(A, X, nev, x0=lk.Vector(ctx, kind, N).put(x0h), kdim=N)
    true = a + 2 * abs(b) * np.cos(np.arange(1, N + 1) * np.pi / (N + 1))
    # fp32 stops as soon as ANY nev Ritz residuals are < rtol_sp = 1e-3 (eighs.fypp:94-99): loose known answer
    assert np.abs(ev - true[:nev]).max() < (lk.RTOL[kind] * 4 if kind in "dz" else 3e-2)
    evo, reso, Xo, infoo = oracle.eighs(oracle.Op.dense(Ah), N, nev, x0h, kdim=N)
    if kind in "dz":
        assert info == infoo
    assert np.abs(ev - evo).max() < (1e-10 if kind in "dz" else 1e-4) * np.abs(evo).max()
    Xg = X.get()
    assert np.abs(Ah @ Xg - Xg * ev.astype(dt)).max() < (1e-6 if kind in "dz" else 5e-2)
    assert np.abs(Xg.conj().T @ Xg - np.eye(nev)).max() < lk.RTOL[kind] * 4


@pytest.mark.parametrize("kind", ["d", "z"])
def test_svds_known_answer_and_oracle(lk, ctx, oracle, kind):
    """TestIterativeSolvers.fypp:440-489 (Strang matrix) + a rectangular random CSR vs oracle."""
    dt = lk.DTYPES[kind]; nsv = 8
    Ah = _toeplitz(N, -1.0, 2.0, -1.0, dt)
    u0h = randn(np.random.default_rng(24), N, dt)
    A = lk.LinOp.dense(ctx, Ah)
    U = lk.Basis(ctx, kind, N, nsv); V = lk.Basis(ctx, kind, N, nsv)
    S, res, info = lk.svds(A, U, V, nsv, u0=lk.Vector(ctx, kind, N).put(u0h), kdim=N)
    true = 2 * (1 + np.cos(np.arange(1, N + 1) * np.pi / (N + 1)))
    assert np.abs(S - true[:nsv]).max() < lk.RTOL[kind]
    Ug, Vg = U.get(), V.get()
    assert np.abs(Ah @ Vg - Ug * S.astype(dt)).max() < 1e-6
    assert np.abs(Ug.conj().T @ Ug - np.eye(nsv)).max() < lk.RTOL[kind]
    So, reso, Uo, Vo, infoo = oracle.svds(oracle.Op.dense(Ah), nsv, u0h, kdim=N)
    assert info == infoo and np.abs(S - So).max() < 1e-10 * So.max()
    # config-5 shaped: rectangular CSR, cdp/rdp
    m, n = 900, 700
    Sp = random_csr(np.random.default_rng(46), m, n, 32, dt)
    Ac = lk.LinOp.csr(ctx, m, n, Sp.indptr, Sp.indices, Sp.data.astype(dt))
    Aco = oracle.Op.csr(m, n, Sp.indptr, Sp.indices, Sp.data.astype(dt))
    u0h = oracle.fill(m, kind, "normal", 47)
    U = lk.Basis(ctx, kind, m, nsv); V = lk.Basis(ctx, kind, n, nsv)
    S, res, info = lk.svds(Ac, U, V, nsv, u0=lk.Vector(ctx, kind, m).put(u0h), kdim=32)
    So, reso, Uo, Vo, infoo = oracle.svds(Aco, nsv, u0h, kdim=32)
    assert info == infoo and np.abs(S - So).max() < 1e-10 * So.max()
    sv_true = np.linalg.svd(Sp.toarray(), compute_uv=False)
    assert abs(S[0] - sv_true[0]) < 1e-6 * sv_true[0]


def test_eigs_convdiff_stencil_vs_oracle(lk, ctx, oracle):
    """Config-3 shaped: nonsymmetric 7-point convection-diffusion, eigs nev=4 with Krylov-Schur."""
    dims = (12, 10, 8); n = int(np.prod(dims)); nev = 4
    A = lk.LinOp.stencil7(ctx, "d", *dims, CONVDIFF7); Ao = oracle.Op.stencil("d", dims, CONVDIFF7)
    x0h = oracle.fill(n, "d", "uniform", 44)
    X = lk.Basis(ctx, "d", n, nev)
    ev, res, info = lk.eigs(A, X, nev, x0=lk.Vector(ctx, "d", n).put(x0h), kdim=24, tolerance=1e-8)
    evo, reso, Xo, infoo = oracle.eigs(Ao, n, nev, x0h, kdim=24, tolerance=1e-8)
    assert info == infoo
    assert _match(ev, evo) < 1e-10 * np.abs(evo).max()


@pytest.mark.parametrize("kind", ["d", "z", "s"])
def test_kexpm_vec_vs_oracle(lk, ctx, oracle, kind):
    """kexpm_vec (src/Expm/ExpmLib.fypp:128-232, SURVEY 8 f4): c = exp(tau A) b on the device vs the oracle restatement:
    same `info` (Krylov dimension used) and the same vector."""
    dims = (24, 20); n = 480
    coef = (-4.0, 1.0, 1.0, 1.0, 1.0)
    A = lk.LinOp.stencil5(ctx, kind, *dims, coef); Ao = oracle.Op.stencil(kind, dims, coef)
    bh = oracle.fill(n, kind, "uniform", 3)
    b = lk.Vector(ctx, kind, n).put(bh); c = lk.Vector(ctx, kind, n)
    tol = 1e-10 if kind in "dz" else 1e-5
    info = lk.kexpm(c, A, b, 0.1, tol)
    co, oinfo = oracle.kexpm_vec(Ao, bh, 0.1, tol)
    assert info == oinfo and info > 1
    assert np.linalg.norm(c.get() - co) < (1e-10 if kind in "dz" else 1e-4) * np.linalg.norm(co)
    # zero input => zero output (ExpmLib.fypp:180-184); transpose of the symmetric operator gives the same vector
    z = lk.Vector(ctx, kind, n); c2 = lk.Vector(ctx, kind, n).put(bh)
    lk.kexpm(c2, A, z, 0.1, tol)
    assert not c2.get().any()
    ct = lk.Vector(ctx, kind, n)
    assert lk.kexpm(ct, A, b, 0.1, tol, trans=True) == info
    assert np.linalg.norm(ct.get() - co) < (1e-10 if kind in "dz" else 1e-4) * np.linalg.norm(co)
    # krylov_exptA (ExpmLib.fypp:364-392) = kexpm_vec with tol = atol_kind, kdim = 30
    ce = lk.Vector(ctx, kind, n); ck = lk.Vector(ctx, kind, n)
    einfo = lk.krylov_exptA(ce, A, b, 0.1)
    assert einfo == lk.kexpm(ck, A, b, 0.1, lk.ATOL[kind], kdim=30) and np.array_equal(ce.get(), ck.get())
    assert einfo == oracle.kexpm_vec(Ao, bh, 0.1, oracle.ATOL[kind], kdim=30)[1]


@pytest.mark.parametrize("kind", ["d", "z"])
def test_kexpm_vec_breakdown_literal_info(lk, ctx, oracle, kind):
    """Arnoldi breakdown inside kexpm_vec: b spans a 3-dimensional invariant subspace of a diagonal operator.  The reference
    overwrites `info` with -2 before its merge(0, ..., info == k), so the error estimate is not zeroed at the breakdown step;
    the loop continues on the refilled vector and stops two steps later with info = kp = 5 and the exact vector
    (ExpmLib.fypp:199-226; literal flow pinned on the CPU by tests/test_oracle_second_opinion.py)."""
    dt = lk.DTYPES[kind]; n = 96
    D = np.asfortranarray(np.diag(np.arange(1, n + 1)).astype(dt))
    A = lk.LinOp.dense(ctx, D); Ao = oracle.Op.dense(D)
    bh = np.zeros(n, dtype=dt); bh[:3] = [1.0, 2.0, -1.5]
    b = lk.Vector(ctx, kind, n).put(bh); c = lk.Vector(ctx, kind, n)
    info = lk.kexpm(c, A, b, 0.2, 1e-12)
    co, oinfo = oracle.kexpm_vec(Ao, bh, 0.2, 1e-12)
    assert info == oinfo == 5
    exact = np.exp(0.2 * np.arange(1, n + 1)) * bh
    assert np.linalg.norm(c.get() - exact) < 1e-12 * np.linalg.norm(exact)


# ---- pivoting QR and block Krylov exponential (SURVEY 8 f2: block Arnoldi's caller `kexpm_mat` with pivoting QR) ----------
@pytest.mark.parametrize("kind", ["d", "z", "s", "c"])
def test_qr_pivoting_vs_oracle(lk, ctx, oracle, kind):
    """qr_with_pivoting (src/Krylov/qr.fypp:32-107) on the device vs the oracle restatement: same pivot order, same R, same Q;
    plus the reference's own assertions (TestKrylov.f90:245-318) on a matrix with 5 exactly-zero columns."""
    dt = lk.DTYPES[kind]; p = 12
    Ah = randn(np.random.default_rng(33), (N, p), dt)
    Q = lk.Basis(ctx, kind, N, p).put(Ah)
    info, R, perm = lk.qr_pivoting(Q)
    Qo = Ah.copy(order="F"); infoo, Ro, permo = oracle.qr_with_pivoting(Qo)
    assert info == infoo == 0 and perm.tolist() == permo.tolist()
    perm_full = permo.copy()
    assert rel_normwise(R, Ro) < tol_for(kind) and rel_normwise(Q.get(), Qo) < tol_for(kind)
    assert np.abs(Ah[:, perm] - Q.get() @ R).max() < lk.RTOL[kind]
    # exact rank deficiency: kdim = 20, 5 zero columns
    kdim, nzero = 20, 5
    rng = np.random.default_rng(34)
    Bh = randn(rng, (N, kdim), dt); Bh[:, rng.choice(kdim, nzero, replace=False)] = 0
    Q = lk.Basis(ctx, kind, N, kdim).put(Bh)
    info, R, perm = lk.qr_pivoting(Q)
    Qo = Bh.copy(order="F"); infoo, Ro, permo = oracle.qr_with_pivoting(Qo)
    rk = kdim - nzero
    assert info == infoo == rk + 1 and perm.tolist() == permo.tolist()
    Qg = Q.get()
    assert rel_normwise(R, Ro) < tol_for(kind) and rel_normwise(Qg[:, :rk], Qo[:, :rk]) < tol_for(kind)
    assert np.abs(Bh[:, perm] - Qg @ R).max() < lk.RTOL[kind]
    assert np.linalg.norm(Qg.conj().T @ Qg - np.eye(kdim)) < lk.RTOL[kind]      # incl. the random orthonormal completion
    assert not R[rk:, :].any()
    # a column section of a larger basis (col0 > 0) leaves the other columns alone
    W = lk.Basis(ctx, kind, N, p + 3).put(np.concatenate([np.ones((N, 2), dtype=dt), Ah, np.ones((N, 1), dtype=dt)], axis=1))
    info, R2, perm2 = lk.qr_pivoting(W, col0=2, p=p)
    Wg = W.get()
    assert info == 0 and perm2.tolist() == perm_full.tolist()
    assert (Wg[:, :2] == 1).all() and (Wg[:, -1] == 1).all() and np.abs(Ah[:, perm2] - Wg[:, 2:2 + p] @ R2).max() < lk.RTOL[kind]


@pytest.mark.parametrize("kind", ["d", "z", "s"])
@pytest.mark.parametrize("p", [1, 3])
def test_kexpm_mat_vs_oracle(lk, ctx, oracle, kind, p):
    """kexpm_mat (src/Expm/ExpmLib.fypp:234-362): C = exp(tau A) B by block Arnoldi on the device vs the oracle restatement:
    same `info` (dimension used), same block; and against the dense exponential (TestExpmlib.f90:334-419)."""
    import scipy.linalg as sla
    dims = (24, 20); n = 480
    coef = (-4.0, 1.0, 0.8, 1.0, 1.2)
    A = lk.LinOp.stencil5(ctx, kind, *dims, coef); Ao = oracle.Op.stencil(kind, dims, coef)
    Bh = np.asfortranarray(np.stack([oracle.fill(n, kind, "uniform", 5 + i) for i in range(p)], axis=1))
    B = lk.Basis(ctx, kind, n, p).put(Bh); Cb = lk.Basis(ctx, kind, n, p)
    tol = 1e-10 if kind in "dz" else 1e-5
    info = lk.kexpm_mat(Cb, A, B, 0.1, tol, kdim=15)
    Co, oinfo = oracle.kexpm_mat(Ao, Bh, 0.1, tol, kdim=15)
    assert info == oinfo and info >= 2 * p
    assert np.linalg.norm(Cb.get() - Co) < tol_for(kind) * np.linalg.norm(Co)
    Ad = np.stack([Ao.apply(e) for e in np.eye(n, dtype=lk.DTYPES[kind])], axis=1).astype(np.complex128)
    ref = sla.expm(0.1 * Ad) @ Bh
    assert np.linalg.norm(Cb.get() - ref) < (1e-9 if kind in "dz" else 1e-4) * np.linalg.norm(ref)
    # transpose flag: exp(tau A^H) B
    Ct = lk.Basis(ctx, kind, n, p)
    tinfo = lk.kexpm_mat(Ct, A, B, 0.1, tol, trans=True, kdim=15)
    Cto, otinfo = oracle.kexpm_mat(Ao, Bh, 0.1, tol, trans=True, kdim=15)
    assert tinfo == otinfo
    assert np.linalg.norm(Ct.get() - Cto) < tol_for(kind) * np.linalg.norm(Cto)
    # zero input => zero output, info = p (ExpmLib.fypp:297-300)
    Z = lk.Basis(ctx, kind, n, p); C2 = lk.Basis(ctx, kind, n, p).put(Bh)
    assert lk.kexpm_mat(C2, A, Z, 0.1, tol, kdim=15) == p
    assert not C2.get().any()


def test_kexpm_mat_breakdown_exits(lk, ctx, oracle):
    """Block-Arnoldi breakdown inside kexpm_mat: the columns of B span a 4-dimensional invariant subspace of a diagonal operator
    (p = 2).  After two block steps the new block is numerically zero, arnoldi returns info = kp, the extended matrix is not
    considered, the error estimate is the norm of an EMPTY section = 0 and the loop exits with info = kp and the exact
    result (ExpmLib.fypp:314-346) -- unlike kexpm_vec, where the estimate is not zeroed."""
    n = 96
    D = np.asfortranarray(np.diag(np.arange(1, n + 1)).astype(np.float64))
    A = lk.LinOp.dense(ctx, D); Ao = oracle.Op.dense(D)
    Bh = np.zeros((n, 2), order="F"); Bh[:4, 0] = [1.0, 2.0, -1.5, 0.5]; Bh[:4, 1] = [0.3, -1.0, 2.0, 1.0]
    B = lk.Basis(ctx, "d", n, 2).put(Bh); Cb = lk.Basis(ctx, "d", n, 2)
    info = lk.kexpm_mat(Cb, A, B, 0.2, 1e-12)
    Co, oinfo = oracle.kexpm_mat(Ao, Bh, 0.2, 1e-12)
    assert info == oinfo == 4
    exact = np.exp(0.2 * np.arange(1, n + 1))[:, None] * Bh
    assert np.linalg.norm(Cb.get() - exact) < 1e-12 * np.linalg.norm(exact)
    assert np.linalg.norm(Co - exact) < 1e-12 * np.linalg.norm(exact)


def test_write_intermediate_sorts_the_residual_table(lk, ctx, oracle, tmp_path):
    """write_results sorts its residual argument IN PLACE (`call sort_index(res, indices)`, intent(inout),
    IterativeSolvers.fypp:882-924), so with write_intermediate (option "write_intermediate"; the reference's default for eigs)
    the residuals a solver returns are entries of the ASCENDING table: for eighs the nev largest ones in non-increasing
    order.  Same `info` and eigenvalues as without the option; the oracle restates the side effect; the table files appear."""
    import os
    nev = 4
    rng = np.random.default_rng(26)
    D = np.diag(np.concatenate([np.linspace(0, 1, N - 4), [2.0, 2.5, 3.0, 4.0]])); Q, _ = np.linalg.qr(rng.standard_normal((N, N)))
    Ah = Q @ D @ Q.T; Ah = np.asfortranarray((Ah + Ah.T) / 2)             # four separated leading eigenvalues: converges at k ~ 16
    x0h = randn(np.random.default_rng(25), N, np.float64)
    A = lk.LinOp.dense(ctx, Ah); x0 = lk.Vector(ctx, "d", N).put(x0h)
    X = lk.Basis(ctx, "d", N, nev)
    ev0, res0, info0 = lk.eighs(A, X, nev, x0=x0, kdim=60, tolerance=1e-6)
    Ag = lk.LinOp.dense(ctx, _toeplitz(N, -0.5, 1.0, 0.5)); Xg = lk.Basis(ctx, "d", N, nev)
    evg0, resg0, infog0 = lk.eigs(Ag, Xg, nev, x0=x0, kdim=4 * nev)
    cwd = os.getcwd()
    try:
        os.chdir(tmp_path)
        ctx.set_option("write_intermediate", 1)
        ev1, res1, info1 = lk.eighs(A, X, nev, x0=x0, kdim=60, tolerance=1e-6)
        evg1, resg1, infog1 = lk.eigs(Ag, Xg, nev, x0=x0, kdim=4 * nev)
    finally:
        ctx.set_option("write_intermediate", 0)
        os.chdir(cwd)
    assert info1 == info0 and 4 < info1 < 60 and np.allclose(ev1, ev0, rtol=1e-13, atol=0)
    assert infog1 == infog0 and np.allclose(evg1, evg0, rtol=1e-13, atol=1e-13)
    assert np.all(res0 < 1e-6)                                               # without the option: the residuals of the returned pairs
    assert np.all(np.diff(res1) <= 0) and res1[-1] > 1e-3                    # with it: the largest entries of the sorted table, descending
    evo, reso, Xo, ko = oracle.eighs(oracle.Op.dense(Ah), N, nev, x0h, kdim=60, tolerance=1e-6, write_intermediate=True)
    assert ko == info1
    np.testing.assert_allclose(res1, reso, rtol=1e-6)
    lines = open(tmp_path / "eighs_output.txt").read().splitlines()
    assert len(lines) == info1 + 1 and lines[0].split() == ["Iter", "value", "residual", "conv"]
    glines = open(tmp_path / "eigs_output.txt").read().splitlines()
    assert glines[0].split() == ["Iter", "Re", "Im", "modulus", "residual", "conv"] and len(glines) >= 2


def _solve_with_failing_callback(lk, ctx, case, fail_at):
    """One small solve whose user callback returns 5 on its `fail_at`-th call (0: never): a host preconditioner (identity) for
    the *_precond cases, a capturable callback operator that applies the 2-D Laplacian for the *_device cases."""
    import ctypes as C
    nx, ny = 48, 40
    n = nx * ny
    S = lk.LinOp.stencil5(ctx, "d", nx, ny, (4.0, -1.0, -1.0, -1.0, -1.0))
    calls = [0]

    def result():
        calls[0] += 1
        return 5 if calls[0] == fail_at else 0

    def wrap(ptr):
        h = C.c_void_p()
        assert ctx.lib.lkb_vec_wrap(ctx.h, lk.KINDS["d"], n, n, 0, ptr, C.byref(h)) == 0
        return lk.Vector(ctx, "d", n, _handle=h)

    def matvec(xp, yp, trans, stream):
        S.matvec(wrap(xp), wrap(yp))
        return result()
    solver, path = case.split("_")
    A, pre = (S, lambda v, nloc, it, cur, tgt, stream: result()) if path == "precond" else \
             (lk.LinOp.callback(ctx, "d", n, n, matvec, capturable=True), None)
    b = lk.Vector(ctx, "d", n).put(np.random.default_rng(40).standard_normal(n))
    x = lk.Vector(ctx, "d", n)
    kw = dict(maxiter=300) if solver == "cg" else dict(kdim=20, maxiter=20)
    info, meta = getattr(lk, solver)(A, b, x, preconditioner=pre, **kw)
    return info, meta["res"], x.get()


@pytest.mark.parametrize("graphs", [True, False])
def test_failing_callback_releases_the_solver_and_leaves_the_context_usable(lk, ctx, graphs):
    """A host preconditioner that fails on its 3rd call (gmres, fgmres, cg) and a capturable callback operator that fails on its
    2nd call (the device GMRES cycle and the device CG loop: inside the graph capture when graphs are on): each solve raises
    LkbError naming the callback, and a clean solve on the same context afterwards is bitwise equal to one on a fresh context."""
    fresh = lk.Context(0)
    try:
        for c in (ctx, fresh):
            c.set_graphs(graphs)
        for case, fail_at in [("gmres_precond", 3), ("fgmres_precond", 3), ("cg_precond", 3), ("gmres_device", 2), ("cg_device", 2)]:
            with pytest.raises(lk.LkbError, match="callback returned 5"):
                _solve_with_failing_callback(lk, ctx, case, fail_at)
            info, res, x = _solve_with_failing_callback(lk, ctx, case, 0)
            info0, res0, x0 = _solve_with_failing_callback(lk, fresh, case, 0)
            assert info == info0 != 0 and res == res0 and np.array_equal(x, x0), case
    finally:
        ctx.set_graphs(True)
        fresh.close()
