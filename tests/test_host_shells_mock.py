"""The product's host shells (lightkrylov_b200/csrc/lkb_eig.cu: eigs incl. the literal post-convergence Krylov-Schur restart,
eighs, svds, krylov_schur; LAPACK in the precision of the kind; stable descending sort_index; write_intermediate side effect)
run WITHOUT a GPU: tests/host_shells_mock.cu includes that translation unit verbatim and replaces the device underneath it
-- CUDA runtime calls by host memory, the Krylov steps by the C oracle -- so the C++ control flow sees exactly the
Hessenberg / tridiagonal / bidiagonal columns the Python oracle shells see, and the two must agree (same `info`, same
eigenvalue ORDER, same residuals, same vectors).  The real device path is checked by the -m gpu tests; this suite is the CPU
regression net of the host logic (it is how changes to the shells are verified when no GPU is at hand)."""
import ctypes as C
import glob
import os
import shutil
import subprocess

import numpy as np
import pytest

from helpers import randn

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "lightkrylov_b200", "csrc")
NVCC = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
KINDS = {"s": 0, "d": 1, "c": 2, "z": 3}
N = 128

pytestmark = pytest.mark.skipif(not os.path.exists(NVCC) and shutil.which("nvcc") is None, reason="needs nvcc to compile the harness")


@pytest.fixture(scope="module")
def oracle():
    from oracle import lk_oracle
    lk_oracle.lib()
    return lk_oracle


def _declare_alloc_hooks(lib):
    lib.mock_fail_at.argtypes = [C.c_int64]
    lib.mock_allocs.restype = C.c_int64
    lib.mock_live.argtypes = [C.c_void_p]


def _live(lib):
    out = (C.c_int64 * 4)()                                      # bases, vectors, pinned blocks, device buffers
    lib.mock_live(out)
    return list(out)


LKB_ERR_ALLOC = -6


def _fail_each_allocation(lib, call):
    """`call()` runs one solver and returns its code.  Counts the N allocations a successful call makes, then fails the n-th one
    for every n = 1..N: the call must return LKB_ERR_ALLOC and leave no basis, vector, pinned block or device buffer behind."""
    lib.mock_fail_at(0)
    before = _live(lib)
    assert call() == 0, lib.mock_last_error()
    nalloc = lib.mock_allocs()
    assert nalloc > 0 and _live(lib) == before
    try:
        for n in range(1, nalloc + 1):
            lib.mock_fail_at(n)
            rc = call()
            assert (rc, _live(lib)) == (LKB_ERR_ALLOC, before), (n, nalloc)
    finally:
        lib.mock_fail_at(0)
    return nalloc


@pytest.fixture(scope="module")
def mock(tmp_path_factory, oracle):
    import scipy
    import __graft_entry__
    __graft_entry__.build()
    out = str(tmp_path_factory.mktemp("mock") / "libhost_shells_mock.so")
    nvcc = NVCC if os.path.exists(NVCC) else shutil.which("nvcc")
    odir = os.path.join(ROOT, "oracle")
    subprocess.check_call([nvcc, "-gencode", "arch=compute_100a,code=sm_100a", "-O1", "-std=c++17", "-shared", "-Xcompiler", "-fPIC",
                           "-diag-suppress", "174", "-I", CSRC, os.path.join(ROOT, "tests", "host_shells_mock.cu"), "-o", out,
                           "-L", CSRC, "-llkb", "-L", odir, "-llk_oracle", "-ldl", "-Xlinker", "-rpath=" + CSRC,
                           "-Xlinker", "-rpath=" + odir, "-Xlinker", "-Bsymbolic"], stderr=subprocess.DEVNULL)
    lib = C.CDLL(out)
    vp, i32, i64, dbl = C.c_void_p, C.c_int32, C.c_int64, C.c_double
    lib.mock_ctx_new.restype = vp; lib.mock_ctx_new.argtypes = [C.c_int]
    lib.mock_ctx_free.argtypes = [vp]
    lib.mock_op_new.restype = vp; lib.mock_op_new.argtypes = [vp, C.c_int, i64, i64, vp]
    lib.mock_op_free.argtypes = [vp]
    lib.mock_vec_new.restype = vp; lib.mock_vec_new.argtypes = [vp, C.c_int, i64, vp]
    lib.mock_vec_free.argtypes = [vp]
    lib.mock_basis_get.argtypes = [vp, vp]; lib.mock_basis_put.argtypes = [vp, vp]
    lib.mock_last_error.restype = C.c_char_p
    lib.lkb_basis_create.argtypes = [vp, C.c_int, i64, i64, i64, C.c_int, C.POINTER(vp)]
    lib.lkb_basis_destroy.argtypes = [vp]
    lib.lkb_set_lapack.argtypes = [C.c_char_p, C.c_char_p, C.c_char_p]
    lib.lkb_eigs.argtypes = [vp, vp, C.c_int, vp, vp, C.POINTER(i32), vp, i32, dbl, i32]
    lib.lkb_eighs.argtypes = [vp, vp, C.c_int, vp, vp, C.POINTER(i32), vp, i32, dbl]
    lib.lkb_svds.argtypes = [vp, vp, vp, vp, C.c_int, vp, C.POINTER(i32), vp, i32, dbl]
    lib.lkb_krylov_schur.argtypes = [vp, vp, C.c_int, C.c_int, C.POINTER(i32)]
    _declare_alloc_hooks(lib)
    blas = glob.glob(os.path.join(os.path.dirname(os.path.dirname(scipy.__file__)), "scipy.libs", "libscipy_openblas*.so"))[0]
    assert lib.lkb_set_lapack(blas.encode(), b"scipy_", b"_") == 0, lib.mock_last_error()
    return lib


class Shells:
    """thin driver of the C++ shells on host memory"""

    def __init__(self, lib, kind, write_intermediate=False):
        self.lib, self.kind, self.dt = lib, kind, {"s": np.float32, "d": np.float64, "c": np.complex64, "z": np.complex128}[kind]
        self.ctx = lib.mock_ctx_new(int(write_intermediate))
        self.keep = []

    def close(self):
        self.lib.mock_ctx_free(self.ctx)

    def op(self, oracle_op):
        self.keep.append(oracle_op)
        return self.lib.mock_op_new(self.ctx, KINDS[self.kind], oracle_op.m, oracle_op.n, C.addressof(oracle_op.st))

    def basis(self, n, ncols, data=None):
        h = C.c_void_p()
        assert self.lib.lkb_basis_create(self.ctx, KINDS[self.kind], n, n, 0, ncols, C.byref(h)) == 0
        if data is not None:
            a = np.asfortranarray(data, dtype=self.dt); self.lib.mock_basis_put(h, a.ctypes.data)
        return h

    def get(self, h, n, ncols):
        out = np.zeros((n, ncols), dtype=self.dt, order="F")
        self.lib.mock_basis_get(h, out.ctypes.data)
        return out

    def vec(self, x):
        a = np.ascontiguousarray(x, dtype=self.dt); self.keep.append(a)
        return self.lib.mock_vec_new(self.ctx, KINDS[self.kind], a.size, a.ctypes.data)

    def check(self, rc):
        assert rc == 0, self.lib.mock_last_error()

    def eigs(self, A, n, nev, x0, kdim=0, tol=-1.0, trans=False):
        X = self.basis(n, nev); ev = np.zeros(2 * nev); res = np.zeros(nev); info = C.c_int32()
        self.check(self.lib.lkb_eigs(A, X, nev, ev.ctypes.data, res.ctypes.data, C.byref(info), self.vec(x0), kdim, tol, int(trans)))
        return ev[0::2] + 1j * ev[1::2], res, self.get(X, n, nev), info.value

    def eighs(self, A, n, nev, x0, kdim=0, tol=-1.0):
        X = self.basis(n, nev); ev = np.zeros(nev); res = np.zeros(nev); info = C.c_int32()
        self.check(self.lib.lkb_eighs(A, X, nev, ev.ctypes.data, res.ctypes.data, C.byref(info), self.vec(x0), kdim, tol))
        return ev, res, self.get(X, n, nev), info.value

    def svds(self, A, m, n, nsv, u0, kdim=0, tol=-1.0):
        U = self.basis(m, nsv); V = self.basis(n, nsv); S = np.zeros(nsv); res = np.zeros(nsv); info = C.c_int32()
        self.check(self.lib.lkb_svds(A, U, S.ctypes.data, V, nsv, res.ctypes.data, C.byref(info), self.vec(u0), kdim, tol))
        return S, res, self.get(U, m, nsv), self.get(V, n, nsv), info.value


def _toeplitz(n, sub, diag, sup, dt):
    A = np.zeros((n, n), dtype=dt); i = np.arange(n)
    A[i, i] = diag; A[i[1:], i[:-1]] = sub; A[i[:-1], i[1:]] = sup
    return np.asfortranarray(A)


def _tol(kind):
    return 1e-11 if kind in "dz" else 2e-4


def _aligned(X, Xo, ev, kind):
    """Ritz vectors agree up to the complex phase LAPACK's normalisation leaves open ("largest component real" flips between two
    components of nearly equal modulus under rounding-level perturbations): 1 - |<v, vo>| / (|v| |vo|) per eigenvector; real
    kinds: columns (i, i+1) of a conjugate pair hold (Re, Im) of the first eigenvalue's vector."""
    worst, i, nev = 0.0, 0, X.shape[1]
    while i < nev:
        if kind in "cz" or ev[i].imag == 0:
            v, vo = X[:, i].astype(np.complex128), Xo[:, i].astype(np.complex128); i += 1
        elif i + 1 < nev:
            v, vo = X[:, i] + 1j * X[:, i + 1], Xo[:, i] + 1j * Xo[:, i + 1]; i += 2
        else:
            break
        worst = max(worst, abs(1.0 - abs(np.vdot(v, vo)) / (np.linalg.norm(v) * np.linalg.norm(vo))))
        worst = max(worst, abs(np.linalg.norm(v) - np.linalg.norm(vo)))
    return worst


@pytest.mark.parametrize("kind", ["d", "z", "s", "c"])
def test_eigs_shell_matches_oracle_shell(mock, oracle, kind):
    """nev = 8, kdim = 32: Krylov-Schur restarts, the literal extra restart after convergence, stable descending sort --
    same niter, same eigenvalues IN THE SAME ORDER, same residual entries, same Ritz vectors."""
    dt = oracle.DTYPES[kind]; nev = 8
    # complex kinds: a diagonal ramp breaks the +/- symmetry of the spectrum, so no two Ritz values have (nearly) equal moduli --
    # the order of near-ties would be decided by rounding noise
    Ah = _toeplitz(N, -0.5, 1.0, 0.5, dt) if kind in "sd" else np.asfortranarray(
        (_toeplitz(N, -0.5, 1.0, 0.5, dt) + np.diag((0.2 + 0.3j) * np.linspace(0, 1, N))).astype(dt))
    x0 = randn(np.random.default_rng(21), N, dt)
    sh = Shells(mock, kind)
    ev, res, X, info = sh.eigs(sh.op(oracle.Op.dense(Ah)), N, nev, x0, kdim=4 * nev)
    evo, reso, Xo, infoo = oracle.eigs(oracle.Op.dense(Ah), N, nev, x0, kdim=4 * nev)
    sh.close()
    assert info == infoo and info > 4 * nev
    assert np.abs(ev - evo).max() < _tol(kind) * np.abs(evo).max()              # elementwise: same order
    # eigs' returned residuals are entries of the PRE-restart table picked with POST-restart indices (the reference's literal flow,
    # DESIGN.md section 1): which entry lands where depends on the order geev lists the restarted Schur block, i.e. on rounding
    # noise -- they are not comparable elementwise, only sane
    assert np.all(np.isfinite(res)) and np.all(res >= 0) and np.all(np.isfinite(reso))
    assert _aligned(X, Xo, ev, kind) < (1e-8 if kind in "dz" else 5e-3)
    if kind in "sd":
        assert ev[0].imag > 0 and ev[1] == np.conj(ev[0])                       # a conjugate pair stays (+, -)


def test_eigs_shell_transpose_and_random_start(mock, oracle):
    """transpose = .true. runs the factorisation on A^H (same spectrum for a real matrix, other Ritz vectors); x0 absent =
    normalised random start vector (no comparison possible: the shell must converge to the same leading eigenvalues)."""
    nev = 4
    rng = np.random.default_rng(30)
    Ah = np.asfortranarray(np.diag(np.concatenate([np.linspace(0, 1, N - 4), [2.0, 2.5, 3.0, 4.0]])) + 0.05 * rng.standard_normal((N, N)))
    x0 = randn(rng, N, np.float64)
    sh = Shells(mock, "d")
    A = sh.op(oracle.Op.dense(Ah))
    ev, res, X, info = sh.eigs(A, N, nev, x0, kdim=24, trans=True)
    evo, reso, Xo, infoo = oracle.eigs(oracle.Op.dense(Ah), N, nev, x0, kdim=24, trans=True)
    assert info == infoo and np.abs(ev - evo).max() < 1e-10 * np.abs(evo).max()
    assert np.all(ev.imag == 0) and np.abs(Ah.T @ X - X * ev.real[None, :]).max() < 1e-6      # left eigenvectors: A^T X = X diag(E)
    # no start vector: lkb_eigs(..., x0 = NULL, ...)
    Xh = sh.basis(N, nev); evr = np.zeros(2 * nev); resr = np.zeros(nev); infor = C.c_int32()
    sh.check(mock.lkb_eigs(A, Xh, nev, evr.ctypes.data, resr.ctypes.data, C.byref(infor), None, 24, -1.0, 0))
    sh.close()
    lead = np.sort(np.abs(np.linalg.eigvals(Ah)))[::-1][:nev]
    assert infor.value > 0 and np.abs(np.sort(np.hypot(evr[0::2], evr[1::2]))[::-1] - lead).max() < 1e-6


def test_eigs_full_spectrum_default_kdim(mock, oracle):
    """the reference's test_evp_rdp: nev = n, kdim = 4 nev > n; elementwise against the analytic spectrum (pair order)."""
    a, b = 1.0, 0.5
    Ah = _toeplitz(N, -b, a, b, np.float64); x0 = np.random.default_rng(20).standard_normal(N)
    sh = Shells(mock, "d")
    ev, res, X, info = sh.eigs(sh.op(oracle.Op.dense(Ah)), N, N, x0)
    sh.close()
    true = np.zeros(N, dtype=np.complex128)
    for k in range(1, N // 2 + 1):
        true[2 * k - 2] = a + 2j * b * np.cos(k * np.pi / (N + 1)); true[2 * k - 1] = np.conj(true[2 * k - 2])
    assert info == N
    assert np.max(np.abs(ev - true) / np.abs(true)) < oracle.RTOL["d"]
    v = X[:, 0] + 1j * X[:, 1]
    assert np.linalg.norm(Ah @ v - ev[0] * v) < 1e-8 * np.linalg.norm(v)         # columns (Re, Im) of the pair's first eigenvalue


@pytest.mark.parametrize("kind", ["d", "z", "s", "c"])
def test_eighs_and_svds_shells_match_oracle_shells(mock, oracle, kind):
    dt = oracle.DTYPES[kind]; nev = 6
    rng = np.random.default_rng(26)
    D = np.diag(np.concatenate([np.linspace(0, 1, N - 4), [2.0, 2.5, 3.0, 4.0]])); Q, _ = np.linalg.qr(randn(rng, (N, N), np.complex128 if kind in "cz" else np.float64))
    Ah = Q @ D @ Q.conj().T; Ah = np.asfortranarray(((Ah + Ah.conj().T) / 2).astype(dt))
    x0 = randn(np.random.default_rng(25), N, dt)
    sh = Shells(mock, kind)
    ev, res, X, info = sh.eighs(sh.op(oracle.Op.dense(Ah)), N, nev, x0, kdim=80)
    evo, reso, Xo, infoo = oracle.eighs(oracle.Op.dense(Ah), N, nev, x0, kdim=80)
    assert info == infoo and 4 < info < 80
    assert np.abs(ev - evo).max() < _tol(kind) * np.abs(evo).max()
    np.testing.assert_allclose(res, reso, rtol=1e-3 if kind in "dz" else 0.3, atol=(1e-3 if kind in "dz" else 0.1) * oracle.RTOL[kind])
    assert np.abs(X - Xo).max() < (1e-8 if kind in "dz" else 5e-3)
    # svds on a rectangular operator
    m, n, nsv = 90, 70, 5
    M = np.asfortranarray(randn(rng, (m, n), dt)); u0 = randn(rng, m, dt)
    S, sres, U, V, sinfo = sh.svds(sh.op(oracle.Op.dense(M)), m, n, nsv, u0, kdim=40)
    So, sreso, Uo, Vo, sinfoo = oracle.svds(oracle.Op.dense(M), nsv, u0, kdim=40)
    sh.close()
    assert sinfo == sinfoo
    assert np.abs(S - So).max() < _tol(kind) * So.max()
    np.testing.assert_allclose(sres, sreso, rtol=1e-3 if kind in "dz" else 0.3, atol=(1e-3 if kind in "dz" else 0.1) * oracle.RTOL[kind])
    assert np.abs(U - Uo).max() < (1e-8 if kind in "dz" else 5e-3) and np.abs(V - Vo).max() < (1e-8 if kind in "dz" else 5e-3)


def test_write_intermediate_side_effect_in_the_shells(mock, oracle, tmp_path):
    """write_results sorts the residual table in place (IterativeSolvers.fypp:882-924): with the option on, the C++ shells
    return the same residuals as the oracle restatement of that side effect, write the table files, and keep info / values."""
    kind, nev = "d", 4
    rng = np.random.default_rng(26)
    D = np.diag(np.concatenate([np.linspace(0, 1, N - 4), [2.0, 2.5, 3.0, 4.0]])); Q, _ = np.linalg.qr(rng.standard_normal((N, N)))
    Ah = Q @ D @ Q.T; Ah = np.asfortranarray((Ah + Ah.T) / 2)
    x0 = randn(np.random.default_rng(25), N, np.float64)
    Ag = _toeplitz(N, -0.5, 1.0, 0.5, np.float64)
    off = Shells(mock, kind); on = Shells(mock, kind, write_intermediate=True)
    ev0, res0, X0, info0 = off.eighs(off.op(oracle.Op.dense(Ah)), N, nev, x0, kdim=60, tol=1e-6)
    evg0, resg0, Xg0, infog0 = off.eigs(off.op(oracle.Op.dense(Ag)), N, nev, x0, kdim=16)
    cwd = os.getcwd()
    try:
        os.chdir(tmp_path)
        ev1, res1, X1, info1 = on.eighs(on.op(oracle.Op.dense(Ah)), N, nev, x0, kdim=60, tol=1e-6)
        evg1, resg1, Xg1, infog1 = on.eigs(on.op(oracle.Op.dense(Ag)), N, nev, x0, kdim=16)
        M = np.asfortranarray(randn(rng, (60, 50), np.float64)); u0 = randn(rng, 60, np.float64)
        S1, sres1, U1, V1, sinfo1 = on.svds(on.op(oracle.Op.dense(M)), 60, 50, 3, u0, kdim=30)
    finally:
        os.chdir(cwd)
    off.close(); on.close()
    assert info1 == info0 and np.allclose(ev1, ev0, rtol=1e-13) and 4 < info1 < 60
    assert infog1 == infog0 and np.allclose(evg1, evg0, rtol=1e-13, atol=1e-13)
    assert np.all(res0 < 1e-6) and np.all(np.diff(res1) <= 0) and res1[-1] > 1e-3
    _, reso, _, ko = oracle.eighs(oracle.Op.dense(Ah), N, nev, x0, kdim=60, tolerance=1e-6, write_intermediate=True)
    assert ko == info1
    np.testing.assert_allclose(res1, reso, rtol=1e-8)
    _, resgo, _, infogo = oracle.eigs(oracle.Op.dense(Ag), N, nev, x0, kdim=16, write_intermediate=True)
    assert infogo == infog1 and np.all(np.isfinite(resg1)) and np.all(resg1 >= 0)      # (eigs residuals: not comparable elementwise)
    _, sreso, _, _, sinfoo = oracle.svds(oracle.Op.dense(M), 3, u0, kdim=30, write_intermediate=True)
    assert sinfoo == sinfo1
    np.testing.assert_allclose(sres1, sreso, rtol=1e-8, atol=1e-14)
    lines = open(tmp_path / "eighs_output.txt").read().splitlines()
    assert len(lines) == info1 + 1 and lines[0].split() == ["Iter", "value", "residual", "conv"]
    assert open(tmp_path / "eigs_output.txt").read().splitlines()[0].split() == ["Iter", "Re", "Im", "modulus", "residual", "conv"]
    assert len(open(tmp_path / "svds_output.txt").read().splitlines()) == sinfo1 + 1


@pytest.mark.parametrize("kind", ["d", "z", "s"])
def test_krylov_schur_shell_matches_oracle(mock, oracle, kind):
    """lkb_krylov_schur (BaseKrylov.fypp:782-834) on a full Arnoldi factorisation: same n, same restarted H and basis."""
    dt = oracle.DTYPES[kind]; kdim = 32
    rng = np.random.default_rng(22)
    Ah = np.asfortranarray((randn(rng, (N, N), dt) / np.sqrt(N)).astype(dt))
    X = np.zeros((N, kdim + 1), dtype=dt, order="F"); X[:, 0] = randn(rng, N, dt); oracle.normalize(X[:, 0])
    H = np.zeros((kdim + 1, kdim), dtype=dt, order="F")
    assert oracle.arnoldi(oracle.Op.dense(Ah), X, H) == 0
    Xo, Ho = X.copy(order="F"), H.copy(order="F")
    nko = oracle.krylov_schur(Xo, Ho)
    sh = Shells(mock, kind)
    hX = sh.basis(N, kdim + 1, X); Hc = H.copy(order="F"); nk = C.c_int32()
    sh.check(mock.lkb_krylov_schur(hX, Hc.ctypes.data, kdim + 1, kdim, C.byref(nk)))
    Xc = sh.get(hX, N, kdim + 1)
    sh.close()
    assert nk.value == nko and 0 < nko < kdim
    tol = 1e-10 if kind in "dz" else 1e-3
    assert np.abs(Hc - Ho).max() < tol and np.abs(Xc - Xo).max() < tol
    assert np.abs(Ah @ Xc[:, :nko] - Xc[:, :nko + 1] @ Hc[:nko + 1, :nko]).max() < oracle.RTOL[kind]


# ---- the Krylov-exponential shells (lkb_expm.cu) on the mocked device ------------------------------------------------------------------
_QR_CB = C.CFUNCTYPE(C.c_int, C.c_int, C.c_int64, C.c_int, C.c_void_p, C.c_int64, C.c_void_p, C.c_int, C.POINTER(C.c_int32), C.c_double,
                     C.POINTER(C.c_int32))


@pytest.fixture(scope="module")
def expm_mock(tmp_path_factory, oracle):
    import __graft_entry__
    __graft_entry__.build()
    out = str(tmp_path_factory.mktemp("expm_mock") / "libhost_expm_mock.so")
    nvcc = NVCC if os.path.exists(NVCC) else shutil.which("nvcc")
    odir = os.path.join(ROOT, "oracle")
    subprocess.check_call([nvcc, "-gencode", "arch=compute_100a,code=sm_100a", "-O1", "-std=c++17", "-shared", "-Xcompiler", "-fPIC",
                           "-diag-suppress", "174", "-I", CSRC, os.path.join(ROOT, "tests", "host_expm_mock.cu"), "-o", out,
                           "-L", odir, "-llk_oracle", "-ldl", "-Xlinker", "-rpath=" + odir, "-Xlinker", "-Bsymbolic"],
                          stderr=subprocess.DEVNULL)
    lib = C.CDLL(out)
    vp, i32, i64, dbl = C.c_void_p, C.c_int32, C.c_int64, C.c_double
    lib.mock_ctx_new.restype = vp; lib.mock_ctx_new.argtypes = [C.c_int]
    lib.mock_ctx_free.argtypes = [vp]
    lib.mock_op_new.restype = vp; lib.mock_op_new.argtypes = [vp, C.c_int, i64, i64, vp]
    lib.mock_vec_new.restype = vp; lib.mock_vec_new.argtypes = [vp, C.c_int, i64, vp]
    lib.mock_basis_get.argtypes = [vp, vp]; lib.mock_basis_put.argtypes = [vp, vp]
    lib.mock_last_error.restype = C.c_char_p
    lib.lkb_basis_create.argtypes = [vp, C.c_int, i64, i64, i64, C.c_int, C.POINTER(vp)]
    lib.lkb_kexpm_vec.argtypes = [vp, vp, vp, dbl, dbl, C.POINTER(i32), i32, i32]
    lib.lkb_kexpm_mat.argtypes = [vp, vp, vp, C.c_int, dbl, dbl, C.POINTER(i32), i32, i32]
    lib.lkb_krylov_expta.argtypes = [vp, vp, vp, dbl, C.POINTER(i32), i32]
    _declare_alloc_hooks(lib)
    dts = {0: np.float32, 1: np.float64, 2: np.complex64, 3: np.complex128}

    def qr_pivoting(kind, n, p, Qp, ld, Rp, ldr, permp, tol, infop):          # lkb_qr_pivoting -> oracle.qr_with_pivoting, in place
        dt = np.dtype(dts[kind])
        assert ld == n
        Q = np.frombuffer((C.c_char * (n * p * dt.itemsize)).from_address(Qp), dtype=dt).reshape((n, p), order="F")
        info, R, perm = oracle.qr_with_pivoting(Q, tol=None if tol < 0 else tol)
        Rout = np.frombuffer((C.c_char * (ldr * p * dt.itemsize)).from_address(Rp), dtype=dt).reshape((ldr, p), order="F")
        Rout[:p, :p] = R
        for i in range(p):
            permp[i] = int(perm[i]) + 1
        infop[0] = info
        return 0

    lib._cb = _QR_CB(qr_pivoting)                                              # keep the trampoline alive
    lib.mock_set_qr_pivoting.argtypes = [_QR_CB]
    lib.mock_set_qr_pivoting(lib._cb)
    return lib


class ExpmShells(Shells):
    def kexpm(self, A, b, tau, tol, trans=False, kdim=0):
        n = b.size
        c = self.vec(np.zeros(n, dtype=self.dt)); info = C.c_int32()
        self.check(self.lib.lkb_kexpm_vec(c, A, self.vec(b), tau, tol, C.byref(info), int(trans), kdim))
        return self._vec_get(c, n), info.value

    def exptA(self, A, b, tau, trans=False):
        n = b.size
        c = self.vec(np.zeros(n, dtype=self.dt)); info = C.c_int32()
        self.check(self.lib.lkb_krylov_expta(c, A, self.vec(b), tau, C.byref(info), int(trans)))
        return self._vec_get(c, n), info.value

    def kexpm_mat(self, A, B, tau, tol, trans=False, kdim=0):
        n, p = B.shape
        hB = self.basis(n, p, B); hC = self.basis(n, p); info = C.c_int32()
        self.check(self.lib.lkb_kexpm_mat(hC, A, hB, p, tau, tol, C.byref(info), int(trans), kdim))
        return self.get(hC, n, p), info.value

    def _vec_get(self, v, n):
        # lkb_vec_s { ctx, kind, n, n_global, row0, d, owns }: the data pointer is the 6th 8-byte field
        d = C.cast(v, C.POINTER(C.c_void_p))[5]
        return np.frombuffer((C.c_char * (n * np.dtype(self.dt).itemsize)).from_address(d), dtype=self.dt).copy()


@pytest.mark.parametrize("kind", ["d", "z", "s", "c"])
def test_kexpm_vec_shell_matches_oracle_shell(expm_mock, oracle, kind):
    """lkb_kexpm_vec / lkb_krylov_expta (ExpmLib.fypp:128-232, 364-392) on the mocked device vs oracle.kexpm_vec: same info (dimension
    used), same vector -- incl. the literal behaviour on Arnoldi breakdown (info = k + 2) and the zero input."""
    dt = oracle.DTYPES[kind]; dims = (24, 20); n = 480
    Ao = oracle.Op.stencil(kind, dims, (-4.0, 1.0, 0.8, 1.0, 1.2))
    b = oracle.fill(n, kind, "uniform", 3)
    tol = 1e-10 if kind in "dz" else 1e-5
    sh = ExpmShells(expm_mock, kind)
    A = sh.op(Ao)
    c, info = sh.kexpm(A, b, 0.1, tol)
    co, infoo = oracle.kexpm_vec(Ao, b, 0.1, tol)
    assert info == infoo and info > 1
    assert np.linalg.norm(c - co) < (1e-12 if kind in "dz" else 1e-5) * np.linalg.norm(co)
    ct, tinfo = sh.kexpm(A, b, 0.1, tol, trans=True)
    cto, tinfoo = oracle.kexpm_vec(Ao, b, 0.1, tol, trans=True)
    assert tinfo == tinfoo and np.linalg.norm(ct - cto) < (1e-12 if kind in "dz" else 1e-5) * np.linalg.norm(cto)
    ce, einfo = sh.exptA(A, b, 0.1)
    ceo, einfoo = oracle.kexpm_vec(Ao, b, 0.1, oracle.ATOL[kind], kdim=30)
    assert einfo == einfoo and np.linalg.norm(ce - ceo) < (1e-12 if kind in "dz" else 1e-5) * np.linalg.norm(ceo)
    z, zinfo = sh.kexpm(A, np.zeros(n, dtype=dt), 0.1, tol)
    assert zinfo == 1 and not z.any()
    if kind in "dz":                                                            # breakdown: 3-dimensional invariant subspace
        m = 96
        D = np.asfortranarray(np.diag(np.arange(1, m + 1)).astype(dt))
        b3 = np.zeros(m, dtype=dt); b3[:3] = [1.0, 2.0, -1.5]
        c3, i3 = sh.kexpm(sh.op(oracle.Op.dense(D)), b3, 0.2, 1e-12)
        exact = np.exp(0.2 * np.arange(1, m + 1)) * b3
        assert i3 == 5 == oracle.kexpm_vec(oracle.Op.dense(D), b3, 0.2, 1e-12)[1]
        assert np.linalg.norm(c3 - exact) < 1e-12 * np.linalg.norm(exact)
    sh.close()


@pytest.mark.parametrize("kind", ["d", "z", "s"])
@pytest.mark.parametrize("p", [1, 3])
def test_kexpm_mat_shell_matches_oracle_shell(expm_mock, oracle, kind, p):
    """lkb_kexpm_mat (ExpmLib.fypp:234-362) on the mocked device vs oracle.kexpm_mat: same info, same block; the work basis grows
    on demand (info = 30 for p = 3 means 9 block steps > the initial room for 8); transpose; zero input; breakdown exit."""
    dt = oracle.DTYPES[kind]; dims = (24, 20); n = 480
    Ao = oracle.Op.stencil(kind, dims, (-4.0, 1.0, 0.8, 1.0, 1.2))
    B = np.asfortranarray(np.stack([oracle.fill(n, kind, "uniform", 5 + i) for i in range(p)], axis=1))
    tol = 1e-10 if kind in "dz" else 1e-5
    sh = ExpmShells(expm_mock, kind)
    A = sh.op(Ao)
    Cm, info = sh.kexpm_mat(A, B, 0.1, tol, kdim=15)
    Co, infoo = oracle.kexpm_mat(Ao, B, 0.1, tol, kdim=15)
    assert info == infoo and info >= 2 * p
    if kind in "dz":
        assert info // p - 1 > 8                                                # the growth path was taken
    assert np.linalg.norm(Cm - Co) < (1e-11 if kind in "dz" else 1e-4) * np.linalg.norm(Co)
    Ct, tinfo = sh.kexpm_mat(A, B, 0.1, tol, trans=True, kdim=15)
    Cto, tinfoo = oracle.kexpm_mat(Ao, B, 0.1, tol, trans=True, kdim=15)
    assert tinfo == tinfoo and np.linalg.norm(Ct - Cto) < (1e-11 if kind in "dz" else 1e-4) * np.linalg.norm(Cto)
    Z, zinfo = sh.kexpm_mat(A, np.zeros_like(B), 0.1, tol, kdim=15)
    assert zinfo == p and not Z.any()
    if kind == "d" and p == 3:                                                  # breakdown: p = 2 columns in a 4-dimensional invariant subspace
        m = 96
        D = np.asfortranarray(np.diag(np.arange(1, m + 1)).astype(dt))
        Bh = np.zeros((m, 2), order="F"); Bh[:4, 0] = [1.0, 2.0, -1.5, 0.5]; Bh[:4, 1] = [0.3, -1.0, 2.0, 1.0]
        Cb, binfo = sh.kexpm_mat(sh.op(oracle.Op.dense(D)), Bh, 0.2, 1e-12)
        exact = np.exp(0.2 * np.arange(1, m + 1))[:, None] * Bh
        assert binfo == 4 == oracle.kexpm_mat(oracle.Op.dense(D), Bh, 0.2, 1e-12)[1]
        assert np.linalg.norm(Cb - exact) < 1e-12 * np.linalg.norm(exact)
    sh.close()


def test_eig_shells_release_everything_when_an_allocation_fails(mock, oracle):
    """eigs (with Krylov-Schur restarts: a device buffer per restart), eighs and svds: every allocation, work bases and pinned
    step slots included, may fail; each failure is reported as LKB_ERR_ALLOC with nothing left allocated.  A clean call afterwards
    still matches the oracle."""
    i32 = C.c_int32
    nev = 8
    Ah = _toeplitz(N, -0.5, 1.0, 0.5, np.float64)
    x0 = randn(np.random.default_rng(21), N, np.float64)
    sh = Shells(mock, "d")
    A = sh.op(oracle.Op.dense(Ah)); X = sh.basis(N, nev); v0 = sh.vec(x0)
    ev, res, info = np.zeros(2 * nev), np.zeros(nev), i32()
    n_eigs = _fail_each_allocation(mock, lambda: mock.lkb_eigs(A, X, nev, ev.ctypes.data, res.ctypes.data, C.byref(info), v0,
                                                               4 * nev, -1.0, 0))
    assert n_eigs > 4                                                          # Xwrk, two pinned slots, restarts
    D = np.diag(np.concatenate([np.linspace(0, 1, N - 4), [2.0, 2.5, 3.0, 4.0]]))
    Ahs = np.asfortranarray(D)
    As = sh.op(oracle.Op.dense(Ahs)); Xs = sh.basis(N, 4)
    evs, ress = np.zeros(4), np.zeros(4)
    assert _fail_each_allocation(mock, lambda: mock.lkb_eighs(As, Xs, 4, evs.ctypes.data, ress.ctypes.data, C.byref(info), v0,
                                                              40, -1.0)) == 3
    m, n, nsv = 90, 70, 3
    M = np.asfortranarray(randn(np.random.default_rng(26), (m, n), np.float64)); u0 = sh.vec(randn(np.random.default_rng(27), m, np.float64))
    Am = sh.op(oracle.Op.dense(M)); U = sh.basis(m, nsv); V = sh.basis(n, nsv)
    S, sres = np.zeros(nsv), np.zeros(nsv)
    assert _fail_each_allocation(mock, lambda: mock.lkb_svds(Am, U, S.ctypes.data, V, nsv, sres.ctypes.data, C.byref(info), u0,
                                                             30, -1.0)) == 4
    ev1, _, X1, info1 = sh.eigs(A, N, nev, x0, kdim=4 * nev)
    sh.close()
    evo, _, Xo, infoo = oracle.eigs(oracle.Op.dense(Ah), N, nev, x0, kdim=4 * nev)
    assert info1 == infoo and np.abs(ev1 - evo).max() < _tol("d") * np.abs(evo).max()
    assert _aligned(X1, Xo, ev1, "d") < 1e-8


def test_expm_shells_release_everything_when_an_allocation_fails(expm_mock, oracle):
    """kexpm_vec and kexpm_mat (p = 3, through the growth of the work basis and the per-column views of C): each allocation fails
    in turn with LKB_ERR_ALLOC and nothing left allocated; a clean call afterwards still matches the oracle."""
    n, p, tol = 480, 3, 1e-10
    Ao = oracle.Op.stencil("d", (24, 20), (-4.0, 1.0, 0.8, 1.0, 1.2))
    b = oracle.fill(n, "d", "uniform", 3)
    B = np.asfortranarray(np.stack([oracle.fill(n, "d", "uniform", 5 + i) for i in range(p)], axis=1))
    sh = ExpmShells(expm_mock, "d")
    A = sh.op(Ao); cv = sh.vec(np.zeros(n)); bv = sh.vec(b); hB = sh.basis(n, p, B); hC = sh.basis(n, p)
    info = C.c_int32()
    assert _fail_each_allocation(expm_mock, lambda: expm_mock.lkb_kexpm_vec(cv, A, bv, 0.1, tol, C.byref(info), 0, 0)) == 1
    n_mat = _fail_each_allocation(expm_mock, lambda: expm_mock.lkb_kexpm_mat(hC, A, hB, p, 0.1, tol, C.byref(info), 0, 15))
    c, cinfo = sh.kexpm(A, b, 0.1, tol)
    Cm, minfo = sh.kexpm_mat(A, B, 0.1, tol, kdim=15)
    assert minfo // p - 1 > 8 and n_mat == 3 + p                               # Xwrk, X, the doubled X, one view per column
    sh.close()
    co, coinfo = oracle.kexpm_vec(Ao, b, 0.1, tol)
    Co, moinfo = oracle.kexpm_mat(Ao, B, 0.1, tol, kdim=15)
    assert cinfo == coinfo and np.linalg.norm(c - co) < 1e-12 * np.linalg.norm(co)
    assert minfo == moinfo and np.linalg.norm(Cm - Co) < 1e-11 * np.linalg.norm(Co)


# ------------------------------------------------------------------------------------------------------------------------------
# The same C++ shells against REFERENCE-PRODUCED fixtures (tests/golden/ref_solvers.npz: outputs of LightKrylov's own eigs / eighs /
# svds code executed by oracle/f90run.py, see tests/test_ref_golden.py): the product's host control flow -- convergence tests, the
# literal post-convergence Krylov-Schur restart, LAPACK post-processing, sort order, the write_intermediate side effect -- must
# return the reference's `info`, spectra and vectors.  Direct product-vs-reference evidence that needs no GPU.
# ------------------------------------------------------------------------------------------------------------------------------
class _ShellsBackend:
    """adapter of the cases in tests/golden/ref_cases.py onto the mocked-device shells (operators = oracle operators)"""

    def __init__(self, lib, kind, oracle, write_intermediate=False):
        self.sh, self.oracle, self.kind = Shells(lib, kind, write_intermediate=write_intermediate), oracle, kind

    def linop(self, kind, A, sym=False):
        return self.sh.op(self.oracle.Op.dense(np.asfortranarray(A)))

    def stencil(self, kind, dims, coef, sym=False):
        return self.sh.op(self.oracle.Op.stencil(kind, tuple(dims), tuple(float(c) for c in coef)))

    def eigs(self, A, nev, x0, kdim, tolerance, n=None):
        return self.sh.eigs(A, x0.shape[0], nev, x0, kdim=kdim, tol=tolerance)

    def eighs(self, A, nev, x0, kdim, tolerance, write_intermediate=False):
        return self.sh.eighs(A, x0.shape[0], nev, x0, kdim=kdim, tol=tolerance)

    def csr(self, kind, m, n, rowptr, col, val):
        return self.sh.op(self.oracle.Op.csr(m, n, rowptr, col, val))

    def svds(self, A, nsv, u0, kdim, tolerance, write_intermediate=False, shape=None):
        return self.sh.svds(A, u0.shape[0], u0.shape[0] if shape is None else shape[1], nsv, u0, kdim=kdim, tol=tolerance)


@pytest.mark.parametrize("kind", ["d", "z"])
@pytest.mark.parametrize("case", ["eigs_solve", "eighs_solve", "svds_solve", "eighs_write_intermediate", "svds_write_intermediate",
                                  "stencil3d_eigs", "csr_svds"])
def test_cpp_shells_reproduce_reference_outputs(mock, oracle, case, kind, tmp_path, monkeypatch):
    import sys
    sys.path.insert(0, os.path.join(ROOT, "tests", "golden"))
    import ref_cases as rc
    if not rc.applies(case, kind):
        pytest.skip("case not defined for this kind")
    monkeypatch.chdir(tmp_path)                                  # the table files of write_intermediate land here
    fx = np.load(os.path.join(ROOT, "tests", "golden", "ref_solvers.npz"))
    be = _ShellsBackend(mock, kind, oracle, write_intermediate="write_intermediate" in case)
    try:
        got = rc.SOLVER_CASES[case](kind, be)
    finally:
        be.sh.close()
    keys = [k for k in fx.files if k.startswith(f"{case}/{kind}/")]
    assert keys
    for full in keys:
        key = full.split("/")[-1]
        want, have = fx[full], np.asarray(got[key])
        if key == "X" and "eigs" in case:
            continue                                             # (Re, Im) pair layout: free phase, compared through the eigenvalues
        if key.startswith("abs_"):
            assert float(have) < 1e-9
        elif want.dtype.kind in "iub":
            assert np.array_equal(have, want), (full, have.tolist(), want.tolist())
        else:
            err = float(np.abs(have - want).max()) / max(float(np.abs(want).max()), 1e-300)
            assert have.shape == want.shape and err < (1e-8 if key.startswith("abs") else 1e-10), (full, err)
    if "write_intermediate" in case:
        assert os.path.exists(tmp_path / ("eighs_output.txt" if case.startswith("eighs") else "svds_output.txt"))


class _ExpmBackend:
    """kexpm cases of tests/golden/ref_cases.py on the mocked-device exponential shells (lkb_expm.cu)"""

    def __init__(self, lib, kind, oracle):
        self.sh, self.oracle = ExpmShells(lib, kind), oracle

    def linop(self, kind, A, sym=False):
        return self.sh.op(self.oracle.Op.dense(np.asfortranarray(A)))

    def basis(self, kind, ncols, first=None):
        X = np.zeros((N, ncols), dtype=self.sh.dt, order="F")
        if first is not None:
            X[:, :np.asarray(first).reshape(N, -1).shape[1]] = np.asarray(first).reshape(N, -1)
        return X

    def data(self, X):
        return X

    def kexpm(self, c, A, b, tau, tol, kdim):
        out, info = self.sh.kexpm(A, b[:, 0].copy(), tau, tol, kdim=kdim)
        c[:, 0] = out
        return info

    def kexpm_mat(self, Cb, A, B, tau, tol, kdim):
        out, info = self.sh.kexpm_mat(A, B, tau, tol, kdim=kdim)
        Cb[...] = out
        return info


@pytest.mark.parametrize("kind", ["d", "z"])
@pytest.mark.parametrize("case", ["kexpm_solve", "kexpm_block", "kexpm_breakdown"])
def test_cpp_expm_shells_reproduce_reference_outputs(expm_mock, oracle, case, kind):
    """lkb_kexpm_vec / lkb_kexpm_mat (C++ on the mocked device) against what the reference's own kexpm returned: same `info`
    (incl. the literal k + 2 on Arnoldi breakdown), same vectors / block"""
    import sys
    sys.path.insert(0, os.path.join(ROOT, "tests", "golden"))
    import ref_cases as rc
    fx = np.load(os.path.join(ROOT, "tests", "golden", "ref_solvers.npz"))
    be = _ExpmBackend(expm_mock, kind, oracle)
    try:
        got = rc.SOLVER_CASES[case](kind, be)
    finally:
        be.sh.close()
    assert int(got["info"]) == int(fx[f"{case}/{kind}/info"])
    key = "C" if case == "kexpm_block" else "c"
    want = fx[f"{case}/{kind}/{key}"]
    assert float(np.abs(np.asarray(got[key]) - want).max()) / float(np.abs(want).max()) < 1e-10
