"""CPU checks of the Chebyshev preconditioner: the host reference against the closed form and its positive definiteness with
the default bounds, the Gershgorin bound of the Laplacians, and the new kernels on the built library (128-bit streaming
loads in k_cheb_update, no spills in the update, Gershgorin and fused stencil kernels)."""
import os
import re
import shutil
import subprocess

import numpy as np
import pytest

from chebyshev_cases import chebyshev_apply, chebyshev_closed_form, gershgorin, stencil_csr
from helpers import LAPLACE7, POISSON5


def _hermitian(n, cplx, seed):
    """A Hermitian positive definite matrix with a positive, varying diagonal and kappa(D^-1 A) of a few hundred."""
    rng = np.random.default_rng(seed)
    X = rng.standard_normal((n, n)) + (1j * rng.standard_normal((n, n)) if cplx else 0)
    Q, _ = np.linalg.qr(X)
    A = (Q * np.geomspace(1e-2, 1.0, n)) @ Q.conj().T
    s = np.geomspace(0.5, 4.0, n)
    return s[:, None] * (A + A.conj().T) / 2 * s[None, :]


@pytest.mark.parametrize("cplx", [False, True])
@pytest.mark.parametrize("m", [1, 2, 3, 8, 16])
def test_reference_matches_closed_form(oracle, cplx, m):
    n = 40
    A = _hermitian(n, cplx, 3 + m)
    Ao = oracle.Op.dense(np.asfortranarray(A))
    invd = 1.0 / np.diag(A)
    b = gershgorin(A)
    for a in (b / 100.0, b / 7.0):
        Mc = chebyshev_closed_form(A, m, a, b)
        R = np.eye(n, dtype=A.dtype)
        Mr = np.column_stack([chebyshev_apply(Ao, invd, R[:, j].copy(), m, a, b) for j in range(n)])
        assert np.abs(Mr - Mc).max() <= 1e-13 * np.abs(Mc).max(), (m, a)
        MrH = np.column_stack([chebyshev_apply(Ao, invd, R[:, j].copy(), m, a, b, trans=True) for j in range(n)])
        assert np.abs(MrH - Mc.conj().T).max() <= 1e-13 * np.abs(Mc).max(), (m, a)


@pytest.mark.parametrize("cplx", [False, True])
@pytest.mark.parametrize("m", [1, 2, 3, 8, 16])
def test_default_bounds_give_hermitian_positive_definite_m(oracle, cplx, m):
    n = 40
    A = _hermitian(n, cplx, 30 + m)
    Ao = oracle.Op.dense(np.asfortranarray(A))
    b = gershgorin(A)
    assert b >= np.abs(np.linalg.eigvals(A / np.diag(A)[:, None])).max()        # never below the spectral radius of D^-1 A
    R = np.eye(n, dtype=A.dtype)
    M = np.column_stack([chebyshev_apply(Ao, 1.0 / np.diag(A), R[:, j].copy(), m, b / 100.0, b) for j in range(n)])
    assert np.abs(M - M.conj().T).max() <= 1e-13 * np.abs(M).max()
    assert np.linalg.eigvalsh((M + M.conj().T) / 2).min() > 0.0


def test_gershgorin_of_laplacians_is_two():
    assert gershgorin(stencil_csr((33, 17), POISSON5)) == 2.0
    assert gershgorin(stencil_csr((12, 9, 7), LAPLACE7)) == 2.0
    # the stencil bound the library computes from the coefficients alone
    assert sum(abs(c) for c in POISSON5) / abs(POISSON5[0]) == 2.0
    assert sum(abs(c) for c in LAPLACE7) / abs(LAPLACE7[0]) == 2.0


@pytest.fixture(scope="module")
def so_path():
    from lightkrylov_b200 import build
    return build.build()


def _demangle(names):
    return subprocess.run(["c++filt"], input="\n".join(names), capture_output=True, text=True).stdout.splitlines()


def test_cheb_update_uses_128bit_streaming_loads(so_path):
    if not shutil.which("cuobjdump") or not shutil.which("c++filt"):
        pytest.skip("cuobjdump not available")
    out = subprocess.run(["cuobjdump", "-sass", so_path], capture_output=True, text=True).stdout
    chunks = out.split("Function : ")[1:]
    names = _demangle([c.split("\n", 1)[0].strip() for c in chunks])
    hits = [(n, c) for n, c in zip(names, chunks) if n.startswith("void lkb::k_cheb_update<")]
    assert len(hits) == 4, [n for n, _ in hits]
    for n, body in hits:
        assert "LDG.E.NA.128" in body, n


def test_chebyshev_kernels_do_not_spill(tmp_path):
    from lightkrylov_b200 import build
    if not os.path.exists(build.NVCC):
        pytest.skip("nvcc not available")
    seen = {}
    for src in ("kernels_vec.cu", "kernels_ops.cu"):
        r = subprocess.run([build.NVCC] + build.FLAGS + ["-Xptxas", "-v", "-c", os.path.join(build.CSRC, src),
                            "-o", str(tmp_path / src.replace(".cu", ".o"))], capture_output=True, text=True)
        assert r.returncode == 0, r.stderr[-2000:]
        cur = None
        for line in r.stderr.splitlines():
            m = re.search(r"Compiling entry function '(\w+)'", line)
            if m:
                cur = _demangle([m.group(1)])[0]
                cur = cur if ("lkb::k_cheb_update<" in cur or "lkb::k_gershgorin<" in cur or "ChebStep" in cur) else None
            elif cur and "spill" in line:
                seen[cur] = line
                assert "0 bytes spill stores, 0 bytes spill loads" in line, (cur, line)
    count = lambda pat: sum(bool(re.match(pat, n)) for n in seen)                 # noqa: E731
    assert count(r"void lkb::k_cheb_update<") == 4
    assert count(r"void lkb::k_gershgorin<") == 12                                # 4 kinds x (csr, blocked csr, dense)
    # 4 kinds x (full pack, PW = 1), z has only PW = 1
    assert count(r"void lkb::k_stencil<.*ChebStep") == 7 and count(r"void lkb::k_stencil_smem<.*ChebStep") == 7
