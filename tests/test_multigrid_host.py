"""CPU checks of the multigrid preconditioner: the structure of the reference hierarchy of tests/mg_cases.py, the library's
host hierarchy builder (lkb_mg.cu: mg_hierarchy, through a host harness that links liblkb.so) against that reference, the
reference V-cycle's symmetry, adjoint and mesh-independent convergence, and the new kernels on the built library (no
spills)."""
import os
import re
import shutil
import subprocess

import numpy as np
import pytest
import scipy.sparse.linalg as spla

from chebyshev_cases import stencil_csr
from helpers import CONVDIFF7, LAPLACE7, POISSON5
from mg_cases import hierarchy, interp1, vcycle

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "lightkrylov_b200", "csrc")
NVCC = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
COMPLEX5 = (4.0 + 0.5j, -1.2 + 0.3j, -0.8 - 0.1j, -1.1 - 0.2j, -0.9 + 0.25j)
COMPLEX7 = COMPLEX5 + (-1.05 + 0.1j, -0.95 - 0.15j)


@pytest.mark.parametrize("n", [4096, 384, 512, 511, 100])
@pytest.mark.parametrize("coef", ["convdiff", "complex"])
def test_reference_structure(n, coef):
    """Along each axis (the operator is a sum of per-axis terms, so 2-D and 3-D are alike) every coarse operator is
    tridiagonal with constant off-diagonals and a constant diagonal but for its last entry, which differs exactly when a
    level on the way had an even size."""
    pairs = [(-1.3, -0.7), (-1.2, -0.8), (-1.1, -0.9)] if coef == "convdiff" else \
        [(COMPLEX7[1], COMPLEX7[2]), (COMPLEX7[3], COMPLEX7[4]), (COMPLEX7[5], COMPLEX7[6])]
    for cm, cp in pairs:
        T = stencil_csr((n,), np.array([0.0, cm, cp], dtype=complex)) - \
            stencil_csr((n,), np.array([cm + cp, 0, 0], dtype=complex))
        even_seen = False
        m = n
        while m >= 2:
            P = interp1(m)
            even_seen = even_seen or m % 2 == 0
            T = (P.T @ T @ P / 2).tocsr()
            m //= 2
            D = T.toarray()
            assert np.count_nonzero(np.triu(D, 2)) == 0 and np.count_nonzero(np.tril(D, -2)) == 0
            scale = np.abs(D).max()
            for k in (-1, 1):
                dk = np.diag(D, k)
                assert dk.size == 0 or np.abs(dk - dk[0]).max() <= 1e-15 * scale, (n, m, k)
            dg = np.diag(D)
            assert m == 1 or np.abs(dg[:-1] - dg[0]).max() <= 1e-15 * scale, (n, m)
            assert (abs(dg[-1] - dg[0]) > 1e-12 * scale) == (even_seen and m > 1), (n, m, dg[-1], dg[0])


def _harness(tmp_path, cases):
    import __graft_entry__
    __graft_entry__.build()
    exe = str(tmp_path / "host_mg_harness")
    nvcc = NVCC if os.path.exists(NVCC) else shutil.which("nvcc")
    subprocess.check_call([nvcc, "-gencode", "arch=compute_100a,code=sm_100a", "-O1", "-std=c++17", "-I", CSRC,
                           os.path.join(ROOT, "tests", "host_mg_harness.cu"), "-o", exe, "-L", CSRC, "-llkb", "-ldl",
                           "-Xlinker", "-rpath=" + CSRC])
    text = ""
    for dims, coef in cases:
        n = tuple(dims) + (1,) * (3 - len(dims))
        c = np.zeros(7, dtype=complex); c[:len(coef)] = coef
        text += f"{len(dims)} {n[0]} {n[1]} {n[2]}\n" + "\n".join(f"{float(v.real)!r} {float(v.imag)!r}" for v in c) + "\n"
    out = subprocess.run([exe], input=text, check=True, capture_output=True, text=True).stdout.splitlines()
    res, i = [], 0
    while i < len(out):
        _, status, nlev, ninv = out[i].split()
        lv = []
        for ln in out[i + 1:i + 1 + int(nlev)]:
            f = ln.split()
            v = [complex(float(f[k]), float(f[k + 1])) for k in range(3, 23, 2)]
            lv.append(dict(dims=tuple(int(x) for x in f[:3]), c0=v[0], cm=v[1::3], cp=v[2::3], e=v[3::3], lmax=float(f[23])))
        i += 1 + int(nlev)
        inv = np.array([complex(*map(float, ln.split())) for ln in out[i:i + int(ninv)]])
        i += int(ninv)
        res.append((int(status), lv, inv))
    return res


HARNESS_CASES = [((4096, 4096), POISSON5), ((384, 384, 384), LAPLACE7), ((512, 512), CONVDIFF7[:5]), ((511, 100), CONVDIFF7[:5]),
                 ((100, 511), COMPLEX5), ((100, 64, 51), CONVDIFF7), ((40, 33, 34), COMPLEX7), ((384, 100), COMPLEX5),
                 ((20, 25), POISSON5)]


@pytest.mark.skipif(not os.path.exists(NVCC) and shutil.which("nvcc") is None, reason="needs nvcc to compile the harness")
def test_builder_matches_reference(tmp_path):
    bad = [((2, 4096), POISSON5), ((64, 63), (3.0, -1.0, -1.0, -1.0, -1.0)), ((2, 16), (1.0, 1.0, 1.0, 0.0, 0.0))]
    res = _harness(tmp_path, HARNESS_CASES + bad)
    assert len(res) == len(HARNESS_CASES) + len(bad)
    for (dims, coef), (status, lv, inv) in zip(HARNESS_CASES, res):
        assert status == 0, dims
        small = int(np.prod(dims)) <= 2_000_000
        ref = hierarchy(dims, coef, assemble=small)
        assert len(lv) == len(ref), dims
        dim = len(dims)
        for got, want in zip(lv, ref):
            assert got["dims"] == tuple(want["dims"]) + (1,) * (3 - dim), dims
            scale = max(abs(want["c0"]), max(abs(np.array(want["cm"] + want["cp"]))))
            for key in ("cm", "cp", "e"):
                assert np.abs(np.array(got[key][:dim]) - np.array(want[key])).max() <= 1e-15 * scale, (dims, key)
            assert abs(got["c0"] - want["c0"]) <= 1e-15 * scale, dims
            if "lmax" in want:
                assert abs(got["lmax"] - want["lmax"]) <= 1e-14 * want["lmax"], (dims, got["lmax"], want["lmax"])
        want_inv = ref[-1]["inv"].ravel(order="F")
        assert inv.size == want_inv.size
        assert np.abs(inv - want_inv).max() <= 1e-12 * np.abs(want_inv).max(), dims
    statuses = [r[0] for r in res[len(HARNESS_CASES):]]
    assert statuses == [-2, -2, -2]                            # too large a coarsest grid, a zero centre, a singular matrix


def _dense_M(lev, n, m=2, trans=False):
    return np.column_stack([vcycle(lev, np.eye(n, dtype=complex)[:, j], m, trans) for j in range(n)])


@pytest.mark.parametrize("dims,coef", [((40, 33), POISSON5), ((12, 11, 10), LAPLACE7)])
def test_reference_spd(dims, coef):
    lev = hierarchy(dims, coef)
    assert len(lev) >= 2
    n = int(np.prod(dims))
    for m in (1, 2, 3):
        M = _dense_M(lev, n, m)
        assert np.abs(M.imag).max() == 0.0
        M = M.real
        assert np.abs(M - M.T).max() <= 1e-13 * np.abs(M).max(), m
        assert np.linalg.eigvalsh((M + M.T) / 2).min() > 0, m


def test_reference_hermitian_complex():
    coef = (4.5, -1.0 + 0.3j, -1.0 - 0.3j, -1.0 - 0.2j, -1.0 + 0.2j)           # c+ = conj(c-): Hermitian, and definite
    dims = (34, 31)
    A = stencil_csr(dims, np.array(coef))
    assert abs(A - A.conj().T).max() == 0
    M = _dense_M(hierarchy(dims, coef), int(np.prod(dims)))
    assert np.abs(M - M.conj().T).max() <= 1e-13 * np.abs(M).max()
    assert np.linalg.eigvalsh((M + M.conj().T) / 2).min() > 0


def test_reference_adjoint_convdiff():
    dims = (14, 12, 11)
    lev = hierarchy(dims, CONVDIFF7)
    rng = np.random.default_rng(3)
    n = int(np.prod(dims))
    x, y = rng.standard_normal(n), rng.standard_normal(n)
    lhs = np.vdot(x, vcycle(lev, y.astype(complex)))
    rhs = np.vdot(vcycle(lev, x.astype(complex), trans=True), y)
    assert abs(lhs - rhs) <= 1e-13 * abs(lhs)
    M = _dense_M(lev, n)
    assert np.abs(M - M.T).max() > 1e-3 * np.abs(M).max()                            # not symmetric: the adjoint matters


@pytest.mark.parametrize("dims", [(255, 255), (256, 256), (512, 512), (1024, 768), (63, 63, 63), (64, 64, 64), (96, 96, 96)])
def test_mesh_independent_pcg(dims):
    """scipy cg with the reference V-cycle (m = 2) reaches rtol 1e-8 in <= 8 iterations at every size."""
    coef = POISSON5 if len(dims) == 2 else LAPLACE7
    lev = hierarchy(dims, coef)
    A = stencil_csr(dims, np.array(coef))
    b = np.random.default_rng(0).random(A.shape[0])
    M = spla.LinearOperator(A.shape, matvec=lambda r: vcycle(lev, r.astype(complex)).real)
    it = [0]
    x, info = spla.cg(A, b, rtol=1e-8, M=M, maxiter=100, callback=lambda xk: it.__setitem__(0, it[0] + 1))
    assert info == 0 and it[0] <= 8, (dims, info, it[0])
    assert np.linalg.norm(b - A @ x) <= 1e-8 * np.linalg.norm(b)


def _demangle(names):
    return subprocess.run(["c++filt"], input="\n".join(names), capture_output=True, text=True).stdout.splitlines()


def test_multigrid_kernels_do_not_spill(tmp_path):
    from lightkrylov_b200 import build
    if not os.path.exists(build.NVCC):
        pytest.skip("nvcc not available")
    r = subprocess.run([build.NVCC] + build.FLAGS + ["-Xptxas", "-v", "-c", os.path.join(build.CSRC, "kernels_ops.cu"),
                        "-o", str(tmp_path / "kernels_ops.o")], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr[-2000:]
    seen, cur = {}, None
    for line in r.stderr.splitlines():
        m = re.search(r"Compiling entry function '(\w+)'", line)
        if m:
            cur = _demangle([m.group(1)])[0]
            cur = cur if ("MgStep" in cur or "lkb::k_mg_" in cur) else None
        elif cur and "spill" in line:
            seen[cur] = line
            assert "0 bytes stack frame, 0 bytes spill stores, 0 bytes spill loads" in line, (cur, line)
    count = lambda pat: sum(bool(re.match(pat, n)) for n in seen)                 # noqa: E731
    assert count(r"void lkb::k_mg_restrict<") == 4 and count(r"void lkb::k_mg_prolong<") == 4
    # 4 kinds x (full pack, PW = 1), z has only PW = 1
    assert count(r"void lkb::k_stencil<.*MgStep") == 7 and count(r"void lkb::k_stencil_smem<.*MgStep") == 7
