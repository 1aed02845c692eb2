"""CPU checks of the GMRES-polynomial preconditioner: the product recurrence of tests/poly_cases.py against the closed form
p(A) = A^-1 (I - prod (I - A/theta_i)), the library's root construction (lkb_poly.cu: gmres_poly_roots, through a host
harness that links liblkb.so) against the numpy reference, and the new kernels on the built library (128-bit streaming loads
in k_poly_update, no spills in k_poly_update and the PolyStep stencil kernels)."""
import glob
import os
import re
import shutil
import subprocess

import numpy as np
import pytest

from poly_cases import extra_copies, gmres_poly_roots, harmonic_ritz, hessenberg_case, poly_apply, poly_closed_form

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "lightkrylov_b200", "csrc")
NVCC = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")


def _matrix(n, cplx, seed):
    """A nonsymmetric matrix with its spectrum in the right half plane around 1 (complex for the real kinds too)."""
    rng = np.random.default_rng(seed)
    X = rng.standard_normal((n, n)) + (1j * rng.standard_normal((n, n)) if cplx else 0)
    return np.eye(n) + 0.35 * X / np.sqrt(n)


ROOT_SETS = {
    "real": [1.6, 0.5, 1.2, 0.8, 1.9, 0.65, 1.4],
    "pair_last": [1.5, 0.7, 1.1 + 0.4j, 1.1 - 0.4j],
    "real_last": [0.9 + 0.5j, 0.9 - 0.5j, 1.7, 0.6 - 0.3j, 0.6 + 0.3j, 1.3],
    "pairs_only": [1.2 + 0.6j, 1.2 - 0.6j, 0.7 + 0.2j, 0.7 - 0.2j],
    "single": [1.1],
    "long": list(np.linspace(0.45, 1.75, 9)) + [1.0 + 0.5j, 1.0 - 0.5j, 1.3 + 0.3j, 1.3 - 0.3j, 0.7 + 0.35j, 0.7 - 0.35j, 1.55],
}


@pytest.mark.parametrize("cplx", [False, True])
@pytest.mark.parametrize("name", sorted(ROOT_SETS))
def test_recurrence_matches_closed_form(oracle, cplx, name):
    roots = np.array(ROOT_SETS[name], dtype=np.complex128)
    assert roots.size <= 16
    if cplx:                                  # complex kinds: any roots, in any order
        roots = roots * np.exp(0.2j)
    n = 30
    A = _matrix(n, cplx, 7 + roots.size)
    Ao = oracle.Op.dense(np.asfortranarray(A))
    Mc = poly_closed_form(A, roots)
    R = np.eye(n, dtype=A.dtype)
    Mr = np.column_stack([poly_apply(Ao, roots, R[:, j].copy()) for j in range(n)])
    assert np.abs(Mr - Mc).max() <= 1e-12 * np.abs(Mc).max(), name
    MrH = np.column_stack([poly_apply(Ao, roots, R[:, j].copy(), trans=True) for j in range(n)])
    assert np.abs(MrH - Mc.conj().T).max() <= 1e-12 * np.abs(Mc).max(), name
    # A M = I - pi(A)
    P = np.eye(n, dtype=np.complex128)
    for t in roots:
        P = P @ (np.eye(n) - A / t)
    assert np.abs(A @ Mr - (np.eye(n) - P)).max() <= 1e-12 * max(1.0, np.abs(P).max())


def test_recurrence_counts_applications():
    """d - 1 applications of A, whatever the mix of roots and pairs."""
    for name, roots in ROOT_SETS.items():
        calls = []
        poly_apply(lambda x: (calls.append(1), 2.0 * x)[1], roots, np.ones(5))
        assert len(calls) == len(roots) - 1, name


def _cases():
    """(name, kind, H, k): real spectrum, complex pairs, a complex kind, a breakdown-sized H and an outlier."""
    yield "real", "d", hessenberg_case([2.0, 1.5, 1.1, 0.8, 0.6, 0.45, 0.3, 0.2], 1), 8
    yield "pairs", "d", hessenberg_case([1 + 1j, 1 - 1j, 2.0, 0.5 + 0.25j, 0.5 - 0.25j, 3.0, 1.5 + 2j, 1.5 - 2j, 0.7, 2.5], 2), 10
    yield "pairs_s", "s", hessenberg_case([1 + 0.6j, 1 - 0.6j, 2.2, 0.4, 1.7 + 0.3j, 1.7 - 0.3j], 3), 6
    yield "complex", "z", hessenberg_case([1 + 1j, 2 - 0.5j, 0.3 + 0.1j, -1 + 2j, 1.5j, 0.8 - 0.9j, 2.5 + 0.2j], 4, cplx=True), 7
    yield "complex_c", "c", hessenberg_case([1 + 0.2j, 0.5 - 0.5j, 2j, 1.2 - 1j], 5, cplx=True), 4
    yield "breakdown", "d", hessenberg_case([3.0, 1.0, 2.0], 6, hk1=1e-17), 3
    yield "outlier", "d", hessenberg_case([1.0, 1.1, 1.25, 1.4, 1.55, 1.7, 1.85, 2.0, 400.0], 7), 9
    yield "outlier_pair", "d", hessenberg_case([1.0, 1.2, 1.4, 1.6, 1.8, 2.0, 2.2, 300 + 50j, 300 - 50j], 8), 9


def _run_harness(tmp_path, cases):
    import scipy
    import __graft_entry__
    __graft_entry__.build()
    exe = str(tmp_path / "host_poly_harness")
    nvcc = NVCC if os.path.exists(NVCC) else shutil.which("nvcc")
    subprocess.check_call([nvcc, "-gencode", "arch=compute_100a,code=sm_100a", "-O1", "-std=c++17", "-I", CSRC,
                           os.path.join(ROOT, "tests", "host_poly_harness.cu"), "-o", exe, "-L", CSRC, "-llkb", "-ldl",
                           "-Xlinker", "-rpath=" + CSRC])
    blas = glob.glob(os.path.join(os.path.dirname(os.path.dirname(scipy.__file__)), "scipy.libs", "libscipy_openblas*.so"))[0]
    text = ""
    for kind, H, k in cases:
        text += f"{kind} {k}\n" + "\n".join(f"{float(v.real)!r} {float(v.imag)!r}" for v in H.ravel(order="F")) + "\n"
    out = subprocess.run([exe, blas], input=text, check=True, capture_output=True, text=True).stdout.splitlines()
    res, i = [], 0
    while i < len(out):
        _, status, count = out[i].split()
        vals = [complex(float(a), float(b)) for a, b in (ln.split() for ln in out[i + 1:i + 1 + int(count)])]
        res.append((int(status), np.array(vals, dtype=np.complex128)))
        i += 1 + int(count)
    return res


@pytest.mark.skipif(not os.path.exists(NVCC) and shutil.which("nvcc") is None, reason="needs nvcc to compile the harness")
def test_library_roots_match_reference(tmp_path):
    cases = list(_cases())
    res = _run_harness(tmp_path, [(kind, H, k) for _, kind, H, k in cases] +
                       [("d", np.triu(np.ones((5, 4)), -1) * np.r_[[[1, 1, 1, 1]] * 4, [[0, 0, 0, 1]]], 4)])   # singular H_k
    assert len(res) == len(cases) + 1
    extras = {}
    for (name, kind, H, k), (status, got) in zip(cases, res):
        cplx = kind in "cz"
        ref = gmres_poly_roots(H, k, cplx)
        assert status == 0, name
        assert got.size == ref.size, (name, got, ref)
        assert np.abs(got - ref).max() <= 1e-10 * np.abs(ref).max(), (name, got, ref)      # same values, same order
        if not cplx:                                      # pairs adjacent, im > 0 first, exact conjugates
            i = 0
            while i < got.size:
                if got[i].imag != 0.0:
                    assert got[i].imag > 0.0 and got[i + 1] == np.conj(got[i]), (name, got)
                    i += 1
                i += 1
        assert np.abs(got[0]) == np.abs(got).max(), name
        extras[name] = got.size - k
        assert extras[name] == sum(extra_copies(harmonic_ritz(H, k, cplx), cplx)), name
    assert extras["outlier"] >= 1 and extras["outlier_pair"] >= 2 and extras["real"] == 0, extras
    brk = res[len(cases) - 3][1]
    assert np.allclose(np.sort(brk.real), [1.0, 2.0, 3.0], rtol=1e-12, atol=0) and np.all(brk.imag == 0), brk
    assert res[-1][0] == -2 and res[-1][1].size == 0                              # singular H_k: LKB_ERR_ARG


@pytest.fixture(scope="module")
def so_path():
    from lightkrylov_b200 import build
    return build.build()


def _demangle(names):
    return subprocess.run(["c++filt"], input="\n".join(names), capture_output=True, text=True).stdout.splitlines()


def test_poly_update_uses_128bit_streaming_loads(so_path):
    if not shutil.which("cuobjdump") or not shutil.which("c++filt"):
        pytest.skip("cuobjdump not available")
    out = subprocess.run(["cuobjdump", "-sass", so_path], capture_output=True, text=True).stdout
    chunks = out.split("Function : ")[1:]
    names = _demangle([c.split("\n", 1)[0].strip() for c in chunks])
    hits = [(n, c) for n, c in zip(names, chunks) if n.startswith("void lkb::k_poly_update<")]
    assert len(hits) == 4, [n for n, _ in hits]
    for n, body in hits:
        assert "LDG.E.NA.128" in body, n


def test_poly_kernels_do_not_spill(tmp_path):
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
                cur = cur if ("lkb::k_poly_update<" in cur or "PolyStep" in cur) else None
            elif cur and "spill" in line:
                seen[cur] = line
                if cur.startswith("void lkb::k_stencil<1, 1, lkb::PolyStep<double> >"):
                    # the 3-D fp64 kernel for rows whose length is odd: ptxas keeps one 16-byte value in local memory
                    m = re.search(r"(\d+) bytes spill stores", line)
                    assert m and int(m.group(1)) <= 24, (cur, line)
                    continue
                assert "0 bytes spill stores, 0 bytes spill loads" in line, (cur, line)
    count = lambda pat: sum(bool(re.match(pat, n)) for n in seen)                 # noqa: E731
    assert count(r"void lkb::k_poly_update<") == 4
    # 4 kinds x (full pack, PW = 1), z has only PW = 1
    assert count(r"void lkb::k_stencil<.*PolyStep") == 7 and count(r"void lkb::k_stencil_smem<.*PolyStep") == 7
