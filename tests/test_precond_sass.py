"""CPU-side checks of the preconditioner kernels on the built library: the diagonal operator (k_diag) and the diagonal
modes of the CG vector kernels stream with 128-bit L1::no_allocate loads, and none of the new kernels spills."""
import os
import re
import shutil
import subprocess

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def so_path():
    from lightkrylov_b200 import build
    return build.build()


def _demangle(names):
    out = subprocess.run(["c++filt"], input="\n".join(names), capture_output=True, text=True).stdout
    return out.splitlines()


def test_diag_and_jacobi_cg_kernels_use_128bit_streaming_loads(so_path):
    if not shutil.which("cuobjdump") or not shutil.which("c++filt"):
        pytest.skip("cuobjdump not available")
    out = subprocess.run(["cuobjdump", "-sass", so_path], capture_output=True, text=True).stdout
    assert "arch = sm_100a" in out
    chunks = out.split("Function : ")[1:]
    names = _demangle([c.split("\n", 1)[0].strip() for c in chunks])
    body = dict(zip(names, chunks))
    want = {"k_diag": 8, "k_cg_update": 4, "k_cg_direction": 4}     # k_diag: 4 kinds x (d, conj d); CG: the CG_DIAG mode per kind
    for fn, count in want.items():
        pat = re.compile(rf"void lkb::{fn}<\d+, (true|false)>" if fn == "k_diag" else rf"void lkb::{fn}<\d+, 1>")
        hits = [n for n in names if pat.match(n)]
        assert len(hits) == count, (fn, hits)
        for n in hits:
            assert "LDG.E.NA.128" in body[n], n


def test_preconditioner_kernels_do_not_spill(tmp_path):
    from lightkrylov_b200 import build
    if not os.path.exists(build.NVCC):
        pytest.skip("nvcc not available")
    fns = ("k_diag", "k_jacobi", "k_cg_update", "k_cg_direction")
    seen = set()
    for src in ("kernels_vec.cu", "kernels_ops.cu"):
        r = subprocess.run([build.NVCC] + build.FLAGS + ["-Xptxas", "-v", "-c", os.path.join(build.CSRC, src),
                            "-o", str(tmp_path / src.replace(".cu", ".o"))], capture_output=True, text=True)
        assert r.returncode == 0, r.stderr[-2000:]
        cur = None
        for line in r.stderr.splitlines():
            m = re.search(r"Compiling entry function '(\w+)'", line)
            if m:
                cur = _demangle([m.group(1)])[0]
                cur = cur if any(f"lkb::{f}<" in cur for f in fns) else None
            elif cur and "spill" in line:
                seen.add(cur)
                assert "0 bytes spill stores, 0 bytes spill loads" in line, (cur, line)
    assert sum("k_diag" in n for n in seen) == 8 and sum("k_jacobi" in n for n in seen) == 20
    assert sum("k_cg_update" in n for n in seen) == 12 and sum("k_cg_direction" in n for n in seen) == 8
