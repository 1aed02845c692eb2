"""Every raw CUDA resource of the library has one owner (lkb_internal.h: Owner and its aliases): the calls that allocate or
release one appear only in the allocation helper and the owners' release functions, plus a short list of sites that manage
memory on their own terms.  A hand-written cudaFree anywhere else is a second release path, which is how leaks and double
frees on failed creation come back."""
import os
import re

CSRC = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "lightkrylov_b200", "csrc")

CALLS = re.compile(r"\b(cudaMalloc|cudaMallocHost|cudaFree|cudaFreeHost|cudaIpcCloseMemHandle|cudaGraphExecDestroy|cudaStreamDestroy|"
                   r"CommDestroy)\s*\(")
ALLOWED = {
    "cuda_alloc",        # the allocation helper that fills an owner
    "comm_destroy",      # the communicator owner's release function
    "lkb_dev_free",      # C ABI: releases arrays that lkb_csr_random_device handed to the caller
    "StepSlots",         # pinned staging slots of the eigensolvers, released after a stream synchronisation
    "dev_alloc", "dev_free",   # the stream-ordered pool of vectors, bases and solver work space
}


def _strip_comments(src):
    """Comments become blanks; string literals are kept (a '//' inside one is not a comment)."""
    pat = re.compile(r'//[^\n]*|/\*.*?\*/|"(?:\\.|[^"\\\n])*"', re.S)
    return pat.sub(lambda m: m.group(0) if m.group(0).startswith('"') else re.sub(r"[^\n]", " ", m.group(0)), src)


def _enclosing_names(src, pos):
    """Names of the functions / classes whose bodies contain `pos`, innermost last."""
    stack = []
    for i, ch in enumerate(src[:pos]):
        if ch == "{":
            head = src[max(src.rfind(";", 0, i), src.rfind("}", 0, i), src.rfind("{", 0, i)) + 1:i]
            m = re.search(r"(\w+)\s*\(", head) or re.search(r"\b(?:struct|class)\s+(\w+)", head)
            stack.append(m.group(1) if m else "")
        elif ch == "}" and stack:
            stack.pop()
    return stack


def _violations(path):
    src = _strip_comments(open(path).read())
    out = []
    for m in CALLS.finditer(src):
        names = _enclosing_names(src, m.start())
        if not ALLOWED.intersection(names):
            line = src.count("\n", 0, m.start()) + 1
            out.append(f"{os.path.basename(path)}:{line}: {m.group(1)} in {'::'.join(n for n in names if n) or 'file scope'}")
    return out


def test_cuda_resources_are_released_only_by_their_owners():
    files = sorted(f for f in os.listdir(CSRC) if f.endswith((".cu", ".h", ".cuh")))
    assert "lkb_core.cu" in files and "lkb_internal.h" in files
    bad = [v for f in files for v in _violations(os.path.join(CSRC, f))]
    assert not bad, "raw CUDA allocation / release outside the owners:\n" + "\n".join(bad)


def test_checker_sees_a_hand_written_release(tmp_path):
    p = tmp_path / "x.cu"
    p.write_text("// cudaFree(p) in a comment is fine\n"
                 "int cuda_alloc(void** p) { return cudaMalloc(p, 16); }\n"
                 "struct S { void f() { if (q) { cudaFree(q); } } };\n"
                 "int g() { cudaStreamDestroy(s); nccl_api()->CommDestroy(c); }\n")
    assert [v.split(": ", 1)[1] for v in _violations(str(p))] == [
        "cudaFree in S::f::if", "cudaStreamDestroy in g", "CommDestroy in g"]
