"""CPU-side checks of the drop-in boundary: the C-ABI library loads, exports every symbol that
include/lkb.h declares, the ctypes table covers them all, and the product fails loudly (no CPU
fallback) when no CUDA device is present."""
import ctypes
import os
import re

import pytest

from oracle import ref_exec

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _declared_symbols():
    src = open(os.path.join(ROOT, "include", "lkb.h")).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    names = set(re.findall(r"\b(lkb_[a-z0-9_]+)\s*\(", src))
    names -= {"lkb_matvec_fn"}
    return sorted(names)


@pytest.fixture(scope="module")
def so_path():
    from lightkrylov_b200 import build
    return build.build()


def test_header_symbols_are_exported(so_path):
    lib = ctypes.CDLL(so_path)
    syms = _declared_symbols()
    assert len(syms) >= 60
    missing = [s for s in syms if not hasattr(lib, s)]
    assert not missing, f"declared in include/lkb.h but not exported: {missing}"


def test_ctypes_table_matches_header(so_path):
    from lightkrylov_b200 import _lib
    assert sorted(_lib.SIGNATURES) == _declared_symbols()
    _lib.load()


def test_no_cpu_fallback(so_path):
    """Without a GPU every entry point must fail loudly; nothing may silently run on the CPU."""
    import torch
    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    import lightkrylov_b200 as lk
    with pytest.raises(lk.LkbError, match="no CUDA device"):
        lk.Context(0)


def test_product_never_imports_oracle():
    """oracle/ is test infrastructure: the package and the CUDA sources must not reference it."""
    pkg = os.path.join(ROOT, "lightkrylov_b200")
    for dp, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h", ".cpp")):
                txt = open(os.path.join(dp, f), errors="replace").read()
                assert "lk_oracle" not in txt and "liblk_oracle" not in txt and "from oracle" not in txt, f


def test_sass_has_128bit_loads(so_path):
    """The GS kernels must move data with 128-bit loads, checked on the built cubin: LDG.E.NA.128[.CONSTANT] since round 2
    (NA = L1::no_allocate streaming loads), LDG.E.128 before."""
    import shutil, subprocess
    if not shutil.which("cuobjdump"):
        pytest.skip("cuobjdump not available")
    out = subprocess.run(["cuobjdump", "-sass", so_path], capture_output=True, text=True).stdout
    assert "arch = sm_100a" in out
    # per-function check: the multi-dot and multi-axpy kernels stream with LDG.E.128
    for fn in ("k_multidot", "k_multiaxpy"):
        chunks = [c for c in out.split("Function : ")[1:] if fn in c.split("\n", 1)[0]]
        assert chunks, fn
        assert all(("LDG.E.NA.128" in c) or ("LDG.E.128" in c) for c in chunks), fn
    assert "LDG.E.NA.128.CONSTANT" in out          # the streaming loads do not allocate in L1
    assert "ACQBULK" in out and "PREEXIT" in out   # griddepcontrol.wait / launch_dependents (programmatic dependent launch)


def _build_c_demo(so_path, tmp_path):
    import subprocess
    exe = str(tmp_path / "c_abi_demo")
    libdir = os.path.dirname(so_path)
    subprocess.check_call(["gcc", "-std=c99", "-Wall", "-Werror", "-I" + os.path.join(ROOT, "include"),
                           os.path.join(ROOT, "examples", "c_abi_demo.c"), "-L" + libdir, "-llkb",
                           "-Wl,-rpath," + libdir, "-lm", "-o", exe])
    return exe


def test_header_is_plain_c_and_links(so_path, tmp_path):
    """include/lkb.h must compile as C99 and a C client must link against liblkb.so (no C++/torch types)."""
    import subprocess
    exe = _build_c_demo(so_path, tmp_path)
    import torch
    if not torch.cuda.is_available():
        r = subprocess.run([exe, "64"], capture_output=True, text=True)
        assert r.returncode == 2 and "no CUDA device" in r.stderr      # loud failure, no CPU fallback


@pytest.mark.gpu
def test_c_client_runs_on_gpu(so_path, tmp_path):
    import subprocess
    exe = _build_c_demo(so_path, tmp_path)
    r = subprocess.run([exe, "1024"], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stdout + r.stderr
    assert "info=0" in r.stdout


def _c_prototypes():
    """name -> list of (is_pointer, base type) for every function declared in include/lkb.h."""
    src = open(os.path.join(ROOT, "include", "lkb.h")).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    protos = {}
    for m in re.finditer(r"\b(lkb_[a-z0-9_]+)\s*\(([^;{]*?)\)\s*;", src, flags=re.S):
        name, args = m.group(1), " ".join(m.group(2).split())
        if name in ("lkb_matvec_fn", "lkb_precond_fn"):
            continue
        params = []
        if args and args != "void":
            for a in args.split(","):
                a = a.strip()
                is_ptr = "*" in a
                base = re.sub(r"\bconst\b", "", a).replace("*", " ")
                base = " ".join(base.split()[:-1]) if len(base.split()) > 1 else base.strip()
                params.append((is_ptr, base))
        protos[name] = params
    return protos


HANDLES = {"lkb_ctx_t", "lkb_vec_t", "lkb_basis_t", "lkb_op_t"}
FWIDTH = {"int": "c_int", "int32_t": "c_int32_t", "int64_t": "c_int64_t", "uint64_t": "c_int64_t", "double": "c_double"}


def test_fortran_shim_interfaces_match_header(so_path):
    """The ISO_C_BINDING shim cannot be compiled here (no Fortran compiler, also not on the GPU box), so every bind(C)
    interface of the generated module is checked against the C prototypes of include/lkb.h: the symbol is exported, the
    argument COUNT agrees, and every argument agrees in by-value-ness and width: a C scalar / handle / function pointer
    must be `value` with the matching c_* kind; a C pointer is either `type(c_ptr), value` or a by-reference dummy."""
    import subprocess, sys
    subprocess.check_call([sys.executable, os.path.join(ROOT, "fortran", "gen_shim.py")], stdout=subprocess.DEVNULL)
    raw = open(os.path.join(ROOT, "fortran", "lightkrylov_cuda.f90")).read()
    assert max(len(ln) for ln in raw.splitlines()) <= 132, "free-form Fortran lines are limited to 132 columns"
    src = re.sub(r"&[ \t]*\n[ \t]*", "", raw)                      # join continuation lines
    protos = _c_prototypes()
    lib = ctypes.CDLL(so_path)
    blocks = re.findall(r"function (lkb_[a-z0-9_]+)\(([^)]*)\) bind\(C, name='(lkb_[a-z0-9_]+)'\)(.*?)end function", src, flags=re.S)
    assert len(blocks) >= 40
    for fname, dummies, cname, body in blocks:
        assert fname == cname and hasattr(lib, cname), cname
        cparams = protos[cname]
        names = [d.strip() for d in dummies.split(",") if d.strip()]
        assert len(names) == len(cparams), f"{cname}: {len(names)} Fortran arguments vs {len(cparams)} in lkb.h"
        decl = {}
        for line in body.splitlines():
            if "::" in line:
                left, right = line.split("::")
                for nm in right.split(","):
                    decl[nm.strip()] = left.strip()
        for nm, (is_ptr, base) in zip(names, cparams):
            d = decl[nm]
            by_value = "value" in d
            if base in ("lkb_matvec_fn", "lkb_precond_fn"):
                assert d.startswith("type(c_funptr)") and by_value, (cname, nm, d)
            elif base in HANDLES and not is_ptr:
                assert d.startswith("type(c_ptr)") and by_value, (cname, nm, d)
            elif not is_ptr:
                assert by_value and FWIDTH[base] in d, (cname, nm, d, base)
            else:
                # pointer in C: address passed by value, or a by-reference dummy of the pointee's width
                if d.startswith("type(c_ptr)"):
                    assert by_value or "intent(out)" in d, (cname, nm, d)
                    if "intent(out)" in d:
                        assert base in HANDLES, (cname, nm, d, base)          # handle out-argument (T* where T is a handle)
                else:
                    assert not by_value and FWIDTH.get(base, "?") in d, (cname, nm, d, base)
    # the try-functions exist for all four kinds with the reference's argument lists
    for sfx in ("rsp", "rdp", "csp", "cdp"):
        for fn, args in (("arnoldi", "A, X, H, info, kstart, kend, tol, transpose, blksize"), ("lanczos", "A, X, T, info, kstart, kend, tol"),
                         ("bidiagonalization", "A, U, V, B, info, kstart, kend, tol"), ("qr", "Q, R, info, tol"),
                         ("gmres", "A, b, x, info, rtol, atol, preconditioner, options, transpose, meta"),
                         ("fgmres", "A, b, x, info, rtol, atol, preconditioner, options, transpose, meta"),
                         ("cg", "A, b, x, info, rtol, atol, preconditioner, options, meta"),
                         ("eigs", "A, X, eigvals, residuals, info, x0, kdim, tolerance, transpose, write_intermediate"),
                         ("eighs", "A, X, eigvals, residuals, info, x0, kdim, tolerance, write_intermediate"),
                         ("svds", "A, U, S, V, residuals, info, u0, kdim, tolerance, write_intermediate"),
                         ("dgs_vector", "y, X, info, if_chk_orthonormal, beta"), ("dgs_basis", "Y, X, info, if_chk_orthonormal, beta"),
                         ("orthogonalize_vector", "y, X, info, if_chk_orthonormal, beta"),
                         ("orthogonalize_basis", "Y, X, info, if_chk_orthonormal, beta"),
                         ("qr_pivoting", "Q, R, perm, info, tol"), ("kexpm_vec", "c, A, b, tau, tol, info, trans, kdim"),
                         ("kexpm_mat", "C, A, B, tau, tol, info, trans, kdim"),
                         ("krylov_exptA", "vec_out, A, vec_in, tau, info, trans")):
            assert f"function lkb_try_{fn}_{sfx}({args}) result(done)" in src, (fn, sfx)
    # no component of the device vector is default-initialised (intent(out) dummies must not reset the handle)
    for sfx in ("rsp", "rdp", "csp", "cdp"):
        tdef = src[src.index(f":: cuda_vector_{sfx}\n"):]
        tdef = tdef[:tdef.index("contains")]
        assert "=" not in tdef.replace("=>", ""), tdef


def _strip_fortran_comment(line):
    q = None
    for i, ch in enumerate(line):
        if q:
            if ch == q:
                q = None
        elif ch in "'\"":
            q = ch
        elif ch == "!":
            return line[:i]
    return line


def _fortran_block_lint(raw):
    """Returns the number of block constructs; raises AssertionError on an unmatched / mismatched / unclosed construct."""
    lines = [_strip_fortran_comment(ln).rstrip() for ln in raw.splitlines()]
    joined, cur = [], ""
    for ln in lines:
        if not ln.strip():
            continue
        if ln.endswith("&"):
            cur += ln[:-1].strip() + " "
            continue
        joined.append((cur + ln.strip()).lower()); cur = ""
    assert cur == "", "dangling continuation at the end of the file"
    openers = [
        ("module", re.compile(r"^module (?!procedure)\w+$")),
        ("function", re.compile(r"^(\w+(\([\w=, ]+\))? )*function \w+ ?\(")),
        ("subroutine", re.compile(r"^((pure|elemental|recursive|impure) )*subroutine \w+")),
        ("interface", re.compile(r"^(abstract )?interface( \w+)?$")),
        ("type", re.compile(r"^type(,[^:]*)? :: \w+$|^type \w+$")),
        ("select", re.compile(r"^select (type|case) ?\(")),
        ("if", re.compile(r"^if ?\(.*\) ?then$")),
        ("do", re.compile(r"^do( |$)")),
        ("block", re.compile(r"^block$")),
    ]
    ender = re.compile(r"^end ?(module|function|subroutine|interface|type|select|if|do|block)\b")
    stack, n_blocks = [], 0
    for ln in joined:
        m = ender.match(ln)
        if m:
            assert stack, "unmatched: " + ln
            kind, opened = stack.pop()
            assert kind == m.group(1), f"`{ln}` closes `{opened}`"
            continue
        assert not ln.startswith("end "), "unknown end statement: " + ln
        for kind, rx in openers:
            if rx.match(ln):
                stack.append((kind, ln)); n_blocks += 1
                break
    assert not stack, "left open: " + repr(stack[-3:])
    return n_blocks


def test_fortran_shim_block_structure():
    """No Fortran compiler exists here or on the GPU box, so the generated module is at least checked mechanically for
    well-formedness: every module / function / subroutine / interface / type / select / if-then / do / block construct is
    closed by the matching `end`, in order, and nothing is left open; continuation lines are well-formed.  The linter itself
    is checked on mutated copies (a dropped `end if`, a dropped `end select`, a swapped `end function`)."""
    import subprocess, sys
    subprocess.check_call([sys.executable, os.path.join(ROOT, "fortran", "gen_shim.py")], stdout=subprocess.DEVNULL)
    raw = open(os.path.join(ROOT, "fortran", "lightkrylov_cuda.f90")).read()
    assert _fortran_block_lint(raw) > 400          # 4 kinds x (types, TBPs, try-functions) + ~58 bind(C) interfaces
    for victim, repl in (("            end if\n", "\n"), ("            end select\n", "\n"), ("    end function\n", "    end subroutine\n")):
        assert victim in raw
        with pytest.raises(AssertionError):
            _fortran_block_lint(raw.replace(victim, repl, 1))


def _shim_code_without_comments():
    raw = open(os.path.join(ROOT, "fortran", "lightkrylov_cuda.f90")).read()
    src = re.sub(r"&[ \t]*\n[ \t]*", "", raw)
    return "\n".join(_strip_fortran_comment(ln) for ln in src.splitlines())


def _call_arg_counts(code, name):
    """number of top-level arguments of every `name(...)` reference in `code` (balanced parentheses, literals skipped)"""
    counts = []
    for m in re.finditer(r"\b" + re.escape(name) + r"\s*\(", code):
        i, depth, nargs, q, empty = m.end(), 1, 1, None, True
        while depth:
            ch = code[i]
            if q:
                if ch == q:
                    q = None
            elif ch in "'\"":
                q = ch; empty = False
            elif ch == "(":
                depth += 1; empty = False
            elif ch == ")":
                depth -= 1
            elif ch == "," and depth == 1:
                nargs += 1
            elif not ch.isspace():
                empty = False
            i += 1
        counts.append(0 if empty else nargs)
    return counts


def test_fortran_shim_calls_match_interfaces():
    """Every liblkb entry point the shim calls is declared in its bind(C) interface block, and every call passes exactly
    as many arguments as the interface (= include/lkb.h, checked above) declares."""
    import subprocess, sys
    subprocess.check_call([sys.executable, os.path.join(ROOT, "fortran", "gen_shim.py")], stdout=subprocess.DEVNULL)
    code = _shim_code_without_comments()
    iface = {m.group(1): len([d for d in m.group(2).split(",") if d.strip()])
             for m in re.finditer(r"function (lkb_[a-z0-9_]+)\(([^)]*)\) bind\(C", code)}
    defined = set(re.findall(r"(?:function|subroutine) (lkb_\w+)", code))
    used = set(re.findall(r"\b(lkb_[A-Za-z0-9_]+)\s*\(", re.sub(r"'[^']*'", "", code)))
    assert not (used - set(iface) - defined), sorted(used - set(iface) - defined)
    n_calls = 0
    nolit = re.sub(r"'[^']*'", "''", code)                   # 'lkb_vec_axpby(copy)' is a message, not a call
    for name, nargs in iface.items():
        counts = _call_arg_counts(nolit, name)
        assert counts, name                                     # at least the declaration itself
        for c in counts:
            assert c == nargs, f"{name}: a reference passes {c} arguments, the interface declares {nargs}"
        n_calls += len(counts) - 1
    assert n_calls > 200


_F_KEYWORDS = set("""if then else elseif end endif do enddo call return select type class is case default function subroutine result
contains module use only implicit none external intrinsic integer real complex logical character len kind intent in out inout optional
target pointer allocatable value import interface procedure pass public private save parameter bind c name allocate deallocate present
size int cmplx merge max min abs sqrt aimag conjg true false and or not eq ne lt gt le ge error stop source mold stat block associated
extends abstract generic assignment null trim shape reshape allocated exit cycle while contiguous transfer ubound lbound
c_loc c_funloc c_associated c_null_ptr c_null_char c_null_funptr c_ptr c_funptr c_int c_int32_t c_int64_t c_double c_float c_char c_f_pointer
sp dp""".split())


def _fortran_undeclared(code):
    """identifiers used in executable statements that are neither dummies, locals, results, module-level entities, `use`d names
    nor keywords / intrinsics: [(procedure, identifier, statement)]"""
    lines = code.splitlines()
    text = "\n".join(lines)
    module_level = set(m.lower() for m in re.findall(r"^[ \t]*(?!end\b)(?:[\w()=, ]+ )?(?:function|subroutine)[ \t]+(\w+)", text, flags=re.M | re.I))
    module_level |= set(m.lower() for m in re.findall(r"^[ \t]*type(?:[ \t]*,[^:\n]*)?[ \t]*::[ \t]*(\w+)", text, flags=re.M | re.I))
    for m in re.finditer(r"^[ \t]*use[ \t]+[\w, :]*only[ \t]*:(.*)$", text, flags=re.M | re.I):
        module_level |= set(w.lower() for w in re.findall(r"\w+", m.group(1)))
    proc_re = re.compile(r"^\s*(?:[\w()=, ]+\s)?(function|subroutine)\s+(\w+)\s*\(([^)]*)\)(?:\s*result\s*\((\w+)\))?", re.I)

    def declared_names(decl_lines):
        names = set()
        for b in decl_lines:
            right = b.split("::", 1)[1]
            for _ in range(3):
                right = re.sub(r"\([^()]*\)", "", right)                       # drop dimensions / initialisers' call parentheses
            for part in right.split(","):
                nm = part.split("=")[0].strip()
                if re.fullmatch(r"\w+", nm):
                    names.add(nm.lower())
        return names

    # module-level variables / parameters: declarations outside any procedure and outside derived-type definitions
    depth_proc, in_type, in_iface, mod_decls = 0, False, False, []
    i, procs = 0, []
    while i < len(lines):
        ls = lines[i].strip().lower()
        if re.match(r"^(abstract\s+)?interface\b", ls):
            in_iface = True
        elif ls.startswith("end interface"):
            in_iface = False
        m = proc_re.match(lines[i])
        if m and not ls.startswith("end") and not in_iface:
            j = i + 1
            while not re.match(r"^\s*end (function|subroutine)", lines[j], re.I):
                j += 1
            procs.append((m, lines[i + 1:j])); i = j + 1
            continue
        if re.match(r"^type(\s*,[^:]*)?\s*::\s*\w+$", ls):
            in_type = True
        elif ls.startswith("end type"):
            in_type = False
        elif "::" in ls and not in_type and not in_iface:
            mod_decls.append(lines[i])
        i += 1
    module_level |= declared_names(mod_decls)
    assert len(procs) > 150 and {"lkb_ctx", "lkb_magic", "this_module"} <= module_level

    problems = []
    for m, body in procs:
        known = {a.strip().lower() for a in m.group(3).split(",") if a.strip()} | {m.group(2).lower()}
        if m.group(4):
            known.add(m.group(4).lower())
        known |= declared_names([b for b in body if "::" in b])
        # Fortran is case-insensitive: a local that differs from a dummy (or another local) only by case is a duplicate declaration
        seen = {}
        for b in body:
            if "::" in b:
                for nm in declared_names([b]):
                    if nm in seen:
                        problems.append((m.group(2), nm, "declared twice: `%s` and `%s`" % (seen[nm].strip()[:60], b.strip()[:60])))
                    seen[nm] = b
        for b in body:
            if "::" in b:
                continue
            t = re.sub(r"%\s*\w+", "", b)                                          # component references
            t = re.sub(r"([(,]\s*)\w+\s*=(?!=)", r"\1", t)                         # keyword arguments
            t = re.sub(r"(?<![\w.])\d+(\.\d*)?([ed][+-]?\d+)?(_\w+)?", "", t, flags=re.I)   # literals with kind suffixes
            t = re.sub(r"\.\w+\.", " ", t)                                         # .true. .and. ...
            for tok in re.findall(r"[A-Za-z_]\w*", t):
                tl = tok.lower()
                if tl in _F_KEYWORDS or tl in known or tl in module_level:
                    continue
                problems.append((m.group(2), tok, b.strip()[:100]))
    return problems


def test_fortran_shim_identifiers_are_declared():
    """`implicit none` in a module nobody can compile here: every identifier used in the executable part of a procedure must be a
    dummy argument, a local declaration, the function result, a module-level entity (procedure, type, parameter, variable, bind(C)
    interface), a name imported by `use ..., only:`, or a Fortran keyword / intrinsic.  Catches typos and forgotten declarations;
    the checker itself is checked on a copy with one local declaration removed and on one with a misspelt call."""
    import subprocess, sys
    subprocess.check_call([sys.executable, os.path.join(ROOT, "fortran", "gen_shim.py")], stdout=subprocess.DEVNULL)
    code = re.sub(r"'[^']*'", "''", _shim_code_without_comments())
    assert _fortran_undeclared(code) == []
    victim = "        integer(c_int32_t) :: kd, tr, cinfo\n"
    assert victim in code
    bad = _fortran_undeclared(code.replace(victim, "        integer(c_int32_t) :: kd, cinfo\n", 1))
    assert bad and all(p[1] == "tr" for p in bad)
    bad = _fortran_undeclared(code.replace("call chk(lkb_vec_zero(", "call chk(lkb_vec_zer0(", 1))
    assert [p[1] for p in bad] == ["lkb_vec_zer0"]


REFERENCE = os.path.join(ref_exec.REF, "src")      # the LightKrylov checkout the interpreter tests use ($LK_REFERENCE)
_REF_ROUTINES = {          # try-function -> (reference file, reference routine)
    "arnoldi": ("Krylov/BaseKrylov.fypp", "arnoldi"), "lanczos": ("Krylov/BaseKrylov.fypp", "lanczos_tridiagonalization"),
    "bidiagonalization": ("Krylov/BaseKrylov.fypp", "lanczos_bidiagonalization"), "qr": ("Krylov/BaseKrylov.fypp", "qr_no_pivoting"),
    "qr_pivoting": ("Krylov/BaseKrylov.fypp", "qr_with_pivoting"),
    "orthogonalize_vector": ("Krylov/BaseKrylov.fypp", "orthogonalize_vector_against_basis"),
    "orthogonalize_basis": ("Krylov/BaseKrylov.fypp", "orthogonalize_basis_against_basis"),
    "dgs_vector": ("Krylov/BaseKrylov.fypp", "DGS_vector_against_basis"), "dgs_basis": ("Krylov/BaseKrylov.fypp", "DGS_basis_against_basis"),
    "gmres": ("IterativeSolvers/IterativeSolvers.fypp", "gmres"), "fgmres": ("IterativeSolvers/IterativeSolvers.fypp", "fgmres"),
    "cg": ("IterativeSolvers/IterativeSolvers.fypp", "cg"), "eigs": ("IterativeSolvers/IterativeSolvers.fypp", "eigs"),
    "eighs": ("IterativeSolvers/IterativeSolvers.fypp", "eighs"), "svds": ("IterativeSolvers/IterativeSolvers.fypp", "svds"),
    "kexpm_vec": ("Expm/ExpmLib.fypp", "kexpm_vec"), "kexpm_mat": ("Expm/ExpmLib.fypp", "kexpm_mat"),
    "krylov_exptA": ("Expm/ExpmLib.fypp", "krylov_exptA"),
}


def _dummy_attributes(header_and_body, names):
    """{dummy: (base type keyword, optional?, rank)} from the declaration lines of a procedure"""
    out = {}
    for ln in header_and_body:
        if "::" not in ln:
            continue
        left, right = ln.split("::", 1)
        left = left.strip().lower()
        base = re.match(r"[a-z]+", left).group(0)
        for _ in range(3):
            right_flat = re.sub(r"\([^()]*\)", lambda m: "(" + ":" * (m.group(0).count(",") + 1) + ")" if ":" in m.group(0) or "size" in m.group(0).lower() else "", right)
            right = right_flat
        for part in re.split(r",(?![^()]*\))", right):
            nm = re.match(r"\s*(\w+)", part)
            if nm and nm.group(1).lower() in names:
                rank = part.count(":") if "(" in part else (left.count(":") if "dimension" in left else 0)
                out[nm.group(1).lower()] = (base, "optional" in left, rank)
    return out


@pytest.mark.skipif(not os.path.isdir(REFERENCE), reason="the reference tree is only present in the build container")
def test_fortran_shim_matches_the_reference_signatures():
    """Drop-in check against the reference's own sources (read here only; neither the GPU tests nor the bench touch them): every
    `lkb_try_<routine>_<kind>` has the reference routine's dummy arguments -- same names, same order (Fortran is case-insensitive)
    -- and every dummy agrees in base type (class / real / complex / integer / logical), optional-ness and rank."""
    import subprocess, sys
    subprocess.check_call([sys.executable, os.path.join(ROOT, "fortran", "gen_shim.py")], stdout=subprocess.DEVNULL)
    code = _shim_code_without_comments().splitlines()
    checked = 0
    for fn, (rel, routine) in _REF_ROUTINES.items():
        ref = open(os.path.join(REFERENCE, rel)).read().splitlines()
        pat = re.compile(r"^\s*(?:module\s+)?subroutine\s+" + routine + r"_\$\{type\[0\]\}\$\$\{kind\}\$\s*\(([^)]*)\)", re.I)
        hits = [(i, pat.match(ln)) for i, ln in enumerate(ref) if pat.match(ln)]
        assert hits, routine
        i0, m = hits[0]
        ref_args = [a.strip().lower() for a in m.group(1).split(",")]
        j = i0 + 1
        while not re.match(r"^\s*end\s+subroutine", ref[j], re.I) and j < i0 + 80:
            j += 1
        ref_body = [re.sub(r"\$\{type\}\$", "real(dp)", re.sub(r"\$\{type\[0\]\}\$\$\{kind\}\$", "rdp", re.sub(r"\$\{kind\}\$", "dp", ln.split("!")[0])))
                    for ln in ref[i0 + 1:j]]
        ref_attr = _dummy_attributes(ref_body, set(ref_args))
        assert set(ref_attr) == set(ref_args), (routine, sorted(set(ref_args) - set(ref_attr)))
        # the shim's function for rdp
        spat = re.compile(r"^\s*logical function lkb_try_" + fn + r"_rdp\(([^)]*)\) result\(done\)", re.I)
        shits = [(i, spat.match(ln)) for i, ln in enumerate(code) if spat.match(ln)]
        assert shits, fn
        s0, sm = shits[0]
        shim_args = [a.strip().lower() for a in sm.group(1).split(",")]
        assert shim_args == ref_args, (fn, shim_args, ref_args)
        k = s0 + 1
        while not re.match(r"^\s*end function", code[k], re.I):
            k += 1
        shim_attr = _dummy_attributes(code[s0 + 1:k], set(shim_args))
        for a in ref_args:
            assert shim_attr[a] == ref_attr[a], (fn, a, shim_attr[a], ref_attr[a])
            checked += 1
    assert checked > 100


_REF_TBPS = {   # shim procedure (rdp instance) -> (reference file, abstract interface the deferred binding must conform to)
    "cuda_zero": ("AbstractTypes/AbstractVectors.fypp", "abstract_zero"), "cuda_rand": ("AbstractTypes/AbstractVectors.fypp", "abstract_rand"),
    "cuda_scal": ("AbstractTypes/AbstractVectors.fypp", "abstract_scal"), "cuda_axpby": ("AbstractTypes/AbstractVectors.fypp", "abstract_axpby"),
    "cuda_dot": ("AbstractTypes/AbstractVectors.fypp", "abstract_dot"), "cuda_get_size": ("AbstractTypes/AbstractVectors.fypp", "abstract_get_size"),
    "cuda_matvec": ("AbstractTypes/AbstractLinops.fypp", "abstract_matvec"), "cuda_rmatvec": ("AbstractTypes/AbstractLinops.fypp", "abstract_matvec"),
    "cuda_sym_matvec": ("AbstractTypes/AbstractLinops.fypp", "abstract_sym_matvec"),
}


@pytest.mark.skipif(not os.path.isdir(REFERENCE), reason="the reference tree is only present in the build container")
def test_fortran_shim_type_bound_procedures_conform():
    """The deferred bindings of abstract_vector_* / abstract_linop_* / abstract_sym_linop_* (AbstractVectors.fypp:295-381,
    AbstractLinops.fypp:58-87, 204-256): an overriding procedure must have the abstract interface's dummy arguments -- same names,
    order, base type, optional-ness, rank, and the same intent except for the passed object's class."""
    import subprocess, sys
    subprocess.check_call([sys.executable, os.path.join(ROOT, "fortran", "gen_shim.py")], stdout=subprocess.DEVNULL)
    code = _shim_code_without_comments().splitlines()

    def intents(body, names):
        out = {}
        for ln in body:
            if "::" in ln:
                left, right = ln.split("::", 1)
                m = re.search(r"intent\s*\(\s*(\w+)\s*\)", left, re.I)
                for nm in re.findall(r"\w+", re.sub(r"\([^()]*\)", "", right)):
                    if nm.lower() in names:
                        out[nm.lower()] = m.group(1).lower() if m else None
        return out

    checked = 0
    for proc, (rel, iface) in _REF_TBPS.items():
        ref = open(os.path.join(REFERENCE, rel)).read().splitlines()
        pat = re.compile(r"^\s*(?:subroutine|function)\s+" + iface + r"_\$\{type\[0\]\}\$\$\{kind\}\$\s*\(([^)]*)\)", re.I)
        i0, m = [(i, pat.match(ln)) for i, ln in enumerate(ref) if pat.match(ln)][0]
        ref_args = [a.strip().lower() for a in m.group(1).split(",")]
        j = i0 + 1
        while not re.match(r"^\s*end\s+(subroutine|function)", ref[j], re.I):
            j += 1
        ref_body = [re.sub(r"\$\{type\}\$", "real(dp)", re.sub(r"\$\{type\[0\]\}\$\$\{kind\}\$", "rdp", re.sub(r"\$\{kind\}\$", "dp", ln.split("!")[0])))
                    for ln in ref[i0 + 1:j]]
        spat = re.compile(r"^\s*(?:[\w()]+\s+)?(?:subroutine|function)\s+" + proc + r"_rdp\s*\(([^)]*)\)", re.I)
        s0, sm = [(i, spat.match(ln)) for i, ln in enumerate(code) if spat.match(ln)][0]
        shim_args = [a.strip().lower() for a in sm.group(1).split(",")]
        assert shim_args == ref_args, (proc, shim_args, ref_args)
        k = s0 + 1
        while not re.match(r"^\s*end (subroutine|function)", code[k], re.I):
            k += 1
        ra, sa = _dummy_attributes(ref_body, set(ref_args)), _dummy_attributes(code[s0 + 1:k], set(shim_args))
        ri, si = intents(ref_body, set(ref_args)), intents(code[s0 + 1:k], set(shim_args))
        for a in ref_args:
            assert sa[a] == ra[a], (proc, a, sa[a], ra[a])
            assert si[a] == ri[a], (proc, a, "intent", si[a], ri[a])
            checked += 1
    assert checked >= 20
