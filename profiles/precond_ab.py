"""A/B of the preconditioned solvers on one GPU: no preconditioner, a torch callback (the host-driven path) and a library
operator (the device-resident path), the arms alternating in one process, three repetitions.

    python profiles/precond_ab.py [--reps 3] [--c4 384] [--csr 128] [--c2 4096] [--out DIR]

  C4     7-point Laplacian m^3 fp64, cg: a fixed 200 iterations (iterations/s) and a solve to the default tolerance
  CSR    variable-coefficient 7-point diffusion on an m^3 grid (tests/precond_cases.py, cell coefficient 10^(4u-2)),
         cg to the default tolerance: iterations to convergence and time to solution
  C2     5-point Poisson m^2 fp64, gmres(kdim=50, maxiter=10) with a diagonal M: inner steps/s, callback against operator
Prints one JSON line per measurement (device name and power limit in each) and, with --out, writes them to DIR/precond_ab.jsonl.
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))


def device_info():
    import torch
    name = torch.cuda.get_device_name(0)
    try:
        pl = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"],
                            capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception as e:       # the number is still reported, with the reason the limit is missing
        pl = f"unavailable ({e})"
    return name, pl


class _DevArray:
    def __init__(self, ptr, n, typestr):
        self.__cuda_array_interface__ = {"shape": (n,), "typestr": typestr, "data": (ptr, False), "version": 3}


def torch_diag_callback(ctx, dh):
    """z *= d on the library's stream with torch: the callback path (two host syncs and a copy per CG iteration)."""
    import torch
    dd = torch.from_numpy(np.ascontiguousarray(dh)).cuda()
    ext = torch.cuda.ExternalStream(ctx.stream)

    def precond(ptr, nloc, it, cur, tgt, stream):
        with torch.cuda.stream(ext):
            torch.as_tensor(_DevArray(ptr, nloc, "<f8"), device="cuda").mul_(dd)
        return 0
    return precond


def timed(ctx, fn):
    ctx.sync()
    t0 = time.perf_counter()
    r = fn()
    ctx.sync()
    return r, time.perf_counter() - t0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--c4", type=int, default=384)
    ap.add_argument("--csr", type=int, default=128)
    ap.add_argument("--c2", type=int, default=4096)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    import lightkrylov_b200 as lk
    from precond_cases import varcoef_spd_csr
    dev, plim = device_info()
    ctx = lk.Context(0)
    lines = []

    def emit(**kw):
        kw = dict(device=dev, power_limit=plim, **kw)
        print(json.dumps(kw), flush=True)
        lines.append(kw)

    # ---- C4: 7-point Laplacian m^3 fp64 ----
    m = a.c4; n = m ** 3
    A = lk.LinOp.stencil7(ctx, "d", m, m, m, (6.0, -1.0, -1.0, -1.0, -1.0, -1.0, -1.0))
    b = lk.Vector(ctx, "d", n).fill_random("uniform", 45); x = lk.Vector(ctx, "d", n)
    arms = {"none": None, "callback_jacobi": torch_diag_callback(ctx, np.full(n, 1.0 / 6.0)), "device_jacobi": lk.LinOp.jacobi(A)}
    for name, M in arms.items():                                        # warm-up (pool, graph capture, torch)
        x.zero(); lk.cg(A, b, x, maxiter=20, preconditioner=M)
    for rep in range(a.reps):
        for name, M in arms.items():
            x.zero()
            (info, meta), dt = timed(ctx, lambda: lk.cg(A, b, x, rtol=0.0, atol=1e-300, maxiter=200, preconditioner=M))
            emit(case=f"C4 cg 7-pt Laplacian {m}^3 fp64, fixed 200 iterations", arm=name, rep=rep, n_iter=meta["n_iter"],
                 seconds=dt, iters_per_s=meta["n_iter"] / dt, res_last=meta["res"][-1])
            x.zero()
            (info, meta), dt = timed(ctx, lambda: lk.cg(A, b, x, maxiter=2000, preconditioner=M))
            emit(case=f"C4 cg 7-pt Laplacian {m}^3 fp64, default tolerance", arm=name, rep=rep, info=info, n_iter=meta["n_iter"],
                 seconds_per_solve=dt, iters_per_s=meta["n_iter"] / dt, res_last=meta["res"][-1])
    del A, b, x, arms

    # ---- variable-coefficient SPD CSR on an m^3 grid ----
    m = a.csr; dims = (m, m, m); n = m ** 3
    t0 = time.perf_counter()
    rp, ci, va, diag = varcoef_spd_csr(dims, 5)
    tbuild = time.perf_counter() - t0
    A = lk.LinOp.csr(ctx, n, n, rp, ci, va)
    b = lk.Vector(ctx, "d", n).fill_random("uniform", 45); x = lk.Vector(ctx, "d", n)
    arms = {"none": None, "callback_jacobi": torch_diag_callback(ctx, 1.0 / diag), "device_jacobi": lk.LinOp.jacobi(A)}
    for name, M in arms.items():
        x.zero(); lk.cg(A, b, x, maxiter=20, preconditioner=M)
    for rep in range(a.reps):
        for name, M in arms.items():
            x.zero()
            (info, meta), dt = timed(ctx, lambda: lk.cg(A, b, x, maxiter=50000, preconditioner=M))
            emit(case=f"CSR cg variable-coefficient diffusion {m}^3 ({n} rows, {int(rp[-1])} nnz) fp64, default tolerance",
                 arm=name, rep=rep, info=info, n_iter=meta["n_iter"], converged=meta["converged"], seconds_to_solution=dt,
                 iters_per_s=meta["n_iter"] / dt, res_last=meta["res"][-1], host_build_s=tbuild)
    del A, b, x, arms

    # ---- C2 operator, gmres(kdim=50, maxiter=10), diagonal M ----
    m = a.c2; n = m * m
    A = lk.LinOp.stencil5(ctx, "d", m, m, (4.0, -1.0, -1.0, -1.0, -1.0))
    b = lk.Vector(ctx, "d", n).fill_random("uniform", 43); x = lk.Vector(ctx, "d", n)
    dv = lk.Vector(ctx, "d", n).fill_random("uniform", 99)
    dh = dv.get() + 0.2; dv.put(dh)
    arms = {"callback_diag": torch_diag_callback(ctx, dh), "operator_diag": lk.LinOp.diag(dv)}
    for name, M in arms.items():
        x.zero(); lk.gmres(A, b, x, kdim=50, maxiter=1, preconditioner=M)
    for rep in range(a.reps):
        for name, M in arms.items():
            x.zero()
            (info, meta), dt = timed(ctx, lambda: lk.gmres(A, b, x, kdim=50, maxiter=10, preconditioner=M))
            emit(case=f"C2 gmres(kdim=50, maxiter=10) 5-pt Poisson {m}^2 fp64, diagonal M", arm=name, rep=rep, info=info,
                 n_inner=meta["n_inner"], n_outer=meta["n_outer"], seconds=dt, inner_steps_per_s=meta["n_inner"] / dt,
                 res_last=meta["res"][-1])
    ctx.close()
    if a.out:
        os.makedirs(a.out, exist_ok=True)
        with open(os.path.join(a.out, "precond_ab.jsonl"), "w") as f:
            for kw in lines:
                f.write(json.dumps(kw) + "\n")


if __name__ == "__main__":
    main()
