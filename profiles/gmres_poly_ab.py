"""A/B of the GMRES-polynomial preconditioner on one GPU (include/lkb.h: lkb_op_gmres_poly_create), the arms alternating in
one process, three repetitions.

    python profiles/gmres_poly_ab.py [--reps 3] [--n2 2048] [--c2 4096] [--c4 384] [--cycles 40] [--out DIR]

  convdiff  5-point convection-diffusion stencil n2^2 (cell Peclet 1.5, so a complex spectrum), fp64, gmres(kdim=50) to
            rtol 1e-8 with at most `cycles` restart cycles: no preconditioner, Jacobi, Chebyshev m = 8 (default bounds; a
            reference arm, it assumes a real spectrum) and the GMRES polynomial of degree 5, 10, 20, 40.  Inner steps,
            applications of A, seconds to solution (or the residual at the cap), and the builder's own time
  C2        5-point Poisson c2^2 (bench_configs.py C2), gmres(kdim=50, maxiter=10): residual reached and time per arm
  M alone   one application of the degree-d GMRES polynomial (d = 10, 20) on the C2 grid (c2^2) and on the C4 grid (c4^3),
            fp64: time per application (CUDA events around 20 applications) and bandwidth on the algorithmic bytes of the
            fused steps (stencil input read, output written, held vector read, accumulator read and written)
Prints one JSON line per measurement (device name and power limit in each) and, with --out, writes them to
DIR/gmres_poly_ab.jsonl.
"""
import argparse
import json
import os
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "profiles"))
sys.path.insert(0, os.path.join(ROOT, "tests"))

from poly_cases import convdiff_coef, factors       # noqa: E402
from precond_ab import device_info, timed           # noqa: E402

DEGREES = (5, 10, 20, 40)


def m_bytes(roots, n, es):
    """HBM bytes of one fused application on a stencil (lkb_poly.cu: poly_plan), as multiples of n s."""
    fs = factors(roots, False)
    units, acc_seen, nf = 0, False, len(fs)

    def step(out, v, acc):
        nonlocal units, acc_seen
        units += 1 + out + v + (0 if not acc else (2 if acc_seen else 1))
        acc_seen = acc_seen or acc
    for f, (kind, _) in enumerate(fs):
        last, fold = f + 1 == nf, f + 2 == nf and fs[-1][0] == "root"
        if kind == "root":
            if last:
                step(0, 0, 1)                     # d = 1: k_poly_update reads r, writes z
            elif fold:
                step(0, 0, 1); break
            else:
                step(1, 0, 1)
        elif last:
            step(0, 0, 1)
        else:
            step(1, 0, 1)
            if fold:
                step(0, 1, 1); break
            step(1, 1, 0)
    return units * n * es


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--n2", type=int, default=2048)
    ap.add_argument("--c2", type=int, default=4096)
    ap.add_argument("--c4", type=int, default=384)
    ap.add_argument("--cycles", type=int, default=40)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    import torch
    import lightkrylov_b200 as lk
    dev, plim = device_info()
    lk.set_lapack_from_scipy()
    ctx = lk.Context(0)
    lines = []

    def emit(**kw):
        kw = dict(device=dev, power_limit=plim, **kw)
        print(json.dumps(kw), flush=True)
        lines.append(kw)

    # ---- convection-dominated 2-D stencil: arms alternate within each repetition ----
    m = a.n2; n = m * m
    A = lk.LinOp.stencil5(ctx, "d", m, m, convdiff_coef(2, 1.5))
    b = lk.Vector(ctx, "d", n).fill_random("uniform", 45); x = lk.Vector(ctx, "d", n)
    arms = {"none": (None, 0), "jacobi": (lk.LinOp.jacobi(A), 0), "chebyshev_m8": (lk.LinOp.chebyshev(A, 8), 8)}
    for d in DEGREES:
        ctx.sync(); t0 = time.perf_counter()
        M = lk.LinOp.gmres_poly(A, d, seed=1)
        ctx.sync()
        emit(case=f"builder, convdiff 5-pt {m}^2 fp64", degree=d, seconds=time.perf_counter() - t0, n_roots=len(M.poly_roots()))
        arms[f"gmres_poly_d{d}"] = (M, len(M.poly_roots()))
    for name, (M, _) in arms.items():                                   # warm-up (pool, graph capture)
        x.zero(); lk.gmres(A, b, x, kdim=50, maxiter=1, preconditioner=M)
    for rep in range(a.reps):
        for name, (M, deg) in arms.items():
            x.zero()
            (info, meta), dt = timed(ctx, lambda: lk.gmres(A, b, x, rtol=1e-8, kdim=50, maxiter=a.cycles, preconditioner=M))
            inner = meta["n_inner"]
            apps = inner + meta["n_outer"]                              # + one matvec per restart for the residual
            m_apps = inner + meta["n_outer"] if M is not None else 0
            a_apps = apps + (m_apps * (deg - 1) if deg else 0)
            emit(case=f"convdiff 5-pt {m}^2 Pe 1.5 fp64, gmres kdim 50 rtol 1e-8, at most {a.cycles} cycles", arm=name,
                 rep=rep, info=info, converged=meta["converged"], n_inner=inner, n_outer=meta["n_outer"],
                 a_applications=a_apps, seconds=dt, res_last=meta["res"][-1])
    del A, b, x, arms

    # ---- C2 Poisson, gmres(kdim=50, maxiter=10) ----
    m = a.c2; n = m * m
    A = lk.LinOp.stencil5(ctx, "d", m, m, (4.0, -1.0, -1.0, -1.0, -1.0))
    b = lk.Vector(ctx, "d", n).fill_random("uniform", 45); x = lk.Vector(ctx, "d", n)
    arms = {"none": None, "jacobi": lk.LinOp.jacobi(A), "chebyshev_m8": lk.LinOp.chebyshev(A, 8)}
    arms.update({f"gmres_poly_d{d}": lk.LinOp.gmres_poly(A, d, seed=1) for d in (5, 10, 20)})
    for name, M in arms.items():
        x.zero(); lk.gmres(A, b, x, kdim=50, maxiter=1, preconditioner=M)
    for rep in range(a.reps):
        for name, M in arms.items():
            x.zero()
            (info, meta), dt = timed(ctx, lambda: lk.gmres(A, b, x, kdim=50, maxiter=10, preconditioner=M))
            emit(case=f"C2 Poisson 5-pt {m}^2 fp64, gmres kdim 50 maxiter 10", arm=name, rep=rep, info=info,
                 n_inner=meta["n_inner"], seconds=dt, res_last=meta["res"][-1])
    del A, b, x, arms

    # ---- one application of M, fp64 ----
    for label, make, n in ((f"C2 {a.c2}^2 Poisson", lambda: lk.LinOp.stencil5(ctx, "d", a.c2, a.c2, (4.0, -1.0, -1.0, -1.0, -1.0)), a.c2 ** 2),
                           (f"C4 {a.c4}^3 Laplacian", lambda: lk.LinOp.stencil7(ctx, "d", a.c4, a.c4, a.c4, (6.0,) + (-1.0,) * 6), a.c4 ** 3)):
        A = make()
        r = lk.Vector(ctx, "d", n).fill_random("uniform", 46); y = lk.Vector(ctx, "d", n)
        Ms = {d: lk.LinOp.gmres_poly(A, d, seed=1) for d in (10, 20)}
        stream = torch.cuda.ExternalStream(ctx.stream)
        for d, M in Ms.items():
            M.matvec(r, y)
        for rep in range(a.reps):
            for d, M in Ms.items():
                ctx.sync()
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record(stream)
                for _ in range(20):
                    M.matvec(r, y)
                e1.record(stream)
                e1.synchronize()
                s = e0.elapsed_time(e1) / 1e3 / 20
                th = M.poly_roots()
                nb = m_bytes(th, n, 8)
                emit(case=f"M alone, {label} fp64", degree=d, n_roots=len(th), rep=rep, seconds_per_application=s,
                     algorithmic_bytes=nb, achieved_TBps=nb / s / 1e12, launches=max(len(th) - 1, 1))
        del A, r, y, Ms
    ctx.close()
    if a.out:
        os.makedirs(a.out, exist_ok=True)
        with open(os.path.join(a.out, "gmres_poly_ab.jsonl"), "w") as f:
            for kw in lines:
                f.write(json.dumps(kw) + "\n")


if __name__ == "__main__":
    t0 = time.perf_counter()
    main()
    print(f"# {time.perf_counter() - t0:.0f} s", file=sys.stderr)
