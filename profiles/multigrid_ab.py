"""A/B of the multigrid preconditioner on one GPU (include/lkb.h: lkb_op_multigrid_create), the arms alternating in one
process, three repetitions.

    python profiles/multigrid_ab.py [--reps 3] [--c4 384] [--c2 4096] [--out DIR]

  C4 cg     7-point Laplacian m^3 in fp64 and fp32, cg to the default tolerance with no preconditioner, Chebyshev m = 8 and
            multigrid with smoother degree 1, 2, 3: iterations, fine-grid applications of A (CG's own plus, per application
            of M, m - 1 for Chebyshev and 2 m for multigrid: pre-smoothing m - 1, the restriction's residual, post-smoothing
            m), time to solution
  C2 gmres  5-point Poisson 4096^2, fp64, gmres(kdim=50, maxiter=10) with no preconditioner and with multigrid (m = 2):
            info, inner steps, time
  M alone   one application of multigrid (m = 1, 2, 3) on the C4 and C2 grids, fp64: time per application (CUDA events
            around 20 applications) and achieved bandwidth on the bytes model, summed over the levels above the coarsest:
            pre-smoothing 2 n s for m <= 2 and (5m - 8) n s beyond, restriction 2 n s, prolongation 2 n s, post-smoothing
            3 n s for m = 1 and (5m - 2) n s beyond (m = 2 on the fine level: 14 n s)
Prints one JSON line per measurement (device name and power limit in each) and, with --out, writes them to
DIR/multigrid_ab.jsonl.
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

from precond_ab import device_info, timed      # noqa: E402

MG_DEGREES = (1, 2, 3)


def level_sizes(dims):
    """Unknowns of the levels above the coarsest (every axis halved until <= 512 unknowns or an axis below 2)."""
    sizes, d = [], list(dims)
    while True:
        n = 1
        for v in d:
            n *= v
        if n <= 512 or min(d) < 2:
            return sizes
        sizes.append(n)
        d = [v // 2 for v in d]


def mg_bytes(m, dims, es):
    per = (2 if m <= 2 else 5 * m - 8) + 2 + 2 + (3 if m == 1 else 5 * m - 2)
    return per * sum(level_sizes(dims)) * es


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--c4", type=int, default=384)
    ap.add_argument("--c2", type=int, default=4096)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    import torch
    import lightkrylov_b200 as lk
    dev, plim = device_info()
    ctx = lk.Context(0)
    lines = []

    def emit(**kw):
        kw = dict(device=dev, power_limit=plim, **kw)
        print(json.dumps(kw), flush=True)
        lines.append(kw)

    # ---- C4 cg: arms alternate within each repetition ----
    m = a.c4; n = m ** 3
    for kind in ("d", "s"):
        A = lk.LinOp.stencil7(ctx, kind, m, m, m, (6.0, -1.0, -1.0, -1.0, -1.0, -1.0, -1.0))
        b = lk.Vector(ctx, kind, n).fill_random("uniform", 45); x = lk.Vector(ctx, kind, n)
        arms = {"none": (None, 0), "chebyshev_m8": (lk.LinOp.chebyshev(A, 8), 7)}
        arms.update({f"multigrid_m{d}": (lk.LinOp.multigrid(A, d), 2 * d) for d in MG_DEGREES})
        for name, (M, _) in arms.items():                               # warm-up (pool, graph capture)
            x.zero(); lk.cg(A, b, x, maxiter=20, preconditioner=M)
        for rep in range(a.reps):
            for name, (M, per) in arms.items():
                x.zero()
                (info, meta), dt = timed(ctx, lambda: lk.cg(A, b, x, maxiter=5000, preconditioner=M))
                it = meta["n_iter"]
                emit(case=f"C4 cg 7-pt Laplacian {m}^3 {'fp64' if kind == 'd' else 'fp32'}, default tolerance", arm=name, rep=rep,
                     info=info, n_iter=it, a_applications=it + (it + 1) * per if M is not None else it,
                     seconds_to_solution=dt, res_last=meta["res"][-1])
        del A, b, x, arms

    # ---- C2 gmres(kdim=50, maxiter=10), fp64 ----
    c2 = a.c2; n2 = c2 * c2
    A = lk.LinOp.stencil5(ctx, "d", c2, c2, (4.0, -1.0, -1.0, -1.0, -1.0))
    b = lk.Vector(ctx, "d", n2).fill_random("uniform", 45); x = lk.Vector(ctx, "d", n2)
    arms = {"none": None, "multigrid_m2": lk.LinOp.multigrid(A, 2)}
    for name, M in arms.items():
        x.zero(); lk.gmres(A, b, x, kdim=50, maxiter=1, preconditioner=M)
    for rep in range(a.reps):
        for name, M in arms.items():
            x.zero()
            (info, meta), dt = timed(ctx, lambda: lk.gmres(A, b, x, kdim=50, maxiter=10, preconditioner=M))
            emit(case=f"C2 gmres(kdim=50, maxiter=10) 5-pt Poisson {c2}^2 fp64", arm=name, rep=rep, info=info,
                 converged=meta["converged"], n_inner=meta["n_inner"], seconds=dt, res_last=meta["res"][-1])
    del A, b, x, arms

    # ---- one application of M, fp64 ----
    for label, dims, make in ((f"C4 {m}^3", (m, m, m), lambda: lk.LinOp.stencil7(ctx, "d", m, m, m, (6.0,) + (-1.0,) * 6)),
                              (f"C2 {c2}^2", (c2, c2), lambda: lk.LinOp.stencil5(ctx, "d", c2, c2, (4.0, -1.0, -1.0, -1.0, -1.0)))):
        A = make()
        nn = A.m
        r = lk.Vector(ctx, "d", nn).fill_random("uniform", 46); y = lk.Vector(ctx, "d", nn)
        Ms = {d: lk.LinOp.multigrid(A, d) for d in MG_DEGREES}
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
                emit(case=f"multigrid M alone, {label} fp64", degree=d, rep=rep, seconds_per_application=s,
                     model_bytes=mg_bytes(d, dims, 8), achieved_TBps=mg_bytes(d, dims, 8) / s / 1e12)
        del A, r, y, Ms
    ctx.close()
    if a.out:
        os.makedirs(a.out, exist_ok=True)
        with open(os.path.join(a.out, "multigrid_ab.jsonl"), "w") as f:
            for kw in lines:
                f.write(json.dumps(kw) + "\n")


if __name__ == "__main__":
    t0 = time.perf_counter()
    main()
    print(f"# {time.perf_counter() - t0:.0f} s", file=sys.stderr)
