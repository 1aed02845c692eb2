"""A/B of the Chebyshev preconditioner on one GPU (include/lkb.h: lkb_op_chebyshev_create), the arms alternating in one
process, three repetitions.

    python profiles/chebyshev_ab.py [--reps 3] [--c4 384] [--c2 4096] [--out DIR]

  C4 cg    7-point Laplacian m^3 in fp64 and fp32, cg to the default tolerance with no preconditioner, Jacobi, and
           Chebyshev of degree 2, 4, 8, 16 (default bounds [0.02, 2]): iterations, applications of A, time to solution
  M alone  one application of the degree-m Chebyshev operator on the C4 grid (384^3) and on the C2 grid (5-point 4096^2),
           fp64: time per application (CUDA events around 20 applications) and achieved bandwidth on the algorithmic bytes
           of the fused steps, (5m - 8) n s for m >= 3 and 2 n s for m <= 2 (x, r, d read and d, z written per middle step)
Prints one JSON line per measurement (device name and power limit in each) and, with --out, writes them to
DIR/chebyshev_ab.jsonl.
"""
import argparse
import json
import os
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "profiles"))

from precond_ab import device_info, timed      # noqa: E402

DEGREES = (2, 4, 8, 16)


def m_bytes(m, n, es):
    return (2 if m <= 2 else 5 * m - 8) * n * es


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
        arms = {"none": (None, 0), "jacobi": (lk.LinOp.jacobi(A), 0)}
        arms.update({f"chebyshev_m{d}": (lk.LinOp.chebyshev(A, d), d) for d in DEGREES})
        for name, (M, _) in arms.items():                               # warm-up (pool, graph capture)
            x.zero(); lk.cg(A, b, x, maxiter=20, preconditioner=M)
        for rep in range(a.reps):
            for name, (M, deg) in arms.items():
                x.zero()
                (info, meta), dt = timed(ctx, lambda: lk.cg(A, b, x, maxiter=5000, preconditioner=M))
                it = meta["n_iter"]
                a_apps = it + (it + 1) * (deg - 1) if deg else it
                emit(case=f"C4 cg 7-pt Laplacian {m}^3 {'fp64' if kind == 'd' else 'fp32'}, default tolerance", arm=name, rep=rep,
                     info=info, n_iter=it, a_applications=a_apps, seconds_to_solution=dt, res_last=meta["res"][-1])
        del A, b, x, arms

    # ---- one application of M, fp64 ----
    for label, make, n in ((f"C4 {m}^3", lambda: lk.LinOp.stencil7(ctx, "d", m, m, m, (6.0,) + (-1.0,) * 6), m ** 3),
                           (f"C2 {a.c2}^2", lambda: lk.LinOp.stencil5(ctx, "d", a.c2, a.c2, (4.0, -1.0, -1.0, -1.0, -1.0)), a.c2 ** 2)):
        A = make()
        r = lk.Vector(ctx, "d", n).fill_random("uniform", 46); y = lk.Vector(ctx, "d", n)
        Ms = {d: lk.LinOp.chebyshev(A, d) for d in DEGREES}
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
                emit(case=f"M alone, {label} fp64", degree=d, rep=rep, seconds_per_application=s,
                     algorithmic_bytes=m_bytes(d, n, 8), achieved_TBps=m_bytes(d, n, 8) / s / 1e12,
                     matvec_equivalents=max(d - 1, 1))
        del A, r, y, Ms
    ctx.close()
    if a.out:
        os.makedirs(a.out, exist_ok=True)
        with open(os.path.join(a.out, "chebyshev_ab.jsonl"), "w") as f:
            for kw in lines:
                f.write(json.dumps(kw) + "\n")


if __name__ == "__main__":
    t0 = time.perf_counter()
    main()
    print(f"# {time.perf_counter() - t0:.0f} s", file=sys.stderr)
