"""Worker of tests/test_gpu_precond.py::test_sharded_precond_vs_oracle: run under torchrun with N ranks (one per GPU).
Jacobi-preconditioned CG on a z-sharded 7-point stencil and on a row-sharded CSR matrix, and diagonal-preconditioned GMRES
on a z-sharded convection-diffusion stencil (A's input is then M V(k), not V(k): the halo must follow it), against the
single-process CPU oracle, with results bitwise equal on every rank."""
import os
import sys

import numpy as np
import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))


def main():
    import lightkrylov_b200 as lk
    from oracle import lk_oracle as lo
    from helpers import CONVDIFF7, LAPLACE7
    from precond_cases import varcoef_spd_csr

    rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
    torch.cuda.set_device(local)
    dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    ctx = lk.Context.from_torch_distributed(local)
    assert ctx.world == world and ctx.rank == rank

    def gather_rows(local_arr):
        parts = [None] * world
        dist.all_gather_object(parts, local_arr)
        return np.concatenate(parts, axis=0)

    def same_on_all_ranks(obj):
        objs = [None] * world
        dist.all_gather_object(objs, obj)
        return all(o[0] == objs[0][0] and o[1] == objs[0][1] for o in objs)

    results = {}
    # ---- Jacobi PCG on a z-sharded 7-point Laplacian (ragged slabs) ----
    dims = (20, 16, 13); n3 = int(np.prod(dims))
    A = lk.LinOp.stencil7(ctx, "d", *dims, LAPLACE7)
    b = lk.Vector(ctx, "d", A.n, n_global=n3, row0=A.row0).fill_random("uniform", 43)
    x = lk.Vector(ctx, "d", A.n, n_global=n3, row0=A.row0)
    M = lk.LinOp.jacobi(A)
    info, meta = lk.cg(A, b, x, maxiter=500, preconditioner=M)
    assert same_on_all_ranks((info, meta["res"])), "stencil PCG must agree on all ranks"
    results["stencil_cg"] = (info, meta, gather_rows(x.get()))
    # ---- Jacobi PCG on a row-sharded variable-coefficient CSR (row slab = column slab) ----
    cdims = (12, 11, 10); nc = int(np.prod(cdims))
    rp, ci, va, diag = varcoef_spd_csr(cdims, 5)
    r0, ml = lk.partition(nc, world, rank)
    Ac = lk.LinOp.csr_dist(ctx, nc, nc, rp[r0:r0 + ml + 1] - rp[r0], ci[rp[r0]:rp[r0 + ml]], va[rp[r0]:rp[r0 + ml]])
    bc = lk.Vector(ctx, "d", ml, n_global=nc, row0=r0).fill_random("uniform", 44)
    xc = lk.Vector(ctx, "d", ml, n_global=nc, row0=r0)
    Mc = lk.LinOp.jacobi(Ac)
    cinfo, cmeta = lk.cg(Ac, bc, xc, maxiter=2000, preconditioner=Mc)
    assert same_on_all_ranks((cinfo, cmeta["res"])), "CSR PCG must agree on all ranks"
    results["csr_cg"] = (cinfo, cmeta, gather_rows(xc.get()))
    # ---- diagonal-preconditioned GMRES on a z-sharded convection-diffusion stencil ----
    A2 = lk.LinOp.stencil7(ctx, "d", *dims, CONVDIFF7)
    dv = lk.Vector(ctx, "d", A2.n, n_global=n3, row0=A2.row0).fill_random("uniform", 99)
    dv.put(dv.get() + 0.2)
    M2 = lk.LinOp.diag(dv)
    x2 = lk.Vector(ctx, "d", A2.n, n_global=n3, row0=A2.row0)
    ginfo, gmeta = lk.gmres(A2, b, x2, kdim=20, maxiter=30, preconditioner=M2)
    assert same_on_all_ranks((ginfo, gmeta["res"])), "GMRES must agree on all ranks"
    results["gmres"] = (ginfo, gmeta, gather_rows(x2.get()))
    if rank == 0:
        bh = lo.fill(n3, "d", "uniform", 43)
        dh = 0.2 + lo.fill(n3, "d", "uniform", 99)
        cases = {
            "stencil_cg": lambda xo: lo.cg(lo.Op.stencil("d", dims, LAPLACE7), bh, xo, maxiter=500,
                                           precond=lambda v: v.__imul__(1.0 / 6.0)),
            "csr_cg": lambda xo: lo.cg(lo.Op.csr(nc, nc, rp, ci, va), lo.fill(nc, "d", "uniform", 44), xo, maxiter=2000,
                                       precond=lambda v: v.__imul__(1.0 / diag)),
            "gmres": lambda xo: lo.gmres(lo.Op.stencil("d", dims, CONVDIFF7), bh, xo, kdim=20, maxiter=30,
                                         precond=lambda v: v.__imul__(dh)),
        }
        for name, run in cases.items():
            info_, meta_, xg = results[name]
            xo = np.zeros(xg.size)
            oinfo, ometa = run(xo)
            assert info_ == oinfo > 0, (name, info_, oinfo)
            r, ro = np.array(meta_["res"]), np.array(ometa["res"])
            assert r.shape == ro.shape and np.abs(r - ro).max() < 1e-10 * np.abs(ro).max(), name
            assert np.linalg.norm(xg - xo) / np.linalg.norm(xo) < 1e-8, name       # as tests/mgpu_worker.py: sharded sums
        print(f"MGPU_PRECOND_OK world={world}", flush=True)
    ctx.sync()
    dist.barrier()
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
