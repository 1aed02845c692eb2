"""Worker of tests/test_gpu_poly.py::test_sharded_poly: run under torchrun with N ranks (one per GPU).  The GMRES-polynomial
preconditioner on a z-sharded convection-diffusion stencil with P2P halos and with NCCL halos (p2p = 0), and on a row-sharded
CSR matrix: the builder's roots bitwise equal on every rank and close to the one-GPU roots, M r with given roots equal to the
one-GPU result, and GMRES with M giving the same result on all ranks."""
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
    from poly_cases import convdiff_coef
    import scipy.sparse as sp

    lk.set_lapack_from_scipy()
    rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
    torch.cuda.set_device(local)
    dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    ctx = lk.Context.from_torch_distributed(local)
    solo = lk.Context(local, rank=0, world=1) if rank == 0 else None      # the one-GPU result, on rank 0's device

    def gather_rows(local_arr):
        parts = [None] * world
        dist.all_gather_object(parts, local_arr)
        return np.concatenate(parts, axis=0)

    def same_on_all_ranks(obj):
        objs = [None] * world
        dist.all_gather_object(objs, obj)
        return all(o == objs[0] for o in objs)

    dims = (20, 16, 13); n3 = int(np.prod(dims))
    cf = convdiff_coef(3, 1.5)
    nc = 3000
    rp0, ci0, va0 = lo.csr_random("d", nc, nc, 7, 21)
    S = (sp.csr_matrix((0.5 * va0, ci0, rp0), shape=(nc, nc)) + 2.0 * sp.identity(nc)).tocsr()
    S.sum_duplicates(); S.sort_indices()
    rp, ci, va = S.indptr.astype(np.int64), S.indices.astype(np.int32), S.data
    r0, ml = lk.partition(nc, world, rank)
    roots = np.array([13.0, 2.0 + 1.0j, 2.0 - 1.0j, 6.0, 9.0 + 3.0j, 9.0 - 3.0j, 4.0])
    cases = []
    for p2p in (1, 0):
        ctx.set_option("p2p", p2p)
        A = lk.LinOp.stencil7(ctx, "d", *dims, cf)
        cases.append((f"stencil_p2p{p2p}", A, A.row0, n3, lambda c: lk.LinOp.stencil7(c, "d", *dims, cf)))
    Ac = lk.LinOp.csr_dist(ctx, nc, nc, rp[r0:r0 + ml + 1] - rp[r0], ci[rp[r0]:rp[r0 + ml]], va[rp[r0]:rp[r0 + ml]])
    cases.append(("csr", Ac, r0, nc, lambda c: lk.LinOp.csr(c, nc, nc, rp, ci, va)))
    for name, A, row0, ng, solo_op in cases:
        ctx.set_option("p2p", 1 if name == "stencil_p2p1" else 0)
        th_scale = 1.0 if name.startswith("stencil") else 0.3
        M = lk.LinOp.polynomial(A, roots * th_scale)
        r = lk.Vector(ctx, "d", A.m, n_global=ng, row0=row0).fill_random("uniform", 47)
        y = lk.Vector(ctx, "d", A.m, n_global=ng, row0=row0)
        M.matvec(r, y)
        yg = gather_rows(y.get())
        Mb = lk.LinOp.gmres_poly(A, 10, seed=9)
        th = Mb.poly_roots()
        assert same_on_all_ranks(th.tobytes()), name
        bv = lk.Vector(ctx, "d", A.m, n_global=ng, row0=row0).fill_random("uniform", 43)
        x = lk.Vector(ctx, "d", A.m, n_global=ng, row0=row0)
        info, meta = lk.gmres(A, bv, x, kdim=20, maxiter=40, preconditioner=Mb)
        assert info > 0 and same_on_all_ranks((info, meta["res"])), name
        xg = gather_rows(x.get())
        if rank == 0:
            A1 = solo_op(solo)
            r1 = lk.Vector(solo, "d", ng).put(lo.fill(ng, "d", "uniform", 47)); y1 = lk.Vector(solo, "d", ng)
            lk.LinOp.polynomial(A1, roots * th_scale).matvec(r1, y1)
            assert np.abs(yg - y1.get()).max() <= 1e-13 * np.abs(y1.get()).max(), name
            th1 = lk.LinOp.gmres_poly(A1, 10, seed=9).poly_roots()       # same start vector; sums in another order
            assert th1.size == th.size and np.abs(th1 - th).max() <= 1e-8 * np.abs(th).max(), name
            bh = lo.fill(ng, "d", "uniform", 43)
            res = np.linalg.norm(bh - (S @ xg if name == "csr" else lo.Op.stencil("d", dims, cf).apply(xg)))
            assert res <= 1e-7 * np.linalg.norm(bh), (name, res)
        assert same_on_all_ranks(xg.tobytes()), name
    if rank == 0:
        print(f"MGPU_POLY_OK world={world}", flush=True)
    ctx.sync()
    dist.barrier()
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
