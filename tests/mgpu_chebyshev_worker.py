"""Worker of tests/test_gpu_chebyshev.py::test_sharded_chebyshev: run under torchrun with N ranks (one per GPU).  The
Chebyshev preconditioner on a z-sharded 7-point Laplacian with P2P halos and with NCCL halos (p2p = 0), and on a row-sharded
CSR matrix: M r equal to the one-GPU result, Chebyshev-PCG with the oracle's iteration count, x bitwise equal on all ranks."""
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
    from chebyshev_cases import chebyshev_apply, gershgorin
    from helpers import LAPLACE7
    from precond_cases import varcoef_spd_csr
    import scipy.sparse as sp

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
    cdims = (12, 11, 10); nc = int(np.prod(cdims))
    rp, ci, va, diag = varcoef_spd_csr(cdims, 5)
    bc = gershgorin(sp.csr_matrix((va, ci, rp), shape=(nc, nc)))
    r0, ml = lk.partition(nc, world, rank)
    m = 4
    cases = []
    for p2p in (1, 0):
        ctx.set_option("p2p", p2p)
        A = lk.LinOp.stencil7(ctx, "d", *dims, LAPLACE7)
        cases.append((f"stencil_p2p{p2p}", A, A.row0, n3, lo.Op.stencil("d", dims, LAPLACE7), 1.0 / 6.0, 2.0,
                      lambda c: lk.LinOp.stencil7(c, "d", *dims, LAPLACE7)))
    Ac = lk.LinOp.csr_dist(ctx, nc, nc, rp[r0:r0 + ml + 1] - rp[r0], ci[rp[r0]:rp[r0 + ml]], va[rp[r0]:rp[r0 + ml]])
    cases.append(("csr", Ac, r0, nc, lo.Op.csr(nc, nc, rp, ci, va), 1.0 / diag, bc, lambda c: lk.LinOp.csr(c, nc, nc, rp, ci, va)))
    for name, A, row0, ng, Ao, invd, b, solo_op in cases:
        ctx.set_option("p2p", 1 if name == "stencil_p2p1" else 0)
        M = lk.LinOp.chebyshev(A, m)
        r = lk.Vector(ctx, "d", A.m, n_global=ng, row0=row0).fill_random("uniform", 47)
        y = lk.Vector(ctx, "d", A.m, n_global=ng, row0=row0)
        M.matvec(r, y)
        yg = gather_rows(y.get())
        bv = lk.Vector(ctx, "d", A.m, n_global=ng, row0=row0).fill_random("uniform", 43)
        x = lk.Vector(ctx, "d", A.m, n_global=ng, row0=row0)
        info, meta = lk.cg(A, bv, x, maxiter=2000, preconditioner=M)
        assert same_on_all_ranks((info, meta["res"])), name
        xg = gather_rows(x.get())
        if rank == 0:
            A1 = solo_op(solo)
            r1 = lk.Vector(solo, "d", ng).put(lo.fill(ng, "d", "uniform", 47)); y1 = lk.Vector(solo, "d", ng)
            lk.LinOp.chebyshev(A1, m).matvec(r1, y1)
            assert np.abs(yg - y1.get()).max() <= 1e-14 * np.abs(y1.get()).max(), name
            bh = lo.fill(ng, "d", "uniform", 43)
            xo = np.zeros(ng)

            def precond_host(v):
                v[:] = chebyshev_apply(Ao, invd, v.copy(), m, b / 100.0, b)
            oinfo, ometa = lo.cg(Ao, bh, xo, maxiter=2000, precond=precond_host)
            assert info == oinfo > 0 and meta["n_iter"] == ometa["n_iter"], (name, info, oinfo)
            assert np.linalg.norm(xg - xo) / np.linalg.norm(xo) < 1e-8, name
        # x bitwise identical on all ranks: every rank's gathered copy is the same
        assert same_on_all_ranks(xg.tobytes()), name
    if rank == 0:
        print(f"MGPU_CHEBYSHEV_OK world={world}", flush=True)
    ctx.sync()
    dist.barrier()
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
