"""Failure paths of operator creation on the device: a failed allocation is an ordinary LKB_ERR_ALLOC that leaves the context
usable, and CSR arrays handed over with adopt = 1 stay with the caller when the create call rejects them."""
import ctypes as C

import numpy as np
import pytest

from helpers import POISSON5

pytestmark = pytest.mark.gpu
LKB_ERR_ARG, LKB_ERR_ALLOC = -2, -6


@pytest.fixture(scope="module")
def lk():
    import lightkrylov_b200 as lk
    return lk


def _stencil_arnoldi(lk, ctx):
    nx, ny, kdim = 96, 64, 16
    A = lk.LinOp.stencil5(ctx, "d", nx, ny, POISSON5)
    X = lk.Basis(ctx, "d", nx * ny, kdim + 1)
    X.put(np.random.default_rng(7).standard_normal(nx * ny))
    H = np.zeros((kdim + 1, kdim), order="F")
    info = lk.arnoldi(A, X, H)
    return info, H, X.get()


def test_failed_allocation_leaves_the_context_usable(lk):
    """Sizes no device can hold (>= 1 PB): cudaMalloc returns cudaErrorMemoryAllocation at once.  The create calls return
    LKB_ERR_ALLOC, and the next kernel launch on the context is not reported as failed."""
    ctx, fresh = lk.Context(0), lk.Context(0)
    try:
        lib, kd = ctx.lib, lk.KINDS["d"]
        a = np.zeros(4)
        h = C.c_void_p()
        assert lib.lkb_op_dense_create(ctx.h, kd, 1 << 25, 1 << 25, a.ctypes.data, C.byref(h)) == LKB_ERR_ALLOC    # 8 PB
        assert b"cudaMalloc(" in lib.lkb_last_error() and not h.value
        rp, ci, va = C.c_void_p(), C.c_void_p(), C.c_void_p()
        assert lib.lkb_csr_random_device(ctx.h, kd, 1 << 47, 0, 1000, 8, 1, C.byref(rp), C.byref(ci), C.byref(va)) == LKB_ERR_ALLOC
        assert not (rp.value or ci.value or va.value)
        info, H, X = _stencil_arnoldi(lk, ctx)
        info0, H0, X0 = _stencil_arnoldi(lk, fresh)
        assert info == info0 and np.array_equal(H, H0) and np.array_equal(X, X0)
    finally:
        fresh.close()
        ctx.close()


def _create_adopting(lib, ctx, dist, kind, m, n, rp, ci, va, h):
    if dist:        # a row-sharded operator of one rank: the slab exchange and gather buffers come before the CSR set-up
        return lib.lkb_op_csr_create_dist_device(ctx.h, kind, m, n, 0, m, 0, n, rp, ci, va, 1, C.byref(h))
    return lib.lkb_op_csr_create_device(ctx.h, kind, m, n, rp, ci, va, 1, C.byref(h))


@pytest.mark.parametrize("dist", [False, True])
@pytest.mark.parametrize("blocked", [False, True])
def test_adopted_arrays_survive_a_rejected_create(lk, oracle, blocked, dist):
    """lkb_op_csr_create_device / lkb_op_csr_create_dist_device (adopt = 1) with an n too small for the column indices is
    rejected (LKB_ERR_ARG); the same arrays then make a working operator.  `blocked` forces the L2-blocked layout, which
    replaces the adopted arrays."""
    ctx = lk.Context(0)
    try:
        if blocked:
            ctx.set_option("csr_slice_kb", 4); ctx.set_option("csr_block_min_kb", 0)
        lib = ctx.lib
        for kind in ("d", "z"):
            m, n, pr, seed = 3001, 2003, 32, 46
            rp, ci, va = C.c_void_p(), C.c_void_p(), C.c_void_p()
            assert lib.lkb_csr_random_device(ctx.h, lk.KINDS[kind], m, 0, n, pr, seed, C.byref(rp), C.byref(ci), C.byref(va)) == 0
            h = C.c_void_p()
            assert _create_adopting(lib, ctx, dist, lk.KINDS[kind], m, n // 2, rp, ci, va, h) == LKB_ERR_ARG
            assert b"column index out of range" in lib.lkb_last_error() and not h.value
            assert _create_adopting(lib, ctx, dist, lk.KINDS[kind], m, n, rp, ci, va, h) == 0
            A = lk.LinOp(ctx, kind, h, m, n)
            Ao = oracle.Op.csr(m, n, *oracle.csr_random(kind, m, n, pr, seed))
            xh = oracle.fill(n, kind, "normal", 3); uh = oracle.fill(m, kind, "normal", 4)
            x = lk.Vector(ctx, kind, n).put(xh); u = lk.Vector(ctx, kind, m).put(uh)
            y = lk.Vector(ctx, kind, m); v = lk.Vector(ctx, kind, n)
            l0 = ctx.kernel_launches
            A.matvec(x, y)
            assert ctx.kernel_launches - l0 == (2 if blocked else 1)        # the blocked layout: one sweep per column block
            A.rmatvec(u, v)
            np.testing.assert_allclose(y.get(), Ao.apply(xh), rtol=1e-11, atol=1e-11)
            np.testing.assert_allclose(v.get(), Ao.apply(uh, trans=True), rtol=1e-11, atol=1e-11)
            del A
    finally:
        ctx.close()
