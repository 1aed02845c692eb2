"""Host-side mirror of LightKrylov's operator / vector / Krylov-process interface on top of the
C ABI (include/lkb.h).  Names, argument meaning and info semantics follow the reference:

    arnoldi(A, X, H, kstart, kend, tol, transpose, blksize) -> info      src/Krylov/BaseKrylov.fypp:132-152
    lanczos(A, X, T, kstart, kend, tol) -> info                          :221-234
    bidiagonalization(A, U, V, B, kstart, kend, tol) -> info             :311-330
    double_gram_schmidt_step(y, X, if_chk_orthonormal, beta) -> info     :679-709
    qr(Q, R, tol) -> info                                                :395-417
    gmres / cg / eigs / eighs / svds                                     src/IterativeSolvers

The reference toolchain (Fortran) is absent in this image, so this Python layer plays the role of
the Fortran shim (fortran/lightkrylov_cuda.f90) for tests and benchmarks.  Everything numeric
happens inside liblkb.so on the GPU; numpy is only used to marshal host arrays.
"""
from __future__ import annotations

import ctypes as C
import os
from typing import Optional, Sequence

import numpy as np

from . import _lib
from ._lib import LkbError, check

KINDS = {"s": 0, "d": 1, "c": 2, "z": 3}
DTYPES = {"s": np.float32, "d": np.float64, "c": np.complex64, "z": np.complex128}
ATOL = {"s": 1e-6, "d": 1e-15, "c": 1e-6, "z": 1e-15}
RTOL = {k: float(np.sqrt(v)) for k, v in ATOL.items()}


def kind_of(dtype) -> str:
    dt = np.dtype(dtype)
    for k, v in DTYPES.items():
        if np.dtype(v) == dt:
            return k
    raise TypeError(f"unsupported dtype {dt}")


def _scalar(kind: str, v):
    return np.array([v], dtype=DTYPES[kind])


def partition(n_slow: int, world: int, rank: int):
    """1-D block partition of the slowest grid axis / rows: returns (start, count)."""
    base, rem = divmod(n_slow, world)
    start = rank * base + min(rank, rem)
    return start, base + (1 if rank < rem else 0)


class Context:
    """One context per process per GPU (lkb_init / lkb_init_dist)."""

    def __init__(self, device: int = 0, rank: int = 0, world: int = 1, unique_id: Optional[bytes] = None):
        self.lib = _lib.load()
        h = C.c_void_p()
        if world > 1:
            assert unique_id is not None and len(unique_id) == 128
            buf = C.create_string_buffer(unique_id, 128)
            check(self.lib.lkb_init_dist(device, rank, world, buf, C.byref(h)), "lkb_init_dist")
        else:
            check(self.lib.lkb_init(device, C.byref(h)), "lkb_init")
        self.h, self.rank, self.world, self.device = h, rank, world, device
        self.p2p = False

    @staticmethod
    def nccl_unique_id() -> bytes:
        lib = _lib.load()
        buf = C.create_string_buffer(128)
        check(lib.lkb_nccl_unique_id(buf), "lkb_nccl_unique_id")
        return buf.raw

    @classmethod
    def from_torch_distributed(cls, device: int):
        """Rendezvous through torch.distributed (plumbing only): rank 0 creates the NCCL id."""
        import torch.distributed as dist
        rank, world = dist.get_rank(), dist.get_world_size()
        if world == 1:
            return cls(device)
        obj = [cls.nccl_unique_id() if rank == 0 else None]
        dist.broadcast_object_list(obj, src=0)
        ctx = cls(device, rank, world, obj[0])
        if world <= 8 and os.environ.get("LKB_P2P", "1") != "0":
            # in-kernel NVLink allreduce: exchange CUDA-IPC handles of the per-rank exchange buffers.
            # Every step is collective and the ranks agree on the outcome, so a local failure (no peer
            # access, IPC disabled) downgrades ALL ranks to the NCCL path instead of desynchronising them.
            ok = 1
            try:
                mine = ctx.p2p_export()
            except LkbError:
                mine, ok = b"\0" * 64, 0
            handles = [None] * world
            dist.all_gather_object(handles, mine)
            if ok:
                try:
                    ctx.p2p_attach(b"".join(handles))
                except LkbError as e:
                    ok = 0
                    import warnings
                    warnings.warn(f"p2p allreduce unavailable, using NCCL: {e}")
            flags = [None] * world
            dist.all_gather_object(flags, ok)
            if all(flags):
                ctx.p2p = True
            else:
                ctx.set_option("p2p", 0)
            dist.barrier()
        return ctx

    def p2p_export(self) -> bytes:
        buf = C.create_string_buffer(64)
        check(self.lib.lkb_p2p_export(self.h, buf), "lkb_p2p_export")
        return buf.raw

    def p2p_attach(self, handles: bytes):
        buf = C.create_string_buffer(handles, len(handles))
        check(self.lib.lkb_p2p_attach(self.h, buf), "lkb_p2p_attach")

    def sync(self):
        check(self.lib.lkb_sync(self.h), "lkb_sync")

    def set_seed(self, seed: int):
        check(self.lib.lkb_set_seed(self.h, seed))

    def set_graphs(self, enable: bool):
        check(self.lib.lkb_set_graphs(self.h, int(enable)))

    def set_profile(self, enable: bool):
        check(self.lib.lkb_set_profile(self.h, int(enable)))

    def set_option(self, name: str, value: int):
        check(self.lib.lkb_set_option(self.h, name.encode(), int(value)), "set_option")

    def get_profile(self):
        ms = (C.c_double * 8)(); n = (C.c_int64 * 8)()
        check(self.lib.lkb_get_profile(self.h, ms, n))
        names = ["matvec", "multidot", "multiaxpy", "other", "fused_axpy_dot"]
        return {k: (ms[i], n[i]) for i, k in enumerate(names)}

    @property
    def stream(self) -> int:
        return int(self.lib.lkb_stream(self.h) or 0)

    @property
    def kernel_launches(self) -> int:
        return int(self.lib.lkb_kernel_launches(self.h))

    def close(self):
        if self.h:
            self.lib.lkb_finalize(self.h)
            self.h = None


class Vector:
    """Device-resident abstract_vector (AbstractVectors.fypp:295-381)."""

    def __init__(self, ctx: Context, kind: str, n_local: int, n_global: Optional[int] = None, row0: int = 0,
                 _handle=None, _owner=None):
        self.ctx, self.kind, self.n = ctx, kind, n_local
        self.n_global = n_local if n_global is None else n_global
        self.row0 = row0
        self._owner = _owner
        if _handle is None:
            h = C.c_void_p()
            check(ctx.lib.lkb_vec_create(ctx.h, KINDS[kind], n_local, self.n_global, row0, C.byref(h)), "lkb_vec_create")
            self.h = h
        else:
            self.h = _handle

    def zero(self):
        check(self.ctx.lib.lkb_vec_zero(self.h)); return self

    def rand(self, ifnorm: bool = False):
        check(self.ctx.lib.lkb_vec_rand(self.h, int(ifnorm))); return self

    def fill_random(self, dist: str, seed: int):
        check(self.ctx.lib.lkb_vec_fill_random(self.h, 0 if dist == "normal" else 1, seed)); return self

    def scal(self, alpha):
        a = _scalar(self.kind, alpha)
        check(self.ctx.lib.lkb_vec_scal(self.h, a.ctypes.data)); return self

    def axpby(self, alpha, vec: "Vector", beta):
        """self = alpha*vec + beta*self"""
        a, b = _scalar(self.kind, alpha), _scalar(self.kind, beta)
        check(self.ctx.lib.lkb_vec_axpby(a.ctypes.data, vec.h, b.ctypes.data, self.h), "axpby"); return self

    def dot(self, vec: "Vector"):
        out = np.zeros(1, dtype=DTYPES[self.kind])
        check(self.ctx.lib.lkb_vec_dot(self.h, vec.h, out.ctypes.data), "dot")
        return out[0]

    def norm(self) -> float:
        out = C.c_double()
        check(self.ctx.lib.lkb_vec_norm(self.h, C.byref(out)), "norm")
        return out.value

    def add(self, vec): return self.axpby(1, vec, 1)
    def sub(self, vec): return self.axpby(-1, vec, 1)
    def chsgn(self): return self.scal(-1)
    def get_size(self) -> int: return int(self.ctx.lib.lkb_vec_size(self.h))

    def clone(self) -> "Vector":
        h = C.c_void_p()
        check(self.ctx.lib.lkb_vec_clone(self.h, C.byref(h)), "clone")
        return Vector(self.ctx, self.kind, self.n, self.n_global, self.row0, _handle=h)

    def put(self, host: np.ndarray):
        a = np.ascontiguousarray(host, dtype=DTYPES[self.kind])
        assert a.size == self.n
        check(self.ctx.lib.lkb_vec_put(self.h, a.ctypes.data), "put"); return self

    def get(self) -> np.ndarray:
        out = np.empty(self.n, dtype=DTYPES[self.kind])
        check(self.ctx.lib.lkb_vec_get(self.h, out.ctypes.data), "get")
        return out

    @property
    def ptr(self) -> int:
        return int(self.ctx.lib.lkb_vec_ptr(self.h))

    def __del__(self):
        try:
            if getattr(self, "h", None) and self.ctx.h:
                self.ctx.lib.lkb_vec_destroy(self.h)
        except Exception:
            pass


class Basis:
    """X(:) -- contiguous column-major device array of abstract_vectors."""

    def __init__(self, ctx: Context, kind: str, n_local: int, ncols: int, n_global: Optional[int] = None, row0: int = 0):
        self.ctx, self.kind, self.n, self.ncols = ctx, kind, n_local, ncols
        self.n_global = n_local if n_global is None else n_global
        self.row0 = row0
        h = C.c_void_p()
        check(ctx.lib.lkb_basis_create(ctx.h, KINDS[kind], n_local, self.n_global, row0, ncols, C.byref(h)), "lkb_basis_create")
        self.h = h

    def col(self, i: int) -> Vector:
        """0-based column view (X(i+1) in the reference's numbering)."""
        h = C.c_void_p()
        check(self.ctx.lib.lkb_basis_col(self.h, i, C.byref(h)), "basis_col")
        return Vector(self.ctx, self.kind, self.n, self.n_global, self.row0, _handle=h, _owner=self)

    def __getitem__(self, i): return self.col(i)
    def __len__(self): return self.ncols

    @classmethod
    def _from_handle(cls, parent: "Basis", h, ncols: int) -> "Basis":
        b = cls.__new__(cls)
        b.ctx, b.kind, b.n, b.ncols, b.n_global, b.row0, b.h, b._parent = parent.ctx, parent.kind, parent.n, ncols, parent.n_global, parent.row0, h, parent
        return b

    def view(self, col0: int, ncols: int) -> "Basis":
        """Non-owning view of columns [col0, col0+ncols): the array section X(col0+1 : col0+ncols) of the reference."""
        h = C.c_void_p()
        check(self.ctx.lib.lkb_basis_view(self.h, col0, ncols, C.byref(h)), "basis_view")
        return Basis._from_handle(self, h, ncols)

    def axpby(self, alpha, X: "Basis", beta, xcol0: int = 0, ycol0: int = 0, ncols: Optional[int] = None):
        """axpby_basis: self(:, ycol0+q) = alpha X(:, xcol0+q) + beta self(:, ycol0+q)  (AbstractVectors.fypp:697-709)"""
        a, b = _scalar(self.kind, alpha), _scalar(self.kind, beta)
        ncols = min(self.ncols - ycol0, X.ncols - xcol0) if ncols is None else ncols
        check(self.ctx.lib.lkb_basis_axpby(a.ctypes.data, X.h, xcol0, b.ctypes.data, self.h, ycol0, ncols), "basis_axpby"); return self

    def copy_from(self, X: "Basis", xcol0: int = 0, ycol0: int = 0, ncols: Optional[int] = None):
        """copy(out, from) = out%axpby(1, from, 0)  (AbstractVectors.fypp:717-723)"""
        return self.axpby(1, X, 0, xcol0, ycol0, ncols)

    def rand(self, col0: int = 0, ncols: Optional[int] = None, ifnorm: bool = False):
        """rand_basis (AbstractVectors.fypp:725-730)"""
        check(self.ctx.lib.lkb_basis_rand(self.h, col0, self.ncols - col0 if ncols is None else ncols, int(ifnorm)), "basis_rand"); return self

    def orthonormalize(self, col0: int = 0, p: Optional[int] = None) -> int:
        """orthonormalize_basis (src/Krylov/utilities.fypp:70-81)"""
        info = C.c_int32()
        check(self.ctx.lib.lkb_orthonormalize_basis(self.h, col0, self.ncols - col0 if p is None else p, C.byref(info)), "orthonormalize_basis")
        return info.value

    def zero(self, col0: int = 0, ncols: Optional[int] = None):
        check(self.ctx.lib.lkb_basis_zero(self.h, col0, self.ncols - col0 if ncols is None else ncols)); return self

    def put(self, host: np.ndarray, col0: int = 0):
        a = np.asfortranarray(host, dtype=DTYPES[self.kind])
        if a.ndim == 1:
            a = a.reshape(-1, 1, order="F")
        assert a.shape[0] == self.n
        check(self.ctx.lib.lkb_basis_put(self.h, col0, a.shape[1], a.ctypes.data, a.shape[0]), "basis_put"); return self

    def get(self, col0: int = 0, ncols: Optional[int] = None) -> np.ndarray:
        ncols = self.ncols - col0 if ncols is None else ncols
        out = np.empty((self.n, ncols), dtype=DTYPES[self.kind], order="F")
        check(self.ctx.lib.lkb_basis_get(self.h, col0, ncols, out.ctypes.data, self.n), "basis_get")
        return out

    def innerprod(self, j: int, W: "Basis", wcol0: int = 0, p: int = 1) -> np.ndarray:
        out = np.zeros((max(j, 1), p), dtype=DTYPES[self.kind], order="F")
        check(self.ctx.lib.lkb_basis_innerprod(self.h, j, W.h, wcol0, p, out.ctypes.data, out.shape[0]), "innerprod")
        return out[:j]

    def lincomb_sub(self, j: int, coef: np.ndarray, W: "Basis", wcol0: int = 0):
        cf = np.asfortranarray(coef, dtype=DTYPES[self.kind]).reshape(j, -1, order="F")
        check(self.ctx.lib.lkb_basis_lincomb_sub(self.h, j, cf.ctypes.data, j, W.h, wcol0, cf.shape[1]), "lincomb_sub")

    def linear_combination(self, j: int, coef: np.ndarray, y: Vector):
        cf = np.ascontiguousarray(coef, dtype=DTYPES[self.kind])
        check(self.ctx.lib.lkb_basis_lincomb(self.h, j, cf.ctypes.data, y.h), "lincomb")

    def __del__(self):
        try:
            if getattr(self, "h", None) and self.ctx.h:
                self.ctx.lib.lkb_basis_destroy(self.h)
        except Exception:
            pass


class LinOp:
    """Device abstract_linop (AbstractLinops.fypp:58-87): matvec / rmatvec with counters."""

    def __init__(self, ctx: Context, kind: str, handle, m: int, n: int, keep=None):
        self.ctx, self.kind, self.h, self.m, self.n, self._keep = ctx, kind, handle, m, n, keep

    @classmethod
    def stencil5(cls, ctx: Context, kind: str, nx: int, ny: int, coef: Sequence, slab=None) -> "LinOp":
        y0, nyl = slab if slab is not None else partition(ny, ctx.world, ctx.rank)
        cf = np.array(coef, dtype=DTYPES[kind]); assert cf.size == 5
        h = C.c_void_p()
        check(ctx.lib.lkb_op_stencil5_create(ctx.h, KINDS[kind], nx, ny, cf.ctypes.data, y0, nyl, C.byref(h)), "stencil5")
        op = cls(ctx, kind, h, nx * nyl, nx * nyl)
        op.row0, op.n_global = nx * y0, nx * ny
        return op

    @classmethod
    def stencil7(cls, ctx: Context, kind: str, nx: int, ny: int, nz: int, coef: Sequence, slab=None) -> "LinOp":
        z0, nzl = slab if slab is not None else partition(nz, ctx.world, ctx.rank)
        cf = np.array(coef, dtype=DTYPES[kind]); assert cf.size == 7
        h = C.c_void_p()
        check(ctx.lib.lkb_op_stencil7_create(ctx.h, KINDS[kind], nx, ny, nz, cf.ctypes.data, z0, nzl, C.byref(h)), "stencil7")
        op = cls(ctx, kind, h, nx * ny * nzl, nx * ny * nzl)
        op.row0, op.n_global = nx * ny * z0, nx * ny * nz
        return op

    @classmethod
    def csr(cls, ctx: Context, m: int, n: int, rowptr, col, val) -> "LinOp":
        kind = kind_of(val.dtype)
        rp = np.ascontiguousarray(rowptr, dtype=np.int64); ci = np.ascontiguousarray(col, dtype=np.int32)
        va = np.ascontiguousarray(val)
        h = C.c_void_p()
        check(ctx.lib.lkb_op_csr_create(ctx.h, KINDS[kind], m, n, rp.ctypes.data, ci.ctypes.data, va.ctypes.data, C.byref(h)), "csr")
        op = cls(ctx, kind, h, m, n)
        op.row0, op.n_global = 0, n
        return op

    @classmethod
    def csr_random(cls, ctx: Context, kind: str, m: int, n: int, per_row: int, seed: int) -> "LinOp":
        """Synthetic config-5 matrix generated and transposed ON THE DEVICE (lkb_csr_random_device +
        lkb_op_csr_create_device, adopt = 1): `per_row` uniformly drawn, sorted column indices per row, normal values.
        The oracle builds the same matrix with `csr_random_host` below."""
        rp, ci, va = C.c_void_p(), C.c_void_p(), C.c_void_p()
        check(ctx.lib.lkb_csr_random_device(ctx.h, KINDS[kind], m, 0, n, per_row, seed, C.byref(rp), C.byref(ci), C.byref(va)), "csr_random")
        h = C.c_void_p()
        rc = ctx.lib.lkb_op_csr_create_device(ctx.h, KINDS[kind], m, n, rp, ci, va, 1, C.byref(h))
        if rc != 0:
            for ptr in (rp, ci, va):
                ctx.lib.lkb_dev_free(ptr)
            check(rc, "csr_create_device")
        op = cls(ctx, kind, h, m, n)
        op.row0, op.n_global = 0, n
        return op

    @classmethod
    def csr_random_dist(cls, ctx: Context, kind: str, m: int, n: int, per_row: int, seed: int) -> "LinOp":
        """The config-5 matrix ROW-SHARDED over the ranks of ctx: every rank generates its row block on its own GPU
        (same counter RNG keyed on the global row, so the global matrix equals `csr_random`'s) and hands it to
        lkb_op_csr_create_dist_device.  Collective."""
        r0, ml = partition(m, ctx.world, ctx.rank)
        c0, nl = partition(n, ctx.world, ctx.rank)
        rp, ci, va = C.c_void_p(), C.c_void_p(), C.c_void_p()
        check(ctx.lib.lkb_csr_random_device(ctx.h, KINDS[kind], ml, r0, n, per_row, seed, C.byref(rp), C.byref(ci), C.byref(va)), "csr_random")
        h = C.c_void_p()
        rc = ctx.lib.lkb_op_csr_create_dist_device(ctx.h, KINDS[kind], m, n, r0, ml, c0, nl, rp, ci, va, 1, C.byref(h))
        if rc != 0:
            for ptr in (rp, ci, va):
                ctx.lib.lkb_dev_free(ptr)
            check(rc, "csr_create_dist_device")
        op = cls(ctx, kind, h, ml, nl)
        op.row0, op.n_global = c0, n
        op.out_row0, op.m_global = r0, m
        return op

    @classmethod
    def csr_dist(cls, ctx: Context, m: int, n: int, rowptr_local, col_global, val, row_slab=None, col_slab=None) -> "LinOp":
        """Row-sharded CSR: this rank passes ITS rows (local rowptr, global column indices).  Collective."""
        kind = kind_of(val.dtype)
        r0, ml = row_slab if row_slab is not None else partition(m, ctx.world, ctx.rank)
        c0, nl = col_slab if col_slab is not None else partition(n, ctx.world, ctx.rank)
        rp = np.ascontiguousarray(rowptr_local, dtype=np.int64); ci = np.ascontiguousarray(col_global, dtype=np.int32)
        va = np.ascontiguousarray(val)
        assert rp.size == ml + 1
        h = C.c_void_p()
        check(ctx.lib.lkb_op_csr_create_dist(ctx.h, KINDS[kind], m, n, r0, ml, c0, nl, rp.ctypes.data, ci.ctypes.data,
                                             va.ctypes.data, C.byref(h)), "csr_dist")
        op = cls(ctx, kind, h, ml, nl)
        op.row0, op.n_global = c0, n            # layout of the column-space vectors
        op.out_row0, op.m_global = r0, m        # layout of the row-space vectors
        return op

    @classmethod
    def dense(cls, ctx: Context, A: np.ndarray) -> "LinOp":
        kind = kind_of(A.dtype)
        Af = np.asfortranarray(A)
        h = C.c_void_p()
        check(ctx.lib.lkb_op_dense_create(ctx.h, KINDS[kind], A.shape[0], A.shape[1], Af.ctypes.data, C.byref(h)), "dense")
        op = cls(ctx, kind, h, A.shape[0], A.shape[1])
        op.row0, op.n_global = 0, A.shape[1]
        return op

    @classmethod
    def callback(cls, ctx: Context, kind: str, m_local: int, n_local: int, fn, capturable: bool = False) -> "LinOp":
        """fn(x_ptr, y_ptr, trans, stream) -> int : a user-written device matvec."""
        cfn = _lib.MATVEC_FN(lambda user, x, y, trans, stream: int(fn(x, y, trans, stream) or 0))
        h = C.c_void_p()
        check(ctx.lib.lkb_op_callback_create(ctx.h, KINDS[kind], m_local, n_local, cfn, None, int(capturable), C.byref(h)), "callback")
        op = cls(ctx, kind, h, m_local, n_local, keep=cfn)
        op.row0, op.n_global = 0, n_local
        return op

    @classmethod
    def diag(cls, d: Vector) -> "LinOp":
        """M = diag(d): matvec d * x, rmatvec conj(d) * x, x may be y.  The values of d are copied; M has d's layout."""
        h = C.c_void_p()
        check(d.ctx.lib.lkb_op_diag_create(d.h, C.byref(h)), "diag")
        op = cls(d.ctx, d.kind, h, d.n, d.n)
        op.row0, op.n_global = d.row0, d.n_global
        return op

    @classmethod
    def jacobi(cls, A: "LinOp") -> "LinOp":
        """Jacobi preconditioner M = diag(A)^-1, built on the device: a diagonal operator with A's row layout."""
        h = C.c_void_p()
        check(A.ctx.lib.lkb_op_jacobi_create(A.h, C.byref(h)), "jacobi")
        op = cls(A.ctx, A.kind, h, A.m, A.m)
        op.row0 = getattr(A, "out_row0", A.row0)
        op.n_global = getattr(A, "m_global", A.n_global)
        return op

    @classmethod
    def chebyshev(cls, A: "LinOp", degree: int, lmin: Optional[float] = None, lmax: Optional[float] = None) -> "LinOp":
        """Chebyshev polynomial preconditioner of `degree` on D^-1 A (include/lkb.h: lkb_op_chebyshev_create), built on
        the device.  lmax None: the Gershgorin bound of D^-1 A; lmin None: lmax / 100.  Keeps A alive."""
        h = C.c_void_p()
        check(A.ctx.lib.lkb_op_chebyshev_create(A.h, int(degree), 0.0 if lmin is None else float(lmin),
                                                0.0 if lmax is None else float(lmax), C.byref(h)), "chebyshev")
        op = cls(A.ctx, A.kind, h, A.m, A.m, keep=A)
        op.row0 = getattr(A, "out_row0", A.row0)
        op.n_global = getattr(A, "m_global", A.n_global)
        return op

    @classmethod
    def polynomial(cls, A: "LinOp", roots) -> "LinOp":
        """Polynomial preconditioner M = p(A), p(z) = (1 - prod_i (1 - z / roots[i])) / z, applied in the order of `roots`
        (a complex array; in a real kind a complex root is immediately followed by its conjugate) (include/lkb.h:
        lkb_op_poly_create).  Keeps A alive."""
        th = np.ascontiguousarray(np.asarray(roots, dtype=np.complex128).ravel())
        ri = np.ascontiguousarray(np.column_stack([th.real, th.imag]).ravel())
        h = C.c_void_p()
        check(A.ctx.lib.lkb_op_poly_create(A.h, int(th.size), ri.ctypes.data_as(C.POINTER(C.c_double)), C.byref(h)), "polynomial")
        return cls._on(A, h)

    @classmethod
    def gmres_poly(cls, A: "LinOp", degree: int, seed: int = 0) -> "LinOp":
        """GMRES-polynomial preconditioner of `degree` (include/lkb.h: lkb_op_gmres_poly_create): the roots are the
        harmonic Ritz values of `degree` Arnoldi steps on A from a seeded random vector.  Collective; keeps A alive."""
        h = C.c_void_p()
        check(A.ctx.lib.lkb_op_gmres_poly_create(A.h, int(degree), int(seed), C.byref(h)), "gmres_poly")
        return cls._on(A, h)

    @classmethod
    def multigrid(cls, A: "LinOp", degree: int = 2) -> "LinOp":
        """Geometric multigrid preconditioner of a 5- / 7-point stencil (include/lkb.h: lkb_op_multigrid_create): one
        V-cycle with Chebyshev smoothing of `degree` on every level.  Keeps A alive."""
        h = C.c_void_p()
        check(A.ctx.lib.lkb_op_multigrid_create(A.h, int(degree), C.byref(h)), "multigrid")
        return cls._on(A, h)

    @classmethod
    def _on(cls, A: "LinOp", h) -> "LinOp":
        op = cls(A.ctx, A.kind, h, A.m, A.m, keep=A)
        op.row0 = getattr(A, "out_row0", A.row0)
        op.n_global = getattr(A, "m_global", A.n_global)
        return op

    def poly_roots(self) -> np.ndarray:
        """The roots of a polynomial operator in application order (complex128)."""
        n = C.c_int32()
        buf = np.zeros(2 * 256, dtype=np.float64)
        check(self.ctx.lib.lkb_op_poly_roots(self.h, 256, C.byref(n), buf.ctypes.data_as(C.POINTER(C.c_double))), "poly_roots")
        return buf[0:2 * n.value:2] + 1j * buf[1:2 * n.value:2]

    def matvec(self, x: Vector, y: Vector):
        check(self.ctx.lib.lkb_op_matvec(self.h, x.h, y.h), "matvec")

    def rmatvec(self, x: Vector, y: Vector):
        check(self.ctx.lib.lkb_op_rmatvec(self.h, x.h, y.h), "rmatvec")

    def counters(self):
        a, b = C.c_int64(), C.c_int64()
        check(self.ctx.lib.lkb_op_counters(self.h, C.byref(a), C.byref(b)))
        return a.value, b.value

    def reset_counter(self):
        check(self.ctx.lib.lkb_op_reset_counters(self.h))

    def __del__(self):
        try:
            if getattr(self, "h", None) and self.ctx.h:
                self.ctx.lib.lkb_op_destroy(self.h)
        except Exception:
            pass


def _hostmat(M: np.ndarray, kind: str):
    if not (isinstance(M, np.ndarray) and M.flags.f_contiguous and M.dtype == DTYPES[kind] and M.ndim == 2):
        raise TypeError("H/T/B must be a Fortran-ordered 2-D numpy array of the basis kind (it is updated in place)")
    return M


def arnoldi(A: LinOp, X: Basis, H: np.ndarray, kstart: int = 0, kend: int = 0, tol: float = -1.0,
            transpose: bool = False, blksize: int = 1) -> int:
    _hostmat(H, X.kind)
    info = C.c_int32()
    check(A.ctx.lib.lkb_arnoldi(A.h, X.h, H.ctypes.data, H.shape[0], C.byref(info), kstart, kend, tol,
                                int(transpose), blksize), "arnoldi")
    return info.value


def lanczos(A: LinOp, X: Basis, T: np.ndarray, kstart: int = 0, kend: int = 0, tol: float = -1.0) -> int:
    _hostmat(T, X.kind)
    info = C.c_int32()
    check(A.ctx.lib.lkb_lanczos(A.h, X.h, T.ctypes.data, T.shape[0], C.byref(info), kstart, kend, tol), "lanczos")
    return info.value


def bidiagonalization(A: LinOp, U: Basis, V: Basis, B: np.ndarray, kstart: int = 0, kend: int = 0,
                      tol: float = -1.0) -> int:
    _hostmat(B, U.kind)
    info = C.c_int32()
    check(A.ctx.lib.lkb_bidiag(A.h, U.h, V.h, B.ctypes.data, B.shape[0], C.byref(info), kstart, kend, tol), "bidiag")
    return info.value


def double_gram_schmidt_step(W: Basis, wcol0: int, p: int, X: Basis, j: int, if_chk_orthonormal: bool = True,
                             want_beta: bool = True):
    """Orthogonalise W(:, wcol0:wcol0+p) against X(:, :j) twice; returns (info, beta[j, p])."""
    beta = np.zeros((max(j, 1), p), dtype=DTYPES[X.kind], order="F")
    info = C.c_int32()
    check(X.ctx.lib.lkb_dgs_step(X.h, j, W.h, wcol0, p, int(if_chk_orthonormal),
                                 beta.ctypes.data if want_beta else None, beta.shape[0], C.byref(info)), "dgs")
    return info.value, beta[:j]


def orthogonalize_against_basis(W: Basis, wcol0: int, p: int, X: Basis, j: int, if_chk_orthonormal: bool = True):
    beta = np.zeros((max(j, 1), p), dtype=DTYPES[X.kind], order="F")
    info = C.c_int32()
    check(X.ctx.lib.lkb_orthogonalize_against_basis(X.h, j, W.h, wcol0, p, int(if_chk_orthonormal),
                                                    beta.ctypes.data, beta.shape[0], C.byref(info)), "orthogonalize")
    return info.value, beta[:j]


def qr(Q: Basis, col0: int = 0, p: Optional[int] = None, tol: float = -1.0):
    p = Q.ncols - col0 if p is None else p
    R = np.zeros((p, p), dtype=DTYPES[Q.kind], order="F")
    info = C.c_int32()
    check(Q.ctx.lib.lkb_qr(Q.h, col0, p, R.ctypes.data, p, tol, C.byref(info)), "qr")
    return info.value, R


def qr_pivoting(Q: Basis, col0: int = 0, p: Optional[int] = None, tol: float = -1.0):
    """qr(Q, R, perm, info, tol) with column pivoting (src/Krylov/qr.fypp:32-107): in place, A[:, perm] = Q R.
    Returns (info, R, perm) with perm 0-based (the C ABI / the reference return it 1-based)."""
    p = Q.ncols - col0 if p is None else p
    R = np.zeros((p, p), dtype=DTYPES[Q.kind], order="F")
    perm = np.zeros(p, dtype=np.int32)
    info = C.c_int32()
    check(Q.ctx.lib.lkb_qr_pivoting(Q.h, col0, p, R.ctypes.data, p, perm.ctypes.data_as(C.POINTER(C.c_int32)), tol,
                                    C.byref(info)), "qr_pivoting")
    return info.value, R, perm.astype(np.int64) - 1


def _wrap_precond(preconditioner):
    """preconditioner(vec_ptr, n_local, iter, current_residual, target_residual, stream) -> None/int
    (a host callback; a LinOp preconditioner goes to the *_precond_op entry points instead)"""
    return _lib.PRECOND_FN(lambda user, v, n, it, cur, tgt, stream: int(preconditioner(v, n, it, cur, tgt, stream) or 0))


def gmres(A: LinOp, b: Vector, x: Vector, rtol: float = -1.0, atol: float = -1.0, kdim: int = 30,
          maxiter: int = 10, transpose: bool = False, preconditioner=None):
    cap = (kdim + 2) * (maxiter + 2) + 8
    res = (C.c_double * cap)()
    io = _lib.GmresIO(kdim=kdim, maxiter=maxiter, res=res, res_cap=cap)
    info = C.c_int32()
    if preconditioner is None:
        check(A.ctx.lib.lkb_gmres(A.h, b.h, x.h, C.byref(info), rtol, atol, int(transpose), C.byref(io)), "gmres")
    elif isinstance(preconditioner, LinOp):
        check(A.ctx.lib.lkb_gmres_precond_op(A.h, b.h, x.h, C.byref(info), rtol, atol, int(transpose), C.byref(io),
                                             preconditioner.h), "gmres")
    else:
        cb = _wrap_precond(preconditioner)
        check(A.ctx.lib.lkb_gmres_precond(A.h, b.h, x.h, C.byref(info), rtol, atol, int(transpose), C.byref(io),
                                          cb, None), "gmres")
    meta = dict(n_iter=io.n_iter, n_inner=io.n_inner, n_outer=io.n_outer, converged=bool(io.converged),
                info=io.info, res=[res[i] for i in range(min(io.res_len, cap))])
    return info.value, meta


def fgmres(A: LinOp, b: Vector, x: Vector, rtol: float = -1.0, atol: float = -1.0, kdim: int = 30,
           maxiter: int = 10, transpose: bool = False, preconditioner=None):
    """Flexible GMRES (GMRES/fgmres.fypp): same options / metadata as gmres.  The preconditioner is a callable: fgmres
    exists for preconditioners that change between inner steps, and with a fixed operator it is gmres."""
    if isinstance(preconditioner, LinOp):
        raise TypeError("fgmres takes a callable preconditioner; pass a LinOp preconditioner to gmres")
    cap = (kdim + 2) * (maxiter + 2) + 8
    res = (C.c_double * cap)()
    io = _lib.GmresIO(kdim=kdim, maxiter=maxiter, res=res, res_cap=cap)
    info = C.c_int32()
    cb = _wrap_precond(preconditioner) if preconditioner is not None else C.cast(None, _lib.PRECOND_FN)
    check(A.ctx.lib.lkb_fgmres(A.h, b.h, x.h, C.byref(info), rtol, atol, int(transpose), C.byref(io), cb, None), "fgmres")
    meta = dict(n_iter=io.n_iter, n_inner=io.n_inner, n_outer=io.n_outer, converged=bool(io.converged),
                info=io.info, res=[res[i] for i in range(min(io.res_len, cap))])
    return info.value, meta


def cg(A: LinOp, b: Vector, x: Vector, rtol: float = -1.0, atol: float = -1.0, maxiter: int = 100,
       preconditioner=None):
    cap = maxiter + 8
    res = (C.c_double * cap)()
    io = _lib.CgIO(maxiter=maxiter, res=res, res_cap=cap)
    info = C.c_int32()
    if preconditioner is None:
        check(A.ctx.lib.lkb_cg(A.h, b.h, x.h, C.byref(info), rtol, atol, C.byref(io)), "cg")
    elif isinstance(preconditioner, LinOp):
        check(A.ctx.lib.lkb_cg_precond_op(A.h, b.h, x.h, C.byref(info), rtol, atol, C.byref(io), preconditioner.h), "cg")
    else:
        cb = _wrap_precond(preconditioner)
        check(A.ctx.lib.lkb_cg_precond(A.h, b.h, x.h, C.byref(info), rtol, atol, C.byref(io), cb, None), "cg")
    meta = dict(n_iter=io.n_iter, converged=bool(io.converged), info=io.info,
                res=[res[i] for i in range(min(io.res_len, cap))])
    return info.value, meta


def set_lapack_from_scipy() -> None:
    """Point the host k x k algebra (geev/gees/trsen/syev/gesvd) at scipy's bundled OpenBLAS."""
    import glob, os, scipy
    root = os.path.dirname(os.path.dirname(scipy.__file__))
    cands = glob.glob(os.path.join(root, "scipy.libs", "libscipy_openblas*.so"))
    if not cands:
        raise LkbError("no libscipy_openblas found for the host LAPACK provider")
    check(_lib.load().lkb_set_lapack(cands[0].encode(), b"scipy_", b"_"), "set_lapack")


def eigs(A: LinOp, X: Basis, nev: int, x0: Optional[Vector] = None, kdim: int = 0, tolerance: float = -1.0,
         transpose: bool = False):
    eigvals = np.zeros(nev, dtype=np.complex128); residuals = np.zeros(nev)
    info = C.c_int32()
    check(A.ctx.lib.lkb_eigs(A.h, X.h, nev, eigvals.ctypes.data_as(C.POINTER(C.c_double)),
                             residuals.ctypes.data_as(C.POINTER(C.c_double)), C.byref(info),
                             x0.h if x0 is not None else None, kdim, tolerance, int(transpose)), "eigs")
    return eigvals, residuals, info.value


def eighs(A: LinOp, X: Basis, nev: int, x0: Optional[Vector] = None, kdim: int = 0, tolerance: float = -1.0):
    eigvals = np.zeros(nev); residuals = np.zeros(nev)
    info = C.c_int32()
    check(A.ctx.lib.lkb_eighs(A.h, X.h, nev, eigvals.ctypes.data_as(C.POINTER(C.c_double)),
                              residuals.ctypes.data_as(C.POINTER(C.c_double)), C.byref(info),
                              x0.h if x0 is not None else None, kdim, tolerance), "eighs")
    return eigvals, residuals, info.value


def svds(A: LinOp, U: Basis, V: Basis, nsv: int, u0: Optional[Vector] = None, kdim: int = 0, tolerance: float = -1.0):
    S = np.zeros(nsv); residuals = np.zeros(nsv)
    info = C.c_int32()
    check(A.ctx.lib.lkb_svds(A.h, U.h, S.ctypes.data_as(C.POINTER(C.c_double)), V.h, nsv,
                             residuals.ctypes.data_as(C.POINTER(C.c_double)), C.byref(info),
                             u0.h if u0 is not None else None, kdim, tolerance), "svds")
    return S, residuals, info.value


def initialize_krylov_subspace(X: Basis, X0: Optional[Basis] = None, p0: Optional[int] = None) -> None:
    """initialize_krylov_subspace(X [, X0]) (src/Krylov/utilities.fypp:32-46, BaseKrylov.fypp:490-517): zero X, copy the
    p0 starting vectors into X(:p0) and orthonormalise them."""
    if X0 is None:
        check(X.ctx.lib.lkb_initialize_krylov_subspace(X.h, None, 0, 0), "initialize_krylov_subspace")
    else:
        check(X.ctx.lib.lkb_initialize_krylov_subspace(X.h, X0.h, 0, X0.ncols if p0 is None else p0), "initialize_krylov_subspace")


def initialize_random_orthonormal_basis(X: Basis, col0: int = 0, p: Optional[int] = None) -> None:
    """utilities.fypp:52-62"""
    check(X.ctx.lib.lkb_initialize_random_orthonormal_basis(X.h, col0, X.ncols - col0 if p is None else p), "initialize_random_orthonormal_basis")


def kexpm(c: Vector, A: LinOp, b: Vector, tau: float, tol: float, trans: bool = False, kdim: int = 0) -> int:
    """kexpm_vec(c, A, b, tau, tol, info, trans, kdim)  (src/Expm/ExpmLib.fypp:128-232): c = exp(tau A) b; returns info."""
    info = C.c_int32()
    check(A.ctx.lib.lkb_kexpm_vec(c.h, A.h, b.h, float(tau), float(tol), C.byref(info), int(trans), int(kdim)), "kexpm_vec")
    return info.value


def kexpm_mat(Cb: Basis, A: LinOp, B: Basis, tau: float, tol: float, trans: bool = False, kdim: int = 0, p: Optional[int] = None) -> int:
    """kexpm_mat(C, A, B, tau, tol, info, trans, kdim)  (src/Expm/ExpmLib.fypp:234-362): C = exp(tau A) B by block Arnoldi with
    blksize p = size(B); returns info (dimension used, or -1)."""
    p = B.ncols if p is None else p
    info = C.c_int32()
    check(A.ctx.lib.lkb_kexpm_mat(Cb.h, A.h, B.h, int(p), float(tau), float(tol), C.byref(info), int(trans), int(kdim)), "kexpm_mat")
    return info.value


def krylov_exptA(vec_out: Vector, A: LinOp, vec_in: Vector, tau: float, trans: bool = False) -> int:
    """krylov_exptA (src/Expm/ExpmLib.fypp:364-392): kexpm_vec with tol = atol_kind and kdim = 30; returns info."""
    info = C.c_int32()
    check(A.ctx.lib.lkb_krylov_expta(vec_out.h, A.h, vec_in.h, float(tau), C.byref(info), int(trans)), "krylov_exptA")
    return info.value


def write_results(filename: str, vals: np.ndarray, res: np.ndarray, tol: float) -> np.ndarray:
    """write_results (IterativeSolvers.fypp:882-924); returns the residuals in the sorted order the reference leaves them in."""
    v = np.ascontiguousarray(vals)
    cplx = np.iscomplexobj(v)
    vv = np.ascontiguousarray(v.astype(np.complex128).view(np.float64) if cplx else v.astype(np.float64))
    rr = np.ascontiguousarray(res, dtype=np.float64).copy()
    check(_lib.load().lkb_write_results(filename.encode(), int(cplx), vv.ctypes.data_as(C.POINTER(C.c_double)),
                                   rr.ctypes.data_as(C.POINTER(C.c_double)), int(rr.size), float(tol)), "write_results")
    return rr


def save_eigenspectrum(lam: np.ndarray, residuals: np.ndarray, fname: str) -> None:
    """save_eigenspectrum (IterativeSolvers.fypp:941-960): .npy, k x 3 (Re, Im, residual) or k x 2 (value, residual)."""
    v = np.ascontiguousarray(lam)
    cplx = np.iscomplexobj(v)
    single = v.dtype in (np.float32, np.complex64)
    vv = np.ascontiguousarray(v.astype(np.complex128).view(np.float64) if cplx else v.astype(np.float64))
    rr = np.ascontiguousarray(residuals, dtype=np.float64)
    check(_lib.load().lkb_save_eigenspectrum(fname.encode(), int(cplx), int(single), vv.ctypes.data_as(C.POINTER(C.c_double)),
                                        rr.ctypes.data_as(C.POINTER(C.c_double)), int(rr.size)), "save_eigenspectrum")


def krylov_schur(X: Basis, H: np.ndarray, kdim: int) -> int:
    _hostmat(H, X.kind)
    n = C.c_int32()
    check(X.ctx.lib.lkb_krylov_schur(X.h, H.ctypes.data, H.shape[0], kdim, C.byref(n)), "krylov_schur")
    return n.value
