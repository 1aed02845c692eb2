"""High-precision restatements shared by the kernel tests (test_gpu_block_kernels.py, test_gpu_cgs2_kernels.py).

References run in float64 for s / c and in np.longdouble for d / z (a compensated Dot2 where longdouble is no wider than
double).  The tables give each kind's pack width, element sizes and unit roundoff as the kernels see them."""
import math

import numpy as np

KINDS = ["s", "d", "c", "z"]
EPP = {"s": 4, "d": 2, "c": 2, "z": 1}                     # elements per 16-byte pack (lkb_types.cuh: Tr<K>::EPP)
ESZ = {"s": 4, "d": 8, "c": 8, "z": 16}                    # sizeof(E)
WSZ = {"s": 8, "d": 8, "c": 16, "z": 16}                   # sizeof(W): the accumulators are double / double2
CPLX = {"s": False, "d": False, "c": True, "z": True}
U = {"s": 2.0 ** -24, "d": 2.0 ** -53, "c": 2.0 ** -24, "z": 2.0 ** -53}
DT = {"s": np.float32, "d": np.float64, "c": np.complex64, "z": np.complex128}
MD_THREADS = 256                                           # lkb_kernels.h
B200_SMS, B200_OPTIN = 148, 232448                         # used when no device is present (CPU rehearsal)


def device_shape():
    """(SM count, opt-in shared memory per block) of device 0, or the B200's values without a device."""
    try:
        import torch
        if torch.cuda.is_available():
            p = torch.cuda.get_device_properties(0)
            return p.multi_processor_count, p.shared_memory_per_block_optin
    except Exception:
        pass
    return B200_SMS, B200_OPTIN


# ---- high-precision arithmetic ---------------------------------------------------------------------------------------
LD_WIDER = np.finfo(np.longdouble).eps < np.finfo(np.float64).eps


def hp(kind, a):
    """a in the reference precision: float64 / complex128 for s / c, longdouble for d / z."""
    if kind in "sc":
        return np.asarray(a, dtype=np.complex128 if CPLX[kind] else np.float64)
    return np.asarray(a, dtype=np.clongdouble if CPLX[kind] else np.longdouble)


def _two_prod(a, b):
    """Dekker / Veltkamp: a * b = p + e exactly (float64)."""
    p = a * b
    sp = 134217729.0
    ah = a * sp; ah = ah - (ah - a); al = a - ah
    bh = b * sp; bh = bh - (bh - b); bl = b - bh
    return p, ((ah * bh - p) + ah * bl + al * bh) + al * bl


def _dot2_real(A, B):
    """A^T B with Ogita-Rump-Oishi Dot2 per entry (error ~ u^2 cond + u): products split exactly, sums by fsum."""
    out = np.empty((A.shape[1], B.shape[1]))
    for i in range(A.shape[1]):
        for j in range(B.shape[1]):
            p, e = _two_prod(A[:, i], B[:, j])
            out[i, j] = math.fsum(np.concatenate([p, e]))
    return out


def _blocks(n):
    """Side of the three-level split of a sum over n rows (see matmul_h)."""
    return max(1, math.ceil(round(n ** (1.0 / 3.0), 9)))


def sum_depth(kind, n):
    """Rounding depth of the reference's sums over n rows: BLAS (float64, any order) for s / c, the three-level split for
    d / z (longdouble carries only 11 more bits than double, so a plain n-term chain would cost them at n = 10^6)."""
    return n if kind in "sc" else 3 * _blocks(n)


def matmul_h(kind, A, B):
    """A^H B in the reference precision.  In longdouble the rows are summed in three nested levels of <= n^(1/3)."""
    if kind in "sc":
        return hp(kind, A).conj().T @ hp(kind, B)
    if LD_WIDER:
        A, B = hp(kind, A), hp(kind, B)
        n = A.shape[0]
        b = _blocks(n)
        pad = b ** 3 - n
        if pad:
            A = np.concatenate([A, np.zeros((pad, A.shape[1]), A.dtype)])
            B = np.concatenate([B, np.zeros((pad, B.shape[1]), B.dtype)])
        P = np.einsum("xyzi,xyzj->xyij", A.conj().reshape(b, b, b, -1), B.reshape(b, b, b, -1))
        for _ in range(2):
            acc = P[0].copy()
            for t in range(1, P.shape[0]):
                acc += P[t]
            P = acc
        return P
    A = np.asarray(A, np.complex128 if CPLX[kind] else np.float64); B = np.asarray(B, A.dtype)
    if not CPLX[kind]:
        return _dot2_real(A, B)
    ar, ai, br, bi = A.real, A.imag, B.real, B.imag      # conj(a) b = (ar br + ai bi) + i (ar bi - ai br)
    re = _dot2_real(np.vstack([ar, ai]), np.vstack([br, bi]))
    im = _dot2_real(np.vstack([ar, -ai]), np.vstack([bi, br]))
    return re + 1j * im


def matmul(kind, A, B):
    """A B in the reference precision."""
    if kind in "sc" or LD_WIDER:
        return hp(kind, A) @ hp(kind, B)
    return matmul_h(kind, np.conj(np.asarray(A)).T, B)
