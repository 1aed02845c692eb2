"""Block Gram-Schmidt (k_multidot2 / k_multiaxpy2) and the basis GEMM (k_basis_gemm_dmma, k_basis_gemm<K,PB>) against
high-precision restatements of what they compute, at the shapes where their index arithmetic changes regime, and the
shared-memory limits of every launcher whose dynamic shared memory grows with j or k.

Shapes follow the launchers (kernels_gs.cu, kernels_gemm.cu) and the device's SM count; every case asserts the regime it
is meant to reach.  References run in float64 for s / c and in np.longdouble for d / z (a compensated Dot2 where
longdouble is no wider than double).  Every entry is checked against a componentwise bound kappa * u * (|X|^T |w| ...),
with kappa argued next to each bound, and the reduction cases are built so that dropping the rows of one CTA, its first or
last row, or a ragged tail row moves the reference by more than 100 tolerances (test_block_cases_are_sensitive)."""
import numpy as np
import pytest

from kernel_ref import CPLX, EPP, ESZ, KINDS, MD_THREADS, U, WSZ, device_shape, hp, matmul, matmul_h, sum_depth

WEIGHT = 256.0                                             # weight of the rows the sensitivity check watches


# ---- the launchers' formulas -------------------------------------------------------------------------------------------
def md2_partition(kind, n, sms):
    """multidot2_t (kernels_gs.cu: nb = min(2 SMs, ntiles)) and k_multidot2 (tper = ceil(ntiles / nb), CTA b owns tiles
    [b tper, (b + 1) tper) of MD_THREADS packs): each CTA's row range, and the ragged tail rows done by CTA 0's thread 0."""
    e = EPP[kind]
    npk = n // e
    ntiles = -(-npk // MD_THREADS)
    nb = max(1, min(2 * sms, ntiles))
    tper = -(-ntiles // nb)
    ranges = []
    for b in range(nb):
        t0, t1 = b * tper, min(ntiles, (b + 1) * tper)
        ranges.append((min(t0 * MD_THREADS, npk) * e, min(t1 * MD_THREADS, npk) * e) if t0 < t1 else None)
    return ranges, list(range(npk * e, n)), tper


def ma2_passes(kind, n, sms):
    """Grid-stride passes of k_multiaxpy2 (multiaxpy2_t: nb = min(ceil(npk / 256), 4 SMs))."""
    npk = n // EPP[kind]
    nb = max(1, min(-(-npk // 256), 4 * sms))
    return -(-npk // (nb * 256))


def md2_smem(kind, j):       # multidot2_t: (MD_THREADS / 32) * 2 * (j + 1) * sizeof(W)
    return 8 * 2 * (j + 1) * WSZ[kind]


def md_smem(kind, j):        # multidot_t: (MD_THREADS / 32) * (j + 1) * sizeof(W)
    return 8 * (j + 1) * WSZ[kind]


def ma_smem(kind, j):        # multiaxpy_t / multiaxpy_fin_t: j * sizeof(E)
    return max(j, 1) * ESZ[kind]


def gemm_pb(kind):           # gemm_t: PB = 16 real / 8 complex output columns per sweep
    return 8 if CPLX[kind] else 16


def gemm_smem(kind, k):      # gemm_t: k * PB * sizeof(E)
    return k * gemm_pb(kind) * ESZ[kind]


def dmma_runs(kind, k, nk):
    """launch_basis_gemm: rdp with p >= 8 goes to gemm_dmma, which declines when its shared memory
    ((kpad * 68 + 3 * 8 * 260) * 8 B, kpad = k rounded up to 8) passes 220 KB: k > 320."""
    kpad = -(-k // 8) * 8
    return kind == "d" and nk >= 8 and (kpad * 68 + 3 * 8 * 260) * 8 <= 220 * 1024


def ks_chunk(kind, n, nk):
    """lkb_eig.cu:335-337 -- the rows per staging chunk of lkb_krylov_schur."""
    chunk = (1 << 30) // (nk * ESZ[kind])
    chunk = max(4096, (chunk // 4096) * 4096)
    return min(chunk, ((n + 4095) // 4096) * 4096)


# ---- (a) one block Gram-Schmidt step -----------------------------------------------------------------------------------
def block_cases(sms, optin):
    """(id, kind, p, k, n): arnoldi(kstart = kend = k, blksize = p) orthogonalises the block X(:, kp : kp + p), kp = k p."""
    cases = []
    for kind in KINDS:
        for p in (2, 3, 4):
            cases.append((f"{kind}-p{p}-onecta", kind, p, 2, 2 * p + 6))
            cases.append((f"{kind}-p{p}-n4099", kind, p, 3, 4099))
        # ntiles = 2 SMs + 1: the grid is 2 SMs CTAs of tper = 2 tiles, so the upper half owns none
        e = EPP[kind]
        n_idle = (2 * sms * MD_THREADS + 1) * e + (e - 1)
        for p in (2, 3):
            cases.append((f"{kind}-p{p}-idlectas", kind, p, 132 // p, n_idle))
        for kp, p in ((2, 2), (16, 4), (18, 3)):
            cases.append((f"{kind}-kp{kp}-n1000003", kind, p, kp // p, 1000003))
    # k_multidot2's old attribute (100 KB): the last j that fitted and the first that did not
    for kind, j_ok, j_bad in (("d", 799, 800), ("z", 399, 400)):
        assert md2_smem(kind, j_ok) <= 100 * 1024 < md2_smem(kind, j_bad)
        p_ok = next(p for p in range(2, 64) if j_ok % p == 0)
        cases.append((f"{kind}-kp{j_ok}-oldlimit-fits", kind, p_ok, j_ok // p_ok, 4099))
        cases.append((f"{kind}-kp{j_bad}-oldlimit-failed", kind, 2, j_bad // 2, 4099))
        # past the device's limit: the pairs take the per-column path
        kp = optin // (16 * WSZ[kind])
        kp += kp % 2
        assert md2_smem(kind, kp) > optin
        cases.append((f"{kind}-kp{kp}-pastdevice", kind, 2, kp // 2, 4099))
    return cases


def block_inputs(kind, p, k, n, sms, seed=0):
    """X(:, :kp + p) with X(:, :kp) orthonormal (host QR, cast to the kind) and the diagonal d of A (powers of two, so that
    A x is exact in every kind).  The rows the sensitivity check watches -- the ragged tail and the first and last row of
    every CTA's range -- carry weight WEIGHT in the columns of the block being orthogonalised (spread round-robin over the
    p columns), so that each of them holds a visible share of the block's entries after the QR."""
    kp = k * p
    rng = np.random.default_rng(seed + 7 * n + 131 * kp + p)
    X0 = rng.standard_normal((n, kp))
    if CPLX[kind]:
        X0 = X0 + 1j * rng.standard_normal((n, kp))
    ranges, tail, _ = md2_partition(kind, n, sms)
    watch = sorted(set(tail) | {r for rg in ranges if rg for r in (rg[0], rg[1] - 1)})
    for i, r in enumerate(watch):
        X0[r, kp - p + i % p] += WEIGHT * (1 if i % 3 else -1)
    Q, _ = np.linalg.qr(X0)
    X = np.zeros((n, kp + p), dtype={"s": np.float32, "d": np.float64, "c": np.complex64, "z": np.complex128}[kind], order="F")
    X[:, :kp] = Q
    d = np.ldexp(1.0, rng.integers(-2, 3, n)).astype(X.dtype)
    d[watch] = 4
    return X, d, watch


def block_reference(kind, X, d, kp, p):
    """The literal step in high precision: W = A X(:, kp - p : kp); two-pass classical Gram-Schmidt against X(:, :kp)
    (c1 = X^H W, W' = W - X c1, c2 = X^H W', W'' = W' - X c2, H = c1 + c2), then qr_no_pivoting of W'' column by column
    (two-pass Gram-Schmidt against the previous columns, R(j, j) = ||q||, q / R(j, j)).  Also the scales of the bounds."""
    V = X[:, :kp]
    W = d[:, None] * X[:, kp - p:kp]                       # exact in the kind
    C1 = matmul_h(kind, V, W)
    W1 = hp(kind, W) - matmul(kind, V, C1)
    C2 = matmul_h(kind, V, W1)
    W2 = W1 - matmul(kind, V, C2)
    Q = W2.copy()
    R = np.zeros((p, p), dtype=Q.dtype)
    for j in range(p):
        q = Q[:, j]
        a = Q[:, :j].conj().T @ q; q = q - Q[:, :j] @ a
        b = Q[:, :j].conj().T @ q; q = q - Q[:, :j] @ b
        R[:j, j] = a + b
        R[j, j] = np.sqrt(np.real(np.vdot(q, q)))
        Q[:, j] = q / R[j, j]
    aV = np.abs(hp(kind, V)); aW = np.abs(hp(kind, W))
    scale_w = aW + aV @ (np.abs(C1) + np.abs(C2))          # |W| + |X| (|c1| + |c2|): what the two updates round against
    return dict(H=C1 + C2, C1=C1, R=R, Q=Q, W=W, aV=aV, scale_w=scale_w)


def block_kappa(kind, n, kp, p, sms):
    """kappa of the step's bounds.  The multi-dot sums, per entry, EPP products and a 5-level warp fold in the kind; then,
    in double, <= tper tiles, 8 warps and the two-level tree over <= 2 SMs CTAs (16 + 64 rows).  For s / c the double
    sums are 2^29 times finer than u and count once; for d / z they are in the kind: depth m.  Each of the two updates is
    an FMA chain over kp terms in the kind, the QR adds chains over < p terms, and H, R are rounded to the kind once:
    kappa = 2 (kp + p + 2) + m."""
    _, _, tper = md2_partition(kind, n, sms)
    m = EPP[kind] + 6 + (tper + 8 + 80 if kind in "dz" else 1)
    return 2 * (kp + p + 2) + m


def block_tolerances(kind, ref, kp, p, kappa):
    """Componentwise bounds kappa u (...):
       H(:kp)  : |X|^T (|W| + |X||c1|) + |c1|     (c1's error cancels in c1 + c2 up to the update's rounding, which c2
                                                  sees through |X|^T; + the narrowing of c1 and of H to the kind)
       R, Q    : the QR of W'' perturbed by dW'' <= kappa u scale_w: |dR| <= |Q|^T (scale_w + |Q||R|),
                 |dQ| <= (scale_w + |Q||R|) |R^-1|."""
    u = U[kind]
    aV = ref["aV"]
    tH = kappa * u * (aV.T @ (np.abs(hp(kind, ref["W"])) + aV @ np.abs(ref["C1"])) + np.abs(ref["C1"]))
    aQ, aR = np.abs(ref["Q"]), np.abs(ref["R"])
    base = ref["scale_w"] + aQ @ aR
    tR = kappa * u * (aQ.T @ base)
    Rinv = np.linalg.inv(np.asarray(ref["R"], dtype=np.complex128 if CPLX[kind] else np.float64))
    tQ = kappa * u * (base @ hp(kind, np.abs(Rinv)))
    return tH, tR, tQ


def sensitivity(kind, X, d, kp, p, tH, n, sms):
    """For each watched row set, max |reference moved by dropping it| / tolerance over the block's H entries."""
    ranges, tail, _ = md2_partition(kind, n, sms)
    V = X[:, :kp]
    W = d[:, None] * X[:, kp - p:kp]
    sets = [("tail", [r]) for r in tail]
    for b, rg in enumerate(ranges):
        if rg is None:
            continue
        sets += [(f"cta{b}.first", [rg[0]]), (f"cta{b}.last", [rg[1] - 1]), (f"cta{b}.all", slice(rg[0], rg[1]))]
    out = {}
    for name, rows in sets:
        delta = matmul_h(kind, V[rows], W[rows])
        out[name] = float(np.max(np.abs(delta) / tH))
    return out


# ---- (b) the basis GEMM through krylov_schur --------------------------------------------------------------------------------
def gemm_cases():
    """(id, kind, n, k).  nk (the Schur vectors kept) is ~k/2 by the median selector; the test asserts the regime."""
    cases = [("d-dmma-n200-k140", "d", 200, 140), ("d-dmma-n512-k140", "d", 512, 140), ("d-dmma-n513-k140", "d", 513, 140),
             ("d-dmma-n768-k320", "d", 768, 320), ("d-dmma-n769-k320", "d", 769, 320),
             ("d-fma-k321", "d", 1001, 321), ("d-fma-nk-lt-8", "d", 4099, 10)]
    cases += [(f"{kind}-{'dmma' if kind == 'd' else 'fma'}-n4099-k37", kind, 4099, 37) for kind in KINDS]
    cases += [(f"{kind}-fma-n1000003-k37", kind, 1000003, 37) for kind in ("s", "c")]
    for kind in ("d", "z"):                               # the old 160 KB attribute: k = 1280 fitted, 1281 did not
        assert gemm_smem(kind, 1280) <= 160 * 1024 < gemm_smem(kind, 1281)
        cases += [(f"{kind}-k1280-oldlimit-fits", kind, 1280 + 67, 1280), (f"{kind}-k1281-oldlimit-failed", kind, 1281 + 67, 1281)]
    return cases


def gemm_inputs(kind, n, k, seed=0):
    rng = np.random.default_rng(seed + n + 17 * k)
    dt = {"s": np.float32, "d": np.float64, "c": np.complex64, "z": np.complex128}[kind]
    X = np.zeros((n, k + 1), dtype=dt, order="F")
    X[:k, :k] = np.eye(k)
    R = rng.standard_normal((n - k, k)) + (1j * rng.standard_normal((n - k, k)) if CPLX[kind] else 0)
    X[k:, :k] = R
    X[:, k] = rng.standard_normal(n) + (1j * rng.standard_normal(n) if CPLX[kind] else 0)
    H = np.triu(rng.standard_normal((k + 1, k)) + (1j * rng.standard_normal((k + 1, k)) if CPLX[kind] else 0), -1)
    return X, np.asfortranarray(H.astype(dt))


def check_gemm_result(kind, X, Xn, k, nk, rows=None):
    """X_new(:k, :nk) is the Z the kernel used (1 z + exact zeros); every row of X_new(k:, :nk) against R Z, the kept
    column moved bitwise, the rest zero.  kappa = k + 4: one FMA chain over k terms per entry (the FMA kernel in the kind,
    DMMA in fp64), ragged k and the zero padding add exact zeros, + the store."""
    Z = Xn[:k, :nk]
    u = U[kind]
    G = matmul_h(kind, Z, Z)
    assert np.max(np.abs(G - np.eye(nk))) < 8 * k * (u if kind in "dz" else 2.0 ** -24)
    rows = np.arange(k, X.shape[0]) if rows is None else rows
    R = X[rows, :k]
    ref = matmul(kind, R, Z)
    tol = (k + 4) * u * (np.abs(hp(kind, R)) @ np.abs(hp(kind, Z)))
    err = np.abs(hp(kind, Xn[rows, :nk]) - ref)
    bad = np.argwhere(err > tol)
    assert bad.size == 0, f"{len(bad)} entries out of bound, first row {rows[bad[0][0]]} col {bad[0][1]}"


# ---- (d) the CPU rehearsal -------------------------------------------------------------------------------------------------
def test_block_cases_are_sensitive():
    """Builds every (a) case's inputs and reference without a device, checks that each case reaches its regime, and that
    dropping any watched row (ragged tail, first / last row of a CTA's range) or a whole CTA's range moves the reference
    by more than 100 tolerances, with the reference's own error below 1/100 of the tolerance."""
    sms, optin = device_shape()
    for cid, kind, p, k, n in block_cases(sms, optin):
        kp = k * p
        ranges, tail, tper = md2_partition(kind, n, sms)
        if "onecta" in cid:
            assert len(ranges) == 1
        if "idlectas" in cid:
            assert tper == 2 and ranges[-1] is None and kp == 132
        if "1000003" in cid:
            assert (tail or kind == "z") and ma2_passes(kind, n, sms) >= 2 and len([r for r in ranges if r]) > sms
        if kp > 500 or n > 400000 and kind in "dz":
            continue                                      # the big references are exercised on the device run
        X, d, _ = block_inputs(kind, p, k, n, sms)
        ref = block_reference(kind, X, d, kp, p)
        kappa = block_kappa(kind, n, kp, p, sms)
        tH, tR, tQ = block_tolerances(kind, ref, kp, p, kappa)
        depth = sum_depth(kind, n) + 2 * kp + 4
        ref_err = depth * np.finfo(np.float64 if kind in "sc" else np.longdouble).eps * (ref["aV"].T @ ref["scale_w"])
        assert np.all(ref_err < tH / 100), cid
        sens = sensitivity(kind, X, d, kp, p, tH, n, sms)
        weak = {s: v for s, v in sens.items() if v <= 100}
        assert not weak, (cid, sorted(weak.items())[:5])


# ---- device tests ------------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def lk():
    import lightkrylov_b200 as lk
    lk.set_lapack_from_scipy()
    return lk


@pytest.fixture(scope="module")
def ctx(lk):
    c = lk.Context(0)
    yield c
    c.close()


def expected_launches(kind, n, kp, p, pairs):
    """Per-class launches of one block step: arnoldi_block (lkb_krylov.cu) then lkb_qr of the block.  A pair is 2 multi-dots
    + 2 multi-axpys; a single column is dgs_enqueue (multi-dot, fused axpy+dot when axpy_dot_ok allows it -- j <= 128,
    n % EPP == 0, n >= 32 EPP -- else multi-axpy + multi-dot, k_gsinfo, multi-axpy); the QR adds one dgs_enqueue with norm
    per column (column 0: one multi-dot for its norm) and one k_scal."""
    c = dict(matvec=p, multidot=0, multiaxpy=0, other=0, fused_axpy_dot=0)
    fused = lambda j: 1 <= j <= 128 and n % EPP[kind] == 0 and n >= 32 * EPP[kind]

    def dgs(j):
        if j == 0:
            c["multidot"] += 1
            return
        c["multidot"] += 1
        if fused(j):
            c["fused_axpy_dot"] += 1
        else:
            c["multiaxpy"] += 1; c["multidot"] += 1
        c["other"] += 1; c["multiaxpy"] += 1
    i = 0
    while i < p:
        if pairs and i + 1 < p:
            c["multidot"] += 2; c["multiaxpy"] += 2; i += 2
        else:
            dgs(kp); i += 1
    for j in range(p):
        dgs(j); c["other"] += 1
    return c


def run_block_step(lk, ctx, kind, X, d, k, p):
    n = X.shape[0]
    Xd = lk.Basis(ctx, kind, n, X.shape[1]).put(X)
    A = lk.LinOp.diag(lk.Vector(ctx, kind, n).put(d))
    H = np.zeros((X.shape[1], k * p), dtype=X.dtype, order="F")
    ctx.set_profile(True)
    try:
        info = lk.arnoldi(A, Xd, H, kstart=k, kend=k, blksize=p)
        prof = {c: v for c, (_, v) in ctx.get_profile().items()}
    finally:
        ctx.set_profile(False)
    return info, Xd.get(), H, prof


@pytest.mark.gpu
@pytest.mark.parametrize("case", block_cases(*device_shape()), ids=lambda c: c[0])
def test_block_gram_schmidt_step(lk, ctx, case):
    cid, kind, p, k, n = case
    sms, optin = device_shape()
    kp = k * p
    X, d, _ = block_inputs(kind, p, k, n, sms)
    info, Xn, H, prof = run_block_step(lk, ctx, kind, X, d, k, p)
    assert info == 0
    ref = block_reference(kind, X, d, kp, p)
    tH, tR, tQ = block_tolerances(kind, ref, kp, p, block_kappa(kind, n, kp, p, sms))
    blk = slice(kp - p, kp)
    eH = np.abs(hp(kind, H[:kp, blk]) - ref["H"])
    assert np.all(eH <= tH), (cid, float(np.max(eH / tH)))
    eR = np.abs(hp(kind, H[kp:kp + p, blk]) - ref["R"])
    assert np.all(eR <= tR), (cid, float(np.max(eR / tR)))
    assert np.all(np.real(np.diag(H[kp:kp + p, blk])) > 0) and not np.any(np.imag(np.diag(H[kp:kp + p, blk])))
    eQ = np.abs(hp(kind, Xn[:, kp:kp + p]) - ref["Q"])
    assert np.all(eQ <= tQ), (cid, float(np.max(eQ / tQ)))
    orth = np.abs(matmul_h(kind, X[:, :kp], Xn[:, kp:kp + p]))          # X(:kp)^H Q_ref is zero up to the reference's error
    assert np.all(orth <= ref["aV"].T @ (tQ + block_kappa(kind, n, kp, p, sms) * U[kind] * np.abs(ref["Q"]))), cid
    assert np.array_equal(Xn[:, :kp], X[:, :kp])
    # which path ran
    pairs = md2_smem(kind, kp) <= optin
    assert pairs == ("pastdevice" not in cid)
    if pairs:
        assert md2_smem(kind, kp) <= optin - 1024           # far from the static-memory band of the limit
    assert prof == expected_launches(kind, n, kp, p, pairs), cid
    # determinism: the same inputs give the same bits
    info2, Xn2, H2, _ = run_block_step(lk, ctx, kind, X, d, k, p)
    assert info2 == 0 and np.array_equal(Xn2, Xn) and np.array_equal(H2, H)


@pytest.mark.gpu
@pytest.mark.parametrize("case", gemm_cases(), ids=lambda c: c[0])
def test_basis_gemm_through_krylov_schur(lk, ctx, oracle, case):
    cid, kind, n, k = case
    X, H = gemm_inputs(kind, n, k)
    Ho = np.asfortranarray(H.copy())
    nk_ref = oracle.krylov_schur(np.zeros((1, k + 1), X.dtype, order="F"), Ho)      # only the kept count is needed
    Xd = lk.Basis(ctx, kind, n, k + 1).put(X)
    nk = lk.krylov_schur(Xd, H, k)
    assert nk == nk_ref and nk >= 1
    if "dmma" in cid:
        assert dmma_runs(kind, k, nk)
        if k in (140, 320):
            assert nk > 64 and (k % 8 == 4 or k == 320) and (n < 256 or n % 256 in (0, 1))
    else:
        assert not dmma_runs(kind, k, nk)
        assert gemm_smem(kind, k) <= device_shape()[1]
    if "n4099" in cid:
        assert (n % EPP[kind] or kind == "z") and k % 4 and nk > gemm_pb(kind)
    if "nk-lt-8" in cid:
        assert nk < 8
    Xn = Xd.get()
    check_gemm_result(kind, X, Xn, k, nk)
    assert np.array_equal(Xn[:, nk], X[:, k])
    assert not np.any(Xn[:, nk + 1:])


class _DevArray:
    def __init__(self, ptr, n, typestr):
        self.__cuda_array_interface__ = {"shape": (n,), "typestr": typestr, "data": (ptr, False), "version": 3}


@pytest.mark.gpu
def test_basis_gemm_multi_chunk(lk, ctx, oracle):
    """lkb_krylov_schur's row chunks: n = 2 chunk + 4097 rows in rdp (about 4.4 GB), checked around every chunk boundary,
    at the last rows and at 10^4 random rows, which are regenerated on the host from the device generator's seeds."""
    import torch
    kind, k = "d", 16
    rng = np.random.default_rng(5)
    H = np.asfortranarray(np.triu(rng.standard_normal((k + 1, k)), -1))
    nk_ref = oracle.krylov_schur(np.zeros((1, k + 1), order="F"), H.copy(order="F"))
    chunk = ks_chunk(kind, 1 << 40, nk_ref)
    n = 2 * chunk + 4097
    assert ks_chunk(kind, n, nk_ref) == chunk and -(-n // chunk) == 3
    X = lk.Basis(ctx, kind, n, k + 1)
    seeds = [1000 + i for i in range(k + 1)]
    for i in range(k + 1):
        X.col(i).fill_random("uniform", seeds[i])
    ext = torch.cuda.ExternalStream(ctx.stream)
    cols = [torch.as_tensor(_DevArray(X.col(i).ptr, n, "<f8"), device="cuda") for i in range(k + 1)]
    with torch.cuda.stream(ext):
        for i in range(k):
            cols[i][:k] = 0
            cols[i][i] = 1
    ext.synchronize()
    nk = lk.krylov_schur(X, H, k)
    assert nk == nk_ref
    rows = set()
    for b in (chunk, 2 * chunk):
        rows |= set(range(b - 2, b + 3))
    rows |= set(range(n - 5, n)) | set(range(k, k + 3))
    rows |= set(int(r) for r in rng.integers(k, n, 10000))
    rows = np.array(sorted(rows))
    Xn = np.stack([cols[i][torch.as_tensor(rows, device="cuda")].cpu().numpy() for i in range(k + 1)], axis=1)
    Zt = torch.stack([cols[i][:k] for i in range(nk)], dim=1).cpu().numpy()
    X0 = np.stack([np.array([oracle.fill(1, kind, "uniform", seeds[i], row0=int(r))[0] for r in rows]) for i in range(k + 1)], axis=1)
    Xn_full = np.zeros((len(rows) + k, nk)); Xn_full[:k] = Zt; Xn_full[k:] = Xn[:, :nk]
    X_in = np.zeros((len(rows) + k, k + 1)); X_in[:k, :k] = np.eye(k); X_in[k:] = X0
    check_gemm_result(kind, X_in, Xn_full, k, nk)
    assert np.array_equal(Xn[:, nk], X0[:, k])
    assert not np.any(Xn[:, nk + 1:])


# ---- (c) the shared-memory limits -------------------------------------------------------------------------------------------
def limit_cases(optin):
    """(id, kind, j, fits): multidot through innerprod, multiaxpy through lincomb_sub.  The old attributes were 160 KB for
    k_multidot and the 48 KB default for k_multiaxpy; past the device's opt-in maximum the call must fail cleanly."""
    cases = []
    for kind, j_ok in (("d", 2559), ("z", 1279)):
        assert md_smem(kind, j_ok) <= 160 * 1024 < md_smem(kind, j_ok + 1)
        j_past = optin // (8 * WSZ[kind])
        assert md_smem(kind, j_past) > optin
        cases += [("innerprod", kind, j_ok, True), ("innerprod", kind, j_ok + 1, True), ("innerprod", kind, j_past, False)]
    for kind, j_ok in (("s", 12288), ("z", 3072)):
        assert ma_smem(kind, j_ok) <= 48 * 1024 < ma_smem(kind, j_ok + 1)
        j_past = optin // ESZ[kind] + 1
        assert ma_smem(kind, j_past) > optin
        cases += [("lincomb_sub", kind, j_ok, True), ("lincomb_sub", kind, j_ok + 1, True), ("lincomb_sub", kind, j_past, False)]
    return cases


def _rand(rng, kind, shape):
    a = rng.standard_normal(shape) + (1j * rng.standard_normal(shape) if CPLX[kind] else 0)
    return np.asfortranarray(a.astype({"s": np.float32, "d": np.float64, "c": np.complex64, "z": np.complex128}[kind]))


@pytest.mark.gpu
@pytest.mark.parametrize("case", limit_cases(device_shape()[1]), ids=lambda c: f"{c[0]}-{c[1]}-j{c[2]}")
def test_gs_launcher_shared_memory_limits(lk, ctx, case):
    """n = 67 rows (ragged in every kind but z): every row is a tail row or one CTA's, and each row alone moves the result
    by more than the tolerance (kappa = depth of the multi-dot's sums: EPP products, the 5-level fold, <= 2 CTAs x 8
    warps, the tree; the multi-axpy: an FMA chain over j terms)."""
    op, kind, j, fits = case
    n = 67
    rng = np.random.default_rng(j)
    X = _rand(rng, kind, (n, j))
    Xd = lk.Basis(ctx, kind, n, j).put(X)
    W = _rand(rng, kind, (n, 1))
    Wd = lk.Basis(ctx, kind, n, 1).put(W)
    if not fits:
        with pytest.raises(lk.LkbError) as e:
            Xd.innerprod(j, Wd) if op == "innerprod" else Xd.lincomb_sub(j, _rand(rng, kind, (j, 1)), Wd)
        assert "code -2" in str(e.value) and "shared memory" in str(e.value) and "limit of" in str(e.value)
        small = Xd.innerprod(4, Wd)
        assert np.max(np.abs(hp(kind, small) - matmul_h(kind, X[:, :4], W))) < 1e-3
        return
    u = U[kind]
    if op == "innerprod":
        got = Xd.innerprod(j, Wd)
        ref = matmul_h(kind, X, W)
        tol = (EPP[kind] + 6 + (2 + 8 + 80 if kind in "dz" else 1)) * u * (np.abs(hp(kind, X)).T @ np.abs(hp(kind, W)))
        contrib = np.abs(hp(kind, X).conj() * hp(kind, W))            # dropping row r moves entry i by contrib[r, i]
        assert np.all((contrib / tol.T).max(axis=1) > 100)
    else:
        C = _rand(rng, kind, (j, 1))
        Xd.lincomb_sub(j, C, Wd)
        got = Wd.get()
        ref = hp(kind, W) - matmul(kind, X, C)
        tol = (j + 2) * u * (np.abs(hp(kind, W)) + np.abs(hp(kind, X)) @ np.abs(hp(kind, C)))
    err = np.abs(hp(kind, got) - ref)
    assert np.all(err <= tol), float(np.max(err / tol))


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["d", "z"])
def test_basis_gemm_past_device_limit(lk, ctx, kind):
    """k_basis_gemm<K,PB> keeps k x PB coefficients in shared memory: past the device's limit the launcher refuses the
    GEMM, krylov_schur fails with LKB_ERR_ARG naming the limit and leaves X and H as they were, and the context stays
    usable."""
    optin = device_shape()[1]
    k = optin // (gemm_pb(kind) * ESZ[kind]) + 1
    assert gemm_smem(kind, k) > optin
    X0, H = gemm_inputs(kind, k + 64, k)
    H0 = H.copy(order="F")
    X = lk.Basis(ctx, kind, k + 64, k + 1).put(X0)
    with pytest.raises(lk.LkbError) as e:
        lk.krylov_schur(X, H, k)
    assert "code -2" in str(e.value) and "limit of" in str(e.value) and f"k = {k}" in str(e.value)
    assert np.array_equal(X.get(), X0) and np.array_equal(H, H0)
    Xs, Hs = gemm_inputs(kind, 300, 12)
    Xd = lk.Basis(ctx, kind, 300, 13).put(Xs)
    nk = lk.krylov_schur(Xd, Hs, 12)
    check_gemm_result(kind, Xs, Xd.get(), 12, nk)
