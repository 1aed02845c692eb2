"""The single-vector CGS2 step kernels -- k_dot2, k_multidot, k_axpy_dot, k_multiaxpy and k_multiaxpy_fin -- against a
literal CGS2 in high precision, at the shapes where each launcher's row partition changes regime.

Each kernel is isolated through the entry point that exposes its output: Basis.innerprod (k_dot2 for j = 1, k_multidot
otherwise), Basis.lincomb_sub (k_multiaxpy), double_gram_schmidt_step with the "fused" option on and off (pass 1, then
k_axpy_dot or its two-kernel fallback, then the last multi-axpy) and arnoldi(kstart = kend = k) with the "fin" and
"serpentine" options on and off (the whole step tail, k_multiaxpy_fin included).  The launchers' partitions are restated
below (kernels_gs.cu, kernels_fused.cu, lkb_reduce.cuh) and every case asserts the regime it claims.

References follow the kernels' data flow (c1 narrowed to the kind before the update, w' stored in the kind) in float64
for s / c and in longdouble (or Dot2) for d / z.  Bounds are componentwise, kappa_E u_E (...) + kappa_W u_W (...), where
kappa_E and kappa_W are the longest sequential chains a kernel sums in the kind (E) and in double (W); each is derived
next to its plan function.  test_cgs2_cases_are_sensitive checks without a device that each case reaches its regime,
that the reference's own error is far below the bound, and that dropping a watched row, a CTA's range, an axpy_dot
tile or the upper half of the final pass's split moves the result by more than 100 bounds."""
import numpy as np
import pytest

from kernel_ref import CPLX, DT, EPP, ESZ, KINDS, U, device_shape, hp, matmul, matmul_h, sum_depth

UW = 2.0 ** -53                                   # unit roundoff of W (double / double2)
CF = {"s": 1, "d": 1, "c": 2, "z": 2}             # sequential FMAs per element product (complex: two per component)
WEIGHT = 256.0                                    # weight of the watched rows in w
CHUNK = 1 << 20                                   # rows per block of the big references


def cdiv(a, b):
    return -(-a // b)


def tree_depth(nb):
    """reduce_rows_tree: level A sums groups of <= 16 partial rows, level B the G = ceil(nb / 16) group rows in steps
    of 8 (padded with zeros): a chain of min(16, nb) + 8 ceil(G / 8) adds."""
    return min(16, nb) + 8 * cdiv(cdiv(nb, 16), 8)


# ---- the launchers' formulas ---------------------------------------------------------------------------------------------
def dot2_plan(kind, n, sms):
    """multidot_t, j = 1 -> k_dot2: nb = clamp(ceil(npk / 1024), 1, min(4 SMs, 960)), 256 threads, a U = 4 main loop
    over packs pk, pk + s, pk + 2s, pk + 3s (s = 256 nb), then a stride-s remainder; the n mod EPP tail rows go to CTA 0,
    thread 0.  CTA b owns the packs with (pk mod s) in [256 b, 256 b + 256)."""
    e = EPP[kind]
    npk = n // e
    nb = max(1, min(cdiv(npk, 1024), 4 * sms, 960))
    s = 256 * nb

    def iters(g):
        main = max(0, cdiv(npk - 3 * s - g, 4 * s))
        p0 = g + 4 * s * main
        return main, max(0, cdiv(npk - p0, s))
    main0, rem0 = iters(0)
    rem_any = any(iters(g)[1] for g in range(min(s, npk)))
    ctas = []
    for b in range(nb):
        first = 256 * b
        if first >= npk:
            continue
        r = (npk - 1) % s
        base = npk - 1 - r
        last = base + 256 * b + 255 if r >= 256 * b + 255 else (npk - 1 if r >= 256 * b else base - s + 256 * b + 255)
        ctas.append((first * e, last * e + e - 1))
    return dict(nb=nb, stride=s, main=main0, rem=rem0, rem_any=rem_any, passes=cdiv(npk, s), tail=list(range(npk * e, n)),
                ctas=ctas)


def dot2_kappa(kind, n, sms):
    """(kappa_E, kappa_W) of out[0] = x^H y.  Each thread keeps one E chain over all its packs (U EPP products per main
    iteration, EPP per remainder pack) and, in CTA 0's thread 0, the tail elements; then the chain is widened and W adds
    the 5-level warp sum, 8 warps and the tree.  (s at 4096^2: 28 packs, 112 float terms per chain.)"""
    p = dot2_plan(kind, n, sms)
    ke = (4 * p["main"] + p["rem"]) * EPP[kind] * CF[kind] + CF[kind] * len(p["tail"])
    kw = 5 + 8 + tree_depth(p["nb"])
    return (ke, kw) if kind in "sc" else (ke + kw, 0)


def md_plan(kind, n, sms):
    """multidot_t, j >= 2 -> k_multidot: nb = clamp(min(2 SMs, ceil(npk / 32)), 1, 960); nfull = npk / (1024 nb) rounds
    of 4-pack tiles (round r, CTA b: packs [(r nb + b) 1024, + 1024)); the remainder split in 32-pack groups, CTA b owning
    [rem0 + floor(b rg / nb) 32, min(npk, rem0 + floor((b + 1) rg / nb) 32)), walked in 256-pack tiles, the last one
    masked; the tail rows go to CTA 0, thread 0.  desc visits the same tiles in reverse order."""
    e = EPP[kind]
    npk = n // e
    nb = max(1, min(2 * sms, cdiv(npk, 32), 960))
    nfull = npk // (1024 * nb)
    rem0 = nfull * 1024 * nb
    rg = cdiv(npk - rem0, 32)
    shares = [(rem0 + (b * rg // nb) * 32, min(npk, rem0 + ((b + 1) * rg // nb) * 32)) for b in range(nb)]
    tiles = [nfull + (q1 - q0) // 256 + (1 if (q1 - q0) % 256 else 0) for q0, q1 in shares]
    return dict(nb=nb, nfull=nfull, rem0=rem0, rg=rg, shares=[(q0 * e, q1 * e) for q0, q1 in shares], tiles=tiles,
                masked=[(q1 - q0) % 256 != 0 for q0, q1 in shares], tail=list(range(npk * e, n)), npk=npk)


def md_kappa(kind, n, sms):
    """(kappa_E, kappa_W) of a column of k_multidot: per (tile, chunk) a thread sums PT EPP products (PT <= 4) in E and
    the warp folds 32 lanes in 5 levels, then the column is widened: E chain <= 4 EPP CF + 5.  In W: one add per tile of
    the CTA, a tail element each, 8 warps and the tree."""
    p = md_plan(kind, n, sms)
    ke = 4 * EPP[kind] * CF[kind] + 5
    kw = max(p["tiles"]) + len(p["tail"]) + 8 + tree_depth(p["nb"])
    return (ke, kw) if kind in "sc" else (ke + kw, 0)


def axpy_dot_plan(kind, n, j, sms):
    """axpy_dot_ok / axpy_dot_t: eligible iff 1 <= j <= 128, n mod EPP = 0 and n >= 32 EPP (a Basis column is 16-byte
    aligned; the tensor-map limit n sizeof(E) / word < 2^31 holds for every n here).  jc = ceil(j / 16) 16; tp = 32 if
    jc > 64, else 64 if jc > 32 or s, else 128; ntiles = ceil(npk / tp), nb = min(SMs, ntiles, 960), tiles dealt
    round-robin (CTA b: tiles b, b + nb, ...); nst stages from the 222 KB budget (<= 8); rs = min(tp / 32, 8 / nchunk)
    row slices per 16-column chunk."""
    e = EPP[kind]
    npk = n // e
    ok = 1 <= j <= 128 and n % e == 0 and n >= 32 * e and n * ESZ[kind] // (4 if kind == "s" else 8) < 2 ** 31
    jc = cdiv(j, 16) * 16
    tp = 32 if jc > 64 else (64 if (jc > 32 or kind == "s") else 128)
    ntiles = cdiv(npk, tp)
    nb = min(sms, ntiles, 960)
    nmine = [cdiv(ntiles - b, nb) for b in range(nb)]
    fixed = 9 * tp * 16 + 128
    nst = min(8, (222 * 1024 - fixed) // (jc * tp * 16 + tp * 16 + 16))
    nchunk = jc // 16
    rs = min(tp // 32, 8 // nchunk)
    return dict(ok=ok, jc=jc, tp=tp, ntiles=ntiles, nb=nb, nmine=nmine, nst=nst, rs=rs, nchunk=nchunk, npk=npk)


def axpy_dot_kappa(kind, n, j, sms):
    """(kappa_E, kappa_W) of c2 from k_axpy_dot.  Phase B: per tile a lane adds (tp / 32) / rs packs of EPP products per
    column to accumulators that persist in E over all the CTA's tiles; one 5-level fold per warp at the end, then W adds
    the rs slices and the tree.  (s at 4096^2, j <= 64: 443 tiles, ~1770 float terms per chain.)"""
    p = axpy_dot_plan(kind, n, j, sms)
    ke = (p["tp"] // 32 // p["rs"]) * EPP[kind] * CF[kind] * max(p["nmine"]) + 5
    kw = p["rs"] + tree_depth(p["nb"])
    return (ke, kw) if kind in "sc" else (ke + kw, 0)


def ma_plan(kind, n, sms):
    """multiaxpy_t / multiaxpy_fin_t: nb = clamp(ceil(npk / 256), 1, min(4 SMs, 1024)), one pack per thread per pass.
    k_multiaxpy_fin with nb >= 2 runs two waves (half = ceil(nb / 2) CTAs, then the rest), each striding over one half of
    the packs, split at mid = min(npk, ceil((npk / 2) / 32) 32); desc swaps the halves and reverses each walk."""
    npk = n // EPP[kind]
    nb = max(1, min(cdiv(npk, 256), 4 * sms, 1024))
    p = dict(nb=nb, passes=cdiv(npk, nb * 256), npk=npk, tail=list(range(npk * EPP[kind], n)))
    if nb >= 2:
        half = cdiv(nb, 2)
        mid = min(npk, (npk // 2 + 31) // 32 * 32)
        p.update(half=half, mid=mid, passes_lo=cdiv(mid, half * 256), passes_hi=cdiv(npk - mid, (nb - half) * 256))
    return p


# ---- references -----------------------------------------------------------------------------------------------------------
def mm_h(kind, A, B):
    """A^H B in the reference precision, in row blocks of CHUNK (bounded host memory for the 4096^2 cases)."""
    if A.shape[0] <= CHUNK:
        return matmul_h(kind, A, B)
    acc = None
    for r in range(0, A.shape[0], CHUNK):
        t = matmul_h(kind, A[r:r + CHUNK], B[r:r + CHUNK])
        acc = t if acc is None else acc + t
    return acc


def mm(kind, A, B):
    """A B in the reference precision, in row blocks."""
    out = np.empty((A.shape[0], B.shape[1]), dtype=hp(kind, np.zeros(1, DT[kind])).dtype)
    for r in range(0, A.shape[0], CHUNK):
        out[r:r + CHUNK] = matmul(kind, A[r:r + CHUNK], B)
    return out


def narrow(kind, a):
    return hp(kind, np.asarray(a).astype(DT[kind]))


def cgs2_reference(kind, V, w):
    """The literal step: c1 = V^H w; w' = fl_E(w - V fl_E(c1)); c2 = V^H w'; w'' = w' - V fl_E(c2); H = c1 + c2."""
    w = w.reshape(-1, 1)
    c1 = mm_h(kind, V, w)
    w1 = narrow(kind, hp(kind, w) - mm(kind, V, narrow(kind, c1)))
    c2 = mm_h(kind, V, w1)
    w2 = w1 - mm(kind, V, narrow(kind, c2))
    return dict(c1=c1[:, 0], c2=c2[:, 0], H=(c1 + c2)[:, 0], w1=w1[:, 0], w2=w2[:, 0])


def step_bounds(kind, V, w, ref, k_dot, k_upd):
    """Componentwise bounds of one CGS2 step.  k_dot = (kappa_E, kappa_W) of the pass-2 dot, k_upd the longest chain of
    an update entry (j CF FMAs, + the E combine of k_axpy_dot's chunks, + the store).
      H  : u_E (k_upd + 2) |V|^T S1 + (k_dot) |V|^T |w'| + u_E |H|     S1 = |w| + |V| |c1|
           (c1's own error cancels in c1 + c2: c2 = V^H (w - V c1) sees it with the opposite sign; the update's rounding
           and c2's sums remain, then H is narrowed to E)
      w'': (I - V V^H) of pass 1's rounding, pass 2's rounding, and V times c2's error."""
    u = U[kind]
    ke, kw = k_dot
    dotc = ke * u + kw * UW
    f64 = lambda a: np.abs(np.asarray(a)).astype(np.float64)       # bounds need no extra precision
    a1, c1, c2 = f64(ref["w1"]), f64(ref["c1"]), f64(ref["c2"])
    S1 = np.empty(V.shape[0]); VtS1 = 0; Vtw1 = 0
    for r in range(0, V.shape[0], CHUNK):
        aV = f64(V[r:r + CHUNK])
        S1[r:r + CHUNK] = f64(w[r:r + CHUNK]) + aV @ c1
        VtS1 = VtS1 + aV.T @ S1[r:r + CHUNK]
        Vtw1 = Vtw1 + aV.T @ a1[r:r + CHUNK]
    tH = u * (k_upd + 2) * VtS1 + dotc * Vtw1 + u * f64(ref["H"])
    tW = np.empty(V.shape[0])
    for r in range(0, V.shape[0], CHUNK):
        aV = f64(V[r:r + CHUNK])
        S2 = a1[r:r + CHUNK] + aV @ c2
        tW[r:r + CHUNK] = u * (k_upd + 2) * (S1[r:r + CHUNK] + aV @ VtS1 + S2) + dotc * (aV @ Vtw1)
    return 2 * tH, 2 * tW


# ---- the cases ------------------------------------------------------------------------------------------------------------
def innerprod_cases(sms):
    """(id, kind, j, n): Basis.innerprod runs k_dot2 (j = 1) or k_multidot alone."""
    cases = []
    for kind in KINDS:
        e = EPP[kind]
        cases += [(f"{kind}-dot2-nb1", kind, 1, 700 * e + e - 1), (f"{kind}-dot2-main-norem", kind, 1, 1024 * e),
                  (f"{kind}-dot2-rem", kind, 1, 3372 * e + e - 1),
                  (f"{kind}-dot2-passes", kind, 1, (4 * sms * 1024 * 3 + 777) * e + e - 1)]
        for j in (2, 16, 17, 129):
            cases.append((f"{kind}-md-j{j}-nfull0", kind, j, 4099))
        cases += [(f"{kind}-md-j33-nfull2-norem", kind, 33, 2048 * 2 * sms * e),
                  (f"{kind}-md-j17-fewgroups", kind, 17, (1024 * 2 * sms + 32 * 10 + 7) * e + e - 1),
                  (f"{kind}-md-j16-masked", kind, 16, (1024 * 2 * sms + 32 * (2 * sms * 9 + 5)) * e),
                  (f"{kind}-md-j33-nb1", kind, 33, 20 * e + e - 1), (f"{kind}-md-j33-nb16", kind, 33, 500 * e + e - 1),
                  (f"{kind}-md-j33-nb17", kind, 33, 530 * e)]
    for kind in ("s", "z"):
        for j in (15, 33, 128, 300):
            cases.append((f"{kind}-md-j{j}-n100003", kind, j, 100003))
    return cases


def check_innerprod_regime(cid, kind, j, n, sms):
    if j == 1:
        p = dot2_plan(kind, n, sms)
        if "nb1" in cid:
            assert p["nb"] == 1
        if "main-norem" in cid:
            assert p["main"] >= 1 and not p["rem_any"]
        if "-rem" in cid:
            assert p["rem_any"] and p["main"] >= 1
        if "passes" in cid:
            assert p["nb"] == 4 * sms and p["passes"] >= 8
        return p
    p = md_plan(kind, n, sms)
    if "nfull0" in cid:
        assert p["nfull"] == 0
    if "nfull2-norem" in cid:
        assert p["nfull"] == 2 and p["rg"] == 0 and p["nb"] == 2 * sms
    if "fewgroups" in cid:
        assert p["nfull"] == 1 and 0 < p["rg"] < p["nb"] and any(q0 == q1 for q0, q1 in p["shares"])
    if "masked" in cid:
        assert p["nfull"] == 1 and p["nb"] == 2 * sms and any(p["masked"]) and min(p["tiles"]) >= 3
    for tag, nb in (("nb1", 1), ("nb16", 16), ("nb17", 17)):
        if cid.endswith("-" + tag):
            assert p["nb"] == nb
    if n % EPP[kind]:
        assert p["tail"]
    return p


def innerprod_watch(kind, j, n, sms):
    """Rows whose loss a correct bound must see: the tail, the first / last row of every CTA's range or share."""
    if j == 1:
        p = dot2_plan(kind, n, sms)
        rows = {r for a, b in p["ctas"] for r in (a, b)}
    else:
        p = md_plan(kind, n, sms)
        e = EPP[kind]
        rows = set()
        for b in range(p["nb"]):
            for r in range(p["nfull"]):
                t0 = (r * p["nb"] + b) * 1024 * e
                rows |= {t0, t0 + 1024 * e - 1}
            q0, q1 = p["shares"][b]
            if q1 > q0:
                rows |= {q0, q1 - 1}
    return sorted(rows | set(p["tail"]))


def innerprod_inputs(kind, j, n, sms, seed=0):
    rng = np.random.default_rng(seed + 31 * n + j)
    V = rng.standard_normal((n, j)).astype(DT[kind]) if not CPLX[kind] else \
        (rng.standard_normal((n, j)) + 1j * rng.standard_normal((n, j))).astype(DT[kind])
    V = np.asfortranarray(V)
    w = rng.standard_normal(n) + (1j * rng.standard_normal(n) if CPLX[kind] else 0)
    watch = innerprod_watch(kind, j, n, sms)
    w[watch] = (w[watch] + np.sign(w[watch].real)) * WEIGHT * len(watch) ** 0.5
    V[watch] += np.sign(V[watch].real).astype(V.dtype)         # |Re v|, |Re w| / weight >= 1 on the watched rows
    return V, w.astype(DT[kind]), watch


def innerprod_tol(kind, V, w, j, n, sms):
    ke, kw = dot2_kappa(kind, n, sms) if j == 1 else md_kappa(kind, n, sms)
    ref = mm_h(kind, V, w.reshape(-1, 1))[:, 0]
    scale = np.abs(hp(kind, V)).T @ np.abs(hp(kind, w))
    return ref, (ke * U[kind] + kw * UW) * scale + U[kind] * np.abs(ref)


def lincomb_cases(sms):
    cases = []
    for kind in KINDS:
        for j in (1, 7, 8, 9, 128, 300):
            cases.append((f"{kind}-j{j}-n100003", kind, j, 100003))
        cases.append((f"{kind}-j9-passes", kind, 9, (4 * sms * 256 * 3 + 5) * EPP[kind] + EPP[kind] - 1))
    return cases


def dgs_cases(sms):
    """(id, kind, j, n) for double_gram_schmidt_step: every tp regime of k_axpy_dot with ntiles < SMs and with
    ntiles = q SMs + 1, q = 2 nst + 1 (the ring wraps twice, the mbarrier parity flips), partial last tiles, j mod 16 != 0,
    and the three ineligible shapes."""
    cases = []
    for kind in KINDS:
        e = EPP[kind]
        for j in (16, 47, 100, 128):
            p = axpy_dot_plan(kind, 4096 * e, j, sms)
            tp, nst = p["tp"], p["nst"]
            cases.append((f"{kind}-j{j}-tp{tp}-few", kind, j, (tp * (sms // 2) + tp // 2) * e))
            if j != 128:
                q = 2 * nst + 1
                cases.append((f"{kind}-j{j}-tp{tp}-wrap", kind, j, (tp * q * sms + tp // 3) * e))
        if e > 1:
            cases.append((f"{kind}-j16-ragged-fallback", kind, 16, 1001 * e + 1))
        cases.append((f"{kind}-j16-short-fallback", kind, 16, 31 * e))
        cases.append((f"{kind}-j129-fallback", kind, 129, 4096 * e))
    return cases


def dgs_inputs(kind, j, n, sms):
    """V = X(:, :j) orthonormal, w = A X(:, j) with the rows of the first and the (partial) last axpy_dot tile weighted,
    so that each tile holds a visible share of c2."""
    X, d = step_inputs(kind, j + 1, n)
    w = d * X[:, j]
    p = axpy_dot_plan(kind, n, j, sms)
    e, tp = EPP[kind], p["tp"]
    for t in (0, p["ntiles"] - 1):
        w[t * tp * e:min(n, (t + 1) * tp * e)] *= DT[kind](WEIGHT)
    return X[:, :j], w.astype(DT[kind])


def check_dgs_regime(cid, kind, j, n, sms):
    p = axpy_dot_plan(kind, n, j, sms)
    assert p["ok"] == ("fallback" not in cid)
    if not p["ok"]:
        return p
    assert f"tp{p['tp']}" in cid
    if "few" in cid:
        assert p["ntiles"] < sms and max(p["nmine"]) == 1 <= p["nst"]
    if "wrap" in cid:
        assert p["ntiles"] % sms == 1 and max(p["nmine"]) > 2 * p["nst"]
    assert p["npk"] % p["tp"], "the last tile is partial"
    return p


def fin_cases(sms):
    """(id, kind, k, n) for arnoldi(kstart = kend = k): k_multiaxpy_fin with nb = 1, 2, 3 and 4 SMs (several passes per
    half), npk < 64; k odd and even flips the serpentine direction."""
    cases = []
    for kind in KINDS:
        e = EPP[kind]
        for tag, npk in (("npk50", 50), ("nb1", 200), ("nb2", 500), ("nb3", 700), ("nbmax", 4 * sms * 256 * 4 + 77)):
            for k in (5, 6):
                cases.append((f"{kind}-{tag}-k{k}", kind, k, npk * e + e - 1))
    return cases


def check_fin_regime(cid, kind, k, n, sms):
    p = ma_plan(kind, n, sms)
    for tag, nb in (("npk50", 1), ("nb1", 1), ("nb2", 2), ("nb3", 3)):
        if f"-{tag}-" in cid:
            assert p["nb"] == nb
    if "npk50" in cid:
        assert p["npk"] < 64
    if "nbmax" in cid:
        assert p["nb"] == 4 * sms and p["passes_lo"] >= 2 and p["passes_hi"] >= 2
    return p


def step_inputs(kind, k, n, seed=0):
    """X(:, :k) orthonormal (host QR, narrowed), d a diagonal of powers of two (A x exact in every kind), and the rows
    of X(:, k - 1) the sensitivity check watches weighted."""
    rng = np.random.default_rng(seed + 7 * n + k)
    X0 = rng.standard_normal((n, k)) + (1j * rng.standard_normal((n, k)) if CPLX[kind] else 0)
    Q, _ = np.linalg.qr(X0)
    X = np.zeros((n, k + 1), dtype=DT[kind], order="F")
    X[:, :k] = Q
    d = np.ldexp(1.0, rng.integers(-2, 3, n)).astype(DT[kind])
    return X, d


# ---- CPU rehearsal ----------------------------------------------------------------------------------------------------------
def test_cgs2_cases_are_sensitive():
    """Without a device: every case reaches its regime; the reference's own error is below 1/100 of the bound; dropping a
    watched row, a CTA's whole range, one axpy_dot tile (the partial last one included) or the upper half of the final
    pass's split moves the result by more than 100 bounds."""
    sms, _ = device_shape()
    for cid, kind, j, n in innerprod_cases(sms):
        check_innerprod_regime(cid, kind, j, n, sms)
        if n * j > 3e6:
            continue                                   # exercised on the device run; the regime is checked above
        V, w, watch = innerprod_inputs(kind, j, n, sms)
        ref, tol = innerprod_tol(kind, V, w, j, n, sms)
        eps = np.finfo(np.float64 if kind in "sc" else np.longdouble).eps
        ref_err = sum_depth(kind, n) * eps * (np.abs(hp(kind, V)).T @ np.abs(hp(kind, w)))
        assert np.all(ref_err < tol / 100), cid
        for r in watch:
            moved = np.abs(hp(kind, V[r]).conj() * hp(kind, w[r]))
            assert np.max(moved / tol) > 100, (cid, r)
        if j > 1:
            p = md_plan(kind, n, sms)
            for b, (q0, q1) in enumerate(p["shares"]):
                if q1 > q0:
                    moved = np.abs(mm_h(kind, V[q0:q1], w[q0:q1].reshape(-1, 1))[:, 0])
                    assert np.max(moved / tol) > 100, (cid, "share", b)
    for cid, kind, j, n in dgs_cases(sms):
        p = check_dgs_regime(cid, kind, j, n, sms)
        if not p["ok"] or n * j > 4e6:
            continue
        V, w = dgs_inputs(kind, j, n, sms)
        ref = cgs2_reference(kind, V, w)
        tH, _ = step_bounds(kind, V, w, ref, axpy_dot_kappa(kind, n, j, sms), j * CF[kind] + p["nchunk"] + 1)
        e, tp = EPP[kind], p["tp"]
        for t in (0, p["ntiles"] - 1):                 # first and (partial) last tile of the pass-2 dot
            r0, r1 = t * tp * e, min(n, (t + 1) * tp * e)
            moved = np.abs(mm_h(kind, V[r0:r1], ref["w1"][r0:r1].reshape(-1, 1))[:, 0])
            assert np.max(moved / tH) > 100, (cid, "tile", t)
    for cid, kind, k, n in fin_cases(sms):
        p = check_fin_regime(cid, kind, k, n, sms)
        if p["nb"] < 2 or n > 400000:
            continue
        X, d = step_inputs(kind, k, n)
        V, w = X[:, :k], d * X[:, k - 1]
        ref = cgs2_reference(kind, V, w)
        _, tW = step_bounds(kind, V, w, ref, md_kappa(kind, n, sms), k * CF[kind] + 2)
        beta = np.sqrt(np.sum(np.abs(ref["w2"]) ** 2))
        e = EPP[kind]
        lo, hi = p["mid"] * e, p["npk"] * e
        moved = np.abs(ref["w1"][lo:hi] - ref["w2"][lo:hi] / beta) * beta      # rows left unprocessed, in w'' units
        assert np.max(moved / tW[lo:hi]) > 100, (cid, "upper half")


# ---- device tests -------------------------------------------------------------------------------------------------------------
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


def profiled(ctx, run):
    ctx.set_profile(True)
    try:
        out = run()
        return out, {c: v for c, (_, v) in ctx.get_profile().items()}
    finally:
        ctx.set_profile(False)


@pytest.mark.gpu
@pytest.mark.parametrize("case", innerprod_cases(device_shape()[0]), ids=lambda c: c[0])
def test_innerprod_kernels(lk, ctx, case):
    cid, kind, j, n = case
    sms = device_shape()[0]
    check_innerprod_regime(cid, kind, j, n, sms)
    V, w, _ = innerprod_inputs(kind, j, n, sms)
    Vd = lk.Basis(ctx, kind, n, j).put(V)
    Wd = lk.Basis(ctx, kind, n, 1).put(w)
    got, prof = profiled(ctx, lambda: Vd.innerprod(j, Wd))
    assert prof == dict(matvec=0, multidot=1, multiaxpy=0, other=0, fused_axpy_dot=0)
    ref, tol = innerprod_tol(kind, V, w, j, n, sms)
    err = np.abs(hp(kind, got[:, 0]) - ref)
    assert np.all(err <= tol), (cid, float(np.max(err / tol)))
    assert np.array_equal(Vd.innerprod(j, Wd), got)


@pytest.mark.gpu
@pytest.mark.parametrize("case", lincomb_cases(device_shape()[0]), ids=lambda c: c[0])
def test_lincomb_sub_kernel(lk, ctx, case):
    """k_multiaxpy: each entry is an FMA chain over j CF terms in E after w is loaded: kappa = j CF + 2."""
    cid, kind, j, n = case
    sms = device_shape()[0]
    p = ma_plan(kind, n, sms)
    if "passes" in cid:
        assert p["passes"] >= 3 and p["nb"] == 4 * sms and p["tail"] or kind == "z"
    rng = np.random.default_rng(j + n)
    V, w, _ = innerprod_inputs(kind, j, n, sms)
    C = (rng.standard_normal((j, 1)) + (1j * rng.standard_normal((j, 1)) if CPLX[kind] else 0)).astype(DT[kind])
    Vd = lk.Basis(ctx, kind, n, j).put(V)
    Wd = lk.Basis(ctx, kind, n, 1).put(w)
    _, prof = profiled(ctx, lambda: Vd.lincomb_sub(j, C, Wd))
    assert prof == dict(matvec=0, multidot=0, multiaxpy=1, other=0, fused_axpy_dot=0)
    got = Wd.get()[:, 0]
    ref = hp(kind, w) - mm(kind, V, C)[:, 0]
    tol = (j * CF[kind] + 2) * U[kind] * (np.abs(hp(kind, w)) + np.abs(hp(kind, V)) @ np.abs(hp(kind, C[:, 0])))
    err = np.abs(hp(kind, got) - ref)
    assert np.all(err <= tol), (cid, float(np.max(err / tol)))


def dgs_launches(fused):
    return dict(matvec=0, multidot=1 if fused else 2, multiaxpy=1 if fused else 2, other=1, fused_axpy_dot=int(fused))


@pytest.mark.gpu
@pytest.mark.parametrize("case", dgs_cases(device_shape()[0]), ids=lambda c: c[0])
def test_dgs_step_fused_and_unfused(lk, ctx, case):
    cid, kind, j, n = case
    sms = device_shape()[0]
    p = check_dgs_regime(cid, kind, j, n, sms)
    V, w = dgs_inputs(kind, j, n, sms)
    ref = cgs2_reference(kind, V, w)
    Vd = lk.Basis(ctx, kind, n, j).put(V)
    out = {}
    try:
        for fused in (1, 0):
            ctx.set_option("fused", fused)
            Wd = lk.Basis(ctx, kind, n, 1).put(w)
            (info, beta), prof = profiled(ctx, lambda: lk.double_gram_schmidt_step(Wd, 0, 1, Vd, j, if_chk_orthonormal=False))
            assert info == 0
            assert prof == dgs_launches(fused and p["ok"]), (cid, prof)
            kdot = (axpy_dot_kappa if (fused and p["ok"]) else lambda k_, n_, j_, s_: md_kappa(k_, n_, s_))(kind, n, j, sms)
            tH, tW = step_bounds(kind, V, w, ref, kdot, j * CF[kind] + p["nchunk"] + 1)
            eH = np.abs(hp(kind, beta[:, 0]) - ref["H"])
            assert np.all(eH <= tH), (cid, fused, "H", float(np.max(eH / tH)))
            w2 = Wd.get()[:, 0]
            eW = np.abs(hp(kind, w2) - ref["w2"])
            assert np.all(eW <= tW), (cid, fused, "w''", float(np.max(eW / tW)), int(np.argmax(eW / tW)))
            out[fused] = (beta.copy(), w2)
            Wd2 = lk.Basis(ctx, kind, n, 1).put(w)
            _, beta2 = lk.double_gram_schmidt_step(Wd2, 0, 1, Vd, j, if_chk_orthonormal=False)
            assert np.array_equal(beta2, beta) and np.array_equal(Wd2.get()[:, 0], w2)
    finally:
        ctx.set_option("fused", 1)
    if not p["ok"]:
        assert all(np.array_equal(a, b) for a, b in zip(out[0], out[1]))


def run_step(lk, ctx, A, Xd, kind, k, profile=False):
    H = np.zeros((k + 1, k), dtype=DT[kind], order="F")
    if profile:
        info, prof = profiled(ctx, lambda: lk.arnoldi(A, Xd, H, kstart=k, kend=k))
    else:
        info, prof = lk.arnoldi(A, Xd, H, kstart=k, kend=k), None
    assert info == 0
    return H[:, k - 1].copy(), Xd.col(k).get(), prof


def step_launches(fused, fin):
    return dict(matvec=1, multidot=1 if fused else 2, multiaxpy=1 if fused else 2, other=1 if fin else 2,
                fused_axpy_dot=int(fused))


def ww_kappa(kind, n, j, fused, sms):
    """Depth, in units of u_E, of ||w'||^2 as k_multiaxpy_fin receives it (entry j of c2).  Fused: k_axpy_dot sums |w'|^2
    of one pack per tile in double over the CTA's tiles, then warp, 8 warps and the tree.  Unfused: k_multidot's w^H w,
    one E chain over all the CTA's tiles, or, for j = 1, k_dot2's y^H y."""
    r = UW / U[kind]
    if fused:
        p = axpy_dot_plan(kind, n, j, sms)
        return 2 + r * (max(p["nmine"]) * EPP[kind] * CF[kind] + 13 + tree_depth(p["nb"]))
    if j == 1:
        ke, kw = dot2_kappa(kind, n, sms)
        return ke + r * kw
    p = md_plan(kind, n, sms)
    ke = max(p["tiles"]) * 4 * EPP[kind] * CF[kind] + CF[kind] * len(p["tail"])
    kw = 13 + tree_depth(p["nb"])
    return ke + (r * kw if kind in "sc" else kw)


def check_step(kind, V, w, ref, h, x, k_dot, k_upd, wwk, cid):
    """H(:k, k-1) and x = X(:, k) of one arnoldi step against the reference.  beta: the exact path computes ||w''||; the
    predicted one sqrt(||w'||^2 - ||c2||^2) with ||w'||^2 from a reduction wwk deep (ww_kappa; relative error
    wwk u ||w'||^2 / (2 beta^2)), and ||w'||^2 - ||c2||^2 - ||w''||^2 is of the size of the orthogonality of V."""
    u = U[kind]
    j = V.shape[1]
    tH, tW = step_bounds(kind, V, w, ref, k_dot, k_upd)
    eH = np.abs(hp(kind, h[:j]) - ref["H"])
    assert np.all(eH <= tH), (cid, "H", float(np.max(eH / tH)))
    beta = np.sqrt(np.sum(np.abs(ref["w2"]) ** 2))
    ww = np.sum(np.abs(ref["w1"]) ** 2)
    tb = u * ((wwk + 4 * j + 8) * ww / (2 * beta) + beta) + np.sqrt(np.sum(tW ** 2))
    eb = abs(float(np.real(h[j])) - float(beta))
    assert eb <= tb, (cid, "beta", eb / tb)
    tx = tW / beta + np.abs(ref["w2"]) * tb / beta ** 2 + 2 * u * np.abs(ref["w2"]) / beta
    ex = np.abs(hp(kind, x) - ref["w2"] / beta)
    assert np.all(ex <= tx), (cid, "x", float(np.max(ex / tx)), int(np.argmax(ex / tx)))


@pytest.mark.gpu
@pytest.mark.parametrize("case", fin_cases(device_shape()[0]), ids=lambda c: c[0])
def test_arnoldi_step_tail(lk, ctx, case):
    cid, kind, k, n = case
    sms = device_shape()[0]
    check_fin_regime(cid, kind, k, n, sms)
    X, d = step_inputs(kind, k, n)
    V, w = X[:, :k], (d * X[:, k - 1]).astype(DT[kind])
    ref = cgs2_reference(kind, V, w)
    fused = axpy_dot_plan(kind, n, k, sms)["ok"]
    kdot = axpy_dot_kappa(kind, n, k, sms) if fused else md_kappa(kind, n, sms)
    wwk = ww_kappa(kind, n, k, fused, sms)
    A = lk.LinOp.diag(lk.Vector(ctx, kind, n).put(d))
    Xd = lk.Basis(ctx, kind, n, k + 1).put(X)
    res = {}
    try:
        for fin in (1, 0):
            for serp in (1, 0):
                ctx.set_option("fin", fin); ctx.set_option("serpentine", serp)
                h, x, prof = run_step(lk, ctx, A, Xd, kind, k, profile=True)
                assert prof == step_launches(fused, fin), (cid, fin, serp, prof)
                check_step(kind, V, w, ref, h, x, kdot, k * CF[kind] + 3, wwk, f"{cid}-fin{fin}-serp{serp}")
                h2, x2, _ = run_step(lk, ctx, A, Xd, kind, k)              # graphs on, profile off: same bits
                assert np.array_equal(h2, h) and np.array_equal(x2, x), (cid, fin, serp)
                res[fin, serp] = (h, x)
        ctx.set_graphs(False)
        h3, x3, _ = run_step(lk, ctx, A, Xd, kind, k)
        assert np.array_equal(h3, res[0, 0][0]) and np.array_equal(x3, res[0, 0][1])
    finally:
        ctx.set_option("fin", 1); ctx.set_option("serpentine", 1); ctx.set_graphs(True)
    # With the fused final pass, serpentine sweeps reverse the pass-1 dot, the fused middle and the final pass at alternate
    # steps, which reorders their reductions (each direction is checked against the bounds above).  Without it every
    # kernel of the step walks the rows upwards, so the option must not change a bit.
    assert all(np.array_equal(a, b) for a, b in zip(res[0, 1], res[0, 0])), cid


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["s", "d"])
@pytest.mark.parametrize("side", ["below", "above"])
def test_fin_predicted_norm_threshold(lk, ctx, kind, side):
    """A non-orthonormal V (one column scaled) makes r = ||c2||^2 / ||w'||^2 tunable.  Below 1e-2 k_multiaxpy_fin trusts
    the predicted norm sqrt(||w'||^2 - ||c2||^2) -- wrong for this V, and far from ||w''|| -- above it the norm is computed
    exactly and k_scale_dev normalises the vector."""
    n, k = 5003, 6
    X, d = step_inputs(kind, k, n)
    target = 0.9e-2 if side == "below" else 1.1e-2

    def ratio(a):
        Y = X.copy(); Y[:, 0] *= DT[kind](a)
        V, w = Y[:, :k], (d * Y[:, k - 1]).astype(DT[kind])
        ref = cgs2_reference(kind, V, w)
        return float(np.sum(np.abs(ref["c2"]) ** 2) / np.sum(np.abs(ref["w1"]) ** 2)), Y, V, w, ref
    lo, hi = 1.5, 3.0
    for _ in range(60):                              # r grows with the scale of column 0 on [1.5, 3] (0.0006 .. 0.1)
        mid = 0.5 * (lo + hi)
        if ratio(mid)[0] < target:
            lo = mid
        else:
            hi = mid
    r, Y, V, w, ref = ratio(lo)
    assert abs(r / target - 1) < 0.02
    A = lk.LinOp.diag(lk.Vector(ctx, kind, n).put(d))
    Xd = lk.Basis(ctx, kind, n, k + 1).put(Y)
    h, x, prof = run_step(lk, ctx, A, Xd, kind, k, profile=True)
    ww = np.sum(np.abs(ref["w1"]) ** 2); s2 = np.sum(np.abs(ref["c2"]) ** 2)
    exact = float(np.sqrt(np.sum(np.abs(ref["w2"]) ** 2)))
    pred = float(np.sqrt(ww - s2))
    bound = 64 * U[kind] * float(np.sqrt(ww))
    assert abs(pred - exact) > 100 * bound
    beta = float(np.real(h[k]))
    if side == "below":
        assert abs(beta - pred) <= bound, (beta, pred, exact)
    else:
        assert abs(beta - exact) <= bound, (beta, pred, exact)
        assert abs(np.linalg.norm(hp(kind, x).astype(np.float64)) - 1) < 8 * U[kind] * 100


@pytest.mark.gpu
@pytest.mark.parametrize("kind", KINDS)
def test_step_nan_is_an_error(lk, ctx, kind):
    n, k = 4099, 4
    X, d = step_inputs(kind, k, n)
    X[17, k - 1] = np.nan
    A = lk.LinOp.diag(lk.Vector(ctx, kind, n).put(d))
    Xd = lk.Basis(ctx, kind, n, k + 1).put(X)
    H = np.zeros((k + 1, k), dtype=DT[kind], order="F")
    with pytest.raises(lk.LkbError, match="NaN"):
        lk.arnoldi(A, Xd, H, kstart=k, kend=k)


# ---- the benchmark's shape: one step on the 4096^2 5-point stencil -------------------------------------------------------
BENCH_COEF = (4.0, -1.0, -1.0, -1.0, -1.0)
# Step-level accuracy: ||V^H x||_inf <= C u_E with one C per kind, set from the unfused path at 4096^2 and held by the
# fused one too.  Measured on an NVIDIA B200 (1000 W): unfused 0.086 / 0.104 (s, k = 16 / 64), 0.075 / 0.009 (c, k = 16 /
# 32), <= 0.008 (d at 4096^2), 0.028 (d, 1024^2, k = 128); the fused path within 5 % of these in every case.
ORTH_C = {"s": 0.25, "c": 0.25, "d": 0.05}


def stencil_cases():
    return ([("d", 4096, 1), ("d", 4096, 16), ("d", 4096, 31), ("s", 4096, 16), ("s", 4096, 64), ("c", 4096, 16),
             ("c", 4096, 32), ("d", 1024, 128)])


@pytest.mark.gpu
@pytest.mark.parametrize("case", stencil_cases(), ids=lambda c: f"{c[0]}-{c[1]}sq-k{c[2]}")
def test_step_on_benchmark_stencil(lk, ctx, case):
    """X(:, :k) is made on the device (fill_random + qr) and read back, w = A X(:, k - 1) by a separate matvec (the
    stencil has no reduction: two matvecs are bitwise equal).  Componentwise bounds as above, and the step-level
    orthogonality ||V^H x||_inf <= C u_E held by the fused and the unfused path alike."""
    kind, side, k = case
    sms = device_shape()[0]
    n = side * side
    A = lk.LinOp.stencil5(ctx, kind, side, side, BENCH_COEF)
    Xd = lk.Basis(ctx, kind, n, k + 1)
    for i in range(k):
        Xd.col(i).fill_random("normal", 100 + i)
    info, _ = lk.qr(Xd, 0, k)
    assert info == 0
    V = Xd.get(0, k)
    y1, y2 = lk.Vector(ctx, kind, n), lk.Vector(ctx, kind, n)
    A.matvec(Xd.col(k - 1), y1); A.matvec(Xd.col(k - 1), y2)
    w = y1.get()
    assert np.array_equal(w, y2.get())
    ref = cgs2_reference(kind, V, w)
    ok = axpy_dot_plan(kind, n, k, sms)["ok"]
    assert ok == (k <= 128)
    orth = {}
    try:
        for fused in (1, 0):
            ctx.set_option("fused", fused)
            use = fused and ok
            kdot = axpy_dot_kappa(kind, n, k, sms) if use else (dot2_kappa(kind, n, sms) if k == 1 else md_kappa(kind, n, sms))
            wwk = ww_kappa(kind, n, k, use, sms)
            h, x, prof = run_step(lk, ctx, A, Xd, kind, k, profile=True)
            assert prof == step_launches(use, True), prof
            check_step(kind, V, w, ref, h, x, kdot, k * CF[kind] + 3, wwk, f"{case}-fused{fused}")
            o = float(np.max(np.abs(mm_h(kind, V, x.reshape(-1, 1))))) / U[kind]
            orth[fused] = o
            h2, x2, _ = run_step(lk, ctx, A, Xd, kind, k)
            assert np.array_equal(h2, h) and np.array_equal(x2, x)
    finally:
        ctx.set_option("fused", 1)
    for fused, o in orth.items():
        assert o <= ORTH_C[kind], (case, fused, o)
