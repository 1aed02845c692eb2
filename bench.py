#!/usr/bin/env python
"""bench.py -- Arnoldi steps/s on BASELINE.json's config C2 (5-point Poisson 4096^2, fp64, kdim=128).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nproc-per-node N ... bench.py --gpus N ...

One bench "step" = one pass of the hot path over one start vector = one full kstart=1..kend=128
Arnoldi factorisation (128 Arnoldi steps: matvec + CGS2 + Hessenberg update each).  `value` is
Arnoldi steps per second = 128*K / time, the strong-scaling metric BASELINE.json names (global
n = 16.8M rows sharded by grid rows over the N ranks).  The start vector is seeded, so two builds run with the same
arguments and --dump-outputs can be compared output for output.

Prints ONE JSON line on rank 0 (see DESIGN.md "Measurement" for every key).
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
# keep stdout to the single JSON line: NCCL prints its version banner to stdout at DEBUG=VERSION
if os.environ.get("NCCL_DEBUG", "VERSION").upper() == "VERSION":
    os.environ["NCCL_DEBUG"] = "WARN"

METRIC = "arnoldi_steps_per_s"
UNIT = "steps/s"
POISSON5 = (4.0, -1.0, -1.0, -1.0, -1.0)
# --dump-outputs keeps the whole H and a fixed row sample of the basis (17 GB at full size): at most 16384 rows, fewer when
# kdim is so large that H and the sample would exceed DUMP_BYTES (default size: 16384 x 129 fp64 = 17 MB)
DUMP_ROWS = 16384
DUMP_BYTES = 64 << 20
DUMP_SEED = 2024


def dump_rows(n: int, kdim: int) -> np.ndarray:
    """The sorted global rows of the basis that --dump-outputs keeps, drawn from a fixed seed."""
    budget = (DUMP_BYTES - (kdim + 1) * kdim * 8) // ((kdim + 1) * 8)
    return np.sort(np.random.default_rng(DUMP_SEED).choice(n, size=min(n, DUMP_ROWS, budget), replace=False))


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--nx", type=int, default=4096)
    ap.add_argument("--ny", type=int, default=4096)
    ap.add_argument("--kdim", type=int, default=128)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-profile-pass", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-fused", action="store_true", help="disable the fused axpy+dot CGS2 kernel (A/B)")
    ap.add_argument("--no-p2p", action="store_true", help="use ncclAllReduce instead of the in-kernel NVLink allreduce (A/B)")
    ap.add_argument("--opt", action="append", default=[], metavar="NAME=0|1",
                    help="lkb_set_option A/B switches: fused, fin (fused final pass), fused_halo, p2p, graphs")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the last timed step computed to DIR: H.npy (the Hessenberg matrix) and X_sample.npy "
                         f"(all columns of the Krylov basis at up to {DUMP_ROWS} fixed, seeded, sorted global rows), float64, "
                         f"{DUMP_BYTES >> 20} MB at most")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be >= 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs needs --impl ours (the reference arm times sampled steps, not whole factorisations)")
    if args.dump_outputs and (args.kdim + 1) ** 2 * 8 > DUMP_BYTES:
        ap.error(f"--dump-outputs: H and one row of the basis exceed {DUMP_BYTES >> 20} MB at this --kdim")
    return args


def alg_bytes_step(j: int, n: int, s: int = 8) -> int:
    """Official algorithmic bytes of one Arnoldi step with j basis vectors (SURVEY 8d)."""
    return 2 * n * s + 4 * j * n * s


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index, self.proc, self.lines = index, None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-i", str(self.index), "-lms", "100"], stdout=subprocess.PIPE, text=True)
            self.thr = threading.Thread(target=self._read, daemon=True); self.thr.start()
        except Exception:
            self.proc = None

    def _read(self):
        for ln in self.proc.stdout:
            self.lines.append(ln.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons, pw = [], [], set(), []
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 8:
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2])); pw.append(float(f[3]))
            except ValueError:
                continue
            for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[4:8]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
        return {"sm_mhz": float(np.median(sm)), "sm_max_mhz": float(max(mx)), "reasons": sorted(reasons),
                "power_w_max": max(pw), "samples": len(sm)}


# ------------------------------------------------------------------------------------------------
# CPU arm: the oracle (C restatement of the reference's per-vector algorithm) on the host cores
# ------------------------------------------------------------------------------------------------
WORKLOAD = "arnoldi kdim={kdim} on 5-pt Poisson {nx}x{ny} (n={n}) fp64 [BASELINE configs[1]]"


class CpuArnoldi:
    """The reference's CPU path for this workload: the oracle (C restatement of LightKrylov's per-vector algorithm,
    OpenMP over `threads` host cores) on the full-size operator.  One SAMPLE = oracle Arnoldi steps at step indices
    `js` spread over the whole 1..kdim range on a basis that is pre-filled ONCE with normalised random columns
    (the cost of a step depends on j, not on the values), so t(j) = a + b*j is fitted by INTERPOLATION and summed
    over j = 1..kdim.  (Round 1 sampled j = 1..8 only and extrapolated; VERDICT r01 weak #6.)"""

    def __init__(self, nx, ny, kdim, threads):
        from oracle import lk_oracle as lo
        self.lo, self.nx, self.ny, self.kdim, self.threads = lo, nx, ny, kdim, threads
        self.n = nx * ny
        self.A = lo.Op.stencil("d", (nx, ny), POISSON5)
        self.X = None

    def _prefill(self, jmax):
        lo = self.lo
        lo.set_threads(host_threads())
        if self.X is None:
            self.X = np.zeros((self.n, self.kdim + 1), order="F")
            self.filled = 0
        for i in range(self.filled, jmax):
            self.X[:, i] = lo.fill(self.n, "d", "uniform", 42 + i)
            lo.normalize(self.X[:, i])
        self.filled = max(self.filled, jmax)

    def sample(self, js):
        """Returns (steps_per_s, seconds_spent, description)."""
        lo = self.lo
        js = sorted(set(min(max(int(j), 1), self.kdim) for j in js))
        self._prefill(max(js))
        lo.set_threads(self.threads)
        H = np.zeros((self.kdim + 1, self.kdim), order="F")
        ts = []
        t00 = time.perf_counter()
        for k in js:
            t0 = time.perf_counter()
            info = lo.arnoldi(self.A, self.X, H, kstart=k, kend=k)
            ts.append(time.perf_counter() - t0)
            assert info == 0
        spent = time.perf_counter() - t00
        if len(js) >= 2:
            b, a = np.polyfit(np.array(js, dtype=float), np.array(ts), 1)
        else:
            a, b = 0.0, ts[-1] / js[-1]
        total = sum(max(a + b * j, 0.0) for j in range(1, self.kdim + 1))
        desc = (f"oracle arnoldi steps at j={js} of 1..{self.kdim} at full n={self.n} (5-pt Poisson {self.nx}x{self.ny}, fp64, "
                f"{self.threads} thread(s)), per-step times fitted t(j)=a+b*j (a={a:.3f}s, b={b:.4f}s) and summed over j=1..{self.kdim}")
        return self.kdim / total, spent, desc


def host_threads() -> int:
    """All the host cores this process may use (torchrun exports OMP_NUM_THREADS=1, which must not shrink the CPU arm)."""
    try:
        return max(1, len(os.sched_getaffinity(0)))
    except AttributeError:
        return max(1, os.cpu_count() or 1)


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    threads = host_threads()
    cpu = CpuArnoldi(args.nx, args.ny, args.kdim, threads)
    kd = args.kdim
    js = sorted(set([1, kd // 4, kd // 2, (3 * kd) // 4, kd]))
    vals = []
    desc = ""
    for i in range(args.warmup + args.steps):
        v, spent, desc = cpu.sample(js)
        if i >= args.warmup:
            vals.append((v, spent))
    value = float(np.mean([v for v, _ in vals]))
    ms = float(np.mean([s for _, s in vals])) * 1e3
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True,
        "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": WORKLOAD.format(kdim=args.kdim, nx=args.nx, ny=args.ny, n=args.nx * args.ny),
                   "bench_step": "bounded CPU sample: " + desc},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": threads, "kind": "port", "sample": desc},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
        "note": "reference = CPU oracle (C restatement of LightKrylov's per-vector algorithm, OpenMP); the Fortran "
                "reference cannot be built in this image or on the GPU box (no Fortran compiler / fpm / stdlib; probed in round 2)",
    }
    emit(line)


# ------------------------------------------------------------------------------------------------
def basis_sample(X, rows: np.ndarray, row0: int, world: int):
    """All columns of the (row-sharded) basis X at the given ascending global rows, gathered on rank 0 (None on the other
    ranks).  The rows are picked on the device, so only the sample crosses to the host."""
    import torch
    import torch.distributed as dist

    class _Column:                                   # a device column of X as a torch tensor, without a copy
        def __init__(self, v):
            self.__cuda_array_interface__ = {"shape": (v.n,), "typestr": "<f8", "data": (v.ptr, False), "version": 2}

    X.ctx.sync()
    mine = rows[(rows >= row0) & (rows < row0 + X.n)] - row0
    idx = torch.as_tensor(mine, device=torch.cuda.current_device())
    part = torch.stack([torch.as_tensor(_Column(X.col(j)), device=idx.device)[idx] for j in range(X.ncols)], dim=1)
    part = part.cpu().numpy()
    if world == 1:
        return part
    parts = [None] * world if dist.get_rank() == 0 else None
    dist.gather_object(part, parts, dst=0)       # rank r holds the r-th slab of grid rows: rank order is row order
    return np.concatenate(parts) if parts else None


def run_ours(args):
    import torch
    import torch.distributed as dist
    import lightkrylov_b200 as lk

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (no CPU fallback)")
    torch.cuda.set_device(local)
    if args.no_p2p:
        os.environ["LKB_P2P"] = "0"
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
        ctx = lk.Context.from_torch_distributed(local)
    else:
        ctx = lk.Context(local)
    assert world == args.gpus or world == 1, "--gpus must equal WORLD_SIZE"
    if args.no_fused:
        ctx.set_option("fused", 0)
    for o in args.opt:
        name, val = o.split("=")
        ctx.set_option(name, int(val))

    nx, ny, kdim = args.nx, args.ny, args.kdim
    n = nx * ny
    y0, nyl = lk.partition(ny, world, rank)
    nloc, row0 = nx * nyl, nx * y0
    A = lk.LinOp.stencil5(ctx, "d", nx, ny, POISSON5)
    X = lk.Basis(ctx, "d", nloc, kdim + 1, n_global=n, row0=row0)
    H = np.zeros((kdim + 1, kdim), order="F")
    x0 = X.col(0)
    x0.fill_random("uniform", 42)
    x0.scal(1.0 / x0.norm())

    ext = torch.cuda.ExternalStream(ctx.stream, device=torch.device("cuda", local))

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        ctx.sync()

    def timed(fn, reps):
        barrier()
        e0 = torch.cuda.Event(enable_timing=True); e1 = torch.cuda.Event(enable_timing=True)
        with torch.cuda.stream(ext):
            e0.record(ext)
            for _ in range(reps):
                fn()
            e1.record(ext)
        barrier()
        ms = e0.elapsed_time(e1)
        if world > 1:
            t = torch.tensor([ms], device=f"cuda:{local}", dtype=torch.float64)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t.item())
        return ms

    # ---- device-resident arm: inputs (operator, start vector) already in HBM -------------------
    def step_resident():
        info = lk.arnoldi(A, X, H)
        assert info == 0

    for _ in range(args.warmup):
        step_resident()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    l0 = ctx.kernel_launches
    ms_total = timed(step_resident, args.steps)
    launches = ctx.kernel_launches - l0
    clocks = sampler.stop() if rank == 0 else None
    value = args.steps * kdim / (ms_total * 1e-3)
    # ---- the outputs of the last timed step, taken before anything below runs the factorisation again ----------
    if args.dump_outputs:
        outputs = {"H": H.copy(), "X_sample": basis_sample(X, dump_rows(n, kdim), row0, world)}
        if rank == 0:
            os.makedirs(args.dump_outputs, exist_ok=True)
            for name, a in outputs.items():
                np.save(os.path.join(args.dump_outputs, name + ".npy"), a)

    # ---- parity record (outside the timed region): H and Ritz values of THIS run, at THIS number of ranks, against the
    # committed oracle Hessenberg matrix of the same workload (tests/golden/c2_full_H.npz, all 128 steps on the CPU) ----
    parity = None
    gold_path = os.path.join(ROOT, "tests", "golden", "c2_full_H.npz")
    if (nx, ny, kdim) == (4096, 4096, 128) and os.path.exists(gold_path):
        g = np.load(gold_path)
        Hg = g["H"]
        herr = float(np.abs(H - Hg).max() / np.abs(Hg).max())
        ritz = np.sort(np.linalg.eigvals(H[:kdim, :kdim]).real)
        rerr = float(np.abs(ritz - g["ritz"]).max() / np.abs(g["ritz"]).max())
        # ||V^H V - I||_max over the first and last 8 columns, evaluated on the device (all ranks take part in the reductions)
        Gm = X.innerprod(kdim + 1, X, wcol0=0, p=8); Gl = X.innerprod(kdim + 1, X, wcol0=kdim - 7, p=8)
        E = np.eye(kdim + 1)
        orth = float(max(np.abs(Gm - E[:, :8]).max(), np.abs(Gl - E[:, kdim - 7:]).max()))
        same = True
        if world > 1:      # H must be bitwise identical on every rank
            hs = [None] * world
            dist.all_gather_object(hs, H.tobytes())
            same = all(h == hs[0] for h in hs)
        # the same workload computed by the REFERENCE's own arnoldi sources (tests/golden/make_ref_golden_c2.py, executed by the
        # interpreter oracle/f90run.py): a second, independent comparison of this run's H (data file only -- nothing is executed)
        ref_err = None
        ref_path = os.path.join(ROOT, "tests", "golden", "ref_c2_full_H.npz")
        if os.path.exists(ref_path):
            try:
                Hr = np.load(ref_path)["H"]
                ref_err = float(np.abs(H - Hr).max() / np.abs(Hr).max())
            except Exception:                 # a damaged fixture must not take the benchmark down
                ref_err = None
        parity = {"oracle": "tests/golden/c2_full_H.npz (CPU oracle, 128 steps, same start vector)",
                  "oracle_pinned_by": "tests/golden/ref_c2_full_H.npz: this workload at full size computed by the reference's own Fortran "
                                      "sources executed by oracle/f90run.py (no Fortran compiler exists here); agrees with the oracle matrix "
                                      "to 1.1e-14 (tests/test_ref_golden.py)",
                  "max_rel_err_H_vs_reference_sources": ref_err,
                  "max_rel_err_H": herr, "max_rel_err_ritz": rerr, "orth_err_first_last_8_cols": orth,
                  "H_identical_on_all_ranks": bool(same), "tol": 1e-10, "orth_tol": 1e-12,
                  "ok": bool(herr < 1e-10 and rerr < 1e-10 and orth <= 1e-12 and same)}

    # ---- end-to-end arm: host start vector in pinned memory -> H on the host ---------------------
    x0_host = torch.empty(nloc, dtype=torch.float64).pin_memory()
    x0_host.copy_(torch.from_numpy(x0.get()))
    Hh = np.zeros((kdim + 1, kdim), order="F")
    lib = ctx.lib

    def step_e2e():
        # H2D of this step's input, normalisation (eigs' x0 handling), factorisation, H back on the host
        rc = lib.lkb_vec_put(x0.h, x0_host.data_ptr())
        assert rc == 0
        x0.scal(1.0 / x0.norm())
        info = lk.arnoldi(A, X, Hh)
        assert info == 0

    if args.no_e2e:
        ms_e2e = float("nan")
    else:
        step_e2e()
        ms_e2e = timed(step_e2e, args.steps)
    e2e_value = args.steps * kdim / (ms_e2e * 1e-3)
    # whole-job bytes per bench step: every rank uploads its slab of the start vector and reads back H + flags
    h2d = n * 8
    d2h = world * ((kdim + 1) * kdim * 8 + 32 + 2 * 16)

    # ---- per-kernel-class device time: separate profiled pass (events on the launching stream) ---
    peak, peak_src = load_peaks()
    roof = None
    kernels = {}
    if not args.no_profile_pass:
        ctx.set_profile(True)
        step_resident()
        prof = ctx.get_profile()
        ctx.set_profile(False)
        s = 8
        fused_on = prof.get("fused_axpy_dot", (0.0, 0))[1] > 0
        npass = 1 if fused_on else 2
        algb = {
            "matvec": kdim * 2 * nloc * s,
            "multidot": sum(npass * (j + 1) * nloc * s for j in range(1, kdim + 1)),   # V_j + w per launch
            "multiaxpy": sum(npass * (j + 2) * nloc * s for j in range(1, kdim + 1)),  # V_j + w read + w write
            "fused_axpy_dot": sum((j + 2) * nloc * s for j in range(1, kdim + 1)) if fused_on else 0,
            "other": kdim * 2 * nloc * s,                                              # normalisation sweep
        }
        for name, (ms, nl) in prof.items():
            gbs = algb[name] / (ms * 1e-3) / 1e9 if ms > 0 else 0.0
            kernels[name] = {"ms_total": ms, "launches": nl, "alg_bytes": algb[name], "GBps": gbs, "frac": gbs / peak}
        dom = max(("multidot", "multiaxpy", "fused_axpy_dot"), key=lambda k: kernels[k]["ms_total"])
        nl = max(kernels[dom]["launches"], 1)
        traffic_ncu = None
        try:   # DRAM bytes of ONE captured launch (j = 101) from the committed ncu capture, with its algorithmic bytes
            import glob
            tf = sorted(glob.glob(os.path.join(ROOT, "profiles", "r*_traffic.json")))[-1]
            tj = json.load(open(tf))
            t = tj.get({"multidot": "multidot", "multiaxpy": "multiaxpy_fin", "fused_axpy_dot": "axpy_dot"}[dom]) or tj.get(dom)
            if t and world == 1 and (nx, ny) == (4096, 4096):
                jcap = 101
                alg = {"multidot": jcap + 1, "multiaxpy": jcap + 2, "fused_axpy_dot": jcap + 2}[dom] * nloc * 8
                traffic_ncu = {"file": os.path.basename(tf), "j": jcap, "dram_bytes": t["dram_bytes_read"] + t["dram_bytes_write"],
                               "alg_bytes": alg, "ratio": (t["dram_bytes_read"] + t["dram_bytes_write"]) / alg}
        except Exception:
            traffic_ncu = None
        roof = {"bound": "hbm", "kernel": dom, "achieved": kernels[dom]["GBps"], "peak": peak, "unit": "GB/s",
                "frac": kernels[dom]["GBps"] / peak,
                "traffic": (traffic_ncu["ratio"] * algb[dom] / max(kernels[dom]["launches"], 1)) if traffic_ncu else None,
                "traffic_source": "NOT measured in this run: DRAM bytes / algorithmic bytes of ONE launch (j = 101) in the committed "
                                  "ncu --set full capture, scaled to this run's average launch",
                "traffic_from_committed_ncu": traffic_ncu,
                "alg_bytes_per_launch_avg": algb[dom] / nl, "avg_launch_ms": kernels[dom]["ms_total"] / nl,
                "peak_source": peak_src,
                "how": "separate profiled factorisation in the same process: CUDA events on the context stream around "
                       "every launch of the class (graphs off), algorithmic bytes summed over the launches of the class (kdim with the fused CGS2 kernel, 2*kdim without)"}
    # ---- cross-GPU exchange cost (N > 1): in-kernel %globaltimer totals of the time the last CTA of k_multidot / k_axpy_dot
    # spends in the NVLink allreduce (latency + waiting for the slowest rank), one extra factorisation, per rank ----
    sync_profile = None
    if world > 1 and ctx.p2p:
        import ctypes as C
        NW = 4 * 1024 + 16
        lk._lib.check(lib.lkb_debug_ktime(ctx.h, 1), "ktime")
        step_resident()
        buf = (C.c_uint64 * NW)()
        lk._lib.check(lib.lkb_debug_ktime_read(ctx.h, buf, NW), "ktime_read")
        lk._lib.check(lib.lkb_debug_ktime(ctx.h, 0), "ktime")
        t = np.frombuffer(buf, dtype=np.uint64).astype(np.float64)[4096:]
        mine = [t[8] / max(t[9], 1) / 1e3, t[10] / max(t[11], 1) / 1e3, int(t[9]), int(t[11])]
        allr = [None] * world
        dist.all_gather_object(allr, mine)
        sync_profile = {"what": "average time (us) per launch that the last CTA spends inside the in-kernel NVLink allreduce "
                                "(LL protocol: one-way latency + wait for the slowest rank), per rank, over one factorisation",
                        "multidot_allreduce_us": [round(a[0], 2) for a in allr], "fused_allreduce_us": [round(a[1], 2) for a in allr],
                        "launches": [allr[0][2], allr[0][3]]}
    # whole-step roofline with the official per-step bytes (matvec + 4*j*n*s), per GPU
    total_alg = sum(alg_bytes_step(j, nloc) for j in range(1, kdim + 1))
    step_gbs = total_alg * args.steps / (ms_total * 1e-3) / 1e9
    actual_b = sum((3 * j + 7) * nloc * 8 for j in range(1, kdim + 1))
    actual_gbs = actual_b * args.steps / (ms_total * 1e-3) / 1e9

    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        thr = host_threads()
        v_all, _, desc = CpuArnoldi(nx, ny, kdim, thr).sample([1, kdim // 2, kdim])
        v_one, _, desc1 = CpuArnoldi(nx, ny, kdim, 1).sample([1, 12])
        cpu = {"value": v_all, "unit": UNIT, "cores": thr, "kind": "port", "sample": desc,
               "serial": {"value": v_one, "cores": 1, "sample": desc1}}

    if rank == 0:
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms_total / args.steps, "higher_is_better": True,
            "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": WORKLOAD.format(kdim=kdim, nx=nx, ny=ny, n=n),
                       "bench_step": f"one kstart=1..kend={kdim} factorisation = {kdim} Arnoldi steps",
                       "partition": f"grid rows over {world} rank(s), {nloc} rows/rank",
                       "l2": "working set 17.3 GB/GPU-share >> 126 MB L2 (inputs larger than L2, no flush needed)",
                       "cuda_graph": True, "fused_cgs2": not args.no_fused,
                       "step_kernels": "matvec, multi-dot, fused axpy+dot (TMA ring, programmatic launch), final multi-axpy "
                                       "(predicted norm + normalisation + H column [+ halo push]), gated scale (no-op on the fast path); "
                                       "serpentine row sweeps, L1::no_allocate streaming loads",
                       "allreduce": ("in-kernel NVLink p2p" if ctx.p2p else "ncclAllReduce") if world > 1 else "none"},
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                    "ms_per_step": ms_e2e / args.steps,
                    "what": "pinned host start vector -> H2D -> normalise -> lkb_arnoldi -> Hessenberg matrix on the host"},
            "gpu_launches": int(launches),
            "roofline": roof,
            "step_roofline": {"alg_bytes_per_factorisation_per_gpu": total_alg, "achieved_GBps_per_gpu": step_gbs,
                              "frac_of_measured": step_gbs / peak, "frac_of_nominal_8TBps": step_gbs / 8000.0,
                              # what the fused step really moves: 3 sweeps of V (multi-dot, fused axpy+dot, final axpy) and
                              # 7 vector passes (matvec 2, w in pass 1, w r/w in the fused kernel, w r/w in the final pass);
                              # round 1 moved (3j+9) n s, the normalisation sweep is gone since round 2
                              "actual_bytes_per_factorisation_per_gpu": actual_b, "actual_GBps_per_gpu": actual_gbs,
                              "actual_frac_of_measured": actual_gbs / peak},
            "kernels": kernels,
            "cpu_baseline": cpu,
            "parity": parity,
            "sync_profile": sync_profile,
            "clocks": clocks,
        }
        emit(line)
    ctx.sync()
    del X, A, x0
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


_REAL_STDOUT = None


def _quiet_stdout():
    """Route fd 1 to stderr while the benchmark runs (NCCL / torchrun banners are printed to stdout by
    native code); the single JSON line is written to the saved descriptor at the end."""
    global _REAL_STDOUT
    sys.stdout.flush()
    _REAL_STDOUT = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)


def emit(line: dict):
    out = _REAL_STDOUT or sys.stdout
    out.write(json.dumps(line) + "\n")
    out.flush()


def main():
    args = parse()
    _quiet_stdout()
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
