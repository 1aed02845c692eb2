"""bench.py contract checks that run without a GPU: the reference (CPU oracle) arm prints exactly one JSON
line on stdout with the keys the driver reads, and the own arm fails loudly without a CUDA device."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_json_line():
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--nx", "192", "--ny", "160",
                        "--kdim", "32", "--steps", "2", "--warmup", "1"], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [ln for ln in r.stdout.splitlines() if ln.strip()]
    assert len(lines) == 1, lines
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == "arnoldi_steps_per_s" and d["unit"] == "steps/s"
    assert d["higher_is_better"] is True and d["value"] > 0 and d["steps"] == 2 and d["warmup"] == 1
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1 and d["cpu_baseline"]["value"] == d["value"]
    assert d["e2e"] == {"value": d["value"], "unit": "steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert d["vs_baseline"] is None and d["dtype"] == "f64" and "workload" in d["config"]


def test_reference_arm_other_ranks_exit_quietly():
    env = dict(os.environ, RANK="1", WORLD_SIZE="2", LOCAL_RANK="1")
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2", "--nx", "64",
                        "--ny", "64", "--kdim", "8", "--steps", "1", "--warmup", "0"], capture_output=True, text=True,
                       timeout=120, env=env)
    assert r.returncode == 0 and r.stdout.strip() == ""


def test_arguments_are_checked_before_any_work():
    for extra in (["--steps", "0"], ["--impl", "reference", "--dump-outputs", "out"], ["--kdim", "4096", "--dump-outputs", "out"]):
        r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py")] + extra, capture_output=True, text=True, timeout=120)
        assert r.returncode == 2 and r.stdout.strip() == "", (extra, r.stderr[-2000:])


@pytest.mark.gpu
def test_dump_outputs_match_the_oracle_and_steps_set_the_timed_work(oracle, tmp_path):
    """--dump-outputs writes H and a seeded row sample of the basis; both agree with the oracle's factorisation of the
    same seeded start vector and are bitwise the same whatever the number of timed steps.  --steps 3 launches three
    times the kernels of --steps 1 inside the timed region."""
    sys.path.insert(0, ROOT)
    import bench
    nx, ny, kdim = 192, 160, 32
    n = nx * ny
    x0 = oracle.fill(n, "d", "uniform", 42); oracle.normalize(x0)
    Xo = np.zeros((n, kdim + 1), order="F"); Xo[:, 0] = x0
    Ho = np.zeros((kdim + 1, kdim), order="F")
    assert oracle.arnoldi(oracle.Op.stencil("d", (nx, ny), bench.POISSON5), Xo, Ho) == 0
    rows = bench.dump_rows(n, kdim)
    assert rows.size == min(n, bench.DUMP_ROWS)
    dumps, launches = [], []
    for steps in ("1", "3"):
        out = tmp_path / steps
        r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--nx", str(nx), "--ny", str(ny), "--kdim", str(kdim),
                            "--steps", steps, "--warmup", "1", "--no-cpu-baseline", "--no-profile-pass", "--no-e2e",
                            "--dump-outputs", str(out)], capture_output=True, text=True, timeout=600)
        assert r.returncode == 0, r.stderr[-4000:]
        line = json.loads(r.stdout.strip().splitlines()[-1])
        assert line["steps"] == int(steps)
        launches.append(line["gpu_launches"])
        H, Xs = np.load(out / "H.npy"), np.load(out / "X_sample.npy")
        assert sorted(os.listdir(out)) == ["H.npy", "X_sample.npy"]
        assert H.dtype == Xs.dtype == np.float64 and H.shape == Ho.shape and Xs.shape == (rows.size, kdim + 1)
        assert np.abs(H - Ho).max() < 1e-10 * np.abs(Ho).max()
        assert np.abs(Xs - Xo[rows]).max() < 1e-10 * np.abs(Xo[rows]).max()
        dumps.append((H, Xs))
    assert all(np.array_equal(a, b) for a, b in zip(*dumps))
    assert launches[0] > 0 and launches[1] == 3 * launches[0], launches


def test_own_arm_needs_a_gpu():
    import torch
    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "1", "--warmup", "1"],
                       capture_output=True, text=True, timeout=300)
    assert r.returncode != 0 and "CUDA" in (r.stderr + r.stdout)
    assert not [ln for ln in r.stdout.splitlines() if ln.startswith("{")]     # no number without a GPU
