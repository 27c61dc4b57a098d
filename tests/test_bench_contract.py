"""bench.py's reference arm (the oracle port timed on the host cores) prints ONE JSON line with the keys the driver
reads, on a tiny bounded sample; the canonical byte formula is the one of SURVEY.md 8(d); --steps and --dump-outputs
(CPU, and one GPU test of the timed CUDA fit)."""
import json
import os
import subprocess
import sys
import warnings

import numpy as np
import pytest

from helpers import col_err, rel_err

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_prints_the_contract_line():
    cmd = [sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0", "--n", "300",
           "--cpu-p", "400", "--components", "3"]
    # torchrun exports OMP_NUM_THREADS=1 to every rank: the CPU arm must still use the host's cores (VERDICT round 1)
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=300, cwd=ROOT, env=dict(os.environ, OMP_NUM_THREADS="1"))
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [ln for ln in r.stdout.splitlines() if ln.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["unit"] == "GB/s" and d["higher_is_better"] is True and d["dtype"] == "f64"
    assert d["n_gpus"] == 1 and d["steps"] == 1 and d["value"] > 0 and d["ms_per_step"] > 0
    sys.path.insert(0, ROOT)
    from oracle import refshim
    # the unmodified reference when its tree is mounted (this container), the numpy port on the GPU box
    assert d["cpu_baseline"]["kind"] == ("reference" if refshim.available() else "port")
    assert d["cpu_baseline"]["cores"] >= min(2, os.cpu_count()) and d["cpu_baseline"]["value"] == d["value"]
    assert len(d["linear_in_p"]) == 2 and all(v["gbs"] > 0 for v in d["linear_in_p"].values())
    assert d["nan_10pct"]["value"] > 0 and "nan_frac=0.1" in d["nan_10pct"]["sample"]
    assert d["e2e"] == {"value": d["value"], "unit": "GB/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert d["trips_per_component"] == [2, 2, 2]  # PLS1: two trips per component, like the reference
    assert "workload" in d["config"] and d["gpu_launches"] == 0


def test_other_ranks_of_the_reference_arm_stay_silent():
    env = dict(os.environ, RANK="1", WORLD_SIZE="2")
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2"], capture_output=True,
                       text=True, timeout=120, cwd=ROOT, env=env)
    assert r.returncode == 0 and r.stdout.strip() == ""


def test_canonical_byte_formula():
    sys.path.insert(0, ROOT)
    import bench
    # 16 n p (1 + K + sum of trips): standardise 1R+1W, per trip 2 reads, per component 1R+1W (SURVEY.md 8d)
    assert bench.fit_bytes(10_000, 1_000_000, 20, [2] * 20) == 16.0 * 10_000 * 1_000_000 * (1 + 20 + 40) == 9.76e12


def _run_dumping(args, out_dir, timeout):
    """bench.py with --dump-outputs: (the printed JSON line, {file name: array})."""
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *args, "--dump-outputs", str(out_dir)], capture_output=True,
                       text=True, timeout=timeout, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-2000:]
    line = json.loads([ln for ln in r.stdout.splitlines() if ln.startswith("{")][-1])
    return line, {f: np.load(os.path.join(out_dir, f)) for f in sorted(os.listdir(out_dir))}


# the seeded workload of the dump tests, passed explicitly so that the tests can rebuild its inputs
WORKLOAD = ["--seed", "7", "--noise", "0.02", "--decay", "0.85", "--max-iter", "200"]


def _oracle_fit(X, Y, K):
    from oracle import OracleMBPLS
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        return OracleMBPLS(n_components=K, method="NIPALS", max_iter=200).fit(X, Y)


def test_dump_outputs_of_the_reference_arm(tmp_path):
    """--dump-outputs writes the last timed fit's attributes as float64 .npy files, the same from run to run, with the
    per-feature arrays of a wide fit cut to a seeded sample of rows; the values are those of the same fit made here, row
    for row; --steps is the number of timed fits."""
    sys.path.insert(0, ROOT)
    import bench
    from oracle.cases import latent_blocks
    runs = []
    for tag, steps in (("a", 2), ("b", 1)):
        args = ["--impl", "reference", "--steps", str(steps), "--warmup", "0", "--n", "300", "--cpu-p", "40000", "--components", "3",
                "--no-nan-variant", *WORKLOAD]
        line, out = _run_dumping(args, tmp_path / tag, 300)
        assert line["steps"] == steps and len(line["step_ms"]) == steps
        runs.append(out)
    a, b = runs
    assert a.keys() == b.keys() and {"beta_.npy", "Ts_.npy", "R_.npy", "W_.0.npy", "P_.3.npy", "xs_mean.3.npy"} <= a.keys()
    for name, arr in a.items():
        assert arr.dtype == np.float64 and arr.ndim >= 1 and arr.size > 0 and np.array_equal(arr, b[name]), name
    assert a["beta_.npy"].shape == (bench.DUMP_ROWS, 1) and a["R_.npy"].shape == (bench.DUMP_ROWS, 3)  # p = 40,000 features
    assert a["Ts_.npy"].shape == (300, 3) and a["W_.0.npy"].shape == (4000, 3)
    assert sum(arr.nbytes for arr in a.values()) <= bench.DUMP_BYTES
    sizes = [max(8, int(round(40000 * s / sum(bench.SIZES_FULL)))) for s in bench.SIZES_FULL]
    X, Y = latent_blocks(300, sizes, 1, 3, seed=7, noise=0.02, decay=0.85)
    m = _oracle_fit(X, Y, 3)
    rows = np.sort(np.random.default_rng(40000).choice(40000, bench.DUMP_ROWS, replace=False))
    assert col_err(a["Ts_.npy"], m.Ts_) <= 1e-9 and col_err(a["W_.0.npy"], m.W_[0]) <= 1e-9 and col_err(a["P_.3.npy"], m.P_[3]) <= 1e-9
    assert rel_err(a["beta_.npy"], m.beta_[rows]) <= 1e-9 and col_err(a["R_.npy"], m.R_[rows]) <= 1e-9
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "0"], capture_output=True,
                       text=True, timeout=120, cwd=ROOT)
    assert r.returncode != 0 and "--steps" in r.stderr


@pytest.mark.gpu
def test_dump_outputs_of_the_timed_gpu_fit(tmp_path):
    """The CUDA arm at a small size: --steps timed fits, and the dumped attributes of two runs are bitwise equal (the inputs
    are regenerated on the device from the seed), carry the trip counts of the printed line, and match the numpy oracle
    fitted here on the same device-generated inputs."""
    import torch
    from mbpls_b200 import synth
    runs = []
    for tag, steps in (("a", 2), ("b", 3)):
        args = ["--n", "1000", "--scale", "0.002", "--components", "4", "--steps", str(steps), "--warmup", "1", "--no-e2e", "--no-cpu",
                "--no-nan-variant", "--no-configs", "--no-parity", *WORKLOAD]
        line, out = _run_dumping(args, tmp_path / tag, 600)
        assert line["steps"] == steps and len(line["step_ms"]) == steps
        assert list(out["n_iter_.npy"]) == line["trips_per_component"] == [2, 2, 2, 2]
        runs.append(out)
    a, b = runs
    assert a.keys() == b.keys() and {"beta_.npy", "Ts_.npy", "W_.0.npy", "P_.3.npy", "xs_scale.3.npy"} <= a.keys()
    for name, arr in a.items():
        assert arr.dtype == np.float64 and arr.ndim >= 1 and arr.size > 0 and np.array_equal(arr, b[name]), name
    assert a["beta_.npy"].shape == (2000, 1) and a["Ts_.npy"].shape == (1000, 4) and a["W_.3.npy"].shape == (800, 4)
    n, K, sizes, dev = 1000, 4, [200, 400, 600, 800], torch.device("cuda", 0)
    Xt = torch.zeros((sum(sizes), n), dtype=torch.float64, device=dev)
    synth.fill_feature_major(Xt, n, 0, sum(sizes), K, 7, noise=0.02, decay=0.85)
    X = Xt.t().cpu().numpy()
    edges = np.cumsum([0] + sizes)
    m = _oracle_fit([np.ascontiguousarray(X[:, edges[b]:edges[b + 1]]) for b in range(len(sizes))],
                    synth.response(n, 1, K, dev, 7, decay=0.85).cpu().numpy(), K)
    assert list(m.n_iter_) == [2, 2, 2, 2] and col_err(a["Ts_.npy"], m.Ts_) <= 1e-8 and rel_err(a["beta_.npy"], m.beta_) <= 1e-8
    for b in range(len(sizes)):
        assert col_err(a[f"W_.{b}.npy"], m.W_[b]) <= 1e-8 and col_err(a[f"P_.{b}.npy"], m.P_[b]) <= 1e-8, b
        assert rel_err(a[f"xs_scale.{b}.npy"], m.x_scalers_[b].scale_) <= 1e-12, b
