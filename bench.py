#!/usr/bin/env python
"""bench.py -- MB-PLS NIPALS fit throughput on B200 (BASELINE.json: "MB-PLS fit s & HBM GB/s
(n=10k, p=1M, 20 LV) at 1/2/4/8 B200 vs host CPU").

One *step* = one complete fp64 multiblock NIPALS fit (column standardisation, 20 latent variables,
finalisation of R_/beta_) of n=10,000 samples x p=1,000,000 features in 4 blocks (100k/200k/300k/400k)
with a single response (PLS1: the NIPALS loop takes exactly 2 trips per component, so the work per
step is data-independent; see DESIGN.md "Benchmark workload").  Synthetic latent-structure data is
generated on the device (feature-major); because `fit` standardises and deflates X in place the input
is regenerated before every step, outside the timed region.

metric/unit: algorithmic HBM GB/s = 16*n*p*(1 + K + sum_k I_k) bytes / fit seconds (SURVEY.md 8d: the traffic of an
exact two-pass NIPALS); `fit_s` is the absolute time.  The one-pass kernels (csrc/fused.cu) read X once per trip, so
the canonical figure can exceed the HBM peak; `hbm_gbs_actual_traffic` / `passes_over_X_per_step` report what the
kernels really move and `roofline` times the dominant kernel against its own bytes.  N > 1: the feature axis is sharded (strong scaling), one NCCL
all-reduce of the (n x B + B) partial block scores per trip.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--dump-outputs DIR]

--dump-outputs DIR writes the fitted attributes of the last timed fit as DIR/<name>.npy (see dump_outputs), so that two
builds can be compared output for output on the same seeded inputs.  With N > 1 GPUs rank 0 writes them, and the
per-feature attributes (W_, P_, R_, beta_, the scalers) are its shard of the features.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import time
import warnings

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "MB-PLS NIPALS fit: algorithmic HBM GB/s (n=10k, p=1M, 4 blocks, 20 LV, fp64)"
SIZES_FULL = (100_000, 200_000, 300_000, 400_000)


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--n", type=int, default=10_000)
    ap.add_argument("--scale", type=float, default=1.0, help="scale the feature counts (debug / small GPUs)")
    ap.add_argument("--components", type=int, default=20)
    ap.add_argument("--q", type=int, default=1)
    ap.add_argument("--nan-frac", type=float, default=0.0)
    ap.add_argument("--max-iter", type=int, default=200, help="safety cap on trips per component for both arms")
    ap.add_argument("--noise", type=float, default=0.02)
    ap.add_argument("--decay", type=float, default=0.85)
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-nan-variant", action="store_true", help="skip the extra 10 %% NaN fit reported under `variants`")
    ap.add_argument("--two-pass", action="store_true", help="force the two-pass NIPALS kernels (X'u and X w as separate reads)")
    ap.add_argument("--e2e-steps", type=int, default=1)
    ap.add_argument("--cpu-p", type=int, default=0, help="features of the CPU sample (0: auto)")
    ap.add_argument("--no-configs", action="store_true", help="skip the other BASELINE configurations (C2 / C3 q=10 / C5) reported under `configs`")
    ap.add_argument("--no-parity", action="store_true", help="skip the in-bench parity gate (GPU fit vs numpy oracle on a column slice)")
    ap.add_argument("--parity-features", type=int, default=1024, help="features per block of the dense parity slice (NaN slice: a quarter)")
    ap.add_argument("--seed", type=int, default=20261017)
    ap.add_argument("--verbose", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write the fitted attributes of the last timed fit as DIR/<name>.npy "
                         "(N > 1 GPUs: rank 0 writes, per-feature attributes are its feature shard)")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be at least 1 and --warmup at least 0")
    return args


VERBOSE = False
_T0 = time.time()


def log(*a):
    if VERBOSE:
        print(f"[bench +{time.time() - _T0:7.1f}s]", *a, file=sys.stderr, flush=True)


def fit_bytes(n, p, K, trips):
    """Canonical algorithmic traffic of one NIPALS fit (SURVEY.md 8d / BASELINE.md section 4)."""
    return 16.0 * n * p * (1 + K + sum(trips))


DUMP_BYTES = 64 << 20   # --dump-outputs: at most this much in all
DUMP_ROWS = 16384       # ... and at first this many rows of an array; halved until the budget holds


def dump_outputs(model, out_dir, write=True):
    """Fitted attributes of `model` -- every array the golden fixtures record (oracle.make_golden.snapshot) and the NIPALS
    trip counts -- as out_dir/<name>.npy in float64 ("T_/0" -> "T_.0.npy"; integer arrays widened, scalars stored as one
    element; empty arrays such as the W_concat_ of a fit that never builds it hold nothing to compare and are left out).
    An array with more rows than the row budget (the per-feature results of the full-size workload) keeps a sorted sample of rows drawn from a
    generator seeded with its row count, so two builds keep the same rows.  Every rank must call this (materialising the
    attributes may communicate); only `write` ranks write."""
    import numpy as np
    from oracle.make_golden import snapshot
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        arrays = snapshot(model)
        if hasattr(model, "n_iter_"):
            arrays["n_iter_"] = np.asarray(model.n_iter_)
    if not write:
        return
    arrays = {k.replace("/", "."): np.atleast_1d(np.asarray(v, dtype=np.float64)) for k, v in arrays.items() if np.size(v) > 0}

    def sample(a, rows):
        if a.shape[0] <= rows:
            return a
        return a[np.sort(np.random.default_rng(a.shape[0]).choice(a.shape[0], rows, replace=False))]

    rows = DUMP_ROWS
    out = {k: sample(a, rows) for k, a in arrays.items()}
    while rows > 1 and sum(a.nbytes for a in out.values()) > DUMP_BYTES:
        rows //= 2
        out = {k: sample(a, rows) for k, a in arrays.items()}
    os.makedirs(out_dir, exist_ok=True)
    for k, a in out.items():
        np.save(os.path.join(out_dir, k + ".npy"), a)


# ------------------------------------------------------------------------------------------------
# reference arm / cpu_baseline: the numpy oracle port of mbpls/mbpls.py on the host cores
# ------------------------------------------------------------------------------------------------
CPU_P_DENSE = 20_000        # BASELINE.md section 3: dense CPU sample at n=10,000 x p=20,000 ...
CPU_P_SECOND = 10_000       # ... and a second width to show the time is linear in p
CPU_NAN_SHAPE = (2_000, 4_000)  # NaN-mode CPU sample (Python-loop-bound on the host, BASELINE.md section 3)


def _host_threads():
    """All host cores for BLAS, whatever OMP_NUM_THREADS said at import (torchrun exports OMP_NUM_THREADS=1)."""
    import threadpoolctl
    return threadpoolctl.threadpool_limits(limits=os.cpu_count())


def cpu_sample(args, p_sample, repeats=1, n=None, nan_frac=None):
    """One bounded CPU fit of the benchmark's workload shape: the reference's own MBPLS (unmodified, through the
    check_array shim of oracle/refshim.py) when /root/reference is mounted, else the numpy port (oracle/mbpls_oracle.py)."""
    import numpy as np
    import threadpoolctl
    from oracle import OracleMBPLS, refshim
    from oracle.cases import latent_blocks
    n = args.n if n is None else n
    nan_frac = args.nan_frac if nan_frac is None else nan_frac
    K = args.components
    frac = [s / sum(SIZES_FULL) for s in SIZES_FULL]
    sizes = [max(8, int(round(p_sample * f))) for f in frac]
    X, Y = latent_blocks(n, sizes, args.q, K, seed=args.seed % 100000, noise=args.noise, decay=args.decay, nan_frac=nan_frac)
    use_ref = refshim.available()
    times, trips = [], None
    with _host_threads():
        info = threadpoolctl.threadpool_info()
        threads = max([i.get("num_threads", 1) for i in info] or [1])
        for _ in range(repeats):
            Xc, Yc = [x.copy() for x in X], Y.copy()
            with warnings.catch_warnings():
                warnings.simplefilter("ignore")
                if use_ref:
                    m = refshim.load()(n_components=K, method='NIPALS', sparse_data=nan_frac > 0)
                    t0 = time.perf_counter()
                    m.fit(Xc, Yc)
                    dt = time.perf_counter() - t0
                    trips = trips or [2] * K if args.q == 1 else None  # the reference does not expose its trip counts
                else:
                    m = OracleMBPLS(n_components=K, method="NIPALS", sparse_data=nan_frac > 0, max_iter=args.max_iter)
                    t0 = time.perf_counter()
                    m.fit(Xc, Yc)
                    dt = time.perf_counter() - t0
                    trips = list(m.n_iter_)
            times.append(dt)
    if trips is None:  # PLS2 through the real reference: count the trips once with the (untimed) port
        with warnings.catch_warnings():
            warnings.simplefilter("ignore")
            trips = list(OracleMBPLS(n_components=K, method="NIPALS", sparse_data=nan_frac > 0, max_iter=args.max_iter)
                         .fit([x.copy() for x in X], Y.copy()).n_iter_)
    p = sum(sizes)
    best = min(times)
    what = "mbpls/mbpls.py of the reference (unmodified, check_array shim)" if use_ref else "oracle numpy/OpenBLAS port of mbpls.py"
    return dict(seconds=best, mean_seconds=sum(times) / len(times), gbs=fit_bytes(n, p, K, trips) / best / 1e9, trips=trips,
                cores=threads, kind="reference" if use_ref else "port", p=p, n=n, model=m,
                sample=f"{what}, NIPALS, n={n}, p={p} in 4 blocks, q={args.q}, K={K}, nan_frac={nan_frac}, "
                       f"{threads} BLAS threads of {os.cpu_count()} cpus, best of {repeats}")


def cpu_p_for_budget(args, budget_s):
    """The CPU sample is p = 20,000 features (BASELINE.md section 3) unless one fit at ~8 GB/s would not fit `budget_s`."""
    if args.cpu_p:
        return args.cpu_p
    per_feature = 16.0 * args.n * (1 + args.components + (2 if args.q == 1 else 40) * args.components) / 8e9
    return int(max(1_000, min(CPU_P_DENSE, budget_s / per_feature)))


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    steps, warm = max(1, args.steps), max(0, args.warmup)
    p_sample = cpu_p_for_budget(args, max(4.0, 170.0 / (steps + warm)))
    for _ in range(warm):
        cpu_sample(args, p_sample)
    times, res = [], None
    for _ in range(steps):
        res = cpu_sample(args, p_sample)
        times.append(res["seconds"])
    if args.dump_outputs:
        dump_outputs(res["model"], args.dump_outputs)
    sec = sum(times) / len(times)
    gbs = res["gbs"] * res["seconds"] / sec
    # a second width: the fit time is linear in p (so GB/s at the sample width stands for the full width), and the NaN-mode
    # sample that goes with variants.nan_10pct of the GPU arm
    second = cpu_sample(args, max(500, p_sample // 2))
    extra = {"linear_in_p": {str(res["p"]): {"seconds": min(times), "gbs": res["gbs"] * res["seconds"] / min(times)},
                             str(second["p"]): {"seconds": second["seconds"], "gbs": second["gbs"]}}}
    if args.nan_frac == 0 and not args.no_nan_variant:
        nn, pp = min(CPU_NAN_SHAPE[0], args.n), min(CPU_NAN_SHAPE[1], p_sample)
        nan = cpu_sample(args, pp, n=nn, nan_frac=0.10)
        extra["nan_10pct"] = {"value": nan["gbs"], "unit": "GB/s", "seconds": nan["seconds"], "cores": nan["cores"], "kind": nan["kind"],
                              "sample": nan["sample"]}
    line = {
        "impl": "reference", "metric": METRIC, "value": gbs, "unit": "GB/s", "n_gpus": args.gpus, "steps": len(times),
        "warmup": warm, "ms_per_step": sec * 1e3, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
        "dtype": "f64", "data": "synthetic",
        "config": workload_config(args, note=f"bounded CPU sample: p={res['p']} features instead of {int(sum(SIZES_FULL) * args.scale)} "
                                             "(fit time is linear in p, see linear_in_p); GB/s is size-normalised"),
        "trips_per_component": res["trips"], "best_of_steps_s": min(times),
        "cpu_baseline": {"value": gbs, "unit": "GB/s", "cores": res["cores"], "kind": res["kind"], "sample": res["sample"]},
        "e2e": {"value": gbs, "unit": "GB/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0, "step_ms": [t * 1e3 for t in times], **extra,
    }
    print(json.dumps(line), flush=True)


def workload_config(args, note=None):
    sizes = [int(s * args.scale) for s in SIZES_FULL]
    cfg = {"workload": f"NIPALS MB-PLS fit n={args.n} p={sum(sizes)} blocks={sizes} q={args.q} K={args.components} "
                       f"nan_frac={args.nan_frac} standardize=True calc_all=True max_tol=1e-14; latent-structure data "
                       f"(r=K+5 factors, decay {args.decay}, noise {args.noise})",
           "parallelism": f"feature-sharded x{args.gpus}", "l2_policy": "inputs (>=10 GB per GPU) larger than the 126 MB L2",
           "timing": "per-step CUDA-event bracket (barrier + synchronize both sides); X regenerated between steps outside it"}
    if note:
        cfg["note"] = note
    return cfg


# ------------------------------------------------------------------------------------------------
# parity gate (SURVEY.md 8d "parity gate run with every benchmark"; mbpls/tests/test_mbpls.py:66-117 is the model)
# ------------------------------------------------------------------------------------------------
def _col_err(o, r):
    """max over components of the relative error after sign alignment (columns are components)."""
    import numpy as np
    o, r = np.asarray(o, float), np.asarray(r, float)
    if o.shape != r.shape:
        return float("inf")
    worst = 0.0
    for k in range(r.shape[1]):
        den = np.linalg.norm(r[:, k]) or 1.0
        worst = max(worst, min(np.linalg.norm(o[:, k] - r[:, k]), np.linalg.norm(o[:, k] + r[:, k])) / den)
    return float(worst)


def parity_gate(args, dev, group, rank, world, nan_frac, feats_per_block):
    """The SAME device-generated data the timed fits use -- the first `feats_per_block` features of each of the 4 blocks,
    all n samples, same Y -- fitted (a) by the GPU path, feature-sharded over the ranks of this run exactly like the timed
    fit, and (b) on rank 0 by the numpy oracle (oracle/mbpls_oracle.py, the restatement of mbpls/mbpls.py pinned to the
    reference's golden vectors).  Reports the worst per-component relative error after sign alignment over
    Ts_, T_, W_, P_, U_, V_ and of beta_ / A_ (no alignment), whether the NIPALS trip counts are equal, and (NaN variant)
    whether the NaN census and the scalers' observed counts are equal."""
    import numpy as np
    import torch
    import torch.distributed as dist
    from mbpls_b200 import MBPLS, synth
    from mbpls_b200 import engine as E
    n, K, q = args.n, args.components, args.q
    full = [int(s * args.scale) for s in SIZES_FULL]
    starts = [sum(full[:b]) for b in range(len(full))]
    sizes = [min(feats_per_block, s) for s in full]
    ld = E.round_ld(n)
    shard = E.ShardMap.build(sizes, rank, world)
    Yd = synth.response(n, q, K, dev, args.seed, decay=args.decay)

    def gen(dst, b, c0, c1):  # features [c0, c1) of the slice of block b == global features starts[b] + [c0, c1)
        synth.fill_feature_major(dst, n, starts[b] + c0, starts[b] + c1, K, args.seed, noise=args.noise, decay=args.decay,
                                 nan_frac=nan_frac)

    Xl = torch.zeros((max(shard.p_local, 1), ld), dtype=torch.float64, device=dev)
    for b, (c0, c1) in enumerate(shard.local_ranges):
        if c1 > c0:
            gen(Xl[shard.block_off[b]:shard.block_off[b + 1]], b, c0, c1)
    local = [Xl[shard.block_off[b]:shard.block_off[b + 1], :n].t() for b in range(len(sizes))]
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        m = MBPLS(n_components=K, method="NIPALS", standardize=True, calc_all=True, sparse_data=nan_frac > 0, copy=True)
        m.set_runtime(device=dev, group=group, materialize=True, global_sizes=sizes if world > 1 else None, max_iter=args.max_iter,
                      one_pass=False if args.two_pass else None, gather="all")  # rank 0 compares the complete attributes
        m.fit(local, Yd)
    out = None
    if rank == 0:
        import threadpoolctl
        from oracle import OracleMBPLS
        host = []
        for b, pb in enumerate(sizes):
            t = torch.zeros((pb, ld), dtype=torch.float64, device=dev)
            gen(t, b, 0, pb)
            host.append(np.ascontiguousarray(t[:, :n].t().cpu().numpy()))
            del t
        Yh = Yd.cpu().numpy()
        t0 = time.perf_counter()
        with warnings.catch_warnings(), threadpoolctl.threadpool_limits(limits=os.cpu_count()):
            warnings.simplefilter("ignore")
            o = OracleMBPLS(n_components=K, method="NIPALS", sparse_data=nan_frac > 0, max_iter=args.max_iter).fit(
                [x.copy() for x in host], Yh.copy())
        oracle_s = time.perf_counter() - t0
        errs = {"Ts_": _col_err(m.Ts_, o.Ts_), "U_": _col_err(m.U_, o.U_), "V_": _col_err(m.V_, o.V_),
                "T_": max(_col_err(a, b_) for a, b_ in zip(m.T_, o.T_)), "W_": max(_col_err(a, b_) for a, b_ in zip(m.W_, o.W_)),
                "P_": max(_col_err(a, b_) for a, b_ in zip(m.P_, o.P_)),
                "beta_": float(np.linalg.norm(m.beta_ - o.beta_) / np.linalg.norm(o.beta_)),
                "A_": float(np.linalg.norm(m.A_ - o.A_) / np.linalg.norm(o.A_))}
        census_equal = None
        if nan_frac > 0:
            census_equal = all(np.array_equal(a, b_) for blk in range(len(sizes))
                               for a, b_ in zip(m.sparse_X_info_[blk], o.sparse_X_info_[blk]))
            census_equal = bool(census_equal and all(
                np.array_equal(np.asarray(a.n_samples_seen_), np.asarray(b_.n_samples_seen_)) for a, b_ in zip(m.x_scalers_, o.x_scalers_)))
        worst = max(errs.values())
        out = {"max_rel_err": worst, "per_attribute": errs, "trips_equal": list(m.n_iter_) == list(o.n_iter_),
               "trips_gpu": list(m.n_iter_), "trips_oracle": list(o.n_iter_), "census_equal": census_equal,
               "tolerance": 1e-8, "ok": bool(worst <= 1e-8 and list(m.n_iter_) == list(o.n_iter_) and census_equal is not False),
               "oracle_seconds": oracle_s,
               "slice": f"first {sizes} features of the 4 blocks of the benchmark's device-generated data (global starts {starts}), "
                        f"all n={n} samples, K={K}, q={q}, nan_frac={nan_frac}; GPU fit feature-sharded over {world} rank(s); "
                        "oracle = oracle/mbpls_oracle.py (numpy restatement of mbpls/mbpls.py) on rank 0"}
    del m, Xl
    if world > 1:
        dist.barrier(group=group)
    return out


# ------------------------------------------------------------------------------------------------
# the other BASELINE.json configurations, measured in the same run (reported under `configs`)
# ------------------------------------------------------------------------------------------------
def fp64_peaks(dev):
    """cuBLAS DGEMM and DSYRK rates on this GPU (8192^3, best of 3): the FP64 roofline SURVEY.md 8(d) asks to measure once
    per box.  DSYRK is credited n^2 k flops (the executed half)."""
    import ctypes
    import glob
    import torch
    N = 8192
    A = torch.randn((N, N), dtype=torch.float64, device=dev)
    out = {}

    def best(fn, reps=3):
        fn()
        torch.cuda.synchronize(dev)
        ts = []
        for _ in range(reps):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            fn()
            e1.record()
            torch.cuda.synchronize(dev)
            ts.append(e0.elapsed_time(e1))
        return min(ts)

    ms = best(lambda: torch.matmul(A, A.t()))
    out["dgemm_tflops"] = 2.0 * N ** 3 / ms / 1e9
    try:
        libs = glob.glob(os.path.join(os.path.dirname(torch.__file__), "..", "nvidia", "cublas", "lib", "libcublas.so*")) + \
            glob.glob(os.path.join(os.path.dirname(torch.__file__), "lib", "libcublas.so*")) + ["libcublas.so.12"]
        lib = None
        for path in libs:
            try:
                lib = ctypes.CDLL(path)
                break
            except OSError:
                continue
        Cm = torch.zeros((N, N), dtype=torch.float64, device=dev)
        one, zero = ctypes.c_double(1.0), ctypes.c_double(0.0)
        handle = ctypes.c_void_p(torch.cuda.current_blas_handle())
        lib.cublasDsyrk_v2.restype = ctypes.c_int
        lib.cublasDsyrk_v2.argtypes = [ctypes.c_void_p, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_void_p,
                                       ctypes.c_void_p, ctypes.c_int, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int]

        def syrk():  # C = A A' (column-major view of the same buffer), upper triangle
            rc = lib.cublasDsyrk_v2(handle, 1, 0, N, N, ctypes.byref(one), ctypes.c_void_p(A.data_ptr()), N, ctypes.byref(zero),
                                    ctypes.c_void_p(Cm.data_ptr()), N)
            if rc != 0:
                raise RuntimeError(f"cublasDsyrk status {rc}")
        ms = best(syrk)
        out["dsyrk_tflops_executed"] = 1.0 * N ** 3 / ms / 1e9
    except Exception as exc:  # the probe must never take the benchmark line down
        out["dsyrk_error"] = repr(exc)[:160]
    return out


def run_configs(args, dev, group, rank, world, peak_gbs):
    """BASELINE.json configs 2, 3 and 5 on device-generated data of their full size (fp64, same generator as the headline):
    time, algorithmic bytes or flops, and the fraction of the measured HBM / FP64 peak.  N > 1: C3 and C2-SIMPLS shard the
    feature axis, C5 KERNEL / UNIPALS shard the sample axis (p x p, resp. per-component p-vector all-reduces)."""
    import numpy as np
    import torch
    import torch.distributed as dist
    from mbpls_b200 import MBPLS, synth
    from mbpls_b200 import engine as E
    out = {}
    sc = args.scale

    def sync_max(seconds):
        t = torch.tensor([seconds], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX, group=group)
        return float(t.item())

    def barrier():
        if world > 1:
            dist.barrier(group=group)
        torch.cuda.synchronize(dev)

    def timed(fn, reps=2):
        best, res = None, None
        for _ in range(reps):
            prep = fn(None)
            barrier()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            with warnings.catch_warnings():
                warnings.simplefilter("ignore")
                res = fn(prep)
            e1.record()
            barrier()
            dt = sync_max(e0.elapsed_time(e1) / 1e3)
            best = dt if best is None else min(best, dt)
        return best, res

    peaks = fp64_peaks(dev) if rank == 0 else {}
    out["fp64_peaks"] = peaks
    fp64_peak = max(peaks.get("dgemm_tflops", 0.0), 1e-9)

    # ---- C3: 8 uneven blocks, n = 2,000, Y n x 10 (the reference paper's own q, runtime_analysis_rowincrease.py:58), K = 20
    n, K, q = 2000, 20, 10
    sizes = [int(s * sc) for s in (20000, 35000, 60000, 95000, 140000, 180000, 220000, 450000)]
    shard = E.ShardMap.build(sizes, rank, world)
    ld = E.round_ld(n)
    Xb = torch.empty((max(shard.p_local, 1), ld), dtype=torch.float64, device=dev)
    Yd = synth.response(n, q, K, dev, args.seed + 3, decay=args.decay)

    def c3(prep):
        if prep is None:
            synth.fill_feature_major(Xb, n, shard.lo, shard.hi, K, args.seed + 3, noise=args.noise, decay=args.decay)
            return True
        blocks = [Xb[shard.block_off[b]:shard.block_off[b + 1], :n].t() for b in range(len(sizes))]
        prof = {}
        m = MBPLS(n_components=K, method="NIPALS", copy=False).set_runtime(device=dev, group=group, materialize=False,
                                                                           global_sizes=sizes, max_iter=2000, profile=prof).fit(blocks, Yd)
        return m, prof

    dt, (m, prof) = timed(c3)
    trips = list(m.n_iter_)
    p = sum(sizes)
    passes = sum(len(prof.get(k, [])) * w for k, w in (("trip", 1), ("xtu", 1), ("xw", 1), ("deflate", 2), ("loadings", 1), ("standardize", 2)))
    out["c3_pls2_q10_nipals"] = {
        "workload": f"NIPALS n={n} p={p} blocks={sizes} q={q} K={K}", "fit_s": dt, "trips_per_component": trips, "trips_total": sum(trips),
        "value": fit_bytes(n, p, K, trips) / dt / 1e9, "unit": "GB/s (canonical two-pass bytes)",
        "hbm_gbs_actual_traffic": passes * 8.0 * n * p / dt / 1e9, "frac_of_hbm_peak_actual_traffic": passes * 8.0 * n * p / dt / 1e9 / (peak_gbs * world),
        "ms_per_trip": dt / max(sum(trips), 1) * 1e3}
    del m, Xb

    # ---- C2: single-block PLS1, n = 5,000 x p = 50,000, K = 10: KERNEL (P > N: XX' on the FP64 tensor cores) and SIMPLS
    n, K, q = 5000, 10, 1
    sizes = [int(50000 * sc)]
    p = sizes[0]
    shard = E.ShardMap.build(sizes, rank, world)
    ld = E.round_ld(n)
    Xb = torch.empty((max(shard.p_local, 1), ld), dtype=torch.float64, device=dev)
    Yd = synth.response(n, q, K, dev, args.seed + 2, decay=args.decay)
    for method in ("KERNEL", "SIMPLS"):
        def c2(prep, method=method):
            if prep is None:
                synth.fill_feature_major(Xb, n, shard.lo, shard.hi, K, args.seed + 2, noise=args.noise, decay=args.decay)
                return True
            blocks = [Xb[:shard.p_local, :n].t()]
            return MBPLS(n_components=K, method=method, copy=False, full_svd=True).set_runtime(
                device=dev, group=group, materialize=False, global_sizes=sizes).fit(blocks, Yd)
        dt, m = timed(c2)
        ent = {"workload": f"{method} PLS1 n={n} p={p} K={K} calc_all=True", "fit_s": dt}
        if method == "KERNEL":
            flops = 2.0 * n * n * p  # XX' as a GEMM; the symmetric kernel executes half
            ent.update({"crossproduct_flops_as_gemm": flops, "tflops_whole_fit_as_gemm": flops / dt / 1e12,
                        "frac_of_measured_dgemm_whole_fit": flops / dt / 1e12 / (fp64_peak * world) if peaks else None,
                        "note": "whole fit (cross product + K rank-2 deflations of the n x n matrix + calc_all passes) over the GEMM-credited flops"})
        else:
            bts = 8.0 * n * p * (1 + 2 * K)
            ent.update({"algorithmic_bytes": bts, "value": bts / dt / 1e9, "unit": "GB/s", "frac_of_hbm_peak": bts / dt / 1e9 / (peak_gbs * world)})
        out[f"c2_pls1_{method.lower()}"] = ent
        del m
    del Xb

    # ---- C5: tall n = 1,000,000 x p = 2,000 (2 blocks), q = 4, K = 30: KERNEL and UNIPALS (n >> p), then batched predict
    n, K, q = int(1_000_000 * sc), 30, 4
    sizes = [1000, 1000]
    p = sum(sizes)
    ld = E.round_ld(n)
    Xb = torch.empty((p, ld), dtype=torch.float64, device=dev)  # N > 1: every rank generates the matrix and ingests its rows
    Yd = synth.response(n, q, K, dev, args.seed + 5, decay=0.9)
    model = None
    for method in ("KERNEL", "UNIPALS"):
        def c5(prep, method=method):
            if prep is None:
                synth.fill_feature_major(Xb, n, 0, p, K, args.seed + 5, noise=args.noise, decay=0.9)
                return True
            blocks = [Xb[:1000, :n].t(), Xb[1000:, :n].t()]
            return MBPLS(n_components=K, method=method, copy=world > 1, full_svd=True, calc_all=False).set_runtime(
                device=dev, group=group, materialize=False).fit(blocks, Yd)
        dt, m = timed(c5, reps=2 if method == "KERNEL" else 1)
        ent = {"workload": f"{method} n={n} p={p} (2 blocks) q={q} K={K} calc_all=False; " +
                           ("sample axis sharded over the ranks" if world > 1 else "one GPU"), "fit_s": dt}
        if method == "KERNEL":
            flops = 2.0 * n * p * p
            ent.update({"crossproduct_flops_as_gemm": flops, "tflops_whole_fit_as_gemm": flops / dt / 1e12,
                        "frac_of_measured_dgemm_whole_fit": flops / dt / 1e12 / (fp64_peak * world) if peaks else None})
            model = m
        else:
            bts = 8.0 * n * p * (1 + 4 * K)  # standardise + per component: X'Y, X w, X'ts (reads) and the deflation (R+W) ~ 5, fused: 4
            ent.update({"x_bytes": 8.0 * n * p, "seconds_per_component": dt / K,
                        "x_passes_per_component_equivalent": dt / K / (8.0 * n * p / (peak_gbs * 1e9 * world)),
                        "note": "x_passes_per_component_equivalent = time per component / time of one read of X at the measured HBM peak"})
        out[f"c5_tall_{method.lower()}"] = ent
        if method != "KERNEL":
            del m
    # batched predict on a fresh tall batch (device-resident feature-major input, numpy output)
    synth.fill_feature_major(Xb, n, 0, p, K, args.seed + 6, noise=args.noise, decay=0.9)
    blocks = [Xb[:1000, :n].t(), Xb[1000:, :n].t()]
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        model.predict(blocks)
        barrier()
        t0 = time.perf_counter()
        yh = model.predict(blocks)
        torch.cuda.synchronize(dev)
        dt = sync_max(time.perf_counter() - t0)
    out["c5_predict"] = {"workload": f"predict {n} x {p} -> {tuple(yh.shape)} (replicated model, every rank predicts the whole batch)",
                         "predict_s": dt, "rows_per_s": n / dt, "value": 8.0 * n * p / dt / 1e9, "unit": "GB/s",
                         "frac_of_hbm_peak": 8.0 * n * p / dt / 1e9 / peak_gbs}
    del model, Xb, yh
    torch.cuda.empty_cache()
    return out


# ------------------------------------------------------------------------------------------------
# clocks sampler (B200_PROFILING.md)
# ------------------------------------------------------------------------------------------------
class Clocks:
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.proc, self.path = None, f"/tmp/mbpls_clocks_{os.getpid()}.csv"
        try:
            self.f = open(self.path, "w")
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "200",
                                          "-i", str(index)], stdout=self.f, stderr=subprocess.DEVNULL)
        except Exception:
            self.proc = None

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": []}
        if self.proc is None:
            return out
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        self.f.close()
        sm, mx, reasons = [], [], set()
        for ln in open(self.path):
            parts = [x.strip() for x in ln.split(",")]
            if len(parts) < 9:
                continue
            try:
                sm.append(float(parts[1])); mx.append(float(parts[2]))
            except ValueError:
                continue
            for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), parts[5:9]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        if sm:
            busy = [s for s in sm if s > 0]
            out = {"sm_mhz": statistics.median(busy), "sm_max_mhz": max(mx), "reasons": sorted(reasons), "samples": len(sm)}
        try:
            os.remove(self.path)
        except OSError:
            pass
        return out


# ------------------------------------------------------------------------------------------------
# our arm
# ------------------------------------------------------------------------------------------------
def run_ours(args):
    import numpy as np
    import torch
    import torch.distributed as dist
    from mbpls_b200 import MBPLS, _cabi, synth
    from mbpls_b200 import engine as E

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    group = None
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
        group = dist.group.WORLD
    n, K, q = args.n, args.components, args.q
    sizes = [int(s * args.scale) for s in SIZES_FULL]
    p = sum(sizes)
    shard = E.ShardMap.build(sizes, rank, world)
    ld = E.round_ld(n)
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    peak_gbs = float(peaks.get("hbm_gbs", 6650.0))
    peak_src = "measured (MEASURED_PEAKS.json hbm_gbs)" if "hbm_gbs" in peaks else "fallback 6.65 TB/s (B200_PROFILING.md)"

    Xbuf = torch.empty((max(shard.p_local, 1), ld), dtype=torch.float64, device=dev)
    Yd = synth.response(n, q, K, dev, args.seed, decay=args.decay)  # n x q, identical on every rank

    def regenerate(nan_frac=None):
        synth.fill_feature_major(Xbuf, n, shard.lo, shard.hi, K, args.seed, noise=args.noise, decay=args.decay,
                                 nan_frac=args.nan_frac if nan_frac is None else nan_frac)

    def local_blocks():
        return [Xbuf[shard.block_off[b]:shard.block_off[b + 1], :n].t() for b in range(len(sizes))]

    def barrier():
        if world > 1:
            dist.barrier(group=group)
        torch.cuda.synchronize(dev)

    one_pass = False if args.two_pass else None

    def make_model(profile=None, materialize=False, sparse=None):
        m = MBPLS(n_components=K, method="NIPALS", standardize=True, calc_all=True,
                  sparse_data=(args.nan_frac > 0) if sparse is None else sparse, copy=False)
        m.set_runtime(device=dev, group=group, materialize=materialize, global_sizes=sizes, profile=profile,
                      max_iter=args.max_iter, one_pass=one_pass)
        return m

    def one_fit(profile=None, nan_frac=None):
        regenerate(nan_frac)
        barrier()
        log("regenerated")
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        with warnings.catch_warnings():
            warnings.simplefilter("ignore")
            m = make_model(profile, sparse=None if nan_frac is None else nan_frac > 0).fit(local_blocks(), Yd)
        e1.record()
        barrier()
        ms = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX, group=group)
        return float(ms.item()), m

    log("setup done; p_local", shard.p_local)
    for _ in range(max(args.warmup, 0)):
        ms, _m = one_fit()
        log("warmup fit ms", ms, "trips", _m.n_iter_)
        del _m  # (a model kept alive across the timed steps changes the allocation pattern inside them: the second timed fit then
        #          goes back to cudaMalloc, which costs 60-90 ms per call once peer mappings exist -- 228 ms instead of 111 at N = 8)
    clocks = Clocks(local) if rank == 0 else None
    profile, times, model = {}, [], None
    launches0 = _cabi.launch_count
    for _ in range(max(args.steps, 1)):
        model = None  # steady state: the previous step's model is released before the next fit allocates
        ms, model = one_fit(profile)
        times.append(ms)
        log("timed fit ms", ms)
    launches = _cabi.launch_count - launches0
    clk = clocks.stop() if clocks else None
    if args.dump_outputs:  # N > 1: rank 0's feature shard of the per-feature attributes
        dump_outputs(model, args.dump_outputs, write=rank == 0)
    # BASELINE config 4 as written: the same fit with 10 % i.i.d. NaN holes (sparse_data=True), reported beside the headline
    variants = {}
    if args.nan_frac == 0 and not args.no_nan_variant:
        one_fit(nan_frac=0.10)
        nan_ms, nan_model = one_fit(nan_frac=0.10)
        nt = list(nan_model.n_iter_)
        variants["nan_10pct"] = {"fit_s": nan_ms / 1e3, "value": fit_bytes(n, p, K, nt) / (nan_ms / 1e3) / 1e9, "unit": "GB/s",
                                 "trips_per_component": nt, "kernels": "one-pass kernels with NaN read as zero + masked denominators from the NaN bit matrix (DESIGN.md 3a)"}
        del nan_model
    trips = list(model.n_iter_)
    exchange = model.__dict__.get("_exchange")
    ms_step = sum(times) / len(times)
    value = fit_bytes(n, p, K, trips) / (ms_step / 1e3) / 1e9

    # X-sized transfers the kernels of one step really make (reads + writes), from the launches timed above
    passes = sum(len(profile.get(k, [])) * m_ for k, m_ in (("trip", 1), ("xtu", 1), ("xw", 1), ("deflate", 2), ("loadings", 1),
                                                             ("standardize", 2))) / max(len(times), 1)
    # per-kernel roofline (rank 0's shard): algorithmic bytes of one launch / mean CUDA-event duration
    def mean_ms(key):
        ev = profile.get(key, [])
        return sum(a.elapsed_time(b) for a, b in ev) / len(ev) if ev else None

    x_bytes_local = 8.0 * n * shard.p_local
    kern = {}
    for key, mult in (("trip", 1.0), ("xtu", 1.0), ("xw", 1.0), ("deflate", 2.0), ("loadings", 1.0), ("standardize", 2.0),
                      ("xchg", 0.0)):  # xchg: split sums + exchange between the GPUs + superlevel step (no X traffic; time incl. peer wait)
        t = mean_ms(key)
        if t:
            kern[key] = {"ms": t, "launches": len(profile[key]), "algorithmic_bytes": mult * x_bytes_local,
                         "gbs": mult * x_bytes_local / (t / 1e3) / 1e9}
    # multi-GPU: every trip ends in an all-reduce, so the slowest rank sets the pace; report the spread of the per-rank means
    rank_skew = None
    if world > 1:
        try:
            keys = ("trip", "deflate", "standardize", "loadings", "xchg")
            mine = torch.tensor([kern[k]["ms"] if k in kern else 0.0 for k in keys], dtype=torch.float64, device=dev)
            allv = [torch.zeros_like(mine) for _ in range(world)]
            dist.all_gather(allv, mine, group=group)
            stack = torch.stack(allv).cpu()
            rank_skew = {k: {"min_ms": float(stack[:, i].min()), "max_ms": float(stack[:, i].max())} for i, k in enumerate(keys)}
        except Exception as exc:  # diagnostics must never take the benchmark line down
            rank_skew = {"error": repr(exc)[:200]}
    # dominant kernel by share of the step: the loadings+deflation(+next first trip) pass when the one-pass kernels run
    # (1 read + 1 write of X per launch), else the X w pass of the two-pass kernels
    dominant = max(kern, key=lambda k: kern[k]["ms"] * kern[k]["launches"]) if kern else None
    names = {"trip": "fused_trip_kernel (X'u and X w in one read)", "deflate": "fused_deflate_kernel / loadings_deflate_*",
             "xw": "xw_kernel", "xtu": "xtu_kernel", "standardize": "standardize_*", "loadings": "xtu_kernel (loadings)"}
    traffic = None
    try:  # dram__bytes_read.sum + dram__bytes_write.sum of one launch from the committed ncu --set full capture
        prof = json.load(open(os.path.join(ROOT, "profiles", "ncu_summary.json")))
        entry = prof.get(dominant, {})
        if dominant and entry.get("algorithmic_bytes_per_launch"):
            # the capture may have been taken on a different shard size: scale by the algorithmic bytes
            traffic = entry["dram_bytes_per_launch"] * kern[dominant]["algorithmic_bytes"] / entry["algorithmic_bytes_per_launch"]
    except Exception:
        pass
    roofline = None
    if dominant:
        roofline = {"bound": "hbm", "kernel": names.get(dominant, dominant) + (" [NaN mode]" if args.nan_frac > 0 else ""),
                    "achieved": kern[dominant]["gbs"], "peak": peak_gbs, "unit": "GB/s",
                    "frac": kern[dominant]["gbs"] / peak_gbs, "traffic": traffic, "peak_source": peak_src,
                    "algorithmic_bytes_per_launch": kern[dominant]["algorithmic_bytes"], "per_kernel": kern}

    # ---- parity gate: the timed configuration's own data (a column slice of it) through the GPU path and the oracle
    parity = None
    if not args.no_parity:
        log("parity gate (dense)")
        parity = {"dense" if args.nan_frac == 0 else "nan": parity_gate(args, dev, group, rank, world, args.nan_frac, args.parity_features)}
        if args.nan_frac == 0 and not args.no_nan_variant:
            log("parity gate (10 % NaN)")
            parity["nan_10pct"] = parity_gate(args, dev, group, rank, world, 0.10, max(16, args.parity_features // 4))
        if rank == 0:
            parity["ok"] = all(v["ok"] for v in parity.values())
            parity["max_rel_err"] = max(v["max_rel_err"] for k, v in parity.items() if isinstance(v, dict))
            parity["trips_equal"] = all(v["trips_equal"] for k, v in parity.items() if isinstance(v, dict))
        log("parity", parity)

    # ---- end to end through the public API with HOST buffers (pinned, row-major like the reference's inputs)
    e2e = None
    del model
    if not args.no_e2e:
        import psutil
        need = 8.0 * n * shard.p_local
        avail = psutil.virtual_memory().available / max(world, 1)
        ok = torch.tensor([1 if need < 0.6 * avail else 0], device=dev)
        if world > 1:
            dist.all_reduce(ok, op=dist.ReduceOp.MIN, group=group)
        if int(ok.item()):
            log("e2e: building pinned host copy")
            regenerate()
            host = []
            for b in range(len(sizes)):
                o0, o1 = shard.block_off[b], shard.block_off[b + 1]
                h = torch.empty((n, o1 - o0), dtype=torch.float64, pin_memory=(o1 > o0))
                for c in range(0, o1 - o0, 8192):
                    c1 = min(o1 - o0, c + 8192)
                    h[:, c:c1].copy_(Xbuf[o0 + c:o0 + c1, :n].t())
                host.append(h)
            Yh = Yd.cpu().pin_memory()
            torch.cuda.synchronize(dev)
            del Xbuf
            torch.cuda.empty_cache()
            e_times, d2h = [], 0
            n_e2e = 1 + max(1, args.e2e_steps)   # one untimed warm-up repetition (pinned result buffers are cached after it)
            for it in range(n_e2e + (1 if VERBOSE else 0)):  # --verbose: one more, untimed, with per-phase wall clocks
                barrier()
                t0 = time.perf_counter()
                with warnings.catch_warnings():
                    warnings.simplefilter("ignore")
                    m = MBPLS(n_components=K, method="NIPALS", sparse_data=args.nan_frac > 0, copy=True)
                    phases = {} if it >= n_e2e else None
                    m.set_runtime(device=dev, group=group, materialize=True, global_sizes=sizes, max_iter=args.max_iter, timings=phases)
                    m.fit(host, Yh)
                    if phases is not None:
                        log("e2e phases (s)", {k: round(v, 4) for k, v in phases.items()})
                barrier()
                dt = torch.tensor([time.perf_counter() - t0], dtype=torch.float64, device=dev)
                if world > 1:
                    dist.all_reduce(dt, op=dist.ReduceOp.MAX, group=group)
                log("e2e fit s", float(dt.item()))
                if 0 < it < n_e2e:
                    e_times.append(float(dt.item()))
                d2h = sum(a.nbytes for a in [m.Ts_, m.U_, m.V_, m.R_, m.beta_, m.A_] + m.T_ + m.W_ + m.P_ + m.W_non_normal_)
                e_trips = list(m.n_iter_)
                del m
                torch.cuda.empty_cache()
            es = sum(e_times) / len(e_times)
            e2e = {"value": fit_bytes(n, p, K, e_trips) / es / 1e9, "unit": "GB/s", "fit_s": es,
                   "h2d_bytes_per_step": int(8 * n * shard.p_local + 8 * n * q), "d2h_bytes_per_step": int(d2h),
                   "what": "MBPLS.fit(list of pinned row-major host blocks, Y) -> numpy attributes; wall clock, max over ranks"}
        else:
            e2e = {"value": None, "unit": "GB/s", "skipped": "host RAM too small for the full-size input"}

    configs = None
    if not args.no_configs:
        try:
            del Xbuf
        except NameError:
            pass
        torch.cuda.empty_cache()
        log("other BASELINE configurations")
        try:
            configs = run_configs(args, dev, group, rank, world, peak_gbs)
        except Exception as exc:  # secondary measurements must not take the headline line down
            configs = {"error": repr(exc)[:300]}
        log("configs", configs)

    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu:
        p_cpu = cpu_p_for_budget(args, 30.0)
        log("cpu baseline sample p", p_cpu)
        r = cpu_sample(args, p_cpu)
        log("cpu baseline done", r["seconds"])
        cpu = {"value": r["gbs"], "unit": "GB/s", "cores": r["cores"], "kind": r["kind"], "sample": r["sample"],
               "seconds": r["seconds"], "trips_per_component": r["trips"]}
        if "nan_10pct" in variants:
            nn, pp = min(CPU_NAN_SHAPE[0], args.n), min(CPU_NAN_SHAPE[1], p_cpu)
            rn = cpu_sample(args, pp, n=nn, nan_frac=0.10)
            variants["nan_10pct"]["cpu_baseline"] = {"value": rn["gbs"], "unit": "GB/s", "cores": rn["cores"], "kind": rn["kind"],
                                                     "sample": rn["sample"], "seconds": rn["seconds"]}

    if rank == 0:
        line = {
            "metric": METRIC, "value": value, "unit": "GB/s", "n_gpus": world, "steps": len(times), "warmup": args.warmup,
            "ms_per_step": ms_step, "fit_s": ms_step / 1e3, "higher_is_better": True, "scaling": "strong",
            "vs_baseline": None, "dtype": "f64", "data": "synthetic (device-generated latent-structure blocks)",
            "config": workload_config(args), "trips_per_component": trips, "algorithmic_bytes_per_step": fit_bytes(n, p, K, trips),
            "frac_of_hbm_peak": value / (peak_gbs * world),
            "frac_of_hbm_peak_actual_traffic": passes * 8.0 * n * p / (ms_step / 1e3) / 1e9 / (peak_gbs * world), "roofline": roofline, "cpu_baseline": cpu, "e2e": e2e,
            "exchange": exchange, "parity": parity, "configs": configs, "gpu_launches": launches, "clocks": clk, "step_ms": times, "variants": variants, "rank_skew": rank_skew,
            "passes_over_X_per_step": passes, "hbm_gbs_actual_traffic": passes * 8.0 * n * p / (ms_step / 1e3) / 1e9,
        }
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def main():
    global VERBOSE
    args = parse()
    VERBOSE = args.verbose
    # torchrun exports OMP_NUM_THREADS=1; the CPU legs (reference arm, cpu_baseline, the parity gate's oracle) run on rank 0 and
    # should see the host's cores (numpy / torch are imported after this point; threadpoolctl raises the limit again at use)
    if int(os.environ.get("RANK", "0")) == 0:
        for var in ("OMP_NUM_THREADS", "OPENBLAS_NUM_THREADS", "MKL_NUM_THREADS"):
            os.environ[var] = str(os.cpu_count() or 1)
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
