"""Block permutation test on the notebook shape (100 x (200 + 250), y 100 x 1, 10-fold, k = 1..15, 1,000 permutations per
block), dense and with 10 % i.i.d. NaN in X (sparse_data=True): the batched path (every fit in one slot-mode launch of
smallfit_kernel, 22,011 fits) against the per-fit path (one MBPLS.fit on the streaming kernels per fold, permutation and block,
and per fit on all rows).  The per-fit path runs a few permutations and is extrapolated linearly to 1,000 (keys
*_per_fit_path_extrapolated_s); everything else is measured.  Prints one JSON line."""
import json, os, subprocess, sys, time, warnings
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np, torch
from sklearn.model_selection import KFold
from mbpls_b200 import MBPLS
from mbpls_b200.model_selection import block_permutation_test
from oracle.cases import latent_blocks

warnings.simplefilter("ignore")
X, Y = latent_blocks(100, (200, 250), 1, 15, seed=7)
rng = np.random.default_rng(11)
Xnan = [x.copy() for x in X]
for x in Xnan:
    x[rng.random(x.shape) < 0.10] = np.nan
ks = list(range(1, 16))
cv = KFold(10)
NPERM, NPERM_FIT = 1000, 2
B, nf = len(X), cv.get_n_splits()


def best_of(fn, reps=3):
    fn(); torch.cuda.synchronize()                     # warm-up
    best, out = None, None
    for _ in range(reps):
        t0 = time.perf_counter(); out = fn(); torch.cuda.synchronize(); dt = time.perf_counter() - t0
        best = dt if best is None else min(best, dt)
    return best, out


def once(fn):
    t0 = time.perf_counter(); out = fn(); torch.cuda.synchronize()
    return time.perf_counter() - t0, out


def run(Xs, sparse, small, nperm):
    est = MBPLS(n_components=1, sparse_data=sparse).set_runtime(small_path=small)
    return block_permutation_test(est, Xs, Y, cv=cv, n_permutations=nperm, n_components_list=ks)


def max_diff(a, b):
    """largest absolute difference of the scores and A_ of the first NPERM_FIT permutations of two results"""
    d = [abs(a["score"][k] - b["score"][k]) for k in ks]
    d += [float(np.max(np.abs(a["permutation_scores"][k][:, :NPERM_FIT] - b["permutation_scores"][k]))) for k in ks]
    d += [float(np.max(np.abs(a["A_"] - b["A_"]))), float(np.max(np.abs(a["A_permuted"][:, :NPERM_FIT] - b["A_permuted"])))]
    return max(d)


line = dict(case="block permutation test 100 x (200+250), 10-fold, k = 1..15, 1,000 permutations per block; dense and "
                 "sparse_data=True with 10 % NaN in X", n_permutations=NPERM,
            fits=(1 + B * NPERM) * (nf + 1), per_fit_path_perms=NPERM_FIT)
for tag, Xs, sparse in (("dense", X, False), ("nan", Xnan, True)):
    t_batch, res = best_of(lambda: run(Xs, sparse, True, NPERM))
    t_fit, res_fit = once(lambda: run(Xs, sparse, False, NPERM_FIT))  # every fit through MBPLS.fit
    line.update({f"{tag}_batched_s": t_batch, f"{tag}_per_fit_path_s": t_fit,
                 f"{tag}_per_fit_path_extrapolated_s": t_fit * (1 + B * NPERM) / (1 + B * NPERM_FIT),
                 f"{tag}_max_abs_diff_batched_vs_per_fit": max_diff(res, res_fit),
                 f"{tag}_score_k15": res["score"][15], f"{tag}_pvalue_k15": [float(v) for v in res["pvalue"][15]],
                 f"{tag}_A_pvalue_k1": [float(v) for v in res["A_pvalue"][:, 0]]})

try:
    power = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
except (OSError, subprocess.SubprocessError):
    power = "unknown"
line.update(gpu=torch.cuda.get_device_name(0), power_limit=power)
print(json.dumps(line), flush=True)
