"""Permutation test and bootstrap with missing values (sparse_data=True) on the notebook shape (100 x (200 + 250), y 100 x 1,
10 % i.i.d. NaN in X, 10-fold, k = 1..15): the batched path (every fit of every permutation in one slot-mode launch of
smallfit_kernel's NaN mode) against the per-fit path (one MBPLS.fit on the streaming kernels per permutation and fold).  The
per-fit path runs a few permutations and is extrapolated linearly to 1,000 (key per_fit_path_extrapolated_s); everything else
is measured.  Prints one JSON line."""
import json, os, subprocess, sys, time, warnings
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np, torch
from sklearn.model_selection import KFold
from mbpls_b200 import MBPLS
from mbpls_b200.model_selection import bootstrap, permutation_test_score
from oracle.cases import latent_blocks

warnings.simplefilter("ignore")
X, Y = latent_blocks(100, (200, 250), 1, 15, seed=7)
rng = np.random.default_rng(11)
for x in X:
    x[rng.random(x.shape) < 0.10] = np.nan
nan_share = float(np.mean(np.isnan(np.hstack(X))))
ks = list(range(1, 16))
cv = KFold(10)
NPERM, NPERM_FIT, NRES = 1000, 3, 1000


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


est = lambda small, K=1: MBPLS(n_components=K, sparse_data=True).set_runtime(small_path=small)
pts = lambda small, nperm: permutation_test_score(est(small), X, Y, cv=cv, n_permutations=nperm, n_components_list=ks)
t_batch, res = best_of(lambda: pts(True, NPERM))
t_fit, res_fit = once(lambda: pts(False, NPERM_FIT))  # every refit through MBPLS.fit on the streaming kernels
diff = max(float(np.max(np.abs(res[k][1][:NPERM_FIT] - res_fit[k][1]))) for k in ks)
diff_score = max(abs(res[k][0] - res_fit[k][0]) for k in ks)

t_boot, boot = best_of(lambda: bootstrap(est(True, 15), X, Y, n_resamples=NRES))

try:
    power = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
except (OSError, subprocess.SubprocessError):
    power = "unknown"
nf = cv.get_n_splits()
print(json.dumps(dict(
    case="sparse_data=True permutation test 100 x (200+250), 10 % NaN in X, 10-fold, k = 1..15; bootstrap K = 15",
    gpu=torch.cuda.get_device_name(0), power_limit=power, nan_share_x=nan_share,
    n_permutations=NPERM, fits=(NPERM + 1) * nf,
    batched_permutation_test_s=t_batch,
    per_fit_path_perms=NPERM_FIT, per_fit_path_s=t_fit,
    per_fit_path_extrapolated_s=t_fit * (NPERM + 1) / (NPERM_FIT + 1),
    max_abs_diff_batched_vs_per_fit_scores=max(diff, diff_score),
    score_k15=res[15][0], pvalue_k15=res[15][2],
    bootstrap_resamples=NRES, batched_bootstrap_s=t_boot,
    bootstrap_A_block0_k1_p2_5_p97_5=[float(v) for v in np.percentile(boot["A_"][:, 0, 0], [2.5, 97.5])])), flush=True)
