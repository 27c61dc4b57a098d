"""Permutation test and bootstrap on the notebook shape (100 x (200 + 250), y 100 x 1, 10-fold, k = 1..15): the batched path
(every fit of every permutation in one slot-mode launch of smallfit_kernel) against the per-fit path (one MBPLS.fit per
permutation and fold) and the numpy oracle's refit loop.  The per-fit path and the oracle run a few permutations and are
extrapolated linearly to 1,000 (keys *_extrapolated_s); everything else is measured.  Prints one JSON line."""
import json, os, subprocess, sys, time, warnings
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np, torch
from sklearn.model_selection import KFold
from mbpls_b200 import MBPLS
from mbpls_b200.model_selection import _permutations, bootstrap, permutation_test_score
from oracle import OracleMBPLS
from oracle.cases import latent_blocks

warnings.simplefilter("ignore")
X, Y = latent_blocks(100, (200, 250), 1, 15, seed=7)
y = Y.ravel()
ks = list(range(1, 16))
cv = KFold(10)
NPERM, NPERM_FIT, NPERM_ORACLE, NRES = 1000, 20, 2, 1000


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


pts = lambda small, nperm: permutation_test_score(MBPLS().set_runtime(small_path=small), X, y, cv=cv, n_permutations=nperm,
                                                  n_components_list=ks)
t_batch, res = best_of(lambda: pts(True, NPERM))
t_fit, res_fit = once(lambda: pts(False, NPERM_FIT))  # every refit through MBPLS.fit (one-kernel path chosen by size)
diff = max(float(np.max(np.abs(res[k][1][:NPERM_FIT] - res_fit[k][1]))) for k in ks)

folds = list(cv.split(np.arange(100)))
t0 = time.perf_counter()
for pi in _permutations(100, NPERM_ORACLE, 0)[1:]:
    for tr, te in folds:
        OracleMBPLS(n_components=15).fit([x[tr] for x in X], y[pi[tr]]).predict([x[te] for x in X])
t_oracle = time.perf_counter() - t0

t_boot, boot = best_of(lambda: bootstrap(MBPLS(n_components=15).set_runtime(small_path=True), X, y, n_resamples=NRES))

try:
    power = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
except (OSError, subprocess.SubprocessError):
    power = "unknown"
nf = len(folds)
print(json.dumps(dict(
    case="permutation test 100 x (200+250), 10-fold, k = 1..15; bootstrap K = 15",
    gpu=torch.cuda.get_device_name(0), power_limit=power,
    n_permutations=NPERM, fits=(NPERM + 1) * nf,
    batched_permutation_test_s=t_batch,
    per_fit_path_perms=NPERM_FIT, per_fit_path_s=t_fit,
    per_fit_path_extrapolated_s=t_fit * (NPERM + 1) / (NPERM_FIT + 1),
    oracle_numpy_perms=NPERM_ORACLE, oracle_numpy_k15_s=t_oracle,
    oracle_numpy_k15_extrapolated_s=t_oracle * (NPERM + 1) / NPERM_ORACLE,
    max_abs_diff_batched_vs_per_fit_scores=diff,
    score_k15=res[15][0], pvalue_k15=res[15][2],
    bootstrap_resamples=NRES, batched_bootstrap_s=t_boot,
    bootstrap_A_block0_k1_p2_5_p97_5=[float(v) for v in np.percentile(boot["A_"][:, 0, 0], [2.5, 97.5])])), flush=True)
