"""GPU: permutation tests and bootstrap of multiblock fits (mbpls_b200/model_selection.py) -- the batched path (every fit of
every permutation / resample in one slot-mode launch of smallfit_kernel) and the generic refit path against scikit-learn's
permutation_test_score and explicit loops over the numpy oracle; slot mode bitwise equal to one CTA per fit.  (conftest.py
switches the automatic small path off, so the batched cases ask for it with small_path=True.)"""
import warnings

import numpy as np
import pytest
from sklearn import metrics

from helpers import assert_trips, rel_err

pytestmark = pytest.mark.gpu

METRIC = {None: metrics.r2_score, "neg_mean_squared_error": lambda a, b: -metrics.mean_squared_error(a, b)}


def _launches():
    from mbpls_b200 import _cabi
    return _cabi.launch_count


def _oracle_permutation_scores(kw, X, Y, folds, perms, scoring=None):
    """mean over folds of the score of OracleMBPLS fitted on X[tr], Y[pi[tr]] and scored on X[te] against Y[pi[te]]"""
    from oracle import OracleMBPLS
    out = []
    for pi in perms:
        s = []
        for tr, te in folds:
            with warnings.catch_warnings():
                warnings.simplefilter("ignore")
                m = OracleMBPLS(**kw).fit([x[tr] for x in X], Y[pi[tr]])
                s.append(METRIC[scoring](Y[pi[te]], np.asarray(m.predict([x[te] for x in X])).reshape(Y[pi[te]].shape)))
        out.append(np.mean(s))
    return np.array(out)


@pytest.mark.parametrize("scoring", [None, "neg_mean_squared_error"])
def test_single_array_matches_sklearn_permutation_test_score(scoring):
    from sklearn.model_selection import permutation_test_score as sk_pts
    from mbpls_b200 import MBPLS
    from mbpls_b200.model_selection import permutation_test_score
    from oracle.cases import latent_blocks
    X, Y = latent_blocks(40, (25,), 1, 3, seed=61)
    x, y = X[0], Y.ravel()
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        score, perm, pv = permutation_test_score(MBPLS(n_components=3).set_runtime(small_path=True), x, y, cv=5,
                                                 n_permutations=30, random_state=7, scoring=scoring)
        s2, perm2, pv2 = sk_pts(MBPLS(n_components=3), x, y, cv=5, n_permutations=30, random_state=7, scoring=scoring)
    assert abs(score - s2) <= 1e-9 * abs(s2)
    assert perm.shape == (30,) and np.all(np.abs(perm - perm2) <= 1e-9 * np.abs(perm2))
    assert pv == pv2


def test_block_list_component_path_matches_oracle_loop():
    from sklearn.model_selection import KFold
    from mbpls_b200 import MBPLS
    from mbpls_b200.model_selection import _permutations, permutation_test_score
    from oracle.cases import latent_blocks
    X, Y = latent_blocks(36, (14, 9, 11), 2, 3, seed=62)
    cv = KFold(4)
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        got = permutation_test_score(MBPLS(n_components=1).set_runtime(small_path=True), X, Y, cv=cv, n_permutations=15,
                                     random_state=3, n_components_list=[1, 2, 3])
    folds = list(cv.split(np.arange(36)))
    perms = _permutations(36, 15, 3)
    for k in (1, 2, 3):
        want = _oracle_permutation_scores(dict(n_components=k), X, Y, folds, perms)
        score, perm, pv = got[k]
        assert rel_err(score, want[0]) < 1e-9 and rel_err(perm, want[1:]) < 1e-9, k
        assert pv == (np.sum(want[1:] >= want[0]) + 1.0) / 16.0


def test_more_fits_than_two_slots_per_sm_take_one_launch():
    import torch
    from mbpls_b200 import MBPLS
    from mbpls_b200.model_selection import permutation_test_score
    from oracle.cases import latent_blocks
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    nperm = 2 * sms // 5 + 1                    # (1 + nperm) * 5 folds > 2 x SM count
    X, Y = latent_blocks(30, (12, 10), 1, 2, seed=63)
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        c0 = _launches()
        _, perm, _ = permutation_test_score(MBPLS(n_components=2).set_runtime(small_path=True), X, Y, cv=5,
                                            n_permutations=nperm)
        assert _launches() - c0 == 1
    assert perm.shape == (nperm,) and np.all(np.isfinite(perm))


def test_slot_mode_is_bitwise_equal_to_one_cta_per_fit():
    import torch
    from mbpls_b200 import _cabi, engine as E
    from mbpls_b200 import smallfit as SF
    from mbpls_b200.model_selection import _permutations
    from oracle.cases import latent_blocks
    X, Y = latent_blocks(33, (10, 7), 2, 4, seed=64)
    dev = torch.device("cuda", 0)
    D, n, sizes, p, q, ldx = SF.pack_source(X, Y, dev)
    perms = _permutations(n, 6, 1)
    folds = [(np.setdiff1d(np.arange(n), te), te) for te in np.array_split(np.arange(n), 4)]
    tr = [f[0].astype(np.int32) for _ in perms for f in folds]
    te = [f[1].astype(np.int32) for _ in perms for f in folds]
    ys = [pi[f[0]].astype(np.int32) for pi in perms for f in folds]
    boff = E.ShardMap.build(sizes, 0, 1).block_off
    res = []
    for nslots in (3, 0):
        lay, out, fp, keep = SF.launch(D, n, p, q, ldx, boff, 4, True, 0, 1e-14, 10**6, tr, te, y_sets=ys, nslots=nslots,
                                       fit_preds=True)
        res.append((lay.section(out, "small").clone(), lay.section(out, "beta").clone(), fp.clone()))
    torch.cuda.synchronize()
    for a, b in zip(*res):  # bit patterns (the prediction rows past a fold's test size hold NaN)
        assert torch.equal(a.view(torch.int64), b.view(torch.int64))
    assert torch.isfinite(res[0][2]).any()
    with pytest.raises(_cabi.MbplsCudaError):  # sample-indexed predictions overlap between permutations: not in slot mode
        SF.launch(D, n, p, q, ldx, boff, 4, True, 0, 1e-14, 10**6, tr, te, y_sets=ys, nslots=3)


def test_batched_and_generic_paths_agree_for_nipals():
    from mbpls_b200 import MBPLS
    from mbpls_b200.model_selection import permutation_test_score
    from oracle.cases import latent_blocks
    X, Y = latent_blocks(30, (16, 8), 1, 2, seed=65)
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        a = permutation_test_score(MBPLS(n_components=2).set_runtime(small_path=True), X, Y, cv=3, n_permutations=8,
                                   n_components_list=[1, 2])
        b = permutation_test_score(MBPLS(n_components=2).set_runtime(small_path=False), X, Y, cv=3, n_permutations=8,
                                   n_components_list=[1, 2])
    for k in (1, 2):
        assert rel_err(a[k][0], b[k][0]) < 1e-9 and rel_err(a[k][1], b[k][1]) < 1e-9 and a[k][2] == b[k][2], k


@pytest.mark.parametrize("method", ["KERNEL", "UNIPALS", "SIMPLS"])
def test_generic_path_matches_oracle_loop(method):
    from mbpls_b200 import MBPLS
    from mbpls_b200.model_selection import _folds, _permutations, permutation_test_score
    from oracle.cases import latent_blocks
    X, Y = latent_blocks(24, (10, 6), 1, 2, seed=66)
    kw = dict(n_components=2, method=method, full_svd=True)
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        score, perm, pv = permutation_test_score(MBPLS(**kw), X, Y, cv=4, n_permutations=5, random_state=2)
    want = _oracle_permutation_scores(kw, X, Y, _folds(24, 4), _permutations(24, 5, 2))
    assert rel_err(score, want[0]) < 1e-9 and rel_err(perm, want[1:]) < 1e-9
    assert pv == (np.sum(want[1:] >= want[0]) + 1.0) / 6.0


def test_bootstrap_matches_oracle_on_resampled_rows():
    from mbpls_b200 import MBPLS
    from mbpls_b200.model_selection import bootstrap
    from oracle import OracleMBPLS
    from oracle.cases import latent_blocks
    X, Y = latent_blocks(40, (18, 13), 2, 3, seed=67)
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        c0 = _launches()
        got = bootstrap(MBPLS(n_components=3).set_runtime(small_path=True), X, Y, n_resamples=12, random_state=5)
        assert _launches() - c0 == 1
    assert got["indices"].shape == (12, 40) and got["A_"].shape == (12, 2, 3) and got["beta_"].shape == (12, 31, 2)
    assert got["n_iter_"].shape == (12, 3) and got["explained_var_xblocks_"].shape == (12, 2, 3)
    for r, idx in enumerate(got["indices"]):
        with warnings.catch_warnings():
            warnings.simplefilter("ignore")
            o = OracleMBPLS(n_components=3).fit([x[idx] for x in X], Y[idx])
        for name in ("A_", "beta_", "A_corrected_", "explained_var_x_", "explained_var_y_", "explained_var_xblocks_"):
            assert rel_err(got[name][r], np.asarray(getattr(o, name))) < 1e-9, (r, name)
        assert_trips(list(got["n_iter_"][r]), list(o.n_iter_), o.diff_trace_, 1e-14, f"resample {r}")


def test_rank_deficient_bootstrap_refits_singular_resamples_through_fit():
    """K above the rank: every resample is flagged singular in the batched launch and refit through MBPLS.fit (the reference's
    pseudo-inverse).  The components beyond the rank are fitted to rounding noise, so there the streaming kernels and the
    one-kernel path legitimately differ; the components the data determines agree with the generic path."""
    from mbpls_b200 import MBPLS
    from mbpls_b200.model_selection import bootstrap
    rng = np.random.default_rng(8)
    Z = rng.standard_normal((10, 2))
    X = [Z @ rng.standard_normal((2, 5)), Z @ rng.standard_normal((2, 4))]   # rank 2: four components are more than the rank
    y = Z @ np.array([1.0, -0.5])
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        a = bootstrap(MBPLS(n_components=4).set_runtime(small_path=True), X, y, n_resamples=6, random_state=1)
        b = bootstrap(MBPLS(n_components=4).set_runtime(small_path=False), X, y, n_resamples=6, random_state=1)
    assert np.array_equal(a["indices"], b["indices"])
    assert np.all(np.isfinite(a["beta_"])) and np.all(np.isfinite(b["beta_"]))
    for r, idx in enumerate(a["indices"]):
        with warnings.catch_warnings():
            warnings.simplefilter("ignore")
            m = MBPLS(n_components=4).set_runtime(small_path=True).fit([x[idx] for x in X], y[idx])
        assert np.array_equal(a["beta_"][r], m.beta_) and np.array_equal(a["A_"][r], m.A_), r
    for name in ("A_", "A_corrected_", "explained_var_xblocks_"):
        assert rel_err(a[name][:, :, :2], b[name][:, :, :2]) < 1e-9, name
    assert rel_err(a["explained_var_y_"][:, :2], b["explained_var_y_"][:, :2]) < 1e-9
