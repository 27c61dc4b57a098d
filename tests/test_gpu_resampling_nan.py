"""GPU: cross-validation, permutation tests and bootstrap of missing-data NIPALS fits (sparse_data=True) in one launch of
smallfit_kernel's NaN mode, against the per-fit path (MBPLS.fit on the streaming kernels, small_path=False) and against the
numpy oracle refitted fold by fold.  (conftest.py switches the automatic small path off, so the batched cases ask for it with
small_path=True.)"""
import warnings

import numpy as np
import pytest
from sklearn import metrics

from helpers import assert_trips, rel_err

pytestmark = pytest.mark.gpu
SIZES = (14, 9, 11)


def _launches():
    from mbpls_b200 import _cabi
    return _cabi.launch_count


# --------------------------------------------------------------------------------------------- #
# missing-data generators
# --------------------------------------------------------------------------------------------- #
def iid_holes(X, Y, frac, seed, y_cols=(), y_frac=0.3, y_rows=None):
    """i.i.d. holes in every feature but the first of each block (so no sample loses a whole block: the reference divides 0/0
    there).  Y columns y_cols miss about y_frac of the rows that have a hole in the LAST X block (restricted to y_rows): the
    reference's Y-score step divides exactly those rows by the masked v'v (mbpls.py:903), a Y hole anywhere else turns its
    fit NaN."""
    rng = np.random.default_rng(seed)
    Xh = [x.copy() for x in X]
    for x in Xh:
        hole = rng.random(x.shape) < frac
        hole[:, 0] = False
        x[hole] = np.nan
    Yh = Y.copy()
    sparse = np.flatnonzero(np.isnan(Xh[-1]).any(axis=1))
    if y_rows is not None:
        sparse = np.intersect1d(sparse, y_rows)
    for c in y_cols:
        Yh[sparse[rng.random(len(sparse)) < y_frac], c] = np.nan
    return Xh, Yh


def structured_holes(X, Y, seed, *, heavy=0, blockwise=(2, 0.25, 1)):
    """The structured holes of test_gpu_long_and_missing.py at n ~ 40: features 2..3 of block `heavy` miss 55 % and 80 % of
    the samples; for a share of the samples every feature of block b except the first `keep` is missing."""
    rng = np.random.default_rng(seed)
    n = Y.shape[0]
    Xh = [x.copy() for x in X]
    for j, share in zip((2, 3), (0.55, 0.80)):
        Xh[heavy][rng.choice(n, round(share * n), replace=False), j] = np.nan
    b, frac, keep = blockwise
    rows = rng.choice(n, int(frac * n), replace=False)
    Xh[b][np.ix_(rows, np.arange(keep, Xh[b].shape[1]))] = np.nan
    return Xh, Y.copy()


def _data(n, q, seed, K=4):
    from oracle.cases import latent_blocks
    X, Y = latent_blocks(n, SIZES, q, K, seed=seed)
    return X, Y.reshape(n, q)


# --------------------------------------------------------------------------------------------- #
# references
# --------------------------------------------------------------------------------------------- #
def _oracle_cv(kw, X, Y, folds, ks):
    from oracle import OracleMBPLS
    out = {k: np.full(Y.shape, np.nan) for k in ks}
    for tr, te in folds:
        for k in ks:
            with warnings.catch_warnings():
                warnings.simplefilter("ignore")
                m = OracleMBPLS(**dict(kw, n_components=k)).fit([x[tr] for x in X], Y[tr])
                out[k][te] = np.asarray(m.predict([x[te] for x in X])).reshape(len(te), -1)
    return out


def _cv(small_path, X, Y, cv, ks, **kw):
    from mbpls_b200 import MBPLS
    from mbpls_b200.model_selection import cross_val_predict
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        c0 = _launches()
        got = cross_val_predict(MBPLS(n_components=max(ks), sparse_data=True, **kw).set_runtime(small_path=small_path),
                                [x.copy() for x in X], Y.copy(), cv=cv, n_components_list=ks)
        return got, _launches() - c0


def _folds(n, cv):
    from mbpls_b200.model_selection import _folds
    return _folds(n, cv)


# --------------------------------------------------------------------------------------------- #
# cross-validation
# --------------------------------------------------------------------------------------------- #
@pytest.mark.parametrize("q", [1, 3])
@pytest.mark.parametrize("cv", [5, "loo"])
@pytest.mark.parametrize("holes", ["iid", "structured"])
def test_cross_val_predict_nan_in_x_one_launch(q, cv, holes):
    n = 36
    X, Y = _data(n, q, seed=71 + q)
    X, Y = iid_holes(X, Y, 0.1, seed=5) if holes == "iid" else structured_holes(X, Y, seed=6)
    cv = n if cv == "loo" else cv
    ks = [1, 2, 3, 4, 5]
    got, launches = _cv(True, X, Y, cv, ks)
    assert launches == 1
    want, _ = _cv(False, X, Y, cv, ks)
    oracle = _oracle_cv(dict(sparse_data=True), X, Y, _folds(n, cv), ks)
    for k in ks:
        assert np.all(np.isfinite(got[k])), k
        assert rel_err(got[k], want[k]) <= 1e-9, (k, rel_err(got[k], want[k]))
        assert rel_err(got[k], oracle[k]) <= 1e-8, (k, rel_err(got[k], oracle[k]))


def test_cross_val_predict_nan_in_y_start_column_per_fold():
    """Y column 0 has holes only among the test rows of fold 0, column 2 in every fold, column 1 nowhere: fold 0 starts its Y
    scores from column 0, every other fold from column 1 (mbpls.py:832-836)."""
    n, q = 40, 3
    X, Y = _data(n, q, seed=81)
    folds = _folds(n, 5)
    X, Y = iid_holes(X, Y, 0.12, seed=8, y_cols=(0,), y_frac=0.6, y_rows=folds[0][1])
    X, Y = X, iid_holes(X, Y, 0.0, seed=9, y_cols=(2,), y_frac=0.4)[1]
    assert np.isnan(Y[folds[0][1], 0]).any() and not np.isnan(Y[folds[0][0], 0]).any()
    assert not np.isnan(Y[:, 1]).any() and all(np.isnan(Y[tr, 2]).any() for tr, _ in folds)
    ks = [1, 2, 3, 4]
    got, launches = _cv(True, X, Y, 5, ks)
    assert launches == 1
    want, _ = _cv(False, X, Y, 5, ks)
    oracle = _oracle_cv(dict(sparse_data=True), X, Y, folds, ks)
    for k in ks:
        assert np.all(np.isfinite(got[k])), k
        assert rel_err(got[k], want[k]) <= 1e-9, k
        assert rel_err(got[k], oracle[k]) <= 1e-8, k


def test_non_orthogonal_scores_prefix_models_match_oracle():
    """About 30 % holes: the superscores are far from orthogonal, so P'W is far from upper triangular and every prefix model
    needs its own inverse (the dense path's triangular substitution would be wrong here)."""
    from oracle import OracleMBPLS
    n, q, K = 40, 2, 5
    X, Y = _data(n, q, seed=91, K=6)
    X, Y = iid_holes(X, Y, 0.3, seed=10)
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        o = OracleMBPLS(n_components=K, sparse_data=True).fit(X, Y)
    Wn = np.concatenate(o.W_non_normal_, axis=0)
    G = np.concatenate(o.P_, axis=0).T @ (Wn / np.linalg.norm(Wn, axis=0))
    assert np.max(np.abs(np.tril(G, -1))) > 1e-2 * np.max(np.abs(np.diag(G)))
    ks = [1, 2, 3, 4, 5]
    got, launches = _cv(True, X, Y, 5, ks)
    assert launches == 1
    oracle = _oracle_cv(dict(sparse_data=True), X, Y, _folds(n, 5), ks)
    want, _ = _cv(False, X, Y, 5, ks)
    for k in ks:
        assert rel_err(got[k], oracle[k]) <= 1e-8, (k, rel_err(got[k], oracle[k]))
        assert rel_err(got[k], want[k]) <= 1e-9, k


def test_rank_deficient_folds_are_refit_through_fit():
    """More components than the data has rank: the batch flags P'W as singular and every fold is refit through MBPLS.fit,
    which applies the pseudo-inverse like the reference, so the result is the per-fit path's.  (Holes break an exact rank
    deficiency -- the masked regressions leave a residual -- so the data here has none; sparse_data=True still runs the NaN
    mode.)"""
    rng = np.random.default_rng(12)
    Z = rng.standard_normal((20, 2))
    X = [Z @ rng.standard_normal((2, 6)), Z @ rng.standard_normal((2, 5))]
    Y = (Z @ np.array([1.0, -0.5])).reshape(-1, 1)
    ks = [1, 2, 3, 4]
    got, launches = _cv(True, X, Y, 4, ks)
    assert launches > 1
    want, _ = _cv(False, X, Y, 4, ks)
    for k in ks:
        assert np.array_equal(got[k], want[k], equal_nan=True), k


# --------------------------------------------------------------------------------------------- #
# routing to the per-fit path
# --------------------------------------------------------------------------------------------- #
def _seeded(fn):
    """fn() with the global numpy random state reset: MBPLS.fit draws its start vector from it when no Y column is whole."""
    np.random.seed(1234)
    try:
        return fn()
    except ValueError as e:
        return e


def _same(a, b):
    if isinstance(a, Exception) or isinstance(b, Exception):
        return type(a) is type(b) and str(a) == str(b)
    if isinstance(a, dict):
        return a.keys() == b.keys() and all(_same(a[k], b[k]) for k in a)
    if isinstance(a, tuple):
        return len(a) == len(b) and all(_same(x, y) for x, y in zip(a, b))
    return np.array_equal(np.asarray(a, float), np.asarray(b, float), equal_nan=True)


def test_fold_with_an_unobserved_feature_goes_to_the_fold_loop():
    from mbpls_b200 import smallfit as SF
    n = 30
    X, Y = _data(n, 2, seed=101)
    X, Y = iid_holes(X, Y, 0.08, seed=13)
    folds = _folds(n, 5)
    X[1][folds[0][0], 4] = np.nan          # block 1 feature 4 is seen only among fold 0's test rows
    x_obs = np.hstack([~np.isnan(x) for x in X])
    ok = SF.nan_fits_eligible(x_obs, ~np.isnan(Y), [tr for tr, _ in folds], [tr for tr, _ in folds])
    assert ok.tolist() == [False, True, True, True, True]
    ks = [1, 2, 3]
    got = _seeded(lambda: _cv(True, X, Y, 5, ks))
    want = _seeded(lambda: _cv(False, X, Y, 5, ks))
    if isinstance(want, Exception):  # whatever MBPLS.fit does with the unobserved feature, the batch does the same
        assert _same(got, want)
    else:
        assert got[1] > 1 and _same(got[0], want[0])


def test_no_fully_observed_y_column_goes_to_the_per_fit_path():
    """Both Y columns have holes in every fold's training rows: the reference starts from np.random.rand, so these fits go to
    MBPLS.fit; with the global random state reset the two paths draw the same start vectors."""
    from mbpls_b200 import MBPLS
    from mbpls_b200.model_selection import permutation_test_score
    n = 32
    X, Y = _data(n, 2, seed=111)
    X, Y = iid_holes(X, Y, 0.15, seed=14, y_cols=(0, 1), y_frac=0.5)
    folds = _folds(n, 4)
    assert all(np.isnan(Y[tr]).any(axis=0).all() for tr, _ in folds)
    got = _seeded(lambda: _cv(True, X, Y, 4, [1, 2]))
    want = _seeded(lambda: _cv(False, X, Y, 4, [1, 2]))
    assert not isinstance(got, Exception) and got[1] > 1
    assert _same(got[0], want[0])

    def pts(small_path):
        with warnings.catch_warnings():
            warnings.simplefilter("ignore")
            return permutation_test_score(MBPLS(n_components=2, sparse_data=True).set_runtime(small_path=small_path),
                                          [x.copy() for x in X], Y.copy(), cv=4, n_permutations=3, random_state=1)
    assert _same(_seeded(lambda: pts(True)), _seeded(lambda: pts(False)))


def test_infinity_is_rejected_and_nan_accepted():
    from mbpls_b200 import MBPLS
    from mbpls_b200.model_selection import bootstrap, cross_val_predict, permutation_test_score
    X, Y = _data(24, 1, seed=121)
    X, Y = iid_holes(X, Y, 0.1, seed=15)
    est = MBPLS(n_components=2, sparse_data=True).set_runtime(small_path=True)
    Xi = [x.copy() for x in X]
    Xi[1][3, 2] = np.inf
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        for call in (lambda A: cross_val_predict(est, A, Y, cv=3), lambda A: permutation_test_score(est, A, Y, cv=3, n_permutations=2),
                     lambda A: bootstrap(est, A, Y, n_resamples=2)):
            with pytest.raises(ValueError, match="infinity"):
                call(Xi)
            call(X)


# --------------------------------------------------------------------------------------------- #
# permutation test
# --------------------------------------------------------------------------------------------- #
def test_permutation_test_score_nan_matches_generic_path_and_oracle():
    from sklearn.model_selection import KFold
    from mbpls_b200 import MBPLS
    from mbpls_b200.model_selection import _permutations, permutation_test_score
    from oracle import OracleMBPLS
    n = 36
    X, Y = _data(n, 2, seed=131)
    X, Y = iid_holes(X, Y, 0.1, seed=16)
    cv = KFold(4)
    ks = [1, 2, 3]

    def run(small_path):
        with warnings.catch_warnings():
            warnings.simplefilter("ignore")
            c0 = _launches()
            r = permutation_test_score(MBPLS(n_components=1, sparse_data=True).set_runtime(small_path=small_path), X, Y, cv=cv,
                                       n_permutations=15, random_state=3, n_components_list=ks)
            return r, _launches() - c0
    got, launches = run(True)
    assert launches == 1
    gen, _ = run(False)
    folds = list(cv.split(np.arange(n)))
    perms = _permutations(n, 15, 3)
    for k in ks:
        want = []
        for pi in perms:
            s = []
            for tr, te in folds:
                with warnings.catch_warnings():
                    warnings.simplefilter("ignore")
                    m = OracleMBPLS(n_components=k, sparse_data=True).fit([x[tr] for x in X], Y[pi[tr]])
                    s.append(metrics.r2_score(Y[pi[te]], m.predict([x[te] for x in X])))
            want.append(np.mean(s))
        want = np.array(want)
        score, perm, pv = got[k]
        assert rel_err(score, gen[k][0]) <= 1e-9 and rel_err(perm, gen[k][1]) <= 1e-9 and pv == gen[k][2], k
        assert rel_err(score, want[0]) <= 1e-9 and rel_err(perm, want[1:]) <= 1e-9, k
        assert pv == (np.sum(want[1:] >= want[0]) + 1.0) / 16.0


# --------------------------------------------------------------------------------------------- #
# bootstrap
# --------------------------------------------------------------------------------------------- #
@pytest.mark.parametrize("holes", ["iid", "structured"])
def test_bootstrap_nan_matches_oracle_on_resampled_rows(holes):
    from mbpls_b200 import MBPLS
    from mbpls_b200.model_selection import bootstrap
    from oracle import OracleMBPLS
    n, q, K = 40, 2, 3
    X, Y = _data(n, q, seed=141)
    X, Y = iid_holes(X, Y, 0.1, seed=17) if holes == "iid" else structured_holes(X, Y, seed=18)

    def run(small_path):
        with warnings.catch_warnings():
            warnings.simplefilter("ignore")
            c0 = _launches()
            r = bootstrap(MBPLS(n_components=K, sparse_data=True).set_runtime(small_path=small_path), X, Y, n_resamples=10,
                          random_state=5)
            return r, _launches() - c0
    got, launches = run(True)
    gen, _ = run(False)
    assert launches == 1
    assert np.array_equal(got["n_iter_"], gen["n_iter_"])
    compared = 0
    for r, idx in enumerate(got["indices"]):
        with warnings.catch_warnings():
            warnings.simplefilter("ignore")
            o = OracleMBPLS(n_components=K, sparse_data=True).fit([x[idx] for x in X], Y[idx])
        if max(o.n_iter_) >= o.max_iter:
            # missing-data NIPALS need not converge: a component that oscillates until the trip cap ends in a state that
            # depends on every rounding on the way (structured resample 0, component 3: diff_t 0.26 after 100,000 trips)
            continue
        compared += 1
        for name in ("A_", "beta_", "A_corrected_", "explained_var_x_", "explained_var_y_", "explained_var_xblocks_"):
            assert rel_err(got[name][r], np.asarray(getattr(o, name))) <= 1e-8, (r, name)
            assert rel_err(got[name][r], gen[name][r]) <= 1e-9, (r, name)
        assert_trips(list(got["n_iter_"][r]), list(o.n_iter_), o.diff_trace_, 1e-14, f"resample {r}")
    assert compared >= 8


def test_bootstrap_resamples_the_batch_cannot_run_are_refit():
    """A feature observed in two rows only: the resamples that miss both go to MBPLS.fit, the others stay in the launch."""
    from mbpls_b200 import MBPLS
    from mbpls_b200.model_selection import _resamples, bootstrap
    n = 12
    X0, Y = _data(n, 1, seed=151)
    X, Y = iid_holes(X0, Y, 0.05, seed=19)
    X[0][:2, 5] = X0[0][:2, 5]
    X[0][2:, 5] = np.nan
    idx = _resamples(n, 12, 2)
    miss = [not np.isin([0, 1], r).any() for r in idx]
    assert any(miss) and not all(miss)

    def run(small_path):
        with warnings.catch_warnings():
            warnings.simplefilter("ignore")
            c0 = _launches()
            r = bootstrap(MBPLS(n_components=2, sparse_data=True).set_runtime(small_path=small_path), X, Y, n_resamples=12,
                          random_state=2)
            return r, _launches() - c0
    got, launches = run(True)
    gen, _ = run(False)
    assert launches > 1
    for r in range(12):
        for name in ("A_", "beta_", "n_iter_"):
            if miss[r]:  # the same MBPLS.fit on both sides
                assert np.array_equal(got[name][r], gen[name][r], equal_nan=True), (r, name)
            else:
                assert rel_err(got[name][r], gen[name][r]) <= 1e-9, (r, name)


# --------------------------------------------------------------------------------------------- #
# slot mode
# --------------------------------------------------------------------------------------------- #
def test_nan_slot_mode_is_bitwise_equal_to_one_cta_per_fit():
    import torch
    from mbpls_b200 import engine as E
    from mbpls_b200 import smallfit as SF
    from mbpls_b200.model_selection import _permutations
    X, Y = _data(33, 3, seed=161)
    X, Y = iid_holes(X, Y, 0.12, seed=20, y_cols=(0,))
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
                                       fit_preds=True, nanmode=True)
        res.append((lay.section(out, "small").clone(), lay.section(out, "beta").clone(), fp.clone()))
    torch.cuda.synchronize()
    for a, b in zip(*res):  # bit patterns (the prediction rows past a fold's test size hold NaN)
        assert torch.equal(a.view(torch.int64), b.view(torch.int64))
    flags = res[0][0][:, -1].cpu().numpy()
    assert np.any(flags == 0.0) and torch.isfinite(res[0][2]).any()
