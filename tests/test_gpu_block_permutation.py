"""GPU: block permutation tests of multiblock fits (mbpls_b200/model_selection.py block_permutation_test) -- the row map of
smallfit_kernel (a fit reads one block's columns from permuted rows) bitwise against a host-permuted source, the batched path
and the generic refit path against loops over the numpy oracle, with missing values, and one launch for many fits.
(conftest.py switches the automatic small path off, so the batched cases ask for it with small_path=True.)"""
import warnings

import numpy as np
import pytest
from sklearn import metrics

from helpers import rel_err

pytestmark = pytest.mark.gpu

METRIC = {None: metrics.r2_score, "neg_mean_absolute_error": lambda a, b: -metrics.mean_absolute_error(a, b)}


def _launches():
    from mbpls_b200 import _cabi
    return _cabi.launch_count


def _iid_holes(X, frac, seed):
    """i.i.d. holes in every feature but the first of each block (no sample loses a whole block)."""
    rng = np.random.default_rng(seed)
    out = [x.copy() for x in X]
    for x in out:
        hole = rng.random(x.shape) < frac
        hole[:, 0] = False
        x[hole] = np.nan
    return out


def _run(X, Y, small_path=True, **kw):
    from mbpls_b200 import MBPLS
    from mbpls_b200.model_selection import block_permutation_test
    est = {k: kw.pop(k) for k in ("n_components", "method", "sparse_data", "full_svd") if k in kw}
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        return block_permutation_test(MBPLS(**est).set_runtime(small_path=small_path), [x.copy() for x in X], Y.copy(), **kw)


def _oracle(kw, X, Y, folds, perms, ks, scoring=None, with_A=True):
    """The test by explicit loops: OracleMBPLS fitted on X with X[b] replaced by X[b][pi], scored on the folds, and on all
    rows for A_.  Returns ({k: (score, (B, R) scores, (B,) p-values)}, A_, A_permuted)."""
    from oracle import OracleMBPLS
    B, R, K = len(X), len(perms), max(ks)
    variants = [list(X)] + [[x[pi] if c == b else x for c, x in enumerate(X)] for b in range(B) for pi in perms]
    S = np.zeros((len(variants), len(ks)))
    A = np.zeros((len(variants), B, K))
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        for v, Xv in enumerate(variants):
            for j, k in enumerate(ks):
                s = []
                for tr, te in folds:
                    m = OracleMBPLS(**dict(kw, n_components=k)).fit([x[tr] for x in Xv], Y[tr])
                    s.append(METRIC[scoring](Y[te], np.asarray(m.predict([x[te] for x in Xv])).reshape(Y[te].shape)))
                S[v, j] = np.mean(s)
            if with_A:
                A[v] = OracleMBPLS(**dict(kw, n_components=K)).fit(Xv, Y).A_
    res = {}
    for j, k in enumerate(ks):
        ps = S[1:, j].reshape(B, R)
        res[k] = (S[0, j], ps, (np.sum(ps >= S[0, j], axis=1) + 1.0) / (R + 1.0))
    Ap = np.stack([A[1 + b * R:1 + (b + 1) * R, b] for b in range(B)])
    return res, A[0], Ap


def _check_against_oracle(got, want, ks, tol):
    res, A0, Ap = want
    for k in ks:
        g = (got["score"][k], got["permutation_scores"][k], got["pvalue"][k]) if isinstance(got["score"], dict) else \
            (got["score"], got["permutation_scores"], got["pvalue"])
        assert rel_err(g[0], res[k][0]) < tol and rel_err(g[1], res[k][1]) < tol, k
        assert np.array_equal(g[2], res[k][2]), (k, g[2], res[k][2])
    assert rel_err(got["A_"], A0) < tol and rel_err(got["A_permuted"], Ap) < tol
    R = Ap.shape[1]
    assert np.array_equal(got["A_pvalue"], (np.sum(Ap >= A0[:, None, :], axis=1) + 1.0) / (R + 1.0))


# --------------------------------------------------------------------------------------------- #
# the kernel's row map
# --------------------------------------------------------------------------------------------- #
@pytest.mark.parametrize("nanmode", [False, True])
@pytest.mark.parametrize("nslots", [0, 3])
def test_row_map_is_bitwise_equal_to_a_host_permuted_block(nanmode, nslots):
    import torch
    from mbpls_b200 import engine as E
    from mbpls_b200 import smallfit as SF
    from mbpls_b200.model_selection import _permutations
    from oracle.cases import latent_blocks
    X, Y = latent_blocks(33, (10, 7, 8), 2, 4, seed=81)
    if nanmode:
        X = _iid_holes(X, 0.1, seed=3)
    dev = torch.device("cuda", 0)
    n, b = 33, 1
    perms = _permutations(n, 3, 4)[1:]
    folds = [(np.setdiff1d(np.arange(n), te), te) for te in np.array_split(np.arange(n), 4)]
    tr = [f[0].astype(np.int32) for f in folds]
    te = [f[1].astype(np.int32) for f in folds]
    boff = E.ShardMap.build([x.shape[1] for x in X], 0, 1).block_off

    def launch(blocks, block_perm=None):
        D, n_, sizes, p, q, ldx = SF.pack_source(blocks, Y, dev)
        lay, out, fp, keep = SF.launch(D, n_, p, q, ldx, boff, 4, True, 0, 1e-14, 10**6, tr + tr, te + te, nslots=nslots,
                                       fit_preds=True, nanmode=nanmode, block_perm=block_perm)
        torch.cuda.synchronize()
        return lay.section(out, "small").clone(), fp.clone()

    # fits 0..3 permute block b by permutation 2, fits 4..7 permute nothing
    got = launch(X, (perms, [(2, b)] * 4 + [(-1, 0)] * 4))
    host = launch([x[perms[2]] if c == b else x for c, x in enumerate(X)])
    plain = launch(X)
    bits = lambda t: t.view(torch.int64)
    for g, h, o in zip(got, host, plain):
        assert torch.equal(bits(g[:4]), bits(h[:4])) and torch.equal(bits(g[4:]), bits(o[4:]))
    assert torch.isfinite(got[1]).any() and not torch.equal(bits(got[0][:4]), bits(plain[0][:4]))


def test_row_map_rejects_bad_pairs():
    import torch
    from mbpls_b200 import _cabi, engine as E
    from mbpls_b200 import smallfit as SF
    from oracle.cases import latent_blocks
    X, Y = latent_blocks(20, (6, 5), 1, 2, seed=82)
    dev = torch.device("cuda", 0)
    D, n, sizes, p, q, ldx = SF.pack_source(X, Y, dev)
    boff = E.ShardMap.build(sizes, 0, 1).block_off
    perms = np.stack([np.random.default_rng(0).permutation(n) for _ in range(2)])
    tr = [np.arange(n, dtype=np.int32)]
    for pair in ((2, 0), (0, 2), (-2, 0), (1, -1)):
        with pytest.raises(_cabi.MbplsCudaError):
            SF.launch(D, n, p, q, ldx, boff, 2, True, 0, 1e-14, 10**6, tr, block_perm=(perms, [pair]))
    with pytest.raises(ValueError):  # every sample of the source, in order: no index tables to map
        SF.launch(D, n, p, q, ldx, boff, 2, True, 0, 1e-14, 10**6, None, block_perm=(perms, [(0, 0)]))


# --------------------------------------------------------------------------------------------- #
# block_permutation_test against the oracle
# --------------------------------------------------------------------------------------------- #
@pytest.mark.parametrize("q,scoring", [(1, None), (3, "neg_mean_absolute_error")])
def test_batched_path_matches_oracle_loop(q, scoring):
    from sklearn.model_selection import KFold
    from mbpls_b200.model_selection import _permutations
    from oracle.cases import latent_blocks
    n, ks = 30, [1, 2, 3]
    X, Y = latent_blocks(n, (8, 6, 7), q, 3, seed=83 + q)
    Y = Y.reshape(n, q)
    cv = KFold(3)
    c0 = _launches()
    got = _run(X, Y.ravel() if q == 1 else Y, n_components=1, cv=cv, n_permutations=6, random_state=5, scoring=scoring,
               n_components_list=ks)
    assert _launches() - c0 == 1
    assert got["permutation_scores"][3].shape == (3, 6) and got["pvalue"][3].shape == (3,)
    assert got["A_"].shape == (3, 3) and got["A_permuted"].shape == (3, 6, 3) and got["A_pvalue"].shape == (3, 3)
    want = _oracle({}, X, Y, list(cv.split(np.arange(n))), _permutations(n, 6, 5)[1:], ks, scoring)
    _check_against_oracle(got, want, ks, 1e-9)


@pytest.mark.parametrize("q,method", [(2, "NIPALS"), (1, "KERNEL")])
def test_generic_path_agrees_with_the_batched_path(q, method):
    """small_path=False refits every fit through MBPLS.fit; KERNEL fits the same model as NIPALS for one y column."""
    from oracle.cases import latent_blocks
    X, Y = latent_blocks(28, (9, 7, 6), q, 3, seed=85)
    kw = dict(cv=4, n_permutations=5, random_state=2, n_components_list=[1, 2])
    a = _run(X, Y, True, n_components=2, **kw)
    c0 = _launches()
    b = _run(X, Y, False, n_components=2, method=method, full_svd=True, **kw)
    assert _launches() - c0 > 1
    for k in (1, 2):
        assert rel_err(a["score"][k], b["score"][k]) < 1e-9
        assert rel_err(a["permutation_scores"][k], b["permutation_scores"][k]) < 1e-9
        assert np.array_equal(a["pvalue"][k], b["pvalue"][k])
    for name in ("A_", "A_permuted"):
        assert rel_err(a[name], b[name]) < 1e-9, name
    assert np.array_equal(a["A_pvalue"], b["A_pvalue"])


def test_simpls_has_no_importance_keys():
    from mbpls_b200.model_selection import _folds, _permutations
    from oracle.cases import latent_blocks
    X, Y = latent_blocks(24, (8, 6), 1, 2, seed=86)
    got = _run(X, Y, False, n_components=2, method="SIMPLS", full_svd=True, cv=4, n_permutations=4, random_state=1)
    assert set(got) == {"score", "permutation_scores", "pvalue"}
    res, _, _ = _oracle(dict(method="SIMPLS", full_svd=True), X, Y, _folds(24, 4), _permutations(24, 4, 1)[1:], [2],
                        with_A=False)
    assert rel_err(got["score"], res[2][0]) < 1e-9 and rel_err(got["permutation_scores"], res[2][1]) < 1e-9
    assert np.array_equal(got["pvalue"], res[2][2])


def test_more_fits_than_two_slots_per_sm_take_one_launch():
    import torch
    from oracle.cases import latent_blocks
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    nperm = sms // 6 + 1                            # (1 + 2 nperm) units x (5 folds + 1) fits > 2 x SM count
    X, Y = latent_blocks(30, (12, 10), 1, 2, seed=87)
    c0 = _launches()
    got = _run(X, Y, n_components=2, cv=5, n_permutations=nperm)
    assert _launches() - c0 == 1
    assert (1 + 2 * nperm) * 6 > 2 * sms
    assert got["permutation_scores"].shape == (2, nperm) and np.all(np.isfinite(got["permutation_scores"]))
    assert got["A_permuted"].shape == (2, nperm, 2) and np.all(np.isfinite(got["A_permuted"]))


# --------------------------------------------------------------------------------------------- #
# missing values
# --------------------------------------------------------------------------------------------- #
def test_nan_mode_iid_holes_match_oracle_loop():
    from sklearn.model_selection import KFold
    from mbpls_b200.model_selection import _permutations
    from oracle.cases import latent_blocks
    n, ks = 32, [1, 2, 3]
    X, Y = latent_blocks(n, (9, 7, 8), 2, 3, seed=88)
    X = _iid_holes(X, 0.1, seed=9)
    c0 = _launches()
    got = _run(X, Y, n_components=3, sparse_data=True, cv=KFold(4), n_permutations=5, random_state=3, n_components_list=ks)
    assert _launches() - c0 == 1
    want = _oracle(dict(sparse_data=True), X, Y, list(KFold(4).split(np.arange(n))), _permutations(n, 5, 3)[1:], ks)
    _check_against_oracle(got, want, ks, 1e-8)
    per_fit = _run(X, Y, False, n_components=3, sparse_data=True, cv=KFold(4), n_permutations=5, random_state=3,
                   n_components_list=ks)
    for k in ks:
        assert rel_err(got["permutation_scores"][k], per_fit["permutation_scores"][k]) < 1e-9
    assert rel_err(got["A_permuted"], per_fit["A_permuted"]) < 1e-9


def test_nan_mode_structured_holes_match_oracle_loop():
    """A feature missing 80 % of the samples and a block missing all but one feature on a quarter of them: the holes move
    with the permuted block's rows."""
    from mbpls_b200.model_selection import _folds, _permutations
    from oracle.cases import latent_blocks
    n = 36
    X, Y = latent_blocks(n, (9, 7, 8), 1, 3, seed=89)
    rng = np.random.default_rng(4)
    X[0][rng.choice(n, round(0.8 * n), replace=False), 3] = np.nan
    X[2][np.ix_(rng.choice(n, n // 4, replace=False), np.arange(1, 8))] = np.nan
    got = _run(X, Y, n_components=2, sparse_data=True, cv=4, n_permutations=5, random_state=6)
    want = _oracle(dict(sparse_data=True), X, Y, _folds(n, 4), _permutations(n, 5, 6)[1:], [2])
    _check_against_oracle(got, want, [2], 1e-8)


def test_permuted_block_with_a_feature_unobserved_on_training_rows_goes_to_fit():
    """Block 0 feature 2 is observed on two rows only: unpermuted, every fold's training rows see one of them; some
    permutations put both among one fold's test rows.  Those fits go to MBPLS.fit, and the batch returns whatever the per-fit
    path returns."""
    from mbpls_b200 import smallfit as SF
    from mbpls_b200.model_selection import _folds, _permutations
    from oracle.cases import latent_blocks
    n, R = 30, 8
    X, Y = latent_blocks(n, (6, 5), 1, 2, seed=90)
    X[0][:, 2] = np.nan
    X[0][[0, 15], 2] = 1.0, -1.0
    folds = _folds(n, 3)
    perms = _permutations(n, R, 7)[1:]
    x_obs = np.hstack([~np.isnan(x) for x in X])
    y_obs = np.ones((n, 1), dtype=bool)
    rows = [tr for _ in range(R) for tr, _ in folds]
    ok = SF.nan_fits_eligible(x_obs, y_obs, rows, rows, [(0, 6)] * len(rows), [pi[tr] for pi in perms for tr, _ in folds])
    assert SF.nan_fits_eligible(x_obs, y_obs, rows[:3], rows[:3]).all() and not ok.all()

    def run(small_path):
        np.random.seed(1234)
        try:
            return _run(X, Y, small_path, n_components=2, sparse_data=True, cv=3, n_permutations=R, random_state=7)
        except Exception as e:  # noqa: BLE001 -- compared below by type and message
            return e
    a, b = run(True), run(False)
    if isinstance(a, Exception) or isinstance(b, Exception):
        assert type(a) is type(b) and str(a) == str(b)
        return
    assert np.isnan(a["permutation_scores"]).any()  # the reference's SVD does not converge either (as the fold loop does)
    for name in a:
        assert np.allclose(np.asarray(a[name], float), np.asarray(b[name], float), rtol=1e-9, atol=0, equal_nan=True), name


# --------------------------------------------------------------------------------------------- #
# sanity
# --------------------------------------------------------------------------------------------- #
def test_informative_block_is_significant_and_noise_block_is_not():
    rng = np.random.default_rng(12)
    n, R = 40, 49
    z = rng.standard_normal(n)
    X = [np.outer(z, rng.standard_normal(10)) + 0.3 * rng.standard_normal((n, 10)), rng.standard_normal((n, 12))]
    y = z + 0.1 * rng.standard_normal(n)
    got = _run(X, y, n_components=1, cv=5, n_permutations=R, random_state=0)
    assert got["pvalue"][0] == 1.0 / (R + 1) and got["pvalue"][1] > 0.05
    assert got["A_pvalue"][0, 0] == 1.0 / (R + 1)
