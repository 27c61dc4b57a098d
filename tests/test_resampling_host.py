"""CPU: host logic of the permutation test and the bootstrap (mbpls_b200/model_selection.py) -- the vectorised scorers against
sklearn.metrics, the random draws against scikit-learn's, and the rejection of an unknown scoring before any device work."""
import warnings

import numpy as np
import pytest
from sklearn import metrics

from mbpls_b200.model_selection import _check_scoring, _permutations, _resamples, _scores

SKLEARN = {
    None: metrics.r2_score,
    "r2": metrics.r2_score,
    "explained_variance": metrics.explained_variance_score,
    "neg_mean_squared_error": lambda a, b: -metrics.mean_squared_error(a, b),
    "neg_root_mean_squared_error": lambda a, b: -metrics.root_mean_squared_error(a, b),
    "neg_mean_absolute_error": lambda a, b: -metrics.mean_absolute_error(a, b),
}


def _each(scoring, yt, yp):
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        return np.array([SKLEARN[scoring](a, b) for a, b in zip(yt, yp)])


@pytest.mark.parametrize("scoring", list(SKLEARN))
@pytest.mark.parametrize("m,q", [(7, 1), (12, 3), (1, 1), (1, 2), (2, 2)])
def test_vectorised_scores_match_sklearn(scoring, m, q):
    rng = np.random.default_rng(m * 10 + q)
    yt = rng.standard_normal((9, m, q))
    yp = yt + 0.3 * rng.standard_normal((9, m, q))
    yp[0] = yt[0]                          # perfect predictions
    yt[1] = 2.5                            # constant target, imperfect predictions
    yt[2], yp[2] = 1.5, 1.5                # constant target, perfect predictions
    if q > 1:
        yt[3, :, 0] = -1.0                 # one constant output among several
    got = _scores(scoring, yt, yp)
    want = _each(scoring, yt, yp)
    assert got.shape == (9,)
    assert np.array_equal(np.isnan(got), np.isnan(want)), (got, want)
    ok = ~np.isnan(want)
    np.testing.assert_allclose(got[ok], want[ok], rtol=1e-12, atol=1e-15)


def test_one_sample_fold_is_nan_for_r2_as_in_sklearn():
    yt, yp = np.array([[[1.0]]]), np.array([[[2.0]]])
    assert np.isnan(_scores("r2", yt, yp)[0]) and np.isnan(_scores(None, yt, yp)[0])
    assert _scores("explained_variance", yt, yp)[0] == _each("explained_variance", yt, yp)[0]


def test_scores_broadcast_over_prefix_models():
    rng = np.random.default_rng(3)
    yt = rng.standard_normal((4, 6, 2))
    yp = rng.standard_normal((4, 5, 6, 2))
    got = _scores("r2", yt[:, None], yp)
    assert got.shape == (4, 5)
    for k in range(5):
        np.testing.assert_allclose(got[:, k], _each("r2", yt, yp[:, k]), rtol=1e-12)


def test_permutations_are_drawn_like_sklearn_shuffle():
    from sklearn.model_selection._validation import _shuffle
    from sklearn.utils import check_random_state
    y = np.arange(23) * 1.0
    got = _permutations(23, 6, 7)
    rs = check_random_state(7)
    want = [np.arange(23)] + [_shuffle(y, None, rs).astype(int) for _ in range(6)]
    assert np.array_equal(got, np.stack(want))


def test_resamples_are_drawn_like_sklearn_resample():
    from sklearn.utils import check_random_state, resample
    got = _resamples(17, 5, 3)
    rs = check_random_state(3)
    assert np.array_equal(got, np.stack([resample(np.arange(17), random_state=rs) for _ in range(5)]))
    assert got.shape == (5, 17)


@pytest.mark.parametrize("bad", ["accuracy", "r2_score", 3, "neg_median_absolute_error"])
def test_unknown_scoring_is_rejected_before_any_device_work(bad):
    from mbpls_b200 import MBPLS
    from mbpls_b200.model_selection import permutation_test_score
    with pytest.raises(ValueError):
        _check_scoring(bad)
    # raises before any device is looked for (this machine may have none)
    with pytest.raises(ValueError):
        permutation_test_score(MBPLS(n_components=1), np.zeros((6, 3)), np.zeros(6), scoring=bad)
