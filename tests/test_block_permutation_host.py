"""CPU: the host side of block_permutation_test (mbpls_b200/model_selection.py): which block-permuted fits with missing values
the one-kernel batch runs (smallfit.nan_fits_eligible with a block's columns counted on other rows), the result's p-values,
shapes and keys, and the arguments it refuses before any device work."""
import numpy as np
import pytest

from mbpls_b200.smallfit import nan_fits_eligible


def _brute(x_obs, y_obs, x_rows, y_rows, cols, brows):
    out = []
    for f, (xr, yr) in enumerate(zip(x_rows, y_rows)):
        seen = x_obs[xr].sum(axis=0)
        if cols[f] is not None:
            lo, hi = cols[f]
            seen[lo:hi] = x_obs[brows[f]][:, lo:hi].sum(axis=0)
        yseen = y_obs[yr].sum(axis=0)
        out.append(bool((seen > 0).all() and (yseen > 0).all() and (yseen == len(yr)).any()))
    return out


def test_block_rows_eligibility_matches_a_brute_force_count():
    rng = np.random.default_rng(1)
    n, off = 24, [0, 4, 9, 12]
    x_obs = rng.random((n, 12)) > 0.35
    y_obs = rng.random((n, 2)) > 0.1
    y_obs[:, 1] = True
    perms = [rng.permutation(n) for _ in range(4)]
    x_rows, cols, brows = [], [], []
    for m in (3, 8, 20, 24):
        for b in (None, 0, 1, 2):
            for r in range(len(perms)):
                tr = np.sort(rng.choice(n, size=m, replace=False))
                x_rows.append(tr)
                cols.append(None if b is None else (off[b], off[b + 1]))
                brows.append(None if b is None else perms[r][tr])
    got = nan_fits_eligible(x_obs, y_obs, x_rows, x_rows, cols, brows)
    want = _brute(x_obs, y_obs, x_rows, x_rows, cols, brows)
    assert got.tolist() == want
    assert 0 < sum(want) < len(want)
    # without block maps: the same as the call without the new arguments
    assert nan_fits_eligible(x_obs, y_obs, x_rows, x_rows, [None] * len(x_rows), brows).tolist() == \
        nan_fits_eligible(x_obs, y_obs, x_rows, x_rows).tolist()


def test_feature_seen_only_on_rows_the_permutation_moves_out():
    x_obs = np.ones((6, 3), dtype=bool)
    x_obs[2:, 1] = False                             # feature 1 (block 1 = columns 1..2) seen in rows 0 and 1
    y_obs = np.ones((6, 1), dtype=bool)
    tr = np.arange(3)
    pi = np.array([3, 4, 5, 0, 1, 2])               # rows 0..2 of block 1 read source rows 3..5
    got = nan_fits_eligible(x_obs, y_obs, [tr, tr, tr], [tr, tr, tr], [None, (1, 3), (0, 1)], [None, pi[tr], pi[tr]])
    assert got.tolist() == [True, False, True]


def test_result_pvalues_shapes_and_keys():
    from mbpls_b200.model_selection import _block_permutation_result
    B, R, K = 2, 4, 3
    S = np.array([[0.5, 0.7], [0.1, 0.8], [0.6, 0.2], [0.5, 0.6], [0.0, 0.0], [0.4, 0.9], [0.9, 0.9], [0.2, 0.1], [0.3, 0.2]])
    A = np.zeros((1 + B * R, B, K))
    A[0] = [[0.6, 0.5, 0.1], [0.4, 0.5, 0.9]]
    A[1:5, 0] = [[0.7, 0.1, 0.1], [0.1, 0.5, 0.0], [0.2, 0.2, 0.2], [0.6, 0.6, 0.6]]
    A[5:9, 1] = [[0.1, 0.1, 0.1], [0.3, 0.3, 0.3], [0.5, 0.5, 0.95], [0.4, 0.4, 0.4]]
    A[1:5, 1] = A[5:9, 0] = 7.0                      # rows of the blocks that were not permuted are not part of the null
    got = _block_permutation_result(S, A, B, R, [1, 2])
    assert set(got) == {"score", "permutation_scores", "pvalue", "A_", "A_permuted", "A_pvalue"}
    assert got["score"] == {1: 0.5, 2: 0.7}
    assert np.array_equal(got["permutation_scores"][1], [[0.1, 0.6, 0.5, 0.0], [0.4, 0.9, 0.2, 0.3]])
    assert np.array_equal(got["pvalue"][1], [3 / 5, 2 / 5])     # >= counts ties
    assert np.array_equal(got["pvalue"][2], [2 / 5, 3 / 5])
    assert got["A_"].shape == (B, K) and got["A_permuted"].shape == (B, R, K)
    assert np.array_equal(got["A_permuted"][1], A[5:9, 1])
    assert np.array_equal(got["A_pvalue"], [[3 / 5, 3 / 5, 4 / 5], [3 / 5, 2 / 5, 2 / 5]])
    one = _block_permutation_result(S[:, 1:], None, B, R, None)
    assert set(one) == {"score", "permutation_scores", "pvalue"} and one["score"] == 0.7
    assert one["permutation_scores"].shape == (B, R) and np.array_equal(one["pvalue"], [2 / 5, 3 / 5])


@pytest.mark.parametrize("X", ["array", "one_block"])
def test_single_block_is_rejected(X):
    from mbpls_b200 import MBPLS
    from mbpls_b200.model_selection import block_permutation_test
    x = np.random.default_rng(0).standard_normal((10, 4))
    with pytest.raises(ValueError):
        block_permutation_test(MBPLS(), x if X == "array" else [x], np.arange(10.0))


def test_bad_scoring_is_rejected():
    from mbpls_b200 import MBPLS
    from mbpls_b200.model_selection import block_permutation_test
    x = np.random.default_rng(0).standard_normal((10, 4))
    with pytest.raises(ValueError):
        block_permutation_test(MBPLS(), [x, x], np.arange(10.0), scoring="accuracy")


def test_process_group_is_rejected():
    from mbpls_b200 import MBPLS
    from mbpls_b200.model_selection import block_permutation_test
    x = np.random.default_rng(0).standard_normal((10, 4))
    with pytest.raises(NotImplementedError):
        block_permutation_test(MBPLS().set_runtime(group=object()), [x, x], np.arange(10.0))
