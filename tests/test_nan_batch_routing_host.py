"""CPU: which fits of a cross-validation, permutation test or bootstrap with missing values (sparse_data=True) the one-kernel
NaN batch runs, and which go to MBPLS.fit (mbpls_b200/smallfit.py nan_fits_eligible), on hand-made hole patterns."""
import numpy as np

from mbpls_b200.smallfit import nan_fits_eligible


def _obs(shape, holes):
    o = np.ones(shape, dtype=bool)
    for i, j in holes:
        o[i, j] = False
    return o


def test_scattered_holes_are_eligible():
    x = _obs((6, 3), [(0, 1), (3, 2), (5, 0)])
    y = _obs((6, 2), [(0, 0)])                       # column 1 is fully observed: the Y scores start there
    got = nan_fits_eligible(x, y, [np.arange(6), np.arange(1, 6)], [np.arange(6), np.arange(1, 6)])
    assert got.tolist() == [True, True]


def test_feature_unobserved_on_the_training_rows_goes_to_fit():
    x = _obs((6, 3), [(2, 1), (3, 1), (4, 1), (5, 1)])  # feature 1 is seen in rows 0 and 1 only
    y = np.ones((6, 1), dtype=bool)
    rows = [np.arange(6), np.array([2, 3, 4, 5]), np.array([1, 2, 3]), np.array([0, 0, 3])]
    assert nan_fits_eligible(x, y, rows, rows).tolist() == [True, False, True, True]


def test_y_column_unobserved_on_the_y_rows_goes_to_fit():
    x = np.ones((5, 2), dtype=bool)
    y = _obs((5, 2), [(0, 0), (1, 0), (2, 1)])           # column 0 seen in rows 2..4 only
    xr = [np.arange(5), np.arange(5)]
    yr = [np.array([0, 1, 0, 1, 1]), np.array([2, 3, 4, 3, 2])]  # permuted / resampled Y rows paired with the X rows
    assert nan_fits_eligible(x, y, xr, yr).tolist() == [False, True]


def test_no_fully_observed_y_column_goes_to_fit():
    x = np.ones((6, 2), dtype=bool)
    y = _obs((6, 3), [(0, 0), (1, 1), (2, 2)])
    rows = [np.arange(6), np.array([3, 4, 5]), np.array([1, 2, 3, 4]), np.array([0, 3, 3])]
    # fit 0: every column has a hole; fit 1: none has; fit 2: column 0 is whole; fit 3: columns 1 and 2 are whole
    assert nan_fits_eligible(x, y, rows, rows).tolist() == [False, True, True, True]


def test_repeated_rows_count_once_per_occurrence():
    x = _obs((4, 2), [(1, 0), (2, 0), (3, 0)])
    y = _obs((4, 2), [(0, 1)])
    # X feature 0 is seen only in row 0; Y column 1 misses row 0, column 0 is whole
    rows = [np.array([1, 1, 2, 3]), np.array([0, 0, 0, 1]), np.array([3, 3, 3, 3])]
    assert nan_fits_eligible(x, y, rows, rows).tolist() == [False, True, False]


def test_fits_of_different_sizes_in_one_call():
    rng = np.random.default_rng(0)
    x = rng.random((30, 7)) > 0.2
    x[:, 0] = True
    y = rng.random((30, 3)) > 0.3
    y[:, 2] = True
    rows = [rng.choice(30, size=m, replace=True) for m in (1, 5, 29, 30, 12)]
    yrows = [rng.permutation(30)[:len(r)] for r in rows]
    got = nan_fits_eligible(x, y, rows, yrows)
    want = [x[r].any(axis=0).all() and y[yr].any(axis=0).all() and y[yr].all(axis=0).any() for r, yr in zip(rows, yrows)]
    assert got.tolist() == want
