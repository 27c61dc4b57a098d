"""CPU: the numpy oracle against the committed golden vectors (the reference's KAT CSVs and stored runs of the
unmodified reference)."""
import os

import numpy as np
import pytest

from oracle import OracleMBPLS, OracleScaler, nan_census
from oracle.make_golden import run_model

from helpers import GOLDEN, assert_fixture_trips, compare, live_cases, load_live


@pytest.mark.parametrize("tag,methods", [("pn", ["UNIPALS", "NIPALS", "KERNEL", "SIMPLS"]), ("np", ["UNIPALS", "KERNEL"])])
def test_oracle_matches_reference_kat_csvs(tag, methods):
    """Same assertions as mbpls/tests/test_mbpls.py:66-117, on inputs regenerated with the 2018 ortho_group."""
    z = np.load(os.path.join(GOLDEN, f"kat_{tag}.npz"))
    X = [z["in/x1_train"], z["in/x2_train"]]
    Xt = [z["in/x1_test"], z["in/x2_test"]]
    for method in methods:
        kw = dict(n_components=2, method=method, standardize=True, full_svd=True)
        s = run_model(OracleMBPLS, kw, [x.copy() for x in X], z["in/y_train"].copy(), [x.copy() for x in Xt], z["in/y_test"].copy())
        csv = lambda nm: z[f"csv/{method}/{nm}"]
        pairs = {"P1": s["P_/0"], "P2": s["P_/1"], "Ts": s["Ts_"], "U": s["U_"], "V": s["V_"], "Ts_test": s["tr_Ts"],
                 "U_test": s["tr_U"]}
        if method != "SIMPLS":
            pairs["T"] = np.concatenate([s["T_/0"], s["T_/1"]], axis=1)
            pairs["T_test"] = np.concatenate([s["tr_T/0"], s["tr_T/1"]], axis=1)
            assert np.allclose(s["A_"], csv("A"))
        for nm, val in pairs.items():
            assert np.allclose(abs(val), abs(csv(nm))), (method, nm)
        assert np.allclose(s["beta_"], csv("beta"))
        assert np.allclose(s["predict"], csv("Y_predict_test"))


@pytest.mark.parametrize("name", live_cases())
def test_oracle_matches_live_reference_fixtures(name):
    X, Y, Xt, Yt, kwargs, ref = load_live(name)
    cp = (lambda a: [x.copy() for x in a] if isinstance(a, list) else a.copy())
    ours = run_model(OracleMBPLS, kwargs, cp(X), cp(Y), cp(Xt), cp(Yt))
    compare(ours, ref, 1e-9, name)
    if "n_iter_" in ref:
        assert_fixture_trips(ours["n_iter_"], name, ref)


def test_oracle_scaler_matches_sklearn():
    from sklearn.preprocessing import StandardScaler
    rng = np.random.default_rng(0)
    X = rng.standard_normal((50, 7)) * rng.uniform(0.1, 50, 7) + rng.uniform(-5, 5, 7)
    X[:, 3] = 2.5  # constant column -> scale 1
    Xn = X.copy()
    Xn[rng.random(X.shape) < 0.1] = np.nan
    for A in (X, Xn):
        a, b = OracleScaler().fit(A), StandardScaler().fit(A)
        assert np.allclose(a.mean_, b.mean_, rtol=1e-14, atol=0, equal_nan=True)
        assert np.allclose(a.var_, b.var_, rtol=1e-13, atol=1e-300, equal_nan=True)
        assert np.allclose(a.scale_, b.scale_, rtol=1e-13, equal_nan=True)
        assert np.array_equal(np.asarray(a.n_samples_seen_), np.asarray(b.n_samples_seen_))
        assert np.allclose(a.transform(A), b.transform(A), rtol=1e-13, atol=1e-15, equal_nan=True)


def test_nan_census_shapes_and_warning():
    A = np.zeros((4, 3))
    A[0, 1] = np.nan
    r, c, dr, dc = nan_census(A)
    assert list(r) == [0] and list(c) == [1] and list(dr) == [1, 2, 3] and list(dc) == [0, 2]
    A[:, :] = np.nan
    with pytest.warns(UserWarning):
        nan_census(A)

