"""The third-party arithmetic restated inside the oracle (numpy mean/round, scikit-learn predict_proba) against the
installed libraries themselves."""
import ctypes as C
import os
import warnings

import numpy as np
import pytest

import golden_cases as gc


def _bits(x):
    return np.float64(x).view(np.uint64)


def test_np_mean_order(oracle):
    """orc_np_mean equals np.mean as bits (the sign of a zero included): every count numpy sums differently (left to right
    below 8, 8 lanes and a tail up to 128, recursive halving above, counts past numpy's 8192-element buffer), and columns
    of -0.0 values, which numpy's reduction turns into 0.0 by starting it from 0.0."""
    L = oracle.lib()
    rng = np.random.default_rng(1)
    for n in list(range(1, 40)) + [64, 127, 128, 129, 200, 300, 1000, 4097, 8193, 65534, 100000]:
        for _ in range(50 if n <= 1000 else 3):
            a = np.round(rng.uniform(-20, 20, n), 4)
            got = L.orc_np_mean(a.ctypes.data_as(C.c_void_p), C.c_int64(n))
            assert _bits(got) == _bits(np.mean(list(a))), n
    for n in (1, 7, 8, 129):
        a = np.full(n, -0.0)
        got = L.orc_np_mean(a.ctypes.data_as(C.c_void_p), C.c_int64(n))
        assert _bits(got) == _bits(np.mean(list(a))) == _bits(0.0), n


def test_np_round4(oracle):
    L = oracle.lib()
    rng = np.random.default_rng(2)
    for _ in range(20000):
        ev, md = "%.2f" % rng.uniform(40, 140), "%.2f" % rng.uniform(40, 140)
        x = float(ev) - float(md)
        assert L.orc_np_round(x, 4) == float(np.round(x, 4))
    for x in (0.00005, -0.00005, 0.00015, 1.23455, -7.000049999, 0.0, -0.0):
        assert L.orc_np_round(x, 4) == float(np.round(x, 4))


def _X(n=400, seed=3):
    rng = np.random.default_rng(seed)
    X = rng.normal(0, 3, (n, 7))
    X[:, 6] = rng.uniform(3, 20, n)
    return X


@pytest.mark.parametrize("pkl", [gc.R95, gc.R94, gc.CAAY_BARE])
def test_mlp_matches_sklearn(pkl, oracle):
    m = oracle.load_pickle(os.path.join(gc.GOLD, "models", pkl))
    ests = list(m.values()) if isinstance(m, dict) else [m]
    X = _X()
    for est in ests:
        with warnings.catch_warnings():
            warnings.simplefilter("ignore")
            want = est.predict_proba(X)[:, 1]
        got = oracle.predict(est, X)
        assert np.max(np.abs(got - want)) < 1e-12


def _fit_alt(kind):
    from sklearn.ensemble import RandomForestClassifier
    from sklearn.linear_model import LogisticRegression
    from sklearn.naive_bayes import GaussianNB
    rng = np.random.default_rng(7)
    X = _X(3000, 9)
    y = np.where(X[:, 2] - X[:, 3] + 0.3 * X[:, 0] + rng.normal(0, 1.5, len(X)) > 0, "m6A", "A")
    if kind == "RF":      # hyper-parameters of train_model.py:39-45 (minus the removed min_impurity_split)
        est = RandomForestClassifier(n_estimators=50, criterion="entropy", max_depth=10, max_features=4, min_samples_leaf=2,
                                     min_samples_split=3, random_state=0)
    elif kind == "LR":
        est = LogisticRegression()
    else:
        est = GaussianNB()
    return est.fit(X, y)


@pytest.mark.parametrize("kind,tol", [("RF", 1e-12), ("LR", 1e-12), ("NBC", 1e-10)])
def test_alt_classifiers_match_sklearn(kind, tol, oracle):
    est = _fit_alt(kind)
    X = _X(500, 11)
    want = est.predict_proba(X)[:, 1]
    got = oracle.predict(est, X)
    assert np.max(np.abs(got - want)) < tol
