#!/usr/bin/env python
"""Fits the alternative classifiers the reference offers with -c RF / LR / NBC (train_model.py:39-60) on deterministic
synthetic feature rows and pickles them as {'MG': est, 'MH': est} (the layout mCaller.py expects with -b A, SURVEY.md Q9)
under tests/golden/models/ -- the reference ships no such pickles.  tools/make_golden.py then runs the UNMODIFIED
reference on them (cases rf_gatc / lr_gatc / nbc_gatc), so the tree-walk / linear / naive-Bayes kernels are pinned against
the reference end to end, not only against scikit-learn.

    python tools/make_alt_models.py
"""
import gzip
import os
import pickle
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
OUT = os.path.join(os.path.dirname(HERE), "tests", "golden", "models")


def fit(kind):
    from sklearn.ensemble import RandomForestClassifier
    from sklearn.linear_model import LogisticRegression
    from sklearn.naive_bayes import GaussianNB
    rng = np.random.RandomState(5)
    # features like the window builder's: six current deviations (pA) and a mean read quality
    X = np.column_stack([rng.normal(0.0, 2.4, size=(6000, 6)), rng.uniform(3.0, 24.0, size=6000)])
    y = np.where(X[:, 2] - 0.8 * X[:, 3] + 0.4 * X[:, 0] + rng.normal(0, 1.2, 6000) > 0.3, "m6A", "A")
    if kind == "RF":       # hyper-parameters of train_model.py:39-45 (minus the arguments scikit-learn has dropped since)
        est = RandomForestClassifier(n_estimators=50, criterion="entropy", max_depth=10, max_features=4, min_samples_leaf=2,
                                     min_samples_split=3, random_state=0)
    elif kind == "LR":     # train_model.py:55-57
        est = LogisticRegression()
    else:                  # train_model.py:59-60
        est = GaussianNB()
    return est.fit(X, y)


if __name__ == "__main__":
    os.makedirs(OUT, exist_ok=True)
    for kind in ("RF", "LR", "NBC"):
        est = fit(kind)
        path = os.path.join(OUT, "alt_%s_6_m6A.pkl" % kind)
        data = pickle.dumps({"MG": est, "MH": est}, protocol=2)
        if kind == "RF":                # 2.4 MB of trees: stored gzipped, tests/golden_cases.py unpacks it for the runs
            path += ".gz"
            data = gzip.compress(data, 9, mtime=0)
        with open(path, "wb") as fh:
            fh.write(data)
        print(path, os.path.getsize(path))
