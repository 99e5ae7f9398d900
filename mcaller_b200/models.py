"""Loading the pickled scikit-learn models mCaller ships / trains (unchanged files) and exporting their fitted
parameters to device memory for stage 6 (reference extract_contexts.py:121-131 load, :195-207 apply)."""
import pickle
import warnings

import numpy as np
import torch

from ._lib import MC_GNB, MC_LR, MC_MLP, MC_RF, Model

_ACT = {"identity": 0, "logistic": 1, "tanh": 2, "relu": 3}


class _AliasingUnpickler(pickle.Unpickler):
    """The shipped r94/r95 pickles were written by python2-era scikit-learn whose module paths have since moved."""
    _MAP = {"sklearn.neural_network.multilayer_perceptron": "sklearn.neural_network._multilayer_perceptron",
            "sklearn.preprocessing.label": "sklearn.preprocessing._label",
            "sklearn.ensemble.forest": "sklearn.ensemble._forest", "sklearn.tree.tree": "sklearn.tree._classes",
            "sklearn.linear_model.logistic": "sklearn.linear_model._logistic",
            "sklearn.naive_bayes": "sklearn.naive_bayes"}

    def find_class(self, module, name):
        return super().find_class(self._MAP.get(module, module), name)


def load_model_file(path):
    """pickle.load(modfi, encoding='latin') with module aliasing (extract_contexts.py:123-125)."""
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        with open(path, "rb") as fh:
            return _AliasingUnpickler(fh, encoding="latin").load()


def select_models(model, base):
    """(estimator for 'MH'/'general', estimator for 'MG' or None, two_models flag) -- extract_contexts.py:126-131 and
    base_models :99-106.  Extension (SURVEY.md Q9): a {'general': est} dict is accepted (the reference raises KeyError)."""
    if not isinstance(model, dict):
        return model, None, False
    if base == "A" and "MG" in model and "MH" in model:
        return model["MH"], model["MG"], True
    if "general" in model:
        return model["general"], None, False
    raise KeyError("model dict has neither MG/MH (base A) nor 'general'")


def input_width(est):
    """Number of features a supported estimator takes (read from its fitted parameters, so older pickles without
    n_features_in_ work too)."""
    tn = type(est).__name__
    if tn == "MLPClassifier":
        return int(est.coefs_[0].shape[0])
    if tn == "LogisticRegression":
        return int(est.coef_.shape[1])
    if tn == "GaussianNB":
        return int(est.theta_.shape[1])
    if tn == "RandomForestClassifier":
        return int(est.n_features_in_)
    raise TypeError("unsupported estimator type %s (supported: MLPClassifier, RandomForestClassifier, LogisticRegression, GaussianNB)" % tn)


class DeviceModels(object):
    """Two mc_model structs (index 0 = 'MH'/'general', 1 = 'MG') backed by device tensors.  Both must be of one estimator
    type: mc_classify runs one kernel for all rows (the reference would apply each key's estimator on its own; mCaller's
    own training never writes a mixed dict).  `n_in`: the input width both must have (k + 1); checked, like the types,
    before anything is copied to the device."""

    def __init__(self, est0, est1=None, device="cuda", n_in=None):
        if est1 is not None and type(est0).__name__ != type(est1).__name__:
            raise TypeError("model dict mixes estimator types: 'MH' is %s, 'MG' is %s (both keys must have one type)"
                            % (type(est0).__name__, type(est1).__name__))
        if n_in is not None:
            named = (("model 'MH'", est0), ("model 'MG'", est1)) if est1 is not None else (("model", est0),)
            for what, est in named:
                if input_width(est) != n_in:
                    raise ValueError("%s expects %d inputs but -n %d gives %d" % (what, input_width(est), n_in - 1, n_in))
        self.device = torch.device(device)
        self._keep = []
        arr = (Model * 2)()
        self._export(est0, arr[0])
        self._export(est1 if est1 is not None else est0, arr[1])
        self.array = arr
        self.kind = arr[0].kind
        self.n_in = arr[0].n_in

    def _dev(self, a, dtype):
        t = torch.from_numpy(np.ascontiguousarray(np.asarray(a), dtype=dtype)).to(self.device)
        self._keep.append(t)
        return t.data_ptr()

    def _export(self, est, m):
        tn = type(est).__name__
        if tn == "MLPClassifier":
            sizes = [est.coefs_[0].shape[0]] + [c.shape[1] for c in est.coefs_]
            if sizes[-1] != 1 or est.out_activation_ != "logistic":
                raise ValueError("only binary MLPClassifier models are supported")
            m.kind, m.n_in, m.n_layers, m.hidden_act = MC_MLP, sizes[0], len(est.coefs_), _ACT[est.activation]
            for i, s in enumerate(sizes):
                m.sizes[i] = s
            m.d_weights = self._dev(np.concatenate([np.asarray(c, dtype=np.float64).ravel() for c in est.coefs_]), np.float64)
            m.d_biases = self._dev(np.concatenate([np.asarray(b, dtype=np.float64).ravel() for b in est.intercepts_]), np.float64)
        elif tn == "LogisticRegression":
            m.kind, m.n_in = MC_LR, est.coef_.shape[1]
            m.d_weights, m.d_biases = self._dev(est.coef_.ravel(), np.float64), self._dev(est.intercept_.ravel(), np.float64)
        elif tn == "GaussianNB":
            var = est.var_ if hasattr(est, "var_") else est.sigma_
            m.kind, m.n_in = MC_GNB, est.theta_.shape[1]
            m.d_weights = self._dev(np.concatenate([est.theta_.ravel(), np.asarray(var).ravel()]), np.float64)
            m.d_biases = self._dev(np.log(est.class_prior_), np.float64)
        elif tn == "RandomForestClassifier":
            off, L, R, F, T, P = [0], [], [], [], [], []
            for t in est.estimators_:
                tr = t.tree_
                L.append(tr.children_left); R.append(tr.children_right); F.append(np.maximum(tr.feature, 0)); T.append(tr.threshold)
                v = tr.value[:, 0, :]
                P.append(v[:, 1] / v.sum(axis=1))
                off.append(off[-1] + tr.node_count)
            m.kind, m.n_in, m.n_trees = MC_RF, est.n_features_in_, len(est.estimators_)
            m.max_nodes = int(max(np.diff(off)))
            m.d_tree_off = self._dev(off, np.int32)
            m.d_left, m.d_right = self._dev(np.concatenate(L), np.int32), self._dev(np.concatenate(R), np.int32)
            m.d_feature = self._dev(np.concatenate(F), np.int32)
            m.d_threshold, m.d_leaf_p1 = self._dev(np.concatenate(T), np.float64), self._dev(np.concatenate(P), np.float64)
        else:
            raise TypeError("unsupported estimator type %s (supported: MLPClassifier, RandomForestClassifier, LogisticRegression, GaussianNB)" % tn)
