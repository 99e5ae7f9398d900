"""Training a model for `mCaller --train` (INTEGRATION.md, "Training"): the labelled `.diffs.<k>.train` rows -> one
estimator per model key, pickled as `{key: estimator}` for the inference path (models.load_model_file / select_models).

Per key: the two labels, the majority class downsampled to the minority count (RandomState(seed), file order kept),
5-fold GroupKFold cross-validation over sites (contig, position, strand) with each fold's held-out accuracy printed, and a
final fit on all balanced rows.  `-c NN` fits scikit-learn 1.9's MLPClassifier(**SHIPPED_NN, random_state=seed) on the
GPU (k_mlp_train, csrc/train.cu): all fits of a run are jobs of one call, and the result is that estimator's `fit` to
rounding.  `-c NBC` fits GaussianNB on the host (closed form).
"""
import concurrent.futures
import os
import warnings

import numpy as np

# the settings of every MLP mCaller ships (tests/golden/models/*NN*.pkl)
SHIPPED_NN = dict(hidden_layer_sizes=100, activation="tanh", solver="adam", alpha=0.001, learning_rate_init=0.001, max_iter=200,
                  tol=1e-4, n_iter_no_change=10, batch_size="auto", shuffle=True)
CV_FOLDS = 5
IDX_BLOCK_BYTES = 256 << 20         # host + device memory for one block of epochs' sample orders (twice, double-buffered)
MAX_BLOCK_EPOCHS = 16


class TrainRows(object):
    """Labelled windows in file order: site keys, features (n x (k+1)), labels and model keys."""

    def __init__(self, sites, x, labels, keys):
        self.sites, self.x, self.labels, self.keys = sites, x, labels, keys


def read_train_tsv(path):
    """Rows of a `.diffs.<k>.train` file (the reference's tsv2matrix): chrom, read, position, context, features, strand,
    label -> (sites, features, labels, contexts)."""
    sites, feats, labels, ctxs = [], [], [], []
    with open(path) as fh:
        for ln in fh:
            f = ln.rstrip("\n").split("\t")
            if len(f) < 7:
                continue
            sites.append((f[0], int(f[2]), f[5]))
            feats.append([float(v) for v in f[4].split(",")])
            labels.append(f[6])
            ctxs.append(f[3])
    if len(set(len(r) for r in feats)) > 1:
        raise ValueError("%s: rows with different feature counts" % path)
    return sites, np.asarray(feats, dtype=np.float64).reshape(len(feats), -1), labels, ctxs


def keys_from_contexts(ctxs, base, k):
    """Model key per row of a `.train` file, from the two letters at the centre of its 2k-1 context -- the reference's
    base_models table (extract_contexts.base_models) the window builder's model_sel follows."""
    from .extract_contexts import base_models
    if base != "A":
        return ["general"] * len(ctxs)
    table = base_models(base, twobase=True)
    return [table[c[k - 1:k + 1]] for c in ctxs]


def balance(labels, seed):
    """Row indices (ascending) with the majority label downsampled to the minority count by RandomState(seed)."""
    labels = np.asarray(labels)
    classes = sorted(set(labels.tolist()))
    idx = [np.flatnonzero(labels == c) for c in classes]
    n_min = min(len(i) for i in idx)
    rs = np.random.RandomState(seed)
    keep = [i if len(i) == n_min else np.sort(rs.choice(i, n_min, replace=False)) for i in idx]
    return np.sort(np.concatenate(keep))


def cv_folds(groups, seed):
    """GroupKFold(5) splits over the given site groups (no site in both train and test); None below 5 sites."""
    from sklearn.model_selection import GroupKFold
    first = {}
    codes = np.asarray([first.setdefault(g, len(first)) for g in groups], dtype=np.int64)
    if len(first) < CV_FOLDS:
        return None
    gkf = GroupKFold(CV_FOLDS, shuffle=True, random_state=seed)
    return list(gkf.split(np.zeros((len(groups), 1)), groups=codes))


def make_mlp(params, classes, n_features, n_iter, loss_curve, best_loss, n_samples, seed, no_improve=0):
    """An sklearn MLPClassifier with the given fitted d-100-1 parameters (W0, W1, c0, c1), set up as its own fit would
    leave it."""
    from sklearn.neural_network import MLPClassifier
    from sklearn.preprocessing import LabelBinarizer
    W0, W1, c0, c1 = params
    est = MLPClassifier(random_state=seed, **SHIPPED_NN)
    est._label_binarizer = LabelBinarizer().fit(np.asarray(classes))
    est.classes_ = est._label_binarizer.classes_
    est.n_features_in_ = int(n_features)
    est.n_outputs_ = 1
    est.n_layers_ = 3
    est.out_activation_ = "logistic"
    est.coefs_ = [np.asarray(W0, dtype=np.float64).reshape(n_features, -1), np.asarray(W1, dtype=np.float64).reshape(-1, 1)]
    est.intercepts_ = [np.asarray(c0, dtype=np.float64).ravel(), np.asarray(c1, dtype=np.float64).ravel()]
    est.n_iter_ = int(n_iter)
    est.t_ = int(n_iter) * int(n_samples)
    est.loss_curve_ = [float(v) for v in loss_curve]
    est.loss_ = est.loss_curve_[-1]
    est.best_loss_ = float(best_loss)
    est._no_improvement_count = int(no_improve)
    est.validation_scores_ = None
    est.best_validation_score_ = None
    return est


def _init_params(rs, d):
    """_initialize / _init_coef of MLPClassifier: Glorot-uniform W0, c0, W1, c1 drawn in that order from rs."""
    h = SHIPPED_NN["hidden_layer_sizes"]
    b0, b1 = np.sqrt(6.0 / (d + h)), np.sqrt(6.0 / (h + 1))
    W0 = rs.uniform(-b0, b0, (d, h))
    c0 = rs.uniform(-b0, b0, h)
    W1 = rs.uniform(-b1, b1, (h, 1))
    c1 = rs.uniform(-b1, b1, 1)
    return W0, W1, c0, c1


class _Orders(object):
    """One job's sample orders: _fit_stochastic's `sample_idx = shuffle(sample_idx, random_state=rs)` per epoch, the
    shuffles composing, mapped to rows of the uploaded feature matrix."""

    def __init__(self, rs, rows):
        self.rs, self.rows = rs, np.asarray(rows, dtype=np.int32)
        self.order = np.arange(len(rows), dtype=np.int32)

    def draw(self, out, epochs):
        n = len(self.rows)
        for e in range(epochs):
            perm = np.arange(n, dtype=np.int32)
            self.rs.shuffle(perm)
            self.order = self.order[perm]
            np.take(self.rows, self.order, out=out[e * n:(e + 1) * n])


def fit_mlp_jobs(x, y, jobs, device="cuda", stats=None):
    """Fit MLPClassifier(**SHIPPED_NN, random_state=seed) on rows `rows` of (x, y) for every job (rows, seed), all in one
    GPU call sequence.  y holds 0/1 (1 = the label that sorts last).  Returns per job (params (W0, W1, c0, c1), n_iter,
    loss_curve, best_loss, no_improvement_count).  `stats`, a dict, receives `draw_s`, the host's time drawing sample
    orders, and `wait_s`, the part of it the GPU sat idle for after finishing a block."""
    import time
    import torch
    from . import _lib, engine
    engine.require_cuda()
    lib = _lib.lib()
    dev = torch.device(device)
    x = np.ascontiguousarray(x, dtype=np.float64)
    n_all, d = x.shape
    if not 1 <= d <= _lib.MC_MAXK + 1:
        raise ValueError("%d features per row; the trainer supports 1..%d" % (d, _lib.MC_MAXK + 1))
    h = SHIPPED_NN["hidden_layer_sizes"]
    npar = d * h + 2 * h + 1
    max_iter = SHIPPED_NN["max_iter"]
    ns = [len(r) for r, _ in jobs]
    if min(ns) < 1:
        raise ValueError("a training job has no rows")
    # epochs per block: as many as IDX_BLOCK_BYTES holds, at most MAX_BLOCK_EPOCHS; the first blocks are 1, 2, 4 ... epochs
    # so the GPU starts after one epoch's shuffles
    cap = int(max(1, min(MAX_BLOCK_EPOCHS, IDX_BLOCK_BYTES // (4 * sum(ns)))))
    offs = np.concatenate([[0], np.cumsum(ns)[:-1]]) * cap
    d_x = torch.from_numpy(x).to(dev)
    d_y = torch.from_numpy(np.ascontiguousarray(y, dtype=np.float64)).to(dev)
    d_w = torch.zeros((len(jobs), 3 * npar), dtype=torch.float64)
    d_loss = torch.zeros((len(jobs), max_iter), dtype=torch.float64, device=dev)
    orders = []
    for j, (rows, seed) in enumerate(jobs):
        rs = np.random.RandomState(seed)
        d_w[j, :npar] = torch.from_numpy(np.concatenate([p.ravel() for p in _init_params(rs, d)]))
        orders.append(_Orders(rs, rows))
    d_w = d_w.to(dev)
    h_idx = [torch.zeros(cap * sum(ns), dtype=torch.int32).pin_memory() for _ in range(2)]
    d_idx = [torch.zeros(cap * sum(ns), dtype=torch.int32, device=dev) for _ in range(2)]
    arr = (_lib.TrainJob * len(jobs))()
    for j, n in enumerate(ns):
        arr[j].d_x, arr[j].d_y = d_x.data_ptr(), d_y.data_ptr()
        arr[j].d_w, arr[j].d_loss_curve = d_w[j].data_ptr(), d_loss[j].data_ptr()
        arr[j].idx_off, arr[j].n, arr[j].d = int(offs[j]), n, d
        arr[j].max_iter, arr[j].n_iter_no_change = max_iter, SHIPPED_NN["n_iter_no_change"]
        arr[j].alpha, arr[j].lr, arr[j].tol = SHIPPED_NN["alpha"], SHIPPED_NN["learning_rate_init"], SHIPPED_NN["tol"]
    d_jobs = torch.frombuffer(bytearray(bytes(arr)), dtype=torch.uint8).to(dev)
    stream = torch.cuda.current_stream(dev).cuda_stream
    _lib.check(lib.mc_mlp_train_init(d_jobs.data_ptr(), len(jobs), stream))

    pool = concurrent.futures.ThreadPoolExecutor(max_workers=max(1, min(len(jobs), os.cpu_count() or 1)))
    driver = concurrent.futures.ThreadPoolExecutor(max_workers=1)        # runs `draw`, which waits on `pool`
    draw_s = wait_s = 0.0

    def draw(buf, epochs, live):
        t0 = time.perf_counter()
        hv = h_idx[buf].numpy()
        list(pool.map(lambda j: orders[j].draw(hv[offs[j]:offs[j] + epochs * ns[j]], epochs), live))
        return time.perf_counter() - t0

    try:
        done, live, blk = 0, list(range(len(jobs))), 0
        epochs = 1
        draw_s += draw(0, epochs, live)
        while live:
            for j in live:
                d_idx[blk % 2][offs[j]:offs[j] + epochs * ns[j]].copy_(h_idx[blk % 2][offs[j]:offs[j] + epochs * ns[j]], non_blocking=True)
            _lib.check(lib.mc_mlp_train_epochs(d_jobs.data_ptr(), len(jobs), d_idx[blk % 2].data_ptr(), epochs, stream))
            done += epochs
            nxt = min(cap, 2 * epochs, max_iter - done)
            fut = driver.submit(draw, (blk + 1) % 2, nxt, live) if nxt > 0 else None
            state = (_lib.TrainJob * len(jobs)).from_buffer_copy(d_jobs.cpu().numpy().tobytes())     # waits for the block
            if fut is not None:
                t0 = time.perf_counter()
                draw_s += fut.result()
                wait_s += time.perf_counter() - t0
            live = [j for j in live if not state[j].stopped]
            epochs, blk = nxt, blk + 1
            if live and nxt <= 0:
                raise RuntimeError("training jobs still running after max_iter epochs")
    finally:
        driver.shutdown(wait=True)
        pool.shutdown(wait=True)
    w = d_w.cpu().numpy()
    curves = d_loss.cpu().numpy()
    if stats is not None:
        stats["draw_s"], stats["wait_s"] = draw_s, wait_s
    out = []
    for j in range(len(jobs)):
        p = w[j, :npar]
        params = (p[:d * h].reshape(d, h).copy(), p[d * h:d * h + h].reshape(h, 1).copy(), p[d * h + h:d * h + 2 * h].copy(),
                  p[d * h + 2 * h:].copy())
        out.append((params, state[j].n_iter, curves[j, :state[j].n_iter].tolist(), state[j].best_loss, state[j].no_improve))
    return out


def _fit_all(classifier, x, y01, jobs, classes):
    """Estimators for jobs [(rows, seed)] on (x, y01): MLPs on the GPU, GaussianNB on the host."""
    if classifier == "NBC":
        from sklearn.naive_bayes import GaussianNB
        lab = np.asarray(classes)[y01.astype(np.int64)]
        return [GaussianNB().fit(x[rows], lab[rows]) for rows, _ in jobs]
    res = fit_mlp_jobs(x, y01, jobs)
    out = []
    for (rows, seed), (params, n_iter, curve, best, noimp) in zip(jobs, res):
        if n_iter == SHIPPED_NN["max_iter"] and noimp <= SHIPPED_NN["n_iter_no_change"]:
            from sklearn.exceptions import ConvergenceWarning
            warnings.warn("Stochastic Optimizer: Maximum iterations (%d) reached and the optimization hasn't converged yet."
                          % n_iter, ConvergenceWarning)
        out.append(make_mlp(params, classes, x.shape[1], n_iter, curve, best, len(rows), seed, noimp))
    return out


def train(rows, classifier, seed, mod_label, required_keys):
    """The training procedure: per key balance, cross-validate, fit; returns {key: estimator}."""
    keys = sorted(set(rows.keys))
    missing = [k for k in required_keys if k not in keys]
    if missing:
        raise ValueError("no labelled windows for model key(s) %s" % ", ".join(missing))
    xs, ys, jobs, plan, classes_of = [], [], [], [], {}
    base_row = 0
    for key in keys:
        sel = np.flatnonzero(np.asarray(rows.keys) == key)
        labels = [rows.labels[i] for i in sel]
        classes = sorted(set(labels))
        if len(classes) != 2:
            raise ValueError("model key %s has label(s) %s; training needs exactly two" % (key, classes))
        if classes[1] != mod_label:
            raise ValueError("model key %s: labels %s; the methylated label %s must sort last" % (key, classes, mod_label))
        keep = sel[balance(labels, seed)]
        x = rows.x[keep]
        y01 = np.asarray([rows.labels[i] == classes[1] for i in keep], dtype=np.float64)
        print("%s: %d windows (%d per label after balancing)" % (key, len(keep), len(keep) // 2))
        folds = cv_folds([rows.sites[i] for i in keep], seed)
        if folds is None:
            print("%s: fewer than %d sites, cross-validation skipped" % (key, CV_FOLDS))
            folds = []
        for f, (tr, te) in enumerate(folds):
            jobs.append((base_row + tr, seed))
            plan.append((key, f, base_row + te))
        jobs.append((base_row + np.arange(len(keep)), seed))
        plan.append((key, None, None))
        classes_of[key] = classes
        xs.append(x)
        ys.append(y01)
        base_row += len(keep)
    x_all, y_all = np.concatenate(xs), np.concatenate(ys)
    # one set of classes per run keeps the fits one call; every key has the same two labels when -b selects one mod
    cls = {tuple(c) for c in classes_of.values()}
    if len(cls) != 1:
        raise ValueError("model keys disagree on the labels: %s" % sorted(cls))
    classes = list(cls.pop())
    ests = _fit_all(classifier, x_all, y_all, jobs, classes)
    model = {}
    for (key, fold, te), est in zip(plan, ests):
        if fold is None:
            model[key] = est
        else:
            acc = float(np.mean(est.predict(x_all[te]) == np.asarray(classes)[y_all[te].astype(np.int64)]))
            print("%s: fold %d held-out accuracy %.4f (%d windows)" % (key, fold + 1, acc, len(te)))
    return model
