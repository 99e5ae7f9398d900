"""Stage-level GPU tests through the C ABI: tokeniser records vs a Python split of the same bytes, device generator vs
the numpy generator, classifiers vs the oracle / scikit-learn, histogram vs the oracle's aggregation, and a larger
device-generated workload checked against the CPU oracle plus size-independent properties."""
import ctypes as C
import os

import numpy as np
import pytest

import golden_cases as gc

pytestmark = pytest.mark.gpu


def _setup(case_name, tmp_path, k=6):
    import torch
    from mcaller_b200 import engine, models, read_qual, refmark
    from mcaller_b200.refindex import ReferenceIndex
    case = gc.CASES[case_name]
    inp = gc.build_inputs(case, str(tmp_path))
    seqs = refmark.read_fasta(inp["fasta"])
    base = case.get("base", "A")
    ref = ReferenceIndex(seqs, base, motif=case.get("motif"), positions_file=inp.get("positions"), k=k)
    model = models.load_model_file(inp["model"])
    e0, e1, two = models.select_models(model, base)
    dm = models.DeviceModels(e0, e1)
    qt = read_qual.build_quality_table(read_qual.extract_read_quality(inp["fastq"]))
    return case, inp, ref, dm, two, qt


def test_scan_records_match_python_split(tmp_path, cuda_lib):
    """Dense mode: one record per kept line, every parsed field equal to what Python's split/int/float give."""
    from mcaller_b200 import engine
    case, inp, ref, dm, two, qt = _setup("adversarial", tmp_path)
    data = open(inp["tsv"], "rb").read()
    eng = engine.Engine(ref, models=dm, qual_table=qt, skip_thresh=1, two_models=two, dense=True)
    res = eng.run_chunk(eng.upload(data), len(data))
    rec = eng.records(res.n_records)
    want = []
    off = 0
    n_lines = n_short = n_unknown = n_nnn = 0
    for ln in data.split(b"\n")[:-1]:
        n_lines += 1
        f = ln.split()
        if len(f) < 12:
            n_short += 1
        elif f[0].decode() not in ref.names:
            n_unknown += 1
        elif f[9] == b"NNNNNN":
            n_nnn += 1
        else:
            d = float(np.round(float(f[6]) - float(f[10]), 4))
            want.append((off, int(f[1]), int(f[5]), d, f[2] == f[9], ref.names.index(f[0].decode()), f[3], ln.find(f[3])))
        off += len(ln) + 1
    assert res.counters["lines"] == n_lines and res.counters["short"] == n_short
    assert res.counters["unknown_contig"] == n_unknown and res.counters["nnn"] == n_nnn
    assert res.counters["kept"] == len(want) == res.n_records
    for r, w in zip(rec, want):
        line = int(r["line_lo"]) | (int(r["line_hi"]) << 32)
        assert (line, int(r["pos"]), int(r["event_idx"]), float(r["diff"]), bool(r["flags"] & 1), int(r["contig"])) == w[:6]
        assert data[line + int(r["name_off"]):line + int(r["name_off"]) + int(r["name_len"])] == w[6] and int(r["name_off"]) == w[7]
        assert not (r["flags"] & 12)


def test_record_values_of_odd_number_shapes(cuda_lib):
    """k_finish_records parses the usual shapes ("1234", "87.41", 6-mers) from 8-byte register loads and everything else
    with byte loops: event index, np.round(float(ev) - float(model), 4) and the k-mer equality flag must equal Python's
    for mixed shapes (no fraction, 1-5 fraction digits, signs, leading zeros, wide integers, long k-mer tokens)."""
    import random
    from mcaller_b200 import engine, synth
    from mcaller_b200.refindex import ReferenceIndex
    spec = synth.SynthSpec(seed=71, contigs=[("ctg", 8000)], n_reads=12, len_min=200, len_max=500)
    tsv, fasta, fastq, quals = synth.generate(spec)
    rnd = random.Random(4)

    def reshape(x):
        v = float(x)
        u = rnd.random()
        if u < 0.5:
            return x
        return rnd.choice(["%d" % int(v), "%.1f" % v, "%.3f" % v, "%.5f" % v, "+%.2f" % v, "0%.2f" % v, "%.2f" % (v + 1000.0), "%d." % int(v)])

    out = []
    for ln in tsv.decode().split("\n"):
        f = ln.split("\t")
        if len(f) >= 13 and f[9] != "NNNNNN":
            f[6], f[10] = reshape(f[6]), reshape(f[10])
            u = rnd.random()
            if u < 0.1:
                f[5] = "+" + f[5]
            elif u < 0.2:
                f[5] = "00" + f[5]
            elif u < 0.25:
                f[5] = "1234" + f[5]
            elif u < 0.3:
                f[5] = "-" + f[5]
            if rnd.random() < 0.1:
                f[2] = f[2] + "ACGT"                       # long tokens: equality decided by the byte loop
                if rnd.random() < 0.5:
                    f[9] = f[2]
        out.append("\t".join(f))
    data = "\n".join(out).encode()
    seqs = {"ctg": synth.genome(spec, 0).tobytes().decode()}
    ref = ReferenceIndex(seqs, "A", motif="GATC", k=6)
    from mcaller_b200 import models, read_qual
    model = models.load_model_file(os.path.join(gc.GOLD, "models", gc.R95))
    dm = models.DeviceModels(model["MH"], model["MG"])
    quals = {k.split("_")[0]: v for k, v in quals.items()}
    eng = engine.Engine(ref, models=dm, qual_table=read_qual.build_quality_table(quals), skip_thresh=1, two_models=True, dense=True)
    res = eng.run_chunk(eng.upload(data), len(data))
    rec = eng.records(res.n_records)
    want = []
    for ln in data.split(b"\n"):
        f = ln.split()
        if len(f) >= 12 and f[9] != b"NNNNNN":
            want.append((int(f[5]), float(np.round(float(f[6]) - float(f[10]), 4)), f[2] == f[9]))
    assert len(want) == res.n_records > 3000
    for r, w in zip(rec, want):
        assert (int(r["event_idx"]), float(r["diff"]), bool(r["flags"] & 1)) == w
        assert not (r["flags"] & 12)


def test_sparse_records_are_subset_with_same_calls(tmp_path, cuda_lib):
    """Sparse mode (candidates + closers only) must give exactly the rows of dense mode."""
    from mcaller_b200 import engine
    case, inp, ref, dm, two, qt = _setup("gatc_s1", tmp_path)
    data = open(inp["tsv"], "rb").read()
    outs = []
    for dense in (False, True):
        eng = engine.Engine(ref, models=dm, qual_table=qt, skip_thresh=1, two_models=two, dense=dense)
        res = eng.run_chunk(eng.upload(data), len(data))
        c = res.calls()
        outs.append((res.n_records, c[["mpos", "kind", "rev", "n_empty", "label"]].tolist(), c["feat"].tolist(), c["prob"].tolist()))
    assert outs[0][0] < outs[1][0] * 0.5
    assert outs[0][1:] == outs[1][1:]


def test_device_generator_matches_numpy_generator(cuda_lib):
    import torch
    from mcaller_b200 import synth, synth_device
    from mcaller_b200.refindex import ReferenceIndex
    spec = synth.SynthSpec(seed=5, contigs=[("zeta", 9000), ("alpha", 7000)], n_reads=14, len_min=150, len_max=600)
    seqs = {nm: synth.genome(spec, ci).tobytes().decode() for ci, (nm, _) in enumerate(spec.contigs)}
    ref = ReferenceIndex(seqs, "A", motif="GATC", k=6)
    meth = {}
    for ci, (nm, ln) in enumerate(spec.contigs):
        b0 = int(ref.contig_base[ref.names.index(nm)])
        meth[ci] = (synth.meth_sites(spec, ci, ref.site_fwd_bits[b0:b0 + ln]), synth.meth_sites(spec, ci, ref.site_rev_bits[b0:b0 + ln]))
    gen = synth_device.DeviceSynth(spec, ref, meth)
    d_text, n, offs = gen.generate(0, spec.n_reads)
    dev_bytes = d_text[:n].cpu().numpy().tobytes()
    host_bytes, _, _, _ = synth.generate(spec, meth)
    assert dev_bytes == host_bytes
    assert bytes(d_text[n:n + 64].cpu().numpy()) == b"\n" * 64
    g = gen.genome_check().cpu().numpy()
    for ci, (nm, ln) in enumerate(spec.contigs):
        b0 = int(ref.contig_base[ref.names.index(nm)])
        assert g[b0:b0 + ln].tobytes().decode() == seqs[nm]
    # a slice in the middle equals the corresponding slice of the whole
    d2, n2, _ = gen.generate(3, 5)
    o = offs.cpu().numpy()
    assert d2[:n2].cpu().numpy().tobytes() == host_bytes[int(o[3]):int(o[8])]


def _Xw(n, d, seed):
    """n feature rows of width d: column means around 0, then a read quality (as test_oracle_numerics._X for d = 7)."""
    rng = np.random.default_rng(seed)
    X = rng.normal(0, 3, (n, d))
    X[:, d - 1] = rng.uniform(3, 20, n)
    return X


def _y(X, seed):
    rng = np.random.default_rng(seed)
    z = X[:, 0] - 0.5 * X[:, min(1, X.shape[1] - 1)] + rng.normal(0, 1.5, len(X))
    return np.where(z > np.median(z), "m6A", "A")


def _mlp(n_in, hidden, act, seed):
    """A seeded MLPClassifier of the given shape; a few iterations: the shape matters, not the fit."""
    import warnings
    from sklearn.neural_network import MLPClassifier
    X = _Xw(400, n_in, 50 + seed)
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        return MLPClassifier(hidden_layer_sizes=hidden, activation=act, max_iter=4, random_state=seed).fit(X, _y(X, seed))


def _rf(seed, n=3000, d=7, **kw):
    from sklearn.ensemble import RandomForestClassifier
    X = _Xw(n, d, 70 + seed)
    return RandomForestClassifier(random_state=seed, **kw).fit(X, _y(X, seed))


def _rf_nodes(leaves):
    """One tree grown to exactly `leaves` leaves (2 * leaves - 1 nodes) on label noise."""
    from sklearn.ensemble import RandomForestClassifier
    rng = np.random.default_rng(leaves)
    X = rng.normal(size=(4 * leaves, 7))
    rf = RandomForestClassifier(n_estimators=1, bootstrap=False, max_leaf_nodes=leaves, random_state=0).fit(X, rng.integers(0, 2, len(X)))
    assert rf.estimators_[0].tree_.node_count == 2 * leaves - 1
    return rf


def _mlp_branch(est0, est1, alias=False):
    """Which MLP kernel mc_classify launches (the dispatch rule of classify.cu, restated): '1hidden' (k_mlp_1hidden),
    'staged' (k_mlp<true>) or 'global' (k_mlp<false>)."""
    def sizes(e):
        return [e.coefs_[0].shape[0]] + [c.shape[1] for c in e.coefs_]

    def params(e):
        s = sizes(e)
        return sum(s[i] * s[i + 1] + s[i + 1] for i in range(len(s) - 1))

    def one_hidden(e):
        return len(e.coefs_) == 2 and sizes(e)[0] <= 9

    width = max([8] + sizes(est0) + sizes(est1))
    width = (width + 3) & ~3
    weight_bytes = 8 * (params(est0) + (0 if alias else params(est1)))
    if one_hidden(est0) and (alias or one_hidden(est1)) and weight_bytes <= 100 * 1024:
        return "1hidden"
    if 8 * 2 * width * 8 + weight_bytes <= 100 * 1024:
        return "staged"
    return "global"


def _classifier_case(name):
    """(est0 ('MH'), est1 ('MG'), input width, alias) of a classifier-matrix case."""
    from mcaller_b200 import models
    from test_oracle_numerics import _fit_alt
    from sklearn.linear_model import LogisticRegression
    from sklearn.naive_bayes import GaussianNB
    if name == "NN":
        m = models.load_model_file(os.path.join(gc.GOLD, "models", gc.R95))
        return m["MH"], m["MG"], 7, False
    if name in ("RF", "LR", "NBC"):
        e = _fit_alt(name)
        return e, e, 7, False
    f = name.split(":")
    if f[0] == "1h":                               # 1h:<n_in>:<H>:<act>
        n_in, H, act = int(f[1]), int(f[2]), f[3]
        return _mlp(n_in, (H,), act, 1), _mlp(n_in, (H,), act, 2), n_in, False
    if f[0] == "1h_alias":                         # one estimator for both keys, given once (model 1 aliases model 0)
        e = _mlp(7, (100,), "tanh", 3)
        return e, e, 7, True
    if f[0] == "1h_same":                          # one estimator for both keys, exported twice
        e = _mlp(7, (100,), "tanh", 3)
        return e, e, 7, False
    if name == "staged_64_32_relu":
        return _mlp(7, (64, 32), "relu", 4), _mlp(7, (64, 32), "relu", 5), 7, False
    if name == "staged_16_7_3_logistic":
        return _mlp(7, (16, 7, 3), "logistic", 6), _mlp(7, (16, 7, 3), "logistic", 7), 7, False
    if name == "staged_1h_with_2h":
        return _mlp(7, (100,), "tanh", 8), _mlp(7, (40, 20), "tanh", 9), 7, False
    if name.startswith("global_300_200_"):
        act = name.rsplit("_", 1)[1]
        return _mlp(7, (300, 200), act, 10), _mlp(7, (300, 200), act, 11), 7, False
    if name == "RF_leaf":                          # every tree is a single leaf
        e = _rf(1, n=200, n_estimators=4, min_samples_split=1000)
        return e, e, 7, False
    if name == "RF_sizes":                         # forests of different tree counts and node counts per key
        return _rf(2, n_estimators=3, max_depth=4), _rf(3, n_estimators=7, max_depth=14), 7, False
    if name == "RF_wide":
        return _rf(4, d=9, n_estimators=5, max_depth=10), _rf(5, d=9, n_estimators=2), 9, False
    if name == "RF_7313_nodes":                    # largest tree just under the shared-memory staging limit (7 314 nodes)
        return _rf_nodes(3657), _rf_nodes(3657), 7, False
    if name == "LR_wide":
        X = _Xw(500, 3, 1)
        return LogisticRegression().fit(X, _y(X, 1)), LogisticRegression(C=0.1).fit(X, _y(X, 2)), 3, False
    if name == "NBC_tiny_smoothing":
        X = _Xw(500, 9, 2)
        return GaussianNB(var_smoothing=1e-15).fit(X, _y(X, 3)), GaussianNB().fit(X, _y(X, 4)), 9, False
    raise KeyError(name)


_MLP_1H = ["1h:%d:%d:%s" % (n_in, H, act) for n_in in (1, 5, 9) for H in (1, 3, 17, 100, 129, 512)
           for act in ("identity", "logistic", "tanh", "relu") if act == "tanh" or H in (3, 129)]
_MLP_OTHER = ["1h_alias", "1h_same", "staged_64_32_relu", "staged_16_7_3_logistic", "staged_1h_with_2h", "global_300_200_identity",
              "global_300_200_relu"]
_OTHER = ["RF_leaf", "RF_sizes", "RF_wide", "RF_7313_nodes", "LR_wide", "NBC_tiny_smoothing"]
_TOL = {"NBC": 1e-10}
_CLASSIFIER_CASES = ([pytest.param(k, t, None, id="%s-%s" % (k, t)) for k, t in [("RF", 1e-12), ("LR", 1e-12), ("NBC", 1e-10), ("NN", 1e-12)]]
                     + [pytest.param(k, _TOL.get(k[:3], 1e-12), None, id=k) for k in _MLP_1H + _MLP_OTHER + _OTHER]
                     + [pytest.param(k, _TOL.get(k, 1e-12), n, id="%s-rows%d" % (k, n))
                        for k in ("NN", "staged_16_7_3_logistic", "global_300_200_relu", "RF", "LR", "NBC") for n in (0, 1, 33, 200000)])


def test_classifier_matrix_reaches_every_mlp_kernel():
    """The parametrization of test_classifiers_match_sklearn reaches each of the three MLP kernels, so a later change to
    the dispatch rule cannot silently drop one from the tests."""
    seen = {}
    for name in _MLP_1H + _MLP_OTHER + ["NN"]:
        e0, e1, _, alias = _classifier_case(name)
        seen.setdefault(_mlp_branch(e0, e1, alias), []).append(name)
    assert set(seen) == {"1hidden", "staged", "global"}
    assert seen["staged"] == ["staged_64_32_relu", "staged_16_7_3_logistic", "staged_1h_with_2h"]
    assert seen["global"] == ["global_300_200_identity", "global_300_200_relu"]


def _run_classify(cuda_lib, model_array, calls, n_live):
    import torch
    from mcaller_b200 import _lib
    d = torch.from_numpy(calls.view(np.uint8).reshape(-1).copy()).cuda()
    d_n = torch.tensor([n_live], dtype=torch.int64, device="cuda")
    d_ws = torch.zeros(int(cuda_lib.mc_classify_workspace_bytes(len(calls))), dtype=torch.uint8, device="cuda")
    rc = cuda_lib.mc_classify(C.c_void_p(d.data_ptr()), C.c_void_p(d_n.data_ptr()), len(calls), model_array, C.c_void_p(d_ws.data_ptr()),
                              C.c_void_p(torch.cuda.current_stream().cuda_stream))
    return rc, d.cpu().numpy().view(_lib.CALL_DTYPE)


@pytest.mark.parametrize("kind,tol,rows", _CLASSIFIER_CASES)
def test_classifiers_match_sklearn(kind, tol, rows, cuda_lib, oracle):
    """mc_classify on synthetic feature rows vs scikit-learn predict_proba and the oracle's restatement (float64 on all
    sides): every MLP kernel (the shipped shape, other input widths, hidden widths and activations, deeper and wider
    nets), RF at its float32 split edges, single-leaf trees, forests of different sizes and the largest tree that fits the
    shared-memory staging, LR and GaussianNB where p saturates to exactly 0 and 1.  Rows of another kind (every 50th),
    rows beyond the device-side count and feature slots beyond the model's width (NaN here) must not be touched or read."""
    import warnings
    from mcaller_b200 import _lib, models
    est0, est1, n_in, alias = _classifier_case(kind)
    dm = models.DeviceModels(est0, est1, n_in=n_in)
    if alias:
        dm.array[1] = dm.array[0]                 # model 1 is model 0: its weights are staged once
        assert _mlp_branch(est0, est1, alias=True) == "1hidden"
    n_live = 777 - 20 if rows is None else rows
    X = _Xw(n_live + 20, n_in, 13)
    sel = np.arange(len(X)) % 2
    special = []                                  # (model selector, feature row) placed from row 1 on
    if kind.startswith("RF"):
        # features exactly at float32(threshold), one float32 ulp either side, and the float64 neighbours of the threshold
        # (which may round to float32 on either side of it), each evaluated by the forest the threshold belongs to
        for m, e in enumerate((est0, est1)):
            tr = e.estimators_[0].tree_
            for f, t in [(int(f), float(t)) for f, t in zip(tr.feature, tr.threshold) if f >= 0][:30]:
                t32 = np.float32(t)
                for v in (t32, np.nextafter(t32, np.float32(-np.inf)), np.nextafter(t32, np.float32(np.inf)), t, np.nextafter(t, -np.inf),
                          np.nextafter(t, np.inf)):
                    r = X[(len(special) + 1) % len(X)].copy()
                    r[f] = float(v)
                    special.append((m, r))
    if kind.startswith(("LR", "NBC")):
        # far out along each axis and the diagonal, both signs: p saturates to exactly 0 and exactly 1
        for m in (0, 1):
            for j in range(n_in + 1):
                for sgn in (-1e3, 1e3):
                    r = np.full(n_in, sgn) if j == n_in else np.zeros(n_in)
                    if j < n_in:
                        r[j] = sgn
                    special.append((m, r))
    all_special = len(special) < n_live       # room for every special row among the live ones (row 0 stays plain)
    special = special[:max(0, n_live - 1)]
    for r, (m, row) in enumerate(special):
        X[r + 1], sel[r + 1] = row, m
    calls = np.zeros(len(X), dtype=_lib.CALL_DTYPE)
    calls["feat"][:, :n_in] = X
    calls["feat"][:, n_in:] = np.nan
    calls["model_sel"] = sel
    calls["kind"][::50] = 1                       # non-call rows must be left untouched
    # the row count lives on the device; the capacity only sizes the launch: the last 20 rows lie beyond the count
    rc, out = _run_classify(cuda_lib, dm.array, calls, n_live)
    _lib.check(rc)
    assert np.all(out["prob"][n_live:] == 0) and np.all(out["label"][n_live:] == 0)
    calls["kind"][n_live:] = 1
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        w0, w1 = est0.predict_proba(X)[:, 1], est1.predict_proba(X)[:, 1]
    want = np.where(sel == 1, w1, w0)
    live = calls["kind"] == 0
    assert np.max(np.abs(out["prob"][live] - want[live]), initial=0.0) < tol
    assert np.array_equal(out["label"][live], (want[live] >= 0.5).astype(np.uint8))
    assert np.all(out["prob"][~live] == 0) and np.all(out["label"][~live] == 0)
    if kind.startswith(("LR", "NBC")) and all_special:
        assert {0.0, 1.0} <= set(want[live].tolist())
    # the oracle's restatement of predict_proba, on all rows (a fixed sample of them for the largest count)
    idx = np.flatnonzero(live)
    if len(idx) > 3000:
        idx = np.concatenate([idx[:1000], np.random.default_rng(0).choice(idx[1000:], 1000, replace=False)])
    for m, est in ((0, est0), (1, est1)):
        j = idx[sel[idx] == m]
        if len(j):
            assert np.max(np.abs(out["prob"][j] - oracle.predict(est, X[j]))) < tol


def test_rf_tree_over_the_shared_memory_limit_is_refused(cuda_lib):
    """A tree of 7 315 nodes does not fit the 200 KB shared-memory staging of k_rf: mc_classify refuses it on the host
    (MC_EINVAL, McallerCudaError) and launches nothing."""
    from mcaller_b200 import _lib, models
    e = _rf_nodes(3658)
    dm = models.DeviceModels(e, e, n_in=7)
    calls = np.zeros(64, dtype=_lib.CALL_DTYPE)
    calls["feat"][:, :7] = _Xw(64, 7, 1)
    rc, out = _run_classify(cuda_lib, dm.array, calls, 64)
    assert rc == -1                                # MC_EINVAL
    with pytest.raises(_lib.McallerCudaError, match="RF tree too large"):
        _lib.check(rc)
    assert np.all(out["prob"] == 0) and np.all(out["label"] == 0)


def _kind_est(kind):
    from test_oracle_numerics import _fit_alt
    if kind == "MLP":
        return _mlp(7, (10,), "tanh", 1)
    if kind == "RF":
        return _rf(1, n=300, n_estimators=2, max_depth=3)
    return _fit_alt(kind)


_KINDS = ["MLP", "RF", "LR", "NBC"]


@pytest.mark.parametrize("k0,k1", [(a, b) for a in _KINDS for b in _KINDS if a != b])
def test_mixed_estimator_types_are_refused_on_the_host(k0, k1, cuda_lib):
    """One classifier kernel serves both keys, so a dict whose 'MH' and 'MG' estimators differ in type is refused:
    DeviceModels raises TypeError naming both before exporting anything, and mc_classify given such a pair (built by
    hand) returns MC_EINVAL.  The device-side row count is 0, so no kernel could touch a row even without the check."""
    from mcaller_b200 import _lib, models
    e0, e1 = _kind_est(k0), _kind_est(k1)
    with pytest.raises(TypeError, match="'MH' is %s, 'MG' is %s" % (type(e0).__name__, type(e1).__name__)):
        models.DeviceModels(e0, e1)
    d0, d1 = models.DeviceModels(e0), models.DeviceModels(e1)
    arr = (_lib.Model * 2)()
    arr[0], arr[1] = d0.array[0], d1.array[0]
    calls = np.zeros(64, dtype=_lib.CALL_DTYPE)
    calls["model_sel"] = np.arange(64) % 2
    rc, out = _run_classify(cuda_lib, arr, calls, 0)
    assert rc == -1                                # MC_EINVAL
    assert "different kinds" in cuda_lib.mc_last_error().decode()
    assert np.all(out["prob"] == 0)


def test_histogram_matches_oracle_aggregation(tmp_path, cuda_lib, oracle):
    """Device histogram (stage 7) == make_bed counts computed by the oracle from the rows of the same run."""
    import json
    from mcaller_b200 import engine
    case, inp, ref, dm, two, qt = _setup("gatc_s2", tmp_path)
    data = open(inp["tsv"], "rb").read()
    eng = engine.Engine(ref, models=dm, qual_table=qt, skip_thresh=2, two_models=two)
    res = eng.run_chunk(eng.upload(data), len(data))
    depth, meth, first = eng.histogram_host()
    gold = json.load(open(os.path.join(gc.GOLD, "gatc_s2.json")))
    rows = oracle.aggregate(gold["diffs"], 1, 0.0, False)
    want = {}
    for r in rows:
        f = r.split("\t")
        want[(f[0], int(f[1]), f[5])] = (int(f[6]), float(f[4]))
    got = {}
    order = np.argsort(first, kind="stable")
    seen = []
    for s in order:
        if depth[s]:
            key = (ref.names[ref.site_contig[s]], int(ref.site_pos[s]), "-" if ref.site_rev[s] else "+")
            got[key] = (int(depth[s]), meth[s] / depth[s])
            seen.append(key)
    assert got == want
    assert seen == [(r.split("\t")[0], int(r.split("\t")[1]), r.split("\t")[5]) for r in rows]     # first-seen order
    assert int(depth.sum()) == eng.count_rows(res)["calls"]


def test_device_workload_against_oracle_and_properties(cuda_lib, oracle):
    """~120 MB of device-generated TSV: CUDA rows == oracle rows (keys exact, features and probabilities bit-equal), the
    same workload streamed in chunks through pinned host memory gives the same totals, and histogram mass == calls."""
    import torch
    from mcaller_b200 import engine, models, read_qual, stream, synth, synth_device
    from mcaller_b200.refindex import ReferenceIndex
    spec = synth.SynthSpec(seed=9, contigs=[("ecoli", 400000)], n_reads=260, len_min=500, len_max=1500)
    seqs = {"ecoli": synth.genome(spec, 0).tobytes().decode()}
    ref = ReferenceIndex(seqs, "A", motif="GATC", k=6)
    meth = {0: (synth.meth_sites(spec, 0, ref.site_fwd_bits[:400000]), synth.meth_sites(spec, 0, ref.site_rev_bits[:400000]))}
    gen = synth_device.DeviceSynth(spec, ref, meth)
    d_text, n, offs = gen.generate(0, spec.n_reads)
    keys, q = synth_device.quality_table_for(spec)
    quals = dict(zip(keys, q.tolist()))
    model = models.load_model_file(os.path.join(gc.GOLD, "models", gc.R95))
    dm = models.DeviceModels(model["MH"], model["MG"])
    eng = engine.Engine(ref, models=dm, qual_table=read_qual.build_quality_table(quals), skip_thresh=1, two_models=True)
    res = eng.run_chunk(d_text, n)
    calls = res.calls()
    host = d_text[:n].cpu().numpy().tobytes()
    want = oracle.extract(host, seqs, quals, k=6, skip_thresh=1, model=model, base="A", motif="GATC", cap=200000)
    mine = calls[(calls["kind"] == 0) & (calls["close_rec"] != 0xFFFFFFFF)]
    assert len(mine) == len(want["calls"]) > 500
    for c, w in zip(mine, want["calls"]):
        assert int(c["mpos"]) == w["mpos"] and bool(c["rev"]) == w["rev"] and int(c["empty_mask"]) == w["empty_mask"]
        assert host[int(c["read_off"]):int(c["read_off"]) + int(c["read_len"])].decode() == w["read"]
        assert [float(x) for x in c["feat"][:7]] == w["feat"]                 # bit-equal float64 features
        assert abs(float(c["prob"]) - w["prob"]) < 1e-12 and int(c["label"]) == w["label"]
    st = eng.count_rows(res)
    assert st["calls"] == len(mine) and st["errors"] == 0
    depth, meth_whole, first_whole = [a.copy() for a in eng.histogram_host()]
    assert int(depth.sum()) == st["calls"]
    assert st["too_many_skips"] == want["counters"]["too_many_skips"]
    # the same bytes streamed from pinned host memory in read-aligned chunks
    eng.reset_histogram()
    hbuf = torch.empty(n, dtype=torch.uint8, pin_memory=True)
    hbuf.copy_(d_text[:n])
    torch.cuda.synchronize()
    hs = stream.HostStreamer(eng, chunk_bytes=8 << 20)
    cuts = stream.plan_chunks(offs.cpu().numpy(), n, hs.chunk_bytes)
    assert len(cuts) > 5
    tot = hs.run(hbuf, cuts)
    assert tot["calls"] == st["calls"] and tot["too_many_skips"] == st["too_many_skips"]
    d2, m2, f2 = eng.histogram_host()
    # windows open at a chunk edge are carried on the device and land in the histogram like any other row: exact
    assert int(d2.sum()) == tot["calls"]
    assert (d2 == depth).all() and (m2 == meth_whole).all()
    assert (np.argsort(f2, kind="stable") == np.argsort(first_whole, kind="stable")).all()      # same first-seen order


def _rename_reads(tsv, quals, style, seed):
    """Rewrite read names (column 4) to stress line layouts: 'short' -> ~70-byte lines (more than 32 lines per
    chunk: multi-pass), 'long' -> 420-byte names (first 12 columns outrun the look-ahead: global-memory slow path),
    'mixed' -> both plus normal names."""
    import random
    rnd = random.Random(seed)
    mapping, new_quals, out = {}, {}, []
    for ln in tsv.decode().split("\n"):
        f = ln.split("\t")
        if len(f) < 13:
            out.append(ln)
            continue
        old = f[3]
        if old not in mapping:
            kind = style if style != "mixed" else rnd.choice(["short", "long", "normal", "wide"])
            i = len(mapping)
            if kind == "short":
                nm = "r%d" % i
            elif kind == "long":
                nm = "L%d-" % i + "x" * 420
            elif kind == "wide":
                nm = "W%d-" % i + "y" * 170          # columns 10/12 beyond the 160-byte window, inside the look-ahead
            else:
                nm = old
            mapping[old] = nm
            new_quals[nm.split(":")[0].split("_")[0]] = quals[old.split(":")[0].split("_")[0]]
        f[3] = mapping[old]
        out.append("\t".join(f))
    return "\n".join(out).encode(), new_quals


@pytest.mark.parametrize("style", ["short", "long", "mixed"])
def test_odd_line_layouts_match_oracle(style, cuda_lib, oracle):
    from mcaller_b200 import engine, models, read_qual, synth
    from mcaller_b200.refindex import ReferenceIndex
    spec = synth.SynthSpec(seed=31, contigs=[("a_rather_long_contig_name|quiver", 9000), ("b", 7000)], n_reads=40, len_min=200, len_max=700)
    tsv, fasta, fastq, quals = synth.generate(spec)
    quals = {k.split("_")[0]: v for k, v in quals.items()}
    tsv, quals = _rename_reads(tsv, quals, style, 5)
    seqs = {nm: synth.genome(spec, ci).tobytes().decode() for ci, (nm, _) in enumerate(spec.contigs)}
    ref = ReferenceIndex(seqs, "A", motif="GATC", k=6)
    model = models.load_model_file(os.path.join(gc.GOLD, "models", gc.R95))
    dm = models.DeviceModels(model["MH"], model["MG"])
    want = oracle.extract(tsv, seqs, quals, k=6, skip_thresh=1, model=model, base="A", motif="GATC", cap=100000)
    for dense in (False, True):
        eng = engine.Engine(ref, models=dm, qual_table=read_qual.build_quality_table(quals), skip_thresh=1, two_models=True, dense=dense)
        res = eng.run_chunk(eng.upload(tsv), len(tsv))
        assert res.missing_quality == 0
        if style in ("long", "mixed"):
            assert res.counters["longline"] > 0          # the slow path really ran
        calls = res.calls()
        mine = calls[(calls["kind"] == 0) & (calls["close_rec"] != 0xFFFFFFFF)]
        assert len(mine) == len(want["calls"]) > 50
        for c, w in zip(mine, want["calls"]):
            assert int(c["mpos"]) == w["mpos"] and bool(c["rev"]) == w["rev"]
            assert tsv[int(c["read_off"]):int(c["read_off"]) + int(c["read_len"])].decode() == w["read"]
            assert [float(x) for x in c["feat"][:7]] == w["feat"]
            assert abs(float(c["prob"]) - w["prob"]) < 1e-12
        st = eng.count_rows(res)
        assert st["too_many_skips"] == want["counters"]["too_many_skips"] and st["errors"] == 0


def _mutate_layout(tsv, seed):
    """Structure-only mutations of an eventalign TSV (numeric fields and read order stay intact): whitespace runs instead
    of tabs, leading whitespace, CR before LF, truncated lines, extra trailing columns, bursts of tiny lines (more than
    32 lines in a chunk, more than 3 line starts in a lane's 128 bytes), junk lines of an unknown contig up to 9 KB."""
    import random
    rnd = random.Random(seed)
    out = []
    for ln in tsv.decode().split("\n"):
        f = ln.split("\t")
        if len(f) < 13:
            out.append(ln)
            continue
        u = rnd.random()
        if u < 0.03:
            ln = "".join(x + rnd.choice(["\t", " ", "  ", "\t ", " \t\t", "\x0b", "\x1f\t"]) for x in f[:-1]) + f[-1]
        elif u < 0.04:
            ln = rnd.choice([" ", "\t", " \t "]) + ln
        elif u < 0.05:
            ln = ln + "\r"
        elif u < 0.06:
            ln = "\t".join(f[:rnd.randint(1, 11)])
        elif u < 0.07:
            ln = ln + "\t" + ",".join("%.2f" % rnd.uniform(50, 120) for _ in range(rnd.randint(5, 120)))
        elif u < 0.08:
            out.extend(rnd.choice(["", "x", "a\tb", "\t", "q r s"]) for _ in range(rnd.randint(20, 90)))
        elif u < 0.085:
            out.append("\t".join(["junk%d" % rnd.randint(0, 9)] + ["z" * rnd.randint(1, 700) for _ in range(rnd.randint(3, 16))]))
        elif u < 0.09:
            out.append("nosuchcontig\t" + "\t".join(f[1:]))
        out.append(ln)
    return "\n".join(out).encode()


@pytest.mark.parametrize("seed", [1, 2, 3, 4, 5, 6])
def test_layout_fuzz_matches_oracle(seed, cuda_lib, oracle):
    """Randomly mutated line layouts: every row, feature bit and counter equals the CPU oracle's, sparse and dense."""
    from mcaller_b200 import engine, models, read_qual, synth
    from mcaller_b200.refindex import ReferenceIndex
    spec = synth.SynthSpec(seed=100 + seed, contigs=[("ctgA", 12000), ("c", 9000)], n_reads=60, len_min=300, len_max=900)
    tsv, fasta, fastq, quals = synth.generate(spec)
    quals = {k.split("_")[0]: v for k, v in quals.items()}
    tsv = _mutate_layout(tsv, seed)
    seqs = {nm: synth.genome(spec, ci).tobytes().decode() for ci, (nm, _) in enumerate(spec.contigs)}
    ref = ReferenceIndex(seqs, "A", motif="GATC", k=6)
    model = models.load_model_file(os.path.join(gc.GOLD, "models", gc.R95))
    dm = models.DeviceModels(model["MH"], model["MG"])
    s = seed % 3
    want = oracle.extract(tsv, seqs, quals, k=6, skip_thresh=s, model=model, base="A", motif="GATC", cap=100000)
    for dense in (False, True):
        eng = engine.Engine(ref, models=dm, qual_table=read_qual.build_quality_table(quals), skip_thresh=s, two_models=True, dense=dense)
        res = eng.run_chunk(eng.upload(tsv), len(tsv))
        assert res.missing_quality == 0
        calls = res.calls()
        mine = calls[(calls["kind"] == 0) & (calls["close_rec"] != 0xFFFFFFFF)]
        assert len(mine) == len(want["calls"]) > 30
        for c, w in zip(mine, want["calls"]):
            assert int(c["mpos"]) == w["mpos"] and bool(c["rev"]) == w["rev"] and int(c["empty_mask"]) == w["empty_mask"]
            assert tsv[int(c["read_off"]):int(c["read_off"]) + int(c["read_len"])].decode() == w["read"]
            assert [float(x) for x in c["feat"][:7]] == w["feat"]
            assert abs(float(c["prob"]) - w["prob"]) < 1e-12
        st = eng.count_rows(res)
        assert st["too_many_skips"] == want["counters"]["too_many_skips"] and st["errors"] == 0


def _junk_blocks(tsv, seed):
    """Insert blocks of 40-120 lines that are NOT kept (model_kmer NNNNNN, or fewer than 12 columns) but start like any
    other line of the read (known contig, plain position): the line that closes an open window then lies one or more
    3840-byte chunks after the window's last event.  Positions of the junk lines are either the previous line's (often a
    candidate position: full parse) or far from it (usually not a candidate: the quick look passes them)."""
    import random
    rnd = random.Random(seed)
    out = []
    for ln in tsv.decode().split("\n"):
        out.append(ln)
        f = ln.split("\t")
        if len(f) < 13 or rnd.random() > 0.03:
            continue
        far = rnd.random() < 0.7
        for _ in range(rnd.randint(40, 120)):
            pos = int(f[1]) + (rnd.randint(30, 60) if far else 0)
            if rnd.random() < 0.5:
                g = list(f)
                g[1], g[9], g[10], g[11], g[12] = str(pos), "NNNNNN", "0.00", "0.00", "inf"
                out.append("\t".join(g))
            else:
                out.append("\t".join([f[0], str(pos)] + f[2:rnd.randint(3, 11)]))
    return "\n".join(out).encode()


@pytest.mark.parametrize("run_len", [0, 1, 3, 64, 200])
@pytest.mark.parametrize("variant", ["junk", "fuzz", "plain"])
def test_scan_runs_and_quiet_chunks_match_oracle(variant, run_len, cuda_lib, oracle):
    """The sparse scan passes over chunks whose lines all sit on non-candidate positions and carries the 'last kept line'
    state along runs of consecutive chunks (mc_scan_set_run_len forces the run length; small inputs would otherwise use
    runs of one chunk).  Rows, features and counters must equal the oracle's for every run length, also when the closing
    line of a window is several chunks away and when line layouts are mutated."""
    from mcaller_b200 import _lib, engine, models, read_qual, synth
    from mcaller_b200.refindex import ReferenceIndex
    spec = synth.SynthSpec(seed=211, contigs=[("NC_000913.3", 14000), ("c", 9000)], n_reads=50, len_min=300, len_max=900)   # 11- and 1-byte names
    tsv, fasta, fastq, quals = synth.generate(spec)
    quals = {k.split("_")[0]: v for k, v in quals.items()}
    if variant == "junk":
        tsv = _junk_blocks(tsv, 9)
    elif variant == "fuzz":
        tsv = _mutate_layout(tsv, 12)
    seqs = {nm: synth.genome(spec, ci).tobytes().decode() for ci, (nm, _) in enumerate(spec.contigs)}
    ref = ReferenceIndex(seqs, "A", motif="GATC", k=6)
    model = models.load_model_file(os.path.join(gc.GOLD, "models", gc.R95))
    dm = models.DeviceModels(model["MH"], model["MG"])
    want = oracle.extract(tsv, seqs, quals, k=6, skip_thresh=1, model=model, base="A", motif="GATC", cap=100000)
    n_lines = tsv.count(b"\n") + (0 if tsv.endswith(b"\n") else 1)
    L = _lib.lib()
    before = L.mc_scan_set_run_len(run_len)
    try:
        outs = []
        for dense in (False, True):
            eng = engine.Engine(ref, models=dm, qual_table=read_qual.build_quality_table(quals), skip_thresh=1, two_models=True, dense=dense)
            res = eng.run_chunk(eng.upload(tsv), len(tsv))
            assert res.missing_quality == 0 and res.counters["lines"] == n_lines and res.counters["kept"] > 0
            calls = res.calls()
            mine = calls[(calls["kind"] == 0) & (calls["close_rec"] != 0xFFFFFFFF)]
            assert len(mine) == len(want["calls"]) > 30
            for c, w in zip(mine, want["calls"]):
                assert int(c["mpos"]) == w["mpos"] and bool(c["rev"]) == w["rev"] and int(c["empty_mask"]) == w["empty_mask"]
                assert tsv[int(c["read_off"]):int(c["read_off"]) + int(c["read_len"])].decode() == w["read"]
                assert [float(x) for x in c["feat"][:7]] == w["feat"]
                assert abs(float(c["prob"]) - w["prob"]) < 1e-12
            st = eng.count_rows(res)
            assert st["too_many_skips"] == want["counters"]["too_many_skips"] and st["errors"] == 0
            outs.append(res.n_records)
        assert outs[0] < outs[1]                      # sparse mode really recorded fewer lines than dense mode
    finally:
        L.mc_scan_set_run_len(before)


def _lead_junk(tsv, seed):
    """Put 1-60 lines that are NOT kept (NNNNNN, or fewer than 12 columns) in front of the first line of about half of the
    reads, under the read's own name: the read's first KEPT line is then not its first line, and may sit chunks later."""
    import random
    rnd = random.Random(seed)
    out, last = [], None
    for ln in tsv.decode().split("\n"):
        f = ln.split("\t")
        if len(f) >= 13 and f[3] != last:
            last = f[3]
            if rnd.random() < 0.5:
                for _ in range(rnd.randint(1, 60)):
                    if rnd.random() < 0.5:
                        g = list(f)
                        g[9], g[10], g[11], g[12] = "NNNNNN", "0.00", "0.00", "inf"
                        out.append("\t".join(g))
                    else:
                        out.append("\t".join(f[:rnd.randint(4, 11)]))
        out.append(ln)
    return "\n".join(out).encode()


@pytest.mark.parametrize("run_len", [0, 1, 5])
@pytest.mark.parametrize("motif", ["GATCG", "GAT"])
@pytest.mark.parametrize("variant", ["plain", "junk", "lead_junk", "names", "fuzz"])
def test_quality_filter_with_sparse_scan_matches_oracle(variant, motif, run_len, cuda_lib, oracle):
    """-q drops whole reads (extract_contexts.py:167) before the window logic sees their lines, so a window left open at the
    end of a read is closed by the first kept line of the next read that PASSES, and the row takes that line's contig (:179,
    :214).  The scan's read-first mode (mc_scan dense == 2) records the first kept line of every read for this; rows
    (contig column included), features and counters must equal the oracle's with about half of the reads filtered, most
    reads without any site of the rare motif (GATCG) or many windows open at read ends (GAT), reads of three contigs in
    random order, and junk in front of / behind the lines that matter."""
    import random
    from mcaller_b200 import _lib, engine, models, read_qual, synth
    from mcaller_b200.refindex import ReferenceIndex
    spec = synth.SynthSpec(seed=77, contigs=[("NC_000913.3", 9000), ("c", 7000), ("plasmid_pB171_2", 5000)], n_reads=400, len_min=30, len_max=200)
    order = list(range(spec.n_reads))
    random.Random(5).shuffle(order)
    tsv, fasta, fastq, quals = synth.generate(spec, reads=order)
    quals = {k.split("_")[0]: v for k, v in quals.items()}
    if variant == "junk":
        tsv = _junk_blocks(tsv, 4)
    elif variant == "lead_junk":
        tsv = _lead_junk(tsv, 6)
    elif variant == "names":
        tsv, quals = _rename_reads(tsv, quals, "mixed", 8)
    elif variant == "fuzz":
        tsv = _mutate_layout(tsv, 3)
    seqs = {nm: synth.genome(spec, ci).tobytes().decode() for ci, (nm, _) in enumerate(spec.contigs)}
    ref = ReferenceIndex(seqs, "A", motif=motif, k=6)
    model = models.load_model_file(os.path.join(gc.GOLD, "models", gc.R95))
    dm = models.DeviceModels(model["MH"], model["MG"])
    qt = float(np.median(list(quals.values())))
    want = oracle.extract(tsv, seqs, quals, k=6, skip_thresh=1, qual_thresh=qt, model=model, base="A", motif=motif, cap=100000)
    all_rows = oracle.extract(tsv, seqs, quals, k=6, skip_thresh=1, model=model, base="A", motif=motif, cap=100000)
    assert 10 < len(want["calls"]) < len(all_rows["calls"])
    if motif == "GAT":
        assert sum(1 for w in want["calls"] if w["chrom"] != w["win_contig"]) >= 2       # rows closed by a line of another contig
    names = [nm for nm, _ in spec.contigs]
    L = _lib.lib()
    before = L.mc_scan_set_run_len(run_len)
    try:
        outs = []
        for dense in (None, True):
            eng = engine.Engine(ref, models=dm, qual_table=read_qual.build_quality_table(quals), skip_thresh=1, qual_thresh=qt,
                                two_models=True, dense=dense)
            assert eng.scan_mode == (1 if dense else 2)
            res = eng.run_chunk(eng.upload(tsv), len(tsv))
            assert res.missing_quality == 0
            calls = res.calls()
            mine = calls[(calls["kind"] == 0) & (calls["close_rec"] != 0xFFFFFFFF)]
            assert len(mine) == len(want["calls"])
            for c, w in zip(mine, want["calls"]):
                assert names[int(c["chrom_contig"])] == w["chrom"] and names[int(c["win_contig"])] == w["win_contig"]
                assert int(c["mpos"]) == w["mpos"] and bool(c["rev"]) == w["rev"] and int(c["empty_mask"]) == w["empty_mask"]
                assert tsv[int(c["read_off"]):int(c["read_off"]) + int(c["read_len"])].decode() == w["read"]
                assert [float(x) for x in c["feat"][:7]] == w["feat"]
                assert abs(float(c["prob"]) - w["prob"]) < 1e-12
            st = eng.count_rows(res)
            assert st["too_many_skips"] == want["counters"]["too_many_skips"] and st["errors"] == 0
            outs.append(res.n_records)
        # (far) fewer records than one per kept line -- except that names of more than 64 bytes ("names") always count as a
        # new read, so all their kept lines are recorded
        assert outs[0] < outs[1] // (3 if (motif == "GATCG" and variant != "names") else 1)
    finally:
        L.mc_scan_set_run_len(before)


@pytest.mark.parametrize("mode", ["A_dense", "p_one_strand"])
def test_window_units_in_other_site_regimes(mode, tmp_path, cuda_lib, oracle):
    """The window builder cuts reads into units at non-candidate records; GATC gives short units.  Two other regimes against
    the oracle: `-m A` (every fourth position a target: long candidate runs, multi-M carries everywhere, skips allowed) and
    `-p` with targets on one strand per contig (reads of the other strand are all candidates without a single 'M': the
    first-'M' pre-pass finds nothing and every unit is a no-op)."""
    from mcaller_b200 import engine, models, read_qual, synth
    from mcaller_b200.refindex import ReferenceIndex
    one, two = "contig_with_a_31_character_name", "a_contig_name_of_32_characters__"      # longest name the quick look handles, and one more
    spec = synth.SynthSpec(seed=808, contigs=[(one, 15000), (two, 11000)], n_reads=120, len_min=300, len_max=1200)
    tsv, fasta, fastq, quals = synth.generate(spec)
    quals = {k.split("_")[0]: v for k, v in quals.items()}
    seqs = {nm: synth.genome(spec, ci).tobytes().decode() for ci, (nm, _) in enumerate(spec.contigs)}
    model = models.load_model_file(os.path.join(gc.GOLD, "models", gc.R95))
    dm = models.DeviceModels(model["MH"], model["MG"])
    if mode == "A_dense":
        kw_ref, kw_orc, s = dict(motif="A"), dict(motif="A"), 2
    else:
        import random
        rnd = random.Random(5)
        pos_path = os.path.join(str(tmp_path), "pos.txt")
        with open(pos_path, "w") as fh:
            for p, c in enumerate(seqs[one]):
                if c == "A" and 20 < p < len(seqs[one]) - 20 and rnd.random() < 0.03:
                    fh.write("%s\t%d\t+\tm6A\n" % (one, p))
            for p, c in enumerate(seqs[two]):
                if c == "T" and 20 < p < len(seqs[two]) - 20 and rnd.random() < 0.03:
                    fh.write("%s\t%d\t-\tm6A\n" % (two, p))
        kw_ref, kw_orc, s = dict(positions_file=pos_path), dict(positions=pos_path), 1
    ref = ReferenceIndex(seqs, "A", k=6, **kw_ref)
    want = oracle.extract(tsv, seqs, quals, k=6, skip_thresh=s, model=model, base="A", cap=400000, **kw_orc)
    eng = engine.Engine(ref, models=dm, qual_table=read_qual.build_quality_table(quals), skip_thresh=s, two_models=True)
    from mcaller_b200 import _lib
    before = _lib.lib().mc_scan_set_run_len(16)          # small input: force runs so that chunks are passed over
    try:
        res = eng.run_chunk(eng.upload(tsv), len(tsv))
    finally:
        _lib.lib().mc_scan_set_run_len(before)
    calls = res.calls()
    mine = calls[(calls["kind"] == 0) & (calls["close_rec"] != 0xFFFFFFFF)]
    assert len(mine) == len(want["calls"]) > 100
    for c, w in zip(mine, want["calls"]):
        assert int(c["mpos"]) == w["mpos"] and bool(c["rev"]) == w["rev"] and int(c["empty_mask"]) == w["empty_mask"]
        assert tsv[int(c["read_off"]):int(c["read_off"]) + int(c["read_len"])].decode() == w["read"]
        assert [float(x) for x in c["feat"][:7]] == w["feat"]
        assert abs(float(c["prob"]) - w["prob"]) < 1e-12
    st = eng.count_rows(res)
    assert st["too_many_skips"] == want["counters"]["too_many_skips"] and st["multi"] == want["counters"]["multi"] and st["errors"] == 0


def test_streamed_text_rows_match_oracle(tmp_path, cuda_lib, oracle):
    """HostStreamer + TextSink (pinned host TSV -> H2D -> kernels -> rows D2H -> native multi-threaded writer): with one chunk
    the text is the oracle's `.diffs` rows byte for byte, and so it is with several chunks: a window open at a chunk edge is
    carried on the device and written, completed, with the first rows of the next chunk.  The same holds for FileStreamer
    reading the TSV from disk in small chunks through its ring of three pinned buffers (each goes back to the reader only
    after its chunk's rows are rendered)."""
    import torch
    from mcaller_b200 import engine, extract_contexts as ec, models, read_qual, stream, synth
    from mcaller_b200.refindex import ReferenceIndex
    spec = synth.SynthSpec(seed=93, contigs=[("ecoli", 60000)], n_reads=400, len_min=400, len_max=1500)
    tsv, fasta, fastq, quals = synth.generate(spec)
    quals = {k.split("_")[0]: v for k, v in quals.items()}
    seqs = {"ecoli": synth.genome(spec, 0).tobytes().decode()}
    ref = ReferenceIndex(seqs, "A", motif="GATC", k=6)
    model = models.load_model_file(os.path.join(gc.GOLD, "models", gc.R95))
    dm = models.DeviceModels(model["MH"], model["MG"])
    want = oracle.extract(tsv, seqs, quals, k=6, skip_thresh=0, model=model, base="A", motif="GATC", cap=200000)
    want_text = "".join(r + "\n" for r in want["rows"]).encode()
    assert len(want["rows"]) > 1000
    eng = engine.Engine(ref, models=dm, qual_table=read_qual.build_quality_table(quals), skip_thresh=0, two_models=True)
    host = torch.empty(len(tsv), dtype=torch.uint8, pin_memory=True)
    host.copy_(torch.frombuffer(bytearray(tsv), dtype=torch.uint8))
    offs, o = [], 0
    last = None
    for ln in tsv.split(b"\n")[:-1]:
        f = ln.split(b"\t")
        if len(f) > 3 and f[3] != last:
            offs.append(o)
            last = f[3]
        o += len(ln) + 1
    for chunk_bytes in (len(tsv) + 1, len(tsv) // 5):
        hs = stream.HostStreamer(eng, chunk_bytes=chunk_bytes)
        sink = stream.TextSink(ref, 6, "A", keep=True)
        eng.reset_histogram()
        cuts = stream.plan_chunks(offs, len(tsv), hs.chunk_bytes)
        hs.run(host, cuts, sink=sink)
        got = b"".join(sink.kept)
        assert len(cuts) == 1 or len(cuts) >= 4
        assert got == want_text
    path = tmp_path / "syn.eventalign.tsv"
    path.write_bytes(tsv)
    fs = stream.FileStreamer(eng, len(tsv) // 40, ec.read_boundary_before, slots=3)
    sink = stream.TextSink(ref, 6, "A", keep=True)
    eng.reset_histogram()
    tot = fs.run(str(path), 0, len(tsv), render=sink.render)
    assert len(sink.kept) >= 30 and fs.h2d_bytes == len(tsv)
    assert b"".join(sink.kept) == want_text
    assert sink.n_obs == tot["calls"] == len(want["rows"])


def test_fastq_quality_on_device_matches_host(tmp_path, cuda_lib):
    """mc_fastq_index + mc_fastq_quality == read_qual.extract_read_quality (keys, means bit-equal, last duplicate wins)."""
    import gzip, random
    from mcaller_b200 import read_qual
    rnd = random.Random(3)
    recs = []
    for i in range(3000):
        style = i % 4
        rid = ["%08x-aaaa_Basecall_1D_template" % rnd.getrandbits(32), "ch%d:read%d:template" % (i, i), "plain%d" % i,
               "dup_key_%d" % (i % 7)][style]
        n = rnd.randint(1, 400)
        q = "".join(chr(33 + rnd.randint(0, 60)) for _ in range(n))
        recs.append("@%s some description\n%s\n+\n%s\n" % (rid, "A" * n, q))
    text = "".join(recs)
    p = tmp_path / "r.fastq"
    p.write_text(text)
    host = read_qual.extract_read_quality(str(p))
    for path in (str(p), str(tmp_path / "r.fastq.gz")):
        if path.endswith(".gz"):
            with gzip.open(path, "wt") as fh:
                fh.write(text[:-1])          # also: no trailing newline
            host_ref = read_qual.extract_read_quality(path)
        else:
            host_ref = host
        dt = read_qual.extract_read_quality_device(path)
        assert dt.bad_headers == 0 and dt.n_records == 3000
        tab = dt.to_host()
        live = tab[tab["hash"] != 0]
        assert len(live) == len(host_ref)
        want = read_qual.build_quality_table(host_ref)
        w = want[want["hash"] != 0]
        a = {(int(e["hash"]), int(e["check"]), int(e["len"])): float(e["qual"]) for e in live}
        b = {(int(e["hash"]), int(e["check"]), int(e["len"])): float(e["qual"]) for e in w}
        assert a == b


def test_cli_end_to_end_with_device_fastq(tmp_path, capsys, cuda_lib):
    """python -m mcaller_b200.cli mCaller ... (FASTQ scanned on the GPU) then make_bed: byte-identical to the reference."""
    import json
    from mcaller_b200 import cli
    case = gc.CASES["gatc_s1"]
    gold = json.load(open(os.path.join(gc.GOLD, "gatc_s1.json")))
    inp = gc.build_inputs(case, str(tmp_path))
    for threads in ("1", "3"):
        cli.mcaller_main(["-m", "GATC", "-r", inp["fasta"], "-e", inp["tsv"], "-f", inp["fastq"], "-d", inp["model"], "-b", "A", "-s", "1",
                          "-t", threads])
        out = os.path.join(str(tmp_path), "syn.eventalign.diffs.6")
        assert open(out).read() == gold["diffs"]
        os.remove(out)


def test_iupac_motif_with_general_dict_model(tmp_path, cuda_lib, oracle, capsys):
    """BASELINE configs[4] semantics: `-m CAAYNNNNNRTAC` with the shipped {'general'} pickle.  The reference cannot run
    this as written (KeyError); its defined equivalent (SURVEY.md Q9) is `-p` with the IUPAC-expanded positions and the
    bare estimator, which the oracle runs.  Rows must be identical."""
    import random
    from mcaller_b200 import extract_contexts as ec, read_qual, refmark, synth
    spec = synth.SynthSpec(seed=41, contigs=[("m1", 9000), ("m2", 6000)], n_reads=50, len_min=300, len_max=800)
    tsv, fasta, fastq, quals = synth.generate(spec)
    seqs = {nm: synth.genome(spec, ci).tobytes().decode() for ci, (nm, _) in enumerate(spec.contigs)}
    rnd = random.Random(2)
    for nm in seqs:                       # plant motif instances on both strands (the TSV never looks at the FASTA)
        s = list(seqs[nm])
        for _ in range(25):
            p = rnd.randrange(40, len(s) - 40)
            inst = "CAA" + rnd.choice("CT") + "".join(rnd.choice("ACGT") for _ in range(5)) + rnd.choice("AG") + "TAC"
            if rnd.random() < 0.5:
                inst = refmark.revcomp(inst)
            s[p:p + 13] = inst
        seqs[nm] = "".join(s)
    d = str(tmp_path)
    with open(os.path.join(d, "ref.fasta"), "w") as fh:
        for nm, s in seqs.items():
            fh.write(">%s\n%s\n" % (nm, s))
    with open(os.path.join(d, "syn.eventalign.tsv"), "wb") as fh:
        fh.write(tsv)
    with open(os.path.join(d, "syn.fastq"), "w") as fh:
        fh.write(fastq)
    pos_path = os.path.join(d, "pos.txt")
    rc = "GTAYNNNNNRTTG"
    with open(pos_path, "w") as fh:
        for nm, s in seqs.items():
            for p in refmark.expand_iupac_sites(s, "CAAYNNNNNRTAC", "A"):
                fh.write("%s\t%d\t+\tm6A\n" % (nm, p))
            for p in refmark.expand_iupac_sites(s, rc, "T"):
                fh.write("%s\t%d\t-\tm6A\n" % (nm, p))
    q = orc_quals = oracle.read_fastq_quals(os.path.join(d, "syn.fastq"))
    want = oracle.extract(tsv, os.path.join(d, "ref.fasta"), orc_quals, k=6, skip_thresh=1,
                          model=oracle.load_pickle(os.path.join(gc.GOLD, "models", gc.CAAY_BARE)), base="A", positions=pos_path)
    assert len(want["rows"]) > 20
    ec.extract_features(os.path.join(d, "syn.eventalign.tsv"), os.path.join(d, "ref.fasta"), read_qual.extract_read_quality(os.path.join(d, "syn.fastq")),
                        6, 1, 0.0, os.path.join(gc.GOLD, "models", "CAAYNNNNNRTAC_model_6_m6A.pkl"), "NN", 0,
                        endline=len(tsv), base="A", motif="CAAYNNNNNRTAC")
    mine = open(os.path.join(d, "syn.eventalign.diffs.6.tmp0")).read()
    assert mine == "".join(r + "\n" for r in want["rows"])


def test_size_independent_properties_at_scale(cuda_lib):
    """1.5 GB of device-generated TSV (3 000 reads): chunk-invariance (streamed from host in 128 MB read-aligned chunks ==
    one pass), shard-invariance (two read slices with the slice-edge hand-off == one pass, histograms add up), idempotence,
    and conservation (histogram mass == closed calls)."""
    import torch
    from mcaller_b200 import engine, models, read_qual, stream, synth, synth_device
    from mcaller_b200.refindex import ReferenceIndex
    spec = synth.SynthSpec(seed=77, contigs=[("ecoli", 1000000)], n_reads=3000, len_min=1000, len_max=3000)
    seqs = {"ecoli": synth.genome(spec, 0).tobytes().decode()}
    ref = ReferenceIndex(seqs, "A", motif="GATC", k=6)
    gen = synth_device.DeviceSynth(spec, ref, None)
    keys, q = synth_device.quality_table_for(spec)
    model = models.load_model_file(os.path.join(gc.GOLD, "models", gc.R95))
    dm = models.DeviceModels(model["MH"], model["MG"])
    eng = engine.Engine(ref, models=dm, qual_table=read_qual.build_quality_table(dict(zip(keys, q.tolist()))), skip_thresh=1, two_models=True)
    d_text, n, offs = gen.generate(0, spec.n_reads)
    assert n > 1.2e9
    res = eng.run_chunk(d_text, n)
    whole = eng.count_rows(res)
    hist_whole = [a.copy() for a in eng.histogram_host()]
    assert whole["errors"] == 0 and whole["calls"] > 10000
    assert int(hist_whole[0].sum()) == whole["calls"]                            # conservation
    # idempotence
    eng.reset_histogram()
    res2 = eng.run_chunk(d_text, n)
    assert eng.count_rows(res2) == whole and all((a == b).all() for a, b in zip(eng.histogram_host(), hist_whole))
    # chunk-invariance through the host streaming path
    eng.reset_histogram()
    hbuf = torch.empty(n, dtype=torch.uint8, pin_memory=True)
    hbuf.copy_(d_text[:n])
    torch.cuda.synchronize()
    hs = stream.HostStreamer(eng, chunk_bytes=128 << 20)
    tot = hs.run(hbuf, stream.plan_chunks(offs.cpu().numpy(), n, hs.chunk_bytes))
    assert tot["calls"] == whole["calls"] and tot["open_at_end"] == whole["pending"] + whole["pending_too_many_skips"]
    assert tot["too_many_skips"] == whole["too_many_skips"] and tot["multi"] == whole["multi"]
    d_s, m_s, f_s = eng.histogram_host()
    # windows open at a chunk edge are carried on the device: the streamed histogram IS the one-pass histogram
    assert int(d_s.sum()) == whole["calls"]
    assert (d_s == hist_whole[0]).all() and (m_s == hist_whole[1]).all()
    assert (np.argsort(f_s, kind="stable") == np.argsort(hist_whole[2], kind="stable")).all()
    # shard-invariance: two read slices as two ranks would run them (row bases rank << 40), the slice-edge window closed
    # with the second slice's first kept contig (dist.close_and_reduce without the collectives), histograms added
    from mcaller_b200 import dist as mdist
    o = offs.cpu().numpy()
    half = 1500
    cut = int(o[half])
    eng.reset_histogram(mdist.rank_row_base(0))
    a = eng.run_chunk(d_text[:cut + engine.MC_TEXT_PAD + 64].clone().index_fill_(0, torch.arange(cut, cut + engine.MC_TEXT_PAD + 64, device=d_text.device), 10), cut)
    sa = eng.count_rows(a)
    open_a, first_a = eng.carry_state()
    assert open_a == bool(sa["pending"] + sa["pending_too_many_skips"]) and first_a == 0
    eng_b = engine.Engine(ref, models=dm, qual_table=read_qual.build_quality_table(dict(zip(keys, q.tolist()))), skip_thresh=1, two_models=True)
    eng_b.reset_histogram(mdist.rank_row_base(1))
    d_b = torch.full((eng_b.padded_capacity(n - cut),), 10, dtype=torch.uint8, device=d_text.device)
    d_b[: n - cut] = d_text[cut:n]
    b = eng_b.run_chunk(d_b, n - cut)
    sb = eng_b.count_rows(b)
    allk = torch.cat([eng.first_kept_contig_dev(), eng_b.first_kept_contig_dev()])
    row_a = eng.close_carry(next_contigs=allk, start=1)
    row_b = eng_b.close_carry(next_contigs=allk, start=2)
    assert int(row_b[0]["kind"]) == 3                                     # nobody closes the last rank's window
    closed_call = int(row_a[0]["kind"] == 0)
    closed_tms = int(row_a[0]["kind"] == 1)
    assert closed_call == sa["pending"] and closed_tms == sa["pending_too_many_skips"]
    assert sa["calls"] + sb["calls"] + closed_call == whole["calls"]
    assert sa["too_many_skips"] + sb["too_many_skips"] + closed_tms == whole["too_many_skips"]
    d_a, m_a, f_a = eng.histogram_host()
    d_bb, m_bb, f_bb = eng_b.histogram_host()
    assert ((d_a + d_bb) == hist_whole[0]).all() and ((m_a + m_bb) == hist_whole[1]).all()
    f_ab = np.minimum(f_a, f_bb)
    assert (np.argsort(f_ab, kind="stable") == np.argsort(hist_whole[2], kind="stable")).all()


def test_diffs_value_parse_is_exact(tmp_path, cuda_lib):
    """mc_diffs_colstats parses the feature column like Python's float(): bit-exact for <= 19 significant digits and
    decimal exponents in [-27, 0] (everything repr(float64) prints for |x| >= 1e-11), within 1 ulp outside (counted)."""
    import random
    import struct
    from mcaller_b200 import make_bed as mb
    rng = random.Random(11)
    toks = []
    for i in range(36000):
        u = i % 12
        if u == 0:
            x = rng.gauss(0, 3)
        elif u == 1:
            x = rng.gauss(0, 3) * 10 ** rng.randint(-9, 3)
        elif u == 2:
            x = round(rng.gauss(0, 50), rng.randint(0, 6))
        elif u == 3:
            x = struct.unpack("<d", struct.pack("<Q", rng.getrandbits(64) & 0x7FFFFFFFFFFFFFFF))[0]
            x = x if (x == x and 1e-11 <= abs(x) < 1e15) else rng.random()
        elif u == 4:
            x = rng.randint(-10 ** 6, 10 ** 6) / 10 ** rng.randint(0, 8)
        elif u == 5:
            x = float(rng.randint(0, 10 ** 15))
        elif u == 6:
            x = rng.gauss(0, 1) * 1e-5
        else:
            x = rng.uniform(-200, 200)
        t = repr(x)
        if u == 7:
            t = "%.17g" % x
        elif u == 8:
            t = "%.4f" % x
        elif u == 9:
            t = "%.12e" % x
        elif u == 10:
            t = "+" + repr(abs(x))
        elif u == 11:
            t = str(rng.randint(-99999, 99999))
        toks.append(t)
    toks[5], toks[17], toks[29] = "0", "-0.0", "1e-05"
    rows = []
    per = 9
    for r in range(len(toks) // per):
        vals = toks[r * per:(r + 1) * per]
        rows.append("ctg\tread%d\t100\tAAAAAMAAAAA\t%s,9.5\t+\tm6A\t0.7\n" % (r, ",".join(vals)))
    path = os.path.join(str(tmp_path), "v.diffs.6")
    with open(path, "w") as fh:
        fh.write("".join(rows))
    pos = os.path.join(str(tmp_path), "p.txt")
    with open(pos, "w") as fh:
        fh.write("ctg\t100\t101\t+\n")
    agg = mb._Aggregation(path, mb.make_pos_set(pos))
    assert len(agg.loci) == 1 and agg.loci[0][4] == len(rows)
    agg.index_rows()
    agg.column_tests()
    assert agg.counters[6] == 0
    got = agg.vals[:, :per]
    want = np.array([[float(t) for t in toks[r * per:(r + 1) * per]] for r in range(len(rows))])
    exact = got.view(np.uint64) == want.view(np.uint64)
    n_bad = int((~exact).sum())
    assert n_bad <= int(agg.counters[7]), (n_bad, int(agg.counters[7]), [(toks[i], got.ravel()[i], want.ravel()[i]) for i in np.nonzero(~exact.ravel())[0][:5]])
    assert np.allclose(got, want, rtol=3e-16, atol=0)
    assert int(agg.counters[7]) < 0.02 * len(toks)
