"""mCaller --train: the host procedure (balancing, folds, `.train` parsing, the pickled estimator, the CLI's refusals), the C
ABI of the fit kernel, and on the GPU the fit against scikit-learn 1.9's own MLPClassifier.fit and the CLI end to end."""
import ctypes as C
import os
import pickle
import warnings

import numpy as np
import pytest

import golden_cases as gc


def _blobs(n, seed, d=7, noise=1.0):
    rng = np.random.RandomState(seed)
    x = rng.normal(size=(n, d))
    y = (x[:, 0] - 0.5 * x[:, 1] + noise * rng.normal(size=n) > 0).astype(np.float64)
    return x, y


# ---- host (no GPU) --------------------------------------------------------------------------------------------------

def test_balance_is_seeded_and_keeps_file_order():
    from mcaller_b200 import train as tr
    labels = ["A"] * 30 + ["m6A"] * 10 + ["A"] * 20
    a, b, c = tr.balance(labels, 0), tr.balance(labels, 0), tr.balance(labels, 1)
    assert np.array_equal(a, b) and not np.array_equal(a, c)
    assert np.all(np.diff(a) > 0)
    kept = [labels[i] for i in a]
    assert kept.count("A") == kept.count("m6A") == 10
    assert set(range(30, 40)) <= set(a.tolist())


def test_group_kfold_keeps_each_site_in_one_fold():
    from mcaller_b200 import train as tr
    rng = np.random.RandomState(3)
    sites = [("c", int(p), "+-"[int(p) % 2]) for p in rng.randint(0, 40, size=400)]
    folds = tr.cv_folds(sites, 0)
    assert len(folds) == 5
    seen = {}
    for f, (trn, te) in enumerate(folds):
        assert not {sites[i] for i in trn} & {sites[i] for i in te}
        for i in te:
            assert seen.setdefault(sites[i], f) == f
    assert sorted(np.concatenate([te for _, te in folds]).tolist()) == list(range(400))
    assert tr.cv_folds([("c", 1, "+")] * 10 + [("c", 2, "+")] * 10, 0) is None


def test_parse_train_file_gives_the_exported_rows(tmp_path):
    from mcaller_b200 import extract_contexts as ec, train as tr
    rows = [["ctgA", "read1", "120", "ACGTAMTCGAT", "1.5,-0.25,0,3.0,2.5e-05,1.0,9.5", "+", "m6A"],
            ["ctgB", "read2", "7", "GGATCMGATCC", "0,0,1.125,-7.0,0.5,0.1,10.25", "-", "A"]]
    path = str(tmp_path / "x.diffs.6.train")
    ec.writefi(rows, path)
    sites, x, labels, ctxs = tr.read_train_tsv(path)
    assert sites == [("ctgA", 120, "+"), ("ctgB", 7, "-")]
    assert labels == ["m6A", "A"] and ctxs == ["ACGTAMTCGAT", "GGATCMGATCC"]
    assert np.array_equal(x, np.array([[float(v) for v in r[4].split(",")] for r in rows]))
    assert tr.keys_from_contexts(ctxs, "A", 6) == ["MH", "MG"]
    assert tr.keys_from_contexts(ctxs, "C", 6) == ["general", "general"]


def test_sample_orders_compose_like_sklearn_shuffle():
    from sklearn.utils import shuffle
    from mcaller_b200 import train as tr
    rows = np.arange(50, 80)
    o = tr._Orders(np.random.RandomState(4), rows)
    out = np.zeros(3 * len(rows), dtype=np.int32)
    o.draw(out, 3)
    rs, idx = np.random.RandomState(4), np.arange(len(rows))
    for e in range(3):
        idx = shuffle(idx, random_state=rs)
        assert np.array_equal(out[e * len(rows):(e + 1) * len(rows)], rows[idx])


def test_built_estimator_is_a_fitted_mlp_with_the_shipped_settings():
    from scipy.special import expit
    from mcaller_b200 import models, train as tr
    rng = np.random.RandomState(0)
    W0, W1, c0, c1 = rng.normal(size=(7, 100)) * 0.3, rng.normal(size=(100, 1)) * 0.3, rng.normal(size=100) * 0.1, rng.normal(size=1)
    est = tr.make_mlp((W0, W1, c0, c1), ["A", "m6A"], 7, 12, np.linspace(0.7, 0.5, 12), 0.5, 1000, 5)
    x = rng.normal(size=(50, 7))
    p = expit(np.tanh(x @ W0 + c0) @ W1 + c1)[:, 0]
    assert np.allclose(est.predict_proba(x)[:, 1], p, rtol=1e-14, atol=1e-15)
    assert list(est.predict(x)) == ["m6A" if v > 0.5 else "A" for v in p]
    assert est.t_ == 12000 and est.n_iter_ == 12 and list(est.classes_) == ["A", "m6A"] and est.n_features_in_ == 7
    shipped = models.load_model_file(os.path.join(gc.GOLD, "models", "r94_model_NN_6_m6A.pkl"))    # pickled by an older sklearn
    mine = est.get_params()
    assert mine.pop("random_state") == 5
    keys = set(tr.SHIPPED_NN)
    assert {k: mine[k] for k in keys} == tr.SHIPPED_NN
    have = [k for k in keys if hasattr(shipped, k)]               # n_iter_no_change was a fixed 10 before it became a setting
    assert set(keys) - set(have) <= {"n_iter_no_change"} and {k: getattr(shipped, k) for k in have} == {k: mine[k] for k in have}
    assert {k: v for k, v in mine.items() if k not in keys} == {k: v for k, v in est.__class__().get_params().items()
                                                                if k not in keys and k != "random_state"}


@pytest.mark.parametrize("extra,exc", [(["--train", "-c", "RF"], NotImplementedError), (["--train", "-c", "LR"], NotImplementedError),
                                       (["--train", "--plot_training"], NotImplementedError),
                                       (["--train", "--gpus", "2"], NotImplementedError)])
def test_cli_train_refuses_unsupported_options(extra, exc, tmp_path):
    from mcaller_b200 import cli
    with pytest.raises(exc):
        cli.mcaller_main(["-p", "x", "-r", "r.fa", "-e", "x.tsv", "-f", "x.fq"] + extra)


def test_cli_train_needs_labelled_positions(tmp_path, capsys):
    from mcaller_b200 import cli
    with pytest.raises(SystemExit):
        cli.mcaller_main(["--train", "-m", "GATC", "-r", "r.fa", "-e", "x.tsv", "-f", "x.fq"])
    assert "labelled positions" in capsys.readouterr().err
    pos = tmp_path / "p.txt"
    pos.write_text("ctgA\t10\t+\n")
    with pytest.raises(SystemExit):
        cli.mcaller_main(["--train", "-p", str(pos), "-r", "r.fa", "-e", "x.tsv", "-f", "x.fq"])
    assert "no label column" in capsys.readouterr().err


def test_train_entry_points_declared_exported_and_bound():
    from mcaller_b200 import _lib, build
    build.build()
    hdr = open(os.path.join(os.path.dirname(gc.GOLD), "..", "include", "mcaller_b200.h")).read()
    lib = _lib.load()
    for fn in ("mc_mlp_train_init", "mc_mlp_train_epochs"):
        assert ("int %s(" % fn) in hdr and fn in _lib.EXPORTS and hasattr(lib, fn)
    assert lib.mc_sizeof(9) == C.sizeof(_lib.TrainJob) == 104
    assert "#define MC_TRAIN_HIDDEN 100" in hdr and "#define MC_TRAIN_BATCH 200" in hdr


# ---- GPU ------------------------------------------------------------------------------------------------------------

# (seed, rows, input width): the shipped width 7, and 2 and 9 (-n 1 and -n 8), whose fits index every array by d
CASES = [(s, n, 7) for s in (0, 1, 2) for n in (150, 20000, 20001)] + [(1, n, 2) for n in (150, 20001)] + [(2, n, 9) for n in (150, 20001)]


@pytest.fixture(scope="module")
def fits_vs_sklearn(cuda_lib):
    """Per case (CASES, then a noisy 150-row set of width 7 that runs to max_iter): (x, y, rows, seed, fit result).  The
    cases of one width are jobs of one call (rows 0..n of one matrix): fit_mlp_jobs takes one matrix."""
    from mcaller_b200 import train as tr
    out = {}
    for d in sorted({c[2] for c in CASES}):
        x, y = _blobs(20001, 7, d=d)
        idx = [i for i, c in enumerate(CASES) if c[2] == d]
        jobs = [(np.arange(CASES[i][1]), CASES[i][0]) for i in idx]
        if d == 7:
            xm, ym = _blobs(150, 8, noise=3.0)
            x, y = np.concatenate([x, xm]), np.concatenate([y, ym])
            idx.append(len(CASES))
            jobs.append((20001 + np.arange(150), 3))
        for i, job, r in zip(idx, jobs, tr.fit_mlp_jobs(x, y, jobs)):
            out[i] = (x, y, job[0], job[1], r)
    return out


@pytest.mark.gpu
@pytest.mark.parametrize("case", list(range(len(CASES) + 1)))
def test_gpu_fit_matches_sklearn(case, fits_vs_sklearn):
    from sklearn.neural_network import MLPClassifier
    from mcaller_b200 import train as tr
    xa, ya, rows, seed, res = fits_vs_sklearn[case]
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        ref = MLPClassifier(random_state=seed, **tr.SHIPPED_NN).fit(xa[rows], ya[rows])
    params, n_iter, curve, best, noimp = res
    if case == len(CASES):
        assert ref.n_iter_ == tr.SHIPPED_NN["max_iter"]
    assert n_iter == ref.n_iter_
    assert np.allclose(curve, ref.loss_curve_, rtol=1e-10, atol=0)
    W0, W1, c0, c1 = params
    assert W0.shape == (xa.shape[1], 100)
    assert np.max(np.abs(W0 - ref.coefs_[0])) < 1e-9 and np.max(np.abs(W1 - ref.coefs_[1])) < 1e-9
    assert np.max(np.abs(c0 - ref.intercepts_[0])) < 1e-9 and np.max(np.abs(c1 - ref.intercepts_[1])) < 1e-9
    est = tr.make_mlp(params, [0.0, 1.0], xa.shape[1], n_iter, curve, best, len(rows), seed, noimp)
    held, _ = _blobs(500, 99, d=xa.shape[1])
    assert np.allclose(est.predict_proba(held), ref.predict_proba(held), rtol=1e-10, atol=0)
    assert est.best_loss_ == pytest.approx(ref.best_loss_, rel=1e-10) and est.t_ == ref.t_


@pytest.mark.gpu
def test_gpu_fit_is_deterministic_and_independent_of_other_jobs(cuda_lib):
    from mcaller_b200 import train as tr
    x, y = _blobs(3000, 11)
    jobs = [(np.arange(500 + 200 * j), j % 4) for j in range(12)]
    together = tr.fit_mlp_jobs(x, y, jobs)
    for j, job in enumerate(jobs):
        alone = tr.fit_mlp_jobs(x, y, [job])[0]
        assert alone[1] == together[j][1] and alone[2] == together[j][2]
        for a, b in zip(alone[0], together[j][0]):
            assert a.tobytes() == b.tobytes()


def _labelled_set(d, seed, n_reads=500):
    """A seeded synthetic set whose A sites of GATC and TAGC (after-target bases T and G: both model keys) carry the
    methylation signal on the meth_sites half; -p file labelling every such site m6A or A.  Returns paths and truth."""
    from mcaller_b200 import refmark, synth
    spec = synth.SynthSpec(seed=seed, contigs=[("ctgA", 24000), ("ctgB", 18000)], n_reads=n_reads, len_min=300, len_max=900, meth=True)
    genomes = [synth.genome(spec, ci) for ci in range(len(spec.contigs))]
    pos_rows, site_maps, truth = [], {}, {}
    for ci, (nm, _) in enumerate(spec.contigs):
        seq = genomes[ci].tobytes().decode()
        maps = []
        for strand_ix, st in enumerate("+-"):
            bm = np.zeros(len(seq), dtype=np.uint8)
            for motif in ("GATC", "TAGC"):
                bm |= refmark.site_bitmap(refmark.mark_reference(seq, "A", motif=motif, contig=nm)[strand_ix])
            meth = synth.meth_sites(spec, ci, bm)
            maps.append(meth)
            for p in np.flatnonzero(bm):
                lab = "m6A" if meth[p] else "A"
                truth[(nm, int(p), st)] = lab
                pos_rows.append("%s\t%d\t%s\t%s\n" % (nm, p, st, lab))
        site_maps[ci] = tuple(maps)
    tsv, fasta, fastq, _ = synth.generate(spec, site_maps)
    paths = {"tsv": os.path.join(d, "syn.eventalign.tsv"), "fasta": os.path.join(d, "ref.fasta"), "fastq": os.path.join(d, "syn.fastq"),
             "positions": os.path.join(d, "pos.txt")}
    for key, data in (("tsv", tsv), ("fasta", fasta.encode()), ("fastq", fastq.encode()), ("positions", "".join(pos_rows).encode())):
        with open(paths[key], "wb") as fh:
            fh.write(data)
    return paths, truth


@pytest.mark.gpu
def test_cli_train_end_to_end(tmp_path, cuda_lib, capsys):
    from sklearn.neural_network import MLPClassifier
    from mcaller_b200 import cli, models, train as tr
    d1, d2 = tmp_path / "one", tmp_path / "two"
    d1.mkdir()
    d2.mkdir()
    inp, _ = _labelled_set(str(d1), 31)
    common = ["-p", inp["positions"], "-r", inp["fasta"], "-e", inp["tsv"], "-f", inp["fastq"], "-b", "A"]
    pk1, pk3, pk_tsv = (str(tmp_path / n) for n in ("t1.pkl", "t3.pkl", "tsv.pkl"))
    assert cli.mcaller_main(["--train", "-d", pk1] + common) == 0
    train_file = os.path.join(str(d1), "syn.eventalign.diffs.6.train")
    t1 = open(train_file, "rb").read()
    assert cli.mcaller_main(["--train", "-t", "3", "-d", pk3] + common) == 0
    assert open(train_file, "rb").read() == t1
    assert not [f for f in os.listdir(str(d1)) if ".tmp" in f]
    assert cli.mcaller_main(["--training_tsv", train_file, "-d", pk_tsv] + common) == 0
    out = capsys.readouterr().out
    assert "fold 5 held-out accuracy" in out
    b1 = open(pk1, "rb").read()
    assert open(pk3, "rb").read() == b1 and open(pk_tsv, "rb").read() == b1
    model = models.load_model_file(pk1)
    assert sorted(model) == ["MG", "MH"]
    e0, e1, two = models.select_models(model, "A")
    assert two and type(e0).__name__ == "MLPClassifier" and list(e0.classes_) == ["A", "m6A"]

    # sklearn's own fit on the same balanced rows
    sites, x, labels, ctxs = tr.read_train_tsv(train_file)
    keys = np.asarray(tr.keys_from_contexts(ctxs, "A", 6))
    ref = {}
    for key in ("MG", "MH"):
        sel = np.flatnonzero(keys == key)
        keep = sel[tr.balance([labels[i] for i in sel], 0)]
        with warnings.catch_warnings():
            warnings.simplefilter("ignore")
            ref[key] = MLPClassifier(random_state=0, **tr.SHIPPED_NN).fit(x[keep], np.asarray(labels)[keep])
        assert model[key].n_iter_ == ref[key].n_iter_
    pk_ref = str(tmp_path / "ref.pkl")
    with open(pk_ref, "wb") as fh:
        pickle.dump(ref, fh)

    inp2, truth = _labelled_set(str(d2), 32)
    common2 = ["-p", inp2["positions"], "-r", inp2["fasta"], "-e", inp2["tsv"], "-f", inp2["fastq"], "-b", "A"]
    diffs = os.path.join(str(d2), "syn.eventalign.diffs.6")
    assert cli.mcaller_main(common2 + ["-d", pk1]) == 0
    mine = open(diffs).read()
    assert cli.mcaller_main(common2 + ["-d", pk_ref]) == 0
    assert open(diffs).read() == mine
    rows = [ln.split("\t") for ln in mine.splitlines()]
    assert len(rows) > 500
    acc = np.mean([r[6] == truth[(r[0], int(r[2]), r[5])] for r in rows])
    assert acc > 0.5, acc
