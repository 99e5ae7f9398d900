"""`-n` (k, the number of window columns) other than the default 6.  Everything that depends on k -- the candidate and
k-mer bit maps, the whole-read unit rule, the column-slot permutation of the multi-M carry, the context bounds, the k + 1
features, the writer's 2k-1 context -- is run for k = 2..8 against the CPU oracle, with (k + 1)-input MLPs fitted here.

The reference itself only ever ran with -n 6 in this project's golden cases and is not part of the repository, so at
k != 6 the oracle's literal restatement of the reference's state machine (oracle/mcaller_oracle.c) is the reference."""
import functools
import os
import pickle
import warnings

import numpy as np
import pytest

KS = [2, 3, 4, 5, 7, 8]


def _features(n, d, seed):
    """n rows of d features shaped like the window features: k column means around 0, then a read quality."""
    rng = np.random.RandomState(seed)
    x = rng.normal(0, 3, (n, d))
    x[:, -1] = rng.uniform(3, 20, n)
    return x


@functools.lru_cache(maxsize=None)
def _model_dict(n_in):
    """{'MH', 'MG'}: two different seeded MLPClassifier fits (100 tanh units, the shipped shape) taking n_in inputs.  A few
    iterations only: the shapes matter here, not the quality of the fit."""
    from sklearn.neural_network import MLPClassifier
    x = _features(600, n_in, 100 + n_in)
    rules = {"MH": x[:, 0] > 0, "MG": x[:, 0] - (0.5 * x[:, 1] if n_in > 2 else 0) < 0.5}
    out = {}
    for seed, (key, y) in enumerate(sorted(rules.items())):
        with warnings.catch_warnings():
            warnings.simplefilter("ignore")
            out[key] = MLPClassifier(hidden_layer_sizes=(100,), activation="tanh", max_iter=5, random_state=seed).fit(
                x, np.where(y, "m6A", "A"))
    return out


def _synth(seed, n_reads=40, contigs=(("ctg_one", 9000), ("c2", 6000)), len_min=300, len_max=900):
    from mcaller_b200 import synth
    spec = synth.SynthSpec(seed=seed, contigs=list(contigs), n_reads=n_reads, len_min=len_min, len_max=len_max)
    tsv, fasta, fastq, quals = synth.generate(spec)
    seqs = {nm: synth.genome(spec, ci).tobytes().decode() for ci, (nm, _) in enumerate(spec.contigs)}
    return spec, tsv, fastq, {q.split("_")[0]: v for q, v in quals.items()}, seqs


# ---- host (no GPU) --------------------------------------------------------------------------------------------------

def test_oracle_refuses_k1_on_the_model_key(oracle):
    """At k = 1 the context has one letter, so the model key context[k-1:k+1] (extract_contexts.py:197, base_models
    :99-106) is one letter: KeyError, with a model and without one.  k = 2 writes rows."""
    _, tsv, _, quals, seqs = _synth(5, n_reads=30)
    for model in (_model_dict(2), None):
        with pytest.raises(oracle.OracleError, match="KeyError: model key"):
            oracle.extract(tsv, seqs, quals, k=1, skip_thresh=0, model=model, base="A", motif="GATC", cap=100000)
    assert len(oracle.extract(tsv, seqs, quals, k=2, skip_thresh=0, model=_model_dict(3), base="A", motif="GATC", cap=100000)["rows"]) > 20


@pytest.mark.parametrize("k", [0, 9])
def test_reference_index_refuses_k_outside_1_to_8(k):
    from mcaller_b200.refindex import ReferenceIndex
    with pytest.raises(ValueError, match="num_variables must be in 1..8"):
        ReferenceIndex({"c": "ACGTGATCAA" * 10}, "A", motif="GATC", k=k)


@pytest.mark.parametrize("k", [1, 4, 8])
def test_cli_skip_threshold_must_be_under_half_of_k(k, tmp_path):
    """mCaller.py's `skip_thresh < num_variables / 2` assertion: -s ceil(k/2) is refused, -s (k-1)//2 passes it (and the run
    then stops at the missing FASTQ, the next check)."""
    from mcaller_b200 import cli
    model = tmp_path / "m.pkl"
    model.write_bytes(b"x")
    args = ["-m", "GATC", "-r", "r.fa", "-e", "x.tsv", "-f", str(tmp_path / "missing.fq"), "-d", str(model), "-n", str(k)]
    with pytest.raises(AssertionError, match="too many skips with only %d variables" % k):
        cli.mcaller_main(args + ["-s", str((k + 1) // 2)])
    with pytest.raises(AssertionError, match="fastq file not found"):
        cli.mcaller_main(args + ["-s", str((k - 1) // 2)])


@pytest.mark.parametrize("wrong", ["MH", "MG"])
def test_model_of_the_wrong_width_is_refused_before_device_work(wrong):
    """Both estimators of a two-model pickle must take k + 1 inputs (scikit-learn would raise ValueError on the first
    call); checked on the host before anything is copied to the device, and the error names the key."""
    from mcaller_b200 import models
    k = 4
    m = dict(_model_dict(k + 1))
    m[wrong] = _model_dict(k + 2)["MH"]
    with pytest.raises(ValueError, match="model '%s' expects %d inputs but -n %d gives %d" % (wrong, k + 2, k, k + 1)):
        models.DeviceModels(m["MH"], m["MG"], device="cpu", n_in=k + 1)
    with pytest.raises(ValueError, match="model expects 7 inputs but -n 4 gives 5"):
        models.DeviceModels(_model_dict(7)["MH"], device="cpu", n_in=k + 1)


# ---- GPU ------------------------------------------------------------------------------------------------------------

def _sweep_cases():
    out = []
    for k in KS:
        for regime in ("GATC", "A"):
            for s in sorted({0, (k - 1) // 2}):
                out.append((k, regime, s))
    return out


@pytest.mark.gpu
@pytest.mark.parametrize("k,regime,s", _sweep_cases())
def test_windows_and_calls_match_oracle_at_k(k, regime, s, cuda_lib, oracle):
    """Window rows of the device path at k = 2..8 == the oracle's: GATC (short units) and `-m A` (every fourth position a
    target: long candidate runs and multi-M carries everywhere, so the column-slot permutation runs, k = 8 included), with
    and without skips, sparse and dense scan, the scan forced to pass over chunks in short runs."""
    from mcaller_b200 import _lib, engine, models, read_qual
    from mcaller_b200.refindex import ReferenceIndex
    _, tsv, _, quals, seqs = _synth(300 + k, n_reads=40 if regime == "GATC" else 24)
    model = _model_dict(k + 1)
    dm = models.DeviceModels(model["MH"], model["MG"], n_in=k + 1)
    ref = ReferenceIndex(seqs, "A", motif=regime, k=k)
    want = oracle.extract(tsv, seqs, quals, k=k, skip_thresh=s, model=model, base="A", motif=regime, cap=400000)
    assert len(want["calls"]) > 30
    assert {w["label"] for w in want["calls"]} == {0, 1}
    if regime == "A":                                        # GATC: the base after the target is always T ('MH')
        assert {w["model_sel"] for w in want["calls"]} == {0, 1} and want["counters"]["multi"] > 10
    L = _lib.lib()
    before = L.mc_scan_set_run_len(8)
    try:
        for dense in (None, True):
            eng = engine.Engine(ref, models=dm, qual_table=read_qual.build_quality_table(quals), skip_thresh=s, two_models=True, dense=dense)
            res = eng.run_chunk(eng.upload(tsv), len(tsv))
            assert res.missing_quality == 0
            calls = res.calls()
            mine = calls[(calls["kind"] == _lib.MC_CALL) & (calls["close_rec"] != _lib.PENDING)]
            assert len(mine) == len(want["calls"])
            for c, w in zip(mine, want["calls"]):
                assert int(c["mpos"]) == w["mpos"] and bool(c["rev"]) == w["rev"] and int(c["empty_mask"]) == w["empty_mask"]
                assert tsv[int(c["read_off"]):int(c["read_off"]) + int(c["read_len"])].decode() == w["read"]
                assert [float(x) for x in c["feat"][:k + 1]] == w["feat"]
                assert np.all(c["feat"][k + 1:] == 0)
                assert int(c["model_sel"]) == w["model_sel"]
                assert abs(float(c["prob"]) - w["prob"]) < 1e-12 and int(c["label"]) == w["label"]
            st = eng.count_rows(res)
            assert st["too_many_skips"] == want["counters"]["too_many_skips"] and st["multi"] == want["counters"]["multi"]
            assert st["errors"] == 0
    finally:
        L.mc_scan_set_run_len(before)


@pytest.mark.gpu
def test_k1_raises_the_model_key_error(cuda_lib, oracle):
    """k = 1: every call row whose context is in bounds carries the model-key error, and the writer raises what the
    reference does at its first such row (KeyError in base_models, caught with a message and sys.exit: ReferenceAbort)."""
    import torch
    from mcaller_b200 import _lib, engine, extract_contexts as ec, models, read_qual, stream
    from mcaller_b200.refindex import ReferenceIndex
    _, tsv, _, quals, seqs = _synth(5, n_reads=30)
    model = _model_dict(2)
    with pytest.raises(oracle.OracleError, match="KeyError: model key"):
        oracle.extract(tsv, seqs, quals, k=1, skip_thresh=0, model=model, base="A", motif="GATC", cap=100000)
    ref = ReferenceIndex(seqs, "A", motif="GATC", k=1)
    eng = engine.Engine(ref, models=models.DeviceModels(model["MH"], model["MG"], n_in=2), qual_table=read_qual.build_quality_table(quals),
                        skip_thresh=0, two_models=True)
    res = eng.run_chunk(eng.upload(tsv), len(tsv))
    calls = res.calls()
    mine = calls[(calls["kind"] == _lib.MC_CALL) & (calls["close_rec"] != _lib.PENDING)]
    assert len(mine) > 20
    assert np.all((mine["err"] & (_lib.MC_CE_MODELKEY | _lib.MC_CE_CONTEXT)) != 0)
    assert np.any(mine["err"] == _lib.MC_CE_MODELKEY)
    host = torch.empty(len(tsv), dtype=torch.uint8, pin_memory=True)
    host.copy_(torch.frombuffer(bytearray(tsv), dtype=torch.uint8))
    hs = stream.HostStreamer(eng, chunk_bytes=len(tsv) + 1)
    with pytest.raises(ec.ReferenceAbort, match="base after target"):
        hs.run(host, stream.plan_chunks(_read_starts(tsv), len(tsv), hs.chunk_bytes), sink=stream.TextSink(ref, 1, "A"))


def _read_starts(tsv):
    offs, o, last = [], 0, None
    for ln in tsv.split(b"\n")[:-1]:
        f = ln.split(b"\t")
        if len(f) > 3 and f[3] != last:
            offs.append(o)
            last = f[3]
        o += len(ln) + 1
    return offs


@pytest.mark.gpu
@pytest.mark.parametrize("k", [2, 8])
def test_streamed_text_at_k_matches_oracle(k, cuda_lib, oracle):
    """HostStreamer + TextSink at k = 2 and 8, in one chunk and in several: the `.diffs.<k>` text (2k-1 context letters, k
    feature fields and the quality, label, probability) is the oracle's byte for byte, also for the windows carried over
    chunk edges.  At k = 8 the same input is also run with -q (the scan's read-first mode)."""
    import torch
    from mcaller_b200 import engine, models, read_qual, stream
    from mcaller_b200.refindex import ReferenceIndex
    _, tsv, _, quals, seqs = _synth(900 + k, n_reads=120, contigs=(("ecoli", 40000),), len_min=400, len_max=1500)
    model = _model_dict(k + 1)
    dm = models.DeviceModels(model["MH"], model["MG"], n_in=k + 1)
    ref = ReferenceIndex(seqs, "A", motif="GATC", k=k)
    host = torch.empty(len(tsv), dtype=torch.uint8, pin_memory=True)
    host.copy_(torch.frombuffer(bytearray(tsv), dtype=torch.uint8))
    offs = _read_starts(tsv)
    qts = [0.0] + ([float(np.median(list(quals.values())))] if k == 8 else [])
    for qt in qts:
        want = oracle.extract(tsv, seqs, quals, k=k, skip_thresh=(k - 1) // 2, qual_thresh=qt, model=model, base="A", motif="GATC",
                              cap=200000)
        want_text = "".join(r + "\n" for r in want["rows"]).encode()
        assert len(want["rows"]) > (100 if qt else 250)
        eng = engine.Engine(ref, models=dm, qual_table=read_qual.build_quality_table(quals), skip_thresh=(k - 1) // 2, qual_thresh=qt,
                            two_models=True)
        if qt:
            assert eng.scan_mode == 2
        for chunk_bytes in (len(tsv) + 1, len(tsv) // 6):
            hs = stream.HostStreamer(eng, chunk_bytes=chunk_bytes)
            sink = stream.TextSink(ref, k, "A", keep=True)
            eng.reset_histogram()
            cuts = stream.plan_chunks(offs, len(tsv), hs.chunk_bytes)
            assert len(cuts) == 1 or len(cuts) >= 4
            hs.run(host, cuts, sink=sink)
            assert b"".join(sink.kept) == want_text
            assert sink.n_obs == len(want["rows"])


@pytest.mark.gpu
def test_cli_at_k8_with_bed_matches_oracle(tmp_path, cuda_lib, oracle):
    """python -m mcaller_b200.cli mCaller -n 8 ... --gpus 1 --bed with a pickled (k + 1)-input model dict: the `.diffs.8`
    file is the oracle's rows and the BED is the oracle's make_bed aggregation of them."""
    import subprocess
    import sys
    _, tsv, fastq, quals, seqs = _synth(77, n_reads=150, contigs=(("ctg", 6000),), len_min=300, len_max=900)
    model = _model_dict(9)
    d = str(tmp_path)
    paths = {n: os.path.join(d, n) for n in ("ref.fasta", "syn.eventalign.tsv", "syn.fastq", "m.pkl")}
    with open(paths["ref.fasta"], "w") as fh:
        for nm, s in seqs.items():
            fh.write(">%s\n%s\n" % (nm, s))
    with open(paths["syn.eventalign.tsv"], "wb") as fh:
        fh.write(tsv)
    with open(paths["syn.fastq"], "w") as fh:
        fh.write(fastq)
    with open(paths["m.pkl"], "wb") as fh:
        pickle.dump(model, fh)
    want = oracle.extract(tsv, seqs, oracle.read_fastq_quals(paths["syn.fastq"]), k=8, skip_thresh=3, model=model, base="A",
                          motif="GATC", cap=200000)
    want_text = "".join(r + "\n" for r in want["rows"])
    bed = oracle.aggregate(want_text, 3, 0.5, False)
    assert len(want["rows"]) > 300 and len(bed) > 5
    env = dict(os.environ)
    env["PYTHONPATH"] = os.path.dirname(os.path.dirname(os.path.abspath(__file__))) + os.pathsep + env.get("PYTHONPATH", "")
    env["MCALLER_B200_CHUNK_BYTES"] = "70000"                    # several chunks: windows carried over chunk edges
    cmd = [sys.executable, "-m", "mcaller_b200.cli", "mCaller", "-m", "GATC", "-r", paths["ref.fasta"], "-e", paths["syn.eventalign.tsv"],
           "-f", paths["syn.fastq"], "-d", paths["m.pkl"], "-b", "A", "-n", "8", "-s", "3", "--gpus", "1", "--bed",
           "--bed_min_read_depth", "3", "--bed_mod_threshold", "0.5"]
    p = subprocess.run(cmd, cwd=d, env=env, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True, timeout=900)
    assert p.returncode == 0, p.stdout[-3000:]
    assert open(os.path.join(d, "syn.eventalign.diffs.8")).read() == want_text
    assert open(os.path.join(d, "syn.methylation.summary.bed")).read() == "".join(b + "\n" for b in bed)
