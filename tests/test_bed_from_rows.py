"""make_bed's per-read modes (--vo, -p) in the multi-GPU product path (`mCaller --gpus N --bed --bed_vo / --bed_positions`):
the rows each rank logs on the device (Engine.enable_row_log), gathered to rank 0 and grouped by locus there
(make_bed.aggregate_from_rows), give byte for byte the file of the unmodified reference's make_bed.py (goldens) and of
the drop-in make_bed.aggregate_by_pos on the run's own `.diffs` text."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

import golden_cases as gc

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _args(a):
    """make_bed argument vector -> keyword arguments of aggregate_from_rows / aggregate_by_pos."""
    return dict(depth_thresh=int(a[a.index("-d") + 1]), mod_thresh=float(a[a.index("-t") + 1]), control="--control" in a,
                verbose_results="--vo" in a, gff="--gff" in a)


def _stream(case, inp, tmp_path, positions=None, chunk=None, n_feat=6):
    """One worker over the whole file with the histogram and the row log (n_feat features per entry: 0 is the layout of
    `--bed_vo` alone); the last open window is dropped (end of file)."""
    from mcaller_b200 import extract_contexts as ec, make_bed as mb, read_qual
    base = case.get("base", "A")
    motif = case.get("motif")
    if motif and len(motif) == 1:
        base = motif
    tmp = ec.diffs_name(inp["tsv"], 6, 0)
    if os.path.exists(tmp):
        os.remove(tmp)
    old = ec.CHUNK_BYTES
    if chunk:
        ec.CHUNK_BYTES = chunk
    try:
        run = ec.RangeRun(inp["tsv"], inp["fasta"], read_qual.extract_read_quality(inp["fastq"]), 6, case.get("s", 0), case.get("q", 0.0),
                          inp["model"], 0, endline=os.path.getsize(inp["tsv"]), base=base, motif=motif, positions_list=inp.get("positions"),
                          histogram=True)
        run.eng.enable_row_log(n_feat, mb.site_flags(run.ref, mb.make_pos_set(positions)) if positions else None)
        run.stream()
    finally:
        ec.CHUNK_BYTES = old
    row = run.eng.close_carry(-1)
    assert int(row[0]["kind"]) == 3
    return run


def _from_rows(run, out, a, pos_list, ref=None):
    from mcaller_b200 import make_bed as mb
    depth, meth, first = run.eng.histogram_host()
    d_log, n_log = run.eng.row_log()
    kw = _args(a)
    mb.aggregate_from_rows(run.ref, depth, meth, first, d_log, n_log, run.eng.log_nfeat, out, kw["depth_thresh"], kw["mod_thresh"],
                           pos_list=pos_list, control=kw["control"], verbose_results=kw["verbose_results"], gff=kw["gff"], ref=ref,
                           odd_rows=run.eng.odd_rows())
    return open(out).read()


def _from_text(diffs, out, a, pos_list, ref=None):
    from mcaller_b200 import make_bed as mb
    kw = _args(a)
    mb.aggregate_by_pos(diffs, out, kw["depth_thresh"], kw["mod_thresh"], pos_list, kw["control"], kw["verbose_results"], kw["gff"], ref,
                        False, "x", False)
    return open(out).read()


def _per_read_beds(gold):
    return [b for b in gold["beds"] if "-p" in b["args"] or "--vo" in b["args"]]


# ---- GPU: one rank, against the reference's goldens --------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("name", ["gatc_s0", "gatc_s2"])
@pytest.mark.parametrize("chunk", [None, 60000])
def test_per_read_beds_from_device_rows_match_reference(name, chunk, tmp_path, capsys, cuda_lib):
    case = gc.CASES[name]
    gold = json.load(open(os.path.join(gc.GOLD, name + ".json")))
    inp = gc.build_inputs(case, str(tmp_path))
    beds = _per_read_beds(gold)
    assert beds and all(b["rc"] == 0 for b in beds)
    pos = os.path.join(str(tmp_path), "bedpos.txt")
    gc.write_bed_positions(gold["diffs"], pos)
    runs = {}
    for b in beds:
        a = b["args"]
        p = pos if "-p" in a else None
        if p not in runs:                                     # --vo alone: the 24-byte entries without features
            runs[p] = _stream(case, inp, tmp_path, positions=p, chunk=chunk, n_feat=6 if p else 0)
            assert open(runs[p].tsv_output).read() == gold["diffs"]
        assert _from_rows(runs[p], os.path.join(str(tmp_path), "r.bed"), a, p) == b["bed"], a
    capsys.readouterr()


# ---- GPU: one rank, against the drop-in on the run's own text ------------------------------------------------------------
FLAG_SETS = [["-d", "1", "-t", "0.5", "--vo"], ["-d", "2", "-t", "0.4", "--gff", "--vo"], ["-d", "1", "-t", "0.5", "--control", "--vo"],
             ["-d", "1", "-t", "0.5", "--ref", "--vo"], ["-d", "1", "-t", "0.5", "-p"], ["-d", "1", "-t", "0.5", "-p", "--vo"]]


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["A_s0", "gat_q_handoff", "A_q_handoff", "pos_p", "cg_c", "rf_gatc"])
def test_per_read_beds_from_device_rows_match_drop_in(name, tmp_path, capsys, cuda_lib):
    case = gc.CASES[name]
    inp = gc.build_inputs(case, str(tmp_path))
    d = str(tmp_path)
    pos = os.path.join(d, "bedpos.txt")
    nomatch = os.path.join(d, "nomatch.txt")
    with open(nomatch, "w") as fh:
        fh.write("nosuchcontig\t10\t11\t+\n")
    run_all = _stream(case, inp, tmp_path)
    diffs = os.path.join(d, "syn.eventalign.diffs.6")
    os.replace(run_all.tsv_output, diffs)
    text = open(diffs).read()
    gc.write_bed_positions(text, pos)
    run_pos = _stream(case, inp, tmp_path, positions=pos)
    assert open(run_pos.tsv_output).read() == text
    run_none = _stream(case, inp, tmp_path, positions=nomatch)
    run_vo = _stream(case, inp, tmp_path, n_feat=0)
    for a in FLAG_SETS:
        ref = inp["fasta"] if "--ref" in a else None
        if "-p" in a:
            for run, p in ((run_pos, pos), (run_none, nomatch), (run_all, pos)):        # run_all: log unfiltered, loci filtered
                assert _from_rows(run, os.path.join(d, "r.bed"), a, p) == _from_text(diffs, os.path.join(d, "t.bed"), a, p), (a, p)
        else:
            want = _from_text(diffs, os.path.join(d, "t.bed"), a, None, ref)
            assert want
            for run in (run_vo, run_all):
                assert _from_rows(run, os.path.join(d, "r.bed"), a, None, ref) == want, a
    capsys.readouterr()


# ---- GPU: deep coverage (every branch of the pairwise sums, loci of more than 1 024 rows) --------------------------------
DEEP_CASE = dict(spec=dict(seed=41, contigs=[("deep", 90), ("mid", 120)], n_reads=10000, len_min=40, len_max=40), motif="AT", model=gc.R95,
                 base="A")


@pytest.mark.gpu
def test_per_read_beds_deep_loci_match_drop_in(tmp_path, capsys, cuda_lib):
    d = str(tmp_path)
    inp = gc.build_inputs(DEEP_CASE, d)
    run = _stream(DEEP_CASE, inp, tmp_path, chunk=8 << 20)
    depth, _, _ = run.eng.histogram_host()
    dep = depth[depth > 0]
    assert dep.max() > 1024 and ((dep > 128) & (dep <= 1024)).any() and (dep <= 128).any(), sorted(dep.tolist())
    diffs = os.path.join(d, "syn.eventalign.diffs.6")
    os.replace(run.tsv_output, diffs)
    pos = os.path.join(d, "bedpos.txt")
    text = open(diffs).read()
    gc.write_bed_positions(text, pos)
    for a in (["-d", "1", "-t", "0.5", "--vo"], ["-d", "1", "-t", "0.5", "-p", "--vo"], ["-d", "1", "-t", "0.5", "--gff", "--vo"]):
        p = pos if "-p" in a else None
        assert _from_rows(run, os.path.join(d, "r.bed"), a, p) == _from_text(diffs, os.path.join(d, "t.bed"), a, p), a
    capsys.readouterr()


# ---- GPU: the CLI's ranks (gloo on one GPU, NCCL on two) -------------------------------------------------------------------
def _cli_ranks(name, world, tmp_path, extra, backend=None):
    case = gc.CASES[name]
    inp = gc.build_inputs(case, str(tmp_path))
    env = dict(os.environ)
    env["PYTHONPATH"] = ROOT + os.pathsep + env.get("PYTHONPATH", "")
    if backend:
        env["MCALLER_B200_DIST_BACKEND"] = backend
    env["MCALLER_B200_CHUNK_BYTES"] = "70000"
    cmd = [sys.executable, "-m", "mcaller_b200.cli", "mCaller"] + gc.cli_args(case, inp) + ["--gpus", str(world), "--bed"] + extra
    p = subprocess.run(cmd, cwd=str(tmp_path), env=env, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True, timeout=900)
    assert p.returncode == 0, p.stdout[-3000:]
    return p.stdout


# (golden make_bed args, CLI flags, output file)
RANK_VARIANTS = [(["-d", "1", "-t", "0.5", "--vo"], ["--bed_vo"], "syn.methylation.summary.bed"),
                 (["-d", "2", "-t", "0.4", "--gff", "--vo"], ["--bed_vo", "--bed_gff"], "syn.methylation.summary.gff"),
                 (["-d", "1", "-t", "0.5", "-p", "bedpos.txt", "--vo"], ["--bed_positions", "bedpos.txt", "--bed_vo"],
                  "syn.methylation.positions.summary.bed")]


def _check_ranks(world, tmp_path, backend):
    gold = json.load(open(os.path.join(gc.GOLD, "gatc_s0.json")))
    for i, (a, flags, out) in enumerate(RANK_VARIANTS):
        d = tmp_path / ("v%d" % i)
        d.mkdir()
        gc.write_bed_positions(gold["diffs"], str(d / "bedpos.txt"))
        extra = ["--bed_min_read_depth", a[a.index("-d") + 1], "--bed_mod_threshold", a[a.index("-t") + 1]] + flags
        _cli_ranks("gatc_s0", world, d, extra, backend)
        assert open(str(d / "syn.eventalign.diffs.6")).read() == gold["diffs"]
        want = [b for b in gold["beds"] if b["args"] == a][0]["bed"]
        assert open(str(d / out)).read() == want, a
        assert not [f for f in os.listdir(str(d)) if ".tmp" in f]


@pytest.mark.gpu
@pytest.mark.parametrize("world", [2, 3])
def test_per_read_beds_from_ranks_on_one_gpu(world, tmp_path, cuda_lib):
    _check_ranks(world, tmp_path, "gloo")


@pytest.mark.gpu
def test_per_read_beds_from_ranks_nccl(tmp_path, cuda_lib):
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    _check_ranks(2, tmp_path, None)


# ---- CPU ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("extra", [["--bed_vo"], ["--bed_positions", "p.txt"], ["--gpus", "2", "--bed_vo"], ["--bed", "--bed_vo"],
                                   ["--bed", "--bed_positions", "p.txt"]])
def test_per_read_flags_need_gpus_and_bed(extra, tmp_path, capsys):
    from mcaller_b200 import cli
    with pytest.raises(SystemExit) as e:
        cli.mcaller_main(["-m", "GATC", "-r", "r.fa", "-e", "x.tsv", "-f", "x.fq"] + extra)
    assert e.value.code == 2
    assert "--bed_vo and --bed_positions need --gpus N --bed" in capsys.readouterr().err


def test_missing_positions_file_fails_before_any_rank(tmp_path, monkeypatch):
    from mcaller_b200 import cli, multigpu

    def no_ranks(*a, **k):
        raise AssertionError("ranks spawned")
    monkeypatch.setattr(multigpu, "run", no_ranks)
    with pytest.raises(AssertionError, match="positions file not found at " + str(tmp_path / "missing.txt")):
        cli.mcaller_main(["-m", "GATC", "-r", "r.fa", "-e", "x.tsv", "-f", "x.fq", "--gpus", "2", "--bed", "--bed_positions",
                          str(tmp_path / "missing.txt")])


def test_row_log_entry_points_declared_exported_bound():
    import ctypes as C
    from mcaller_b200 import _lib, build
    build.build()
    hdr = open(os.path.join(ROOT, "include", "mcaller_b200.h")).read()
    lib = _lib.load()
    for fn in ("mc_rowlog_stride", "mc_rowlog_append", "mc_rowlog_group_workspace_bytes", "mc_rowlog_group", "mc_colstats", "mc_format_probs"):
        assert (" %s(" % fn) in hdr and fn in _lib.EXPORTS and hasattr(lib, fn), fn
    assert lib.mc_version() == 3
    assert lib.mc_sizeof(10) == _lib.ROW_ENTRY_DTYPE.itemsize == 24
    assert lib.mc_rowlog_stride(0) == 24 and lib.mc_rowlog_stride(6) == 24 + 48
    assert lib.mc_rowlog_group_workspace_bytes(1000, 10) > 1000 * 28


def test_probability_text_is_the_diffs_column():
    """mc_format_probs renders str(np.round(p, 2)) with the .diffs writer's code, in one thread and in several."""
    import ctypes as C
    from mcaller_b200 import _lib, build
    build.build()
    lib = _lib.load()
    rng = np.random.default_rng(3)
    p = np.concatenate([rng.random(200000), [0.0, 1.0, 0.005, 0.015, 0.125, 0.995, 0.5, 1e-20, 0.994999999]])
    for threads in (1, 0):
        buf = np.zeros(32 * len(p), dtype=np.uint8)
        offs = np.zeros(len(p) + 1, dtype=np.int64)
        n = lib.mc_format_probs(p.ctypes.data_as(C.c_void_p), len(p), threads, buf.ctypes.data_as(C.c_void_p), len(buf),
                                offs.ctypes.data_as(C.c_void_p))
        text = buf[:n].tobytes().decode()
        got = [text[offs[i]:offs[i + 1]] for i in range(len(p))]
        assert got == [str(np.round(x, 2)) for x in p]


def test_ttest_finish_is_the_previous_column_tests_finish():
    """The factored finish of column_tests (Student-t tail, -log10, rounding) gives on fixed statistics exactly what the
    finish inside _Aggregation.column_tests gave before it was factored out, and scipy's ttest_1samp's values."""
    import warnings
    from scipy import special, stats as ss
    from mcaller_b200 import make_bed as mb
    rng = np.random.default_rng(5)
    sizes = [2, 3, 9, 17, 130, 1]
    cols = [rng.normal(0.2 * i, 1.5, size=(n, 6)) for i, n in enumerate(sizes)]
    st = np.zeros((len(sizes), 6, 2))
    for li, x in enumerate(cols):
        m = np.mean(x, axis=0)
        st[li, :, 0] = m
        st[li, :, 1] = np.add.reduce((x - m) ** 2, axis=0)
    off = np.concatenate([[0], np.cumsum(sizes)]).astype(np.uint32)
    got = mb.ttest_finish(st, off)
    n = (off[1:].astype(np.int64) - off[:-1].astype(np.int64)).astype(np.float64)[:, None]
    with warnings.catch_warnings(), np.errstate(all="ignore"):
        warnings.simplefilter("ignore")
        var = (st[:, :, 1] / n) * (n / (n - 1.0))
        t = st[:, :, 0] / np.sqrt(var / n)
        p = 2 * special.stdtr(n - 1.0, -np.abs(t))
        want = []
        for li in range(len(sizes)):
            pvals = [(p[li, c], t[li, c]) for c in range(6)]
            pval = (sum([-np.log10(x[0]) for x in pvals]), max([x[1] for x in pvals]))
            want.append([np.round(x, 3) for x in [pval[1], pval[0]]])
    assert str(got) == str(want)
    for li, x in enumerate(cols[:-1]):
        pv = [ss.ttest_1samp(x[:, c], 0) for c in range(6)]
        assert [float(v) for v in got[li]] == pytest.approx([max(r[0] for r in pv), sum(-np.log10(r[1]) for r in pv)], abs=1.01e-3)
