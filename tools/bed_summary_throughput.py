#!/usr/bin/env python
"""Cost of make_bed's per-read summaries in the multi-GPU product path (`mCaller --gpus N --bed --bed_vo` and
`--bed_positions FILE`), on device-generated input (synthetic E. coli, -m GATC, r95 NN model) at the configs[2] size per GPU
(BASELINE.json: 125k reads per GPU).  One JSON line:
  summary_s       -- rank 0's time from the end of streaming to the written file, per mode, on 1 GPU and on all visible GPUs
  log_kernel_ms   -- the per-chunk time mc_rowlog_append adds: CUDA events around back-to-back replays of it on the last
                     chunk's rows (`vo`: every row, no features; `positions`: the rows of the listed sites, with features)
  text_path_s     -- the alternative: make_bed.aggregate_by_pos --vo / -p on the merged `.diffs` file
  gpu, power_limit_w -- the card and its power limit, read in the same run.
usage: python tools/bed_summary_throughput.py [--reads-per-gpu N] [--dir D]"""
import argparse
import contextlib
import ctypes as C
import io
import json
import os
import re
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
MODEL = os.path.join(ROOT, "tests", "golden", "models", "r95_twobase_model_NN_6_m6A.pkl")


def _inputs(d, reads):
    """TSV / FASTA / FASTQ of `reads` synthetic reads, the TSV written by the device generator."""
    import torch
    from mcaller_b200 import synth, synth_device
    from mcaller_b200.refindex import ReferenceIndex
    spec = synth.SynthSpec(seed=0, contigs=[("ecoli", 4600000)], n_reads=reads, len_min=1000, len_max=3000)
    seqs = {"ecoli": synth.genome(spec, 0).tobytes().decode()}
    ref = ReferenceIndex(seqs, "A", motif="GATC", k=6)
    meth = {0: (synth.meth_sites(spec, 0, ref.site_fwd_bits[:4600000]), synth.meth_sites(spec, 0, ref.site_rev_bits[:4600000]))}
    gen = synth_device.DeviceSynth(spec, ref, meth)
    tsv, fasta, fastq = (os.path.join(d, f) for f in ("syn.eventalign.tsv", "ref.fasta", "syn.fastq"))
    with open(tsv, "wb") as fh:
        for r0 in range(0, reads, 20000):                       # bounded device memory per piece
            d_text, n, _ = gen.generate(r0, min(20000, reads - r0))
            for o in range(0, n, 1 << 28):
                fh.write(d_text[o:min(n, o + (1 << 28))].cpu().numpy().tobytes())
            del d_text
    with open(fasta, "w") as fh:
        fh.write(">ecoli\n%s\n" % seqs["ecoli"])
    with open(fastq, "w") as fh:
        for i in range(reads):
            qs, _ = synth.read_quality_string(spec, i)
            fh.write("@%s\n%s\n+\n%s\n" % (synth.read_name(spec, i), "A" * len(qs), qs))
    del gen
    torch.cuda.empty_cache()
    return tsv, fasta, fastq


def _cli(d, tsv, fasta, fastq, gpus, extra):
    cmd = [sys.executable, "-m", "mcaller_b200.cli", "mCaller", "-m", "GATC", "-r", fasta, "-e", tsv, "-f", fastq, "-d", MODEL, "-b", "A",
           "--gpus", str(gpus), "--bed", "--bed_min_read_depth", "15", "--bed_mod_threshold", "0.5"] + extra
    env = dict(os.environ, PYTHONPATH=ROOT + os.pathsep + os.environ.get("PYTHONPATH", ""))
    p = subprocess.run(cmd, cwd=d, env=env, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    if p.returncode:
        sys.exit(p.stdout[-3000:])
    m = re.search(r"^rank 0: .* written ([0-9.]+) s after the end of streaming$", p.stdout, re.M)
    return float(m.group(1))


def _log_kernel_ms(tsv, fasta, fastq, pos, reps=50):
    """Stream the file once with the row log, then replay mc_rowlog_append on the last chunk's rows, `reps` launches back
    to back between two CUDA events (the log holds every replay's entries, so no write is skipped and nothing else runs
    in between): `vo` = 24-byte entries of every row, `positions` = entries with 6 features of the rows whose site is in
    the positions file (its site flags)."""
    import torch
    from mcaller_b200 import extract_contexts as ec, make_bed as mb, read_qual
    from mcaller_b200 import engine as E
    run = ec.RangeRun(tsv, fasta, read_qual.extract_read_quality_device(fastq), 6, 0, 0.0, MODEL, 0, endline=os.path.getsize(tsv), base="A",
                      motif="GATC", histogram=True)
    run.eng.enable_row_log(6)
    with contextlib.redirect_stdout(io.StringIO()):
        run.stream()
    os.remove(run.tsv_output)
    eng = run.eng
    calls = eng._bufs["calls"]
    n_rows = int(eng.h_small[E.S_NROWS])
    cap = calls.numel() // E.CALL_DTYPE.itemsize
    flags = torch.from_numpy(mb.site_flags(eng.ref, mb.make_pos_set(pos))).to(eng.device)
    out = {}
    for name, n_feat, d_flags in (("vo", 0, None), ("positions", 6, flags)):
        log_cap = (reps + 5) * n_rows + cap
        log = torch.empty(log_cap * int(eng.L.mc_rowlog_stride(n_feat)), dtype=torch.uint8, device=eng.device)
        cnt = torch.zeros(1, dtype=torch.int64, device=eng.device)
        fl = C.c_void_p(d_flags.data_ptr()) if d_flags is not None else None
        st = eng._sptr()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        for i in range(reps + 5):
            if i == 5:
                e0.record()
            eng.L.mc_rowlog_append(C.c_void_p(calls.data_ptr()), eng._status_ptr(E.S_NROWS), cap, eng._persist_ptr(E.P_ROW_BASE), fl,
                                   eng.ref.n_sites, n_feat, C.c_void_p(log.data_ptr()), log_cap, C.c_void_p(cnt.data_ptr()), None, None, st)
        e1.record()
        torch.cuda.synchronize()
        out[name] = dict(ms=round(e0.elapsed_time(e1) / reps, 4), rows_in_chunk=n_rows, rows_logged=int(cnt.item()) // (reps + 5))
    return out


def _text_path_s(d, diffs):
    from mcaller_b200 import make_bed as mb
    import golden_cases as gc
    pos = os.path.join(d, "bedpos.txt")
    gc.write_bed_positions(open(diffs).read(), pos)
    res = {}
    for name, kw in (("vo", dict(pos_list=None, vo=True)), ("positions", dict(pos_list=pos, vo=False))):
        t0 = time.perf_counter()
        with contextlib.redirect_stdout(io.StringIO()):
            mb.aggregate_by_pos(diffs, os.path.join(d, "text.bed"), 15, 0.5, kw["pos_list"], False, kw["vo"], False, None, False, "x", False)
        res[name] = round(time.perf_counter() - t0, 3)
    return res, pos


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reads-per-gpu", type=int, default=125000)
    ap.add_argument("--dir", default=None)
    a = ap.parse_args()
    import torch
    n_gpu = torch.cuda.device_count()
    gpu = torch.cuda.get_device_name(0)
    try:
        power = float(subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader,nounits", "-i", "0"],
                                     stdout=subprocess.PIPE, text=True).stdout.strip())
    except (OSError, ValueError):
        power = None
    base = a.dir or tempfile.mkdtemp(prefix="mc_bedsum_")
    res = dict(gpu=gpu, power_limit_w=power, reads_per_gpu=a.reads_per_gpu, summary_s={}, text_path_s={},
               timed=dict(summary_s="rank 0: end of streaming -> summary file written (mCaller --gpus N --bed, -d 15 -t 0.5)",
                          text_path_s="make_bed.aggregate_by_pos on the merged .diffs file, same thresholds",
                          log_kernel_ms="one mc_rowlog_append launch on one chunk's rows (mean of back-to-back replays)"))
    for gpus in sorted({1, n_gpu}):
        d = os.path.join(base, "g%d" % gpus)
        os.makedirs(d, exist_ok=True)
        tsv, fasta, fastq = _inputs(d, a.reads_per_gpu * gpus)
        _cli(d, tsv, fasta, fastq, gpus, ["--bed_vo"])                   # warms the page cache; the merged .diffs for the text path
        text, pos = _text_path_s(d, os.path.join(d, "syn.eventalign.diffs.6"))
        res["text_path_s"]["%d_gpu" % gpus] = text
        res["summary_s"]["%d_gpu" % gpus] = dict(vo=_cli(d, tsv, fasta, fastq, gpus, ["--bed_vo"]),
                                                 positions=_cli(d, tsv, fasta, fastq, gpus, ["--bed_positions", pos]))
        if gpus == 1:
            res["log_kernel_ms"] = _log_kernel_ms(tsv, fasta, fastq, pos)
    print(json.dumps(res))


if __name__ == "__main__":
    main()
