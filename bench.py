#!/usr/bin/env python
"""bench.py -- per-read methylation site calls/sec of the mCaller hot path on B200 (BASELINE.json metric).

A step = one pass of the hot path (TSV scan -> window features -> classifier -> per-site histogram) over one batch of
synthetic eventalign text resident in HBM.  The workload follows BASELINE.json `configs`:

  N = 1 (default)   configs[1]: synthetic E. coli 4.6 Mb, 100k reads, -m GATC, NN model (r95), -n 6, -s 0.
  N > 1 (torchrun)  configs[2]: the same at 1M reads over 8 GPUs = 125k reads per GPU (weak scaling: per-GPU work fixed
                    for N = 2/4/8), -s 1, reads sharded over the ranks, the slice-edge windows closed across ranks, the
                    per-site histograms all-reduced over NCCL and make_bed.py's -d 15 -t 0.5 thresholds applied to the
                    combined histogram -- all inside the timed region.
  --config 3        configs[3]: -c RF (tree-walk kernel).     --config 4: configs[4]: motif CAAYNNNNNRTAC + its model.
  --motif A         dense regime (every A is a target: no quiet chunks in the scan).
  --qual Q          -q read-quality filter (sparse scan in read-first mode; --scan-dense: every kept line recorded, as round 1).

`value` times the pass with the text already resident in HBM (CUDA events, max over ranks); `e2e` times the same metric
through the public host-buffer path (pinned host memory -> H2D -> kernels -> rows D2H -> `.diffs` text); `roofline` is the
scan kernel against the measured HBM bandwidth; `cpu_baseline` (N = 1) and `--impl reference` time the UNMODIFIED
reference (`python oracle/_ref/mCaller.py ... -t <cores>`, laid out by oracle/make_ref.sh) on a bounded sample of the
same workload, and `parity_check` compares the GPU rows on that sample with the reference's and the oracle's.
`--dump-outputs DIR` writes the rows and the histogram of the last timed step as .npy files: the inputs are seeded, so two
builds run with the same arguments can be compared output for output.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--config 1|2|3|4] [--reads R]
                    [--dump-outputs DIR] ...
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import numpy as np  # noqa: E402

MODELS = os.path.join(ROOT, "tests", "golden", "models")
MODEL = os.path.join(MODELS, "r95_twobase_model_NN_6_m6A.pkl")
MODEL_CAAY = os.path.join(MODELS, "CAAYNNNNNRTAC_model_6_m6A.pkl")
METRIC = "per-read site calls/sec"
UNIT = "calls/s"
BED_DEPTH, BED_THRESH = 15, 0.5           # make_bed.py -d 15 -t 0.5 (BASELINE configs[2])


def positive_int(s):
    v = int(s)
    if v < 1:
        raise argparse.ArgumentTypeError("must be at least 1")
    return v


def parse_args():
    p = argparse.ArgumentParser()
    p.add_argument("--gpus", type=int, default=1)
    p.add_argument("--steps", type=positive_int, default=10, help="timed steps (of the main region and of the e2e leg)")
    p.add_argument("--warmup", type=int, default=3)
    p.add_argument("--impl", default="ours", choices=["ours", "reference"])
    p.add_argument("--config", type=int, default=0, choices=[0, 1, 2, 3, 4],
                   help="BASELINE.json configs index (0: 1 on one GPU, 2 under torchrun)")
    p.add_argument("--reads", type=int, default=0, help="reads per GPU (0: the config's: 100k, configs[2] 125k)")
    p.add_argument("--e2e-bytes", type=float, default=8e9, help="size of the pinned host sample streamed by the e2e leg")
    p.add_argument("--e2e-chunk", type=int, default=1 << 30)
    p.add_argument("--cpu-reads", type=int, default=4000, help="reads in the bounded CPU-baseline sample")
    p.add_argument("--skip", type=int, default=-1, help="-s skip threshold (-1: the config's)")
    p.add_argument("--motif", default="", help="-m motif (default: the config's, GATC)")
    p.add_argument("--qual", type=float, default=0.0, help="-q read-quality threshold (0: no filter; the synthetic read means spread around 9-13)")
    p.add_argument("--scan-dense", action="store_true", help="record every kept line in the scan (round-1 behaviour under -q)")
    p.add_argument("--classifier", default="", choices=["", "NN", "RF"],
                   help="NN: the shipped MLP pickle; RF: a forest with the reference's -c RF hyper-parameters "
                        "(train_model.py:39-45) fitted on synthetic features (configs[3], tree-walk kernel)")
    p.add_argument("--contig-name", default="ecoli", help="name of the synthetic contig (column 1 of every line)")
    p.add_argument("--no-e2e", action="store_true")
    p.add_argument("--no-cpu", action="store_true")
    p.add_argument("--no-bind", action="store_true", help="do not bind the rank to a core set / NUMA node")
    p.add_argument("--budget-s", type=float, default=240.0, help="wall-clock budget of the reference arm's timed steps")
    p.add_argument("--dump-outputs", metavar="DIR", default="",
                   help="after the timed steps, write what the last one computed as DIR/<name>.npy (see dump_outputs)")
    a = p.parse_args()
    if a.dump_outputs and a.impl != "ours":
        p.error("--dump-outputs needs --impl ours")
    return a


def resolve_config(args, world):
    """BASELINE.json configs -> the knobs of this run."""
    cfg = args.config or (1 if world == 1 else 2)
    c = dict(index=cfg, motif="GATC", skip=0, classifier="NN", reads=100000, bed=False, model=MODEL,
             name="configs[%d]" % cfg)
    if cfg == 2:
        c.update(skip=1, reads=125000, bed=True)
    elif cfg == 3:
        c.update(classifier="RF")
    elif cfg == 4:
        c.update(motif="CAAYNNNNNRTAC", model=MODEL_CAAY)
    if args.motif:
        c["motif"] = args.motif
        if args.motif == "A" and not args.reads:
            c["reads"] = 20000                   # every A is a target: ~50 rows per read-kb; keeps rows + records in a few GB
    if args.skip >= 0:
        c["skip"] = args.skip
    if args.classifier:
        c["classifier"] = args.classifier
    if args.reads:
        c["reads"] = args.reads
    c["qual"] = float(args.qual)
    c["scan_dense"] = bool(args.scan_dense)
    return c


def workload_text(c, nbytes=None, world=1):
    model = ("NN model (%s)" % os.path.basename(c["model"]).split("_model")[0]) if c["classifier"] == "NN" else \
        "RF model (50 trees, depth 10, reference hyper-parameters, fitted on synthetic features)"
    s = "%s: synthetic E. coli 4.6 Mb, %d reads per GPU%s, -m %s, %s, -n 6, -s %d" % (
        c["name"], c["reads"], (" (%.1f GB eventalign TSV)" % (nbytes / 1e9)) if nbytes else "", c["motif"], model, c["skip"])
    if c.get("qual"):
        s += ", -q %g%s" % (c["qual"], " (dense scan)" if c.get("scan_dense") else "")
    if c["bed"]:
        s += ", make_bed -d %d -t %s on the all-reduced histogram" % (BED_DEPTH, BED_THRESH)
    if c["index"] == 2:
        s += " (1M reads at 8 GPUs)"
    if c["index"] == 4:
        s += " (10M reads at 8 GPUs = 12.5 steps of this size per GPU)"
    return s


class ClockSampler(threading.Thread):
    """Samples SM clocks / throttle reasons of one GPU while the timed region runs: NVML (a query takes ~0.1 ms, so even a
    100 ms region gets hundreds of samples) when the bindings load, else the nvidia-smi query of the profiling recipe."""

    NAMES = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.rows, self.stop_flag, self.source = index, [], False, "nvidia-smi"
        self.mem_rows, self.power_rows = [], []
        self.nvml = self.handle = None
        try:
            import pynvml
            pynvml.nvmlInit()
            # NVML enumerates physical devices: map through CUDA_VISIBLE_DEVICES when it lists plain indices
            vis = os.environ.get("CUDA_VISIBLE_DEVICES", "")
            phys = index
            if vis and all(x.strip().isdigit() for x in vis.split(",")) and index < len(vis.split(",")):
                phys = int(vis.split(",")[index])
            self.handle = pynvml.nvmlDeviceGetHandleByIndex(phys)
            self.max_mhz = int(pynvml.nvmlDeviceGetMaxClockInfo(self.handle, pynvml.NVML_CLOCK_SM))
            self.nvml, self.source = pynvml, "nvml"
        except Exception:
            self.nvml = None

    def _sample_nvml(self):
        n = self.nvml
        mhz = int(n.nvmlDeviceGetClockInfo(self.handle, n.NVML_CLOCK_SM))
        try:
            self.mem_rows.append(int(n.nvmlDeviceGetClockInfo(self.handle, n.NVML_CLOCK_MEM)))
            self.power_rows.append(int(n.nvmlDeviceGetPowerUsage(self.handle)) // 1000)
        except Exception:
            pass
        r = int(n.nvmlDeviceGetCurrentClocksEventReasons(self.handle))
        bits = [n.nvmlClocksEventReasonHwSlowdown, n.nvmlClocksEventReasonHwThermalSlowdown, n.nvmlClocksEventReasonSwThermalSlowdown,
                n.nvmlClocksEventReasonSwPowerCap]
        self.rows.append([str(mhz), str(self.max_mhz)] + ["Active" if (r & b) else "Not Active" for b in bits])

    def run(self):
        q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        while not self.stop_flag:
            try:
                if self.nvml is not None:
                    self._sample_nvml()
                    time.sleep(0.002)
                    continue
                out = subprocess.run(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + q, "--format=csv,noheader,nounits"],
                                     stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True, timeout=5).stdout.strip()
                if out:
                    self.rows.append([x.strip() for x in out.split(",")])
            except Exception:
                if self.nvml is not None:
                    self.nvml = None                     # fall back to nvidia-smi for the rest of the run
                    self.source = "nvidia-smi"
            time.sleep(0.1)

    def summary(self):
        self.stop_flag = True
        self.join(timeout=6)
        if not self.rows:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["unavailable"]}
        sm = sorted(int(r[0]) for r in self.rows if r[0].isdigit())
        reasons = [n for j, n in enumerate(self.NAMES) if any(len(r) > 2 + j and r[2 + j].lower().startswith("active") for r in self.rows)]
        out = {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": int(self.rows[0][1]) if self.rows[0][1].isdigit() else None,
               "reasons": reasons, "samples": len(self.rows), "source": self.source}
        if self.mem_rows:
            out["mem_mhz"] = sorted(self.mem_rows)[len(self.mem_rows) // 2]
        if self.power_rows:
            out["power_w"] = sorted(self.power_rows)[len(self.power_rows) // 2]
        return out


def measured_peak_hbm():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        try:
            return float(json.load(open(path))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def fit_reference_rf():
    """{'MG': rf, 'MH': rf} with the hyper-parameters of the reference's -c RF (train_model.py:39-45 minus the arguments
    current scikit-learn has dropped), fitted on 40 000 synthetic feature rows -- no RF pickle is shipped (SURVEY.md 4)."""
    from sklearn.ensemble import RandomForestClassifier
    rng = np.random.RandomState(0)
    X = np.column_stack([rng.normal(0.0, 2.4, size=(40000, 6)), rng.uniform(3.0, 24.0, size=40000)])
    y = np.where(X[:, 2] - 0.6 * X[:, 3] + 0.3 * rng.normal(size=40000) > 0.5, "m6A", "A")
    rf = RandomForestClassifier(n_estimators=50, criterion="entropy", max_depth=10, max_features=4, min_samples_leaf=2,
                                min_samples_split=3, random_state=0, n_jobs=-1).fit(X, y)
    return {"MG": rf, "MH": rf}


def bind_rank(local_rank, local_world, device_index):
    """One disjoint core set per rank, taken from the NUMA node of the rank's GPU when the box has several: the rank's
    Python thread, the reader / writer thread pools and (first touch) its pinned buffers then stay on that node."""
    info = {"bound": False}
    try:
        avail = sorted(os.sched_getaffinity(0))
        node_cpus = None
        try:
            import pynvml
            pynvml.nvmlInit()
            vis = os.environ.get("CUDA_VISIBLE_DEVICES", "")
            phys = device_index
            if vis and all(x.strip().isdigit() for x in vis.split(",")) and device_index < len(vis.split(",")):
                phys = int(vis.split(",")[device_index])
            bus = pynvml.nvmlDeviceGetPciInfo(pynvml.nvmlDeviceGetHandleByIndex(phys)).busId
            bus = bus.decode() if isinstance(bus, bytes) else bus
            node = int(open("/sys/bus/pci/devices/%s/numa_node" % bus.lower()[-12:]).read().strip())
            info["gpu_numa_node"] = node
            if node >= 0:
                cl = open("/sys/devices/system/node/node%d/cpulist" % node).read().strip()
                cpus = []
                for part in cl.split(","):
                    a, _, b = part.partition("-")
                    cpus.extend(range(int(a), int(b or a) + 1))
                node_cpus = [c for c in cpus if c in set(avail)]
        except Exception:
            node_cpus = None
        n_nodes = len([d for d in os.listdir("/sys/devices/system/node") if d.startswith("node")]) if os.path.isdir("/sys/devices/system/node") else 1
        info["numa_nodes"] = n_nodes
        pool = node_cpus if (node_cpus and n_nodes > 1) else avail
        # ranks that share the pool split it evenly (with one NUMA node: all ranks share all cores)
        sharers = local_world if pool is avail or n_nodes <= 1 else max(1, local_world // n_nodes)
        idx = local_rank % sharers
        per = max(1, len(pool) // sharers)
        mine = pool[idx * per:(idx + 1) * per] or pool
        os.sched_setaffinity(0, mine)
        info.update(bound=True, cores=len(mine), first_core=mine[0])
    except Exception as e:                         # binding is an optimisation, never a requirement
        info["error"] = str(e)[:100]
    return info


def build_world(args, cfg, rank, world, n_generate=None):
    """Reference index, models, quality table and this rank's synthetic text in HBM."""
    import torch
    from mcaller_b200 import engine as eng_mod, models, read_qual, synth, synth_device
    from mcaller_b200.refindex import ReferenceIndex
    reads = cfg["reads"]
    spec = synth.SynthSpec(seed=0, contigs=[(args.contig_name, 4600000)], n_reads=reads * world, len_min=1000, len_max=3000)
    genome = synth.genome(spec, 0)
    seqs = {args.contig_name: genome.tobytes().decode()}
    motif = cfg["motif"]
    base = motif if len(motif) == 1 else "A"
    ref = ReferenceIndex(seqs, base, motif=motif, k=6)
    meth = {0: (synth.meth_sites(spec, 0, ref.site_fwd_bits[:4600000]), synth.meth_sites(spec, 0, ref.site_rev_bits[:4600000]))}
    gen = synth_device.DeviceSynth(spec, ref, meth)
    lo, hi = rank * reads, (rank + 1) * reads
    if n_generate is not None:
        hi = lo + min(n_generate, hi - lo)
    d_text, nbytes, offs = gen.generate(lo, hi - lo)
    torch.cuda.synchronize()
    keys, q = synth_device.quality_table_for(spec, lo, hi)
    qt = read_qual.build_quality_table(dict(zip(keys, q.tolist())))
    model = models.load_model_file(cfg["model"]) if cfg["classifier"] == "NN" else fit_reference_rf()
    e0, e1, two = models.select_models(model, base)
    dm = models.DeviceModels(e0, e1)
    engine = eng_mod.Engine(ref, models=dm, qual_table=qt, skip_thresh=cfg["skip"], qual_thresh=cfg["qual"], two_models=two, histogram=True,
                            dense=True if cfg["scan_dense"] else None)
    return dict(spec=spec, ref=ref, gen=gen, d_text=d_text, nbytes=nbytes, offs=offs, engine=engine, seqs=seqs, lo=lo, hi=hi,
                quals=dict(zip(keys, q.tolist())), model=model, base=base, motif=motif)


# ---- the CPU side: the unmodified reference (oracle/_ref) and the C restatement (oracle/) ------------------------------------

def write_reference_inputs(W, cfg, n_reads, workdir):
    """The first n_reads reads of this rank's text as files the reference CLI can run on: TSV, FASTA, FASTQ, model pickle.
    Returns dict(paths..., sample bytes, read offsets)."""
    import pickle
    from mcaller_b200 import synth
    spec, offs_all = W["spec"], W["offs"].cpu().numpy()
    n_reads = min(n_reads, len(offs_all))
    end = int(offs_all[n_reads]) if n_reads < len(offs_all) else W["nbytes"]
    sample = W["d_text"][:end].cpu().numpy().tobytes()
    p = dict(tsv=os.path.join(workdir, "syn.eventalign.tsv"), fasta=os.path.join(workdir, "ref.fa"), fastq=os.path.join(workdir, "syn.fastq"))
    with open(p["tsv"], "wb") as fh:
        fh.write(sample)
    name = list(W["seqs"])[0]
    seq = W["seqs"][name]
    with open(p["fasta"], "w") as fh:
        fh.write(">%s\n" % name)
        fh.write("\n".join(seq[j:j + 60] for j in range(0, len(seq), 60)) + "\n")
    with open(p["fastq"], "w") as fh:
        for i in range(W["lo"], W["lo"] + n_reads):
            qs, _ = synth.read_quality_string(spec, i)
            fh.write("@%s\n%s\n+\n%s\n" % (synth.read_name(spec, i), "A" * len(qs), qs))
    if cfg["classifier"] == "NN" and cfg["model"] == MODEL:
        p["model"] = cfg["model"]
    else:                                           # fitted RF / {'general'} dict: a pickle the reference's loader accepts
        m = W["model"]
        if isinstance(m, dict) and "general" in m:
            m = m["general"]                        # SURVEY.md Q9: the reference crashes on {'general'} dicts; the bare estimator runs
        p["model"] = os.path.join(workdir, "model.pkl")
        with open(p["model"], "wb") as fh:
            pickle.dump(m, fh)
    p.update(sample=sample, read_offsets=[int(x) for x in offs_all[:n_reads]], n_reads=n_reads, nbytes=end)
    return p


def reference_motif_args(W, cfg, workdir):
    """The reference matches -m literally (str.replace) and cannot take IUPAC motifs (SURVEY.md Q9): those run with the
    equivalent -p positions file (the IUPAC expansion on both strands)."""
    from mcaller_b200 import refmark
    motif = cfg["motif"]
    if all(ch in "ACGT" for ch in motif):
        return dict(motif=motif)
    name = list(W["seqs"])[0]
    seq = W["seqs"][name]
    path = os.path.join(workdir, "positions.txt")
    fwd, rev = refmark.mark_reference(seq, W["base"], motif=motif)
    with open(path, "w") as fh:
        for strand, marked in (("+", fwd), ("-", rev)):
            start = marked.find("M")
            while start >= 0:
                fh.write("%s\t%d\t%s\tm6A\n" % (name, start, strand))
                start = marked.find("M", start + 1)
    return dict(positions=path)


def reference_pass(files, W, cfg, workdir, threads):
    """One run of the unmodified reference CLI on the sample -> (rows, seconds, path of its .diffs file)."""
    from oracle import ref_run
    r = ref_run.run_mcaller(workdir, files["tsv"], files["fasta"], files["fastq"], files["model"], threads=threads, base=W["base"],
                            skip=cfg["skip"], qual=cfg["qual"], classifier=cfg["classifier"], **files["motif_args"])
    if r["rc"] != 0 or r["diffs"] is None:
        raise RuntimeError("reference run failed (rc=%d): %s" % (r["rc"], (r["stdout"][-800:] + r["stderr"][-1500:])))
    with open(r["diffs"], "rb") as fh:
        rows = sum(1 for _ in fh)
    return rows, r["wall_s"], r["diffs"]


def oracle_cap(cfg, nbytes):
    """Row capacity for the oracle: one row per ~85 KB of text for sparse motifs, one per few hundred bytes for -m A."""
    return max(4096, nbytes // (150 if len(cfg["motif"]) == 1 else 2000))


def cpu_oracle_pass(text_bytes, read_offsets, W, cfg, threads):
    """The CPU restatement (oracle/mcaller_oracle.c) over a host sample, read-aligned slices on `threads` host threads.
    Returns (calls, seconds).  Slices are independent files here: each drops its own last open window (reference Q3)."""
    from concurrent.futures import ThreadPoolExecutor
    from oracle import oracle as orc
    orc.lib()
    n = len(read_offsets)
    threads = max(1, min(threads, n))
    bounds = [read_offsets[(n * t) // threads] for t in range(threads)] + [len(text_bytes)]
    mv = memoryview(text_bytes)
    # reference marking, quality table and model are marshalled once (the reference also loads them once per worker)
    prep = orc.prepare(W["seqs"], W["quals"], model=W["model"], base=W["base"], motif=W["motif"])

    def work(t):
        sl = bytes(mv[bounds[t]:bounds[t + 1]])
        r = orc.extract(sl, None, None, k=6, skip_thresh=cfg["skip"], qual_thresh=cfg["qual"], cap=oracle_cap(cfg, len(sl)), count_only=True,
                        prepared=prep)
        return r["counters"]["observations"]

    t0 = time.perf_counter()
    with ThreadPoolExecutor(max_workers=threads) as ex:
        calls = sum(ex.map(work, range(threads)))
    return calls, time.perf_counter() - t0


def gpu_rows_of_sample(W, cfg, files):
    """`.diffs` text of the sample through the public streaming path (HostStreamer + TextSink), as one bytes object."""
    import torch
    from mcaller_b200 import stream as stream_mod
    engine = W["engine"]
    host = torch.frombuffer(bytearray(files["sample"]), dtype=torch.uint8).pin_memory()
    hs = stream_mod.HostStreamer(engine, chunk_bytes=min(1 << 29, max(len(files["sample"]), 1 << 20)))
    cuts = stream_mod.plan_chunks(np.asarray(files["read_offsets"]), len(files["sample"]), hs.chunk_bytes)
    sink = stream_mod.TextSink(W["ref"], 6, W["base"], keep=True)
    engine.reset_histogram()
    hs.run(host, cuts, sink=sink)
    engine.close_carry(-1)                             # end of the file: the last open window is dropped (reference Q3)
    return b"".join(sink.kept)


def parity_check(W, cfg, files, ref_diffs_path):
    """GPU rows of the sample vs (a) the oracle's rows (-t 1 semantics, byte for byte, order included) and (b) the rows the
    unmodified reference just wrote with -t <cores> (its merge sorts and de-duplicates whole lines: compared as sorted
    unique lines).  Label / probability-text agreement is counted on the rows both sides have."""
    from oracle import oracle as orc
    gpu = gpu_rows_of_sample(W, cfg, files)
    want = orc.extract(files["sample"], W["seqs"], W["quals"], k=6, skip_thresh=cfg["skip"], qual_thresh=cfg["qual"], model=W["model"],
                       base=W["base"], motif=W["motif"], cap=oracle_cap(cfg, len(files["sample"])))
    oracle_text = "".join(r + "\n" for r in want["rows"]).encode()
    gpu_rows = gpu.split(b"\n")[:-1]
    out = {"slice_reads": files["n_reads"], "gpu_calls": len(gpu_rows), "oracle_calls": len(want["rows"]),
           "equal": gpu == oracle_text, "what": "`.diffs.6` text of the sample, GPU streaming path vs CPU oracle, byte for byte"}

    def keyed(rows):
        d = {}
        for r in rows:
            f = r.split(b"\t")
            d[(f[0], f[1], f[2], f[5])] = (f[6], f[7]) if len(f) > 7 else (None, None)
        return d
    if ref_diffs_path is not None:
        ref_rows = open(ref_diffs_path, "rb").read().split(b"\n")
        ref_rows = [r for r in ref_rows if r]
        gs, rs = set(gpu_rows), set(ref_rows)
        gk, rk = keyed(gpu_rows), keyed(ref_rows)
        common = [kx for kx in gk if kx in rk]
        lab = sum(1 for kx in common if gk[kx][0] == rk[kx][0])
        prob = sum(1 for kx in common if gk[kx][1] == rk[kx][1])
        out["reference"] = {"rows": len(rs), "gpu_rows": len(gs), "identical_rows": len(gs & rs), "only_gpu": len(gs - rs),
                            "only_reference": len(rs - gs), "set_equal": gs == rs,
                            "label_agreement": (lab / len(common)) if common else None,
                            "prob_text_agreement": (prob / len(common)) if common else None,
                            "what": "unique rows of the unmodified reference (-t cores: workers overlap, merge = sort | uniq) vs unique "
                                    "GPU rows; label = m6A/A at the 0.5 threshold, prob text = np.round(p, 2)"}
    else:
        gk, ok = keyed(gpu_rows), keyed([r.encode() for r in want["rows"]])
        common = [kx for kx in gk if kx in ok]
        out["label_agreement"] = (sum(1 for kx in common if gk[kx][0] == ok[kx][0]) / len(common)) if common else None
    return out


DUMP_BYTES = 64 * 10 ** 6
DUMP_HEADER_BYTES = 128                   # per .npy file


def dump_outputs(engine, cfg, out_dir):
    """Writes what the last timed step computed, as a caller of the step receives it, to out_dir/<name>.npy:
      rows_*  the step's `.diffs` rows (kind MC_CALL, in output order): byte offset of the read in the text, position,
              strand (1 = '-'), the k + 1 features (empty columns are 0 with their bit set in rows_empty_mask), the
              classifier's probability and label (1 = methylated);
      hist_*  the per-site histogram (all-reduced over ranks): depth, methylated calls, first-seen global row index (-1:
              no row), and with BED thresholds in the step the per-site selection flag.
    float64, float32 where every value is a small integer.  Outputs larger than DUMP_BYTES keep a seeded sample of the rows
    and of the site slots (the same entries on every run with the same arguments).  Returns a summary for the JSON line."""
    from mcaller_b200 import _lib, engine as eng_mod
    n_rows = int(engine.d_small[eng_mod.S_NROWS].item())
    rows = engine._bufs["calls"][: n_rows * _lib.CALL_DTYPE.itemsize].cpu().numpy().view(_lib.CALL_DTYPE)
    rows = rows[rows["kind"] == _lib.MC_CALL]
    k1 = 7                                 # -n 6 current differences + the read quality
    f64, f32 = np.float64, np.float32
    row_cols = {"rows_read_offset": (rows["read_off"], f64), "rows_position": (rows["mpos"], f64), "rows_strand": (rows["rev"], f32),
                "rows_features": (rows["feat"][:, :k1], f64), "rows_empty_mask": (rows["empty_mask"], f32),
                "rows_probability": (rows["prob"], f64), "rows_label": (rows["label"], f32)}
    ns = max(engine.ref.n_sites, 1)
    first = engine.d_first.cpu().numpy()
    first = np.where(first == 2 ** 63 - 1, -1, first)
    site_cols = {"hist_depth": (engine.d_depth.cpu().numpy(), f32), "hist_methylated": (engine.d_meth.cpu().numpy(), f32),
                 "hist_first_row": (first, f64)}
    if cfg["bed"]:
        site_cols["hist_bed_selected"] = (engine.d_bed_flags.cpu().numpy(), f32)

    def width(cols):
        return sum(np.dtype(dt).itemsize * int(np.prod(a.shape[1:])) for a, dt in cols.values())
    total = len(rows) * width(row_cols) + ns * width(site_cols)
    budget = DUMP_BYTES - DUMP_HEADER_BYTES * (len(row_cols) + len(site_cols))
    scale = min(1.0, budget / total) if total else 1.0

    def sample(n, seed):
        keep = int(n * scale)
        if keep >= n:
            return np.arange(n)
        return np.sort(np.random.default_rng(seed).choice(n, keep, replace=False))
    os.makedirs(out_dir, exist_ok=True)
    row_idx, site_idx = sample(len(rows), 0), sample(ns, 1)
    for cols, idx in ((row_cols, row_idx), (site_cols, site_idx)):
        for name, (a, dt) in cols.items():
            np.save(os.path.join(out_dir, name + ".npy"), np.ascontiguousarray(a[idx], dtype=dt))
    return {"dir": out_dir, "rows": len(rows), "rows_written": len(row_idx), "sites": ns, "sites_written": len(site_idx)}


_REAL_STDOUT = None


def emit_line(obj):
    """The one JSON line of the contract goes to the real stdout; everything else (NCCL banners, library prints) was
    redirected to stderr at start-up."""
    data = (json.dumps(obj) + "\n").encode()
    if _REAL_STDOUT is None:
        sys.stdout.write(data.decode())
        sys.stdout.flush()
    else:
        os.write(_REAL_STDOUT, data)


def reference_arm(args, cfg, W, host_cores):
    """--impl reference: the unmodified reference CLI on a bounded sample, all host cores, wall clock (imports included)."""
    from oracle import ref_run
    if not ref_run.available():
        try:
            ref_run.build()
        except Exception:
            pass
    workdir = ref_run.scratch_dir()
    try:
        n_s = min(args.cpu_reads, cfg["reads"])
        files = write_reference_inputs(W, cfg, n_s, workdir)
        files["motif_args"] = reference_motif_args(W, cfg, workdir)
        sample_desc = None
        if ref_run.available():
            kind = "reference"
            startup = ref_run.startup_seconds(workdir)
            rows, t, _ = reference_pass(files, W, cfg, workdir, host_cores)                  # warm-up (page cache, .pyc)
            if t * args.steps > args.budget_s and n_s > 500:
                # keep the whole arm within minutes: shrink the sample so that `steps` runs fit the budget
                work_t = max(t - startup, 0.2 * t)
                target = max(args.budget_s / args.steps - startup, 0.5)
                n_s = max(500, int(n_s * min(1.0, target / work_t)))
                files = write_reference_inputs(W, cfg, n_s, workdir)
                files["motif_args"] = reference_motif_args(W, cfg, workdir)
                reference_pass(files, W, cfg, workdir, host_cores)

            def one():
                return reference_pass(files, W, cfg, workdir, host_cores)[:2]
            sample_desc = ("unmodified reference: python mCaller.py -m %s ... -t %d (oracle/_ref) on %d reads (%.2f GB of eventalign TSV) in "
                           "/dev/shm per step; wall clock of the whole process, imports (%.1f s) included"
                           % (cfg["motif"], host_cores, files["n_reads"], files["nbytes"] / 1e9, startup))
        else:
            kind = "port"

            def one():
                return cpu_oracle_pass(files["sample"], files["read_offsets"], W, cfg, host_cores)
            one()
            sample_desc = ("oracle/_ref is absent (run oracle/make_ref.sh where /root/reference exists): C restatement of the reference "
                           "(oracle/mcaller_oracle.c) on %d reads (%.2f GB), %d host threads" % (files["n_reads"], files["nbytes"] / 1e9, host_cores))
        tot_calls, tot_t = 0, 0.0
        for _ in range(args.steps):
            c, t = one()
            tot_calls += c
            tot_t += t
        v = tot_calls / tot_t
        return {"impl": "reference", "metric": METRIC, "value": v, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
                "warmup": 1, "ms_per_step": 1e3 * tot_t / args.steps, "higher_is_better": True, "scaling": "weak",
                "vs_baseline": None, "dtype": "f64", "data": "synthetic",
                "config": {"workload": workload_text(cfg), "sample": sample_desc},
                "cpu_baseline": {"value": v, "unit": UNIT, "cores": host_cores, "kind": kind, "sample": sample_desc},
                "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}, "gpu_launches": 0}
    finally:
        ref_run.cleanup(workdir)


def main():
    global _REAL_STDOUT
    args = parse_args()
    sys.stdout.flush()
    _REAL_STDOUT = os.dup(1)
    os.dup2(2, 1)                       # fd 1 -> stderr for the rest of the run
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    local_world = int(os.environ.get("LOCAL_WORLD_SIZE", str(world)))
    if args.impl == "reference" and rank != 0:
        return 0
    cfg = resolve_config(args, world)
    host_cores = os.cpu_count() or 1
    binding = {"bound": False}
    if args.impl == "ours" and world > 1 and not args.no_bind:
        binding = bind_rank(local_rank, local_world, local_rank)
    import torch
    from mcaller_b200 import dist as mdist, engine as eng_mod, stream as stream_mod
    eng_mod.require_cuda()
    torch.cuda.set_device(local_rank)
    use_dist = world > 1 and args.impl == "ours"
    if use_dist:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))

    W = build_world(args, cfg, rank, 1 if args.impl == "reference" else world,
                    n_generate=min(args.cpu_reads, cfg["reads"]) if args.impl == "reference" else None)
    engine, d_text, nbytes = W["engine"], W["d_text"], W["nbytes"]
    dev = engine.device

    # ------------------------------------------------------------------------------------------------ reference arm
    if args.impl == "reference":
        emit_line(reference_arm(args, cfg, W, host_cores))
        return 0

    # ------------------------------------------------------------------------------------------------ our arm
    scan_pairs = []

    def step(record_scan=False, sync=True):
        """One pass over this rank's text: every stage of the chunk is queued back to back, then the slice-edge window is
        closed with the next rank's first kept line and the histograms are combined -- both consumed on the device, no host
        read.  Warm-up steps read the chunk's status (buffer capacities are learned from it); timed steps do not read
        anything back: K steps are K uninterrupted launch sequences, an overflow would raise the engine's sticky flag."""
        engine.reset_histogram(mdist.rank_row_base(rank))
        if record_scan:
            engine.scan_events = []
        res = None
        if sync:
            res = engine.run_chunk(d_text, nbytes)
        else:
            engine.launch_chunk(d_text, nbytes)
        if use_dist:
            mdist.close_and_reduce(engine, rank, fetch=False)
        else:
            engine.close_carry(-1, fetch=False)          # one rank = the whole file: its last open window is dropped
        if cfg["bed"]:
            engine.bed_select(BED_DEPTH, BED_THRESH)
        if record_scan and engine.scan_events:
            scan_pairs.extend(engine.scan_events)
            engine.scan_events = None
        return res

    for _ in range(max(args.warmup, 3)):
        res = step()
    if use_dist:
        dist.barrier()
    torch.cuda.synchronize()
    engine.overflowed()                 # clear the sticky flag: the warm-up steps grew the buffers where needed
    sampler = ClockSampler(local_rank)
    sampler.start()
    launches0 = engine.launches
    redone0 = engine.redone
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record()
    for _ in range(args.steps):
        step(record_scan=True, sync=False)
    ev1.record()
    torch.cuda.synchronize()
    if use_dist:
        dist.barrier()
    if engine.overflowed():
        raise RuntimeError("a timed step outgrew the buffers learned in the warm-up steps")
    elapsed_ms = ev0.elapsed_time(ev1)
    scan_ms = [a.elapsed_time(b) for a, b in scan_pairs]
    launches = engine.launches - launches0
    clocks = sampler.summary()
    # calls of one step = mass of the (all-reduced) histogram + the rows keyed on the host (every step is the same pass)
    calls_per_step = int(engine.d_depth.sum().item())
    n_odd = torch.tensor([len(engine.odd_rows())], dtype=torch.int64, device=dev)
    bed_loci = int(engine.d_bed_count.item()) if cfg["bed"] else None
    if use_dist:
        t = torch.tensor([elapsed_ms], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        elapsed_ms = float(t[0])
        dist.all_reduce(n_odd, op=dist.ReduceOp.SUM)
    calls_per_step += int(n_odd[0])
    total_calls = calls_per_step * args.steps
    value = total_calls / (elapsed_ms / 1e3)
    dumped = dump_outputs(engine, cfg, args.dump_outputs) if args.dump_outputs and rank == 0 else None

    # N > 1 runs configs[2] while the driver's N = 1 run is configs[1] (fewer calls per byte): so that the scaling of THIS
    # workload can be read off the line, rank 0 also times its own slice alone (no collectives, the other ranks wait)
    solo = None
    if use_dist:
        if rank == 0:
            s0, s1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            s0.record()
            for _ in range(args.steps):
                engine.reset_histogram(0)
                engine.run_chunk(d_text, nbytes)
                engine.close_carry(-1, fetch=False)
                engine.bed_select(BED_DEPTH, BED_THRESH)
            s1.record()
            torch.cuda.synchronize()
            solo_calls = int(engine.d_depth.sum().item()) + len(engine.odd_rows())
            solo = {"value": solo_calls * args.steps / (s0.elapsed_time(s1) / 1e3), "unit": UNIT, "ms_per_step": s0.elapsed_time(s1) / args.steps,
                    "what": "rank 0's slice of the same workload timed alone on one GPU after the multi-GPU region (no collectives)"}
        dist.barrier()

    # roofline of the dominant kernel (k_scan): algorithmic bytes = the text once + 32 B per record written
    peak, peak_src = measured_peak_hbm()
    alg_bytes = nbytes + 32 * res.n_records
    scan_avg_ms = float(np.mean(scan_ms)) if scan_ms else None
    achieved = alg_bytes / (scan_avg_ms / 1e3) / 1e9 if scan_avg_ms else None
    roofline = {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": (achieved / peak) if achieved else None,
                "traffic": None, "kernel": "k_scan", "kernel_ms": scan_avg_ms, "algorithmic_bytes": alg_bytes, "peak_source": peak_src,
                "step_frac": (alg_bytes / (elapsed_ms / args.steps / 1e3) / 1e9 / peak) if elapsed_ms else None}
    tr = os.path.join(ROOT, "profiles", "k_scan_traffic.json")
    if os.path.exists(tr) and cfg["index"] == 1 and not args.motif:
        try:
            roofline["traffic"] = json.load(open(tr)).get("dram_bytes_per_launch_at_bench_size")
        except Exception:
            pass

    # ------------------------------------------------------------------------------------------------ e2e leg
    e2e = None
    if not args.no_e2e:
        offs_all = W["offs"].cpu().numpy()
        n_e = int(np.searchsorted(offs_all, args.e2e_bytes, side="right"))
        n_e = max(1, min(n_e, len(offs_all)))
        end = int(offs_all[n_e]) if n_e < len(offs_all) else nbytes
        host = torch.empty(end, dtype=torch.uint8, pin_memory=True)
        host.copy_(d_text[:end])
        torch.cuda.synchronize()
        # concurrent H2D ceiling of this box: every rank copies from its pinned buffer at the same time, back to back for the
        # whole window (a sustained figure, like the streaming leg it is compared with -- not the best single copy)
        probe_n = min(end, 2 << 30)
        dst = torch.empty(probe_n, dtype=torch.uint8, device=dev)
        dst.copy_(host[:probe_n], non_blocking=True)               # warm-up
        torch.cuda.synchronize()
        if use_dist:
            dist.barrier()
        probe_reps = 4
        t0 = time.perf_counter()
        for _ in range(probe_reps):
            dst.copy_(host[:probe_n], non_blocking=True)
        torch.cuda.synchronize()
        best = probe_reps * probe_n / (time.perf_counter() - t0) / 1e9
        del dst
        ceil_t = torch.tensor([best], dtype=torch.float64, device=dev)
        ceil_min = ceil_t.clone()
        if use_dist:
            dist.all_reduce(ceil_t, op=dist.ReduceOp.SUM)
            ceil_t /= world
            dist.all_reduce(ceil_min, op=dist.ReduceOp.MIN)
        h2d_ceiling, h2d_ceiling_min = float(ceil_t[0]), float(ceil_min[0])
        streamer = stream_mod.HostStreamer(engine, chunk_bytes=min(args.e2e_chunk, max(end, 1 << 20)))
        cuts = stream_mod.plan_chunks(offs_all[:n_e], end, streamer.chunk_bytes)
        fmt_threads = binding.get("cores", 0) if binding.get("bound") else 0
        sink = stream_mod.TextSink(W["ref"], 6, W["base"], max_threads=fmt_threads)      # rows rendered as .diffs text on host threads

        def e2e_pass():
            engine.reset_histogram(mdist.rank_row_base(rank))
            tot = streamer.run(host, cuts, sink=sink)
            if use_dist:
                row = mdist.close_and_reduce(engine, rank)
            else:
                row = engine.close_carry(-1)
            sink.render(row.view(np.uint8), 1, 0)          # the slice-edge row, completed by the next rank (nothing on one GPU)
            if cfg["bed"]:
                engine.bed_select(BED_DEPTH, BED_THRESH)
            return tot["calls"] + int(row[0]["kind"] == 0)
        e2e_pass()                                                 # warm-up (buffer growth, pinned result buffers)
        streamer.h2d_bytes = streamer.d2h_bytes = 0
        sink.text_bytes = 0
        sink.render_seconds = 0.0
        if use_dist:
            dist.barrier()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        e_calls = 0
        e_steps = args.steps
        for _ in range(e_steps):
            e_calls += e2e_pass()
        torch.cuda.synchronize()
        dt = time.perf_counter() - t0
        dt_fastest = dt
        if use_dist:
            t = torch.tensor([dt], dtype=torch.float64, device=dev)
            tmin = t.clone()
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            dist.all_reduce(tmin, op=dist.ReduceOp.MIN)
            dt, dt_fastest = float(t[0]), float(tmin[0])
            c = torch.tensor([e_calls], dtype=torch.int64, device=dev)
            dist.all_reduce(c, op=dist.ReduceOp.SUM)
            e_calls = int(c[0])
        h2d_rate = streamer.h2d_bytes / dt / 1e9
        e2e = {"value": e_calls / dt, "unit": UNIT, "h2d_bytes_per_step": streamer.h2d_bytes // e_steps,
               "d2h_bytes_per_step": streamer.d2h_bytes // e_steps, "diffs_text_bytes_per_step": sink.text_bytes // e_steps,
               "host_writer_ms_per_step": 1e3 * sink.render_seconds / e_steps, "ms_per_step": 1e3 * dt / e_steps,
               "ms_per_step_fastest_rank": 1e3 * dt_fastest / e_steps,
               "h2d_gbs_per_gpu": h2d_rate, "h2d_ceiling_gbs_per_gpu": h2d_ceiling, "h2d_ceiling_slowest_rank_gbs": h2d_ceiling_min,
               "h2d_frac_of_ceiling": (h2d_rate / h2d_ceiling) if h2d_ceiling else None,
               "h2d_frac_of_slowest_rank_ceiling": (h2d_rate / h2d_ceiling_min) if h2d_ceiling_min else None,
               "sample": "%d reads (%.2f GB TSV) per GPU streamed from pinned host memory in %d chunks, rows copied back and "
                         "rendered as .diffs text by the native writer; ceiling = mean (and slowest rank) over ranks of %d back-to-back "
                         "pinned->device copies of %.1f GB, all %d ranks copying at once; the step ends with the slowest rank" % (n_e, end / 1e9, len(cuts), probe_reps, probe_n / 1e9, world)}
        del host

    # ------------------------------------------------------------------------------------------------ CPU baseline + parity
    cpu = parity = None
    if rank == 0 and world == 1 and not args.no_cpu:
        from oracle import ref_run
        if not ref_run.available():
            try:
                ref_run.build()
            except Exception:
                pass
        workdir = ref_run.scratch_dir()
        try:
            n_s = min(args.cpu_reads, cfg["reads"])
            files = write_reference_inputs(W, cfg, n_s, workdir)
            files["motif_args"] = reference_motif_args(W, cfg, workdir)
            cpu_oracle_pass(files["sample"], files["read_offsets"], W, cfg, host_cores)          # warm-up pass
            p_calls, p_t = cpu_oracle_pass(files["sample"], files["read_offsets"], W, cfg, host_cores)
            port = {"value": p_calls / p_t, "unit": UNIT, "cores": host_cores, "kind": "port",
                    "sample": "C restatement of the reference (oracle/mcaller_oracle.c), %d host threads, %.1f s" % (host_cores, p_t)}
            ref_diffs = None
            if ref_run.available():
                startup = ref_run.startup_seconds(workdir)
                r_rows, r_t, ref_diffs = reference_pass(files, W, cfg, workdir, host_cores)
                cpu = {"value": r_rows / r_t, "unit": UNIT, "cores": host_cores, "kind": "reference",
                       "sample": "unmodified reference: python mCaller.py -m %s ... -t %d (oracle/_ref) on %d reads (%.2f GB TSV) in /dev/shm, "
                                 "one run, %.1f s wall clock of the whole process, imports (%.1f s) included"
                                 % (cfg["motif"], host_cores, files["n_reads"], files["nbytes"] / 1e9, r_t, startup),
                       "port": port}
            else:
                cpu = dict(port, sample="oracle/_ref absent; " + port["sample"])
            parity = parity_check(W, cfg, files, ref_diffs)
        finally:
            ref_run.cleanup(workdir)

    if rank == 0:
        line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3),
                "ms_per_step": elapsed_ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
                "dtype": "f64", "data": "synthetic",
                "config": {"workload": workload_text(cfg, nbytes, world),
                           "l2": "inputs (%.1f GB) larger than L2 (126 MB); no flush needed" % (nbytes / 1e9),
                           "parallelism": "reads sharded over %d GPU(s); slice-edge window closed across ranks + one SUM and one MIN "
                                          "all-reduce of the per-site histogram per step" % world,
                           "calls_per_step": calls_per_step, "lines_per_step_per_gpu": res.counters["lines"],
                           "records_per_step_per_gpu": res.n_records, "bed_loci": bed_loci, "single_gpu_same_workload": solo, "chunks_redone": engine.redone - redone0,
                           "binding": binding},
                "clocks": clocks, "e2e": e2e, "gpu_launches": launches, "roofline": roofline, "cpu_baseline": cpu,
                "parity_check": parity}
        if dumped:
            line["outputs_dumped"] = dumped
        emit_line(line)
    if use_dist:
        dist.destroy_process_group()
    if parity is not None and not parity["equal"]:
        sys.stderr.write("bench.py: GPU rows differ from the oracle on the shared sample\n")
        return 3
    return 0


if __name__ == "__main__":
    sys.exit(main())
