"""Command lines with the reference's flags (mCaller.py:122-141, make_bed.py:169-182) on top of the GPU path.

    python -m mcaller_b200.cli mCaller  -m GATC -r ref.fa -e x.eventalign.tsv -f x.fastq -d model.pkl -b A
    python -m mcaller_b200.cli make_bed -f x.eventalign.diffs.6 -d 15 -t 0.5
    python -m mcaller_b200.cli mCaller --train -p labelled_positions.txt -r ref.fa -e x.eventalign.tsv -f x.fastq -b A -c NN

The reference's own mCaller.py / make_bed.py can be used unchanged instead (INTEGRATION.md); these entry points exist
so the path can be run where the reference checkout is absent.  `-t N` splits the TSV into N read-aligned byte ranges
like the reference (mCaller.py:63-68); range i is handled on GPU i mod n_gpus, one after another in this process.
`--gpus N` (extension) runs N ranks at once, one process per GPU (mcaller_b200.multigpu): rows are written per rank and
concatenated, the per-site histograms are all-reduced over NCCL, and with `--bed` rank 0 writes make_bed.py's BED / GFF
straight from the combined histogram (`--bed_min_read_depth`, `--bed_mod_threshold`, `--bed_control`, `--bed_gff`,
`--bed_ref` mirror make_bed.py's -d / -t / --control / --gff / --ref).  `--bed_vo` and `--bed_positions FILE` mirror
make_bed.py's per-read modes --vo and -p FILE: the ranks keep the rows of each locus on the device and rank 0 writes the
probability lists and per-column t-tests from them, again without any `.diffs` text.
"""
import os
import sys
from argparse import ArgumentParser


def mcaller_main(argv=None):
    from . import extract_contexts as ec, multigpu, read_qual, refmark
    p = ArgumentParser(description="Classify bases as methylated or unmethylated", prog="mCaller")
    g = p.add_mutually_exclusive_group(required=True)
    g.add_argument("-p", "--positions", type=str)
    g.add_argument("-m", "--motif", type=str)
    p.add_argument("-r", "--reference", type=str, required=True)
    p.add_argument("-e", "--tsv", type=str, required=True)
    p.add_argument("-f", "--fastq", type=str, required=True)
    p.add_argument("-t", "--threads", type=int, default=1)
    p.add_argument("-b", "--base", type=str, default="A")
    p.add_argument("-n", "--num_variables", type=int, default=6)
    p.add_argument("--train", action="store_true", default=False)
    p.add_argument("--training_tsv", type=str)
    p.add_argument("-d", "--modelfile", type=str)
    p.add_argument("-s", "--skip_thresh", type=int, default=0)
    p.add_argument("-q", "--qual_thresh", type=float, default=0)
    p.add_argument("-c", "--classifier", type=str, default="NN")
    p.add_argument("--plot_training", action="store_true", default=False)
    p.add_argument("-v", "--version", action="version", version="%(prog)s v1.0 (mcaller_b200)")
    p.add_argument("--gpus", type=int, default=0, help="run N ranks, one process per GPU (0: single process, -t ranges in turn)")
    p.add_argument("--bed", action="store_true", help="with --gpus: write the make_bed.py summary from the all-reduced histogram")
    p.add_argument("--bed_min_read_depth", type=int, default=15)
    p.add_argument("--bed_mod_threshold", type=float, default=0.5)
    p.add_argument("--bed_control", action="store_true")
    p.add_argument("--bed_gff", action="store_true")
    p.add_argument("--bed_ref", type=str)
    p.add_argument("--bed_vo", action="store_true", help="with --gpus --bed: make_bed.py --vo (per-locus probability lists)")
    p.add_argument("--bed_positions", type=str, help="with --gpus --bed: make_bed.py -p FILE (listed loci, per-column t-tests)")
    p.add_argument("--seed", type=int, default=0, help="random_state of the training's balancing, folds and fits")
    a = p.parse_args(argv)
    if (a.bed_vo or a.bed_positions) and not (a.gpus and a.gpus > 0 and a.bed):
        p.error("--bed_vo and --bed_positions need --gpus N --bed")
    if a.bed_positions:
        assert os.path.isfile(a.bed_positions), "positions file not found at " + a.bed_positions
    if a.base == "A":
        mod = "m6A"
    elif a.base == "C":
        mod = "m5C"
    else:
        print("classification only available for A or C bases so far")
        return 0
    if a.train or a.training_tsv:
        return _train_main(p, a, mod)
    modelfile = a.modelfile or (os.path.dirname(os.path.realpath(sys.argv[0])) + "/model_" + a.classifier + "_" + str(a.num_variables) + "_" + mod + ".pkl")
    assert os.path.isfile(modelfile), "model file not found at " + modelfile
    base = a.motif if (a.motif and len(a.motif) == 1) else a.base
    assert a.skip_thresh < a.num_variables / 2, "too many skips with only " + str(a.num_variables) + " variables - try < half"
    assert os.path.isfile(a.fastq), "fastq file not found at " + a.fastq
    k = a.num_variables
    if a.gpus and a.gpus > 0:
        print("%d contigs" % len(refmark.read_fasta(a.reference)))
        print("%d GPUs" % a.gpus)
        multigpu.run(dict(tsv=a.tsv, reference=a.reference, fastq=a.fastq, modelfile=modelfile, k=k, skip=a.skip_thresh, qual=a.qual_thresh,
                          base=base, motif=a.motif, positions=a.positions, bed=a.bed, bed_depth=a.bed_min_read_depth,
                          bed_thresh=a.bed_mod_threshold, bed_control=a.bed_control, bed_gff=a.bed_gff, bed_ref=a.bed_ref,
                          bed_vo=a.bed_vo, bed_positions=a.bed_positions), a.gpus)
        print("Finished extracting signals")
        return 0
    read2qual = read_qual.extract_read_quality_device(a.fastq)        # FASTQ scanned on the GPU (same mapping as read_qual.py)
    print("%d contigs" % len(refmark.read_fasta(a.reference)))
    print("%d threads" % a.threads)
    ranges = multigpu.byte_ranges(os.path.getsize(a.tsv), max(1, a.threads))
    for start, end in ranges:
        tmp = multigpu.ec_tmp_name(a.tsv, k, start)
        if os.path.exists(tmp):
            os.remove(tmp)                       # the reference appends to stale files (quirk Q7); we start clean
        ec.extract_features(a.tsv, a.reference, read2qual, k, a.skip_thresh, a.qual_thresh, modelfile, a.classifier, start,
                            endline=end, train=False, base=base, motif=a.motif, positions_list=a.positions)
    print("Finished extracting signals")
    multigpu.merge_outputs(a.tsv, k, len(ranges))
    return 0


def _train_main(p, a, mod):
    """--train: labelled windows -> `<prefix>.diffs.<k>.train` -> model fit -> pickle; --training_tsv: fit on an existing
    `.train` file (INTEGRATION.md, "Training")."""
    import pickle
    from . import extract_contexts as ec, multigpu, read_qual, refmark, train as tr
    if a.classifier in ("RF", "LR"):
        raise NotImplementedError("-c %s training is not supported: the reference's RandomForest / LogisticRegression settings "
                                  "are rejected by scikit-learn 1.9" % a.classifier)
    if a.classifier not in ("NN", "NBC"):
        p.error("-c must be NN, NBC, RF or LR")
    if a.plot_training:
        raise NotImplementedError("--plot_training: training plots are not produced")
    if a.gpus:
        raise NotImplementedError("--train runs in one process; --gpus applies to calling only")
    k = a.num_variables
    out = a.modelfile or "model_%s_%d_%s.pkl" % (a.classifier, k, mod)
    if a.training_tsv:
        assert os.path.isfile(a.training_tsv), "training file not found at " + a.training_tsv
        sites, x, labels, ctxs = tr.read_train_tsv(a.training_tsv)
        keys = tr.keys_from_contexts(ctxs, a.base, k)
    else:
        if not a.positions:
            p.error("--train needs labelled positions (-p, 4th column: label), not a motif")
        pos_label = {}
        with open(a.positions) as fh:
            for ln in fh:
                f = ln.split()
                if not f:
                    continue
                if len(f) < 4:
                    p.error("--train: %s has no label column (contig, position, strand, label)" % a.positions)
                pos_label[(f[0], int(f[1]), f[2])] = f[3]
        assert a.skip_thresh < k / 2, "too many skips with only " + str(k) + " variables - try < half"
        assert os.path.isfile(a.fastq), "fastq file not found at " + a.fastq
        read2qual = read_qual.extract_read_quality_device(a.fastq)
        print("%d contigs" % len(refmark.read_fasta(a.reference)))
        print("%d threads" % a.threads)
        ranges = multigpu.byte_ranges(os.path.getsize(a.tsv), max(1, a.threads))
        keys = []
        for start, end in ranges:
            tmp = ec.diffs_name(a.tsv, k, start, train=True)
            if os.path.exists(tmp):
                os.remove(tmp)
            run = ec.RangeRun(a.tsv, a.reference, read2qual, k, a.skip_thresh, a.qual_thresh, None, start, endline=end, train=True,
                              pos_label=pos_label, base=a.base, positions_list=a.positions)
            run.stream()
            run.close_by_probe()
            run.print_counters()
            keys += run.fmt.keys
        print("Finished extracting signals")
        sites, x, labels, _ = tr.read_train_tsv(multigpu.merge_outputs(a.tsv, k, len(ranges), train=True))
        if len(keys) != len(labels):
            raise RuntimeError("%d rows written, %d model keys" % (len(labels), len(keys)))
    model = tr.train(tr.TrainRows(sites, x, labels, keys), a.classifier, a.seed, mod, ["MG", "MH"] if a.base == "A" else ["general"])
    with open(out, "wb") as fh:
        pickle.dump(model, fh)
    print("model written to %s" % out)
    return 0


def make_bed_main(argv=None):
    from . import make_bed as mb
    p = ArgumentParser(description="Produce bed file of methylated positions based on mCaller output")
    p.add_argument("-d", "--min_read_depth", type=int, default=15)
    p.add_argument("-t", "--mod_threshold", type=float, default=0.5)
    p.add_argument("-f", "--mCaller_file", type=str, required=True)
    p.add_argument("-p", "--positions", type=str)
    p.add_argument("--control", action="store_true")
    p.add_argument("--gff", action="store_true")
    p.add_argument("--ref", type=str)
    p.add_argument("--plot", action="store_true")
    p.add_argument("--plotsummary", action="store_true")
    p.add_argument("--plotdir", type=str, default="mCaller_position_plots")
    p.add_argument("--vo", action="store_true")
    a = p.parse_args(argv)
    assert os.path.isfile(a.mCaller_file), "file not found at " + a.mCaller_file
    out = mb.output_name(a.mCaller_file, a.positions, a.control, a.gff)
    print(a.mCaller_file)
    mb.aggregate_by_pos(a.mCaller_file, out, a.min_read_depth, a.mod_threshold, a.positions, a.control, a.vo, a.gff, a.ref, a.plot,
                        a.plotdir, a.plotsummary)
    return 0


if __name__ == "__main__":
    if len(sys.argv) < 2 or sys.argv[1] not in ("mCaller", "make_bed"):
        sys.exit("usage: python -m mcaller_b200.cli {mCaller|make_bed} [flags of the reference CLI]")
    sys.exit(mcaller_main(sys.argv[2:]) if sys.argv[1] == "mCaller" else make_bed_main(sys.argv[2:]))
