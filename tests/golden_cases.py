"""Shared table of golden cases + deterministic input builders.

Used by tools/make_golden.py (build container: runs the real reference on these inputs) and by
the tests (any box: rebuild the same inputs, run oracle / CUDA path, compare with the stored
reference outputs in tests/golden/<case>.json).
"""
import gzip
import os
import random

import numpy as np

from mcaller_b200 import refmark, synth

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")

_SPEC3 = dict(seed=11, contigs=[("ctgA", 6000), ("ctgB", 5000), ("ctgC", 4500)], n_reads=60, len_min=300, len_max=900, header=True)
_SPEC_A = dict(seed=12, contigs=[("c1", 1500), ("c2", 1500)], n_reads=10, len_min=150, len_max=300)
_SPEC_G = dict(seed=13, contigs=[("chrG", 8000)], n_reads=40, len_min=300, len_max=700)
_SPEC_P = dict(seed=14, contigs=[("p1", 5000), ("p2", 4000)], n_reads=40, len_min=300, len_max=800, header=True)

R95 = "r95_twobase_model_NN_6_m6A.pkl"
R94 = "r94_model_NN_6_m6A.pkl"
CAAY_BARE = "CAAY_bare_model_6_m6A.pkl"

CASES = {
    # reference's own fixture (README.md:132 command) and the survey's extra regression run
    "masonread1_p": dict(fixture="masonread1", positions="test_positions_m6A.txt", model=R95, base="A"),
    "masonread1_gatc": dict(fixture="masonread1", motif="GATC", model=R95, base="A"),
    "masonread1_gatc_s2": dict(fixture="masonread1", motif="GATC", model=R95, base="A", s=2),
    # synthetic, three contigs + header line, methylation signal on half the sites
    "gatc_s0": dict(spec=_SPEC3, motif="GATC", model=R95, base="A", meth=True,
                    beds=[["-d", "1", "-t", "0.5"], ["-d", "3", "-t", "0.3"], ["-d", "1", "-t", "0.5", "--gff"],
                          ["-d", "2", "-t", "0.4", "--ref", "ref.fasta"], ["-d", "1", "-t", "0.6", "--control", "--gff", "--ref", "ref.fasta"],
                          ["-d", "1", "-t", "0.5", "--vo"], ["-d", "2", "-t", "0.4", "--gff", "--vo"],
                          ["-d", "1", "-t", "0.5", "-p", "bedpos.txt"], ["-d", "1", "-t", "0.5", "-p", "bedpos.txt", "--vo"]]),
    "gatc_s1": dict(spec=_SPEC3, motif="GATC", model=R95, base="A", meth=True, s=1),
    "gatc_s2": dict(spec=_SPEC3, motif="GATC", model=R95, base="A", meth=True, s=2,
                    beds=[["-d", "2", "-t", "0.5"], ["-d", "2", "-t", "0.5", "--control"], ["-d", "2", "-t", "0.5", "-p", "bedpos.txt"]]),
    # dense multi-M windows (every A is a target), reads truncated so windows stay open across reads/contigs
    "A_s0": dict(spec=_SPEC_A, motif="A", model=R95, base="A", post="truncate"),
    "A_s2": dict(spec=_SPEC_A, motif="A", model=R95, base="A", s=2, post="truncate"),
    "gaa_s1": dict(spec=_SPEC_G, motif="GAA", model=R95, base="A", s=1),
    "gaa_s2": dict(spec=_SPEC_G, motif="GAA", model=R95, base="A", s=2),
    # positions file on both strands
    "pos_p": dict(spec=_SPEC_P, positions="random", model=R95, base="A", s=1),
    # read-quality filter
    "gatc_q": dict(spec=_SPEC3, motif="GATC", model=R95, base="A", meth=True, q=13.5),
    # read-quality filter where it matters: reads of three contigs in random order, cut short so that windows stay open at read
    # ends, half of the reads below the threshold -- a window is then closed by the first kept line of the next read that
    # PASSES and takes that line's contig (extract_contexts.py:167 before :179, :214)
    "gat_q_handoff": dict(spec=dict(seed=31, contigs=[("ctgA", 5000), ("ctgB", 4000), ("ctgC", 3000)], n_reads=90, len_min=40, len_max=160),
                          motif="GAT", model=R95, base="A", s=1, q=13.5, post="truncate", shuffle=9),
    # the same with every A a target: each read ends inside an open window
    "A_q_handoff": dict(spec=dict(seed=32, contigs=[("c1", 1500), ("c2", 1200), ("c3", 900)], n_reads=30, len_min=60, len_max=200),
                        motif="A", model=R95, base="A", s=2, q=13.5, post="truncate", shuffle=4),
    # malformed / odd lines
    "adversarial": dict(spec=_SPEC3, motif="GATC", model=R95, base="A", meth=True, s=1, post="adversarial"),
    # bare estimator pickles -> 'general' model path
    "bare_r94": dict(spec=_SPEC3, motif="GATC", model=R94, base="A", meth=True),
    "bare_caay_p": dict(spec=_SPEC_P, positions="random", model=CAAY_BARE, base="A"),
    # cytosine targets
    "cg_c": dict(spec=_SPEC_G, motif="CG", model=R94, base="C", s=1),
    # the reference's alternative classifiers (-c RF / LR / NBC; pickles fitted by tools/make_alt_models.py, the reference
    # ships none): tree-walk, linear and naive-Bayes kernels pinned against the reference end to end
    "rf_gatc": dict(spec=_SPEC3, motif="GATC", model="alt_RF_6_m6A.pkl.gz", base="A", meth=True, s=1, classifier="RF"),
    "lr_gatc": dict(spec=_SPEC3, motif="GATC", model="alt_LR_6_m6A.pkl", base="A", meth=True, classifier="LR"),
    "nbc_gatc": dict(spec=_SPEC3, motif="GATC", model="alt_NBC_6_m6A.pkl", base="A", meth=True, classifier="NBC"),
}


# A case large enough for multi-chunk streaming (>= 10^3 reads, ~0.6 GB of TSV): the reference's outputs are stored as row
# counts + sha256 (tools/make_golden.py), the inputs are regenerated on the GPU by the device generator (bit-identical to the
# host generator, see test_device_generator_matches_numpy_generator)
BIG_CASES = {
    "gatc_1k_s1": dict(spec=dict(seed=21, contigs=[("ecoli", 600000)], n_reads=1200, len_min=1000, len_max=3000), motif="GATC",
                       model=R95, base="A", meth=True, s=1, beds=[["-d", "2", "-t", "0.5"], ["-d", "3", "-t", "0.3", "--control"]]),
}


def _fixture_fasta(tsv_bytes, length, out_path):
    """Rebuild the missing assembly FASTA: N everywhere except what TSV column 3 pins (SURVEY.md 8c)."""
    seq = bytearray(b"N" * length)
    for ln in tsv_bytes.split(b"\n"):
        f = ln.split(b"\t")
        if len(f) < 3:
            continue
        p = int(f[1])
        seq[p:p + len(f[2])] = f[2]
    with open(out_path, "w") as fh:
        fh.write(">ecoli\n")
        s = seq.decode()
        fh.write("\n".join(s[i:i + 60] for i in range(0, length, 60)) + "\n")


def _post_truncate(lines, seed):
    """Cut each read at a random line so that windows are left open at read ends."""
    rnd = random.Random(seed)
    out, cur, cur_name = [], [], None
    def flush():
        if cur:
            keep = rnd.randint(max(1, len(cur) // 2), len(cur))
            out.extend(cur[:keep])
    for ln in lines:
        f = ln.split("\t")
        nm = f[3] if len(f) > 3 else None
        if nm != cur_name:
            flush()
            cur, cur_name = [], nm
        cur.append(ln)
    flush()
    return out


def _post_adversarial(lines, seed):
    rnd = random.Random(seed)
    out = []
    for i, ln in enumerate(lines):
        r = rnd.random()
        f = ln.split("\t")
        if len(f) < 13 or f[0] == "contig":
            out.append(ln)
            continue
        if r < 0.01:
            out.append("\t".join(f[:5]))                      # short line (<12 fields) -> dropped
        elif r < 0.02:
            out.append("\t".join(["ghost"] + f[1:]))          # unknown contig -> dropped, state untouched
        elif r < 0.03:
            out.append(ln + "\t1.5,2.5,3.5")                  # extra samples column
        elif r < 0.04:
            out.append(f[0] + "\t\t" + "\t".join(f[1:]))      # doubled tab collapses in str.split()
        elif r < 0.05:
            out.append(ln + " ")                              # trailing blank (a CR would hang the reference:
                                                              # its char count never reaches the byte size, :144-148)
        elif r < 0.055:
            out.append("")                                    # empty line
        elif r < 0.065:
            out.append("\t".join(f[:12]))                     # exactly 12 fields (minimum accepted)
        elif r < 0.075:
            out.append("\t".join(f[:11]))                     # 11 fields -> dropped
        elif r < 0.085:
            continue                                          # line deleted (position gaps / event gaps)
        out.append(ln)
    return out


POSTS = {"truncate": _post_truncate, "adversarial": _post_adversarial}


def _random_positions(spec, genomes, seed, frac=0.04):
    rnd = random.Random(seed)
    rows = []
    for ci, (nm, ln) in enumerate(spec.contigs):
        g = genomes[ci]
        for p in range(12, ln - 12):
            if g[p] == 65 and rnd.random() < frac:
                rows.append((nm, p, "+"))
            elif g[p] == 84 and rnd.random() < frac:
                rows.append((nm, p, "-"))
    return rows


def build_inputs(case, outdir, models_dir=None):
    """Write tsv / fasta / fastq / (positions) for `case` into outdir; return dict of paths."""
    models_dir = models_dir or os.path.join(GOLD, "models")
    paths = {"tsv": os.path.join(outdir, "syn.eventalign.tsv"), "fasta": os.path.join(outdir, "ref.fasta"),
             "fastq": os.path.join(outdir, "syn.fastq"), "model": os.path.join(models_dir, case["model"])}
    if case["model"].endswith(".gz"):                      # large pickles are stored compressed; the runs read the plain file
        paths["model"] = os.path.join(outdir, case["model"][:-3])
        with gzip.open(os.path.join(models_dir, case["model"]), "rb") as src, open(paths["model"], "wb") as dst:
            dst.write(src.read())
    if "fixture" in case:
        fx = os.path.join(GOLD, case["fixture"])
        tsv = gzip.open(os.path.join(fx, "masonread1.eventalign.tsv.gz"), "rb").read()
        with open(paths["tsv"], "wb") as fh:
            fh.write(tsv)
        _fixture_fasta(tsv, 4734145, paths["fasta"])
        with open(paths["fastq"], "w") as fh:
            fh.write(open(os.path.join(fx, "masonread1.fastq")).read())
        if case.get("positions"):
            paths["positions"] = os.path.join(outdir, "positions.txt")
            with open(paths["positions"], "w") as fh:
                fh.write(open(os.path.join(fx, case["positions"])).read())
        return paths
    spec = synth.SynthSpec(**case["spec"])
    genomes = [synth.genome(spec, ci) for ci in range(len(spec.contigs))]
    base = case.get("base", "A")
    if case.get("positions") == "random":
        rows = _random_positions(spec, genomes, spec.seed + 1000)
        paths["positions"] = os.path.join(outdir, "positions.txt")
        with open(paths["positions"], "w") as fh:
            for nm, p, st in rows:
                fh.write("%s\t%d\t%s\tm6A\n" % (nm, p, st))
    site_maps = None
    if case.get("meth"):
        site_maps = {}
        for ci, (nm, ln) in enumerate(spec.contigs):
            seq = genomes[ci].tobytes().decode()
            fwd, rev = refmark.mark_reference(seq, base, motif=case.get("motif"), positions_file=paths.get("positions"), contig=nm)
            site_maps[ci] = (synth.meth_sites(spec, ci, refmark.site_bitmap(fwd)),
                             synth.meth_sites(spec, ci, refmark.site_bitmap(rev)))
    order = None
    if case.get("shuffle") is not None:                      # reads in random order instead of contig by contig
        order = list(range(spec.n_reads))
        random.Random(case["shuffle"]).shuffle(order)
    tsv, fasta, fastq, _ = synth.generate(spec, site_maps, reads=order)
    if case.get("post"):
        lines = tsv.decode().split("\n")
        if lines and lines[-1] == "":
            lines.pop()
        lines = POSTS[case["post"]](lines, spec.seed + 77)
        tsv = ("\n".join(lines) + "\n").encode()
    with open(paths["tsv"], "wb") as fh:
        fh.write(tsv)
    with open(paths["fasta"], "w") as fh:
        fh.write(fasta)
    with open(paths["fastq"], "w") as fh:
        fh.write(fastq)
    return paths


def cli_args(case, inputs):
    """Argument vector of the reference CLI (mCaller.py:122-141) for this case."""
    a = []
    if case.get("positions"):
        a += ["-p", inputs["positions"]]
    else:
        a += ["-m", case["motif"]]
    a += ["-r", inputs["fasta"], "-e", inputs["tsv"], "-f", inputs["fastq"], "-d", inputs["model"],
          "-b", case.get("base", "A"), "-n", str(case.get("k", 6))]
    if case.get("s"):
        a += ["-s", str(case["s"])]
    if case.get("q"):
        a += ["-q", str(case["q"])]
    if case.get("classifier"):
        a += ["-c", case["classifier"]]
    return a


def write_bed_positions(diffs_text, path):
    """Positions file for `make_bed.py -p` derived from a `.diffs` text: every second locus in first-seen order
    (chrom, start, start+1, strand), one entry whose end column is wrong (never matches, make_bed.py:83-84), one unknown
    contig and one short line (skipped by make_pos_set, make_bed.py:17)."""
    seen, order = set(), []
    for ln in diffs_text.split("\n"):
        f = ln.split("\t")
        if len(f) < 7:
            continue
        key = (f[0], f[2], f[5])
        if key not in seen:
            seen.add(key)
            order.append(key)
    with open(path, "w") as fh:
        for i, (chrom, pos, strand) in enumerate(order):
            if i % 2 == 0:
                fh.write("%s\t%s\t%d\t%s\n" % (chrom, pos, int(pos) + 1, strand))
            elif i % 7 == 1:
                fh.write("%s\t%s\t%d\t%s\n" % (chrom, pos, int(pos) + 2, strand))
        fh.write("nosuchcontig\t10\t11\t+\n")
        fh.write("x\n")


# ---- make_bed-only golden: deep coverage (pairwise-summation paths of the t-tests, 17-digit and scientific-notation values) ----
BED_DEEP_VARIANTS = [["-d", "1", "-t", "0.5", "-p", "bedpos.txt"], ["-d", "1", "-t", "0.5", "-p", "bedpos.txt", "--vo"],
                     ["-d", "1", "-t", "0.5", "--vo"], ["-d", "5", "-t", "0.3", "--gff", "--vo"], ["-d", "5", "-t", "0.3", "--gff"]]


def deep_diffs_text(seed=7):
    """Deterministic `.diffs.6` text with loci of depth 1..520, rows interleaved across loci, feature text as repr(float64)."""
    import random
    rng = random.Random(seed)
    depths = [1, 2, 3, 5, 7, 8, 9, 15, 16, 17, 23, 24, 64, 127, 128, 129, 130, 136, 255, 256, 257, 300, 400, 520]
    rows = []
    for li, depth in enumerate(depths):
        chrom = "ctgA" if li % 3 else "ctgB"
        pos = 1000 + 37 * li
        strand = "+" if li % 2 else "-"
        ctx = "".join(rng.choice("ACGT") for _ in range(5)) + "M" + "".join(rng.choice("ACGT") for _ in range(5))
        shift = rng.uniform(-1.5, 1.5)
        for d in range(depth):
            feats = []
            for c in range(6):
                u = rng.random()
                if u < 0.05:
                    feats.append("0")                                   # empty column
                elif u < 0.10:
                    feats.append(repr(rng.gauss(0, 3) * 1e-5))           # scientific notation
                elif u < 0.30:
                    feats.append(repr(round(rng.gauss(shift, 2), 4)))    # few digits
                else:
                    feats.append(repr(rng.gauss(shift, 2)))              # 16-17 significant digits
            feats.append(repr(round(rng.uniform(5, 15), 3)))
            p = round(rng.random(), 2)
            label = "m6A" if p >= 0.5 else "A"
            rows.append((rng.random(), "%s\tread%d_%d\t%d\t%s\t%s\t%s\t%s\t%s\n" % (chrom, li, d, pos, ctx, ",".join(feats), strand, label, repr(p))))
    rows.sort()
    return "".join(r[1] for r in rows)
