"""Window column means at every event count numpy sums differently.

A window feature is `np.mean` of the `np.round(event_level_mean - model_mean, 4)` values of the lines that fed one column
(extract_contexts.py:186).  numpy sums fewer than 8 values left to right, up to 128 in 8 lanes and a tail, more by
recursive halving; k_windows restates each order separately (a running sum in shared memory, col_sum_big re-reading the
tagged records, the spill arena and an explicit stack), and its per-slot event count saturates at 65 535.  The synthetic
generator never puts more than 20 events on a position, so here a stall injector replaces the lines of chosen positions
by N events each -- the pore holding one k-mer -- and every stall's column mean is checked, as bits, against numpy itself
(the oracle restates numpy too, so only numpy can catch an order both get wrong), against the CPU oracle's rows and
against the device's: in the GATC and `-m A` regimes, sparse, dense and read-first (-q) scans, across k_windows block
edges, across chunk edges, with a spill arena too small for the input, and at the 65 535-event limit."""
import functools
import os

import numpy as np
import pytest

import golden_cases as gc

WIN_RECS = 1536             # records one k_windows block stages (WIN_THREADS * WIN_ITEMS, mcaller_b200/csrc/windows.cu:42)
COUNTS = [1, 7, 8, 9, 16, 17, 21, 64, 127, 128, 129, 136, 137, 256, 257, 1000, 1537, 4097, 8193]
BIG = 65534                 # the most events a column may hold: used once per input
NEG_ZERO = (1, 7, 8, 9, 129)  # counts with one column whose currents all round to -0.0 (numpy's mean: 0.0)
REGIMES = [("GATC", 6, 1), ("A", 6, 2), ("A", 8, 3)]     # motif, k, -s


def _bits(x):
    return int(np.float64(x).view(np.uint64))


def _spec(seed, n_reads, len_min=300, len_max=700):
    from mcaller_b200 import synth
    return synth.SynthSpec(seed=seed, contigs=[("ctgA", 40000), ("ctgB", 30000)], n_reads=n_reads, len_min=len_min, len_max=len_max)


def _split_reads(tsv):
    """The lines of a synth.generate TSV as one list of field lists per read, in file order (read i of the spec)."""
    reads = []
    for ln in tsv.decode().split("\n"):
        if not ln:
            continue
        f = ln.split("\t")
        if not reads or reads[-1][0][3] != f[3]:
            reads.append([])
        reads[-1].append(f)
    return reads


def _groups(lines):
    """(position, first line index, end line index) of each run of lines at one position."""
    out, a = [], 0
    for i in range(1, len(lines) + 1):
        if i == len(lines) or lines[i][1] != lines[a][1]:
            out.append((int(lines[a][1]), a, i))
            a = i
    return out


class Stall(object):
    """N events of one read at one position: their currents, and `want`, numpy's mean of their rounded differences."""

    def __init__(self, read, rev, pos, first_m, evs, model):
        self.read, self.rev, self.pos, self.first_m, self.evs, self.model = read, rev, pos, first_m, evs, model
        self.n = len(evs)
        self.diffs = [np.round(float(ev) - float(model), 4) for ev in evs]
        self.want = np.mean(self.diffs)

    def feature(self, k):
        """Index of the stall's column among the row's features: forward reads are flipped (extract_contexts.py:186-188)."""
        return self.first_m if self.rev else k - 1 - self.first_m


def _left_to_right(v):
    """Mean of a plain running sum: numpy's order below 8 values only."""
    acc = 0.0
    for x in v:
        acc += x
    return acc / len(v)


def _lanes8(v):
    """Mean of numpy's 8-lane sum applied to the whole column, without the recursive halving above 128 values."""
    r = list(v[:8])
    i = 8
    while i < len(v) - len(v) % 8:
        for j in range(8):
            r[j] += v[i + j]
        i += 8
    acc = ((r[0] + r[1]) + (r[2] + r[3])) + ((r[4] + r[5]) + (r[6] + r[7]))
    for x in v[i:]:
        acc += x
    return (acc + 0.0) / len(v)


def _order_shows(st):
    """Would a kernel that summed this column in the wrong order get another mean?"""
    if st.n < 8:
        return True
    return _bits(_left_to_right(st.diffs)) != _bits(st.want) and (st.n <= 128 or _bits(_lanes8(st.diffs)) != _bits(st.want))


def _currents(rng, model, n, neg_zero):
    """n event_level_mean strings whose difference to `model` (a %.2f string) rounds to values of both signs and magnitudes
    from 0.0001 to about 40, about a tenth of them exactly 0; with neg_zero, 5-decimal currents 0.00001-0.00004 below the
    model, whose rounded differences are all -0.0."""
    m = float(model)
    if neg_zero:
        return ["%.5f" % (m - 1e-5 * u) for u in rng.integers(1, 5, n)]
    mag = 10.0 ** rng.uniform(-4, np.log10(40.0), n)
    d = np.round(np.where(rng.random(n) < 0.5, -mag, mag), 4)
    d[rng.random(n) < 0.1] = 0.0
    return [model if x == 0.0 else "%.4f" % (m + x) for x in d]


def _target(ref, contig, pos, rev):
    """Index of the first target of the k-mer at `pos` on the read's strand, or -1 (the ReferenceIndex site bit maps)."""
    bits = ref.site_rev_bits if rev else ref.site_fwd_bits
    g = int(ref.contig_base[ref.names.index(contig)]) + pos
    hit = np.flatnonzero(bits[g:g + ref.k])
    return int(hit[0]) if len(hit) else -1


def _candidates(ref, lines, rev):
    """(position, first target index, template line index) of the read's positions that feed a window column; the template
    is a line of that position that is not NNNNNN (its columns are copied into the stall's lines).  Positions within k of
    the read's ends are left out: their windows lack the columns before the read's start and usually have too many skips."""
    out = []
    lo, hi = int(lines[0][1]) + ref.k, int(lines[-1][1]) - ref.k
    for pos, a, b in _groups(lines):
        tmpl = [i for i in range(a, b) if lines[i][9] != "NNNNNN"]
        f = _target(ref, lines[a][0], pos, rev)
        if tmpl and f >= 0 and lo <= pos <= hi:
            out.append((pos, f, tmpl[0]))
    return out


def _stall_read(lines, at, first_m, n, rng, neg_zero, rev):
    """Replaces the lines of the position group holding line `at` by n lines copied from line `at` with drawn currents
    -> (new lines, Stall)."""
    pos = lines[at][1]
    a = at
    while a > 0 and lines[a - 1][1] == pos:
        a -= 1
    b = at
    while b < len(lines) and lines[b][1] == pos:
        b += 1
    tmpl = lines[at]
    while True:                       # columns of 8 or more values are redrawn until the summation order shows in their mean
        st = Stall(tmpl[3], rev, int(pos), first_m, _currents(rng, tmpl[10], n, neg_zero), tmpl[10])
        if neg_zero or _order_shows(st):
            break
    new = [list(tmpl[:6]) + [ev] + list(tmpl[7:]) for ev in st.evs]
    return lines[:a] + new + lines[b:], st


def _renumber(spec, reads):
    """event_index strictly monotonic over each whole read: ascending on forward reads, descending on reverse reads, as
    synth.read_lines writes them."""
    from mcaller_b200 import synth
    for i, lines in enumerate(reads):
        rev, e0 = synth.read_meta(spec, i)[3], synth.read_meta(spec, i)[4]
        n = len(lines)
        for j, f in enumerate(lines):
            f[5] = str(e0 + (n - 1 - j if rev else j))


def _join(reads):
    return ("\n".join("\t".join(f) for lines in reads for f in lines) + "\n").encode()


def inject_stalls(spec, tsv, ref, plan, seed):
    """plan: [(read index, position, N, neg_zero)] -> (stalled TSV bytes, [Stall]).  Every planned position must feed a
    window column on the read's strand."""
    from mcaller_b200 import synth
    rng = np.random.default_rng(seed)
    reads = _split_reads(tsv)
    stalls = []
    for ri, pos, n, neg in plan:
        rev = bool(synth.read_meta(spec, ri)[3])
        lines = reads[ri]
        cand = {p: (f, t) for p, f, t in _candidates(ref, lines, rev)}
        f, at = cand[pos]
        reads[ri], st = _stall_read(lines, at, f, n, rng, neg, rev)
        stalls.append(st)
    _renumber(spec, reads)
    return _join(reads), stalls


def _plan(spec, tsv, ref, counts, seed, per_read=2):
    """Three stalls per count (strands fwd/rev/fwd or rev/fwd/rev) and BIG once, placed in file order by increasing N (the
    first chunks of a streamed run hold the small ones), at most `per_read` per read and 2k positions apart."""
    from mcaller_b200 import synth
    rng = np.random.default_rng(seed)
    reads = _split_reads(tsv)
    want = []
    for ci, n in enumerate(counts):
        s = ci % 2
        want += [(n, s, False), (n, 1 - s, n in NEG_ZERO), (n, s, False)]
    want.append((BIG, 1, False))
    used = {}
    nxt = [0, 0]
    plan = []
    for n, strand, neg in want:
        while True:
            ri = nxt[strand]
            assert ri < len(reads) - 1, "not enough reads for the plan"
            if bool(synth.read_meta(spec, ri)[3]) == bool(strand) and len(used.get(ri, [])) < per_read:
                taken = used.setdefault(ri, [])
                ok = [c for c in _candidates(ref, reads[ri], bool(strand)) if all(abs(c[0] - p) > 2 * ref.k for p in taken)]
                if ok:
                    pos = ok[int(rng.integers(len(ok)))][0]
                    taken.append(pos)
                    plan.append((ri, pos, n, neg))
                    break
            nxt[strand] += 1
    return plan


@functools.lru_cache(maxsize=None)
def _models(k):
    from mcaller_b200 import models
    if k == 6:
        return models.load_model_file(os.path.join(gc.GOLD, "models", gc.R95))
    from test_num_variables import _model_dict
    return _model_dict(k + 1)


@functools.lru_cache(maxsize=None)
def _case(motif, k):
    """Stalled input of one regime: (tsv, seqs, quals, stalls, -q threshold, read offsets)."""
    from mcaller_b200 import synth
    from mcaller_b200.refindex import ReferenceIndex
    spec = _spec(41 + k + (0 if motif == "GATC" else 100), 90 if motif == "GATC" else 50)
    tsv, _, _, quals = synth.generate(spec)
    seqs = {nm: synth.genome(spec, ci).tobytes().decode() for ci, (nm, _) in enumerate(spec.contigs)}
    ref = ReferenceIndex(seqs, "A", motif=motif, k=k, device="cpu")
    plan = _plan(spec, tsv, ref, COUNTS, 7 + k)
    tsv, stalls = inject_stalls(spec, tsv, ref, plan, 11 + k)
    quals = {q.split("_")[0]: v for q, v in quals.items()}
    return tsv, seqs, quals, stalls, float(np.median(list(quals.values())))


@functools.lru_cache(maxsize=None)
def _oracle_rows(motif, k, s, q):
    from oracle import oracle as orc
    tsv, seqs, quals, stalls, qt = _case(motif, k)
    return orc.extract(tsv, seqs, quals, k=k, skip_thresh=s, qual_thresh=qt if q else 0.0, model=_models(k), base="A", motif=motif,
                       cap=400000)


def _landed(rows, stalls, k, quals, qual_thresh):
    """Checks every stall whose window became a call row ((read, mpos) -> features, empty mask): its column holds numpy's
    mean as bits.  Returns (stalls landed, stalls on reads the quality filter keeps)."""
    landed = eligible = 0
    for st in stalls:
        if quals[st.read.split("_")[0]] < qual_thresh:
            continue
        eligible += 1
        row = rows.get((st.read, st.pos + st.first_m))
        if row is None:
            continue
        feat, empty = row
        j = st.feature(k)
        assert not (empty >> j) & 1, (st.read, st.pos, st.n)
        assert _bits(feat[j]) == _bits(st.want), (st.read, st.pos, st.n, feat[j], st.want)
        landed += 1
    return landed, eligible


# ---- host (no GPU) --------------------------------------------------------------------------------------------------

@pytest.mark.parametrize("motif,k,s", REGIMES)
def test_stalled_inputs_have_teeth(motif, k, s):
    """The drawn currents make the summation order visible: for every N >= 8 a left-to-right mean differs from np.mean in
    at least one column, and for N > 128 so does an 8-lane sum without the halving; the -0.0 columns really are -0.0;
    every count appears three times, on both strands; event indices stay strictly monotonic in each read."""
    tsv, seqs, quals, stalls, qt = _case(motif, k)

    by_n = {}
    for st in stalls:
        by_n.setdefault(st.n, []).append(st)
    assert sorted(by_n) == sorted(COUNTS + [BIG])
    for n, group in by_n.items():
        assert len(group) == (1 if n == BIG else 3) and (n == BIG or {st.rev for st in group} == {False, True})
        if n >= 8:
            assert any(_bits(_left_to_right(st.diffs)) != _bits(st.want) for st in group), n
        if n > 128:
            assert any(_bits(_lanes8(st.diffs)) != _bits(st.want) for st in group), n
        neg = [st for st in group if all(_bits(d) == _bits(-0.0) for d in st.diffs)]
        assert len(neg) == (1 if n in NEG_ZERO else 0), n
        for st in neg:
            assert _bits(st.want) == _bits(0.0)
    direction = {st.read: st.rev for st in stalls}
    for lines in _split_reads(tsv):
        d = np.diff([int(f[5]) for f in lines])
        assert np.all(d > 0) or np.all(d < 0)
        if lines[0][3] in direction and len(d):
            assert (d[0] < 0) == direction[lines[0][3]]


@pytest.mark.parametrize("q", [False, True])
@pytest.mark.parametrize("motif,k,s", REGIMES)
def test_oracle_column_means_equal_numpy(motif, k, s, q, oracle):
    """The CPU oracle's rows carry each stall's numpy mean, as bits, in the stall's column; at least 80 % of the stalls on
    reads the quality filter keeps land in a call row."""
    tsv, seqs, quals, stalls, qt = _case(motif, k)
    want = _oracle_rows(motif, k, s, q)
    rows = {(w["read"], w["mpos"]): (w["feat"], w["empty_mask"]) for w in want["calls"]}
    landed, eligible = _landed(rows, stalls, k, quals, qt if q else 0.0)
    assert eligible >= (len(stalls) // 3 if q else len(stalls)) and landed >= 0.8 * eligible, (landed, eligible)


# ---- GPU ------------------------------------------------------------------------------------------------------------

def _engine(motif, k, s, qual_thresh=0.0, dense=None, seqs=None, quals=None):
    from mcaller_b200 import engine, models, read_qual
    from mcaller_b200.refindex import ReferenceIndex
    m = _models(k)
    ref = ReferenceIndex(seqs, "A", motif=motif, k=k)
    dm = models.DeviceModels(m["MH"], m["MG"], n_in=k + 1)
    return engine.Engine(ref, models=dm, qual_table=read_qual.build_quality_table(quals), skip_thresh=s, qual_thresh=qual_thresh,
                         two_models=True, dense=dense)


def _check_rows(res, tsv, want, stalls, k, quals, qual_thresh):
    """Device rows == oracle rows (keys, features as bits, probability within 1e-12), the counters equal, and each stall's
    numpy mean in its column; returns the number of stalls that landed."""
    from mcaller_b200 import _lib
    assert res.missing_quality == 0
    calls = res.calls()
    mine = calls[(calls["kind"] == _lib.MC_CALL) & (calls["close_rec"] != _lib.PENDING)]
    assert len(mine) == len(want["calls"])
    rows = {}
    for c, w in zip(mine, want["calls"]):
        read = tsv[int(c["read_off"]):int(c["read_off"]) + int(c["read_len"])].decode()
        assert (int(c["mpos"]), bool(c["rev"]), int(c["empty_mask"]), read, int(c["model_sel"]), int(c["label"])) == \
            (w["mpos"], w["rev"], w["empty_mask"], w["read"], w["model_sel"], w["label"])
        assert np.array_equal(c["feat"][:k + 1].view(np.uint64), np.array(w["feat"], dtype=np.float64).view(np.uint64))
        assert abs(float(c["prob"]) - w["prob"]) < 1e-12
        rows[(read, int(c["mpos"]))] = (c["feat"][:k + 1].copy(), int(c["empty_mask"]))
    st = res.stats
    multi = calls[calls["kind"] == _lib.MC_MULTI_M]
    assert st["too_many_skips"] == want["counters"]["too_many_skips"] and st["errors"] == 0
    assert len({(int(a), int(b)) for a, b in zip(multi["seg"], multi["mpos"])}) == want["counters"]["multi"]
    landed, eligible = _landed(rows, stalls, k, quals, qual_thresh)
    assert landed >= 0.8 * eligible
    return landed


@pytest.mark.gpu
@pytest.mark.parametrize("mode", ["sparse", "dense", "q"])
@pytest.mark.parametrize("motif,k,s", REGIMES)
def test_device_column_means_equal_oracle_and_numpy(motif, k, s, mode, cuda_lib, oracle):
    """Stalls of 1 to 65 534 events, on both strands, in the GATC regime (short windows) and the `-m A` regime at k = 6 and 8
    (multi-M carries reuse a stalled column in consecutive windows and permute the column slots), with the sparse scan, the
    dense scan and the read-first scan of -q (threshold: the median read quality): every row, feature bit and counter equals
    the oracle's, and every stall's column holds numpy's mean."""
    tsv, seqs, quals, stalls, qt = _case(motif, k)
    q = qt if mode == "q" else 0.0
    eng = _engine(motif, k, s, qual_thresh=q, dense=True if mode == "dense" else None, seqs=seqs, quals=quals)
    res = eng.run_chunk(eng.upload(tsv), len(tsv))
    _check_rows(res, tsv, _oracle_rows(motif, k, s, mode == "q"), stalls, k, quals, q)


def _block_edge_case():
    """`-m A`, k = 6: stalls of 9, 100, 129 and 300 events with a multiple of WIN_RECS records strictly inside (in dense mode
    one record is one kept line), and one of 3 100 across two block edges.  -> (tsv, seqs, quals, stalls)."""
    from mcaller_b200 import synth
    from mcaller_b200.refindex import ReferenceIndex
    spec = _spec(77, 40, 500, 900)
    tsv, _, _, quals = synth.generate(spec)
    seqs = {nm: synth.genome(spec, ci).tobytes().decode() for ci, (nm, _) in enumerate(spec.contigs)}
    ref = ReferenceIndex(seqs, "A", motif="A", k=6, device="cpu")
    reads = _split_reads(tsv)
    rng = np.random.default_rng(5)
    stalls, ri = [], 0
    for n in (9, 100, 129, 300, 3100):
        edges = 2 if n == 3100 else 1
        placed = False
        while not placed:
            ri += 1                                     # one stall per read, the first read left alone
            assert ri < len(reads) - 1
            rev = bool(synth.read_meta(spec, ri)[3])
            before = sum(f[9] != "NNNNNN" for lines in reads[:ri] for f in lines)
            for pos, f, at in _candidates(ref, reads[ri], rev):
                a = at
                while a > 0 and reads[ri][a - 1][1] == reads[ri][at][1]:
                    a -= 1
                r0 = before + sum(x[9] != "NNNNNN" for x in reads[ri][:a])       # record index of the stall's first line
                edge = -(-(r0 + 1) // WIN_RECS) * WIN_RECS                        # first block edge after it
                if edge + (edges - 1) * WIN_RECS <= r0 + n - 1:
                    reads[ri], st = _stall_read(reads[ri], at, f, n, rng, False, rev)
                    stalls.append(st)
                    placed = True
                    break
    _renumber(spec, reads)
    tsv = _join(reads)
    return tsv, seqs, {q.split("_")[0]: v for q, v in quals.items()}, stalls


@pytest.mark.gpu
def test_columns_across_block_edges(cuda_lib, oracle):
    """Stalled columns whose records straddle k_windows block edges (tags of the records past a block's staged range live in
    global memory): rows equal the oracle's, each stall's column is numpy's mean, dense and sparse scan alike."""
    tsv, seqs, quals, stalls = _block_edge_case()
    want = oracle.extract(tsv, seqs, quals, k=6, skip_thresh=2, model=_models(6), base="A", motif="A", cap=400000)
    for dense in (True, None):
        eng = _engine("A", 6, 2, dense=dense, seqs=seqs, quals=quals)
        res = eng.run_chunk(eng.upload(tsv), len(tsv))
        assert _check_rows(res, tsv, want, stalls, 6, quals, 0.0) == len(stalls)
        if dense:
            rec = eng.records(res.n_records)
            line = rec["line_lo"].astype(np.int64) | (rec["line_hi"].astype(np.int64) << 32)
            for st in stalls:                           # the stall's records: its read's records at its position
                name = st.read.encode()
                idx = np.flatnonzero(rec["pos"] == st.pos)
                idx = [i for i in idx if tsv[line[i] + int(rec["name_off"][i]):line[i] + int(rec["name_off"][i]) + len(name)] == name]
                assert len(idx) == st.n and idx[-1] - idx[0] == st.n - 1
                inside = [b for b in range(idx[0] + 1, idx[-1] + 1) if b % WIN_RECS == 0]
                assert len(inside) == (2 if st.n == 3100 else 1), (st.n, idx[0])


def _stream(eng, tsv, chunk_bytes):
    """HostStreamer + TextSink over read-aligned chunks -> (text, chunks, histogram)."""
    import torch
    from mcaller_b200 import stream
    offs, p = [], 0
    last = None
    for ln in tsv.split(b"\n")[:-1]:
        name = ln.split(b"\t", 4)[3]
        if name != last:
            offs.append(p)
            last = name
        p += len(ln) + 1
    hbuf = torch.empty(len(tsv), dtype=torch.uint8, pin_memory=True)
    hbuf.copy_(torch.from_numpy(np.frombuffer(tsv, dtype=np.uint8).copy()))
    cuts = stream.plan_chunks(offs, len(tsv), chunk_bytes)
    sink = stream.TextSink(eng.ref, eng.ref.k, "A", with_prob=True, keep=True)
    stream.HostStreamer(eng, chunk_bytes).run(hbuf, cuts, sink=sink)
    return b"".join(sink.kept), len(cuts), [a.copy() for a in eng.histogram_host()]


@pytest.mark.gpu
def test_columns_across_chunk_edges_and_a_small_spill_arena(monkeypatch, cuda_lib):
    """The GATC input streamed in read-aligned chunks: the text equals the oracle's rows byte for byte and the histogram
    equals a one-chunk run's, first-seen order included.  Then the same with a 1 024-double spill arena, which the stalls of
    the later chunks outgrow: each such chunk is run again with a grown arena (the failed attempt leaves the histogram and
    the carried window untouched), in one run_chunk over the whole input and in the stream alike."""
    from mcaller_b200 import engine
    tsv, seqs, quals, stalls, qt = _case("GATC", 6)
    text = "".join(r + "\n" for r in _oracle_rows("GATC", 6, 1, False)["rows"]).encode()
    one, n1, hist1 = _stream(_engine("GATC", 6, 1, seqs=seqs, quals=quals), tsv, 1 << 30)
    assert n1 == 1 and one == text
    many, n, hist = _stream(_engine("GATC", 6, 1, seqs=seqs, quals=quals), tsv, len(tsv) // 6)
    assert n >= 4 and many == text
    assert all(np.array_equal(a, b) for a, b in zip(hist[:2], hist1[:2]))
    assert np.array_equal(np.argsort(hist[2], kind="stable"), np.argsort(hist1[2], kind="stable"))

    monkeypatch.setattr(engine, "SPILL_CAP", 1024)
    eng = _engine("GATC", 6, 1, seqs=seqs, quals=quals)
    res = eng.run_chunk(eng.upload(tsv), len(tsv))
    assert eng.redone >= 1 and eng.spill_cap > 1024
    _check_rows(res, tsv, _oracle_rows("GATC", 6, 1, False), stalls, 6, quals, 0.0)
    eng = _engine("GATC", 6, 1, seqs=seqs, quals=quals)
    small, n2, hist2 = _stream(eng, tsv, len(tsv) // 6)
    assert n2 == n and small == text and eng.redone >= 1
    assert all(np.array_equal(a, b) for a, b in zip(hist2, hist))


def _limit_case(n, d):
    """A GATC input with one stall of n events, written to directory d with a FASTQ and a labelled positions file (every
    GATC site, labels alternating) for the training export -> (paths, tsv, seqs, quals, stall)."""
    from mcaller_b200 import synth
    from mcaller_b200.refindex import ReferenceIndex
    spec = _spec(91, 8)
    tsv, fasta, fastq, quals = synth.generate(spec)
    seqs = {nm: synth.genome(spec, ci).tobytes().decode() for ci, (nm, _) in enumerate(spec.contigs)}
    ref = ReferenceIndex(seqs, "A", motif="GATC", k=6, device="cpu")
    reads = _split_reads(tsv)
    ri = next(i for i in range(1, len(reads) - 1) if _candidates(ref, reads[i], bool(synth.read_meta(spec, i)[3])))
    pos = _candidates(ref, reads[ri], bool(synth.read_meta(spec, ri)[3]))[0][0]
    tsv, stalls = inject_stalls(spec, tsv, ref, [(ri, pos, n, False)], 3)
    pos_rows = ["%s\t%d\t%s\t%s\n" % (ref.names[c], p, "-" if r else "+", "m6A" if i % 2 else "A")
                for i, (c, p, r) in enumerate(zip(ref.site_contig, ref.site_pos, ref.site_rev))]
    paths = {"tsv": os.path.join(d, "stall.eventalign.tsv"), "fasta": os.path.join(d, "ref.fasta"), "fastq": os.path.join(d, "stall.fastq"),
             "positions": os.path.join(d, "pos.txt")}
    for key, data in (("tsv", tsv), ("fasta", fasta.encode()), ("fastq", fastq.encode()), ("positions", "".join(pos_rows).encode())):
        with open(paths[key], "wb") as fh:
            fh.write(data)
    return paths, tsv, seqs, {q.split("_")[0]: v for q, v in quals.items()}, stalls[0]


@pytest.mark.gpu
@pytest.mark.parametrize("n", [65534, 65535, 70000])
def test_event_count_limit_of_a_column(n, tmp_path, cuda_lib, oracle):
    """65 534 events in one column give numpy's mean; at 65 535 and more the per-slot count of k_windows saturates, and the
    `.diffs` writer and the training export both raise an error naming the limit instead of writing the row."""
    from mcaller_b200 import cli, extract_contexts as ec
    paths, tsv, seqs, quals, st = _limit_case(n, str(tmp_path))
    want = oracle.extract(tsv, seqs, quals, k=6, skip_thresh=1, model=_models(6), base="A", motif="GATC", cap=400000)
    assert (st.read, st.pos + st.first_m) in {(w["read"], w["mpos"]) for w in want["calls"]}    # the stall's window is a call row
    text = "".join(r + "\n" for r in want["rows"]).encode()
    eng = _engine("GATC", 6, 1, seqs=seqs, quals=quals)
    if n < 65535:
        res = eng.run_chunk(eng.upload(tsv), len(tsv))
        assert _check_rows(res, tsv, want, [st], 6, quals, 0.0) == 1
        eng.reset_histogram()
        assert _stream(eng, tsv, 1 << 30)[0] == text
        return
    with pytest.raises(ValueError, match="65535 or more events"):
        _stream(eng, tsv, 1 << 30)
    pk = str(tmp_path / "m.pkl")
    with pytest.raises(ValueError, match="65535 or more events"):
        cli.mcaller_main(["--train", "-d", pk, "-p", paths["positions"], "-r", paths["fasta"], "-e", paths["tsv"], "-f", paths["fastq"],
                          "-b", "A", "-s", "1"])
    train = ec.diffs_name(paths["tsv"], 6, 0, train=True)
    rows = open(train).read().splitlines() if os.path.exists(train) else []
    assert not [r for r in rows if r.split("\t")[1] == st.read and int(r.split("\t")[2]) == st.pos + st.first_m]
    assert not os.path.exists(pk)
