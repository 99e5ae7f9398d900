"""Host-side logic that runs without a GPU: reference marking, model-key table, chunk / worker-range cutting,
read-quality ingest and lookup table, synthetic generator determinism, C-ABI surface."""
import io
import os
import random
import re

import numpy as np
import pytest

import golden_cases as gc
from mcaller_b200 import extract_contexts as ec, read_qual, refmark, synth


def test_revcomp_and_strand():
    assert ec.revcomp("GATCM") == "MGATC"
    assert ec.revcomp("GATC", False) == "GATC"
    assert ec.comp("ACGTNM") == "TGCANM"
    assert ec.strand(True) == "-" and ec.strand(False) == "+"
    with pytest.raises(KeyError):
        ec.revcomp("CAAY")          # reference has no IUPAC codes in base_comps (:11)


def test_mark_motif_semantics():
    # every `base` of the motif is marked, matching is leftmost non-overlapping (reference :39-40)
    assert refmark.mark_motif("TTGATCGATCAA", "GATC", "A") == "TTGMTCGMTCAA"
    assert refmark.mark_motif("GAGAGAG", "GAGAG", "A") == "GMGMGAG"
    assert refmark.mark_motif("CAAC", "AA", "A") == "CMMC"
    f, r = refmark.mark_reference("TTGATCAAT", "A", motif="GATC")
    assert f == "TTGMTCAAT" and r == "TTGAMCAAT"
    f, r = refmark.mark_reference("ACGT", "A", motif="A")
    assert f == "MCGT" and r == "ACGM"


def test_mark_positions(tmp_path):
    p = tmp_path / "pos.txt"
    p.write_text("c1\t1\t+\tm6A\nc1\t3\t-\tm6A\nc2\t0\t+\tm6A\n\n")
    f, r = refmark.mark_reference("CATT", "A", positions_file=str(p), contig="c1")
    assert f == "CMTT" and r == "CATM"
    with pytest.raises(refmark.MarkError):
        refmark.mark_reference("CCTT", "A", positions_file=str(p), contig="c1")


def test_base_models_table():
    t = ec.base_models("A", True)
    assert t["MG"] == "MG" and t["AG"] == "MG"
    for kx in ("MC", "MA", "MT", "MM", "AT", "AC", "AA", "AM"):
        assert t[kx] == "MH"
    g = ec.base_models("C", True)
    assert set(g.values()) == {"general"} and "MG" in g and "TM" in g
    assert ec.base_models("A", False)["MG"] == "general"


def _mk_tsv(n_reads, rnd, junk=False):
    lines, starts = [], []
    off = 0
    for r in range(n_reads):
        starts.append(off)
        for j in range(rnd.randint(1, 30)):
            ln = "ctg\t%d\tACGTAC\tread%04d_x\tt\t%d\t80.00\t1.0\t0.001\tACGTAC\t81.00\t1.5\t0.1\n" % (100 + j, r, j)
            lines.append(ln)
            off += len(ln)
            if junk and rnd.random() < 0.3:          # malformed lines inside a read must not look like read boundaries
                jl = rnd.choice(["\n", "ctg\t5\tAAA\tother\tt\n", "x y z\n"])
                lines.append(jl)
                off += len(jl)
    return "".join(lines).encode(), starts


@pytest.mark.parametrize("junk", [False, True])
def test_read_boundary_helpers(tmp_path, junk):
    rnd = random.Random(5)
    data, starts = _mk_tsv(40, rnd, junk)
    path = tmp_path / "x.tsv"
    path.write_bytes(data)
    sset = sorted(starts)
    with open(path, "rb") as fh:
        for off in [0, 1, 5, starts[3], starts[3] + 1, starts[10] - 1, len(data) - 1, len(data)]:
            want = min([s for s in sset if s >= off] + [len(data)])
            assert ec.read_boundary_after(fh, off, len(data), probe=257) == want, off
    for lim in [len(data), len(data) - 3, starts[7] + 5, starts[1] + 1, 10]:
        buf = data[:lim]
        comp_end = buf.rfind(b"\n") + 1
        good = [i for i in range(comp_end) if (i == 0 or buf[i - 1:i] == b"\n") and len(buf[i:buf.find(b"\n", i)].split()) >= 12]
        want = max([s for s in sset if good and s <= good[-1]] + [0])
        assert ec.read_boundary_before(buf) == want, lim


def test_read_quality_and_table(tmp_path):
    fq = tmp_path / "r.fastq"
    fq.write_text("@abc_Basecall_1D_template extra\nACGT\n+\n!!II\n@zz:1D_000:template\nAC\n+\n5I\n")
    q = read_qual.extract_read_quality(str(fq))
    assert set(q) == {"abc", "zz"}
    assert q["abc"] == np.mean([0, 0, 40, 40]) and q["zz"] == np.mean([20, 40])
    import gzip
    gz = tmp_path / "r.fastq.gz"
    with gzip.open(gz, "wt") as fh:
        fh.write(fq.read_text())
    assert read_qual.extract_read_quality(str(gz)) == q
    d = {"r%d" % i: float(i) / 7 for i in range(5000)}
    t = read_qual.build_quality_table(d)
    assert len(t) & (len(t) - 1) == 0 and (t["hash"] != 0).sum() == len(d)
    h, h2, ln = read_qual.fnv_pair([k.encode() for k in d])
    mask = len(t) - 1
    for i, k in enumerate(list(d)[:500]):
        s = int(h[i]) & mask
        while True:
            assert t["hash"][s] != 0
            if t["hash"][s] == h[i] and t["len"][s] == ln[i] and t["check"][s] == int(h2[i]) >> 32:
                assert t["qual"][s] == d[k]
                break
            s = (s + 1) & mask


def test_fixture_quality_matches_reference_value():
    q = read_qual.extract_read_quality(os.path.join(gc.GOLD, "masonread1", "masonread1.fastq"))
    assert q == {"26dd376e-9d82-41fc-921e-71e559c8e8d1": 7.055265349382997}     # SURVEY.md section 4


def test_synth_is_deterministic_and_wellformed():
    spec = synth.SynthSpec(seed=21, contigs=[("a", 3000), ("b", 2500)], n_reads=6, len_min=100, len_max=300, header=True)
    t1, fa1, fq1, q1 = synth.generate(spec)
    t2, fa2, fq2, q2 = synth.generate(synth.SynthSpec(seed=21, contigs=[("a", 3000), ("b", 2500)], n_reads=6, len_min=100, len_max=300, header=True))
    assert t1 == t2 and fa1 == fa2 and fq1 == fq2
    lines = t1.decode().split("\n")[1:-1]
    assert all(len(l.split("\t")) == 13 for l in lines)
    g = {"a": synth.genome(spec, 0).tobytes().decode(), "b": synth.genome(spec, 1).tobytes().decode()}
    for l in lines[:500]:
        f = l.split("\t")
        assert g[f[0]][int(f[1]):int(f[1]) + 6] == f[2]
        assert f[9] in (f[2], refmark.revcomp(f[2]), "NNNNNN")
        assert re.fullmatch(r"\d+\.\d\d", f[6])


def test_golden_inputs_are_stable(tmp_path):
    """The committed golden outputs are only meaningful if the inputs can be rebuilt bit for bit."""
    import hashlib, json
    for name in ("gatc_s0", "A_s0", "adversarial", "masonread1_p"):
        gold = json.load(open(os.path.join(gc.GOLD, name + ".json")))
        d = tmp_path / name
        d.mkdir()
        inp = gc.build_inputs(gc.CASES[name], str(d))
        assert hashlib.sha256(open(inp["tsv"], "rb").read()).hexdigest() == gold["tsv_sha256"]


def test_c_abi_v3_exports_match_header():
    """ABI version 3: every function declared in include/mcaller_b200.h is exported by the built library and bound in
    _lib, and the unused mc_diffs_aggregate that version 2 exported is gone."""
    from mcaller_b200 import _lib, build
    build.build()
    hdr = open(os.path.join(os.path.dirname(gc.GOLD), "..", "include", "mcaller_b200.h")).read()
    declared = set(re.findall(r"^(?:int|int64_t|const char \*)\s*\*?\s*(mc_[a-z0-9_]+)\s*\(", hdr, re.M))
    assert declared, "no declarations parsed"
    lib = _lib.load()
    for fn in declared:
        assert hasattr(lib, fn), fn
    assert declared == set(_lib.EXPORTS)
    assert not hasattr(lib, "mc_diffs_aggregate")
    assert lib.mc_version() == _lib.MC_ABI_VERSION == 3
    assert lib.mc_num_tiles(1) == 1 and lib.mc_num_tiles(3840) == 1 and lib.mc_num_tiles(3841) == 2
    assert lib.mc_workspace_bytes(1000) > 8000


def test_struct_sizes_match_abi():
    import ctypes as C
    from mcaller_b200 import _lib
    assert _lib.RECORD_DTYPE.itemsize == 32 and _lib.CALL_DTYPE.itemsize == 128 and _lib.QUAL_DTYPE.itemsize == 24
    from mcaller_b200 import build
    build.build()
    lib = _lib.load()
    assert lib.mc_sizeof(0) == _lib.RECORD_DTYPE.itemsize and lib.mc_sizeof(1) == _lib.CALL_DTYPE.itemsize
    assert lib.mc_sizeof(2) == C.sizeof(_lib.RefIndex) and lib.mc_sizeof(3) == C.sizeof(_lib.Model)
    assert lib.mc_sizeof(4) == _lib.QUAL_DTYPE.itemsize and lib.mc_sizeof(5) == C.sizeof(_lib.SynthSpec)
    assert lib.mc_sizeof(6) == C.sizeof(_lib.LocusEntry) == 32
    assert lib.mc_sizeof(7) == _lib.DIFFS_ROW_DTYPE.itemsize == 32


def test_no_cpu_fallback_without_cuda():
    import torch
    if torch.cuda.is_available():
        pytest.skip("CUDA present")
    from mcaller_b200 import _lib, engine
    with pytest.raises(_lib.McallerCudaError):
        engine.require_cuda()
    with pytest.raises(_lib.McallerCudaError):
        ec.extract_features("x.tsv", "x.fa", {}, 6, 0, 0, "m.pkl", "NN", 0, endline=1, base="A", motif="GATC")


def test_iupac_expansion_matches_regex():
    """Documented extension (SURVEY.md Q9): IUPAC motifs are expanded on both strands (all, also overlapping, matches)."""
    import re as _re
    rnd = random.Random(9)
    seq = "".join(rnd.choice("ACGT") for _ in range(20000))
    for motif, base in (("CAAYNNNNNRTAC", "A"), ("GANTC", "A"), ("CCWGG", "C"), ("RAACY", "A")):
        pat = "".join("[%s]" % refmark.IUPAC[c] for c in motif)
        want = set()
        for m in _re.finditer("(?=(%s))" % pat, seq):
            for j, ch in enumerate(motif):
                if ch == base:
                    want.add(m.start() + j)
        assert refmark.expand_iupac_sites(seq, motif, base) == sorted(want)
    f, r = refmark.mark_reference("TTCAACGGGGGATACTTGTATCCCCCGTTGAA", "A", motif="CAAYNNNNNRTAC")
    assert f.count("M") == 3 and r.count("M") == 3          # one instance per strand, three A's / T's each


def test_native_row_writer_matches_python_repr():
    """mc_format_rows (host-side C++): shortest round-trip float text == repr(float) / str(np.float64), np.round(p, 2),
    integer 0 for empty columns, revcomp'd context for '-' rows."""
    import ctypes as C
    from mcaller_b200 import _lib, build
    build.build()
    lib = _lib.load()
    rnd = random.Random(1)
    vals = [0.0, -0.0, 1.0, -1.5, 1e-5, 5e-05, 0.0001, 0.00011, 123456789012345678.0, 1e16, 9999999999999998.0, 1e15, 0.1 + 0.2, -4.55,
            7.055265349382997, 1e-300, float("nan"), 3.0, 100000.0, 1e22, 1.7976931348623157e308, -0.4066666666666667]
    vals += [rnd.uniform(-20, 20) for _ in range(2000)] + [float(np.round(rnd.uniform(-10, 10), 4)) for _ in range(2000)]
    vals += [rnd.uniform(-1, 1) * 10 ** rnd.randint(-8, 18) for _ in range(1000)]
    n = len(vals)
    calls = np.zeros(n, dtype=_lib.CALL_DTYPE)
    calls["feat"][:, 0] = vals
    calls["feat"][:, 1] = 11.5
    calls["prob"] = [abs(v) % 1 if v == v else 0.5 for v in vals]
    calls["mpos"] = 10
    calls["read_len"] = 2
    calls["rev"] = np.arange(n) % 2
    calls["empty_mask"][5::7] = 1
    calls["kind"][3::11] = 1                      # non-call rows are skipped
    text = b"rd" + b"\n" * 16
    fwd, rev = b"ACGTACGTACMCGTACGTACGTAAAA", b"TTGTACGTACMCGGACGTACGTAAAA"
    names = (C.c_char_p * 1)(b"c1")
    a_f, a_r, ln = (C.c_char_p * 1)(fwd), (C.c_char_p * 1)(rev), (C.c_int64 * 1)(26)
    out = C.create_string_buffer(400 * n)
    r = lib.mc_format_rows(calls.ctypes.data_as(C.c_void_p), n, text, None, 0, names, a_f, a_r, ln, 1, 1, b"A", b"m6A", 1, 0, out, len(out))
    assert r > 0, lib.mc_last_error()
    rows = out.raw[:r].decode().split("\n")[:-1]
    live = [i for i in range(n) if calls["kind"][i] == 0]
    assert len(rows) == len(live)
    for i, row in zip(live, rows):
        f = row.split("\t")
        c = calls[i]
        want_feat = "0" if c["empty_mask"] & 1 else repr(float(vals[i]))
        assert f[:4] == ["c1", "rd", "10", "M"] and f[5] == ("-" if c["rev"] else "+")
        assert f[4] == want_feat + ",11.5"
        assert f[6] == ("m6A" if c["prob"] >= 0.5 else "A") and f[7] == str(np.round(np.float64(c["prob"]), 2))
    # the 5 022 rows above are rendered by several host threads (one per ~2k rows); slices of 1 000 rows are rendered by one
    # thread each and must concatenate to the same bytes
    whole = out.raw[:r]
    parts = []
    for a in range(0, n, 1000):
        sl = np.ascontiguousarray(calls[a:a + 1000])
        r2 = lib.mc_format_rows(sl.ctypes.data_as(C.c_void_p), len(sl), text, None, 0, names, a_f, a_r, ln, 1, 1, b"A", b"m6A", 1, 0, out, len(out))
        assert r2 >= 0
        parts.append(out.raw[:r2])
    assert b"".join(parts) == whole
    # an error flag on a row is reported with the row, whichever thread meets it
    bad = calls.copy()
    bad["err"][4321] = 4
    r3 = lib.mc_format_rows(bad.ctypes.data_as(C.c_void_p), n, text, None, 0, names, a_f, a_r, ln, 1, 1, b"A", b"m6A", 1, 0, out, len(out))
    assert r3 == -104 and b"4321" in lib.mc_last_error()
    # k = 3: context is cut from the strand's marked copy and reverse-complemented for '-' rows
    calls2 = np.zeros(2, dtype=_lib.CALL_DTYPE)
    calls2["mpos"], calls2["read_len"], calls2["rev"] = 10, 2, [0, 1]
    r = lib.mc_format_rows(calls2.ctypes.data_as(C.c_void_p), 2, text, None, 0, names, a_f, a_r, ln, 1, 3, b"A", b"m6A", 0, 0, out, len(out))
    rows = out.raw[:r].decode().split("\n")[:-1]
    assert rows[0].split("\t")[3] == fwd[8:13].decode() and rows[1].split("\t")[3] == refmark.revcomp(rev[8:13].decode())
    assert len(rows[0].split("\t")) == 6
    # a row carried over a chunk edge (read_off < 0) takes its read name from the caller; MC_NONE slots are skipped; the
    # thread cap does not change the bytes
    calls3 = np.zeros(3, dtype=_lib.CALL_DTYPE)
    calls3["mpos"], calls3["read_len"], calls3["rev"] = 10, 2, [0, 1, 0]
    calls3["read_off"][0] = -1
    calls3["kind"][2] = _lib.MC_NONE
    r = lib.mc_format_rows(calls3.ctypes.data_as(C.c_void_p), 3, text, b"carried-read", 12, names, a_f, a_r, ln, 1, 3, b"A", b"m6A", 0, 1, out, len(out))
    rows = out.raw[:r].decode().split("\n")[:-1]
    assert len(rows) == 2 and rows[0].split("\t")[1] == "carried-read" and rows[1].split("\t")[1] == "rd"
    assert lib.mc_format_rows(calls3.ctypes.data_as(C.c_void_p), 3, text, None, 0, names, a_f, a_r, ln, 1, 3, b"A", b"m6A", 0, 0, out, len(out)) == -1
    # a context over a reference letter outside ACGTNM: the reference raises KeyError in revcomp; here an error, not a NUL byte
    a_bad = (C.c_char_p * 1)(b"TTGTACGTRCMCGGACGTACGTAAAA")
    r = lib.mc_format_rows(calls2.ctypes.data_as(C.c_void_p), 2, text, None, 0, names, a_f, a_bad, ln, 1, 3, b"A", b"m6A", 0, 0, out, len(out))
    assert r == -1 and b"ACGTNM" in lib.mc_last_error()


def test_tail_search_of_last_read_boundary_equals_full_search():
    """stream.last_boundary (the file reader's cut point, searched in a growing tail of the pinned buffer) returns what
    extract_contexts.read_boundary_before gives on the whole buffer: random read lengths incl. reads longer than the
    first tail, malformed lines, a partial last line, buffers without any boundary."""
    from mcaller_b200 import extract_contexts as ec, stream
    rnd = random.Random(11)

    def line(read, pos):
        return ("ctg\t%d\tACGTAC\t%s\tt\t%d\t90.12\t1.5\t0.003\tACGTAC\t89.9\t1.2\t0.1\n" % (pos, read, pos)).encode()

    for trial in range(40):
        parts, n_reads = [], rnd.randint(1, 6)
        for r in range(n_reads):
            for j in range(rnd.choice([1, 3, 40, 400, 3000])):
                parts.append(line("read%d_%d" % (trial, r), j))
                if rnd.random() < 0.02:
                    parts.append(rnd.choice([b"\n", b"x y z\n", b"ctg\t5\tshort\n"]))
        buf = b"".join(parts)
        if rnd.random() < 0.5:
            buf = buf[:len(buf) - rnd.randint(1, 60)]                  # partial last line
        arr = np.frombuffer(buf, dtype=np.uint8)
        want = ec.read_boundary_before(buf, len(buf))
        for span in (64, 1000, 50000, 1 << 22):
            assert stream.last_boundary(arr, len(buf), ec.read_boundary_before, span=span) == want, (trial, span)


def test_multigpu_run_reports_a_failed_rank(tmp_path):
    """`cli mCaller --gpus N` spawns its ranks with plain multiprocessing (the parent never imports torch); a rank that
    dies -- here: no such TSV, or no CUDA device -- takes the others down and surfaces as one RuntimeError."""
    from mcaller_b200 import multigpu
    with pytest.raises(RuntimeError, match="rank [01] of 2 exited"):
        multigpu.run(dict(tsv=str(tmp_path / "missing.eventalign.tsv"), k=6), 2)
