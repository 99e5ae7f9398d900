"""stream.TextSink, the one `.diffs.<k>` writer of the CLI, the ranks and the benchmark, on the CPU: output buffer sizing
for long read and contig names, and the reference's exceptions for rows it cannot write."""
import hashlib
import random

import numpy as np
import pytest

from mcaller_b200 import _lib, build, extract_contexts as ec, refmark, stream

FWD, REV = b"ACGTACGTACMCGTACGTACGTAAAA", b"TTGTACGTACMCGGACGTACGTAAAA"


class _Ref(object):
    """What TextSink reads from a ReferenceIndex: contig names and the marked copies of each strand."""

    def __init__(self, name, fwd=FWD, rev=REV):
        self.names = [name]
        self._marked = (fwd, rev)

    def marked_bytes(self, strand):
        return [self._marked[strand]]


@pytest.fixture(scope="module", autouse=True)
def _built():
    build.build()


def _rows(read_len, n=2000, seed=5):
    """n closed call rows at position 10 of contig 0, row i naming read i of a text of n read_len-byte names."""
    rnd = random.Random(seed)
    names = b"".join((b"r%05d" % i).ljust(read_len, b"x")[:read_len] for i in range(n))
    rows = np.zeros(n, dtype=_lib.CALL_DTYPE)
    rows["read_off"] = np.arange(n) * read_len
    rows["read_len"] = read_len
    rows["mpos"] = 10
    rows["rev"] = np.arange(n) % 2
    rows["seg"] = np.arange(n) // 4
    rows["feat"][:, :4] = [[rnd.uniform(-20, 20) * 10 ** rnd.randint(-6, 6) for _ in range(4)] for _ in range(n)]
    rows["empty_mask"][3::5] = 2
    rows["n_empty"][3::5] = 1
    rows["prob"] = [rnd.random() for _ in range(n)]
    return rows, np.frombuffer(names, dtype=np.uint8)


def _render(sink, rows, text):
    r = sink.render(rows.view(np.uint8), len(rows), text.ctypes.data)
    return sink.out.raw[:r]


def test_long_read_names_fit_the_output_buffer():
    """2 000 rows with 1 000-byte read names (k = 3): every row is written, byte for byte what the writer produced before
    the CLI and the benchmark shared it, and the five counters count them."""
    rows, text = _rows(1000)
    sink = stream.TextSink(_Ref("c1"), 3, "A")
    out = _render(sink, rows, text)
    assert len(out) == 2200286 and out.count(b"\n") == 2000
    assert hashlib.sha256(out).hexdigest() == "48796281ce2ebe8761ebbcedf97c60f40a134ea12880905139677f54503ce9a1"
    assert (sink.n_obs, len(sink.pos_set), len(sink.multi), len(sink.wskips), len(sink.toomany)) == (2000, 1, 0, 400, 0)


def test_long_contig_name_fits_the_output_buffer():
    """2 000 rows on a 300-byte contig name with 2-byte read names (k = 3), checked field by field."""
    contig = "c" * 300
    rows, text = _rows(2)
    out = _render(stream.TextSink(_Ref(contig), 3, "A"), rows, text)
    lines = out.decode().split("\n")
    assert lines[-1] == "" and len(lines) == 2001
    for c, line in zip(rows, lines):
        f = line.split("\t")
        feats = ["0" if (c["empty_mask"] >> j) & 1 else repr(float(c["feat"][j])) for j in range(3)] + [repr(float(c["feat"][3]))]
        ctx = refmark.revcomp(REV[8:13].decode()) if c["rev"] else FWD[8:13].decode()
        assert f == [contig, text[c["read_off"]:c["read_off"] + 2].tobytes().decode(), "10", ctx, ",".join(feats), "-" if c["rev"] else "+",
                     "m6A" if c["prob"] >= 0.5 else "A", str(np.round(np.float64(c["prob"]), 2))]


def test_row_errors_raise_what_the_reference_raises():
    """A row carrying an error flag raises ReferenceAbort with the window's position; a context over a reference letter
    outside ACGTNM raises KeyError, as revcomp does in the reference."""
    rows, text = _rows(2, n=10)
    rows["err"][6] = _lib.MC_CE_CONTEXT
    rows["mpos"][6] = 11
    with pytest.raises(ec.ReferenceAbort, match="window at 11 "):
        _render(stream.TextSink(_Ref("c1"), 3, "A"), rows, text)
    rows, text = _rows(2, n=10)
    with pytest.raises(KeyError, match="outside ACGTNM"):
        _render(stream.TextSink(_Ref("c1", rev=b"TTGTACGTRCMCGGACGTACGTAAAA"), 3, "A"), rows, text)
