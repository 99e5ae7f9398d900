"""Drop-in replacement for the reference module `extract_contexts` (al-mcintyre/mCaller).

Same public names and signatures as the reference file (extract_contexts.py:11-110), so the unmodified
`mCaller.py` (`from extract_contexts import *`, mCaller.py:18) and `make_bed.py` (`from extract_contexts import
revcomp`, make_bed.py:8) run on it when this directory precedes the reference on sys.path (INTEGRATION.md).
`extract_features` keeps its contract -- it appends `.diffs.<k>` rows to `<tsv prefix>.diffs.<k>.tmp<startline>` and
prints the five counters -- but the work is done by the CUDA pipeline in libmcaller_b200.so (engine.Engine); there is
no CPU implementation behind it.
"""
import os
import sys

import numpy as np

from . import refmark
from .refmark import comp, revcomp, strand  # noqa: F401  (re-exported, reference :14-29)

base_comps = {"A": "T", "C": "G", "T": "A", "G": "C", "N": "N", "M": "M"}

CHUNK_BYTES = int(os.environ.get("MCALLER_B200_CHUNK_BYTES", str(1 << 30)))
READ_THREADS = int(os.environ.get("MCALLER_B200_READ_THREADS", str(min(16, os.cpu_count() or 1))))   # parallel preads of the file reader


class ReferenceAbort(RuntimeError):
    """A condition on which the reference prints a diagnostic and calls sys.exit(0) or dies with an exception."""


def methylate_motifs(ref_seq, motif, meth_base, meth_position=None):
    """reference :33-41 (the meth_position branch of the reference is unreachable from its CLI and not mirrored)."""
    return refmark.mark_motif(ref_seq, motif, meth_base)


def methylate_positions(ref_seq, positions, meth_base):
    """reference :45-56; raises where the reference prints and quits."""
    return refmark.mark_positions(ref_seq, positions, meth_base)


def methylate_references(ref_seq, base, motif=None, positions=None, train=False, contig=None):
    """reference :60-73."""
    if not positions and not motif:
        print("no motifs or positions specified")
        raise ReferenceAbort("no motifs or positions specified")
    return refmark.mark_reference(ref_seq, base, motif=motif, positions_file=positions, contig=contig)


def find_and_methylate(refname, contigname, base, motif, positions_list):
    """reference :76-81 (returns None when the contig is absent)."""
    seqs = refmark.read_fasta(refname)
    if contigname in seqs:
        return methylate_references(seqs[contigname], base, motif=motif, positions=positions_list, contig=contigname)
    return None


def writefi(data, fi):
    """reference :83-86 (append mode)."""
    with open(fi, "a") as outfi:
        for entry in data:
            outfi.write("\t".join(entry) + "\n")


def diffs_name(tsv_input, k, start=None, train=False):
    """`<tsv prefix>.diffs.<k>`, the merged output of a run; with `start`, the file the worker whose byte range starts there
    appends to, `<tsv prefix>.diffs.<k>[.train].tmp<start>` (the reference's names)."""
    stem = ".".join(tsv_input.split(".")[:-1]) + ".diffs." + str(k) + (".train" if train else "")
    return stem if start is None else stem + ".tmp" + str(start)


def base_models(base, twobase=False):
    """reference :99-106: two-letter context after the target -> model key."""
    if base == "A" and twobase:
        table = {"M" + b: "MH" for b in "CATMH"}
        table.update({"A" + b: "MH" for b in "TCAM"})
        table["MG"] = "MG"
        table["AG"] = "MG"
        return table
    return {f + b: "general" for f in "MAT" for b in "ACGTM"}


# ---- helpers -------------------------------------------------------------------------------------------------------

def _line_name(buf, start):
    """Read name (4th whitespace-separated field) of the line starting at `start`, or None for lines with fewer than
    12 fields -- those are dropped by the tokeniser (:149-152) and must not look like read boundaries."""
    end = buf.find(b"\n", start)
    if end < 0:
        end = len(buf)
    f = buf[start:end].split(None, 12)
    return f[3] if len(f) >= 12 else None


def read_boundary_before(buf, limit=None):
    """Largest start s of a complete line of buf at which a new read begins (its name differs from the previous
    well-formed line's); 0 if there is none.  Everything from s on (the possibly incomplete last read and any partial
    last line) is meant to be carried into the next chunk."""
    end = buf.rfind(b"\n", 0, len(buf) if limit is None else limit) + 1       # end of the complete lines
    if end <= 0:
        return 0
    cur = buf.rfind(b"\n", 0, end - 1) + 1                                     # start of the last complete line
    cur_name = _line_name(buf, cur)
    while cur > 0:
        prev = buf.rfind(b"\n", 0, cur - 1) + 1
        prev_name = _line_name(buf, prev)
        if cur_name is None:                       # malformed line: transparent
            cur, cur_name = prev, prev_name
            continue
        if prev_name is None:                      # skip malformed predecessors
            p2 = prev
            while p2 > 0 and prev_name is None:
                p2 = buf.rfind(b"\n", 0, p2 - 1) + 1
                prev_name = _line_name(buf, p2)
            if prev_name is None:
                return 0
            if prev_name != cur_name:
                return cur
            cur, cur_name = p2, prev_name
            continue
        if cur_name != prev_name:
            return cur
        cur, cur_name = prev, prev_name
    return 0


def read_boundary_after(fh, offset, fsize, probe=1 << 22):
    """Smallest file offset s >= offset at which a line starts that begins a new read (or s == 0), else fsize."""
    if offset <= 0:
        return 0
    if offset >= fsize:
        return fsize
    # start far enough back to know the name of the last well-formed line before `offset`
    back = min(offset, 1 << 16)
    while True:
        fh.seek(offset - back)
        head = fh.read(back)
        p = head.find(b"\n")
        names = []
        if p >= 0:
            q = p + 1
            while q < len(head):
                e = head.find(b"\n", q)
                if e < 0:
                    break
                nm = _line_name(head, q)
                if nm is not None:
                    names.append(nm)
                q = e + 1
        if names or back == offset:
            break
        back = min(offset, back * 4)
    if back == offset:
        base, prev_name = 0, None
    else:
        # restart the scan at the first complete line of `head`
        base, prev_name = offset - back + p + 1, None
    while True:
        fh.seek(base)
        buf = fh.read(probe)
        if not buf:
            return fsize
        at_eof = base + len(buf) >= fsize
        cur = 0
        last_complete = -1
        while cur < len(buf):
            e = buf.find(b"\n", cur)
            if e < 0 and not at_eof:
                break                              # partial line: refill starting at it
            nm = _line_name(buf, cur)
            if nm is not None:
                if base + cur >= offset and prev_name is not None and nm != prev_name:
                    return base + cur
                if base + cur >= offset and prev_name is None and base + cur == 0:
                    return 0
                prev_name = nm
            last_complete = cur
            cur = (e + 1) if e >= 0 else len(buf)
        if at_eof:
            return fsize
        if last_complete < 0:
            probe *= 4
        else:
            base += cur


def _fmt(x):
    return repr(float(x))


def raise_row_error(err, mpos):
    """The reference's failure for a window whose row carries MC_CE_* error flags."""
    if err & 1:
        raise ReferenceAbort("window at %d lies within k of a contig end (reference: IndexError / sys.exit at extract_contexts.py:195/:224)" % mpos)
    if err & 2:
        raise ReferenceAbort("base after target %d is not one of ACGTM (reference: KeyError -> sys.exit, :218-223)" % mpos)
    if err & 4:
        raise ValueError("unsupported numeric field in a line feeding the window at %d" % mpos)
    if err & 16:
        raise ReferenceAbort("n diffs off (multi-M spacing 0) at %d" % mpos)


class _RowFormatter(object):
    """Training export: the closed call rows of a chunk as the reference's labelled `.diffs.<k>.train` rows (writer :216)
    and the signal / context matrices train_model takes.  The carried window's read name and the counters are the
    TextSink's (`sink`)."""

    def __init__(self, refindex, k, pos_label, sink, two_models=False):
        self.ref, self.k, self.pos_label, self.sink, self.two_models = refindex, k, pos_label, sink, two_models
        self.signals, self.contexts = {}, {}
        self.keys = []                 # model key of each row written, from the window builder's model_sel (mCaller --train)

    def _row(self, c, read):
        k = self.k
        mpos = int(c["mpos"])
        raise_row_error(int(c["err"]), mpos)
        rev = bool(c["rev"])
        ctx = self.ref.context(int(c["win_contig"]), mpos, rev)
        em = int(c["empty_mask"])
        feat = c["feat"]
        feats = ["0" if (em >> j) & 1 else _fmt(feat[j]) for j in range(k)] + [_fmt(feat[k])]
        chrom = self.ref.names[int(c["chrom_contig"])]
        label = self.pos_label[(chrom, mpos, strand(rev))]
        self.signals.setdefault("general", {}).setdefault(label, []).append([float(x) for x in feat[:k + 1]])
        self.contexts.setdefault("general", {}).setdefault(label, []).append(ctx)
        self.keys.append(("MG" if c["model_sel"] else "MH") if self.two_models else "general")
        return [chrom, read.decode(), str(mpos), ctx, ",".join(feats), strand(rev), label]

    def consume(self, calls, host_text_ptr, n_segments):
        """Rows of one chunk (host structured array, slot 0 first; read names at host_text_ptr) -> list of row lists."""
        import ctypes as C
        from . import _lib
        out = []
        for c in calls:
            if int(c["kind"]) != _lib.MC_CALL or int(c["close_rec"]) == _lib.PENDING:
                continue
            ro = int(c["read_off"])
            read = self.sink.carry[0] if ro < 0 else C.string_at(host_text_ptr + ro, int(c["read_len"]))
            out.append(self._row(c, read))
        self.sink.advance(calls, host_text_ptr, n_segments)
        return out


def _select_device(startline, endline):
    """SURVEY.md 8e: the reference's `-t N` workers (mCaller.py:63-70) own the byte ranges [chunk*i, chunk*(i+1)); worker i
    runs on GPU i mod n_gpus.  MCALLER_B200_DEVICE pins the device instead (one process per GPU launchers set it)."""
    import torch
    n = torch.cuda.device_count()
    env = os.environ.get("MCALLER_B200_DEVICE")
    if env is not None:
        idx = int(env) % max(n, 1)
    elif endline is not None and endline > startline and n > 1:
        idx = int(startline // (endline - startline)) % n
    else:
        idx = torch.cuda.current_device()
    torch.cuda.set_device(idx)
    return idx


class RangeRun(object):
    """One worker's byte range of an eventalign file on one GPU: reference index, models, engine and row writer, the
    streaming of the range into `<prefix>.diffs.<k>[.train].tmp<startline>` and the ways its last open window gets closed
    (probing the text after the range -- forked workers that cannot talk to each other -- or the next rank's first kept
    line in a multi-GPU run, mcaller_b200.multigpu)."""

    def __init__(self, tsv_input, fasta_input, read2qual, k, skip_thresh, qual_thresh, modelfile, startline, endline=None, train=False,
                 pos_label=None, base=None, motif=None, positions_list=None, histogram=False, row_base=0):
        from . import engine as _engine, models as _models, read_qual as _rq, stream as _stream
        from .refindex import ReferenceIndex
        _engine.require_cuda()
        self.device_index = _select_device(startline, endline)
        self.k = k = int(k)
        self.train, self.tsv_input, self.qual_thresh = train, tsv_input, qual_thresh
        seqs = refmark.read_fasta(fasta_input)
        try:
            self.ref = ReferenceIndex(seqs, base, motif=motif, positions_file=positions_list, k=k)
        except refmark.MarkError as e:
            print(str(e) + " - quitting thread now")
            raise ReferenceAbort(str(e))
        dm, two = None, train and base == "A"        # training -b A: rows get the MG/MH choice of a two-model pickle
        self.tsv_output = diffs_name(tsv_input, k, startline, train)
        if not train:
            model = _models.load_model_file(modelfile)
            e0, e1, two = _models.select_models(model, base)
            dm = _models.DeviceModels(e0, e1, n_in=k + 1)     # both models' widths are checked before any export
        # read2qual: the reference's dict, or a read_qual.DeviceQualityTable built on the GPU from the FASTQ
        qt = read2qual if isinstance(read2qual, _rq.DeviceQualityTable) else _rq.build_quality_table(read2qual)
        if isinstance(qt, _rq.DeviceQualityTable) and qt.table.device.index != self.device_index:
            qt = _rq.DeviceQualityTable(qt.table.to("cuda:%d" % self.device_index), qt.size, qt.n_records, qt.bad_headers)
        self.eng = _engine.Engine(self.ref, models=dm, qual_table=qt, skip_thresh=skip_thresh, qual_thresh=qual_thresh, two_models=two,
                                  histogram=histogram and dm is not None)
        if row_base:
            self.eng.reset_stream_state(row_base)
        self.sink = _stream.TextSink(self.ref, k, base, with_prob=dm is not None)
        self.fmt = _RowFormatter(self.ref, k, pos_label, self.sink, two_models=two) if train else None
        self.fsize = os.path.getsize(tsv_input)
        if endline is None:
            endline = self.fsize
        with open(tsv_input, "rb") as fh:
            self.lo = read_boundary_after(fh, startline, self.fsize)
            self.hi = read_boundary_after(fh, min(endline, self.fsize), self.fsize)
        self.bytes_done = 0

    def _render(self, h_calls, n_calls, host_text_ptr, n_segments=0):
        """Rows of one chunk, or the completed carried row, appended to the tmp file (like writefi, :83-86)."""
        from . import stream as _stream
        if self.train:
            writefi(self.fmt.consume(_stream.row_view(h_calls, n_calls), host_text_ptr, n_segments), self.tsv_output)
            return
        r = self.sink.render(h_calls, n_calls, host_text_ptr, n_segments)
        with open(self.tsv_output, "ab") as outfi:
            outfi.write(memoryview(self.sink.out)[:r])

    def stream(self):
        """Rows of the reads whose first line lies in [lo, hi) -> the tmp file: reader thread -> pinned buffers -> H2D on a
        side stream -> kernels -> rows back -> writer."""
        from . import stream as _stream
        open(self.tsv_output, "a").close()
        # chunk size: the configured one (1 GiB) for long ranges -- fewest per-chunk costs: 25.7 GB/s from the page cache
        # against 19.6 GB/s with 256 MiB chunks --, 1/32 of a shorter range: pinning three 1.25 GiB host buffers costs a
        # fresh process 3.4 s, three of 320 MiB 1.1 s, and reading, copying and computing still overlap
        chunk = min(CHUNK_BYTES, max(32 << 20, (self.hi - self.lo + 31) // 32))
        fs = _stream.FileStreamer(self.eng, chunk, read_boundary_before, readers=READ_THREADS)

        def check(res, text):
            _raise_on_counters(res)
            self._check_marking(text)
        fs.run(self.tsv_input, self.lo, self.hi, render=self._render, check=check)
        self.bytes_done += fs.h2d_bytes

    def _check_marking(self, text):
        """The reference marks a contig when the TSV first names it and quits on a bad positions row then
        (extract_contexts.py:45-56, :154-160).  Contigs whose marking failed were kept without targets (ReferenceIndex):
        the run stops as soon as one of them actually occurs in the text -- a rare path, searched on the host."""
        if not self.ref.mark_errors:
            return
        buf = text.tobytes() if isinstance(text, np.ndarray) else bytes(text)
        for nm, err in self.ref.mark_errors.items():
            key = nm.encode()
            if buf.startswith(key + b"\t") or buf.startswith(key + b" ") or (b"\n" + key + b"\t") in buf or (b"\n" + key + b" ") in buf:
                print(str(err) + " - quitting thread now")
                raise ReferenceAbort(str(err))

    def close_by_probe(self):
        """A window still open at the end of the range is closed by the first kept line after it, which lies in the next
        worker's range (mCaller.py:63-68): keep feeding text from there -- line-aligned pieces, growing -- until the carried
        window comes back completed as slot 0 (mc_carry_rows); the pieces' own rows belong to the next worker and are
        ignored, as are its input problems.  At the end of the file nothing closes it (reference: dropped, SURVEY.md Q3)."""
        from . import _lib
        eng = self.eng
        if self.sink.carry is None or self.hi >= self.fsize:
            return
        with open(self.tsv_input, "rb") as fh:
            ppos, size = self.hi, 4 << 20
            while ppos < self.fsize:
                fh.seek(ppos)
                probe = fh.read(size)
                at_eof = ppos + len(probe) >= self.fsize
                cutp = len(probe) if at_eof else probe.rfind(b"\n") + 1
                if cutp <= 0:                                  # no complete line in the piece: look at a larger one
                    size *= 4
                    continue
                res = eng.run_chunk(eng.upload(probe[:cutp]), cutp)
                row0 = res.calls()[:1]
                if len(row0) and row0[0]["kind"] != _lib.MC_NONE:
                    self.consume_closed(row0)
                    return
                ppos += cutp
                size = min(size * 2, 1 << 28)

    def consume_closed(self, row):
        """The carried window, completed (by close_by_probe or Engine.close_carry), goes to the end of the tmp file."""
        from . import _lib
        if len(row) and row[0]["kind"] != _lib.MC_NONE:
            self._render(row.view(np.uint8), 1, 0)

    def print_counters(self):
        sink = self.sink
        print("thread finished processing...:")
        print("%d observations" % sink.n_obs)
        print("%d positions" % len(sink.pos_set))
        print("%d regions with multiple methylated bases" % len(sink.multi))
        print("%d observations with skips included" % len(sink.wskips))
        print("%d observations with too many skips" % len(sink.toomany))


def extract_features(tsv_input, fasta_input, read2qual, k, skip_thresh, qual_thresh, modelfile, classifier, startline, endline=None,
                     train=False, pos_label=None, base=None, motif=None, positions_list=None):
    """GPU implementation behind the reference signature (extract_contexts.py:110).

    startline/endline are byte offsets like the reference's (mCaller.py:58, :63-68); a worker owns the reads whose
    first line starts inside [startline, endline) (ranges are snapped to read boundaries instead of the reference's
    '-500 characters / 8 MB overrun' overlap, SURVEY.md Q6), so concatenating the workers' files in offset order gives
    exactly the -t 1 output.  Worker i of a `-t N` run uses GPU i mod n_gpus (SURVEY.md 8e).
    """
    run = RangeRun(tsv_input, fasta_input, read2qual, k, skip_thresh, qual_thresh, modelfile, startline, endline=endline, train=train,
                   pos_label=pos_label, base=base, motif=motif, positions_list=positions_list)
    run.stream()
    run.close_by_probe()
    run.print_counters()
    if train:
        return run.fmt.signals, run.fmt.contexts


def _raise_on_counters(res):
    c = res.counters
    if c["badpos"]:
        raise ValueError("%d lines on known contigs have a non-integer position column" % c["badpos"])
    if res.missing_quality:
        raise KeyError("%d reads of the eventalign file are missing from the fastq" % res.missing_quality)
