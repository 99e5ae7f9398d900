"""Streaming eventalign text through the Engine: read-aligned chunks, double-buffered H2D copies on a side stream
overlapped with the kernels, the rows of every chunk copied back and rendered as `.diffs` text one chunk behind the GPU
(host memory -> PCIe -> HBM -> kernels -> rows back -> text).  The chunks come from a pinned host buffer (HostStreamer,
what bench.py times as `e2e`) or from a file (FileStreamer, the CLI and extract_features); both run the same pipeline and
the same writer (TextSink)."""
import ctypes as C
import time

import numpy as np
import torch

from . import _lib
from ._lib import CALL_DTYPE, MC_TEXT_PAD


def plan_chunks(read_offsets, total_bytes, chunk_bytes):
    """Chunk end offsets that fall on read boundaries; read_offsets = byte offset of the first line of each read."""
    offs = np.asarray(read_offsets, dtype=np.int64)
    cuts, start = [], 0
    while start < total_bytes:
        lim = start + chunk_bytes
        if lim >= total_bytes:
            cuts.append(int(total_bytes))
            break
        j = int(np.searchsorted(offs, lim, side="right")) - 1
        end = int(offs[j]) if j >= 0 and offs[j] > start else None
        if end is None:                       # a single read larger than the chunk: take it whole
            j2 = int(np.searchsorted(offs, start, side="right"))
            end = int(offs[j2]) if j2 < len(offs) else int(total_bytes)
        cuts.append(end)
        start = end
    return cuts


def row_view(h_calls, n_calls):
    """The first n_calls rows of a pinned uint8 tensor or numpy uint8 array as a structured array (no copy)."""
    raw = h_calls.numpy() if isinstance(h_calls, torch.Tensor) else h_calls
    return raw[:n_calls * CALL_DTYPE.itemsize].view(CALL_DTYPE)


class TextSink(object):
    """Renders the rows of a chunk as `.diffs.<k>` text with the native writer (mc_format_rows, host threads) straight from
    the pinned row buffer and the host copy of the TSV (read names are cut from it), and keeps the reference's five
    counters (extract_contexts.py:295-301).  Row 0 of every chunk is the slot of the window carried over the chunk edge
    (mc_carry_rows): kind MC_NONE when empty, else the completed row (read_off < 0) whose read name lies in an earlier
    chunk's text, so the sink keeps those bytes, and the row's read-segment key, when it sees the open row."""

    def __init__(self, refindex, k, base="A", with_prob=True, keep=False, max_threads=0):
        names = refindex.names
        n = len(names)
        self._keep = [nm.encode() for nm in names] + list(refindex.marked_bytes(0)) + list(refindex.marked_bytes(1))
        self.names, self.fwd, self.rev = (C.c_char_p * n)(*self._keep[:n]), (C.c_char_p * n)(*self._keep[n:2 * n]), (C.c_char_p * n)(*self._keep[2 * n:])
        self.lens = (C.c_int64 * n)(*[len(x) for x in self._keep[n:2 * n]])
        self.name_len = max([len(x) for x in self._keep[:n]] + [0])
        self.n, self.k, self.with_prob = n, int(k), 1 if with_prob else 0
        self.base, self.mod = base.encode(), (b"m6A" if base == "A" else b"m" + base.encode())
        self.max_threads = int(max_threads)
        self.out = None
        self.text_bytes = 0
        self.render_seconds = 0.0             # host time spent in the native writer
        self.carry = None                     # (read name, segment key) of the window currently open across a chunk edge
        self.seg_base = 0                     # read segments of the chunks so far: segment keys are unique over the range
        self.n_obs = 0
        self.pos_set, self.multi, self.wskips, self.toomany = set(), set(), set(), set()
        self.kept = [] if keep else None      # rendered text per chunk (tests)

    def render(self, h_calls, n_calls, host_text_ptr, n_segments=0):
        """h_calls: pinned uint8 tensor (or numpy uint8 array) holding n_calls rows; host_text_ptr: address of the chunk's
        first byte in host memory (0 when the rows carry no read_off into a text, e.g. the row of Engine.close_carry).
        Returns the number of bytes rendered into self.out; row errors raise what the reference raises."""
        rows = row_view(h_calls, n_calls)
        r = 0
        if n_calls > 0:
            name = self.carry[0] if self.carry is not None else None
            nlen = len(name) if name is not None else 0
            # per row at most: contig and read name, 2k-1 context letters, k+1 floats of <= 24 characters, label,
            # probability, position, strand and separators
            cap = n_calls * (96 + 26 * (self.k + 1) + self.name_len + max(int(rows["read_len"].max()), nlen)) + 4096
            if self.out is None or len(self.out) < cap:
                self.out = C.create_string_buffer(int(cap * 1.25))
            t0 = time.perf_counter()
            r = int(_lib.lib().mc_format_rows(C.c_void_p(rows.ctypes.data), n_calls, C.c_void_p(host_text_ptr), name, nlen, self.names,
                                              self.fwd, self.rev, self.lens, self.n, self.k, self.base, self.mod, self.with_prob,
                                              self.max_threads, self.out, len(self.out)))
            self.render_seconds += time.perf_counter() - t0
            if r < 0:
                self._raise(r, rows)
            self.text_bytes += r
            if self.kept is not None:
                self.kept.append(self.out.raw[:r])
        self.advance(rows, host_text_ptr, n_segments)
        return r

    @staticmethod
    def _raise(r, rows):
        from .extract_contexts import raise_row_error
        if r <= -100:
            bad = rows[(rows["kind"] == _lib.MC_CALL) & (rows["close_rec"] != _lib.PENDING) & (rows["err"] != 0)][0]
            raise_row_error(int(bad["err"]), int(bad["mpos"]))
        try:
            _lib.check(r)
        except _lib.McallerCudaError as e:
            if "outside ACGTNM" in str(e):
                raise KeyError(str(e))               # the reference: KeyError in revcomp (extract_contexts.py:11-15)
            raise

    def advance(self, rows, host_text_ptr, n_segments):
        """Counts one chunk's rows (vectorised) and moves the carried window on: the one completed in slot 0 is done, a
        call or too-many-skips window still open after the last row is kept with its read name.  render calls it; the
        training export, which writes its own rows, calls it directly."""
        n = len(rows)
        if n:
            kind = rows["kind"]
            pend = rows["close_rec"] == _lib.PENDING
            carried = rows["read_off"] < 0
            segkey = rows["seg"].astype(np.int64) + self.seg_base
            segkey[carried] = self.carry[1] if self.carry is not None else -1
            pair = (segkey << 32) | rows["mpos"].astype(np.int64)
            closed = (kind == _lib.MC_CALL) & ~pend
            self.multi.update(np.unique(pair[kind == _lib.MC_MULTI_M]).tolist())
            self.toomany.update(np.unique(pair[(kind == _lib.MC_TOO_MANY_SKIPS) & ~pend]).tolist())
            self.wskips.update(np.unique(pair[closed & (rows["n_empty"] > 0)]).tolist())
            self.pos_set.update(np.unique(rows["mpos"][closed]).tolist())
            self.n_obs += int(closed.sum())
            if kind[0] != _lib.MC_NONE and carried[0]:
                self.carry = None             # the carried window has been written (or counted) with this chunk
            last = rows[n - 1]
            if pend[n - 1] and kind[n - 1] in (_lib.MC_CALL, _lib.MC_TOO_MANY_SKIPS) and not carried[n - 1]:
                self.carry = (C.string_at(host_text_ptr + int(last["read_off"]), int(last["read_len"])), int(segkey[n - 1]))
        self.seg_base += n_segments


def last_boundary(arr, total, boundary_before, span=1 << 22):
    """Offset of the last read boundary inside arr[:total] (uint8 numpy array; 0: none) -- what
    boundary_before(bytes(arr[:total])) returns, but only a tail is searched (and copied).  The tail starts at a line start,
    so the first line seen is complete, and grows until it holds a boundary."""
    while True:
        a = max(0, total - span)
        if a > 0:
            nl = np.flatnonzero(arr[a:min(total, a + (1 << 20))] == 10)
            if len(nl) == 0:
                span *= 4
                continue
            a += int(nl[0]) + 1
        tail = arr[a:total].tobytes()
        cut = boundary_before(tail, len(tail))
        if cut > 0:
            return a + cut
        if a == 0:
            return 0
        span *= 4


class _Pipeline(object):
    """The device side of both sources: double-buffered H2D staging of the text on a side stream (chunk i+1 is copied
    while chunk i is in the kernels), Engine.run_chunk, the pinned D2H of the rows and their rendering one chunk behind."""

    def __init__(self, engine):
        self.eng, self.dev = engine, engine.device
        self.dbuf = [None, None]
        self.copy_stream = torch.cuda.Stream(device=self.dev)
        self.ready = [torch.cuda.Event() for _ in range(2)]
        self.free = [torch.cuda.Event() for _ in range(2)]
        self.h_calls = None                   # pinned rows: chunk i-1 is rendered before chunk i's rows are copied in
        self.calls_done = torch.cuda.Event()
        self.h2d_bytes = 0
        self.d2h_bytes = 0

    def _enqueue_copy(self, dslot, src, n):
        cap = self.eng.padded_capacity(n)
        if self.dbuf[dslot] is None or self.dbuf[dslot].numel() < cap:
            self.free[dslot].synchronize()
            self.dbuf[dslot] = torch.empty(int(cap * 1.1) + 4096, dtype=torch.uint8, device=self.dev)
        with torch.cuda.stream(self.copy_stream):
            self.copy_stream.wait_event(self.free[dslot])
            self.dbuf[dslot][:n].copy_(src[:n], non_blocking=True)
            self.dbuf[dslot][n:n + MC_TEXT_PAD + 16].fill_(10)
            self.ready[dslot].record(self.copy_stream)
        self.h2d_bytes += n

    def _stream(self, chunks, render=None, check=None, fetch_calls=True):
        """chunks: iterator of (pinned uint8 tensor with the chunk's text at [0, n), n, release or None).  check(res, text)
        runs as soon as chunk i's kernels are done, before any of its rows is rendered; render(h_calls, n_calls,
        host_text_ptr, n_segments) gets chunk i's rows once chunk i+1 is in the kernels' queue.  Chunk i-1 is rendered and
        released before chunk i+1 is taken: a source that cuts its chunks out of a ring of buffers (FileStreamer) needs that
        slot back to hand chunk i+1 over.  Windows open at a chunk end are carried on the device (Engine.d_carry); the one
        still open after the last chunk is left for the caller (Engine.close_carry: next rank / end of file)."""
        eng = self.eng
        fetch_calls = fetch_calls or render is not None
        cur = torch.cuda.current_stream(self.dev)
        for e in self.free:
            e.record(cur)
        tot = dict(calls=0, too_many_skips=0, multi=0, errors=0, methylated=0, records=0, lines=0, rows=0)
        late = None                                   # (n_calls, text address, n_segments, release) of chunk i-1

        def finish(n_c, ptr, n_seg, release):
            if render is not None:
                if n_c:
                    self.calls_done.synchronize()
                render(self.h_calls, n_c, ptr, n_seg)
            if release is not None:
                release()
        chunks = iter(chunks)
        nxt = next(chunks, None)
        if nxt is not None:
            self._enqueue_copy(0, nxt[0], nxt[1])
        st, i = None, 0
        while nxt is not None:
            src, n, release = nxt
            if late is not None:
                finish(*late)
            nxt = next(chunks, None)
            if nxt is not None:
                self._enqueue_copy((i + 1) & 1, nxt[0], nxt[1])
            cur.wait_event(self.ready[i & 1])
            res = eng.run_chunk(self.dbuf[i & 1], n)
            if check is not None:
                check(res, src.numpy()[:n])
            st = res.stats
            n_c = res.n_calls if fetch_calls else 0
            if n_c:
                nb = n_c * CALL_DTYPE.itemsize
                if self.h_calls is None or self.h_calls.numel() < nb:
                    self.h_calls = torch.empty(int(nb * 1.5) + 4096, dtype=torch.uint8, pin_memory=True)
                self.h_calls[:nb].copy_(res.calls_dev[:nb], non_blocking=True)
                self.calls_done.record(cur)
                self.d2h_bytes += nb
            late = (n_c, src.data_ptr(), res.n_segments, release)
            self.free[i & 1].record(cur)
            for kx in ("calls", "too_many_skips", "multi", "errors", "methylated"):
                tot[kx] += st[kx]
            tot["records"] += res.n_records
            tot["lines"] += res.counters["lines"]
            tot["rows"] += res.n_calls
            i += 1
        cur.synchronize()
        if late is not None:
            finish(*late)
        # the window (call or too-many-skips event) still open after the last chunk: Engine.close_carry decides its fate
        tot["open_at_end"] = (st["pending"] + st["pending_too_many_skips"]) if st is not None else 0
        return tot


class FileStreamer(_Pipeline):
    """A byte range of an eventalign file -> read-aligned chunks through the pipeline: a reader thread fills a ring of
    pinned host buffers with parallel preads, cutting at the last read boundary and carrying the incomplete read into the
    next buffer.  A buffer goes back to the reader once its chunk's rows are rendered (read names are cut from its text).
    `boundary_before(bytes) -> offset` finds the last read boundary of a buffer (extract_contexts.read_boundary_before)."""

    def __init__(self, engine, chunk_bytes, boundary_before, slots=3, readers=4):
        _Pipeline.__init__(self, engine)
        self.chunk_bytes = int(chunk_bytes)
        self.boundary_before = boundary_before
        self.n_slots, self.readers = int(slots), int(readers)
        self.pin = [None] * self.n_slots          # pinned uint8 tensors, grown on demand

    def _ensure_pin(self, slot, nbytes, keep=0):
        t = self.pin[slot]
        if t is None or t.numel() < nbytes:
            nt = torch.empty(int(nbytes * 1.25) + (1 << 16), dtype=torch.uint8, pin_memory=True)
            if t is not None and keep:
                nt[:keep].copy_(t[:keep])
            self.pin[slot] = nt
        return self.pin[slot]

    def _producer(self, path, lo, hi, q_free, q_ready):
        import os
        from concurrent.futures import ThreadPoolExecutor
        try:
            fd = os.open(path, os.O_RDONLY)
            try:
                with ThreadPoolExecutor(max_workers=self.readers) as pool:
                    def read_into(mv, off):
                        done = 0
                        while done < len(mv):
                            got = os.preadv(fd, [mv[done:]], off + done)
                            if got <= 0:
                                raise IOError("short read at offset %d" % (off + done))
                            done += got

                    pos, carry, slot = lo, 0, q_free.get()
                    while pos < hi or carry:
                        want = min(self.chunk_bytes, hi - pos)
                        arr = self._ensure_pin(slot, carry + want, keep=carry).numpy()
                        if want:
                            step = max(1 << 24, (want + self.readers - 1) // self.readers)
                            futs = [pool.submit(read_into, memoryview(arr[carry + a:carry + min(want, a + step)]), pos + a)
                                    for a in range(0, want, step)]
                            for f in futs:
                                f.result()
                        pos += want
                        total = carry + want
                        if pos < hi:
                            cut = last_boundary(arr, total, self.boundary_before)
                            if cut == 0:                     # a single read larger than the chunk: keep reading into this slot
                                carry = total
                                continue
                            nslot = q_free.get()
                            narr = self._ensure_pin(nslot, total - cut + self.chunk_bytes).numpy()
                            narr[:total - cut] = arr[cut:total]
                            q_ready.put((slot, cut))
                            slot, carry = nslot, total - cut
                        else:
                            if total:
                                q_ready.put((slot, total))
                            carry = 0
            finally:
                os.close(fd)
            q_ready.put(None)
        except BaseException as e:                          # surfaces in the consumer
            q_ready.put(e)

    def run(self, path, lo, hi, render=None, check=None):
        """Streams the file's bytes [lo, hi) (read-aligned) through the pipeline; returns the totals of _Pipeline._stream."""
        import queue
        import threading
        q_free, q_ready = queue.Queue(), queue.Queue()
        for sl in range(self.n_slots):
            q_free.put(sl)
        th = threading.Thread(target=self._producer, args=(path, lo, hi, q_free, q_ready), daemon=True)
        th.start()

        def chunks():
            while True:
                item = q_ready.get()
                if isinstance(item, BaseException):
                    raise item
                if item is None:
                    return
                slot, n = item
                yield self.pin[slot], n, lambda s=slot: q_free.put(s)
        tot = self._stream(chunks(), render=render, check=check)
        th.join()
        return tot


class HostStreamer(_Pipeline):
    """Chunks are slices of a pinned host buffer at plan_chunks cuts (bench.py's e2e leg)."""

    def __init__(self, engine, chunk_bytes=1 << 30):
        _Pipeline.__init__(self, engine)
        self.chunk_bytes = int(chunk_bytes)

    def run(self, host_buf, cuts, fetch_calls=True, sink=None):
        """host_buf: pinned uint8 CPU tensor; cuts: chunk end offsets from plan_chunks.  Returns dict of totals; rows of
        every chunk are copied to pinned host memory when fetch_calls (the D2H leg of the end-to-end path) and, with a
        TextSink, rendered as `.diffs` text."""
        bounds = [0] + list(cuts)
        return self._stream(((host_buf[a:b], b - a, None) for a, b in zip(bounds, bounds[1:])),
                            render=sink.render if sink is not None else None, fetch_calls=fetch_calls)
