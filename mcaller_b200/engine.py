"""Host driver of the GPU pipeline: one `run_chunk` = stages 1-7 of include/mcaller_b200.h over one chunk of
eventalign TSV text resident in device memory.  PyTorch is used only to own device buffers and streams.

A chunk is ONE asynchronous sequence of launches: every count a stage hands to the next (records, read segments,
rows) stays in device memory, the window still open at the end of the chunk is carried to the next one in a
device-resident `mc_carry`, and the host reads a single status block when the chunk is done.  Buffer capacities are
learned from the chunks seen so far; a chunk that outgrows them is detected on the device (mc_chunk_guard: the stages
that touch cross-chunk state then do nothing) and simply run again with larger buffers.

The engine never computes anything on the CPU: without a CUDA device or the built library it raises.
"""
import ctypes as C

import numpy as np
import torch

from . import _lib
from ._lib import CALL_DTYPE, CARRY_BYTES, MC_C_COUNT, MC_TEXT_PAD, RECORD_DTYPE, check

C_LINES, C_KEPT, C_RECORDS, C_SHORT, C_UNKNOWN, C_NNN, C_BADPOS, C_LONGLINE, C_OVERFLOW = range(9)

# layout of the per-chunk status block (uint64 slots): 0..15 the counters of mc_scan, then
S_NSEG, S_MISSING_QUAL, S_NCALLS, S_CALL_OVERFLOW, S_ABORT, S_NREC, S_NROWS = 16, 17, 18, 19, 20, 21, 22
S_NLOG = 23                 # entries mc_rowlog_append added in this chunk (row log enabled only)
S_STATS = 24                # 7 row statistics of mc_count_calls
S_WORDS = 32
# persistent device state (uint64 slots): global row index of the next chunk's slot 0, rows in the odd-row list, the sticky
# overflow flag, entries in the row log
P_ROW_BASE, P_N_ODD, P_POISON, P_N_LOG = 0, 1, 2, 3
SPILL_CAP = 1 << 22         # doubles: values of columns with more than 128 events (a stalled read) while numpy's halving is replayed;
                            # the initial size of the arena, which a chunk that needs more grows (and runs again)
ODD_CAP = 1 << 16           # rows whose closing contig differs from their window's (reference quirk Q4); merged on the host


def require_cuda():
    if not torch.cuda.is_available():
        raise _lib.McallerCudaError("mcaller_b200 needs a CUDA device (B200, sm_100a); there is no CPU fallback")


class ChunkResult(object):
    """Device-side results of one chunk plus the scalar counters copied to the host.  `n_calls` rows start at
    `calls_dev`: slot 0 is the window carried in from the previous chunk (kind MC_NONE when there was none or this
    chunk has no kept line to close it), the chunk's own rows follow; a row with close_rec == 0xFFFFFFFF is still open
    and will be slot 0 of a later chunk."""
    __slots__ = ("n_calls", "n_records", "n_segments", "counters", "calls_dev", "missing_quality", "stats", "nbytes")

    def calls(self):
        """All rows (kinds 0/1/2/3) as a host numpy structured array (D2H copy)."""
        if self.n_calls == 0:
            return np.zeros(0, dtype=CALL_DTYPE)
        raw = self.calls_dev[: self.n_calls * CALL_DTYPE.itemsize].cpu().numpy()
        return raw.view(CALL_DTYPE)


class Engine(object):
    def __init__(self, refindex, models=None, qual_table=None, skip_thresh=0, qual_thresh=0.0, two_models=False,
                 device="cuda", dense=None, histogram=True):
        require_cuda()
        self.L = _lib.lib()
        self.ref = refindex
        self.models = models
        self.device = torch.device(device)
        if self.device.index is None:
            self.device = torch.device("cuda", torch.cuda.current_device())
        if refindex.device != self.device:
            raise ValueError("reference index lives on %s, engine on %s" % (refindex.device, self.device))
        self.skip_thresh = int(skip_thresh)
        self.qual_thresh = float(qual_thresh)
        self.two_models = 1 if two_models else 0
        # scan mode: 1 = every kept line gets a record; 0 = candidates, their successors and run-first lines; 2 = mode 0 plus
        # the first kept line of every read -- the -q filter drops whole reads, and a window left open at the end of a read
        # is closed by the first kept line of the next read that passes (extract_contexts.py:167 before :179)
        self.dense = bool(dense) if dense is not None else False
        self.scan_mode = 1 if self.dense else (2 if self.qual_thresh > 0.0 else 0)
        with torch.cuda.device(self.device):
            if qual_table is None:
                qual_table = np.zeros(16, dtype=_lib.QUAL_DTYPE)
            if hasattr(qual_table, "table") and hasattr(qual_table, "size"):          # read_qual.DeviceQualityTable
                self.qual_table_size = int(qual_table.size)
                self.d_qual = qual_table.table
            else:
                self.qual_table_size = len(qual_table)
                self.d_qual = torch.from_numpy(qual_table.view(np.uint8).reshape(-1).copy()).to(self.device)
            self.histogram = histogram
            ns = max(refindex.n_sites, 1)
            # depth | meth in one buffer so a multi-GPU run combines both with one SUM all-reduce
            self.d_counts = torch.zeros(2 * ns, dtype=torch.int32, device=self.device)
            self.d_depth, self.d_meth = self.d_counts[:ns], self.d_counts[ns:]
            self.d_first = torch.full((ns,), 2 ** 63 - 1, dtype=torch.int64, device=self.device)   # 'never seen'
            self._bufs = {}
            self.d_small = torch.zeros(S_WORDS, dtype=torch.int64, device=self.device)      # per-chunk status block
            self.d_persist = torch.zeros(8, dtype=torch.int64, device=self.device)          # row base, odd-row count
            self.d_carry = torch.zeros(CARRY_BYTES, dtype=torch.uint8, device=self.device)
            self.d_carry_out = torch.zeros(CALL_DTYPE.itemsize, dtype=torch.uint8, device=self.device)
            self.d_odd = torch.zeros(ODD_CAP * CALL_DTYPE.itemsize, dtype=torch.uint8, device=self.device)
            self.spill_cap = SPILL_CAP
            self.d_spill = torch.zeros(self.spill_cap, dtype=torch.float64, device=self.device)
            self.h_small = np.zeros(S_WORDS, dtype=np.uint64)
            self.rec_per_byte = self.call_per_byte = self.seg_per_byte = 0.0     # largest demand per text byte seen so far
            self.launches = 0
            self.redone = 0                   # chunks run a second time because a buffer was too small
            self.scan_events = None           # set to [] to collect (start, end) CUDA events around the scan kernel
            self.d_log = None                 # row log (enable_row_log): off unless a per-read summary is asked for
            self.reset_stream_state()

    # ---- buffers -----------------------------------------------------------------------------------------------
    def _buf(self, name, nbytes):
        nbytes = int(max(nbytes, 256))
        t = self._bufs.get(name)
        if t is None or t.numel() < nbytes:
            t = torch.empty(int(nbytes * 1.25) + 256, dtype=torch.uint8, device=self.device)
            self._bufs[name] = t
        return t

    def _sptr(self):
        # launches go to torch's current stream: wrap calls in `with torch.cuda.stream(s)` to use another one
        return C.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)

    def _status_ptr(self, slot):
        return C.c_void_p(self.d_small.data_ptr() + 8 * slot)

    def _persist_ptr(self, slot):
        return C.c_void_p(self.d_persist.data_ptr() + 8 * slot)

    def _read_status(self):
        check(self.L.mc_read_u64(C.c_void_p(self.d_small.data_ptr()), S_WORDS, self.h_small.ctypes.data_as(C.c_void_p), self._sptr()))
        return self.h_small

    @staticmethod
    def padded_capacity(nbytes):
        return ((nbytes + 15) // 16) * 16 + MC_TEXT_PAD + 64

    def upload(self, data):
        """Host bytes -> device text tensor with the '\\n' padding the scan kernel requires."""
        n = len(data)
        t = torch.full((self.padded_capacity(n),), 10, dtype=torch.uint8, device=self.device)
        if n:
            t[:n] = torch.from_numpy(np.frombuffer(data, dtype=np.uint8).copy()).to(self.device)
        return t

    # ---- cross-chunk state -------------------------------------------------------------------------------------
    def reset_stream_state(self, row_base=0):
        """Start of a byte range / file: no window carried in, first-seen row numbering restarts at row_base."""
        check(self.L.mc_carry_reset(C.c_void_p(self.d_carry.data_ptr()), self._sptr()))
        self.d_persist[:2].zero_()                # row base, odd-row count (the sticky overflow flag stays)
        if row_base:
            self.d_persist[P_ROW_BASE] = int(row_base)
        self.launches += 1

    def reset_histogram(self, row_base=0):
        self.d_counts.zero_()
        self.d_first.fill_(2 ** 63 - 1)
        if self.d_log is not None:
            self.d_persist[P_N_LOG] = 0
            self.log_bound = 0
        self.reset_stream_state(row_base)

    # ---- row log (make_bed --vo / -p summaries of the multi-GPU product path) ---------------------------------------------
    def enable_row_log(self, n_feat=0, site_flags=None):
        """Log every row the histogram counts (mc_rowlog_append): global row index, site slot, probability and, with
        n_feat > 0, the first n_feat features.  site_flags (uint8 per site slot, host or device) restricts the log to the
        flagged site slots; rows closed by another contig's line are always logged."""
        if not (self.histogram and self.models is not None):
            raise ValueError("the row log needs the histogram and the models")
        self.log_nfeat = int(n_feat)
        self.log_stride = int(self.L.mc_rowlog_stride(self.log_nfeat))
        self.d_log_flags = None
        if site_flags is not None:
            self.d_log_flags = torch.as_tensor(np.ascontiguousarray(site_flags, dtype=np.uint8)).to(self.device)
        self.log_cap = 0
        # entries logged so far as the host knows them without a synchronisation of its own: the exact count from each
        # chunk's status read (S_NLOG), a chunk's row capacity where no status is read
        self.log_bound = 0
        self.d_log = torch.empty(0, dtype=torch.uint8, device=self.device)
        self.d_persist[P_N_LOG] = 0
        self._log_room(1 << 16)

    def _log_room(self, rows):
        """Grow the log so that `rows` more entries fit after every entry that may have been logged so far."""
        need = self.log_bound + int(rows)
        if need <= self.log_cap:
            return
        cap = max(need, 2 * self.log_cap)
        new = torch.empty(cap * self.log_stride, dtype=torch.uint8, device=self.device)
        if self.log_cap:
            new[:self.log_cap * self.log_stride].copy_(self.d_log)
        self.d_log, self.log_cap = new, cap

    def _log_rows(self, d_calls, d_nrows, row_cap, d_row_base, d_n_added, d_abort):
        V = C.c_void_p
        flags = V(self.d_log_flags.data_ptr()) if self.d_log_flags is not None else None
        check(self.L.mc_rowlog_append(d_calls, d_nrows, row_cap, d_row_base, flags, self.ref.n_sites, self.log_nfeat,
                                      V(self.d_log.data_ptr()), self.log_cap, self._persist_ptr(P_N_LOG), d_n_added, d_abort,
                                      self._sptr()))
        self.launches += 1

    def row_log(self):
        """(uint8 device tensor of the logged entries, their count) -- 8-byte D2H, synchronises."""
        if self.d_log is None:
            raise ValueError("the row log is not enabled")
        n = int(self.d_persist[P_N_LOG].item())
        if n > self.log_cap:
            raise _lib.McallerCudaError("row log holds %d entries, capacity %d" % (n, self.log_cap))
        return self.d_log[:n * self.log_stride], n

    def carry_state(self):
        """(open window carried out of the last chunk?, contig of the first kept line since the reset or -1) -- 16-byte D2H."""
        tail = self.d_carry[CALL_DTYPE.itemsize:CALL_DTYPE.itemsize + 8].cpu().numpy()
        return bool(tail.view(np.uint32)[0]), int(tail.view(np.int32)[1])

    def first_kept_contig_dev(self):
        """int64 device tensor [1]: contig of the first kept line since the reset, -1 if none (for an all-gather over ranks)."""
        return self.d_carry[CALL_DTYPE.itemsize + 4:CALL_DTYPE.itemsize + 8].view(torch.int32).to(torch.int64)

    def close_carry(self, closing_contig=-1, next_contigs=None, start=0, fetch=True):
        """End of the byte range: the window still open is closed by the first kept line after the range -- its contig is
        `closing_contig` (found by the host) or the first entry >= 0 of next_contigs[start:] (int64 device tensor: the
        first kept contigs of the following ranks).  The completed row enters the histogram after all rows of this range.
        Returns the row as a 1-element host array (kind MC_NONE when there was nothing to close) or None when not fetched."""
        hist = self.histogram and self.models is not None
        cnt = int(next_contigs.numel()) if next_contigs is not None else 0
        # first-seen index: after every row of this range (the device-side row base has advanced past them)
        check(self.L.mc_carry_close(C.c_void_p(self.d_carry.data_ptr()), int(closing_contig),
                                    C.c_void_p(next_contigs.data_ptr()) if next_contigs is not None else None, int(start), cnt,
                                    C.c_void_p(self.d_carry_out.data_ptr()),
                                    C.c_void_p(self.d_depth.data_ptr()) if hist else None, C.c_void_p(self.d_meth.data_ptr()) if hist else None,
                                    C.c_void_p(self.d_first.data_ptr()) if hist else None, self.ref.n_sites,
                                    self._persist_ptr(P_ROW_BASE), self._sptr()))
        self.launches += 1
        if hist and self.d_log is not None:
            self._log_room(1)
            self._log_rows(C.c_void_p(self.d_carry_out.data_ptr()), None, 1, None, None, None)    # its index is in pad1/pad2
            self.log_bound += 1
        if not fetch:
            return None
        return self.d_carry_out.cpu().numpy().view(CALL_DTYPE)

    # ---- the pipeline --------------------------------------------------------------------------------------------
    def _default_rec_cap(self, nbytes, n_tiles):
        # sparse mode: ~3 records per 29-line chunk plus the reservation blocks of the resident warps
        slack = 256 * min(n_tiles, 8192) + 4096
        return (nbytes // 24 + slack) if self.dense else (nbytes // 1024 + 2 * n_tiles + slack)

    def _caps(self, nbytes, n_tiles):
        """Capacities only size launches and buffers: heuristics for the first chunk, afterwards what the chunks so far needed
        per byte of text (+25 %); a chunk that outgrows them is run again (mc_chunk_guard)."""
        slack = 256 * min(n_tiles, 8192) + 4096
        if self.rec_per_byte:
            rec_cap = int(self.rec_per_byte * nbytes * 1.25) + slack
            call_cap = int(self.call_per_byte * nbytes * 1.25) + 1024
            seg_cap = int(self.seg_per_byte * nbytes * 1.5) + 1024
        else:
            rec_cap = self._default_rec_cap(nbytes, n_tiles)
            call_cap = rec_cap // 8 + 1024
            seg_cap = rec_cap
        rec_cap = int(min(max(rec_cap, 1), 2 ** 32 - 2))
        return rec_cap, int(max(call_cap, 1)), int(min(max(seg_cap, 1), rec_cap))

    def run_chunk(self, d_text, nbytes, rec_cap=None, call_cap=None):
        """d_text: uint8 device tensor, >= padded_capacity(nbytes) long, bytes past nbytes all '\\n'."""
        L = self.L
        if d_text.numel() < nbytes + MC_TEXT_PAD:
            raise ValueError("text tensor lacks the MC_TEXT_PAD newline padding")
        res = ChunkResult()
        res.nbytes = nbytes
        n_tiles = int(L.mc_num_tiles(nbytes))
        slack = 256 * min(n_tiles, 8192) + 4096
        if rec_cap is None and call_cap is None:
            rec_cap, call_cap, seg_cap = self._caps(nbytes, n_tiles)
        else:
            d_rec, d_call, d_seg = self._caps(nbytes, n_tiles)
            rec_cap = int(min(max(rec_cap if rec_cap is not None else d_rec, 1), 2 ** 32 - 2))
            call_cap = int(max(call_cap if call_cap is not None else d_call, 1))
            seg_cap = int(min(d_seg, rec_cap))
        attempts = 0
        while True:
            cnt = self._launch_chunk(d_text, nbytes, n_tiles, rec_cap, call_cap, seg_cap)
            reserved, n_rec, n_calls, n_seg = int(cnt[C_RECORDS]), int(cnt[S_NREC]), int(cnt[S_NCALLS]), int(cnt[S_NSEG])
            if nbytes > 0:
                self.rec_per_byte = max(self.rec_per_byte, reserved / nbytes)
                self.call_per_byte = max(self.call_per_byte, n_calls / nbytes)
                self.seg_per_byte = max(self.seg_per_byte, n_seg / nbytes)
            if not cnt[S_ABORT]:
                break
            self.redone += 1
            attempts += 1
            if attempts > 6:
                raise _lib.McallerCudaError("chunk keeps overflowing its buffers (counters: %s)" % list(map(int, cnt[:MC_C_COUNT])))
            if cnt[C_OVERFLOW] or reserved > rec_cap:
                if rec_cap >= 2 ** 32 - 2:
                    raise _lib.McallerCudaError("chunk produces more than 2^32 records; use smaller chunks")
                rec_cap = int(min(max(reserved, rec_cap * 2 if cnt[C_OVERFLOW] and reserved <= rec_cap else 0) + slack, 2 ** 32 - 2))
                call_cap = max(call_cap, rec_cap // 8 + 1024)
            elif n_seg > seg_cap:
                seg_cap = min(n_seg + 1024, rec_cap)
            else:
                over = int(cnt[S_CALL_OVERFLOW])           # k_check_cap: bit 0 rows over call_cap, bits 1-63 spill demand
                if over & 1:
                    call_cap = n_calls + 1024
                if over >> 1:
                    self.spill_cap = int((over >> 1) * 1.25)
                    self.d_spill = torch.empty(self.spill_cap, dtype=torch.float64, device=self.device)
        if attempts:
            self.d_persist[P_POISON] = 0              # the overflow was handled here: nothing is pending for overflowed()
        res.counters = {nm: int(cnt[i]) for i, nm in enumerate(_lib.COUNTER_NAMES)}
        res.n_records = n_rec
        res.n_segments = int(cnt[S_NSEG])
        res.missing_quality = int(cnt[S_MISSING_QUAL])
        res.n_calls = int(cnt[S_NROWS])
        res.calls_dev = self._bufs["calls"]
        v = cnt[S_STATS:S_STATS + 7]
        res.stats = dict(calls=int(v[0]), pending=int(v[1]), too_many_skips=int(v[2]), multi=int(v[3]), errors=int(v[4]), methylated=int(v[5]),
                         pending_too_many_skips=int(v[6]))
        return res

    def _launch_chunk(self, d_text, nbytes, n_tiles, rec_cap, call_cap, seg_cap, read_status=True):
        """All stages of one chunk, back to back on the current stream; one status read at the end."""
        L, st = self.L, self._sptr()
        V = C.c_void_p
        tile_tab = self._buf("tile_tab", 8 * max(n_tiles, 1))
        run_len = max(int(L.mc_scan_run_len(nbytes)), 1)
        n_runs = max((n_tiles + run_len - 1) // run_len, 1)
        run_tab = self._buf("run_tab", 8 * n_runs)
        run_first = self._buf("run_first", 4 * n_runs)
        rec_a = self._buf("rec_a", 32 * rec_cap)
        rec_b = self._buf("rec_b", 32 * rec_cap)
        ws = self._buf("ws", L.mc_workspace_bytes(max(rec_cap, n_tiles)))
        seg_start = self._buf("seg_start", 4 * (rec_cap + 2))
        seg_flags = self._buf("seg_flags", 4 * rec_cap)
        seg_qual = self._buf("seg_qual", 8 * seg_cap)
        seg_count = self._buf("seg_count", 4 * seg_cap)
        calls = self._buf("calls", CALL_DTYPE.itemsize * (call_cap + 1))          # slot 0 + the chunk's rows
        self.d_small.zero_()
        if self.scan_events is not None:
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
        check(L.mc_scan(V(d_text.data_ptr()), nbytes, self.ref.ref(), self.scan_mode, V(rec_a.data_ptr()), rec_cap,
                        V(tile_tab.data_ptr()), V(run_tab.data_ptr()), V(self.d_small.data_ptr()), st))
        if self.scan_events is not None:
            e1.record()
            self.scan_events.append((e0, e1))
        check(L.mc_order_records(V(d_text.data_ptr()), nbytes, self.ref.ref(), V(tile_tab.data_ptr()), n_tiles, V(run_tab.data_ptr()), run_len, V(rec_a.data_ptr()), rec_cap,
                                 V(self.d_small.data_ptr()), V(rec_b.data_ptr()), rec_cap, self._status_ptr(S_NREC), V(seg_flags.data_ptr()),
                                 V(run_first.data_ptr()), V(ws.data_ptr()), st))
        check(L.mc_segment_reads(V(d_text.data_ptr()), V(rec_b.data_ptr()), self._status_ptr(S_NREC), rec_cap, V(seg_flags.data_ptr()), V(run_first.data_ptr()),
                                 n_runs if n_tiles else 0, V(seg_start.data_ptr()),
                                 self._status_ptr(S_NSEG), V(ws.data_ptr()), st))
        check(L.mc_segment_quality(V(d_text.data_ptr()), V(rec_b.data_ptr()), V(seg_start.data_ptr()), self._status_ptr(S_NSEG), seg_cap,
                                   V(self.d_qual.data_ptr()), self.qual_table_size, V(seg_qual.data_ptr()), self._status_ptr(S_MISSING_QUAL), st))
        rows1 = V(calls.data_ptr() + CALL_DTYPE.itemsize)
        check(L.mc_build_windows(V(rec_b.data_ptr()), self._status_ptr(S_NREC), rec_cap, V(seg_start.data_ptr()), self._status_ptr(S_NSEG),
                                 seg_cap, V(seg_qual.data_ptr()), self.ref.ref(), self.skip_thresh, self.qual_thresh, self.two_models,
                                 rows1, call_cap, V(seg_count.data_ptr()), self._status_ptr(S_NCALLS), V(ws.data_ptr()),
                                 V(self.d_spill.data_ptr()), self.spill_cap, st))
        check(L.mc_chunk_guard(V(self.d_small.data_ptr()), rec_cap, self._status_ptr(S_NREC), rec_cap, self._status_ptr(S_NSEG), seg_cap,
                               self._status_ptr(S_NCALLS), call_cap, self._status_ptr(S_ABORT), self._persist_ptr(P_POISON), st))
        check(L.mc_carry_rows(V(calls.data_ptr()), self._status_ptr(S_NCALLS), V(rec_b.data_ptr()), self._status_ptr(S_NREC),
                              V(seg_start.data_ptr()), self._status_ptr(S_NSEG), V(seg_qual.data_ptr()), self.qual_thresh,
                              V(self.d_carry.data_ptr()), self._status_ptr(S_NROWS), self._status_ptr(S_ABORT), st))
        # 1 scan + 5 order (run resolution, 3 scan kernels, gather + finish) + 5 segmentation + 1 quality
        # + 7 windows (first-'M', 2 passes, 3 scan kernels, capacity check) + guard + carry
        self.launches += 1 + 5 + 5 + 1 + 7 + 2
        if self.models is not None:
            cls_ws = self._buf("cls_ws", L.mc_classify_workspace_bytes(call_cap + 1))
            check(L.mc_classify(V(calls.data_ptr()), self._status_ptr(S_NROWS), call_cap + 1, self.models.array, V(cls_ws.data_ptr()), st))
            self.launches += 2                       # index list of the call rows + the classifier
            if self.histogram:
                if self.d_log is not None:
                    # before mc_hist_accumulate, which advances the row base past this chunk
                    self._log_room(call_cap + 1)
                    self._log_rows(V(calls.data_ptr()), self._status_ptr(S_NROWS), call_cap + 1, self._persist_ptr(P_ROW_BASE),
                                   self._status_ptr(S_NLOG), self._status_ptr(S_ABORT))
                check(L.mc_hist_accumulate(V(calls.data_ptr()), self._status_ptr(S_NROWS), call_cap + 1, V(self.d_depth.data_ptr()),
                                           V(self.d_meth.data_ptr()), V(self.d_first.data_ptr()), self.ref.n_sites, self._persist_ptr(P_ROW_BASE),
                                           V(self.d_odd.data_ptr()), ODD_CAP, self._persist_ptr(P_N_ODD), self._status_ptr(S_ABORT), st))
                self.launches += 2
        check(L.mc_count_calls(V(calls.data_ptr()), self._status_ptr(S_NROWS), call_cap + 1, self._status_ptr(S_STATS), st))
        self.launches += 1
        log = self.d_log is not None and self.models is not None and self.histogram
        if not read_status:
            if log:
                self.log_bound += call_cap + 1
            return None
        cnt = self._read_status().copy()
        if log:
            self.log_bound += int(cnt[S_NLOG])            # 0 when the chunk overflowed and logged nothing
        return cnt

    def launch_chunk(self, d_text, nbytes):
        """Queues every stage of a chunk WITHOUT reading its status: for back-to-back passes over inputs whose buffer needs are
        already known (a repeated benchmark step).  Capacities come from the chunks seen so far; should one overflow anyway
        the device keeps a sticky flag (`overflowed()`) and leaves all cross-chunk state untouched for that chunk."""
        if not self.rec_per_byte:
            raise _lib.McallerCudaError("launch_chunk needs a preceding run_chunk (capacities are learned from it)")
        n_tiles = int(self.L.mc_num_tiles(nbytes))
        rec_cap, call_cap, seg_cap = self._caps(nbytes, n_tiles)
        self._launch_chunk(d_text, nbytes, n_tiles, rec_cap, call_cap, seg_cap, read_status=False)

    def overflowed(self, clear=True):
        """Did any chunk since the last check outgrow its buffers (8-byte D2H, synchronises)?"""
        v = int(self.d_persist[P_POISON].item())
        if clear and v:
            self.d_persist[P_POISON] = 0
        return bool(v)

    def count_rows(self, res):
        """Row statistics of a chunk (computed on the device as part of run_chunk)."""
        return dict(res.stats)

    def records(self, n_rec):
        """Ordered stage-1 records of the last chunk (host copy; test helper)."""
        return self._bufs["rec_b"][: n_rec * 32].cpu().numpy().view(RECORD_DTYPE)

    def histogram_host(self):
        return (self.d_depth.cpu().numpy().view(np.uint32), self.d_meth.cpu().numpy().view(np.uint32),
                self.d_first.cpu().numpy().view(np.uint64))

    def bed_select(self, depth_thresh, mod_thresh, control=False):
        """check_thresh (make_bed.py:21-28) over the device histogram -> (uint8 device tensor of flags per site slot, int64
        device tensor [1] with their count); asynchronous."""
        ns = max(self.ref.n_sites, 1)
        if getattr(self, "d_bed_flags", None) is None:
            self.d_bed_flags = torch.zeros(ns, dtype=torch.uint8, device=self.device)
            self.d_bed_count = torch.zeros(1, dtype=torch.int64, device=self.device)
        check(self.L.mc_bed_select(C.c_void_p(self.d_depth.data_ptr()), C.c_void_p(self.d_meth.data_ptr()), self.ref.n_sites, int(depth_thresh),
                                   float(mod_thresh), 1 if control else 0, C.c_void_p(self.d_bed_flags.data_ptr()),
                                   C.c_void_p(self.d_bed_count.data_ptr()), self._sptr()))
        self.launches += 1
        return self.d_bed_flags, self.d_bed_count

    def odd_rows(self):
        """Rows the histogram could not key by site slot (closing contig != window contig, quirk Q4), with their global row
        index in pad1/pad2 -> host structured array."""
        n = int(self.d_persist[P_N_ODD].item())
        if n > ODD_CAP:
            raise _lib.McallerCudaError("more than %d rows close on another contig than their window's" % ODD_CAP)
        return self.d_odd[: n * CALL_DTYPE.itemsize].cpu().numpy().view(CALL_DTYPE)
