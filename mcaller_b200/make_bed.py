"""Drop-in replacement for the hot part of the reference's make_bed.py: `aggregate_by_pos` (make_bed.py:67-164) and
`check_thresh` (:21-28) with the same signatures.  The per-position depth / methylated counts are built on the GPU
(mc_diffs_aggregate_ex: tab-split of the `.diffs.<k>` rows + integer atomics in a hash table); the host formats the
BED/GFF rows of the surviving loci in first-seen order.

Variants (SURVEY.md section 8f rank 3):
* `--vo` (verbose_results): the GPU indexes the used rows (mc_diffs_rows); the host joins the probability strings of each
  locus in file order (:158-159) and, with `--gff`, calls the same scipy/numpy functions as the reference on them
  (fracLow / fracUp / identificationQv, :147-151).
* `-p positions`: rows are filtered on the GPU through a hash set of the positions file; the per-locus, per-column
  one-sample t-tests of :115-127 are computed from exactly parsed values with numpy's summation order on the GPU
  (mc_diffs_colstats) and finished (Student-t tail, -log10, rounding) on the host with scipy's own special function.
`--plot` / `--plotsummary` (matplotlib figures) are out of scope and raise NotImplementedError.  The reference's debugging
`print(values_dict)` / `print(aggfi)` lines are not reproduced.
"""
import ctypes as C
import os

import numpy as np

LOCUS_DTYPE = np.dtype([("hash", "<u8"), ("first_off", "<u8"), ("check", "<u8"), ("depth", "<u4"), ("meth", "<u4")])

_FNV_OFF, _FNV_PRIME, _M64 = 14695981039346656037, 1099511628211, (1 << 64) - 1


def check_thresh(locus_list, mod_thresh, depth_thresh, control):
    """reference make_bed.py:21-28 on a 0/1 list (kept for API compatibility)."""
    if len(locus_list) >= depth_thresh:
        frac = np.mean(locus_list)
        if not control and frac >= mod_thresh:
            return True
        if control and frac < mod_thresh:
            return True
        return False


def _check_counts(depth, meth, mod_thresh, depth_thresh, control):
    if depth >= depth_thresh:
        frac = np.float64(meth) / np.float64(depth)        # np.mean of a 0/1 list
        return (not control and frac >= mod_thresh) or (control and frac < mod_thresh)
    return False


def make_pos_set(pos_list):
    """reference make_bed.py:13-19."""
    pos_set = set()
    with open(pos_list, "r") as fi:
        for line in fi:
            if len(line) > 3:
                pos_set.add(tuple(line.strip().split("\t")[:4]))
    return pos_set


def _fnv(parts):
    h = _FNV_OFF
    for i, part in enumerate(parts):
        if i:
            h = ((h ^ 9) * _FNV_PRIME) & _M64
        for b in part:
            h = ((h ^ b) * _FNV_PRIME) & _M64
    return h or 1


def _pos_keys(pos_set):
    """(chrom, pos, strand) of the entries a row can match: the reference tests (csome, pos, str(int(pos)+1), strand) in
    pos_set (:83-84), so an entry whose end column is not start + 1 never matches."""
    keys = set()
    for t in pos_set:
        if len(t) != 4:
            continue
        chrom, start, end, strand = t
        try:
            if str(int(start) + 1) != end:
                continue
        except ValueError:
            continue
        keys.add((chrom, start, strand))
    return keys


def _pos_hash_set(pos_set):
    """Open-addressing set of FNV-1a("chrom\\tpos\\tstrand") of _pos_keys(pos_set)."""
    keys = set(_fnv([chrom.encode(), start.encode(), strand.encode()]) for chrom, start, strand in _pos_keys(pos_set))
    size = 64
    while size < 2 * len(keys) + 2:
        size *= 2
    tab = np.zeros(size, dtype=np.uint64)
    mask = size - 1
    for k in keys:
        s = k & mask
        while tab[s] != 0 and tab[s] != k:
            s = (s + 1) & mask
        tab[s] = k
    return tab


STREAM_BYTES = int(os.environ.get("MCALLER_B200_BED_CHUNK_BYTES", str(256 << 20)))     # piece size of the streamed `.diffs` file


def _empty_table(torch, size, dev):
    init = np.zeros(size, dtype=LOCUS_DTYPE)
    init["first_off"] = np.uint64(0xFFFFFFFFFFFFFFFF)
    return torch.from_numpy(init.view(np.uint8).reshape(-1)).to(dev)


class _Aggregation(object):
    """GPU passes over one `.diffs.<k>` file.  The default mode streams the file in line-aligned pieces into one device
    locus table that grows with the loci seen (the reference streams line by line, make_bed.py:75); the modes that need
    per-read lists (-p, --vo) keep the whole file on the device for their second pass."""

    def __init__(self, meth_fi, pos_set=None, keep_text=None):
        import torch
        from . import _lib, engine
        engine.require_cuda()
        self.torch, self._lib, self.L = torch, _lib, _lib.lib()
        self.path = meth_fi
        self.n = os.path.getsize(meth_fi)
        self.dev = torch.device("cuda", torch.cuda.current_device())
        self.loci = []            # (chrom, pos, context, strand, depth, meth) in first-seen order
        self.slots = np.zeros(0, dtype=np.int64)
        self.counters = np.zeros(8, dtype=np.int64)
        self.data = None
        if keep_text is None:
            keep_text = pos_set is not None       # the per-read passes (index_rows / column_tests) need the text on the device
        if self.n == 0:
            return
        self.d_posset = None
        self.posset_size = 0
        if pos_set is not None:
            tab = _pos_hash_set(pos_set)
            self.d_posset = torch.from_numpy(tab.view(np.int64)).to(self.dev)
            self.posset_size = len(tab)
        self.d_cnt = torch.zeros(8, dtype=torch.int64, device=self.dev)
        self.table_size = 1024
        self.d_table = _empty_table(torch, self.table_size, self.dev)
        n_loci = 0
        if keep_text:
            self.data = open(meth_fi, "rb").read()
            self.d_text = torch.from_numpy(np.frombuffer(self.data, dtype=np.uint8).copy()).to(self.dev)
            self._ensure_room(n_loci, self.n)
            _lib.check(self.L.mc_diffs_aggregate_ex(self._p(self.d_text), self.n, 0, self._p(self.d_posset), self.posset_size,
                                                    self._p(self.d_table), self.table_size, self._p(self.d_cnt), self._stream()))
        else:
            with open(meth_fi, "rb") as fh:
                base, carry = 0, b""
                while True:
                    piece = fh.read(STREAM_BYTES)
                    buf = carry + piece
                    if not buf:
                        break
                    if piece:
                        cut = buf.rfind(b"\n") + 1
                        if cut == 0:                              # no complete line yet
                            carry = buf
                            continue
                    else:
                        cut = len(buf)                            # last line without a newline
                    self._ensure_room(n_loci, cut)
                    d_piece = torch.from_numpy(np.frombuffer(buf, dtype=np.uint8, count=cut).copy()).to(self.dev)
                    _lib.check(self.L.mc_diffs_aggregate_ex(self._p(d_piece), cut, base, self._p(self.d_posset), self.posset_size,
                                                            self._p(self.d_table), self.table_size, self._p(self.d_cnt), self._stream()))
                    n_loci = int((self.d_table.view(torch.int64).view(-1, 4)[:, 0] != 0).sum().item())
                    base += cut
                    carry = buf[cut:]
                    if not piece:
                        break
        cnt = self.d_cnt.cpu().numpy()
        self.counters = cnt
        if cnt[1]:
            raise ValueError("%d rows of %s do not have 7 or 8 tab-separated fields" % (cnt[1], meth_fi))
        if cnt[3]:
            raise RuntimeError("locus table overflow")
        if cnt[7]:
            raise RuntimeError("%d rows of %s collide with another locus in the 64-bit key hash" % (cnt[7], meth_fi))
        table = self.d_table.cpu().numpy().view(LOCUS_DTYPE)
        used = np.nonzero(table["hash"] != 0)[0]
        order = np.argsort(table["first_off"][used], kind="stable")
        self.slots = used[order]                              # table slot of each locus, first-seen order
        with open(meth_fi, "rb") as fh:
            for e in table[self.slots]:
                fh.seek(int(e["first_off"]))
                f = fh.readline().rstrip(b"\n").split(b"\t")
                self.loci.append((f[0].decode(), f[2].decode(), f[3].decode(), f[5].decode(), int(e["depth"]), int(e["meth"])))

    def _ensure_room(self, n_loci, piece_bytes):
        """The table keeps a load factor <= 0.5 even if every row of the next piece were a new locus (a row is >= 48 bytes)."""
        need = 2 * (n_loci + piece_bytes // 48 + 16)
        if self.table_size >= need:
            return
        size = self.table_size
        while size < need:
            size *= 2
        new = _empty_table(self.torch, size, self.dev)
        self._lib.check(self.L.mc_diffs_rehash(self._p(self.d_table), self.table_size, self._p(new), size, self._p(self.d_cnt), self._stream()))
        self.d_table, self.table_size = new, size

    def _p(self, t):
        return C.c_void_p(t.data_ptr()) if t is not None else C.c_void_p(0)

    def _stream(self):
        return C.c_void_p(self.torch.cuda.current_stream(self.dev).cuda_stream)

    def index_rows(self):
        """Row index grouped by locus (first-seen order) and in file order inside a locus: (rows, order, locus_off)."""
        torch, _lib = self.torch, self._lib
        n_rows = int(sum(l[4] for l in self.loci))
        self.n_rows = n_rows
        if n_rows == 0:
            self.rows = np.zeros(0, dtype=_lib.DIFFS_ROW_DTYPE)
            self.order = np.zeros(0, dtype=np.uint32)
            self.locus_off = np.zeros(len(self.loci) + 1, dtype=np.uint32)
            return
        self.d_rows = torch.zeros(n_rows * _lib.DIFFS_ROW_DTYPE.itemsize, dtype=torch.uint8, device=self.dev)
        d_n = torch.zeros(1, dtype=torch.int64, device=self.dev)
        _lib.check(self.L.mc_diffs_rows(self._p(self.d_text), self.n, self._p(self.d_posset), self.posset_size, self._p(self.d_table),
                                        self.table_size, self._p(self.d_rows), n_rows, self._p(d_n), self._stream()))
        got = int(d_n.cpu()[0])
        if got != n_rows:
            raise RuntimeError("row index holds %d rows, the locus table counted %d" % (got, n_rows))
        rows = self.d_rows.cpu().numpy().view(_lib.DIFFS_ROW_DTYPE)
        rank = np.full(self.table_size, -1, dtype=np.int64)
        rank[self.slots] = np.arange(len(self.slots))
        self.rows = rows
        self.order = np.lexsort((rows["line_off"], rank[rows["slot"]])).astype(np.uint32)
        depth = np.array([l[4] for l in self.loci], dtype=np.int64)
        self.locus_off = np.concatenate([[0], np.cumsum(depth)]).astype(np.uint32)

    def prob_strings(self, li):
        """pos_dict_verbose[locus] (:96-97): the stripped probability column of the locus's rows, file order."""
        out = []
        for j in self.order[self.locus_off[li]:self.locus_off[li + 1]]:
            r = self.rows[j]
            a = int(r["line_off"]) + int(r["prob_off"])
            out.append(self.data[a:a + int(r["prob_len"])].decode())
        return out

    def column_tests(self):
        """values_dict[locus] of :115-127: [np.round(max t, 3), np.round(sum -log10 p, 3)] per locus."""
        torch, _lib = self.torch, self._lib
        n_loci = len(self.loci)
        if n_loci == 0:
            return []
        # number of columns = features per row minus the trailing read quality (:91); taken from the first used row
        r0 = self.rows[self.order[0]]
        a = int(r0["line_off"]) + int(r0["values_off"])
        ncols = len(self.data[a:a + int(r0["values_len"])].split(b",")) - 1
        if ncols < 1 or ncols > _lib.MC_MAXK + 1:
            raise ValueError("rows of %s hold %d feature columns" % (self.path, ncols))
        d_order = torch.from_numpy(self.order.astype(np.int32)).to(self.dev)
        d_off = torch.from_numpy(self.locus_off.astype(np.int32)).to(self.dev)
        d_vals = torch.zeros(self.n_rows * (_lib.MC_MAXK + 1), dtype=torch.float64, device=self.dev)
        d_ncol = torch.zeros(self.n_rows, dtype=torch.int32, device=self.dev)
        d_stats = torch.zeros(n_loci * ncols * 2, dtype=torch.float64, device=self.dev)
        _lib.check(self.L.mc_diffs_colstats(self._p(self.d_text), self._p(self.d_rows), self._p(d_order), self.n_rows, self._p(d_off),
                                            n_loci, ncols, self._p(d_vals), self._p(d_ncol), self._p(d_stats), self._p(self.d_cnt),
                                            self._stream()))
        cnt = self.d_cnt.cpu().numpy()
        self.counters = cnt
        if cnt[6]:
            raise ValueError("%d feature values of %s are not plain floats" % (cnt[6], self.path))
        ncol = d_ncol.cpu().numpy()
        self.vals = d_vals.cpu().numpy().reshape(self.n_rows, _lib.MC_MAXK + 1)     # parsed features, grouped row order
        if (ncol != ncols).any():
            raise ValueError("rows of %s do not all hold %d feature columns" % (self.path, ncols))
        return ttest_finish(d_stats.cpu().numpy().reshape(n_loci, ncols, 2), self.locus_off)


def ttest_finish(stats, locus_off):
    """values_dict[locus] of :115-127 from the device statistics: stats[n_loci][ncols][2] = (np.mean(x), np.add.reduce((x -
    mean)**2)) per locus and column, locus_off[n_loci + 1] the CSR of the rows -> [np.round(max t, 3), np.round(sum -log10 p,
    3)] per locus (Student-t tail, -log10 and rounding as the reference's scipy / numpy calls)."""
    import warnings
    from scipy import special
    n_loci, ncols = stats.shape[0], stats.shape[1]
    locus_off = np.asarray(locus_off)
    n = (locus_off[1:].astype(np.int64) - locus_off[:-1].astype(np.int64)).astype(np.float64)[:, None]
    out = []
    with warnings.catch_warnings(), np.errstate(all="ignore"):
        warnings.simplefilter("ignore")
        # scipy.stats.ttest_1samp(x, 0): mean, _var = mean((x-mean)**2) * (n / (n-1)), t = mean / sqrt(var / n),
        # p = 2 * stdtr(n-1, -|t|)
        mean = stats[:, :, 0]
        var = (stats[:, :, 1] / n) * (n / (n - 1.0))
        t = mean / np.sqrt(var / n)
        p = 2 * special.stdtr(n - 1.0, -np.abs(t))
        for li in range(n_loci):
            pvals = [(p[li, c], t[li, c]) for c in range(ncols)]
            pval = (sum([-np.log10(x[0]) for x in pvals]), max([x[1] for x in pvals]))
            out.append([np.round(x, 3) for x in [pval[1], pval[0]]])
    return out


def count_loci(meth_fi):
    """GPU pass over the file -> list of (chrom, pos, context, strand, depth, meth) in first-seen order."""
    return _Aggregation(meth_fi).loci


def _read_fasta(ref):
    seqs = {}
    name, parts = None, []
    for ln in open(ref):                         # make_bed.py:36-40 keeps the case of the file
        if ln.startswith(">"):
            if name is not None:
                seqs[name] = "".join(parts)
            t = ln[1:].split()
            name, parts = (t[0] if t else ""), []
        elif name is not None:
            parts.append(ln.strip())
    if name is not None:
        seqs[name] = "".join(parts)
    return seqs


def aggregate_by_pos(meth_fi, aggfi, depth_thresh, mod_thresh, pos_list, control, verbose_results, gff, ref, plot, plotdir, plotsummary):
    """reference make_bed.py:67: default mode, --control, --gff, --ref, --vo and -p."""
    if plot or plotsummary:
        raise NotImplementedError("make_bed --plot/--plotsummary are outside the accelerated path")
    pos_set = make_pos_set(pos_list) if pos_list else None
    agg = _Aggregation(meth_fi, pos_set, keep_text=bool(verbose_results or pos_list))
    loci = agg.loci
    if verbose_results and agg.counters[5]:
        raise ValueError("--vo needs the 8-column format: %d rows of %s have no probability column" % (agg.counters[5], meth_fi))
    tests = None
    if verbose_results or pos_list:
        agg.index_rows()
    if pos_list:
        tests = agg.column_tests()
    return _write_loci(loci, aggfi, depth_thresh, mod_thresh, pos_list, control, verbose_results, gff, ref, agg, tests)


def _write_loci(loci, aggfi, depth_thresh, mod_thresh, pos_list, control, verbose_results, gff, ref, agg=None, tests=None):
    """Thresholds (check_thresh, make_bed.py:21-28) and the BED / GFF rows (:132-159) for loci in first-seen order."""
    contexts = None
    if ref:
        from . import refmark
        seqs = _read_fasta(ref)
        contexts = {}
        for chrom, pos, ctx, strand, _, _ in loci:
            if chrom in seqs:
                cx = seqs[chrom][int(pos) - 20:int(pos) + 21].upper()
                contexts[(chrom, pos, ctx, strand)] = refmark.revcomp(cx) if strand == "-" else cx
    count = 0
    with open(aggfi, "w") as outfi:
        for li, (chrom, pos, ctx, strand, depth, meth) in enumerate(loci):
            # :134-136 -- thresholds apply without -p; with -p every locus of the positions file is reported
            if not pos_list and not _check_counts(depth, meth, mod_thresh, depth_thresh, control):
                continue
            count += 1
            frac = np.float64(meth) / np.float64(depth)
            cx = contexts[(chrom, pos, ctx, strand)] if contexts is not None else ctx
            nextpos = str(int(pos) + 1)
            if gff:
                deets = "coverage=" + str(depth) + ";context=" + cx + ";IPDRatio=5;frac=" + str(frac)
                if verbose_results:                                      # :147-151
                    from scipy import stats
                    probs = [float(x) for x in agg.prob_strings(li)]
                    se_95 = 2 * stats.sem(probs)
                    deets = deets + ";fracLow=" + str(frac - se_95) + ";fracUp=" + str(frac + se_95) + ";identificationQv=" + \
                        str(int(100 * np.mean([float(x) for x in probs])))
                outfi.write("\t".join([chrom, "kinModCall", "m6A", nextpos, nextpos, "10", strand, ".", deets]) + "\n")
            else:
                out_line = "\t".join([chrom, pos, nextpos, ctx, str(frac), strand, str(depth)])
                if pos_list:
                    out_line = out_line + "\t" + "\t".join([str(x) for x in tests[li]])
                if verbose_results:
                    out_line = out_line + "\t" + ",".join(agg.prob_strings(li))
                outfi.write(out_line + "\n")
    if not pos_list:
        if not control:
            print(count, "methylated loci found with min depth", depth_thresh, "reads")
        else:
            print(count, "unmethylated loci found with min depth", depth_thresh, "reads")
    return count


def _locus_entries(refindex, depth, meth, first, odd_rows=None):
    """Loci of the device histogram in first-seen order: (locus tuple, site slot or -1, global row indices of its odd rows)."""
    depth = np.asarray(depth).astype(np.int64)
    meth = np.asarray(meth).astype(np.int64)
    first = np.asarray(first).astype(np.uint64)
    used = np.flatnonzero(depth > 0)
    entries = []                                  # (first-seen index, locus tuple, site slot, odd row indices)
    for s_ in used.tolist():
        ci, pos, rev = int(refindex.site_contig[s_]), int(refindex.site_pos[s_]), bool(refindex.site_rev[s_])
        entries.append((int(first[s_]), (refindex.names[ci], str(pos), refindex.context(ci, pos, rev), "-" if rev else "+",
                                         int(depth[s_]), int(meth[s_])), s_, ()))
    if odd_rows is not None and len(odd_rows):
        extra = {}
        for c in odd_rows:
            rev = bool(c["rev"])
            key = (refindex.names[int(c["chrom_contig"])], str(int(c["mpos"])), refindex.context(int(c["win_contig"]), int(c["mpos"]), rev),
                   "-" if rev else "+")
            idx = int(c["pad1"]) | (int(c["pad2"]) << 32)
            e = extra.setdefault(key, [idx, 0, 0, []])
            e[0] = min(e[0], idx)
            e[1] += 1
            e[2] += int(c["label"])
            e[3].append(idx)
        for key, (idx, d_, m_, rows) in extra.items():
            entries.append((idx, key + (d_, m_), -1, tuple(rows)))
    entries.sort(key=lambda t: t[0])
    return [e[1:] for e in entries]


def loci_from_histogram(refindex, depth, meth, first, odd_rows=None):
    """The per-site histogram of the fused pipeline (mc_hist_accumulate; all-reduced over the ranks of a multi-GPU run)
    -> list of (chrom, pos, context, strand, depth, meth) in first-seen order, i.e. what make_bed.py:75-98 builds from
    the `.diffs` rows.  A site slot IS the reference's key (chrom, pos, pos+1, context, strand): the context is a function of
    contig, position and strand.  `odd_rows` (Engine.odd_rows(), gathered over ranks) are the rows whose column 1 names
    another contig than their window's (reference quirk, extract_contexts.py:216): they form loci of their own."""
    return [e[0] for e in _locus_entries(refindex, depth, meth, first, odd_rows)]


def aggregate_from_histogram(refindex, depth, meth, first, aggfi, depth_thresh, mod_thresh, control=False, gff=False, ref=None,
                             odd_rows=None):
    """make_bed.py's default output (also --control / --gff / --ref) straight from the device histogram: no `.diffs` text is
    parsed.  The modes that need per-read lists (-p, --vo) take the rows the ranks logged on the device as well:
    aggregate_from_rows."""
    loci = loci_from_histogram(refindex, depth, meth, first, odd_rows)
    return _write_loci(loci, aggfi, depth_thresh, mod_thresh, None, control, False, gff, ref)


def site_flags(refindex, pos_set):
    """uint8 per site slot: 1 where the slot's (contig, str(pos), strand) -- the key a `.diffs` row of that site carries --
    matches an entry of pos_set (make_pos_set) as make_bed.py:84 matches rows."""
    flags = np.zeros(max(refindex.n_sites, 1), dtype=np.uint8)
    names = {nm: i for i, nm in enumerate(refindex.names)}
    g_site = refindex.contig_base[refindex.site_contig] + refindex.site_pos       # ascending within each strand
    nf, ns = refindex.n_fwd, refindex.n_sites
    for chrom, start, strand in _pos_keys(pos_set):
        ci = names.get(chrom)
        if ci is None or strand not in ("+", "-"):
            continue
        try:
            pos = int(start)
        except ValueError:
            continue
        if str(pos) != start or pos < 0 or pos >= int(refindex.contig_len[ci]):
            continue
        g = int(refindex.contig_base[ci]) + pos
        lo, hi = (0, nf) if strand == "+" else (nf, ns)
        j = lo + int(np.searchsorted(g_site[lo:hi], g))
        if j < hi and int(g_site[j]) == g:
            flags[j] = 1
    return flags


class _RowGroups(object):
    """The per-locus row lists of the multi-GPU product path: the rows the ranks logged on the device (mc_rowlog_append),
    gathered to this rank and grouped by locus on the device (mc_rowlog_group).  Offers what _write_loci takes from
    _Aggregation -- prob_strings(li) -- and the t-test statistics of column_tests, with no `.diffs` text."""

    def __init__(self, refindex, entries, d_log, n_log, n_feat, want_probs=True, want_vals=False):
        import torch
        from . import _lib
        self.torch, self._lib, self.L = torch, _lib, _lib.lib()
        dev = d_log.device
        self.dev = dev
        self.n_feat = int(n_feat)
        n_loci = len(entries)
        depth = np.zeros(n_loci + 1, dtype=np.uint32)
        depth[:n_loci] = [e[0][4] for e in entries]
        self.n_loci, self.n_rows = n_loci, int(depth.sum(dtype=np.int64))
        locus_of_site = np.full(max(refindex.n_sites, 1), -1, dtype=np.int32)
        odd_idx, odd_loc = [], []
        for li, (_, site, rows) in enumerate(entries):
            if site >= 0:
                locus_of_site[site] = li
            odd_idx += rows
            odd_loc += [li] * len(rows)
        o = np.argsort(np.array(odd_idx, dtype=np.uint64), kind="stable")
        odd_rows = np.array(odd_idx, dtype=np.uint64)[o]
        odd_locus = np.array(odd_loc, dtype=np.int32)[o]

        def up(a):
            return torch.from_numpy(np.ascontiguousarray(a)).to(dev)

        def p(t):
            return C.c_void_p(t.data_ptr()) if t is not None else None
        d_los, d_depth = up(locus_of_site), up(depth.view(np.int32))
        d_odd_rows, d_odd_locus = up(odd_rows.view(np.int64) if len(odd_rows) else np.zeros(1, np.int64)), up(odd_locus if len(odd_locus) else np.zeros(1, np.int32))
        d_off = torch.empty(n_loci + 1, dtype=torch.int32, device=dev)
        self.d_prob = torch.empty(max(self.n_rows, 1), dtype=torch.float64, device=dev)
        self.d_vals = self.d_ncol = None
        if want_vals:
            self.d_vals = torch.empty(max(self.n_rows, 1) * (_lib.MC_MAXK + 1), dtype=torch.float64, device=dev)
            self.d_ncol = torch.empty(max(self.n_rows, 1), dtype=torch.int32, device=dev)
        ws = torch.empty(int(self.L.mc_rowlog_group_workspace_bytes(self.n_rows, n_loci)), dtype=torch.uint8, device=dev)
        d_cnt = torch.zeros(2, dtype=torch.int64, device=dev)
        st = C.c_void_p(torch.cuda.current_stream(dev).cuda_stream)
        _lib.check(self.L.mc_rowlog_group(p(d_log), int(n_log), self.n_feat, p(d_los), refindex.n_sites, p(d_odd_rows), p(d_odd_locus),
                                          len(odd_rows), p(d_depth), n_loci, self.n_rows, p(d_off), p(self.d_prob), p(self.d_vals),
                                          p(self.d_ncol), p(ws), p(d_cnt), st))
        self.d_off = d_off
        cnt = d_cnt.cpu().numpy()
        if cnt[1] or int(n_log) - int(cnt[0]) != self.n_rows:
            raise _lib.McallerCudaError("the row log holds %d rows of the reported loci, the histogram counted %d"
                                        % (int(n_log) - int(cnt[0]) - int(cnt[1]), self.n_rows))
        self.locus_off = d_off.cpu().numpy().view(np.uint32)
        self.text, self.offs = "", [0]
        if want_probs and self.n_rows:
            probs = self.d_prob[:self.n_rows].cpu().numpy()
            buf = np.empty(32 * self.n_rows, dtype=np.uint8)
            offs = np.empty(self.n_rows + 1, dtype=np.int64)
            total = self.L.mc_format_probs(probs.ctypes.data_as(C.c_void_p), self.n_rows, 0, buf.ctypes.data_as(C.c_void_p), len(buf),
                                           offs.ctypes.data_as(C.c_void_p))
            if total < 0:
                _lib.check(int(total))
            self.text = buf[:total].tobytes().decode("ascii")
            self.offs = offs.tolist()

    def prob_strings(self, li):
        """pos_dict_verbose[locus] (:96-97): the `.diffs` probability text of the locus's rows, file order."""
        t, o = self.text, self.offs
        return [t[o[j]:o[j + 1]] for j in range(int(self.locus_off[li]), int(self.locus_off[li + 1]))]

    def column_tests(self):
        """values_dict[locus] of :115-127 from the logged features (k columns: the trailing read quality is not logged, :91)."""
        torch, _lib = self.torch, self._lib
        if self.n_loci == 0:
            return []
        if self.d_vals is None or not (1 <= self.n_feat <= _lib.MC_MAXK):
            raise ValueError("the row log holds no feature columns")
        d_stats = torch.zeros(self.n_loci * self.n_feat * 2, dtype=torch.float64, device=self.dev)
        _lib.check(self.L.mc_colstats(C.c_void_p(self.d_vals.data_ptr()), C.c_void_p(self.d_ncol.data_ptr()), C.c_void_p(self.d_off.data_ptr()),
                                      self.n_loci, self.n_feat, C.c_void_p(d_stats.data_ptr()),
                                      C.c_void_p(torch.cuda.current_stream(self.dev).cuda_stream)))
        return ttest_finish(d_stats.cpu().numpy().reshape(self.n_loci, self.n_feat, 2), self.locus_off)


def aggregate_from_rows(refindex, depth, meth, first, d_log, n_log, n_feat, aggfi, depth_thresh, mod_thresh, pos_list=None, control=False,
                        verbose_results=False, gff=False, ref=None, odd_rows=None):
    """make_bed.py --vo and -p (also with each other and with --gff / --control / --ref, combined as aggregate_by_pos combines
    them) from the device histogram and the rows logged on the device (Engine.enable_row_log; gathered over the ranks of a
    multi-GPU run, dist.gather_row_log): d_log holds n_log entries with n_feat features each (the k feature columns,
    needed with pos_list).  No `.diffs` text is parsed."""
    entries = _locus_entries(refindex, depth, meth, first, odd_rows)
    if pos_list:
        keys = _pos_keys(make_pos_set(pos_list))
        entries = [e for e in entries if (e[0][0], e[0][1], e[0][3]) in keys]
    groups = _RowGroups(refindex, entries, d_log, n_log, n_feat, want_probs=bool(verbose_results), want_vals=bool(pos_list))
    tests = groups.column_tests() if pos_list else None
    return _write_loci([e[0] for e in entries], aggfi, depth_thresh, mod_thresh, pos_list, control, verbose_results, gff, ref, groups, tests)


def output_name(mCaller_file, positions=None, control=False, gff=False):
    """File naming of reference make_bed.py:184-194 (first '.' of the whole path, quirk Q8)."""
    stem = mCaller_file.split(".")[0]
    if positions:
        out = stem + ".methylation.positions.summary"
    elif not control:
        out = stem + ".methylation.summary"
    else:
        out = stem + ".methylation.control.summary"
    return out + (".gff" if gff else ".bed")
