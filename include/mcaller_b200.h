/*
 * mcaller_b200.h -- C ABI of libmcaller_b200.so: the B200-native (sm_100a) implementation of
 * mCaller's data-parallel hot path.
 *
 * The reference (al-mcintyre/mCaller) is pure Python and exposes no FFI; its boundary for this
 * path is the Python function extract_features() (extract_contexts.py:110) called from
 * mCaller.py:53/58/60, and aggregate_by_pos() (make_bed.py:67) called from make_bed.py:200.
 * The replacement modules mcaller_b200/extract_contexts.py and mcaller_b200/make_bed.py keep
 * those signatures and drive the entry points below through ctypes (see INTEGRATION.md for
 * the binding a maintainer would add).  Each entry point names the reference lines it
 * replaces.
 *
 * Conventions
 *   - every function returns 0 on success, a negative MC_E* code otherwise; the text of the last
 *     error of the calling thread is available from mc_last_error();
 *   - all pointers named d_* are DEVICE pointers owned by the caller (the host side allocates
 *     them as torch tensors); the library never allocates device memory and keeps no state;
 *   - every launch is asynchronous on `stream` (a cudaStream_t passed as void*); the only host
 *     synchronisation is mc_read_u64();
 *   - item counts produced by one stage and consumed by the next (records, read segments, rows) stay in device memory:
 *     consumers take a device pointer to the count (`d_n_*`) plus a host-side capacity that only sizes the launch, so a
 *     chunk runs from mc_scan to mc_hist_accumulate without a host round trip;
 *   - no torch / C++ types cross this boundary.
 */
#ifndef MCALLER_B200_H
#define MCALLER_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define MC_ABI_VERSION 3

/* text chunks: one warp tokenises MC_TILE_BYTES of TSV; the caller must keep MC_TEXT_PAD readable bytes,
 * all '\n', after the last text byte (so a final line without newline and tile look-ahead are safe). */
#define MC_TILE_BYTES 3840
#define MC_TEXT_PAD 4096
#define MC_MAXK 8            /* largest -n/--num_variables supported (reference default 6) */

enum {
    MC_OK = 0,
    MC_EINVAL = -1,      /* bad argument */
    MC_ECUDA = -2,       /* CUDA runtime error (see mc_last_error) */
    MC_ECAPACITY = -3    /* an output buffer is too small */
};

/* ---- device-resident reference index (built once per run by the host from the marked reference,
 *      replaces the per-contig meth_fwd/meth_rev strings of extract_contexts.py:154-160) --------------- */
typedef struct mc_refindex {
    int32_t n_contigs;
    int32_t k;                     /* -n */
    const uint8_t *d_names;        /* concatenated contig ids */
    const int32_t *d_name_off;     /* [n_contigs+1] offsets into d_names */
    const int64_t *d_base;         /* [n_contigs] first global coordinate of the contig (multiple of 64) */
    const int32_t *d_len;          /* [n_contigs] contig length */
    const uint32_t *d_site_fwd;    /* bit g: forward-strand copy holds 'M' at global coordinate g */
    const uint32_t *d_site_rev;    /* same for the reverse-strand copy (forward coordinates) */
    const uint32_t *d_cand;        /* bit g: some 'M' (either strand) inside [g, g+k) */
    const uint32_t *d_rank_fwd;    /* per 32-bit word: number of forward sites before the word */
    const uint32_t *d_rank_rev;    /* same for reverse sites, offset by the total number of forward sites */
    const uint8_t *d_bases;        /* reference letters at global coordinates (upper case) */
    int64_t total_bits;            /* size of the global coordinate space (multiple of 64) */
} mc_refindex;

/* ---- stage 1 output: one record per TSV line that can open, feed or close a window ------------------- */
typedef struct mc_record {
    uint32_t line_lo;      /* byte offset of the line inside the chunk, low 32 bits */
    uint16_t line_hi;      /* high 16 bits */
    uint16_t name_off;     /* offset of the read-name field (column 4) from the line start */
    int32_t pos;           /* column 2, reference position */
    int32_t event_idx;     /* column 6 */
    double diff;           /* np.round(float(col7) - float(col11), 4), extract_contexts.py:286 */
    uint16_t name_len;
    uint16_t contig;       /* contig index */
    uint8_t flags;         /* MC_RF_* */
    uint8_t kbits_fwd;     /* bit c: the forward-strand marked copy holds 'M' at pos + c, c < k (meth_fwd[pos:pos+k], :176) */
    uint8_t kbits_rev;     /* same for the reverse-strand copy */
    uint8_t pad;
} mc_record;               /* 32 bytes */

#define MC_RF_EQ 1u        /* reference_kmer (col 3) == model_kmer (col 10) */
#define MC_RF_CAND 2u      /* k-mer window touches a target on either strand */
#define MC_RF_BADNUM 4u    /* event/model mean not a plain decimal (<= 18 digits) */
#define MC_RF_BADIDX 8u    /* event index not a plain integer */
#define MC_RF_RAW 16u      /* stage-1 form: event_idx / diff / name span are not filled in yet; mc_order_records does and clears the flag */
#define MC_RF_NEWREAD 32u  /* read name differs from the previous record's (valid when MC_RF_SEGKNOWN is set) */
#define MC_RF_SEGKNOWN 64u /* mc_order_records compared the read name with the previous record's */

/* counters written by mc_scan (uint64 each) */
enum {
    MC_C_LINES = 0,        /* lines owned by the scanned range */
    MC_C_KEPT,             /* >= 12 fields, known contig, model_kmer != NNNNNN (see mc_scan for the sparse mode) */
    MC_C_RECORDS,          /* record slots reserved (allocation cursor, >= records written) */
    MC_C_SHORT,            /* lines with < 12 whitespace separated fields (:149-152) */
    MC_C_UNKNOWN_CONTIG,   /* contig not in the reference (:154-160) */
    MC_C_NNN,              /* model_kmer == 'NNNNNN' (:167) */
    MC_C_BADPOS,           /* column 2 not a non-negative integer on a known contig (reference: ValueError) */
    MC_C_LONGLINE,         /* lines whose first 12 columns outran the look-ahead and took the byte-wise slow path (informational) */
    MC_C_OVERFLOW,         /* records dropped because rec_cap was too small */
    MC_C_RUN_CURSOR,       /* internal: next unclaimed run of chunks (dynamic work distribution of mc_scan) */
    MC_C_QUIET,            /* chunks (MC_TILE_BYTES each) passed over after the look at their first columns (informational) */
    MC_C_COUNT = 16
};

/* ---- stage 5 output: one row per closed window ----------------------------------------------------- */
typedef struct mc_call {
    int64_t read_off;      /* read name: byte offset inside the chunk ... */
    double prob;           /* P(methylated), filled by mc_classify */
    double feat[MC_MAXK + 1];   /* k column means in output order (5'->3' on the read strand) + read quality */
    int32_t read_len;      /* ... and length */
    int32_t mpos;          /* target position (column 3 of the .diffs row) */
    int32_t site;          /* dense site slot (forward sites first, then reverse) for the histogram */
    uint32_t close_rec;    /* ordered index of the record that closed the window; 0xFFFFFFFF = still open at the end of the chunk */
    uint16_t win_contig;   /* contig of the window (context is cut from its marked copy, :194) */
    uint16_t chrom_contig; /* contig of the closing line (column 1, :216); 0xFFFF while pending */
    uint8_t kind;          /* MC_CALL / MC_TOO_MANY_SKIPS / MC_MULTI_M */
    uint8_t rev;           /* strand: 1 = '-' */
    uint8_t n_empty;       /* empty columns (skips) */
    uint8_t empty_mask;    /* bit c: output feature c is an empty column (printed as integer 0) */
    uint8_t model_sel;     /* 0 = 'MH' / 'general', 1 = 'MG' (base_models, :99-106) */
    uint8_t label;         /* prob >= 0.5 */
    uint8_t err;           /* MC_CE_* */
    uint8_t pad0;
    uint32_t seg;          /* read segment index inside the chunk */
    uint32_t pad1;
    uint32_t pad2;
} mc_call;                 /* 128 bytes */

enum { MC_CALL = 0, MC_TOO_MANY_SKIPS = 1, MC_MULTI_M = 2, MC_NONE = 3 /* empty slot: every consumer skips it */ };
#define MC_CE_CONTEXT 1u   /* window within k of a contig end (reference: IndexError / sys.exit, :195, :224) */
#define MC_CE_MODELKEY 2u  /* base after the target not in ACGTM (reference: KeyError -> sys.exit, :218-223) */
#define MC_CE_BADNUM 4u    /* a fed line had an unsupported numeric field */
#define MC_CE_COLUMN 8u    /* a column holds 65535 or more events: its count saturated, the mean is not computed */
#define MC_CE_SPACING 16u  /* multi-M shift of 0 (reference: 'n diffs off' -> sys.exit, :257-266) */

/* ---- classifier (host struct holding device pointers; layout mirrors sklearn's fitted attributes) ---- */
enum { MC_MLP = 0, MC_LR = 1, MC_GNB = 2, MC_RF = 3 };
enum { MC_ACT_IDENTITY = 0, MC_ACT_LOGISTIC = 1, MC_ACT_TANH = 2, MC_ACT_RELU = 3 };
typedef struct mc_model {
    int32_t kind;
    int32_t n_in;
    int32_t n_layers;          /* MLP: number of weight matrices */
    int32_t hidden_act;
    int32_t sizes[8];          /* MLP: layer widths, sizes[0] = n_in ... sizes[n_layers] = 1 */
    const double *d_weights;   /* MLP: coefs_ concatenated (row-major [in][out]); LR: coef_; GNB: theta_[2][n] then var_[2][n] */
    const double *d_biases;    /* MLP: intercepts_ concatenated; LR: intercept_; GNB: log class_prior_[2] */
    int32_t n_trees;           /* RF */
    int32_t max_nodes;         /* RF: largest tree (for shared-memory staging) */
    const int32_t *d_tree_off; /* [n_trees+1] */
    const int32_t *d_left;     /* child index inside the tree, -1 = leaf */
    const int32_t *d_right;
    const int32_t *d_feature;
    const double *d_threshold;
    const double *d_leaf_p1;   /* class-1 fraction of the node's value */
} mc_model;

/* read-quality table entry (open addressing, power-of-two size, key = FNV-1a of the read-name prefix) */
typedef struct mc_qual_entry {
    uint64_t hash;             /* 0 = empty slot */
    uint32_t check;            /* second hash (different basis), guards against 64-bit collisions */
    uint32_t len;              /* prefix length */
    double qual;               /* mean phred (read_qual.py:13) */
} mc_qual_entry;

/* ---------------------------------------------------------------------------------------------------- */

int mc_version(void);
/* sizeof of the ABI structs: 0 mc_record, 1 mc_call, 2 mc_refindex, 3 mc_model, 4 mc_qual_entry, 5 mc_synth_spec, 6 mc_locus_entry,
 * 7 mc_diffs_row, 8 mc_carry */
int mc_sizeof(int what);
const char *mc_last_error(void);

/* copy n uint64 from device to host and synchronise the stream */
int mc_read_u64(const uint64_t *d_src, int64_t n, uint64_t *h_dst, void *stream);

/*
 * Stage 1 -- tokenise + filter.  Replaces the reader/tokeniser and the per-line filters of
 * extract_contexts.py:140-176 (readlines, line.split()[:12], contig lookup, NNNNNN filter, k-mer
 * 'has M' test).  One warp per MC_TILE_BYTES chunk; a line belongs to the chunk holding its first byte.
 * Emits a record for every kept line that is a candidate (k-mer window touches a target on either
 * strand), that follows a candidate, or that is the first kept line of a run of chunks; with dense == 1 for
 * every kept line; with dense == 2 ("read-first", the mode for -q) additionally for the first kept line of every read
 * (maximal block of lines with the same read name), so that whole reads can be dropped by quality later and a window left
 * open at the end of a read still finds its closer: the first kept line of the next read that passes
 * (extract_contexts.py:167 runs before :179).  Records of one chunk are contiguous and in line order; warps reserve slots in
 * blocks from d_counters[MC_C_RECORDS] (so that counter is an upper bound of the record count and the buffer has
 * holes); d_tile_tab[chunk] = {first record slot, count | flags} and d_run_tab[run] = {records of the run, flags} are consumed
 * by mc_order_records, which also drops the run-first records whose predecessor line turns out not to be a candidate.
 * Records leave this stage raw (MC_RF_RAW): line offset, position, contig, candidate flag and -- parked in the fields that are
 * still empty -- the first 128 field-start bits of the line; mc_order_records finishes them at full lane occupancy.
 * With dense != 1, groups of lines that all sit on non-candidate positions of the current contig (and, with dense == 2,
 * all carry the read name of the line before them) are passed over after
 * a look at their first two columns, so MC_C_KEPT / MC_C_SHORT / MC_C_NNN / MC_C_BADPOS count only the lines that were
 * parsed in full: MC_C_KEPT is exact with dense == 1 and otherwise > 0 exactly when the range holds a kept line.
 * d_counters (MC_C_COUNT uint64) must be zeroed by the caller; d_text must be 16-byte and d_tile_tab 8-byte aligned.
 */
int mc_scan(const uint8_t *d_text, int64_t nbytes, const mc_refindex *ref, int dense,
            mc_record *d_rec, int64_t rec_cap, uint32_t *d_tile_tab /* [2*n_tiles] */, uint32_t *d_run_tab /* [2*n_runs] */,
            uint64_t *d_counters, void *stream);

/* Chunks per run mc_scan uses for nbytes of text on the current device (consecutive chunks parsed by one warp); the run
 * table holds ceil(mc_num_tiles(nbytes) / run length) entries of two uint32: {records of the run, flags}.  mc_order_records
 * must be given the same run length. */
int mc_scan_run_len(int64_t nbytes);

/* Test / tuning hook: chunks per run of mc_scan (consecutive chunks parsed by one warp, which carries the
 * "last kept line" state between them).  0 = automatic (32, shortened for small inputs so every warp gets runs to
 * balance on).  Results do not depend on it.  Returns the previous setting. */
int mc_scan_set_run_len(int run_len);

/* number of tiles mc_scan uses for nbytes */
int64_t mc_num_tiles(int64_t nbytes);

/* bytes of scratch needed by the scan-based stages below for up to n items */
int64_t mc_workspace_bytes(int64_t n);

/* Stage 2 -- put the records into file order (exclusive scan of the run table, then one warp per run gathers its chunks).  d_rec_in is the stage-1
 * buffer (rec_in_cap = its capacity; slots are reserved in blocks, so it has holes); d_n_out[0] receives the number of
 * records, which land densely in d_rec_out (rec_out_cap slots; rec_in_cap is always enough).  Records arrive in raw form
 * (MC_RF_RAW) and are finished here, one thread per record: event index, the float64 np.round(event_mean - model_mean, 4)
 * from exact decimal parsing, the k-mer equality flag (extract_contexts.py:150, :169, :286), the read-name span and the
 * target bits of the k-mer on both strands (kbits_fwd / kbits_rev, from `ref`); read-name changes between neighbouring
 * records of a run are flagged (MC_RF_SEGKNOWN / MC_RF_NEWREAD), the first record of a run is left to mc_segment_reads.
 * d_seg_flags / d_run_first (optional, together): the read-change flag of every ordered record as 0 / 1 (placeholder 1 for the
 * first record of a run) and, per run, the ordered index of its first record (0xFFFFFFFF: none) -- with them
 * mc_segment_reads only has to look at one record per run.  d_scan_counters: the counter block mc_scan wrote
 * (may be NULL); when it shows that stage 1 ran out of record slots nothing is ordered and d_n_out[0] = 0, so every later
 * stage of the chunk is a no-op until the caller has grown the buffer and scanned again. */
int mc_order_records(const uint8_t *d_text, int64_t nbytes, const mc_refindex *ref, const uint32_t *d_tile_tab, int64_t n_tiles,
                     uint32_t *d_run_tab, int run_len, const mc_record *d_rec_in, int64_t rec_in_cap, const uint64_t *d_scan_counters,
                     mc_record *d_rec_out, int64_t rec_out_cap, uint64_t *d_n_out, uint32_t *d_seg_flags /* [rec_out_cap] or NULL */,
                     uint32_t *d_run_first /* [n_runs] or NULL */, void *d_ws, void *stream);

/*
 * Stage 3 -- read segmentation: a new segment starts where the read name (column 4) differs from the
 * previous record's (extract_contexts.py:161, `read_name != last_read`).  Writes the first record index of
 * each segment to d_seg_start (capacity rec_cap+1, terminated by the record count) and the segment count to
 * d_nseg[0].  d_n_records[0] (device) is the record count written by mc_order_records; rec_cap >= it sizes the launch.
 * Records whose flags do not yet say whether a new read starts there (MC_RF_SEGKNOWN clear) are compared with their
 * predecessor in the text and get MC_RF_SEGKNOWN / MC_RF_NEWREAD written back.
 */
int mc_segment_reads(const uint8_t *d_text, mc_record *d_rec, const uint64_t *d_n_records, int64_t rec_cap,
                     uint32_t *d_seg_flags /* from mc_order_records, or NULL */, const uint32_t *d_run_first, int64_t n_runs,
                     uint32_t *d_seg_start, uint64_t *d_nseg, void *d_ws, void *stream);

/*
 * Stage 4 -- read quality per segment: read2qual[name] else read2qual[name.split(':')[0].split('_')[0]]
 * (extract_contexts.py:163-166, read_qual.py:6-19).  Missing reads get NaN and are counted in d_err[0]
 * (the reference raises KeyError).  d_nseg[0] (device) segments, seg_cap >= it.
 */
int mc_segment_quality(const uint8_t *d_text, const mc_record *d_rec, const uint32_t *d_seg_start, const uint64_t *d_nseg,
                       int64_t seg_cap, const mc_qual_entry *d_table, int64_t table_size, double *d_seg_qual, uint64_t *d_err,
                       void *stream);

/*
 * Stage 5 -- window builder: the state machine of extract_contexts.py:169-291 (strand inference, window
 * open/feed/close, skip filter, multi-M carry, orientation flip, np.mean of np.round(ev-model,4) per column in
 * numpy's summation order, any number of events per column).  A read is cut into units at its non-candidate records
 * (after which the reference's state is closed and empty); one thread per unit, two passes (count, exclusive scan,
 * write) so rows come out in file order.  d_rec must come from mc_order_records (MC_RF_SEGKNOWN / MC_RF_NEWREAD set)
 * and d_seg_start from mc_segment_reads on the same records.  d_seg_count is scratch of seg_cap uint32.  d_ncalls[0]
 * receives the number of rows (all kinds).  Segments whose quality is below qual_thresh are skipped entirely (:167).
 * d_ws: mc_workspace_bytes(rec_cap).  d_spill (spill_cap doubles) holds the values of columns with more than 128 events
 * while numpy's recursive halving is replayed on them (a stalled read).  d_ncalls[1] is 0 when every buffer sufficed;
 * otherwise bit 0 says rows beyond call_cap were dropped and bits 1-63 hold the doubles the spill arena would have needed
 * when that is more than spill_cap (the rows of such columns are then wrong).  Either way the rows must be discarded and
 * the chunk built again with larger buffers (mc_chunk_guard aborts on a nonzero d_ncalls[1]).
 */
int mc_build_windows(const mc_record *d_rec, const uint64_t *d_n_records, int64_t rec_cap, const uint32_t *d_seg_start,
                     const uint64_t *d_nseg, int64_t seg_cap, const double *d_seg_qual, const mc_refindex *ref, int skip_thresh,
                     double qual_thresh, int two_models, mc_call *d_calls, int64_t call_cap, uint32_t *d_seg_count,
                     uint64_t *d_ncalls, void *d_ws, double *d_spill, int64_t spill_cap, void *stream);

/*
 * Chunk / rank edges.  The reference closes a window when it reads the NEXT kept line (extract_contexts.py:179), so the
 * window still open at the end of a chunk of text belongs to the rows of the following chunk, and the one open at the
 * end of a worker's byte range is closed by the first kept line of the next range (mCaller.py:63-68); only the last
 * window of the file is dropped (SURVEY.md Q3).  mc_carry is the device-resident state that carries that one row.
 *
 * mc_carry_rows: d_rows[0] is a slot reserved by the caller in front of the rows mc_build_windows wrote at d_rows + 1
 *   (d_ncalls[0] of them).  If the carry holds a row and this chunk has a kept line (first record of the first read
 *   segment that passes the quality filter), the carried row is completed -- chrom_contig = contig of that line (:216),
 *   close_rec = its record index, read_off = -1 (the read name lies in the previous chunk's text; the host keeps it) --
 *   and placed in d_rows[0]; otherwise d_rows[0].kind = MC_NONE.  A row of this chunk that is still pending
 *   (close_rec == 0xFFFFFFFF, always the last row) becomes the new carry.  d_nrows_out[0] = d_ncalls[0] + 1: the rows
 *   d_rows[0 .. ] that the classifier, histogram, statistics and the writer consume.  The first kept contig seen since
 *   mc_carry_reset is remembered in the carry (what the previous rank needs to close ITS last window).  d_abort (may be
 *   NULL): see mc_chunk_guard.
 * mc_carry_close: end of a byte range.  closing_contig >= 0: contig of the first kept line after the range (found by the
 *   host, or -1 with d_next_contigs: first_kept_contig of the following ranks, all-gathered; the first entry >= 0 among
 *   [from, count) closes).  The completed row goes to d_row_out (kind MC_NONE when there is nothing to close or nobody
 *   closes it = end of file) and, when it is a call with prob/label already set by mc_classify, into the histogram
 *   (d_depth may be NULL: no histogram) with first-seen index d_row_base[0] -- the device-side row counter
 *   mc_hist_accumulate advances, i.e. after every row of the range -- which is then advanced by one.
 */
typedef struct mc_carry {
    mc_call row;                   /* the open window (valid != 0) */
    uint32_t valid;
    int32_t first_kept_contig;     /* contig of the first kept line seen since mc_carry_reset, -1 = none yet */
    uint64_t chunks;               /* chunks seen since the reset (informational) */
    uint64_t pad[6];
} mc_carry;                        /* 192 bytes */
int mc_carry_reset(mc_carry *d_carry, void *stream);
int mc_carry_rows(mc_call *d_rows, const uint64_t *d_ncalls, const mc_record *d_rec, const uint64_t *d_n_records,
                  const uint32_t *d_seg_start, const uint64_t *d_nseg, const double *d_seg_qual, double qual_thresh,
                  mc_carry *d_carry, uint64_t *d_nrows_out, const uint64_t *d_abort, void *stream);
/* Overflow guard of a chunk: d_abort[0] = 1 when a buffer of the stages so far was too small (mc_scan's overflow counter, reserved
 * record slots > rec_cap, ordered records > rec_out_cap, read segments > seg_cap, rows > call_cap), else 0.  The stages that change state across chunks
 * (mc_carry_rows, mc_hist_accumulate) take d_abort and do nothing when it is set, so the host can grow its buffers and run the
 * chunk again without having synchronised in between. */
int mc_chunk_guard(const uint64_t *d_counters, int64_t rec_cap, const uint64_t *d_n_records, int64_t rec_out_cap,
                   const uint64_t *d_nseg, int64_t seg_cap, const uint64_t *d_ncalls, int64_t call_cap, uint64_t *d_abort,
                   uint64_t *d_sticky /* may be NULL: set to 1 on overflow, never cleared here */, void *stream);
int mc_carry_close(mc_carry *d_carry, int closing_contig, const int64_t *d_next_contigs, int from, int count, mc_call *d_row_out,
                   uint32_t *d_depth, uint32_t *d_meth, uint64_t *d_first, int64_t n_sites, uint64_t *d_row_base, void *stream);

/*
 * Stage 6 -- classifier: model[key].predict_proba([x])[0][1] and the 0.5 label threshold
 * (extract_contexts.py:195-207) for every MC_CALL row; float64 arithmetic.  models[0] = 'MH'/'general',
 * models[1] = 'MG' (used for rows with model_sel == 1; pass models[0] again when there is one model).  Both must be of one
 * kind and take one input width, and each is validated on the host before any launch (MC_EINVAL otherwise).
 * d_nrows[0] (device) rows, row_cap >= it.  d_ws: scratch of
 * mc_classify_workspace_bytes(row_cap) bytes (index list of the call rows, so the kernels run with every lane busy).
 */
int64_t mc_classify_workspace_bytes(int64_t row_cap);
int mc_classify(mc_call *d_calls, const uint64_t *d_nrows, int64_t row_cap, const mc_model *models, void *d_ws, void *stream);

/*
 * Stage 7 -- per-position aggregation (make_bed.py:86-96): depth and methylated counts per site slot, plus the
 * smallest global row index that touched the slot (first-seen order of make_bed.py:134).  d_depth/d_meth are
 * uint32[n_sites], d_first uint64[n_sites] (initialise to ~0); d_row_base[0] (device) is added to the row index and then
 * advanced by the number of rows, so consecutive chunks keep file order.  Rows whose closing contig differs from the
 * window contig (reference quirk, :216: column 1 of the row names another contig than the site's) cannot be keyed by
 * site slot: they are appended to d_odd (capacity odd_cap rows, count in d_n_odd[0], the row's pad1/pad2 receive the
 * low / high half of its global row index) for the host to merge.  Pending rows and MC_NONE slots are skipped.
 */
int mc_hist_accumulate(const mc_call *d_calls, const uint64_t *d_nrows, int64_t row_cap, uint32_t *d_depth, uint32_t *d_meth,
                       uint64_t *d_first, int64_t n_sites, uint64_t *d_row_base, mc_call *d_odd, int64_t odd_cap, uint64_t *d_n_odd,
                       const uint64_t *d_abort /* may be NULL */, void *stream);

/* Thresholds of the summary (check_thresh, make_bed.py:21-28) on the device histogram: d_flags[s] = 1 for the site slots
 * that make_bed.py -d depth_thresh -t mod_thresh [--control] reports (depth >= depth_thresh and float64 meth / depth >= mod_thresh,
 * or < with control), d_count[0] = how many.  The host formats only those (mcaller_b200.make_bed.aggregate_from_histogram). */
int mc_bed_select(const uint32_t *d_depth, const uint32_t *d_meth, int64_t n_sites, int64_t depth_thresh, double mod_thresh,
                  int control, uint8_t *d_flags, uint64_t *d_count, void *stream);

/* Row statistics on the device (adds to d_out[7], which the caller zeroes): calls closed in the chunk, calls still
 * pending, too-many-skips events closed in the chunk, multi-M events, rows with an error flag, calls labelled
 * methylated, too-many-skips events still pending (counted by the reference only once a later kept line closes them). */
int mc_count_calls(const mc_call *d_calls, const uint64_t *d_nrows, int64_t row_cap, uint64_t *d_out, void *stream);

/*
 * make_bed drop-in: aggregate a `.diffs.<k>` text file (make_bed.py:75-98, default mode).  d_table is an open-addressing
 * table (power-of-two entries; hash == 0 means empty, first_off must be initialised to ~0) keyed by the FNV-1a hash of
 * "chrom\tpos\tcontext\tstrand"; first_off is the smallest byte offset of a row with that key (first-seen order, :134).
 * d_counters[8] (see mc_diffs_aggregate_ex): rows, malformed rows (field count not 7/8), rows skipped by the centre-'M'
 * test (:84), table-full drops, ...
 */
typedef struct mc_locus_entry {
    unsigned long long hash;
    unsigned long long first_off;
    unsigned long long check;   /* independent second hash of the locus key (0 = not set): two loci with one `hash` are counted in d_counters[7] */
    uint32_t depth;
    uint32_t meth;
} mc_locus_entry;

/*
 * make_bed variants that need per-read lists (make_bed.py -p and --vo; SURVEY.md section 8f rank 3).
 *
 * mc_diffs_aggregate_ex: the aggregation above with the `-p` filter of make_bed.py:73-74/:84 and a base offset, so a file can be
 *   streamed in line-aligned pieces into one table (first_off = base_off + offset inside the piece) -- d_posset (may be NULL) is an
 *   open-addressing set (power-of-two entries, 0 = empty) of FNV-1a hashes of "chrom\tpos\tstrand" built by the host from
 *   the positions file (entries whose end column is not start + 1 can never match and are left out).
 *   d_counters[8]: rows, malformed, centre-not-'M', table-full drops, rows outside the positions set, old-format rows,
 *   [6] see mc_diffs_colstats, [7] rows whose 64-bit locus key matched a slot holding another locus (check hash differs)
 *   (7 fields), value tokens float() would not parse, value tokens outside the exactly-rounded range.
 * mc_diffs_rows: second pass; one mc_diffs_row per used row in arbitrary order (sort by line_off for file order):
 *   the locus slot in d_table, and the spans of the values (column 5) and stripped probability (column 8) fields.
 * mc_diffs_colstats: the one-sample t-test inputs of make_bed.py:115-127 (scipy.stats.ttest_1samp, popmean 0).  d_order
 *   lists the row indices grouped by locus in file order, d_locus_off[n_loci + 1] is the CSR over that order.  Values are
 *   parsed like `[float(v) for v in values.split(',')][:-1]` (exactly rounded) into d_vals[n_rows][MC_MAXK + 1] /
 *   d_ncol[n_rows]; d_stats[n_loci][ncols][2] receives np.mean(x) and np.add.reduce((x - mean)**2) in numpy's pairwise
 *   summation order, so t = mean / sqrt(ss / n * (n / (n - 1)) / n) is bit-identical to scipy's.
 */
typedef struct mc_diffs_row {
    uint64_t line_off;         /* byte offset of the row in the file */
    uint32_t slot;             /* index of its locus in d_table */
    uint32_t values_off;       /* column 5 (comma-joined features), relative to line_off */
    uint32_t values_len;
    uint32_t prob_off;         /* column 8 without surrounding whitespace; length 0 for old-format rows */
    uint32_t prob_len;
    uint32_t pad;
} mc_diffs_row;                /* 32 bytes */
int mc_diffs_aggregate_ex(const uint8_t *d_text, int64_t nbytes, int64_t base_off, const uint64_t *d_posset, int64_t posset_size,
                          mc_locus_entry *d_table, int64_t table_size, uint64_t *d_counters, void *stream);
/* moves the used entries of d_old into the (initialised, larger) table d_table; table-full drops are counted in d_counters[3] */
int mc_diffs_rehash(const mc_locus_entry *d_old, int64_t old_size, mc_locus_entry *d_table, int64_t table_size,
                    uint64_t *d_counters, void *stream);
int mc_diffs_rows(const uint8_t *d_text, int64_t nbytes, const uint64_t *d_posset, int64_t posset_size,
                  const mc_locus_entry *d_table, int64_t table_size, mc_diffs_row *d_rows, int64_t row_cap, uint64_t *d_nrows,
                  void *stream);
int mc_diffs_colstats(const uint8_t *d_text, const mc_diffs_row *d_rows, const uint32_t *d_order, int64_t n_rows,
                      const uint32_t *d_locus_off, int64_t n_loci, int ncols, double *d_vals, uint32_t *d_ncol,
                      double *d_stats, uint64_t *d_counters, void *stream);

/*
 * Host-side writer (no device work): renders the MC_CALL rows of a chunk (host copy of the mc_call array; rows still
 * pending are skipped) as `.diffs.<k>` text exactly like the reference (extract_contexts.py:216, :83-86): chrom, read,
 * position, 2k-1 context cut from the marked reference copies, comma-joined features (shortest round-trip repr, integer 0
 * for empty columns) + read quality, strand, and -- with_prob -- label and np.round(prob, 2).  h_text is the host copy
 * of the chunk (read names); a row with read_off < 0 (a window carried over from the previous chunk, mc_carry_rows) takes
 * its read name from carry_name[0 .. carry_name_len).  Returns the number of bytes written, MC_ECAPACITY when out_cap is
 * too small, -100 - err when a row carries MC_CE_* error flags, or MC_EINVAL when a context covers a reference letter
 * outside ACGTNM (the reference raises KeyError in revcomp, extract_contexts.py:11-15).  max_threads <= 0: one host
 * thread per hardware thread.
 */
int64_t mc_format_rows(const mc_call *h_calls, int64_t n_calls, const uint8_t *h_text, const uint8_t *carry_name,
                       int32_t carry_name_len, const char *const *contig_names, const char *const *marked_fwd,
                       const char *const *marked_rev, const int64_t *contig_len, int32_t n_contigs, int32_t k,
                       const char *base_label, const char *mod_label, int32_t with_prob, int32_t max_threads, char *out,
                       int64_t out_cap);

/*
 * FASTQ read-quality ingest (reference read_qual.py:6-19) on the device.  mc_fastq_index builds the byte offset of every
 * line start (d_line_start[0] = 0, capacity line_cap; *d_n_newlines = number of '\n' in the buffer; d_tile_cnt/d_tile_off
 * hold mc_fastq_tiles(nbytes) uint32 each, d_ws >= mc_workspace_bytes(tiles)).  The buffer must be readable up to the next
 * multiple of 16 bytes.  mc_fastq_quality then treats lines 4r..4r+3 as record r (d_line_start[n_lines] must hold the offset
 * one past the newline that ends the last line -- nbytes + 1 when the file has no final newline) and inserts
 * {id.split(':')[0].split('_')[0] -> mean(ord(c) - 33 over the quality line)} into the open-addressing table probed by
 * mc_segment_quality (d_owner: uint32[table_size], zeroed; d_rec_mean: double[n_lines/4] scratch; the last record with a
 * given key wins, like the reference's dict).  d_stats[3]: records inserted, records whose header does not start with '@', inserts dropped (table full).
 */
int64_t mc_fastq_tiles(int64_t nbytes);
int mc_fastq_index(const uint8_t *d_text, int64_t nbytes, uint32_t *d_tile_cnt, uint32_t *d_tile_off, uint64_t *d_line_start,
                   int64_t line_cap, uint64_t *d_n_newlines, void *d_ws, void *stream);
int mc_fastq_quality(const uint8_t *d_text, int64_t nbytes, const uint64_t *d_line_start, int64_t n_lines, mc_qual_entry *d_table,
                     int64_t table_size, uint32_t *d_owner, double *d_rec_mean, uint64_t *d_stats, void *stream);

/*
 * MLP training (mCaller --train -c NN): scikit-learn 1.9 MLPClassifier(hidden_layer_sizes=MC_TRAIN_HIDDEN,
 * activation='tanh', solver='adam', batch_size='auto', shuffle=True).fit on a binary target, float64, one CTA per job.
 * The caller draws the initial parameters and every epoch's sample order from numpy's RandomState(seed) as scikit-learn
 * does, writes the parameters to d_w (W0 [d][100] row-major, W1 [100], c0 [100], c1 [1]; n_params = 102 d + 101) and the
 * job array to device memory, and calls mc_mlp_train_init once (Adam moments zeroed, state reset).  Each
 * mc_mlp_train_epochs call then runs up to `epochs` epochs of every job not yet stopped: epoch e of job j visits the rows
 * d_idx[idx_off + e*n .. + n) (indices into d_x / d_y) in batches of min(MC_TRAIN_BATCH, n), the last one possibly short.
 * After an epoch the kernel appends the epoch loss to d_loss_curve and applies the no-improvement rule (loss > best - tol
 * counts; stop when the count exceeds n_iter_no_change, stopped = 1) and the iteration limit (stopped = 2).  The state
 * stays in d_w and the job array between calls, so the caller can draw the next epochs' orders while a call runs, and
 * read `stopped` back after it.  Requirements: 1 <= d <= MC_MAXK + 1, n >= 1; d_idx entries index valid rows for every
 * epoch of the call (also the epochs of a job that stops early).
 */
#define MC_TRAIN_HIDDEN 100
#define MC_TRAIN_BATCH 200
typedef struct mc_train_job {
    const double *d_x;           /* [rows][d] features, row-major */
    const double *d_y;           /* [rows] target, 0.0 or 1.0 */
    double *d_w;                 /* [3][n_params]: parameters (in: initial, out: fitted), Adam m, Adam v */
    double *d_loss_curve;        /* [max_iter] epoch losses (scikit-learn's loss_curve_) */
    int64_t idx_off;             /* this job's [epochs][n] sample orders in the d_idx of each call */
    int32_t n, d;                /* training rows, features */
    int32_t max_iter, n_iter_no_change;
    double alpha, lr, tol;
    /* kept by the kernels */
    double best_loss;
    int32_t n_iter, no_improve, stopped, pad;
} mc_train_job;                  /* 104 bytes */

int mc_mlp_train_init(mc_train_job *d_jobs, int32_t n_jobs, void *stream);
int mc_mlp_train_epochs(mc_train_job *d_jobs, int32_t n_jobs, const int32_t *d_idx, int32_t epochs, void *stream);

/* ---- synthetic eventalign generator (bench / test tooling; bit-identical to mcaller_b200/synth.py) ---- */
typedef struct mc_synth_spec {
    uint64_t seed;
    int32_t n_contigs;
    int32_t len_min, len_max, p_skip, p_nnn, margin;
    int32_t meth;                  /* add METH_OFFSETS at methylated sites */
    const uint8_t *d_names;        /* contig ids, concatenated */
    const int32_t *d_name_off;     /* [n_contigs+1] */
    const int32_t *d_contig_len;   /* [n_contigs] */
    const int64_t *d_read_bounds;  /* [n_contigs+1] read index ranges per contig */
    const int64_t *d_gbase;        /* [n_contigs] global coordinate base (as in mc_refindex) */
    const uint8_t *d_genome;       /* letters at global coordinates */
    const uint32_t *d_meth_fwd;    /* methylated-site bitmaps (global coordinates), may be NULL when !meth */
    const uint32_t *d_meth_rev;
    const int32_t *d_model_mean;   /* [4096] centi-pA */
    const int32_t *d_model_sd;     /* [4096] */
} mc_synth_spec;

/* genome letters for all contigs (global coordinates) */
int mc_synth_genome(const mc_synth_spec *spec, uint8_t *d_genome_out, int64_t total_bits, void *stream);
/* pass 1: bytes of TSV text of reads [read0, read0+n) -> d_sizes[n] */
int mc_synth_sizes(const mc_synth_spec *spec, int64_t read0, int64_t n, int64_t n_total_reads, uint64_t *d_sizes, void *stream);
/* pass 2: write the text of each read at d_offsets[i] (exclusive scan of the sizes) */
int mc_synth_write(const mc_synth_spec *spec, int64_t read0, int64_t n, int64_t n_total_reads, const uint64_t *d_offsets,
                   uint8_t *d_text, void *stream);

#ifdef __cplusplus
}
#endif
#endif
