"""ctypes binding of libmcaller_b200.so (C ABI in include/mcaller_b200.h).

There is no CPU fallback: importing this module's `lib()` without the built library, or calling
into it without a CUDA device, raises.
"""
import ctypes as C
import os

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("MCALLER_B200_LIB") or os.path.join(HERE, "libmcaller_b200.so")      # the env var selects a tuning build

MC_TILE_BYTES = 3840
MC_TEXT_PAD = 4096
MC_MAXK = 8
MC_C_COUNT = 16
COUNTER_NAMES = ["lines", "kept", "records", "short", "unknown_contig", "nnn", "badpos", "longline", "overflow", "run_cursor", "quiet_chunks"]

MC_ABI_VERSION = 3
MC_CALL, MC_TOO_MANY_SKIPS, MC_MULTI_M, MC_NONE = 0, 1, 2, 3
MC_CE_CONTEXT, MC_CE_MODELKEY, MC_CE_BADNUM, MC_CE_COLUMN, MC_CE_SPACING = 1, 2, 4, 8, 16
MC_MLP, MC_LR, MC_GNB, MC_RF = 0, 1, 2, 3
PENDING = 0xFFFFFFFF


class RefIndex(C.Structure):
    _fields_ = [("n_contigs", C.c_int32), ("k", C.c_int32), ("d_names", C.c_void_p), ("d_name_off", C.c_void_p),
                ("d_base", C.c_void_p), ("d_len", C.c_void_p), ("d_site_fwd", C.c_void_p), ("d_site_rev", C.c_void_p),
                ("d_cand", C.c_void_p), ("d_rank_fwd", C.c_void_p), ("d_rank_rev", C.c_void_p), ("d_bases", C.c_void_p),
                ("total_bits", C.c_int64)]


class Model(C.Structure):
    _fields_ = [("kind", C.c_int32), ("n_in", C.c_int32), ("n_layers", C.c_int32), ("hidden_act", C.c_int32),
                ("sizes", C.c_int32 * 8), ("d_weights", C.c_void_p), ("d_biases", C.c_void_p), ("n_trees", C.c_int32),
                ("max_nodes", C.c_int32), ("d_tree_off", C.c_void_p), ("d_left", C.c_void_p), ("d_right", C.c_void_p),
                ("d_feature", C.c_void_p), ("d_threshold", C.c_void_p), ("d_leaf_p1", C.c_void_p)]


class SynthSpec(C.Structure):
    _fields_ = [("seed", C.c_uint64), ("n_contigs", C.c_int32), ("len_min", C.c_int32), ("len_max", C.c_int32),
                ("p_skip", C.c_int32), ("p_nnn", C.c_int32), ("margin", C.c_int32), ("meth", C.c_int32),
                ("d_names", C.c_void_p), ("d_name_off", C.c_void_p), ("d_contig_len", C.c_void_p),
                ("d_read_bounds", C.c_void_p), ("d_gbase", C.c_void_p), ("d_genome", C.c_void_p),
                ("d_meth_fwd", C.c_void_p), ("d_meth_rev", C.c_void_p), ("d_model_mean", C.c_void_p),
                ("d_model_sd", C.c_void_p)]


RECORD_DTYPE = np.dtype([("line_lo", "<u4"), ("line_hi", "<u2"), ("name_off", "<u2"), ("pos", "<i4"), ("event_idx", "<i4"),
                         ("diff", "<f8"), ("name_len", "<u2"), ("contig", "<u2"), ("flags", "u1"), ("kbits_fwd", "u1"), ("kbits_rev", "u1"), ("pad", "u1")])
assert RECORD_DTYPE.itemsize == 32

CALL_DTYPE = np.dtype([("read_off", "<i8"), ("prob", "<f8"), ("feat", "<f8", (MC_MAXK + 1,)), ("read_len", "<i4"),
                       ("mpos", "<i4"), ("site", "<i4"), ("close_rec", "<u4"), ("win_contig", "<u2"), ("chrom_contig", "<u2"),
                       ("kind", "u1"), ("rev", "u1"), ("n_empty", "u1"), ("empty_mask", "u1"), ("model_sel", "u1"),
                       ("label", "u1"), ("err", "u1"), ("pad0", "u1"), ("seg", "<u4"), ("pad1", "<u4"), ("pad2", "<u4")])
assert CALL_DTYPE.itemsize == 128

class LocusEntry(C.Structure):
    _fields_ = [("hash", C.c_uint64), ("first_off", C.c_uint64), ("check", C.c_uint64), ("depth", C.c_uint32), ("meth", C.c_uint32)]


class TrainJob(C.Structure):
    _fields_ = [("d_x", C.c_void_p), ("d_y", C.c_void_p), ("d_w", C.c_void_p), ("d_loss_curve", C.c_void_p), ("idx_off", C.c_int64),
                ("n", C.c_int32), ("d", C.c_int32), ("max_iter", C.c_int32), ("n_iter_no_change", C.c_int32), ("alpha", C.c_double),
                ("lr", C.c_double), ("tol", C.c_double), ("best_loss", C.c_double), ("n_iter", C.c_int32), ("no_improve", C.c_int32),
                ("stopped", C.c_int32), ("pad", C.c_int32)]


MC_TRAIN_HIDDEN, MC_TRAIN_BATCH = 100, 200

CARRY_BYTES = 192          # sizeof(mc_carry): the row (128 B), valid, first_kept_contig, chunk count, padding

QUAL_DTYPE = np.dtype([("hash", "<u8"), ("check", "<u4"), ("len", "<u4"), ("qual", "<f8")])
assert QUAL_DTYPE.itemsize == 24
DIFFS_ROW_DTYPE = np.dtype([("line_off", "<u8"), ("slot", "<u4"), ("values_off", "<u4"), ("values_len", "<u4"), ("prob_off", "<u4"),
                            ("prob_len", "<u4"), ("pad", "<u4")])
assert DIFFS_ROW_DTYPE.itemsize == 32


class McallerCudaError(RuntimeError):
    pass


_lib = None

_PROTOS = {
    "mc_version": (C.c_int, []),
    "mc_sizeof": (C.c_int, [C.c_int]),
    "mc_last_error": (C.c_char_p, []),
    "mc_read_u64": (C.c_int, [C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p]),
    "mc_scan": (C.c_int, [C.c_void_p, C.c_int64, C.POINTER(RefIndex), C.c_int, C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p,
                          C.c_void_p]),
    "mc_scan_run_len": (C.c_int, [C.c_int64]),
    "mc_scan_set_run_len": (C.c_int, [C.c_int]),
    "mc_num_tiles": (C.c_int64, [C.c_int64]),
    "mc_workspace_bytes": (C.c_int64, [C.c_int64]),
    # d_text, nbytes, ref, d_tile_tab, n_tiles, d_run_tab, run_len, d_rec_in, rec_in_cap, d_scan_counters, d_rec_out, rec_out_cap,
    # d_n_out, d_seg_flags, d_run_first, d_ws, stream
    "mc_order_records": (C.c_int, [C.c_void_p, C.c_int64, C.POINTER(RefIndex), C.c_void_p, C.c_int64, C.c_void_p, C.c_int, C.c_void_p,
                                   C.c_int64, C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    # d_text, d_rec, d_n_records, rec_cap, d_seg_flags, d_run_first, n_runs, d_seg_start, d_nseg, d_ws, stream
    "mc_segment_reads": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p,
                                   C.c_void_p, C.c_void_p]),
    # d_text, d_rec, d_seg_start, d_nseg, seg_cap, d_table, table_size, d_seg_qual, d_err, stream
    "mc_segment_quality": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p, C.c_int64, C.c_void_p,
                                     C.c_void_p, C.c_void_p]),
    # d_rec, d_n_records, rec_cap, d_seg_start, d_nseg, seg_cap, d_seg_qual, ref, skip, qual, two_models, d_calls, call_cap,
    # d_seg_count, d_ncalls, d_ws, d_spill, spill_cap, stream
    "mc_build_windows": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p, C.POINTER(RefIndex),
                                   C.c_int, C.c_double, C.c_int, C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                   C.c_int64, C.c_void_p]),
    "mc_carry_reset": (C.c_int, [C.c_void_p, C.c_void_p]),
    # d_rows, d_ncalls, d_rec, d_n_records, d_seg_start, d_nseg, d_seg_qual, qual_thresh, d_carry, d_nrows_out, d_abort, stream
    "mc_carry_rows": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_double, C.c_void_p,
                                C.c_void_p, C.c_void_p, C.c_void_p]),
    # d_counters, rec_cap, d_n_records, rec_out_cap, d_nseg, seg_cap, d_ncalls, call_cap, d_abort, d_sticky, stream
    "mc_chunk_guard": (C.c_int, [C.c_void_p, C.c_int64, C.c_void_p, C.c_int64, C.c_void_p, C.c_int64, C.c_void_p, C.c_int64, C.c_void_p,
                                 C.c_void_p, C.c_void_p]),
    # d_carry, closing_contig, d_next_contigs, from, count, d_row_out, d_depth, d_meth, d_first, n_sites, d_row_base, stream
    "mc_carry_close": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                 C.c_int64, C.c_void_p, C.c_void_p]),
    "mc_classify_workspace_bytes": (C.c_int64, [C.c_int64]),
    # d_calls, d_nrows, row_cap, models, d_ws, stream
    "mc_classify": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.POINTER(Model), C.c_void_p, C.c_void_p]),
    # d_calls, d_nrows, row_cap, d_depth, d_meth, d_first, n_sites, d_row_base, d_odd, odd_cap, d_n_odd, d_abort, stream
    "mc_hist_accumulate": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p,
                                     C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p]),
    "mc_count_calls": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p]),
    # d_depth, d_meth, n_sites, depth_thresh, mod_thresh, control, d_flags, d_count, stream
    "mc_bed_select": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_int64, C.c_double, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p]),
    # h_calls, n_calls, h_text, carry_name, carry_name_len, contig_names, marked_fwd, marked_rev, contig_len, n_contigs, k,
    # base_label, mod_label, with_prob, max_threads, out, out_cap
    "mc_format_rows": (C.c_int64, [C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                   C.c_int32, C.c_int32, C.c_char_p, C.c_char_p, C.c_int32, C.c_int32, C.c_void_p, C.c_int64]),
    "mc_fastq_tiles": (C.c_int64, [C.c_int64]),
    "mc_fastq_index": (C.c_int, [C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p]),
    "mc_fastq_quality": (C.c_int, [C.c_void_p, C.c_int64, C.c_void_p, C.c_int64, C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p,
                                   C.c_void_p]),
    "mc_synth_genome": (C.c_int, [C.POINTER(SynthSpec), C.c_void_p, C.c_int64, C.c_void_p]),
    "mc_synth_sizes": (C.c_int, [C.POINTER(SynthSpec), C.c_int64, C.c_int64, C.c_int64, C.c_void_p, C.c_void_p]),
    "mc_synth_write": (C.c_int, [C.POINTER(SynthSpec), C.c_int64, C.c_int64, C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p]),
    "mc_diffs_aggregate_ex": (C.c_int, [C.c_void_p, C.c_int64, C.c_int64, C.c_void_p, C.c_int64, C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p]),
    "mc_diffs_rehash": (C.c_int, [C.c_void_p, C.c_int64, C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p]),
    "mc_diffs_rows": (C.c_int, [C.c_void_p, C.c_int64, C.c_void_p, C.c_int64, C.c_void_p, C.c_int64, C.c_void_p, C.c_int64, C.c_void_p,
                                C.c_void_p]),
    # d_jobs, n_jobs, stream
    "mc_mlp_train_init": (C.c_int, [C.c_void_p, C.c_int32, C.c_void_p]),
    # d_jobs, n_jobs, d_idx, epochs, stream
    "mc_mlp_train_epochs": (C.c_int, [C.c_void_p, C.c_int32, C.c_void_p, C.c_int32, C.c_void_p]),
    "mc_diffs_colstats": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p, C.c_int64, C.c_int, C.c_void_p, C.c_void_p,
                                    C.c_void_p, C.c_void_p, C.c_void_p]),
}

# symbols every build must export (checked by the CPU test-suite against include/mcaller_b200.h)
EXPORTS = sorted(_PROTOS)


def load(path=LIB_PATH):
    """dlopen the library and attach prototypes (no CUDA call is made)."""
    if not os.path.exists(path):
        raise McallerCudaError("libmcaller_b200.so is not built (%s); run `python -m mcaller_b200.build` -- there is no CPU fallback" % path)
    lib = C.CDLL(path)
    for name, (res, args) in _PROTOS.items():
        fn = getattr(lib, name)
        fn.restype = res
        fn.argtypes = args
    return lib


def lib():
    global _lib
    if _lib is None:
        _lib = load()
        if _lib.mc_version() != MC_ABI_VERSION:
            raise McallerCudaError("ABI version mismatch")
    return _lib


def check(rc):
    if rc != 0:
        raise McallerCudaError("libmcaller_b200: rc=%d %s" % (rc, lib().mc_last_error().decode(errors="replace")))
