"""ctypes binding of libbbk.so (include/bbk.h).  There is no fallback: if the CUDA library is
missing or does not load, importing a kernel entry point raises."""
import ctypes
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "lib", "libbbk.so")

FIT_S_GIVEN = 7777          # input value of FitResult.status: use FitResult.smoothing as s
FIT_TOO_MANY_BINS = -13
PHIST_BINS = 4096
PHIST_LEN = PHIST_BINS + 2
BH_UNSORTED = 0
BH_POSITIONAL = 1

FIT_STATUS = {
    0: None,
    -11: (ZeroDivisionError, "float division by zero (a distance bin holds no possible pairs; fithic.py:216)"),
    -12: (ValueError, "m > k must hold (fewer than 4 equal-occupancy bins came out; scipy UnivariateSpline)"),
    -13: (RuntimeError, "more equal-occupancy bins than the workspace was sized for"),
    -14: (ZeroDivisionError, "float division by zero (no in-range contacts: observedIntraInRangeSum == 0; fithic.py:216)"),
    -15: (ValueError, "x must be increasing if s > 0"),
    -16: (ValueError, "no genomic distance lies inside [min(x), max(x)]; nothing to evaluate the spline on"),
    -17: (RuntimeError, "the fit problem's sizes, pointers or workspace do not allow the fit (bbk_fit_batched)"),
}


class BbkError(RuntimeError):
    pass


class FitResult(ctypes.Structure):
    _fields_ = [
        ("status", ctypes.c_int32), ("n_out", ctypes.c_int32), ("k0", ctypes.c_int32), ("L", ctypes.c_int32),
        ("n_knots", ctypes.c_int32), ("ier", ctypes.c_int32), ("S", ctypes.c_int64),
        ("min_x", ctypes.c_double), ("max_x", ctypes.c_double), ("residual", ctypes.c_double),
        ("fp", ctypes.c_double), ("smoothing", ctypes.c_double), ("phase_cycles", ctypes.c_int64 * 6),
        ("spline_diag", ctypes.c_int64 * 8), ("y_min", ctypes.c_double),
    ]


class FitProblem(ctypes.Structure):
    _fields_ = [("d_possible", ctypes.c_void_p), ("d_obs_sum", ctypes.c_void_p), ("d_totals", ctypes.c_void_p),
                ("d_result", ctypes.c_void_p), ("d_x", ctypes.c_void_p), ("d_y", ctypes.c_void_p), ("d_bin_of_key", ctypes.c_void_p),
                ("d_spline_y", ctypes.c_void_p), ("d_spline_raw", ctypes.c_void_p), ("d_knots", ctypes.c_void_p),
                ("d_coefs", ctypes.c_void_p), ("d_workspace", ctypes.c_void_p), ("workspace_bytes", ctypes.c_uint64),
                ("nkeys", ctypes.c_int32), ("max_bins", ctypes.c_int32)]


class BiasTable(ctypes.Structure):
    _fields_ = [("d_bias", ctypes.c_void_p), ("d_chrom_base", ctypes.c_void_p), ("d_mid0", ctypes.c_void_p),
                ("n_chrom", ctypes.c_int32), ("step", ctypes.c_int64)]


class ScoreState(ctypes.Structure):
    _fields_ = [("n_list", ctypes.c_uint64), ("n_cand", ctypes.c_uint64), ("overflow", ctypes.c_int32),
                ("cand_overflow", ctypes.c_int32), ("exact", ctypes.c_int32), ("reserved", ctypes.c_int32)]


class DeferredList(ctypes.Structure):
    _fields_ = [("d_row", ctypes.c_void_p), ("d_count", ctypes.c_void_p), ("d_prior", ctypes.c_void_p),
                ("capacity", ctypes.c_int64)]


TILE_ROWS = 2048
PACK_CHUNK = 4096


class PackState(ctypes.Structure):
    _fields_ = [("n_p", ctypes.c_uint64), ("n_q", ctypes.c_uint64), ("overflow", ctypes.c_int32), ("reserved", ctypes.c_int32)]


class Candidates(ctypes.Structure):
    _fields_ = [("d_keys", ctypes.c_void_p), ("d_rows", ctypes.c_void_p), ("capacity", ctypes.c_int64)]


class BhSegment(ctypes.Structure):
    _fields_ = [("d_p_hist", ctypes.c_void_p), ("d_state", ctypes.c_void_p), ("cands", Candidates), ("n_tests", ctypes.c_int64)]


_vp, _i32, _i64, _f64, _sz = ctypes.c_void_p, ctypes.c_int32, ctypes.c_int64, ctypes.c_double, ctypes.c_size_t

# name -> (restype, argtypes); exactly the prototypes of include/bbk.h
SIGNATURES = {
    "bbk_version": (ctypes.c_int, []),
    "bbk_last_error": (ctypes.c_int, [ctypes.c_char_p, _sz]),
    "bbk_sm_count": (ctypes.c_int, []),
    "bbk_hist_init": (ctypes.c_int, [_vp, _i32, _vp, _vp]),
    "bbk_hist_pairs": (ctypes.c_int, [_vp, _vp, _vp, _vp, _vp, _i64, _i64, _i64, _i64, _i32, _vp, _vp, _vp]),
    "bbk_hist_pairs_excluding": (ctypes.c_int, [_vp, _vp, _vp, _vp, _vp, _vp, _f64, _i64, _i64, _i64, _i64, _i32, _vp, _vp, _vp]),
    "bbk_possible_pairs": (ctypes.c_int, [_vp, _vp, _i32, _i64, _i32, _vp, _vp]),
    "bbk_fit_workspace_bytes": (_sz, [_i32, _i32]),
    "bbk_fit": (ctypes.c_int, [_vp, _vp, _i32, _vp, _i32, _i64, _i64, _i64, _i32, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp,
                               _vp, _sz, _vp]),
    "bbk_fit_batched": (ctypes.c_int, [_vp, _i32, _i32, _i64, _i64, _i64, _vp]),
    "bbk_fit_from_bins": (ctypes.c_int, [_vp, _vp, _i32, _i32, _i64, _vp, _vp, _vp, _vp, _vp, _vp, _sz, _vp]),
    "bbk_pvalues": (ctypes.c_int, [_vp, _vp, _vp, _vp, _vp, _i64, _i32, _i64, _i64, _i64, _vp, _vp,
                                   ctypes.POINTER(BiasTable), _vp, _vp, _vp]),
    "bbk_bh_workspace_bytes": (_sz, [_i64]),
    "bbk_bh_qvalues": (ctypes.c_int, [_vp, _i64, _i64, _i32, _vp, _vp, _vp, _vp, _sz, _vp]),
    "bbk_decimate_workspace_bytes": (_sz, [_i64]),
    "bbk_decimate": (ctypes.c_int, [_vp, _i64, _i64, _vp, _vp, _vp, _sz, _vp]),
    "bbk_contact_band_ingest": (ctypes.c_int, [_vp, _vp, _vp, _i64, _i64, _i32, _vp, _vp, _vp, _vp, _vp]),
    "bbk_contact_band_normalize": (ctypes.c_int, [_vp, _vp, _vp, _i64, _vp, _vp, _i32, _vp, _vp, _vp]),
    "bbk_bh_select": (ctypes.c_int, [_vp, _i64, _i64, _vp, _vp, _vp, _vp, _i64, _vp, _vp, _sz, _vp]),
    "bbk_bh_fix_ones_dev": (ctypes.c_int, [_vp, _i64, _vp, _vp, _vp]),
    "bbk_count_band": (ctypes.c_int, [_vp, _i64, _f64, _f64, _vp, _vp]),
    "bbk_stats_pack": (ctypes.c_int, [_vp, _vp, _i32, _i32, _vp]),
    "bbk_stats_unpack": (ctypes.c_int, [_vp, _vp, _i32, _vp]),
    "bbk_score_begin": (ctypes.c_int, [_vp, _vp, _vp]),
    "bbk_bias_flags_bytes": (_sz, [_i64]),
    "bbk_bias_flags": (ctypes.c_int, [_vp, _i64, _vp, _vp]),
    "bbk_score_guard": (ctypes.c_int, [_vp, _vp, _vp, _vp]),
    "bbk_score_pairs": (ctypes.c_int, [_vp, _vp, _vp, _i64, _i32, _i64, _i64, _i64, _vp, _vp, ctypes.POINTER(BiasTable), _vp, _i64,
                                       _vp, _vp, _vp, ctypes.POINTER(Candidates), ctypes.POINTER(DeferredList), _vp, _vp]),
    "bbk_score_deferred": (ctypes.c_int, [ctypes.POINTER(DeferredList), _vp, _vp, _vp, _vp, ctypes.POINTER(Candidates), _vp, _vp]),
    "bbk_extract_workspace_bytes": (_sz, [_i64]),
    "bbk_extract_contacts": (ctypes.c_int, [_vp, _i64, _f64, _f64, _i32, _f64, _f64, _vp, _i64, _vp, _vp, _sz, _vp]),
    "bbk_pack_chunks": (_i64, [_i64]),
    "bbk_pack_code_words": (_i64, [_i64]),
    "bbk_pack_scores": (ctypes.c_int, [_vp, _vp, _i64, _vp, _vp, _vp, _i64, _vp, _i64, _vp, _vp]),
    "bbk_unpack_records": (ctypes.c_int, [_vp, _i64, _i64, _vp, _vp, _vp, _vp]),
    "bbk_bh_qvalues_listed": (ctypes.c_int, [_vp, _i64, _i64, _vp, _vp, ctypes.POINTER(Candidates), _vp, _vp, _sz, _vp]),
    "bbk_bh_segmented_workspace_bytes": (_sz, [_i64, _i32]),
    "bbk_bh_qvalues_segmented": (ctypes.c_int, [_vp, _i64, _vp, _vp, _i32, _vp, _vp, _sz, _vp]),
    "bbk_bh_select_listed": (ctypes.c_int, [_vp, _i64, _i64, _vp, _vp, ctypes.POINTER(Candidates), _vp, _vp, _vp, _i64, _vp, _vp, _sz, _vp]),
    "bbk_bh_gathered_workspace_bytes": (_sz, [_i32, _i64]),
    "bbk_bh_pack_count": (ctypes.c_int, [_vp, _vp, _vp]),
    "bbk_bh_rank_gathered_padded": (ctypes.c_int, [_vp, _i32, _i64, _i32, _vp, _vp, _vp, _vp, _vp, _vp, _sz, _vp]),
    "bbk_bh_rank_gathered_all": (ctypes.c_int, [_vp, _i32, _i64, _vp, _vp, _vp, _vp, _vp, _sz, _vp]),
    "bbk_synth_contacts_range": (ctypes.c_int, [_i64, _i64, _i64, _f64, _f64, ctypes.c_uint64, _vp, _i64, _i64, _vp, _vp, _vp, _vp]),
    "bbk_synth_n_pairs": (_i64, [_i64, _i64]),
    "bbk_synth_contacts": (ctypes.c_int, [_i64, _i64, _i64, _f64, _f64, ctypes.c_uint64, _vp, _vp, _vp, _vp, _vp]),
}

_lib = None


def load():
    """Load libbbk.so (once).  Raises BbkError when it is missing - there is no CPU path."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise BbkError("%s not found: build it with `python -m blueberry_b200.build` "
                       "(blueberry_b200 has no CPU fallback)" % LIB_PATH)
    lib = ctypes.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def last_error():
    buf = ctypes.create_string_buffer(512)
    load().bbk_last_error(buf, 512)
    return buf.value.decode(errors="replace")


def check(rc, what):
    if rc != 0:
        raise BbkError("%s failed (code %d): %s" % (what, rc, last_error()))


def ptr(t):
    """Device pointer of a torch tensor (or None)."""
    return None if t is None else ctypes.c_void_p(t.data_ptr())


def stream_ptr(stream=None):
    import torch
    s = stream if stream is not None else torch.cuda.current_stream()
    return ctypes.c_void_p(s.cuda_stream)
