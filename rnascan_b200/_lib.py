"""ctypes binding of librnascan_b200.so (the C ABI declared in include/rnascan_b200.h).

There is no CPU fallback: if the shared library is missing or cannot be loaded the import
of this module raises, and every device entry point raises ``RnascanCudaError`` when the
CUDA runtime reports an error (including "no device").
"""
import ctypes
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "librnascan_b200.so")

RS_OK, RS_ERR_INVALID, RS_ERR_CUDA, RS_ERR_WORKSPACE = 0, 1, 2, 3
RS_F32, RS_F64 = 0, 1
RS_MODE_STRUCT, RS_MODE_AND = 0, 1
RS_ROWS_F32, RS_ROWS_F32_SHADOW, RS_ROWS_Q8, RS_ROWS_Q4 = 0, 1, 2, 3
RS_SEP, RS_RNA_OTHER, RS_SS_OTHER, RS_MAX_W = 0xFF, 0x0C, 0x0F, 64
RS_ALPHA_OTHER, RS_ALPHA_LOWER = 0x1F, 0x20
RS_MILLI_NAN, RS_MILLI_NINF, RS_MILLI_NEG0, RS_MILLI_RANGE = -2147483648, -2147483647, -2147483646, -2147483645


class RnascanCudaError(RuntimeError):
    pass


def _load():
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            "rnascan_b200: %s not found -- build it with `python -c 'import __graft_entry__ as g; "
            "g.build()'` or `make -C rnascan_b200/csrc` (there is no CPU fallback)" % LIB_PATH)
    return ctypes.CDLL(LIB_PATH)


lib = _load()

_i64, _vp, _int, _dbl = ctypes.c_int64, ctypes.c_void_p, ctypes.c_int, ctypes.c_double
_u32 = ctypes.c_uint32
_SIGS = {
    "rs_version": ([], _int),
    "rs_last_error": ([], ctypes.c_char_p),
    "rs_device_info": ([_vp, _vp, _vp], _int),
    "rs_padded_count": ([_i64], _i64),
    "rs_scan_workspace_bytes": ([_i64, _i64], _i64),
    "rs_set_reserved_sms": ([_int], _int),
    "rs_prof_begin": ([_int], _int),
    "rs_prof_end": ([_vp, _int, _vp], _int),
    "rs_host_fasta_index": ([_vp, _i64, _vp, _vp, _vp], _int),
    "rs_host_fasta_fill": ([_vp, _i64, _int, _vp, _vp, _vp, _vp, _vp, _vp], _int),
    "rs_host_profiles_open": ([_vp, _i64, _int, _vp, _vp], _int),
    "rs_host_profiles_fill": ([_vp, _int, _vp, _vp, _vp], _int),
    "rs_host_profiles_close": ([_vp], _int),
    "rs_host_parse_doubles": ([ctypes.c_char_p, _i64, _vp, _i64, _vp, _vp], _int),
    "rs_host_encode_rna": ([_vp, _i64, _vp], _int),
    "rs_host_encode_struct": ([_vp, _i64, _vp], _int),
    "rs_host_encode_alpha": ([_vp, _i64, ctypes.c_char_p, _int, _vp], _int),
    "rs_host_log_odds": ([_vp, _vp, _int, _int, _vp], _int),
    "rs_host_annotate_structures": ([_vp, _vp, _vp, _i64, _vp, _vp], _int),
    "rs_host_format_hits": ([_i64, _i64, _vp, ctypes.c_char_p, _vp, ctypes.c_char_p, _vp, ctypes.c_char_p, _vp, _i64,
                             _vp, _vp, _int, _vp, _vp, _i64, _vp], _int),
    "rs_host_format_hits_combined": ([_i64, _i64, _vp, ctypes.c_char_p, _vp, ctypes.c_char_p, _vp, ctypes.c_char_p,
                                      _vp, ctypes.c_char_p, ctypes.c_char_p, _vp, _i64, _vp, _vp, _vp, _int, _vp,
                                      _int, _vp, _vp, _i64, _vp], _int),
    "rs_hist": ([_vp, _i64, _vp, _vp], _int),
    "rs_hist_rna": ([_vp, _i64, _vp, _vp], _int),
    "rs_hist_alpha": ([_vp, _i64, _vp, _vp], _int),
    "rs_scores_dense_seq": ([_vp, _i64, _vp, _int, _vp, _vp], _int),
    "rs_scores_dense_struct": ([_vp, _i64, _vp, _int, _vp, _vp], _int),
    "rs_scores_dense_struct_milli": ([_vp, _i64, _vp, _int, _vp, _vp], _int),
    "rs_scores_dense_alpha": ([_vp, _i64, _vp, _int, _int, _vp, _vp], _int),
    "rs_scores_dense_profile": ([_vp, _int, _i64, _vp, _vp, _int, _vp, _vp], _int),
    "rs_profile_stats": ([_vp, _int, _i64, _vp, _vp], _int),
    "rs_scan_seq": ([_vp, _i64, _vp, _int, _dbl, _i64, _vp, _vp, _vp, _vp, _i64, _vp], _int),
    "rs_scan_struct_onehot": ([_vp, _i64, _vp, _int, _dbl, _i64, _vp, _vp, _vp, _vp, _i64, _vp], _int),
    "rs_scan_alpha": ([_vp, _i64, _vp, _int, _int, _dbl, _i64, _vp, _vp, _vp, _vp, _i64, _vp], _int),
    "rs_scan_pair_onehot": ([_vp, _vp, _i64, _vp, _vp, _int, _dbl, _i64, _vp, _vp, _vp, _vp, _vp, _i64,
                             _vp], _int),
    "rs_scan_fused": ([_vp, _vp, _int, _i64, _vp, _vp, _int, _dbl, _dbl, _int, _i64, _vp, _vp, _vp, _vp,
                       _vp, _i64, _vp], _int),
    "rs_provisional_table": ([_vp, _vp, _int, _int, _vp, _vp], _int),
    "rs_scan_onehot_begin": ([_int, _vp, _i64, _vp, _vp, _int, _dbl, _dbl, _i64, _vp, _i64, _vp], _int),
    "rs_scan_onehot_begin_notify": ([_int, _vp, _i64, _vp, _vp, _int, _dbl, _dbl, _i64, _vp, _i64, _vp, _u32, _vp,
                                     _vp], _int),
    "rs_scan_onehot_finish": ([_int, _vp, _i64, _vp, _int, _dbl, _i64, _vp, _vp, _vp, _vp, _i64, _vp], _int),
    "rs_refine_hits_seq": ([_vp, _i64, _vp, _int, _dbl, _vp, _i64, _vp, _vp, _vp, _vp, _vp, _i64, _vp], _int),
    "rs_scan_fused_candidates": ([_vp, _vp, _int, _i64, _vp, _int, _dbl, _dbl, _i64, _vp, _vp, _i64, _vp, _vp], _int),
    "rs_scan_fused_candidates_counting": ([_vp, _vp, _int, _i64, _vp, _int, _dbl, _dbl, _i64, _vp, _vp, _vp, _i64, _vp,
                                           _vp], _int),
    "rs_scan_fused_resolve": ([_vp, _i64, _vp, _int, _dbl, _i64, _i64, _vp, _vp, _vp, _vp, _vp, _i64, _vp], _int),
    "rs_filter_workspace_bytes": ([_i64, _i64], _i64),
    "rs_filter_profile": ([_vp, _vp, _int, _dbl, _i64, _vp, _vp, _int, _dbl, _dbl, _i64, _i64, _vp, _i64, _vp, _vp, _vp,
                           _vp, _i64, _vp], _int),
    "rs_refine_packed_workspace_bytes": ([_i64], _i64),
    "rs_refine_candidates_packed": ([_vp, _vp, _i64, _vp, _int, _dbl, _vp, _vp, _vp, _i64, _vp], _int),
    "rs_resolve_workspace_bytes": ([_i64], _i64),
    "rs_resolve_candidates": ([_vp, _i64, _vp, _int, _vp, _vp, _vp, _int, _dbl, _vp, _vp, _vp, _vp, _vp, _i64,
                               _vp], _int),
    "rs_host_rows_stats": ([_vp, _int, _i64, _int, _vp], _int),
    "rs_host_rows_to_f32": ([_vp, _i64, _vp, _int], _int),
    "rs_host_copy": ([_vp, _vp, _i64, _int], _int),
    "rs_host_quantize_q8": ([_vp, _int, _i64, _vp, _dbl, _vp, _int, _vp], _int),
    "rs_host_quantize_q4": ([_vp, _int, _i64, _vp, _dbl, _vp, _int, _vp], _int),
    "rs_host_gather_windows": ([_vp, _int, _i64, _vp, _i64, _vp, _i64, _int, _vp, _vp, _int], _int),
    "rs_scan_batched_workspace_bytes": ([_i64, _int, _int, _i64], _i64),
    "rs_set_batched_path": ([_int], _int),
    "rs_last_batched_path": ([], _int),
    "rs_scan_batched": ([_vp, _vp, _int, _i64, _int, _vp, _vp, _vp, _int, _dbl, _dbl, _int, _i64, _vp, _vp,
                         _vp, _vp, _vp, _vp, _vp, _i64, _vp], _int),
    "rs_scan_onehot_many_workspace_bytes": ([_int, _i64, _int, _int], _i64),
    "rs_scan_onehot_many": ([_int, _vp, _i64, _int, _vp, _vp, _int, _dbl, _i64, _vp, _vp, _vp, _vp, _vp, _vp, _i64,
                             _vp], _int),
    "rs_scan_pair_onehot_many_workspace_bytes": ([_i64, _int, _int], _i64),
    "rs_scan_pair_onehot_many": ([_vp, _vp, _i64, _int, _vp, _vp, _vp, _int, _dbl, _i64, _vp, _vp, _vp, _vp, _vp,
                                  _vp, _i64, _vp], _int),
    "rs_scan_batched_shadow": ([_vp, _vp, _vp, _i64, _int, _vp, _vp, _vp, _int, _dbl, _dbl, _int, _i64, _vp, _vp,
                                _vp, _vp, _vp, _vp, _vp, _i64, _vp], _int),
}
EXPORTS = sorted(_SIGS)
for _name, (_args, _res) in _SIGS.items():
    _fn = getattr(lib, _name)          # AttributeError here == header/library mismatch
    _fn.argtypes = _args
    _fn.restype = _res


def last_error():
    return lib.rs_last_error().decode("utf-8", "replace")


def check(rc):
    """Raise the Python exception matching the C status (the reference raises ValueError
    for malformed matrices, _pwm.c:96-113)."""
    if rc == RS_OK:
        return
    msg = last_error()
    if rc == RS_ERR_INVALID:
        raise ValueError(msg)
    if rc == RS_ERR_WORKSPACE:
        raise MemoryError(msg)
    raise RnascanCudaError(msg)
