"""ctypes binding of libhanselx.so (see include/hanselx.h).  No CPU fallback: if the
library is missing or a call fails this raises."""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libhanselx.so")

HX_OK, HX_HOLE = 0, 1
HX_E_CUDA, HX_E_ARG, HX_E_BAND, HX_E_READ, HX_E_NOMEM, HX_E_STATE = -1, -2, -3, -4, -5, -6
HX_F_VSITE_TO, HX_F_KEEP_UNSYMBOLS = 1, 2

_p, _i32, _i64, _u64, _int, _dbl, _flt = C.c_void_p, C.c_int32, C.c_int64, C.c_uint64, C.c_int, C.c_double, C.c_float
_pp = C.POINTER(C.c_void_p)

# name -> (restype, argtypes); must list every symbol include/hanselx.h declares
SIGNATURES = {
    "hx_last_error": (C.c_char_p, []),
    "hx_version": (_int, []),
    "hx_device_count": (_int, [C.POINTER(_int)]),
    "hx_create": (_int, [_i32, _i32, _i32, _pp]),
    "hx_destroy": (_int, [_p]),
    "hx_copy": (_int, [_p, _pp]),
    "hx_info": (_int, [_p, C.POINTER(_i32), C.POINTER(_i32), C.POINTER(_i32)]),
    "hx_stream": (_int, [_p, _pp]),
    "hx_set_stream": (_int, [_p, _p]),
    "hx_sync": (_int, [_p]),
    "hx_ingest_host": (_int, [_p, _p, _p, _p, _i64, _p]),
    "hx_counts_pack": (_int, [_p, _i32, _pp, C.POINTER(_i64)]),
    "hx_counts_unpack": (_int, [_p, C.POINTER(_i32)]),
    "hx_counts_unpack_async": (_int, [_p, _p]),
    "hx_counts_pack_overflowed": (_int, [_p, C.POINTER(_i32)]),
    "hx_counts_max": (_int, [_p, C.POINTER(C.c_uint32)]),
    "hx_ingest_host_compact": (_int, [_p, _p, _p, _p, _i64, _i64, _p]),
    "hx_dense_encode": (_int, [_p, _p, _p, _i64, _int, _p]),
    "hx_dense_free": (None, [_p]),
    "hx_ingest_host_dense": (_int, [_p, _p, _p, _p, _i64, _p, _i32, _p, _p, _i64, _i64, _i64, _p]),
    "hx_ingest_device": (_int, [_p, _p, _p, _p, _i64]),
    "hx_set_ingest_kernel": (_int, [_p, _int]),
    "hx_set_ingest_sms": (_int, [_p, _int]),
    "hx_ingest_totals": (_int, [_p, _p]),
    "hx_counts_buffer": (_int, [_p, _pp, C.POINTER(_i64), _pp, C.POINTER(_i64)]),
    "hx_counts_ipc_export": (_int, [_p, _i32, _p]),
    "hx_counts_ipc_import": (_int, [_p, _p, _i32, _i32]),
    "hx_counts_ipc_close": (_int, [_p]),
    "hx_finalize_counts": (_int, [_p]),
    "hx_reset_counts": (_int, [_p]),
    "hx_add_observation": (_int, [_p, _int, _int, _i32, _i32, _flt]),
    "hx_get_observation": (_int, [_p, _int, _int, _i32, _i32, C.POINTER(_flt)]),
    "hx_reweight_observation": (_int, [_p, _int, _int, _i32, _i32, _dbl, C.POINTER(_dbl)]),
    "hx_reweight_matrix": (_int, [_p, _dbl]),
    "hx_counts_all": (_int, [_p, _p]),
    "hx_marginal_of_at": (_int, [_p, _int, _i32, C.POINTER(_dbl)]),
    "hx_edge_weights_at": (_int, [_p, _i32, _p, _i32, _int, _p, C.POINTER(_dbl), C.POINTER(_int)]),
    "hx_generate_path": (_int, [_p, _p, _i32, _int, _p, _p, C.POINTER(_i32)]),
    "hx_reweight_path": (_int, [_p, _p, _dbl, C.POINTER(_dbl)]),
    "hx_recover": (_int, [_p, _p, _i32, _int, _i32, _dbl, _p, _p, C.POINTER(_i32)]),
    "hx_assign_reads": (_int, [_p, _p, _i32, _p, _p, _p, _i64, _i32, _p, _p, _p, _p, _p, _p, _p]),
    "hx_read_classes": (_int, [_p, _p, _i32, _p, _p, _p, _i64, _i32, _p, _p, _p]),
    "hx_read_classes_get": (_int, [_p, _p, _p, _p]),
    "hx_em_abundance": (_int, [_i32, _i64, _p, _p, _p, _i32, _dbl, _p, _p, _p, _p]),
    "hx_em_bootstrap": (_int, [_p, _i32, _i64, _p, _p, _p, _i32, _u64, _i32, _dbl, _p, _p, _p, _p, _p]),
    "hx_score_paths": (_int, [_p, _p, _i32, _i32, _int, _p, _p, _p, _p, _p, _p, _p]),
    "hx_pack_bam": (_int, [C.c_char_p, C.c_char_p, _i32, _i32, _p, _i32, _int, _int, _p]),
    "hx_pack_bam_ex": (_int, [C.c_char_p, C.c_char_p, _i32, _i32, _p, _i32, _int, _int, _i32, _p, _p]),
    "hx_pack_free": (None, [_p]),
    "hx_count_coverage": (_int, [C.c_char_p, C.c_char_p, _i32, _i32, _int, _p]),
    "hx_count_coverage_gpu": (_int, [C.c_char_p, C.c_char_p, _i32, _i32, _int, _i32, _p]),
    "hx_bam_contig_length": (_int, [C.c_char_p, C.c_char_p, C.POINTER(_i32)]),
    "hx_inflate_raw": (_int, [_p, _i64, _i64, _p, _i64, _i32]),
    "hx_probe_expected_rows": (_int, [_p, _p, _p, _p, _i64, _p]),
    "hx_counts_row_sums": (_int, [_p, _p]),
    "hx_device_math": (_int, [_i32, _int, _p, _p, _i64]),
    "hx_band_to_host": (_int, [_p, _p]),
    "hx_band_from_host": (_int, [_p, _p]),
    "hx_to_dense": (_int, [_p, _p]),
    "hx_last_kernel_ms": (_int, [_p, _int, C.POINTER(_flt)]),
    "hx_launch_count": (_int, [_p, C.POINTER(_i64)]),
}

class HxPacked(C.Structure):
    _fields_ = [("rank", C.POINTER(C.c_int32)), ("off", C.POINTER(C.c_int64)), ("codes", C.POINTER(C.c_uint8)),
                ("n_reads", C.c_int64), ("n_codes", C.c_int64), ("n_records", C.c_int64)]


class HxDense(C.Structure):
    _fields_ = [("blob", C.POINTER(C.c_uint8)), ("blob_bytes", C.c_int64), ("n_reads", C.c_int64),
                ("n_codes", C.c_int64), ("n_exc", C.c_int64), ("n_esc", C.c_int64), ("o_klen", C.c_int64),
                ("o_codes2", C.c_int64), ("o_exc", C.c_int64), ("o_esc_idx", C.c_int64), ("o_esc_delta", C.c_int64),
                ("klen_bytes", C.c_int32)]


_LIB = None


class HanselxError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__("hanselx error %d: %s" % (code, msg))
        self.code = code


def load():
    """dlopen libhanselx.so and type every entry point.  Raises if it is not built."""
    global _LIB
    if _LIB is not None:
        return _LIB
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(
            "gretel_b200: %s is missing - build it with `python -m gretel_b200.build` "
            "(nvcc, sm_100a).  There is no CPU fallback." % LIB_PATH)
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)
        fn.restype = res
        fn.argtypes = args
    _LIB = lib
    return lib


def check(rc, allow=()):
    if rc == HX_OK or rc in allow:
        return rc
    raise HanselxError(rc, load().hx_last_error().decode(errors="replace"))
