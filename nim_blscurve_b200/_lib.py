"""ctypes binding of libblsgpu.so (C ABI in include/blsgpu.h).

The library is the product; this module only loads it and declares prototypes.  There is no
fallback: if the shared object is missing or no CUDA device is visible, calls raise.
"""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("BLSGPU_LIB") or os.path.join(_HERE, "libblsgpu.so")   # env override: kernel-variant experiments

# every symbol include/blsgpu.h declares (tests check the export list against the header)
SYMBOLS = [
    "blsgpu_device_count", "blsgpu_create", "blsgpu_create_multi", "blsgpu_device_span", "blsgpu_destroy", "blsgpu_last_error", "blsgpu_capacity",
    "blsgpu_set_stream", "blsgpu_rlc_scalars", "blsgpu_batch_verify", "blsgpu_batch_verify_dev",
    "blsgpu_partial", "blsgpu_partial_dev", "blsgpu_finalize", "blsgpu_finalize_dev", "blsgpu_hash_to_g2", "blsgpu_aggregate_g1", "blsgpu_aggregate_g2",
    "blsgpu_msm_g1", "blsgpu_msm_g1_dev", "blsgpu_msm_g2", "blsgpu_msm_g2_dev", "blsgpu_combine", "blsgpu_last_stage_ms", "blsgpu_stage_name", "blsgpu_last_launches",
    "blsgpu_subtract_g1", "blsgpu_subtract_g2", "blsgpu_aggregate_g1_segments", "blsgpu_aggregate_verify", "blsgpu_fast_aggregate_verify",
    "blsgpu_pubkeys_from_bytes", "blsgpu_signatures_from_bytes", "blsgpu_pubkeys_to_bytes", "blsgpu_signatures_to_bytes",
    "blsgpu_test_fp", "blsgpu_test_field", "blsgpu_test_small_hash", "blsgpu_imad_peak", "blsgpu_fpmul_peak", "blsgpu_make_sets", "blsgpu_msm_make_inputs",
]

_lib = None


class BlsGpuError(RuntimeError):
    pass


def lib():
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise BlsGpuError(f"{LIB_PATH} not built: run `python -c 'import __graft_entry__ as g; g.build()'` "
                          "(nvcc, sm_100a). There is no CPU fallback.")
    L = C.CDLL(LIB_PATH)
    vp, sz, u8p = C.c_void_p, C.c_size_t, C.c_char_p
    L.blsgpu_device_count.restype = C.c_int
    L.blsgpu_create.restype = vp
    L.blsgpu_create.argtypes = [C.c_int, sz]
    L.blsgpu_create_multi.restype = vp
    L.blsgpu_create_multi.argtypes = [vp, C.c_int, sz]
    L.blsgpu_device_span.argtypes = [vp]
    L.blsgpu_destroy.argtypes = [vp]
    L.blsgpu_last_error.restype = C.c_char_p
    L.blsgpu_last_error.argtypes = [vp]
    L.blsgpu_capacity.restype = sz
    L.blsgpu_capacity.argtypes = [vp]
    L.blsgpu_set_stream.argtypes = [vp, vp]
    L.blsgpu_rlc_scalars.argtypes = [vp, u8p, sz, C.c_uint32, vp]
    L.blsgpu_batch_verify.argtypes = [vp, vp, sz, u8p, C.c_uint32, vp, vp]
    L.blsgpu_batch_verify_dev.argtypes = [vp, vp, sz, u8p, C.c_uint32, vp, vp]
    L.blsgpu_partial.argtypes = [vp, vp, C.c_int, sz, sz, sz, u8p, C.c_uint32, vp, vp, vp]
    L.blsgpu_finalize.argtypes = [vp, vp, sz, vp]
    L.blsgpu_partial_dev.argtypes = [vp, vp, sz, sz, sz, u8p, C.c_uint32, vp, vp]
    L.blsgpu_finalize_dev.argtypes = [vp, vp, sz, vp, vp]
    L.blsgpu_hash_to_g2.argtypes = [vp, vp, sz, sz, vp, sz, vp, vp]
    L.blsgpu_test_small_hash.argtypes = [vp, vp, sz, vp, vp]
    L.blsgpu_aggregate_g1.argtypes = [vp, vp, sz, vp]
    L.blsgpu_aggregate_g2.argtypes = [vp, vp, sz, vp]
    L.blsgpu_subtract_g1.argtypes = [vp, vp, vp, sz]
    L.blsgpu_subtract_g2.argtypes = [vp, vp, vp, sz]
    L.blsgpu_msm_g1.argtypes = [vp, vp, vp, sz, sz, vp]
    L.blsgpu_msm_g1_dev.argtypes = [vp, vp, vp, sz, sz, vp]
    L.blsgpu_msm_g2.argtypes = [vp, vp, vp, sz, sz, vp]
    L.blsgpu_msm_g2_dev.argtypes = [vp, vp, vp, sz, sz, vp]
    L.blsgpu_combine.argtypes = [vp, u8p, vp, vp, sz, vp, vp]
    L.blsgpu_aggregate_g1_segments.argtypes = [vp, vp, vp, sz, vp]
    L.blsgpu_aggregate_verify.argtypes = [vp, vp, sz, vp, vp, vp, sz, vp, vp]
    L.blsgpu_fast_aggregate_verify.argtypes = [vp, vp, sz, vp, sz, vp, sz, vp, vp]
    L.blsgpu_pubkeys_from_bytes.argtypes = [vp, vp, sz, sz, C.c_int, vp, vp]
    L.blsgpu_signatures_from_bytes.argtypes = [vp, vp, sz, sz, C.c_int, vp, vp]
    L.blsgpu_pubkeys_to_bytes.argtypes = [vp, vp, sz, vp]
    L.blsgpu_signatures_to_bytes.argtypes = [vp, vp, sz, vp]
    L.blsgpu_last_stage_ms.argtypes = [vp, vp, C.c_int]
    L.blsgpu_stage_name.restype = C.c_char_p
    L.blsgpu_stage_name.argtypes = [C.c_int]
    L.blsgpu_last_launches.argtypes = [vp]
    L.blsgpu_test_fp.argtypes = [vp, C.c_int, vp, vp, sz, vp]
    L.blsgpu_test_field.argtypes = [vp, C.c_int, vp, sz, sz, vp, sz]
    L.blsgpu_imad_peak.restype = C.c_double
    L.blsgpu_imad_peak.argtypes = [vp, C.c_int]
    L.blsgpu_fpmul_peak.restype = C.c_double
    L.blsgpu_fpmul_peak.argtypes = [vp, C.c_int, C.c_int]
    L.blsgpu_make_sets.argtypes = [vp, C.c_uint64, sz, sz, vp, C.c_int]
    L.blsgpu_msm_make_inputs.argtypes = [vp, C.c_uint64, sz, vp, vp]
    _lib = L
    return L
