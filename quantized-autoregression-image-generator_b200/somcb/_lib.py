"""ctypes binding of libsomcb.so (C-ABI declared in include/somcb.h).

The library is built in-tree by ``build.py`` (nvcc, sm_100a).  There is NO fallback: if the
shared object is missing, or a call is made without a CUDA device, this module raises.
"""
import ctypes
import os
from ctypes import c_char_p, c_double, c_float, c_int, c_int64, c_size_t, c_void_p, POINTER

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libsomcb.so")

SOM_BMU_AUTO, SOM_BMU_FFMA, SOM_BMU_TC3X, SOM_BMU_TC_TF32, SOM_BMU_TC_F16 = 0, 1, 2, 3, 4

# name -> (restype, argtypes); mirrors include/somcb.h one to one
SIGNATURES = {
    "som_version": (c_int, []),
    "som_last_error": (c_char_p, []),
    "som_launch_count": (ctypes.c_uint64, []),
    "som_device_info": (c_int, [POINTER(c_int), POINTER(c_int), POINTER(c_int)]),
    "som_prepare_codebook_f32": (c_int, [c_void_p, c_int, c_int, c_void_p, c_void_p]),
    "som_prepare_codebook_w16": (c_int, [c_void_p, c_int, c_int, c_int, c_void_p, c_void_p]),
    "som_bmu_workspace_bytes": (c_size_t, [c_int64, c_int, c_int, c_int]),
    "som_bmu_pick_variant": (c_int, [c_int64, c_int, c_int]),
    "som_bmu_split_mode": (c_int, [c_int64, c_int, c_int]),
    "som_bmu_nchw_f32": (c_int, [c_void_p, c_int64, c_int, c_int, c_int, c_int, c_int,
                                 c_void_p, c_void_p, c_int, c_int64, c_void_p, c_void_p,
                                 c_void_p, c_size_t, c_int, c_void_p]),
    "som_bmu_can_stage": (c_int, [c_int64, c_int, c_int, c_int]),
    "som_bmu_stage_nchw_f32": (c_int, [c_void_p, c_int64, c_int, c_int, c_int, c_int, c_int,
                                       c_void_p, c_void_p, c_int, c_int64, c_void_p, c_void_p, c_void_p,
                                       c_void_p, c_size_t, c_int, c_void_p]),
    "som_bmu_f16_native": (c_int, [c_int64, c_int, c_int, c_int]),
    "som_bmu_stage_nchw_f16": (c_int, [c_void_p, c_int64, c_int, c_int, c_int, c_int, c_int,
                                       c_void_p, c_void_p, c_int, c_int64, c_void_p, c_void_p, c_void_p,
                                       c_void_p, c_size_t, c_int, c_void_p]),
    "som_bmu_stage_nchw_bf16": (c_int, [c_void_p, c_int64, c_int, c_int, c_int, c_int, c_int,
                                        c_void_p, c_void_p, c_int, c_int64, c_void_p, c_void_p, c_void_p,
                                        c_void_p, c_size_t, c_int, c_void_p]),
    "som_convert_f16_f32": (c_int, [c_void_p, c_int64, c_void_p, c_void_p]),
    "som_convert_bf16_f32": (c_int, [c_void_p, c_int64, c_void_p, c_void_p]),
    "som_bmu_w16_workspace_bytes": (c_size_t, [c_int64, c_int, c_int, c_int]),
    "som_bmu_w16_nchw": (c_int, [c_void_p, c_int, c_int64, c_int, c_int, c_int, c_int, c_int, c_void_p, c_int,
                                 c_void_p, c_int, c_int64, c_void_p, c_void_p, c_void_p, c_size_t, c_int, c_void_p]),
    "som_bmu_flat_f32": (c_int, [c_void_p, c_int64, c_int, c_void_p, c_void_p, c_int, c_int64, c_void_p, c_void_p,
                                 c_void_p, c_size_t, c_int, c_void_p]),
    "som_backward_nchw_f32": (c_int, [c_void_p, c_int64, c_int, c_int, c_int, c_int, c_int, c_void_p, c_int,
                                      c_void_p, c_void_p, c_size_t, c_void_p]),
    "som_merge_candidates": (c_int, [c_void_p, c_void_p, c_int, c_int64, c_void_p, c_void_p, c_void_p]),
    "som_histogram_i64": (c_int, [c_void_p, c_int64, c_int, c_void_p, c_void_p]),
    "som_filter_f32": (c_int, [c_void_p, c_void_p, c_int, c_int, c_double, c_float, c_void_p]),
    "som_filter_workspace_bytes": (c_size_t, [c_int, c_int, c_double]),
    "som_filter_half_width": (c_int, [c_int, c_double]),
    "som_filter_ws_f32": (c_int, [c_void_p, c_void_p, c_int, c_int, c_double, c_float, c_void_p, c_size_t,
                                  c_void_p]),
    "som_accumulate_workspace_bytes": (c_size_t, [c_int64, c_int, c_int]),
    "som_accumulate_nchw_f32": (c_int, [c_void_p, c_int64, c_int, c_int, c_int, c_int, c_int,
                                        c_void_p, c_void_p, c_int, c_void_p, c_void_p, c_void_p,
                                        c_void_p, c_size_t, c_void_p]),
    "som_accumulate_packed_nchw_f32": (c_int, [c_void_p, c_int64, c_int, c_int, c_int, c_int, c_int,
                                               c_void_p, c_void_p, c_int, c_void_p, c_void_p, c_size_t, c_void_p]),
    "som_adam_dp_f32": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_int64, c_int, c_double, c_double,
                                c_double, c_double, c_void_p, c_void_p, c_void_p, c_void_p]),
    "som_step_small_workspace_bytes": (c_size_t, [c_int64, c_int, c_int, c_double]),
    "som_step_small_f32": (c_int, [c_void_p, c_int64, c_int, c_int, c_int, c_int, c_int, c_void_p, c_void_p, c_void_p,
                                   c_int, c_double, c_double, c_double, c_double, c_double, c_void_p, c_void_p, c_void_p,
                                   c_void_p, c_size_t, c_void_p]),
    "som_peer_signal_bytes": (c_size_t, []),
    "som_peer_allreduce_f32": (c_int, [c_void_p, c_int64, c_void_p, c_void_p, c_int, c_int, c_void_p, c_int, c_void_p]),
    "som_peer_reduce_rows_f32": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int, c_void_p, c_void_p,
                                         c_int, c_int, c_void_p, c_int, c_void_p]),
    "som_peer_reduce_filter_rows_f32": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int, c_double, c_float,
                                                c_void_p, c_void_p, c_void_p, c_int, c_int, c_void_p, c_int, c_void_p,
                                                c_size_t, c_void_p]),
    "som_peer_bcast_rows_f32": (c_int, [c_void_p, c_void_p, c_int64, c_int64, c_int, c_int, c_void_p, c_int,
                                        c_void_p]),
    "som_peer_adam_slice_f32": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int64, c_int64, c_int,
                                        c_double, c_double, c_double, c_double, c_void_p, c_void_p, c_void_p,
                                        c_int, c_int, c_void_p, c_int, c_void_p]),
    "som_quantize_nchw_f32": (c_int, [c_void_p, c_void_p, c_int, c_int64, c_int, c_int, c_int,
                                      c_int, c_int, c_void_p, c_void_p]),
    "som_quantize_nchw_b16": (c_int, [c_void_p, c_void_p, c_int, c_int64, c_int, c_int, c_int,
                                      c_int, c_int, c_void_p, c_void_p]),
    "som_adam_f32": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_int64, c_double, c_double,
                             c_double, c_double, c_int64, c_void_p]),
    "som_adam_devstep_f32": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_int64, c_double, c_double,
                                     c_double, c_double, c_void_p, c_void_p]),
    "som_gather_rows_f32": (c_int, [c_void_p, c_int, c_void_p, c_int64, c_void_p, c_void_p]),
    "som_gather_rows_b16": (c_int, [c_void_p, c_int, c_void_p, c_int64, c_void_p, c_void_p]),
    "som_assemble_tokens_i64": (c_int, [c_void_p, c_void_p, c_int64, c_int, c_int, c_int64, c_int64, c_int,
                                        c_void_p, c_void_p, c_void_p]),
}

_lib = None


class SomError(RuntimeError):
    """Non-zero return from libsomcb (negative: SOM_E_*, positive: cudaError_t)."""

    def __init__(self, fn, code, msg):
        super().__init__(f"{fn} failed with code {code}: {msg}")
        self.code = code


def load():
    """Load libsomcb.so once and attach the prototypes.  Raises if it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(
            f"libsomcb.so not found at {LIB_PATH}. Build it with "
            "`python quantized-autoregression-image-generator_b200/build.py` "
            "(or __graft_entry__.build()); there is no CPU fallback.")
    lib = ctypes.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)          # AttributeError if the symbol is not exported
        fn.restype = res
        fn.argtypes = args
    from . import SOM_ABI_VERSION
    got = lib.som_version()
    if got != SOM_ABI_VERSION:
        raise RuntimeError(f"libsomcb ABI version {got} != expected {SOM_ABI_VERSION}; rebuild")
    _lib = lib
    return lib


def check(fn_name, rc):
    if rc != 0:
        msg = load().som_last_error()
        raise SomError(fn_name, rc, msg.decode("utf-8", "replace") if msg else "")
