"""ctypes binding of the C ABI in ``include/radiorust_b200.h``.

The shared library is built in-tree by ``radiorust_b200.build``.  There is no
CPU fallback: if the library is missing, loading fails loudly.
"""
from __future__ import annotations

import ctypes as C
import os

HERE = os.path.dirname(os.path.abspath(__file__))
# RR_LIB_PATH: load another build of the same library (A/B measurements of kernel variants)
LIB_PATH = os.environ.get("RR_LIB_PATH") or os.path.join(HERE, "lib", "libradiorust_b200.so")

RR_OK = 0
RR_ERR_INVALID = -1
RR_ERR_CUDA = -2
RR_ERR_UNSUPPORTED = -3
RR_ERR_NOMEM = -4
RR_ERR_CAPACITY = -5

RR_C32, RR_C64 = 0, 1
(RR_STAGE_FREQSHIFT, RR_STAGE_FILTER, RR_STAGE_DOWNSAMPLE, RR_STAGE_UPSAMPLE, RR_STAGE_FMDEMOD, RR_STAGE_GAIN,
 RR_STAGE_FOURIER, RR_STAGE_FMMOD, RR_STAGE_RECHUNK, RR_STAGE_OVERLAP) = range(1, 11)
RR_WINDOW_KAISER, RR_WINDOW_RECTANGULAR, RR_WINDOW_CUSTOM = 0, 1, 2

FREQ_RESP_FN = C.CFUNCTYPE(None, C.c_void_p, C.c_int64, C.c_double, C.POINTER(C.c_double), C.POINTER(C.c_double))
WINDOW_FN = C.CFUNCTYPE(C.c_double, C.c_void_p, C.c_double)


class StageDesc(C.Structure):
    _fields_ = [
        ("kind", C.c_int32),
        ("window_kind", C.c_int32),
        ("precision", C.c_double),
        ("shift", C.c_double),
        ("freq_resp", FREQ_RESP_FN),
        ("freq_resp_user", C.c_void_p),
        ("window_beta", C.c_double),
        ("window_fn", WINDOW_FN),
        ("window_user", C.c_void_p),
        ("output_chunk_len", C.c_uint64),
        ("output_rate", C.c_double),
        ("bandwidth", C.c_double),
        ("quality", C.c_double),
        ("deviation", C.c_double),
        ("gain", C.c_double),
        ("center_dc", C.c_int32),
        ("chunk_count", C.c_int32),
    ]


class ChainDesc(C.Structure):
    _fields_ = [
        ("dtype", C.c_int32),
        ("n_streams", C.c_int32),
        ("n_stages", C.c_int32),
        ("reserved", C.c_int32),
        ("stages", C.POINTER(StageDesc)),
    ]


# name -> (restype, argtypes).  Every symbol include/radiorust_b200.h declares.
_P = C.c_void_p
_SZ = C.c_size_t
_D = C.c_double
_I = C.c_int
SIGNATURES = {
    "rr_last_error": (C.c_char_p, []),
    "rr_version": (_I, [C.POINTER(_I), C.POINTER(_I)]),
    "rr_kernel_launch_count": (C.c_uint64, []),
    "rr_ctx_create": (_I, [_I, C.POINTER(_P)]),
    "rr_ctx_destroy": (_I, [_P]),
    "rr_ctx_device": (_I, [_P]),
    "rr_pool_create": (_I, [_P, C.POINTER(_P)]),
    "rr_pool_destroy": (_I, [_P]),
    "rr_pool_get": (_I, [_P, _SZ, C.POINTER(_P), C.POINTER(_SZ)]),
    "rr_pool_put": (_I, [_P, _P]),
    "rr_pool_trim": (_I, [_P]),
    "rr_pool_stats": (_I, [_P, C.POINTER(C.c_uint64), C.POINTER(C.c_uint64), C.POINTER(C.c_uint64), C.POINTER(C.c_uint64)]),
    "rr_pinned_alloc": (_I, [_P, _SZ, C.POINTER(_P)]),
    "rr_pinned_free": (_I, [_P, _P]),
    "rr_host_register": (_I, [_P, _P, _SZ]),
    "rr_host_unregister": (_I, [_P, _P]),
    "rr_device_alloc": (_I, [_P, _SZ, C.POINTER(_P)]),
    "rr_device_free": (_I, [_P, _P]),
    "rr_ipc_export": (_I, [_P, _P, _P]),
    "rr_ipc_open": (_I, [_P, _P, C.POINTER(_P)]),
    "rr_ipc_close": (_I, [_P, _P]),
    "rr_memcpy_h2d": (_I, [_P, _P, _P, _SZ]),
    "rr_memcpy_d2h": (_I, [_P, _P, _P, _SZ]),
    "rr_metering_level": (_I, [_P, C.c_int32, _P, _SZ, _SZ, _SZ, _I, C.POINTER(_D)]),
    "rr_metering_bandwidth": (_I, [_P, C.c_int32, _P, _SZ, _SZ, _SZ, _I, _D, _D, C.POINTER(_D)]),
    "rr_metering_rescale_energy": (_I, [_P, C.c_int32, _P, _SZ, _SZ, _SZ, _I, _SZ, _P]),
    "rr_bessel_i0": (_D, [_D]),
    "rr_sinc": (_D, [_D]),
    "rr_kaiser_rel_with_beta": (_D, [_D, _D]),
    "rr_kaiser_null_at_bin_to_beta": (_D, [_D]),
    "rr_deemphasis_factor": (None, [_D, _D, C.POINTER(_D), C.POINTER(_D)]),
    "rr_freq_to_ratio": (_I, [_D, _D, _D, C.POINTER(C.c_int64), C.POINTER(C.c_int64)]),
    "rr_design_filter_response": (_I, [FREQ_RESP_FN, _P, C.c_int32, _D, WINDOW_FN, _P, _D, _SZ, C.c_int32, C.POINTER(_D)]),
    "rr_design_downsampler_taps": (_I, [_D, _D, _D, _D, C.POINTER(_SZ), C.POINTER(_D)]),
    "rr_design_upsampler_taps": (_I, [_D, _D, _D, _D, C.POINTER(_SZ), C.POINTER(_D)]),
    "rr_design_fused_rank": (_I, [FREQ_RESP_FN, _P, C.c_int32, _D, WINDOW_FN, _P, _D, _SZ, _D, _D, _D, _D, _I,
                                  C.POINTER(_I), C.POINTER(_D), C.POINTER(_D)]),
    "rr_chain_create": (_I, [_P, C.POINTER(ChainDesc), C.POINTER(_P)]),
    "rr_chain_destroy": (_I, [_P]),
    "rr_chain_set_shift": (_I, [_P, _I, _I, _D]),
    "rr_chain_set_shifts": (_I, [_P, _I, C.POINTER(_D), _I]),
    "rr_chain_get_shift": (_I, [_P, _I, _I, C.POINTER(_D)]),
    "rr_chain_update_filter": (_I, [_P, _I, FREQ_RESP_FN, _P, C.c_int32, _D, WINDOW_FN, _P, _I]),
    "rr_chain_set_deviation": (_I, [_P, _I, _D]),
    "rr_chain_set_gain": (_I, [_P, _I, _D]),
    "rr_chain_set_output_chunk_len": (_I, [_P, _I, _SZ]),
    "rr_chain_samples_lost_count": (C.c_uint64, [_P]),
    "rr_chain_event": (_I, [_P, _I]),
    "rr_chain_max_output": (_SZ, [_P, _D, _SZ, _SZ]),
    "rr_chain_push": (_I, [_P, _D, _SZ, _SZ, _P, _SZ, _P, _SZ, _SZ, C.POINTER(_SZ), C.POINTER(_D)]),
    "rr_chain_push_device": (_I, [_P, _D, _SZ, _SZ, _P, _SZ, _P, _SZ, _SZ, C.POINTER(_SZ), C.POINTER(_D)]),
    "rr_chain_push_shared": (_I, [_P, _D, _SZ, _SZ, _P, _P, _SZ, _SZ, C.POINTER(_SZ), C.POINTER(_D)]),
    "rr_chain_push_shared_device": (_I, [_P, _D, _SZ, _SZ, _P, _P, _SZ, _SZ, C.POINTER(_SZ), C.POINTER(_D)]),
    "rr_chain_push_summed": (_I, [_P, _D, _SZ, _SZ, _P, _SZ, _P, _SZ, C.POINTER(_SZ), C.POINTER(_D)]),
    "rr_chain_push_summed_device": (_I, [_P, _D, _SZ, _SZ, _P, _SZ, _P, _SZ, C.POINTER(_SZ), C.POINTER(_D)]),
    "rr_chain_sync": (_I, [_P]),
    "rr_chain_copy_out_async": (_I, [_P, _P, _SZ, _P, _SZ, _SZ]),
    "rr_chain_set_fast_path": (_I, [_P, _I]),
    "rr_chain_set_timing": (_I, [_P, _I]),
    "rr_chain_kernel_time": (_I, [_P, C.POINTER(_D), C.POINTER(_I), C.POINTER(C.c_char_p)]),
    "rr_chain_kernel_breakdown": (C.c_char_p, [_P]),
    "rr_chain_cuda_stream": (_P, [_P]),
    "rr_chain_plan": (C.c_char_p, [_P]),
}

_lib = None


def load() -> C.CDLL:
    """Load the CUDA library (no fallback: raises if it has not been built)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(
            f"{LIB_PATH} is missing: build it with `python -m radiorust_b200.build` "
            "(radiorust_b200 has no CPU fallback)"
        )
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)  # AttributeError if the header and the library disagree
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


class RadiorustError(RuntimeError):
    def __init__(self, code: int, msg: str):
        super().__init__(f"radiorust_b200 error {code}: {msg}")
        self.code = code


def check(code: int) -> None:
    if code != RR_OK:
        msg = load().rr_last_error()
        raise RadiorustError(code, msg.decode() if msg else "")
