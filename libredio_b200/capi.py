"""ctypes binding of include/libredio_cuda.h -- the same C ABI the Rust FFI crate (rust/libredio-cuda-sys)
and the C++ kpn blocks (kpn/gpu_blocks.hpp) bind.  PyTorch appears here only as the owner of device memory
and streams; every computation goes through libredio_cuda.so.  There is NO CPU fallback: a missing
library or a missing GPU raises.
"""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libredio_cuda.so")

OK, ERR_INVALID, ERR_CUDA, ERR_UNSUPPORTED, ERR_NOMEM, ERR_CAPACITY, ERR_ODD_LENGTH, ERR_LENGTH = range(8)
WINDOW_NONE, WINDOW_HANN = 0, 1


class LrcError(RuntimeError):
    def __init__(self, status: int, what: str, detail: str):
        super().__init__(f"{what}: status {status} ({detail})")
        self.status = status


class OokPacket(C.Structure):
    _fields_ = [("stream", C.c_uint32), ("proto", C.c_uint32), ("seq", C.c_uint32), ("nbits", C.c_uint32),
                ("bits", C.c_uint8 * 40)]


_vp, _sz, _i, _u8p, _fp = C.c_void_p, C.c_size_t, C.c_int, C.c_void_p, C.c_void_p
_pp = C.POINTER(C.c_void_p)
_szp = C.POINTER(C.c_size_t)

# name -> (restype, argtypes); every symbol include/libredio_cuda.h declares
SIGNATURES = {
    "lrc_version": (_i, []),
    "lrc_strerror": (C.c_char_p, [_i]),
    "lrc_last_error": (C.c_char_p, []),
    "lrc_ctx_create": (_i, [_i, _pp]),
    "lrc_ctx_destroy": (_i, [_vp]),
    "lrc_ctx_sync": (_i, [_vp]),
    "lrc_ctx_sm_count": (_i, [_vp, C.POINTER(_i)]),
    "lrc_ctx_numa_node": (_i, [_vp, C.POINTER(_i), C.POINTER(_i)]),
    "lrc_ctx_bind_thread": (_i, [_vp, C.POINTER(_i)]),
    "lrc_host_alloc": (_i, [_vp, _sz, _pp]),
    "lrc_host_free": (_i, [_vp, _vp]),
    "lrc_dev_alloc": (_i, [_vp, _sz, _pp]),
    "lrc_dev_free": (_i, [_vp, _vp]),
    "lrc_dev_memset": (_i, [_vp, _vp, _i, _sz, _vp]),
    "lrc_stream_create": (_i, [_vp, _pp]),
    "lrc_stream_destroy": (_i, [_vp, _vp]),
    "lrc_stream_sync": (_i, [_vp, _vp]),
    "lrc_event_create": (_i, [_vp, _pp]),
    "lrc_event_destroy": (_i, [_vp, _vp]),
    "lrc_event_record": (_i, [_vp, _vp, _vp]),
    "lrc_event_sync": (_i, [_vp, _vp]),
    "lrc_copy_h2d_async": (_i, [_vp, _vp, _vp, _sz, _vp]),
    "lrc_copy_d2h_async": (_i, [_vp, _vp, _vp, _sz, _vp]),
    "lrc_copy_to_host": (_i, [_vp, _vp, _vp, _sz]),
    "lrc_unpack_u8_cf32": (_i, [_vp, _u8p, _sz, _fp, _vp]),
    "lrc_fir_create": (_i, [_vp, _fp, _i, _i, _pp]),
    "lrc_fir_destroy": (_i, [_vp]),
    "lrc_fir_out_len": (_sz, [_vp, _sz]),
    "lrc_fir_run_cf32": (_i, [_vp, _fp, _sz, _sz, _sz, _fp, _sz, _vp]),
    "lrc_fir_run_u8": (_i, [_vp, _u8p, _sz, _sz, _sz, _fp, _sz, _vp]),
    "lrc_fir_stream_create": (_i, [_vp, _sz, _sz, _i, _pp]),
    "lrc_fir_stream_destroy": (_i, [_vp]),
    "lrc_fir_stream_push": (_i, [_vp, _vp, _sz, _sz, _fp, _sz, _szp, _vp]),
    "lrc_fft_create": (_i, [_vp, _i, _i, _pp]),
    "lrc_fft_destroy": (_i, [_vp]),
    "lrc_fft_run": (_i, [_vp, _fp, _fp, _sz, _vp]),
    "lrc_fft_run_host": (_i, [_vp, _fp, _fp, _sz]),
    "lrc_rfft_create": (_i, [_vp, _i, _i, _pp]),
    "lrc_rfft_destroy": (_i, [_vp]),
    "lrc_rfft_run": (_i, [_vp, _fp, _fp, _sz, _vp]),
    "lrc_rfft_run_host": (_i, [_vp, _fp, _fp, _sz]),
    "lrc_psd_create": (_i, [_vp, _i, _i, _pp]),
    "lrc_psd_set_window": (_i, [_vp, _fp]),
    "lrc_psd_destroy": (_i, [_vp]),
    "lrc_psd_run": (_i, [_vp, _fp, _sz, _sz, _fp, _vp]),
    "lrc_psdpng_rows": (_i, [_vp, _vp, _sz, _i, _i, _i, _i, _fp, _szp, _vp]),
    "lrc_chain_create": (_i, [_vp, _fp, _i, _i, _i, _i, _pp]),
    "lrc_chain_destroy": (_i, [_vp]),
    "lrc_chain_frames": (_sz, [_vp, _sz]),
    "lrc_chain_kind": (_i, [_vp]),
    "lrc_chain_run": (_i, [_vp, _fp, _sz, _sz, _fp, _szp, _vp]),
    "lrc_chain_run_u8": (_i, [_vp, _u8p, _sz, _sz, _fp, _szp, _vp]),
    "lrc_chain_run_host": (_i, [_vp, _fp, _sz, _sz, _fp, _szp]),
    "lrc_chain_run_host_u8": (_i, [_vp, _u8p, _sz, _sz, _fp, _szp]),
    "lrc_fastfir_create": (_i, [_vp, _fp, _sz, _sz, _pp]),
    "lrc_fastfir_destroy": (_i, [_vp]),
    "lrc_fastfir_nfft": (_sz, [_vp]),
    "lrc_fastfir_out_len": (_sz, [_vp, _sz, _i]),
    "lrc_fastfir_run": (_i, [_vp, _fp, _sz, _fp, _i, _szp, _vp]),
    "lrc_fmdemod_run": (_i, [_vp, _fp, _sz, _sz, _sz, _fp, _fp, _sz, _vp]),
    "lrc_resampler_create": (_i, [_vp, C.c_double, _sz, _sz, _pp]),
    "lrc_resampler_destroy": (_i, [_vp]),
    "lrc_resampler_reset": (_i, [_vp]),
    "lrc_resampler_get_taps": (_i, [_vp, _vp, _sz, _szp, C.POINTER(_i), C.POINTER(_i)]),
    "lrc_resampler_next_out_len": (_sz, [_vp, _sz]),
    "lrc_resampler_process": (_i, [_vp, _fp, _sz, _sz, _fp, _sz, _szp, _vp]),
    "lrc_resampler_process_host": (_i, [_vp, _fp, _sz, _fp, _sz, _szp]),
    "lrc_fmrx_create": (_i, [_vp, _fp, _i, _i, C.c_double, _sz, _sz, _pp]),
    "lrc_fmrx_destroy": (_i, [_vp]),
    "lrc_fmrx_reset": (_i, [_vp]),
    "lrc_fmrx_is_fused": (_i, [_vp]),
    "lrc_fmrx_next_out_len": (_sz, [_vp, _sz]),
    "lrc_fmrx_push": (_i, [_vp, _u8p, _sz, _sz, _fp, _sz, _szp, _vp]),
    "lrc_ook_create": (_i, [_vp, _sz, _sz, C.c_uint, _sz, _sz, _pp]),
    "lrc_ook_destroy": (_i, [_vp]),
    "lrc_ook_decode": (_i, [_vp, _u8p, _sz, _vp]),
    "lrc_ook_fetch_packets": (_i, [_vp, _vp, _sz, _szp]),
    "lrc_ook_debug_ptrs": (_i, [_vp, _pp, _pp, _pp, _pp]),
    "lrc_ook_stream_create": (_i, [_vp, _sz, _sz, C.c_uint, _sz, _sz, _sz, _pp]),
    "lrc_ook_stream_destroy": (_i, [_vp]),
    "lrc_ook_stream_reset": (_i, [_vp]),
    "lrc_ook_stream_push": (_i, [_vp, _u8p, _sz, _sz, _vp]),
    "lrc_ook_stream_fetch_packets": (_i, [_vp, _vp, _sz, _szp]),
    "lrc_ook_stream_debug_ptrs": (_i, [_vp, _pp, _pp, _pp, _pp]),
    "lrc_eat": (_i, [_vp, _sz, _vp, _sz, _vp]),
    "lrc_ook_envelope_table": (_i, [_vp, _fp, _vp]),
    "lrc_gather_create": (_i, [_vp, _i, _i, _sz, _i, _pp]),
    "lrc_gather_create_host": (_i, [_vp, _i, _i, _sz, _i, C.c_char_p, _i, _pp]),
    "lrc_gather_destroy": (_i, [_vp]),
    "lrc_gather_wait_host": (_i, [_vp, _i, C.c_uint]),
    "lrc_gather_set_root": (_i, [_vp, _i]),
    "lrc_gather_handle_bytes": (_sz, []),
    "lrc_gather_export": (_i, [_vp, _vp, _sz]),
    "lrc_gather_connect": (_i, [_vp, _vp]),
    "lrc_gather_connect_local": (_i, [_vp, _pp]),
    "lrc_gather_push": (_i, [_vp, _i, _vp, _vp]),
    "lrc_gather_wait_sent": (_i, [_vp, _i, _vp]),
    "lrc_gather_wait": (_i, [_vp, _i, _vp]),
    "lrc_gather_buffer": (_i, [_vp, _i, _pp, _szp]),
}

_lib = None


def load() -> C.CDLL:
    """dlopen libredio_cuda.so and type every entry point.  Raises if the library was not built."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise ImportError(
                f"{LIB_PATH} is missing: build it with `python -m libredio_b200.build` "
                "(there is no CPU fallback)")
        lib = C.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(lib, name)          # AttributeError if the symbol is not exported
            fn.restype = res
            fn.argtypes = args
        _lib = lib
    return _lib


def check(status: int, what: str) -> None:
    if status != OK:
        lib = load()
        detail = lib.lrc_last_error().decode() or lib.lrc_strerror(status).decode()
        raise LrcError(status, what, detail)
