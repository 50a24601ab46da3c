"""ctypes binding of libbsrnn_b200.so (the C ABI declared in include/bsrnn_b200.h).

The product path has NO CPU fallback: if the shared library is missing, or the device is not sm_100, every op
raises.  Build with ``./build.sh`` (or ``__graft_entry__.build()``); the .so is kept in-tree under ``_C/``.
"""
from __future__ import annotations

import ctypes as C
import os

import numpy as np
import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "_C", "libbsrnn_b200.so")

c_void_p, c_int, c_long, c_float, c_double = C.c_void_p, C.c_int, C.c_long, C.c_float, C.c_double

# name -> argtypes (restype is int for all but bsrnn_last_error)
PROTOTYPES = {
    "bsrnn_abi_version": [],
    "bsrnn_device_check": [],
    "bsrnn_launch_count": [c_int],
    "bsrnn_fft_twiddle": [c_void_p, c_int, c_void_p],
    "bsrnn_stft_fwd": [c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int, c_float, c_float,
                       c_void_p],
    "bsrnn_istft_fwd": [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int,
                        c_int, c_int, c_float, c_float, c_void_p],
    "bsrnn_gn_stats": [c_void_p, c_void_p, c_int, c_long, c_int, c_long, c_void_p],
    "bsrnn_band_stats": [c_void_p, c_void_p, c_int, c_int, c_long, c_void_p, c_void_p, c_int, c_void_p],
    "bsrnn_gn_finalize": [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_void_p,
                          c_float, c_int, c_void_p],
    "bsrnn_gemm_f32": [c_void_p, c_int, c_int, c_int, c_void_p],
    "bsrnn_blstm_recurrence_f32": [c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_long, c_long,
                                   c_long, c_long, c_void_p],
    "bsrnn_norm_cast_kb8": [c_void_p, c_void_p, c_void_p, c_void_p, c_long, c_int, c_int, c_int, c_int, c_int, c_int,
                            c_long, c_long, c_long, c_long, c_long, c_int, c_void_p],
    "bsrnn_norm_cast_kb8_ones": [c_void_p, c_void_p, c_void_p, c_void_p, c_long, c_int, c_int, c_int, c_int, c_int,
                                 c_int, c_long, c_long, c_long, c_long, c_long, c_int, c_int, c_void_p],
    "bsrnn_gemm_tc": [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int, c_long,
                      c_int, c_int, c_long, c_int, c_int, c_long, c_long, c_long, c_long, c_void_p],
    "bsrnn_gemm_tc_ex": [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int, c_long,
                         c_int, c_int, c_long, c_int, c_int, c_long, c_long, c_long, c_long, c_int, c_int, c_void_p],
    "bsrnn_gemm_tc_grouped": [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_long,
                              c_int, c_long, c_int, c_int, c_long, c_long, c_long, c_long, c_void_p],
    "bsrnn_gemm_tc_limit_ctas": [c_int],
    "bsrnn_blstm_fused_train_tc": [c_int, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_long, c_void_p, c_void_p, c_void_p,
                                   c_void_p, c_int, c_int, c_int, c_int, c_int, c_void_p, c_void_p],
    "bsrnn_blstm_fused_train_scratch_bytes": [c_int, c_int],
    "bsrnn_band_norm_cast_kb8": [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int,
                                 c_long, c_int, c_int, c_int, c_void_p],
    "bsrnn_lstm_step_tc": [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_long, c_void_p],
    "bsrnn_blstm_step_tc": [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p,
                            c_int, c_int, c_int, c_int, c_long, c_void_p],
    "bsrnn_blstm_recurrence_tc": [c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_void_p],
    "bsrnn_blstm_recurrence_tc_ex": [c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int,
                                     c_void_p],
    "bsrnn_blstm_recurrence_tc_flag": [c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int,
                                       c_void_p, c_void_p],
    "bsrnn_blstm_fused_tc": [c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int, c_void_p, c_void_p],
    "bsrnn_blstm_fused768_tc": [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_long, c_int, c_int, c_int, c_int, c_int,
                                c_void_p, c_void_p],
    "bsrnn_blstm_fused768_max_groups": [],
    "bsrnn_blstm_fused768_train_tc": [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_long, c_void_p, c_void_p, c_void_p,
                                      c_void_p, c_int, c_int, c_int, c_int, c_int, c_void_p, c_void_p],
    "bsrnn_blstm_fused768_train_scratch_bytes": [c_int, c_int],
    "bsrnn_blstm_fused7_tc": [c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int, c_void_p, c_void_p],
    "bsrnn_blstm_fused7_max_groups": [],
    "bsrnn_blstm_fused14_tc": [c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int, c_void_p, c_void_p],
    "bsrnn_blstm_fused14_max_groups": [],
    "bsrnn_blstm_fused_max_groups": [],
    "bsrnn_blstm_fused_sync_bytes": [],
    "bsrnn_blstm_tc_flag_max_groups": [],
    "bsrnn_blstm_tc_sync_bytes": [],
    "bsrnn_blstm_tc_max_clusters": [],
    "bsrnn_blstm_tc_max_pair_clusters": [],
    "bsrnn_debug_set_lstm_schedule": [c_int],
    "bsrnn_blstm_train_fwd_f32": [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_long, c_long,
                                  c_long, c_long, c_void_p],
    "bsrnn_blstm_train_bwd_f32": [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int,
                                  c_long, c_long, c_long, c_long, c_void_p],
    "bsrnn_grad_sumsq": [c_void_p, c_long, c_void_p, c_void_p],
    "bsrnn_adamw_step": [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_long, c_void_p, c_float, c_float, c_float,
                         c_float, c_float, c_float, c_float, c_int, c_float, c_void_p],
    "bsrnn_adamw_step2": [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_long, c_void_p, c_void_p, c_int, c_float,
                          c_float, c_float, c_float, c_float, c_float, c_float, c_float, c_void_p],
    "bsrnn_blstm_step_train_tc": [c_void_p] * 12 + [c_int, c_int, c_int, c_int, c_long, c_void_p],
    "bsrnn_blstm_bwd_step_tc": [c_void_p] * 16 + [c_int, c_int, c_int, c_int, c_long, c_long, c_int, c_void_p],
    "bsrnn_blstm_train_fwd_tc": [c_void_p] * 8 + [c_int, c_int, c_int, c_int, c_int, c_void_p],
    "bsrnn_blstm_train_bwd_tc": [c_void_p] * 11 + [c_int, c_int, c_int, c_int, c_int, c_int, c_void_p],
    "bsrnn_gemm_tc_scaled": [c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_long, c_int, c_float,
                             c_void_p, c_int, c_int, c_int, c_long, c_long, c_long, c_long, c_void_p],
    "bsrnn_kb8_transpose": [c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int, c_long, c_long, c_void_p],
    "bsrnn_stft_stats_fwd": [c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int, c_float, c_float,
                             c_void_p, c_void_p, c_int, c_void_p],
    "bsrnn_band_split_fwd": [c_void_p] * 10 + [c_int, c_long, c_int, c_int, c_int, c_int, c_long, c_int, c_int, c_void_p],
    "bsrnn_istft_bwd": [c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int, c_void_p],
    "bsrnn_l1_time_fwd_bwd": [c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_float, c_void_p],
    "bsrnn_mrl1_spec_fwd_bwd": [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_float, c_void_p],
    "bsrnn_time_embed": [c_void_p, c_void_p, c_void_p, c_int, c_int, c_void_p],
    "bsrnn_conv5x5_glu": [c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_void_p],
    "bsrnn_euler_step": [c_void_p, c_void_p, c_void_p, c_float, c_long, c_void_p],
    "bsrnn_axpy_complex": [c_void_p, c_void_p, c_void_p, c_float, c_long, c_void_p],
    "bsrnn_complex_mask": [c_void_p, c_void_p, c_void_p, c_void_p, c_float, c_long, c_void_p],
    "bsrnn_mix_conv_scratch_bytes": [c_int, c_int, c_int, c_int],
    "bsrnn_mix_conv": [c_void_p] * 7 + [c_int, c_int, c_int, c_int, c_int, c_void_p],
    "bsrnn_mix_snr_scratch_bytes": [c_int, c_int],
    "bsrnn_mix_snr": [c_void_p] * 7 + [c_int, c_int, c_void_p],
    "bsrnn_mix_quantiles": [c_void_p] * 4 + [c_int, c_int, c_void_p],
    "bsrnn_mix_finish": [c_void_p] * 5 + [c_int, c_int, c_void_p, c_int, c_int, c_void_p],
    "bsrnn_resample_poly": [c_void_p, c_void_p, c_int, c_int, c_void_p, c_int, c_int, c_int, c_void_p, c_void_p, c_int,
                            c_void_p],
    "bsrnn_estoi_compact_scratch_bytes": [c_int, c_int],
    "bsrnn_estoi_compact": [c_void_p] * 3 + [c_int, c_int] + [c_void_p] * 5,
    "bsrnn_estoi_bands": [c_void_p] * 3 + [c_int, c_int] + [c_void_p] * 4 + [c_int, c_void_p],
    "bsrnn_estoi_score": [c_void_p, c_void_p, c_int, c_int, c_void_p, c_void_p, c_void_p],
    "bsrnn_sdr_scratch_bytes": [c_int, c_int],
    "bsrnn_sdr": [c_void_p] * 3 + [c_int, c_int] + [c_void_p] * 3,
}

# mirrors `bsrnn_gemm_desc` (include/bsrnn_b200.h); 144 bytes
GEMM_DESC = np.dtype([
    ("A", "<u8"), ("W", "<u8"), ("bias", "<u8"), ("C", "<u8"), ("scale", "<u8"), ("shift", "<u8"),
    ("a_inner", "<i8"), ("a_outer_stride", "<i8"), ("a_inner_stride", "<i8"),
    ("c_inner", "<i8"), ("c_outer_stride", "<i8"), ("c_inner_stride", "<i8"),
    ("rows_per_sample", "<i8"), ("ss_stride", "<i8"),
    ("M", "<i4"), ("N", "<i4"), ("K", "<i4"), ("k_valid", "<i4"), ("ldw", "<i4"), ("epilogue", "<i4"),
    ("n_store", "<i4"), ("pad_", "<i4"),
])
assert GEMM_DESC.itemsize == 144

EPI_STORE, EPI_TANH, EPI_RESIDUAL, EPI_GLU = 0, 1, 2, 3
TC_F16_ROWS, TC_RESID_F32, TC_TANH_KB8, TC_GLU_F32, TC_F16_KB8 = 0, 1, 2, 3, 4      # bsrnn_gemm_tc epilogues
TC_TANH_F32 = 7
TC_RESID_TMA = 8        # epilogue 1 with the residual rows moved by bulk (TMA) copies through a shared-memory row buffer

_lib = None


class NativeLibraryError(RuntimeError):
    pass


def lib():
    """Load (once) and return the ctypes handle; raises NativeLibraryError if the extension was not built."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise NativeLibraryError(
                f"{LIB_PATH} not found: the CUDA extension is not built (run ./build.sh). "
                "There is no CPU or PyTorch fallback for this path.")
        handle = C.CDLL(LIB_PATH)
        for name, argtypes in PROTOTYPES.items():
            fn = getattr(handle, name)
            fn.argtypes = argtypes
            fn.restype = c_int
        handle.bsrnn_launch_count.restype = C.c_long
        handle.bsrnn_blstm_fused_train_scratch_bytes.restype = C.c_long
        handle.bsrnn_blstm_fused768_train_scratch_bytes.restype = C.c_long
        handle.bsrnn_mix_conv_scratch_bytes.restype = C.c_long
        handle.bsrnn_mix_snr_scratch_bytes.restype = C.c_long
        handle.bsrnn_estoi_compact_scratch_bytes.restype = C.c_long
        handle.bsrnn_sdr_scratch_bytes.restype = C.c_long
        handle.bsrnn_last_error.restype = C.c_char_p
        handle.bsrnn_last_error.argtypes = []
        _lib = handle
    return _lib


def check(rc: int, what: str):
    if rc != 0:
        raise RuntimeError(f"{what} failed (rc={rc}): {lib().bsrnn_last_error().decode()}")


_DEVICE_OK = set()


def require_device():
    if not torch.cuda.is_available():
        raise NativeLibraryError("no CUDA device: the B200 path has no CPU fallback")
    dev = torch.cuda.current_device()
    if dev not in _DEVICE_OK:                          # once per device and process
        check(lib().bsrnn_device_check(), "bsrnn_device_check")
        _DEVICE_OK.add(dev)


def ptr(t):
    """Device pointer of a tensor (or None)."""
    if t is None:
        return None
    return t.data_ptr()


def stream_ptr():
    return torch.cuda.current_stream().cuda_stream


def call(name, *args):
    check(getattr(lib(), name)(*args), name)
