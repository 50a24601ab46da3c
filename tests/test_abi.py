"""CPU tests of the drop-in boundary: libbsrnn_b200.so loads and exports every symbol include/bsrnn_b200.h declares,
the ctypes prototypes cover them, and the product path fails loudly without a GPU (no CPU fallback)."""
import ctypes
import os
import re
import subprocess

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HEADER = os.path.join(ROOT, "include", "bsrnn_b200.h")


def declared_symbols():
    src = open(HEADER).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(bsrnn_[a-z0-9_]+)\s*\(", src)))


@pytest.fixture(scope="module")
def lib_path():
    from urgent2026_challenge_track1_b200 import _lib
    if not os.path.exists(_lib.LIB_PATH):
        subprocess.run(["bash", os.path.join(ROOT, "build.sh")], check=True, cwd=ROOT)
    return _lib.LIB_PATH


def test_header_declares_the_hot_path():
    syms = declared_symbols()
    for need in ("bsrnn_stft_fwd", "bsrnn_istft_fwd", "bsrnn_gemm_f32", "bsrnn_blstm_recurrence_f32", "bsrnn_gemm_tc",
                 "bsrnn_blstm_recurrence_tc", "bsrnn_norm_cast_kb8", "bsrnn_gn_stats", "bsrnn_band_stats",
                 "bsrnn_gn_finalize", "bsrnn_euler_step", "bsrnn_conv5x5_glu", "bsrnn_time_embed", "bsrnn_last_error"):
        assert need in syms


def test_library_exports_every_declared_symbol(lib_path):
    h = ctypes.CDLL(lib_path)
    missing = [s for s in declared_symbols() if not hasattr(h, s)]
    assert not missing, missing
    assert h.bsrnn_abi_version() >= 1


def test_ctypes_prototypes_cover_the_header(lib_path):
    from urgent2026_challenge_track1_b200 import _lib
    protos = set(_lib.PROTOTYPES) | {"bsrnn_last_error"}
    assert set(declared_symbols()) <= protos, set(declared_symbols()) - protos
    _lib.lib()                                      # binds every prototype; raises on a missing symbol


def test_gemm_desc_layout_matches_header():
    from urgent2026_challenge_track1_b200 import _lib
    # 6 pointers + 8 longs + 8 ints (include/bsrnn_b200.h: bsrnn_gemm_desc)
    assert _lib.GEMM_DESC.itemsize == 6 * 8 + 8 * 8 + 8 * 4
    assert _lib.GEMM_DESC.fields["M"][1] == 112 and _lib.GEMM_DESC.fields["rows_per_sample"][1] == 96


@pytest.mark.skipif(torch.cuda.is_available(), reason="checks the no-GPU failure mode")
def test_no_cpu_fallback(lib_path):
    from urgent2026_challenge_track1_b200 import BSRNN_SE, NativeLibraryError
    m = BSRNN_SE(16, 1)
    with pytest.raises(NativeLibraryError):
        m(torch.zeros(1, 4000), torch.tensor([4000]), 16000)


# bsrnn_gemm_tc_ex calls whose epilogue would store outside what include/bsrnn_b200.h promises: (epilogue, n_tiles, BN, ldo,
# n_valid, out_kcores, expected error).  Epilogues 0 and 4 store every column of every N tile.
_OUT_OF_CONTRACT = {
    "f16_rows_last_tile_past_ldo": (0, 2, 64, 120, 120, 0, "epilogue 0 stores"),
    "f16_kb8_last_tile_past_out_kcores": (4, 2, 64, 0, 128, 15, "epilogue 4 stores"),
    "resid_rows_overlap": (1, 1, 208, 192, 196, 0, "n_valid <= ldo"),
    "resid_tma_rows_overlap": (8, 1, 208, 192, 196, 0, "n_valid <= ldo"),
    "tanh_rows_overlap": (7, 1, 64, 40, 48, 0, "n_valid <= ldo"),
    "glu_rows_overlap": (3, 1, 64, 20, 26, 0, "n_valid <= ldo"),
}


@pytest.mark.skipif(torch.cuda.is_available(), reason="on a GPU an accepted call would launch")
@pytest.mark.parametrize("case", sorted(_OUT_OF_CONTRACT))
def test_gemm_tc_rejects_out_of_contract_stores(lib_path, case):
    from urgent2026_challenge_track1_b200 import _lib
    epi, n_tiles, BN, ldo, n_valid, out_kcores, msg = _OUT_OF_CONTRACT[case]
    h = _lib.lib()
    p = 1 << 20                                          # never dereferenced: the call must fail its argument checks
    rc = h.bsrnn_gemm_tc_ex(p, p, None, p, None, 2, n_tiles, 26, BN, epi, ldo, n_valid, out_kcores, 256, 2, 256, 1 << 40, 0, 1,
                            0, 1, 0, None)
    err = h.bsrnn_last_error().decode()
    assert rc != 0 and msg in err, (rc, err)


@pytest.mark.skipif(torch.cuda.is_available(), reason="on a GPU an accepted call would launch")
@pytest.mark.parametrize("ksplit", [1, 4])
def test_gemm_tc_scaled_rejects_overlapping_rows(lib_path, ksplit):
    from urgent2026_challenge_track1_b200 import _lib
    h = _lib.lib()
    p = 1 << 20
    rc = h.bsrnn_gemm_tc_scaled(p, p, None, p, 2, 1, 26, 208, 192, 196, 0.5, None, ksplit, 2, 256, 1 << 40, 0, 1, 0, None)
    err = h.bsrnn_last_error().decode()
    assert rc != 0 and "n_valid <= ldo" in err, (rc, err)


def test_missing_library_raises(monkeypatch, tmp_path):
    from urgent2026_challenge_track1_b200 import _lib
    monkeypatch.setattr(_lib, "_lib", None)
    monkeypatch.setattr(_lib, "LIB_PATH", str(tmp_path / "nope.so"))
    with pytest.raises(_lib.NativeLibraryError):
        _lib.lib()


# Spectral calls the kernels cannot serve: each must fail its argument checks, with its message, before any launch.
_P = 1 << 20                                             # never dereferenced
_SPECTRAL_REJECTS = {
    "stft_L_at_half_n_fft": ("bsrnn_stft_fwd", (_P, None, _P, _P, 1, 80, 160, 80, 0, 1.0, 1.0, None), "stft_fwd: bad dims"),
    "stft_stats_L_at_half_n_fft": ("bsrnn_stft_stats_fwd", (_P, None, _P, _P, 1, 80, 160, 80, 0, 1.0, 1.0, _P, _P, 4, None),
                                   "stft_stats_fwd: bad dims"),
    "stft_prime_97": ("bsrnn_stft_fwd", (_P, None, _P, _P, 1, 1000, 97, 48, 0, 1.0, 1.0, None), "cannot factorise n_fft=97"),
    "stft_stats_prime_101": ("bsrnn_stft_stats_fwd", (_P, None, _P, _P, 1, 1000, 101, 50, 0, 1.0, 1.0, _P, _P, 4, None),
                             "cannot factorise n_fft=101"),
    "istft_prime_194": ("bsrnn_istft_fwd", (_P, None, None, None, _P, _P, 1, 10, 1000, 194, 97, 0, 1.0, 1.0, None),
                        "cannot factorise n_fft=194"),
    "istft_prime_101": ("bsrnn_istft_fwd", (_P, None, None, None, _P, _P, 1, 10, 1000, 101, 50, 0, 1.0, 1.0, None),
                        "cannot factorise n_fft=101"),
    "istft_bwd_prime_97": ("bsrnn_istft_bwd", (_P, _P, _P, 1, 10, 1000, 97, 48, None), "cannot factorise n_fft=97"),
    "istft_bwd_prime_194": ("bsrnn_istft_bwd", (_P, _P, _P, 1, 10, 1000, 194, 97, None), "cannot factorise n_fft=194"),
    "istft_mask_without_resid": ("bsrnn_istft_fwd", (_P, _P, None, None, _P, _P, 1, 10, 1000, 160, 80, 0, 1.0, 1.0, None),
                                 "mask and resid must come together"),
    "mrl1_odd_window": ("bsrnn_mrl1_spec_fwd_bwd", (_P, _P, _P, _P, _P, 1, 1000, 255, 0.5, None),
                        "mrl1_spec_fwd_bwd: bad dims"),
    "mrl1_L_at_half_window": ("bsrnn_mrl1_spec_fwd_bwd", (_P, _P, _P, _P, _P, 1, 128, 256, 0.5, None),
                              "mrl1_spec_fwd_bwd: bad dims"),
    "mrl1_prime_194": ("bsrnn_mrl1_spec_fwd_bwd", (_P, _P, _P, _P, _P, 1, 1000, 194, 0.5, None), "cannot factorise window=194"),
}


@pytest.mark.skipif(torch.cuda.is_available(), reason="on a GPU an accepted call would launch")
@pytest.mark.parametrize("case", sorted(_SPECTRAL_REJECTS))
def test_spectral_calls_reject_what_the_kernels_cannot_serve(lib_path, case):
    from urgent2026_challenge_track1_b200 import _lib
    name, args, msg = _SPECTRAL_REJECTS[case]
    h = _lib.lib()
    rc = getattr(h, name)(*args)
    err = h.bsrnn_last_error().decode()
    assert rc != 0 and msg in err, (rc, err)


# CUDA-core calls the kernels cannot serve: each must fail its argument checks, with its message, before any launch.
# bsrnn_band_split_fwd reads its host channel offsets: bands of 8 channels and, last, one of 224 at N = 256 (over 227 KB), so
# the check must run before the first band's launch.
_C_OFF = (ctypes.c_int32 * 4)(0, 8, 16, 240)
_BS = lambda N, ldo, out_width, out_col: (_P, _P, _P, _P, _P, _P, _P, _P, _P, ctypes.addressof(_C_OFF), 3, 1000, 10, 600, N,
                                          224, ldo, out_width, out_col, None)
_CORE_REJECTS = {
    "band_split_N_not_4": ("bsrnn_band_split_fwd", _BS(198, 600, 200, 0), "multiples of 4"),
    "band_split_out_col_not_4": ("bsrnn_band_split_fwd", _BS(196, 600, 200, 2), "multiples of 4"),
    "band_split_out_width_not_4": ("bsrnn_band_split_fwd", _BS(196, 600, 198, 0), "multiples of 4"),
    "band_split_ldo_not_4": ("bsrnn_band_split_fwd", _BS(196, 602, 200, 0), "multiples of 4"),
    "band_split_wide_band_last": ("bsrnn_band_split_fwd", _BS(256, 768, 256, 0), "band of 224 channels does not fit"),
    "band_cast_cmax_too_large": ("bsrnn_band_norm_cast_kb8", (_P, _P, _P, _P, _P, _P, _P, _P, 3, 1000, 10, 600, 900, None),
                                 "band of 900 channels does not fit"),
    "gn_stats_rows_0": ("bsrnn_gn_stats", (_P, _P, 2, 0, 196, 196, None), "gn_stats: bad arguments"),
    "gn_stats_C_0": ("bsrnn_gn_stats", (_P, _P, 2, 10, 0, 196, None), "gn_stats: bad arguments"),
    "gn_stats_B_neg": ("bsrnn_gn_stats", (_P, _P, -1, 10, 196, 196, None), "gn_stats: bad arguments"),
    "band_stats_T_0": ("bsrnn_band_stats", (_P, _P, 2, 0, 392, _P, _P, 2, None), "band_stats: bad arguments"),
    "gn_finalize_G_0": ("bsrnn_gn_finalize", (_P, _P, _P, None, _P, _P, 0, 196, _P, 1e-5, 1, None), "gn_finalize: bad arguments"),
    "gn_finalize_C_0": ("bsrnn_gn_finalize", (_P, _P, _P, None, _P, _P, 4, 0, _P, 1e-5, 1, None), "gn_finalize: bad arguments"),
    "gn_finalize_G_inner_0": ("bsrnn_gn_finalize", (_P, _P, _P, None, _P, _P, 4, 196, _P, 1e-5, 0, None),
                              "gn_finalize: bad arguments"),
    "conv5x5_T_0": ("bsrnn_conv5x5_glu", (_P, _P, _P, _P, 1, 0, 32, 32, None), "conv5x5_glu: bad arguments"),
    "conv5x5_Fp_0": ("bsrnn_conv5x5_glu", (_P, _P, _P, _P, 1, 4, 0, 32, None), "conv5x5_glu: bad arguments"),
    "conv5x5_F_neg": ("bsrnn_conv5x5_glu", (_P, _P, _P, _P, 1, 4, 32, -1, None), "conv5x5_glu: bad arguments"),
    "blstm_recurrence_seq_inner_0": ("bsrnn_blstm_recurrence_f32", (_P, _P, _P, _P, 4, 3, 8, 0, 3, 1, 1, None),
                                     "blstm_recurrence_f32: bad dims"),
    "blstm_train_fwd_seq_inner_neg": ("bsrnn_blstm_train_fwd_f32", (_P, _P, _P, _P, _P, 4, 3, 8, -1, 3, 1, 1, None),
                                      "blstm_train_fwd_f32: bad dims"),
    "blstm_train_bwd_seq_inner_0": ("bsrnn_blstm_train_bwd_f32", (_P, _P, _P, _P, _P, _P, 4, 3, 8, 0, 3, 1, 1, None),
                                    "blstm_train_bwd_f32: bad dims"),
}


@pytest.mark.skipif(torch.cuda.is_available(), reason="on a GPU an accepted call would launch")
@pytest.mark.parametrize("case", sorted(_CORE_REJECTS))
def test_cuda_core_calls_reject_what_the_kernels_cannot_serve(lib_path, case):
    from urgent2026_challenge_track1_b200 import _lib
    name, args, msg = _CORE_REJECTS[case]
    h = _lib.lib()
    rc = getattr(h, name)(*args)
    err = h.bsrnn_last_error().decode()
    assert rc == 1 and msg in err, (rc, err)
