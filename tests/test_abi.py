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
