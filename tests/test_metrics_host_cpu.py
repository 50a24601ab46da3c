"""CPU tests of the host side of the GPU metrics (metrics.py, evaluate.py): the resampling filter, the resampled lengths
and the band table against oracle/metrics.py, the scp pairing of the evaluation entry point, and the missing-GPU error."""
import numpy as np
import pytest
import torch

from oracle import metrics as ORC
from urgent2026_challenge_track1_b200 import metrics as MET

RATES = (8000, 16000, 22050, 24000, 32000, 44100, 48000)


@pytest.mark.parametrize("fs", RATES)
def test_resample_taps_match_the_oracle(fs):
    up, down = MET.resample_ratio(fs)
    h = MET.resample_taps(up, down)
    ho = ORC._resample_window_oct(ORC.FS, fs)
    ho = ho / np.sum(ho) * up                                        # resample_poly's normalisation and gain
    assert h.shape == ho.shape
    assert np.abs(h - ho).max() <= 1e-12
    P = MET.polyphase(h, up)
    assert P.shape == (up, -(-h.size // up))
    for ph in (0, up - 1):
        assert np.array_equal(P[ph, : len(h[ph::up])], h[ph::up]) and not P[ph, len(h[ph::up]):].any()


def test_long_filters_have_the_expected_size():
    assert MET.resample_taps(*MET.resample_ratio(44100)).size == 31947
    assert MET.resample_taps(*MET.resample_ratio(22050)).size == 31947


@pytest.mark.parametrize("fs", RATES)
def test_resampled_lengths_match_the_oracle(fs):
    up, down = MET.resample_ratio(fs)
    for n in (1, 255, 4001, fs + 7):
        assert MET.resampled_length(n, up, down) == ORC.resample_oct(np.ones(n), ORC.FS, fs).size


def test_band_table_matches_thirdoct():
    lo, hi = MET.third_octave_bands()
    obm, _ = ORC.thirdoct(ORC.FS, ORC.NFFT, ORC.NUMBAND, ORC.MINFREQ)
    f = np.arange(obm.shape[1])
    for k in range(ORC.NUMBAND):
        assert np.array_equal(obm[k], ((f >= lo[k]) & (f < hi[k])).astype(float))


def test_frame_count_matches_the_framing():
    for n in (0, 256, 257, 384, 385, 10000):
        assert MET.n_frames(n) == len(range(0, n - 256, 128))


def _wav(path, n, fs):
    from urgent2026_challenge_track1_b200.inference import _write_wav
    _write_wav(str(path), np.zeros(n, np.float32), fs)
    return str(path)


def _scp(path, entries):
    path.write_text("".join(f"{u} {p}\n" for u, p in entries))
    return str(path)


def test_pairing_follows_the_estimate_list(tmp_path):
    from urgent2026_challenge_track1_b200 import evaluate as EV
    r = [(u, _wav(tmp_path / f"r_{u}.wav", 800 + i, 16000)) for i, u in enumerate("abc")]
    e = [(u, _wav(tmp_path / f"e_{u}.wav", 800 + i, 16000)) for i, u in enumerate("abc")]
    pairs = EV.pair_scps(_scp(tmp_path / "ref.scp", r), _scp(tmp_path / "inf.scp", [e[2], e[0]]))
    assert [(p[0], p[3], p[4]) for p in pairs] == [("c", 802, 16000), ("a", 800, 16000)]


def test_pairing_rejects_a_missing_uid(tmp_path):
    from urgent2026_challenge_track1_b200 import evaluate as EV
    ref = _scp(tmp_path / "ref.scp", [("a", _wav(tmp_path / "r.wav", 800, 16000))])
    inf = _scp(tmp_path / "inf.scp", [("a", _wav(tmp_path / "a.wav", 800, 16000)), ("zz", _wav(tmp_path / "z.wav", 800, 16000))])
    with pytest.raises(ValueError, match="'zz'"):
        EV.pair_scps(ref, inf)


@pytest.mark.parametrize("what", ["length", "rate"])
def test_pairing_rejects_a_mismatched_pair(tmp_path, what):
    from urgent2026_challenge_track1_b200 import evaluate as EV
    ref = _scp(tmp_path / "ref.scp", [("u1", _wav(tmp_path / "r.wav", 800, 16000))])
    n, fs = (801, 16000) if what == "length" else (800, 8000)
    inf = _scp(tmp_path / "inf.scp", [("u1", _wav(tmp_path / "e.wav", n, fs))])
    with pytest.raises(ValueError, match="'u1'"):
        EV.pair_scps(ref, inf)


def test_main_rejects_before_touching_the_device(tmp_path, monkeypatch):
    from urgent2026_challenge_track1_b200 import evaluate as EV
    monkeypatch.setattr(EV, "score", lambda *a, **k: pytest.fail("scored despite a bad list"))
    ref = _scp(tmp_path / "ref.scp", [("u1", _wav(tmp_path / "r.wav", 800, 16000))])
    inf = _scp(tmp_path / "inf.scp", [("u1", _wav(tmp_path / "e.wav", 700, 16000))])
    args = EV.build_parser().parse_args(["--ref_scp", ref, "--inf_scp", inf, "--output_dir", str(tmp_path / "out")])
    with pytest.raises(ValueError, match="'u1'"):
        EV.main(args)


@pytest.mark.skipif(torch.cuda.is_available(), reason="checks the no-GPU failure mode")
@pytest.mark.parametrize("metric", ["estoi", "sdr"])
def test_metrics_without_a_gpu_raise(metric):
    from urgent2026_challenge_track1_b200 import NativeLibraryError
    x = torch.zeros(1, 16000)
    with pytest.raises(NativeLibraryError):
        if metric == "estoi":
            MET.estoi(x, x, [16000], 16000)
        else:
            MET.sdr(x, x, [16000])
