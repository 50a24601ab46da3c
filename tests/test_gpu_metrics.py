"""ESTOI and SDR on the GPU (csrc/metrics.cu through metrics.py) against oracle/metrics.py: every ESTOI stage against its
oracle function, the final scores at every sample rate, the SDR cases of the f64 reference, the documented divergences for
degenerate input, ragged batches with garbage in their padding, and inference.py -> evaluate.py end to end."""
import os

import numpy as np
import pytest
import torch

from oracle import metrics as ORC
from urgent2026_challenge_track1_b200 import metrics as MET
from urgent2026_challenge_track1_b200.synth import synth_pair

pytestmark = pytest.mark.gpu
dev = torch.device("cuda")
RATES = (8000, 10000, 16000, 22050, 24000, 32000, 44100, 48000)
GARBAGE = 7.5e3


def _speechlike(n, fs, seed, floor_db=-25.0):
    """(clean, noisy) f32: synth_pair plus a broadband floor shared by both (a well-conditioned reference)."""
    c, x = synth_pair(1, n, fs, seed=seed)
    rng = np.random.RandomState(seed)
    fl = rng.randn(n) * float(c.std()) * 10 ** (floor_db / 20)
    return ((c[0].numpy() + fl).astype(np.float32), (x[0].numpy() + fl).astype(np.float32))


def _batch(sigs):
    """Rows padded with garbage to the longest -> (device (B, T) f32, device lengths int32)."""
    T = max(len(s) for s in sigs)
    a = np.full((len(sigs), T), GARBAGE, np.float32)
    for r, s in enumerate(sigs):
        a[r, : len(s)] = s
    return torch.from_numpy(a).to(dev), torch.tensor([len(s) for s in sigs], dtype=torch.int32, device=dev)


def _f64(x):
    return np.asarray(x, np.float64)


def _pairs(fs, seconds=(2.5, 1.7)):
    out = []
    for i, s in enumerate(seconds):
        c, x = _speechlike(int(s * fs), fs, 10 + i)
        out.append((c, x))
    return out


def _stages(pairs, fs):
    ref, lens = _batch([c for c, _ in pairs])
    inf, _ = _batch([x for _, x in pairs])
    return MET.estoi_stages(ref, inf, lens, fs)


# ------------------------------------------------------------------------------------------------ ESTOI stages
@pytest.mark.parametrize("fs", [r for r in RATES if r != 10000])
def test_resampling_matches_resample_oct(fs):
    pairs = _pairs(fs)
    st = _stages(pairs, fs)
    x10, n10 = st["x10"].cpu().numpy(), st["n10"].cpu().numpy()
    for r, (c, _) in enumerate(pairs):
        want = ORC.resample_oct(_f64(c), ORC.FS, fs)
        assert n10[r] == want.size
        assert np.abs(x10[r, : n10[r]] - want).max() <= 2e-7 * np.abs(want).max()
        assert not x10[r, n10[r]:].any()


def _with_silence(fs, seed):
    """A pair whose reference has a stretch 60 dB down: silent frames to drop."""
    c, x = _speechlike(int(2.5 * fs), fs, seed)
    a, b = int(0.8 * fs), int(1.4 * fs)
    c[a:b] *= 1e-3
    x[a:b] *= 1e-3
    return c, x


@pytest.mark.parametrize("fs", [16000, 44100])
def test_silent_frame_removal_matches_the_oracle(fs):
    pairs = [_with_silence(fs, 3), _speechlike(int(1.2 * fs), fs, 4)]
    st = _stages(pairs, fs)
    x10, y10, n10 = st["x10"].cpu().numpy(), st["y10"].cpu().numpy(), st["n10"].cpu().numpy()
    xc, yc, c_len = st["xc"].cpu().numpy(), st["yc"].cpu().numpy(), st["c_len"].cpu().numpy()
    for r in range(len(pairs)):
        wx, wy = ORC.remove_silent_frames(_f64(x10[r, : n10[r]]), _f64(y10[r, : n10[r]]), ORC.DYN_RANGE, ORC.N_FRAME,
                                          ORC.N_FRAME // 2)
        assert c_len[r] == wx.size
        for got, want in ((xc[r], wx), (yc[r], wy)):
            assert np.abs(got[: c_len[r]] - want).max() <= 2e-7 * np.abs(want).max()
            assert not got[c_len[r]:].any()
    assert c_len[0] < n10[0] - 0.5 * ORC.FS                                   # the silent stretch is gone


@pytest.mark.parametrize("fs", [16000, 48000])
def test_band_envelopes_match_the_oracle(fs):
    pairs = [_with_silence(fs, 5), _speechlike(int(1.5 * fs), fs, 6)]
    st = _stages(pairs, fs)
    xc, yc, c_len, tob = st["xc"].cpu().numpy(), st["yc"].cpu().numpy(), st["c_len"].cpu().numpy(), st["tob"].cpu().numpy()
    obm, _ = ORC.thirdoct(ORC.FS, ORC.NFFT, ORC.NUMBAND, ORC.MINFREQ)
    for r in range(len(pairs)):
        for z, sig in enumerate((xc, yc)):
            spec = ORC._stft(_f64(sig[r, : c_len[r]]), ORC.N_FRAME, ORC.NFFT).T
            want = np.sqrt(obm @ np.square(np.abs(spec)))
            got = tob[r, z, :, : want.shape[1]]
            assert want.shape[1] == MET.n_frames(c_len[r]) >= 30
            assert np.linalg.norm(got - want) <= 1e-5 * np.linalg.norm(want)
            assert np.abs(got - want).max() <= 1e-5 * want.max()


@pytest.mark.parametrize("fs", RATES)
def test_estoi_matches_the_oracle_at_every_rate(fs):
    pairs = _pairs(fs)
    c, x = pairs[0]
    pairs.append((c, c + 3.0 * (x - c)))                                      # a worse estimate
    ref, lens = _batch([p[0] for p in pairs])
    inf, _ = _batch([p[1] for p in pairs])
    got = MET.estoi(ref, inf, lens, fs).cpu().numpy()
    want = np.array([ORC.estoi(_f64(a), _f64(b), fs) for a, b in pairs])
    assert np.abs(got - want).max() <= 1e-5, (got, want)
    assert 0.0 < want[2] < want[0] < 1.0


# ------------------------------------------------------------------------------------------------ SDR
def _sdr_cases():
    rng = np.random.RandomState(0)
    x = rng.randn(16000 * 2).astype(np.float32)
    cases = {}
    for snr in (0.0, 10.0, 20.0):
        cases[f"white_{snr:g}dB"] = (x, (x + rng.randn(x.size) * 10 ** (-snr / 20)).astype(np.float32))
    cases["delay_100"] = (x, np.concatenate([np.zeros(100, np.float32), x[:-100]]))
    cases["clamp_plus50"] = (x, 3.0 * x)
    cases["clamp_minus50"] = (x, np.zeros_like(x))
    c, n = _speechlike(300, 16000, 7)
    cases["short_300"] = (c, n)
    c, n = _speechlike(6000, 16000, 5)
    cases["speech_6000"] = (c, n)
    cases["lowpass_4k_floor_-60dB"] = _lowpassed(-60.0)
    return cases


def _lowpassed(floor_db):
    """A 48 kHz reference low-passed at 4 kHz (and its estimate), with a broadband floor floor_db below it or none."""
    from scipy.signal import butter, sosfilt
    fs = 48000
    c, x = synth_pair(1, fs * 2, fs, seed=3)
    c, x = c[0].numpy().astype(np.float64), x[0].numpy().astype(np.float64)
    sos = butter(12, 4000, fs=fs, output="sos")
    c, x = sosfilt(sos, c), sosfilt(sos, x)
    if floor_db is not None:
        f = np.random.RandomState(0).randn(c.size) * c.std() * 10 ** (floor_db / 20)
        c, x = c + f, x + f
    return c.astype(np.float32), x.astype(np.float32)


def test_sdr_matches_the_oracle():
    cases = _sdr_cases()
    names = sorted(cases)
    ref, lens = _batch([cases[k][0] for k in names])
    inf, _ = _batch([cases[k][1] for k in names])
    got = MET.sdr(ref, inf, lens).cpu().numpy()
    for k, g in zip(names, got):
        want = ORC.sdr(_f64(cases[k][0]), _f64(cases[k][1]))
        assert abs(g - want) <= 1e-3, (k, g, want)
    assert got[names.index("clamp_plus50")] == pytest.approx(50.0, abs=1e-9)
    assert got[names.index("clamp_minus50")] == pytest.approx(-50.0, abs=1e-9)


# ------------------------------------------------------------------------------------------------ documented divergences
def test_ill_conditioned_reference_stays_finite():
    c, x = _lowpassed(None)                                                   # cond ~ 4e19: outside the parity domain
    ref, lens = _batch([c, c])
    inf, _ = _batch([x, c])
    got = MET.sdr(ref, inf, lens).cpu().numpy()
    assert np.isfinite(got).all() and (np.abs(got) <= 50.0).all(), got


def test_degenerate_inputs():
    fs = 16000
    c, x = _speechlike(fs * 2, fs, 8)
    z = np.zeros_like(c)
    ref, lens = _batch([z, c, c[:2000], c[:200]])
    inf, _ = _batch([x, z, x[:2000], x[:200]])
    s = MET.sdr(ref, inf, lens).cpu().numpy()
    e = MET.estoi(ref, inf, lens, fs).cpu().numpy()
    assert np.isnan(s[0])                                                     # zero reference: no solution
    assert s[1] == pytest.approx(-50.0, abs=1e-9) and e[1] == 0.0              # zero estimate
    assert e[2] == 1e-5 and e[3] == 1e-5                                      # under 30 frames; no full frame at all
    assert ORC.estoi(_f64(c[:2000]), _f64(x[:2000]), fs) == 1e-5
    assert np.isfinite(s[1:]).all()


# ------------------------------------------------------------------------------------------------ batching
@pytest.mark.parametrize("fs", [16000, 44100])
def test_ragged_batch_is_bitwise_the_single_scores(fs):
    pairs = [_speechlike(int(s * fs), fs, 20 + i) for i, s in enumerate((2.2, 0.9, 1.6, 0.03))]
    ref, lens = _batch([c for c, _ in pairs])
    inf, _ = _batch([x for _, x in pairs])
    e_all = MET.estoi(ref, inf, lens, fs).cpu()
    s_all = MET.sdr(ref, inf, lens).cpu()
    for r, (c, x) in enumerate(pairs):
        r1, l1 = _batch([c])
        i1, _ = _batch([x])
        assert torch.equal(MET.estoi(r1, i1, l1, fs).cpu(), e_all[r: r + 1]), r
        assert torch.equal(MET.sdr(r1, i1, l1).cpu(), s_all[r: r + 1]), r
    again = MET.estoi(ref, inf, lens, fs).cpu()
    assert torch.equal(again, e_all)


# ------------------------------------------------------------------------------------------------ end to end
def test_inference_then_evaluate(tmp_path):
    from urgent2026_challenge_track1_b200 import evaluate as EV
    from urgent2026_challenge_track1_b200 import inference as I
    from urgent2026_challenge_track1_b200.checkpoint import save_checkpoint
    from urgent2026_challenge_track1_b200.config import Config
    from urgent2026_challenge_track1_b200.d_model import SEModel
    torch.manual_seed(0)
    cfg = Config(se_model="bsrnn", model_configs={"num_channel": 32, "num_layer": 1})
    ckpt = save_checkpoint(str(tmp_path / "se.ckpt"), SEModel(cfg, precision="fp32"), cfg)
    specs = [(16000, 24000), (16000, 17000), (8000, 12000), (48000, 60000)]
    ins, refs = [], []
    for i, (fs, n) in enumerate(specs):
        c, x = _speechlike(n, fs, 40 + i)
        pc, px = str(tmp_path / f"clean_{i}.wav"), str(tmp_path / f"noisy_{i}.wav")
        I._write_wav(pc, c, fs)
        I._write_wav(px, x, fs)
        refs.append(f"utt{i} {pc}")
        ins.append(f"utt{i} {px}")
    (tmp_path / "clean.scp").write_text("\n".join(refs) + "\n")
    (tmp_path / "wav.scp").write_text("\n".join(ins) + "\n")
    out = str(tmp_path / "enh")
    I.main(I.build_parser().parse_args(["--input_scp", str(tmp_path / "wav.scp"), "--output_dir", out, "--ckpt_path", ckpt,
                                        "--precision", "fp32"]))
    ev = str(tmp_path / "scores")
    EV.main(EV.build_parser().parse_args(["--ref_scp", str(tmp_path / "clean.scp"), "--inf_scp",
                                          os.path.join(out, "inf.scp"), "--output_dir", ev, "--max_batch", "2"]))
    listed = [l.split() for l in open(os.path.join(out, "inf.scp")).read().split("\n") if l]
    got = {}
    for name in ("ESTOI", "SDR"):
        rows = [l.split() for l in open(os.path.join(ev, f"{name}.scp")).read().split("\n") if l]
        assert [u for u, _ in rows] == [u for u, _ in listed]                 # inf.scp order
        got[name] = {u: float(v) for u, v in rows}
    for uid, path in listed:
        i = int(uid[3:])
        c, fs = I._read_wav(str(tmp_path / f"clean_{i}.wav"))
        e, fs2 = I._read_wav(path)
        assert fs == fs2 == specs[i][0]
        assert abs(got["ESTOI"][uid] - ORC.estoi(_f64(c), _f64(e), fs)) <= 1e-5, uid
        assert abs(got["SDR"][uid] - ORC.sdr(_f64(c), _f64(e))) <= 1e-3, uid
    res = dict(l.split(": ") for l in open(os.path.join(ev, "RESULTS.txt")).read().strip().split("\n"))
    for name in ("ESTOI", "SDR"):
        assert res[name] == f"{np.nanmean(list(got[name].values())):.4f}"
