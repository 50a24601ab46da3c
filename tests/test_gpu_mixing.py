"""Dynamic mixing on the GPU: each kernel of csrc/mix.cu against the f64 reference of mixing_ref, ragged batches with
garbage in their padding, bitwise reproducibility, the whole simulate() chain, train_se end to end on a dynamic-mixing set
(SE and FlowSE) and the simulated batches of a resumed run."""
import os

import numpy as np
import pytest
import torch
import yaml

import mixing_ref as REF
from test_corpus_cpu import make_set
from test_mixing_cpu import _pink, _rir, make_mix_set
from urgent2026_challenge_track1_b200 import data as D
from urgent2026_challenge_track1_b200 import mixing as M
from urgent2026_challenge_track1_b200.config import Config

pytestmark = pytest.mark.gpu
dev = torch.device("cuda")


def rel(a, b):
    a, b = np.asarray(a, np.float64), np.asarray(b, np.float64)
    return float(np.linalg.norm(a - b) / max(np.linalg.norm(b), 1e-300))


def _batch(lens, T, seed, garbage=True):
    """(B, T) f32 rows of 1/f noise valid on [0, len); the padding holds garbage (large values) unless garbage=False."""
    rng = np.random.default_rng(seed)
    x = np.full((len(lens), T), 7.5e3 if garbage else 0.0, np.float32)
    for r, n in enumerate(lens):
        x[r, :n] = _pink(n, rng)
    return x


def _dev(a):
    return torch.from_numpy(np.ascontiguousarray(a)).to(dev)


def test_reverb_conv_short_and_long_rirs():
    fs, T = 16000, 9000
    lens = [9000, 6150, 2047, 4100]
    x = _batch(lens, T, 1)
    rng = np.random.default_rng(2)
    rirs = [_rir(fs, rng, s) for s in (0.05, 0.7, 0.3)] + [np.zeros(0)]   # 800 taps; longer than every utterance; none
    Lh = max(len(h) for h in rirs)
    h = np.full((len(lens), Lh), -3e3, np.float32)                      # garbage beyond each RIR
    for r, g in enumerate(rirs):
        h[r, : len(g)] = g
    early = [min(len(g), int(np.argmax(np.abs(g))) + 800) if len(g) else 0 for g in rirs]
    h_len = np.array([[len(g), e] for g, e in zip(rirs, early)], np.int32)
    y = M.conv(_dev(x), _dev(np.array(lens, np.int32)), _dev(h), _dev(h_len)).cpu().numpy()
    for r, n in enumerate(lens):
        for f, L in enumerate(h_len[r]):
            ref = REF.reverb(x[r], h[r, :L], n)
            if L == 0:
                assert np.array_equal(y[f, r, :n], x[r, :n])
            else:
                assert rel(y[f, r, :n], ref) <= 1e-5, (r, f, rel(y[f, r, :n], ref))
            assert not np.any(y[f, r, n:])


@pytest.mark.parametrize("fs", [16000, 22050, 24000, 32000, 44100, 48000])
def test_zero_phase_lowpass_every_rate_pair(fs):
    lower = [r for r in M.RATES if r < fs]
    lens = [int(0.3 * fs) - 37 * i for i in range(len(lower))]
    T = max(lens)
    x = _batch(lens, T, fs)
    taps = [M.lowpass_taps(fs, r) for r in lower]
    Lh = max(len(t) for t in taps)
    h = np.zeros((len(lower), Lh), np.float32)
    for r, t in enumerate(taps):
        h[r, : len(t)] = t
    h_len = np.array([[len(t)] for t in taps], np.int32)
    y = M.conv(_dev(x), _dev(np.array(lens, np.int32)), _dev(h), _dev(h_len), centered=True)[0].cpu().numpy()
    for r, (n, f_new) in enumerate(zip(lens, lower)):
        ref = REF.zero_phase(x[r], REF.lowpass(fs, f_new), n)
        assert rel(y[r, :n], ref) <= 1e-5, (f_new, rel(y[r, :n], ref))
        assert not np.any(y[r, n:])
        spec = np.abs(np.fft.rfft(y[r, :n].astype(np.float64)))             # the stopband is gone
        f = np.fft.rfftfreq(n, 1 / fs)
        assert spec[f > 1.05 * f_new / 2].max() < 1e-3 * spec.max()


def test_snr_mixing_hits_the_drawn_snr():
    T = 20000
    lens = [20000, 15001, 700, 9999]
    s, z = _batch(lens, T, 3), _batch(lens, T, 4)
    s[1, :5000] *= 1e-3                                                   # a quiet stretch: inactive frames
    snr = np.array([-5.0, 0.0, 7.3, 20.0], np.float32)
    noisy, gain = M.snr_mix(_dev(s), _dev(z), _dev(np.array(lens, np.int32)), _dev(snr))
    noisy, gain = noisy.cpu().numpy(), gain.cpu().numpy()
    for r, n in enumerate(lens):
        ps, pn = REF.active_power(s[r], n), REF.active_power(z[r], n)
        achieved = 10 * np.log10(ps / (float(gain[r]) ** 2 * pn))
        assert abs(achieved - float(snr[r])) <= 1e-3, (r, achieved, snr[r])
        assert rel(noisy[r, :n], s[r, :n].astype(np.float64) + float(gain[r]) * z[r, :n]) <= 1e-6
        assert not np.any(noisy[r, n:])


def test_quantile_clipping_packet_loss_and_peak():
    T = 30000
    lens = [30000, 12345, 2, 1]
    x = _batch(lens, T, 5) * 9.0                                         # peaks well above 0.9
    c = _batch(lens, T, 6)
    x[0, :100] = 0.25                                                    # ties
    q = np.array([[0.03, 0.97], [0.0, 1.0], [0.1, 0.9], [0.05, 0.95]])
    thr = M.quantiles(_dev(x), _dev(np.array(lens, np.int32)), _dev(q)).cpu().numpy()
    for r, n in enumerate(lens):
        for i in range(2):
            ref = np.float32(REF.quantile(x[r], n, q[r, i]))
            assert abs(int(thr[r, i].view(np.int32)) - int(ref.view(np.int32))) <= 1, (r, i, thr[r, i], ref)
    pkt = 320
    rng = np.random.default_rng(8)
    lost = (rng.random((len(lens), -(-T // pkt))) < 0.2).astype(np.uint8)
    xn, xc = _dev(x), _dev(c)
    M.finish(xn, xc, _dev(np.array(lens, np.int32)), _dev(thr), _dev(lost), pkt)
    xn, xc = xn.cpu().numpy(), xc.cpu().numpy()
    for r, n in enumerate(lens):
        rn, rc = REF.finish(x[r], c[r], n, q[r, 0], q[r, 1], lost[r], pkt)
        assert rel(xn[r, :n], rn) <= 1e-6 and rel(xc[r, :n], rc) <= 1e-6
        assert max(np.abs(xn[r, :n]).max(), np.abs(xc[r, :n]).max()) <= 0.9 + 1e-6
        for k in np.nonzero(lost[r])[0]:
            assert not np.any(xn[r, k * pkt: min((k + 1) * pkt, n)])
        assert not np.any(xn[r, n:]) and not np.any(xc[r, n:])


@pytest.fixture(scope="module")
def mixset(tmp_path_factory):
    root = tmp_path_factory.mktemp("mixgpu")
    make_mix_set(root, n_per_rate=4, rates=(16000, 22050, 48000), seed=2)
    return M.MixCorpus(str(root))


_ALL = dict(prob_reverb=1.0, prob_bandwidth_limit=1.0, prob_clipping=1.0, prob_packet_loss=1.0)


def _simulated(corpus, params, max_len, seed=3, epoch=1):
    out = []
    for idx in D.train_batches(corpus, 3, max_len, 0, 1, epoch, seed)[0]:
        b = M.collate(corpus, idx, max_len, params, seed, epoch)
        out.append((idx, b, [t.cpu() if torch.is_tensor(t) else t for t in M.simulate(b, dev)]))
    return out


def test_simulate_chain_matches_the_reference_and_repeats_bitwise(mixset):
    for over in (_ALL, {}):
        params = M.mix_params(Config(dynamic_mixing=over))
        a, b = _simulated(mixset, params, 8000), _simulated(mixset, params, 8000)
        for (idx, batch, (clean, noisy, fs, lens)), (_, _, (c2, n2, _, l2)) in zip(a, b):
            assert torch.equal(clean, c2) and torch.equal(noisy, n2) and torch.equal(lens, l2)
            speech, noise, rir, lost, _, prm = batch
            for r in range(len(idx)):
                n = int(lens[r])
                p = prm[r].tolist()
                rc, rn = REF.chain(speech[r].numpy(), noise[r].numpy(), rir[r, : int(p[M.P_RIR_LEN])].numpy(), n, int(fs),
                                   p[M.P_SNR], int(p[M.P_EARLY_LEN]), int(p[M.P_BW_RATE]), p[M.P_QMIN], p[M.P_QMAX],
                                   lost[r].numpy() if p[M.P_LOSS] else None, int(fs) // 50)
                assert rel(clean[r, 0, :n], rc) <= 1e-5 and rel(noisy[r, 0, :n], rn) <= 1e-4, (r, p)
                assert not clean[r, 0, n:].any() and not noisy[r, 0, n:].any()
                assert max(float(clean[r].abs().max()), float(noisy[r].abs().max())) <= 0.9 + 1e-6


def test_garbage_in_the_padding_never_reaches_a_valid_sample(mixset):
    params = M.mix_params(Config(dynamic_mixing=_ALL))
    idx = D.train_batches(mixset, 3, 8000, 0, 1, 0, 3)[0][0]
    batch = M.collate(mixset, idx, 8000, params, 3, 0)
    speech, noise, rir, lost, fs, prm = batch
    lens = prm[:, M.P_LEN].long()
    dirty = [t.clone() for t in (speech, noise, rir)]
    for r in range(len(idx)):
        dirty[0][r, lens[r]:] = float("nan")
        dirty[1][r, lens[r]:] = 1e30
        dirty[2][r, int(prm[r, M.P_RIR_LEN]):] = float("nan")
    ref = M.simulate(batch, dev)
    got = M.simulate((*dirty, lost, fs, prm), dev)
    assert torch.equal(ref[0].cpu(), got[0].cpu()) and torch.equal(ref[1].cpu(), got[1].cpu())


def _write_yaml(tmp_path, name, **over):
    cfg = dict(model_configs={"num_channel": 32, "num_layer": 1}, train_precision="fp16", train_set_dynamic_mixing=True,
               num_worker=2, seed=11, learning_rate=1e-3, dynamic_mixing=dict(prob_reverb=0.7, prob_bandwidth_limit=0.5,
                                                                                prob_clipping=0.5, prob_packet_loss=0.5))
    cfg.update(over)
    p = tmp_path / f"{name}.yaml"
    p.write_text(yaml.safe_dump(cfg))
    return str(p)


def _run(tmp_path, monkeypatch, yml, *flags):
    from urgent2026_challenge_track1_b200 import train_se
    monkeypatch.chdir(tmp_path)
    return train_se.main(["--config_file", yml, *flags])


@pytest.fixture(scope="module")
def sets(tmp_path_factory):
    root = tmp_path_factory.mktemp("dm")
    make_mix_set(root / "train", n_per_rate=4, rates=(8000, 22050, 48000), seed=0)
    make_set(root / "valid", n_per_rate=2, rates=(8000, 22050, 48000), seed=1)
    return str(root / "train"), str(root / "valid")


def test_train_se_dynamic_mixing_end_to_end(tmp_path, monkeypatch, sets):
    from urgent2026_challenge_track1_b200 import inference as I
    from urgent2026_challenge_track1_b200.d_model import SEModel
    train, valid = sets
    yml = _write_yaml(tmp_path, "se_dm")
    hist = _run(tmp_path, monkeypatch, yml, "--train_set_path", train, "--valid_set_path", valid, "--val_check_interval", "2",
                "--save_top_k", "2", "--batch_size", "2", "--max_duration", "8000", "--num_train_epochs", "1")
    ck_dir = tmp_path / "exp" / "se_dm" / "baseline" / "version_0" / "checkpoints"
    files = sorted(os.listdir(ck_dir))
    print(files, [(v["step"], v["val_loss"]) for v in hist["val"]])
    assert hist["global_step"] == 6 and len(hist["val"]) == 3
    assert all(np.isfinite(v["val_loss"]) for v in hist["val"])
    assert 1 <= len(files) <= 2 and all(f.startswith("best_") and "-val_loss=" in f for f in files)
    ckpt = str(ck_dir / files[0])
    model = I.load_model(ckpt, torch.device("cuda"))
    assert isinstance(model, SEModel)
    wav = os.path.join(valid, "u22050_0_n.wav")
    (tmp_path / "in.scp").write_text(f"utt {wav}\n")
    I.main(I.build_parser().parse_args(["--input_scp", str(tmp_path / "in.scp"), "--output_dir", str(tmp_path / "out"),
                                        "--ckpt_path", ckpt]))
    y, sr = I._read_wav(str(tmp_path / "out" / "wav" / "utt.wav"))
    assert sr == 22050 and np.isfinite(y).all()


def test_train_flowse_dynamic_mixing(tmp_path, monkeypatch, sets):
    import types
    from oracle import ref_loader
    from urgent2026_challenge_track1_b200.flow_model import FlowSEModel
    train, valid = sets
    cfg = dict(vars(ref_loader.flowse_config(types.SimpleNamespace(Config=Config), num_layer=1)))
    cfg = {k: v for k, v in cfg.items() if k not in ("config_file", "train_tag", "model_configs")}
    cfg.update(model_type="flowse", train_set_dynamic_mixing=True, num_worker=1, train_set_path=train, valid_set_path=valid,
               max_steps=3, val_check_interval=2, batch_size=2, max_duration=8000,
               dynamic_mixing=dict(prob_reverb=1.0, prob_bandwidth_limit=0.5, prob_clipping=0.5, prob_packet_loss=0.5))
    yml = tmp_path / "flowse_dm.yaml"
    yml.write_text(yaml.safe_dump(cfg))
    hist = _run(tmp_path, monkeypatch, str(yml))
    assert hist["global_step"] == 3 and [v["step"] for v in hist["val"]] == [2, 3]
    assert all(np.isfinite(v["val_loss"]) for v in hist["val"])
    d = tmp_path / "exp" / "flowse_dm" / "baseline" / "version_0" / "checkpoints"
    files = sorted(os.listdir(d))
    assert files
    FlowSEModel.load_from_checkpoint(str(d / files[0]), map_location="cuda")


def test_resumed_run_simulates_bitwise_equal_batches(tmp_path, monkeypatch, sets):
    """6 steps uninterrupted against 3 + resume + 3 on a set of 4 batches per epoch (the resume lands mid-epoch and crosses
    an epoch end): every simulated batch of the resumed run equals the uninterrupted one bit for bit."""
    train, valid = sets
    yml = _write_yaml(tmp_path, "dm_resume")
    record = []
    real = M.simulate

    def spy(batch, device):
        out = real(batch, device)
        record.append(tuple(t.detach().cpu().clone() for t in out))
        return out
    monkeypatch.setattr(M, "simulate", spy)
    common = ["--train_set_path", train, "--valid_set_path", valid, "--val_check_interval", "3", "--save_top_k", "-1",
              "--batch_size", "3", "--max_duration", "6000", "--num_train_epochs", "3"]
    _run(tmp_path, monkeypatch, yml, *common, "--train_name", "full", "--max_steps", "6")
    full, record[:] = list(record), []
    _run(tmp_path, monkeypatch, yml, *common, "--train_name", "split", "--max_steps", "3")
    h = _run(tmp_path, monkeypatch, yml, *common, "--train_name", "split", "--max_steps", "6")
    assert h["global_step"] == 6 and len(full) == len(record) == 6
    for a, b in zip(full, record):
        assert all(torch.equal(x, y) for x, y in zip(a, b))
