"""Dynamic-mixing set reader, parameter draws, the ``dynamic_mixing:`` key validation and the worker collate (mixing.py), on
small WAV sets written into tmp_path; the low-pass taps against the independent f64 reference of mixing_ref."""
import os

import numpy as np
import pytest
import torch

from test_corpus_cpu import _wav
from urgent2026_challenge_track1_b200 import data as D
from urgent2026_challenge_track1_b200 import mixing as M
from urgent2026_challenge_track1_b200.config import Config
from urgent2026_challenge_track1_b200.synth import synth_pair

import mixing_ref

RATES = (8000, 16000, 48000)


def _pink(n, rng):
    spec = np.fft.rfft(rng.standard_normal(n))
    spec /= np.sqrt(np.maximum(np.arange(spec.size), 1.0))
    x = np.fft.irfft(spec, n)
    return 0.1 * x / np.sqrt(np.mean(x ** 2))


def _rir(fs, rng, seconds):
    n = int(seconds * fs)
    t = np.arange(n) / fs
    h = rng.standard_normal(n) * np.exp(-6.9 * t / rng.uniform(0.3, 1.0)) * 0.1
    d = int(rng.integers(0, fs // 200))
    h[:d] = 0.0
    h[d] = 1.0
    return h


def make_mix_set(root, n_per_rate=4, rates=RATES, seed=0, rir=True, fs_column=False):
    """Speech of 0.25-0.6 s from synth_pair, per rate one short (0.1 s, tiled) and one long (2 s) 1/f noise as 16-bit PCM,
    and RIRs of 0.05-0.2 s (one longer than most utterances); scp lines in shuffled order, 2 or 3 columns."""
    root.mkdir(parents=True, exist_ok=True)
    rng = np.random.default_rng(seed)
    lines = {"speech.scp": [], "noise.scp": [], "rir.scp": []}
    meta = {}

    def line(uid, fs, path):
        return f"{uid} {fs} {path}" if fs_column else f"{uid} {path}"
    for fs in rates:
        for i in range(n_per_rate):
            uid = f"s{fs}_{i}"
            n = int(rng.integers(fs // 4, fs * 6 // 10))
            clean, _ = synth_pair(1, n, fs, seed=seed * 1000 + i + fs)
            _wav(root / f"{uid}.wav", clean[0].numpy(), fs)
            lines["speech.scp"].append(line(uid, fs, root / f"{uid}.wav"))
            meta[uid] = (n, fs)
        for j, sec in enumerate((0.1, 2.0)):
            from scipy.io import wavfile
            x = (np.clip(_pink(int(sec * fs), rng), -1, 1) * 32767).astype(np.int16)
            wavfile.write(str(root / f"n{fs}_{j}.wav"), fs, x)
            lines["noise.scp"].append(line(f"n{fs}_{j}", fs, root / f"n{fs}_{j}.wav"))
        if rir:
            for j, sec in enumerate((0.05, 0.2, 0.7)):
                h = _rir(fs, rng, sec)
                _wav(root / f"r{fs}_{j}.wav", np.stack([h, 0.5 * h], 1), fs)           # two channels: the first is used
                lines["rir.scp"].append(line(f"r{fs}_{j}", fs, root / f"r{fs}_{j}.wav"))
    for name, ls in lines.items():
        if ls:
            rng.shuffle(ls)
            (root / name).write_text("\n".join(ls) + "\n")
    return meta


@pytest.fixture(scope="module")
def mixset(tmp_path_factory):
    root = tmp_path_factory.mktemp("mix")
    meta = make_mix_set(root)
    return M.MixCorpus(str(root)), meta


def test_reader_reads_headers_and_pools(mixset):
    c, meta = mixset
    assert sorted(c.uids) == sorted(meta) and c.has_rir
    for u, n, fs in zip(c.uids, c.lengths, c.rates):
        assert (n, fs) == meta[u]
    assert sorted(c.noise) == sorted(c.rir) == list(RATES)
    for fs in RATES:
        assert sorted(n for _, n in c.noise[fs]) == [int(0.1 * fs), int(2.0 * fs)]
        assert all(f"{fs}_" in p for p, _ in c.noise[fs] + c.rir[fs])
    batches, dropped = D.train_batches(c, 2, 6000, 0, 1, 0, 1)                  # the pair sampler, unchanged
    assert dropped == 0 and all(len({c.rates[i] for i in b}) == 1 for b in batches)


def test_three_column_scp_lines(tmp_path):
    make_mix_set(tmp_path / "s", n_per_rate=2, rates=(16000,), fs_column=True)
    c = M.MixCorpus(str(tmp_path / "s"))
    assert len(c) == 2 and c.rates == [16000, 16000]
    lines = (tmp_path / "s" / "speech.scp").read_text().splitlines()
    uid, _, path = lines[0].split()
    lines[0] = f"{uid} 8000 {path}"
    (tmp_path / "s" / "speech.scp").write_text("\n".join(lines) + "\n")
    with pytest.raises(ValueError, match=f"{uid}.*8000.*16000 Hz"):
        M.MixCorpus(str(tmp_path / "s"))
    lines[0] = f"{uid} 16000 {path} extra"
    (tmp_path / "s" / "speech.scp").write_text("\n".join(lines) + "\n")
    with pytest.raises(ValueError, match="uid path"):
        M.MixCorpus(str(tmp_path / "s"))


def test_reader_errors(tmp_path):
    root = tmp_path / "s"
    make_mix_set(root, n_per_rate=2, rates=(8000, 16000))
    for name in ("speech.scp", "noise.scp"):
        os.rename(root / name, root / "bak")
        with pytest.raises(FileNotFoundError, match=name):
            M.MixCorpus(str(root))
        os.rename(root / "bak", root / name)
    M.MixCorpus(str(root))
    speech = (root / "speech.scp").read_text().splitlines()
    (root / "speech.scp").write_text("\n".join(speech + speech[:1]) + "\n")                  # a uid listed twice
    with pytest.raises(ValueError, match=f"{speech[0].split()[0]}.*twice"):
        M.MixCorpus(str(root))
    (root / "speech.scp").write_text("\n".join(speech) + "\n")
    noise = (root / "noise.scp").read_text().splitlines()
    (root / "noise.scp").write_text("\n".join(l for l in noise if "n16000" not in l) + "\n")  # a rate without noise
    with pytest.raises(ValueError, match="noise.scp.*16000 Hz"):
        M.MixCorpus(str(root))
    (root / "noise.scp").write_text("\n".join(noise) + "\n")
    rir = (root / "rir.scp").read_text().splitlines()
    (root / "rir.scp").write_text("\n".join(l for l in rir if "r8000" not in l) + "\n")      # a rate without RIRs
    with pytest.raises(ValueError, match="rir.scp.*8000 Hz"):
        M.MixCorpus(str(root))
    os.remove(root / "rir.scp")                                                               # rir.scp is optional
    c = M.MixCorpus(str(root))
    assert not c.has_rir and c.rir == {}
    uid, path = noise[0].split()
    with open(path, "wb") as f:                                                               # not a WAV file
        f.write(b"this is not a RIFF file" * 10)
    with pytest.raises(ValueError, match=f"{uid}.*WAV"):
        M.MixCorpus(str(root))


def test_dynamic_mixing_key_validation():
    p = M.mix_params(Config())
    assert p == dict(snr_range=(-5.0, 20.0), prob_reverb=0.5, early_rir_ms=50.0, prob_bandwidth_limit=0.25,
                     prob_clipping=0.25, prob_packet_loss=0.1)
    p = M.mix_params(Config(dynamic_mixing={"snr_range": [0, 5], "prob_clipping": 1}))
    assert p["snr_range"] == (0.0, 5.0) and p["prob_clipping"] == 1.0 and p["prob_reverb"] == 0.5
    for bad, msg in (({"snr": [0, 1]}, "unknown key 'snr'"), ({"snr_range": [5, 0]}, "snr_range"),
                     ({"snr_range": [1]}, "snr_range"), ({"prob_reverb": 1.5}, "prob_reverb"),
                     ({"prob_packet_loss": -0.1}, "prob_packet_loss"), ({"early_rir_ms": -1}, "early_rir_ms"),
                     ([0.5], "mapping")):
        with pytest.raises(ValueError, match=msg):
            M.mix_params(Config(dynamic_mixing=bad))


def test_draws_are_a_pure_function_of_seed_epoch_uid(mixset):
    c, _ = mixset
    params = M.mix_params(Config(dynamic_mixing=dict(prob_reverb=0.5, prob_bandwidth_limit=0.5, prob_clipping=0.5,
                                                     prob_packet_loss=0.5)))
    seen = {k: set() for k in ("bw", "rir", "clip", "loss")}
    for i in range(len(c)):
        n, fs = min(c.lengths[i], 6000), c.rates[i]
        per_epoch = []
        for epoch in range(8):
            d = M.draw(c, i, n, params, 7, epoch)
            e = M.draw(c, i, n, params, 7, epoch)
            assert repr(d) == repr(e)
            per_epoch.append(repr(d))
            assert -5.0 <= d["snr"] <= 20.0
            assert any(p == d["noise_path"] for p, _ in c.noise[fs])
            off_max = d["noise_n"] - n if d["noise_n"] >= n else d["noise_n"] - 1
            assert 0 <= d["noise_off"] <= off_max
            if d["bw_rate"]:
                assert d["bw_rate"] in M.RATES and d["bw_rate"] < fs
            assert fs != 8000 or d["bw_rate"] == 0
            if d["rir"] is not None:
                assert any(p == d["rir"] for p, _ in c.rir[fs])
            if (d["qmin"], d["qmax"]) != (0.0, 1.0):
                assert 0.0 <= d["qmin"] <= 0.1 and 0.9 <= d["qmax"] <= 1.0
                seen["clip"].add(True)
            if d["lost"] is not None:
                assert d["lost"].shape == (-(-n // (fs // 50)),) and d["lost"].dtype == bool
                seen["loss"].add(True)
            seen["bw"].add(bool(d["bw_rate"]))
            seen["rir"].add(d["rir"] is not None)
        assert len(set(per_epoch)) == len(per_epoch)                          # a new mixture every epoch
        assert repr(M.draw(c, i, n, params, 8, 0)) != per_epoch[0]             # and per seed
    assert seen["bw"] == {True, False} and seen["rir"] == {True, False} and seen["clip"] and seen["loss"]


def test_collate_reads_windows_and_pads(mixset):
    c, _ = mixset
    params = M.mix_params(Config(dynamic_mixing=dict(prob_reverb=1.0, prob_packet_loss=1.0)))
    max_len = 3000
    for idx in D.train_batches(c, 2, max_len, 0, 1, 0, 1)[0]:
        speech, noise, rir, lost, fs, prm = M.collate(c, idx, max_len, params, 5, 2)
        lens = [min(c.lengths[i], max_len) for i in idx]
        assert int(fs) == c.rates[idx[0]] and speech.shape == noise.shape == (len(idx), max(lens))
        assert prm.dtype == torch.float64 and prm[:, M.P_LEN].tolist() == lens
        pkt = int(fs) // 50
        assert lost.dtype == torch.uint8 and lost.shape == (len(idx), -(-max(lens) // pkt))
        for row, i in enumerate(idx):
            n = lens[row]
            d = M.draw(c, i, n, params, 5, 2)
            x, _ = D._read_wav(c.paths[i])
            off = D.crop_offset(5, 2, c.uids[i], c.lengths[i], max_len) if c.lengths[i] > max_len else 0
            assert torch.equal(speech[row, :n], torch.from_numpy(x[off: off + n]))
            z, _ = D._read_wav(d["noise_path"])
            want = z[(d["noise_off"] + np.arange(n)) % len(z)]
            assert torch.equal(noise[row, :n], torch.from_numpy(want))
            h, _ = D._read_wav(d["rir"])
            h = h[:n]
            r = int(prm[row, M.P_RIR_LEN])
            assert r == len(h) and torch.equal(rir[row, :r], torch.from_numpy(h))
            assert int(prm[row, M.P_EARLY_LEN]) == min(r, int(np.argmax(np.abs(h))) + int(fs) * 50 // 1000)
            assert float(prm[row, M.P_SNR]) == d["snr"] and int(prm[row, M.P_BW_RATE]) == d["bw_rate"]
            assert lost[row, : len(d["lost"])].tolist() == d["lost"].astype(int).tolist()
            for t in (speech, noise):
                assert float(t[row, n:].abs().sum()) == 0.0
            assert float(rir[row, r:].abs().sum()) == 0.0


def test_lowpass_taps_match_the_reference():
    for fs in M.RATES:
        for f_new in [r for r in M.RATES if r < fs]:
            h = M.lowpass_taps(fs, f_new)
            ref = mixing_ref.lowpass(fs, f_new)
            assert len(h) == len(ref) and len(h) % 2 == 1
            assert np.abs(h - ref).max() <= 1e-6 * np.abs(ref).max()


def test_fit_corpus_still_raises_on_a_pre_simulated_set(tmp_path):
    from test_corpus_cpu import make_set
    from urgent2026_challenge_track1_b200.train_se import fit_corpus
    make_set(tmp_path / "pairs", n_per_rate=1, rates=(16000,))
    cfg = Config(train_set_path=str(tmp_path / "pairs"), train_set_dynamic_mixing=True)
    with pytest.raises(NotImplementedError, match="speech.scp.*noise.scp.*train_set_dynamic_mixing: false"):
        fit_corpus(None, cfg, 0, 1, None, False, "unused")
