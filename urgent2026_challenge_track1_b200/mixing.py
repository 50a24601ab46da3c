"""Dynamic mixing: a new noisy mixture for every utterance in every epoch (the reference's DynamicMixingDataset,
dataset.py:154-335, enabled by ``train_set_dynamic_mixing: true``), simulated on the GPU.

A set is a directory holding ``speech.scp`` (clean speech), ``noise.scp`` and optionally ``rir.scp``; each line is
``uid path`` or ``uid fs path`` (when given, fs must equal the WAV header's rate).  Noise and RIRs are used only at the
speech's own rate.  The DataLoader workers read audio only (collate): the speech window, the noise segment through a
memory-mapped read of that window, channel 0 of the RIR.  ``simulate`` then runs, per utterance and on the device:
reverberation -> noise at the drawn SNR -> bandwidth limitation -> clipping -> packet loss -> peak normalisation (csrc/mix.cu).
Only the noisy signal is degraded; the target is the early-reverberant speech, or the dry speech without an RIR.

Every random choice of an utterance comes from ``np.random.default_rng([seed, epoch, crc32(uid), _DOMAIN])``: a pure
function of (seed, epoch, uid), like data.crop_offset, so a resumed run repeats its mixtures exactly.
"""
from __future__ import annotations

import math
import os
import zlib

import numpy as np
import torch

from . import data as D

RATES = (8000, 16000, 22050, 24000, 32000, 44100, 48000)
DEFAULTS = dict(snr_range=(-5.0, 20.0), prob_reverb=0.5, early_rir_ms=50.0, prob_bandwidth_limit=0.25, prob_clipping=0.25,
                prob_packet_loss=0.1)
PACKET_MS = 20
_DOMAIN = 0x6D6978                  # separates these draws from crop_offset's stream of the same (seed, epoch, uid)

# columns of the per-utterance parameter tensor (float64; integers are exact)
P_LEN, P_SNR, P_RIR_LEN, P_EARLY_LEN, P_BW_RATE, P_QMIN, P_QMAX, P_LOSS = range(8)
N_PARAMS = 8


# ------------------------------------------------------------------------------------------------ parameters
def mix_params(cfg):
    """The ``dynamic_mixing:`` mapping of the YAML merged over DEFAULTS.  Unknown keys and out-of-range values raise."""
    given = getattr(cfg, "dynamic_mixing", None) or {}
    if not isinstance(given, dict):
        raise ValueError(f"dynamic_mixing: expected a mapping, got {given!r}")
    unknown = sorted(set(given) - set(DEFAULTS))
    if unknown:
        raise ValueError(f"dynamic_mixing: unknown key {unknown[0]!r} (known: {', '.join(sorted(DEFAULTS))})")
    p = dict(DEFAULTS, **given)
    snr = p["snr_range"]
    if (not isinstance(snr, (list, tuple)) or len(snr) != 2 or not all(isinstance(v, (int, float)) for v in snr)
            or not math.isfinite(snr[0]) or not math.isfinite(snr[1]) or snr[0] > snr[1]):
        raise ValueError(f"dynamic_mixing: snr_range must be [low, high] with low <= high, got {snr!r}")
    p["snr_range"] = (float(snr[0]), float(snr[1]))
    for k in ("prob_reverb", "prob_bandwidth_limit", "prob_clipping", "prob_packet_loss"):
        v = p[k]
        if isinstance(v, bool) or not isinstance(v, (int, float)) or not 0.0 <= v <= 1.0:
            raise ValueError(f"dynamic_mixing: {k} must be in [0, 1], got {v!r}")
        p[k] = float(v)
    v = p["early_rir_ms"]
    if isinstance(v, bool) or not isinstance(v, (int, float)) or not 0.0 <= v <= 1000.0:
        raise ValueError(f"dynamic_mixing: early_rir_ms must be in [0, 1000], got {v!r}")
    p["early_rir_ms"] = float(v)
    return p


# ------------------------------------------------------------------------------------------------ set
def read_list(path):
    """-> [(uid, fs or None, path)] of an scp whose lines are ``uid path`` or ``uid fs path``; a uid listed twice raises."""
    out, seen = [], set()
    with open(path) as f:
        for no, line in enumerate(f, 1):
            parts = line.split()
            if not parts:
                continue
            if len(parts) == 2:
                uid, fs, wav = parts[0], None, parts[1]
            elif len(parts) == 3:
                uid, wav = parts[0], parts[2]
                try:
                    fs = int(parts[1])
                except ValueError:
                    raise ValueError(f"{path}:{no}: the fs column of uid {uid!r} is not an integer: {parts[1]!r}") from None
            else:
                raise ValueError(f"{path}:{no}: expected 'uid path' or 'uid fs path', got {line.strip()!r}")
            if uid in seen:
                raise ValueError(f"{path}: uid {uid!r} listed twice")
            seen.add(uid)
            out.append((uid, fs, wav))
    return out


def _open_list(root, name):
    path = os.path.join(root, name)
    entries = []
    for uid, fs, wav in read_list(path):
        n, sr = D._probe(uid, wav)
        if fs is not None and fs != sr:
            raise ValueError(f"{path}: uid {uid!r} lists fs {fs} but {wav} is {sr} Hz")
        entries.append((uid, wav, n, sr))
    return sorted(entries)


def is_mix_set(root):
    return all(os.path.isfile(os.path.join(root, n)) for n in ("speech.scp", "noise.scp"))


class MixCorpus:
    """A dynamic-mixing set: ``uids``, ``lengths``, ``rates`` and ``paths`` of the speech (sorted by uid; what the sampler
    reads), and per-rate pools ``noise[fs]`` / ``rir[fs]`` of (path, n_samples).  ``rir`` is empty without rir.scp."""

    def __init__(self, root):
        for name in ("speech.scp", "noise.scp"):
            if not os.path.isfile(os.path.join(root, name)):
                raise FileNotFoundError(f"{root}: missing {name} (a dynamic-mixing set holds speech.scp, noise.scp and "
                                        "optionally rir.scp)")
        self.root = root
        speech = _open_list(root, "speech.scp")
        self.uids = [e[0] for e in speech]
        self.paths = [e[1] for e in speech]
        self.lengths = [e[2] for e in speech]
        self.rates = [e[3] for e in speech]
        self.noise, self.rir = {}, {}
        for name, pools in (("noise.scp", self.noise), ("rir.scp", self.rir)):
            if name == "rir.scp" and not os.path.isfile(os.path.join(root, name)):
                continue
            for _, wav, n, sr in _open_list(root, name):
                pools.setdefault(sr, []).append((wav, n))
            for fs in sorted(set(self.rates)):
                if fs not in pools:
                    raise ValueError(f"{os.path.join(root, name)}: no entry at {fs} Hz, the rate of speech uid "
                                     f"{self.uids[self.rates.index(fs)]!r}")
        self.has_rir = bool(self.rir)

    def __len__(self):
        return len(self.uids)


# ------------------------------------------------------------------------------------------------ draws
def draw(corpus, i, n, params, seed, epoch):
    """The random choices of speech utterance i with a training window of n samples: a dict with the noise path, its start
    (``noise_off``; a noise shorter than n is tiled from that phase), snr, the RIR path or None, the bandwidth-limit rate
    (0 = none), the clipping quantiles (0, 1 = none) and the lost-packet bitmap (None = no loss).  Every value is drawn
    whether or not its stage is taken, so the stream of one stage does not depend on the others."""
    uid, fs = corpus.uids[i], corpus.rates[i]
    rng = np.random.default_rng([int(seed) & 0xFFFFFFFF, int(epoch), zlib.crc32(uid.encode()), _DOMAIN])
    noises = corpus.noise[fs]
    noise_path, noise_n = noises[int(rng.integers(len(noises)))]
    noise_off = int(rng.integers(noise_n - n + 1)) if noise_n >= n else int(rng.integers(noise_n))
    snr = float(rng.uniform(*params["snr_range"]))
    reverb = rng.random() < params["prob_reverb"]
    rirs = corpus.rir.get(fs, [])
    rir_pick = int(rng.integers(max(len(rirs), 1)))
    lower = [r for r in RATES if r < fs]
    bw = rng.random() < params["prob_bandwidth_limit"]
    bw_pick = int(rng.integers(max(len(lower), 1)))
    clip = rng.random() < params["prob_clipping"]
    qmin, qmax = float(rng.uniform(0.0, 0.1)), float(rng.uniform(0.9, 1.0))
    loss = rng.random() < params["prob_packet_loss"]
    rate = float(rng.uniform(0.05, 0.25))
    pkt = fs * PACKET_MS // 1000
    bitmap = rng.random(-(-n // pkt)) < rate
    return dict(noise_path=noise_path, noise_n=noise_n, noise_off=noise_off, snr=snr,
                rir=rirs[rir_pick][0] if (reverb and rirs) else None,
                bw_rate=lower[bw_pick] if (bw and lower) else 0,
                qmin=qmin if clip else 0.0, qmax=qmax if clip else 1.0,
                lost=bitmap if loss else None)


# ------------------------------------------------------------------------------------------------ worker collate
def read_window(path, off, n):
    """n samples of channel 0 from off, wrapping around the end of the file; a memory-mapped read touches only them."""
    from scipy.io import wavfile
    _, x = wavfile.read(path, mmap=True)
    total = x.shape[0]
    if off + n <= total:
        return D._to_float(x[off: off + n])
    idx = (off + np.arange(n)) % total
    return D._to_float(x[idx])


def collate(corpus, idx, max_len, params, seed, epoch):
    """Reads one batch: speech windows (crop_offset for speech longer than max_len), noise segments and RIRs, right-zero-
    padded to the batch's width and to its longest RIR.  -> (speech (B,T), noise (B,T), rir (B,Lr), lost (B,npk) uint8,
    fs int32 scalar, params (B, N_PARAMS) float64), all on the CPU.  No arithmetic beyond I/O, padding and locating the
    RIR's direct path."""
    fs = corpus.rates[idx[0]]
    lens = [min(corpus.lengths[i], max_len) for i in idx]
    T, B = max(lens), len(idx)
    pkt = fs * PACKET_MS // 1000
    speech = torch.zeros(B, T, dtype=torch.float32)
    noise = torch.zeros(B, T, dtype=torch.float32)
    lost = torch.zeros(B, -(-T // pkt), dtype=torch.uint8)
    prm = torch.zeros(B, N_PARAMS, dtype=torch.float64)
    rirs = []
    for row, i in enumerate(idx):
        n_full, n = corpus.lengths[i], lens[row]
        off = D.crop_offset(seed, epoch, corpus.uids[i], n_full, max_len) if n_full > max_len else 0
        x, sr = D._read_wav(corpus.paths[i])
        if sr != fs or x.shape[0] != n_full:
            raise ValueError(f"uid {corpus.uids[i]!r}: {corpus.paths[i]} changed since the set was opened")
        speech[row, :n] = torch.from_numpy(x[off: off + n])
        d = draw(corpus, i, n, params, seed, epoch)
        noise[row, :n] = torch.from_numpy(read_window(d["noise_path"], d["noise_off"], n))
        rir_len = early = 0
        if d["rir"] is not None:
            h, _ = D._read_wav(d["rir"])
            h = h[:n]                   # taps at or beyond n never reach an output sample of [0, n)
            rir_len = h.shape[0]
            early = min(rir_len, int(np.argmax(np.abs(h))) + int(round(params["early_rir_ms"] * fs / 1000)))
            rirs.append((row, h))
        if d["lost"] is not None:
            lost[row, : d["lost"].shape[0]] = torch.from_numpy(d["lost"].astype(np.uint8))
        prm[row] = torch.tensor([n, d["snr"], rir_len, early, d["bw_rate"], d["qmin"], d["qmax"],
                                 float(d["lost"] is not None)], dtype=torch.float64)
    rir = torch.zeros(B, max([h.shape[0] for _, h in rirs], default=0), dtype=torch.float32)
    for row, h in rirs:
        rir[row, : h.shape[0]] = torch.from_numpy(h)
    return speech, noise, rir, lost, torch.tensor(fs, dtype=torch.int32), prm


class MixDataset(torch.utils.data.Dataset):
    """One item = one collated batch (DataLoader with batch_size=None)."""

    def __init__(self, corpus, batches, max_len, params, seed, epoch):
        self.corpus, self.batches, self.max_len, self.params, self.seed, self.epoch = corpus, batches, max_len, params, seed, epoch

    def __len__(self):
        return len(self.batches)

    def __getitem__(self, i):
        return collate(self.corpus, self.batches[i], self.max_len, self.params, self.seed, self.epoch)


def make_loader(corpus, batches, max_len, params, num_workers, seed, epoch):
    return torch.utils.data.DataLoader(MixDataset(corpus, batches, max_len, params, seed, epoch), batch_size=None,
                                       shuffle=False, num_workers=int(num_workers), pin_memory=torch.cuda.is_available())


# ------------------------------------------------------------------------------------------------ low-pass taps
KAISER_BETA = 14.769656459379492       # resampy's kaiser_best: beta, rolloff and zero crossings per side
ROLLOFF = 0.9475937167399596
ZERO_CROSSINGS = 64


def lowpass_taps(fs, f_new):
    """Linear-phase Kaiser windowed-sinc low-pass for limiting fs to the band of f_new: cutoff ROLLOFF * f_new / 2,
    ZERO_CROSSINGS zero crossings of the sinc on each side, unit DC gain.  -> float32 (L,), L odd."""
    fc = ROLLOFF * f_new / 2.0 / fs                        # cycles per sample
    half = int(math.ceil(ZERO_CROSSINGS / (2.0 * fc)))
    t = np.arange(-half, half + 1, dtype=np.float64)
    h = 2 * fc * np.sinc(2 * fc * t) * np.kaiser(2 * half + 1, KAISER_BETA)
    return (h / h.sum()).astype(np.float32)


_TAPS = {}
_TWIDDLE = {}


def _device_taps(fs, f_new, device):
    key = (fs, f_new, str(device))
    if key not in _TAPS:
        _TAPS[key] = torch.from_numpy(lowpass_taps(fs, f_new)).to(device)
    return _TAPS[key]


def twiddle(device, n=2048):
    from . import _lib as L
    key = (str(device), n)
    if key not in _TWIDDLE:
        tw = torch.empty(n, 2, dtype=torch.float32, device=device)
        L.call("bsrnn_fft_twiddle", tw.data_ptr(), n, L.stream_ptr())
        _TWIDDLE[key] = tw
    return _TWIDDLE[key]


# ------------------------------------------------------------------------------------------------ device chain
def conv(x, x_len, h, h_len, centered=False):
    """bsrnn_mix_conv: x (B,T) f32, x_len (B) int32, h (B,Lh) f32, h_len (B, nfilt) int32, all on the device ->
    (nfilt, B, T)."""
    from . import _lib as L
    B, T = x.shape
    Lh, nfilt = h.shape[1], h_len.shape[1]
    y = torch.empty(nfilt, B, T, dtype=torch.float32, device=x.device)
    scratch = torch.empty(max(L.lib().bsrnn_mix_conv_scratch_bytes(B, T, Lh, nfilt) // 4, 1), dtype=torch.float32,
                          device=x.device)
    L.call("bsrnn_mix_conv", x.data_ptr(), x_len.data_ptr(), h.data_ptr() if Lh else None, h_len.data_ptr(), y.data_ptr(),
           scratch.data_ptr(), twiddle(x.device).data_ptr(), B, T, Lh, nfilt, int(centered), L.stream_ptr())
    return y


def snr_mix(speech, noise, x_len, snr_db):
    """bsrnn_mix_snr -> (noisy (B,T), gain (B))."""
    from . import _lib as L
    B, T = speech.shape
    noisy = torch.empty_like(speech)
    gain = torch.empty(B, dtype=torch.float32, device=speech.device)
    scratch = torch.empty(L.lib().bsrnn_mix_snr_scratch_bytes(B, T) // 8, dtype=torch.float64, device=speech.device)
    L.call("bsrnn_mix_snr", speech.data_ptr(), noise.data_ptr(), x_len.data_ptr(), snr_db.data_ptr(), noisy.data_ptr(),
           gain.data_ptr(), scratch.data_ptr(), B, T, L.stream_ptr())
    return noisy, gain


def quantiles(x, x_len, q):
    """bsrnn_mix_quantiles: q (B,2) f64 -> thresholds (B,2) f32."""
    from . import _lib as L
    B, T = x.shape
    thr = torch.empty(B, 2, dtype=torch.float32, device=x.device)
    L.call("bsrnn_mix_quantiles", x.data_ptr(), x_len.data_ptr(), q.data_ptr(), thr.data_ptr(), B, T, L.stream_ptr())
    return thr


def finish(noisy, clean, x_len, thr, lost, pkt):
    """bsrnn_mix_finish, in place on noisy and clean."""
    from . import _lib as L
    B, T = noisy.shape
    peak = torch.empty(B, dtype=torch.int32, device=noisy.device)
    L.call("bsrnn_mix_finish", noisy.data_ptr(), clean.data_ptr(), x_len.data_ptr(), thr.data_ptr(),
           lost.data_ptr() if lost is not None else None, lost.shape[1] if lost is not None else 0, pkt, peak.data_ptr(),
           B, T, L.stream_ptr())


def simulate(batch, device):
    """One collated batch -> (clean (B,1,T), noisy (B,1,T), fs int32 scalar, lengths (B,) int32): the tuple the trainers'
    step takes.  Runs on the current stream; the signals may already be on the device (data.prefetch_to_device)."""
    from . import _lib as L
    L.require_device()
    speech, noise, rir, lost, fs, prm = batch
    fs_i = int(fs)
    B, T = speech.shape
    speech, noise, rir, lost = (t.to(device, non_blocking=True) for t in (speech, noise, rir, lost))
    lens = prm[:, P_LEN].to(torch.int32)
    ints = torch.stack([prm[:, P_LEN], prm[:, P_RIR_LEN], prm[:, P_EARLY_LEN]], 1).to(torch.int32).to(device)
    x_len = ints[:, 0].contiguous()
    # reverberation: filter 0 the whole RIR (the noisy path), filter 1 its early part (the target)
    rev, clean = conv(speech, x_len, rir, ints[:, 1:3].contiguous())
    snr = prm[:, P_SNR].to(torch.float32).to(device)
    noisy, _ = snr_mix(rev, noise, x_len, snr)
    bw = prm[:, P_BW_RATE].to(torch.int64).tolist()
    if any(bw):
        taps = [_device_taps(fs_i, r, device) if r else None for r in bw]
        Lf = max(t.numel() for t in taps if t is not None)
        h = torch.zeros(B, Lf, dtype=torch.float32, device=device)
        for row, t in enumerate(taps):
            if t is not None:
                h[row, : t.numel()] = t
        h_len = torch.tensor([[t.numel() if t is not None else 0] for t in taps], dtype=torch.int32).to(device)
        noisy = conv(noisy, x_len, h, h_len, centered=True)[0]
    q = prm[:, P_QMIN: P_QMAX + 1].contiguous()
    if bool(((q[:, 0] > 0) | (q[:, 1] < 1)).any()):
        thr = quantiles(noisy, x_len, q.to(device))          # (0, 1) rows clamp to their own min and max: no change
    else:
        thr = torch.tensor([[-math.inf, math.inf]] * B, dtype=torch.float32).to(device)
    clean = clean.contiguous()
    finish(noisy, clean, x_len, thr, lost if bool((prm[:, P_LOSS] > 0).any()) else None, fs_i * PACKET_MS // 1000)
    return clean.view(B, 1, T), noisy.view(B, 1, T), torch.tensor(fs_i, dtype=torch.int32), lens
