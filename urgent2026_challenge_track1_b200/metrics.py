"""Intrusive speech-enhancement metrics on the GPU: ESTOI and SDR of a batch of (reference, estimate) pairs, the two
restatable scores of the reference's ``evaluation_metrics/calculate_intrusive_se_metrics.py`` (ESTOI through
``pystoi.stoi(extended=True)``, SDR through ``fast_bss_eval`` with a 512-tap distortion filter clamped to +-50 dB).

Inputs are device tensors: ``ref`` and ``inf`` (B, T) f32, valid on [0, lengths[b]) (the padding may hold anything and
never reaches a score), one sample rate per batch.  Scores come back as (B,) f64 device tensors, and an utterance's
score is bit-identical whether it is scored alone or inside any batch (csrc/metrics.cu has no floating-point atomics).

The host side only designs the resampling filter (the Octave-compatible Kaiser window pystoi uses), the one-third octave
band table and the buffer sizes; every pass over the audio is a kernel of csrc/metrics.cu.  There is no CPU fallback:
without the library or a GPU every call raises ``NativeLibraryError``.

Where these scores differ from pystoi / fast_bss_eval on purpose (DESIGN.md §7d):
  * ESTOI adds no ``EPS * randn`` jitter before its normalisations; a row or column of zero norm normalises to zeros.
    An all-zero estimate scores exactly 0 (pystoi: a tiny random value).  Fewer than 30 frames after silence removal
    (including no frame at all) score 1e-5, pystoi's fallback.
  * SDR of an all-zero reference is NaN (fast_bss_eval's solve fails).  When the Levinson recursion of an extremely
    ill-conditioned reference breaks down (a non-positive pivot), the solution of the largest leading system that was
    still positive definite is used, so the score stays finite and inside [-50, 50].
"""
from __future__ import annotations

import math

import numpy as np
import torch

FS = 10000                      # ESTOI's internal rate
N_FRAME = 256                   # frame length (and STFT window) at 10 kHz; hop N_FRAME / 2
NFFT = 512
NUMBAND = 15
MINFREQ = 150


# ------------------------------------------------------------------------------------------------ host-side design
def resample_ratio(fs):
    """(up, down) of the resampling fs -> 10 kHz, reduced by their gcd (resample_poly's first step)."""
    g = math.gcd(FS, int(fs))
    return FS // g, int(fs) // g


def resample_taps(up, down):
    """The Octave-compatible Kaiser low-pass pystoi resamples with (``_resample_window_oct``), normalised to unit sum and
    scaled by ``up`` as resample_poly applies it.  f64, 2 L + 1 taps."""
    g = math.gcd(up, down)
    up, down = up // g, down // g
    stopband_cutoff_f = 1.0 / (2 * max(up, down))
    roll_off_width = stopband_cutoff_f / 10
    rejection_db = 60.0                                     # -20 * log10_rejection, log10_rejection = -3
    L = int(np.ceil((rejection_db - 8) / (28.714 * roll_off_width)))
    t = np.arange(-L, L + 1)
    ideal = 2 * up * stopband_cutoff_f * np.sinc(2 * stopband_cutoff_f * t)
    beta = 0.1102 * (rejection_db - 8.7)                    # rejection_db > 50
    h = np.kaiser(2 * L + 1, beta) * ideal
    return h / np.sum(h) * up


def polyphase(h, up):
    """(up, J) table of the taps by phase, P[ph, j] = h[ph + j up] (zero past the end): the layout the resampling kernel
    reads, so that one output's taps are contiguous."""
    J = -(-h.size // up)
    return np.ascontiguousarray(np.pad(h, (0, J * up - h.size)).reshape(J, up).T)


def resampled_length(n, up, down):
    """resample_poly's output length ceil(n up / down)."""
    return -(-int(n) * up // down)


def n_frames(n):
    """Frames of ``range(0, n - 256, 128)``: pystoi's framing of the silence removal and of the STFT."""
    return (n - N_FRAME - 1) // (N_FRAME // 2) + 1 if n > N_FRAME else 0


def third_octave_bands(fs=FS, nfft=NFFT, num_bands=NUMBAND, min_freq=MINFREQ):
    """(lo, hi) int32 bin ranges of the one-third octave bands: band k sums bins [lo[k], hi[k]) (pystoi's ``thirdoct``
    matrix, which is one on exactly that range)."""
    f = np.linspace(0, fs, nfft + 1)[: nfft // 2 + 1]
    k = np.arange(num_bands, dtype=float)
    freq_low = min_freq * 2.0 ** ((2 * k - 1) / 6)
    freq_high = min_freq * 2.0 ** ((2 * k + 1) / 6)
    lo = np.array([np.argmin(np.square(f - fl)) for fl in freq_low], np.int32)
    hi = np.array([np.argmin(np.square(f - fh)) for fh in freq_high], np.int32)
    return lo, hi


# ------------------------------------------------------------------------------------------------ device calls
_CACHE = {}


def _cached(key, make):
    if key not in _CACHE:
        _CACHE[key] = make()
    return _CACHE[key]


def _prepare(ref, inf, lengths):
    from . import _lib as L
    L.require_device()
    if ref.shape != inf.shape or ref.dim() != 2:
        raise ValueError(f"ref and inf must be (B, T) of the same shape, got {tuple(ref.shape)} and {tuple(inf.shape)}")
    if ref.dtype != torch.float32 or inf.dtype != torch.float32 or not ref.is_cuda or not inf.is_cuda:
        raise ValueError("ref and inf must be float32 CUDA tensors")
    B, T = ref.shape
    lens = torch.as_tensor(lengths).to(device=ref.device, dtype=torch.int32).reshape(-1).contiguous()
    if lens.numel() != B:
        raise ValueError(f"{lens.numel()} lengths for {B} utterances")
    return ref.contiguous(), inf.contiguous(), lens, B, T


def _resample(x, lens, fs):
    """bsrnn_resample_poly of x (B, T) to 10 kHz -> (y (B, T10), y_len (B) int32)."""
    from . import _lib as L
    up, down = resample_ratio(fs)
    B, T = x.shape

    def design():
        h = resample_taps(up, down)
        return torch.from_numpy(polyphase(h, up)).to(x.device), h.size

    taps, n_taps = _cached(("taps", up, down, str(x.device)), design)
    T10 = resampled_length(T, up, down)
    y = torch.empty(B, T10, dtype=torch.float32, device=x.device)
    y_len = torch.empty(B, dtype=torch.int32, device=x.device)
    L.call("bsrnn_resample_poly", x.data_ptr(), lens.data_ptr(), B, T, taps.data_ptr(), n_taps, up, down, y.data_ptr(),
           y_len.data_ptr(), T10, L.stream_ptr())
    return y, y_len


def estoi_stages(ref, inf, lengths, fs):
    """Every intermediate of ESTOI (for tests and inspection): the 10 kHz signals and lengths, the silence-compacted
    signals and their lengths, the band envelopes (B, 2, 15, F) f64 (index 0 = ref, 1 = inf) with room for F frames, and
    the scores."""
    from . import _lib as L
    ref, inf, lens, B, T = _prepare(ref, inf, lengths)
    dev = ref.device
    if int(fs) != FS:
        x10, n10 = _resample(ref, lens, fs)
        y10, _ = _resample(inf, lens, fs)
    else:
        x10, y10, n10 = ref, inf, lens
    T10 = x10.shape[1]
    NF = max(n_frames(T10), 1)
    xc = torch.empty(B, T10, dtype=torch.float32, device=dev)
    yc = torch.empty_like(xc)
    c_len = torch.empty(B, dtype=torch.int32, device=dev)
    scratch = torch.empty(-(-L.lib().bsrnn_estoi_compact_scratch_bytes(B, T10) // 8), dtype=torch.float64, device=dev)
    L.call("bsrnn_estoi_compact", x10.data_ptr(), y10.data_ptr(), n10.data_ptr(), B, T10, xc.data_ptr(), yc.data_ptr(),
           c_len.data_ptr(), scratch.data_ptr(), L.stream_ptr())
    band = _cached(("bands", str(dev)), lambda: torch.from_numpy(np.concatenate(third_octave_bands())).to(dev))
    tw = _cached(("twiddle", str(dev)), lambda: _twiddle(dev))
    tob = torch.empty(B, 2, NUMBAND, NF, dtype=torch.float64, device=dev)
    L.call("bsrnn_estoi_bands", xc.data_ptr(), yc.data_ptr(), c_len.data_ptr(), B, T10, tw.data_ptr(), band.data_ptr(),
           band[NUMBAND:].data_ptr(), tob.data_ptr(), NF, L.stream_ptr())
    out = torch.empty(B, dtype=torch.float64, device=dev)
    seg = torch.empty(B * NF, dtype=torch.float64, device=dev)
    L.call("bsrnn_estoi_score", tob.data_ptr(), c_len.data_ptr(), B, NF, seg.data_ptr(), out.data_ptr(), L.stream_ptr())
    return dict(x10=x10, y10=y10, n10=n10, xc=xc, yc=yc, c_len=c_len, tob=tob, estoi=out)


def _twiddle(dev):
    from . import _lib as L
    tw = torch.empty(NFFT, 2, dtype=torch.float32, device=dev)
    L.call("bsrnn_fft_twiddle", tw.data_ptr(), NFFT, L.stream_ptr())
    return tw


def estoi(ref, inf, lengths, fs):
    """ESTOI (pystoi 0.4, extended=True) of each pair -> (B,) f64 on the device."""
    return estoi_stages(ref, inf, lengths, fs)["estoi"]


def sdr(ref, inf, lengths):
    """BSS-eval v3 SDR with a 512-tap distortion filter, clamped to +-50 dB, of each pair -> (B,) f64 on the device."""
    from . import _lib as L
    ref, inf, lens, B, T = _prepare(ref, inf, lengths)
    out = torch.empty(B, dtype=torch.float64, device=ref.device)
    scratch = torch.empty(-(-L.lib().bsrnn_sdr_scratch_bytes(B, T) // 8), dtype=torch.float64, device=ref.device)
    L.call("bsrnn_sdr", ref.data_ptr(), inf.data_ptr(), lens.data_ptr(), B, T, out.data_ptr(), scratch.data_ptr(),
           L.stream_ptr())
    return out
