"""f64 NumPy / SciPy reference of the dynamic-mixing chain (urgent2026_challenge_track1_b200/mixing.py, csrc/mix.cu), from
the same f32 inputs the kernels receive: scipy.signal.fftconvolve for the convolutions, the Kaiser low-pass built here
independently of mixing.lowpass_taps, np.quantile(method="linear"), and the active-level SNR definition."""
import math

import numpy as np
from scipy.signal import fftconvolve

FRAME, HOP = 1024, 512


def reverb(x, h, n):
    """s * h truncated to the speech length (offset 0)."""
    x = np.asarray(x[:n], np.float64)
    if len(h) == 0:
        return x
    return fftconvolve(x, np.asarray(h, np.float64))[:n]


def lowpass(fs, f_new, beta=14.769656459379492, rolloff=0.9475937167399596, zeros=64):
    """Kaiser windowed sinc, cutoff rolloff * f_new / 2, `zeros` zero crossings per side, unit DC gain (f64)."""
    from scipy.signal.windows import kaiser
    cut = rolloff * f_new / 2.0                             # Hz
    spacing = fs / (2.0 * cut)                              # samples between zero crossings
    half = int(math.ceil(zeros * spacing))
    n = np.arange(-half, half + 1)
    h = np.sinc(n / spacing) * kaiser(2 * half + 1, beta, sym=True)
    return h / h.sum()


def zero_phase(x, h, n):
    """x (valid on [0, n)) filtered by the odd-length linear-phase h, output aligned on the input: offset (L-1)/2."""
    x = np.asarray(x[:n], np.float64)
    off = (len(h) - 1) // 2
    return fftconvolve(x, np.asarray(h, np.float64))[off: off + n]


def frame_powers(x, n):
    x = np.asarray(x[:n], np.float64)
    nf = 0 if n <= 0 else (1 + (n - FRAME) // HOP if n >= FRAME else 1)
    return np.array([np.mean(x[t * HOP: min(t * HOP + FRAME, n)] ** 2) for t in range(nf)])


def active_power(x, n):
    p = frame_powers(x, n)
    act = p[p > 0.01 * p.mean()]
    return float(act.mean()) if act.size else 0.0


def snr_gain(s, z, n, snr_db):
    return 10 ** (-snr_db / 20) * math.sqrt(active_power(s, n) / max(active_power(z, n), 1e-10))


def quantile(x, n, q):
    return float(np.quantile(np.asarray(x[:n], np.float64), q, method="linear"))


def finish(noisy, clean, n, qmin, qmax, lost, pkt):
    """clip at the quantiles, zero the lost packets, joint peak normalisation to 0.9 -> (noisy, clean) f64."""
    y = np.clip(np.asarray(noisy[:n], np.float64), quantile(noisy, n, qmin), quantile(noisy, n, qmax))
    if lost is not None:
        for k in range(-(-n // pkt)):
            if k < len(lost) and lost[k]:
                y[k * pkt: (k + 1) * pkt] = 0.0
    c = np.asarray(clean[:n], np.float64)
    peak = max(np.abs(y).max(initial=0.0), np.abs(c).max(initial=0.0))
    scale = 0.9 / peak if peak > 0.9 else 1.0
    return y * scale, c * scale


def chain(speech, noise, rir, n, fs, snr_db, early_len, bw_rate, qmin, qmax, lost, pkt):
    """The whole chain of one utterance -> (clean, noisy) f64 of n samples."""
    rev = reverb(speech, rir, n)
    clean = reverb(speech, np.asarray(rir)[:early_len], n) if len(rir) else rev
    z = np.asarray(noise[:n], np.float64)
    noisy = rev + snr_gain(rev, z, n, snr_db) * z
    if bw_rate:
        noisy = zero_phase(noisy, lowpass(fs, bw_rate), n)
    noisy, clean = finish(noisy, clean, n, qmin, qmax, lost, pkt)
    return clean, noisy
