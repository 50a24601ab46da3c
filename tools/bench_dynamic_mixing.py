"""Dynamic mixing at BASELINE config 5's shape (B = 4 x 96 000 samples at 48 kHz), in one process:
  (a) mixing.simulate() per batch on the GPU (CUDA events over >= 200 batches, every RIR width warmed up), with every
      stage forced on and at the default probabilities;
  (b) the same chain per utterance in NumPy / SciPy f32 on one host core (fftconvolve for the RIR and the low-pass,
      np.quantile), which is what a DataLoader worker would pay instead;
  (c) SE fp16 graph-replay training steps (BSRNN_baseline) fed from a dynamic-mixing set against a pre-simulated set of
      the same shape, in alternating rounds as tools/bench_train_corpus.py does.
  python tools/bench_dynamic_mixing.py [--utts 96] [--rounds 3] [--workers 4] [--batches 200]
Inputs are generated from a seed into a temporary directory: speech from synth.synth_pair (2-4 s, so every utterance is
cropped to 96 000 samples), 1/f noise (5-20 s), RIRs as an exponential decay over noise with a direct-path impulse
(RT60 0.3-1.0 s, 0.5-1.5 s long).  Prints one JSON line, with the GPU name and power limit read in the same run.
On one NVIDIA B200 at its 1000 W power limit: (a) 0.63 ms per batch with every stage on, 0.48 ms at the default
probabilities; (b) 8.1 ms per utterance (median of 16, 7.4-10.8 ms), 32 ms per batch of 4; (c) 66.5 ms per step fed from
the dynamic-mixing set against 67.7 ms from the pre-simulated set (best of 3 alternating rounds of 24 steps, rounds
66.5-70.0 and 67.7-69.6 ms)."""
import argparse, json, os, shutil, subprocess, sys, tempfile, time
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch
from scipy.io import wavfile
from scipy.signal import fftconvolve
from urgent2026_challenge_track1_b200 import BSRNN_SE, data as D, mixing as M
from urgent2026_challenge_track1_b200.config import Config
from urgent2026_challenge_track1_b200.synth import synth_pair
from urgent2026_challenge_track1_b200.training import SETrainer

ap = argparse.ArgumentParser()
ap.add_argument("--utts", type=int, default=96); ap.add_argument("--batch", type=int, default=4)
ap.add_argument("--max-duration", type=int, default=96000); ap.add_argument("--rounds", type=int, default=3)
ap.add_argument("--workers", type=int, default=4); ap.add_argument("--batches", type=int, default=200)
ap.add_argument("--host-utts", type=int, default=16)
ap.add_argument("--channels", type=int, default=196); ap.add_argument("--layers", type=int, default=6)
a = ap.parse_args()
FS = 48000
dev = torch.device("cuda", 0)
torch.cuda.set_device(dev)


def smi(q):
    try:
        return subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader", "-i", "0"], capture_output=True,
                              text=True, timeout=30).stdout.strip()
    except Exception as e:
        return f"unavailable ({e})"


def pink(n, rng):
    spec = np.fft.rfft(rng.standard_normal(n))
    x = np.fft.irfft(spec / np.sqrt(np.maximum(np.arange(spec.size), 1.0)), n)
    return (0.1 * x / np.sqrt(np.mean(x ** 2))).astype(np.float32)


def rir(rng):
    n = int(rng.uniform(0.5, 1.5) * FS)
    t = np.arange(n) / FS
    h = 0.1 * rng.standard_normal(n) * np.exp(-6.9 * t / rng.uniform(0.3, 1.0))
    h[0] = 1.0
    return h.astype(np.float32)


def write_sets(root, n, seed):
    """A dynamic-mixing set and a pre-simulated set with the same speech (so the same batch shapes)."""
    rng = np.random.default_rng(seed)
    mix, pairs = os.path.join(root, "mix"), os.path.join(root, "pairs")
    os.makedirs(mix)
    os.makedirs(pairs)
    with open(os.path.join(mix, "speech.scp"), "w") as fs_, open(os.path.join(pairs, "wav.scp"), "w") as fn, \
            open(os.path.join(pairs, "spk1.scp"), "w") as fc:
        for i in range(n):
            clean, noisy = synth_pair(1, int(rng.uniform(2.0, 4.0) * FS), FS, seed=seed + i)
            for f, x, p in ((fs_, clean, f"{mix}/s{i:05d}.wav"), (fn, noisy, f"{pairs}/n{i:05d}.wav"),
                            (fc, clean, f"{pairs}/c{i:05d}.wav")):
                wavfile.write(p, FS, x[0].numpy())
                print(f"u{i:05d} {p}", file=f)
    for name, gen, count in (("noise", lambda: pink(int(rng.uniform(5, 20) * FS), rng), 16), ("rir", lambda: rir(rng), 16)):
        with open(os.path.join(mix, f"{name}.scp"), "w") as f:
            for j in range(count):
                p = f"{mix}/{name}{j:03d}.wav"
                wavfile.write(p, FS, gen())
                print(f"{name}{j:03d} {p}", file=f)
    return M.MixCorpus(mix), D.PairCorpus(pairs)


def timed(fn):
    torch.cuda.synchronize(dev)
    t0 = time.perf_counter()
    n = fn()
    torch.cuda.synchronize(dev)
    return (time.perf_counter() - t0) * 1e3 / n, n


tmp = tempfile.mkdtemp(prefix="bench_dynamic_mixing_")
mixc, pairc = write_sets(tmp, a.utts, 1)

# ---------------------------------------------------------------- (a) simulate() per batch
results_a = {}
for label, over in (("all_stages", dict(prob_reverb=1.0, prob_bandwidth_limit=1.0, prob_clipping=1.0, prob_packet_loss=1.0)),
                    ("defaults", {})):
    params = M.mix_params(Config(dynamic_mixing=over))
    host = []
    for ep in range(3):
        for idx in D.train_batches(mixc, a.batch, a.max_duration, 0, 1, ep, 1996)[0]:
            host.append(M.collate(mixc, idx, a.max_duration, params, 1996, ep))
    batches = [tuple(t.to(dev) if i < 4 else t for i, t in enumerate(b)) for b in host]
    for b in batches:                                        # warm every shape (RIR width) and cache every FIR
        M.simulate(b, dev)
    torch.cuda.synchronize(dev)
    n = max(a.batches, len(batches))
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(n):
        M.simulate(batches[i % len(batches)], dev)
    e1.record()
    torch.cuda.synchronize(dev)
    results_a[label] = {"ms_per_batch": e0.elapsed_time(e1) / n, "batches": n, "distinct_batches": len(batches)}

# ---------------------------------------------------------------- (b) the same chain on one host core
params = M.mix_params(Config(dynamic_mixing=dict(prob_reverb=1.0, prob_bandwidth_limit=1.0, prob_clipping=1.0,
                                                 prob_packet_loss=1.0)))
host_ms = []
for idx in D.train_batches(mixc, a.batch, a.max_duration, 0, 1, 0, 1996)[0]:
    speech, noise, h, lost, fs, prm = M.collate(mixc, idx, a.max_duration, params, 1996, 0)
    for r in range(len(idx)):
        if len(host_ms) >= a.host_utts:
            break
        n, p = int(prm[r, M.P_LEN]), prm[r].tolist()
        s, z, hr = speech[r, :n].numpy(), noise[r, :n].numpy(), h[r, : int(p[M.P_RIR_LEN])].numpy()
        taps = M.lowpass_taps(FS, int(p[M.P_BW_RATE]))
        t0 = time.perf_counter()
        rev = fftconvolve(s, hr)[:n].astype(np.float32)
        clean = fftconvolve(s, hr[: int(p[M.P_EARLY_LEN])])[:n].astype(np.float32)

        def active(x):
            nf = 1 + (n - 1024) // 512
            pw = np.array([np.mean(x[t * 512: t * 512 + 1024] ** 2) for t in range(nf)], np.float32)
            return pw[pw > 0.01 * pw.mean()].mean()
        g = np.float32(10 ** (-p[M.P_SNR] / 20) * np.sqrt(active(rev) / max(active(z), 1e-10)))
        noisy = rev + g * z
        off = (len(taps) - 1) // 2
        noisy = fftconvolve(noisy, taps)[off: off + n].astype(np.float32)
        lo, hi = np.quantile(noisy, [p[M.P_QMIN], p[M.P_QMAX]])
        noisy = np.clip(noisy, lo, hi)
        pkt = FS // 50
        for k in np.nonzero(lost[r].numpy())[0]:
            noisy[k * pkt: (k + 1) * pkt] = 0
        peak = max(np.abs(noisy).max(), np.abs(clean).max())
        if peak > 0.9:
            noisy, clean = noisy * (0.9 / peak), clean * (0.9 / peak)
        host_ms.append((time.perf_counter() - t0) * 1e3)
    if len(host_ms) >= a.host_utts:
        break

# ---------------------------------------------------------------- (c) training steps fed from each set
torch.manual_seed(0)
m = BSRNN_SE(a.channels, a.layers, precision="fp32").to(dev)
tr = SETrainer(m, lr=1e-3, precision="fp16", cuda_graph=True)
mix_defaults = M.mix_params(Config())


def mix_epoch(ep):
    batches, _ = D.train_batches(mixc, a.batch, a.max_duration, 0, 1, ep, 1996)
    loader = M.make_loader(mixc, batches, a.max_duration, mix_defaults, a.workers, 1996, ep)
    n = 0
    for b in D.prefetch_to_device(loader, dev):
        clean, noisy, fs, lens = M.simulate(b, dev)
        tr.step(noisy, clean, lens, fs)
        n += 1
    return n


def pair_epoch(ep):
    batches, _ = D.train_batches(pairc, a.batch, a.max_duration, 0, 1, ep, 1996)
    loader = D.make_loader(pairc, batches, a.max_duration, True, a.workers, seed=1996, epoch=ep)
    n = 0
    for clean, noisy, fs, lens in D.prefetch_to_device(loader, dev):
        tr.step(noisy, clean, lens, fs)
        n += 1
    return n


pair_epoch(0)                                                # captures the one graph, starts the loaders once
mix_epoch(0)
mix_ms, pair_ms = [], []
for r in range(a.rounds):
    mix_ms.append(timed(lambda: mix_epoch(r + 1))[0])
    pair_ms.append(timed(lambda: pair_epoch(r + 1))[0])
steps = len(D.train_batches(mixc, a.batch, a.max_duration, 0, 1, 0, 1996)[0])
out = {"metric": "dynamic mixing at config 5 (B=4 x 96000 samples, 48 kHz)",
       "a_simulate_ms_per_batch": results_a,
       "b_host_numpy_f32_ms_per_utterance": {"median": float(np.median(host_ms)), "min": float(np.min(host_ms)),
                                             "max": float(np.max(host_ms)), "utterances": len(host_ms),
                                             "per_batch_of_4_median": 4 * float(np.median(host_ms))},
       "c_train_step_ms": {"dynamic_mixing": min(mix_ms), "pre_simulated": min(pair_ms),
                           "ratio": min(mix_ms) / min(pair_ms), "rounds_dynamic_mixing": mix_ms,
                           "rounds_pre_simulated": pair_ms, "steps_per_epoch": steps, "graph_captures": tr.captures},
       "gpu": torch.cuda.get_device_name(dev), "power_limit": smi("power.limit"), "sm_clock_max": smi("clocks.max.sm"),
       "config": {"batch": a.batch, "samples": a.max_duration, "fs": FS, "utts": a.utts, "workers": a.workers,
                  "channels": a.channels, "layers": a.layers}}
print(json.dumps(out))
shutil.rmtree(tmp, ignore_errors=True)
