"""Throughput of the GPU metrics (metrics.estoi / metrics.sdr, csrc/metrics.cu), in one process:
  (a) one batch of 64 x 10 s at 48 kHz (245 MB of input, larger than the 126 MB L2);
  (b) a sweep over the seven rates, 8 ragged utterances (2-9 s) per rate;
  (c) oracle/metrics.py (numpy / scipy f64) on this host's CPU for a few 10 s 48 kHz utterances, extrapolated to (a) --
      labelled as an extrapolation.
Each GPU figure is CUDA events around `--reps` back-to-back calls after a warm-up of every shape, ending in a synchronise;
throughput is audio-seconds scored per second of wall time.  Writes bench_metrics.json to --out_dir and prints it, with the
card's name, power limit and max SM clock read in the same run.
  python tools/bench_metrics.py [--out_dir exp/bench_metrics] [--reps 10] [--cpu-utts 3]"""
import argparse, json, os, subprocess, sys, time
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch
from oracle import metrics as ORC
from urgent2026_challenge_track1_b200 import metrics as MET
from urgent2026_challenge_track1_b200.synth import synth_pair

ap = argparse.ArgumentParser()
ap.add_argument("--out_dir", default="exp/bench_metrics"); ap.add_argument("--reps", type=int, default=10)
ap.add_argument("--cpu-utts", type=int, default=3)
a = ap.parse_args()
dev = torch.device("cuda", 0)
torch.cuda.set_device(dev)
RATES = (8000, 16000, 22050, 24000, 32000, 44100, 48000)


def smi(q):
    try:
        return subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader", "-i", "0"], capture_output=True,
                              text=True, timeout=30).stdout.strip()
    except Exception as e:
        return f"unavailable ({e})"


def pairs(lengths, fs, seed, distinct=4):
    """(ref, inf) (B, T) f32 on the host, rows valid on [0, lengths[b]): `distinct` generated pairs with a -25 dB
    broadband floor, reused (scaled) for the other rows; padding zero."""
    T = max(lengths)
    base = [synth_pair(1, T, fs, seed=seed + i) for i in range(distinct)]
    rng = np.random.default_rng(seed)
    ref = np.zeros((len(lengths), T), np.float32)
    inf = np.zeros_like(ref)
    for r, n in enumerate(lengths):
        c, x = (t[0].numpy()[:n].astype(np.float64) for t in base[r % distinct])
        fl = rng.standard_normal(n) * c.std() * 10 ** (-25 / 20)
        s = 1.0 + 0.01 * r
        ref[r, :n], inf[r, :n] = s * (c + fl), s * (x + fl)
    return ref, inf


def gpu_time(fn, reps):
    fn()
    torch.cuda.synchronize(dev)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        fn()
    e1.record()
    torch.cuda.synchronize(dev)
    return e0.elapsed_time(e1) / reps


def run(ref, inf, lengths, fs):
    r, i = torch.from_numpy(ref).to(dev), torch.from_numpy(inf).to(dev)
    lens = torch.tensor(lengths, dtype=torch.int32, device=dev)
    ms_e = gpu_time(lambda: MET.estoi(r, i, lens, fs), a.reps)
    ms_s = gpu_time(lambda: MET.sdr(r, i, lens), a.reps)
    return ms_e, ms_s


out = {"metric": "ESTOI / SDR throughput, audio-seconds scored per second", "reps": a.reps}

# ---------------------------------------------------------------- (a) 64 x 10 s at 48 kHz
FS = 48000
la = [10 * FS] * 64
ref, inf = pairs(la, FS, 1)
ms_e, ms_s = run(ref, inf, la, FS)
audio_a = sum(la) / FS
out["a_64x10s_48k"] = {"estoi_ms": ms_e, "sdr_ms": ms_s, "audio_s": audio_a, "estoi_audio_s_per_s": audio_a / ms_e * 1e3,
                       "sdr_audio_s_per_s": audio_a / ms_s * 1e3, "both_audio_s_per_s": audio_a / (ms_e + ms_s) * 1e3}

# ---------------------------------------------------------------- (b) seven rates, 8 ragged utterances each
sweep, tot = {}, {"audio_s": 0.0, "estoi_ms": 0.0, "sdr_ms": 0.0}
for k, fs in enumerate(RATES):
    lengths = [int((2.0 + i) * fs) + 37 * i for i in range(8)]
    ref, inf = pairs(lengths, fs, 100 + k)
    ms_e, ms_s = run(ref, inf, lengths, fs)
    au = sum(lengths) / fs
    sweep[str(fs)] = {"estoi_ms": ms_e, "sdr_ms": ms_s, "audio_s": au, "estoi_audio_s_per_s": au / ms_e * 1e3,
                      "sdr_audio_s_per_s": au / ms_s * 1e3}
    tot["audio_s"] += au
    tot["estoi_ms"] += ms_e
    tot["sdr_ms"] += ms_s
sweep["all_rates"] = dict(tot, estoi_audio_s_per_s=tot["audio_s"] / tot["estoi_ms"] * 1e3,
                          sdr_audio_s_per_s=tot["audio_s"] / tot["sdr_ms"] * 1e3)
out["b_rate_sweep_8_ragged"] = sweep

# ---------------------------------------------------------------- (c) oracle on the CPU, extrapolated
ref, inf = pairs([10 * FS] * a.cpu_utts, FS, 1)
t_e, t_s = [], []
for r in range(a.cpu_utts):
    c, x = ref[r].astype(np.float64), inf[r].astype(np.float64)
    t0 = time.perf_counter(); ORC.estoi(c, x, FS); t_e.append(time.perf_counter() - t0)
    t0 = time.perf_counter(); ORC.sdr(c, x); t_s.append(time.perf_counter() - t0)
out["c_cpu_oracle_10s_48k"] = {"utterances": a.cpu_utts, "estoi_ms_per_utt_median": 1e3 * float(np.median(t_e)),
                               "sdr_ms_per_utt_median": 1e3 * float(np.median(t_s)),
                               "extrapolated_to_a_s": 64 * float(np.median(t_e) + np.median(t_s)),
                               "note": "numpy/scipy f64 oracle, one process on the GPU host's CPU; batch (a) extrapolated "
                                       "from the median per utterance, not measured"}
out.update({"gpu": torch.cuda.get_device_name(dev), "power_limit": smi("power.limit"), "sm_clock_max": smi("clocks.max.sm")})
os.makedirs(a.out_dir, exist_ok=True)
with open(os.path.join(a.out_dir, "bench_metrics.json"), "w") as f:
    json.dump(out, f, indent=1)
print(json.dumps(out))
