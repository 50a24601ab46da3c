"""Corpus-fed training step against device-resident synthetic batches of the same shape (BASELINE config 5:
BSRNN_baseline, B = 4 x 96 000 samples at 48 kHz, fp16 BLSTM blocks, CUDA-graph replay), in one process.
  python tools/bench_train_corpus.py [--utts 384] [--rounds 3] [--workers 4]
A 48 kHz WAV set of 2-4 s utterances (so every one is cropped to 96 000 samples) is written to a temporary directory
from synth.synth_pair and read through data.make_loader + data.prefetch_to_device, as train_se does.  Rounds alternate
an epoch fed from the set with as many steps on tensors already on the device.  Then a mixed-rate set (all seven rates,
same durations) runs one epoch: graph captures per epoch, device memory per captured graph.
Prints one JSON line, with the GPU name and power limit read in the same run.  Also: the private pool of a captured FlowSE
step at the published width (48 kHz and 8 kHz, same B x samples), which decides how many FlowSE graphs fit.
On a B200 at its 1000 W limit: 61.9 ms per step fed from the 48 kHz set against 61.1 ms from device tensors (96-step
epochs, DataLoader start included).  Mixed-rate set (28 steps per epoch, 21 shapes): 134, 184 and 79.9 ms per step in
epochs 1-3 (captures in the first two; 8 graphs kept, 13 shapes eager) against 89.1 ms for an eager trainer; SE pools up
to 8.7 GB.  FlowSE pools 20.6 GB at 48 kHz and 67.2 GB at 8 kHz."""
import argparse, json, os, shutil, subprocess, sys, tempfile, time
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch
from scipy.io import wavfile
from urgent2026_challenge_track1_b200 import BSRNN_SE, data as D
from urgent2026_challenge_track1_b200.synth import synth_pair
from urgent2026_challenge_track1_b200.training import SETrainer

RATES = (8000, 16000, 22050, 24000, 32000, 44100, 48000)

ap = argparse.ArgumentParser()
ap.add_argument("--utts", type=int, default=384); ap.add_argument("--mixed-utts", type=int, default=112)
ap.add_argument("--batch", type=int, default=4); ap.add_argument("--max-duration", type=int, default=96000)
ap.add_argument("--rounds", type=int, default=3); ap.add_argument("--workers", type=int, default=4)
ap.add_argument("--channels", type=int, default=196); ap.add_argument("--layers", type=int, default=6)
a = ap.parse_args()
dev = torch.device("cuda", 0)
torch.cuda.set_device(dev)


def write_set(root, n, rates, seed):
    rng = np.random.default_rng(seed)
    os.makedirs(root)
    with open(os.path.join(root, "wav.scp"), "w") as fn, open(os.path.join(root, "spk1.scp"), "w") as fc:
        for i in range(n):
            fs = rates[i % len(rates)]
            clean, noisy = synth_pair(1, int(rng.uniform(2.0, 4.0) * fs), fs, seed=seed + i)
            for f, x, tag in ((fn, noisy, "n"), (fc, clean, "c")):
                p = os.path.join(root, f"u{i:05d}_{tag}.wav")
                wavfile.write(p, fs, x[0].numpy())
                print(f"u{i:05d} {p}", file=f)
    return D.PairCorpus(root)


def smi(q):
    try:
        return subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader", "-i", "0"], capture_output=True,
                              text=True, timeout=30).stdout.strip()
    except Exception as e:
        return f"unavailable ({e})"


torch.manual_seed(0)
m = BSRNN_SE(a.channels, a.layers, precision="fp32").to(dev)
tr = SETrainer(m, lr=1e-3, precision="fp16", cuda_graph=True)
tmp = tempfile.mkdtemp(prefix="bench_train_corpus_")
corpus = write_set(os.path.join(tmp, "fs48k"), a.utts, (48000,), 1)
clean_s, noisy_s = synth_pair(a.batch, a.max_duration, 48000, seed=5)
clean_s, noisy_s = clean_s.view(a.batch, 1, -1).to(dev), noisy_s.view(a.batch, 1, -1).to(dev)
lens_s = torch.full((a.batch,), a.max_duration, dtype=torch.int32)


def corpus_epoch(c, epoch, per_step=None):
    batches, _ = D.train_batches(c, a.batch, a.max_duration, 0, 1, epoch, 1996)
    loader = D.make_loader(c, batches, a.max_duration, True, a.workers, seed=1996, epoch=epoch)
    n = 0
    for clean, noisy, fs, lens in D.prefetch_to_device(loader, dev):
        before = tr.captures
        tr.step(noisy, clean, lens, fs)
        if per_step is not None and tr.captures > before:
            key = (tuple(noisy.shape), tuple(clean.shape), int(fs))
            per_step.append((int(fs), int(noisy.shape[-1]), tr.pool_bytes[key]))
        n += 1
    return n


def synthetic_epoch():
    for _ in range(steps):
        tr.step(noisy_s, clean_s, lens_s, 48000)
    return steps


def timed(fn):
    torch.cuda.synchronize(dev)
    t0 = time.perf_counter()
    n = fn()
    torch.cuda.synchronize(dev)
    return (time.perf_counter() - t0) * 1e3 / n, n


# warm-up: capture the one 48 kHz graph, start the loader once, bring the synthetic feed to steady state
corpus_epoch(corpus, 0)
for _ in range(3):
    tr.step(noisy_s, clean_s, lens_s, 48000)
steps = len(D.train_batches(corpus, a.batch, a.max_duration, 0, 1, 0, 1996)[0])
corpus_ms, synth_ms = [], []
for r in range(a.rounds):
    ms, _ = timed(lambda: corpus_epoch(corpus, r + 1))
    corpus_ms.append(ms)
    ms, _ = timed(synthetic_epoch)
    synth_ms.append(ms)
captures_48k = tr.captures
# mixed-rate set: three epochs (a shape is captured the second time it comes, if it fits), every capture logged with its
# pool size; the same epoch on an eager trainer for comparison
mixed = write_set(os.path.join(tmp, "mixed"), a.mixed_utts, RATES, 7)
tr._graphs.clear()
tr._seen.clear()
tr._eager_only.clear()
torch.cuda.empty_cache()
c0 = tr.captures
per_graph = []
mixed_ms = []
for ep in range(3):
    ms, n_mixed = timed(lambda: corpus_epoch(mixed, ep, per_graph))
    mixed_ms.append(ms)
captures_mixed = tr.captures - c0
graphs_kept = len(tr._graphs)
eager_only = len(tr._eager_only)
se_pool = max(tr.pool_bytes.values())
tr._graphs.clear()
tr.cuda_graph = False                                       # (the graphs' pools are released here)
mixed_eager_ms, _ = timed(lambda: corpus_epoch(mixed, 0))
del tr, m
torch.cuda.empty_cache()
# FlowSE at the published width (N = 384, 6 layers): the private pool of one captured step at 48 kHz and at 8 kHz (most
# frames), same B x samples
from urgent2026_challenge_track1_b200.config import Config
from urgent2026_challenge_track1_b200.flow_model import FlowSEModel
torch.manual_seed(0)
fm = FlowSEModel(Config(model_type="flowse", ema_decay=0.999, sigma_max=0.5, sigma_min=0.05, t_eps=0.03, T_rev=1.0,
                        loss_type="mse", loss_abs_exponent=0.5, n_fft=1536, hop_length=384, spec_transform_type="exponent",
                        spec_abs_exponent=0.667, spec_factor=0.065, bsrnn_hidden=384, num_layer=6, learning_rate=1e-4)).to(dev)
ftr = fm.configure_optimizers(precision="fp16", cuda_graph=True)
flowse_pool = {}
for fs in (48000, 8000):
    c, n = synth_pair(a.batch, a.max_duration, fs, seed=9)
    c, n = c.view(a.batch, 1, -1).to(dev), n.view(a.batch, 1, -1).to(dev)
    for _ in range(2):                                       # eager (measures the peak), then the capture if it fits
        ftr.step(n, c, lens_s, fs)
    key = ((a.batch, 1, a.max_duration), (a.batch, 1, a.max_duration), fs)
    flowse_pool[fs] = {"eager_peak_bytes": ftr._seen[key], "pool_bytes": ftr.pool_bytes.get(key)}
torch.cuda.synchronize(dev)
out = {"metric": "corpus-fed vs synthetic training step, config 5 (BSRNN_baseline, fp16, graph replay)",
       "ms_per_step_corpus": min(corpus_ms), "ms_per_step_synthetic": min(synth_ms),
       "corpus_over_synthetic": min(corpus_ms) / min(synth_ms), "rounds_corpus_ms": corpus_ms, "rounds_synthetic_ms": synth_ms,
       "steps_per_epoch": steps, "captures_48k_total": captures_48k,
       "mixed_rate": {"steps_per_epoch": n_mixed, "ms_per_step_graphed_by_epoch": mixed_ms,
                      "ms_per_step_eager": mixed_eager_ms, "captures_in_three_epochs": captures_mixed,
                      "graphs_kept": graphs_kept, "eager_only_shapes": eager_only, "se_pool_bytes_max": se_pool,
                      "per_capture": [{"fs": f, "width": w, "pool_bytes": b} for f, w, b in per_graph]},
       "flowse_published_width": flowse_pool,
       "gpu": torch.cuda.get_device_name(dev), "power_limit": smi("power.limit"), "sm_clock_max": smi("clocks.max.sm"),
       "config": {"batch": a.batch, "samples": a.max_duration, "fs": 48000, "channels": a.channels, "layers": a.layers,
                  "utts": a.utts, "workers": a.workers}}
print(json.dumps(out))
shutil.rmtree(tmp, ignore_errors=True)
