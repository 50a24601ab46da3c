"""FlowSE training-step timing at the published config (BSRNN_flowse.yaml: N = 384, H = 768, 6 layers, 103 M parameters).
  python tools/bench_flowse_train.py [--batch 4] [--samples 96000] [--steps 5] [--rounds 3]     (or under torchrun)
Defaults: B = 4 x 96 000 samples at 48 kHz per GPU (config 5's shape: T = 251 frames, K = 48 bands, 48 192 tokens per BLSTM
axis), fp16 tensor-core blocks, CUDA-graph replay.  Two trainers from the same seed, one whose graph holds the fused H = 768
training forward (bsrnn_blstm_fused768_train_tc) and one the step-wise forward, are replayed in alternating rounds in this
process.  One eager step of the default trainer gives the forward / backward / optimizer split and the native launches
per step.  Prints one JSON line; the device name, power limit and max SM clock are read in the same run."""
import argparse
import json
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
import torch.distributed as dist

from urgent2026_challenge_track1_b200 import _lib as L, training_tc as TT
from urgent2026_challenge_track1_b200.config import Config
from urgent2026_challenge_track1_b200.flow_model import FlowSEModel

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
FLOWSE = dict(model_type="flowse", ema_decay=0.999, sigma_max=0.5, sigma_min=0.05, t_eps=0.03, T_rev=1.0, loss_type="mse",
              loss_abs_exponent=0.5, n_fft=1536, hop_length=384, spec_transform_type="exponent", spec_abs_exponent=0.667,
              spec_factor=0.065, bsrnn_hidden=384, num_layer=6, learning_rate=1e-4)          # BSRNN_flowse.yaml:31-53


def flops_per_token(N, H, layers, subbands, F_bins, K):
    """Forward multiply-adds x 2 per (frame, band) token, from shapes: the 2 x layers (BLSTM + Linear(2H -> N)) blocks, the
    condition Linear(2N -> N), both BandSplits (Conv1d(2 s_k -> N) per band), and the GradDecoder (Conv1d(N -> 16 s_k)
    per band and family, Conv2d(16 -> 4, 5 x 5) per bin and family).  SURVEY §8d config 4: ~185 MFLOP."""
    block = 2 * (2 * 4 * H * (N + H)) + 2 * 2 * H * N
    per_frame = 2 * sum(2 * 2 * s * N for s in subbands[:K])                    # band_split_x + band_split_y
    per_frame += 2 * sum(2 * N * 16 * s for s in subbands[:K])                  # mask + residual Conv1d
    per_frame += 2 * 2 * 16 * 4 * 25 * sum(subbands[:K])                        # mask + residual Conv2d
    return 2 * layers * block + 2 * 2 * N * N + per_frame / K


def device_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
        name, power, clock = [v.strip() for v in out[int(os.environ.get("LOCAL_RANK", 0)) % len(out)].split(",")]
        return {"name": name, "power_limit": power, "max_sm_clock": clock}
    except Exception as e:                       # report what is missing rather than guess
        return {"name": torch.cuda.get_device_name(), "power_limit": None, "max_sm_clock": None, "nvidia_smi": repr(e)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, default=4)
    ap.add_argument("--samples", type=int, default=96000)
    ap.add_argument("--steps", type=int, default=5, help="timed replays per trainer and round")
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--layers", type=int, default=6)
    ap.add_argument("--precision", default="fp16")
    a = ap.parse_args()
    rank, world, local = int(os.environ.get("RANK", 0)), int(os.environ.get("WORLD_SIZE", 1)), int(os.environ.get("LOCAL_RANK", 0))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    L.require_device()
    info = device_info()
    fs = 48000
    g = torch.Generator().manual_seed(1 + rank)
    clean = (0.05 * torch.randn(a.batch, 1, a.samples, generator=g)).to(dev)
    noisy = clean + (0.03 * torch.randn(a.batch, 1, a.samples, generator=g)).to(dev)
    lens = torch.full((a.batch,), a.samples, dtype=torch.int32)
    fs_t = torch.tensor(fs, dtype=torch.int32)

    def trainer(fused, graph=True):
        torch.manual_seed(0)
        m = FlowSEModel(Config(**dict(FLOWSE, num_layer=a.layers))).to(dev)
        if world > 1:
            for p in m.parameters():
                dist.broadcast(p.data, 0)
        tr = m.configure_optimizers(precision=a.precision, cuda_graph=graph)
        TT.FUSED_TRAIN = fused                   # read while the graph is captured: each graph keeps its forward
        for _ in range(2):
            tr.step(noisy, clean, lens, fs_t)
        torch.cuda.synchronize()
        return m, tr

    default_fused = TT.FUSED_TRAIN
    torch.cuda.reset_peak_memory_stats(dev)
    m_f, tr_f = trainer(True)
    peak_one = torch.cuda.max_memory_allocated(dev)
    m_s, tr_s = trainer(False)
    TT.FUSED_TRAIN = default_fused
    ms = {True: [], False: []}
    for _ in range(a.rounds):
        for fused, tr in ((True, tr_f), (False, tr_s)):
            if world > 1:
                dist.barrier()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(a.steps):
                tr.step(noisy, clean, lens, fs_t)
            e1.record()
            torch.cuda.synchronize()
            ms[fused].append(e0.elapsed_time(e1) / a.steps)
    best = {k: min(v) for k, v in ms.items()}

    # eager split of the default trainer's step (host launches: the forward / backward boundary is visible)
    tr_f.cuda_graph = False
    ev = lambda: torch.cuda.Event(enable_timing=True)
    split = {"forward": [], "backward": [], "optimizer": []}
    launches = 0
    for _ in range(2):
        e = [ev() for _ in range(4)]
        L.lib().bsrnn_launch_count(1)            # reset the host-side counter of native launches
        e[0].record()
        tr_f.flat.zero_grad()
        loss, _ = tr_f.loss(noisy, clean, lens, fs_t)
        e[1].record()
        loss.backward()
        tr_f.flat.gather_grads()
        e[2].record()
        tr_f.apply_gradients()
        e[3].record()
        torch.cuda.synchronize()
        launches = L.lib().bsrnn_launch_count(0)
        for k, i in (("forward", 0), ("backward", 1), ("optimizer", 2)):
            split[k].append(e[i].elapsed_time(e[i + 1]))

    T = a.samples // 384 + 1
    from urgent2026_challenge_track1_b200.runtime import BandPlan
    plan = BandPlan.make(m_f.dnn.band_split_x.subbands, 1536 // 2 + 1)
    tokens = a.batch * T * plan.K
    fpt = flops_per_token(384, 768, a.layers, m_f.dnn.band_split_x.subbands, 1536 // 2 + 1, plan.K)
    step_flop = 3 * fpt * tokens
    peaks = {}
    pp = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(pp):
        peaks = json.load(open(pp))
    peak_tf = peaks.get("bf16_tflops_sustained", 1400.0)
    audio_s = a.batch * a.samples / fs
    fastest = min(best, key=best.get)
    res = {
        "what": "FlowSE training step (BSRNN_flowse: N=384, H=768, %d layers), fp16 tensor-core blocks, CUDA-graph replay" % a.layers,
        "device": info, "world": world, "batch_per_gpu": a.batch, "samples": a.samples, "fs": fs, "frames": T, "bands": plan.K,
        "tokens": tokens, "params": sum(p.numel() for p in m_f.parameters()),
        "ms_per_step": {"fused_forward": best[True], "stepwise_forward": best[False]},
        "ms_per_step_rounds": {"fused_forward": ms[True], "stepwise_forward": ms[False]},
        "faster_forward": "fused" if fastest else "stepwise",
        "audio_s_per_s": {"fused_forward": world * audio_s / (best[True] / 1e3), "stepwise_forward": world * audio_s / (best[False] / 1e3)},
        "eager_split_ms": {k: min(v) for k, v in split.items()},
        "native_launches_per_eager_step": launches,
        "peak_memory_gb": {"one_trainer": peak_one / 1e9, "both_trainers": torch.cuda.max_memory_allocated(dev) / 1e9},
        "mflop_per_token_forward": fpt / 1e6, "tflop_per_step": step_flop / 1e12,
        "achieved_tflops": {k: step_flop / (v / 1e3) / 1e12 for k, v in (("fused_forward", best[True]), ("stepwise_forward", best[False]))},
        "share_of_sustained_peak": {k: step_flop / (v / 1e3) / 1e12 / peak_tf for k, v in (("fused_forward", best[True]), ("stepwise_forward", best[False]))},
        "peak_tflops": peak_tf,
        "peak_source": "MEASURED_PEAKS.json (bf16_tflops_sustained)" if peaks else "fallback (B200_PROFILING.md), as bench.py",
    }
    if rank == 0:
        print(json.dumps(res), flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
