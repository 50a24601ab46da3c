#!/usr/bin/env python
"""bench.py — BSRNN audio-seconds enhanced per second at 48 kHz (BASELINE.json metric) on N B200s of one node.

  python bench.py --gpus 1 --steps K --warmup W            # our arm (libbsrnn_b200 through the C ABI), BASELINE config 2
  python bench.py --impl reference ...                     # the reference's own CPU path on the box's host cores
  torchrun --nproc-per-node N ... bench.py --gpus N ...    # one rank per GPU, utterances sharded, no collective
  python bench.py --config 3|4|5 ...                       # sample-rate sweep | FlowSE 32x10 s NFE 15 | training step
  python bench.py ... --dump-outputs DIR                   # + what the last timed step computed (rank 0), DIR/<name>.npy

Config 2 (default, the headline): a step = one BSRNN_SE forward (STFT -> BandSplit -> 6x[time BLSTM, band BLSTM] ->
MaskDecoder -> mask+iSTFT) over one batch of synthetic noisy utterances with random-init BSRNN_baseline.yaml weights
(N=196, 6 layers).  `value` times the forward with inputs resident in HBM; `e2e` times the public call path with pinned
HOST buffers, H2D of the waveforms and D2H of the enhanced waveforms inside the timed region.  Under torchrun the
primary number keeps 64 utterances PER GPU ("weak"); the partition BASELINE.json names -- 64 utterances sharded 64/G
per GPU -- is measured in the same run and reported under "strong" (or made the headline with --scaling strong).
At N=1 the line also carries `cpu_baseline` (the reference's CPU path on the host cores), `library_baseline` (the
reference's own modules on this GPU under stock torch eager: cuDNN LSTM / cuBLAS / cuFFT -- the bar the kernels must
beat) and `fp32_mode` (the f32 CUDA-core kernels).
"""
import argparse
import json
import os
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

FS = 48000
NUM_CHANNEL, NUM_LAYER = 196, 6                      # conf/models/BSRNN_baseline.yaml:36-38
METRIC, UNIT = "BSRNN audio-sec/sec enhanced at 48 kHz", "audio-s/s"
RATES = (8000, 16000, 22050, 24000, 32000, 44100, 48000)          # SURVEY.md §8d cfg3
DUMP_BYTES = 60_000_000                              # --dump-outputs: data of all arrays together (64 MB with the headers)


def dump_outputs(out_dir, arrays):
    """--dump-outputs: {name: tensor} -> out_dir/<name>.npy, so that two builds can be compared output for output.
    Complex tensors get a trailing (re, im) axis; float64 stays float64, everything else is written as float32.  When
    the arrays together hold more than DUMP_BYTES, each keeps the same fraction of its elements, flattened to 1-D: the
    sorted distinct flat indices drawn by numpy's default_rng(0).  They depend on the array's size and on the total
    size of all the arrays, so runs with the same arguments write the same elements.  Files of the same names are
    overwritten; other files already in out_dir are left as they are."""
    import numpy as np
    arrays = {k: torch.view_as_real(t.detach()) if t.is_complex() else t.detach() for k, t in arrays.items()}
    arrays = {k: t if t.dtype == torch.float64 else t.float() for k, t in arrays.items()}
    total = sum(t.numel() * t.element_size() for t in arrays.values())
    os.makedirs(out_dir, exist_ok=True)
    for name, t in arrays.items():
        if total > DUMP_BYTES:
            keep = max(1, t.numel() * DUMP_BYTES // total)
            idx = np.unique(np.random.default_rng(0).integers(0, t.numel(), size=keep))
            t = t.reshape(-1)[torch.from_numpy(idx).to(t.device)]
        np.save(os.path.join(out_dir, name + ".npy"), t.cpu().numpy())


def lstm_flops(tokens, N=NUM_CHANNEL, layers=NUM_LAYER):
    """2 x MACs of the weight GEMMs of the dual path (SURVEY.md §8d): per token-layer 4 directions x 4H(N+H) + 2 x 4N*N."""
    H = 2 * N
    return dict(lstm_rec=tokens * layers * 4 * (4 * H * H) * 2, lstm_in=tokens * layers * 4 * (4 * H * N) * 2,
                fc=tokens * layers * 2 * (4 * N * N) * 2)


class ClockSampler(threading.Thread):
    """Samples SM clock + throttle reasons during the timed region (B200_PROFILING.md clocks line) via NVML."""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.samples, self.reasons, self.stop_flag, self.max_mhz = index, [], set(), False, None
        self.times = []

    def run(self):
        try:
            import pynvml as nv
            nv.nvmlInit()
            h = nv.nvmlDeviceGetHandleByIndex(self.index)
            self.max_mhz = nv.nvmlDeviceGetMaxClockInfo(h, nv.NVML_CLOCK_SM)
            names = {nv.nvmlClocksEventReasonSwPowerCap: "sw_power_cap", nv.nvmlClocksThrottleReasonHwSlowdown: "hw_slowdown",
                     nv.nvmlClocksThrottleReasonHwThermalSlowdown: "hw_thermal_slowdown",
                     nv.nvmlClocksThrottleReasonSwThermalSlowdown: "sw_thermal_slowdown"}
            while not self.stop_flag:
                self.samples.append(nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM))
                self.times.append(time.monotonic())
                r = nv.nvmlDeviceGetCurrentClocksEventReasons(h)
                for bit, name in names.items():
                    if r & bit:
                        self.reasons.add(name)
                time.sleep(0.1)
        except Exception as e:  # noqa: BLE001
            self.reasons.add(f"nvml_error:{type(e).__name__}")

    def median(self, t0=None, t1=None):
        s = sorted(v for v, t in zip(self.samples, self.times) if (t0 is None or t >= t0) and (t1 is None or t <= t1))
        return s[len(s) // 2] if s else None

    def summary(self, t0=None, t1=None, t2=None):
        """sm_mhz: median over [t0, t1] (the device-resident timed loop); sm_mhz_e2e: over [t1, t2]."""
        return {"sm_mhz": self.median(t0, t1), "sm_mhz_e2e": self.median(t1, t2), "sm_max_mhz": self.max_mhz,
                "reasons": sorted(self.reasons)}

    def finish(self):
        self.stop_flag = True
        if self.is_alive():
            self.join(timeout=2)


# ---------------------------------------------------------------------------------------------------- reference legs
def _reference_module():
    """The reference's own BSRNN_SE (verbatim files from /root/reference or the oracle/_ref snapshot, on the espnet2
    shim) when importable -> (module, 'reference'); else the oracle port as a callable -> (callable, 'port')."""
    from oracle import ref_loader
    torch.manual_seed(0)
    if ref_loader.available():
        ns = ref_loader.load()
        return ns.BSRNN_SE(num_channel=NUM_CHANNEL, num_layer=NUM_LAYER).eval(), "reference"
    from oracle import restated as R
    from urgent2026_challenge_track1_b200.bsrnn import BSRNN_SE
    sd = BSRNN_SE(NUM_CHANNEL, NUM_LAYER).state_dict()
    return (lambda x, lens, fs: R.bsrnn_se_forward(sd, x, lens, fs, NUM_LAYER)), "port"


def cpu_reference_throughput(seconds, threads, steps=3, warmup=1):
    """The reference's CPU path on the box's host cores (SURVEY.md §8d: torch.no_grad, all cores, 1 warm-up + 3 runs of
    one 10 s @48 kHz utterance; the 64-utterance batch of config 2 is 64 such independent units).
    -> (audio_s_per_s, cores, sample description, kind)."""
    from urgent2026_challenge_track1_b200.synth import synth_noisy
    torch.set_num_threads(threads)
    model, kind = _reference_module()
    n = int(seconds * FS)
    x = synth_noisy(1, n, FS)
    lens = torch.tensor([n])
    with torch.no_grad():
        for _ in range(warmup):
            model(x, lens, FS)
        t0 = time.perf_counter()
        for _ in range(steps):
            model(x, lens, FS)
        dt = (time.perf_counter() - t0) / steps
    what = "the reference's own baseline_code files (verbatim) on the espnet2 shim" if kind == "reference" else "oracle port"
    return seconds / dt, threads, f"1x{seconds:g}s@48kHz utterance, f32, {steps} run(s) after {warmup} warm-up; {what}", kind


def library_baseline(x_dev, lens, steps=2):
    """The reference's modules moved to this GPU under stock torch eager (cuDNN LSTM, cuBLASLt, cuFFT) on the SAME
    batch: TF32 matmuls (what train_se.py:39 'medium' precision allows) and fp16 autocast.  SURVEY.md §2.1 / BASELINE.md
    §3: this, not the CPU, is the bar for the kernels."""
    out = {}
    try:
        model, kind = _reference_module()
        if kind != "reference":
            return {"unavailable": "verbatim reference files not present (oracle/_ref missing)"}
        model = model.to(x_dev.device)
        lens_d = lens.to(x_dev.device)
        audio_s = float(lens.sum()) / FS
        old = torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.allow_tf32
        for name, tf32, amp in (("tf32", True, False), ("fp16_autocast", True, True), ("fp32", False, False)):
            torch.backends.cuda.matmul.allow_tf32 = torch.backends.cudnn.allow_tf32 = tf32
            try:
                with torch.no_grad(), torch.autocast("cuda", dtype=torch.float16, enabled=amp):
                    model(x_dev, lens_d, FS)
                    torch.cuda.synchronize()
                    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    e0.record()
                    for _ in range(steps):
                        model(x_dev, lens_d, FS)
                    e1.record()
                    torch.cuda.synchronize()
                ms = e0.elapsed_time(e1) / steps
                out[name] = {"value": audio_s / (ms / 1e3), "ms_per_step": ms}
            except Exception as e:  # noqa: BLE001  (e.g. out of memory at this batch in one of the modes)
                out[name] = {"unavailable": f"{type(e).__name__}: {str(e)[:120]}"}
                torch.cuda.empty_cache()
        torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.allow_tf32 = old
        out.update(unit=UNIT, impl="reference modules (verbatim baseline_code + espnet2 shim) on cuda, stock torch "
                   f"{torch.__version__} eager: cuDNN LSTM, cuBLAS, cuFFT", batch=int(x_dev.shape[0]), steps=steps)
        del model
        torch.cuda.empty_cache()
    except Exception as e:  # noqa: BLE001
        out = {"unavailable": f"{type(e).__name__}: {str(e)[:160]}"}
    return out


_JSON_FD = None


def _claim_stdout():
    """The contract is ONE JSON line on stdout.  Libraries write there too (NCCL prints its version banner on fd 1 when
    the box sets NCCL_DEBUG): keep a private duplicate of the real stdout for the JSON line and point fd 1 at stderr."""
    global _JSON_FD
    if _JSON_FD is None:
        sys.stdout.flush()
        _JSON_FD = os.dup(1)
        os.dup2(2, 1)


def _emit(obj):
    data = (json.dumps(obj) + "\n").encode()
    if _JSON_FD is None:
        sys.stdout.write(data.decode()); sys.stdout.flush()
    else:
        os.write(_JSON_FD, data)


def workload_config(args):
    """`config` of the JSON line: names the WORKLOAD only, identical for our arm and the reference arm."""
    if args.config == 2:
        return {"workload": f"BASELINE config 2: BSRNN_baseline (N=196, L=6) inference, {args.batch}x{args.seconds:g}s@48kHz "
                            "synthetic utterances", "baseline_config": 2, "weights": "random-init seed 0",
                "sharding": "utterances over ranks, no data-path collective"}
    if args.config == 3:
        return {"workload": "BASELINE config 3: BSRNN_baseline inference, sample-rate sweep 8/16/22.05/24/32/44.1/48 kHz, per "
                            f"rate one {args.sweep_batch}x{args.seconds:g}s batch + one ragged batch ({args.seconds:g}..{0.6 * args.seconds:g} s)",
                "baseline_config": 3, "weights": "random-init seed 0", "sharding": "rates over ranks, no collective"}
    if args.config == 4:
        return {"workload": f"BASELINE config 4: BSRNN_flowse (N=384, L=6) generative inference, {args.flow_batch}x{args.seconds:g}s@48kHz, "
                            f"{args.nfe} Euler steps", "baseline_config": 4, "weights": "random-init seed 0",
                "sharding": "utterances over ranks, no data-path collective"}
    return {"workload": f"BASELINE config 5: BSRNN_baseline training step, B={args.train_batch} x {args.train_samples} samples @48kHz per GPU, "
                        "fwd + MultiResL1SpecLoss + bwd + gradient allreduce + clip + AdamW", "baseline_config": 5,
            "weights": "random-init seed 0", "sharding": "data parallel, one NCCL allreduce of the flat gradient buffer"}


class Ctx:
    def __init__(self, args):
        self.args = args
        self.rank = int(os.environ.get("RANK", "0"))
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        self.local_rank = int(os.environ.get("LOCAL_RANK", "0"))
        self.cores = os.cpu_count() or 1
        self.peaks = {}
        pp = os.path.join(ROOT, "MEASURED_PEAKS.json")
        if os.path.exists(pp):
            self.peaks = json.load(open(pp))
        self.peak_tf = self.peaks.get("bf16_tflops_sustained", 1400.0)
        self.hbm_peak = self.peaks.get("hbm_gbs", 6650.0)
        self.peak_source = "MEASURED_PEAKS.json (bf16_tflops_sustained, hbm_gbs)" if self.peaks else "fallback (B200_PROFILING.md)"

    def init_device(self):
        import torch.distributed as dist
        from urgent2026_challenge_track1_b200 import _lib
        torch.cuda.set_device(self.local_rank)
        self.dev = torch.device("cuda", self.local_rank)
        if self.world > 1:
            dist.init_process_group("nccl", device_id=self.dev)
        _lib.require_device()
        self.lib = _lib.lib()

    def barrier(self):
        if self.world > 1:
            import torch.distributed as dist
            dist.barrier()
        torch.cuda.synchronize()

    def gather(self, values):
        """per-rank float list -> (world, len) tensor on the CPU (the only exchange of the inference benches)."""
        mine = torch.tensor(values, dtype=torch.float64, device=self.dev)
        rows = [mine]
        if self.world > 1:
            import torch.distributed as dist
            rows = [torch.zeros_like(mine) for _ in range(self.world)]
            dist.all_gather(rows, mine)
        return torch.stack(rows).cpu()

    def finish(self):
        if self.world > 1:
            import torch.distributed as dist
            dist.destroy_process_group()


def timed_forward(ctx, model, x_dev, lens, steps, warmup, graph=True):
    """W warm-up + K timed replays of the product path on a device-resident batch -> ms for K steps (this rank)."""
    model.cuda_graph = graph
    for _ in range(max(1, warmup)):
        model(x_dev, lens, FS)
    ctx.barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        model(x_dev, lens, FS)
    e1.record()
    ctx.barrier()
    return e0.elapsed_time(e1)


def timed_e2e(ctx, model, host, lens, steps, fs=FS):
    """K steps through pipeline.StreamedEnhancer (the package's batched front-end, used by inference.py): every step
    copies its input batch from pinned host memory and its enhanced waveforms back to pinned host memory inside the
    timed region -> (ms, h2d bytes per step, d2h bytes per step)."""
    from urgent2026_challenge_track1_b200.pipeline import StreamedEnhancer
    enh = StreamedEnhancer(model)
    for _ in enh.run((host, lens, fs) for _ in range(2)):          # untimed: allocates the staging / pinned slots
        pass
    ctx.barrier()
    enh.h2d_bytes = enh.d2h_bytes = 0
    f0, f1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    f0.record()
    n_out = 0
    for out, _, _ in enh.run((host, lens, fs) for _ in range(steps)):
        n_out += out.shape[0]                                      # result is complete in pinned host memory here
    f1.record()
    ctx.barrier()
    assert n_out == host.shape[0] * steps
    return f0.elapsed_time(f1), enh.h2d_bytes // steps, enh.d2h_bytes // steps


# ---------------------------------------------------------------------------------------------------- config 2
def run_config2(ctx, args):
    from urgent2026_challenge_track1_b200 import BSRNN_SE, runtime, runtime_tc as TC
    from urgent2026_challenge_track1_b200.sharding import shard_batch
    from urgent2026_challenge_track1_b200.synth import synth_batch
    rank, world, dev = ctx.rank, ctx.world, ctx.dev
    torch.manual_seed(0)
    model = BSRNN_SE(NUM_CHANNEL, NUM_LAYER, precision=args.precision).to(dev)
    n = int(args.seconds * FS)
    B_weak = args.batch                                       # 64 utterances on every GPU
    first, B_strong = shard_batch(args.batch, rank, world)    # 64 utterances split over the GPUs (BASELINE config 2)
    primary = args.scaling
    B = B_weak if primary == "weak" else B_strong
    host = synth_batch(B_weak, n, FS, seed=1 + rank).pin_memory()
    lens_all = torch.full((B_weak,), n, dtype=torch.int32)
    host_p, lens = host[:B], lens_all[:B]
    x_dev = host_p.to(dev)

    # setup, in this order so that the GPU is under continuous load from the region passes to the timed loop (a 1 kW
    # part that goes idle -> full load overshoots its power cap and clocks down for about a second):
    #   1. one eager forward (packs weights, sizes workspaces) and, for the product path, the CUDA-graph capture;
    #   2. REGION_PASSES eager forwards with per-region CUDA events (roofline leg; averaged) + the kernel count;
    #   3. W warm-up steps of the product path, barrier, K timed steps.
    model(x_dev, lens, FS)
    ctx.barrier()
    if not args.no_graph:
        model.cuda_graph = True
        model(x_dev, lens, FS)                               # capture (+ first replay)
        ctx.barrier()
        model.cuda_graph = False
    REGION_PASSES = 3
    ctx.lib.bsrnn_launch_count(1)
    with runtime.Profile() as prof:
        for _ in range(REGION_PASSES):
            model(x_dev, lens, FS)
        ctx.barrier()
        regions = {k: (v[0] / REGION_PASSES, v[1] // REGION_PASSES) for k, v in prof.totals_ms().items()}
    launches_per_step = ctx.lib.bsrnn_launch_count(0) // REGION_PASSES
    sampler = ClockSampler(ctx.local_rank)
    if os.environ.get("BSRNN_BENCH_NO_NVML", "0") != "1":
        sampler.start()
    model.cuda_graph = not args.no_graph
    for _ in range(args.warmup):
        model(x_dev, lens, FS)
    ctx.barrier()
    t_a = time.monotonic()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(args.steps):
        wav, spec = model(x_dev, lens, FS)
    e1.record()
    ctx.barrier()
    t_b = time.monotonic()
    ms = e0.elapsed_time(e1)
    outputs = {"wav": wav, "spec": spec}                     # fresh tensors: later calls do not overwrite them
    ms_e2e, h2d, d2h = timed_e2e(ctx, model, host_p, lens, args.steps)
    t_c = time.monotonic()

    # the other partition of the same 64-utterance workload, same run (N > 1 only: at N = 1 the two coincide)
    other = None
    if world > 1:
        B2 = B_strong if primary == "weak" else B_weak
        h2, l2 = host[:B2], lens_all[:B2]
        x2 = h2.to(dev)
        model.cuda_graph = False
        model(x2, l2, FS)                                    # sizes the workspaces of this shape
        ms2 = timed_forward(ctx, model, x2, l2, args.steps, args.warmup, graph=not args.no_graph)
        ms2_e2e, _, _ = timed_e2e(ctx, model, h2, l2, args.steps)
        other = (B2, ms2, ms2_e2e)
    sampler.finish()
    clk = sampler.summary(t_a, t_b, t_c)

    vals = [ms, ms_e2e, float(clk["sm_mhz"] or 0), float(B)] + ([other[1], other[2], float(other[0])] if other else [])
    per_rank = ctx.gather(vals)
    ms, ms_e2e = float(per_rank[:, 0].max()), float(per_rank[:, 1].max())      # max over ranks
    utts = float(per_rank[:, 3].sum())
    audio_s = utts * args.seconds * args.steps
    value, e2e = audio_s / (ms / 1e3), audio_s / (ms_e2e / 1e3)
    if rank != 0:
        return
    T, K = 1 + n // 480, 34
    fl = lstm_flops(B * T * K)
    rec_ms, rec_calls = regions.get("lstm_time", (0.0, 0))
    rec_ms_b, rec_calls_b = regions.get("lstm_freq", (0.0, 0))
    # dominant kernel family: the BLSTM recurrence (60 % of algorithmic FLOPs); one "launch" = one BLSTM layer call
    # With the fused layer kernel (runtime_tc.FUSED_AXES, the default) a launch also contains the input projection
    # x W_ih^T: its algorithmic FLOPs count for that axis.
    calls = max(1, rec_calls + rec_calls_b)
    fused_axes = TC.FUSED_AXES if args.precision != "fp32" else ()
    fl_axis = {ax: (fl["lstm_rec"] + (fl["lstm_in"] if ax in fused_axes else 0)) / (2 * NUM_LAYER) for ax in ("time", "freq")}
    flops_per_call = (fl_axis["time"] * rec_calls + fl_axis["freq"] * rec_calls_b) / calls
    achieved = flops_per_call / ((rec_ms + rec_ms_b) / calls / 1e3) / 1e12 if rec_ms + rec_ms_b > 0 else 0.0
    per_axis = {}
    for ax, (m_, c_) in (("time", (rec_ms, rec_calls)), ("freq", (rec_ms_b, rec_calls_b))):
        if m_ > 0:
            tf = fl_axis[ax] / (m_ / c_ / 1e3) / 1e12
            per_axis[ax] = {"ms_per_launch": m_ / c_, "achieved": tf, "frac": tf / ctx.peak_tf, "fused_input_projection": ax in fused_axes,
                            "algorithmic_flops_per_launch": fl_axis[ax]}
    # ncu --set full capture of the recurrence kernel at this workload: dram__bytes_read.sum + dram__bytes_write.sum per
    # launch, committed under profiles/ (traffic.json names the source file)
    traffic = None
    for rnd in ("r02", "r01"):
        tp = os.path.join(ROOT, "profiles", rnd, "traffic.json")
        if os.path.exists(tp) and B == 64 and args.seconds == 10.0:
            tj = json.load(open(tp))
            traffic = tj.get("blstm_fused" if fused_axes else "blstm_recurrence", tj.get("blstm_recurrence", {})).get("dram_bytes_per_launch")
            break
    # memory-bound kernel families (SURVEY.md §8d): algorithmic bytes per call at this workload / measured time
    tok = B * T * K
    kb = lambda kc: tok * kc * 16                                   # bytes of a KB8 fp16 operand with kc k-cores
    wav_b, spec_b = B * n * 4, B * T * 481 * 8
    alg = {"inproj": kb(26) + kb(400), "fc": kb(100) + 2 * tok * NUM_CHANNEL * 4, "norm": tok * NUM_CHANNEL * 4 + kb(26),
           "stft": wav_b + spec_b, "istft": spec_b + wav_b, "bandsplit": spec_b + tok * NUM_CHANNEL * 4}
    others = {}
    for name, nbytes in alg.items():
        ms_r, n_r = regions.get(name, (0.0, 0))
        if ms_r > 0:
            gbs = nbytes * n_r / (ms_r / 1e3) / 1e9
            others[name] = {"bound": "hbm", "achieved": gbs, "peak": ctx.hbm_peak, "unit": "GB/s", "frac": gbs / ctx.hbm_peak,
                            "algorithmic_bytes_per_call": nbytes, "calls": n_r}
    total_flops = sum(fl.values()) + 2 * B * T * (1.73e12 + 0.024e12) / (64 * 1001) / 2 * 2 / 2   # + mask decoder, band split
    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": primary, "vs_baseline": None,
        "dtype": "f32" if args.precision == "fp32" else "fp16", "data": "synthetic",
        "config": workload_config(args),
        "impl_notes": {"precision": args.precision, "utterances_per_gpu": B, "global_utterances": int(utts),
                       "l2": "inputs and activations larger than L2 (no flush needed)",
                       "launch": "host launches" if args.no_graph else "CUDA graph replay of the per-step kernel sequence",
                       "recurrence_schedule": ("fused layer kernel (CTA pairs + flag groups) on " + ",".join(fused_axes)) if fused_axes
                       else os.environ.get("BSRNN_LSTM_SCHED", "flag")},
        "e2e": {"value": e2e, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h},
        "gpu_launches": int(launches_per_step * args.steps),
        "clocks": clk,
        "per_rank": {"ms_per_step": [round(float(v) / args.steps, 3) for v in per_rank[:, 0]],
                     "e2e_ms_per_step": [round(float(v) / args.steps, 3) for v in per_rank[:, 1]],
                     "sm_mhz": [int(v) for v in per_rank[:, 2]], "utterances": [int(v) for v in per_rank[:, 3]]},
        "roofline": {"bound": "tensor", "kernel": "lstm_fused_kernel (BLSTM layer: input projection + recurrence)" if fused_axes
                     else "blstm_recurrence", "achieved": achieved, "peak": ctx.peak_tf,
                     "unit": "TFLOP/s", "frac": achieved / ctx.peak_tf, "traffic": traffic,
                     "algorithmic_flops_per_launch": flops_per_call, "launches_per_step": calls, "per_axis": per_axis,
                     "whole_step": {"algorithmic_tflop": total_flops / 1e12,
                                    "achieved": total_flops / (ms / args.steps / 1e3) / 1e12,
                                    "frac": total_flops / (ms / args.steps / 1e3) / 1e12 / ctx.peak_tf},
                     "other_kernels": others, "peak_source": ctx.peak_source,
                     "regions_ms_per_step": {k: v[0] for k, v in regions.items()}},
    }
    if other is not None:
        B2s = float(per_rank[:, 6].sum())
        m2, m2e = float(per_rank[:, 4].max()), float(per_rank[:, 5].max())
        name = "strong" if primary == "weak" else "weak"
        line[name] = {"value": B2s * args.seconds * args.steps / (m2 / 1e3), "unit": UNIT,
                      "e2e": B2s * args.seconds * args.steps / (m2e / 1e3), "ms_per_step": m2 / args.steps,
                      "global_utterances": int(B2s), "utterances_per_gpu": [int(v) for v in per_rank[:, 6]],
                      "note": ("BASELINE config 2's partition: one 64-utterance batch sharded 64/G per GPU" if name == "strong"
                               else "64 utterances on every GPU")}
    if world == 1:                                           # reported at N=1 only (bounded samples, rank 0)
        if not args.no_cpu_baseline:
            v, c, sample, kind = cpu_reference_throughput(args.cpu_seconds, ctx.cores)
            line["cpu_baseline"] = {"value": v, "unit": UNIT, "cores": c, "kind": kind, "sample": sample}
        if not args.no_library_baseline:
            line["library_baseline"] = library_baseline(x_dev, lens)
        if not args.no_fp32 and args.precision != "fp32":
            m32 = BSRNN_SE(NUM_CHANNEL, NUM_LAYER, precision="fp32")
            m32.load_state_dict(model.state_dict())
            m32 = m32.to(dev)
            Bs = min(B, args.fp32_batch)
            xs, ls = x_dev[:Bs].contiguous(), lens[:Bs]
            m32(xs, ls, FS)
            ms32 = timed_forward(ctx, m32, xs, ls, 2, 1, graph=False)
            line["fp32_mode"] = {"value": Bs * args.seconds * 2 / (ms32 / 1e3), "unit": UNIT, "ms_per_step": ms32 / 2,
                                 "batch": Bs, "dtype": "f32", "note": "precision='fp32': CUDA-core f32 kernels for every op "
                                 "(parity ~1e-6 vs the reference); bounded batch"}
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, outputs)
    _emit(line)


# ---------------------------------------------------------------------------------------------------- config 3
def run_config3(ctx, args):
    """Mixed-sample-rate sweep (SURVEY.md §8d cfg3): per rate one full batch and one ragged batch; rates are dealt over
    the ranks; value = audio seconds of the whole sweep / device time of the whole sweep (max over ranks)."""
    from urgent2026_challenge_track1_b200 import BSRNN_SE
    from urgent2026_challenge_track1_b200.synth import synth_batch
    rank, world, dev = ctx.rank, ctx.world, ctx.dev
    torch.manual_seed(0)
    model = BSRNN_SE(NUM_CHANNEL, NUM_LAYER, precision=args.precision).to(dev)
    Bs = args.sweep_batch
    batches = []
    for fs in RATES[rank::world]:
        n = int(args.seconds * fs)
        x = synth_batch(Bs, n, fs, seed=fs).pin_memory()
        full = torch.full((Bs,), n, dtype=torch.int32)
        ragged = torch.tensor([int(n * (1.0 - 0.4 * i / max(1, Bs - 1))) for i in range(Bs)], dtype=torch.int32)
        batches += [(fs, x, full), (fs, x, ragged)]
    dev_batches = [(fs, x.to(dev), lens) for fs, x, lens in batches]
    # one host-launched pass: counts this rank's kernel launches per sweep (graph replays do not pass through the C ABI
    # counter) and the algorithmic FLOPs of the dual path (tokens = B x frames x bands of each batch)
    from urgent2026_challenge_track1_b200 import runtime as RT
    model.cuda_graph = False
    ctx.lib.bsrnn_launch_count(1)
    flops = 0.0
    for fs, x, lens in dev_batches:
        model(x, lens, fs)
        n_fft, hop = RT.stft_dims(fs, model.N_FFT, model.HOP, model.DEFAULT_FS)
        K = RT.BandPlan.make(model.bsrnn.bsrnn.band_split.subbands, n_fft // 2 + 1).K
        flops += sum(lstm_flops(x.shape[0] * (1 + x.shape[1] // hop) * K).values())
    torch.cuda.synchronize()
    launches_per_sweep = ctx.lib.bsrnn_launch_count(0)
    model.cuda_graph = not args.no_graph
    for _ in range(max(1, args.warmup)):
        for fs, x, lens in dev_batches:
            model(x, lens, fs)
    ctx.barrier()
    sampler = ClockSampler(ctx.local_rank)
    sampler.start()
    t_a = time.monotonic()
    per_batch = []
    outputs = {}
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(args.steps):
        for i, (fs, x, lens) in enumerate(dev_batches):
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record(); wav, spec = model(x, lens, fs); b.record()
            per_batch.append((fs, float(lens.sum()) / fs, a, b))
            kind = ("full", "ragged")[i % 2]
            outputs[f"wav_{fs}_{kind}"], outputs[f"spec_{fs}_{kind}"] = wav, spec
    e1.record()
    ctx.barrier()
    t_b = time.monotonic()
    ms = e0.elapsed_time(e1)
    # e2e: every batch from pinned host memory and back
    from urgent2026_challenge_track1_b200.pipeline import StreamedEnhancer
    enh = StreamedEnhancer(model)
    for _ in enh.run((x, lens, fs) for fs, x, lens in batches):
        pass
    ctx.barrier()
    enh.h2d_bytes = enh.d2h_bytes = 0
    f0, f1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    f0.record()
    for _ in range(args.steps):
        for _ in enh.run((x, lens, fs) for fs, x, lens in batches):
            pass
    f1.record()
    ctx.barrier()
    ms_e2e = f0.elapsed_time(f1)
    sampler.finish()
    clk = sampler.summary(t_a, t_b, time.monotonic())
    audio_rank = sum(float(lens.sum()) / fs for fs, _, lens in batches) * args.steps
    per_rank = ctx.gather([ms, ms_e2e, audio_rank, float(launches_per_sweep), flops])
    per_fs = {}
    for fs, secs, a, b in per_batch:
        d = per_fs.setdefault(fs, [0.0, 0.0])
        d[0] += secs; d[1] += a.elapsed_time(b)
    mine = torch.zeros(len(RATES), 2, dtype=torch.float64)
    for i, fs in enumerate(RATES):
        if fs in per_fs:
            mine[i] = torch.tensor(per_fs[fs])
    allfs = ctx.gather(mine.flatten().tolist()).view(world, len(RATES), 2).sum(0)
    if rank != 0:
        return
    audio = float(per_rank[:, 2].sum())
    ms, ms_e2e = float(per_rank[:, 0].max()), float(per_rank[:, 1].max())
    line = {"metric": METRIC.replace("at 48 kHz", "over the sample-rate sweep"), "value": audio / (ms / 1e3), "unit": UNIT,
            "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms / args.steps,
            "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
            "dtype": "f32" if args.precision == "fp32" else "fp16", "data": "synthetic", "config": workload_config(args),
            "e2e": {"value": audio / (ms_e2e / 1e3), "unit": UNIT, "h2d_bytes_per_step": enh.h2d_bytes // args.steps,
                    "d2h_bytes_per_step": enh.d2h_bytes // args.steps},
            "per_rate": {str(fs): {"audio_s_per_s": float(allfs[i, 0] / (allfs[i, 1] / 1e3)) if allfs[i, 1] > 0 else None,
                                   "ms": float(allfs[i, 1]) / args.steps} for i, fs in enumerate(RATES)},
            "clocks": clk, "gpu_launches": int(per_rank[:, 3].sum()) * args.steps,
            "roofline": {"bound": "tensor", "kernel": "whole sweep (fused BLSTM layer kernels, small-batch geometries)",
                         "achieved": float(per_rank[:, 4].sum()) * args.steps / (ms / 1e3) / 1e12, "peak": ctx.peak_tf * world,
                         "unit": "TFLOP/s", "frac": float(per_rank[:, 4].sum()) * args.steps / (ms / 1e3) / 1e12 / (ctx.peak_tf * world),
                         "traffic": None, "algorithmic_flops_per_step": float(per_rank[:, 4].sum()),
                         "note": "dual-path GEMM FLOPs (SURVEY 8d) of all batches of the sweep / device time; 8-utterance batches sit "
                                 "on the recurrence's per-step dependency chain, not on the tensor pipe",
                         "peak_source": "MEASURED_PEAKS.json (bf16_tflops_sustained)"},
            "impl_notes": {"precision": args.precision, "launch": "host launches" if args.no_graph else "CUDA graph per batch signature"}}
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, outputs)
    _emit(line)


# ---------------------------------------------------------------------------------------------------- config 4
def flowse_cfg(hidden=384, layers=6):
    from urgent2026_challenge_track1_b200.config import Config
    return Config(model_type="flowse", ema_decay=0.999, sigma_max=0.5, sigma_min=0.05, t_eps=0.03, T_rev=1.0,
                  loss_type="mse", loss_abs_exponent=0.5, n_fft=1536, hop_length=384, spec_transform_type="exponent",
                  spec_abs_exponent=0.667, spec_factor=0.065, bsrnn_hidden=hidden, num_layer=layers, learning_rate=1e-4)


def run_config4(ctx, args):
    """BSRNN_flowse generative inference (conf/models/BSRNN_flowse.yaml: N=384, 6 layers), 32 x 10 s @48 kHz, 15 Euler
    steps through FlowSEModel.enhance (flow_model.py:189-200).  A step = one whole enhance() of the batch."""
    from urgent2026_challenge_track1_b200.flow_model import FlowSEModel
    from urgent2026_challenge_track1_b200.sharding import shard_batch
    from urgent2026_challenge_track1_b200.synth import synth_batch
    rank, world, dev = ctx.rank, ctx.world, ctx.dev
    torch.manual_seed(0)
    m = FlowSEModel(flowse_cfg()).to(dev).eval(no_ema=True)
    m.dnn.precision = "fp32" if args.precision == "fp32" else "fp16"
    m.dnn.cuda_graph = not args.no_graph
    _, B = shard_batch(args.flow_batch, rank, world) if args.scaling == "strong" else (0, args.flow_batch)
    n = int(args.seconds * FS)
    host = synth_batch(B, n, FS, seed=5 + rank).pin_memory()
    lens = torch.full((B,), n, dtype=torch.int32)
    y = host.to(dev)
    ctx.lib.bsrnn_launch_count(1)
    for _ in range(max(1, args.warmup)):
        torch.manual_seed(2)
        m.enhance(y, FS, lens, N=args.nfe)
    ctx.barrier()
    launches_per_step = ctx.lib.bsrnn_launch_count(0) // max(1, args.warmup)
    sampler = ClockSampler(ctx.local_rank)
    sampler.start()
    t_a = time.monotonic()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(args.steps):
        enhanced = m.enhance(y, FS, lens, N=args.nfe)
    e1.record()
    ctx.barrier()
    t_b = time.monotonic()
    ms = e0.elapsed_time(e1)
    out_host = torch.empty(B, n, dtype=torch.float32).pin_memory()
    f0, f1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    f0.record()
    for _ in range(args.steps):
        out_host.copy_(m.enhance(host.to(dev, non_blocking=True), FS, lens, N=args.nfe), non_blocking=True)
    f1.record()
    ctx.barrier()
    ms_e2e = f0.elapsed_time(f1)
    sampler.finish()
    clk = sampler.summary(t_a, t_b, time.monotonic())
    per_rank = ctx.gather([ms, ms_e2e, float(B)])
    if rank != 0:
        return
    ms, ms_e2e, utts = float(per_rank[:, 0].max()), float(per_rank[:, 1].max()), float(per_rank[:, 2].sum())
    audio = utts * args.seconds * args.steps
    flops = 1.112e12 * args.seconds * args.nfe * B                      # SURVEY.md §8d: 1.112 TFLOP per audio-s per NFE
    tf = flops / (ms / args.steps / 1e3) / 1e12
    line = {"metric": "BSRNN_flowse audio-sec/sec enhanced at 48 kHz", "value": audio / (ms / 1e3), "unit": UNIT, "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms / args.steps, "higher_is_better": True,
            "scaling": args.scaling, "vs_baseline": None, "dtype": "f32" if args.precision == "fp32" else "fp16",
            "data": "synthetic", "config": workload_config(args),
            "e2e": {"value": audio / (ms_e2e / 1e3), "unit": UNIT, "h2d_bytes_per_step": B * n * 4, "d2h_bytes_per_step": B * n * 4},
            "gpu_launches": int(launches_per_step * args.steps), "clocks": clk,
            "roofline": {"bound": "tensor", "kernel": "whole enhance() (recurrence step kernels dominate)", "achieved": tf,
                         "peak": ctx.peak_tf, "unit": "TFLOP/s", "frac": tf / ctx.peak_tf, "traffic": None,
                         "algorithmic_flops_per_step": flops, "peak_source": ctx.peak_source},
            "impl_notes": {"utterances_per_gpu": B, "nfe": args.nfe,
                           "launch": "host launches" if args.no_graph else "one network evaluation per CUDA-graph replay"}}
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, {"enhanced": enhanced})
    _emit(line)


# ---------------------------------------------------------------------------------------------------- config 5
def run_config5(ctx, args):
    """Training step (train_se.py -> SEModel.training_step, d_model.py:61-113): B x 96 000 samples @48 kHz per GPU,
    forward + loss + backward + ONE NCCL allreduce of the flat gradient buffer + clip + AdamW."""
    from urgent2026_challenge_track1_b200 import BSRNN_SE
    from urgent2026_challenge_track1_b200.synth import synth_pair
    from urgent2026_challenge_track1_b200.training import SETrainer
    rank, world, dev = ctx.rank, ctx.world, ctx.dev
    torch.manual_seed(0)
    m = BSRNN_SE(NUM_CHANNEL, NUM_LAYER, precision="fp32").to(dev)
    tr = SETrainer(m, lr=1e-3, precision=args.train_precision, cuda_graph=not args.no_graph)
    B, ns = args.train_batch, args.train_samples
    clean_h, noisy_h = synth_pair(B, ns, FS, seed=1 + rank)
    clean_h, noisy_h = clean_h.view(B, 1, ns).pin_memory(), noisy_h.view(B, 1, ns).pin_memory()
    lens = torch.full((B,), ns, dtype=torch.int32)
    fs_t = torch.tensor(FS, dtype=torch.int32)
    clean, noisy = clean_h.to(dev), noisy_h.to(dev)
    ev = lambda: torch.cuda.Event(enable_timing=True)
    ctx.lib.bsrnn_launch_count(1)
    for _ in range(max(1, args.warmup)):
        tr.step(noisy, clean, lens, fs_t)
    ctx.barrier()
    launches_per_step = ctx.lib.bsrnn_launch_count(0) // max(1, args.warmup)
    sampler = ClockSampler(ctx.local_rank)
    sampler.start()
    t_a = time.monotonic()
    e0, e1 = ev(), ev()
    e0.record()
    for _ in range(args.steps):
        loss, sisnr = tr.step(noisy, clean, lens, fs_t)
    e1.record()
    ctx.barrier()
    t_b = time.monotonic()
    ms = e0.elapsed_time(e1)
    n_par = tr.flat.numel                                    # the passes below update the weights again: copy them now
    outputs = {"loss": loss, "sisnr": sisnr, "params": tr.flat.flat[:n_par].clone(), "grads": tr.flat.grad[:n_par].clone()}
    # split of one step (separate EAGER pass: host launches, so the forward / backward shares are upper bounds of what
    # the graph replay spends there)
    a0, a1, a2, a3, a4 = ev(), ev(), ev(), ev(), ev()
    tr.flat.zero_grad()
    a0.record(); l2, _ = tr.loss(noisy, clean, lens, fs_t); a1.record()
    l2.backward(); tr.flat.gather_grads(); a2.record()
    tr.allreduce_gradients(); a3.record()
    tr.apply_gradients(); a4.record()
    ctx.barrier()
    split = {"fwd_loss_ms": a0.elapsed_time(a1), "bwd_ms": a1.elapsed_time(a2), "allreduce_ms": a2.elapsed_time(a3),
             "allreduce_clip_adamw_ms": a3.elapsed_time(a4)}
    # e2e: the batch comes from pinned host memory and the loss goes back to the host every step
    f0, f1 = ev(), ev()
    f0.record()
    for _ in range(args.steps):
        loss, _ = tr.step(noisy_h.to(dev, non_blocking=True), clean_h.to(dev, non_blocking=True), lens, fs_t)
        loss_host = float(loss)
    f1.record()
    ctx.barrier()
    ms_e2e = f0.elapsed_time(f1)
    sampler.finish()
    clk = sampler.summary(t_a, t_b, time.monotonic())
    per_rank = ctx.gather([ms, ms_e2e])
    if rank != 0:
        return
    ms, ms_e2e = float(per_rank[:, 0].max()), float(per_rank[:, 1].max())
    audio = world * B * ns / FS * args.steps
    T = 1 + ns // 480
    flops = 3.0 * (sum(lstm_flops(B * T * 34).values()) + 1.75e12 * B * T / (64 * 1001))   # fwd + ~2x bwd (SURVEY §8d cfg5)
    tf = flops / (ms / args.steps / 1e3) / 1e12
    line = {"metric": "BSRNN_baseline training audio-sec/sec at 48 kHz", "value": audio / (ms / 1e3), "unit": UNIT, "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms / args.steps, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": getattr(tr, "precision", "f32"), "data": "synthetic",
            "config": workload_config(args),
            "e2e": {"value": audio / (ms_e2e / 1e3), "unit": UNIT, "h2d_bytes_per_step": 2 * B * ns * 4, "d2h_bytes_per_step": 4},
            "gpu_launches": int(launches_per_step * args.steps), "clocks": clk, "split_ms": split,
            "allreduce_bytes": int(tr.flat.grad.numel() * 4), "loss": loss_host,
            "roofline": {"bound": "tensor", "kernel": "whole training step", "achieved": tf, "peak": ctx.peak_tf, "unit": "TFLOP/s",
                         "frac": tf / ctx.peak_tf, "traffic": None, "algorithmic_flops_per_step": flops,
                         "peak_source": ctx.peak_source},
            "impl_notes": {"batch_per_gpu": B, "samples": ns, "precision": tr.precision,
                           "blstm": "forward: fused layer kernel with the activations for BPTT saved by its epilogue; backward: one "
                                    "tensor-core step kernel per time step, split-K weight-gradient GEMMs",
                           "launch": "host launches" if args.no_graph else "CUDA graph replay of forward + loss + backward; "
                                     "allreduce and the fused clip+AdamW tail eager"}}
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, outputs)
    _emit(line)


def reference_arm(ctx, args):
    """`--impl reference`: the reference's own CPU implementation of the path on the box's host cores, all threads, on
    a bounded sample of the workload (one 10 s @48 kHz utterance per step; config 2 is 64 such independent units).
    Rank 0 alone runs it; the other ranks exit 0."""
    if ctx.rank != 0:
        return
    v, c, sample, kind = cpu_reference_throughput(args.cpu_seconds, ctx.cores, steps=max(1, args.steps), warmup=min(args.warmup, 1))
    _emit({"impl": "reference", "metric": METRIC, "value": v, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
           "warmup": args.warmup, "ms_per_step": 1e3 * args.cpu_seconds / v, "higher_is_better": True, "scaling": args.scaling,
           "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": workload_config(args),
           "cpu_baseline": {"value": v, "unit": UNIT, "cores": c, "kind": kind, "sample": sample},
           "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}})


def main():
    _claim_stdout()
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=None)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--config", type=int, default=2, choices=[2, 3, 4, 5], help="BASELINE.json config (default 2, the headline)")
    ap.add_argument("--scaling", default="weak", choices=["weak", "strong"],
                    help="config 2/4 under torchrun: weak = the batch on every GPU, strong = the batch sharded B/G per GPU")
    ap.add_argument("--precision", default=os.environ.get("BSRNN_B200_PRECISION", "fp16"))
    ap.add_argument("--batch", type=int, default=64, help="config 2: utterances (BASELINE: 64)")
    ap.add_argument("--seconds", type=float, default=10.0)
    ap.add_argument("--cpu-seconds", type=float, default=10.0, help="length of the bounded CPU-baseline utterance (SURVEY §8d: 10 s)")
    ap.add_argument("--sweep-batch", type=int, default=8)
    ap.add_argument("--flow-batch", type=int, default=32)
    ap.add_argument("--nfe", type=int, default=15)
    ap.add_argument("--train-batch", type=int, default=4)
    ap.add_argument("--train-samples", type=int, default=96000)
    ap.add_argument("--train-precision", default="fp16", help="config 5: fp16 = BLSTM blocks fwd+bwd on tensor cores; fp32")
    ap.add_argument("--fp32-batch", type=int, default=8)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-library-baseline", action="store_true")
    ap.add_argument("--no-fp32", action="store_true")
    ap.add_argument("--no-graph", action="store_true", help="launch every kernel from the host instead of replaying the "
                    "per-step kernel sequence from a captured CUDA graph")
    ap.add_argument("--dump-outputs", metavar="DIR", help="after the timed steps, write what the last timed step computed "
                    "as DIR/<name>.npy (float32 / float64, at most 64 MB in all: a fixed seeded sample of larger outputs); "
                    "other files in DIR are kept, so give each run its own DIR")
    args = ap.parse_args()
    if args.steps is None:
        args.steps = {2: 3, 3: 2, 4: 1, 5: 5}[args.config]
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be >= 1 and --warmup >= 0")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes the outputs of --impl b200")
    ctx = Ctx(args)
    if args.impl == "reference":
        reference_arm(ctx, args)
        return
    ctx.init_device()
    {2: run_config2, 3: run_config3, 4: run_config4, 5: run_config5}[args.config](ctx, args)
    ctx.finish()


if __name__ == "__main__":
    main()
