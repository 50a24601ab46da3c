"""Times the tcgen05 GEMM alone at BASELINE config-2 shapes (input projection / Linear+skip), for ncu and A/B runs.

  python tools/prof_gemm.py --which inproj --axis time [--reps 5]
"""
import argparse, os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
from urgent2026_challenge_track1_b200 import runtime_tc as tc, _lib as L

ap = argparse.ArgumentParser()
ap.add_argument("--which", default="inproj", choices=["inproj", "fc"])
ap.add_argument("--axis", default="time"); ap.add_argument("--reps", type=int, default=5)
ap.add_argument("--tma", action="store_true", help="fc: residual rows through the TMA unit (epilogue 8)")
ap.add_argument("--nobias", action="store_true", help="inproj: bias folded into the weights (bias pointer NULL)")
ap.add_argument("--B", type=int, default=64); ap.add_argument("--T", type=int, default=1001); ap.add_argument("--K", type=int, default=34)
a = ap.parse_args()
B, T, K, N = a.B, a.T, a.K, 196
if a.axis == "time":
    R, steps, addr = B * K, T, (K, T * K, 1, K)
else:
    R, steps, addr = B * T, K, (1, K, 0, 1)
tiles = (R + 127) // 128
ntile = steps * tiles
M = B * T * K
st = L.stream_ptr()
dev = "cuda"
torch.manual_seed(0)
if a.which == "inproj":
    kc = 26
    A = (torch.randn(ntile * kc * 1024, device=dev) * 0.5).half()
    W = (torch.randn(16 * kc * 208 * 8, device=dev) * 0.05).half()
    bias = torch.randn(16 * 208, device=dev)
    out = torch.empty(ntile * 416 * 1024, dtype=torch.float16, device=dev)
    run = lambda: L.call("bsrnn_gemm_tc", A.data_ptr(), W.data_ptr(), None if a.nobias else bias.data_ptr(), out.data_ptr(), None, ntile, 16, kc, 208,
                         L.TC_F16_KB8, 0, 3328, 416, T * K, tiles, R, *addr, st)
    bytes_alg = A.numel() * 2 + out.numel() * 2
    flops = 2.0 * ntile * 128 * 208 * 3328
else:
    kc = 100
    A = torch.empty(ntile * kc * 1024, dtype=torch.float16, device=dev)
    for i in range(0, A.numel(), 1 << 26):
        n = min(1 << 26, A.numel() - i)
        A[i:i + n] = (torch.randn(n, device=dev) * 0.3).half()
    W = (torch.randn(kc * 208 * 8, device=dev) * 0.03).half()
    bias = torch.randn(208, device=dev)
    out = torch.randn(B, T, K, N, device=dev)
    stats = torch.zeros(B, 2, dtype=torch.float64, device=dev)
    run = lambda: L.call("bsrnn_gemm_tc", A.data_ptr(), W.data_ptr(), bias.data_ptr(), out.data_ptr(), stats.data_ptr(), ntile, 1, kc,
                         208, L.TC_RESID_TMA if a.tma else L.TC_RESID_F32, N, N, 0, T * K, tiles, R, *addr, st)
    bytes_alg = A.numel() * 2 + 2 * out.numel() * 4
    flops = 2.0 * ntile * 128 * 800 * 208
run(); torch.cuda.synchronize()
for _ in range(a.reps):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(); run(); e1.record(); torch.cuda.synchronize()
    ms = e0.elapsed_time(e1)
    print(f"[gemm {a.which} {a.axis}{' nobias' if a.nobias else ''}{' tma' if a.tma else ''}] {ms:.3f} ms  {bytes_alg / ms / 1e6:.0f} GB/s algorithmic  {flops / ms / 1e9:.0f} TFLOP/s", flush=True)
