"""Tensor-core training path of the BLSTM blocks (reference: autograd through nn.LSTM + nn.Linear inside
SEModel.training_step / FlowSEModel.training_step, d_model.py:61-95, flow_model.py:149-187, bsrnn_flowse.py:296-307;
SURVEY.md §8a rows a5, a6, a16).

``BLSTMBlockTC`` is one (BLSTM -> Linear(4N->N)) block as an autograd Function whose forward AND backward run on the
tcgen05 kernels of csrc/gemm_tc.cu with fp16 operands, f32 accumulation and f32 master weights / gradients:

  forward   x --norm_cast--> xhat (KB8) --gemm_tc--> input projection rows --[per step] bsrnn_blstm_step_train_tc-->
            h tiles (KB8), activated gates (in place of the projection), c_t --gemm_tc (residual epilogue)--> Linear output
  backward  d_out --norm_cast (x loss scale S)--> KB8 --gemm_tc--> dy rows --[per step] bsrnn_blstm_bwd_step_tc-->
            dG tiles (KB8) --gemm_tc_scaled--> dx ;  dW_ih = dG^T xhat, dW_hh = dG^T h_prev, dW_fc = d_out^T y through
            bsrnn_kb8_transpose (tokens become the K axis) + gemm_tc_scaled (1/S removed in f32).

The step-wise recurrence (one launch per time step, both directions) serves any hidden size with H % 8 == 0 (K padded to 16) -- the
same kernels serve BSRNN (H = 392) and FlowSE (H = 768).  At the two published widths the forward instead runs on the persistent
fused layer kernel (input projection + every step in one launch); BPTT stays step-wise.  Only bias gradients (two small reductions) use torch ops.
Gradients are loss-scaled by a power of two chosen per call from max|d_out| so that fp16 neither overflows nor flushes.
"""
from __future__ import annotations

import math
import os

import torch

from . import _lib as L
from .runtime_tc import to_kb8, FC_EPI, gate_row_map, lstm_ws, pack_steps, tile_width
from .runtime_tc import pack_fused as pack_fused_train      # the fused forward's weights: the inference layout, repacked per step

BIG = 1 << 40


def _bn_cover(rows, mult=16):
    """(BN, n_tiles) with BN a multiple of `mult` <= 256 and n_tiles * BN >= rows, fewest tiles then least padding."""
    nt = (rows + 255) // 256
    bn = ((rows + nt - 1) // nt + mult - 1) // mult * mult
    return bn, nt


NARROW_BN = int(os.environ.get("BSRNN_BWD_BN", "0"))      # 0 = automatic (see pack_block)


@torch.no_grad()
def pack_block(w_ih, w_hh, b_ih, b_hh, w_ih_r, w_hh_r, b_ih_r, b_hh_r, fc_w, narrow_bwd=False, fwd_steps=True):
    """All tensor-core operands of one block, from the f32 master weights (nn.LSTM / nn.Linear layouts).
    narrow_bwd: BPTT output tiles of 64 hidden units instead of up to 256 (few row tiles = small batch: more CTAs share a
    step and each epilogue warp owns a single 32-unit chunk).
    fwd_steps=False (the fused forward): the input operand carries the constant-one bias column N, so kc_in and the
    x^T tiles (bn_n x nt_n rows) cover N + 1 columns.  At N = 196 that column sits in the padding already; at N = 384
    it needs two more k-cores (kc_in = 50), and every operand built on kc_in (dD, fcT, xT) follows."""
    H, N = w_hh.shape[1], w_ih.shape[1]
    if H % 8:
        raise NotImplementedError(f"tensor-core training BLSTM needs H % 8 == 0, got {H}")
    kc_h = (H + 15) // 16 * 2                        # k-cores of an h tile: K padded to a multiple of 16, pad core = 0
    n_in = N if fwd_steps else N + 1                 # + the constant-one column of the fused forward's operand
    kc_in = (n_in + 15) // 16 * 2
    BN = tile_width(4 * H, 32)
    bn_h, nt_h = _bn_cover(H, 32)                    # BPTT output tiles over the H hidden units (32-column chunks)
    if narrow_bwd and H > 64:
        # one BPTT step is a single wave of tiles x ceil(H / bn) x 2 CTAs that each stream the whole 4H-wide dG tile: the narrowest
        # tile that still fits one wave of 148 SMs (config 5: 63.3 ms per step with 32, 68.0 with 64, 75.0 with 128; call74)
        bn_h = NARROW_BN if NARROW_BN > 0 else (32 if isinstance(narrow_bwd, int) and not isinstance(narrow_bwd, bool)
                                                 and 2 * narrow_bwd * ((H + 31) // 32) <= 148 else 64)
        nt_h = (H + bn_h - 1) // bn_h
    bn_n, nt_n = _bn_cover(n_in, 16)
    p = dict(H=H, N=N, kc_in=kc_in, kc_h=kc_h, BN=BN, n_tiles=4 * H // BN, bn_h=bn_h, nt_h=nt_h, bn_n=bn_n, nt_n=nt_n)
    if fwd_steps:                                      # operands of the step-wise forward (the fused forward packs its own)
        p.update(pack_steps((w_ih, w_hh, b_ih, b_hh, w_ih_r, w_hh_r, b_ih_r, b_hh_r), kc_in, BN))
    # BPTT: TRUE weights, rows of the step-wise layout transposed (rows = unit u / input n, K = packed gate column)
    perm = gate_row_map(H, 1, H, w_hh.device)[0][0]
    p.update(whhT=[to_kb8(wh.float()[perm].t(), bn_h, 4 * H // 8) for wh in (w_hh, w_hh_r)],
             wihT=[to_kb8(wi.float()[perm].t(), bn_n, 4 * H // 8) for wi in (w_ih, w_ih_r)])
    fw = fc_w.float()                                                                    # (N, 2H)
    n16 = (N + 15) // 16 * 16
    fc_bn = tile_width(n16, 16)
    p.update(fc_bn=fc_bn, fc_nt=n16 // fc_bn, fcw=[to_kb8(fw[:, :H], fc_bn, kc_h), to_kb8(fw[:, H:], fc_bn, kc_h)])
    bn_y = tile_width(2 * H, 16)
    p.update(bn_y=bn_y, nt_y=2 * H // bn_y, fcT=to_kb8(fw.t().contiguous(), bn_y, kc_in))   # rows = y column, K = n
    return p


# BLSTM forward of the training step on the fused layer kernel (bsrnn_blstm_fused_train_tc at H = 392,
# bsrnn_blstm_fused768_train_tc at H = 768 / N = 384): one persistent launch per block instead of one input-projection GEMM
# + one launch per time step.  BSRNN_TRAIN_FUSED=0: the step-wise forward.
FUSED_TRAIN = os.environ.get("BSRNN_TRAIN_FUSED", "1") == "1"


def _geom(B, T, K, axis):
    if axis == "time":
        R, steps, addr = B * K, T, (K, T * K, 1, K)
    else:
        R, steps, addr = B * T, K, (1, K, 0, 1)
    return R, steps, (R + 127) // 128, addr


def _cast_kb8(x, kcores, steps, tiles, R, addr, tokens_per_sample, scale=None):
    """(B,T,K,C) f32 token-major -> KB8 fp16 operand tiles in the axis' (step, sequence tile) order, optionally x scale."""
    C = x.shape[-1]
    out = torch.empty(steps * tiles * kcores * 1024, dtype=torch.float16, device=x.device)
    sc = sh = None
    if scale is not None:                            # python float or 0-dim device tensor
        if torch.is_tensor(scale):
            sc = scale.reshape(1, 1).expand(x.shape[0], C).contiguous()
        else:
            sc = torch.full((x.shape[0], C), float(scale), dtype=torch.float32, device=x.device)
        sh = torch.zeros_like(sc)
    L.call("bsrnn_norm_cast_kb8", x.data_ptr(), L.ptr(sc), L.ptr(sh), out.data_ptr(), C, 0, C, kcores, steps * tiles, tiles, R,
           *addr, tokens_per_sample, 1, L.stream_ptr())
    return out


def _transpose(src, src_m0, m_count, kc_src, BN, n_tiles, dst_kcores, dst_kc0, zero):
    dev = src.device
    alloc = torch.zeros if zero else torch.empty
    dst = alloc(n_tiles * dst_kcores * BN * 8, dtype=torch.float16, device=dev)
    L.call("bsrnn_kb8_transpose", src.data_ptr(), dst.data_ptr(), src_m0, m_count, kc_src, BN, n_tiles, dst_kcores, dst_kc0,
           L.stream_ptr())
    return dst


class BLSTMBlockTC(torch.autograd.Function):
    """out (B,T,K,N) = Linear(4N->N)(BLSTM_axis(x)) for a token-major x (B,T,K,N) f32 (already normalised)."""

    @staticmethod
    def forward(ctx, x, w_ih, w_hh, b_ih, b_hh, w_ih_r, w_hh_r, b_ih_r, b_hh_r, fc_w, fc_b, axis):
        L.require_device()
        B, T, K, N = x.shape
        dev = x.device
        st = L.stream_ptr()
        R, steps, tiles, addr = _geom(B, T, K, axis)
        Hh, Nn = w_hh.shape[1], w_ih.shape[1]
        fused = FUSED_TRAIN and ((Hh == 392 and Nn % 4 == 0 and Nn % 16 != 0) or (Hh == 768 and Nn == 384))
        with torch.profiler.record_function("tc_pack_block"):
            p = pack_block(w_ih, w_hh, b_ih, b_hh, w_ih_r, w_hh_r, b_ih_r, b_hh_r, fc_w, narrow_bwd=(tiles if tiles <= 16 else False),
                           fwd_steps=not fused)
        H, BN, nt = p["H"], p["BN"], p["n_tiles"]
        m_all = steps * tiles
        x = x.contiguous().float()
        gates = torch.empty(m_all * 128, 8 * H, dtype=torch.float16, device=dev)
        tile_halves = p["kc_h"] * 1024
        y = [torch.zeros(m_all * tile_halves, dtype=torch.float16, device=dev) for _ in range(2)]     # pad k-core stays 0
        c_all = [torch.empty(steps, tiles * 128, H, dtype=torch.float32, device=dev) for _ in range(2)]
        zero = torch.zeros(tiles * tile_halves, dtype=torch.float16, device=dev)
        assert not fused or N < p["kc_in"] * 8
        if fused:
            # x -> operand tiles with the constant-one column (the bias rides in the weights), then ONE persistent launch:
            # input projection + recurrence, activated gates and c_t saved by the epilogue for BPTT
            geo = 768 if H == 768 else 14 if (tiles + 1) // 2 <= 3 else 7
            xhat = torch.empty(m_all * p["kc_in"] * 1024, dtype=torch.float16, device=dev)
            L.call("bsrnn_norm_cast_kb8_ones", x.data_ptr(), None, None, xhat.data_ptr(), N, 0, N, p["kc_in"], m_all, tiles, R,
                   *addr, T * K, 1, N, st)
            wf = pack_fused_train((w_ih, w_hh, b_ih, b_hh, w_ih_r, w_hh_r, b_ih_r, b_hh_r), geo, p["kc_in"], N)
            sync = torch.empty(L.lib().bsrnn_blstm_fused_sync_bytes(), dtype=torch.uint8, device=dev)
            scratch = torch.empty(m_all * 128 * H * 24, dtype=torch.uint8, device=dev)      # bsrnn_blstm_fused*_train_scratch_bytes
            with torch.profiler.record_function("tc_fwd_fused"):
                if geo == 768:
                    L.call("bsrnn_blstm_fused768_train_tc", xhat.data_ptr(), wf.data_ptr(), zero.data_ptr(), y[0].data_ptr(),
                           y[1].data_ptr(), tile_halves, gates.data_ptr(), c_all[0].data_ptr(), c_all[1].data_ptr(),
                           scratch.data_ptr(), R, steps, tiles, 0, 0, sync.data_ptr(), st)
                else:
                    L.call("bsrnn_blstm_fused_train_tc", geo, xhat.data_ptr(), wf.data_ptr(), zero.data_ptr(), y[0].data_ptr(),
                           y[1].data_ptr(), tile_halves, gates.data_ptr(), c_all[0].data_ptr(), c_all[1].data_ptr(),
                           scratch.data_ptr(), R, steps, tiles, 0, 0, sync.data_ptr(), st)
        else:
            xhat = _cast_kb8(x, p["kc_in"], steps, tiles, R, addr, T * K)
            L.call("bsrnn_gemm_tc", xhat.data_ptr(), p["wih"].data_ptr(), p["bias"].data_ptr(), gates.data_ptr(), None, m_all,
                   2 * nt, p["kc_in"], BN, L.TC_F16_ROWS, 8 * H, 8 * H, 0, 1, m_all, m_all * 128, BIG, 0, 1, 0, st)
            with torch.profiler.record_function("tc_fwd_steps"):
                L.call("bsrnn_blstm_train_fwd_tc", zero.data_ptr(), y[0].data_ptr(), y[1].data_ptr(), p["whh"][0].data_ptr(),
                       p["whh"][1].data_ptr(), gates.data_ptr(), c_all[0].data_ptr(), c_all[1].data_ptr(), steps, tiles, nt, BN, H, st)
        out = torch.zeros(B, T, K, N, dtype=torch.float32, device=dev)
        n16 = p["fc_nt"] * p["fc_bn"]
        bias = torch.zeros(n16, dtype=torch.float32, device=dev)
        bias[:N] = fc_b.detach().float()
        zbias = torch.zeros_like(bias)
        for half, bb in ((0, bias), (1, zbias)):                   # out = y_fwd W_f^T + b, then += y_bwd W_b^T
            L.call("bsrnn_gemm_tc", y[half].data_ptr(), p["fcw"][half].data_ptr(), bb.data_ptr(), out.data_ptr(), None,
                   m_all, p["fc_nt"], p["kc_h"], p["fc_bn"], FC_EPI, N, N, 0, T * K, tiles, R, *addr, st)
        ctx.p, ctx.dims, ctx.fused = p, (B, T, K, N, axis), fused
        ctx.save_for_backward(xhat, gates, y[0], y[1], c_all[0], c_all[1])
        return out

    @staticmethod
    def backward(ctx, d_out):
        xhat, gates, y0, y1, c0, c1 = ctx.saved_tensors
        y, c_all = (y0, y1), (c0, c1)
        p = ctx.p
        B, T, K, N, axis = ctx.dims
        H, kc_in = p["H"], p["kc_in"]
        dev = d_out.device
        st = L.stream_ptr()
        R, steps, tiles, addr = _geom(B, T, K, axis)
        m_all = steps * tiles
        kc_g = 4 * H // 8
        d_out = d_out.contiguous().float()
        # loss scale S = 2^floor(log2(64 / max|d_out|)), kept ON THE DEVICE (no host sync): fp16 operands then sit around
        # 2^5..2^6 at their largest; non-finite or zero gradients fall back to S = 1
        amax = d_out.abs().max()
        S = torch.exp2(torch.floor(torch.log2(64.0 / amax)).clamp(-24.0, 24.0))
        S = torch.where(torch.isfinite(S) & (S > 0), S, torch.ones_like(S)).float()
        inv_s = (1.0 / S).reshape(1).contiguous()
        # ---- Linear backward: dy rows (tokens, 2H) = d_out W_fc
        dD = _cast_kb8(d_out, kc_in, steps, tiles, R, addr, T * K, scale=S)
        dy = torch.empty(m_all * 128, 2 * H, dtype=torch.float16, device=dev)
        L.call("bsrnn_gemm_tc", dD.data_ptr(), p["fcT"].data_ptr(), None, dy.data_ptr(), None, m_all, p["nt_y"], kc_in, p["bn_y"],
               L.TC_F16_ROWS, 2 * H, 2 * H, 0, 1, m_all, m_all * 128, BIG, 0, 1, 0, st)
        # ---- BPTT, one launch per step (both directions)
        dG = [torch.empty(m_all * kc_g * 1024, dtype=torch.float16, device=dev) for _ in range(2)]
        dc = [torch.zeros(tiles * 128, H, dtype=torch.float32, device=dev) for _ in range(2)]
        zero = torch.zeros(tiles * kc_g * 1024, dtype=torch.float16, device=dev)
        L.call("bsrnn_blstm_train_bwd_tc", zero.data_ptr(), dG[0].data_ptr(), dG[1].data_ptr(), p["whhT"][0].data_ptr(),
               p["whhT"][1].data_ptr(), gates.data_ptr(), dy.data_ptr(), c_all[0].data_ptr(), c_all[1].data_ptr(),
               dc[0].data_ptr(), dc[1].data_ptr(), steps, tiles, p["nt_h"], p["bn_h"], H, R, st)
        # ---- dx = sum_d dG_d W_ih_d   (token-major f32, loss scale removed)
        dx = torch.zeros(B, T, K, N, dtype=torch.float32, device=dev)
        for d in (0, 1):
            L.call("bsrnn_gemm_tc_scaled", dG[d].data_ptr(), p["wihT"][d].data_ptr(), None, dx.data_ptr(), m_all, p["nt_n"], kc_g,
                   p["bn_n"], N, N, 0.0, inv_s.data_ptr(), 1, tiles, R, *addr, st)
        # ---- weight gradients: tokens as the K axis
        kc_tok = m_all * 16
        nt_g = (4 * H + 127) // 128
        ksplit = max(1, min(16, kc_tok // 256))                       # ~13 output tiles x ksplit CTAs; >= 2048 tokens each
        xT = _transpose(xhat, 0, m_all, kc_in, p["bn_n"], p["nt_n"], kc_tok, 0, zero=False)
        grads_w = []
        for d in (0, 1):
            dGT = _transpose(dG[d], 0, m_all, kc_g, 128, nt_g, kc_tok, 0, zero=False)
            # fused forward: xhat carries the constant-one column N, so column N of dG^T xhat IS the bias gradient (sum of dG over
            # tokens) -- 4 more output columns instead of a reduction pass over dG per direction
            nv = N + 4 if ctx.fused else N
            dwih_full = torch.zeros(4 * H, nv, dtype=torch.float32, device=dev)
            L.call("bsrnn_gemm_tc_scaled", dGT.data_ptr(), xT.data_ptr(), None, dwih_full.data_ptr(), nt_g, p["nt_n"], kc_tok,
                   p["bn_n"], nv, nv, 0.0, inv_s.data_ptr(), ksplit, 1 << 30, 4 * H, 4, 1, H, 0, st)   # GEMM row 4u+g -> gradient row g*H + u
            dwih = dwih_full[:, :N]
            # h_{t-1}: the y tiles shifted by one step along the direction of the recurrence (zeros at its first step)
            if steps > 1:
                hT = _transpose(y[d], 0 if d == 0 else tiles, m_all - tiles, p["kc_h"], p["bn_h"], p["nt_h"], kc_tok,
                                tiles * 16 if d == 0 else 0, zero=True)
            else:
                hT = torch.zeros(p["nt_h"] * kc_tok * p["bn_h"] * 8, dtype=torch.float16, device=dev)
            dwhh = torch.zeros(4 * H, H, dtype=torch.float32, device=dev)
            L.call("bsrnn_gemm_tc_scaled", dGT.data_ptr(), hT.data_ptr(), None, dwhh.data_ptr(), nt_g, p["nt_h"], kc_tok, p["bn_h"],
                   H, H, 0.0, inv_s.data_ptr(), ksplit, 1 << 30, 4 * H, 4, 1, H, 0, st)
            # (f32 accumulation straight from the fp16 tiles: .float() first materialised a 2x copy of dG per direction)
            if ctx.fused:
                db = dwih_full[:, N]
            else:
                db = dG[d].view(m_all, kc_g, 128, 8).sum(dim=(0, 2), dtype=torch.float32).reshape(H, 4).t().reshape(4 * H) * inv_s
            grads_w.append((dwih, dwhh, db))
        nt_d = (N + 127) // 128
        dDT = _transpose(dD, 0, m_all, kc_in, 128, nt_d, kc_tok, 0, zero=False)
        dfcw = torch.zeros(N, 2 * H, dtype=torch.float32, device=dev)
        for d in (0, 1):
            yT = _transpose(y[d], 0, m_all, p["kc_h"], p["bn_h"], p["nt_h"], kc_tok, 0, zero=False)
            L.call("bsrnn_gemm_tc_scaled", dDT.data_ptr(), yT.data_ptr(), None, dfcw.data_ptr() + 4 * d * H, nt_d, p["nt_h"], kc_tok,
                   p["bn_h"], 2 * H, H, 0.0, inv_s.data_ptr(), ksplit, 1 << 30, N, BIG, 0, 1, 0, st)
        dfcb = d_out.sum(dim=(0, 1, 2))
        (wf, hf, bf), (wr, hr, br) = grads_w
        return dx, wf, hf, bf, bf, wr, hr, br, br, dfcw, dfcb, None


def blstm_block_tc(x, rnn, fc, axis):
    return BLSTMBlockTC.apply(x, *lstm_ws(rnn), fc.weight, fc.bias, axis)
