"""Training path of BSRNN_SE (reference train_se.py -> SEModel.training_step d_model.py:61-113, SURVEY.md §8a rows
a15-a17, §8e): differentiable forward, loss, backward, gradient allreduce, clip + AdamW.

What runs where (round-1 state, see DESIGN.md §7):
  * the 12 BLSTMs (91 % of the FLOPs): the sequential recurrence, forward AND back-propagation through time, are the
    hand-written kernels bsrnn_blstm_train_fwd_f32 / bsrnn_blstm_train_bwd_f32 (csrc/lstm_f32.cu) behind
    `BLSTMFunction`; the batched GEMMs around them (x W_ih^T, dG W_ih, dG^T x, dG^T h_prev) are plain library GEMMs
    (torch.matmul -> cuBLAS);
  * the input STFT is bsrnn_stft_fwd (no gradient flows into the noisy input);
  * BandSplit, GroupNorms, Linear+residual, MaskDecoder, complex mask, iSTFT and the loss are torch autograd ops over
    the SAME nn.Parameters (the reference's names/shapes), so `state_dict()` stays checkpoint-compatible;
  * the optimizer tail is two kernels on one flat buffer (csrc/optim.cu): global grad-norm + non-finite flag, then
    clip(0.5) + AdamW (+ EMA).  Data parallelism = ONE allreduce of that flat gradient buffer (NCCL on GPUs, gloo in
    the CPU tests); parameters unused on a rank (bands beyond K' at low sample rates) contribute zeros, which is what
    the reference's `ddp_find_unused_parameters_true` does (train_se.py:82).
"""
from __future__ import annotations

import math

import torch
import torch.nn.functional as F

from . import _lib as L
from . import runtime as R
from .losses import multires_l1_spec_loss, si_snr_loss


# ------------------------------------------------------------------------------------------------ BLSTM
class BLSTMFunction(torch.autograd.Function):
    """nn.LSTM(N, H, batch_first, bidirectional) over one axis of a token-major (B,T,K,N) tensor -> (B,T,K,2H)."""

    @staticmethod
    def forward(ctx, x, w_ih, w_hh, b_ih, b_hh, w_ih_r, w_hh_r, b_ih_r, b_hh_r, axis):
        B, T, K, N = x.shape
        H = w_hh.shape[1]
        M = B * T * K
        dev = x.device
        st = L.stream_ptr()
        x2 = x.reshape(M, N).contiguous()
        wih = torch.cat([w_ih, w_ih_r], 0).contiguous()                      # (8H, N)
        bias = torch.cat([b_ih + b_hh, b_ih_r + b_hh_r], 0)
        whh = torch.stack([w_hh, w_hh_r], 0).contiguous()                    # (2, 4H, H)
        gates = torch.addmm(bias, x2, wih.t())                               # (M, 8H) = (tokens, 2, 4H)
        if axis == "time":
            Rr, steps, addr = B * K, T, (K, T * K, 1, K)
        else:
            Rr, steps, addr = B * T, K, (1, K, 0, 1)
        y = torch.empty(M, 2 * H, dtype=torch.float32, device=dev)
        saved = torch.empty(M, 2, 5, H, dtype=torch.float32, device=dev)
        cst = torch.empty(2 * Rr * H, dtype=torch.float32, device=dev)
        L.call("bsrnn_blstm_train_fwd_f32", gates.data_ptr(), whh.data_ptr(), y.data_ptr(), cst.data_ptr(), saved.data_ptr(),
               Rr, steps, H, *addr, st)
        ctx.save_for_backward(x2, wih, whh, y, saved)
        ctx.dims = (B, T, K, N, H, Rr, steps, addr, axis)
        return y.view(B, T, K, 2 * H)

    @staticmethod
    def backward(ctx, dy):
        x2, wih, whh, y, saved = ctx.saved_tensors
        B, T, K, N, H, Rr, steps, addr, axis = ctx.dims
        M = B * T * K
        dev = dy.device
        st = L.stream_ptr()
        dy = dy.reshape(M, 2 * H).contiguous().float()
        dG = torch.empty(M, 2, 4 * H, dtype=torch.float32, device=dev)
        dh = torch.empty(2 * Rr * H, dtype=torch.float32, device=dev)
        dc = torch.empty(2 * Rr * H, dtype=torch.float32, device=dev)
        L.call("bsrnn_blstm_train_bwd_f32", dy.data_ptr(), saved.data_ptr(), whh.data_ptr(), dG.data_ptr(), dh.data_ptr(),
               dc.data_ptr(), Rr, steps, H, *addr, st)
        dG2 = dG.view(M, 8 * H)
        dx = (dG2 @ wih).view(B, T, K, N)
        dwih = dG2.t() @ x2                                                   # (8H, N)
        dbias = dG2.sum(0)
        # h_{t-1} per direction: y shifted by one step along the recurrence axis (zeros at the sequence start)
        y5 = y.view(B, T, K, 2, H)
        hp_f, hp_b = torch.zeros_like(y5[..., 0, :]), torch.zeros_like(y5[..., 1, :])
        if axis == "time":
            hp_f[:, 1:] = y5[:, :-1, :, 0]
            hp_b[:, :-1] = y5[:, 1:, :, 1]
        else:
            hp_f[:, :, 1:] = y5[:, :, :-1, 0]
            hp_b[:, :, :-1] = y5[:, :, 1:, 1]
        dwhh_f = dG[:, 0].t() @ hp_f.reshape(M, H)
        dwhh_b = dG[:, 1].t() @ hp_b.reshape(M, H)
        h4 = 4 * H
        return (dx, dwih[:h4], dwhh_f, dbias[:h4], dbias[:h4], dwih[h4:], dwhh_b, dbias[h4:], dbias[h4:], None)


def blstm(x, rnn, axis):
    return BLSTMFunction.apply(x, rnn.weight_ih_l0, rnn.weight_hh_l0, rnn.bias_ih_l0, rnn.bias_hh_l0,
                               rnn.weight_ih_l0_reverse, rnn.weight_hh_l0_reverse, rnn.bias_ih_l0_reverse,
                               rnn.bias_hh_l0_reverse, axis)


# ------------------------------------------------------------------------------------------------ differentiable forward
def _gn(x, dims, weight, bias, eps=1e-5):
    """GroupNorm(1, C) with the channel axis last: statistics over `dims` per sample, affine over the last axis."""
    mean = x.mean(dim=dims, keepdim=True)
    var = x.var(dim=dims, unbiased=False, keepdim=True)
    return (x - mean) * torch.rsqrt(var + eps) * weight + bias


def band_split_diff(bs, spec, plan):
    """BandSplit [bsrnn_flowse.py:65-86 / espnet2 BandSplit] on a (B,T,F,2) spectrum -> (B,T,K',N), differentiable."""
    B, T = spec.shape[0], spec.shape[1]
    zs = []
    for k in range(plan.K):
        s, b0, w = plan.subbands[k], plan.bin0[k], plan.width[k]
        xk = spec[:, :, b0:b0 + w, :]
        if w < s:
            xk = F.pad(xk, (0, 0, 0, s - w))
        xk = xk.reshape(B, T, 2 * s)
        xk = _gn(xk, (1, 2), bs.norm[k].weight, bs.norm[k].bias, bs.norm[k].eps)
        zs.append(F.linear(xk, bs.fc[k].weight[:, :, 0], bs.fc[k].bias))
    return torch.stack(zs, dim=2)


_BAND_TABLES = {}


def _band_tables(plan, dev):
    """Index tables of the batched per-band ops, cached per (plan, device): gather index into the flattened (F*2) axis,
    validity mask and per-band channel count of BandSplit; the (band, bin) -> output bin selection of the decoders."""
    key = (plan.subbands, plan.F, plan.K, str(dev))
    t = _BAND_TABLES.get(key)
    if t is None:
        K = plan.K
        smax = max(plan.subbands[:K])
        idx = torch.zeros(K, 2 * smax, dtype=torch.long)
        mask = torch.zeros(K, 2 * smax)
        sel = []
        for k in range(K):
            s, b0, w = plan.subbands[k], plan.bin0[k], plan.width[k]
            idx[k, : 2 * w] = 2 * b0 + torch.arange(2 * w)
            mask[k, : 2 * w] = 1.0
            sel += [k * smax + f for f in range(s)]
        chans = torch.tensor([2.0 * plan.subbands[k] for k in range(K)])
        t = _BAND_TABLES[key] = dict(smax=smax, idx=idx.to(dev), mask=mask.to(dev), chans=chans.to(dev),
                                     sel=torch.tensor(sel[: plan.F], dtype=torch.long, device=dev))
    return t


def _pad_rows(w, rows):
    return w if w.shape[0] == rows else F.pad(w, (0, 0, 0, rows - w.shape[0]))


def band_split_batched(bs, spec, plan):
    """band_split_diff with the K' per-band GroupNorm + Conv1d pairs as ONE gather, one set of reductions and one batched
    GEMM over zero-padded bands (the loop launches ~40 tiny kernels per band in forward + backward; at the training batch the
    step was bound by their count, not their work).  Same arithmetic per band: statistics over the 2 s_k channels x T frames
    (zeros of a truncated band included), padded channels carry zero weights."""
    B, T = spec.shape[0], spec.shape[1]
    K = plan.K
    tb = _band_tables(plan, spec.device)
    cmax = 2 * tb["smax"]
    x = spec.reshape(B, T, -1)[:, :, tb["idx"]] * tb["mask"]                     # (B,T,K,cmax)
    cnt = (tb["chans"] * T)[None, :]                                            # (1,K)
    mean = x.sum(dim=(1, 3)) / cnt                                              # (B,K)
    d = (x - mean[:, None, :, None]) * (torch.arange(cmax, device=x.device)[None, :] < tb["chans"][:, None])
    var = (d * d).sum(dim=(1, 3)) / cnt
    eps = bs.norm[0].eps
    gamma = torch.stack([F.pad(bs.norm[k].weight, (0, cmax - 2 * plan.subbands[k])) for k in range(K)])    # (K,cmax)
    beta = torch.stack([F.pad(bs.norm[k].bias, (0, cmax - 2 * plan.subbands[k])) for k in range(K)])
    xn = d * torch.rsqrt(var + eps)[:, None, :, None] * gamma + beta
    W = torch.stack([F.pad(bs.fc[k].weight[:, :, 0], (0, cmax - 2 * plan.subbands[k])) for k in range(K)])  # (K,N,cmax)
    bias = torch.stack([bs.fc[k].bias for k in range(K)])                       # (K,N)
    z = torch.bmm(xn.permute(2, 0, 1, 3).reshape(K, B * T, cmax), W.transpose(1, 2)) + bias[:, None, :]
    return z.reshape(K, B, T, -1).permute(1, 2, 0, 3).contiguous()


def mask_decoder_batched(md, skip, plan, F_bins):
    """mask_decoder_diff with the per-band MLPs as three batched GEMMs per family (bands zero-padded to the widest one in
    the last Conv1d, value and gate halves padded separately so that GLU pairs stay aligned)."""
    B, T, K, N = skip.shape
    tb = _band_tables(plan, skip.device)
    smax = tb["smax"]
    mean = skip.mean(dim=(1, 3), keepdim=True)
    d = skip - mean
    var = (d * d).mean(dim=(1, 3), keepdim=True)
    outs = []
    for mlps in (md.mlp_mask, md.mlp_residual):
        m0 = mlps[0]
        gamma = torch.stack([mlps[k][0].weight for k in range(K)])              # (K,N)
        beta = torch.stack([mlps[k][0].bias for k in range(K)])
        xn = d * torch.rsqrt(var + m0[0].eps) * gamma + beta                    # (B,T,K,N)
        W1 = torch.stack([mlps[k][1].weight[:, :, 0] for k in range(K)])        # (K,4N,N)
        b1 = torch.stack([mlps[k][1].bias for k in range(K)])
        h = torch.tanh(torch.bmm(xn.permute(2, 0, 1, 3).reshape(K, B * T, N), W1.transpose(1, 2)) + b1[:, None, :])
        W2, b2 = [], []
        for k in range(K):
            w, b = mlps[k][3].weight[:, :, 0], mlps[k][3].bias                   # (4s, 4N): rows [0,2s) value, [2s,4s) gate
            hs = w.shape[0] // 2
            W2.append(torch.cat([_pad_rows(w[:hs], 2 * smax), _pad_rows(w[hs:], 2 * smax)], 0))
            b2.append(torch.cat([F.pad(b[:hs], (0, 2 * smax - hs)), F.pad(b[hs:], (0, 2 * smax - hs))], 0))
        W2, b2 = torch.stack(W2), torch.stack(b2)                               # (K,4 smax,4N), (K,4 smax)
        o = F.glu(torch.bmm(h, W2.transpose(1, 2)) + b2[:, None, :], dim=-1)    # (K,B*T,2 smax)
        o = o.reshape(K, B, T, smax, 2).permute(1, 2, 0, 3, 4).reshape(B, T, K * smax, 2)
        outs.append(torch.view_as_complex(o[:, :, tb["sel"], :].contiguous()))
    return outs[0], outs[1]


def grad_decoder_batched(gd, skip, plan, F_bins):
    """grad_decoder_diff with the 2 x K' per-band GN -> Conv1d(N, 16 s) -> tanh as one set of reductions and one batched
    GEMM per family.  Each band's 16 s output channels (channel c = 16-index * s + f) are padded per sub-channel to
    16 smax, so that one reshape turns the GEMM output into (B,16,K smax,T); a gather then keeps the sum(s_k) real bins,
    the padded tail of a truncated last band included (the 5x5 Conv2d sees it, as in the per-band loop).  The Conv2d +
    GLU stays one torch op per family."""
    B, T, K, N = skip.shape
    sc = gd.sub_channel
    tb = _band_tables(plan, skip.device)
    smax = tb["smax"]
    sel = tb.get("sel_all")
    if sel is None:                                   # every bin of the K' bands (F' = sum s_k >= F), (band, bin) order
        sel = tb["sel_all"] = torch.tensor([k * smax + f for k in range(K) for f in range(plan.subbands[k])], dtype=torch.long,
                                           device=skip.device)
    mean = skip.mean(dim=(1, 3), keepdim=True)
    d = skip - mean
    var = (d * d).mean(dim=(1, 3), keepdim=True)
    outs = []
    for mlps, conv in ((gd.mlp_mask, gd.conv_after_mask), (gd.mlp_residual, gd.conv_after_residual)):
        gamma = torch.stack([mlps[k][0].weight for k in range(K)])              # (K,N)
        beta = torch.stack([mlps[k][0].bias for k in range(K)])
        xn = d * torch.rsqrt(var + mlps[0][0].eps) * gamma + beta               # (B,T,K,N)
        W, b = [], []
        for k in range(K):
            s = plan.subbands[k]
            W.append(F.pad(mlps[k][1].weight[:, :, 0].reshape(sc, s, N), (0, 0, 0, smax - s)).reshape(sc * smax, N))
            b.append(F.pad(mlps[k][1].bias.reshape(sc, s), (0, smax - s)).reshape(sc * smax))
        W, b = torch.stack(W), torch.stack(b)                                   # (K,16 smax,N), (K,16 smax)
        h = torch.tanh(torch.bmm(xn.permute(2, 0, 1, 3).reshape(K, B * T, N), W.transpose(1, 2)) + b[:, None, :])
        g = h.reshape(K, B, T, sc, smax).permute(1, 3, 0, 4, 2).reshape(B, sc, K * smax, T)[:, :, sel, :]   # (B,16,F',T)
        g = F.glu(F.conv2d(g, conv[0].weight, conv[0].bias, padding=2), dim=1)   # (B,2,F',T)
        g = g.permute(0, 3, 2, 1)                                                # (B,T,F',2)
        if g.shape[2] < F_bins:
            g = F.pad(g, (0, 0, 0, F_bins - g.shape[2]))
        outs.append(torch.view_as_complex(g[:, :, :F_bins, :].contiguous()))
    return outs[0], outs[1]


def block_f32(x, rnn, fc, axis):
    """(BLSTM -> Linear) block, f32: CUDA-core recurrence kernels + library GEMMs (parity ~1e-6)."""
    return F.linear(blstm(x, rnn, axis), fc.weight, fc.bias)


def block_tc(x, rnn, fc, axis):
    """(BLSTM -> Linear) block on tensor cores, forward and backward (training_tc.BLSTMBlockTC)."""
    from .training_tc import blstm_block_tc
    return blstm_block_tc(x, rnn, fc, axis)


BLOCKS = {"fp32": block_f32, "fp16": block_tc, "bf16": block_tc}


def dual_path_diff(core, skip, t_emb=None, blstm_fn=None):
    """The 2*num_layer (GN -> [+ t-embedding] -> BLSTM -> Linear -> residual) blocks [bsrnn_flowse.py:288-307] on a
    token-major (B,T,K,N) tensor.  t_emb: list of (B,N) per layer, added after the time-axis GroupNorm (:293-294).
    blstm_fn(x, rnn, fc, axis) -> Linear(BLSTM(x)): block_f32 (default) or block_tc."""
    blstm_fn = blstm_fn or block_f32
    for i in range(core.num_layer):
        for axis, norm, rnn, fc in (("time", core.norm_time[i], core.rnn_time[i], core.fc_time[i]),
                                    ("freq", core.norm_freq[i], core.rnn_freq[i], core.fc_freq[i])):
            out = _gn(skip, (1, 2, 3), norm.weight, norm.bias, norm.eps)
            if t_emb is not None and axis == "time":
                out = out + t_emb[i][:, None, None, :]
            skip = skip + blstm_fn(out, rnn, fc, axis)
    return skip


def mask_decoder_diff(md, skip, plan, F_bins):
    """espnet2 MaskDecoder: per band GN -> Conv1d(N,4N) -> tanh -> Conv1d(4N,4s) -> GLU -> (mask, resid) complex (B,T,F)."""
    B, T = skip.shape[0], skip.shape[1]
    outs = []
    for mlps in (md.mlp_mask, md.mlp_residual):
        parts = []
        for k in range(plan.K):
            m = mlps[k]
            xk = _gn(skip[:, :, k, :], (1, 2), m[0].weight, m[0].bias, m[0].eps)
            hk = torch.tanh(F.linear(xk, m[1].weight[:, :, 0], m[1].bias))
            ok = F.glu(F.linear(hk, m[3].weight[:, :, 0], m[3].bias), dim=-1)   # (B,T,2s)
            parts.append(ok.reshape(B, T, plan.subbands[k], 2))
        outs.append(torch.cat(parts, dim=2)[:, :, :F_bins, :])
    return torch.view_as_complex(outs[0].contiguous()), torch.view_as_complex(outs[1].contiguous())


def grad_decoder_diff(gd, skip, plan, F_bins):
    """GradDecoder [bsrnn_flowse.py:136-168]: per band GN -> Conv1d(N,16 s) -> tanh -> (B,16,s,T); cat over bins;
    Conv2d(16->4, 5x5, pad 2) + GLU(dim=1) -> (mask, resid) complex (B,T,F)."""
    B, T = skip.shape[0], skip.shape[1]
    sc = gd.sub_channel
    outs = []
    for mlps, conv in ((gd.mlp_mask, gd.conv_after_mask), (gd.mlp_residual, gd.conv_after_residual)):
        parts = []
        for k in range(plan.K):
            m = mlps[k]
            xk = _gn(skip[:, :, k, :], (1, 2), m[0].weight, m[0].bias, m[0].eps)
            ok = torch.tanh(F.linear(xk, m[1].weight[:, :, 0], m[1].bias))       # (B,T,16 s), channel c = sc*s + f
            parts.append(ok.reshape(B, T, sc, plan.subbands[k]).permute(0, 2, 3, 1))   # (B,16,s,T)
        g = torch.cat(parts, dim=2)                                              # (B,16,F',T)
        g = F.glu(F.conv2d(g, conv[0].weight, conv[0].bias, padding=2), dim=1)   # (B,2,F',T)
        g = g.permute(0, 3, 2, 1)                                                # (B,T,F',2)
        if g.shape[2] < F_bins:
            g = F.pad(g, (0, 0, 0, F_bins - g.shape[2]))
        outs.append(torch.view_as_complex(g[:, :, :F_bins, :].contiguous()))
    return outs[0], outs[1]


class ISTFTFunction(torch.autograd.Function):
    """STFTDecoder / torch.istft (window, overlap-add, envelope division, trim) as our kernels in both directions:
    forward bsrnn_istft_fwd, backward its exact adjoint bsrnn_istft_bwd.  (torch.istft is also not CUDA-graph capturable:
    it reads the window envelope back to the host.)"""

    @staticmethod
    def forward(ctx, spec_ri, L_out, n_fft, hop):
        ctx.dims = (L_out, n_fft, hop, spec_ri.shape[1])
        wav, _ = R.istft(spec_ri.contiguous().float(), None, None, L_out, n_fft, hop, want_spec=False)
        return wav

    @staticmethod
    def backward(ctx, d_wav):
        L_out, n_fft, hop, T = ctx.dims
        d_wav = d_wav.contiguous().float()
        B = d_wav.shape[0]
        d_spec = torch.empty(B, T, n_fft // 2 + 1, 2, dtype=torch.float32, device=d_wav.device)
        L.call("bsrnn_istft_bwd", d_wav.data_ptr(), d_spec.data_ptr(), R.twiddle(n_fft, d_wav.device).data_ptr(), B, T, L_out,
               n_fft, hop, L.stream_ptr())
        return d_spec, None, None, None


def bsrnn_se_train_forward(model, wav, lens, fs, blstm_fn=None):
    """Differentiable BSRNN_SE.forward on CUDA tensors: wav (B,L) f32, lens (B,) int -> (enhanced (B, max len),
    enhanced spectrum (B,T,F) complex64).  Same arithmetic as the inference kernels / the reference
    (bsrnn.py:36-41; espnet2 BSRNN.forward, SURVEY.md Appendix A), zeros of padded frames and truncated bands
    included in every GroupNorm statistic (§8g.1)."""
    core = model.bsrnn.bsrnn
    fs = int(fs)
    n_fft, hop = R.stft_dims(fs, model.N_FFT, model.HOP, model.DEFAULT_FS)
    F_bins = n_fft // 2 + 1
    plan = R.BandPlan.make(core.band_split.subbands, F_bins)
    lens_dev = R.device_lengths(lens, wav.device)
    with torch.no_grad():
        spec = R.stft(wav.contiguous().float(), lens_dev, n_fft, hop)           # (B,T,F,2), frames >= olens are zeros
    skip = band_split_batched(core.band_split, spec, plan)                      # (B,T,K',N)
    skip = dual_path_diff(core, skip, blstm_fn=blstm_fn)
    m_c, r_c = mask_decoder_batched(core.mask_decoder, skip, plan, F_bins)
    est = m_c * torch.view_as_complex(spec) + r_c                               # (B,T,F)
    if torch.cuda.is_current_stream_capturing():
        # reading device lengths would be a sync inside the capture: the output is the padded width, which is
        # max(lengths) for every batch SETrainer replays (it checks that on the host)
        L_out = wav.shape[1]
    else:
        L_out = int(torch.as_tensor(lens).max()) if not (torch.is_tensor(lens) and lens.is_cuda) else int(lens.max())
    wav_out = ISTFTFunction.apply(torch.view_as_real(est), L_out, n_fft, hop)
    return wav_out, est


def flow_bsrnn_train_forward(dnn, x_btf, y_btf, t, blstm_fn=None):
    """Differentiable flow BSRNN.forward [bsrnn_flowse.py:255-318] on the kernel layout: x_t, y (B,T,F,2) f32, t (B,) ->
    g = m*x_t + r as complex (B,T,F).  (FlowSEModel.forward negates it: flow_model.py:203-209.)"""
    import math
    F_bins = x_btf.shape[2]
    plan = R.BandPlan.make(dnn.band_split_x.subbands, F_bins)
    xx = band_split_batched(dnn.band_split_x, x_btf, plan)
    yy = band_split_batched(dnn.band_split_y, y_btf, plan)
    skip = F.linear(torch.cat([xx, yy], dim=-1), dnn.condition_fc.weight, dnn.condition_fc.bias)    # :284-285
    t = t.to(device=x_btf.device, dtype=torch.float32)
    t_emb = []
    for i in range(dnn.num_layer):                                               # GaussianFourierProjection :90-99
        proj = t[:, None] * dnn.t_cond[i].W[None, :] * 2 * math.pi
        t_emb.append(torch.cat([torch.sin(proj), torch.cos(proj)], dim=-1))
    skip = dual_path_diff(dnn, skip, t_emb=t_emb, blstm_fn=blstm_fn)
    m_c, r_c = grad_decoder_batched(dnn.grad_decoder, skip, plan, F_bins)
    return m_c * torch.view_as_complex(x_btf.contiguous()) + r_c


# ------------------------------------------------------------------------------------------------ flat parameters + step
class FlatParams:
    """All trainable parameters of a module re-pointed into ONE contiguous f32 buffer (and their .grad into another),
    so the allreduce is a single collective and the optimizer tail a single pair of kernels."""

    def __init__(self, module):
        self.params = [p for p in module.parameters() if p.requires_grad]
        self.numel = sum(p.numel() for p in self.params)
        dev = self.params[0].device
        pad = (-self.numel) % 4
        self.flat = torch.zeros(self.numel + pad, dtype=torch.float32, device=dev)
        self.grad = torch.zeros_like(self.flat)
        self.offsets = []
        self.touched = [False] * len(self.params)      # did autograd deliver a gradient for parameter i this step?
        off = 0
        for i, p in enumerate(self.params):
            n = p.numel()
            self.flat[off:off + n].copy_(p.data.reshape(-1))
            p.data = self.flat[off:off + n].view_as(p)
            p.grad = self.grad[off:off + n].view_as(p)
            self.offsets.append(off)
            p.register_post_accumulate_grad_hook(lambda _p, i=i: self._touch(i))
            off += n

    def _touch(self, i):
        self.touched[i] = True

    def untouched_ranges(self, touched=None):
        """Merged [lo, hi) element ranges of the parameters that got no gradient (bands beyond K' at low sample
        rates): torch AdamW skips grad=None parameters altogether, and so does bsrnn_adamw_step2."""
        touched = self.touched if touched is None else touched
        out = []
        for p, off, t in zip(self.params, self.offsets, touched):
            if t:
                continue
            if out and out[-1][1] == off:
                out[-1][1] = off + p.numel()
            else:
                out.append([off, off + p.numel()])
        return out

    def zero_grad(self):
        self.grad.zero_()
        self.touched = [False] * len(self.params)
        for p, off in zip(self.params, self.offsets):           # autograd may have replaced .grad: re-attach the views
            n = p.numel()
            view = self.grad[off:off + n].view_as(p)
            if p.grad is None or p.grad.data_ptr() != view.data_ptr():
                p.grad = view

    def gather_grads(self):
        """Make sure every gradient autograd produced lives in the flat buffer (it normally accumulates in place)."""
        for p, off in zip(self.params, self.offsets):
            n = p.numel()
            view = self.grad[off:off + n].view_as(p)
            if p.grad is not None and p.grad.data_ptr() != view.data_ptr():
                view.copy_(p.grad)
                p.grad = view


class SETrainer:
    """One optimisation step of the reference's SEModel [d_model.py:61-113 + Trainer(gradient_clip_val=0.5),
    train_se.py:74-83]:  forward -> MultiResL1SpecLoss.mean() (NaN loss -> zero loss, d_model.py:75-77) -> backward ->
    allreduce(avg) -> clip-by-norm -> AdamW(lr, eps=adam_epsilon, weight_decay) -> optional EMA; StepLR via set_lr()."""

    def __init__(self, se_model, lr=1e-3, weight_decay=1e-6, eps=1e-8, betas=(0.9, 0.999), gradient_clip=0.5,
                 ema_decay=None, process_group=None, forward_fn=None, loss_fn=None, precision="fp32", cuda_graph=False):
        # precision: "fp32" = f32 recurrence kernels + library GEMMs; "fp16" (alias "bf16") = the BLSTM blocks forward and
        # backward on tcgen05 with fp16 operands, f32 accumulation and f32 master weights (training_tc.py)
        if precision not in BLOCKS:
            raise NotImplementedError(f"precision {precision!r}")
        self.precision = precision
        self.block_fn = BLOCKS[precision]
        self.cuda_graph = bool(cuda_graph)
        self._graphs = {}                  # (noisy shape, clean shape, fs) -> captured step
        self.captures = 0
        self._seen = {}                    # shape -> peak device bytes of its first (eager) step
        self._eager_only = set()           # shapes that did not fit beside the graphs kept
        self.pool_bytes = {}               # signature -> device bytes of the private pool its capture took
        self.model = se_model
        self.loss_fn = loss_fn             # (model, noisy, clean, lengths, fs) -> (loss, logged scalar): other criteria
        self.flat = FlatParams(se_model)
        self.lr, self.weight_decay, self.eps, self.betas, self.clip = lr, weight_decay, eps, betas, gradient_clip
        self.exp_avg = torch.zeros_like(self.flat.flat)
        self.exp_avg_sq = torch.zeros_like(self.flat.flat)
        self.ema = self.flat.flat.clone() if ema_decay else None
        self.ema_decay, self.ema_updates = ema_decay, 0
        # {sum g^2, non-finite flag, adam steps, ema updates, 1-b1^t, 1-b2^t, ema decay, -}: the counters live on the
        # device so a step skipped for non-finite gradients does not advance them (bsrnn_adamw_step2)
        self.stats = torch.zeros(8, dtype=torch.float64, device=self.flat.flat.device)
        self._skip_cache = {}
        self.group = process_group
        self.forward_fn = forward_fn or bsrnn_se_train_forward

    def set_lr(self, lr):
        self.lr = lr

    def world_size(self):
        import torch.distributed as dist
        return dist.get_world_size(self.group) if (dist.is_available() and dist.is_initialized()) else 1

    def loss(self, noisy, clean, lengths, fs):
        """SEModel.forward_step [d_model.py:61-89]: returns (loss scalar, SI-SNR in dB averaged over the batch)."""
        if self.loss_fn is not None:
            return self.loss_fn(self.model, noisy, clean, lengths, fs, blstm_fn=self.block_fn)
        Bn = clean.shape[0]
        clean, noisy = clean.reshape(Bn, -1).float(), noisy.reshape(Bn, -1).float()
        est = self.forward_fn(self.model, noisy, lengths, fs, blstm_fn=self.block_fn)[0]
        loss = multires_l1_spec_loss(clean, est).mean()
        # d_model.py:75-77 (NaN loss -> est.mean() * 0), selected on the device: `if torch.isnan(loss)` is a host sync
        loss = torch.where(torch.isnan(loss), est.mean() * 0, loss)
        with torch.no_grad():
            sisnr = -si_snr_loss(clean, est).mean()
        return loss, sisnr

    def step(self, noisy, clean, lengths, fs):
        if self.cuda_graph:
            return self._step_graphed(noisy, clean, lengths, fs)
        return self._step_eager(noisy, clean, lengths, fs)

    def _step_eager(self, noisy, clean, lengths, fs):
        self.flat.zero_grad()
        loss, sisnr = self.loss(noisy, clean, lengths, fs)
        loss.backward()
        self.flat.gather_grads()
        self.apply_gradients()
        return loss.detach(), sisnr

    # ---- CUDA-graph replay of forward + loss + backward (the step is launch-bound: ~8 700 kernels, profiles/r02 call05) ----
    # Graphs are kept per (batch shape, rate), and a corpus with utterances shorter than max_duration has many shapes.  Each
    # graph pins a private pool about as large as the eager step's peak, which depends on the model AND the rate (config 5
    # on a B200: SE up to 9.7 GB; FlowSE at the published width 20.6 GB at 48 kHz, 67 GB at 8 kHz), so what fits is decided
    # at run time from free device memory.  Evicting graphs to capture others thrashes when a corpus has more shapes than
    # fit (measured on a seven-rate set: 420 ms per step against 90 ms eager), so graphs are kept and a shape that does not
    # fit runs eager.
    MAX_GRAPHS = 8

    def _step_graphed(self, noisy, clean, lengths, fs):
        """One captured graph per batch shape and rate: zero_grad + forward + loss + backward + gather are replayed; the
        allreduce and the fused optimizer tail stay eager (two kernels and one collective).  The lengths are device data
        of the graph (a static buffer written before each replay), so one graph serves every batch of that shape; the
        padded width must be the longest length, which the training collate guarantees (checked on the host for host
        lengths; device lengths are checked once, at the first step of a shape, and must keep it after).

        The first batch of a shape runs eager and measures its peak device memory (resetting the allocator's peak
        statistics), so a width seen once costs no capture.  The second is captured if MAX_GRAPHS allows it and the free
        device memory holds that peak (for the graph's pool) plus the largest eager peak seen (for the shapes that keep
        running eager); otherwise that shape runs eager from then on.  Random draws inside the loss (FlowSE's t and z)
        use the graph-safe CUDA generator, so every replay draws afresh."""
        dev = self.flat.flat.device
        lens_src = lengths if (torch.is_tensor(lengths) and lengths.is_cuda) else torch.as_tensor(lengths)
        key = (tuple(noisy.shape), tuple(clean.shape), int(fs))
        entry = self._graphs.get(key)
        if not lens_src.is_cuda or key not in self._seen:      # (host lengths: pinned from the loader, so the copy is async)
            longest = int(lens_src.max())
            if longest != noisy.shape[-1]:
                raise ValueError(f"graphed step: max(lengths) = {longest} but the batch is padded to {noisy.shape[-1]}")
        if entry is None and key not in self._seen:
            torch.cuda.reset_peak_memory_stats(dev)
            base = torch.cuda.memory_allocated(dev)
            out = self._step_eager(noisy, clean, lengths, fs)
            self._seen[key] = torch.cuda.max_memory_allocated(dev) - base
            return out
        if entry is None and key in self._eager_only:
            return self._step_eager(noisy, clean, lengths, fs)
        if entry is None:
            torch.cuda.synchronize(dev)
            torch.cuda.empty_cache()
            need = self._seen[key] + max(self._seen.values())
            if len(self._graphs) >= self.MAX_GRAPHS or torch.cuda.mem_get_info(dev)[0] < need:
                self._eager_only.add(key)
                return self._step_eager(noisy, clean, lengths, fs)
            n_s, c_s = torch.empty_like(noisy, device=dev), torch.empty_like(clean, device=dev)
            l_s = torch.empty(lens_src.shape, dtype=torch.int32, device=dev)
            n_s.copy_(noisy); c_s.copy_(clean); l_s.copy_(lens_src)
            side = torch.cuda.Stream(dev)
            side.wait_stream(torch.cuda.current_stream(dev))
            with torch.cuda.stream(side):                     # warm-up on a side stream (allocator, caches, lazy inits)
                for _ in range(2):
                    self.flat.zero_grad()
                    l0, _ = self.loss(n_s, c_s, l_s, fs)
                    l0.backward()
                    self.flat.gather_grads()
            torch.cuda.current_stream(dev).wait_stream(side)
            torch.cuda.synchronize(dev)
            touched = list(self.flat.touched)                  # hooks do not run at replay: the set is part of the signature
            del l0
            torch.cuda.empty_cache()                           # the warm-up's blocks go back before the pool is filled
            free0 = torch.cuda.mem_get_info(dev)[0]
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g):
                self.flat.zero_grad()
                loss, logged = self.loss(n_s, c_s, l_s, fs)
                loss.backward()
                self.flat.gather_grads()
            torch.cuda.synchronize(dev)
            self.pool_bytes[key] = free0 - torch.cuda.mem_get_info(dev)[0]
            self.captures += 1
            entry = self._graphs[key] = (g, n_s, c_s, l_s, loss, logged, touched)
        g, n_s, c_s, l_s, loss, logged, touched = entry
        n_s.copy_(noisy, non_blocking=True)
        c_s.copy_(clean, non_blocking=True)
        l_s.copy_(lens_src, non_blocking=True)
        g.replay()
        self.flat.touched = list(touched)
        self.apply_gradients()
        return loss.detach().clone(), logged.detach().clone()

    # ---- trainer state (checkpoints, resume) ----
    def state_dict(self):
        """Optimizer state beside the weights: the flat AdamW moments, the flat EMA, the device counters, the lr."""
        cpu = lambda t: None if t is None else t.detach().cpu().clone()
        return {"numel": self.flat.numel, "exp_avg": cpu(self.exp_avg), "exp_avg_sq": cpu(self.exp_avg_sq),
                "ema": cpu(self.ema), "stats": cpu(self.stats), "lr": float(self.lr)}

    def load_state_dict(self, state):
        if int(state["numel"]) != self.flat.numel or state["exp_avg"].numel() != self.exp_avg.numel():
            raise ValueError(f"trainer state for {state['numel']} parameters, this model has {self.flat.numel}")
        self.exp_avg.copy_(state["exp_avg"])
        self.exp_avg_sq.copy_(state["exp_avg_sq"])
        if self.ema is not None and state.get("ema") is not None:
            self.ema.copy_(state["ema"])
        self.stats.copy_(state["stats"])
        self.lr = float(state["lr"])

    def allreduce_gradients(self):
        """ONE collective over the flat gradient buffer (sum; the 1/world factor is folded into the optimizer kernel).
        Parameters that received no gradient on this rank hold zeros, so ranks with different sample rates (different
        K') still agree on what is reduced — the semantics of ddp_find_unused_parameters_true (train_se.py:82)."""
        import torch.distributed as dist
        world = self.world_size()
        if world > 1:
            dist.all_reduce(self.flat.grad, op=dist.ReduceOp.SUM, group=self.group)
        return world

    def _touched_any_rank(self, world):
        """Which parameters received a gradient on ANY rank (after the allreduce those hold real gradients everywhere,
        like the zeros-contributing unused parameters of ddp_find_unused_parameters_true)."""
        touched = list(self.flat.touched)
        if world > 1:
            import torch.distributed as dist
            t = torch.tensor(touched, dtype=torch.int32, device=self.flat.grad.device)
            dist.all_reduce(t, op=dist.ReduceOp.MAX, group=self.group)
            touched = [bool(v) for v in t.tolist()]
        return touched

    def _skip_ranges(self, world):
        ranges = self.flat.untouched_ranges(self._touched_any_rank(world))
        if len(ranges) > 32:                       # cannot happen for BSRNN (4 contiguous band suffixes); stay correct
            ranges = []
        key = tuple(map(tuple, ranges))
        dev = self._skip_cache.get(key)
        if dev is None:
            flat = [v for r in ranges for v in r] or [0, 0]
            dev = self._skip_cache[key] = torch.tensor(flat, dtype=torch.int64, device=self.flat.grad.device)
        return dev, len(ranges)

    @property
    def step_count(self):
        """Optimizer steps actually taken (device counter; non-finite steps are not counted)."""
        return int(self.stats[2])

    def apply_gradients(self):
        """allreduce (sum) of the flat gradient buffer, then the fused clip + AdamW (+EMA) tail."""
        world = self.allreduce_gradients()
        g = self.flat.grad
        if not g.is_cuda:
            raise L.NativeLibraryError("SETrainer.apply_gradients needs CUDA parameters (no CPU fallback)")
        skip, n_skip = self._skip_ranges(world)
        st = L.stream_ptr()
        L.call("bsrnn_grad_sumsq", g.data_ptr(), g.numel(), self.stats.data_ptr(), st)
        L.call("bsrnn_adamw_step2", self.flat.flat.data_ptr(), g.data_ptr(), self.exp_avg.data_ptr(),
               self.exp_avg_sq.data_ptr(), L.ptr(self.ema), g.numel(), self.stats.data_ptr(), skip.data_ptr(), n_skip,
               1.0 / world, float(self.clip or 0.0), self.lr, self.betas[0], self.betas[1], self.eps,
               self.weight_decay, float(self.ema_decay or 0.0), st)
        R.invalidate_packed()          # the kernel wrote the parameters through raw pointers: packed copies are stale

    def grad_norm(self):
        """Global L2 norm of the (averaged) gradients of the last step — the reference logs it as `Grad_norm`."""
        return math.sqrt(float(self.stats[0])) / self.world_size()


# ------------------------------------------------------------------------------------------------ FlowSE
def flowse_forward_step(model, noisy, clean, lengths, fs, t=None, z=None, blstm_fn=None):
    """FlowSEModel.forward_step [flow_model.py:149-187]: STFT (+ exponent compression) of clean and noisy, t ~
    min((1-U)(T_rev - t_eps) + t_eps, T_rev), x_t = (1-t) x0 + t y + sigma_t z, target condVF = (sigma_max - sigma_min) z
    + (y - x0) [odes.py:74-98], loss = mean_b 0.5 * sum |v - condVF|^2 with v = -dnn([x_t, y], t) [:122-132, :203-209].
    ``t`` (B,) and ``z`` complex (B,T,F) may be passed in for parity tests (the reference draws them with torch.rand /
    randn_like).  Returns (loss, loss detached) in SETrainer's (loss, logged scalar) convention."""
    B = clean.shape[0]
    clean = torch.nan_to_num(clean.reshape(B, -1).float(), nan=0.0)
    noisy = torch.nan_to_num(noisy.reshape(B, -1).float(), nan=0.0)
    with torch.no_grad():
        x0 = torch.view_as_complex(model._encode(clean, fs, lengths))              # (B,T,F) compressed spectra
        y = torch.view_as_complex(model._encode(noisy, fs, lengths))
        dev = x0.device
        if t is None:
            rdm = (1 - torch.rand(B, device=dev)) * (model.T_rev - model.t_eps) + model.t_eps
            t = torch.clamp(rdm, max=model.T_rev)
        t = t.to(dev).float()
        if z is None:
            z = torch.randn_like(x0)
        z = z.to(dev)
        ode = model.ode
        std = ((1 - t) * ode.sigma_min + t * ode.sigma_max)[:, None, None]
        xt = (1 - t)[:, None, None] * x0 + t[:, None, None] * y + std * z
        cond_vf = (ode.sigma_max - ode.sigma_min) * z + (y - x0)
    g = flow_bsrnn_train_forward(model.dnn, torch.view_as_real(xt).contiguous(), torch.view_as_real(y).contiguous(), t,
                                 blstm_fn=blstm_fn)
    err = (-g) - cond_vf
    loss = (0.5 * (err.real ** 2 + err.imag ** 2).reshape(B, -1).sum(-1)).mean()
    return loss, loss.detach()


class FlowSETrainer(SETrainer):
    """FlowSEModel's optimisation step [flow_model.py:66-84,149-187,238-249]: flow-matching loss, AdamW, and the
    torch_ema update fused into the optimizer kernel; ``sync_ema()`` writes the flat EMA back into ``model.ema`` (what
    ``eval()`` swaps in and ``on_save_checkpoint`` stores)."""

    def __init__(self, flow_model, **kw):
        kw.setdefault("lr", flow_model.lr)
        kw.setdefault("ema_decay", flow_model.ema_decay)
        super().__init__(flow_model, loss_fn=flowse_forward_step, **kw)

    def sync_ema(self):
        n_upd = int(self.stats[3])
        shadow = self.model.ema.shadow_params
        by_id = {id(p): i for i, p in enumerate(self.model.parameters())}
        with torch.no_grad():
            for p, off in zip(self.flat.params, self.flat.offsets):
                shadow[by_id[id(p)]].copy_(self.ema[off:off + p.numel()].view_as(p))
        self.model.ema.num_updates = n_upd

    def load_ema_from_model(self):
        """The inverse of sync_ema: ``model.ema`` (e.g. a checkpoint's ``ema`` entry) into the flat EMA and its counter."""
        shadow = self.model.ema.shadow_params
        by_id = {id(p): i for i, p in enumerate(self.model.parameters())}
        with torch.no_grad():
            for p, off in zip(self.flat.params, self.flat.offsets):
                self.ema[off:off + p.numel()].copy_(shadow[by_id[id(p)]].reshape(-1))
        self.stats[3] = float(self.model.ema.num_updates or 0)
