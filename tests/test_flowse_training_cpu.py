"""CPU tests of the FlowSE training path's host logic: the batched GradDecoder against the per-band loop, the operand
sizes of the H = 768 fused training forward, and the argument checks of its C entry point."""
import types

import pytest
import torch

from oracle import ref_loader


def _flowse(**over):
    from urgent2026_challenge_track1_b200.config import Config
    from urgent2026_challenge_track1_b200.flow_model import FlowSEModel
    return FlowSEModel(ref_loader.flowse_config(types.SimpleNamespace(Config=Config), **over))


@pytest.mark.parametrize("fs", [16000, 22050, 48000])
def test_grad_decoder_batched_equals_the_per_band_loop(fs):
    """training.grad_decoder_batched (one set of GN reductions + one batched GEMM per family) against grad_decoder_diff
    (the per-band loop that mirrors bsrnn_flowse.py:136-168) in f64: outputs and every GradDecoder gradient, truncated last
    band included (22.05 kHz and 16 kHz end inside a band)."""
    from urgent2026_challenge_track1_b200 import runtime as RT, training as TR
    torch.manual_seed(0)
    m = _flowse(bsrnn_hidden=16, num_layer=1).double()
    gd = m.dnn.grad_decoder
    for p in gd.parameters():
        p.data = p.data + 0.1 * torch.randn_like(p)
    n_fft, hop = RT.stft_dims(fs, m.n_fft, m.hop_length, m.DEFAULT_FS)
    Fb = n_fft // 2 + 1
    plan = RT.BandPlan.make(m.dnn.band_split_x.subbands, Fb)
    skip = torch.randn(2, 7, plan.K, 16, dtype=torch.float64)
    if fs != 48000:
        assert plan.width[-1] < plan.subbands[plan.K - 1] or sum(plan.subbands[:plan.K]) > Fb

    def run(fn):
        for p in gd.parameters():
            p.grad = None
        x = skip.clone().requires_grad_(True)
        mc, rc = fn(gd, x, plan, Fb)
        ((mc.abs() ** 2).sum() + (rc.real * 1.3 + rc.imag * 0.7).sum()).backward()
        return mc.detach(), rc.detach(), x.grad, {n: p.grad.clone() for n, p in gd.named_parameters() if p.grad is not None}

    a = run(TR.grad_decoder_diff)
    b = run(TR.grad_decoder_batched)
    rel = lambda x, y: float((x - y).abs().max() / (y.abs().max() + 1e-30))
    assert a[0].shape == b[0].shape == (2, 7, Fb)
    assert rel(b[0], a[0]) < 1e-12 and rel(b[1], a[1]) < 1e-12 and rel(b[2], a[2]) < 1e-12
    assert set(a[3]) == set(b[3])                  # bands the spectrum does not reach get no gradient in either
    assert max(rel(b[3][n], a[3][n]) for n in a[3]) < 1e-12


@pytest.mark.parametrize("N,H,kc_in,rows", [(196, 392, 26, 208), (384, 768, 50, 416)])
def test_fused_block_operands_cover_the_bias_column(N, H, kc_in, rows):
    """The fused forward's input operand carries the constant-one column N: kc_in and the x^T tiles of the weight
    gradient cover it (column N of dG^T xhat is the bias gradient).  At N = 196 it sits in the padding; at N = 384 it needs
    two more k-cores.  The step-wise operands keep K = N."""
    from urgent2026_challenge_track1_b200 import training_tc as TT
    torch.manual_seed(2)
    rnn, fc = torch.nn.LSTM(N, H, bidirectional=True), torch.nn.Linear(2 * H, N)
    ws = [getattr(rnn, n + sfx) for sfx in ("", "_reverse") for n in ("weight_ih_l0", "weight_hh_l0", "bias_ih_l0", "bias_hh_l0")]
    fused = TT.pack_block(*ws, fc.weight, fwd_steps=False)
    assert fused["kc_in"] == kc_in and fused["bn_n"] * fused["nt_n"] == rows and N + 4 <= rows
    assert fused["fcT"].numel() == fused["nt_y"] * fused["bn_y"] * kc_in * 8          # K of dy = dD W_fc spans kc_in
    steps = TT.pack_block(*ws, fc.weight, fwd_steps=True)
    assert steps["kc_in"] == (N + 15) // 16 * 2
    if N == 196:                                  # H = 392 operands are the same either way
        assert steps["kc_in"] == fused["kc_in"] and steps["bn_n"] == fused["bn_n"] and steps["nt_n"] == fused["nt_n"]


# (description, argument overrides, expected error) for bsrnn_blstm_fused768_train_tc
_BAD_CALLS = {
    "null_xhat": (dict(xhat=None), "null pointer"),
    "null_gates": (dict(gates=None), "null pointer"),
    "null_scratch": (dict(scratch=None), "null pointer"),
    "null_sync": (dict(sync=None), "null pointer"),
    "zero_rows": (dict(R=0), "bad dims"),
    "zero_steps": (dict(steps=0), "bad dims"),
    "too_few_tiles": (dict(R=300, tiles=2), "bad dims"),
    "short_y_stride": (dict(y_stride=95 * 1024), "bad y_stride"),
    "odd_y_stride": (dict(y_stride=96 * 1024 + 4), "bad y_stride"),
}


@pytest.mark.skipif(torch.cuda.is_available(), reason="on a GPU an accepted call would launch")
@pytest.mark.parametrize("case", sorted(_BAD_CALLS))
def test_fused768_train_rejects_bad_arguments(case):
    from urgent2026_challenge_track1_b200 import _lib
    over, msg = _BAD_CALLS[case]
    p = 1 << 20                                   # never dereferenced: the call must fail its argument checks
    a = dict(xhat=p, gates=p, scratch=p, sync=p, R=256, steps=3, tiles=2, y_stride=96 * 1024)
    a.update(over)
    h = _lib.lib()
    rc = h.bsrnn_blstm_fused768_train_tc(a["xhat"], p, p, p, p, a["y_stride"], a["gates"], p, p, a["scratch"], a["R"],
                                         a["steps"], a["tiles"], 0, 0, a["sync"], None)
    err = h.bsrnn_last_error().decode()
    assert rc != 0 and "blstm_fused768_train_tc" in err and msg in err, (rc, err)
    assert h.bsrnn_blstm_fused768_train_scratch_bytes(3, 2) == 3 * 2 * 128 * 768 * 24
