"""CPU tests: every packed BLSTM weight layout decodes back to nn.LSTM's tensors exactly.

The decoders (tests/lstm_packs.py) invert each packer's index map and remove GATE_SCALE.  The decoded tensors must equal
fp16(w * scale) / scale of the nn.LSTM tensors bit for bit, and every padding row, column and k-core of the pack must be
zero.  Training hands the packers nn.Parameters that require grad, inference packs under no_grad: both are decoded.  The
GPU tests (test_gpu_lstm_tc.py) build their f64 references from the same decoders."""
import itertools

import pytest
import torch

from lstm_packs import (decode_fused_pairs, decode_lstm_steps, decode_lstm_tc, decode_pack_block, lstm_tensors, rounded)
from urgent2026_challenge_track1_b200 import runtime_tc as TC
from urgent2026_challenge_track1_b200 import runtime_tc_steps as TS
from urgent2026_challenge_track1_b200 import training_tc as TT


GRAD = pytest.mark.parametrize("grad", [True, False], ids=["requires_grad", "no_grad"])


def _lstm(N, H, seed):
    torch.manual_seed(seed)
    rnn = torch.nn.LSTM(N, H, batch_first=True, bidirectional=True)
    with torch.no_grad():
        for p in rnn.parameters():           # magnitudes that exercise fp16 rounding, subnormals and the exponent range
            p.copy_(torch.randn_like(p) * torch.exp2(torch.randint(-16, 3, p.shape).float()))
    return rnn


def _same(a, b, what):
    assert a.shape == b.shape, f"{what}: shape {tuple(a.shape)} != {tuple(b.shape)}"
    diff = (a != b) & ~(torch.isnan(a) & torch.isnan(b))
    assert not bool(diff.any()), f"{what}: {int(diff.sum())} elements differ (first at {torch.nonzero(diff)[0].tolist()})"


def test_pack_and_decode_lstm_tc():
    rnn = _lstm(196, 392, 1)
    p = TC.pack_lstm_tc(rnn)
    dec = decode_lstm_tc(p)
    for d, (wi, wh, b) in enumerate(lstm_tensors(rnn)):
        _same(dec["wih"][d][0], rounded(wi), f"wih[{d}]")
        _same(dec["wih"][d][1], rounded(b), f"wih[{d}] bias column")
        _same(dec["whh"][d], rounded(wh), f"whh[{d}]")
        _same(dec["bih"][d], b.double(), f"bih[{d}] (f32, not rounded)")
        fwi, fwh, fb = dec["wfused"][d]
        _same(fwi, rounded(wi), f"wfused[{d}] W_ih")
        _same(fwh, rounded(wh), f"wfused[{d}] W_hh")
        _same(fb, rounded(b), f"wfused[{d}] bias")


# geometry -> (N, H, kc_in, pairs, packed rows per pair): the fused layer kernel's four group geometries at their widths
FUSED = {8: (196, 392, 26, 8, 208), 7: (196, 392, 26, 7, 224), 14: (196, 392, 26, 14, 112), 768: (384, 768, 50, 24, 128)}


@GRAD
@pytest.mark.parametrize("geo", sorted(FUSED))
def test_pack_and_decode_fused(geo, grad):
    N, H, kc_in, P, rows = FUSED[geo]
    rnn = _lstm(N, H, geo)
    with torch.set_grad_enabled(grad):
        wf = TC.pack_fused(TC.lstm_ws(rnn), geo, kc_in, N)
    assert tuple(wf.shape) == (2, P, 2, kc_in + (H + 15) // 16 * 2, rows // 2, 8) and wf.dtype == torch.float16
    for d, ((wi, wh, b), (dwi, dwh, db)) in enumerate(zip(lstm_tensors(rnn), decode_fused_pairs(wf, H, N, kc_in, N))):
        _same(dwi, rounded(wi), f"fused{geo}[{d}] W_ih")
        _same(dwh, rounded(wh), f"fused{geo}[{d}] W_hh")
        _same(db, rounded(b), f"fused{geo}[{d}] bias")


def test_pack_and_decode_lstm_steps_and_fused768():
    """pack_lstm_steps_tc at the FlowSE width (with the fused layer kernel's weights) and at (N, H) = (64, 32), in both grad
    modes."""
    for (N, H), grad in itertools.product([(384, 768), (64, 32)], [True, False]):
        rnn = _lstm(N, H, 3)
        with torch.set_grad_enabled(grad):
            p = TS.pack_lstm_steps_tc(rnn)
        assert ("wfused" in p) == (H == 768)
        steps = decode_lstm_steps(p)
        for d, (wi, wh, b) in enumerate(lstm_tensors(rnn)):
            _same(steps[d][0], rounded(wi), f"steps{H} wih[{d}]")
            _same(steps[d][1], rounded(wh), f"steps{H} whh[{d}]")
            _same(steps[d][2], b.double(), f"steps{H} bias[{d}] (f32, not rounded)")
        if H == 768:
            assert tuple(p["wfused"].shape) == (2, 24, 2, 146, 64, 8) and p["kc_fused"] == 50 and p["one_col"] == 384
            for d, ((wi, wh, b), fused) in enumerate(zip(lstm_tensors(rnn), decode_fused_pairs(p["wfused"], 768, 384, 50, 384))):
                _same(fused[0], rounded(wi), f"fused768[{d}] W_ih")
                _same(fused[1], rounded(wh), f"fused768[{d}] W_hh")
                _same(fused[2], rounded(b), f"fused768[{d}] bias")


@pytest.mark.parametrize("N,H", [(196, 392), (384, 768), (36, 40)])
@pytest.mark.parametrize("fwd_steps", [True, False])
@pytest.mark.parametrize("narrow", [False, 2])
def test_pack_and_decode_pack_block(N, H, fwd_steps, narrow):
    rnn = _lstm(N, H, H + N)
    fc_w = torch.randn(N, 2 * H)
    for grad in (True, False):
        with torch.set_grad_enabled(grad):
            p = TT.pack_block(*TC.lstm_ws(rnn), fc_w, narrow_bwd=narrow, fwd_steps=fwd_steps)
        assert p["nt_h"] * p["bn_h"] >= H and p["nt_n"] * p["bn_n"] >= N
        dec = decode_pack_block(p)
        for d, (wi, wh, b) in enumerate(lstm_tensors(rnn)):
            _same(dec[d]["whhT"], rounded(wh, scale_rows=False), f"whhT[{d}]")
            _same(dec[d]["wihT"], rounded(wi, scale_rows=False), f"wihT[{d}]")
            if fwd_steps:
                _same(dec[d]["whh"], rounded(wh), f"block whh[{d}]")
                _same(dec[d]["wih"], rounded(wi), f"block wih[{d}]")
                _same(dec[d]["b"], b.double(), f"block bias[{d}]")
            else:
                assert "whh" not in dec[d]


def test_decoders_reject_a_corrupted_pack():
    """the decoders see a moved weight (wrong row), a non-zero padding element and a wrong scale."""
    rnn = _lstm(196, 392, 5)
    wf = TC.pack_fused(TC.lstm_ws(rnn), 7, 26, 196)
    wi = lstm_tensors(rnn)[0][0]
    bad = wf.clone()
    bad[0, 0, 0, :, [0, 1]] = bad[0, 0, 0, :, [1, 0]]                 # i and f rows of unit 0 swapped
    assert not torch.equal(decode_fused_pairs(bad, 392, 196, 26, 196)[0][0], rounded(wi))
    bad = wf.clone()
    bad[1, 3, 1, 25, 7, 5] = 1.0                                        # x column 205: padding between bias and W_hh
    with pytest.raises(AssertionError, match="padding"):
        decode_fused_pairs(bad, 392, 196, 26, 196)
    rnn = _lstm(64, 32, 6)
    p = TS.pack_lstm_steps_tc(rnn)
    p["whh"][0] = p["whh"][0] * 2                                       # an unremoved factor 2 (g rows packed like i, f, o)
    assert not torch.equal(decode_lstm_steps(p)[0][1], rounded(lstm_tensors(rnn)[0][1]))
