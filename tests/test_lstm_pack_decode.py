"""CPU tests: every packed BLSTM weight layout decodes back to nn.LSTM's tensors exactly.

The decoders (tests/lstm_packs.py) invert each packer's index map and remove GATE_SCALE.  The decoded tensors must equal
fp16(w * scale) / scale of the nn.LSTM tensors bit for bit, and every padding row, column and k-core of the pack must be
zero.  The existing pack tests compare the training packer with the inference packer; these compare both with nn.LSTM,
and the GPU tests (test_gpu_lstm_tc.py) build their f64 references from the same decoders."""
import pytest
import torch

from lstm_packs import (decode_fused_pairs, decode_lstm_steps, decode_lstm_tc, decode_pack_block, lstm_tensors, rounded)
from urgent2026_challenge_track1_b200 import runtime_tc as TC
from urgent2026_challenge_track1_b200 import runtime_tc_steps as TS
from urgent2026_challenge_track1_b200 import training_tc as TT


def _lstm(N, H, seed):
    torch.manual_seed(seed)
    rnn = torch.nn.LSTM(N, H, batch_first=True, bidirectional=True)
    with torch.no_grad():
        for p in rnn.parameters():           # magnitudes that exercise fp16 rounding, subnormals and the exponent range
            p.copy_(torch.randn_like(p) * torch.exp2(torch.randint(-16, 3, p.shape).float()))
    return rnn


def _ws(rnn):
    return (rnn.weight_ih_l0, rnn.weight_hh_l0, rnn.bias_ih_l0, rnn.bias_hh_l0, rnn.weight_ih_l0_reverse,
            rnn.weight_hh_l0_reverse, rnn.bias_ih_l0_reverse, rnn.bias_hh_l0_reverse)


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


@pytest.mark.parametrize("P,U", [(7, 56), (14, 28)])
def test_pack_and_decode_lstm_fused7(P, U):
    rnn = _lstm(196, 392, P)
    wf = TC.pack_lstm_fused7(rnn, 26, 196, P=P, U=U)
    assert tuple(wf.shape) == (2, P, 2, 76, 2 * U, 8)
    for d, ((wi, wh, b), (dwi, dwh, db)) in enumerate(zip(lstm_tensors(rnn), decode_fused_pairs(wf, 392, 196, 26, 196))):
        _same(dwi, rounded(wi), f"fused{P}[{d}] W_ih")
        _same(dwh, rounded(wh), f"fused{P}[{d}] W_hh")
        _same(db, rounded(b), f"fused{P}[{d}] bias")


def test_pack_and_decode_lstm_steps_and_fused768():
    rnn = _lstm(384, 768, 3)
    p = TS.pack_lstm_steps_tc(rnn)
    assert tuple(p["wfused"].shape) == (2, 24, 2, 146, 64, 8)
    steps = decode_lstm_steps(p)
    fused = decode_fused_pairs(p["wfused"], 768, 384, 50, 384)
    for d, (wi, wh, b) in enumerate(lstm_tensors(rnn)):
        _same(steps[d][0], rounded(wi), f"steps wih[{d}]")
        _same(steps[d][1], rounded(wh), f"steps whh[{d}]")
        _same(steps[d][2], b.double(), f"steps bias[{d}] (f32, not rounded)")
        _same(fused[d][0], rounded(wi), f"fused768[{d}] W_ih")
        _same(fused[d][1], rounded(wh), f"fused768[{d}] W_hh")
        _same(fused[d][2], rounded(b), f"fused768[{d}] bias")


@pytest.mark.parametrize("N,H", [(196, 392), (384, 768), (36, 40)])
@pytest.mark.parametrize("fwd_steps", [True, False])
@pytest.mark.parametrize("narrow", [False, 2])
def test_pack_and_decode_pack_block(N, H, fwd_steps, narrow):
    rnn = _lstm(N, H, H + N)
    fc_w = torch.randn(N, 2 * H)
    p = TT.pack_block(*_ws(rnn), fc_w, narrow_bwd=narrow, fwd_steps=fwd_steps)
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


@pytest.mark.parametrize("geo,N,H,kc_in", [(7, 196, 392, 26), (14, 196, 392, 26), (768, 384, 768, 50)])
def test_pack_and_decode_fused_train(geo, N, H, kc_in):
    rnn = _lstm(N, H, geo)
    wf = TT.pack_fused_train(_ws(rnn), geo, kc_in, N)
    for d, ((wi, wh, b), (dwi, dwh, db)) in enumerate(zip(lstm_tensors(rnn), decode_fused_pairs(wf, H, N, kc_in, N))):
        _same(dwi, rounded(wi), f"train{geo}[{d}] W_ih")
        _same(dwh, rounded(wh), f"train{geo}[{d}] W_hh")
        _same(db, rounded(b), f"train{geo}[{d}] bias")


def test_pack_and_decode_rejects_a_corrupted_pack():
    """the decoders see a moved weight (wrong row), a non-zero padding element and a wrong scale."""
    rnn = _lstm(196, 392, 5)
    wf = TC.pack_lstm_fused7(rnn, 26, 196, P=7, U=56)
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
