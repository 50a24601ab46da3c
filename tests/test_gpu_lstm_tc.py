"""GPU tests (-m gpu) of the tensor-core BLSTM recurrences against f64 references, step by step:

  * the step kernels of csrc/gemm_tc.cu (EPI_LSTM_STEP / EPI_LSTM_BWD): bsrnn_lstm_step_tc, bsrnn_blstm_step_tc,
    bsrnn_blstm_step_train_tc, bsrnn_blstm_bwd_step_tc and the whole-sequence drivers bsrnn_blstm_train_fwd_tc / _bwd_tc;
  * the fused layer kernels of csrc/lstm_fused.cu (geometries 8, 7, 14 at H = 392 and 768, with their SAVE variants);
  * the gates_x recurrences of csrc/lstm_tc.cu (cluster schedules 4 / 5 / 6 / 8 / 9, the pair schedule 7, flag groups).

Method: TEACHER FORCING.  The kernels publish what they consumed: h_{t-1} is the fp16 y block of the previous step, the
training variants store c_t (f32) and the activated gates (fp16), BPTT stores dG_t.  The reference of step t takes the
kernel's own h_{t-1} (and c_{t-1}, dG_{t+1} where stored) and computes step t in f64, so errors do not compound and the
bar is ELEMENTWISE: a wrong, stale or racy read of h at any step, row or unit fails at that element.  Kernels that store no
c carry c in f64 from the teacher-forced gates; the c update is contractive (|f| <= 1), so its error bound only adds up.

The weights of the reference are the DECODED packs (tests/lstm_packs.py): kernel and reference multiply identical operands,
fp16-rounded bias included.  Bounds (derived, not fitted; K = k-cores of the contraction, 2 f32 ulps per K = 16 MMA step):

  z (i/f/o rows halved)  e_z = 2^-23 (K + 2) (sum |a||w| + |gx|)
  sigmoid gates          0.5 (e_z + TANH_ERR |tanh|) + 2^-24          g: e_z + TANH_ERR |g|
  c_t                    |c_{t-1}| e_f + |f| e_c,t-1 + |g| e_i + |i| e_g (+ products of errors) + f32 rounding
  h_t                    |tanh c| e_o + |o| (e_c + TANH_ERR |tanh c|) + f32 rounding, + half an fp16 ulp when stored
  saved gates            gate bound + half an fp16 ulp
  BPTT                   the EPI_LSTM_BWD formulas (gemm_tc.cu) with the saved fp16 gates and c as exact inputs

TANH_ERR = 2^-10.987 is the documented maximum relative error of tanh.approx.f32.  Every case prints its worst err/bound.
Memory the kernels must not write starts as a NaN bit pattern and must come back bit-identical; every case also checks
that each value the kernel stores -- padding rows of valid tiles included -- is finite and within its bound.
"""
import math
import os
import subprocess
import sys

import pytest
import torch

from lstm_packs import decode_fused_pairs, decode_lstm_tc, decode_pack_block
from test_gpu_gemm_tc import (GUARD, TANH_ERR, U23, U24, bits, half_ulp16, kb8_pack, kb8_unpack, sentinel, worst_ratio)

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CHILD = "BSRNN_LSTM_TC_TEST_CHILD"
F64 = torch.float64
DEV = "cuda"
GSC = (0.5, 0.5, 1.0, 0.5)


@pytest.fixture(scope="module")
def L():
    from urgent2026_challenge_track1_b200 import _lib
    _lib.require_device()
    return _lib


def gen(name):
    return torch.Generator(device=DEV).manual_seed(sum(map(ord, name)) * 7919)


def rand(g, *shape, scale=1.0):
    return torch.randn(*shape, device=DEV, generator=g, dtype=torch.float32) * scale


def gate_scale(H):
    return torch.tensor(GSC, dtype=F64, device=DEV).repeat_interleave(H)            # LSTM row order (gate*H + u)


def rand_lstm(g, N, H, sat=False):
    """per direction (W_ih, W_hh, b) f32 in nn.LSTM layout.  sat: weights x4 and forget bias +3 -- |c| grows well past 1 and
    the gates reach fp16 1.0."""
    out = []
    k = 1.0 / math.sqrt(H)
    for _ in range(2):
        wi = (torch.rand(4 * H, N, device=DEV, generator=g) * 2 - 1) * k
        wh = (torch.rand(4 * H, H, device=DEV, generator=g) * 2 - 1) * k
        b = (torch.rand(4 * H, device=DEV, generator=g) * 2 - 1) * 2 * k
        if sat:
            wi, wh, b = wi * 4, wh * 4, b * 4
            b[H:2 * H] += 3.0
        out.append((wi, wh, b))
    return out


def ratio(got, ref, bound):
    return worst_ratio(got, ref, bound)


# ---------------------------------------------------------------------------------------------------- reference cells
def cell_ref(zp, mag, kc, cprev, e_cprev):
    """one LSTM cell in f64.  zp: (rows, 4, H) pre-activations in the kernels' scale (i, f, o halved: sigmoid(z) =
    0.5 tanh(z/2) + 0.5), mag: the magnitude sum |a||w| (+ |gx|) of the same scale, kc: k-cores of the contraction,
    cprev / e_cprev: c_{t-1} and its error bound.  Returns the exact gates, c, h and their bounds (before fp16 rounding)."""
    ez = U23 * (kc + 2) * mag
    th = torch.tanh(zp)
    i, f, gg, o = 0.5 * th[:, 0] + 0.5, 0.5 * th[:, 1] + 0.5, th[:, 2], 0.5 * th[:, 3] + 0.5
    esig = lambda k: 0.5 * (ez[:, k] + TANH_ERR * th[:, k].abs()) + U24          # fma(tanh, .5, .5): one rounding of <= 1
    ei, ef, eo = esig(0), esig(1), esig(3)
    eg = ez[:, 2] + TANH_ERR * gg.abs()
    ig = i * gg
    c = f * cprev + ig
    A = cprev.abs() * ef + f * e_cprev + ef * e_cprev + gg.abs() * ei + i * eg + ei * eg
    ec = A + U24 * (ig.abs() + c.abs() + 2 * A)                                    # i*g and the fma round once each
    tc = torch.tanh(c)
    etc = ec + TANH_ERR * (tc.abs() + ec)                                          # tanh' <= 1
    h = o * tc
    B = tc.abs() * eo + o * etc + eo * etc
    eh = B + U24 * (h.abs() + B)
    return dict(gates=torch.stack([i, f, gg, o], 1), egates=torch.stack([ei, ef, eg, eo], 1), c=c, ec=ec, h=h, eh=eh)


def f16_bound(v, e):
    return e + half_ulp16(v.abs() + e)


def bwd_ref(acc, mag, kc, dy, sg, ct, cp, dc_in, e_dc):
    """EPI_LSTM_BWD in f64 (gemm_tc.cu): acc / mag (rows, H) = dG_{t+1} W_hh and its magnitude; dy (rows, H); sg (rows, 4, H)
    the saved fp16 gates i, f, g, o; ct / cp c_t / c_{t-1}; dc_in carry with bound e_dc.  Returns dG (rows, 4, H), dc_out and
    their bounds (dG before fp16 rounding)."""
    i, f, gg, o = sg[:, 0], sg[:, 1], sg[:, 2], sg[:, 3]
    eacc = U23 * (kc + 2) * mag
    dh = dy + acc
    edh = eacc + U24 * (dh.abs() + eacc)
    tc = torch.tanh(ct)
    etc = TANH_ERR * tc.abs()
    d_o = dh * tc
    edo = tc.abs() * edh + dh.abs() * etc + edh * etc + U24 * d_o.abs()
    s = 1 - tc * tc
    es = 2 * tc.abs() * etc + etc * etc + 2 * U24
    p = dh * o * s
    ep = o * (s.abs() * edh + dh.abs() * es + edh * es) + 2 * U24 * (p.abs() + o * (s.abs() * edh + dh.abs() * es))
    dc = dc_in + p
    edc = e_dc + ep + U24 * (dc.abs() + e_dc + ep)
    d_i, d_g, d_f = dc * gg, dc * i, dc * cp
    edi, edg, edf = gg.abs() * edc + U24 * d_i.abs(), i * edc + U24 * d_g.abs(), cp.abs() * edc + U24 * d_f.abs()
    dc_out = dc * f
    edco = f * edc + U24 * (dc_out.abs() + f * edc)
    gi, gf, gG, go = d_i * i * (1 - i), d_f * f * (1 - f), d_g * (1 - gg * gg), d_o * o * (1 - o)
    egi = i * (1 - i) * edi + 2 * U24 * (gi.abs() + i * (1 - i) * edi)
    egf = f * (1 - f) * edf + 2 * U24 * (gf.abs() + f * (1 - f) * edf)
    egG = (1 - gg * gg).abs() * edg + 2 * U24 * d_g.abs() + U24 * (gG.abs() + (1 - gg * gg).abs() * edg)
    ego = o * (1 - o) * edo + 2 * U24 * (go.abs() + o * (1 - o) * edo)
    return dict(dG=torch.stack([gi, gf, gG, go], 1), edG=torch.stack([egi, egf, egG, ego], 1), dc=dc_out, edc=edco)


def fwd_check(tag, H, kc, steps, W, hk, xin=None, gx=None, gk=None, ck=None, worst=None, verbose=True):
    """Teacher-forced check of a whole recurrence, both directions (direction 0 walks 0..steps-1, 1 walks steps-1..0).
    W[d] = (wx (4H, Kx) or None, wh (4H, H)) decoded f64 (scale removed); xin(p) -> (rows, Kx) operand of step p;
    gx(d, p) -> (rows, 4, H) input projection in the kernel's scale; hk(d, p) -> (rows, H) kernel h; gk(d, p) -> (rows, 4, H)
    saved gates; ck(d, p) -> (rows, H) saved c (then c is teacher-forced too, else carried in f64).  Returns worst ratios."""
    worst = dict(h=0.0, gates=0.0, c=0.0) if worst is None else worst
    S = gate_scale(H)[:, None]
    for d in range(2):
        wx, wh = W[d]
        whs, whsa = (wh * S).t(), (wh * S).abs().t()
        wxs, wxsa = ((wx * S).t(), (wx * S).abs().t()) if wx is not None else (None, None)
        prev, cprev, ecp = None, 0.0, 0.0
        for p in (range(steps) if d == 0 else range(steps - 1, -1, -1)):
            h_here = hk(d, p)
            rows = h_here.shape[0]
            if prev is None:
                zp = torch.zeros(rows, 4 * H, dtype=F64, device=DEV)
                mag = torch.zeros_like(zp)
            else:
                hp = hk(d, prev)
                zp, mag = hp @ whs, hp.abs() @ whsa
            if wx is not None:
                a = xin(p)
                zp, mag = zp + a @ wxs, mag + a.abs() @ wxsa
            zp, mag = zp.view(rows, 4, H), mag.view(rows, 4, H)
            if gx is not None:
                gv = gx(d, p)
                zp, mag = zp + gv, mag + gv.abs()
            if ck is not None:
                cprev, ecp = (ck(d, prev) if prev is not None else 0.0), 0.0
            r = cell_ref(zp, mag, kc, torch.as_tensor(cprev, dtype=F64, device=DEV), torch.as_tensor(ecp, dtype=F64, device=DEV))
            worst["h"] = max(worst["h"], ratio(h_here, r["h"], f16_bound(r["h"], r["eh"])))
            if gk is not None:
                worst["gates"] = max(worst["gates"], ratio(gk(d, p), r["gates"], f16_bound(r["gates"], r["egates"])))
            if ck is not None:
                worst["c"] = max(worst["c"], ratio(ck(d, p), r["c"], r["ec"]))
            else:
                cprev, ecp = r["c"], r["ec"]
            prev = p
    if verbose:
        print(f"{tag}: worst err/bound " + ", ".join(f"{k} {v:.3g}" for k, v in worst.items() if v > 0))
    return worst


def assert_worst(tag, worst):
    for k, v in worst.items():
        assert v <= 1.0, f"{tag}: {k} worst err/bound {v:.3g}"


def guarded(n, dtype, fill=None):
    """sentinel buffer of n elements + GUARD; `fill` (tensor of n) written into the first n."""
    b = sentinel(n + GUARD, dtype)
    if fill is not None:
        b[:n] = fill.reshape(-1).to(dtype)
    return b


def assert_guard(tag, buf, n):
    s = sentinel(GUARD, buf.dtype)
    assert torch.equal(bits(buf[n:]), bits(s)), f"{tag}: guard tail written"


def assert_finite(tag, t):
    assert bool(torch.isfinite(t).all()), f"{tag}: {int((~torch.isfinite(t)).sum())} stored values are not finite"


# ---------------------------------------------------------------------------------------------------- layout helpers
def kb8_rows(buf, tiles, kc, base=0, stride=None):
    """(tiles*128, kc*8) f64 matrix of KB8 blocks [kc][128][8] at buf[base + j*stride] (stride default kc*1024)."""
    stride = kc * 1024 if stride is None else stride
    v = buf.as_strided((tiles, kc, 128, 8), (stride, 1024, 8, 1), buf.storage_offset() + base)
    return kb8_unpack(v).double()


def gate_rows(mat, H, col0=0):
    """rows of packed gate columns col0 + 4u + gate -> (rows, 4, H) in LSTM order."""
    return mat[:, col0:col0 + 4 * H].double().view(-1, H, 4).permute(0, 2, 1)


def to_gate_cols(z):
    """(rows, 4, H) -> (rows, 4H) packed columns 4u + gate."""
    return z.permute(0, 2, 1).reshape(z.shape[0], -1)


def step_pack(w, H, BN, n_tiles, kc, scaled=True):
    """(4H, K) LSTM-order matrix -> KB8 [n_tiles][kc][BN][8] with rows 4u + gate (scaled) -- the step kernels' W layout."""
    u = torch.arange(H, device=DEV)
    perm = (torch.arange(4, device=DEV)[None, :] * H + u[:, None]).reshape(-1)
    m = w.float()[perm]
    if scaled:
        m = m * torch.tensor(GSC, device=DEV).repeat(H)[:, None]
    full = torch.zeros(n_tiles * BN, kc * 8, device=DEV)
    full[:4 * H, :m.shape[1]] = m
    return kb8_pack(full.half(), BN, kc)


def unpack_step_w(W8, H, K):
    """inverse of step_pack (scale removed), f64 (4H, K)."""
    m = kb8_unpack(W8).double()
    u = torch.arange(H, device=DEV)
    perm = (torch.arange(4, device=DEV)[:, None] + 4 * u[None, :]).reshape(-1)    # LSTM row g*H + u <- packed 4u + g
    return m[perm, :K] / gate_scale(H)[:, None]


# ---------------------------------------------------------------------------------------------------- a. step kernels
# (H, BN, n_tiles, m_tiles): every BN the packers choose (tile_width / _bn_for: widest divisor; _bn_cover; narrow 32 / 64), one
# n_tiles*BN > 4H, padded k-cores at H = 40 and 392
STEP_CASES = {
    "h32_bn128_m1": (32, 128, 1, 1),
    "h40_bn160_m2": (40, 160, 1, 2),
    "h40_bn96_cover_m3": (40, 96, 2, 3),              # 192 > 160 gate columns: the last chunk has no units
    "h64_bn256_m2": (64, 256, 1, 2),
    "h64_bn32_m3": (64, 32, 8, 3),
    "h392_bn224_m2": (392, 224, 7, 2),
    "h392_bn256_cover_m1": (392, 256, 7, 1),          # 1792 > 1568
    "h768_bn256_m3": (768, 256, 12, 3),
    "h768_bn96_m5": (768, 96, 32, 5),
}


def _step_inputs(name, H, m_tiles, n_tiles, BN, cprev_null=False, saturate=False):
    g = gen(name)
    kc = (H + 15) // 16 * 2
    rows = m_tiles * 128
    data = []
    for d in range(2):                                                     # different data per direction
        wh = (torch.rand(4 * H, H, device=DEV, generator=g) * 2 - 1) / math.sqrt(H) * (4 if saturate else 1)
        W8 = step_pack(wh, H, BN, n_tiles, kc)
        h = torch.zeros(rows, kc * 8, device=DEV)
        h[:, :H] = torch.tanh(rand(g, rows, H))
        A8 = kb8_pack(h.half(), 128, kc)
        c = None if cprev_null else rand(g, rows, H, scale=3.0 if saturate else 1.0)
        data.append(dict(W8=W8, A8=A8, wh=unpack_step_w(W8, H, H), h=kb8_unpack(A8).double()[:, :H], c=c))
    gx = rand(g, rows, 8 * H, scale=2.0).half()                          # rows of 8H: direction d at column 4H*d
    return kc, data, gx


def step_fwd_ref(H, kc, dd, gxd, cprev):
    """teacher-forced reference of one step of direction data dd with input projection gxd (rows, 4H packed) fp16."""
    S = gate_scale(H)[:, None]
    rows = dd["h"].shape[0]
    zp = (dd["h"] @ (dd["wh"] * S).t()).view(rows, 4, H)
    mag = (dd["h"].abs() @ (dd["wh"] * S).abs().t()).view(rows, 4, H)
    gv = gate_rows(gxd, H)
    cp = torch.zeros(rows, H, dtype=F64, device=DEV) if cprev is None else cprev.double()
    return cell_ref(zp + gv, mag + gv.abs(), kc, cp, torch.zeros_like(cp))


@pytest.mark.parametrize("name", sorted(STEP_CASES))
@pytest.mark.parametrize("kind", ["single", "blstm", "train", "train_c0"])
def test_step_kernel(L, name, kind):
    H, BN, n_tiles, m_tiles = STEP_CASES[name]
    if kind == "single" and name not in ("h40_bn96_cover_m3", "h768_bn256_m3", "h392_bn224_m2"):
        pytest.skip("single-direction launcher: three shapes")
    tag = f"{kind}[{name}]"
    c0 = kind == "train_c0"
    kc, data, gx = _step_inputs(tag, H, m_tiles, n_tiles, BN, cprev_null=c0)
    rows = m_tiles * 128
    n_y = m_tiles * kc * 1024
    st = L.stream_ptr()
    ys = []
    for d in range(2):
        y = guarded(n_y, torch.float16)
        if kc * 8 > H:                                               # the pad k-core starts (and must stay) zero
            y[:n_y].view(m_tiles, kc, 128, 8)[:, kc - 1] = 0
        ys.append(y)
    # one buffer of 8H-wide rows per direction holding only that direction's half (the other half and a guard tail are NaN
    # patterns: neither may be read or written)
    gxbs = []
    for d in range(2):
        b = guarded(rows * 8 * H, torch.float16)
        b[:rows * 8 * H].view(rows, 8 * H)[:, 4 * H * d:4 * H * (d + 1)] = gx[:, 4 * H * d:4 * H * (d + 1)]
        gxbs.append(b)
    gx_snaps = [bits(b).clone() for b in gxbs]
    train = kind.startswith("train")
    ndir = 1 if kind == "single" else 2
    cins = [None if c0 else guarded(rows * H, torch.float32, data[d]["c"]) for d in range(2)]
    couts = [guarded(rows * H, torch.float32) for d in range(2)] if train else cins
    args = []
    for d in range(2):
        args += [data[d]["A8"].data_ptr(), data[d]["W8"].data_ptr(), gxbs[d].data_ptr() + 2 * 4 * H * d]
        args += [L.ptr(cins[d]), couts[d].data_ptr(), ys[d].data_ptr()] if train else [cins[d].data_ptr(), ys[d].data_ptr()]
    if kind == "single":
        L.call("bsrnn_lstm_step_tc", *args[:5], m_tiles, n_tiles, BN, H, 8 * H, st)
    elif kind == "blstm":
        L.call("bsrnn_blstm_step_tc", *args, m_tiles, n_tiles, BN, H, 8 * H, st)
    else:
        L.call("bsrnn_blstm_step_train_tc", *args, m_tiles, n_tiles, BN, H, 8 * H, st)
    torch.cuda.synchronize()
    worst = dict(h=0.0, gates=0.0, c=0.0)
    for d in range(ndir):
        r = step_fwd_ref(H, kc, data[d], gx[:, 4 * H * d:4 * H * (d + 1)], data[d]["c"])
        hk = kb8_rows(ys[d], m_tiles, kc)
        assert_finite(tag, hk[:, :H])
        worst["h"] = max(worst["h"], ratio(hk[:, :H], r["h"], f16_bound(r["h"], r["eh"])))
        if kc * 8 > H:
            assert bool((hk[:, H:] == 0).all()), f"{tag}: pad k-core of h written"
        assert_guard(tag + " y", ys[d], n_y)
        ck = couts[d][:rows * H].view(rows, H).double()
        assert_finite(tag, ck)
        worst["c"] = max(worst["c"], ratio(ck, r["c"], r["ec"]))
        assert_guard(tag + " c", couts[d], rows * H)
        keep = torch.ones(rows * 8 * H + GUARD, dtype=torch.bool, device=DEV)
        if train:
            sg = gate_rows(gxbs[d][:rows * 8 * H].view(rows, 8 * H), H, 4 * H * d)
            worst["gates"] = max(worst["gates"], ratio(sg, r["gates"], f16_bound(r["gates"], r["egates"])))
            if not c0:
                assert torch.equal(bits(cins[d]), bits(guarded(rows * H, torch.float32, data[d]["c"]))), f"{tag}: c_prev written"
            keep[:rows * 8 * H].view(rows, 2, 4 * H)[:, d] = False
        assert torch.equal(bits(gxbs[d])[keep], gx_snaps[d][keep]), f"{tag}: gates row written outside this direction's half"
    gx_after = gxbs[0][:rows * 8 * H].view(rows, 8 * H)
    print(f"{tag}: worst err/bound " + ", ".join(f"{k} {v:.3g}" for k, v in worst.items() if v > 0))
    assert_worst(tag, worst)
    if name == "h392_bn224_m2" and kind == "train":
        # sharpness: one h element 3x its bound off, one saved gate a few fp16 ulps off
        r = step_fwd_ref(H, kc, data[0], gx[:, :4 * H], data[0]["c"])
        hk = kb8_rows(ys[0], m_tiles, kc)[:, :H]
        bnd = f16_bound(r["h"], r["eh"])
        bad = hk.clone()
        k = int(bnd.reshape(-1).argmax())
        bad.view(-1)[k] += 3 * bnd.view(-1)[k]
        assert ratio(bad, r["h"], bnd) > 1, f"{tag}: a 3x-bound h error passes"
        # (a gate in [0.5, 1): there an fp16 ulp is 2^-11, well above the z error; near 0 a few ulps are below it)
        sg = gate_rows(gx_after, H).contiguous()
        gb = f16_bound(r["gates"], r["egates"])
        k = int(torch.nonzero(((sg >= 0.5) & (sg < 0.999)).reshape(-1))[0])
        sg.view(-1)[k] += 3 * 2.0 ** -11
        assert ratio(sg, r["gates"], gb) > 1, f"{tag}: a saved gate 3 fp16 ulps off passes"


def test_step_and_step_train_agree(L):
    """bsrnn_blstm_step_tc and bsrnn_blstm_step_train_tc run the same cell code: identical h and c, bit for bit."""
    H, BN, n_tiles, m_tiles = STEP_CASES["h392_bn224_m2"]
    kc, data, gx = _step_inputs("agree", H, m_tiles, n_tiles, BN)
    rows, st = m_tiles * 128, L.stream_ptr()
    y1 = [torch.zeros(m_tiles * kc * 1024, dtype=torch.float16, device=DEV) for _ in range(2)]
    y2 = [torch.zeros_like(y) for y in y1]
    c1 = [data[d]["c"].clone() for d in range(2)]
    c2 = [torch.empty_like(c) for c in c1]
    gx2 = gx.clone()
    a1, a2 = [], []
    for d in range(2):
        a1 += [data[d]["A8"].data_ptr(), data[d]["W8"].data_ptr(), gx.data_ptr() + 2 * 4 * H * d, c1[d].data_ptr(), y1[d].data_ptr()]
        a2 += [data[d]["A8"].data_ptr(), data[d]["W8"].data_ptr(), gx2.data_ptr() + 2 * 4 * H * d, data[d]["c"].data_ptr(),
               c2[d].data_ptr(), y2[d].data_ptr()]
    L.call("bsrnn_blstm_step_tc", *a1, m_tiles, n_tiles, BN, H, 8 * H, st)
    L.call("bsrnn_blstm_step_train_tc", *a2, m_tiles, n_tiles, BN, H, 8 * H, st)
    torch.cuda.synchronize()
    for d in range(2):
        assert torch.equal(bits(y1[d]), bits(y2[d])), f"direction {d}: h differs"
        assert torch.equal(bits(c1[d]), bits(c2[d])), f"direction {d}: c differs"
    print("blstm_step_tc vs blstm_step_train_tc: h and c bit-identical")


# (H, BN, n_tiles, m_tiles, valid_rows, dy scale)
BWD_CASES = {
    "h40_bn64_m2_vr200": (40, 64, 1, 2, 200, 64.0),
    "h40_bn32_m1_vr1": (40, 32, 2, 1, 1, 1.0),            # 2*32 > 40: the second tile holds one 8-unit sub-block
    "h64_bn64_m3_vr300": (64, 64, 1, 3, 300, 2.0 ** -12),  # dG near the fp16 subnormal range
    "h392_bn224_m2_vr256": (392, 224, 2, 2, 256, 64.0),   # _bn_cover(392, 32): 2 x 224
    "h392_bn32_m1_vr77": (392, 32, 13, 1, 77, 1.0),       # narrow BPTT tiles, 416 > 392
    "h768_bn64_m2_vr129": (768, 64, 12, 2, 129, 64.0),
    "h768_bn256_m1_vr128": (768, 256, 3, 1, 128, 2.0 ** -12),
}


def _bwd_inputs(name, H, m_tiles, BN, n_tiles, dy_scale, cprev_null=False):
    g = gen(name)
    rows = m_tiles * 128
    kc = 4 * H // 8
    per = []
    for d in range(2):
        wh = (torch.rand(4 * H, H, device=DEV, generator=g) * 2 - 1) / math.sqrt(H)
        # W^T tiles: row = unit u, K = packed gate column 4u' + gate, TRUE weights
        u = torch.arange(H, device=DEV)
        pcol = (4 * u[None, :] + torch.arange(4, device=DEV)[:, None]).reshape(-1)
        wt = torch.zeros(n_tiles * BN, 4 * H, device=DEV)
        wt[:H, pcol] = wh.t()
        WT = kb8_pack(wt.half(), BN, kc)
        whd = kb8_unpack(WT).double()[:H][:, pcol].t().contiguous()             # (4H, H) LSTM order, as stored
        dG1 = (rand(g, rows, 4 * H) * dy_scale * 0.05).half()
        A8 = kb8_pack(dG1, 128, kc)
        sg = torch.rand(rows, 4, H, device=DEV, generator=g)
        sg[:, 2] = sg[:, 2] * 2 - 1
        sg = sg.half()
        ct = rand(g, rows, H, scale=2.0)
        cp = None if cprev_null else rand(g, rows, H, scale=2.0)
        dc = rand(g, rows, H, scale=dy_scale * 0.5)
        per.append(dict(WT=WT, wh=whd, A8=A8, dG1=dG1.double(), sg=sg, ct=ct, cp=cp, dc=dc))
    dy = (rand(g, rows, 2 * H) * dy_scale / 3).clamp(-dy_scale, dy_scale).half()
    return kc, per, dy


def bwd_step_ref(H, kc, pd, dyd, dc_in, e_dc=0.0):
    rows = pd["dG1"].shape[0]
    dgl = gate_rows(pd["dG1"], H).reshape(rows, 4 * H)                           # LSTM order
    acc, mag = dgl @ pd["wh"], dgl.abs() @ pd["wh"].abs()
    cp = torch.zeros(rows, H, dtype=F64, device=DEV) if pd["cp"] is None else pd["cp"].double()
    return bwd_ref(acc, mag, kc, dyd.double(), pd["sg"].double(), pd["ct"].double(), cp, dc_in.double(),
                   torch.as_tensor(e_dc, dtype=F64, device=DEV))


@pytest.mark.parametrize("name", sorted(BWD_CASES))
@pytest.mark.parametrize("cprev", ["cprev", "cprev_null"])
def test_bwd_step(L, name, cprev):
    H, BN, n_tiles, m_tiles, vr, dys = BWD_CASES[name]
    tag = f"bwd_step[{name},{cprev}]"
    kc, per, dy = _bwd_inputs(tag, H, m_tiles, BN, n_tiles, dys, cprev_null=cprev == "cprev_null")
    rows, st = m_tiles * 128, L.stream_ptr()
    n_g = rows * 4 * H
    outs, dcs, sgs, args = [], [], [], []
    dyb = guarded(rows * 2 * H, torch.float16, dy)
    for d in range(2):
        pd = per[d]
        sgb = guarded(rows * 8 * H, torch.float16)                     # rows of 8H, direction d's half at 4H*d
        sgb[:rows * 8 * H].view(rows, 2, H, 4)[:, d] = pd["sg"].permute(0, 2, 1)
        sgs.append(sgb)
        dcs.append(guarded(rows * H, torch.float32, pd["dc"]))
        outs.append(guarded(n_g, torch.float16))
        args += [pd["A8"].data_ptr(), pd["WT"].data_ptr(), sgb.data_ptr() + 2 * 4 * H * d, dyb.data_ptr() + 2 * H * d,
                 pd["ct"].data_ptr(), L.ptr(pd["cp"]), dcs[d].data_ptr(), outs[d].data_ptr()]
    snaps = [bits(b).clone() for b in sgs] + [bits(dyb).clone()]
    L.call("bsrnn_blstm_bwd_step_tc", *args, m_tiles, n_tiles, BN, H, 8 * H, 2 * H, vr, st)
    torch.cuda.synchronize()
    worst = dict(dG=0.0, dc=0.0)
    for d in range(2):
        pd = per[d]
        r = bwd_step_ref(H, kc, pd, dy[:, H * d:H * (d + 1)], pd["dc"])
        got = gate_rows(kb8_rows(outs[d], m_tiles, kc), H)
        assert_guard(tag + " dG", outs[d], n_g)
        live = torch.arange(rows, device=DEV) < vr
        assert bool((got[~live] == 0).all()) and bool((bits(outs[d][:n_g]).view(m_tiles, kc, 128, 8).permute(0, 2, 1, 3)
                                                        .reshape(rows, -1)[~live] == 0).all()), f"{tag}: dG rows >= valid_rows not +0"
        worst["dG"] = max(worst["dG"], ratio(got[live], r["dG"][live], f16_bound(r["dG"], r["edG"])[live]))
        dck = dcs[d][:rows * H].view(rows, H)
        worst["dc"] = max(worst["dc"], ratio(dck[live].double(), r["dc"][live], r["edc"][live]))
        assert torch.equal(bits(dck[~live]), bits(pd["dc"][~live])), f"{tag}: dc rows >= valid_rows written"
        assert_guard(tag + " dc", dcs[d], rows * H)
        if d == 0 and name == "h392_bn224_m2_vr256" and cprev == "cprev":
            gb = f16_bound(r["dG"], r["edG"])[live]
            bad = got.clone()
            bad[:128, :2] = 0                                           # one dG core (8 gate columns of 2 units) zeroed
            assert ratio(bad[live], r["dG"][live], gb) > 1, f"{tag}: a zeroed dG core passes"
    for b, s in zip(sgs + [dyb], snaps):
        assert torch.equal(bits(b), s), f"{tag}: an input buffer was written"
    print(f"{tag}: worst err/bound dG {worst['dG']:.3g}, dc {worst['dc']:.3g}")
    assert_worst(tag, worst)


# ---------------------------------------------------------------------------------------------------- b. sequence drivers
@pytest.mark.parametrize("H,tiles,steps,R", [(40, 2, 9, 200), (392, 1, 5, 77), (768, 2, 3, 129)])
def test_train_drivers(L, H, tiles, steps, R):
    """bsrnn_blstm_train_fwd_tc / _bwd_tc, teacher-forced at every step of both directions.  The backward walks each direction
    against its forward order (f: steps-1..0, b: 0..steps-1); the reference pairs dG_t with dG_{t+1} of the same direction."""
    tag = f"train_drivers[H{H},t{tiles},s{steps},R{R}]"
    g = gen(tag)
    st = L.stream_ptr()
    kc = (H + 15) // 16 * 2
    kg = 4 * H // 8
    rows = tiles * 128
    m_all = steps * tiles
    from urgent2026_challenge_track1_b200 import training_tc as TT
    ws = []
    for (wi, wh, b) in rand_lstm(g, 16, H):
        ws += [wi, wh, b, torch.zeros_like(b)]
    p = TT.pack_block(*ws, torch.zeros(16, 2 * H, device=DEV), narrow_bwd=tiles, fwd_steps=True)
    cpu = lambda v: [t.cpu() for t in v] if isinstance(v, list) else (v.cpu() if torch.is_tensor(v) else v)
    dec = [{k: v.to(DEV) for k, v in e.items()} for e in decode_pack_block({k: cpu(v) for k, v in p.items()})]
    proj = (rand(g, steps * rows, 8 * H, scale=1.5)).half()
    gates = guarded(steps * rows * 8 * H, torch.float16, proj)
    y = [guarded(m_all * kc * 1024, torch.float16, torch.zeros(m_all * kc * 1024, device=DEV)) for _ in range(2)]
    c = [guarded(steps * rows * H, torch.float32) for _ in range(2)]
    zero = torch.zeros(tiles * max(kc, kg) * 1024, dtype=torch.float16, device=DEV)
    L.call("bsrnn_blstm_train_fwd_tc", zero.data_ptr(), y[0].data_ptr(), y[1].data_ptr(), p["whh"][0].data_ptr(),
           p["whh"][1].data_ptr(), gates.data_ptr(), c[0].data_ptr(), c[1].data_ptr(), steps, tiles, p["n_tiles"], p["BN"], H, st)
    torch.cuda.synchronize()
    for d in range(2):
        assert_guard(tag, y[d], m_all * kc * 1024)
        assert_guard(tag, c[d], steps * rows * H)
    assert_guard(tag, gates, steps * rows * 8 * H)
    G = gates[:steps * rows * 8 * H].view(steps, rows, 8 * H)
    P = proj.view(steps, rows, 8 * H)
    Y = [kb8_rows(y[d], m_all, kc).view(steps, rows, kc * 8) for d in range(2)]
    C = [c[d][:steps * rows * H].view(steps, rows, H).double() for d in range(2)]
    for d in range(2):
        if kc * 8 > H:
            assert bool((Y[d][..., H:] == 0).all()), f"{tag}: pad k-core of y written"
        assert_finite(tag, Y[d][..., :H])
        assert_finite(tag, C[d])
    W = [(None, dec[d]["whh"]) for d in range(2)]
    worst = fwd_check(tag + " fwd", H, kc, steps, W, hk=lambda d, p_: Y[d][p_, :, :H],
                      gx=lambda d, p_: gate_rows(P[p_], H, 4 * H * d),
                      gk=lambda d, p_: gate_rows(G[p_], H, 4 * H * d), ck=lambda d, p_: C[d][p_])
    assert_worst(tag + " fwd", worst)
    # ---- backward
    dy = (rand(g, steps * rows, 2 * H) * 20).clamp(-64, 64).half()
    dG = [guarded(m_all * kg * 1024, torch.float16) for _ in range(2)]
    dc = [guarded(rows * H, torch.float32, torch.zeros(rows * H, device=DEV)) for _ in range(2)]
    L.call("bsrnn_blstm_train_bwd_tc", zero.data_ptr(), dG[0].data_ptr(), dG[1].data_ptr(), p["whhT"][0].data_ptr(),
           p["whhT"][1].data_ptr(), gates.data_ptr(), dy.data_ptr(), c[0].data_ptr(), c[1].data_ptr(), dc[0].data_ptr(),
           dc[1].data_ptr(), steps, tiles, p["nt_h"], p["bn_h"], H, R, st)
    torch.cuda.synchronize()
    DY = dy.view(steps, rows, 2 * H).double()
    live = torch.arange(rows, device=DEV) < R
    wb = dict(dG=0.0, dc=0.0)
    for d in range(2):
        assert_guard(tag, dG[d], m_all * kg * 1024)
        assert_guard(tag, dc[d], rows * H)
        DG = gate_rows(kb8_rows(dG[d], m_all, kg), H).reshape(steps, rows, 4, H)
        wt = dec[d]["whhT"]                                                # (4H, H) TRUE weights
        order = range(steps - 1, -1, -1) if d == 0 else range(steps)
        nxt, dcr, edc = None, torch.zeros(rows, H, dtype=F64, device=DEV), torch.zeros(rows, H, dtype=F64, device=DEV)
        for p_ in order:
            if nxt is None:
                acc = mag = torch.zeros(rows, H, dtype=F64, device=DEV)
            else:
                a = DG[nxt].reshape(rows, 4 * H)
                acc, mag = a @ wt, a.abs() @ wt.abs()
            prevc = p_ - 1 if d == 0 else p_ + 1
            cp = C[d][prevc] if 0 <= prevc < steps else torch.zeros(rows, H, dtype=F64, device=DEV)
            r = bwd_ref(acc, mag, kg, DY[p_, :, H * d:H * (d + 1)], gate_rows(G[p_], H, 4 * H * d), C[d][p_], cp, dcr, edc)
            assert bool((DG[p_][~live] == 0).all()), f"{tag}: dG rows >= valid_rows not zero"
            wb["dG"] = max(wb["dG"], ratio(DG[p_][live], r["dG"][live], f16_bound(r["dG"], r["edG"])[live]))
            dcr, edc = r["dc"], r["edc"]
            nxt = p_
        dck = dc[d][:rows * H].view(rows, H)
        wb["dc"] = max(wb["dc"], ratio(dck[live].double(), dcr[live], edc[live]))
        assert bool((dck[~live] == 0).all()), f"{tag}: dc rows >= valid_rows written"
    print(f"{tag} bwd: worst err/bound dG {wb['dG']:.3g}, dc {wb['dc']:.3g}")
    assert_worst(tag + " bwd", wb)


# ---------------------------------------------------------------------------------------------------- c. fused layer kernels
GEOS = {   # geo -> (H, N, kc_in, kc_h, P, U)
    8: (392, 196, 26, 50, 8, 49), 7: (392, 196, 26, 50, 7, 56), 14: (392, 196, 26, 50, 14, 28), 768: (768, 384, 50, 96, 24, 32)}


def fused_pack(geo, ws):
    from urgent2026_challenge_track1_b200 import runtime_tc as TC
    H, N, kc_in, kc_h, P, U = GEOS[geo]
    flat = []
    for (wi, wh, b) in ws:
        flat += [wi, wh, b, torch.zeros_like(b)]
    wf = TC.pack_fused(flat, geo, kc_in, N)
    W = []
    for wi, wh, b in decode_fused_pairs(wf.cpu(), H, N, kc_in, N):
        W.append((torch.cat([wi, b[:, None]], 1).to(DEV), wh.to(DEV)))     # x operand: columns 0..N-1 and the one column N
    return wf.contiguous(), W


def make_xhat(g, steps, tiles, N, kc_in, scale=1.0):
    x = torch.zeros(steps * tiles * 128, kc_in * 8, device=DEV)
    x[:, :N] = rand(g, steps * tiles * 128, N, scale=scale)
    x[:, N] = 1.0
    xh = x.half()
    return kb8_pack(xh, 128, kc_in).reshape(-1).contiguous(), xh.double()[:, :N + 1]


class FusedBufs:
    """y (+ gates, c, scratch for SAVE) with sentinel fill, pad core zero, guard tails; layout per geometry."""

    def __init__(self, L, geo, steps, tiles, train, y_layout="sep", gap=0):
        H, N, kc_in, kc_h, P, U = GEOS[geo]
        self.geo, self.steps, self.tiles, self.train, self.kc_h, self.H = geo, steps, tiles, train, kc_h, H
        blk = kc_h * 1024
        m_all = steps * tiles
        if geo in (8, 7, 14) and not train:               # inference H = 392: one interleaved buffer [..][dir][50][128][8]
            self.y_stride, self.offs, nbuf = 2 * blk, (0, blk), 1
        elif y_layout == "inter":                           # H = 768 interleaved: y_b = y_f + 96*1024, stride 2*96*1024
            self.y_stride, self.offs, nbuf = 2 * blk, (0, blk), 1
        else:
            self.y_stride, self.offs, nbuf = blk + gap, (0, 0), 2
        self.ny = m_all * self.y_stride
        self.y = [guarded(self.ny, torch.float16) for _ in range(nbuf)]
        for d in range(2):
            yb = self.ybuf(d)
            v = yb.as_strided((m_all, kc_h, 128, 8), (self.y_stride, 1024, 8, 1), yb.storage_offset() + self.offs[d])
            if kc_h * 8 > H:
                v[:, kc_h - 1] = 0                            # pad k-core starts zero and must stay zero
        self.snap = [bits(b).clone() for b in self.y]
        self.zero = torch.zeros(blk, dtype=torch.float16, device=DEV)
        self.sync = torch.zeros(L.lib().bsrnn_blstm_fused_sync_bytes() // 4, dtype=torch.int32, device=DEV)
        if train:
            fn = "bsrnn_blstm_fused768_train_scratch_bytes" if geo == 768 else "bsrnn_blstm_fused_train_scratch_bytes"
            self.nscr = int(getattr(L.lib(), fn)(steps, tiles))
            self.scratch = guarded(self.nscr // 2, torch.float16)
            self.ng = m_all * 128 * 8 * H
            self.gates = guarded(self.ng, torch.float16)
            self.nc = m_all * 128 * H
            self.c = [guarded(self.nc, torch.float32) for _ in range(2)]

    def ybuf(self, d):
        return self.y[0] if len(self.y) == 1 else self.y[d]

    def yptr(self, d):
        return self.ybuf(d).data_ptr() + 2 * self.offs[d]

    def h(self, d, p):
        yb = self.ybuf(d)
        return kb8_rows(yb, self.tiles, self.kc_h, base=self.offs[d] + p * self.tiles * self.y_stride, stride=self.y_stride)

    def launch(self, L, xhat, wf, R, slots, max_groups):
        st = L.stream_ptr()
        a = (xhat.data_ptr(), wf.data_ptr(), self.zero.data_ptr())
        tail = (R, self.steps, self.tiles, max_groups, slots, self.sync.data_ptr(), st)
        if self.train:
            mid = (self.yptr(0), self.yptr(1), self.y_stride, self.gates.data_ptr(), self.c[0].data_ptr(), self.c[1].data_ptr(),
                   self.scratch.data_ptr())
            if self.geo == 768:
                L.call("bsrnn_blstm_fused768_train_tc", *a, *mid, *tail)
            else:
                L.call("bsrnn_blstm_fused_train_tc", self.geo, *a, *mid, *tail)
        elif self.geo == 768:
            L.call("bsrnn_blstm_fused768_tc", *a, self.yptr(0), self.yptr(1), self.y_stride, *tail)
        else:
            fn = {8: "bsrnn_blstm_fused_tc", 7: "bsrnn_blstm_fused7_tc", 14: "bsrnn_blstm_fused14_tc"}[self.geo]
            L.call(fn, *a, self.y[0].data_ptr(), *tail)
        torch.cuda.synchronize()

    def check_memory(self, tag):
        """bits outside the stored y cores unchanged (gaps, pad core, guard); scratch / gates / c guards."""
        m_all = self.steps * self.tiles
        H, kc_h = self.H, self.kc_h
        for i, yb in enumerate(self.y):
            keep = torch.ones(yb.numel(), dtype=torch.bool, device=DEV)
            ds = (0, 1) if len(self.y) == 1 else (i,)
            for d in ds:
                v = keep.as_strided((m_all, kc_h, 128, 8), (self.y_stride, 1024, 8, 1), self.offs[d])
                v[:, :H // 8] = False
            assert torch.equal(bits(yb)[keep], self.snap[i][keep]), f"{tag}: y written outside the h cores (gap, pad core or guard)"
        if self.train:
            assert_guard(tag + " scratch", self.scratch, self.nscr // 2)
            assert_guard(tag + " gates", self.gates, self.ng)
            for cb in self.c:
                assert_guard(tag + " c", cb, self.nc)

    def saved(self):
        m_all, H = self.steps * self.tiles, self.H
        G = self.gates[:self.ng].view(self.steps, self.tiles * 128, 8 * H)
        C = [cb[:self.nc].view(self.steps, self.tiles * 128, H).double() for cb in self.c]
        return G, C

    def all_h(self):
        return [torch.stack([self.h(d, p) for p in range(self.steps)]) for d in range(2)]


def check_fused(tag, B, W, X, geo, verbose=True):
    H, N, kc_in, kc_h, P, U = GEOS[geo]
    rows = B.tiles * 128
    Y = B.all_h()
    for d in range(2):
        assert_finite(tag, Y[d][..., :H])
    xin = lambda p: X[p * rows:(p + 1) * rows]
    kw = {}
    if B.train:
        G, C = B.saved()
        assert_finite(tag + " gates", G.double())
        for d in range(2):
            assert_finite(tag + " c", C[d])
        kw = dict(gk=lambda d, p: gate_rows(G[p], H, 4 * H * d), ck=lambda d, p: C[d][p])
    return fwd_check(tag, H, kc_in + kc_h, B.steps, W, hk=lambda d, p: Y[d][p, :, :H], xin=xin, verbose=verbose, **kw)


# (geo, R, steps, seq_tiles (0 = ceil(R/128)), saturating, train, y layout / gap)
FUSED_CASES = {
    "g8_r300_s9": (8, 300, 9, 0, False, False, "sep", 0),
    "g8_r1_s2": (8, 1, 2, 0, False, False, "sep", 0),
    "g7_r129_s9_sat": (7, 129, 9, 0, True, False, "sep", 0),
    "g7_r2300_s40": (7, 2300, 40, 0, False, False, "sep", 0),
    "g14_r127_s2": (14, 127, 2, 0, False, False, "sep", 0),
    "g14_r128_s1_tiles3": (14, 128, 1, 3, False, False, "sep", 0),
    "g768_r300_s9_gap": (768, 300, 9, 0, False, False, "sep", 64),
    "g768_r2300_s40_inter": (768, 2300, 40, 0, False, False, "inter", 0),
    "g768_r129_s2_sat": (768, 129, 2, 0, True, False, "sep", 0),
    "g7S_r300_s9": (7, 300, 9, 0, False, True, "sep", 0),
    "g14S_r129_s9_sat": (14, 129, 9, 0, True, True, "sep", 0),
    "g768S_r300_s9": (768, 300, 9, 0, False, True, "sep", 0),
    "g768S_r2300_s40_gap": (768, 2300, 40, 0, True, True, "sep", 64),
    "g14S_r1_s2_tiles4": (14, 1, 2, 4, False, True, "sep", 0),
}
CONFIGS = [(0, 0), (1, 1), (2, 3), (3, 0), (1, 3)]        # (slots, max_groups)


@pytest.mark.parametrize("name", sorted(FUSED_CASES))
def test_fused_layer(L, name):
    geo, R, steps, seq_tiles, sat, train, layout, gap = FUSED_CASES[name]
    H, N, kc_in, kc_h, P, U = GEOS[geo]
    tiles = seq_tiles or -(-R // 128)
    g = gen(name)
    wf, W = fused_pack(geo, rand_lstm(g, N, H, sat))
    xhat, X = make_xhat(g, steps, tiles, N, kc_in, scale=2.0 if sat else 1.0)
    B = FusedBufs(L, geo, steps, tiles, train, layout, gap)
    worst = None
    first = None
    for k, (slots, mg) in enumerate(CONFIGS):
        B.launch(L, xhat, wf, R, slots, mg)
        tag = f"fused[{name}] slots={slots} max_groups={mg}"
        B.check_memory(tag)
        cur = [bits(y).clone() for y in B.y] + ([bits(B.gates).clone()] + [bits(c).clone() for c in B.c] if train else [])
        if k == 0:
            worst = check_fused(tag, B, W, X, geo)
            assert_worst(tag, worst)
            first = cur
            if name in ("g7S_r300_s9", "g768S_r300_s9", "g8_r300_s9", "g768_r300_s9_gap"):
                sharpness(tag, B, W, X, geo)
        else:
            same = all(torch.equal(a, b) for a, b in zip(first, cur))
            print(f"{tag}: bit-identical to slots=0 max_groups=0: {same}")
            if not same:
                w = check_fused(tag, B, W, X, geo)
                assert_worst(tag, w)
            assert same, f"{tag}: outputs differ from the first configuration"
    # stale reads: a second launch with DIFFERENT inputs into the same y / gates / c / sync buffers
    xhat2, X2 = make_xhat(gen(name + "#2"), steps, tiles, N, kc_in, scale=2.0 if sat else 1.0)
    B.launch(L, xhat2, wf, R, 0, 0)
    tag = f"fused[{name}] relaunch"
    B.check_memory(tag)
    assert_worst(tag, check_fused(tag, B, W, X2, geo))


def sharpness(tag, B, W, X, geo):
    """corrupt the kernel's real output; the teacher-forced check must reject each corruption."""
    H = GEOS[geo][0]
    yb = B.ybuf(0)
    s = B.steps // 2
    r0 = 5
    keep = yb.clone()
    try:
        # h of step s replaced by h of step s-1 for one row (direction 0)
        blk = lambda p: yb.as_strided((B.kc_h, 128, 8), (1024, 8, 1), yb.storage_offset() + B.offs[0] + p * B.tiles * B.y_stride)
        if B.steps >= 2:
            blk(s)[:, r0] = blk(s - 1)[:, r0].clone()
            w = check_fused(tag + " [h_t <- h_t-1]", B, W, X, geo, verbose=False)
            assert w["h"] > 1, f"{tag}: h_t replaced by h_t-1 in one row passes"
            yb.copy_(keep)
        # one h element 3x its bound off: the bound of that element is at most a few fp16 ulps, 3 * 2^-11 * |h| + 2^-20 exceeds it
        v = blk(s)[3, r0, 2]
        blk(s)[3, r0, 2] = (v.float() + 3 * max(2.0 ** -9 * abs(float(v)), 2.0 ** -18)).half()
        w = check_fused(tag + " [h +3 bound]", B, W, X, geo, verbose=False)
        assert w["h"] > 1, f"{tag}: a 3x-bound h error passes"
    finally:
        yb.copy_(keep)
    if B.train:
        gk = B.gates.clone()
        try:
            G = B.gates[:B.ng].view(B.steps, B.tiles * 128, 8 * H)
            row = G[s, r0].float()
            col = int(torch.nonzero((row >= 0.5) & (row < 0.999))[0])          # a gate in [0.5, 1): fp16 ulp 2^-11
            G[s, r0, col] = (row[col] + 3 * 2.0 ** -11).half()
            w = check_fused(tag + " [gate +3 ulp]", B, W, X, geo, verbose=False)
            assert w["gates"] > 1, f"{tag}: a saved gate 3 fp16 ulps off passes"
        finally:
            B.gates.copy_(gk)
    print(f"{tag}: every corruption rejected")


def test_fused_twins_bit_identical(L):
    """a SAVE kernel and its inference twin (7 / 7S, 14 / 14S, 768 / 768S) run the same cell code: bit-identical y; and
    geometries 8 / 7 / 14 compared with each other (reported; they split the gate columns differently)."""
    g = gen("twins")
    R, steps = 300, 9
    tiles = -(-R // 128)
    res = {}
    for H, N, kc_in, geos in ((392, 196, 26, (8, 7, 14)), (768, 384, 50, (768,))):
        ws = rand_lstm(g, N, H)
        xhat, X = make_xhat(g, steps, tiles, N, kc_in)
        for geo in geos:
            wf, _ = fused_pack(geo, ws)
            for train in ((False, True) if geo != 8 else (False,)):
                B = FusedBufs(L, geo, steps, tiles, train)
                B.launch(L, xhat, wf, R, 0, 0)
                res[(geo, train)] = [torch.stack([B.h(d, p) for p in range(steps)]) for d in range(2)]
    diffs = []
    for geo in (7, 14, 768):
        same = all(torch.equal(a, b) for a, b in zip(res[(geo, False)], res[(geo, True)]))
        print(f"geometry {geo}: inference vs SAVE y bit-identical: {same}")
        if not same:
            diffs.append(geo)
    for a, b in ((8, 7), (8, 14), (7, 14)):
        ne = sum(int((x != y).sum()) for x, y in zip(res[(a, False)], res[(b, False)]))
        print(f"geometry {a} vs {b}: {ne} of {sum(x.numel() for x in res[(a, False)])} y elements differ")
    assert not diffs, f"SAVE and inference kernels differ at geometries {diffs}"


# ---------------------------------------------------------------------------------------------------- d. lstm_tc.cu recurrences
def tc_inputs(g, R, steps, tiles):
    from urgent2026_challenge_track1_b200 import runtime_tc as TC
    ws = rand_lstm(g, 196, 392)
    rnn = torch.nn.LSTM(196, 392, bidirectional=True)
    with torch.no_grad():
        for (wi, wh, b), sfx in zip(ws, ("", "_reverse")):
            getattr(rnn, "weight_ih_l0" + sfx).copy_(wi.cpu())
            getattr(rnn, "weight_hh_l0" + sfx).copy_(wh.cpu())
            getattr(rnn, "bias_ih_l0" + sfx).copy_(b.cpu())
            getattr(rnn, "bias_hh_l0" + sfx).zero_()
    p = TC.pack_lstm_tc(rnn)
    whh = p["whh"].to(DEV).contiguous()
    W = [(None, w.to(DEV)) for w in decode_lstm_tc(p)["whh"]]
    # gates_x [step][tile][dir][q][26][128][8] fp16, random (the pad columns 196..207 of each q too)
    gxt = (rand(g, steps * tiles * 2 * 8 * 26 * 1024, scale=1.5)).half()
    return whh, W, gxt


def tc_gx(gxt, steps, tiles):
    """(d, p) -> (rows, 4, H) input projection in the kernel's scale, from the documented gates_x layout."""
    v = gxt.view(steps, tiles, 2, 8, 26, 128, 8).permute(0, 1, 5, 2, 3, 4, 6).reshape(steps, tiles * 128, 2, 8, 208)
    v = v[..., :196].reshape(steps, tiles * 128, 2, 8, 49, 4)             # packed column 4u + gate of CTA q
    v = v.permute(0, 1, 2, 5, 3, 4).reshape(steps, tiles * 128, 2, 4, 392)  # [gate][49q + u]
    return lambda d, p: v[p, :, d].double()


SCHEDULES = ["v4", "v5", "v6", "v7", "v8", "v9", "flag"]
TC_CASES = {"r300_s9": (300, 9), "r129_s2": (129, 2), "r1_s1": (1, 1)}
TC_CONFIGS = [(0, 0), (1, 1), (3, 2), (2, 1)]        # (slots, max_clusters / max_groups)
_TC_Y = {}


@pytest.mark.parametrize("case", sorted(TC_CASES))
@pytest.mark.parametrize("sched", SCHEDULES)
def test_lstm_tc_recurrence(L, sched, case):
    R, steps = TC_CASES[case]
    tiles = -(-R // 128)
    g = gen("tc" + case)
    whh, W, gxt = tc_inputs(g, R, steps, tiles)
    gxf = tc_gx(gxt, steps, tiles)
    ny = steps * tiles * 2 * 50 * 1024
    y = guarded(ny, torch.float16)
    y[:ny].view(steps * tiles, 2, 50, 1024)[:, :, 49] = 0
    snap = bits(y).clone()
    zero = torch.zeros(50 * 1024, dtype=torch.float16, device=DEV)
    sync = torch.zeros(L.lib().bsrnn_blstm_tc_sync_bytes() // 4, dtype=torch.int32, device=DEV)
    st = L.stream_ptr()

    def run(gx, slots, mc):
        if sched == "flag":
            L.call("bsrnn_blstm_recurrence_tc_flag", gx.data_ptr(), whh.data_ptr(), zero.data_ptr(), y.data_ptr(), R, steps, tiles, mc,
                   slots, sync.data_ptr(), st)
        else:
            L.lib().bsrnn_debug_set_lstm_schedule(int(sched[1:]))
            try:
                L.call("bsrnn_blstm_recurrence_tc_ex", gx.data_ptr(), whh.data_ptr(), zero.data_ptr(), y.data_ptr(), R, steps, tiles,
                       mc, slots, st)
            finally:
                L.lib().bsrnn_debug_set_lstm_schedule(-1)
        torch.cuda.synchronize()

    def hk_of():
        Y = kb8_rows(y, steps * tiles * 2, 50).view(steps, tiles, 2, 128, 400)
        return lambda d, p: Y[p, :, d].reshape(tiles * 128, 400)[:, :392]

    def mem(tag):
        keep = torch.ones(y.numel(), dtype=torch.bool, device=DEV)
        keep[:ny].view(steps * tiles * 2, 50, 1024)[:, :49] = False
        assert torch.equal(bits(y)[keep], snap[keep]), f"{tag}: y written outside the h cores (pad core 49 or guard)"

    first = None
    for k, (slots, mc) in enumerate(TC_CONFIGS):
        tag = f"lstm_tc[{sched},{case}] slots={slots} max={mc}"
        run(gxt, slots, mc)
        mem(tag)
        cur = bits(y).clone()
        if k == 0:
            assert_finite(tag, y[:ny].view(-1, 50, 1024)[:, :49].double())
            w = fwd_check(tag, 392, 50, steps, W, hk=hk_of(), gx=lambda d, p: gxf(d, p))
            assert_worst(tag, w)
            first = cur
            if sched == "v8" and case == "r300_s9":
                hk = hk_of()
                good = y.clone()
                y.view(-1)[:ny].view(steps, tiles, 2, 50, 128, 8)[4, 0, 0, :, 7] = \
                    y.view(-1)[:ny].view(steps, tiles, 2, 50, 128, 8)[3, 0, 0, :, 7].clone()
                w2 = fwd_check(tag + " [h_t <- h_t-1]", 392, 50, steps, W, hk=hk_of(), gx=lambda d, p: gxf(d, p), verbose=False)
                y.copy_(good)
                assert w2["h"] > 1, f"{tag}: h_t replaced by h_t-1 in one row passes"
        else:
            same = torch.equal(first, cur)
            print(f"{tag}: bit-identical to the first configuration: {same}")
            assert same, f"{tag}: y differs from slots=0 max=0"
    # stale reads: different gates_x into the same y / sync
    gxt2 = (rand(gen("tc2" + case), gxt.numel(), scale=1.5)).half()
    run(gxt2, 0, 0)
    tag = f"lstm_tc[{sched},{case}] relaunch"
    mem(tag)
    assert_worst(tag, fwd_check(tag, 392, 50, steps, W, hk=hk_of(), gx=tc_gx(gxt2, steps, tiles)))
    _TC_Y[(sched, case)] = first


def test_lstm_tc_schedules_compared():
    """the lstm_tc.cu schedules against each other, bit for bit (reported; each was checked against its bound above)."""
    cases = sorted({c for _, c in _TC_Y})
    if not cases:
        pytest.skip("no recurrence case ran in this process")
    for case in cases:
        ref = _TC_Y.get(("v8", case))
        for s in SCHEDULES:
            y = _TC_Y.get((s, case))
            if ref is None or y is None:
                continue
            print(f"lstm_tc {case}: {s} vs v8: {int((y != ref).sum())} of {y.numel()} y bit patterns differ")


# ---------------------------------------------------------------------------------------------------- i. launcher switches
def run_child(env, kexpr):
    env = dict(os.environ, **env, **{CHILD: "1", "COLUMNS": "250"})
    cmd = [sys.executable, "-m", "pytest", os.path.abspath(__file__), "-m", "gpu", "-q", "-x", "-p", "no:cacheprovider", "-k", kexpr]
    r = subprocess.run(cmd, cwd=ROOT, env=env, capture_output=True, text=True, timeout=900)
    return r.returncode, "\n".join((r.stdout + r.stderr).splitlines()[-25:])


child_only = pytest.mark.skipif(os.environ.get(CHILD) == "1", reason="runs in the parent process only")
SWITCHES = [
    ({"BSRNN_FUSED14_CLS": "4"}, "fused_layer and g14 and not g14S"),
]


@child_only
@pytest.mark.parametrize("env,kexpr", SWITCHES, ids=[",".join(f"{k}={v}" for k, v in e.items()) for e, _ in SWITCHES])
def test_launcher_switch_passes(env, kexpr):
    rc, tail = run_child(env, kexpr)
    print(tail)
    assert rc == 0 and " passed" in tail, f"{env}: child exit {rc}\n{tail}"
