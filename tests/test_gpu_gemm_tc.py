"""GPU tests (-m gpu) of the tcgen05 GEMM family (csrc/gemm_tc.cu: bsrnn_gemm_tc_ex, _grouped, _scaled) and the two operand
builders that feed it (bsrnn_norm_cast_kb8[_ones], bsrnn_kb8_transpose), each against a plain f64 restatement of what
include/bsrnn_b200.h promises.

Reference: an f64 matmul of the fp16 operands as stored, plus the bias, then the epilogue in f64.  The bar is ELEMENTWISE:
fp16 x fp16 products are exact in f32, and each of the <= K + a few f32 additions that follow (tensor-pipe accumulation,
bias, scale, residual, split-K atomics) is off by at most one f32 ulp (2^-23, covering truncation as well as rounding) of a
partial sum bounded by sum_k |a_k w_k| (+ |bias|, |residual|).  So

    |got - ref| <= 2^-23 * (K + extra adds) * (|A| |W|^T + |bias|) [* |scale| + |residual|]       (c = 1, not fitted)

plus the epilogue's own error: half an fp16 ulp for fp16 outputs, 2^-10.987 * |tanh| for tanh.approx.f32 (PTX ISA, maximum
relative error; tanh' <= 1 carries the GEMM error through unchanged) and, for the GLU gate, the same inside
sigmoid(x) = 0.5 tanh(x / 2) + 0.5.  Every case prints its worst err / bound.

Everything the kernel must NOT write -- rows of tokens outside the row map, columns n_valid .. ldo, neighbouring segments
of a row when the output pointer is offset, KB8 cores >= out_kcores, a guard tail after the buffer -- starts as a NaN bit
pattern and must come back bit-identical.  One case per epilogue also corrupts the kernel's real output (a zeroed core, two
swapped rows, one element 3x its bound off) and asserts that the checker rejects each, so the bar is not slack.

Each GEMM case runs on the default persistent grid and under bsrnn_gemm_tc_limit_ctas (3 CTAs, or n_tiles for the
weight-resident schedule) so that every CTA walks many tiles: both TMEM accumulators and their phase flips, the row-buffer
refill of epilogue 8, and the later steps of the tile iterator (reverse M, band innermost, grouped).  The BSRNN_GEMM_DEBUG
modes that break the result on purpose are read once per process: they run in child pytest processes of this file, and
each must fail.
"""
import math
import os
import subprocess
import sys

import pytest
import torch

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CHILD = "BSRNN_GEMM_TC_TEST_CHILD"          # set in the child processes: the subprocess tests themselves do not recurse
U23, U24 = 2.0 ** -23, 2.0 ** -24
TANH_ERR = 2.0 ** -10.987                   # tanh.approx.f32: maximum relative error (PTX ISA)
BIG = 1 << 40
GUARD = 4096                                # elements of guard tail after every output buffer
SENT32 = 0x7F8DEAD1                         # NaN bit patterns of the untouched regions
SENT16 = 0x7E5B


# ---------------------------------------------------------------------------------------------------- reference machinery
def _kb8_index(tiles, kcores, rpt, dev):
    t = torch.arange(tiles, device=dev).view(-1, 1, 1, 1)
    c = torch.arange(kcores, device=dev).view(1, -1, 1, 1)
    r = torch.arange(rpt, device=dev).view(1, 1, -1, 1)
    e = torch.arange(8, device=dev).view(1, 1, 1, -1)
    return t * rpt + r, 8 * c + e              # (matrix row, matrix column) of element [t][c][r][e]


def kb8_pack(x, rpt, kcores):
    """(rows, K) matrix -> KB8 tiles [tiles][kcores][rpt][8] of the same dtype, element [t][c][r][e] = x[t*rpt + r, 8c + e]
    (umma.cuh, bsrnn_b200.h), rows and columns zero padded."""
    rows, K = x.shape
    tiles = -(-rows // rpt)
    full = torch.zeros(tiles * rpt, kcores * 8, dtype=x.dtype, device=x.device)
    full[:rows, :K] = x
    ri, ci = _kb8_index(tiles, kcores, rpt, x.device)
    return full[ri, ci]


def kb8_unpack(p):
    """KB8 tiles [tiles][kcores][rpt][8] -> (tiles*rpt, kcores*8) matrix of the same dtype."""
    tiles, kcores, rpt, _ = p.shape
    out = torch.empty(tiles * rpt, kcores * 8, dtype=p.dtype, device=p.device)
    ri, ci = _kb8_index(tiles, kcores, rpt, p.device)
    out[ri, ci] = p
    return out


def row_tokens(m_tiles, rows, dev="cuda"):
    """Token of every GEMM row m_tile*128 + r (-1 = not mapped), restated from the header:
    m_tile = step*tiles_per_step + j ; seq = j*128 + r (valid iff seq < R) ;
    token = (seq / seq_inner)*seq_outer + (seq % seq_inner)*seq_inner_stride + step*step_stride."""
    tps, R, si, so, sis, ss = rows
    m = torch.arange(m_tiles, device=dev, dtype=torch.long).view(-1, 1)
    r = torch.arange(128, device=dev, dtype=torch.long).view(1, -1)
    step = m // tps
    seq = (m - step * tps) * 128 + r
    tok = (seq // si) * so + (seq % si) * sis + step * ss
    return torch.where(seq < R, tok, torch.full_like(tok, -1)).reshape(-1)


def gemm_ref(A, W, bias=None):
    """f64 A W^T (+ bias) of the fp16 operands and the magnitude |A| |W|^T (+ |bias|) the accumulation error scales with."""
    Ad, Wd = A.double(), W.double()
    acc, mag = Ad @ Wd.t(), Ad.abs() @ Wd.abs().t()
    if bias is not None:
        acc += bias.double()
        mag += bias.double().abs()
    return acc, mag


def half_ulp16(x):
    """half the fp16 spacing at magnitude x (f64 tensor), subnormals included."""
    e = torch.floor(torch.log2(x.abs().clamp(min=2.0 ** -14)))
    return torch.exp2(e - 11)


def worst_ratio(got, ref, bound):
    """max err / bound (inf where an error meets a zero bound, or a value is not finite)."""
    err = (got - ref).abs()
    ratio = torch.where(bound > 0, err / bound.clamp(min=1e-300), torch.where(err > 0, math.inf, 0.0))
    return float(torch.nan_to_num(ratio, nan=math.inf).max()) if ratio.numel() else 0.0


def assert_within(name, got, ref, bound):
    w = worst_ratio(got, ref, bound)
    print(f"{name}: worst err/bound = {w:.3g}")
    assert w <= 1.0, f"{name}: worst err/bound {w:.3g}"
    return w


def assert_checker_is_sharp(name, got, ref, bound):
    """Corrupt a correct result three ways; the elementwise check must reject each."""
    assert got.shape[0] >= 2
    bad = got.clone()
    bad[:128, :8] = 0.0                                                   # one 8-column core of one row tile zeroed
    assert worst_ratio(bad, ref, bound) > 1.0, f"{name}: a zeroed core passes"
    bad = got.clone()
    bad[[0, 1]] = bad[[1, 0]]                                             # rows 0 and 1 of the tile swapped
    assert worst_ratio(bad, ref, bound) > 1.0, f"{name}: swapped rows pass"
    bad = got.clone()
    k = int(bound.reshape(-1).argmax())
    bad.view(-1)[k] += 3.0 * bound.reshape(-1)[k]                          # one element 3x its bound off
    assert worst_ratio(bad, ref, bound) > 1.0, f"{name}: a 3x-bound error passes"


def sentinel(n, dtype):
    if dtype == torch.float32:
        return torch.full((n,), SENT32, dtype=torch.int32, device="cuda").view(torch.float32)
    return torch.full((n,), SENT16, dtype=torch.int16, device="cuda").view(torch.float16)


def bits(t):
    return t.view(torch.int32 if t.dtype == torch.float32 else torch.int16)


def assert_untouched(name, buf, snap, written):
    keep = torch.ones(buf.numel(), dtype=torch.bool, device=buf.device)
    keep[written.reshape(-1)] = False
    same = bits(buf)[keep] == snap[keep]
    if not bool(same.all()):
        first = int(torch.nonzero(keep).reshape(-1)[~same][0])
        raise AssertionError(f"{name}: {int((~same).sum())} elements outside the output contract were written "
                             f"(first at flat index {first} of {buf.numel()})")


def rand(g, *shape, scale=1.0):
    return torch.randn(*shape, device="cuda", generator=g, dtype=torch.float32) * scale


@pytest.fixture(scope="module")
def L():
    from urgent2026_challenge_track1_b200 import _lib
    _lib.require_device()
    return _lib


def num_sms():
    return torch.cuda.get_device_properties(0).multi_processor_count


@pytest.fixture(params=["all", "few"])
def ctas(request, L):
    """Sets the persistent-CTA bound of the case (0 = every SM, or a small count) and restores the previous bound."""
    prev = L.lib().bsrnn_gemm_tc_limit_ctas(0)
    L.lib().bsrnn_gemm_tc_limit_ctas(prev)

    def apply(few_limit):
        L.lib().bsrnn_gemm_tc_limit_ctas(few_limit if request.param == "few" else 0)
        return request.param
    try:
        yield apply
    finally:
        L.lib().bsrnn_gemm_tc_limit_ctas(prev)


def test_kb8_pack_matches_the_runtime_packer():
    from urgent2026_challenge_track1_b200.runtime_tc import to_kb8
    g = torch.Generator().manual_seed(1)
    w = torch.randn(300, 197, generator=g)
    mine = kb8_pack(w.half(), 128, 26)
    assert torch.equal(bits(mine), bits(to_kb8(w, 128, 26)))
    assert torch.equal(kb8_unpack(mine)[:300, :197], w.half())


def test_row_map_restatement():
    # time axis of (B, T, K) = (2, 3, 4): seq = b*K + k, token = (b*T + t)*K + k at step t
    tok = row_tokens(3, (1, 8, 4, 12, 1, 4), dev="cpu").view(3, 128)
    assert tok[1, :8].tolist() == [4, 5, 6, 7, 16, 17, 18, 19] and bool((tok[:, 8:] == -1).all())
    # band axis: seq = b*T + t, token = seq*K + k at step k
    tok = row_tokens(4, (1, 6, 1, 4, 0, 1), dev="cpu").view(4, 128)
    assert tok[2, :6].tolist() == [2, 6, 10, 14, 18, 22]


# ---------------------------------------------------------------------------------------------------- row epilogues
# rows: (tiles_per_step, R, seq_inner, seq_outer, seq_inner_stride, step_stride); n_tok: tokens of the output matrix (the row
# map leaves some of them out).  "res_nt": m_tiles = 2*(SMs / n_tiles) + 1, the weight-resident schedule.
def _band(B, T, Kt, steps):             # (B, T, Kt) tokens, bands [0, steps) mapped: seq = b*T + t, step = band
    R = B * T
    tiles = -(-R // 128)
    return dict(rows=(tiles, R, 1, Kt, 0, 1), m_tiles=steps * tiles, n_tok=B * T * Kt, tps=T * Kt)


def _time_rows(B, T, Kt, Kused):        # time axis over bands [0, Kused) of Kt: seq = b*Kused + k, step = frame
    R = B * Kused
    tiles = -(-R // 128)
    return dict(rows=(tiles, R, Kused, T * Kt, 1, Kt), m_tiles=T * tiles, n_tok=B * T * Kt, tps=T * Kt)


def _plain(M, m_tiles, stride=1, tps=100):   # plain rows: token = seq * stride
    return dict(rows=(m_tiles, M, BIG, 0, stride, 0), m_tiles=m_tiles, n_tok=M * stride, tps=tps)


def _wgrad(H, m_tiles):                 # weight-gradient GEMM: GEMM row 4u + g -> gradient row g*H + u
    return dict(rows=(1 << 30, 4 * H, 4, 1, H, 0), m_tiles=m_tiles, n_tok=4 * H, tps=1)


ROW_CASES = {
    # epilogue 0: LSTM input-projection rows (8H = 3136 in 14 tiles of 224; 8H = 6144 in 24 tiles of 256), ragged R, ldo > n_tiles*BN
    "f16rows_h392": dict(epi=0, n_tiles=14, BN=224, kcores=26, ldo=3136 + 8, **_plain(300, 3), selfcheck=True),
    "f16rows_h392_resident": dict(epi=0, n_tiles=14, BN=224, kcores=26, ldo=3136, res_nt=True, **_plain(0, 0)),
    "f16rows_h768": dict(epi=0, n_tiles=24, BN=256, kcores=48, ldo=6144, **_plain(200, 2)),
    "f16rows_k2": dict(epi=0, n_tiles=2, BN=64, kcores=2, ldo=136, **_plain(333, 3, stride=2)),
    # epilogues 1 / 8 (Linear + skip): band axis (tensor map, band innermost), plain rows with holes (one copy per row, two N
    # tiles of 192 = N 384), time axis with stats per (sample, band) (run-merged copies), n_valid % 8 == 0 single tile
    "resid_band": dict(n_tiles=1, BN=208, kcores=100, n_valid=196, ldo=200, stats=True, **_band(3, 50, 5, 4)),
    "resid_plain384": dict(n_tiles=2, BN=192, kcores=34, n_valid=384, ldo=392, stats=True, **_plain(300, 3, stride=2)),
    "resid_time": dict(n_tiles=1, BN=208, kcores=2, n_valid=196, ldo=196, stats=True, stats_inner=22, **_time_rows(9, 6, 22, 20)),
    "resid_plain192": dict(n_tiles=1, BN=192, kcores=26, n_valid=192, ldo=200, stats=True, **_plain(250, 2)),
    # epilogue 8 store-only (BandSplit): tensor-map and run-merged forms
    "store_band": dict(epi=8, flags=1, n_tiles=1, BN=208, kcores=6, n_valid=196, ldo=200, stats=True, **_band(2, 70, 3, 3)),
    "store_time": dict(epi=8, flags=1, n_tiles=1, BN=208, kcores=4, n_valid=196, ldo=196, stats=True, **_time_rows(7, 4, 20, 20)),
    # epilogue 3 (mask decoder Conv1d + GLU): odd band widths, output at 2*bin0 inside rows of 2F floats, reverse M walk
    "glu_w3": dict(epi=3, n_tiles=1, BN=16, kcores=100, n_valid=6, ldo=40, off=14, **_plain(600, 5), selfcheck=True),
    "glu_w13": dict(epi=3, n_tiles=1, BN=64, kcores=26, n_valid=26, ldo=40, off=6, **_plain(450, 4)),
    # epilogue 7 (GradDecoder Conv1d + Tanh): 3 subbands x 16 channels at column 32 of rows of 160, second N tile half valid
    "tanh32": dict(epi=7, n_tiles=2, BN=32, kcores=26, n_valid=48, ldo=160, off=32, **_plain(400, 4), selfcheck=True),
    # bsrnn_gemm_tc_scaled (epilogue 1, training backward): constant / device scale, split-K with a short last split
    "scaled_const": dict(api="scaled", scale=0.375, n_tiles=1, BN=208, kcores=26, n_valid=196, ldo=200, **_plain(300, 3)),
    "scaled_ptr_time": dict(api="scaled", scale_ptr=2.0 ** -5, n_tiles=1, BN=208, kcores=98, n_valid=196, ldo=196,
                            **_time_rows(5, 3, 34, 34)),
    "splitk3": dict(api="scaled", scale_ptr=0.25, ksplit=3, bias=False, n_tiles=1, BN=208, kcores=50, n_valid=200, ldo=200,
                    **_wgrad(40, 2), selfcheck=True),
    "splitk16": dict(api="scaled", scale_ptr=0.5, ksplit=16, bias=False, n_tiles=1, BN=64, kcores=194, n_valid=40, ldo=80, off=40,
                     **_wgrad(40, 2)),
    # config-5 dW GEMM: time axis at 4 x 96 000 samples @48 kHz -> T = 201 frames, K = 34 bands, ceil(4*34/128) = 2 sequence
    # tiles: 201*2*128 = 51 456 tokens as the K axis, ksplit 16 (training_tc: min(16, kc_tok // 256))
    "splitk_config5": dict(api="scaled", scale_ptr=2.0 ** -6, ksplit=16, bias=False, n_tiles=1, BN=208, kcores=201 * 2 * 16,
                           n_valid=200, ldo=200, **_wgrad(32, 1)),
}
for _name in ("resid_band", "resid_plain384", "resid_time", "resid_plain192"):
    ROW_CASES[_name.replace("resid", "epi1")] = dict(ROW_CASES[_name], epi=1, selfcheck=_name == "resid_band")
    ROW_CASES[_name.replace("resid", "epi8")] = dict(ROW_CASES.pop(_name), epi=8, selfcheck=_name == "resid_band")


def run_row_case(L, name, c, few):
    sms = num_sms()
    dev = "cuda"
    g = torch.Generator(device=dev).manual_seed(sum(map(ord, name)))
    epi, n_tiles, BN, kc = c.get("epi", 1), c["n_tiles"], c["BN"], c["kcores"]
    rows, m_tiles, n_tok = c["rows"], c["m_tiles"], c["n_tok"]
    if c.get("res_nt"):                 # weight-resident schedule: m_tiles >= 2 * (SMs / n_tiles)
        m_tiles = 2 * (sms // n_tiles) + 1
        R = m_tiles * 128 - 37
        rows, n_tok = (m_tiles, R, BIG, 0, 1, 0), R
    resident = bool(c.get("res_nt"))
    mode = few(n_tiles if resident else 3)
    ncols, Kd = n_tiles * BN, 8 * kc
    nv = c.get("n_valid", ncols)
    ldo, off, api = c["ldo"], c.get("off", 0), c.get("api", "ex")
    ksplit, flags = c.get("ksplit", 1), c.get("flags", 0)
    A = rand(g, m_tiles * 128, Kd, scale=0.5).half()
    W = rand(g, ncols, Kd, scale=Kd ** -0.5).half()
    bias = rand(g, ncols) if c.get("bias", True) else None
    A8, W8 = kb8_pack(A, 128, kc), kb8_pack(W, BN, kc)
    toks = row_tokens(m_tiles, rows)
    valid = toks >= 0
    tv = toks[valid]
    cols_out = ncols if epi == 0 else nv
    pos = off + tv[:, None] * ldo + torch.arange(cols_out, device=dev)[None, :]
    odt = torch.float16 if epi == 0 else torch.float32
    buf = sentinel(off + n_tok * ldo + GUARD, odt)
    if epi in (1, 8):
        buf[pos] = rand(g, *pos.shape)                                     # the residual stream
    old = buf[pos].double() if epi in (1, 8) else None
    snap = bits(buf).clone()
    stats = None
    if c.get("stats"):
        si = c.get("stats_inner", 1)
        n_stat = (n_tok // c["tps"] + 1) * si
        stats = torch.zeros(n_stat, 2, dtype=torch.float64, device=dev)
    st = L.stream_ptr()
    sc = c.get("scale", 0.0)
    sc_dev = torch.tensor([c["scale_ptr"]], dtype=torch.float32, device=dev) if "scale_ptr" in c else None
    if api == "ex":
        L.call("bsrnn_gemm_tc_ex", A8.data_ptr(), W8.data_ptr(), L.ptr(bias), buf.data_ptr() + off * buf.element_size(),
               L.ptr(stats), m_tiles, n_tiles, kc, BN, epi, ldo, nv, 0, c.get("tps", 1), *rows, c.get("stats_inner", 1), flags, st)
    else:
        L.call("bsrnn_gemm_tc_scaled", A8.data_ptr(), W8.data_ptr(), L.ptr(bias), buf.data_ptr() + off * 4, m_tiles, n_tiles, kc,
               BN, ldo, nv, sc, L.ptr(sc_dev), ksplit, *rows, st)
    torch.cuda.synchronize()
    tag = f"{name}[{mode}]"
    assert_untouched(tag, buf, snap, pos)
    acc, mag = gemm_ref(A, W, bias)
    acc, mag = acc[valid], mag[valid]
    got = buf[pos].double()
    if epi == 0:
        ref = acc
        gb = U23 * (Kd + 2) * mag
        bound = gb + half_ulp16(ref.abs() + gb)
    elif epi in (1, 8):
        s = c.get("scale_ptr", sc if sc != 0.0 else 1.0)
        base = torch.zeros_like(old) if flags & 1 else old
        ref = base + s * acc[:, :nv]
        bound = U23 * (Kd + ksplit + 3) * (abs(s) * mag[:, :nv] + base.abs())
    elif epi == 7:
        ref = torch.tanh(acc[:, :nv])
        bound = U23 * (Kd + 2) * mag[:, :nv] + (TANH_ERR + U24) * ref.abs()
    else:                               # GLU on (value, gate)-interleaved columns
        v, gt = acc[:, 0::2][:, :nv], acc[:, 1::2][:, :nv]
        ev, eg = (U23 * (Kd + 2) * mag[:, 0::2][:, :nv]), (U23 * (Kd + 2) * mag[:, 1::2][:, :nv])
        th = torch.tanh(0.5 * gt)
        sg = 0.5 * th + 0.5
        ref = v * sg
        e_sg = 0.5 * (TANH_ERR * th.abs() + 0.5 * eg) + U24
        bound = ev * sg + v.abs() * e_sg + ev * e_sg + U24 * ref.abs()
    assert_within(tag, got, ref, bound)
    if c.get("selfcheck") and mode == "all":
        assert_checker_is_sharp(tag, got, ref, bound)
    if stats is not None:
        si = c.get("stats_inner", 1)
        srow = (tv // c["tps"]) * si + (tv % si if si > 1 else 0)
        want = torch.zeros_like(stats)
        want[:, 0].index_add_(0, srow, ref.sum(1))
        want[:, 1].index_add_(0, srow, (ref * ref).sum(1))
        sb = torch.zeros_like(stats)
        sb[:, 0].index_add_(0, srow, (bound + U23 * (BN + 8) * ref.abs()).sum(1))
        sb[:, 1].index_add_(0, srow, (2 * ref.abs() * bound + bound * bound + U23 * (BN + 8) * ref * ref).sum(1))
        assert_within(tag + " stats", stats, want, sb)
        if c.get("selfcheck") and mode == "all":
            bad = stats.clone()
            bad[int(srow[0])] += 3.0 * sb[int(srow[0])]
            assert worst_ratio(bad, want, sb) > 1.0, f"{tag}: statistics 3x their bound off pass"


@pytest.mark.parametrize("name", sorted(ROW_CASES))
def test_row_epilogue(L, ctas, name):
    run_row_case(L, name, ROW_CASES[name], ctas)


# ---------------------------------------------------------------------------------------------------- KB8 epilogues 2 / 4
KB8_CASES = {
    # epilogue 4, generic (bias in the epilogue); two spare k-cores per row tile that nobody writes
    "f16kb8_generic": dict(epi=4, n_tiles=3, BN=64, kcores=26, out_kcores=26, m_tiles=5, selfcheck=True),
    "f16kb8_generic_k100": dict(epi=4, n_tiles=2, BN=128, kcores=100, out_kcores=34, m_tiles=3),
    # epilogue 4, the specialised input-projection kernel: 16 N tiles of 208, kc 26, bias through the constant-one column 196
    "f16kb8_special": dict(epi=4, n_tiles=16, BN=208, kcores=26, out_kcores=418, one_col=196, res_nt=True),
    # epilogue 2, generic: n_valid = 100, out_kcores = 14 (columns 100..111 must be zeros, 112..127 are clipped); the bias of the
    # padding columns is NOT zero, so the zeros must come from the epilogue
    "tanhkb8_generic": dict(epi=2, n_tiles=2, BN=64, kcores=26, n_valid=100, out_kcores=14, m_tiles=4, selfcheck=True),
    # epilogue 2, the specialised bulk-store kernel: Conv1d(N -> 4N = 784) in 4 N tiles of 208, bias through the ones column,
    # destination of 100 k-cores (the K = 800 operand of the GLU GEMM)
    "tanhkb8_special": dict(epi=2, n_tiles=4, BN=208, kcores=26, n_valid=784, out_kcores=100, one_col=196, res_nt=True),
}


def run_kb8_case(L, name, c, few):
    sms = num_sms()
    dev = "cuda"
    g = torch.Generator(device=dev).manual_seed(sum(map(ord, name)))
    epi, n_tiles, BN, kc, okc = c["epi"], c["n_tiles"], c["BN"], c["kcores"], c["out_kcores"]
    resident = bool(c.get("res_nt"))
    m_tiles = 2 * (sms // n_tiles) + 1 if resident else c["m_tiles"]
    mode = few(n_tiles if resident else 3)
    ncols, Kd = n_tiles * BN, 8 * kc
    nv = c.get("n_valid", ncols)
    oc = c.get("one_col", -1)
    A = rand(g, m_tiles * 128, Kd, scale=0.5)
    W = rand(g, ncols, Kd, scale=Kd ** -0.5)
    bias = rand(g, ncols)
    if oc >= 0:                         # bias as weight column `oc` against the operand's constant-one column (no epilogue bias)
        A[:, oc] = 1.0
        A[:, oc + 1:] = 0.0
        W[:, oc] = bias
        W[:, oc + 1:] = 0.0
        if epi == 2:
            W[nv:] = 0.0                # the padding channels of the hidden operand come from zero weight rows
        bias = None
    A, W = A.half(), W.half()
    A8, W8 = kb8_pack(A, 128, kc), kb8_pack(W, BN, kc)
    buf = sentinel(m_tiles * okc * 1024 + GUARD, torch.float16)
    snap = bits(buf).clone()
    L.call("bsrnn_gemm_tc_ex", A8.data_ptr(), W8.data_ptr(), L.ptr(bias), buf.data_ptr(), None, m_tiles, n_tiles, kc, BN, epi,
           0, nv, okc, 1, m_tiles, m_tiles * 128, BIG, 0, 1, 0, 1, 0, L.stream_ptr())
    torch.cuda.synchronize()
    tag = f"{name}[{mode}]"
    cols = torch.arange(min(ncols, 8 * okc), device=dev)
    if epi == 4 and resident and BN == 208:
        # the specialised input-projection kernel does not store core 25 of an N tile (gate columns 200..207: the padding of a
        # 49-unit slice, never read by the recurrence): those columns are neither checked nor required untouched
        skip = cols[(cols % 208) >= 200]
        cols = cols[(cols % 208) < 200]
    else:
        skip = cols[:0]
    rows = torch.arange(m_tiles * 128, device=dev)
    pos_of = lambda cc: (((rows[:, None] // 128) * okc + cc[None, :] // 8) * 128 + rows[:, None] % 128) * 8 + cc[None, :] % 8
    pos = pos_of(cols)
    assert_untouched(tag, buf, snap, torch.cat([pos.reshape(-1), pos_of(skip).reshape(-1)]))
    acc, mag = gemm_ref(A, W, bias)
    got = buf[pos].double()
    gb = U23 * (Kd + 2) * mag
    if epi == 4:
        ref = acc[:, cols]
        bound = gb[:, cols] + half_ulp16(ref.abs() + gb[:, cols])
    else:
        pad = got[:, nv:]
        assert bool((pad == 0).all()), f"{tag}: padding columns {nv}..{8 * okc} of the hidden operand are not zero"
        got = got[:, :nv]
        ref = torch.tanh(acc[:, :nv])
        e = gb[:, :nv] + (TANH_ERR + U24) * ref.abs()
        bound = e + half_ulp16(ref.abs() + e)
    assert_within(tag, got, ref, bound)
    if c.get("selfcheck") and mode == "all":
        assert_checker_is_sharp(tag, got, ref, bound)


@pytest.mark.parametrize("name", sorted(KB8_CASES))
def test_kb8_epilogue(L, ctas, name):
    run_kb8_case(L, name, KB8_CASES[name], ctas)


# ---------------------------------------------------------------------------------------------------- grouped (BandSplit)
def test_grouped_bandsplit(L, ctas):
    """bsrnn_gemm_tc_grouped: 4 bands with kcores 2, 6, 4, 6 (kc_max = 6), per-band operand / weight / bias / output offsets,
    per-sample statistics over all bands, rows of K*N + 8 floats (the last 8 untouched)."""
    dev = "cuda"
    g = torch.Generator(device=dev).manual_seed(7)
    kcs, N, BN, B, T = [2, 6, 4, 6], 196, 208, 3, 100
    K = len(kcs)
    R = B * T
    tiles = -(-R // 128)
    ldo = K * N + 8
    mode = ctas(3)
    A = [rand(g, tiles * 128, 8 * k, scale=0.5).half() for k in kcs]
    W = [rand(g, BN, 8 * k, scale=(8 * k) ** -0.5).half() for k in kcs]
    bias = rand(g, K * BN)
    A8 = torch.cat([kb8_pack(a, 128, k).reshape(-1) for a, k in zip(A, kcs)])
    W8 = torch.cat([kb8_pack(w, BN, k).reshape(-1) for w, k in zip(W, kcs)])
    a_off = [sum(tiles * k * 1024 for k in kcs[:i]) for i in range(K)]
    w_off = [sum(BN * k * 8 for k in kcs[:i]) for i in range(K)]
    groups = torch.tensor([[a_off[i], w_off[i], i * N, i * BN, kcs[i]] for i in range(K)], dtype=torch.int64, device=dev)
    buf = sentinel(R * ldo + GUARD, torch.float32)
    tok = torch.arange(R, device=dev)
    pos = tok[:, None] * ldo + torch.arange(K * N, device=dev)[None, :]
    buf[pos] = rand(g, *pos.shape)          # store-only: whatever was there is replaced
    snap = bits(buf).clone()
    stats = torch.zeros(B + 1, 2, dtype=torch.float64, device=dev)
    L.call("bsrnn_gemm_tc_grouped", A8.data_ptr(), W8.data_ptr(), bias.data_ptr(), buf.data_ptr(), stats.data_ptr(),
           groups.data_ptr(), K, tiles, max(kcs), BN, ldo, N, T, tiles, R, BIG, 0, 1, 0, L.stream_ptr())
    torch.cuda.synchronize()
    tag = f"grouped[{mode}]"
    assert_untouched(tag, buf, snap, pos)
    refs, bounds = [], []
    for i in range(K):
        acc, mag = gemm_ref(A[i], W[i], bias[i * BN:(i + 1) * BN])
        refs.append(acc[:R, :N])
        bounds.append(U23 * (8 * kcs[i] + 3) * mag[:R, :N])
    ref, bound = torch.cat(refs, 1), torch.cat(bounds, 1)
    got = buf[pos].double()
    assert_within(tag, got, ref, bound)
    srow = tok // T
    want, sb = torch.zeros_like(stats), torch.zeros_like(stats)
    want[:, 0].index_add_(0, srow, ref.sum(1))
    want[:, 1].index_add_(0, srow, (ref * ref).sum(1))
    sb[:, 0].index_add_(0, srow, (bound + U23 * (BN + 8) * ref.abs()).sum(1))
    sb[:, 1].index_add_(0, srow, (2 * ref.abs() * bound + bound * bound + U23 * (BN + 8) * ref * ref).sum(1))
    assert_within(tag + " stats", stats, want, sb)
    if mode == "all":
        assert_checker_is_sharp(tag, got, ref, bound)


# ---------------------------------------------------------------------------------------------------- operand builders
NORM_CASES = {
    # time axis (B, T, K) = (3, 4, 34), dense rows (run-merged copies), per-sample scale, constant-one column 196
    "time_ones": dict(C=196, col0=0, ldx=196, kcores=26, one_col=196, g_inner=1, scale=True, **_time_rows(3, 4, 34, 34)),
    # band axis (tensor-map copies), per-(sample, band) scale: g_inner = K
    "band_ginner": dict(C=196, col0=0, ldx=196, kcores=26, one_col=-1, g_inner=5, scale=True, **_band(2, 70, 5, 5)),
    # rows of 204 floats from column 4 (one bulk copy per row), no affine
    "plain_col0": dict(C=196, col0=4, ldx=204, kcores=26, one_col=200, g_inner=1, scale=False, **_plain(300, 3)),
    # C % 4 != 0: the scalar path, g_inner = 3
    "scalar_c30": dict(C=30, col0=2, ldx=37, kcores=4, one_col=-1, g_inner=3, scale=True, **_plain(200, 2, tps=50)),
}


@pytest.mark.parametrize("name", sorted(NORM_CASES))
def test_norm_cast_kb8(L, name):
    c = NORM_CASES[name]
    dev = "cuda"
    g = torch.Generator(device=dev).manual_seed(sum(map(ord, name)))
    m_tiles, rows, n_tok, tps = c["m_tiles"], c["rows"], c["n_tok"], c["tps"]
    C, col0, ldx, kc, oc, gi = c["C"], c["col0"], c["ldx"], c["kcores"], c["one_col"], c["g_inner"]
    x = rand(g, n_tok * ldx + 8, scale=2.0)
    n_grp = (n_tok // tps + 1) * gi
    scale = rand(g, n_grp, C) if c["scale"] else None
    shift = rand(g, n_grp, C) if c["scale"] else None
    buf = sentinel(m_tiles * kc * 1024 + GUARD, torch.float16)
    snap = bits(buf).clone()
    L.call("bsrnn_norm_cast_kb8_ones", x.data_ptr(), L.ptr(scale), L.ptr(shift), buf.data_ptr(), ldx, col0, C, kc, m_tiles,
           *rows, tps, gi, oc, L.stream_ptr())
    torch.cuda.synchronize()
    n_out = m_tiles * kc * 1024
    assert torch.equal(bits(buf)[n_out:], snap[n_out:]), f"{name}: guard tail written"
    got = kb8_unpack(buf[:n_out].view(m_tiles, kc, 128, 8)).double()        # (m_tiles*128, kc*8)
    toks = row_tokens(m_tiles, rows)
    valid = toks >= 0
    tv = toks[valid]
    xv = x.double()[tv[:, None] * ldx + col0 + torch.arange(C, device=dev)[None, :]]
    if scale is not None:
        grp = (tv // tps) * gi + (tv % gi if gi > 1 else 0)
        ref = xv * scale.double()[grp] + shift.double()[grp]
        mag = (xv * scale.double()[grp]).abs() + shift.double()[grp].abs()
    else:
        ref, mag = xv, xv.abs()
    bound = U24 * mag + half_ulp16(ref.abs() * (1 + U23) + U24 * mag)
    assert_within(f"norm_cast {name}", got[valid][:, :C], ref, bound)
    pad = got[:, C:].clone()
    if oc >= 0:
        assert bool((pad[:, oc - C] == 1.0).all()), f"{name}: constant-one column is not 1"
        pad[:, oc - C] = 0.0
    assert bool((pad == 0).all()), f"{name}: padding columns are not 0"
    assert bool((got[~valid][:, :C] == 0).all()), f"{name}: rows outside the row map are not 0"


@pytest.mark.parametrize("src_tiles,kc_src,BN,n_tiles,src_m0,m_count,dst_kcores,dst_kc0", [
    (5, 26, 128, 2, 1, 3, 3 * 16 + 20, 8),          # columns 208..255 read as zero; k-cores 0..7 and 56..67 untouched
    (2, 6, 64, 1, 0, 2, 40, 0),                     # k-cores 32..39 untouched
    (3, 100, 256, 4, 2, 1, 16, 0),                  # wide source, the last of its tiles only
])
def test_kb8_transpose_bit_exact(L, src_tiles, kc_src, BN, n_tiles, src_m0, m_count, dst_kcores, dst_kc0):
    dev = "cuda"
    g = torch.Generator(device=dev).manual_seed(kc_src + BN)
    src = rand(g, src_tiles * 128, kc_src * 8).half()
    src8 = kb8_pack(src, 128, kc_src)
    dst = sentinel(n_tiles * dst_kcores * BN * 8 + GUARD, torch.float16)
    snap = bits(dst).clone()
    L.call("bsrnn_kb8_transpose", src8.data_ptr(), dst.data_ptr(), src_m0, m_count, kc_src, BN, n_tiles, dst_kcores, dst_kc0,
           L.stream_ptr())
    torch.cuda.synchronize()
    # documented map: dst row n*BN + c = source column, dst k index = dst_kc0*8 + (m - src_m0)*128 + r; columns >= kc_src*8 = 0
    n_dst = n_tiles * dst_kcores * BN * 8
    want = kb8_unpack(snap[:n_dst].view(n_tiles, dst_kcores, BN, 8))                 # (n_tiles*BN, dst_kcores*8) of bits
    srcb = torch.zeros(src_tiles * 128, max(kc_src * 8, n_tiles * BN), dtype=torch.int16, device=dev)
    srcb[:, :kc_src * 8] = bits(src)
    for m in range(m_count):
        k0 = dst_kc0 * 8 + m * 128
        want[:, k0:k0 + 128] = srcb[(src_m0 + m) * 128:(src_m0 + m + 1) * 128, :n_tiles * BN].t()
    want = kb8_pack(want, BN, dst_kcores).reshape(-1)
    assert torch.equal(bits(dst)[:n_dst], want)
    assert torch.equal(bits(dst)[n_dst:], snap[n_dst:])


# ---------------------------------------------------------------------------------------------------- child processes
def run_child(env_var, value, kexpr):
    env = dict(os.environ, **{env_var: value, CHILD: "1", "COLUMNS": "250"})      # untruncated summary lines
    cmd = [sys.executable, "-m", "pytest", os.path.abspath(__file__), "-m", "gpu", "-q", "-x", "-p", "no:cacheprovider",
           "-k", kexpr]
    r = subprocess.run(cmd, cwd=ROOT, env=env, capture_output=True, text=True, timeout=900)
    tail = "\n".join((r.stdout + r.stderr).splitlines()[-25:])
    return r.returncode, tail


child_only = pytest.mark.skipif(os.environ.get(CHILD) == "1", reason="runs in the parent process only")


# BSRNN_GEMM_DEBUG modes that break the result on purpose (all stay in bounds) -> a case that must catch it
DEBUG_MODES = [
    ("1", "f16kb8_special and all"),                # every tile of the specialised kernels stores into tile 0's block
    ("2", "tanhkb8_special and all"),               # no stores
    ("4", "epi1_plain192 and all"),                 # epilogue 1: no residual traffic at all
    ("8", "epi1_plain192 and all"),                 # epilogue 1: residual stored but not read
    ("16", "epi1_plain192 and all"),                # epilogue 1: no statistics
]


@child_only
@pytest.mark.parametrize("value,kexpr", DEBUG_MODES, ids=[f"BSRNN_GEMM_DEBUG={v}" for v, _ in DEBUG_MODES])
def test_debug_mode_is_caught(value, kexpr):
    rc, tail = run_child("BSRNN_GEMM_DEBUG", value, kexpr)
    print(tail)
    case = kexpr.split()[0]
    caught = any(line.startswith("FAILED") and case in line and "AssertionError" in line for line in tail.splitlines())
    assert rc == 1 and caught, f"BSRNN_GEMM_DEBUG={value}: child exit {rc}\n{tail}"
