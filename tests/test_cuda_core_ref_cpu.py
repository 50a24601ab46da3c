"""CPU checks of tests/cuda_core_ref.py: each f64 reference against an independent implementation (torch.addmm / F.glu /
tanh, nn.LSTM and autograd, the oracle's BandSplit / GroupNorm / GaussianFourierProjection / prior / Euler sampler, an
unfolded convolution), each bound small against its reference, and the restated launcher geometry against hand-worked
values."""
import math

import pytest
import torch
import torch.nn.functional as F

import cuda_core_ref as R
from oracle import restated as O


def _close(a, b, tol=1e-12):
    a, b = a.double(), b.double()
    scale = max(1.0, float(b.abs().max()))
    assert float((a - b).abs().max()) <= tol * scale, float((a - b).abs().max())


def _relbound(ref, bound, lim):
    """Bounds stay a small multiple of u of the result scale (so the GPU checks have teeth)."""
    assert bool((bound >= 0).all())
    assert float(bound.max()) <= lim * max(1.0, float(ref.abs().max()))


# ------------------------------------------------------------------------------------------------------------ gemm_f32
@pytest.mark.parametrize("epi", [0, 1, 2, 3])
@pytest.mark.parametrize("scaled", [False, True])
def test_gemm_ref_matches_torch(epi, scaled):
    g = torch.Generator().manual_seed(epi + 4 * scaled)
    M, N, K, kv = 37, 66, 29, 23
    A = torch.randn(M, K, generator=g)
    W = torch.randn(N, K, generator=g) / 5
    b = torch.randn(N, generator=g)
    sc = torch.rand(M, K, generator=g) + 0.5 if scaled else None
    sh = torch.randn(M, K, generator=g) if scaled else None
    C0 = torch.randn(M, N, generator=g)
    ref, bound = R.gemm_f32_ref(A, W, b, sc, sh, kv, epi, C0)
    Ad = A.double().clone()
    Ad[:, kv:] = 0
    if scaled:
        Ad = Ad * sc.double() + sh.double()
    v = torch.addmm(b.double(), Ad, W.double().t())
    want = {0: v, 1: torch.tanh(v), 2: v + C0.double(), 3: F.glu(v, dim=1)}[epi]
    _close(ref, want)
    assert ref.shape == want.shape and bound.shape == want.shape
    _relbound(ref, bound, 1e-4)


def test_gemm_geometry_hand_worked():
    assert R.gemm_grid(1000, 784, 3) == (25, 16, 3)
    assert R.gemm_group_tiles(1000, 784, 0) == (13, 16)           # 64-column tiles
    assert R.gemm_group_tiles(65, 240, 3) == (4, 2)               # GLU: 120 logical columns in 32-column tiles
    # mask decoder: max_n = 2 * max(s) = 120 for N = 4 s = 240 -> 4 column tiles, exactly covered
    assert R.gemm_grid(10, 120, 1)[0] == 4
    b = R.gemm_branches(65, 240, 17, 15, 3, 100, True, 1000, 240)
    assert {"epilogue3", "scaled", "early_exit", "partial_row_tile", "partial_k_tile", "k_valid", "n_store",
            "glu_partial_w"} <= b
    with pytest.raises(AssertionError):
        R.gemm_branches(1000, 784, 16, 16, 0, 784, False, 1000, 384)   # 12 < 13 column tiles


# ------------------------------------------------------------------------------------------------------------ BLSTM
def _token_major_sequences(B, T, K, axis):
    """(R, S) tokens of a (B, T, K) token-major tensor along an axis, built with permutes (independent of seq_tokens)."""
    tok = torch.arange(B * T * K).view(B, T, K)
    if axis == "time":
        return tok.permute(0, 2, 1).reshape(B * K, T)
    return tok.reshape(B * T, K)


@pytest.mark.parametrize("axis", ["time", "band"])
def test_seq_tokens_match_both_axes(axis):
    B, T, K = 2, 5, 3
    want = _token_major_sequences(B, T, K, axis)
    addr = (K, T * K, 1, K) if axis == "time" else (1, K, 0, 1)
    R_, S = want.shape
    assert torch.equal(R.seq_tokens(R_, S, *addr), want)


def _lstm_setup(seed, B, T, K, N, H, axis):
    g = torch.Generator().manual_seed(seed)
    rnn = torch.nn.LSTM(N, H, batch_first=True, bidirectional=True).double()
    with torch.no_grad():
        for p in rnn.parameters():
            p.copy_(torch.randn(p.shape, generator=g, dtype=torch.float64) * 0.4)
    x = torch.randn(B, T, K, N, generator=g, dtype=torch.float64)
    seq = _token_major_sequences(B, T, K, axis)
    xs = x.reshape(-1, N)[seq]                                               # (R, S, N)
    gx = torch.stack([xs @ rnn.weight_ih_l0.t() + rnn.bias_ih_l0 + rnn.bias_hh_l0,
                      xs @ rnn.weight_ih_l0_reverse.t() + rnn.bias_ih_l0_reverse + rnn.bias_hh_l0_reverse])
    whh = torch.stack([rnn.weight_hh_l0, rnn.weight_hh_l0_reverse]).detach()
    return rnn, xs, gx.detach(), whh


@pytest.mark.parametrize("axis", ["time", "band"])
def test_lstm_forward_ref_matches_nn_lstm(axis):
    rnn, xs, gx, whh = _lstm_setup(1, 2, 6, 3, 5, 7, axis)
    with torch.no_grad():
        want = rnn(xs)[0]
    _close(R.lstm_forward_ref(gx, whh), want)


def test_lstm_step_bound_small():
    g = torch.Generator().manual_seed(2)
    gx, whh = torch.randn(9, 32, generator=g), torch.randn(32, 8, generator=g) / 3
    st = R.lstm_step_ref(gx, whh, torch.randn(9, 8, generator=g).tanh(), torch.randn(9, 8, generator=g))
    for k, (v, b) in st.items():
        _relbound(v, b, 1e-5)


def _unidirectional_autograd(gx, whh, dy):
    """dL/d gates_x of one direction via nn.LSTM with an identity input weight (gates_x is the input)."""
    H = whh.shape[1]
    lstm = torch.nn.LSTM(4 * H, H, batch_first=True).double()
    with torch.no_grad():
        lstm.weight_ih_l0.copy_(torch.eye(4 * H, dtype=torch.float64))
        lstm.weight_hh_l0.copy_(whh)
        lstm.bias_ih_l0.zero_()
        lstm.bias_hh_l0.zero_()
    inp = gx.clone().requires_grad_(True)
    y = lstm(inp)[0]
    (y * dy).sum().backward()
    return inp.grad


@pytest.mark.parametrize("axis", ["time", "band"])
def test_lstm_bptt_ref_matches_autograd(axis):
    _, _, gx, whh = _lstm_setup(3, 2, 5, 4, 3, 6, axis)
    Rn, S, _ = gx.shape[1:]
    H = whh.shape[2]
    g = torch.Generator().manual_seed(4)
    dy = torch.randn(2, Rn, S, H, generator=g, dtype=torch.float64)
    # saved (i, f, g, o, c) from the f64 forward
    saved = torch.zeros(2, Rn, S, 5, H, dtype=torch.float64)
    for d in range(2):
        h = c = None
        for q in range(S):
            s = q if d == 0 else S - 1 - q
            st = R.lstm_step_ref(gx[d, :, s], whh[d], h, c)
            saved[d, :, s] = torch.stack([st[k][0] for k in "ifgoc"], 1)
            h, c = st["h"][0], st["c"][0]
    got, bound = R.lstm_bwd_ref(saved, dy, whh)
    want0 = _unidirectional_autograd(gx[0], whh[0], dy[0])
    want1 = _unidirectional_autograd(gx[1].flip(1), whh[1], dy[1].flip(1)).flip(1)
    _close(got[0], want0)
    _close(got[1], want1)
    _relbound(got, bound, 1e-4)
    # the running bound grows against the processing order of each direction
    assert float(bound[0, :, 0].sum()) > float(bound[0, :, -1].sum())
    assert float(bound[1, :, -1].sum()) > float(bound[1, :, 0].sum())


def test_lstm_grids_hand_worked():
    f, g1, g2 = R.lstm_grids(70000, 392)
    assert f == (25, 1094, 2) and g1 == (2, 65535, 2) and g2 == (7, 1094, 2)


# ------------------------------------------------------------------------------------------------------------ BandSplit / GN
def _band_tables(subbands, F):
    plan_bin0, plan_w, lo = [], [], 0
    for s in subbands:
        plan_bin0.append(lo)
        plan_w.append(min(s, F - lo))
        lo += s
        if lo >= F:
            break
    K = len(plan_bin0)
    c_off = [0]
    for s in subbands[:K]:
        c_off.append(c_off[-1] + 2 * s)
    return K, plan_bin0, [2 * w for w in plan_w], c_off


@pytest.mark.parametrize("F_bins", [161, 221, 481])              # 16 k (truncated last band), 22.05 k, 48 k
def test_band_split_and_gn_match_oracle(F_bins):
    subbands = O.SUBBANDS_481
    g = torch.Generator().manual_seed(F_bins)
    B, T, N = 2, 7, 12
    K, bin0, width2, c_off = _band_tables(subbands, F_bins)
    cmax = 2 * max(subbands)
    spec = torch.randn(B, T, F_bins, 2, generator=g) * 3 + 0.5
    sd, prefix = {}, "bs."
    gamma = torch.zeros(K, cmax)
    beta = torch.zeros(K, cmax)
    wT = []
    for k in range(K):
        s = subbands[k]
        sd[f"bs.norm.{k}.weight"] = torch.rand(2 * s, generator=g) + 0.5
        sd[f"bs.norm.{k}.bias"] = torch.randn(2 * s, generator=g)
        sd[f"bs.fc.{k}.weight"] = torch.randn(N, 2 * s, 1, generator=g) / 4
        sd[f"bs.fc.{k}.bias"] = torch.randn(N, generator=g)
        gamma[k, :2 * s], beta[k, :2 * s] = sd[f"bs.norm.{k}.weight"], sd[f"bs.norm.{k}.bias"]
        wT.append(sd[f"bs.fc.{k}.weight"][:, :, 0].t())
    wT = torch.cat(wT).contiguous()
    bias = torch.stack([sd[f"bs.fc.{k}.bias"] for k in range(K)])
    rows = spec.reshape(B * T, 2 * F_bins)
    # statistics (the real bins; the padded ones enter only through the count) -> finalize -> BandSplit
    stats = torch.zeros(B * K, 2, dtype=torch.float64)
    geo = R.band_stats_geometry(B, T, K, max(width2))
    for k in range(K):
        xb = rows[:, 2 * bin0[k]: 2 * bin0[k] + width2[k]].reshape(B, -1)
        s_, q_, bs_, bq_ = R.sums_ref(xb, geo["m"])
        stats[k::K, 0], stats[k::K, 1] = s_, q_
        _relbound(s_, bs_, 1e-4)
    counts = torch.tensor([2.0 * subbands[k] * T for k in range(K)], dtype=torch.float64)
    (sc, dsc), (sh, dsh) = R.gn_finalize_ref(stats, gamma, beta, None, counts, O.EPS_NORM1D, K)
    _relbound(sc, dsc, 1e-5)
    got = R.band_split_ref(rows, T, sc.float(), sh.float(), wT, bias, c_off, bin0, width2, cmax, N)
    want = O.band_split(sd, prefix, spec, subbands)                        # (B, T, K, N)
    for k, (ref, bound) in enumerate(got):
        _close(ref.view(B, T, N), want[:, :, k], 1e-5)                     # scale / shift rounded to f32 on the way
        _relbound(ref, bound, 1e-4)


def test_gn_finalize_matches_group_norm_and_clamps():
    g = torch.Generator().manual_seed(5)
    B, C, n = 3, 10, 40
    x = torch.randn(B, C, n, generator=g, dtype=torch.float64) * 2 + 1000.0             # DC offset
    gamma, beta, extra = torch.randn(1, C, generator=g), torch.randn(1, C, generator=g), torch.randn(B, C, generator=g)
    stats = torch.stack([x.sum((1, 2)), (x * x).sum((1, 2))], 1)
    (sc, _), (sh, _) = R.gn_finalize_ref(stats, gamma, beta, extra, torch.tensor([float(C * n)]), 1e-5, 1)
    want = O._gn(x, gamma[0].double(), beta[0].double(), 1e-5) + extra.double()[:, :, None]
    _close(sc[:, :, None] * x + sh[:, :, None], want, 1e-8)
    # variance below zero is clamped: rstd = 1 / sqrt(eps)
    st = torch.tensor([[4.0, 0.0]], dtype=torch.float64)
    (sc, _), (sh, _) = R.gn_finalize_ref(st, torch.ones(1, 2), torch.zeros(1, 2), None, torch.tensor([2.0]), 0.25, 1)
    assert torch.allclose(sc, torch.full((1, 2), 2.0, dtype=torch.float64)) and torch.allclose(sh, torch.full((1, 2), -4.0, dtype=torch.float64))


def test_stats_geometry_hand_worked():
    # contiguous: B = 1 -> 1184 chunks; 100 rows -> 1 row per block, 100 blocks; 196 floats per block -> 1 term per partial
    assert R.gn_stats_geometry(1, 100, 196, 196) == dict(chunks=1184, rpb=1, blocks=100, contiguous=True, m=1)
    # B = 3: 395 chunks; 4000 rows -> 11 rows per block (364 blocks), 11 * 196 / 256 -> 9 terms
    assert R.gn_stats_geometry(3, 4000, 196, 196) == dict(chunks=395, rpb=11, blocks=364, contiguous=True, m=9)
    # flushed at 64: B = 1200 -> 1 chunk, 500 rows x 196 = 98000 floats -> 383 per thread, flushed every 64
    assert R.gn_stats_geometry(1200, 500, 196, 196)["m"] == 64
    # strided: C = 300 > 256 -> 2 terms per row, 11 rows per block
    assert R.gn_stats_geometry(3, 4000, 300, 320) == dict(chunks=395, rpb=11, blocks=364, contiguous=False, m=22)
    # band_stats: B K > 1184 -> tchunks = 1 (one block per (b, k) walks all T)
    assert R.band_stats_geometry(40, 100, 30, 196) == dict(tchunks=1, tpb=100, zblocks=1, m=64)
    assert R.band_stats_geometry(2, 100, 30, 8) == dict(tchunks=20, tpb=5, zblocks=20, m=1)
    assert R.band_stats_geometry(2, 1, 30, 8)["tchunks"] == 1


def test_band_split_runs_hand_worked():
    N = 196
    # SE table: 2 s = 10, 8 x 19, 20 x 6, 80 x 7, 120 -> padded 12 / 8 / 20 / 80 / 120 channels x (N + 128) floats; 20 -> 80
    # is more than 2x, 80 -> 120 is not: two runs
    K, _, _, c_off = _band_tables(O.SUBBANDS_481, 481)
    runs = R.band_split_runs(c_off, N)
    assert [(a, b) for a, b, _ in runs] == [(0, 26), (26, 34)]
    assert runs[0][2] == 20 * (N + 128) * 4 and runs[-1][2] == 120 * (N + 128) * 4
    assert [(a, b) for a, b, _ in R.band_split_runs([0, 8, 40, 48, 52, 212], N)] == [(0, 1), (1, 2), (2, 4), (4, 5)]
    # 2 s = 112 at N = 384 comes within 3 KB of the limit and still fits; 116 does not
    assert R.band_split_smem(112, 384) == 229376 <= R.SMEM_LIMIT < R.band_split_smem(116, 384)
    assert R.kb8_geometry(10, 300) == (2, 3, 6144) and R.kb8_geometry(120, 128) == (16, 1, 16384)


# ------------------------------------------------------------------------------------------------------------ flow
def test_conv5x5_glu_ref_matches_unfolded_conv():
    g = torch.Generator().manual_seed(6)
    B, T, Fp, F_out = 2, 9, 11, 14
    x = torch.randn(B, T, Fp, 16, generator=g)
    w, b = torch.randn(4, 16, 5, 5, generator=g) / 8, torch.randn(4, generator=g)
    ref, bound = R.conv5x5_glu_ref(x, w, b, F_out)
    img = x.double().permute(0, 3, 2, 1)                                     # (B, 16, F', T)
    cols = F.unfold(img, 5, padding=2)                                       # (B, 400, F' T) in (ci, df, dt) order
    acc = (w.double().reshape(4, 400) @ cols).view(B, 4, Fp, T) + b.double()[:, None, None]
    want = F.glu(acc, dim=1).permute(0, 3, 2, 1)                              # (B, T, F', 2)
    _close(ref[:, :, :Fp], want)
    assert bool((ref[:, :, Fp:] == 0).all()) and bool((bound[:, :, Fp:] == 0).all())
    _relbound(ref, bound, 1e-3)                                              # gamma_400 of |v| |w| sums ~ 40 |out|
    assert R.conv_grid(3, 100, 33, 31) == (2, 13, 3)


def test_time_embed_ref_matches_oracle():
    g = torch.Generator().manual_seed(7)
    t, W = torch.rand(5, generator=g), torch.randn(64, generator=g) * 16
    ref, bound = R.time_embed_ref(t, W)
    want = O.gaussian_fourier(W.double(), t.double())
    # the f32 phase differs from the f64 one by three roundings of |phase|
    p = (t.double()[:, None] * W.double()[None, :] * 2 * math.pi).abs()
    assert bool(((ref - want).abs() <= torch.cat([p, p], 1) * 3 * R.U * 1.01 + 1e-15).all())
    _relbound(ref, bound, 1e-6)


def test_prior_and_euler_match_oracle():
    g = torch.Generator().manual_seed(8)
    B, T, Fb = 2, 5, 7
    y = torch.randn(B, T, Fb, 2, generator=g)
    z, x = torch.randn(B, T, Fb, 2, generator=g), torch.randn(B, T, Fb, 2, generator=g)
    m, r = torch.randn(B, T, Fb, 2, generator=g), torch.randn(B, T, Fb, 2, generator=g)
    smin, smax = 0.0, 0.5
    got, bound = R.axpy_ref(y, z, smax)
    want = O.fm_prior(torch.view_as_complex(y.double()), torch.view_as_complex(z.double()), smin, smax)
    _close(got, torch.view_as_real(want))
    _relbound(got, bound, 1e-6)
    mc, rc = torch.view_as_complex(m.double()), torch.view_as_complex(r.double())
    _, steps = O.euler_schedule(1.0, 0.03, 1)
    want = O.ode_sample(lambda xx, t, yy: -(mc * xx + rc), torch.view_as_complex(y.double()),
                        torch.view_as_complex(x.double()), N=1)                     # vf = -(m x + r), dt = -step
    got, bound = R.euler_step_ref(x, m, r, float(steps[0]))
    _close(got, torch.view_as_real(want))
    got2, _ = R.complex_mask_ref(x, m, r, -1.0)
    _close(got2, torch.view_as_real(-(mc * torch.view_as_complex(x.double()) + rc)))
    assert R.flow_grid_passes(303104) == 1 and R.flow_grid_passes(303105) == 2
