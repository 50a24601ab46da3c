"""f64 references and elementwise error bounds of the CUDA-core kernels -- the f32 grouped GEMM (csrc/gemm_f32.cu), the f32
BLSTM recurrence and its backward (csrc/lstm_f32.cu), BandSplit and its tensor-core operand builder (csrc/bandsplit.cu), the
GroupNorm statistics and tables (csrc/norm.cu) and the FlowSE pieces (csrc/flow.cu) -- and a restatement of their launchers'
geometry.  Used by tests/test_gpu_cuda_core.py; validated on the CPU by tests/test_cuda_core_ref_cpu.py.  Nothing here reads
a kernel's output, except where a reference is stated step-locally: it then takes the kernel's own previous state as input.

Every reference takes the f32 values the kernel receives and computes the operation in f64.  Notation: u = 2^-24 (unit
roundoff of f32, round to nearest), ulp(y) <= 2^-23 |y| for normal y, gamma_n = n u / (1 - n u).  Bounds are first order;
products of two bound terms are carried through (|x| + dx) factors, and the remaining second-order terms (u times a bound)
are covered by the factor SECOND = 1 + 2^-10.

gemm_f32.  A' = a * scale + shift is one fmaf or a rounded product and a rounded sum (contraction allowed): <= 2u (|a scale|
  + |shift|); rows k >= k_valid enter as a = 0, so A' = shift exactly.  The 64x64x16 tiles run ONE sequential fmaf chain
  over k = 0 .. K-1 from 0 (padding k >= K adds exact zeros): gamma_K sum_k |A' w|; the bias add rounds once:
      |v - ref| <= (2u [scale] + gamma_{K+1}) (sum_k (|a scale| + |shift|) |w| + |bias|)          (bound_v)
  tanhf <= 2 ulp (CUDA C++ Programming Guide, standard single-precision functions) and tanh' <= 1; the residual add rounds
  once.  GLU: out = v * 1 / (1 + __expf(-g)); __expf is off by at most 2 + floor(|1.173 x|) ulp (intrinsic functions table),
  1 + E rounds once and the IEEE division once, so with s = sigmoid(g) and sigmoid' <= 1/4:
      ds <= bound_g / 4 + s (1 - s) e_exp + u s ,     dout <= (s + ds) bound_v + |v| ds + u |out|.
lstm_f32 forward, step-local.  pre = (H-term fmaf chain of h_{s-1} W_hh^T from 0) + gates_x: gamma_{H+1} (sum |h w| +
  |gates_x|); at step 0 there is no chain and pre = 0 + gates_x exactly.  sigmoid = 1 / (1 + expf(-p)): expf <= 2 ulp, add
  and division one rounding each: ds <= dp / 4 + s (1 - s) 2^-22 + 2u s.  tanhf: dt <= dp + 2^-22 |t|.
  c = f c_prev + i g (two products and a sum, contraction allowed): 2u (|f c_prev| + |i g|) plus the propagated gate errors;
  h = o tanhf(c): one more rounding.  h_{s-1} (from y) and c_{s-1} (from saved) are the kernel's own, so errors do not
  compound over steps.
lstm_f32 backward.  The f64 BPTT runs from the kernel's saved (i, f, g, o, c) with the same recursion as the kernel; next to
  it a running error bound on magnitudes: dh = dy + dh_rec adds u |dh| to the carried e_rec; dc = dh o (1 - t^2) + dc_carry
  carries e_dh and e_carry and adds the tanhf error and 4 roundings; dc_carry' = dc f; each dG is a product of up to four
  factors (4 roundings, 1 - x rounds at most once) and dh_rec' = dG W_hh is a 4H-term fmaf chain:
      e_rec' = sum_n e_dG,n |W_nk| + gamma_{4H} sum_n |dG_n W_nk|.
  So the bound grows along the sequence exactly as the true error can.
band_split_fwd.  xn = fmaf(x, scale, shift) rounds once (u |xn|); the conv is ONE chain of 2 s_k fmaf starting from the bias
  (groups of four, padding channels add exact zeros): gamma_{2s} (|bias| + sum |xn w|) + u sum |xn| |w|.
band_norm_cast_kb8.  fmaf rounds once to f32 (u |v|), then __float2half_rn adds half an fp16 ulp of the f32 value.
gn_stats / band_stats.  Float partials of m terms (m restated per path below), each promoted to double: gamma_m sum |x| for
  the sum, gamma_{m+1} sum x^2 for the sum of squares (v * v rounds once more); the double warp / block / atomic sums add
  gamma^(53)_{n + 64} of the same magnitudes (n elements; order of atomics is free).
gn_finalize.  mean and var in double (4 double roundings of |Q/cnt| + mean^2, clamped at 0 exactly as the kernel does);
  mean -> f32 and rstd -> f32 round once each; sc = rstd ga one rounding; sh = be - mu sc one or two (contraction allowed);
  + extra one rounding.
conv5x5_glu.  One chain of 400 fmaf in (df, dt, ci) order from the bias: gamma_400 (|b| + sum |v w|); GLU with expf (<= 2 ulp)
  and IEEE division, sigmoid' <= 1/4 as above.
time_embed.  The phase ((t W) 2) pi is evaluated in f32 in the kernel's association; the same f32 products in torch round
  identically, so the phase is exact; sinf / cosf <= 2 ulp over the full range.
euler_step / complex_mask / axpy_complex.  Each component is a few roundings of the complex formula, contraction allowed:
  gamma_3 for m x + r, gamma_2 more for x + step (.), gamma_2 for y + sigma z.
"""
import math

import torch
import torch.nn.functional as F

U = 2.0 ** -24
ULP = 2.0 ** -23                       # ulp(y) <= ULP |y| for normal f32 y
U53 = 2.0 ** -53
SECOND = 1.0 + 2.0 ** -10              # second-order terms (see docstring)
TINY = 2.0 ** -140                     # absolute slack for results in the f32 subnormal range
SMEM_LIMIT = 227 * 1024                # bandsplit.cu: dynamic shared memory per block
STAT_CTAS = 148 * 8                    # norm.cu launchers: target CTA count of the statistics kernels
STAT_THREADS = 256
FLUSH = 64                             # norm.cu: float partials are flushed to double every 64 terms (flushed paths)
FLOW_CTAS, FLOW_THREADS = 148 * 8, 256 # flow.cu: grid-stride kernels


def gam(n, u=U):
    return n * u / (1.0 - n * u)


def cdiv(a, b):
    return -(-a // b)


def _d(x):
    return x.double()


# ---------------------------------------------------------------------------------------------------------- gemm_f32
GEMM_BM, GEMM_BN = 64, 64


def gemm_grid(max_m, max_n, n_groups):
    """bsrnn_gemm_f32: grid (ceil(max_n / 32), ceil(max_m / 64), n_groups) -- sized for 32-column GLU tiles."""
    return cdiv(max_n, GEMM_BN // 2), cdiv(max_m, GEMM_BM), n_groups


def gemm_group_tiles(M, N, epilogue):
    """(column tiles, row tiles) a group needs: GLU tiles produce 32 of the N / 2 logical columns, the others 64 of N."""
    glu = epilogue == 3
    n_out = N // 2 if glu else N
    return cdiv(n_out, GEMM_BN // 2 if glu else GEMM_BN), cdiv(M, GEMM_BM)


def gemm_branches(M, N, K, k_valid, epilogue, n_store, scaled, max_m, max_n):
    """Launcher / kernel branches one group of a bsrnn_gemm_f32 call reaches (for the static coverage test)."""
    gx, gy, _ = gemm_grid(max_m, max_n, 1)
    tx, ty = gemm_group_tiles(M, N, epilogue)
    assert gx >= tx and gy >= ty, "grid does not cover the group"
    n_out = N // 2 if epilogue == 3 else N
    b = {f"epilogue{epilogue}", "scaled" if scaled else "unscaled"}
    if gx > tx or gy > ty:
        b.add("early_exit")
    if M % GEMM_BM:
        b.add("partial_row_tile")
    if K % 16:
        b.add("partial_k_tile")
    if k_valid < K:
        b.add("k_valid")
    if n_store < n_out:
        b.add("n_store")
    if epilogue == 3 and n_out % 32:
        b.add("glu_partial_w")
    elif epilogue != 3 and N % GEMM_BN:
        b.add("partial_col_tile")
    return b


GEMM_BRANCHES = {"epilogue0", "epilogue1", "epilogue2", "epilogue3", "scaled", "unscaled", "early_exit", "partial_row_tile",
                 "partial_k_tile", "k_valid", "n_store", "glu_partial_w", "partial_col_tile"}


def _glu_bound(v, g, bv, bg):
    """out = v sigmoid(g) with sigmoid from __expf (gemm_f32) -- value and bound."""
    s = torch.sigmoid(g)
    e_exp = (2.0 + torch.floor(1.173 * (g.abs() + bg))) * ULP
    ds = bg / 4 + s * (1 - s) * e_exp + U * s
    out = v * s
    return out, ((s + ds) * bv + v.abs() * ds + U * out.abs()) * SECOND + TINY


def gemm_f32_ref(A, W, bias=None, scale=None, shift=None, k_valid=None, epilogue=0, C_old=None):
    """f64 reference of one bsrnn_gemm_f32 group on gathered operands: A (M, K) rows of A, W (N, K), bias (N), scale / shift
    (M, K) per row (the sample's table row), C_old (M, N') the output before a residual epilogue.  Returns (ref, bound) of
    the logical output (M, N) or (M, N / 2) for GLU."""
    Ad = _d(A).clone()
    M, K = Ad.shape
    if k_valid is not None and k_valid < K:
        Ad[:, k_valid:] = 0.0
    if scale is not None:
        Ap = Ad * _d(scale) + _d(shift)
        amag = (Ad * _d(scale)).abs() + _d(shift).abs()
        c_a = 2 * U
    else:
        Ap, amag, c_a = Ad, Ad.abs(), 0.0
    Wd = _d(W)
    v = Ap @ Wd.t()
    mag = amag @ Wd.abs().t()
    if bias is not None:
        v = v + _d(bias)
        mag = mag + _d(bias).abs()
    bv = (c_a + gam(K + 1)) * mag * SECOND
    if epilogue == 0:
        return v, bv
    if epilogue == 1:
        t = torch.tanh(v)
        return t, bv + 2 * ULP * t.abs() * SECOND + TINY
    if epilogue == 2:
        c = _d(C_old)
        return v + c, bv + U * (v.abs() + c.abs() + bv) * SECOND
    assert epilogue == 3
    h = v.shape[1] // 2
    return _glu_bound(v[:, :h], v[:, h:], bv[:, :h], bv[:, h:])


# ---------------------------------------------------------------------------------------------------------- lstm_f32
LSTM_LM, LSTM_LU = 64, 16


def lstm_grids(R, H):
    """Forward step grid (ceil(H/16), ceil(R/64), 2); backward gates grid (ceil(H/256), min(R, 65535), 2) looping over rows;
    backward dh grid (ceil(H/64), ceil(R/64), 2)."""
    return ((cdiv(H, LSTM_LU), cdiv(R, LSTM_LM), 2), (cdiv(H, 256), min(R, 65535), 2), (cdiv(H, 64), cdiv(R, 64), 2))


def seq_tokens(R, steps, seq_inner, seq_outer, seq_inner_stride, step_stride):
    """(R, steps) token of sequence r at step s (include/bsrnn_b200.h: SeqAddr)."""
    r = torch.arange(R, dtype=torch.long).view(-1, 1)
    s = torch.arange(steps, dtype=torch.long).view(1, -1)
    return (r // seq_inner) * seq_outer + (r % seq_inner) * seq_inner_stride + s * step_stride


def _sig_err(p, dp):
    s = torch.sigmoid(p)
    return s, dp / 4 + s * (1 - s) * 2 * ULP + 2 * U * s


def lstm_step_ref(gx, whh, h_prev=None, c_prev=None):
    """One step of one direction, f64.  gx (R, 4H) gates_x at this step, whh (4H, H), h_prev / c_prev (R, H) the kernel's
    previous state (None at step 0).  Returns dict of (ref, bound) for i, f, g, o, c and h."""
    gxd = _d(gx)
    H = whh.shape[1]
    if h_prev is None:
        pre, bp = gxd, torch.zeros_like(gxd)
    else:
        hd, wd = _d(h_prev), _d(whh)
        pre = gxd + hd @ wd.t()
        bp = gam(H + 1) * (hd.abs() @ wd.abs().t() + gxd.abs())
    pi, pf, pg, po = pre.split(H, 1)
    bi, bf, bg, bo = bp.split(H, 1)
    i, di = _sig_err(pi, bi)
    f, df = _sig_err(pf, bf)
    o, do = _sig_err(po, bo)
    g = torch.tanh(pg)
    dg = bg + 2 * ULP * g.abs()
    cp = torch.zeros_like(i) if c_prev is None else _d(c_prev)
    c = f * cp + i * g
    dc = cp.abs() * df + (g.abs() + dg) * di + (i + di) * dg + 2 * U * ((f * cp).abs() + (i * g).abs())
    tc = torch.tanh(c)
    dtc = dc + 2 * ULP * tc.abs()
    h = o * tc
    dh = tc.abs() * do + (o + do) * dtc + U * h.abs()
    out = dict(i=(i, di), f=(f, df), g=(g, dg), o=(o, do), c=(c, dc), h=(h, dh))
    return {k: (v, b * SECOND + TINY) for k, (v, b) in out.items()}


def lstm_forward_ref(gx, whh):
    """Full f64 BLSTM recurrence on sequence-major operands (the CPU check against nn.LSTM): gx (2, R, S, 4H), whh (2, 4H, H)
    -> y (R, S, 2H); direction 1 runs backwards."""
    _, R, S, H4 = gx.shape
    H = H4 // 4
    y = torch.zeros(R, S, 2 * H, dtype=torch.float64, device=gx.device)
    for d in range(2):
        h = c = None
        for q in range(S):
            s = q if d == 0 else S - 1 - q
            st = lstm_step_ref(gx[d, :, s], whh[d], h, c)
            h, c = st["h"][0], st["c"][0]
            y[:, s, d * H:(d + 1) * H] = h
    return y


def lstm_bwd_ref(saved, dy, whh):
    """f64 BPTT from the kernel's saved activations, with a running error bound.  Sequence-major operands: saved (2, R, S, 5,
    H) = (i, f, g, o, c), dy (2, R, S, H) = dL/dy of that direction, whh (2, 4H, H).  Returns dgates (2, R, S, 4H) and its
    bound.  Direction 0 is processed from s = S-1 down (predecessor s-1), direction 1 from s = 0 up (predecessor s+1)."""
    _, R, S, _, H = saved.shape
    sv, dyd = _d(saved), _d(dy)
    out = torch.zeros(2, R, S, 4 * H, dtype=torch.float64, device=saved.device)
    bnd = torch.zeros_like(out)
    for d in range(2):
        wd = _d(whh[d])
        wa = wd.abs()
        rec = carry = e_rec = e_carry = None
        order = range(S - 1, -1, -1) if d == 0 else range(S)
        for s in order:
            i, f, g, o, c = sv[d, :, s].unbind(1)
            sp = s - 1 if d == 0 else s + 1
            cp = sv[d, :, sp, 4] if 0 <= sp < S else torch.zeros_like(c)
            dh = dyd[d, :, s] + (0 if rec is None else rec)
            e_dh = (0 if e_rec is None else e_rec) + U * dh.abs()
            tc = torch.tanh(c)
            dtc = 2 * ULP * tc.abs()
            om = 1 - tc * tc
            e_om = 2 * tc.abs() * dtc + U * (tc * tc + om.abs())
            term = dh * o * om
            dc = term + (0 if carry is None else carry)
            e_dc = (e_dh * (o * om).abs() + (dh * o).abs() * e_om + 2 * U * term.abs()
                    + (0 if e_carry is None else e_carry) + U * dc.abs())
            gi = dc * g * i * (1 - i)
            gf = dc * cp * f * (1 - f)
            gg = dc * i * (1 - g * g)
            go = dh * tc * o * (1 - o)
            e_gi = e_dc * (g * i * (1 - i)).abs() + 5 * U * gi.abs()
            e_gf = e_dc * (cp * f * (1 - f)).abs() + 5 * U * gf.abs()
            e_gg = e_dc * (i * (1 - g * g)).abs() + (dc * i).abs() * U * (g * g + (1 - g * g).abs()) + 3 * U * gg.abs()
            e_go = e_dh * (tc * o * (1 - o)).abs() + (dh * o * (1 - o)).abs() * dtc + 5 * U * go.abs()
            dG = torch.cat([gi, gf, gg, go], 1)
            eG = torch.cat([e_gi, e_gf, e_gg, e_go], 1) * SECOND + TINY
            out[d, :, s], bnd[d, :, s] = dG, eG
            carry = dc * f
            e_carry = e_dc * f + U * carry.abs()
            rec = dG @ wd
            e_rec = (eG @ wa + gam(4 * H) * (dG.abs() @ wa)) * SECOND
    return out, bnd


# ---------------------------------------------------------------------------------------------------------- bandsplit
BS_ROWS = 128


def band_split_smem(C, N):
    """bandsplit.cu smem_of: the band's transposed weight and the 128-row input tile, channels padded to 4."""
    Cp = (C + 3) & ~3
    return Cp * N * 4 + BS_ROWS * Cp * 4


def band_split_runs(c_off, N):
    """The launches of bsrnn_band_split_fwd: consecutive bands whose shared-memory need is within 2x of the run's maximum
    share one launch.  Returns [(k_lo, k_hi, smem bytes)]."""
    K = len(c_off) - 1
    runs, k = [], 0
    while k < K:
        need = band_split_smem(c_off[k + 1] - c_off[k], N)
        e = k + 1
        while e < K:
            s = band_split_smem(c_off[e + 1] - c_off[e], N)
            if s > 2 * need or 2 * s < need:
                break
            need = max(need, s)
            e += 1
        runs.append((k, e, need))
        k = e
    return runs


def band_split_fits(c_off, N):
    return all(band_split_smem(c_off[j + 1] - c_off[j], N) <= SMEM_LIMIT for j in range(len(c_off) - 1))


def band_inputs(spec, T, bin0, width2, C, k, K, cmax, scale, shift):
    """Band k's normalised inputs of bsrnn_band_split_fwd / _kb8, f64: x (rows, C) zero beyond width2 (a truncated band is
    padded BEFORE the norm), xn = x * scale[b*K + k] + shift[...].  spec (rows, F2).  Returns (x, xn)."""
    rows = spec.shape[0]
    x = torch.zeros(rows, C, dtype=torch.float64, device=spec.device)
    x[:, :width2] = _d(spec[:, 2 * bin0: 2 * bin0 + width2])
    b = torch.arange(rows, device=spec.device) // T
    sc = _d(scale.view(-1, K, cmax)[b, k, :C])
    sh = _d(shift.view(-1, K, cmax)[b, k, :C])
    return x, sc, sh


def band_split_ref(spec, T, scale, shift, wT, bias, c_off, bin0, width2, cmax, N):
    """f64 BandSplit per band: list of (ref, bound), each (rows, N)."""
    K = len(c_off) - 1
    res = []
    for k in range(K):
        C = c_off[k + 1] - c_off[k]
        x, sc, sh = band_inputs(spec, T, bin0[k], width2[k], C, k, K, cmax, scale, shift)
        xn = x * sc + sh
        w = _d(wT[c_off[k]: c_off[k + 1]])
        b = _d(bias.view(K, N)[k])
        ref = xn @ w + b
        mag = xn.abs() @ w.abs()
        res.append((ref, ((gam(C) + U) * mag + gam(C) * b.abs()) * SECOND + TINY))
    return res


def half_ulp16(x):
    """half the fp16 spacing at magnitude x (f64 tensor), subnormals included."""
    e = torch.floor(torch.log2(x.abs().clamp(min=2.0 ** -14)))
    return torch.exp2(e - 11)


def band_cast_ref(spec, T, scale, shift, c_off, bin0, width2, cmax, k):
    """Band k of bsrnn_band_norm_cast_kb8 as a (rows, C) matrix: ref and bound (one f32 fmaf rounding, then fp16)."""
    K = len(c_off) - 1
    C = c_off[k + 1] - c_off[k]
    x, sc, sh = band_inputs(spec, T, bin0[k], width2[k], C, k, K, cmax, scale, shift)
    v = x * sc + sh
    return v, U * v.abs() + half_ulp16(v.abs() * (1 + U))


def kb8_geometry(C, rows):
    """bsrnn_band_norm_cast_kb8: kc = 2 ceil(C / 16) cores of 8 halves, row tiles of 128; band extent kc * 1024 per tile."""
    kc = 2 * cdiv(C, 16)
    return kc, cdiv(rows, 128), kc * 1024 * cdiv(rows, 128)


# ---------------------------------------------------------------------------------------------------------- GroupNorm
def gn_stats_geometry(B, rows_per_sample, C, row_stride):
    """bsrnn_gn_stats: chunks = ceil(1184 / B), rows per block = max(1, ceil(rows / chunks)), grid.x = ceil(rows / rpb); the
    number of terms per float partial: <= 64 on the contiguous path (flushed every 64, each thread takes every 256th
    element of the block's range), rows_per_block * ceil(C / 256) on the strided path (no flush)."""
    chunks = cdiv(STAT_CTAS, B)
    rpb = max(1, cdiv(rows_per_sample, chunks))
    blocks = cdiv(rows_per_sample, rpb)
    contiguous = row_stride == C
    if contiguous:
        m = min(FLUSH, cdiv(rpb * C, STAT_THREADS))
    else:
        m = rpb * cdiv(C, STAT_THREADS)
    return dict(chunks=chunks, rpb=rpb, blocks=blocks, contiguous=contiguous, m=m)


def band_stats_geometry(B, T, n_bands, max_width):
    """bsrnn_band_stats: tchunks = min(T, 1184 // (B n_bands) + 1), t_per_block = ceil(T / tchunks), grid.z = ceil(T / tpb);
    per float partial at most min(64, ceil(tpb * width / 256)) terms (flushed)."""
    tchunks = min(T, STAT_CTAS // (B * n_bands) + 1)
    tpb = cdiv(T, tchunks)
    return dict(tchunks=tchunks, tpb=tpb, zblocks=cdiv(T, tpb), m=min(FLUSH, cdiv(tpb * max_width, STAT_THREADS)))


def sums_ref(x, m):
    """{sum, sum of squares} of f32 values x (..., n) over the last dim, f64, and their bounds for float partials of m terms
    promoted to double (plus the double sums of n + 64 terms)."""
    xd = _d(x)
    n = x.shape[-1]
    a, q = xd.abs().sum(-1), (xd * xd).sum(-1)
    dbl = gam(n + 64, U53)
    return xd.sum(-1), q, (gam(m) + dbl) * a * SECOND, (gam(m + 1) + dbl) * q * SECOND


def gn_finalize_ref(stats, gamma, beta, extra, counts, eps, G_inner):
    """f64 reference of bsrnn_gn_finalize: stats (G, 2) double, gamma / beta (G_inner, C), counts (G_inner), extra (G, C) or
    None.  Returns (scale, bound), (shift, bound), each (G, C)."""
    G = stats.shape[0]
    gi = torch.arange(G, device=stats.device) % G_inner
    cnt = _d(counts)[gi]
    S, Q = _d(stats[:, 0]), _d(stats[:, 1])
    mean = S / cnt
    ex2 = Q / cnt
    var = (ex2 - mean * mean).clamp(min=0.0)
    dvar = 4 * U53 * (ex2.abs() + mean * mean)
    rstd = 1.0 / torch.sqrt(var + eps)
    drstd = 0.5 * ((var - dvar).clamp(min=0.0) + eps) ** -1.5 * dvar + U * rstd
    dmu = U * mean.abs() + 2 * U53 * mean.abs()
    ga, be = _d(gamma)[gi], _d(beta)[gi]
    sc = rstd[:, None] * ga
    dsc = ga.abs() * drstd[:, None] + U * sc.abs()
    sh = be - mean[:, None] * sc
    dsh = (mean.abs()[:, None] * dsc + (sc.abs() + dsc) * dmu[:, None]
           + U * (mean[:, None] * sc).abs() + U * sh.abs())
    if extra is not None:
        sh = sh + _d(extra)
        dsh = dsh + U * sh.abs()
    return (sc, dsc * SECOND + TINY), (sh, dsh * SECOND + TINY)


# ---------------------------------------------------------------------------------------------------------- flow
CONV_CT, CONV_CF = 8, 32


def conv_grid(B, T, Fp, F):
    """bsrnn_conv5x5_glu: grid (ceil(max(F, Fp) / 32), ceil(T / 8), B)."""
    return cdiv(max(F, Fp), CONV_CF), cdiv(T, CONV_CT), B


def conv5x5_glu_ref(g, weight, bias, F_out):
    """g (B, T, Fp, 16) channel-last -> (B, T, F_out, 2) f64 and bound: Conv2d(16 -> 4, 5x5, pad 2) over the (F', T) image,
    GLU over the 4 channels, bins >= Fp exactly 0."""
    B, T, Fp, _ = g.shape
    img = _d(g).permute(0, 3, 2, 1)                                        # (B, 16, Fp, T)
    w, b = _d(weight), _d(bias)
    acc = F.conv2d(img, w, b, padding=2)                                   # (B, 4, Fp, T)
    mag = F.conv2d(img.abs(), w.abs(), b.abs(), padding=2)
    bv = gam(400) * mag * SECOND
    outs, bnds = [], []
    for j in range(2):
        s = torch.sigmoid(acc[:, j + 2])
        ds = bv[:, j + 2] / 4 + s * (1 - s) * 2 * ULP + U * s
        o = acc[:, j] * s
        outs.append(o)
        bnds.append(((s + ds) * bv[:, j] + acc[:, j].abs() * ds + U * o.abs()) * SECOND + TINY)
    ref = torch.zeros(B, T, F_out, 2, dtype=torch.float64, device=g.device)
    bnd = torch.zeros_like(ref)
    n = min(Fp, F_out)
    ref[:, :, :n] = torch.stack(outs, -1).permute(0, 2, 1, 3)[:, :, :n]
    bnd[:, :, :n] = torch.stack(bnds, -1).permute(0, 2, 1, 3)[:, :, :n]
    return ref, bnd


def time_phase_f32(t, W):
    """The kernel's f32 phase ((t W) 2) pi, evaluated left to right in f32 (B, E)."""
    return ((t.float()[:, None] * W.float()[None, :]) * 2.0) * torch.tensor(math.pi, dtype=torch.float32)


def time_embed_ref(t, W):
    """(B, 2E) [sin, cos] of the f32 phase, f64, and the 2-ulp bound."""
    p = _d(time_phase_f32(t, W))
    ref = torch.cat([torch.sin(p), torch.cos(p)], -1)
    return ref, 2 * ULP * ref.abs() * SECOND + 2.0 ** -148


def _cmul_add(x, m, r):
    xd, md, rd = _d(x), _d(m), _d(r)
    gx = md[..., 0] * xd[..., 0] - md[..., 1] * xd[..., 1] + rd[..., 0]
    gy = md[..., 0] * xd[..., 1] + md[..., 1] * xd[..., 0] + rd[..., 1]
    ax = (md[..., 0] * xd[..., 0]).abs() + (md[..., 1] * xd[..., 1]).abs() + rd[..., 0].abs()
    ay = (md[..., 0] * xd[..., 1]).abs() + (md[..., 1] * xd[..., 0]).abs() + rd[..., 1].abs()
    return torch.stack([gx, gy], -1), gam(3) * torch.stack([ax, ay], -1)


def complex_mask_ref(x, m, r, sign):
    """sign (m x + r) on (..., 2) re/im pairs."""
    g, b = _cmul_add(x, m, r)
    return sign * g, b * SECOND + TINY


def euler_step_ref(x, m, r, step):
    """x + step (m x + r)."""
    g, b = _cmul_add(x, m, r)
    xd = _d(x)
    step = float(torch.tensor(step, dtype=torch.float32))
    out = xd + step * g
    return out, (abs(step) * b + gam(2) * (xd.abs() + abs(step) * (g.abs() + b))) * SECOND + TINY


def axpy_ref(y, z, sigma):
    """y + sigma z."""
    sigma = float(torch.tensor(sigma, dtype=torch.float32))
    yd, zd = _d(y), _d(z)
    out = yd + sigma * zd
    return out, gam(2) * (yd.abs() + abs(sigma) * zd.abs()) * SECOND + TINY


def flow_grid_passes(n_complex):
    """Grid-stride passes of the flow.cu elementwise kernels (1184 CTAs x 256 threads)."""
    return cdiv(n_complex, FLOW_CTAS * FLOW_THREADS)
