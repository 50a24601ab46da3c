"""Decoders of the packed fp16 BLSTM weight layouts (runtime_tc, runtime_tc_steps, training_tc) back to nn.LSTM's tensors.

Every decoder maps a packed buffer to per-direction (W_ih, W_hh, b) in nn.LSTM row order (gate*H + unit, gates i, f, g, o)
as f64 with GATE_SCALE removed, and asserts that every packed element that no LSTM element maps to (padding rows, padding
columns, padding k-cores) is exactly zero.  The packers promise

    decoded == fp16(w * scale) / scale          (scale = 0.5 for the i, f, o rows, 1 for g; scale = 1 for the TRUE-weight
                                                 transposes of BPTT)

so the GPU tests take the weights of their f64 reference from these decoders: kernel and reference then multiply the same
operands, bias included (the fp16-rounded bias in the constant-one operand column).
"""
import torch

GATE_SCALE = (0.5, 0.5, 1.0, 0.5)


def rounded(w, scale_rows=True):
    """fp16(w * scale) / scale in f64 for a (4H, ...) or (4H,) LSTM tensor: what a packer keeps of it."""
    w = w.detach().float()
    H = w.shape[0] // 4
    s = torch.tensor(GATE_SCALE if scale_rows else (1.0,) * 4, dtype=torch.float32).repeat_interleave(H)
    s = s.view(-1, *([1] * (w.dim() - 1)))
    return (w * s).half().double() / s.double()


def lstm_tensors(rnn):
    """per direction (W_ih, W_hh, b_ih + b_hh) of an nn.LSTM, f32 (the bias sum in the module's precision, as the packers)."""
    out = []
    for sfx in ("", "_reverse"):
        g = lambda n: getattr(rnn, n + sfx).detach().float()
        out.append((g("weight_ih_l0"), g("weight_hh_l0"), g("bias_ih_l0") + g("bias_hh_l0")))
    return out


def _unkb8(t):
    """[tiles][kcores][rpt][8] -> (tiles*rpt, kcores*8) f64."""
    tiles, kc, rpt, _ = t.shape
    return t.double().permute(0, 2, 1, 3).reshape(tiles * rpt, kc * 8)


def _scale_of_rows(gate):
    return torch.tensor(GATE_SCALE, dtype=torch.float64)[gate]


def zero_outside(mat, rows_used, cols_used, what):
    """every element of the 2-D `mat` outside rows_used x cols_used is exactly zero."""
    keep = torch.ones_like(mat, dtype=torch.bool)
    keep[rows_used[:, None], cols_used[None, :]] = False
    bad = mat[keep]
    assert bool((bad == 0).all()), f"{what}: {int((bad != 0).sum())} padding elements are not zero"


def decode_gate_rows(W, H, K, scaled=True, what="pack"):
    """KB8 weight tiles [n_tiles][kc][BN][8] whose packed row 4u + gate holds LSTM row gate*H + u (pack_lstm_steps_tc's
    whh / wih, pack_block's whh / wih): -> (4H, K) f64, scale removed; rows >= 4H and columns >= K must be zero."""
    return _decode_rows(_unkb8(W), H, K, scaled, what)


def _decode_rows(m, H, K, scaled=True, what="pack"):
    u = torch.arange(H)
    g = torch.arange(4)
    prow = (4 * u[None, :] + g[:, None]).reshape(-1)                    # packed row of LSTM row gate*H + u
    zero_outside(m, prow, torch.arange(K), what)
    out = m[prow, :K]
    if scaled:
        out = out / _scale_of_rows(g.repeat_interleave(H))[:, None]
    return out


def decode_lstm_steps(p):
    """runtime_tc_steps.pack_lstm_steps_tc -> [(W_ih, W_hh, b)] * 2.  wih: [2*4H/BN][kc_in][BN][8] (directions stacked);
    bias: f32 (2*4H,) scaled, NOT fp16-rounded; whh: per direction [4H/BN][H/8][BN][8]."""
    H, N, BN = p["H"], p["N"], p["BN"]
    wih = _unkb8(p["wih"])
    assert wih.shape[0] == 8 * H
    out = []
    for d in range(2):
        wi = _decode_rows(wih[d * 4 * H:(d + 1) * 4 * H], H, N, what=f"steps wih[{d}]")
        wh = decode_gate_rows(p["whh"][d], H, H, what=f"steps whh[{d}]")
        b = p["bias"][d * 4 * H:(d + 1) * 4 * H].double().view(H, 4).t().reshape(-1)
        b = b / _scale_of_rows(torch.arange(4).repeat_interleave(H))
        out.append((wi, wh, b))
    return out


def decode_lstm_tc(p):
    """runtime_tc.pack_lstm_tc -> dict(wih=[(W_ih, b_ih_col)] per direction from `wih` (+ the bias column when one_col >= 0),
    bih: the f32 bias table, whh: W_hh per direction, wfused: [(W_ih, W_hh, b)] per direction (None without one_col)).
    Layout: 8 CTAs q x 208 gate columns, packed column c = 4u + gate (u < 49) <- LSTM row gate*H + 49q + u; c >= 196 pads."""
    H, N, kc_in, oc = p["H"], p["N"], p["kc_in"], p["one_col"]
    assert H == 392
    CL, LU, LBN = 8, 49, 208
    u = torch.arange(LU)
    g = torch.arange(4)
    prow = (4 * u[None, :] + g[:, None]).reshape(-1)                    # [gate][u] -> packed column inside a CTA
    lrow = (g[:, None] * H + u[None, :]).reshape(-1)                    # [gate][u] -> LSTM row (q = 0)
    inv_s = 1.0 / _scale_of_rows(g.repeat_interleave(LU))
    wih = _unkb8(p["wih"])                                              # (16*208, kc_in*8)
    whh = p["whh"]                                                      # [2][8][50][208][8]
    bih = p["bih"].double()
    xcols = torch.arange(N) if oc < 0 else torch.cat([torch.arange(N), torch.tensor([oc])])
    res = dict(wih=[], bih=[], whh=[], wfused=[])
    for d in range(2):
        Wi = torch.zeros(4 * H, N, dtype=torch.float64)
        Wh = torch.zeros(4 * H, H, dtype=torch.float64)
        bc = torch.zeros(4 * H, dtype=torch.float64)
        bt = torch.zeros(4 * H, dtype=torch.float64)
        for q in range(CL):
            t = d * CL + q
            m = wih[t * LBN:(t + 1) * LBN]
            zero_outside(m, prow, xcols, f"lstm_tc wih[{d},{q}]")
            Wi[lrow + LU * q] = m[prow, :N] * inv_s[:, None]
            if oc >= 0:
                bc[lrow + LU * q] = m[prow, oc] * inv_s
            bq = bih[t * LBN:(t + 1) * LBN]
            assert bool((bq[torch.arange(4 * LU, LBN)] == 0).all()), f"lstm_tc bih[{d},{q}]: padding columns not zero"
            bt[lrow + LU * q] = bq[prow] * inv_s
            mh = _unkb8(whh[d, q][None])
            zero_outside(mh, prow, torch.arange(H), f"lstm_tc whh[{d},{q}]")
            Wh[lrow + LU * q] = mh[prow, :H] * inv_s[:, None]
        res["wih"].append((Wi, bc if oc >= 0 else None))
        res["bih"].append(bt)
        res["whh"].append(Wh)
    if "wfused" in p:
        # [dir][q][half e][kc_in + 50][104][8]: half e holds packed columns e*104 .. e*104 + 103 of CTA q
        wf = p["wfused"]
        P = wf.shape[1]
        for d in range(2):
            blocks = torch.stack([torch.cat([_unkb8(wf[d, q, e][None]) for e in range(2)], 0) for q in range(P)])
            res["wfused"].append(_decode_fused_blocks(blocks, H, N, kc_in, 50, oc, LU, prow_of=lambda U: prow, what="lstm_tc wfused"))
    else:
        res["wfused"] = None
    return res


def _decode_fused_blocks(blocks, H, N, kc_in, kc_h, oc, U, prow_of, what):
    """blocks (P, rows of a pair, (kc_in + kc_h)*8) f64: pair q's packed rows over K = [x cores (column oc = bias) | h cores]."""
    P = blocks.shape[0]
    g = torch.arange(4)
    u = torch.arange(U)
    prow = prow_of(U)
    lrow = (g[:, None] * H + u[None, :]).reshape(-1)
    inv_s = 1.0 / _scale_of_rows(g.repeat_interleave(U))
    cols = torch.cat([torch.arange(N), torch.tensor([oc]), kc_in * 8 + torch.arange(H)])
    Wi = torch.zeros(4 * H, N, dtype=torch.float64)
    Wh = torch.zeros(4 * H, H, dtype=torch.float64)
    b = torch.zeros(4 * H, dtype=torch.float64)
    assert blocks.shape[2] == (kc_in + kc_h) * 8
    for q in range(P):
        m = blocks[q]
        zero_outside(m, prow, cols, f"{what}[pair {q}]")
        rows = lrow + U * q
        Wi[rows] = m[prow, :N] * inv_s[:, None]
        b[rows] = m[prow, oc] * inv_s
        Wh[rows] = m[prow, kc_in * 8:kc_in * 8 + H] * inv_s[:, None]
    return (Wi, Wh, b)


def decode_fused_pairs(wf, H, N, kc_in, oc):
    """runtime_tc.pack_fused (P/U = 8/49, 7/56, 14/28, 24/32): [dir][pair q][half e][kc_in + kc_h k-cores][rh rows][8],
    rh = ceil16(4U) / 2; pair q's packed row 4*u_local + gate (half e = rows e*rh ..) <- LSTM row gate*H + U*q + u_local,
    rows >= 4U padding (208-row pairs at P = 8), K = [W_ih | bias at column oc | pad | W_hh | pad]."""
    _, P, _, kct, rh, _ = wf.shape
    U = H // P
    assert U * P == H and rh == (4 * U + 15) // 16 * 8
    kc_h = kct - kc_in
    g = torch.arange(4)
    out = []
    for d in range(2):
        blocks = torch.stack([torch.cat([_unkb8(wf[d, q, e][None]) for e in range(2)], 0) for q in range(P)])
        pr = lambda U_: (4 * torch.arange(U_)[None, :] + g[:, None]).reshape(-1)
        out.append(_decode_fused_blocks(blocks, H, N, kc_in, kc_h, oc, U, pr, f"fused P={P} dir {d}"))
    return out


def decode_transposed(WT, H, K_rows, what):
    """pack_block's whhT / wihT: KB8 [nt][4H/8][bn][8], row = unit u (whhT) or input n (wihT), K = packed gate column
    4u' + gate, TRUE weights -> (4H, K_rows) f64 in LSTM row order; rows >= K_rows must be zero."""
    m = _unkb8(WT)                                                      # (nt*bn, 4H)
    assert m.shape[1] == 4 * H
    zero_outside(m, torch.arange(K_rows), torch.arange(4 * H), what)
    u = torch.arange(H)
    g = torch.arange(4)
    pcol = (4 * u[None, :] + g[:, None]).reshape(-1)                    # packed column of LSTM row gate*H + u
    return m[:K_rows, pcol].t().contiguous()


def decode_pack_block(p):
    """training_tc.pack_block -> per direction dict(whhT=W_hh, wihT=W_ih) (TRUE weights) and, when the step-wise forward
    operands exist, whh / wih / b (scaled, from `whh`, `wih`, `bias`)."""
    H, N = p["H"], p["N"]
    out = []
    for d in range(2):
        e = dict(whhT=decode_transposed(p["whhT"][d], H, H, f"whhT[{d}]"), wihT=decode_transposed(p["wihT"][d], H, N, f"wihT[{d}]"))
        if "whh" in p:
            e["whh"] = decode_gate_rows(p["whh"][d], H, H, what=f"block whh[{d}]")
            e["wih"] = _decode_rows(_unkb8(p["wih"])[d * 4 * H:(d + 1) * 4 * H], H, N, what=f"block wih[{d}]")
            b = p["bias"][d * 4 * H:(d + 1) * 4 * H].double().view(H, 4).t().reshape(-1)
            e["b"] = b / _scale_of_rows(torch.arange(4).repeat_interleave(H))
        out.append(e)
    return out
