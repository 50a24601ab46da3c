"""Step-wise tensor-core BLSTM for hidden sizes the persistent cluster kernel does not cover (FlowSE: N = 384, H = 768;
reference nn.LSTM(N, 2N, bidirectional), bsrnn_flowse.py:226-238, called at :296-297 / :303-304).

One launch per (time step, direction): `bsrnn_lstm_step_tc` = tcgen05 GEMM h_{t-1} * W_hh^T whose epilogue adds the input
projection, applies the gates (f32, MUFU tanh), updates c in place and writes h_t in the KB8 tile layout -- the tile is
the next step's A operand and the layer output.  The input projection of ALL steps and both directions is one
`bsrnn_gemm_tc` launch (fp16 rows, bias in its epilogue).  Gate columns are interleaved (4u + gate) and the i/f/o rows
of W_ih / W_hh / bias pre-halved, exactly as in runtime_tc.pack_lstm_tc.

Layouts (rows of an axis are grouped in tiles of 128 sequences; m = step*tiles + j):
  xhat   [steps*tiles][kc_in][128][8] fp16          (bsrnn_norm_cast_kb8 with the axis' row map)
  gates  rows [m*128 + r][2 * 4H] fp16              (direction-major columns)
  y[d]   [steps*tiles][H/8][128][8] fp16            (per direction: the fc GEMM consumes the two as K halves)
"""
from __future__ import annotations

import torch

from . import _lib as L
from .runtime_tc import to_kb8, FC_EPI, lstm_ws, pack_fused, pack_steps, tile_width


def _bn_for(cols, kcores=None):
    """N-tile width of the step GEMM (widest that divides the gate columns).  BSRNN_STEP_RESIDENT=1 instead picks the widest
    tile whose W_hh slice stays RESIDENT in shared memory beside a 4-stage A ring (H = 768 -> BN = 96, 147 KB) with the h
    tiles multicast across clusters of N-tile CTAs -- measured slower (52 vs 34 us per step, profiles/r02 call13): the
    narrow tiles pay the per-K-stage pipeline handshake 2.7x more often; kept as an A/B switch."""
    import os
    forced = int(os.environ.get("BSRNN_STEP_BN", "0"))
    if forced:
        return forced
    if kcores is not None and os.environ.get("BSRNN_STEP_RESIDENT", "0") == "1":      # A/B switch, off: see launch_tc
        for bn in range(256, 63, -32):
            if cols % bn == 0 and kcores * bn * 16 + 65536 + 1024 <= 225 * 1024:
                return bn
    return tile_width(cols, 32)


def pack_lstm_steps_tc(rnn):
    """nn.LSTM(N, H, bidirectional), H % 16 == 0 -> the step-wise operands (runtime_tc.pack_steps) in BN-row tiles; at the
    FlowSE width (N = 384, H = 768) also the fused layer kernel's weights (pack_lstm_fused768)."""
    ws = lstm_ws(rnn)
    H, N = ws[1].shape[1], ws[0].shape[1]
    if H % 16:
        raise NotImplementedError(f"step-wise tensor-core LSTM needs H % 16 == 0, got {H}")
    kc_in = (N + 15) // 16 * 2
    BN = _bn_for(4 * H, H // 8)
    out = dict(pack_steps(ws, kc_in, BN), BN=BN, H=H, N=N, kc_in=kc_in, n_tiles=4 * H // BN)
    if H == 768 and N == 384:
        out.update(pack_lstm_fused768(rnn))
    return out


def pack_lstm_fused768(rnn):
    """nn.LSTM(384, 768, bidirectional) -> dict(wfused, kc_fused, one_col) for bsrnn_blstm_fused768_tc: runtime_tc.pack_fused
    at geometry 768, the bias in operand column 384 (norm_cast_kb8_ones writes the constant 1 there) of kc_fused = 50 k-cores."""
    N = rnn.weight_ih_l0.shape[1]
    return dict(wfused=pack_fused(lstm_ws(rnn), 768, 50, N), kc_fused=50, one_col=N)


# BSRNN_FLOWSE_FUSED=0 returns to the input-projection GEMM + one bsrnn_blstm_step_tc launch per time step
import os as _os
FLOWSE_FUSED = _os.environ.get("BSRNN_FLOWSE_FUSED", "1") == "1"
_FUSED_SLOTS = {"time": 0, "freq": 0}
for _kv in _os.environ.get("BSRNN_FLOWSE_FUSED_SLOTS", "").split(","):
    if "=" in _kv:
        _ax, _sv = _kv.split("=")
        _FUSED_SLOTS[_ax] = int(_sv)


class StepsWorkspace:
    def __init__(self, steps, tiles, H, dev):
        rows = steps * tiles * 128
        self.gates = torch.empty(rows, 2 * 4 * H, dtype=torch.float16, device=dev)
        self.y = [torch.empty(steps * tiles * (H // 8) * 1024, dtype=torch.float16, device=dev) for _ in range(2)]
        self.c = [torch.empty(tiles * 128, H, dtype=torch.float32, device=dev) for _ in range(2)]
        self.zero = torch.zeros(tiles * (H // 8) * 1024, dtype=torch.float16, device=dev)
        self.sync = torch.zeros(L.lib().bsrnn_blstm_fused_sync_bytes() // 4, dtype=torch.int32, device=dev)


def blstm_steps_tc(xhat, p, steps, tiles, ws: StepsWorkspace):
    """xhat: KB8 operand tiles of the normalised input (steps*tiles m-tiles).  Fills ws.y[0] (forward) / ws.y[1]."""
    st = L.stream_ptr()
    H, BN, nt = p["H"], p["BN"], p["n_tiles"]
    m_all = steps * tiles
    # all steps, both directions: gates rows = m*128 + r (identity row map), bias added in the epilogue
    L.call("bsrnn_gemm_tc", xhat.data_ptr(), p["wih"].data_ptr(), p["bias"].data_ptr(), ws.gates.data_ptr(), None, m_all,
           2 * nt, p["kc_in"], BN, L.TC_F16_ROWS, 8 * H, 8 * H, 0, 1, m_all, m_all * 128, 1 << 40, 0, 1, 0, st)
    tile_halves = (H // 8) * 1024
    for d in (0, 1):
        ws.c[d].zero_()
    g0 = ws.gates.data_ptr()
    for s in range(steps):
        ptrs = []
        for d in (0, 1):
            cur = s if d == 0 else steps - 1 - s
            prev = cur - 1 if d == 0 else cur + 1
            a_ptr = ws.zero.data_ptr() if s == 0 else ws.y[d].data_ptr() + 2 * prev * tiles * tile_halves
            ptrs += [a_ptr, p["whh"][d].data_ptr(), g0 + 2 * (cur * tiles * 128 * 8 * H + d * 4 * H), ws.c[d].data_ptr(),
                     ws.y[d].data_ptr() + 2 * cur * tiles * tile_halves]
        # both directions of the step in one launch: their launch / prologue / first-load latencies overlap
        L.call("bsrnn_blstm_step_tc", *ptrs, tiles, nt, BN, H, 8 * H, st)
    return ws.y


# ------------------------------------------------------------------------------------------------ dual path (FlowSE)
def pack_dual_path_steps(mod):
    """Tensor-core packing of the 2*num_layer (GN, BLSTM, Linear) blocks of a module with norm_/rnn_/fc_{time,freq}
    ModuleLists, for the step-wise kernels: the Linear(2H -> N) is split into its forward / backward K halves."""
    layers = []
    for i in range(mod.num_layer):
        e = {}
        for axis in ("time", "freq"):
            norm, rnn, fc = getattr(mod, f"norm_{axis}")[i], getattr(mod, f"rnn_{axis}")[i], getattr(mod, f"fc_{axis}")[i]
            p = pack_lstm_steps_tc(rnn)
            H, N = p["H"], fc.weight.shape[0]
            bn = tile_width((N + 15) // 16 * 16)
            nt = ((N + 15) // 16 * 16) // bn
            w = fc.weight.float()
            bias = torch.zeros(nt * bn, device=w.device)
            bias[:N] = fc.bias.float()
            p.update(gamma=norm.weight.float().contiguous(), beta=norm.bias.float().contiguous(), eps=float(norm.eps),
                     fcw=[to_kb8(w[:, :H], bn, H // 8), to_kb8(w[:, H:], bn, H // 8)], fcb=bias,
                     fcb0=torch.zeros_like(bias), fc_bn=bn, fc_nt=nt)
            if "wfused" in p:                # fused layer kernel: y is one [dir][96] operand, Linear(2H -> N) is ONE GEMM
                p["fc1"] = pack_linear_tc(fc)
            e[axis] = p
        layers.append(e)
    return layers


def pack_linear_tc(fc):
    """nn.Linear(K -> N) -> KB8 weight tiles + padded bias for bsrnn_gemm_tc (N tiles of bn columns, bn | ceil16(N))."""
    N, K = fc.weight.shape
    n16 = (N + 15) // 16 * 16
    bn = tile_width(n16)
    bias = torch.zeros(n16, device=fc.weight.device)
    bias[:N] = fc.bias.float()
    return dict(w=to_kb8(fc.weight.float(), bn, (K + 7) // 8), b=bias, bn=bn, nt=n16 // bn)


_WS = {}


def dual_path_tc_steps(skip, layers, t_emb=None):
    """In-place 2*num_layer residual blocks on skip (B,T,K,N) f32 with fp16 tensor-core GEMMs and the step-wise BLSTM.
    Same call pattern as runtime.dual_path_f32 (t_emb: list of (B,N) per layer, added after the time-axis GroupNorm)."""
    from .runtime import _layer_norm_tables, region
    if FLOWSE_FUSED and all("wfused" in lay[ax] for lay in layers for ax in ("time", "freq")):
        return dual_path_tc_fused768(skip, layers, t_emb)
    B, T, K, N = skip.shape
    dev = skip.device
    st = L.stream_ptr()
    H = layers[0]["time"]["H"]
    tiles_t, tiles_f = (B * K + 127) // 128, (B * T + 127) // 128
    key = (B, T, K, N, H, str(dev))
    ws = _WS.get(key)
    if ws is None:
        _WS.clear()
        kc_in = layers[0]["time"]["kc_in"]
        ntile = max(T * tiles_t, K * tiles_f)
        ws = _WS[key] = dict(xhat=torch.empty(ntile * kc_in * 1024, dtype=torch.float16, device=dev),
                             time=StepsWorkspace(T, tiles_t, H, dev), freq=StepsWorkspace(K, tiles_f, H, dev))
    for i, lay in enumerate(layers):
        for axis in ("time", "freq"):
            w = lay[axis]
            extra = t_emb[i] if (t_emb is not None and axis == "time") else None      # bsrnn_flowse.py:293-294
            if axis == "time":
                R_, steps, tiles, addr = B * K, T, tiles_t, (K, T * K, 1, K)
            else:
                R_, steps, tiles, addr = B * T, K, tiles_f, (1, K, 0, 1)
            with region("norm"):
                scale, shift = _layer_norm_tables(skip, w["gamma"], w["beta"], extra, w["eps"])
                L.call("bsrnn_norm_cast_kb8", skip.data_ptr(), scale.data_ptr(), shift.data_ptr(), ws["xhat"].data_ptr(),
                       N, 0, N, w["kc_in"], steps * tiles, tiles, R_, *addr, T * K, 1, st)
            with region(f"lstm_{axis}"):
                y = blstm_steps_tc(ws["xhat"], w, steps, tiles, ws[axis])
            with region("fc"):
                for half, bias in ((0, w["fcb"]), (1, w["fcb0"])):       # skip += y_fwd W_f^T + b, then += y_bwd W_b^T
                    L.call("bsrnn_gemm_tc", y[half].data_ptr(), w["fcw"][half].data_ptr(), bias.data_ptr(), skip.data_ptr(),
                           None, steps * tiles, w["fc_nt"], H // 8, w["fc_bn"], FC_EPI, N, N, 0, T * K,
                           tiles, R_, *addr, st)
    return skip


class Fused768Workspace:
    """Buffers of the fused FlowSE dual path for one (B, T, K) shape."""

    def __init__(self, B, T, K, N, H, kc, dev):
        from .runtime import _f64
        tiles_t, tiles_f = (B * K + 127) // 128, (B * T + 127) // 128
        ntile = max(T * tiles_t, K * tiles_f)
        self.xhat = torch.empty(ntile * kc * 1024, dtype=torch.float16, device=dev)
        self.y = torch.empty(ntile * 2 * (H // 8) * 1024, dtype=torch.float16, device=dev)     # [step][tile][dir][96][128][8]
        self.zero = torch.zeros((H // 8) * 1024, dtype=torch.float16, device=dev)
        self.sync = torch.zeros(L.lib().bsrnn_blstm_fused_sync_bytes() // 4, dtype=torch.int32, device=dev)
        self.stats = torch.zeros(B, 2, dtype=torch.float64, device=dev)
        self.scale = torch.empty(B, N, dtype=torch.float32, device=dev)
        self.shift = torch.empty(B, N, dtype=torch.float32, device=dev)
        self.counts = _f64([float(T) * K * N], dev)


def dual_path_tc_fused768(skip, layers, t_emb=None):
    """The 2*num_layer (GN, BLSTM, Linear) residual blocks of BSRNN_flowse (N = 384, H = 768) with ONE persistent kernel per
    BLSTM layer (bsrnn_blstm_fused768_tc: input projection + every time step of both directions), ONE Linear GEMM whose
    epilogue adds the residual and accumulates the next GroupNorm's statistics, and one normalise-and-cast pass: 3 launches
    per block instead of steps + 4."""
    from .runtime import region, keepalive
    B, T, K, N = skip.shape
    dev = skip.device
    st = L.stream_ptr()
    H = layers[0]["time"]["H"]
    tiles_t, tiles_f = (B * K + 127) // 128, (B * T + 127) // 128
    key = ("fused", B, T, K, N, H, str(dev))
    ws = _WS.get(key)
    if ws is None:
        _WS.clear()
        ws = _WS[key] = Fused768Workspace(B, T, K, N, H, layers[0]["time"]["kc_fused"], dev)
    keepalive(ws)
    y_tile = (H // 8) * 1024
    L.call("bsrnn_gn_stats", skip.data_ptr(), ws.stats.data_ptr(), B, T * K, N, N, st)
    for i, lay in enumerate(layers):
        for axis in ("time", "freq"):
            w = lay[axis]
            extra = t_emb[i] if (t_emb is not None and axis == "time") else None      # bsrnn_flowse.py:293-294
            if axis == "time":
                R_, steps, tiles, addr = B * K, T, tiles_t, (K, T * K, 1, K)
            else:
                R_, steps, tiles, addr = B * T, K, tiles_f, (1, K, 0, 1)
            with region("norm"):
                L.call("bsrnn_gn_finalize", ws.stats.data_ptr(), w["gamma"].data_ptr(), w["beta"].data_ptr(), L.ptr(extra),
                       ws.scale.data_ptr(), ws.shift.data_ptr(), B, N, ws.counts.data_ptr(), w["eps"], 1, st)
                # 50 k-cores: column 384 = 1 carries the bias through the fused contraction
                L.call("bsrnn_norm_cast_kb8_ones", skip.data_ptr(), ws.scale.data_ptr(), ws.shift.data_ptr(),
                       ws.xhat.data_ptr(), N, 0, N, w["kc_fused"], steps * tiles, tiles, R_, *addr, T * K, 1, w["one_col"], st)
            with region(f"lstm_{axis}"):
                L.call("bsrnn_blstm_fused768_tc", ws.xhat.data_ptr(), w["wfused"].data_ptr(), ws.zero.data_ptr(),
                       ws.y.data_ptr(), ws.y.data_ptr() + 2 * y_tile, 2 * y_tile, R_, steps, tiles, 0, _FUSED_SLOTS[axis],
                       ws.sync.data_ptr(), st)
            with region("fc"):
                ws.stats.zero_()
                fc = w["fc1"]
                L.call("bsrnn_gemm_tc", ws.y.data_ptr(), fc["w"].data_ptr(), fc["b"].data_ptr(), skip.data_ptr(),
                       ws.stats.data_ptr(), steps * tiles, fc["nt"], 2 * (H // 8), fc["bn"], FC_EPI, N, N, 0, T * K,
                       tiles, R_, *addr, st)
    return skip


# ------------------------------------------------------------------------------------------------ GradDecoder (FlowSE)
def pack_grad_decoder_tc(gd):
    """GradDecoder [reference bsrnn_flowse.py:103-168] for the tensor-core path: per band the Conv1d(N -> 16 s) as KB8
    weight tiles with rows permuted from c = sc*s + f to c' = f*16 + sc (the GEMM then writes the channel-last
    (B,T,F',16) image the 5x5 conv kernel reads), plus what runtime.pack_grad_decoder keeps (norm affine, conv weights)."""
    from .runtime import pack_grad_decoder
    base = pack_grad_decoder(gd)
    for name in ("mlp_mask", "mlp_residual"):
        p = base[name]
        N = p["w1"][0].shape[1]
        kc = (N + 15) // 16 * 2
        w, b, bn, nt = [], [], [], []
        for k, wk in enumerate(p["w1"]):                    # (16 s, N), rows already in c' order
            n16 = (wk.shape[0] + 15) // 16 * 16
            bk = tile_width(n16)
            w.append(to_kb8(wk, bk, kc))
            bb = torch.zeros(n16, device=wk.device); bb[: wk.shape[0]] = p["b1"][k]
            b.append(bb); bn.append(bk); nt.append(n16 // bk)
        p.update(w1_tc=w, b1_tc=b, bn=bn, nt=nt, kc=kc)
    return base


def grad_decoder_tc(skip, plan, gd_pack, sub_channel=16):
    """skip (B,T,K',N) -> mask, resid (B,T,F,2): the per-band Conv1d + Tanh as tcgen05 GEMMs (fp16 operands, f32 image),
    then the f32 5x5 conv + GLU kernel.  Mirrors runtime.grad_decoder_f32 (35.5 ms of CUDA-core GEMM per evaluation at
    BASELINE config 4, profiles/r02 call31)."""
    from .runtime import _decoder_norm_tables, region
    B, T, K, N = skip.shape
    F = plan.F
    Fp = sum(plan.subbands[:K])
    dev = skip.device
    st = L.stream_ptr()
    tabs = _decoder_norm_tables(skip, gd_pack)
    tiles = (B * T + 127) // 128
    img = torch.empty(2, B, T, Fp, sub_channel, dtype=torch.float32, device=dev)
    outs = []
    with region("graddec"):
        for gi, name in enumerate(("mlp_mask", "mlp_residual")):
            p = gd_pack[name]
            scale, shift = tabs[name][0], tabs[name][1]
            xhat = torch.empty(K * tiles * p["kc"] * 1024, dtype=torch.float16, device=dev)
            # rows of tile (k, j) are the (b,t) tokens of band k; GroupNorm(1,N) per (sample, band) folded into the cast
            L.call("bsrnn_norm_cast_kb8", skip.data_ptr(), scale.data_ptr(), shift.data_ptr(), xhat.data_ptr(), N, 0, N,
                   p["kc"], K * tiles, tiles, B * T, 1, K, 0, 1, T * K, K, st)
            base = img.data_ptr() + 4 * gi * B * T * Fp * sub_channel
            for k in range(K):
                L.call("bsrnn_gemm_tc", xhat.data_ptr() + 2 * k * tiles * p["kc"] * 1024, p["w1_tc"][k].data_ptr(),
                       p["b1_tc"][k].data_ptr(), base + 4 * plan.bin0[k] * sub_channel, None, tiles, p["nt"][k], p["kc"],
                       p["bn"][k], L.TC_TANH_F32, Fp * sub_channel, sub_channel * plan.subbands[k], 0, B * T, tiles, B * T,
                       1 << 60, 0, 1, 0, st)
            o = torch.empty(B, T, F, 2, dtype=torch.float32, device=dev)
            L.call("bsrnn_conv5x5_glu", img[gi].data_ptr(), p["cw"].data_ptr(), p["cb"].data_ptr(), o.data_ptr(), B, T, Fp, F, st)
            outs.append(o)
    return outs[0], outs[1]
