"""Tensor-core ("fp16") mode of the runtime: weight packing into the UMMA-native KB8 tiling and the sequencing of
bsrnn_norm_cast_kb8 / bsrnn_gemm_tc / bsrnn_blstm_recurrence_tc (include/bsrnn_b200.h).  H = 2N = 392 only
(BSRNN_baseline, N = 196): the recurrence kernel is specialised for that size (csrc/lstm_tc.cu).
"""
from __future__ import annotations

import torch

from . import _lib as L
from .runtime import region, _f64, keepalive

import os

BIG = 1 << 60
# recurrence schedule per axis: interleaved slots of bsrnn_blstm_recurrence_tc_ex, e.g. BSRNN_LSTM_SLOTS="time=3,freq=2"
_LSTM_SLOTS = {"time": 3, "freq": 3}
for _kv in os.environ.get("BSRNN_LSTM_SLOTS", "").split(","):
    if "=" in _kv:
        _ax, _sv = _kv.split("=")
        _LSTM_SLOTS[_ax] = int(_sv)
# recurrence schedule: "flag" = groups of 8 CTAs synchronised through global-memory counters (18 groups = 144 SMs),
# "cluster" = 8-CTA thread-block clusters (15 co-resident = 120 SMs).  BSRNN_LSTM_SCHED overrides.
LSTM_SCHED = os.environ.get("BSRNN_LSTM_SCHED", "flag")
_FLAG_SLOTS = {"time": 0, "freq": 0}    # 0 = automatic (fewest interleaved tiles that cover all units in one wave)
for _kv in os.environ.get("BSRNN_LSTM_FLAG_SLOTS", "").split(","):
    if "=" in _kv:
        _ax, _sv = _kv.split("=")
        _FLAG_SLOTS[_ax] = int(_sv)
# axes whose BLSTM runs as ONE fused kernel (input projection inside the recurrence, csrc/lstm_fused.cu):
# BSRNN_LSTM_FUSED="time,freq" (default) | "freq" | "none" (separate input-projection GEMM + bsrnn_blstm_recurrence_tc*)
FUSED_AXES = tuple(a for a in os.environ.get("BSRNN_LSTM_FUSED", "time,freq").split(",") if a in ("time", "freq"))
# group geometry of the fused kernel: 8 pairs x 49 units (9 groups), 7 pairs x 56 units (10 groups = 5 per direction) or
# 14 pairs x 28 units (5 groups; small batches: half the per-step chain).  BSRNN_LSTM_FUSED_GEO = 8 | 7 | 14 | auto (default)
FUSED_GEO = os.environ.get("BSRNN_LSTM_FUSED_GEO", "auto")


GEO14_MAX_PTILES = int(os.environ.get("BSRNN_LSTM_GEO14_MAX_PTILES", "3"))


def _passes(ptiles, groups, slots):
    """(passes, interleaved pairs) of the cheapest schedule: a step costs max(dependency chain ~ 2.3 items, slots items)."""
    best = None
    for s in range(1, min(slots, ptiles) + 1):
        gpd = (ptiles + s - 1) // s
        t = ((2 * gpd + groups - 1) // groups) * max(2.3, float(s))
        if best is None or t < best - 1e-9:
            best = t
    return best


def fused_geometry(tiles):
    """7 when the 10-group geometry needs fewer item times for this tile count (an item costs 8 % more there: N = 224)."""
    if FUSED_GEO in ("7", "8", "14"):
        return int(FUSED_GEO)
    ptiles = (tiles + 1) // 2
    if ptiles <= GEO14_MAX_PTILES:          # chain-bound regime: few tile pairs, every unit (nearly) alone on a group
        return 14
    return 7 if 1.08 * _passes(ptiles, 10, 3) < _passes(ptiles, 9, 3) - 1e-9 else 8


_FUSED_SLOTS = {"time": 0, "freq": 0}
for _kv in os.environ.get("BSRNN_LSTM_FUSED_SLOTS", "").split(","):
    if "=" in _kv:
        _ax, _sv = _kv.split("=")
        _FUSED_SLOTS[_ax] = int(_sv)
# epilogue of the Linear(4N->N) + skip GEMM: residual rows through the TMA unit (bsrnn_gemm_tc epilogue 8, default) or
# register-staged 16-byte loads / stores (epilogue 1, BSRNN_FC_EPI=ldst)
FC_EPI = L.TC_RESID_F32 if os.environ.get("BSRNN_FC_EPI", "tma") == "ldst" else L.TC_RESID_TMA
CL, LU, LBN, LKC = 8, 49, 208, 50       # cluster size, units per CTA, gate columns per CTA, k-cores of h (K = 400)
LGC = LBN // 8                           # gates_x cores per CTA
GATE_SCALE = (0.5, 0.5, 1.0, 0.5)       # i, f, o rows pre-halved: sigmoid(x) = 0.5*tanh(x/2) + 0.5 in the kernel


def to_kb8(w, rows_per_tile, kcores):
    """(rows, K) -> fp16 [n_tiles][kcores][rows_per_tile][8]; rows / K zero padded."""
    rows, K = w.shape
    n_tiles = (rows + rows_per_tile - 1) // rows_per_tile
    buf = torch.zeros(n_tiles * rows_per_tile, kcores * 8, dtype=torch.float32, device=w.device)
    buf[:rows, :K] = w
    return buf.view(n_tiles, rows_per_tile, kcores, 8).permute(0, 2, 1, 3).contiguous().to(torch.float16)


def from_kb8(t, rows, K):
    """inverse of to_kb8 (test helper): [n_tiles][kcores][rpt][8] -> (rows, K) f32."""
    n_tiles, kcores, rpt, _ = t.shape
    return t.permute(0, 2, 1, 3).reshape(n_tiles * rpt, kcores * 8)[:rows, :K].float()


def tile_width(cols, mult=16):
    """widest multiple of `mult` <= 256 that divides cols: the N-tile width of a GEMM over cols output columns."""
    for bn in range(256, mult - 1, -mult):
        if cols % bn == 0:
            return bn
    raise NotImplementedError(f"no tile width for {cols} columns")


# ------------------------------------------------------------------------------------------------ packed BLSTM weights
# Every tensor-core BLSTM layout is cut from one block of gate rows per (direction, pair q): packed row 4*u + gate of pair q
# is LSTM row gate*H + U*q + u (gates i, f, g, o), its i, f and o rows pre-halved by GATE_SCALE.  The step-wise kernels see a
# single pair (P = 1, U = H).

# fused layer kernel geometry -> (pairs per group P, hidden units per pair U): PPG / UPP of the csrc/lstm_fused.cu struct
FUSED_PAIRS = {8: (8, 49),         # Geo392
               7: (7, 56),         # Geo392x7
               14: (14, 28),       # Geo392x14
               768: (24, 32)}      # Geo768
_GATE_ROWS = {}


def lstm_ws(rnn):
    """the 8 tensors of a one-layer bidirectional nn.LSTM in the packers' order: w_ih, w_hh, b_ih, b_hh, then the reverse four."""
    return tuple(getattr(rnn, n + sfx) for sfx in ("", "_reverse") for n in ("weight_ih_l0", "weight_hh_l0", "bias_ih_l0", "bias_hh_l0"))


def gate_row_map(H, P, U, dev):
    """(rows (P, R) int64, scale (R, 1) f32), R = ceil16(4U): rows[q, 4*u + gate] = gate*H + U*q + u, and 4H (a zero row of
    gate_rows' source) for the padding rows past 4U; scale = GATE_SCALE of each packed row.  Built once per (H, P, U, device):
    an H2D copy from pageable memory is a stream synchronisation, and the training step packs inside every block."""
    key = (H, P, U, str(dev))
    t = _GATE_ROWS.get(key)
    if t is None:
        R = (4 * U + 15) // 16 * 16
        q = torch.arange(P, device=dev)[:, None, None]
        u = torch.arange(U, device=dev)[None, :, None]
        g = torch.arange(4, device=dev)[None, None, :]
        rows = torch.full((P, R), 4 * H, dtype=torch.long, device=dev)
        rows[:, :4 * U] = (g * H + U * q + u).reshape(P, 4 * U)
        scale = torch.zeros(R, device=dev)
        scale[:4 * U] = torch.tensor(GATE_SCALE, device=dev).repeat(U)
        t = _GATE_ROWS[key] = (rows, scale[:, None])
    return t


@torch.no_grad()
def gate_rows(ws, P, U, kc_in, one_col=-1):
    """The gate rows of the 8 LSTM tensors ws (lstm_ws order) for groups of P pairs x U units: (w (2, P, R, (kc_in + kc_h) * 8),
    b (2, P, R)) f32, R = ceil16(4U), kc_h = ceil16(H) / 8, rows past 4U zero.  Columns of w: [W_ih | pad | W_hh | pad] over
    kc_in + kc_h k-cores, and b_ih + b_hh in column one_col too when one_col >= 0 (the operand's constant-one column).  b is
    the f32 bias.  Both carry GATE_SCALE.  A few batched ops without a host synchronisation: it runs in every training step."""
    w_ih, w_hh, b_ih, b_hh, w_ih_r, w_hh_r, b_ih_r, b_hh_r = ws
    H, N = w_hh.shape[1], w_ih.shape[1]
    K = (kc_in + (H + 15) // 16 * 2) * 8
    rows, scale = gate_row_map(H, P, U, w_hh.device)
    src = torch.zeros(2, 4 * H + 1, K + 1, device=w_hh.device)         # row 4H stays zero; column K holds the bias
    lstm = src[:, :4 * H]
    lstm[..., :N] = torch.stack((w_ih, w_ih_r))
    lstm[..., kc_in * 8: kc_in * 8 + H] = torch.stack((w_hh, w_hh_r))
    lstm[..., K] = torch.stack((b_ih + b_hh, b_ih_r + b_hh_r))
    if one_col >= 0:
        src[:, :, one_col] = src[:, :, K]
    w = src[:, rows] * scale                                             # (2, P, R, K + 1)
    return w[..., :K], w[..., K]


def pack_fused(ws, geo, kc_in, one_col):
    """Weights of the fused layer kernel of geometry `geo` (FUSED_PAIRS): [dir][pair q][half e][kc_in + kc_h k-cores][R/2][8]
    fp16, half e holding gate rows e*R/2 .. of pair q; the bias rides in operand column one_col."""
    P, U = FUSED_PAIRS[geo]
    w = gate_rows(ws, P, U, kc_in, one_col)[0]
    R, K = w.shape[2:]
    return w.view(2, P, 2, R // 2, K // 8, 8).permute(0, 1, 2, 4, 3, 5).contiguous().to(torch.float16)


def pack_steps(ws, kc_in, BN):
    """Operands of the step-wise kernels (one pair of U = H units, BN-row tiles): wih [2*4H/BN][kc_in][BN][8] (directions
    stacked) for the input-projection GEMM, whose epilogue adds `bias` (2*4H) f32; whh per direction [4H/BN][kc_h][BN][8]."""
    H = ws[1].shape[1]
    kc_h = (H + 15) // 16 * 2
    w, b = gate_rows(ws, 1, H, kc_in)
    w, k0 = w[:, 0], kc_in * 8
    return dict(wih=to_kb8(w[..., :k0].reshape(8 * H, k0), BN, kc_in), whh=[to_kb8(w[d, :, k0:], BN, kc_h) for d in (0, 1)],
                bias=b.flatten().contiguous())


def pack_lstm_tc(rnn):
    """nn.LSTM(N, H=392, bidirectional) -> dict(wih [16][26][208][8], bih (16*208) f32, whh [2][8][50][208][8]): 8 CTAs of
    49 units, 208 gate rows each.

    When the operand has a padding column (N < kc_in*8) the bias b_ih + b_hh is ALSO stored as weight column N
    (`one_col`): norm_cast_kb8_ones writes the constant 1 there and the input-projection GEMM runs without a bias
    epilogue (its epilogue is then a pure convert-and-store at HBM write speed).  The fused layer kernel needs that column:
    only then are its weights packed (`wfused`, geometry 8; the others on first use, fused_weights)."""
    ws = lstm_ws(rnn)
    H, N = ws[1].shape[1], ws[0].shape[1]
    if H != CL * LU:
        raise NotImplementedError(f"tensor-core BLSTM kernel is specialised for H=392, got H={H}")
    kc_in = (N + 15) // 16 * 2
    one_col = N if (N % 4 == 0 and N < kc_in * 8) else -1
    w, b = gate_rows(ws, CL, LU, kc_in, one_col)
    out = dict(wih=to_kb8(w[..., :kc_in * 8].reshape(-1, kc_in * 8), LBN, kc_in), bih=b.flatten().contiguous(),
               whh=to_kb8(w[..., kc_in * 8:].reshape(-1, LKC * 8), LBN, LKC).view(2, CL, LKC, LBN, 8),
               kc_in=kc_in, H=H, N=N, one_col=one_col)
    if one_col >= 0:
        out.update(wfused=pack_fused(ws, 8, kc_in, one_col), _ws=ws)
    return out


def fused_weights(w, geo):
    """Packed weights of the fused layer kernel for group geometry `geo` (8, 7 or 14), built on first use and kept in the
    layer's pack dict (which PackedCache rebuilds whenever a parameter changes)."""
    key = "wfused" if geo == 8 else f"wfused{geo}"
    if key not in w:
        w[key] = pack_fused(w["_ws"], geo, w["kc_in"], w["one_col"])
    return w[key]


def pack_fc_tc(fc, H):
    """Linear(2H -> N): K re-indexed to the y tile's [dir][400] columns; one N tile of BN = ceil16(N)."""
    N = fc.weight.shape[0]
    BN = (N + 15) // 16 * 16
    w = torch.zeros(N, 2 * LKC * 8, device=fc.weight.device)
    w[:, :H] = fc.weight[:, :H]
    w[:, LKC * 8: LKC * 8 + H] = fc.weight[:, H:]
    bias = torch.zeros(BN, device=w.device)
    bias[:N] = fc.bias
    return dict(w=to_kb8(w, BN, 2 * LKC), b=bias, BN=BN, N=N)


def pack_dual_path_tc(mod):
    layers = []
    for i in range(mod.num_layer):
        e = {}
        for axis in ("time", "freq"):
            norm, rnn, fc = getattr(mod, f"norm_{axis}")[i], getattr(mod, f"rnn_{axis}")[i], getattr(mod, f"fc_{axis}")[i]
            p = pack_lstm_tc(rnn)
            p.update(gamma=norm.weight.float().contiguous(), beta=norm.bias.float().contiguous(), eps=float(norm.eps),
                     fc=pack_fc_tc(fc, p["H"]))
            e[axis] = p
        layers.append(e)
    return layers


class TcWorkspace:
    """Per-shape buffers of the tensor-core dual path (kept across calls: y must stay zero in its padding)."""

    def __init__(self, B, T, K, N, dev):
        self.key = (B, T, K, N, str(dev))
        M = B * T * K
        self.m_tiles = (M + 127) // 128
        self.tiles_time = (B * K + 127) // 128
        self.tiles_freq = (B * T + 127) // 128
        kc_in = (N + 15) // 16 * 2
        ntile = max(T * self.tiles_time, K * self.tiles_freq)     # (step, sequence tile) pairs of either axis
        self.xhat = torch.empty(ntile * kc_in * 128 * 8, dtype=torch.float16, device=dev)
        self.gates = torch.empty(ntile * 2 * CL * LGC * 128 * 8, dtype=torch.float16, device=dev)
        self.zero_tile = torch.zeros(LKC * 128 * 8, dtype=torch.float16, device=dev)
        self.y = torch.zeros(ntile * 2 * LKC * 128 * 8, dtype=torch.float16, device=dev)
        self.stats = torch.zeros(B, 2, dtype=torch.float64, device=dev)
        self.scale = torch.empty(B, N, dtype=torch.float32, device=dev)
        self.shift = torch.empty(B, N, dtype=torch.float32, device=dev)
        self.counts = _f64([float(T) * K * N], dev)
        self.sync = torch.zeros(max(L.lib().bsrnn_blstm_tc_sync_bytes(), L.lib().bsrnn_blstm_fused_sync_bytes()) // 4,
                                dtype=torch.int32, device=dev)
        self.nbytes = sum(t.numel() * t.element_size() for t in (self.xhat, self.gates, self.y))


_WS = {}                                 # insertion-ordered: least recently used first
WS_BUDGET_BYTES = int(os.environ.get("BSRNN_WS_BUDGET_GB", "64")) << 30


def workspace(B, T, K, N, dev):
    """Per-shape workspaces, least-recently-used eviction under a byte budget (config 2 needs ~25 GB for one shape; a
    mixed-sample-rate sweep alternates between many small ones and must not re-zero y on every batch)."""
    key = (B, T, K, N, str(dev))
    ws = _WS.pop(key, None)
    if ws is None:
        ws = TcWorkspace(B, T, K, N, dev)
        while _WS and sum(w.nbytes for w in _WS.values()) + ws.nbytes > WS_BUDGET_BYTES:
            _WS.pop(next(iter(_WS)))
    _WS[key] = ws
    return ws


_EXACT_STATS = os.environ.get("BSRNN_TC_EXACT_STATS", "0") == "1"


def dual_path_tc(skip, layers, t_emb=None, max_clusters=0, stats_ready=False, band_stats=None):
    """In-place 2*num_layer residual blocks on skip (B,T,K,N) f32, tensor-core mode.
    stats_ready: the per-sample sums of `skip` already sit in workspace(...).stats (written by band_split_tc's GEMM
    epilogues).  band_stats: (B,K,2) f64 zeros -- the last Linear + skip then accumulates per-(sample, band) sums of the
    final stream there (the statistics of the mask decoder's GroupNorms) instead of the per-sample ones nobody reads."""
    B, T, K, N = skip.shape
    dev = skip.device
    st = L.stream_ptr()
    ws = workspace(B, T, K, N, dev)
    keepalive(ws)
    M = B * T * K
    if not stats_ready:
        L.call("bsrnn_gn_stats", skip.data_ptr(), ws.stats.data_ptr(), B, T * K, N, N, st)
    for i, lay in enumerate(layers):
        for axis in ("time", "freq"):
            last = band_stats is not None and FC_EPI == L.TC_RESID_TMA and i == len(layers) - 1 and axis == "freq"
            w = lay[axis]
            extra = t_emb[i] if (t_emb is not None and axis == "time") else None
            if axis == "time":
                R, steps, tiles, addr = B * K, T, ws.tiles_time, (K, T * K, 1, K)
            else:
                R, steps, tiles, addr = B * T, K, ws.tiles_freq, (1, K, 0, 1)
            with region("norm"):
                L.call("bsrnn_gn_finalize", ws.stats.data_ptr(), w["gamma"].data_ptr(), w["beta"].data_ptr(), L.ptr(extra),
                       ws.scale.data_ptr(), ws.shift.data_ptr(), B, N, ws.counts.data_ptr(), w["eps"], 1, st)
                # operand tiles in the axis' (step, sequence tile) order: the GEMM output tiles are then the
                # recurrence kernel's gates_x tiles
                L.call("bsrnn_norm_cast_kb8_ones", skip.data_ptr(), ws.scale.data_ptr(), ws.shift.data_ptr(),
                       ws.xhat.data_ptr(), N, 0, N, w["kc_in"], steps * tiles, tiles, R, *addr, T * K, 1, w["one_col"], st)
            if axis in FUSED_AXES and "wfused" in w:
                # input projection inside the recurrence: gates_t = [x_t | h_{t-1}] [W_ih | W_hh]^T, no gates_x tensor
                with region(f"lstm_{axis}"):
                    geo = fused_geometry(tiles)
                    if geo in (7, 14):
                        L.call(f"bsrnn_blstm_fused{geo}_tc", ws.xhat.data_ptr(), fused_weights(w, geo).data_ptr(),
                               ws.zero_tile.data_ptr(), ws.y.data_ptr(), R, steps, tiles, max_clusters, _FUSED_SLOTS[axis],
                               ws.sync.data_ptr(), st)
                    else:
                        L.call("bsrnn_blstm_fused_tc", ws.xhat.data_ptr(), w["wfused"].data_ptr(), ws.zero_tile.data_ptr(),
                               ws.y.data_ptr(), R, steps, tiles, max_clusters, _FUSED_SLOTS[axis], ws.sync.data_ptr(), st)
            else:
                with region("inproj"):
                    L.call("bsrnn_gemm_tc", ws.xhat.data_ptr(), w["wih"].data_ptr(),
                           None if w["one_col"] >= 0 else w["bih"].data_ptr(), ws.gates.data_ptr(), None,
                           steps * tiles, 2 * CL, w["kc_in"], LBN, L.TC_F16_KB8, 0, 2 * CL * LBN, 2 * CL * LGC, T * K,
                           tiles, R, *addr, st)
                with region(f"lstm_{axis}"):
                    if LSTM_SCHED == "flag":
                        L.call("bsrnn_blstm_recurrence_tc_flag", ws.gates.data_ptr(), w["whh"].data_ptr(),
                               ws.zero_tile.data_ptr(), ws.y.data_ptr(), R, steps, tiles, max_clusters, _FLAG_SLOTS[axis],
                               ws.sync.data_ptr(), st)
                    else:
                        L.call("bsrnn_blstm_recurrence_tc_ex", ws.gates.data_ptr(), w["whh"].data_ptr(),
                               ws.zero_tile.data_ptr(), ws.y.data_ptr(), R, steps, tiles, max_clusters, _LSTM_SLOTS[axis], st)
            with region("fc"):
                ws.stats.zero_()
                fc = w["fc"]
                L.call("bsrnn_gemm_tc_ex", ws.y.data_ptr(), fc["w"].data_ptr(), fc["b"].data_ptr(), skip.data_ptr(),
                       band_stats.data_ptr() if last else ws.stats.data_ptr(), steps * tiles, 1, 2 * LKC, fc["BN"], FC_EPI,
                       N, N, 0, T * K, tiles, R, *addr, K if last else 1, 0, st)
                if _EXACT_STATS:                       # diagnosis: statistics from a separate pass over skip
                    ws.stats.zero_()
                    L.call("bsrnn_gn_stats", skip.data_ptr(), ws.stats.data_ptr(), B, T * K, N, N, st)
    return band_stats is not None and FC_EPI == L.TC_RESID_TMA          # True: band_stats holds the decoder statistics


# ------------------------------------------------------------------------------------------------ band split
BAND_SPLIT_TC = os.environ.get("BSRNN_BAND_SPLIT_TC", "1") == "1"      # 0: the f32 CUDA-core kernel (A/B, bandsplit.cu)


def pack_band_split_tc(bs):
    """BandSplit Conv1d(2 s_k -> N, 1) weights as fp16 KB8 tiles (one 208-row N tile per band, K padded to 16) + bias table;
    a_unit[k] = k-cores of band k's operand tile."""
    K = len(bs.subbands)
    N = bs.fc[0].weight.shape[0]
    dev = bs.fc[0].weight.device
    BN = (N + 15) // 16 * 16
    kcs = [((2 * s + 15) // 16) * 2 for s in bs.subbands]
    w = [to_kb8(bs.fc[k].weight[:, :, 0].float(), BN, kcs[k]).reshape(-1) for k in range(K)]
    w_off, tot = [], 0
    for k in range(K):
        w_off.append(tot)
        tot += w[k].numel()
    bias = torch.zeros(K, BN, device=dev)
    for k in range(K):
        bias[k, :N] = bs.fc[k].bias
    return dict(w=torch.cat(w).contiguous(), w_off=w_off, bias=bias, kcs=kcs, BN=BN, N=N)


def band_split_tc(spec, plan, bs_pack, bs_tc, N, stats):
    """spec (B,T,F,2) -> skip (B,T,K',N) f32 on tensor cores [reference bsrnn_flowse.py:65-86]: one operand-builder launch
    (per-band GroupNorm applied on the fly) + one store-only tcgen05 GEMM launch for all bands.  The GEMM epilogue also accumulates the
    per-sample sums of the result into workspace(...).stats: the first dual-path GroupNorm needs no pass of its own."""
    from .runtime import _i32, _const_table
    B, T, F, _ = spec.shape
    dev = spec.device
    K = plan.K
    cmax = bs_pack["cmax"]
    st = L.stream_ptr()
    ws = workspace(B, T, K, N, dev)
    keepalive(ws)
    counts = _f64([2.0 * plan.subbands[k] * T for k in range(K)], dev)      # padded bins count (bsrnn_flowse.py:68-73)
    scale = torch.empty(B * K, cmax, dtype=torch.float32, device=dev)
    shift = torch.empty_like(scale)
    L.call("bsrnn_gn_finalize", stats.data_ptr(), bs_pack["gamma"].data_ptr(), bs_pack["beta"].data_ptr(), None,
           scale.data_ptr(), shift.data_ptr(), B * K, cmax, counts.data_ptr(), bs_pack["eps"], K, st)
    tiles = (B * T + 127) // 128
    offs, tot = [], 0
    for k in range(K):
        offs.append(tot)
        tot += tiles * bs_tc["kcs"][k] * 1024
    a_off_d = _const_table(offs, torch.int64, dev)
    xhat = torch.empty(tot, dtype=torch.float16, device=dev)
    wid = _i32([2 * w for w in plan.width], dev)
    bin0 = _i32(list(plan.bin0), dev)
    L.call("bsrnn_band_norm_cast_kb8", spec.data_ptr(), scale.data_ptr(), shift.data_ptr(), xhat.data_ptr(),
           bs_pack["c_off"].data_ptr(), bin0.data_ptr(), wid.data_ptr(), a_off_d.data_ptr(), K, B * T, T, 2 * F, cmax, st)
    out = torch.empty(B, T, K, N, dtype=torch.float32, device=dev)
    ws.stats.zero_()
    # one launch for all bands, band innermost in the tile order: co-running CTAs write adjacent 4N-byte segments of the
    # same rows of the (B,T,K,N) stream
    desc = []
    for k in range(K):
        desc += [offs[k], bs_tc["w_off"][k], k * N, k * bs_tc["BN"], bs_tc["kcs"][k]]
    groups = _const_table(desc, torch.int64, dev)
    L.call("bsrnn_gemm_tc_grouped", xhat.data_ptr(), bs_tc["w"].data_ptr(), bs_tc["bias"].data_ptr(), out.data_ptr(),
           ws.stats.data_ptr(), groups.data_ptr(), K, tiles, max(bs_tc["kcs"][:K]), bs_tc["BN"], K * N, N, T, tiles,
           B * T, BIG, 0, 1, 0, st)
    return out


# ------------------------------------------------------------------------------------------------ mask decoder
def pack_mask_decoder_tc(md):
    """espnet2-style MaskDecoder for the tensor-core path: Conv1d(N,4N) as 208-column tiles, Conv1d(4N,4s) with rows
    interleaved (value, gate) so the GLU pairs sit in adjacent accumulator columns."""
    out = {}
    for name in ("mlp_mask", "mlp_residual"):
        mlps = getattr(md, name)
        N = mlps[0][1].weight.shape[1]
        kc1 = (N + 15) // 16 * 2
        H4 = 4 * N
        kc2 = (H4 + 15) // 16 * 2
        nt1 = (H4 + LBN - 1) // LBN
        w1, b1, w2, b2, bn2 = [], [], [], [], []
        # bias of Conv1d(N,4N) as weight column N against the operand's constant-one column (bsrnn_norm_cast_kb8_ones): the
        # GEMM then runs bias-free on the bulk-store tanh kernel (gemm_tc.cu, EPI_TANH_KB8 / BNC = 208).  Widths without a
        # padding column for it (N % 16 == 0, or N % 4 != 0) keep the bias vector and one normalised operand per family.
        one_col = N if (N % 4 == 0 and kc1 * 8 > N) else -1
        for k, m in enumerate(mlps):
            wk = m[1].weight[:, :, 0].float()
            if one_col >= 0:
                # W (z * gamma + beta) + b = (W diag(gamma)) z + (W beta + b): with the per-channel affine of this family's
                # GroupNorm folded in, BOTH families read one operand z = (x - mean) * rstd (one norm_cast, not two)
                bk = m[1].bias.float() + wk @ m[0].bias.float()
                wk = torch.cat([wk * m[0].weight.float()[None, :], bk[:, None]], 1)
            w1.append(to_kb8(wk, LBN, kc1))
            bb = torch.zeros(nt1 * LBN, device=m[1].bias.device); bb[:H4] = m[1].bias
            b1.append(bb)
            w = m[3].weight[:, :, 0].float()                     # (4s, 4N): first 2s rows = value, last 2s = gate
            half = w.shape[0] // 2
            order = torch.stack([torch.arange(half), torch.arange(half) + half], 1).reshape(-1).to(w.device)
            BN = (w.shape[0] + 15) // 16 * 16
            w2.append(to_kb8(w[order], BN, kc2))
            bb = torch.zeros(BN, device=w.device); bb[: w.shape[0]] = m[3].bias[order]
            b2.append(bb)
            bn2.append(BN)
        out[name] = dict(gamma=torch.stack([m[0].weight for m in mlps]).float().contiguous(),
                         beta=torch.stack([m[0].bias for m in mlps]).float().contiguous(),
                         w1=w1, b1=b1, w2=w2, b2=b2, bn2=bn2, kc1=kc1, kc2=kc2, nt1=nt1, N=N, one_col=one_col,
                         shared_norm=one_col >= 0,
                         eps=float(mlps[0][0].eps))
    return out


def mask_decoder_tc(skip, plan, md_pack, band_stats=None):
    """skip (B,T,K',N) -> mask, resid (B,T,F,2) f32, tensor-core mode.  band_stats: (B,K,2) per-(sample, band) sums of
    skip when the last Linear + skip already took them (dual_path_tc)."""
    from .runtime import _decoder_norm_tables
    B, T, K, N = skip.shape
    F = plan.F
    dev = skip.device
    st = L.stream_ptr()
    names = ("mlp_residual", "mlp_mask")
    shared = (all(md_pack[n]["shared_norm"] for n in names) and len({md_pack[n]["eps"] for n in names}) == 1
              and len({(md_pack[n]["kc1"], md_pack[n]["one_col"]) for n in names}) == 1)
    if shared:        # the affine halves live in the weights: one table of (rstd, -mean * rstd) per (sample, band)
        ones = _ones_pack(K, N, dev, md_pack[names[0]]["eps"])
        tabs = _decoder_norm_tables(skip, {"shared": ones}, stats=band_stats)
        tabs = {n: tabs["shared"] for n in names}
    else:
        tabs = _decoder_norm_tables(skip, md_pack, stats=band_stats)
    tiles = (B * T + 127) // 128
    outs = {}
    # The mask and the residual MLP families are independent chains of 2 x K small GEMMs: they run on two streams (two
    # parallel branches of a captured graph), so one chain's launch gaps and tile tails are filled by the other's.
    main = torch.cuda.current_stream()
    side = _side_stream(dev)
    fork = torch.cuda.Event()
    capturing = torch.cuda.is_current_stream_capturing()
    bufs = {}
    xshared = None
    for name in names:                                   # every buffer belongs to the main stream's allocator pool
        p = md_pack[name]
        if xshared is None or not shared:
            xshared = torch.empty(K * tiles * p["kc1"] * 1024, dtype=torch.float16, device=dev)
        bufs[name] = (xshared,
                      torch.empty(tiles * p["kc2"] * 1024, dtype=torch.float16, device=dev),
                      torch.empty(B, T, F, 2, dtype=torch.float32, device=dev))
    with region("maskdec"):
        if shared:
            p = md_pack[names[0]]
            scale, shift = tabs[names[0]][0], tabs[names[0]][1]
            L.call("bsrnn_norm_cast_kb8_ones", skip.data_ptr(), scale.data_ptr(), shift.data_ptr(), xshared.data_ptr(), N, 0, N,
                   p["kc1"], K * tiles, tiles, B * T, 1, K, 0, 1, T * K, K, p["one_col"], st)
        fork.record(main)
        side.wait_event(fork)
        for name, stream in (("mlp_residual", side), ("mlp_mask", main)):
            p = md_pack[name]
            scale, shift = tabs[name][0], tabs[name][1]
            xhat, hidden, o = bufs[name]
            with torch.cuda.stream(stream):
                st = L.stream_ptr()
                # rows of tile (k, j) are the (b,t) tokens of band k: same row map as the band-axis BLSTM
                if not shared:
                    L.call("bsrnn_norm_cast_kb8_ones", skip.data_ptr(), scale.data_ptr(), shift.data_ptr(), xhat.data_ptr(), N, 0,
                           N, p["kc1"], K * tiles, tiles, B * T, 1, K, 0, 1, T * K, K, p["one_col"], st)
                for k in range(K):
                    L.call("bsrnn_gemm_tc", xhat.data_ptr() + 2 * k * tiles * p["kc1"] * 1024, p["w1"][k].data_ptr(),
                           None if p["one_col"] >= 0 else p["b1"][k].data_ptr(), hidden.data_ptr(), None, tiles, p["nt1"],
                           p["kc1"], LBN, L.TC_TANH_KB8,
                           0, 4 * N, p["kc2"], B * T, tiles, B * T, BIG, 0, 1, 0, st)
                    L.call("bsrnn_gemm_tc", hidden.data_ptr(), p["w2"][k].data_ptr(), p["b2"][k].data_ptr(),
                           o.data_ptr() + 8 * plan.bin0[k], None, tiles, 1, p["kc2"], p["bn2"][k], L.TC_GLU_F32, 2 * F,
                           2 * plan.width[k], 0, B * T, tiles, B * T, BIG, 0, 1, 0, st)
            if stream is side and not capturing:
                for t in (xhat, hidden, o, skip, scale, shift):
                    t.record_stream(side)
            outs[name] = o
        main.wait_stream(side)
    return outs["mlp_mask"], outs["mlp_residual"]


_SIDE = {}
_ONES = {}


def _ones_pack(K, N, dev, eps):
    key = (K, N, str(dev), eps)
    t = _ONES.get(key)
    if t is None:
        t = _ONES[key] = dict(gamma=torch.ones(K, N, device=dev), beta=torch.zeros(K, N, device=dev), eps=eps)
    return t


def _side_stream(dev):
    key = str(dev)
    if key not in _SIDE:
        _SIDE[key] = torch.cuda.Stream(device=dev)
    return _SIDE[key]
