"""GPU tests (-m gpu) of the CUDA-core kernels -- bsrnn_gemm_f32 (csrc/gemm_f32.cu), bsrnn_blstm_recurrence_f32 /
_train_fwd_f32 / _train_bwd_f32 (csrc/lstm_f32.cu), bsrnn_band_split_fwd and bsrnn_band_norm_cast_kb8 (csrc/bandsplit.cu),
bsrnn_gn_stats / bsrnn_band_stats / bsrnn_gn_finalize (csrc/norm.cu), bsrnn_conv5x5_glu, bsrnn_time_embed, bsrnn_euler_step,
bsrnn_axpy_complex and bsrnn_complex_mask (csrc/flow.cu) -- each called through the C ABI against the plain f64 restatement
in tests/cuda_core_ref.py.

The bar is ELEMENTWISE, with bounds derived in cuda_core_ref's docstring from the operation order of each kernel (not
fitted); every case prints its worst err / bound and asserts it <= 1.  The BLSTM forward is checked step-locally (each step
from the kernel's own previous h and c), its backward against an f64 BPTT from the kernel's saved activations with a running
error bound.

Everything a kernel must not write -- a guard tail after every output, columns >= n_store, rows outside a descriptor's row
map, the neighbouring column segments of a wider row, the unused half of GLU tiles, W columns >= K, table entries of other
samples -- starts as a NaN bit pattern and must come back bit-identical (inputs the kernel must not read are NaN too, so a
stray read shows up as a NaN result).  Padding a kernel must write as zero (KB8 padding columns and rows, GradDecoder bins in
[F', F)) must be exactly 0.  One case per family corrupts the kernel's real output (a zeroed row tile, two swapped rows or
bands, one element 3x its bound off) and asserts that the checker rejects each.  The launcher branches are restated in
cuda_core_ref and the case lists are asserted to reach every one of them; the band-split launch runs also through
bsrnn_launch_count.
"""
import math

import numpy as np
import pytest
import torch

import cuda_core_ref as R
from oracle import restated as O

pytestmark = pytest.mark.gpu

GUARD = 1024
SENT32 = 0x7F8DEAD1
SENT64 = 0x7FF4DEADBEEF0001
SENT16 = 0x7E5B
DEV = "cuda"


def _lib():
    from urgent2026_challenge_track1_b200 import _lib as L
    L.require_device()
    return L


# ------------------------------------------------------------------------------------------------------------ machinery
def sentinel(n, dtype=torch.float32):
    if dtype == torch.float64:
        return torch.full((n + GUARD,), SENT64, dtype=torch.int64, device=DEV).view(torch.float64)
    if dtype == torch.float16:
        return torch.full((n + GUARD,), SENT16, dtype=torch.int16, device=DEV).view(torch.float16)
    return torch.full((n + GUARD,), SENT32, dtype=torch.int32, device=DEV).view(torch.float32)


def bits(t):
    return t.view({torch.float64: torch.int64, torch.float32: torch.int32, torch.float16: torch.int16}[t.dtype])


def guard_ok(buf, n, name):
    assert torch.equal(bits(buf[n:]), bits(sentinel(0, buf.dtype)[:buf.numel() - n])), f"{name}: guard tail written"


def untouched_ok(after, before, written_idx, name):
    """Every element outside the flat indices written_idx is bit-identical to its initial state."""
    keep = torch.ones(after.numel(), dtype=torch.bool, device=DEV)
    keep[written_idx.reshape(-1)] = False
    assert torch.equal(bits(after)[keep], bits(before)[keep]), f"{name}: wrote outside its output"


def worst_ratio(got, ref, bound):
    err = (got.double() - ref).abs()
    ratio = torch.where(bound > 0, err / bound.clamp(min=1e-300), torch.where(err > 0, math.inf, 0.0))
    return float(torch.nan_to_num(ratio, nan=math.inf).max()) if ratio.numel() else 0.0


def assert_within(name, got, ref, bound):
    w = worst_ratio(got, ref, bound)
    print(f"{name}: worst err/bound = {w:.3g}")
    assert w <= 1.0, f"{name}: worst err/bound {w:.3g}"
    return w


def assert_checker_is_sharp(name, got, ref, bound, tile=64):
    """Corrupt a correct (rows, cols) result three ways; the elementwise check must reject each."""
    assert got.shape[0] >= 2
    bad = got.clone()
    bad[:tile] = 0.0                                                      # one row tile zeroed
    assert worst_ratio(bad, ref, bound) > 1.0, f"{name}: a zeroed row tile passes"
    bad = got.clone()
    bad[[0, 1]] = bad[[1, 0]]                                             # two rows (bands, steps) swapped
    assert worst_ratio(bad, ref, bound) > 1.0, f"{name}: swapped rows pass"
    bad = got.double().contiguous().clone()
    k = int(bound.reshape(-1).argmax())
    bad.view(-1)[k] = ref.reshape(-1)[k] + 3.0 * bound.reshape(-1)[k]    # one element 3x its bound off
    assert worst_ratio(bad, ref, bound) > 1.0, f"{name}: a 3x-bound error passes"


def rnd(*shape, scale=1.0, offset=0.0, seed=0):
    g = torch.Generator(device=DEV).manual_seed(seed)
    return torch.randn(*shape, generator=g, device=DEV) * scale + offset


# ------------------------------------------------------------------------------------------------------------ gemm_f32
def _gemm_group(M, N, K, epilogue=0, k_valid=None, n_store=None, scaled=False, rows_per_sample=None, ss_extra=0,
                a_map=None, c_map=None, ldw_extra=0, bias=True):
    """Geometry of one synthetic group.  a_map / c_map: (inner, outer_stride, inner_stride) of a two-level row map; default
    dense rows of K (A) and of the output width plus 3 (C)."""
    n_out = N // 2 if epilogue == 3 else N
    return dict(M=M, N=N, K=K, epilogue=epilogue, k_valid=K if k_valid is None else k_valid,
                n_store=n_out if n_store is None else n_store, scaled=scaled,
                rows_per_sample=rows_per_sample or M, ss_stride=K + ss_extra,
                a_map=a_map or (1 << 60, 0, K + 1), c_map=c_map or (1 << 60, 0, n_out + 3), ldw=K + ldw_extra, bias=bias)


def _from_rows_desc(d, scaled, bias=True):
    """A group with the geometry of a descriptor built by runtime._rows_desc (pointers are replaced by the harness)."""
    return dict(M=d["M"], N=d["N"], K=d["K"], epilogue=d["epilogue"], k_valid=d["k_valid"], n_store=d["n_store"],
                scaled=scaled, rows_per_sample=d["rows_per_sample"], ss_stride=max(d["ss_stride"], d["K"]),
                a_map=(d["a_inner"], d["a_outer_stride"], d["a_inner_stride"]),
                c_map=(d["c_inner"], d["c_outer_stride"], d["c_inner_stride"]), ldw=d["ldw"], bias=bias)


def _row_offsets(M, mp):
    r = torch.arange(M, device=DEV, dtype=torch.long)
    return (r // mp[0]) * mp[1] + (r % mp[0]) * mp[2]


def run_gemm(name, groups, max_n=None, seed=0, sharp=False):
    """Build every group's buffers, run them in ONE bsrnn_gemm_f32 launch, check each group elementwise and everything
    around its output bit-identical."""
    L = _lib()
    from urgent2026_challenge_track1_b200 import runtime
    recs, state = [], []
    for gi, g in enumerate(groups):
        M, N, K = g["M"], g["N"], g["K"]
        n_out = N // 2 if g["epilogue"] == 3 else N
        ao, co = _row_offsets(M, g["a_map"]), _row_offsets(M, g["c_map"])
        A = rnd(int(ao.max()) + K + GUARD, seed=seed * 100 + gi)
        W = sentinel(N * g["ldw"])
        W[:N * g["ldw"]].view(N, g["ldw"])[:, :K] = rnd(N, K, scale=1 / math.sqrt(K), seed=seed * 100 + gi + 50)
        b = rnd(N, scale=0.5, seed=seed * 100 + gi + 60) if g["bias"] else None
        n_smp = -(-M // g["rows_per_sample"])
        sc = sh = None
        if g["scaled"]:
            sc, sh = sentinel(n_smp * g["ss_stride"]), sentinel(n_smp * g["ss_stride"])
            sc[:n_smp * g["ss_stride"]].view(n_smp, -1)[:, :K] = rnd(n_smp, K, scale=0.3, offset=1.0, seed=seed + 7 * gi)
            sh[:n_smp * g["ss_stride"]].view(n_smp, -1)[:, :K] = rnd(n_smp, K, scale=0.5, seed=seed + 7 * gi + 3)
        cw = min(n_out, g["n_store"])
        widx = co[:, None] + torch.arange(cw, device=DEV)[None, :]
        C = sentinel(int(co.max()) + n_out + 8)
        if g["epilogue"] == 2:
            C[widx] = rnd(M, cw, seed=seed + 11 * gi)
        C0 = C.clone()
        recs.append(runtime._rows_desc(A.data_ptr(), W.data_ptr(), L.ptr(b), C.data_ptr(), M, N, K, a_stride=0, c_stride=0,
                                       k_valid=g["k_valid"], ldw=g["ldw"], epilogue=g["epilogue"], n_store=g["n_store"],
                                       scale=L.ptr(sc), shift=L.ptr(sh), rows_per_sample=g["rows_per_sample"],
                                       ss_stride=g["ss_stride"]))
        recs[-1].update(a_inner=g["a_map"][0], a_outer_stride=g["a_map"][1], a_inner_stride=g["a_map"][2],
                        c_inner=g["c_map"][0], c_outer_stride=g["c_map"][1], c_inner_stride=g["c_map"][2])
        state.append((g, A, W, b, sc, sh, C, C0, ao, widx, n_out, cw))
    arr = np.zeros(len(recs), dtype=L.GEMM_DESC)
    for i, r in enumerate(recs):
        for k, v in r.items():
            arr[i][k] = v if v is not None else 0
    descs = torch.from_numpy(np.frombuffer(arr.tobytes(), dtype=np.uint8).copy()).to(DEV)
    max_m = max(g["M"] for g in groups)
    max_n = max_n or max(s[10] for s in state)
    L.call("bsrnn_gemm_f32", descs.data_ptr(), len(groups), max_m, max_n, L.stream_ptr())
    torch.cuda.synchronize()
    worst, tallest = 0.0, max(range(len(groups)), key=lambda i: groups[i]["M"])
    for gi, (g, A, W, b, sc, sh, C, C0, ao, widx, n_out, cw) in enumerate(state):
        M, N, K = g["M"], g["N"], g["K"]
        Ag = A[ao[:, None] + torch.arange(K, device=DEV)[None, :]]
        Wg = W[:N * g["ldw"]].view(N, g["ldw"])[:, :K]
        scg = shg = None
        if sc is not None:
            s = torch.arange(M, device=DEV) // g["rows_per_sample"]
            scg = sc[:-GUARD].view(-1, g["ss_stride"])[s, :K]
            shg = sh[:-GUARD].view(-1, g["ss_stride"])[s, :K]
        ref, bound = R.gemm_f32_ref(Ag, Wg, b, scg, shg, g["k_valid"], g["epilogue"], C0[widx] if g["epilogue"] == 2 else None)
        got = C[widx]
        tag = f"{name}[{gi}] M={M} N={N} K={K} epi={g['epilogue']}"
        worst = max(worst, assert_within(tag, got, ref[:, :cw], bound[:, :cw]))
        untouched_ok(C, C0, widx, tag)
        if sharp and gi == tallest:
            assert_checker_is_sharp(tag, got, ref[:, :cw], bound[:, :cw])
    return worst


GEMM_CASES = {
    # every epilogue, each with M / N / K edges; several groups of different extents share one launch (early exits)
    "epilogues_mixed": [
        _gemm_group(1, 1, 1),
        _gemm_group(63, 4, 15, epilogue=1),
        _gemm_group(65, 33, 17, epilogue=2),
        _gemm_group(1000, 196, 196, epilogue=3, scaled=True, rows_per_sample=250, ss_extra=5),
        _gemm_group(64, 784, 784, epilogue=0, ldw_extra=3),
    ],
    "sizes_M1_K784": [_gemm_group(1, 784, 784, epilogue=1), _gemm_group(1037, 1, 1, epilogue=2)],
    "k_valid_scaled": [_gemm_group(130, 196, 17, k_valid=9, scaled=True, rows_per_sample=40, ss_extra=2),
                       _gemm_group(70, 33, 15, k_valid=1, epilogue=1)],
    "k_valid_unscaled": [_gemm_group(65, 4, 196, k_valid=150, epilogue=2)],
    # per-sample scale rows: a sample boundary inside each 64-row tile; ss_stride != C
    "per_sample_scale": [_gemm_group(300, 64, 40, scaled=True, rows_per_sample=7, ss_extra=11, epilogue=1)],
    # two-level row maps on A and C (token-major sequences of a (B, T, K) tensor along the time axis)
    "two_level_rows": [_gemm_group(3 * 5 * 29, 33, 20, a_map=(29, 5 * 29 * 21, 21), c_map=(29, 5 * 29 * 40, 40),
                                   scaled=True, rows_per_sample=5 * 29, epilogue=0)],
    # GLU with N/2 not a multiple of 32 and n_store < N/2
    "glu_edges": [_gemm_group(129, 2 * 45, 33, epilogue=3, n_store=41), _gemm_group(64, 2 * 1, 4, epilogue=3),
                  _gemm_group(65, 2 * 120, 196, epilogue=3, n_store=118, bias=False)],
    # the residual epilogue in place on a wide row (C's neighbouring columns are another layer's)
    "residual_in_place": [_gemm_group(200, 196, 784, epilogue=2, c_map=(1 << 60, 0, 3 * 196))],
}


def _real_groups():
    """Descriptors with the geometry runtime.py builds (same runtime._rows_desc calls, small B, T)."""
    from urgent2026_challenge_track1_b200 import runtime
    dsc = runtime._rows_desc
    B, T = 2, 9
    out = {}
    # band_split_f32 GEMM fallback (FlowSE table at N = 384 does not fit the band-split kernel); bands 0, 36 and the last
    # truncated band of a 44.1 kHz spectrum (F = 1411 // 2 + 1 = 706 bins of the 769-bin table)
    plan = runtime.BandPlan.make(runtime.SUBBANDS[769], 706)
    N, K, cmax, Fb = 384, plan.K, 2 * max(plan.subbands), plan.F
    grp = []
    for k in (0, 36, plan.K - 1):
        s = plan.subbands[k]
        d = dsc(0, 0, 0, 0, B * T, N, 2 * s, a_stride=2 * Fb, c_stride=K * N, k_valid=2 * plan.width[k],
                scale=1, shift=1, rows_per_sample=T, ss_stride=K * cmax)
        grp.append(_from_rows_desc(d, True))
    assert grp[-1]["k_valid"] < grp[-1]["K"]
    out["band_split_f32_fallback"] = (grp, N)
    # dual_path_f32 at N = 196, H = 392: input projection 8H = 3136 columns (scaled), Linear 2H -> N with residual
    N, H, K = 196, 392, 34
    M = B * T * K
    out["dual_path_inproj"] = ([_from_rows_desc(dsc(0, 0, 0, 0, M, 8 * H, N, a_stride=N, c_stride=8 * H, scale=1, shift=1,
                                                    rows_per_sample=T * K, ss_stride=N), True)], 8 * H)
    out["dual_path_fc"] = ([_from_rows_desc(dsc(0, 0, 0, 0, M, N, 2 * H, a_stride=2 * H, c_stride=N, epilogue=2), False)], N)
    # mask_decoder_f32 (SE table, 16 kHz: 161 bins, last band truncated): tanh MLP N -> 4N, GLU 4N -> 4 s with n_store
    plan = runtime.BandPlan.make(runtime.SUBBANDS[481], 161)
    K, Fb = plan.K, plan.F
    g1, g2 = [], []
    for k in (0, K - 1):
        s = plan.subbands[k]
        g1.append(_from_rows_desc(dsc(0, 0, 0, 0, B * T, 4 * N, N, a_stride=K * N, c_stride=4 * N, epilogue=1, scale=1,
                                      shift=1, rows_per_sample=T, ss_stride=K * N), True))
        g2.append(_from_rows_desc(dsc(0, 0, 0, 0, B * T, 4 * s, 4 * N, a_stride=4 * N, c_stride=2 * Fb, epilogue=3,
                                      n_store=2 * plan.width[k]), False))
    assert g2[-1]["n_store"] < g2[-1]["N"] // 2
    out["mask_decoder_mlp1"] = (g1, 4 * N)
    out["mask_decoder_mlp2"] = (g2, 2 * max(plan.subbands[:K]))
    # grad_decoder_f32: tanh MLP N -> 16 s into the channel-last (B, T, F', 16) image
    plan = runtime.BandPlan.make(runtime.SUBBANDS[769], 769)
    Fp = sum(plan.subbands[:plan.K])
    out["grad_decoder_mlp"] = ([_from_rows_desc(dsc(0, 0, 0, 0, B * T, 16 * s, N, a_stride=plan.K * N,
                                                    c_stride=Fp * 16, epilogue=1, scale=1, shift=1, rows_per_sample=T,
                                                    ss_stride=plan.K * N), True) for s in (5, 60)], 16 * 60)
    # FlowSE condition_fc: Linear(2N -> N) over the concatenated band-split outputs, N = 196 and 384
    for n in (196, 384):
        out[f"condition_fc_{n}"] = ([_from_rows_desc(dsc(0, 0, 0, 0, B * T * 48, n, 2 * n, a_stride=2 * n, c_stride=n), False)],
                                    n)
    return out


@pytest.mark.parametrize("case", sorted(GEMM_CASES))
def test_gemm_f32_synthetic(case):
    run_gemm(case, GEMM_CASES[case], seed=len(case), sharp=case == "epilogues_mixed")


def test_gemm_f32_runtime_descriptors():
    for name, (groups, max_n) in _real_groups().items():
        run_gemm(name, groups, max_n=max_n, seed=len(name), sharp=name == "mask_decoder_mlp2")


def test_gemm_f32_cases_reach_every_branch():
    reached = set()
    for groups in GEMM_CASES.values():
        max_m = max(g["M"] for g in groups)
        max_n = max(g["N"] // 2 if g["epilogue"] == 3 else g["N"] for g in groups)
        for g in groups:
            reached |= R.gemm_branches(g["M"], g["N"], g["K"], g["k_valid"], g["epilogue"], g["n_store"], g["scaled"],
                                       max_m, max_n)
    print("gemm_f32 branches reached:", sorted(reached))
    assert reached == R.GEMM_BRANCHES, R.GEMM_BRANCHES - reached
    for groups, max_n in _real_groups().values():                            # the runtime's max_n covers its groups
        for g in groups:
            R.gemm_branches(g["M"], g["N"], g["K"], g["k_valid"], g["epilogue"], g["n_store"], g["scaled"],
                            max(x["M"] for x in groups), max_n)


# ------------------------------------------------------------------------------------------------------------ lstm_f32
def _lstm_geometry(R_, steps, axis):
    """(B, T, K, addr) of a token-major tensor whose `axis` sequences are R_ sequences of `steps` steps."""
    inner = 100 if R_ % 100 == 0 and R_ > 100 else R_
    B = R_ // inner
    if axis == "time":
        T, K = steps, inner
        return B, T, K, (K, T * K, 1, K)
    T, K = inner, steps
    return B, T, K, (1, K, 0, 1)


def run_lstm(R_, steps, H, axis, seed=0, backward=True, check_fwd=True, sharp=False):
    L = _lib()
    B, T, K, addr = _lstm_geometry(R_, steps, axis)
    tokens = B * T * K
    tag = f"lstm_f32 {axis} R={R_} steps={steps} H={H}"
    gx = rnd(tokens, 2, 4 * H, scale=1.0, seed=seed)
    whh = rnd(2, 4 * H, H, scale=1.5 / math.sqrt(H), seed=seed + 1)
    y, c_st, saved = sentinel(tokens * 2 * H), sentinel(2 * R_ * H), sentinel(tokens * 10 * H)
    st = L.stream_ptr()
    L.call("bsrnn_blstm_train_fwd_f32", gx.data_ptr(), whh.data_ptr(), y.data_ptr(), c_st.data_ptr(), saved.data_ptr(), R_,
           steps, H, *addr, st)
    y2, c2 = sentinel(tokens * 2 * H), sentinel(2 * R_ * H)
    L.call("bsrnn_blstm_recurrence_f32", gx.data_ptr(), whh.data_ptr(), y2.data_ptr(), c2.data_ptr(), R_, steps, H, *addr, st)
    torch.cuda.synchronize()
    for buf, n, what in ((y, tokens * 2 * H, "y"), (c_st, 2 * R_ * H, "c_state"), (saved, tokens * 10 * H, "saved"),
                         (y2, tokens * 2 * H, "y (recurrence)")):
        guard_ok(buf, n, f"{tag} {what}")
    assert torch.equal(bits(y2), bits(y)), f"{tag}: recurrence_f32 y differs from train_fwd_f32 y"
    assert torch.equal(bits(c2), bits(c_st)), f"{tag}: recurrence_f32 c_state differs"
    tok = R.seq_tokens(R_, steps, *addr).to(DEV)                             # (R, S)
    yv = y[:-GUARD].view(tokens, 2, H)
    sv = saved[:-GUARD].view(tokens, 2, 5, H)
    cv = c_st[:-GUARD].view(2, R_, H)
    assert torch.equal(bits(cv[0]), bits(sv[tok[:, -1], 0, 4])), f"{tag}: final c (fwd) is not the last saved c"
    assert torch.equal(bits(cv[1]), bits(sv[tok[:, 0], 1, 4])), f"{tag}: final c (bwd) is not the last saved c"
    if check_fwd:
        for d in range(2):
            # all steps at once, each from the kernel's own previous state; step 0 of the direction from zeros
            s = torch.arange(steps, device=DEV)
            sp = s - 1 if d == 0 else s + 1
            first = (sp < 0) | (sp >= steps)
            spc = sp.clamp(0, steps - 1)
            t_cur, t_prev = tok[:, s].reshape(-1), tok[:, spc].reshape(-1)
            hp = torch.where(first.repeat(R_)[:, None], 0.0, yv[t_prev, d])
            cp = torch.where(first.repeat(R_)[:, None], 0.0, sv[t_prev, d, 4])
            ref = R.lstm_step_ref(gx[t_cur, d], whh[d], hp, cp)
            for j, k in enumerate("ifgoc"):
                assert_within(f"{tag} d={d} {k}", sv[t_cur, d, j], *ref[k])
            assert_within(f"{tag} d={d} h", yv[t_cur, d], *ref["h"])
            if sharp and d == 0 and R_ >= 2:
                assert_checker_is_sharp(tag + " h", yv[t_cur, d], *ref["h"], tile=min(64, R_ * steps))
    if not backward:
        return
    dy = rnd(tokens, 2 * H, seed=seed + 2)
    dg = sentinel(tokens * 8 * H)
    dh_rec, dc_carry = torch.empty(2 * R_ * H, device=DEV), torch.empty(2 * R_ * H, device=DEV)
    L.call("bsrnn_blstm_train_bwd_f32", dy.data_ptr(), saved.data_ptr(), whh.data_ptr(), dg.data_ptr(), dh_rec.data_ptr(),
           dc_carry.data_ptr(), R_, steps, H, *addr, st)
    torch.cuda.synchronize()
    guard_ok(dg, tokens * 8 * H, f"{tag} dgates")
    sv_sm = sv[tok].permute(2, 0, 1, 3, 4)                                   # (2, R, S, 5, H)
    dy_sm = dy.view(tokens, 2, H)[tok].permute(2, 0, 1, 3)                   # (2, R, S, H)
    ref, bound = R.lstm_bwd_ref(sv_sm, dy_sm, whh)
    got = dg[:-GUARD].view(tokens, 2, 4 * H)[tok].permute(2, 0, 1, 3)
    assert_within(f"{tag} dgates", got.reshape(-1, 4 * H), ref.reshape(-1, 4 * H), bound.reshape(-1, 4 * H))
    if sharp:
        assert_checker_is_sharp(tag + " dgates", got.reshape(-1, 4 * H), ref.reshape(-1, 4 * H), bound.reshape(-1, 4 * H))


LSTM_SMALL = [(R_, steps, H, axis) for H in (8, 24) for R_ in (1, 63, 64, 65, 300) for steps in (1, 2, 33)
              for axis in ("time", "band")]
LSTM_WIDE = [(65, 33, 392, "time"), (300, 2, 392, "band"), (1, 33, 392, "band"), (64, 1, 392, "time"),
             (65, 2, 768, "time"), (300, 33, 768, "band"), (63, 33, 768, "time")]


@pytest.mark.parametrize("H", [8, 24])
def test_blstm_f32_small_widths(H):
    for i, (R_, steps, h, axis) in enumerate(c for c in LSTM_SMALL if c[2] == H):
        run_lstm(R_, steps, h, axis, seed=i, sharp=(R_, steps, axis) == (65, 33, "time"))


@pytest.mark.parametrize("case", LSTM_WIDE, ids=[f"{a}-R{r}-S{s}-H{h}" for r, s, h, a in LSTM_WIDE])
def test_blstm_f32_model_widths(case):
    R_, steps, H, axis = case
    run_lstm(R_, steps, H, axis, seed=H + R_)


def test_blstm_f32_backward_beyond_grid_y_limit():
    """R = B T > 65535 sequences on the band axis: the backward gates kernel loops over rows past grid.y's limit."""
    run_lstm(70001, 2, 8, "band", seed=5)


def test_blstm_f32_cases_reach_every_branch():
    cases = LSTM_SMALL + LSTM_WIDE + [(70001, 2, 8, "band")]
    row_tiles = {R.lstm_grids(r, h)[0][1] for r, s, h, a in cases}
    assert {1, 2, 5} <= row_tiles                                  # one tile, a partial second tile, several tiles
    assert any(h % 16 for _, _, h, _ in cases) and any(h % 16 == 0 for _, _, h, _ in cases)   # partial unit tile
    assert {1, 2, 33} <= {s for _, s, _, _ in cases} and {"time", "band"} == {a for *_, a in cases}
    assert any(R.lstm_grids(r, h)[1][1] < r for r, s, h, a in cases)      # gates kernel loops over rows
    assert any(R.lstm_grids(r, h)[1][0] > 1 for r, s, h, a in cases)      # H > 256: two unit blocks in the gates kernel


# ------------------------------------------------------------------------------------------------------------ BandSplit
def _band_table(subbands, F_bins):
    from urgent2026_challenge_track1_b200 import runtime
    plan = runtime.BandPlan.make(tuple(subbands), F_bins)
    c_off = [0]
    for s in plan.subbands[:plan.K]:
        c_off.append(c_off[-1] + 2 * s)
    return plan.K, list(plan.bin0), [2 * w for w in plan.width], c_off


def run_band_split(name, subbands, F_bins, N, B, T, out_width=None, out_col=0, seed=0, sharp=False, cast=True):
    L = _lib()
    K, bin0, width2, c_off = _band_table(subbands, F_bins)
    cmax = max(c_off[k + 1] - c_off[k] for k in range(K)) + 4
    rows = B * T
    F2 = 2 * F_bins
    spec = rnd(rows, F2, scale=2.0, offset=0.3, seed=seed)
    scale = rnd(B * K, cmax, scale=0.3, offset=1.0, seed=seed + 1)
    shift = rnd(B * K, cmax, scale=0.5, seed=seed + 2)
    wT = rnd(c_off[-1], N, scale=0.2, seed=seed + 3)
    bias = rnd(K, N, scale=0.5, seed=seed + 4)
    out_width = out_width or N
    ldo = K * out_width
    out = sentinel(rows * ldo)
    out0 = out.clone()
    dc_off = torch.tensor(c_off, dtype=torch.int32, device=DEV)
    dbin0 = torch.tensor(bin0, dtype=torch.int32, device=DEV)
    dwid = torch.tensor(width2, dtype=torch.int32, device=DEV)
    c_off_host = np.array(c_off, dtype=np.int32)
    L.lib().bsrnn_launch_count(1)
    L.call("bsrnn_band_split_fwd", spec.data_ptr(), scale.data_ptr(), shift.data_ptr(), wT.data_ptr(), bias.data_ptr(),
           out.data_ptr(), dc_off.data_ptr(), dbin0.data_ptr(), dwid.data_ptr(), c_off_host.ctypes.data, K, rows, T, F2, N,
           cmax, ldo, out_width, out_col, L.stream_ptr())
    launches = L.lib().bsrnn_launch_count(1)
    torch.cuda.synchronize()
    runs = R.band_split_runs(c_off, N)
    assert launches == len(runs), (launches, runs)
    refs = R.band_split_ref(spec, T, scale, shift, wT, bias, c_off, bin0, width2, cmax, N)
    r_idx = torch.arange(rows, device=DEV)[:, None] * ldo
    widx, got_all, ref_all, bnd_all = [], [], [], []
    for k, (ref, bound) in enumerate(refs):
        idx = r_idx + k * out_width + out_col + torch.arange(N, device=DEV)[None, :]
        widx.append(idx)
        got_all.append(out[idx])
        ref_all.append(ref)
        bnd_all.append(bound)
    got, ref, bound = torch.stack(got_all), torch.stack(ref_all), torch.stack(bnd_all)      # (K, rows, N)
    tag = f"band_split {name} K={K} N={N} rows={rows} runs={len(runs)}"
    assert_within(tag, got, ref, bound)
    untouched_ok(out, out0, torch.stack(widx), tag)
    if sharp:                                                                # bands swapped / a row tile / one element
        assert_checker_is_sharp(tag, got, ref, bound, tile=1)
        assert_checker_is_sharp(tag + " rows", got[0], ref[0], bound[0], tile=min(128, rows))
    if cast:
        run_band_cast(name, spec, T, scale, shift, c_off, bin0, width2, cmax, dc_off, dbin0, dwid, sharp)
    return len(runs)


def run_band_cast(name, spec, T, scale, shift, c_off, bin0, width2, cmax, dc_off, dbin0, dwid, sharp):
    """bsrnn_band_norm_cast_kb8 on the same operands: per-band a_off with a gap of 512 halves between bands."""
    L = _lib()
    rows, F2 = spec.shape
    K = len(c_off) - 1
    a_off, pos, ext = [], 512, []
    for k in range(K):
        kc, tiles, n = R.kb8_geometry(c_off[k + 1] - c_off[k], rows)
        a_off.append(pos)
        ext.append((kc, tiles, n))
        pos += n + 512
    out = sentinel(pos, torch.float16)
    out0 = out.clone()
    da = torch.tensor(a_off, dtype=torch.int64, device=DEV)
    L.call("bsrnn_band_norm_cast_kb8", spec.data_ptr(), scale.data_ptr(), shift.data_ptr(), out.data_ptr(), dc_off.data_ptr(),
           dbin0.data_ptr(), dwid.data_ptr(), da.data_ptr(), K, rows, T, F2, cmax, L.stream_ptr())
    torch.cuda.synchronize()
    widx, worst = [], 0.0
    for k in range(K):
        kc, tiles, n = ext[k]
        C = c_off[k + 1] - c_off[k]
        idx = torch.arange(a_off[k], a_off[k] + n, device=DEV)
        widx.append(idx)
        m = out[idx].view(tiles, kc, 128, 8).permute(0, 2, 1, 3).reshape(tiles * 128, kc * 8).double()
        ref, bound = R.band_cast_ref(spec, T, scale, shift, c_off, bin0, width2, cmax, k)
        tag = f"band_norm_cast_kb8 {name} band {k}"
        assert bool((m[:, C:] == 0).all()) and bool((m[rows:] == 0).all()), f"{tag}: padding is not exactly 0"
        w = worst_ratio(m[:rows, :C], ref, bound)
        worst = max(worst, w)
        assert w <= 1.0, f"{tag}: worst err/bound {w:.3g}"
        if sharp and k == K - 1 and rows >= 2:
            assert_checker_is_sharp(tag, m[:rows, :C], ref, bound, tile=min(64, rows))
    print(f"band_norm_cast_kb8 {name}: worst err/bound = {worst:.6f}")     # ~1 - 2^-13 near fp16 midpoints
    untouched_ok(out, out0, torch.cat(widx), f"band_norm_cast_kb8 {name}")


SE_RATES = {16000: 161, 22050: 221, 44100: 442, 48000: 481}
# synthetic tables: the shared-memory class changes along the bands (several runs), a band at N = 384 within 3 KB of the
# 227 KB limit, and a truncated last band
SYNTH_TABLES = {
    "classes_5_runs": ((4, 16, 4, 2, 2, 80, 3), 110, 196),
    "near_limit_384": ((2, 56, 8), 60, 384),
    "n4": ((3, 5, 60, 1), 66, 4),
}


@pytest.mark.parametrize("fs", sorted(SE_RATES))
def test_band_split_se_tables(fs):
    run_band_split(f"SE {fs}", runtime_subbands(481), SE_RATES[fs], 196, 2, 67, seed=fs % 97, sharp=fs == 16000)


def runtime_subbands(n):
    from urgent2026_challenge_track1_b200 import runtime
    return runtime.SUBBANDS[n]


def test_band_split_flowse_table():
    """The FlowSE table at its own FFT size (1536 -> 769 bins), into columns [N, 2N) of a (B, T, K, 2N) row (the
    band_split_x / band_split_y pair condition_fc reads)."""
    run_band_split("FlowSE", runtime_subbands(769), 769, 196, 1, 130, out_width=392, out_col=196, seed=3)


@pytest.mark.parametrize("case", sorted(SYNTH_TABLES))
def test_band_split_synthetic_tables(case):
    sub, F_bins, N = SYNTH_TABLES[case]
    run_band_split(case, sub, F_bins, N, 3, 45, out_width=N + 8, out_col=4, seed=len(case))


def test_band_split_cases_reach_every_branch():
    counts = set()
    for sub, F_bins, N in SYNTH_TABLES.values():
        _, _, _, c_off = _band_table(sub, F_bins)
        counts.add(len(R.band_split_runs(c_off, N)))
        assert R.band_split_fits(c_off, N)
    _, _, w2, c_off = _band_table(runtime_subbands(481), 161)
    assert w2[-1] < c_off[-1] - c_off[-2]                                       # truncated last band at 16 kHz
    assert max(counts) >= 4 and len(counts) >= 2, counts
    _, _, _, c_off = _band_table(*SYNTH_TABLES["near_limit_384"][:2])
    assert max(R.band_split_smem(c_off[k + 1] - c_off[k], 384) for k in range(len(c_off) - 1)) > R.SMEM_LIMIT - 4096
    assert {196 // 4 % 32, 384 // 4 % 32} == {17, 0}                            # N = 196: second pass has 17 active lanes


# ------------------------------------------------------------------------------------------------------------ GroupNorm
def run_gn_stats(B, rows, C, row_stride, dc=0.0, std=1.0, seed=0):
    L = _lib()
    x = sentinel(B * rows * row_stride)
    x[:B * rows * row_stride].view(B, rows, row_stride)[:, :, :C] = rnd(B, rows, C, scale=std, offset=dc, seed=seed)
    stats = sentinel(2 * B, torch.float64)
    L.call("bsrnn_gn_stats", x.data_ptr(), stats.data_ptr(), B, rows, C, row_stride, L.stream_ptr())
    torch.cuda.synchronize()
    guard_ok(stats, 2 * B, "gn_stats")
    geo = R.gn_stats_geometry(B, rows, C, row_stride)
    xs = x[:B * rows * row_stride].view(B, rows, row_stride)[:, :, :C].reshape(B, -1)
    s, q, bs, bq = R.sums_ref(xs, geo["m"])
    tag = f"gn_stats B={B} rows={rows} C={C} stride={row_stride} dc={dc} m={geo['m']}"
    got = stats[:2 * B].view(B, 2)
    assert_within(tag + " sum", got[:, 0], s, bs)
    assert_within(tag + " sumsq", got[:, 1], q, bq)
    return geo


GN_CASES = [(B, rows, C, stride, dc) for (B, rows) in ((1, 3000), (3, 400), (64, 50), (1200, 100), (3, 2))
            for (C, stride) in ((1, 1), (196, 196), (300, 300), (196, 200), (300, 320), (1, 5))
            for dc in (0.0, 1000.0)]


@pytest.mark.parametrize("B", sorted({c[0] for c in GN_CASES}))
def test_gn_stats(B):
    for i, (b, rows, C, stride, dc) in enumerate(c for c in GN_CASES if c[0] == B):
        run_gn_stats(b, rows, C, stride, dc, seed=i)


def run_band_stats(B, T, K, N, dc=0.0, seed=0):
    """Decoder layout: x (B, T, K, N), band k = floats [k N, (k+1) N) of every row of K N floats."""
    L = _lib()
    x = rnd(B, T, K, N, offset=dc, seed=seed)
    stats = sentinel(2 * B * K, torch.float64)
    off = torch.tensor([k * N for k in range(K)], dtype=torch.int32, device=DEV)
    wid = torch.tensor([N] * K, dtype=torch.int32, device=DEV)
    L.call("bsrnn_band_stats", x.data_ptr(), stats.data_ptr(), B, T, K * N, off.data_ptr(), wid.data_ptr(), K, L.stream_ptr())
    torch.cuda.synchronize()
    guard_ok(stats, 2 * B * K, "band_stats")
    geo = R.band_stats_geometry(B, T, K, N)
    s, q, bs, bq = R.sums_ref(x.permute(0, 2, 1, 3).reshape(B * K, T * N), geo["m"])
    got = stats[:2 * B * K].view(B * K, 2)
    tag = f"band_stats B={B} T={T} K={K} N={N} tchunks={geo['tchunks']}"
    assert_within(tag + " sum", got[:, 0], s, bs)
    assert_within(tag + " sumsq", got[:, 1], q, bq)
    return geo


BAND_STATS_CASES = [(40, 3, 30, 8, 0.0), (2, 1, 30, 196, 1000.0), (1, 100, 34, 196, 0.0), (3, 700, 2, 100, 0.0)]


def test_band_stats_decoder_layout():
    for i, c in enumerate(BAND_STATS_CASES):
        run_band_stats(*c, seed=i)


def run_gn_finalize(G, C, G_inner, with_extra, clamp=False, pad=0, seed=0):
    L = _lib()
    n = 1000.0
    cnt = torch.full((G_inner,), n, dtype=torch.float64, device=DEV) + torch.arange(G_inner, device=DEV)
    mean = torch.rand(G, device=DEV, dtype=torch.float64) * 2000 - 1000
    var = torch.rand(G, device=DEV, dtype=torch.float64) * 4 + 1e-3
    if clamp:
        var[::2] = -(torch.rand(G, device=DEV, dtype=torch.float64)[::2] + 0.5)         # E[x^2] - E[x]^2 < 0
    gi = torch.arange(G, device=DEV) % G_inner
    stats = torch.stack([mean * cnt[gi], (var + mean * mean) * cnt[gi]], 1).contiguous()
    gamma, beta = rnd(G_inner, C, scale=0.5, offset=1.0, seed=seed), rnd(G_inner, C, seed=seed + 1)
    if pad:
        gamma[:, C - pad:] = 0.0
        beta[:, C - pad:] = 0.0
    extra = rnd(G, C, seed=seed + 2) if with_extra else None
    sc, sh = sentinel(G * C), sentinel(G * C)
    eps = float(np.float32(1e-5))                                            # the f32 argument the kernel receives
    L.call("bsrnn_gn_finalize", stats.data_ptr(), gamma.data_ptr(), beta.data_ptr(), L.ptr(extra), sc.data_ptr(), sh.data_ptr(),
           G, C, cnt.data_ptr(), eps, G_inner, L.stream_ptr())
    torch.cuda.synchronize()
    guard_ok(sc, G * C, "gn_finalize scale")
    guard_ok(sh, G * C, "gn_finalize shift")
    (rs, bs), (rh, bh) = R.gn_finalize_ref(stats, gamma, beta, extra, cnt, eps, G_inner)
    tag = f"gn_finalize G={G} C={C} G_inner={G_inner} extra={with_extra} clamp={clamp} pad={pad}"
    assert_within(tag + " scale", sc[:G * C].view(G, C), rs, bs)
    assert_within(tag + " shift", sh[:G * C].view(G, C), rh, bh)
    if pad and not with_extra:
        assert bool((sc[:G * C].view(G, C)[:, C - pad:] == 0).all()) and bool((sh[:G * C].view(G, C)[:, C - pad:] == 0).all())
    if clamp:
        # rstd = 1/sqrt(eps) exactly where the variance was clamped
        want = torch.tensor(1.0 / math.sqrt(eps), dtype=torch.float32, device=DEV) * gamma[gi[::2]]
        assert torch.equal(sc[:G * C].view(G, C)[::2], want), f"{tag}: clamped rows"


def test_gn_finalize():
    run_gn_finalize(3, 196, 1, True, seed=1)
    run_gn_finalize(64 * 30, 196, 30, False, seed=2)
    run_gn_finalize(2 * 34, 120, 34, False, pad=40, seed=3)
    run_gn_finalize(5, 300, 1, True, clamp=True, seed=4)
    run_gn_finalize(2 * 7, 8, 7, False, clamp=True, pad=3, seed=5)


def test_gn_cases_reach_every_branch():
    geos = [R.gn_stats_geometry(B, rows, C, s) for B, rows, C, s, _ in GN_CASES]
    assert {True, False} == {g["contiguous"] for g in geos}
    assert any(g["m"] == R.FLUSH for g in geos if g["contiguous"])          # a flushed partial
    assert any(g["m"] > R.FLUSH for g in geos if not g["contiguous"])        # strided: unflushed partials of > 64 terms
    assert any(g["chunks"] == 1 for g in geos)                               # B > 1184: one chunk per sample
    assert any(rows < g["chunks"] for (_, rows, *_), g in zip(GN_CASES, geos))    # rows_per_sample < chunks
    assert {1, 196, 300} <= {C for _, _, C, _, _ in GN_CASES}
    bgeo = [R.band_stats_geometry(B, T, K, N) for B, T, K, N, _ in BAND_STATS_CASES]
    assert any(g["tchunks"] == 1 and B * K > R.STAT_CTAS for g, (B, T, K, *_) in zip(bgeo, BAND_STATS_CASES))
    assert any(T == 1 for _, T, *_ in BAND_STATS_CASES) and any(g["tchunks"] > 1 for g in bgeo)


# ------------------------------------------------------------------------------------------------------------ conv5x5_glu
def run_conv(B, T, Fp, F_out, seed=0, sharp=False):
    L = _lib()
    g = rnd(B, T, Fp, 16, scale=0.7, seed=seed)
    w = rnd(4, 16, 5, 5, scale=0.08, seed=seed + 1)
    b = rnd(4, scale=0.3, seed=seed + 2)
    out = sentinel(B * T * F_out * 2)
    L.call("bsrnn_conv5x5_glu", g.data_ptr(), w.data_ptr(), b.data_ptr(), out.data_ptr(), B, T, Fp, F_out, L.stream_ptr())
    torch.cuda.synchronize()
    tag = f"conv5x5_glu B={B} T={T} Fp={Fp} F={F_out}"
    guard_ok(out, B * T * F_out * 2, tag)
    ref, bound = R.conv5x5_glu_ref(g, w, b, F_out)
    got = out[:B * T * F_out * 2].view(B, T, F_out, 2)
    if F_out > Fp:
        assert bool((got[:, :, Fp:] == 0).all()), f"{tag}: bins >= F' are not exactly 0"
    w_ = worst_ratio(got, ref, bound)
    assert w_ <= 1.0, f"{tag}: worst err/bound {w_:.3g}"
    if sharp:
        gv, rv, bv = got.reshape(B * T, -1), ref.reshape(B * T, -1), bound.reshape(B * T, -1)
        assert_checker_is_sharp(tag, gv, rv, bv, tile=8)
    return w_


CONV_CASES = [(3, T, Fp, F_out) for T in (1, 2, 7, 8, 9, 100) for Fp in (1, 4, 31, 32, 33)
              for F_out in sorted({max(1, Fp - 1), Fp, Fp + 3})]


def test_conv5x5_glu_edges():
    worst = max(run_conv(*c, seed=i, sharp=c == (3, 9, 33, 36)) for i, c in enumerate(CONV_CASES))
    print(f"conv5x5_glu ({len(CONV_CASES)} shapes): worst err/bound = {worst:.3g}")


def test_conv5x5_glu_flowse_shape():
    Fp = sum(runtime_subbands(769))
    print(f"conv5x5_glu FlowSE: worst err/bound = {run_conv(1, 51, Fp, 769, seed=9):.3g}")


def test_conv_cases_reach_every_branch():
    assert any(F_ < Fp for _, _, Fp, F_ in CONV_CASES) and any(F_ > Fp for _, _, Fp, F_ in CONV_CASES)
    assert any(F_ == Fp for _, _, Fp, F_ in CONV_CASES)
    assert {T % R.CONV_CT != 0 for _, T, _, _ in CONV_CASES} == {True, False}
    assert {max(Fp, F_) % R.CONV_CF != 0 for _, _, Fp, F_ in CONV_CASES} == {True, False}
    assert any(R.conv_grid(B, T, Fp, F_)[0] > 1 for B, T, Fp, F_ in CONV_CASES)


# ------------------------------------------------------------------------------------------------------------ flow pieces
def test_time_embed():
    L = _lib()
    for B, E, tscale in ((3, 43, 1.0), (1, 1, 1.0), (7, 128, 1.0), (5, 97, 1000.0)):
        t = torch.rand(B, device=DEV) * tscale
        W = rnd(E, scale=16.0, seed=B + E)
        out = sentinel(B * 2 * E)
        L.call("bsrnn_time_embed", t.data_ptr(), W.data_ptr(), out.data_ptr(), B, E, L.stream_ptr())
        torch.cuda.synchronize()
        tag = f"time_embed B={B} E={E} |phase| <= {float(R.time_phase_f32(t, W).abs().max()):.3g}"
        guard_ok(out, B * 2 * E, tag)
        ref, bound = R.time_embed_ref(t.cpu(), W.cpu())
        got = out[:B * 2 * E].view(B, 2 * E)
        assert_within(tag, got, ref.to(DEV), bound.to(DEV))
        if B > 1:
            assert_checker_is_sharp(tag, got, ref.to(DEV), bound.to(DEV), tile=1)


FLOW_N = (1, 303103, 303105, 4 * 1024 * 1024 + 7)


def test_complex_elementwise():
    L = _lib()
    _, steps = O.euler_schedule(1.0, 0.03, 15)
    for i, n in enumerate(FLOW_N):
        x, m, r = rnd(n, 2, seed=i), rnd(n, 2, scale=0.5, seed=i + 10), rnd(n, 2, seed=i + 20)
        st = L.stream_ptr()
        for sign in (1.0, -1.0):
            out = sentinel(2 * n)
            L.call("bsrnn_complex_mask", out.data_ptr(), x.data_ptr(), m.data_ptr(), r.data_ptr(), sign, n, st)
            torch.cuda.synchronize()
            guard_ok(out, 2 * n, "complex_mask")
            assert_within(f"complex_mask n={n} sign={sign:+.0f}", out[:2 * n].view(n, 2), *R.complex_mask_ref(x, m, r, sign))
        sigma = 0.5
        out = sentinel(2 * n)
        L.call("bsrnn_axpy_complex", out.data_ptr(), x.data_ptr(), r.data_ptr(), sigma, n, st)
        torch.cuda.synchronize()
        guard_ok(out, 2 * n, "axpy_complex")
        assert_within(f"axpy_complex n={n}", out[:2 * n].view(n, 2), *R.axpy_ref(x, r, sigma))
        # the Euler sampler: every step size euler_schedule produces, x updated in place
        xs = sentinel(2 * n)
        xs[:2 * n] = x.view(-1)
        for j, step in enumerate(steps.tolist()[:: (1 if n < 10 ** 6 else 7)]):
            before = xs[:2 * n].view(n, 2).clone()
            L.call("bsrnn_euler_step", xs.data_ptr(), m.data_ptr(), r.data_ptr(), step, n, st)
            torch.cuda.synchronize()
            guard_ok(xs, 2 * n, "euler_step")
            ref, bound = R.euler_step_ref(before, m, r, step)
            got = xs[:2 * n].view(n, 2)
            assert_within(f"euler_step n={n} step={step:.4g}", got, ref, bound)
            if j == 0 and n > 1:
                assert_checker_is_sharp(f"euler_step n={n}", got, ref, bound, tile=1)
    assert [R.flow_grid_passes(n) for n in FLOW_N] == [1, 1, 2, 14]
