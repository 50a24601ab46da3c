"""GPU tests (-m gpu) of the spectral kernels -- bsrnn_fft_twiddle, bsrnn_stft_fwd, bsrnn_stft_stats_fwd, bsrnn_istft_fwd,
bsrnn_istft_bwd (csrc/fft.cu, csrc/fft_core.cuh), bsrnn_band_stats (csrc/norm.cu) on the spectrum, bsrnn_mrl1_spec_fwd_bwd and
bsrnn_l1_time_fwd_bwd (csrc/loss.cu) -- each called through the C ABI against a plain f64 restatement in tests/spectral_ref.py.

The bar is ELEMENTWISE, with bounds derived in spectral_ref's docstring from the butterflies, the launchers and the documented
error of __powf (not fitted): every bin of the STFT within u C_plan ||Z_pair||_2 plus its window error (propagated through the
compression by interval arithmetic), every iSTFT sample within the inverse-FFT bound of the frames covering it over the
envelope, every gradient sample of the loss within its phasor errors plus 2 weight per AMBIGUOUS bin (f64 margin within the
magnitude bounds; their count is printed per case).  Every case prints its worst err / bound and asserts it <= 1.  Frames the
kernels must zero (past olen, past the last frame of the iSTFT) have bound 0 and must be exactly 0.

Everything around an output -- a guard tail after every buffer, spec_out's untouched state -- starts as a NaN bit pattern
and must come back bit-identical (or, for spec_out, be written everywhere).  Sharpness cases corrupt the kernels' real output
(one bin 3x its bound off, two frames swapped, the last frame of a CTA zeroed, a stale spec_out frame, the trimmed tail
shifted by a sample, one gradient sample 3x its bound off outside the ambiguous allowance) and require the check to reject
each.  The launcher classes (STFT fpb, iSTFT (fpb, G) and nblocks from L_out or from T, loss fpb) are restated in
spectral_ref and the case lists are asserted to reach every one of them.
"""
import math

import pytest
import torch

import spectral_ref as S
from oracle import restated as R

pytestmark = pytest.mark.gpu

GUARD = 1024
SENT32 = 0x7F8DEAD1
SENT64 = 0x7FF4DEADBEEF0001
SE_SIZES = [(160, 80), (320, 160), (441, 220), (480, 240), (640, 320), (882, 441), (960, 480)]
FLOWSE_SIZES = [(256, 64), (512, 128), (705, 176), (768, 192), (1024, 256), (1411, 352), (1536, 384)]
RATES = (8000, 16000, 22050, 24000, 32000, 44100, 48000)
SWEEP = [n for n in range(4, 201) if S.make_plan(n) is not None]
LOSS_SWEEP = [w for w in SWEEP if w % 2 == 0]
LOSS_MODEL = [(256, 96000, 3), (512, 48000, 2), (768, 32000, 2), (1024, 40000, 2), (2048, 20000, 2)]
EXTRA_STFT = [(3072, 768), (2048, 512)]
FLOWSE_COMP = (0.667, 0.065)


def _lib():
    from urgent2026_challenge_track1_b200 import _lib as L
    L.require_device()
    return L


# ------------------------------------------------------------------------------------------------------------ machinery
def sentinel(n, dtype=torch.float32):
    if dtype == torch.float64:
        return torch.full((n + GUARD,), SENT64, dtype=torch.int64, device="cuda").view(torch.float64)
    return torch.full((n + GUARD,), SENT32, dtype=torch.int32, device="cuda").view(torch.float32)


def guard_ok(buf, n, name):
    raw = buf.view(torch.int64 if buf.dtype == torch.float64 else torch.int32)[n:]
    want = SENT64 if buf.dtype == torch.float64 else SENT32
    assert bool((raw == want).all()), f"{name}: guard tail written"


def worst_ratio(got, ref, bound):
    """max |got - ref| / bound over complex or real elements (inf where an error meets a zero bound or a value is not
    finite)."""
    err = (got - ref).abs()
    ratio = torch.where(bound > 0, err / bound.clamp(min=1e-300), torch.where(err > 0, math.inf, 0.0))
    return float(torch.nan_to_num(ratio, nan=math.inf).max()) if ratio.numel() else 0.0


def assert_within(name, got, ref, bound, extra=""):
    w = worst_ratio(got, ref, bound)
    print(f"{name}: worst err/bound = {w:.3g}{extra}")
    assert w <= 1.0, f"{name}: worst err/bound {w:.3g}"
    return w


def as_complex(buf, shape):
    n = math.prod(shape) * 2
    return torch.view_as_complex(buf[:n].view(*shape, 2).double().cpu().contiguous())


_TW = {}


def twiddle(n):
    if n not in _TW:
        L = _lib()
        buf = sentinel(2 * n)
        L.call("bsrnn_fft_twiddle", buf.data_ptr(), n, L.stream_ptr())
        guard_ok(buf, 2 * n, f"twiddle {n}")
        _TW[n] = buf
    return _TW[n]


def run_stft(wav, lens, n_fft, hop, transform=0, exponent=1.0, factor=1.0, edges=None, stats=None):
    L = _lib()
    B, Ls = wav.shape
    T, Fb = S.n_frames(Ls, hop), n_fft // 2 + 1
    spec = sentinel(B * T * Fb * 2)
    w = wav.cuda().contiguous()
    ln = None if lens is None else torch.tensor(lens, dtype=torch.int32, device="cuda")
    if edges is None:
        L.call("bsrnn_stft_fwd", w.data_ptr(), L.ptr(ln), spec.data_ptr(), twiddle(n_fft).data_ptr(), B, Ls, n_fft, hop,
               transform, exponent, factor, L.stream_ptr())
    else:
        e = torch.tensor(edges, dtype=torch.int32, device="cuda")
        L.call("bsrnn_stft_stats_fwd", w.data_ptr(), L.ptr(ln), spec.data_ptr(), twiddle(n_fft).data_ptr(), B, Ls, n_fft,
               hop, transform, exponent, factor, stats.data_ptr(), e.data_ptr(), len(edges) - 1, L.stream_ptr())
    torch.cuda.synchronize()
    guard_ok(spec, B * T * Fb * 2, f"stft {n_fft}/{hop}")
    return spec, as_complex(spec, (B, T, Fb))


def check_stft(name, wav, lens, n_fft, hop, transform=0, exponent=1.0, factor=1.0):
    _, got = run_stft(wav, lens, n_fft, hop, transform, exponent, factor)
    ref, bound = S.stft_ref(wav, lens, n_fft, hop, transform, exponent, factor)
    assert_within(name, got, ref, bound)
    return got, ref, bound


def wavs(B, L, seed, kind="noise"):
    if kind == "speech":
        return R.synth_noisy(B, L, 16000, seed=seed)
    g = torch.Generator().manual_seed(seed)
    return (0.3 * torch.randn(B, L, generator=g)).float()


def rand_spec(B, T, Fb, seed, scale=1.0):
    g = torch.Generator().manual_seed(seed)
    return (scale * torch.randn(B, T, Fb, 2, generator=g)).float()


def run_istft(spec, mask, resid, L_out, n_fft, hop, want_spec_out, transform=0, exponent=1.0, factor=1.0):
    L = _lib()
    B, T, Fb, _ = spec.shape
    wav = sentinel(B * L_out)
    so = sentinel(B * T * Fb * 2) if want_spec_out else None
    s, m, r = (None if x is None else x.cuda().contiguous() for x in (spec, mask, resid))
    L.call("bsrnn_istft_fwd", s.data_ptr(), L.ptr(m), L.ptr(r), L.ptr(so), wav.data_ptr(), twiddle(n_fft).data_ptr(), B, T,
           L_out, n_fft, hop, transform, exponent, factor, L.stream_ptr())
    torch.cuda.synchronize()
    guard_ok(wav, B * L_out, f"istft {n_fft}/{hop} wav")
    if so is not None:
        guard_ok(so, B * T * Fb * 2, f"istft {n_fft}/{hop} spec_out")
    return wav[:B * L_out].view(B, L_out).double().cpu(), (None if so is None else as_complex(so, (B, T, Fb)))


def istft_expect(spec, mask, resid, L_out, n_fft, hop, transform=0, exponent=1.0, factor=1.0):
    s, ds = S.masked_ref(spec, mask, resid)
    v, dv = (S.decompress_ref(s, ds, exponent, factor) if transform == 1 else (s, ds))
    ref = S.istft_ref(v, n_fft, hop, L_out)
    bound, straddle = S.istft_bound(v, dv, n_fft, hop, L_out)
    return s, ds, ref, bound, straddle


def check_istft(name, spec, mask, resid, L_out, n_fft, hop, want_spec_out=True, transform=0, exponent=1.0, factor=1.0):
    got, so = run_istft(spec, mask, resid, L_out, n_fft, hop, want_spec_out, transform, exponent, factor)
    s, ds, ref, bound, straddle = istft_expect(spec, mask, resid, L_out, n_fft, hop, transform, exponent, factor)
    assert_within(f"{name} wav", got, ref, bound, f" (straddling the envelope threshold: {int(straddle.sum())})")
    if so is not None:
        assert_within(f"{name} spec_out", so, s, ds)            # every frame written: NaN prefill fails the check
    return got, ref, bound, so, s, ds


def run_istft_bwd(g, T, n_fft, hop):
    L = _lib()
    B, L_out = g.shape
    Fb = n_fft // 2 + 1
    out = sentinel(B * T * Fb * 2)
    gg = g.cuda().contiguous()
    L.call("bsrnn_istft_bwd", gg.data_ptr(), out.data_ptr(), twiddle(n_fft).data_ptr(), B, T, L_out, n_fft, hop,
           L.stream_ptr())
    torch.cuda.synchronize()
    guard_ok(out, B * T * Fb * 2, f"istft_bwd {n_fft}/{hop}")
    return as_complex(out, (B, T, Fb))


# ------------------------------------------------------------------------------------------------------------ coverage
def _stft_cases():
    out = [(n, max(1, n // 2)) for n in SWEEP] + [(n, max(1, n // 4)) for n in SWEEP] + SE_SIZES + FLOWSE_SIZES + EXTRA_STFT
    return out


def _istft_cases():
    """(n_fft, hop, T, L_out) of every iSTFT call below."""
    out = []
    for n, h in [(n, max(1, n // 2)) for n in SWEEP] + [(n, max(1, n // 4)) for n in SWEEP]:
        out.append((n, h, 9, 8 * h))
    for n, h in SE_SIZES + FLOWSE_SIZES + EXTRA_STFT:
        T = 23
        out += [(n, h, T, (T - 1) * h)]
    for n, h in EDGE_ISTFT_SIZES:
        ov = (n + h - 1) // h - 1
        for T in sorted({1, 2, max(1, ov - 1), 11}):
            for L_out in _edge_lengths(T, h, n):
                out.append((n, h, T, L_out))
    return out


EDGE_ISTFT_SIZES = [(960, 480), (441, 220), (256, 64), (705, 176), (1536, 384), (3072, 768), (16, 4)]


def _edge_lengths(T, hop, n_fft):
    full = (T - 1) * hop
    return sorted({max(1, full), max(1, full - 3 - (full % 2)), 1, full + n_fft // 2 + 5})       # the 2nd is odd


def test_launcher_classes_are_all_reached():
    stft = {S.stft_fpb(n) for n, _ in _stft_cases()}
    assert stft == {8, 4, 2}, stft
    classes, nb_from_T, nb_from_L = set(), False, False
    for n, h, T, L_out in _istft_cases():
        fpb, ov, G, span, nb = S.istft_geometry(n, h, T, L_out)
        classes.add((fpb, G))
        by_L = -(-(n // 2 + L_out) // span)
        nb_from_T |= nb > by_L
        nb_from_L |= nb == by_L and by_L > -(-T // G)
    need = {(8, 7), (8, 6), (8, 5), (8, 4), (4, 8), (2, 8)}
    assert need <= classes, need - classes
    assert nb_from_T and nb_from_L
    loss = {S.loss_fpb(w) for w in LOSS_SWEEP + [w for w, _, _ in LOSS_MODEL]}
    assert {8, 4, 2} <= loss, loss
    print(f"STFT fpb {sorted(stft)}; iSTFT (fpb, G) {sorted(classes)}; loss fpb {sorted(loss)}")


# ------------------------------------------------------------------------------------------------------------ twiddles
def test_twiddles_are_the_rounded_roots_of_unity():
    worst = 0.0
    for n in sorted(set(SWEEP) | {n for n, _ in SE_SIZES + FLOWSE_SIZES + EXTRA_STFT}):
        got = as_complex(twiddle(n), (n,))
        ref = S.twiddles(n)
        # each component rounded once from the double sincospi: u |component| (+ 2^-50 for the double itself)
        bound = (S.U * ref.real.abs() + 2.0 ** -50) + (S.U * ref.imag.abs() + 2.0 ** -50)
        worst = max(worst, worst_ratio(got, ref, bound))
    print(f"twiddles: worst err/bound = {worst:.3g}")
    assert worst <= 1.0


# ------------------------------------------------------------------------------------------------------------ STFT
@pytest.mark.parametrize("quarter", [False, True])
def test_stft_plan_sweep(quarter):
    """every n_fft 4..200 make_plan accepts (every radix path, generic primes up to 89), hop n/2 and n/4."""
    worst = 0.0
    for n in SWEEP:
        hop = max(1, n // 4 if quarter else n // 2)
        L = max(n // 2 + 1, 11 * hop + n % 5)
        wav = wavs(2, L, n)
        _, got = run_stft(wav, [L, max(1, L - 3 * hop - 1)], n, hop)
        ref, bound = S.stft_ref(wav, [L, max(1, L - 3 * hop - 1)], n, hop)
        w = worst_ratio(got, ref, bound)
        print(f"stft sweep n={n} hop={hop} plan={S.make_plan(n)}: worst err/bound = {w:.3g}")
        assert w <= 1.0, (n, hop, w)
        worst = max(worst, w)
    print(f"stft sweep (hop n/{4 if quarter else 2}): worst err/bound = {worst:.3g}")


@pytest.mark.parametrize("n_fft,hop", SE_SIZES + FLOWSE_SIZES + EXTRA_STFT)
def test_stft_model_sizes(n_fft, hop):
    L = 20 * hop + 7
    wav = wavs(3, L, n_fft, "speech")
    lens = [L, L - 5 * hop - 3, n_fft // 2 + 1]
    check_stft(f"stft {n_fft}/{hop}", wav, lens, n_fft, hop)
    e, f = FLOWSE_COMP if (n_fft, hop) in FLOWSE_SIZES else (0.5, 0.15)
    check_stft(f"stft {n_fft}/{hop} exponent {e} factor {f}", wav, lens, n_fft, hop, 1, e, f)


@pytest.mark.parametrize("n_fft,hop", [(160, 80), (1536, 384), (3072, 768), (705, 176)])
def test_stft_frame_and_length_edges(n_fft, hop):
    """T mod fpb at every residue; olen mid-CTA, on a CTA boundary, = T, = 1; lens NULL; L = n/2 + 1; B in {1, 3, 5}."""
    fpb = S.stft_fpb(n_fft)
    for res in range(fpb):
        T = 3 * fpb + res if res else 2 * fpb
        L = (T - 1) * hop + (res % max(1, hop))
        assert S.n_frames(L, hop) == T
        B = (1, 3, 5)[res % 3]
        lens = [L, (fpb + fpb // 2) * hop + 1, fpb * hop - n_fft // 2 + 1, 1, L - 1][:B]   # = T, mid-CTA, CTA boundary, 1
        lens = [min(L, max(1, v)) for v in lens]
        ol = S.olens(lens, L, n_fft, hop, B)
        for tr in (0, 1):
            wav = wavs(B, L, 7 * res + tr)
            check_stft(f"stft edges {n_fft}/{hop} T={T} (T mod fpb={T % fpb}) B={B} olen={ol} tr={tr}", wav, lens, n_fft,
                       hop, tr, *FLOWSE_COMP)
        check_stft(f"stft edges {n_fft}/{hop} T={T} lens=NULL", wavs(2, L, res), None, n_fft, hop)
    L = n_fft // 2 + 1                                          # smallest accepted length: reflection reaches the far end
    for tr in (0, 1):
        check_stft(f"stft {n_fft}/{hop} L=n/2+1 tr={tr}", wavs(3, L, 5), [L, L - 1, 1], n_fft, hop, tr, *FLOWSE_COMP)


def test_stft_checker_is_sharp():
    n_fft, hop = 960, 480
    L = 30 * hop
    wav = wavs(2, L, 1, "speech")
    got, ref, bound = check_stft("stft sharpness base", wav, None, n_fft, hop)
    bad = got.clone()
    k = int(bound.reshape(-1).argmax())
    bad.view(-1)[k] += 3.0 * bound.reshape(-1)[k]
    assert worst_ratio(bad, ref, bound) > 1.0, "one bin 3x its bound off passes"
    bad = got.clone()
    bad[:, [1, 2]] = bad[:, [2, 1]]
    assert worst_ratio(bad, ref, bound) > 1.0, "two swapped frames pass"
    bad = got.clone()
    bad[1, S.stft_fpb(n_fft) - 1] = 0
    assert worst_ratio(bad, ref, bound) > 1.0, "a zeroed last frame of a CTA passes"


def test_stft_crosstalk_floor():
    """A frame wholly inside a span of digital zeros is 0 in f64; the kernel's carries the rounding of its loud FFT partner.
    It must stay within the pair bound; the floor relative to the loud frames is printed (without and with compression)."""
    n_fft, hop = 960, 480
    L = 40 * hop
    wav = wavs(1, L, 3, "speech") * 10.0
    wav[:, 15 * hop:25 * hop] = 0.0
    for tr, (e, f) in ((0, (1.0, 1.0)), (1, FLOWSE_COMP)):
        got, ref, bound = check_stft(f"stft crosstalk tr={tr}", wav, None, n_fft, hop, tr, e, f)
        quiet = [t for t in range(S.n_frames(L, hop)) if t * hop - n_fft // 2 >= 15 * hop and
                 t * hop + n_fft - n_fft // 2 <= 25 * hop]
        loud = [t for t in quiet if (t ^ 1) not in quiet]
        assert quiet and loud and bool((ref[:, quiet] == 0).all())
        floor = float(got[:, loud].abs().max()) / float(ref.abs().max())
        print(f"crosstalk tr={tr}: quiet frames {quiet}, paired with a loud frame {loud}: max |bin| / max loud |bin| = "
              f"{floor:.3g}; worst quiet err/bound = {worst_ratio(got[:, quiet], ref[:, quiet], bound[:, quiet]):.3g}")


# ------------------------------------------------------------------------------------------------------------ band stats
def _plans():
    from urgent2026_challenge_track1_b200 import runtime as RT
    out = []
    for sub, base in ((RT.SUBBANDS[481], (960, 480)), (RT.SUBBANDS[769], (1536, 384))):
        for fs in RATES:
            n, h = RT.stft_dims(fs, *base)
            plan = RT.BandPlan.make(sub, n // 2 + 1)
            out.append((n, h, plan, list(plan.bin0) + [plan.bin0[-1] + plan.width[-1]]))
    return out


def test_band_stats_fused_and_separate():
    L = _lib()
    from urgent2026_challenge_track1_b200 import runtime as RT
    cases = _plans()
    n, h = 160, 80                                               # synthetic table: its last bands start at or beyond F = 81
    cases.append((n, h, None, [0, 5, 30, 80, 81, 90, 200]))
    for n, h, plan, edges in cases:
        Ls = 17 * h + 3
        K = len(edges) - 1
        stats = sentinel(3 * K * 2, torch.float64)
        lens = [Ls, Ls - 6 * h, n // 2 + 1]
        tr, e, f = (1, *FLOWSE_COMP) if n in {s[0] for s in FLOWSE_SIZES} else (0, 1.0, 1.0)
        for seed in (0, 1):                                     # relaunch into the same buffer: the call zeroes it
            wav = wavs(3, Ls, 100 * n + seed, "speech")
            spec_buf, got = run_stft(wav, lens, n, h, tr, e, f, edges=edges, stats=stats)
            guard_ok(stats, 3 * K * 2, "stft_stats stats")
            ref, bound = S.stft_ref(wav, lens, n, h, tr, e, f)
            assert_within(f"stft_stats {n}/{h} K={K} spectrum", got, ref, bound)
            st = stats[:3 * K * 2].view(3, K, 2).cpu()
            own, own_abs, cnt = S.band_stats_ref(got, edges)
            tol_own = (cnt[None, :, None] + 64) * S.U53 * own_abs      # double sums of f32 values (exact products)
            assert_within(f"stft_stats {n}/{h} seed {seed} vs own spectrum", st, own, tol_own)
            sref, _, _ = S.band_stats_ref(ref, edges)
            d1 = torch.zeros_like(sref)
            for k in range(K):
                k0, k1 = edges[k], min(edges[k + 1], n // 2 + 1)
                if k0 < k1:
                    b = bound[:, :, k0:k1]
                    d1[:, k, 0] = (math.sqrt(2.0) * b).sum(dim=(1, 2))
                    d1[:, k, 1] = (2.0 * ref[:, :, k0:k1].abs() * b + b * b).sum(dim=(1, 2))
            tol_ref = d1 + tol_own
            assert_within(f"stft_stats {n}/{h} seed {seed} vs f64 spectrum", st, sref, tol_ref)
            if plan is None:
                assert bool((st[:, 4:] == 0).all())
                continue
            # bsrnn_band_stats on the same spectrum, offsets and widths of runtime.band_split_f32
            off = torch.tensor([2 * b0 for b0 in plan.bin0], dtype=torch.int32, device="cuda")
            wid = torch.tensor([2 * w for w in plan.width], dtype=torch.int32, device="cuda")
            st2 = sentinel(3 * plan.K * 2, torch.float64)
            T = S.n_frames(Ls, h)
            L.call("bsrnn_band_stats", spec_buf.data_ptr(), st2.data_ptr(), 3, T, 2 * (n // 2 + 1), off.data_ptr(),
                   wid.data_ptr(), plan.K, L.stream_ptr())
            torch.cuda.synchronize()
            guard_ok(st2, 3 * plan.K * 2, "band_stats")
            st2 = st2[:3 * plan.K * 2].view(3, plan.K, 2).cpu()
            tol_f32 = 65 * S.U * own_abs + tol_own     # f32 partials of <= 64 terms (+ v*v rounding)
            assert_within(f"band_stats {n}/{h} seed {seed} vs own spectrum", st2, own, tol_f32)
            assert_within(f"band_stats {n}/{h} seed {seed} vs f64 spectrum", st2, sref, tol_ref + tol_f32)


# ------------------------------------------------------------------------------------------------------------ iSTFT
@pytest.mark.parametrize("quarter", [False, True])
def test_istft_plan_sweep(quarter):
    worst = 0.0
    for n in SWEEP:
        hop = max(1, n // 4 if quarter else n // 2)
        T = 9
        spec = rand_spec(2, T, n // 2 + 1, n)
        got, _ = run_istft(spec, None, None, 8 * hop, n, hop, False)
        _, _, ref, bound, _ = istft_expect(spec, None, None, 8 * hop, n, hop)
        w = worst_ratio(got, ref, bound)
        print(f"istft sweep n={n} hop={hop}: worst err/bound = {w:.3g}")
        assert w <= 1.0, (n, hop, w)
        worst = max(worst, w)
    print(f"istft sweep (hop n/{4 if quarter else 2}): worst err/bound = {worst:.3g}")


@pytest.mark.parametrize("n_fft,hop", SE_SIZES + FLOWSE_SIZES + EXTRA_STFT)
def test_istft_model_sizes(n_fft, hop):
    T, Fb = 23, n_fft // 2 + 1
    spec = rand_spec(3, T, Fb, n_fft)
    mask, resid = rand_spec(3, T, Fb, n_fft + 1), rand_spec(3, T, Fb, n_fft + 2, 0.1)
    print(f"istft {n_fft}/{hop}: (fpb, overlap, G, span, nblocks) = {S.istft_geometry(n_fft, hop, T, (T - 1) * hop)}")
    check_istft(f"istft {n_fft}/{hop} mask", spec, mask, resid, (T - 1) * hop, n_fft, hop)
    check_istft(f"istft {n_fft}/{hop} plain, spec_out", spec, None, None, (T - 1) * hop, n_fft, hop)
    e, f = FLOWSE_COMP if (n_fft, hop) in FLOWSE_SIZES else (0.5, 0.15)
    check_istft(f"istft {n_fft}/{hop} mask exponent {e}", spec * 0.1, mask, resid * 0.1, (T - 1) * hop, n_fft, hop,
                True, 1, e, f)


@pytest.mark.parametrize("n_fft,hop", EDGE_ISTFT_SIZES)
def test_istft_edges(n_fft, hop):
    """T in {1, 2, fewer frames than the overlap, 11}; L_out = (T-1) hop, shorter and odd, 1 (nblocks from T), and past the
    last frame (a zero tail); mask / spec_out / transform present and absent."""
    Fb = n_fft // 2 + 1
    ov = (n_fft + hop - 1) // hop - 1
    for T in sorted({1, 2, max(1, ov - 1), 11}):
        spec = rand_spec(2, T, Fb, 10 * T + n_fft)
        mask, resid = rand_spec(2, T, Fb, 10 * T + 1), rand_spec(2, T, Fb, 10 * T + 2, 0.1)
        for L_out in _edge_lengths(T, hop, n_fft):
            geo = S.istft_geometry(n_fft, hop, T, L_out)
            for k, (m, r, so, tr) in enumerate(((mask, resid, True, 0), (None, None, False, 0), (mask, resid, False, 1),
                                                (None, None, True, 1))):
                if T > 2 and L_out not in (1, (T - 1) * hop) and k > 1:
                    continue
                sc = 0.1 if tr else 1.0
                check_istft(f"istft {n_fft}/{hop} T={T} L_out={L_out} geo={geo} mask={m is not None} spec_out={so} "
                            f"tr={tr}", spec * sc, m, None if r is None else r * sc, L_out, n_fft, hop, so, tr,
                            *FLOWSE_COMP)


def test_istft_checker_is_sharp():
    n_fft, hop = 960, 480
    T, Fb = 20, 481
    spec, mask, resid = rand_spec(2, T, Fb, 1), rand_spec(2, T, Fb, 2), rand_spec(2, T, Fb, 3, 0.1)
    L_out = (T - 1) * hop - 5
    got, ref, bound, so, s, ds = check_istft("istft sharpness base", spec, mask, resid, L_out, n_fft, hop)
    bad = so.clone()
    bad[1, 7] = torch.view_as_complex(spec[1, 7].double().contiguous())      # one spec_out frame left stale (unmasked)
    assert worst_ratio(bad, s, ds) > 1.0, "a stale spec_out frame passes"
    bad = got.clone()
    bad[0, -1] = bad[0, -2]                                                   # the trimmed tail shifted by one sample
    assert worst_ratio(bad, ref, bound) > 1.0, "a wrong last sample passes"
    bad = got.clone()
    k = int(bound.reshape(-1).argmax())
    bad.view(-1)[k] += 3.0 * bound.reshape(-1)[k]
    assert worst_ratio(bad, ref, bound) > 1.0, "one sample 3x its bound off passes"


# ------------------------------------------------------------------------------------------------------------ adjoint
@pytest.mark.parametrize("n_fft,hop", SE_SIZES + FLOWSE_SIZES + EXTRA_STFT)
def test_istft_adjoint(n_fft, hop):
    """elementwise against the f64 transpose, and <istft(s), w> = <s, istft_bwd(w)> from the kernels' outputs."""
    g = torch.Generator().manual_seed(n_fft)
    for T, L_out in ((21, 20 * hop), (21, 20 * hop - 7), (S.stft_fpb(n_fft) * 2 + 1, (2 * S.stft_fpb(n_fft)) * hop + 3)):
        w = (0.5 * torch.randn(2, L_out, generator=g)).float()
        got = run_istft_bwd(w, T, n_fft, hop)
        ref = S.istft_bwd_ref(w, T, n_fft, hop)
        bound = S.istft_bwd_bound(w, T, n_fft, hop)
        assert_within(f"istft_bwd {n_fft}/{hop} T={T} L_out={L_out}", got, ref, bound)
        s = rand_spec(2, T, n_fft // 2 + 1, T)
        y, _ = run_istft(s, None, None, L_out, n_fft, hop, False)
        _, _, yref, ybound, _ = istft_expect(s, None, None, L_out, n_fft, hop)
        sc = torch.view_as_complex(s.double().contiguous())
        lhs, rhs = float((y * w.double()).sum()), S.real_inner(sc, got, n_fft)
        tol = float((w.double().abs() * ybound).sum()) + float(_abs_dot_bound(sc, bound, n_fft))
        tol += 2.0 ** -50 * (abs(lhs) + abs(rhs))
        print(f"adjoint identity {n_fft}/{hop} T={T} L_out={L_out}: |lhs - rhs| / bound = {abs(lhs - rhs) / tol:.3g}")
        assert abs(lhs - rhs) <= tol
        assert abs(float((yref * w.double()).sum()) - S.real_inner(sc, ref, n_fft)) <= 1e-9 * (abs(lhs) + 1)


def _abs_dot_bound(sc, bound, n_fft):
    """sum |s| * bound over the components the inner product reads (each component of a bin within the modulus bound)."""
    return float(((sc.real.abs() + sc.imag.abs()) * bound).sum())


# ------------------------------------------------------------------------------------------------------------ loss
def run_loss(est, tgt, window, weight, prefill, loss0):
    L = _lib()
    B, Ls = est.shape
    e, t = est.cuda().contiguous(), tgt.cuda().contiguous()
    grad = sentinel(B * Ls)
    grad[:B * Ls] = prefill.reshape(-1).cuda()
    loss = sentinel(B, torch.float64)
    loss[:B] = loss0
    L.call("bsrnn_mrl1_spec_fwd_bwd", e.data_ptr(), t.data_ptr(), loss.data_ptr(), grad.data_ptr(), twiddle(window).data_ptr(),
           B, Ls, window, weight, L.stream_ptr())
    torch.cuda.synchronize()
    guard_ok(grad, B * Ls, "loss grad")
    guard_ok(loss, B, "loss value")
    return loss[:B].cpu(), grad[:B * Ls].view(B, Ls).double().cpu()


def check_loss(name, est, tgt, window, weight, want_amb_small=True):
    B, Ls = est.shape
    weight = S.f32(weight)
    g = torch.Generator().manual_seed(window + Ls)
    prefill = torch.randn(B, Ls, generator=g).float()
    loss, grad = run_loss(est, tgt, window, weight, prefill, 1.5)
    value, gref, info = S.loss_spec_ref(est, tgt, window, weight)
    vb, gb, amb_part, amb = S.loss_spec_bound(est, tgt, window, weight, info, prefill.double().abs())
    n_amb, n_bins = int(amb.sum()), amb.numel()
    extra = f" (ambiguous bins {n_amb} of {n_bins})"
    assert_within(f"{name} value", loss, 1.5 + value, vb)
    assert_within(f"{name} grad", grad, prefill.double() + gref, gb, extra)
    if want_amb_small:
        # at most 2 %: the largest generic radix here (47, at w = 94) leaves about 1 % of noise bins within their bound
        assert n_amb <= 0.02 * n_bins, f"{name}: {n_amb} ambiguous bins of {n_bins}: the bound is not sharp"
    else:
        print(f"{name}: kernel's spectral gradient max |grad - prefill| / weight = "
              f"{float((grad - prefill.double()).abs().max()) / weight:.3g}")
    return grad, prefill.double() + gref, gb, amb_part


def test_loss_plan_sweep():
    for w in LOSS_SWEEP:
        Ls = 9 * w // 2 + 3
        t = wavs(2, Ls, w)
        e = (t + 0.5 * wavs(2, Ls, w + 1)).float()
        check_loss(f"mrl1 sweep w={w} plan={S.make_plan(w)} fpb={S.loss_fpb(w)}", e, t, w, 0.125)


@pytest.mark.parametrize("window,Ls,B", LOSS_MODEL)
def test_loss_model_windows(window, Ls, B):
    t = R.synth_noisy(B, Ls, 16000, seed=window)
    e = (t + 0.3 * R.synth_noisy(B, Ls, 16000, seed=window + 1)).float()
    check_loss(f"mrl1 w={window} L={Ls} B={B} speech-like fpb={S.loss_fpb(window)}", e, t, window, 0.125)
    tn = wavs(B, Ls, window)
    check_loss(f"mrl1 w={window} L={Ls} B={B} white noise", (tn + wavs(B, Ls, 1)).float(), tn, window, 0.125)


@pytest.mark.parametrize("window", [256, 1024, 2048])
def test_loss_edges(window):
    Ls = window // 2 + 1
    t = wavs(3, Ls, 1)
    check_loss(f"mrl1 w={window} L=w/2+1", (t + wavs(3, Ls, 2)).float(), t, window, 0.125)
    t = wavs(2, 5 * window, 3)
    check_loss(f"mrl1 w={window} est = tgt", t.clone(), t, window, 0.125, want_amb_small=False)
    z = torch.zeros(2, 5 * window)
    _, grad = run_loss(z, z, window, 0.125, torch.ones(2, 5 * window), 0.0)
    print(f"mrl1 w={window} digital silence: max |grad - prefill| = {float((grad - 1.0).abs().max()):.3g}")
    assert bool((grad == 1.0).all())


def test_loss_gradient_checker_is_sharp():
    tn = wavs(2, 8192, 5)
    grad, ref, bound, amb_part = check_loss("mrl1 sharpness base", (tn + wavs(2, 8192, 6)).float(), tn, 512, 0.125)
    clean = (amb_part == 0).nonzero()
    assert clean.shape[0] > 0, "every sample is covered by an ambiguous bin"
    b, i = clean[clean.shape[0] // 2].tolist()
    bad = grad.clone()
    bad[b, i] += 3.0 * bound[b, i]
    assert worst_ratio(bad, ref, bound) > 1.0, "one gradient sample 3x its bound off passes"


def test_loss_time_term():
    """L not a multiple of 256 and larger than 64 blocks x 1024 (the grid-stride loop)."""
    L = _lib()
    for Ls, B in ((64 * 1024 + 777, 3), (1000, 1), (300001, 2)):
        t = wavs(B, Ls, Ls)
        e = t.clone()
        e[:, ::3] += wavs(B, Ls, 2)[:, ::3]                      # a third of the samples differ, the rest are equal (sgn 0)
        prefill = wavs(B, Ls, 9)
        grad = sentinel(B * Ls)
        grad[:B * Ls] = prefill.reshape(-1).cuda()
        loss = sentinel(B, torch.float64)
        loss[:B] = 0.25
        ec, tc = e.cuda(), t.cuda()
        L.call("bsrnn_l1_time_fwd_bwd", ec.data_ptr(), tc.data_ptr(), loss.data_ptr(), grad.data_ptr(), B, Ls, 0.5,
               L.stream_ptr())
        torch.cuda.synchronize()
        guard_ok(grad, B * Ls, "l1_time grad")
        guard_ok(loss, B, "l1_time loss")
        value, gref, vb, gb = S.loss_time_ref(e, t, 0.5, prefill)
        assert_within(f"l1_time L={Ls} B={B} value", loss[:B].cpu(), 0.25 + value, vb)
        assert_within(f"l1_time L={Ls} B={B} grad", grad[:B * Ls].view(B, Ls).double().cpu(), gref, gb)
