"""CPU tests of tests/spectral_ref.py, the f64 references and launcher restatements the spectral GPU tests
(tests/test_gpu_spectral.py) check the kernels against: the STFT against the oracle's restated encoder, the overlap-add iSTFT
against torch.istft where that is defined, its transpose against autograd (through the restatement and through torch.istft),
the loss core against autograd and the oracle's MultiResL1SpecLoss, and the geometry classes the GPU cases rely on."""
import math

import pytest
import torch

import spectral_ref as S
from oracle import restated as R

SE_SIZES = [(160, 80), (320, 160), (441, 220), (480, 240), (640, 320), (882, 441), (960, 480)]
FLOWSE_SIZES = [(256, 64), (512, 128), (705, 176), (768, 192), (1024, 256), (1411, 352), (1536, 384)]


def test_model_sizes_are_the_stft_dims_of_every_rate():
    rates = (8000, 16000, 22050, 24000, 32000, 44100, 48000)
    assert [R.stft_dims(fs, 960, 480) for fs in rates] == SE_SIZES
    assert [R.stft_dims(fs, 1536, 384) for fs in rates] == FLOWSE_SIZES


def test_plan_restatement_accepts_and_rejects_what_the_factoriser_does():
    assert S.make_plan(705) == [3, 5, 47] and S.make_plan(1411) == [17, 83] and S.make_plan(1536) == [4, 4, 4, 4, 2, 3]
    assert S.make_plan(89) == [89]
    for n in (97, 194, 101, 2 * 101, 199):
        assert S.make_plan(n) is None
    for n in range(4, 201):
        big = max(p for p in range(2, n + 1) if n % p == 0 and all(p % q for q in range(2, p)))
        assert (S.make_plan(n) is None) == (big > 96), n
        if S.make_plan(n):
            assert math.prod(S.make_plan(n)) == n


def test_geometry_classes_of_the_model_sizes():
    assert {S.stft_fpb(n) for n, _ in SE_SIZES + FLOWSE_SIZES if n != 1536} == {8}
    assert S.stft_fpb(1536) == 4 and S.stft_fpb(2048) == 4 and S.stft_fpb(3072) == 2
    assert 1411 * 8 * 9 <= S.SMEM_LIMIT < 1536 * 8 * 9                       # 1411 just under the 8-frame limit
    cls = {(n, h): S.istft_geometry(n, h, 100, 100 * h)[::2][:2] for n, h in SE_SIZES + FLOWSE_SIZES}
    assert {cls[s] for s in SE_SIZES if s != (441, 220)} == {(8, 7)}
    assert cls[(441, 220)] == (8, 6) and cls[(705, 176)] == (8, 4)
    assert {cls[s] for s in FLOWSE_SIZES if s[0] in (256, 512, 768, 1024)} == {(8, 5)}
    assert cls[(1411, 352)] == (4, 8) and cls[(1536, 384)] == (4, 8)
    assert S.istft_geometry(3072, 768, 10, 100)[::2][:2] == (2, 8) and S.istft_geometry(2048, 512, 10, 100)[0] == 4
    assert [S.loss_fpb(w) for w in (256, 512, 768, 1024, 2048)] == [8, 8, 4, 4, 2]
    # nblocks from cdiv(T, G) when L_out is short
    fpb, ov, G, span, nb = S.istft_geometry(960, 480, 40, 1)
    assert nb == -(-40 // G) > -(-(480 + 1) // span)


def test_twiddles_and_window():
    for n in (4, 7, 705, 1411):
        tw = S.twiddles(n)
        assert torch.allclose(tw, torch.exp(-2j * math.pi * torch.arange(n, dtype=torch.float64) / n), atol=1e-15)
        w32 = 0.5 - 0.5 * tw.real.float()
        assert bool(((w32.double() - S.hann(n)).abs() <= S.win_err(n)).all())


@pytest.mark.parametrize("n_fft,hop", [(160, 80), (441, 220), (705, 176), (16, 4), (9, 4)])
@pytest.mark.parametrize("transform", [0, 1])
def test_stft_ref_is_the_restated_encoder(n_fft, hop, transform):
    g = torch.Generator().manual_seed(n_fft)
    L = 7 * hop + 3
    wav = torch.randn(3, L, generator=g).float()
    lens = torch.tensor([L, L - hop - 1, n_fft // 2 + 1])
    spec, bound = S.stft_ref(wav, lens, n_fft, hop, transform, 0.5, 0.15)
    ref, ol = R.stft_encode(wav.double(), lens, 48000, n_fft, hop, 48000, "exponent" if transform else None,
                            S.f32(0.5), S.f32(0.15))
    Tr = ref.shape[1]
    assert torch.allclose(spec[:, :Tr], ref, atol=1e-12, rtol=1e-12)
    assert bool((spec[:, Tr:] == 0).all())
    assert ol.tolist() == S.olens(lens, L, n_fft, hop, 3)
    live = torch.arange(spec.shape[1])[None, :] < ol[:, None]
    assert bool((bound[~live] == 0).all()) and bool((bound[live] > 0).all())


def _rand_spec(B, T, Fb, seed):
    g = torch.Generator().manual_seed(seed)
    return torch.complex(torch.randn(B, T, Fb, generator=g, dtype=torch.float64),
                         torch.randn(B, T, Fb, generator=g, dtype=torch.float64))


@pytest.mark.parametrize("n_fft,hop,T", [(160, 80, 9), (441, 220, 6), (705, 176, 8), (1536, 384, 5), (9, 4, 7), (16, 4, 3)])
def test_istft_ref_matches_torch_istft(n_fft, hop, T):
    v = _rand_spec(2, T, n_fft // 2 + 1, n_fft)                     # not Hermitian-consistent: Im of DC / Nyquist nonzero
    for L_out in ((T - 1) * hop, (T - 1) * hop - 3, 1):
        got = S.istft_ref(v, n_fft, hop, L_out)
        ref = torch.istft(v.transpose(1, 2), n_fft, hop, n_fft, S.hann(n_fft), center=True, length=L_out)
        assert torch.allclose(got, ref, atol=1e-12, rtol=1e-10), L_out
    long = S.istft_ref(v, n_fft, hop, (T - 1) * hop + n_fft)
    assert bool((long[:, (T - 1) * hop + n_fft - n_fft // 2:] == 0).all())  # past the last frame: zeros (documented)


@pytest.mark.parametrize("n_fft,hop,T,L_out", [(160, 80, 9, 640), (441, 220, 6, 1099), (9, 4, 7, 23), (16, 4, 3, 40),
                                               (705, 176, 8, 1001)])
def test_istft_adjoint_is_the_transpose(n_fft, hop, T, L_out):
    Fb = n_fft // 2 + 1
    v = _rand_spec(2, T, Fb, 3).requires_grad_(True)
    g = torch.randn(2, L_out, generator=torch.Generator().manual_seed(4), dtype=torch.float64)
    (S.istft_ref(v, n_fft, hop, L_out) * g).sum().backward()
    adj = S.istft_bwd_ref(g, T, n_fft, hop)
    assert torch.allclose(adj, v.grad, atol=1e-12, rtol=1e-10)
    if L_out <= (T - 1) * hop:
        v2 = v.detach().clone().requires_grad_(True)
        out = torch.istft(v2.transpose(1, 2), n_fft, hop, n_fft, S.hann(n_fft), center=True, length=L_out)
        (out * g).sum().backward()
        assert torch.allclose(adj, v2.grad, atol=1e-12, rtol=1e-10)
    lhs = float((S.istft_ref(v.detach(), n_fft, hop, L_out) * g).sum())
    assert abs(lhs - S.real_inner(v.detach(), adj, n_fft)) <= 1e-10 * (abs(lhs) + 1)
    assert bool((S.istft_bwd_bound(g.float(), T, n_fft, hop) > 0).all())


@pytest.mark.parametrize("window,L", [(4, 3), (256, 1000), (512, 257), (1024, 3000)])
def test_loss_ref_matches_autograd_and_the_oracle(window, L):
    g = torch.Generator().manual_seed(window)
    t = torch.randn(2, L, generator=g, dtype=torch.float64)
    e = (t + 0.3 * torch.randn(2, L, generator=g, dtype=torch.float64)).requires_grad_(True)
    kw = dict(n_fft=window, hop_length=window // 2, win_length=window, window=torch.ones(window, dtype=torch.float64),
              center=True, pad_mode="reflect", return_complex=True)
    val = (torch.stft(e, **kw).abs() - torch.stft(t, **kw).abs()).abs().sum(dim=(1, 2)) * 0.25
    val.sum().backward()
    value, grad, _ = S.loss_spec_ref(e.detach(), t, window, 0.25)
    assert torch.allclose(value, val.detach(), rtol=1e-12)
    assert torch.allclose(grad, e.grad, atol=1e-10, rtol=1e-10)
    if L > window // 2 + 2:                                            # the oracle's loss (std / alpha normalisation inside)
        tn = t / torch.std(t, dim=1, keepdim=True)
        en = e.detach() / torch.std(e.detach(), dim=1, keepdim=True)
        alpha = (en * tn).sum(-1, keepdim=True) / ((en ** 2).sum(-1, keepdim=True) + 1e-6)
        want = R.multires_l1_spec_loss(t, e.detach(), window_sz=(window,), time_domain_weight=0.0)
        assert torch.allclose(S.loss_spec_ref(en * alpha, tn, window, 1.0)[0], want, rtol=1e-12)
        want_td = R.multires_l1_spec_loss(t, e.detach(), window_sz=(window,), time_domain_weight=1.0)
        assert torch.allclose(S.loss_time_ref(en * alpha, tn, 1.0, torch.zeros(2, L))[0], want_td, rtol=1e-12)


def test_loss_ref_zero_phasor_and_equal_inputs():
    t = torch.randn(1, 600, generator=torch.Generator().manual_seed(1), dtype=torch.float64)
    value, grad, info = S.loss_spec_ref(t, t, 256, 0.5)
    assert float(value) == 0.0 and bool((grad == 0).all())
    z = torch.zeros(1, 600, dtype=torch.float64)
    value, grad, _ = S.loss_spec_ref(z, t, 256, 0.5)                    # |E| = 0: sgn = -1 but a zero phasor
    assert float(value) > 0 and bool((grad == 0).all())
    vb, gb, amb_part, amb = S.loss_spec_bound(t, t, 256, 0.5, info, 0.0)
    assert bool(amb.all())


def test_band_stats_ref_bands_beyond_F_are_zero():
    v = _rand_spec(2, 5, 17, 0)
    s, a, n = S.band_stats_ref(v, [0, 4, 10, 17, 20, 30])
    assert bool((s[:, 3:] == 0).all()) and n.tolist()[3:] == [0, 0]
    assert torch.allclose(s[:, 1, 1], (v[:, :, 4:10].abs() ** 2).sum(dim=(1, 2)))


def test_power_map_bound_covers_perturbed_inputs():
    """The interval bound contains the exact map of every input within d, including |z| at or below d."""
    g = torch.Generator().manual_seed(0)
    m = torch.cat([torch.rand(2000, generator=g, dtype=torch.float64) * 3, torch.tensor([0.0, 1e-9, 1e-3])])
    d = torch.rand(m.shape, generator=g, dtype=torch.float64) * 0.05
    Z = torch.polar(m, torch.rand(m.shape, generator=g, dtype=torch.float64) * 6.28)
    ang = torch.rand(m.shape, generator=g, dtype=torch.float64) * 6.28
    z = Z + torch.polar(d * torch.rand(m.shape, generator=g, dtype=torch.float64), ang)
    for p, sc in ((0.667, 0.065), (0.5, 0.15), (1 / 0.667, 1.0)):
        f = lambda x: sc * x.abs() ** p * torch.exp(1j * x.angle()) * (x.abs() > 0)
        assert bool(((f(z) - f(Z)).abs() <= S.power_map_bound(m, d, p, sc)).all())
