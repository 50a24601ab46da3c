"""f64 references and elementwise error bounds of the spectral kernels (csrc/fft.cu, csrc/fft_core.cuh, csrc/loss.cu), and a
restatement of their launchers' geometry choices.  Used by tests/test_gpu_spectral.py; validated on the CPU by
tests/test_spectral_ref_cpu.py.  Nothing here reads a kernel's output.

Notation: u = 2^-24 (unit roundoff of f32, round to nearest).  All bounds are first order in u; the second-order terms are
below u^2 C^2 ~ 1e-6 of the first-order ones at the largest C used here and are not carried.

FFT.  fft_core.cuh computes a Stockham transform: stage s applies, to every group of R_s elements, twiddles
tw[q k tstep] and then an R_s-point DFT.  In exact arithmetic a stage multiplies the 2-norm of the data by sqrt(R_s)
(twiddles are unit, the R-point DFT matrix is sqrt(R) times unitary), so the data after stage s has norm
sqrt(R_1 .. R_s) ||z||, and an error of norm e introduced at stage s leaves the transform with norm
e sqrt(R_{s+1} .. R_S).  If stage s adds at most c(R_s) u times the norm of its own output, the result is within
    ||dZ||_2 <= u C_plan ||Z||_2,     C_plan = sum_s c(R_s) (+ the pair split),   ||Z||_2 = sqrt(N) ||z||_2,
and every bin of it within the same amount.  c(R) per butterfly (complex roundings are u |result| per component pair):
  * twiddle product cmul(v, tw): the f32 table entry is off by at most u (cos, sin each rounded once from double) and the
    product adds at most 2 sqrt(2) u (two roundings per component, each of |v| |tw|): 4 u |v| per twiddled element, i.e.
    4 u ||o|| after the butterfly (a norm-sqrt(R) map of the twiddled vector).                                     -> 4
  * radix 2: one complex add, u ||o||.                                                       c(2) = 4 + 1 = 5
  * radix 4: two levels of complex adds (a, b, c, d then o), each u times the norm of its result, the first one carried
    through a sqrt(2)-norm level: sqrt(2) u sqrt(2) ||v|| = u ||o||, and u ||o||.               c(4) = 4 + 1 + 1 = 6
  * radix 3, 5, 7 and the generic radix R: o_p = v_0 + sum_{q=1}^{R-1} v_q w_pq, R - 1 complex multiply-adds with
    f32-rounded w.  Per component 2R - 1 real operations in one chain: gamma_{2R-1} <= (2R-1) u times the sum of the
    absolute terms, <= sqrt(2) sum_q |v_q| per component, so 2 (2R-1) u sum_q |v_q| complex; the rounded w adds
    u sum_q |v_q|.  sum_q |v_q| <= sqrt(R) ||v||, over R outputs sqrt(R) times that, and ||o|| = sqrt(R) ||v||:
                                                                                              c(R) = 4 + (4R - 1) sqrt(R)
  * pair split X_a = (Z_k + conj Z_{N-k}) / 2 (and X_b): the carried error averages two bin errors (no growth); the two
    roundings are u (|Z_k| + |Z_{N-k}|) / sqrt(2) <= u ||Z||_2.                                                  -> + 1
    The iSTFT's pair build (Z_k = V_a + j V_b, one add per component) is the same kind of step before its inverse.
Z is the transform of the PAIR z = x_a + j x_b (frames 2j, 2j+1 of the STFT and of the adjoint; estimate + j target in the
loss; in the iSTFT two frames of a batch starting at the block's first frame tlo, bounded here by the frame and the louder of
its two neighbours), so ||z||^2 = ||x_a||^2 + ||x_b||^2 and a frame's bins carry the rounding of its partner.

Window.  The kernels take w_n = 0.5 - 0.5 Re tw[n]: the f32 cosine is off by at most u |cos| (rounded once from the double
sincospi, whose own error ~1e-16 is below 2^-50), 0.5 c is exact, the subtraction rounds once:
    |w_f32 - w| <= u/2 |cos| + u w + 2^-50                                               (WIN_ERR; not the f64 Hann)
and every product with a sample rounds once more (u).

__powf (compression).  CUDA C++ Programming Guide, "Intrinsic Functions", single-precision table: __powf(x, y) "derived
from its implementation as exp2f(y * __log2f(x))"; __log2f: absolute error 2^-22 for x in [0.5, 2], 2 ulp otherwise; exp2f:
2 ulp (standard-functions table).  So with a = y log2 x:  relative error <= ln 2 (|y| 2^-22 max(1, |log2 x|) + u |a|)
+ 2^-22 (the product y * log2 rounds once).  Inputs are assumed normal (|z| >= 2^-126): __log2f flushes subnormals.

Envelope.  The iSTFT and its adjoint sum w_f32^2 over the frames covering a sample in f32 (m terms: m u of the sum), each
square off by 2 w dw + u w^2; a sample whose f64 envelope is within that of 1e-11 may be written as 0 or as the quotient.
"""
import math

import torch
import torch.nn.functional as F

U = 2.0 ** -24
U53 = 2.0 ** -53
ENV_EPS = 1e-11                      # fft.cu: env > 1e-11 (the threshold torch.istft checks)
MAX_GENERIC_RADIX = 96               # fft_core.cuh kMaxGenericRadix: v[96] of the generic butterfly
MAX_STAGES = 16                      # fft_core.cuh kMaxStages
SMEM_LIMIT = 100 * 1024              # launchers: dynamic shared memory budget


# ------------------------------------------------------------------------------------------------------- plans and geometry
def make_plan(n):
    """fft_core.cuh make_plan: radices 4, 2, 3, 5, 7 greedily, then odd primes up to 96; None where it returns false."""
    radix, m = [], n
    for r in (4, 2, 3, 5, 7):
        while m % r == 0:
            if len(radix) >= MAX_STAGES:
                return None
            radix.append(r)
            m //= r
    r = 11
    while m > 1:
        while m % r == 0:
            if len(radix) >= MAX_STAGES or r > MAX_GENERIC_RADIX:
                return None
            radix.append(r)
            m //= r
        if r > MAX_GENERIC_RADIX and m > 1:
            return None
        r += 2
    return radix


def c_radix(r):
    """per-stage constant c(R) of the module docstring."""
    if r == 2:
        return 5.0
    if r == 4:
        return 6.0
    return 4.0 + (4 * r - 1) * math.sqrt(r)


def c_plan(n):
    """C_plan of an n-point transform: the stages of make_plan(n) plus the pair split / pair build (+1)."""
    plan = make_plan(n)
    assert plan is not None, n
    return sum(c_radix(r) for r in plan) + 1.0


def stft_fpb(n_fft):
    """fft.cu stft_smem_fpb (STFT and iSTFT adjoint): frames per CTA."""
    fpb = 8
    while fpb > 2 and n_fft * 8 * (1 + 2 * ((fpb + 1) // 2)) > SMEM_LIMIT:
        fpb >>= 1
    return fpb


def istft_geometry(n_fft, hop, T, L_out):
    """fft.cu bsrnn_istft_fwd: (fpb, overlap, G, span, nblocks)."""
    G, fpb = 8, 8
    while fpb > 2 and n_fft * 8 * (1 + 2 * ((fpb + 1) // 2)) + G * hop * 4 > SMEM_LIMIT:
        fpb >>= 1
    overlap = (n_fft + hop - 1) // hop - 1
    if fpb - overlap >= 4:
        G = fpb - overlap
    span = G * hop
    nblocks = max(-(-(n_fft // 2 + L_out) // span), -(-T // G))
    return fpb, overlap, G, span, nblocks


def loss_fpb(window):
    """loss.cu bsrnn_mrl1_spec_fwd_bwd: frames per CTA."""
    fpb = 8
    while fpb > 1 and window * 8 * (1 + 2 * fpb) > SMEM_LIMIT:
        fpb >>= 1
    return fpb


def n_frames(L, hop):
    """T = 1 + L / hop (bsrnn_stft_fwd, runtime.stft)."""
    return 1 + L // hop


def olens(lens, L, n_fft, hop, B):
    """frames >= olen[b] = (len + 2 (n_fft/2) - n_fft) / hop + 1 are written as zeros (include/bsrnn_b200.h)."""
    lens = [L] * B if lens is None else [int(v) for v in lens]
    return [(v + 2 * (n_fft // 2) - n_fft) // hop + 1 for v in lens]


# ------------------------------------------------------------------------------------------------------- small pieces
def twiddles(n):
    """exp(-2 pi i n / N), f64 (B,) complex."""
    k = torch.arange(n, dtype=torch.float64)
    return torch.polar(torch.ones_like(k), -2.0 * math.pi * k / n)


def hann(n):
    return torch.hann_window(n, periodic=True, dtype=torch.float64)


def win_err(n):
    """|w_f32 - w| per n (module docstring)."""
    c = torch.cos(2.0 * math.pi * torch.arange(n, dtype=torch.float64) / n).abs()
    return 0.5 * U * c + U * hann(n) + 2.0 ** -50


def rel_pow_err(xlo, xhi, y, dy=0.0):
    """relative error of __powf(x, y) for x in [xlo, xhi] (module docstring), plus |ln x| dy for an exponent that is
    itself off by dy."""
    lo = xlo.clamp(min=2.0 ** -126)
    hi = xhi.clamp(min=2.0 ** -126)
    lg = torch.maximum(torch.log2(lo).abs(), torch.log2(hi).abs())
    return (math.log(2.0) * (abs(y) * 2.0 ** -22 * lg.clamp(min=1.0) + U * abs(y) * lg) + 2.0 ** -22
            + math.log(2.0) * lg * dy)


def power_map_bound(m, d, p, scale, dy=0.0):
    """Error of the kernel's  scale * |z|^(p-1) * z  when its z is within d of a value of magnitude m, against the f64
    scale * m^p * phase.  Interval arithmetic over |z| in [max(0, m - d), m + d] (covers |z| at or below its own error),
    the direction error |z/|z| - Z/|Z|| <= 2 d / |Z| (<= 2), and the kernel's own roundings: |z| (sum of squares + sqrtf,
    2u, carried with exponent p - 1), __powf, and the products by scale and by z (2u)."""
    hi = m + d
    lo = (m - d).clamp(min=0.0)
    mag = scale * torch.maximum(hi ** p - m ** p, m ** p - lo ** p)
    dirn = torch.where(m > 0, torch.clamp(2.0 * d / m.clamp(min=1e-300), max=2.0), torch.zeros_like(m))
    rnd = 2.0 * U * abs(p - 1.0) + rel_pow_err(lo, hi, p - 1.0, dy) + 2.0 * U
    return mag + scale * hi ** p * (dirn + rnd)


def f32(v):
    """a Python float as the kernel receives it (c_float)."""
    return float(torch.tensor(v, dtype=torch.float32))


# ------------------------------------------------------------------------------------------------------- STFT
def frames_of(wav, n_fft, hop, T):
    """windowed (B, T, N) f64 frames of the reflect-padded rows (center=True), zero frames past the end of the padding."""
    x = wav.double()
    pad = F.pad(x[:, None, :], (n_fft // 2, n_fft // 2), mode="reflect")[:, 0]
    fr = pad.unfold(-1, n_fft, hop)
    out = torch.zeros(x.shape[0], T, n_fft, dtype=torch.float64)
    out[:, :fr.shape[1]] = fr[:, :T]
    return out


def stft_ref(wav, lens, n_fft, hop, transform=0, exponent=1.0, factor=1.0):
    """f64 STFT of the f32 rows as stored: torch.stft (periodic Hann, center=True, reflect padding over all L samples), frames
    >= olen zero, then the optional compression factor |X|^e e^{j arg X}.  Returns (spec (B,T,F) complex, bound (B,T,F)
    per element: a bound on the complex modulus |kernel - ref|, so on each component too)."""
    B, L = wav.shape
    T = n_frames(L, hop)
    Fb = n_fft // 2 + 1
    x = wav.double()
    X = torch.stft(x, n_fft, hop, n_fft, hann(n_fft), center=True, pad_mode="reflect", onesided=True,
                   return_complex=True).transpose(1, 2)
    spec = torch.zeros(B, T, Fb, dtype=torch.complex128)
    spec[:, :X.shape[1]] = X[:, :T]
    ol = olens(lens, L, n_fft, hop, B)
    live = torch.arange(T)[None, :] < torch.tensor(ol)[:, None]                          # (B, T)
    spec[~live] = 0
    raw = frames_of(wav, n_fft, hop, T)                                                   # unwindowed
    xw = raw * hann(n_fft)
    energy = torch.where(live, (xw ** 2).sum(-1), torch.zeros(()))
    t = torch.arange(T)
    partner = t ^ 1
    pe = torch.zeros(B, T, dtype=torch.float64)
    ok = partner < T
    pe[:, ok] = energy[:, partner[ok]]
    pe = torch.where(live, pe, torch.zeros(()))
    fft_err = U * c_plan(n_fft) * math.sqrt(n_fft) * torch.sqrt(energy + pe)
    in_err = (raw.abs() * (win_err(n_fft) + U * hann(n_fft))).sum(-1)                     # window + product rounding
    bound = (fft_err + in_err)[..., None].expand(B, T, Fb).clone()
    if transform == 1:
        e, fa = f32(exponent), f32(factor)
        m = spec.abs()
        spec = torch.where(m > 0, fa * m ** e * torch.exp(1j * spec.angle()), torch.zeros((), dtype=torch.complex128))
        bound = power_map_bound(m, bound, e, fa)
    bound = torch.where(live[..., None], bound, torch.zeros(()))
    return spec, bound


# ------------------------------------------------------------------------------------------------------- iSTFT
def masked_ref(spec, mask=None, resid=None):
    """s = m x + r in f64 of the f32 inputs ((B,T,F,2) real views), and the f32 arithmetic's bound (3 roundings per
    component: 3u (sqrt(2) |m| |x| + |r|))."""
    x = torch.view_as_complex(spec.double().contiguous())
    if mask is None:
        return x, torch.zeros(x.shape, dtype=torch.float64)
    m = torch.view_as_complex(mask.double().contiguous())
    r = torch.view_as_complex(resid.double().contiguous())
    return m * x + r, 3.0 * U * (math.sqrt(2.0) * m.abs() * x.abs() + r.abs())


def decompress_ref(s, ds, exponent, factor):
    """the iSTFT's inverse compression |s / factor|^(1/e) e^{j arg s} and its bound (inv_factor = fl(1/factor): 2u on the
    scaled value; 1/e rounded once: the exponent is off by u / e)."""
    e, fa = f32(exponent), f32(factor)
    m = s.abs() / fa
    d = ds / fa + 2.0 * U * m
    out = torch.where(m > 0, m ** (1.0 / e) * torch.exp(1j * s.angle()), torch.zeros((), dtype=torch.complex128))
    return out, power_map_bound(m, d, 1.0 / e, 1.0, dy=U / e)


def _ola(frames, hop, P):
    """overlap-add (B, T, N) -> (B, P)."""
    B, T, N = frames.shape
    return F.fold(frames.transpose(1, 2), output_size=(1, P), kernel_size=(1, N), stride=(1, hop))[:, 0, 0]


def _hermitian_l1(v, n_fft):
    """sum over all N bins of the Hermitian extension of one-sided magnitudes v (..., F)."""
    w = torch.full((v.shape[-1],), 2.0, dtype=torch.float64)
    w[0] = 1.0
    if n_fft % 2 == 0:
        w[-1] = 1.0
    return (v * w).sum(-1)


def istft_ref(v, n_fft, hop, L_out):
    """Explicit f64 overlap-add iSTFT of (B,T,F) complex: irfft per frame with Im of DC / Nyquist ignored, periodic Hann,
    overlap-add, division by the window-square envelope where env > 1e-11 (0 elsewhere), trim n_fft/2, L_out samples (zeros
    past the last frame)."""
    B, T, Fb = v.shape
    v = v.clone()
    v[..., 0] = v[..., 0].real
    if n_fft % 2 == 0:
        v[..., -1] = v[..., -1].real
    fr = torch.fft.irfft(v, n=n_fft)                                                     # (B, T, N)
    w = hann(n_fft)
    P = (T - 1) * hop + n_fft
    y = _ola(fr * w, hop, P)
    env = _ola((w * w).expand(1, T, n_fft), hop, P)[0]
    yo = torch.where(env > ENV_EPS, y / torch.where(env > ENV_EPS, env, torch.ones(())), torch.zeros(()))
    h = n_fft // 2
    out = torch.zeros(B, L_out, dtype=torch.float64)
    n = max(0, min(L_out, P - h))
    out[:, :n] = yo[:, h:h + n]
    return out


def istft_bound(v, dv, n_fft, hop, L_out):
    """Elementwise bound of bsrnn_istft_fwd's wav_out against istft_ref(v) when the kernel's one-sided spectra are within
    dv of v (module docstring: inverse FFT of the frame pair, the 1/N and window products, the overlap-add and envelope
    sums, the quotient and its threshold).  Returns (bound (B, L_out), straddle mask where 0 is also acceptable)."""
    B, T, Fb = v.shape
    N = n_fft
    vv = v.clone()
    vv[..., 0] = vv[..., 0].real
    if N % 2 == 0:
        vv[..., -1] = vv[..., -1].real
    x = torch.fft.irfft(vv, n=N)                                                         # reference frames (B, T, N)
    mag = v.abs() + dv
    S = _hermitian_l1(mag ** 2, N)                                                       # ||ext V_t||^2 (B, T)
    nb = torch.zeros_like(S)
    nb[:, 1:] = S[:, :-1]
    nb[:, :-1] = torch.maximum(nb[:, :-1], S[:, 1:])
    eps_t = U * c_plan(N) * torch.sqrt(S + nb) / math.sqrt(N) + _hermitian_l1(dv, N) / N   # per-sample frame error
    w = hann(N)
    dw = win_err(N)
    P = (T - 1) * hop + N
    A = _ola(x * w, hop, P)
    absA = _ola(x.abs() * w, hop, P)
    dA_frames = _ola(eps_t[..., None] * w + x.abs() * (dw + 3.0 * U * w), hop, P)
    m = _ola(torch.ones(1, T, N, dtype=torch.float64), hop, P)[0]                        # frames covering each sample
    E = _ola((w * w).expand(1, T, N), hop, P)[0]
    dE = _ola((2.0 * w * dw + dw * dw + U * w * w).expand(1, T, N), hop, P)[0] + m * U * E
    dA = dA_frames + m * U * absA
    Ez = torch.where(E > 0, E, torch.ones(()))
    q = A / Ez
    den = (E - dE).clamp(min=1e-300)
    bnd = (dA + q.abs() * dE) / den + U * (A.abs() + dA) / den
    sure = E - dE > ENV_EPS
    never = E + dE <= ENV_EPS
    straddle = ~sure & ~never
    bnd = torch.where(sure, bnd, torch.zeros(()))
    bnd = torch.where(straddle, bnd + q.abs(), bnd)
    h = N // 2
    out = torch.zeros(B, L_out, dtype=torch.float64)
    st = torch.zeros(L_out, dtype=torch.bool)
    n = max(0, min(L_out, P - h))
    out[:, :n] = bnd[:, h:h + n]
    st[:n] = straddle[h:h + n]
    return out, st


# ------------------------------------------------------------------------------------------------------- iSTFT adjoint
def _edge_weights(n_fft, Fb):
    c = torch.full((Fb,), 2.0, dtype=torch.float64)
    c[0] = 1.0
    if n_fft % 2 == 0:
        c[-1] = 1.0
    return c / n_fft


def istft_bwd_ref(g, T, n_fft, hop):
    """f64 transpose of istft_ref (no mask, no compression): g (B, L_out) -> (B, T, F) complex; bin k of frame t is
    c_k / N * DFT(w * g_pad[t hop + n] / env), c_0 = c_{N/2} = 1 else 2, Im of DC / Nyquist zero, g_pad zero outside the
    trimmed range and where env <= 1e-11."""
    B, L_out = g.shape
    N = n_fft
    P = (T - 1) * hop + N
    h = N // 2
    gp = torch.zeros(B, P, dtype=torch.float64)
    n = max(0, min(L_out, P - h))
    gp[:, h:h + n] = g.double()[:, :n]
    w = hann(N)
    env = _ola((w * w).expand(1, T, N), hop, P)[0]
    y = torch.where(env > ENV_EPS, gp / torch.where(env > ENV_EPS, env, torch.ones(())), torch.zeros(()))
    fr = y.unfold(-1, N, hop)[:, :T] * w
    X = torch.fft.rfft(fr, n=N) * _edge_weights(N, N // 2 + 1)
    X[..., 0] = X[..., 0].real
    if N % 2 == 0:
        X[..., -1] = X[..., -1].real
    return X


def istft_bwd_bound(g, T, n_fft, hop):
    """Elementwise bound of bsrnn_istft_bwd against istft_bwd_ref: per sample the f32 envelope (dE), the products by w and the
    quotient (2u), the window error; per frame the DFT of the pair (2j, 2j+1); then c_k / N (2u)."""
    B, L_out = g.shape
    N = n_fft
    P = (T - 1) * hop + N
    h = N // 2
    gp = torch.zeros(B, P, dtype=torch.float64)
    n = max(0, min(L_out, P - h))
    gp[:, h:h + n] = g.double()[:, :n].abs()
    w = hann(N)
    dw = win_err(N)
    E = _ola((w * w).expand(1, T, N), hop, P)[0]
    m = _ola(torch.ones(1, T, N, dtype=torch.float64), hop, P)[0]
    dE = _ola((2.0 * w * dw + dw * dw + U * w * w).expand(1, T, N), hop, P)[0] + m * U * E
    sure = E - dE > ENV_EPS
    never = E + dE <= ENV_EPS
    den = torch.where(sure, E - dE, torch.ones(()))
    inv = torch.where(sure, 1.0 / den, torch.zeros(()))
    straddle_inv = torch.where(~sure & ~never, 1.0 / torch.full_like(E, ENV_EPS), torch.zeros(()))
    gf = gp.unfold(-1, N, hop)[:, :T]                                                  # |g| per frame sample
    invf = inv.unfold(-1, N, hop)[:T]
    dEf = dE.unfold(-1, N, hop)[:T]
    stf = straddle_inv.unfold(-1, N, hop)[:T]
    y = gf * w * invf                                                                  # |y| (upper, with E - dE)
    dy = gf * (dw * invf + w * dEf * invf * invf + 2.0 * U * w * invf) + gf * w * stf
    energy = ((y + dy) ** 2).sum(-1)                                                    # (B, T)
    t = torch.arange(T)
    partner = t ^ 1
    pe = torch.zeros_like(energy)
    ok = partner < T
    pe[:, ok] = energy[:, partner[ok]]
    fft_err = U * c_plan(N) * math.sqrt(N) * torch.sqrt(energy + pe) + dy.sum(-1)
    c = _edge_weights(N, N // 2 + 1)
    ref_mag = c * (y.sum(-1, keepdim=True))                                             # |bin| <= c/N sum |y|
    return c * fft_err[..., None] + 2.0 * U * (ref_mag + c * fft_err[..., None])


def real_inner(a, b, n_fft):
    """real inner product over (re, im) pairs of two (B,T,F) complex spectra, the imaginary parts of DC and Nyquist
    excluded."""
    a, b = a.clone(), b.clone()
    a[..., 0] = a[..., 0].real
    b[..., 0] = b[..., 0].real
    if n_fft % 2 == 0:
        a[..., -1] = a[..., -1].real
        b[..., -1] = b[..., -1].real
    return float((a.real * b.real + a.imag * b.imag).sum())


# ------------------------------------------------------------------------------------------------------- loss
def reflect_index(L, T, N, hop):
    """(T, N) sample index of frame t, offset n under center=True reflect padding (loss.cu reflect_index)."""
    i = torch.arange(T)[:, None] * hop - N // 2 + torch.arange(N)[None, :]
    i = torch.where(i < 0, -i, i)
    return torch.where(i >= L, 2 * (L - 1) - i, i)


def loss_spec_ref(est, tgt, window, weight):
    """MultiResL1SpecLoss spectral core at one window: rectangular window, hop w/2, center=True reflect padding, one-sided.
    value[b] = weight sum | |E| - |T| |; grad[b, n] = d value / d est[b, n] with sgn(0) = 0 and a zero phasor at |E| = 0.
    Returns (value (B,), grad (B, L), per-bin data for the bounds)."""
    e, t = est.double(), tgt.double()
    B, L = e.shape
    N, hop = window, window // 2
    kw = dict(n_fft=N, hop_length=hop, win_length=N, window=torch.ones(N, dtype=torch.float64), center=True,
              pad_mode="reflect", onesided=True, return_complex=True)
    E = torch.stft(e, **kw).transpose(1, 2)                                              # (B, T, F)
    Tt = torch.stft(t, **kw).transpose(1, 2)
    me, mt = E.abs(), Tt.abs()
    d = me - mt
    value = weight * d.abs().sum(dim=(1, 2))
    phasor = torch.where(me > 0, E / torch.where(me > 0, me, torch.ones(())).to(E.dtype), torch.zeros((), dtype=E.dtype))
    G = weight * torch.sign(d) * phasor
    T = E.shape[1]
    Fb = N // 2 + 1                                  # Re sum_{k<F} G_k e^{+j..}: irfft doubles 0 < k < N/2, reads Re G_0, G_N/2
    cw = torch.full((Fb,), 0.5, dtype=torch.float64)
    cw[0] = 1.0
    cw[-1] = 1.0
    fr = torch.fft.irfft(G * cw, n=N) * N
    idx = reflect_index(L, T, N, hop).reshape(-1)
    grad = torch.zeros(B, L, dtype=torch.float64)
    grad.index_add_(1, idx, fr.reshape(B, -1))
    frames = torch.stack([e[:, reflect_index(L, T, N, hop)], t[:, reflect_index(L, T, N, hop)]])   # (2, B, T, N)
    return value, grad, dict(E=E, T=Tt, d=d, frames=frames, idx=idx, T_frames=T)


def loss_spec_bound(est, tgt, window, weight, info, prefill_abs):
    """Bounds of bsrnn_mrl1_spec_fwd_bwd (module docstring): per bin |E| and |T| within dE = u C_plan sqrt(N) ||(e, t)_frame||
    (+2u |E| for the f32 magnitude); a bin is AMBIGUOUS when its f64 margin | |E| - |T| | is within the two magnitude bounds
    or |E| is within its own bound, and may then put up to 2 weight into every sample its frame covers; any other bin puts
    weight (2 dE / |E| + 4u) (phasor error; the product by s and the division by |E| round once each, |E| itself 2u).
    Per frame and sample: the sum over bins, plus the inverse transform u C_plan sqrt(N) ||G||_2 (||G|| <= weight sqrt(F)).
    Per sample: sum over the (frame, offset) pairs that reflect onto it, plus the f32 atomicAdd order (m adds of terms
    <= weight F, and the prefill).  Value: weight sum (dE + dT + u |d|) plus the double sums.
    Returns (value bound (B,), grad bound (B, L), the part of it from ambiguous bins (B, L), ambiguous mask (B,T,F))."""
    N = window
    Fb = N // 2 + 1
    B, L = est.shape
    E, Tt, d, frames = info["E"], info["T"], info["d"], info["frames"]
    energy = (frames ** 2).sum(-1).sum(0)                                                # (B, T)
    dZ = U * c_plan(N) * math.sqrt(N) * torch.sqrt(energy)[..., None]
    me, mt = E.abs(), Tt.abs()
    dme = dZ + 2.0 * U * (me + dZ)
    dmt = dZ + 2.0 * U * (mt + dZ)
    amb = (d.abs() <= dme + dmt + U * (me + mt)) | (me <= dme)
    phase = 2.0 * dZ / me.clamp(min=1e-300) + 4.0 * U
    dG = torch.where(amb, torch.full_like(me, 2.0 * (1.0 + 2.0 * U)), phase) * weight
    per_frame = dG.sum(-1) + U * c_plan(N) * math.sqrt(N) * weight * math.sqrt(Fb)      # (B, T)
    amb_frame = (amb.double() * 2.0 * (1.0 + 2.0 * U) * weight).sum(-1)
    T = E.shape[1]
    idx = info["idx"]

    def scatter(v):
        out = torch.zeros(B, L, dtype=torch.float64)
        out.index_add_(1, idx, v[..., None].expand(B, T, N).reshape(B, -1))
        return out
    mult = torch.zeros(L, dtype=torch.float64)
    mult.index_add_(0, idx, torch.ones(idx.numel(), dtype=torch.float64))
    gb = scatter(per_frame) + (mult + 1.0) * U * (prefill_abs + mult * weight * Fb * (1.0 + 4.0 * U))
    count = E.shape[1] * Fb
    vb = weight * (dme + dmt + U * d.abs()).sum(dim=(1, 2)) + (count + 64) * U53 * weight * (me + mt).sum(dim=(1, 2))
    return vb, gb, scatter(amb_frame), amb


def loss_time_ref(est, tgt, weight, prefill):
    """time-domain term: value weight sum |e - t| (f32 subtraction: u |e - t| each), gradient prefill + weight sgn(e - t)
    (the f32 difference has the sign of the exact one; the one f32 add rounds: u |result|)."""
    d = est.double() - tgt.double()
    value = weight * d.abs().sum(-1)
    vb = weight * U * d.abs().sum(-1) + (d.shape[-1] + 64) * U53 * value.abs()
    grad = prefill.double() + weight * torch.sign(d)
    return value, grad, vb, U * grad.abs()


# ------------------------------------------------------------------------------------------------------- band statistics
def band_stats_ref(spec, edges):
    """per (b, band) sum of re + im and sum of re^2 + im^2 over bins [edges[k], min(edges[k+1], F)) of a (B,T,F) complex
    spectrum (0 for bands starting at or beyond F), f64; and the sums of |re| + |im| and of the squares for the bounds."""
    B, T, Fb = spec.shape
    K = len(edges) - 1
    s = torch.zeros(B, K, 2, dtype=torch.float64)
    a = torch.zeros(B, K, 2, dtype=torch.float64)
    n = torch.zeros(K, dtype=torch.float64)
    for k in range(K):
        k0, k1 = edges[k], min(edges[k + 1], Fb)
        if k0 >= Fb:
            continue
        v = spec[:, :, k0:k1]
        s[:, k, 0] = (v.real + v.imag).sum(dim=(1, 2))
        s[:, k, 1] = (v.real ** 2 + v.imag ** 2).sum(dim=(1, 2))
        a[:, k, 0] = (v.real.abs() + v.imag.abs()).sum(dim=(1, 2))
        a[:, k, 1] = s[:, k, 1]
        n[k] = 2 * T * (k1 - k0)
    return s, a, n
