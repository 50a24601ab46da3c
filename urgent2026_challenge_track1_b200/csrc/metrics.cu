// metrics.cu — intrusive speech-enhancement metrics on the device (metrics.py): ESTOI (pystoi 0.4, extended=True) in four
// stages -- polyphase resampling to 10 kHz, silent-frame removal, one-third octave band envelopes, segment correlation --
// and BSS-eval v3 SDR (512-tap distortion filter, correlations + Levinson recursion in f64).
// Signals are (B, T) f32 rows valid on [0, len[b]); no padded sample is read.  No floating-point atomics and no sum whose
// order depends on the batch: an utterance's scores are bitwise the same alone or inside any ragged batch.
#include <algorithm>

#include "fft_core.cuh"

namespace bsrnn {

constexpr int kMetFrame = 256;          // ESTOI frame (and STFT window) at 10 kHz
constexpr int kMetHop = 128;
constexpr int kMetNfft = 512;
constexpr int kMetBands = 15;
constexpr int kMetSeg = 30;             // frames per correlation segment
constexpr double kMetDynRange = 40.0;   // dB below the loudest frame that still counts as speech
constexpr double kMetEps = 2.220446049250313e-16;   // np.finfo(float).eps

constexpr int kRsThreads = 256;
constexpr int kEnThreads = 256;         // 8 warps = 8 frames per CTA
constexpr int kSelThreads = 1024;
constexpr int kOlaThreads = 256;
constexpr int kBandThreads = 256;
constexpr int kBandFrames = 8;          // STFT frames per CTA
constexpr int kSegThreads = 32;         // one thread per segment
constexpr int kSegWin = kSegThreads + kMetSeg - 1;
constexpr int kRedThreads = 256;

constexpr int kSdrTaps = 512;
constexpr int kSdrChunk = 2048;         // samples per CTA of the correlation kernel
constexpr int kSdrVals = 2 * kSdrTaps + 1;   // acf[0..512), xcorr[0..512), sum inf^2

__device__ __forceinline__ int met_frames(int n) { return n > kMetFrame ? (n - kMetFrame - 1) / kMetHop + 1 : 0; }

// np.hanning(258)[1:-1]
__device__ __forceinline__ double met_hann(int j) { return 0.5 - 0.5 * cospi(2.0 * (j + 1) / 257.0); }

// fixed-order block sum of a double (all threads get the result)
__device__ double met_block_sum(double v, double* red) {
  v = warp_sum(v);
  const int w = threadIdx.x / 32, nw = blockDim.x / 32;
  __syncthreads();
  if (threadIdx.x % 32 == 0) red[w] = v;
  __syncthreads();
  double s = 0.0;
  for (int i = 0; i < nw; ++i) s += red[i];
  return s;
}

// ----------------------------------------------------------------------------------------------- 1. resampling
// grid (cdiv(T_out, 256), B): y[b, m] = sum_i x[b, i] h[k - i up], k = (m + pre_remove) down - pre_pad, over
// 0 <= i < len[b] (scipy.signal.resample_poly with a given window, zero padding).  poly (up, J) holds h by phase:
// poly[ph, j] = h[ph + j up], so output m reads row ph = k mod up from column 0 on, against x[k / up - j].
__global__ void __launch_bounds__(kRsThreads)
met_resample_kernel(const float* __restrict__ x, const int32_t* __restrict__ len, int T, const double* __restrict__ poly,
                    int J, int up, int down, int pre_pad, int pre_remove, float* __restrict__ y, int32_t* __restrict__ y_len,
                    int T_out) {
  const int b = blockIdx.y;
  const int n = len[b];
  const long n_out = ((long)n * up + down - 1) / down;
  const long m = (long)blockIdx.x * kRsThreads + threadIdx.x;
  if (m == 0) y_len[b] = (int)n_out;
  if (m >= T_out) return;
  float* yb = y + (size_t)b * T_out;
  if (m >= n_out) {
    yb[m] = 0.f;
    return;
  }
  const long k = (m + pre_remove) * (long)down - pre_pad;      // >= 0: pre_remove * down >= half_len + pre_pad - down + 1
  const long ih = k / up;
  const double* h = poly + (size_t)(k - ih * up) * J;
  const float* xb = x + (size_t)b * T;
  const int j0 = (int)max(0L, ih - (n - 1)), j1 = (int)min((long)J, ih + 1);
  double acc = 0.0;
  for (int j = j0; j < j1; ++j) acc = fma((double)__ldg(xb + ih - j), __ldg(h + j), acc);
  yb[m] = (float)acc;
}

// ----------------------------------------------------------------------------------------------- 2. silent frames
// grid (cdiv(NF, 8), B): one warp per frame; en[b, t] = 20 log10(||w * x[128 t, 128 t + 256)|| + eps) in f64.
__global__ void __launch_bounds__(kEnThreads)
met_energy_kernel(const float* __restrict__ x, const int32_t* __restrict__ len, int T, int NF, double* __restrict__ en) {
  __shared__ double w[kMetFrame];
  for (int j = threadIdx.x; j < kMetFrame; j += blockDim.x) w[j] = met_hann(j);
  __syncthreads();
  const int b = blockIdx.y, lane = threadIdx.x % 32;
  const int t = blockIdx.x * (kEnThreads / 32) + threadIdx.x / 32;
  if (t >= met_frames(len[b])) return;
  const float* xb = x + (size_t)b * T + (size_t)t * kMetHop;
  double acc = 0.0;
  for (int j = lane; j < kMetFrame; j += 32) {
    const double v = w[j] * (double)xb[j];
    acc = fma(v, v, acc);
  }
  acc = warp_sum(acc);
  if (lane == 0) en[(size_t)b * NF + t] = 20.0 * log10(sqrt(acc) + kMetEps);
}

// grid (B): keep the frames within 40 dB of the loudest; kept[b, j] = index of the j-th kept frame (in order),
// c_len[b] = length of the overlap-added result, (n_kept - 1) 128 + 256 (0 without frames).
__global__ void __launch_bounds__(kSelThreads)
met_select_kernel(const int32_t* __restrict__ len, int NF, const double* __restrict__ en, int32_t* __restrict__ kept,
                  int32_t* __restrict__ c_len) {
  __shared__ double red[kSelThreads / 32];
  __shared__ int cnt[kSelThreads / 32];
  const int b = blockIdx.x, nf = met_frames(len[b]);
  const double* e = en + (size_t)b * NF;
  double mx = -INFINITY;
  for (int t = threadIdx.x; t < nf; t += blockDim.x) mx = fmax(mx, e[t]);
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) mx = fmax(mx, __shfl_xor_sync(0xffffffffu, mx, o));
  const int w = threadIdx.x / 32, lane = threadIdx.x % 32, nw = blockDim.x / 32;
  if (lane == 0) red[w] = mx;
  __syncthreads();
  for (int i = 0; i < nw; ++i) mx = fmax(mx, red[i]);
  int base = 0;
  for (int t0 = 0; t0 < nf; t0 += blockDim.x) {
    const int t = t0 + threadIdx.x;
    const bool keep = t < nf && (mx - kMetDynRange - e[t]) < 0.0;
    const unsigned bal = __ballot_sync(0xffffffffu, keep);
    __syncthreads();                                            // cnt of the previous chunk has been read
    if (lane == 0) cnt[w] = __popc(bal);
    __syncthreads();
    int off = base;
    for (int i = 0; i < w; ++i) off += cnt[i];
    if (keep) kept[(size_t)b * NF + off + __popc(bal & ((1u << lane) - 1u))] = t;
    for (int i = 0; i < nw; ++i) base += cnt[i];
  }
  if (threadIdx.x == 0) c_len[b] = base > 0 ? (base - 1) * kMetHop + kMetFrame : 0;
}

// grid (cdiv(T, 256), B): xc / yc = overlap-add (hop 128) of the windowed kept frames of x / y; zero from c_len[b] on.
__global__ void __launch_bounds__(kOlaThreads)
met_ola_kernel(const float* __restrict__ x, const float* __restrict__ y, int T, int NF, const int32_t* __restrict__ kept,
               const int32_t* __restrict__ c_len, float* __restrict__ xc, float* __restrict__ yc) {
  const int b = blockIdx.y;
  const int s = blockIdx.x * kOlaThreads + threadIdx.x;
  if (s >= T) return;
  const size_t row = (size_t)b * T;
  const int n = c_len[b];
  if (s >= n) {
    xc[row + s] = 0.f;
    yc[row + s] = 0.f;
    return;
  }
  const int nk = (n - kMetFrame) / kMetHop + 1;
  const int32_t* kb = kept + (size_t)b * NF;
  double ax = 0.0, ay = 0.0;
  for (int j = s / kMetHop - 1; j <= s / kMetHop; ++j) {      // frame j - 1 first: the order np's overlap-add adds in
    if (j < 0 || j >= nk) continue;
    const int o = s - j * kMetHop;
    const double wv = met_hann(o);
    const size_t src = row + (size_t)kb[j] * kMetHop + o;
    ax += wv * (double)x[src];
    ay += wv * (double)y[src];
  }
  xc[row + s] = (float)ax;
  yc[row + s] = (float)ay;
}

// ----------------------------------------------------------------------------------------------- 3. band envelopes
// grid (cdiv(NF, 8), B, 2): 8 STFT frames (Hann 256, hop 128, zero-padded to 512) of xc (z = 0) or yc (z = 1) per CTA;
// tob[b, z, k, t] = sqrt(sum_{lo[k] <= f < hi[k]} |X_t(f)|^2) for t < frames(c_len[b]).
__global__ void __launch_bounds__(kBandThreads)
met_bands_kernel(const float* __restrict__ xc, const float* __restrict__ yc, const int32_t* __restrict__ c_len, int T,
                 const float2* __restrict__ twiddle, const int32_t* __restrict__ lo,
                 const int32_t* __restrict__ hi, int NF, double* __restrict__ tob) {
  extern __shared__ float2 sm[];
  float2* tw = sm;
  float2* b0 = tw + kMetNfft;
  float2* b1 = b0 + kBandFrames * kMetNfft;
  __shared__ float w[kMetFrame];
  __shared__ int band[2 * kMetBands];
  const int b = blockIdx.y, z = blockIdx.z;
  const int nfr = met_frames(c_len[b]);
  const int t0 = blockIdx.x * kBandFrames;
  if (t0 >= nfr) return;
  const float* sig = (z ? yc : xc) + (size_t)b * T;
  for (int j = threadIdx.x; j < kMetFrame; j += blockDim.x) w[j] = (float)met_hann(j);
  for (int i = threadIdx.x; i < kMetNfft; i += blockDim.x) tw[i] = twiddle[i];
  if (threadIdx.x < kMetBands) {
    band[threadIdx.x] = lo[threadIdx.x];
    band[kMetBands + threadIdx.x] = hi[threadIdx.x];
  }
  __syncthreads();
  for (int i = threadIdx.x; i < kBandFrames * kMetNfft; i += blockDim.x) {
    const int f = i / kMetNfft, o = i % kMetNfft, t = t0 + f;
    b0[i] = make_float2((t < nfr && o < kMetFrame) ? w[o] * sig[(size_t)t * kMetHop + o] : 0.f, 0.f);
  }
  __syncthreads();
  // 512 = 4^4 * 2: the radix-4 and radix-2 butterflies of fft_core.cuh only
  float2 *src = b0, *dst = b1;
  for (int st = 0, Ns = 1; st < 5; ++st) {
    const int R = st < 4 ? 4 : 2, per = kMetNfft / R;
    for (int idx = threadIdx.x; idx < kBandFrames * per; idx += blockDim.x) {
      const int f = idx / per, j = idx - f * per;
      if (R == 4) butterfly<4, false>(src + f * kMetNfft, dst + f * kMetNfft, tw, kMetNfft, Ns, j);
      else butterfly<2, false>(src + f * kMetNfft, dst + f * kMetNfft, tw, kMetNfft, Ns, j);
    }
    __syncthreads();
    Ns *= R;
    float2* t = src; src = dst; dst = t;
  }
  const float2* r = src;
  for (int i = threadIdx.x; i < kBandFrames * kMetBands; i += blockDim.x) {
    const int f = i / kMetBands, k = i % kMetBands, t = t0 + f;
    if (t >= nfr) continue;
    const float2* X = r + f * kMetNfft;
    double acc = 0.0;
    for (int q = band[k]; q < band[kMetBands + k]; ++q) acc += (double)X[q].x * X[q].x + (double)X[q].y * X[q].y;
    tob[(((size_t)b * 2 + z) * kMetBands + k) * NF + t] = sqrt(acc);
  }
}

// ----------------------------------------------------------------------------------------------- 4. correlation
// grid (cdiv(NF, 32), B): thread i scores segment m = 32 blockIdx.x + i, frames [m, m + 30) of both envelopes: rows (bands)
// centred and scaled to unit norm, then columns (frames) the same, seg[b, m] = sum(xn yn) / 30.  A zero-norm row or
// column normalises to zeros.
__global__ void __launch_bounds__(kSegThreads)
met_segment_kernel(const double* __restrict__ tob, const int32_t* __restrict__ c_len, int NF, double* __restrict__ seg) {
  __shared__ double win[2][kMetBands][kSegWin];
  __shared__ double mu[2][kMetBands][kSegThreads];
  __shared__ double nrm[2][kMetBands][kSegThreads];
  const int b = blockIdx.y, i = threadIdx.x;
  const int nseg = met_frames(c_len[b]) - kMetSeg + 1;
  const int m0 = blockIdx.x * kSegThreads;
  if (m0 >= nseg) return;
  const int nfr = nseg + kMetSeg - 1;
  for (int q = i; q < 2 * kMetBands * kSegWin; q += blockDim.x) {
    const int z = q / (kMetBands * kSegWin), k = (q / kSegWin) % kMetBands, t = q % kSegWin;
    win[z][k][t] = m0 + t < nfr ? tob[(((size_t)b * 2 + z) * kMetBands + k) * NF + m0 + t] : 0.0;
  }
  __syncthreads();
  if (m0 + i >= nseg) return;
  for (int z = 0; z < 2; ++z)
    for (int k = 0; k < kMetBands; ++k) {
      const double* r = &win[z][k][i];
      double s = 0.0;
      for (int c = 0; c < kMetSeg; ++c) s += r[c];
      const double mk = s / kMetSeg;
      double q = 0.0;
      for (int c = 0; c < kMetSeg; ++c) q += (r[c] - mk) * (r[c] - mk);
      mu[z][k][i] = mk;
      nrm[z][k][i] = sqrt(q);
    }
  double total = 0.0;
  for (int c = 0; c < kMetSeg; ++c) {
    double cm[2], cn[2];
    for (int z = 0; z < 2; ++z) {
      double s = 0.0;
      for (int k = 0; k < kMetBands; ++k) {
        const double d = nrm[z][k][i];
        s += d > 0.0 ? (win[z][k][i + c] - mu[z][k][i]) / d : 0.0;
      }
      cm[z] = s / kMetBands;
      double q = 0.0;
      for (int k = 0; k < kMetBands; ++k) {
        const double d = nrm[z][k][i];
        const double a = (d > 0.0 ? (win[z][k][i + c] - mu[z][k][i]) / d : 0.0) - cm[z];
        q += a * a;
      }
      cn[z] = sqrt(q);
    }
    if (!(cn[0] > 0.0) || !(cn[1] > 0.0)) continue;
    for (int k = 0; k < kMetBands; ++k) {
      const double dx = nrm[0][k][i], dy = nrm[1][k][i];
      const double a = ((dx > 0.0 ? (win[0][k][i + c] - mu[0][k][i]) / dx : 0.0) - cm[0]) / cn[0];
      const double v = ((dy > 0.0 ? (win[1][k][i + c] - mu[1][k][i]) / dy : 0.0) - cm[1]) / cn[1];
      total += a * v / kMetSeg;
    }
  }
  seg[(size_t)b * NF + m0 + i] = total;
}

// grid (B): out[b] = mean of the segment scores, 1e-5 with fewer than 30 frames (pystoi's fallback)
__global__ void __launch_bounds__(kRedThreads)
met_estoi_mean_kernel(const int32_t* __restrict__ c_len, int NF, const double* __restrict__ seg, double* __restrict__ out) {
  __shared__ double red[kRedThreads / 32];
  const int b = blockIdx.x;
  const int nseg = met_frames(c_len[b]) - kMetSeg + 1;
  if (nseg <= 0) {
    if (threadIdx.x == 0) out[b] = 1e-5;
    return;
  }
  double s = 0.0;
  for (int m = threadIdx.x; m < nseg; m += blockDim.x) s += seg[(size_t)b * NF + m];
  s = met_block_sum(s, red);
  if (threadIdx.x == 0) out[b] = s / nseg;
}

// ----------------------------------------------------------------------------------------------- SDR
// grid (cdiv(T, 2048), B), 512 threads: partial sums over the chunk's samples s of
//   acf[k] = r[s] r[s + k], xcorr[k] = r[s] e[s + k] (thread k) and sum e[s]^2 (thread 0), all in f64
// -> part[b, chunk, 0..1025).  Samples at or beyond len[b] count as zeros.
__global__ void __launch_bounds__(kSdrTaps)
met_sdr_corr_kernel(const float* __restrict__ ref, const float* __restrict__ inf, const int32_t* __restrict__ len, int T,
                    int n_chunks, double* __restrict__ part) {
  __shared__ double r[kSdrChunk + kSdrTaps];
  __shared__ double e[kSdrChunk + kSdrTaps];
  const int b = blockIdx.y, n = len[b];
  const long s0 = (long)blockIdx.x * kSdrChunk;
  if (s0 >= n) return;
  const float* rb = ref + (size_t)b * T;
  const float* eb = inf + (size_t)b * T;
  for (int i = threadIdx.x; i < kSdrChunk + kSdrTaps; i += blockDim.x) {
    const long s = s0 + i;
    r[i] = s < n ? (double)rb[s] : 0.0;
    e[i] = s < n ? (double)eb[s] : 0.0;
  }
  __syncthreads();
  const int k = threadIdx.x;
  const int cnt = (int)min((long)kSdrChunk, n - s0);
  double a = 0.0, c = 0.0;
  for (int s = 0; s < cnt; ++s) {
    const double rs = r[s];
    a = fma(rs, r[s + k], a);
    c = fma(rs, e[s + k], c);
  }
  double* p = part + ((size_t)b * n_chunks + blockIdx.x) * kSdrVals;
  p[k] = a;
  p[kSdrTaps + k] = c;
  if (k == 0) {
    double q = 0.0;
    for (int s = 0; s < cnt; ++s) q = fma(e[s], e[s], q);
    p[2 * kSdrTaps] = q;
  }
}

// grid (B), 512 threads: sum the chunk partials in chunk order, normalise as for unit-norm signals, solve the symmetric
// Toeplitz system acf * sol = xcorr by Levinson recursion (one warp), coh = xcorr . sol clamped to [1e-5, 1e5] / (1 + .),
// out = 10 log10(coh / (1 - coh)).  A zero reference gives NaN.  A non-positive pivot (an ill-conditioned system in
// finite precision) ends the recursion at the last order that was still positive definite.
__global__ void __launch_bounds__(kSdrTaps)
met_sdr_solve_kernel(const int32_t* __restrict__ len, int n_chunks, const double* __restrict__ part,
                     double* __restrict__ out) {
  __shared__ double acf[kSdrTaps], xc[kSdrTaps], f[2][kSdrTaps], x[kSdrTaps];
  __shared__ double ee;
  const int b = blockIdx.x, n = len[b];
  const int nc = n > 0 ? (n + kSdrChunk - 1) / kSdrChunk : 0;
  const double* p = part + (size_t)b * n_chunks * kSdrVals;
  for (int v = threadIdx.x; v < kSdrVals; v += blockDim.x) {
    double s = 0.0;
    for (int c = 0; c < nc; ++c) s += p[(size_t)c * kSdrVals + v];
    if (v < kSdrTaps) acf[v] = s;
    else if (v < 2 * kSdrTaps) xc[v - kSdrTaps] = s;
    else ee = s;
  }
  __syncthreads();
  const double rr = acf[0];
  if (!(rr > 0.0)) {
    if (threadIdx.x == 0) out[b] = nan("");
    return;
  }
  const double nr = fmax(sqrt(rr), 1e-12), ne = fmax(sqrt(ee), 1e-12);
  const double sa = 1.0 / (nr * nr), sx = 1.0 / (nr * ne);
  for (int i = threadIdx.x; i < kSdrTaps; i += blockDim.x) {
    acf[i] = acf[i] * sa;
    xc[i] = xc[i] * sx;
    f[0][i] = 0.0;
    f[1][i] = 0.0;
    x[i] = 0.0;
  }
  __syncthreads();
  if (threadIdx.x >= 32) return;
  const int lane = threadIdx.x;
  if (lane == 0) {
    f[0][0] = 1.0 / acf[0];
    x[0] = xc[0] / acf[0];
  }
  __syncwarp();
  int cur = 0;
  for (int m = 1; m < kSdrTaps; ++m) {
    const double* fo = f[cur];
    double ef = 0.0, ex = 0.0;
    for (int i = lane; i < m; i += 32) {
      ef = fma(acf[m - i], fo[i], ef);
      ex = fma(acf[m - i], x[i], ex);
    }
    ef = warp_sum(ef);
    ex = warp_sum(ex);
    const double den = 1.0 - ef * ef;
    if (!(den > 0.0) || !isfinite(ef) || !isfinite(ex)) break;
    double* fn = f[cur ^ 1];
    for (int i = lane; i <= m; i += 32) fn[i] = ((i < m ? fo[i] : 0.0) - ef * (i > 0 ? fo[m - i] : 0.0)) / den;
    __syncwarp();
    const double g = xc[m] - ex;
    for (int i = lane; i <= m; i += 32) x[i] = fma(g, fn[m - i], x[i]);
    __syncwarp();
    cur ^= 1;
  }
  double coh = 0.0;
  for (int i = lane; i < kSdrTaps; i += 32) coh = fma(xc[i], x[i], coh);
  coh = warp_sum(coh);
  if (lane == 0) {
    const double lo = 1e-5;                                     // 10^(-50 / 10)
    coh = fmin(fmax(coh, lo / (1.0 + lo)), 1.0 / (1.0 + lo));   // fmax also maps a NaN to the lower clamp
    out[b] = 10.0 * log10(coh / (1.0 - coh));
  }
}

}  // namespace bsrnn

using namespace bsrnn;

extern "C" int bsrnn_resample_poly(const float* x, const int32_t* len, int B, int T, const double* taps, int n_taps, int up,
                                   int down, float* y, int32_t* y_len, int T_out, void* stream) {
  BSRNN_CHECK_ARG(x && len && taps && y && y_len, "resample_poly: null pointer");
  BSRNN_CHECK_ARG(B > 0 && B <= 65535 && T > 0 && n_taps > 0 && (n_taps & 1) && up > 0 && down > 0 &&
                      T_out >= ((long)T * up + down - 1) / down,
                  "resample_poly: bad dims");
  const int half = (n_taps - 1) / 2;
  const int pre_pad = down - half % down;
  const int pre_remove = (half + pre_pad) / down;
  const int J = (n_taps + up - 1) / up;
  met_resample_kernel<<<dim3(cdiv(T_out, kRsThreads), B), kRsThreads, 0, (cudaStream_t)stream>>>(
      x, len, T, taps, J, up, down, pre_pad, pre_remove, y, y_len, T_out);
  BSRNN_LAUNCH_OK();
  return 0;
}

static int met_nf(int T) { return std::max(T > kMetFrame ? (T - kMetFrame - 1) / kMetHop + 1 : 0, 1); }

extern "C" long bsrnn_estoi_compact_scratch_bytes(int B, int T) {
  if (B <= 0 || T <= 0) return -1;
  return (long)B * met_nf(T) * (long)(sizeof(double) + sizeof(int32_t));
}

extern "C" int bsrnn_estoi_compact(const float* x, const float* y, const int32_t* len, int B, int T, float* xc, float* yc,
                                   int32_t* c_len, void* scratch, void* stream) {
  BSRNN_CHECK_ARG(x && y && len && xc && yc && c_len && scratch, "estoi_compact: null pointer");
  BSRNN_CHECK_ARG(B > 0 && B <= 65535 && T > 0, "estoi_compact: bad dims");
  const int NF = met_nf(T);
  double* en = reinterpret_cast<double*>(scratch);
  int32_t* kept = reinterpret_cast<int32_t*>(en + (size_t)B * NF);
  cudaStream_t st = (cudaStream_t)stream;
  met_energy_kernel<<<dim3(cdiv(NF, kEnThreads / 32), B), kEnThreads, 0, st>>>(x, len, T, NF, en);
  BSRNN_LAUNCH_OK();
  met_select_kernel<<<B, kSelThreads, 0, st>>>(len, NF, en, kept, c_len);
  BSRNN_LAUNCH_OK();
  met_ola_kernel<<<dim3(cdiv(T, kOlaThreads), B), kOlaThreads, 0, st>>>(x, y, T, NF, kept, c_len, xc, yc);
  BSRNN_LAUNCH_OK();
  return 0;
}

extern "C" int bsrnn_estoi_bands(const float* xc, const float* yc, const int32_t* c_len, int B, int T, const float* twiddle,
                                 const int32_t* band_lo, const int32_t* band_hi, double* tob, int NF, void* stream) {
  BSRNN_CHECK_ARG(xc && yc && c_len && twiddle && band_lo && band_hi && tob, "estoi_bands: null pointer");
  BSRNN_CHECK_ARG(B > 0 && B <= 65535 && T > 0 && NF >= met_nf(T), "estoi_bands: bad dims");
  const size_t smem = (size_t)(1 + 2 * kBandFrames) * kMetNfft * sizeof(float2);
  BSRNN_CUDA_OK(cudaFuncSetAttribute(met_bands_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  met_bands_kernel<<<dim3(cdiv(NF, kBandFrames), B, 2), kBandThreads, smem, (cudaStream_t)stream>>>(
      xc, yc, c_len, T, reinterpret_cast<const float2*>(twiddle), band_lo, band_hi, NF, tob);
  BSRNN_LAUNCH_OK();
  return 0;
}

extern "C" int bsrnn_estoi_score(const double* tob, const int32_t* c_len, int B, int NF, double* seg, double* out,
                                 void* stream) {
  BSRNN_CHECK_ARG(tob && c_len && seg && out, "estoi_score: null pointer");
  BSRNN_CHECK_ARG(B > 0 && B <= 65535 && NF > 0, "estoi_score: bad dims");
  cudaStream_t st = (cudaStream_t)stream;
  met_segment_kernel<<<dim3(cdiv(NF, kSegThreads), B), kSegThreads, 0, st>>>(tob, c_len, NF, seg);
  BSRNN_LAUNCH_OK();
  met_estoi_mean_kernel<<<B, kRedThreads, 0, st>>>(c_len, NF, seg, out);
  BSRNN_LAUNCH_OK();
  return 0;
}

extern "C" long bsrnn_sdr_scratch_bytes(int B, int T) {
  if (B <= 0 || T <= 0) return -1;
  return (long)B * cdiv(T, kSdrChunk) * kSdrVals * (long)sizeof(double);
}

extern "C" int bsrnn_sdr(const float* ref, const float* inf, const int32_t* len, int B, int T, double* out, double* scratch,
                         void* stream) {
  BSRNN_CHECK_ARG(ref && inf && len && out && scratch, "sdr: null pointer");
  BSRNN_CHECK_ARG(B > 0 && B <= 65535 && T > 0, "sdr: bad dims");
  const int nc = cdiv(T, kSdrChunk);
  cudaStream_t st = (cudaStream_t)stream;
  met_sdr_corr_kernel<<<dim3(nc, B), kSdrTaps, 0, st>>>(ref, inf, len, T, nc, scratch);
  BSRNN_LAUNCH_OK();
  met_sdr_solve_kernel<<<B, kSdrTaps, 0, st>>>(len, nc, scratch, out);
  BSRNN_LAUNCH_OK();
  return 0;
}
