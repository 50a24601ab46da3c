// mix.cu — dynamic-mixing simulation on the device (mixing.simulate): partitioned FFT convolution (reverberation and the
// bandwidth-limiting low-pass), active-level SNR mixing, quantile clipping, packet loss and the joint peak normalisation.
// Every kernel is batched over the utterances of a batch, reads per-utterance lengths, writes exact zeros beyond each
// length and never reads a padded sample.  No floating-point atomics: the same inputs give bitwise-identical outputs.
#include "fft_core.cuh"

namespace bsrnn {

constexpr int kMixP = 1024;             // partition / output block length
constexpr int kMixN = 2 * kMixP;        // FFT length (radix 4^5 * 2)
constexpr int kMixThreads = 512;
constexpr int kMixFrame = 1024;         // active-level frames
constexpr int kMixHop = 512;
constexpr int kMixPwThreads = 256;      // 8 warps = 8 frames per CTA
constexpr int kMixEwThreads = 256;
constexpr int kMixEwChunk = 8192;       // samples per CTA of the elementwise kernels
constexpr int kMixSelThreads = 1024;

static inline size_t mix_fft_smem() { return 3 * kMixN * sizeof(float2); }   // twiddles + two ping-pong frames

// ----------------------------------------------------------------------------------------------- FFT convolution
// y_f[b, s] = sum_m h_f[b, m] * x[b, s + off_b - m]  for s < x_len[b] (zero for s in [x_len[b], T)), x zero outside
// [0, x_len[b]), h_f zero at and beyond h_len[b, f].  off_b = (h_len[b, 0] - 1) / 2 when `centered` (zero-phase FIR),
// else 0.  An utterance whose h_len[b, f] is 0 gets y_f = x (copied, not convolved).
// Overlap-save with uniform partitions of P = 1024 taps: input frame j holds x'[(j-1)P, (j+1)P) (x' = x shifted by off),
// filter partition p holds h[pP, (p+1)P) zero-padded to 2P; output block k = the last P samples of
// IFFT(sum_{p <= k} X_{k-p} H_p) / 2P.  Grid of the transform launch: (nfr + nfilt * nparts, B).
__global__ void __launch_bounds__(kMixThreads)
mix_conv_spec_kernel(const float* __restrict__ x, const int32_t* __restrict__ x_len, int T, const float* __restrict__ h,
                     const int32_t* __restrict__ h_len, int Lh, int nfilt, int centered, float2* __restrict__ xspec,
                     float2* __restrict__ hspec, const float2* __restrict__ twiddle, FftPlan plan, int nfr, int nparts) {
  extern __shared__ float2 sm[];
  float2* tw = sm;
  float2* b0 = sm + kMixN;
  float2* b1 = b0 + kMixN;
  const int b = blockIdx.y, B = gridDim.y;
  const int32_t* hl = h_len + (size_t)b * nfilt;
  bool any = false;
  for (int f = 0; f < nfilt; ++f) any |= hl[f] > 0;
  if (!any) return;                                           // every output of this utterance is a copy of x
  float2* dst;
  int j = blockIdx.x;
  if (j < nfr) {
    const long n = x_len[b];
    const long base = (long)(j - 1) * kMixP + (centered ? (hl[0] - 1) / 2 : 0);
    const float* xb = x + (size_t)b * T;
    for (int i = threadIdx.x; i < kMixN; i += blockDim.x) {
      const long s = base + i;
      b0[i] = make_float2((s >= 0 && s < n) ? xb[s] : 0.f, 0.f);
    }
    dst = xspec + ((size_t)b * nfr + j) * kMixN;
  } else {
    j -= nfr;
    const int f = j / nparts, p = j - f * nparts;
    const long len = hl[f];
    if ((long)p * kMixP >= len) return;                       // beyond this filter: never read
    const float* hb = h + (size_t)b * Lh;
    for (int i = threadIdx.x; i < kMixN; i += blockDim.x) {
      const long s = (long)p * kMixP + i;
      b0[i] = make_float2((i < kMixP && s < len) ? hb[s] : 0.f, 0.f);
    }
    dst = hspec + (((size_t)f * B + b) * nparts + p) * kMixN;
  }
  for (int i = threadIdx.x; i < kMixN; i += blockDim.x) tw[i] = twiddle[i];
  __syncthreads();
  const float2* r = fft_frames<false>(b0, b1, tw, plan, 1);
  for (int i = threadIdx.x; i < kMixN; i += blockDim.x) dst[i] = r[i];
}

// grid (nfr, nfilt, B): one CTA per (output block, filter, utterance).  Each thread accumulates its bins over the
// partitions in a fixed order, the inverse FFT runs in shared memory, and the valid half is stored.
__global__ void __launch_bounds__(kMixThreads)
mix_conv_acc_kernel(const float* __restrict__ x, const int32_t* __restrict__ x_len, int T, const int32_t* __restrict__ h_len,
                    int nfilt, const float2* __restrict__ xspec, const float2* __restrict__ hspec,
                    const float2* __restrict__ twiddle, FftPlan plan, int nfr, int nparts, float* __restrict__ y) {
  extern __shared__ float2 sm[];
  float2* tw = sm;
  float2* b0 = sm + kMixN;
  float2* b1 = b0 + kMixN;
  const int k = blockIdx.x, f = blockIdx.y, b = blockIdx.z, B = gridDim.z;
  const long n = x_len[b];
  const int len = h_len[(size_t)b * nfilt + f];
  float* out = y + ((size_t)f * B + b) * T;
  const long o0 = (long)k * kMixP;
  if (len == 0) {
    const float* xb = x + (size_t)b * T;
    for (int i = threadIdx.x; i < kMixP; i += blockDim.x) {
      const long s = o0 + i;
      if (s < T) out[s] = s < n ? xb[s] : 0.f;
    }
    return;
  }
  const int np = min((len + kMixP - 1) / kMixP, k + 1);
  const float2* X = xspec + (size_t)b * nfr * kMixN;
  const float2* H = hspec + ((size_t)f * B + b) * nparts * kMixN;
  for (int i = threadIdx.x; i < kMixN; i += blockDim.x) {
    float2 acc = make_float2(0.f, 0.f);
    for (int p = 0; p < np; ++p) {
      const float2 a = X[(size_t)(k - p) * kMixN + i], w = H[(size_t)p * kMixN + i];
      acc.x = fmaf(a.x, w.x, fmaf(-a.y, w.y, acc.x));
      acc.y = fmaf(a.x, w.y, fmaf(a.y, w.x, acc.y));
    }
    b0[i] = acc;
    tw[i] = twiddle[i];
  }
  __syncthreads();
  const float2* r = fft_frames<true>(b0, b1, tw, plan, 1);
  const float inv = 1.f / kMixN;
  for (int i = threadIdx.x; i < kMixP; i += blockDim.x) {
    const long s = o0 + i;
    if (s < T) out[s] = s < n ? r[kMixP + i].x * inv : 0.f;
  }
}

// ----------------------------------------------------------------------------------------------- SNR mixing
__device__ __forceinline__ int mix_nframes(int n) { return n <= 0 ? 0 : (n >= kMixFrame ? 1 + (n - kMixFrame) / kMixHop : 1); }

// grid (cdiv(nf_max, 8), B, 2): one warp per frame; pw[(sig * B + b) * nf_max + t] = mean square of frame t of signal sig
// (0 = speech, 1 = noise).  Frames are 1024 samples at hop 512 inside [0, n); an utterance shorter than a frame is one frame.
__global__ void __launch_bounds__(kMixPwThreads)
mix_frame_power_kernel(const float* __restrict__ speech, const float* __restrict__ noise, const int32_t* __restrict__ len,
                       int T, int nf_max, double* __restrict__ pw) {
  const int b = blockIdx.y, sig = blockIdx.z, B = gridDim.y;
  const int t = blockIdx.x * (kMixPwThreads / 32) + threadIdx.x / 32, lane = threadIdx.x % 32;
  const int n = len[b];
  if (t >= mix_nframes(n)) return;
  const float* xb = (sig ? noise : speech) + (size_t)b * T;
  const int s0 = t * kMixHop, s1 = min(s0 + kMixFrame, n);
  double acc = 0.0;
  for (int s = s0 + lane; s < s1; s += 32) acc += (double)xb[s] * (double)xb[s];
  acc = warp_sum(acc);
  if (lane == 0) pw[((size_t)sig * B + b) * nf_max + t] = acc / (double)(s1 - s0);
}

// fixed-order block sum (all threads get the result)
__device__ double mix_block_sum(double v, double* red) {
  v = warp_sum(v);
  const int w = threadIdx.x / 32, nw = blockDim.x / 32;
  __syncthreads();
  if (threadIdx.x % 32 == 0) red[w] = v;
  __syncthreads();
  double s = 0.0;
  for (int i = 0; i < nw; ++i) s += red[i];
  return s;
}

// active-level power of one signal: mean of the frame powers above 0.01 x the mean frame power
__device__ double mix_active_power(const double* p, int nf, double* red) {
  double s = 0.0;
  for (int t = threadIdx.x; t < nf; t += blockDim.x) s += p[t];
  const double mean = mix_block_sum(s, red) / (double)max(nf, 1);
  double a = 0.0, c = 0.0;
  for (int t = threadIdx.x; t < nf; t += blockDim.x)
    if (p[t] > 0.01 * mean) { a += p[t]; c += 1.0; }
  a = mix_block_sum(a, red);
  c = mix_block_sum(c, red);
  return c > 0.0 ? a / c : 0.0;
}

// grid (cdiv(T, chunk), B): every CTA of an utterance derives the same gain from the frame powers (the same fixed-order
// sums), then mixes its chunk: noisy = speech + g * noise, g = 10^(-snr/20) sqrt(P_s / max(P_n, 1e-10)).
__global__ void __launch_bounds__(kMixEwThreads)
mix_snr_kernel(const float* __restrict__ speech, const float* __restrict__ noise, const int32_t* __restrict__ len,
               const float* __restrict__ snr_db, int T, int nf_max, const double* __restrict__ pw, float* __restrict__ noisy,
               float* __restrict__ gain) {
  __shared__ double red[kMixEwThreads / 32];
  const int b = blockIdx.y, B = gridDim.y;
  const int n = len[b], nf = mix_nframes(n);
  const double ps = mix_active_power(pw + (size_t)b * nf_max, nf, red);
  const double pn = mix_active_power(pw + ((size_t)B + b) * nf_max, nf, red);
  const float g = (float)(pow(10.0, -(double)snr_db[b] / 20.0) * sqrt(ps / fmax(pn, 1e-10)));
  if (blockIdx.x == 0 && threadIdx.x == 0 && gain) gain[b] = g;
  const float* sb = speech + (size_t)b * T;
  const float* nb = noise + (size_t)b * T;
  float* ob = noisy + (size_t)b * T;
  const long s1 = min((long)T, (long)(blockIdx.x + 1) * kMixEwChunk);
  for (long s = (long)blockIdx.x * kMixEwChunk + threadIdx.x; s < s1; s += blockDim.x)
    ob[s] = s < n ? fmaf(g, nb[s], sb[s]) : 0.f;
}

// ----------------------------------------------------------------------------------------------- quantile clipping
// order-preserving image of a float in uint32 (negative values reversed below the positive ones)
__device__ __forceinline__ uint32_t mix_ord(float v) {
  const uint32_t u = __float_as_uint(v);
  return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}
__device__ __forceinline__ float mix_unord(uint32_t u) {
  return __uint_as_float((u & 0x80000000u) ? (u & 0x7fffffffu) : ~u);
}

// the k-th smallest (0-based) ordered image among xb[0, n): radix select, 8 bits per pass, MSB first
__device__ uint32_t mix_select(const float* xb, int n, int k, uint32_t* hist, uint32_t* bc) {
  uint32_t prefix = 0, mask = 0;
  for (int shift = 24; shift >= 0; shift -= 8) {
    for (int i = threadIdx.x; i < 256; i += blockDim.x) hist[i] = 0;
    __syncthreads();
    for (int s = threadIdx.x; s < n; s += blockDim.x) {
      const uint32_t u = mix_ord(xb[s]);
      if ((u & mask) == prefix) atomicAdd(&hist[(u >> shift) & 255u], 1u);
    }
    __syncthreads();
    if (threadIdx.x == 0) {
      uint32_t cum = 0, d = 0;
      while (cum + hist[d] <= (uint32_t)k) cum += hist[d++];
      bc[0] = prefix | (d << shift);
      bc[1] = (uint32_t)k - cum;
    }
    __syncthreads();
    prefix = bc[0];
    k = (int)bc[1];
    mask |= 255u << shift;
    __syncthreads();
  }
  return prefix;
}

// the (k+1)-th smallest given v = the k-th: v again if more than k+1 values are <= v, else the least value above v
__device__ uint32_t mix_next(const float* xb, int n, int k, uint32_t v, uint32_t* bc) {
  if (threadIdx.x == 0) { bc[2] = 0; bc[3] = 0xffffffffu; }
  __syncthreads();
  uint32_t le = 0, mn = 0xffffffffu;
  for (int s = threadIdx.x; s < n; s += blockDim.x) {
    const uint32_t u = mix_ord(xb[s]);
    if (u <= v) ++le; else mn = min(mn, u);
  }
  atomicAdd(&bc[2], le);
  atomicMin(&bc[3], mn);
  __syncthreads();
  const uint32_t r = (bc[2] > (uint32_t)k + 1u) ? v : bc[3];
  __syncthreads();
  return r;
}

// grid (B): thr[b, i] = NumPy's linear-method quantile q[b, i] of the valid samples of x[b] (i = 0 lower, 1 upper)
__global__ void __launch_bounds__(kMixSelThreads)
mix_quantile_kernel(const float* __restrict__ x, const int32_t* __restrict__ len, const double* __restrict__ q, int T,
                    float* __restrict__ thr) {
  __shared__ uint32_t hist[256];
  __shared__ uint32_t bc[4];
  const int b = blockIdx.x, n = len[b];
  const float* xb = x + (size_t)b * T;
  for (int i = 0; i < 2; ++i) {
    if (n <= 0) {
      if (threadIdx.x == 0) thr[2 * b + i] = 0.f;
      continue;
    }
    const double pos = q[2 * b + i] * (double)(n - 1);
    const int lo = min((int)floor(pos), n - 1);
    const double t = pos - (double)lo;
    const uint32_t ua = mix_select(xb, n, lo, hist, bc);
    const uint32_t ub = lo + 1 < n ? mix_next(xb, n, lo, ua, bc) : ua;
    const double a = (double)mix_unord(ua), c = (double)mix_unord(ub), d = c - a;
    if (threadIdx.x == 0) thr[2 * b + i] = (float)(t >= 0.5 ? c - d * (1.0 - t) : a + d * t);
  }
}

// ----------------------------------------------------------------------------------------------- finish
__device__ __forceinline__ float mix_degrade(float v, long s, const float* th, const uint8_t* lost, int npk, int pkt) {
  v = fminf(fmaxf(v, th[0]), th[1]);
  if (pkt > 0) {
    const long k = s / pkt;
    if (k < npk && lost[k]) v = 0.f;
  }
  return v;
}

// grid (cdiv(T, chunk), B): peak[b] = max over the valid samples of |degraded noisy| and |clean|, as float bits (a
// non-negative float orders like its bit pattern, so the integer max is exact and order-free)
__global__ void __launch_bounds__(kMixEwThreads)
mix_peak_kernel(const float* __restrict__ noisy, const float* __restrict__ clean, const int32_t* __restrict__ len,
                const float* __restrict__ thr, const uint8_t* __restrict__ lost, int npk, int pkt, int T,
                uint32_t* __restrict__ peak) {
  __shared__ float red[kMixEwThreads / 32];
  const int b = blockIdx.y, n = len[b];
  const long s1 = min((long)n, (long)(blockIdx.x + 1) * kMixEwChunk);
  const float* th = thr + 2 * b;
  const uint8_t* lb = lost ? lost + (size_t)b * npk : nullptr;
  float m = 0.f;
  for (long s = (long)blockIdx.x * kMixEwChunk + threadIdx.x; s < s1; s += blockDim.x) {
    const float v = mix_degrade(noisy[(size_t)b * T + s], s, th, lb, npk, lb ? pkt : 0);
    m = fmaxf(m, fmaxf(fabsf(v), fabsf(clean[(size_t)b * T + s])));
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
  if (threadIdx.x % 32 == 0) red[threadIdx.x / 32] = m;
  __syncthreads();
  if (threadIdx.x == 0) {
    for (int i = 1; i < kMixEwThreads / 32; ++i) m = fmaxf(m, red[i]);
    atomicMax(&peak[b], __float_as_uint(m));
  }
}

// grid (cdiv(T, chunk), B): clip, drop the lost packets, and scale noisy and clean by 0.9 / peak when peak > 0.9
__global__ void __launch_bounds__(kMixEwThreads)
mix_finish_kernel(float* __restrict__ noisy, float* __restrict__ clean, const int32_t* __restrict__ len,
                  const float* __restrict__ thr, const uint8_t* __restrict__ lost, int npk, int pkt, int T,
                  const uint32_t* __restrict__ peak) {
  const int b = blockIdx.y, n = len[b];
  const float pk = __uint_as_float(peak[b]);
  const float scale = pk > 0.9f ? 0.9f / pk : 1.f;
  const float* th = thr + 2 * b;
  const uint8_t* lb = lost ? lost + (size_t)b * npk : nullptr;
  const long s1 = min((long)T, (long)(blockIdx.x + 1) * kMixEwChunk);
  for (long s = (long)blockIdx.x * kMixEwChunk + threadIdx.x; s < s1; s += blockDim.x) {
    const size_t i = (size_t)b * T + s;
    if (s < n) {
      noisy[i] = mix_degrade(noisy[i], s, th, lb, npk, lb ? pkt : 0) * scale;
      clean[i] = clean[i] * scale;
    } else {
      noisy[i] = 0.f;
      clean[i] = 0.f;
    }
  }
}

}  // namespace bsrnn

using namespace bsrnn;

static void mix_conv_geometry(int T, int Lh, int* nfr, int* nparts) {
  *nfr = cdiv(T, kMixP);
  *nparts = cdiv(Lh, kMixP);
}

extern "C" long bsrnn_mix_conv_scratch_bytes(int B, int T, int Lh, int nfilt) {
  if (B <= 0 || T <= 0 || Lh < 0 || nfilt <= 0) return -1;
  int nfr, nparts;
  mix_conv_geometry(T, Lh, &nfr, &nparts);
  return ((long)B * nfr + (long)nfilt * B * nparts) * kMixN * (long)sizeof(float2);
}

extern "C" int bsrnn_mix_conv(const float* x, const int32_t* x_len, const float* h, const int32_t* h_len, float* y,
                              float* scratch, const float* twiddle, int B, int T, int Lh, int nfilt, int centered,
                              void* stream) {
  BSRNN_CHECK_ARG(x && x_len && h_len && y && twiddle && (scratch || Lh == 0) && (h || Lh == 0), "mix_conv: null pointer");
  BSRNN_CHECK_ARG(B > 0 && B <= 65535 && T > 0 && Lh >= 0 && nfilt > 0 && nfilt <= 65535, "mix_conv: bad dims");
  FftPlan plan;
  make_plan(kMixN, &plan);
  int nfr, nparts;
  mix_conv_geometry(T, Lh, &nfr, &nparts);
  cudaStream_t st = (cudaStream_t)stream;
  float2* xspec = reinterpret_cast<float2*>(scratch);
  float2* hspec = xspec + (size_t)B * nfr * kMixN;
  const float2* tw = reinterpret_cast<const float2*>(twiddle);
  if (nparts > 0) {
    mix_conv_spec_kernel<<<dim3(nfr + nfilt * nparts, B), kMixThreads, mix_fft_smem(), st>>>(
        x, x_len, T, h, h_len, Lh, nfilt, centered, xspec, hspec, tw, plan, nfr, nparts);
    BSRNN_LAUNCH_OK();
  }
  mix_conv_acc_kernel<<<dim3(nfr, nfilt, B), kMixThreads, mix_fft_smem(), st>>>(x, x_len, T, h_len, nfilt, xspec, hspec, tw,
                                                                                 plan, nfr, nparts, y);
  BSRNN_LAUNCH_OK();
  return 0;
}

extern "C" long bsrnn_mix_snr_scratch_bytes(int B, int T) {
  if (B <= 0 || T <= 0) return -1;
  return 2L * B * (1 + T / kMixHop) * (long)sizeof(double);
}

extern "C" int bsrnn_mix_snr(const float* speech, const float* noise, const int32_t* len, const float* snr_db, float* noisy,
                             float* gain, double* scratch, int B, int T, void* stream) {
  BSRNN_CHECK_ARG(speech && noise && len && snr_db && noisy && scratch, "mix_snr: null pointer");
  BSRNN_CHECK_ARG(B > 0 && B <= 65535 && T > 0, "mix_snr: bad dims");
  const int nf_max = 1 + T / kMixHop;                 // >= the frame count of any n <= T
  cudaStream_t st = (cudaStream_t)stream;
  mix_frame_power_kernel<<<dim3(cdiv(nf_max, kMixPwThreads / 32), B, 2), kMixPwThreads, 0, st>>>(speech, noise, len, T,
                                                                                                 nf_max, scratch);
  BSRNN_LAUNCH_OK();
  mix_snr_kernel<<<dim3(cdiv(T, kMixEwChunk), B), kMixEwThreads, 0, st>>>(speech, noise, len, snr_db, T, nf_max, scratch,
                                                                         noisy, gain);
  BSRNN_LAUNCH_OK();
  return 0;
}

extern "C" int bsrnn_mix_quantiles(const float* x, const int32_t* len, const double* q, float* thr, int B, int T,
                                   void* stream) {
  BSRNN_CHECK_ARG(x && len && q && thr, "mix_quantiles: null pointer");
  BSRNN_CHECK_ARG(B > 0 && T > 0, "mix_quantiles: bad dims");
  mix_quantile_kernel<<<B, kMixSelThreads, 0, (cudaStream_t)stream>>>(x, len, q, T, thr);
  BSRNN_LAUNCH_OK();
  return 0;
}

extern "C" int bsrnn_mix_finish(float* noisy, float* clean, const int32_t* len, const float* thr, const uint8_t* lost,
                                int npk, int pkt, uint32_t* peak, int B, int T, void* stream) {
  BSRNN_CHECK_ARG(noisy && clean && len && thr && peak, "mix_finish: null pointer");
  BSRNN_CHECK_ARG(B > 0 && B <= 65535 && T > 0 && (!lost || (npk > 0 && pkt > 0)), "mix_finish: bad dims");
  cudaStream_t st = (cudaStream_t)stream;
  BSRNN_CUDA_OK(cudaMemsetAsync(peak, 0, (size_t)B * sizeof(uint32_t), st));
  const dim3 grid(cdiv(T, kMixEwChunk), B);
  mix_peak_kernel<<<grid, kMixEwThreads, 0, st>>>(noisy, clean, len, thr, lost, npk, pkt, T, peak);
  BSRNN_LAUNCH_OK();
  mix_finish_kernel<<<grid, kMixEwThreads, 0, st>>>(noisy, clean, len, thr, lost, npk, pkt, T, peak);
  BSRNN_LAUNCH_OK();
  return 0;
}
