// bandsplit.cu — BandSplit as ONE kernel family: per band k, GroupNorm(1, 2 s_k) applied on load + Conv1d(2 s_k -> N, 1)
// [reference bsrnn_flowse.py:65-86; espnet2 BandSplit], writing the token-major residual stream (B, T, K', N).
//
// The op is write-bound (config 2: reads the 246 MB spectrum once, writes 1.71 GB; 24 GFLOP): a CTA owns 128 tokens of one
// band, keeps the band's transposed weight (2 s_k x N, <= 94 KB) and the normalised inputs (128 x 2 s_k) in shared memory
// and each warp writes whole 784-byte output rows.  It replaces the generic 64x64x16 SIMT grouped GEMM (gemm_f32.cu), which
// spent 2.83 ms on it (10 % of the copy bandwidth, profiles/r01 call47 / r02 call08).
#include "common.cuh"
#include <cuda_fp16.h>

namespace bsrnn {

constexpr int kBsRows = 128;
constexpr int kBsThreads = 256;

struct BandSplitArgs {
  const float* spec;        // (rows, 2F) interleaved re/im
  const float* scale;       // (B * K, cmax): GroupNorm scale per (sample, band, channel)
  const float* shift;
  const float* wT;          // concatenated transposed weights: band k at row c_off[k], (2 s_k rows) x N
  const float* bias;        // (K, N)
  float* out;
  const int* c_off;         // [K + 1] channel offsets into wT
  const int* bin0;          // [K] first bin of each band
  const int* width2;        // [K] 2 * real bins of the band (the rest of its 2 s_k channels are zero padding)
  long rows;                // B * T
  int T, F2, N, K, cmax, k_lo;
  long ldo;                 // output row stride (floats) = K * out_width
  int out_width, out_col;
};

__global__ void __launch_bounds__(kBsThreads, 2) band_split_kernel(const BandSplitArgs a) {
  extern __shared__ __align__(16) float bs_smem[];
  const int k = a.k_lo + blockIdx.x;                  // band fastest: co-running CTAs write adjacent segments of the same rows
  const int C = a.c_off[k + 1] - a.c_off[k];          // 2 s_k
  const int Cp = (C + 3) & ~3;                        // padded to float4
  const int N = a.N;
  float* Ws = bs_smem;                                // [Cp][N]
  float* xs = bs_smem + (size_t)Cp * N;               // [128][Cp]
  const long r0 = (long)blockIdx.y * kBsRows;
  const float* wsrc = a.wT + (size_t)a.c_off[k] * N;
  for (int i = threadIdx.x; i < Cp * N; i += kBsThreads) Ws[i] = i < C * N ? wsrc[i] : 0.f;
  const int cvalid = a.width2[k];
  const int col0 = 2 * a.bin0[k];
  for (int i = threadIdx.x; i < kBsRows * Cp; i += kBsThreads) {
    const int r = i / Cp, c = i - r * Cp;
    const long row = r0 + r;
    float v = 0.f;
    if (row < a.rows && c < C) {
      const long b = row / a.T;
      const float x = c < cvalid ? a.spec[row * a.F2 + col0 + c] : 0.f;       // truncated band: zero-padded BEFORE the norm
      const size_t g = ((size_t)b * a.K + k) * a.cmax + c;
      v = fmaf(x, a.scale[g], a.shift[g]);
    }
    xs[i] = v;
  }
  __syncthreads();
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int ngrp = N >> 2;                            // float4 column groups (N % 4 == 0)
  const float* bias = a.bias + (size_t)k * N;
  for (int pass = 0; pass * 32 < ngrp; ++pass) {
    const int grp = pass * 32 + lane;
    const bool act = grp < ngrp;
    float4 acc[16];
    const float4 b4 = act ? *reinterpret_cast<const float4*>(bias + 4 * grp) : make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
    for (int r = 0; r < 16; ++r) acc[r] = b4;
    if (act) {
      for (int c = 0; c < Cp; c += 4) {
        const float4 w0 = *reinterpret_cast<const float4*>(Ws + (size_t)(c + 0) * N + 4 * grp);
        const float4 w1 = *reinterpret_cast<const float4*>(Ws + (size_t)(c + 1) * N + 4 * grp);
        const float4 w2 = *reinterpret_cast<const float4*>(Ws + (size_t)(c + 2) * N + 4 * grp);
        const float4 w3 = *reinterpret_cast<const float4*>(Ws + (size_t)(c + 3) * N + 4 * grp);
#pragma unroll
        for (int r = 0; r < 16; ++r) {
          const float4 x = *reinterpret_cast<const float4*>(xs + (size_t)(16 * warp + r) * Cp + c);     // broadcast
          acc[r].x = fmaf(x.x, w0.x, fmaf(x.y, w1.x, fmaf(x.z, w2.x, fmaf(x.w, w3.x, acc[r].x))));
          acc[r].y = fmaf(x.x, w0.y, fmaf(x.y, w1.y, fmaf(x.z, w2.y, fmaf(x.w, w3.y, acc[r].y))));
          acc[r].z = fmaf(x.x, w0.z, fmaf(x.y, w1.z, fmaf(x.z, w2.z, fmaf(x.w, w3.z, acc[r].z))));
          acc[r].w = fmaf(x.x, w0.w, fmaf(x.y, w1.w, fmaf(x.z, w2.w, fmaf(x.w, w3.w, acc[r].w))));
        }
      }
#pragma unroll
      for (int r = 0; r < 16; ++r) {
        const long row = r0 + 16 * warp + r;
        if (row < a.rows)
          *reinterpret_cast<float4*>(a.out + row * a.ldo + (size_t)k * a.out_width + a.out_col + 4 * grp) = acc[r];
      }
    }
  }
}


// ---------------------------------------------------------------------------------------------- tensor-core operand
// Tensor-core BandSplit (fp16 mode): the per-band GroupNorm(1, 2 s_k) is applied while the band's slice of the spectrum
// is re-tiled into the fp16 KB8 operand of a tcgen05 GEMM (bsrnn_gemm_tc_ex, store-only TMA epilogue: out rows of band k
// = A_k W_k^T + b_k, with the statistics of the first dual-path GroupNorm in the epilogue).  One launch covers all bands:
// grid (K, row tiles); band k's tiles start at a_off[k] halves, [tile][kc_k][128][8] with kc_k = 2 * ceil(2 s_k / 16).
struct BandCastArgs {
  const float* spec;        // (rows, F2)
  const float* scale;       // (B * K, cmax)
  const float* shift;
  __half* out;
  const int* c_off;         // [K + 1]
  const int* bin0;          // [K]
  const int* width2;        // [K]
  const long long* a_off;   // [K] halves
  long rows;
  int T, F2, K, cmax;
};

__global__ void __launch_bounds__(256) band_norm_cast_kb8_kernel(const BandCastArgs a) {
  extern __shared__ __align__(16) unsigned char bc_smem[];
  __half* tile = reinterpret_cast<__half*>(bc_smem);
  const int k = blockIdx.x;                           // band fastest: co-running blocks read adjacent slices of the same rows
  const int C = a.c_off[k + 1] - a.c_off[k];
  const int kc = ((C + 15) >> 4) << 1;
  const int kw = kc * 8;
  const int ld = kw + 8;                               // +8 halves: rows land in different banks
  const int cvalid = a.width2[k];
  const int col0 = 2 * a.bin0[k];
  const long r0 = (long)blockIdx.y * 128;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  for (int r = warp; r < 128; r += 8) {
    const long row = r0 + r;
    const bool ok = row < a.rows;
    const long b = ok ? row / a.T : 0;
    const float* src = a.spec + (ok ? row : 0) * a.F2 + col0;
    const size_t g = ((size_t)b * a.K + k) * a.cmax;
    for (int c = lane; c < kw; c += 32) {
      float v = 0.f;
      if (ok && c < C) {
        const float x = c < cvalid ? __ldg(src + c) : 0.f;      // truncated band: zero-padded BEFORE the norm
        v = fmaf(x, __ldg(a.scale + g + c), __ldg(a.shift + g + c));
      }
      tile[r * ld + c] = __float2half_rn(v);
    }
  }
  __syncthreads();
  __half* dst = a.out + a.a_off[k] + (size_t)blockIdx.y * kc * 1024;
  for (int i = threadIdx.x; i < kc * 128; i += 256) {
    const int c8 = i >> 7, r = i & 127;
    *reinterpret_cast<uint4*>(dst + (size_t)i * 8) = *reinterpret_cast<const uint4*>(tile + r * ld + c8 * 8);
  }
}

}  // namespace bsrnn
using namespace bsrnn;

// Launches bands [0, K) in two shared-memory classes (narrow bands: many CTAs per SM; wide bands: up to 157 KB).
extern "C" int bsrnn_band_split_fwd(const float* spec, const float* scale, const float* shift, const float* wT,
                                    const float* bias, float* out, const int32_t* c_off, const int32_t* bin0,
                                    const int32_t* width2, const int32_t* c_off_host, int K, long rows, int T, int F2, int N,
                                    int cmax, long ldo, int out_width, int out_col, void* stream) {
  BSRNN_CHECK_ARG(spec && scale && shift && wT && bias && out && c_off && bin0 && width2 && c_off_host, "band_split_fwd: null pointer");
  BSRNN_CHECK_ARG(K > 0 && rows > 0 && T > 0 && N > 0 && N % 4 == 0 && out_col % 4 == 0 && out_width % 4 == 0 && ldo % 4 == 0,
                  "band_split_fwd: bad dims (N, out_col, out_width and ldo must be multiples of 4)");
  BandSplitArgs a{spec, scale, shift, wT, bias, out, c_off, bin0, width2, rows, T, F2, N, K, cmax, 0, ldo, out_width, out_col};
  auto smem_of = [&](int C) { const int Cp = (C + 3) & ~3; return (size_t)Cp * N * 4 + (size_t)kBsRows * Cp * 4; };
  for (int j = 0; j < K; ++j)                         // every band fits before the first run launches
    BSRNN_CHECK_ARG(smem_of(c_off_host[j + 1] - c_off_host[j]) <= 227 * 1024,
                    "band_split_fwd: band of %d channels does not fit in shared memory", c_off_host[j + 1] - c_off_host[j]);
  // consecutive runs of bands whose shared-memory need is within 2x of the run's maximum share one launch
  int k = 0;
  while (k < K) {
    size_t need = smem_of(c_off_host[k + 1] - c_off_host[k]);
    int e = k + 1;
    while (e < K) {
      const size_t s = smem_of(c_off_host[e + 1] - c_off_host[e]);
      if (s > 2 * need || 2 * s < need) break;
      if (s > need) need = s;
      ++e;
    }
    BSRNN_CUDA_OK(cudaFuncSetAttribute(band_split_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)need));
    a.k_lo = k;
    dim3 grid(e - k, (unsigned)((rows + kBsRows - 1) / kBsRows));
    band_split_kernel<<<grid, kBsThreads, need, (cudaStream_t)stream>>>(a);
    BSRNN_LAUNCH_OK();
    k = e;
  }
  return 0;
}

// Operand builder of the tensor-core BandSplit (see band_norm_cast_kb8_kernel).  a_off: device [K] offsets in halves.
extern "C" int bsrnn_band_norm_cast_kb8(const float* spec, const float* scale, const float* shift, void* out,
                                        const int32_t* c_off, const int32_t* bin0, const int32_t* width2,
                                        const long long* a_off, int K, long rows, int T, int F2, int cmax, void* stream) {
  BSRNN_CHECK_ARG(spec && scale && shift && out && c_off && bin0 && width2 && a_off, "band_norm_cast_kb8: null pointer");
  BSRNN_CHECK_ARG(K > 0 && rows > 0 && T > 0 && F2 > 0 && cmax > 0, "band_norm_cast_kb8: bad dims");
  const int kc_max = ((cmax + 15) >> 4) << 1;
  const size_t smem = (size_t)128 * (kc_max * 8 + 8) * 2;
  BSRNN_CHECK_ARG(smem <= 227 * 1024, "band_norm_cast_kb8: band of %d channels does not fit in shared memory", cmax);
  BSRNN_CUDA_OK(cudaFuncSetAttribute(band_norm_cast_kb8_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  BandCastArgs a{spec, scale, shift, reinterpret_cast<__half*>(out), c_off, bin0, width2, a_off, rows, T, F2, K, cmax};
  dim3 grid(K, (unsigned)((rows + 127) / 128));
  band_norm_cast_kb8_kernel<<<grid, 256, smem, (cudaStream_t)stream>>>(a);
  BSRNN_LAUNCH_OK();
  return 0;
}
