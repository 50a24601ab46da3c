// pack.cu — GroupNorm-apply + cast + re-tile: f32 token-major activations -> fp16 UMMA operand tiles (KB8 layout).
// This is the "normalise" half of nn.GroupNorm(1,N) [reference bsrnn_flowse.py:291,302; decoder norms :146-152]
// fused with the layout change the tensor-core GEMMs need, so the normalised activation is written exactly once, in
// the form the next GEMM's bulk copies fetch.
#include "common.cuh"
#include "umma.cuh"
#include "tmap.cuh"
#include <cuda_fp16.h>

namespace bsrnn {

struct PackArgs {
  const float* x;          // token-major rows of ldx floats
  const float* scale;      // (groups, C) or null
  const float* shift;
  __half* out;             // [m_tiles][kcores][128][8]
  long ldx;
  int col0, C, kcores;
  int tiles_per_step, R;
  long seq_inner, seq_outer, seq_inner_stride, step_stride;
  long tokens_per_sample;  // scale row = (token / tokens_per_sample) * g_inner + (g_inner > 1 ? token % g_inner : 0)
  int g_inner;
  int one_col;           // >= C: this operand column is the constant 1 (bias row of the weights); -1 = none
  int bulk;              // async kernel: rows arrive by one cp.async.bulk per row (1), per run of contiguous rows (2), or by
                         // ONE 2-D tensor copy per block (3, band axis, tmap.cuh)
  int m_inner;           // bulk == 3: blocks walk the tiles with the step (= band) innermost: co-running blocks read adjacent
                         // segments of the same rows of the residual stream
  int tm_col_step;       // bulk == 3: the tile is rows [j*128, +128) x cols [step*tm_col_step, +C) of the matrix view `tmap`
  alignas(64) CUtensorMap tmap;
};

// grid (m_tiles), block 256, dynamic smem 128 * (kcores*8 + 8) halves + 128 row descriptors.
// Work item = (row, 4 consecutive channels): consecutive threads read consecutive float4 of a token row (coalesced
// 16-byte loads, PK_U in flight per thread), apply the affine, and drop 4 halves into the padded tile; the tile then
// leaves as 16-byte KB8 cores.  Needs C % 4 == 0, col0 % 4 == 0 and 16-byte aligned rows; otherwise the scalar path.
// 16-byte loads each thread keeps in flight (profiles/r01/call26: with 4 the kernel sat on the load latency at 2.9 TB/s)
constexpr int PK_U = 8;
struct PackRow {
  long tok;        // token index or -1
  long grp;        // scale/shift row
};

__global__ void __launch_bounds__(256) norm_cast_kb8_kernel(const PackArgs a, int vec_ok) {
  extern __shared__ __align__(128) unsigned char smem_raw[];
  const int ld = a.kcores * 8 + 8;                 // +8 halves: rows land in different banks
  __half* tile = reinterpret_cast<__half*>(smem_raw);
  PackRow* rows = reinterpret_cast<PackRow*>(smem_raw + (size_t)128 * ld * 2);
  const int m = blockIdx.x;
  const int step = m / a.tiles_per_step, j = m - step * a.tiles_per_step;
  const int kw = a.kcores * 8;
  if (threadIdx.x < 128) {
    const int r = threadIdx.x;
    const long seq = (long)j * 128 + r;
    PackRow pr{-1, 0};
    if (seq < a.R) {
      pr.tok = (seq / a.seq_inner) * a.seq_outer + (seq % a.seq_inner) * a.seq_inner_stride + (long)step * a.step_stride;
      if (a.scale) pr.grp = (pr.tok / a.tokens_per_sample) * a.g_inner + (a.g_inner > 1 ? pr.tok % a.g_inner : 0);
    }
    rows[r] = pr;
  }
  __syncthreads();
  if (vec_ok) {
    const int q4 = kw >> 2;                        // float4 slots per row (52 for N = 196)
    const int items = 128 * q4;
    for (int base = threadIdx.x; base < items; base += 256 * PK_U) {
      float4 v[PK_U];
      int rr[PK_U], cc[PK_U];
#pragma unroll
      for (int u = 0; u < PK_U; ++u) {
        const int idx = base + u * 256;
        v[u] = make_float4(0.f, 0.f, 0.f, 0.f);
        rr[u] = -1;
        if (idx < items) {
          rr[u] = idx / q4;
          cc[u] = (idx - rr[u] * q4) * 4;
          const long tok = rows[rr[u]].tok;
          if (tok >= 0 && cc[u] < a.C) v[u] = __ldg(reinterpret_cast<const float4*>(a.x + tok * a.ldx + a.col0 + cc[u]));
          if (cc[u] == a.one_col) v[u].x = 1.f;
        }
      }
#pragma unroll
      for (int u = 0; u < PK_U; ++u) {
        if (rr[u] < 0) continue;
        const PackRow pr = rows[rr[u]];
        if (a.scale && pr.tok >= 0 && cc[u] < a.C) {
          const float4 sc = __ldg(reinterpret_cast<const float4*>(a.scale + pr.grp * a.C + cc[u]));
          const float4 sh = __ldg(reinterpret_cast<const float4*>(a.shift + pr.grp * a.C + cc[u]));
          v[u].x = fmaf(v[u].x, sc.x, sh.x); v[u].y = fmaf(v[u].y, sc.y, sh.y);
          v[u].z = fmaf(v[u].z, sc.z, sh.z); v[u].w = fmaf(v[u].w, sc.w, sh.w);
        }
        __half2 lo = __floats2half2_rn(v[u].x, v[u].y), hi = __floats2half2_rn(v[u].z, v[u].w);
        *reinterpret_cast<uint2*>(tile + rr[u] * ld + cc[u]) =
            make_uint2(*reinterpret_cast<uint32_t*>(&lo), *reinterpret_cast<uint32_t*>(&hi));
      }
    }
  } else {
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    for (int r = warp; r < 128; r += 8) {
      const PackRow pr = rows[r];
      const bool ok = pr.tok >= 0;
      const float* row = a.x + (ok ? pr.tok : 0) * a.ldx + a.col0;
      const float* sc = a.scale ? a.scale + pr.grp * a.C : nullptr;
      const float* sh = a.scale ? a.shift + pr.grp * a.C : nullptr;
      for (int c = lane; c < kw; c += 32) {
        float v = 0.f;
        if (ok && c < a.C) {
          v = row[c];
          if (sc) v = fmaf(v, sc[c], sh[c]);
        }
        if (c == a.one_col) v = 1.f;
        tile[r * ld + c] = __float2half_rn(v);
      }
    }
  }
  __syncthreads();
  __half* dst = a.out + (size_t)m * a.kcores * 128 * 8;
  for (int i = threadIdx.x; i < a.kcores * 128; i += 256) {
    const int kc = i >> 7, r = i & 127;
    *reinterpret_cast<uint4*>(dst + (size_t)i * 8) = *reinterpret_cast<const uint4*>(tile + r * ld + kc * 8);
  }
}


// Asynchronous variant (vectorisable shapes): the block's rows arrive in an f32 shared-memory tile by bulk copies (no
// registers held), and the block then converts from there: thread = (k-core, row) reads 8 floats, applies the affine and
// stores one 16-byte KB8 core entry.  The register-staged kernel above held at most 8 loads per thread and measured
// 0.885 ms = 2.9 TB/s at BASELINE config 2 whatever that count (profiles/r01/call26, call42).
// Row stride LD floats with LD % 8 == 4 (C itself for N = 196, C + 4 for N = 384 / 768): consecutive rows start 4 banks
// apart, so the 8 rows of one 16-byte-access phase cover all 32 banks.
// A block owns PACK_ROWS = 32 rows of every k-core of a tile (four blocks per tile): a block loads, waits, then converts, and
// only co-resident blocks overlap those phases.  MEASURED (profiles/r02 call53 / call54, N = 196, config 2): 128-row blocks
// (2 per SM) 595 / 614 us per call (time / band axis), 64-row blocks 463 / 541 us, 32-row blocks (8 per SM) 402 / 447 us;
// FlowSE config 4 5.78 s (32) vs 5.84 s (64).
constexpr int PACK_ROWS = 32;
__global__ void __launch_bounds__(256) norm_cast_kb8_async_kernel(const __grid_constant__ PackArgs a, int ld) {
  constexpr int ROWS = PACK_ROWS;
  extern __shared__ __align__(128) unsigned char smem_raw[];
  float* tile = reinterpret_cast<float*>(smem_raw);                    // [ROWS][ld]
  PackRow* rows = reinterpret_cast<PackRow*>(smem_raw + (size_t)ROWS * ld * 4);
  constexpr int PARTS = 128 / ROWS;
  int m = blockIdx.x / PARTS;
  const int r0 = (blockIdx.x % PARTS) * ROWS;
  if (a.m_inner > 1) m = (m % a.m_inner) * a.tiles_per_step + m / a.m_inner;     // band innermost (see PackArgs::m_inner)
  const int step = m / a.tiles_per_step, j = m - step * a.tiles_per_step;
  if (threadIdx.x < ROWS) {
    const int r = threadIdx.x;
    const long seq = (long)j * 128 + r0 + r;
    PackRow pr{-1, 0};
    if (seq < a.R) {
      pr.tok = (seq / a.seq_inner) * a.seq_outer + (seq % a.seq_inner) * a.seq_inner_stride + (long)step * a.step_stride;
      if (a.scale) pr.grp = (pr.tok / a.tokens_per_sample) * a.g_inner + (a.g_inner > 1 ? pr.tok % a.g_inner : 0);
    }
    rows[r] = pr;
  }
  __syncthreads();
  // one bulk (1-D TMA) copy per row: C*4 contiguous bytes, completion counted on one mbarrier.  The DMA engine issues
  // whole-row bursts instead of separate 16-byte requests.
  __shared__ uint64_t bar;
  if (threadIdx.x == 0) { umma::mbar_init(&bar, ROWS); umma::fence_barrier_init(); }
  __syncthreads();
  if (a.bulk == 3) {
    if (threadIdx.x < ROWS) {
      if (threadIdx.x == 0) {
        umma::mbar_expect_tx(&bar, (uint32_t)ROWS * (uint32_t)a.C * 4);
        tma_load_2d(tile, &a.tmap, step * a.tm_col_step, j * 128 + r0, &bar);
      } else {
        umma::mbar_arrive(&bar);
      }
    }
  } else if (threadIdx.x < ROWS) {
    const int r = threadIdx.x;
    const long tok = rows[r].tok;
    // dense rows (ldx == C == ld, time axis: the K bands of a frame are consecutive tokens): the rows of a warp whose
    // tokens are consecutive are one contiguous run in HBM and in the tile and arrive by ONE bulk copy
    uint32_t nr = tok >= 0 ? 1u : 0u;
    if (a.bulk == 2) {
      const int lane = threadIdx.x & 31;
      const long ptok = __shfl_up_sync(0xffffffffu, tok, 1);
      const bool head = tok >= 0 && (lane == 0 || ptok < 0 || tok != ptok + 1);
      const unsigned heads = __ballot_sync(0xffffffffu, head), oks = __ballot_sync(0xffffffffu, tok >= 0);
      const unsigned above = lane == 31 ? 0u : ((heads | ~oks) & ~((2u << lane) - 1u));
      nr = head ? (uint32_t)((above ? __ffs(above) - 1 : 32) - lane) : 0u;
    }
    if (nr) {
      umma::mbar_expect_tx(&bar, nr * (uint32_t)a.C * 4);
      umma::bulk_g2s(tile + (size_t)r * ld, a.x + tok * a.ldx + a.col0, nr * (uint32_t)a.C * 4, &bar);
    } else {
      umma::mbar_arrive(&bar);
    }
  }
  umma::mbar_wait(&bar, 0);
  __syncthreads();
  __half* dst = a.out + (size_t)m * a.kcores * 128 * 8;
  for (int i = threadIdx.x; i < a.kcores * ROWS; i += 256) {
    const int kc = i / ROWS, r = i % ROWS;
    const PackRow pr = rows[r];
    const int c0 = kc * 8;
    float v[8];
#pragma unroll
    for (int h = 0; h < 2; ++h) {
      const int c = c0 + 4 * h;
      float4 x4 = make_float4(0.f, 0.f, 0.f, 0.f);
      if (pr.tok >= 0 && c < a.C) {                                    // C % 4 == 0: a 4-group is all valid or all padding
        x4 = *reinterpret_cast<const float4*>(tile + r * ld + c);
        if (a.scale) {
          const float4 sc = __ldg(reinterpret_cast<const float4*>(a.scale + pr.grp * a.C + c));
          const float4 sh = __ldg(reinterpret_cast<const float4*>(a.shift + pr.grp * a.C + c));
          x4.x = fmaf(x4.x, sc.x, sh.x); x4.y = fmaf(x4.y, sc.y, sh.y);
          x4.z = fmaf(x4.z, sc.z, sh.z); x4.w = fmaf(x4.w, sc.w, sh.w);
        }
      }
      if (c == a.one_col) x4.x = 1.f;
      v[4 * h] = x4.x; v[4 * h + 1] = x4.y; v[4 * h + 2] = x4.z; v[4 * h + 3] = x4.w;
    }
    const __half2 p0 = __floats2half2_rn(v[0], v[1]), p1 = __floats2half2_rn(v[2], v[3]);
    const __half2 p2 = __floats2half2_rn(v[4], v[5]), p3 = __floats2half2_rn(v[6], v[7]);
    *reinterpret_cast<uint4*>(dst + ((size_t)kc * 128 + r0 + r) * 8) =
        make_uint4(*reinterpret_cast<const uint32_t*>(&p0), *reinterpret_cast<const uint32_t*>(&p1),
                   *reinterpret_cast<const uint32_t*>(&p2), *reinterpret_cast<const uint32_t*>(&p3));
  }
}

}  // namespace bsrnn
using namespace bsrnn;

extern "C" int bsrnn_norm_cast_kb8_ones(const float* x, const float* scale, const float* shift, void* out, long ldx,
                                   int col0, int C, int kcores, int m_tiles, int tiles_per_step, int R,
                                   long seq_inner, long seq_outer, long seq_inner_stride, long step_stride,
                                   long tokens_per_sample, int g_inner, int one_col, void* stream) {
  BSRNN_CHECK_ARG(x && out && C > 0 && kcores * 8 >= C && m_tiles > 0 && tiles_per_step > 0 && seq_inner > 0 &&
                  tokens_per_sample > 0 && g_inner > 0, "norm_cast_kb8: bad arguments");
  BSRNN_CHECK_ARG((scale == nullptr) == (shift == nullptr), "norm_cast_kb8: scale and shift come together");
  BSRNN_CHECK_ARG(one_col < 0 || (one_col >= C && one_col < kcores * 8 && one_col % 4 == 0),
                  "norm_cast_kb8: the constant-one column must be a padding column (multiple of 4)");
  PackArgs a{x, scale, shift, reinterpret_cast<__half*>(out), ldx, col0, C, kcores, tiles_per_step, R,
             seq_inner, seq_outer, seq_inner_stride, step_stride, tokens_per_sample, g_inner, one_col};
  const size_t smem = (size_t)128 * (kcores * 8 + 8) * 2 + 128 * sizeof(PackRow);
  const int vec_ok = (C % 4 == 0 && col0 % 4 == 0 && ldx % 4 == 0 && (reinterpret_cast<uintptr_t>(x) & 15) == 0 &&
                      (!scale || ((reinterpret_cast<uintptr_t>(scale) & 15) == 0 && (reinterpret_cast<uintptr_t>(shift) & 15) == 0)))
                         ? 1 : 0;
  // asynchronous kernel: vectorisable shapes whose f32 block tile fits (bank-friendly row stride)
  const int ld = (C % 8 == 4) ? C : C + 4;              // bank-friendly row stride of the staging tile
  a.bulk = (ld == C && ldx == C && col0 == 0) ? 2 : 1;
  const size_t smem_async = (size_t)PACK_ROWS * ld * 4 + PACK_ROWS * sizeof(PackRow);
  // band axis (seq_inner == 1: token = seq * seq_outer + step * step_stride): the block's rows are a box of the row-major
  // matrix [R rows][seq_outer * ldx floats] -> one tensor copy (the box is PACK_ROWS x C)
  if (ld == C && col0 == 0 && seq_inner == 1 && seq_inner_stride == 0 &&
      (long)(m_tiles / tiles_per_step - 1) * step_stride * ldx + C <= seq_outer * ldx && step_stride * ldx < (1L << 30) &&
      make_tmap_2d_f32(&a.tmap, x, (uint64_t)(seq_outer * ldx), (uint64_t)R, (uint64_t)(seq_outer * ldx) * 4, (uint32_t)C,
                       (uint32_t)PACK_ROWS)) {
    a.bulk = 3;
    a.tm_col_step = (int)(step_stride * ldx);
    if (m_tiles % tiles_per_step == 0 && m_tiles / tiles_per_step > 1) a.m_inner = m_tiles / tiles_per_step;
  }
  if (vec_ok && C % 4 == 0 && smem_async <= 110 * 1024 && (one_col < 0 || one_col % 4 == 0)) {
    BSRNN_CUDA_OK(cudaFuncSetAttribute(norm_cast_kb8_async_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_async));
    norm_cast_kb8_async_kernel<<<(128 / PACK_ROWS) * m_tiles, 256, smem_async, (cudaStream_t)stream>>>(a, ld);
    BSRNN_LAUNCH_OK();
    return 0;
  }
  BSRNN_CUDA_OK(cudaFuncSetAttribute(norm_cast_kb8_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  norm_cast_kb8_kernel<<<m_tiles, 256, smem, (cudaStream_t)stream>>>(a, vec_ok);
  BSRNN_LAUNCH_OK();
  return 0;
}

extern "C" int bsrnn_norm_cast_kb8(const float* x, const float* scale, const float* shift, void* out, long ldx,
                                   int col0, int C, int kcores, int m_tiles, int tiles_per_step, int R,
                                   long seq_inner, long seq_outer, long seq_inner_stride, long step_stride,
                                   long tokens_per_sample, int g_inner, void* stream) {
  return bsrnn_norm_cast_kb8_ones(x, scale, shift, out, ldx, col0, C, kcores, m_tiles, tiles_per_step, R, seq_inner,
                                  seq_outer, seq_inner_stride, step_stride, tokens_per_sample, g_inner, -1, stream);
}

// ---------------------------------------------------------------------------------------------- KB8 transpose (training)
// The weight-gradient GEMMs contract over TOKENS (dW = dG^T X), so both operands are needed with tokens as the K axis.
// src: KB8 [..][kc_src][128][8] = matrix X[row = m*128 + r][col = kc*8 + e].  dst: KB8 of X^T,
// [n_tiles][dst_kcores][BN][8]: dst row (n*BN + c) = src column, dst k index = dst_kc0*8 + (m - src_m0)*128 + r.
// Source columns >= kc_src*8 read as zero.  grid (m_count, n_tiles); the caller zeroes whatever dst k-cores no source
// tile covers (the one-step shift of h_{t-1} leaves a block of zeros).
namespace bsrnn {
__global__ void __launch_bounds__(256) kb8_transpose_kernel(const __half* __restrict__ src, __half* __restrict__ dst, int kc_src,
                                                            int BN, long dst_kcores, long dst_kc0, int src_m0) {
  extern __shared__ __align__(128) unsigned char smem_raw[];
  __half* tile = reinterpret_cast<__half*>(smem_raw);            // [128][BN + 8]
  const int ld = BN + 8;
  const int m = blockIdx.x, n = blockIdx.y;
  const int ncores = BN >> 3;
  const uint4* s4 = reinterpret_cast<const uint4*>(src) + ((size_t)(src_m0 + m) * kc_src) * 128;
  for (int idx = threadIdx.x; idx < ncores * 128; idx += blockDim.x) {
    const int kc = idx >> 7, r = idx & 127;
    const int gkc = n * ncores + kc;
    uint4 v = make_uint4(0u, 0u, 0u, 0u);
    if (gkc < kc_src) v = __ldg(s4 + (size_t)gkc * 128 + r);
    *reinterpret_cast<uint4*>(tile + (size_t)r * ld + kc * 8) = v;
  }
  __syncthreads();
  uint4* d4 = reinterpret_cast<uint4*>(dst) + ((size_t)n * dst_kcores + dst_kc0 + (size_t)m * 16) * BN;
  for (int idx = threadIdx.x; idx < 16 * BN; idx += blockDim.x) {
    const int kk = idx / BN, c = idx - kk * BN;
    __half h[8];
#pragma unroll
    for (int e = 0; e < 8; ++e) h[e] = tile[(size_t)(kk * 8 + e) * ld + c];
    d4[(size_t)kk * BN + c] = *reinterpret_cast<const uint4*>(h);
  }
}
}  // namespace bsrnn

extern "C" int bsrnn_kb8_transpose(const void* src, void* dst, int src_m0, int m_count, int kc_src, int BN, int n_tiles,
                                   long dst_kcores, long dst_kc0, void* stream) {
  BSRNN_CHECK_ARG(src && dst && m_count > 0 && kc_src > 0 && BN >= 16 && BN <= 256 && BN % 8 == 0 && n_tiles > 0 &&
                  dst_kc0 >= 0 && dst_kc0 + (long)m_count * 16 <= dst_kcores, "kb8_transpose: bad arguments");
  const size_t smem = (size_t)128 * (BN + 8) * 2;
  BSRNN_CUDA_OK(cudaFuncSetAttribute(bsrnn::kb8_transpose_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  dim3 grid(m_count, n_tiles);
  bsrnn::kb8_transpose_kernel<<<grid, 256, smem, (cudaStream_t)stream>>>(reinterpret_cast<const __half*>(src),
                                                                          reinterpret_cast<__half*>(dst), kc_src, BN,
                                                                          dst_kcores, dst_kc0, src_m0);
  BSRNN_LAUNCH_OK();
  return 0;
}
