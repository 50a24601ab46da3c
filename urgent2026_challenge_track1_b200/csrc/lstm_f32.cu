// lstm_f32.cu — f32 BLSTM recurrence (CUDA cores), one launch per step covering both directions.
// Replaces nn.LSTM(N, 2N, batch_first, bidirectional) forward with zero initial state
// [bsrnn_flowse.py:226-238 construct; :296-297 time axis, :303-304 band axis]; gate order i,f,g,o;
// c' = sig(f)*c + sig(i)*tanh(g), h = sig(o)*tanh(c').  The bf16 mode runs the persistent tcgen05 kernel in
// lstm_tc.cu instead.  y doubles as the carrier of h between steps, so no separate hidden-state buffer exists.
#include "common.cuh"

namespace bsrnn {

constexpr int LM = 64, LU = 16, LK = 16, LT = 256;   // 64 sequences x 16 hidden units (x4 gates) per CTA

struct SeqAddr {
  long seq_inner, seq_outer, seq_inner_stride, step_stride;
  __device__ __forceinline__ long token(long r, long s) const {
    return (r / seq_inner) * seq_outer + (r % seq_inner) * seq_inner_stride + s * step_stride;
  }
};

// grid (ceil(H/16), ceil(R/64), 2)
__global__ void __launch_bounds__(LT)
lstm_step_f32_kernel(const float* __restrict__ gates_x, const float* __restrict__ w_hh, float* __restrict__ y,
                     float* __restrict__ c_state, float* __restrict__ saved, int R, int H, int step, int steps,
                     SeqAddr addr) {
  const int d = blockIdx.z;
  const int u0 = blockIdx.x * LU;
  const int r0 = blockIdx.y * LM;
  const int s_cur = d == 0 ? step : steps - 1 - step;
  const int s_prev = d == 0 ? s_cur - 1 : s_cur + 1;
  const int tid = threadIdx.x, tx = tid & 15, ty = tid >> 4;
  const int lr = tid >> 2, lk = (tid & 3) * 4;

  __shared__ float As[LK][LM + 4];
  __shared__ float Bs[LK][LM + 4];
  float acc[4][4];
#pragma unroll
  for (int i = 0; i < 4; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) acc[i][j] = 0.f;

  if (step > 0) {
    const int arow = r0 + lr;
    const float* hp = arow < R ? y + addr.token(arow, s_prev) * (2L * H) + (long)d * H : nullptr;
    const int gate = lr >> 4, ul = lr & 15;
    const bool w_ok = (u0 + ul) < H;
    const float* wp = w_hh + ((long)d * 4 * H + (long)gate * H + u0 + ul) * H;
    for (int k0 = 0; k0 < H; k0 += LK) {
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        const int k = k0 + lk + u;
        As[lk + u][lr] = (hp && k < H) ? hp[k] : 0.f;
        Bs[lk + u][lr] = (w_ok && k < H) ? wp[k] : 0.f;
      }
      __syncthreads();
#pragma unroll
      for (int k = 0; k < LK; ++k) {
        float a[4], b[4];
#pragma unroll
        for (int i = 0; i < 4; ++i) a[i] = As[k][ty * 4 + i];
#pragma unroll
        for (int j = 0; j < 4; ++j) b[j] = Bs[k][tx + 16 * j];
#pragma unroll
        for (int i = 0; i < 4; ++i)
#pragma unroll
          for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(a[i], b[j], acc[i][j]);
      }
      __syncthreads();
    }
  }
  const int u = u0 + tx;
  if (u >= H) return;
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int r = r0 + ty * 4 + i;
    if (r >= R) continue;
    const long tok = addr.token(r, s_cur);
    const float* gx = gates_x + tok * (8L * H) + (long)d * 4 * H;
    const float pi = acc[i][0] + gx[u];
    const float pf = acc[i][1] + gx[H + u];
    const float pg = acc[i][2] + gx[2 * H + u];
    const float po = acc[i][3] + gx[3 * H + u];
    const float ig = 1.f / (1.f + expf(-pi));
    const float fg = 1.f / (1.f + expf(-pf));
    const float gg = tanhf(pg);
    const float og = 1.f / (1.f + expf(-po));
    float* cp = c_state + ((long)d * R + r) * H + u;
    const float c_prev = step > 0 ? *cp : 0.f;
    const float c_new = fg * c_prev + ig * gg;
    *cp = c_new;
    y[tok * (2L * H) + (long)d * H + u] = og * tanhf(c_new);
    if (saved) {                                    // training: gate activations and cell state for the backward pass
      float* sv = saved + (tok * 2 + d) * (5L * H) + u;
      sv[0] = ig; sv[H] = fg; sv[2L * H] = gg; sv[3L * H] = og; sv[4L * H] = c_new;
    }
  }
}

}  // namespace bsrnn
using namespace bsrnn;

extern "C" int bsrnn_blstm_recurrence_f32(const float* gates_x, const float* w_hh, float* y, float* c_state, int R,
                                          int steps, int H, long seq_inner, long seq_outer, long seq_inner_stride,
                                          long step_stride, void* stream) {
  BSRNN_CHECK_ARG(gates_x && w_hh && y && c_state, "blstm_recurrence_f32: null pointer");
  BSRNN_CHECK_ARG(R > 0 && steps > 0 && H > 0 && seq_inner > 0, "blstm_recurrence_f32: bad dims");
  SeqAddr addr{seq_inner, seq_outer, seq_inner_stride, step_stride};
  dim3 grid(cdiv(H, LU), cdiv(R, LM), 2);
  for (int s = 0; s < steps; ++s) {
    lstm_step_f32_kernel<<<grid, LT, 0, (cudaStream_t)stream>>>(gates_x, w_hh, y, c_state, nullptr, R, H, s, steps, addr);
  }
  BSRNN_LAUNCH_OK();
  count_launches(steps - 1);
  return 0;
}

// ---------------------------------------------------------------------------------------------------- training
// Forward that also saves (i, f, g, o, c) per (token, direction): saved (tokens, 2, 5, H) f32.
extern "C" int bsrnn_blstm_train_fwd_f32(const float* gates_x, const float* w_hh, float* y, float* c_state, float* saved,
                                         int R, int steps, int H, long seq_inner, long seq_outer, long seq_inner_stride,
                                         long step_stride, void* stream) {
  BSRNN_CHECK_ARG(gates_x && w_hh && y && c_state && saved, "blstm_train_fwd_f32: null pointer");
  BSRNN_CHECK_ARG(R > 0 && steps > 0 && H > 0 && seq_inner > 0, "blstm_train_fwd_f32: bad dims");
  SeqAddr addr{seq_inner, seq_outer, seq_inner_stride, step_stride};
  dim3 grid(cdiv(H, LU), cdiv(R, LM), 2);
  for (int s = 0; s < steps; ++s)
    lstm_step_f32_kernel<<<grid, LT, 0, (cudaStream_t)stream>>>(gates_x, w_hh, y, c_state, saved, R, H, s, steps, addr);
  BSRNN_LAUNCH_OK();
  count_launches(steps - 1);
  return 0;
}

namespace bsrnn {

// Backward through time, one (elementwise, GEMM) kernel pair per step, both directions per launch.
// q = 0..steps-1 walks each direction against its forward order: position p = steps-1-q (d = 0) or q (d = 1).
//   dh      = dy[p, d] + dh_rec[d]            (dh_rec = dG_{next} W_hh from the step processed just before)
//   dc      = dh * o * (1 - tanh(c)^2) + dc_carry[d]     ; dc_carry <- dc * f
//   dG      = (dc*g*i(1-i), dc*c_prev*f(1-f), dc*i*(1-g^2), dh*tanh(c)*o(1-o))   -> dgates[p, d] (grad of gates_x)
// grid (ceil(H/256), min(R, 65535), 2), block 256: sequences r = blockIdx.y + j * gridDim.y (R = B*T on the band axis
// can exceed the 65535 limit of grid.y)
__global__ void __launch_bounds__(256)
lstm_bwd_gates_kernel(const float* __restrict__ dy, const float* __restrict__ saved, const float* __restrict__ dh_rec,
                      float* __restrict__ dc_carry, float* __restrict__ dgates, int R, int H, int q, int steps,
                      SeqAddr addr) {
  const int u = blockIdx.x * 256 + threadIdx.x;
  const int d = blockIdx.z;
  if (u >= H) return;
  const int p = d == 0 ? steps - 1 - q : q;
  const int p_prev = d == 0 ? p - 1 : p + 1;                 // forward-order predecessor
  for (int r = blockIdx.y; r < R; r += gridDim.y) {
    const long tok = addr.token(r, p);
    const float* sv = saved + (tok * 2 + d) * (5L * H) + u;
    const float ig = sv[0], fg = sv[H], gg = sv[2L * H], og = sv[3L * H], c = sv[4L * H];
    float c_prev = 0.f;
    if (p_prev >= 0 && p_prev < steps) c_prev = saved[(addr.token(r, p_prev) * 2 + d) * (5L * H) + 4L * H + u];
    const long si = ((long)d * R + r) * H + u;
    float dh = dy[tok * (2L * H) + (long)d * H + u];
    float dc = 0.f;
    if (q > 0) { dh += dh_rec[si]; dc = dc_carry[si]; }
    const float tc = tanhf(c);
    dc += dh * og * (1.f - tc * tc);
    dc_carry[si] = dc * fg;
    float* dg = dgates + (tok * 2 + d) * (4L * H) + u;
    dg[0] = dc * gg * ig * (1.f - ig);
    dg[H] = dc * c_prev * fg * (1.f - fg);
    dg[2L * H] = dc * ig * (1.f - gg * gg);
    dg[3L * H] = dh * tc * og * (1.f - og);
  }
}

// dh_rec[d, r, k] = sum_n dgates[p, d, r, n] * W_hh[d, n, k]      (R x 4H) @ (4H x H); 64x64x16 tiles
// grid (ceil(H/64), ceil(R/64), 2), block 256
__global__ void __launch_bounds__(256)
lstm_bwd_dh_kernel(const float* __restrict__ dgates, const float* __restrict__ w_hh, float* __restrict__ dh_rec, int R,
                   int H, int q, int steps, SeqAddr addr) {
  const int d = blockIdx.z;
  const int k0 = blockIdx.x * 64, r0 = blockIdx.y * 64;
  const int p = d == 0 ? steps - 1 - q : q;
  const int tid = threadIdx.x, tx = tid & 15, ty = tid >> 4;
  __shared__ float As[16][64 + 4];      // [n][row]
  __shared__ float Bs[16][64 + 4];      // [n][k]
  float acc[4][4];
#pragma unroll
  for (int i = 0; i < 4; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) acc[i][j] = 0.f;
  const int lr = tid >> 2, ln = (tid & 3) * 4;          // A loader: row lr, 4 consecutive n
  const int bn = tid >> 4, bk = (tid & 15) * 4;          // B loader: n row bn, 4 consecutive k
  const int arow = r0 + lr;
  const float* ap = arow < R ? dgates + (addr.token(arow, p) * 2 + d) * (4L * H) : nullptr;
  const float* wp = w_hh + (long)d * 4 * H * H;
  const int N4 = 4 * H;
  for (int n0 = 0; n0 < N4; n0 += 16) {
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      const int n = n0 + ln + u;
      As[ln + u][lr] = (ap && n < N4) ? ap[n] : 0.f;
    }
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      const int n = n0 + bn, k = k0 + bk + u;
      Bs[bn][bk + u] = (n < N4 && k < H) ? wp[(long)n * H + k] : 0.f;
    }
    __syncthreads();
#pragma unroll
    for (int n = 0; n < 16; ++n) {
      float a[4], b[4];
#pragma unroll
      for (int i = 0; i < 4; ++i) a[i] = As[n][ty * 4 + i];
#pragma unroll
      for (int j = 0; j < 4; ++j) b[j] = Bs[n][tx * 4 + j];
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(a[i], b[j], acc[i][j]);
    }
    __syncthreads();
  }
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int r = r0 + ty * 4 + i;
    if (r >= R) continue;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int k = k0 + tx * 4 + j;
      if (k < H) dh_rec[((long)d * R + r) * H + k] = acc[i][j];
    }
  }
}

}  // namespace bsrnn

// dy (tokens, 2H), saved (tokens, 2, 5, H), w_hh (2, 4H, H) -> dgates (tokens, 2, 4H) = dL/d gates_x.
// scratch: dh_rec and dc_carry, (2, R, H) f32 each.
extern "C" int bsrnn_blstm_train_bwd_f32(const float* dy, const float* saved, const float* w_hh, float* dgates,
                                         float* dh_rec, float* dc_carry, int R, int steps, int H, long seq_inner,
                                         long seq_outer, long seq_inner_stride, long step_stride, void* stream) {
  BSRNN_CHECK_ARG(dy && saved && w_hh && dgates && dh_rec && dc_carry, "blstm_train_bwd_f32: null pointer");
  BSRNN_CHECK_ARG(R > 0 && steps > 0 && H > 0 && seq_inner > 0, "blstm_train_bwd_f32: bad dims");
  SeqAddr addr{seq_inner, seq_outer, seq_inner_stride, step_stride};
  cudaStream_t st = (cudaStream_t)stream;
  dim3 g1(cdiv(H, 256), R < 65535 ? R : 65535, 2), g2(cdiv(H, 64), cdiv(R, 64), 2);
  for (int q = 0; q < steps; ++q) {
    lstm_bwd_gates_kernel<<<g1, 256, 0, st>>>(dy, saved, dh_rec, dc_carry, dgates, R, H, q, steps, addr);
    if (q + 1 < steps) lstm_bwd_dh_kernel<<<g2, 256, 0, st>>>(dgates, w_hh, dh_rec, R, H, q, steps, addr);
  }
  BSRNN_LAUNCH_OK();
  count_launches(2 * steps - 2);
  return 0;
}
