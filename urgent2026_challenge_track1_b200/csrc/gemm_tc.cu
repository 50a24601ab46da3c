// gemm_tc.cu — persistent, warp-specialised fp16-operand GEMM on tcgen05 tensor cores (sm_100a), f32 accumulation
// in TMEM.  (fp16 rather than bf16 operands: same tensor-pipe rate, 3 more mantissa bits; every operand on this path
// is GroupNorm-normalised, a tanh/sigmoid product, or a weight, so the fp16 range is never an issue.)
//
//   C[128*m_tiles, BN*n_tiles] = A_kb8 * W_kb8^T   (+ fused epilogue)
//
// Operands live in HBM in the UMMA-native "KB8" layout (umma.cuh), so each pipeline stage is filled by two plain
// cp.async.bulk copies.  Roles: warp 0 = bulk-copy producer, warp 1 = single-thread tcgen05.mma issuer, warps 2-9 =
// epilogue (tcgen05.ld -> registers -> fused op -> global): two warps per TMEM lane quadrant, each taking half of the
// tile's column chunks (these GEMMs have K <= 800, so a 4-warp epilogue was the pacing stage).  Two 256-column TMEM
// accumulators let the epilogue of tile i overlap the MMAs of tile i+1.  The residual epilogue transposes each
// 32x32 chunk through a per-warp shared-memory scratch so that the f32 read-modify-write of the residual stream
// moves whole 128-byte lines.  One CTA per SM, static round-robin tile schedule with the N tile innermost so
// concurrently running CTAs share the same A tile through L2.
//
// Used for (fp16 tensor-core mode): LSTM input projections, Linear(4N->N)+skip (+GroupNorm statistics of the result),
// MaskDecoder Conv1d(N->4N)+tanh and Conv1d(4N->4s)+GLU   [reference bsrnn_flowse.py:296-307 pattern, espnet2
// MaskDecoder].
#include "common.cuh"
#include "umma.cuh"
#include "tmap.cuh"
#include <cuda_fp16.h>
#include <stdlib.h>

namespace bsrnn {
using namespace umma;

constexpr int TC_STAGES = 8;       // barrier slots; a launch uses a.stages (<= 8, chosen by shared-memory fit) of them
constexpr int TC_KS = 8;            // k-cores (8 halves each) per pipeline stage -> K = 64 per stage
constexpr int TC_EPI_WARPS = 8;
// Epilogue warps per CTA.  The residual epilogue (Linear + skip) runs 12 (16 would cap the kernel at 96 registers and spill 4 KB): it is a scattered-row read-modify-write of the f32
// residual stream whose cost is set by the bytes its warps keep in flight (profiles/r02 call43: 0.81 ms without the
// residual traffic, 1.45 ms store-only, 1.80 ms full, all with 8 warps).
constexpr int TC_RESID_EPI_WARPS = 12;
__host__ __device__ constexpr int tc_epi_warps(int epi) { return (epi == 1 /* EPI_RESID_F32 */ || epi == 8 /* EPI_RESID_TMA */) ? TC_RESID_EPI_WARPS : TC_EPI_WARPS; }
__host__ __device__ constexpr int tc_threads(int epi) { return (2 + tc_epi_warps(epi)) * 32; }
constexpr int TC_SCR_LD = 36;                                   // floats per scratch row (32 + 4: conflict-free 16 B rows)
constexpr int TC_SCR_BYTES = tc_epi_warps(1) * 32 * TC_SCR_LD * 4;  // residual epilogue only
constexpr int TC_ACC_COLS = 256;

struct RowMap {                     // global row (m_tile, r) -> token
  int tiles_per_step;               // m_tile = step * tiles_per_step + j ; seq = j*128 + r
  int R;                            // valid sequences
  long seq_inner, seq_outer, seq_inner_stride, step_stride;
  __device__ __forceinline__ bool map(int m_tile, int r, long* token) const {
    const int step = m_tile / tiles_per_step;
    const int j = m_tile - step * tiles_per_step;
    const int seq = j * 128 + r;                   // < R (int)
    if (seq >= R) return false;
    // the general form costs two 64-bit divisions per row and tile (9 % of the Linear+skip epilogue's samples, profiles/r02
    // call52): band axis / plain rows need none, the time axis one 32-bit division
    if (seq_inner == 1) *token = (long)seq * seq_outer + (long)step * step_stride;
    else if (seq_inner >= (long)R) *token = (long)seq * seq_inner_stride + (long)step * step_stride;
    else {
      const int si = (int)seq_inner, q = seq / si;
      *token = (long)q * seq_outer + (long)(seq - q * si) * seq_inner_stride + (long)step * step_stride;
    }
    return true;
  }
};

struct GemmTcArgs {
  const __half* A;           // [m_tiles][kcores][128][8]
  const __half* W;           // [n_tiles][kcores][BN][8]
  const float* bias;                // [n_tiles*BN] or null
  void* out;
  double* stats;                    // EPI_RESID: (samples, 2) sum / sumsq accumulators or null
  long ldo;                         // output row stride (elements)
  long tokens_per_sample;
  int m_tiles, n_tiles, kcores, BN;
  int n_valid;                      // logical output columns kept
  int out_kcores;                   // EPI_TANH_KB8: k-cores of the destination operand
  int b_resident;                   // 1: each CTA keeps ONE weight tile in shared memory and streams A tiles only
  int pf_dist;                      // A tile this many tiles ahead is bulk-prefetched into L2 (0 = off)
  const __half* gx;                 // EPI_LSTM_STEP: input projection rows [m*128 + r][ld_gx] fp16 (this step, this direction)
  float* cstate;                    // EPI_LSTM_STEP: cell state [m*128 + r][H] f32 (this direction), updated in place
  long ld_gx;
  int H;
  // EPI_LSTM_STEP / EPI_LSTM_BWD, both directions in one launch (streaming schedule): row tiles m >= dir_tiles belong to
  // the second direction and use the *2 pointers with m - dir_tiles (0 = single direction)
  int dir_tiles;
  const __half* A2; const __half* W2; const __half* gx2; float* cstate2; void* out2;
  int debug;                        // BSRNN_GEMM_DEBUG (A/B experiments on the input projection): 1 = every tile
                                    // writes the first tile's output block (stores stay in L2), 2 = no stores
  int stages;                       // pipeline depth: 8 when the shared memory allows (short-K GEMMs: one tile is 4 stages,
                                    // and a ring of one tile exposes the HBM latency of every A tile), else 4 (3 if 4 do not fit)
  RowMap rows;
  float out_scale;                  // EPI_RESID_F32: the accumulator is multiplied by this before it is added (0 = 1)
  const float* out_scale_ptr;       // ... or by *out_scale_ptr (device scalar: no host sync to learn the loss scale)
  // split-K (EPI_RESID_F32 with atomic adds; weight-gradient GEMMs: few output tiles, K = tokens): the launch iterates
  // over m_tiles = m_log * ksplit tiles; tile m' = split * m_log + m covers k-cores [split*kps, split*kps + kps)
  int ksplit, kps, m_log;
  // training (EPI_LSTM_STEP with save_gates, EPI_LSTM_BWD)
  int save_gates;                   // EPI_LSTM_STEP: write the ACTIVATED gates i,f,g,o back over gx (fp16, same columns) and
                                    // c_t to cstate_out (c_{t-1} is read from cstate; null = zeros): what BPTT needs
  float* cstate_out; float* cstate_out2;
  const __half* dy; const __half* dy2;     // EPI_LSTM_BWD: dL/dh_t rows [m*128 + r][ld_dy] (this step, this direction)
  long ld_dy;
  const float* c_cur; const float* c_cur2;    // c_t rows [m*128 + r][H]
  const float* c_prev; const float* c_prev2;  // c_{t-1} rows (null at the first step of the sequence = zeros)
  int valid_rows;                   // rows >= valid_rows (padding of the last sequence tile) get zero gradients
  alignas(64) CUtensorMap tmap;     // use_tmap: the matrix view of `out` (read through the kernel's __grid_constant__ parameter)
  // EPI_RESID_TMA extras (bsrnn_gemm_tc_ex)
  // Grouped launch (EPI_RESID_TMA, one N tile, streaming weights): tile index t = row_tile * n_groups + g; group g (a band of
  // BandSplit) has its own operand / weight / bias / output offsets and K extent: groups[g] = {a_off (halves, tile 0 of the
  // group), w_off (halves), out_off (floats), bias_off (floats), kcores}.  Bands innermost: CTAs that run together write
  // adjacent 784-byte segments of the same output rows.
  const long long* groups;
  int n_groups;
  // streaming launches with one N tile walk the M tiles from the LAST one down: the MaskDecoder's Conv1d+GLU GEMM reads the 100 MB
  // hidden tile its predecessor has just written in ascending order, so the most recently written (still L2-resident) tiles come
  // first instead of the evicted ones
  int reverse_m;
  // band-axis Linear+skip (tensor-map path): tiles are walked with the STEP (= band) innermost, tile = (lin % m_inner) *
  // tiles_per_step + lin / m_inner, so that the CTAs running together read / write adjacent 784-byte segments of the same rows
  // of the residual stream (whole 26.6 KB rows per DRAM page visit) instead of one segment of 148 x 128 different rows
  int m_inner;
  // EPI_RESID_TMA with a 2-D tensor map (tmap.cuh): the tile's rows are `rows [j*128, +128) x cols [step*tm_col_step (+ group
  // offset), +n_valid)` of a row-major matrix over `out` (band axis, BandSplit): ONE tensor copy per tile and direction
  int use_tmap;
  int tm_col_step;
  int run_merge;                    // 1: rows of consecutive tokens move as one bulk copy (set by the launcher, see run_rows)
  int no_resid;                     // 1: out = acc + bias (store only: the residual rows are neither loaded nor added)
  int stats_inner;                  // > 1: statistics row = (token / tokens_per_sample) * stats_inner + token % stats_inner
                                    // (per (sample, band) sums for the mask decoder's GroupNorm(1, N) over (N, T))
};

enum { EPI_F16_ROWS = 0, EPI_RESID_F32 = 1, EPI_TANH_KB8 = 2, EPI_GLU_F32 = 3, EPI_F16_KB8 = 4, EPI_LSTM_STEP = 5,
       EPI_LSTM_BWD = 6, EPI_TANH_F32 = 7, EPI_RESID_TMA = 8 };

__device__ __forceinline__ float fast_tanh(float x) {
  float y;
  asm("tanh.approx.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
__device__ __forceinline__ float fast_sigmoid(float x) { return fmaf(fast_tanh(0.5f * x), 0.5f, 0.5f); }

__device__ __forceinline__ uint32_t pack_h2(float a, float b) {
  __half2 v = __floats2half2_rn(a, b);
  return *reinterpret_cast<uint32_t*>(&v);
}

// EPI_LSTM_BWD: the operands of one 8-unit sub-block of a row (saved gates, dy, c_t, c_{t-1}, dc carry)
struct BwdSub {
  uint4 g[4];
  uint4 dy;
  float4 cc[2], cq[2], dc[2];
};
__device__ __forceinline__ void bwd_load(BwdSub& R, const __half* sgp, const __half* dyp, const float* ccp, const float* cpp,
                                         const float* dcp, int b8) {
#pragma unroll
  for (int i = 0; i < 4; ++i) R.g[i] = __ldg(reinterpret_cast<const uint4*>(sgp + 32 * b8) + i);
  R.dy = __ldg(reinterpret_cast<const uint4*>(dyp + 8 * b8));
  R.cc[0] = __ldg(reinterpret_cast<const float4*>(ccp + 8 * b8));
  R.cc[1] = __ldg(reinterpret_cast<const float4*>(ccp + 8 * b8 + 4));
  R.cq[0] = R.cq[1] = make_float4(0.f, 0.f, 0.f, 0.f);
  if (cpp) {
    R.cq[0] = __ldg(reinterpret_cast<const float4*>(cpp + 8 * b8));
    R.cq[1] = __ldg(reinterpret_cast<const float4*>(cpp + 8 * b8 + 4));
  }
  R.dc[0] = *reinterpret_cast<const float4*>(dcp + 8 * b8);
  R.dc[1] = *reinterpret_cast<const float4*>(dcp + 8 * b8 + 4);
}
__device__ __forceinline__ void bwd_unit(float dh_rec, float dy, float i_, float f_, float g_, float o_, float ct, float cprev,
                                         float& dc_carry, uint32_t& w0, uint32_t& w1) {
  const float dh = dy + dh_rec;
  const float tc = fast_tanh(ct);
  const float d_o = dh * tc;
  const float dc = dc_carry + dh * o_ * (1.f - tc * tc);
  const float d_i = dc * g_, d_g = dc * i_, d_f = dc * cprev;
  dc_carry = dc * f_;
  w0 = pack_h2(d_i * i_ * (1.f - i_), d_f * f_ * (1.f - f_));
  w1 = pack_h2(d_g * (1.f - g_ * g_), d_o * o_ * (1.f - o_));
}
__device__ __forceinline__ void bwd_compute(BwdSub& R, float a0, float a1, float a2, float a3, float a4, float a5, float a6,
                                            float a7, uint32_t (&dgw)[16]) {
  const __half2* gh = reinterpret_cast<const __half2*>(R.g);
  const __half2* dyh = reinterpret_cast<const __half2*>(&R.dy);
  const float acc[8] = {a0, a1, a2, a3, a4, a5, a6, a7};
  const float ct[8] = {R.cc[0].x, R.cc[0].y, R.cc[0].z, R.cc[0].w, R.cc[1].x, R.cc[1].y, R.cc[1].z, R.cc[1].w};
  const float cp[8] = {R.cq[0].x, R.cq[0].y, R.cq[0].z, R.cq[0].w, R.cq[1].x, R.cq[1].y, R.cq[1].z, R.cq[1].w};
  float dcs[8] = {R.dc[0].x, R.dc[0].y, R.dc[0].z, R.dc[0].w, R.dc[1].x, R.dc[1].y, R.dc[1].z, R.dc[1].w};
#pragma unroll
  for (int j = 0; j < 8; ++j) {
    const float2 g_if = __half22float2(gh[2 * j]), g_go = __half22float2(gh[2 * j + 1]);
    const float2 d2 = __half22float2(dyh[j >> 1]);
    bwd_unit(acc[j], (j & 1) ? d2.y : d2.x, g_if.x, g_if.y, g_go.x, g_go.y, ct[j], cp[j], dcs[j], dgw[2 * j], dgw[2 * j + 1]);
  }
  R.dc[0] = make_float4(dcs[0], dcs[1], dcs[2], dcs[3]);
  R.dc[1] = make_float4(dcs[4], dcs[5], dcs[6], dcs[7]);
}

// Epilogue for NC (16 or 32) accumulator columns [c0, c0+NC) of row r of tile (m, n).
template <int EPI, int NC>
__device__ __forceinline__ void epilogue_chunk(const GemmTcArgs& a, int m, int n, int r, int c0, const uint32_t* acc,
                                               bool row_ok, long token, float& s_sum, float& s_sq, float* scr, int lane,
                                               float bias_lane) {
  const int gc0 = n * a.BN + c0;                      // global output column of acc[0]
  // bias_lane = bias[gc0 + lane]: ONE coalesced load per chunk (issued before the accumulator wait), broadcast by
  // shuffles.  32 dependent uniform loads per chunk were 60 % of the epilogue's stall samples (profiles/r01/call21).
  float v[NC];
  if (a.bias) {
#pragma unroll
    for (int i = 0; i < NC; ++i) v[i] = __uint_as_float(acc[i]) + __shfl_sync(0xffffffffu, bias_lane, i);
  } else {               // bias folded into the weights (constant-one operand column): nothing to add
#pragma unroll
    for (int i = 0; i < NC; ++i) v[i] = __uint_as_float(acc[i]);
  }
  if (EPI == EPI_RESID_F32 && (a.out_scale != 0.f || a.out_scale_ptr)) {
    const float sc = a.out_scale_ptr ? __ldg(a.out_scale_ptr) : a.out_scale;
#pragma unroll
    for (int i = 0; i < NC; ++i) v[i] *= sc;
  }

  if (EPI == EPI_F16_ROWS) {
    if (!row_ok) return;
    __half* o = reinterpret_cast<__half*>(a.out) + token * a.ldo + gc0;
#pragma unroll
    for (int i = 0; i < NC; i += 8) {
      uint4 pk = make_uint4(pack_h2(v[i], v[i + 1]), pack_h2(v[i + 2], v[i + 3]), pack_h2(v[i + 4], v[i + 5]),
                            pack_h2(v[i + 6], v[i + 7]));
      *reinterpret_cast<uint4*>(o + i) = pk;
    }
  } else if (EPI == EPI_RESID_F32) {
    // out[token, gc0 + c] += v[c].  Thread r owns row r; the rows of a warp are 32 scattered tokens of ldo floats, so
    // the chunk goes through the warp's scratch (row stride 36 floats): afterwards 8 lanes cover one row's 128
    // bytes and a warp instruction touches 4 whole lines instead of 32 partial ones.
    if (a.debug & 4) return;             // A/B (BSRNN_GEMM_DEBUG=4): no residual traffic at all -- loads + MMAs only
    float* my = scr + (r & 31) * TC_SCR_LD;
#pragma unroll
    for (int i = 0; i < NC; i += 4) *reinterpret_cast<float4*>(my + i) = make_float4(v[i], v[i + 1], v[i + 2], v[i + 3]);
    __syncwarp();
    const int sub = lane >> 3, c4 = (lane & 7) * 4;
    const unsigned okmask = __ballot_sync(0xffffffffu, row_ok);
    const bool col_ok = c4 < NC && gc0 + c4 + 3 < a.n_valid;     // n_valid % 4 == 0 is checked by the launcher
    // all 8 reads of the residual stream are issued before the first store (the rows are scattered tokens: the
    // compiler cannot prove the stores do not alias the later loads and would serialise 8 DRAM round trips)
    float* optr[8];
    float4 old[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      const int rr = 4 * i + sub;
      const long tok = __shfl_sync(0xffffffffu, token, rr);
      optr[i] = (((okmask >> rr) & 1u) && col_ok) ? reinterpret_cast<float*>(a.out) + tok * a.ldo + gc0 + c4 : nullptr;
      old[i] = make_float4(0.f, 0.f, 0.f, 0.f);
      if (optr[i] && a.ksplit <= 1 && !(a.debug & 8)) old[i] = *reinterpret_cast<const float4*>(optr[i]);   // debug 8: store only
    }
    if (a.ksplit > 1) {                  // split-K: several CTAs add into the same rows
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        if (optr[i]) {
          const float4 nv = *reinterpret_cast<const float4*>(scr + (4 * i + sub) * TC_SCR_LD + c4);
          atomicAdd(optr[i], nv.x); atomicAdd(optr[i] + 1, nv.y); atomicAdd(optr[i] + 2, nv.z); atomicAdd(optr[i] + 3, nv.w);
        }
      }
      __syncwarp();
      return;
    }
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      if (optr[i]) {
        float* sp = scr + (4 * i + sub) * TC_SCR_LD + c4;
        float4 nv = *reinterpret_cast<const float4*>(sp);
        nv.x += old[i].x; nv.y += old[i].y; nv.z += old[i].z; nv.w += old[i].w;
        *reinterpret_cast<float4*>(optr[i]) = nv;
        *reinterpret_cast<float4*>(sp) = nv;             // new values back for the row owner's statistics
      }
    }
    __syncwarp();
    if (row_ok && a.stats && !(a.debug & 16)) {        // debug 16: no statistics
#pragma unroll
      for (int i = 0; i < NC; i += 4) {
        if (gc0 + i + 3 < a.n_valid) {
          const float4 nv = *reinterpret_cast<const float4*>(my + i);
          s_sum += nv.x + nv.y + nv.z + nv.w;
          s_sq += nv.x * nv.x + nv.y * nv.y + nv.z * nv.z + nv.w * nv.w;
        }
      }
    }
    __syncwarp();
  } else if (EPI == EPI_F16_KB8) {
    // a warp stores 32 rows x 16 B = 512 contiguous bytes per instruction
    __half* o = reinterpret_cast<__half*>(a.out) + (((long)m * a.out_kcores + (gc0 >> 3)) * 128 + r) * 8;
#pragma unroll
    for (int i = 0; i < NC; i += 8) {
      uint4 pk = make_uint4(pack_h2(v[i], v[i + 1]), pack_h2(v[i + 2], v[i + 3]), pack_h2(v[i + 4], v[i + 5]),
                            pack_h2(v[i + 6], v[i + 7]));
      *reinterpret_cast<uint4*>(o + (long)(i >> 3) * 1024) = pk;
    }
  } else if (EPI == EPI_LSTM_STEP) {
    // One LSTM step for any hidden size (FlowSE, H = 768): the GEMM is h_{t-1} * W_hh^T with gate-interleaved weight
    // rows (column 4u + gate, i/f/o rows pre-halved like lstm_tc.cu), so a chunk of 32 accumulator columns holds the 4
    // gates of 8 hidden units of this row: add the input projection (fp16, same column order), update c in place,
    // and store h_t as ONE 16-byte KB8 core entry of the tile that is next step's A operand and the layer output.
    // [reference nn.LSTM semantics: bsrnn_flowse.py:226-238; zero initial state = zero A tile and zero c]
    if (NC == 32) {
      const int u0 = gc0 >> 2;
      if (u0 < a.H) {
        const bool dir2 = a.dir_tiles > 0 && m >= a.dir_tiles;
        const int md = dir2 ? m - a.dir_tiles : m;
        const long grow = (long)md * 128 + r;
        const uint4* gp = reinterpret_cast<const uint4*>((dir2 ? a.gx2 : a.gx) + grow * a.ld_gx + gc0);
        const float* cin = dir2 ? a.cstate2 : a.cstate;                     // c_{t-1} (null: zeros, training's first step)
        float* cout = dir2 ? a.cstate_out2 : a.cstate_out;                  // c_t (null: in place)
        const float* cp = cin ? cin + grow * a.H + u0 : nullptr;
        float* cpo = cout ? cout + grow * a.H + u0 : const_cast<float*>(cp);
        uint4 g4[4];
        if (a.save_gates) {                // (the buffer is rewritten below: no read-only path)
#pragma unroll
          for (int i = 0; i < 4; ++i) g4[i] = gp[i];
        } else {
#pragma unroll
          for (int i = 0; i < 4; ++i) g4[i] = __ldg(gp + i);
        }
        float4 c4[2] = {make_float4(0.f, 0.f, 0.f, 0.f), make_float4(0.f, 0.f, 0.f, 0.f)};
        if (cp) { c4[0] = *reinterpret_cast<const float4*>(cp); c4[1] = *reinterpret_cast<const float4*>(cp + 4); }
        float* c = reinterpret_cast<float*>(c4);
        const __half2* gh = reinterpret_cast<const __half2*>(g4);
        float h[8];
        uint32_t sv[16];
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          const float2 g01 = __half22float2(gh[2 * j]), g23 = __half22float2(gh[2 * j + 1]);
          const float ig = fmaf(fast_tanh(v[4 * j] + g01.x), 0.5f, 0.5f), fg = fmaf(fast_tanh(v[4 * j + 1] + g01.y), 0.5f, 0.5f);
          const float gg = fast_tanh(v[4 * j + 2] + g23.x), og = fmaf(fast_tanh(v[4 * j + 3] + g23.y), 0.5f, 0.5f);
          c[j] = fmaf(fg, c[j], ig * gg);
          h[j] = og * fast_tanh(c[j]);
          sv[2 * j] = pack_h2(ig, fg);
          sv[2 * j + 1] = pack_h2(gg, og);
        }
        if (a.save_gates) {
          uint4* gw = const_cast<uint4*>(gp);
#pragma unroll
          for (int i = 0; i < 4; ++i) gw[i] = make_uint4(sv[4 * i], sv[4 * i + 1], sv[4 * i + 2], sv[4 * i + 3]);
        }
        *reinterpret_cast<float4*>(cpo) = c4[0];
        *reinterpret_cast<float4*>(cpo + 4) = c4[1];
        __half* o = reinterpret_cast<__half*>(dir2 ? a.out2 : a.out) + (((long)md * a.out_kcores + (u0 >> 3)) * 128 + r) * 8;
        *reinterpret_cast<uint4*>(o) = make_uint4(pack_h2(h[0], h[1]), pack_h2(h[2], h[3]), pack_h2(h[4], h[5]), pack_h2(h[6], h[7]));
      }
    }
  } else if (EPI == EPI_LSTM_BWD) {
    // One step of back-propagation through time (training): the GEMM is dG_{t+1} * W_hh (K = 4H gate columns in the
    // interleaved order 4u + gate, TRUE weights; N = H hidden units), so accumulator column u holds the recurrent part
    // of dL/dh_t[u].  With the activations saved by the forward (i,f,g,o fp16 in gx's place, c_t f32):
    //   dh = dy + acc;  do = dh*tanh(c_t);  dc = dc_carry + dh*o*(1 - tanh(c_t)^2);  di = dc*g;  dg = dc*i;  df = dc*c_{t-1};
    //   dc_carry' = dc*f;   dG = [di*i(1-i), df*f(1-f), dg*(1-g^2), do*o(1-o)]   (w.r.t. the true pre-activations)
    // dG is stored as the KB8 tile that is the next (earlier) step's A operand and the operand of the dx / dW GEMMs.
    // [reference: autograd through nn.LSTM, bsrnn_flowse.py:296-297,303-304; d_model.py:74 loss.backward()]
    if (NC == 32) {
      const int u0 = gc0;
      if (u0 < a.H) {
        const bool dir2 = a.dir_tiles > 0 && m >= a.dir_tiles;
        const int md = dir2 ? m - a.dir_tiles : m;
        const long grow = (long)md * 128 + r;
        const bool live = grow < a.valid_rows;
        const __half* sgp = (dir2 ? a.gx2 : a.gx) + grow * a.ld_gx + 4 * u0;
        const __half* dyp = (dir2 ? a.dy2 : a.dy) + grow * a.ld_dy + u0;
        const float* ccp = (dir2 ? a.c_cur2 : a.c_cur) + grow * a.H + u0;
        const float* cpv = dir2 ? a.c_prev2 : a.c_prev;
        const float* cpp = cpv ? cpv + grow * a.H + u0 : nullptr;
        float* dcp = (dir2 ? a.cstate2 : a.cstate) + grow * a.H + u0;
        __half* o = reinterpret_cast<__half*>(dir2 ? a.out2 : a.out) + (((long)md * a.out_kcores + (u0 >> 1)) * 128 + r) * 8;
        // four 8-unit sub-blocks, one after the other: a double-buffered variant (loads of sub-block b+1 under the math
        // of b) needs ~90 more registers and spilled 4.4 KB at the 168-register cap of this 320-thread kernel; the host
        // instead picks narrow N tiles (BN = 64) for small batches so that a warp owns one chunk and many CTAs share the
        // step (training_tc.pack_block)
        BwdSub ra;
#pragma unroll
        for (int b8 = 0; b8 < 4; ++b8) {
          if (u0 + 8 * b8 >= a.H) break;
          uint32_t dgw[16];
          if (live) {
            bwd_load(ra, sgp, dyp, ccp, cpp, dcp, b8);
            bwd_compute(ra, v[8 * b8], v[8 * b8 + 1], v[8 * b8 + 2], v[8 * b8 + 3], v[8 * b8 + 4], v[8 * b8 + 5], v[8 * b8 + 6],
                        v[8 * b8 + 7], dgw);
            *reinterpret_cast<float4*>(dcp + 8 * b8) = ra.dc[0];
            *reinterpret_cast<float4*>(dcp + 8 * b8 + 4) = ra.dc[1];
          } else {
#pragma unroll
            for (int i = 0; i < 16; ++i) dgw[i] = 0u;
          }
#pragma unroll
          for (int i = 0; i < 4; ++i)
            *reinterpret_cast<uint4*>(o + (size_t)(4 * b8 + i) * 1024) = make_uint4(dgw[4 * i], dgw[4 * i + 1], dgw[4 * i + 2], dgw[4 * i + 3]);
        }
      }
    }
  } else if (EPI == EPI_TANH_KB8) {
    __half* o = reinterpret_cast<__half*>(a.out);
#pragma unroll
    for (int i = 0; i < NC; i += 8) {
      const int kc = (gc0 + i) >> 3;
      if (kc >= a.out_kcores) break;
      float t[8];
#pragma unroll
      for (int j = 0; j < 8; ++j) t[j] = (gc0 + i + j < a.n_valid) ? fast_tanh(v[i + j]) : 0.f;
      uint4 pk = make_uint4(pack_h2(t[0], t[1]), pack_h2(t[2], t[3]), pack_h2(t[4], t[5]), pack_h2(t[6], t[7]));
      *reinterpret_cast<uint4*>(o + (((long)m * a.out_kcores + kc) * 128 + r) * 8) = pk;
    }
  } else if (EPI == EPI_TANH_F32) {
    // out[token, gc0 + c] = tanh(v[c]) as f32 rows (GradDecoder Conv1d + Tanh [reference bsrnn_flowse.py:118-134]: the
    // channel-last image the 5x5 conv kernel reads); n_valid % 4 == 0 is checked by the launcher
    if (!row_ok) return;
    float* o = reinterpret_cast<float*>(a.out) + token * a.ldo + gc0;
#pragma unroll
    for (int i = 0; i < NC; i += 4)
      if (gc0 + i + 3 < a.n_valid)
        *reinterpret_cast<float4*>(o + i) = make_float4(fast_tanh(v[i]), fast_tanh(v[i + 1]), fast_tanh(v[i + 2]), fast_tanh(v[i + 3]));
  } else if (EPI == EPI_GLU_F32) {
    if (!row_ok) return;
    // packed weight rows alternate (value, gate): output column = global column / 2
    float* o = reinterpret_cast<float*>(a.out) + token * a.ldo + (gc0 >> 1);
#pragma unroll
    for (int i = 0; i < NC; i += 2)
      if (((gc0 + i) >> 1) < a.n_valid) o[i >> 1] = v[i] * fast_sigmoid(v[i + 1]);
  }
}

// Static tile schedule.  Streaming mode: tile t = blockIdx + it*grid, N tile innermost (CTAs running together share
// the A tile through L2).  Weight-resident mode: CTA i owns N tile i % n_tiles for the whole launch and walks the M
// tiles g, g+G, ... of its group (g = i / n_tiles, G = grid / n_tiles): the weight tile is fetched once, and the
// n_tiles CTAs of a group still consume the same A tile at the same time.
// The schedule above as an iterator without a division per tile: the control warps have ~1 350 cycles of MMA per tile at
// K = 208 and every dependent integer division costs them ~150 (profiles/r01/call32: the MMA warp spent more time
// between tiles than issuing).
struct TileIter {
  int m, n;
  int dm, dn, n_tiles, m_tiles;
  bool resident;
  __device__ __forceinline__ TileIter(const GemmTcArgs& a) {
    n_tiles = a.n_tiles; m_tiles = a.m_tiles; resident = a.b_resident != 0;
    n = (int)blockIdx.x % n_tiles;
    m = (int)blockIdx.x / n_tiles;
    dm = (int)gridDim.x / n_tiles;
    dn = resident ? 0 : (int)gridDim.x - dm * n_tiles;
    if (a.reverse_m && n_tiles == 1 && !resident) {      // last M tile first (see GemmTcArgs::reverse_m)
      rev = true;
      m = m_tiles - 1 - (int)blockIdx.x;
      dm = -(int)gridDim.x;
    } else if (a.m_inner > 1 && !resident && dn == 0) {        // steps innermost (see GemmTcArgs::m_inner); n stays fixed per CTA
      inner = a.m_inner; tps = a.rows.tiles_per_step;
      lin = m;
      m = (lin % inner) * tps + lin / inner;
    }
  }
  bool rev = false;
  int inner = 0, tps = 0, lin = 0;
  __device__ __forceinline__ bool valid() const { return rev ? m >= 0 : (inner ? lin < m_tiles : m < m_tiles); }
  __device__ __forceinline__ void next() {
    if (inner) {
      lin += dm;
      m = (lin % inner) * tps + lin / inner;
      return;
    }
    m += dm; n += dn;
    if (n >= n_tiles) { n -= n_tiles; ++m; }
  }
  __device__ __forceinline__ TileIter ahead(int k) const {       // k small (prefetch distance / next tile)
    TileIter t = *this;
    for (int i = 0; i < k; ++i) t.next();
    return t;
  }
};

// 32 accumulator columns of one row -> 4 consecutive KB8 cores (16 bytes each, 128 rows x 16 B apart)
template <int NCORES>
__device__ __forceinline__ void store_kb8_cores(__half* o, const uint32_t (&v)[32]) {
#pragma unroll
  for (int i = 0; i < NCORES; ++i) {
    const uint4 pk = make_uint4(pack_h2(__uint_as_float(v[8 * i]), __uint_as_float(v[8 * i + 1])),
                                pack_h2(__uint_as_float(v[8 * i + 2]), __uint_as_float(v[8 * i + 3])),
                                pack_h2(__uint_as_float(v[8 * i + 4]), __uint_as_float(v[8 * i + 5])),
                                pack_h2(__uint_as_float(v[8 * i + 6]), __uint_as_float(v[8 * i + 7])));
    *reinterpret_cast<uint4*>(o + (size_t)i * 1024) = pk;
  }
}

template <int NCORES>
__device__ __forceinline__ void store_kb8_cores_smem(uint8_t* p, const uint32_t (&v)[32]) {
#pragma unroll
  for (int i = 0; i < NCORES; ++i) {
    const uint4 pk = make_uint4(pack_h2(__uint_as_float(v[8 * i]), __uint_as_float(v[8 * i + 1])),
                                pack_h2(__uint_as_float(v[8 * i + 2]), __uint_as_float(v[8 * i + 3])),
                                pack_h2(__uint_as_float(v[8 * i + 4]), __uint_as_float(v[8 * i + 5])),
                                pack_h2(__uint_as_float(v[8 * i + 6]), __uint_as_float(v[8 * i + 7])));
    *reinterpret_cast<uint4*>(p + (size_t)i * 2048) = pk;
  }
}
__device__ __forceinline__ void named_bar_sync(int id, int nthreads) {
  asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(nthreads) : "memory");
}

// BNC > 0: BN is the compile-time constant BNC and the launch is the bias-free, weight-resident LSTM input
// projection (EPI_F16_KB8): its epilogue is then straight-line code (profiles/r01/call26: the generic epilogue spent
// ~440 instructions per tile and warp on 70 useful ones and paced the kernel at 2.8x the MMA time).
template <int EPI, int BNC = 0>
__global__ void __launch_bounds__(tc_threads(EPI), 1) gemm_tc_kernel(const __grid_constant__ GemmTcArgs a) {
  extern __shared__ __align__(128) uint8_t smem[];
  const int BN = a.BN;
  constexpr int KS = TC_KS;
  const uint32_t a_stage_bytes = KS * 128 * 16;
  const uint32_t b_stage_bytes = KS * BN * 16;
  uint8_t* sA = smem;
  const uint32_t NST = (uint32_t)a.stages;
  uint8_t* sB = smem + NST * a_stage_bytes;
  const uint32_t b_region = a.b_resident ? (uint32_t)a.kcores * BN * 16 : NST * b_stage_bytes;
  uint64_t* bars = reinterpret_cast<uint64_t*>(sB + b_region);
  uint64_t* full = bars;                     // [TC_STAGES]
  uint64_t* empty = bars + TC_STAGES;        // [TC_STAGES]
  uint64_t* acc_full = bars + 2 * TC_STAGES;     // [2]
  uint64_t* acc_empty = bars + 2 * TC_STAGES + 2;  // [2]
  uint64_t* b_full = bars + 2 * TC_STAGES + 4;
  uint64_t* res_full = bars + 2 * TC_STAGES + 5;   // EPI_RESID_TMA: the tile's residual rows have landed in the row buffer
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 2 * TC_STAGES + 6);
  uint8_t* smem_scr = reinterpret_cast<uint8_t*>(bars + 2 * TC_STAGES + 8);     // 16-byte aligned (residual epilogues only)

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (threadIdx.x == 0) {
    for (int i = 0; i < TC_STAGES; ++i) { mbar_init(full + i, 1); mbar_init(empty + i, 1); }
    for (int i = 0; i < 2; ++i) { mbar_init(acc_full + i, 1); mbar_init(acc_empty + i, BNC ? TC_EPI_WARPS / 2 : tc_epi_warps(EPI)); }
    mbar_init(b_full, 1);
    mbar_init(res_full, 128);
    fence_barrier_init();
  }
  if (warp == 2) tmem_alloc(tmem_slot, 2 * TC_ACC_COLS);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  // Control warps: the whole role runs inside ONE `if (elect_one())` region.  The compiler then knows a single
  // thread executes it and emits back-to-back UTCHMMA / UBLKCP / UTCBAR with descriptors in uniform registers.  Under
  // `if (lane == 0)` it cannot prove that and wraps every such instruction in an elect-and-retry loop with the
  // descriptors rebuilt in vector registers: ~15 dependent instructions = ~250 cycles per MMA issued, 2.4x the
  // 104-cycle MMA itself (profiles/r01/call26: MMA warp 87 % busy issuing, tensor pipe 40 % active).
  if (warp == 0) {
    if (elect_one()) {
      uint32_t stage = 0, phase = 0;
      TileIter ti(a);
      // weight-resident mode: the CTA of the group whose N tile equals (m mod n_tiles) prefetches A tile m
      int pf_mod = 0, pf_dmod = 0;
      if (a.b_resident && a.pf_dist > 0) {
        const TileIter t3 = ti.ahead(a.pf_dist);
        pf_mod = t3.m % a.n_tiles; pf_dmod = ti.dm % a.n_tiles;
      }
      if (a.b_resident && ti.valid()) {
        const uint8_t* gB = reinterpret_cast<const uint8_t*>(a.W) + (size_t)ti.n * a.kcores * BN * 16;
        const uint32_t bytes = (uint32_t)a.kcores * BN * 16;
        mbar_expect_tx(b_full, bytes);
        for (uint32_t off = 0; off < bytes; off += 32768) bulk_g2s(sB + off, gB + off, min(32768u, bytes - off), b_full);
      }
      for (; ti.valid(); ti.next()) {
        const bool dir2 = a.dir_tiles > 0 && ti.m >= a.dir_tiles;
        const int split = a.ksplit > 1 ? ti.m / a.m_log : 0;
        const int mrow = dir2 ? ti.m - a.dir_tiles : (a.ksplit > 1 ? ti.m - split * a.m_log : ti.m);
        const int kbase = split * a.kps;
        int kcnt = a.ksplit > 1 ? min(a.kps, a.kcores - kbase) : a.kcores;
        const uint8_t* gA = reinterpret_cast<const uint8_t*>(dir2 ? a.A2 : a.A) + ((size_t)mrow * a.kcores + kbase) * 2048;
        const uint8_t* gB = reinterpret_cast<const uint8_t*>(dir2 ? a.W2 : a.W) + ((size_t)ti.n * a.kcores + kbase) * BN * 16;
        if (a.groups) {
          const long long* G = a.groups + 5 * (ti.m % a.n_groups);
          kcnt = (int)__ldg(G + 4);
          gA = reinterpret_cast<const uint8_t*>(a.A + __ldg(G)) + (size_t)(ti.m / a.n_groups) * kcnt * 2048;
          gB = reinterpret_cast<const uint8_t*>(a.W + __ldg(G + 1));
        }
        const int nstage_t = (kcnt + KS - 1) / KS;
        if (a.pf_dist > 0) {                       // the A tile pf_dist tiles ahead -> L2 (one bulk prefetch)
          const TileIter t3 = ti.ahead(a.pf_dist);
          if (t3.valid() && (a.b_resident ? ti.n == pf_mod : t3.n == 0))
            bulk_prefetch_l2(reinterpret_cast<const uint8_t*>(a.A) + (size_t)t3.m * a.kcores * 2048, (uint32_t)a.kcores * 2048);
          pf_mod += pf_dmod;
          if (pf_mod >= a.n_tiles) pf_mod -= a.n_tiles;
        }
        for (int ks = 0; ks < nstage_t; ++ks) {
          const int kc0 = ks * KS;
          const int nk = min(KS, kcnt - kc0);
          mbar_wait(empty + stage, phase ^ 1);
          mbar_expect_tx(full + stage, (uint32_t)nk * (2048 + (a.b_resident ? 0 : BN * 16)));
          bulk_g2s(sA + stage * a_stage_bytes, gA + (size_t)kc0 * 2048, nk * 2048, full + stage);
          if (!a.b_resident)
            bulk_g2s(sB + stage * b_stage_bytes, gB + (size_t)kc0 * BN * 16, nk * BN * 16, full + stage);
          if (++stage == NST) { stage = 0; phase ^= 1; }
        }
      }
    }
  } else if (warp == 1) {
    if (elect_one()) {
      const uint32_t idesc = idesc_f16_f32(128, BN);
      TileIter ti(a);
      if (a.b_resident && ti.valid()) mbar_wait(b_full, 0);
      // descriptors advance by adding to the 14-bit (address >> 4) field: shared memory is < 256 KB, no carry out
      const uint64_t da0 = smem_desc_kb8(smem_u32(sA), 2048, 128);
      const uint64_t db0 = smem_desc_kb8(smem_u32(sB), BN * 16, 128);
      const uint32_t a_step = (2 * 2048) >> 4, b_step = (uint32_t)(2 * BN * 16) >> 4;    // one K = 16 step
      {
        uint32_t stage = 0, phase = 0;
        for (int it = 0; ti.valid(); ti.next(), ++it) {
          const int buf = it & 1;
          const uint32_t acc_phase = (it >> 1) & 1;
          mbar_wait(acc_empty + buf, acc_phase ^ 1);
          tc_fence_after();
          const uint32_t d_tmem = tmem_base + buf * TC_ACC_COLS;
          const int kcnt = a.groups ? (int)__ldg(a.groups + 5 * (ti.m % a.n_groups) + 4)
                                    : (a.ksplit > 1 ? min(a.kps, a.kcores - (ti.m / a.m_log) * a.kps) : a.kcores);
          const int nstage_t = (kcnt + KS - 1) / KS;
          for (int ks = 0; ks < nstage_t; ++ks) {
            const int nk = min(KS, kcnt - ks * KS);
            mbar_wait(full + stage, phase);
            tc_fence_after();
            const uint64_t da = da0 + (uint64_t)(stage * (a_stage_bytes >> 4));
            const uint64_t db = db0 + (uint64_t)(a.b_resident ? (uint32_t)ks * (KS / 2) * b_step : stage * (b_stage_bytes >> 4));
            for (int j = 0; j < nk / 2; ++j) mma_f16_ss(d_tmem, da + (uint64_t)(j * a_step), db + (uint64_t)(j * b_step), idesc, (ks | j) != 0);
            mma_commit(empty + stage);
            if (++stage == NST) { stage = 0; phase ^= 1; }
          }
          mma_commit(acc_full + buf);
        }
      }
    }
  } else {
    const int q = warp & 3;                    // TMEM lane quadrant this warp may access
    const int half = (warp - 2) >> 2;          // which half of the tile's column chunks
    const int r = q * 32 + lane;               // row of the tile
    if constexpr ((EPI == EPI_F16_KB8 || EPI == EPI_TANH_KB8) && BNC == 208) {
      // The two 4-warp groups take ALTERNATE tiles (group g <-> TMEM buffer g), each warp the whole 208-column row
      // of its lane quadrant in two passes (cores [0,14) and [14,26) of the tile's 26 KB8 cores).  A pass is
      // converted into the group's shared-memory staging block -- already in the global layout, a pass is ONE
      // contiguous run of 2 KB cores -- and leaves as a single cp.async.bulk shared->global store.
      // Why not st.global: measured (profiles/r01/call37) 1.95 ms without stores, 3.06 ms with st.global.v4 stores that
      // never leave L2, 3.42 ms with DRAM behind them: the LSU store path (8 warps, 512 B per instruction) paced the
      // kernel at ~19 B/clk/SM, not DRAM.  Bulk stores move the same bytes through the TMA unit.
      const int n = blockIdx.x % a.n_tiles;
      const int mstep = gridDim.x / a.n_tiles;
      constexpr uint32_t STG_BYTES = 14 * 2048;                         // staging block of one group (pass A: 14 cores)
      uint8_t* stg = smem_scr + half * STG_BYTES;
      uint8_t* my_stg = stg + r * 16;                                   // this row's 16 bytes of core 0
      uint8_t* gbase = reinterpret_cast<uint8_t*>(a.out) + (size_t)(n * (BNC / 8)) * 2048;
      const size_t o_tile = (a.debug & 1) ? 0 : (size_t)a.out_kcores * 2048;
      const bool do_store = !(a.debug & 2);
      const bool leader = (warp == 2 + 4 * half) && lane == 0;          // issues and tracks the group's bulk stores
      const uint32_t t_row = tmem_base + half * TC_ACC_COLS + ((uint32_t)(q * 32) << 16);
      const int bar_id = 1 + half;                                      // named barrier of the group (128 threads)
      // EPI_TANH_KB8 (MaskDecoder Conv1d(N->4N)+Tanh, bias folded into the weights through the operand's ones column): the
      // last N tile may reach past the destination's out_kcores k-cores -- its two stores are clipped to the cores that exist
      const int cores_left = a.out_kcores - n * (BNC / 8);
      const uint32_t nA = (uint32_t)(cores_left < 14 ? (cores_left < 0 ? 0 : cores_left) : 14);
      // pass B: the input projection's 26th core (columns 200..207 = the 12 pad gate columns of a 49-unit slice) is never read
      // and not stored; the MaskDecoder's hidden tile uses all 208 columns
      constexpr int NB_MAX = EPI == EPI_TANH_KB8 ? 12 : 11;
      const uint32_t nB = (uint32_t)(cores_left - 14 < 0 ? 0 : (cores_left - 14 > NB_MAX ? NB_MAX : cores_left - 14));
      auto act = [](uint32_t (&v)[32], int cnt) {
        if constexpr (EPI == EPI_TANH_KB8) {
#pragma unroll
          for (int i = 0; i < 32; ++i)
            if (i < cnt) v[i] = __float_as_uint(fast_tanh(__uint_as_float(v[i])));
        }
      };
      uint32_t acc_phase = 0;
      for (int m = blockIdx.x / a.n_tiles + half * mstep; m < a.m_tiles; m += 2 * mstep, acc_phase ^= 1) {
        uint32_t v0[32], v1[32], v2[32], v3[32];
        uint8_t* gdst = gbase + (size_t)m * o_tile;
        mbar_wait(acc_full + half, acc_phase);
        tc_fence_after();
        tmem_ld_x32(t_row, v0);
        tmem_ld_x32(t_row + 32, v1);
        tmem_ld_x32(t_row + 64, v2);
        tmem_ld_x16(t_row + 96, reinterpret_cast<uint32_t(&)[16]>(v3));
        tmem_ld_wait();
        tmem_ld_pin(v0); tmem_ld_pin(v1); tmem_ld_pin(v2); tmem_ld_pin(v3);
        act(v0, 32); act(v1, 32); act(v2, 32); act(v3, 16);
        if (leader) bulk_store_wait_read();                             // previous store has finished reading the staging block
        named_bar_sync(bar_id, 128);
        store_kb8_cores_smem<4>(my_stg, v0);
        store_kb8_cores_smem<4>(my_stg + 4 * 2048, v1);
        store_kb8_cores_smem<4>(my_stg + 8 * 2048, v2);
        store_kb8_cores_smem<2>(my_stg + 12 * 2048, v3);
        fence_proxy_async_shared();                                     // generic-proxy smem writes -> the bulk copy's reads
        named_bar_sync(bar_id, 128);
        if (leader && do_store && nA) bulk_s2g(gdst, stg, nA * 2048);
        tmem_ld_x32(t_row + 112, v0);
        tmem_ld_x32(t_row + 144, v1);
        tmem_ld_x32(t_row + 176, v2);
        tmem_ld_wait();
        tmem_ld_pin(v0); tmem_ld_pin(v1); tmem_ld_pin(v2);
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(acc_empty + half);                   // the accumulator sits in registers: back to the MMA warp
        act(v0, 32); act(v1, 32); act(v2, 32);
        if (leader) bulk_store_wait_read();
        named_bar_sync(bar_id, 128);
        store_kb8_cores_smem<4>(my_stg, v0);
        store_kb8_cores_smem<4>(my_stg + 4 * 2048, v1);
        if constexpr (EPI == EPI_TANH_KB8) store_kb8_cores_smem<4>(my_stg + 8 * 2048, v2);
        else store_kb8_cores_smem<3>(my_stg + 8 * 2048, v2);            // core 25 (columns 200..207) is padding nobody reads
        fence_proxy_async_shared();
        named_bar_sync(bar_id, 128);
        if (leader && do_store && nB) bulk_s2g(gdst + 14 * 2048, stg, nB * 2048);
      }
      if (leader) bulk_store_wait_all();
    } else if constexpr (EPI == EPI_RESID_TMA) {
      // Linear + skip with the residual rows moved by the TMA unit: out[token, n*BN + c] += acc (+ bias), c < ncols.
      // The tile's 128 residual row segments (ncols*4 bytes each, contiguous in HBM) arrive in a shared-memory row buffer
      // by one bulk copy per row, are updated there, and leave by one bulk store per row -- instead of 16-byte
      // loads / stores from 12 warps whose bytes in flight bound the register-staged epilogue (profiles/r02 call43/44).
      // Thread r of epilogue warps 2..5 owns row r's copies; a single buffer suffices: load(i+1) is issued as soon as the
      // stores of tile i have been read out of it, and lands while the MMAs of tile i+1 run.
      constexpr int NPART = tc_epi_warps(EPI) / 4;
      const int nch = (BN + 31) >> 5;
      // floor partition of the column chunks: BN = 208 / N = 196 gives the three warps of a quadrant 64 / 64 / 68 valid columns
      // (chunks [0,2) [2,4) [4,7); the 7th chunk holds 4 valid columns).  The ceil partition gave 96 / 64 / 36, and the tile
      // waits for its slowest warp at the named barrier below (23 % of the samples, profiles/r02 call52)
      const int ch0 = (half * nch) / NPART, ch1 = ((half + 1) * nch) / NPART;
      float* resbuf = reinterpret_cast<float*>((reinterpret_cast<uintptr_t>(smem_scr) + 127) & ~(uintptr_t)127);   // TMA box: 128 B
      const int ncmax = a.n_valid < BN ? a.n_valid : BN;
      const int ldr = (ncmax % 8 == 4) ? ncmax : ncmax + 4;          // bank-friendly row stride (floats)
      const bool loader = half == 0;                                   // warps 2..5: one thread per tile row
      float* myrow = resbuf + (size_t)r * ldr;
      // a.run_merge (dense rows: ldo == n_valid == ldr, one N tile): consecutive rows of a warp whose tokens are consecutive
      // form ONE contiguous run in HBM and in the row buffer (time axis: the 34 bands of a frame) and move as one bulk copy --
      // the TMA unit then sees ~8 copies per tile and direction instead of 128 of 784 bytes.  Returns the rows of the run
      // headed by this thread (0 for the other rows).
      auto run_rows = [&](bool ok, long tok) -> uint32_t {
        if (!a.run_merge) return ok ? 1u : 0u;
        const long ptok = __shfl_up_sync(0xffffffffu, tok, 1);
        const bool pok = __shfl_up_sync(0xffffffffu, ok ? 1 : 0, 1) != 0;
        const bool head = ok && (lane == 0 || !pok || tok != ptok + 1);
        const unsigned heads = __ballot_sync(0xffffffffu, head), oks = __ballot_sync(0xffffffffu, ok);
        if (!head) return 0u;
        const unsigned above = lane == 31 ? 0u : ((heads | ~oks) & ~((2u << lane) - 1u));
        return (uint32_t)((above ? __ffs(above) - 1 : 32) - lane);
      };
      auto issue_loads = [&](const TileIter& t) {                      // this thread's row of tile t -> row buffer
        const int m2 = t.m, n2 = t.n;
        long tok2 = 0;
        const int nc2 = (a.n_valid - n2 * BN < BN ? a.n_valid - n2 * BN : BN);
        if (a.use_tmap) {                                              // one tensor copy for the whole tile (thread of row 0)
          if (r == 0 && !a.no_resid) {
            const int step2 = m2 / a.rows.tiles_per_step;
            mbar_expect_tx(res_full, 128u * (uint32_t)nc2 * 4);
            tma_load_2d(resbuf, &a.tmap, step2 * a.tm_col_step + n2 * BN, (m2 - step2 * a.rows.tiles_per_step) * 128, res_full);
          } else {
            mbar_arrive(res_full);
          }
          return;
        }
        const bool ok2 = !a.no_resid && a.rows.map(m2, r, &tok2) && nc2 > 0;
        const uint32_t nr = run_rows(ok2, tok2);
        if (nr) {
          mbar_expect_tx(res_full, nr * (uint32_t)nc2 * 4);
          bulk_g2s(myrow, reinterpret_cast<const float*>(a.out) + tok2 * a.ldo + (long)n2 * BN, nr * (uint32_t)nc2 * 4, res_full);
        } else {
          mbar_arrive(res_full);
        }
      };
      TileIter ti(a);
      if (loader && ti.valid()) issue_loads(ti);
      for (int it = 0; ti.valid(); ti.next(), ++it) {
        const int m = a.groups ? ti.m / a.n_groups : ti.m, n = ti.n;
        const float* g_bias = a.bias;
        float* g_out = reinterpret_cast<float*>(a.out);
        int tm_col = 0;
        if (a.groups) {                                // grouped launch (store only): this tile's band
          const long long* G = a.groups + 5 * (ti.m % a.n_groups);
          tm_col = (int)__ldg(G + 2);
          g_out += tm_col;
          if (g_bias) g_bias += __ldg(G + 3);
        }
        const int buf = it & 1;
        const uint32_t acc_phase = (it >> 1) & 1;
        long token = 0;
        const bool row_ok = a.rows.map(m, r, &token);
        const int ncols = (a.n_valid - n * BN < BN ? a.n_valid - n * BN : BN);
        float s_sum = 0.f, s_sq = 0.f;
        const TileIter tn = ti.ahead(1);
        {                                              // next tile's residual rows -> L2 while this tile is processed
          long tok2 = 0;
          if (!a.no_resid && tn.valid() && a.rows.map(tn.m, r, &tok2)) {
            const char* p = reinterpret_cast<const char*>(reinterpret_cast<const float*>(a.out) + tok2 * a.ldo + (long)tn.n * BN);
            const int nbytes = (a.n_valid - tn.n * BN < BN ? a.n_valid - tn.n * BN : BN) * 4;
            for (int off = half * 128; off < nbytes; off += NPART * 128) asm volatile("prefetch.global.L2 [%0];" ::"l"(p + off));
          }
        }
        float bl[4] = {0.f, 0.f, 0.f, 0.f};
        if (a.bias) {
#pragma unroll
          for (int i = 0; i < 4; ++i) {
            const int c = (ch0 + i) * 32 + lane;
            if (ch0 + i < ch1 && c < BN) bl[i] = __ldg(g_bias + n * BN + c);
          }
        }
        const float osc = a.out_scale_ptr ? __ldg(a.out_scale_ptr) : (a.out_scale != 0.f ? a.out_scale : 1.f);
        mbar_wait(acc_full + buf, acc_phase);
        tc_fence_after();
        mbar_wait(res_full, (uint32_t)(it & 1));
        const uint32_t t_addr = tmem_base + buf * TC_ACC_COLS + ((uint32_t)(q * 32) << 16);
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          const int ch = ch0 + i;
          if (ch >= ch1) break;
          const int c0 = ch * 32;
          uint32_t acc[32];
          const bool wide = c0 + 32 <= BN;
          if (wide) tmem_ld_x32(t_addr + c0, acc);
          else tmem_ld_x16(t_addr + c0, reinterpret_cast<uint32_t(&)[16]>(acc));
          tmem_ld_wait();
          tmem_ld_pin(acc);
          const int nc = wide ? 32 : 16;
#pragma unroll
          for (int j = 0; j < 32; j += 4) {
            if (j >= nc || c0 + j + 3 >= ncols) continue;      // warp-uniform; n_valid % 4 == 0: a 4-group is all valid or all padding
            const float b0 = a.bias ? __shfl_sync(0xffffffffu, bl[i], j) : 0.f, b1 = a.bias ? __shfl_sync(0xffffffffu, bl[i], j + 1) : 0.f;
            const float b2 = a.bias ? __shfl_sync(0xffffffffu, bl[i], j + 2) : 0.f, b3 = a.bias ? __shfl_sync(0xffffffffu, bl[i], j + 3) : 0.f;
            if (row_ok) {
              float4 o = a.no_resid ? make_float4(0.f, 0.f, 0.f, 0.f) : *reinterpret_cast<float4*>(myrow + c0 + j);
              o.x += (__uint_as_float(acc[j]) + b0) * osc; o.y += (__uint_as_float(acc[j + 1]) + b1) * osc;
              o.z += (__uint_as_float(acc[j + 2]) + b2) * osc; o.w += (__uint_as_float(acc[j + 3]) + b3) * osc;
              *reinterpret_cast<float4*>(myrow + c0 + j) = o;
              s_sum += o.x + o.y + o.z + o.w;
              s_sq += o.x * o.x + o.y * o.y + o.z * o.z + o.w * o.w;
            }
          }
        }
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(acc_empty + buf);
        fence_proxy_async_shared();                    // this thread's generic-proxy writes -> the bulk stores' reads
        named_bar_sync(3, tc_epi_warps(EPI) * 32);     // every warp has updated its share of the row buffer
        if (loader) {
          if (a.use_tmap) {
            if (r == 0) {
              const int step = m / a.rows.tiles_per_step;
              tma_store_2d(&a.tmap, tm_col + step * a.tm_col_step + n * BN, (m - step * a.rows.tiles_per_step) * 128, resbuf);
            }
          } else {
          const uint32_t nr = run_rows(row_ok && ncols > 0, token);
          if (nr) bulk_s2g(g_out + token * a.ldo + (long)n * BN, myrow, nr * (uint32_t)ncols * 4);
          }
          bulk_store_wait_read();                      // the store has finished READING the row: the buffer may be refilled
          named_bar_sync(4, 128);                      // ... for all 128 rows
          if (tn.valid()) issue_loads(tn);
        }
        if (a.stats) {
          const long samp = row_ok ? (a.stats_inner > 1 ? (token / a.tokens_per_sample) * a.stats_inner + token % a.stats_inner : token / a.tokens_per_sample) : -1;
          unsigned todo = __ballot_sync(0xffffffffu, row_ok);
          while (todo) {
            const int leader = __ffs(todo) - 1;
            const long ls = __shfl_sync(0xffffffffu, samp, leader);
            const bool mine = row_ok && samp == ls;
            const float ps = warp_sum(mine ? s_sum : 0.f);
            const float pq = warp_sum(mine ? s_sq : 0.f);
            if (lane == leader) {
              atomicAdd(a.stats + 2 * ls, (double)ps);
              atomicAdd(a.stats + 2 * ls + 1, (double)pq);
            }
            todo &= ~__ballot_sync(0xffffffffu, mine);
          }
        }
      }
      if (loader) bulk_store_wait_all();
    } else {
    const int nch = (BN + 31) >> 5;            // 32-column chunks (the last one may be 16 wide)
    constexpr int NPART = tc_epi_warps(EPI) / 4;                 // warps per TMEM lane quadrant: each takes a share of the chunks
    const int ch0 = (half * nch + NPART - 1) / NPART, ch1 = ((half + 1) * nch + NPART - 1) / NPART;
    float* scr = reinterpret_cast<float*>(smem_scr) + (warp - 2) * 32 * TC_SCR_LD;
    TileIter ti(a);
    for (int it = 0; ti.valid(); ti.next(), ++it) {
      const int m = a.ksplit > 1 ? ti.m % a.m_log : ti.m, n = ti.n;
      const int buf = it & 1;
      const uint32_t acc_phase = (it >> 1) & 1;
      long token = 0;
      const bool row_ok = a.rows.map(m, r, &token);
      float s_sum = 0.f, s_sq = 0.f;
      if (EPI == EPI_RESID_F32) {                      // next tile's residual rows -> L2 while this tile is processed
        const TileIter t2 = ti.ahead(1);
        const int m2 = a.ksplit > 1 ? t2.m % a.m_log : t2.m, n2 = t2.n;
        long tok2 = 0;
        if (t2.valid() && a.rows.map(m2, r, &tok2)) {
          const char* p = reinterpret_cast<const char*>(reinterpret_cast<const float*>(a.out) + tok2 * a.ldo + n2 * a.BN);
          const int nbytes = (a.n_valid - n2 * a.BN < a.BN ? a.n_valid - n2 * a.BN : a.BN) * 4;
          for (int off = half * 128; off < nbytes; off += NPART * 128) asm volatile("prefetch.global.L2 [%0];" ::"l"(p + off));
        }
      }
      float bl[4] = {0.f, 0.f, 0.f, 0.f};          // this lane's bias column of each of the warp's (<= 4) chunks
      if (a.bias) {
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          const int c = (ch0 + i) * 32 + lane;
          if (ch0 + i < ch1 && c < BN) bl[i] = __ldg(a.bias + n * BN + c);
        }
      }
      mbar_wait(acc_full + buf, acc_phase);
      tc_fence_after();
      const uint32_t t_addr = tmem_base + buf * TC_ACC_COLS + ((uint32_t)(q * 32) << 16);
      // software pipeline over the warp's (<= 4) chunks: the TMEM load of chunk i+1 is in flight while chunk i is
      // converted and stored (two register buffers; tcgen05.wait::ld covers every load issued before it)
      uint32_t acc0[32], acc1[32];
      auto issue = [&](int ch, uint32_t (&dst)[32]) {
        const int c0 = ch * 32;
        if (c0 + 32 <= BN) tmem_ld_x32(t_addr + c0, dst);
        else tmem_ld_x16(t_addr + c0, reinterpret_cast<uint32_t(&)[16]>(dst));      // BN % 32 == 16
      };
      auto consume = [&](int ch, int i, uint32_t (&src)[32]) {
        const int c0 = ch * 32;
        tmem_ld_pin(src);
        if (c0 + 32 <= BN) epilogue_chunk<EPI, 32>(a, m, n, r, c0, src, row_ok, token, s_sum, s_sq, scr, lane, bl[i]);
        else epilogue_chunk<EPI, 16>(a, m, n, r, c0, src, row_ok, token, s_sum, s_sq, scr, lane, bl[i]);
      };
      if constexpr (EPI == EPI_RESID_F32 && tc_epi_warps(EPI) > 8) {
        // many warps per SM hide the TMEM latency by themselves: one register buffer (32 registers fewer under the
        // lower per-thread cap of a 14-warp CTA)
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          const int ch = ch0 + i;
          if (ch >= ch1) break;
          issue(ch, acc0);
          tmem_ld_wait();
          consume(ch, i, acc0);
        }
      } else {
      if (ch0 < ch1) issue(ch0, acc0);
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const int ch = ch0 + i;
        if (ch >= ch1) break;
        tmem_ld_wait();
        if ((i & 1) == 0) {
          if (ch + 1 < ch1) issue(ch + 1, acc1);
          consume(ch, i, acc0);
        } else {
          if (ch + 1 < ch1) issue(ch + 1, acc0);
          consume(ch, i, acc1);
        }
      }
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(acc_empty + buf);
      if (EPI == EPI_RESID_F32 && a.stats) {
        // rows of a warp are consecutive sequences: usually one sample, sometimes two or three
        const long samp = row_ok ? (a.stats_inner > 1 ? (token / a.tokens_per_sample) * a.stats_inner + token % a.stats_inner : token / a.tokens_per_sample) : -1;
        unsigned todo = __ballot_sync(0xffffffffu, row_ok);
        while (todo) {
          const int leader = __ffs(todo) - 1;
          const long ls = __shfl_sync(0xffffffffu, samp, leader);
          const bool mine = row_ok && samp == ls;
          const float ps = warp_sum(mine ? s_sum : 0.f);
          const float pq = warp_sum(mine ? s_sq : 0.f);
          if (lane == leader) {
            atomicAdd(a.stats + 2 * ls, (double)ps);
            atomicAdd(a.stats + 2 * ls + 1, (double)pq);
          }
          todo &= ~__ballot_sync(0xffffffffu, mine);
        }
      }
    }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 2) {
    tc_fence_after();
    tmem_dealloc(tmem_base, 2 * TC_ACC_COLS);
  }
}

static size_t tc_smem_bytes(int BN, int kcores, bool resident, bool scratch, int stages, size_t extra = 0) {
  const size_t b = resident ? (size_t)kcores * BN * 16 : (size_t)stages * TC_KS * BN * 16;
  return (size_t)stages * TC_KS * 128 * 16 + b + (2 * TC_STAGES + 8) * 8 + (scratch ? TC_SCR_BYTES : 0) + extra;
}
// EPI_RESID_TMA: 128 residual rows of min(BN, n_valid) floats, row stride padded to 4 (mod 8) floats
static size_t tc_resbuf_bytes(int BN, int n_valid) {
  const int nc = n_valid < BN ? n_valid : BN;
  const int ldr = (nc % 8 == 4) ? nc : nc + 4;
  return (size_t)128 * ldr * 4;
}

// Upper bound on the persistent CTAs of the following bsrnn_gemm_tc* launches (0 = every SM): with a few CTAs every CTA
// walks many tiles of the same launch.
static int g_cta_limit = 0;

// One launch shape per call: a plain launch of gemm_tc_kernel<EPI> (streaming or weight-resident schedule, chosen below), or
// of the specialised straight-line kernel gemm_tc_kernel<EPI, 208> for the input projection (EPI_F16_KB8) and the
// MaskDecoder's Conv1d+Tanh (EPI_TANH_KB8) at BN = 208, K = 208, bias folded into the weights.
template <int EPI>
static int launch_tc(GemmTcArgs a, cudaStream_t st) {
  static int sms = 0;                     // one process per GPU: the SM count is queried once
  if (sms == 0) {
    int dev = 0;
    cudaGetDevice(&dev);
    if (cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || sms <= 0) sms = 148;
  }
  // weight-resident schedule when several N tiles exist, the tile fits beside the A ring, and there is enough M work
  // (the LSTM step kernels run both directions in one launch: dir_tiles > 0 keeps them streaming; measured resident
  // with A-tile multicast: 52 vs 34 us per step at H = 768, profiles/r02 call13)
  a.b_resident = (a.n_tiles > 1 && a.n_tiles <= sms && (size_t)a.kcores * a.BN * 16 <= 120 * 1024 &&
                  a.m_tiles >= 2 * (sms / a.n_tiles) && a.ksplit <= 1 && a.dir_tiles == 0) ? 1 : 0;
  if (EPI == EPI_GLU_F32) a.reverse_m = 1;
  const size_t extra_smem = EPI == EPI_RESID_TMA ? tc_resbuf_bytes(a.BN, a.n_valid) + 128 : 0;
  if (EPI == EPI_RESID_TMA) {
    // matrix view of the output for the tensor-map path: address = seq * row_stride + step * col_step (+ group offset)
    long row_stride = 0, col_step = 0;
    if (a.rows.seq_inner == 1) { row_stride = a.rows.seq_outer * a.ldo; col_step = a.rows.step_stride * a.ldo; }
    else if (a.rows.seq_inner >= (long)a.rows.R) { row_stride = a.rows.seq_inner_stride * a.ldo; col_step = a.rows.step_stride * a.ldo; }
    const long steps = (a.groups ? a.m_tiles / a.n_groups : a.m_tiles) / a.rows.tiles_per_step;
    a.use_tmap = 0;
    if (a.n_tiles == 1 && a.n_valid <= a.BN && a.n_valid % 8 == 4 && row_stride > 0 && a.ksplit <= 1 &&
        a.out_scale == 0.f && a.out_scale_ptr == nullptr && (steps - 1) * col_step + a.n_valid <= row_stride &&
        (!a.groups || col_step == 0) && col_step < (1L << 30) &&
        make_tmap_2d_f32(&a.tmap, a.out, (uint64_t)row_stride, (uint64_t)a.rows.R, (uint64_t)row_stride * 4, (uint32_t)a.n_valid, 128)) {
      a.use_tmap = 1;
      a.tm_col_step = (int)col_step;
      if (!a.groups && steps > 1 && col_step > 0 && a.m_tiles == steps * a.rows.tiles_per_step) a.m_inner = (int)steps;
    }
  }
  // (the same band-innermost walk without a tensor map -- FlowSE, N = 384 = two N tiles of 192, one bulk copy per row -- measures
  // no difference: 5.75 vs 5.73 s on config 4, profiles/r02 call72; it stays step-major there)
  if (EPI == EPI_RESID_TMA && !a.use_tmap)
    a.run_merge = (a.n_tiles == 1 && a.n_valid <= a.BN && a.ldo == a.n_valid && a.n_valid % 8 == 4) ? 1 : 0;
  // Streaming GEMMs whose ring only fits 4 stages of 8 k-cores (Linear 4N->N: the 333 KB weight tile rides beside every
  // 205 KB activation tile) keep 4: 8 stages of 4 k-cores measured no gain (profiles/r02 call41: Linear+skip 25.6 vs 25.5 ms
  // per step at config 2, FlowSE 38.0 vs 38.0 ms per evaluation).
  a.stages = tc_smem_bytes(a.BN, a.kcores, a.b_resident, EPI == EPI_RESID_F32, 8, extra_smem) <= 227 * 1024 ? 8 : 4;
  while (a.stages > 2 && tc_smem_bytes(a.BN, a.kcores, a.b_resident, EPI == EPI_RESID_F32, a.stages, extra_smem) > 227 * 1024) --a.stages;
  // L2 prefetch distance of the A tiles.  Streaming mode has one prefetcher per CTA: at K = 800 (Linear 4N->N, A tile
  // 205 KB) three tiles ahead on 148 CTAs is 91 MB of prefetched lines in a 126 MB L2 that also carries the residual
  // stream -- they were evicted before use and fetched twice (ncu: 9.3 GB read for 5.2 GB algorithmic,
  // profiles/r01/call21_ncu_full_gemm_fc_raw.csv).  Keep the prefetched set under ~32 MB.
  // Measured (profiles/r01/call24_gemm_fc.log, Linear 4N->N at BASELINE config 2): distance 3 / 1 / 0 = 2.09 / 2.01 /
  // 1.60 ms -- with an 8-stage ring the bulk copies already run a full tile ahead, and the extra L2 prefetch only
  // competes with the residual stream.  Streaming mode: off.  Weight-resident mode (short K): 3 tiles ahead.
  a.pf_dist = a.b_resident ? 3 : 0;
  static int dbg = -1;
  if (dbg < 0) { const char* e = getenv("BSRNN_GEMM_DEBUG"); dbg = (e && e[0] >= '0' && e[0] <= '9') ? atoi(e) : 0; }
  a.debug = dbg;
  const int total = a.m_tiles * a.n_tiles;
  const int sms_use = (g_cta_limit > 0 && g_cta_limit < sms) ? g_cta_limit : sms;
  int grid = total < sms_use ? total : sms_use;
  if (a.b_resident) {
    grid = (sms_use / a.n_tiles) * a.n_tiles;
    if (grid < a.n_tiles) grid = a.n_tiles;
  }
  if constexpr (EPI == EPI_F16_KB8 || EPI == EPI_TANH_KB8) {
    // Specialised kernel: 5 ring stages + two 28 KB staging blocks for the bulk stores.  Conv1d(N->4N)+Tanh runs on it too
    // (straight-line epilogue, tile staged in shared memory in the destination layout): the st.global path of the generic
    // epilogue paced it.  (A-tile multicast over clusters of N-tile CTAs measured 42.1 / 43.3 / 45.6 ms per step for
    // 1 / 2 / 4, profiles/r02 call11: the L2->SM re-reads are not what bounds this GEMM.)
    const bool fits = EPI == EPI_F16_KB8 ? a.out_kcores >= a.n_tiles * 26 : a.out_kcores > (a.n_tiles - 1) * 26;
    if (a.BN == 208 && a.kcores == 26 && a.bias == nullptr && a.b_resident && fits) {
      a.stages = 5;
      const size_t smem_ip = tc_smem_bytes(a.BN, a.kcores, true, false, a.stages) + 2 * 14 * 2048;
      BSRNN_CUDA_OK(cudaFuncSetAttribute(gemm_tc_kernel<EPI, 208>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_ip));
      gemm_tc_kernel<EPI, 208><<<grid, tc_threads(EPI), smem_ip, st>>>(a);
      BSRNN_LAUNCH_OK();
      return 0;
    }
  }
  const size_t smem = tc_smem_bytes(a.BN, a.kcores, a.b_resident, EPI == EPI_RESID_F32, a.stages, extra_smem);
  static size_t smem_set = 0;             // per instantiation: the attribute only ever needs to grow (step-wise launches
  if (smem > smem_set) {                  // call this thousands of times per training step)
    BSRNN_CUDA_OK(cudaFuncSetAttribute(gemm_tc_kernel<EPI>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    smem_set = smem;
  }
  gemm_tc_kernel<EPI><<<grid, tc_threads(EPI), smem, st>>>(a);
  BSRNN_LAUNCH_OK();
  return 0;
}

}  // namespace bsrnn
using namespace bsrnn;

// bsrnn_gemm_tc with two extras of the f32-row epilogues 1 / 8: stats_inner (> 1: statistics per (sample, token %
// stats_inner) instead of per sample) and flags (bit 0, epilogue 8 only: store only -- out = A W^T + bias, no residual read).
extern "C" int bsrnn_gemm_tc_ex(const void* A, const void* W, const float* bias, void* out, double* stats,
                                  int m_tiles, int n_tiles, int kcores, int BN, int epilogue, long ldo, int n_valid,
                                  int out_kcores, long tokens_per_sample, int tiles_per_step, int R, long seq_inner,
                                  long seq_outer, long seq_inner_stride, long step_stride, int stats_inner, int flags,
                                  void* stream) {
  BSRNN_CHECK_ARG(A && W && out, "gemm_tc: null pointer");
  BSRNN_CHECK_ARG(m_tiles > 0 && n_tiles > 0 && kcores > 0 && kcores % 2 == 0, "gemm_tc: bad tile counts (kcores=%d)", kcores);
  BSRNN_CHECK_ARG(BN >= 16 && BN <= 256 && BN % 16 == 0, "gemm_tc: BN=%d must be a multiple of 16 in [16,256]", BN);
  BSRNN_CHECK_ARG(tiles_per_step > 0 && seq_inner > 0 && tokens_per_sample > 0, "gemm_tc: bad row map");
  BSRNN_CHECK_ARG((epilogue != EPI_RESID_F32 && epilogue != EPI_TANH_F32 && epilogue != EPI_RESID_TMA) || (n_valid % 4 == 0 && ldo % 4 == 0),
                  "gemm_tc: the f32-row epilogues need n_valid and ldo to be multiples of 4 (got %d, %ld)", n_valid, ldo);
  // the epilogues that do not clip at n_valid / out_kcores store every column of every N tile: reject a launch whose last tile
  // would run into the next row (fp16 rows) or the next row tile (KB8), and row epilogues whose rows overlap
  BSRNN_CHECK_ARG(epilogue != EPI_F16_ROWS || (long)n_tiles * BN <= ldo,
                  "gemm_tc: epilogue 0 stores n_tiles*BN = %d columns per row, more than ldo = %ld", n_tiles * BN, ldo);
  BSRNN_CHECK_ARG(epilogue != EPI_F16_KB8 || n_tiles * BN <= 8 * out_kcores,
                  "gemm_tc: epilogue 4 stores n_tiles*BN = %d columns, more than 8*out_kcores = %d", n_tiles * BN, 8 * out_kcores);
  BSRNN_CHECK_ARG((epilogue != EPI_RESID_F32 && epilogue != EPI_TANH_F32 && epilogue != EPI_RESID_TMA && epilogue != EPI_GLU_F32) ||
                  (n_valid > 0 && ldo >= n_valid),
                  "gemm_tc: the row epilogues need 0 < n_valid <= ldo (got %d, %ld)", n_valid, ldo);
  GemmTcArgs a{};
  a.A = reinterpret_cast<const __half*>(A);
  a.W = reinterpret_cast<const __half*>(W);
  a.bias = bias; a.out = out; a.stats = stats; a.ldo = ldo; a.tokens_per_sample = tokens_per_sample;
  a.m_tiles = m_tiles; a.n_tiles = n_tiles; a.kcores = kcores; a.BN = BN; a.n_valid = n_valid; a.out_kcores = out_kcores;
  a.rows = RowMap{tiles_per_step, R, seq_inner, seq_outer, seq_inner_stride, step_stride};
  BSRNN_CHECK_ARG(stats_inner >= 1 && (flags & ~1) == 0 && (!(flags & 1) || epilogue == EPI_RESID_TMA),
                  "gemm_tc: bad stats_inner / flags (store-only needs epilogue 8)");
  a.stats_inner = stats_inner;
  a.no_resid = flags & 1;
  cudaStream_t st = (cudaStream_t)stream;
  switch (epilogue) {
    case EPI_F16_ROWS: return launch_tc<EPI_F16_ROWS>(a, st);
    case EPI_RESID_F32: return launch_tc<EPI_RESID_F32>(a, st);
    case EPI_TANH_KB8: return launch_tc<EPI_TANH_KB8>(a, st);
    case EPI_GLU_F32: return launch_tc<EPI_GLU_F32>(a, st);
    case EPI_F16_KB8: return launch_tc<EPI_F16_KB8>(a, st);
    case EPI_TANH_F32: return launch_tc<EPI_TANH_F32>(a, st);
    case EPI_RESID_TMA:
      BSRNN_CHECK_ARG(BN % 4 == 0 && (reinterpret_cast<uintptr_t>(out) & 15) == 0, "gemm_tc: the TMA residual epilogue needs 16-byte aligned rows");
      return launch_tc<EPI_RESID_TMA>(a, st);
  }
  set_error("gemm_tc: unknown epilogue %d", epilogue);
  return 1;
}
extern "C" int bsrnn_gemm_tc_limit_ctas(int n) {
  const int prev = g_cta_limit;
  g_cta_limit = n > 0 ? n : 0;
  return prev;
}

// Grouped store-only GEMM (tensor-core BandSplit): out[token*ldo + out_off_g + c] = A_g W_g^T + bias_g for n_groups bands in
// ONE launch, bands innermost in the tile order.  groups: device [n_groups][5] int64 {a_off, w_off, out_off, bias_off,
// kcores} relative to A / W / out / bias; kc_max = largest kcores (sizes the pipeline); m_tiles = row tiles per group.
extern "C" int bsrnn_gemm_tc_grouped(const void* A, const void* W, const float* bias, void* out, double* stats,
                                       const long long* groups, int n_groups, int m_tiles, int kc_max, int BN, long ldo,
                                       int n_valid, long tokens_per_sample, int tiles_per_step, int R, long seq_inner,
                                       long seq_outer, long seq_inner_stride, long step_stride, void* stream) {
  BSRNN_CHECK_ARG(A && W && out && groups && n_groups > 0, "gemm_tc_grouped: null pointer");
  BSRNN_CHECK_ARG(m_tiles > 0 && kc_max > 0 && kc_max % 2 == 0 && BN >= 16 && BN <= 256 && BN % 16 == 0, "gemm_tc_grouped: bad tile dims");
  BSRNN_CHECK_ARG(n_valid > 0 && n_valid <= BN && n_valid % 4 == 0 && ldo % 4 == 0 && (reinterpret_cast<uintptr_t>(out) & 15) == 0,
                  "gemm_tc_grouped: rows must be 16-byte aligned, n_valid <= BN");
  BSRNN_CHECK_ARG(tiles_per_step > 0 && seq_inner > 0 && tokens_per_sample > 0, "gemm_tc_grouped: bad row map");
  GemmTcArgs a{};
  a.A = reinterpret_cast<const __half*>(A);
  a.W = reinterpret_cast<const __half*>(W);
  a.bias = bias; a.out = out; a.stats = stats; a.ldo = ldo; a.tokens_per_sample = tokens_per_sample;
  a.m_tiles = m_tiles * n_groups; a.n_tiles = 1; a.kcores = kc_max; a.BN = BN; a.n_valid = n_valid;
  a.rows = RowMap{tiles_per_step, R, seq_inner, seq_outer, seq_inner_stride, step_stride};
  a.stats_inner = 1; a.no_resid = 1; a.groups = groups; a.n_groups = n_groups;
  return launch_tc<EPI_RESID_TMA>(a, (cudaStream_t)stream);
}

extern "C" int bsrnn_gemm_tc(const void* A, const void* W, const float* bias, void* out, double* stats,
                               int m_tiles, int n_tiles, int kcores, int BN, int epilogue, long ldo, int n_valid,
                               int out_kcores, long tokens_per_sample, int tiles_per_step, int R, long seq_inner,
                               long seq_outer, long seq_inner_stride, long step_stride, void* stream) {
  return bsrnn_gemm_tc_ex(A, W, bias, out, stats, m_tiles, n_tiles, kcores, BN, epilogue, ldo, n_valid, out_kcores,
                          tokens_per_sample, tiles_per_step, R, seq_inner, seq_outer, seq_inner_stride, step_stride, 1, 0, stream);
}

// One time step of an LSTM direction on tensor cores, any H % 8 == 0 (csrc/gemm_tc.cu, EPI_LSTM_STEP):
//   A      [m_tiles][kc][128][8] fp16  h_{t-1} tiles (a zero tile set for the first step); kc = 2*ceil(H/16): K is padded
//                                       to a multiple of 16 and the pad k-core of the tiles must stay zero
//   W      [n_tiles][kc][BN][8]  fp16  W_hh with rows reordered to 4u + gate and i/f/o rows pre-halved; BN % 32 == 0
//   gx     rows [m*128 + r][ld_gx] fp16: input projection (+ bias) of THIS step and direction, same column order
//   cstate [m_tiles*128][H] f32, updated in place;   out_h: h_t tiles, same layout as A
extern "C" int bsrnn_lstm_step_tc(const void* A, const void* W, const void* gx, float* cstate, void* out_h, int m_tiles,
                                  int n_tiles, int BN, int H, long ld_gx, void* stream) {
  BSRNN_CHECK_ARG(A && W && gx && cstate && out_h, "lstm_step_tc: null pointer");
  BSRNN_CHECK_ARG(m_tiles > 0 && n_tiles > 0 && H > 0 && H % 8 == 0 && BN % 32 == 0 && BN >= 32 && BN <= 256 &&
                  (long)n_tiles * BN >= 4L * H && ld_gx >= 4L * H && ld_gx % 8 == 0, "lstm_step_tc: bad dims");
  GemmTcArgs a{};
  a.A = reinterpret_cast<const __half*>(A);
  a.W = reinterpret_cast<const __half*>(W);
  a.bias = nullptr; a.out = out_h; a.stats = nullptr; a.ldo = 0; a.tokens_per_sample = 1;
  a.m_tiles = m_tiles; a.n_tiles = n_tiles; a.kcores = (H + 15) / 16 * 2; a.BN = BN; a.n_valid = 4 * H; a.out_kcores = (H + 15) / 16 * 2;
  a.gx = reinterpret_cast<const __half*>(gx); a.cstate = cstate; a.ld_gx = ld_gx; a.H = H;
  a.rows = RowMap{m_tiles, m_tiles * 128, 1L << 40, 0, 1, 0};
  return launch_tc<EPI_LSTM_STEP>(a, (cudaStream_t)stream);
}

// Both directions of one BLSTM time step in ONE launch (the two chains are independent, so their launch / prologue /
// first-load latencies overlap): the *_f pointers serve row tiles [0, m_tiles), the *_b pointers row tiles
// [m_tiles, 2*m_tiles).  Arguments as bsrnn_lstm_step_tc.
extern "C" int bsrnn_blstm_step_tc(const void* A_f, const void* W_f, const void* gx_f, float* c_f, void* out_f,
                                   const void* A_b, const void* W_b, const void* gx_b, float* c_b, void* out_b, int m_tiles,
                                   int n_tiles, int BN, int H, long ld_gx, void* stream) {
  BSRNN_CHECK_ARG(A_f && W_f && gx_f && c_f && out_f && A_b && W_b && gx_b && c_b && out_b, "blstm_step_tc: null pointer");
  BSRNN_CHECK_ARG(m_tiles > 0 && n_tiles > 0 && H > 0 && H % 8 == 0 && BN % 32 == 0 && BN >= 32 && BN <= 256 &&
                  (long)n_tiles * BN >= 4L * H && ld_gx >= 4L * H && ld_gx % 8 == 0, "blstm_step_tc: bad dims");
  GemmTcArgs a{};
  a.A = reinterpret_cast<const __half*>(A_f); a.W = reinterpret_cast<const __half*>(W_f);
  a.A2 = reinterpret_cast<const __half*>(A_b); a.W2 = reinterpret_cast<const __half*>(W_b);
  a.bias = nullptr; a.out = out_f; a.out2 = out_b; a.stats = nullptr; a.ldo = 0; a.tokens_per_sample = 1;
  a.m_tiles = 2 * m_tiles; a.dir_tiles = m_tiles; a.n_tiles = n_tiles; a.kcores = (H + 15) / 16 * 2; a.BN = BN; a.n_valid = 4 * H;
  a.out_kcores = (H + 15) / 16 * 2;
  a.gx = reinterpret_cast<const __half*>(gx_f); a.gx2 = reinterpret_cast<const __half*>(gx_b);
  a.cstate = c_f; a.cstate2 = c_b; a.ld_gx = ld_gx; a.H = H;
  a.rows = RowMap{2 * m_tiles, 2 * m_tiles * 128, 1L << 40, 0, 1, 0};
  return launch_tc<EPI_LSTM_STEP>(a, (cudaStream_t)stream);
}

// ---------------------------------------------------------------------------------------------- training entry points
// bsrnn_gemm_tc with an output scale (EPI_RESID_F32: out += scale * A W^T): the fp16 gradient operands of the training
// backward carry a power-of-two loss scale that is removed here, in f32.
extern "C" int bsrnn_gemm_tc_scaled(const void* A, const void* W, const float* bias, void* out, int m_tiles, int n_tiles,
                                    int kcores, int BN, long ldo, int n_valid, float out_scale, const float* out_scale_ptr,
                                    int ksplit, int tiles_per_step, int R, long seq_inner, long seq_outer,
                                    long seq_inner_stride, long step_stride, void* stream) {
  BSRNN_CHECK_ARG(A && W && out, "gemm_tc_scaled: null pointer");
  BSRNN_CHECK_ARG(m_tiles > 0 && n_tiles > 0 && kcores > 0 && kcores % 2 == 0, "gemm_tc_scaled: bad tile counts (kcores=%d)", kcores);
  BSRNN_CHECK_ARG(BN >= 16 && BN <= 256 && BN % 16 == 0, "gemm_tc_scaled: BN=%d must be a multiple of 16 in [16,256]", BN);
  BSRNN_CHECK_ARG(tiles_per_step > 0 && seq_inner > 0 && n_valid % 4 == 0 && ldo % 4 == 0, "gemm_tc_scaled: bad row map / strides");
  BSRNN_CHECK_ARG(n_valid > 0 && ldo >= n_valid, "gemm_tc_scaled: need 0 < n_valid <= ldo (got %d, %ld)", n_valid, ldo);
  GemmTcArgs a{};
  a.A = reinterpret_cast<const __half*>(A);
  a.W = reinterpret_cast<const __half*>(W);
  a.bias = bias; a.out = out; a.stats = nullptr; a.ldo = ldo; a.tokens_per_sample = 1;
  a.m_tiles = m_tiles; a.n_tiles = n_tiles; a.kcores = kcores; a.BN = BN; a.n_valid = n_valid; a.out_kcores = 0;
  a.out_scale = out_scale; a.out_scale_ptr = out_scale_ptr;
  a.ksplit = 1; a.kps = kcores; a.m_log = m_tiles;
  if (ksplit > 1) {                                   // K split over CTAs, partial sums meet through atomic adds
    BSRNN_CHECK_ARG(bias == nullptr, "gemm_tc_scaled: split-K has no bias epilogue");
    const int kps = ((kcores + ksplit - 1) / ksplit + TC_KS - 1) / TC_KS * TC_KS;
    a.kps = kps;
    a.ksplit = (kcores + kps - 1) / kps;
    a.m_tiles = m_tiles * a.ksplit;
  }
  a.rows = RowMap{tiles_per_step, R, seq_inner, seq_outer, seq_inner_stride, step_stride};
  return launch_tc<EPI_RESID_F32>(a, (cudaStream_t)stream);
}

// Both directions of one BLSTM time step, TRAINING forward: as bsrnn_blstm_step_tc, but c_{t-1} is read from cprev_*
// (null = zeros: first step of the sequence), c_t is written to cout_*, and the activated gates (i, f, g, o; fp16) replace
// the input projection in gx_* -- the quantities bsrnn_blstm_bwd_step_tc consumes.
extern "C" int bsrnn_blstm_step_train_tc(const void* A_f, const void* W_f, void* gx_f, const float* cprev_f, float* cout_f,
                                         void* out_f, const void* A_b, const void* W_b, void* gx_b, const float* cprev_b,
                                         float* cout_b, void* out_b, int m_tiles, int n_tiles, int BN, int H, long ld_gx,
                                         void* stream) {
  BSRNN_CHECK_ARG(A_f && W_f && gx_f && cout_f && out_f && A_b && W_b && gx_b && cout_b && out_b, "blstm_step_train_tc: null pointer");
  BSRNN_CHECK_ARG(m_tiles > 0 && n_tiles > 0 && H > 0 && H % 8 == 0 && BN % 32 == 0 && BN >= 32 && BN <= 256 &&
                  (long)n_tiles * BN >= 4L * H && ld_gx >= 4L * H && ld_gx % 8 == 0, "blstm_step_train_tc: bad dims");
  GemmTcArgs a{};
  a.A = reinterpret_cast<const __half*>(A_f); a.W = reinterpret_cast<const __half*>(W_f);
  a.A2 = reinterpret_cast<const __half*>(A_b); a.W2 = reinterpret_cast<const __half*>(W_b);
  a.bias = nullptr; a.out = out_f; a.out2 = out_b; a.stats = nullptr; a.ldo = 0; a.tokens_per_sample = 1;
  a.m_tiles = 2 * m_tiles; a.dir_tiles = m_tiles; a.n_tiles = n_tiles; a.kcores = (H + 15) / 16 * 2; a.BN = BN; a.n_valid = 4 * H;
  a.out_kcores = (H + 15) / 16 * 2;
  a.gx = reinterpret_cast<const __half*>(gx_f); a.gx2 = reinterpret_cast<const __half*>(gx_b);
  a.cstate = const_cast<float*>(cprev_f); a.cstate2 = const_cast<float*>(cprev_b);
  a.cstate_out = cout_f; a.cstate_out2 = cout_b; a.save_gates = 1;
  a.ld_gx = ld_gx; a.H = H;
  a.rows = RowMap{2 * m_tiles, 2 * m_tiles * 128, 1L << 40, 0, 1, 0};
  return launch_tc<EPI_LSTM_STEP>(a, (cudaStream_t)stream);
}

// Both directions of one BPTT step (EPI_LSTM_BWD above).  Per direction:
//   A     [m_tiles][4H/8][128][8] fp16  dG of the step processed just before (a zero tile set for the first one)
//   W     [n_tiles][4H/8][BN][8]  fp16  W_hh^T: row = hidden unit u, K = gate column 4u' + gate (true weights); BN % 32 == 0
//   sg    rows [m*128 + r][ld_sg] fp16  activated gates of THIS step (written by bsrnn_blstm_step_train_tc)
//   dy    rows [m*128 + r][ld_dy] fp16  dL/dh_t from the layers above (loss-scaled)
//   ccur / cprev  rows [m*128 + r][H] f32  c_t / c_{t-1} (cprev null = zeros)
//   dc    [m_tiles*128][H] f32 carry, updated in place (zero before the first step)
//   out   dG tiles of THIS step, layout as A.     Rows >= valid_rows get zero gradients.
extern "C" int bsrnn_blstm_bwd_step_tc(const void* A_f, const void* W_f, const void* sg_f, const void* dy_f, const float* ccur_f,
                                       const float* cprev_f, float* dc_f, void* out_f, const void* A_b, const void* W_b,
                                       const void* sg_b, const void* dy_b, const float* ccur_b, const float* cprev_b, float* dc_b,
                                       void* out_b, int m_tiles, int n_tiles, int BN, int H, long ld_sg, long ld_dy,
                                       int valid_rows, void* stream) {
  BSRNN_CHECK_ARG(A_f && W_f && sg_f && dy_f && ccur_f && dc_f && out_f && A_b && W_b && sg_b && dy_b && ccur_b && dc_b && out_b,
                  "blstm_bwd_step_tc: null pointer");
  BSRNN_CHECK_ARG(m_tiles > 0 && n_tiles > 0 && H > 0 && H % 8 == 0 && (4 * H / 8) % 2 == 0 && BN % 32 == 0 && BN >= 32 && BN <= 256 &&
                  (long)n_tiles * BN >= H && ld_sg >= 4L * H && ld_sg % 8 == 0 && ld_dy >= H && ld_dy % 8 == 0 && valid_rows > 0,
                  "blstm_bwd_step_tc: bad dims");
  GemmTcArgs a{};
  a.A = reinterpret_cast<const __half*>(A_f); a.W = reinterpret_cast<const __half*>(W_f);
  a.A2 = reinterpret_cast<const __half*>(A_b); a.W2 = reinterpret_cast<const __half*>(W_b);
  a.bias = nullptr; a.out = out_f; a.out2 = out_b; a.stats = nullptr; a.ldo = 0; a.tokens_per_sample = 1;
  a.m_tiles = 2 * m_tiles; a.dir_tiles = m_tiles; a.n_tiles = n_tiles; a.kcores = 4 * H / 8; a.BN = BN; a.n_valid = H;
  a.out_kcores = 4 * H / 8;
  a.gx = reinterpret_cast<const __half*>(sg_f); a.gx2 = reinterpret_cast<const __half*>(sg_b); a.ld_gx = ld_sg;
  a.dy = reinterpret_cast<const __half*>(dy_f); a.dy2 = reinterpret_cast<const __half*>(dy_b); a.ld_dy = ld_dy;
  a.c_cur = ccur_f; a.c_cur2 = ccur_b; a.c_prev = cprev_f; a.c_prev2 = cprev_b;
  a.cstate = dc_f; a.cstate2 = dc_b; a.H = H; a.valid_rows = valid_rows;
  a.rows = RowMap{2 * m_tiles, 2 * m_tiles * 128, 1L << 40, 0, 1, 0};
  return launch_tc<EPI_LSTM_BWD>(a, (cudaStream_t)stream);
}

// Whole-sequence drivers of the two step kernels above: the host loop over time steps lives here (a launch every few
// microseconds) instead of in the Python caller (tens of microseconds per ctypes call x thousands of steps).
//   y_*   [steps*tiles][kc][128][8] fp16 h tiles (kc = 2*ceil(H/16); zero-initialised by the caller: the pad core stays 0)
//   gates rows [(step*tiles*128 + r)][8H] fp16: input projection on entry, ACTIVATED gates on return (direction-major)
//   c_*   [steps][tiles*128][H] f32
// Direction f walks positions 0..steps-1, direction b walks steps-1..0; position p of either lives at step index p.
extern "C" int bsrnn_blstm_train_fwd_tc(const void* zero_tile, void* y_f, void* y_b, const void* W_f, const void* W_b,
                                        void* gates, float* c_f, float* c_b, int steps, int tiles, int n_tiles, int BN, int H,
                                        void* stream) {
  BSRNN_CHECK_ARG(zero_tile && y_f && y_b && W_f && W_b && gates && c_f && c_b && steps > 0 && tiles > 0,
                  "blstm_train_fwd_tc: bad arguments");
  const size_t kc = (size_t)((H + 15) / 16 * 2);
  const size_t y_step = (size_t)tiles * kc * 1024;            // halves
  const size_t g_step = (size_t)tiles * 128 * 8 * H;          // halves
  const size_t c_step = (size_t)tiles * 128 * H;              // floats
  __half* yf = reinterpret_cast<__half*>(y_f);
  __half* yb = reinterpret_cast<__half*>(y_b);
  __half* g = reinterpret_cast<__half*>(gates);
  for (int s = 0; s < steps; ++s) {
    const int pf = s, pb = steps - 1 - s;
    const int rc = bsrnn_blstm_step_train_tc(
        s == 0 ? zero_tile : (const void*)(yf + (size_t)(pf - 1) * y_step), W_f, g + (size_t)pf * g_step,
        s == 0 ? nullptr : c_f + (size_t)(pf - 1) * c_step, c_f + (size_t)pf * c_step, yf + (size_t)pf * y_step,
        s == 0 ? zero_tile : (const void*)(yb + (size_t)(pb + 1) * y_step), W_b, g + (size_t)pb * g_step + 4 * (size_t)H,
        s == 0 ? nullptr : c_b + (size_t)(pb + 1) * c_step, c_b + (size_t)pb * c_step, yb + (size_t)pb * y_step, tiles, n_tiles,
        BN, H, 8L * H, stream);
    if (rc) return rc;
  }
  return 0;
}

//   dG_*  [steps*tiles][4H/8][128][8] fp16 (output);  dy rows [(step*tiles*128 + r)][2H] fp16;  dc_* [tiles*128][H] f32 zeroed
extern "C" int bsrnn_blstm_train_bwd_tc(const void* zero_tile, void* dG_f, void* dG_b, const void* WT_f, const void* WT_b,
                                        const void* gates, const void* dy, const float* c_f, const float* c_b, float* dc_f,
                                        float* dc_b, int steps, int tiles, int n_tiles, int BN, int H, int valid_rows,
                                        void* stream) {
  BSRNN_CHECK_ARG(zero_tile && dG_f && dG_b && WT_f && WT_b && gates && dy && c_f && c_b && dc_f && dc_b && steps > 0 && tiles > 0,
                  "blstm_train_bwd_tc: bad arguments");
  const size_t dg_step = (size_t)tiles * (4 * H / 8) * 1024;  // halves
  const size_t g_step = (size_t)tiles * 128 * 8 * H;
  const size_t dy_step = (size_t)tiles * 128 * 2 * H;
  const size_t c_step = (size_t)tiles * 128 * H;
  __half* df = reinterpret_cast<__half*>(dG_f);
  __half* db = reinterpret_cast<__half*>(dG_b);
  const __half* g = reinterpret_cast<const __half*>(gates);
  const __half* dyh = reinterpret_cast<const __half*>(dy);
  for (int sb = 0; sb < steps; ++sb) {
    const int pf = steps - 1 - sb, pb = sb;                   // reverse of the forward order of each direction
    const int rc = bsrnn_blstm_bwd_step_tc(
        sb == 0 ? zero_tile : (const void*)(df + (size_t)(pf + 1) * dg_step), WT_f, g + (size_t)pf * g_step,
        dyh + (size_t)pf * dy_step, c_f + (size_t)pf * c_step, pf > 0 ? c_f + (size_t)(pf - 1) * c_step : nullptr, dc_f,
        df + (size_t)pf * dg_step,
        sb == 0 ? zero_tile : (const void*)(db + (size_t)(pb - 1) * dg_step), WT_b, g + (size_t)pb * g_step + 4 * (size_t)H,
        dyh + (size_t)pb * dy_step + H, c_b + (size_t)pb * c_step, pb < steps - 1 ? c_b + (size_t)(pb + 1) * c_step : nullptr, dc_b,
        db + (size_t)pb * dg_step, tiles, n_tiles, BN, H, 8L * H, 2L * H, valid_rows, stream);
    if (rc) return rc;
  }
  return 0;
}
