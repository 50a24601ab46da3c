/* bsrnn_b200.h — C ABI of the B200-native BSRNN / FlowSE hot path (libbsrnn_b200.so, sm_100a only).
 *
 * The reference (urgent-challenge/urgent2026_challenge_track1) defines NO FFI for this path: every device op is
 * a PyTorch library call (SURVEY.md §2.1).  The entry points below are therefore build-defined; each one cites the
 * reference call it replaces (file:line relative to the reference root; `espnet2/...` = the un-vendored
 * espnet==202412 dependency, behaviour in SURVEY.md Appendix A).
 *
 * Conventions
 *   - Stateless and stream-ordered: every pointer is a DEVICE pointer owned by the caller (torch allocates), every
 *     call enqueues on `stream` (a cudaStream_t passed as void*) and returns without synchronising.
 *   - No allocation inside; scratch and workspaces come from the caller (sizes follow from the documented layouts).
 *   - Return value: 0 = ok, non-zero = error; bsrnn_last_error() returns a thread-local message.
 *   - "spec" tensors are complex64 stored as interleaved float pairs, layout (B, T, F, 2).
 *   - "token-major" activations are (B, T, K, N) f32: token index ((b*T + t)*K + k).
 *   - precision modes: the *_f32 entry points compute in f32 on CUDA cores (parity bar 1e-3); the *_tc ones use
 *     tcgen05 tensor cores with fp16 operands (KB8 tiling) and f32 accumulation in TMEM (parity bar 1e-2).
 */
#ifndef BSRNN_B200_H_
#define BSRNN_B200_H_

#include <stdint.h>
#include <stddef.h>

#ifdef __cplusplus
extern "C" {
#endif

/* ---------------------------------------------------------------------------------------------- misc */
const char* bsrnn_last_error(void);
int bsrnn_abi_version(void);                 /* bumped whenever a signature changes */
int bsrnn_device_check(void);                /* 0 iff the current device is compute capability 10.x */
long bsrnn_launch_count(int reset);          /* kernels launched by this library since the last reset */

/* ---------------------------------------------------------------------------------------------- STFT / iSTFT
 * bsrnn_stft_fwd  replaces STFTEncoder.forward -> Stft.forward -> torch.stft (+ frame masking, + optional
 *   "exponent" compression)           [baseline_code/models/bsrnn.py:37, baseline_code/flow_model.py:136]
 *   wav (B, L) f32, lens (B) int32 (may be NULL = all L) -> spec (B, T, F, 2), T = 1 + L/hop, F = n_fft/2+1.
 *   Periodic Hann window of n_fft points, center=True reflect padding over the whole (padded) row of L samples,
 *   frames >= olens[b] = (lens[b] + 2*(n_fft/2) - n_fft)/hop + 1 written as zeros.
 *   transform: 0 none; 1 "exponent": |X|^exponent * e^{j arg X} * factor.
 *   twiddle: (n_fft, 2) f32 table exp(-2*pi*i*n/n_fft) from bsrnn_fft_twiddle().
 */
int bsrnn_fft_twiddle(float* twiddle, int n_fft, void* stream);
int bsrnn_stft_fwd(const float* wav, const int32_t* lens, float* spec, const float* twiddle, int B, int L,
                   int n_fft, int hop, int transform, float exponent, float factor, void* stream);

/* bsrnn_istft_fwd replaces the complex mask  s = m*x + r  (espnet2 BSRNN.forward tail; flow analogue
 *   baseline_code/models/bsrnn_flowse.py:311-316) fused with STFTDecoder.forward -> torch.istft
 *   [baseline_code/models/bsrnn.py:40, baseline_code/flow_model.py:145].
 *   spec (B,T,F,2); mask/resid (B,T,F,2) or NULL (then s = spec).  If spec_out != NULL the masked spectrum s is
 *   also written there (the `enhanced_feature` BSRNN_SE.forward returns).  transform 1 = inverse "exponent"
 *   (s/factor, |.|^(1/exponent)) applied after masking.  wav_out (B, L_out): inverse real DFT, Hann window,
 *   overlap-add, division by the window-square envelope, trim n_fft/2 (center=True), length = L_out.
 */
int bsrnn_istft_fwd(const float* spec, const float* mask, const float* resid, float* spec_out, float* wav_out,
                    const float* twiddle, int B, int T, int L_out, int n_fft, int hop, int transform,
                    float exponent, float factor, void* stream);

/* ---------------------------------------------------------------------------------------------- GroupNorm(1, C)
 * Statistics are per sample over everything else, zeros of padded frames/bins included (SURVEY.md §8g.1).
 * bsrnn_gn_stats:   x viewed as (B, rows_per_sample, C) with row stride `row_stride` floats, sample stride
 *                   rows_per_sample*row_stride; accumulates {sum, sumsq} as double into stats (B,2).
 *                   Replaces the reduction half of nn.GroupNorm at bsrnn_flowse.py:291,302 (norm_time/norm_freq).
 * bsrnn_band_stats: per (b, band) statistics over rows (b,t) of row_len floats; band k = floats
 *                   [band_off[k], band_off[k]+band_width[k]) of every row (device int32 arrays).  BandSplit:
 *                   x = spec (B,T,F,2), row_len 2F, off 2*bin0, width 2*min(s, F-bin0) (missing bins are zeros and
 *                   only enter through the count)  [bsrnn_flowse.py:65-73]; mask / grad decoders: x = skip (B,T,K,N),
 *                   row_len K*N, off k*N, width N  [espnet2 MaskDecoder; bsrnn_flowse.py:146-152].
 *                   stats (B, n_bands, 2) double, zeroed by the call.
 * bsrnn_gn_finalize: scale[b,c] = rstd_b*gamma_c, shift[b,c] = beta_c - mean_b*rstd_b*gamma_c (+ extra[b,c] if
 *                   non-NULL: the FlowSE time embedding added after the norm, bsrnn_flowse.py:293-294).
 *                   stats (G,2) double; gamma/beta (G_inner, C) and counts (G_inner) double (device), selected by
 *                   g % G_inner (G_inner = 1 for a plain layer norm, = n_bands for per-band norms with C the
 *                   padded channel width); scale/shift (G, C).  gn_stats zeroes `stats` itself.
 */
int bsrnn_gn_stats(const float* x, double* stats, int B, long rows_per_sample, int C, long row_stride, void* stream);
int bsrnn_band_stats(const float* x, double* stats, int B, int T, long row_len, const int32_t* band_off,
                     const int32_t* band_width, int n_bands, void* stream);
int bsrnn_gn_finalize(const double* stats, const float* gamma, const float* beta, const float* extra,
                      float* scale, float* shift, int G, int C, const double* counts, float eps, int G_inner,
                      void* stream);

/* ---------------------------------------------------------------------------------------------- grouped GEMM (f32)
 * One descriptor per group g (band / MLP / plain layer):
 *     C[row, n] = epi( sum_k A'[row, k] * W[n, k] + bias[n] ),   A'[row,k] = A[row,k]*scale[s,k] + shift[s,k]
 * with s = row / rows_per_sample (scale==NULL: identity).  Row r of A lives at
 *     A + (r / a_inner) * a_outer_stride + (r % a_inner) * a_inner_stride          (floats), same for C.
 * k >= k_valid reads as 0 before the affine (truncated last band, bsrnn_flowse.py:68-71).
 * epilogue: 0 store, 1 tanh, 2 C += result (residual, bsrnn_flowse.py:300,307), 3 GLU over the N axis
 *           (out[n] = v[n] * sigmoid(v[n + N/2]), n < N/2; nn.GLU(dim=1) in espnet2 MaskDecoder).
 * Only output columns n < n_store are written (bins beyond F of a truncated band are dropped, espnet2
 * BSRNN.forward `m[..., :F]`).
 */
typedef struct {
  const float* A; const float* W; const float* bias; float* C;
  const float* scale; const float* shift;
  long a_inner, a_outer_stride, a_inner_stride;
  long c_inner, c_outer_stride, c_inner_stride;
  long rows_per_sample, ss_stride;      /* scale/shift row of sample s starts at s*ss_stride */
  int M, N, K, k_valid, ldw, epilogue, n_store, pad_;
} bsrnn_gemm_desc;
/* descs: DEVICE array of n_groups descriptors; max_m/max_n: maxima over groups (grid sizing). */
int bsrnn_gemm_f32(const bsrnn_gemm_desc* descs, int n_groups, int max_m, int max_n, void* stream);

/* ---------------------------------------------------------------------------------------------- BLSTM (f32)
 * Replaces nn.LSTM(N, H, batch_first=True, bidirectional=True) forward with zero initial state
 * [bsrnn_flowse.py:226-238 construct, :296-297 (time axis) and :303-304 (band axis) call]; gate order i,f,g,o.
 * Sequences are addressed inside token-major tensors: sequence r = (r / seq_inner, r % seq_inner), step s:
 *     token(r, s) = (r / seq_inner) * seq_outer + (r % seq_inner) * seq_inner_stride + s * step_stride
 * time axis of (B,T,K): seq_inner=K, seq_outer=T*K, seq_inner_stride=1, step_stride=K, steps=T, R=B*K
 * band axis           : seq_inner=1, seq_outer=K,   seq_inner_stride=0, step_stride=1, steps=K, R=B*T
 *   gates_x (tokens, 2, 4H) f32 : x W_ih^T + b_ih + b_hh for both directions (from bsrnn_gemm_f32)
 *   w_hh    (2, 4H, H) f32      : weight_hh_l0, weight_hh_l0_reverse
 *   y       (tokens, 2H) f32    : output, [fwd | bwd] per token (also the h carrier between steps)
 *   c_state (2, R, H) f32       : scratch
 */
int bsrnn_blstm_recurrence_f32(const float* gates_x, const float* w_hh, float* y, float* c_state,
                               int R, int steps, int H, long seq_inner, long seq_outer, long seq_inner_stride,
                               long step_stride, void* stream);

/* ---------------------------------------------------------------------------------------------- tensor-core mode
 * fp16 operands, f32 accumulation in TMEM (tcgen05).  Operands use the UMMA-native "KB8" tiling
 *     X_kb8[tile][K/8][rows_per_tile][8]      (rows_per_tile = 128 for activations, BN for weights)
 * so every pipeline stage is one contiguous bulk copy.  Row tiles map to tokens through
 *     m_tile = step*tiles_per_step + j ;  seq = j*128 + r (valid iff seq < R) ;
 *     token  = (seq / seq_inner)*seq_outer + (seq % seq_inner)*seq_inner_stride + step*step_stride .
 *
 * bsrnn_norm_cast_kb8: out_kb8 = fp16( x[token, col0:col0+C] * scale[g] + shift[g] ), zero padded to kcores*8 columns;
 *     g = (token / tokens_per_sample)*g_inner + (g_inner > 1 ? token % g_inner : 0).  The apply half of
 *     nn.GroupNorm(1,N) [bsrnn_flowse.py:291,302,146-152] fused with the operand re-tiling.
 *     _ones: additionally writes the constant 1 into padding column one_col (C <= one_col < kcores*8, multiple of 4;
 *     -1 = none) so that a bias stored as weight column one_col is added by the GEMM itself (bias = NULL there).
 * bsrnn_gemm_tc: C = A_kb8 * W_kb8^T + bias (bias may be NULL) with epilogue
 *     0: fp16 rows      out[token*ldo + col]                              (LSTM input projection, :296,:303)
 *     1: f32 residual   out[token*ldo + col] += .., col < n_valid; optional per-sample {sum,sumsq} of the new
 *                       values added into stats (samples,2) double        (Linear + skip :298-300,:305-307 and the
 *                       statistics of the next GroupNorm)
 *     2: tanh -> fp16 KB8 operand with out_kcores k-cores                 (MaskDecoder Conv1d(N->4N)+Tanh)
 *     3: GLU on (value,gate)-interleaved columns -> f32 out[token*ldo + col/2], col/2 < n_valid
 *     4: fp16 KB8 tiles out[m_tile][out_kcores][128][8], core = global column / 8 (LSTM input projection in the
 *        layout the recurrence kernel reads with coalesced 16-byte loads)
 *     7: tanh -> f32 rows out[token*ldo + col], col < n_valid             (GradDecoder Conv1d(N->16 s)+Tanh,
 *        bsrnn_flowse.py:118-134: the channel-last image of the 5x5 conv)
 *     8: epilogue 1 (f32 residual + statistics) with the tile's residual row segments moved by one bulk (TMA) copy
 *        per row into a shared-memory row buffer, updated there and stored back by one bulk store per row; rows must be
 *        16-byte aligned (ldo % 4 == 0, BN % 4 == 0, out 16-byte aligned)
 *     Epilogues 0 and 4 store every column of every N tile (they do not clip at n_valid), so a call is rejected unless
 *     n_tiles*BN <= ldo (epilogue 0) or n_tiles*BN <= 8*out_kcores (epilogue 4).  The row epilogues 1, 3, 7 and 8 (and
 *     bsrnn_gemm_tc_scaled) need 0 < n_valid <= ldo.  Epilogue 2 writes k-cores < out_kcores only, with columns
 *     n_valid .. 8*out_kcores - 1 stored as zeros when bias != NULL (the bias-free launches rely on zero weight rows there).
 * bsrnn_blstm_recurrence_tc: persistent cluster kernel, H = 392 only (csrc/lstm_tc.cu).  Sequences are grouped in
 *     tiles of 128 (seq = j*128 + r, valid iff seq < R); all operands are (step, seq_tile)-major:
 *       gates_x [step][seq_tile][dir][q][26][128][8] fp16 — epilogue 4 of bsrnn_gemm_tc over A tiles built with the
 *               axis' row map (m_tile = step*seq_tiles + j) and the packed W_ih of 16 column tiles (dir, q);
 *       w_pack  [dir][q][50][208][8] fp16; zero_tile: 50*128*8 fp16 zeros (h before the first step);
 *       y       [step][seq_tile][dir][50][128][8] fp16 (k-core 49 must stay zero).
 *     The i, f, o gate rows of W_ih / W_hh / bias are pre-multiplied by 0.5 by the packer.
 *     max_clusters <= 0: use every co-resident cluster.  _ex: `slots` = sequence tiles one cluster interleaves
 *     (1..3; <= 0 = 3).
 */
int bsrnn_norm_cast_kb8(const float* x, const float* scale, const float* shift, void* out, long ldx, int col0, int C,
                        int kcores, int m_tiles, int tiles_per_step, int R, long seq_inner, long seq_outer,
                        long seq_inner_stride, long step_stride, long tokens_per_sample, int g_inner, void* stream);
int bsrnn_norm_cast_kb8_ones(const float* x, const float* scale, const float* shift, void* out, long ldx, int col0,
                             int C, int kcores, int m_tiles, int tiles_per_step, int R, long seq_inner, long seq_outer,
                             long seq_inner_stride, long step_stride, long tokens_per_sample, int g_inner, int one_col,
                             void* stream);
int bsrnn_gemm_tc(const void* A, const void* W, const float* bias, void* out, double* stats, int m_tiles, int n_tiles,
                  int kcores, int BN, int epilogue, long ldo, int n_valid, int out_kcores, long tokens_per_sample,
                  int tiles_per_step, int R, long seq_inner, long seq_outer, long seq_inner_stride, long step_stride,
                  void* stream);
/* bsrnn_gemm_tc_ex: bsrnn_gemm_tc with two extras of the f32-row epilogues 1 / 8.
 *     stats_inner > 1: the statistics row is (token / tokens_per_sample) * stats_inner + token % stats_inner, i.e. per
 *       (sample, band) on the (B,T,K,N) residual stream with stats_inner = K: the reduction half of the mask decoder's
 *       per-band GroupNorm(1, N) over (N, T) [espnet2 MaskDecoder; bsrnn_flowse.py:146-152] taken in the epilogue of the
 *       last Linear + skip instead of a separate pass over the stream;
 *     flags bit 0 (epilogue 8 only): store only, out[token*ldo + col] = A W^T + bias (no residual read) -- the
 *       tensor-core BandSplit Conv1d(2 s_k -> N, 1) [bsrnn_flowse.py:65-86], whose statistics are those of the first
 *       dual-path GroupNorm.
 * bsrnn_band_norm_cast_kb8: the operand of that GEMM for ALL bands in one launch: band k's slice of the spectrum (rows,
 *     F2 = 2F floats), zero-padded to 2 s_k = c_off[k+1] - c_off[k] channels BEFORE the per-(sample, band) affine scale /
 *     shift (B*K, cmax), as fp16 tiles [tile][kc_k][128][8] at out + a_off[k] halves, kc_k = 2 * ceil(2 s_k / 16). */
int bsrnn_gemm_tc_ex(const void* A, const void* W, const float* bias, void* out, double* stats, int m_tiles, int n_tiles,
                     int kcores, int BN, int epilogue, long ldo, int n_valid, int out_kcores, long tokens_per_sample,
                     int tiles_per_step, int R, long seq_inner, long seq_outer, long seq_inner_stride, long step_stride,
                     int stats_inner, int flags, void* stream);
/* bsrnn_gemm_tc_grouped: the store-only GEMM of bsrnn_gemm_tc_ex (epilogue 8, flags 1) for n_groups bands in ONE launch:
 *     out[token*ldo + out_off_g + c] = A_g W_g^T + bias_g, c < n_valid, tile order (row tile, band) with the band innermost so
 *     that co-running CTAs write adjacent segments of the same output rows.  groups: device int64 [n_groups][5] =
 *     {a_off (halves into A: the group's tile 0), w_off (halves into W), out_off (floats), bias_off (floats), kcores};
 *     A_g tiles [row tile][kcores_g][128][8], W_g [kcores_g][BN][8]; kc_max = max kcores_g; m_tiles = row tiles per group;
 *     the row map (tiles_per_step ...) applies to the row tile.  BandSplit Conv1d(2 s_k -> N, 1) [bsrnn_flowse.py:65-86]. */
int bsrnn_gemm_tc_grouped(const void* A, const void* W, const float* bias, void* out, double* stats,
                          const long long* groups, int n_groups, int m_tiles, int kc_max, int BN, long ldo, int n_valid,
                          long tokens_per_sample, int tiles_per_step, int R, long seq_inner, long seq_outer,
                          long seq_inner_stride, long step_stride, void* stream);
/* bsrnn_gemm_tc_limit_ctas: upper bound on the persistent CTAs of the following bsrnn_gemm_tc* launches of this process (0 =
 *     every SM); returns the previous bound.  The mask decoder's two MLP families [espnet2 MaskDecoder: mlp_mask /
 *     mlp_residual] run on two streams with half of the SMs each. */
int bsrnn_gemm_tc_limit_ctas(int n);
int bsrnn_band_norm_cast_kb8(const float* spec, const float* scale, const float* shift, void* out, const int32_t* c_off,
                             const int32_t* bin0, const int32_t* width2, const long long* a_off, int K, long rows, int T,
                             int F2, int cmax, void* stream);
/* bsrnn_lstm_step_tc: ONE time step of one LSTM direction on tensor cores for any hidden size H % 16 == 0 (FlowSE: H = 768,
 *     which does not fit the persistent kernel above) [nn.LSTM, bsrnn_flowse.py:226-238]: h_{t-1} * W_hh^T as a tcgen05 GEMM
 *     whose epilogue adds the input projection, applies the gates, updates c in place and writes h_t as the KB8 tile that is
 *     the next step's A operand and the layer output.  A / out_h: [m_tiles][H/8][128][8] fp16 (zero tiles for the first
 *     step); W: [n_tiles][H/8][BN][8] fp16, rows reordered to 4u + gate, i/f/o rows pre-halved, BN % 32 == 0;
 *     gx: rows [m*128 + r][ld_gx] fp16 of this step and direction (same column order, bias included);
 *     cstate: [m_tiles*128][H] f32. */
int bsrnn_lstm_step_tc(const void* A, const void* W, const void* gx, float* cstate, void* out_h, int m_tiles, int n_tiles,
                       int BN, int H, long ld_gx, void* stream);
/* bsrnn_blstm_step_tc: the forward and the backward direction of one BLSTM time step in ONE launch (row tiles
 *     [0, m_tiles) use the *_f pointers, [m_tiles, 2*m_tiles) the *_b pointers); arguments as bsrnn_lstm_step_tc. */
int bsrnn_blstm_step_tc(const void* A_f, const void* W_f, const void* gx_f, float* c_f, void* out_f, const void* A_b,
                        const void* W_b, const void* gx_b, float* c_b, void* out_b, int m_tiles, int n_tiles, int BN,
                        int H, long ld_gx, void* stream);
int bsrnn_blstm_recurrence_tc(const void* gates_x, const void* w_pack, const void* zero_tile, void* y, int R, int steps,
                              int seq_tiles, int max_clusters, void* stream);
int bsrnn_blstm_recurrence_tc_ex(const void* gates_x, const void* w_pack, const void* zero_tile, void* y, int R,
                                 int steps, int seq_tiles, int max_clusters, int slots, void* stream);
int bsrnn_blstm_tc_max_clusters(void);
/* Co-resident 16-CTA clusters of the CTA-pair schedule (BSRNN_LSTM_VER=7: cta_group::2 MMAs, half of the W_hh slice
 * per CTA); <= 0 when the device cannot host one. */
int bsrnn_blstm_tc_max_pair_clusters(void);
/* bsrnn_blstm_recurrence_tc_flag: the same recurrence with FLAG GROUPS instead of thread-block clusters: the 8 CTAs
 *     of a work unit announce "h_t is in L2" through gpu-scope release/acquire counters in sync_ws, so they need not
 *     share a GPC: floor(148/8) = 18 groups (144 SMs) are co-resident instead of 15 clusters (120 SMs).  sync_ws:
 *     bsrnn_blstm_tc_sync_bytes() bytes of caller-owned device memory (zeroed inside, stream-ordered).  max_groups
 *     <= 0: all co-resident groups; slots <= 0: the fewest interleaved tiles per group that cover every unit in one
 *     wave.  The launch must be the only resident kernel of its size class: its CTAs spin on each other. */
int bsrnn_blstm_recurrence_tc_flag(const void* gates_x, const void* w_pack, const void* zero_tile, void* y, int R,
                                   int steps, int seq_tiles, int max_groups, int slots, void* sync_ws, void* stream);
int bsrnn_blstm_tc_flag_max_groups(void);
int bsrnn_blstm_tc_sync_bytes(void);
/* bsrnn_blstm_fused_tc: the whole nn.LSTM(N=196, H=392, bidirectional) layer [reference bsrnn_flowse.py:226-238,
 *     called at :296-297 / :303-304] in ONE persistent kernel: gates_t = [x_t | h_{t-1}] [W_ih | W_hh]^T per step, so
 *     the input-projection GEMM and its gates_x tensor (13.9 GB per call at BASELINE config 2) disappear.  CTA pairs
 *     (tcgen05 cta_group::2, M = 256) hold half of a 208 x 608 weight slice each; groups of 8 pairs synchronise through
 *     gpu-scope counters in sync_ws (bsrnn_blstm_fused_sync_bytes() bytes, zeroed inside, stream-ordered).
 *     xhat: fp16 [steps*seq_tiles][26][128][8] as written by bsrnn_norm_cast_kb8_ones (column 196 = 1 carries the
 *     bias); w_fused: fp16 [2 dirs][8 pairs][2 halves][76 k-cores][104][8]; zero_tile / y as bsrnn_blstm_recurrence_tc.
 *     max_groups <= 0: all co-resident groups; slots <= 0: automatic (1..3 interleaved tile pairs per group). */
int bsrnn_blstm_fused_tc(const void* xhat, const void* w_fused, const void* zero_tile, void* y, int R, int steps,
                         int seq_tiles, int max_groups, int slots, void* sync_ws, void* stream);
int bsrnn_blstm_fused_max_groups(void);
int bsrnn_blstm_fused_sync_bytes(void);
/* bsrnn_blstm_fused7_tc: bsrnn_blstm_fused_tc on groups of 7 CTA pairs x 56 hidden units (224 gate columns, no padding):
 *     10 co-resident groups (140 SMs) instead of 9, i.e. 5 per direction - the schedule for sequence-tile counts that 9
 *     groups split badly (BASELINE config 2 time axis: 9 tile pairs per direction).  w_fused7: fp16
 *     [2][7][2][76][112][8]; every other argument as bsrnn_blstm_fused_tc. */
int bsrnn_blstm_fused7_tc(const void* xhat, const void* w_fused7, const void* zero_tile, void* y, int R, int steps,
                          int seq_tiles, int max_groups, int slots, void* sync_ws, void* stream);
int bsrnn_blstm_fused7_max_groups(void);
/* bsrnn_blstm_fused14_tc: the small-batch geometry: groups of 14 CTA pairs x 28 hidden units (112 gate columns), 5
 *     co-resident groups.  With few sequence tiles the layer is bound by the per-step dependency chain; sharing a tile
 *     among twice as many CTAs halves the epilogue and MMA time of an item (at twice the L2 traffic per item).
 *     w_fused14: fp16 [2][14][2][76][56][8]; every other argument as bsrnn_blstm_fused_tc. */
int bsrnn_blstm_fused14_tc(const void* xhat, const void* w_fused14, const void* zero_tile, void* y, int R, int steps,
                           int seq_tiles, int max_groups, int slots, void* sync_ws, void* stream);
/* bsrnn_blstm_fused_train_tc: TRAINING forward of the BLSTM layer (H = 392) on the fused kernel: geo = 7 | 14 as
 *     bsrnn_blstm_fused7_tc / _fused14_tc, separate output buffers per direction (block (step, tile) of direction d at
 *     y_d + (step*seq_tiles + tile) * y_stride halves, [50][128][8], k-core 49 stays zero), and the activations BPTT needs
 *     written by the epilogue: gates rows [(step*seq_tiles + tile)*128 + r][8H] fp16 = ACTIVATED i, f, g, o at column
 *     dir*4H + 4u + gate; c_f / c_b [step][seq_tiles*128][H] f32 -- the buffers bsrnn_blstm_train_bwd_tc reads
 *     [autograd's saved tensors of nn.LSTM in SEModel.training_step, d_model.py:61-95]. */
int bsrnn_blstm_fused_train_tc(int geo, const void* xhat, const void* w_fused, const void* zero_tile, void* y_f, void* y_b,
                               long y_stride, void* gates, float* c_f, float* c_b, void* scratch, int R, int steps,
                               int seq_tiles, int max_groups, int slots, void* sync_ws, void* stream);
/* scratch of the call above in bytes: the epilogue stores the activations unit-major ([unit][128 rows], coalesced over a
 * warp's rows) and a transpose kernel inside the call writes the row-major buffers. */
long bsrnn_blstm_fused_train_scratch_bytes(int steps, int seq_tiles);
int bsrnn_blstm_fused14_max_groups(void);
/* bsrnn_blstm_fused768_tc: the same fused layer kernel for nn.LSTM(N=384, H=768, bidirectional) of BSRNN_flowse
 *     [reference bsrnn_flowse.py:226-238 at the conf/models/BSRNN_flowse.yaml width]: groups of 24 CTA pairs (32 hidden
 *     units = 128 gate columns per pair), replacing the input-projection GEMM + one bsrnn_blstm_step_tc launch per time
 *     step.  xhat: fp16 [steps*seq_tiles][50][128][8] (bsrnn_norm_cast_kb8_ones with kcores = 50, column 384 = 1);
 *     w_fused: fp16 [2][24][2][146][64][8]; zero_tile: 96*128*8 zeros; the (step, tile) block [96][128][8] of
 *     direction d lives at y_d + (step*seq_tiles + tile) * y_stride halves: two buffers as bsrnn_blstm_step_tc writes
 *     them (y_stride = 96*1024) or one interleaved [..][dir][96][128][8] buffer (y_b = y_f + 96*1024, y_stride =
 *     2*96*1024), which is the K = 1536 operand of ONE Linear(2H -> N) GEMM.  sync_ws as bsrnn_blstm_fused_tc. */
int bsrnn_blstm_fused768_tc(const void* xhat, const void* w_fused, const void* zero_tile, void* y_f, void* y_b,
                            long y_stride, int R, int steps, int seq_tiles, int max_groups, int slots, void* sync_ws,
                            void* stream);
int bsrnn_blstm_fused768_max_groups(void);
/* bsrnn_blstm_fused768_train_tc: TRAINING forward of the H = 768 layer on the fused kernel: xhat, w_fused, zero_tile and
 *     y_f / y_b / y_stride as bsrnn_blstm_fused768_tc (y_stride >= 96*1024, a multiple of 8), plus the activations BPTT
 *     needs, written by the epilogue: gates rows [(step*seq_tiles + tile)*128 + r][8H] fp16 = ACTIVATED i, f, g, o at
 *     column dir*4H + 4u + gate; c_f / c_b [step][seq_tiles*128][H] f32 -- the buffers bsrnn_blstm_train_bwd_tc reads
 *     [autograd's saved tensors of nn.LSTM in FlowSEModel.training_step, flow_model.py:149-187].  sync_ws as
 *     bsrnn_blstm_fused_tc; scratch as below. */
int bsrnn_blstm_fused768_train_tc(const void* xhat, const void* w_fused, const void* zero_tile, void* y_f, void* y_b,
                                  long y_stride, void* gates, float* c_f, float* c_b, void* scratch, int R, int steps,
                                  int seq_tiles, int max_groups, int slots, void* sync_ws, void* stream);
/* scratch of the call above in bytes (unit-major activations, as bsrnn_blstm_fused_train_scratch_bytes at H = 768). */
long bsrnn_blstm_fused768_train_scratch_bytes(int steps, int seq_tiles);

/* Debug / A-B timing: selects the recurrence schedule (4, 5, 6: 8-CTA clusters; 7: CTA pairs); any other value
 * returns to the BSRNN_LSTM_VER environment default. */
void bsrnn_debug_set_lstm_schedule(int ver);

/* ---------------------------------------------------------------------------------------------- training (f32)
 * The sequential parts of the BLSTM forward/backward for train_se.py [reference d_model.py:61-95 -> autograd through
 * nn.LSTM at bsrnn_flowse.py:296-297,303-304]; the batched GEMMs around them (input projection, dW, dx) are plain
 * library GEMMs issued by the host side (training.py).
 * bsrnn_blstm_train_fwd_f32: bsrnn_blstm_recurrence_f32 that also stores saved (tokens, 2, 5, H) = sigmoid(i),
 *     sigmoid(f), tanh(g), sigmoid(o), c per (token, direction).
 * bsrnn_blstm_train_bwd_f32: back-propagation through time.  dy (tokens, 2H) = dL/dy -> dgates (tokens, 2, 4H) =
 *     dL/d gates_x (pre-activations, gate order i,f,g,o).  dh_rec, dc_carry: (2, R, H) f32 scratch.
 * bsrnn_grad_sumsq / bsrnn_adamw_step: the optimizer tail on one flat buffer — stats = {sum g^2, non-finite flag};
 *     gradients are scaled by grad_scale (1/world after a summed allreduce), clipped to max_norm like
 *     torch.nn.utils.clip_grad_norm_ [train_se.py:78], the step is skipped when a non-finite gradient was seen
 *     [d_model.py:48-57], then AdamW with decoupled weight decay [d_model.py:102-109] and, if ema != NULL,
 *     ema -= (1-ema_decay)*(ema - param) [torch_ema, flow_model.py:84].
 */
int bsrnn_blstm_train_fwd_f32(const float* gates_x, const float* w_hh, float* y, float* c_state, float* saved, int R,
                              int steps, int H, long seq_inner, long seq_outer, long seq_inner_stride,
                              long step_stride, void* stream);
int bsrnn_blstm_train_bwd_f32(const float* dy, const float* saved, const float* w_hh, float* dgates, float* dh_rec,
                              float* dc_carry, int R, int steps, int H, long seq_inner, long seq_outer,
                              long seq_inner_stride, long step_stride, void* stream);
int bsrnn_grad_sumsq(const float* grad, long n, double* stats, void* stream);
int bsrnn_adamw_step(float* param, const float* grad, float* exp_avg, float* exp_avg_sq, float* ema, long n,
                     const double* stats, float grad_scale, float max_norm, float lr, float beta1, float beta2,
                     float eps, float weight_decay, int step, float ema_decay, void* stream);
/* bsrnn_adamw_step2: the same tail with the step counters kept ON THE DEVICE, so a step skipped for non-finite
 *     gradients does not advance Adam's bias correction (reference: optimizer.zero_grad() makes AdamW skip every
 *     parameter AND its step counter, d_model.py:48-59) while torch_ema's update still runs (flow_model.py:66-84).
 *     state (double[8]) = {sum g^2, non-finite flag [both written by bsrnn_grad_sumsq], adam steps, ema updates,
 *     1-beta1^t, 1-beta2^t, effective ema decay, -}; zero it once.  skip_ranges: n_skip (<= 32) half-open element
 *     ranges [lo, hi) (long pairs, device memory) of parameters that received NO gradient on any rank this step
 *     (bands beyond K' at low sample rates): torch AdamW skips grad=None parameters entirely -- no weight decay, no
 *     moment decay.  ema_decay is the nominal decay; the warm-up min(decay, (1+n)/(10+n)) is applied inside. */
int bsrnn_adamw_step2(float* param, const float* grad, float* exp_avg, float* exp_avg_sq, float* ema, long n,
                      double* state, const long* skip_ranges, int n_skip, float grad_scale, float max_norm, float lr,
                      float beta1, float beta2, float eps, float weight_decay, float ema_decay, void* stream);

/* ---------------------------------------------------------------------------------------------- training (tensor cores)
 * The BLSTM blocks of the training step on tcgen05 (fp16 operands, f32 accumulation, f32 master weights), replacing
 * autograd through nn.LSTM / nn.Linear [reference d_model.py:61-95, bsrnn_flowse.py:296-307]:
 * bsrnn_blstm_step_train_tc: one forward time step of both directions that also saves what BPTT needs (activated gates
 *     over the input projection, c_t per step).
 * bsrnn_blstm_bwd_step_tc: one BPTT step of both directions: recurrent GEMM dG_{t+1} W_hh + gate derivatives -> dG_t
 *     (KB8 tiles: next step's operand and the operand of the dx / dW GEMMs).
 * bsrnn_gemm_tc_scaled: out += scale * A W^T (f32, row-mapped): dx = dG W_ih, dW = dG^T X (tokens as K), with the fp16
 *     loss scale (a device scalar, so choosing it costs no host sync) removed in f32.
 * bsrnn_kb8_transpose: KB8 operand -> KB8 operand of its transpose (tokens become the K axis for the dW GEMMs). */
int bsrnn_blstm_step_train_tc(const void* A_f, const void* W_f, void* gx_f, const float* cprev_f, float* cout_f, void* out_f,
                              const void* A_b, const void* W_b, void* gx_b, const float* cprev_b, float* cout_b,
                              void* out_b, int m_tiles, int n_tiles, int BN, int H, long ld_gx, void* stream);
int bsrnn_blstm_bwd_step_tc(const void* A_f, const void* W_f, const void* sg_f, const void* dy_f, const float* ccur_f,
                            const float* cprev_f, float* dc_f, void* out_f, const void* A_b, const void* W_b,
                            const void* sg_b, const void* dy_b, const float* ccur_b, const float* cprev_b, float* dc_b,
                            void* out_b, int m_tiles, int n_tiles, int BN, int H, long ld_sg, long ld_dy, int valid_rows,
                            void* stream);
/* whole-sequence drivers (the host loop over the time steps of both directions, in C) */
int bsrnn_blstm_train_fwd_tc(const void* zero_tile, void* y_f, void* y_b, const void* W_f, const void* W_b, void* gates,
                             float* c_f, float* c_b, int steps, int tiles, int n_tiles, int BN, int H, void* stream);
int bsrnn_blstm_train_bwd_tc(const void* zero_tile, void* dG_f, void* dG_b, const void* WT_f, const void* WT_b,
                             const void* gates, const void* dy, const float* c_f, const float* c_b, float* dc_f, float* dc_b,
                             int steps, int tiles, int n_tiles, int BN, int H, int valid_rows, void* stream);
int bsrnn_gemm_tc_scaled(const void* A, const void* W, const float* bias, void* out, int m_tiles, int n_tiles, int kcores,
                         int BN, long ldo, int n_valid, float out_scale, const float* out_scale_ptr, int ksplit,
                         int tiles_per_step, int R, long seq_inner, long seq_outer, long seq_inner_stride,
                         long step_stride, void* stream);   /* scale = *out_scale_ptr (device) if non-null; ksplit > 1:
                         K split over CTAs with atomic adds (weight gradients: few output tiles, K = tokens) */
int bsrnn_kb8_transpose(const void* src, void* dst, int src_m0, int m_count, int kc_src, int BN, int n_tiles,
                        long dst_kcores, long dst_kc0, void* stream);

/* bsrnn_stft_stats_fwd: bsrnn_stft_fwd that also accumulates, per (utterance, band), the sum and the sum of squares of the
 *   spectrum it writes (band_stats (B, n_bands, 2) double, zeroed inside; band_bin0 [n_bands + 1] first bins): the
 *   reduction half of BandSplit's GroupNorm(1, 2 s_k) [bsrnn_flowse.py:72-73] without a second pass over the spectrum.
 * bsrnn_band_split_fwd: BandSplit.forward [bsrnn_flowse.py:65-86] for all bands: normalise on load (scale / shift from
 *   bsrnn_gn_finalize, zero padding of a truncated band BEFORE the norm), Conv1d(2 s_k -> N, 1) with the band's transposed
 *   weight resident in shared memory, rows of the token-major (B, T, K', out_width) output written whole.  wT: all bands'
 *   weights transposed and concatenated ((sum_k 2 s_k) x N); c_off [K+1] channel offsets (device + host copy). */
int bsrnn_stft_stats_fwd(const float* wav, const int32_t* lens, float* spec, const float* twiddle, int B, int L, int n_fft,
                         int hop, int transform, float exponent, float factor, double* band_stats,
                         const int32_t* band_bin0, int n_bands, void* stream);
int bsrnn_band_split_fwd(const float* spec, const float* scale, const float* shift, const float* wT, const float* bias,
                         float* out, const int32_t* c_off, const int32_t* bin0, const int32_t* width2,
                         const int32_t* c_off_host, int K, long rows, int T, int F2, int N, int cmax, long ldo,
                         int out_width, int out_col, void* stream);

/* bsrnn_istft_bwd: backward of bsrnn_istft_fwd (no mask, no transform) for the training step [replaces autograd through
 *   torch.istft, reference d_model.py:71-74]: d_wav (B, L_out) -> d_spec (B, T, F, 2) = c_k / N * DFT(w * d_wav / envelope)
 *   per frame, zero outside [0, L_out), imaginary parts of DC / Nyquist zero. */
int bsrnn_istft_bwd(const float* d_wav, float* d_spec, const float* twiddle, int B, int T, int L_out, int n_fft, int hop,
                    void* stream);

/* ---------------------------------------------------------------------------------------------- training loss
 * The core of espnet2 MultiResL1SpecLoss as configured at d_model.py:24 (window_sz [256,512,768,1024], hop w/2,
 * rectangular window, center=True reflect padding, onesided, reduction "sum"), VALUE AND GRADIENT in one pass
 * [replaces d_model.py:74 forward + the autograd backward of the four torch.stft/abs pairs]:
 *   loss[b] += weight * sum |e - t|                                  (bsrnn_l1_time_fwd_bwd, the time-domain term)
 *   loss[b] += weight * sum_{frames,bins} | |STFT_w(e)| - |STFT_w(t)| |   (bsrnn_mrl1_spec_fwd_bwd, one window size w)
 * and grad (B, L) accumulates d loss[b] / d e[b, :].  est, tgt (B, L) f32 are the already scaled / variance-normalised
 * signals; loss (B) double and grad (B, L) f32 are zeroed by the caller; twiddle from bsrnn_fft_twiddle(window).
 * Call the time-domain term first (plain stores into grad), then the spectral terms (atomic adds). */
int bsrnn_l1_time_fwd_bwd(const float* est, const float* tgt, double* loss, float* grad, int B, int L, float weight,
                          void* stream);
int bsrnn_mrl1_spec_fwd_bwd(const float* est, const float* tgt, double* loss, float* grad, const float* twiddle, int B,
                            int L, int window, float weight, void* stream);

/* ---------------------------------------------------------------------------------------------- FlowSE pieces
 * bsrnn_time_embed: GaussianFourierProjection [bsrnn_flowse.py:90-99]: out (B, 2*E) = [sin(2*pi*t*W), cos(...)].
 * bsrnn_conv5x5_glu: GradDecoder.conv_after_* = Conv2d(16->4, 5x5, pad 2) + GLU(dim=1) [bsrnn_flowse.py:114-117,
 *   163-164] on g (B, T, Fp, 16) channel-last -> out (B, T, F, 2) (bins >= Fp zero, bsrnn_flowse.py:166-167).
 *   weight (4,16,5,5) as in the state_dict, kernel dims ordered (freq, time) like the reference's (F', T) image.
 * bsrnn_euler_step: x <- x + step*(m*x + r)  [sampling/odesolvers.py:76-81 with VF = -dnn, flow_model.py:203-209];
 *   all (B,T,F,2); in place on x.
 * bsrnn_fm_prior: x = y + sigma*z  [models/odes.py:84-91].
 */
int bsrnn_time_embed(const float* t, const float* W, float* out, int B, int E, void* stream);
int bsrnn_conv5x5_glu(const float* g, const float* weight, const float* bias, float* out, int B, int T, int Fp,
                      int F, void* stream);
int bsrnn_euler_step(float* x, const float* mask, const float* resid, float step, long n_complex, void* stream);
int bsrnn_axpy_complex(float* out, const float* y, const float* z, float sigma, long n_complex, void* stream);
/* out = sign * (mask*x + resid): the network output g = m*x_t + r [bsrnn_flowse.py:313-316]; sign=-1 gives the
 * vector field FlowSEModel.forward returns [flow_model.py:203-209]. */
int bsrnn_complex_mask(float* out, const float* x, const float* mask, const float* resid, float sign, long n_complex,
                       void* stream);

#ifdef __cplusplus
}
#endif
#endif  /* BSRNN_B200_H_ */
