// lstm_fused.cu — BLSTM layer with the INPUT PROJECTION FUSED into the persistent recurrence:
//     gates_t = [x_t | h_{t-1}] * [W_ih | W_hh]^T          (one contraction over K = N_in + H per step)
// so the gates_x tensor that the step-wise / lstm_tc.cu kernels read (13.9 GB per BLSTM call at BASELINE config 2, written
// by a separate input-projection GEMM) is never materialised.  Replaces nn.LSTM(N, 2N, bidirectional) [reference
// bsrnn_flowse.py:226-238, called at :296-297 (time axis) and :303-304 (band axis)] including its x * W_ih^T + b half,
// for the two widths the reference configures: N = 196 / H = 392 (BSRNN_baseline) and N = 384 / H = 768 (BSRNN_flowse).
//
// Why CTA pairs.  At H = 392 with 8 CTAs per sequence tile a CTA would have to keep a 208 x 608 fp16 slice (253 KB)
// resident — more than the 227 KB of shared memory.  A CTA PAIR (2-CTA cluster, tcgen05 cta_group::2, M = 256) shares one
// slice: each CTA keeps HALF of the pair's gate columns and supplies its own 128 sequence rows; the MMA delivers all gate
// columns of those rows into the CTA's own TMEM.  Per CTA and item the L2 -> SM traffic is the h tile plus the x tile, the
// same as the h tile plus the gates_x slice before.
//
// Decomposition.  Work unit = (direction, PAIR of 128-sequence tiles).  A GROUP = PPG pairs (any placement: pairs rank
// themselves by an arrival ticket) owns up to 3 interleaved units of one direction; pair q owns hidden units
// [UPP*q, UPP*q + UPP).  The even CTA of each pair serves tile 2j, the odd CTA tile 2j+1; the PPG CTAs of one parity
// exchange h_t of "their" tile through y in L2 and a gpu-scope release/acquire counter in global memory (the flag
// protocol of lstm_tc_flag_kernel), so the only cluster traffic is inside a pair:
//   warp 0  producer : per item the ring stages of x_t (no dependency: they stream ahead) and, once the parity's
//                      counter shows h_{t-1} complete, the stages of h;
//   warp 1  leader   : MMA issuer — tcgen05.mma.cta_group::2 (M=256, N=BN, K=16), commits multicast to both CTAs'
//                      `empty` / `acc_full` barriers;
//           odd CTA  : relays its `full` completions to the leader's `pfull` barriers (RELAXED remote arrive: a
//                      release.cluster arrive costs ~1 000 cycles per stage and paced the whole ring, profiles/r02 call20/21);
//   warp 2  publisher: named barrier with the epilogue warps, then one red.release on the parity's counter;
//   warps 4..        : epilogue, all warps on every item (thread = sequence row x share of the units): tcgen05.ld in
//                      16-column chunks software-pipelined against the MUFU work, c in registers, h_t -> y.
// The bias rides in the weights (operand column N is the constant 1 written by norm_cast_kb8_ones), the i/f/o rows are
// pre-halved (sigmoid(x) = 0.5*tanh(x/2)+0.5), step 0 skips the h half (h_{-1} = 0).
//
//                     H = 392 (Geo392)                          H = 768 (Geo768)
//   pairs per group   8 x 49 units (N = 208 incl. 12 pad)       24 x 32 units (N = 128)
//   K                 26 + 50 k-cores (208 + 400)               50 + 96 k-cores (400 + 768)
//   W half per CTA    76 x 104 x 16 B = 126 KB                  146 x 64 x 16 B = 150 KB
//   ring              5 stages x 10 k-cores (20 KB)             3 stages x 12 k-cores (24 KB)
//   epilogue          12 warps: row x third (16/16/17 units)    16 warps: row x quarter (8 units = one 16-byte k-core row)
//   TMEM              2 accumulators x 256 columns              4 accumulators x 128 columns
//   co-resident       9 groups of 16 CTAs (144 SMs)             3 groups of 48 CTAs (144 SMs)
//
// x (fp16)   : [step][seq_tile][XKC k-cores][128 rows][8]   — what bsrnn_norm_cast_kb8_ones writes
// y (fp16)   : per direction [step][seq_tile][HKC k-cores][128 rows][8]; H = 392 interleaves the directions in one buffer
//              ([step][seq_tile][dir][50]...: the Linear GEMM's 128 x 800 operand tile), H = 768 keeps two buffers
// w pack     : [dir][pair q][parity e][XKC k-cores of W_ih (+bias column) then HKC of W_hh][BN/2 gate rows][8]
#include "lstm_tc_common.cuh"
#include <stdlib.h>

#ifndef BSRNN_FUSED768_CLS
#define BSRNN_FUSED768_CLS 2
#endif

namespace bsrnn {

struct Geo392 {
  static constexpr bool SAVE = false;     // training forward: also write activated gates + c_t (the *S geometries)
  static constexpr int H = 392;            // hidden size (unit-major stride of the saved activations)
  static constexpr int UPP = 49, BN = 208, PPG = 8, XKC = 26, HKC = 50, KS = 10, STAGES = 5;
  static constexpr int EPI_WARPS = 12, ACC = 256, NBUF = 2, EPI_REGS = 152, NC = 17;
  static constexpr int CLS = 2;             // cluster = one CTA pair
};
// H = 392 on groups of 7 pairs x 56 units (N = 224, no padding columns): 10 groups = 140 SMs, so the 9 tile pairs per
// direction of BASELINE config 2's time axis run 2-interleaved on 5 groups per direction instead of 3-interleaved on 3.
struct Geo392x7 {
  static constexpr bool SAVE = false;     // training forward: also write activated gates + c_t (the *S geometries)
  static constexpr int H = 392;
  static constexpr int UPP = 56, BN = 224, PPG = 7, XKC = 26, HKC = 50, KS = 10, STAGES = 4;
  static constexpr int EPI_WARPS = 16, ACC = 256, NBUF = 2, EPI_REGS = 104, NC = 14;
  static constexpr int CLS = 2;
};
// H = 392 on groups of 14 pairs x 28 units (N = 112): the small-batch geometry.  With few sequence tiles the layer is bound
// by the per-step dependency chain (epilogue -> publish -> h tile -> MMAs), and both the MUFU work and the MMA time of an
// item halve when twice as many CTAs share a tile; every CTA still pulls the whole x / h tile, so L2 traffic per item
// doubles - worthwhile only while few items are in flight (runtime_tc.fused_geometry).
struct Geo392x14 {
  static constexpr bool SAVE = false;     // training forward: also write activated gates + c_t (the *S geometries)
  static constexpr int H = 392;
  static constexpr int UPP = 28, BN = 112, PPG = 14, XKC = 26, HKC = 50, KS = 10, STAGES = 7;
  static constexpr int EPI_WARPS = 16, ACC = 128, NBUF = 4, EPI_REGS = 104, NC = 7;
  static constexpr int CLS = 2;
};
struct Geo768 {
  static constexpr bool SAVE = false;     // training forward: also write activated gates + c_t (the *S geometries)
  static constexpr int H = 768;
  static constexpr int UPP = 32, BN = 128, PPG = 24, XKC = 50, HKC = 96, KS = 12, STAGES = 3;
  static constexpr int EPI_WARPS = 16, ACC = 128, NBUF = 4, EPI_REGS = 104, NC = 8;
  // -DBSRNN_FUSED768_CLS=4: clusters of 2 CTA pairs, the two CTAs of a parity fetch half of each ring stage and
  // multicast it to both.  Measured (profiles/r02 call28): no gain per item (8 000 vs 7 670 cycles: the 72 KB ring's
  // round-trip latency paces the loads, not L2 throughput) and only 24 co-resident 4-CTA clusters = 2 groups instead
  // of 3, so the default stays one pair per cluster.
  static constexpr int CLS = BSRNN_FUSED768_CLS;
};
// small-batch geometry in clusters of 2 pairs: the two CTAs of a parity fetch half of every ring stage and multicast it to
// both (the 100 KB h tile of a step is on the dependency chain of a chain-bound launch).  BSRNN_FUSED14_CLS=4 selects it.
struct Geo392x14M : Geo392x14 { static constexpr int CLS = 4; };
struct Geo392x7S : Geo392x7 { static constexpr bool SAVE = true; };
struct Geo392x14S : Geo392x14 { static constexpr bool SAVE = true; };
struct Geo768S : Geo768 { static constexpr bool SAVE = true; };
template <class G>
struct Der {
  static constexpr int BH = G::BN / 2;                                  // B rows (gate columns) per CTA
  static constexpr int UKC = G::XKC + G::HKC;
  static constexpr uint32_t W_BYTES = UKC * BH * 16;
  static constexpr uint32_t STAGE = G::KS * 128 * 16;
  static constexpr int XST = (G::XKC + G::KS - 1) / G::KS;              // ring stages of the x tile (last one partial)
  static constexpr int XLAST = G::XKC - (XST - 1) * G::KS;
  static constexpr int HST = G::HKC / G::KS;
  static constexpr int THREADS = (4 + G::EPI_WARPS) * 32;
  static constexpr int NP = G::CLS / 2;                                 // pairs per cluster
  static constexpr int NBARS = 3 * G::STAGES + LNS + G::NBUF + 3;
  static constexpr size_t SMEM = W_BYTES + G::STAGES * STAGE + NBARS * 8 + 32;   // + TMEM address slot + ticket slot (16 B each)
  static_assert(G::HKC % G::KS == 0 && XLAST % 2 == 0 && G::KS % 2 == 0, "stages hold whole K = 16 MMAs");
  static_assert(SMEM <= 232448, "exceeds the 227 KB per-CTA shared memory limit");
  static_assert(W_BYTES % 64 == 0, "W half is fetched as 4 bulk copies");
  static_assert(G::NBUF * G::ACC <= 512 && (G::NBUF & (G::NBUF - 1)) == 0, "TMEM accumulators");
  static_assert(G::PPG % NP == 0 && (G::KS * 2048 / NP) % 16 == 0 && (XLAST * 2048 / NP) % 16 == 0, "multicast shares");
};
constexpr int U_MAX_GROUPS = 16;
constexpr int U_SYNC_WORDS = 32 + 32 * (U_MAX_GROUPS * LNS * 2);

struct FusedArgs {
  const __half* x;
  const __half* w;
  const __half* zero_tile;   // HKC*128*8 zeros (stands in for the h tile of a missing odd tile)
  __half *y0, *y1;           // per direction: block of (step p, tile j) at y_d + (p*seq_tiles + j) * y_stride
  long y_stride;             // halves
  int R, steps, seq_tiles;
  int gpd;                   // work groups per direction (each = up to `slots` consecutive tile PAIRS)
  unsigned* sync;            // [0] ticket counter, [32 + 32*((3*group + slot)*2 + parity)] h_ready counters
  long long* probe;          // debug (-DBSRNN_FUSED_PROBE): per-role wait / busy cycle totals of pair 0, [16*e + i]
  // training forward (SAVE instantiations): activated gates [tile = step*seq_tiles + j][dir][unit][128 rows][4] fp16 and c_t
  // per direction [tile][unit][128 rows] f32 (unit-major scratch; saved_transpose_kernel makes them row-major for BPTT)
  __half* sv_gates;
  float* sv_c0;
  float* sv_c1;
};
// saved activations, UNIT-major per (tile, direction): gates [tile][dir][unit][128 rows][4] fp16, c [tile][unit][128 rows] f32
constexpr int SVG = 128 * 4, SVC = 128;

#ifdef BSRNN_FUSED_PROBE
#define FP_DECL(cond) const bool prb_ = a.probe && ticket == 0 && (cond); long long pt_ = prb_ ? clock64() : 0
#define FP_MARK(v)                     \
  do {                                 \
    if (prb_) {                        \
      const long long n_ = clock64();  \
      (v) += n_ - pt_;                 \
      pt_ = n_;                        \
    }                                  \
  } while (0)
#else
#define FP_DECL(cond) constexpr bool prb_ = false
#define FP_MARK(v) do { (void)(v); } while (0)
#endif

struct PGroup {
  int d, j0, nact;           // direction, first tile pair, tile pairs
};
__device__ __forceinline__ PGroup pgroup_of(const FusedArgs& a, int g) {
  const int ptiles = (a.seq_tiles + 1) >> 1;
  PGroup r;
  r.d = g / a.gpd;
  const int gi = g - r.d * a.gpd;
  r.j0 = (int)(((long)gi * ptiles) / a.gpd);
  r.nact = (int)(((long)(gi + 1) * ptiles) / a.gpd) - r.j0;
  return r;
}
__device__ __forceinline__ unsigned* uflag_of(const FusedArgs& a, int cid, int k, int e) {
  return a.sync + 32 + 32 * ((3 * cid + k) * 2 + e);
}

// 4 hidden units from 16 accumulator columns (i, f, g, o interleaved)
template <int CH, int NC, int NH>
__device__ __forceinline__ void epif_chunk(const uint32_t (&acc)[16], float (&c)[NC], float (&h)[NH]) {
#pragma unroll
  for (int u = 0; u < 4; ++u)
    gate_update(__uint_as_float(acc[4 * u]), __uint_as_float(acc[4 * u + 1]), __uint_as_float(acc[4 * u + 2]),
                __uint_as_float(acc[4 * u + 3]), c[4 * CH + u], h[4 * CH + u]);
}
// H = 392: one item for one thread (row r, third T of the pair's 49 units).  Unit j of third T is h column
// 49Q + 16T + j -> k-core 6Q + 2T + (Q+j)/8, slot (Q+j)%8 of the y tile (store pattern depends on Q only).
template <int Q>
__device__ __forceinline__ void epif_item392(uint32_t t_col, bool last_third, uint32_t t_col48, __half* ycore, float (&c)[17],
                                             bool st) {
  constexpr size_t CORE = 128 * 8;
  float h[16];
  uint32_t accA[16], accB[16];
  tmem_ld_x16(t_col, accA);
  tmem_ld_wait();
  tmem_ld_x16(t_col + 16, accB);
  tmem_ld_pin16(accA);
  epif_chunk<0>(accA, c, h);
  tmem_ld_wait();
  tmem_ld_x16(t_col + 32, accA);
  tmem_ld_pin16(accB);
  epif_chunk<1>(accB, c, h);
  if (st) {
    if (Q == 0) store_full<0>(ycore, h);
    else store_partial<Q, 8, 0>(ycore, h);              // core A: slots Q..7 <- j = 0..7-Q
  }
  tmem_ld_wait();
  tmem_ld_x16(t_col + 48, accB);
  tmem_ld_pin16(accA);
  epif_chunk<2>(accA, c, h);
  uint32_t a4[4] = {0u, 0u, 0u, 0u};
  tmem_ld_wait();
  if (last_third) tmem_ld_x4(t_col48, a4);
  tmem_ld_pin16(accB);
  epif_chunk<3>(accB, c, h);
  if (st) {
    store_full<8 - Q>(ycore + CORE, h);                 // core B: j = 8-Q .. 15-Q
    if (Q > 0) store_partial<0, Q, 16 - Q>(ycore + 2 * CORE, h);   // core C: slots 0..Q-1 <- j = 16-Q .. 15
  }
  if (last_third) {                                     // local unit 48 -> slot Q of core C
    tmem_ld_wait();
    asm volatile("" : "+r"(a4[0]), "+r"(a4[1]), "+r"(a4[2]), "+r"(a4[3]));
    float h48;
    gate_update(__uint_as_float(a4[0]), __uint_as_float(a4[1]), __uint_as_float(a4[2]), __uint_as_float(a4[3]), c[16], h48);
    if (st) ycore[2 * CORE + Q] = __float2half_rn(h48);
  }
}
// H = 392, 7 pairs: thread = (row r, quarter T of the pair's 56 units): 14 units at h columns 56q + 14T + j, i.e. position
// p = 14T + j of the pair's 7 k-cores (core p/8, slot p%8): the store pattern depends on T only.
// one accumulator chunk of 4 units; SAVE: activated gates / c_t of unit U0 + u go to sg + 4*(U0+u) / sc + U0 + u
template <int CH, int NC, int NH, bool SAVE>
__device__ __forceinline__ void epif_chunk_sv(const uint32_t (&acc)[16], float (&c)[NC], float (&h)[NH], __half* sg, float* sc, bool st) {
#pragma unroll
  for (int u = 0; u < 4; ++u) {
    if (SAVE && st)
      gate_update_save(__uint_as_float(acc[4 * u]), __uint_as_float(acc[4 * u + 1]), __uint_as_float(acc[4 * u + 2]),
                       __uint_as_float(acc[4 * u + 3]), c[4 * CH + u], h[4 * CH + u], sg + SVG * (4 * CH + u), sc + SVC * (4 * CH + u));
    else
      gate_update(__uint_as_float(acc[4 * u]), __uint_as_float(acc[4 * u + 1]), __uint_as_float(acc[4 * u + 2]),
                  __uint_as_float(acc[4 * u + 3]), c[4 * CH + u], h[4 * CH + u]);
  }
}
template <bool SAVE>
__device__ __forceinline__ void gate_update_sv(float pi, float pf, float pg, float po, float& c, float& h, __half* sg, float* sc, bool st) {
  if (SAVE && st) gate_update_save(pi, pf, pg, po, c, h, sg, sc);
  else gate_update(pi, pf, pg, po, c, h);
}
template <int T, bool SAVE = false>
__device__ __forceinline__ void epif_item392x7(uint32_t t_col, __half* ycore, float (&c)[14], bool st, __half* sg = nullptr,
                                               float* sc = nullptr) {
  constexpr size_t CORE = 128 * 8;
  float h[16];
  uint32_t accA[16], accB[16];
  tmem_ld_x16(t_col, accA);
  tmem_ld_wait();
  tmem_ld_x16(t_col + 16, accB);
  tmem_ld_pin16(accA);
  epif_chunk_sv<0, 14, 16, SAVE>(accA, c, h, sg, sc, st);
  tmem_ld_wait();
  tmem_ld_x16(t_col + 32, accA);
  tmem_ld_pin16(accB);
  epif_chunk_sv<1, 14, 16, SAVE>(accB, c, h, sg, sc, st);
  if (st) {
    if (T == 0) store_full<0>(ycore, h);                                   // p 0..7   -> core 0
    if (T == 1) store_partial<6, 8, 0>(ycore + CORE, h);                   // p 14,15  -> core 1 slots 6,7
    if (T == 2) store_partial<4, 8, 0>(ycore + 3 * CORE, h);               // p 28..31 -> core 3 slots 4..7
    if (T == 3) store_partial<2, 8, 0>(ycore + 5 * CORE, h);               // p 42..47 -> core 5 slots 2..7
  }
  uint32_t a8[8];
  tmem_ld_wait();
  tmem_ld_x8(t_col + 48, a8);
  tmem_ld_pin16(accA);
  epif_chunk_sv<2, 14, 16, SAVE>(accA, c, h, sg, sc, st);
  tmem_ld_wait();
  asm volatile("" : "+r"(a8[0]), "+r"(a8[1]), "+r"(a8[2]), "+r"(a8[3]), "+r"(a8[4]), "+r"(a8[5]), "+r"(a8[6]), "+r"(a8[7]));
#pragma unroll
  for (int u = 0; u < 2; ++u)
    gate_update_sv<SAVE>(__uint_as_float(a8[4 * u]), __uint_as_float(a8[4 * u + 1]), __uint_as_float(a8[4 * u + 2]),
                         __uint_as_float(a8[4 * u + 3]), c[12 + u], h[12 + u], sg + SVG * (12 + u), sc + SVC * (12 + u), st);
  if (st) {
    if (T == 0) store_partial<0, 6, 8>(ycore + CORE, h);                   // p 8..13  -> core 1 slots 0..5
    if (T == 1) { store_full<2>(ycore + 2 * CORE, h); store_partial<0, 4, 10>(ycore + 3 * CORE, h); }   // p 16..23, 24..27
    if (T == 2) { store_full<4>(ycore + 4 * CORE, h); store_partial<0, 2, 12>(ycore + 5 * CORE, h); }   // p 32..39, 40,41
    if (T == 3) store_full<6>(ycore + 6 * CORE, h);                        // p 48..55 -> core 6
  }
}
// H = 392, 14 pairs: thread = (row r, quarter T of the pair's 28 units): 7 units at h columns 28q + 7T + j.  With
// QP = q & 1 the pair's columns start 4*QP slots into k-core (28q - 4*QP)/8; position p = 4*QP + 7T + j -> core p/8, slot p%8.
template <int QP, int T, bool SAVE = false>
__device__ __forceinline__ void epif_item392x14(uint32_t t_col, __half* ycore, float (&c)[7], bool st, __half* sg = nullptr,
                                                float* sc = nullptr) {
  constexpr size_t CORE = 128 * 8;
  constexpr int P0 = 4 * QP + 7 * T;                 // first position of this thread's units
  constexpr int C0 = P0 / 8, S0 = P0 % 8;            // first core / slot
  constexpr int N0 = (8 - S0) < 7 ? (8 - S0) : 7;    // units that fall into the first core
  float h[16];
  uint32_t acc[16], a8[8], a4[4];
  tmem_ld_x16(t_col, acc);
  tmem_ld_x8(t_col + 16, a8);
  tmem_ld_x4(t_col + 24, a4);
  tmem_ld_wait();
  tmem_ld_pin16(acc);
  asm volatile("" : "+r"(a8[0]), "+r"(a8[1]), "+r"(a8[2]), "+r"(a8[3]), "+r"(a8[4]), "+r"(a8[5]), "+r"(a8[6]), "+r"(a8[7]));
  asm volatile("" : "+r"(a4[0]), "+r"(a4[1]), "+r"(a4[2]), "+r"(a4[3]));
#pragma unroll
  for (int u = 0; u < 4; ++u)
    gate_update_sv<SAVE>(__uint_as_float(acc[4 * u]), __uint_as_float(acc[4 * u + 1]), __uint_as_float(acc[4 * u + 2]),
                         __uint_as_float(acc[4 * u + 3]), c[u], h[u], sg + SVG * u, sc + SVC * u, st);
#pragma unroll
  for (int u = 0; u < 2; ++u)
    gate_update_sv<SAVE>(__uint_as_float(a8[4 * u]), __uint_as_float(a8[4 * u + 1]), __uint_as_float(a8[4 * u + 2]),
                         __uint_as_float(a8[4 * u + 3]), c[4 + u], h[4 + u], sg + SVG * (4 + u), sc + SVC * (4 + u), st);
  gate_update_sv<SAVE>(__uint_as_float(a4[0]), __uint_as_float(a4[1]), __uint_as_float(a4[2]), __uint_as_float(a4[3]), c[6], h[6],
                       sg + SVG * 6, sc + SVC * 6, st);
  if (st) {
    store_partial<S0, S0 + N0, 0>(ycore + C0 * CORE, h);
    if constexpr (N0 < 7) store_partial<0, 7 - N0, N0>(ycore + (C0 + 1) * CORE, h);
  }
}
// H = 768: thread = (row r, quarter T of the pair's 32 units): 8 units = 32 accumulator columns = one 16-byte row of
// k-core 4q + T of the y tile.  SAVE: the activated gates / c_t of unit u0 + u (u0 = 32q + 8T) go to sg + 4*u / sc + u.
template <bool SAVE = false>
__device__ __forceinline__ void epif_item768(uint32_t t_col, __half* ycore, float (&c)[8], bool st, __half* sg = nullptr,
                                             float* sc = nullptr) {
  float h[8];
  uint32_t accA[16], accB[16];
  tmem_ld_x16(t_col, accA);
  tmem_ld_wait();
  tmem_ld_x16(t_col + 16, accB);
  tmem_ld_pin16(accA);
  epif_chunk_sv<0, 8, 8, SAVE>(accA, c, h, sg, sc, st);
  tmem_ld_wait();
  tmem_ld_pin16(accB);
  epif_chunk_sv<1, 8, 8, SAVE>(accB, c, h, sg, sc, st);
  if (st)
    *reinterpret_cast<uint4*>(ycore) = make_uint4(pack_h2(h[0], h[1]), pack_h2(h[2], h[3]), pack_h2(h[4], h[5]), pack_h2(h[6], h[7]));
}

template <class G, int Q>
__device__ __forceinline__ void epiloguef_role(const FusedArgs& a, uint32_t tmem_base, int T, int quad, int lane, int cid,
                                               int ncl, int e, int q, uint32_t leader, uint64_t* acc_full, uint64_t* acc_empty,
                                               uint64_t* w_free, uint32_t ticket) {
  // G7: the template parameter Q carries the quarter T; G14: Q = 4 * (q & 1) + T
  constexpr bool G392 = G::UPP == 49, G7 = G::UPP == 56, G14 = G::UPP == 28;
  const int r = quad * 32 + lane;
  long long w_acc = 0, w_busy = 0, w_arr = 0;
  FP_DECL(T == 0 && quad == 0 && lane == 0);
  const bool last_third = T == 2;
  const uint32_t t_lane = tmem_base + ((uint32_t)(quad * 32) << 16) + (G392 ? 64 : G7 ? 56 : G14 ? 28 : 32) * T;
  const uint32_t t_lane48 = tmem_base + ((uint32_t)(quad * 32) << 16) + 192;
  const int ngroups = 2 * a.gpd;
  // this thread's first k-core row inside a y tile
  const size_t y_off = (size_t)(G392 ? 6 * Q + 2 * T : G7 ? 7 * q : G14 ? (28 * q - 4 * (q & 1)) / 8 : 4 * q + T) * (128 * 8) + (size_t)r * 8;
  uint32_t it0 = 0, nfull = 0;
  float c0[G::NC], c1[G::NC], c2[G::NC];
  for (int g = cid; g < ngroups; g += ncl) {
    const PGroup GR = pgroup_of(a, g);
#pragma unroll
    for (int i = 0; i < G::NC; ++i) c0[i] = c1[i] = c2[i] = 0.f;
    for (int s = 0; s < a.steps; ++s) {
      const int p = GR.d == 0 ? s : a.steps - 1 - s;
#pragma unroll
      for (int k = 0; k < LNS; ++k) {
        if (k < GR.nact) {
          const int j = 2 * (GR.j0 + k) + e;
          const bool valid = j < a.seq_tiles;                  // odd tile count: the last odd CTA computes and drops
          const size_t tile = (size_t)p * a.seq_tiles + (valid ? j : 0);
          __half* ycore = (GR.d == 0 ? a.y0 : a.y1) + tile * a.y_stride + y_off;
          const uint32_t it = it0 + (uint32_t)(s * GR.nact + k);
          const uint32_t buf = it & (G::NBUF - 1);
          FP_MARK(w_busy);
          mbar_wait(acc_full + k, (nfull >> k) & 1);
          nfull ^= 1u << k;
          tc_fence_after();
          FP_MARK(w_acc);
          if constexpr (G392) {
            if (k == 0) epif_item392<Q>(t_lane + buf * G::ACC, last_third, t_lane48 + buf * G::ACC, ycore, c0, valid);
            else if (k == 1) epif_item392<Q>(t_lane + buf * G::ACC, last_third, t_lane48 + buf * G::ACC, ycore, c1, valid);
            else epif_item392<Q>(t_lane + buf * G::ACC, last_third, t_lane48 + buf * G::ACC, ycore, c2, valid);
          } else if constexpr (G7) {
            __half* sg = nullptr; float* sc = nullptr;
            if constexpr (G::SAVE) {
              const int u0 = 56 * q + 14 * T;
              sg = a.sv_gates + (((tile * 2 + GR.d) * G::H + u0) * 128 + (size_t)r) * 4;
              sc = (GR.d == 0 ? a.sv_c0 : a.sv_c1) + (tile * G::H + u0) * 128 + (size_t)r;
            }
            if (k == 0) epif_item392x7<Q, G::SAVE>(t_lane + buf * G::ACC, ycore, c0, valid, sg, sc);
            else if (k == 1) epif_item392x7<Q, G::SAVE>(t_lane + buf * G::ACC, ycore, c1, valid, sg, sc);
            else epif_item392x7<Q, G::SAVE>(t_lane + buf * G::ACC, ycore, c2, valid, sg, sc);
          } else if constexpr (G14) {
            __half* sg = nullptr; float* sc = nullptr;
            if constexpr (G::SAVE) {
              const int u0 = 28 * q + 7 * T;
              sg = a.sv_gates + (((tile * 2 + GR.d) * G::H + u0) * 128 + (size_t)r) * 4;
              sc = (GR.d == 0 ? a.sv_c0 : a.sv_c1) + (tile * G::H + u0) * 128 + (size_t)r;
            }
            if (k == 0) epif_item392x14<Q / 4, Q % 4, G::SAVE>(t_lane + buf * G::ACC, ycore, c0, valid, sg, sc);
            else if (k == 1) epif_item392x14<Q / 4, Q % 4, G::SAVE>(t_lane + buf * G::ACC, ycore, c1, valid, sg, sc);
            else epif_item392x14<Q / 4, Q % 4, G::SAVE>(t_lane + buf * G::ACC, ycore, c2, valid, sg, sc);
          } else {
            __half* sg = nullptr; float* sc = nullptr;
            if constexpr (G::SAVE) {
              const int u0 = 32 * q + 8 * T;
              sg = a.sv_gates + (((tile * 2 + GR.d) * G::H + u0) * 128 + (size_t)r) * 4;
              sc = (GR.d == 0 ? a.sv_c0 : a.sv_c1) + (tile * G::H + u0) * 128 + (size_t)r;
            }
            if (k == 0) epif_item768<G::SAVE>(t_lane + buf * G::ACC, ycore, c0, valid, sg, sc);
            else if (k == 1) epif_item768<G::SAVE>(t_lane + buf * G::ACC, ycore, c1, valid, sg, sc);
            else epif_item768<G::SAVE>(t_lane + buf * G::ACC, ycore, c2, valid, sg, sc);
          }
          tc_fence_before();
          __syncwarp();
          FP_MARK(w_busy);
          // the pair's MMA issuer counts both CTAs' warps.  Relaxed remote arrive: the accumulator reads were completed
          // by tcgen05.wait::ld; a release at cluster scope would make every warp drain its h stores first (~1 000 cycles)
          if (lane == 0) {
            if (e == 0) mbar_arrive(acc_empty + buf);
            else mbar_arrive_cluster_relaxed(acc_empty + buf, leader);
          }
          FP_MARK(w_arr);
          // h_t slice of this warp is stored: tell the publisher (non-blocking)
          if (s + 1 < a.steps) asm volatile("bar.arrive %0, %1;" ::"r"(1 + k), "n"(G::EPI_WARPS * 32 + 32) : "memory");
        }
      }
    }
    const int gn = g + ncl;                          // next work group of this hardware group switches direction?
    if (gn < ngroups && gn / a.gpd != GR.d) {
      __syncwarp();
      if (lane == 0) mbar_arrive(w_free);            // this warp consumed the last accumulator: W may go
    }
    it0 += (uint32_t)(a.steps * GR.nact);
  }
  FP_MARK(w_busy);
  if (prb_) { a.probe[16 * e + 12] = w_acc; a.probe[16 * e + 13] = w_busy; a.probe[16 * e + 14] = w_arr; }
}

template <class G>
__global__ void __launch_bounds__(Der<G>::THREADS, 1) lstm_fused_kernel(const FusedArgs a) {
  using D = Der<G>;
  extern __shared__ __align__(128) uint8_t smem[];
  uint8_t* sW = smem;
  uint8_t* sA = smem + D::W_BYTES;
  uint64_t* bars = reinterpret_cast<uint64_t*>(sA + G::STAGES * D::STAGE);
  uint64_t* full = bars;                       // [STAGES] this CTA's ring stage landed
  uint64_t* empty = full + G::STAGES;          // [STAGES] MMAs that read the stage retired (multicast commit)
  uint64_t* pfull = empty + G::STAGES;         // [STAGES] leader only: the odd CTA's stage landed (relayed)
  uint64_t* acc_full = pfull + G::STAGES;      // [LNS]
  uint64_t* acc_empty = acc_full + LNS;        // [NBUF] leader only: the epilogue warps of both CTAs
  uint64_t* w_full = acc_empty + G::NBUF;
  uint64_t* w_free = w_full + 1;
  uint64_t* pw_full = w_free + 1;              // leader only: the odd CTA's W half landed (relayed)
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(pw_full + 1);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t crank = cluster_ctarank();
  const int e = (int)(crank & 1u);             // tile parity served by this CTA; the even CTA of a pair is its leader
  const uint32_t pc = crank >> 1;              // pair within the cluster
  const uint32_t leader = crank & ~1u;

  if (threadIdx.x == 0) {
    for (int i = 0; i < G::STAGES; ++i) { mbar_init(full + i, 1); mbar_init(empty + i, D::NP); mbar_init(pfull + i, 1); }
    for (int i = 0; i < LNS; ++i) mbar_init(acc_full + i, 1);
    for (int i = 0; i < G::NBUF; ++i) mbar_init(acc_empty + i, 2 * G::EPI_WARPS);
    mbar_init(w_full, 1);
    mbar_init(w_free, G::EPI_WARPS);
    mbar_init(pw_full, 1);
    fence_barrier_init();
    // the cluster's rank within the launch by arrival order (its own 16-byte slot: racecheck treats the TMEM allocator's
    // result write as touching the words next to tmem_slot[0])
    if (crank == 0) tmem_slot[4] = atomicAdd(a.sync, 1u);
  }
  if (warp == 2) tmem_alloc2(tmem_slot, 512);
  tc_fence_before();
  __syncthreads();
  cluster_sync();                       // both CTAs run and their barriers are initialised
  if (crank != 0 && threadIdx.x == 0) { // the other CTAs read the cluster's ticket from CTA 0's shared memory
    uint32_t remote, v;
    asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(remote) : "r"(smem_u32(tmem_slot + 4)), "r"(0));
    asm volatile("ld.shared::cluster.u32 %0, [%1];" : "=r"(v) : "r"(remote) : "memory");
    tmem_slot[4] = v;
  }
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = tmem_slot[0];
  const uint32_t ticket = tmem_slot[4] * D::NP + pc;     // this pair's rank within the launch
  const uint32_t q = ticket % G::PPG;
  const int cid = (int)(ticket / G::PPG);
  const int ncl = (int)(gridDim.x / (2 * G::PPG));

  const int ngroups = 2 * a.gpd;
  const size_t x_tile = (size_t)G::XKC * 128 * 8;      // halves per (step, tile) of x

  if (warp == 0) {
    // ------------------------------------------------------------------ producer: W half + this CTA's x / h tiles
    asm volatile("setmaxnreg.dec.sync.aligned.u32 40;");
    uint32_t stage = 0, phase = 0, wfphase = 0;
    uint32_t npub0 = 0u, npub1 = 0u, npub2 = 0u;       // h tiles of slot k published so far by each CTA of this parity
    int cur_dir = -1;
    uint16_t mc_mask = 0;                              // the CTAs of my parity in this cluster
    for (int i = 0; i < D::NP; ++i) mc_mask |= (uint16_t)(1u << (2 * i + e));
    (void)mc_mask;
    long long w_h = 0, w_e = 0, w_o = 0;
    FP_DECL(lane == 0);
    for (int g = cid; g < ngroups; g += ncl) {
      const PGroup GR = pgroup_of(a, g);
      if (GR.d != cur_dir) {
        if (cur_dir >= 0) {
          mbar_wait(w_free, wfphase);
          wfphase ^= 1;
        }
        if (elect_one()) {
          mbar_expect_tx(w_full, D::W_BYTES);
          const uint8_t* src = reinterpret_cast<const uint8_t*>(a.w) + (((size_t)GR.d * G::PPG + q) * 2 + e) * D::W_BYTES;
          for (uint32_t off = 0; off < D::W_BYTES; off += D::W_BYTES / 4) bulk_g2s(sW + off, src + off, D::W_BYTES / 4, w_full);
        }
        __syncwarp();
        cur_dir = GR.d;
      }
      for (int s = 0; s < a.steps; ++s) {
        const int p = GR.d == 0 ? s : a.steps - 1 - s;
        const int p_prev = GR.d == 0 ? s - 1 : a.steps - s;        // position whose h feeds this step
        for (int k = 0; k < GR.nact; ++k) {
          const int j = 2 * (GR.j0 + k) + e;
          const bool valid = j < a.seq_tiles;
          const uint8_t* xsrc = reinterpret_cast<const uint8_t*>(a.x + ((size_t)p * a.seq_tiles + (valid ? j : 0)) * x_tile);
          // x comes from DRAM (the operand of a whole BLSTM call is far larger than L2): one pair per group and parity
          // pulls the slot's tile of the NEXT step into L2, so the ring's copies are L2 hits
          if (q == 0 && s + 1 < a.steps && elect_one())
            bulk_prefetch_l2(xsrc + (GR.d == 0 ? 1 : -1) * (long)a.seq_tiles * (long)(x_tile * 2), (uint32_t)(x_tile * 2));
#pragma unroll
          for (int xs = 0; xs < D::XST; ++xs) {
            const uint32_t bytes = (xs == D::XST - 1 ? D::XLAST : G::KS) * 2048;
            FP_MARK(w_o);
            mbar_wait(empty + stage, phase ^ 1);
            FP_MARK(w_e);
            if (elect_one()) {
              mbar_expect_tx(full + stage, bytes);
              if constexpr (D::NP == 1) {
                bulk_g2s(sA + stage * D::STAGE, xsrc + (size_t)xs * D::STAGE, bytes, full + stage);
              } else {             // my share of the stage -> the same ring slot of every CTA of my parity in the cluster
                const uint32_t sh = bytes / D::NP;
                bulk_g2s_multicast(sA + stage * D::STAGE + pc * sh, xsrc + (size_t)xs * D::STAGE + pc * sh, sh, full + stage, mc_mask);
              }
            }
            __syncwarp();
            if (++stage == G::STAGES) { stage = 0; phase ^= 1; }
          }
          if (s > 0) {
            const uint8_t* src = reinterpret_cast<const uint8_t*>(a.zero_tile);
            if (valid) {
              // all PPG CTAs of this parity have released their slice of h_{t-1} (gpu-scope acquire on the counter)
              uint32_t& np = k == 0 ? npub0 : (k == 1 ? npub1 : npub2);
              const uint32_t want = G::PPG * (++np);
              const unsigned* fl = uflag_of(a, cid, k, e);
              uint32_t spins = 0;
              FP_MARK(w_o);
              while ((int32_t)(ld_acquire_gpu(fl) - want) < 0) {
                if (++spins > (1u << 22)) { __trap(); }
              }
              FP_MARK(w_h);
              src = reinterpret_cast<const uint8_t*>((GR.d == 0 ? a.y0 : a.y1) + ((size_t)p_prev * a.seq_tiles + j) * a.y_stride);
            }
#pragma unroll 1
            for (int ks = 0; ks < D::HST; ++ks) {
              FP_MARK(w_o);
              mbar_wait(empty + stage, phase ^ 1);
              FP_MARK(w_e);
              if (elect_one()) {
                if (ks == 0) fence_proxy_async_global();      // peers' generic-proxy h stores -> this thread's async-proxy reads
                mbar_expect_tx(full + stage, D::STAGE);
                if constexpr (D::NP == 1) {
                  bulk_g2s(sA + stage * D::STAGE, src + (size_t)ks * D::STAGE, D::STAGE, full + stage);
                } else {
                  constexpr uint32_t sh = D::STAGE / D::NP;
                  bulk_g2s_multicast(sA + stage * D::STAGE + pc * sh, src + (size_t)ks * D::STAGE + pc * sh, sh, full + stage, mc_mask);
                }
              }
              __syncwarp();
              if (++stage == G::STAGES) { stage = 0; phase ^= 1; }
            }
          }
        }
      }
    }
    FP_MARK(w_o);
    if (prb_) { a.probe[16 * e + 0] = w_h; a.probe[16 * e + 1] = w_e; a.probe[16 * e + 2] = w_o; }
  } else if (warp == 1) {
    asm volatile("setmaxnreg.dec.sync.aligned.u32 40;");
    if (e == 0) {
      // ---------------------------------------------------------------- MMA issuer (leader CTA of the pair)
      const uint32_t idesc = idesc_f16_f32(256, G::BN);
      uint32_t stage = 0, phase = 0, it = 0, wphase = 0;
      int cur_dir = -1;
      // descriptors advance by adding to the 14-bit (address >> 4) field: shared memory is < 256 KB, no carry out
      const uint64_t da0 = smem_desc_kb8(smem_u32(sA), 2048, 128);
      const uint64_t db0 = smem_desc_kb8(smem_u32(sW), D::BH * 16, 128);
      const uint16_t all_mask = (uint16_t)((1u << G::CLS) - 1), pair_mask = (uint16_t)(3u << (2 * pc));
      long long w_a = 0, w_f = 0, w_p = 0, w_o = 0;
      FP_DECL(lane == 0);
      for (int g = cid; g < ngroups; g += ncl) {
        const PGroup GR = pgroup_of(a, g);
        if (GR.d != cur_dir) {
          mbar_wait(w_full, wphase);
          mbar_wait(pw_full, wphase);
          wphase ^= 1;
          cur_dir = GR.d;
        }
        for (int s = 0; s < a.steps; ++s) {
          for (int k = 0; k < GR.nact; ++k, ++it) {
            const uint32_t buf = it & (G::NBUF - 1);
            FP_MARK(w_o);
            mbar_wait(acc_empty + buf, ((it / G::NBUF) & 1) ^ 1);
            FP_MARK(w_a);
            tc_fence_after();
            const uint32_t d_tmem = tmem_base + buf * G::ACC;
#pragma unroll
            for (int xs = 0; xs < D::XST; ++xs) {              // x_t * W_ih^T: k-cores [0, XKC)
              FP_MARK(w_o);
              mbar_wait(full + stage, phase);
              FP_MARK(w_f);
              mbar_wait(pfull + stage, phase);
              FP_MARK(w_p);
              tc_fence_after();
              if (elect_one()) {
                const uint64_t da = da0 + (uint64_t)(stage * (D::STAGE >> 4));
                const uint64_t db = db0 + (uint64_t)(xs * G::KS * ((D::BH * 16) >> 4));
#pragma unroll
                for (int jk = 0; jk < (xs == D::XST - 1 ? D::XLAST : G::KS) / 2; ++jk)
                  mma_f16_ss_2cta(d_tmem, da + (uint64_t)(jk * ((2 * 2048) >> 4)), db + (uint64_t)(jk * ((2 * D::BH * 16) >> 4)),
                                  idesc, (xs | jk) != 0);
                mma_commit2_multicast(empty + stage, all_mask);
                if (s == 0 && xs == D::XST - 1) mma_commit2_multicast(acc_full + k, pair_mask);
              }
              __syncwarp();
              if (++stage == G::STAGES) { stage = 0; phase ^= 1; }
            }
            if (s > 0) {
#pragma unroll
              for (int ks = 0; ks < D::HST; ++ks) {            // h_{t-1} * W_hh^T: k-cores [XKC, XKC + HKC)
                FP_MARK(w_o);
                mbar_wait(full + stage, phase);
                FP_MARK(w_f);
                mbar_wait(pfull + stage, phase);
                FP_MARK(w_p);
                tc_fence_after();
                if (elect_one()) {
                  const uint64_t da = da0 + (uint64_t)(stage * (D::STAGE >> 4));
                  const uint64_t db = db0 + (uint64_t)((G::XKC + ks * G::KS) * ((D::BH * 16) >> 4));
#pragma unroll
                  for (int jk = 0; jk < G::KS / 2; ++jk)
                    mma_f16_ss_2cta(d_tmem, da + (uint64_t)(jk * ((2 * 2048) >> 4)), db + (uint64_t)(jk * ((2 * D::BH * 16) >> 4)),
                                    idesc, 1u);
                  mma_commit2_multicast(empty + stage, all_mask);
                  if (ks == D::HST - 1) mma_commit2_multicast(acc_full + k, pair_mask);
                }
                __syncwarp();
                if (++stage == G::STAGES) { stage = 0; phase ^= 1; }
              }
            }
          }
        }
      }
      FP_MARK(w_o);
      if (prb_) { a.probe[4] = w_a; a.probe[5] = w_f; a.probe[6] = w_p; a.probe[7] = w_o; }
    } else {
      // ---------------------------------------------------------------- relay (odd CTA): my stages -> leader's pfull
      uint32_t stage = 0, phase = 0, wphase = 0;
      int cur_dir = -1;
      for (int g = cid; g < ngroups; g += ncl) {
        const PGroup GR = pgroup_of(a, g);
        if (GR.d != cur_dir) {
          mbar_wait(w_full, wphase);
          wphase ^= 1;
          if (lane == 0) mbar_arrive_cluster_relaxed(pw_full, leader);
          __syncwarp();
          cur_dir = GR.d;
        }
        const int nfills = GR.nact * (D::XST + (a.steps - 1) * (D::XST + D::HST));
        for (int i = 0; i < nfills; ++i) {
          mbar_wait(full + stage, phase);
          if (lane == 0) mbar_arrive_cluster_relaxed(pfull + stage, leader);   // no fence: a release.cluster per stage paces the ring
          __syncwarp();
          if (++stage == G::STAGES) { stage = 0; phase ^= 1; }
        }
      }
    }
  } else if (warp == 2) {
    // ------------------------------------------------------------------ publisher
    asm volatile("setmaxnreg.dec.sync.aligned.u32 40;");
    for (int g = cid; g < ngroups; g += ncl) {
      const PGroup GR = pgroup_of(a, g);
      for (int s = 0; s + 1 < a.steps; ++s) {
        for (int k = 0; k < GR.nact; ++k) {
          // completes once all epilogue warps have stored their h_t slices of slot k
          asm volatile("bar.sync %0, %1;" ::"r"(1 + k), "n"(G::EPI_WARPS * 32 + 32) : "memory");
          if (lane == 0 && 2 * (GR.j0 + k) + e < a.seq_tiles) {
            fence_proxy_async_global();
            red_release_gpu_add(uflag_of(a, cid, k, e), 1u);   // release: the CTA's h stores (ordered by the bar.sync) first
          }
          __syncwarp();
        }
      }
    }
  } else if (warp == 3) {
    asm volatile("setmaxnreg.dec.sync.aligned.u32 40;");      // idle 4th warp of warpgroup 0
  } else {
    // ------------------------------------------------------------------ epilogue: every warp on every item
    asm volatile("setmaxnreg.inc.sync.aligned.u32 %0;" ::"n"(G::EPI_REGS));
    const int T = (warp - 4) >> 2, quad = warp & 3;
    if constexpr (G::UPP == 49) {
#define BSRNN_EPIF_CASE(QQ) \
  case QQ: epiloguef_role<G, QQ>(a, tmem_base, T, quad, lane, cid, ncl, e, QQ, leader, acc_full, acc_empty, w_free, ticket); break;
      switch (q) {
        BSRNN_EPIF_CASE(0) BSRNN_EPIF_CASE(1) BSRNN_EPIF_CASE(2) BSRNN_EPIF_CASE(3)
        BSRNN_EPIF_CASE(4) BSRNN_EPIF_CASE(5) BSRNN_EPIF_CASE(6) BSRNN_EPIF_CASE(7)
      }
#undef BSRNN_EPIF_CASE
    } else if constexpr (G::UPP == 56) {
#define BSRNN_EPIF_CASE(TT) \
  case TT: epiloguef_role<G, TT>(a, tmem_base, TT, quad, lane, cid, ncl, e, (int)q, leader, acc_full, acc_empty, w_free, ticket); break;
      switch (T) { BSRNN_EPIF_CASE(0) BSRNN_EPIF_CASE(1) BSRNN_EPIF_CASE(2) BSRNN_EPIF_CASE(3) }
#undef BSRNN_EPIF_CASE
    } else if constexpr (G::UPP == 28) {
#define BSRNN_EPIF_CASE(QT) \
  case QT: epiloguef_role<G, QT>(a, tmem_base, QT % 4, quad, lane, cid, ncl, e, (int)q, leader, acc_full, acc_empty, w_free, ticket); break;
      switch (4 * (int)(q & 1u) + T) {
        BSRNN_EPIF_CASE(0) BSRNN_EPIF_CASE(1) BSRNN_EPIF_CASE(2) BSRNN_EPIF_CASE(3)
        BSRNN_EPIF_CASE(4) BSRNN_EPIF_CASE(5) BSRNN_EPIF_CASE(6) BSRNN_EPIF_CASE(7)
      }
#undef BSRNN_EPIF_CASE
    } else {
      epiloguef_role<G, 0>(a, tmem_base, T, quad, lane, cid, ncl, e, (int)q, leader, acc_full, acc_empty, w_free, ticket);
    }
  }
  tc_fence_before();
  __syncthreads();
  cluster_sync();                       // neither CTA exits (or frees TMEM) while its peer may still arrive / read
  if (warp == 2) {
    tc_fence_after();
    tmem_dealloc2(tmem_base, 512);
  }
}

template <class G>
static cudaError_t launch_fused(const FusedArgs& a, int ncl, cudaStream_t st, int* occupancy) {
  static bool attr_set = false;
  if (!attr_set) {
    cudaError_t e1 = cudaFuncSetAttribute(lstm_fused_kernel<G>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)Der<G>::SMEM);
    if (e1 != cudaSuccess) return e1;
    attr_set = true;
  }
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3((occupancy ? 64 : ncl) * 2 * G::PPG);
  cfg.blockDim = dim3(Der<G>::THREADS);
  cfg.dynamicSmemBytes = Der<G>::SMEM;
  cfg.stream = st;
  cudaLaunchAttribute at[1];
  at[0].id = cudaLaunchAttributeClusterDimension;
  at[0].val.clusterDim.x = G::CLS; at[0].val.clusterDim.y = 1; at[0].val.clusterDim.z = 1;
  cfg.attrs = at; cfg.numAttrs = 1;
  if (occupancy) return cudaOccupancyMaxActiveClusters(occupancy, lstm_fused_kernel<G>, &cfg);
  return cudaLaunchKernelEx(&cfg, lstm_fused_kernel<G>, a);
}
// co-resident groups of PPG CTA pairs (all CTAs of a launch must be resident: the groups spin on each other's counters)
template <class G>
static int fused_max_groups() {
  static int cached = -1;
  if (cached >= 0) return cached;
  int n = 0;
  FusedArgs dummy{};
  if (launch_fused<G>(dummy, 0, nullptr, &n) != cudaSuccess) { cudaGetLastError(); return -1; }
  cached = (n * Der<G>::NP) / G::PPG;
  if (cached > U_MAX_GROUPS) cached = U_MAX_GROUPS;
  return cached;
}

static long long* g_fused_probe = nullptr;

// slots <= 0: the number of interleaved tile pairs per group (1..3) that minimises passes x step time, with a step
// costing max(dependency chain ~ 2.3 items, slots items).
static int auto_slots(int ptiles, int cap) {
  int best = 1;
  double best_t = 1e30;
  for (int s = 1; s <= LNS && s <= ptiles; ++s) {
    const int gpd = (ptiles + s - 1) / s;
    const int passes = (2 * gpd + cap - 1) / cap;
    const double t = passes * (s > 2.3 ? (double)s : 2.3);
    if (t < best_t - 1e-9) { best_t = t; best = s; }
  }
  return best;
}

template <class G>
static int run_fused(const char* what, const void* xhat, const void* w_fused, const void* zero_tile, void* y_f, void* y_b,
                     long y_stride, int R, int steps, int seq_tiles, int max_groups, int slots, void* sync_ws, void* stream,
                     void* sv_gates = nullptr, float* sv_c0 = nullptr, float* sv_c1 = nullptr) {
  int cap = fused_max_groups<G>();
  if (cap <= 0) {
    cudaGetLastError();
    set_error("%s: kernel does not fit (2-CTA clusters, %d threads, %zu B shared memory)", what, Der<G>::THREADS, Der<G>::SMEM);
    return 2;
  }
  if (max_groups > 0 && cap > max_groups) cap = max_groups;
  const int ptiles = (seq_tiles + 1) / 2;
  if (slots <= 0) slots = auto_slots(ptiles, cap);
  if (slots > LNS) slots = LNS;
  if (slots > ptiles) slots = ptiles;
  FusedArgs a{reinterpret_cast<const __half*>(xhat), reinterpret_cast<const __half*>(w_fused),
              reinterpret_cast<const __half*>(zero_tile), reinterpret_cast<__half*>(y_f), reinterpret_cast<__half*>(y_b),
              y_stride, R, steps, seq_tiles, (ptiles + slots - 1) / slots, reinterpret_cast<unsigned*>(sync_ws), g_fused_probe,
              reinterpret_cast<__half*>(sv_gates), sv_c0, sv_c1};
  int ncl = 2 * a.gpd;
  if (ncl > cap) ncl = cap;
  cudaStream_t st = (cudaStream_t)stream;
  BSRNN_CUDA_OK(cudaMemsetAsync(sync_ws, 0, (size_t)U_SYNC_WORDS * sizeof(unsigned), st));
  cudaError_t le = launch_fused<G>(a, ncl, st, nullptr);
  if (le != cudaSuccess) { set_error("%s: %s", what, cudaGetErrorString(le)); return 3; }
  BSRNN_LAUNCH_OK();
  return 0;
}

}  // namespace bsrnn
using namespace bsrnn;

extern "C" void bsrnn_debug_set_fused_probe(void* p) { g_fused_probe = reinterpret_cast<long long*>(p); }

// Fused BLSTM layer, H = 392 (see the header of this file).  sync_ws: bsrnn_blstm_fused_sync_bytes() of device memory
// owned by the caller (zeroed here, stream-ordered, before every launch).  y: [step][seq_tile][dir][50][128][8].
extern "C" int bsrnn_blstm_fused_tc(const void* xhat, const void* w_fused, const void* zero_tile, void* y, int R, int steps,
                                    int seq_tiles, int max_groups, int slots, void* sync_ws, void* stream) {
  BSRNN_CHECK_ARG(xhat && w_fused && zero_tile && y && sync_ws, "blstm_fused_tc: null pointer");
  BSRNN_CHECK_ARG(R > 0 && steps > 0 && (long)seq_tiles * 128 >= R, "blstm_fused_tc: bad dims");
  const long y_tile = (long)Geo392::HKC * 128 * 8;
  return run_fused<Geo392>("blstm_fused_tc", xhat, w_fused, zero_tile, y, reinterpret_cast<__half*>(y) + y_tile, 2 * y_tile, R,
                           steps, seq_tiles, max_groups, slots, sync_ws, stream);
}
extern "C" int bsrnn_blstm_fused_max_groups(void) { return fused_max_groups<Geo392>(); }
// Same layer on groups of 7 pairs x 56 units (Geo392x7): w_fused7 [2][7][2][76][112][8]; x, zero_tile, y, sync_ws as above.
extern "C" int bsrnn_blstm_fused7_tc(const void* xhat, const void* w_fused7, const void* zero_tile, void* y, int R, int steps,
                                     int seq_tiles, int max_groups, int slots, void* sync_ws, void* stream) {
  BSRNN_CHECK_ARG(xhat && w_fused7 && zero_tile && y && sync_ws, "blstm_fused7_tc: null pointer");
  BSRNN_CHECK_ARG(R > 0 && steps > 0 && (long)seq_tiles * 128 >= R, "blstm_fused7_tc: bad dims");
  const long y_tile = (long)Geo392x7::HKC * 128 * 8;
  return run_fused<Geo392x7>("blstm_fused7_tc", xhat, w_fused7, zero_tile, y, reinterpret_cast<__half*>(y) + y_tile, 2 * y_tile,
                             R, steps, seq_tiles, max_groups, slots, sync_ws, stream);
}
extern "C" int bsrnn_blstm_fused7_max_groups(void) { return fused_max_groups<Geo392x7>(); }
// Same layer on groups of 14 pairs x 28 units (Geo392x14, the small-batch geometry): w_fused14 [2][14][2][76][56][8].
extern "C" int bsrnn_blstm_fused14_tc(const void* xhat, const void* w_fused14, const void* zero_tile, void* y, int R, int steps,
                                      int seq_tiles, int max_groups, int slots, void* sync_ws, void* stream) {
  BSRNN_CHECK_ARG(xhat && w_fused14 && zero_tile && y && sync_ws, "blstm_fused14_tc: null pointer");
  BSRNN_CHECK_ARG(R > 0 && steps > 0 && (long)seq_tiles * 128 >= R, "blstm_fused14_tc: bad dims");
  const long y_tile = (long)Geo392x14::HKC * 128 * 8;
  static int cls_env = -1;
  if (cls_env < 0) { const char* e = getenv("BSRNN_FUSED14_CLS"); cls_env = (e && e[0] == '4') ? 4 : 2; }
  if (cls_env == 4)
    return run_fused<Geo392x14M>("blstm_fused14_tc", xhat, w_fused14, zero_tile, y, reinterpret_cast<__half*>(y) + y_tile, 2 * y_tile,
                                 R, steps, seq_tiles, max_groups, slots, sync_ws, stream);
  return run_fused<Geo392x14>("blstm_fused14_tc", xhat, w_fused14, zero_tile, y, reinterpret_cast<__half*>(y) + y_tile, 2 * y_tile,
                              R, steps, seq_tiles, max_groups, slots, sync_ws, stream);
}
extern "C" int bsrnn_blstm_fused14_max_groups(void) { return fused_max_groups<Geo392x14>(); }
extern "C" int bsrnn_blstm_fused_sync_bytes(void) { return (int)(U_SYNC_WORDS * sizeof(unsigned)); }

// Fused BLSTM layer, H = 768 / N = 384 (BSRNN_flowse): xhat [steps*seq_tiles][50][128][8] (column 384 = 1), w_fused
// [2][24][2][146][64][8], zero_tile 96*128*8 zeros.  The (step, tile) block of direction d is y_d + (step*seq_tiles +
// tile) * y_stride halves, [96][128][8] each: two separate buffers (y_stride = 96*1024) or one interleaved buffer
// [steps*seq_tiles][dir][96][128][8] (y_b = y_f + 96*1024, y_stride = 2*96*1024 = the Linear GEMM's K = 1536 operand).
extern "C" int bsrnn_blstm_fused768_tc(const void* xhat, const void* w_fused, const void* zero_tile, void* y_f, void* y_b,
                                       long y_stride, int R, int steps, int seq_tiles, int max_groups, int slots, void* sync_ws,
                                       void* stream) {
  BSRNN_CHECK_ARG(xhat && w_fused && zero_tile && y_f && y_b && sync_ws, "blstm_fused768_tc: null pointer");
  BSRNN_CHECK_ARG(R > 0 && steps > 0 && (long)seq_tiles * 128 >= R, "blstm_fused768_tc: bad dims");
  BSRNN_CHECK_ARG(y_stride >= (long)Geo768::HKC * 128 * 8 && y_stride % 8 == 0, "blstm_fused768_tc: bad y_stride");
  return run_fused<Geo768>("blstm_fused768_tc", xhat, w_fused, zero_tile, y_f, y_b, y_stride, R, steps, seq_tiles, max_groups,
                           slots, sync_ws, stream);
}
extern "C" int bsrnn_blstm_fused768_max_groups(void) { return fused_max_groups<Geo768>(); }

namespace bsrnn {
// unit-major scratch of the SAVE kernels -> the row-major buffers of bsrnn_blstm_train_bwd_tc.  grid (tiles, 2 directions).
template <int H>
__global__ void __launch_bounds__(256) saved_transpose_kernel(const uint2* __restrict__ gT, const float* __restrict__ cT0,
                                                             const float* __restrict__ cT1, uint2* __restrict__ gates,
                                                             float* __restrict__ c0, float* __restrict__ c1) {
  __shared__ uint2 tg[32][33];
  __shared__ float tc[32][33];
  const int tile = blockIdx.x, d = blockIdx.y;
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;                 // 32 x 8
  const uint2* sg = gT + ((size_t)(tile * 2 + d) * H) * 128;              // [unit][row]
  const float* sc = (d == 0 ? cT0 : cT1) + (size_t)tile * H * 128;
  uint2* dg = gates + (size_t)tile * 128 * (2 * H) + (size_t)d * H;       // row stride 2*H uint2 (= 8H halves)
  float* dc = (d == 0 ? c0 : c1) + (size_t)tile * 128 * H;
  for (int u0 = 0; u0 < H; u0 += 32) {
    for (int r0 = 0; r0 < 128; r0 += 32) {
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        const int u = u0 + ty + 8 * k;
        if (u < H) {
          tg[ty + 8 * k][tx] = sg[(size_t)u * 128 + r0 + tx];
          tc[ty + 8 * k][tx] = sc[(size_t)u * 128 + r0 + tx];
        }
      }
      __syncthreads();
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        const int r = r0 + ty + 8 * k, u = u0 + tx;
        if (u < H) {
          dg[(size_t)r * (2 * H) + u] = tg[tx][ty + 8 * k];
          dc[(size_t)r * H + u] = tc[tx][ty + 8 * k];
        }
      }
      __syncthreads();
    }
  }
}

// scratch of a SAVE launch: unit-major gates (2 directions x 4H halves per row) + c_t (2 directions x H floats per row)
template <int H>
static long fused_train_scratch_bytes(int steps, int seq_tiles) {
  return (long)steps * seq_tiles * 128 * H * (2 * 4 * 2 + 2 * 4);
}

// SAVE launch of geometry G, then the transpose of its scratch into gates / c_f / c_b
template <class G>
static int run_fused_train(const char* what, const void* xhat, const void* w_fused, const void* zero_tile, void* y_f, void* y_b,
                           long y_stride, void* gates, float* c_f, float* c_b, void* scratch, int R, int steps, int seq_tiles,
                           int max_groups, int slots, void* sync_ws, void* stream) {
  static_assert(G::SAVE, "training forward needs a SAVE geometry");
  const size_t m_all = (size_t)steps * seq_tiles;
  __half* gT = reinterpret_cast<__half*>(scratch);
  float* cT0 = reinterpret_cast<float*>(gT + m_all * 128 * 8 * G::H);
  float* cT1 = cT0 + m_all * 128 * G::H;
  const int rc = run_fused<G>(what, xhat, w_fused, zero_tile, y_f, y_b, y_stride, R, steps, seq_tiles, max_groups, slots, sync_ws,
                              stream, gT, cT0, cT1);
  if (rc) return rc;
  saved_transpose_kernel<G::H><<<dim3((unsigned)m_all, 2), 256, 0, (cudaStream_t)stream>>>(
      reinterpret_cast<const uint2*>(gT), cT0, cT1, reinterpret_cast<uint2*>(gates), c_f, c_b);
  BSRNN_LAUNCH_OK();
  return 0;
}
}  // namespace bsrnn

// Training forward of the BLSTM layer (H = 392) on the fused kernel: as bsrnn_blstm_fused7_tc / _fused14_tc (geo = 7 | 14) with
// separate output buffers per direction (block (step, tile) of direction d at y_d + (step*seq_tiles + tile) * y_stride halves,
// [50][128][8] each) and the activations BPTT needs written by the epilogue: gates rows [(step*seq_tiles + tile)*128 + r][8H]
// fp16 = ACTIVATED i, f, g, o at column dir*4H + 4u + gate, c_f / c_b [step][seq_tiles*128][H] f32 -- the buffers
// bsrnn_blstm_train_bwd_tc reads [replaces autograd's saved tensors of nn.LSTM, d_model.py:61-95 / train_se.py:74-84].
// scratch: (2 * steps*seq_tiles*128*4H halves) + (2 * steps*seq_tiles*128*H floats) = bsrnn_blstm_fused_train_scratch_bytes().
extern "C" long bsrnn_blstm_fused_train_scratch_bytes(int steps, int seq_tiles) {
  return fused_train_scratch_bytes<392>(steps, seq_tiles);
}
extern "C" int bsrnn_blstm_fused_train_tc(int geo, const void* xhat, const void* w_fused, const void* zero_tile, void* y_f,
                                          void* y_b, long y_stride, void* gates, float* c_f, float* c_b, void* scratch, int R,
                                          int steps, int seq_tiles, int max_groups, int slots, void* sync_ws, void* stream) {
  BSRNN_CHECK_ARG(xhat && w_fused && zero_tile && y_f && y_b && gates && c_f && c_b && sync_ws && scratch, "blstm_fused_train_tc: null pointer");
  BSRNN_CHECK_ARG(R > 0 && steps > 0 && (long)seq_tiles * 128 >= R, "blstm_fused_train_tc: bad dims");
  BSRNN_CHECK_ARG(geo == 7 || geo == 14, "blstm_fused_train_tc: geo must be 7 or 14");
  BSRNN_CHECK_ARG(y_stride >= (long)Geo392x7::HKC * 128 * 8 && y_stride % 8 == 0, "blstm_fused_train_tc: bad y_stride");
  return geo == 7 ? run_fused_train<Geo392x7S>("blstm_fused_train_tc", xhat, w_fused, zero_tile, y_f, y_b, y_stride, gates, c_f, c_b,
                                               scratch, R, steps, seq_tiles, max_groups, slots, sync_ws, stream)
                  : run_fused_train<Geo392x14S>("blstm_fused_train_tc", xhat, w_fused, zero_tile, y_f, y_b, y_stride, gates, c_f, c_b,
                                                scratch, R, steps, seq_tiles, max_groups, slots, sync_ws, stream);
}

// Training forward of the BLSTM layer at H = 768 / N = 384 (BSRNN_flowse) on the fused kernel (Geo768S): xhat, w_fused,
// zero_tile, y_f / y_b / y_stride as bsrnn_blstm_fused768_tc; gates [(step*seq_tiles + tile)*128 + r][8H] fp16 and c_f / c_b
// [step][seq_tiles*128][H] f32 as bsrnn_blstm_fused_train_tc.  scratch: bsrnn_blstm_fused768_train_scratch_bytes().
extern "C" long bsrnn_blstm_fused768_train_scratch_bytes(int steps, int seq_tiles) {
  return fused_train_scratch_bytes<768>(steps, seq_tiles);
}
extern "C" int bsrnn_blstm_fused768_train_tc(const void* xhat, const void* w_fused, const void* zero_tile, void* y_f, void* y_b,
                                             long y_stride, void* gates, float* c_f, float* c_b, void* scratch, int R, int steps,
                                             int seq_tiles, int max_groups, int slots, void* sync_ws, void* stream) {
  BSRNN_CHECK_ARG(xhat && w_fused && zero_tile && y_f && y_b && gates && c_f && c_b && sync_ws && scratch,
                  "blstm_fused768_train_tc: null pointer");
  BSRNN_CHECK_ARG(R > 0 && steps > 0 && (long)seq_tiles * 128 >= R, "blstm_fused768_train_tc: bad dims");
  BSRNN_CHECK_ARG(y_stride >= (long)Geo768::HKC * 128 * 8 && y_stride % 8 == 0, "blstm_fused768_train_tc: bad y_stride");
  return run_fused_train<Geo768S>("blstm_fused768_train_tc", xhat, w_fused, zero_tile, y_f, y_b, y_stride, gates, c_f, c_b,
                                  scratch, R, steps, seq_tiles, max_groups, slots, sync_ws, stream);
}
