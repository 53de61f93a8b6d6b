// Persistent, epilogue-overlapped WN layer kernel (glow.py:201-220) for C = 256.
//
// Why: when one tile's [128 x 512] fp32 pre-activation fills tensor memory, the gate, the res/skip epilogue, the stores
// and the per-tile prologue all run with the tensor pipe stopped (ncu r1e: 52 % active in f16f8).  Here
//   * a CTA PAIR (cta_group::2, M = 256) is persistent and loops over tile pairs: TMEM, barriers, biases and the
//     folded-`end` weight tiles are set up once per CTA;
//   * GEMM1 runs as two N = 256 SWEEPS over K.  Sweep g computes the tanh AND the sigmoid rows of channels
//     [128g, 128g+128): in the 2-SM MMA each CTA supplies half of the N rows of B, so the leader loads the tanh rows and
//     the follower the sigmoid rows of the same channels - no weight re-packing.  Sweep g accumulates into TMEM region
//     R_g = columns [256g, 256g+256), so the gate of sweep 0 runs under the MMAs of sweep 1;
//   * GEMM2 (res -> R1, folded `end` -> R0[32,64)) follows the gate of sweep 1; its residual epilogue, the x_old loads
//     and the TMA stores of tile i run under sweep 0 of tile i+1 (R0 is released as soon as the 16 `end` columns are
//     read, R1 when the res accumulator has been read).
// Per tile the tensor pipe now only waits for the gate of sweep 1 (half of the gate) and the barrier hand-offs.
// The price: the activation (A) tiles are streamed once per sweep, i.e. twice per tile.
//
// Shared memory (per CTA): twelve 16-KB units.  0-3: A ring; 4-7: B ring (a CTA's half of a [256 x 64] weight tile);
// 8-11: gate outputs that do not live in TMEM (bf16x3: acts lo tiles of the four 64-channel blocks; f16f8: the e5m2
// lo*2^P / hi*2^-Q acts tiles of the two 128-channel groups), re-used after GEMM2 as the x_old / x_new staging of the
// residual epilogue (column group h: units 8+2h (hi) and 9+2h (lo), one 64-channel block at a time).
// TMEM: R0 = [0,256): sweep-0 accumulators (tanh 0-127 | sigmoid 128-255); afterwards acts hi (bf16/fp16 pairs, the A
// operand of GEMM2's ".ts" MMAs) at [0,32) [64,96) [128,160) [192,224) and the folded-`end` accumulator at [32,64).
// R1 = [256,512): sweep-1 accumulators, afterwards the res accumulator.
#include "cwg_tc_common.cuh"

#include <stdlib.h>
#include <string.h>

namespace cwg {

using namespace sm100;
using namespace tc;

namespace {

struct PsArgs {
  const float* b1;        // [2C]
  const float* b2;        // [C]
  const float* eo_b;      // [MG]
  float* eo;              // [B*T'][MG], MG = eo_pitch (16; 32 for the wide group layout, include/cwg.h CWG_GROUP_PAD)
  int eo_pitch;           // wide (32): the follower's 16 folded-`end` rows are real and column group 1 accumulates them
  long long b1_bstride;   // floats between the gate biases of consecutive utterances (ax WN speaker embedding); 0: shared
  uint8_t* xo_l8;         // f16f8: e5m2 planes of x_out, written with plain 16-byte stores
  uint8_t* xo_h8;
  int Tp, dil;
  int w1_row0, w2_row0;
  int has_res, first;
  int pairs_per_utt, n_pairs;
  // layer-0 fold (fused0): x_0 = start(audio_0) is never materialised.  GEMM1 contracts the 3 taps of the <= 8 coupling
  // input channels (+ a constant-1 channel carrying the start bias) with W_in*S (tm_a0_* / tm_w0_*), and the residual
  // epilogue rebuilds x_old = S a + b in fp32 from the audio state
  int fused0;
  const float* audio;     // [B*T'][G] fp32 audio state; audio_0 of row m = audio[m*G + a_off .. + a_nh)
  int G, a_off, a_nh;
  const float* start_w;   // [C][8] (the fold takes the narrow layout, n_half <= 8, only)
  const float* start_b;   // [C]
  int w0_row0;
  int* range_flag;        // f16f8, last residual layer only: |= 2 when x_new leaves the fp16 range (else NULL)
  long long* dbg;         // optional: per CTA {start, end, tiles} clock64 stamps
  // RAGGED only (appended so that the other instantiations keep their parameter offsets): utterance b holds
  // T'_b = len[b] * P valid group-steps and tile pairs [prefix[b], prefix[b+1]); n_pairs = prefix[nb] on the device
  const int* len;         // [nb] mel frames, already clamped to [1, Tm] (cwg_infer_ragged's plan kernel)
  const int* prefix;      // [nb + 1]
  int nb, P;
};

constexpr int P_OFF_WSE = 12 * TILE_A;                 // 196608
constexpr int P_OFF_B1 = P_OFF_WSE + 16384;
constexpr int P_OFF_B2 = P_OFF_B1 + 2048;
constexpr int P_OFF_BAR = P_OFF_B2 + 1024;
constexpr int P_OFF_S = P_OFF_BAR + 256;               // fused0: start weights [256][8] fp32 + bias [256]
constexpr int P_SMEM = P_OFF_S + 256 * 8 * 4 + 1024 + 1024;   // 226560 (<= 232448)
constexpr int P_OFF_R = P_OFF_S + 256 * 8 * 4 + 1024;  // RAGGED: tile-pair prefix sums [nb + 1]
constexpr int P_SMEM_R = P_SMEM + (4 * (CWG_RAGGED_MAX_BATCH + 1) + 15) / 16 * 16;   // 230672
static_assert(P_SMEM_R <= 232448, "ragged prefix sums do not fit next to the layer kernel's shared memory");
constexpr int TILE_S = 4096;                           // [128 rows][16 x 16-bit], 32B swizzle
constexpr int P_EPI_THREADS = 256;
constexpr int P_THREADS = 128 + P_EPI_THREADS;
constexpr int PS_DBG_STRIDE = 24;                      // int64 per CTA in the debug buffer: {start, end, tiles, -}, 12 MMA-thread stamps, 8 epilogue stamps
constexpr uint32_t P_D_RES = 256, P_D_EO = 32;         // TMEM columns of the GEMM2 accumulators

// TMEM column of the packed 16-bit acts of 16-channel chunk c (0..15): sweep g = c / 8 writes into R0 columns the same
// warp has already consumed (g = 0: behind its own tanh read pointer; g = 1: its sigmoid columns of sweep 0)
__device__ __forceinline__ uint32_t P_ACOL(int c) { return (uint32_t)(((c >> 3) << 7) + (((c >> 2) & 1) << 6) + ((c & 3) << 3)); }

// f16f8 residual epilogue: 16 fp32 values -> fp16 hi / lo words (to the in-place staging tiles) and the two e5m2 words
__device__ __forceinline__ void split16_f8_words(const float* v, uint32_t* hi, uint32_t* lo, uint32_t* l8, uint32_t* h8) {
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    float h0, h1;
    hi[i] = pack_f16x2(v[2 * i], v[2 * i + 1]);
    unpack2<true>(hi[i], h0, h1);
    lo[i] = pack_f16x2(v[2 * i] - h0, v[2 * i + 1] - h1);
  }
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    l8[i] = e5m2x4_from_f16x2(lo[2 * i], lo[2 * i + 1], F16X2_2P6);
    h8[i] = e5m2x4_from_f16x2(hi[2 * i], hi[2 * i + 1], F16X2_2M8);
  }
}

// FUSED0: the layer-0 fold variant (compiled separately so that its extra registers do not burden layers 1..L-1)
// RAGGED: per-utterance lengths (cwg_infer_ragged).  Pair p maps to (b, t0) through the prefix sums of the utterances'
// tile pairs, so pairs wholly past T'_b do not exist; rows t >= T'_b of a computed tile are stored as zeros (every
// plane) and leave eo and the range flag alone.  The caller keeps every row t >= T'_b of both x buffers at 0, so the
// dilated taps of valid rows read exactly the zero padding a call for utterance b alone would see.
template <int NPASS, bool FUSED0, bool RAGGED>
__global__ void __launch_bounds__(P_THREADS, 1)
k_layer_ps(const __grid_constant__ CUtensorMap tm_x_hi, const __grid_constant__ CUtensorMap tm_x_lo,
           const __grid_constant__ CUtensorMap tm_h_hi, const __grid_constant__ CUtensorMap tm_h_lo,
           const __grid_constant__ CUtensorMap tm_w1_hi, const __grid_constant__ CUtensorMap tm_w1_lo,
           const __grid_constant__ CUtensorMap tm_w2_hi, const __grid_constant__ CUtensorMap tm_w2_lo,
           const __grid_constant__ CUtensorMap tm_wse_hi, const __grid_constant__ CUtensorMap tm_wse_lo,
           const __grid_constant__ CUtensorMap tm_xo_hi, const __grid_constant__ CUtensorMap tm_xo_lo,
           // e5m2 planes, NPASS == 2 (CWG_MODE_F16F8) only; tm_w2_lo / tm_wse_lo are then the e5m2 hi*2^-P planes of w2
           const __grid_constant__ CUtensorMap tm_x_l8, const __grid_constant__ CUtensorMap tm_x_h8,
           const __grid_constant__ CUtensorMap tm_h_l8, const __grid_constant__ CUtensorMap tm_h_h8,
           const __grid_constant__ CUtensorMap tm_w1_h8, const __grid_constant__ CUtensorMap tm_w1_l8,
           const __grid_constant__ CUtensorMap tm_w2_l8, const __grid_constant__ CUtensorMap tm_wse_l8,
           // layer-0 fold: coupling-input planes (16 channels) and folded weights (3 taps x 16), 32B-swizzled 4-KB tiles
           const __grid_constant__ CUtensorMap tm_a0_hi, const __grid_constant__ CUtensorMap tm_a0_lo,
           const __grid_constant__ CUtensorMap tm_w0_hi, const __grid_constant__ CUtensorMap tm_w0_lo, PsArgs a) {
  constexpr bool F8 = NPASS == 2;
  constexpr bool X3 = NPASS != 1;                 // the gate produces a second (lo / e5m2) set of acts planes
  constexpr int PL = NPASS == 3 ? 2 : 1;          // planes streamed per k-block in GEMM1 of the bf16 modes
  constexpr int PL2 = X3 ? 2 : 1;
  constexpr uint32_t ID256 = F8 ? umma_idesc_f16(256, 256) : umma_idesc_bf16(256, 256);
  constexpr uint32_t ID32 = F8 ? umma_idesc_f16(256, 32) : umma_idesc_bf16(256, 32);
  constexpr uint32_t IDE256 = umma_idesc_e5m2(256, 256), IDE32 = umma_idesc_e5m2(256, 32);

  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = align_1024(smem_raw);
  float* b1s = reinterpret_cast<float*>(smem + P_OFF_B1);
  float* b2s = reinterpret_cast<float*>(smem + P_OFF_B2);
  float* s_tab = reinterpret_cast<float*>(smem + P_OFF_S);            // fused0 only
  float* s_bias = s_tab + 256 * 8;
  uint64_t* full = reinterpret_cast<uint64_t*>(smem + P_OFF_BAR);   // [8]: A slot i -> i, B slot j -> 4 + j
  uint64_t* empty = full + 8;
  uint64_t* wse_full = empty + 8;
  uint64_t* acc_full = wse_full + 1;        // [2]: sweep g complete (multicast commit, both CTAs)
  uint64_t* acts_ready = acc_full + 2;      // leader: both gates of both CTAs are written
  uint64_t* acc2_full = acts_ready + 1;     // GEMM2 complete (both CTAs)
  uint64_t* r_free = acc2_full + 1;         // [2], leader: TMEM region g may be overwritten by the next tile's sweep g
  uint64_t* xold_full = r_free + 2;         // [2]: x_old block of column group h has landed
  uint64_t* acts0_ready = xold_full + 2;    // leader: the gate of sweep 0 (channels [0, 128) of acts) is written in both CTAs
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(acts0_ready + 1);
  int* pre_s = reinterpret_cast<int*>(smem + P_OFF_R);                 // RAGGED only

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (RAGGED)
    for (int i = threadIdx.x; i <= a.nb; i += P_THREADS) pre_s[i] = __ldg(a.prefix + i);
  auto slot = [&](int i) { return smem + i * TILE_A; };
  auto wse = [&](int plane, int kb) { return smem + P_OFF_WSE + plane * 8192 + kb * 2048; };

  if (threadIdx.x == 0) {
    for (int i = 0; i < 8; ++i) { mbar_init(&full[i], 1); mbar_init(&empty[i], 1); }
    mbar_init(wse_full, 1); mbar_init(&acc_full[0], 1); mbar_init(&acc_full[1], 1);
    // epilogue -> MMA hand-offs: ONE elected arrive per warp after __syncwarp (512 per-thread arrives, half of them remote
    // DSMEM transactions, cost ~1.3-2.9 k cycles per hand-off in the per-tile timeline)
    mbar_init(acts_ready, 2 * (P_EPI_THREADS / 32)); mbar_init(acc2_full, 1);
    mbar_init(&r_free[0], a.eo_pitch == 32 ? 2 * (P_EPI_THREADS / 32) : 2 * (P_EPI_THREADS / 64)); mbar_init(&r_free[1], 2 * (P_EPI_THREADS / 32));
    mbar_init(&xold_full[0], 1); mbar_init(&xold_full[1], 1);
    mbar_init(acts0_ready, 2 * (P_EPI_THREADS / 32));
    fence_barrier_init();
  }
  if (warp == 1) tmem_alloc_2sm(tmem_slot, 512);
  tc_fence_before_sync();
  __syncthreads();
  cluster_sync_all();                              // both CTAs' barriers and TMEM exist before anything targets them
  tc_fence_after_sync();
  const uint32_t tmem = *tmem_slot;
  const uint32_t rank = cluster_ctarank();
  const bool leader = rank == 0;
  const int cluster_id = blockIdx.x >> 1, n_clusters = gridDim.x >> 1;

  // loads complete on the LEADER's barrier, armed by the leader for both CTAs' bytes
  auto arm = [&](uint64_t* bar, uint32_t bytes) { if (leader) mbar_arrive_expect_tx(bar, 2 * bytes); };
  auto lda3 = [&](void* dst, const CUtensorMap* m, uint64_t* bar, int c0, int c1, int c2) {
    tma_load_3d_2sm(dst, m, mapa_shared(bar, 0), c0, c1, c2);
  };
  auto ldb2 = [&](void* dst, const CUtensorMap* m, uint64_t* bar, int c0, int row) {
    tma_load_2d_2sm(dst, m, mapa_shared(bar, 0), c0, row);
  };
  auto kblk = [&](uint32_t a_addr, uint32_t b_addr, uint32_t d, uint32_t id, bool first) {
    const uint64_t da = DESC_SW128_HI | (uint64_t)((a_addr & 0x3FFFF) >> 4), db = DESC_SW128_HI | (uint64_t)((b_addr & 0x3FFFF) >> 4);
    umma_bf16_2sm(d, da, db, id, first ? 0u : 1u); umma_bf16_2sm(d, da + 2, db + 2, id, 1u);
    umma_bf16_2sm(d, da + 4, db + 4, id, 1u); umma_bf16_2sm(d, da + 6, db + 6, id, 1u);
  };
  auto kblk8 = [&](uint32_t a_addr, uint32_t b_addr, uint32_t d, uint32_t id) {
    const uint64_t da = DESC_SW128_HI | (uint64_t)((a_addr & 0x3FFFF) >> 4), db = DESC_SW128_HI | (uint64_t)((b_addr & 0x3FFFF) >> 4);
    umma_f8_2sm(d, da, db, id, 1u); umma_f8_2sm(d, da + 2, db + 2, id, 1u);
    umma_f8_2sm(d, da + 4, db + 4, id, 1u); umma_f8_2sm(d, da + 6, db + 6, id, 1u);
  };
  // number of tile pairs of the launch, and the tile of pair p handled by this CTA.  RAGGED: every role walks p upwards,
  // so a per-thread cursor over the prefix sums finds b
  auto n_pairs = [&]() { return RAGGED ? pre_s[a.nb] : a.n_pairs; };
  int ub = 0;
  auto tile_of = [&](int p, int& b, int& t0) {
    if (RAGGED) {
      while (pre_s[ub + 1] <= p) ++ub;
      b = ub;
      t0 = ((p - pre_s[ub]) * 2 + (int)rank) * 128;
    } else {
      b = p / a.pairs_per_utt;
      t0 = ((p - b * a.pairs_per_utt) * 2 + (int)rank) * 128;
    }
  };

  if (warp == 0 && lane == 0) {
    // ---------------- producer A: activation tiles (3 dilated taps of x, then the cond hidden H2), once per sweep
    tma_prefetch_desc(&tm_x_hi); tma_prefetch_desc(&tm_h_hi);
    if (F8) { tma_prefetch_desc(&tm_x_l8); tma_prefetch_desc(&tm_x_h8); }
    if (NPASS == 3) { tma_prefetch_desc(&tm_x_lo); tma_prefetch_desc(&tm_h_lo); }
    int s = 0; uint32_t pm = 0;
    for (int p = cluster_id; p < n_pairs(); p += n_clusters) {
      int b, t0; tile_of(p, b, t0);
      for (int g = 0; g < 2; ++g) {
        if (FUSED0) {
          // one ring item per plane: the 3 tap tiles [128 steps x 16 channels] of the coupling input (4 KB each)
          for (int pl = 0; pl < PL2; ++pl) {
            mbar_wait(&empty[s], ((pm >> s) & 1u) ^ 1u);
            pm ^= 1u << s;
            arm(&full[s], 3 * TILE_S);
            for (int tap = 0; tap < 3; ++tap)
              lda3(slot(s) + tap * TILE_S, pl ? &tm_a0_lo : &tm_a0_hi, &full[s], 0, t0 + (tap - 1) * a.dil, b);
            s = (s + 1) & 3;
          }
        }
        if (F8) {
          // K in groups of 128 channels (taps 0..2 of x: groups 0..5, H2: groups 6, 7); per group two fp16 tiles of 64
          // channels, then the e5m2 tile of lo*2^P and the e5m2 tile of hi*2^-Q (128 channels = 128 bytes per row)
          for (int G = FUSED0 ? 6 : 0; G < 8; ++G)
            for (int it = 0; it < 4; ++it) {
              mbar_wait(&empty[s], ((pm >> s) & 1u) ^ 1u);
              pm ^= 1u << s;
              arm(&full[s], TILE_A);
              const bool cond = G >= 6;
              const int tt = cond ? t0 : t0 + ((G >> 1) - 1) * a.dil;
              const int c0 = (cond ? G - 6 : (G & 1)) * 128;
              if (it < 2) lda3(slot(s), cond ? &tm_h_hi : &tm_x_hi, &full[s], c0 + it * 64, tt, b);
              else if (it == 2) lda3(slot(s), cond ? &tm_h_l8 : &tm_x_l8, &full[s], c0, tt, b);
              else lda3(slot(s), cond ? &tm_h_h8 : &tm_x_h8, &full[s], c0, tt, b);
              s = (s + 1) & 3;
            }
        } else {
          for (int kb = FUSED0 ? 12 : 0; kb < 16; ++kb)
            for (int pl = 0; pl < PL; ++pl) {
              mbar_wait(&empty[s], ((pm >> s) & 1u) ^ 1u);
              pm ^= 1u << s;
              arm(&full[s], TILE_A);
              if (kb < 12) lda3(slot(s), pl ? &tm_x_lo : &tm_x_hi, &full[s], (kb & 3) * 64, t0 + ((kb >> 2) - 1) * a.dil, b);
              else lda3(slot(s), pl ? &tm_h_lo : &tm_h_hi, &full[s], (kb - 12) * 64, t0, b);
              s = (s + 1) & 3;
            }
        }
      }
    }
  } else if (warp == 2 && lane == 0) {
    // ---------------- producer B: this CTA's 128 rows of every weight tile.  Sweep g: leader = tanh rows, follower =
    // sigmoid rows of channels [128g, 128g+128).  Then W2 (res rows [128*rank, +128)).
    tma_prefetch_desc(&tm_w1_hi); tma_prefetch_desc(&tm_w2_hi);
    if (F8) { tma_prefetch_desc(&tm_w1_h8); tma_prefetch_desc(&tm_w1_l8); }
    if (NPASS == 3) tma_prefetch_desc(&tm_w1_lo);
    int j = 0; uint32_t pm = 0;
    auto next_slot = [&]() {
      mbar_wait(&empty[4 + j], ((pm >> j) & 1u) ^ 1u);
      pm ^= 1u << j;
      arm(&full[4 + j], TILE_A);
    };
    const int w2_row = a.w2_row0 + (int)rank * 128;
    for (int p = cluster_id; p < n_pairs(); p += n_clusters) {
      for (int g = 0; g < 2; ++g) {
        const int w1_row = a.w1_row0 + (int)rank * 256 + g * 128;
        if (FUSED0) {
          const int w0_row = a.w0_row0 + (int)rank * 256 + g * 128;
          for (int pl = 0; pl < PL2; ++pl) {
            mbar_wait(&empty[4 + j], ((pm >> j) & 1u) ^ 1u);
            pm ^= 1u << j;
            arm(&full[4 + j], 3 * TILE_S);
            for (int tap = 0; tap < 3; ++tap)
              ldb2(slot(4 + j) + tap * TILE_S, pl ? &tm_w0_lo : &tm_w0_hi, &full[4 + j], tap * 16, w0_row);
            j = (j + 1) & 3;
          }
        }
        if (F8) {
          for (int G = FUSED0 ? 6 : 0; G < 8; ++G)
            for (int it = 0; it < 4; ++it) {
              next_slot();
              if (it < 2) ldb2(slot(4 + j), &tm_w1_hi, &full[4 + j], (2 * G + it) * 64, w1_row);
              else ldb2(slot(4 + j), it == 2 ? &tm_w1_h8 : &tm_w1_l8, &full[4 + j], G * 128, w1_row);
              j = (j + 1) & 3;
            }
        } else {
          for (int kb = FUSED0 ? 12 : 0; kb < 16; ++kb)
            for (int pl = 0; pl < PL; ++pl) {
              next_slot();
              ldb2(slot(4 + j), pl ? &tm_w1_lo : &tm_w1_hi, &full[4 + j], kb * 64, w1_row);
              j = (j + 1) & 3;
            }
        }
      }
      if (a.has_res) {
        if (F8) {
          for (int grp = 0; grp < 2; ++grp)
            for (int it = 0; it < 4; ++it) {          // two fp16 tiles, then the e5m2 hi*2^-P and lo*2^Q tiles of the group
              next_slot();
              if (it < 2) ldb2(slot(4 + j), &tm_w2_hi, &full[4 + j], (2 * grp + it) * 64, w2_row);
              else ldb2(slot(4 + j), it == 2 ? &tm_w2_lo : &tm_w2_l8, &full[4 + j], grp * 128, w2_row);
              j = (j + 1) & 3;
            }
        } else {
          for (int kb = 0; kb < 4; ++kb)
            for (int pl = 0; pl < PL2; ++pl) {
              next_slot();
              ldb2(slot(4 + j), pl ? &tm_w2_lo : &tm_w2_hi, &full[4 + j], kb * 64, w2_row);
              j = (j + 1) & 3;
            }
        }
      }
    }
  } else if (warp == 3 && lane == 0) {
    // ---------------- folded-`end` weight tiles, once per CTA (N = 32 per pair: the leader stages the 16 real rows, the
    // follower the 16 rows that follow them in w2 - they only feed accumulator columns nobody reads)
    arm(wse_full, 4 * 2048 * PL2);
    const int row = a.w2_row0 + 256 + (int)rank * 16;
    for (int kb = 0; kb < 4; ++kb) {
      ldb2(wse(0, kb), &tm_wse_hi, wse_full, kb * 64, row);
      if (X3 && !F8) ldb2(wse(1, kb), &tm_wse_lo, wse_full, kb * 64, row);
    }
    if (F8)       // e5m2 planes of the folded-`end` rows: [16 rows x 128 B] per 128-channel group
      for (int grp = 0; grp < 2; ++grp) {
        ldb2(wse(1, grp), &tm_wse_lo, wse_full, grp * 128, row);
        ldb2(wse(1, 2 + grp), &tm_wse_l8, wse_full, grp * 128, row);
      }
  } else if (warp == 1 && lane == 0 && leader) {
    // ---------------- MMA issuer (leader CTA only)
    int sa = 0, jb = 0; uint32_t cm = 0;
    auto wait_full = [&](int bar) {               // bar: barrier index (A slot i -> i, B slot j -> 4 + j)
      mbar_wait(&full[bar], (cm >> bar) & 1u);
      cm ^= 1u << bar;
    };
    auto commit = [&](uint64_t* bar) { umma_commit_2sm(bar); };
    uint32_t par = 0;
    bool wse_seen = false;
    int it_no = 0;
    long long* tdbg = a.dbg ? a.dbg + (size_t)blockIdx.x * PS_DBG_STRIDE + 4 : nullptr;
    for (int p = cluster_id; p < n_pairs(); p += n_clusters, par ^= 1u, ++it_no) {
      const bool stamp = tdbg && it_no == 2;
      for (int g = 0; g < 2; ++g) {
        if (stamp) tdbg[3 * g] = clock64();
        // region R_g is free once the previous tile's epilogues (both CTAs) have read it
        mbar_wait_cluster(&r_free[g], par ^ 1u);
        tc_fence_after_sync();
        if (stamp) tdbg[3 * g + 1] = clock64();
        const uint32_t d = tmem + g * 256;
        if (FUSED0) {
          // x part of layer 0: 3 taps x (hi*hi [+ lo*hi + hi*lo]) K = 16 MMAs on the 32B-swizzled 4-KB tiles
          const int sa_hi = sa; wait_full(sa); sa = (sa + 1) & 3;
          int sa_lo = sa_hi;
          if (X3) { sa_lo = sa; wait_full(sa); sa = (sa + 1) & 3; }
          const int jb_hi = jb; wait_full(4 + jb); jb = (jb + 1) & 3;
          int jb_lo = jb_hi;
          if (X3) { jb_lo = jb; wait_full(4 + jb); jb = (jb + 1) & 3; }
          tc_fence_after_sync();
          const uint32_t a_hi = smem_u32(slot(sa_hi)), a_lo = smem_u32(slot(sa_lo));
          const uint32_t b_hi = smem_u32(slot(4 + jb_hi)), b_lo = smem_u32(slot(4 + jb_lo));
#pragma unroll
          for (int tap = 0; tap < 3; ++tap) {
            const uint32_t o = tap * TILE_S;
            umma_bf16_2sm(d, umma_desc_sw32(a_hi + o), umma_desc_sw32(b_hi + o), ID256, tap ? 1u : 0u);
            if (X3) {
              umma_bf16_2sm(d, umma_desc_sw32(a_lo + o), umma_desc_sw32(b_hi + o), ID256, 1u);
              umma_bf16_2sm(d, umma_desc_sw32(a_hi + o), umma_desc_sw32(b_lo + o), ID256, 1u);
            }
          }
          commit(&empty[4 + jb_hi]); commit(&empty[sa_hi]);
          if (X3) { commit(&empty[4 + jb_lo]); commit(&empty[sa_lo]); }
        }
        if (F8) {
          for (int G = FUSED0 ? 6 : 0; G < 8; ++G)
            for (int it = 0; it < 4; ++it) {
              const int sa_cur = sa; wait_full(sa); sa = (sa + 1) & 3;
              const int jb_cur = jb; wait_full(4 + jb); jb = (jb + 1) & 3;
              tc_fence_after_sync();
              if (it < 2) kblk(smem_u32(slot(sa_cur)), smem_u32(slot(4 + jb_cur)), d, ID256, G == 0 && it == 0);      // fused0 starts at G = 6: accumulates
              else kblk8(smem_u32(slot(sa_cur)), smem_u32(slot(4 + jb_cur)), d, IDE256);
              commit(&empty[4 + jb_cur]);
              commit(&empty[sa_cur]);
            }
        } else {
          for (int kb = FUSED0 ? 12 : 0; kb < 16; ++kb) {
            const int sa_hi = sa; wait_full(sa); sa = (sa + 1) & 3;
            int sa_lo = 0;
            if (NPASS == 3) { sa_lo = sa; wait_full(sa); sa = (sa + 1) & 3; }
            const int jb_hi = jb; wait_full(4 + jb); jb = (jb + 1) & 3;
            tc_fence_after_sync();
            kblk(smem_u32(slot(sa_hi)), smem_u32(slot(4 + jb_hi)), d, ID256, kb == 0);
            if (NPASS == 3) {
              kblk(smem_u32(slot(sa_lo)), smem_u32(slot(4 + jb_hi)), d, ID256, false);     // lo * hi
              commit(&empty[4 + jb_hi]);
              commit(&empty[sa_lo]);
              const int jb_lo = jb; wait_full(4 + jb); jb = (jb + 1) & 3;
              tc_fence_after_sync();
              kblk(smem_u32(slot(sa_hi)), smem_u32(slot(4 + jb_lo)), d, ID256, false);     // hi * lo
              commit(&empty[4 + jb_lo]);
            } else {
              commit(&empty[4 + jb_hi]);
            }
            commit(&empty[sa_hi]);
          }
        }
        commit(&acc_full[g]);
        if (stamp) tdbg[3 * g + 2] = clock64();
      }
      // GEMM2: [res | folded end] = acts x W2^T; A hi from TMEM (".ts"), lo / e5m2 planes from units 8..11.
      // Channels [0, 128) of acts come from sweep 0's gate, which finished long ago: their folded-`end` MMAs (N = 32,
      // accumulator R0[32, 64), weights resident) are issued FIRST, under the gate of sweep 1; the res MMAs (whose
      // accumulator R1 the gate of sweep 1 is still reading) and the second half follow once acts_ready fires.
      if (!wse_seen) { mbar_wait(wse_full, 0); wse_seen = true; }
      const uint32_t dres = tmem + P_D_RES, d32 = tmem + P_D_EO;
      auto gemm2 = [&](int half0, int half1, bool do_res, bool end_half0, bool end_half1) {
        if (F8) {
          for (int grp = half0; grp < half1; ++grp) {
            const bool do_end = grp == 0 ? end_half0 : end_half1;
            for (int it = 0; it < 4; ++it) {
              uint32_t r = 0; int jb_cur = 0;
              if (do_res) { jb_cur = jb; wait_full(4 + jb); jb = (jb + 1) & 3; tc_fence_after_sync(); r = smem_u32(slot(4 + jb_cur)); }
              if (it < 2) {
                const int kb = 2 * grp + it;
                const uint32_t wv = smem_u32(wse(0, kb));
#pragma unroll
                for (int k = 0; k < 4; ++k) {
                  const uint32_t o = 32 * k, acc = (kb | k) ? 1u : 0u, a_t = tmem + P_ACOL(kb * 4 + k);
                  if (do_res) umma_bf16_ts_2sm(dres, a_t, umma_desc_sw128(r + o), ID256, acc);
                  if (do_end) umma_bf16_ts_2sm(d32, a_t, umma_desc_sw128(wv + o), ID32, acc);
                }
              } else {
                const uint32_t av = smem_u32(slot(8 + 2 * (it - 2) + grp)), wv = smem_u32(wse(1, 2 * (it - 2) + grp));
#pragma unroll
                for (int k = 0; k < 4; ++k) {
                  const uint32_t o = 32 * k;
                  if (do_res) umma_f8_2sm(dres, umma_desc_sw128(av + o), umma_desc_sw128(r + o), IDE256, 1u);
                  if (do_end) umma_f8_2sm(d32, umma_desc_sw128(av + o), umma_desc_sw128(wv + o), IDE32, 1u);
                }
              }
              if (do_res) commit(&empty[4 + jb_cur]);
            }
          }
        } else {
          for (int kb = 2 * half0; kb < 2 * half1; ++kb) {
            const bool do_end = kb < 2 ? end_half0 : end_half1;
            const uint32_t a_lo = smem_u32(slot(8 + kb));
            const uint32_t w_hi = smem_u32(wse(0, kb)), w_lo = smem_u32(wse(1, kb));
            uint32_t r_hi = 0, r_lo = 0;
            int jb_hi = 0, jb_lo = 0;
            if (do_res) {
              jb_hi = jb; wait_full(4 + jb); jb = (jb + 1) & 3;
              if (X3) { jb_lo = jb; wait_full(4 + jb); jb = (jb + 1) & 3; }
              tc_fence_after_sync();
              r_hi = smem_u32(slot(4 + jb_hi)); r_lo = smem_u32(slot(4 + jb_lo));
            }
#pragma unroll
            for (int k = 0; k < 4; ++k) {
              const uint32_t o = 32 * k, acc = (kb | k) ? 1u : 0u, a_t = tmem + P_ACOL(kb * 4 + k);
              if (do_res) umma_bf16_ts_2sm(dres, a_t, umma_desc_sw128(r_hi + o), ID256, acc);
              if (do_end) umma_bf16_ts_2sm(d32, a_t, umma_desc_sw128(w_hi + o), ID32, acc);
              if (X3) {
                if (do_res) umma_bf16_2sm(dres, umma_desc_sw128(a_lo + o), umma_desc_sw128(r_hi + o), ID256, 1u);
                if (do_end) umma_bf16_2sm(d32, umma_desc_sw128(a_lo + o), umma_desc_sw128(w_hi + o), ID32, 1u);
                if (do_res) umma_bf16_ts_2sm(dres, a_t, umma_desc_sw128(r_lo + o), ID256, 1u);
                if (do_end) umma_bf16_ts_2sm(d32, a_t, umma_desc_sw128(w_lo + o), ID32, 1u);
              }
            }
            if (do_res) {
              commit(&empty[4 + jb_hi]);
              if (X3) commit(&empty[4 + jb_lo]);
            }
          }
        }
      };
      mbar_wait_cluster(acts0_ready, par);
      tc_fence_after_sync();
      gemm2(0, 1, false, true, false);                 // `end` of channels [0, 128), under the gate of sweep 1
      mbar_wait_cluster(acts_ready, par);
      tc_fence_after_sync();
      if (stamp) tdbg[6] = clock64();
      gemm2(0, 2, a.has_res != 0, false, true);        // res of all channels, `end` of channels [128, 256)
      commit(acc2_full);
      if (stamp) tdbg[7] = clock64();
    }
  } else if (warp >= 4) {
    // ---------------- epilogue warps: TMEM lane quarter = warp % 4 (one group-step per lane), column group
    // h = (warp - 4) / 4: 64 of the 128 channels of each sweep in the gate, channels [128h, 128h+128) in the res epilogue
    const int quarter = warp & 3, h = (warp - 4) >> 2, row = quarter * 32 + lane;
    const uint32_t trow = tmem + ((uint32_t)(quarter * 32) << 16);
    const bool ldr = quarter == 0 && lane == 0;                // issues this column group's TMA loads / stores
    const float4* b1t = reinterpret_cast<const float4*>(b1s);
    const float4* b1g = reinterpret_cast<const float4*>(b1s + 256);
    const float4* b2v = reinterpret_cast<const float4*>(b2s);
    uint8_t* const u_hi = slot(8 + 2 * h);
    uint8_t* const u_lo = slot(9 + 2 * h);
    {   // biases -> smem, once per CTA; gate biases pre-multiplied by the argument scales of gate_fused
      const int e = threadIdx.x - 128;
      b1s[e] = __ldg(a.b1 + e) * GateK<NPASS>::KA; b1s[256 + e] = __ldg(a.b1 + 256 + e) * GateK<NPASS>::KB;
      b2s[e] = __ldg(a.b2 + e);
      if (FUSED0) {          // start conv of this flow: S [256][8] (columns >= n_half are zero) and its bias
        const float4* sw = reinterpret_cast<const float4*>(a.start_w + (size_t)e * 8);
        reinterpret_cast<float4*>(s_tab)[2 * e] = __ldg(sw); reinterpret_cast<float4*>(s_tab)[2 * e + 1] = __ldg(sw + 1);
        s_bias[e] = __ldg(a.start_b + e);
      }
      asm volatile("bar.sync 1, %0;" ::"n"(P_EPI_THREADS) : "memory");
    }
    const uint32_t r0_bar = mapa_shared(&r_free[0], 0), r1_bar = mapa_shared(&r_free[1], 0), ar_bar = mapa_shared(acts_ready, 0);
    const uint32_t a0_bar = mapa_shared(acts0_ready, 0);
    long long t_start = 0;
    if (a.dbg && warp == 4 && lane == 0) t_start = clock64();
    int n_tiles = 0;
    uint32_t par = 0, xph = 0;
    int b_cur = 0;
    for (int p = cluster_id; p < n_pairs(); p += n_clusters, par ^= 1u, ++n_tiles) {
      int b, t0; tile_of(p, b, t0);
      const bool valid = t0 + row < (RAGGED ? __ldg(a.len + b) * a.P : a.Tp);
      const size_t m = (size_t)b * a.Tp + (size_t)min(t0 + row, a.Tp - 1);
      if (a.b1_bstride != 0 && b != b_cur) {    // per-utterance gate bias (b is uniform over the CTA): reload on a change
        b_cur = b;
        asm volatile("bar.sync 1, %0;" ::"n"(P_EPI_THREADS) : "memory");     // every warp is past the previous tile's gates
        const int e = threadIdx.x - 128;
        const float* bb = a.b1 + (size_t)b * a.b1_bstride;
        b1s[e] = __ldg(bb + e) * GateK<NPASS>::KA; b1s[256 + e] = __ldg(bb + 256 + e) * GateK<NPASS>::KB;
        asm volatile("bar.sync 1, %0;" ::"n"(P_EPI_THREADS) : "memory");
      }
      auto load_xold = [&](int blk) {          // ldr only: x_old (centre tap) tiles of a 64-channel block -> staging
        mbar_arrive_expect_tx(&xold_full[h], 2 * TILE_A);
        tma_load_3d(u_hi, &tm_x_hi, &xold_full[h], blk * 64, t0, b);
        tma_load_3d(u_lo, &tm_x_lo, &xold_full[h], blk * 64, t0, b);
      };
      // bf16: units 8..11 hold no gate output, so the first x_old block can be fetched a whole tile ahead
      if (!X3 && a.has_res && !FUSED0 && ldr) load_xold(2 * h);

      // ---- gates: acts = tanh(pre[:, :C]) * sigmoid(pre[:, C:]) (glow.py:34-41), sweep by sweep
      const bool stamp = a.dbg && n_tiles == 2 && warp == 4 && lane == 0;
      long long* edbg = a.dbg ? a.dbg + (size_t)blockIdx.x * PS_DBG_STRIDE + 16 : nullptr;
#pragma unroll 1
      for (int g = 0; g < 2; ++g) {
        mbar_wait(&acc_full[g], par);
        tc_fence_after_sync();
        if (stamp) edbg[2 * g] = clock64();
        const uint32_t treg = trow + g * 256;
        uint32_t buf[2][32];
        const int i0 = 4 * h;                                       // 16-channel chunk of the sweep: i0 .. i0+3
        tmem_issue16x2(treg + i0 * 16, treg + 128 + i0 * 16, buf[0]);
#pragma unroll
        for (int jj = 0; jj < 4; ++jj) {
          const int c = 8 * g + i0 + jj;                            // chunk of the 256 channels
          uint32_t* cur = buf[jj & 1];
          tmem_wait32(cur);
          if (jj + 1 < 4) tmem_issue16x2(treg + (i0 + jj + 1) * 16, treg + 128 + (i0 + jj + 1) * 16, buf[(jj + 1) & 1]);
          float act[16];
#pragma unroll
          for (int q = 0; q < 4; ++q) {
            const float4 bt = b1t[c * 4 + q], bs = b1g[c * 4 + q];
            act[4 * q + 0] = gate_fused<NPASS>(__uint_as_float(cur[4 * q + 0]), __uint_as_float(cur[16 + 4 * q + 0]), bt.x, bs.x);
            act[4 * q + 1] = gate_fused<NPASS>(__uint_as_float(cur[4 * q + 1]), __uint_as_float(cur[16 + 4 * q + 1]), bt.y, bs.y);
            act[4 * q + 2] = gate_fused<NPASS>(__uint_as_float(cur[4 * q + 2]), __uint_as_float(cur[16 + 4 * q + 2]), bt.z, bs.z);
            act[4 * q + 3] = gate_fused<NPASS>(__uint_as_float(cur[4 * q + 3]), __uint_as_float(cur[16 + 4 * q + 3]), bt.w, bs.w);
          }
          if (F8) store_split16_tmem_f8(act, trow + P_ACOL(c), slot(8 + (c >> 3)), slot(10 + (c >> 3)), row, c & 7);
          else store_split16_tmem<X3, false>(act, trow + P_ACOL(c), slot(8 + (c >> 2)), row, (c & 3) * 2);
        }
        if (stamp) edbg[2 * g + 1] = clock64();
        if (g == 0) {                          // acts of channels [0, 128) are complete: their `end` MMAs may start
          tmem_wait_st();
          tc_fence_before_sync();
          fence_proxy_async_smem();
          __syncwarp();
          if (lane == 0) { if (leader) mbar_arrive(acts0_ready); else mbar_arrive_cluster(a0_bar); }
        }
      }
      tmem_wait_st();
      tc_fence_before_sync();
      fence_proxy_async_smem();
      __syncwarp();
      if (lane == 0) {
        if (leader) mbar_arrive(acts_ready); else mbar_arrive_cluster(ar_bar);
        if (!a.has_res) { if (leader) mbar_arrive(&r_free[1]); else mbar_arrive_cluster(r1_bar); }   // R1 fully consumed
      }

      // prefetch this row's folded-`end` accumulator while GEMM2 runs
      float4 eold[4];
      const bool eo_mine = h == 0 || a.eo_pitch == 32;     // wide layout: column group 1 owns outputs [16, 32)
      if (eo_mine) {
        const float4* e = reinterpret_cast<const float4*>(a.first ? a.eo_b + 16 * h : a.eo + m * a.eo_pitch + 16 * h);
#pragma unroll
        for (int q = 0; q < 4; ++q) eold[q] = __ldg(e + q);
      }

      // ---- res / skip
      mbar_wait(acc2_full, par);
      tc_fence_after_sync();
      if (stamp) edbg[4] = clock64();
      uint32_t sk[16];
      if (eo_mine) {                                             // first of all: release R0 to the next tile's sweep 0
        tmem_issue16(trow + P_D_EO + 16 * h, sk);
        tmem_wait16(sk);
        tc_fence_before_sync();
        __syncwarp();
        if (lane == 0) { if (leader) mbar_arrive(&r_free[0]); else mbar_arrive_cluster(r0_bar); }   // R0: acts consumed by GEMM2, `end` read
      }
      if (X3 && a.has_res && !FUSED0 && ldr) load_xold(2 * h);  // GEMM2 no longer reads units 8..11
      if (eo_mine) {
        if (valid) {
          float4* e = reinterpret_cast<float4*>(a.eo + m * a.eo_pitch + 16 * h);
#pragma unroll
          for (int q = 0; q < 4; ++q)
            e[q] = make_float4(eold[q].x + __uint_as_float(sk[4 * q]), eold[q].y + __uint_as_float(sk[4 * q + 1]),
                               eold[q].z + __uint_as_float(sk[4 * q + 2]), eold[q].w + __uint_as_float(sk[4 * q + 3]));
        }
      }
      if (a.has_res) {
        uint32_t buf[2][16];
        const int c0 = 8 * h;
        float av[8];                                 // fused0: this row's coupling input audio_0 (fp32, exact)
        if (FUSED0) {
          const float* ar = a.audio + m * a.G + a.a_off;
#pragma unroll
          for (int j = 0; j < 8; ++j) av[j] = (valid && j < a.a_nh) ? __ldg(ar + j) : 0.f;
        }
        tmem_issue16(trow + P_D_RES + c0 * 16, buf[0]);
#pragma unroll
        for (int i = 0; i < 8; ++i) {
          const int c = c0 + i;
          uint32_t* cur = buf[i & 1];
          if ((i & 3) == 0 && !FUSED0) { mbar_wait(&xold_full[h], xph); xph ^= 1u; }   // x_old tiles of this 64-channel block have landed
          tmem_wait16(cur);
          if (i + 1 < 8) tmem_issue16(trow + P_D_RES + (c + 1) * 16, buf[(i + 1) & 1]);
          else {                                                           // last TMEM read of this warp: release R1
            tc_fence_before_sync();
            __syncwarp();
            if (lane == 0) { if (leader) mbar_arrive(&r_free[1]); else mbar_arrive_cluster(r1_bar); }
          }
          const uint32_t o0 = sw128_offset(row, (c & 3) * 2), o1 = sw128_offset(row, (c & 3) * 2 + 1);
          float r[16];
#pragma unroll
          for (int q = 0; q < 4; ++q) {
            const float4 bb = b2v[c * 4 + q];
            r[4 * q] = __uint_as_float(cur[4 * q]) + bb.x; r[4 * q + 1] = __uint_as_float(cur[4 * q + 1]) + bb.y;
            r[4 * q + 2] = __uint_as_float(cur[4 * q + 2]) + bb.z; r[4 * q + 3] = __uint_as_float(cur[4 * q + 3]) + bb.w;
          }
          if (FUSED0) {
            // x_old = start(audio_0) = S a + b in fp32 (glow.py:189), never stored: 8 FMAs per channel, S broadcast from smem
#pragma unroll
            for (int q = 0; q < 16; ++q) {
              const float4 s0 = reinterpret_cast<const float4*>(s_tab)[2 * (c * 16 + q)], s1 = reinterpret_cast<const float4*>(s_tab)[2 * (c * 16 + q) + 1];
              float x = s_bias[c * 16 + q];
              x = fmaf(s0.x, av[0], x); x = fmaf(s0.y, av[1], x); x = fmaf(s0.z, av[2], x); x = fmaf(s0.w, av[3], x);
              x = fmaf(s1.x, av[4], x); x = fmaf(s1.y, av[5], x); x = fmaf(s1.z, av[6], x); x = fmaf(s1.w, av[7], x);
              r[q] += x;
            }
          } else {
            const uint4 h0 = *reinterpret_cast<const uint4*>(u_hi + o0), h1 = *reinterpret_cast<const uint4*>(u_hi + o1);
            const uint4 l0 = *reinterpret_cast<const uint4*>(u_lo + o0), l1 = *reinterpret_cast<const uint4*>(u_lo + o1);
            const uint32_t hw[8] = {h0.x, h0.y, h0.z, h0.w, h1.x, h1.y, h1.z, h1.w};
            const uint32_t lw[8] = {l0.x, l0.y, l0.z, l0.w, l1.x, l1.y, l1.z, l1.w};
#pragma unroll
            for (int j = 0; j < 8; ++j) {   // x_new = x_old(hi + lo) + res, glow.py:217
              float f0, f1, g0, g1;
              unpack2<F8>(hw[j], f0, f1); unpack2<F8>(lw[j], g0, g1);
              r[2 * j] += f0 + g0;
              r[2 * j + 1] += f1 + g1;
            }
          }
          if (RAGGED && !valid)      // padding of utterance b: zeros in every plane keep the taps of later layers exact
#pragma unroll
            for (int j = 0; j < 16; ++j) r[j] = 0.f;
          if (F8) {
            uint32_t nh[8], nl[8], l8[4], h8[4];
            if (a.range_flag) {      // the layer that consumes this x has no residual: an Inf here would not reach the waveform
              float mx = 0.f;
#pragma unroll
              for (int j = 0; j < 16; ++j) mx = fmaxf(mx, fabsf(r[j]));
              if (valid && !(mx < 65504.f)) atomicOr(a.range_flag, 2);
            }
            split16_f8_words(r, nh, nl, l8, h8);
            *reinterpret_cast<uint4*>(u_hi + o0) = make_uint4(nh[0], nh[1], nh[2], nh[3]);
            *reinterpret_cast<uint4*>(u_hi + o1) = make_uint4(nh[4], nh[5], nh[6], nh[7]);
            *reinterpret_cast<uint4*>(u_lo + o0) = make_uint4(nl[0], nl[1], nl[2], nl[3]);
            *reinterpret_cast<uint4*>(u_lo + o1) = make_uint4(nl[4], nl[5], nl[6], nl[7]);
            // the two e5m2 planes: 16 bytes per row and chunk, straight to HBM (L2 merges the sectors); RAGGED also
            // stores the zeros of the padded rows below T'_max
            if (RAGGED ? t0 + row < a.Tp : valid) {
              *reinterpret_cast<uint4*>(a.xo_l8 + m * 256 + c * 16) = make_uint4(l8[0], l8[1], l8[2], l8[3]);
              *reinterpret_cast<uint4*>(a.xo_h8 + m * 256 + c * 16) = make_uint4(h8[0], h8[1], h8[2], h8[3]);
            }
          } else {
            store_split16<true>(r, u_hi, u_lo, row, (c & 3) * 2);     // in place (same thread, same addresses)
          }
          if ((i & 3) == 3) {
            // one 64-channel block (hi + lo) is final: store it; the first block's buffers then take the second block
            fence_proxy_async_smem();
            asm volatile("bar.sync %0, 128;" ::"r"(2 + h) : "memory");
            if (ldr) {
              const int blk = c >> 2;
              tma_store_3d(&tm_xo_hi, u_hi, blk * 64, t0, b);
              tma_store_3d(&tm_xo_lo, u_lo, blk * 64, t0, b);
              tma_store_commit();
              tma_store_wait_read();
              if (i == 3 && !FUSED0) load_xold(blk + 1);
            }
            // fused0 has no x_old load (whose mbarrier orders the re-use of the staging tiles in the other path): nobody
            // may overwrite them before the store above has read them
            if (FUSED0 && i == 3) asm volatile("bar.sync %0, 128;" ::"r"(2 + h) : "memory");
          }
        }
        // the staging units become gate outputs of the next tile (written by BOTH column groups)
        asm volatile("bar.sync 1, %0;" ::"n"(P_EPI_THREADS) : "memory");
      }
      if (stamp) edbg[5] = clock64();
    }
    tc_fence_before_sync();
    if (a.dbg && warp == 4 && lane == 0) {
      long long* d = a.dbg + (size_t)blockIdx.x * PS_DBG_STRIDE;
      d[0] = t_start; d[1] = clock64(); d[2] = n_tiles;
    }
  }
  __syncthreads();
  cluster_sync_all();                              // the pair releases TMEM together; no CTA exits with peer traffic pending
  if (warp == 1) { __syncwarp(); tmem_dealloc_2sm(tmem, 512); }
}

// ------------------------------------------------------------------------------------------
// host: tensor maps are encoded once per (buffers, shape, mode) and re-used by every layer launch that sees the same
// buffers (the ping-pong x planes give two entries per infer call) - 12-21 cuTensorMapEncodeTiled calls per launch before.
// ------------------------------------------------------------------------------------------
struct PsMaps {
  CUtensorMap x_hi, x_lo, h_hi, h_lo, w1_hi, w1_lo, w2_hi, w2_lo, wse_hi, wse_lo, xo_hi, xo_lo;
  CUtensorMap x_l8, x_h8, h_l8, h_h8, w1_h8, w1_l8, w2_l8, wse_l8;
  CUtensorMap a0_hi, a0_lo, w0_hi, w0_lo;
};
struct PsKey {
  const void *x_in, *x_out, *h2, *w1, *w2, *w1b, *w2b, *a0, *w0;
  int B, Tp, C, H, K1, N2, npass; long long fl;
};
struct PsEntry { PsKey key; PsMaps maps; bool used; unsigned long long stamp; };
constexpr int PS_CACHE = 8;
thread_local PsEntry g_cache[PS_CACHE];
thread_local unsigned long long g_stamp = 0;

int build_maps(const Dims& d, const cwg_weights* w, int npass, const __nv_bfloat16* x_in, __nv_bfloat16* x_out,
               const __nv_bfloat16* h2, const void* a0, PsMaps* m) {
  const size_t plane = (size_t)d.BT * d.C, hplane = (size_t)d.BT * d.H;
  const uint64_t fl = (uint64_t)d.F * d.L;
  if (int r = map_act(&m->x_hi, x_in, d.C, d.Tp, d.B)) return r;
  if (int r = map_act(&m->x_lo, x_in + plane, d.C, d.Tp, d.B)) return r;
  if (int r = map_act(&m->h_hi, h2, d.H, d.Tp, d.B)) return r;
  if (int r = map_act(&m->h_lo, npass == 2 ? h2 : h2 + hplane, d.H, d.Tp, d.B)) return r;
  if (int r = map_act(&m->xo_hi, x_out, d.C, d.Tp, d.B)) return r;
  if (int r = map_act(&m->xo_lo, x_out + plane, d.C, d.Tp, d.B)) return r;
  // weight tiles: every CTA of a pair loads 128 of the 256 N rows
  if (int r = map_2d(&m->w1_hi, w->w1_hi, d.K1, fl * 2 * d.C, 128)) return r;
  if (int r = map_2d(&m->w2_hi, w->w2_hi, d.C, fl * d.N2, 128)) return r;
  if (int r = map_2d(&m->wse_hi, w->w2_hi, d.C, fl * d.N2, 16)) return r;
  if (npass == 2) {
    // x = [fp16 hi][fp16 lo][e5m2 lo*2^P][e5m2 hi*2^-Q], H2 = [fp16 hi][e5m2 lo*2^P][e5m2 hi*2^-Q]
    const uint8_t* xi8 = reinterpret_cast<const uint8_t*>(x_in) + 4 * plane;
    const uint8_t* h8 = reinterpret_cast<const uint8_t*>(h2) + 2 * hplane;
    m->w1_lo = m->w1_hi;                                           // f16f8 has no 16-bit lo plane of the weights
    if (int r = map_act8(&m->x_l8, xi8, d.C, d.Tp, d.B)) return r;
    if (int r = map_act8(&m->x_h8, xi8 + plane, d.C, d.Tp, d.B)) return r;
    if (int r = map_act8(&m->h_l8, h8, d.H, d.Tp, d.B)) return r;
    if (int r = map_act8(&m->h_h8, h8 + hplane, d.H, d.Tp, d.B)) return r;
    if (int r = map_2d8(&m->w1_h8, w->w1_h8, d.K1, fl * 2 * d.C, 128)) return r;
    if (int r = map_2d8(&m->w1_l8, w->w1_l8, d.K1, fl * 2 * d.C, 128)) return r;
    if (int r = map_2d8(&m->w2_lo, w->w2_h8, d.C, fl * d.N2, 128)) return r;
    if (int r = map_2d8(&m->w2_l8, w->w2_l8, d.C, fl * d.N2, 128)) return r;
    if (int r = map_2d8(&m->wse_lo, w->w2_h8, d.C, fl * d.N2, 16)) return r;
    if (int r = map_2d8(&m->wse_l8, w->w2_l8, d.C, fl * d.N2, 16)) return r;
  } else {
    if (int r = map_2d(&m->w1_lo, w->w1_lo, d.K1, fl * 2 * d.C, 128)) return r;
    if (int r = map_2d(&m->w2_lo, w->w2_lo, d.C, fl * d.N2, 128)) return r;
    if (int r = map_2d(&m->wse_lo, w->w2_lo, d.C, fl * d.N2, 16)) return r;
    m->x_l8 = m->x_h8 = m->h_l8 = m->h_h8 = m->w1_h8 = m->w1_l8 = m->w2_l8 = m->wse_l8 = m->x_hi;
  }
  if (a0) {      // layer-0 fold: planes hi then lo, each [B*T'][16] 16-bit; folded weights [F][2C][48]
    const uint16_t* ap = reinterpret_cast<const uint16_t*>(a0);
    if (int r = map_a0(&m->a0_hi, ap, d.Tp, d.B)) return r;
    if (int r = map_a0(&m->a0_lo, ap + (size_t)d.BT * 16, d.Tp, d.B)) return r;
    if (int r = map_w0(&m->w0_hi, w->w0_hi, (uint64_t)d.F * 2 * d.C)) return r;
    if (int r = map_w0(&m->w0_lo, w->w0_lo, (uint64_t)d.F * 2 * d.C)) return r;
  } else {
    m->a0_hi = m->a0_lo = m->w0_hi = m->w0_lo = m->x_hi;
  }
  return 0;
}

int get_maps(const Dims& d, const cwg_weights* w, int npass, const __nv_bfloat16* x_in, __nv_bfloat16* x_out,
             const __nv_bfloat16* h2, const void* a0, const PsMaps** out) {
  PsKey k;
  memset(&k, 0, sizeof(k));
  k.x_in = x_in; k.x_out = x_out; k.h2 = h2; k.w1 = w->w1_hi; k.w2 = w->w2_hi;
  k.w1b = npass == 2 ? (const void*)w->w1_h8 : (const void*)w->w1_lo;
  k.w2b = npass == 2 ? (const void*)w->w2_h8 : (const void*)w->w2_lo;
  k.a0 = a0; k.w0 = a0 ? (const void*)w->w0_hi : nullptr;
  k.B = d.B; k.Tp = d.Tp; k.C = d.C; k.H = d.H; k.K1 = d.K1; k.N2 = d.N2; k.npass = npass; k.fl = (long long)d.F * d.L;
  int victim = 0;
  for (int i = 0; i < PS_CACHE; ++i) {
    if (g_cache[i].used && memcmp(&g_cache[i].key, &k, sizeof(k)) == 0) {
      g_cache[i].stamp = ++g_stamp;
      *out = &g_cache[i].maps;
      return 0;
    }
    if (!g_cache[i].used) victim = i;
    else if (g_cache[victim].used && g_cache[i].stamp < g_cache[victim].stamp) victim = i;
  }
  PsEntry& e = g_cache[victim];
  e.used = false;
  if (int r = build_maps(d, w, npass, x_in, x_out, h2, a0, &e.maps)) return r;
  e.key = k; e.used = true; e.stamp = ++g_stamp;
  *out = &e.maps;
  return 0;
}

template <int NPASS, bool FUSED0, bool RAGGED>
int max_clusters(int* out) {
  static int cached = 0;                           // per process; all GPUs of a box are the same part
  constexpr int smem = RAGGED ? P_SMEM_R : P_SMEM;
  if (cached == 0) {
    CWG_CHECK_CUDA(cudaFuncSetAttribute(k_layer_ps<NPASS, FUSED0, RAGGED>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
    cudaLaunchConfig_t lc{};
    lc.gridDim = dim3(2 * 148); lc.blockDim = dim3(P_THREADS); lc.dynamicSmemBytes = smem;
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeClusterDimension;
    at[0].val.clusterDim.x = 2; at[0].val.clusterDim.y = 1; at[0].val.clusterDim.z = 1;
    lc.attrs = at; lc.numAttrs = 1;
    int n = 0;
    CWG_CHECK_CUDA(cudaOccupancyMaxActiveClusters(&n, k_layer_ps<NPASS, FUSED0, RAGGED>, &lc));
    CWG_REQUIRE(n >= 1, "k_layer_ps does not fit on this device (cudaOccupancyMaxActiveClusters = %d)", n);
    cached = n;
  }
  *out = cached;
  return 0;
}

template <bool RAGGED>
int max_clusters(int npass, bool f0, int* out) {
  return npass == 3 ? (f0 ? max_clusters<3, true, RAGGED>(out) : max_clusters<3, false, RAGGED>(out))
       : npass == 2 ? (f0 ? max_clusters<2, true, RAGGED>(out) : max_clusters<2, false, RAGGED>(out))
                    : (f0 ? max_clusters<1, true, RAGGED>(out) : max_clusters<1, false, RAGGED>(out));
}

long long* g_ps_dbg = nullptr;

}  // namespace

void debug_set_ps_timing(long long* buf) { g_ps_dbg = buf; }

int launch_layer_ps(const Dims& d, const cwg_weights* w, int npass, int flow, int layer,
                    const __nv_bfloat16* x_in, __nv_bfloat16* x_out, const __nv_bfloat16* h2,
                    float* eo, cudaStream_t s, const void* a0, const float* audio, int a_off, int a_nh,
                    const int* rag_len, const int* rag_prefix) {
  // a0 != NULL (layer 0 only): the layer-0 fold - x_in is not read; see PsArgs::fused0
  // rag_len / rag_prefix != NULL: the ragged form (PsArgs::len / prefix, both device arrays; d.B <= CWG_RAGGED_MAX_BATCH)
  const bool ragged = rag_len != nullptr;
  CWG_REQUIRE(!ragged || (rag_prefix && d.B <= CWG_RAGGED_MAX_BATCH), "ragged layer: bad arguments");
  CWG_REQUIRE(a0 == nullptr || (layer == 0 && w->w0_hi && w->w0_lo && audio && d.L >= 2 && d.MG == 16), "layer-0 fold: bad arguments");
  const PsMaps* m = nullptr;
  if (int r = get_maps(d, w, npass, x_in, x_out, h2, a0, &m)) return r;
  const size_t plane = (size_t)d.BT * d.C;
  const size_t idx = (size_t)flow * d.L + layer;
  PsArgs a{};
  a.b1 = w->b1 + idx * 2 * d.C; a.b2 = w->b2 + idx * d.C; a.eo_b = w->eo_b + (size_t)flow * d.MG;
  if (d.b1_batch) { a.b1 = d.b1_batch + idx * 2 * d.C; a.b1_bstride = (long long)d.F * d.L * 2 * d.C; }
  a.eo = eo; a.eo_pitch = d.MG;
  a.xo_l8 = reinterpret_cast<uint8_t*>(x_out) + 4 * plane; a.xo_h8 = a.xo_l8 + plane;
  a.Tp = d.Tp; a.dil = 1 << layer;
  a.w1_row0 = (int)(idx * 2 * d.C); a.w2_row0 = (int)(idx * d.N2);
  a.has_res = layer < d.L - 1; a.first = layer == 0;
  const int tiles = (d.Tp + 127) / 128;
  a.pairs_per_utt = (tiles + 1) / 2;                // an odd tile count gets one tile fully past T' (TMA zero-fills / clips)
  a.n_pairs = a.pairs_per_utt * d.B;
  a.dbg = g_ps_dbg;
  a.fused0 = a0 != nullptr; a.audio = audio; a.G = d.G; a.a_off = a_off; a.a_nh = a_nh;
  a.start_w = w->start_w + (size_t)flow * d.C * (d.MG / 2); a.start_b = w->start_b + (size_t)flow * d.C;
  a.w0_row0 = flow * 2 * d.C;
  a.range_flag = (npass == 2 && (layer == d.L - 2 || range_all_layers())) ? range_flag() : nullptr;
  a.len = rag_len; a.prefix = rag_prefix; a.nb = d.B; a.P = d.P;
  int ncl = 0;
  const bool f0 = a0 != nullptr;
  if (int r = ragged ? max_clusters<true>(npass, f0, &ncl) : max_clusters<false>(npass, f0, &ncl)) return r;
  if (ncl > a.n_pairs) ncl = a.n_pairs;            // ragged: the padded count bounds the device-side one
  cudaLaunchConfig_t lc{};
  lc.gridDim = dim3(2 * ncl); lc.blockDim = dim3(P_THREADS); lc.dynamicSmemBytes = ragged ? P_SMEM_R : P_SMEM; lc.stream = s;
  cudaLaunchAttribute at[1];
  at[0].id = cudaLaunchAttributeClusterDimension;
  at[0].val.clusterDim.x = 2; at[0].val.clusterDim.y = 1; at[0].val.clusterDim.z = 1;
  lc.attrs = at; lc.numAttrs = 1;
#define CWG_LAUNCH_PS(NP, F0)                                                                                          \
  CWG_CHECK_CUDA(cudaLaunchKernelEx(&lc, ragged ? k_layer_ps<NP, F0, true> : k_layer_ps<NP, F0, false>,               \
                                    m->x_hi, m->x_lo, m->h_hi, m->h_lo, m->w1_hi, m->w1_lo,                            \
                                    m->w2_hi, m->w2_lo, m->wse_hi, m->wse_lo, m->xo_hi, m->xo_lo, m->x_l8, m->x_h8,    \
                                    m->h_l8, m->h_h8, m->w1_h8, m->w1_l8, m->w2_l8, m->wse_l8, m->a0_hi, m->a0_lo,  \
                                    m->w0_hi, m->w0_lo, a))
  if (f0) { if (npass == 3) CWG_LAUNCH_PS(3, true); else if (npass == 2) CWG_LAUNCH_PS(2, true); else CWG_LAUNCH_PS(1, true); }
  else { if (npass == 3) CWG_LAUNCH_PS(3, false); else if (npass == 2) CWG_LAUNCH_PS(2, false); else CWG_LAUNCH_PS(1, false); }
#undef CWG_LAUNCH_PS
  return 0;
}

}  // namespace cwg
