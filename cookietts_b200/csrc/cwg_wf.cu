// WaveFlow (BASELINE config 5) on sm_100a: the autoregressive-over-height inverse of the reference's
// "ax" model.  Reference lines (CookieTTS/_4_mtw/waveglow/):
//   efficient_model_ax.py:279-357  WaveGlow.inverse              -> cwg_wf_infer
//   efficient_model_ax.py:171-182  _upsample_mels (interpolate)  -> k_wf_mel_up
//   efficient_modules.py:42-65     WaveFlowCoupling.inverse      -> row loop in cwg_wf_infer + k_wf_row
//   glow_ax.py:556-635             WN_2d.forward (conv queues)   -> k_wf_layer_tc (one launch per layer per row)
//   efficient_modules.py:360-403   PermuteHeight.inverse         -> column bookkeeping on the host (no data movement)
//
// One autoregressive row step of one layer is the same fused kernel shape as the 1-D WN layer
// (cwg_ps.cu): implicit GEMM over K = (kh rows) x (kw dilated taps) x C + padded mel, gate epilogue,
// res/skip GEMM, residual update.  The "conv queue" of the reference is a kernel_h-slot ring of each
// layer's input rows kept in HBM; rows that do not exist yet (zero queue) are simply skipped.
//
// Two in_layer layouts run on the tensor cores:
//   dense 3x3 (k_wf_layer_tc; a separable 3x3 is folded into it at pack time): K = 9 x C + mel.
//   depthwise-separable, kernel_h <= 7 x odd kernel_w <= 7 (k_wf_sep_tc; the layout of the reference author's
//   trained checkpoints, glow_ax.py:525-531): the depthwise conv runs on the CUDA cores inside the layer kernel
//   and writes its output straight into shared memory as the A operand of the pointwise GEMM, K = C + mel.
#include "cwg_tc_common.cuh"

namespace cwg {

using namespace sm100;
using namespace tc;

namespace {

constexpr int WF_C = 128, WF_KH = 3, WF_KW = 3, WF_HP = CWG_WF_COND_PAD;
constexpr int WF_K1 = WF_KH * WF_KW * WF_C + WF_HP;     // 1280
constexpr int WF_N2 = WF_C + CWG_EO_PAD;                // 144
constexpr int WF_TC_MAX_GROUP = 32;                    // squeeze height (only host arrays are sized by it)
constexpr int WF_SEP_MAX_KH = 7, WF_SEP_MAX_KW = 7;     // separable in_layers: kernel_h <= 7, odd kernel_w <= 7
constexpr uint32_t IDESC_N144 = umma_idesc_bf16(128, 144);

struct WfDims {
  int B, Tp, F, L, G, M, KH;
  long long BT;
};

// ------------------------------------------------------------------------------------------
// mel -> [B][T'][128] bf16 hi/lo: zero-extended by pad frames, interpolated to T' steps
// (F.interpolate(..., mode='linear', align_corners=True) or 'nearest'), channels padded to 128.
// ------------------------------------------------------------------------------------------
__global__ void k_wf_mel_up(const float* __restrict__ mel, __nv_bfloat16* __restrict__ hi, __nv_bfloat16* __restrict__ lo,
                            int B, int M, int frames, int frames_padded, int Tp, int linear) {
  long long n = (long long)B * Tp * WF_HP;
  long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  int c = (int)(i % WF_HP);
  long long m = i / WF_HP;
  int t = (int)(m % Tp), b = (int)(m / Tp);
  float v = 0.f;
  if (c < M) {
    const float* row = mel + ((size_t)b * M + c) * frames;
    auto at = [&](int f) { return f < frames ? row[f] : 0.f; };
    if (linear) {
      double src = Tp > 1 ? (double)t * (double)(frames_padded - 1) / (double)(Tp - 1) : 0.0;
      int i0 = min((int)floor(src), frames_padded - 1);
      int i1 = min(i0 + 1, frames_padded - 1);
      float w = (float)(src - (double)i0);
      v = at(i0) * (1.f - w) + at(i1) * w;
    } else {
      int i0 = min((int)floor((double)t * ((double)frames_padded / (double)Tp)), frames_padded - 1);
      v = at(i0);
    }
  }
  __nv_bfloat16 h = __float2bfloat16_rn(v);
  hi[i] = h;
  lo[i] = __float2bfloat16_rn(v - __bfloat162float(h));
}

// ------------------------------------------------------------------------------------------
// Row kernel: finishes AR step `row-1` and prepares step `row`:
//   val = in[col_in]*in_scale                       (init: row 0 passes through, efficient_modules.py:49)
//   val = (val - t) * exp(-log_s)                   (efficient_modules.py:62-63) when do_couple
//   out[col_out] = val ;  x0 = start(val)           (glow_ax.py:558) -> ring slot of layer 0
// ------------------------------------------------------------------------------------------
struct WfRowP {
  long long BT; int G;
  const float* in; float in_scale; int col_in;
  float* out; int col_out;
  const float* eo; int do_couple;
  const float* start_w; const float* start_b;
  __nv_bfloat16* x_hi; __nv_bfloat16* x_lo;     // destination ring slot (layer 0), may be null for the last row
};

__global__ void __launch_bounds__(256) k_wf_row(WfRowP p) {
  __shared__ float v_s[64];
  const long long m0 = (long long)blockIdx.x * 64;
  const int tid = threadIdx.x;
  if (tid < 64) {
    long long m = m0 + tid;
    if (m < p.BT) {
      float v = p.in[m * p.G + p.col_in] * p.in_scale;
      if (p.do_couple) {
        const float log_s = p.eo[m * CWG_EO_PAD], t = p.eo[m * CWG_EO_PAD + 1];
        v = (v - t) * expf(-log_s);
      }
      p.out[m * p.G + p.col_out] = v;
      v_s[tid] = v;
    }
  }
  if (p.x_hi == nullptr) return;
  __syncthreads();
  const int nrow = (int)min((long long)64, p.BT - m0);
  const int cp = tid & 63, rq = tid >> 6;          // channel pair, row quarter
  const int c = 2 * cp;
  const float w0 = __ldg(p.start_w + c), w1 = __ldg(p.start_w + c + 1);
  const float b0 = __ldg(p.start_b + c), b1 = __ldg(p.start_b + c + 1);
  for (int r = rq; r < nrow; r += 4) {
    const float v = v_s[r];
    const float x0 = fmaf(w0, v, b0), x1 = fmaf(w1, v, b1);
    const size_t idx = (size_t)(m0 + r) * WF_C + c;
    const __nv_bfloat162 h = __floats2bfloat162_rn(x0, x1);
    *reinterpret_cast<__nv_bfloat162*>(p.x_hi + idx) = h;
    *reinterpret_cast<__nv_bfloat162*>(p.x_lo + idx) = __floats2bfloat162_rn(x0 - __low2float(h), x1 - __high2float(h));
  }
}

// ------------------------------------------------------------------------------------------
// WN_2d layer, one AR row step
// ------------------------------------------------------------------------------------------
struct WfLayerArgs {
  const float* b1;        // [2C]
  const float* b2;        // [C]
  const float* eo_b;      // [16]
  float* eo;              // [B*T'][16]
  int Tp, dil;
  int w1_row0, w2_row0;
  int ring_in, ring_out;  // 4th tensor-map coordinate base of the layer's input ring / next layer's ring
  int row;                // AR row index (newest row), ring slot = row % 3 (row % kh when separable)
  int rows_valid;         // min(row + 1, 3): rows of the conv queue that exist
                          // full-height form (FULL): row = blockIdx.z, set in the kernel with rows_valid and eo's row; x rows
                          // are absolute (ring_in + row), eo is [G-1][B*T'][16]
  int has_res, first;
  // separable in_layers only (k_wf_sep_tc)
  const __nv_bfloat16* x; // ring hi plane; the lo plane follows at x + xplane
  long long xplane, BT;
  const float* dw_w;      // [C][kh * kw] depthwise weights of this (flow, layer)
  const float* dw_b;      // [C]
  int kh, kw;
};

// Two CTAs per SM (each: 6 smem units = 96 KB, 256 TMEM columns), so one CTA's epilogues overlap
// the other's MMAs.  Pool: A units 0,1 (barriers 0,1); weight slots [256 x 64] = unit pairs (2,3) and
// (4,5) (barriers 2,3).  After GEMM1: acts hi -> units 0,1, lo -> units 2,3; W2 tiles use slot 1
// only when acts lo occupies slot 0 (NPASS = 3).  x_old tiles / x_new staging reuse units 0..3.
// TMEM: pre-activation in columns 0..255; [res | folded end] reuses columns 0..143 after the gate.
constexpr int W_NS = 6, W_NA = 2, W_NBAR = 4;
constexpr int W_OFF_B1 = W_NS * TILE_A;                // 98304
constexpr int W_OFF_B2 = W_OFF_B1 + 1024;
constexpr int W_OFF_BAR = W_OFF_B2 + 512;
constexpr int W_SMEM = W_OFF_BAR + 256 + 1024;
constexpr int W_THREADS = 384, W_EPI_THREADS = 256;

template <int NPASS, bool FULL = false>
__global__ void __launch_bounds__(W_THREADS, 2)
k_wf_layer_tc(const __grid_constant__ CUtensorMap tm_x_hi, const __grid_constant__ CUtensorMap tm_x_lo,
              const __grid_constant__ CUtensorMap tm_m_hi, const __grid_constant__ CUtensorMap tm_m_lo,
              const __grid_constant__ CUtensorMap tm_w1_hi, const __grid_constant__ CUtensorMap tm_w1_lo,
              const __grid_constant__ CUtensorMap tm_w2_hi, const __grid_constant__ CUtensorMap tm_w2_lo, WfLayerArgs a) {
  constexpr int PL = NPASS == 3 ? 2 : 1;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = align_1024(smem_raw);
  float* b1s = reinterpret_cast<float*>(smem + W_OFF_B1);
  float* b2s = reinterpret_cast<float*>(smem + W_OFF_B2);
  uint64_t* full = reinterpret_cast<uint64_t*>(smem + W_OFF_BAR);
  uint64_t* empty = full + W_NBAR;
  uint64_t* acc1_full = empty + W_NBAR;
  uint64_t* acts_ready = acc1_full + 1;
  uint64_t* acc2_full = acts_ready + 1;
  uint64_t* xold_full = acc2_full + 1;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(xold_full + 1);

  if constexpr (FULL) {                              // full-height form: one CTA row per height row
    a.row = blockIdx.z;
    a.rows_valid = min(a.row + 1, WF_KH);
    a.eo += (size_t)a.row * a.BT * CWG_EO_PAD;
  }
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int t0 = blockIdx.x * 128, b = blockIdx.y;
  auto slot = [&](int i) { return smem + i * TILE_A; };
  auto bslot = [&](int j) { return smem + (W_NA + 2 * j) * TILE_A; };
  const int nkb_x = a.rows_valid * (WF_KW * 2);      // k-blocks over x: rows x taps x 2 channel blocks
  const int nkb = nkb_x + WF_HP / 64;

  if (threadIdx.x == 0) {
    for (int i = 0; i < W_NBAR; ++i) { mbar_init(&full[i], 1); mbar_init(&empty[i], 1); }
    mbar_init(acc1_full, 1); mbar_init(acts_ready, W_EPI_THREADS); mbar_init(acc2_full, 1); mbar_init(xold_full, 1);
    fence_barrier_init();
  }
  if (warp == 1) tmem_alloc(tmem_slot, 256);
  if (warp >= 4) {
    const int e = threadIdx.x - 128;
    b1s[e] = __ldg(a.b1 + e);
    if (e < WF_C) b2s[e] = __ldg(a.b2 + e);
  }
  tc_fence_before_sync();
  __syncthreads();
  tc_fence_after_sync();
  const uint32_t tmem = *tmem_slot;

  // k-block -> (source, coordinates).  x blocks: oldest existing row first.
  //   kb < nkb_x : j = kb / 6 -> kernel row kh = 3 - rows_valid + j (row index a.row - 2 + kh),
  //                kw = (kb % 6) / 2, cb = kb % 2
  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&tm_x_hi); tma_prefetch_desc(&tm_m_hi);
    int s = 0; uint32_t pm = 0;
    for (int kb = 0; kb < nkb; ++kb) {
      for (int pl = 0; pl < PL; ++pl) {
        mbar_wait(&empty[s], ((pm >> s) & 1u) ^ 1u);
        pm ^= 1u << s;
        mbar_arrive_expect_tx(&full[s], TILE_A);
        if (kb < nkb_x) {
          const int j = kb / 6, kh = WF_KH - a.rows_valid + j, kw = (kb % 6) >> 1, cb = kb & 1;
          const int r = a.row - (WF_KH - 1) + kh;                  // absolute row of this kernel row
          asm volatile(
              "cp.async.bulk.tensor.4d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6}], [%2];"
              ::"r"(smem_u32(slot(s))), "l"(reinterpret_cast<uint64_t>(pl ? &tm_x_lo : &tm_x_hi)), "r"(smem_u32(&full[s])),
                "r"(cb * 64), "r"(t0 + (kw - 1) * a.dil), "r"(b), "r"(a.ring_in + (FULL ? r : r % 3))
              : "memory");
        } else {
          tma_load_3d(slot(s), pl ? &tm_m_lo : &tm_m_hi, &full[s], (kb - nkb_x) * 64, t0, b);
        }
        s = (s + 1 == W_NA) ? 0 : s + 1;
      }
    }
  } else if (warp == 2 && lane == 0) {
    tma_prefetch_desc(&tm_w1_hi); tma_prefetch_desc(&tm_w2_hi);
    int j = 0; uint32_t pm = 0;
    auto put = [&](const CUtensorMap* m, int c0, int r0, uint32_t bytes, bool only1) {
      if (only1) j = 1;
      mbar_wait(&empty[W_NA + j], ((pm >> j) & 1u) ^ 1u);
      pm ^= 1u << j;
      mbar_arrive_expect_tx(&full[W_NA + j], bytes);
      tma_load_2d(bslot(j), m, &full[W_NA + j], c0, r0);
      j ^= 1;
    };
    for (int kb = 0; kb < nkb; ++kb) {
      int col;
      if (kb < nkb_x) {
        const int jj = kb / 6, kh = WF_KH - a.rows_valid + jj, kw = (kb % 6) >> 1, cb = kb & 1;
        col = (kh * WF_KW + kw) * WF_C + cb * 64;
      } else {
        col = WF_KH * WF_KW * WF_C + (kb - nkb_x) * 64;
      }
      for (int pl = 0; pl < PL; ++pl) put(pl ? &tm_w1_lo : &tm_w1_hi, col, a.w1_row0, 2 * TILE_A, false);
    }
    for (int kb = 0; kb < 2; ++kb)
      for (int pl = 0; pl < PL; ++pl) put(pl ? &tm_w2_lo : &tm_w2_hi, kb * 64, a.w2_row0, WF_N2 * 128, NPASS == 3);
  } else if (warp == 1 && lane == 0) {
    int sa = 0, jb = 0; uint32_t cm = 0;
    auto wait_full = [&](int bar) { mbar_wait(&full[bar], (cm >> bar) & 1u); cm ^= 1u << bar; };
    // GEMM1: pre[128 x 256] (tanh | sigmoid halves) in TMEM columns 0..255
    for (int kb = 0; kb < nkb; ++kb) {
      const int sa_hi = sa; wait_full(sa); sa ^= 1;
      int sa_lo = 0;
      if (NPASS == 3) { sa_lo = sa; wait_full(sa); sa ^= 1; }
      const int jb_hi = jb; wait_full(W_NA + jb); jb ^= 1;     // slots: waited for just before first use, released after last use
      tc_fence_after_sync();
      issue_kblock_fast(smem_u32(slot(sa_hi)), smem_u32(bslot(jb_hi)), tmem, IDESC_N256, kb == 0);
      if (NPASS == 3) {
        issue_kblock_fast(smem_u32(slot(sa_lo)), smem_u32(bslot(jb_hi)), tmem, IDESC_N256, false);
        umma_commit(&empty[W_NA + jb_hi]);
        umma_commit(&empty[sa_lo]);
        const int jb_lo = jb; wait_full(W_NA + jb); jb ^= 1;
        tc_fence_after_sync();
        issue_kblock_fast(smem_u32(slot(sa_hi)), smem_u32(bslot(jb_lo)), tmem, IDESC_N256, false);
        umma_commit(&empty[W_NA + jb_lo]);
      } else {
        umma_commit(&empty[W_NA + jb_hi]);
      }
      umma_commit(&empty[sa_hi]);
    }
    umma_commit(acc1_full);
    // GEMM2: [res (128) | folded end (16)] = acts x W2^T, reusing TMEM columns 0..143
    mbar_wait(acts_ready, 0);
    tc_fence_after_sync();
    for (int kb = 0; kb < 2; ++kb) {
      const uint32_t a_hi = smem_u32(slot(kb)), a_lo = smem_u32(slot(2 + kb));
      if (NPASS == 3) jb = 1;
      const int jb_hi = jb; wait_full(W_NA + jb); jb ^= 1;
      tc_fence_after_sync();
      issue_kblock_fast(a_hi, smem_u32(bslot(jb_hi)), tmem, IDESC_N144, kb == 0);
      if (NPASS == 3) {
        issue_kblock_fast(a_lo, smem_u32(bslot(jb_hi)), tmem, IDESC_N144, false);
        umma_commit(&empty[W_NA + jb_hi]);
        wait_full(W_NA + 1);                 // W2 lo tile arrives in the same (only) slot
        tc_fence_after_sync();
        issue_kblock_fast(a_hi, smem_u32(bslot(1)), tmem, IDESC_N144, false);
        umma_commit(&empty[W_NA + 1]);
      } else {
        umma_commit(&empty[W_NA + jb_hi]);
      }
    }
    umma_commit(acc2_full);
    if (a.has_res) {
      // this row's input tiles (the conv's newest row, centre tap) -> units 0..3 for the residual add
      mbar_wait(acc2_full, 0);
      mbar_arrive_expect_tx(xold_full, 4 * TILE_A);
      for (int kb = 0; kb < 2; ++kb)
        for (int pl = 0; pl < 2; ++pl)
          asm volatile(
              "cp.async.bulk.tensor.4d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6}], [%2];"
              ::"r"(smem_u32(slot(2 * pl + kb))), "l"(reinterpret_cast<uint64_t>(pl ? &tm_x_lo : &tm_x_hi)), "r"(smem_u32(xold_full)),
                "r"(kb * 64), "r"(t0), "r"(b), "r"(a.ring_in + (FULL ? a.row : a.row % 3))
              : "memory");
    }
  } else if (warp >= 4) {
    const int quarter = warp & 3, half = (warp - 4) >> 2, row = quarter * 32 + lane;
    const uint32_t trow = tmem + ((uint32_t)(quarter * 32) << 16);
    const bool valid = t0 + row < a.Tp;
    const size_t m = (size_t)b * a.Tp + (size_t)min(t0 + row, a.Tp - 1);
    const float4* b1t = reinterpret_cast<const float4*>(b1s);
    const float4* b1g = reinterpret_cast<const float4*>(b1s + WF_C);

    mbar_wait(acc1_full, 0);
    tc_fence_after_sync();
    {
      uint32_t buf[2][32];
      const int c0 = half * 4;
      tmem_issue16x2(trow + c0 * 16, trow + WF_C + c0 * 16, buf[0]);
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const int c = c0 + i;
        uint32_t* cur = buf[i & 1];
        tmem_wait32(cur);
        if (i + 1 < 4) tmem_issue16x2(trow + (c + 1) * 16, trow + WF_C + (c + 1) * 16, buf[(i + 1) & 1]);
        float act[16];
#pragma unroll
        for (int q = 0; q < 4; ++q) {
          const float4 bt = b1t[c * 4 + q], bs = b1g[c * 4 + q];
          act[4 * q + 0] = gate<NPASS>(__uint_as_float(cur[4 * q + 0]) + bt.x, __uint_as_float(cur[16 + 4 * q + 0]) + bs.x);
          act[4 * q + 1] = gate<NPASS>(__uint_as_float(cur[4 * q + 1]) + bt.y, __uint_as_float(cur[16 + 4 * q + 1]) + bs.y);
          act[4 * q + 2] = gate<NPASS>(__uint_as_float(cur[4 * q + 2]) + bt.z, __uint_as_float(cur[16 + 4 * q + 2]) + bs.z);
          act[4 * q + 3] = gate<NPASS>(__uint_as_float(cur[4 * q + 3]) + bt.w, __uint_as_float(cur[16 + 4 * q + 3]) + bs.w);
        }
        store_split16<NPASS == 3>(act, slot(c >> 2), slot(2 + (c >> 2)), row, (c & 3) * 2);
      }
    }
    tc_fence_before_sync();
    fence_proxy_async_smem();
    mbar_arrive(acts_ready);

    float4 eold[4];
    if (half == 0) {
      const float4* e = reinterpret_cast<const float4*>(a.first ? a.eo_b : a.eo + m * CWG_EO_PAD);
#pragma unroll
      for (int q = 0; q < 4; ++q) eold[q] = __ldg(e + q);
    }
    mbar_wait(acc2_full, 0);
    tc_fence_after_sync();
    if (half == 0) {
      uint32_t sk[16];
      tmem_issue16(trow + WF_C, sk);
      tmem_wait16(sk);
      if (valid) {
        float4* e = reinterpret_cast<float4*>(a.eo + m * CWG_EO_PAD);
#pragma unroll
        for (int q = 0; q < 4; ++q) {
          float4 v = eold[q];
          v.x += __uint_as_float(sk[4 * q]); v.y += __uint_as_float(sk[4 * q + 1]);
          v.z += __uint_as_float(sk[4 * q + 2]); v.w += __uint_as_float(sk[4 * q + 3]);
          e[q] = v;
        }
      }
    }
    if (a.has_res) {
      const float4* b2v = reinterpret_cast<const float4*>(b2s);
      uint32_t buf[2][16];
      const int c0 = half * 4;
      tmem_issue16(trow + c0 * 16, buf[0]);
      mbar_wait(xold_full, 0);
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const int c = c0 + i;
        uint32_t* cur = buf[i & 1];
        tmem_wait16(cur);
        if (i + 1 < 4) tmem_issue16(trow + (c + 1) * 16, buf[(i + 1) & 1]);
        uint8_t* thi = slot(c >> 2);
        uint8_t* tlo = slot(2 + (c >> 2));
        const uint32_t o0 = sw128_offset(row, (c & 3) * 2), o1 = sw128_offset(row, (c & 3) * 2 + 1);
        const uint4 h0 = *reinterpret_cast<const uint4*>(thi + o0), h1 = *reinterpret_cast<const uint4*>(thi + o1);
        const uint4 l0 = *reinterpret_cast<const uint4*>(tlo + o0), l1 = *reinterpret_cast<const uint4*>(tlo + o1);
        const uint32_t hw[8] = {h0.x, h0.y, h0.z, h0.w, h1.x, h1.y, h1.z, h1.w};
        const uint32_t lw[8] = {l0.x, l0.y, l0.z, l0.w, l1.x, l1.y, l1.z, l1.w};
        float r[16];
#pragma unroll
        for (int q = 0; q < 4; ++q) {
          const float4 bb = b2v[c * 4 + q];
          r[4 * q] = __uint_as_float(cur[4 * q]) + bb.x; r[4 * q + 1] = __uint_as_float(cur[4 * q + 1]) + bb.y;
          r[4 * q + 2] = __uint_as_float(cur[4 * q + 2]) + bb.z; r[4 * q + 3] = __uint_as_float(cur[4 * q + 3]) + bb.w;
        }
#pragma unroll
        for (int j = 0; j < 8; ++j) {   // audio += res_skip_acts[:, :C], glow_ax.py:615-620
          r[2 * j] += __uint_as_float(hw[j] << 16) + __uint_as_float(lw[j] << 16);
          r[2 * j + 1] += __uint_as_float(hw[j] & 0xFFFF0000u) + __uint_as_float(lw[j] & 0xFFFF0000u);
        }
        store_split16<true>(r, thi, tlo, row, (c & 3) * 2);
      }
      // each column half owns one 64-channel tile (hi + lo)
      fence_proxy_async_smem();
      asm volatile("bar.sync %0, 128;" ::"r"(2 + half) : "memory");
      if (quarter == 0 && lane == 0) {
        for (int pl = 0; pl < 2; ++pl)
          asm volatile("cp.async.bulk.tensor.4d.global.shared::cta.bulk_group [%0, {%2, %3, %4, %5}], [%1];"
                       ::"l"(reinterpret_cast<uint64_t>(pl ? &tm_x_lo : &tm_x_hi)), "r"(smem_u32(slot(2 * pl + half))),
                         "r"(half * 64), "r"(t0), "r"(b), "r"(a.ring_out + (FULL ? a.row : a.row % 3))
                       : "memory");
        tma_store_commit();
        tma_store_wait_read();
      }
    }
    tc_fence_before_sync();
  }
  __syncthreads();
  if (warp == 1) { __syncwarp(); tmem_dealloc(tmem, 256); }
}

// Separable layout (k_wf_sep_tc), one CTA per SM: the same pool (units 0..5), plus the depthwise output d - GEMM1's
// x operand, hi in units 6,7 and lo in units 8,9 - and the depthwise weights transposed to [tap][C].
constexpr int S_NS = W_NS + 4;
constexpr int S_OFF_DW = S_NS * TILE_A;                                   // 163840
constexpr int S_OFF_DWB = S_OFF_DW + WF_SEP_MAX_KH * WF_SEP_MAX_KW * WF_C * 4;
constexpr int S_OFF_B1 = S_OFF_DWB + WF_C * 4;
constexpr int S_OFF_B2 = S_OFF_B1 + 1024;
constexpr int S_OFF_BAR = S_OFF_B2 + 512;
constexpr int S_SMEM = S_OFF_BAR + 256 + 1024;                             // 192256

// Depthwise part of a separable in_layer (glow_ax.py:525-528) for the 128 steps of this tile, by the 8 epilogue warps
// while the mel k-blocks of GEMM1 run:
//   d[t][c] = dw_b[c] + sum_{a,b} dw_w[c][a][b] * x[row - (kh-1-a)][t + (b - kw/2) * dil][c]     in fp32, x = hi + lo,
// causal in height (rows that do not exist yet are the zero queue), zero-padded in width per utterance.  A lane owns 4
// channels and a warp one step at a time, so each load is a 256-byte run of channels.  d is written as 128B-swizzled
// bf16 hi (and lo) tiles, one per 64-channel k-block; it never goes to HBM.
template <int NPASS, bool FULL>
__device__ __forceinline__ void wf_depthwise_tile(const WfLayerArgs& a, const float* dws, const float* dwb, int b, int t0,
                                                  int ew, int lane, uint8_t* d_hi, uint8_t* d_lo) {
  // A warp handles 16 steps in two passes of S.  The loop is not bound by load latency (issuing two taps' loads at once
  // was slower), so its instruction count is kept down: per bf16x2 word two FFMA2 (hi, then lo; no separate hi + lo add),
  // and a pass checks the utterance bounds once when all S steps of a tap are inside (the common case).
  constexpr int S = 8;
  const int c = 4 * lane, chunk = (lane & 15) >> 1, sub = (lane & 1) * 8;
  uint8_t* th = d_hi + (lane >> 4) * TILE_A;
  uint8_t* tl = d_lo + (lane >> 4) * TILE_A;
  const float4 bias = *reinterpret_cast<const float4*>(dwb + c);
  auto lo2 = [](uint32_t v) { return make_float2(__uint_as_float(v << 16), __uint_as_float(v & 0xFFFF0000u)); };
  for (int s0 = ew * 16; s0 < ew * 16 + 16; s0 += S) {
    float2 acc[S][2];
#pragma unroll
    for (int i = 0; i < S; ++i) { acc[i][0] = make_float2(bias.x, bias.y); acc[i][1] = make_float2(bias.z, bias.w); }
    for (int ah = 0; ah < a.kh; ++ah) {
      const int r = a.row - (a.kh - 1 - ah);
      if (r < 0) continue;
      const __nv_bfloat16* xh = a.x + ((size_t)(a.ring_in + (FULL ? r : r % a.kh)) * a.BT + (size_t)b * a.Tp) * WF_C + c;
      const __nv_bfloat16* xl = xh + a.xplane;
      for (int bw = 0; bw < a.kw; ++bw) {
        const float4 w = *reinterpret_cast<const float4*>(dws + (ah * a.kw + bw) * WF_C + c);
        const float2 w01 = make_float2(w.x, w.y), w23 = make_float2(w.z, w.w);
        const int tt0 = t0 + s0 + (bw - a.kw / 2) * a.dil;
        uint2 h[S], l[S];
        if (tt0 >= 0 && tt0 + S <= a.Tp) {
#pragma unroll
          for (int i = 0; i < S; ++i) {
            h[i] = __ldg(reinterpret_cast<const uint2*>(xh + (size_t)(tt0 + i) * WF_C));
            l[i] = __ldg(reinterpret_cast<const uint2*>(xl + (size_t)(tt0 + i) * WF_C));
          }
        } else {
#pragma unroll
          for (int i = 0; i < S; ++i) {
            const int tt = tt0 + i;
            h[i] = l[i] = make_uint2(0u, 0u);
            if (tt >= 0 && tt < a.Tp) {
              h[i] = __ldg(reinterpret_cast<const uint2*>(xh + (size_t)tt * WF_C));
              l[i] = __ldg(reinterpret_cast<const uint2*>(xl + (size_t)tt * WF_C));
            }
          }
        }
#pragma unroll
        for (int i = 0; i < S; ++i) {
          acc[i][0] = __ffma2_rn(w01, lo2(l[i].x), __ffma2_rn(w01, lo2(h[i].x), acc[i][0]));
          acc[i][1] = __ffma2_rn(w23, lo2(l[i].y), __ffma2_rn(w23, lo2(h[i].y), acc[i][1]));
        }
      }
    }
#pragma unroll
    for (int i = 0; i < S; ++i) {
      const uint32_t off = sw128_offset(s0 + i, chunk) + sub;
      const float2 d01 = acc[i][0], d23 = acc[i][1];
      const uint32_t h0 = pack_bf16x2(d01.x, d01.y), h1 = pack_bf16x2(d23.x, d23.y);
      *reinterpret_cast<uint2*>(th + off) = make_uint2(h0, h1);
      if (NPASS == 3) {
        float e0, e1, e2, e3;
        unpack2<false>(h0, e0, e1); unpack2<false>(h1, e2, e3);
        *reinterpret_cast<uint2*>(tl + off) = make_uint2(pack_bf16x2(d01.x - e0, d01.y - e1), pack_bf16x2(d23.x - e2, d23.y - e3));
      }
    }
  }
}

// The layer step with separable in_layers, one CTA per SM: GEMM1 runs over the 2 mel k-blocks (TMA, issued first), then
// the 2 k-blocks of d, which the epilogue warps compute in the meantime (wf_depthwise_tile).  Gate, GEMM2 ([res | folded
// end], N = 144), residual update and eo accumulation are those of k_wf_layer_tc, whose source is kept as it is.
template <int NPASS, bool FULL = false>
__global__ void __launch_bounds__(W_THREADS, 1)
k_wf_sep_tc(const __grid_constant__ CUtensorMap tm_x_hi, const __grid_constant__ CUtensorMap tm_x_lo,
            const __grid_constant__ CUtensorMap tm_m_hi, const __grid_constant__ CUtensorMap tm_m_lo,
            const __grid_constant__ CUtensorMap tm_w1_hi, const __grid_constant__ CUtensorMap tm_w1_lo,
            const __grid_constant__ CUtensorMap tm_w2_hi, const __grid_constant__ CUtensorMap tm_w2_lo, WfLayerArgs a) {
  constexpr int PL = NPASS == 3 ? 2 : 1;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = align_1024(smem_raw);
  float* b1s = reinterpret_cast<float*>(smem + S_OFF_B1);
  float* b2s = reinterpret_cast<float*>(smem + S_OFF_B2);
  uint64_t* full = reinterpret_cast<uint64_t*>(smem + S_OFF_BAR);
  uint64_t* empty = full + W_NBAR;
  uint64_t* acc1_full = empty + W_NBAR;
  uint64_t* acts_ready = acc1_full + 1;
  uint64_t* acc2_full = acts_ready + 1;
  uint64_t* xold_full = acc2_full + 1;
  uint64_t* d_ready = xold_full + 1;                 // depthwise tiles written
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(d_ready + 1);

  if constexpr (FULL) {                              // full-height form: one CTA row per height row
    a.row = blockIdx.z;
    a.eo += (size_t)a.row * a.BT * CWG_EO_PAD;
  }
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int t0 = blockIdx.x * 128, b = blockIdx.y;
  auto slot = [&](int i) { return smem + i * TILE_A; };
  auto bslot = [&](int j) { return smem + (W_NA + 2 * j) * TILE_A; };
  constexpr int nkb = WF_HP / 64;                   // mel k-blocks through the A ring
  constexpr int NKB_D = WF_C / 64;                  // k-blocks of d, after the mel ones
  const int nslot = a.kh;                           // ring slots per layer

  if (threadIdx.x == 0) {
    for (int i = 0; i < W_NBAR; ++i) { mbar_init(&full[i], 1); mbar_init(&empty[i], 1); }
    mbar_init(acc1_full, 1); mbar_init(acts_ready, W_EPI_THREADS); mbar_init(acc2_full, 1); mbar_init(xold_full, 1);
    mbar_init(d_ready, W_EPI_THREADS);
    fence_barrier_init();
  }
  if (warp == 1) tmem_alloc(tmem_slot, 256);
  if (warp >= 4) {
    const int e = threadIdx.x - 128;
    b1s[e] = __ldg(a.b1 + e);
    if (e < WF_C) b2s[e] = __ldg(a.b2 + e);
    float* dws = reinterpret_cast<float*>(smem + S_OFF_DW);
    const int ntap = a.kh * a.kw;
    for (int i = e; i < ntap * WF_C; i += W_EPI_THREADS) dws[(i % ntap) * WF_C + i / ntap] = __ldg(a.dw_w + i);
    if (e < WF_C) reinterpret_cast<float*>(smem + S_OFF_DWB)[e] = __ldg(a.dw_b + e);
  }
  tc_fence_before_sync();
  __syncthreads();
  tc_fence_after_sync();
  const uint32_t tmem = *tmem_slot;

  // k-block order of GEMM1: the 2 mel k-blocks (A ring), then the 2 channel k-blocks of d
  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&tm_x_hi); tma_prefetch_desc(&tm_m_hi);
    int s = 0; uint32_t pm = 0;
    for (int kb = 0; kb < nkb; ++kb) {
      for (int pl = 0; pl < PL; ++pl) {
        mbar_wait(&empty[s], ((pm >> s) & 1u) ^ 1u);
        pm ^= 1u << s;
        mbar_arrive_expect_tx(&full[s], TILE_A);
        tma_load_3d(slot(s), pl ? &tm_m_lo : &tm_m_hi, &full[s], kb * 64, t0, b);
        s = (s + 1 == W_NA) ? 0 : s + 1;
      }
    }
  } else if (warp == 2 && lane == 0) {
    tma_prefetch_desc(&tm_w1_hi); tma_prefetch_desc(&tm_w2_hi);
    int j = 0; uint32_t pm = 0;
    auto put = [&](const CUtensorMap* m, int c0, int r0, uint32_t bytes, bool only1) {
      if (only1) j = 1;
      mbar_wait(&empty[W_NA + j], ((pm >> j) & 1u) ^ 1u);
      pm ^= 1u << j;
      mbar_arrive_expect_tx(&full[W_NA + j], bytes);
      tma_load_2d(bslot(j), m, &full[W_NA + j], c0, r0);
      j ^= 1;
    };
    for (int kb = 0; kb < nkb + NKB_D; ++kb) {
      const int col = kb < nkb ? WF_C + kb * 64 : (kb - nkb) * 64;          // w1 columns: pointwise (C) | mel
      for (int pl = 0; pl < PL; ++pl) put(pl ? &tm_w1_lo : &tm_w1_hi, col, a.w1_row0, 2 * TILE_A, false);
    }
    for (int kb = 0; kb < 2; ++kb)
      for (int pl = 0; pl < PL; ++pl) put(pl ? &tm_w2_lo : &tm_w2_hi, kb * 64, a.w2_row0, WF_N2 * 128, NPASS == 3);
  } else if (warp == 1 && lane == 0) {
    int sa = 0, jb = 0; uint32_t cm = 0;
    auto wait_full = [&](int bar) { mbar_wait(&full[bar], (cm >> bar) & 1u); cm ^= 1u << bar; };
    // GEMM1: pre[128 x 256] (tanh | sigmoid halves) in TMEM columns 0..255
    for (int kb = 0; kb < nkb; ++kb) {
      const int sa_hi = sa; wait_full(sa); sa ^= 1;
      int sa_lo = 0;
      if (NPASS == 3) { sa_lo = sa; wait_full(sa); sa ^= 1; }
      const int jb_hi = jb; wait_full(W_NA + jb); jb ^= 1;     // slots: waited for just before first use, released after last use
      tc_fence_after_sync();
      issue_kblock_fast(smem_u32(slot(sa_hi)), smem_u32(bslot(jb_hi)), tmem, IDESC_N256, kb == 0);
      if (NPASS == 3) {
        issue_kblock_fast(smem_u32(slot(sa_lo)), smem_u32(bslot(jb_hi)), tmem, IDESC_N256, false);
        umma_commit(&empty[W_NA + jb_hi]);
        umma_commit(&empty[sa_lo]);
        const int jb_lo = jb; wait_full(W_NA + jb); jb ^= 1;
        tc_fence_after_sync();
        issue_kblock_fast(smem_u32(slot(sa_hi)), smem_u32(bslot(jb_lo)), tmem, IDESC_N256, false);
        umma_commit(&empty[W_NA + jb_lo]);
      } else {
        umma_commit(&empty[W_NA + jb_hi]);
      }
      umma_commit(&empty[sa_hi]);
    }
    mbar_wait(d_ready, 0);
    tc_fence_after_sync();
    for (int kd = 0; kd < NKB_D; ++kd) {
      const uint32_t d_hi = smem_u32(slot(W_NS + kd)), d_lo = smem_u32(slot(W_NS + NKB_D + kd));
      const int jb_hi = jb; wait_full(W_NA + jb); jb ^= 1;
      tc_fence_after_sync();
      issue_kblock_fast(d_hi, smem_u32(bslot(jb_hi)), tmem, IDESC_N256, false);
      if (NPASS == 3) {
        issue_kblock_fast(d_lo, smem_u32(bslot(jb_hi)), tmem, IDESC_N256, false);
        umma_commit(&empty[W_NA + jb_hi]);
        const int jb_lo = jb; wait_full(W_NA + jb); jb ^= 1;
        tc_fence_after_sync();
        issue_kblock_fast(d_hi, smem_u32(bslot(jb_lo)), tmem, IDESC_N256, false);
        umma_commit(&empty[W_NA + jb_lo]);
      } else {
        umma_commit(&empty[W_NA + jb_hi]);
      }
    }
    umma_commit(acc1_full);
    // GEMM2: [res (128) | folded end (16)] = acts x W2^T, reusing TMEM columns 0..143
    mbar_wait(acts_ready, 0);
    tc_fence_after_sync();
    for (int kb = 0; kb < 2; ++kb) {
      const uint32_t a_hi = smem_u32(slot(kb)), a_lo = smem_u32(slot(2 + kb));
      if (NPASS == 3) jb = 1;
      const int jb_hi = jb; wait_full(W_NA + jb); jb ^= 1;
      tc_fence_after_sync();
      issue_kblock_fast(a_hi, smem_u32(bslot(jb_hi)), tmem, IDESC_N144, kb == 0);
      if (NPASS == 3) {
        issue_kblock_fast(a_lo, smem_u32(bslot(jb_hi)), tmem, IDESC_N144, false);
        umma_commit(&empty[W_NA + jb_hi]);
        wait_full(W_NA + 1);                 // W2 lo tile arrives in the same (only) slot
        tc_fence_after_sync();
        issue_kblock_fast(a_hi, smem_u32(bslot(1)), tmem, IDESC_N144, false);
        umma_commit(&empty[W_NA + 1]);
      } else {
        umma_commit(&empty[W_NA + jb_hi]);
      }
    }
    umma_commit(acc2_full);
    if (a.has_res) {
      // this row's input tiles (the conv's newest row, centre tap) -> units 0..3 for the residual add
      mbar_wait(acc2_full, 0);
      mbar_arrive_expect_tx(xold_full, 4 * TILE_A);
      for (int kb = 0; kb < 2; ++kb)
        for (int pl = 0; pl < 2; ++pl)
          asm volatile(
              "cp.async.bulk.tensor.4d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6}], [%2];"
              ::"r"(smem_u32(slot(2 * pl + kb))), "l"(reinterpret_cast<uint64_t>(pl ? &tm_x_lo : &tm_x_hi)), "r"(smem_u32(xold_full)),
                "r"(kb * 64), "r"(t0), "r"(b), "r"(a.ring_in + (FULL ? a.row : a.row % nslot))
              : "memory");
    }
  } else if (warp >= 4) {
    const int quarter = warp & 3, half = (warp - 4) >> 2, row = quarter * 32 + lane;
    const uint32_t trow = tmem + ((uint32_t)(quarter * 32) << 16);
    const bool valid = t0 + row < a.Tp;
    const size_t m = (size_t)b * a.Tp + (size_t)min(t0 + row, a.Tp - 1);
    const float4* b1t = reinterpret_cast<const float4*>(b1s);
    const float4* b1g = reinterpret_cast<const float4*>(b1s + WF_C);

    // the mel k-blocks of GEMM1 run meanwhile
    wf_depthwise_tile<NPASS, FULL>(a, reinterpret_cast<const float*>(smem + S_OFF_DW), reinterpret_cast<const float*>(smem + S_OFF_DWB),
                             b, t0, warp - 4, lane, slot(W_NS), slot(W_NS + NKB_D));
    tc_fence_before_sync();
    fence_proxy_async_smem();
    mbar_arrive(d_ready);
    mbar_wait(acc1_full, 0);
    tc_fence_after_sync();
    {
      uint32_t buf[2][32];
      const int c0 = half * 4;
      tmem_issue16x2(trow + c0 * 16, trow + WF_C + c0 * 16, buf[0]);
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const int c = c0 + i;
        uint32_t* cur = buf[i & 1];
        tmem_wait32(cur);
        if (i + 1 < 4) tmem_issue16x2(trow + (c + 1) * 16, trow + WF_C + (c + 1) * 16, buf[(i + 1) & 1]);
        float act[16];
#pragma unroll
        for (int q = 0; q < 4; ++q) {
          const float4 bt = b1t[c * 4 + q], bs = b1g[c * 4 + q];
          act[4 * q + 0] = gate<NPASS>(__uint_as_float(cur[4 * q + 0]) + bt.x, __uint_as_float(cur[16 + 4 * q + 0]) + bs.x);
          act[4 * q + 1] = gate<NPASS>(__uint_as_float(cur[4 * q + 1]) + bt.y, __uint_as_float(cur[16 + 4 * q + 1]) + bs.y);
          act[4 * q + 2] = gate<NPASS>(__uint_as_float(cur[4 * q + 2]) + bt.z, __uint_as_float(cur[16 + 4 * q + 2]) + bs.z);
          act[4 * q + 3] = gate<NPASS>(__uint_as_float(cur[4 * q + 3]) + bt.w, __uint_as_float(cur[16 + 4 * q + 3]) + bs.w);
        }
        store_split16<NPASS == 3>(act, slot(c >> 2), slot(2 + (c >> 2)), row, (c & 3) * 2);
      }
    }
    tc_fence_before_sync();
    fence_proxy_async_smem();
    mbar_arrive(acts_ready);

    float4 eold[4];
    if (half == 0) {
      const float4* e = reinterpret_cast<const float4*>(a.first ? a.eo_b : a.eo + m * CWG_EO_PAD);
#pragma unroll
      for (int q = 0; q < 4; ++q) eold[q] = __ldg(e + q);
    }
    mbar_wait(acc2_full, 0);
    tc_fence_after_sync();
    if (half == 0) {
      uint32_t sk[16];
      tmem_issue16(trow + WF_C, sk);
      tmem_wait16(sk);
      if (valid) {
        float4* e = reinterpret_cast<float4*>(a.eo + m * CWG_EO_PAD);
#pragma unroll
        for (int q = 0; q < 4; ++q) {
          float4 v = eold[q];
          v.x += __uint_as_float(sk[4 * q]); v.y += __uint_as_float(sk[4 * q + 1]);
          v.z += __uint_as_float(sk[4 * q + 2]); v.w += __uint_as_float(sk[4 * q + 3]);
          e[q] = v;
        }
      }
    }
    if (a.has_res) {
      const float4* b2v = reinterpret_cast<const float4*>(b2s);
      uint32_t buf[2][16];
      const int c0 = half * 4;
      tmem_issue16(trow + c0 * 16, buf[0]);
      mbar_wait(xold_full, 0);
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const int c = c0 + i;
        uint32_t* cur = buf[i & 1];
        tmem_wait16(cur);
        if (i + 1 < 4) tmem_issue16(trow + (c + 1) * 16, buf[(i + 1) & 1]);
        uint8_t* thi = slot(c >> 2);
        uint8_t* tlo = slot(2 + (c >> 2));
        const uint32_t o0 = sw128_offset(row, (c & 3) * 2), o1 = sw128_offset(row, (c & 3) * 2 + 1);
        const uint4 h0 = *reinterpret_cast<const uint4*>(thi + o0), h1 = *reinterpret_cast<const uint4*>(thi + o1);
        const uint4 l0 = *reinterpret_cast<const uint4*>(tlo + o0), l1 = *reinterpret_cast<const uint4*>(tlo + o1);
        const uint32_t hw[8] = {h0.x, h0.y, h0.z, h0.w, h1.x, h1.y, h1.z, h1.w};
        const uint32_t lw[8] = {l0.x, l0.y, l0.z, l0.w, l1.x, l1.y, l1.z, l1.w};
        float r[16];
#pragma unroll
        for (int q = 0; q < 4; ++q) {
          const float4 bb = b2v[c * 4 + q];
          r[4 * q] = __uint_as_float(cur[4 * q]) + bb.x; r[4 * q + 1] = __uint_as_float(cur[4 * q + 1]) + bb.y;
          r[4 * q + 2] = __uint_as_float(cur[4 * q + 2]) + bb.z; r[4 * q + 3] = __uint_as_float(cur[4 * q + 3]) + bb.w;
        }
#pragma unroll
        for (int j = 0; j < 8; ++j) {   // audio += res_skip_acts[:, :C], glow_ax.py:615-620
          r[2 * j] += __uint_as_float(hw[j] << 16) + __uint_as_float(lw[j] << 16);
          r[2 * j + 1] += __uint_as_float(hw[j] & 0xFFFF0000u) + __uint_as_float(lw[j] & 0xFFFF0000u);
        }
        store_split16<true>(r, thi, tlo, row, (c & 3) * 2);
      }
      // each column half owns one 64-channel tile (hi + lo)
      fence_proxy_async_smem();
      asm volatile("bar.sync %0, 128;" ::"r"(2 + half) : "memory");
      if (quarter == 0 && lane == 0) {
        for (int pl = 0; pl < 2; ++pl)
          asm volatile("cp.async.bulk.tensor.4d.global.shared::cta.bulk_group [%0, {%2, %3, %4, %5}], [%1];"
                       ::"l"(reinterpret_cast<uint64_t>(pl ? &tm_x_lo : &tm_x_hi)), "r"(smem_u32(slot(2 * pl + half))),
                         "r"(half * 64), "r"(t0), "r"(b), "r"(a.ring_out + (FULL ? a.row : a.row % nslot))
                       : "memory");
        tma_store_commit();
        tma_store_wait_read();
      }
    }
    tc_fence_before_sync();
  }
  __syncthreads();
  if (warp == 1) { __syncwarp(); tmem_dealloc(tmem, 256); }
}

struct WfWorkspace {
  __nv_bfloat16* x;      // hi plane then lo plane, each [L][KH][B][T'][C] (KH = kernel_h: 3 for the dense layout)
  __nv_bfloat16* mel_up; // hi, lo planes [B][T'][128]
  float* eo;             // [B*T'][16]
  float* state;          // [B*T'][G] scratch audio state (flows F-1 .. 1)
  size_t bytes;
};

void wf_carve(const WfDims& d, void* base, WfWorkspace* ws) {
  size_t off = 0;
  auto take = [&](size_t bytes) { size_t o = off; off = align_up(off + bytes, 1024); return (char*)base + o; };
  ws->eo = (float*)take((size_t)d.BT * CWG_EO_PAD * 4);
  ws->state = (float*)take((size_t)d.BT * d.G * 4);
  ws->mel_up = (__nv_bfloat16*)take((size_t)d.BT * WF_HP * 2 * 2);
  ws->x = (__nv_bfloat16*)take((size_t)d.L * d.KH * d.BT * WF_C * 2 * 2);
  ws->bytes = off;
}

// Forward direction (cwg_wf_forward): all G-1 height rows of a flow are known before it runs.
struct WfFwdWorkspace {
  __nv_bfloat16* x;      // hi plane then lo plane, each two full-height buffers [2][G-1][B][T'][C] (layers ping-pong)
  __nv_bfloat16* mel_up; // hi, lo planes [B][T'][128]
  float* eo;             // [G-1][B*T'][16]
  double* ls_part;       // [F][B][nblk] block sums of log_s
  double* z2_part;       // [B][nblk] block sums of z^2
  double* ld_zero;       // [F] zeros: the log|det| of PermuteHeight that k_fwd_reduce adds
  size_t bytes;
};

void wf_fwd_carve(const WfDims& d, void* base, WfFwdWorkspace* ws) {
  size_t off = 0;
  auto take = [&](size_t bytes) { size_t o = off; off = align_up(off + bytes, 1024); return (char*)base + o; };
  const size_t nblk = (size_t)wf_fwd_blocks(d.Tp);
  ws->eo = (float*)take((size_t)(d.G - 1) * d.BT * CWG_EO_PAD * 4);
  ws->ls_part = (double*)take((size_t)d.F * d.B * nblk * 8);
  ws->z2_part = (double*)take((size_t)d.B * nblk * 8);
  ws->ld_zero = (double*)take((size_t)d.F * 8);
  ws->mel_up = (__nv_bfloat16*)take((size_t)d.BT * WF_HP * 2 * 2);
  ws->x = (__nv_bfloat16*)take((size_t)2 * (d.G - 1) * d.BT * WF_C * 2 * 2);
  ws->bytes = off;
}

int wf_check(const cwg_wf_config* c, int mode, int batch, int t_samples) {
  CWG_REQUIRE(c != nullptr, "cfg is NULL");
  CWG_REQUIRE(mode == CWG_MODE_BF16X3 || mode == CWG_MODE_BF16, "WaveFlow supports the tensor-core modes only");
  CWG_REQUIRE(c->n_channels == WF_C && ((c->kernel_h == WF_KH && c->kernel_w == WF_KW) ||
                                        (c->kernel_h >= 1 && c->kernel_h <= WF_SEP_MAX_KH && c->kernel_w >= 1 &&
                                         c->kernel_w <= WF_SEP_MAX_KW && c->kernel_w % 2 == 1)),
              "the tensor-core WaveFlow kernels take n_channels=128 with a dense or separable 3x3 kernel, or separable in_layers "
              "of kernel_h <= %d and odd kernel_w <= %d (got %d, %dx%d)", WF_SEP_MAX_KH, WF_SEP_MAX_KW, c->n_channels, c->kernel_h,
              c->kernel_w);
  CWG_REQUIRE(c->n_group >= 2 && c->n_group <= WF_TC_MAX_GROUP, "n_group must be in [2, %d]", WF_TC_MAX_GROUP);
  CWG_REQUIRE(c->n_mel >= 1 && c->n_mel <= WF_HP, "n_mel must be <= %d", WF_HP);
  CWG_REQUIRE(c->n_flows >= 1 && c->n_layers >= 1 && c->n_layers <= 16, "bad n_flows / n_layers");
  CWG_REQUIRE(c->gate == CWG_GATE_GTU, "the tensor-core WaveFlow kernels implement the GTU gate only (use CWG_MODE_FFMA)");
  CWG_REQUIRE(c->n_early_every == 0 && c->mix_first_off == 0 && c->mixing_conv == 0,
              "early outputs / mix_first = 0 / 1x1conv mixing run in CWG_MODE_FFMA only");
  for (int l = 0; l < c->n_layers; ++l)
    CWG_REQUIRE((c->dilations_w[l] == 0 || c->dilations_w[l] == (1 << l)) && c->dilations_h[l] <= 1,
                "the tensor-core WaveFlow kernels take dilation_w 2^i and dilation_h 1 only (use CWG_MODE_FFMA)");
  CWG_REQUIRE(batch >= 1 && t_samples >= c->n_group && t_samples % c->n_group == 0, "t_samples must be a positive multiple of n_group");
  return 0;
}

WfDims wf_dims(const cwg_wf_config* c, int batch, int t_samples) {
  WfDims d;
  d.B = batch; d.Tp = t_samples / c->n_group; d.F = c->n_flows; d.L = c->n_layers; d.G = c->n_group; d.M = c->n_mel;
  d.BT = (long long)batch * d.Tp;
  d.KH = c->kernel_h;
  return d;
}

// PermuteHeight index list of flow k (efficient_modules.py:341-353,377-383)
void wf_perm(int k, int h, int* idx) {
  for (int i = 0; i < h; ++i) idx[i] = i;
  if (k % 4 == 2 || k % 4 == 3) {
    int half = h / 2;
    for (int i = 0; i < half; ++i) idx[i] = half - 1 - i;
    for (int i = half; i < h; ++i) idx[i] = h - 1 - (i - half);
  } else {
    for (int i = 0; i < h; ++i) idx[i] = h - 1 - i;
  }
}

// Separable in_layers (cwg_wf_weights.dw_w set) run k_wf_sep_tc, everything else the dense 3x3 kernel.
int wf_check_weights(const cwg_wf_config* c, const cwg_wf_weights* w) {
  CWG_REQUIRE(w->dw_w != nullptr || (c->kernel_h == WF_KH && c->kernel_w == WF_KW),
              "a %dx%d WaveFlow in_layer runs on the tensor cores only as a depthwise-separable conv (cwg_wf_weights.dw_w)",
              c->kernel_h, c->kernel_w);
  CWG_REQUIRE(w->dw_w == nullptr || w->dw_b != nullptr, "dw_b missing");
  return 0;
}

template <bool FULL>
void wf_go(bool sep, int npass, dim3 grid, const CUtensorMap* m, const WfLayerArgs& a, cudaStream_t s) {
  if (sep && npass == 3) k_wf_sep_tc<3, FULL><<<grid, W_THREADS, S_SMEM, s>>>(m[0], m[1], m[2], m[3], m[4], m[5], m[6], m[7], a);
  else if (sep) k_wf_sep_tc<1, FULL><<<grid, W_THREADS, S_SMEM, s>>>(m[0], m[1], m[2], m[3], m[4], m[5], m[6], m[7], a);
  else if (npass == 3) k_wf_layer_tc<3, FULL><<<grid, W_THREADS, W_SMEM, s>>>(m[0], m[1], m[2], m[3], m[4], m[5], m[6], m[7], a);
  else k_wf_layer_tc<1, FULL><<<grid, W_THREADS, W_SMEM, s>>>(m[0], m[1], m[2], m[3], m[4], m[5], m[6], m[7], a);
}

// One WN_2d layer.  row >= 0: the step of AR row `row`, x = the conv-queue rings [L][KH][B][T'][C] (hi plane, then lo).
// row < 0 (forward direction): all G-1 height rows in one launch, x = two full-height buffers [2][G-1][B][T'][C] per plane;
// layer l reads buffer l % 2 and writes buffer (l + 1) % 2, eo is [G-1][B*T'][16].
int wf_launch_layer(const cwg_wf_config* cfg, const WfDims& d, const cwg_wf_weights* w, int npass, int flow, int layer,
                    int row, __nv_bfloat16* x, const __nv_bfloat16* mel_up, float* eo, cudaStream_t s) {
  const bool sep = w->dw_w != nullptr, full = row < 0;
  const uint64_t xrows = full ? 2ull * (d.G - 1) : (uint64_t)d.L * d.KH;
  const size_t xplane = (size_t)xrows * d.BT * WF_C, mplane = (size_t)d.BT * WF_HP;
  const uint64_t fl = (uint64_t)d.F * d.L;
  CUtensorMap tx_hi, tx_lo, tm_hi, tm_lo, tw1_hi, tw1_lo, tw2_hi, tw2_lo;
  {
    uint64_t dims[4] = {WF_C, (uint64_t)d.Tp, (uint64_t)d.B, xrows};
    uint64_t st[3] = {WF_C * 2, (uint64_t)d.Tp * WF_C * 2, (uint64_t)d.BT * WF_C * 2};
    uint32_t box[4] = {64, 128, 1, 1};
    if (int r = make_map(&tx_hi, x, 4, dims, st, box)) return r;
    if (int r = make_map(&tx_lo, x + xplane, 4, dims, st, box)) return r;
  }
  if (int r = map_act(&tm_hi, mel_up, WF_HP, d.Tp, d.B)) return r;
  if (int r = map_act(&tm_lo, mel_up + mplane, WF_HP, d.Tp, d.B)) return r;
  const uint64_t k1 = sep ? WF_C + WF_HP : WF_K1;               // separable: pointwise columns | mel
  if (int r = map_2d(&tw1_hi, w->w1_hi, k1, fl * 2 * WF_C, 256)) return r;
  if (int r = map_2d(&tw1_lo, w->w1_lo, k1, fl * 2 * WF_C, 256)) return r;
  if (int r = map_2d(&tw2_hi, w->w2_hi, WF_C, fl * WF_N2, WF_N2)) return r;
  if (int r = map_2d(&tw2_lo, w->w2_lo, WF_C, fl * WF_N2, WF_N2)) return r;
  const size_t idx = (size_t)flow * d.L + layer;
  WfLayerArgs a{};
  a.b1 = w->b1 + idx * 2 * WF_C; a.b2 = w->b2 + idx * WF_C; a.eo_b = w->eo_b + (size_t)flow * CWG_EO_PAD;
  a.eo = eo; a.Tp = d.Tp; a.dil = 1 << layer;
  a.w1_row0 = (int)(idx * 2 * WF_C); a.w2_row0 = (int)(idx * WF_N2);
  if (full) {
    a.ring_in = (layer & 1) * (d.G - 1); a.ring_out = ((layer + 1) & 1) * (d.G - 1);
  } else {
    a.ring_in = layer * d.KH; a.ring_out = (layer + 1) * d.KH;
    a.row = row; a.rows_valid = row + 1 < WF_KH ? row + 1 : WF_KH;
  }
  a.has_res = layer < d.L - 1; a.first = layer == 0;
  a.x = x; a.xplane = (long long)xplane; a.BT = d.BT;
  dim3 grid((unsigned)((d.Tp + 127) / 128), d.B, full ? d.G - 1 : 1);
  if (sep) {
    a.kh = cfg->kernel_h; a.kw = cfg->kernel_w;
    a.dw_w = w->dw_w + idx * WF_C * a.kh * a.kw; a.dw_b = w->dw_b + idx * WF_C;
  }
  if (full) {
    if (int r = sep ? (npass == 3 ? set_smem(k_wf_sep_tc<3, true>, S_SMEM) : set_smem(k_wf_sep_tc<1, true>, S_SMEM))
                    : (npass == 3 ? set_smem(k_wf_layer_tc<3, true>, W_SMEM) : set_smem(k_wf_layer_tc<1, true>, W_SMEM)))
      return r;
  } else {
    if (int r = sep ? (npass == 3 ? set_smem(k_wf_sep_tc<3>, S_SMEM) : set_smem(k_wf_sep_tc<1>, S_SMEM))
                    : (npass == 3 ? set_smem(k_wf_layer_tc<3>, W_SMEM) : set_smem(k_wf_layer_tc<1>, W_SMEM)))
      return r;
  }
  const CUtensorMap maps[8] = {tx_hi, tx_lo, tm_hi, tm_lo, tw1_hi, tw1_lo, tw2_hi, tw2_lo};
  if (full) wf_go<true>(sep, npass, grid, maps, a, s);
  else wf_go<false>(sep, npass, grid, maps, a, s);
  CWG_CHECK_CUDA(cudaGetLastError());
  return 0;
}

}  // namespace
}  // namespace cwg

using namespace cwg;

extern "C" {

size_t cwg_wf_workspace_bytes(const cwg_wf_config* cfg, int mode, int batch, int frames, int t_samples) {
  (void)frames;
  if (mode == CWG_MODE_FFMA) return wff_workspace_bytes(cfg, batch, t_samples);
  if (wf_check(cfg, mode, batch, t_samples)) return 0;
  WfDims d = wf_dims(cfg, batch, t_samples);
  WfWorkspace ws;
  wf_carve(d, nullptr, &ws);
  return ws.bytes + 1024;
}

int cwg_wf_launch_count(const cwg_wf_config* cfg) {
  if (!cfg) return -1;
  return 1 + cfg->n_flows * (1 + (cfg->n_group - 1) * (cfg->n_layers + 1));
}

int cwg_wf_layer(const cwg_wf_config* cfg, const cwg_wf_weights* w, int mode, int flow, int layer, int row,
                 void* x_rings, const void* mel_up, float* eo, int batch, int t_samples, void* cuda_stream) {
  if (int r = wf_check(cfg, mode, batch, t_samples)) return r;
  CWG_REQUIRE(w && w->w1_hi && w->w1_lo && w->w2_hi && w->w2_lo && w->b1 && w->b2 && w->eo_b, "missing weight arrays");
  if (int r = wf_check_weights(cfg, w)) return r;
  CWG_REQUIRE(flow >= 0 && flow < cfg->n_flows && layer >= 0 && layer < cfg->n_layers && row >= 0 && row < cfg->n_group - 1,
              "flow/layer/row out of range");
  WfDims d = wf_dims(cfg, batch, t_samples);
  return wf_launch_layer(cfg, d, w, mode == CWG_MODE_BF16X3 ? 3 : 1, flow, layer, row, (__nv_bfloat16*)x_rings,
                         (const __nv_bfloat16*)mel_up, eo, (cudaStream_t)cuda_stream);
}

int cwg_wf_infer(const cwg_wf_config* cfg, const cwg_wf_weights* w, int mode,
                 const float* mel, int frames, int pad_frames, const float* z, float sigma,
                 float* audio, void* workspace, size_t workspace_bytes,
                 int batch, int t_samples, void* cuda_stream) {
  return cwg_wf_infer_profiled(cfg, w, mode, mel, frames, pad_frames, z, sigma, audio, workspace, workspace_bytes, batch,
                               t_samples, cuda_stream, nullptr, nullptr, 0);
}

int cwg_wf_infer_profiled(const cwg_wf_config* cfg, const cwg_wf_weights* w, int mode,
                          const float* mel, int frames, int pad_frames, const float* z, float sigma,
                          float* audio, void* workspace, size_t workspace_bytes,
                          int batch, int t_samples, void* cuda_stream,
                          void** layer_ev_begin, void** layer_ev_end, int n_events) {
  if (mode == CWG_MODE_FFMA) {
    CWG_REQUIRE(n_events == 0 || (layer_ev_begin && layer_ev_end), "event arrays are NULL");
    CWG_REQUIRE(mel && z && audio && frames >= 1 && pad_frames >= 0, "bad tensor arguments");
    CWG_REQUIRE(workspace != nullptr && ((uintptr_t)workspace % 1024) == 0, "workspace must be 1024-byte aligned");
    return wff_infer(cfg, w, mel, frames, pad_frames, z, sigma, audio, workspace, workspace_bytes, batch, t_samples,
                     (cudaStream_t)cuda_stream, layer_ev_begin, layer_ev_end, n_events);
  }
  if (int r = wf_check(cfg, mode, batch, t_samples)) return r;
  CWG_REQUIRE(n_events == 0 || (layer_ev_begin && layer_ev_end), "event arrays are NULL");
  int ev = 0;
  CWG_REQUIRE(w && w->w1_hi && w->w1_lo && w->w2_hi && w->w2_lo && w->b1 && w->b2 && w->eo_b && w->start_w && w->start_b,
              "missing weight arrays");
  if (int r = wf_check_weights(cfg, w)) return r;
  CWG_REQUIRE(mel && z && audio && frames >= 1 && pad_frames >= 0, "bad tensor arguments");
  CWG_REQUIRE(workspace != nullptr && ((uintptr_t)workspace % 1024) == 0, "workspace must be 1024-byte aligned");
  WfDims d = wf_dims(cfg, batch, t_samples);
  WfWorkspace ws;
  wf_carve(d, workspace, &ws);
  CWG_REQUIRE(ws.bytes <= workspace_bytes, "workspace too small: need %zu, got %zu", ws.bytes, workspace_bytes);
  cudaStream_t s = (cudaStream_t)cuda_stream;
  const int npass = mode == CWG_MODE_BF16X3 ? 3 : 1;
  const int h = d.G, F = d.F, L = d.L;
  const size_t xplane = (size_t)L * d.KH * d.BT * WF_C, slot_elems = (size_t)d.BT * WF_C, mplane = (size_t)d.BT * WF_HP;

  {   // cond = interpolate(mel) once; every flow's cond layer rides in its W1 columns
    long long n = d.BT * WF_HP;
    k_wf_mel_up<<<(unsigned)((n + 255) / 256), 256, 0, s>>>(mel, ws.mel_up, ws.mel_up + mplane, d.B, d.M, frames,
                                                           frames + pad_frames, d.Tp, cfg->upsample_linear);
    CWG_CHECK_CUDA(cudaGetLastError());
  }
  // phys[c]: physical column of logical height row c in the state buffer (PermuteHeight is bookkeeping)
  int phys[WF_TC_MAX_GROUP], perm[WF_TC_MAX_GROUP], nxt[WF_TC_MAX_GROUP];
  for (int c = 0; c < h; ++c) phys[c] = c;
  const unsigned row_grid = (unsigned)((d.BT + 63) / 64);
  for (int k = F - 1; k >= 0; --k) {                                   // efficient_model_ax.py:325
    wf_perm(k, h, perm);
    const bool first_flow = k == F - 1, last_flow = k == 0;
    for (int i = -1; i < h - 1; ++i) {                                  // efficient_modules.py:49,56
      if (i >= 0)
        for (int l = 0; l < L; ++l, ++ev) {
          if (ev < n_events) CWG_CHECK_CUDA(cudaEventRecord((cudaEvent_t)layer_ev_begin[ev], s));
          if (int r = wf_launch_layer(cfg, d, w, npass, k, l, i, ws.x, ws.mel_up, ws.eo, s)) return r;
          if (ev < n_events) CWG_CHECK_CUDA(cudaEventRecord((cudaEvent_t)layer_ev_end[ev], s));
        }
      const int j = i + 1;                                              // logical row produced now
      WfRowP p{};
      p.BT = d.BT; p.G = h;
      p.in = first_flow ? z : ws.state; p.in_scale = first_flow ? sigma : 1.f; p.col_in = phys[j];
      // the last flow writes straight into `audio` at the column its PermuteHeight sends row j to
      p.out = last_flow ? audio : ws.state;
      p.col_out = last_flow ? perm[j] : phys[j];
      p.eo = ws.eo; p.do_couple = i >= 0;
      p.start_w = w->start_w + (size_t)k * WF_C; p.start_b = w->start_b + (size_t)k * WF_C;
      if (j < h - 1) {
        p.x_hi = ws.x + (size_t)(j % d.KH) * slot_elems;                // ring of layer 0
        p.x_lo = p.x_hi + xplane;
      }
      k_wf_row<<<row_grid, 256, 0, s>>>(p);
      CWG_CHECK_CUDA(cudaGetLastError());
    }
    for (int c = 0; c < h; ++c) nxt[c] = phys[perm[c]];                 // z = permute_channels(audio_out), :336-337
    for (int c = 0; c < h; ++c) phys[c] = nxt[c];
  }
  return 0;
}

static int wf_fwd_check(const cwg_wf_config* cfg, int mode, int batch, int t_samples) {
  CWG_REQUIRE(cfg != nullptr, "cfg is NULL");
  CWG_REQUIRE(mode != CWG_MODE_FFMA, "the WaveFlow forward direction runs in CWG_MODE_BF16X3 / CWG_MODE_BF16 only, not CWG_MODE_FFMA");
  return wf_check(cfg, mode, batch, t_samples);
}

size_t cwg_wf_forward_workspace_bytes(const cwg_wf_config* cfg, int mode, int batch, int frames, int t_samples) {
  if (wf_fwd_check(cfg, mode, batch, t_samples)) return 0;
  if (frames < 1) { set_error("frames must be >= 1"); return 0; }
  WfDims d = wf_dims(cfg, batch, t_samples);
  WfFwdWorkspace ws;
  wf_fwd_carve(d, nullptr, &ws);
  return ws.bytes + 1024;
}

int cwg_wf_forward_launch_count(const cwg_wf_config* cfg) {
  if (!cfg) return -1;
  return cfg->n_flows * (cfg->n_layers + 1) + 3;      // mel, F + 1 boundaries, F * L full-height layers, reduction
}

int cwg_wf_forward_layer(const cwg_wf_config* cfg, const cwg_wf_weights* w, int mode, int flow, int layer, void* x_bufs,
                         const void* mel_up, float* eo, int batch, int t_samples, void* cuda_stream) {
  if (int r = wf_fwd_check(cfg, mode, batch, t_samples)) return r;
  CWG_REQUIRE(w && w->w1_hi && w->w1_lo && w->w2_hi && w->w2_lo && w->b1 && w->b2 && w->eo_b, "missing weight arrays (NULL)");
  if (int r = wf_check_weights(cfg, w)) return r;
  CWG_REQUIRE(x_bufs && mel_up && eo, "NULL tensor argument");
  CWG_REQUIRE(flow >= 0 && flow < cfg->n_flows && layer >= 0 && layer < cfg->n_layers, "flow/layer out of range");
  WfDims d = wf_dims(cfg, batch, t_samples);
  return wf_launch_layer(cfg, d, w, mode == CWG_MODE_BF16X3 ? 3 : 1, flow, layer, -1, (__nv_bfloat16*)x_bufs,
                         (const __nv_bfloat16*)mel_up, eo, (cudaStream_t)cuda_stream);
}

int cwg_wf_forward(const cwg_wf_config* cfg, const cwg_wf_weights* w, int mode, const float* mel, int frames,
                   const float* audio, int t_samples, float* z, double* logp_terms, void* workspace, size_t workspace_bytes,
                   int batch, void* cuda_stream) {
  if (int r = wf_fwd_check(cfg, mode, batch, t_samples)) return r;
  CWG_REQUIRE(w && w->w1_hi && w->w1_lo && w->w2_hi && w->w2_lo && w->b1 && w->b2 && w->eo_b && w->start_w && w->start_b,
              "missing weight arrays (NULL)");
  if (int r = wf_check_weights(cfg, w)) return r;
  CWG_REQUIRE(mel && audio && z && logp_terms, "NULL tensor argument");
  CWG_REQUIRE(frames >= 1, "frames must be >= 1");
  CWG_REQUIRE(workspace != nullptr && ((uintptr_t)workspace % 1024) == 0, "workspace must be 1024-byte aligned (NULL)");
  WfDims d = wf_dims(cfg, batch, t_samples);
  WfFwdWorkspace ws;
  wf_fwd_carve(d, workspace, &ws);
  CWG_REQUIRE(ws.bytes <= workspace_bytes, "workspace too small: need %zu, got %zu", ws.bytes, workspace_bytes);
  cudaStream_t s = (cudaStream_t)cuda_stream;
  const int npass = mode == CWG_MODE_BF16X3 ? 3 : 1;
  const int h = d.G, F = d.F, L = d.L, nblk = wf_fwd_blocks(d.Tp);
  const long long xplane = 2ll * (h - 1) * d.BT * WF_C;
  {
    const long long n = d.BT * WF_HP, mplane = n;
    k_wf_mel_up<<<(unsigned)((n + 255) / 256), 256, 0, s>>>(mel, ws.mel_up, ws.mel_up + mplane, d.B, d.M, frames, frames,
                                                           d.Tp, cfg->upsample_linear);
    CWG_CHECK_CUDA(cudaGetLastError());
  }
  // phys[c]: physical column of logical height row c in z; x = permute_height(x, k) before flow k's coupling
  int phys[WF_TC_MAX_GROUP], perm[WF_TC_MAX_GROUP], nxt[WF_TC_MAX_GROUP];
  for (int c = 0; c < h; ++c) phys[c] = c;
  auto permute = [&](int k) {
    wf_perm(k, h, perm);
    for (int c = 0; c < h; ++c) nxt[c] = phys[perm[c]];
    for (int c = 0; c < h; ++c) phys[c] = nxt[c];
  };
  permute(0);
  if (int r = launch_wf_fwd_boundary(d.B, d.Tp, h, F, audio, z, nullptr, nullptr, phys, w->start_w, w->start_b, ws.x, xplane,
                                     nullptr, nullptr, ws.ld_zero, s)) return r;
  for (int k = 0; k < F; ++k) {
    for (int l = 0; l < L; ++l)
      if (int r = wf_launch_layer(cfg, d, w, npass, k, l, -1, ws.x, ws.mel_up, ws.eo, s)) return r;
    int done[WF_TC_MAX_GROUP];
    for (int c = 0; c < h; ++c) done[c] = phys[c];
    const bool last = k + 1 == F;
    if (!last) permute(k + 1);
    if (int r = launch_wf_fwd_boundary(d.B, d.Tp, h, F, nullptr, z, ws.eo, done, last ? nullptr : phys,
                                       last ? nullptr : w->start_w + (size_t)(k + 1) * WF_C,
                                       last ? nullptr : w->start_b + (size_t)(k + 1) * WF_C, ws.x, xplane,
                                       ws.ls_part + (size_t)k * d.B * nblk, last ? ws.z2_part : nullptr, nullptr, s)) return r;
  }
  return launch_fwd_reduce(F, d.B, nblk, d.Tp, ws.ls_part, ws.z2_part, ws.ld_zero, logp_terms, s);
}

}  // extern "C"
