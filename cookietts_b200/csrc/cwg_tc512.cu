// WN layer for n_channels = 512 (BASELINE config 4 model) on tcgen05.  The pre-activation of one
// 128-step tile is [128 x 1024] fp32 - twice the 512 TMEM columns - and the res/skip accumulator
// [128 x 528] does not fit either, so the layer is two kernels with the gated activations staged
// in HBM as bf16 hi/lo planes (2-4 KB per group-step, still far on the compute side of the ridge):
//
//   k_gate512_tc : grid.z = channel half p.  GEMM1 for tanh rows [256p, 256p+256) and the matching
//                  sigmoid rows (K = 3*512 + 256 = 28 k-blocks) -> gate -> acts[:, 256p:256p+256]
//   k_res512_tc  : grid.z = res channel half q.  acts [128 x 512] x W2[256q:256q+256]^T (8 k-blocks),
//                  residual add + TMA store; the q = 0 CTAs also accumulate the folded `end` (N = 16).
//
// Same reference lines as cwg_ps.cu (glow.py:201-222).
#include "cwg_tc_common.cuh"

namespace cwg {

using namespace sm100;
using namespace tc;

namespace {

constexpr int C5 = 512;
constexpr int G_NS = 12, G_NA = 4, G_NBAR = 8;
// k_gate512: [12 units][b1 2 KB][barriers]; k_res512: [12 units][Wse 8 kb x 2 planes x 2 KB][b2 1 KB][barriers]
constexpr int GA_OFF_B1 = G_NS * TILE_A;
constexpr int GA_OFF_BAR = GA_OFF_B1 + 2048;
constexpr int GA_SMEM = GA_OFF_BAR + 256 + 1024;
constexpr int GR_OFF_WSE = G_NS * TILE_A;
constexpr int GR_OFF_B2 = GR_OFF_WSE + 32768;
constexpr int GR_OFF_BAR = GR_OFF_B2 + 1024;
constexpr int GR_SMEM = GR_OFF_BAR + 256 + 1024;        // 231680 <= 232448
constexpr int G_THREADS = 384;

struct Gate512Args {
  const float* b1;       // [2C] of this layer
  int Tp, dil, w1_row0;
};

template <int NPASS>
__global__ void __launch_bounds__(G_THREADS, 1)
k_gate512_tc(const __grid_constant__ CUtensorMap tm_x_hi, const __grid_constant__ CUtensorMap tm_x_lo,
             const __grid_constant__ CUtensorMap tm_h_hi, const __grid_constant__ CUtensorMap tm_h_lo,
             const __grid_constant__ CUtensorMap tm_w1_hi, const __grid_constant__ CUtensorMap tm_w1_lo,
             const __grid_constant__ CUtensorMap tm_a_hi, const __grid_constant__ CUtensorMap tm_a_lo, Gate512Args a) {
  constexpr int PL = NPASS == 3 ? 2 : 1;
  constexpr int NKB = 3 * C5 / 64 + 4;                  // 28
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = align_1024(smem_raw);
  float* b1s = reinterpret_cast<float*>(smem + GA_OFF_B1);
  uint64_t* full = reinterpret_cast<uint64_t*>(smem + GA_OFF_BAR);
  uint64_t* empty = full + G_NBAR;
  uint64_t* acc1_full = empty + G_NBAR;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(acc1_full + 1);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int t0 = blockIdx.x * 128, b = blockIdx.y, p = blockIdx.z;
  auto slot = [&](int i) { return smem + i * TILE_A; };
  auto bslot = [&](int j) { return smem + (G_NA + 2 * j) * TILE_A; };

  if (threadIdx.x == 0) {
    for (int i = 0; i < G_NBAR; ++i) { mbar_init(&full[i], 1); mbar_init(&empty[i], 1); }
    mbar_init(acc1_full, 1);
    fence_barrier_init();
  }
  if (warp == 1) tmem_alloc(tmem_slot, 512);
  if (warp >= 4) {
    const int e = threadIdx.x - 128;
    b1s[e] = __ldg(a.b1 + 256 * p + e);
    b1s[256 + e] = __ldg(a.b1 + C5 + 256 * p + e);
  }
  tc_fence_before_sync();
  __syncthreads();
  tc_fence_after_sync();
  const uint32_t tmem = *tmem_slot;

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&tm_x_hi); tma_prefetch_desc(&tm_h_hi);
    int s = 0; uint32_t pm = 0;
    for (int kb = 0; kb < NKB; ++kb)
      for (int pl = 0; pl < PL; ++pl) {
        mbar_wait(&empty[s], ((pm >> s) & 1u) ^ 1u);
        pm ^= 1u << s;
        mbar_arrive_expect_tx(&full[s], TILE_A);
        if (kb < 24) {
          const int tap = kb >> 3, cb = kb & 7;
          tma_load_3d(slot(s), pl ? &tm_x_lo : &tm_x_hi, &full[s], cb * 64, t0 + (tap - 1) * a.dil, b);
        } else {
          tma_load_3d(slot(s), pl ? &tm_h_lo : &tm_h_hi, &full[s], (kb - 24) * 64, t0, b);
        }
        s = (s + 1 == G_NA) ? 0 : s + 1;
      }
  } else if (warp == 2 && lane == 0) {
    tma_prefetch_desc(&tm_w1_hi);
    int j = 0; uint32_t pm = 0;
    for (int kb = 0; kb < NKB; ++kb)
      for (int g = 0; g < 2; ++g)
        for (int pl = 0; pl < PL; ++pl) {
          mbar_wait(&empty[4 + j], ((pm >> j) & 1u) ^ 1u);
          pm ^= 1u << j;
          mbar_arrive_expect_tx(&full[4 + j], 2 * TILE_A);
          tma_load_2d(bslot(j), pl ? &tm_w1_lo : &tm_w1_hi, &full[4 + j], kb * 64, a.w1_row0 + g * C5 + 256 * p);
          j = (j + 1) & 3;
        }
  } else if (warp == 1 && lane == 0) {
    int sa = 0, jb = 0; uint32_t cm = 0;
    auto wait_full = [&](int bar) { mbar_wait(&full[bar], (cm >> bar) & 1u); cm ^= 1u << bar; };
    for (int kb = 0; kb < NKB; ++kb) {
      const int sa_hi = sa; wait_full(sa); sa = (sa + 1) & 3;
      int sa_lo = 0;
      if (NPASS == 3) { sa_lo = sa; wait_full(sa); sa = (sa + 1) & 3; }
      for (int g = 0; g < 2; ++g) {      // slots are waited for just before first use, released right after last use
        const int jb_hi = jb; wait_full(4 + jb); jb = (jb + 1) & 3;
        tc_fence_after_sync();
        const uint32_t d = tmem + g * 256;
        issue_kblock_fast(smem_u32(slot(sa_hi)), smem_u32(bslot(jb_hi)), d, IDESC_N256, kb == 0);
        if (NPASS == 3) {
          issue_kblock_fast(smem_u32(slot(sa_lo)), smem_u32(bslot(jb_hi)), d, IDESC_N256, false);
          umma_commit(&empty[4 + jb_hi]);
          if (g == 1) umma_commit(&empty[sa_lo]);
          const int jb_lo = jb; wait_full(4 + jb); jb = (jb + 1) & 3;
          tc_fence_after_sync();
          issue_kblock_fast(smem_u32(slot(sa_hi)), smem_u32(bslot(jb_lo)), d, IDESC_N256, false);
          umma_commit(&empty[4 + jb_lo]);
        } else {
          umma_commit(&empty[4 + jb_hi]);
        }
      }
      umma_commit(&empty[sa_hi]);
    }
    umma_commit(acc1_full);
  } else if (warp >= 4) {
    const int quarter = warp & 3, half = (warp - 4) >> 2, row = quarter * 32 + lane;
    const uint32_t trow = tmem + ((uint32_t)(quarter * 32) << 16);
    const float4* b1t = reinterpret_cast<const float4*>(b1s);
    const float4* b1g = reinterpret_cast<const float4*>(b1s + 256);
    mbar_wait(acc1_full, 0);
    tc_fence_after_sync();
    uint32_t buf[2][32];
    const int c0 = half * 8;
    tmem_issue16x2(trow + c0 * 16, trow + 256 + c0 * 16, buf[0]);
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      const int c = c0 + i;
      uint32_t* cur = buf[i & 1];
      tmem_wait32(cur);
      if (i + 1 < 8) tmem_issue16x2(trow + (c + 1) * 16, trow + 256 + (c + 1) * 16, buf[(i + 1) & 1]);
      float act[16];
#pragma unroll
      for (int q = 0; q < 4; ++q) {
        const float4 bt = b1t[c * 4 + q], bs = b1g[c * 4 + q];
        act[4 * q + 0] = gate<NPASS>(__uint_as_float(cur[4 * q + 0]) + bt.x, __uint_as_float(cur[16 + 4 * q + 0]) + bs.x);
        act[4 * q + 1] = gate<NPASS>(__uint_as_float(cur[4 * q + 1]) + bt.y, __uint_as_float(cur[16 + 4 * q + 1]) + bs.y);
        act[4 * q + 2] = gate<NPASS>(__uint_as_float(cur[4 * q + 2]) + bt.z, __uint_as_float(cur[16 + 4 * q + 2]) + bs.z);
        act[4 * q + 3] = gate<NPASS>(__uint_as_float(cur[4 * q + 3]) + bt.w, __uint_as_float(cur[16 + 4 * q + 3]) + bs.w);
      }
      store_split16<NPASS == 3>(act, slot(c >> 2), slot(4 + (c >> 2)), row, (c & 3) * 2);
      if ((i & 3) == 3) {
        fence_proxy_async_smem();
        asm volatile("bar.sync %0, 128;" ::"r"(2 + half) : "memory");
        if (quarter == 0 && lane == 0) {
          const int kb = c >> 2;
          tma_store_3d(&tm_a_hi, slot(kb), 256 * p + kb * 64, t0, b);
          if (NPASS == 3) tma_store_3d(&tm_a_lo, slot(4 + kb), 256 * p + kb * 64, t0, b);
          tma_store_commit();
        }
      }
    }
    if (quarter == 0 && lane == 0) tma_store_wait_read();
    tc_fence_before_sync();
  }
  __syncthreads();
  if (warp == 1) { __syncwarp(); tmem_dealloc(tmem, 512); }
}

struct Res512Args {
  const float* b2;        // [C]
  const float* eo_b;      // [16]
  float* eo;
  int Tp, w2_row0, has_res, first;
};

template <int NPASS>
__global__ void __launch_bounds__(G_THREADS, 1)
k_res512_tc(const __grid_constant__ CUtensorMap tm_a_hi, const __grid_constant__ CUtensorMap tm_a_lo,
            const __grid_constant__ CUtensorMap tm_w2_hi, const __grid_constant__ CUtensorMap tm_w2_lo,
            const __grid_constant__ CUtensorMap tm_wse_hi, const __grid_constant__ CUtensorMap tm_wse_lo,
            const __grid_constant__ CUtensorMap tm_x_hi, const __grid_constant__ CUtensorMap tm_x_lo,
            const __grid_constant__ CUtensorMap tm_xo_hi, const __grid_constant__ CUtensorMap tm_xo_lo, Res512Args a) {
  constexpr int PL = NPASS == 3 ? 2 : 1;
  constexpr int NKB = C5 / 64;                          // 8
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = align_1024(smem_raw);
  float* b2s = reinterpret_cast<float*>(smem + GR_OFF_B2);
  uint64_t* full = reinterpret_cast<uint64_t*>(smem + GR_OFF_BAR);
  uint64_t* empty = full + G_NBAR;
  uint64_t* wse_full = empty + G_NBAR;
  uint64_t* acc2_full = wse_full + 1;
  uint64_t* xold_full = acc2_full + 1;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(xold_full + 1);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int t0 = blockIdx.x * 128, b = blockIdx.y, q = blockIdx.z;
  const bool do_eo = q == 0, do_res = a.has_res != 0;
  auto slot = [&](int i) { return smem + i * TILE_A; };
  auto bslot = [&](int j) { return smem + (G_NA + 2 * j) * TILE_A; };
  auto wse = [&](int plane, int kb) { return smem + GR_OFF_WSE + plane * 16384 + kb * 2048; };

  if (threadIdx.x == 0) {
    for (int i = 0; i < G_NBAR; ++i) { mbar_init(&full[i], 1); mbar_init(&empty[i], 1); }
    mbar_init(wse_full, 1); mbar_init(acc2_full, 1); mbar_init(xold_full, 1);
    fence_barrier_init();
  }
  if (warp == 1) tmem_alloc(tmem_slot, 512);
  if (warp >= 4) b2s[threadIdx.x - 128] = __ldg(a.b2 + 256 * q + (threadIdx.x - 128));
  tc_fence_before_sync();
  __syncthreads();
  tc_fence_after_sync();
  const uint32_t tmem = *tmem_slot;

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&tm_a_hi);
    if (do_eo) {
      mbar_arrive_expect_tx(wse_full, NKB * 2048 * PL);
      for (int kb = 0; kb < NKB; ++kb) {
        tma_load_2d(wse(0, kb), &tm_wse_hi, wse_full, kb * 64, a.w2_row0 + C5);
        if (NPASS == 3) tma_load_2d(wse(1, kb), &tm_wse_lo, wse_full, kb * 64, a.w2_row0 + C5);
      }
    }
    int s = 0; uint32_t pm = 0;
    for (int kb = 0; kb < NKB; ++kb)
      for (int pl = 0; pl < PL; ++pl) {
        mbar_wait(&empty[s], ((pm >> s) & 1u) ^ 1u);
        pm ^= 1u << s;
        mbar_arrive_expect_tx(&full[s], TILE_A);
        tma_load_3d(slot(s), pl ? &tm_a_lo : &tm_a_hi, &full[s], kb * 64, t0, b);
        s = (s + 1 == G_NA) ? 0 : s + 1;
      }
  } else if (warp == 2 && lane == 0) {
    if (do_res) {
      tma_prefetch_desc(&tm_w2_hi);
      int j = 0; uint32_t pm = 0;
      for (int kb = 0; kb < NKB; ++kb)
        for (int pl = 0; pl < PL; ++pl) {
          mbar_wait(&empty[4 + j], ((pm >> j) & 1u) ^ 1u);
          pm ^= 1u << j;
          mbar_arrive_expect_tx(&full[4 + j], 2 * TILE_A);
          tma_load_2d(bslot(j), pl ? &tm_w2_lo : &tm_w2_hi, &full[4 + j], kb * 64, a.w2_row0 + 256 * q);
          j = (j + 1) & 3;
        }
    }
  } else if (warp == 1 && lane == 0) {
    int sa = 0, jb = 0; uint32_t cm = 0;
    auto wait_full = [&](int bar) { mbar_wait(&full[bar], (cm >> bar) & 1u); cm ^= 1u << bar; };
    if (do_eo) mbar_wait(wse_full, 0);
    const uint32_t d16 = tmem + 256;
    for (int kb = 0; kb < NKB; ++kb) {
      const int sa_hi = sa; wait_full(sa); sa = (sa + 1) & 3;
      int sa_lo = 0;
      if (NPASS == 3) { sa_lo = sa; wait_full(sa); sa = (sa + 1) & 3; }
      int jb_hi = 0, jb_lo = 0;
      if (do_res) {
        jb_hi = jb; wait_full(4 + jb); jb = (jb + 1) & 3;
        if (NPASS == 3) { jb_lo = jb; wait_full(4 + jb); jb = (jb + 1) & 3; }
      }
      tc_fence_after_sync();
      const uint32_t a_hi = smem_u32(slot(sa_hi)), a_lo = smem_u32(slot(sa_lo));
      const uint32_t r_hi = smem_u32(bslot(jb_hi)), r_lo = smem_u32(bslot(jb_lo));
      const uint32_t w_hi = smem_u32(wse(0, kb)), w_lo = smem_u32(wse(1, kb));
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        const uint32_t o = 32 * k, acc = (kb | k) ? 1u : 0u;
        if (do_res) umma_bf16(tmem, umma_desc_sw128(a_hi + o), umma_desc_sw128(r_hi + o), IDESC_N256, acc);
        if (do_eo) umma_bf16(d16, umma_desc_sw128(a_hi + o), umma_desc_sw128(w_hi + o), IDESC_N16, acc);
        if (NPASS == 3) {
          if (do_res) umma_bf16(tmem, umma_desc_sw128(a_lo + o), umma_desc_sw128(r_hi + o), IDESC_N256, 1u);
          if (do_eo) umma_bf16(d16, umma_desc_sw128(a_lo + o), umma_desc_sw128(w_hi + o), IDESC_N16, 1u);
          if (do_res) umma_bf16(tmem, umma_desc_sw128(a_hi + o), umma_desc_sw128(r_lo + o), IDESC_N256, 1u);
          if (do_eo) umma_bf16(d16, umma_desc_sw128(a_hi + o), umma_desc_sw128(w_lo + o), IDESC_N16, 1u);
        }
      }
      if (do_res) { umma_commit(&empty[4 + jb_hi]); if (NPASS == 3) umma_commit(&empty[4 + jb_lo]); }
      umma_commit(&empty[sa_hi]);
      if (NPASS == 3) umma_commit(&empty[sa_lo]);
    }
    umma_commit(acc2_full);
    if (do_res) {
      mbar_wait(acc2_full, 0);
      mbar_arrive_expect_tx(xold_full, 8 * TILE_A);
      for (int kb = 0; kb < 4; ++kb) {
        tma_load_3d(slot(kb), &tm_x_hi, xold_full, 256 * q + kb * 64, t0, b);
        tma_load_3d(slot(4 + kb), &tm_x_lo, xold_full, 256 * q + kb * 64, t0, b);
      }
    }
  } else if (warp >= 4) {
    const int quarter = warp & 3, half = (warp - 4) >> 2, row = quarter * 32 + lane;
    const uint32_t trow = tmem + ((uint32_t)(quarter * 32) << 16);
    const bool valid = t0 + row < a.Tp;
    const size_t m = (size_t)b * a.Tp + (size_t)min(t0 + row, a.Tp - 1);
    float4 eold[4];
    if (do_eo && half == 0) {
      const float4* e = reinterpret_cast<const float4*>(a.first ? a.eo_b : a.eo + m * CWG_EO_PAD);
#pragma unroll
      for (int i = 0; i < 4; ++i) eold[i] = __ldg(e + i);
    }
    mbar_wait(acc2_full, 0);
    tc_fence_after_sync();
    if (do_eo && half == 0) {
      uint32_t sk[16];
      tmem_issue16(trow + 256, sk);
      tmem_wait16(sk);
      if (valid) {
        float4* e = reinterpret_cast<float4*>(a.eo + m * CWG_EO_PAD);
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          float4 v = eold[i];
          v.x += __uint_as_float(sk[4 * i]); v.y += __uint_as_float(sk[4 * i + 1]);
          v.z += __uint_as_float(sk[4 * i + 2]); v.w += __uint_as_float(sk[4 * i + 3]);
          e[i] = v;
        }
      }
    }
    if (do_res) {
      const float4* b2v = reinterpret_cast<const float4*>(b2s);
      uint32_t buf[2][16];
      const int c0 = half * 8;
      tmem_issue16(trow + c0 * 16, buf[0]);
      mbar_wait(xold_full, 0);
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        const int c = c0 + i;
        uint32_t* cur = buf[i & 1];
        tmem_wait16(cur);
        if (i + 1 < 8) tmem_issue16(trow + (c + 1) * 16, buf[(i + 1) & 1]);
        uint8_t* thi = slot(c >> 2);
        uint8_t* tlo = slot(4 + (c >> 2));
        const uint32_t o0 = sw128_offset(row, (c & 3) * 2), o1 = sw128_offset(row, (c & 3) * 2 + 1);
        const uint4 h0 = *reinterpret_cast<const uint4*>(thi + o0), h1 = *reinterpret_cast<const uint4*>(thi + o1);
        const uint4 l0 = *reinterpret_cast<const uint4*>(tlo + o0), l1 = *reinterpret_cast<const uint4*>(tlo + o1);
        const uint32_t hw[8] = {h0.x, h0.y, h0.z, h0.w, h1.x, h1.y, h1.z, h1.w};
        const uint32_t lw[8] = {l0.x, l0.y, l0.z, l0.w, l1.x, l1.y, l1.z, l1.w};
        float r[16];
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          const float4 bb = b2v[c * 4 + j];
          r[4 * j] = __uint_as_float(cur[4 * j]) + bb.x; r[4 * j + 1] = __uint_as_float(cur[4 * j + 1]) + bb.y;
          r[4 * j + 2] = __uint_as_float(cur[4 * j + 2]) + bb.z; r[4 * j + 3] = __uint_as_float(cur[4 * j + 3]) + bb.w;
        }
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          r[2 * j] += __uint_as_float(hw[j] << 16) + __uint_as_float(lw[j] << 16);
          r[2 * j + 1] += __uint_as_float(hw[j] & 0xFFFF0000u) + __uint_as_float(lw[j] & 0xFFFF0000u);
        }
        store_split16<true>(r, thi, tlo, row, (c & 3) * 2);
        if ((i & 3) == 3) {
          fence_proxy_async_smem();
          asm volatile("bar.sync %0, 128;" ::"r"(2 + half) : "memory");
          if (quarter == 0 && lane == 0) {
            const int kb = c >> 2;
            tma_store_3d(&tm_xo_hi, slot(kb), 256 * q + kb * 64, t0, b);
            tma_store_3d(&tm_xo_lo, slot(4 + kb), 256 * q + kb * 64, t0, b);
            tma_store_commit();
          }
        }
      }
      if (quarter == 0 && lane == 0) tma_store_wait_read();
    }
    tc_fence_before_sync();
  }
  __syncthreads();
  if (warp == 1) { __syncwarp(); tmem_dealloc(tmem, 512); }
}

}  // namespace

int launch_layer_tc512(const Dims& d, const cwg_weights* w, int npass, int flow, int layer,
                       const __nv_bfloat16* x_in, __nv_bfloat16* x_out, const __nv_bfloat16* h2,
                       __nv_bfloat16* acts, float* eo, cudaStream_t s) {
  CWG_REQUIRE(d.MG == 16 && d.b1_batch == nullptr, "the 512-channel kernels take n_group <= 16 and a shared gate bias");
  const size_t plane = (size_t)d.BT * d.C, hplane = (size_t)d.BT * d.H;
  const uint64_t fl = (uint64_t)d.F * d.L;
  CUtensorMap tx_hi, tx_lo, th_hi, th_lo, tw1_hi, tw1_lo, ta_hi, ta_lo, tw2_hi, tw2_lo, tse_hi, tse_lo, to_hi, to_lo;
  if (int r = map_act(&tx_hi, x_in, d.C, d.Tp, d.B)) return r;
  if (int r = map_act(&tx_lo, x_in + plane, d.C, d.Tp, d.B)) return r;
  if (int r = map_act(&th_hi, h2, d.H, d.Tp, d.B)) return r;
  if (int r = map_act(&th_lo, h2 + hplane, d.H, d.Tp, d.B)) return r;
  if (int r = map_2d(&tw1_hi, w->w1_hi, d.K1, fl * 2 * d.C, 256)) return r;
  if (int r = map_2d(&tw1_lo, w->w1_lo, d.K1, fl * 2 * d.C, 256)) return r;
  if (int r = map_act(&ta_hi, acts, d.C, d.Tp, d.B)) return r;
  if (int r = map_act(&ta_lo, acts + plane, d.C, d.Tp, d.B)) return r;
  if (int r = map_2d(&tw2_hi, w->w2_hi, d.C, fl * d.N2, 256)) return r;
  if (int r = map_2d(&tw2_lo, w->w2_lo, d.C, fl * d.N2, 256)) return r;
  if (int r = map_2d(&tse_hi, w->w2_hi, d.C, fl * d.N2, 16)) return r;
  if (int r = map_2d(&tse_lo, w->w2_lo, d.C, fl * d.N2, 16)) return r;
  if (int r = map_act(&to_hi, x_out, d.C, d.Tp, d.B)) return r;
  if (int r = map_act(&to_lo, x_out + plane, d.C, d.Tp, d.B)) return r;
  const size_t idx = (size_t)flow * d.L + layer;
  const bool has_res = layer < d.L - 1;
  Gate512Args ga{};
  ga.b1 = w->b1 + idx * 2 * d.C; ga.Tp = d.Tp; ga.dil = 1 << layer; ga.w1_row0 = (int)(idx * 2 * d.C);
  Res512Args ra{};
  ra.b2 = w->b2 + idx * d.C; ra.eo_b = w->eo_b + (size_t)flow * CWG_EO_PAD; ra.eo = eo;
  ra.Tp = d.Tp; ra.w2_row0 = (int)(idx * d.N2); ra.has_res = has_res; ra.first = layer == 0;
  dim3 g1((unsigned)((d.Tp + 127) / 128), d.B, 2);
  dim3 g2((unsigned)((d.Tp + 127) / 128), d.B, has_res ? 2 : 1);
  if (npass == 3) {
    if (int r = set_smem(k_gate512_tc<3>, GA_SMEM)) return r;
    if (int r = set_smem(k_res512_tc<3>, GR_SMEM)) return r;
    k_gate512_tc<3><<<g1, G_THREADS, GA_SMEM, s>>>(tx_hi, tx_lo, th_hi, th_lo, tw1_hi, tw1_lo, ta_hi, ta_lo, ga);
    CWG_CHECK_CUDA(cudaGetLastError());
    k_res512_tc<3><<<g2, G_THREADS, GR_SMEM, s>>>(ta_hi, ta_lo, tw2_hi, tw2_lo, tse_hi, tse_lo, tx_hi, tx_lo, to_hi, to_lo, ra);
  } else {
    if (int r = set_smem(k_gate512_tc<1>, GA_SMEM)) return r;
    if (int r = set_smem(k_res512_tc<1>, GR_SMEM)) return r;
    k_gate512_tc<1><<<g1, G_THREADS, GA_SMEM, s>>>(tx_hi, tx_lo, th_hi, th_lo, tw1_hi, tw1_lo, ta_hi, ta_lo, ga);
    CWG_CHECK_CUDA(cudaGetLastError());
    k_res512_tc<1><<<g2, G_THREADS, GR_SMEM, s>>>(ta_hi, ta_lo, tw2_hi, tw2_lo, tse_hi, tse_lo, tx_hi, tx_lo, to_hi, to_lo, ra);
  }
  CWG_CHECK_CUDA(cudaGetLastError());
  return 0;
}

}  // namespace cwg
