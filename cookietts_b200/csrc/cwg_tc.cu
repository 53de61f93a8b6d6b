// Tensor-core path of the WaveGlow inverse pass for sm_100a: TMA-fed tcgen05.mma kernels with
// TMEM accumulators.
//
//   k_cond_tc   : folded upsample+squeeze+cond_layers[0..1] GEMM (glow.py:318-324,198-199)
//                 H2[b, f*P+p, :] = mel4[b, f, :] @ cond_w[p*H:(p+1)*H, :]^T + bias
//
// Operand precision: every fp32 quantity q that feeds an MMA is stored as two bf16 planes,
// q ~= hi + lo.  NPASS = 1 issues hi*hi only (CWG_MODE_BF16); NPASS = 3 issues
// hi*hi + lo*hi + hi*lo (CWG_MODE_BF16X3, ~2^-17 relative operand error).  Accumulation is fp32 in
// TMEM; the residual stream always keeps both planes.
#include "cwg_tc_common.cuh"

namespace cwg {

using namespace sm100;
using namespace tc;

namespace {


// ------------------------------------------------------------------------------------------
// mel4 im2col: mel4[b*Tm + f][j*M + ci] = mel[b][ci][f - j] (0 for f < j), bf16 hi / lo planes
// ------------------------------------------------------------------------------------------
__global__ void k_im2col_mel(const float* __restrict__ mel, __nv_bfloat16* __restrict__ hi, __nv_bfloat16* __restrict__ lo,
                             int B, int M, int Tm, int J, int KCp, int f16) {
  long long n = (long long)B * Tm * KCp;
  long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  long long row = i / KCp; int kk = (int)(i - row * KCp);
  int b = (int)(row / Tm), f = (int)(row - (long long)b * Tm);
  int j = kk / M, ci = kk - j * M;
  float v = (j < J && f >= j) ? mel[((size_t)b * M + ci) * Tm + (f - j)] : 0.f;   // columns >= J*M are zero padding
  if (f16) {                                                                        // CWG_MODE_F16F8: fp16 hi / lo
    const __half h = __float2half_rn(v);
    reinterpret_cast<__half*>(hi)[i] = h;
    reinterpret_cast<__half*>(lo)[i] = __float2half_rn(v - __half2float(h));
    return;
  }
  __nv_bfloat16 h = __float2bfloat16_rn(v);
  hi[i] = h;
  lo[i] = __float2bfloat16_rn(v - __bfloat162float(h));
}

// ------------------------------------------------------------------------------------------
// cond GEMM: tile 128 rows (b,f) x 256 columns (one phase p, all H=256 hidden channels)
// ------------------------------------------------------------------------------------------
struct CondArgs {
  const float* bias;      // cond_bias + flow*H ; [B] stride bias_bstride
  int bias_bstride;
  int M, Tm, B;
  int w_row0;             // flow * P * H
  int nkb;                // KC / 64
  int* range_flag;        // f16f8: |= 2 when an H2 value leaves the fp16 range (may be NULL)
};

template <int NPASS>
struct CondCfg {
  static constexpr int PL = NPASS != 1 ? 2 : 1;               // NPASS 2 (f16f8): three fp16 products like bf16x3
  static constexpr int STAGE = (TILE_A + 2 * TILE_A) * PL;     // A 16 KB + B 32 KB per plane
  // One (bf16x3) / two (bf16) stages of 96 / 48 KB: two CTAs are co-resident per SM (2 x 256 TMEM columns), so one
  // CTA's loads and MMAs overlap the other's epilogue and stores (the K loop is only 5 k-blocks long).
  static constexpr int NST = NPASS != 1 ? 1 : 2;
  static constexpr int SMEM = NST * STAGE + 256 + 1024;
};

template <int NPASS>
__global__ void __launch_bounds__(320, 2)
k_cond_tc(const __grid_constant__ CUtensorMap tm_a_hi, const __grid_constant__ CUtensorMap tm_a_lo,
          const __grid_constant__ CUtensorMap tm_b_hi, const __grid_constant__ CUtensorMap tm_b_lo,
          const __grid_constant__ CUtensorMap tm_c_hi, const __grid_constant__ CUtensorMap tm_c_lo,
          const __grid_constant__ CUtensorMap tm_c_h8, CondArgs a) {   // f16f8: tm_c_lo = e5m2 lo*2^P plane, tm_c_h8 = e5m2 hi*2^-Q
  using Cfg = CondCfg<NPASS>;
  constexpr bool F8 = NPASS == 2;
  constexpr uint32_t ID256 = F8 ? IDESC_F16_N256 : IDESC_N256;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = align_1024(smem_raw);
  uint64_t* full = reinterpret_cast<uint64_t*>(smem + Cfg::NST * Cfg::STAGE);
  uint64_t* empty = full + Cfg::NST;
  uint64_t* acc_full = empty + Cfg::NST;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(acc_full + 1);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int p = blockIdx.x, m0 = blockIdx.y * 128;

  if (threadIdx.x == 0) {
    for (int i = 0; i < Cfg::NST; ++i) { mbar_init(&full[i], 1); mbar_init(&empty[i], 1); }
    mbar_init(acc_full, 1);
    fence_barrier_init();
  }
  if (warp == 1) tmem_alloc(tmem_slot, 256);
  tc_fence_before_sync();
  __syncthreads();
  tc_fence_after_sync();
  const uint32_t tmem = *tmem_slot;

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&tm_a_hi); tma_prefetch_desc(&tm_b_hi);
    int s = 0; uint32_t ph = 0;
    for (int kb = 0; kb < a.nkb; ++kb) {
      mbar_wait(&empty[s], ph ^ 1u);
      uint8_t* st = smem + s * Cfg::STAGE;
      mbar_arrive_expect_tx(&full[s], Cfg::STAGE);
      tma_load_2d(st, &tm_a_hi, &full[s], kb * 64, m0);
      tma_load_2d(st + TILE_A, &tm_b_hi, &full[s], kb * 64, a.w_row0 + p * 256);
      if (NPASS != 1) {
        tma_load_2d(st + 3 * TILE_A, &tm_a_lo, &full[s], kb * 64, m0);
        tma_load_2d(st + 4 * TILE_A, &tm_b_lo, &full[s], kb * 64, a.w_row0 + p * 256);
      }
      ring_advance(s, ph, Cfg::NST);
    }
  } else if (warp == 1 && lane == 0) {
    int s = 0; uint32_t ph = 0;
    for (int kb = 0; kb < a.nkb; ++kb) {
      mbar_wait(&full[s], ph);
      tc_fence_after_sync();
      uint32_t st = smem_u32(smem + s * Cfg::STAGE);
      issue_kblock(st, st + TILE_A, tmem, ID256, kb == 0);
      if (NPASS != 1) {
        issue_kblock(st + 3 * TILE_A, st + TILE_A, tmem, ID256, false);   // lo * hi
        issue_kblock(st, st + 4 * TILE_A, tmem, ID256, false);            // hi * lo
      }
      umma_commit(&empty[s]);
      ring_advance(s, ph, Cfg::NST);
    }
    umma_commit(acc_full);
  } else if (warp >= 2) {
    // 8 epilogue warps: TMEM lane quarter = warp % 4 (one row per lane), column group cg = (warp - 2) / 4 takes 4 of the 8
    // 16-column chunks of each 128-column half
    const int quarter = warp & 3, cg = (warp - 2) >> 2, row = quarter * 32 + lane;
    const uint32_t trow = tmem + ((uint32_t)(quarter * 32) << 16);
    int m = m0 + row;
    int b = min(m / a.Tm, a.B - 1);
    const float4* bias4 = reinterpret_cast<const float4*>(a.bias + (size_t)b * a.bias_bstride);
    mbar_wait(acc_full, 0);
    tc_fence_after_sync();
    // staging aliases the (now idle) pipeline stage, 128 columns at a time: hi boxes at 0..32 KB, lo boxes at 32..64 KB
#pragma unroll 1
    for (int half = 0; half < 2; ++half) {
#pragma unroll 1
      for (int c = 8 * half + 4 * cg; c < 8 * half + 4 * cg + 4; ++c) {
        float v[16];
        tmem_ld16_sync(trow + c * 16, v);
#pragma unroll
        for (int q = 0; q < 4; ++q) {
          float4 bb = __ldg(bias4 + c * 4 + q);
          v[4 * q] += bb.x; v[4 * q + 1] += bb.y; v[4 * q + 2] += bb.z; v[4 * q + 3] += bb.w;
        }
        if (F8 && a.range_flag) {
          float mx = 0.f;
#pragma unroll
          for (int q = 0; q < 16; ++q) mx = fmaxf(mx, fabsf(v[q]));
          if (!(mx < 65504.f)) atomicOr(a.range_flag, 2);
        }
        uint8_t* thi = smem + ((c >> 2) & 1) * TILE_A;
        if (F8) store_split16_f8(v, thi, nullptr, smem + 2 * TILE_A, smem + 3 * TILE_A, row, (c & 3) * 2, c & 7);
        else store_split16<NPASS == 3>(v, thi, thi + 2 * TILE_A, row, (c & 3) * 2);
      }
      tc_fence_before_sync();
      fence_proxy_async_smem();
      asm volatile("bar.sync 1, 256;" ::: "memory");
      if (warp == 2 && lane == 0) {
        for (int j = 0; j < 2; ++j) {
          tma_store_2d(&tm_c_hi, smem + j * TILE_A, p * 256 + (2 * half + j) * 64, m0);
          if (NPASS == 3) tma_store_2d(&tm_c_lo, smem + (2 + j) * TILE_A, p * 256 + (2 * half + j) * 64, m0);
        }
        if (F8) {                                   // one [128 rows x 128 B] e5m2 tile per plane and half
          tma_store_2d(&tm_c_lo, smem + 2 * TILE_A, p * 256 + half * 128, m0);
          tma_store_2d(&tm_c_h8, smem + 3 * TILE_A, p * 256 + half * 128, m0);
        }
        tma_store_commit();
        tma_store_wait_read();                 // the second half reuses the staging tiles
      }
      asm volatile("bar.sync 1, 256;" ::: "memory");
    }
    if (warp == 2 && lane == 0) tma_store_wait_all();
  }
  __syncthreads();
  if (warp == 1) { __syncwarp(); tmem_dealloc(tmem, 256); }
}

}  // namespace

int launch_cond_tc(const Dims& d, const cwg_weights* w, int npass, int flow, const float* mel,
                   const float* cond_bias, __nv_bfloat16* h2_planes, __nv_bfloat16* mel4_planes,
                   cudaStream_t s, const int* mel_len) {
  const size_t n4 = (size_t)d.B * d.Tm * d.KCp;
  __nv_bfloat16* m4_hi = mel4_planes; __nv_bfloat16* m4_lo = mel4_planes + n4;
  if (mel != nullptr) {
    k_im2col_mel<<<(unsigned)((n4 + 255) / 256), 256, 0, s>>>(mel, m4_hi, m4_lo, d.B, d.M, d.Tm, d.J, d.KCp, npass == 2);
    CWG_CHECK_CUDA(cudaGetLastError());
    if (mel_len)      // row f of utterance b reads frames <= f only (causal upsampler): rows f < len[b] are unaffected
      if (int r = launch_ragged_rows(m4_hi, nullptr, n4 * 2, 2, d.B, d.Tm, d.KCp / 2, mel_len, 1, s)) return r;
  }
  const uint64_t rows = (uint64_t)d.B * d.Tm, ncol = (uint64_t)d.P * d.H;
  CUtensorMap ta_hi, ta_lo, tb_hi, tb_lo, tc_hi, tc_lo;
  if (int r = map_2d(&ta_hi, m4_hi, d.KCp, rows, 128)) return r;
  if (int r = map_2d(&ta_lo, m4_lo, d.KCp, rows, 128)) return r;
  if (int r = map_2d(&tb_hi, w->cond_w_hi, d.KCp, (uint64_t)d.F * ncol, 256)) return r;
  if (int r = map_2d(&tb_lo, w->cond_w_lo, d.KCp, (uint64_t)d.F * ncol, 256)) return r;
  if (int r = map_2d(&tc_hi, h2_planes, ncol, rows, 128)) return r;
  CUtensorMap tc_h8 = tc_hi;
  if (npass == 2) {       // H2 = [fp16 hi][e5m2 lo*2^P][e5m2 hi*2^-Q]
    uint8_t* h8 = reinterpret_cast<uint8_t*>(h2_planes) + 2 * (size_t)d.BT * d.H;
    if (int r = map_2d8(&tc_lo, h8, ncol, rows, 128)) return r;
    if (int r = map_2d8(&tc_h8, h8 + (size_t)d.BT * d.H, ncol, rows, 128)) return r;
  } else {
    if (int r = map_2d(&tc_lo, h2_planes + (size_t)d.BT * d.H, ncol, rows, 128)) return r;
  }
  CondArgs a{};
  a.bias = cond_bias + (size_t)flow * d.H; a.bias_bstride = d.F * d.H;
  a.M = (int)rows; a.Tm = d.Tm; a.B = d.B; a.w_row0 = flow * (int)ncol; a.nkb = d.KCp / 64;
  a.range_flag = npass == 2 ? range_flag() : nullptr;
  dim3 grid(d.P, (unsigned)((rows + 127) / 128));
  if (npass == 3) {
    if (int r = set_smem(k_cond_tc<3>, CondCfg<3>::SMEM)) return r;
    k_cond_tc<3><<<grid, 320, CondCfg<3>::SMEM, s>>>(ta_hi, ta_lo, tb_hi, tb_lo, tc_hi, tc_lo, tc_h8, a);
  } else if (npass == 2) {
    if (int r = set_smem(k_cond_tc<2>, CondCfg<2>::SMEM)) return r;
    k_cond_tc<2><<<grid, 320, CondCfg<2>::SMEM, s>>>(ta_hi, ta_lo, tb_hi, tb_lo, tc_hi, tc_lo, tc_h8, a);
  } else {
    if (int r = set_smem(k_cond_tc<1>, CondCfg<1>::SMEM)) return r;
    k_cond_tc<1><<<grid, 320, CondCfg<1>::SMEM, s>>>(ta_hi, ta_lo, tb_hi, tb_lo, tc_hi, tc_lo, tc_h8, a);
  }
  CWG_CHECK_CUDA(cudaGetLastError());
  return 0;
}

}  // namespace cwg
