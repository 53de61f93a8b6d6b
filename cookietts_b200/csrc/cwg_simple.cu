// CUDA-core (fp32 FFMA) kernels of the WaveGlow inverse pass, plus the flow-boundary kernel
// that both arithmetic modes share.  This path keeps exact fp32 semantics (CWG_MODE_FFMA) and
// doubles as the on-device cross-check for the tcgen05 path (cwg_tc.cu, cwg_ps.cu, cwg_tc512.cu).
//
// Reference lines implemented (CookieTTS/_4_mtw/waveglow/glow.py):
//   cond GEMM        : upsample + squeeze + cond_layers[0..1]  :318-324, :198-199 (folded, see packing.py)
//   layer GEMM1+gate : in_layers[i] + cond_layers[2] slice + fused_add_tanh_sigmoid_multiply :201-209, :34-41
//   layer GEMM2      : res_skip_layers[i], residual/skip update, `end` (folded) :211-222
//   flow boundary    : affine coupling inverse, W^-1, early-z concat, start conv :329-347, :189
#include "cwg_common.cuh"
#include "cwg_sm100.cuh"
#include <cuda_fp16.h>

namespace cwg {

namespace {

constexpr int BM = 64, BN = 64, BK = 16, TM = 4, TN = 4;

struct GemmP {
  int M, N, K;
  const float* W; int ldw;          // [N][ldw]
  const float* a0; const float* a1; // A sources
  int Tm, Tp, nmel, C, ks, dil, H;
  float* o0; float* o1;
  const float* bias; const float* bias2; const float* xin;
  long long bias_bstride;           // cond / gate: batch stride of a per-utterance bias (0: shared)
  int has_res, first, eo_pad;       // eo_pad: row pitch MG of the folded-`end` accumulator
};

// A(m, kk) for the three GEMMs.
template <int AMODE>
__device__ __forceinline__ float load_a(const GemmP& p, int m, int kk) {
  if (m >= p.M || kk >= p.K) return 0.f;
  if (AMODE == 0) {             // mel4[b, f, j*nmel + ci] = mel[b, ci, f - j]
    int b = m / p.Tm, f = m - b * p.Tm;
    int j = kk / p.nmel, ci = kk - j * p.nmel;
    int ff = f - j;
    return ff >= 0 ? __ldg(p.a0 + ((size_t)b * p.nmel + ci) * p.Tm + ff) : 0.f;
  } else if (AMODE == 1) {      // [x taps | h2]
    int kx = p.ks * p.C;
    if (kk < kx) {
      int b = m / p.Tp, t = m - b * p.Tp;
      int tap = kk / p.C, c = kk - tap * p.C;
      int tt = t + (tap - p.ks / 2) * p.dil;
      return (tt >= 0 && tt < p.Tp) ? __ldg(p.a0 + ((size_t)b * p.Tp + tt) * p.C + c) : 0.f;
    }
    return __ldg(p.a1 + (size_t)m * p.H + (kk - kx));
  } else {
    return __ldg(p.a0 + (size_t)m * p.K + kk);
  }
}

template <int EMODE>
__device__ __forceinline__ void store_c(const GemmP& p, int m, int n, float acc) {
  if (m >= p.M || n >= p.N) return;
  if (EMODE == 0) {             // H2[m][n] (+ per-utterance cond bias of channel n % H)
    int b = m / p.Tm;
    p.o0[(size_t)m * p.N + n] = acc + __ldg(p.bias + (size_t)b * p.bias_bstride + (n % p.H));
  } else if (EMODE == 1) {      // pre-activation (+ the per-utterance gate bias of the ax WN-level speaker embedding)
    p.o0[(size_t)m * p.N + n] = acc + __ldg(p.bias + (size_t)(m / p.Tp) * p.bias_bstride + n);
  } else {                      // res / folded end
    if (n < p.C) {
      if (p.has_res) p.o0[(size_t)m * p.C + n] = __ldg(p.xin + (size_t)m * p.C + n) + acc + __ldg(p.bias + n);
    } else {
      int j = n - p.C;
      float* e = p.o1 + (size_t)m * p.eo_pad + j;
      *e = (p.first ? __ldg(p.bias2 + j) : *e) + acc;
    }
  }
}

template <int AMODE, int EMODE>
__global__ void __launch_bounds__(256) k_sgemm(GemmP p) {
  __shared__ float As[BK][BM + 4];
  __shared__ float Bs[BK][BN + 4];
  const int tid = threadIdx.x, tx = tid % 16, ty = tid / 16;
  const int m0 = blockIdx.x * BM, n0 = blockIdx.y * BN;
  float acc[TM][TN] = {};
  for (int k0 = 0; k0 < p.K; k0 += BK) {
#pragma unroll
    for (int r = 0; r < (BM * BK) / 256; ++r) {
      int idx = tid + r * 256;
      int row, kk;
      if (AMODE == 0) { kk = idx / BM; row = idx % BM; } else { row = idx / BK; kk = idx % BK; }
      As[kk][row] = load_a<AMODE>(p, m0 + row, k0 + kk);
    }
#pragma unroll
    for (int r = 0; r < (BN * BK) / 256; ++r) {
      int idx = tid + r * 256;
      int n = idx / BK, kk = idx % BK;
      Bs[kk][n] = (n0 + n < p.N && k0 + kk < p.K) ? __ldg(p.W + (size_t)(n0 + n) * p.ldw + k0 + kk) : 0.f;
    }
    __syncthreads();
#pragma unroll
    for (int kk = 0; kk < BK; ++kk) {
      float a[TM], b[TN];
#pragma unroll
      for (int i = 0; i < TM; ++i) a[i] = As[kk][ty * TM + i];
#pragma unroll
      for (int j = 0; j < TN; ++j) b[j] = Bs[kk][tx * TN + j];
#pragma unroll
      for (int i = 0; i < TM; ++i)
#pragma unroll
        for (int j = 0; j < TN; ++j) acc[i][j] = fmaf(a[i], b[j], acc[i][j]);
    }
    __syncthreads();
  }
#pragma unroll
  for (int i = 0; i < TM; ++i)
#pragma unroll
    for (int j = 0; j < TN; ++j) store_c<EMODE>(p, m0 + ty * TM + i, n0 + tx * TN + j, acc[i][j]);
}

// acts[m][c] = tanh(pre[m][c]) * sigmoid(pre[m][C + c])   (glow.py:34-41)
__global__ void k_gate(const float* __restrict__ pre, float* __restrict__ acts, long long n, int C) {
  long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  long long m = i / C; int c = (int)(i - m * C);
  float a = pre[m * 2 * C + c], b = pre[m * 2 * C + C + c];
  acts[i] = tanhf(a) * (1.f / (1.f + expf(-b)));
}

constexpr int TB = 32;   // group-steps per block in the boundary kernel

struct BoundaryP {
  long long BT; int G, C;
  int init, do_flow, do_mix, do_start, ignore_nan;
  int n_rem, n_half;          // of flow_done (coupling)
  int n_rem_mix;              // channels of the inverse 1x1 conv applied after the coupling
  int n_rem2, n_half2;        // of flow_next
  const float* z; float sigma;
  float* audio; const float* eo;
  const float* winv;          // [MG][MG] of the mixing flow
  int* range_flag;            // CWG_MODE_F16F8: |= 2 when a start-conv output leaves the fp16 range (may be NULL)
  const float* start_w;       // [C][MG/2] of flow_next
  const float* start_b;       // [C]
  void* x_out;
  void* a0_out;               // layer-0 fold: planes hi, lo [BT][16] 16-bit of (audio_0 | 1 | 0...) instead of x (tensor-core modes)
};

// One block handles TB consecutive group-steps (rows of the [B*T'][G] audio state, which IS
// the [B, T] output buffer: latent channel c of step s lives at audio[b, s*G + c], so the
// early-z concat (glow.py:342-347) and the final un-squeeze (:349) are no-ops by layout).
// MG = CWG_GROUP_PAD(n_group): 16, or 32 for the wide layout (16 < n_group <= 32)
template <int XFMT, int MG>
__global__ void __launch_bounds__(256) k_flow_boundary(BoundaryP p) {
  __shared__ float a_s[TB][MG];
  const long long m0 = (long long)blockIdx.x * TB;
  const int tid = threadIdx.x;
  if (tid < TB) {
    long long m = m0 + tid;
    if (m < p.BT) {
      float a[MG];
      for (int g = 0; g < p.G; ++g)
        a[g] = p.init ? p.sigma * p.z[m * p.G + g] : p.audio[m * p.G + g];
      if (p.do_flow) {
        const int off = p.G - p.n_rem;
        const float* e = p.eo + m * MG;
        for (int j = 0; j < p.n_rem - p.n_half; ++j) {
          // audio_1 = (audio_1 - b) / exp(s), glow.py:337
          float b = e[j], s = e[p.n_half + j];
          a[off + p.n_half + j] = (a[off + p.n_half + j] - b) * expf(-s);
        }
        if (p.ignore_nan)                              // efficient_model_ax.py:12-15,331-332 (NaN -> 0 after the coupling)
          for (int c = 0; c < p.n_rem; ++c) if (isnan(a[off + c])) a[off + c] = 0.f;
      }
      if (p.do_mix) {                                 // z = conv1d(z, W^-1), glow.py:98
        const int off = p.G - p.n_rem_mix;
        float v[MG];
        for (int c = 0; c < p.n_rem_mix; ++c) v[c] = a[off + c];
        for (int r = 0; r < p.n_rem_mix; ++r) {
          float acc = 0.f;
          for (int c = 0; c < p.n_rem_mix; ++c) acc = fmaf(__ldg(p.winv + r * MG + c), v[c], acc);
          a[off + r] = acc;
        }
      }
      if (p.init || p.do_flow || p.do_mix)
        for (int g = 0; g < p.G; ++g) p.audio[m * p.G + g] = a[g];
      for (int g = 0; g < p.G; ++g) a_s[tid][g] = a[g];
    }
  }
  if (!p.do_start) return;
  __syncthreads();
  const int off2 = p.G - p.n_rem2;
  const int nrow = (int)min((long long)TB, p.BT - m0);
  // audio = start(audio_0), glow.py:189.  Thread -> channel pair (4-byte bf16x2 / 8-byte fp32 stores,
  // 128 B per warp store); the two halves of the block take alternate rows.
  const int npair = p.C >> 1, rpar = tid >> 7;
  for (int cp = tid & 127; cp < npair; cp += 128) {
    const int c = 2 * cp;
    float w0[MG / 2], w1[MG / 2];
    for (int j = 0; j < p.n_half2; ++j) {
      w0[j] = __ldg(p.start_w + c * (MG / 2) + j);
      w1[j] = __ldg(p.start_w + (c + 1) * (MG / 2) + j);
    }
    const float bias0 = __ldg(p.start_b + c), bias1 = __ldg(p.start_b + c + 1);
    for (int r = rpar; r < nrow; r += 2) {
      float x0 = bias0, x1 = bias1;
      for (int j = 0; j < p.n_half2; ++j) {
        const float av = a_s[r][off2 + j];
        x0 = fmaf(w0[j], av, x0); x1 = fmaf(w1[j], av, x1);
      }
      const size_t idx = (size_t)(m0 + r) * p.C + c;
      if (XFMT == 0) {
        *reinterpret_cast<float2*>(reinterpret_cast<float*>(p.x_out) + idx) = make_float2(x0, x1);
      } else {
        __nv_bfloat16* hi = reinterpret_cast<__nv_bfloat16*>(p.x_out);
        __nv_bfloat16* lo = hi + (size_t)p.BT * p.C;
        const __nv_bfloat162 h = __floats2bfloat162_rn(x0, x1);
        *reinterpret_cast<__nv_bfloat162*>(hi + idx) = h;
        *reinterpret_cast<__nv_bfloat162*>(lo + idx) = __floats2bfloat162_rn(x0 - __low2float(h), x1 - __high2float(h));
      }
    }
  }
}

// Same work for C % 8 == 0, laid out for 128-bit HBM access: one block = TBV group-steps.  Phase 1: thread ->
// group-step (coupling, NaN flush, W^-1; the audio row is read and written as float4).  Phase 2: warp -> group-step,
// lane -> 8 consecutive channels of the start conv, so every warp store is one contiguous 512-byte (bf16 hi, then lo)
// or 1-KB (fp32) run of the channels-last activation row; the lane's 8 x n_half weights stay in registers.
constexpr int TBV = 256;

template <int XFMT, int MG>
__global__ void __launch_bounds__(TBV) k_flow_boundary_v(BoundaryP p) {
  __shared__ __align__(16) float a_s[TBV][MG / 2];      // the n_half2 inputs of the next start conv
  const long long m0 = (long long)blockIdx.x * TBV;
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  {
    const long long m = m0 + tid;
    if (m < p.BT) {
      float a[MG];
      const float* src = p.init ? p.z + m * p.G : p.audio + m * p.G;
      if ((p.G & 3) == 0) {
        for (int g = 0; g < p.G; g += 4) {
          const float4 v = *reinterpret_cast<const float4*>(src + g);
          a[g] = v.x; a[g + 1] = v.y; a[g + 2] = v.z; a[g + 3] = v.w;
        }
      } else {
        for (int g = 0; g < p.G; ++g) a[g] = src[g];
      }
      if (p.init) for (int g = 0; g < p.G; ++g) a[g] *= p.sigma;
      if (p.do_flow) {
        const int off = p.G - p.n_rem;
        float e[MG];
        const float4* ev = reinterpret_cast<const float4*>(p.eo + m * MG);
#pragma unroll
        for (int q = 0; q < MG / 4; ++q) { const float4 v = __ldcs(ev + q); e[4 * q] = v.x; e[4 * q + 1] = v.y; e[4 * q + 2] = v.z; e[4 * q + 3] = v.w; }
        for (int j = 0; j < p.n_rem - p.n_half; ++j)                 // audio_1 = (audio_1 - b) / exp(s), glow.py:337
          a[off + p.n_half + j] = (a[off + p.n_half + j] - e[j]) * expf(-e[p.n_half + j]);
        if (p.ignore_nan)
          for (int c = 0; c < p.n_rem; ++c) if (isnan(a[off + c])) a[off + c] = 0.f;
      }
      if (p.do_mix) {                                                // z = conv1d(z, W^-1), glow.py:98
        const int off = p.G - p.n_rem_mix;
        float v[MG];
        for (int c = 0; c < p.n_rem_mix; ++c) v[c] = a[off + c];
        for (int r = 0; r < p.n_rem_mix; ++r) {
          float acc = 0.f;
          for (int c = 0; c < p.n_rem_mix; ++c) acc = fmaf(__ldg(p.winv + r * MG + c), v[c], acc);
          a[off + r] = acc;
        }
      }
      if (p.init || p.do_flow || p.do_mix) {
        float* dst = p.audio + m * p.G;
        if ((p.G & 3) == 0) for (int g = 0; g < p.G; g += 4) *reinterpret_cast<float4*>(dst + g) = make_float4(a[g], a[g + 1], a[g + 2], a[g + 3]);
        else for (int g = 0; g < p.G; ++g) dst[g] = a[g];
      }
      if (p.do_start && p.a0_out) {
        // layer-0 fold: the next flow's first layer contracts (audio_0, 1) with in_layers.0 * start itself; the constant-1
        // channel carries the start bias and vanishes, like the conv's zero padding, where TMA zero-fills out-of-range steps
        const int off2 = p.G - p.n_rem2;
        float v[16];
#pragma unroll
        for (int j = 0; j < 16; ++j) v[j] = j < p.n_half2 ? a[off2 + j < MG ? off2 + j : 0] : (j == p.n_half2 ? 1.f : 0.f);
        uint32_t hi[8], lo[8];
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          float h0, h1;
          hi[j] = sm100::pack2<XFMT == 2>(v[2 * j], v[2 * j + 1]);
          sm100::unpack2<XFMT == 2>(hi[j], h0, h1);
          lo[j] = sm100::pack2<XFMT == 2>(v[2 * j] - h0, v[2 * j + 1] - h1);
        }
        uint4* oh = reinterpret_cast<uint4*>(reinterpret_cast<uint16_t*>(p.a0_out) + (size_t)m * 16);
        uint4* ol = reinterpret_cast<uint4*>(reinterpret_cast<uint16_t*>(p.a0_out) + ((size_t)p.BT + m) * 16);
        oh[0] = make_uint4(hi[0], hi[1], hi[2], hi[3]); oh[1] = make_uint4(hi[4], hi[5], hi[6], hi[7]);
        ol[0] = make_uint4(lo[0], lo[1], lo[2], lo[3]); ol[1] = make_uint4(lo[4], lo[5], lo[6], lo[7]);
      } else if (p.do_start) {
        const int off2 = p.G - p.n_rem2;
        for (int j = 0; j < MG / 2; ++j) a_s[tid][j] = j < p.n_half2 ? a[off2 + j] : 0.f;
      }
    }
  }
  if (!p.do_start || p.a0_out) return;
  __syncthreads();
  const int nrow = (int)min((long long)TBV, p.BT - m0);
  if (MG != 16) {
    // wide layout (n_half2 <= 16): lane -> 4 consecutive channels, so that the 4 x 16 weights still fit in registers
    for (int cg = lane; cg < (p.C >> 2); cg += 32) {
      const int c = cg * 4;
      float w[4][MG / 2], bias[4];
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        bias[i] = __ldg(p.start_b + c + i);
#pragma unroll
        for (int j = 0; j < MG / 2; ++j) w[i][j] = j < p.n_half2 ? __ldg(p.start_w + (c + i) * (MG / 2) + j) : 0.f;
      }
      for (int r = warp; r < nrow; r += TBV / 32) {
        float x[4] = {bias[0], bias[1], bias[2], bias[3]};
#pragma unroll
        for (int jq = 0; jq < MG / 8; ++jq) {
          const float4 a4 = *reinterpret_cast<const float4*>(&a_s[r][4 * jq]);
          const float av[4] = {a4.x, a4.y, a4.z, a4.w};
#pragma unroll
          for (int i = 0; i < 4; ++i)
#pragma unroll
            for (int j = 0; j < 4; ++j) x[i] = fmaf(w[i][4 * jq + j], av[j], x[i]);
        }
        const size_t idx = (size_t)(m0 + r) * p.C + c;
        if (XFMT == 0) {
          *reinterpret_cast<float4*>(reinterpret_cast<float*>(p.x_out) + idx) = make_float4(x[0], x[1], x[2], x[3]);
        } else {
          constexpr bool F16 = XFMT == 2;
          const size_t plane = (size_t)p.BT * p.C;
          uint16_t* hi = reinterpret_cast<uint16_t*>(p.x_out);
          if (F16 && p.range_flag) {
            const float mx = fmaxf(fmaxf(fabsf(x[0]), fabsf(x[1])), fmaxf(fabsf(x[2]), fabsf(x[3])));
            if (!(mx < 65504.f)) atomicOr(p.range_flag, 2);
          }
          uint32_t h[2], l[2];
#pragma unroll
          for (int i = 0; i < 2; ++i) {
            float h0, h1;
            h[i] = sm100::pack2<F16>(x[2 * i], x[2 * i + 1]);
            sm100::unpack2<F16>(h[i], h0, h1);
            l[i] = sm100::pack2<F16>(x[2 * i] - h0, x[2 * i + 1] - h1);
          }
          *reinterpret_cast<uint2*>(hi + idx) = make_uint2(h[0], h[1]);
          *reinterpret_cast<uint2*>(hi + plane + idx) = make_uint2(l[0], l[1]);
          if (F16) {                          // e5m2(lo * 2^P), e5m2(hi * 2^-Q) planes
            uint8_t* p8 = reinterpret_cast<uint8_t*>(p.x_out) + 4 * plane;
            *reinterpret_cast<uint32_t*>(p8 + idx) = sm100::e5m2x4_from_f16x2(l[0], l[1], sm100::F16X2_2P6);
            *reinterpret_cast<uint32_t*>(p8 + plane + idx) = sm100::e5m2x4_from_f16x2(h[0], h[1], sm100::F16X2_2M8);
          }
        }
      }
    }
    return;
  }
  for (int cg = lane; cg < (p.C >> 3); cg += 32) {                   // audio = start(audio_0), glow.py:189
    const int c = cg * 8;
    float w[8][MG / 2], bias[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      bias[i] = __ldg(p.start_b + c + i);
#pragma unroll
      for (int j = 0; j < MG / 2; ++j) w[i][j] = j < p.n_half2 ? __ldg(p.start_w + (c + i) * (MG / 2) + j) : 0.f;
    }
    for (int r = warp; r < nrow; r += TBV / 32) {
      const float4 a0 = *reinterpret_cast<const float4*>(&a_s[r][0]), a1 = *reinterpret_cast<const float4*>(&a_s[r][4]);
      const float av[8] = {a0.x, a0.y, a0.z, a0.w, a1.x, a1.y, a1.z, a1.w};
      float x[8];
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        float acc = bias[i];
#pragma unroll
        for (int j = 0; j < MG / 2; ++j) acc = fmaf(w[i][j], av[j], acc);
        x[i] = acc;
      }
      const size_t idx = (size_t)(m0 + r) * p.C + c;
      if (XFMT == 0) {
        float4* o = reinterpret_cast<float4*>(reinterpret_cast<float*>(p.x_out) + idx);
        o[0] = make_float4(x[0], x[1], x[2], x[3]); o[1] = make_float4(x[4], x[5], x[6], x[7]);
      } else if (XFMT == 2) {                  // CWG_MODE_F16F8: fp16 hi, fp16 lo, e5m2(lo * 2^P), e5m2(hi * 2^-Q)
        const size_t plane = (size_t)p.BT * p.C;
        __half* hi = reinterpret_cast<__half*>(p.x_out);
        uint8_t* p8 = reinterpret_cast<uint8_t*>(p.x_out) + 4 * plane;
        uint32_t h[4], l[4];
        float hf[8], df[8];
        if (p.range_flag) {
          float mx = 0.f;
#pragma unroll
          for (int i = 0; i < 8; ++i) mx = fmaxf(mx, fabsf(x[i]));
          if (!(mx < 65504.f)) atomicOr(p.range_flag, 2);
        }
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          const __half2 hh = __floats2half2_rn(x[2 * i], x[2 * i + 1]);
          hf[2 * i] = __low2float(hh); hf[2 * i + 1] = __high2float(hh);
          df[2 * i] = x[2 * i] - hf[2 * i]; df[2 * i + 1] = x[2 * i + 1] - hf[2 * i + 1];
          const __half2 ll = __floats2half2_rn(df[2 * i], df[2 * i + 1]);
          h[i] = *reinterpret_cast<const uint32_t*>(&hh); l[i] = *reinterpret_cast<const uint32_t*>(&ll);
        }
        *reinterpret_cast<uint4*>(hi + idx) = make_uint4(h[0], h[1], h[2], h[3]);
        *reinterpret_cast<uint4*>(hi + plane + idx) = make_uint4(l[0], l[1], l[2], l[3]);
        uint32_t l8[2], h8[2];
#pragma unroll
        for (int i = 0; i < 2; ++i) {
          l8[i] = sm100::e5m2x4_from_f16x2(l[2 * i], l[2 * i + 1], sm100::F16X2_2P6);
          h8[i] = sm100::e5m2x4_from_f16x2(h[2 * i], h[2 * i + 1], sm100::F16X2_2M8);
        }
        *reinterpret_cast<uint2*>(p8 + idx) = make_uint2(l8[0], l8[1]);
        *reinterpret_cast<uint2*>(p8 + plane + idx) = make_uint2(h8[0], h8[1]);
      } else {
        __nv_bfloat16* hi = reinterpret_cast<__nv_bfloat16*>(p.x_out);
        __nv_bfloat16* lo = hi + (size_t)p.BT * p.C;
        uint32_t h[4], l[4];
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          const __nv_bfloat162 hh = __floats2bfloat162_rn(x[2 * i], x[2 * i + 1]);
          const __nv_bfloat162 ll = __floats2bfloat162_rn(x[2 * i] - __low2float(hh), x[2 * i + 1] - __high2float(hh));
          h[i] = *reinterpret_cast<const uint32_t*>(&hh); l[i] = *reinterpret_cast<const uint32_t*>(&ll);
        }
        *reinterpret_cast<uint4*>(hi + idx) = make_uint4(h[0], h[1], h[2], h[3]);
        *reinterpret_cast<uint4*>(lo + idx) = make_uint4(l[0], l[1], l[2], l[3]);
      }
    }
  }
}

// mel [B][M][frames] -> cond [B][T'][H] (channels >= M are zero): zero-extended by pad frames and
// interpolated to T' steps like F.interpolate(mode='linear', align_corners=True) / 'nearest'
// (efficient_model_ax.py:171-182).  XFMT 0: fp32; 1: bf16 hi plane then lo plane.
template <int XFMT>
__global__ void k_mel_up(const float* __restrict__ mel, void* __restrict__ out, int B, int M, int frames,
                         int frames_padded, int Tp, int H, int linear, int* range_flag) {
  long long n = (long long)B * Tp * H;
  long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  int c = (int)(i % H);
  long long m = i / H;
  int t = (int)(m % Tp), b = (int)(m / Tp);
  float v = 0.f;
  if (c < M) {
    const float* row = mel + ((size_t)b * M + c) * frames;
    if (linear) {
      double src = Tp > 1 ? (double)t * (double)(frames_padded - 1) / (double)(Tp - 1) : 0.0;
      int i0 = min((int)floor(src), frames_padded - 1);
      int i1 = min(i0 + 1, frames_padded - 1);
      float w = (float)(src - (double)i0);
      float v0 = i0 < frames ? row[i0] : 0.f, v1 = i1 < frames ? row[i1] : 0.f;
      v = v0 * (1.f - w) + v1 * w;
    } else {
      int i0 = min((int)floor((double)t * ((double)frames_padded / (double)Tp)), frames_padded - 1);
      v = i0 < frames ? row[i0] : 0.f;
    }
  }
  if (XFMT == 0) {
    reinterpret_cast<float*>(out)[i] = v;
  } else if (XFMT == 2) {                     // CWG_MODE_F16F8 cond planes: fp16 hi, e5m2(lo * 2^P), e5m2(hi * 2^-Q)
    const __half h = __float2half_rn(v);
    const float hf = __half2float(h);
    if (range_flag && !(fabsf(v) < 65504.f)) atomicOr(range_flag, 2);
    reinterpret_cast<__half*>(out)[i] = h;
    uint8_t* p8 = reinterpret_cast<uint8_t*>(out) + 2 * n;
    p8[i] = (uint8_t)(sm100::pack_e5m2x4((v - hf) * F8_LO_SCALE, 0.f, 0.f, 0.f) & 0xffu);
    p8[n + i] = (uint8_t)(sm100::pack_e5m2x4(hf * F8_HI_SCALE, 0.f, 0.f, 0.f) & 0xffu);
  } else {
    __nv_bfloat16* hi = reinterpret_cast<__nv_bfloat16*>(out);
    __nv_bfloat16 h = __float2bfloat16_rn(v);
    hi[i] = h;
    hi[n + i] = __float2bfloat16_rn(v - __bfloat162float(h));
  }
}

}  // namespace

int launch_mel_up(int xfmt, const float* mel, void* out, int B, int M, int frames, int frames_padded, int Tp, int H,
                  int linear, cudaStream_t s) {
  long long n = (long long)B * Tp * H;
  unsigned grid = (unsigned)((n + 255) / 256);
  if (xfmt == 2) k_mel_up<2><<<grid, 256, 0, s>>>(mel, out, B, M, frames, frames_padded, Tp, H, linear, range_flag());
  else if (xfmt == 0) k_mel_up<0><<<grid, 256, 0, s>>>(mel, out, B, M, frames, frames_padded, Tp, H, linear, nullptr);
  else           k_mel_up<1><<<grid, 256, 0, s>>>(mel, out, B, M, frames, frames_padded, Tp, H, linear, nullptr);
  CWG_CHECK_CUDA(cudaGetLastError());
  return 0;
}

int launch_cond_ffma(const Dims& d, const cwg_weights* w, int flow, const float* mel,
                     const float* cond_bias, float* h2, cudaStream_t s) {
  GemmP p{};
  p.M = d.B * d.Tm; p.N = d.P * d.H; p.K = d.KC;
  p.W = w->cond_w_f32 + (size_t)flow * p.N * d.KCp; p.ldw = d.KCp;
  p.a0 = mel; p.Tm = d.Tm; p.nmel = d.M; p.H = d.H;
  p.o0 = h2; p.bias = cond_bias + (size_t)flow * d.H; p.bias_bstride = (long long)d.F * d.H;
  dim3 grid((p.M + BM - 1) / BM, (p.N + BN - 1) / BN);
  k_sgemm<0, 0><<<grid, 256, 0, s>>>(p);
  CWG_CHECK_CUDA(cudaGetLastError());
  return 0;
}

int launch_layer_ffma(const Dims& d, const cwg_weights* w, int flow, int layer, const float* x_in,
                      float* x_out, const float* h2, float* eo, float* pre, float* acts, cudaStream_t s) {
  const size_t fl = (size_t)flow * d.L + layer;
  GemmP p{};
  p.M = (int)d.BT; p.N = 2 * d.C; p.K = d.K1;
  p.W = w->w1_f32 + fl * (size_t)(2 * d.C) * d.K1; p.ldw = d.K1;
  p.a0 = x_in; p.a1 = h2; p.Tp = d.Tp; p.C = d.C; p.ks = d.ks; p.dil = 1 << layer; p.H = d.H;
  p.o0 = pre; p.bias = w->b1 + fl * (size_t)(2 * d.C);
  if (d.b1_batch) { p.bias = d.b1_batch + fl * (size_t)(2 * d.C); p.bias_bstride = (long long)d.F * d.L * 2 * d.C; }
  dim3 g1((p.M + BM - 1) / BM, (p.N + BN - 1) / BN);
  k_sgemm<1, 1><<<g1, 256, 0, s>>>(p);
  CWG_CHECK_CUDA(cudaGetLastError());

  long long n = d.BT * d.C;
  k_gate<<<(unsigned)((n + 255) / 256), 256, 0, s>>>(pre, acts, n, d.C);
  CWG_CHECK_CUDA(cudaGetLastError());

  GemmP q{};
  q.M = (int)d.BT; q.N = d.N2; q.K = d.C;
  q.W = w->w2_f32 + fl * (size_t)d.N2 * d.C; q.ldw = d.C;
  q.a0 = acts; q.C = d.C;
  q.o0 = x_out; q.o1 = eo; q.xin = x_in;
  q.bias = w->b2 + fl * (size_t)d.C; q.bias2 = w->eo_b + (size_t)flow * d.MG; q.eo_pad = d.MG;
  q.has_res = layer < d.L - 1; q.first = layer == 0;
  dim3 g2((q.M + BM - 1) / BM, (q.N + BN - 1) / BN);
  k_sgemm<2, 2><<<g2, 256, 0, s>>>(q);
  CWG_CHECK_CUDA(cudaGetLastError());
  return 0;
}

int launch_flow_boundary(const cwg_config* cfg, const Dims& d, const cwg_weights* w, int xfmt,
                         int flow_done, int flow_next, const float* z, float sigma, float* audio,
                         const float* eo, void* x_out, cudaStream_t s, int mix_flow, int ignore_nan, void* a0_out) {
  // mix_flow: flow whose inverse 1x1 conv follows the coupling; -2 = the classic order (flow_done)
  if (mix_flow == -2) mix_flow = flow_done;
  BoundaryP p{};
  p.BT = d.BT; p.G = d.G; p.C = d.C;
  p.init = z != nullptr; p.do_flow = flow_done >= 0; p.do_start = flow_next >= 0; p.do_mix = mix_flow >= 0;
  p.z = z; p.sigma = sigma; p.audio = audio; p.eo = eo; p.x_out = x_out; p.ignore_nan = ignore_nan;
  p.range_flag = xfmt == 2 ? range_flag() : nullptr;
  p.a0_out = (xfmt != 0 && flow_next >= 0) ? a0_out : nullptr;
  if (p.do_flow) flow_channels(cfg, flow_done, &p.n_rem, &p.n_half);
  if (p.do_mix) {
    int nh;
    flow_channels(cfg, mix_flow, &p.n_rem_mix, &nh);
    p.winv = w->winv + (size_t)mix_flow * d.MG * d.MG;
  }
  if (p.do_start) {
    flow_channels(cfg, flow_next, &p.n_rem2, &p.n_half2);
    p.start_w = w->start_w + (size_t)flow_next * d.C * (d.MG / 2);
    p.start_b = w->start_b + (size_t)flow_next * d.C;
  }
  const bool wide = d.MG != 16;
  CWG_REQUIRE(!wide || p.a0_out == nullptr, "the layer-0 fold takes n_group <= 16");
  if ((d.C & 7) == 0 && ((uintptr_t)x_out & 15) == 0) {
    unsigned grid = (unsigned)((d.BT + TBV - 1) / TBV);
    if (wide) {
      if (xfmt == 0) k_flow_boundary_v<0, 32><<<grid, TBV, 0, s>>>(p);
      else if (xfmt == 2) k_flow_boundary_v<2, 32><<<grid, TBV, 0, s>>>(p);
      else           k_flow_boundary_v<1, 32><<<grid, TBV, 0, s>>>(p);
    } else {
      if (xfmt == 0) k_flow_boundary_v<0, 16><<<grid, TBV, 0, s>>>(p);
      else if (xfmt == 2) k_flow_boundary_v<2, 16><<<grid, TBV, 0, s>>>(p);
      else           k_flow_boundary_v<1, 16><<<grid, TBV, 0, s>>>(p);
    }
  } else {
    CWG_REQUIRE(xfmt != 2, "CWG_MODE_F16F8 needs n_channels % 8 == 0");
    CWG_REQUIRE(p.a0_out == nullptr, "the layer-0 fold needs n_channels % 8 == 0");
    unsigned grid = (unsigned)((d.BT + TB - 1) / TB);
    if (wide) {
      if (xfmt == 0) k_flow_boundary<0, 32><<<grid, 256, 0, s>>>(p);
      else           k_flow_boundary<1, 32><<<grid, 256, 0, s>>>(p);
    } else {
      if (xfmt == 0) k_flow_boundary<0, 16><<<grid, 256, 0, s>>>(p);
      else           k_flow_boundary<1, 16><<<grid, 256, 0, s>>>(p);
    }
  }
  CWG_CHECK_CUDA(cudaGetLastError());
  return 0;
}

// non-finite scan of a result buffer: *flag |= 1 when any element is NaN / Inf (128-bit loads, grid-stride)
__global__ void k_nonfinite(const float* __restrict__ x, size_t n, int* __restrict__ flag) {
  const size_t n4 = n >> 2;
  const float4* x4 = reinterpret_cast<const float4*>(x);
  bool bad = false;
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += (size_t)gridDim.x * blockDim.x) {
    const float4 v = __ldg(x4 + i);
    // |v| < inf is false for NaN and for +-Inf
    bad |= !(fabsf(v.x) < INFINITY) | !(fabsf(v.y) < INFINITY) | !(fabsf(v.z) < INFINITY) | !(fabsf(v.w) < INFINITY);
  }
  if (blockIdx.x == 0 && threadIdx.x < (n & 3)) bad |= !(fabsf(x[(n4 << 2) + threadIdx.x]) < INFINITY);
  if (__any_sync(0xffffffffu, bad) && (threadIdx.x & 31) == 0) atomicOr(flag, 1);
}

int launch_nonfinite(const float* x, size_t n, int* flag, cudaStream_t s, bool clear) {
  CWG_REQUIRE(((uintptr_t)x & 15) == 0, "cwg_nonfinite: buffer must be 16-byte aligned");
  if (clear) CWG_CHECK_CUDA(cudaMemsetAsync(flag, 0, sizeof(int), s));
  if (n == 0) return 0;
  size_t blocks = (n / 4 + 255) / 256;
  if (blocks > 148 * 8) blocks = 148 * 8;
  if (blocks == 0) blocks = 1;
  k_nonfinite<<<(unsigned)blocks, 256, 0, s>>>(x, n, flag);
  CWG_CHECK_CUDA(cudaGetLastError());
  return 0;
}

// ragged calls (cwg_infer_ragged): zero the rows of every utterance past its length, copying the valid rows from src
// when given.  Grid: (RR_BLOCKS, B, planes), grid-stride over one utterance's plane; without src only the padded rows
// are visited, so a batch without padding costs a few thousand empty blocks
constexpr int RR_BLOCKS = 64;

__global__ void k_ragged_rows(uint32_t* __restrict__ dst, const uint32_t* __restrict__ src, size_t plane_words, int T,
                              int row_words, const int* __restrict__ len, int mult) {
  const int b = blockIdx.y;
  const long long n = (long long)T * row_words;
  const long long lim = min((long long)__ldg(len + b) * mult * row_words, n);      // first word of the padding
  const size_t o = blockIdx.z * plane_words + (size_t)b * n;
  for (long long i = (src ? 0 : lim) + (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n;
       i += (long long)gridDim.x * blockDim.x)
    dst[o + i] = i < lim ? src[o + i] : 0u;
}

int launch_ragged_rows(void* dst, const void* src, size_t plane_bytes, int n_planes, int B, int T, int row_words,
                       const int* len, int mult, cudaStream_t s) {
  CWG_REQUIRE(dst && len && plane_bytes % 4 == 0 && ((uintptr_t)dst & 3) == 0, "ragged rows: bad arguments");
  const long long blocks = ((long long)T * row_words + 255) / 256;
  dim3 grid((unsigned)(blocks < RR_BLOCKS ? blocks : RR_BLOCKS), (unsigned)B, (unsigned)n_planes);
  k_ragged_rows<<<grid, 256, 0, s>>>((uint32_t*)dst, (const uint32_t*)src, plane_bytes / 4, T, row_words, len, mult);
  CWG_CHECK_CUDA(cudaGetLastError());
  return 0;
}

}  // namespace cwg
