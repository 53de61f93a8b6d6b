// Flow boundary of WaveGlow's forward direction (audio -> z, glow.py `WaveGlow.forward` in NVIDIA's formulation):
//   flow k   : audio_1 = exp(log_s) * audio_1 + b            (coupling, after WN_k)
//   flow k+1 : audio   = W_{k+1} audio   on the trailing n_rem_{k+1} columns, then start_{k+1}(audio_0) -> x_0
// The ax model with mix_first=False (cwg_ax_forward) mixes after the coupling instead: flow k's W_k follows its own
// coupling in the same launch (k_fwd_boundary_mixlast).
// The WN layers between two boundaries are the kernels `infer` runs (cwg_ps.cu, cwg_tc512.cu, cwg_simple.cu).
// Sums are deterministic: each block writes one fp64 partial per utterance (a fixed shuffle tree), and k_fwd_reduce adds
// the partials in a fixed order.  No float atomics.
#include "cwg_common.cuh"
#include "cwg_sm100.cuh"
#include <cuda_fp16.h>

namespace cwg {

namespace {

constexpr int TBF = 256;   // group-steps per block (one utterance per grid row)

struct FwdP {
  int Tp, G, C, nblk;
  long long BT;
  int vec4;                   // the audio rows may be read / written as float4
  const float* audio_in;      // first launch: the waveform [B*T'][G] (may alias `audio`); NULL afterwards
  float* audio;               // audio state [B*T'][G]: ends as z in the repo's layout z[b, s*G + c]
  int do_flow, n_rem, n_half; // coupling of flow_done
  const float* eo;            // [B*T'][MG]: b = eo[0, n_half), log_s = eo[n_half, 2 n_half)
  float* log_s;               // [B][n_half][T'] of flow_done, or NULL
  double* ls_part;            // [B][nblk]: per-block sum of log_s of flow_done
  double* z2_part;            // [B][nblk]: per-block sum of z^2 (last launch), or NULL
  int do_next, n_rem2, n_half2;   // mixing + start conv of flow_next
  const float* wmix;          // [MG][MG] W of flow_next (not inverted)
  const float* start_w;       // [C][MG/2]
  const float* start_b;       // [C]
  void* x_out;
  void* a0_out;               // layer-0 fold planes hi, lo [BT][16] instead of x (tensor-core modes, MG = 16)
  int* range_flag;            // CWG_MODE_F16F8: |= 2 when a start-conv output leaves the fp16 range (may be NULL)
};

// Sum of v over the block; the result is valid in thread 0.  Fixed reduction order: bit-reproducible.
__device__ __forceinline__ double block_sum(double v, double* red) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_down_sync(0xffffffffu, v, o);
  if (lane == 0) red[warp] = v;
  __syncthreads();
  double s = 0.0;
  if (threadIdx.x == 0)
    for (int w = 0; w < TBF / 32; ++w) s += red[w];
  __syncthreads();
  return s;
}

// x[0..N) of row m -> the activation planes of format XFMT at element idx (N = 4 or 8 consecutive channels)
template <int XFMT, int N>
__device__ __forceinline__ void store_x(const FwdP& p, size_t idx, const float* x) {
  if constexpr (XFMT == 0) {
    float4* o = reinterpret_cast<float4*>(reinterpret_cast<float*>(p.x_out) + idx);
#pragma unroll
    for (int q = 0; q < N / 4; ++q) o[q] = make_float4(x[4 * q], x[4 * q + 1], x[4 * q + 2], x[4 * q + 3]);
    return;
  }
  constexpr bool F16 = XFMT == 2;
  const size_t plane = (size_t)p.BT * p.C;
  uint16_t* hi = reinterpret_cast<uint16_t*>(p.x_out);
  if (F16 && p.range_flag) {
    float mx = 0.f;
#pragma unroll
    for (int i = 0; i < N; ++i) mx = fmaxf(mx, fabsf(x[i]));
    if (!(mx < 65504.f)) atomicOr(p.range_flag, 2);
  }
  uint32_t h[N / 2], l[N / 2];
#pragma unroll
  for (int i = 0; i < N / 2; ++i) {
    float h0, h1;
    h[i] = sm100::pack2<F16>(x[2 * i], x[2 * i + 1]);
    sm100::unpack2<F16>(h[i], h0, h1);
    l[i] = sm100::pack2<F16>(x[2 * i] - h0, x[2 * i + 1] - h1);
  }
  if constexpr (N == 8) {
    *reinterpret_cast<uint4*>(hi + idx) = make_uint4(h[0], h[1], h[2], h[3]);
    *reinterpret_cast<uint4*>(hi + plane + idx) = make_uint4(l[0], l[1], l[2], l[3]);
  } else {
    *reinterpret_cast<uint2*>(hi + idx) = make_uint2(h[0], h[1]);
    *reinterpret_cast<uint2*>(hi + plane + idx) = make_uint2(l[0], l[1]);
  }
  if constexpr (F16) {                        // e5m2(lo * 2^P), e5m2(hi * 2^-Q) planes
    uint8_t* p8 = reinterpret_cast<uint8_t*>(p.x_out) + 4 * plane;
    if constexpr (N == 8) {
      *reinterpret_cast<uint2*>(p8 + idx) = make_uint2(sm100::e5m2x4_from_f16x2(l[0], l[1], sm100::F16X2_2P6),
                                                       sm100::e5m2x4_from_f16x2(l[2], l[3], sm100::F16X2_2P6));
      *reinterpret_cast<uint2*>(p8 + plane + idx) = make_uint2(sm100::e5m2x4_from_f16x2(h[0], h[1], sm100::F16X2_2M8),
                                                               sm100::e5m2x4_from_f16x2(h[2], h[3], sm100::F16X2_2M8));
    } else {
      *reinterpret_cast<uint32_t*>(p8 + idx) = sm100::e5m2x4_from_f16x2(l[0], l[1], sm100::F16X2_2P6);
      *reinterpret_cast<uint32_t*>(p8 + plane + idx) = sm100::e5m2x4_from_f16x2(h[0], h[1], sm100::F16X2_2M8);
    }
  }
}

// One block = TBF group-steps of utterance blockIdx.y.  Phase 1: thread -> group-step (input copy, coupling of flow_done,
// log_s store, mixing, layer-0 fold planes); block partial sums.  Phase 2 (no fold): the start conv of flow_next, warp ->
// group-step and lane -> 8 (MG = 16) or 4 (MG = 32) consecutive channels; VEC = false: any C (fp32).
// MIX_LAST = false: W_{flow_next} mixes before the start conv (p.wmix).  MIX_LAST = true (the ax model's mix_first=False):
// wmix_done (may be NULL) mixes the trailing n_rem_done columns right after the coupling, and nothing mixes before the
// start conv - flow_next's own W follows its coupling in the next launch.
template <int XFMT, int MG, bool VEC, bool MIX_LAST>
__device__ __forceinline__ void fwd_boundary(const FwdP& p, const float* wmix_done, int n_rem_done) {
  __shared__ __align__(16) float a_s[TBF][MG / 2];
  __shared__ double red[TBF / 32];
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31, b = blockIdx.y;
  const int t0 = blockIdx.x * TBF, t = t0 + tid;
  const long long m0 = (long long)b * p.Tp + t0, m = m0 + tid;
  double lsum = 0.0, z2 = 0.0;
  if (t < p.Tp) {
    float a[MG];
    const float* src = p.audio_in ? p.audio_in + m * p.G : p.audio + m * p.G;
    if (p.vec4) {
      for (int g = 0; g < p.G; g += 4) {
        const float4 v = *reinterpret_cast<const float4*>(src + g);
        a[g] = v.x; a[g + 1] = v.y; a[g + 2] = v.z; a[g + 3] = v.w;
      }
    } else {
      for (int g = 0; g < p.G; ++g) a[g] = src[g];
    }
    if (p.do_flow) {                                               // audio_1 = exp(log_s) * audio_1 + b
      const int off = p.G - p.n_rem;
      float e[MG];
      const float4* ev = reinterpret_cast<const float4*>(p.eo + m * MG);
#pragma unroll
      for (int q = 0; q < MG / 4; ++q) { const float4 v = __ldcs(ev + q); e[4 * q] = v.x; e[4 * q + 1] = v.y; e[4 * q + 2] = v.z; e[4 * q + 3] = v.w; }
      for (int j = 0; j < p.n_half; ++j) {
        const float ls = e[p.n_half + j];
        a[off + p.n_half + j] = fmaf(expf(ls), a[off + p.n_half + j], e[j]);
        lsum += (double)ls;
        if (p.log_s) __stcs(p.log_s + ((size_t)b * p.n_half + j) * p.Tp + t, ls);
      }
    }
    if constexpr (MIX_LAST) {
      if (wmix_done) {                                             // efficient_model_ax.py mix_first=False: W_k after coupling k
        const int off = p.G - n_rem_done;
        float v[MG];
        for (int c = 0; c < n_rem_done; ++c) v[c] = a[off + c];
        for (int r = 0; r < n_rem_done; ++r) {
          float acc = 0.f;
          for (int c = 0; c < n_rem_done; ++c) acc = fmaf(__ldg(wmix_done + r * MG + c), v[c], acc);
          a[off + r] = acc;
        }
      }
      if (!p.do_next)
        for (int g = 0; g < p.G; ++g) z2 = fma((double)a[g], (double)a[g], z2);
    } else if (p.do_next) {                                        // audio = conv1d(audio, W), glow.py:85-99 (forward branch)
      const int off = p.G - p.n_rem2;
      float v[MG];
      for (int c = 0; c < p.n_rem2; ++c) v[c] = a[off + c];
      for (int r = 0; r < p.n_rem2; ++r) {
        float acc = 0.f;
        for (int c = 0; c < p.n_rem2; ++c) acc = fmaf(__ldg(p.wmix + r * MG + c), v[c], acc);
        a[off + r] = acc;
      }
    } else {
      for (int g = 0; g < p.G; ++g) z2 = fma((double)a[g], (double)a[g], z2);
    }
    float* dst = p.audio + m * p.G;
    if (p.vec4) for (int g = 0; g < p.G; g += 4) *reinterpret_cast<float4*>(dst + g) = make_float4(a[g], a[g + 1], a[g + 2], a[g + 3]);
    else for (int g = 0; g < p.G; ++g) dst[g] = a[g];
    if (p.do_next && p.a0_out) {
      // layer-0 fold: (audio_0 | 1 | 0...) as 16-bit hi / lo planes, exactly as the inverse direction builds them
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
    } else if (p.do_next) {
      const int off2 = p.G - p.n_rem2;
      for (int j = 0; j < MG / 2; ++j) a_s[tid][j] = j < p.n_half2 ? a[off2 + j] : 0.f;
    }
  }
  if (p.do_flow) {
    const double s = block_sum(lsum, red);
    if (tid == 0) p.ls_part[(size_t)b * p.nblk + blockIdx.x] = s;
  }
  if (p.z2_part) {
    const double s = block_sum(z2, red);
    if (tid == 0) p.z2_part[(size_t)b * p.nblk + blockIdx.x] = s;
  }
  if (!p.do_next || p.a0_out) return;
  __syncthreads();
  const int nrow = min(TBF, p.Tp - t0);
  if (!VEC) {                                                      // fp32, any C: thread -> channel
    for (int c = tid; c < p.C; c += TBF) {
      float w[MG / 2];
      for (int j = 0; j < MG / 2; ++j) w[j] = j < p.n_half2 ? __ldg(p.start_w + c * (MG / 2) + j) : 0.f;
      const float bias = __ldg(p.start_b + c);
      for (int r = 0; r < nrow; ++r) {
        float acc = bias;
        for (int j = 0; j < p.n_half2; ++j) acc = fmaf(w[j], a_s[r][j], acc);
        reinterpret_cast<float*>(p.x_out)[(size_t)(m0 + r) * p.C + c] = acc;
      }
    }
    return;
  }
  constexpr int NC = MG == 16 ? 8 : 4;                             // channels per lane (weights stay in registers)
  for (int cg = lane; cg < p.C / NC; cg += 32) {                   // audio = start(audio_0), glow.py:189
    const int c = cg * NC;
    float w[NC][MG / 2], bias[NC];
#pragma unroll
    for (int i = 0; i < NC; ++i) {
      bias[i] = __ldg(p.start_b + c + i);
#pragma unroll
      for (int j = 0; j < MG / 2; ++j) w[i][j] = j < p.n_half2 ? __ldg(p.start_w + (c + i) * (MG / 2) + j) : 0.f;
    }
    for (int r = warp; r < nrow; r += TBF / 32) {
      float x[NC];
#pragma unroll
      for (int i = 0; i < NC; ++i) x[i] = bias[i];
#pragma unroll
      for (int jq = 0; jq < MG / 8; ++jq) {
        const float4 a4 = *reinterpret_cast<const float4*>(&a_s[r][4 * jq]);
        const float av[4] = {a4.x, a4.y, a4.z, a4.w};
#pragma unroll
        for (int i = 0; i < NC; ++i)
#pragma unroll
          for (int j = 0; j < 4; ++j) x[i] = fmaf(w[i][4 * jq + j], av[j], x[i]);
      }
      store_x<XFMT, NC>(p, (size_t)(m0 + r) * p.C + c, x);
    }
  }
}

template <int XFMT, int MG, bool VEC>
__global__ void __launch_bounds__(TBF) k_fwd_boundary(FwdP p) {
  fwd_boundary<XFMT, MG, VEC, false>(p, nullptr, 0);
}

template <int XFMT, int MG, bool VEC>
__global__ void __launch_bounds__(TBF) k_fwd_boundary_mixlast(FwdP p, const float* wmix_done, int n_rem_done) {
  fwd_boundary<XFMT, MG, VEC, true>(p, wmix_done, n_rem_done);
}

// terms[b] = {sum z^2, sum log_s (all flows), T' * sum_k log|det W_k|}: the block partials added in a fixed order
__global__ void __launch_bounds__(TBF) k_fwd_reduce(const double* __restrict__ ls_part, const double* __restrict__ z2_part,
                                                    const double* __restrict__ logabsdet, int F, int B, int nblk, int Tp,
                                                    double* __restrict__ terms) {
  __shared__ double red[TBF / 32];
  const int b = blockIdx.x;
  double z2 = 0.0, ls = 0.0;
  for (int i = threadIdx.x; i < nblk; i += TBF) z2 += z2_part[(size_t)b * nblk + i];
  for (int i = threadIdx.x; i < F * nblk; i += TBF) {
    const int k = i / nblk, j = i - k * nblk;
    ls += ls_part[((size_t)k * B + b) * nblk + j];
  }
  z2 = block_sum(z2, red);
  ls = block_sum(ls, red);
  if (threadIdx.x == 0) {
    double ld = 0.0;
    for (int k = 0; k < F; ++k) ld += logabsdet[k];
    terms[(size_t)b * 3 + 0] = z2;
    terms[(size_t)b * 3 + 1] = ls;
    terms[(size_t)b * 3 + 2] = (double)Tp * ld;
  }
}

// ------------------------------------------------------------------------------------------
// WaveFlow's forward direction (cwg_wf_forward): one launch per flow boundary, a thread per group-step of the state
// [B*T'][G] (z), whose columns are read and written through the host's phys[] maps: PermuteHeight moves no data.
//   flow done: x[phys[r+1]] = x[phys[r+1]] * exp(log_s_r) + t_r, r = 0 .. G-2 (eo [G-1][B*T'][16]: log_s, t)
//   flow next: x0[r] = start(x[phys'[r]]), r = 0 .. G-2, as bf16 hi / lo planes [G-1][B*T'][128]
//   last     : z[c] = x[phys[c]] in logical order, and the block's sum of z^2
// ------------------------------------------------------------------------------------------
constexpr int WF_FWD_MAXG = 32, WF_FWD_C = 128;

struct WfFwdP {
  int Tp, G, nblk, F;
  long long BT, xplane;
  const float* audio_in;          // first launch: the waveform [B*T'][G]; NULL afterwards
  float* z;                       // the state, physical columns; the last launch leaves z in logical order
  const float* eo;                // coupling of the flow done, or NULL (first launch)
  double* ls_part;                // [B][nblk] sums of log_s of the flow done
  double* z2_part;                // [B][nblk] sums of z^2 (last launch), or NULL
  double* ld_zero;                // first launch: zeroes the [F] log|det| array k_fwd_reduce adds (PermuteHeight: 0)
  const float* start_w;           // [C] start conv of the next flow, or NULL (last launch)
  const float* start_b;
  __nv_bfloat16* x0;              // hi plane; the lo plane at x0 + xplane
  int phys_done[WF_FWD_MAXG], phys_next[WF_FWD_MAXG];
};

__global__ void __launch_bounds__(TBF) k_wf_fwd_boundary(WfFwdP p) {
  __shared__ float v_s[WF_FWD_MAXG - 1][TBF];
  __shared__ double red[TBF / 32];
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31, b = blockIdx.y;
  const int t0 = blockIdx.x * TBF, t = t0 + tid;
  const long long m0 = (long long)b * p.Tp + t0, m = m0 + tid;
  const bool next = p.start_w != nullptr;
  if (p.ld_zero && blockIdx.x == 0 && b == 0)
    for (int k = tid; k < p.F; k += TBF) p.ld_zero[k] = 0.0;
  double lsum = 0.0, z2 = 0.0;
  if (t < p.Tp) {
    float a[WF_FWD_MAXG];
    const float* src = (p.audio_in ? p.audio_in : p.z) + m * p.G;
    for (int g = 0; g < p.G; ++g) a[g] = src[g];
    if (p.eo) {                                                    // efficient_modules.py:42-65 run forward
      for (int r = 0; r + 1 < p.G; ++r) {
        const float2 e = __ldcs(reinterpret_cast<const float2*>(p.eo + ((size_t)r * p.BT + m) * CWG_EO_PAD));
        const int c = p.phys_done[r + 1];
        a[c] = fmaf(expf(e.x), a[c], e.y);
        lsum += (double)e.x;
      }
    }
    float* dst = p.z + m * p.G;
    if (next) {
      for (int r = 0; r + 1 < p.G; ++r) v_s[r][tid] = a[p.phys_next[r]];
      for (int g = 0; g < p.G; ++g) dst[g] = a[g];
    } else {
      for (int c = 0; c < p.G; ++c) {
        const float v = a[p.phys_done[c]];
        z2 = fma((double)v, (double)v, z2);
        dst[c] = v;
      }
    }
  }
  if (p.eo) {
    const double s = block_sum(lsum, red);
    if (tid == 0) p.ls_part[(size_t)b * p.nblk + blockIdx.x] = s;
  }
  if (!next) {
    const double s = block_sum(z2, red);
    if (tid == 0) p.z2_part[(size_t)b * p.nblk + blockIdx.x] = s;
    return;
  }
  __syncthreads();
  // start conv (glow_ax.py:558): warp -> group-step, lane -> 4 consecutive channels
  const int nrow = min(TBF, p.Tp - t0), c = 4 * lane;
  const float4 w4 = __ldg(reinterpret_cast<const float4*>(p.start_w + c));
  const float4 b4 = __ldg(reinterpret_cast<const float4*>(p.start_b + c));
  for (int r = 0; r + 1 < p.G; ++r) {
    for (int i = warp; i < nrow; i += TBF / 32) {
      const float v = v_s[r][i];
      const float x0 = fmaf(w4.x, v, b4.x), x1 = fmaf(w4.y, v, b4.y), x2 = fmaf(w4.z, v, b4.z), x3 = fmaf(w4.w, v, b4.w);
      const __nv_bfloat162 h01 = __floats2bfloat162_rn(x0, x1), h23 = __floats2bfloat162_rn(x2, x3);
      const __nv_bfloat162 l01 = __floats2bfloat162_rn(x0 - __low2float(h01), x1 - __high2float(h01));
      const __nv_bfloat162 l23 = __floats2bfloat162_rn(x2 - __low2float(h23), x3 - __high2float(h23));
      const size_t idx = ((size_t)r * p.BT + m0 + i) * WF_FWD_C + c;
      *reinterpret_cast<uint2*>(p.x0 + idx) = make_uint2(*reinterpret_cast<const uint32_t*>(&h01), *reinterpret_cast<const uint32_t*>(&h23));
      *reinterpret_cast<uint2*>(p.x0 + p.xplane + idx) =
          make_uint2(*reinterpret_cast<const uint32_t*>(&l01), *reinterpret_cast<const uint32_t*>(&l23));
    }
  }
}

template <int XFMT, int MG>
void launch_fb(dim3 grid, bool vec, const FwdP& p, bool mix_last, const float* wmix_done, int n_rem_done, cudaStream_t s) {
  if (mix_last) {
    if (vec) k_fwd_boundary_mixlast<XFMT, MG, true><<<grid, TBF, 0, s>>>(p, wmix_done, n_rem_done);
    else if constexpr (XFMT == 0) k_fwd_boundary_mixlast<XFMT, MG, false><<<grid, TBF, 0, s>>>(p, wmix_done, n_rem_done);
    return;
  }
  if (vec) k_fwd_boundary<XFMT, MG, true><<<grid, TBF, 0, s>>>(p);
  else if constexpr (XFMT == 0) k_fwd_boundary<XFMT, MG, false><<<grid, TBF, 0, s>>>(p);   // other widths: fp32 only
}

}  // namespace

int fwd_blocks(const Dims& d) { return (d.Tp + TBF - 1) / TBF; }

int launch_fwd_boundary(const cwg_config* cfg, const Dims& d, const cwg_weights* w, const float* w_fwd, int xfmt,
                        int flow_done, int flow_next, const float* audio_in, float* audio, const float* eo, float* log_s,
                        double* ls_part, double* z2_part, void* x_out, void* a0_out, cudaStream_t s, int mix_flow) {
  const bool mix_last = mix_flow != -2;
  FwdP p{};
  p.Tp = d.Tp; p.G = d.G; p.C = d.C; p.BT = d.BT; p.nblk = fwd_blocks(d);
  p.audio_in = audio_in; p.audio = audio;
  p.vec4 = (d.G & 3) == 0 && ((uintptr_t)audio & 15) == 0 && ((uintptr_t)(audio_in ? audio_in : audio) & 15) == 0;
  p.do_flow = flow_done >= 0; p.do_next = flow_next >= 0;
  p.eo = eo; p.log_s = log_s; p.ls_part = ls_part; p.z2_part = p.do_next ? nullptr : z2_part;
  p.x_out = x_out;
  p.a0_out = (xfmt != 0 && p.do_next) ? a0_out : nullptr;
  p.range_flag = xfmt == 2 ? range_flag() : nullptr;
  if (p.do_flow) { int nr; flow_channels(cfg, flow_done, &nr, &p.n_half); p.n_rem = nr; }
  if (p.do_next) {
    flow_channels(cfg, flow_next, &p.n_rem2, &p.n_half2);
    p.wmix = mix_last ? nullptr : w_fwd + (size_t)flow_next * d.MG * d.MG;
    p.start_w = w->start_w + (size_t)flow_next * d.C * (d.MG / 2);
    p.start_b = w->start_b + (size_t)flow_next * d.C;
  }
  CWG_REQUIRE(p.do_flow || p.do_next, "forward boundary: nothing to do");
  CWG_REQUIRE(!p.do_flow || (eo && ls_part), "forward boundary: eo / partials missing");
  CWG_REQUIRE(p.do_next || z2_part, "forward boundary: z^2 partials missing");
  CWG_REQUIRE(mix_flow >= -2 && mix_flow < cfg->n_flows, "forward boundary: mix flow out of range");
  const float* wmix_done = nullptr;
  int n_rem_done = 0;
  if (mix_flow >= 0) {
    int nh;
    flow_channels(cfg, mix_flow, &n_rem_done, &nh);
    wmix_done = w_fwd + (size_t)mix_flow * d.MG * d.MG;
  }
  const bool wide = d.MG != 16;
  CWG_REQUIRE(!wide || p.a0_out == nullptr, "the layer-0 fold takes n_group <= 16");
  const bool vec = (d.C & 7) == 0 && ((uintptr_t)x_out & 15) == 0;
  CWG_REQUIRE(vec || xfmt == 0, "the tensor-core modes need n_channels % 8 == 0");
  const dim3 grid((unsigned)p.nblk, (unsigned)d.B);
  if (wide) {
    if (xfmt == 0) launch_fb<0, 32>(grid, vec, p, mix_last, wmix_done, n_rem_done, s);
    else if (xfmt == 2) launch_fb<2, 32>(grid, vec, p, mix_last, wmix_done, n_rem_done, s);
    else launch_fb<1, 32>(grid, vec, p, mix_last, wmix_done, n_rem_done, s);
  } else {
    if (xfmt == 0) launch_fb<0, 16>(grid, vec, p, mix_last, wmix_done, n_rem_done, s);
    else if (xfmt == 2) launch_fb<2, 16>(grid, vec, p, mix_last, wmix_done, n_rem_done, s);
    else launch_fb<1, 16>(grid, vec, p, mix_last, wmix_done, n_rem_done, s);
  }
  CWG_CHECK_CUDA(cudaGetLastError());
  return 0;
}

int launch_fwd_reduce(const Dims& d, const double* ls_part, const double* z2_part, const double* logabsdet, double* terms,
                      cudaStream_t s) {
  return launch_fwd_reduce(d.F, d.B, fwd_blocks(d), d.Tp, ls_part, z2_part, logabsdet, terms, s);
}

int launch_fwd_reduce(int F, int B, int nblk, int Tp, const double* ls_part, const double* z2_part, const double* logabsdet,
                      double* terms, cudaStream_t s) {
  k_fwd_reduce<<<B, TBF, 0, s>>>(ls_part, z2_part, logabsdet, F, B, nblk, Tp, terms);
  CWG_CHECK_CUDA(cudaGetLastError());
  return 0;
}

int wf_fwd_blocks(int Tp) { return (Tp + TBF - 1) / TBF; }

int launch_wf_fwd_boundary(int B, int Tp, int G, int F, const float* audio_in, float* z, const float* eo,
                           const int* phys_done, const int* phys_next, const float* start_w, const float* start_b,
                           __nv_bfloat16* x0, long long xplane, double* ls_part, double* z2_part, double* ld_zero,
                           cudaStream_t s) {
  CWG_REQUIRE(G >= 2 && G <= WF_FWD_MAXG, "forward boundary: n_group must be in [2, %d]", WF_FWD_MAXG);
  CWG_REQUIRE((eo == nullptr) == (phys_done == nullptr) && (start_w == nullptr) == (phys_next == nullptr),
              "forward boundary: inconsistent arguments");
  CWG_REQUIRE(start_w || (phys_done && z2_part), "forward boundary: the last launch needs the flow done and z^2 partials");
  WfFwdP p{};
  p.Tp = Tp; p.G = G; p.F = F; p.BT = (long long)B * Tp; p.nblk = wf_fwd_blocks(Tp); p.xplane = xplane;
  p.audio_in = audio_in; p.z = z; p.eo = eo; p.ls_part = ls_part; p.z2_part = z2_part; p.ld_zero = ld_zero;
  p.start_w = start_w; p.start_b = start_b; p.x0 = x0;
  for (int c = 0; c < G; ++c) {
    p.phys_done[c] = phys_done ? phys_done[c] : c;
    p.phys_next[c] = phys_next ? phys_next[c] : c;
  }
  k_wf_fwd_boundary<<<dim3((unsigned)p.nblk, (unsigned)B), TBF, 0, s>>>(p);
  CWG_CHECK_CUDA(cudaGetLastError());
  return 0;
}

}  // namespace cwg
