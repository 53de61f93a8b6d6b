// cwg_pack_weights: reference state_dict (device fp32 tensors, glow.py parameter names) -> the packed arrays of
// cwg_weights, on the device, in fp64.  The three exact rewrites of DESIGN.md "Packed weights":
//   1. weight-norm folded (w = g * v / ||v||; glow.py:136-186 applies torch.nn.utils.weight_norm to every WN conv);
//   2. cond_layers[1] . cond_layers[0] (glow.py:198-199) folded with the ConvTranspose1d upsampler + squeeze
//      (glow.py:238-241, 318-324) into one per-phase map from J mel frames to the H-wide hidden cond vector;
//      cond_layers[2] becomes H extra K columns of every in_layer GEMM;
//   3. `end` (glow.py:222) folded into the skip half of res_skip: 2*n_half output rows instead of a C-wide skip sum.
// W^-1 of every Invertible1x1Conv (glow.py:85-99) is computed here too (Gauss-Jordan with partial pivoting, fp64).
// The numpy version of the same algebra (cookietts_b200/packing.py) is what tests/test_pack_c.py checks this against.
#include "cwg_common.cuh"

#include <cuda_fp16.h>
#include <cuda_fp8.h>
#include <string.h>

namespace cwg {
namespace {

// ---------------------------------------------------------------------------------- output planes
struct Planes {
  float* f32;
  uint16_t *hi, *lo;
  uint8_t *h8, *l8;
  int fmt;                // 0: fp32; 1: bf16 hi + lo; 2: fp16 hi + lo (+ the two e5m2 planes when h8 != NULL)
};

__device__ __forceinline__ uint8_t e5m2_sat(double x) {
  float f = (float)x;
  f = fminf(fmaxf(f, -57344.f), 57344.f);
  return (uint8_t)__nv_cvt_float_to_fp8(f, __NV_SATFINITE, __NV_E5M2);
}

__device__ __forceinline__ void emit(const Planes& p, size_t i, double w) {
  if (p.fmt == 0) {
    p.f32[i] = (float)w;
  } else if (p.fmt == 1) {
    const __nv_bfloat16 h = __float2bfloat16_rn((float)w);
    const __nv_bfloat16 l = __float2bfloat16_rn((float)(w - (double)__bfloat162float(h)));
    p.hi[i] = __bfloat16_as_ushort(h);
    p.lo[i] = __bfloat16_as_ushort(l);
  } else {
    const __half h = __double2half(w);
    const double hd = (double)__half2float(h);
    const __half l = __double2half(w - hd);
    p.hi[i] = __half_as_ushort(h);
    p.lo[i] = __half_as_ushort(l);
    if (p.h8) {                                      // packing.py f8_correction_planes: 2^-P on hi, 2^Q on lo
      p.h8[i] = e5m2_sat(hd * (1.0 / 64.0));
      p.l8[i] = e5m2_sat((w - hd) * 256.0);
    }
  }
}

// ---------------------------------------------------------------------------------- kernels
// effective weight of a (possibly weight-normed) conv, one block per output row: out[r][:] = g[r] * v[r][:] / ||v[r]||
__global__ void k_effective(const float* __restrict__ v, const float* __restrict__ g, int cols, double* __restrict__ out) {
  const int r = blockIdx.x;
  const float* vr = v + (size_t)r * cols;
  double* o = out + (size_t)r * cols;
  __shared__ double red[256];
  double scale = 1.0;
  if (g) {
    double s = 0.0;
    for (int c = threadIdx.x; c < cols; c += blockDim.x) { const double x = vr[c]; s += x * x; }
    red[threadIdx.x] = s;
    __syncthreads();
    for (int k = blockDim.x / 2; k > 0; k >>= 1) {
      if (threadIdx.x < k) red[threadIdx.x] += red[threadIdx.x + k];
      __syncthreads();
    }
    scale = (double)g[r] / sqrt(red[0]);
  }
  for (int c = threadIdx.x; c < cols; c += blockDim.x) o[c] = g ? (double)vr[c] * scale : (double)vr[c];
}

// out[m][n] = sum_k a[m][k] * b[k][n]
__global__ void k_matmul64(const double* __restrict__ a, const double* __restrict__ b, int M, int K, int N, double* __restrict__ out) {
  const int n = blockIdx.x * blockDim.x + threadIdx.x, m = blockIdx.y;
  if (n >= N) return;
  double s = 0.0;
  for (int k = 0; k < K; ++k) s += a[(size_t)m * K + k] * b[(size_t)k * N + n];
  out[(size_t)m * N + n] = s;
}

// cond_w[p*H + h][j*M + ci] = sum_{m,g} w21[h][m*G + g] * w_up[ci][m][j*hop + p*G + g]   (taps past `win` are zero)
__global__ void k_cond_w(const double* __restrict__ w21, int ld21, const float* __restrict__ w_up, int M, int G, int P, int J,
                         int H, int hop, int win, int KCp, Planes out, size_t out0) {
  const int col = blockIdx.x * blockDim.x + threadIdx.x, row = blockIdx.y;
  if (col >= KCp) return;
  const int p = row / H, h = row - p * H;
  double s = 0.0;
  if (col < J * M) {
    const int j = col / M, ci = col - j * M;
    const int t0 = j * hop + p * G;
    for (int m = 0; m < M; ++m) {
      const float* wu = w_up + ((size_t)ci * M + m) * win;
      const double* w2 = w21 + (size_t)h * ld21 + (size_t)m * G;
      for (int g = 0; g < G; ++g)
        if (t0 + g < win) s += w2[g] * (double)wu[t0 + g];
    }
  }
  emit(out, out0 + (size_t)row * KCp + col, s);
}

// cond_b[h] = sum_{m,g} w21[h][m*G+g] * b_up[m] + sum_j c1[h][j] * cb0[j] + cb1[h];  cond_w_spk[h][e] = w21[h][M*G + e]
__global__ void k_cond_b(const double* __restrict__ w21, int ld21, const double* __restrict__ c1, const float* __restrict__ b_up,
                         const float* __restrict__ cb0, const float* __restrict__ cb1, int M, int G, int H, int E,
                         float* __restrict__ cond_b, float* __restrict__ cond_w_spk) {
  const int h = blockIdx.x * blockDim.x + threadIdx.x;
  if (h >= H) return;
  double s = (double)cb1[h];
  for (int m = 0; m < M; ++m)
    for (int g = 0; g < G; ++g) s += w21[(size_t)h * ld21 + m * G + g] * (double)b_up[m];
  for (int j = 0; j < H; ++j) s += c1[(size_t)h * H + j] * (double)cb0[j];
  cond_b[h] = (float)s;
  for (int e = 0; e < E; ++e) cond_w_spk[(size_t)h * E + e] = (float)w21[(size_t)h * ld21 + M * G + e];
}

// w1[o][tap*C + c] = in_layer[o][c][tap];  w1[o][ks*C + h] = cond_layers.2[2C*i + o][h];  b1[o] = in_bias[o] + cb2[2C*i + o]
__global__ void k_w1(const double* __restrict__ w_in, const double* __restrict__ c2, const float* __restrict__ b_in,
                     const float* __restrict__ cb2, int C, int ks, int H, int layer, Planes out, size_t out0, float* __restrict__ b1) {
  const int K1 = ks * C + H;
  const int col = blockIdx.x * blockDim.x + threadIdx.x, o = blockIdx.y;
  if (col >= K1) return;
  double v;
  if (col < ks * C) {
    const int tap = col / C, c = col - tap * C;
    v = w_in[((size_t)o * C + c) * ks + tap];
  } else {
    v = c2[((size_t)2 * C * layer + o) * H + (col - ks * C)];
  }
  emit(out, out0 + (size_t)o * K1 + col, v);
  if (col == 0) b1[o] = (float)((double)b_in[o] + (double)cb2[2 * C * layer + o]);
}

// w2[row][c]: rows < C = alpha * res rows (zero for the last layer), rows [C, C + 2 n_half) = W_end (alpha W_skip), rest 0
__global__ void k_w2(const double* __restrict__ w_rs, const double* __restrict__ w_end, const float* __restrict__ b_rs,
                     const float* __restrict__ alpha, int C, int n2h, int last, Planes out, size_t out0, float* __restrict__ b2) {
  const int c = blockIdx.x * blockDim.x + threadIdx.x, row = blockIdx.y;
  if (c >= C) return;
  const double al = alpha ? (double)alpha[0] : 1.0;
  double v = 0.0;
  if (row < C) {
    if (!last) v = w_rs[(size_t)row * C + c] * al;
    if (c == 0) b2[row] = last ? 0.f : (float)((double)b_rs[row] * al);
  } else if (row < C + n2h) {
    const double* we = w_end + (size_t)(row - C) * C;
    const double* ws = w_rs + (last ? 0 : (size_t)C * C);
    for (int k = 0; k < C; ++k) v += we[k] * (ws[(size_t)k * C + c] * al);
  }
  emit(out, out0 + (size_t)row * C + c, v);
}

// layer-0 fold: w0[o][tap*16 + j] = sum_c in_layers.0[o][c][tap] * (j < n_half ? start[c][j] : j == n_half ? start_bias[c] : 0)
__global__ void k_w0(const double* __restrict__ w_in, const double* __restrict__ w_start, const float* __restrict__ b_start,
                     int C, int ks, int n_half, Planes out, size_t out0) {
  const int col = threadIdx.x, o = blockIdx.x;             // 48 columns, 2C rows
  if (col >= 48) return;
  const int tap = col / 16, j = col - tap * 16;
  double v = 0.0;
  if (tap < ks && j <= n_half)
    for (int c = 0; c < C; ++c)
      v += w_in[((size_t)o * C + c) * ks + tap] * (j < n_half ? w_start[(size_t)c * n_half + j] : (double)b_start[c]);
  // only the 16-bit hi / lo planes exist for w0 (three products in every tensor-core mode)
  Planes p = out; p.h8 = nullptr; p.l8 = nullptr;
  emit(p, out0 + (size_t)o * 48 + col, v);
}

struct EoArgs { const float* b_rs[16]; const float* alpha[16]; };
// eo_b[r] = b_end[r] + sum_i sum_c W_end[r][c] * alpha_i * b_skip_i[c]
__global__ void k_eo_b(const double* __restrict__ w_end, const float* __restrict__ b_end, EoArgs a, int C, int L, int n2h,
                       int mg, float* __restrict__ eo_b) {
  const int r = threadIdx.x;
  if (r >= mg) return;
  double s = 0.0;
  if (r < n2h) {
    s = (double)b_end[r];
    for (int i = 0; i < L; ++i) {
      const double al = a.alpha[i] ? (double)a.alpha[i][0] : 1.0;
      const float* bs = a.b_rs[i] + (i < L - 1 ? C : 0);
      for (int c = 0; c < C; ++c) s += w_end[(size_t)r * C + c] * ((double)bs[c] * al);
    }
  }
  eo_b[r] = (float)s;
}

__global__ void k_start(const double* __restrict__ w, const float* __restrict__ b, int C, int n_half, int mg, float* __restrict__ start_w,
                        float* __restrict__ start_b) {
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= C) return;
  for (int j = 0; j < mg / 2; ++j) start_w[(size_t)c * (mg / 2) + j] = j < n_half ? (float)w[(size_t)c * n_half + j] : 0.f;
  start_b[c] = b[c];
}

// W^-1 of the n x n mixing matrix (glow.py:93 inverts in fp32; fp64 here), zero-padded to [mg][mg] (mg = CWG_GROUP_PAD(n_group))
__global__ void k_winv(const float* __restrict__ W, int n, int mg, float* __restrict__ out, int* __restrict__ singular) {
  __shared__ double a[CWG_MAX_GROUP][2 * CWG_MAX_GROUP];
  if (threadIdx.x != 0) return;
  for (int i = 0; i < n; ++i)
    for (int j = 0; j < n; ++j) { a[i][j] = (double)W[i * n + j]; a[i][n + j] = i == j ? 1.0 : 0.0; }
  for (int col = 0; col < n; ++col) {
    int piv = col;
    for (int r = col + 1; r < n; ++r) if (fabs(a[r][col]) > fabs(a[piv][col])) piv = r;
    if (a[piv][col] == 0.0) { *singular = 1; return; }
    if (piv != col) for (int j = 0; j < 2 * n; ++j) { const double t = a[col][j]; a[col][j] = a[piv][j]; a[piv][j] = t; }
    const double d = a[col][col];
    for (int j = 0; j < 2 * n; ++j) a[col][j] /= d;
    for (int r = 0; r < n; ++r) {
      if (r == col) continue;
      const double f = a[r][col];
      if (f != 0.0) for (int j = 0; j < 2 * n; ++j) a[r][j] -= f * a[col][j];
    }
  }
  for (int i = 0; i < mg; ++i)
    for (int j = 0; j < mg; ++j) out[i * mg + j] = (i < n && j < n) ? (float)a[i][n + j] : 0.f;
}

// Forward direction: W itself zero-padded to [mg][mg], and log det W from an fp64 LU with partial pivoting.
// logdet[flow] follows torch.logdet (NaN for det < 0, -inf for det = 0); logdet[n_flows + flow] = log|det W|.
__global__ void k_wfwd(const float* __restrict__ W, int n, int mg, int flow, int n_flows, float* __restrict__ out,
                       double* __restrict__ logdet) {
  __shared__ double a[CWG_MAX_GROUP][CWG_MAX_GROUP];
  if (threadIdx.x != 0) return;
  for (int i = 0; i < mg; ++i)
    for (int j = 0; j < mg; ++j) out[i * mg + j] = (i < n && j < n) ? W[i * n + j] : 0.f;
  for (int i = 0; i < n; ++i)
    for (int j = 0; j < n; ++j) a[i][j] = (double)W[i * n + j];
  double logabs = 0.0;
  int neg = 0;
  for (int col = 0; col < n; ++col) {
    int piv = col;
    for (int r = col + 1; r < n; ++r) if (fabs(a[r][col]) > fabs(a[piv][col])) piv = r;
    if (a[piv][col] == 0.0) { logabs = -INFINITY; neg = 0; break; }
    if (piv != col) {
      neg ^= 1;
      for (int j = col; j < n; ++j) { const double t = a[col][j]; a[col][j] = a[piv][j]; a[piv][j] = t; }
    }
    const double d = a[col][col];
    if (d < 0.0) neg ^= 1;
    logabs += log(fabs(d));
    for (int r = col + 1; r < n; ++r) {
      const double f = a[r][col] / d;
      if (f != 0.0) for (int j = col; j < n; ++j) a[r][j] -= f * a[col][j];
    }
  }
  logdet[flow] = neg ? (double)NAN : logabs;
  logdet[n_flows + flow] = logabs;
}

// cond_bias[b][f][h] = cond_b_base[f][h] + sum_e cond_w_spk[f][h][e] * speaker_embed_f[ids[b]][e]   (glow.py:193-196)
__global__ void k_cond_bias(const float* __restrict__ base, const float* __restrict__ wspk, const float* __restrict__ emb,
                            const long long* __restrict__ ids, int F, int H, int E, int S, float* __restrict__ out) {
  const int h = blockIdx.x * blockDim.x + threadIdx.x, f = blockIdx.y, b = blockIdx.z;
  if (h >= H) return;
  float s = base[(size_t)f * H + h];
  if (E > 0 && ids) {
    long long id = ids[b];
    id = id < 0 ? 0 : (id >= S ? S - 1 : id);            // the host checks the range; never read out of bounds
    const float* e = emb + ((size_t)f * S + id) * E;
    const float* w = wspk + ((size_t)f * H + h) * E;
    float acc = 0.f;
    for (int k = 0; k < E; ++k) acc += w[k] * e[k];
    s += acc;
  }
  out[((size_t)b * F + f) * H + h] = s;
}

// ---------------------------------------------------------------------------------- host side
const cwg_tensor* find(const cwg_tensor* sd, int n, const char* name) {
  for (int i = 0; i < n; ++i)
    if (sd[i].name && strcmp(sd[i].name, name) == 0) return &sd[i];
  return nullptr;
}

long long numel(const cwg_tensor* t) {
  long long k = 1;
  for (int i = 0; i < t->ndim; ++i) k *= t->shape[i];
  return k;
}

struct Layout {
  size_t cond_w, w1, w2, b1, b2, eo_b, start_w, start_b, winv, cond_b_base, cond_w_spk, spk_embed;   // element counts
  size_t off_cond_w[3], off_w1[3], off_w2[3], off_w1_8[2], off_w2_8[2], off_w0[2], w0;
  size_t off_b1, off_b2, off_eo_b, off_start_w, off_start_b, off_winv, off_cond_b_base, off_cond_w_spk, off_spk_embed;
  size_t bytes;
};

Layout make_layout(const cwg_config* c, int mode, int E, int S) {
  Layout l;
  memset(&l, 0, sizeof(l));
  const Dims d = make_dims(c, 1, 1);
  const size_t F = d.F, L = d.L, C = d.C, H = d.H;
  l.cond_w = F * d.P * H * d.KCp; l.w1 = F * L * 2 * C * d.K1; l.w2 = F * L * d.N2 * C;
  l.b1 = F * L * 2 * C; l.b2 = F * L * C; l.eo_b = F * (size_t)d.MG;
  l.start_w = F * C * (size_t)(d.MG / 2); l.start_b = F * C; l.winv = F * (size_t)d.MG * d.MG;
  l.cond_b_base = F * H; l.cond_w_spk = F * H * (size_t)(E > 0 ? E : 1); l.spk_embed = F * (size_t)S * E;
  size_t off = 0;
  auto take = [&](size_t bytes) { const size_t o = off; off = align_up(off + bytes, 256); return o; };
  if (mode == CWG_MODE_FFMA) {
    l.off_cond_w[0] = take(l.cond_w * 4); l.off_w1[0] = take(l.w1 * 4); l.off_w2[0] = take(l.w2 * 4);
  } else {
    l.off_cond_w[1] = take(l.cond_w * 2); l.off_cond_w[2] = take(l.cond_w * 2);
    l.off_w1[1] = take(l.w1 * 2); l.off_w1[2] = take(l.w1 * 2);
    l.off_w2[1] = take(l.w2 * 2); l.off_w2[2] = take(l.w2 * 2);
    if (mode == CWG_MODE_F16F8) {
      l.off_w1_8[0] = take(l.w1); l.off_w1_8[1] = take(l.w1);
      l.off_w2_8[0] = take(l.w2); l.off_w2_8[1] = take(l.w2);
    }
    if (d.ks == 3 && C == 256) {                      // layer-0 fold planes (the persistent 256-channel layer kernel)
      l.w0 = F * 2 * C * 48;
      l.off_w0[0] = take(l.w0 * 2); l.off_w0[1] = take(l.w0 * 2);
    }
  }
  l.off_b1 = take(l.b1 * 4); l.off_b2 = take(l.b2 * 4); l.off_eo_b = take(l.eo_b * 4);
  l.off_start_w = take(l.start_w * 4); l.off_start_b = take(l.start_b * 4); l.off_winv = take(l.winv * 4);
  l.off_cond_b_base = take(l.cond_b_base * 4); l.off_cond_w_spk = take(l.cond_w_spk * 4);
  l.off_spk_embed = take((l.spk_embed ? l.spk_embed : 1) * 4);
  l.bytes = off;
  return l;
}

void view(const Layout& l, int mode, int E, int S, void* packed, cwg_weights* w) {
  char* p = (char*)packed;
  memset(w, 0, sizeof(*w));
  if (mode == CWG_MODE_FFMA) {
    w->cond_w_f32 = (const float*)(p + l.off_cond_w[0]); w->w1_f32 = (const float*)(p + l.off_w1[0]);
    w->w2_f32 = (const float*)(p + l.off_w2[0]);
  } else {
    w->cond_w_hi = (const uint16_t*)(p + l.off_cond_w[1]); w->cond_w_lo = (const uint16_t*)(p + l.off_cond_w[2]);
    w->w1_hi = (const uint16_t*)(p + l.off_w1[1]); w->w1_lo = (const uint16_t*)(p + l.off_w1[2]);
    w->w2_hi = (const uint16_t*)(p + l.off_w2[1]); w->w2_lo = (const uint16_t*)(p + l.off_w2[2]);
    if (mode == CWG_MODE_F16F8) {
      w->w1_h8 = (const uint8_t*)(p + l.off_w1_8[0]); w->w1_l8 = (const uint8_t*)(p + l.off_w1_8[1]);
      w->w2_h8 = (const uint8_t*)(p + l.off_w2_8[0]); w->w2_l8 = (const uint8_t*)(p + l.off_w2_8[1]);
    }
    if (l.w0) { w->w0_hi = (const uint16_t*)(p + l.off_w0[0]); w->w0_lo = (const uint16_t*)(p + l.off_w0[1]); }
  }
  w->b1 = (const float*)(p + l.off_b1); w->b2 = (const float*)(p + l.off_b2); w->eo_b = (const float*)(p + l.off_eo_b);
  w->start_w = (const float*)(p + l.off_start_w); w->start_b = (const float*)(p + l.off_start_b);
  w->winv = (const float*)(p + l.off_winv);
  w->cond_b_base = (const float*)(p + l.off_cond_b_base); w->cond_w_spk = (const float*)(p + l.off_cond_w_spk);
  w->spk_embed = E > 0 ? (const float*)(p + l.off_spk_embed) : nullptr;
  w->speaker_embed_dim = E; w->n_speakers = S;
}

Planes planes_of(const cwg_weights& w, int mode, int which) {      // which: 0 cond_w, 1 w1, 2 w2
  Planes p;
  memset(&p, 0, sizeof(p));
  p.fmt = mode == CWG_MODE_FFMA ? 0 : (mode == CWG_MODE_F16F8 ? 2 : 1);
  if (which == 0) { p.f32 = (float*)w.cond_w_f32; p.hi = (uint16_t*)w.cond_w_hi; p.lo = (uint16_t*)w.cond_w_lo; }
  if (which == 1) { p.f32 = (float*)w.w1_f32; p.hi = (uint16_t*)w.w1_hi; p.lo = (uint16_t*)w.w1_lo; p.h8 = (uint8_t*)w.w1_h8; p.l8 = (uint8_t*)w.w1_l8; }
  if (which == 2) { p.f32 = (float*)w.w2_f32; p.hi = (uint16_t*)w.w2_hi; p.lo = (uint16_t*)w.w2_lo; p.h8 = (uint8_t*)w.w2_h8; p.l8 = (uint8_t*)w.w2_l8; }
  return p;
}

// speaker_embed_dim / n_speakers / rezero are properties of the checkpoint: read them off the state_dict
int inspect(const cwg_tensor* sd, int n, int* E, int* S, int* rezero) {
  CWG_REQUIRE(sd != nullptr && n > 0, "state_dict is empty");
  const cwg_tensor* t = find(sd, n, "WN.0.speaker_embed.weight");
  *E = 0; *S = 0;
  if (t) { CWG_REQUIRE(t->ndim == 2, "WN.0.speaker_embed.weight must be 2-D"); *S = (int)t->shape[0]; *E = (int)t->shape[1]; }
  *rezero = find(sd, n, "WN.0.alpha_i.0") != nullptr;
  return 0;
}

size_t pack_ws_bytes(const cwg_config* c, int E) {
  const Dims d = make_dims(c, 1, 1);
  const size_t C = d.C, H = d.H, L = d.L, n0 = (size_t)d.M * d.G + E;
  size_t dbl = 2 * H * n0 + H * H + 2 * C * L * H + 2 * C * C * d.ks + 2 * C * C + (size_t)CWG_MAX_GROUP * C + C * (CWG_MAX_GROUP / 2);
  return dbl * 8 + 8 * 256 + 256;
}

// effective (weight-norm folded) weight of conv `prefix` -> out64 [rows][cols]
int effective(const cwg_tensor* sd, int n, const char* prefix, long long rows, long long cols, double* out, cudaStream_t s) {
  char name[160];
  snprintf(name, sizeof(name), "%s.weight_g", prefix);
  const cwg_tensor* g = find(sd, n, name);
  snprintf(name, sizeof(name), g ? "%s.weight_v" : "%s.weight", prefix);
  const cwg_tensor* v = find(sd, n, name);
  CWG_REQUIRE(v != nullptr, "state_dict has no %s", name);
  CWG_REQUIRE(v->ndim >= 1 && v->shape[0] == rows && numel(v) == rows * cols,
              "%s: expected %lld x %lld elements, got shape[0] = %lld, numel = %lld", name, rows, cols, (long long)v->shape[0], numel(v));
  if (g) CWG_REQUIRE(numel(g) == rows, "%s.weight_g: expected %lld elements", prefix, rows);
  k_effective<<<(unsigned)rows, 256, 0, s>>>(v->data, g ? g->data : nullptr, (int)cols, out);
  CWG_CHECK_CUDA(cudaGetLastError());
  return 0;
}

int need(const cwg_tensor* sd, int n, const char* name, long long count, const float** out) {
  const cwg_tensor* t = find(sd, n, name);
  CWG_REQUIRE(t != nullptr, "state_dict has no %s", name);
  CWG_REQUIRE(numel(t) == count, "%s: expected %lld elements, got %lld", name, count, numel(t));
  *out = t->data;
  return 0;
}

}  // namespace
}  // namespace cwg

using namespace cwg;

extern "C" {

size_t cwg_packed_bytes(const cwg_config* cfg, int mode, int speaker_embed_dim, int n_speakers) {
  if (!cfg || speaker_embed_dim < 0 || n_speakers < 0) { set_error("cwg_packed_bytes: bad arguments"); return 0; }
  return make_layout(cfg, mode, speaker_embed_dim, n_speakers).bytes;
}

size_t cwg_pack_workspace_bytes(const cwg_config* cfg, int speaker_embed_dim) {
  if (!cfg || speaker_embed_dim < 0) { set_error("cwg_pack_workspace_bytes: bad arguments"); return 0; }
  return pack_ws_bytes(cfg, speaker_embed_dim);
}

int cwg_state_dict_info(const cwg_tensor* sd, int n_tensors, int* speaker_embed_dim, int* n_speakers, int* rezero) {
  int E, S, rz;
  if (int r = inspect(sd, n_tensors, &E, &S, &rz)) return r;
  if (speaker_embed_dim) *speaker_embed_dim = E;
  if (n_speakers) *n_speakers = S;
  if (rezero) *rezero = rz;
  return 0;
}

int cwg_packed_view(const cwg_config* cfg, int mode, int speaker_embed_dim, int n_speakers, void* packed, size_t packed_bytes,
                    cwg_weights* out) {
  CWG_REQUIRE(cfg && packed && out, "cwg_packed_view: NULL argument");
  const Layout l = make_layout(cfg, mode, speaker_embed_dim, n_speakers);
  CWG_REQUIRE(packed_bytes >= l.bytes, "packed buffer too small: %zu < %zu bytes", packed_bytes, l.bytes);
  CWG_REQUIRE(((uintptr_t)packed & 255) == 0, "packed buffer must be 256-byte aligned");
  view(l, mode, speaker_embed_dim, n_speakers, packed, out);
  return 0;
}

int cwg_pack_weights(const cwg_config* cfg, int mode, const cwg_tensor* sd, int n_tensors, void* packed, size_t packed_bytes,
                     void* workspace, size_t workspace_bytes, cwg_weights* out, void* cuda_stream) {
  CWG_REQUIRE(cfg && packed && workspace && out, "cwg_pack_weights: NULL argument");
  CWG_REQUIRE(mode == CWG_MODE_FFMA || mode == CWG_MODE_BF16X3 || mode == CWG_MODE_BF16 || mode == CWG_MODE_F16F8, "unknown mode %d", mode);
  CWG_REQUIRE(cfg->n_group % 2 == 0 && cfg->n_group >= 2 && cfg->n_group <= CWG_MAX_GROUP && cfg->hop_length % cfg->n_group == 0 &&
              cfg->n_layers >= 1 && cfg->n_layers <= 16 && cfg->kernel_size % 2 == 1, "bad configuration");
  int E, S, rezero;
  if (int r = inspect(sd, n_tensors, &E, &S, &rezero)) return r;
  const Layout l = make_layout(cfg, mode, E, S);
  CWG_REQUIRE(packed_bytes >= l.bytes, "packed buffer too small: %zu < %zu bytes", packed_bytes, l.bytes);
  CWG_REQUIRE(workspace_bytes >= pack_ws_bytes(cfg, E), "pack workspace too small: %zu < %zu bytes", workspace_bytes, pack_ws_bytes(cfg, E));
  CWG_REQUIRE(((uintptr_t)packed & 255) == 0 && ((uintptr_t)workspace & 255) == 0, "buffers must be 256-byte aligned");
  cudaStream_t s = (cudaStream_t)cuda_stream;
  cwg_weights w;
  view(l, mode, E, S, packed, &w);
  const Dims d = make_dims(cfg, 1, 1);
  const int F = d.F, L = d.L, C = d.C, H = d.H, M = d.M, G = d.G, ks = d.ks, n0 = M * G + E;

  // fp64 scratch (re-used flow after flow; everything runs on one stream)
  double* ws = (double*)workspace;
  double* c0 = ws;            ws += (size_t)H * n0;
  double* c1 = ws;            ws += (size_t)H * H;
  double* c2 = ws;            ws += (size_t)2 * C * L * H;
  double* w21 = ws;           ws += (size_t)H * n0;
  double* w_in = ws;          ws += (size_t)2 * C * C * ks;
  double* w_rs = ws;          ws += (size_t)2 * C * C;
  double* w_end = ws;         ws += (size_t)CWG_MAX_GROUP * C;
  double* w_start = ws;       ws += (size_t)C * (CWG_MAX_GROUP / 2);
  int* singular = (int*)ws;
  CWG_CHECK_CUDA(cudaMemsetAsync(singular, 0, sizeof(int), s));
  CWG_CHECK_CUDA(cudaMemsetAsync(packed, 0, l.bytes, s));

  const cwg_tensor* up = find(sd, n_tensors, "upsample.weight");
  CWG_REQUIRE(up && up->ndim == 3 && up->shape[0] == M && up->shape[1] == M && up->shape[2] == cfg->win_length,
              "upsample.weight must be [%d, %d, %d] (only upsample_mode='normal' is supported)", M, M, cfg->win_length);
  const float* b_up;
  if (int r = need(sd, n_tensors, "upsample.bias", M, &b_up)) return r;
  const Planes p_cond = planes_of(w, mode, 0), p_w1 = planes_of(w, mode, 1), p_w2 = planes_of(w, mode, 2);
  char nm[160];

  for (int k = 0; k < F; ++k) {
    int n_rem, n_half;
    flow_channels(cfg, k, &n_rem, &n_half);
    const int n2h = 2 * n_half;
    // ---- cond chain folded with upsample + squeeze
    snprintf(nm, sizeof(nm), "WN.%d.cond_layers.0", k); if (int r = effective(sd, n_tensors, nm, H, n0, c0, s)) return r;
    snprintf(nm, sizeof(nm), "WN.%d.cond_layers.1", k); if (int r = effective(sd, n_tensors, nm, H, H, c1, s)) return r;
    snprintf(nm, sizeof(nm), "WN.%d.cond_layers.2", k); if (int r = effective(sd, n_tensors, nm, (long long)2 * C * L, H, c2, s)) return r;
    const float *cb0, *cb1, *cb2;
    snprintf(nm, sizeof(nm), "WN.%d.cond_layers.0.bias", k); if (int r = need(sd, n_tensors, nm, H, &cb0)) return r;
    snprintf(nm, sizeof(nm), "WN.%d.cond_layers.1.bias", k); if (int r = need(sd, n_tensors, nm, H, &cb1)) return r;
    snprintf(nm, sizeof(nm), "WN.%d.cond_layers.2.bias", k); if (int r = need(sd, n_tensors, nm, (long long)2 * C * L, &cb2)) return r;
    k_matmul64<<<dim3((n0 + 127) / 128, H), 128, 0, s>>>(c1, c0, H, H, n0, w21);
    k_cond_w<<<dim3((d.KCp + 63) / 64, d.P * H), 64, 0, s>>>(w21, n0, up->data, M, G, d.P, d.J, H, cfg->hop_length, cfg->win_length,
                                                            d.KCp, p_cond, (size_t)k * d.P * H * d.KCp);
    k_cond_b<<<(H + 63) / 64, 64, 0, s>>>(w21, n0, c1, b_up, cb0, cb1, M, G, H, E, (float*)w.cond_b_base + (size_t)k * H,
                                         (float*)w.cond_w_spk + (size_t)k * H * (E > 0 ? E : 1));
    if (E > 0) {
      const float* emb;
      snprintf(nm, sizeof(nm), "WN.%d.speaker_embed.weight", k); if (int r = need(sd, n_tensors, nm, (long long)S * E, &emb)) return r;
      CWG_CHECK_CUDA(cudaMemcpyAsync((float*)w.spk_embed + (size_t)k * S * E, emb, (size_t)S * E * 4, cudaMemcpyDeviceToDevice, s));
    }
    // ---- end / start / W^-1
    snprintf(nm, sizeof(nm), "WN.%d.end", k); if (int r = effective(sd, n_tensors, nm, n2h, C, w_end, s)) return r;
    const float* b_end;
    snprintf(nm, sizeof(nm), "WN.%d.end.bias", k); if (int r = need(sd, n_tensors, nm, n2h, &b_end)) return r;
    snprintf(nm, sizeof(nm), "WN.%d.start", k); if (int r = effective(sd, n_tensors, nm, C, n_half, w_start, s)) return r;
    const float* b_start;
    snprintf(nm, sizeof(nm), "WN.%d.start.bias", k); if (int r = need(sd, n_tensors, nm, C, &b_start)) return r;
    k_start<<<(C + 127) / 128, 128, 0, s>>>(w_start, b_start, C, n_half, d.MG, (float*)w.start_w + (size_t)k * C * (d.MG / 2),
                                           (float*)w.start_b + (size_t)k * C);
    const float* Wm;
    snprintf(nm, sizeof(nm), "convinv.%d.conv.weight", k); if (int r = need(sd, n_tensors, nm, (long long)n_rem * n_rem, &Wm)) return r;
    k_winv<<<1, 32, 0, s>>>(Wm, n_rem, d.MG, (float*)w.winv + (size_t)k * d.MG * d.MG, singular);
    // ---- layers
    EoArgs ea;
    memset(&ea, 0, sizeof(ea));
    for (int i = 0; i < L; ++i) {
      const bool last = i == L - 1;
      const size_t idx = (size_t)k * L + i;
      snprintf(nm, sizeof(nm), "WN.%d.in_layers.%d", k, i);
      if (int r = effective(sd, n_tensors, nm, 2 * C, (long long)C * ks, w_in, s)) return r;
      const float* b_in;
      snprintf(nm, sizeof(nm), "WN.%d.in_layers.%d.bias", k, i); if (int r = need(sd, n_tensors, nm, 2 * C, &b_in)) return r;
      k_w1<<<dim3((d.K1 + 127) / 128, 2 * C), 128, 0, s>>>(w_in, c2, b_in, cb2, C, ks, H, i, p_w1, idx * 2 * C * d.K1,
                                                         (float*)w.b1 + idx * 2 * C);
      if (i == 0 && w.w0_hi) {
        Planes p0 = p_w1;
        p0.hi = (uint16_t*)w.w0_hi; p0.lo = (uint16_t*)w.w0_lo; p0.f32 = nullptr;
        k_w0<<<2 * C, 64, 0, s>>>(w_in, w_start, b_start, C, ks, n_half, p0, (size_t)k * 2 * C * 48);
      }
      const int rs_rows = last ? C : 2 * C;
      snprintf(nm, sizeof(nm), "WN.%d.res_skip_layers.%d", k, i);
      if (int r = effective(sd, n_tensors, nm, rs_rows, C, w_rs, s)) return r;
      snprintf(nm, sizeof(nm), "WN.%d.res_skip_layers.%d.bias", k, i); if (int r = need(sd, n_tensors, nm, rs_rows, &ea.b_rs[i])) return r;
      if (rezero) { snprintf(nm, sizeof(nm), "WN.%d.alpha_i.%d", k, i); if (int r = need(sd, n_tensors, nm, 1, &ea.alpha[i])) return r; }
      k_w2<<<dim3((C + 127) / 128, d.N2), 128, 0, s>>>(w_rs, w_end, ea.b_rs[i], ea.alpha[i], C, n2h, last ? 1 : 0, p_w2,
                                                     idx * d.N2 * C, (float*)w.b2 + idx * C);
    }
    k_eo_b<<<1, 32, 0, s>>>(w_end, b_end, ea, C, L, n2h, d.MG, (float*)w.eo_b + (size_t)k * d.MG);
    CWG_CHECK_CUDA(cudaGetLastError());
  }
  *out = w;
  return 0;
}

int cwg_pack_forward(const cwg_config* cfg, const cwg_tensor* sd, int n_tensors, float* w_fwd, double* logdet,
                     void* cuda_stream) {
  CWG_REQUIRE(cfg && sd && w_fwd && logdet, "cwg_pack_forward: NULL argument");
  CWG_REQUIRE(cfg->n_group % 2 == 0 && cfg->n_group >= 2 && cfg->n_group <= CWG_MAX_GROUP && cfg->n_flows >= 1 &&
              cfg->n_early_every >= 1, "bad configuration");
  const int F = cfg->n_flows, mg = CWG_GROUP_PAD(cfg->n_group);
  cudaStream_t s = (cudaStream_t)cuda_stream;
  char nm[160];
  for (int k = 0; k < F; ++k) {
    int n_rem, n_half;
    flow_channels(cfg, k, &n_rem, &n_half);
    const float* Wm;
    snprintf(nm, sizeof(nm), "convinv.%d.conv.weight", k); if (int r = need(sd, n_tensors, nm, (long long)n_rem * n_rem, &Wm)) return r;
    k_wfwd<<<1, 32, 0, s>>>(Wm, n_rem, mg, k, F, w_fwd + (size_t)k * mg * mg, logdet);
  }
  CWG_CHECK_CUDA(cudaGetLastError());
  return 0;
}

int cwg_cond_bias(const cwg_config* cfg, const cwg_weights* w, const int64_t* speaker_ids, int batch, float* cond_bias,
                  void* cuda_stream) {
  CWG_REQUIRE(cfg && w && cond_bias && batch >= 1, "cwg_cond_bias: bad arguments");
  CWG_REQUIRE(w->cond_b_base != nullptr, "cwg_cond_bias: weights were not produced by cwg_pack_weights (cond_b_base is NULL)");
  const int E = w->speaker_embed_dim;
  if (E > 0) CWG_REQUIRE(speaker_ids && w->cond_w_spk && w->spk_embed && w->n_speakers > 0,
                         "this model has speaker embeddings: speaker_ids (one per utterance) is required");
  const int H = cfg->cond_hidden, F = cfg->n_flows;
  k_cond_bias<<<dim3((H + 127) / 128, F, batch), 128, 0, (cudaStream_t)cuda_stream>>>(
      w->cond_b_base, w->cond_w_spk, w->spk_embed, (const long long*)speaker_ids, F, H, E, w->n_speakers, cond_bias);
  CWG_CHECK_CUDA(cudaGetLastError());
  return 0;
}

}  // extern "C"
