// extern "C" entry points of libcwg (see include/cwg.h): argument checks, workspace carving and
// the launch sequence of WaveGlow.infer (glow.py:314-350).  No allocation, no host sync.
#include "cwg_common.cuh"

#include <stdarg.h>
#include <stdlib.h>
#include <string.h>

namespace cwg {

static thread_local char g_err[512] = "";

void set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}

static thread_local int* g_range_flag = nullptr;
static thread_local bool g_range_all = false;
int* range_flag() { return g_range_flag; }
void set_range_flag(int* flag) { g_range_flag = flag; }
bool range_all_layers() { return g_range_all; }
void set_range_all_layers(bool on) { g_range_all = on; }

namespace {

struct Workspace {
  int* status;            // first word of the workspace: see cwg_infer in cwg.h
  // FFMA mode
  float *x[2], *h2, *pre, *acts;
  // tensor-core modes (each: hi plane then lo plane)
  __nv_bfloat16 *xb[2], *h2b, *mel4, *actsb;
  void* a0;               // layer-0 fold: planes hi, lo [BT][16] 16-bit
  float* eo;
  size_t bytes;
};

int check_config(const cwg_config* c) {
  CWG_REQUIRE(c != nullptr, "cfg is NULL");
  CWG_REQUIRE(c->n_group % 2 == 0 && c->n_group >= 2 && c->n_group <= CWG_MAX_GROUP,
              "n_group must be even and <= %d", CWG_MAX_GROUP);
  CWG_REQUIRE(c->hop_length > 0 && c->hop_length % c->n_group == 0, "hop_length must be a multiple of n_group");
  CWG_REQUIRE(c->win_length >= c->hop_length, "win_length < hop_length");
  CWG_REQUIRE(c->kernel_size % 2 == 1, "kernel_size must be odd");
  CWG_REQUIRE(c->n_flows >= 1 && c->n_layers >= 1 && c->n_layers <= 16, "bad n_flows / n_layers");
  CWG_REQUIRE(c->n_channels >= 2 && c->n_channels % 2 == 0 && c->n_mel >= 1 && c->cond_hidden >= 1, "bad channel counts");
  CWG_REQUIRE(c->n_early_every >= 1 && c->n_early_size % 2 == 0, "bad early-output settings");
  int n_rem, n_half;
  flow_channels(c, c->n_flows - 1, &n_rem, &n_half);
  CWG_REQUIRE(n_half >= 1, "too many early outputs for n_group");
  return 0;
}

int check_mode(const cwg_config* c, int mode, bool cond_gemm = true) {
  CWG_REQUIRE(mode == CWG_MODE_FFMA || mode == CWG_MODE_BF16X3 || mode == CWG_MODE_BF16 || mode == CWG_MODE_F16F8,
              "unknown mode %d", mode);
  if (mode == CWG_MODE_F16F8)
    CWG_REQUIRE(c->n_channels == 256, "CWG_MODE_F16F8 is built for the 256-channel layer kernel");
  if (mode != CWG_MODE_FFMA && c->n_group > 16)
    CWG_REQUIRE(c->n_channels == 256, "n_group > 16 runs in CWG_MODE_FFMA or, for n_channels = 256, in the tensor-core modes");
  if (mode != CWG_MODE_FFMA) {
    CWG_REQUIRE((c->n_channels == 256 || c->n_channels == 512) && c->cond_hidden == 256 && c->kernel_size == 3,
                "tensor-core modes are built for n_channels in {256, 512}, cond_hidden=256, kernel_size=3 "
                "(got %d, %d, %d); use CWG_MODE_FFMA", c->n_channels, c->cond_hidden, c->kernel_size);
    (void)cond_gemm;   // the cond GEMM's K = n_mel * ceil(win/hop) is zero-padded to a multiple of 64
  }
  return 0;
}

void carve(const Dims& d, int mode, void* base, Workspace* ws) {
  size_t off = 0;
  auto take = [&](size_t bytes) { size_t o = off; off = align_up(off + bytes, 1024); return (char*)base + o; };
  memset(ws, 0, sizeof(*ws));
  ws->status = (int*)take(1024);
  ws->eo = (float*)take((size_t)d.BT * d.MG * sizeof(float));
  if (mode == CWG_MODE_FFMA) {
    ws->x[0] = (float*)take((size_t)d.BT * d.C * 4);
    ws->x[1] = (float*)take((size_t)d.BT * d.C * 4);
    ws->h2 = (float*)take((size_t)d.BT * d.H * 4);
    ws->pre = (float*)take((size_t)d.BT * 2 * d.C * 4);
    ws->acts = (float*)take((size_t)d.BT * d.C * 4);
  } else {
    const size_t xe = mode == CWG_MODE_F16F8 ? 6 : 4;       // bytes per element of the x planes (see cwg.h)
    ws->xb[0] = (__nv_bfloat16*)take((size_t)d.BT * d.C * xe);
    ws->xb[1] = (__nv_bfloat16*)take((size_t)d.BT * d.C * xe);
    ws->h2b = (__nv_bfloat16*)take((size_t)d.BT * d.H * 2 * 2);
    ws->mel4 = (__nv_bfloat16*)take((size_t)d.B * d.Tm * d.KCp * 2 * 2);
    if (d.C == 512) ws->actsb = (__nv_bfloat16*)take((size_t)d.BT * d.C * 2 * 2);   // gated activations (two-kernel layer)
    ws->a0 = take((size_t)d.BT * 16 * 2 * 2);
  }
  ws->bytes = off;
}

// tensor-core modes: is layer 0 run from the (audio_0 | 1) planes instead of a materialised x_0 (the start conv folded
// into in_layers.0)?
bool fold_active(const Dims& d, const cwg_weights* w) {
  return d.C == 256 && d.L >= 2 && d.MG == 16 && w->w0_hi && w->w0_lo;
}

int layer_tc(const cwg_config* cfg, const Dims& d, const cwg_weights* w, int npass, int k, int i, const Workspace& ws,
             const float* audio, cudaStream_t s, const int* rag_len = nullptr, const int* rag_prefix = nullptr) {
  if (d.C == 512)
    return launch_layer_tc512(d, w, npass, k, i, ws.xb[i & 1], ws.xb[(i + 1) & 1], ws.h2b, ws.actsb, ws.eo, s);
  if (i == 0 && audio && fold_active(d, w)) {
    int n_rem, n_half;
    flow_channels(cfg, k, &n_rem, &n_half);
    return launch_layer_ps(d, w, npass, k, i, ws.xb[0], ws.xb[1], ws.h2b, ws.eo, s, ws.a0, audio, d.G - n_rem, n_half,
                           rag_len, rag_prefix);
  }
  return launch_layer_ps(d, w, npass, k, i, ws.xb[i & 1], ws.xb[(i + 1) & 1], ws.h2b, ws.eo, s, nullptr, nullptr, 0, 0,
                         rag_len, rag_prefix);
}

// ---- ragged calls (cwg_infer_ragged) ----
// pairs of 128-step tiles an utterance of `frames` mel frames runs per WN layer
__host__ __device__ inline int ragged_pairs_of(int frames, int P) { return ((frames * P + 127) / 128 + 1) / 2; }

int check_ragged(const cwg_config* cfg, int mode, int batch) {
  CWG_REQUIRE(mode != CWG_MODE_FFMA && cfg->n_channels == 256,
              "ragged batches need the 256-channel persistent layer kernel in a tensor-core mode (f16f8, bf16x3, bf16); "
              "the 512-channel kernel pair and CWG_MODE_FFMA have no ragged form");
  CWG_REQUIRE(batch <= CWG_RAGGED_MAX_BATCH, "ragged batches hold at most %d utterances (got %d); split the batch",
              CWG_RAGGED_MAX_BATCH, batch);
  return 0;
}

// Workspace of a ragged call: cwg_infer's, then len [B] (clamped frames) and the tile-pair prefix sums [B + 1]
size_t ragged_plan_offset(const Dims& d, int mode) {
  Workspace ws;
  carve(d, mode, nullptr, &ws);
  return ws.bytes;
}
size_t ragged_plan_bytes(int batch) { return align_up((size_t)(2 * batch + 1) * sizeof(int), 1024); }

// one block: clamp the lengths into [1, Tm] (status bit 2 on a clamp) and scan the utterances' tile pairs
__global__ void k_ragged_plan(const int32_t* __restrict__ lengths, int B, int Tm, int P, int* __restrict__ len,
                              int* __restrict__ prefix, int* __restrict__ status) {
  __shared__ int pairs[CWG_RAGGED_MAX_BATCH];
  for (int b = threadIdx.x; b < B; b += blockDim.x) {
    int l = lengths[b];
    if (l < 1 || l > Tm) { atomicOr(status, 4); l = l < 1 ? 1 : Tm; }
    len[b] = l;
    pairs[b] = ragged_pairs_of(l, P);
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    int acc = 0;
    for (int b = 0; b < B; ++b) { prefix[b] = acc; acc += pairs[b]; }
    prefix[B] = acc;
  }
}

int check_run(const cwg_config* cfg, const cwg_weights* w, int mode, int batch, int t_mel) {
  if (int r = check_config(cfg)) return r;
  if (int r = check_mode(cfg, mode)) return r;
  CWG_REQUIRE(w != nullptr, "weights is NULL");
  CWG_REQUIRE(batch >= 1 && t_mel >= 1, "batch and t_mel must be >= 1");
  CWG_REQUIRE((long long)batch * t_mel * (cfg->hop_length / cfg->n_group) < (1ll << 31) / 4,
              "batch * T' too large for one call; split the batch");
  CWG_REQUIRE(w->b1 && w->b2 && w->eo_b && w->start_w && w->start_b && w->winv, "missing weight arrays");
  if (mode == CWG_MODE_FFMA) CWG_REQUIRE(w->cond_w_f32 && w->w1_f32 && w->w2_f32, "fp32 weight planes missing");
  else if (mode == CWG_MODE_F16F8)
    CWG_REQUIRE(w->cond_w_hi && w->cond_w_lo && w->w1_hi && w->w1_h8 && w->w1_l8 && w->w2_hi && w->w2_h8 && w->w2_l8,
                "fp16 / e5m2 weight planes missing");
  else CWG_REQUIRE(w->cond_w_hi && w->w1_hi && w->w2_hi && w->cond_w_lo && w->w1_lo && w->w2_lo,
                   "bf16 hi/lo weight planes missing");
  return 0;
}


// b1_batch[b][fl][n] = b1[fl][n] + <spk_w[fl][n][:], spk_embed[f][id_b][:]>  (glow_ax.py:378-381 folded into the gate bias)
__global__ void k_ax_speaker_bias(const float* __restrict__ b1, const float* __restrict__ spk_w,
                                  const float* __restrict__ spk_embed, const int64_t* __restrict__ ids, int E, int S,
                                  int L, int N, int FL, float* __restrict__ out) {
  extern __shared__ float emb_s[];
  const int fl = blockIdx.x, b = blockIdx.y, f = fl / L;
  long long id = ids[b];
  id = id < 0 ? 0 : (id >= S ? S - 1 : id);          // cwg_ax_speaker_bias rejects out-of-range ids on the host side
  for (int e = threadIdx.x; e < E; e += blockDim.x) emb_s[e] = spk_embed[((size_t)f * S + id) * E + e];
  __syncthreads();
  for (int n = threadIdx.x; n < N; n += blockDim.x) {
    const float* wr = spk_w + ((size_t)fl * N + n) * E;
    float acc = 0.f;
    for (int e = 0; e < E; ++e) acc = fmaf(__ldg(wr + e), emb_s[e], acc);
    out[((size_t)b * FL + fl) * N + n] = b1[(size_t)fl * N + n] + acc;
  }
}
}  // namespace
}  // namespace cwg

using namespace cwg;

extern "C" {

int cwg_abi_version(void) { return CWG_ABI_VERSION; }

// Debug only (not in cwg.h): the persistent layer kernel writes {start, end, tiles, -} clock64 stamps per CTA (4 x int64
// each) into `buf`.
void cwg_debug_set_ps_timing(void* buf) { cwg::debug_set_ps_timing((long long*)buf); }

// Debug only: layer 0 of `flow` through the layer-0 fold (a0 planes built from `audio`, then the fused persistent kernel);
// x_out / eo as in cwg_wn_layer.  a0_scratch: >= batch*T'*64 bytes.
int cwg_debug_layer0_fused(const cwg_config* cfg, const cwg_weights* w, int mode, int flow, float* audio, void* x_out,
                           const void* h2, float* eo, void* a0_scratch, int batch, int t_mel, void* cuda_stream) {
  if (int r = check_run(cfg, w, mode, batch, t_mel)) return r;
  CWG_REQUIRE(mode != CWG_MODE_FFMA && cfg->n_channels == 256 && w->w0_hi && w->w0_lo, "layer-0 fold not available for this model / mode");
  Dims d = make_dims(cfg, batch, t_mel);
  cudaStream_t s = (cudaStream_t)cuda_stream;
  if (int r = launch_flow_boundary(cfg, d, w, mode_xfmt(mode), -1, flow, nullptr, 1.f, audio, nullptr, x_out, s, -2, 0, a0_scratch)) return r;
  int n_rem, n_half;
  flow_channels(cfg, flow, &n_rem, &n_half);
  return launch_layer_ps(d, w, mode_npass(mode), flow, 0, (const __nv_bfloat16*)x_out, (__nv_bfloat16*)x_out, (const __nv_bfloat16*)h2, eo, s,
                         a0_scratch, audio, d.G - n_rem, n_half);
}

const char* cwg_last_error(void) { return cwg::g_err; }

size_t cwg_workspace_bytes(const cwg_config* cfg, int mode, int batch, int t_mel) {
  if (check_config(cfg) || check_mode(cfg, mode) || batch < 1 || t_mel < 1) return 0;
  if ((long long)batch * t_mel * (cfg->hop_length / cfg->n_group) >= (1ll << 31) / 4) {
    set_error("batch * T' too large for one call; split the batch");
    return 0;
  }
  Dims d = make_dims(cfg, batch, t_mel);
  Workspace ws;
  carve(d, mode, nullptr, &ws);
  return ws.bytes + 1024;
}

int cwg_launch_count(const cwg_config* cfg, int mode) {
  if (check_config(cfg) || check_mode(cfg, mode)) return -1;
  // per flow: cond (+ mel4 build in tensor modes), L layers, one boundary; plus the initial boundary
  int per_layer = mode == CWG_MODE_FFMA ? 3 : (cfg->n_channels == 512 ? 2 : 1);
  int cond = mode == CWG_MODE_FFMA ? 1 : 1;
  int once = mode == CWG_MODE_FFMA ? 1 : 2;   // init boundary (+ mel4 im2col)
  if (mode == CWG_MODE_F16F8) once += 1;   // non-finite scan of the waveform (range guard)
  return once + cfg->n_flows * (cond + per_layer * cfg->n_layers + 1);
}

int cwg_cond(const cwg_config* cfg, const cwg_weights* w, int mode, int flow,
             const float* mel, const float* cond_bias, void* h2_out,
             void* workspace, size_t workspace_bytes, int batch, int t_mel, void* cuda_stream) {
  if (int r = check_run(cfg, w, mode, batch, t_mel)) return r;
  CWG_REQUIRE(flow >= 0 && flow < cfg->n_flows, "flow out of range");
  Dims d = make_dims(cfg, batch, t_mel);
  cudaStream_t s = (cudaStream_t)cuda_stream;
  if (mode == CWG_MODE_FFMA) return launch_cond_ffma(d, w, flow, mel, cond_bias, (float*)h2_out, s);
  Workspace ws;
  CWG_REQUIRE(workspace != nullptr && ((uintptr_t)workspace % 1024) == 0, "workspace must be 1024-byte aligned");
  carve(d, mode, workspace, &ws);
  CWG_REQUIRE(ws.bytes <= workspace_bytes, "workspace too small: need %zu, got %zu", ws.bytes, workspace_bytes);
  return launch_cond_tc(d, w, mode_npass(mode), flow, mel, cond_bias,
                        (__nv_bfloat16*)h2_out, ws.mel4, s);
}

int cwg_wn_layer(const cwg_config* cfg, const cwg_weights* w, int mode, int flow, int layer,
                 const void* x_in, void* x_out, const void* h2, float* eo,
                 void* workspace, size_t workspace_bytes, int batch, int t_mel, void* cuda_stream) {
  if (int r = check_run(cfg, w, mode, batch, t_mel)) return r;
  CWG_REQUIRE(flow >= 0 && flow < cfg->n_flows && layer >= 0 && layer < cfg->n_layers, "flow/layer out of range");
  Dims d = make_dims(cfg, batch, t_mel);
  cudaStream_t s = (cudaStream_t)cuda_stream;
  if (mode == CWG_MODE_FFMA) {
    Workspace ws;
    CWG_REQUIRE(workspace != nullptr && ((uintptr_t)workspace % 1024) == 0, "workspace must be 1024-byte aligned");
    carve(d, mode, workspace, &ws);
    CWG_REQUIRE(ws.bytes <= workspace_bytes, "workspace too small: need %zu, got %zu", ws.bytes, workspace_bytes);
    return launch_layer_ffma(d, w, flow, layer, (const float*)x_in, (float*)x_out, (const float*)h2, eo,
                             ws.pre, ws.acts, s);
  }
  if (d.C == 512) {
    Workspace ws;
    CWG_REQUIRE(workspace != nullptr && ((uintptr_t)workspace % 1024) == 0, "workspace must be 1024-byte aligned");
    carve(d, mode, workspace, &ws);
    CWG_REQUIRE(ws.bytes <= workspace_bytes, "workspace too small: need %zu, got %zu", ws.bytes, workspace_bytes);
    return launch_layer_tc512(d, w, mode_npass(mode), flow, layer, (const __nv_bfloat16*)x_in,
                              (__nv_bfloat16*)x_out, (const __nv_bfloat16*)h2, ws.actsb, eo, s);
  }
  return launch_layer_ps(d, w, mode_npass(mode), flow, layer, (const __nv_bfloat16*)x_in,
                         (__nv_bfloat16*)x_out, (const __nv_bfloat16*)h2, eo, s);
}

int cwg_flow_boundary(const cwg_config* cfg, const cwg_weights* w, int mode,
                      int flow_done, int flow_next, const float* z, float sigma,
                      float* audio, const float* eo, void* x_out,
                      int batch, int t_mel, void* cuda_stream) {
  if (int r = check_run(cfg, w, mode, batch, t_mel)) return r;
  CWG_REQUIRE(flow_done < cfg->n_flows && flow_next < cfg->n_flows, "flow out of range");
  Dims d = make_dims(cfg, batch, t_mel);
  return launch_flow_boundary(cfg, d, w, mode_xfmt(mode), flow_done, flow_next, z, sigma,
                              audio, eo, x_out, (cudaStream_t)cuda_stream);
}

int cwg_infer_status(const void* workspace, int32_t* status, void* cuda_stream) {
  CWG_REQUIRE(workspace && status, "cwg_infer_status: NULL argument");
  CWG_CHECK_CUDA(cudaMemcpyAsync(status, workspace, sizeof(int32_t), cudaMemcpyDeviceToDevice, (cudaStream_t)cuda_stream));
  return 0;
}

int cwg_nonfinite(const float* x, size_t n, int32_t* flag, void* cuda_stream) {
  CWG_REQUIRE(x && flag, "cwg_nonfinite: NULL argument");
  return launch_nonfinite(x, n, (int*)flag, (cudaStream_t)cuda_stream, true);
}

int cwg_infer(const cwg_config* cfg, const cwg_weights* w, int mode,
              const float* mel, const float* cond_bias, const float* z, float sigma,
              float* audio, void* workspace, size_t workspace_bytes,
              int batch, int t_mel, void* cuda_stream) {
  return cwg_infer_profiled(cfg, w, mode, mel, cond_bias, z, sigma, audio, workspace, workspace_bytes,
                            batch, t_mel, cuda_stream, nullptr, nullptr, 0);
}

int cwg_infer_profiled(const cwg_config* cfg, const cwg_weights* w, int mode,
                       const float* mel, const float* cond_bias, const float* z, float sigma,
                       float* audio, void* workspace, size_t workspace_bytes,
                       int batch, int t_mel, void* cuda_stream,
                       void** layer_ev_begin, void** layer_ev_end, int n_events) {
  if (int r = check_run(cfg, w, mode, batch, t_mel)) return r;
  CWG_REQUIRE(n_events == 0 || (layer_ev_begin && layer_ev_end), "event arrays are NULL");
  CWG_REQUIRE(mel && cond_bias && z && audio, "NULL tensor argument");
  CWG_REQUIRE(workspace != nullptr && ((uintptr_t)workspace % 1024) == 0, "workspace must be 1024-byte aligned");
  Dims d = make_dims(cfg, batch, t_mel);
  Workspace ws;
  carve(d, mode, workspace, &ws);
  CWG_REQUIRE(ws.bytes <= workspace_bytes, "workspace too small: need %zu, got %zu", ws.bytes, workspace_bytes);
  cudaStream_t s = (cudaStream_t)cuda_stream;
  const bool tc = mode != CWG_MODE_FFMA;
  const int npass = mode_npass(mode);
  const int xfmt = mode_xfmt(mode);
  const int F = cfg->n_flows, L = cfg->n_layers;

  // status word (first 4 bytes of the workspace): bit 1 (2) = an fp16 plane of CWG_MODE_F16F8 left the fp16 range,
  // bit 0 (1) = the waveform holds a NaN / Inf.  Zero in the other modes.
  CWG_CHECK_CUDA(cudaMemsetAsync(ws.status, 0, sizeof(int), s));
  set_range_flag(mode == CWG_MODE_F16F8 ? ws.status : nullptr);
  auto run = [&]() -> int {
  // audio = sigma * z (glow.py:326; early z already sits in its final columns), x = start_{F-1}(audio_0)
  void* x0 = tc ? (void*)ws.xb[0] : (void*)ws.x[0];
  void* a0 = (tc && fold_active(d, w)) ? ws.a0 : nullptr;
  if (int r = launch_flow_boundary(cfg, d, w, xfmt, -1, F - 1, z, sigma, audio, nullptr, x0, s, -2, 0, a0)) return r;
  for (int k = F - 1; k >= 0; --k) {                       // glow.py:328
    if (tc) {
      if (int r = launch_cond_tc(d, w, npass, k, k == F - 1 ? mel : nullptr, cond_bias, ws.h2b, ws.mel4, s)) return r;
    } else {
      if (int r = launch_cond_ffma(d, w, k, mel, cond_bias, ws.h2, s)) return r;
    }
    for (int i = 0; i < L; ++i) {                          // glow.py:201-220
      const int ev = (F - 1 - k) * L + i;
      if (ev < n_events) CWG_CHECK_CUDA(cudaEventRecord((cudaEvent_t)layer_ev_begin[ev], s));
      if (tc) {
        if (int r = layer_tc(cfg, d, w, npass, k, i, ws, audio, s)) return r;
      } else {
        if (int r = launch_layer_ffma(d, w, k, i, ws.x[i & 1], ws.x[(i + 1) & 1], ws.h2, ws.eo, ws.pre, ws.acts, s)) return r;
      }
      if (ev < n_events) CWG_CHECK_CUDA(cudaEventRecord((cudaEvent_t)layer_ev_end[ev], s));
    }
    // coupling inverse + W^-1 of flow k, then start conv of flow k-1 (glow.py:329-347, :189)
    if (int r = launch_flow_boundary(cfg, d, w, xfmt, k, k - 1, nullptr, sigma, audio, ws.eo, x0, s, -2, 0, a0)) return r;
  }
  return 0;
  };
  const int rc = run();
  set_range_flag(nullptr);
  if (rc) return rc;
  if (mode == CWG_MODE_F16F8) return launch_nonfinite(audio, (size_t)batch * t_mel * cfg->hop_length, ws.status, s, false);
  return 0;
}

// ---------------------------------------------------------------------------------------------
// Ragged batches: cwg_infer's launch sequence with per-utterance lengths.  Zero invariant: throughout the call every row
// t >= T'_b of the audio state, of eo, of both x buffers (all planes) and of the layer-0-fold planes is 0, so that a
// dilated tap of a valid row reads the zero padding a call for utterance b alone would see, and nothing of the padding
// (z, mel, stale workspace) can reach a valid row, the range flag or the waveform.  It is established once here (eo, x,
// z -> audio); the layers keep it (k_layer_ps<..., RAGGED>), padded audio stays 0 through the boundaries (eo = 0 there:
// (0 - 0) * exp(-0)), and the start-conv rows the boundaries write into the padding are zeroed after each of them.
// ---------------------------------------------------------------------------------------------
size_t cwg_ragged_workspace_bytes(const cwg_config* cfg, int mode, int batch, int t_mel) {
  if (check_config(cfg) || check_mode(cfg, mode) || check_ragged(cfg, mode, batch)) return 0;
  const size_t base = cwg_workspace_bytes(cfg, mode, batch, t_mel);
  if (base == 0) return 0;
  return ragged_plan_offset(make_dims(cfg, batch, t_mel), mode) + ragged_plan_bytes(batch) + 1024;
}

int cwg_ragged_pairs(const cwg_config* cfg, const int32_t* lengths, int batch, int t_mel, int32_t* prefix) {
  if (check_config(cfg)) return -1;
  if (!lengths || batch < 1 || t_mel < 1) { set_error("cwg_ragged_pairs: NULL lengths or batch / t_mel < 1"); return -1; }
  const int P = cfg->hop_length / cfg->n_group;
  if ((long long)t_mel * P >= (1ll << 31) / 4) { set_error("cwg_ragged_pairs: t_mel too large"); return -1; }
  long long acc = 0;
  for (int b = 0; b < batch; ++b) {
    if (lengths[b] < 1 || lengths[b] > t_mel) {
      set_error("lengths[%d] = %d is outside [1, t_mel = %d]", b, (int)lengths[b], t_mel);
      return -1;
    }
    if (prefix) prefix[b] = (int32_t)acc;
    acc += ragged_pairs_of(lengths[b], P);
  }
  if (acc >= (1ll << 31)) { set_error("cwg_ragged_pairs: too many tile pairs"); return -1; }
  if (prefix) prefix[batch] = (int32_t)acc;
  return (int)acc;
}

int cwg_infer_ragged(const cwg_config* cfg, const cwg_weights* w, int mode,
                     const float* mel, const float* cond_bias, const float* z, float sigma, const int32_t* lengths,
                     float* audio, void* workspace, size_t workspace_bytes,
                     int batch, int t_mel, void* cuda_stream) {
  if (int r = check_run(cfg, w, mode, batch, t_mel)) return r;
  if (int r = check_ragged(cfg, mode, batch)) return r;
  CWG_REQUIRE(mel && cond_bias && z && audio && lengths, "NULL tensor argument");
  CWG_REQUIRE(workspace != nullptr && ((uintptr_t)workspace % 1024) == 0, "workspace must be 1024-byte aligned");
  Dims d = make_dims(cfg, batch, t_mel);
  Workspace ws;
  carve(d, mode, workspace, &ws);
  CWG_REQUIRE(ws.bytes + ragged_plan_bytes(batch) <= workspace_bytes, "workspace too small: need %zu, got %zu",
              ws.bytes + ragged_plan_bytes(batch), workspace_bytes);
  int* len = (int*)((char*)workspace + ws.bytes);
  int* prefix = len + batch;
  cudaStream_t s = (cudaStream_t)cuda_stream;
  const int npass = mode_npass(mode), xfmt = mode_xfmt(mode);
  const int F = cfg->n_flows, L = cfg->n_layers;
  void* a0 = fold_active(d, w) ? ws.a0 : nullptr;
  const size_t plane = (size_t)d.BT * d.C;

  CWG_CHECK_CUDA(cudaMemsetAsync(ws.status, 0, sizeof(int), s));       // status word as in cwg_infer, + bit 2
  set_range_flag(mode == CWG_MODE_F16F8 ? ws.status : nullptr);
  // padded rows of the start-conv output the boundaries write: x_0 (or the layer-0-fold planes, constant-1 channel
  // included) must read as the conv's zero padding
  auto clear_x = [&](void* x) -> int {
    if (int r = launch_ragged_rows(x, nullptr, plane * 2, 2, d.B, d.Tp, d.C / 2, len, d.P, s)) return r;   // 16-bit hi, lo
    if (mode == CWG_MODE_F16F8)                                                                             // e5m2 planes
      return launch_ragged_rows((char*)x + 4 * plane, nullptr, plane, 2, d.B, d.Tp, d.C / 4, len, d.P, s);
    return 0;
  };
  auto clear_start = [&]() -> int {
    return a0 ? launch_ragged_rows(a0, nullptr, (size_t)d.BT * 32, 2, d.B, d.Tp, 8, len, d.P, s) : clear_x(ws.xb[0]);
  };
  auto run = [&]() -> int {
  k_ragged_plan<<<1, 1024, 0, s>>>(lengths, batch, t_mel, d.P, len, prefix, ws.status);
  CWG_CHECK_CUDA(cudaGetLastError());
  if (int r = launch_ragged_rows(ws.eo, nullptr, 0, 1, d.B, d.Tp, d.MG, len, d.P, s)) return r;
  if (int r = clear_x(ws.xb[0])) return r;
  if (int r = clear_x(ws.xb[1])) return r;
  // audio = z with the padding zeroed; the first boundary then scales it in place (audio = sigma * audio)
  if (int r = launch_ragged_rows(audio, z, 0, 1, d.B, d.Tp, d.G, len, d.P, s)) return r;
  if (int r = launch_flow_boundary(cfg, d, w, xfmt, -1, F - 1, audio, sigma, audio, nullptr, ws.xb[0], s, -2, 0, a0)) return r;
  if (int r = clear_start()) return r;
  for (int k = F - 1; k >= 0; --k) {
    if (int r = launch_cond_tc(d, w, npass, k, k == F - 1 ? mel : nullptr, cond_bias, ws.h2b, ws.mel4, s, len)) return r;
    for (int i = 0; i < L; ++i)
      if (int r = layer_tc(cfg, d, w, npass, k, i, ws, audio, s, len, prefix)) return r;
    if (int r = launch_flow_boundary(cfg, d, w, xfmt, k, k - 1, nullptr, sigma, audio, ws.eo, ws.xb[0], s, -2, 0, a0)) return r;
    if (k > 0)
      if (int r = clear_start()) return r;
  }
  return 0;
  };
  const int rc = run();
  set_range_flag(nullptr);
  if (rc) return rc;
  if (mode == CWG_MODE_F16F8) return launch_nonfinite(audio, (size_t)batch * t_mel * cfg->hop_length, ws.status, s, false);
  return 0;
}

// ---------------------------------------------------------------------------------------------
// Forward direction (audio -> z, log_s, log det W): NVIDIA's WaveGlow.forward, of which glow.py is derived.  Flows run
// k = 0 .. F-1; flow k mixes with W_k, runs WN_k on audio_0 and applies audio_1 = exp(log_s) * audio_1 + b.  The WN work
// is the launch sequence of cwg_infer; the flow boundaries are cwg_forward.cu's.
// ---------------------------------------------------------------------------------------------
namespace {
struct FwdLayout {
  Dims d;           // layer dims: T' = t_samples / n_group per utterance (Tm = tf, the frames the cond GEMM runs on)
  Dims dc;          // cond GEMM dims: tf = ceil(t_samples / hop) frames, tf * P group-steps per utterance
  size_t ls_part, z2_part, cond, mel, bytes;   // byte offsets of the extra regions (cond / mel: 0 = not needed)
};

int fwd_check(const cwg_config* cfg, int mode, int batch, int t_mel, int t_samples) {
  if (int r = check_config(cfg)) return r;
  if (int r = check_mode(cfg, mode)) return r;
  CWG_REQUIRE(batch >= 1 && t_mel >= 1, "batch and t_mel must be >= 1");
  CWG_REQUIRE(t_samples >= cfg->n_group && t_samples % cfg->n_group == 0,
              "t_samples must be a positive multiple of n_group = %d (got %d)", cfg->n_group, t_samples);
  CWG_REQUIRE((long long)t_samples <= (long long)t_mel * cfg->hop_length,
              "t_samples = %d exceeds t_mel * hop_length = %lld: the upsampled mel must cover the audio", t_samples,
              (long long)t_mel * cfg->hop_length);
  CWG_REQUIRE((long long)batch * ((t_samples + cfg->hop_length - 1) / cfg->hop_length) * (cfg->hop_length / cfg->n_group) <
              (1ll << 31) / 4, "batch * T' too large for one call; split the batch");
  return 0;
}

FwdLayout fwd_layout(const cwg_config* cfg, int mode, int batch, int t_mel, int t_samples) {
  FwdLayout l;
  const int tf = (t_samples + cfg->hop_length - 1) / cfg->hop_length;
  l.dc = make_dims(cfg, batch, tf);
  l.d = l.dc;
  l.d.Tp = t_samples / cfg->n_group;
  l.d.BT = (long long)batch * l.d.Tp;
  Workspace ws;
  carve(l.d, mode, nullptr, &ws);
  size_t off = ws.bytes;
  auto take = [&](size_t bytes) { size_t o = off; off = align_up(off + bytes, 1024); return o; };
  const size_t nblk = (size_t)fwd_blocks(l.d);
  l.ls_part = take((size_t)l.d.F * batch * nblk * sizeof(double));
  l.z2_part = take((size_t)batch * nblk * sizeof(double));
  l.cond = l.dc.Tp != l.d.Tp ? take((size_t)l.dc.BT * l.d.H * 4) : 0;     // every cond format is 4 bytes per element
  l.mel = t_mel != tf ? take((size_t)batch * l.d.M * tf * sizeof(float)) : 0;
  l.bytes = off;
  return l;
}
}  // namespace

size_t cwg_forward_workspace_bytes(const cwg_config* cfg, int mode, int batch, int t_mel, int t_samples) {
  if (fwd_check(cfg, mode, batch, t_mel, t_samples)) return 0;
  return fwd_layout(cfg, mode, batch, t_mel, t_samples).bytes + 1024;
}

int cwg_forward_launch_count(const cwg_config* cfg, int mode) {
  const int n = cwg_launch_count(cfg, mode);
  return n < 0 ? n : n + 1;       // the inverse pass's sequence (one boundary per flow plus one) + the final reduction
}

int cwg_forward(const cwg_config* cfg, const cwg_weights* w, const float* w_fwd, const double* logdet, int mode,
                const float* mel, const float* cond_bias, const float* audio, int t_samples,
                float* z, float* log_s, double* logp_terms,
                void* workspace, size_t workspace_bytes, int batch, int t_mel, void* cuda_stream) {
  if (int r = fwd_check(cfg, mode, batch, t_mel, t_samples)) return r;
  if (int r = check_run(cfg, w, mode, batch, (t_samples + cfg->hop_length - 1) / cfg->hop_length)) return r;
  CWG_REQUIRE(w_fwd && logdet && mel && cond_bias && audio && z && logp_terms, "NULL tensor argument");
  CWG_REQUIRE(workspace != nullptr && ((uintptr_t)workspace % 1024) == 0, "workspace must be 1024-byte aligned");
  const FwdLayout l = fwd_layout(cfg, mode, batch, t_mel, t_samples);
  CWG_REQUIRE(l.bytes <= workspace_bytes, "workspace too small: need %zu, got %zu", l.bytes, workspace_bytes);
  const Dims& d = l.d;
  Workspace ws;
  carve(d, mode, workspace, &ws);
  char* base = (char*)workspace;
  double* ls_part = (double*)(base + l.ls_part);
  double* z2_part = (double*)(base + l.z2_part);
  cudaStream_t s = (cudaStream_t)cuda_stream;
  const bool tc = mode != CWG_MODE_FFMA;
  const int npass = mode_npass(mode), xfmt = mode_xfmt(mode);
  const int F = cfg->n_flows, L = cfg->n_layers, tf = l.dc.Tm;
  const size_t nblk = (size_t)fwd_blocks(d);

  CWG_CHECK_CUDA(cudaMemsetAsync(ws.status, 0, sizeof(int), s));     // status word as in cwg_infer (cwg_infer_status)
  set_range_flag(mode == CWG_MODE_F16F8 ? ws.status : nullptr);
  auto run = [&]() -> int {
  // the cond GEMM reads [B][n_mel][tf]: a longer mel is cut to the tf frames the audio needs (ConvTranspose1d is causal
  // in frames: sample o depends on frames <= o / hop only)
  const float* melc = mel;
  if (l.mel) {
    melc = (const float*)(base + l.mel);
    CWG_CHECK_CUDA(cudaMemcpy2DAsync((void*)melc, (size_t)tf * 4, mel, (size_t)t_mel * 4, (size_t)tf * 4,
                                     (size_t)batch * d.M, cudaMemcpyDeviceToDevice, s));
  }
  void* h2 = tc ? (void*)ws.h2b : (void*)ws.h2;
  void* h2c = l.cond ? (void*)(base + l.cond) : h2;       // T % hop != 0: cond of tf * P steps, compacted to T' below
  // One fp32 plane of one utterance already holds its first T' rows in place; every other layout needs the compaction
  // (the offsets of the lo / e5m2 planes and of utterance b > 0 depend on the row count)
  const bool compact = l.cond && (tc || batch > 1);
  const float* h2f = compact ? ws.h2 : (const float*)h2c;  // cond rows of the fp32 layers
  void* x0 = tc ? (void*)ws.xb[0] : (void*)ws.x[0];
  void* a0 = (tc && fold_active(d, w)) ? ws.a0 : nullptr;
  // z = audio, then W_0 and the start conv of flow 0
  if (int r = launch_fwd_boundary(cfg, d, w, w_fwd, xfmt, -1, 0, audio, z, nullptr, nullptr, nullptr, nullptr, x0, a0, s)) return r;
  size_t ls_off = 0;
  for (int k = 0; k < F; ++k) {
    if (tc) {
      if (int r = launch_cond_tc(l.dc, w, npass, k, k == 0 ? melc : nullptr, cond_bias, (__nv_bfloat16*)h2c, ws.mel4, s)) return r;
    } else {
      if (int r = launch_cond_ffma(l.dc, w, k, melc, cond_bias, (float*)h2c, s)) return r;
    }
    if (compact) {
      // per plane: the first T' of the tf * P rows of every utterance (planes: fp32 | bf16 hi, lo | fp16, e5m2, e5m2)
      const int ne[3] = {xfmt == 0 ? 4 : 2, xfmt == 0 ? 0 : (xfmt == 1 ? 2 : 1), xfmt == 2 ? 1 : 0};
      size_t so = 0, dof = 0;
      for (int q = 0; q < 3 && ne[q]; ++q) {
        const size_t row = (size_t)d.H * ne[q];
        CWG_CHECK_CUDA(cudaMemcpy2DAsync((char*)h2 + dof, (size_t)d.Tp * row, (const char*)h2c + so, (size_t)l.dc.Tp * row,
                                         (size_t)d.Tp * row, (size_t)batch, cudaMemcpyDeviceToDevice, s));
        so += (size_t)l.dc.BT * row;
        dof += (size_t)d.BT * row;
      }
    }
    for (int i = 0; i < L; ++i) {
      if (tc) {
        if (int r = layer_tc(cfg, d, w, npass, k, i, ws, z, s)) return r;
      } else {
        if (int r = launch_layer_ffma(d, w, k, i, ws.x[i & 1], ws.x[(i + 1) & 1], h2f, ws.eo, ws.pre, ws.acts, s)) return r;
      }
    }
    int n_rem, n_half;
    flow_channels(cfg, k, &n_rem, &n_half);
    float* ls_k = log_s ? log_s + ls_off : nullptr;
    ls_off += (size_t)batch * n_half * d.Tp;
    // coupling of flow k, then W_{k+1} and the start conv of flow k+1 (the last boundary reduces z^2 instead)
    if (int r = launch_fwd_boundary(cfg, d, w, w_fwd, xfmt, k, k + 1 < F ? k + 1 : -1, nullptr, z, ws.eo, ls_k,
                                    ls_part + (size_t)k * batch * nblk, z2_part, x0, a0, s)) return r;
  }
  return launch_fwd_reduce(d, ls_part, z2_part, logdet + F, logp_terms, s);
  };
  const int rc = run();
  set_range_flag(nullptr);
  if (rc) return rc;
  if (mode == CWG_MODE_F16F8) return launch_nonfinite(z, (size_t)batch * t_samples, ws.status, s, false);
  return 0;
}

// ---------------------------------------------------------------------------------------------
// ax WaveGlow (waveflow=False): efficient_model_ax.py:279-357 with AffineCouplingBlock.inverse
// (efficient_modules.py:94-105), glow_ax.WN.forward (:375-418), InvertibleConv1x1.inverse (:269-286)
// or PermuteHeight as the channel mixing (packed as a permutation matrix in `winv`).
// Same layer / boundary kernels as the classic model; the cond vector is the interpolated mel
// (channels padded to cfg->cond_hidden) and the WN's single 1x1 cond layer rides in w1's K columns.
// ---------------------------------------------------------------------------------------------
namespace {
Dims ax_dims(const cwg_config* cfg, int batch, int frames, int t_samples) {
  Dims d = make_dims(cfg, batch, frames);
  d.Tp = t_samples / cfg->n_group;
  d.BT = (long long)batch * d.Tp;
  return d;
}
int ax_check(const cwg_config* cfg, int mode, int batch, int frames, int t_samples) {
  if (int r = check_config(cfg)) return r;
  if (int r = check_mode(cfg, mode, false)) return r;
  CWG_REQUIRE(batch >= 1 && frames >= 1 && t_samples >= cfg->n_group && t_samples % cfg->n_group == 0,
              "t_samples must be a positive multiple of n_group");
  CWG_REQUIRE(cfg->n_mel <= cfg->cond_hidden, "n_mel must be <= cond_hidden (the padded cond width)");
  return 0;
}
}  // namespace

size_t cwg_ax_workspace_bytes(const cwg_config* cfg, int mode, int batch, int frames, int t_samples) {
  if (ax_check(cfg, mode, batch, frames, t_samples)) return 0;
  Dims d = ax_dims(cfg, batch, frames, t_samples);
  Workspace ws;
  carve(d, mode, nullptr, &ws);
  return ws.bytes + 1024;
}

int cwg_ax_infer(const cwg_config* cfg, const cwg_weights* w, int mode,
                 const float* mel, int frames, int pad_frames, int upsample_linear, int mix_first,
                 const float* z, float sigma, float* audio, void* workspace, size_t workspace_bytes,
                 int batch, int t_samples, const float* b1_batch, void* cuda_stream) {
  if (int r = ax_check(cfg, mode, batch, frames, t_samples)) return r;
  CWG_REQUIRE(w && w->b1 && w->b2 && w->eo_b && w->start_w && w->start_b && w->winv, "missing weight arrays");
  if (mode == CWG_MODE_FFMA) CWG_REQUIRE(w->w1_f32 && w->w2_f32, "fp32 weight planes missing");
  else if (mode == CWG_MODE_F16F8) CWG_REQUIRE(w->w1_hi && w->w1_h8 && w->w1_l8 && w->w2_hi && w->w2_h8 && w->w2_l8, "fp16 / e5m2 weight planes missing");
  else CWG_REQUIRE(w->w1_hi && w->w2_hi && w->w1_lo && w->w2_lo, "bf16 hi/lo weight planes missing");
  CWG_REQUIRE(mel && z && audio && pad_frames >= 0, "bad tensor arguments");
  CWG_REQUIRE(workspace != nullptr && ((uintptr_t)workspace % 1024) == 0, "workspace must be 1024-byte aligned");
  Dims d = ax_dims(cfg, batch, frames, t_samples);
  d.b1_batch = b1_batch;             // per-utterance gate bias (WN-level speaker embedding, cwg_ax_speaker_bias) or NULL
  Workspace ws;
  carve(d, mode, workspace, &ws);
  CWG_REQUIRE(ws.bytes <= workspace_bytes, "workspace too small: need %zu, got %zu", ws.bytes, workspace_bytes);
  cudaStream_t s = (cudaStream_t)cuda_stream;
  const bool tc = mode != CWG_MODE_FFMA;
  const int npass = mode_npass(mode);
  const int xfmt = mode_xfmt(mode);
  const int F = cfg->n_flows, L = cfg->n_layers;
  void* x0 = tc ? (void*)ws.xb[0] : (void*)ws.x[0];
  void* h2 = tc ? (void*)ws.h2b : (void*)ws.h2;
  // status word as in cwg_infer (cwg_infer_status): the fp16 planes of CWG_MODE_F16F8 are range-checked
  CWG_CHECK_CUDA(cudaMemsetAsync(ws.status, 0, sizeof(int), s));
  set_range_flag(mode == CWG_MODE_F16F8 ? ws.status : nullptr);
  auto run = [&]() -> int {
  // cond = interpolate(mel) once for all flows (upsample_first), efficient_model_ax.py:313-314
  if (int r = launch_mel_up(xfmt, mel, h2, d.B, d.M, frames, frames + pad_frames, d.Tp, d.H, upsample_linear, s)) return r;
  // z -> audio state; mix_first=False applies the channel mixing of flow F-1 before its coupling
  void* a0 = (tc && fold_active(d, w)) ? ws.a0 : nullptr;       // layer-0 fold, as in cwg_infer
  if (int r = launch_flow_boundary(cfg, d, w, xfmt, -1, F - 1, z, sigma, audio, nullptr, x0, s, mix_first ? -1 : F - 1, 0, a0)) return r;
  for (int k = F - 1; k >= 0; --k) {                       // efficient_model_ax.py:325
    for (int i = 0; i < L; ++i) {
      if (tc) {
        if (int r = layer_tc(cfg, d, w, npass, k, i, ws, audio, s)) return r;
      } else {
        if (int r = launch_layer_ffma(d, w, k, i, ws.x[i & 1], ws.x[(i + 1) & 1], ws.h2, ws.eo, ws.pre, ws.acts, s)) return r;
      }
    }
    // coupling inverse of flow k, then (mix_first) mixing of flow k or (else) mixing of flow k-1
    // after the early-z concat, then the start conv of flow k-1
    if (int r = launch_flow_boundary(cfg, d, w, xfmt, k, k - 1, nullptr, sigma, audio, ws.eo, x0, s,
                                     mix_first ? k : k - 1, /*ignore_nan=*/1, a0)) return r;
  }
  return 0;
  };
  set_range_all_layers(true);      // ignore_nan flushes NaNs at every flow boundary: no overflow may rely on reaching the waveform
  const int rc = run();
  set_range_all_layers(false);
  set_range_flag(nullptr);
  if (rc) return rc;
  if (mode == CWG_MODE_F16F8) return launch_nonfinite(audio, (size_t)batch * t_samples, ws.status, s, false);
  return 0;
}

// Forward direction of the ax model (audio -> z): flows k = 0 .. F-1, each on the trailing n_rem_k columns (early
// outputs stay where they are).  mix_first: W_k, WN_k + coupling;  else: WN_k + coupling, W_k.  In flow k the WN sees
// audio_0 and the cond of the inverse, so the layer launches are cwg_ax_infer's; only the boundaries differ.
namespace {
struct AxFwdLayout {
  Dims d;
  size_t ls_part, z2_part, bytes;
};

AxFwdLayout ax_fwd_layout(const cwg_config* cfg, int mode, int batch, int frames, int t_samples) {
  AxFwdLayout l;
  l.d = ax_dims(cfg, batch, frames, t_samples);
  Workspace ws;
  carve(l.d, mode, nullptr, &ws);
  size_t off = ws.bytes;
  auto take = [&](size_t bytes) { size_t o = off; off = align_up(off + bytes, 1024); return o; };
  const size_t nblk = (size_t)fwd_blocks(l.d);
  l.ls_part = take((size_t)l.d.F * batch * nblk * sizeof(double));
  l.z2_part = take((size_t)batch * nblk * sizeof(double));
  l.bytes = off;
  return l;
}
}  // namespace

size_t cwg_ax_forward_workspace_bytes(const cwg_config* cfg, int mode, int batch, int frames, int t_samples) {
  if (ax_check(cfg, mode, batch, frames, t_samples)) return 0;
  return ax_fwd_layout(cfg, mode, batch, frames, t_samples).bytes + 1024;
}

int cwg_ax_forward_launch_count(const cwg_config* cfg, int mode) {
  if (check_config(cfg) || check_mode(cfg, mode, false)) return -1;
  const int per_layer = mode == CWG_MODE_FFMA ? 3 : (cfg->n_channels == 512 ? 2 : 1);
  // cond interpolation, first boundary, per flow L layers and a boundary, the reduction (+ the non-finite scan of z)
  return 3 + (mode == CWG_MODE_F16F8 ? 1 : 0) + cfg->n_flows * (per_layer * cfg->n_layers + 1);
}

int cwg_ax_forward(const cwg_config* cfg, const cwg_weights* w, const float* w_fwd, const double* logabsdet, int mode,
                   const float* mel, int frames, int upsample_linear, int mix_first, const float* audio, int t_samples,
                   float* z, double* logp_terms, void* workspace, size_t workspace_bytes, int batch,
                   const float* b1_batch, void* cuda_stream) {
  if (int r = ax_check(cfg, mode, batch, frames, t_samples)) return r;
  CWG_REQUIRE(w && w->b1 && w->b2 && w->eo_b && w->start_w && w->start_b, "missing weight arrays");
  if (mode == CWG_MODE_FFMA) CWG_REQUIRE(w->w1_f32 && w->w2_f32, "fp32 weight planes missing");
  else if (mode == CWG_MODE_F16F8) CWG_REQUIRE(w->w1_hi && w->w1_h8 && w->w1_l8 && w->w2_hi && w->w2_h8 && w->w2_l8, "fp16 / e5m2 weight planes missing");
  else CWG_REQUIRE(w->w1_hi && w->w2_hi && w->w1_lo && w->w2_lo, "bf16 hi/lo weight planes missing");
  CWG_REQUIRE(w_fwd && logabsdet && mel && audio && z && logp_terms, "NULL tensor argument");
  CWG_REQUIRE(workspace != nullptr && ((uintptr_t)workspace % 1024) == 0, "workspace must be 1024-byte aligned");
  const AxFwdLayout l = ax_fwd_layout(cfg, mode, batch, frames, t_samples);
  CWG_REQUIRE(l.bytes <= workspace_bytes, "workspace too small: need %zu, got %zu", l.bytes, workspace_bytes);
  Dims d = l.d;
  d.b1_batch = b1_batch;             // per-utterance gate bias (cwg_ax_speaker_bias) or NULL
  Workspace ws;
  carve(d, mode, workspace, &ws);
  double* ls_part = (double*)((char*)workspace + l.ls_part);
  double* z2_part = (double*)((char*)workspace + l.z2_part);
  cudaStream_t s = (cudaStream_t)cuda_stream;
  const bool tc = mode != CWG_MODE_FFMA;
  const int npass = mode_npass(mode), xfmt = mode_xfmt(mode);
  const int F = cfg->n_flows, L = cfg->n_layers;
  const size_t nblk = (size_t)fwd_blocks(d);
  void* x0 = tc ? (void*)ws.xb[0] : (void*)ws.x[0];
  void* h2 = tc ? (void*)ws.h2b : (void*)ws.h2;
  void* a0 = (tc && fold_active(d, w)) ? ws.a0 : nullptr;
  CWG_CHECK_CUDA(cudaMemsetAsync(ws.status, 0, sizeof(int), s));     // status word as in cwg_forward
  set_range_flag(mode == CWG_MODE_F16F8 ? ws.status : nullptr);
  auto run = [&]() -> int {
  if (int r = launch_mel_up(xfmt, mel, h2, d.B, d.M, frames, frames, d.Tp, d.H, upsample_linear, s)) return r;
  // z = audio, then (mix_first) W_0 and the start conv of flow 0
  if (int r = launch_fwd_boundary(cfg, d, w, w_fwd, xfmt, -1, 0, audio, z, nullptr, nullptr, nullptr, nullptr, x0, a0, s,
                                  mix_first ? -2 : -1)) return r;
  for (int k = 0; k < F; ++k) {
    for (int i = 0; i < L; ++i) {
      if (tc) {
        if (int r = layer_tc(cfg, d, w, npass, k, i, ws, z, s)) return r;
      } else {
        if (int r = launch_layer_ffma(d, w, k, i, ws.x[i & 1], ws.x[(i + 1) & 1], ws.h2, ws.eo, ws.pre, ws.acts, s)) return r;
      }
    }
    // coupling of flow k, then W_k (mix last) or W_{k+1} (mix first), then the start conv of flow k+1 (last: z^2)
    if (int r = launch_fwd_boundary(cfg, d, w, w_fwd, xfmt, k, k + 1 < F ? k + 1 : -1, nullptr, z, ws.eo, nullptr,
                                    ls_part + (size_t)k * batch * nblk, z2_part, x0, a0, s, mix_first ? -2 : k)) return r;
  }
  return launch_fwd_reduce(d, ls_part, z2_part, logabsdet, logp_terms, s);
  };
  const int rc = run();
  set_range_flag(nullptr);
  if (rc) return rc;
  if (mode == CWG_MODE_F16F8) return launch_nonfinite(z, (size_t)batch * t_samples, ws.status, s, false);
  return 0;
}

int cwg_ax_speaker_bias(const cwg_config* cfg, const float* b1, const float* spk_w, const float* spk_embed,
                        int speaker_embed_dim, int n_speakers, const int64_t* speaker_ids, int batch,
                        float* b1_batch, void* cuda_stream) {
  if (int r = check_config(cfg)) return r;
  CWG_REQUIRE(b1 && spk_w && spk_embed && speaker_ids && b1_batch, "cwg_ax_speaker_bias: NULL argument");
  CWG_REQUIRE(speaker_embed_dim >= 1 && speaker_embed_dim <= 4096 && n_speakers >= 1 && batch >= 1, "cwg_ax_speaker_bias: bad sizes");
  const int FL = cfg->n_flows * cfg->n_layers, N = 2 * cfg->n_channels;
  k_ax_speaker_bias<<<dim3(FL, batch), 256, speaker_embed_dim * sizeof(float), (cudaStream_t)cuda_stream>>>(
      b1, spk_w, spk_embed, speaker_ids, speaker_embed_dim, n_speakers, cfg->n_layers, N, FL, b1_batch);
  CWG_CHECK_CUDA(cudaGetLastError());
  return 0;
}

}  // extern "C"
