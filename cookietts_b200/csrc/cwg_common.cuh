// Shared declarations for the cwg (CookieTTS WaveGlow, B200) kernels.
#pragma once

#include <cuda_runtime.h>
#include <cuda_bf16.h>
#include <stdint.h>
#include <stdio.h>

#include "../../include/cwg.h"

namespace cwg {

// Derived problem dimensions (all in elements).
struct Dims {
  int B, Tm, Tp;        // batch, mel frames, group-steps T' = Tm * P
  int F, L, C, H;       // flows, WN layers, WN channels, cond hidden
  int G, M, P, J, ks;   // n_group, n_mel, phases hop/G, upsampler taps, WN kernel size
  int K1, N2, KC, KCp;  // ks*C + H, C + MG, J*M, J*M padded to a multiple of 64 (cond_w row pitch)
  int MG;               // group padding CWG_GROUP_PAD(G): 16, or 32 for 16 < n_group <= 32 (include/cwg.h)
  long long BT;         // B * Tp
  const float* b1_batch;   // per-utterance gate bias [B][F][L][2C] (ax WN-level speaker embedding) or NULL: w->b1
};

inline Dims make_dims(const cwg_config* c, int batch, int t_mel) {
  Dims d;
  d.B = batch; d.Tm = t_mel;
  d.F = c->n_flows; d.L = c->n_layers; d.C = c->n_channels; d.H = c->cond_hidden;
  d.G = c->n_group; d.M = c->n_mel; d.P = c->hop_length / c->n_group;
  d.J = (c->win_length + c->hop_length - 1) / c->hop_length; d.ks = c->kernel_size;
  d.Tp = t_mel * d.P;
  d.MG = CWG_GROUP_PAD(c->n_group); d.b1_batch = nullptr;
  d.K1 = d.ks * d.C + d.H; d.N2 = d.C + d.MG; d.KC = d.J * d.M; d.KCp = (d.KC + 63) / 64 * 64;
  d.BT = (long long)batch * d.Tp;
  return d;
}

// (n_remaining_channels, n_half) of flow k; glow.py:251-264.
inline void flow_channels(const cwg_config* c, int k, int* n_rem, int* n_half) {
  int nh = c->n_group / 2, nr = c->n_group;
  for (int j = 1; j <= k; ++j)
    if (j % c->n_early_every == 0) { nh -= c->n_early_size / 2; nr -= c->n_early_size; }
  *n_rem = nr; *n_half = nh;
}

void set_error(const char* fmt, ...);

#define CWG_CHECK_CUDA(expr)                                                              \
  do {                                                                                    \
    cudaError_t _e = (expr);                                                              \
    if (_e != cudaSuccess) {                                                              \
      cwg::set_error("%s failed: %s (%s:%d)", #expr, cudaGetErrorString(_e), __FILE__, __LINE__); \
      return 1;                                                                           \
    }                                                                                     \
  } while (0)

#define CWG_REQUIRE(cond, ...)                  \
  do {                                          \
    if (!(cond)) { cwg::set_error(__VA_ARGS__); return 2; } \
  } while (0)

static inline size_t align_up(size_t x, size_t a) { return (x + a - 1) / a * a; }

// The gated units of glow_ax.py:36-166 on the two halves (a, b) of the pre-activation (gate = CWG_GATE_*).  The SIREN
// variants scale the first half by 16 in place before the sine (:113,:131,:140,:149); rrelu in eval mode is
// leaky_relu((lower + upper) / 2).
#ifdef __CUDACC__
__device__ __forceinline__ float gated_unit(int gate, float a, float b) {
  float fa, fb;
  switch (gate) {
    case CWG_GATE_GLU: fa = a; break;
    case CWG_GATE_GTSU: case CWG_GATE_GTSRU: fa = a - tanhf(a); break;
    case CWG_GATE_GSIU: fa = sinf(a); break;
    case CWG_GATE_GSIRU: case CWG_GATE_GSIRRU: case CWG_GATE_GSIRLRU: case CWG_GATE_GSIRRLRU: fa = sinf(16.f * a); break;
    default: fa = tanhf(a);
  }
  switch (gate) {
    case CWG_GATE_GTRU: case CWG_GATE_GTSRU: case CWG_GATE_GSIRRU: fb = fmaxf(b, 0.f); break;
    case CWG_GATE_GTLRU: case CWG_GATE_GSIRLRU: fb = b > 0.f ? b : 0.01f * b; break;
    case CWG_GATE_GSIRRLRU: fb = b > 0.f ? b : 0.055f * b; break;
    case CWG_GATE_TTU: fb = tanhf(b); break;
    case CWG_GATE_STU: fb = 1.0507009873554804934f * (b > 0.f ? b : 1.6732632423543772848f * expm1f(b)); break;
    case CWG_GATE_SPTU: fb = b > 20.f ? b : log1pf(expf(b)); break;
    default: fb = 1.f / (1.f + expf(-b));
  }
  return fa * fb;
}
#endif

// CWG_MODE_F16F8 scaling of the e5m2 correction operands (cookietts_b200/packing.py F8_P, F8_Q)
constexpr float F8_LO_SCALE = 64.f;            // 2^P applied to activation lo parts (weights hi carry 2^-P)
constexpr float F8_HI_SCALE = 1.f / 256.f;     // 2^-Q applied to activation hi parts (weights lo carry 2^Q)
// npass argument of the tensor-core launchers: 1 = bf16, 3 = bf16x3, 2 = f16f8
inline int mode_npass(int mode) { return mode == CWG_MODE_BF16X3 ? 3 : (mode == CWG_MODE_F16F8 ? 2 : 1); }
inline int mode_xfmt(int mode) { return mode == CWG_MODE_FFMA ? 0 : (mode == CWG_MODE_F16F8 ? 2 : 1); }

// ---- launchers implemented in cwg_simple.cu (CUDA-core fp32 path + shared boundary kernels) ----
int launch_cond_ffma(const Dims& d, const cwg_weights* w, int flow, const float* mel,
                     const float* cond_bias, float* h2, cudaStream_t s);
int launch_layer_ffma(const Dims& d, const cwg_weights* w, int flow, int layer, const float* x_in,
                      float* x_out, const float* h2, float* eo, float* pre, float* acts, cudaStream_t s);
// xfmt: 0 = fp32 [BT][C]; 1 = bf16 hi plane followed by lo plane (each [BT][C]); 2 = CWG_MODE_F16F8 planes
// (fp16 hi, fp16 lo, e5m2(lo * 2^F8_P), e5m2(hi * 2^-F8_Q))
int launch_flow_boundary(const cwg_config* cfg, const Dims& d, const cwg_weights* w, int xfmt,
                         int flow_done, int flow_next, const float* z, float sigma, float* audio,
                         const float* eo, void* x_out, cudaStream_t s, int mix_flow = -2, int ignore_nan = 0,
                         void* a0_out = nullptr);   // a0_out: write the layer-0-fold planes [BT][16] hi, lo instead of x

// CWG_MODE_F16F8 range guard: device status word the producers of fp16 planes OR bit 1 (value 2) into when a value leaves
// +-65504 (set by cwg_infer around its launches; NULL = no check).  Host-side, thread-local.
int* range_flag();
void set_range_flag(int* flag);
// ax models flush NaNs at flow boundaries (ignore_nan), so there every residual layer checks its x_new, not only the last
bool range_all_layers();
void set_range_all_layers(bool on);

int launch_nonfinite(const float* x, size_t n, int* flag, cudaStream_t s, bool clear);

// Ragged calls: n_planes planes of [B][T] rows of row_words 4-byte words, plane_bytes apart.  Row t of utterance b is
// valid when t < len[b] * mult: valid rows are copied from src (src == NULL: left as they are), the others set to 0.
int launch_ragged_rows(void* dst, const void* src, size_t plane_bytes, int n_planes, int B, int T, int row_words,
                       const int* len, int mult, cudaStream_t s);

int launch_mel_up(int xfmt, const float* mel, void* out, int B, int M, int frames, int frames_padded, int Tp, int H,
                  int linear, cudaStream_t s);

// ---- forward direction (audio -> z), cwg_forward.cu ----
// One launch per flow boundary: coupling of flow_done (-1: none; audio_in != NULL copies the waveform in first), log_s
// store (log_s may be NULL), per-block sums of log_s into ls_part [B][fwd_blocks], then W of flow_next and its start conv
// into x_out (or the layer-0 fold planes into a0_out).  flow_next = -1 ends the pass: per-block sums of z^2 into z2_part.
// mix_flow: -2 = W of flow_next before its start conv (mix first); otherwise W of flow mix_flow over its n_rem right after
// the coupling, and none before the start conv (mix last; -1 = no mixing in this launch).
int fwd_blocks(const Dims& d);
int launch_fwd_boundary(const cwg_config* cfg, const Dims& d, const cwg_weights* w, const float* w_fwd, int xfmt,
                        int flow_done, int flow_next, const float* audio_in, float* audio, const float* eo, float* log_s,
                        double* ls_part, double* z2_part, void* x_out, void* a0_out, cudaStream_t s, int mix_flow = -2);
// terms [B][3] = {sum z^2, sum log_s, T' * sum_k log|det W_k|} from the partials (ls_part [F][B][fwd_blocks])
int launch_fwd_reduce(const Dims& d, const double* ls_part, const double* z2_part, const double* logabsdet, double* terms,
                      cudaStream_t s);
int launch_fwd_reduce(int F, int B, int nblk, int Tp, const double* ls_part, const double* z2_part, const double* logabsdet,
                      double* terms, cudaStream_t s);
// WaveFlow (cwg_wf_forward): one launch per flow boundary, k_wf_fwd_boundary in cwg_forward.cu.  phys_done: column map of
// the flow just run (NULL: first launch, which reads audio_in and zeroes ld_zero [F]); phys_next / start_*: the flow to
// prepare (NULL: last launch, z in logical order and z^2 partials).  Partials are [B][wf_fwd_blocks(Tp)].
int wf_fwd_blocks(int Tp);
int launch_wf_fwd_boundary(int B, int Tp, int G, int F, const float* audio_in, float* z, const float* eo,
                           const int* phys_done, const int* phys_next, const float* start_w, const float* start_b,
                           __nv_bfloat16* x0, long long xplane, double* ls_part, double* z2_part, double* ld_zero,
                           cudaStream_t s);

// ---- launchers implemented in cwg_tc.cu (tcgen05 / TMA path) ----
// mel_len != NULL (ragged calls): frames f >= mel_len[b] of the im2col matrix are zeroed before the GEMM, so the cond rows
// of the padding hold the bias alone - finite whatever the padded mel holds, and never tripping the f16f8 range check
int launch_cond_tc(const Dims& d, const cwg_weights* w, int npass, int flow, const float* mel,
                   const float* cond_bias, __nv_bfloat16* h2_planes, __nv_bfloat16* mel4_planes,
                   cudaStream_t s, const int* mel_len = nullptr);

// n_channels = 256: one persistent, epilogue-overlapped kernel per WN layer (cwg_ps.cu)
int launch_layer_ps(const Dims& d, const cwg_weights* w, int npass, int flow, int layer,
                    const __nv_bfloat16* x_in, __nv_bfloat16* x_out, const __nv_bfloat16* h2,
                    float* eo, cudaStream_t s, const void* a0 = nullptr, const float* audio = nullptr,
                    int a_off = 0, int a_nh = 0, const int* rag_len = nullptr, const int* rag_prefix = nullptr);
void debug_set_ps_timing(long long* buf);

// n_channels = 512: two kernels per layer (cwg_tc512.cu); `acts` = bf16 hi/lo planes [B*T'][512]
int launch_layer_tc512(const Dims& d, const cwg_weights* w, int npass, int flow, int layer,
                       const __nv_bfloat16* x_in, __nv_bfloat16* x_out, const __nv_bfloat16* h2,
                       __nv_bfloat16* acts, float* eo, cudaStream_t s);

// ---- fp32 CUDA-core WaveFlow path (cwg_wf_ffma.cu), dispatched by cwg_wf_* for CWG_MODE_FFMA ----
int wff_check(const cwg_wf_config* c, int batch, int t_samples);
size_t wff_workspace_bytes(const cwg_wf_config* c, int batch, int t_samples);
int wff_launch_count(const cwg_wf_config* c);
int wff_infer(const cwg_wf_config* cfg, const cwg_wf_weights* w, const float* mel, int frames, int pad_frames,
              const float* z, float sigma, float* audio, void* workspace, size_t workspace_bytes, int batch, int t_samples,
              cudaStream_t s, void** ev_begin, void** ev_end, int n_events);

}  // namespace cwg
