/* cwg.h - C ABI of the B200 (sm_100a) WaveGlow inverse pass.
 *
 * This is the drop-in boundary for the reference's mel->wave hot path
 *   CookieTTS/_4_mtw/waveglow/glow.py:314-350   WaveGlow.infer(spect, speaker_id, sigma)
 * and the functions it calls (WN.forward :188-222, Invertible1x1Conv.forward(reverse=True)
 * :85-99, fused_add_tanh_sigmoid_multiply :34-41).  The reference has no FFI of its own
 * (pure Python on torch); the bindings a maintainer adds are in INTEGRATION.md: the torch.ops shim
 * (cookietts_b200/csrc/torch_ops.cpp, what cookietts_b200.WaveGlow.infer calls) and the ctypes stub
 * (cookietts_b200/_cabi.py, what the stage-level tests call).
 *
 * Conventions
 *  - Every pointer in cwg_weights / cwg_infer is a DEVICE pointer owned by the caller.
 *    The library allocates nothing, keeps no mutable global state except the last error
 *    string (thread local), never synchronises the host, and enqueues all work on the
 *    stream it is given.
 *  - Return value: 0 on success, non-zero on error; cwg_last_error() describes it.
 *  - Layouts: mel [B, n_mel, T_mel] fp32 (the reference layout); z and audio [B, T] fp32 with
 *    T = T_mel*hop; latent channel c of group-step s is z[b, s*n_group + c], channels ordered
 *    as the reference stacks them at the end of infer (early outputs of the lowest flow
 *    first, the main latent last; glow.py:326,342-347).
 *  - Packed weights are produced by cwg_pack_weights below from the reference state_dict (weight-norm folded, the
 *    linear cond chain folded with the transposed-conv upsampler, `end` folded into the skip half of res_skip,
 *    `start` folded into in_layers.0; see DESIGN.md "Packed weights").  cookietts_b200/packing.py is the numpy
 *    statement of the same algebra that the tests hold it to (and that the ax / WaveFlow packers build on).
 */
#ifndef CWG_H
#define CWG_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define CWG_ABI_VERSION 5

/* Arithmetic modes of the WN contractions. */
#define CWG_MODE_FFMA   0   /* fp32 weights/activations, CUDA-core FFMA (exact fp32 semantics)        */
#define CWG_MODE_BF16X3 1   /* tcgen05 bf16 MMA, operands split hi+lo, 3 products, fp32 accumulate   */
#define CWG_MODE_BF16   2   /* tcgen05 bf16 MMA, single product, fp32 accumulate + hi/lo residual    */
#define CWG_MODE_F16F8  3   /* fp32-accurate at 2 MMA passes instead of 3 (256-channel classic model): operands split into
                               fp16 hi + lo; the in_layer GEMM issues hi*hi in fp16 and the two cross terms as e5m2 fp8
                               MMAs (twice the rate): a*w ~= a16*w16 + e5m2(a_lo*2^6)*e5m2(w16*2^-6) + e5m2(a16*2^-8)*e5m2(w_lo*2^8);
                               the res/skip GEMM likewise, the small cond GEMM uses three fp16 products                                */

#define CWG_EO_PAD 16       /* padded width of the folded `end` output for n_group <= 16 (2*n_half <= 16) */
#define CWG_MAX_GROUP 32    /* n_group <= 32                                                         */
/* ABI 4: group padding MG of the arrays indexed by latent channels.  n_group <= 16 keeps the round-1 layout (MG = 16);
 * 16 < n_group <= 32 (the ax notebook model: n_group 24) doubles it.  start_w is [F][C][MG/2], winv [F][MG][MG], the
 * folded `end` output (eo, eo_b, the last rows of w2) is MG wide and N2 = C + MG.  The wide layout runs in CWG_MODE_FFMA
 * and, for n_channels = 256, in the tensor-core modes (cwg_ps.cu; layer 0 unfolded). */
#define CWG_GROUP_PAD(n_group) ((n_group) <= 16 ? 16 : 32)

/* Mirrors the constructor arguments of the reference WaveGlow (glow.py:226-227) and
 * WN_config (glow.py:116-117) that the inverse pass depends on. */
typedef struct cwg_config {
  int32_t n_mel;          /* n_mel_channels                                   */
  int32_t n_flows;
  int32_t n_group;
  int32_t n_early_every;
  int32_t n_early_size;
  int32_t win_length;     /* ConvTranspose1d kernel                           */
  int32_t hop_length;     /* ConvTranspose1d stride                           */
  int32_t n_layers;       /* WN layers L                                      */
  int32_t n_channels;     /* WN channels C                                    */
  int32_t kernel_size;    /* WN dilated conv taps (odd)                       */
  int32_t cond_hidden;    /* H: width of the folded cond chain output (256)   */
} cwg_config;

/* Device pointers to the packed weights.  F = n_flows, L = n_layers, C = n_channels,
 * H = cond_hidden, P = hop/n_group, J = ceil(win/hop), M = n_mel, K1 = kernel_size*C + H,
 * N2 = C + MG, MG = CWG_GROUP_PAD(n_group).  fp32 arrays are used by CWG_MODE_FFMA, the bf16 hi/lo planes by the
 * tensor-core modes (lo = bf16(w - float(hi))); unused ones may be NULL. */
typedef struct cwg_weights {
  const float*    cond_w_f32;   /* [F][P*H][KCp]   row p*H+h, col j*M+ci; KCp = J*M rounded up to 64, zero padded */
  const uint16_t* cond_w_hi;    /* same, bf16                                          */
  const uint16_t* cond_w_lo;
  const float*    w1_f32;       /* [F][L][2C][K1]  col tap*C+c | kernel_size*C+h        */
  const uint16_t* w1_hi;
  const uint16_t* w1_lo;
  const float*    b1;           /* [F][L][2C]      in_layer bias + cond_layers.2 bias   */
  const float*    w2_f32;       /* [F][L][N2][C]   rows <C: res, rows >=C: end*skip     */
  const uint16_t* w2_hi;
  const uint16_t* w2_lo;
  const float*    b2;           /* [F][L][C]       res bias (0 for the last layer)      */
  const float*    eo_b;         /* [F][MG]         end bias + end*(sum of skip biases)  */
  const float*    start_w;      /* [F][C][MG/2]                                         */
  const float*    start_b;      /* [F][C]                                               */
  const float*    winv;         /* [F][MG][MG]     W^-1, row major                      */
  /* CWG_MODE_F16F8 only (there *_hi / *_lo are fp16 planes): e5m2 planes of w1, same shape as w1_hi */
  const uint8_t*  w1_h8;        /* e5m2(fp16(w1) * 2^-6)                                */
  const uint8_t*  w1_l8;        /* e5m2((w1 - fp16(w1)) * 2^8)                          */
  const uint8_t*  w2_h8;        /* the same two planes of w2 ([F][L][N2][C])            */
  const uint8_t*  w2_l8;
  /* ABI 3: what cwg_cond_bias needs (filled by cwg_pack_weights; NULL / 0 when the caller passes its own cond_bias) */
  const float*    cond_b_base;  /* [F][H]        bias of the folded cond chain without the speaker branch          */
  const float*    cond_w_spk;   /* [F][H][E]     speaker columns of cond_layers.1 * cond_layers.0 (glow.py:193-199) */
  const float*    spk_embed;    /* [F][S][E]     WN.k.speaker_embed.weight of every flow (glow.py:144-147)          */
  /* layer-0 fold (tensor-core modes, C = 256; optional - NULL selects the unfused layer 0): in_layers.0 * start per flow,
   * [F][2C][48] 16-bit planes (bf16, or fp16 in CWG_MODE_F16F8), col = tap*16 + j: j < n_half the coupling input
   * channels, j = n_half the start bias (contracted with a constant-1 channel), other columns zero */
  const uint16_t* w0_hi;
  const uint16_t* w0_lo;
  int32_t         speaker_embed_dim;   /* E (0: single-speaker model) */
  int32_t         n_speakers;          /* S: rows of the embedding tables */
} cwg_weights;

int         cwg_abi_version(void);
const char* cwg_last_error(void);

/* ---- checkpoint -> packed weights (replaces the per-forward weight handling of glow.py:136-186, 74-83, 238-241) ----
 * One entry of the reference checkpoint's state_dict: the parameter names of glow.py (SURVEY Appendix A), e.g.
 * "upsample.weight", "WN.3.in_layers.2.weight_g", "WN.3.in_layers.2.weight_v", "WN.3.cond_layers.0.bias",
 * "WN.3.end.weight", "convinv.3.conv.weight", "WN.3.speaker_embed.weight", "WN.3.alpha_i.2".  Weight-normed
 * (weight_g / weight_v) and plain (weight) layouts are both accepted, per tensor. */
typedef struct cwg_tensor {
  const char*  name;
  const float* data;        /* DEVICE pointer, fp32, contiguous in the torch layout */
  int32_t      ndim;
  int64_t      shape[4];
} cwg_tensor;

/* speaker_embed_dim / n_speakers (shape of WN.0.speaker_embed.weight, 0 if absent) and rezero (WN.0.alpha_i.0 present)
 * are properties of the checkpoint; any out pointer may be NULL. */
int cwg_state_dict_info(const cwg_tensor* sd, int n_tensors, int* speaker_embed_dim, int* n_speakers, int* rezero);

/* Bytes of the packed blob for (cfg, mode) and of the fp64 scratch cwg_pack_weights needs.  0 on error. */
size_t cwg_packed_bytes(const cwg_config* cfg, int mode, int speaker_embed_dim, int n_speakers);
size_t cwg_pack_workspace_bytes(const cwg_config* cfg, int speaker_embed_dim);

/* Folds the checkpoint into the arrays of cwg_weights, in fp64, on the device, on `cuda_stream`:
 * weight-norm folded; cond_layers[1]*cond_layers[0]*squeeze*ConvTranspose1d folded into cond_w; cond_layers[2] appended to
 * every in_layer's K; `end` folded into the skip rows of res_skip; ReZero alphas folded; W^-1 of every
 * Invertible1x1Conv.  `packed` (256-byte aligned, cwg_packed_bytes) receives the planes `mode` uses; *out points into it.
 * Only the planes of `mode` are written (BF16 and BF16X3 share theirs). */
int cwg_pack_weights(const cwg_config* cfg, int mode, const cwg_tensor* sd, int n_tensors,
                     void* packed, size_t packed_bytes, void* workspace, size_t workspace_bytes,
                     cwg_weights* out, void* cuda_stream);

/* Re-derives the cwg_weights pointers of a blob written by cwg_pack_weights (pure host arithmetic). */
int cwg_packed_view(const cwg_config* cfg, int mode, int speaker_embed_dim, int n_speakers,
                    void* packed, size_t packed_bytes, cwg_weights* out);

/* cond_bias [batch][F][H] for cwg_infer / cwg_cond: cond_b_base plus, for multispeaker checkpoints, the speaker-embedding
 * branch glow.py:193-196 (speaker_ids: DEVICE int64 [batch]; required when speaker_embed_dim > 0, else ignored). */
int cwg_cond_bias(const cwg_config* cfg, const cwg_weights* w, const int64_t* speaker_ids, int batch,
                  float* cond_bias, void* cuda_stream);

/* Bytes of device workspace cwg_infer needs for (batch, t_mel) in `mode`. 0 on error. */
size_t cwg_workspace_bytes(const cwg_config* cfg, int mode, int batch, int t_mel);

/* WaveGlow.infer with explicit latent (glow.py:314-350).
 *   mel        [batch][n_mel][t_mel] fp32
 *   cond_bias  [batch][F][H] fp32: folded cond-chain bias per utterance (carries the speaker
 *              embedding branch glow.py:193-196 when speaker_embed_dim > 0)
 *   z          [batch][t_mel*hop] fp32 standard normal
 *   audio      [batch][t_mel*hop] fp32 out
 * All work is enqueued on `cuda_stream` (a cudaStream_t). */
int cwg_infer(const cwg_config* cfg, const cwg_weights* w, int mode,
              const float* mel, const float* cond_bias, const float* z, float sigma,
              float* audio, void* workspace, size_t workspace_bytes,
              int batch, int t_mel, void* cuda_stream);

/* Same as cwg_infer; additionally records the CUDA events layer_ev_begin[e] / layer_ev_end[e]
 * (cudaEvent_t handles owned by the caller) on `cuda_stream` around the e-th WN-layer launch,
 * e = (n_flows-1-flow)*n_layers + layer, for e < n_events.  bench.py uses it to time the dominant
 * kernel inside the real step. */
int cwg_infer_profiled(const cwg_config* cfg, const cwg_weights* w, int mode,
                       const float* mel, const float* cond_bias, const float* z, float sigma,
                       float* audio, void* workspace, size_t workspace_bytes,
                       int batch, int t_mel, void* cuda_stream,
                       void** layer_ev_begin, void** layer_ev_end, int n_events);

/* Status word of the last cwg_infer / cwg_infer_profiled that used `workspace` (the first 4 bytes of the workspace, DEVICE
 * memory), copied to the DEVICE int32 *status on `cuda_stream`:  0 = fine;  bit 0 (1) = the waveform holds a NaN / Inf;
 * bit 1 (2) = CWG_MODE_F16F8 only: a value of an fp16 operand plane (cond hidden vector, `start` output, residual stream
 * entering the last layer) left +-65504, i.e. the result is not trustworthy - re-run in CWG_MODE_BF16X3 (fp32 range).
 * Other modes always report 0 (they have fp32's exponent range; use cwg_nonfinite for a NaN scan). */
int cwg_infer_status(const void* workspace, int32_t* status, void* cuda_stream);

/* Range guard of the fp16-based mode: *flag (DEVICE int32) = 1 when x[0..n) holds a NaN or Inf, else 0.  In CWG_MODE_F16F8
 * the residual stream and the cond hidden vector are stored as fp16 hi + lo planes: a value beyond +-65504 becomes Inf
 * there, turns into NaN in the next GEMM and reaches the waveform, so a finite waveform proves no overflow happened.
 * cookietts_b200.WaveGlow re-runs the call in CWG_MODE_BF16X3 (fp32 range) when the flag is set. */
int cwg_nonfinite(const float* x, size_t n, int32_t* flag, void* cuda_stream);

/* Number of kernels cwg_infer launches for this configuration (bench.py's gpu_launches). */
int cwg_launch_count(const cwg_config* cfg, int mode);

/* ---- ragged batches: per-utterance lengths ------------------------------------------------------------------------
 * cwg_infer_ragged is cwg_infer on a padded batch whose utterance b holds lengths[b] mel frames (1 <= lengths[b] <=
 * t_mel).  Utterance b is computed as if it were alone: audio[b][0 .. lengths[b]*hop) equals, byte for byte, what
 * cwg_infer returns for mel[b][:][0 .. lengths[b]) and z[b][0 .. lengths[b]*hop) in the same mode; audio[b][lengths[b]*hop
 * ..) is 0.  WN-layer tiles wholly past an utterance's end are not computed.  Tensor-core modes of the 256-channel layer
 * kernel only (CWG_MODE_F16F8, CWG_MODE_BF16X3, CWG_MODE_BF16); batch <= CWG_RAGGED_MAX_BATCH.
 *   lengths    DEVICE int32 [batch], mel frames per utterance.  The device checks them: a value outside [1, t_mel] is
 *              clamped into it and sets bit 2 (4) of the status word (cwg_infer_status), which otherwise works as for
 *              cwg_infer.  Check lengths on the host (cwg_ragged_pairs) to reject them before any work is enqueued.
 * The other arguments are cwg_infer's; the workspace size is cwg_ragged_workspace_bytes'. */
#define CWG_RAGGED_MAX_BATCH 1024
size_t cwg_ragged_workspace_bytes(const cwg_config* cfg, int mode, int batch, int t_mel);
int cwg_infer_ragged(const cwg_config* cfg, const cwg_weights* w, int mode,
                     const float* mel, const float* cond_bias, const float* z, float sigma, const int32_t* lengths,
                     float* audio, void* workspace, size_t workspace_bytes,
                     int batch, int t_mel, void* cuda_stream);
/* Host-side tile-pair plan of a ragged call (pure host arithmetic): utterance b runs ceil(ceil(T'_b / 128) / 2) pairs of
 * 128-step tiles per WN layer, T'_b = lengths[b] * hop / n_group.  lengths: HOST int32 [batch].  Writes the prefix sums
 * [batch + 1] to prefix (may be NULL) and returns their total (the pairs every WN layer launch computes), or -1 on bad
 * arguments (a length outside [1, t_mel] included; see cwg_last_error).  A padded call computes
 * batch * ceil(ceil(t_mel * hop / n_group / 128) / 2). */
int cwg_ragged_pairs(const cwg_config* cfg, const int32_t* lengths, int batch, int t_mel, int32_t* prefix);

/* ---- stage-level entry points (tests bisect the pipeline with these) ---------------- */

/* Folded cond chain for one flow: H2 [batch][T'][H] (fp32 in FFMA mode; bf16 hi/lo planes,
 * hi first then lo, each [batch][T'][H], in the bf16 modes; in CWG_MODE_F16F8 an fp16 plane followed by the two
 * e5m2 planes e5m2(lo * 2^6), e5m2(hi * 2^-8), 4 bytes per element in total). */
int cwg_cond(const cwg_config* cfg, const cwg_weights* w, int mode, int flow,
             const float* mel, const float* cond_bias, void* h2_out,
             void* workspace, size_t workspace_bytes, int batch, int t_mel, void* cuda_stream);

/* One WN layer: x_in -> x_out (fp32 [batch][T'][C] in FFMA mode; hi/lo bf16 planes in the bf16 modes; in
 * CWG_MODE_F16F8 fp16 hi, fp16 lo, e5m2(lo * 2^6), e5m2(hi * 2^-8) planes, 6 bytes per element),
 * eo [batch][T'][MG] fp32 accumulated (written when layer == 0). */
int cwg_wn_layer(const cwg_config* cfg, const cwg_weights* w, int mode, int flow, int layer,
                 const void* x_in, void* x_out, const void* h2, float* eo,
                 void* workspace, size_t workspace_bytes, int batch, int t_mel, void* cuda_stream);

/* Flow boundary: optional init (audio = sigma*z), optional coupling + W^-1 of flow `flow_done`
 * (glow.py:329-340) and optional `start` conv of flow `flow_next` (glow.py:189). -1 disables. */
int cwg_flow_boundary(const cwg_config* cfg, const cwg_weights* w, int mode,
                      int flow_done, int flow_next, const float* z, float sigma,
                      float* audio, const float* eo, void* x_out,
                      int batch, int t_mel, void* cuda_stream);

/* ---- forward direction: audio -> z, log_s, log det W (no-grad evaluation; NVIDIA WaveGlow.forward) ----------------
 * Flows run k = 0 .. F-1: early channels leave at k % n_early_every == 0, k > 0 (they stay in their columns of the
 * [batch][T'][n_group] audio state, which ends as z in the repo's layout z[b, s*n_group + c]); audio = W_k audio;
 * (b, log_s) = WN_k(audio_0, cond); audio_1 = exp(log_s) * audio_1 + b.  The cond is the upsampled mel cut to t_samples.
 *
 * Mixing matrices for the forward direction, from the state_dict's convinv.{k}.conv.weight (device fp32):
 *   w_fwd  [F][MG][MG] fp32 device out: W_k zero-padded (MG = CWG_GROUP_PAD(n_group))
 *   logdet [2][F] fp64 device out: logdet[k] = log det W_k as torch.logdet gives it (NaN for det < 0, -inf for det = 0),
 *          logdet[F + k] = log|det W_k|; fp64 LU with partial pivoting. */
int cwg_pack_forward(const cwg_config* cfg, const cwg_tensor* sd, int n_tensors, float* w_fwd, double* logdet,
                     void* cuda_stream);

/* Bytes of device workspace cwg_forward needs. 0 on error (cwg_last_error says why). */
size_t cwg_forward_workspace_bytes(const cwg_config* cfg, int mode, int batch, int t_mel, int t_samples);

/* Kernels cwg_forward launches (device-to-device copies not counted). */
int cwg_forward_launch_count(const cwg_config* cfg, int mode);

/* Forward pass.  mel [batch][n_mel][t_mel] fp32, cond_bias as in cwg_infer (cwg_cond_bias), audio [batch][t_samples]
 * fp32 with t_samples a positive multiple of n_group and <= t_mel * hop_length (need not be a multiple of hop_length).
 *   z          [batch][t_samples] fp32 out (may alias audio)
 *   log_s      NULL, or fp32 out: for k = 0 .. F-1 one [batch][n_half_k][T'] block after the other (T' = t_samples / n_group)
 *   logp_terms [batch][3] fp64 out: sum z^2, sum_k sum log_s_k, T' * sum_k log|det W_k| per utterance
 * Sums are reduced in a fixed order: identical calls give identical bytes.  The status word (cwg_infer_status) works as
 * for cwg_infer, with z in place of the waveform. */
int cwg_forward(const cwg_config* cfg, const cwg_weights* w, const float* w_fwd, const double* logdet, int mode,
                const float* mel, const float* cond_bias, const float* audio, int t_samples,
                float* z, float* log_s, double* logp_terms,
                void* workspace, size_t workspace_bytes, int batch, int t_mel, void* cuda_stream);

/* ax WaveGlow with waveflow=False (efficient_model_ax.py:279-357; AffineCouplingBlock.inverse
 * efficient_modules.py:94-105; glow_ax.WN.forward :375-418; InvertibleConv1x1.inverse :269-286 or
 * PermuteHeight, packed as a permutation matrix in `winv`).  Uses cwg_config / cwg_weights:
 * cond_hidden = padded width of the interpolated mel (256 in the tensor-core modes), w1's last
 * cond_hidden columns hold the WN's 1x1 cond layer, cond_w_* are unused, eo rows are ordered
 * [t | log_s].  mel [batch][n_mel][frames] is zero-extended by pad_frames and interpolated to
 * T' = t_samples / n_group steps.  mix_first selects coupling-then-mixing (1) or mixing-then-coupling (0). */
size_t cwg_ax_workspace_bytes(const cwg_config* cfg, int mode, int batch, int frames, int t_samples);
int cwg_ax_infer(const cwg_config* cfg, const cwg_weights* w, int mode,
                 const float* mel, int frames, int pad_frames, int upsample_linear, int mix_first,
                 const float* z, float sigma, float* audio, void* workspace, size_t workspace_bytes,
                 int batch, int t_samples, const float* b1_batch, void* cuda_stream);

/* Forward direction of the same model (audio -> z, log-likelihood terms; no-grad evaluation).  Flows run k = 0 .. F-1:
 * at k % n_early_every == 0, k > 0 the first n_early_size channels leave (they stay in their columns of the
 * [batch][T'][n_group] state, which ends as z in the layout cwg_ax_infer takes); then mix_first: audio = W_k audio,
 * (t, log_s) = WN_k(audio_0, cond), audio_1 = exp(log_s) * audio_1 + t;  mix_first = 0: the coupling first, then W_k.
 * The cond is the one cwg_ax_infer builds from the same mel (no pad frames), and the layer launches are its own.
 *   w_fwd      [F][MG][MG] fp32 device: W_k zero-padded (convinv.{k}.weight; for PermuteHeight the transpose of winv[k])
 *   logabsdet  [F] fp64 device: log|det W_k| (0 for a permutation)
 *   audio      [batch][t_samples] fp32, t_samples a positive multiple of n_group
 *   z          [batch][t_samples] fp32 out (may alias audio)
 *   logp_terms [batch][3] fp64 out: sum z^2, sum_k sum log_s_k, T' * sum_k log|det W_k| per utterance
 *   b1_batch   as in cwg_ax_infer (WN-level speaker embeddings) or NULL
 * Sums are reduced in a fixed order: identical calls give identical bytes, and row b of a batch equals the call for
 * utterance b alone.  The status word (cwg_infer_status) works as for cwg_forward, with z in place of the waveform. */
size_t cwg_ax_forward_workspace_bytes(const cwg_config* cfg, int mode, int batch, int frames, int t_samples);
/* Kernels cwg_ax_forward launches: F * (L * per-layer launches + 1) + 3, plus 1 in CWG_MODE_F16F8. -1 on error. */
int cwg_ax_forward_launch_count(const cwg_config* cfg, int mode);
int cwg_ax_forward(const cwg_config* cfg, const cwg_weights* w, const float* w_fwd, const double* logabsdet, int mode,
                   const float* mel, int frames, int upsample_linear, int mix_first, const float* audio, int t_samples,
                   float* z, double* logp_terms, void* workspace, size_t workspace_bytes, int batch,
                   const float* b1_batch, void* cuda_stream);

/* WN-level speaker embedding (glow_ax.py:284-286, :378-381: every flow's WN concatenates speaker_embed(speaker_id),
 * constant over time, to its cond input before the 1x1 cond layer).  A time-constant input of a 1x1 conv is a bias, so
 * the branch is evaluated once per call instead of per group-step:
 *   b1_batch[b][f][l][n] = b1[f][l][n] + sum_e spk_w[f][l][n][e] * spk_embed[f][speaker_ids[b]][e]
 * spk_w [F][L][2C][E] holds the speaker columns of every flow's cond_layers.0, spk_embed [F][S][E] the embedding tables.
 * The result ([batch][F][L][2C] fp32, device) is what cwg_ax_infer takes as `b1_batch` (NULL: the shared w->b1).  The
 * same commutation - interpolate(conv1x1(x)) == conv1x1(interpolate(x)) because the interpolation weights sum to 1 - is
 * what lets `upsample_first=False` models (cond layer at frame rate, then WN._upsample_mels, glow_ax.py:361-373, :389)
 * run on the same kernels. */
int cwg_ax_speaker_bias(const cwg_config* cfg, const float* b1, const float* spk_w, const float* spk_embed,
                        int speaker_embed_dim, int n_speakers, const int64_t* speaker_ids, int batch,
                        float* b1_batch, void* cuda_stream);

/* =====================================================================================
 * WaveFlow (BASELINE config 5): the reference's "ax" model with waveflow=True
 *   efficient_model_ax.py:279-357  WaveGlow.inverse      efficient_modules.py:42-65  WaveFlowCoupling.inverse
 *   glow_ax.py:556-635             WN_2d.forward          efficient_modules.py:360-403 PermuteHeight
 * Tensor-core modes (CWG_MODE_BF16X3 / CWG_MODE_BF16): channel_mixing='permuteheight', mix_first, upsample_first
 * (model-level F.interpolate of the mel), WN_2d with one 1x1 cond layer, dilation_h 1, dilation_w 2^i, n_channels 128,
 * GTU gate, res_skip without merge, n_group <= 32, and either a dense 3x3 in_layer or a depthwise-separable one
 * (glow_ax.py:525-531) of kernel_h <= 7 x odd kernel_w <= 7 (cwg_wf_weights.dw_w set; the trained checkpoints' 7x7).
 * CWG_MODE_FFMA runs general shapes and the WN_config variants.
 * ===================================================================================== */
#define CWG_WF_COND_PAD 128  /* mel channels padded to two 64-wide k-blocks */

typedef struct cwg_wf_config {
  int32_t n_mel;
  int32_t n_flows;
  int32_t n_group;        /* squeeze height h, 2 .. 32 */
  int32_t n_layers;
  int32_t n_channels;     /* 128 */
  int32_t kernel_h, kernel_w;   /* tensor-core modes: 3 x 3, or separable kernel_h <= 7 x odd kernel_w <= 7 */
  int32_t hop_length;
  int32_t upsample_linear;      /* 1: F.interpolate(mode='linear', align_corners=True); 0: 'nearest' */
  /* ABI 5 - WN_config variants of WN_2d, CWG_MODE_FFMA only (the tensor-core kernels take the defaults: all zero) */
  int32_t gate;                 /* CWG_GATE_* (glow_ax.py:168-198); 0 = GTU                                        */
  int32_t dilations_w[16];      /* n_layers_dilations_w (glow_ax.py:514); 0 = the default 2^i                      */
  int32_t dilations_h[16];      /* n_layers_dilations_h (:513,:517: causal padding (kernel_h-1)*dilation_h); 0 = 1 */
  int32_t n_early_every;        /* early outputs (efficient_model_ax.py:151-167,:319-340): 0 = none; a flow then works on  */
  int32_t n_early_size;         /*   the trailing n_rem height rows only                                                    */
  int32_t mix_first_off;        /* 1: mix_first = False (PermuteHeight.inverse BEFORE the coupling, :326-337); 0: after    */
  int32_t mixing_conv;          /* 1: channel_mixing = '1x1conv' (InvertibleConv1x1 over the height rows, efficient_modules.py */
                                /*    :269-286; cwg_wf_weights.winv); 0: PermuteHeight                                        */
} cwg_wf_config;

/* K1 = kernel_h*kernel_w*C + CWG_WF_COND_PAD (dense in_layers) or C + CWG_WF_COND_PAD (separable), N2 = C + CWG_EO_PAD */
typedef struct cwg_wf_weights {
  const uint16_t* w1_hi;   /* [F][L][2C][K1]  col (kh*kw_n + kw)*C + c | 9C + mel channel; separable: c | C + mel channel */
  const uint16_t* w1_lo;
  const float*    b1;      /* [F][L][2C]      in_layer bias + cond layer bias slice          */
  const uint16_t* w2_hi;   /* [F][L][N2][C]   rows <C res (0 for last layer; all 0 with merge_res_skip, where the hidden
                              tensor is never updated, glow_ax.py:613-626), C: log_s, C+1: t (end folded) */
  const uint16_t* w2_lo;
  const float*    b2;      /* [F][L][C]                                                      */
  const float*    eo_b;    /* [F][CWG_EO_PAD]                                                */
  const float*    start_w; /* [F][C]   Conv2d(1, C, 1x1)                                     */
  const float*    start_b; /* [F][C]                                                         */
  /* CWG_MODE_FFMA (fp32 CUDA cores; any even C, any kernel_h x odd kernel_w, n_group <= 32, any n_mel): the same two
   * matrices in fp32 with K1 = kernel_h*kernel_w*C + n_mel (the cond columns are not padded); hi / lo may then be NULL */
  const float*    w1_f32;
  const float*    w2_f32;
  /* ABI 5, CWG_MODE_FFMA, optional (NULL: the shared b1): per-utterance gate bias [batch][F][L][2C] of this call - the
   * WN-level speaker embedding (glow_ax.py:464-466,:567-570) is a time-constant input of the 1x1 cond layer, i.e. a bias;
   * cwg_ax_speaker_bias evaluates it */
  const float*    b1_batch;
  /* ABI 5, CWG_MODE_FFMA, mixing_conv = 1: W^-1 of every flow's InvertibleConv1x1, [F][32][32] row major (the flow's
   * n_rem x n_rem matrix in the top-left corner) */
  const float*    winv;
  /* ABI 5, CWG_MODE_FFMA, optional: the output of every flow's WN cond path evaluated by the caller - multi-layer / activated
   * cond stacks, a WN-level TransposedUpsampleNet (glow_ax.py:476-505,:565-579) - as [F][batch][2*C*L][T'] fp32.  When set,
   * w1_f32 has no cond columns (K1 = kernel_h*kernel_w*C), b1 holds the in_layer biases only and `mel` is not read. */
  const float*    c_all;
  /* ABI 5, optional: depthwise-separable in_layers (glow_ax.py:525-531) kept separable instead of folded to a dense
   * kernel_h x kernel_w conv (the layout of the reference author's trained checkpoints: 7x7 -> 49x fewer MACs).
   * dw_w [F][L][C][kernel_h*kernel_w], dw_b [F][L][C]: the depthwise conv (fp32 in every mode); w1_f32 is then
   * [F][L][2C][C + n_mel] and w1_hi / w1_lo [F][L][2C][C + CWG_WF_COND_PAD] (pointwise weights | cond layer), b1 the
   * pointwise + cond biases.  The tensor-core modes run it in one kernel per layer step (k_wf_sep_tc: the depthwise conv
   * on the CUDA cores feeds the pointwise GEMM through shared memory); NULL there means a dense 3x3 in_layer. */
  const float*    dw_w;
  const float*    dw_b;
} cwg_wf_weights;

size_t cwg_wf_workspace_bytes(const cwg_wf_config* cfg, int mode, int batch, int frames, int t_samples);

/* WaveGlow.inverse of the ax model (explicit latent): mel [batch][n_mel][frames] fp32, zero-extended
 * to frames + pad_frames (infer's artifact_trimming pad, efficient_model_ax.py:370-371) and
 * interpolated to T' = t_samples / n_group steps; z [batch][t_samples] standard normal (scaled by
 * sigma inside); audio [batch][t_samples] out.  mode: CWG_MODE_BF16X3 or CWG_MODE_BF16 (tcgen05 kernels: C = 128, dense
 * 3x3 or separable kernel_h <= 7 x odd kernel_w <= 7, n_group <= 32, n_mel <= 128), or CWG_MODE_FFMA (exact fp32 on the
 * CUDA cores, general shapes; csrc/cwg_wf_ffma.cu). */
int cwg_wf_infer(const cwg_wf_config* cfg, const cwg_wf_weights* w, int mode,
                 const float* mel, int frames, int pad_frames, const float* z, float sigma,
                 float* audio, void* workspace, size_t workspace_bytes,
                 int batch, int t_samples, void* cuda_stream);

/* Same; additionally records the caller's cudaEvent_t pairs around the e-th WN_2d layer launch (order: flows n_flows-1..0,
 * row steps 0..n_group-2, layers 0..n_layers-1) for e < n_events - bench.py times k_wf_layer_tc inside the real call. */
int cwg_wf_infer_profiled(const cwg_wf_config* cfg, const cwg_wf_weights* w, int mode,
                          const float* mel, int frames, int pad_frames, const float* z, float sigma,
                          float* audio, void* workspace, size_t workspace_bytes,
                          int batch, int t_samples, void* cuda_stream,
                          void** layer_ev_begin, void** layer_ev_end, int n_events);

int cwg_wf_launch_count(const cwg_wf_config* cfg);

/* Stage entry point (tests): one WN_2d layer of one autoregressive row step, either layout (tensor-core modes).
 * x_rings: bf16 planes (hi then lo), each [L][kernel_h][batch][T'][C]; mel_up planes [batch][T'][128];
 * reads ring slots of rows row .. row-kernel_h+1 (those >= 0) of layer `layer`, writes slot row%kernel_h of layer+1. */
int cwg_wf_layer(const cwg_wf_config* cfg, const cwg_wf_weights* w, int mode, int flow, int layer, int row,
                 void* x_rings, const void* mel_up, float* eo, int batch, int t_samples, void* cuda_stream);

/* Forward direction (audio -> z) of the tensor-core subset above, CWG_MODE_BF16X3 / CWG_MODE_BF16 (CWG_MODE_FFMA and the
 * WN_config variants are errors).  With x = audio.view(B, T', h).transpose(1, 2) and the cond of cwg_wf_infer, flows
 * k = 0 .. F-1 do x = permute_height(x, k), then (log_s_r, t_r) = WN_2d(rows 0 .. h-2 of x, causal in height) and
 * x[r+1] = x[r+1] * exp(log_s_r) + t_r; z = x in the [batch][t_samples] layout cwg_wf_infer takes (z[b, s*h + c]).
 * Every height row is known before a flow runs, so each WN_2d layer is one launch over all h-1 rows.
 *   mel        [batch][n_mel][frames] fp32, interpolated to T' = t_samples / n_group steps (no pad frames)
 *   audio      [batch][t_samples] fp32; z [batch][t_samples] fp32 out
 *   logp_terms [batch][3] fp64 out: sum z^2, sum_k sum log_s_k, 0 (PermuteHeight has |det| = 1) per utterance
 * Sums are reduced in a fixed order: identical calls give identical bytes, and row b of a batch equals the
 * single-utterance call. */
size_t cwg_wf_forward_workspace_bytes(const cwg_wf_config* cfg, int mode, int batch, int frames, int t_samples);
int cwg_wf_forward_launch_count(const cwg_wf_config* cfg);     /* n_flows * (n_layers + 1) + 3 */
int cwg_wf_forward(const cwg_wf_config* cfg, const cwg_wf_weights* w, int mode, const float* mel, int frames,
                   const float* audio, int t_samples, float* z, double* logp_terms, void* workspace, size_t workspace_bytes,
                   int batch, void* cuda_stream);

/* Stage entry point (tests): one full-height WN_2d layer of the forward direction.  x_bufs: bf16 planes (hi then lo), each
 * two buffers [2][n_group-1][batch][T'][C]; reads buffer layer % 2 at rows r-kernel_h+1 .. r (those >= 0) for every row
 * r = 0 .. n_group-2 and writes buffer (layer+1) % 2 (not for the last layer); eo [n_group-1][batch*T'][CWG_EO_PAD]. */
int cwg_wf_forward_layer(const cwg_wf_config* cfg, const cwg_wf_weights* w, int mode, int flow, int layer, void* x_bufs,
                         const void* mel_up, float* eo, int batch, int t_samples, void* cuda_stream);

/* =====================================================================================
 * Denoiser post-filter (SURVEY 8f-1): CookieTTS/_4_mtw/waveglow/denoiser.py:59-71 on the conv-based STFT of
 * CookieTTS/utils/audio/stft.py:79-146 (reflect pad, windowed Fourier bases, window-sum-square synthesis).
 *   fwd_basis   [2*cutoff][fl]   windowed forward basis (real rows then imaginary rows), cutoff = fl/2 + 1
 *   inv_basis_t [fl][2*cutoff]   windowed inverse (pinv) basis, transposed
 *   window_sum  [fl + hop*(NF-1)]  audio_processing.py:7-57, NF = (T + 2*(fl/2) - fl)/hop + 1
 *   bias_spec   [n_bias][cutoff] mean magnitude of the vocoder's output for a near-silent mel; bias_index [B]
 *               selects a row per utterance (NULL = row 0)
 *   out         [B][cwg_denoise_out_samples(T, fl, hop)]
 * ===================================================================================== */
size_t cwg_denoise_workspace_bytes(int batch, int n_samples, int filter_length, int hop_length);
int    cwg_denoise_out_samples(int n_samples, int filter_length, int hop_length);
int    cwg_stft_mean_magnitude(const float* audio, int batch, int n_samples, int filter_length, int hop_length,
                               const float* fwd_basis, float* mean_mag, void* workspace, size_t workspace_bytes,
                               void* cuda_stream);
int    cwg_denoise(const float* audio, int batch, int n_samples, int filter_length, int hop_length,
                   const float* fwd_basis, const float* inv_basis_t, const float* window_sum,
                   const float* bias_spec, const int32_t* bias_index, float strength,
                   float* out, void* workspace, size_t workspace_bytes, void* cuda_stream);

/* =====================================================================================
 * 16-bit PCM output (SURVEY 8f-2): CookieTTS/_5_infer/t2s_server/text2speech.py:672-694 - per utterance, samples
 * past n_valid[b] (= output_length*hop; NULL = all of t_stride) become silence, the rest is
 * (audio * 2**15).astype('int16') (truncation toward zero).  out [B][out_stride]; out_stride may exceed
 * t_stride (the `cat_silence_s` padding).  saturate = 0 reproduces numpy's wrap-around for |audio| >= 1,
 * saturate = 1 clips instead.
 * ===================================================================================== */
int cwg_pcm16(const float* audio, int batch, int t_stride, const int32_t* n_valid, int16_t* out, int out_stride,
              int saturate, void* cuda_stream);

/* =====================================================================================
 * Conditioning front-end and output filters of the "ax" models (SURVEY 8f-3), fp32, channels-first [B, C, T]
 * like the reference tensors.  pad_mode: 0 zeros, 1 replicate, 2 reflect, 3 circular.  act: 0 none, 1 relu,
 * 2 leaky relu (slope), 3 tanh, 4 sigmoid.
 *   cwg_conv1d            y = res + out_scale * act(conv1d(x, w[c_out][c_in][k], padding) + bias); res may be NULL.
 *                         nn.Conv1d of efficient_model_ax.py:74-113 (cond_layers, res_conv), applied at :293-307.
 *   cwg_conv_transpose1d  y = out_scale * act(conv_transpose1d(x, stride, padding) + bias), nn.ConvTranspose1d of
 *                         TransposedUpsampleNet (glow_ax.py:201-242).  w_phases is the torch weight [c_in][c_out][k]
 *                         re-packed per output phase r: [stride][c_out][c_in][ceil(k/stride)], tap jj = w[ci][co][r + stride*jj].
 *   cwg_resample1d        F.interpolate along T (mode 0 nearest, 1 linear align_corners=True, 2 linear
 *                         align_corners=False) to t_virtual samples, of which [crop, crop + t_out) are written
 *                         (or added when accumulate != 0); scale_factor > 0 is the value given to F.interpolate.
 *   cwg_deemphasis        y[n] = x[n] + coef*y[n-1] per utterance in fp64 (scipy.signal.lfilter([1],[1,-coef]),
 *                         efficient_model_ax.py:351-355), after the optional inverse volume map (:343-345).
 * ===================================================================================== */
int cwg_conv1d(const float* x, int batch, int c_in, int t_in, const float* w, const float* bias, int c_out, int k,
               int padding, int pad_mode, int act, float slope, float out_scale, const float* res, float* y,
               void* cuda_stream);
int cwg_conv_transpose1d(const float* x, int batch, int c_in, int t_in, const float* w_phases, const float* bias,
                         int c_out, int k, int stride, int padding, int act, float slope, float out_scale, float* y,
                         void* cuda_stream);
int cwg_resample1d(const float* x, int batch, int channels, int t_in, long long x_batch_stride, float* y, int t_out,
                   long long y_batch_stride, int mode, int t_virtual, int crop, float scale_factor, int accumulate,
                   void* cuda_stream);
int cwg_deemphasis(const float* x, int batch, int t_samples, double coef, int vol_scaling, float* y, void* cuda_stream);

/* =====================================================================================
 * Mel-domain flow decoders (SURVEY 8f-4): FlowDecoder.inverse of the reference's text-to-mel models
 *   CookieTTS/_2_ttm/flowtts/waveglow/glow.py:302-343 (WN.forward :133-172, modules.py:36-47, :234-250) and
 *   CookieTTS/_2_ttm/untts/waveglow/glow.py (same, plus the constant padding of the first flow's hidden tensor, :80,126).
 * fp32, the reference's channels-first layout.  z [batch][n_group][T] is updated in place: on entry the latent (already
 * multiplied by sigma, viewed as the reference's z.view(B, n_group, -1)), on return the mel; the active channels of flow k
 * are the trailing n_rem_k ones (early outputs sit in front, glow.py:317-321,339-340).  cond [batch][cond_channels][T].
 * Supported: WN with one 1x1 cond layer without activation (the hparams defaults), any n_layers <= 16 / dilations /
 * odd kernel size, res_skip on or off, merge_res_skip on or off, mix_first on or off, no decoder-level cond layers.
 * ===================================================================================== */
#define CWG_FD_MAX_LAYERS 16

typedef struct cwg_fd_config {
  int32_t n_group, n_flows, n_early_every, n_early_size, mix_first;
  int32_t cond_channels;
  int32_t n_layers, n_channels, kernel_size;
  int32_t dilations[CWG_FD_MAX_LAYERS];
  int32_t res_skip;          /* hparams.wn_res_skip       */
  int32_t merge_res_skip;    /* hparams.wn_merge_res_skip */
  float   first_pad_value;   /* untts decoder_padding_value: pads the hidden tensor of flow 0's in_layers; 0 for flowtts */
} cwg_fd_config;

/* Device fp32 arrays, weight-norm folded.  F flows, L layers, C channels, Cc cond channels, ks kernel size; n_rem_k /
 * n_half_k = n_rem_k / 2 per flow (glow.py:205-220).  "concatenated" = flow after flow with the per-flow shape given. */
typedef struct cwg_fd_weights {
  const float* start_w;   /* concatenated [C][n_half_k]                  */
  const float* start_b;   /* [F][C]                                       */
  const float* cond_w;    /* [F][2CL][Cc]   WN.cond_layers.0              */
  const float* cond_b;    /* [F][2CL]                                     */
  const float* in_w;      /* [F][L][2C][C][ks]                            */
  const float* in_b;      /* [F][L][2C]                                   */
  const float* rs_w;      /* [F][L][2C][C]  (rows past the layer's res_skip width unused); NULL when res_skip = 0 */
  const float* rs_b;      /* [F][L][2C]                                   */
  const float* end_w;     /* concatenated [2 n_half_k][C]                 */
  const float* end_b;     /* concatenated [2 n_half_k]                    */
  const float* winv;      /* concatenated [n_rem_k][n_rem_k]  W^-1, row major */
  /* ABI 5, optional: the output of every flow's WN cond stack evaluated by the caller (several cond layers / kernel sizes /
   * activations, glow.py:74-101,:145-148) as [F][batch][2CL][T]; cond_w / cond_b and `cond` are then not read */
  const float* c_all;
} cwg_fd_weights;

size_t cwg_fd_workspace_bytes(const cwg_fd_config* cfg, int batch, int t_steps);
int    cwg_fd_launch_count(const cwg_fd_config* cfg);
int    cwg_fd_inverse(const cwg_fd_config* cfg, const cwg_fd_weights* w, const float* cond, float* z,
                      void* workspace, size_t workspace_bytes, int batch, int t_steps, void* cuda_stream);

/* =====================================================================================
 * General fp32 mode of the ax 1-D WN (glow_ax.py:245-418) for the WN_config variants the packed tensor-core / FFMA layer
 * kernels are not specialised for: any of the 14 gated units of glow_ax.py:36-198, listed dilations
 * (n_layers_dilations_w, :331-335), merge_res_skip / res_skip=False (:259-263,:352,:399-414: the hidden tensor is then
 * never updated and every layer's res_skip output is accumulated), and WN cond stacks of several layers / activations /
 * kernel sizes (:297-329) - the caller evaluates the cond stack (cwg_conv1d, cwg_resample1d) and hands over its output
 * c_all [batch][2*C*L][T'].  One call = one flow of WaveGlow.inverse (efficient_model_ax.py:325-340): channel mixing
 * (before or after, mix_first), WN, AffineCouplingBlock.inverse (efficient_modules.py:99-105), ignore_nan.
 * z is the reference's channels-first view [batch][n_group][T'] (cwg_group_transpose converts from / to [batch][T]),
 * updated in place; the active channels of the flow are the trailing n_rem rows.
 * ===================================================================================== */
#define CWG_GATE_GTU      0   /* tanh * sigmoid          */
#define CWG_GATE_GTRU     1   /* tanh * relu             */
#define CWG_GATE_GTLRU    2   /* tanh * leaky_relu(0.01) */
#define CWG_GATE_GLU      3   /* x * sigmoid             */
#define CWG_GATE_TTU      4   /* tanh * tanh             */
#define CWG_GATE_STU      5   /* tanh * selu             */
#define CWG_GATE_GTSU     6   /* tanhshrink * sigmoid    */
#define CWG_GATE_SPTU     7   /* tanh * softplus         */
#define CWG_GATE_GSIU     8   /* sin * sigmoid           */
#define CWG_GATE_GSIRU    9   /* sin(16 x) * sigmoid     */
#define CWG_GATE_GTSRU    10  /* tanhshrink * relu       */
#define CWG_GATE_GSIRRU   11  /* sin(16 x) * relu        */
#define CWG_GATE_GSIRLRU  12  /* sin(16 x) * leaky_relu(0.01) */
#define CWG_GATE_GSIRRLRU 13  /* sin(16 x) * rrelu(0.01, 0.1) in eval mode = leaky_relu(0.055) */
#define CWG_GATE_COUNT    14

typedef struct cwg_axg_config {
  int32_t n_group;           /* rows of z                                               */
  int32_t n_rem;             /* active (trailing) channels of this flow, even            */
  int32_t mix_first;         /* 1: coupling then mixing, 0: mixing then coupling         */
  int32_t n_layers, n_channels, kernel_size;
  int32_t dilations[CWG_FD_MAX_LAYERS];
  int32_t res_skip;          /* WN_config['res_skip']                                    */
  int32_t merge_res_skip;    /* WN_config['merge_res_skip']                              */
  int32_t gate;              /* CWG_GATE_*                                               */
  int32_t ignore_nan;        /* efficient_model_ax.py:331-332                            */
} cwg_axg_config;

/* Device fp32 arrays of ONE flow, weight-norm folded, separable in_layers folded to dense (C = n_channels, L = n_layers,
 * ks = kernel_size, n_half = n_rem / 2). */
typedef struct cwg_axg_weights {
  const float* start_w;   /* [C][n_half]                                                  */
  const float* start_b;   /* [C]                                                          */
  const float* in_w;      /* [L][2C][C][ks]                                               */
  const float* in_b;      /* [L][2C]                                                      */
  const float* rs_w;      /* [L][2C][C]  rows past a layer's res_skip width unused; NULL when res_skip = 0 */
  const float* rs_b;      /* [L][2C]                                                      */
  const float* end_w;     /* [2 n_half][C]   rows: log_s then t                           */
  const float* end_b;     /* [2 n_half]                                                   */
  const float* winv;      /* [n_rem][n_rem]  W^-1 (or the PermuteHeight permutation matrix), row major */
} cwg_axg_weights;

size_t cwg_axg_workspace_bytes(const cwg_axg_config* cfg, int batch, int t_steps);
int    cwg_axg_launch_count(const cwg_axg_config* cfg);
int    cwg_axg_flow(const cwg_axg_config* cfg, const cwg_axg_weights* w, const float* c_all, float* z,
                    void* workspace, size_t workspace_bytes, int batch, int t_steps, void* cuda_stream);

/* z.view(B, -1, n_group).transpose(1, 2) and back (efficient_model_ax.py:310,347): to_channels_first = 1 reads
 * in [batch][T'][n_group] and writes out [batch][n_group][T']; 0 is the inverse. */
int cwg_group_transpose(const float* in, float* out, int batch, int t_steps, int n_group, int to_channels_first,
                        void* cuda_stream);

#ifdef __cplusplus
}
#endif
#endif /* CWG_H */
