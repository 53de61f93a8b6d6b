// torch.ops.cookietts_b200.* - the reference-side binding of the C ABI (include/cwg.h) for PyTorch callers.
// This is the ONLY file of the repo that sees torch types: it unpacks tensors into plain pointers / sizes, takes the
// current CUDA stream and calls libcwg.so.  cookietts_b200.WaveGlow.infer (the drop-in for glow.py:314-350) calls
// torch.ops.cookietts_b200.waveglow_pack once per checkpoint and torch.ops.cookietts_b200.waveglow_infer per call.
#include <ATen/ATen.h>
#include <c10/cuda/CUDAGuard.h>
#include <c10/cuda/CUDAStream.h>
#include <torch/library.h>

#include <string>
#include <tuple>
#include <vector>

#include "../../include/cwg.h"

namespace {

cwg_config config_from(at::IntArrayRef v) {
  TORCH_CHECK(v.size() == 11, "cfg must hold the 11 fields of cwg_config, got ", v.size());
  cwg_config c;
  c.n_mel = (int32_t)v[0]; c.n_flows = (int32_t)v[1]; c.n_group = (int32_t)v[2]; c.n_early_every = (int32_t)v[3];
  c.n_early_size = (int32_t)v[4]; c.win_length = (int32_t)v[5]; c.hop_length = (int32_t)v[6]; c.n_layers = (int32_t)v[7];
  c.n_channels = (int32_t)v[8]; c.kernel_size = (int32_t)v[9]; c.cond_hidden = (int32_t)v[10];
  return c;
}

void check(int rc) { TORCH_CHECK(rc == 0, "libcwg error ", rc, ": ", cwg_last_error()); }

void* aligned(const at::Tensor& t, size_t a) {
  return (void*)(((uintptr_t)t.data_ptr() + a - 1) / a * a);
}

// names: the state_dict keys joined by '\n', in the order of `tensors`
std::vector<std::string> split_names(const std::string& names) {
  std::vector<std::string> keys;
  size_t pos = 0;
  while (pos <= names.size()) {
    const size_t e = names.find('\n', pos);
    keys.push_back(names.substr(pos, e == std::string::npos ? std::string::npos : e - pos));
    if (e == std::string::npos) break;
    pos = e + 1;
  }
  return keys;
}

at::Tensor waveglow_pack(at::TensorList tensors, std::string names, at::IntArrayRef cfg, int64_t mode) {
  TORCH_CHECK(!tensors.empty(), "empty state_dict");
  const cwg_config c = config_from(cfg);
  const std::vector<std::string> keys = split_names(names);
  TORCH_CHECK(keys.size() == tensors.size(), "names / tensors length mismatch: ", keys.size(), " vs ", tensors.size());
  const at::Device dev = tensors[0].device();
  TORCH_CHECK(dev.is_cuda(), "waveglow_pack needs the parameters on a CUDA device (no CPU fallback)");
  c10::cuda::CUDAGuard guard(dev);
  std::vector<at::Tensor> keep;
  std::vector<cwg_tensor> sd(tensors.size());
  for (size_t i = 0; i < tensors.size(); ++i) {
    TORCH_CHECK(tensors[i].device() == dev, keys[i], " is on another device");
    TORCH_CHECK(tensors[i].dim() <= 4, keys[i], " has more than 4 dimensions");
    keep.push_back(tensors[i].detach().to(at::kFloat).contiguous());
    sd[i].name = keys[i].c_str();
    sd[i].data = keep.back().data_ptr<float>();
    sd[i].ndim = (int32_t)keep.back().dim();
    for (int k = 0; k < 4; ++k) sd[i].shape[k] = k < keep.back().dim() ? keep.back().size(k) : 1;
  }
  int E = 0, S = 0, rz = 0;
  check(cwg_state_dict_info(sd.data(), (int)sd.size(), &E, &S, &rz));
  const size_t bytes = cwg_packed_bytes(&c, (int)mode, E, S), ws_bytes = cwg_pack_workspace_bytes(&c, E);
  TORCH_CHECK(bytes > 0 && ws_bytes > 0, "libcwg: ", cwg_last_error());
  const auto u8 = at::TensorOptions().dtype(at::kByte).device(dev);
  at::Tensor packed = at::empty({(int64_t)bytes + 256}, u8), ws = at::empty({(int64_t)ws_bytes + 256}, u8);
  cwg_weights w;
  check(cwg_pack_weights(&c, (int)mode, sd.data(), (int)sd.size(), aligned(packed, 256), bytes, aligned(ws, 256), ws_bytes, &w,
                         (void*)c10::cuda::getCurrentCUDAStream(dev.index()).stream()));
  return packed;
}

std::tuple<at::Tensor, at::Tensor> waveglow_infer(const at::Tensor& packed, at::IntArrayRef cfg, int64_t mode, int64_t embed_dim, int64_t n_speakers,
                          const at::Tensor& mel, const c10::optional<at::Tensor>& speaker_ids, const at::Tensor& z, double sigma,
                          at::IntArrayRef ev_begin, at::IntArrayRef ev_end) {
  const cwg_config c = config_from(cfg);
  TORCH_CHECK(mel.is_cuda() && z.is_cuda() && packed.is_cuda(), "waveglow_infer needs CUDA tensors (no CPU fallback)");
  TORCH_CHECK(mel.scalar_type() == at::kFloat && z.scalar_type() == at::kFloat && mel.is_contiguous() && z.is_contiguous(),
              "mel and z must be contiguous fp32");
  TORCH_CHECK(mel.dim() == 3 && mel.size(1) == c.n_mel, "mel must be [B, ", c.n_mel, ", T_mel]");
  const int64_t B = mel.size(0), Tm = mel.size(2), T = Tm * c.hop_length;
  TORCH_CHECK(z.dim() == 2 && z.size(0) == B && z.size(1) == T, "z must be [B, T_mel*hop]");
  TORCH_CHECK(ev_begin.size() == ev_end.size(), "event lists differ in length");
  const at::Device dev = mel.device();
  c10::cuda::CUDAGuard guard(dev);
  void* stream = (void*)c10::cuda::getCurrentCUDAStream(dev.index()).stream();
  cwg_weights w;
  check(cwg_packed_view(&c, (int)mode, (int)embed_dim, (int)n_speakers, aligned(packed, 256), (size_t)packed.numel() - 256, &w));
  const int64_t* ids = nullptr;
  at::Tensor ids_t;
  if (embed_dim > 0) {
    TORCH_CHECK(speaker_ids.has_value(), "this model has speaker embeddings: pass speaker ids");
    ids_t = speaker_ids->to(dev, at::kLong).contiguous();
    TORCH_CHECK(ids_t.numel() == B, "speaker ids must hold one entry per utterance");
    ids = ids_t.data_ptr<int64_t>();
  }
  const auto f32 = at::TensorOptions().dtype(at::kFloat).device(dev);
  at::Tensor cond_bias = at::empty({B, c.n_flows, c.cond_hidden}, f32);
  check(cwg_cond_bias(&c, &w, ids, (int)B, cond_bias.data_ptr<float>(), stream));
  const size_t ws_bytes = cwg_workspace_bytes(&c, (int)mode, (int)B, (int)Tm);
  TORCH_CHECK(ws_bytes > 0, "libcwg: ", cwg_last_error());
  at::Tensor ws = at::empty({(int64_t)ws_bytes + 1024}, at::TensorOptions().dtype(at::kByte).device(dev));
  at::Tensor audio = at::empty({B, T}, f32);
  if (ev_begin.empty()) {
    check(cwg_infer(&c, &w, (int)mode, mel.data_ptr<float>(), cond_bias.data_ptr<float>(), z.data_ptr<float>(), (float)sigma,
                    audio.data_ptr<float>(), aligned(ws, 1024), ws_bytes, (int)B, (int)Tm, stream));
  } else {
    std::vector<void*> eb(ev_begin.size()), ee(ev_end.size());
    for (size_t i = 0; i < eb.size(); ++i) { eb[i] = (void*)(uintptr_t)ev_begin[i]; ee[i] = (void*)(uintptr_t)ev_end[i]; }
    check(cwg_infer_profiled(&c, &w, (int)mode, mel.data_ptr<float>(), cond_bias.data_ptr<float>(), z.data_ptr<float>(),
                             (float)sigma, audio.data_ptr<float>(), aligned(ws, 1024), ws_bytes, (int)B, (int)Tm, stream,
                             eb.data(), ee.data(), (int)eb.size()));
  }
  at::Tensor status = at::empty({1}, at::TensorOptions().dtype(at::kInt).device(dev));
  check(cwg_infer_status(aligned(ws, 1024), status.data_ptr<int32_t>(), stream));
  return std::make_tuple(audio, status);
}

// waveglow_infer with per-utterance lengths (cwg_infer_ragged): lengths int32 [B] mel frames, 1 <= lengths[b] <= T_mel
std::tuple<at::Tensor, at::Tensor> waveglow_infer_ragged(const at::Tensor& packed, at::IntArrayRef cfg, int64_t mode,
                                                         int64_t embed_dim, int64_t n_speakers, const at::Tensor& mel,
                                                         const c10::optional<at::Tensor>& speaker_ids, const at::Tensor& z,
                                                         double sigma, const at::Tensor& lengths) {
  const cwg_config c = config_from(cfg);
  TORCH_CHECK(mel.is_cuda() && z.is_cuda() && packed.is_cuda() && lengths.is_cuda(),
              "waveglow_infer_ragged needs CUDA tensors (no CPU fallback)");
  TORCH_CHECK(mel.scalar_type() == at::kFloat && z.scalar_type() == at::kFloat && mel.is_contiguous() && z.is_contiguous(),
              "mel and z must be contiguous fp32");
  TORCH_CHECK(mel.dim() == 3 && mel.size(1) == c.n_mel, "mel must be [B, ", c.n_mel, ", T_mel]");
  const int64_t B = mel.size(0), Tm = mel.size(2), T = Tm * c.hop_length;
  TORCH_CHECK(z.dim() == 2 && z.size(0) == B && z.size(1) == T, "z must be [B, T_mel*hop]");
  TORCH_CHECK(lengths.scalar_type() == at::kInt && lengths.is_contiguous() && lengths.dim() == 1 && lengths.size(0) == B,
              "lengths must be a contiguous int32 [B] tensor");
  const at::Device dev = mel.device();
  TORCH_CHECK(lengths.device() == dev, "lengths must be on the device of mel");
  c10::cuda::CUDAGuard guard(dev);
  void* stream = (void*)c10::cuda::getCurrentCUDAStream(dev.index()).stream();
  cwg_weights w;
  check(cwg_packed_view(&c, (int)mode, (int)embed_dim, (int)n_speakers, aligned(packed, 256), (size_t)packed.numel() - 256, &w));
  const int64_t* ids = nullptr;
  at::Tensor ids_t;
  if (embed_dim > 0) {
    TORCH_CHECK(speaker_ids.has_value(), "this model has speaker embeddings: pass speaker ids");
    ids_t = speaker_ids->to(dev, at::kLong).contiguous();
    TORCH_CHECK(ids_t.numel() == B, "speaker ids must hold one entry per utterance");
    ids = ids_t.data_ptr<int64_t>();
  }
  const auto f32 = at::TensorOptions().dtype(at::kFloat).device(dev);
  at::Tensor cond_bias = at::empty({B, c.n_flows, c.cond_hidden}, f32);
  check(cwg_cond_bias(&c, &w, ids, (int)B, cond_bias.data_ptr<float>(), stream));
  const size_t ws_bytes = cwg_ragged_workspace_bytes(&c, (int)mode, (int)B, (int)Tm);
  TORCH_CHECK(ws_bytes > 0, "libcwg: ", cwg_last_error());
  at::Tensor ws = at::empty({(int64_t)ws_bytes + 1024}, at::TensorOptions().dtype(at::kByte).device(dev));
  at::Tensor audio = at::empty({B, T}, f32);
  check(cwg_infer_ragged(&c, &w, (int)mode, mel.data_ptr<float>(), cond_bias.data_ptr<float>(), z.data_ptr<float>(),
                         (float)sigma, lengths.data_ptr<int32_t>(), audio.data_ptr<float>(), aligned(ws, 1024), ws_bytes,
                         (int)B, (int)Tm, stream));
  at::Tensor status = at::empty({1}, at::TensorOptions().dtype(at::kInt).device(dev));
  check(cwg_infer_status(aligned(ws, 1024), status.data_ptr<int32_t>(), stream));
  return std::make_tuple(audio, status);
}

// Forward-direction mixing matrices: uint8 blob = W_k padded [F][MG][MG] fp32, then logdet [2][F] fp64 (cwg_pack_forward)
at::Tensor waveglow_pack_forward(at::TensorList tensors, std::string names, at::IntArrayRef cfg) {
  TORCH_CHECK(!tensors.empty(), "empty state_dict");
  const cwg_config c = config_from(cfg);
  const std::vector<std::string> keys = split_names(names);
  TORCH_CHECK(keys.size() == tensors.size(), "names / tensors length mismatch: ", keys.size(), " vs ", tensors.size());
  const at::Device dev = tensors[0].device();
  TORCH_CHECK(dev.is_cuda(), "waveglow_pack_forward needs the parameters on a CUDA device (no CPU fallback)");
  c10::cuda::CUDAGuard guard(dev);
  std::vector<at::Tensor> keep;
  std::vector<cwg_tensor> sd;
  for (size_t i = 0; i < tensors.size(); ++i) {
    if (keys[i].rfind("convinv.", 0) != 0) continue;         // only the mixing matrices are read
    TORCH_CHECK(tensors[i].device() == dev, keys[i], " is on another device");
    keep.push_back(tensors[i].detach().to(at::kFloat).contiguous());
    cwg_tensor t;
    t.name = keys[i].c_str();
    t.data = keep.back().data_ptr<float>();
    t.ndim = (int32_t)std::min<int64_t>(keep.back().dim(), 4);
    for (int k = 0; k < 4; ++k) t.shape[k] = k < keep.back().dim() ? keep.back().size(k) : 1;
    sd.push_back(t);
  }
  const int64_t mg = CWG_GROUP_PAD(c.n_group), wbytes = (int64_t)c.n_flows * mg * mg * 4;
  at::Tensor blob = at::empty({wbytes + 2 * (int64_t)c.n_flows * 8}, at::TensorOptions().dtype(at::kByte).device(dev));
  check(cwg_pack_forward(&c, sd.data(), (int)sd.size(), (float*)blob.data_ptr(), (double*)((char*)blob.data_ptr() + wbytes),
                         (void*)c10::cuda::getCurrentCUDAStream(dev.index()).stream()));
  return blob;
}

// (z [B, T], log_s (flat, empty unless want_log_s), logp_terms [B, 3] fp64, status int32 [1])
std::tuple<at::Tensor, at::Tensor, at::Tensor, at::Tensor> waveglow_forward(
    const at::Tensor& packed, const at::Tensor& packed_fwd, at::IntArrayRef cfg, int64_t mode, int64_t embed_dim,
    int64_t n_speakers, const at::Tensor& mel, const c10::optional<at::Tensor>& speaker_ids, const at::Tensor& audio,
    bool want_log_s) {
  const cwg_config c = config_from(cfg);
  TORCH_CHECK(mel.is_cuda() && audio.is_cuda() && packed.is_cuda() && packed_fwd.is_cuda(),
              "waveglow_forward needs CUDA tensors (no CPU fallback)");
  TORCH_CHECK(mel.scalar_type() == at::kFloat && audio.scalar_type() == at::kFloat && mel.is_contiguous() && audio.is_contiguous(),
              "mel and audio must be contiguous fp32");
  TORCH_CHECK(mel.dim() == 3 && mel.size(1) == c.n_mel, "mel must be [B, ", c.n_mel, ", T_mel]");
  const int64_t B = mel.size(0), Tm = mel.size(2);
  TORCH_CHECK(audio.dim() == 2 && audio.size(0) == B, "audio must be [B, T]");
  const int64_t T = audio.size(1);
  const int64_t mg = CWG_GROUP_PAD(c.n_group), wbytes = (int64_t)c.n_flows * mg * mg * 4;
  TORCH_CHECK(packed_fwd.numel() == wbytes + 2 * (int64_t)c.n_flows * 8, "packed_fwd does not match cfg");
  const at::Device dev = mel.device();
  c10::cuda::CUDAGuard guard(dev);
  void* stream = (void*)c10::cuda::getCurrentCUDAStream(dev.index()).stream();
  cwg_weights w;
  check(cwg_packed_view(&c, (int)mode, (int)embed_dim, (int)n_speakers, aligned(packed, 256), (size_t)packed.numel() - 256, &w));
  const int64_t* ids = nullptr;
  at::Tensor ids_t;
  if (embed_dim > 0) {
    TORCH_CHECK(speaker_ids.has_value(), "this model has speaker embeddings: pass speaker ids");
    ids_t = speaker_ids->to(dev, at::kLong).contiguous();
    TORCH_CHECK(ids_t.numel() == B, "speaker ids must hold one entry per utterance");
    ids = ids_t.data_ptr<int64_t>();
  }
  const auto f32 = at::TensorOptions().dtype(at::kFloat).device(dev);
  at::Tensor cond_bias = at::empty({B, c.n_flows, c.cond_hidden}, f32);
  check(cwg_cond_bias(&c, &w, ids, (int)B, cond_bias.data_ptr<float>(), stream));
  const size_t ws_bytes = cwg_forward_workspace_bytes(&c, (int)mode, (int)B, (int)Tm, (int)T);
  TORCH_CHECK(ws_bytes > 0, "libcwg: ", cwg_last_error());
  at::Tensor ws = at::empty({(int64_t)ws_bytes + 1024}, at::TensorOptions().dtype(at::kByte).device(dev));
  at::Tensor z = at::empty({B, T}, f32);
  int64_t n_log_s = 0;
  if (want_log_s) {
    int nh = c.n_group / 2;
    for (int k = 0; k < c.n_flows; ++k) {
      if (k > 0 && k % c.n_early_every == 0) nh -= c.n_early_size / 2;
      n_log_s += B * nh * (T / c.n_group);
    }
  }
  at::Tensor log_s = at::empty({n_log_s}, f32);
  at::Tensor terms = at::empty({B, 3}, at::TensorOptions().dtype(at::kDouble).device(dev));
  const char* pf = (const char*)packed_fwd.data_ptr();
  check(cwg_forward(&c, &w, (const float*)pf, (const double*)(pf + wbytes), (int)mode, mel.data_ptr<float>(),
                    cond_bias.data_ptr<float>(), audio.data_ptr<float>(), (int)T, z.data_ptr<float>(),
                    want_log_s ? log_s.data_ptr<float>() : nullptr, terms.data_ptr<double>(), aligned(ws, 1024), ws_bytes,
                    (int)B, (int)Tm, stream));
  at::Tensor status = at::empty({1}, at::TensorOptions().dtype(at::kInt).device(dev));
  check(cwg_infer_status(aligned(ws, 1024), status.data_ptr<int32_t>(), stream));
  return std::make_tuple(z, log_s, terms, status);
}

// int32 [1] device tensor: 1 when `x` holds a NaN / Inf (cwg_nonfinite), else 0
at::Tensor nonfinite(const at::Tensor& x) {
  TORCH_CHECK(x.is_cuda() && x.scalar_type() == at::kFloat && x.is_contiguous(), "nonfinite needs a contiguous fp32 CUDA tensor");
  c10::cuda::CUDAGuard guard(x.device());
  at::Tensor flag = at::empty({1}, at::TensorOptions().dtype(at::kInt).device(x.device()));
  check(cwg_nonfinite(x.data_ptr<float>(), (size_t)x.numel(), flag.data_ptr<int32_t>(),
                      (void*)c10::cuda::getCurrentCUDAStream(x.device().index()).stream()));
  return flag;
}

int64_t waveglow_launch_count(at::IntArrayRef cfg, int64_t mode) {
  const cwg_config c = config_from(cfg);
  return cwg_launch_count(&c, (int)mode);
}

int64_t abi_version() { return cwg_abi_version(); }

}  // namespace

TORCH_LIBRARY(cookietts_b200, m) {
  m.def("waveglow_pack(Tensor[] tensors, str names, int[] cfg, int mode) -> Tensor");
  m.def("waveglow_infer(Tensor packed, int[] cfg, int mode, int embed_dim, int n_speakers, Tensor mel, Tensor? speaker_ids, "
        "Tensor z, float sigma, int[] ev_begin, int[] ev_end) -> (Tensor, Tensor)");
  m.def("waveglow_infer_ragged(Tensor packed, int[] cfg, int mode, int embed_dim, int n_speakers, Tensor mel, "
        "Tensor? speaker_ids, Tensor z, float sigma, Tensor lengths) -> (Tensor, Tensor)");
  m.def("waveglow_pack_forward(Tensor[] tensors, str names, int[] cfg) -> Tensor");
  m.def("waveglow_forward(Tensor packed, Tensor packed_fwd, int[] cfg, int mode, int embed_dim, int n_speakers, Tensor mel, "
        "Tensor? speaker_ids, Tensor audio, bool want_log_s) -> (Tensor z, Tensor log_s, Tensor logp_terms, Tensor status)");
  m.def("nonfinite(Tensor x) -> Tensor");
  m.def("waveglow_launch_count(int[] cfg, int mode) -> int", &waveglow_launch_count);
  m.def("abi_version() -> int", &abi_version);
}

TORCH_LIBRARY_IMPL(cookietts_b200, CUDA, m) {
  m.impl("waveglow_pack", &waveglow_pack);
  m.impl("waveglow_infer", &waveglow_infer);
  m.impl("waveglow_infer_ragged", &waveglow_infer_ragged);
  m.impl("waveglow_pack_forward", &waveglow_pack_forward);
  m.impl("waveglow_forward", &waveglow_forward);
  m.impl("nonfinite", &nonfinite);
}
