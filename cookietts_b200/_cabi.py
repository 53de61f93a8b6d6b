"""ctypes binding of libcwg.so (include/cwg.h).

The product path has NO fallback: if the shared library is missing or a symbol is absent,
importing the binding raises.  Build it with `python __graft_entry__.py` (or
`make -C cookietts_b200/csrc`)."""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("CWG_LIB") or os.path.join(_HERE, "libcwg.so")    # CWG_LIB: A/B builds of the kernels

MODE_FFMA, MODE_BF16X3, MODE_BF16, MODE_F16F8 = 0, 1, 2, 3
MODES = {"ffma": MODE_FFMA, "bf16x3": MODE_BF16X3, "bf16": MODE_BF16, "f16f8": MODE_F16F8}
EO_PAD = 16          # narrow layout; see packing.group_pad / include/cwg.h CWG_GROUP_PAD
MAX_GROUP = 32
RAGGED_MAX_BATCH = 1024  # include/cwg.h CWG_RAGGED_MAX_BATCH
ABI_VERSION = 5


class CwgConfig(C.Structure):
    _fields_ = [(n, C.c_int32) for n in (
        "n_mel", "n_flows", "n_group", "n_early_every", "n_early_size", "win_length",
        "hop_length", "n_layers", "n_channels", "kernel_size", "cond_hidden")]


WEIGHT_FIELDS = ("cond_w_f32", "cond_w_hi", "cond_w_lo", "w1_f32", "w1_hi", "w1_lo", "b1",
                 "w2_f32", "w2_hi", "w2_lo", "b2", "eo_b", "start_w", "start_b", "winv", "w1_h8", "w1_l8", "w2_h8", "w2_l8")


WEIGHT_FIELDS_V3 = ("cond_b_base", "cond_w_spk", "spk_embed", "w0_hi", "w0_lo")


class CwgWeights(C.Structure):
    _fields_ = ([(n, C.c_void_p) for n in WEIGHT_FIELDS + WEIGHT_FIELDS_V3]
                + [("speaker_embed_dim", C.c_int32), ("n_speakers", C.c_int32)])


class CwgTensor(C.Structure):
    """cwg_tensor: one state_dict entry (device fp32 data)"""
    _fields_ = [("name", C.c_char_p), ("data", C.c_void_p), ("ndim", C.c_int32), ("shape", C.c_int64 * 4)]


EXPORTS = ("cwg_abi_version", "cwg_last_error", "cwg_workspace_bytes", "cwg_launch_count",
           "cwg_state_dict_info", "cwg_packed_bytes", "cwg_pack_workspace_bytes", "cwg_pack_weights", "cwg_packed_view",
           "cwg_cond_bias", "cwg_nonfinite", "cwg_infer_status", "cwg_infer", "cwg_infer_profiled", "cwg_cond", "cwg_wn_layer", "cwg_flow_boundary",
           "cwg_ax_workspace_bytes", "cwg_ax_infer", "cwg_ax_speaker_bias",
           "cwg_wf_workspace_bytes", "cwg_wf_infer", "cwg_wf_infer_profiled", "cwg_wf_launch_count", "cwg_wf_layer",
           "cwg_wf_forward_workspace_bytes", "cwg_wf_forward_launch_count", "cwg_wf_forward", "cwg_wf_forward_layer",
           "cwg_denoise_workspace_bytes", "cwg_denoise_out_samples", "cwg_stft_mean_magnitude", "cwg_denoise", "cwg_pcm16",
           "cwg_conv1d", "cwg_conv_transpose1d", "cwg_resample1d", "cwg_deemphasis",
           "cwg_fd_workspace_bytes", "cwg_fd_launch_count", "cwg_fd_inverse",
           "cwg_axg_workspace_bytes", "cwg_axg_launch_count", "cwg_axg_flow", "cwg_group_transpose",
           "cwg_pack_forward", "cwg_forward_workspace_bytes", "cwg_forward_launch_count", "cwg_forward",
           "cwg_ax_forward_workspace_bytes", "cwg_ax_forward_launch_count", "cwg_ax_forward",
           "cwg_ragged_workspace_bytes", "cwg_infer_ragged", "cwg_ragged_pairs")


class CwgError(RuntimeError):
    pass


_lib = None


def load():
    """Load libcwg.so once; raises if it is missing (no CPU fallback exists)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise CwgError(f"{LIB_PATH} not found - build the CUDA extension first "
                       f"(python -c 'import __graft_entry__ as g; g.build()')")
    lib = C.CDLL(LIB_PATH)
    for name in EXPORTS:
        if not hasattr(lib, name):
            raise CwgError(f"libcwg.so does not export {name}")
    lib.cwg_abi_version.restype = C.c_int
    lib.cwg_last_error.restype = C.c_char_p
    lib.cwg_workspace_bytes.restype = C.c_size_t
    lib.cwg_workspace_bytes.argtypes = [C.POINTER(CwgConfig), C.c_int, C.c_int, C.c_int]
    lib.cwg_launch_count.restype = C.c_int
    lib.cwg_state_dict_info.restype = C.c_int
    lib.cwg_state_dict_info.argtypes = [C.POINTER(CwgTensor), C.c_int, C.POINTER(C.c_int), C.POINTER(C.c_int), C.POINTER(C.c_int)]
    lib.cwg_packed_bytes.restype = C.c_size_t
    lib.cwg_packed_bytes.argtypes = [C.POINTER(CwgConfig), C.c_int, C.c_int, C.c_int]
    lib.cwg_pack_workspace_bytes.restype = C.c_size_t
    lib.cwg_pack_workspace_bytes.argtypes = [C.POINTER(CwgConfig), C.c_int]
    lib.cwg_pack_weights.restype = C.c_int
    lib.cwg_pack_weights.argtypes = [C.POINTER(CwgConfig), C.c_int, C.POINTER(CwgTensor), C.c_int, C.c_void_p, C.c_size_t,
                                     C.c_void_p, C.c_size_t, C.POINTER(CwgWeights), C.c_void_p]
    lib.cwg_packed_view.restype = C.c_int
    lib.cwg_packed_view.argtypes = [C.POINTER(CwgConfig), C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_size_t, C.POINTER(CwgWeights)]
    lib.cwg_nonfinite.restype = C.c_int
    lib.cwg_nonfinite.argtypes = [C.c_void_p, C.c_size_t, C.c_void_p, C.c_void_p]
    lib.cwg_infer_status.restype = C.c_int
    lib.cwg_infer_status.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p]
    lib.cwg_cond_bias.restype = C.c_int
    lib.cwg_cond_bias.argtypes = [C.POINTER(CwgConfig), C.POINTER(CwgWeights), C.c_void_p, C.c_int, C.c_void_p, C.c_void_p]
    lib.cwg_launch_count.argtypes = [C.POINTER(CwgConfig), C.c_int]
    lib.cwg_infer.restype = C.c_int
    lib.cwg_infer.argtypes = [C.POINTER(CwgConfig), C.POINTER(CwgWeights), C.c_int,
                              C.c_void_p, C.c_void_p, C.c_void_p, C.c_float,
                              C.c_void_p, C.c_void_p, C.c_size_t, C.c_int, C.c_int, C.c_void_p]
    lib.cwg_infer_profiled.restype = C.c_int
    lib.cwg_infer_profiled.argtypes = lib.cwg_infer.argtypes + [C.POINTER(C.c_void_p), C.POINTER(C.c_void_p), C.c_int]
    lib.cwg_ragged_workspace_bytes.restype = C.c_size_t
    lib.cwg_ragged_workspace_bytes.argtypes = [C.POINTER(CwgConfig), C.c_int, C.c_int, C.c_int]
    lib.cwg_infer_ragged.restype = C.c_int
    lib.cwg_infer_ragged.argtypes = [C.POINTER(CwgConfig), C.POINTER(CwgWeights), C.c_int,
                                     C.c_void_p, C.c_void_p, C.c_void_p, C.c_float, C.c_void_p,
                                     C.c_void_p, C.c_void_p, C.c_size_t, C.c_int, C.c_int, C.c_void_p]
    lib.cwg_ragged_pairs.restype = C.c_int
    lib.cwg_ragged_pairs.argtypes = [C.POINTER(CwgConfig), C.c_void_p, C.c_int, C.c_int, C.c_void_p]
    lib.cwg_cond.restype = C.c_int
    lib.cwg_cond.argtypes = [C.POINTER(CwgConfig), C.POINTER(CwgWeights), C.c_int, C.c_int,
                             C.c_void_p, C.c_void_p, C.c_void_p,
                             C.c_void_p, C.c_size_t, C.c_int, C.c_int, C.c_void_p]
    lib.cwg_wn_layer.restype = C.c_int
    lib.cwg_wn_layer.argtypes = [C.POINTER(CwgConfig), C.POINTER(CwgWeights), C.c_int, C.c_int, C.c_int,
                                 C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                 C.c_void_p, C.c_size_t, C.c_int, C.c_int, C.c_void_p]
    lib.cwg_flow_boundary.restype = C.c_int
    lib.cwg_flow_boundary.argtypes = [C.POINTER(CwgConfig), C.POINTER(CwgWeights), C.c_int,
                                      C.c_int, C.c_int, C.c_void_p, C.c_float,
                                      C.c_void_p, C.c_void_p, C.c_void_p,
                                      C.c_int, C.c_int, C.c_void_p]
    lib.cwg_pack_forward.restype = C.c_int
    lib.cwg_pack_forward.argtypes = [C.POINTER(CwgConfig), C.POINTER(CwgTensor), C.c_int, C.c_void_p, C.c_void_p, C.c_void_p]
    lib.cwg_forward_workspace_bytes.restype = C.c_size_t
    lib.cwg_forward_workspace_bytes.argtypes = [C.POINTER(CwgConfig), C.c_int, C.c_int, C.c_int, C.c_int]
    lib.cwg_forward_launch_count.restype = C.c_int
    lib.cwg_forward_launch_count.argtypes = [C.POINTER(CwgConfig), C.c_int]
    lib.cwg_forward.restype = C.c_int
    lib.cwg_forward.argtypes = [C.POINTER(CwgConfig), C.POINTER(CwgWeights), C.c_void_p, C.c_void_p, C.c_int,
                                C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p,
                                C.c_void_p, C.c_size_t, C.c_int, C.c_int, C.c_void_p]
    lib.cwg_denoise_workspace_bytes.restype = C.c_size_t
    lib.cwg_denoise_workspace_bytes.argtypes = [C.c_int] * 4
    lib.cwg_denoise_out_samples.restype = C.c_int
    lib.cwg_denoise_out_samples.argtypes = [C.c_int] * 3
    lib.cwg_stft_mean_magnitude.restype = C.c_int
    lib.cwg_stft_mean_magnitude.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p,
                                            C.c_void_p, C.c_size_t, C.c_void_p]
    lib.cwg_denoise.restype = C.c_int
    lib.cwg_denoise.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p,
                                C.c_void_p, C.c_void_p, C.c_float, C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p]
    lib.cwg_pcm16.restype = C.c_int
    lib.cwg_pcm16.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_void_p]
    lib.cwg_conv1d.restype = C.c_int
    lib.cwg_conv1d.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int,
                               C.c_int, C.c_int, C.c_float, C.c_float, C.c_void_p, C.c_void_p, C.c_void_p]
    lib.cwg_conv_transpose1d.restype = C.c_int
    lib.cwg_conv_transpose1d.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_int, C.c_int,
                                         C.c_int, C.c_int, C.c_int, C.c_float, C.c_float, C.c_void_p, C.c_void_p]
    lib.cwg_resample1d.restype = C.c_int
    lib.cwg_resample1d.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_longlong, C.c_void_p, C.c_int,
                                   C.c_longlong, C.c_int, C.c_int, C.c_int, C.c_float, C.c_int, C.c_void_p]
    lib.cwg_deemphasis.restype = C.c_int
    lib.cwg_deemphasis.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_double, C.c_int, C.c_void_p, C.c_void_p]
    if lib.cwg_abi_version() != ABI_VERSION:
        raise CwgError(f"libcwg.so ABI {lib.cwg_abi_version()} != binding ABI {ABI_VERSION}; rebuild")
    _lib = lib
    return lib


def check(rc: int):
    if rc != 0:
        raise CwgError(f"libcwg error {rc}: {load().cwg_last_error().decode()}")


def make_config(pc) -> CwgConfig:
    return CwgConfig(n_mel=pc.n_mel, n_flows=pc.n_flows, n_group=pc.n_group,
                     n_early_every=pc.n_early_every, n_early_size=pc.n_early_size,
                     win_length=pc.win_length, hop_length=pc.hop_length, n_layers=pc.n_layers,
                     n_channels=pc.n_channels, kernel_size=pc.kernel_size, cond_hidden=pc.cond_hidden)
