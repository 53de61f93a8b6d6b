"""fp64 numpy statement of cwg_axg_flow (csrc/cwg_fd.cu), the general fp32 mode's one-flow call, on the packed arrays of
cookietts_b200.waveglow_ax.pack_ax_general.  Pinned to the reference goldens on the CPU by tests/test_ax_general_packing.py;
the kernels are held to it at larger shapes on the GPU by tests/test_gpu_fp32_shapes.py."""
import numpy as np

from oracle.waveglow_ax_oracle import GATED_UNITS as ORACLE_UNITS


def _mm(w, x):
    return np.einsum("oc,bct->bot", w.astype(np.float64), x, optimize=True)


def flow_packed(pk, cfg, n_rem, c_all, z, ignore_nan=False):
    """cwg_axg_flow on channels-first z [B, G, T] (in place), c_all [B, 2CL, T].  With `ignore_nan` a NaN coming out of
    the coupling becomes 0 before the mixing (efficient_model_ax.py:331-332)."""
    G, C, L, ks = cfg.n_group, cfg.n_channels, cfg.n_layers, cfg.kernel_size
    nh, off = n_rem // 2, G - n_rem
    T = z.shape[2]
    ua, ub = ORACLE_UNITS[cfg.gated_unit.upper()]

    def mix():
        z[:, off:] = _mm(pk["winv"], z[:, off:])
    if not cfg.mix_first:
        mix()
    h = _mm(pk["start_w"], z[:, off:off + nh]) + pk["start_b"][None, :, None]
    out = np.zeros_like(h)
    split = cfg.res_skip and not cfg.merge_res_skip
    for i in range(L):
        d = cfg.dilation(i)
        pad = d * (ks // 2)
        hp = np.pad(h, ((0, 0), (0, 0), (pad, pad)))
        pre = np.zeros((z.shape[0], 2 * C, T))
        for j in range(ks):
            pre += _mm(pk["in_w"][i, :, :, j], hp[:, :, j * d:j * d + T])
        pre += pk["in_b"][i][None, :, None] + c_all[:, 2 * C * i:2 * C * (i + 1)]
        acts = ua(pre[:, :C]) * ub(pre[:, C:])
        if cfg.res_skip:
            rs = _mm(pk["rs_w"][i], acts) + pk["rs_b"][i][None, :, None]
            if split and i < L - 1:
                h = h + rs[:, :C]
                out += rs[:, C:]
            else:
                out += rs[:, :C]
        else:
            out += acts
    e = _mm(pk["end_w"], out) + pk["end_b"][None, :, None]
    z[:, off + nh:] = (z[:, off + nh:] - e[:, nh:]) / np.exp(e[:, :nh])
    if ignore_nan:
        z[:, off + nh:] = np.where(np.isnan(z[:, off + nh:]), 0.0, z[:, off + nh:])
    if cfg.mix_first:
        mix()
