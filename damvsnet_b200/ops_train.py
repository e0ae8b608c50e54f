"""Tensor-level wrappers over the training-path entry points of the C ABI (include/damvs.h):
BatchNorm statistics / apply / backward, convolution weight gradients, head backward, and the forward /
backward kernels of the fused warp + aggregation and of the fused warp + group-wise correlation.  Same conventions
as ``ops.py``: CUDA tensors in, outputs allocated with torch, torch's current stream, no fallback.
"""
from __future__ import annotations

import ctypes
from typing import List, Optional, Sequence, Tuple

import torch

from . import _lib
from .ops import AGG_ADAPTIVE, AGG_VARIANCE, _dt, _hyp_flags, _p, _stream, conv_desc

_VOL_DTYPES = (torch.float32, torch.bfloat16)


def _vol_dims(t: torch.Tensor) -> Tuple[int, int, int, int, int]:
    if t.dim() != 6 or t.shape[-1] != 8 or t.dtype not in _VOL_DTYPES or not t.is_cuda or not t.is_contiguous():
        raise ValueError("expected a contiguous CUDA G8 volume [B,C/8,D,H,W,8] in fp32 or bf16")
    b, g, d, h, w, _ = t.shape
    return b, g * 8, d, h, w


def _f32c(t: Optional[torch.Tensor], n: int, name: str) -> Optional[torch.Tensor]:
    if t is None:
        return None
    if t.dtype != torch.float32 or t.numel() != n or not t.is_cuda:
        raise ValueError(f"{name}: expected {n} fp32 CUDA values")
    return t.contiguous()


# --------------------------------------------------------------------------
# BatchNorm pieces
# --------------------------------------------------------------------------
def bn_stats(y: torch.Tensor) -> torch.Tensor:
    """G8 volume -> fp64 [C,2] = per-channel (sum y, sum y^2) over (B,D,H,W)."""
    b, c, d, h, w = _vol_dims(y)
    sums = torch.zeros((c, 2), dtype=torch.float64, device=y.device)
    with torch.cuda.device_of(y):
        _lib.check(_lib.load().damvs_bn_stats(_p(y), _dt(y.dtype), b, c, d, h, w, _p(sums), _stream()))
    return sums


def bn_apply(y: torch.Tensor, scale: torch.Tensor, shift: torch.Tensor, skip: Optional[torch.Tensor], relu: bool) -> torch.Tensor:
    """out = skip + act(y * scale[c] + shift[c])."""
    b, c, d, h, w = _vol_dims(y)
    if skip is not None and (skip.shape != y.shape or skip.dtype != y.dtype):
        raise ValueError("skip volume must match y")
    out = torch.empty_like(y)
    with torch.cuda.device_of(y):
        _lib.check(_lib.load().damvs_bn_apply(_p(y), _p(_f32c(scale, c, "scale")), _p(_f32c(shift, c, "shift")),
                                              _p(None if skip is None else skip.contiguous()), _p(out), _dt(y.dtype),
                                              b, c, d, h, w, int(relu), _stream()))
    return out


def bn_bwd(g_out: torch.Tensor, y: torch.Tensor, scale, shift, k1, k2, k3, relu: bool, want_gy: bool, want_sums: bool):
    """See damvs_bn_bwd: returns (g_y | None, sums fp64 [C,2] | None)."""
    b, c, d, h, w = _vol_dims(y)
    if g_out.shape != y.shape or g_out.dtype != y.dtype:
        raise ValueError("g_out must match y")
    g_out = g_out.contiguous()
    g_y = torch.empty_like(y) if want_gy else None
    sums = torch.zeros((c, 2), dtype=torch.float64, device=y.device) if want_sums else None
    with torch.cuda.device_of(y):
        _lib.check(_lib.load().damvs_bn_bwd(_p(g_out), _p(y), _p(_f32c(scale, c, "scale")), _p(_f32c(shift, c, "shift")),
                                            _p(_f32c(k1, c, "k1")), _p(_f32c(k2, c, "k2")), _p(_f32c(k3, c, "k3")),
                                            _p(g_y), _p(sums), _dt(y.dtype), b, c, d, h, w, int(relu), _stream()))
    return g_y, sums


def bn_finalize(sums: torch.Tensor, gamma, beta, running_mean, running_var, count: int, momentum: float, eps: float):
    """sums fp64 [C,2] -> (scale, shift, mean, rstd) fp32 [C]; running buffers (or None) updated in place."""
    c = sums.shape[0]
    dev = sums.device
    scale, shift, mean, rstd = (torch.empty(c, dtype=torch.float32, device=dev) for _ in range(4))
    with torch.cuda.device_of(sums):
        _lib.check(_lib.load().damvs_bn_finalize(_p(sums), _p(_f32c(gamma, c, "gamma")), _p(_f32c(beta, c, "beta")), _p(running_mean),
                                                 _p(running_var), float(count), float(momentum), float(eps), _p(scale), _p(shift),
                                                 _p(mean), _p(rstd), c, _stream()))
    return scale, shift, mean, rstd


def bn_bwd_coeffs(sums: torch.Tensor, scale, mean, rstd, count: int, batch_stats: bool):
    """sums fp64 [C,2] -> (k1, k2, k3 | None x3, g_gamma, g_beta) fp32 [C]."""
    c = sums.shape[0]
    dev = sums.device
    g_gamma, g_beta = (torch.empty(c, dtype=torch.float32, device=dev) for _ in range(2))
    k1 = k2 = k3 = None
    if batch_stats:
        k1, k2, k3 = (torch.empty(c, dtype=torch.float32, device=dev) for _ in range(3))
    with torch.cuda.device_of(sums):
        _lib.check(_lib.load().damvs_bn_bwd_coeffs(_p(sums), _p(scale), _p(mean), _p(rstd), float(count), _p(k1), _p(k2), _p(k3),
                                                   _p(g_gamma), _p(g_beta), c, _stream()))
    return k1, k2, k3, g_gamma, g_beta


def plain_to_g8(t: torch.Tensor, dtype: torch.dtype) -> torch.Tensor:
    """[B,D,H,W] fp32 -> G8 volume [B,1,D,H,W,8] (channel 0 = value, the rest zero)."""
    if t.dtype != torch.float32 or t.dim() != 4 or not t.is_cuda:
        raise ValueError("expected a CUDA fp32 [B,D,H,W] tensor")
    t = t.contiguous()
    b, d, h, w = t.shape
    out = torch.empty((b, 1, d, h, w, 8), dtype=dtype, device=t.device)
    with torch.cuda.device_of(t):
        _lib.check(_lib.load().damvs_plain_to_g8(_p(t), _p(out), _dt(dtype), t.numel(), _stream()))
    return out


# --------------------------------------------------------------------------
# convolution weight gradient / head backward
# --------------------------------------------------------------------------
def conv3d_wgrad(x: torch.Tensor, g_y: torch.Tensor, cin: int, cout: int, stride: int, transposed: bool) -> torch.Tensor:
    """dW in PyTorch layout ([Cout,Cin,3,3,3], transposed [Cin,Cout,3,3,3]) from G8 x and g_y.  For cout < 8
    g_y carries one zero-padded channel group (plain_to_g8)."""
    b, cx, d, h, w = _vol_dims(x)
    _vol_dims(g_y)
    if cx != cin:
        raise ValueError("x channel mismatch")
    desc = conv_desc(b, cin, cout, d, h, w, stride, transposed, 0, x.dtype, g_y.dtype, False, 0)
    shape = (cin, cout, 3, 3, 3) if transposed else (cout, cin, 3, 3, 3)
    dw = torch.empty(shape, dtype=torch.float32, device=x.device)
    with torch.cuda.device_of(x):
        _lib.check(_lib.load().damvs_conv3d_wgrad(ctypes.byref(desc), _p(x), _p(g_y.contiguous()), _p(dw), _stream()))
    return dw


def softmax_regress_bwd(prob, depth_values, depth, g_depth, g_var, g_prob, want_hyp_grad: bool = False):
    """Gradients of (depth, variance, prob_volume) w.r.t. the logits (and optionally per-pixel hypotheses)."""
    b, d, h, w = prob.shape
    dv, per_pixel, _ = _hyp_flags(depth_values, b, h, w)
    g_logits = torch.empty_like(prob)
    g_hyp = torch.empty_like(prob) if (want_hyp_grad and per_pixel) else None

    def c(t):
        return None if t is None else t.contiguous().float()

    with torch.cuda.device_of(prob):
        _lib.check(_lib.load().damvs_softmax_regress_bwd(_p(prob.contiguous()), _p(dv), _p(depth.contiguous()), _p(c(g_depth)),
                                                         _p(c(g_var)), _p(c(g_prob)), _p(g_logits), _p(g_hyp), b, d, h, w,
                                                         per_pixel, _stream()))
    return g_logits, g_hyp


# --------------------------------------------------------------------------
# warp + aggregation, training kernels
# --------------------------------------------------------------------------
def _ptrs(ts: Sequence[torch.Tensor]):
    return (ctypes.c_void_p * len(ts))(*[t.data_ptr() for t in ts])


def _warp_common(ref: torch.Tensor, srcs: Sequence[torch.Tensor], rot_trans: torch.Tensor, depth_values: torch.Tensor):
    b, h, w, c = ref.shape
    for s in srcs:
        if s.shape != ref.shape or not s.is_contiguous() or s.dtype != torch.float32:
            raise ValueError("source features must be contiguous fp32 NHWC shaped like the reference feature")
    if tuple(rot_trans.shape) != (len(srcs), b, 12):
        raise ValueError("rot_trans must be [n_src,B,12]")
    dv, per_pixel, d = _hyp_flags(depth_values, b, h, w)
    return b, h, w, c, d, dv, per_pixel


def warp_agg_bwd(ref, srcs, rot_trans, depth_values, wnet, g_vol: torch.Tensor, mode: str):
    """Backward of ops.warp_aggregate with a per-voxel (eval-mode) view-weight net: (g_ref, [g_src], g_wnet | None)."""
    b, h, w, c, d, dv, per_pixel = _warp_common(ref, srcs, rot_trans, depth_values)
    g_ref = torch.empty_like(ref)
    g_srcs = [torch.zeros_like(s) for s in srcs]
    g_wnet = torch.zeros(c + 5, dtype=torch.float32, device=ref.device) if mode == "adaptive" else None
    m = AGG_ADAPTIVE if mode == "adaptive" else AGG_VARIANCE
    with torch.cuda.device_of(ref):
        _lib.check(_lib.load().damvs_warp_agg_bwd(_p(ref.contiguous()), _ptrs(srcs), len(srcs), _p(rot_trans.contiguous()), _p(dv),
                                                  _p(wnet), _p(g_vol.contiguous()), _dt(g_vol.dtype), _p(g_ref), _ptrs(g_srcs),
                                                  _p(g_wnet), b, c, d, h, w, m, per_pixel, _stream()))
    return g_ref, g_srcs, g_wnet


def _gwc_common(ref, srcs, rot_trans, depth_values, groups: int):
    b, h, w, c, d, dv, per_pixel = _warp_common(ref, srcs, rot_trans, depth_values)
    if c not in (8, 16, 32) or groups not in (4, 8, 16, 32) or groups > c:
        raise ValueError(f"group-wise correlation needs C in (8,16,32), groups in (4,8,16,32) and groups <= C; got C={c}, groups={groups}")
    return b, h, w, c, d, dv, per_pixel


def warp_gwc_train_fwd(ref, srcs, rot_trans, depth_values, groups: int, out_dtype: torch.dtype) -> torch.Tensor:
    """Group-wise correlation at the training kernels' sampling coordinates -> G8 data tensor of max(groups, 8)
    channels (fp32 or bf16; for groups = 4 channels 4..7 are zero)."""
    b, h, w, c, d, dv, per_pixel = _gwc_common(ref, srcs, rot_trans, depth_values, groups)
    if out_dtype not in _VOL_DTYPES:
        raise ValueError("out_dtype must be fp32 or bf16")
    out = torch.empty((b, max(groups, 8) // 8, d, h, w, 8), dtype=out_dtype, device=ref.device)
    with torch.cuda.device_of(ref):
        _lib.check(_lib.load().damvs_warp_gwc_train_fwd(_p(ref.contiguous()), _ptrs(srcs), len(srcs), _p(rot_trans.contiguous()), _p(dv),
                                                        _p(out), b, c, groups, d, h, w, per_pixel, _dt(out_dtype), _stream()))
    return out


def warp_gwc_bwd(ref, srcs, rot_trans, depth_values, g_vol: torch.Tensor, groups: int):
    """Backward of warp_gwc_train_fwd: (g_ref, [g_src]).  The padding channels of a groups = 4 g_vol are ignored."""
    b, h, w, c, d, dv, per_pixel = _gwc_common(ref, srcs, rot_trans, depth_values, groups)
    g_vol = g_vol.contiguous()
    if _vol_dims(g_vol) != (b, max(groups, 8), d, h, w):
        raise ValueError(f"g_vol must be a G8 volume [B,{max(groups, 8) // 8},D,H,W,8]")
    g_ref = torch.empty_like(ref)
    g_srcs = [torch.zeros_like(s) for s in srcs]
    with torch.cuda.device_of(ref):
        _lib.check(_lib.load().damvs_warp_gwc_bwd(_p(ref.contiguous()), _ptrs(srcs), len(srcs), _p(rot_trans.contiguous()), _p(dv),
                                                  _p(g_vol), _dt(g_vol.dtype), _p(g_ref), _ptrs(g_srcs), b, c, groups, d, h, w,
                                                  per_pixel, _stream()))
    return g_ref, g_srcs


def warp_score_fwd(ref, srcs, rot_trans, depth_values, w1: torch.Tensor) -> torch.Tensor:
    """s[v,b,d,y,x] = sum_c w1[c] (ref - warp_v)[c]^2 -> fp32 [n_src,B,D,H,W]."""
    b, h, w, c, d, dv, per_pixel = _warp_common(ref, srcs, rot_trans, depth_values)
    s_vol = torch.empty((len(srcs), b, d, h, w), dtype=torch.float32, device=ref.device)
    with torch.cuda.device_of(ref):
        _lib.check(_lib.load().damvs_warp_score_fwd(_p(ref.contiguous()), _ptrs(srcs), len(srcs), _p(rot_trans.contiguous()), _p(dv),
                                                    _p(_f32c(w1, c, "w1")), _p(s_vol), b, c, d, h, w, per_pixel, _stream()))
    return s_vol


def warp_weighted_fwd(ref, srcs, rot_trans, depth_values, wt_vol: torch.Tensor, out_dtype: torch.dtype) -> torch.Tensor:
    """vol = sum_v (wt_v + 1) (ref - warp_v)^2 / n_src -> G8 data tensor."""
    b, h, w, c, d, dv, per_pixel = _warp_common(ref, srcs, rot_trans, depth_values)
    if tuple(wt_vol.shape) != (len(srcs), b, d, h, w) or wt_vol.dtype != torch.float32:
        raise ValueError("wt_vol must be fp32 [n_src,B,D,H,W]")
    out = torch.empty((b, c // 8, d, h, w, 8), dtype=out_dtype, device=ref.device)
    with torch.cuda.device_of(ref):
        _lib.check(_lib.load().damvs_warp_weighted_fwd(_p(ref.contiguous()), _ptrs(srcs), len(srcs), _p(rot_trans.contiguous()), _p(dv),
                                                       _p(wt_vol.contiguous()), _p(out), b, c, d, h, w, per_pixel, _dt(out_dtype),
                                                       _stream()))
    return out


def warp_gwt(ref, srcs, rot_trans, depth_values, g_vol) -> torch.Tensor:
    """d loss / d wt_v = sum_c g_vol[c] (ref - warp_v)[c]^2 / n_src -> fp32 [n_src,B,D,H,W]; no feature gradients."""
    b, h, w, c, d, dv, per_pixel = _warp_common(ref, srcs, rot_trans, depth_values)
    g_wt = torch.empty((len(srcs), b, d, h, w), dtype=torch.float32, device=ref.device)
    with torch.cuda.device_of(ref):
        _lib.check(_lib.load().damvs_warp_gwt(_p(ref.contiguous()), _ptrs(srcs), len(srcs), _p(rot_trans.contiguous()), _p(dv),
                                              _p(g_vol.contiguous()), _dt(g_vol.dtype), _p(g_wt), b, c, d, h, w, per_pixel, _stream()))
    return g_wt


def warp_merged_bwd(ref, srcs, rot_trans, depth_values, w1, wt_vol, g_s_vol, g_vol, g_ref, g_srcs: List[torch.Tensor]) -> torch.Tensor:
    """One scatter for both paths into the features (through the aggregate and through the score); returns g_w1 [C]."""
    b, h, w, c, d, dv, per_pixel = _warp_common(ref, srcs, rot_trans, depth_values)
    g_w1 = torch.zeros(c, dtype=torch.float32, device=ref.device)
    with torch.cuda.device_of(ref):
        _lib.check(_lib.load().damvs_warp_merged_bwd(_p(ref.contiguous()), _ptrs(srcs), len(srcs), _p(rot_trans.contiguous()), _p(dv),
                                                     _p(_f32c(w1, c, "w1")), _p(wt_vol.contiguous()), _p(g_s_vol.contiguous().float()),
                                                     _p(g_vol.contiguous()), _dt(g_vol.dtype), _p(g_ref), _ptrs(g_srcs), _p(g_w1),
                                                     b, c, d, h, w, per_pixel, _stream()))
    return g_w1


def wnet_chain_fwd(s_vol: torch.Tensor, bn1, w2: torch.Tensor, bn2):
    """Scalar tail of the weight net with batch statistics per view: s_vol [n_src,B,D,H,W] -> (wt_vol, state [n_src,8]).
    bn1 / bn2 are the nn.BatchNorm3d(1) modules: their affine parameters are read, their running buffers updated view by
    view (momentum must be a number), num_batches_tracked advanced by n_src."""
    n = s_vol.shape[0]
    m = s_vol.numel() // n
    dev = s_vol.device
    if bn1.momentum is None or bn2.momentum is None or bn1.momentum != bn2.momentum or bn1.eps != bn2.eps:
        raise NotImplementedError("native weight-net chain needs one numeric BatchNorm momentum and eps")
    sums = torch.zeros(4 * n, dtype=torch.float64, device=dev)
    state = torch.empty((n, 8), dtype=torch.float32, device=dev)
    wt = torch.empty_like(s_vol)
    track = bn1.track_running_stats and bn1.running_mean is not None
    with torch.no_grad():
        if track:
            bn1.num_batches_tracked += n
            bn2.num_batches_tracked += n
    with torch.cuda.device_of(s_vol):
        _lib.check(_lib.load().damvs_wnet_chain_fwd(
            _p(s_vol.contiguous()), n, m, _p(bn1.weight.detach()), _p(bn1.bias.detach()), _p(bn1.running_mean if track else None),
            _p(bn1.running_var if track else None), _p(w2.detach().reshape(-1).float()), _p(bn2.weight.detach()), _p(bn2.bias.detach()),
            _p(bn2.running_mean if track else None), _p(bn2.running_var if track else None), float(bn1.momentum), float(bn1.eps),
            _p(sums), _p(state), _p(wt), _stream()))
    return wt, state


def wnet_chain_bwd(s_vol: torch.Tensor, g_wt: torch.Tensor, state: torch.Tensor, w2: torch.Tensor):
    """Backward of wnet_chain_fwd: (g_s [n_src,B,D,H,W], g_params [5] = d gamma1, d beta1, d w2, d gamma2, d beta2)."""
    n = s_vol.shape[0]
    m = s_vol.numel() // n
    dev = s_vol.device
    sums = torch.zeros(4 * n + 2, dtype=torch.float64, device=dev)
    coef = torch.empty((n, 6), dtype=torch.float32, device=dev)
    g_s = torch.empty_like(s_vol)
    g_params = torch.empty(5, dtype=torch.float32, device=dev)
    with torch.cuda.device_of(s_vol):
        _lib.check(_lib.load().damvs_wnet_chain_bwd(_p(s_vol.contiguous()), _p(g_wt.contiguous()), n, m, _p(state), _p(w2.detach().reshape(-1).float()),
                                                    _p(sums), _p(coef), _p(g_s), _p(g_params), _stream()))
    return g_s, g_params
