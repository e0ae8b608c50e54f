"""Host-side mirror of the reference's ``models/module.py`` for the hot path.

Same names, constructor arguments, parameter/buffer names (so reference
checkpoints load with ``strict=True``) and call signatures as the reference:
``Conv3d``, ``Deconv3d``, ``CostRegNet``, ``AggWeightNetVolume``,
``homo_warping``, ``depth_regression``.  The arithmetic runs in the CUDA library
behind include/damvs.h; parameters stay ordinary fp32 ``nn.Parameter``s in
PyTorch layout and are repacked (BatchNorm folded, weights reordered / cast)
into a per-module cache keyed on the parameters' version counters.

Inference (``eval()`` under ``no_grad``) runs the fused kernels (BatchNorm folded into the
convolution epilogue).  With gradients enabled, or in ``train()`` mode (batch statistics),
the blocks run through ``damvsnet_b200.autograd``: raw convolution -> statistics ->
normalise/ReLU/skip, with native backward kernels.
"""
from __future__ import annotations

from typing import Dict, Optional, Tuple

import torch
import torch.nn as nn

from . import autograd as ag
from . import ops
from .ops import G8Volume

__all__ = ["Conv3d", "Deconv3d", "CostRegNet", "AggWeightNetVolume", "homo_warping", "depth_regression",
           "uncertainty_aware_samples", "invalidate_packed"]

# Packed-weight / folded-BatchNorm caches are keyed on (epoch, data_ptr, tensor._version) of every tensor they were
# built from.  In-place writes through autograd-visible ops (optimizer steps, load_state_dict, copy_ under no_grad)
# bump `_version`; module moves (`.to()`, `.cuda()`, DataParallel replication through `_apply`) bump the epoch here.
# Writes that bypass both -- `p.data.copy_(...)`, `dist.broadcast(p.data)`, EMA swaps through `.data` -- do NOT bump
# `_version`: call `invalidate_packed()` after them (damvsnet_b200.training.broadcast_module_state does).
_EPOCH = [0]


def invalidate_packed() -> None:
    """Drop every cached packed weight / folded BatchNorm of this process (they are rebuilt on next use).  Needed only
    after parameters or BatchNorm buffers were written through `.data` (which leaves `tensor._version` unchanged)."""
    _EPOCH[0] += 1


class _EpochOnApply(nn.Module):
    """Mixin: `module._apply` (device / dtype moves, DataParallel replicas) invalidates the caches, because a moved
    parameter can land at a recycled address with a `_version` that matches a stale cache entry."""

    def _apply(self, fn, *args, **kwargs):
        invalidate_packed()
        return super()._apply(fn, *args, **kwargs)


def _bn_affine(bn: nn.BatchNorm3d) -> Tuple[torch.Tensor, torch.Tensor]:
    """Eval-mode BatchNorm as (scale, shift) (reference models/module.py:141,150; SURVEY.md appendix A)."""
    scale = bn.weight.detach() / torch.sqrt(bn.running_var + bn.eps)
    shift = bn.bias.detach() - bn.running_mean * scale
    return scale.float().contiguous(), shift.float().contiguous()


def _versions(*tensors) -> tuple:
    return (_EPOCH[0],) + tuple((t.data_ptr(), t._version) for t in tensors if t is not None)


class _ConvBlock(_EpochOnApply):
    """Shared machinery of Conv3d / Deconv3d: parameters as in the reference, packed-weight cache."""

    transposed = False

    def _init_cache(self):
        self._packed: Dict[tuple, tuple] = {}

    def _cached(self, key, ver, make):
        hit = self._packed.get(key)
        if hit is not None and hit[0] == ver:
            return hit[1]
        val = make()
        self._packed[key] = (ver, val)
        return val

    def packed_weight(self, impl: int) -> torch.Tensor:
        """Packed convolution weights alone (no BatchNorm fold): the training path applies BatchNorm separately."""
        w = self.conv.weight
        return self._cached(("w", impl, w.device), _versions(w), lambda: ops.conv3d_pack_weight(
            w.detach().float(), self.in_channels, self.out_channels, self.transposed, impl, self.stride))

    def packed_adjoint(self, impl: int) -> torch.Tensor:
        """Packed weights of the adjoint convolution (data gradient).  Stride-1: transposed + flipped weights;
        stride-2 conv <-> transposed conv share the weight tensor as it is."""
        w = self.conv.weight
        cin, cout = self.in_channels, self.out_channels

        def make():
            wd = w.detach().float()
            if self.transposed:          # adjoint: Conv3d(cout -> cin, stride 2), weight [cin, cout, ...] as is
                return ops.conv3d_pack_weight(wd.contiguous(), cout, cin, False, impl, 2)
            if self.stride == 2:         # adjoint: ConvTranspose3d(cout -> cin), weight [cout, cin, ...] as is
                return ops.conv3d_pack_weight(wd.contiguous(), cout, cin, True, impl, 2)
            return ops.conv3d_pack_weight(wd.transpose(0, 1).flip(2, 3, 4).contiguous(), cout, cin, False, impl, 1)
        return self._cached(("adj", impl, w.device), _versions(w), make)

    def prepared(self, impl: int, dtype: torch.dtype = torch.bfloat16):
        """(packed weight, scale, shift) for `impl` and volumes of `dtype` on the parameters' device, rebuilt when they
        change (the tcgen05 kernels hold the weights in the volumes' 2-byte type)."""
        w = self.conv.weight
        bn = self.bn
        key = (impl, w.device, dtype if dtype in ops.HALF_DTYPES else None)
        ver = _versions(w, *( (bn.weight, bn.bias, bn.running_mean, bn.running_var) if bn is not None else () ))
        hit = self._packed.get(key)
        if hit is not None and hit[0] == ver:
            return hit[1]
        cin, cout = self.in_channels, self.out_channels
        packed = ops.conv3d_pack_weight(w.detach().float(), cin, cout, self.transposed, impl, self.stride, dtype)
        if bn is not None:
            scale, shift = _bn_affine(bn)
        elif self.conv.bias is not None:
            scale = torch.ones(cout, dtype=torch.float32, device=w.device)
            shift = self.conv.bias.detach().float().contiguous()
        else:
            scale = shift = None
        val = (packed, scale, shift)
        self._packed[key] = (ver, val)
        return val

    def forward_g8(self, vol: G8Volume, skip: Optional[G8Volume] = None, out_dtype: Optional[torch.dtype] = None) -> G8Volume:
        """out = skip + relu(bn(conv(vol))) on G8 volumes (the path CostRegNet uses)."""
        if self.kernel_size != 3:
            raise NotImplementedError("native conv blocks are 3x3x3 only")
        bn = self.bn
        batch_stats = bn is not None and (self.training or not bn.track_running_stats)
        params = (self.conv.weight,) + ((bn.weight, bn.bias) if bn is not None else (self.conv.bias,))
        if batch_stats or ag.wants_grad(vol.data, None if skip is None else skip.data, *params):
            if vol.dtype == torch.float16:
                raise NotImplementedError("precision 'fp16' is the inference pipeline; train in 'bf16' or 'fp32'")
            if out_dtype is not None and out_dtype != vol.dtype:
                raise NotImplementedError("training path keeps one volume dtype")
            out = ag.ConvBlockFn.apply(vol.data, None if skip is None else skip.data, self.conv.weight,
                                       None if bn is None else bn.weight, None if bn is None else bn.bias,
                                       self.conv.bias if bn is None else None, self)
            return G8Volume(out)
        impl = ops.conv_impl_for(self.in_channels, self.out_channels, self.stride, self.transposed)
        packed, scale, shift = self.prepared(impl, vol.dtype)
        return ops.conv3d(vol, packed, scale, shift, self.out_channels, self.stride, self.transposed, self.relu, skip,
                          out_dtype or vol.dtype, False, impl)

    def forward(self, x: torch.Tensor) -> torch.Tensor:
        """Reference call signature: [B,C,D,H,W] fp32 in and out (repacked to/from G8 around the kernel)."""
        if self.kernel_size != 3 or x.shape[1] % 8 or self.out_channels % 8 or self._padding != 1:
            raise NotImplementedError(
                "stand-alone Conv3d/Deconv3d forward is native for kernel 3, padding 1, channels % 8 == 0 only; "
                "the 1x1x1 view-weight convs are fused into the warp/aggregate kernel (see DepthNet)")
        vol = G8Volume(ag.NcdhwToG8Fn.apply(x, ops.volume_dtype()))
        return ag.G8ToNcdhwFn.apply(self.forward_g8(vol).data)


class Conv3d(_ConvBlock):
    """3-D convolution + BatchNorm + ReLU block (reference models/module.py:117-159)."""

    def __init__(self, in_channels, out_channels, kernel_size=3, stride=1, relu=True, bn=True, bn_momentum=0.1,
                 init_method="xavier", **kwargs):
        super().__init__()
        self.in_channels = in_channels
        self.out_channels = out_channels
        self.kernel_size = kernel_size
        assert stride in [1, 2]
        self.stride = stride
        self._padding = kwargs.get("padding", 0)
        self.conv = nn.Conv3d(in_channels, out_channels, kernel_size, stride=stride, bias=(not bn), **kwargs)
        self.bn = nn.BatchNorm3d(out_channels, momentum=bn_momentum) if bn else None
        self.relu = relu
        self._init_cache()


class Deconv3d(_ConvBlock):
    """3-D transposed convolution + BatchNorm + ReLU block (reference models/module.py:161-202)."""

    transposed = True

    def __init__(self, in_channels, out_channels, kernel_size=3, stride=1, relu=True, bn=True, bn_momentum=0.1,
                 init_method="xavier", **kwargs):
        super().__init__()
        self.in_channels = in_channels
        self.out_channels = out_channels
        self.kernel_size = kernel_size
        assert stride in [1, 2]
        self.stride = stride
        self._padding = kwargs.get("padding", 0)
        if kernel_size == 3 and not (stride == 2 and kwargs.get("padding", 0) == 1 and kwargs.get("output_padding", 0) == 1):
            raise NotImplementedError("native Deconv3d supports the reference's only configuration: k3, s2, p1, op1")
        self.conv = nn.ConvTranspose3d(in_channels, out_channels, kernel_size, stride=stride, bias=(not bn), **kwargs)
        self.bn = nn.BatchNorm3d(out_channels, momentum=bn_momentum) if bn else None
        self.relu = relu
        self._init_cache()


class CostRegNet(_EpochOnApply):
    """3-level 3-D U-Net regulariser (reference models/module.py:510-541)."""

    def __init__(self, in_channels, base_channels):
        super().__init__()
        self.conv0 = Conv3d(in_channels, base_channels, padding=1)
        self.conv1 = Conv3d(base_channels, base_channels * 2, stride=2, padding=1)
        self.conv2 = Conv3d(base_channels * 2, base_channels * 2, padding=1)
        self.conv3 = Conv3d(base_channels * 2, base_channels * 4, stride=2, padding=1)
        self.conv4 = Conv3d(base_channels * 4, base_channels * 4, padding=1)
        self.conv5 = Conv3d(base_channels * 4, base_channels * 8, stride=2, padding=1)
        self.conv6 = Conv3d(base_channels * 8, base_channels * 8, padding=1)
        self.conv7 = Deconv3d(base_channels * 8, base_channels * 4, stride=2, padding=1, output_padding=1)
        self.conv9 = Deconv3d(base_channels * 4, base_channels * 2, stride=2, padding=1, output_padding=1)
        self.conv11 = Deconv3d(base_channels * 2, base_channels * 1, stride=2, padding=1, output_padding=1)
        self.prob = nn.Conv3d(base_channels, 1, 3, stride=1, padding=1, bias=False)
        self.in_channels = in_channels
        self.base_channels = base_channels
        self._prob_packed: Dict[tuple, tuple] = {}

    def _prob_prepared(self, impl: int, dtype: torch.dtype = torch.bfloat16) -> torch.Tensor:
        w = self.prob.weight
        key = (impl, w.device, dtype if dtype in ops.HALF_DTYPES else None)
        ver = _versions(w)
        hit = self._prob_packed.get(key)
        if hit is not None and hit[0] == ver:
            return hit[1]
        packed = ops.conv3d_pack_weight(w.detach().float(), self.base_channels, 1, False, impl, 1, dtype)
        self._prob_packed[key] = (ver, packed)
        return packed

    def _prob_adjoint(self, impl: int) -> torch.Tensor:
        """Packed weights of the adjoint of `prob`: Conv3d(8 (zero-padded from 1) -> base_channels)."""
        w = self.prob.weight
        key = ("adj", impl, w.device)
        ver = _versions(w)
        hit = self._prob_packed.get(key)
        if hit is not None and hit[0] == ver:
            return hit[1]
        wd = w.detach().float()                                              # [1, C, 3,3,3]
        padded = torch.zeros((8,) + tuple(wd.shape[1:]), dtype=torch.float32, device=w.device)
        padded[:1] = wd
        packed = ops.conv3d_pack_weight(padded.transpose(0, 1).flip(2, 3, 4).contiguous(), 8, self.base_channels, False, impl)
        self._prob_packed[key] = (ver, packed)
        return packed

    def forward_g8(self, vol: G8Volume, head_hypotheses: Optional[torch.Tensor] = None):
        """G8 cost volume -> logits [B,D,H,W] fp32 (the squeeze(1) of the reference output).

        With `head_hypotheses` = per-pixel depth_values [B,D,H,W] (inference only) and ops.set_fusion(prob_head=True),
        the last layer runs fused with the softmax / regression head when the shape qualifies and the call returns the tuple
        (prob_volume, depth, photometric_confidence, variance) instead of logits -- callers check the type."""
        b, c, d, h, w = vol.shape
        if c != self.in_channels:
            raise ValueError(f"CostRegNet expects {self.in_channels} channels, got {c}")
        if d % 8 or h % 8 or w % 8:
            raise ValueError(f"CostRegNet needs D,H,W divisible by 8 (three stride-2 levels), got {(d, h, w)}")
        conv0 = self.conv0.forward_g8(vol)
        conv2 = self.conv2.forward_g8(self.conv1.forward_g8(conv0))
        conv4 = self.conv4.forward_g8(self.conv3.forward_g8(conv2))
        x = self.conv6.forward_g8(self.conv5.forward_g8(conv4))
        x = self.conv7.forward_g8(x, skip=conv4)     # conv4 + conv7(x)
        x = self.conv9.forward_g8(x, skip=conv2)
        x = self.conv11.forward_g8(x, skip=conv0)
        if ag.wants_grad(x.data, self.prob.weight):
            return ag.ProbConvFn.apply(x.data, self.prob.weight, self)
        impl = ops.conv_impl_for(self.base_channels, 1, 1, False)
        if ops.fuse_prob_head() and head_hypotheses is not None and head_hypotheses.dim() == 4 \
                and not head_hypotheses.requires_grad and ops.prob_head_supported(x, impl):
            return ops.prob_head(x, self._prob_prepared(impl, x.dtype), head_hypotheses, impl)
        return ops.conv3d(x, self._prob_prepared(impl, x.dtype), None, None, 1, 1, False, False, None, torch.float32, True, impl)

    def forward(self, x: torch.Tensor) -> torch.Tensor:
        """Reference call signature: [B,C,D,H,W] -> [B,1,D,H,W]."""
        vol = G8Volume(ag.NcdhwToG8Fn.apply(x, ops.volume_dtype()))
        return self.forward_g8(vol).unsqueeze(1)


class AggWeightNetVolume(_EpochOnApply):
    """Per-view, per-voxel visibility weight net (reference models/module.py:544-563).

    Parameters mirror the reference exactly, including the dead ``conv0``.  In
    ``DepthNet`` the two 1x1x1 blocks are folded into five scalars plus a C-vector
    (``folded()``) and evaluated inside the fused warp/aggregate kernel.
    """

    def __init__(self, in_channels=32):
        super().__init__()
        self.conv0 = Conv3d(in_channels, 1, kernel_size=1, stride=1, padding=0)
        self.w_net = nn.Sequential(
            Conv3d(in_channels, 1, kernel_size=1, stride=1, padding=0),
            Conv3d(1, 1, kernel_size=1, stride=1, padding=0),
        )
        self.in_channels = in_channels
        self._folded: Dict[torch.device, tuple] = {}

    def folded(self) -> torch.Tensor:
        """[C+5] fp32: w1[C], scale1, shift1, w2, scale2, shift2 (include/damvs.h, damvs_warp_agg_fwd)."""
        a, b = self.w_net[0], self.w_net[1]
        if self.training:
            raise RuntimeError("folded() is the eval-mode form; in training DepthNet runs autograd.WarpAdaptiveTrainFn")
        tensors = (a.conv.weight, a.bn.weight, a.bn.bias, a.bn.running_mean, a.bn.running_var,
                   b.conv.weight, b.bn.weight, b.bn.bias, b.bn.running_mean, b.bn.running_var)
        ver = _versions(*tensors)
        dev = a.conv.weight.device
        hit = self._folded.get(dev)
        if hit is not None and hit[0] == ver:
            return hit[1]
        s1, b1 = _bn_affine(a.bn)
        s2, b2 = _bn_affine(b.bn)
        vec = torch.cat([a.conv.weight.detach().float().reshape(-1), s1, b1,
                         b.conv.weight.detach().float().reshape(-1), s2, b2]).contiguous()
        self._folded[dev] = (ver, vec)
        return vec

    def folded_with_grad(self) -> torch.Tensor:
        """folded() as a differentiable function of the parameters (eval-mode BatchNorm, gradients enabled):
        the kernel's gradient w.r.t. the C+5 vector flows back to conv weights, gamma and beta through autograd."""
        a, b = self.w_net[0], self.w_net[1]

        def affine(bn):
            scale = bn.weight / torch.sqrt(bn.running_var + bn.eps)
            return scale, bn.bias - bn.running_mean * scale
        s1, b1 = affine(a.bn)
        s2, b2 = affine(b.bn)
        return torch.cat([a.conv.weight.reshape(-1), s1, b1, b.conv.weight.reshape(-1), s2, b2]).float().contiguous()

    def forward(self, x: torch.Tensor) -> torch.Tensor:
        """Stand-alone reference signature [B,C,D,H,W] -> [B,1,D,H,W] (reference models/module.py:555-563).  NOT on the
        hot path: DepthNet evaluates the weight net inside the fused warp/aggregate kernels.  This entry exists so the
        class is a complete stand-in for the reference's: the two 1x1x1 conv + BatchNorm + ReLU blocks on C-to-1 /
        1-to-1 channels are C- and scalar-sized per-voxel affine maps, written here with tensor ops in both modes --
        eval(): the folded form the kernel uses; train(): batch statistics over (B,D,H,W), running buffers updated with
        momentum 0.1 and the unbiased variance, gradients through autograd, exactly as nn.BatchNorm3d does."""
        a, b = self.w_net[0], self.w_net[1]
        c = self.in_channels
        if not self.training and not ag.wants_grad(x, *self.w_net.parameters()):
            v = self.folded()
            s = (x * v[:c].view(1, c, 1, 1, 1)).sum(dim=1, keepdim=True)
            h = torch.relu(s * v[c] + v[c + 1])
            return torch.relu((h * v[c + 2]) * v[c + 3] + v[c + 4])
        y = (x * a.conv.weight.view(1, c, 1, 1, 1)).sum(dim=1, keepdim=True)
        for blk, pre in ((a, None), (b, b.conv.weight.view(()))):
            if pre is not None:
                y = y * pre
            bn = blk.bn
            factor = 0.0
            if self.training and bn.track_running_stats:
                bn.num_batches_tracked += 1                                 # nn.BatchNorm3d.forward does this first
                factor = bn.momentum if bn.momentum is not None else 1.0 / float(bn.num_batches_tracked)
            y = torch.relu(torch.nn.functional.batch_norm(y, bn.running_mean, bn.running_var, bn.weight, bn.bias,
                                                          self.training, factor, bn.eps))
        return y


def homo_warping(src_fea: torch.Tensor, src_proj: torch.Tensor, ref_proj: torch.Tensor,
                 depth_values: torch.Tensor) -> torch.Tensor:
    """Reference signature (models/module.py:297-302): src_fea [B,C,H,W], src_proj/ref_proj [B,4,4],
    depth_values [B,D] or [B,D,H,W] -> warped volume [B,C,D,H,W].  Forward only: the library has no stand-alone warp
    backward (DepthNet differentiates the fused warp + aggregation instead), so inputs that require grad are rejected
    rather than silently detached."""
    if ag.wants_grad(src_fea, src_proj, ref_proj, depth_values):
        raise NotImplementedError("homo_warping has no backward kernel; DepthNet's fused warp + aggregation is differentiable")
    rot_trans = ops.relative_rot_trans(src_proj.float(), ref_proj.float())
    return ops.homo_warp(ops.features_to_nhwc(src_fea), rot_trans, depth_values)


def depth_regression(p: torch.Tensor, depth_values: torch.Tensor) -> torch.Tensor:
    """Reference signature (models/module.py:609-615): sum_d p * depth_values."""
    if depth_values.dim() == 1:
        depth_values = depth_values.view(1, -1).expand(p.shape[0], -1)
    return ag.DepthRegressionFn.apply(p, depth_values.to(torch.float32))


def uncertainty_aware_samples(cur_depth: torch.Tensor, exp_var: torch.Tensor, ndepth, dtype=None, device=None, shape=None) -> torch.Tensor:
    """Reference signature (models/module.py:999): cur_depth [B,Dtot] (first stage) or [B,1,H,W], exp_var [B,1,H,W]
    -> depth hypotheses [B,D,H,W].  The [B,1,H,W] branch runs the native kernel (at the inputs' own resolution);
    the first-stage branch is a [B,D] range broadcast over (H,W), as in the reference.  Under the reference's default
    grad_method="detach" (cas_mvsnet.py:237-239) the inputs carry no gradient and the kernel runs; inputs that require
    grad (grad_method="undetach") take a differentiable tensor-op route so that gradient path is not lost."""
    ndepth = int(ndepth)
    if cur_depth.dim() == 2:
        lo, hi = cur_depth[:, 0], cur_depth[:, -1]
        interval = (hi - lo) / (ndepth - 1)
        rng = lo.unsqueeze(1) + torch.arange(0, ndepth, device=cur_depth.device, dtype=cur_depth.dtype).reshape(1, -1) * interval.unsqueeze(1)
        return rng.unsqueeze(-1).unsqueeze(-1).repeat(1, 1, shape[1], shape[2])
    if cur_depth.dim() != 4 or cur_depth.shape[1] != 1 or exp_var.shape != cur_depth.shape:
        raise ValueError("cur_depth and exp_var must be [B,1,H,W]")
    b, _, h, w = cur_depth.shape
    if ag.wants_grad(cur_depth, exp_var):
        # grad_method != "detach" (reference models/cas_mvsnet.py:236-243): the samples carry gradient back into the
        # previous stage's depth and variance.  Training-only side path, D small planes of element-wise math: kept on
        # the autograd tape with tensor ops (same formula as csrc/hypotheses.cu at scale 1; models/module.py:1012-1036).
        eps = 1e-12
        low = -torch.minimum(cur_depth, exp_var)
        step = (exp_var - low) / (float(ndepth) - 1.0)
        idx = torch.arange(ndepth, device=cur_depth.device, dtype=cur_depth.dtype).view(1, ndepth, 1, 1)
        lin = low + step * idx                                             # [B,D,H,W]
        offset = torch.softmax(3.0 * lin / (exp_var + eps), dim=1)
        return cur_depth + lin + eps + offset * step
    return ops.stage_hypotheses(cur_depth.reshape(b, h, w).float(), exp_var.reshape(b, h, w).float(), ndepth, h, w, 1)
