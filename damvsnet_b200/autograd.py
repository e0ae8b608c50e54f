"""Training path: ``torch.autograd.Function`` shells around the native forward / backward kernels.

The reference trains through PyTorch autograd over ``F.grid_sample``, ``nn.Conv3d`` / ``nn.ConvTranspose3d``,
``nn.BatchNorm3d`` and the softmax head (reference models/cas_mvsnet.py:18-134, models/module.py:117-202,
297-332, 510-563).  Here autograd is only the tape: every volume-sized operation, forward and backward, is a
kernel of libdamvs_b200.so.

* ``ConvBlockFn``  conv -> BatchNorm (batch or running statistics) -> ReLU (+ skip).  Backward: BatchNorm/ReLU
  backward kernel, data gradient = the adjoint convolution run by the same conv kernels on re-packed weights
  (stride-1 <-> stride-1 with transposed, flipped weights; stride-2 <-> transposed with the SAME weight tensor),
  weight gradient kernel.
* ``ProbConvFn``   the final 8 -> 1 convolution writing fp32 logits.
* ``HeadFn``       softmax + depth + confidence + variance; closed-form backward kernel.
* ``WarpAggFn``    fused warp + aggregation with a per-voxel weight net (eval-mode BN) or variance aggregation.
* ``WarpAdaptiveTrainFn``  the adaptive aggregation when the weight net's BatchNorms use batch statistics: score ->
  native scalar chain -> weighted, one scatter pass in the backward (csrc/warp_agg_train.cu, csrc/wnet_chain.cu).
* ``WarpGwcFn``    fused warp + group-wise correlation (not in the reference); forward and backward sample at the same
  coordinates (csrc/warp_gwc_train.cu).
"""
from __future__ import annotations

from typing import Optional

import torch

from . import ops, ops_train
from .ops import G8Volume


# --------------------------------------------------------------------------
# BatchNorm coefficient algebra (C-sized, host side of damvs_bn_*)
# --------------------------------------------------------------------------
def _batch_norm_coeffs(bn: torch.nn.BatchNorm3d, y: torch.Tensor, gamma, beta):
    """Batch statistics of a G8 volume -> (scale, shift, mean, rstd), with the running-buffer update of
    nn.BatchNorm3d.forward in training mode; two launches (damvs_bn_stats, damvs_bn_finalize)."""
    c = y.shape[1] * 8
    m = y.numel() // c
    sums = ops_train.bn_stats(y)
    track = bn.track_running_stats and bn.running_mean is not None
    f = 0.0
    if track:
        with torch.no_grad():
            bn.num_batches_tracked += 1
        # momentum None = cumulative average; needs the counter's value (a host read, as in nn.BatchNorm itself)
        f = 1.0 / float(bn.num_batches_tracked) if bn.momentum is None else bn.momentum
    g = None if gamma is None else gamma.detach().float()
    b = None if beta is None else beta.detach().float()
    rm = bn.running_mean if track and bn.running_mean.dtype == torch.float32 else None
    rv = bn.running_var if rm is not None else None
    return ops_train.bn_finalize(sums, g, b, rm, rv, m, f, bn.eps)


class ConvBlockFn(torch.autograd.Function):
    """out = skip + act(bn(conv(x))) on G8 data tensors.  `blk` is the Conv3d / Deconv3d module (configuration,
    packed-weight caches, BatchNorm buffers)."""

    @staticmethod
    def forward(ctx, x, skip, weight, gamma, beta, bias, blk):
        cin, cout, stride, tr = blk.in_channels, blk.out_channels, blk.stride, blk.transposed
        impl = ops.conv_impl_for(cin, cout, stride, tr)
        y = ops.conv3d(G8Volume(x), blk.packed_weight(impl), None, None, cout, stride, tr, False, None, x.dtype, False,
                       impl).data
        bn = blk.bn
        batch = bn is not None and (blk.training or not bn.track_running_stats)
        if bn is not None and batch:
            scale, shift, mean, rstd = _batch_norm_coeffs(bn, y, gamma, beta)
        elif bn is not None:
            mean, rstd = bn.running_mean.float(), torch.rsqrt(bn.running_var.float() + bn.eps)
            g = gamma.detach().float() if gamma is not None else torch.ones_like(mean)
            scale = g * rstd
            shift = (beta.detach().float() if beta is not None else torch.zeros_like(mean)) - mean * scale
        else:
            mean = torch.zeros(cout, dtype=torch.float32, device=x.device)
            rstd = torch.ones_like(mean)
            scale = torch.ones_like(mean)
            shift = bias.detach().float() if bias is not None else torch.zeros_like(mean)
        out = ops_train.bn_apply(y, scale, shift, skip, blk.relu)
        ctx.blk, ctx.batch, ctx.has_skip = blk, batch, skip is not None
        ctx.save_for_backward(x, y, scale, shift, mean, rstd)
        return out

    @staticmethod
    def backward(ctx, g_out):
        x, y, scale, shift, mean, rstd = ctx.saved_tensors
        blk = ctx.blk
        cin, cout, stride, tr = blk.in_channels, blk.out_channels, blk.stride, blk.transposed
        g_out = g_out.contiguous()
        m = y.numel() // cout
        if ctx.batch:
            _, sums = ops_train.bn_bwd(g_out, y, scale, shift, None, None, None, blk.relu, False, True)
            k1, k2, k3, dgamma, dbeta = ops_train.bn_bwd_coeffs(sums, scale, mean, rstd, m, True)
            g_y, _ = ops_train.bn_bwd(g_out, y, scale, shift, k1, k2, k3, blk.relu, True, False)
        else:
            g_y, sums = ops_train.bn_bwd(g_out, y, scale, shift, scale, None, None, blk.relu, True, True)
            _, _, _, dgamma, dbeta = ops_train.bn_bwd_coeffs(sums, scale, mean, rstd, m, False)
        g_x = g_w = g_gamma = g_beta = g_bias = None
        if ctx.needs_input_grad[0]:
            a_stride, a_tr = (1, False) if (stride == 1 and not tr) else ((2, False) if tr else (2, True))
            impl = ops.conv_impl_for(cout, cin, a_stride, a_tr)
            g_x = ops.conv3d(G8Volume(g_y), blk.packed_adjoint(impl), None, None, cin, a_stride, a_tr, False, None, g_y.dtype,
                             False, impl).data
            if g_x.shape != x.shape:
                # the adjoint of a stride-2 conv over an odd extent is a transposed conv one plane longer than x (2 * ceil(n/2)
                # planes); the extra plane pairs with no input voxel, so the data gradient is its crop
                g_x = g_x[:, :, :x.shape[2], :x.shape[3], :x.shape[4]].contiguous()
        if ctx.needs_input_grad[2]:
            g_w = ops_train.conv3d_wgrad(x, g_y, cin, cout, stride, tr)
        if blk.bn is not None:
            if ctx.needs_input_grad[3]:
                g_gamma = dgamma
            if ctx.needs_input_grad[4]:
                g_beta = dbeta
        elif ctx.needs_input_grad[5]:
            g_bias = dbeta               # without BatchNorm the conv bias is the shift: its gradient is the channel sum of g_z
        g_skip = g_out if (ctx.has_skip and ctx.needs_input_grad[1]) else None
        return g_x, g_skip, g_w, g_gamma, g_beta, g_bias, None


class ProbConvFn(torch.autograd.Function):
    """CostRegNet.prob (reference models/module.py:530): Conv3d(8 -> 1, k3, p1, no bias) -> fp32 logits [B,D,H,W]."""

    @staticmethod
    def forward(ctx, x, weight, net):
        impl = ops.conv_impl_for(net.base_channels, 1, 1, False)
        logits = ops.conv3d(G8Volume(x), net._prob_prepared(impl), None, None, 1, 1, False, False, None, torch.float32, True, impl)
        ctx.net = net
        ctx.save_for_backward(x)
        return logits

    @staticmethod
    def backward(ctx, g_logits):
        (x,) = ctx.saved_tensors
        net = ctx.net
        c = net.base_channels
        g8 = ops_train.plain_to_g8(g_logits.contiguous().float(), x.dtype)
        g_x = g_w = None
        if ctx.needs_input_grad[0]:
            impl = ops.conv_impl_for(8, c, 1, False)
            g_x = ops.conv3d(G8Volume(g8), net._prob_adjoint(impl), None, None, c, 1, False, False, None, x.dtype, False, impl).data
        if ctx.needs_input_grad[1]:
            g_w = ops_train.conv3d_wgrad(x, g8, c, 1, 1, False)
        return g_x, g_w, None


class HeadFn(torch.autograd.Function):
    """softmax + depth regression + photometric confidence + hypothesis variance (reference
    models/cas_mvsnet.py:105-124).  The confidence is computed under no_grad in the reference and is
    non-differentiable here too."""

    @staticmethod
    def forward(ctx, logits, depth_values):
        prob, depth, conf, var = ops.softmax_regress(logits, depth_values)
        ctx.save_for_backward(prob, depth_values, depth)
        ctx.mark_non_differentiable(conf)
        return prob, depth, conf, var

    @staticmethod
    def backward(ctx, g_prob, g_depth, _g_conf, g_var):
        prob, dv, depth = ctx.saved_tensors
        g_logits, g_hyp = ops_train.softmax_regress_bwd(prob, dv, depth, g_depth, g_var, g_prob,
                                                        want_hyp_grad=ctx.needs_input_grad[1])
        return g_logits, g_hyp


class DepthRegressionFn(torch.autograd.Function):
    """depth = sum_d p * depth_values (native kernel); backward g_p = g * dv, g_dv = g * p (D planes of tensor ops)."""

    @staticmethod
    def forward(ctx, p, depth_values):
        ctx.save_for_backward(p, depth_values)
        return ops.depth_regression(p, depth_values)

    @staticmethod
    def backward(ctx, g):
        p, dv = ctx.saved_tensors
        g = g.unsqueeze(1)
        dv4 = dv if dv.dim() == 4 else dv.view(*dv.shape, 1, 1)
        g_p = g * dv4 if ctx.needs_input_grad[0] else None
        g_dv = None
        if ctx.needs_input_grad[1]:
            g_dv = g * p if dv.dim() == 4 else (g * p).sum(dim=(2, 3))
        return g_p, g_dv


class NcdhwToG8Fn(torch.autograd.Function):
    """[B,C,D,H,W] fp32 -> G8 data tensor of `dtype` (layout kernel); the backward is the opposite layout kernel."""

    @staticmethod
    def forward(ctx, x, dtype):
        return G8Volume.from_ncdhw(x, dtype).data

    @staticmethod
    def backward(ctx, g):
        return G8Volume(g.contiguous()).to_ncdhw(), None


class G8ToNcdhwFn(torch.autograd.Function):
    """G8 data tensor -> [B,C,D,H,W] fp32 (layout kernel); the backward is the opposite layout kernel."""

    @staticmethod
    def forward(ctx, data):
        ctx.dtype = data.dtype
        return G8Volume(data).to_ncdhw()

    @staticmethod
    def backward(ctx, g):
        return G8Volume.from_ncdhw(g.contiguous().float(), ctx.dtype).data


class NhwcFn(torch.autograd.Function):
    """[B,C,H,W] -> contiguous [B,H,W,C] (native repack kernel); the gradient is the permuted view."""

    @staticmethod
    def forward(ctx, x):
        return ops.features_to_nhwc(x)

    @staticmethod
    def backward(ctx, g):
        return g.permute(0, 3, 1, 2)


class WarpAggFn(torch.autograd.Function):
    """Fused warp + aggregation, per-voxel weight net (folded eval-mode BN, `wnet` = [C+5]) or variance."""

    @staticmethod
    def forward(ctx, wnet, rot_trans, depth_values, mode, out_dtype, ref, *srcs):
        vol = ops.warp_aggregate(ref, list(srcs), rot_trans, depth_values, wnet, mode, out_dtype).data
        ctx.mode = mode
        ctx.save_for_backward(wnet, rot_trans, depth_values, ref, *srcs)
        return vol

    @staticmethod
    def backward(ctx, g_vol):
        wnet, rot_trans, dv, ref, *srcs = ctx.saved_tensors
        g_ref, g_srcs, g_wnet = ops_train.warp_agg_bwd(ref, srcs, rot_trans, dv, wnet, g_vol, ctx.mode)
        return (g_wnet, None, None, None, None, g_ref, *g_srcs)


class WarpGwcFn(torch.autograd.Function):
    """Fused warp + group-wise correlation -> G8 volume of max(groups, 8) channels.  Saves only its inputs; the
    backward re-projects and re-samples (one scatter pass to the source features)."""

    @staticmethod
    def forward(ctx, rot_trans, depth_values, groups, out_dtype, ref, *srcs):
        vol = ops_train.warp_gwc_train_fwd(ref, list(srcs), rot_trans, depth_values, groups, out_dtype)
        ctx.groups = groups
        ctx.save_for_backward(rot_trans, depth_values, ref, *srcs)
        return vol

    @staticmethod
    def backward(ctx, g_vol):
        rot_trans, dv, ref, *srcs = ctx.saved_tensors
        g_ref, g_srcs = ops_train.warp_gwc_bwd(ref, srcs, rot_trans, dv, g_vol, ctx.groups)
        return (None, None, None, None, g_ref, *g_srcs)


class WarpAdaptiveTrainFn(torch.autograd.Function):
    """The adaptive aggregation with the weight net in training mode as ONE node: score -> scalar chain -> weighted in
    the forward; in the backward d loss / d wt (no scatter), the chain's own backward on the scalar volumes, then a
    single scatter pass that carries both paths into the features (through the aggregate and through the score).
    Every step is a kernel of the library (csrc/warp_agg_train.cu, csrc/wnet_chain.cu).  `wn` is the
    AggWeightNetVolume module (its BatchNorm buffers are updated once, in the forward)."""

    @staticmethod
    def forward(ctx, w1, g1, b1, w2, g2, b2, rot_trans, depth_values, out_dtype, wn, ref, *srcs):
        srcs = list(srcs)
        a, b = wn.w_net[0], wn.w_net[1]
        s_vol = ops_train.warp_score_fwd(ref, srcs, rot_trans, depth_values, w1.detach().reshape(-1).float())
        wt_vol, state = ops_train.wnet_chain_fwd(s_vol, a.bn, w2, b.bn)
        vol = ops_train.warp_weighted_fwd(ref, srcs, rot_trans, depth_values, wt_vol, out_dtype)
        ctx.save_for_backward(w1, w2, s_vol, wt_vol, state, rot_trans, depth_values, ref, *srcs)
        return vol

    @staticmethod
    def backward(ctx, g_vol):
        w1, w2, s_vol, wt_vol, state, rot_trans, dv, ref, *srcs = ctx.saved_tensors
        g_wt = ops_train.warp_gwt(ref, srcs, rot_trans, dv, g_vol)
        g_s, gp = ops_train.wnet_chain_bwd(s_vol, g_wt, state, w2)
        g_ref = torch.zeros_like(ref)
        g_srcs = [torch.zeros_like(s) for s in srcs]
        g_w1 = ops_train.warp_merged_bwd(ref, srcs, rot_trans, dv, w1.detach().reshape(-1).float(), wt_vol, g_s, g_vol, g_ref, g_srcs)
        need = ctx.needs_input_grad
        return (g_w1.view_as(w1) if need[0] else None, gp[0:1] if need[1] else None, gp[1:2] if need[2] else None,
                gp[2:3].view_as(w2) if need[3] else None, gp[3:4] if need[4] else None, gp[4:5] if need[5] else None,
                None, None, None, None, g_ref, *g_srcs)


def wants_grad(*tensors: Optional[torch.Tensor]) -> bool:
    return torch.is_grad_enabled() and any(t is not None and t.requires_grad for t in tensors)
