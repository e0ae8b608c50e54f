"""Host-side mirror of the reference's ``models/cas_mvsnet.py`` hot path: ``DepthNet``.

``DepthNet.forward`` keeps the reference signature and output dict
(models/cas_mvsnet.py:18, :133-134) and runs three native kernels per stage:
fused warp+aggregate -> CostRegNet conv blocks -> softmax/regression head.
"""
from __future__ import annotations

from typing import Dict, List, Optional, Sequence

import torch
import torch.nn as nn

from . import autograd as ag
from . import ops
from .module import AggWeightNetVolume, CostRegNet

__all__ = ["DepthNet", "stage_volume_channels"]


def stage_volume_channels(mode: str, in_channels: Sequence[int], groups: Optional[Sequence[int]]) -> List[int]:
    """Channels of each stage's cost volume, i.e. CostRegNet's in_channels: the feature width, or for mode
    "groupwise" max(G_s, 8) (a G = 4 volume is zero-padded to one 8-channel group).  `groups` holds one count per
    stage, or fewer, the last repeated (as DepthNet reads it)."""
    if mode != "groupwise":
        return list(in_channels)
    if groups is None:
        raise ValueError('mode "groupwise" needs groups=(G per stage)')
    gs = [int(g) for g in (groups if isinstance(groups, (list, tuple)) else [groups])]
    return [max(gs[min(s, len(gs) - 1)], 8) for s in range(len(in_channels))]


class DepthNet(nn.Module):
    """Per-stage cost-volume pipeline (reference models/cas_mvsnet.py:10-134)."""

    def __init__(self, mode="adaptive", in_channels=None, groups=None, trainable: bool = False):
        """mode "variance" / "adaptive" are the reference's (models/cas_mvsnet.py:11-16).  mode "groupwise" with
        `groups` = per-stage group counts is NOT in the reference: the group-wise correlation cost volume BASELINE.json's
        north star names (CostRegNet(in_channels=max(groups, 8)) consumes it).  It is inference-only unless
        `trainable` is set: then features that require grad go through the training kernels (csrc/warp_gwc_train.cu),
        in fp32 or bf16; without grad the inference kernel runs either way.  `trainable` means nothing for the
        other modes, which always train."""
        super().__init__()
        self.mode = mode
        assert mode in ("variance", "adaptive", "groupwise"), "Don't support {}!".format(mode)
        self.trainable = bool(trainable)
        self.groups = None
        if mode == "groupwise":
            if groups is None:
                raise ValueError('mode "groupwise" needs groups=[G per stage]')
            self.groups = [int(g) for g in (groups if isinstance(groups, (list, tuple)) else [groups])]
        if self.mode == "adaptive":
            self.weight_net = nn.ModuleList([AggWeightNetVolume(in_channels[i]) for i in range(len(in_channels))])

    @staticmethod
    def stage_rot_trans(proj_matrices: torch.Tensor) -> torch.Tensor:
        """[B,N,2,4,4] -> [N-1,B,12]: per source view, rows 0-2 of P_src @ inverse(P_ref)
        with P = [K @ E[:3,:4]; E[3]] (reference models/cas_mvsnet.py:44-47, models/module.py:308-310)."""
        p = ops.compose_projection(proj_matrices.float())          # [B,N,4,4]
        ref = p[:, 0:1]                                             # [B,1,4,4]
        rt = ops.relative_rot_trans(p[:, 1:], ref.expand(-1, p.shape[1] - 1, -1, -1).contiguous())  # [B,N-1,12]
        return rt.permute(1, 0, 2).contiguous()

    def cost_volume(self, stage_idx: int, features: List[torch.Tensor], proj_matrices: torch.Tensor,
                    depth_values: torch.Tensor, out_dtype: Optional[torch.dtype] = None) -> ops.G8Volume:
        """Aggregated cost volume (reference models/cas_mvsnet.py:30-87) as a G8 volume."""
        rot_trans = self.stage_rot_trans(proj_matrices)
        out_dtype = out_dtype or ops.volume_dtype()
        if self.mode == "groupwise":
            g = self.groups[min(stage_idx, len(self.groups) - 1)]
            if ag.wants_grad(*features):
                if not self.trainable:
                    raise NotImplementedError("group-wise correlation is an inference-only variant here: build "
                                              "DepthNet(..., trainable=True) to train through it")
                if out_dtype == torch.float16:
                    raise NotImplementedError("precision 'fp16' is the inference pipeline; train in 'bf16' or 'fp32'")
                with torch.no_grad():
                    rot_trans = rot_trans.detach()      # the sampling grid is not differentiated (module.py:307)
                    dv = depth_values.detach().contiguous()
                nhwc = [ag.NhwcFn.apply(f) for f in features]
                return ops.G8Volume(ag.WarpGwcFn.apply(rot_trans, dv, g, out_dtype, *nhwc))
            half = out_dtype in ops.HALF_DTYPES and ops.half_features()
            nhwc = ops.features_to_nhwc_half_multi(features) if half else [ops.features_to_nhwc(f) for f in features]
            return ops.warp_groupwise(nhwc[0], nhwc[1:], rot_trans, depth_values, g, out_dtype)
        wn = self.weight_net[stage_idx] if self.mode == "adaptive" else None
        batch_stats = wn is not None and wn.training
        params = tuple(wn.w_net.parameters()) if wn is not None else ()
        if batch_stats or ag.wants_grad(*features, *params):
            if out_dtype == torch.float16:
                raise NotImplementedError("precision 'fp16' is the inference pipeline; train in 'bf16' or 'fp32'")
            # training path: same kernels' worth of work, recorded on the autograd tape (damvsnet_b200/autograd.py)
            with torch.no_grad():
                rot_trans = rot_trans.detach()          # the sampling grid is not differentiated (module.py:307)
                dv = depth_values.detach().contiguous()
            nhwc = [ag.NhwcFn.apply(f) for f in features]
            if batch_stats:
                a, b2 = wn.w_net[0], wn.w_net[1]
                return ops.G8Volume(ag.WarpAdaptiveTrainFn.apply(a.conv.weight, a.bn.weight, a.bn.bias, b2.conv.weight, b2.bn.weight,
                                                                 b2.bn.bias, rot_trans, dv, out_dtype, wn, *nhwc))
            wnet = wn.folded_with_grad() if wn is not None else None
            return ops.G8Volume(ag.WarpAggFn.apply(wnet, rot_trans, dv, self.mode, out_dtype, *nhwc))
        # bf16 pipeline: fp16 NHWC features (half the gather bytes); fp32 pipeline: exact fp32 features
        half = out_dtype in ops.HALF_DTYPES and ops.half_features()
        nhwc = ops.features_to_nhwc_half_multi(features) if half else [ops.features_to_nhwc(f) for f in features]
        wnet = wn.folded() if wn is not None else None
        return ops.warp_aggregate(nhwc[0], nhwc[1:], rot_trans, depth_values, wnet, self.mode, out_dtype)

    def forward(self, stage_idx, features, proj_matrices, depth_values, num_depth, cost_regularization,
                prob_volume_init=None) -> Dict[str, torch.Tensor]:
        assert len(features) == proj_matrices.shape[1], "Different number of images and projection matrices"
        assert depth_values.shape[1] == num_depth, "depth_values.shape[1]:{}  num_depth:{}".format(
            depth_values.shape[1], num_depth)
        if not isinstance(cost_regularization, CostRegNet):
            raise TypeError("cost_regularization must be a damvsnet_b200 CostRegNet")
        volume = self.cost_volume(stage_idx, features, proj_matrices, depth_values)
        # inference with per-pixel hypotheses: the last conv layer and the head run as one launch where the shape allows
        fuse = prob_volume_init is None and depth_values.dim() == 4
        logits = cost_regularization.forward_g8(volume, head_hypotheses=depth_values if fuse else None)
        if isinstance(logits, tuple):
            prob, depth, conf, var = logits
            return {"depth": depth, "photometric_confidence": conf, "variance": var,
                    "prob_volume": prob, "depth_values": depth_values}
        if prob_volume_init is not None:                                       # dead in the reference (always None)
            logits = logits + prob_volume_init
        dv = depth_values
        if dv.dim() == 2:
            b, _, h, w = logits.shape
            dv = dv.view(b, -1, 1, 1).expand(-1, -1, h, w).contiguous()
        if ag.wants_grad(logits, dv):
            prob, depth, conf, var = ag.HeadFn.apply(logits, dv)
        else:
            prob, depth, conf, var = ops.softmax_regress(logits, dv)
        return {"depth": depth, "photometric_confidence": conf, "variance": var,
                "prob_volume": prob, "depth_values": depth_values}
