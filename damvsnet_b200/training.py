"""Data-parallel training step of the hot path (BASELINE.json configs[3]).

One process per GPU.  Each rank runs forward + backward of the three stages on its own batch through the native
kernels (``damvsnet_b200.autograd``), then the gradients of the hot-path parameters are summed across ranks:
``GradientBucket`` flattens a parameter set into ONE contiguous fp32 buffer (3.5 MB for the whole path at base_channels
8, SURVEY.md 8e) so that one ``all_reduce`` (NCCL over NVLink on the GPUs, gloo in the CPU test) replaces ~70 per-tensor
collectives; ``OverlappedBuckets`` keeps one bucket per cascade stage and starts its collective from gradient hooks as
soon as that stage's backward is complete, so it overlaps the backward kernels of the remaining stages; the averaged
values are scattered back into ``param.grad``.  BatchNorm statistics stay per GPU, as in the reference
(plain ``DistributedDataParallel``, no SyncBN: train.py:474-479); buffers are broadcast from rank 0 once at
start, like DDP's initial sync.  Parameters that never receive a gradient (the dead ``conv0`` of the view-weight
net, SURVEY.md appendix B) are left out of the bucket -- the reference as committed needs
``find_unused_parameters`` for them.

The loss is the reference's ``cas_mvsnet_loss`` (models/module.py:695-719): masked smooth-L1 depth term per stage,
weighted by ``dlossw`` (train.py:65 default 0.5,1.0,2.0), plus -- when images and cameras are handed to
``train_step`` -- 12 x the cross-view photometric term (``damvsnet_b200.losses.cross_view_loss``, native).
"""
from __future__ import annotations

from typing import Dict, Iterable, List, Optional, Sequence, Tuple

import torch
import torch.distributed as dist
import torch.nn.functional as F

from . import synthetic
from .cas_mvsnet import DepthNet, stage_volume_channels
from .module import CostRegNet

StageInput = Tuple[List[torch.Tensor], torch.Tensor, torch.Tensor]


class GradientBucket:
    """Flat fp32 gradient buffer over a fixed parameter list; `allreduce` averages it across the group."""

    def __init__(self, params: Iterable[torch.nn.Parameter]):
        self.params = [p for p in params if p.requires_grad]
        if not self.params:
            raise ValueError("no trainable parameters")
        dev = self.params[0].device
        self.numel = sum(p.numel() for p in self.params)
        self.flat = torch.zeros(self.numel, dtype=torch.float32, device=dev)
        self.views = []
        off = 0
        for p in self.params:
            self.views.append(self.flat[off:off + p.numel()].view_as(p))
            off += p.numel()

    def gather(self) -> None:
        for p, v in zip(self.params, self.views):
            if p.grad is None:
                v.zero_()
            else:
                v.copy_(p.grad)

    def scatter(self) -> None:
        for p, v in zip(self.params, self.views):
            if p.grad is None:
                p.grad = v.clone()
            else:
                p.grad.copy_(v)

    def allreduce(self, group=None, async_op: bool = False):
        """Average gradients across ranks.  No-op without an initialised process group (single GPU)."""
        if not (dist.is_available() and dist.is_initialized()) or dist.get_world_size(group) == 1:
            return None
        self.gather()
        world = dist.get_world_size(group)
        work = dist.all_reduce(self.flat, op=dist.ReduceOp.SUM, group=group, async_op=async_op)

        def finish():
            if work is not None:
                work.wait()
            self.flat.div_(world)
            self.scatter()
        if async_op:
            return finish
        finish()
        return None


class OverlappedBuckets:
    """One GradientBucket per cascade stage, all-reduced as soon as the backward pass has produced the last gradient of
    that stage (autograd runs the stages in reverse, so the collective of stage 3 overlaps the backward kernels of
    stages 2 and 1).  Hooks fire on gradient accumulation; `finish()` waits for the collectives and scatters the
    averages back.  Without a process group everything is a no-op."""

    def __init__(self, stage_params: Sequence[Sequence[torch.nn.Parameter]], group=None):
        self.group = group
        self.buckets = [GradientBucket(ps) for ps in stage_params if any(p.requires_grad for p in ps)]
        self.active = dist.is_available() and dist.is_initialized() and dist.get_world_size(group) > 1
        self._left: List[int] = []
        self._done: List[object] = []
        self._handles = []
        if self.active:
            for i, b in enumerate(self.buckets):
                for p in b.params:
                    self._handles.append(p.register_post_accumulate_grad_hook(lambda _p, i=i: self._ready(i)))
        self.reset()

    def reset(self) -> None:
        self._left = [len(b.params) for b in self.buckets]
        self._done = [None] * len(self.buckets)
        self._next = len(self.buckets) - 1        # collectives are issued in ONE order on every rank: last stage first

    def close(self) -> None:
        """Remove the gradient hooks (a second trainer over the same parameters would otherwise double-count)."""
        for h in self._handles:
            h.remove()
        self._handles = []
        self.active = False

    def _issue_ready(self) -> None:
        # bucket i is started only once every later bucket has been started, so ranks whose buckets complete in a
        # different order (e.g. one rank has a parameter without gradient) still pair the same collectives
        while self._next >= 0 and self._left[self._next] == 0:
            self._done[self._next] = self.buckets[self._next].allreduce(self.group, async_op=True)
            self._next -= 1

    def _ready(self, i: int) -> None:
        self._left[i] -= 1
        if self._left[i] < 0:
            raise RuntimeError("OverlappedBuckets: a second backward() before finish() (gradient accumulation) is not "
                               "supported: call finish() after every backward, or use GradientBucket.allreduce directly")
        self._issue_ready()

    def finish(self) -> None:
        if self.active:
            # buckets the hooks could not start (a parameter got no gradient on this rank) go now, in the same order
            while self._next >= 0:
                self._done[self._next] = self.buckets[self._next].allreduce(self.group, async_op=True)
                self._next -= 1
            for fin in reversed(self._done):
                if fin is not None:
                    fin()
        self.reset()


def broadcast_module_state(modules: Sequence[torch.nn.Module], src: int = 0, group=None) -> None:
    """Parameters and buffers of rank `src` to every rank (DDP's construction-time sync)."""
    if not (dist.is_available() and dist.is_initialized()) or dist.get_world_size(group) == 1:
        return
    from .module import invalidate_packed
    with torch.no_grad():
        for m in modules:
            for t in list(m.parameters()) + list(m.buffers()):
                dist.broadcast(t, src=src, group=group)     # in place on the tensor itself: bumps t._version
    invalidate_packed()                                      # belt and braces: packed-weight caches are rebuilt


def depth_loss(outputs: Sequence[Dict[str, torch.Tensor]], depth_gt: Sequence[torch.Tensor], masks: Sequence[torch.Tensor],
               dlossw: Sequence[float] = (0.5, 1.0, 2.0)) -> torch.Tensor:
    """Depth term of cas_mvsnet_loss (reference models/module.py:702-714)."""
    total = None
    for out, gt, mask, w in zip(outputs, depth_gt, masks, dlossw):
        m = mask > 0.5
        term = w * F.smooth_l1_loss(out["depth"][m], gt[m], reduction="mean")
        total = term if total is None else total + term
    return total


class HotPathTrainer:
    """DepthNet + per-stage CostRegNets in train() mode, Adam (train.py:439), one bucketed gradient all-reduce.
    mode "groupwise" (not in the reference) takes `groups` = per-stage group counts; its cost volume has no parameters,
    so only the CostRegNets (in_channels = max(G, 8)) train."""

    def __init__(self, state_dict: Optional[Dict[str, torch.Tensor]] = None, mode: str = "adaptive",
                 in_channels: Sequence[int] = synthetic.STAGE_CHANNELS, base_channels: Sequence[int] = (8, 8, 8),
                 device: torch.device | str = "cuda:0", lr: float = 1e-3, weight_decay: float = 0.0, group=None,
                 groups: Optional[Sequence[int]] = None):
        self.device = torch.device(device)
        self.group = group
        vol_channels = stage_volume_channels(mode, in_channels, groups)
        self.depthnet = DepthNet(mode, list(in_channels), groups, trainable=True)
        self.cost_regularization = torch.nn.ModuleList([CostRegNet(c, b) for c, b in zip(vol_channels, base_channels)])
        if state_dict is not None:
            if mode == "adaptive":
                self.depthnet.load_state_dict({k[len("DepthNet."):]: v for k, v in state_dict.items()
                                               if k.startswith("DepthNet.")}, strict=True)
            self.cost_regularization.load_state_dict({k[len("cost_regularization."):]: v for k, v in state_dict.items()
                                                      if k.startswith("cost_regularization.")}, strict=True)
        self.depthnet.to(self.device).train()
        self.cost_regularization.to(self.device).train()
        # the dead conv0 block of AggWeightNetVolume never gets a gradient (models/module.py:547)
        for wn in getattr(self.depthnet, "weight_net", []):
            for p in wn.conv0.parameters():
                p.requires_grad_(False)
        broadcast_module_state([self.depthnet, self.cost_regularization], group=group)
        self.params = [p for p in list(self.depthnet.parameters()) + list(self.cost_regularization.parameters())
                       if p.requires_grad]
        self.bucket = GradientBucket(self.params)          # the whole hot path as one buffer (size report, tests)
        n_stage = len(self.cost_regularization)
        per_stage = [[p for p in list(self.cost_regularization[s].parameters()) +
                      (list(self.depthnet.weight_net[s].parameters()) if mode == "adaptive" else []) if p.requires_grad]
                     for s in range(n_stage)]
        self.overlap = OverlappedBuckets(per_stage, group)
        self.optimizer = torch.optim.Adam(self.params, lr=lr, betas=(0.9, 0.999), weight_decay=weight_decay)

    def forward(self, stages: Sequence[StageInput]) -> List[Dict[str, torch.Tensor]]:
        return [self.depthnet(i, f, p, d, d.shape[1], self.cost_regularization[i]) for i, (f, p, d) in enumerate(stages)]

    def train_step(self, stages: Sequence[StageInput], depth_gt: Sequence[torch.Tensor], masks: Sequence[torch.Tensor],
                   dlossw: Sequence[float] = (0.5, 1.0, 2.0), imgs: Optional[torch.Tensor] = None,
                   sample_cams: Optional[Dict[str, torch.Tensor]] = None, cpc_weight: float = 12.0) -> torch.Tensor:
        """forward -> loss -> backward -> gradient all-reduce -> Adam step.  Returns the (local) loss tensor.
        With `imgs` [B,N,3,H,W] and `sample_cams` {stageK: [B,N,2,4,4]} the loss is the reference's full
        cas_mvsnet_loss: depth term + 12 x cross-view photometric term (models/module.py:700-717)."""
        self.optimizer.zero_grad(set_to_none=False)
        outs = self.forward(stages)
        loss = depth_loss(outs, depth_gt, masks, dlossw)
        if imgs is not None:
            from .losses import cross_view_loss
            named = {f"stage{i + 1}": o for i, o in enumerate(outs)}
            gts = {f"stage{i + 1}": g for i, g in enumerate(depth_gt)}
            loss = loss + cpc_weight * cross_view_loss(named, imgs, sample_cams, gts, list(dlossw))
        loss.backward()          # per-stage gradient all-reduces start from hooks inside the backward pass
        self.overlap.finish()
        self.optimizer.step()
        return loss.detach()
