"""Three-stage hot-path runner: the call a user of this package makes per reference view.

``HotPathRunner`` owns one ``DepthNet`` and the per-stage ``CostRegNet``s (loaded from a
reference-keyed state_dict) and exposes

* ``run_device(stages)``  -- inputs already resident in HBM;
* ``run_host(stages)``    -- inputs in (pinned) host memory: per view it uploads the
  stage inputs on a copy stream, runs the three stages on the compute stream and
  reads depth / confidence / variance back to pinned host buffers.  Uploads of
  stage s+1 overlap the kernels of stage s.

A "stage input" is ``(features: list of N [B,C,h,w] fp32, proj_matrices [B,N,2,4,4],
depth_values [B,D,h,w])`` exactly as ``DepthNet.forward`` receives them in the
reference (models/cas_mvsnet.py:292-298).
"""
from __future__ import annotations

from typing import Dict, List, Sequence, Tuple

import torch

from . import synthetic
from .cas_mvsnet import DepthNet, stage_volume_channels
from .module import CostRegNet

StageInput = Tuple[List[torch.Tensor], torch.Tensor, torch.Tensor]


class HotPathRunner:
    def __init__(self, state_dict: Dict[str, torch.Tensor], mode: str = "adaptive",
                 in_channels: Sequence[int] = synthetic.STAGE_CHANNELS, base_channels: Sequence[int] = (8, 8, 8),
                 device: torch.device | str = "cuda:0", groups: Sequence[int] | None = None):
        """mode "groupwise" (not in the reference) takes `groups` = per-stage group counts; the state dict then holds
        CostRegNets of in_channels max(G, 8), as HotPathTrainer(mode="groupwise") trains them."""
        self.device = torch.device(device)
        self.mode = mode
        vol_channels = stage_volume_channels(mode, in_channels, groups)
        self.depthnet = DepthNet(mode, list(in_channels), groups).eval()
        if mode == "adaptive":
            self.depthnet.load_state_dict({k[len("DepthNet."):]: v for k, v in state_dict.items()
                                           if k.startswith("DepthNet.")}, strict=True)
        self.cost_regularization = torch.nn.ModuleList(
            [CostRegNet(c, b) for c, b in zip(vol_channels, base_channels)]).eval()
        self.cost_regularization.load_state_dict({k[len("cost_regularization."):]: v for k, v in state_dict.items()
                                                  if k.startswith("cost_regularization.")}, strict=True)
        self.depthnet.to(self.device)
        self.cost_regularization.to(self.device)
        self._copy_stream = None
        self._host_out = None
        self._graphs = {}

    # ------------------------------------------------------------------ device-resident
    @torch.no_grad()
    def run_stage(self, stage_idx: int, features, proj, depth_values) -> Dict[str, torch.Tensor]:
        return self.depthnet(stage_idx, features, proj, depth_values, depth_values.shape[1],
                             self.cost_regularization[stage_idx])

    @torch.no_grad()
    def run_device(self, stages: Sequence[StageInput]) -> List[Dict[str, torch.Tensor]]:
        return [self.run_stage(i, f, p, d) for i, (f, p, d) in enumerate(stages)]

    # ------------------------------------------------------------------ chained cascade
    @torch.no_grad()
    def run_cascade(self, features: Sequence[Sequence[torch.Tensor]], proj_matrices: Dict[str, torch.Tensor],
                    depth_values: torch.Tensor, ndepths: Sequence[int], height: int, width: int,
                    scales: Sequence[int] = synthetic.STAGE_SCALES) -> Dict[str, object]:
        """The stage loop of CascadeMVSNet.forward (reference models/cas_mvsnet.py:210-307) on given per-stage
        features: stage-1 hypotheses from the plane-sweep range, stages 2/3 from the previous stage's depth and
        variance through the fused sampling kernel, every stage through DepthNet.  `features[s]` is the list of N
        stage-s feature maps (the reference refines the reference-view features between stages with its PyTorch
        GeoFeatureFusionNet; pass the refined maps in if that is wanted).  Returns the reference's output dict:
        "stage1".."stage3" plus the last stage's five keys at top level (cas_mvsnet.py:306-307)."""
        from . import ops
        outputs: Dict[str, object] = {}
        depth = var = None
        for s, nd in enumerate(ndepths):
            f = features[s]
            b, _, h, w = f[0].shape
            if depth is None:
                lo, hi = depth_values[:, 0], depth_values[:, -1]
                rng = lo.unsqueeze(1) + torch.arange(nd, device=depth_values.device, dtype=torch.float32).view(1, -1) * \
                    ((hi - lo) / (nd - 1)).unsqueeze(1)                         # module.py:1003-1008
                dv = rng.view(b, nd, 1, 1).expand(b, nd, h, w).contiguous()
            else:
                dv = ops.stage_hypotheses(depth, var, nd, height, width, scales[s])
            out = self.run_stage(s, f, proj_matrices[f"stage{s + 1}"], dv)
            depth, var = out["depth"], out["variance"]
            outputs[f"stage{s + 1}"] = out
            outputs.update(out)
        return outputs

    # ------------------------------------------------------------------ CUDA-graph replay
    @staticmethod
    def _signature(stages: Sequence[StageInput]):
        return tuple((tuple(f.data_ptr() for f in fs), p.data_ptr(), d.data_ptr(), tuple(d.shape), fs[0].shape[1])
                     for fs, p, d in stages)

    @torch.no_grad()
    def run_device_graphed(self, stages: Sequence[StageInput]) -> List[Dict[str, torch.Tensor]]:
        """Same result as run_device, replayed from a CUDA graph captured on first use for these input
        buffers (pointers and shapes are baked in: callers refill the same tensors between calls).
        One graph launch replaces ~60 kernel launches + ~70 small torch ops of host work per view."""
        from . import ops
        key = (self._signature(stages),) + tuple(sorted(ops._POLICY.items()))     # every policy knob that shapes the captured step
        hit = self._graphs.get(key)
        if hit is None:
            # warm-up outside capture: weight packing synchronises and fills the per-module caches
            self.run_device(stages)
            torch.cuda.synchronize(self.device)
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g):
                outs = self.run_device(stages)
            hit = (g, outs)
            self._graphs[key] = hit
        hit[0].replay()
        return hit[1]

    # ------------------------------------------------------------------ host buffers
    @staticmethod
    def pin_stages(stages: Sequence[StageInput], feature_format: str = "nchw_f32") -> List[StageInput]:
        """Host inputs -> pinned host inputs.  feature_format "nchw_f32" keeps the reference layout; "nhwc_f16" stores
        each feature map as an fp16 channels_last [B,C,h,w] tensor -- the width and layout the bf16 pipeline's gather
        kernel consumes, so the upload is half the bytes and the device side is zero-copy (no repack launch)."""
        if feature_format not in ("nchw_f32", "nhwc_f16"):
            raise ValueError(f"unknown feature_format {feature_format!r}")

        def feat(f):
            if feature_format == "nhwc_f16":
                f = f.clamp(-65504.0, 65504.0).to(torch.float16).contiguous(memory_format=torch.channels_last)
            return f.pin_memory()

        def pin(t):
            if t is None:
                return None
            if isinstance(t, (tuple, list)):
                return tuple(pin(x) for x in t)
            return t.pin_memory()
        return [([feat(f) for f in feats], proj.pin_memory(), pin(dv)) for feats, proj, dv in stages]

    @staticmethod
    def h2d_bytes(stages: Sequence[StageInput]) -> int:
        def nb(t):
            if t is None:
                return 0
            if isinstance(t, (tuple, list)):
                return sum(nb(x) for x in t)
            return t.numel() * t.element_size()
        return sum(nb(feats) + nb(proj) + nb(dv) for feats, proj, dv in stages)

    @staticmethod
    def d2h_bytes(stages: Sequence[StageInput]) -> int:
        return sum(3 * f[0].shape[0] * f[0].shape[2] * f[0].shape[3] * 4 for f, _, _ in stages)

    @torch.no_grad()
    def submit_host(self, stages: Sequence[StageInput], cascade=None) -> "HostTicket":
        """Enqueue one view whose inputs live in (pinned) host memory: H2D on the copy stream, the three stages
        on the compute stream (stage s waits only for its own inputs), D2H of depth / confidence / variance on
        the readback stream.  Returns immediately; `collect` waits.  Submitting view i+1 before collecting
        view i overlaps its upload with view i's kernels.

        `cascade` = (depth_range [B,Dtot] host tensor, ndepths, height, width) chains the stages as
        CascadeMVSNet.forward does (reference models/cas_mvsnet.py:236-296): a stage whose hypotheses are `None`
        gets them on the device -- stage 1 from the plane-sweep range, later stages from the previous stage's depth
        and variance through the fused sampling kernel -- so only features and cameras cross PCIe.  A stage may also
        carry a `(prev_depth, prev_variance)` pair of [B,hp,wp] host maps in place of its hypotheses (teacher-forced
        cascade): they are uploaded (h*w*8 bytes instead of D*h*w*4) and sampled on the device by the same kernel."""
        dev = self.device
        if self._copy_stream is None:
            self._copy_stream = torch.cuda.Stream(device=dev)
            self._d2h_stream = torch.cuda.Stream(device=dev)
            self._host_pool = []
            self._dev_in = [None, None]
            self._set_done = [None, None]
            self._submits = 0
        compute = torch.cuda.current_stream(dev)
        copy, d2h = self._copy_stream, self._d2h_stream
        # two persistent sets of device input buffers (no allocator traffic, hence no implicit device syncs):
        # set k is overwritten only after the kernels that last read it have finished
        bset = self._submits % 2
        self._submits += 1
        def shp(t):
            if t is None:
                return None
            if isinstance(t, (tuple, list)):
                return tuple(shp(x) for x in t)
            return (tuple(t.shape), t.dtype, tuple(t.stride()))

        def dev_like(t):
            # empty_like keeps the strides (channels_last features stay channels_last: one flat memcpy each)
            if t is None:
                return None
            if isinstance(t, (tuple, list)):
                return tuple(dev_like(x) for x in t)
            return torch.empty_like(t, device=dev)

        def upload(src, dst):
            if src is None:
                return
            if isinstance(src, (tuple, list)):
                for a, b2 in zip(src, dst):
                    upload(a, b2)
                return
            dst.copy_(src, non_blocking=True)
        if self._dev_in[bset] is None or [[shp(t) for t in st[0]] + [shp(st[1]), shp(st[2])] for st in self._dev_in[bset]] != \
                [[shp(f) for f in feats] + [shp(proj), shp(dv)] for feats, proj, dv in stages]:
            self._dev_in[bset] = [([dev_like(f) for f in feats], dev_like(proj), dev_like(dv)) for feats, proj, dv in stages]
            self._set_done[bset] = None
        if self._set_done[bset] is not None:
            copy.wait_event(self._set_done[bset])
        uploaded, ready = [], []
        with torch.cuda.stream(copy):
            for (feats, proj, dv), (bfe, bpr, bdv) in zip(stages, self._dev_in[bset]):
                upload(feats, bfe)
                upload(proj, bpr)
                upload(dv, bdv)
                ev = torch.cuda.Event()
                ev.record(copy)
                uploaded.append((bfe, bpr, bdv))
                ready.append(ev)
        shapes = [(f[0].shape[0], f[0].shape[2], f[0].shape[3]) for f, _, _ in stages]
        host = None
        for i, cand in enumerate(self._host_pool):
            if [tuple(o["depth"].shape) for o in cand] == shapes:
                host = self._host_pool.pop(i)
                break
        if host is None:
            host = [{k: torch.empty(sh, dtype=torch.float32).pin_memory()
                     for k in ("depth", "photometric_confidence", "variance")} for sh in shapes]
        prev = None
        for i, ((dfe, dpr, ddv), ev) in enumerate(zip(uploaded, ready)):
            compute.wait_event(ev)
            if ddv is None or isinstance(ddv, tuple):
                from . import ops
                rng_host, ndepths, height, width = cascade
                b, _, h, w = dfe[0].shape
                if isinstance(ddv, tuple):   # teacher-forced cascade: the previous stage's (depth, variance) maps were handed in
                    ddv = ops.stage_hypotheses(ddv[0], ddv[1], ndepths[i], height, width, height // h)
                elif prev is None:          # plane-sweep range -> evenly spaced hypotheses (models/module.py:1003-1010)
                    ddv = self.range_hypotheses(rng_host, ndepths[i], b, h, w)
                else:
                    ddv = ops.stage_hypotheses(prev["depth"], prev["variance"], ndepths[i], height, width, height // h)
            out = self.run_stage(i, dfe, dpr, ddv)
            prev = out
            done = torch.cuda.Event()
            done.record(compute)
            d2h.wait_event(done)
            with torch.cuda.stream(d2h):
                for k, h in host[i].items():
                    out[k].record_stream(d2h)
                    h.copy_(out[k], non_blocking=True)
        used = torch.cuda.Event()
        used.record(compute)
        self._set_done[bset] = used
        fin = torch.cuda.Event()
        fin.record(d2h)
        return HostTicket(host, fin)

    def range_hypotheses(self, depth_range: torch.Tensor, ndepth: int, b: int, h: int, w: int) -> torch.Tensor:
        """First-stage hypotheses [B,D,h,w] from the plane-sweep range [B,Dtot] (reference models/module.py:1003-1010)."""
        rng = depth_range.to(self.device, non_blocking=True)
        lo, hi = rng[:, 0], rng[:, -1]
        vals = lo.unsqueeze(1) + torch.arange(ndepth, device=self.device, dtype=torch.float32).view(1, -1) * ((hi - lo) / (ndepth - 1)).unsqueeze(1)
        return vals.view(b, -1, 1, 1).expand(b, ndepth, h, w).contiguous()

    def collect(self, ticket: "HostTicket") -> List[Dict[str, torch.Tensor]]:
        """Wait for a submitted view; the returned pinned host tensors are recycled by a later submit_host
        once `release` is called (or the ticket is dropped)."""
        ticket.event.synchronize()
        return ticket.host

    def release(self, ticket: "HostTicket") -> None:
        self._host_pool.append(ticket.host)

    @torch.no_grad()
    def run_host(self, stages: Sequence[StageInput]) -> List[Dict[str, torch.Tensor]]:
        """Host tensors in, pinned host tensors (depth, photometric_confidence, variance per stage) out.
        Returns after the results have landed on the host."""
        if getattr(self, "_last_ticket", None) is not None:
            self.release(self._last_ticket)      # buffers handed out by the previous call are recycled now
        t = self.submit_host(stages)
        self._last_ticket = t
        return self.collect(t)


class ViewPipeline:
    """K independent views in flight: one captured CUDA graph per input set (a whole 3-stage view each), replayed
    round-robin on K streams.  Reference views are independent units of work (SURVEY.md 8e), so this is the
    single-GPU form of the view sharding: kernels of different views fill each other's tails and idle issue
    slots (the conv kernels are persistent and latency-bound, the warp kernel is issue-bound).
    Measured on B200 at the DTU-test shape: 3.86 / 3.59 / 3.34 ms per view for K = 1 / 2 / 3."""

    def __init__(self, runner: "HotPathRunner", stage_sets: Sequence[Sequence[StageInput]]):
        self.runner = runner
        self.streams = [torch.cuda.Stream(device=runner.device) for _ in stage_sets]
        self.graphs, self.outputs = [], []
        for st, stream in zip(stage_sets, self.streams):
            with torch.cuda.stream(stream):
                runner.run_device(st)                       # warm-up: weight packing synchronises, fills caches
                torch.cuda.synchronize(runner.device)
                g = torch.cuda.CUDAGraph()
                with torch.cuda.graph(g, stream=stream):
                    outs = runner.run_device(st)
            self.graphs.append(g)
            self.outputs.append(outs)
        torch.cuda.synchronize(runner.device)
        self._next = 0

    def fork(self) -> None:
        """Order the K streams after everything already enqueued on the current stream."""
        ev = torch.cuda.Event()
        ev.record()
        for s in self.streams:
            s.wait_event(ev)

    def submit(self, n_views: int) -> None:
        k = len(self.graphs)
        for _ in range(n_views):
            i = self._next % k
            self._next += 1
            with torch.cuda.stream(self.streams[i]):
                self.graphs[i].replay()

    def join(self) -> None:
        """Order the current stream after the K streams (no host synchronisation)."""
        cur = torch.cuda.current_stream(self.runner.device)
        for s in self.streams:
            ev = torch.cuda.Event()
            ev.record(s)
            cur.wait_event(ev)

    def last_outputs(self) -> List[Dict[str, torch.Tensor]]:
        """The output buffers of the view submitted last (complete once the current stream has passed join())."""
        return self.outputs[(self._next - 1) % len(self.graphs)]


class HostTicket:
    def __init__(self, host, event):
        self.host = host
        self.event = event


def make_workload(height: int, width: int, nviews: int, ndepths: Sequence[int], batch: int = 1, seed: int = 0,
                  device: torch.device | str | None = None) -> List[StageInput]:
    """Synthetic three-stage DepthNet inputs of the given image size (SURVEY.md section 8d)."""
    stages = []
    for s, d in enumerate(ndepths):
        feats, proj, dv = synthetic.make_stage_inputs(s, batch, nviews, height, width, d, seed=seed)
        if device is not None:
            feats = [f.to(device) for f in feats]
            proj, dv = proj.to(device), dv.to(device)
        stages.append((feats, proj, dv))
    return stages
