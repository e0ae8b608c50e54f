"""Every training-path op against a float64 autograd reference of the same operation, op by op.

The checker is torch on the CPU in float64: F.conv3d / F.conv_transpose3d, F.batch_norm(training=True) with float64
copies of the running buffers, O.regress_head, and a warp built from the fp32 sampling coordinates of
O.relative_projection-style rot/trans + O.warp_coordinates (the rounding the kernels reproduce) cast to float64 and
sampled with O.bilinear_zeros.  Gradients are compared in G8 layout through a torch permute/view, never through the
library's own layout kernels.

bf16 cases model the kernels' 2-byte storage so that the bounds measure arithmetic, not storage: inputs, weights and
upstream gradients are bf16-representable, the raw conv output y is rounded with a straight-through bf16 round in the
forward, and gradients stored as bf16 between kernels (g_y) are rounded in the backward by `GradRound`.

Tolerances (derived, not tuned):
* fp32, one op against float64: relative L2 <= 1e-5 and elementwise <= 1e-4 * max|ref|.  fp32 arithmetic on sums of at
  most a few thousand terms has relative error ~ sqrt(n) * 2^-24 < 1e-5 in L2; the elementwise bound leaves room for
  the worst single sum (n * 2^-24 ~ 1e-4 for n ~ 1700, the largest conv reduction here).
* blocks with batch statistics: relative L2 <= 1e-4.  The normalisation divides by a std computed from fp32 partial
  sums over the whole channel and the backward subtracts two per-channel means: each step adds ~1e-6..1e-5.
* bf16 with the roundings modelled: elementwise <= 2^-7 * |ref| + floor.  One bf16 rounding of the result is 2^-8
  relative; a stored input (y) that rounds the other way at a tie contributes another 2^-8.  The floor is the fp32
  accumulation-order noise of an O(1) sum, scaled by the magnitude of the reference (2^-8 * max|ref| / 4).
"""
import copy

import pytest
import torch
import torch.nn.functional as F

from oracle import damvs_oracle as O

F64 = torch.float64


def dev():
    return torch.device("cuda:0")


# --------------------------------------------------------------------------------------------------------------------
# helpers (CPU, usable without a GPU)
# --------------------------------------------------------------------------------------------------------------------
def bfr(t):
    """Round to bf16 and back (same dtype)."""
    return t.to(torch.bfloat16).to(t.dtype)


class StraightRound(torch.autograd.Function):
    """bf16 rounding in the forward, identity in the backward (a value the kernel stores in 2 bytes)."""

    @staticmethod
    def forward(ctx, x):
        return bfr(x)

    @staticmethod
    def backward(ctx, g):
        return g


class GradRound(torch.autograd.Function):
    """Identity in the forward, bf16 rounding of the gradient in the backward (a gradient stored in 2 bytes)."""

    @staticmethod
    def forward(ctx, x):
        return x.view_as(x)

    @staticmethod
    def backward(ctx, g):
        return bfr(g)


def to_g8(x):
    """[B,C,D,H,W] -> [B,C/8,D,H,W,8] (differentiable)."""
    b, c, d, h, w = x.shape
    return x.reshape(b, c // 8, 8, d, h, w).permute(0, 1, 3, 4, 5, 2).contiguous()


def from_g8(t):
    b, g, d, h, w, _ = t.shape
    return t.permute(0, 1, 5, 2, 3, 4).reshape(b, g * 8, d, h, w)


def rel(a, b):
    a, b = a.detach().double().cpu(), b.detach().double().cpu()
    return ((a - b).norm() / b.norm().clamp_min(1e-300)).item()


def check_fp32(got, ref, name, rl2=1e-5, elt=1e-4):
    got, ref = got.detach().double().cpu(), ref.detach().double().cpu()
    assert got.shape == ref.shape, (name, got.shape, ref.shape)
    assert torch.isfinite(got).all(), name
    r = rel(got, ref)
    e = (got - ref).abs().max().item()
    m = ref.abs().max().item()
    assert r <= rl2 and e <= elt * m + 1e-30, f"{name}: rel L2 {r:.3e} (<= {rl2:.0e}), max err {e:.3e} vs {elt:.0e} * {m:.3e}"


def check_bf16(got, ref, name, floor_frac=2 ** -8 / 4, rtol=2 ** -7):
    got, ref = got.detach().double().cpu(), ref.detach().double().cpu()
    assert got.shape == ref.shape, (name, got.shape, ref.shape)
    assert torch.isfinite(got).all(), name
    floor = floor_frac * ref.abs().max().item()
    err = (got - ref).abs()
    bad = err > rtol * ref.abs() + floor
    assert not bad.any(), f"{name}: {int(bad.sum())}/{bad.numel()} outside 2^-7|ref| + {floor:.2e}; max err {err.max().item():.3e}"


def check(got, ref, name, bf16, batch=False):
    if bf16:
        check_bf16(got, ref, name)
    else:
        check_fp32(got, ref, name, rl2=1e-4 if batch else 1e-5, elt=1e-3 if batch else 1e-4)


# ---- warp / aggregation checker ----------------------------------------------------------------------------------
def warp_coords(rot_trans, dv, h, w):
    """fp32 sampling coordinates (the kernels' rounding) -> float64 ix, iy [B, D*H*W]."""
    b = rot_trans.shape[0]
    rot = rot_trans[:, :9].reshape(b, 3, 3).float()
    trans = rot_trans[:, 9:].float()
    ix, iy = O.warp_coordinates(rot, trans, dv.float(), h, w)
    d = dv.shape[1]
    return ix.expand(b, d, h * w).reshape(b, -1).double(), iy.expand(b, d, h * w).reshape(b, -1).double()


def warp64(src, coords, d, h, w):
    b, c = src.shape[:2]
    ix, iy = coords
    return O.bilinear_zeros(src, ix, iy).view(b, c, d, h, w)


def wnet_view_weight(sq, p, training, bufs=None, momentum=0.1, eps=1e-5):
    """AggWeightNetVolume restated: two 1x1x1 conv + BatchNorm + ReLU blocks on [B,C,D,H,W] -> [B,1,D,H,W].
    `p` = dict of float64 parameters (w1 [C], g1, b1, w2, g2, b2); `bufs` = dict of float64 running buffers, updated
    in place in training mode (one forward call = one update, as nn.BatchNorm3d)."""
    s = (sq * p["w1"].view(1, -1, 1, 1, 1)).sum(dim=1, keepdim=True)
    a = torch.relu(F.batch_norm(s, bufs["rm1"], bufs["rv1"], p["g1"], p["b1"], training, momentum, eps))
    t = a * p["w2"].view(())
    return torch.relu(F.batch_norm(t, bufs["rm2"], bufs["rv2"], p["g2"], p["b2"], training, momentum, eps))


def aggregate64(ref, srcs, rts, dv, mode, p=None, bufs=None, training=False):
    """Cost volume [B,C,D,H,W] in float64 from float64 NCHW features, as oracle/damvs_oracle.py:aggregate."""
    b, c, h, w = ref.shape
    d = dv.shape[1]
    ref_vol = ref.unsqueeze(2).expand(-1, -1, d, -1, -1)
    n = len(srcs)
    if mode == "variance":
        vsum, vsq = ref_vol, ref_vol ** 2
        for s, rt in zip(srcs, rts):
            wv = warp64(s, warp_coords(rt, dv, h, w), d, h, w)
            vsum = vsum + wv
            vsq = vsq + wv ** 2
        return vsq / (n + 1) - (vsum / (n + 1)) ** 2
    acc = 0
    for s, rt in zip(srcs, rts):
        sq = (ref_vol - warp64(s, warp_coords(rt, dv, h, w), d, h, w)) ** 2
        acc = acc + (wnet_view_weight(sq, p, training, bufs) + 1) * sq
    return acc / n


def make_cameras(n, b, g):
    """rot_trans [n, B, 12] fp32: view 0 near identity (taps straddle every image border: ix in (-1,0) at x = 0 and
    in (W-1,W) at x = W-1, likewise iy), view 1 shifted and slightly rotated, view 2 looking away from the scene
    (every sample out of range), further views random small motions."""
    cams = []
    for v in range(n):
        rot = torch.eye(3).expand(b, 3, 3).clone()
        trans = torch.zeros(b, 3)
        kind = v if v < 3 else 1
        if kind == 0:
            rot = rot + 1e-4 * torch.randn(b, 3, 3, generator=g)
        elif kind == 1:
            rot = rot + 0.02 * torch.randn(b, 3, 3, generator=g)
            trans = torch.tensor([1.5, -1.0, 0.05]) + 0.5 * torch.randn(b, 3, generator=g)
        else:           # every ray maps to u = v = 30 (beyond the image) at every depth
            rot = torch.tensor([[0.0, 0.0, -30.0], [0.0, 0.0, -30.0], [0.0, 0.0, -1.0]]).expand(b, 3, 3).clone()
        cams.append(torch.cat([rot.reshape(b, 9), trans], dim=1))
    return torch.stack(cams).float().contiguous()


def make_hyp(b, d, h, w, per_pixel, g):
    base = 2.0 + 0.25 * torch.arange(d, dtype=torch.float32)
    if per_pixel:
        return (base.view(1, d, 1, 1) + 0.3 * torch.rand(b, 1, h, w, generator=g)).contiguous()
    return (base.view(1, d) + 0.3 * torch.rand(b, 1, generator=g)).contiguous()


def make_wnet_params(c, g):
    return {"w1": 0.2 + 0.3 * torch.rand(c, generator=g), "g1": torch.tensor([0.9]), "b1": torch.tensor([0.2]),
            "w2": torch.tensor([0.8]), "g2": torch.tensor([1.1]), "b2": torch.tensor([0.1])}


def load_wnet(wn, p, rm=0.3, rv=1.5):
    a, b2 = wn.w_net[0], wn.w_net[1]
    with torch.no_grad():
        a.conv.weight.copy_(p["w1"].view_as(a.conv.weight))
        a.bn.weight.copy_(p["g1"]); a.bn.bias.copy_(p["b1"])
        b2.conv.weight.copy_(p["w2"].view_as(b2.conv.weight))
        b2.bn.weight.copy_(p["g2"]); b2.bn.bias.copy_(p["b2"])
        for bn in (a.bn, b2.bn):
            bn.running_mean.fill_(rm)
            bn.running_var.fill_(rv)


def wnet_leaves(p):
    return {k: v.double().clone().requires_grad_(True) for k, v in p.items()}


def wnet_bufs(rm=0.3, rv=1.5):
    return {"rm1": torch.tensor([rm], dtype=F64), "rv1": torch.tensor([rv], dtype=F64),
            "rm2": torch.tensor([rm], dtype=F64), "rv2": torch.tensor([rv], dtype=F64)}


# --------------------------------------------------------------------------------------------------------------------
# checker self-tests (CPU)
# --------------------------------------------------------------------------------------------------------------------
def _grid_sample_aggregate(ref, srcs, rts, dv, mode, wn):
    """fp32 aggregation through F.grid_sample autograd (the reference's own warp) and the module's weight net."""
    b, c, h, w = ref.shape
    d = dv.shape[1]
    ref_vol = ref.unsqueeze(2).expand(-1, -1, d, -1, -1)
    warps = []
    for s, rt in zip(srcs, rts):
        rot = rt[:, :9].reshape(b, 3, 3)
        ix, iy = O.warp_coordinates(rot, rt[:, 9:], dv, h, w)
        ix = ix.expand(b, d, h * w)
        iy = iy.expand(b, d, h * w)
        grid = torch.stack(((2 * ix + 1) / w - 1, (2 * iy + 1) / h - 1), dim=-1).view(b, d * h, w, 2)
        warps.append(F.grid_sample(s, grid, mode="bilinear", padding_mode="zeros", align_corners=False).view(b, c, d, h, w))
    if mode == "variance":
        n = len(srcs) + 1
        vsum = ref_vol + sum(warps)
        vsq = ref_vol ** 2 + sum(wv ** 2 for wv in warps)
        return vsq / n - (vsum / n) ** 2
    acc = 0
    for wv in warps:
        sq = (ref_vol - wv) ** 2
        acc = acc + (wn(sq) + 1) * sq
    return acc / len(srcs)


@pytest.mark.parametrize("mode,per_pixel", [("variance", True), ("adaptive", False), ("adaptive", True)])
def test_checker_aggregation_matches_grid_sample(mode, per_pixel):
    """The float64 checker (bilinear_zeros on fp32 coordinates) against the fp32 oracle through F.grid_sample, forward
    and feature / weight-net gradients; fp32 vs float64 on O(1) values: 1e-4 relative L2."""
    import damvsnet_b200 as dm
    g = torch.Generator().manual_seed(3)
    B, C, D, H, W, n = 2, 8, 4, 7, 11, 3
    feats = [torch.randn(B, C, H, W, generator=g) for _ in range(n + 1)]
    rts = make_cameras(n, B, g)
    dv = make_hyp(B, D, H, W, per_pixel, g)
    p = make_wnet_params(C, g)
    wn = dm.AggWeightNetVolume(C).eval()
    load_wnet(wn, p)
    f32 = [f.clone().requires_grad_(True) for f in feats]
    v32 = _grid_sample_aggregate(f32[0], f32[1:], rts, dv, mode, wn)
    r = torch.randn(v32.shape, generator=g)
    (v32 * r).sum().backward()
    f64 = [f.double().requires_grad_(True) for f in feats]
    p64 = wnet_leaves(p)
    v64 = aggregate64(f64[0], f64[1:], rts, dv, mode, p64, wnet_bufs(), False)
    (v64 * r.double()).sum().backward()
    assert rel(v32, v64) < 1e-5
    for a, b in zip(f32, f64):
        assert rel(a.grad, b.grad) < 1e-4
    if mode == "adaptive":
        assert rel(wn.w_net[0].conv.weight.grad.reshape(-1), p64["w1"].grad) < 1e-4
        assert rel(wn.w_net[1].bn.bias.grad.reshape(-1), p64["b2"].grad) < 1e-4


def test_checker_weight_net_chain_matches_module_train():
    """wnet_view_weight in training mode, called once per view, against AggWeightNetVolume.forward in train() mode:
    outputs, gradients and running buffers after the sequential updates (fp32 module vs float64 checker)."""
    import damvsnet_b200 as dm
    g = torch.Generator().manual_seed(4)
    C, n = 8, 3
    sqs = [torch.rand(2, C, 3, 5, 6, generator=g) * (v + 1) for v in range(n)]
    p = make_wnet_params(C, g)
    wn = dm.AggWeightNetVolume(C).train()
    load_wnet(wn, p)
    outs = [wn(s) for s in sqs]
    r = [torch.randn(o.shape, generator=g) for o in outs]
    sum((o * rr).sum() for o, rr in zip(outs, r)).backward()
    p64, bufs = wnet_leaves(p), wnet_bufs()
    outs64 = [wnet_view_weight(s.double(), p64, True, bufs) for s in sqs]
    sum((o * rr.double()).sum() for o, rr in zip(outs64, r)).backward()
    for o, o64 in zip(outs, outs64):
        assert rel(o, o64) < 1e-5
    a, b2 = wn.w_net[0], wn.w_net[1]
    for got, k in ((a.conv.weight, "w1"), (a.bn.weight, "g1"), (a.bn.bias, "b1"), (b2.bn.weight, "g2"), (b2.bn.bias, "b2")):
        assert rel(got.grad.reshape(-1), p64[k].grad) < 1e-4, k
    for got, k in ((a.bn.running_mean, "rm1"), (a.bn.running_var, "rv1"), (b2.bn.running_mean, "rm2"), (b2.bn.running_var, "rv2")):
        assert rel(got, bufs[k]) < 1e-6, k
    assert int(a.bn.num_batches_tracked) == n


def test_grad_round_helpers():
    x = torch.tensor([1.0 + 2 ** -10, 3.0], requires_grad=True)
    y = StraightRound.apply(x)
    assert y[0].item() == 1.0
    GradRound.apply(y).backward(torch.tensor([1.0 + 2 ** -10, 2.0]))
    assert x.grad[0].item() == 1.0 and x.grad[1].item() == 2.0


# --------------------------------------------------------------------------------------------------------------------
# GPU tests
# --------------------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def dm():
    import damvsnet_b200 as dm
    from damvsnet_b200 import _lib
    _lib.check(_lib.load().damvs_check_device(0))
    return dm


# ---- BatchNorm kernels, called directly ----------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("stats", ["batch", "batch_cumulative", "fixed"])
@pytest.mark.parametrize("relu,skip", [(True, True), (True, False), (False, True), (False, False)])
@pytest.mark.parametrize("offset", [0, 10, 100])
@pytest.mark.parametrize("C", [8, 64])
@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
def test_bn_kernels_match_float64(dm, dtype, C, offset, relu, skip, stats):
    """bn_stats / bn_finalize / bn_apply / bn_bwd / bn_bwd_coeffs exactly as ConvBlockFn chains them, against
    F.batch_norm in float64.  5895 voxels per (batch, channel group): one full 256 x 16 reduction block and a ragged
    one.  Channel means sit `offset` standard deviations from zero: the sums must not lose the variance to
    cancellation.  The ReLU mask is the kernel's own pre-activation sign (bn_apply without ReLU), so an element whose
    pre-activation is within rounding of zero cannot flip between kernel and reference.  Bounds: module docstring
    (fp32 outputs 1e-5 relative L2, batch statistics 1e-4; bf16: 2^-7 |ref| + floor)."""
    from damvsnet_b200 import ops_train
    bf = dtype == torch.bfloat16
    batch = stats != "fixed"
    g = torch.Generator().manual_seed(C * 7 + offset + 3 * relu + skip)
    B, D, H, W = 2, 5, 9, 131
    m = B * D * H * W
    std = 0.5 + 1.5 * torch.rand(C, generator=g, dtype=F64)
    mu = offset * std * torch.where(torch.rand(C, generator=g) < 0.5, -1.0, 1.0).double()
    y = mu.view(1, C, 1, 1, 1) + std.view(1, C, 1, 1, 1) * torch.randn(B, C, D, H, W, generator=g, dtype=F64)
    y = y.to(dtype).double()
    gamma = 0.5 + torch.rand(C, generator=g, dtype=F64)
    beta = 0.2 * torch.randn(C, generator=g, dtype=F64)
    rm0 = mu + 0.1 * torch.randn(C, generator=g, dtype=F64)
    rv0 = (std * (0.8 + 0.4 * torch.rand(C, generator=g, dtype=F64))) ** 2
    rm0, rv0 = rm0.float().double(), rv0.float().double()
    sk = torch.randn(B, C, D, H, W, generator=g, dtype=F64).to(dtype).double() if skip else None
    gout = torch.randn(B, C, D, H, W, generator=g, dtype=F64).to(dtype).double()
    momentum = 1.0 / 3 if stats == "batch_cumulative" else 0.1   # momentum None at num_batches_tracked = 3

    yd = to_g8(y).to(dtype).to(dev())
    gamma_d, beta_d = gamma.float().to(dev()), beta.float().to(dev())
    rm_d, rv_d = rm0.float().to(dev()), rv0.float().to(dev())
    if batch:
        sums = ops_train.bn_stats(yd)
        scale, shift, mean, rstd = ops_train.bn_finalize(sums, gamma_d, beta_d, rm_d, rv_d, m, momentum, 1e-5)
    else:
        mean, rstd = rm_d, torch.rsqrt(rv_d + 1e-5)
        scale = gamma_d * rstd
        shift = beta_d - mean * scale
    z_k = ops_train.bn_apply(yd, scale, shift, None, False)
    out = ops_train.bn_apply(yd, scale, shift, None if sk is None else to_g8(sk).to(dtype).to(dev()), relu)
    god = to_g8(gout).to(dtype).to(dev())
    if batch:
        _, s2 = ops_train.bn_bwd(god, yd, scale, shift, None, None, None, relu, False, True)
        k1, k2, k3, dgamma, dbeta = ops_train.bn_bwd_coeffs(s2, scale, mean, rstd, m, True)
        g_y, _ = ops_train.bn_bwd(god, yd, scale, shift, k1, k2, k3, relu, True, False)
    else:
        g_y, s2 = ops_train.bn_bwd(god, yd, scale, shift, scale, None, None, relu, True, True)
        _, _, _, dgamma, dbeta = ops_train.bn_bwd_coeffs(s2, scale, mean, rstd, m, False)

    yr = y.clone().requires_grad_(True)
    gr, br = gamma.clone().requires_grad_(True), beta.clone().requires_grad_(True)
    rm, rv = rm0.clone(), rv0.clone()
    z = F.batch_norm(yr, rm, rv, gr, br, batch, momentum, 1e-5)
    mask = (from_g8(z_k.cpu().double()) > 0).double() if relu else torch.ones_like(y)
    o = z * mask + (sk if sk is not None else 0)
    (o * gout).sum().backward()

    name = f"{dtype} C={C} offset={offset} {stats}"
    check(from_g8(out.cpu()), o, "out " + name, bf, batch)
    check(from_g8(g_y.cpu()), yr.grad, "g_y " + name, bf, batch)
    check_fp32(dgamma, gr.grad, "g_gamma " + name, rl2=1e-4 if batch else 1e-5, elt=1e-3 if batch else 1e-4)
    check_fp32(dbeta, br.grad, "g_beta " + name, elt=1e-4)
    if batch:
        # the mean is stored in fp32 (half an ulp of |mean|); its arithmetic error scales with the channel's spread
        ym = y.mean(dim=(0, 2, 3, 4))
        assert ((mean.cpu().double() - ym).abs() <= 2 ** -24 * ym.abs() + 1e-6 * std).all(), "mean " + name
        check_fp32(rstd, 1 / torch.sqrt(y.var(dim=(0, 2, 3, 4), unbiased=False) + 1e-5), "rstd " + name, rl2=1e-5, elt=1e-5)
        check_fp32(rm_d, rm, "running_mean " + name, rl2=1e-6, elt=1e-6)
        check_fp32(rv_d, rv, "running_var " + name, rl2=1e-5, elt=1e-5)


# ---- conv blocks through ConvBlockFn -----------------------------------------------------------------------------
LAYERS = [  # cin, cout, stride, transposed: the 11 CostRegNet layers at base channels 8 (conv0 .. conv11)
    (8, 8, 1, False), (8, 16, 2, False), (16, 16, 1, False), (16, 32, 2, False), (32, 32, 1, False),
    (32, 64, 2, False), (64, 64, 1, False), (64, 32, 2, True), (32, 16, 2, True), (16, 8, 2, True),
]


def _make_block(dm, cin, cout, stride, tr, bn, relu, g):
    if tr:
        blk = dm.Deconv3d(cin, cout, stride=2, relu=relu, bn=bn, padding=1, output_padding=1)
    else:
        blk = dm.Conv3d(cin, cout, stride=stride, relu=relu, bn=bn, padding=1)
    with torch.no_grad():
        blk.conv.weight.copy_(bfr(0.3 * torch.randn(blk.conv.weight.shape, generator=g) / (cin ** 0.5)))
        if bn:
            blk.bn.weight.copy_(0.8 + 0.4 * torch.rand(cout, generator=g))
            blk.bn.bias.copy_(0.1 * torch.randn(cout, generator=g))
            blk.bn.running_mean.copy_(0.05 * torch.randn(cout, generator=g))
            blk.bn.running_var.copy_(0.5 + torch.rand(cout, generator=g))
        else:
            blk.conv.bias.copy_(0.1 * torch.randn(cout, generator=g))
    return blk


def _block_reference(blk, x, skip, gout, train, bf):
    """float64 conv -> BatchNorm -> ReLU (+ skip) with autograd; returns output and gradients."""
    tr, bn = blk.transposed, blk.bn
    xr = x.double().clone().requires_grad_(True)
    w = blk.conv.weight.detach().double().clone().requires_grad_(True)
    bias = blk.conv.bias.detach().double().clone().requires_grad_(True) if blk.conv.bias is not None else None
    y = F.conv_transpose3d(xr, w, None, stride=2, padding=1, output_padding=1) if tr else F.conv3d(xr, w, None, stride=blk.stride, padding=1)
    if bf:
        y = GradRound.apply(StraightRound.apply(y))
    res = {"x": xr, "w": w}
    bufs = None
    if bn is not None:
        gm = bn.weight.detach().double().clone().requires_grad_(True)
        bt = bn.bias.detach().double().clone().requires_grad_(True)
        rm, rv = bn.running_mean.detach().double().clone(), bn.running_var.detach().double().clone()
        z = F.batch_norm(y, rm, rv, gm, bt, train, bn.momentum, bn.eps)
        res.update(gamma=gm, beta=bt)
        bufs = (rm, rv)
    else:
        z = y + bias.view(1, -1, 1, 1, 1)
        res["bias"] = bias
    a = torch.relu(z) if blk.relu else z
    sr = None
    if skip is not None:
        sr = skip.double().clone().requires_grad_(True)
        a = a + sr
    (a * gout.double()).sum().backward()
    return a.detach(), res, sr, bufs


def _run_block(dm, prec, impl, cin, cout, stride, tr, ext, bn=True, relu=True, train=True, with_skip=False, seed=0):
    g = torch.Generator().manual_seed(seed + cin * 100 + cout + 7 * stride + 3 * tr)
    blk = _make_block(dm, cin, cout, stride, tr, bn, relu, g)
    B = 2
    x = bfr(torch.randn(B, cin, *ext, generator=g))
    d, h, w = ext
    oext = (2 * d, 2 * h, 2 * w) if tr else tuple((n - 1) // stride + 1 for n in ext)
    skip = bfr(torch.randn(B, cout, *oext, generator=g)) if with_skip else None
    gout = bfr(torch.randn(B, cout, *oext, generator=g))
    bf = prec == "bf16"
    blk.train(train)
    ref_blk = copy.deepcopy(blk)
    dtype = torch.bfloat16 if bf else torch.float32
    blk = blk.to(dev())
    with dm.precision(prec, impl):
        xd = to_g8(x).to(dtype).to(dev()).requires_grad_(True)
        sd = to_g8(skip).to(dtype).to(dev()).requires_grad_(True) if skip is not None else None
        out = blk.forward_g8(dm.G8Volume(xd), None if sd is None else dm.G8Volume(sd)).data
        (out.float() * to_g8(gout).to(dev())).sum().backward()
    want, res, sr, bufs = _block_reference(ref_blk, x, skip, gout, train, bf)
    batch = bn and train
    name = f"{prec}/{impl} {cin}->{cout} s{stride}{'T' if tr else ''} {ext} bn={bn} relu={relu} train={train}"
    check(from_g8(out.detach().cpu()), want, "out " + name, bf, batch)
    check(from_g8(xd.grad.cpu()), res["x"].grad, "g_x " + name, bf, batch)
    # weight / affine gradients are sums over every voxel in fp32 (bf16 operands): fp32-style relative L2 bounds
    wtol = 4e-3 if bf else (1e-4 if batch else 1e-5)
    assert rel(blk.conv.weight.grad.cpu(), res["w"].grad) <= wtol, ("g_w " + name, rel(blk.conv.weight.grad.cpu(), res["w"].grad))
    if bn:
        assert rel(blk.bn.weight.grad.cpu(), res["gamma"].grad) <= wtol, ("g_gamma " + name, rel(blk.bn.weight.grad.cpu(), res["gamma"].grad))
        assert rel(blk.bn.bias.grad.cpu(), res["beta"].grad) <= wtol, ("g_beta " + name, rel(blk.bn.bias.grad.cpu(), res["beta"].grad))
        if train:
            torch.testing.assert_close(blk.bn.running_mean.cpu().double(), bufs[0], rtol=1e-5 if not bf else 4e-3, atol=1e-6)
            torch.testing.assert_close(blk.bn.running_var.cpu().double(), bufs[1], rtol=1e-5 if not bf else 4e-3, atol=1e-6)
            assert int(blk.bn.num_batches_tracked) == 1
        else:
            assert int(blk.bn.num_batches_tracked) == 0
    else:
        assert blk.conv.bias.grad is not None, "conv bias gradient missing: " + name
        assert rel(blk.conv.bias.grad.cpu(), res["bias"].grad) <= wtol, ("g_bias " + name, rel(blk.conv.bias.grad.cpu(), res["bias"].grad))
    if skip is not None:
        check(from_g8(sd.grad.float().cpu()), sr.grad, "g_skip " + name, bf)


@pytest.mark.gpu
@pytest.mark.parametrize("cin,cout,stride,tr", LAYERS)
@pytest.mark.parametrize("train", [True, False])
def test_conv_block_fp32(dm, cin, cout, stride, tr, train):
    """fp32 (direct kernels): forward, g_x through the adjoint convolution, g_w, BatchNorm gradients and buffers;
    ragged extents (5 x 7 x 19 in, 3 x 4 x 10 for the decoder layers), skip on the transposed layers."""
    ext = (3, 4, 10) if tr else (5, 7, 19)
    _run_block(dm, "fp32", "direct", cin, cout, stride, tr, ext, train=train, with_skip=tr)


@pytest.mark.gpu
@pytest.mark.parametrize("cin,cout,stride,tr", LAYERS)
@pytest.mark.parametrize("impl", ["tcgen05", "direct"])
def test_conv_block_bf16(dm, cin, cout, stride, tr, impl):
    """bf16 with the raw output and g_y roundings modelled (module docstring); both convolution implementations."""
    ext = (2, 4, 9) if tr else (4, 8, 18)
    _run_block(dm, "bf16", impl, cin, cout, stride, tr, ext, train=True, with_skip=tr)


@pytest.mark.gpu
@pytest.mark.parametrize("ext", [(5, 7, 9), (1, 3, 5), (3, 1, 2)])
@pytest.mark.parametrize("cin,cout", [(8, 16), (16, 32)])
def test_conv_block_stride2_odd_extents(dm, cin, cout, ext):
    """Stride-2 Conv3d over odd extents: the adjoint (transposed) convolution yields one extra plane, which the data
    gradient must crop; extents smaller than one tile."""
    _run_block(dm, "fp32", "direct", cin, cout, 2, False, ext)


@pytest.mark.gpu
@pytest.mark.parametrize("bn,relu", [(False, True), (False, False), (True, False)])
@pytest.mark.parametrize("prec", ["fp32", "bf16"])
def test_conv_block_without_bn_or_relu(dm, bn, relu, prec):
    """Conv3d(bn=False) trains its conv bias (the shift of the BatchNorm-less block) and relu=False passes the gradient
    everywhere; with a skip input."""
    _run_block(dm, prec, "direct", 8, 16, 1, False, (3, 6, 11), bn=bn, relu=relu, with_skip=True)


@pytest.mark.gpu
@pytest.mark.parametrize("ext", [(1, 3, 5), (2, 2, 2)])
def test_conv_block_smaller_than_tile(dm, ext):
    _run_block(dm, "fp32", "direct", 8, 8, 1, False, ext)
    _run_block(dm, "bf16", "tcgen05", 8, 8, 1, False, ext)


# ---- prob conv -----------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("prec", ["fp32", "bf16"])
def test_prob_conv_gradients(dm, prec):
    """ProbConvFn (8 -> 1, fp32 logits): g_x through the zero-padded adjoint and plain_to_g8, g_w; ragged 5 x 9 x 21."""
    from damvsnet_b200 import autograd as ag
    g = torch.Generator().manual_seed(11)
    bf = prec == "bf16"
    dtype = torch.bfloat16 if bf else torch.float32
    net = dm.CostRegNet(8, 8)
    with torch.no_grad():
        net.prob.weight.copy_(bfr(0.2 * torch.randn(net.prob.weight.shape, generator=g)))
    B, D, H, W = 2, 5, 9, 21
    x = bfr(torch.randn(B, 8, D, H, W, generator=g))
    r = torch.randn(B, D, H, W, generator=g)
    xr = x.double().requires_grad_(True)
    wr = net.prob.weight.detach().double().clone().requires_grad_(True)
    lo = F.conv3d(xr, wr, None, padding=1)[:, 0]
    ((GradRound.apply(lo) if bf else lo) * r.double()).sum().backward()   # plain_to_g8 stores the logit gradient in bf16
    net = net.to(dev())
    with dm.precision(prec, "tcgen05" if bf else "direct"):
        xd = to_g8(x).to(dtype).to(dev()).requires_grad_(True)
        logits = ag.ProbConvFn.apply(xd, net.prob.weight, net)
        (logits * r.to(dev())).sum().backward()
    check_fp32(logits, lo, "logits")             # fp32 logits of bf16-representable operands in both precisions
    check(from_g8(xd.grad.float().cpu()), xr.grad, "g_x", bf)
    assert rel(net.prob.weight.grad.cpu(), wr.grad) <= (1e-4 if bf else 1e-5), rel(net.prob.weight.grad.cpu(), wr.grad)


# ---- head ----------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("which", ["all", "depth", "variance", "prob"])
@pytest.mark.parametrize("per_pixel", [True, False])
@pytest.mark.parametrize("D", [2, 8, 12, 48, 64, 96, 100])
def test_head_backward(dm, D, per_pixel, which):
    """HeadFn / softmax_regress_bwd against autograd of O.regress_head in float64: g_logits and (per-pixel) g_hyp;
    each upstream gradient alone and all together; 7 x 13 pixels (not a multiple of 4); a third of the pixels
    peaked (logit gap 60: variance sum near underflow) must still give finite gradients.  fp32 single-op bounds."""
    from damvsnet_b200 import autograd as ag
    g = torch.Generator().manual_seed(D * 10 + per_pixel)
    B, H, W = 2, 7, 13
    logits = torch.randn(B, D, H, W, generator=g)
    peak = torch.rand(B, 1, H, W, generator=g) < 0.33
    logits = torch.where(peak & (torch.arange(D).view(1, D, 1, 1) == D // 2), logits + 60.0, logits)
    hyp = make_hyp(B, D, H, W, True, g) * 100
    if not per_pixel:
        hyp2 = hyp[:, :, 0, 0].contiguous()
        hyp = hyp2.view(B, D, 1, 1).expand(B, D, H, W)
    r_d = torch.randn(B, H, W, generator=g) if which in ("all", "depth") else torch.zeros(B, H, W)
    r_v = torch.randn(B, H, W, generator=g) if which in ("all", "variance") else torch.zeros(B, H, W)
    r_p = torch.randn(B, D, H, W, generator=g) if which in ("all", "prob") else torch.zeros(B, D, H, W)
    lr = logits.double().requires_grad_(True)
    hr = hyp.double().clone().requires_grad_(True)
    o = O.regress_head(lr, hr)
    ((o["depth"] * r_d).sum() + (o["variance"] * r_v).sum() + (o["prob_volume"] * r_p).sum()).backward()
    ld = logits.to(dev()).requires_grad_(True)
    hd = (hyp.contiguous() if per_pixel else hyp2).to(dev()).requires_grad_(per_pixel)
    if per_pixel:
        prob, depth, conf, var = ag.HeadFn.apply(ld, hd)
    else:
        prob, depth, conf, var = ag.HeadFn.apply(ld, hd.view(B, D, 1, 1).expand(B, D, H, W).contiguous())
    ((depth * r_d.to(dev())).sum() + (var * r_v.to(dev())).sum() + (prob * r_p.to(dev())).sum()).backward()
    assert torch.isfinite(ld.grad).all()
    check_fp32(depth, o["depth"], "depth")
    check_fp32(var, o["variance"], "variance", elt=1e-4)
    check_fp32(ld.grad, lr.grad, f"g_logits D={D} {which}")
    if per_pixel:
        check_fp32(hd.grad, hr.grad, f"g_hyp D={D} {which}")


# ---- warp + aggregation ------------------------------------------------------------------------------------------
def _warp_inputs(C, n, per_pixel, seed):
    g = torch.Generator().manual_seed(seed)
    B, D, H, W = 2, 5, 9, 13
    feats = [torch.randn(B, C, H, W, generator=g) for _ in range(n + 1)]
    rts = make_cameras(n, B, g)
    dv = make_hyp(B, D, H, W, per_pixel, g)
    return g, feats, rts, dv


@pytest.mark.gpu
@pytest.mark.parametrize("gdt", [torch.float32, torch.bfloat16])
@pytest.mark.parametrize("per_pixel", [True, False])
@pytest.mark.parametrize("n", [1, 2, 6])
@pytest.mark.parametrize("C", [8, 16, 32])
@pytest.mark.parametrize("mode", ["variance", "adaptive"])
def test_warp_agg_backward(dm, mode, C, n, per_pixel, gdt):
    """WarpAggFn (warp_agg_bwd): variance and adaptive-eval aggregation; feature gradients (the bilinear atomic
    scatter with its own border clamping) and, adaptive, the gradients of the weight net's conv weights, gamma and
    beta through folded_with_grad.  Cameras straddle every image border and one looks away.  g_vol in fp32 and bf16
    (the upstream gradient is bf16-representable, so the bf16 case changes storage only).  fp32 single-op bounds."""
    from damvsnet_b200 import autograd as ag
    g, feats, rts, dv = _warp_inputs(C, n, per_pixel, C * 10 + n + 100 * per_pixel)
    p = make_wnet_params(C, g)
    f64 = [f.double().requires_grad_(True) for f in feats]
    p64 = wnet_leaves(p)
    want = aggregate64(f64[0], f64[1:], rts, dv, mode, p64, wnet_bufs(), False)
    r = bfr(torch.randn(want.shape, generator=g))
    (want * r.double()).sum().backward()
    wn = None
    if mode == "adaptive":
        wn = dm.AggWeightNetVolume(C).eval()
        load_wnet(wn, p)
        wn = wn.to(dev())
    fs = [f.to(dev()).requires_grad_(True) for f in feats]
    nhwc = [ag.NhwcFn.apply(f) for f in fs]
    wnet = wn.folded_with_grad() if wn is not None else None
    vol = ag.WarpAggFn.apply(wnet, rts.to(dev()), dv.to(dev()), mode, gdt, *nhwc)
    (vol.float() * to_g8(r).to(dev())).sum().backward()
    name = f"{mode} C={C} n={n} per_pixel={per_pixel} {gdt}"
    if gdt == torch.bfloat16:
        check_bf16(from_g8(vol.detach().cpu()), want.detach(), "vol " + name)
    else:
        check_fp32(from_g8(vol.detach().cpu()), want.detach(), "vol " + name)
    for i, (a, b) in enumerate(zip(fs, f64)):
        check_fp32(a.grad, b.grad, f"g_feat[{i}] " + name)
    if wn is not None:
        a_, b_ = wn.w_net[0], wn.w_net[1]
        check_fp32(a_.conv.weight.grad.reshape(-1), p64["w1"].grad, "g_w1 " + name)
        # each scalar gradient is one fp32 atomic sum over B*D*H*W*n voxels of terms of both signs (and d gamma a difference
        # of two: (d scale - running_mean * d shift) * rstd), accumulated in a run-dependent order; the cancellation
        # amplifies the rounding: measured on the B200 up to 2.4e-4 relative (g_w2, C = 8, n = 6)
        for got, k in ((a_.bn.weight, "g1"), (a_.bn.bias, "b1"), (b_.conv.weight, "w2"), (b_.bn.weight, "g2"), (b_.bn.bias, "b2")):
            check_fp32(got.grad.reshape(-1), p64[k].grad, f"g_{k} " + name, rl2=1e-3, elt=1e-3)


def _train_chain_run(dm, C, n, per_pixel, gdt, seed):
    from damvsnet_b200 import autograd as ag
    g, feats, rts, dv = _warp_inputs(C, n, per_pixel, seed)
    p = make_wnet_params(C, g)
    f64 = [f.double().requires_grad_(True) for f in feats]
    p64, bufs = wnet_leaves(p), wnet_bufs()
    want = aggregate64(f64[0], f64[1:], rts, dv, "adaptive", p64, bufs, True)
    r = bfr(torch.randn(want.shape, generator=g))
    (want * r.double()).sum().backward()
    wn = dm.AggWeightNetVolume(C).train()
    load_wnet(wn, p)
    wn = wn.to(dev())
    a, b2 = wn.w_net[0], wn.w_net[1]
    fs = [f.to(dev()).requires_grad_(True) for f in feats]
    nhwc = [ag.NhwcFn.apply(f) for f in fs]
    vol = ag.WarpAdaptiveTrainFn.apply(a.conv.weight, a.bn.weight, a.bn.bias, b2.conv.weight, b2.bn.weight, b2.bn.bias,
                                       rts.to(dev()), dv.to(dev()), gdt, wn, *nhwc)
    (vol.float() * to_g8(r).to(dev())).sum().backward()
    return want, f64, p64, bufs, vol, fs, wn


@pytest.mark.gpu
@pytest.mark.parametrize("gdt", [torch.float32, torch.bfloat16])
@pytest.mark.parametrize("per_pixel", [True, False])
@pytest.mark.parametrize("n", [1, 2, 6])
@pytest.mark.parametrize("C", [8, 16, 32])
def test_warp_adaptive_train(dm, C, n, per_pixel, gdt):
    """WarpAdaptiveTrainFn (warp_score_fwd -> wnet_chain_fwd -> warp_weighted_fwd; warp_gwt -> wnet_chain_bwd ->
    warp_merged_bwd) against the float64 checker with one weight-net call per source view (batch statistics per view,
    running buffers updated view by view): volume, feature gradients, g_w1, the five scalar-chain gradients, both
    BatchNorms' running buffers and num_batches_tracked += n.  Batch-statistics bounds (1e-4 relative L2)."""
    want, f64, p64, bufs, vol, fs, wn = _train_chain_run(dm, C, n, per_pixel, gdt, C * 10 + n + 100 * per_pixel + 1)
    name = f"C={C} n={n} per_pixel={per_pixel} {gdt}"
    if gdt == torch.bfloat16:
        check_bf16(from_g8(vol.detach().cpu()), want.detach(), "vol " + name)
    else:
        check_fp32(from_g8(vol.detach().cpu()), want.detach(), "vol " + name, rl2=1e-4, elt=1e-3)
    for i, (a, b) in enumerate(zip(fs, f64)):
        check_fp32(a.grad, b.grad, f"g_feat[{i}] " + name, rl2=1e-4, elt=1e-3)
    a_, b_ = wn.w_net[0], wn.w_net[1]
    for got, k in ((a_.conv.weight, "w1"), (a_.bn.weight, "g1"), (a_.bn.bias, "b1"), (b_.bn.weight, "g2"), (b_.bn.bias, "b2")):
        check_fp32(got.grad.reshape(-1), p64[k].grad, f"g_{k} " + name, rl2=1e-4, elt=1e-3)
    # w2 feeds a batch-statistics BatchNorm directly: its true gradient is zero up to eps effects
    assert abs(b_.conv.weight.grad.item() - p64["w2"].grad.item()) <= 1e-3 * (1.0 + p64["g1"].grad.abs().item())
    for got, k in ((a_.bn.running_mean, "rm1"), (a_.bn.running_var, "rv1"), (b_.bn.running_mean, "rm2"), (b_.bn.running_var, "rv2")):
        check_fp32(got.cpu(), bufs[k], f"{k} " + name, rl2=1e-5, elt=1e-5)
    assert int(a_.bn.num_batches_tracked) == n and int(b_.bn.num_batches_tracked) == n


@pytest.mark.gpu
def test_wnet_chain_direct(dm):
    """wnet_chain_fwd / wnet_chain_bwd called directly on score volumes with a mean offset, against the float64 chain."""
    from damvsnet_b200 import ops_train
    g = torch.Generator().manual_seed(21)
    n, M = 3, 3 * 4 * 37 * 41
    s = (5.0 + torch.rand(n, 3, 4, 37, 41, generator=g) * torch.arange(1, n + 1).view(n, 1, 1, 1, 1)).contiguous()
    gw = torch.randn(s.shape, generator=g)
    p = make_wnet_params(8, g)
    wn = dm.AggWeightNetVolume(8).train()
    load_wnet(wn, p)
    wn = wn.to(dev())
    a, b2 = wn.w_net[0], wn.w_net[1]
    wt, state = ops_train.wnet_chain_fwd(s.to(dev()), a.bn, b2.conv.weight, b2.bn)
    g_s, gp = ops_train.wnet_chain_bwd(s.to(dev()), gw.to(dev()), state, b2.conv.weight)
    p64, bufs = wnet_leaves(p), wnet_bufs()
    sr = s.double().requires_grad_(True)
    outs = []
    for v in range(n):
        x = sr[v].unsqueeze(1)
        h = torch.relu(F.batch_norm(x, bufs["rm1"], bufs["rv1"], p64["g1"], p64["b1"], True, 0.1, 1e-5))
        outs.append(torch.relu(F.batch_norm(h * p64["w2"].view(()), bufs["rm2"], bufs["rv2"], p64["g2"], p64["b2"], True, 0.1, 1e-5)))
    want = torch.stack([o.squeeze(1) for o in outs])
    (want * gw.double()).sum().backward()
    check_fp32(wt, want, "wt", rl2=1e-4, elt=1e-3)
    check_fp32(g_s, sr.grad, "g_s", rl2=1e-4, elt=1e-3)
    ref_gp = torch.stack([p64[k].grad.reshape(()) for k in ("g1", "b1", "w2", "g2", "b2")])
    for i in (0, 1, 3, 4):
        assert abs(gp[i].item() - ref_gp[i].item()) <= 1e-4 * ref_gp[i].abs().item() + 1e-6, (i, gp.tolist(), ref_gp.tolist())
    for got, k in ((a.bn.running_mean, "rm1"), (a.bn.running_var, "rv1"), (b2.bn.running_mean, "rm2"), (b2.bn.running_var, "rv2")):
        check_fp32(got.cpu(), bufs[k], k, rl2=1e-5, elt=1e-5)
    assert int(a.bn.num_batches_tracked) == n


# ---- weight gradient kernel: extents the existing test does not reach ---------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("B,ext", [(2, (1, 3, 5)), (2, (5, 7, 9)), (3, (48, 3, 5))])
@pytest.mark.parametrize("cin,cout,stride,tr", [(8, 8, 1, False), (8, 16, 2, False), (16, 8, 2, True), (8, 1, 1, False)])
def test_conv_wgrad_edges(dm, B, ext, cin, cout, stride, tr):
    """conv3d_wgrad on extents smaller than one tile, odd stride-2 inputs, 48 planes and B = 3; bf16 (mma kernel) with
    bf16 operands (sums of fp32 products: 1e-5 relative L2 up to accumulation order, bounded at 1e-4) and fp32
    (CUDA-core kernel, 1e-5)."""
    from damvsnet_b200 import ops_train
    g = torch.Generator().manual_seed(cin + cout + sum(ext) + B)
    x = bfr(torch.randn(B, cin, *ext, generator=g)).double()
    w = torch.randn((cin, cout, 3, 3, 3) if tr else (cout, cin, 3, 3, 3), generator=g, dtype=F64).requires_grad_(True)
    y = F.conv_transpose3d(x, w, None, stride=2, padding=1, output_padding=1) if tr else F.conv3d(x, w, None, stride=stride, padding=1)
    gy = bfr(torch.randn(y.shape, generator=g, dtype=F64))
    (y * gy).sum().backward()
    gy_p = gy
    if cout % 8:
        gy_p = torch.zeros(B, 8, *gy.shape[2:], dtype=F64)
        gy_p[:, :cout] = gy
    for dtype, tol in ((torch.bfloat16, 1e-4), (torch.float32, 1e-5)):
        dw = ops_train.conv3d_wgrad(to_g8(x).to(dtype).to(dev()), to_g8(gy_p).to(dtype).to(dev()), cin, cout, stride, tr).cpu()
        assert dw.shape == w.shape
        assert rel(dw, w.grad) <= tol, (dtype, rel(dw, w.grad))


# ---- reference-signature entry points ------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["conv_s1", "conv_s2_odd", "deconv"])
def test_reference_signature_blocks_propagate_gradients(dm, kind):
    """Conv3d / Deconv3d.forward(x) on [B,C,D,H,W] fp32 with x requiring grad: x.grad and the parameter gradients equal
    the float64 reference (the layout conversions are differentiable)."""
    g = torch.Generator().manual_seed(31)
    if kind == "deconv":
        blk, ext = _make_block(dm, 16, 8, 2, True, True, True, g), (2, 3, 5)
    else:
        blk, ext = _make_block(dm, 8, 16, 2 if kind == "conv_s2_odd" else 1, False, True, True, g), (5, 7, 9)
    blk.train()
    ref_blk = copy.deepcopy(blk)
    x = torch.randn(2, blk.in_channels, *ext, generator=g)
    with dm.precision("fp32"):
        blk = blk.to(dev())
        xd = x.to(dev()).requires_grad_(True)
        out = blk(xd)
        assert out.grad_fn is not None
        r = torch.randn(out.shape, generator=g)
        (out * r.to(dev())).sum().backward()
    want, res, _, _ = _block_reference(ref_blk, x, None, r, True, False)
    check_fp32(out.detach(), want, "out", rl2=1e-4, elt=1e-3)
    assert xd.grad is not None
    check_fp32(xd.grad, res["x"].grad, "g_x", rl2=1e-4, elt=1e-3)
    assert rel(blk.conv.weight.grad.cpu(), res["w"].grad) <= 1e-4


@pytest.mark.gpu
def test_reference_signature_costregnet_propagates_gradients(dm):
    """CostRegNet.forward(x) with x requiring grad: x.grad equals the float64 oracle network.  Ten chained
    batch-statistics BatchNorms, the deepest over 2 x 2 x 2 voxels per batch item, amplify fp32 rounding: 1e-3."""
    g = torch.Generator().manual_seed(32)
    net = dm.CostRegNet(8, 8)
    sd = {k: v.clone() for k, v in net.state_dict().items()}
    for k in sd:
        if k.endswith("conv.weight") or k == "prob.weight":
            sd[k] = 0.3 * torch.randn(sd[k].shape, generator=g) / (sd[k].shape[1] ** 0.5)
    net.load_state_dict(sd)
    net.train()
    x = torch.randn(2, 8, 16, 16, 16, generator=g)
    r = torch.randn(2, 1, 16, 16, 16, generator=g)
    xr = x.double().requires_grad_(True)
    sd64 = {"cost_regularization.0." + k: v.double() for k, v in sd.items()}
    (O.cost_reg_net(xr, sd64, 0, training=True) * r.double()).sum().backward()
    with dm.precision("fp32"):
        net = net.to(dev())
        xd = x.to(dev()).requires_grad_(True)
        out = net(xd)
        (out * r.to(dev())).sum().backward()
    assert xd.grad is not None
    check_fp32(xd.grad, xr.grad, "CostRegNet g_x", rl2=1e-3, elt=1e-2)


@pytest.mark.gpu
@pytest.mark.parametrize("per_pixel", [True, False])
def test_depth_regression_gradients(dm, per_pixel):
    g = torch.Generator().manual_seed(33)
    B, D, H, W = 2, 7, 5, 9
    p = torch.softmax(torch.randn(B, D, H, W, generator=g), 1)
    dv = make_hyp(B, D, H, W, per_pixel, g)
    r = torch.randn(B, H, W, generator=g)
    pr, dr = p.double().requires_grad_(True), dv.double().requires_grad_(True)
    (O.depth_regression(pr, dr) * r.double()).sum().backward()
    pd, dd = p.to(dev()).requires_grad_(True), dv.to(dev()).requires_grad_(True)
    out = dm.depth_regression(pd, dd)
    (out * r.to(dev())).sum().backward()
    check_fp32(pd.grad, pr.grad, "g_p")
    check_fp32(dd.grad, dr.grad, "g_dv")


@pytest.mark.gpu
def test_homo_warping_refuses_gradients(dm):
    """homo_warping has no backward kernel: with inputs that require grad it raises instead of detaching."""
    g = torch.Generator().manual_seed(34)
    src = torch.randn(1, 8, 6, 10, generator=g, device="cpu").to(dev())
    proj = torch.eye(4).view(1, 4, 4).to(dev())
    dv = make_hyp(1, 4, 6, 10, False, g).to(dev())
    out = dm.homo_warping(src, proj, proj, dv)
    assert out.shape == (1, 8, 4, 6, 10)
    with pytest.raises(NotImplementedError):
        dm.homo_warping(src.requires_grad_(True), proj, proj, dv)


# ---- NaN propagation through the head kernels ---------------------------------------------------------------------
def _nan_check(prob, depth, conf, var, bad):
    """bad: bool [B,H,W] of pixels that saw a NaN logit."""
    for name, t in (("depth", depth), ("conf", conf), ("variance", var)):
        t = t.cpu()
        assert torch.isnan(t[bad]).all(), name
        assert torch.isfinite(t[~bad]).all(), name
    pc = prob.cpu()
    assert torch.isnan(pc.permute(0, 2, 3, 1)[bad]).all()
    assert torch.isfinite(pc.permute(0, 2, 3, 1)[~bad]).all()


@pytest.mark.gpu
@pytest.mark.parametrize("D,per_pixel,hw", [
    (8, True, (5, 13)), (16, True, (5, 13)), (32, True, (5, 13)), (48, True, (5, 13)), (64, True, (5, 13)), (96, True, (5, 13)),
    (12, True, (4, 16)), (16, False, (4, 16)), (64, False, (4, 16)),
    (12, True, (5, 13)), (16, False, (5, 13)), (100, True, (4, 16)),
])
def test_head_nan_logit_propagates(dm, D, per_pixel, hw):
    """A NaN logit gives NaN prob / depth / conf / variance at its pixel, all other pixels finite: head_reg_kernel
    (per-pixel, D in {8,16,32,48,64,96}), head_staged_kernel (D <= 64, H*W % 4 == 0) and head_stream_kernel."""
    from damvsnet_b200 import ops
    g = torch.Generator().manual_seed(D)
    B, (H, W) = 2, hw
    logits = torch.randn(B, D, H, W, generator=g)
    logits[0, D // 3, 1, 2] = float("nan")
    logits[1, D - 1, H - 1, W - 1] = float("nan")
    bad = torch.zeros(B, H, W, dtype=torch.bool)
    bad[0, 1, 2] = bad[1, H - 1, W - 1] = True
    dv = make_hyp(B, D, H, W, per_pixel, g).to(dev())
    _nan_check(*ops.softmax_regress(logits.to(dev()), dv), bad)


@pytest.mark.gpu
@pytest.mark.parametrize("prec", ["fp16", "bf16"])
def test_prob_head_nan_propagates(dm, prec):
    """The fused prob conv + head: a NaN voxel of the input volume makes NaN logits at the 3 x 3 pixels around it,
    which must come out NaN; every other pixel stays finite."""
    from damvsnet_b200 import ops
    from damvsnet_b200.ops import CONV_TCGEN05
    hd = torch.float16 if prec == "fp16" else torch.bfloat16
    g = torch.Generator().manual_seed(5)
    B, D, H, W = 1, 8, 12, 40
    x = torch.randn(B, 8, D, H, W, generator=g)
    x[0, 3, 4, 6, 20] = float("nan")
    bad = torch.zeros(B, H, W, dtype=torch.bool)
    bad[0, 5:8, 19:22] = True
    net = dm.CostRegNet(8, 8).to(dev())
    vol = dm.G8Volume(to_g8(x).to(hd).to(dev()))
    if not ops.prob_head_supported(vol, CONV_TCGEN05):
        pytest.fail("prob_head does not support the test shape")
    dv = make_hyp(B, D, H, W, True, g).to(dev())
    _nan_check(*ops.prob_head(vol, net._prob_prepared(CONV_TCGEN05, hd), dv, CONV_TCGEN05), bad)
