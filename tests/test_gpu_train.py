"""GPU parity tests of the training path (native forward + backward kernels through the C ABI).

Checked against (1) gradients produced by the reference itself (tests/golden/train_grads.npz) and (2) the CPU
oracle differentiated by torch autograd on fresh seeded inputs.  fp32 mode: relative L2 error of every gradient
<= 5e-3 with fixed BatchNorm statistics, <= 1e-2 with batch statistics (eleven chained batch-stat BatchNorms on a
16x24 volume amplify fp32 summation-order noise: the reference on CPU and the oracle on CPU already differ by 2e-3);
bf16 mode (tensor-core convolutions, bf16 volumes and volume gradients): relative L2 error <= twice the value
measured on the B200 for each gradient (BF16_MEASURED).  w_net.1.conv.weight feeds a BatchNorm directly, so its true gradient is zero up to eps
effects (|g| ~ 1e-4): only its magnitude is checked.
"""
import pytest
import torch

pytestmark = pytest.mark.gpu

from oracle import damvs_oracle as O  # noqa: E402
from tests.golden_io import load_train_grads  # noqa: E402


def dev():
    return torch.device("cuda:0")


@pytest.fixture(scope="module")
def dm():
    import damvsnet_b200 as dm
    from damvsnet_b200 import _lib
    _lib.check(_lib.load().damvs_check_device(0))
    return dm


def rel(a, b, drop: int = 0):
    """Relative L2 error; `drop` ignores that many worst elements (a ReLU whose pre-activation is within 1e-5 of
    zero flips between implementations and moves one summand of a per-channel gradient)."""
    d = (a - b).flatten()
    if drop and d.numel() > drop:
        keep = torch.ones_like(d, dtype=torch.bool)
        keep[d.abs().topk(drop).indices] = False
        return (d[keep].norm() / b.flatten()[keep].norm().clamp_min(1e-12)).item()
    return (d.norm() / b.norm().clamp_min(1e-12)).item()


def build(dm, sd, mode, cin, train):
    net = dm.DepthNet(mode, [cin])
    cr = dm.CostRegNet(cin, 8)
    if mode == "adaptive":
        net.load_state_dict({k[len("DepthNet."):]: v for k, v in sd.items() if k.startswith("DepthNet.")}, strict=True)
    pre = "cost_regularization.0."
    cr.load_state_dict({k[len(pre):]: v for k, v in sd.items() if k.startswith(pre)}, strict=True)
    net.train(train)
    cr.train(train)
    return net.to(dev()), cr.to(dev())


def native_step(dm, net, cr, feats, proj, dv, r_depth, r_prob, r_var):
    fs = [f.to(dev()).requires_grad_(True) for f in feats]
    out = net(0, fs, proj.to(dev()), dv.to(dev()), dv.shape[1], cr)
    loss = (out["depth"] * r_depth.to(dev())).sum() + (out["prob_volume"] * r_prob.to(dev())).sum() + \
        (out["variance"] * r_var.to(dev())).sum()
    loss.backward()
    grads = {}
    for prefix, mod in (("DepthNet.", net), ("cost_regularization.0.", cr)):
        for k, p in mod.named_parameters():
            if p.grad is not None:
                grads[prefix + k] = p.grad.detach().cpu()
    return out, loss.item(), [f.grad.detach().cpu() for f in fs], grads


@pytest.mark.parametrize("mode", ["adaptive", "variance"])
@pytest.mark.parametrize("bn_mode", ["train", "eval"])
def test_fp32_gradients_match_reference_fixture(dm, mode, bn_mode):
    fx = load_train_grads(mode, bn_mode)
    with dm.precision("fp32"):
        net, cr = build(dm, fx["sd"], mode, 8, bn_mode == "train")
        out, loss, g_feats, grads = native_step(dm, net, cr, fx["features"], fx["proj"], fx["depth_values"],
                                                fx["r_depth"], fx["r_prob"], fx["r_var"])
    assert abs(loss - fx["loss"]) <= 5e-4 * abs(fx["loss"])
    for k in ("depth", "variance", "prob_volume"):
        assert rel(out[k].detach().cpu(), fx["out"][k]) < 2e-4, k
    tol = 1e-2 if bn_mode == "train" else 5e-3
    for got, want in zip(g_feats, fx["g_features"]):
        assert rel(got, want) < tol
    assert set(grads) == set(fx["grads"]), set(grads) ^ set(fx["grads"])
    for k, want in fx["grads"].items():
        if bn_mode == "train" and k.endswith("w_net.1.conv.weight"):
            assert float(grads[k].abs().max()) < 1e-3
            continue
        assert rel(grads[k], want, drop=1) < tol or float((grads[k] - want).abs().max()) < 2e-5, (k, rel(grads[k], want))
    if bn_mode == "train":     # running buffers after one training step (momentum 0.1, unbiased variance)
        bufs = {}
        for prefix, mod in (("DepthNet.", net), ("cost_regularization.0.", cr)):
            for k, b in mod.named_buffers():
                bufs[prefix + k] = b.detach().cpu()
        for k, want in fx["buffers"].items():
            if "conv0" in k and k.startswith("DepthNet."):
                continue           # dead block of the weight net: never run
            if want.dtype.is_floating_point:
                torch.testing.assert_close(bufs[k], want, rtol=2e-4, atol=2e-5, msg=k)
            else:
                assert int(bufs[k]) == int(want), k


# Relative L2 error of the bf16 training step's gradients against the fp32 reference fixture, measured on an NVIDIA B200
# (1000 W power limit): feature gradients (max over the three views) and every parameter gradient of >= 64 elements.
# The bounds are twice these values.  The error is the bf16 cost volume / activations / weights of the whole network
# (eleven layers, peaked softmax), not one kernel: the per-op bounds are in tests/test_gpu_train_ops.py.
BF16_MEASURED = {
    "adaptive": {"features": 0.2635, "conv0": 0.2930, "conv1": 0.2599, "conv2": 0.2510, "conv3": 0.2656, "conv4": 0.2438,
                 "conv5": 0.2796, "conv5.bn": 0.2618, "conv6": 0.1878, "conv6.bn": 0.1683, "conv7": 0.1743, "conv9": 0.1282,
                 "conv11": 0.0840, "prob": 0.0169},
    "variance": {"features": 0.2149, "conv0": 0.2119, "conv1": 0.1956, "conv2": 0.1803, "conv3": 0.1990, "conv4": 0.1723,
                 "conv5": 0.1965, "conv5.bn": 0.2188, "conv6": 0.1881, "conv6.bn": 0.1989, "conv7": 0.1679, "conv9": 0.1050,
                 "conv11": 0.0780, "prob": 0.0166},
}


def _bf16_key(k):
    name = k[len("cost_regularization.0."):]
    layer = name.split(".")[0]
    return layer + ".bn" if ".bn." in name else layer


@pytest.mark.parametrize("mode", ["adaptive", "variance"])
def test_bf16_gradients_close_to_reference_fixture(dm, mode):
    """Relative L2 of every feature gradient and every parameter gradient of >= 64 elements <= 2x the value measured on
    the B200 (BF16_MEASURED)."""
    fx = load_train_grads(mode, "train")
    with dm.precision("bf16"):
        net, cr = build(dm, fx["sd"], mode, 8, True)
        out, loss, g_feats, grads = native_step(dm, net, cr, fx["features"], fx["proj"], fx["depth_values"],
                                                fx["r_depth"], fx["r_prob"], fx["r_var"])
    assert abs(loss - fx["loss"]) <= 3e-2 * abs(fx["loss"])
    measured = BF16_MEASURED[mode]
    for got, want in zip(g_feats, fx["g_features"]):
        assert rel(got, want) <= 2 * measured["features"], rel(got, want)
    big = [k for k, w in fx["grads"].items() if w.numel() >= 64]
    assert big
    for k in big:
        assert rel(grads[k], fx["grads"][k]) <= 2 * measured[_bf16_key(k)], (k, rel(grads[k], fx["grads"][k]))


@pytest.mark.parametrize("cin,stage", [(16, 1), (32, 0)])
def test_fp32_gradients_match_oracle_autograd(dm, cin, stage):
    """Fresh seeded inputs at the other channel widths (lanes-per-pixel 2 and 4), B=1, N=4, D=16."""
    from damvsnet_b200 import synthetic
    B, N, D, H, W = 1, 4, 16, 24 * synthetic.STAGE_SCALES[stage], 32 * synthetic.STAGE_SCALES[stage]
    feats, proj, dv = synthetic.make_stage_inputs(stage, B, N, H, W, D, seed=9)
    h, w = dv.shape[2:]
    sd_all = synthetic.hot_path_state_dict(seed=2)
    sd = {}
    for k, v in sd_all.items():
        for src, dst in ((f"cost_regularization.{stage}.", "cost_regularization.0."), (f"DepthNet.weight_net.{stage}.", "DepthNet.weight_net.0.")):
            if k.startswith(src):
                sd[dst + k[len(src):]] = v
    g = torch.Generator().manual_seed(5)
    r_depth, r_prob, r_var = torch.randn(B, h, w, generator=g) * 0.1, torch.randn(B, D, h, w, generator=g), torch.rand(B, h, w, generator=g) * 0.05
    # oracle
    fo = [f.clone().requires_grad_(True) for f in feats]
    so = {k: (v.clone().requires_grad_(True) if v.dtype.is_floating_point and "running" not in k else v.clone()) for k, v in sd.items()}
    oo = O.depthnet_forward(0, fo, proj, dv, so, "adaptive", training=True)
    lo = (oo["depth"] * r_depth).sum() + (oo["prob_volume"] * r_prob).sum() + (oo["variance"] * r_var).sum()
    lo.backward()
    with dm.precision("fp32"):
        net, cr = build(dm, sd, "adaptive", cin, True)
        out, loss, g_feats, grads = native_step(dm, net, cr, feats, proj, dv, r_depth, r_prob, r_var)
    assert abs(loss - lo.item()) <= 5e-4 * abs(lo.item())
    for got, f in zip(g_feats, fo):
        assert rel(got, f.grad) < 1e-2
    for k, got in grads.items():
        want = so[k].grad
        assert want is not None, k
        if k.endswith("w_net.1.conv.weight"):
            assert float(got.abs().max()) < 5e-2        # mathematically zero; fp32 cancellation over 0.6 M voxels
            continue
        assert rel(got, want, drop=1) < 1e-2 or float((got - want).abs().max()) < 2e-5, (k, rel(got, want))


def test_head_backward_matches_autograd(dm):
    from damvsnet_b200 import autograd as ag
    g = torch.Generator().manual_seed(1)
    B, D, H, W = 2, 12, 9, 14
    logits = torch.randn(B, D, H, W, generator=g)
    hyp = (425 + 2.65 * torch.arange(D, dtype=torch.float32).view(1, D, 1, 1) + torch.rand(B, 1, H, W, generator=g)).expand(B, D, H, W).contiguous()
    r1, r2, r3 = torch.randn(B, H, W, generator=g), torch.randn(B, D, H, W, generator=g), torch.randn(B, H, W, generator=g)
    lc, hc = logits.clone().requires_grad_(True), hyp.clone().requires_grad_(True)
    o = O.regress_head(lc, hc)
    ((o["depth"] * r1).sum() + (o["prob_volume"] * r2).sum() + (o["variance"] * r3).sum()).backward()
    lg, hg = logits.to(dev()).requires_grad_(True), hyp.to(dev()).requires_grad_(True)
    prob, depth, conf, var = ag.HeadFn.apply(lg, hg)
    ((depth * r1.to(dev())).sum() + (prob * r2.to(dev())).sum() + (var * r3.to(dev())).sum()).backward()
    assert rel(lg.grad.cpu(), lc.grad) < 1e-4
    assert rel(hg.grad.cpu(), hc.grad) < 1e-4


def test_eval_no_grad_path_unchanged_by_training_code(dm):
    """The inference path (fused kernels) and the autograd path agree on the forward outputs."""
    fx = load_train_grads("adaptive", "eval")
    with dm.precision("fp32"):
        net, cr = build(dm, fx["sd"], "adaptive", 8, False)
        fs = [f.to(dev()) for f in fx["features"]]
        with torch.no_grad():
            a = net(0, fs, fx["proj"].to(dev()), fx["depth_values"].to(dev()), 8, cr)
        b = net(0, [f.clone().requires_grad_(True) for f in fs], fx["proj"].to(dev()), fx["depth_values"].to(dev()), 8, cr)
    assert rel(b["depth"].detach().cpu(), a["depth"].cpu()) < 1e-5
    assert rel(b["prob_volume"].detach().cpu(), a["prob_volume"].cpu()) < 1e-4


@pytest.mark.parametrize("cin,cout,stride,transposed", [
    (8, 8, 1, False), (16, 8, 1, False), (32, 8, 1, False), (64, 64, 1, False), (8, 1, 1, False),
    (8, 16, 2, False), (16, 32, 2, False), (32, 64, 2, False),
    (64, 32, 2, True), (32, 16, 2, True), (16, 8, 2, True)])
def test_weight_gradient_kernels_match_torch(dm, cin, cout, stride, transposed):
    """damvs_conv3d_wgrad (tensor-core kernel for bf16 volumes, CUDA-core kernel for fp32) against autograd of
    F.conv3d / F.conv_transpose3d on the same (bf16-rounded) operands; ragged extents, 2 batch items."""
    import torch.nn.functional as F
    from damvsnet_b200 import ops_train
    g = torch.Generator().manual_seed(cin * 100 + cout)
    B, D, H, W = 2, 6, 10, 38
    x = torch.randn(B, cin, D, H, W, generator=g).bfloat16().float()
    w = torch.randn((cin, cout, 3, 3, 3) if transposed else (cout, cin, 3, 3, 3), generator=g).requires_grad_(True)
    y = F.conv_transpose3d(x, w, None, stride=2, padding=1, output_padding=1) if transposed else F.conv3d(x, w, None, stride=stride, padding=1)
    gy = torch.randn(y.shape, generator=g).bfloat16().float()
    (y * gy).sum().backward()
    gy_p = gy
    if cout % 8:
        gy_p = torch.zeros(B, 8, *gy.shape[2:])
        gy_p[:, :cout] = gy
    for dtype, tol in ((torch.bfloat16, 2e-3), (torch.float32, 1e-4)):
        xv = dm.G8Volume.from_ncdhw(x.to(dev()), dtype).data
        gv = dm.G8Volume.from_ncdhw(gy_p.to(dev()), dtype).data
        dw = ops_train.conv3d_wgrad(xv, gv, cin, cout, stride, transposed).cpu()
        assert dw.shape == w.shape
        assert rel(dw, w.grad) < tol, (dtype, rel(dw, w.grad))


def test_trainer_step_with_full_reference_loss_decreases_loss(dm):
    """HotPathTrainer: three stages, depth + 12 x cross-view loss (models/module.py:700-717), Adam; a few steps on one
    fixed batch reduce the loss and keep every parameter finite."""
    from damvsnet_b200 import synthetic
    from damvsnet_b200.runner import make_workload
    from damvsnet_b200.training import HotPathTrainer
    B, N, H, W, nds = 2, 3, 64, 96, [16, 8, 8]
    with dm.precision("bf16"):
        tr = HotPathTrainer(synthetic.hot_path_state_dict(seed=4), device=dev(), lr=2e-3)
        stages = make_workload(H, W, N, nds, batch=B, seed=3, device=dev())
        stages = [([f.requires_grad_(True) for f in fs], p, d) for fs, p, d in stages]
        gts = [d[:, d.shape[1] // 2].contiguous() for _, _, d in stages]
        masks = [torch.ones_like(g) for g in gts]
        imgs = synthetic.make_images(B, N, H, W, seed=1).to(dev())
        cams = {f"stage{i + 1}": p for i, (_, p, _) in enumerate(stages)}
        losses = [float(tr.train_step(stages, gts, masks, imgs=imgs, sample_cams=cams)) for _ in range(6)]
    assert all(torch.isfinite(p).all() for p in tr.params)
    assert losses[-1] < losses[0], losses
