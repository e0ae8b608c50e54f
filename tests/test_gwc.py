"""Group-wise correlation cost volume (NOT in the reference: BASELINE.json north star / configs[4]).

CPU: the own-restatement oracle (oracle/gwc_oracle.py) against a direct formulation built on F.grid_sample, and on the
stored outputs of the reference's own ``homo_warping``.  GPU (-m gpu): csrc/warp_gwc.cu against that
oracle for every supported (C, G), both feature widths, ragged extents, [B,D] and [B,D,H,W] hypotheses, and through
CostRegNet + head as a DepthNet mode.
"""
import pytest
import torch
import torch.nn.functional as F

from oracle import damvs_oracle as O
from oracle import gwc_oracle

CASES = [(8, 4), (8, 8), (16, 4), (16, 8), (16, 16), (32, 4), (32, 8), (32, 16), (32, 32)]


def _inputs(stage, batch, nviews, H, W, D, seed, channels):
    from damvsnet_b200 import synthetic
    return synthetic.make_stage_inputs(stage, batch, nviews, H, W, D, seed=seed, channels=channels)


def test_gwc_oracle_matches_a_direct_grid_sample_formulation():
    feats, pm, dv = _inputs(1, 2, 4, 32, 48, 6, 3, 16)
    got = gwc_oracle.groupwise_correlation(feats, pm, dv, 8)
    b, c, h, w = feats[0].shape
    d = dv.shape[1]
    projs = [O.compose_projection(p) for p in torch.unbind(pm, 1)]
    want = torch.zeros(b, 8, d, h, w)
    for src, sp in zip(feats[1:], projs[1:]):
        rot, trans = O.relative_projection(sp, projs[0])
        ix, iy = O.warp_coordinates(rot, trans, dv, h, w)                       # un-normalised sample coordinates [B,D,HW]
        grid = torch.stack(((2 * ix + 1) / w - 1, (2 * iy + 1) / h - 1), dim=-1).view(b, d * h, w, 2)
        warped = F.grid_sample(src, grid, mode="bilinear", padding_mode="zeros", align_corners=False).view(b, c, d, h, w)
        want += (feats[0].unsqueeze(2) * warped).view(b, 8, 2, d, h, w).mean(2)
    want /= 3
    torch.testing.assert_close(got, want, rtol=1e-4, atol=1e-5)
    assert got.shape == (2, 8, 6, 16, 24)          # stage 2 of a 32x48 image


def test_gwc_oracle_uses_the_references_warp():
    """Against the reference's own homo_warping outputs stored in tests/golden/homo_warping.npz (one source view, [B,D,H,W]
    and [B,D] hypotheses).  The stored projections are already composed, so they enter as extrinsics with identity
    intrinsics."""
    from tests import golden_io
    g = golden_io.load_homo()
    src = g["src"]
    b, c, h, w = src.shape
    eye = torch.eye(4).expand(b, 4, 4)
    pm = torch.stack([torch.stack([g["ref_proj"], eye], 1), torch.stack([g["src_proj"], eye], 1)], 1)     # [B,2,2,4,4]
    ref = torch.randn(b, c, h, w, generator=torch.Generator().manual_seed(4))
    for dv, warped in ((g["dv4"], g["out4"]), (g["dv2"], g["out2"])):
        got = gwc_oracle.groupwise_correlation([ref, src], pm, dv, 4)
        want = (ref.unsqueeze(2) * warped).view(b, 4, c // 4, dv.shape[1], h, w).mean(2)
        torch.testing.assert_close(got, want, rtol=1e-4, atol=1e-5)


# ------------------------------------------------------------------------------------------------ GPU
@pytest.mark.gpu
@pytest.mark.parametrize("c,g", CASES)
@pytest.mark.parametrize("half", [False, True])
def test_gwc_kernel_matches_oracle(c, g, half):
    import damvsnet_b200 as dm
    from damvsnet_b200 import ops
    dev = torch.device("cuda:0")
    stage = {32: 0, 16: 1, 8: 2}[c]
    scale = (4, 2, 1)[stage]
    H, W = 37 * scale, 45 * scale                               # ragged: partial warps and CTAs in both directions
    feats, pm, dv = _inputs(stage, 2, 4, H, W, 5, 7 + g, c)
    if half:
        feats = [f.half().float() for f in feats]               # same fp16-representable values on both sides
    want = gwc_oracle.groupwise_correlation(feats, pm, dv, g)
    net = dm.DepthNet("groupwise", [32, 16, 8], groups=[g, g, g]).to(dev)
    for out_dtype in ((torch.float16, torch.bfloat16) if half else (torch.float32,)):
        with dm.precision("fp16" if half else "fp32"), torch.no_grad():
            vol = net.cost_volume(stage, [f.to(dev) for f in feats], pm.to(dev), dv.to(dev), out_dtype=out_dtype)
        got = vol.to_ncdhw().cpu()
        assert got.shape == (2, max(g, 8), 5, H // scale, W // scale)
        tol = {torch.float32: 2e-4, torch.float16: 2e-3, torch.bfloat16: 1.2e-2}[out_dtype]
        s = max(want.abs().mean().item(), 1e-3)
        err = (got[:, :g] - want).abs()
        assert (err <= tol * (want.abs() + s)).all(), (out_dtype, err.max().item(), s)
        if g < 8:
            assert (got[:, g:] == 0).all()                      # zero padding channels
    # [B,D] hypotheses take the broadcast path
    dv2 = dv[:, :, 0, 0].contiguous()
    want2 = gwc_oracle.groupwise_correlation(feats, pm, dv2.view(2, 5, 1, 1).expand_as(dv).contiguous(), g)
    nhwc = [ops.features_to_nhwc(f.to(dev)) for f in feats]
    rt = net.stage_rot_trans(pm.to(dev))
    got2 = ops.warp_groupwise(nhwc[0], nhwc[1:], rt, dv2.to(dev), g, torch.float32).to_ncdhw().cpu()
    s2 = max(want2.abs().mean().item(), 1e-3)
    assert ((got2[:, :g] - want2).abs() <= 2e-4 * (want2.abs() + s2)).all()


@pytest.mark.gpu
def test_gwc_depthnet_end_to_end_and_validation():
    """DepthNet(mode="groupwise") -> CostRegNet(in_channels=max(G,8)) -> head against the oracle chain (fp32), and the
    argument checks of the wrapper."""
    import damvsnet_b200 as dm
    from damvsnet_b200 import ops, synthetic
    dev = torch.device("cuda:0")
    g = 8
    sd = synthetic.hot_path_state_dict(in_channels=(8, 8, 8), seed=5, mode="variance")
    feats, pm, dv = _inputs(0, 1, 3, 64, 96, 8, 2, 32)
    net = dm.DepthNet("groupwise", [32, 16, 8], groups=[g]).to(dev).eval()
    cr = dm.CostRegNet(8, 8).eval()
    pre = "cost_regularization.0."
    cr.load_state_dict({k[len(pre):]: v for k, v in sd.items() if k.startswith(pre)}, strict=True)
    cr = cr.to(dev)
    with dm.precision("fp32"), torch.no_grad():
        out = net(0, [f.to(dev) for f in feats], pm.to(dev), dv.to(dev), 8, cr)
    vol = gwc_oracle.groupwise_correlation(feats, pm, dv, g)
    want = O.regress_head(O.cost_reg_net(vol, sd, 0).squeeze(1), dv)
    rel = ((out["depth"].cpu() - want["depth"]).abs() / want["depth"].abs())
    assert rel.max().item() < 1e-4, rel.max().item()
    assert (out["prob_volume"].cpu() - want["prob_volume"]).abs().max() < 2e-3
    with pytest.raises(ValueError):
        dm.DepthNet("groupwise", [32, 16, 8])
    nhwc = [ops.features_to_nhwc(f.to(dev)) for f in feats]
    with pytest.raises(ValueError):
        ops.warp_groupwise(nhwc[0], nhwc[1:], net.stage_rot_trans(pm.to(dev)), dv.to(dev), 3, torch.float32)
    with pytest.raises(NotImplementedError):
        net.cost_volume(0, [f.to(dev).requires_grad_(True) for f in feats], pm.to(dev), dv.to(dev))
