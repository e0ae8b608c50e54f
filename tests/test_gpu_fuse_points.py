"""Point emission of the geometric-consistency filter on the device (damvs_geo_consistency_points, fusion.fuse_views).

The kernel filters a reference view and writes the points of its final mask, compacted in row-major pixel order, at the
end of a scan-wide buffer.  It is checked against the per-view composition it replaces: filter_reference_view, then
backproject_valid on the averaged depth and final mask, then the reference image's colours at the mask.  Both paths use
one device function for the masks, so counts, order and colours must agree exactly.  The world coordinates are the
same float64 expression summed in a possibly different order, so after the cast to float32 they agree within 1 ulp,
except where the terms cancel: a coordinate that is 0 in exact arithmetic (the principal point's row or column of a
camera at the origin) comes out as float64 rounding noise of terms as large as the scene, a few 1e-16 of its size."""
import ctypes
import functools
import os
import sys

import numpy as np
import pytest
import torch

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


@pytest.fixture(scope="module")
def lib():
    from damvsnet_b200 import _lib, build
    build.build()
    return _lib.load()


# ---- argument checks (no GPU) ---------------------------------------------------------------------------------------

def _call(lib, n_src=4, H=8, W=8, capacity=16, null=None):
    """The entry point with pointers that must never be dereferenced: every call here fails its host-side checks."""
    fake = {k: ctypes.c_void_p(4096) for k in ("depth", "c1", "c2", "c3", "image", "xyz", "rgb", "total", "ws")}
    if null:
        fake[null] = None
    cams = np.zeros(18 + 42 * 11)
    world = np.zeros(12)
    srcs = (ctypes.c_void_p * 11)(*([4096] * 11))
    dbl = ctypes.POINTER(ctypes.c_double)
    return lib.damvs_geo_consistency_points(fake["depth"], fake["c1"], fake["c2"], fake["c3"], srcs, cams.ctypes.data_as(dbl),
                                            world.ctypes.data_as(dbl), n_src, H, W, 0.1, 0.15, 0.9, 0.25, 1 / 1300, fake["image"],
                                            capacity, fake["xyz"], fake["rgb"], fake["total"], fake["ws"], None)


@pytest.mark.parametrize("case,kw,msg", [
    ("null depth", dict(null="depth"), b"null pointer"),
    ("null xyz", dict(null="xyz"), b"null pointer"),
    ("null total", dict(null="total"), b"null pointer"),
    ("null workspace", dict(null="ws"), b"null pointer"),
    ("no source view", dict(n_src=0), b"n_src=0 outside [1,10]"),
    ("eleven source views", dict(n_src=11), b"n_src=11 outside [1,10]"),
    ("negative capacity", dict(capacity=-1), b"capacity=-1 is negative"),
    ("empty image", dict(H=0), b"bad shape"),
])
def test_points_argument_validation_needs_no_gpu(lib, case, kw, msg):
    assert _call(lib, **kw) == 1, case
    assert msg in lib.damvs_last_error(), (case, lib.damvs_last_error())


def test_points_workspace_grows_with_image(lib):
    ws = lib.damvs_geo_consistency_points_workspace_bytes
    assert ws(0, 16) == 0 and ws(16, 0) == 0
    assert 0 < ws(1, 1) <= ws(8, 128) < ws(8, 129) <= ws(8, 256) < ws(8, 257) < ws(16, 257) < ws(1152, 1600)
    assert all(ws(h, w) % 8 == 0 for h, w in ((1, 1), (8, 129), (1152, 1600)))


# ---- GPU ------------------------------------------------------------------------------------------------------------

def dev():
    return torch.device("cuda:0")


def to_dev(a):
    return torch.from_numpy(np.ascontiguousarray(a)).to(dev())


def make_scene(seed, H, W, n_src):
    sys.path.insert(0, GOLDEN)
    from make_golden_filter import make_scene as _make
    return _make(seed, H, W, n_src)


@functools.lru_cache(maxsize=None)
def scan(name):
    """(depths, confidences, images, Ks, Es, pairs) on the device for the named case (read, never written)."""
    from tests.golden_io import load_fusion_filter
    rs = np.random.RandomState(11)
    if name in ("a", "b", "scan3"):
        fx = load_fusion_filter()
        fx = {k: fx[("a" if name == "scan3" else name) + "/" + k] for k in ("K", "E", "depths", "confs")}
        K, E, d = list(fx["K"]), list(fx["E"]), list(fx["depths"])
        confs = [to_dev(c) for c in fx["confs"]]
        if name == "scan3":
            K, E, d = K[:3], E[:3], d[:3]
            pairs = [(0, [1, 2]), (1, [0, 2]), (2, [1, 0])]       # those of test_gpu_filter's three-view scan
        else:
            pairs = [(0, list(range(1, len(d))))]
    else:
        H, W, n = {"full": (1152, 1600, 4), "five": (48, 200, 4)}[name]
        K, E, d = make_scene(3, H, W, n)
        crs = np.random.RandomState(0)
        confs = [to_dev(crs.rand(H, W).astype(np.float32)) for _ in range(3)]
        pairs = [(0, [1, 2, 3, 4])] if name == "full" else [(v, [s for s in range(5) if s != v]) for v in range(5)]
    images = [to_dev(rs.rand(*x.shape, 3).astype(np.float32)) for x in d]
    return [to_dev(x) for x in d], [confs] * len(d), images, K, E, pairs


def old_composition(depths, confidences, images, Ks, Es, pairs, **kw):
    """Per view: filter_reference_view -> backproject_valid -> (image[mask] * 255).to(uint8)."""
    from damvsnet_b200 import fusion
    xyz, rgb = [], []
    for ref, srcs in pairs:
        out = fusion.filter_reference_view(depths[ref], confidences[ref], Ks[ref], Es[ref], [depths[s] for s in srcs],
                                           [Ks[s] for s in srcs], [Es[s] for s in srcs], **kw)
        m = out["final_mask"]
        xyz.append(fusion.backproject_valid(out["depth_est_averaged"], m, Ks[ref], Es[ref]).cpu().numpy())
        rgb.append((images[ref][m] * 255).to(torch.uint8).cpu().numpy())
    return xyz, rgb


def assert_points_equal(xyz, rgb, want_xyz, want_rgb):
    """Same count, same order, identical colours, coordinates within 1 float32 ulp or, near 0, 1e-12 of the scene's
    extent (thousands of float64 ulps of the cancelling terms, far below a float32 ulp of any coordinate above 1e-4)."""
    xyz = xyz.cpu().numpy() if isinstance(xyz, torch.Tensor) else xyz
    rgb = rgb.cpu().numpy() if isinstance(rgb, torch.Tensor) else rgb
    assert xyz.shape == want_xyz.shape and rgb.shape == want_rgb.shape
    np.testing.assert_array_equal(rgb, want_rgb)
    tol = np.spacing(np.maximum(np.abs(xyz), np.abs(want_xyz))) + 1e-12 * (np.abs(want_xyz).max() if want_xyz.size else 0.0)
    bad = np.abs(xyz.astype(np.float64) - want_xyz) > tol
    assert not bad.any(), f"{bad.sum()} coordinates differ by more than 1 ulp, first at {np.argwhere(bad)[0]}"


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["a", "b", "scan3", "full"])
def test_points_match_old_composition(name):
    from damvsnet_b200 import fusion
    args = scan(name)
    want_xyz, want_rgb = old_composition(*args)
    xyz, rgb = fusion.fuse_views(*args)
    assert xyz.dtype == torch.float32 and rgb.dtype == torch.uint8 and xyz.device == dev()
    counts = [len(x) for x in want_xyz]
    assert len(xyz) == sum(counts) and min(counts) > 0
    start = 0
    for n, wx, wr in zip(counts, want_xyz, want_rgb):
        assert_points_equal(xyz[start:start + n], rgb[start:start + n], wx, wr)
        start += n


@pytest.mark.gpu
@pytest.mark.parametrize("W", [130, 257])
def test_points_row_major_with_partial_tiles(W):
    """Row tails shorter than a tile: a real scene, a view checked against copies of itself with every photometric
    threshold below 0 (every pixel is a point: the full row-major grid), and thresholds above 1 (no point)."""
    from damvsnet_b200 import fusion
    H = 24
    K, E, d = make_scene(7, H, W, 3)
    rs = np.random.RandomState(W)
    confs = [to_dev(rs.rand(H, W).astype(np.float32)) for _ in range(3)]
    images = [to_dev(rs.rand(H, W, 3).astype(np.float32)) for _ in d]
    depths = [to_dev(x) for x in d]
    pairs = [(0, [1, 2, 3])]
    args = (depths, [confs] * 4, images, K, E, pairs)
    got, want = fusion.fuse_views(*args), old_composition(*args)
    assert 0 < len(want[0][0]) < H * W
    assert_points_equal(*got, want[0][0], want[1][0])

    same = ([depths[0]] * 3, [confs] * 3, [images[0]] * 3, [K[0]] * 3, [E[0]] * 3, [(0, [1, 2])])
    kw = dict(conf_thr=(-1.0, -1.0, -1.0))
    xyz, rgb = fusion.fuse_views(*same, **kw)
    want_xyz, _ = old_composition(*same, **kw)
    assert len(xyz) == H * W
    assert_points_equal(xyz, rgb, want_xyz[0], (images[0].reshape(-1, 3) * 255).to(torch.uint8).cpu().numpy())

    xyz, rgb = fusion.fuse_views(*args, conf_thr=(1.5, 1.5, 1.5))
    assert tuple(xyz.shape) == (0, 3) and tuple(rgb.shape) == (0, 3)
    sentinel = run_direct(depths, confs, images[0], K, E, pairs[0], capacity=H * W, conf_thr=(1.5, 1.5, 1.5))
    assert sentinel["total"] == 0 and sentinel["untouched_xyz"] == H * W + 128 and sentinel["untouched_rgb"] == H * W + 128


SENTINEL_XYZ, SENTINEL_RGB = -12345.0, 77


def run_direct(depths, confs, image, Ks, Es, pair, capacity, conf_thr=(0.1, 0.15, 0.9)):
    """One call of the entry point through ctypes into sentinel-filled buffers one tile (128 points) longer than
    `capacity`.  Returns the buffers, the total and how many rows still hold the sentinel."""
    from damvsnet_b200 import _lib, fusion
    lib = _lib.load()
    ref, srcs = pair
    h, w = depths[ref].shape
    xyz = torch.full((capacity + 128, 3), SENTINEL_XYZ, device=dev())
    rgb = torch.full((capacity + 128, 3), SENTINEL_RGB, dtype=torch.uint8, device=dev())
    total = torch.zeros((), dtype=torch.int64, device=dev())
    ws = torch.zeros(lib.damvs_geo_consistency_points_workspace_bytes(h, w), dtype=torch.uint8, device=dev())
    cams = fusion.pack_cameras(Ks[ref], Es[ref], [Ks[s] for s in srcs], [Es[s] for s in srcs])
    world = np.ascontiguousarray(np.linalg.inv(np.asarray(Es[ref], np.float64))[:3])
    ptrs = (ctypes.c_void_p * len(srcs))(*[depths[s].data_ptr() for s in srcs])
    dbl = ctypes.POINTER(ctypes.c_double)
    p = lambda t: ctypes.c_void_p(t.data_ptr())
    _lib.check(lib.damvs_geo_consistency_points(
        p(depths[ref]), p(confs[0]), p(confs[1]), p(confs[2]), ptrs, cams.ctypes.data_as(dbl), world.ctypes.data_as(dbl),
        len(srcs), h, w, *[float(c) for c in conf_thr], 0.25, 1 / 1300, p(image), capacity, p(xyz), p(rgb), p(total), p(ws),
        ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)))
    torch.cuda.synchronize()
    return {"xyz": xyz.cpu().numpy(), "rgb": rgb.cpu().numpy(), "total": int(total.item()),
            "untouched_xyz": int((xyz == SENTINEL_XYZ).all(1).sum()), "untouched_rgb": int((rgb == SENTINEL_RGB).all(1).sum())}


@pytest.mark.gpu
def test_points_past_capacity_are_counted_not_written():
    depths, confidences, images, K, E, pairs = scan("a")
    want_xyz, want_rgb = old_composition(depths, confidences, images, K, E, pairs)
    n = len(want_xyz[0])
    cap = n // 2 + 3                                                 # not a multiple of any tile's count
    out = run_direct(depths, confidences[0], images[0], K, E, pairs[0], capacity=cap)
    assert out["total"] == n
    assert_points_equal(out["xyz"][:cap], out["rgb"][:cap], want_xyz[0][:cap], want_rgb[0][:cap])
    assert (out["xyz"][cap:] == SENTINEL_XYZ).all() and (out["rgb"][cap:] == SENTINEL_RGB).all()


@pytest.mark.gpu
def test_views_append_in_pairs_order():
    from damvsnet_b200 import fusion
    depths, confidences, images, K, E, pairs = scan("five")
    want_xyz, want_rgb = old_composition(depths, confidences, images, K, E, pairs)
    counts = [len(x) for x in want_xyz]
    assert len(set(counts)) > 1                                      # the blocks are told apart by their sizes too
    xyz, rgb = fusion.fuse_views(depths, confidences, images, K, E, pairs)
    offsets = np.concatenate([[0], np.cumsum(counts)])
    for k in range(5):
        assert_points_equal(xyz[offsets[k]:offsets[k + 1]], rgb[offsets[k]:offsets[k + 1]], want_xyz[k], want_rgb[k])
    rxyz, rrgb = fusion.fuse_views(depths, confidences, images, K, E, pairs[::-1])
    start = 0
    for k in reversed(range(5)):
        n = counts[k]
        assert torch.equal(rxyz[start:start + n], xyz[offsets[k]:offsets[k + 1]])
        assert torch.equal(rrgb[start:start + n], rgb[offsets[k]:offsets[k + 1]])
        start += n


@pytest.mark.gpu
def test_one_launch_and_no_sync_per_view():
    from damvsnet_b200 import _lib, fusion
    args = scan("five")
    fusion.fuse_views(*args)                                         # warm-up: allocator, module load
    n0 = _lib.launch_count()
    fusion.fuse_views(*args)
    assert _lib.launch_count() - n0 == len(args[-1])
    torch.cuda.synchronize()
    mode = torch.cuda.get_sync_debug_mode()
    torch.cuda.set_sync_debug_mode("error")
    try:
        total, xyz, rgb = fusion._enqueue_points(*args, (0.1, 0.15, 0.9), 1 / 4, 1 / 1300)
    finally:
        torch.cuda.set_sync_debug_mode(mode)
    assert int(total.item()) == sum(len(x) for x in old_composition(*args)[0])


@pytest.mark.gpu
def test_points_are_deterministic():
    from damvsnet_b200 import fusion
    args = scan("full")
    a, b = fusion.fuse_views(*args), fusion.fuse_views(*args)
    assert torch.equal(a[0].view(torch.int32), b[0].view(torch.int32)) and torch.equal(a[1], b[1])
