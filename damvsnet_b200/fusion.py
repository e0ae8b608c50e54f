"""Geometric-consistency filtering of a reference view (the downstream neighbour of the hot path, SURVEY.md 8f rank 2).

Host-side mirror of what reference ``filter/dypcd.py:filter_depth`` does per reference view (lines 205-257, calling
``check_geometric_consistency`` :135-159 and ``reproject_with_depth`` :98-132): the depth maps stay on the GPU, one
native kernel (``damvs_geo_consistency_fuse``) replaces the numpy + ``cv2.remap`` loop over source views, and the
PFM round trip through disk between ``test_uni.py:246-287`` and the filter goes away.  Camera products are formed in
float64 numpy exactly as the reference forms them.
"""
from __future__ import annotations

import ctypes
from typing import Dict, Sequence

import numpy as np
import torch

from . import _lib
from .ops import _p, _stream

MAX_SRC_VIEWS = 10


def pack_cameras(ref_K: np.ndarray, ref_E: np.ndarray, src_Ks: Sequence[np.ndarray], src_Es: Sequence[np.ndarray]) -> np.ndarray:
    """float64 vector in the layout damvs_geo_consistency_fuse expects (include/damvs.h)."""
    ref_K, ref_E = np.asarray(ref_K, np.float64), np.asarray(ref_E, np.float64)
    out = [ref_K.reshape(-1), np.linalg.inv(ref_K).reshape(-1)]
    for K, E in zip(src_Ks, src_Es):
        K, E = np.asarray(K, np.float64), np.asarray(E, np.float64)
        out += [np.matmul(E, np.linalg.inv(ref_E))[:3].reshape(-1), K.reshape(-1), np.linalg.inv(K).reshape(-1),
                np.matmul(ref_E, np.linalg.inv(E))[:3].reshape(-1)]
    return np.ascontiguousarray(np.concatenate(out))


def filter_reference_view(ref_depth: torch.Tensor, confidences: Sequence[torch.Tensor], ref_K, ref_E,
                          src_depths: Sequence[torch.Tensor], src_Ks, src_Es, conf_thr: Sequence[float] = (0.1, 0.15, 0.9),
                          dist_base: float = 1 / 4, rel_diff_base: float = 1 / 1300) -> Dict[str, torch.Tensor]:
    """ref_depth [H,W] and confidences (stage 1, 2, 3, each [H,W]) of the reference view, src_depths n x [H,W], all CUDA
    fp32; intrinsics 3x3 / extrinsics 4x4 as numpy.  Returns depth_est_averaged (fp32) and the photo / geo / final masks
    (bool) of filter/dypcd.py:254-262.  Defaults are the reference's (test_uni.py:104-109)."""
    n = len(src_depths)
    if not 1 <= n <= MAX_SRC_VIEWS:
        raise ValueError(f"1..{MAX_SRC_VIEWS} source views supported (the reference's mask list covers dy_range <= 11)")
    h, w = ref_depth.shape
    tensors = [ref_depth, *confidences, *src_depths]
    if len(confidences) != 3 or any(t.dtype != torch.float32 or not t.is_cuda or tuple(t.shape) != (h, w) for t in tensors):
        raise ValueError("expected CUDA fp32 [H,W] maps: depth, three confidences, n source depths")
    tensors = [t.contiguous() for t in tensors]
    cams = pack_cameras(ref_K, ref_E, src_Ks, src_Es)
    dev = ref_depth.device
    depth_avg = torch.empty((h, w), dtype=torch.float32, device=dev)
    photo, geo, final = (torch.empty((h, w), dtype=torch.uint8, device=dev) for _ in range(3))
    src_ptrs = (ctypes.c_void_p * n)(*[t.data_ptr() for t in tensors[4:]])
    with torch.cuda.device_of(ref_depth):
        _lib.check(_lib.load().damvs_geo_consistency_fuse(
            _p(tensors[0]), _p(tensors[1]), _p(tensors[2]), _p(tensors[3]), src_ptrs,
            cams.ctypes.data_as(ctypes.POINTER(ctypes.c_double)), n, h, w, float(conf_thr[0]), float(conf_thr[1]), float(conf_thr[2]),
            float(dist_base), float(rel_diff_base), _p(depth_avg), _p(photo), _p(geo), _p(final), _stream()))
    return {"depth_est_averaged": depth_avg, "photo_mask": photo.bool(), "geo_mask": geo.bool(), "final_mask": final.bool()}


def backproject_valid(depth: torch.Tensor, mask: torch.Tensor, K, E) -> torch.Tensor:
    """World-space points of the masked pixels, [n,3] (filter/dypcd.py:281-299): inv(E) [inv(K) [x,y,1] d; 1]."""
    ys, xs = torch.nonzero(mask, as_tuple=True)
    d = depth[ys, xs].double()
    pix = torch.stack([xs.double() * d, ys.double() * d, d], 0)
    Ki = torch.from_numpy(np.linalg.inv(np.asarray(K, np.float64))).to(depth.device)
    Ei = torch.from_numpy(np.linalg.inv(np.asarray(E, np.float64))).to(depth.device)
    cam = Ki @ pix
    world = Ei[:3, :3] @ cam + Ei[:3, 3:4]
    return world.t().float()


def _enqueue_points(depths, confidences, images, Ks, Es, pairs, conf_thr, dist_base, rel_diff_base):
    """Enqueue one damvs_geo_consistency_points launch per (ref, srcs) of `pairs`, all appending to one buffer, with
    no host synchronisation.  Returns (total, xyz, rgb): the device int64 point count and the [capacity,3] buffers,
    capacity being the number of reference pixels, so that no scan can overflow it."""
    if not pairs:
        raise ValueError("pairs is empty")
    dev = depths[pairs[0][0]].device
    if dev.type != "cuda":
        raise ValueError("expected CUDA tensors")
    views = []
    for ref, srcs in pairs:
        if not 1 <= len(srcs) <= MAX_SRC_VIEWS:
            raise ValueError(f"1..{MAX_SRC_VIEWS} source views supported (the reference's mask list covers dy_range <= 11)")
        maps = [depths[ref], *confidences[ref], *[depths[s] for s in srcs]]
        h, w = maps[0].shape
        if len(confidences[ref]) != 3 or any(t.dtype != torch.float32 or t.device != dev or tuple(t.shape) != (h, w) for t in maps):
            raise ValueError("expected CUDA fp32 [H,W] maps on one device: depth, three confidences, n source depths")
        img = images[ref]
        if img.dtype != torch.float32 or img.device != dev or tuple(img.shape) != (h, w, 3):
            raise ValueError("expected a CUDA fp32 [H,W,3] image per reference view, on the device of the depth maps")
        views.append((ref, srcs, [t.contiguous() for t in maps], img.contiguous()))
    lib = _lib.load()
    capacity = sum(maps[0].numel() for _, _, maps, _ in views)
    ws_bytes = [lib.damvs_geo_consistency_points_workspace_bytes(*maps[0].shape) for _, _, maps, _ in views]
    xyz = torch.empty((capacity, 3), dtype=torch.float32, device=dev)
    rgb = torch.empty((capacity, 3), dtype=torch.uint8, device=dev)
    total = torch.zeros((), dtype=torch.int64, device=dev)
    workspace = torch.zeros(sum(ws_bytes), dtype=torch.uint8, device=dev)   # one zeroed slice per launch
    offset = 0
    with torch.cuda.device_of(total):
        for (ref, srcs, maps, img), nbytes in zip(views, ws_bytes):
            cams = pack_cameras(Ks[ref], Es[ref], [Ks[s] for s in srcs], [Es[s] for s in srcs])
            world_from_cam = np.ascontiguousarray(np.linalg.inv(np.asarray(Es[ref], np.float64))[:3])
            src_ptrs = (ctypes.c_void_p * len(srcs))(*[t.data_ptr() for t in maps[4:]])
            _lib.check(lib.damvs_geo_consistency_points(
                _p(maps[0]), _p(maps[1]), _p(maps[2]), _p(maps[3]), src_ptrs, cams.ctypes.data_as(ctypes.POINTER(ctypes.c_double)),
                world_from_cam.ctypes.data_as(ctypes.POINTER(ctypes.c_double)), len(srcs), *maps[0].shape,
                float(conf_thr[0]), float(conf_thr[1]), float(conf_thr[2]), float(dist_base), float(rel_diff_base),
                _p(img), capacity, _p(xyz), _p(rgb), _p(total), ctypes.c_void_p(workspace.data_ptr() + offset), _stream()))
            offset += nbytes
    return total, xyz, rgb


def fuse_views(depths: Sequence[torch.Tensor], confidences: Sequence[Sequence[torch.Tensor]], images: Sequence[torch.Tensor],
               Ks, Es, pairs: Sequence[tuple], conf_thr: Sequence[float] = (0.1, 0.15, 0.9), dist_base: float = 1 / 4,
               rel_diff_base: float = 1 / 1300):
    """The loop of reference filter/dypcd.py:filter_depth (:190-300) over a scan that is already on the GPU: for every
    (ref_view, src_views) of `pairs` the fused filter, then the world-space points of the final mask with the reference
    image's colours.  depths[v] [H,W], confidences[v] = (stage1, stage2, stage3) maps, images[v] [H,W,3] in [0,1].
    Returns (xyz [n,3] fp32, rgb [n,3] uint8) on the device, in the reference's order (views, then row-major pixels).
    One native launch per view writes the points straight into a scan-wide buffer; the host waits once, for the count."""
    total, xyz, rgb = _enqueue_points(depths, confidences, images, Ks, Es, pairs, conf_thr, dist_base, rel_diff_base)
    n = int(total.item())
    if n > len(xyz):
        raise RuntimeError(f"fuse_views: {n} points overflow the buffer of {len(xyz)}")
    return xyz[:n].clone(), rgb[:n].clone()


def write_ply(path: str, xyz, rgb) -> None:
    """Binary little-endian PLY with the vertex layout the reference writes through plyfile (filter/dypcd.py:308-321):
    x, y, z float32 and red, green, blue uint8."""
    xyz = np.ascontiguousarray(xyz.detach().cpu().numpy() if isinstance(xyz, torch.Tensor) else xyz, dtype="<f4")
    rgb = np.ascontiguousarray(rgb.detach().cpu().numpy() if isinstance(rgb, torch.Tensor) else rgb, dtype=np.uint8)
    assert xyz.ndim == 2 and xyz.shape[1] == 3 and rgb.shape == xyz.shape
    vert = np.empty(len(xyz), dtype=[("x", "<f4"), ("y", "<f4"), ("z", "<f4"), ("red", "u1"), ("green", "u1"), ("blue", "u1")])
    for i, k in enumerate(("x", "y", "z")):
        vert[k] = xyz[:, i]
    for i, k in enumerate(("red", "green", "blue")):
        vert[k] = rgb[:, i]
    header = ("ply\nformat binary_little_endian 1.0\nelement vertex %d\nproperty float x\nproperty float y\nproperty float z\n"
              "property uchar red\nproperty uchar green\nproperty uchar blue\nend_header\n" % len(xyz))
    with open(path, "wb") as f:
        f.write(header.encode("ascii"))
        f.write(vert.tobytes())
