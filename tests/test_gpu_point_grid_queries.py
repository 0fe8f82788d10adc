"""GPU: the read-outs, spatial queries and carve of the point grids, predicted exactly from their own block dumps.

The point-average grid (`VoxelBlockGrid`) and both semantic grids are fed the golden inputs, then every query is
restated in numpy from `dump_blocks()`, which lists blocks in pool order like the read-outs do:
  count (and confidence) threshold -> block-key range -> voxel-key range -> mean position -> box or frustum test.
Key bounds are floor(bound * (double)inv_voxel_size) with the grid's float32 inverse voxel size; the frustum's key
bounds come from the world AABB of its 8 corners.  The projection is ((R0 x + R1 y) + R2 z) + t in float64, then
float(fx * (x / z) + cx).  The mean is a float32 division for the point-average grid and a float64 division for the
semantic grid.  Outputs are compared with array_equal: same voxels, same order, same bits."""

import os

import numpy as np
import pytest

from pyslam_b200 import (BoundingBox3D, CameraFrustrum, VoxelBlockGrid, VoxelBlockSemanticGrid,
                         VoxelBlockSemanticProbabilisticGrid)
from tests._util import GOLDEN

pytestmark = pytest.mark.gpu

_T = np.arange(512)
LOCAL = np.stack([_T & 7, (_T >> 3) & 7, _T >> 6], axis=1)   # voxel index lx + 8 ly + 64 lz -> (lx, ly, lz)


def key_bounds(bb, inv_vs):
    s = float(np.float32(inv_vs))
    return (np.floor(np.asarray(bb[:3], np.float64) * s).astype(np.int32),
            np.floor(np.asarray(bb[3:], np.float64) * s).astype(np.int32))


def frustum_query(K, W, H, Tcw, depth_max, depth_min):
    """The frustum query as the library builds it: world AABB of the 8 frustum corners, in float64."""
    fx, fy, cx, cy = (float(np.float32(k)) for k in K)
    T = np.asarray(Tcw, np.float64)
    R = [[float(T[i, j]) for j in range(3)] for i in range(3)]
    t = [float(T[i, 3]) for i in range(3)]
    Rwc = [[R[j][i] for j in range(3)] for i in range(3)]
    twc = [-(Rwc[i][0] * t[0] + Rwc[i][1] * t[1] + Rwc[i][2] * t[2]) for i in range(3)]
    lo, hi = [1e300] * 3, [-1e300] * 3
    for u, v in ((0.0, 0.0), (float(W), 0.0), (float(W), float(H)), (0.0, float(H))):
        xn, yn = (u - cx) / fx, (v - cy) / fy
        for d in (float(np.float32(depth_min)), float(np.float32(depth_max))):
            pc = (xn * d, yn * d, d)
            for a in range(3):
                w = Rwc[a][0] * pc[0] + Rwc[a][1] * pc[1] + Rwc[a][2] * pc[2] + twc[a]
                lo[a], hi[a] = min(lo[a], w), max(hi[a], w)
    return dict(bb=np.array(lo + hi), R=np.array(R), t=np.array(t), fx=fx, fy=fy, cx=cx, cy=cy, W=W, H=H,
                depth_min=np.float32(depth_min), depth_max=np.float32(depth_max))


def project(q, p):
    """CameraFrustrum::contains of float64 positions p [..., 3]: (inside, u, v, depth)."""
    R, t = q["R"], q["t"]
    x, y, z = p[..., 0], p[..., 1], p[..., 2]
    pc = [((R[a, 0] * x + R[a, 1] * y) + R[a, 2] * z) + t[a] for a in range(3)]
    depth = pc[2].astype(np.float32)
    u = (q["fx"] * (pc[0] / pc[2]) + q["cx"]).astype(np.float32)
    v = (q["fy"] * (pc[1] / pc[2]) + q["cy"]).astype(np.float32)
    inside = ((depth >= q["depth_min"]) & (depth <= q["depth_max"]) & (u >= 0) & (u < np.float32(q["W"]))
              & (v >= 0) & (v < np.float32(q["H"])))
    return inside, u, v, depth


def spatial_stages(keys, mean, bb, inv_vs, fine):
    """The spatial filter stages of a query on every voxel of a dump, as cumulative masks [nb, 512]."""
    lo, hi = key_bounds(bb, inv_vs)
    blk = np.all((keys >= (lo >> 3)) & (keys <= (hi >> 3)), axis=1)[:, None] & np.ones((1, 512), bool)
    vk = keys[:, None, :].astype(np.int64) * 8 + LOCAL[None]
    vox = blk & np.all((vk >= lo) & (vk <= hi), axis=2)
    return [("block-key range", blk), ("voxel-key range", vox), ("position test", vox & fine(mean))]


def box_test(bb):
    bb = np.asarray(bb, np.float64)
    return lambda p: np.all((p >= bb[:3]) & (p <= bb[3:]), axis=-1)


def quantile_box(p):
    """A box from the 20 % and 80 % quantiles of the voxel means: it cuts through blocks and voxels."""
    return np.concatenate([np.quantile(p, 0.2, axis=0), np.quantile(p, 0.8, axis=0)])


def check_stages(count_mask, stages):
    """Every stage rejects at least one voxel that passed the stages before it; returns the final mask."""
    assert count_mask.any() and not count_mask.all()
    prev = count_mask
    for name, m in stages:
        cur = prev & m
        assert (prev & ~cur).any(), f"the {name} stage rejects nothing"
        prev = cur
    assert prev.any()
    return prev


def feed_point_grid():
    g = np.load(os.path.join(GOLDEN, "refgrid_T0.npz"))
    grid = VoxelBlockGrid(float(g["voxel_size"]), 8, capacity_blocks=4096)
    start = 0
    for n in g["frame_counts"]:
        grid.integrate(g["points"][start:start + n], g["colors"][start:start + n])
        start += int(n)
    return g, grid


def point_grid_means(d):
    with np.errstate(all="ignore"):
        c = d["count"].astype(np.float32)[..., None]
        return d["pos_sum"] / c, d["col_sum"] / c


def point_frustum_args(g):
    K = g["query_K"]
    H, W = g["query_depth"].shape
    return K, W, H, g["query_Tcw"]


def test_point_average_grid_read_outs_equal_their_restatement():
    g, grid = feed_point_grid()
    inv_vs = np.float32(1.0) / np.float32(g["voxel_size"])
    d = grid.dump_blocks()
    count, keys = d["count"], d["keys"]
    mean, col = point_grid_means(d)
    for min_count in (0, 1, 3):
        out = grid.get_voxels(min_count=min_count)
        keep = count >= min_count
        assert np.array_equal(out.points, mean[keep], equal_nan=True)
        assert np.array_equal(out.colors, col[keep], equal_nan=True)
    assert grid.size() == int((count >= 1).sum())

    pos64 = mean.astype(np.float64)
    bbox = quantile_box(pos64[count > 0])
    keep = check_stages(count >= 2, spatial_stages(keys, pos64, bbox, inv_vs, box_test(bbox)))
    out = grid.get_voxels_in_bb(BoundingBox3D(*bbox), min_count=2)
    assert np.array_equal(out.points, mean[keep]) and np.array_equal(out.colors, col[keep])

    K, W, H, Tcw = point_frustum_args(g)
    q = frustum_query(K, W, H, Tcw, 2.0, 0.05)
    keep = check_stages(count >= 2, spatial_stages(keys, pos64, q["bb"], inv_vs, lambda p: project(q, p)[0]))
    fr = CameraFrustrum(K[0], K[1], K[2], K[3], W, H, Tcw, depth_max=2.0, depth_min=0.05)
    out = grid.get_voxels_in_camera_frustrum(fr, min_count=2)
    assert np.array_equal(out.points, mean[keep]) and np.array_equal(out.colors, col[keep])


def carve_reset(count, keys, mean64, q, inv_vs, depth, thr):
    """The voxels a carve resets: in the frustum (count >= 1) and in front of the observed depth by more than thr."""
    keep = check_stages(count >= 1, spatial_stages(keys, mean64, q["bb"], inv_vs, lambda p: project(q, p)[0]))
    with np.errstate(all="ignore"):
        _, u, v, z = project(q, mean64)
    img = np.zeros(count.shape, np.float32)
    img[keep] = depth[v[keep].astype(np.int32), u[keep].astype(np.int32)]
    reset = keep & (img > 0) & np.isfinite(img) & (z < img - np.float32(thr))
    assert reset.any() and (keep & ~reset).any()
    return reset


def test_point_average_grid_carve_resets_the_restated_voxels():
    g, grid = feed_point_grid()
    inv_vs = np.float32(1.0) / np.float32(g["voxel_size"])
    d = grid.dump_blocks()
    mean, _ = point_grid_means(d)
    K, W, H, Tcw = point_frustum_args(g)
    q = frustum_query(K, W, H, Tcw, 3.0, 0.05)
    with np.errstate(all="ignore"):
        reset = carve_reset(d["count"], d["keys"], mean.astype(np.float64), q, inv_vs, g["query_depth"], 0.05)
    grid.carve(CameraFrustrum(K[0], K[1], K[2], K[3], W, H, Tcw, depth_max=3.0, depth_min=0.05), g["query_depth"],
               depth_threshold=0.05)
    after = grid.dump_blocks()
    assert np.array_equal(after["keys"], d["keys"])
    assert np.array_equal(after["count"], np.where(reset, 0, d["count"]))
    assert np.array_equal(after["pos_sum"], np.where(reset[..., None], np.float32(0), d["pos_sum"]))


def feed_semantic_grid(tag):
    g = np.load(os.path.join(GOLDEN, "semantic_T0.npz"))
    cls_t = VoxelBlockSemanticGrid if tag == "vote" else VoxelBlockSemanticProbabilisticGrid
    grid = cls_t(float(g["voxel_size"]), 8, capacity_blocks=1024)
    grid.set_depth_threshold(float(g[f"{tag}_depth_threshold"]))
    grid.set_depth_decay_rate(float(g[f"{tag}_depth_decay_rate"]))
    for i in range(int(g["n_frames"])):
        grid.integrate(*[g[f"{tag}_{n}_{i}"] for n in ("points", "colors", "cls", "inst", "depths")])
    return g, grid


def semantic_emit(d):
    """What a read-out returns for every voxel: float64 mean (0 for an empty voxel), float32 colour mean, labels."""
    c = d["count"]
    with np.errstate(all="ignore"):
        pts = np.where(c[..., None] > 0, d["pos_sum"] / c[..., None].astype(np.float64), 0.0)
        cols = np.where(c[..., None] > 0, d["col_sum"] / c[..., None].astype(np.float32), np.float32(0))
    return pts, cols


def assert_semantic_out(out, d, pts, cols, keep):
    assert np.array_equal(out.points, pts[keep]) and np.array_equal(out.colors, cols[keep])
    assert np.array_equal(out.class_ids, d["class_id"][keep])
    assert np.array_equal(out.object_ids, d["object_id"][keep])
    assert np.array_equal(out.confidences, d["confidence"][keep])


def semantic_frustum_args():
    a = np.load(os.path.join(GOLDEN, "semantic_assoc_T0.npz"))
    return np.array(a["K"], np.float32), 96, 72, a["Tcw_2"], a["depth_2"]


@pytest.mark.parametrize("tag", ["vote", "prob"])
def test_semantic_grid_read_outs_equal_their_restatement(tag):
    g, grid = feed_semantic_grid(tag)
    inv_vs = np.float32(1.0) / np.float32(g["voxel_size"])
    d = grid.dump_blocks(8)
    count, keys, conf = d["count"], d["keys"], d["confidence"]
    pts, cols = semantic_emit(d)
    for min_count, min_conf in ((0, 0.0), (1, 0.0), (3, 0.0), (1, 0.6), (3, 0.6)):
        keep = (count >= min_count) & (conf >= np.float32(min_conf))
        assert keep.any() and (min_count == 0 or not keep.all())
        assert_semantic_out(grid.get_voxels(min_count, min_conf), d, pts, cols, keep)

    bbox = quantile_box(pts[count > 0])
    keep = check_stages((count >= 2) & (conf >= np.float32(0.3)),
                        spatial_stages(keys, pts, bbox, inv_vs, box_test(bbox)))
    assert_semantic_out(grid.get_voxels_in_bb(BoundingBox3D(*bbox), 2, 0.3), d, pts, cols, keep)

    K, W, H, Tcw, _ = semantic_frustum_args()
    q = frustum_query(K, W, H, Tcw, 2.0, 0.05)
    with np.errstate(all="ignore"):
        keep = check_stages((count >= 2) & (conf >= np.float32(0.3)),
                            spatial_stages(keys, pts, q["bb"], inv_vs, lambda p: project(q, p)[0]))
    fr = CameraFrustrum(K[0], K[1], K[2], K[3], W, H, Tcw, depth_max=2.0, depth_min=0.05)
    assert_semantic_out(grid.get_voxels_in_camera_frustrum(fr, 2, 0.3), d, pts, cols, keep)


@pytest.mark.parametrize("tag", ["vote", "prob"])
def test_semantic_grid_carve_resets_the_restated_voxels(tag):
    g, grid = feed_semantic_grid(tag)
    inv_vs = np.float32(1.0) / np.float32(g["voxel_size"])
    d = grid.dump_blocks(8)
    K, W, H, Tcw, depth = semantic_frustum_args()
    c = d["count"][..., None].astype(np.float64)
    with np.errstate(all="ignore"):
        reset = carve_reset(d["count"], d["keys"], d["pos_sum"] / c, frustum_query(K, W, H, Tcw, 3.0, 0.05),
                            inv_vs, depth, 0.02)
    grid.carve(CameraFrustrum(K[0], K[1], K[2], K[3], W, H, Tcw, depth_max=3.0, depth_min=0.05), depth,
               depth_threshold=0.02)
    after = grid.dump_blocks(8)
    assert np.array_equal(after["keys"], d["keys"])
    assert np.array_equal(after["count"], np.where(reset, 0, d["count"]))
    assert np.array_equal(after["object_id"], np.where(reset, -1, d["object_id"]))
