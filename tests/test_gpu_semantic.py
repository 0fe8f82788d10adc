"""GPU: semantic voxel-block grids (SURVEY.md §8(f) rank 2) through the C ABI (b2v_sgrid_*).

(1) the reference's own known-answer tests (cpp/test_volumetric_voxel_semantic.py:20-229), assertion for assertion;
(2) the committed dump of the UNMODIFIED compiled reference (tests/golden/semantic_T0.npz): block keys, hashes,
    counts, float64 position sums, float32 colour sums, labels and counters BIT-EXACT; label evidence bit-exact
    except for one-ulp expf differences (glibc vs float64-rounded) on a handful of depth-decay weights;
    Bayesian confidence within 2e-6 relative;
(3) live against oracle/_ref when it travelled, with edits (remove / merge) and every input-dtype variant."""

import os

import numpy as np
import pytest

import oracle
from pyslam_b200 import (VoxelBlockSemanticGrid, VoxelBlockSemanticProbabilisticGrid, VoxelSemanticGrid,
                         VoxelSemanticGridProbabilistic)
from tests._util import GOLDEN, SEGMENT_QUERIES, feed_segment_blobs, golden_segments, segment_blobs, sort_dump

pytestmark = pytest.mark.gpu

BASE_LOG = 0.10536051565782628


def _zeros_points(n):
    return np.zeros((n, 3), dtype=np.float64)


def _zeros_colors(n):
    return np.zeros((n, 3), dtype=np.uint8)


# ---- (1) the reference KATs ------------------------------------------------------------------------------------
def test_kat_voting_label_switch_and_confidence():
    grid = VoxelSemanticGrid(0.1)
    grid.integrate(_zeros_points(2), _zeros_colors(2), np.array([1, 2], np.int32), np.array([1, 2], np.int32))
    v = grid.get_voxels(min_count=1, min_confidence=0.0)
    assert len(v.object_ids) == 1 and v.object_ids[0] == 2 and v.class_ids[0] == 2
    assert v.confidences[0] == pytest.approx(0.5, abs=1e-3)


def test_kat_probabilistic_majority_depth_decay_and_strong_majority():
    grid = VoxelSemanticGridProbabilistic(0.1)
    grid.integrate(_zeros_points(4), _zeros_colors(4), np.array([5, 5, 5, 6], np.int32),
                   np.array([1, 1, 1, 2], np.int32))
    v = grid.get_voxels(min_count=1, min_confidence=0.0)
    assert len(v.object_ids) == 1 and v.object_ids[0] == 1 and v.class_ids[0] == 5 and v.confidences[0] > 0.5
    grid = VoxelSemanticGridProbabilistic(0.1)
    grid.integrate(_zeros_points(2), _zeros_colors(2), np.array([7, 8], np.int32), np.array([3, 4], np.int32),
                   np.array([1.0, 20.0], np.float32))
    v = grid.get_voxels(min_count=1, min_confidence=0.0)
    assert len(v.object_ids) == 1 and v.object_ids[0] == 3 and v.class_ids[0] == 7 and v.confidences[0] > 0.5
    grid = VoxelSemanticGridProbabilistic(0.1)
    grid.integrate(_zeros_points(13), _zeros_colors(13), np.array([5] * 12 + [6], np.int32),
                   np.array([1] * 12 + [2], np.int32))
    v = grid.get_voxels(min_count=1, min_confidence=0.0)
    assert v.object_ids[0] == 1 and v.class_ids[0] == 5 and v.confidences[0] > 0.7


def test_kat_labels_across_voxels():
    grid = VoxelSemanticGrid(0.1)
    grid.integrate(np.array([[0.0, 0.0, 0.0], [0.2, 0.0, 0.0]]), _zeros_colors(2), np.array([10, 20], np.int32),
                   np.array([101, 202], np.int32))
    v = grid.get_voxels(min_count=1, min_confidence=0.0)
    paired = sorted(zip(map(tuple, v.points), v.object_ids, v.class_ids))
    assert len(paired) == 2 and paired[0][1:] == (101, 10) and paired[1][1:] == (202, 20)


def test_kat_label_noise_and_joint_softmax():
    for cls_t, seed, maj, noise, labels in ((VoxelSemanticGridProbabilistic, 0, 50, 5, ((111, 11), (222, 12))),
                                            (VoxelSemanticGrid, 1, 30, 3, ((210, 21), (220, 22)))):
        rng = np.random.default_rng(seed)
        tot = maj + noise
        pts = rng.uniform(low=0.0, high=0.05, size=(tot, 3)).astype(np.float64)
        cls = np.array([labels[0][1]] * maj + [labels[1][1]] * noise, np.int32)
        ins = np.array([labels[0][0]] * maj + [labels[1][0]] * noise, np.int32)
        perm = rng.permutation(tot)
        grid = cls_t(0.2)
        grid.integrate(pts[perm], _zeros_colors(tot), cls[perm], ins[perm])
        v = grid.get_voxels(min_count=1, min_confidence=0.0)
        assert len(v.object_ids) == 1 and (v.object_ids[0], v.class_ids[0]) == labels[0]
        if cls_t is VoxelSemanticGridProbabilistic:
            assert v.confidences[0] > 0.75
        else:
            assert v.confidences[0] == pytest.approx((maj - noise) / float(tot), abs=1e-2)
    pc = {(1, 10): 3, (1, 11): 3, (2, 10): 4}
    ins = np.concatenate([[o] * k for (o, c), k in pc.items()]).astype(np.int32)
    cls = np.concatenate([[c] * k for (o, c), k in pc.items()]).astype(np.int32)
    perm = np.random.default_rng(42).permutation(10)
    grid = VoxelSemanticGridProbabilistic(0.1)
    grid.integrate(_zeros_points(10), _zeros_colors(10), cls[perm], ins[perm])
    v = grid.get_voxels(min_count=1, min_confidence=0.0)
    lp = np.array([4, 3, 3]) * BASE_LOG
    assert v.object_ids[0] == 2 and v.class_ids[0] == 10
    assert v.confidences[0] == pytest.approx(np.exp(lp[0]) / np.exp(lp).sum(), rel=1e-4, abs=1e-4)


# ---- (2) golden dump of the compiled reference --------------------------------------------------------------------
def _compare_dumps(a, b, kind):
    assert np.array_equal(a["keys"], b["keys"]) and np.array_equal(a["hashes"], b["hashes"])
    for k in ("count", "pos_sum", "col_sum", "object_id", "class_id", "aux"):
        assert np.array_equal(a[k], b[k]), k
    if kind == "prob":
        assert np.array_equal(a["lab_obj"], b["lab_obj"]) and np.array_equal(a["lab_cls"], b["lab_cls"])
        # evidence: bit-exact except where glibc's expf (not correctly rounded) and the GPU's float64-rounded exp
        # disagree by one ulp on a depth-decay weight - a handful of the ~10^5 observations
        fa, fb = np.isfinite(a["lab_logp"]), np.isfinite(b["lab_logp"])
        assert np.array_equal(fa, fb)
        ndiff = int((a["lab_logp"][fa] != b["lab_logp"][fb]).sum())
        assert ndiff <= max(2, fa.sum() // 1000), ndiff
        assert np.allclose(a["lab_logp"][fa], b["lab_logp"][fb], rtol=1e-6, atol=0)
        bad = np.argwhere(~np.isclose(a["confidence"], b["confidence"], rtol=2e-6, atol=1e-9))
        assert len(bad) == 0, (len(bad), [(tuple(i), a["confidence"][tuple(i)], b["confidence"][tuple(i)],
                                           b["count"][tuple(i)], b["aux"][tuple(i)], b["object_id"][tuple(i)],
                                           b["class_id"][tuple(i)], b["lab_obj"][tuple(i)].tolist(),
                                           b["lab_cls"][tuple(i)].tolist(), b["lab_logp"][tuple(i)].tolist())
                                          for i in bad[:4]])
    else:
        assert np.array_equal(a["confidence"], b["confidence"])


@pytest.mark.parametrize("tag", ["vote", "prob"])
def test_golden_reference_dump(tag):
    g = np.load(os.path.join(GOLDEN, "semantic_T0.npz"))
    cls_t = VoxelBlockSemanticGrid if tag == "vote" else VoxelBlockSemanticProbabilisticGrid
    grid = cls_t(float(g["voxel_size"]), 8, capacity_blocks=1024)
    grid.set_depth_threshold(float(g[f"{tag}_depth_threshold"]))
    grid.set_depth_decay_rate(float(g[f"{tag}_depth_decay_rate"]))
    for i in range(int(g["n_frames"])):
        grid.integrate(g[f"{tag}_points_{i}"], g[f"{tag}_colors_{i}"], g[f"{tag}_cls_{i}"], g[f"{tag}_inst_{i}"],
                       g[f"{tag}_depths_{i}"])
    ref = {k: g[f"{tag}_{k}"] for k in ("keys", "hashes", "count", "pos_sum", "col_sum", "object_id", "class_id",
                                         "confidence", "aux", "lab_obj", "lab_cls", "lab_logp")}
    _compare_dumps(sort_dump(grid.dump_blocks(8)), ref, tag)
    assert grid.label_overflows() == 0
    v = grid.get_voxels(2, 0.4)
    order = np.lexsort((v.points[:, 2], v.points[:, 1], v.points[:, 0]))
    # voxels whose confidence sits within float rounding of 0.4 may flip for the Bayesian grid
    if len(order) == len(g[f"{tag}_voxels_points"]):
        assert np.array_equal(v.points[order], g[f"{tag}_voxels_points"])
        assert np.array_equal(v.colors[order], g[f"{tag}_voxels_colors"])
        assert np.array_equal(v.class_ids[order], g[f"{tag}_voxels_class_ids"])
        assert np.array_equal(v.object_ids[order], g[f"{tag}_voxels_object_ids"])
        assert np.allclose(v.confidences[order], g[f"{tag}_voxels_confidences"], rtol=2e-6)
    else:
        assert tag == "prob" and abs(len(order) - len(g[f"{tag}_voxels_points"])) <= 2
    assert grid.num_blocks() == len(ref["keys"]) and grid.size() == int((ref["count"] > 0).sum())
    grid.clear()
    assert grid.empty() and len(grid.get_voxels(1, 0.0).points) == 0


# ---- (3) live against the compiled reference ----------------------------------------------------------------------
@pytest.mark.skipif(not oracle.have_ref_semantic(), reason="compiled reference (oracle/_ref) not on this box")
@pytest.mark.parametrize("kind", ["voting", "probabilistic"])
def test_live_against_compiled_reference_with_edits(kind):
    rng = np.random.default_rng(11)
    vs = 0.05
    cls_t = VoxelBlockSemanticGrid if kind == "voting" else VoxelBlockSemanticProbabilisticGrid
    ref = oracle.RefSemanticGrid(vs, kind)
    grid = cls_t(vs, 8, capacity_blocks=1 << 12)
    thr, rate = (2.0, 0.0) if kind == "voting" else (1.5, 0.8)
    ref.set_depth_threshold(thr)
    grid.set_depth_threshold(thr)
    if kind == "probabilistic":
        ref.set_depth_decay_rate(rate)
        grid.set_depth_decay_rate(rate)
    tag = "vote" if kind == "voting" else "prob"
    variants = [dict(f64=True, u8=False, inst=True, depth=True), dict(f64=False, u8=True, inst=True, depth=False),
                dict(f64=True, u8=False, inst=False, depth=True), dict(f64=False, u8=False, inst=False, depth=False)]
    for var in variants:
        n = 30000
        dirs = rng.normal(size=(n, 3))
        dirs /= np.linalg.norm(dirs, axis=1, keepdims=True)
        pts = dirs * (0.5 + 0.01 * rng.normal(size=(n, 1))) + [0.05, -0.1, 0.02]   # shell across the origin
        pts = pts.astype(np.float64 if var["f64"] else np.float32)
        cols_u8 = rng.integers(0, 256, size=(n, 3), dtype=np.uint8)
        # the reference harness takes float colours; uint8 goes through c * (1.0f / 255.0f) (voxel_data.h:82-85)
        cols_f = (cols_u8.astype(np.float32) * (np.float32(1.0) / np.float32(255.0))) if var["u8"] \
            else rng.random((n, 3)).astype(np.float32)
        side = (pts[:, 0] > 0).astype(np.int32)
        flip, noise = rng.random(n) < 0.2, rng.integers(-1, 1, n)    # correlated label noise incl. the invalid id -1
        cls = np.where(flip, noise, 1 + side).astype(np.int32)
        ins = np.where(flip, noise, 10 + side).astype(np.int32)
        dep = rng.uniform(0.5, 4.0, n).astype(np.float32)
        ref.integrate(pts, cols_f, cls, ins if var["inst"] else None, dep if var["depth"] else None)
        grid.integrate(pts, cols_u8 if var["u8"] else cols_f, cls, ins if var["inst"] else None,
                       dep if var["depth"] else None)
    a, b = sort_dump(grid.dump_blocks(8)), sort_dump(ref.dump_blocks(8))
    assert b["aux"].max() <= 8 or kind == "voting"
    _compare_dumps(a, b, tag)
    # edits: merge two objects, drop one, drop low-count voxels, then compare again
    for g_ in (ref, grid):
        g_.merge_segments(10, 11)
        g_.remove_segment(0)
        g_.remove_low_count_voxels(3)
    a, b = sort_dump(grid.dump_blocks(8)), sort_dump(ref.dump_blocks(8))
    assert np.array_equal(a["count"], b["count"]) and np.array_equal(a["object_id"], b["object_id"])
    assert np.array_equal(a["class_id"], b["class_id"])
    assert np.allclose(a["confidence"], b["confidence"], rtol=2e-6, atol=1e-9)
    rv = ref.get_voxels(2, 0.3)
    gv = grid.get_voxels(2, 0.3)
    assert abs(len(gv.points) - len(rv["points"])) <= 2 and len(rv["points"]) > 50
    for g_ in (ref, grid):
        g_.remove_low_confidence_segments(1)      # int threshold: everything below confidence 1 goes
    a, b = sort_dump(grid.dump_blocks(1)), sort_dump(ref.dump_blocks(1))
    assert np.array_equal(a["count"], b["count"]) and (b["count"] > 0).sum() > 0


def test_label_overflow_is_counted_and_keeps_the_majority():
    grid = VoxelBlockSemanticProbabilisticGrid(0.1, 8, capacity_blocks=64)
    n_noise = 11                                   # 11 distinct minority pairs + the majority pair > 8 slots
    cls = np.array([5] * 20 + list(range(100, 100 + n_noise)), np.int32)
    ins = np.array([1] * 20 + list(range(200, 200 + n_noise)), np.int32)
    perm = np.random.default_rng(3).permutation(len(cls))
    grid.integrate(np.zeros((len(cls), 3), np.float32), np.zeros((len(cls), 3), np.float32), cls[perm], ins[perm])
    v = grid.get_voxels(1, 0.0)
    assert (v.object_ids[0], v.class_ids[0]) == (1, 5)
    assert grid.label_overflows() == n_noise + 1 - 8
    with pytest.raises(RuntimeError):
        grid.integrate(np.zeros((2, 3), np.float32), None, None, np.array([1, 2], np.int32))
    with pytest.raises(RuntimeError):
        grid.integrate(np.zeros((2, 3), np.float32), np.zeros((2, 3), np.float32), np.array([1], np.int32))
    with pytest.raises(RuntimeError):
        VoxelBlockSemanticGrid(0.1, 4)


def test_fused_rgbd_front_end_matches_the_reference_pipeline():
    """integrate_rgbd(depth, color, class / object images) == the reference's own front-end functions
    (filter_shadow_points, depth2pointcloud with label images; tests/golden/semantic_frontend_T0.npz) feeding the
    compiled reference grid.  The reference transforms with BLAS (`inv_pose @ points.T`), so a point may land one
    float32 ulp away and cross a voxel face: a handful of voxels out of ~1800 may differ; all others are exact."""
    from pyslam_b200 import synthetic as S
    g = np.load(os.path.join(GOLDEN, "semantic_frontend_T0.npz"))
    grid = VoxelBlockSemanticProbabilisticGrid(float(g["voxel_size"]), 8, capacity_blocks=1024)
    grid.set_depth_threshold(float(g["depth_threshold"]))
    grid.set_depth_decay_rate(float(g["depth_decay_rate"]))
    for i in range(g["depth"].shape[0]):
        grid.integrate_rgbd(g["depth"][i], g["color"][i], g["K"], S.inv_T(g["Tcw"][i]), g["class_image"][i],
                            g["object_image"][i], max_depth=float(g["max_depth"]), use_depths=True,
                            filter_shadow_points=True)
    d = sort_dump(grid.dump_blocks(8))
    assert np.array_equal(d["keys"], g["keys"]) and np.array_equal(d["hashes"], g["hashes"])
    same = d["count"] == g["count"]
    assert int((~same).sum()) <= 6, int((~same).sum())
    occ = same & (g["count"] > 0)
    exact = occ & np.all(d["pos_sum"] == g["pos_sum"], axis=-1)
    assert exact.sum() >= 0.99 * occ.sum()                       # same points in the same order: float64 sums equal
    assert np.array_equal(d["col_sum"][exact], g["col_sum"][exact])
    assert np.array_equal(d["object_id"][exact], g["object_id"][exact])
    assert np.array_equal(d["class_id"][exact], g["class_id"][exact])
    assert np.array_equal(d["aux"][exact], g["aux"][exact])
    fin = np.isfinite(g["lab_logp"][exact])
    assert np.array_equal(np.isfinite(d["lab_logp"][exact]), fin)
    assert np.allclose(d["lab_logp"][exact][fin], g["lab_logp"][exact][fin], rtol=1e-6, atol=0)
    assert np.allclose(d["confidence"][exact], g["confidence"][exact], rtol=2e-6, atol=1e-9)
    # the explicit-array path fed the same frame gives the same grid as the fused one (no filter, no BLAS involved)
    a = VoxelBlockSemanticGrid(0.05, 8, capacity_blocks=1024)
    b = VoxelBlockSemanticGrid(0.05, 8, capacity_blocks=1024)
    dep, col, K, T = g["depth"][0], g["color"][0], g["K"], S.inv_T(g["Tcw"][0])
    a.integrate_rgbd(dep, col, K, T, g["class_image"][0], g["object_image"][0], max_depth=float(g["max_depth"]))
    valid = (dep > 0) & (dep < float(g["max_depth"]))
    z = dep[valid].astype(np.float64)
    rows, cols = np.where(valid)
    x, y = (cols - K[2]) * z * (1.0 / K[0]), (rows - K[3]) * z * (1.0 / K[1])
    pw = np.stack([x * T[r, 0] + y * T[r, 1] + z * T[r, 2] + T[r, 3] for r in range(3)], axis=1).astype(np.float32)
    b.integrate(pw, (col[valid] / 255.0).astype(np.float32), g["class_image"][0][valid], g["object_image"][0][valid],
                dep[valid])
    da, db = sort_dump(a.dump_blocks(1)), sort_dump(b.dump_blocks(1))
    for k in ("keys", "count", "pos_sum", "col_sum", "object_id", "class_id", "aux", "confidence"):
        assert np.array_equal(da[k], db[k]), k


def test_replica_shape_frame_split_equals_whole():
    """BASELINE config 3 shape (1200x680, labelled): a size-independent property of the order-preserving fusion -
    integrating a frame's points in one call equals integrating its two halves in two calls, bit for bit; counts
    add up to the number of points; the voting confidence stays in [0, 1]."""
    rng = np.random.default_rng(5)
    h, w = 680, 1200
    n = h * w
    u, v = np.meshgrid(np.arange(w), np.arange(h))
    z = 2.0 + 0.3 * np.sin(u / 90.0) + 0.2 * np.cos(v / 70.0)
    pts = np.stack([(u - 600) / 600.0 * z, (v - 340) / 600.0 * z, z], axis=-1).reshape(-1, 3).astype(np.float32)
    cols = rng.integers(0, 256, (n, 3), dtype=np.uint8)
    cls = (1 + (u // 150 + v // 170) % 5).reshape(-1).astype(np.int32)
    cls = np.where(rng.random(n) < 0.1, rng.integers(0, 6, n), cls).astype(np.int32)
    ins = (cls * 100 + (u // 300).reshape(-1)).astype(np.int32)
    dep = z.reshape(-1).astype(np.float32)
    for cls_t in (VoxelBlockSemanticGrid, VoxelBlockSemanticProbabilisticGrid):
        whole = cls_t(0.005, 8, capacity_blocks=1 << 15)
        halves = cls_t(0.005, 8, capacity_blocks=1 << 15)
        for g_ in (whole, halves):
            g_.set_depth_threshold(2.1)
        whole.integrate(pts, cols, cls, ins, dep)
        m = n // 2 + 12345
        halves.integrate(pts[:m], cols[:m], cls[:m], ins[:m], dep[:m])
        halves.integrate(pts[m:], cols[m:], cls[m:], ins[m:], dep[m:])
        va, vb = whole.get_voxels(1, 0.0), halves.get_voxels(1, 0.0)
        oa = np.lexsort((va.points[:, 2], va.points[:, 1], va.points[:, 0]))
        ob = np.lexsort((vb.points[:, 2], vb.points[:, 1], vb.points[:, 0]))
        assert len(oa) == len(ob) > 100000
        for name in ("points", "colors", "class_ids", "object_ids", "confidences"):
            assert np.array_equal(getattr(va, name)[oa], getattr(vb, name)[ob]), name
        assert va.confidences.min() >= 0.0 and va.confidences.max() <= 1.0
        assert whole.label_overflows() == 0
        whole.close()
        halves.close()


@pytest.mark.parametrize("tag", ["vote", "prob"])
def test_instance_association_pipeline_matches_the_reference(tag):
    """The reference integrator's loop body (assign_object_ids_to_instance_ids with carving -> remap_instance_ids ->
    integrate) replayed over 4 frames whose 2-D instance ids change every frame, against the maps and the final
    grid of the UNMODIFIED compiled reference (tests/golden/semantic_assoc_T0.npz).  New object ids are handed out
    in a different order (ascending instance id here, block-iteration order there), so ids are compared through
    the bijection the maps themselves define."""
    from pyslam_b200 import CameraFrustrum, remap_instance_ids
    from pyslam_b200 import synthetic as S
    g = np.load(os.path.join(GOLDEN, "semantic_assoc_T0.npz"))
    cls_t = VoxelBlockSemanticGrid if tag == "vote" else VoxelBlockSemanticProbabilisticGrid
    grid = cls_t(float(g["voxel_size"]), 8, capacity_blocks=1024)
    grid.set_depth_threshold(10.0)
    K = g["K"]
    phi = {-1: -1, 0: 0}           # reference object id -> our object id
    for i in range(int(g["n_frames"])):
        d, c, T = g[f"depth_{i}"], g[f"color_{i}"], g[f"Tcw_{i}"]
        cls_img, inst_img = g[f"class_image_{i}"], g[f"instance_image_{i}"]
        h, w = d.shape
        fr = CameraFrustrum(K[0], K[1], K[2], K[3], w, h, T, depth_max=float(g["param_depth_max"]),
                            depth_min=float(g["param_depth_min"]))
        m = grid.assign_object_ids_to_instance_ids(fr, cls_img, inst_img, d, float(g["param_depth_threshold"]),
                                                   bool(g["param_do_carving"]), float(g["param_min_vote_ratio"]),
                                                   int(g["param_min_votes"]))
        ref = dict(zip(g[f"{tag}_map_inst_{i}"].tolist(), g[f"{tag}_map_obj_{i}"].tolist()))
        assert sorted(m) == sorted(ref), (i, m, ref)
        for k, ro in ref.items():
            assert phi.setdefault(ro, m[k]) == m[k], (i, k, ro, m[k], phi)
        obj_img = remap_instance_ids(inst_img, m)
        Twc = S.inv_T(T)
        valid = (d > 0) & (d < float(g["max_depth"]))
        z = d[valid].astype(np.float64)
        rows, cols = np.where(valid)
        x, y = (cols - K[2]) * z * (1.0 / K[0]), (rows - K[3]) * z * (1.0 / K[1])
        pw = np.stack([x * Twc[r, 0] + y * Twc[r, 1] + z * Twc[r, 2] + Twc[r, 3] for r in range(3)],
                      axis=1).astype(np.float32)
        grid.integrate(pw, (c[valid] / 255.0).astype(np.float32), cls_img[valid], obj_img[valid], d[valid])
    assert len(set(phi.values())) == len(phi)                      # a bijection
    assert grid.get_next_object_id() == int(g[f"{tag}_next_object_id"])
    dmp = sort_dump(grid.dump_blocks(1))
    assert np.array_equal(dmp["keys"], g[f"{tag}_keys"])
    # carving compares float depths against the image: a voxel within rounding of the threshold may flip
    same = dmp["count"] == g[f"{tag}_count"]
    assert int((~same).sum()) <= 4, int((~same).sum())
    lut = np.vectorize(lambda o: phi.get(int(o), -12345))
    occ = same & (g[f"{tag}_count"] > 0)
    assert np.array_equal(dmp["object_id"][occ], lut(g[f"{tag}_object_id"][occ]))
    assert np.array_equal(dmp["class_id"][occ], g[f"{tag}_class_id"][occ])
    assert np.allclose(dmp["confidence"][occ], g[f"{tag}_confidence"][occ], rtol=2e-6, atol=1e-9)
    assert (g[f"{tag}_object_id"][occ] > 0).sum() > 200           # objects really were associated
    # soft failures and argument checks
    assert grid.assign_object_ids_to_instance_ids(fr, cls_img[:5], inst_img) == {}
    grid.carve(fr, d[:5])                                          # wrong size: no-op
    before = sort_dump(grid.dump_blocks(1))["count"]
    grid.carve(fr, d + 0.5, depth_threshold=0.05)                  # the surface moved back: carve what is in front
    after = sort_dump(grid.dump_blocks(1))["count"]
    assert (after > 0).sum() < (before > 0).sum()


@pytest.mark.skipif(not oracle.have_ref_semantic(), reason="compiled reference (oracle/_ref) not on this box")
@pytest.mark.parametrize("tag", ["vote", "prob"])
def test_spatial_read_outs_match_the_compiled_reference(tag):
    """get_voxels_in_camera_frustrum / get_voxels_in_bb (with labels) against the compiled reference fed the same
    stream (tests/golden/semantic_T0.npz inputs).  Compared as sets ordered by position; a voxel whose projection
    or mean lies within float rounding of a bound, or whose Bayesian confidence lies within rounding of the
    threshold, may flip (<= 3 voxels)."""
    from pyslam_b200 import BoundingBox3D, CameraFrustrum
    g = np.load(os.path.join(GOLDEN, "semantic_T0.npz"))
    a = np.load(os.path.join(GOLDEN, "semantic_assoc_T0.npz"))
    kind = "voting" if tag == "vote" else "probabilistic"
    cls_t = VoxelBlockSemanticGrid if tag == "vote" else VoxelBlockSemanticProbabilisticGrid
    ref = oracle.RefSemanticGrid(float(g["voxel_size"]), kind)
    grid = cls_t(float(g["voxel_size"]), 8, capacity_blocks=1024)
    for g_ in (ref, grid):
        g_.set_depth_threshold(float(g[f"{tag}_depth_threshold"]))
        g_.set_depth_decay_rate(float(g[f"{tag}_depth_decay_rate"]))
    for i in range(int(g["n_frames"])):
        args = [g[f"{tag}_{n}_{i}"] for n in ("points", "colors", "cls", "inst", "depths")]
        ref.integrate(*args)
        grid.integrate(*args)
    K = np.array(a["K"], np.float32)
    T = a["Tcw_2"]

    def same(out, r):
        assert abs(len(out.points) - len(r["points"])) <= 3 and len(r["points"]) > 20
        if len(out.points) != len(r["points"]):
            return
        o1 = np.lexsort((out.points[:, 2], out.points[:, 1], out.points[:, 0]))
        o2 = np.lexsort((r["points"][:, 2], r["points"][:, 1], r["points"][:, 0]))
        assert np.array_equal(out.points[o1], r["points"][o2])
        assert np.array_equal(out.colors[o1], r["colors"][o2])
        assert np.array_equal(out.class_ids[o1], r["class_ids"][o2])
        assert np.array_equal(out.object_ids[o1], r["object_ids"][o2])
        assert np.allclose(out.confidences[o1], r["confidences"][o2], rtol=2e-6, atol=1e-9)

    fr = CameraFrustrum(K[0], K[1], K[2], K[3], 96, 72, T, depth_max=3.0, depth_min=0.05)
    same(grid.get_voxels_in_camera_frustrum(fr, 2, 0.3), ref.get_voxels_in_camera_frustrum(K, 96, 72, T, 3.0, 0.05, 2, 0.3))
    pts = ref.get_voxels(1, 0.0)["points"]
    box = np.concatenate([np.quantile(pts, 0.2, axis=0), np.quantile(pts, 0.8, axis=0)])
    same(grid.get_voxels_in_bb(BoundingBox3D(*box), 1, 0.2), ref.get_voxels_in_bb(box, 1, 0.2))
    same(grid.get_voxels(1, 0.0), ref.get_voxels(1, 0.0))


@pytest.mark.parametrize("kind", ["voting", "probabilistic"])
def test_object_and_class_segments_and_integrate_segment_match_the_reference(kind):
    """get_object_segments / get_class_segments / integrate_segment (voxel_block_semantic_grid.hpp:52-99, 204-316)
    against the stored segments of the same stream (tests/golden/segments_T0.npz; its `source` says what recorded it,
    and test_oracle_semantic.py::test_compiled_reference_reproduces_the_segment_goldens compares it with the
    UNMODIFIED compiled reference at these tolerances): same segment ids, the same voxels (positions, colours) in
    every segment, class ids, confidence ranges; PCA boxes to 1e-9."""
    from pyslam_b200 import VoxelBlockSemanticGrid, VoxelBlockSemanticProbabilisticGrid
    ref = np.load(os.path.join(GOLDEN, "segments_T0.npz"))
    tag = "vote" if kind == "voting" else "prob"
    Cls = VoxelBlockSemanticGrid if kind == "voting" else VoxelBlockSemanticProbabilisticGrid
    g = Cls(float(ref["voxel_size"]), 8, capacity_blocks=1 << 13)
    blobs = segment_blobs(np.random.default_rng(3), 3000)
    feed_segment_blobs(g, blobs)
    with pytest.raises(RuntimeError):
        g.integrate_segment(blobs[0][2], blobs[0][3][:5], 1, 1)
    for query, (by_class, min_count, min_conf) in enumerate(SEGMENT_QUERIES):
        a = (g.get_class_segments if by_class else g.get_object_segments)(min_count, min_conf)
        b = golden_segments(ref, tag, query)
        av = a.class_vector if by_class else a.object_vector
        ids_a = [x.class_id if by_class else x.object_id for x in av]
        assert sorted(ids_a) == sorted(s["id"] for s in b) and len(b) == 3
        for x in av:
            s = next(s for s in b if s["id"] == (x.class_id if by_class else x.object_id))
            oa = np.lexsort(np.asarray(x.points).T[::-1])
            ob = np.lexsort(s["points"].T[::-1])
            assert np.array_equal(np.asarray(x.points)[oa], s["points"][ob])       # float64 means, bit for bit
            assert np.allclose(np.asarray(x.colors)[oa], s["colors"][ob], rtol=0, atol=1e-6)
            assert abs(x.confidence_min - s["confidence_min"]) < 1e-5
            assert abs(x.confidence_max - s["confidence_max"]) < 1e-5
            if not by_class:
                assert x.class_id == s["class_id"]
                box = x.oriented_bounding_box
                assert np.abs(box.center - s["obb_center"]).max() < 1e-9
                assert np.abs(box.size - s["obb_size"]).max() < 1e-9
    g.close()
