"""CPU: pin the semantic-fusion oracle.  (1) The reference's own known-answer tests
(cpp/test_volumetric_voxel_semantic.py:20-229) run against the UNMODIFIED compiled reference block grids
(oracle/_ref/libref_semantic.so).  (2) The committed golden dump (tests/golden/semantic_T0.npz, produced by that
library) obeys the rules the GPU implementation restates: voting confidence = min(1, counter / count), Bayesian
confidence = softmax of the label evidence, argmax = label with the largest evidence."""

import os

import numpy as np
import pytest

import oracle
from tests._util import GOLDEN

BASE_LOG = 0.10536051565782628  # voxel_data_semantic.h:287

needs_ref = pytest.mark.skipif(not oracle.have_ref_semantic(), reason="oracle/_ref/libref_semantic.so not built")


def _one_voxel(kind, voxel, cls, inst, depths=None, points=None):
    g = oracle.RefSemanticGrid(voxel, kind)
    g.set_depth_threshold(10.0 if kind == "voting" else 5.0)   # class defaults (voxel_data_semantic.h:107,251-254)
    if kind == "probabilistic":
        g.set_depth_decay_rate(0.07)
    n = len(cls)
    g.integrate(np.zeros((n, 3)) if points is None else points, np.zeros((n, 3), np.float32), cls, inst, depths)
    return g.get_voxels(1, 0.0)


@needs_ref
def test_reference_kats_hold_for_the_compiled_block_grids():
    v = _one_voxel("voting", 0.1, [1, 2], [1, 2])                         # :20-36 label switch, confidence 0.5
    assert list(v["object_ids"]) == [2] and list(v["class_ids"]) == [2]
    assert v["confidences"][0] == pytest.approx(0.5, abs=1e-3)
    v = _one_voxel("probabilistic", 0.1, [5, 5, 5, 6], [1, 1, 1, 2])      # :39-55 majority
    assert (v["object_ids"][0], v["class_ids"][0]) == (1, 5) and v["confidences"][0] > 0.5
    v = _one_voxel("probabilistic", 0.1, [7, 8], [3, 4], [1.0, 20.0])     # :58-76 depth decay
    assert (v["object_ids"][0], v["class_ids"][0]) == (3, 7) and v["confidences"][0] > 0.5
    v = _one_voxel("voting", 0.1, [10, 20], [101, 202], points=np.array([[0.0, 0, 0], [0.2, 0, 0]]))  # :79-97
    pairs = sorted(zip(map(tuple, v["points"]), v["object_ids"], v["class_ids"]))
    assert [p[1:] for p in pairs] == [(101, 10), (202, 20)]
    v = _one_voxel("probabilistic", 0.1, [5] * 12 + [6], [1] * 12 + [2])  # :100-120 strong majority
    assert (v["object_ids"][0], v["class_ids"][0]) == (1, 5) and v["confidences"][0] > 0.7
    # :123-185 seeded noise
    for kind, seed, maj, noise, labels, bound in (("probabilistic", 0, 50, 5, ((111, 11), (222, 12)), 0.75),
                                                  ("voting", 1, 30, 3, ((210, 21), (220, 22)), None)):
        rng = np.random.default_rng(seed)
        tot = maj + noise
        pts = rng.uniform(0.0, 0.05, size=(tot, 3))
        cls = np.array([labels[0][1]] * maj + [labels[1][1]] * noise, np.int32)
        ins = np.array([labels[0][0]] * maj + [labels[1][0]] * noise, np.int32)
        perm = rng.permutation(tot)
        v = _one_voxel(kind, 0.2, cls[perm], ins[perm], points=pts[perm])
        assert (v["object_ids"][0], v["class_ids"][0]) == labels[0]
        if bound:
            assert v["confidences"][0] > bound
        else:
            assert v["confidences"][0] == pytest.approx((maj - noise) / tot, abs=1e-2)
    # :188-229 exact softmax of k * BASE_LOG
    pc = {(1, 10): 3, (1, 11): 3, (2, 10): 4}
    ins = np.concatenate([[o] * k for (o, c), k in pc.items()]).astype(np.int32)
    cls = np.concatenate([[c] * k for (o, c), k in pc.items()]).astype(np.int32)
    perm = np.random.default_rng(42).permutation(10)
    v = _one_voxel("probabilistic", 0.1, cls[perm], ins[perm])
    lp = np.array([4, 3, 3]) * BASE_LOG
    assert (v["object_ids"][0], v["class_ids"][0]) == (2, 10)
    assert v["confidences"][0] == pytest.approx(np.exp(lp[0]) / np.exp(lp).sum(), rel=1e-4, abs=1e-4)


def test_golden_dump_obeys_the_fusion_rules():
    g = np.load(os.path.join(GOLDEN, "semantic_T0.npz"))
    # voting: confidence = min(1, counter / count) (voxel_data_semantic.h:117-132)
    cnt, ctr = g["vote_count"], g["vote_aux"]
    occ = cnt > 0
    exp = np.minimum(1.0, ctr[occ].astype(np.float32) / cnt[occ].astype(np.float32))
    assert np.array_equal(g["vote_confidence"][occ], exp.astype(np.float32))
    assert (ctr[occ] < cnt[occ]).any() and (g["vote_object_id"][occ] == -1).any()   # gated + invalid ids occur
    # Bayesian: argmax + softmax over the label evidence (voxel_data_semantic.h:561-570, 607-624)
    lp = g["prob_lab_logp"].astype(np.float64)
    nl = g["prob_aux"]
    occ = (g["prob_count"] > 0) & (nl > 0)
    assert nl.max() <= 8 and nl[occ].min() >= 1 and (nl[occ] > 2).any()
    best = lp[occ].max(axis=1)
    k = lp[occ].argmax(axis=1)
    rows = np.arange(len(k))
    obj, cls = g["prob_lab_obj"][occ][rows, k], g["prob_lab_cls"][occ][rows, k]
    valid = (obj != -1) & (cls != -1)
    # ties keep the earlier label, so compare labels only where the maximum is unique
    srt = np.sort(lp[occ], axis=1)
    unique = (srt[:, -1] - srt[:, -2] > 1e-6) | (nl[occ] == 1)
    assert np.array_equal(g["prob_object_id"][occ][unique], obj[unique])
    assert np.array_equal(g["prob_class_id"][occ][unique], cls[unique])
    soft = np.exp(best - np.log(np.exp(lp[occ]).sum(axis=1)))
    conf = g["prob_confidence"][occ]
    chosen_valid = (g["prob_object_id"][occ] != -1) & (g["prob_class_id"][occ] != -1)
    assert np.allclose(conf[unique & chosen_valid], soft[unique & chosen_valid], rtol=2e-6, atol=1e-7)
    assert np.all(conf[~chosen_valid] == 0.0) and valid.any()


@needs_ref
@pytest.mark.parametrize("tag", ["vote", "prob"])
def test_compiled_reference_reproduces_the_semantic_goldens(tag):
    """The committed dumps are exactly what the compiled reference produces from the committed inputs (so the GPU
    tests that compare against the .npz compare against the reference itself)."""
    from tests._util import sort_dump
    g = np.load(os.path.join(GOLDEN, "semantic_T0.npz"))
    kind = "voting" if tag == "vote" else "probabilistic"
    r = oracle.RefSemanticGrid(float(g["voxel_size"]), kind)
    r.set_depth_threshold(float(g[f"{tag}_depth_threshold"]))
    if kind == "probabilistic":
        r.set_depth_decay_rate(float(g[f"{tag}_depth_decay_rate"]))
    for i in range(int(g["n_frames"])):
        r.integrate(*[g[f"{tag}_{n}_{i}"] for n in ("points", "colors", "cls", "inst", "depths")])
    d = sort_dump(r.dump_blocks(8))
    for k in ("keys", "hashes", "count", "pos_sum", "col_sum", "object_id", "class_id", "confidence", "aux",
              "lab_obj", "lab_cls", "lab_logp"):
        assert np.array_equal(d[k], g[f"{tag}_{k}"]), k
    # the association replay: same maps, same allocator end value
    a = np.load(os.path.join(GOLDEN, "semantic_assoc_T0.npz"))
    from pyslam_b200 import remap_instance_ids
    from pyslam_b200 import synthetic as S
    oracle.RefSemanticGrid.set_next_object_id(1)
    r2 = oracle.RefSemanticGrid(float(a["voxel_size"]), kind)
    r2.set_depth_threshold(10.0)
    K = a["K"]
    for i in range(int(a["n_frames"])):
        dep, col, T = a[f"depth_{i}"], a[f"color_{i}"], a[f"Tcw_{i}"]
        cls_img, inst_img = a[f"class_image_{i}"], a[f"instance_image_{i}"]
        m = r2.assign_object_ids_to_instance_ids(np.array(K, np.float32), dep.shape[1], dep.shape[0], T,
                                                 float(a["param_depth_max"]), float(a["param_depth_min"]), cls_img,
                                                 inst_img, dep, float(a["param_depth_threshold"]),
                                                 bool(a["param_do_carving"]), float(a["param_min_vote_ratio"]),
                                                 int(a["param_min_votes"]))
        assert m == dict(zip(a[f"{tag}_map_inst_{i}"].tolist(), a[f"{tag}_map_obj_{i}"].tolist()))
        Twc = S.inv_T(T)
        valid = (dep > 0) & (dep < float(a["max_depth"]))
        z = dep[valid].astype(np.float64)
        rows, cols = np.where(valid)
        x, y = (cols - K[2]) * z * (1.0 / K[0]), (rows - K[3]) * z * (1.0 / K[1])
        pw = np.stack([x * Twc[q, 0] + y * Twc[q, 1] + z * Twc[q, 2] + Twc[q, 3] for q in range(3)],
                      axis=1).astype(np.float32)
        obj_img = remap_instance_ids(inst_img, m)
        r2.integrate(pw, (col[valid] / 255.0).astype(np.float32), cls_img[valid], obj_img[valid], dep[valid])
    assert oracle.RefSemanticGrid.get_next_object_id() == int(a[f"{tag}_next_object_id"])
    d2 = sort_dump(r2.dump_blocks(1))
    assert np.array_equal(d2["count"], a[f"{tag}_count"]) and np.array_equal(d2["object_id"], a[f"{tag}_object_id"])


def _quat_matrix(q):
    """Rotation matrix of a unit quaternion (w, x, y, z)."""
    w, x, y, z = q
    return np.array([[1 - 2 * (y * y + z * z), 2 * (x * y - z * w), 2 * (x * z + y * w)],
                     [2 * (x * y + z * w), 1 - 2 * (x * x + z * z), 2 * (y * z - x * w)],
                     [2 * (x * z - y * w), 2 * (y * z + x * w), 1 - 2 * (x * x + y * y)]])


@needs_ref
@pytest.mark.parametrize("kind", ["voting", "probabilistic"])
def test_compiled_reference_reproduces_the_segment_goldens(kind):
    """tests/golden/segments_T0.npz against the segments and PCA boxes (bounding_boxes_3d.cpp:373-556) of the
    compiled reference fed the same stream, at the tolerances of the segment tests that compare against the file."""
    from tests._util import SEGMENT_QUERIES, feed_segment_blobs, golden_segments, segment_blobs
    g = np.load(os.path.join(GOLDEN, "segments_T0.npz"))
    r = oracle.RefSemanticGrid(float(g["voxel_size"]), kind)
    feed_segment_blobs(r, segment_blobs(np.random.default_rng(3), 3000))
    for q, (by_class, min_count, min_conf) in enumerate(SEGMENT_QUERIES):
        ref = {t["id"]: t for t in (r.get_class_segments if by_class else r.get_object_segments)(min_count, min_conf)}
        gold = golden_segments(g, "vote" if kind == "voting" else "prob", q)
        assert sorted(ref) == sorted(s["id"] for s in gold)
        for s in gold:
            t = ref[s["id"]]
            oa, ob = np.lexsort(s["points"].T[::-1]), np.lexsort(t["points"].T[::-1])
            assert np.array_equal(s["points"][oa], t["points"][ob])
            assert np.allclose(s["colors"][oa], t["colors"][ob], rtol=0, atol=1e-6)
            assert abs(s["confidence_min"] - t["confidence_min"]) < 1e-5
            assert abs(s["confidence_max"] - t["confidence_max"]) < 1e-5
            if not by_class:
                assert s["class_id"] == t["class_id"]
                assert np.abs(s["obb_center"] - t["obb_center"]).max() < 1e-9
                assert np.abs(s["obb_size"] - t["obb_size"]).max() < 1e-9
                Rs, Rt = _quat_matrix(s["obb_quat_wxyz"]), _quat_matrix(t["obb_quat_wxyz"])
                assert np.abs(np.abs(np.sum(Rs * Rt, axis=0)) - 1.0).max() < 1e-9     # same axes, sign aside


def test_pca_oriented_box_equals_the_compiled_reference():
    """The product's OrientedBoundingBox3D.compute_from_points (numpy) on the object segments of
    tests/golden/segments_T0.npz: centre and size to 1e-9 and the axes (up to the eigenvector sign the eigen-solver
    happens to return) against the stored boxes, which test_compiled_reference_reproduces_the_segment_goldens
    compares with the boxes the UNMODIFIED reference attaches to its segments (bounding_boxes_3d.cpp:373-556 via
    voxel_block_semantic_grid.hpp:248-252).  Independently of any stored box: a right-handed frame whose axes carry
    descending variance, extents that just enclose the points, and the quaternion of that frame (w, x, y, z) as
    scipy converts it."""
    from scipy.spatial.transform import Rotation

    from pyslam_b200.volume import OrientedBoundingBox3D
    from tests._util import golden_segments
    segs = golden_segments(np.load(os.path.join(GOLDEN, "segments_T0.npz")), "vote", 0)
    assert sorted(s["id"] for s in segs) == [1, 2, 3]
    for s in segs:
        P = s["points"]
        b = OrientedBoundingBox3D.compute_from_points(P)
        assert np.abs(b.center - s["obb_center"]).max() < 1e-9 and np.abs(b.size - s["obb_size"]).max() < 1e-9
        Rr = _quat_matrix(s["obb_quat_wxyz"])
        assert np.abs(np.abs(np.sum(b.R * Rr, axis=0)) - 1.0).max() < 1e-9     # same axes, sign aside
        assert s["class_id"] == s["id"] + 10 and len(P) > 1000
        assert np.abs(b.R.T @ b.R - np.eye(3)).max() < 1e-12 and abs(np.linalg.det(b.R) - 1.0) < 1e-12
        var = ((P - P.mean(axis=0)) @ b.R).var(axis=0)
        assert var[0] > var[1] > var[2]
        assert np.abs(np.abs((P - b.center) @ b.R).max(axis=0) - b.size / 2).max() < 1e-9
        x, y, z, w = Rotation.from_matrix(b.R).as_quat()
        qs = np.array([w, x, y, z])
        assert min(np.abs(b.orientation - qs).max(), np.abs(b.orientation + qs).max()) < 1e-9
    # degenerate inputs
    assert np.array_equal(OrientedBoundingBox3D.compute_from_points(np.zeros((0, 3))).size, np.zeros(3))
    b1 = OrientedBoundingBox3D.compute_from_points([[1.0, 2.0, 3.0]])
    assert np.array_equal(b1.center, [1.0, 2.0, 3.0]) and np.array_equal(b1.size, np.zeros(3))
    b2 = OrientedBoundingBox3D.compute_from_points([[0.0, 0, 0], [2.0, 0, 0]])
    assert np.allclose(b2.center, [1.0, 0, 0]) and np.allclose(b2.size, [2.0, 0, 0])
