"""Golden segments of the semantic grids (get_object_segments / get_class_segments with their PCA boxes), for the
segment tests in tests/test_gpu_semantic.py and tests/test_oracle_semantic.py:
    python tests/golden/make_golden_segments.py [out.npz]

The segments come from the UNMODIFIED compiled reference (oracle.RefSemanticGrid) when oracle/_ref is built, and
otherwise from this project's GPU grids; `source` in the file says which.  The committed file has source "pyslam_b200":
it was recorded where the pySLAM sources were not available.  Where they are,
test_oracle_semantic.py::test_compiled_reference_reproduces_the_segment_goldens compares it with the reference.

segments_T0.npz  the stream of tests/_util.feed_segment_blobs (three blobs of 3000 points, default_rng(3)) into
                 VoxelBlockSemanticGrid ("vote") and VoxelBlockSemanticProbabilisticGrid ("prob") at 5 cm voxels.
                 points float64 [n,3] / colors [n,3]: every voxel of the object segments (1, 0.0) of "vote", sorted;
                 both kinds hold the same voxels.  For each kind and each query q of tests/_util.SEGMENT_QUERIES:
                 {kind}_{q}_ids, _conf_min, _conf_max per segment; _member int8 [n] = the segment each voxel belongs
                 to (-1: none); for object queries also _class_ids and _obb [k,10] = centre, size, quaternion wxyz."""
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)

import oracle  # noqa: E402
from tests._util import GOLDEN, SEGMENT_QUERIES, feed_segment_blobs, segment_blobs  # noqa: E402

VOXEL = 0.05


def reference_segments(kind):
    """kind -> query -> segment dicts, from the compiled reference."""
    g = oracle.RefSemanticGrid(VOXEL, kind)
    feed_segment_blobs(g, segment_blobs(np.random.default_rng(3), 3000))
    return [(g.get_class_segments if by_class else g.get_object_segments)(min_count, min_conf)
            for by_class, min_count, min_conf in SEGMENT_QUERIES]


def product_segments(kind):
    """The same from this project's GPU grids, in the reference's dict form."""
    from pyslam_b200 import VoxelBlockSemanticGrid, VoxelBlockSemanticProbabilisticGrid
    cls_t = VoxelBlockSemanticGrid if kind == "voting" else VoxelBlockSemanticProbabilisticGrid
    g = cls_t(VOXEL, 8, capacity_blocks=1 << 13)
    feed_segment_blobs(g, segment_blobs(np.random.default_rng(3), 3000))
    out = []
    for by_class, min_count, min_conf in SEGMENT_QUERIES:
        grp = (g.get_class_segments if by_class else g.get_object_segments)(min_count, min_conf)
        segs = []
        for s in (grp.class_vector if by_class else grp.object_vector):
            d = dict(id=s.class_id if by_class else s.object_id, points=np.asarray(s.points),
                     colors=np.asarray(s.colors), confidence_min=s.confidence_min, confidence_max=s.confidence_max)
            if not by_class:
                b = s.oriented_bounding_box
                d.update(class_id=s.class_id, obb_center=b.center, obb_size=b.size, obb_quat_wxyz=b.orientation)
            segs.append(d)
        out.append(segs)
    g.close()
    return out


def main(path):
    source = "reference" if oracle.have_ref_semantic() else "pyslam_b200"
    out = dict(voxel_size=VOXEL, source=source)
    row_of = None
    for tag, kind in (("vote", "voting"), ("prob", "probabilistic")):
        per_query = reference_segments(kind) if source == "reference" else product_segments(kind)
        for q, segs in enumerate(per_query):
            if row_of is None:   # the voxel table: "vote", object segments (1, 0.0)
                pts = np.concatenate([s["points"] for s in segs])
                cols = np.concatenate([s["colors"] for s in segs])
                order = np.lexsort(pts.T[::-1])
                out["points"], out["colors"] = pts[order], cols[order]
                row_of = {p.tobytes(): i for i, p in enumerate(out["points"])}
                assert len(row_of) == len(pts)
            member = np.full(len(out["points"]), -1, np.int8)
            for k, s in enumerate(segs):
                rows = np.array([row_of[p.tobytes()] for p in s["points"]], np.int64)
                assert np.array_equal(out["colors"][rows], s["colors"]) and (member[rows] == -1).all()
                member[rows] = k
            out[f"{tag}_{q}_member"] = member
            out[f"{tag}_{q}_ids"] = np.array([s["id"] for s in segs], np.int32)
            out[f"{tag}_{q}_conf_min"] = np.array([s["confidence_min"] for s in segs], np.float64)
            out[f"{tag}_{q}_conf_max"] = np.array([s["confidence_max"] for s in segs], np.float64)
            if not SEGMENT_QUERIES[q][0]:
                out[f"{tag}_{q}_class_ids"] = np.array([s["class_id"] for s in segs], np.int32)
                out[f"{tag}_{q}_obb"] = np.array([np.concatenate([s["obb_center"], s["obb_size"], s["obb_quat_wxyz"]])
                                                  for s in segs])
            print(tag, q, "segments", len(segs), "voxels", int((member >= 0).sum()))
    np.savez_compressed(path, **out)
    print("source", source, "size", os.path.getsize(path))


if __name__ == "__main__":
    main(sys.argv[1] if len(sys.argv) > 1 else os.path.join(GOLDEN, "segments_T0.npz"))
