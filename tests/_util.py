"""Shared helpers for the parity tests."""

import os

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLDEN = os.path.join(ROOT, "tests", "golden")


def sort_dump(dump):
    """Order a block dump (keys [nb,3] + per-block arrays) by key so two dumps can be compared."""
    k = dump["keys"]
    order = np.lexsort((k[:, 2], k[:, 1], k[:, 0]))
    return {name: np.asarray(arr)[order] for name, arr in dump.items()}


def sorted_keys(keys):
    k = np.asarray(keys).reshape(-1, 3)
    return k[np.lexsort((k[:, 2], k[:, 1], k[:, 0]))]


def blocks_checksum(dump_sorted):
    """Order-independent integer checksum of a sorted dump's float planes (bit patterns)."""
    bits = np.ascontiguousarray(dump_sorted["vox"]).view(np.uint32).astype(np.uint64)
    per_block = bits.reshape(bits.shape[0], -1).sum(axis=1, dtype=np.uint64)
    return per_block


def segment_blobs(rng, n):
    """Three anisotropic Gaussian blobs (object ids 1..3, class id = object id + 10), n points each, with colours."""
    out = []
    for oid, (c, sc) in enumerate([((0, 0, 1), (0.5, 0.2, 0.1)), ((2, 1, 1), (0.1, 0.6, 0.3)), ((-1, 2, 0.5), (0.3, 0.3, 0.3))], 1):
        Q, _ = np.linalg.qr(rng.normal(size=(3, 3)))
        out.append((oid, oid + 10, (rng.normal(size=(n, 3)) * np.array(sc)) @ Q.T + np.array(c),
                    rng.random((n, 3)).astype(np.float32)))
    return out


def feed_segment_blobs(grid, blobs):
    """Each blob three times (the second time through integrate_segment), then a segment with a negative class id,
    which integrate_segment skips."""
    for rep in range(3):
        for oid, cid, p, col in blobs:
            if rep == 1:
                grid.integrate_segment(p, col, cid, oid)
            else:
                grid.integrate(p, col, np.full(len(p), cid, np.int32), np.full(len(p), oid, np.int32))
    grid.integrate_segment(blobs[0][2], blobs[0][3], -1, 5)


# get_object_segments / get_class_segments arguments of the segment parity tests and tests/golden/segments_T0.npz
SEGMENT_QUERIES = [(by_class, min_count, min_conf) for by_class in (False, True)
                   for min_count, min_conf in ((1, 0.0), (2, 0.5))]


def golden_segments(g, tag, query):
    """The segments stored for one kind ("vote" / "prob") and one SEGMENT_QUERIES index, as dicts shaped like
    oracle.RefSemanticGrid.get_object_segments' (obb_* only for object segments)."""
    member = g[f"{tag}_{query}_member"]
    out = []
    for k, seg_id in enumerate(g[f"{tag}_{query}_ids"]):
        s = dict(id=int(seg_id), points=g["points"][member == k], colors=g["colors"][member == k],
                 confidence_min=float(g[f"{tag}_{query}_conf_min"][k]),
                 confidence_max=float(g[f"{tag}_{query}_conf_max"][k]))
        if f"{tag}_{query}_obb" in g:
            obb = g[f"{tag}_{query}_obb"][k]
            s.update(class_id=int(g[f"{tag}_{query}_class_ids"][k]), obb_center=obb[0:3], obb_size=obb[3:6],
                     obb_quat_wxyz=obb[6:10])
        out.append(s)
    return out


def has_gpu() -> bool:
    try:
        import torch
        return torch.cuda.is_available()
    except Exception:
        return False
