"""GPU: mesh and point-cloud extraction (pyslam_b200/csrc/b2v_mesh.cu) against the Open3D-order restatement of
ScalableTSDFVolume::ExtractTriangleMesh and ::ExtractPointCloud (oracle/open3d_order.c).

The restatement is seeded with the GPU volume's own `dump_blocks()` (or with the blocks uploaded to it), so both
sides extract from the same float32 voxels: mesh edges, triangles, vertices and colours, point positions and point
colours must then be equal bit for bit.  Integrated scenes are also compared end to end, with the restatement
integrating the same frames: there the only difference is Open3D's float64 colour mean, so colours get 1e-5 on the
0..1 scale.

The seeded volumes are built to reach what smooth scenes do not: every marching-cubes case, the per-block list
maxima of the emit kernels, special tsdf values (-0.0, +-0.98f, denormals, products that underflow), crossings that
only a neighbour block's sign summary reveals, far and negative block keys, and more tiles than the persistent grids
have CTAs.  tests/test_oracle_extraction.py pins the restatement's new code against numpy and the CPU twin."""

import os

import numpy as np
import pytest

import oracle
from pyslam_b200 import B200TsdfVolume
from pyslam_b200 import synthetic as S

pytestmark = pytest.mark.gpu

NT = max(1, min(len(os.sched_getaffinity(0)), 64))
VL, TAU = 0.013, 0.05      # voxel length / truncation of the seeded volumes (not a power of two: positions round)
_L = np.arange(512)
_LX, _LY, _LZ = _L % 8, (_L // 8) % 8, _L // 64
# the 7 neighbour offsets of a block's 2x2x2 tile, in the classify kernel's order (o & 1, o >> 1 & 1, o >> 2 & 1)
TILE_OFFSETS = [(o & 1, (o >> 1) & 1, (o >> 2) & 1) for o in range(1, 8)]


# ---- seeded volumes: (keys int32 [n,3], vox float32 [n,5,512]) --------------------------------------------------

def _voxel_coords(keys):
    """Global voxel coordinates [n,512] (int64) of every voxel of the blocks."""
    k = np.asarray(keys, np.int64).reshape(-1, 3)
    return k[:, :1] * 8 + _LX, k[:, 1:2] * 8 + _LY, k[:, 2:3] * 8 + _LZ


def _blocks(keys, tsdf, weight, rng):
    keys = np.asarray(keys, np.int32).reshape(-1, 3)
    vox = np.empty((len(keys), 5, 512), np.float32)
    vox[:, 0] = tsdf
    vox[:, 1] = weight
    vox[:, 2:] = rng.uniform(0.0, 255.0, (len(keys), 3, 512)).astype(np.float32)
    return keys, vox


def _sphere(keys, centre, radius, rng):
    """Signed distance to a sphere (voxel units, truncated at 3 voxels), float64 coordinates for far keys."""
    x, y, z = _voxel_coords(keys)
    d = np.sqrt(sum((g - c).astype(np.float64) ** 2 for g, c in zip((x, y, z), centre))) - radius
    t = np.clip(d / 3.0, -1.0, 1.0).astype(np.float32)
    return _blocks(keys, t, rng.integers(1, 30, t.shape).astype(np.float32), rng)


def _cube_keys(lo, side):
    g = np.stack(np.meshgrid(*[np.arange(side)] * 3, indexing="ij"), -1).reshape(-1, 3)
    return (g + np.asarray(lo)).astype(np.int32)


SPECIAL_TSDF = np.array([0.0, -0.0, 0.98, -0.98, np.nextafter(np.float32(0.98), np.float32(0)),
                         np.nextafter(np.float32(-0.98), np.float32(0)), 1.0, -1.0, 1e-40, -1e-40, 1e-30, -1e-30],
                        np.float32)


def random_volume(seed=1):
    """A 27^3-block region around the origin with ~40 % of its blocks removed (~11 800 left): tsdf uniform(-1, 1) with
    a quarter of the voxels replaced by SPECIAL_TSDF (+-0, +-0.98f and their inner neighbours, +-1, denormals, and
    +-1e-30 whose products underflow to -0), 15 % zero weights, colours uniform in [0, 255]."""
    rng = np.random.default_rng(seed)
    keys = _cube_keys((-13, -13, -13), 27)
    keys = keys[rng.random(len(keys)) >= 0.4]
    n = len(keys)
    t = rng.uniform(-1.0, 1.0, (n, 512)).astype(np.float32)
    pick = rng.random((n, 512)) < 0.25
    t[pick] = SPECIAL_TSDF[rng.integers(0, len(SPECIAL_TSDF), int(pick.sum()))]
    w = rng.integers(1, 100, (n, 512)).astype(np.float32)
    w[rng.random((n, 512)) < 0.15] = 0.0
    return _blocks(keys, t, w, rng)


def checkerboard_volume(seed=2):
    """4^3 blocks with tsdf +-0.5 by global voxel parity: every interior voxel owns 3 vertices and 3 points, every
    cube is case 0x5A or 0xA5 (4 triangles), so the 27 blocks with all 7 upper neighbours reach 1536 vertices and
    2048 triangles, the sizes of the emit kernels' shared-memory lists."""
    rng = np.random.default_rng(seed)
    keys = _cube_keys((3, -2, 5), 4)
    x, y, z = _voxel_coords(keys)
    t = np.where((x + y + z) % 2 == 0, 0.5, -0.5).astype(np.float32)
    return _blocks(keys, t, np.ones_like(t), rng)


def _layer(o, far):
    """Voxels [512] on the face / edge / corner of a block that touches its neighbour at +o (far=True) or at -o."""
    m = np.ones(512, bool)
    for a, l in enumerate((_LX, _LY, _LZ)):
        if o[a]:
            m &= l == (7 if far else 0)
    return m


def face_only_anchor(variant, j):
    """Key of block A of face_only_volume's pair for variant `variant` and tile offset TILE_OFFSETS[j]."""
    return np.array([4 * j - 9, 4 * variant - 5, -3])


def face_only_volume(seed=3, zero_weight=False):
    """For each of the 7 tile offsets o, a block A and its neighbour B = A + o, placed 4 blocks apart, plus every block
    A + s between them (s != 0, s != o, s <= o componentwise), filled with A's bulk sign.  Those fillers complete the
    cubes rooted in A that reach B across an edge or the corner; without them such cubes have unobserved corners.
      variant 0: A and the fillers all tsdf > 0, B < 0 only on the layer touching A: every crossing in A's tile lies
                 on B's layer, and only B's sign summary keeps the tile;
      variant 1: the mirror: B all > 0, A < 0 on the layer touching B;
      variant 2: variant 0 with every sign swapped.
    zero_weight=True: variant 0 only, with B's negative layer at weight 0, which must emit nothing."""
    rng = np.random.default_rng(seed)
    keys, tsdf, weight = [], [], []
    for variant in ((0,) if zero_weight else (0, 1, 2)):
        for j, o in enumerate(TILE_OFFSETS):
            a = face_only_anchor(variant, j)
            ta = rng.uniform(0.1, 0.9, 512)
            tb = rng.uniform(0.1, 0.9, 512)
            wa, wb = np.ones(512), np.ones(512)
            if variant == 1:
                ta[_layer(o, True)] *= -1
            else:
                tb[_layer(o, False)] *= -1
                if zero_weight:
                    wb[_layer(o, False)] = 0.0
            if variant == 2:
                ta, tb = -ta, -tb
            keys += [a, a + np.array(o)]
            tsdf += [ta, tb]
            weight += [wa, wb]
            for s in TILE_OFFSETS:
                if s != o and all(si <= oi for si, oi in zip(s, o)):
                    keys.append(a + np.array(s))
                    tsdf.append(rng.uniform(0.1, 0.9, 512) * (-1.0 if variant == 2 else 1.0))
                    weight.append(np.ones(512))
    return _blocks(keys, np.array(tsdf, np.float32), np.array(weight, np.float32), rng)


def topology_volume(seed=4):
    """An isolated block holding a closed sphere, and 8 copies of a 2x2x2 cluster cut by one sphere, each copy with
    another of its blocks removed; the clusters are 6 blocks apart."""
    rng = np.random.default_rng(seed)
    parts = [_sphere(np.array([[-7, 2, 1]]), (-7 * 8 + 4, 2 * 8 + 4, 1 * 8 + 4), 2.6, rng)]
    for j in range(8):
        lo = np.array([6 * j, -1, 2])
        keys = np.delete(_cube_keys(lo, 2), j, axis=0)
        parts.append(_sphere(keys, tuple(lo * 8 + 8), 5.3, rng))
    return np.concatenate([p[0] for p in parts]), np.concatenate([p[1] for p in parts])


def far_keys_volume(seed=5):
    """3^3-block clusters cut by a sphere around block keys (-1,-1,-1), (-2^20, 2^19, -3) and (2^20-1, 5, -2^19):
    negative keys split into units by a floor, and edge ids near +-2^23."""
    rng = np.random.default_rng(seed)
    parts = []
    for c in ((-1, -1, -1), (-(1 << 20), 1 << 19, -3), ((1 << 20) - 1, 5, -(1 << 19))):
        c = np.array(c, np.int64)
        parts.append(_sphere(_cube_keys(c - 1, 3), tuple(c * 8 + 4), 9.5, rng))
    return np.concatenate([p[0] for p in parts]), np.concatenate([p[1] for p in parts])


def all_positive_volume(seed=6):
    rng = np.random.default_rng(seed)
    keys = _cube_keys((-1, 0, 2), 3)
    t = rng.uniform(0.0, 1.0, (len(keys), 512)).astype(np.float32)
    return _blocks(keys, t, np.ones_like(t), rng)


def empty_volume():
    return np.zeros((0, 3), np.int32), np.zeros((0, 5, 512), np.float32)


SEEDED = {
    "random": random_volume,
    "checkerboard": checkerboard_volume,
    "face_only": face_only_volume,
    "face_only_zero_weight": lambda: face_only_volume(zero_weight=True),
    "topology": topology_volume,
    "far_keys": far_keys_volume,
    "all_positive": all_positive_volume,
    "empty": empty_volume,
}
EMPTY_OUTPUT = ("face_only_zero_weight", "all_positive", "empty")


# ---- comparison ----------------------------------------------------------------------------------------------

def seeded_restatement(keys, vox, R, vl=VL, tau=TAU):
    o3 = oracle.Open3DOrderVolume(vl, tau, R, 4)
    o3.set_blocks(keys, vox)
    return o3


def sort_points(points, colors):
    """Rows sorted by position, then colour (a degenerate weight ratio can put two points on one voxel centre)."""
    p, c = np.asarray(points), np.asarray(colors)
    order = np.lexsort((c[:, 2], c[:, 1], c[:, 0], p[:, 2], p[:, 1], p[:, 0]))
    return p[order], c[order]


def assert_same_mesh(m, ref, colour_tol=0.0):
    a = oracle.canonical_mesh(m.vertices, m.vertex_colors, m.edge_ids, m.triangles)
    b = oracle.canonical_mesh(ref["vertices"], ref["colors"], ref["edges"], ref["triangles"])
    assert m.vertices.shape == (len(ref["vertices"]), 3) and m.triangles.shape == (len(ref["triangles"]), 3)
    for name in ("edges", "triangles", "vertices"):
        assert np.array_equal(a[name], b[name]), name
    if colour_tol == 0.0:
        assert np.array_equal(a["colors"], b["colors"]), "colors"
    elif len(a["colors"]):
        assert np.abs(a["colors"] - b["colors"]).max() < colour_tol


def assert_same_points(pc, ref, colour_tol=0.0):
    assert pc.points.shape == ref["points"].shape and pc.colors.shape == ref["colors"].shape
    pa, ca = sort_points(pc.points, pc.colors)
    pb, cb = sort_points(ref["points"], ref["colors"])
    assert np.array_equal(pa, pb), "points"
    if colour_tol == 0.0:
        assert np.array_equal(ca, cb), "colors"
    elif len(ca):
        assert np.abs(ca - cb).max() < colour_tol


def check_stats(vol, mesh):
    st = vol.last_mesh_stats()
    assert st["blocks"] == vol.num_blocks()
    assert 0 <= st["vertex_blocks"] <= st["tiles_with_both_signs"] <= st["candidate_tiles"] <= st["blocks"]
    assert 0 <= st["triangle_blocks"] <= st["tiles_with_both_signs"]
    if not mesh:
        assert st["triangle_blocks"] == 0
    return st


def extract_both(vol):
    m = vol.extract_mesh()
    check_stats(vol, True)
    p = vol.extract_point_cloud()
    check_stats(vol, False)
    return m, p


def assert_matches_dump(vol, m=None, p=None):
    """Both extractions of `vol` equal, bit for bit, the restatement seeded with the volume's current blocks."""
    if m is None:
        m, p = extract_both(vol)
    d = vol.dump_blocks()
    o3 = seeded_restatement(d["keys"], d["vox"], vol.volume_unit_resolution, vol.voxel_length, vol.sdf_trunc)
    assert_same_mesh(m, o3.extract_triangle_mesh())
    assert_same_points(p, o3.extract_point_cloud())
    return m, p


def _volume(cfg_or_vl, tau=None, unit=16, capacity=1 << 16):
    if tau is None:
        cfg = cfg_or_vl
        return B200TsdfVolume(cfg.voxel_size, cfg.sdf_trunc, cfg.depth_trunc, capacity_blocks=capacity,
                              volume_unit_resolution=unit)
    return B200TsdfVolume(cfg_or_vl, tau, 4.0, capacity_blocks=capacity, volume_unit_resolution=unit)


# ---- a. integrated scenes --------------------------------------------------------------------------------------

@pytest.mark.parametrize("cfg_name,frames,unit", [
    ("T0", [0, 1, 2, 3], 16),
    ("T0", [0, 1, 2, 3], 8),
    ("C1", [0, 1, 2, 50], 16),
    ("C5", [0, 40], 16),                           # 10 cm voxels, width 1241
    ("C2", ([0, 1, 2, 3], [4, 5]), 16),            # a fused batch, then single frames
])
def test_integrated_scene_extractions_equal_open3d(cfg_name, frames, unit):
    cfg = S.CONFIGS[cfg_name]
    vol = _volume(cfg, unit=unit, capacity=1 << 17)
    batch, singles = frames if isinstance(frames, tuple) else ([], frames)
    rendered = {i: S.render_frame(cfg, i) for i in batch + singles}
    if batch:
        vol.integrate_batch(np.stack([rendered[i][0] for i in batch]), np.stack([rendered[i][1] for i in batch]),
                            cfg.K, np.stack([rendered[i][2] for i in batch]))
    for i in singles:
        vol.integrate(*rendered[i][:2], cfg.K, rendered[i][2])
    m, p = assert_matches_dump(vol)
    assert len(p.points) > 1000 and len(m.triangles) > 1000
    if unit != 16:
        return   # decision D1 allocates 8^3 units by pyslam's key rule, not by Open3D's LocateVolumeUnit
    o3 = oracle.Open3DOrderVolume(cfg.voxel_size, cfg.sdf_trunc, 16, 4)
    for i in batch + singles:
        d, c, T = rendered[i]
        o3.integrate(d, c, cfg.K, T, cfg.depth_trunc, nthreads=NT)
    assert_same_mesh(m, o3.extract_triangle_mesh(), colour_tol=1e-5)
    assert_same_points(p, o3.extract_point_cloud(), colour_tol=1e-5)


# ---- b. seeded worst-case volumes ------------------------------------------------------------------------------

@pytest.fixture(scope="module")
def seeded():
    return {name: make() for name, make in SEEDED.items()}


@pytest.mark.parametrize("unit", [8, 16])
@pytest.mark.parametrize("name", list(SEEDED))
def test_seeded_volume_extractions_equal_open3d(seeded, name, unit):
    keys, vox = seeded[name]
    vol = _volume(VL, TAU, unit=unit, capacity=1 << 15)
    vol.upload_blocks(keys, vox)
    assert vol.num_blocks() == len(keys)
    m, p = extract_both(vol)
    o3 = seeded_restatement(keys, vox, unit)
    assert_same_mesh(m, o3.extract_triangle_mesh())
    assert_same_points(p, o3.extract_point_cloud())
    st = check_stats(vol, False)
    if name in EMPTY_OUTPUT:
        for a in (m.vertices, m.vertex_colors, m.triangles, p.points, p.colors):
            assert a.shape == (0, 3)
        return
    assert len(m.triangles) > 0 and len(p.points) > 0
    if name == "random":
        # more work than the persistent grids have CTAs, and a two-level scan over more than 10 chunks
        assert st["blocks"] > 10 * 1024 and st["tiles_with_both_signs"] > 148 * 16
    if name == "checkerboard":
        owner = m.edge_ids[:, :3] // 8
        _, per_block = np.unique(owner, axis=0, return_counts=True)
        assert per_block.max() == 1536
        assert len(m.triangles) >= 27 * 2048
    # a second extraction of each kind is identical, array for array
    m2, p2 = extract_both(vol)
    for a, b in ((m.vertices, m2.vertices), (m.vertex_colors, m2.vertex_colors), (m.edge_ids, m2.edge_ids),
                 (m.triangles, m2.triangles), (p.points, p2.points), (p.colors, p2.colors)):
        assert np.array_equal(a, b)


# ---- c. sign summaries across every write path ----------------------------------------------------------------

def test_sign_summaries_follow_every_write_path():
    """PoolMeta::block_flags must cover the signs present after every path that writes voxels; a missing bit drops
    the tile, so the outputs lose triangles and points and differ from the restatement."""
    import torch
    cfg = S.CONFIGS["T0"]
    rng = np.random.default_rng(11)
    vol = _volume(cfg, capacity=1 << 14)
    # 1. upload: the blocks of frame 0 as the twin integrates them, every tsdf made non-negative, so a block's
    #    negative bit can only come from a later write
    twin = oracle.TsdfOracle(cfg.voxel_size, cfg.sdf_trunc, cfg.depth_trunc)
    d, c, T = S.render_frame(cfg, 0)
    twin.integrate(d, c, cfg.K, T)
    seed = twin.dump_blocks()
    seed["vox"][:, 0] = np.abs(seed["vox"][:, 0])
    vol.upload_blocks(seed["keys"], seed["vox"])
    m, p = assert_matches_dump(vol)
    assert len(m.triangles) == 0 and len(p.points) == 0
    # 2. the per-frame update kernel
    for i in (1, 2):
        d, c, T = S.render_frame(cfg, i)
        vol.integrate(d, c, cfg.K, T)
        assert_matches_dump(vol)
    # 3. the fused group kernel, then the same batch path unfused; frames far along the trajectory allocate blocks
    #    whose only flags come from these kernels
    for fuse, idx in ((True, [8, 9, 10, 11]), (False, [16, 17, 18])):
        fr = [S.render_frame(cfg, i) for i in idx]
        vol.set_fusion(fuse)
        vol.integrate_batch(np.stack([f[0] for f in fr]), np.stack([f[1] for f in fr]), cfg.K,
                            np.stack([f[2] for f in fr]))
        assert_matches_dump(vol)
    vol.set_fusion(True)
    # 4. re-upload blocks with their signs flipped: blocks that held only non-negative observed voxels now hold only
    #    negative ones, and some mixed blocks; the upload must recompute their summaries, so the flipped blocks get the
    #    negative bit (a summary that also kept the old bits would only be wider, which no output comparison can see)
    d = vol.dump_blocks()
    obs = d["vox"][:, 1] != 0
    neg = (obs & (d["vox"][:, 0] < 0)).any(axis=1)
    pos = (obs & ~(d["vox"][:, 0] < 0)).any(axis=1)
    only_pos = np.flatnonzero(pos & ~neg & (obs.sum(axis=1) > 64))
    mixed = np.flatnonzero(pos & neg)
    pick = np.concatenate([rng.choice(only_pos, min(24, len(only_pos)), replace=False),
                           rng.choice(mixed, min(8, len(mixed)), replace=False)])
    assert len(pick) > 16
    flipped = d["vox"][pick].copy()
    flipped[:, 0] = -flipped[:, 0]
    vol.upload_blocks(d["keys"][pick], flipped)
    m, p = assert_matches_dump(vol)
    # 5. device export / import into a second volume
    keys, vox = vol.export_blocks_torch()
    other = _volume(cfg, capacity=1 << 14)
    other.import_blocks_torch(keys, vox)
    m2, p2 = assert_matches_dump(other)
    assert_same_mesh(m2, dict(vertices=m.vertices, colors=m.vertex_colors, edges=m.edge_ids, triangles=m.triangles))
    assert_same_points(p2, dict(points=p.points, colors=p.colors))
    del keys, vox
    torch.cuda.synchronize()
    other.close()
    # 6. reset, then integrate again
    vol.reset()
    assert vol.num_blocks() == 0
    m, p = extract_both(vol)
    assert len(m.vertices) == 0 and len(p.points) == 0
    for i in (3, 4):
        d, c, T = S.render_frame(cfg, i)
        vol.integrate(d, c, cfg.K, T)
        m, p = assert_matches_dump(vol)
    assert len(p.points) > 100
    vol.close()


# ---- d. scratch shared by the two extractions ------------------------------------------------------------------

def test_alternating_extractions_while_the_volume_grows():
    """Mesh and point extraction share MeshBuffers (regrown by ensure_mesh_scratch): alternate them, grow the volume
    past twice its block count, alternate again; every result equals the restatement, repeats are identical."""
    cfg = S.CONFIGS["T0"]
    vol = _volume(cfg, capacity=1 << 14)
    d, c, T = S.render_frame(cfg, 0)
    vol.integrate(np.ascontiguousarray(d[:30, :40]), np.ascontiguousarray(c[:30, :40]), cfg.K, T)
    n0 = vol.num_blocks()
    assert n0 > 0
    m1 = vol.extract_mesh()
    check_stats(vol, True)
    p1 = vol.extract_point_cloud()
    check_stats(vol, False)
    m2 = vol.extract_mesh()
    check_stats(vol, True)
    assert_matches_dump(vol, m1, p1)
    for name in ("vertices", "vertex_colors", "edge_ids", "triangles"):
        assert np.array_equal(getattr(m1, name), getattr(m2, name)), name
    i = 1
    while vol.num_blocks() <= 2 * n0:
        d, c, T = S.render_frame(cfg, i)
        vol.integrate(d, c, cfg.K, T)
        i += 1
    p3 = vol.extract_point_cloud()
    check_stats(vol, False)
    m3 = vol.extract_mesh()
    check_stats(vol, True)
    p4 = vol.extract_point_cloud()
    check_stats(vol, False)
    assert_matches_dump(vol, m3, p3)
    assert np.array_equal(p3.points, p4.points) and np.array_equal(p3.colors, p4.colors)
    assert len(p3.points) > len(p1.points)
    vol.close()
