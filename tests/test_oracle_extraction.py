"""CPU: the extraction side of the Open3D-order restatement (oracle/open3d_order.c) that tests/test_gpu_extraction.py
compares the kernels with.

- `extract_point_cloud` (ScalableTSDFVolume::ExtractPointCloud) equals an independent vectorised numpy restatement
  bit for bit, on the seeded worst-case volumes and on T0 frames the restatement integrates itself.
- `set_blocks` puts every voxel where the CPU twin's `set_block` does: the two meshes are equal bit for bit.
- The random seeded volume contains every one of the 254 non-trivial marching-cubes cases."""

import importlib.util
import os

import numpy as np
import pytest

import oracle
from pyslam_b200 import synthetic as S
from tests import test_gpu_extraction as gx
from tests._util import ROOT

f32 = np.float32
# marching-cubes corner order {000, 100, 110, 010, 001, 101, 111, 011} as (x, y, z) shifts
MC_CORNERS = [(0, 0, 0), (1, 0, 0), (1, 1, 0), (0, 1, 0), (0, 0, 1), (1, 0, 1), (1, 1, 1), (0, 1, 1)]


@pytest.fixture(scope="module")
def seeded():
    return {name: make() for name, make in gx.SEEDED.items()}


def _neighbour_index(keys, offset):
    """Row of the block at key + offset for every block, -1 where it is missing."""
    index = {k: i for i, k in enumerate(map(tuple, keys.tolist()))}
    return np.array([index.get((k[0] + offset[0], k[1] + offset[1], k[2] + offset[2]), -1)
                     for k in keys.tolist()], np.int64)


def _plus_one(a, nbr, axis):
    """a [n, ..., z, y, x]: the value at +1 along `axis` (-1 = x, -2 = y, -3 = z); the last layer comes from the
    first layer of the neighbour block, zero where that block is missing."""
    nxt = np.take(a, [0], axis=axis)[nbr]
    nxt[nbr < 0] = 0
    return np.concatenate([np.take(a, range(1, 8), axis=axis), nxt], axis=axis)


def numpy_point_cloud(keys, vox, voxel_length, R):
    """ExtractPointCloud per block and per axis in numpy: float32 tsdf / weight / colour and their arithmetic,
    float64 positions built unit-relative, no FMA."""
    keys = np.asarray(keys, np.int64).reshape(-1, 3)
    n = len(keys)
    f = np.asarray(vox[:, 0], np.float32).reshape(n, 8, 8, 8)          # [block, z, y, x]
    w = np.asarray(vox[:, 1], np.float32).reshape(n, 8, 8, 8)
    c = np.asarray(vox[:, 2:], np.float32).reshape(n, 3, 8, 8, 8)
    S_ = R // 8
    unit = keys // S_                                                     # floor, also for negative keys
    x_in_unit = [((keys[:, a] - unit[:, a] * S_) * 8)[:, None, None, None] + l for a, l in
                 enumerate((np.arange(8)[None, None, :], np.arange(8)[None, :, None], np.arange(8)[:, None, None]))]
    vl, half, L = float(voxel_length), float(voxel_length) * 0.5, float(voxel_length) * R
    p0 = [np.broadcast_to((half + vl * x_in_unit[a].astype(np.float64)) +
                          unit[:, a, None, None, None].astype(np.float64) * L, f.shape) for a in range(3)]
    ok0 = (w != 0) & (f < f32(0.98)) & (f >= f32(-0.98))
    r0 = np.abs(f)
    points, colors = [], []
    for a in range(3):
        e = [0, 0, 0]
        e[a] = 1
        nbr = _neighbour_index(keys, e)
        f1, w1 = _plus_one(f, nbr, -1 - a), _plus_one(w, nbr, -1 - a)
        c1 = _plus_one(c, nbr, -1 - a)
        with np.errstate(under="ignore"):
            q = ok0 & (w1 != 0) & (f1 < f32(0.98)) & (f1 >= f32(-0.98)) & (f * f1 < f32(0))
        r1 = np.abs(f1)
        rs = r0 + r1                          # 0 only where q is false
        p = [p0[k][q] for k in range(3)]
        p[a] = (p0[a][q] * r1[q].astype(np.float64) + (p0[a][q] + vl) * r0[q].astype(np.float64)) / \
            rs[q].astype(np.float64)
        points.append(np.stack(p, axis=1))
        with np.errstate(invalid="ignore"):
            col = (c * r1[:, None] + c1 * r0[:, None]) / rs[:, None] / f32(255.0)
        assert col.dtype == np.float32
        colors.append(np.moveaxis(col, 1, -1)[q].astype(np.float64))
    return np.concatenate(points), np.concatenate(colors)


def _assert_points_equal(ref, keys, vox, voxel_length, R):
    pa, ca = gx.sort_points(ref["points"], ref["colors"])
    pb, cb = gx.sort_points(*numpy_point_cloud(keys, vox, voxel_length, R))
    assert pa.shape == pb.shape
    assert np.array_equal(pa, pb), "points"
    assert np.array_equal(ca, cb), "colors"
    return len(pa)


@pytest.mark.parametrize("R", [8, 16])
@pytest.mark.parametrize("name", list(gx.SEEDED))
def test_point_cloud_restatement_equals_numpy_on_seeded_volumes(seeded, name, R):
    keys, vox = seeded[name]
    o3 = gx.seeded_restatement(keys, vox, R)
    n = _assert_points_equal(o3.extract_point_cloud(), keys, vox, gx.VL, R)
    assert (n == 0) == (name in gx.EMPTY_OUTPUT)


@pytest.mark.parametrize("R", [8, 16])
def test_point_cloud_restatement_equals_numpy_on_integrated_frames(R):
    cfg = S.CONFIGS["T0"]
    o3 = oracle.Open3DOrderVolume(cfg.voxel_size, cfg.sdf_trunc, R, 4)
    for i in range(4):
        d, c, T = S.render_frame(cfg, i)
        o3.integrate(d, c, cfg.K, T, cfg.depth_trunc, nthreads=4)
    dump = o3.dump_blocks()     # float64 planes; tsdf and weight are float32 values, colour Open3D's float64 mean
    assert _assert_points_equal(o3.extract_point_cloud(), dump["keys"], dump["vox"], cfg.voxel_size, R) > 1000


@pytest.mark.parametrize("name", list(gx.SEEDED))
def test_set_blocks_mesh_equals_the_twins(seeded, name):
    keys, vox = seeded[name]
    twin = oracle.TsdfOracle(gx.VL, gx.TAU, 4.0)
    for k, v in zip(keys, vox):
        twin.set_block(k, v)
    b = twin.extract_mesh()
    cb = oracle.canonical_mesh(b["vertices"], b["colors"], b["edges"], b["triangles"])
    for R in (8, 16):
        a = gx.seeded_restatement(keys, vox, R).extract_triangle_mesh()
        ca = oracle.canonical_mesh(a["vertices"], a["colors"], a["edges"], a["triangles"])
        for part in ("edges", "triangles", "vertices", "colors"):
            assert np.array_equal(ca[part], cb[part]), (R, part)
    assert (len(cb["triangles"]) == 0) == (name in gx.EMPTY_OUTPUT)


def cube_case_grid(keys, vox):
    """Marching-cubes case [n, z, y, x] of the cube rooted at every voxel, from the blocks' 9^3 tiles, and whether its
    8 corners are all observed (w != 0)."""
    keys = np.asarray(keys, np.int64)
    n = len(keys)
    f = np.asarray(vox[:, 0], np.float32).reshape(n, 8, 8, 8)
    w = np.asarray(vox[:, 1], np.float32).reshape(n, 8, 8, 8)
    tf, tw = np.zeros((n, 9, 9, 9), np.float32), np.zeros((n, 9, 9, 9), np.float32)
    for o in range(8):
        dx, dy, dz = o & 1, (o >> 1) & 1, (o >> 2) & 1
        nbr = np.arange(n) if o == 0 else _neighbour_index(keys, (dx, dy, dz))
        have = nbr >= 0
        dst = (have,) + tuple(slice(8, 9) if d else slice(0, 8) for d in (dz, dy, dx))
        src = tuple(slice(0, 1) if d else slice(0, 8) for d in (dz, dy, dx))
        tf[dst] = f[nbr[have]][(slice(None),) + src]
        tw[dst] = w[nbr[have]][(slice(None),) + src]
    case = np.zeros((n, 8, 8, 8), np.int32)
    observed = np.ones((n, 8, 8, 8), bool)
    for i, (sx, sy, sz) in enumerate(MC_CORNERS):
        corner = (slice(None), slice(sz, sz + 8), slice(sy, sy + 8), slice(sx, sx + 8))
        case |= (tf[corner] < 0).astype(np.int32) << i
        observed &= tw[corner] != 0
    return case, observed


def cube_cases(keys, vox):
    """Marching-cubes case of every cube whose 8 corners are observed."""
    case, observed = cube_case_grid(keys, vox)
    return case[observed]


def test_face_only_crossings_are_seen_only_through_the_neighbour(seeded):
    """In variants 0 and 2 of the face-only volume, block A holds one sign only, and so does every other block of its
    2x2x2 tile except B = A + o.  Yet for each of the 7 offsets o, cubes rooted in A emit triangles.  So the tile is
    kept only if the filter ORs B's sign summary, whichever of the 7 neighbours B is."""
    keys, vox = seeded["face_only"]
    case, observed = cube_case_grid(keys, vox)
    row = {k: i for i, k in enumerate(map(tuple, keys.tolist()))}
    obs = vox[:, 1] != 0
    neg = (obs & (vox[:, 0] < 0)).any(axis=1)
    pos = (obs & ~(vox[:, 0] < 0)).any(axis=1)
    for variant in (0, 2):
        for j, o in enumerate(gx.TILE_OFFSETS):
            a = gx.face_only_anchor(variant, j)
            tile = [row.get(tuple(int(v) for v in a + np.array(s))) for s in [(0, 0, 0)] + gx.TILE_OFFSETS]
            b = row[tuple(int(v) for v in a + np.array(o))]
            assert neg[b] and pos[b]
            for r in tile:
                if r is not None and r != b:
                    assert neg[r] != pos[r] and neg[r] == (variant == 2)
            c = case[tile[0]][observed[tile[0]]]
            assert ((c != 0) & (c != 255)).sum() > 0, (variant, o)


def test_random_volume_covers_every_cube_case(seeded):
    keys, vox = seeded["random"]
    cases = np.unique(cube_cases(keys, vox))
    assert set(range(1, 255)) <= set(cases.tolist())
    # and the restatement meshes them: its triangle count is the table's count summed over those cubes
    mesh = gx.seeded_restatement(keys, vox, 8).extract_triangle_mesh()
    num_tris = np.array(_mc_tables().num_tris_table())
    assert len(mesh["triangles"]) == int(num_tris[cube_cases(keys, vox)].sum())


def _mc_tables():
    spec = importlib.util.spec_from_file_location("mc_tables", os.path.join(ROOT, "tools", "mc_tables.py"))
    m = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(m)
    return m

