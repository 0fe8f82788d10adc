"""TEST INFRASTRUCTURE ONLY: ctypes front-ends for the oracle libraries + numpy cross-checks."""

from __future__ import annotations

import ctypes as C
import os
import subprocess

import numpy as np

_DIR = os.path.dirname(os.path.abspath(__file__))
_TSDF_SO = os.path.join(_DIR, "liboracle_tsdf.so")
_REF_SO = os.path.join(_DIR, "_ref", "libref_grid.so")

_f32p = np.ctypeslib.ndpointer(np.float32, flags="C_CONTIGUOUS")
_f64p = np.ctypeslib.ndpointer(np.float64, flags="C_CONTIGUOUS")
_u8p = np.ctypeslib.ndpointer(np.uint8, flags="C_CONTIGUOUS")
_i32p = np.ctypeslib.ndpointer(np.int32, flags="C_CONTIGUOUS")
_u64p = np.ctypeslib.ndpointer(np.uint64, flags="C_CONTIGUOUS")


def build(quiet: bool = True) -> None:
    """Compile the oracle libraries (the C restatement always; `_ref` when /root/reference exists)."""
    subprocess.run(["make", "-C", _DIR, "all"], check=True,
                   stdout=subprocess.DEVNULL if quiet else None)


def have_ref() -> bool:
    return os.path.exists(_REF_SO)


_tsdf_lib = None
_ref_lib = None


def _tsdf():
    global _tsdf_lib
    if _tsdf_lib is None:
        if not os.path.exists(_TSDF_SO):
            build()
        L = C.CDLL(_TSDF_SO)
        L.tsdf_oracle_create.restype = C.c_void_p
        L.tsdf_oracle_create.argtypes = [C.c_float, C.c_int, C.c_float, C.c_float, C.c_int]
        L.tsdf_oracle_destroy.argtypes = [C.c_void_p]
        L.tsdf_oracle_reset.argtypes = [C.c_void_p]
        L.tsdf_oracle_num_blocks.restype = C.c_int64
        L.tsdf_oracle_num_blocks.argtypes = [C.c_void_p]
        L.tsdf_oracle_num_touched.restype = C.c_int64
        L.tsdf_oracle_num_touched.argtypes = [C.c_void_p]
        L.tsdf_oracle_integrate.restype = C.c_int64
        L.tsdf_oracle_integrate.argtypes = [C.c_void_p, _f32p, _u8p, C.c_int, C.c_int, _f64p, _f64p,
                                            C.c_int]
        L.tsdf_oracle_last_touched.restype = C.c_int64
        L.tsdf_oracle_last_touched.argtypes = [C.c_void_p, _i32p]
        L.tsdf_oracle_dump.restype = C.c_int64
        L.tsdf_oracle_dump.argtypes = [C.c_void_p, _i32p, _u64p, _f32p]
        L.tsdf_oracle_extract_mesh.argtypes = [C.c_void_p, C.POINTER(C.c_int64), C.POINTER(C.c_int64)]
        L.tsdf_oracle_mesh_copy.argtypes = [_f64p, _f64p, _i32p, _i32p]
        L.tsdf_oracle_block_key_hash.restype = C.c_uint64
        L.tsdf_oracle_block_key_hash.argtypes = [C.c_int32] * 3
        L.tsdf_oracle_floor_div.restype = C.c_int64
        L.tsdf_oracle_floor_div.argtypes = [C.c_int64, C.c_int64]
        L.tsdf_oracle_voxel_coord.restype = C.c_int32
        L.tsdf_oracle_voxel_coord.argtypes = [C.c_float, C.c_float]
        L.tsdf_oracle_max_threads.restype = C.c_int
        L.tsdf_oracle_set_block.argtypes = [C.c_void_p, C.c_int32, C.c_int32, C.c_int32, _f32p]
        L.tsdf_oracle_set_units.argtypes = [C.c_void_p, C.c_int, C.c_double, C.c_double]
        _tsdf_lib = L
    return _tsdf_lib


def _ref():
    global _ref_lib
    if _ref_lib is None:
        if not have_ref():
            raise RuntimeError("oracle/_ref/libref_grid.so missing (needs /root/reference to build)")
        L = C.CDLL(_REF_SO)
        L.refgrid_create.restype = C.c_void_p
        L.refgrid_create.argtypes = [C.c_float, C.c_int]
        L.refgrid_destroy.argtypes = [C.c_void_p]
        L.refgrid_clear.argtypes = [C.c_void_p]
        L.refgrid_integrate.restype = C.c_double
        L.refgrid_integrate.argtypes = [C.c_void_p, _f32p, C.c_void_p, C.c_int64]
        L.refgrid_integrate_f64.restype = C.c_double
        L.refgrid_integrate_f64.argtypes = [C.c_void_p, _f64p, C.c_void_p, C.c_int64]
        L.refgrid_num_blocks.restype = C.c_int64
        L.refgrid_num_blocks.argtypes = [C.c_void_p]
        L.refgrid_block_size.argtypes = [C.c_void_p]
        L.refgrid_inv_voxel_size.restype = C.c_float
        L.refgrid_inv_voxel_size.argtypes = [C.c_void_p]
        L.refgrid_dump_blocks.restype = C.c_int64
        L.refgrid_dump_blocks.argtypes = [C.c_void_p] * 6
        L.refgrid_get_voxels.restype = C.c_int64
        L.refgrid_get_voxels.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p,
                                         C.POINTER(C.c_double)]
        L.refgrid_remove_low_count_voxels.argtypes = [C.c_void_p, C.c_int]
        L.refgrid_carve.argtypes = [C.c_void_p, C.c_float, C.c_float, C.c_float, C.c_float, C.c_int,
                                    C.c_int, _f64p, C.c_float, C.c_float, _f32p, C.c_float]
        L.refgrid_get_voxels_in_frustum.restype = C.c_int64
        L.refgrid_get_voxels_in_frustum.argtypes = [C.c_void_p, C.c_float, C.c_float, C.c_float, C.c_float,
                                                    C.c_int, C.c_int, _f64p, C.c_float, C.c_float, C.c_int,
                                                    C.c_void_p, C.c_void_p]
        L.refgrid_get_voxels_in_bb.restype = C.c_int64
        L.refgrid_get_voxels_in_bb.argtypes = [C.c_void_p, _f64p, C.c_int, C.c_void_p, C.c_void_p]
        L.ref_voxel_key_inv.argtypes = [C.c_float] * 4 + [_i32p]
        L.ref_floor_div.restype = C.c_int64
        L.ref_floor_div.argtypes = [C.c_int64, C.c_int64]
        L.ref_block_and_local_key.argtypes = [_i32p, C.c_int, _i32p, _i32p]
        L.ref_block_key_hash.restype = C.c_uint64
        L.ref_block_key_hash.argtypes = [C.c_int32] * 3
        L.ref_sizeof_voxel_data.restype = C.c_int
        _ref_lib = L
    return _ref_lib


# ---------------------------------------------------------------------------------------------
# compiled reference
# ---------------------------------------------------------------------------------------------

def ref_block_key_hash(x, y, z) -> int:
    return int(_ref().ref_block_key_hash(int(x), int(y), int(z)))


def ref_floor_div(a, b) -> int:
    return int(_ref().ref_floor_div(int(a), int(b)))


def ref_keys(point, voxel_size, block_size=8):
    """(voxel key, block key, local key) of one point exactly as the reference computes them."""
    L = _ref()
    inv = np.float32(1.0) / np.float32(voxel_size)
    vk = np.zeros(3, np.int32)
    L.ref_voxel_key_inv(float(np.float32(point[0])), float(np.float32(point[1])),
                        float(np.float32(point[2])), float(inv), vk)
    bk, lk = np.zeros(3, np.int32), np.zeros(3, np.int32)
    L.ref_block_and_local_key(vk, int(block_size), bk, lk)
    return vk, bk, lk


class RefGrid:
    """The unmodified reference `volumetric::VoxelBlockGrid` (sequential branch)."""

    def __init__(self, voxel_size: float, block_size: int = 8):
        self._L = _ref()
        self._h = self._L.refgrid_create(float(voxel_size), int(block_size))
        self.block_size = block_size
        self.last_elapsed_s = 0.0

    def __del__(self):
        if getattr(self, "_h", None):
            self._L.refgrid_destroy(self._h)
            self._h = None

    def integrate(self, points, colors=None) -> float:
        f64 = np.asarray(points).dtype == np.float64        # the reference's float64-points overload
        pts = np.ascontiguousarray(points, dtype=np.float64 if f64 else np.float32)
        assert pts.ndim == 2 and pts.shape[1] == 3
        cp = None
        if colors is not None:
            cols = np.ascontiguousarray(colors, dtype=np.float32)
            assert cols.shape == pts.shape
            cp = cols.ctypes.data
        fn = self._L.refgrid_integrate_f64 if f64 else self._L.refgrid_integrate
        self.last_elapsed_s = fn(self._h, pts.reshape(-1) if f64 else pts, cp, pts.shape[0])
        return self.last_elapsed_s

    def num_blocks(self) -> int:
        return int(self._L.refgrid_num_blocks(self._h))

    def clear(self):
        self._L.refgrid_clear(self._h)

    def dump_blocks(self):
        nb = self.num_blocks()
        nv = self.block_size ** 3
        keys = np.zeros((nb, 3), np.int32)
        hashes = np.zeros(nb, np.uint64)
        count = np.zeros((nb, nv), np.int32)
        pos = np.zeros((nb, nv, 3), np.float32)
        col = np.zeros((nb, nv, 3), np.float32)
        self._L.refgrid_dump_blocks(self._h, keys.ctypes.data, hashes.ctypes.data, count.ctypes.data,
                                    pos.ctypes.data, col.ctypes.data)
        return dict(keys=keys, hashes=hashes, count=count, pos_sum=pos, col_sum=col)

    def get_voxels(self, min_count=1):
        el = C.c_double(0.0)
        n = self._L.refgrid_get_voxels(self._h, int(min_count), None, None, C.byref(el))
        pts = np.zeros((n, 3), np.float32)
        cols = np.zeros((n, 3), np.float32)
        if n:
            self._L.refgrid_get_voxels(self._h, int(min_count), pts.ctypes.data, cols.ctypes.data,
                                       C.byref(el))
        self.last_elapsed_s = el.value
        return pts, cols

    def remove_low_count_voxels(self, min_count):
        self._L.refgrid_remove_low_count_voxels(self._h, int(min_count))

    def get_voxels_in_frustum(self, K, width, height, Tcw, min_count=1, depth_max=10.0, depth_min=1e-2):
        T = np.ascontiguousarray(Tcw, np.float64).reshape(16)
        a = (self._h, K[0], K[1], K[2], K[3], int(width), int(height), T, depth_max, depth_min, int(min_count))
        n = self._L.refgrid_get_voxels_in_frustum(*a, None, None)
        pts, cols = np.zeros((n, 3), np.float32), np.zeros((n, 3), np.float32)
        if n:
            self._L.refgrid_get_voxels_in_frustum(*a, pts.ctypes.data, cols.ctypes.data)
        return pts, cols

    def get_voxels_in_bb(self, bbox, min_count=1):
        bb = np.ascontiguousarray(bbox, np.float64).reshape(6)
        n = self._L.refgrid_get_voxels_in_bb(self._h, bb, int(min_count), None, None)
        pts, cols = np.zeros((n, 3), np.float32), np.zeros((n, 3), np.float32)
        if n:
            self._L.refgrid_get_voxels_in_bb(self._h, bb, int(min_count), pts.ctypes.data, cols.ctypes.data)
        return pts, cols

    def carve(self, K, width, height, Tcw, depth, depth_threshold=1e-2, depth_max=10.0,
              depth_min=1e-2):
        d = np.ascontiguousarray(depth, np.float32)
        T = np.ascontiguousarray(Tcw, np.float64).reshape(16)
        self._L.refgrid_carve(self._h, K[0], K[1], K[2], K[3], int(width), int(height), T,
                              depth_max, depth_min, d, depth_threshold)


# ---------------------------------------------------------------------------------------------
# C restatement of the TSDF path
# ---------------------------------------------------------------------------------------------

class TsdfOracle:
    def __init__(self, voxel_size, sdf_trunc, depth_trunc, block_size=8, stride=4, unit_resolution=16):
        self._L = _tsdf()
        self.block_size = block_size
        self.nvox = block_size ** 3
        self._h = self._L.tsdf_oracle_create(float(np.float32(voxel_size)), int(block_size),
                                             float(np.float32(sdf_trunc)),
                                             float(np.float32(depth_trunc)), int(stride))
        self.set_units(unit_resolution, voxel_size, sdf_trunc)

    def __del__(self):
        if getattr(self, "_h", None):
            self._L.tsdf_oracle_destroy(self._h)
            self._h = None

    @staticmethod
    def max_threads() -> int:
        return int(_tsdf().tsdf_oracle_max_threads())

    def reset(self):
        self._L.tsdf_oracle_reset(self._h)

    def set_units(self, unit_resolution, voxel_length, sdf_trunc):
        """Open3D volume-unit resolution: 16 = the reference's setting (allocation by LocateVolumeUnit), 8 = decision
        D1 (allocation by the float32 pyslam key range); voxel_length / sdf_trunc as the float64 values Open3D holds."""
        self._L.tsdf_oracle_set_units(self._h, int(unit_resolution), float(voxel_length), float(sdf_trunc))

    def integrate(self, depth, color, K, Tcw, nthreads=1) -> int:
        d = np.ascontiguousarray(depth, np.float32)
        c = np.ascontiguousarray(color, np.uint8)
        H, W = d.shape
        assert c.shape == (H, W, 3)
        return int(self._L.tsdf_oracle_integrate(self._h, d, c, H, W,
                                                 np.ascontiguousarray(K, np.float64).reshape(4),
                                                 np.ascontiguousarray(Tcw, np.float64).reshape(16),
                                                 int(nthreads)))

    def num_blocks(self) -> int:
        return int(self._L.tsdf_oracle_num_blocks(self._h))

    def set_block(self, key, vox):
        """test hook: overwrite / create one block with vox f32 [5, B^3]"""
        v = np.ascontiguousarray(vox, np.float32).reshape(5 * self.nvox)
        self._L.tsdf_oracle_set_block(self._h, int(key[0]), int(key[1]), int(key[2]), v)

    def last_touched(self):
        n = int(self._L.tsdf_oracle_num_touched(self._h))
        keys = np.zeros((n, 3), np.int32)
        self._L.tsdf_oracle_last_touched(self._h, keys)
        return keys

    def dump_blocks(self):
        nb = self.num_blocks()
        keys = np.zeros((nb, 3), np.int32)
        hashes = np.zeros(nb, np.uint64)
        vox = np.zeros((nb, 5, self.nvox), np.float32)
        self._L.tsdf_oracle_dump(self._h, keys, hashes, vox)
        return dict(keys=keys, hashes=hashes, vox=vox)

    def extract_mesh(self):
        nv, nt = C.c_int64(0), C.c_int64(0)
        self._L.tsdf_oracle_extract_mesh(self._h, C.byref(nv), C.byref(nt))
        V64 = np.zeros((nv.value, 3), np.float64)
        Cc = np.zeros((nv.value, 3), np.float64)
        E = np.zeros((nv.value, 4), np.int32)
        T = np.zeros((nt.value, 3), np.int32)
        self._L.tsdf_oracle_mesh_copy(V64.reshape(-1), Cc.reshape(-1), E.reshape(-1), T.reshape(-1))
        return dict(vertices=V64, colors=Cc, edges=E, triangles=T)


# ---------------------------------------------------------------------------------------------
# Open3D ScalableTSDFVolume in Open3D's own operation order (oracle/open3d_order.c)
# ---------------------------------------------------------------------------------------------
_O3D_SO = os.path.join(_DIR, "libopen3d_order.so")
_o3d_lib = None


def _o3d():
    global _o3d_lib
    if _o3d_lib is None:
        if not os.path.exists(_O3D_SO):
            build()
        L = C.CDLL(_O3D_SO)
        vp = C.c_void_p
        L.o3d_create.restype = vp
        L.o3d_create.argtypes = [C.c_double, C.c_double, C.c_int, C.c_int]
        L.o3d_destroy.argtypes = [vp]
        L.o3d_reset.argtypes = [vp]
        L.o3d_num_units.restype = C.c_int64
        L.o3d_num_units.argtypes = [vp]
        L.o3d_num_touched.restype = C.c_int64
        L.o3d_num_touched.argtypes = [vp]
        L.o3d_prepare_depth.argtypes = [_f32p, _f32p, C.c_int64, C.c_double, C.c_double]
        L.o3d_multiplier.argtypes = [_f32p, C.c_int, C.c_int, _f64p]
        L.o3d_integrate.restype = C.c_int64
        L.o3d_integrate.argtypes = [vp, _f32p, _u8p, _f32p, C.c_int, C.c_int, _f64p, _f64p, C.c_int]
        L.o3d_last_touched.restype = C.c_int64
        L.o3d_last_touched.argtypes = [vp, _i32p]
        L.o3d_dump_blocks.restype = C.c_int64
        L.o3d_dump_blocks.argtypes = [vp, vp, vp]
        L.o3d_extract_mesh.argtypes = [vp, C.POINTER(C.c_int64), C.POINTER(C.c_int64)]
        L.o3d_mesh_copy.argtypes = [_f64p, _f64p, _i32p, _i32p]
        L.o3d_set_block.argtypes = [vp, C.c_int32, C.c_int32, C.c_int32, _f32p]
        L.o3d_extract_point_cloud.argtypes = [vp, C.POINTER(C.c_int64)]
        L.o3d_points_copy.argtypes = [_f64p, _f64p]
        _o3d_lib = L
    return _o3d_lib


class Open3DOrderVolume:
    """`o3d.pipelines.integration.ScalableTSDFVolume(voxel_length, sdf_trunc, RGB8, volume_unit_resolution,
    depth_sampling_stride)` as the reference constructs it (volumetric_integrator_tsdf.py:104-108), restated in
    Open3D's own operation order and types.  `integrate` takes what the reference passes at tsdf.py:215-223:
    a float32 depth in metres (depth_scale 1.0), the depth truncation of create_from_color_and_depth, RGB u8,
    the intrinsics and the world->camera pose."""

    def __init__(self, voxel_length, sdf_trunc, volume_unit_resolution=16, depth_sampling_stride=4):
        self._L = _o3d()
        self.R = int(volume_unit_resolution)
        assert self.R % 8 == 0
        self._h = self._L.o3d_create(float(voxel_length), float(sdf_trunc), self.R, int(depth_sampling_stride))
        self._mult_key, self._mult = None, None

    def __del__(self):
        if getattr(self, "_h", None):
            self._L.o3d_destroy(self._h)
            self._h = None

    def reset(self):
        self._L.o3d_reset(self._h)

    def integrate(self, depth, color, K, Tcw, depth_trunc, depth_scale=1.0, nthreads=1) -> int:
        d_in = np.ascontiguousarray(depth, np.float32)
        c = np.ascontiguousarray(color, np.uint8)
        H, W = d_in.shape
        assert c.shape == (H, W, 3)
        d = np.empty_like(d_in)
        self._L.o3d_prepare_depth(d_in.reshape(-1), d.reshape(-1), d.size, float(depth_scale), float(depth_trunc))
        K4 = np.ascontiguousarray(K, np.float64).reshape(4)
        key = (H, W, tuple(K4))
        if self._mult_key != key:
            self._mult = np.zeros((H, W), np.float32)
            self._L.o3d_multiplier(self._mult.reshape(-1), H, W, K4)
            self._mult_key = key
        return int(self._L.o3d_integrate(self._h, d.reshape(-1), c.reshape(-1), self._mult.reshape(-1), H, W, K4,
                                         np.ascontiguousarray(Tcw, np.float64).reshape(16), int(nthreads)))

    def num_units(self) -> int:
        return int(self._L.o3d_num_units(self._h))

    def last_touched_units(self):
        n = int(self._L.o3d_num_touched(self._h))
        idx = np.zeros((n, 3), np.int32)
        self._L.o3d_last_touched(self._h, idx.reshape(-1))
        return idx

    def dump_blocks(self):
        """Every unit as (R/8)^3 blocks in the product's layout: keys int32 [nb,3], vox float64 [nb,5,512]."""
        nb = self.num_units() * (self.R // 8) ** 3
        keys = np.zeros((nb, 3), np.int32)
        vox = np.zeros((nb, 5, 512), np.float64)
        self._L.o3d_dump_blocks(self._h, keys.ctypes.data, vox.ctypes.data)
        return dict(keys=keys, vox=vox)

    def extract_triangle_mesh(self):
        nv, nt = C.c_int64(0), C.c_int64(0)
        self._L.o3d_extract_mesh(self._h, C.byref(nv), C.byref(nt))
        V = np.zeros((nv.value, 3), np.float64)
        Cc = np.zeros((nv.value, 3), np.float64)
        E = np.zeros((nv.value, 4), np.int32)
        T = np.zeros((nt.value, 3), np.int32)
        self._L.o3d_mesh_copy(V.reshape(-1), Cc.reshape(-1), E.reshape(-1), T.reshape(-1))
        return dict(vertices=V, colors=Cc, edges=E, triangles=T)

    def set_blocks(self, keys, vox):
        """Seed blocks in the product's layout (keys int32 [n,3], vox float32 [n,5,512]), e.g. a GPU volume's
        `dump_blocks()`: each goes to its place in unit floor(key / (R/8)); the unit's other voxels keep weight 0."""
        k = np.ascontiguousarray(keys, np.int32).reshape(-1, 3)
        v = np.ascontiguousarray(vox, np.float32).reshape(k.shape[0], 5 * 512)
        for key, block in zip(k, v):
            self._L.o3d_set_block(self._h, int(key[0]), int(key[1]), int(key[2]), block)

    def extract_point_cloud(self):
        """ScalableTSDFVolume::ExtractPointCloud: points and colours float64 [n,3], in Open3D's loop order."""
        n = C.c_int64(0)
        self._L.o3d_extract_point_cloud(self._h, C.byref(n))
        P = np.zeros((n.value, 3), np.float64)
        Cc = np.zeros((n.value, 3), np.float64)
        self._L.o3d_points_copy(P.reshape(-1), Cc.reshape(-1))
        return dict(points=P, colors=Cc)


def canonical_mesh(vertices, colors, edges, triangles):
    """Order-independent form of a welded mesh: vertices sorted by canonical edge id
    (gx,gy,gz,axis); triangles re-indexed, each rotated so its smallest index leads (winding kept),
    then sorted.  Two extractions of the same volume are equal iff these arrays are equal."""
    edges = np.asarray(edges)
    order = np.lexsort((edges[:, 3], edges[:, 2], edges[:, 1], edges[:, 0]))
    inv = np.empty_like(order)
    inv[order] = np.arange(order.size)
    tri = inv[np.asarray(triangles)] if len(triangles) else np.zeros((0, 3), np.int64)
    if len(tri):
        k = np.argmin(tri, axis=1)
        idx = (k[:, None] + np.arange(3)[None, :]) % 3
        tri = np.take_along_axis(tri, idx, axis=1)
        tri = tri[np.lexsort((tri[:, 2], tri[:, 1], tri[:, 0]))]
    return dict(vertices=np.asarray(vertices)[order], colors=np.asarray(colors)[order],
                edges=edges[order], triangles=tri.astype(np.int64))


# ---------------------------------------------------------------------------------------------
# independent numpy restatement (pins the C oracle; float32 numpy, no FMA -> tolerance compare)
# ---------------------------------------------------------------------------------------------

def numpy_touched_blocks(depth, K, Tcw, voxel_size, sdf_trunc, depth_trunc, block_size=8, stride=4):
    """A.2 touched-block set of one frame as a sorted int32 [n,3] array (numpy, vectorised)."""
    fx, fy, cx, cy = [float(v) for v in K]
    d = np.asarray(depth, np.float32)[::stride, ::stride]
    H, W = d.shape
    jj, ii = np.meshgrid(np.arange(W) * stride, np.arange(H) * stride)
    valid = (d > 0) & (d < np.float32(depth_trunc))
    z = d[valid].astype(np.float64)
    x = (jj[valid].astype(np.float64) - cx) * z / fx
    y = (ii[valid].astype(np.float64) - cy) * z / fy
    Tcw = np.asarray(Tcw, np.float64).reshape(4, 4)
    R = Tcw[:3, :3].T
    t = -np.stack([(R[a, 0] * Tcw[0, 3] + R[a, 1] * Tcw[1, 3]) + R[a, 2] * Tcw[2, 3]
                   for a in range(3)])
    pw = np.stack([((R[a, 0] * x + R[a, 1] * y) + R[a, 2] * z) + t[a] for a in range(3)], axis=1)
    tau = float(np.float32(sdf_trunc))
    inv_vs = np.float32(1.0) / np.float32(voxel_size)
    lo = np.floor((pw - tau).astype(np.float32) * inv_vs).astype(np.int64) // block_size
    hi = np.floor((pw + tau).astype(np.float32) * inv_vs).astype(np.int64) // block_size
    keys = set()
    span = (hi - lo).max(axis=0) + 1 if len(lo) else np.zeros(3, np.int64)
    for dx in range(int(span[0])):
        for dy in range(int(span[1])):
            for dz in range(int(span[2])):
                k = lo + np.array([dx, dy, dz])
                ok = np.all(k <= hi, axis=1)
                keys.update(map(tuple, k[ok]))
    out = np.array(sorted(keys), dtype=np.int32).reshape(-1, 3)
    return out


def numpy_integrate_block(vox, key, depth, color, K, Tcw, voxel_size, sdf_trunc, depth_trunc,
                          block_size=8):
    """A.3 update of one block in float32 numpy (no FMA, true divisions): an independent second
    restatement.  vox: f32 [5, B^3] -> new f32 [5, B^3]."""
    B = block_size
    f32 = np.float32
    vs, tau = f32(voxel_size), f32(sdf_trunc)
    fx, fy, cx, cy = [f32(v) for v in K]
    E = np.asarray(Tcw, np.float64).reshape(4, 4).astype(np.float32)
    H, W = depth.shape
    l = np.arange(B ** 3)
    lx, ly, lz = l % B, (l // B) % B, l // (B * B)
    c = np.stack([(f32(key[0] * B) + lx.astype(np.float32) + f32(0.5)) * vs,
                  (f32(key[1] * B) + ly.astype(np.float32) + f32(0.5)) * vs,
                  (f32(key[2] * B) + lz.astype(np.float32) + f32(0.5)) * vs], axis=1)
    p = (c.astype(np.float64) @ E[:3, :3].astype(np.float64).T + E[:3, 3].astype(np.float64))
    p = p.astype(np.float32)
    out = np.array(vox, dtype=np.float32, copy=True)
    pz = p[:, 2]
    with np.errstate(divide="ignore", invalid="ignore"):
        u_f = p[:, 0] * fx / pz + cx + f32(0.5)
        v_f = p[:, 1] * fy / pz + cy + f32(0.5)
    ok = (pz > 0) & (u_f >= f32(0.0001)) & (u_f < f32(W) - f32(0.0001)) & \
         (v_f >= f32(0.0001)) & (v_f < f32(H) - f32(0.0001))
    u = np.where(ok, u_f, 0).astype(np.int64)
    v = np.where(ok, v_f, 0).astype(np.int64)
    d = depth[v, u].astype(np.float32)
    ok &= (d > 0) & (d < f32(depth_trunc))
    xx = (u.astype(np.float32) - cx) / fx
    yy = (v.astype(np.float32) - cy) / fy
    lam = np.sqrt(xx * xx + yy * yy + f32(1.0))
    sdf = (d - pz) * lam
    ok &= sdf > -tau
    t = np.minimum(f32(1.0), sdf / tau)
    w = out[1]
    wn = w + f32(1.0)
    rgb = color[v, u].astype(np.float32)
    new_t = (out[0] * w + t) / wn
    out[0] = np.where(ok, new_t, out[0])
    for k in range(3):
        out[2 + k] = np.where(ok, (out[2 + k] * w + rgb[:, k]) / wn, out[2 + k])
    out[1] = np.where(ok, wn, w)
    return out, ok


# ---------------------------------------------------------------------------------------------
# compiled reference: semantic voxel-block grids (SURVEY.md §8(f) rank 2)
# ---------------------------------------------------------------------------------------------
_EIGEN_SO = os.path.join(_DIR, "_ref", "libeigen_ops.so")


def have_eigen_ops() -> bool:
    return os.path.exists(_EIGEN_SO)


class EigenOps:
    """The three Eigen expressions of Open3D's TSDF path, evaluated by the Eigen vendored in the reference tree
    (oracle/eigen_ops.cpp; x86-64 baseline like Open3D's wheels).  Row-major numpy in and out."""

    def __init__(self):
        if not have_eigen_ops():
            raise RuntimeError("oracle/_ref/libeigen_ops.so missing (needs /root/reference to build)")
        self._L = C.CDLL(_EIGEN_SO)
        self.version = int(self._L.eig_version())

    def mat4f_times_vec4f(self, M, v):
        M = np.ascontiguousarray(M, np.float32).reshape(4, 4)
        v = np.ascontiguousarray(v, np.float32).reshape(4)
        out = np.zeros(4, np.float32)
        self._L.eig_mat4f_times_vec4f(C.c_void_p(M.ctypes.data), C.c_void_p(v.ctypes.data), C.c_void_p(out.ctypes.data))
        return out

    def mat4d_times_vec4d(self, M, v):
        M = np.ascontiguousarray(M, np.float64).reshape(4, 4)
        v = np.ascontiguousarray(v, np.float64).reshape(4)
        out = np.zeros(4, np.float64)
        self._L.eig_mat4d_times_vec4d(C.c_void_p(M.ctypes.data), C.c_void_p(v.ctypes.data), C.c_void_p(out.ctypes.data))
        return out

    def mat4d_inverse(self, M):
        M = np.ascontiguousarray(M, np.float64).reshape(4, 4)
        out = np.zeros((4, 4), np.float64)
        self._L.eig_mat4d_inverse(C.c_void_p(M.ctypes.data), C.c_void_p(out.ctypes.data))
        return out


def open3d_order_inverse4(M):
    """The float64 cofactor inverse oracle/open3d_order.c uses for camera_pose = extrinsic.inverse()."""
    L = _o3d()
    M = np.ascontiguousarray(M, np.float64).reshape(4, 4)
    out = np.zeros((4, 4), np.float64)
    L.o3d_inverse4(C.c_void_p(M.ctypes.data), C.c_void_p(out.ctypes.data))
    return out


_SEM_SO = os.path.join(_DIR, "_ref", "libref_semantic.so")
_sem_lib = None


def have_ref_semantic() -> bool:
    return os.path.exists(_SEM_SO)


def _sem():
    global _sem_lib
    if _sem_lib is None:
        if not have_ref_semantic():
            raise RuntimeError("oracle/_ref/libref_semantic.so missing (needs /root/reference to build)")
        L = C.CDLL(_SEM_SO)
        vp = C.c_void_p
        L.refsem_create.restype = vp
        L.refsem_create.argtypes = [C.c_int, C.c_double, C.c_int]
        L.refsem_destroy.argtypes = [vp]
        L.refsem_clear.argtypes = [vp]
        L.refsem_set_depth_threshold.argtypes = [C.c_int, C.c_float]
        L.refsem_set_depth_decay_rate.argtypes = [C.c_float]
        L.refsem_get_depth_threshold.restype = C.c_float
        L.refsem_get_depth_threshold.argtypes = [C.c_int]
        L.refsem_get_depth_decay_rate.restype = C.c_float
        L.refsem_integrate.argtypes = [vp, _f64p, C.c_int64, vp, vp, vp, vp]
        L.refsem_integrate_f32.argtypes = [vp, _f32p, C.c_int64, vp, vp, vp, vp]
        L.refsem_num_blocks.restype = C.c_int64
        L.refsem_num_blocks.argtypes = [vp]
        L.refsem_dump_blocks.restype = C.c_int64
        L.refsem_dump_blocks.argtypes = [vp] * 10 + [C.c_int] + [vp] * 3
        L.refsem_get_voxels.restype = C.c_int64
        L.refsem_get_voxels.argtypes = [vp, C.c_int, C.c_float, vp, vp, vp, vp, vp]
        L.refsem_assign_object_ids.restype = C.c_int64
        L.refsem_assign_object_ids.argtypes = [vp, _f32p, C.c_int, C.c_int, _f64p, C.c_float, C.c_float, _i32p, _i32p,
                                               vp, C.c_float, C.c_int, C.c_float, C.c_int, _i32p, _i32p, C.c_int64]
        L.refsem_query.restype = C.c_int64
        L.refsem_query.argtypes = [vp, vp, C.c_int, C.c_int, vp, C.c_float, C.c_float, vp, C.c_int, C.c_float, vp, vp,
                                   vp, vp, vp]
        L.refsem_carve.argtypes = [vp, _f32p, C.c_int, C.c_int, _f64p, C.c_float, C.c_float, _f32p, C.c_float]
        L.refsem_set_next_object_id.argtypes = [C.c_int32]
        L.refsem_get_next_object_id.restype = C.c_int32
        L.refsem_integrate_segment.argtypes = [vp, _f64p, C.c_int64, _f32p, C.c_int, C.c_int]
        L.refsem_segments.restype = C.c_int64
        L.refsem_segments.argtypes = [vp, C.c_int, C.c_int, C.c_float] + [vp] * 8 + [C.POINTER(C.c_int64)]
        L.refsem_remove_low_count_voxels.argtypes = [vp, C.c_int]
        L.refsem_remove_low_confidence_segments.argtypes = [vp, C.c_int]
        L.refsem_merge_segments.argtypes = [vp, C.c_int, C.c_int]
        L.refsem_remove_segment.argtypes = [vp, C.c_int]
        _sem_lib = L
    return _sem_lib


class RefSemanticGrid:
    """The unmodified reference `VoxelBlockSemanticGrid` (kind="voting") or
    `VoxelBlockSemanticProbabilisticGrid` (kind="probabilistic"), sequential branch.  The depth threshold
    and decay rate are class-static in the reference (process-wide): set them right before use."""

    KINDS = {"voting": 0, "probabilistic": 1}

    def __init__(self, voxel_size: float, kind: str = "voting", block_size: int = 8):
        self._L = _sem()
        self.kind = self.KINDS[kind]
        self._h = self._L.refsem_create(self.kind, float(voxel_size), int(block_size))

    def __del__(self):
        if getattr(self, "_h", None):
            self._L.refsem_destroy(self._h)
            self._h = None

    def set_depth_threshold(self, v):
        self._L.refsem_set_depth_threshold(self.kind, float(v))

    def set_depth_decay_rate(self, v):
        self._L.refsem_set_depth_decay_rate(float(v))

    def integrate(self, points, colors=None, class_ids=None, instance_ids=None, depths=None):
        """float32 points take the reference's float overload (keys computed in float32), anything else float64."""
        f32 = np.asarray(points).dtype == np.float32
        pts = np.ascontiguousarray(points, np.float32 if f32 else np.float64)
        n = pts.shape[0]
        cols = np.ascontiguousarray(colors if colors is not None else np.zeros((n, 3)), np.float32)
        hold = [pts, cols]

        def ptr(a, dt):
            if a is None:
                return None
            b = np.ascontiguousarray(a, dt)
            assert b.shape == (n,)
            hold.append(b)
            return b.ctypes.data

        fn = self._L.refsem_integrate_f32 if f32 else self._L.refsem_integrate
        fn(self._h, pts, n, cols.ctypes.data, ptr(class_ids, np.int32), ptr(instance_ids, np.int32),
           ptr(depths, np.float32))

    def integrate_segment(self, points, colors, class_id, object_id):
        pts = np.ascontiguousarray(points, np.float64)
        cols = np.ascontiguousarray(colors, np.float32)
        self._L.refsem_integrate_segment(self._h, pts.reshape(-1), pts.shape[0], cols.reshape(-1), int(class_id),
                                         int(object_id))

    def _segments(self, by_class, min_count, min_confidence):
        tot = C.c_int64(0)
        a = (self._h, int(by_class), int(min_count), float(min_confidence))
        n = self._L.refsem_segments(*a, None, None, None, None, None, None, None, None, C.byref(tot))
        ids, cls, npts = np.zeros(n, np.int32), np.zeros(n, np.int32), np.zeros(n, np.int64)
        cmin, cmax, obb = np.zeros(n, np.float32), np.zeros(n, np.float32), np.zeros((n, 10), np.float64)
        pts, cols = np.zeros((tot.value, 3), np.float64), np.zeros((tot.value, 3), np.float32)
        if n:
            self._L.refsem_segments(*a, ids.ctypes.data, cls.ctypes.data, npts.ctypes.data, cmin.ctypes.data,
                                    cmax.ctypes.data, obb.ctypes.data, pts.ctypes.data, cols.ctypes.data, C.byref(tot))
        out, off = [], 0
        for k in range(n):
            m = int(npts[k])
            out.append(dict(id=int(ids[k]), class_id=int(cls[k]), points=pts[off:off + m], colors=cols[off:off + m],
                            confidence_min=float(cmin[k]), confidence_max=float(cmax[k]), obb_center=obb[k, 0:3],
                            obb_size=obb[k, 3:6], obb_quat_wxyz=obb[k, 6:10]))
            off += m
        return out

    def get_object_segments(self, min_count=1, min_confidence=0.0):
        return self._segments(0, min_count, min_confidence)

    def get_class_segments(self, min_count=1, min_confidence=0.0):
        return self._segments(1, min_count, min_confidence)

    def num_blocks(self):
        return int(self._L.refsem_num_blocks(self._h))

    def clear(self):
        self._L.refsem_clear(self._h)

    def dump_blocks(self, K=8):
        nb, nv = self.num_blocks(), 512
        d = dict(keys=np.zeros((nb, 3), np.int32), hashes=np.zeros(nb, np.uint64),
                 count=np.zeros((nb, nv), np.int32), pos_sum=np.zeros((nb, nv, 3), np.float64),
                 col_sum=np.zeros((nb, nv, 3), np.float32), object_id=np.zeros((nb, nv), np.int32),
                 class_id=np.zeros((nb, nv), np.int32), confidence=np.zeros((nb, nv), np.float32),
                 aux=np.zeros((nb, nv), np.int32), lab_obj=np.zeros((nb, nv, K), np.int32),
                 lab_cls=np.zeros((nb, nv, K), np.int32), lab_logp=np.zeros((nb, nv, K), np.float32))
        a = d
        self._L.refsem_dump_blocks(self._h, a["keys"].ctypes.data, a["hashes"].ctypes.data, a["count"].ctypes.data,
                                   a["pos_sum"].ctypes.data, a["col_sum"].ctypes.data, a["object_id"].ctypes.data,
                                   a["class_id"].ctypes.data, a["confidence"].ctypes.data, a["aux"].ctypes.data,
                                   int(K), a["lab_obj"].ctypes.data, a["lab_cls"].ctypes.data,
                                   a["lab_logp"].ctypes.data)
        return d

    def get_voxels(self, min_count=1, min_confidence=0.0):
        n = self._L.refsem_get_voxels(self._h, int(min_count), float(min_confidence), None, None, None, None, None)
        out = dict(points=np.zeros((n, 3), np.float64), colors=np.zeros((n, 3), np.float32),
                   class_ids=np.zeros(n, np.int32), object_ids=np.zeros(n, np.int32),
                   confidences=np.zeros(n, np.float32))
        if n:
            self._L.refsem_get_voxels(self._h, int(min_count), float(min_confidence), out["points"].ctypes.data,
                                      out["colors"].ctypes.data, out["class_ids"].ctypes.data,
                                      out["object_ids"].ctypes.data, out["confidences"].ctypes.data)
        return out

    def assign_object_ids_to_instance_ids(self, K, width, height, Tcw, depth_max, depth_min, class_image,
                                          instance_image, depth_image=None, depth_threshold=0.1, do_carving=False,
                                          min_vote_ratio=0.5, min_votes=3):
        """-> dict instance id -> object id (voxel_semantic_data_association.h:69-373)."""
        K4 = np.ascontiguousarray(K, np.float32)
        T = np.ascontiguousarray(np.asarray(Tcw, np.float64).reshape(16))
        ci = np.ascontiguousarray(class_image, np.int32)
        ii = np.ascontiguousarray(instance_image, np.int32)
        di = None if depth_image is None else np.ascontiguousarray(depth_image, np.float32)
        ids, objs = np.zeros(4096, np.int32), np.zeros(4096, np.int32)
        n = self._L.refsem_assign_object_ids(self._h, K4, int(width), int(height), T, float(depth_max),
                                             float(depth_min), ci, ii, None if di is None else di.ctypes.data,
                                             float(depth_threshold), int(bool(do_carving)), float(min_vote_ratio),
                                             int(min_votes), ids, objs, 4096)
        assert n <= 4096
        return {int(i): int(o) for i, o in zip(ids[:n], objs[:n])}

    def _query(self, K, width, height, Tcw, depth_max, depth_min, bbox, min_count, min_confidence):
        kp = tp = bp = None
        hold = []
        if K is not None:
            K4 = np.ascontiguousarray(K, np.float32)
            T = np.ascontiguousarray(np.asarray(Tcw, np.float64).reshape(16))
            hold += [K4, T]
            kp, tp = K4.ctypes.data, T.ctypes.data
        else:
            bb = np.ascontiguousarray(bbox, np.float64).reshape(6)
            hold.append(bb)
            bp = bb.ctypes.data
        args = (self._h, kp, int(width), int(height), tp, float(depth_max), float(depth_min), bp, int(min_count),
                float(min_confidence))
        n = self._L.refsem_query(*args, None, None, None, None, None)
        out = dict(points=np.zeros((n, 3), np.float64), colors=np.zeros((n, 3), np.float32),
                   class_ids=np.zeros(n, np.int32), object_ids=np.zeros(n, np.int32),
                   confidences=np.zeros(n, np.float32))
        if n:
            self._L.refsem_query(*args, out["points"].ctypes.data, out["colors"].ctypes.data,
                                 out["class_ids"].ctypes.data, out["object_ids"].ctypes.data,
                                 out["confidences"].ctypes.data)
        return out

    def get_voxels_in_camera_frustrum(self, K, width, height, Tcw, depth_max, depth_min, min_count=1,
                                      min_confidence=0.0):
        return self._query(K, width, height, Tcw, depth_max, depth_min, None, min_count, min_confidence)

    def get_voxels_in_bb(self, bbox, min_count=1, min_confidence=0.0):
        return self._query(None, 0, 0, None, 0.0, 0.0, bbox, min_count, min_confidence)

    def carve(self, K, width, height, Tcw, depth_max, depth_min, depth_image, depth_threshold):
        self._L.refsem_carve(self._h, np.ascontiguousarray(K, np.float32), int(width), int(height),
                             np.ascontiguousarray(np.asarray(Tcw, np.float64).reshape(16)), float(depth_max),
                             float(depth_min), np.ascontiguousarray(depth_image, np.float32), float(depth_threshold))

    @staticmethod
    def set_next_object_id(v):
        _sem().refsem_set_next_object_id(int(v))

    @staticmethod
    def get_next_object_id():
        return int(_sem().refsem_get_next_object_id())

    def remove_low_count_voxels(self, min_count):
        self._L.refsem_remove_low_count_voxels(self._h, int(min_count))

    def remove_low_confidence_segments(self, min_confidence):
        self._L.refsem_remove_low_confidence_segments(self._h, int(min_confidence))

    def merge_segments(self, a, b):
        self._L.refsem_merge_segments(self._h, int(a), int(b))

    def remove_segment(self, object_id):
        self._L.refsem_remove_segment(self._h, int(object_id))
