// b2v_points.cuh — device code shared by the point grids: the point-average grid (b2v_grid.cu) and the semantic
// grids (b2v_semantic.cu).  Block insert, RGBD back-projection and the spatial-query tests, each defined once.
#pragma once

#include "b2v_internal.h"

namespace b2v {

// voxel coordinate of a point in its own precision: get_voxel_key_inv<Tpos, Tpos> (voxel_hashing.h:69-75) with the
// float32 inverse voxel size widened for float64 points (voxel_block_grid.hpp:473)
__device__ __forceinline__ int point_voxel_coord(float x, float inv_vs) { return voxel_coord(x, inv_vs); }
__device__ __forceinline__ int point_voxel_coord(double x, float inv_vs) {
    return __double2int_rd(__dmul_rn(x, static_cast<double>(inv_vs)));
}

// Find-or-create the block (bx, by, bz) of this lane's point; every lane of a full warp calls it, `have` = false for
// a lane without a point.  One lane per distinct block of the warp probes the table (neighbouring points share
// blocks); a new block takes the next pool index.  counters[kGridError]: 1 = pool full, 2 = table full.
__device__ __forceinline__ void insert_block_warp(bool have, int bx, int by, int bz, const HashTable &T,
                                                  int4 *block_keys, uint32_t *counters, uint32_t capacity) {
    const int lane = threadIdx.x & 31;
    const unsigned long long pk = have ? (static_cast<unsigned long long>(slot_hash(bx, by, bz)) << 32 |
                                          static_cast<uint32_t>(bx * 73856093 ^ by * 19349663 ^ bz * 83492791))
                                       : ((1ull << 63) | static_cast<unsigned long long>(lane) << 40 | 0xFFFFFFull);
    const unsigned grp = __match_any_sync(0xffffffffu, pk);
    // hash equality is not key equality: only skip when the leader's key really matches
    const int leader = __ffs(grp) - 1;
    const int lbx = __shfl_sync(0xffffffffu, bx, leader), lby = __shfl_sync(0xffffffffu, by, leader),
              lbz = __shfl_sync(0xffffffffu, bz, leader);
    if (!have) return;
    if (leader != lane && lbx == bx && lby == by && lbz == bz) return;
    bool is_new;
    const uint32_t slot = table_insert(T, bx, by, bz, &is_new);
    if (slot == kEmpty) {
        atomicOr(counters + kGridError, 2u);
        return;
    }
    if (is_new) {
        const uint32_t idx = atomicAdd(counters + kGridPool, 1u);
        uint32_t *w = reinterpret_cast<uint32_t *>(T.entries + slot) + 3;
        if (idx < capacity) {
            block_keys[idx] = make_int4(bx, by, bz, 0);
            *w = idx;
        } else {
            *w = kNoBlock;
            atomicOr(counters + kGridError, 1u);
        }
    }
}

// ---- RGBD front-end: depth2pointcloud (pyslam/utilities/depth.py:45-85) + world transform ----------------------
// world point of pixel i, false for an invalid depth: float64 in the reference's operation order, then float32
// (voxel_grid.py:262-265, 281; semantic_grid.py:411-415, 434-436)
__device__ __forceinline__ bool rgbd_point(const RgbdParams &P, const float *__restrict__ depth, int64_t i,
                                           float pt[3]) {
    const float d = depth[i];
    if (!(d > P.min_depth && d < P.max_depth)) return false;  // depth.py:62
    const int row = static_cast<int>(i / P.W), col = static_cast<int>(i % P.W);
    const double z = static_cast<double>(d);
    const double x = __dmul_rn(__dmul_rn(__dsub_rn(static_cast<double>(col), P.cx), z), P.fx_inv);  // depth.py:72
    const double y = __dmul_rn(__dmul_rn(__dsub_rn(static_cast<double>(row), P.cy), z), P.fy_inv);  // depth.py:73
#pragma unroll
    for (int a = 0; a < 3; ++a)
        pt[a] = __double2float_rn(__dadd_rn(
            __dadd_rn(__dadd_rn(__dmul_rn(x, P.R[3 * a]), __dmul_rn(y, P.R[3 * a + 1])), __dmul_rn(z, P.R[3 * a + 2])),
            P.t[a]));
    return true;
}

// image / 255.0 in float64, then float32 (depth.py:76)
__device__ __forceinline__ float rgbd_color(uint8_t c) {
    return __double2float_rn(__ddiv_rn(static_cast<double>(c), 255.0));
}

// ---- spatial queries (GridQuery) ---------------------------------------------------------------------------------
__device__ __forceinline__ bool block_in_range(const GridQuery &Q, const int4 key) {
    const int k[3] = {key.x, key.y, key.z};
#pragma unroll
    for (int a = 0; a < 3; ++a)
        if (k[a] < block_coord(Q.min_key[a]) || k[a] > block_coord(Q.max_key[a])) return false;
    return true;
}

// voxel t of block `key`
__device__ __forceinline__ bool voxel_key_in_range(const GridQuery &Q, const int4 key, int t) {
    const int vk[3] = {key.x * kB + (t & 7), key.y * kB + ((t >> 3) & 7), key.z * kB + (t >> 6)};
#pragma unroll
    for (int a = 0; a < 3; ++a)
        if (vk[a] < Q.min_key[a] || vk[a] > Q.max_key[a]) return false;
    return true;
}

struct ImagePoint {
    float u, v, depth;
};

// CameraFrustrum::contains (camera_frustrum.cpp:174-196): world point -> (inside?, pixel, depth)
__device__ __forceinline__ bool frustum_contains(const GridQuery &Q, const double p[3], ImagePoint *ip) {
    double pc[3];
#pragma unroll
    for (int a = 0; a < 3; ++a)
        pc[a] = __dadd_rn(__dadd_rn(__dadd_rn(__dmul_rn(Q.R[3 * a], p[0]), __dmul_rn(Q.R[3 * a + 1], p[1])),
                                    __dmul_rn(Q.R[3 * a + 2], p[2])),
                          Q.t[a]);
    const float depth = static_cast<float>(pc[2]);
    if (!(depth >= Q.depth_min && depth <= Q.depth_max)) return false;
    ip->u = static_cast<float>(__dadd_rn(__dmul_rn(static_cast<double>(Q.fx), __ddiv_rn(pc[0], pc[2])),
                                         static_cast<double>(Q.cx)));
    ip->v = static_cast<float>(__dadd_rn(__dmul_rn(static_cast<double>(Q.fy), __ddiv_rn(pc[1], pc[2])),
                                         static_cast<double>(Q.cy)));
    ip->depth = depth;
    return ip->u >= 0.0f && ip->u < static_cast<float>(Q.W) && ip->v >= 0.0f && ip->v < static_cast<float>(Q.H);
}

// the fine test of a box or frustum query on a voxel's mean position (double arithmetic like the reference).  An
// empty voxel's 0/0 mean fails both.
__device__ __forceinline__ bool position_in_query(const GridQuery &Q, const double p[3], ImagePoint *ip) {
    if (Q.mode == kQueryBox)  // BoundingBox3D::contains (bounding_boxes_3d.cpp:207-210)
        return p[0] >= Q.bb[0] && p[0] <= Q.bb[3] && p[1] >= Q.bb[1] && p[1] <= Q.bb[4] && p[2] >= Q.bb[2] &&
               p[2] <= Q.bb[5];
    return frustum_contains(Q, p, ip);
}

}  // namespace b2v
