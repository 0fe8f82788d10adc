// b2v_internal.h — host-side state of a volume and the kernel launchers (one .cu per kernel family).
#pragma once

#include <cstdint>
#include <cuda.h>
#include <cuda_runtime.h>
#include <string>

#include "b2v_device.cuh"

namespace b2v {

// Constants of the projective update of one frame (Open3D UniformTSDFVolume::IntegrateWithDepthToCameraDistance-
// Multiplier): passed in kernel-parameter space, so the kernels read them as constant-bank operands.
struct IntFrame {
    float E[12];     // Tcw rows 0..2 as float32 (extrinsic.cast<float>())
    float Es[3];     // E[2], E[6], E[10] times voxel_length_f (extrinsic_scaled_f(:, 2)): the per-z-step increment
    float fxf, fyf, cxf, cyf;
    float safe_w, safe_h;   // W - 0.0001f, H - 0.0001f
    float tau, inv_tau;
    int32_t W;
    const float4 *tex;      // packed {valid depth | 0, lambda, rgbx, 0} texels of the frame
};

// camera -> world of one frame, float64 (allocation samples)
struct FramePose {
    double Rwc[9];   // rigid inverse of Tcw, row-major
    double twc[3];
};

// Per-frame constants of the allocate kernels (+ the update constants of the frame-by-frame path).
struct FrameParams {
    // f64 back-projection of the allocation samples (Open3D CreatePointCloudFromFloatDepthImage)
    double fx, fy, cx, cy;
    FramePose pose;
    double tau_d;    // sdf_trunc as float64 (unit mode: the value Open3D holds; D1: (double)sdf_trunc_f)
    double unit_len; // voxel_length * unit resolution, float64 (volume_unit_length_)
    IntFrame I;
    float inv_fx, inv_fy;   // 1.0f / fx, 1.0f / fy (lambda image)
    float inv_vs, depth_trunc;
    int32_t unit_shift;     // log2(blocks per unit side): 0 = 8^3 units (D1 allocation), 1 = Open3D's 16^3 units
    int32_t H, W, stride;
    uint32_t frame_id;
    int32_t shard_rank, shard_count;
    // fused group mode (b2v_integrate_batch): this frame is bit `group_bit` of group buffer
    // `group_buf`; -1 = per-frame mode (frame stamps + per-frame active lists)
    int32_t group_bit, group_buf;
};

// Volume-wide constants of the update kernels (frame independent).
struct VolumeConsts {
    double unit_len;     // float64 volume-unit length
    float vs, half_vs;   // voxel_length_f, voxel_length_f * 0.5f
    int32_t unit_shift;
};

// Fused group integration: up to kMaxGroup consecutive frames are applied to a block while it is
// resident in registers.
constexpr int kMaxGroup = 32;   // frames per fused group (bits of the membership mask); the default group is 16
// group state (masks, union list, texel images, counters) is kGroupBufs-deep: the allocation of group g+3 may
// run while group g is still being integrated
constexpr int kGroupBufs = 4;
struct GroupArgs {
    IntFrame f[kMaxGroup];
    VolumeConsts V;
    int32_t count;
};

// Device-resident bookkeeping of one volume.
struct PoolMeta {
    float *pool;              // [capacity][5][512] float32 planes: tsdf, weight, r, g, b
    int4 *block_keys;         // [capacity] key of pool block i (w unused)
    uint32_t *counters;       // device counters, see Counter
    uint32_t *active_slots;   // [kActiveRing][capacity] table slots touched by a frame
    uint32_t *group_mask;     // [kGroupBufs][table capacity] bit k: the slot is touched by frame k of the group
    uint32_t *union_slots;    // [kGroupBufs][capacity] slots touched by any frame of the group
    uint32_t *block_flags;    // [capacity] sign summary for the mesh extraction's tile filter: bit 0 = some store left
                              // an observed voxel (w != 0) with tsdf < 0, bit 1 = with tsdf >= 0; bits are only ever
                              // set, so the union over a tile is a superset of the signs present now
    uint32_t capacity;
};

enum Counter : int {
    kCtrPool = 0,            // number of allocated blocks (may exceed capacity on overflow)
    kCtrError = 1,           // sticky error flag (1 = pool overflow, 2 = table full)
    kCtrUpdatesLo = 2,       // 64-bit total of (block, frame) updates since reset (8-byte aligned)
    kCtrUpdatesHi = 3,
    kCtrActive0 = 4,         // [kActiveRing] per-frame counts of touched blocks
    kCtrNew0 = 8,            // [kActiveRing] per-frame counts of newly allocated blocks
    kCtrVisitsLo = 12,       // 64-bit total of block visits (one block read + written) since reset
    kCtrVisitsHi = 13,
    kCtrGroup0 = 16,         // [kGroupBufs][kGroupCtrStride] per-group-buffer counters, contiguous so that ONE
                             // memset re-arms a buffer: see GroupCounter
    kNumCounters = 16 + 4 * (4 + 32)
};
// offsets inside one group buffer's counter block (M.counters + kCtrGroup0 + buf * kGroupCtrStride)
enum GroupCounter : int {
    kGcUnion = 0,    // number of slots in the group's union list
    kGcNext = 1,     // work-stealing cursor of the fused kernel
    kGcNew = 2,      // blocks newly allocated by the group
    kGcTouched0 = 4  // [kMaxGroup] blocks touched by frame k of the group
};
constexpr int kGroupCtrStride = 4 + kMaxGroup;
__host__ __device__ __forceinline__ constexpr int group_ctr(int buf, int which) {
    return kCtrGroup0 + buf * kGroupCtrStride + which;
}
constexpr int kActiveRing = 4;
static_assert(kGcTouched0 + kMaxGroup <= kGroupCtrStride && kCtrGroup0 + kGroupBufs * kGroupCtrStride <= kNumCounters,
              "counter layout");

struct VolumeGeometry {   // set once per volume (b2v_create)
    float vs, tau, depth_trunc;
    double voxel_length, tau_d;   // float64 values as Open3D holds them
    int32_t unit_shift, stride;
    int32_t shard_rank, shard_count;
};
void fill_frame_params(FrameParams *p, const double K[4], const double Tcw[16], int H, int W,
                       const VolumeGeometry &g, uint32_t frame_id);
VolumeConsts volume_consts(const VolumeGeometry &g);

// ---- kernels (b2v_tsdf.cu) ----
// lambda image (Open3D's depth-to-camera-distance multiplier) for the current intrinsics
cudaError_t launch_lambda(const FrameParams &p, float *lam, cudaStream_t stream);
// TMA descriptors of one frame's images (2-D tiled: depth f32, colour u8 x3 interleaved, lambda f32)
struct FrameMaps {
    alignas(64) CUtensorMap depth;
    alignas(64) CUtensorMap color;
    const void *color_ptr = nullptr;  // host-side cache validation only
};
struct LambdaMap {
    alignas(64) CUtensorMap lam;
};
// TMA tile staging needs 16-byte aligned bases and row pitches (W % 16 == 0) and the 32x32 tile
bool tma_tiles_usable(int W, int stride, const void *depth, const void *color, const void *lam);
// returns false if the driver entry point is unavailable or encoding fails
bool encode_frame_maps(FrameMaps *maps, const float *depth, const uint8_t *color, int H, int W, int tile);
bool encode_lambda_map(LambdaMap *map, const float *lam, int H, int W, int tile);
// frame packing ({valid depth, lambda, rgbx} texels) + allocation + touched-set of one frame;
// zeroes the next frame's ring counters.  maps != nullptr: the image tiles are staged into shared
// memory with TMA (cp.async.bulk.tensor.2d); nullptr: plain loads.
cudaError_t launch_allocate(const FrameParams &p, const float *depth, const uint8_t *color,
                            const float *lam, float4 *texels, const HashTable &table,
                            const PoolMeta &meta, int ring, const FrameMaps *maps, const LambdaMap *lmap,
                            cudaStream_t stream);
// projective TSDF + colour update of every block touched by the frame
cudaError_t launch_integrate(const FrameParams &p, const VolumeConsts &vc, const HashTable &table,
                             const PoolMeta &meta, int ring, int grid_ctas, cudaStream_t stream);
// all frames of a group in ONE launch (blockIdx.z = frame): the per-frame latency chains overlap
struct GroupAllocArgs {
    FrameParams P;                 // constants shared by the frames of the group (P.pose / P.I unused)
    FramePose pose[kMaxGroup];
    const float *depth[kMaxGroup];
    const uint8_t *color[kMaxGroup];
    float4 *tex[kMaxGroup];
    FrameMaps maps[kMaxGroup];
    LambdaMap lmap;
    uint32_t frame_id0;            // frame id of the group's first frame
    int32_t count, use_tma;
};
static_assert(sizeof(GroupAllocArgs) < 32000, "kernel parameter space");
cudaError_t launch_allocate_group(const GroupAllocArgs &args, const float *lam, const HashTable &table,
                                  const PoolMeta &meta, cudaStream_t stream);
int integrate_max_resident_ctas_per_sm();
// d_bad[0]: reciprocals (3 x 2^23 inputs), d_bad[1]: quotients (`pairs` inputs) whose fast path differs from IEEE
cudaError_t launch_selftest_division(unsigned long long *d_bad, uint64_t pairs, cudaStream_t stream);
// fused update of a group of frames (each block is read and written once per group)
cudaError_t launch_integrate_group(const GroupArgs &args, const HashTable &table, const PoolMeta &meta,
                                   int group_buf, int grid_ctas, cudaStream_t stream);
// hashes[i] = BlockKeyHash(block_keys[i])
cudaError_t launch_block_hashes(const int4 *block_keys, uint64_t *hashes, uint32_t n,
                                cudaStream_t stream);
// keys of the slots in an active list
cudaError_t launch_gather_active_keys(const HashTable &table, const uint32_t *active_slots,
                                      uint32_t n, int4 *out, cudaStream_t stream);

// find-or-create the blocks of `keys` (unique) and copy `vox` [n][5][512] into them
cudaError_t launch_upload_blocks(const int4 *keys, const float *vox, uint32_t n, uint32_t *scratch_idx,
                                 const HashTable &table, const PoolMeta &meta, cudaStream_t stream);

// ---- mesh (b2v_mesh.cu) ----
// Scratch and outputs of one extraction.  Per-voxel scratch is indexed [pool block][voxel].
struct MeshBuffers {
    uint32_t n_blocks;
    int32_t *nbr;            // [n_blocks][8] pool index of the block at +(dx,dy,dz) (bit0=x), -1 if missing
    uint8_t *cube;           // [n_blocks][512] marching-cubes case of the cube rooted here (0 = none)
    uint32_t *edge_mask;     // [n_blocks][128] byte per voxel: bit a = a vertex lives on its +a edge
    uint32_t *local;         // [n_blocks][512] position of the voxel's first vertex (low 16 bits) / triangle (high) in its block
    uint32_t *sums;          // [2][n_blocks] per-block vertex / triangle counts
    uint32_t *offs;          // [2][n_blocks] exclusive scans of sums
    uint32_t *partials;      // [2][ceil(n_blocks / 1024)] chunk sums of the two-level scan
    uint32_t *totals;        // [8] total vertices, triangles; blocks with vertices, blocks with triangles; candidate
                             // tiles (sign-summary filter), classified tiles (see MeshTotal)
    uint32_t *work;          // [4][n_blocks] the blocks with vertices / with triangles (what the emit kernels visit);
                             // candidate tiles; tiles with a sign change (what classify / block sums visit)
    double *vertices;        // [nv][3] float64, Open3D's formula
    double *colors;          // [nv][3] in [0,1]
    int32_t *edge_ids;       // [nv][4] canonical weld key (voxel x,y,z, axis)
    int32_t *triangles;      // [nt][3]
};
enum MeshTotal : int { kMtVertices = 0, kMtTriangles = 1, kMtVertexBlocks = 2, kMtTriangleBlocks = 3,
                       kMtCandidates = 4, kMtTiles = 5, kNumMeshTotals = 8 };
// neighbour lookup (7 hash probes per block) + candidate tiles from the blocks' sign summaries, then the
// marching-cubes case per voxel + vertex ownership masks of the candidates (Open3D ExtractTriangleMesh semantics)
cudaError_t launch_mesh_classify(const HashTable &table, const PoolMeta &meta, const MeshBuffers &mb, int grid_ctas,
                                 cudaStream_t stream);
// the same front end + zero-crossing masks of Open3D ExtractPointCloud (no cube validity requirement)
cudaError_t launch_point_masks(const HashTable &table, const PoolMeta &meta, const MeshBuffers &mb, int grid_ctas,
                               cudaStream_t stream);
// per-block sums + exclusive scans -> offs, totals
cudaError_t launch_mesh_scan(const MeshBuffers &mb, int grid_ctas, cudaStream_t stream);
cudaError_t launch_mesh_vertices(const PoolMeta &meta, const MeshBuffers &mb, double voxel_length, int unit_shift,
                                 bool points, uint32_t work_blocks, cudaStream_t stream);
cudaError_t launch_mesh_triangles(const MeshBuffers &mb, uint32_t work_blocks, cudaStream_t stream);

// ---- point grids: the point-average grid (b2v_grid.cu) and the semantic grids (b2v_semantic.cu) ----
// device counters of a point grid
enum GridCounter : int {
    kGridPool = 0,         // number of allocated blocks (may exceed the capacity on overflow)
    kGridError = 1,        // sticky error flags: 1 = pool full, 2 = hash table full
    kGridNumCounters = 2
};

// Fused front-end of the RGBD paths: depth2pointcloud (pyslam/utilities/depth.py:45-85) + world transform
// (pyslam/dense/volumetric_integrator_voxel_grid.py:262-281) without materialising the point cloud.  float64
// arithmetic in the reference's operation order, then float32 like the front-end.
struct RgbdParams {
    double fx_inv, fy_inv, cx, cy;   // 1.0 / fx, 1.0 / fy (depth.py:67-68)
    double R[9], t[3];               // Twc (camera -> world)
    float min_depth, max_depth;
    int32_t H, W;
};
RgbdParams rgbd_params(const double K[4], const double Twc[16], int H, int W, float min_depth, float max_depth);

// Spatial queries / carving over the existing blocks (voxel_block_grid.hpp:717-1195, 1334-1540;
// voxel_grid_carving.h:47-80; camera_frustrum.cpp:174-196).  A voxel qualifies if count >= min_count and, for a box
// or frustum query, its key lies in [min_key, max_key] and its mean position passes the fine test (double
// arithmetic like the reference).
enum QueryMode : int32_t { kQueryAll = 0, kQueryBox = 1, kQueryFrustum = 2 };
struct GridQuery {
    int32_t mode, min_count;
    int32_t min_key[3], max_key[3];
    double bb[6];                 // min xyz, max xyz
    double R[9], t[3];            // world -> camera
    float fx, fy, cx, cy, depth_min, depth_max;
    int32_t W, H;
};
// every voxel with count >= min_count (get_voxels)
inline void fill_all_query(GridQuery *q, int min_count) {
    *q = GridQuery{};
    q->mode = kQueryAll;
    q->min_count = min_count;
}
// box: voxel key bounds of `bbox` in double with the float inverse voxel size (voxel_block_grid.hpp:828-831)
void fill_box_query(GridQuery *q, const double bbox[6], int min_count, float inv_vs);
// frustum: world AABB of the frustum corners -> voxel key bounds
void fill_frustum_query(GridQuery *q, const float K[4], int W, int H, const double Tcw[16], float depth_max,
                        float depth_min, int min_count, float inv_vs);

// Copies a point grid's n device counters to the pinned mirror h (on `device`) and waits for the stream.  Returns
// the CUDA status; *full gets the "table / pool full" message when an insert ran out of capacity, else nullptr.
cudaError_t read_grid_counters(int device, cudaStream_t stream, const uint32_t *d, uint32_t *h, int n,
                               const char **full);
// blocks with storage: the pool counter clamped to the capacity
inline uint32_t grid_blocks_used(const uint32_t *h, uint32_t capacity) {
    return h[kGridPool] < capacity ? h[kGridPool] : capacity;
}
// block dumps: keys [n][3] and BlockKeyHash [n] of the pool's block keys (either output may be null)
void dump_block_keys(const int4 *k, int64_t n, int32_t *keys, uint64_t *hashes);

// ---- host helpers (b2v_api.cu) ----
// Sets obj->err and returns B2V_ERR_CUDA from the calling function when `call` fails.
#define B2V_CUDA(obj, call)                                                                \
    do {                                                                                   \
        cudaError_t e_ = (call);                                                           \
        if (e_ != cudaSuccess) {                                                           \
            (obj)->err = std::string(#call) + ": " + cudaGetErrorString(e_);               \
            return B2V_ERR_CUDA;                                                           \
        }                                                                                  \
    } while (0)
uint32_t next_pow2(uint64_t v);
// device or managed memory, which kernels read in place
bool is_device_pointer(const void *p);
// *out = src when the device reads it in place, else a new device copy *tmp (enqueued on `stream`; the caller frees
// *tmp, which stays null when no copy was made)
cudaError_t device_input(const void *src, size_t bytes, void **tmp, const void **out, cudaStream_t stream);
// frees *p and allocates n (at least 1) elements
template <typename T> cudaError_t regrow(T **p, size_t n) {
    cudaFree(*p);
    *p = nullptr;
    return cudaMalloc(p, (n ? n : 1) * sizeof(T));
}

// raw uint16 depth -> float32 metres (b2v_prep.cu)
cudaError_t launch_depth_u16_to_f32(const uint16_t *src, float *dst, size_t n, float scale, cudaStream_t stream);

// filter_shadow_points (pyslam/utilities/depth.py:103-146) on the device; scratch: 64 + 16384 bytes
constexpr size_t kShadowScratchBytes = 64 + 4096 * sizeof(uint32_t);
cudaError_t launch_filter_shadow_points(const float *depth, int H, int W, int dx, int dy, float fill, float *out,
                                        void *scratch, cudaStream_t stream);

// cv2.remap equivalents (bit-exact fixed-point bilinear for 8-bit x3, nearest for 32-bit pixels)
cudaError_t launch_remap_u8c3_linear(const uint8_t *src, int H, int W, const float *mapx, const float *mapy,
                                     uint8_t *dst, int swap_rb, cudaStream_t stream);
cudaError_t launch_remap_b32_nearest(const void *src, int H, int W, const float *mapx, const float *mapy, void *dst,
                                     cudaStream_t stream);

}  // namespace b2v
