// b2v_grid.cu — point-average voxel block grid (pySLAM's own `volumetric.VoxelBlockGrid`), sm_100a: kernels and
// the C ABI of include/b2v.h (b2v_grid_*).
//
// Replaces VoxelBlockGridT<VoxelData>::integrate_raw / get_voxels / remove_low_count_voxels
// (cpp/volumetric/voxel_block_grid.hpp:115-136, 524-614, 625-647, 717-819).  Per voxel the
// reference keeps {count, position_sum[3], color_sum[3]} (cpp/volumetric/voxel_data.h:118-133);
// here each block stores the same seven fields as 512-wide planes so a warp's accesses coalesce.
//   keys: voxel = floor(p * inv_vs) (voxel_hashing.h:69-75), block = floor_div(voxel, 8),
//         local index lx + 8 ly + 64 lz (voxel_block.h:67-70) -- bit exact.
//   sums: float atomics => same values as the reference up to summation order.
#include <algorithm>
#include <cmath>
#include <cstring>
#include <new>
#include <string>
#include <vector>

#include "../../include/b2v.h"
#include "b2v_points.cuh"
#include "b2v_scan.cuh"

namespace b2v {

constexpr int kGridPlanes = 7;  // count(int32), px, py, pz, cr, cg, cb
constexpr int kGridBlockWords = kGridPlanes * kVox;

struct GridMeta {
    uint32_t *pool;        // [capacity][7][512] planes: count(int32), px, py, pz, cr, cg, cb (float32)
    int4 *block_keys;      // [capacity]
    uint32_t *counters;    // [kGridNumCounters]
    uint32_t capacity;
};

// ---- pass 1: make sure every point's block exists -------------------------------------------
template <typename Tp>
__global__ void __launch_bounds__(256)
grid_insert_kernel(const Tp *__restrict__ pts, const int64_t n, const float inv_vs,
                   const HashTable T, const GridMeta G) {
    const int64_t i = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
    const bool have = i < n;
    int bx = 0, by = 0, bz = 0;
    if (have) {
        bx = block_coord(point_voxel_coord(pts[3 * i + 0], inv_vs));
        by = block_coord(point_voxel_coord(pts[3 * i + 1], inv_vs));
        bz = block_coord(point_voxel_coord(pts[3 * i + 2], inv_vs));
    }
    insert_block_warp(have, bx, by, bz, T, G.block_keys, G.counters, G.capacity);
}

// ---- pass 2: accumulate ----------------------------------------------------------------------
// colour of a point as the voxel accumulates it: float passthrough, uint8 * (1.0f / 255.0f) (voxel_data.h:79-97)
__device__ __forceinline__ float color_value(float c) { return c; }
__device__ __forceinline__ float color_value(uint8_t c) { return __fmul_rn(static_cast<float>(c), 1.0f / 255.0f); }

// adds a point to voxel v: position sums, colour sums color(0..2) if has_color, count.  A point whose block got no
// storage is dropped.
template <typename ColorFn>
__device__ __forceinline__ void grid_add_point(const HashTable &T, const GridMeta &G, const int v[3], const float p[3],
                                               bool has_color, ColorFn color) {
    const uint32_t slot = table_find(T, block_coord(v[0]), block_coord(v[1]), block_coord(v[2]));
    if (slot == kEmpty) return;
    const uint32_t idx = T.entries[slot].w;
    if (idx >= G.capacity) return;
    const int l = local_coord(v[0]) + (local_coord(v[1]) << 3) + (local_coord(v[2]) << 6);
    uint32_t *blk = G.pool + static_cast<size_t>(idx) * kGridBlockWords;
    float *fb = reinterpret_cast<float *>(blk);
#pragma unroll
    for (int a = 0; a < 3; ++a) atomicAdd(fb + (1 + a) * kVox + l, p[a]);
    if (has_color)
#pragma unroll
        for (int a = 0; a < 3; ++a) atomicAdd(fb + (4 + a) * kVox + l, color(a));
    atomicAdd(reinterpret_cast<int *>(blk) + l, 1);
}

template <typename Tp, typename Tc>
__global__ void __launch_bounds__(256)
grid_accumulate_kernel(const Tp *__restrict__ pts, const Tc *__restrict__ cols, const int64_t n,
                       const float inv_vs, const HashTable T, const GridMeta G) {
    const int64_t i = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const int v[3] = {point_voxel_coord(pts[3 * i + 0], inv_vs), point_voxel_coord(pts[3 * i + 1], inv_vs),
                      point_voxel_coord(pts[3 * i + 2], inv_vs)};
    // position_sum += static_cast<float>(x) (voxel_data.h:53-57)
    const float p[3] = {static_cast<float>(pts[3 * i + 0]), static_cast<float>(pts[3 * i + 1]),
                        static_cast<float>(pts[3 * i + 2])};
    grid_add_point(T, G, v, p, cols != nullptr, [&](int a) { return color_value(cols[3 * i + a]); });
}

// ---- fused RGBD front-end: back-project + insert / accumulate ---------------------------------
__global__ void __launch_bounds__(256)
grid_rgbd_insert_kernel(const RgbdParams P, const float *__restrict__ depth, const float inv_vs,
                        const HashTable T, const GridMeta G) {
    const int64_t n = static_cast<int64_t>(P.H) * P.W;
    const int64_t i = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
    float pt[3];
    const bool have = i < n && rgbd_point(P, depth, i, pt);
    int bx = 0, by = 0, bz = 0;
    if (have) {
        bx = block_coord(voxel_coord(pt[0], inv_vs));
        by = block_coord(voxel_coord(pt[1], inv_vs));
        bz = block_coord(voxel_coord(pt[2], inv_vs));
    }
    insert_block_warp(have, bx, by, bz, T, G.block_keys, G.counters, G.capacity);
}

__global__ void __launch_bounds__(256)
grid_rgbd_accumulate_kernel(const RgbdParams P, const float *__restrict__ depth, const uint8_t *__restrict__ rgb,
                            const float inv_vs, const HashTable T, const GridMeta G) {
    const int64_t n = static_cast<int64_t>(P.H) * P.W;
    const int64_t i = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
    float pt[3];
    if (i >= n || !rgbd_point(P, depth, i, pt)) return;
    const int v[3] = {voxel_coord(pt[0], inv_vs), voxel_coord(pt[1], inv_vs), voxel_coord(pt[2], inv_vs)};
    // voxel_grid.py:271-273: the front-end's float64 colour, narrowed to float32
    grid_add_point(T, G, v, pt, true, [&](int a) { return rgbd_color(rgb[3 * i + a]); });
}

// ---- read-outs: count -> scan -> emit; carve ---------------------------------------------------
// the reference's per-voxel filter chain: count threshold, then for a box or frustum query the voxel-key range and
// the fine test of the float32 mean (voxel_data.h:58-69) widened to double
__device__ __forceinline__ bool query_voxel(const GridQuery &Q, const uint32_t *blk, const int4 key, int t,
                                            ImagePoint *ip) {
    const int c = reinterpret_cast<const int *>(blk)[t];
    if (c < Q.min_count) return false;
    if (Q.mode == kQueryAll) return true;
    if (!voxel_key_in_range(Q, key, t)) return false;
    const float *fb = reinterpret_cast<const float *>(blk);
    const float fc = static_cast<float>(c);
    const double p[3] = {__fdiv_rn(fb[1 * kVox + t], fc), __fdiv_rn(fb[2 * kVox + t], fc),
                         __fdiv_rn(fb[3 * kVox + t], fc)};
    return position_in_query(Q, p, ip);
}

__device__ __forceinline__ bool grid_keep(const GridMeta &G, const GridQuery &Q, uint32_t b, int t) {
    const int4 key = G.block_keys[b];
    ImagePoint ip;
    return (Q.mode == kQueryAll || block_in_range(Q, key)) &&
           query_voxel(Q, G.pool + static_cast<size_t>(b) * kGridBlockWords, key, t, &ip);
}

__global__ void __launch_bounds__(kVox)
grid_query_count_kernel(const GridMeta G, const GridQuery Q, uint32_t *__restrict__ sums) {
    __shared__ uint32_t s_warp[16];
    block_count_512(grid_keep(G, Q, blockIdx.x, threadIdx.x), s_warp, sums);
}

__global__ void __launch_bounds__(kVox)
grid_query_emit_kernel(const GridMeta G, const GridQuery Q, const uint32_t *__restrict__ offs,
                       float *__restrict__ out_pts, float *__restrict__ out_cols) {
    __shared__ uint32_t s_warp[16];
    const uint32_t b = blockIdx.x;
    const int t = threadIdx.x;
    const bool keep = grid_keep(G, Q, b, t);
    const uint32_t o = offs[b] + block_excl_scan_512(keep ? 1u : 0u, s_warp);
    if (!keep) return;
    const uint32_t *blk = G.pool + static_cast<size_t>(b) * kGridBlockWords;
    const float *fb = reinterpret_cast<const float *>(blk);
    const float fc = static_cast<float>(reinterpret_cast<const int *>(blk)[t]);  // voxel_data.h:64-67,104-107
#pragma unroll
    for (int k = 0; k < 3; ++k) {
        out_pts[3 * static_cast<size_t>(o) + k] = __fdiv_rn(fb[(1 + k) * kVox + t], fc);
        out_cols[3 * static_cast<size_t>(o) + k] = __fdiv_rn(fb[(4 + k) * kVox + t], fc);
    }
}

__global__ void __launch_bounds__(kVox)
grid_remove_low_count_kernel(const GridMeta G, const int min_count) {
    uint32_t *blk = G.pool + static_cast<size_t>(blockIdx.x) * kGridBlockWords;
    const int t = threadIdx.x;
    if (reinterpret_cast<const int *>(blk)[t] < min_count) {  // voxel_block_grid.hpp:641-643 -> reset()
#pragma unroll
        for (int k = 0; k < kGridPlanes; ++k) blk[k * kVox + t] = 0u;
    }
}

// carve (voxel_grid_carving.h:47-80): reset voxels that lie in front of the observed depth by more
// than the threshold.  The depth image is indexed with TRUNCATED pixel coordinates, like at<float>(v, u).
__global__ void __launch_bounds__(kVox)
grid_carve_kernel(const GridMeta G, const GridQuery Q, const float *__restrict__ depth, const float thr) {
    const uint32_t b = blockIdx.x;
    const int t = threadIdx.x;
    const int4 key = G.block_keys[b];
    if (!block_in_range(Q, key)) return;
    uint32_t *blk = G.pool + static_cast<size_t>(b) * kGridBlockWords;
    ImagePoint ip;
    if (!query_voxel(Q, blk, key, t, &ip)) return;
    const float image_depth = depth[static_cast<size_t>(static_cast<int>(ip.v)) * Q.W + static_cast<int>(ip.u)];
    if (image_depth <= 0.0f || !isfinite(image_depth)) return;
    if (ip.depth < image_depth - thr) {
#pragma unroll
        for (int k = 0; k < kGridPlanes; ++k) blk[k * kVox + t] = 0u;
    }
}

// ---- host helpers shared with the semantic grids (b2v_internal.h) ------------------------------
RgbdParams rgbd_params(const double K[4], const double Twc[16], int H, int W, float min_depth, float max_depth) {
    RgbdParams P;
    P.fx_inv = 1.0 / K[0];
    P.fy_inv = 1.0 / K[1];
    P.cx = K[2];
    P.cy = K[3];
    for (int i = 0; i < 3; ++i) {
        for (int j = 0; j < 3; ++j) P.R[3 * i + j] = Twc[4 * i + j];
        P.t[i] = Twc[4 * i + 3];
    }
    P.min_depth = min_depth;
    P.max_depth = max_depth;
    P.H = H;
    P.W = W;
    return P;
}

// voxel key bounds of q->bb in double (voxel_block_grid.hpp:828-831, 1340-1345: get_voxel_key_inv<double,double>
// with the float inv_voxel_size)
static void fill_key_bounds(GridQuery *q, float inv_vs) {
    for (int a = 0; a < 3; ++a) {
        q->min_key[a] = static_cast<int32_t>(std::floor(q->bb[a] * static_cast<double>(inv_vs)));
        q->max_key[a] = static_cast<int32_t>(std::floor(q->bb[3 + a] * static_cast<double>(inv_vs)));
    }
}

void fill_box_query(GridQuery *q, const double bbox[6], int min_count, float inv_vs) {
    std::memset(q, 0, sizeof(*q));
    q->mode = kQueryBox;
    q->min_count = min_count;
    for (int a = 0; a < 6; ++a) q->bb[a] = bbox[a];
    fill_key_bounds(q, inv_vs);
}

// frustum: AABB of the 8 frustum corners (camera_frustrum.cpp:209-260) -> voxel key bounds
void fill_frustum_query(GridQuery *q, const float K[4], int W, int H, const double Tcw[16], float depth_max,
                        float depth_min, int min_count, float inv_vs) {
    std::memset(q, 0, sizeof(*q));
    q->mode = kQueryFrustum;
    q->min_count = min_count;
    q->fx = K[0];
    q->fy = K[1];
    q->cx = K[2];
    q->cy = K[3];
    q->depth_min = depth_min;
    q->depth_max = depth_max;
    q->W = W;
    q->H = H;
    double Rwc[9], twc[3];
    for (int i = 0; i < 3; ++i) {
        for (int j = 0; j < 3; ++j) {
            q->R[3 * i + j] = Tcw[4 * i + j];
            Rwc[3 * i + j] = Tcw[4 * j + i];
        }
        q->t[i] = Tcw[4 * i + 3];
    }
    for (int i = 0; i < 3; ++i) twc[i] = -(Rwc[3 * i] * q->t[0] + Rwc[3 * i + 1] * q->t[1] + Rwc[3 * i + 2] * q->t[2]);
    for (int a = 0; a < 3; ++a) {
        q->bb[a] = 1e300;
        q->bb[3 + a] = -1e300;
    }
    const double us[4] = {0.0, static_cast<double>(W), static_cast<double>(W), 0.0};
    const double vs[4] = {0.0, 0.0, static_cast<double>(H), static_cast<double>(H)};
    for (int c = 0; c < 4; ++c) {
        const double xn = (us[c] - static_cast<double>(q->cx)) / static_cast<double>(q->fx);
        const double yn = (vs[c] - static_cast<double>(q->cy)) / static_cast<double>(q->fy);
        for (int far = 0; far < 2; ++far) {
            const double d = far ? static_cast<double>(depth_max) : static_cast<double>(depth_min);
            const double pc[3] = {xn * d, yn * d, d};
            for (int a = 0; a < 3; ++a) {
                const double w = Rwc[3 * a] * pc[0] + Rwc[3 * a + 1] * pc[1] + Rwc[3 * a + 2] * pc[2] + twc[a];
                q->bb[a] = std::min(q->bb[a], w);
                q->bb[3 + a] = std::max(q->bb[3 + a], w);
            }
        }
    }
    fill_key_bounds(q, inv_vs);
}

cudaError_t read_grid_counters(int device, cudaStream_t stream, const uint32_t *d, uint32_t *h, int n,
                               const char **full) {
    cudaError_t e = cudaSetDevice(device);
    if (e == cudaSuccess) e = cudaMemcpyAsync(h, d, n * sizeof(uint32_t), cudaMemcpyDeviceToHost, stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(stream);
    if (full)
        *full = e != cudaSuccess || !h[kGridError] ? nullptr
                : (h[kGridError] & 2u)             ? "hash table full: raise capacity_blocks"
                                                   : "block pool full: raise capacity_blocks";
    return e;
}

void dump_block_keys(const int4 *k, int64_t n, int32_t *keys, uint64_t *hashes) {
    for (int64_t i = 0; i < n; ++i) {
        if (keys) {
            keys[3 * i + 0] = k[i].x;
            keys[3 * i + 1] = k[i].y;
            keys[3 * i + 2] = k[i].z;
        }
        if (hashes) hashes[i] = block_key_hash(k[i].x, k[i].y, k[i].z);
    }
}

}  // namespace b2v

// ====================================================================================================================
// host side: the C ABI of include/b2v.h (b2v_grid_*)
// ====================================================================================================================
using namespace b2v;

struct b2v_grid {
    float voxel_size = 0.0f, inv_voxel_size = 0.0f;
    int device = 0;
    cudaStream_t stream = nullptr;
    HashTable table{};
    GridMeta meta{};
    uint32_t *h_counters = nullptr;
    float *d_pts = nullptr, *d_cols = nullptr;
    size_t stage_points = 0;
    uint32_t *d_sums = nullptr, *d_offs = nullptr, *d_total = nullptr;
    uint32_t scan_cap = 0;
    float *d_out_pts = nullptr, *d_out_cols = nullptr;
    size_t out_cap = 0;
    int64_t last_n = 0;
    std::string err;
};

extern "C" const char *b2v_grid_last_error(const b2v_grid *g) { return g ? g->err.c_str() : "null grid"; }

static int grid_clear_device(b2v_grid *g, uint32_t used_blocks) {
    const size_t tcap = static_cast<size_t>(g->table.mask) + 1;
    B2V_CUDA(g, cudaMemsetAsync(g->table.entries, 0xFF, tcap * sizeof(uint4), g->stream));
    B2V_CUDA(g, cudaMemsetAsync(g->meta.counters, 0, kGridNumCounters * sizeof(uint32_t), g->stream));
    B2V_CUDA(g, cudaMemsetAsync(g->meta.pool, 0,
                                static_cast<size_t>(used_blocks) * kGridBlockWords * sizeof(uint32_t), g->stream));
    return B2V_OK;
}

extern "C" int b2v_grid_create(float voxel_size, int32_t block_size, uint32_t capacity_blocks,
                               int32_t device, b2v_grid **out) {
    if (!out) return B2V_ERR_INVALID_ARGUMENT;
    *out = nullptr;
    if (block_size != B2V_BLOCK_SIZE || !(voxel_size > 0.0f) || capacity_blocks == 0)
        return B2V_ERR_INVALID_ARGUMENT;
    b2v_grid *g = new (std::nothrow) b2v_grid();
    if (!g) return B2V_ERR_INVALID_ARGUMENT;
    g->voxel_size = voxel_size;
    g->inv_voxel_size = 1.0f / voxel_size;  // voxel_block_grid.hpp:6
    g->device = device;
    *out = g;
    B2V_CUDA(g, cudaSetDevice(device));
    B2V_CUDA(g, cudaStreamCreateWithFlags(&g->stream, cudaStreamNonBlocking));
    const uint32_t tcap = next_pow2(static_cast<uint64_t>(capacity_blocks) * 2);
    g->table.mask = tcap - 1;
    g->table.stamp = nullptr;
    g->meta.capacity = capacity_blocks;
    B2V_CUDA(g, cudaMalloc(&g->table.entries, static_cast<size_t>(tcap) * sizeof(uint4)));
    B2V_CUDA(g, cudaMalloc(&g->meta.pool, static_cast<size_t>(capacity_blocks) * kGridBlockWords * sizeof(uint32_t)));
    B2V_CUDA(g, cudaMalloc(&g->meta.block_keys, static_cast<size_t>(capacity_blocks) * sizeof(int4)));
    B2V_CUDA(g, cudaMalloc(&g->meta.counters, kGridNumCounters * sizeof(uint32_t)));
    B2V_CUDA(g, cudaMalloc(&g->d_total, sizeof(uint32_t)));
    B2V_CUDA(g, cudaMallocHost(&g->h_counters, kGridNumCounters * sizeof(uint32_t)));
    int rc = grid_clear_device(g, capacity_blocks);
    if (rc != B2V_OK) return rc;
    B2V_CUDA(g, cudaStreamSynchronize(g->stream));
    return B2V_OK;
}

extern "C" int b2v_grid_destroy(b2v_grid *g) {
    if (!g) return B2V_OK;
    cudaSetDevice(g->device);
    if (g->stream) cudaStreamSynchronize(g->stream);
    void *ptrs[] = {g->table.entries, g->meta.pool, g->meta.block_keys, g->meta.counters, g->d_pts, g->d_cols,
                    g->d_sums, g->d_offs, g->d_total, g->d_out_pts, g->d_out_cols};
    for (void *p : ptrs) cudaFree(p);
    cudaFreeHost(g->h_counters);
    if (g->stream) cudaStreamDestroy(g->stream);
    delete g;
    return B2V_OK;
}

static int grid_read_counters(b2v_grid *g) {
    const char *full;
    B2V_CUDA(g, read_grid_counters(g->device, g->stream, g->meta.counters, g->h_counters, kGridNumCounters, &full));
    if (full) {
        g->err = full;
        return B2V_ERR_CAPACITY;
    }
    return B2V_OK;
}

static uint32_t grid_block_count(const b2v_grid *g) { return grid_blocks_used(g->h_counters, g->meta.capacity); }

extern "C" int b2v_grid_clear(b2v_grid *g) {
    if (!g) return B2V_ERR_INVALID_ARGUMENT;
    int rc = grid_read_counters(g);
    if (rc == B2V_ERR_CUDA) return rc;
    rc = grid_clear_device(g, grid_block_count(g));
    if (rc != B2V_OK) return rc;
    g->err.clear();
    B2V_CUDA(g, cudaStreamSynchronize(g->stream));
    return B2V_OK;
}

static int grid_integrate_any(b2v_grid *g, const void *points, bool f64, const void *colors, bool u8, int64_t n_points) {
    if (!g) return B2V_ERR_INVALID_ARGUMENT;
    if (n_points < 0 || (n_points > 0 && !points)) {
        g->err = "b2v_grid_integrate: bad arguments";
        return B2V_ERR_INVALID_ARGUMENT;
    }
    if (n_points == 0) return B2V_OK;  // voxel_block_grid.hpp:22-24,121-123
    B2V_CUDA(g, cudaSetDevice(g->device));
    const void *d_p = points;
    const void *d_c = colors;
    const bool dev_p = is_device_pointer(points);
    const bool dev_c = colors ? is_device_pointer(colors) : true;
    if (!dev_p || !dev_c) {
        if (static_cast<size_t>(n_points) > g->stage_points) {
            B2V_CUDA(g, cudaStreamSynchronize(g->stream));
            B2V_CUDA(g, regrow(&g->d_pts, static_cast<size_t>(n_points) * 3 * 2));  // room for float64 points
            B2V_CUDA(g, regrow(&g->d_cols, static_cast<size_t>(n_points) * 3));
            g->stage_points = static_cast<size_t>(n_points);
        }
        if (!dev_p) {
            B2V_CUDA(g, cudaMemcpyAsync(g->d_pts, points, static_cast<size_t>(n_points) * 3 * (f64 ? sizeof(double) : sizeof(float)),
                                        cudaMemcpyHostToDevice, g->stream));
            d_p = g->d_pts;
        }
        if (colors && !dev_c) {
            B2V_CUDA(g, cudaMemcpyAsync(g->d_cols, colors, static_cast<size_t>(n_points) * 3 * (u8 ? 1 : sizeof(float)),
                                        cudaMemcpyHostToDevice, g->stream));
            d_c = g->d_cols;
        }
    }
    const unsigned grid = static_cast<unsigned>((n_points + 255) / 256);
    cudaStream_t s = g->stream;
    const float inv = g->inv_voxel_size;
    if (f64) {
        const double *p = static_cast<const double *>(d_p);
        grid_insert_kernel<<<grid, 256, 0, s>>>(p, n_points, inv, g->table, g->meta);
        if (u8)
            grid_accumulate_kernel<<<grid, 256, 0, s>>>(p, static_cast<const uint8_t *>(d_c), n_points, inv, g->table, g->meta);
        else
            grid_accumulate_kernel<<<grid, 256, 0, s>>>(p, static_cast<const float *>(d_c), n_points, inv, g->table, g->meta);
    } else {
        const float *p = static_cast<const float *>(d_p);
        grid_insert_kernel<<<grid, 256, 0, s>>>(p, n_points, inv, g->table, g->meta);
        if (u8)
            grid_accumulate_kernel<<<grid, 256, 0, s>>>(p, static_cast<const uint8_t *>(d_c), n_points, inv, g->table, g->meta);
        else
            grid_accumulate_kernel<<<grid, 256, 0, s>>>(p, static_cast<const float *>(d_c), n_points, inv, g->table, g->meta);
    }
    B2V_CUDA(g, cudaGetLastError());
    return B2V_OK;
}

extern "C" int b2v_grid_integrate(b2v_grid *g, const float *points, const float *colors, int64_t n_points) {
    return grid_integrate_any(g, points, false, colors, false, n_points);
}

extern "C" int b2v_grid_integrate_f64(b2v_grid *g, const double *points, const float *colors, int64_t n_points) {
    return grid_integrate_any(g, points, true, colors, false, n_points);
}

extern "C" int b2v_grid_integrate_ex(b2v_grid *g, const void *points, int32_t points_f64, const void *colors,
                                     int32_t colors_u8, int64_t n_points) {
    return grid_integrate_any(g, points, points_f64 != 0, colors, colors_u8 != 0, n_points);
}

extern "C" int b2v_grid_integrate_rgbd(b2v_grid *g, const float *depth, const uint8_t *color, int32_t height,
                                       int32_t width, const double K[4], const double Twc[16], float max_depth,
                                       float min_depth, int32_t filter_shadow_points) {
    if (!g) return B2V_ERR_INVALID_ARGUMENT;
    if (!depth || !color || !K || !Twc || height <= 0 || width <= 0) {
        g->err = "b2v_grid_integrate_rgbd: bad arguments";
        return B2V_ERR_INVALID_ARGUMENT;
    }
    B2V_CUDA(g, cudaSetDevice(g->device));
    const size_t pixels = static_cast<size_t>(height) * width;
    void *tmp_d = nullptr, *tmp_c = nullptr;
    const void *d_depth = nullptr, *d_color = nullptr;
    cudaError_t e = device_input(depth, pixels * sizeof(float), &tmp_d, &d_depth, g->stream);
    if (e == cudaSuccess) e = device_input(color, pixels * 3, &tmp_c, &d_color, g->stream);
    float *filtered = nullptr;
    void *scratch = nullptr;
    if (e == cudaSuccess && filter_shadow_points) {  // voxel_grid.py:238-245: depth2pointcloud sees the filtered depth
        e = cudaMalloc(&filtered, pixels * sizeof(float));
        if (e == cudaSuccess) e = cudaMalloc(&scratch, kShadowScratchBytes);
        if (e == cudaSuccess && (height <= 2 || width <= 2)) e = cudaErrorInvalidValue;
        if (e == cudaSuccess)
            e = launch_filter_shadow_points(static_cast<const float *>(d_depth), height, width, 2, 2, -1.0f, filtered,
                                            scratch, g->stream);
        d_depth = filtered;
    }
    if (e == cudaSuccess) {
        const RgbdParams P = rgbd_params(K, Twc, height, width, min_depth, max_depth);
        const unsigned grid = static_cast<unsigned>((pixels + 255) / 256);
        const float *dd = static_cast<const float *>(d_depth);
        grid_rgbd_insert_kernel<<<grid, 256, 0, g->stream>>>(P, dd, g->inv_voxel_size, g->table, g->meta);
        grid_rgbd_accumulate_kernel<<<grid, 256, 0, g->stream>>>(P, dd, static_cast<const uint8_t *>(d_color),
                                                                 g->inv_voxel_size, g->table, g->meta);
        e = cudaGetLastError();
    }
    if (e == cudaSuccess && (tmp_d || tmp_c || filtered)) e = cudaStreamSynchronize(g->stream);
    cudaFree(tmp_d);
    cudaFree(tmp_c);
    cudaFree(filtered);
    cudaFree(scratch);
    if (e != cudaSuccess) {
        g->err = std::string("b2v_grid_integrate_rgbd: ") + cudaGetErrorString(e);
        return B2V_ERR_CUDA;
    }
    return B2V_OK;
}

extern "C" int b2v_grid_synchronize(b2v_grid *g) {
    if (!g) return B2V_ERR_INVALID_ARGUMENT;
    return grid_read_counters(g);
}

extern "C" int64_t b2v_grid_num_blocks(b2v_grid *g) {
    if (!g) return -1;
    if (grid_read_counters(g) == B2V_ERR_CUDA) return -1;
    return grid_block_count(g);
}

// count pass of a read-out: the number of voxels the query keeps (-1 on a device error); *nb = blocks in use
static int64_t grid_query_total(b2v_grid *g, const GridQuery &q, uint32_t *nb) {
    if (grid_read_counters(g) == B2V_ERR_CUDA) return -1;
    *nb = grid_block_count(g);
    if (*nb == 0) return 0;
    if (*nb > g->scan_cap) {
        if (regrow(&g->d_sums, *nb) != cudaSuccess || regrow(&g->d_offs, *nb) != cudaSuccess) return -1;
        g->scan_cap = *nb;
    }
    grid_query_count_kernel<<<*nb, kVox, 0, g->stream>>>(g->meta, q, g->d_sums);
    exclusive_scan_kernel<<<1, 1024, 0, g->stream>>>(g->d_sums, g->d_offs, g->d_total, *nb);
    uint32_t total = 0;
    if (cudaGetLastError() != cudaSuccess) return -1;
    if (cudaMemcpyAsync(&total, g->d_total, sizeof(uint32_t), cudaMemcpyDeviceToHost, g->stream) != cudaSuccess) return -1;
    if (cudaStreamSynchronize(g->stream) != cudaSuccess) return -1;
    return total;
}

static int64_t grid_run_query(b2v_grid *g, const GridQuery &q) {
    uint32_t nb = 0;
    const int64_t n = grid_query_total(g, q, &nb);
    if (n < 0) return -1;
    if (static_cast<size_t>(n) > g->out_cap) {
        if (regrow(&g->d_out_pts, static_cast<size_t>(n) * 3) != cudaSuccess) return -1;
        if (regrow(&g->d_out_cols, static_cast<size_t>(n) * 3) != cudaSuccess) return -1;
        g->out_cap = static_cast<size_t>(n);
    }
    if (nb) {
        grid_query_emit_kernel<<<nb, kVox, 0, g->stream>>>(g->meta, q, g->d_offs, g->d_out_pts, g->d_out_cols);
        if (cudaGetLastError() != cudaSuccess) return -1;
    }
    if (cudaStreamSynchronize(g->stream) != cudaSuccess) return -1;
    g->last_n = n;
    return n;
}

extern "C" int64_t b2v_grid_size(b2v_grid *g) {
    if (!g) return -1;
    GridQuery q;
    fill_all_query(&q, 1);
    uint32_t nb;
    return grid_query_total(g, q, &nb);
}

extern "C" int64_t b2v_grid_get_voxels(b2v_grid *g, int32_t min_count) {
    if (!g) return -1;
    GridQuery q;
    fill_all_query(&q, min_count);
    return grid_run_query(g, q);
}

extern "C" int b2v_grid_copy_voxels(b2v_grid *g, float *points, float *colors) {
    if (!g) return B2V_ERR_INVALID_ARGUMENT;
    const size_t n = static_cast<size_t>(g->last_n);
    if (points && n) B2V_CUDA(g, cudaMemcpy(points, g->d_out_pts, n * 3 * sizeof(float), cudaMemcpyDeviceToHost));
    if (colors && n) B2V_CUDA(g, cudaMemcpy(colors, g->d_out_cols, n * 3 * sizeof(float), cudaMemcpyDeviceToHost));
    return B2V_OK;
}

extern "C" int b2v_grid_remove_low_count_voxels(b2v_grid *g, int32_t min_count) {
    if (!g) return B2V_ERR_INVALID_ARGUMENT;
    const int rc = grid_read_counters(g);
    if (rc == B2V_ERR_CUDA) return rc;
    const uint32_t nb = grid_block_count(g);
    if (nb) {
        grid_remove_low_count_kernel<<<nb, kVox, 0, g->stream>>>(g->meta, min_count);
        B2V_CUDA(g, cudaGetLastError());
    }
    return B2V_OK;
}

extern "C" int64_t b2v_grid_get_voxels_in_frustum(b2v_grid *g, const float K[4], int32_t width, int32_t height,
                                                  const double Tcw[16], float depth_max, float depth_min,
                                                  int32_t min_count) {
    if (!g || !K || !Tcw || width <= 0 || height <= 0) return -1;
    GridQuery q;
    fill_frustum_query(&q, K, width, height, Tcw, depth_max, depth_min, min_count, g->inv_voxel_size);
    return grid_run_query(g, q);
}

extern "C" int64_t b2v_grid_get_voxels_in_bb(b2v_grid *g, const double bbox[6], int32_t min_count) {
    if (!g || !bbox) return -1;
    GridQuery q;
    fill_box_query(&q, bbox, min_count, g->inv_voxel_size);
    return grid_run_query(g, q);
}

extern "C" int b2v_grid_carve(b2v_grid *g, const float K[4], int32_t width, int32_t height, const double Tcw[16],
                              float depth_max, float depth_min, const float *depth, float depth_threshold) {
    if (!g) return B2V_ERR_INVALID_ARGUMENT;
    if (!K || !Tcw || !depth || width <= 0 || height <= 0) {
        g->err = "b2v_grid_carve: bad arguments";
        return B2V_ERR_INVALID_ARGUMENT;
    }
    const int rc = grid_read_counters(g);
    if (rc == B2V_ERR_CUDA) return rc;
    void *tmp = nullptr;
    const void *d_depth = nullptr;
    cudaError_t e = device_input(depth, static_cast<size_t>(width) * height * sizeof(float), &tmp, &d_depth, g->stream);
    const uint32_t nb = grid_block_count(g);
    if (e == cudaSuccess && nb) {
        GridQuery q;
        fill_frustum_query(&q, K, width, height, Tcw, depth_max, depth_min, 1, g->inv_voxel_size);
        grid_carve_kernel<<<nb, kVox, 0, g->stream>>>(g->meta, q, static_cast<const float *>(d_depth), depth_threshold);
        e = cudaGetLastError();
    }
    if (e == cudaSuccess) e = cudaStreamSynchronize(g->stream);
    cudaFree(tmp);
    if (e != cudaSuccess) {
        g->err = cudaGetErrorString(e);
        return B2V_ERR_CUDA;
    }
    return B2V_OK;
}

extern "C" int64_t b2v_grid_dump_blocks(b2v_grid *g, int32_t *keys, uint64_t *hashes, int32_t *count,
                                        float *pos_sum, float *col_sum) {
    if (!g) return -1;
    if (grid_read_counters(g) == B2V_ERR_CUDA) return -1;
    const uint32_t nb = grid_block_count(g);
    if (nb == 0) return 0;
    std::vector<int4> k(nb);
    if (cudaMemcpy(k.data(), g->meta.block_keys, nb * sizeof(int4), cudaMemcpyDeviceToHost) != cudaSuccess)
        return -1;
    dump_block_keys(k.data(), nb, keys, hashes);
    if (count || pos_sum || col_sum) {
        std::vector<uint32_t> raw(static_cast<size_t>(nb) * kGridBlockWords);
        if (cudaMemcpy(raw.data(), g->meta.pool, raw.size() * sizeof(uint32_t), cudaMemcpyDeviceToHost) != cudaSuccess)
            return -1;
        for (size_t b = 0; b < nb; ++b) {
            const uint32_t *blk = raw.data() + b * kGridBlockWords;
            const float *fb = reinterpret_cast<const float *>(blk);
            for (int l = 0; l < kVox; ++l) {
                if (count) count[b * kVox + l] = static_cast<int32_t>(blk[l]);
                for (int c = 0; c < 3; ++c) {
                    if (pos_sum) pos_sum[(b * kVox + l) * 3 + c] = fb[(1 + c) * kVox + l];
                    if (col_sum) col_sum[(b * kVox + l) * 3 + c] = fb[(4 + c) * kVox + l];
                }
            }
        }
    }
    return nb;
}
