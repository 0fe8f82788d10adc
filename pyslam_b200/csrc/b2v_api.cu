// b2v_api.cu — the C ABI (include/b2v.h) of the TSDF volume: lifetime, frame staging and stream pipelining,
// parity hooks; and the stand-alone prep entry points (b2v_remap, b2v_filter_shadow_points).  Host code only;
// kernels live in b2v_tsdf.cu, b2v_mesh.cu, b2v_prep.cu.  The point grids keep their ABI beside their kernels
// (b2v_grid.cu, b2v_semantic.cu).
//
// Per frame (b2v_integrate):   copy stream:    H2D depth, colour  -> event ready[s]
//                              compute stream: wait ready[s]; allocate_kernel; integrate_kernel;
//                                              event free[s]
// with a ring of kStage device staging slots, so the upload of frame f+1 overlaps the kernels of
// frame f.  Nothing synchronises with the host until b2v_synchronize / an inspection call.
#include <algorithm>
#include <cmath>
#include <cstring>
#include <new>
#include <string>
#include <unordered_map>
#include <vector>

#include "../../include/b2v.h"
#include "b2v_internal.h"

using namespace b2v;

namespace b2v {

// Host-side pose algebra, same operation order as the oracle (and -ffp-contract=off on the host
// compiler), so allocation keys agree bit for bit.
void fill_frame_params(FrameParams *p, const double K[4], const double Tcw[16], int H, int W,
                       const VolumeGeometry &g, uint32_t frame_id) {
    p->fx = K[0];
    p->fy = K[1];
    p->cx = K[2];
    p->cy = K[3];
    for (int i = 0; i < 3; ++i)
        for (int j = 0; j < 3; ++j) p->pose.Rwc[3 * i + j] = Tcw[4 * j + i];
    for (int i = 0; i < 3; ++i)
        p->pose.twc[i] = -((p->pose.Rwc[3 * i + 0] * Tcw[3] + p->pose.Rwc[3 * i + 1] * Tcw[7]) +
                           p->pose.Rwc[3 * i + 2] * Tcw[11]);
    p->tau_d = g.unit_shift > 0 ? g.tau_d : static_cast<double>(g.tau);
    p->unit_len = g.voxel_length * static_cast<double>(kB << g.unit_shift);
    IntFrame &I = p->I;
    for (int i = 0; i < 12; ++i) I.E[i] = static_cast<float>(Tcw[i]);
    for (int i = 0; i < 3; ++i) I.Es[i] = I.E[4 * i + 2] * g.vs;  // extrinsic_f * voxel_length_f, column 2
    I.fxf = static_cast<float>(K[0]);
    I.fyf = static_cast<float>(K[1]);
    I.cxf = static_cast<float>(K[2]);
    I.cyf = static_cast<float>(K[3]);
    I.safe_w = static_cast<float>(W) - 0.0001f;
    I.safe_h = static_cast<float>(H) - 0.0001f;
    I.tau = g.tau;
    I.inv_tau = 1.0f / g.tau;
    I.W = W;
    I.tex = nullptr;
    p->inv_fx = 1.0f / I.fxf;
    p->inv_fy = 1.0f / I.fyf;
    p->inv_vs = 1.0f / g.vs;  // voxel_block_grid.hpp:6
    p->depth_trunc = g.depth_trunc;
    p->unit_shift = g.unit_shift;
    p->H = H;
    p->W = W;
    p->stride = g.stride;
    p->frame_id = frame_id;
    p->shard_rank = g.shard_rank;
    p->shard_count = g.shard_count;
    p->group_bit = -1;
    p->group_buf = 0;
}

VolumeConsts volume_consts(const VolumeGeometry &g) {
    VolumeConsts c;
    c.unit_len = g.voxel_length * static_cast<double>(kB << g.unit_shift);
    c.vs = g.vs;
    c.half_vs = g.vs * 0.5f;
    c.unit_shift = g.unit_shift;
    return c;
}

uint32_t next_pow2(uint64_t v) {
    uint64_t p = 1;
    while (p < v) p <<= 1;
    return static_cast<uint32_t>(p);
}

bool is_device_pointer(const void *p) {
    cudaPointerAttributes a;
    if (cudaPointerGetAttributes(&a, p) != cudaSuccess) {
        cudaGetLastError();
        return false;
    }
    return a.type == cudaMemoryTypeDevice || a.type == cudaMemoryTypeManaged;
}

cudaError_t device_input(const void *src, size_t bytes, void **tmp, const void **out, cudaStream_t stream) {
    *tmp = nullptr;
    *out = src;
    if (is_device_pointer(src)) return cudaSuccess;
    cudaError_t e = cudaMalloc(tmp, bytes);
    if (e == cudaSuccess) e = cudaMemcpyAsync(*tmp, src, bytes, cudaMemcpyHostToDevice, stream);
    *out = *tmp;
    return e;
}

}  // namespace b2v

namespace {

static_assert(kCtrNew0 == kCtrActive0 + kActiveRing, "the ring counters are cleared with one memset");
constexpr int kFrameStage = 4;                       // staging ring of the frame-by-frame path
constexpr int kGroupStage = kGroupBufs * kMaxGroup;  // group buffers x kMaxGroup frames
constexpr int kStage = kGroupStage + kFrameStage;    // raw-frame staging slots (device copies of host frames)

// Depth images of an integrate call: float32 metres (u16_scale == 0) or raw uint16 that the device widens to
// float(depth) * u16_scale.
struct DepthInput {
    const void *ptr;
    float u16_scale;
};

// The images of one integrate call: frames of H x W pixels back to back, each kind on the host (staged through the
// copy stream) or on the device (read in place).
struct FrameImages {
    DepthInput depth;
    const uint8_t *color;
    int32_t H, W;
    bool dev_depth, dev_color;
};

}  // namespace

struct b2v_volume {
    b2v_config cfg{};
    VolumeGeometry geo{};
    cudaStream_t compute = nullptr, copy = nullptr, alloc = nullptr;
    cudaStream_t last_stream = nullptr;  // caller stream of the most recent frame (synchronised on reads)
    bool overlap = true;                 // allocate(f+1) on its own stream, concurrent with integrate(f)
    bool inputs_fenced = false;          // batch call: device inputs already ordered before the alloc stream
    bool fuse = true;                    // b2v_integrate_batch fuses groups of up to kMaxGroup frames
    int group_frames = 16;               // frames per fused group (1..kMaxGroup), b2v_set_group_size
    LambdaMap lam_map{};
    bool lam_map_ok = false;
    cudaEvent_t input_event = nullptr;   // b2v_set_input_event: readiness of the next batch's device inputs
    bool rings_stale = false;            // a fused batch advanced frame_id: the per-frame ring counters must be re-armed
    uint32_t group_id = 0;
    cudaEvent_t ev_galloc[kGroupBufs] = {}, ev_group_done[kGroupBufs] = {};
    int last_group_buf = -1, last_group_count = 0;  // most recent frame came from a fused group
    int64_t prof_frames = 0, prof_int_launches = 0;
    // optional rectification stage (b2v_set_rectification)
    float *d_mapx = nullptr, *d_mapy = nullptr;
    int rect_H = 0, rect_W = 0, rect_swap = 0;
    // TMA descriptors are cached per image address (encoding costs ~1 us of host time each)
    std::unordered_map<uintptr_t, FrameMaps> map_cache;
    int map_H = 0, map_W = 0;
    const float *map_lam = nullptr;
    cudaEvent_t ev_in = nullptr, ev_alloc_done[kActiveRing] = {}, ev_int_done[kActiveRing] = {};
    // Frame staging (ensure_staging): one allocation per image kind, holding slots of stage_pixels pixels.  The
    // kStage raw and rectified slots are the kGroupStage slots of the group buffers followed by the kFrameStage
    // slots of the per-frame ring; the texel kinds hold only the slots of their own path.
    size_t stage_pixels = 0;
    float *d_depth = nullptr;       // raw float32 depth: host uploads and widened uint16 depth
    uint8_t *d_color = nullptr;     // raw colour
    uint16_t *d_depth16 = nullptr;  // raw uint16 depth; allocated on first use
    float *d_rdepth = nullptr;      // rectified frames; allocated while maps are installed
    uint8_t *d_rcolor = nullptr;
    float4 *d_texel = nullptr;      // kFrameStage packed {depth, lambda, rgbx} frames read by integrate_kernel
    float4 *d_gtex = nullptr;       // kGroupStage texel images of the group buffers; allocated on first use
    float *d_lambda = nullptr;      // lambda image of the cached intrinsics
    double lam_K[4] = {0, 0, 0, 0};
    int lam_H = 0, lam_W = 0;
    cudaEvent_t ev_ready[kStage] = {}, ev_free[kStage] = {};
    HashTable table{};
    PoolMeta meta{};
    uint32_t frame_id = 0;  // frames integrated since reset (stamp = frame_id + 1)
    int grid_ctas = 0;
    int sm_count = 0;
    int64_t launches = 0;
    uint32_t *h_counters = nullptr;  // pinned mirror
    std::string err;
    // mesh / point-cloud extraction
    MeshBuffers mb{};
    uint32_t mesh_blocks_cap = 0;
    size_t mesh_v_cap = 0, mesh_t_cap = 0;
    int64_t last_nv = 0, last_nt = 0;
    uint32_t *h_totals = nullptr;
    // optional per-kernel timing (b2v_profile_*)
    bool prof_enabled = false;
    std::vector<cudaEvent_t> prof_events;  // quadruples: allocate begin/end, integrate begin/end
    size_t prof_used = 0;

    // image k of the run of frames staged from slot s0 of `base`: a run starts on a slot boundary and holds its
    // frames of `pixels` pixels back to back, so it uploads with one copy per image kind
    template <typename T> T *staged(T *base, int s0, size_t pixels, int k = 0, int channels = 1) const {
        return base + (stage_pixels * s0 + pixels * k) * channels;
    }
};

static int volume_clear_device(b2v_volume *v) {
    const size_t tcap = static_cast<size_t>(v->table.mask) + 1;
    B2V_CUDA(v, cudaMemsetAsync(v->table.entries, 0xFF, tcap * sizeof(uint4), v->compute));
    B2V_CUDA(v, cudaMemsetAsync(v->table.stamp, 0, tcap * sizeof(uint32_t), v->compute));
    B2V_CUDA(v, cudaMemsetAsync(v->meta.group_mask, 0, tcap * kGroupBufs * sizeof(uint32_t), v->compute));
    B2V_CUDA(v, cudaMemsetAsync(v->meta.counters, 0, kNumCounters * sizeof(uint32_t), v->compute));
    return B2V_OK;
}

// frees every staging kind (ensure_staging); the caller has waited for the device
static void free_staging(b2v_volume *v) {
    auto release = [](auto *&p) {
        cudaFree(p);
        p = nullptr;
    };
    release(v->d_depth);
    release(v->d_color);
    release(v->d_depth16);
    release(v->d_rdepth);
    release(v->d_rcolor);
    release(v->d_texel);
    release(v->d_gtex);
    release(v->d_lambda);
    v->stage_pixels = 0;
    v->lam_H = v->lam_W = 0;
}

extern "C" int b2v_version(void) { return 100; }

extern "C" int b2v_selftest_division(int32_t device, uint64_t pairs, uint64_t *bad_reciprocals, uint64_t *bad_quotients) {
    if (cudaSetDevice(device) != cudaSuccess) return B2V_ERR_CUDA;
    unsigned long long *d = nullptr, h[2] = {0, 0};
    if (cudaMalloc(&d, sizeof(h)) != cudaSuccess) return B2V_ERR_CUDA;
    cudaError_t e = cudaMemset(d, 0, sizeof(h));
    if (e == cudaSuccess) e = launch_selftest_division(d, pairs, nullptr);
    if (e == cudaSuccess) e = cudaMemcpy(h, d, sizeof(h), cudaMemcpyDeviceToHost);
    cudaFree(d);
    if (e != cudaSuccess) return B2V_ERR_CUDA;
    if (bad_reciprocals) *bad_reciprocals = h[0];
    if (bad_quotients) *bad_quotients = h[1];
    return B2V_OK;
}

extern "C" int b2v_device_sm_count(int32_t device) {
    int n = 0;
    if (cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, device) != cudaSuccess) return -1;
    return n;
}

extern "C" const char *b2v_last_error(const b2v_volume *v) { return v ? v->err.c_str() : "null volume"; }

extern "C" int b2v_create(const b2v_config *cfg, b2v_volume **out) {
    if (!cfg || !out) return B2V_ERR_INVALID_ARGUMENT;
    *out = nullptr;
    if (cfg->block_size != B2V_BLOCK_SIZE || !(cfg->voxel_size > 0.0f) || !(cfg->sdf_trunc > 0.0f) ||
        !(cfg->depth_trunc > 0.0f) || cfg->capacity_blocks == 0 || cfg->shard_count < 1 ||
        cfg->shard_rank < 0 || cfg->shard_rank >= cfg->shard_count ||
        (cfg->unit_resolution != 0 && cfg->unit_resolution != 8 && cfg->unit_resolution != 16) ||
        static_cast<float>(cfg->voxel_length > 0.0 ? cfg->voxel_length : cfg->voxel_size) != cfg->voxel_size ||
        static_cast<float>(cfg->sdf_trunc_d > 0.0 ? cfg->sdf_trunc_d : cfg->sdf_trunc) != cfg->sdf_trunc)
        return B2V_ERR_INVALID_ARGUMENT;
    // allocate_kernel packs 21 bits per axis inside one frustum
    if (static_cast<double>(cfg->depth_trunc) / (static_cast<double>(cfg->voxel_size) * kB) > 5.0e5)
        return B2V_ERR_UNSUPPORTED;
    b2v_volume *v = new (std::nothrow) b2v_volume();
    if (!v) return B2V_ERR_INVALID_ARGUMENT;
    v->cfg = *cfg;
    if (v->cfg.depth_stride < 1) v->cfg.depth_stride = 4;
    if (v->cfg.unit_resolution == 0) v->cfg.unit_resolution = 16;
    if (!(v->cfg.voxel_length > 0.0)) v->cfg.voxel_length = static_cast<double>(cfg->voxel_size);
    if (!(v->cfg.sdf_trunc_d > 0.0)) v->cfg.sdf_trunc_d = static_cast<double>(cfg->sdf_trunc);
    v->geo.vs = cfg->voxel_size;
    v->geo.tau = cfg->sdf_trunc;
    v->geo.depth_trunc = cfg->depth_trunc;
    v->geo.voxel_length = v->cfg.voxel_length;
    v->geo.tau_d = v->cfg.sdf_trunc_d;
    v->geo.unit_shift = v->cfg.unit_resolution == 16 ? 1 : 0;
    v->geo.stride = v->cfg.depth_stride;
    v->geo.shard_rank = cfg->shard_rank;
    v->geo.shard_count = cfg->shard_count;
    *out = v;  // returned even on CUDA failure so the caller can read b2v_last_error and destroy
    B2V_CUDA(v, cudaSetDevice(cfg->device));
    B2V_CUDA(v, cudaStreamCreateWithFlags(&v->compute, cudaStreamNonBlocking));
    B2V_CUDA(v, cudaStreamCreateWithFlags(&v->copy, cudaStreamNonBlocking));
    B2V_CUDA(v, cudaStreamCreateWithFlags(&v->alloc, cudaStreamNonBlocking));
    B2V_CUDA(v, cudaEventCreateWithFlags(&v->ev_in, cudaEventDisableTiming));
    for (int r = 0; r < kActiveRing; ++r) {
        B2V_CUDA(v, cudaEventCreateWithFlags(&v->ev_alloc_done[r], cudaEventDisableTiming));
        B2V_CUDA(v, cudaEventCreateWithFlags(&v->ev_int_done[r], cudaEventDisableTiming));
    }
    for (int b = 0; b < kGroupBufs; ++b) {
        B2V_CUDA(v, cudaEventCreateWithFlags(&v->ev_galloc[b], cudaEventDisableTiming));
        B2V_CUDA(v, cudaEventCreateWithFlags(&v->ev_group_done[b], cudaEventDisableTiming));
    }
    for (int s = 0; s < kStage; ++s) {
        B2V_CUDA(v, cudaEventCreateWithFlags(&v->ev_ready[s], cudaEventDisableTiming));
        B2V_CUDA(v, cudaEventCreateWithFlags(&v->ev_free[s], cudaEventDisableTiming));
    }
    const uint32_t cap = cfg->capacity_blocks;
    const uint32_t tcap = next_pow2(static_cast<uint64_t>(cap) * 2);
    v->table.mask = tcap - 1;
    v->meta.capacity = cap;
    B2V_CUDA(v, cudaMalloc(&v->table.entries, static_cast<size_t>(tcap) * sizeof(uint4)));
    B2V_CUDA(v, cudaMalloc(&v->table.stamp, static_cast<size_t>(tcap) * sizeof(uint32_t)));
    B2V_CUDA(v, cudaMalloc(&v->meta.pool, static_cast<size_t>(cap) * kBlockFloats * sizeof(float)));
    B2V_CUDA(v, cudaMalloc(&v->meta.block_keys, static_cast<size_t>(cap) * sizeof(int4)));
    B2V_CUDA(v, cudaMalloc(&v->meta.counters, kNumCounters * sizeof(uint32_t)));
    B2V_CUDA(v, cudaMalloc(&v->meta.active_slots, static_cast<size_t>(cap) * kActiveRing * sizeof(uint32_t)));
    B2V_CUDA(v, cudaMalloc(&v->meta.group_mask, static_cast<size_t>(tcap) * kGroupBufs * sizeof(uint32_t)));
    B2V_CUDA(v, cudaMalloc(&v->meta.union_slots, static_cast<size_t>(cap) * kGroupBufs * sizeof(uint32_t)));
    B2V_CUDA(v, cudaMalloc(&v->meta.block_flags, static_cast<size_t>(cap) * sizeof(uint32_t)));
    B2V_CUDA(v, cudaMemsetAsync(v->meta.block_flags, 0, static_cast<size_t>(cap) * sizeof(uint32_t), v->compute));
    B2V_CUDA(v, cudaMallocHost(&v->h_counters, kNumCounters * sizeof(uint32_t)));
    B2V_CUDA(v, cudaMallocHost(&v->h_totals, kNumMeshTotals * sizeof(uint32_t)));
    std::memset(v->h_totals, 0, kNumMeshTotals * sizeof(uint32_t));
    B2V_CUDA(v, cudaMemsetAsync(v->meta.pool, 0, static_cast<size_t>(cap) * kBlockFloats * sizeof(float),
                                v->compute));
    int rc = volume_clear_device(v);
    if (rc != B2V_OK) return rc;
    const int sms = b2v_device_sm_count(cfg->device);
    // persistent grid: exactly one wave of resident CTAs
    v->grid_ctas = (sms > 0 ? sms : 148) * integrate_max_resident_ctas_per_sm();
    v->sm_count = sms;
    B2V_CUDA(v, cudaStreamSynchronize(v->compute));
    return B2V_OK;
}

extern "C" int b2v_destroy(b2v_volume *v) {
    if (!v) return B2V_OK;
    cudaSetDevice(v->cfg.device);
    cudaDeviceSynchronize();
    if (v->ev_in) cudaEventDestroy(v->ev_in);
    for (int r = 0; r < kActiveRing; ++r) {
        if (v->ev_alloc_done[r]) cudaEventDestroy(v->ev_alloc_done[r]);
        if (v->ev_int_done[r]) cudaEventDestroy(v->ev_int_done[r]);
    }
    for (int s = 0; s < kStage; ++s) {
        if (v->ev_ready[s]) cudaEventDestroy(v->ev_ready[s]);
        if (v->ev_free[s]) cudaEventDestroy(v->ev_free[s]);
    }
    free_staging(v);
    cudaFree(v->d_mapx);
    cudaFree(v->d_mapy);
    for (int b = 0; b < kGroupBufs; ++b) {
        if (v->ev_galloc[b]) cudaEventDestroy(v->ev_galloc[b]);
        if (v->ev_group_done[b]) cudaEventDestroy(v->ev_group_done[b]);
    }
    cudaFree(v->meta.group_mask);
    cudaFree(v->meta.union_slots);
    cudaFree(v->meta.block_flags);
    cudaFree(v->table.entries);
    cudaFree(v->table.stamp);
    cudaFree(v->meta.pool);
    cudaFree(v->meta.block_keys);
    cudaFree(v->meta.counters);
    cudaFree(v->meta.active_slots);
    cudaFree(v->mb.nbr);
    cudaFree(v->mb.cube);
    cudaFree(v->mb.edge_mask);
    cudaFree(v->mb.local);
    cudaFree(v->mb.sums);
    cudaFree(v->mb.offs);
    cudaFree(v->mb.work);
    cudaFree(v->mb.totals);
    cudaFree(v->mb.partials);
    cudaFree(v->mb.vertices);
    cudaFree(v->mb.colors);
    cudaFree(v->mb.edge_ids);
    cudaFree(v->mb.triangles);
    cudaFreeHost(v->h_counters);
    cudaFreeHost(v->h_totals);
    for (cudaEvent_t e : v->prof_events)
        if (e) cudaEventDestroy(e);
    if (v->compute) cudaStreamDestroy(v->compute);
    if (v->copy) cudaStreamDestroy(v->copy);
    if (v->alloc) cudaStreamDestroy(v->alloc);
    delete v;
    return B2V_OK;
}

static int read_counters(b2v_volume *v) {
    B2V_CUDA(v, cudaSetDevice(v->cfg.device));
    B2V_CUDA(v, cudaStreamSynchronize(v->copy));
    B2V_CUDA(v, cudaStreamSynchronize(v->alloc));
    if (v->last_stream) B2V_CUDA(v, cudaStreamSynchronize(v->last_stream));
    B2V_CUDA(v, cudaMemcpyAsync(v->h_counters, v->meta.counters, kNumCounters * sizeof(uint32_t),
                                cudaMemcpyDeviceToHost, v->compute));
    B2V_CUDA(v, cudaStreamSynchronize(v->compute));
    if (v->h_counters[kCtrError]) {
        v->err = (v->h_counters[kCtrError] & 2u) ? "hash table full: raise capacity_blocks"
                                                 : "block pool full: raise capacity_blocks";
        return B2V_ERR_CAPACITY;
    }
    return B2V_OK;
}

static uint32_t block_count(const b2v_volume *v) {
    const uint32_t n = v->h_counters[kCtrPool];
    return n < v->meta.capacity ? n : v->meta.capacity;
}

extern "C" int b2v_reset(b2v_volume *v) {
    if (!v) return B2V_ERR_INVALID_ARGUMENT;
    int rc = read_counters(v);
    if (rc == B2V_ERR_CUDA) return rc;
    const uint32_t nb = block_count(v);
    B2V_CUDA(v, cudaMemsetAsync(v->meta.pool, 0, static_cast<size_t>(nb) * kBlockFloats * sizeof(float),
                                v->compute));
    B2V_CUDA(v, cudaMemsetAsync(v->meta.block_flags, 0, static_cast<size_t>(nb) * sizeof(uint32_t), v->compute));
    rc = volume_clear_device(v);
    if (rc != B2V_OK) return rc;
    v->frame_id = 0;
    v->group_id = 0;
    v->last_group_buf = -1;
    v->rings_stale = false;
    v->err.clear();
    B2V_CUDA(v, cudaStreamSynchronize(v->compute));
    return B2V_OK;
}

// Allocates the staging kinds that the next frames need, for images of `pixels` pixels: raw depth and colour, the
// per-frame texels and the lambda image always; raw uint16 depth, the group texels and the rectified frames once a
// call needs them.  Larger images reallocate every kind.  Kernels on any stream, a caller's stream included, may still
// read the old buffers, so that waits for the whole device; it happens only when the image size grows.
static int ensure_staging(b2v_volume *v, size_t pixels, bool u16, bool group) {
    if (pixels > v->stage_pixels) {
        B2V_CUDA(v, cudaDeviceSynchronize());
        free_staging(v);
        v->stage_pixels = pixels;
    }
    const size_t n = v->stage_pixels;
    auto alloc = [](auto *&p, size_t elems) { return p ? cudaSuccess : cudaMalloc(&p, elems * sizeof(*p)); };
    B2V_CUDA(v, alloc(v->d_depth, n * kStage));
    B2V_CUDA(v, alloc(v->d_color, n * 3 * kStage));
    B2V_CUDA(v, alloc(v->d_texel, n * kFrameStage));
    B2V_CUDA(v, alloc(v->d_lambda, n));
    if (u16) B2V_CUDA(v, alloc(v->d_depth16, n * kStage));
    if (group) B2V_CUDA(v, alloc(v->d_gtex, n * kGroupStage));
    if (v->d_mapx) {
        B2V_CUDA(v, alloc(v->d_rdepth, n * kStage));
        B2V_CUDA(v, alloc(v->d_rcolor, n * 3 * kStage));
    }
    return B2V_OK;
}

// The four timing events of one allocate / update launch pair (allocate begin, end, update begin, end) while
// profiling is on, else nullptr.  `frames`: the frames the pair integrates.
static int profile_events(b2v_volume *v, int frames, cudaEvent_t **pe) {
    *pe = nullptr;
    if (!v->prof_enabled) return B2V_OK;
    if (v->prof_used + 4 > v->prof_events.size()) {
        const size_t old = v->prof_events.size();
        v->prof_events.resize(old + 4 * 256, nullptr);
        for (size_t k = old; k < v->prof_events.size(); ++k) B2V_CUDA(v, cudaEventCreate(&v->prof_events[k]));
    }
    *pe = &v->prof_events[v->prof_used];
    v->prof_used += 4;
    v->prof_frames += frames;
    v->prof_int_launches += 1;
    return B2V_OK;
}

// cached TMA descriptors of a frame (keyed by the depth image address; colour address is checked)
static const FrameMaps *frame_maps(b2v_volume *v, const float *d_depth, const uint8_t *d_color, int H, int W) {
    if (!tma_tiles_usable(W, v->cfg.depth_stride, d_depth, d_color, v->d_lambda)) return nullptr;
    if (v->map_H != H || v->map_W != W || v->map_lam != v->d_lambda || v->map_cache.size() > 4096) {
        v->map_cache.clear();
        v->map_H = H;
        v->map_W = W;
        v->map_lam = v->d_lambda;
        v->lam_map_ok = encode_lambda_map(&v->lam_map, v->d_lambda, H, W, 32);
    }
    if (!v->lam_map_ok) return nullptr;
    auto it = v->map_cache.find(reinterpret_cast<uintptr_t>(d_depth));
    if (it != v->map_cache.end() && it->second.color_ptr == d_color) return &it->second;
    FrameMaps m;
    if (!encode_frame_maps(&m, d_depth, d_color, H, W, 32)) return nullptr;
    m.color_ptr = d_color;
    auto res = v->map_cache.insert_or_assign(reinterpret_cast<uintptr_t>(d_depth), m);
    return &res.first->second;
}

// recomputes the lambda image when the intrinsics or the image size change
static int refresh_lambda(b2v_volume *v, const FrameParams &P, const double K[4], int H, int W, cudaStream_t as) {
    if (v->lam_H == H && v->lam_W == W && std::memcmp(v->lam_K, K, sizeof(v->lam_K)) == 0) return B2V_OK;
    if (v->overlap) {  // the lambda image is read by allocate kernels that may still be in flight
        B2V_CUDA(v, cudaStreamSynchronize(v->alloc));
    }
    B2V_CUDA(v, launch_lambda(P, v->d_lambda, as));
    std::memcpy(v->lam_K, K, sizeof(v->lam_K));
    v->lam_H = H;
    v->lam_W = W;
    v->launches += 1;
    return B2V_OK;
}

// The checks that every integrate entry point makes, reported under the entry point's name `fn`; also finds where
// the images of `in` live.
static int check_integrate(b2v_volume *v, const char *fn, bool u16, int32_t n_frames, FrameImages *in,
                           const double *K, const double *Tcw, void *stream) {
    const char *why = nullptr;
    if (u16 && !(in->depth.u16_scale > 0.0f)) {
        why = "depth_scale must be positive";
    } else if (n_frames < 0 || in->H <= 0 || in->W <= 0 ||
               (n_frames > 0 && (!in->depth.ptr || !in->color || !K || !Tcw))) {
        why = "null pointer, negative frame count or non-positive image size";
    } else if (n_frames > 0 && !(K[0] > 0.0 && K[1] > 0.0)) {
        why = "focal lengths must be positive";
    } else if (n_frames > 0) {
        B2V_CUDA(v, cudaSetDevice(v->cfg.device));
        in->dev_depth = is_device_pointer(in->depth.ptr);
        in->dev_color = is_device_pointer(in->color);
        if (stream != nullptr && !(in->dev_depth && in->dev_color))
            why = "a caller stream requires device image pointers";
    }
    if (!why) return B2V_OK;
    v->err = std::string(fn) + ": " + why;
    return B2V_ERR_INVALID_ARGUMENT;
}

// Stages `count` consecutive frames of `in`, from frame f0 on, into the run of slots that starts at slot s0, for the
// allocate stream `as`.  Host images are uploaded on the copy stream, one copy per image kind, once `ev_free` has
// fired (the previous reader of the run is done); `ev_ready` orders `as` after the uploads.  Raw uint16 depth is
// widened in one launch, and every frame is rectified while maps are installed.  Returns the device images that the
// allocate kernels read, one per frame.
static int prepare_frames(b2v_volume *v, const FrameImages &in, size_t f0, int count, int s0, cudaEvent_t ev_free,
                          cudaEvent_t ev_ready, cudaStream_t as, const float **d_depth, const uint8_t **d_color) {
    const size_t pixels = static_cast<size_t>(in.H) * in.W;
    const float scale = in.depth.u16_scale;
    const size_t depth_bytes = scale > 0.0f ? sizeof(uint16_t) : sizeof(float);
    const void *depth = static_cast<const char *>(in.depth.ptr) + pixels * depth_bytes * f0;
    const uint8_t *color = in.color + pixels * 3 * f0;
    float *raw_depth = v->staged(v->d_depth, s0, pixels);
    uint8_t *raw_color = v->staged(v->d_color, s0, pixels, 0, 3);
    if (!in.dev_depth || !in.dev_color) {
        B2V_CUDA(v, cudaStreamWaitEvent(v->copy, ev_free, 0));
        if (!in.dev_depth) {
            void *dst = scale > 0.0f ? static_cast<void *>(v->staged(v->d_depth16, s0, pixels)) : raw_depth;
            B2V_CUDA(v, cudaMemcpyAsync(dst, depth, pixels * depth_bytes * count, cudaMemcpyHostToDevice, v->copy));
            depth = dst;
        }
        if (!in.dev_color) {
            B2V_CUDA(v, cudaMemcpyAsync(raw_color, color, pixels * 3 * count, cudaMemcpyHostToDevice, v->copy));
            color = raw_color;
        }
        B2V_CUDA(v, cudaEventRecord(ev_ready, v->copy));
        B2V_CUDA(v, cudaStreamWaitEvent(as, ev_ready, 0));
    }
    if (scale > 0.0f) {  // widen into the float slots: float(u16) * scale, one rounding
        B2V_CUDA(v, launch_depth_u16_to_f32(static_cast<const uint16_t *>(depth), raw_depth, pixels * count, scale, as));
        depth = raw_depth;
        v->launches += 1;
    }
    for (int k = 0; k < count; ++k) {
        d_depth[k] = static_cast<const float *>(depth) + pixels * k;
        d_color[k] = color + pixels * 3 * k;
    }
    if (!v->d_mapx) return B2V_OK;
    if (in.H != v->rect_H || in.W != v->rect_W) {
        v->err = "rectification maps were installed for a different image size";
        return B2V_ERR_INVALID_ARGUMENT;
    }
    for (int k = 0; k < count; ++k) {
        float *rdepth = v->staged(v->d_rdepth, s0, pixels, k);
        uint8_t *rcolor = v->staged(v->d_rcolor, s0, pixels, k, 3);
        B2V_CUDA(v, launch_remap_b32_nearest(d_depth[k], in.H, in.W, v->d_mapx, v->d_mapy, rdepth, as));
        B2V_CUDA(v, launch_remap_u8c3_linear(d_color[k], in.H, in.W, v->d_mapx, v->d_mapy, rcolor, v->rect_swap, as));
        d_depth[k] = rdepth;
        d_color[k] = rcolor;
        v->launches += 2;
    }
    return B2V_OK;
}

// frame f of `in` (pose Tcw) through allocate_kernel + integrate_kernel, staged in the per-frame ring of slots
static int integrate_frame(b2v_volume *v, const FrameImages &in, size_t f, const double K[4], const double Tcw[16],
                           void *stream) {
    cudaStream_t cs = stream ? static_cast<cudaStream_t>(stream) : v->compute;
    cudaStream_t as = v->overlap ? v->alloc : cs;  // stream of the allocate kernel
    v->last_stream = stream ? cs : nullptr;
    const int s = kGroupStage + static_cast<int>(v->frame_id % kFrameStage);
    const int ring = static_cast<int>(v->frame_id % kActiveRing);
    const size_t pixels = static_cast<size_t>(in.H) * in.W;
    const bool staged = !(in.dev_depth && in.dev_color);
    const bool u16 = in.depth.u16_scale > 0.0f;
    int rc = ensure_staging(v, pixels, u16, false);
    if (rc != B2V_OK) return rc;
    if (!staged && v->overlap && !v->inputs_fenced) {
        // device inputs were produced by earlier work on the caller's stream (a batch call fences once:
        // an event recorded now would also wait for the previous frame's integrate kernel)
        B2V_CUDA(v, cudaEventRecord(v->ev_in, cs));
        B2V_CUDA(v, cudaStreamWaitEvent(as, v->ev_in, 0));
    }
    if (v->rings_stale) {
        // first single frame after a fused batch: the batch advanced frame_id without passing through the
        // per-frame rings, so the ring this frame counts into may still hold an old frame's counts (only the
        // previous per-frame allocate re-arms the next ring).  Rare transition: order it after everything on the
        // compute stream and clear all ring counters.
        B2V_CUDA(v, cudaEventRecord(v->ev_in, cs));
        B2V_CUDA(v, cudaStreamWaitEvent(as, v->ev_in, 0));
        B2V_CUDA(v, cudaMemsetAsync(v->meta.counters + kCtrActive0, 0, 2 * kActiveRing * sizeof(uint32_t), as));
        v->rings_stale = false;
    } else if (v->overlap && v->frame_id >= 3) {
        // allocate(f) recycles the ring slot / texel buffer last read by integrate(f - 3) .. (f - 4)
        B2V_CUDA(v, cudaStreamWaitEvent(as, v->ev_int_done[(v->frame_id - 3) % kActiveRing], 0));
    }
    const float *d_depth;
    const uint8_t *d_color;
    rc = prepare_frames(v, in, f, 1, s, v->ev_free[s], v->ev_ready[s], as, &d_depth, &d_color);
    if (rc != B2V_OK) return rc;
    FrameParams P;
    fill_frame_params(&P, K, Tcw, in.H, in.W, v->geo, v->frame_id + 1);
    rc = refresh_lambda(v, P, K, in.H, in.W, as);
    if (rc != B2V_OK) return rc;
    cudaEvent_t *pe;
    rc = profile_events(v, 1, &pe);
    if (rc != B2V_OK) return rc;
    if (pe) B2V_CUDA(v, cudaEventRecord(pe[0], as));
    float4 *tex = v->staged(v->d_texel, s - kGroupStage, pixels);
    P.I.tex = tex;
    B2V_CUDA(v, launch_allocate(P, d_depth, d_color, v->d_lambda, tex, v->table, v->meta, ring,
                                frame_maps(v, d_depth, d_color, in.H, in.W), &v->lam_map, as));
    if (staged || u16) B2V_CUDA(v, cudaEventRecord(v->ev_free[s], as));  // the raw frame is consumed by allocate only
    v->launches += 1;
    v->frame_id += 1;
    v->last_group_buf = -1;
    if (pe) B2V_CUDA(v, cudaEventRecord(pe[1], as));
    if (v->overlap) {
        B2V_CUDA(v, cudaEventRecord(v->ev_alloc_done[ring], as));
        B2V_CUDA(v, cudaStreamWaitEvent(cs, v->ev_alloc_done[ring], 0));
    }
    if (pe) B2V_CUDA(v, cudaEventRecord(pe[2], cs));
    B2V_CUDA(v, launch_integrate(P, volume_consts(v->geo), v->table, v->meta, ring, v->grid_ctas, cs));
    if (pe) B2V_CUDA(v, cudaEventRecord(pe[3], cs));
    if (v->overlap) B2V_CUDA(v, cudaEventRecord(v->ev_int_done[ring], cs));
    v->launches += 1;
    return B2V_OK;
}

extern "C" int b2v_integrate(b2v_volume *v, const float *depth, const uint8_t *color, int32_t height,
                             int32_t width, const double K[4], const double Tcw[16], void *stream) {
    if (!v) return B2V_ERR_INVALID_ARGUMENT;
    FrameImages in{{depth, 0.0f}, color, height, width};
    const int rc = check_integrate(v, "b2v_integrate", false, 1, &in, K, Tcw, stream);
    return rc != B2V_OK ? rc : integrate_frame(v, in, 0, K, Tcw, stream);
}

extern "C" int b2v_set_rectification(b2v_volume *v, const float *map_x, const float *map_y, int32_t height,
                                     int32_t width, int32_t swap_rb) {
    if (!v) return B2V_ERR_INVALID_ARGUMENT;
    B2V_CUDA(v, cudaSetDevice(v->cfg.device));
    B2V_CUDA(v, cudaDeviceSynchronize());  // remap kernels on any stream may still read the maps and rectified slots
    cudaFree(v->d_mapx);
    cudaFree(v->d_mapy);
    cudaFree(v->d_rdepth);
    cudaFree(v->d_rcolor);
    v->d_mapx = v->d_mapy = v->d_rdepth = nullptr;
    v->d_rcolor = nullptr;  // ensure_staging allocates the rectified slots while maps are installed
    v->rect_H = v->rect_W = 0;
    v->rect_swap = swap_rb;
    v->map_cache.clear();
    if (!map_x || !map_y) return B2V_OK;
    if (height <= 0 || width <= 0) {
        v->err = "b2v_set_rectification: bad image size";
        return B2V_ERR_INVALID_ARGUMENT;
    }
    const size_t pixels = static_cast<size_t>(height) * width;
    B2V_CUDA(v, cudaMalloc(&v->d_mapx, pixels * sizeof(float)));
    B2V_CUDA(v, cudaMalloc(&v->d_mapy, pixels * sizeof(float)));
    B2V_CUDA(v, cudaMemcpy(v->d_mapx, map_x, pixels * sizeof(float), cudaMemcpyHostToDevice));
    B2V_CUDA(v, cudaMemcpy(v->d_mapy, map_y, pixels * sizeof(float), cudaMemcpyHostToDevice));
    v->rect_H = height;
    v->rect_W = width;
    return B2V_OK;
}

extern "C" int b2v_remap(const void *src, int32_t kind, int32_t height, int32_t width, const float *map_x,
                         const float *map_y, void *dst, int32_t swap_rb, int32_t device) {
    if (!src || !dst || !map_x || !map_y || height <= 0 || width <= 0 || (kind != 0 && kind != 1))
        return B2V_ERR_INVALID_ARGUMENT;
    if (cudaSetDevice(device) != cudaSuccess) return B2V_ERR_CUDA;
    const size_t pixels = static_cast<size_t>(height) * width;
    const size_t bytes = pixels * (kind == 0 ? 3 : 4);
    void *d_src = nullptr, *d_dst = nullptr;
    float *d_mx = nullptr, *d_my = nullptr;
    cudaError_t e = cudaMalloc(&d_src, bytes);
    if (e == cudaSuccess) e = cudaMalloc(&d_dst, bytes);
    if (e == cudaSuccess) e = cudaMalloc(&d_mx, pixels * sizeof(float));
    if (e == cudaSuccess) e = cudaMalloc(&d_my, pixels * sizeof(float));
    if (e == cudaSuccess) e = cudaMemcpy(d_src, src, bytes, cudaMemcpyHostToDevice);
    if (e == cudaSuccess) e = cudaMemcpy(d_mx, map_x, pixels * sizeof(float), cudaMemcpyHostToDevice);
    if (e == cudaSuccess) e = cudaMemcpy(d_my, map_y, pixels * sizeof(float), cudaMemcpyHostToDevice);
    if (e == cudaSuccess)
        e = kind == 0 ? launch_remap_u8c3_linear(static_cast<const uint8_t *>(d_src), height, width, d_mx, d_my,
                                                 static_cast<uint8_t *>(d_dst), swap_rb, nullptr)
                      : launch_remap_b32_nearest(d_src, height, width, d_mx, d_my, d_dst, nullptr);
    if (e == cudaSuccess) e = cudaDeviceSynchronize();
    if (e == cudaSuccess) e = cudaMemcpy(dst, d_dst, bytes, cudaMemcpyDeviceToHost);
    cudaFree(d_src);
    cudaFree(d_dst);
    cudaFree(d_mx);
    cudaFree(d_my);
    return e == cudaSuccess ? B2V_OK : B2V_ERR_CUDA;
}

// the frames of `in` in fused groups of group_frames: per group, the uploads, ONE allocate_group launch and ONE
// integrate_group launch (frame by frame when fusion is off)
static int integrate_batch(b2v_volume *v, int32_t n_frames, const FrameImages &in, const double K[4],
                           const double *Tcw, void *stream) {
    cudaStream_t cs = stream ? static_cast<cudaStream_t>(stream) : v->compute;
    cudaStream_t as = v->overlap ? v->alloc : cs;
    const bool dev_inputs = in.dev_depth && in.dev_color;
    struct FenceGuard {  // every exit path (errors included) drops the batch-wide input fence
        b2v_volume *v;
        ~FenceGuard() { v->inputs_fenced = false; }
    } fence_guard{v};
    if (v->overlap) {
        // one fence for the whole batch: by default everything enqueued on the caller's stream so far (the inputs'
        // producers, earlier per-frame work) happens before the batch's allocate kernels.  A caller that knows better
        // (b2v_set_input_event: "the inputs are ready when this event fires") keeps the allocate kernels of this batch
        // from also waiting for the update kernels of the previous one.
        if (v->input_event && dev_inputs) {
            B2V_CUDA(v, cudaStreamWaitEvent(v->alloc, v->input_event, 0));
        } else {
            B2V_CUDA(v, cudaEventRecord(v->ev_in, cs));
            B2V_CUDA(v, cudaStreamWaitEvent(v->alloc, v->ev_in, 0));
        }
        v->inputs_fenced = true;
    } else if (v->input_event && dev_inputs) {
        B2V_CUDA(v, cudaStreamWaitEvent(cs, v->input_event, 0));
    }
    v->input_event = nullptr;
    int rc = B2V_OK;
    if (!v->fuse || n_frames < 2) {
        for (int32_t f = 0; f < n_frames && rc == B2V_OK; ++f)
            rc = integrate_frame(v, in, f, K, Tcw + 16 * static_cast<size_t>(f), stream);
        return rc;
    }
    const size_t pixels = static_cast<size_t>(in.H) * in.W;
    rc = ensure_staging(v, pixels, in.depth.u16_scale > 0.0f, true);
    if (rc != B2V_OK) return rc;
    v->rings_stale = true;
    v->last_stream = stream ? cs : nullptr;
    const int gsz = std::max(1, std::min(v->group_frames, kMaxGroup));
    for (int32_t g0 = 0; g0 < n_frames; g0 += gsz) {
        const int count = std::min<int32_t>(gsz, n_frames - g0);
        const int buf = static_cast<int>(v->group_id % kGroupBufs);
        const int s0 = buf * kMaxGroup;
        // the group buffer (masks, union list, texel images) was last used by group id - kGroupBufs
        B2V_CUDA(v, cudaStreamWaitEvent(as, v->ev_group_done[buf], 0));
        B2V_CUDA(v, cudaMemsetAsync(v->meta.counters + group_ctr(buf, 0), 0, kGroupCtrStride * sizeof(uint32_t), as));
        static thread_local GroupAllocArgs aargs;  // ~15 KB: keep it off the stack
        static thread_local GroupArgs args;
        std::memset(&args, 0, sizeof(args));
        args.V = volume_consts(v->geo);
        args.count = count;
        aargs.count = count;
        aargs.use_tma = 1;
        for (int k = 0; k < count; ++k) {
            FrameParams P;
            fill_frame_params(&P, K, Tcw + 16 * static_cast<size_t>(g0 + k), in.H, in.W, v->geo, v->frame_id + 1);
            P.group_bit = k;
            P.group_buf = buf;
            aargs.pose[k] = P.pose;
            if (k == 0) {
                aargs.P = P;
                aargs.frame_id0 = v->frame_id + 1;
                rc = refresh_lambda(v, P, K, in.H, in.W, as);
                if (rc != B2V_OK) return rc;
            }
            float4 *tex = v->staged(v->d_gtex, s0, pixels, k);
            aargs.tex[k] = tex;
            P.I.tex = tex;
            args.f[k] = P.I;
            v->frame_id += 1;
        }
        // the raw slots of this buffer were consumed by the allocate launch of group id - kGroupBufs
        rc = prepare_frames(v, in, g0, count, s0, v->ev_galloc[buf], v->ev_ready[buf], as, aargs.depth, aargs.color);
        if (rc != B2V_OK) return rc;
        for (int k = 0; k < count; ++k) {  // the TMA descriptors of the final images
            const FrameMaps *fm = frame_maps(v, aargs.depth[k], aargs.color[k], in.H, in.W);
            if (fm) aargs.maps[k] = *fm; else aargs.use_tma = 0;
        }
        cudaEvent_t *pe;
        rc = profile_events(v, count, &pe);
        if (rc != B2V_OK) return rc;
        if (pe) B2V_CUDA(v, cudaEventRecord(pe[0], as));
        aargs.lmap = v->lam_map;
        B2V_CUDA(v, launch_allocate_group(aargs, v->d_lambda, v->table, v->meta, as));
        if (pe) B2V_CUDA(v, cudaEventRecord(pe[1], as));
        B2V_CUDA(v, cudaEventRecord(v->ev_galloc[buf], as));
        if (v->overlap) B2V_CUDA(v, cudaStreamWaitEvent(cs, v->ev_galloc[buf], 0));
        if (pe) B2V_CUDA(v, cudaEventRecord(pe[2], cs));
        B2V_CUDA(v, launch_integrate_group(args, v->table, v->meta, buf, v->grid_ctas, cs));
        if (pe) B2V_CUDA(v, cudaEventRecord(pe[3], cs));
        B2V_CUDA(v, cudaEventRecord(v->ev_group_done[buf], cs));
        v->launches += 3;
        v->last_group_buf = buf;
        v->last_group_count = count;
        v->group_id += 1;
    }
    return B2V_OK;
}

extern "C" int b2v_integrate_batch(b2v_volume *v, int32_t n_frames, const float *depth,
                                   const uint8_t *color, int32_t height, int32_t width,
                                   const double K[4], const double *Tcw, void *stream) {
    if (!v) return B2V_ERR_INVALID_ARGUMENT;
    FrameImages in{{depth, 0.0f}, color, height, width};
    const int rc = check_integrate(v, "b2v_integrate_batch", false, n_frames, &in, K, Tcw, stream);
    return rc != B2V_OK || n_frames == 0 ? rc : integrate_batch(v, n_frames, in, K, Tcw, stream);
}

// Raw 16-bit depth (e.g. TUM / ScanNet PNGs): uploaded as uint16 (2 instead of 4 bytes per pixel over PCIe) and
// widened on the device to float(u16) * depth_scale in float32 - the value numpy's
// `depth.astype(np.float32) * depth_factor` produces (volumetric_integrator_base.py:1008-1015).
extern "C" int b2v_integrate_batch_u16(b2v_volume *v, int32_t n_frames, const uint16_t *depth, float depth_scale,
                                       const uint8_t *color, int32_t height, int32_t width, const double K[4],
                                       const double *Tcw, void *stream) {
    if (!v) return B2V_ERR_INVALID_ARGUMENT;
    FrameImages in{{depth, depth_scale}, color, height, width};
    const int rc = check_integrate(v, "b2v_integrate_batch_u16", true, n_frames, &in, K, Tcw, stream);
    return rc != B2V_OK || n_frames == 0 ? rc : integrate_batch(v, n_frames, in, K, Tcw, stream);
}

extern "C" int b2v_integrate_u16(b2v_volume *v, const uint16_t *depth, float depth_scale, const uint8_t *color,
                                 int32_t height, int32_t width, const double K[4], const double Tcw[16],
                                 void *stream) {
    if (!v) return B2V_ERR_INVALID_ARGUMENT;
    FrameImages in{{depth, depth_scale}, color, height, width};
    const int rc = check_integrate(v, "b2v_integrate_u16", true, 1, &in, K, Tcw, stream);
    return rc != B2V_OK ? rc : integrate_frame(v, in, 0, K, Tcw, stream);
}

extern "C" int b2v_set_input_event(b2v_volume *v, void *event) {
    if (!v) return B2V_ERR_INVALID_ARGUMENT;
    v->input_event = static_cast<cudaEvent_t>(event);
    return B2V_OK;
}

extern "C" int b2v_set_group_size(b2v_volume *v, int32_t frames) {
    if (!v) return B2V_ERR_INVALID_ARGUMENT;
    if (frames < 1 || frames > kMaxGroup) {
        v->err = "b2v_set_group_size: 1..32 frames";
        return B2V_ERR_INVALID_ARGUMENT;
    }
    const int rc = read_counters(v);
    if (rc == B2V_ERR_CUDA) return rc;
    v->group_frames = frames;
    return B2V_OK;
}

extern "C" int b2v_set_fusion(b2v_volume *v, int32_t enable) {
    if (!v) return B2V_ERR_INVALID_ARGUMENT;
    const int rc = read_counters(v);
    if (rc == B2V_ERR_CUDA) return rc;
    v->fuse = enable != 0;
    return B2V_OK;
}

extern "C" int b2v_synchronize(b2v_volume *v) {
    if (!v) return B2V_ERR_INVALID_ARGUMENT;
    return read_counters(v);
}

extern "C" int64_t b2v_num_blocks(b2v_volume *v) {
    if (!v) return -1;
    const int rc = read_counters(v);
    if (rc == B2V_ERR_CUDA) return -1;
    return block_count(v);
}

extern "C" int b2v_last_frame_stats(b2v_volume *v, int64_t *touched_blocks, int64_t *new_blocks) {
    if (!v) return B2V_ERR_INVALID_ARGUMENT;
    const int rc = read_counters(v);
    if (rc == B2V_ERR_CUDA) return rc;
    const int ring = v->frame_id ? static_cast<int>((v->frame_id - 1) % kActiveRing) : 0;
    if (touched_blocks) {
        if (v->frame_id == 0)
            *touched_blocks = 0;
        else if (v->last_group_buf >= 0)
            *touched_blocks = v->h_counters[group_ctr(v->last_group_buf, kGcTouched0) + v->last_group_count - 1];
        else
            *touched_blocks = v->h_counters[kCtrActive0 + ring];
    }
    if (new_blocks) {
        if (v->frame_id == 0)
            *new_blocks = 0;
        else if (v->last_group_buf >= 0)  // after a fused batch: blocks allocated by the last group
            *new_blocks = v->h_counters[group_ctr(v->last_group_buf, kGcNew)];
        else
            *new_blocks = v->h_counters[kCtrNew0 + ring];
    }
    return rc;
}

extern "C" int b2v_set_overlap(b2v_volume *v, int32_t enable) {
    if (!v) return B2V_ERR_INVALID_ARGUMENT;
    const int rc = read_counters(v);  // drains every stream first
    if (rc == B2V_ERR_CUDA) return rc;
    v->overlap = enable != 0;
    return B2V_OK;
}

extern "C" int b2v_profile_enable(b2v_volume *v, int32_t enable) {
    if (!v) return B2V_ERR_INVALID_ARGUMENT;
    v->prof_enabled = enable != 0;
    v->prof_used = 0;
    v->prof_frames = 0;
    v->prof_int_launches = 0;
    return B2V_OK;
}

extern "C" int b2v_profile_read(b2v_volume *v, double *allocate_ms, double *integrate_ms, int64_t *frames,
                                int64_t *integrate_launches) {
    if (!v) return B2V_ERR_INVALID_ARGUMENT;
    B2V_CUDA(v, cudaSetDevice(v->cfg.device));
    double a = 0.0, b = 0.0;
    for (size_t k = 0; k + 3 < v->prof_used; k += 4) {
        B2V_CUDA(v, cudaEventSynchronize(v->prof_events[k + 1]));
        B2V_CUDA(v, cudaEventSynchronize(v->prof_events[k + 3]));
        float ms = 0.0f;
        B2V_CUDA(v, cudaEventElapsedTime(&ms, v->prof_events[k], v->prof_events[k + 1]));
        a += ms;
        B2V_CUDA(v, cudaEventElapsedTime(&ms, v->prof_events[k + 2], v->prof_events[k + 3]));
        b += ms;
    }
    if (allocate_ms) *allocate_ms = a;
    if (integrate_ms) *integrate_ms = b;
    if (frames) *frames = v->prof_frames;
    if (integrate_launches) *integrate_launches = v->prof_int_launches;
    v->prof_used = 0;
    v->prof_frames = 0;
    v->prof_int_launches = 0;
    return B2V_OK;
}

extern "C" int b2v_counters(b2v_volume *v, int64_t *block_updates, int64_t *kernel_launches,
                            int64_t *block_visits) {
    if (!v) return B2V_ERR_INVALID_ARGUMENT;
    const int rc = read_counters(v);
    if (rc == B2V_ERR_CUDA) return rc;
    if (block_updates)
        *block_updates = static_cast<int64_t>(static_cast<uint64_t>(v->h_counters[kCtrUpdatesLo]) |
                                              (static_cast<uint64_t>(v->h_counters[kCtrUpdatesHi]) << 32));
    if (kernel_launches) *kernel_launches = v->launches;
    if (block_visits)
        *block_visits = static_cast<int64_t>(static_cast<uint64_t>(v->h_counters[kCtrVisitsLo]) |
                                             (static_cast<uint64_t>(v->h_counters[kCtrVisitsHi]) << 32));
    return rc;
}

extern "C" int64_t b2v_dump_blocks(b2v_volume *v, int32_t *keys, uint64_t *hashes, float *voxels) {
    if (!v) return -1;
    if (read_counters(v) == B2V_ERR_CUDA) return -1;
    const uint32_t nb = block_count(v);
    if (nb == 0) return 0;
    if (keys) {
        std::vector<int4> tmp(nb);
        if (cudaMemcpy(tmp.data(), v->meta.block_keys, nb * sizeof(int4), cudaMemcpyDeviceToHost) != cudaSuccess)
            return -1;
        for (uint32_t i = 0; i < nb; ++i) {
            keys[3 * i + 0] = tmp[i].x;
            keys[3 * i + 1] = tmp[i].y;
            keys[3 * i + 2] = tmp[i].z;
        }
    }
    if (hashes) {
        uint64_t *d_h = nullptr;
        if (cudaMalloc(&d_h, nb * sizeof(uint64_t)) != cudaSuccess) return -1;
        cudaError_t e = launch_block_hashes(v->meta.block_keys, d_h, nb, v->compute);
        if (e == cudaSuccess) e = cudaStreamSynchronize(v->compute);
        if (e == cudaSuccess) e = cudaMemcpy(hashes, d_h, nb * sizeof(uint64_t), cudaMemcpyDeviceToHost);
        cudaFree(d_h);
        v->launches += 1;
        if (e != cudaSuccess) return -1;
    }
    if (voxels) {
        if (cudaMemcpy(voxels, v->meta.pool, static_cast<size_t>(nb) * kBlockFloats * sizeof(float),
                       cudaMemcpyDeviceToHost) != cudaSuccess)
            return -1;
    }
    return nb;
}

extern "C" int b2v_upload_blocks(b2v_volume *v, int64_t n_blocks, const int32_t *keys, const float *voxels) {
    if (!v) return B2V_ERR_INVALID_ARGUMENT;
    if (n_blocks < 0 || (n_blocks > 0 && (!keys || !voxels))) {
        v->err = "b2v_upload_blocks: bad arguments";
        return B2V_ERR_INVALID_ARGUMENT;
    }
    if (n_blocks == 0) return B2V_OK;
    B2V_CUDA(v, cudaSetDevice(v->cfg.device));
    const size_t n = static_cast<size_t>(n_blocks);
    std::vector<int4> k4(n);
    for (size_t i = 0; i < n; ++i) k4[i] = make_int4(keys[3 * i], keys[3 * i + 1], keys[3 * i + 2], 0);
    int4 *d_k = nullptr;
    float *d_v = nullptr;
    uint32_t *d_i = nullptr;
    cudaError_t e = cudaMalloc(&d_k, n * sizeof(int4));
    if (e == cudaSuccess) e = cudaMalloc(&d_v, n * kBlockFloats * sizeof(float));
    if (e == cudaSuccess) e = cudaMalloc(&d_i, n * sizeof(uint32_t));
    if (e == cudaSuccess) e = cudaMemcpyAsync(d_k, k4.data(), n * sizeof(int4), cudaMemcpyHostToDevice, v->compute);
    if (e == cudaSuccess)
        e = cudaMemcpyAsync(d_v, voxels, n * kBlockFloats * sizeof(float), cudaMemcpyHostToDevice, v->compute);
    if (e == cudaSuccess)
        e = launch_upload_blocks(d_k, d_v, static_cast<uint32_t>(n), d_i, v->table, v->meta, v->compute);
    if (e == cudaSuccess) e = cudaStreamSynchronize(v->compute);
    cudaFree(d_k);
    cudaFree(d_v);
    cudaFree(d_i);
    v->launches += 2;
    if (e != cudaSuccess) {
        v->err = std::string("b2v_upload_blocks: ") + cudaGetErrorString(e);
        return B2V_ERR_CUDA;
    }
    return read_counters(v);
}

// Device-to-device block exchange (multi-GPU mesh gather, SURVEY.md 8e): keys as int32 x 4 {x, y, z, 0}
extern "C" int64_t b2v_export_blocks_device(b2v_volume *v, int32_t *d_keys4, float *d_voxels, int64_t max_blocks) {
    if (!v) return -1;
    if (read_counters(v) == B2V_ERR_CUDA) return -1;
    const uint32_t nb = block_count(v);
    if (!d_keys4 && !d_voxels) return nb;
    if (static_cast<int64_t>(nb) > max_blocks) {
        v->err = "b2v_export_blocks_device: destination too small";
        return -1;
    }
    if (nb == 0) return 0;
    cudaError_t e = cudaSuccess;
    if (d_keys4) e = cudaMemcpyAsync(d_keys4, v->meta.block_keys, nb * sizeof(int4), cudaMemcpyDeviceToDevice, v->compute);
    if (e == cudaSuccess && d_voxels)
        e = cudaMemcpyAsync(d_voxels, v->meta.pool, static_cast<size_t>(nb) * kBlockFloats * sizeof(float),
                            cudaMemcpyDeviceToDevice, v->compute);
    if (e == cudaSuccess) e = cudaStreamSynchronize(v->compute);
    if (e != cudaSuccess) {
        v->err = std::string("b2v_export_blocks_device: ") + cudaGetErrorString(e);
        return -1;
    }
    return nb;
}

extern "C" int b2v_import_blocks_device(b2v_volume *v, int64_t n_blocks, const int32_t *d_keys4, const float *d_voxels) {
    if (!v) return B2V_ERR_INVALID_ARGUMENT;
    if (n_blocks < 0 || (n_blocks > 0 && (!d_keys4 || !d_voxels))) {
        v->err = "b2v_import_blocks_device: bad arguments";
        return B2V_ERR_INVALID_ARGUMENT;
    }
    if (n_blocks == 0) return B2V_OK;
    B2V_CUDA(v, cudaSetDevice(v->cfg.device));
    uint32_t *d_i = nullptr;
    cudaError_t e = cudaMalloc(&d_i, static_cast<size_t>(n_blocks) * sizeof(uint32_t));
    if (e == cudaSuccess)
        e = launch_upload_blocks(reinterpret_cast<const int4 *>(d_keys4), d_voxels, static_cast<uint32_t>(n_blocks), d_i,
                                 v->table, v->meta, v->compute);
    if (e == cudaSuccess) e = cudaStreamSynchronize(v->compute);
    cudaFree(d_i);
    v->launches += 2;
    if (e != cudaSuccess) {
        v->err = std::string("b2v_import_blocks_device: ") + cudaGetErrorString(e);
        return B2V_ERR_CUDA;
    }
    return read_counters(v);
}

extern "C" int64_t b2v_last_touched_keys(b2v_volume *v, int32_t *keys, int64_t max_keys) {
    if (!v) return -1;
    if (read_counters(v) == B2V_ERR_CUDA) return -1;
    if (v->frame_id == 0) return 0;
    const int ring = static_cast<int>((v->frame_id - 1) % kActiveRing);
    const bool grp = v->last_group_buf >= 0;  // after a fused batch: the last group's union of touched blocks
    uint32_t n = grp ? v->h_counters[group_ctr(v->last_group_buf, kGcUnion)] : v->h_counters[kCtrActive0 + ring];
    if (n > v->meta.capacity) n = v->meta.capacity;
    if (!keys) return n;
    if (static_cast<int64_t>(n) > max_keys) n = static_cast<uint32_t>(max_keys);
    if (n == 0) return 0;
    int4 *d_k = nullptr;
    if (cudaMalloc(&d_k, n * sizeof(int4)) != cudaSuccess) return -1;
    std::vector<int4> tmp(n);
    const uint32_t *list = grp ? v->meta.union_slots + static_cast<size_t>(v->last_group_buf) * v->meta.capacity
                               : v->meta.active_slots + static_cast<size_t>(ring) * v->meta.capacity;
    cudaError_t e = launch_gather_active_keys(v->table, list, n, d_k, v->compute);
    if (e == cudaSuccess) e = cudaStreamSynchronize(v->compute);
    if (e == cudaSuccess) e = cudaMemcpy(tmp.data(), d_k, n * sizeof(int4), cudaMemcpyDeviceToHost);
    cudaFree(d_k);
    v->launches += 1;
    if (e != cudaSuccess) return -1;
    for (uint32_t i = 0; i < n; ++i) {
        keys[3 * i + 0] = tmp[i].x;
        keys[3 * i + 1] = tmp[i].y;
        keys[3 * i + 2] = tmp[i].z;
    }
    return n;
}

// ---- mesh / point cloud ---------------------------------------------------------------------

static int ensure_mesh_scratch(b2v_volume *v, uint32_t nb) {
    if (!v->mb.totals) B2V_CUDA(v, cudaMalloc(&v->mb.totals, kNumMeshTotals * sizeof(uint32_t)));
    if (nb <= v->mesh_blocks_cap) return B2V_OK;
    const size_t n = nb;
    B2V_CUDA(v, regrow(&v->mb.nbr, n * 8));
    B2V_CUDA(v, regrow(&v->mb.cube, n * kVox));
    B2V_CUDA(v, regrow(&v->mb.edge_mask, n * (kVox / 4)));
    B2V_CUDA(v, regrow(&v->mb.local, n * kVox));
    B2V_CUDA(v, regrow(&v->mb.sums, n * 2));
    B2V_CUDA(v, regrow(&v->mb.offs, n * 2));
    B2V_CUDA(v, regrow(&v->mb.partials, 2 * ((n + 1023) / 1024)));
    B2V_CUDA(v, regrow(&v->mb.work, n * 4));
    v->mesh_blocks_cap = nb;
    return B2V_OK;
}

static int extract_common(b2v_volume *v, bool mesh, int64_t *n_vertices, int64_t *n_triangles) {
    int rc = read_counters(v);
    if (rc == B2V_ERR_CUDA) return rc;
    const uint32_t nb = block_count(v);
    rc = ensure_mesh_scratch(v, nb);
    if (rc != B2V_OK) return rc;
    v->mb.n_blocks = nb;
    cudaStream_t cs = v->compute;
    const int sms = v->sm_count > 0 ? v->sm_count : 148;
    if (mesh) {
        B2V_CUDA(v, launch_mesh_classify(v->table, v->meta, v->mb, sms, cs));
    } else {
        B2V_CUDA(v, launch_point_masks(v->table, v->meta, v->mb, sms, cs));
    }
    B2V_CUDA(v, launch_mesh_scan(v->mb, sms, cs));
    B2V_CUDA(v, cudaMemcpyAsync(v->h_totals, v->mb.totals, kNumMeshTotals * sizeof(uint32_t), cudaMemcpyDeviceToHost, cs));
    B2V_CUDA(v, cudaStreamSynchronize(cs));
    const size_t nv = v->h_totals[kMtVertices], nt = v->h_totals[kMtTriangles];
    if (nv > v->mesh_v_cap) {
        B2V_CUDA(v, regrow(&v->mb.vertices, nv * 3));
        B2V_CUDA(v, regrow(&v->mb.colors, nv * 3));
        B2V_CUDA(v, regrow(&v->mb.edge_ids, nv * 4));
        v->mesh_v_cap = nv;
    }
    if (nt > v->mesh_t_cap) {
        B2V_CUDA(v, regrow(&v->mb.triangles, nt * 3));
        v->mesh_t_cap = nt;
    }
    B2V_CUDA(v, launch_mesh_vertices(v->meta, v->mb, v->geo.voxel_length, v->geo.unit_shift, !mesh, v->h_totals[kMtVertexBlocks], cs));
    if (mesh) B2V_CUDA(v, launch_mesh_triangles(v->mb, v->h_totals[kMtTriangleBlocks], cs));
    B2V_CUDA(v, cudaStreamSynchronize(cs));
    v->launches += mesh ? 6 : 5;
    v->last_nv = static_cast<int64_t>(nv);
    v->last_nt = mesh ? static_cast<int64_t>(nt) : 0;
    if (n_vertices) *n_vertices = v->last_nv;
    if (n_triangles) *n_triangles = v->last_nt;
    return rc;
}

extern "C" int b2v_last_mesh_stats(b2v_volume *v, int64_t stats[5]) {
    if (!v || !stats) return B2V_ERR_INVALID_ARGUMENT;
    stats[0] = v->mb.n_blocks;
    stats[1] = v->h_totals[kMtCandidates];
    stats[2] = v->h_totals[kMtTiles];
    stats[3] = v->h_totals[kMtVertexBlocks];
    stats[4] = v->h_totals[kMtTriangleBlocks];
    return B2V_OK;
}

extern "C" int b2v_extract_mesh(b2v_volume *v, int64_t *n_vertices, int64_t *n_triangles) {
    if (!v) return B2V_ERR_INVALID_ARGUMENT;
    return extract_common(v, true, n_vertices, n_triangles);
}

extern "C" int b2v_copy_mesh(b2v_volume *v, double *vertices, double *colors, int32_t *edge_ids,
                             int32_t *triangles) {
    if (!v) return B2V_ERR_INVALID_ARGUMENT;
    const size_t nv = static_cast<size_t>(v->last_nv), nt = static_cast<size_t>(v->last_nt);
    if (vertices && nv) B2V_CUDA(v, cudaMemcpy(vertices, v->mb.vertices, nv * 3 * sizeof(double), cudaMemcpyDeviceToHost));
    if (colors && nv) B2V_CUDA(v, cudaMemcpy(colors, v->mb.colors, nv * 3 * sizeof(double), cudaMemcpyDeviceToHost));
    if (edge_ids && nv) B2V_CUDA(v, cudaMemcpy(edge_ids, v->mb.edge_ids, nv * 4 * sizeof(int32_t), cudaMemcpyDeviceToHost));
    if (triangles && nt) B2V_CUDA(v, cudaMemcpy(triangles, v->mb.triangles, nt * 3 * sizeof(int32_t), cudaMemcpyDeviceToHost));
    return B2V_OK;
}

extern "C" int b2v_extract_points(b2v_volume *v, int64_t *n_points) {
    if (!v) return B2V_ERR_INVALID_ARGUMENT;
    return extract_common(v, false, n_points, nullptr);
}

extern "C" int b2v_copy_points(b2v_volume *v, double *points, double *colors) {
    return b2v_copy_mesh(v, points, colors, nullptr, nullptr);
}

extern "C" int b2v_filter_shadow_points(const float *depth, int32_t height, int32_t width, int32_t delta_x,
                                        int32_t delta_y, float fill_value, float *out, int32_t device) {
    if (!depth || !out || height <= 0 || width <= 0 || delta_x < 0 || delta_y < 0 || delta_x >= width ||
        delta_y >= height)
        return B2V_ERR_INVALID_ARGUMENT;
    if (cudaSetDevice(device) != cudaSuccess) return B2V_ERR_CUDA;
    const size_t pixels = static_cast<size_t>(height) * width;
    const bool din = is_device_pointer(depth), dout = is_device_pointer(out);
    float *d_in = nullptr, *d_out = nullptr;
    void *scratch = nullptr;
    cudaError_t e = cudaMalloc(&scratch, kShadowScratchBytes);
    if (e == cudaSuccess && !din) {
        e = cudaMalloc(&d_in, pixels * sizeof(float));
        if (e == cudaSuccess) e = cudaMemcpy(d_in, depth, pixels * sizeof(float), cudaMemcpyHostToDevice);
    }
    if (e == cudaSuccess && !dout) e = cudaMalloc(&d_out, pixels * sizeof(float));
    if (e == cudaSuccess)
        e = launch_filter_shadow_points(din ? depth : d_in, height, width, delta_x, delta_y, fill_value,
                                        dout ? out : d_out, scratch, nullptr);
    if (e == cudaSuccess) e = cudaDeviceSynchronize();
    if (e == cudaSuccess && !dout) e = cudaMemcpy(out, d_out, pixels * sizeof(float), cudaMemcpyDeviceToHost);
    cudaFree(scratch);
    cudaFree(d_in);
    cudaFree(d_out);
    return e == cudaSuccess ? B2V_OK : B2V_ERR_CUDA;
}
