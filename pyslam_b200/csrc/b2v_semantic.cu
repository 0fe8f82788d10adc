// b2v_semantic.cu — semantic voxel-block grids on sm_100a (SURVEY.md §8(f) rank 2, Appendix D).
//
// Replaces, for the `integrate(points, colors, class_ids, instance_ids, depths)` path and its read-outs,
//   VoxelBlockSemanticGrid               = VoxelBlockSemanticGridT<VoxelSemanticData>               (voting)
//   VoxelBlockSemanticProbabilisticGrid  = VoxelBlockSemanticGridT<VoxelSemanticDataProbabilistic>  (Bayesian)
// (cpp/volumetric/voxel_block_semantic_grid.h:118-121; voxel data: voxel_data_semantic.h:106-199, 249-672;
//  integrate: voxel_block_grid.hpp:12-112, 220-288, 524-614; get_voxels :717-819).
//
// Both label rules are ORDER DEPENDENT in the reference (the voting counter is a sequential state machine; the
// Bayesian argmax keeps the earlier label on ties; float sums round in input order).  The reference's
// deterministic build processes the points of one call in input order, so this implementation does the same
// per voxel:
//   1. insert   one thread per point: block key (bit-exact, in the point's own precision) -> 128-bit-CAS table
//   2. keys     one thread per point: sort key = pool_index * 512 + local voxel index
//   3. sort     stable LSD radix sort of (key, point index) pairs (cub::DeviceRadixSort - library code)
//   4. runs     the first element of every run of equal keys walks its run in input order and applies the
//               reference's per-observation update: count, position_sum (float64), color_sum (float32), labels
// => counts, sums, labels and log-evidence are bit-identical to the sequential reference.  Only exp / log of the
// confidence read-out are evaluated in float64 and rounded (glibc's expf / logf are within 1 ulp of that).
//
// Bayesian labels: the reference keeps a std::map<(object, class), float> per voxel (typically 1-5 entries);
// here a voxel has kSemLabels = 8 fixed slots.  A ninth distinct pair evicts the slot with the least evidence
// that is not the current argmax and bumps the overflow counter (b2v_sgrid_label_overflows) - a documented
// deviation that no test or reference KAT reaches.
#include <cub/device/device_radix_sort.cuh>

#include <climits>
#include <limits>
#include <map>
#include <new>
#include <string>
#include <vector>

#include "../../include/b2v.h"
#include "b2v_points.cuh"
#include "b2v_scan.cuh"

namespace b2v {

constexpr int kSemLabels = B2V_SEM_MAX_LABELS;
constexpr uint32_t kBadVid = 0xFFFFFFFFu;
constexpr float kBaseLogProb = 0.10536051565782628f;  // voxel_data_semantic.h:287, -log(0.9)

// the point-grid counters (GridCounter) + the label slot evictions
enum SemCounter : int { kSemOverflow = kGridNumCounters, kSemNumCounters };

struct SemGrid {
    uint32_t *counters;
    int4 *block_keys;   // [capacity]
    int32_t *count;     // [V]            V = capacity * 512, voxel id = pool index * 512 + lx + 8 ly + 64 lz
    double *pos;        // [V][3]
    float *col;         // [V][3]
    int32_t *obj, *cls; // [V]            current label (voting) / cached argmax (Bayesian)
    int32_t *counter;   // [V]            voting: confidence counter; Bayesian: number of label slots in use
    float *ml_logp;     // [V]            Bayesian: evidence of the argmax
    float *conf;        // [V]            Bayesian: cached confidence
    int32_t *lab_obj, *lab_cls;  // [V][kSemLabels]
    float *lab_logp;             // [V][kSemLabels]
    uint32_t capacity;
    int32_t kind;
    float depth_threshold, depth_decay_rate;
};

// ---- 1. make sure every point's block exists ---------------------------------------------------------------
template <typename T>
__global__ void __launch_bounds__(256)
sem_insert_kernel(const T *__restrict__ pts, const uint8_t *__restrict__ valid, const int64_t n,
                  const float inv_vs, const HashTable H, const SemGrid G) {
    const int64_t i = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
    const bool have = i < n && (valid == nullptr || valid[i]);
    int bx = 0, by = 0, bz = 0;
    if (have) {
        bx = block_coord(point_voxel_coord(pts[3 * i + 0], inv_vs));
        by = block_coord(point_voxel_coord(pts[3 * i + 1], inv_vs));
        bz = block_coord(point_voxel_coord(pts[3 * i + 2], inv_vs));
    }
    insert_block_warp(have, bx, by, bz, H, G.block_keys, G.counters, G.capacity);
}

// ---- 2. sort keys --------------------------------------------------------------------------------------------
template <typename T>
__global__ void __launch_bounds__(256)
sem_keys_kernel(const T *__restrict__ pts, const uint8_t *__restrict__ valid, const int64_t n, const float inv_vs,
                const HashTable H, const SemGrid G, uint32_t *__restrict__ vid, uint32_t *__restrict__ order) {
    const int64_t i = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const int vx = point_voxel_coord(pts[3 * i + 0], inv_vs), vy = point_voxel_coord(pts[3 * i + 1], inv_vs),
              vz = point_voxel_coord(pts[3 * i + 2], inv_vs);
    uint32_t key = kBadVid;
    const uint32_t slot = (valid == nullptr || valid[i])
                              ? table_find(H, block_coord(vx), block_coord(vy), block_coord(vz))
                              : kEmpty;
    if (slot != kEmpty) {
        const uint32_t idx = H.entries[slot].w;
        if (idx < G.capacity)
            key = idx * kVox + static_cast<uint32_t>(local_coord(vx) + (local_coord(vy) << 3) + (local_coord(vz) << 6));
    }
    vid[i] = key;
    order[i] = static_cast<uint32_t>(i);
}

// ---- fused front-end: depth2pointcloud + world transform of one labelled RGBD frame ------------------------
// (pyslam/utilities/depth.py:45-85; pyslam/dense/volumetric_integrator_voxel_semantic_grid.py:392-453).  One
// thread per pixel writes the point record the reference front-end would have produced for it; invalid pixels
// are masked instead of compacted - their sort key is kBadVid, so the per-voxel order of the valid ones is the
// row-major pixel order, i.e. the reference's point order.
__global__ void __launch_bounds__(256)
sem_rgbd_points_kernel(const RgbdParams P, const float *__restrict__ depth, const uint8_t *__restrict__ rgb,
                       const int32_t *__restrict__ class_img, const int32_t *__restrict__ object_img,
                       float *__restrict__ pts, float *__restrict__ cols, int32_t *__restrict__ cls,
                       int32_t *__restrict__ inst, float *__restrict__ depths, uint8_t *__restrict__ valid) {
    const int64_t n = static_cast<int64_t>(P.H) * P.W;
    const int64_t i = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
    if (i >= n) return;
    float pt[3];
    const bool ok = rgbd_point(P, depth, i, pt);
    valid[i] = ok ? 1 : 0;
    if (!ok) return;
#pragma unroll
    for (int a = 0; a < 3; ++a) {
        pts[3 * i + a] = pt[a];
        cols[3 * i + a] = rgbd_color(rgb[3 * i + a]);
    }
    if (class_img) cls[i] = class_img[i];
    if (object_img) inst[i] = object_img[i];
    depths[i] = depth[i];  // points[:, 2] narrowed back to float32 (:408-409) is the depth itself
}

// ---- 4. per-voxel sequential update ------------------------------------------------------------------------
struct SemInputs {
    const void *pts;      // float or double [n][3]
    const void *cols;     // nullptr, float [n][3] or uint8 [n][3]
    const int32_t *cls;   // nullptr or [n]
    const int32_t *inst;  // nullptr or [n]
    const float *depths;  // nullptr or [n]
    int32_t pts_f64, cols_u8;
};

__device__ __forceinline__ float exp_rn(float x) { return __double2float_rn(exp(static_cast<double>(x))); }
__device__ __forceinline__ float log_rn(float x) { return __double2float_rn(log(static_cast<double>(x))); }

// log_add_exp (voxel_data_semantic.h:626-635)
__device__ __forceinline__ float log_add_exp(float a, float b) {
    const float ninf = __uint_as_float(0xFF800000u);
    if (a == ninf) return b;
    if (b == ninf) return a;
    const float m = fmaxf(a, b);
    return __fadd_rn(m, log_rn(__fadd_rn(exp_rn(__fsub_rn(a, m)), exp_rn(__fsub_rn(b, m)))));
}

// confidence of the argmax: exp(max - logsumexp) with the sum folded in std::map order, i.e. ascending
// (object, class) (voxel_data_semantic.h:561-570, 607-624)
__device__ float bayes_confidence(const int32_t *lo, const int32_t *lc, const float *lp, int nl, int mo, int mc,
                                  float mlp) {
    if (mo == -1 || mc == -1 || nl == 0) return 0.0f;
    float sum = __uint_as_float(0xFF800000u);
    long long prev = LLONG_MIN;
    for (int k = 0; k < nl; ++k) {  // selection in key order; nl <= 8
        long long best = LLONG_MAX;
        int bi = -1;
        for (int j = 0; j < nl; ++j) {
            const long long key = (static_cast<long long>(lo[j]) << 32) + (static_cast<long long>(lc[j]) + 0x80000000LL);
            if (key > prev && key < best) {
                best = key;
                bi = j;
            }
        }
        if (bi < 0) break;
        prev = best;
        sum = log_add_exp(sum, lp[bi]);
    }
    return exp_rn(__fsub_rn(mlp, sum));
}

__global__ void __launch_bounds__(128)
sem_runs_kernel(const uint32_t *__restrict__ vid, const uint32_t *__restrict__ order, const int64_t n,
                const SemInputs in, const SemGrid G) {
    const int64_t j0 = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
    if (j0 >= n) return;
    const uint32_t v = vid[j0];
    if (v == kBadVid || (j0 > 0 && vid[j0 - 1] == v)) return;  // not the head of a run

    int32_t count = G.count[v];
    double px = G.pos[3 * static_cast<size_t>(v) + 0], py = G.pos[3 * static_cast<size_t>(v) + 1],
           pz = G.pos[3 * static_cast<size_t>(v) + 2];
    float cr = G.col[3 * static_cast<size_t>(v) + 0], cg = G.col[3 * static_cast<size_t>(v) + 1],
          cb = G.col[3 * static_cast<size_t>(v) + 2];
    int32_t obj = G.obj[v], cls = G.cls[v], ctr = G.counter[v];
    const bool bayes = G.kind == B2V_SEM_PROBABILISTIC;
    const bool semantics = in.cls != nullptr && in.cols != nullptr;  // no colours => positions only (hpp:228-231)
    float mlp = 0.0f;
    int32_t lo[kSemLabels], lc[kSemLabels];
    float lp[kSemLabels];
    int nl = 0;
    if (bayes && semantics) {
        mlp = G.ml_logp[v];
        nl = ctr;
        for (int k = 0; k < kSemLabels; ++k) {
            lo[k] = G.lab_obj[static_cast<size_t>(v) * kSemLabels + k];
            lc[k] = G.lab_cls[static_cast<size_t>(v) * kSemLabels + k];
            lp[k] = G.lab_logp[static_cast<size_t>(v) * kSemLabels + k];
        }
    }

    for (int64_t j = j0; j < n && vid[j] == v; ++j) {
        const uint32_t i = order[j];
        double x, y, z;
        if (in.pts_f64) {
            const double *p = static_cast<const double *>(in.pts) + 3 * static_cast<size_t>(i);
            x = p[0], y = p[1], z = p[2];
        } else {
            const float *p = static_cast<const float *>(in.pts) + 3 * static_cast<size_t>(i);
            x = p[0], y = p[1], z = p[2];
        }
        px = __dadd_rn(px, x);  // voxel_data.h:53-57
        py = __dadd_rn(py, y);
        pz = __dadd_rn(pz, z);
        if (in.cols != nullptr) {  // voxel_data.h:79-90
            float r, g, b;
            if (in.cols_u8) {
                const uint8_t *c = static_cast<const uint8_t *>(in.cols) + 3 * static_cast<size_t>(i);
                const float inv255 = 1.0f / 255.0f;
                r = __fmul_rn(static_cast<float>(c[0]), inv255);
                g = __fmul_rn(static_cast<float>(c[1]), inv255);
                b = __fmul_rn(static_cast<float>(c[2]), inv255);
            } else {
                const float *c = static_cast<const float *>(in.cols) + 3 * static_cast<size_t>(i);
                r = c[0], g = c[1], b = c[2];
            }
            cr = __fadd_rn(cr, r);
            cg = __fadd_rn(cg, g);
            cb = __fadd_rn(cb, b);
        }
        if (semantics) {
            const int32_t oc = in.cls[i];
            const int32_t oo = in.inst ? in.inst[i] : 0;  // no instance ids: object id 0 (hpp:259-286)
            const bool has_depth = in.depths != nullptr;
            const float depth = has_depth ? in.depths[i] : 0.0f;
            if (!bayes) {
                // voting (voxel_data_semantic.h:153-198): observations at depth >= threshold are ignored
                if (!has_depth || depth < G.depth_threshold) {
                    if (count == 0) {
                        obj = oo, cls = oc, ctr = 1;
                    } else if (obj == oo && cls == oc) {
                        ++ctr;
                    } else if (--ctr <= 0) {
                        obj = oo, cls = oc, ctr = 1;
                    }
                }
            } else {
                // Bayesian (voxel_data_semantic.h:312-451): evidence w * -log(0.9), w = 1 up to the depth threshold,
                // exp(-(depth - threshold) * rate) beyond it
                float w = kBaseLogProb;
                if (has_depth && !(depth <= G.depth_threshold))
                    w = __fmul_rn(exp_rn(__fmul_rn(-__fsub_rn(depth, G.depth_threshold), G.depth_decay_rate)),
                                  kBaseLogProb);
                int k = 0;
                while (k < nl && !(lo[k] == oo && lc[k] == oc)) ++k;
                if (count == 0) {  // initialize_semantics_log_prob: map[key] = w, argmax = key
                    if (k == nl) {
                        k = nl < kSemLabels ? nl++ : 0;
                        lo[k] = oo, lc[k] = oc;
                    }
                    lp[k] = w;
                    obj = oo, cls = oc, mlp = w;
                } else if (k < nl) {  // known pair: accumulate; a strictly larger value takes the argmax
                    lp[k] = __fadd_rn(lp[k], w);
                    if (lo[k] == obj && lc[k] == cls) {
                        mlp = lp[k];
                    } else if (lp[k] > mlp) {
                        mlp = lp[k];
                        obj = oo, cls = oc;
                    }
                } else {  // new pair
                    if (nl < kSemLabels) {
                        k = nl++;
                    } else {  // out of slots: evict the weakest pair that is not the argmax
                        k = -1;
                        for (int q = 0; q < kSemLabels; ++q)
                            if (!(lo[q] == obj && lc[q] == cls) && (k < 0 || lp[q] < lp[k])) k = q;
                        atomicAdd(G.counters + kSemOverflow, 1u);
                    }
                    lo[k] = oo, lc[k] = oc, lp[k] = w;
                    if (w > mlp) {
                        mlp = w;
                        obj = oo, cls = oc;
                    }
                }
            }
        }
        ++count;
    }

    G.count[v] = count;
    G.pos[3 * static_cast<size_t>(v) + 0] = px;
    G.pos[3 * static_cast<size_t>(v) + 1] = py;
    G.pos[3 * static_cast<size_t>(v) + 2] = pz;
    G.col[3 * static_cast<size_t>(v) + 0] = cr;
    G.col[3 * static_cast<size_t>(v) + 1] = cg;
    G.col[3 * static_cast<size_t>(v) + 2] = cb;
    if (semantics) {
        G.obj[v] = obj;
        G.cls[v] = cls;
        if (!bayes) {
            G.counter[v] = ctr;
        } else {
            G.counter[v] = nl;
            G.ml_logp[v] = mlp;
            for (int k = 0; k < kSemLabels; ++k) {
                G.lab_obj[static_cast<size_t>(v) * kSemLabels + k] = lo[k];
                G.lab_cls[static_cast<size_t>(v) * kSemLabels + k] = lc[k];
                G.lab_logp[static_cast<size_t>(v) * kSemLabels + k] = lp[k];
            }
            G.conf[v] = bayes_confidence(lo, lc, lp, nl, obj, cls, mlp);
        }
    }
}

// ---- read-outs -------------------------------------------------------------------------------------------------
__device__ __forceinline__ float sem_confidence(const SemGrid &G, uint32_t v, int32_t count) {
    if (count == 0) return 0.0f;
    if (G.kind == B2V_SEM_PROBABILISTIC) return G.conf[v];
    // voting (voxel_data_semantic.h:117-132): min(1, counter / count)
    return fminf(1.0f, __fdiv_rn(static_cast<float>(G.counter[v]), static_cast<float>(count)));
}

__device__ __forceinline__ void sem_reset_voxel(const SemGrid &G, uint32_t v) {  // VoxelSemanticData*::reset()
    G.count[v] = 0;
    for (int a = 0; a < 3; ++a) {
        G.pos[3 * static_cast<size_t>(v) + a] = 0.0;
        G.col[3 * static_cast<size_t>(v) + a] = 0.0f;
    }
    G.obj[v] = -1;
    G.cls[v] = -1;
    G.counter[v] = 0;
    if (G.kind == B2V_SEM_PROBABILISTIC) {
        G.ml_logp[v] = __uint_as_float(0xFF800000u);
        G.conf[v] = 0.0f;
    }
}

// set_object_id (voxel_data_semantic.h:135, 455-460): the Bayesian voxel collapses onto the forced pair
__device__ __forceinline__ void sem_set_object_id(const SemGrid &G, uint32_t v, int32_t id) {
    G.obj[v] = id;
    if (G.kind == B2V_SEM_PROBABILISTIC) {
        const int32_t cl = G.cls[v];
        if (id >= 0 && cl >= 0) {
            G.counter[v] = 1;
            G.lab_obj[static_cast<size_t>(v) * kSemLabels] = id;
            G.lab_cls[static_cast<size_t>(v) * kSemLabels] = cl;
            G.lab_logp[static_cast<size_t>(v) * kSemLabels] = 0.0f;
            G.ml_logp[v] = 0.0f;
            G.conf[v] = 1.0f;
        } else {
            G.counter[v] = 0;
            G.ml_logp[v] = __uint_as_float(0xFF800000u);
            G.conf[v] = 0.0f;
        }
    }
}

// op 0: remove_low_count_voxels(a)  1: remove_low_confidence_segments(a)  2: remove_segment(a)
// op 3: merge_segments(a, b)  (voxel_block_grid.hpp:625-647; voxel_block_semantic_grid.hpp:101-183)
__global__ void __launch_bounds__(kVox) sem_edit_kernel(const SemGrid G, const int op, const int a, const int b) {
    const uint32_t v = blockIdx.x * kVox + threadIdx.x;
    const int c = G.count[v];
    if (op == 0) {
        if (c < a) sem_reset_voxel(G, v);
    } else if (op == 1) {
        if (sem_confidence(G, v, c) < static_cast<float>(a)) sem_reset_voxel(G, v);
    } else if (op == 2) {
        if (G.obj[v] == a) sem_reset_voxel(G, v);
    } else if (G.obj[v] == b) {
        sem_set_object_id(G, v, a);
    }
}

// ---- spatial queries: read-outs, carve and instance -> object association ------------------------------------
// the per-voxel stages of a box or frustum query (voxel_block_grid.hpp:822-1195, 1336-1460) on voxel t of pool block
// b before the fine test: count threshold and voxel-key range; p = the voxel's float64 mean position
__device__ __forceinline__ bool sem_voxel_in_range(const SemGrid &G, const GridQuery &Q, uint32_t b, int t,
                                                   double p[3]) {
    const uint32_t v = b * kVox + t;
    const int c = G.count[v];
    if (c < Q.min_count || !voxel_key_in_range(Q, G.block_keys[b], t)) return false;
    const double dc = static_cast<double>(c);
#pragma unroll
    for (int a = 0; a < 3; ++a) p[a] = __ddiv_rn(G.pos[3 * static_cast<size_t>(v) + a], dc);
    return true;
}

// the filter of a read-out: count and confidence thresholds (voxel_block_grid.hpp:797-803), then the query's
// spatial stages
__device__ __forceinline__ bool sem_keep(const SemGrid &G, const GridQuery &Q, uint32_t b, int t, float min_conf,
                                         float *conf_out) {
    const uint32_t v = b * kVox + t;
    const int c = G.count[v];
    const float conf = sem_confidence(G, v, c);
    *conf_out = conf;
    if (!(c >= Q.min_count && conf >= min_conf)) return false;
    if (Q.mode == kQueryAll) return true;
    double p[3];
    ImagePoint ip;
    return block_in_range(Q, G.block_keys[b]) && sem_voxel_in_range(G, Q, b, t, p) && position_in_query(Q, p, &ip);
}

__global__ void __launch_bounds__(kVox)
sem_count_kernel(const SemGrid G, const GridQuery Q, const float min_conf, uint32_t *__restrict__ sums) {
    __shared__ uint32_t s_warp[16];
    float conf;
    block_count_512(sem_keep(G, Q, blockIdx.x, threadIdx.x, min_conf, &conf), s_warp, sums);
}

__global__ void __launch_bounds__(kVox)
sem_emit_kernel(const SemGrid G, const GridQuery Q, const float min_conf,
                const uint32_t *__restrict__ offs, double *__restrict__ out_pts, float *__restrict__ out_cols,
                int32_t *__restrict__ out_cls, int32_t *__restrict__ out_obj, float *__restrict__ out_conf) {
    __shared__ uint32_t s_warp[16];
    const uint32_t v = blockIdx.x * kVox + threadIdx.x;
    float conf;
    const bool keep = sem_keep(G, Q, blockIdx.x, threadIdx.x, min_conf, &conf);
    const size_t pos = offs[blockIdx.x] + block_excl_scan_512(keep ? 1u : 0u, s_warp);
    if (!keep) return;
    const int c = G.count[v];
    const double dc = static_cast<double>(c);
    const float fc = static_cast<float>(c);
    for (int a = 0; a < 3; ++a) {  // voxel_data.h:58-69, 98-109: sum / (T)count, zero for an empty voxel
        out_pts[3 * pos + a] = c ? __ddiv_rn(G.pos[3 * static_cast<size_t>(v) + a], dc) : 0.0;
        out_cols[3 * pos + a] = c ? __fdiv_rn(G.col[3 * static_cast<size_t>(v) + a], fc) : 0.0f;
    }
    out_cls[pos] = G.cls[v];
    out_obj[pos] = G.obj[v];
    out_conf[pos] = conf;
}

// carve (voxel_grid_carving.h:47-80): reset voxels in front of the observed surface by more than the threshold;
// the depth image is indexed with truncated pixel coordinates, like at<float>(v, u)
__global__ void __launch_bounds__(kVox)
sem_carve_kernel(const SemGrid G, const GridQuery Q, const float *__restrict__ depth, const float thr) {
    const uint32_t b = blockIdx.x;
    if (!block_in_range(Q, G.block_keys[b])) return;
    double p[3];
    ImagePoint ip;
    if (!sem_voxel_in_range(G, Q, b, threadIdx.x, p) || !frustum_contains(Q, p, &ip)) return;
    const float image_depth = depth[static_cast<size_t>(static_cast<int>(ip.v)) * Q.W + static_cast<int>(ip.u)];
    if (image_depth <= 0.0f || !isfinite(image_depth)) return;
    if (ip.depth < image_depth - thr) sem_reset_voxel(G, b * kVox + threadIdx.x);
}

// process_point of assign_object_ids_to_instance_ids (voxel_semantic_data_association.h:171-229): every voxel in
// the frustum whose class equals the pixel's class and that lies on the observed surface votes
// "image instance id -> my object id".  Voxels without an object id are recorded as pending (pend[v] = instance
// id); the host turns the vote records into the instance -> object map.
constexpr int32_t kAssocPending = INT_MIN;
__global__ void __launch_bounds__(kVox)
sem_assoc_kernel(const SemGrid G, const GridQuery Q, const int32_t *__restrict__ class_img,
                 const int32_t *__restrict__ inst_img, const float *__restrict__ depth_img, const float thr,
                 const int do_carving, int32_t *__restrict__ pend, int2 *__restrict__ records,
                 uint32_t *__restrict__ n_records, const uint32_t cap_records) {
    const uint32_t b = blockIdx.x;
    if (!block_in_range(Q, G.block_keys[b])) return;
    double p[3];
    ImagePoint ip;
    if (!sem_voxel_in_range(G, Q, b, threadIdx.x, p) || !frustum_contains(Q, p, &ip)) return;
    const uint32_t v = b * kVox + threadIdx.x;
    const size_t px = static_cast<size_t>(static_cast<int>(ip.v)) * Q.W + static_cast<int>(ip.u);
    const int32_t image_class = class_img[px];
    if (image_class < 0) return;
    const int32_t point_class = G.cls[v];
    if (point_class < 0 || point_class != image_class) return;
    const int32_t image_instance = inst_img[px];
    if (image_instance < 0) return;
    int32_t point_object = G.obj[v];
    if (depth_img != nullptr) {
        const float image_depth = depth_img[px];
        if (image_depth <= 0.0f || !isfinite(image_depth)) return;
        if (do_carving && ip.depth < image_depth - thr) {
            sem_reset_voxel(G, v);
            return;
        }
        if (ip.depth > image_depth + thr) return;
    }
    if (point_object < 0) {
        if (image_instance == 0) {
            point_object = 0;
            sem_set_object_id(G, v, 0);
        } else {
            point_object = kAssocPending;  // one new object id per instance id, handed out by the host
            pend[v] = image_instance;
        }
    }
    const uint32_t r = atomicAdd(n_records, 1u);
    if (r < cap_records) records[r] = make_int2(image_instance, point_object);
}

// deferred assignment (voxel_semantic_data_association.h:354-370): pending voxels take their instance's final id
__global__ void __launch_bounds__(kVox)
sem_assoc_apply_kernel(const SemGrid G, const int32_t *__restrict__ pend, const int32_t *__restrict__ map_inst,
                       const int32_t *__restrict__ map_obj, const int n_map) {
    const uint32_t v = blockIdx.x * kVox + threadIdx.x;
    const int32_t inst = pend[v];
    if (inst < 0) return;
    int lo = 0, hi = n_map - 1;
    while (lo <= hi) {  // map_inst is sorted
        const int mid = (lo + hi) >> 1;
        const int32_t m = map_inst[mid];
        if (m == inst) {
            if (map_obj[mid] >= 0) sem_set_object_id(G, v, map_obj[mid]);
            return;
        }
        if (m < inst) lo = mid + 1; else hi = mid - 1;
    }
}

__global__ void sem_fill_kernel(const SemGrid G, const size_t n_vox) {
    for (size_t v = static_cast<size_t>(blockIdx.x) * blockDim.x + threadIdx.x; v < n_vox;
         v += static_cast<size_t>(gridDim.x) * blockDim.x) {
        G.obj[v] = -1;
        G.cls[v] = -1;
        if (G.kind == B2V_SEM_PROBABILISTIC) G.ml_logp[v] = __uint_as_float(0xFF800000u);
    }
}

}  // namespace b2v

// ====================================================================================================================
// host side: the C ABI of include/b2v.h (b2v_sgrid_*)
// ====================================================================================================================
using namespace b2v;

struct b2v_sgrid {
    double voxel_size = 0.0;
    float inv_voxel_size = 0.0f;
    int device = 0;
    cudaStream_t stream = nullptr;
    HashTable table{};
    SemGrid G{};
    uint32_t *h_counters = nullptr;
    // staging
    void *d_pts = nullptr, *d_cols = nullptr;
    int32_t *d_cls = nullptr, *d_inst = nullptr;
    float *d_depths = nullptr;
    uint32_t *d_vid[2] = {nullptr, nullptr}, *d_ord[2] = {nullptr, nullptr};
    void *d_sort_tmp = nullptr;
    size_t sort_tmp_bytes = 0, stage_points = 0;
    // fused RGBD front-end
    float *d_img_depth = nullptr, *d_img_filtered = nullptr;
    uint8_t *d_img_rgb = nullptr, *d_valid = nullptr;
    int32_t *d_img_cls = nullptr, *d_img_obj = nullptr;
    void *d_shadow_scratch = nullptr;
    size_t img_pixels = 0;
    // instance -> object association
    int32_t *d_pend = nullptr;
    int2 *d_records = nullptr;
    uint32_t *d_n_records = nullptr;
    size_t records_cap = 0;
    int32_t next_object_id = 1;  // VoxelSemanticSharedData::next_object_id (process-wide in the reference)
    std::vector<int32_t> map_inst, map_obj;
    // read-out
    uint32_t *d_sums = nullptr, *d_offs = nullptr, *d_total = nullptr;
    uint32_t scan_cap = 0;
    double *d_out_pts = nullptr;
    float *d_out_cols = nullptr, *d_out_conf = nullptr;
    int32_t *d_out_cls = nullptr, *d_out_obj = nullptr;
    size_t out_cap = 0;
    int64_t last_n = 0;
    std::string err;
};

extern "C" const char *b2v_sgrid_last_error(const b2v_sgrid *g) { return g ? g->err.c_str() : "null grid"; }

static int sgrid_clear_device(b2v_sgrid *g, uint32_t used_blocks) {
    const size_t tcap = static_cast<size_t>(g->table.mask) + 1;
    const size_t nv = static_cast<size_t>(used_blocks) * kVox;
    B2V_CUDA(g, cudaMemsetAsync(g->table.entries, 0xFF, tcap * sizeof(uint4), g->stream));
    B2V_CUDA(g, cudaMemsetAsync(g->G.counters, 0, kSemNumCounters * sizeof(uint32_t), g->stream));
    if (nv == 0) return B2V_OK;
    B2V_CUDA(g, cudaMemsetAsync(g->G.count, 0, nv * sizeof(int32_t), g->stream));
    B2V_CUDA(g, cudaMemsetAsync(g->G.pos, 0, nv * 3 * sizeof(double), g->stream));
    B2V_CUDA(g, cudaMemsetAsync(g->G.col, 0, nv * 3 * sizeof(float), g->stream));
    B2V_CUDA(g, cudaMemsetAsync(g->G.counter, 0, nv * sizeof(int32_t), g->stream));
    if (g->G.kind == B2V_SEM_PROBABILISTIC) B2V_CUDA(g, cudaMemsetAsync(g->G.conf, 0, nv * sizeof(float), g->stream));
    sem_fill_kernel<<<592, 256, 0, g->stream>>>(g->G, nv);
    B2V_CUDA(g, cudaGetLastError());
    return B2V_OK;
}

extern "C" int b2v_sgrid_create(double voxel_size, int32_t block_size, uint32_t capacity_blocks, int32_t kind,
                                int32_t device, b2v_sgrid **out) {
    if (!out) return B2V_ERR_INVALID_ARGUMENT;
    *out = nullptr;
    if (block_size != B2V_BLOCK_SIZE || !(voxel_size > 0.0) || capacity_blocks == 0 ||
        capacity_blocks > (1u << 22) || (kind != B2V_SEM_VOTING && kind != B2V_SEM_PROBABILISTIC))
        return B2V_ERR_INVALID_ARGUMENT;
    b2v_sgrid *g = new (std::nothrow) b2v_sgrid();
    if (!g) return B2V_ERR_INVALID_ARGUMENT;
    g->voxel_size = voxel_size;
    // the reference stores the voxel size as float and inverts it in float (voxel_block_grid.h:225-226, .hpp:6)
    g->inv_voxel_size = 1.0f / static_cast<float>(voxel_size);
    g->device = device;
    g->G.kind = kind;
    g->G.capacity = capacity_blocks;
    // class defaults (voxel_data_semantic.h:107-108, 251-254)
    g->G.depth_threshold = kind == B2V_SEM_VOTING ? 10.0f : 5.0f;
    g->G.depth_decay_rate = 0.07f;
    *out = g;
    B2V_CUDA(g, cudaSetDevice(device));
    B2V_CUDA(g, cudaStreamCreateWithFlags(&g->stream, cudaStreamNonBlocking));
    const size_t tcap = next_pow2(static_cast<uint64_t>(capacity_blocks) * 2);
    g->table.mask = static_cast<uint32_t>(tcap - 1);
    g->table.stamp = nullptr;
    const size_t nv = static_cast<size_t>(capacity_blocks) * kVox;
    B2V_CUDA(g, cudaMalloc(&g->table.entries, tcap * sizeof(uint4)));
    B2V_CUDA(g, cudaMalloc(&g->G.counters, kSemNumCounters * sizeof(uint32_t)));
    B2V_CUDA(g, cudaMalloc(&g->G.block_keys, static_cast<size_t>(capacity_blocks) * sizeof(int4)));
    B2V_CUDA(g, cudaMalloc(&g->G.count, nv * sizeof(int32_t)));
    B2V_CUDA(g, cudaMalloc(&g->G.pos, nv * 3 * sizeof(double)));
    B2V_CUDA(g, cudaMalloc(&g->G.col, nv * 3 * sizeof(float)));
    B2V_CUDA(g, cudaMalloc(&g->G.obj, nv * sizeof(int32_t)));
    B2V_CUDA(g, cudaMalloc(&g->G.cls, nv * sizeof(int32_t)));
    B2V_CUDA(g, cudaMalloc(&g->G.counter, nv * sizeof(int32_t)));
    if (kind == B2V_SEM_PROBABILISTIC) {
        B2V_CUDA(g, cudaMalloc(&g->G.ml_logp, nv * sizeof(float)));
        B2V_CUDA(g, cudaMalloc(&g->G.conf, nv * sizeof(float)));
        B2V_CUDA(g, cudaMalloc(&g->G.lab_obj, nv * kSemLabels * sizeof(int32_t)));
        B2V_CUDA(g, cudaMalloc(&g->G.lab_cls, nv * kSemLabels * sizeof(int32_t)));
        B2V_CUDA(g, cudaMalloc(&g->G.lab_logp, nv * kSemLabels * sizeof(float)));
    }
    B2V_CUDA(g, cudaMalloc(&g->d_total, sizeof(uint32_t)));
    B2V_CUDA(g, cudaMallocHost(&g->h_counters, kSemNumCounters * sizeof(uint32_t)));
    const int rc = sgrid_clear_device(g, capacity_blocks);
    if (rc != B2V_OK) return rc;
    B2V_CUDA(g, cudaStreamSynchronize(g->stream));
    return B2V_OK;
}

extern "C" int b2v_sgrid_destroy(b2v_sgrid *g) {
    if (!g) return B2V_OK;
    cudaSetDevice(g->device);
    if (g->stream) cudaStreamSynchronize(g->stream);
    void *ptrs[] = {g->table.entries, g->G.counters, g->G.block_keys, g->G.count, g->G.pos, g->G.col, g->G.obj,
                    g->G.cls, g->G.counter, g->G.ml_logp, g->G.conf, g->G.lab_obj, g->G.lab_cls, g->G.lab_logp,
                    g->d_pts, g->d_cols, g->d_cls, g->d_inst, g->d_depths, g->d_vid[0], g->d_vid[1], g->d_ord[0],
                    g->d_ord[1], g->d_sort_tmp, g->d_sums, g->d_offs, g->d_total, g->d_out_pts, g->d_out_cols,
                    g->d_out_conf, g->d_out_cls, g->d_out_obj, g->d_img_depth, g->d_img_filtered, g->d_img_rgb,
                    g->d_valid, g->d_img_cls, g->d_img_obj, g->d_shadow_scratch, g->d_pend, g->d_records,
                    g->d_n_records};
    for (void *p : ptrs) cudaFree(p);
    cudaFreeHost(g->h_counters);
    if (g->stream) cudaStreamDestroy(g->stream);
    delete g;
    return B2V_OK;
}

static int sgrid_read_counters(b2v_sgrid *g) {
    const char *full;
    B2V_CUDA(g, read_grid_counters(g->device, g->stream, g->G.counters, g->h_counters, kSemNumCounters, &full));
    if (full) {
        g->err = full;
        return B2V_ERR_CAPACITY;
    }
    return B2V_OK;
}

extern "C" int b2v_sgrid_clear(b2v_sgrid *g) {
    if (!g) return B2V_ERR_INVALID_ARGUMENT;
    B2V_CUDA(g, read_grid_counters(g->device, g->stream, g->G.counters, g->h_counters, kSemNumCounters, nullptr));
    const int rc = sgrid_clear_device(g, grid_blocks_used(g->h_counters, g->G.capacity));
    if (rc != B2V_OK) return rc;
    B2V_CUDA(g, cudaStreamSynchronize(g->stream));
    return B2V_OK;
}

extern "C" int b2v_sgrid_set_depth_threshold(b2v_sgrid *g, float depth_threshold) {
    if (!g) return B2V_ERR_INVALID_ARGUMENT;
    g->G.depth_threshold = depth_threshold;
    return B2V_OK;
}

extern "C" int b2v_sgrid_set_depth_decay_rate(b2v_sgrid *g, float depth_decay_rate) {
    if (!g) return B2V_ERR_INVALID_ARGUMENT;
    if (g->G.kind == B2V_SEM_PROBABILISTIC) g->G.depth_decay_rate = depth_decay_rate;  // semantic_grid.hpp:31-36
    return B2V_OK;
}

static int sgrid_ensure_stage(b2v_sgrid *g, size_t n) {
    if (n <= g->stage_points) return B2V_OK;
    B2V_CUDA(g, cudaStreamSynchronize(g->stream));
    void **bufs[] = {&g->d_pts, &g->d_cols, reinterpret_cast<void **>(&g->d_cls), reinterpret_cast<void **>(&g->d_inst),
                     reinterpret_cast<void **>(&g->d_depths), reinterpret_cast<void **>(&g->d_vid[0]),
                     reinterpret_cast<void **>(&g->d_vid[1]), reinterpret_cast<void **>(&g->d_ord[0]),
                     reinterpret_cast<void **>(&g->d_ord[1]), &g->d_sort_tmp};
    for (void **b : bufs) {
        cudaFree(*b);
        *b = nullptr;
    }
    g->stage_points = 0;  // stays 0 if an allocation below fails
    const size_t cap = n + n / 4 + 1024;
    B2V_CUDA(g, cudaMalloc(&g->d_pts, cap * 3 * sizeof(double)));
    B2V_CUDA(g, cudaMalloc(&g->d_cols, cap * 3 * sizeof(float)));
    B2V_CUDA(g, cudaMalloc(&g->d_cls, cap * sizeof(int32_t)));
    B2V_CUDA(g, cudaMalloc(&g->d_inst, cap * sizeof(int32_t)));
    B2V_CUDA(g, cudaMalloc(&g->d_depths, cap * sizeof(float)));
    for (int k = 0; k < 2; ++k) {
        B2V_CUDA(g, cudaMalloc(&g->d_vid[k], cap * sizeof(uint32_t)));
        B2V_CUDA(g, cudaMalloc(&g->d_ord[k], cap * sizeof(uint32_t)));
    }
    size_t tmp = 0;
    B2V_CUDA(g, cub::DeviceRadixSort::SortPairs(nullptr, tmp, g->d_vid[0], g->d_vid[1], g->d_ord[0], g->d_ord[1],
                                               static_cast<int64_t>(cap), 0, 32, g->stream));
    B2V_CUDA(g, cudaMalloc(&g->d_sort_tmp, tmp));
    g->sort_tmp_bytes = tmp;
    g->stage_points = cap;
    return B2V_OK;
}

// insert -> keys -> sort -> runs over the staged point records (valid: optional per-point mask)
static int sgrid_fuse_staged(b2v_sgrid *g, int64_t n, const SemInputs &in, const uint8_t *valid) {
    cudaStream_t s = g->stream;
    const unsigned grid = static_cast<unsigned>((n + 255) / 256);
    if (in.pts_f64) {
        sem_insert_kernel<double><<<grid, 256, 0, s>>>(static_cast<const double *>(in.pts), valid, n,
                                                       g->inv_voxel_size, g->table, g->G);
        sem_keys_kernel<double><<<grid, 256, 0, s>>>(static_cast<const double *>(in.pts), valid, n, g->inv_voxel_size,
                                                     g->table, g->G, g->d_vid[0], g->d_ord[0]);
    } else {
        sem_insert_kernel<float><<<grid, 256, 0, s>>>(static_cast<const float *>(in.pts), valid, n, g->inv_voxel_size,
                                                      g->table, g->G);
        sem_keys_kernel<float><<<grid, 256, 0, s>>>(static_cast<const float *>(in.pts), valid, n, g->inv_voxel_size,
                                                    g->table, g->G, g->d_vid[0], g->d_ord[0]);
    }
    B2V_CUDA(g, cudaGetLastError());
    size_t tmp = g->sort_tmp_bytes;  // all 32 key bits: kBadVid (points without storage) must sort last
    B2V_CUDA(g, cub::DeviceRadixSort::SortPairs(g->d_sort_tmp, tmp, g->d_vid[0], g->d_vid[1], g->d_ord[0], g->d_ord[1],
                                               n, 0, 32, s));
    sem_runs_kernel<<<static_cast<unsigned>((n + 127) / 128), 128, 0, s>>>(g->d_vid[1], g->d_ord[1], n, in, g->G);
    B2V_CUDA(g, cudaGetLastError());
    return B2V_OK;
}

extern "C" int b2v_sgrid_integrate(b2v_sgrid *g, int64_t n, const void *points, int32_t points_f64,
                                   const void *colors, int32_t colors_u8, const int32_t *class_ids,
                                   const int32_t *instance_ids, const float *depths) {
    if (!g) return B2V_ERR_INVALID_ARGUMENT;
    if (n < 0 || (n > 0 && !points) || n > 0x7FFFFFF0LL) {
        g->err = "b2v_sgrid_integrate: bad arguments";
        return B2V_ERR_INVALID_ARGUMENT;
    }
    if (instance_ids && !class_ids) {  // voxel_block_grid.hpp:43-46
        g->err = "instance_ids but no class_ids is not supported";
        return B2V_ERR_INVALID_ARGUMENT;
    }
    if (n == 0) return B2V_OK;
    B2V_CUDA(g, cudaSetDevice(g->device));
    int rc = sgrid_ensure_stage(g, static_cast<size_t>(n));
    if (rc != B2V_OK) return rc;
    const size_t m = static_cast<size_t>(n);
    cudaStream_t s = g->stream;
    B2V_CUDA(g, cudaMemcpyAsync(g->d_pts, points, m * 3 * (points_f64 ? sizeof(double) : sizeof(float)),
                               cudaMemcpyDefault, s));
    if (colors)
        B2V_CUDA(g, cudaMemcpyAsync(g->d_cols, colors, m * 3 * (colors_u8 ? 1 : sizeof(float)), cudaMemcpyDefault, s));
    if (class_ids) B2V_CUDA(g, cudaMemcpyAsync(g->d_cls, class_ids, m * sizeof(int32_t), cudaMemcpyDefault, s));
    if (instance_ids) B2V_CUDA(g, cudaMemcpyAsync(g->d_inst, instance_ids, m * sizeof(int32_t), cudaMemcpyDefault, s));
    if (depths) B2V_CUDA(g, cudaMemcpyAsync(g->d_depths, depths, m * sizeof(float), cudaMemcpyDefault, s));
    SemInputs in{};
    in.pts = g->d_pts;
    in.cols = colors ? g->d_cols : nullptr;
    in.cls = class_ids ? g->d_cls : nullptr;
    in.inst = instance_ids ? g->d_inst : nullptr;
    in.depths = depths ? g->d_depths : nullptr;
    in.pts_f64 = points_f64 ? 1 : 0;
    in.cols_u8 = colors_u8 ? 1 : 0;
    rc = sgrid_fuse_staged(g, n, in, nullptr);
    if (rc != B2V_OK) return rc;
    return sgrid_read_counters(g);  // also the completion fence: the inputs are free when this returns
}

extern "C" int b2v_sgrid_integrate_rgbd(b2v_sgrid *g, const float *depth, const uint8_t *color,
                                        const int32_t *class_image, const int32_t *object_image, int32_t height,
                                        int32_t width, const double K[4], const double Twc[16], float max_depth,
                                        float min_depth, int32_t use_depths, int32_t filter_shadow_points) {
    if (!g) return B2V_ERR_INVALID_ARGUMENT;
    if (!depth || !color || !K || !Twc || height <= 0 || width <= 0 || (object_image && !class_image)) {
        g->err = "b2v_sgrid_integrate_rgbd: bad arguments";
        return B2V_ERR_INVALID_ARGUMENT;
    }
    B2V_CUDA(g, cudaSetDevice(g->device));
    const size_t pixels = static_cast<size_t>(height) * width;
    int rc = sgrid_ensure_stage(g, pixels);
    if (rc != B2V_OK) return rc;
    if (pixels > g->img_pixels) {
        B2V_CUDA(g, cudaStreamSynchronize(g->stream));
        void **bufs[] = {reinterpret_cast<void **>(&g->d_img_depth), reinterpret_cast<void **>(&g->d_img_filtered),
                         reinterpret_cast<void **>(&g->d_img_rgb), reinterpret_cast<void **>(&g->d_img_cls),
                         reinterpret_cast<void **>(&g->d_img_obj), reinterpret_cast<void **>(&g->d_valid),
                         &g->d_shadow_scratch};
        for (void **b : bufs) {
            cudaFree(*b);
            *b = nullptr;
        }
        g->img_pixels = 0;  // stays 0 if an allocation below fails
        B2V_CUDA(g, cudaMalloc(&g->d_img_depth, pixels * sizeof(float)));
        B2V_CUDA(g, cudaMalloc(&g->d_img_filtered, pixels * sizeof(float)));
        B2V_CUDA(g, cudaMalloc(&g->d_img_rgb, pixels * 3));
        B2V_CUDA(g, cudaMalloc(&g->d_img_cls, pixels * sizeof(int32_t)));
        B2V_CUDA(g, cudaMalloc(&g->d_img_obj, pixels * sizeof(int32_t)));
        B2V_CUDA(g, cudaMalloc(&g->d_valid, pixels));
        B2V_CUDA(g, cudaMalloc(&g->d_shadow_scratch, kShadowScratchBytes));
        g->img_pixels = pixels;
    }
    cudaStream_t s = g->stream;
    B2V_CUDA(g, cudaMemcpyAsync(g->d_img_depth, depth, pixels * sizeof(float), cudaMemcpyDefault, s));
    B2V_CUDA(g, cudaMemcpyAsync(g->d_img_rgb, color, pixels * 3, cudaMemcpyDefault, s));
    if (class_image) B2V_CUDA(g, cudaMemcpyAsync(g->d_img_cls, class_image, pixels * sizeof(int32_t), cudaMemcpyDefault, s));
    if (object_image) B2V_CUDA(g, cudaMemcpyAsync(g->d_img_obj, object_image, pixels * sizeof(int32_t), cudaMemcpyDefault, s));
    const float *d_depth = g->d_img_depth;
    if (filter_shadow_points) {  // semantic_grid.py:332-341: everything downstream sees the filtered depth
        if (height <= 2 || width <= 2) {
            g->err = "b2v_sgrid_integrate_rgbd: image too small for the shadow filter";
            return B2V_ERR_INVALID_ARGUMENT;
        }
        B2V_CUDA(g, launch_filter_shadow_points(d_depth, height, width, 2, 2, -1.0f, g->d_img_filtered,
                                               g->d_shadow_scratch, s));
        d_depth = g->d_img_filtered;
    }
    const RgbdParams P = rgbd_params(K, Twc, height, width, min_depth, max_depth);
    const int64_t n = static_cast<int64_t>(pixels);
    sem_rgbd_points_kernel<<<static_cast<unsigned>((n + 255) / 256), 256, 0, s>>>(
        P, d_depth, g->d_img_rgb, class_image ? g->d_img_cls : nullptr, object_image ? g->d_img_obj : nullptr,
        static_cast<float *>(g->d_pts), static_cast<float *>(g->d_cols), g->d_cls, g->d_inst, g->d_depths, g->d_valid);
    B2V_CUDA(g, cudaGetLastError());
    SemInputs in{};
    in.pts = g->d_pts;
    in.cols = g->d_cols;
    in.cls = class_image ? g->d_cls : nullptr;
    in.inst = object_image ? g->d_inst : nullptr;
    in.depths = use_depths ? g->d_depths : nullptr;
    rc = sgrid_fuse_staged(g, n, in, g->d_valid);
    if (rc != B2V_OK) return rc;
    return sgrid_read_counters(g);
}

extern "C" int64_t b2v_sgrid_num_blocks(b2v_sgrid *g) {
    if (!g) return -1;
    if (read_grid_counters(g->device, g->stream, g->G.counters, g->h_counters, kSemNumCounters, nullptr) != cudaSuccess)
        return -1;
    return grid_blocks_used(g->h_counters, g->G.capacity);
}

extern "C" int b2v_sgrid_label_overflows(b2v_sgrid *g, uint64_t *out) {
    if (!g || !out) return B2V_ERR_INVALID_ARGUMENT;
    if (b2v_sgrid_num_blocks(g) < 0) return B2V_ERR_CUDA;
    *out = g->h_counters[kSemOverflow];
    return B2V_OK;
}

static int64_t sgrid_run_readout(b2v_sgrid *g, const GridQuery &q, float min_confidence) {
    const int64_t nb64 = b2v_sgrid_num_blocks(g);
    if (nb64 < 0) {
        g->err = "semantic read-out: device error";
        return -1;
    }
    const uint32_t nb = static_cast<uint32_t>(nb64);
    g->last_n = 0;
    if (nb == 0) return 0;
    auto fail = [&](cudaError_t e) {
        g->err = std::string("semantic read-out: ") + cudaGetErrorString(e);
        return static_cast<int64_t>(-1);
    };
    cudaError_t e;
    if (nb > g->scan_cap) {
        cudaFree(g->d_sums);
        cudaFree(g->d_offs);
        g->d_sums = g->d_offs = nullptr;
        if ((e = cudaMalloc(&g->d_sums, static_cast<size_t>(nb) * 2 * sizeof(uint32_t))) != cudaSuccess) return fail(e);
        if ((e = cudaMalloc(&g->d_offs, static_cast<size_t>(nb) * 2 * sizeof(uint32_t))) != cudaSuccess) return fail(e);
        g->scan_cap = nb * 2;
    }
    sem_count_kernel<<<nb, kVox, 0, g->stream>>>(g->G, q, min_confidence, g->d_sums);
    exclusive_scan_kernel<<<1, 1024, 0, g->stream>>>(g->d_sums, g->d_offs, g->d_total, nb);
    uint32_t total = 0;
    if ((e = cudaMemcpyAsync(&total, g->d_total, sizeof(uint32_t), cudaMemcpyDeviceToHost, g->stream)) != cudaSuccess)
        return fail(e);
    if ((e = cudaStreamSynchronize(g->stream)) != cudaSuccess) return fail(e);
    if (total > g->out_cap) {
        void *old[] = {g->d_out_pts, g->d_out_cols, g->d_out_conf, g->d_out_cls, g->d_out_obj};
        for (void *p : old) cudaFree(p);
        g->d_out_pts = nullptr;
        g->d_out_cols = g->d_out_conf = nullptr;
        g->d_out_cls = g->d_out_obj = nullptr;
        g->out_cap = 0;
        const size_t cap = static_cast<size_t>(total) + total / 4 + 1024;
        if ((e = cudaMalloc(&g->d_out_pts, cap * 3 * sizeof(double))) != cudaSuccess) return fail(e);
        if ((e = cudaMalloc(&g->d_out_cols, cap * 3 * sizeof(float))) != cudaSuccess) return fail(e);
        if ((e = cudaMalloc(&g->d_out_conf, cap * sizeof(float))) != cudaSuccess) return fail(e);
        if ((e = cudaMalloc(&g->d_out_cls, cap * sizeof(int32_t))) != cudaSuccess) return fail(e);
        if ((e = cudaMalloc(&g->d_out_obj, cap * sizeof(int32_t))) != cudaSuccess) return fail(e);
        g->out_cap = cap;
    }
    if (total) {
        sem_emit_kernel<<<nb, kVox, 0, g->stream>>>(g->G, q, min_confidence, g->d_offs, g->d_out_pts, g->d_out_cols,
                                                    g->d_out_cls, g->d_out_obj, g->d_out_conf);
        if ((e = cudaGetLastError()) != cudaSuccess) return fail(e);
    }
    g->last_n = total;
    return total;
}

extern "C" int64_t b2v_sgrid_get_voxels(b2v_sgrid *g, int32_t min_count, float min_confidence) {
    if (!g) return -1;
    GridQuery q;
    fill_all_query(&q, min_count);
    return sgrid_run_readout(g, q, min_confidence);
}

extern "C" int64_t b2v_sgrid_get_voxels_in_bb(b2v_sgrid *g, const double bbox[6], int32_t min_count,
                                              float min_confidence) {
    if (!g || !bbox) return -1;
    GridQuery q;
    fill_box_query(&q, bbox, min_count, g->inv_voxel_size);
    return sgrid_run_readout(g, q, min_confidence);
}

extern "C" int64_t b2v_sgrid_get_voxels_in_frustum(b2v_sgrid *g, const float K[4], int32_t width, int32_t height,
                                                   const double Tcw[16], float depth_max, float depth_min,
                                                   int32_t min_count, float min_confidence) {
    if (!g || !K || !Tcw || width <= 0 || height <= 0) return -1;
    GridQuery q;
    fill_frustum_query(&q, K, width, height, Tcw, depth_max, depth_min, min_count, g->inv_voxel_size);
    return sgrid_run_readout(g, q, min_confidence);
}

extern "C" int b2v_sgrid_copy_voxels(b2v_sgrid *g, double *points, float *colors, int32_t *class_ids,
                                     int32_t *object_ids, float *confidences) {
    if (!g) return B2V_ERR_INVALID_ARGUMENT;
    const size_t n = static_cast<size_t>(g->last_n);
    B2V_CUDA(g, cudaSetDevice(g->device));
    if (n) {
        if (points) B2V_CUDA(g, cudaMemcpyAsync(points, g->d_out_pts, n * 3 * sizeof(double), cudaMemcpyDefault, g->stream));
        if (colors) B2V_CUDA(g, cudaMemcpyAsync(colors, g->d_out_cols, n * 3 * sizeof(float), cudaMemcpyDefault, g->stream));
        if (class_ids) B2V_CUDA(g, cudaMemcpyAsync(class_ids, g->d_out_cls, n * sizeof(int32_t), cudaMemcpyDefault, g->stream));
        if (object_ids) B2V_CUDA(g, cudaMemcpyAsync(object_ids, g->d_out_obj, n * sizeof(int32_t), cudaMemcpyDefault, g->stream));
        if (confidences) B2V_CUDA(g, cudaMemcpyAsync(confidences, g->d_out_conf, n * sizeof(float), cudaMemcpyDefault, g->stream));
    }
    B2V_CUDA(g, cudaStreamSynchronize(g->stream));
    return B2V_OK;
}

static int sgrid_edit(b2v_sgrid *g, int op, int a, int b) {
    if (!g) return B2V_ERR_INVALID_ARGUMENT;
    const int64_t nb = b2v_sgrid_num_blocks(g);
    if (nb < 0) return B2V_ERR_CUDA;
    if (nb == 0) return B2V_OK;
    sem_edit_kernel<<<static_cast<unsigned>(nb), kVox, 0, g->stream>>>(g->G, op, a, b);
    B2V_CUDA(g, cudaGetLastError());
    B2V_CUDA(g, cudaStreamSynchronize(g->stream));
    return B2V_OK;
}

extern "C" int b2v_sgrid_remove_low_count_voxels(b2v_sgrid *g, int32_t min_count) { return sgrid_edit(g, 0, min_count, 0); }
extern "C" int b2v_sgrid_remove_low_confidence_segments(b2v_sgrid *g, int32_t min_confidence) {
    return sgrid_edit(g, 1, min_confidence, 0);
}
extern "C" int b2v_sgrid_remove_segment(b2v_sgrid *g, int32_t object_id) { return sgrid_edit(g, 2, object_id, 0); }
extern "C" int b2v_sgrid_merge_segments(b2v_sgrid *g, int32_t object_id1, int32_t object_id2) {
    return sgrid_edit(g, 3, object_id1, object_id2);
}

// Parity hook.  Arrays are [nb][512]...; any output may be NULL.  `aux` = voting confidence counter, or the
// number of label pairs of a Bayesian voxel; lab_* [nb][512][K] in ascending (object, class) order, padded with
// (-1, -1, -inf) (K <= B2V_SEM_MAX_LABELS).
extern "C" int64_t b2v_sgrid_dump_blocks(b2v_sgrid *g, int32_t *keys, uint64_t *hashes, int32_t *count, double *pos_sum,
                                         float *col_sum, int32_t *object_id, int32_t *class_id, float *confidence,
                                         int32_t *aux, int32_t K, int32_t *lab_obj, int32_t *lab_cls,
                                         float *lab_logp) {
    if (!g) return -1;
    const int64_t nb = b2v_sgrid_num_blocks(g);
    if (nb <= 0) return nb;
    const size_t nv = static_cast<size_t>(nb) * kVox;
    bool ok = true;
    auto d2h = [&](void *dst, const void *src, size_t bytes) {
        if (dst && src) ok = ok && cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDeviceToHost, g->stream) == cudaSuccess;
    };
    std::vector<int4> hk(static_cast<size_t>(nb));
    d2h(hk.data(), g->G.block_keys, hk.size() * sizeof(int4));
    d2h(count, g->G.count, nv * sizeof(int32_t));
    d2h(pos_sum, g->G.pos, nv * 3 * sizeof(double));
    d2h(col_sum, g->G.col, nv * 3 * sizeof(float));
    d2h(object_id, g->G.obj, nv * sizeof(int32_t));
    d2h(class_id, g->G.cls, nv * sizeof(int32_t));
    d2h(aux, g->G.counter, nv * sizeof(int32_t));
    std::vector<int32_t> h_count, h_ctr, lo, lc;
    std::vector<float> lp;
    const bool bayes = g->G.kind == B2V_SEM_PROBABILISTIC;
    const bool want_labels = bayes && K > 0 && (lab_obj || lab_cls || lab_logp);
    if (confidence) {
        if (bayes) {
            d2h(confidence, g->G.conf, nv * sizeof(float));
        } else {
            h_count.resize(nv);
            h_ctr.resize(nv);
            d2h(h_count.data(), g->G.count, nv * sizeof(int32_t));
            d2h(h_ctr.data(), g->G.counter, nv * sizeof(int32_t));
        }
    }
    if (want_labels) {
        if (h_ctr.empty()) {
            h_ctr.resize(nv);
            d2h(h_ctr.data(), g->G.counter, nv * sizeof(int32_t));
        }
        lo.resize(nv * kSemLabels);
        lc.resize(nv * kSemLabels);
        lp.resize(nv * kSemLabels);
        d2h(lo.data(), g->G.lab_obj, lo.size() * sizeof(int32_t));
        d2h(lc.data(), g->G.lab_cls, lc.size() * sizeof(int32_t));
        d2h(lp.data(), g->G.lab_logp, lp.size() * sizeof(float));
    }
    ok = ok && cudaStreamSynchronize(g->stream) == cudaSuccess;
    if (!ok) {
        g->err = "b2v_sgrid_dump_blocks: device copy failed";
        return -1;
    }
    dump_block_keys(hk.data(), nb, keys, hashes);
    if (confidence && !bayes)
        for (size_t v = 0; v < nv; ++v) {
            const float c = h_count[v] ? static_cast<float>(h_ctr[v]) / static_cast<float>(h_count[v]) : 0.0f;
            confidence[v] = h_count[v] ? (c < 1.0f ? c : 1.0f) : 0.0f;
        }
    if (want_labels) {
        const float ninf = -std::numeric_limits<float>::infinity();
        for (size_t v = 0; v < nv; ++v) {
            int idx[kSemLabels];
            const int nl = h_ctr[v] < kSemLabels ? h_ctr[v] : kSemLabels;
            for (int k = 0; k < nl; ++k) idx[k] = k;
            for (int a = 1; a < nl; ++a)  // insertion sort by (object, class)
                for (int q = a; q > 0; --q) {
                    const size_t i0 = v * kSemLabels + idx[q - 1], i1 = v * kSemLabels + idx[q];
                    if (lo[i0] < lo[i1] || (lo[i0] == lo[i1] && lc[i0] <= lc[i1])) break;
                    const int t = idx[q];
                    idx[q] = idx[q - 1];
                    idx[q - 1] = t;
                }
            for (int k = 0; k < K; ++k) {
                const bool have = k < nl;
                const size_t src = v * kSemLabels + (have ? idx[k] : 0);
                if (lab_obj) lab_obj[v * K + k] = have ? lo[src] : -1;
                if (lab_cls) lab_cls[v * K + k] = have ? lc[src] : -1;
                if (lab_logp) lab_logp[v * K + k] = have ? lp[src] : ninf;
            }
        }
    }
    return nb;
}


// ---- carve / instance -> object association -------------------------------------------------------------------------
extern "C" int b2v_sgrid_carve(b2v_sgrid *g, const float K[4], int32_t width, int32_t height, const double Tcw[16],
                               float depth_max, float depth_min, const float *depth, float depth_threshold) {
    if (!g) return B2V_ERR_INVALID_ARGUMENT;
    if (!K || !Tcw || !depth || width <= 0 || height <= 0) {
        g->err = "b2v_sgrid_carve: bad arguments";
        return B2V_ERR_INVALID_ARGUMENT;
    }
    const int64_t nb = b2v_sgrid_num_blocks(g);
    if (nb < 0) return B2V_ERR_CUDA;
    if (nb == 0) return B2V_OK;
    void *tmp = nullptr;
    const void *d_depth = nullptr;
    cudaError_t e = device_input(depth, static_cast<size_t>(width) * height * sizeof(float), &tmp, &d_depth, g->stream);
    if (e == cudaSuccess) {
        GridQuery q;
        fill_frustum_query(&q, K, width, height, Tcw, depth_max, depth_min, 1, g->inv_voxel_size);
        sem_carve_kernel<<<static_cast<unsigned>(nb), kVox, 0, g->stream>>>(g->G, q, static_cast<const float *>(d_depth),
                                                                             depth_threshold);
        e = cudaGetLastError();
    }
    if (e == cudaSuccess) e = cudaStreamSynchronize(g->stream);
    cudaFree(tmp);
    if (e != cudaSuccess) {
        g->err = std::string("b2v_sgrid_carve: ") + cudaGetErrorString(e);
        return B2V_ERR_CUDA;
    }
    return B2V_OK;
}

extern "C" int b2v_sgrid_set_next_object_id(b2v_sgrid *g, int32_t next_object_id) {
    if (!g) return B2V_ERR_INVALID_ARGUMENT;
    g->next_object_id = next_object_id;
    return B2V_OK;
}

extern "C" int32_t b2v_sgrid_get_next_object_id(const b2v_sgrid *g) { return g ? g->next_object_id : -1; }

extern "C" int64_t b2v_sgrid_assign_object_ids_to_instance_ids(
    b2v_sgrid *g, const float K[4], int32_t width, int32_t height, const double Tcw[16], float depth_max,
    float depth_min, const int32_t *class_image, const int32_t *instance_image, const float *depth_image,
    float depth_threshold, int32_t do_carving, float min_vote_ratio, int32_t min_votes) {
    if (!g) return -1;
    g->map_inst.clear();
    g->map_obj.clear();
    if (!K || !Tcw || !class_image || !instance_image || width <= 0 || height <= 0) {
        g->err = "b2v_sgrid_assign_object_ids_to_instance_ids: bad arguments";
        return -1;
    }
    const int64_t nb = b2v_sgrid_num_blocks(g);
    if (nb < 0) return -1;
    const size_t pixels = static_cast<size_t>(width) * height;
    const size_t nv = static_cast<size_t>(nb) * kVox;
    auto fail = [&](const char *what, cudaError_t e) {
        g->err = std::string("b2v_sgrid_assign_object_ids_to_instance_ids: ") + what + ": " + cudaGetErrorString(e);
        return static_cast<int64_t>(-1);
    };
    // host copies of the label images: the map must cover every (instance >= 0, class >= 0) pixel (:322-352)
    std::vector<int32_t> h_cls(pixels), h_inst(pixels);
    cudaError_t e = cudaMemcpy(h_cls.data(), class_image, pixels * sizeof(int32_t), cudaMemcpyDefault);
    if (e == cudaSuccess) e = cudaMemcpy(h_inst.data(), instance_image, pixels * sizeof(int32_t), cudaMemcpyDefault);
    if (e != cudaSuccess) return fail("label images", e);

    std::vector<int2> rec;
    if (nb > 0) {
        void *t_cls = nullptr, *t_inst = nullptr, *t_depth = nullptr;
        const void *d_cls = nullptr, *d_inst = nullptr, *d_depth = nullptr;
        e = device_input(class_image, pixels * sizeof(int32_t), &t_cls, &d_cls, g->stream);
        if (e == cudaSuccess) e = device_input(instance_image, pixels * sizeof(int32_t), &t_inst, &d_inst, g->stream);
        if (e == cudaSuccess && depth_image)
            e = device_input(depth_image, pixels * sizeof(float), &t_depth, &d_depth, g->stream);
        int rc = e == cudaSuccess ? B2V_OK : B2V_ERR_CUDA;
        if (rc == B2V_OK && nv > g->records_cap) {
            cudaFree(g->d_pend);
            cudaFree(g->d_records);
            g->d_pend = nullptr;
            g->d_records = nullptr;
            g->records_cap = 0;
            e = cudaMalloc(&g->d_pend, nv * sizeof(int32_t));
            if (e == cudaSuccess) e = cudaMalloc(&g->d_records, nv * sizeof(int2));
            if (e == cudaSuccess && !g->d_n_records) e = cudaMalloc(&g->d_n_records, sizeof(uint32_t));
            if (e != cudaSuccess) rc = B2V_ERR_CUDA; else g->records_cap = nv;
        }
        uint32_t n_rec = 0;
        if (rc == B2V_OK) {
            GridQuery q;
            fill_frustum_query(&q, K, width, height, Tcw, depth_max, depth_min, 1, g->inv_voxel_size);
            e = cudaMemsetAsync(g->d_pend, 0xFF, nv * sizeof(int32_t), g->stream);
            if (e == cudaSuccess) e = cudaMemsetAsync(g->d_n_records, 0, sizeof(uint32_t), g->stream);
            if (e == cudaSuccess) {
                sem_assoc_kernel<<<static_cast<unsigned>(nb), kVox, 0, g->stream>>>(
                    g->G, q, static_cast<const int32_t *>(d_cls), static_cast<const int32_t *>(d_inst),
                    static_cast<const float *>(d_depth), depth_threshold, (do_carving && depth_image) ? 1 : 0, g->d_pend,
                    g->d_records, g->d_n_records, static_cast<uint32_t>(nv));
                e = cudaGetLastError();
            }
            if (e == cudaSuccess) e = cudaMemcpyAsync(&n_rec, g->d_n_records, sizeof(uint32_t), cudaMemcpyDeviceToHost, g->stream);
            if (e == cudaSuccess) e = cudaStreamSynchronize(g->stream);
            if (e == cudaSuccess && n_rec) {
                rec.resize(n_rec);
                e = cudaMemcpy(rec.data(), g->d_records, n_rec * sizeof(int2), cudaMemcpyDeviceToHost);
            }
            if (e != cudaSuccess) rc = B2V_ERR_CUDA;
        }
        cudaFree(t_cls);
        cudaFree(t_inst);
        cudaFree(t_depth);
        if (rc != B2V_OK) return e != cudaSuccess ? fail("device pass", e) : -1;
    }

    // votes: instance id -> (object id -> count); pending voxels vote for their instance's NEW object id, handed
    // out here in ascending instance-id order (the reference hands them out in block-iteration order, :118-141)
    std::map<int32_t, std::map<int32_t, int>> votes;
    std::map<int32_t, int32_t> new_id;
    for (const int2 &r : rec)
        if (r.y == kAssocPending) new_id.emplace(r.x, 0);
    for (auto &kv : new_id) kv.second = g->next_object_id++;
    for (const int2 &r : rec) votes[r.x][r.y == kAssocPending ? new_id[r.x] : r.y] += 1;
    std::map<int32_t, int32_t> result;
    for (const auto &[inst, ov] : votes) {  // :287-320
        int max_votes = 0, winner = -1, total = 0;
        for (const auto &[obj, cnt] : ov) {
            total += cnt;
            if (cnt > max_votes) {
                max_votes = cnt;
                winner = obj;
            }
        }
        if (total < min_votes || static_cast<float>(max_votes) / static_cast<float>(total) < min_vote_ratio)
            result[inst] = -1;
        else
            result[inst] = winner;
    }
    for (size_t i = 0; i < pixels; ++i) {  // :322-352: every labelled instance of the image gets an entry
        const int32_t inst = h_inst[i];
        if (inst < 0 || h_cls[i] < 0) continue;
        if (inst == 0)
            result[0] = 0;
        else
            result.emplace(inst, -1);
    }
    for (const auto &[inst, obj] : result) {
        g->map_inst.push_back(inst);
        g->map_obj.push_back(obj);
    }
    if (!new_id.empty() && nb > 0) {  // deferred assignment of the pending voxels
        int32_t *d_mi = nullptr, *d_mo = nullptr;
        const size_t m = g->map_inst.size();
        e = cudaMalloc(&d_mi, m * sizeof(int32_t));
        if (e == cudaSuccess) e = cudaMalloc(&d_mo, m * sizeof(int32_t));
        if (e == cudaSuccess) e = cudaMemcpyAsync(d_mi, g->map_inst.data(), m * sizeof(int32_t), cudaMemcpyHostToDevice, g->stream);
        if (e == cudaSuccess) e = cudaMemcpyAsync(d_mo, g->map_obj.data(), m * sizeof(int32_t), cudaMemcpyHostToDevice, g->stream);
        if (e == cudaSuccess) {
            sem_assoc_apply_kernel<<<static_cast<unsigned>(nb), kVox, 0, g->stream>>>(g->G, g->d_pend, d_mi, d_mo,
                                                                                       static_cast<int>(m));
            e = cudaGetLastError();
        }
        if (e == cudaSuccess) e = cudaStreamSynchronize(g->stream);
        cudaFree(d_mi);
        cudaFree(d_mo);
        if (e != cudaSuccess) return fail("apply", e);
    }
    return static_cast<int64_t>(g->map_inst.size());
}

extern "C" int b2v_sgrid_copy_instance_map(b2v_sgrid *g, int32_t *instance_ids, int32_t *object_ids) {
    if (!g) return B2V_ERR_INVALID_ARGUMENT;
    for (size_t i = 0; i < g->map_inst.size(); ++i) {
        if (instance_ids) instance_ids[i] = g->map_inst[i];
        if (object_ids) object_ids[i] = g->map_obj[i];
    }
    return B2V_OK;
}
