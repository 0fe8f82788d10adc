// b2v_scan.cuh — single-CTA exclusive scan over per-block counts (n <= a few million entries).
// Used by the count -> scan -> emit passes of the mesher and of the point grids' read-outs.
#pragma once

#include <cstdint>
#include <cuda_runtime.h>

namespace b2v {

// out[i] = sum(in[0..i)), *total = sum(in[0..n)).  blockIdx.x selects one of several independent
// arrays laid out back to back with stride n.
static __global__ void __launch_bounds__(1024)
exclusive_scan_kernel(const uint32_t *__restrict__ in_all, uint32_t *__restrict__ out_all,
                      uint32_t *__restrict__ totals, const uint32_t n) {
    __shared__ uint32_t s_warp[32];
    __shared__ uint32_t s_carry;
    const uint32_t *in = in_all + static_cast<size_t>(blockIdx.x) * n;
    uint32_t *out = out_all + static_cast<size_t>(blockIdx.x) * n;
    const int t = threadIdx.x, lane = t & 31, wid = t >> 5;
    if (t == 0) s_carry = 0;
    __syncthreads();
    for (uint32_t base = 0; base < n; base += 1024) {
        const uint32_t i = base + t;
        const uint32_t v = i < n ? in[i] : 0u;
        uint32_t x = v;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            const uint32_t y = __shfl_up_sync(0xffffffffu, x, d);
            if (lane >= d) x += y;
        }
        if (lane == 31) s_warp[wid] = x;
        __syncthreads();
        if (wid == 0) {
            uint32_t w = s_warp[lane];
#pragma unroll
            for (int d = 1; d < 32; d <<= 1) {
                const uint32_t y = __shfl_up_sync(0xffffffffu, w, d);
                if (lane >= d) w += y;
            }
            s_warp[lane] = w;
        }
        __syncthreads();
        const uint32_t carry = s_carry;
        const uint32_t incl = x + (wid ? s_warp[wid - 1] : 0u);
        if (i < n) out[i] = carry + incl - v;
        __syncthreads();
        if (t == 1023) s_carry = carry + incl;
        __syncthreads();
    }
    if (t == 0) totals[blockIdx.x] = s_carry;
}

// ---- two-level scan for the mesher (n ~ 1e5 .. 5e5: the single-CTA loop above costs ~1 us per 1024 entries) ----
// grid = (chunks of 1024, arrays).  Pass 1 reduces every chunk; pass 2 adds the partials before the CTA's chunk (at most
// 512 of them) and scans the chunk.
static __global__ void __launch_bounds__(1024)
scan_reduce_kernel(const uint32_t *__restrict__ in_all, uint32_t *__restrict__ partials, const uint32_t n) {
    __shared__ uint32_t s_warp[32];
    const uint32_t *in = in_all + static_cast<size_t>(blockIdx.y) * n;
    const int t = threadIdx.x, lane = t & 31, wid = t >> 5;
    const uint32_t i = blockIdx.x * 1024u + t;
    uint32_t x = i < n ? in[i] : 0u;
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) x += __shfl_down_sync(0xffffffffu, x, d);
    if (lane == 0) s_warp[wid] = x;
    __syncthreads();
    if (wid == 0) {
        uint32_t w = s_warp[lane];
#pragma unroll
        for (int d = 16; d > 0; d >>= 1) w += __shfl_down_sync(0xffffffffu, w, d);
        if (lane == 0) partials[blockIdx.y * gridDim.x + blockIdx.x] = w;
    }
}

static __global__ void __launch_bounds__(1024)
scan_apply_kernel(const uint32_t *__restrict__ in_all, uint32_t *__restrict__ out_all,
                  const uint32_t *__restrict__ partials, uint32_t *__restrict__ totals, const uint32_t n) {
    __shared__ uint32_t s_warp[32];
    __shared__ uint32_t s_prefix;
    const uint32_t *in = in_all + static_cast<size_t>(blockIdx.y) * n;
    uint32_t *out = out_all + static_cast<size_t>(blockIdx.y) * n;
    const uint32_t *part = partials + blockIdx.y * gridDim.x;
    const int t = threadIdx.x, lane = t & 31, wid = t >> 5;
    // sum of the chunks before this one
    uint32_t p = 0;
    for (uint32_t c = t; c < blockIdx.x; c += 1024u) p += part[c];
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) p += __shfl_down_sync(0xffffffffu, p, d);
    if (lane == 0) s_warp[wid] = p;
    __syncthreads();
    if (wid == 0) {
        uint32_t w = s_warp[lane];
#pragma unroll
        for (int d = 16; d > 0; d >>= 1) w += __shfl_down_sync(0xffffffffu, w, d);
        if (lane == 0) s_prefix = w;
    }
    __syncthreads();
    const uint32_t prefix = s_prefix;
    // scan of the chunk
    const uint32_t i = blockIdx.x * 1024u + t;
    const uint32_t v = i < n ? in[i] : 0u;
    uint32_t x = v;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        const uint32_t y = __shfl_up_sync(0xffffffffu, x, d);
        if (lane >= d) x += y;
    }
    __syncthreads();   // s_warp is reused
    if (lane == 31) s_warp[wid] = x;
    __syncthreads();
    if (wid == 0) {
        uint32_t w = s_warp[lane];
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            const uint32_t y = __shfl_up_sync(0xffffffffu, w, d);
            if (lane >= d) w += y;
        }
        s_warp[lane] = w;
    }
    __syncthreads();
    const uint32_t incl = x + (wid ? s_warp[wid - 1] : 0u);
    if (i < n) out[i] = prefix + incl - v;
    if (blockIdx.x == gridDim.x - 1 && t == 1023) totals[blockIdx.y] = prefix + incl;
}

// sums[blockIdx.x] = the number of threads of a 512-thread CTA that pass `keep`; s_warp: 16 words
static __device__ __forceinline__ void block_count_512(bool keep, uint32_t *s_warp, uint32_t *sums) {
    const int t = threadIdx.x;
    const uint32_t x = __reduce_add_sync(0xffffffffu, keep ? 1u : 0u);
    if ((t & 31) == 0) s_warp[t >> 5] = x;
    __syncthreads();
    if (t == 0) {
        uint32_t s = 0;
        for (int k = 0; k < 16; ++k) s += s_warp[k];
        sums[blockIdx.x] = s;
    }
}

// block-wide exclusive scan of one value per thread for a 512-thread CTA; s_warp: 16 words
static __device__ __forceinline__ uint32_t block_excl_scan_512(uint32_t v, uint32_t *s_warp) {
    const int t = threadIdx.x, lane = t & 31, wid = t >> 5;
    uint32_t x = v;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        const uint32_t y = __shfl_up_sync(0xffffffffu, x, d);
        if (lane >= d) x += y;
    }
    if (lane == 31) s_warp[wid] = x;
    __syncthreads();
    if (wid == 0) {
        uint32_t w = lane < 16 ? s_warp[lane] : 0u;
#pragma unroll
        for (int d = 1; d < 16; d <<= 1) {
            const uint32_t y = __shfl_up_sync(0xffffffffu, w, d);
            if (lane >= d) w += y;
        }
        if (lane < 16) s_warp[lane] = w;
    }
    __syncthreads();
    return x - v + (wid ? s_warp[wid - 1] : 0u);
}

}  // namespace b2v
