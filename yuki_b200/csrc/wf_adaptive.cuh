// Adaptive sampling (yk_render_opts.adaptive): at each check point, the still sampling pixels of a pixel group that have
// converged get their films and sample counts, and the others are compacted, in order, into the group's next job list.
// Separate kernels, launched only for adaptive renders: the render's own kernels are unchanged.
// Part of the single translation unit render.cu (compiled --fmad=false: every float op is the reference's un-fused IEEE op).
#pragma once
#include "wf_common.cuh"
#include "wf_aov.cuh"

namespace {

constexpr int kAdaptiveThreads = 256;  // block size of k_adaptive_check and k_adaptive_compact (one per-block survivor count)
constexpr int kAdaptiveScanThreads = 1024;

// The stopping rule of one channel after n samples (yuki_gpu.h, yk_adaptive): the squared standard error of the mean within
// (rel * mean + abs)^2. Only + - * / and comparisons, un-fused, so that a float32 restatement on the host gives the same
// decision; a NaN compares false and never stops.
__device__ __forceinline__ bool adaptive_converged(float s, float q, float n, float rel, float abs_err) {
    const float m = s / n;
    float v = q / n - m * m;
    if (v < 0.0f) v = 0.0f;
    const float e2 = v / (n - 1.0f);
    const float t = rel * m + abs_err;
    return e2 <= t * t;
}

// One thread per job after `count` samples of each: a pixel stops when all three channels converged (every pixel with
// `stop_all`, the group's last samples), and then gets film = sum / n (k_film_store's division), each requested companion film
// its sum / n, and its count. `keep[j]` marks the survivors and `block_keep` counts them per block (both null with stop_all).
// `sums.v[kAovRadianceSq]` holds the pixels' sums of li * li.
__global__ void k_adaptive_check(const Job* jobs, uint32_t n_jobs, uint32_t res_x, uint32_t count, uint32_t stop_all, float rel,
                                 float abs_err, const float* accum, AovSums sums, AovSums views, float* film, uint32_t* counts,
                                 uint8_t* keep, uint32_t* block_keep) {
    const uint32_t j = blockIdx.x * blockDim.x + threadIdx.x;
    bool stop = true;
    if (j < n_jobs) {
        const Job job = jobs[j];
        const size_t px = (size_t)job.y * res_x + job.x, p = px * 3;
        const float n = (float)count;
        if (!stop_all) {
            const float* q = sums.v[kAovRadianceSq];
            stop = adaptive_converged(accum[p], q[p], n, rel, abs_err) && adaptive_converged(accum[p + 1], q[p + 1], n, rel, abs_err) &&
                   adaptive_converged(accum[p + 2], q[p + 2], n, rel, abs_err);
        }
        if (stop) {
            film[p] = accum[p] / n;
            film[p + 1] = accum[p + 1] / n;
            film[p + 2] = accum[p + 2] / n;
            for (int k = 0; k < kAovViews; ++k) {
                if (!views.v[k]) continue;
                views.v[k][p] = sums.v[k][p] / n;
                views.v[k][p + 1] = sums.v[k][p + 1] / n;
                views.v[k][p + 2] = sums.v[k][p + 2] / n;
            }
            if (counts) counts[px] = count;
        }
        if (keep) keep[j] = stop ? 0 : 1;
    }
    if (block_keep) {  // (uniform over the block)
        const int kept = __syncthreads_count(!stop);
        if (threadIdx.x == 0) block_keep[blockIdx.x] = (uint32_t)kept;
    }
}

// One block: the exclusive prefix sum of the per-block survivor counts, in place, and their total.
__global__ void k_adaptive_scan(uint32_t* v, uint32_t n, uint32_t* total) {
    __shared__ uint32_t warp_incl[32];
    __shared__ uint32_t carry;
    const uint32_t lane = threadIdx.x & 31, warp = threadIdx.x >> 5, n_warps = blockDim.x >> 5;
    if (threadIdx.x == 0) carry = 0;
    for (uint32_t base = 0; base < n; base += blockDim.x) {
        __syncthreads();
        const uint32_t i = base + threadIdx.x;
        const uint32_t x = i < n ? v[i] : 0u;
        uint32_t incl = x;
        for (int d = 1; d < 32; d <<= 1) {
            const uint32_t y = __shfl_up_sync(0xffffffffu, incl, d);
            if ((int)lane >= d) incl += y;
        }
        if (lane == 31) warp_incl[warp] = incl;
        __syncthreads();
        if (warp == 0) {
            uint32_t t = lane < n_warps ? warp_incl[lane] : 0u;
            for (int d = 1; d < 32; d <<= 1) {
                const uint32_t y = __shfl_up_sync(0xffffffffu, t, d);
                if ((int)lane >= d) t += y;
            }
            warp_incl[lane] = t;
        }
        __syncthreads();
        const uint32_t c = carry;
        if (i < n) v[i] = c + (warp ? warp_incl[warp - 1] : 0u) + incl - x;
        __syncthreads();
        if (threadIdx.x == 0) carry = c + warp_incl[n_warps - 1];
    }
    __syncthreads();
    if (threadIdx.x == 0) *total = carry;
}

// The survivors' jobs, in their order, to `out` at the block's offset (k_adaptive_scan) plus their rank within the block: a
// warp of the next batch still holds neighbouring pixels, and the list does not depend on scheduling.
__global__ void k_adaptive_compact(const Job* jobs, uint32_t n_jobs, const uint8_t* keep, const uint32_t* block_off, Job* out) {
    __shared__ uint32_t warp_kept[kAdaptiveThreads / 32];
    const uint32_t j = blockIdx.x * blockDim.x + threadIdx.x;
    const uint32_t lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const bool k = j < n_jobs && keep[j];
    const uint32_t ballot = __ballot_sync(0xffffffffu, k);
    if (lane == 0) warp_kept[warp] = (uint32_t)__popc(ballot);
    __syncthreads();
    if (!k) return;
    uint32_t off = block_off[blockIdx.x];
    for (uint32_t w = 0; w < warp; ++w) off += warp_kept[w];
    out[off + (uint32_t)__popc(ballot & ((1u << lane) - 1u))] = jobs[j];
}

}  // namespace
