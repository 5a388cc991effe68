// Companion films of a Path / Whitted render (yk_render_opts.aovs): the debug integrators' views of the first hit, and each
// pixel's sum of squared radiance. Separate kernels, launched only when a view is requested: the render's own kernels are
// unchanged.
// Part of the single translation unit render.cu (compiled --fmad=false: every float op is the reference's un-fused IEEE op).
#pragma once
#include "wf_common.cuh"
#include "wf_shade.cuh"

namespace {

constexpr int kAovViews = 5;  // yk_aov_films order: bvh_intersections, geometry_normals, shading_normals, shading_uvs, radiance_sq
constexpr int kAovRadianceSq = 4;

// Per-pixel sums the views add into: the accumulators carried across batches (zeroed per pixel group, like yk_context::d_accum),
// or the views themselves for accumulating films. Null = not requested.
struct AovSums {
    float* v[kAovViews];
};

// One pixel's view sum: `sum += c` over ascending samples in registers (averaging films), or, for accumulating films (one sample
// per pixel per batch), one atomicAdd as k_film_add does, so that tiles of one sample index that overlap lose no add.
struct AovAcc {
    float r = 0.0f, g = 0.0f, b = 0.0f;
    __device__ void load(const float* o) { r = o[0]; g = o[1]; b = o[2]; }
    __device__ void add(float* o, bool atomic, float cr, float cg, float cb) {
        if (atomic) { atomicAdd(o, cr); atomicAdd(o + 1, cg); atomicAdd(o + 2, cb); }
        else { r = r + cr; g = g + cg; b = b + cb; }
    }
    __device__ void store(float* o) const { o[0] = r; o[1] = g; o[2] = b; }
};

// k_debug_shade's four films (bvh_heatmap.rs, geometry_normals.rs, shading_normals.rs, shading_uvs.rs) from bounce 0 of a
// Path / Whitted batch, summed like k_film_accumulate: one thread per pixel job, its samples in ascending order. Runs between
// bounce 0's closest-hit kernel and bounce 1's, which overwrites the hits, the counters and st[0]'s rays (slot == path here).
// `atomic`: accumulating film (bt.n_samples == 1), the views are added into with k_film_add's atomics.
__global__ void k_aov_first_hit(DevScene sc, Wave w, Batch bt, AovSums a, uint32_t res_x, uint32_t atomic) {
    const uint32_t j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= bt.n_jobs) return;
    const Job job = bt.jobs[j];
    const size_t px = ((size_t)job.y * res_x + job.x) * 3;
    float* o[4];
    AovAcc acc[4];
    for (int k = 0; k < 4; ++k) {
        o[k] = a.v[k] ? a.v[k] + px : nullptr;
        if (o[k] && !atomic) acc[k].load(o[k]);
    }
    const bool surface = o[1] || o[2] || o[3];
    for (uint32_t s = 0; s < bt.n_samples; ++s) {
        const size_t path = (size_t)s * bt.n_jobs + j;
        const uint2 h = w.hit[path];
        if (o[0]) {
            const uint2 cnt = w.bvh_counts[path];
            const RGB c = rgb((float)cnt.x, (float)cnt.y, h.y != kMiss ? (float)cnt.y : 0.0f);
            acc[0].add(o[0], atomic, c.r, c.g, c.b);
        }
        if (!surface) continue;
        RGB c3[3] = {gray(0.0f), gray(0.0f), gray(0.0f)};
        if (h.y != kMiss) {
            Surface si;
            uint32_t m;
            make_surface(sc, h.y, f4v(w.st[0].ray_o[path]), f4v(w.st[0].ray_d[path]), &si, &m);
            c3[0] = rgb(si.n.x, si.n.y, si.n.z) / 2.0f + gray(0.5f);
            c3[1] = rgb(si.sh_n.x, si.sh_n.y, si.sh_n.z) / 2.0f + gray(0.5f);
            c3[2] = rgb(si.uv.x, si.uv.y, 0.0f);
        }
        for (int k = 0; k < 3; ++k)
            if (o[1 + k]) acc[1 + k].add(o[1 + k], atomic, c3[k].r, c3[k].g, c3[k].b);
    }
    if (!atomic)
        for (int k = 0; k < 4; ++k)
            if (o[k]) acc[k].store(o[k]);
}

// k_film_accumulate for `li * li`: the per-channel second moment, in the film's sample order (`atomic`: accumulating film, as
// k_aov_first_hit).
__global__ void k_film_accumulate_sq(Wave w, Batch bt, float* sums, uint32_t res_x, uint32_t atomic) {
    const uint32_t j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= bt.n_jobs) return;
    const Job job = bt.jobs[j];
    float* o = sums + ((size_t)job.y * res_x + job.x) * 3;
    AovAcc acc;
    if (!atomic) acc.load(o);
    for (uint32_t s = 0; s < bt.n_samples; ++s) {
        const float4 L = w.L[(size_t)s * bt.n_jobs + j];
        acc.add(o, atomic, L.x * L.x, L.y * L.y, L.z * L.z);
    }
    if (!atomic) acc.store(o);
}

}  // namespace
