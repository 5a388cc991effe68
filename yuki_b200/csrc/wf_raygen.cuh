// Per-group set-up and ray generation kernels: pixel jobs expanded from the tile list, the (pixel, dimension) hash table,
// the sampler seek table, and camera rays (integrators/mod.rs:145-169).
// Part of the single translation unit render.cu (compiled --fmad=false: every float op is the reference's un-fused IEEE op).
#pragma once
#include "wf_common.cuh"

namespace {

// ---- pixel jobs of one pixel group, expanded on the device from the tile list -----------------------------------
// Job j of a render is pixel (j - off[t]) of tile t in row-major order (Bounds2 iteration, math/bounds.rs:102-126), tiles
// in list order; `off` is the prefix sum of the tile areas. Also hash_values!(pixel.x, pixel.y), the pixel's sampler
// stream (uniform.rs:77, stratified.rs:95). The host uploads 16 bytes per tile instead of 8 per pixel.
__global__ void k_jobs_expand(const yk_tile* tiles, const unsigned long long* off, uint32_t t_lo, uint32_t t_hi, unsigned long long j0,
                              uint32_t n, uint32_t accumulate, Job* out) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const unsigned long long j = j0 + i;
    uint32_t lo = t_lo, hi = t_hi;  // off[lo] <= j < off[hi]
    while (hi - lo > 1) {
        const uint32_t mid = lo + (hi - lo) / 2;
        if (off[mid] <= j) lo = mid;
        else hi = mid;
    }
    const yk_tile tl = tiles[lo];
    const uint32_t local = (uint32_t)(j - off[lo]), w = (uint32_t)tl.x1 - tl.x0;
    const uint32_t row = local / w;
    Job o;
    o.x = (uint16_t)(tl.x0 + (local - row * w));
    o.y = (uint16_t)(tl.y0 + row);
    o.sample_begin = accumulate ? tl.sample : 0u;
    o.rng_inc = (hash_pixel(o.x, o.y) << 1) | 1ULL;
    out[i] = o;
}

// yk_debug_ray: the freshly cloned sampler of launch_debug_ray draws from PCG stream 0 (`Pcg32::new(seed, 0)`, stratified.rs:73,
// uniform.rs:57), not from the pixel's stream
__global__ void k_debug_job(Job* jobs) { jobs[0].rng_inc = 1ULL; }

// hash_values!(pixel.x, pixel.y, dimension, seed) for every (dimension, pixel) of a pixel group (SamplerCfg::hash_table)
__global__ void k_dim_hashes(const Job* jobs, uint32_t n_jobs, uint32_t n_dims, unsigned long long seed, uint32_t* out) {
    const uint32_t j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= n_jobs) return;
    const Job job = jobs[j];
    for (uint32_t dim = blockIdx.y; dim < n_dims; dim += gridDim.y)
        out[(size_t)dim * n_jobs + j] = (uint32_t)hash_pixel_dim_seed(job.x, job.y, dim, seed);
}

// ---- raygen: Integrator::render loop head (integrators/mod.rs:145-169) -----------------------------
// `rng.advance(sample_index * 65536)` (uniform.rs:81-83, stratified.rs:99-101) is an LCG jump: state' = M * state + inc * P
// with M, P functions of the distance only (the jump's additive term is linear in the stream increment). A tiny kernel
// (k_sample_jumps) tabulates (M, P) for the batch's consecutive sample indices, so seeking costs two multiplies instead of the
// O(log n) loop — which was most of this kernel's instructions.
constexpr uint32_t kMaxBatchSamples = 1024;  // consecutive sample indices of a pixel per batch (size of the jump table)
struct SampleJump {
    unsigned long long mult, plus;
};
// jumps[k] = the (M, P) of Lcg64Xsh32::advance((first_sample + k) * 65536) for increment 1
__global__ void k_sample_jumps(uint32_t first_sample, uint32_t n, SampleJump* jumps) {
    const uint32_t k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= n) return;
    unsigned long long delta = (unsigned long long)(first_sample + k) * 65536ull, am = 1, ap = 0, cm = kPcgMult, cp = 1;
    while (delta) {
        if (delta & 1ull) { am *= cm; ap = ap * cm + cp; }
        cp = (cm + 1ull) * cp;
        cm *= cm;
        delta >>= 1;
    }
    jumps[k] = SampleJump{am, ap};
}
// sampling/mod.rs:68-87 (ConcentricSampleDisk), the map cosine_hemisphere inlines; restated here so that the shading kernels'
// code stays as it is
__device__ __forceinline__ V2 concentric_disk(V2 u) {
    const float ox = u.x * 2.0f - 1.0f, oy = u.y * 2.0f - 1.0f;
    if (ox == 0.0f && oy == 0.0f) return {0.0f, 0.0f};
    float theta, r;
    if (fabsf(ox) > fabsf(oy)) { theta = kPiOver4 * (oy / ox); r = ox; }
    else { theta = kPiOver2 - kPiOver4 * (ox / oy); r = oy; }
    return {cos_f32(theta) * r, sin_f32(theta) * r};
}
__global__ void k_raygen(Wave w, RenderCfg cfg, Batch bt, uint32_t first_sample, uint32_t n_jumps, const SampleJump* jumps, IterCounters* first) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= bt.n_paths) return;
    if (i == 0) first->n_active = bt.n_paths;
    const uint32_t si = bt.div_jobs.div(i), ji = i - si * bt.n_jobs;
    const Job job = bt.jobs[ji];
    const uint32_t sample = job.sample_begin + bt.sample_off + si;
    SamplerState s;
    const uint32_t slot = sample - first_sample;
    if (slot < n_jumps) {  // (always, for the batches yk_render builds)
        s.px = job.x; s.py = job.y; s.index = sample; s.dim = 0; s.job = ji;
        s.rng.inc = job.rng_inc;
        const unsigned long long seeded = (cfg.sampler.seed + job.rng_inc) * kPcgMult + job.rng_inc;  // Lcg64Xsh32::new
        const SampleJump j = jumps[slot];
        s.rng.state = j.mult * seeded + job.rng_inc * j.plus;
    } else {
        s.start(cfg.sampler, job.x, job.y, sample, job.rng_inc, ji);
    }
    const V2 j = s.get_2d(cfg.sampler);
    // Camera::ray, camera.rs:105-114
    // (yk_debug_ray: the sampler belongs to pixel (0, 0) — a fresh clone, window.rs:884 — but the ray leaves through debug_px)
    const float fx = cfg.debug_log ? cfg.debug_px[0] : (float)job.x, fy = cfg.debug_log ? cfg.debug_px[1] : (float)job.y;
    const V3 p_cam = xf_point(cfg.r2c, mk(fx + j.x, fy + j.y, 0.0f));
    const V3 d_cam = unit(p_cam);
    const V3 o = xf_point(cfg.c2w, mk(0.0f, 0.0f, 0.0f));
    const V3 d = xf_vec(cfg.c2w, d_cam);
    st_once(&w.st[0].ray_o[i], make_float4(o.x, o.y, o.z, __int_as_float(0x7f800000)));
    st_once(&w.st[0].ray_d[i], make_float4(d.x, d.y, d.z, 0.0f));
    st_once(&w.st[0].rng[i], (unsigned long long)s.rng.state);
    if (cfg.integrator == YK_INTEGRATOR_WHITTED) st_once(&w.st[0].beta[i], make_float4(__uint_as_float(s.dim), 1.0f, 1.0f, __uint_as_float(kFlagAlive)));
    else st_once(&w.st[0].beta[i], make_float4(1.0f, 1.0f, 1.0f, __uint_as_float(kFlagAlive | (s.dim << kDimShift))));
    st_once(&w.L[i], make_float4(0.0f, 0.0f, 0.0f, 0.0f));
}

// k_raygen for a thin lens of radius > 0 (yk_thin_lens, include/yuki_gpu.h: pbrt-v3's PerspectiveCamera::GenerateRay): the path's
// second get_2d is the lens sample. A kernel of its own, so that the pinhole's code stays as it is.
__global__ void k_raygen_lens(Wave w, RenderCfg cfg, Batch bt, uint32_t first_sample, uint32_t n_jumps, const SampleJump* jumps, IterCounters* first,
                              float lens_radius, float focal_distance) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= bt.n_paths) return;
    if (i == 0) first->n_active = bt.n_paths;
    const uint32_t si = bt.div_jobs.div(i), ji = i - si * bt.n_jobs;
    const Job job = bt.jobs[ji];
    const uint32_t sample = job.sample_begin + bt.sample_off + si;
    SamplerState s;
    const uint32_t slot = sample - first_sample;
    if (slot < n_jumps) {
        s.px = job.x; s.py = job.y; s.index = sample; s.dim = 0; s.job = ji;
        s.rng.inc = job.rng_inc;
        const unsigned long long seeded = (cfg.sampler.seed + job.rng_inc) * kPcgMult + job.rng_inc;
        const SampleJump j = jumps[slot];
        s.rng.state = j.mult * seeded + job.rng_inc * j.plus;
    } else {
        s.start(cfg.sampler, job.x, job.y, sample, job.rng_inc, ji);
    }
    const V2 j = s.get_2d(cfg.sampler);
    const V3 p_cam = xf_point(cfg.r2c, mk((float)job.x + j.x, (float)job.y + j.y, 0.0f));
    const V3 d_cam = unit(p_cam);
    const V2 l = concentric_disk(s.get_2d(cfg.sampler));
    const float lx = lens_radius * l.x, ly = lens_radius * l.y;
    const float ft = focal_distance / d_cam.z;
    const V3 f = d_cam * ft;  // the point on the plane of focus
    const V3 o_cam = mk(lx, ly, 0.0f);
    const V3 o = xf_point(cfg.c2w, o_cam);
    const V3 d = xf_vec(cfg.c2w, unit(f - o_cam));
    st_once(&w.st[0].ray_o[i], make_float4(o.x, o.y, o.z, __int_as_float(0x7f800000)));
    st_once(&w.st[0].ray_d[i], make_float4(d.x, d.y, d.z, 0.0f));
    st_once(&w.st[0].rng[i], (unsigned long long)s.rng.state);
    if (cfg.integrator == YK_INTEGRATOR_WHITTED) st_once(&w.st[0].beta[i], make_float4(__uint_as_float(s.dim), 1.0f, 1.0f, __uint_as_float(kFlagAlive)));
    else st_once(&w.st[0].beta[i], make_float4(1.0f, 1.0f, 1.0f, __uint_as_float(kFlagAlive | (s.dim << kDimShift))));
    st_once(&w.L[i], make_float4(0.0f, 0.0f, 0.0f, 0.0f));
}

}  // namespace
