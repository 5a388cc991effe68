// Ray-batch queries against a scene's BVH: BoundingVolumeHierarchy::intersect / any_intersect (bvh.rs:160-302) called
// directly, the way the reference's own callers outside the integrators do (Scene::intersect from launch_debug_ray,
// VisibilityTester::unoccluded). The traversal kernels are the wavefront's; these kernels only move caller rays into
// the wavefront's ray arrays and results back out.
#pragma once
#include "wf_common.cuh"
#include "wf_shade.cuh"

namespace {

// rays (o, d, t_max) -> bounce-0 ray stream; the queue is the identity (slot i = ray i). `nan_flag` (device-resident rays,
// whose t_max the host cannot scan) is set to 1 when a t_max is NaN (Ray::new, math/ray.rs).
__global__ void k_query_pack(Wave w, const float* __restrict__ o, const float* __restrict__ d, const float* __restrict__ t_max, uint32_t n,
                             int* __restrict__ nan_flag) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const float tm = t_max ? t_max[i] : __int_as_float(0x7f800000);
    if (nan_flag && tm != tm) *nan_flag = 1;
    w.st[0].ray_o[i] = make_float4(o[3 * i], o[3 * i + 1], o[3 * i + 2], t_max ? tm + 0.0f : tm);  // (-0 -> +0)
    w.st[0].ray_d[i] = make_float4(d[3 * i], d[3 * i + 1], d[3 * i + 2], 0.0f);
}
// hits -> t (inf on a miss), the shape's original id (-1 on a miss), and the (tests, hits) node counters of bvh.rs:177-179;
// a null output is not written
__global__ void k_query_unpack(DevScene sc, Wave w, uint32_t n, float* __restrict__ t_out, int32_t* __restrict__ id_out, uint32_t* __restrict__ counts) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const uint2 h = w.hit[i];
    const bool hit = h.y != kMiss;
    if (t_out) t_out[i] = hit ? __uint_as_float(h.x) : __int_as_float(0x7f800000);
    if (id_out) id_out[i] = hit ? (int32_t)__float_as_uint(sc.tris[3 * h.y + 2].w) : -1;
    if (counts) {
        const uint2 c = w.bvh_counts[i];
        counts[2 * i] = c.x;
        counts[2 * i + 1] = c.y;
    }
}
// Scene::intersect's SurfaceInteraction for the traced rays: make_surface called as k_debug_shade calls it (the caller's ray
// from the bounce-0 stream, the hit slot from w.hit). Misses: surface 0, material and area light -1. Null outputs are skipped.
struct QuerySurfaceOut {
    int32_t* material;
    int32_t* area_light;
    float *p, *n, *uv, *sh_n, *sh_dpdu;
};
__global__ void k_query_surface(DevScene sc, Wave w, uint32_t n, QuerySurfaceOut out) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const uint2 h = w.hit[i];
    Surface si{};
    si.area_light = -1;
    int32_t material = -1;
    if (h.y != kMiss) {
        uint32_t m;
        make_surface(sc, h.y, f4v(w.st[0].ray_o[i]), f4v(w.st[0].ray_d[i]), &si, &m);
        material = (int32_t)m;
    }
    auto st3 = [i](float* dst, V3 v) {
        if (dst) { dst[3 * i] = v.x; dst[3 * i + 1] = v.y; dst[3 * i + 2] = v.z; }
    };
    if (out.material) out.material[i] = material;
    if (out.area_light) out.area_light[i] = si.area_light;
    st3(out.p, si.p);
    st3(out.n, si.n);
    if (out.uv) { out.uv[2 * i] = si.uv.x; out.uv[2 * i + 1] = si.uv.y; }
    st3(out.sh_n, si.sh_n);
    st3(out.sh_dpdu, si.sh_dpdu);
}

// Segments o -> o + d as the one "light" of path i, with a unit contribution and no target area light: after the shadow /
// fold kernel L[i].x is 1 for an unoccluded segment and 0 for an occluded one.
__global__ void k_query_pack_segments(Wave w, const float* __restrict__ o, const float* __restrict__ d, uint32_t n) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    w.sh_path[i] = i;
    w.sh_mask[i] = 1u;
    w.pend_extra[i] = make_float4(0.0f, 0.0f, 0.0f, __uint_as_float(1u));
    w.pend_beta[i] = make_float4(1.0f, 1.0f, 1.0f, 0.0f);
    w.L[i] = make_float4(0.0f, 0.0f, 0.0f, 0.0f);
    w.lt_o[i] = make_float4(o[3 * i], o[3 * i + 1], o[3 * i + 2], 1.0f);
    w.lt_d[i] = make_float4(d[3 * i], d[3 * i + 1], d[3 * i + 2], 0.0f);
    w.lt_c[i] = make_float2(0.0f, __int_as_float(-1));
}
// per_ray: the segments went through k_trace_shadow_rays (an occluded segment lost its bit); else through k_trace_shadow's fold
__global__ void k_query_unpack_segments(Wave w, uint32_t n, int per_ray, uint8_t* __restrict__ out) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    out[i] = per_ray ? ((w.sh_mask[i] & 1u) ? 0 : 1) : (w.L[i].x == 0.0f ? 1 : 0);
}

// Sampler::{start_pixel_sample(p, index, 0), get_1d, get_2d} (sampling/mod.rs:46-57, uniform.rs:72-94, stratified.rs:90-143)
// for n (pixel, sample index) pairs: each thread starts a sampler the way Integrator::render does (integrators/mod.rs:163)
// and performs the same sequence of draws (pattern[k] = 1: get_1d, 2: get_2d); out holds sum(pattern) floats per pair.
__global__ void k_sampler_draws(SamplerCfg cfg, const uint32_t* __restrict__ pixel_index, uint32_t n, const uint8_t* __restrict__ pattern,
                                uint32_t n_pattern, uint32_t floats_per_pair, float* __restrict__ out) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const uint32_t px = pixel_index[3 * i], py = pixel_index[3 * i + 1], index = pixel_index[3 * i + 2];
    SamplerState s;
    s.start(cfg, px, py, index, (hash_pixel(px, py) << 1) | 1ULL, 0);
    float* o = out + (size_t)i * floats_per_pair;
    for (uint32_t k = 0; k < n_pattern; ++k) {
        if (pattern[k] == 1) {
            *o++ = s.get_1d(cfg);
        } else {
            const V2 u = s.get_2d(cfg);
            *o++ = u.x;
            *o++ = u.y;
        }
    }
}

}  // namespace
