// The material sort (classify) and the per-material shading kernels: surface set-up, BSDFs, light sampling, the Path and
// Whitted integrator bodies (integrators/path.rs, whitted.rs), and the debug integrators.
// Part of the single translation unit render.cu (compiled --fmad=false: every float op is the reference's un-fused IEEE op).
#pragma once
#include "wf_common.cuh"
#include "wf_trace.cuh"
#include "wf_sort.cuh"

namespace {

// ---- whitted recursion frames ----------------------------------------------------------------------------
// Whitted::li_internal recurses (whitted.rs:132-170): a node's radiance is `lights (+ Le)`, then
// `+= f * li(child) * |cos|` for the reflection child, then for the transmission child. The wavefront walks that tree
// depth first, one node per path and bounce, and evaluates it bottom-up like the recursion does, so every float
// operation has the reference's operands: frame d of a path holds the partial sum of its depth-d node, the factor of the
// child being evaluated and, while the reflection subtree runs, the waiting transmission child.
//   frame[0] = sum_li.rgb | -          frame[1] = f.rgb | |cos| of the running child
//   frame[2] = waiting child: o.xyz | d.x   frame[3] = d.yz | f.rg   frame[4] = f.b | |cos| | flags (0 = none) | -
constexpr int kFrameWords = 5;
constexpr uint32_t kFramePending = 0x80000000u;
struct TreeRay {
    V3 o, d;
    uint32_t flags;  // depth | specular | transmission
};
__device__ __forceinline__ float4* frame_of(const Wave& w, uint32_t depth, uint32_t path) {
    return w.stack + ((size_t)depth * w.cap + path) * kFrameWords;
}
// The depth-`depth` node of `path` finished with radiance `li`: hand it to the parent (`sum_li += s.f * child.li * |cos|`,
// whitted.rs:160-166) and climb while the parents finish too. Returns true with the next ray of the tree when a parent
// still has its transmission child waiting; false once the root is done (its radiance is then the path's L).
__device__ __forceinline__ bool tree_return(const Wave& w, uint32_t path, uint32_t depth, RGB li, TreeRay* next) {
    while (depth > 0) {
        float4* fr = frame_of(w, depth - 1, path);
        const float4 a = fr[0], cf = fr[1], p4 = fr[4];
        const RGB sum = rgb(a.x, a.y, a.z) + rgb(cf.x, cf.y, cf.z) * li * cf.w;
        const uint32_t pflags = __float_as_uint(p4.z);
        if (pflags & kFramePending) {
            const float4 p2 = fr[2], p3 = fr[3];
            fr[0] = make_float4(sum.r, sum.g, sum.b, 0.0f);
            fr[1] = make_float4(p3.z, p3.w, p4.x, p4.y);
            fr[4] = make_float4(0.0f, 0.0f, 0.0f, 0.0f);
            next->o = mk(p2.x, p2.y, p2.z);
            next->d = mk(p2.w, p3.x, p3.y);
            next->flags = pflags & ~kFramePending;
            return true;
        }
        li = sum;
        depth -= 1;
    }
    w.L[path] = make_float4(li.r, li.g, li.b, 0.0f);
    return false;
}
// Writes a tree node as the path's next ray (the sampler state carries on: the reference shares one sampler through
// the recursion).
__device__ __forceinline__ void stream_node(const Wave::Stream& st, uint32_t pos, const TreeRay& e, uint32_t dim, unsigned long long rng) {
    st.ray_o[pos] = make_float4(e.o.x, e.o.y, e.o.z, __int_as_float(0x7f800000));
    st.ray_d[pos] = make_float4(e.d.x, e.d.y, e.d.z, 0.0f);
    st.beta[pos] = make_float4(__uint_as_float(dim), 1.0f, 1.0f, __uint_as_float(e.flags | kFlagAlive));
    st.rng[pos] = rng;
}

// ---- classify: miss handling + compaction by material ("ray-queue sort/compaction pass") ---------------
// K items per thread and block round (K * blockDim.x rays per global atomic): the queue counters are single addresses, and
// same-address atomics, not bandwidth, bound this kernel. Whitted's tree walk re-queues rays here and runs with K = 1.
#ifndef YK_CLASSIFY_ITEMS
#define YK_CLASSIFY_ITEMS 8
#endif
template <int K, bool WHITTED>
__global__ void k_classify(DevScene sc, Wave w, RenderCfg cfg, Batch bt, const uint32_t* queue, int b, IterCounters* cur,
                           IterCounters* nxt, int first_iteration, uint32_t* q_next, const uint32_t* perm) {
    const uint32_t n = cur->n_active;
    const uint32_t per_round = gridDim.x * blockDim.x * K;
    const uint32_t rounds = (n + per_round - 1) / per_round;
    for (uint32_t r = 0; r < rounds; ++r) {
        const uint32_t block_first = (r * gridDim.x + blockIdx.x) * blockDim.x * K;
        if (block_first >= n) break;  // block-uniform
        uint32_t idx[K], path[K], hit_slot[K];
        int key[K];
        TreeRay node[WHITTED ? K : 1];
        uint32_t node_dim[WHITTED ? K : 1];
        unsigned long long hh = 0;
#pragma unroll
        for (int k = 0; k < K; ++k) {
            const uint32_t j = block_first + k * blockDim.x + threadIdx.x;
            idx[k] = j;
            path[k] = 0; hit_slot[k] = kMiss; key[k] = -1;
            if (j >= n) continue;
            const uint32_t i = perm ? __ldg(&perm[j]) : j;  // the ray's queue slot (sorted renders walk the queue through perm)
            YK_ASSERT(i < n);
            idx[k] = i;
            path[k] = queue ? queue[i] : i;
            const uint2 h = ld_once(&w.hit[i]);
            hit_slot[k] = h.y;
            uint32_t orig = 0xffffffffu;
            if (h.y != kMiss) {
                key[k] = (int)((__float_as_uint(__ldg(&sc.tris[3 * h.y + 1]).w) >> 28) & 3u);
                if (first_iteration) orig = __float_as_uint(__ldg(&sc.tris[3 * h.y + 2]).w);
            } else if (first_iteration != 2) {  // (2 = debug integrators: their li() returns no background)
                const float4 bw = w.st[b].beta[i];
                if (WHITTED) {  // whitted.rs:174: this node's radiance is the background
                    node_dim[WHITTED ? k : 0] = __float_as_uint(bw.x);
                    const uint32_t depth = __float_as_uint(bw.w) & kDepthMask;
                    if (tree_return(w, path[k], depth, rgb(sc.background[0], sc.background[1], sc.background[2]), &node[WHITTED ? k : 0])) key[k] = 4;
                } else {  // path.rs:155-160: background weighted by the throughput
                    float4 L = w.L[path[k]];
                    L.x = L.x + bw.x * sc.background[0];
                    L.y = L.y + bw.y * sc.background[1];
                    L.z = L.z + bw.z * sc.background[2];
                    w.L[path[k]] = L;
                }
            }
            if (first_iteration) {
                const uint32_t si = bt.div_jobs.div(path[k]);
                const Job job = bt.jobs[path[k] - si * bt.n_jobs];
                const uint32_t sample = job.sample_begin + bt.sample_off + si;
                hh += mix_hit(job.x, job.y, sample, orig);
                if (cfg.hit_ids && sample == cfg.aux_sample) cfg.hit_ids[(size_t)job.y * cfg.res_x + job.x] = (int32_t)orig;
            }
        }
        uint32_t* const queues[5] = {w.q_mat, w.q_mat + (size_t)w.cap, w.q_mat + (size_t)2 * w.cap, w.q_mat + (size_t)3 * w.cap, q_next};
        uint32_t* const counters[5] = {&cur->mat[0], &cur->mat[1], &cur->mat[2], &cur->mat[3], &nxt->n_active};
        uint32_t pos[K];
        block_scatter_multi<5, K>(key, path, queues, counters, pos);
#pragma unroll
        for (int k = 0; k < K; ++k) {
            if (key[k] >= 0 && key[k] < 4) {
                st_once(&w.q_mat_tri[(size_t)key[k] * w.cap + pos[k]], hit_slot[k]);
                st_once(&w.q_mat_slot[(size_t)key[k] * w.cap + pos[k]], idx[k]);
            } else if (WHITTED && key[k] == 4) {
                stream_node(w.st[b ^ 1], pos[k], node[WHITTED ? k : 0], node_dim[WHITTED ? k : 0], w.st[b].rng[idx[k]]);
            }
        }
        if (first_iteration) {
            hh = warp_sum(hh);
            if ((threadIdx.x & 31) == 0 && hh) atomicAdd(&w.totals->hit_hash, hh);
        }
    }
}

// ---- surface set-up: Triangle::intersect's SurfaceInteraction part (triangle.rs:141-226) ----------------
__device__ __forceinline__ void make_surface(const DevScene& sc, uint32_t tri, V3 o, V3 d, Surface* si, uint32_t* material) {
    const float4 a4 = __ldg(&sc.tris[3 * tri]), b4 = __ldg(&sc.tris[3 * tri + 1]), c4 = __ldg(&sc.tris[3 * tri + 2]);
    const V3 p0 = mk(a4.x, b4.x, c4.x), p1 = mk(a4.y, b4.y, c4.y), p2 = mk(a4.z, b4.z, c4.z);  // stored transposed
    const uint32_t packed = __float_as_uint(b4.w);
    const uint32_t flags = (packed >> 24) & 0xfu;
    *material = packed & 0xffffffu;
    if (flags & YK_TRI_IS_SPHERE) {
        sphere_surface(sc.spheres[-2 - __float_as_int(a4.w)], o, d, si);
        return;
    }
    // Barycentrics: re-run the (deterministic) triangle test that the traversal accepted.
    TriRay tr;
    tr.setup(d);
    TriHit h{0, 0, 0, 0};
    tri_test(tr, o, __int_as_float(0x7f800000), p0, p1, p2, &h);
    V2 uv0{0.0f, 0.0f}, uv1{1.0f, 0.0f}, uv2{1.0f, 1.0f};  // triangle.rs:143-155
    if (flags & YK_TRI_HAS_UVS) {
        const float* u = sc.uvs + (size_t)tri * 6;
        uv0 = {u[0], u[1]}; uv1 = {u[2], u[3]}; uv2 = {u[4], u[5]};
    }
    const float du02 = uv0.x - uv2.x, dv02 = uv0.y - uv2.y, du12 = uv1.x - uv2.x, dv12 = uv1.y - uv2.y;
    const V3 dp02 = p0 - p2, dp12 = p1 - p2;
    const float uv_det = du02 * dv12 - dv02 * du12;
    V3 dpdu;
    if (uv_det == 0.0f) {
        V3 unused;
        frame_from(unit(cross64(p2 - p0, p1 - p0)), &dpdu, &unused);
    } else {
        const float inv = 1.0f / uv_det;
        dpdu = (dp02 * dv12 - dp12 * dv02) * inv;
    }
    si->p = p0 * h.b0 + p1 * h.b1 + p2 * h.b2;
    si->uv = {uv0.x * h.b0 + uv1.x * h.b1 + uv2.x * h.b2, uv0.y * h.b0 + uv1.y * h.b1 + uv2.y * h.b2};
    si->wo = -d;
    si->area_light = __float_as_int(a4.w);
    V3 n = unit(cross64(dp02, dp12));
    if (flags & YK_TRI_SWAPS_HANDEDNESS) n = -n;
    si->n = n;
    si->sh_n = n;
    si->sh_dpdu = dpdu;
    if (flags & YK_TRI_HAS_NORMALS) {  // triangle.rs:197-224 + set_shading_geometry, interaction.rs:126-132
        const float* nn = sc.normals + (size_t)tri * 9;
        const V3 n0 = mk(nn[0], nn[1], nn[2]), n1 = mk(nn[3], nn[4], nn[5]), n2 = mk(nn[6], nn[7], nn[8]);
        V3 ns = unit(n0 * h.b0 + n1 * h.b1 + n2 * h.b2);
        if (dot0(ns, ns) > 0.0f) ns = unit(ns);
        else ns = si->n;
        V3 ss = unit(dpdu);
        V3 ts = cross64(ss, ns);
        if (dot0(ts, ts) > 0.0f) {
            ts = unit(ts);
            ss = cross64(ts, ns);
        } else {
            frame_from(ns, &ss, &ts);
        }
        si->sh_n = unit(cross64(ss, ts));
        si->n = flip_toward_n(si->n, si->sh_n);
        si->sh_dpdu = ss;
    }
}

// textures/constant.rs:23-30, textures/image_texture.rs:81-111
__device__ __noinline__ RGB tex_image_eval(const DevTexture& t, V2 uv);
__device__ __forceinline__ RGB tex_eval(const DevScene& sc, int32_t index, V2 uv) {
    const DevTexture& t = sc.textures[index];
    if (t.kind == YK_TEX_CONSTANT) return rgb(t.value[0], t.value[1], t.value[2]);
    return tex_image_eval(t, uv);
}
__device__ __noinline__ RGB tex_image_eval(const DevTexture& t, V2 uv) {
    float sx = uv.x - truncf(uv.x), sy = uv.y - truncf(uv.y);
    if (sx < 0.0f) sx = 1.0f + sx;
    if (sy < 0.0f) sy = 1.0f + sy;
    sy = 1.0f - sy;
    sx = sx * (float)t.width - 0.5f;
    sy = sy * (float)t.height - 0.5f;
    const uint32_t ix = sx > 0.0f ? (uint32_t)sx : 0u, iy = sy > 0.0f ? (uint32_t)sy : 0u;
    const float* px = t.texels + ((size_t)iy * t.width + ix) * 3;
    return rgb(__ldg(px), __ldg(px + 1), __ldg(px + 2));
}

static __device__ __noinline__ float roughness_to_alpha(float r) {  // trowbridge_reitz.rs:22-30 (rare: image-textured roughness)
    const float x = yklibm::logf_glibc(fmaxf(r, 0.001f));  // f32::ln = glibc's logf, restated (yk_libm.h)
    return 1.62142f + 0.819955f * x + 0.1734f * x * x + 0.0171201f * x * x * x + 0.000640711f * x * x * x * x;
}

template <uint32_t KIND>
__device__ __forceinline__ void make_bsdf(const DevScene& sc, const DevMaterial& m, const Surface& si, Bsdf* b) {
    b->kind = KIND;
    b->empty = false;
    b->ng = si.n;
    b->ns = si.sh_n;
    b->ss = unit(si.sh_dpdu);
    b->ts = cross64(b->ns, b->ss);
    b->c1 = gray(0.0f);
    b->p0 = 0.0f;
    b->p1 = -1.0f;
    if (KIND == YK_MAT_MATTE) {  // matte.rs:22-40, oren_nayar.rs:18-25
        b->c0 = tex_eval(sc, m.tex[0], si.uv);
        const float sigma = tex_eval(sc, m.tex[1], si.uv).r;
        b->empty = black(b->c0);
        if (sigma != 0.0f) {
            const float s2 = sigma * sigma;
            b->p0 = 1.0f - (s2 / (2.0f * (s2 + 0.33f)));
            b->p1 = 0.45f * s2 / (s2 + 0.09f);
            if (b->p1 < 0.0f) b->p1 = 0.0f;  // cannot happen for real sigma; keeps the Lambertian tag (p1 < 0) unambiguous
        }
    } else if (KIND == YK_MAT_GLASS) {  // glass.rs:27-45
        b->c0 = tex_eval(sc, m.tex[0], si.uv);
        b->c1 = tex_eval(sc, m.tex[1], si.uv);
        b->p0 = m.eta;
    } else if (KIND == YK_MAT_METAL) {  // metal.rs:34-61, trowbridge_reitz.rs:16-20
        b->c0 = tex_eval(sc, m.tex[0], si.uv);
        b->c1 = tex_eval(sc, m.tex[1], si.uv);
        if (m.const_alpha >= 0.0f) b->p0 = m.const_alpha;
        else {
            float r = tex_eval(sc, m.tex[2], si.uv).r;
            if (m.remap) r = roughness_to_alpha(r);
            b->p0 = fmaxf(r, 0.001f);
        }
    } else {  // glossy.rs:32-58 (alpha = roughness^2)
        b->c0 = tex_eval(sc, m.tex[0], si.uv);
        if (m.const_alpha >= 0.0f) b->p0 = m.const_alpha;
        else {
            float r = tex_eval(sc, m.tex[1], si.uv).r;
            if (m.remap) r = roughness_to_alpha(r);
            b->p0 = fmaxf(r * r, 0.001f);
        }
    }
}

// Light::sample_li for the four light kinds (lights/*.rs). Returns false when no visibility test exists.
struct LightSample {
    V3 l;
    RGB li;
    float pdf;
    bool has_vis;
    Ray vis;
    int vis_light;
};
__device__ __forceinline__ void sample_light(const yk_light& L, int index, const Surface& si, V2 u, LightSample* s) {
    s->vis_light = -1;
    s->pdf = 1.0f;
    s->has_vis = true;
    const RGB I = rgb(L.i[0], L.i[1], L.i[2]);
    const V3 lp = mk(L.p[0], L.p[1], L.p[2]);
    if (L.kind == YK_LIGHT_POINT) {  // point_light.rs:27-49
        const V3 to = lp - si.p;
        const float d2 = dot0(to, to);
        s->li = I / d2;
        s->l = to / sqrtf(d2);
        s->vis = spawn_ray_to(si.p, si.n, lp);
    } else if (L.kind == YK_LIGHT_SPOT) {  // spot_light.rs:38-80
        const V3 to = lp - si.p;
        const float d2 = dot0(to, to);
        s->l = to / sqrtf(d2);
        const float ct = unit(xf_vec(L.world_to_light, -s->l)).z;
        float fall;
        if (ct < L.cos_total_width) fall = 0.0f;
        else if (ct > L.cos_falloff_start) fall = 1.0f;
        else {
            const float dl = (ct - L.cos_total_width) / (L.cos_falloff_start - L.cos_total_width);
            fall = (dl * dl) * (dl * dl);
        }
        s->li = I * fall / d2;
        s->has_vis = !black(s->li);
        s->vis = spawn_ray_to(si.p, si.n, lp);
    } else if (L.kind == YK_LIGHT_RECT) {  // rectangular_light.rs:46-72
        const V3 p = xf_point(L.sample_to_world, mk(u.x, 0.0f, u.y));
        const V3 n = xf_normal(L.sample_to_world_inv, mk(0.0f, -1.0f, 0.0f));
        const V3 wi = unit(p - si.p);
        const float c = dotn(n, -wi);
        s->li = c > 0.0f ? I : gray(0.0f);
        s->l = wi;
        s->vis = spawn_ray_to(si.p, si.n, p);
        s->vis_light = index;
        const V3 dp = si.p - p;
        s->pdf = dot0(dp, dp) / (fabsf(c) * L.area);
    } else {  // distant_light.rs:24-43
        s->li = I;
        s->l = lp;
        s->vis = spawn_ray_to(si.p, si.n, si.p + lp * 10000.0f);
    }
}

// ---- shading: one kernel instance per material kind ----------------------------------------------------
// Covers Material::compute_scattering_functions, the light fold (path.rs:102-119 / whitted.rs:109-126), the
// emitted term, BSDF sampling + throughput update + Russian roulette (path.rs:121-171), and the specular
// recursion of whitted.rs:132-170 flattened onto a per-sample DFS stack (children inherit weight * f * |cos|).
// Radiance is not summed here: each light that needs a visibility test leaves its shadow ray and contribution in
// lt_*, and k_trace_shadow adds the unoccluded terms in light order. Surviving paths are appended to the next
// active queue (one atomic per block).
// Measured: prefetching a block's queue lines two rounds ahead takes 5 % off the shading kernels (+1.6 % Cornell render);
// prefetching the state those entries point to (next round's, or this round's late-used beta / rng / job) adds nothing.
#ifndef YK_SHADE_PREFETCH
#define YK_SHADE_PREFETCH 1
#endif
__device__ __forceinline__ void prefetch_l2(const void* p) { asm volatile("prefetch.global.L2 [%0];" ::"l"(p)); }

// What one shaded path hands to the survivor compaction.
struct ShadeOut {
    float4 nx_o, nx_d, nx_beta;  // the survivor's state for the next bounce, written after the compaction assigns its position
    unsigned long long nx_rng;
    uint32_t nx_key;             // ray sort: the survivor's coherence key (wf_sort.cuh)
    uint32_t path;
    bool alive;
};

// One queue entry. SYNC: the calling block is full (every thread has an entry), so the body may hold block barriers — they keep
// the block's warps inside the same phase of the ~100 KB of straight-line code (surface + BSDF set-up | one light at a time |
// emission + BSDF sampling), whose top stall with the warps spread all over it is `no_instruction` (32 KB instruction cache,
// profiles/r02/ncu_shade_room.txt). The last, partial block of a queue runs the barrier-free instantiation.
template <uint32_t KIND, bool PATH, bool SYNC>
__device__ __forceinline__ void shade_item(const DevScene& sc, const Wave& w, const RenderCfg& cfg, const Batch& bt, const uint32_t* queue,
                                           const uint32_t* queue_tri, const uint32_t* queue_slot, int b, uint32_t i, uint32_t g, ShadeOut* out) {
    const uint32_t path = ld_once(&queue[i]);
    out->path = path;
    st_once(&w.sh_path[g], path);
    const uint32_t hit_slot = ld_once(&queue_tri[i]), slot = ld_once(&queue_slot[i]);
    YK_ASSERT(path < w.cap && slot < w.cap && g < w.cap && hit_slot < sc.n_tris);
    const float4 ro = ld_once(&w.st[b].ray_o[slot]), rd = ld_once(&w.st[b].ray_d[slot]);
    const V3 o = f4v(ro), d = f4v(rd);
    Surface si;
    uint32_t mat_index;
    make_surface(sc, hit_slot, o, d, &si, &mat_index);
    Bsdf bsdf;
    make_bsdf<KIND>(sc, sc.materials[mat_index], si, &bsdf);

    const float4 beta4 = ld_once(&w.st[b].beta[slot]);
    RGB beta = rgb(beta4.x, beta4.y, beta4.z);
    const uint32_t flags = __float_as_uint(beta4.w) & kFlagMask;
    const uint32_t depth = flags & kDepthMask;  // path: bounces so far; whitted: node depth
    const bool was_specular = (flags & kFlagSpecular) != 0;

    const uint32_t sample_i = bt.div_jobs.div(path), job_i = path - sample_i * bt.n_jobs;
    const Job job = bt.jobs[job_i];
    SamplerState smp;
    smp.rng.state = ld_once(&w.st[b].rng[slot]);
    smp.rng.inc = job.rng_inc;
    smp.dim = PATH ? __float_as_uint(beta4.w) >> kDimShift : __float_as_uint(beta4.x);
    smp.px = job.x;
    smp.py = job.y;
    smp.index = job.sample_begin + bt.sample_off + sample_i;
    smp.job = job_i;

    // Light fold: every light consumes one get_2d whether it is used or not (path.rs:103).
    uint32_t shadow_mask = 0;
    for (uint32_t k = 0; k < sc.n_lights; ++k) {
        if (SYNC) __syncthreads();
        const V2 u = smp.get_2d(cfg.sampler);
        LightSample ls;
        sample_light(sc.lights[k], (int)k, si, u, &ls);
        if (!black(ls.li)) {
            const RGB f = bsdf.f(si.wo, ls.l);
            if (ls.has_vis && !black(f)) {
                const RGB c = f * ls.li * clamp01ish(dotn(si.sh_n, ls.l), 0.0f, 1.0f) / ls.pdf;
                const size_t ref = (size_t)k * w.cap + g;
                st_once(&w.lt_o[ref], make_float4(ls.vis.o.x, ls.vis.o.y, ls.vis.o.z, c.r));
                st_once(&w.lt_d[ref], make_float4(ls.vis.d.x, ls.vis.d.y, ls.vis.d.z, c.g));
                st_once(&w.lt_c[ref], make_float2(c.b, __int_as_float(ls.vis_light)));
                shadow_mask |= 1u << k;
            }
        }
    }
    if (SYNC) __syncthreads();
    if (cfg.shadow_per_ray) st_once(&w.sh_mask[g], shadow_mask);  // (k_trace_shadow reads the mask from pend_extra.w)

    // Emitted radiance: interaction.rs:134-138 + rectangular_light.rs:74-81
    RGB le = gray(0.0f);
    // The integrators pass -ray.d here and (Path) to sample_f, but si.wo to Bsdf::f; the two differ for spheres, whose
    // si.wo went through object_to_world once more (sphere.rs:116, interaction.rs:155).
    const V3 wo_ray = -d;
    if (si.area_light >= 0 && dotn(si.n, wo_ray) > 0.0f) {
        const yk_light& al = sc.lights[si.area_light];
        le = rgb(al.i[0], al.i[1], al.i[2]);
    }
    const bool add_le = depth == 0 || was_specular;

    bool alive = false;
    uint32_t new_flags = 0;
    if (PATH) {
        // path.rs:121-129 — beta multiplies the emitted term here and again in the fold (reference quirk)
        const RGB extra = add_le ? beta * le : gray(0.0f);
        st_once(&w.pend_extra[g], make_float4(extra.r, extra.g, extra.b, __uint_as_float(shadow_mask)));
        st_once(&w.pend_beta[g], make_float4(beta.r, beta.g, beta.b, (depth > 0 && cfg.has_clamp) ? 1.0f : 0.0f));
        const Bsdf::Sample s = bsdf.sample_f(wo_ray, smp.get_2d(cfg.sampler), BX_ALL);  // path.rs:131-137 (wo = -ray.d)
        if (!(black(s.f) || s.pdf == 0.0f)) {
            alive = true;
            const bool spec = (s.type & BX_SPECULAR) != 0;
            beta = beta * (s.f * fabsf(dotn(s.wi, si.sh_n)) / s.pdf);
            const Ray nr = spawn_ray(si.p, si.n, s.wi);
            if (depth > 3) {  // Russian roulette, path.rs:163-169
                // q == 1 (beta.g == 0) ends the path even when the stratified draw rounds up to exactly 1.0f: path.rs would go on
                // with beta * 1 / 0 and turn the pixel into NaN. The draw is still taken, as in the oracle.
                const float q = fmaxf(1.0f - beta.g, 0.05f);
                if (smp.get_1d(cfg.sampler) < q || q >= 1.0f) alive = false;
                else beta = beta * (gray(1.0f) / (1.0f - q));
            }
            const uint32_t bounces = depth + 1;
            if (bounces >= cfg.max_depth) alive = false;
            new_flags = (bounces & kDepthMask) | (spec ? kFlagSpecular : 0u) | ((s.type & BX_TRANSMISSION) ? kFlagTransmission : 0u);
            out->nx_o = make_float4(nr.o.x, nr.o.y, nr.o.z, nr.t_max);
            out->nx_d = make_float4(nr.d.x, nr.d.y, nr.d.z, 0.0f);
            out->nx_beta = make_float4(beta.r, beta.g, beta.b, __uint_as_float(new_flags | kFlagAlive | (smp.dim << kDimShift)));
            if (cfg.sort_key_mode) out->nx_key = ray_sort_key(sc, cfg, hit_slot, nr.o.x, nr.o.y, nr.o.z, nr.d.x, nr.d.y, nr.d.z);
        }
    } else {
        // whitted.rs:128-170: this node's own terms go to the shadow / fold kernel; k_tree_return then either parks
        // their sum in the node's frame (children pending) or hands it to the parent
        const RGB extra = add_le ? le : gray(0.0f);
        st_once(&w.pend_extra[g], make_float4(extra.r, extra.g, extra.b, __uint_as_float(shadow_mask)));
        TreeRay child[2];
        RGB child_f[2];
        float child_cos[2];
        int n_child = 0;
        if (KIND == YK_MAT_GLASS && depth + 1 < cfg.max_depth) {  // only Glass owns SPECULAR lobes
            const uint32_t wants[2] = {BX_SPECULAR | BX_REFLECTION, BX_SPECULAR | BX_TRANSMISSION};
#pragma unroll
            for (int c = 0; c < 2; ++c) {
                const Bsdf::Sample s = bsdf.sample_f(si.wo, V2{0.0f, 0.0f}, wants[c]);
                if (s.type == 0u) continue;  // BxdfType::NONE: no ray, no radiance
                const Ray nr = spawn_ray(si.p, si.n, s.wi);
                TreeRay e;
                e.o = nr.o;
                e.d = nr.d;
                e.flags = ((depth + 1) & kDepthMask) | ((s.type & BX_SPECULAR) ? kFlagSpecular : 0u) | (c == 1 ? kFlagTransmission : 0u);
                child_f[n_child] = s.f;
                child_cos[n_child] = fabsf(dotn(s.wi, si.sh_n));
                child[n_child++] = e;
            }
        }
        alive = n_child >= 1;
        st_once(&w.pend_beta[g], make_float4(__uint_as_float(depth | (alive ? 0x100u : 0u)), __uint_as_float(smp.dim), 0.0f, -1.0f));
        if (alive) {
            float4* fr = frame_of(w, depth, path);
            fr[1] = make_float4(child_f[0].r, child_f[0].g, child_f[0].b, child_cos[0]);
            if (n_child == 2) {  // transmission waits until the reflection subtree is done
                fr[2] = make_float4(child[1].o.x, child[1].o.y, child[1].o.z, child[1].d.x);
                fr[3] = make_float4(child[1].d.y, child[1].d.z, child_f[1].r, child_f[1].g);
                fr[4] = make_float4(child_f[1].b, child_cos[1], __uint_as_float(child[1].flags | kFramePending), 0.0f);
            } else {
                fr[4] = make_float4(0.0f, 0.0f, 0.0f, 0.0f);
            }
            const TreeRay& e = child[0];
            out->nx_o = make_float4(e.o.x, e.o.y, e.o.z, __int_as_float(0x7f800000));
            out->nx_d = make_float4(e.d.x, e.d.y, e.d.z, 0.0f);
            out->nx_beta = make_float4(__uint_as_float(smp.dim), 1.0f, 1.0f, __uint_as_float(e.flags | kFlagAlive));
        } else {
            w.tree_rng[g] = smp.rng.state;  // the sampler goes on with whichever node the tree visits next
        }
    }
    out->nx_rng = smp.rng.state;
    out->alive = alive;
}

// PHASED: blocks of kShadeThreads with the phase barriers of shade_item (scenes with several lights / material kinds, where the
// instruction cache is the limiter); else blocks of kShadeThreadsPlain without barriers (the Cornell-box class: one light, two
// kinds — measured 0.7 % faster there with two pipes, while the room gains 5 % from the phases; profiles/r02).
template <uint32_t KIND, bool PATH, bool PHASED>
__global__ void __launch_bounds__(PHASED ? kShadeThreads : kShadeThreadsPlain, PHASED ? YK_SHADE_MIN_BLOCKS : (1024 / kShadeThreadsPlain))
    k_shade(DevScene sc, Wave w, RenderCfg cfg, Batch bt, const uint32_t* queue, const uint32_t* queue_tri, const uint32_t* queue_slot, int b,
            IterCounters* cur, IterCounters* nxt, uint32_t* q_next) {
    const uint32_t n = cur->mat[KIND];
    uint32_t g_base = 0;  // shading position of this kind's first queue entry (classify has finished: the counts are final)
    if (KIND > 0) g_base += cur->mat[0];
    if (KIND > 1) g_base += cur->mat[1];
    if (KIND > 2) g_base += cur->mat[2];
    const uint32_t rounds = (n + gridDim.x * blockDim.x - 1) / (gridDim.x * blockDim.x);
    for (uint32_t r = 0; r < rounds; ++r) {
        const uint32_t block_first = (r * gridDim.x + blockIdx.x) * blockDim.x;
        if (block_first >= n) break;  // block-uniform
        const uint32_t i = block_first + threadIdx.x;
#if YK_SHADE_PREFETCH
        // the block's queue entries two rounds ahead: pull them into the L2 now (one 128-byte line per warp and queue)
        if ((threadIdx.x & 31) == 0) {
            const uint32_t i_ahead = i + 2 * gridDim.x * blockDim.x;
            if (i_ahead < n) { prefetch_l2(queue + i_ahead); prefetch_l2(queue_tri + i_ahead); prefetch_l2(queue_slot + i_ahead); }
        }
#endif
        ShadeOut so;
        so.nx_o = so.nx_d = so.nx_beta = make_float4(0, 0, 0, 0);
        so.nx_rng = 0; so.nx_key = 0; so.path = 0; so.alive = false;
        if (PHASED && block_first + blockDim.x <= n) shade_item<KIND, PATH, true>(sc, w, cfg, bt, queue, queue_tri, queue_slot, b, i, g_base + i, &so);
        else if (i < n) shade_item<KIND, PATH, false>(sc, w, cfg, bt, queue, queue_tri, queue_slot, b, i, g_base + i, &so);
        uint32_t* const queues[1] = {q_next};
        uint32_t* const counters[1] = {&nxt->n_active};
        const uint32_t npos = block_scatter<1>(so.alive ? 0 : -1, so.path, queues, counters);
        if (so.alive) {  // a finished path's ray / throughput / sampler state is never read again
            YK_ASSERT(npos < w.cap);
            const Wave::Stream& out = w.st[b ^ 1];
            st_once(&out.ray_o[npos], so.nx_o);
            st_once(&out.ray_d[npos], so.nx_d);
            st_once(&out.beta[npos], so.nx_beta);
            st_once(&out.rng[npos], so.nx_rng);
            if (PATH && cfg.sort_key_mode) w.sort_key[npos] = so.nx_key;
        }
    }
}

// ---- Whitted: nodes shaded this bounce return their radiance ---------------------------------------------
// Runs after the shadow / fold kernel, which left `lights (+ Le)` of every node shaded this bounce in pend_extra. A node
// with children parks it in its frame; a finished node hands it up the tree (tree_return), which may release a waiting
// transmission ray into the next bounce's queue.
__global__ void k_tree_return(Wave w, int b, IterCounters* cur, IterCounters* nxt, uint32_t* q_next) {
    const uint32_t n = cur->mat[0] + cur->mat[1] + cur->mat[2] + cur->mat[3];
    const uint32_t rounds = (n + gridDim.x * blockDim.x - 1) / (gridDim.x * blockDim.x);
    for (uint32_t r = 0; r < rounds; ++r) {
        const uint32_t block_first = (r * gridDim.x + blockIdx.x) * blockDim.x;
        if (block_first >= n) break;  // block-uniform
        const uint32_t g = block_first + threadIdx.x;
        bool alive = false;
        uint32_t path = 0, dim = 0;
        TreeRay next;
        if (g < n) {
            path = w.sh_path[g];
            const float4 info = w.pend_beta[g], li4 = w.pend_extra[g];
            const uint32_t word = __float_as_uint(info.x), depth = word & kDepthMask;
            dim = __float_as_uint(info.y);
            if (word & 0x100u) frame_of(w, depth, path)[0] = make_float4(li4.x, li4.y, li4.z, 0.0f);
            else alive = tree_return(w, path, depth, rgb(li4.x, li4.y, li4.z), &next);
        }
        uint32_t* const queues[1] = {q_next};
        uint32_t* const counters[1] = {&nxt->n_active};
        const uint32_t npos = block_scatter<1>(alive ? 0 : -1, path, queues, counters);
        if (alive) stream_node(w.st[b ^ 1], npos, next, dim, w.tree_rng[g]);
    }
}

// ---- Integrator::li_debug (integrators/mod.rs:103-118): the ray list of one path ------------------------
// yk_debug_ray renders a single path through the ordinary wavefront kernels; this one-thread kernel runs after each bounce's
// closest-hit kernel and appends what Path / Whitted::li_internal collect (path.rs:71-113, whitted.rs:89-121): the bounce ray
// (cut at the hit, else at the scene bounds for Path's secondary rays), the geometric normal at the hit, and the shadow ray
// of every light sample that carries a visibility test. It re-draws the light samples from a copy of the path's sampler
// state, exactly as the shading kernel that follows does.
__global__ void k_debug_log(DevScene sc, Wave w, RenderCfg cfg, Batch bt, int b, const IterCounters* cur) {
    if (threadIdx.x != 0 || blockIdx.x != 0 || cur->n_active == 0) return;
    DebugLog* log = cfg.debug_log;
    auto push = [&](V3 o, V3 d, float t_max, uint32_t type) {
        const uint32_t k = log->count++;
        if (k >= log->cap) return;
        yk_integrator_ray r;
        r.o[0] = o.x; r.o[1] = o.y; r.o[2] = o.z;
        r.d[0] = d.x; r.d[1] = d.y; r.d[2] = d.z;
        r.t_max = t_max;
        r.ray_type = type;
        log->rays[k] = r;
    };
    const float4 ro = w.st[b].ray_o[0], rd = w.st[b].ray_d[0], beta4 = w.st[b].beta[0];
    const V3 o = f4v(ro), d = f4v(rd);
    const uint2 h = w.hit[0];
    const uint32_t word = __float_as_uint(beta4.w), depth = word & kDepthMask;
    const uint32_t type = depth == 0 ? YK_RAY_DIRECT : ((word & kFlagTransmission) ? YK_RAY_REFRACTION : YK_RAY_REFLECTION);
    float t_log = ro.w;  // ray.t_max
    if (h.y != kMiss) {
        t_log = __uint_as_float(h.x);
    } else if (cfg.integrator == YK_INTEGRATOR_PATH && type != YK_RAY_DIRECT) {  // Bounds3::intersections, math/bounds.rs:176-205
        const float ix = 1.0f / d.x, iy = 1.0f / d.y, iz = 1.0f / d.z;
        const float t0x = (sc.root_min[0] - o.x) * ix, t0y = (sc.root_min[1] - o.y) * iy, t0z = (sc.root_min[2] - o.z) * iz;
        const float t1x = (sc.root_max[0] - o.x) * ix, t1y = (sc.root_max[1] - o.y) * iy, t1z = (sc.root_max[2] - o.z) * iz;
        const float tmin = fmaxf(fmaxf(fminf(t0x, t1x), fmaxf(fminf(t0y, t1y), fminf(t0z, t1z))), 0.0f);
        const float tmax = fminf(fminf(fmaxf(t0x, t1x), fminf(fmaxf(t0y, t1y), fmaxf(t0z, t1z))), ro.w);
        t_log = tmin <= tmax ? tmax : log->min_len;
    }
    push(o, d, t_log, type);
    if (h.y == kMiss) return;
    Surface si;
    uint32_t mat_index;
    make_surface(sc, h.y, o, d, &si, &mat_index);
    push(si.p, si.n, log->min_len, YK_RAY_NORMAL);
    const Job job = bt.jobs[0];
    SamplerState smp;
    smp.rng.state = w.st[b].rng[0];
    smp.rng.inc = job.rng_inc;
    smp.dim = cfg.integrator == YK_INTEGRATOR_WHITTED ? __float_as_uint(beta4.x) : word >> kDimShift;
    smp.px = job.x;
    smp.py = job.y;
    smp.index = job.sample_begin + bt.sample_off;
    smp.job = 0;
    for (uint32_t k = 0; k < sc.n_lights; ++k) {
        const V2 u = smp.get_2d(cfg.sampler);
        LightSample ls;
        sample_light(sc.lights[k], (int)k, si, u, &ls);
        if (!black(ls.li) && ls.has_vis) push(ls.vis.o, ls.vis.d, ls.vis.t_max, YK_RAY_SHADOW);
    }
}

// ---- debug integrators (bvh_heatmap.rs, geometry_normals.rs, shading_normals.rs, shading_uvs.rs) --------
__global__ void k_debug_shade(DevScene sc, Wave w, RenderCfg cfg, uint32_t n) {
    const uint32_t path = blockIdx.x * blockDim.x + threadIdx.x;
    if (path >= n) return;
    const uint2 h = w.hit[path];
    RGB c = gray(0.0f);
    if (cfg.integrator == YK_INTEGRATOR_BVH_INTERSECTIONS) {
        const uint2 cnt = w.bvh_counts[path];
        c = rgb((float)cnt.x, (float)cnt.y, h.y != kMiss ? (float)cnt.y : 0.0f);
    } else if (h.y != kMiss) {
        Surface si;
        uint32_t m;
        make_surface(sc, h.y, f4v(w.st[0].ray_o[path]), f4v(w.st[0].ray_d[path]), &si, &m);  // first bounce: slot == path
        if (cfg.integrator == YK_INTEGRATOR_GEOMETRY_NORMALS) c = rgb(si.n.x, si.n.y, si.n.z) / 2.0f + gray(0.5f);
        else if (cfg.integrator == YK_INTEGRATOR_SHADING_NORMALS) c = rgb(si.sh_n.x, si.sh_n.y, si.sh_n.z) / 2.0f + gray(0.5f);
        else c = rgb(si.uv.x, si.uv.y, 0.0f);
    }
    w.L[path] = make_float4(c.r, c.g, c.b, 0.0f);
}

}  // namespace
