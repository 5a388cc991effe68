// ORACLE — TEST INFRASTRUCTURE ONLY (see yko_math.h header).
//
// CPU restatement of yuki's integrators (integrators/{mod,whitted,path,bvh_heatmap,geometry_normals,
// shading_normals,shading_uvs}.rs), film tiling (film.rs) and the tile-queue worker model of
// renderer/{render_manager,render_worker}.rs. PARITY UNPINNED (no reference tests/goldens exist for the
// path); follows the cited lines, quirks included.
#pragma once
#include <atomic>
#include <deque>
#include <mutex>
#include <thread>

#include "yko_bsdf.h"

namespace yko {

enum IntegratorKind : uint32_t {
    INTEGRATOR_WHITTED = 0,
    INTEGRATOR_PATH = 1,
    INTEGRATOR_BVH_INTERSECTIONS = 2,
    INTEGRATOR_GEOMETRY_NORMALS = 3,
    INTEGRATOR_SHADING_NORMALS = 4,
    INTEGRATOR_SHADING_UVS = 5,
};
struct Integrator {
    IntegratorKind kind;
    uint32_t max_depth;      // whitted.rs:21-25 / path.rs:25-32: default 3
    bool has_clamp;
    float indirect_clamp;
};

struct RadianceResult {
    Spec li{0, 0, 0};
    uint64_t rays = 0;
};

struct ThreadStats {
    TraversalStats ts;
    uint64_t shadow_rays = 0;
    uint64_t primary_hit_hash = 0;
};

// Order-independent digest of every primary hit: sum over (pixel, sample) of mix(x, y, sample, id).
inline uint64_t mix_hit(uint32_t x, uint32_t y, uint32_t sample, uint32_t id) {
    uint64_t h = ((uint64_t)x << 48) ^ ((uint64_t)y << 32) ^ ((uint64_t)sample << 8) ^ (uint64_t)id * 0x9E3779B97F4A7C15ULL;
    h ^= h >> 31; h *= 0xBF58476D1CE4E5B9ULL; h ^= h >> 29;
    return h;
}

struct RenderCtx {
    const Scene& scene;
    const Integrator& integ;
    ThreadStats* st;
};

// integrators/mod.rs:76-89: the rays li_debug() collects for the ray visualisation.
enum RayType : uint32_t { RAY_DIRECT = 0, RAY_REFLECTION = 1, RAY_REFRACTION = 2, RAY_NORMAL = 3, RAY_SHADOW = 4 };
struct IntegratorRay {
    Ray ray;
    uint32_t ray_type;
};
using RayLog = std::vector<IntegratorRay>;

// whitted.rs:84-88 / path.rs:58-62
inline float min_debug_ray_length(const Scene& scene) {
    Bounds3 b = scene.bounds();
    int i = maximum_extent(b);
    const float hi = i == 0 ? b.p_max.x : (i == 1 ? b.p_max.y : b.p_max.z), lo = i == 0 ? b.p_min.x : (i == 1 ? b.p_min.y : b.p_min.z);
    return (hi - lo) / 10.0f;
}
// Bounds3::intersections, math/bounds.rs:196-205: the far slab distance, if the ray meets the box at all.
inline bool bounds_intersections_tmax(const Bounds3& b, const Ray& ray, float* t_max) {
    V3 inv_dir = {1.0f / ray.d.x, 1.0f / ray.d.y, 1.0f / ray.d.z};
    V3 a0 = b.p_min - ray.o, a1 = b.p_max - ray.o;
    V3 t0 = {a0.x * inv_dir.x, a0.y * inv_dir.y, a0.z * inv_dir.z};
    V3 t1 = {a1.x * inv_dir.x, a1.y * inv_dir.y, a1.z * inv_dir.z};
    float tmin = fmax_(max_comp(vmin(t0, t1)), 0.0f);
    float tmax = fmin_(min_comp(vmax(t0, t1)), ray.t_max);
    *t_max = tmax;
    return tmin <= tmax;
}

// Direct lighting fold shared by Whitted (whitted.rs:109-126) and Path (path.rs:102-119). `rays` (li_debug only) receives
// the shadow ray of every light sample that carries a visibility test, occluded or not, black f or not.
inline Spec light_fold(const RenderCtx& c, const SurfaceInteraction& si, const Bsdf& bsdf, Sampler& sampler, RayLog* rays = nullptr) {
    Spec acc = spec1(0.0f);
    for (int32_t li = 0; li < (int32_t)c.scene.lights.size(); ++li) {
        LightSample ls = sample_li(c.scene, li, si, sampler.get_2d());  // every light consumes a get_2d
        if (!is_black(ls.li)) {
            Spec f = bsdf.f(si.wo, ls.l, BXDF_ALL);
            if (ls.has_vis) {
                if (rays) rays->push_back({ls.vis_ray, RAY_SHADOW});
                if (!is_black(f)) {
                    c.st->shadow_rays += 1;
                    if (!c.scene.any_intersect(ls.vis_ray, ls.vis_area_light, &c.st->ts))
                        acc = acc + f * ls.li * clampf(dot_nv(si.sh_n, ls.l), 0.0f, 1.0f) / ls.pdf;
                }
            }
        }
    }
    return acc;
}

// whitted.rs:74-182 (+ specular_contribution :38-70)
inline RadianceResult whitted_li(const RenderCtx& c, Ray ray, uint32_t depth, Sampler& sampler, bool is_specular,
                                 int32_t* primary_id, RayLog* rays = nullptr) {
    IntersectionResult ir = c.scene.intersect(ray, &c.st->ts);
    if (primary_id) *primary_id = ir.has_hit ? (int32_t)c.scene.shapes[ir.hit.shape].orig_id : -1;
    if (rays) {  // :89-105
        rays->push_back({ray, RAY_DIRECT});
        if (ir.has_hit) {
            rays->back().ray.t_max = ir.hit.t;
            rays->push_back({Ray{ir.hit.si.p, ir.hit.si.n, min_debug_ray_length(c.scene)}, RAY_NORMAL});
        }
    }
    RadianceResult out;
    if (!ir.has_hit) {
        out.li = c.scene.background;
        out.rays = 1;
        return out;
    }
    const SurfaceInteraction& si = ir.hit.si;
    const Triangle& tri = c.scene.shapes[ir.hit.shape];
    Bsdf bsdf = compute_scattering_functions(c.scene, c.scene.materials[tri.material], si);
    uint64_t ray_count = 1;
    Spec sum_li = light_fold(c, si, bsdf, sampler, rays);
    if (depth == 0 || is_specular) sum_li += emitted_radiance(c.scene, si, -ray.d);
    if (depth + 1 < c.integ.max_depth) {
        const uint8_t kinds[2] = {BXDF_REFLECTION, BXDF_TRANSMISSION};
        for (int k = 0; k < 2; ++k) {
            BxdfSample s = bsdf.sample_f(si.wo, V2{0.0f, 0.0f}, (uint8_t)(BXDF_SPECULAR | kinds[k]));
            if (s.sample_type == BXDF_NONE) continue;  // zero radiance, zero rays
            Ray refl = spawn_ray(si.p, si.n, s.wi);
            const size_t first_child_ray = rays ? rays->size() : 0;
            RadianceResult child =
                whitted_li(c, refl, depth + 1, sampler, (s.sample_type & BXDF_SPECULAR) != 0, nullptr, rays);
            // :136-160: the subtree's rays are appended with its first ray re-typed
            if (rays && rays->size() > first_child_ray) (*rays)[first_child_ray].ray_type = k == 0 ? RAY_REFLECTION : RAY_REFRACTION;
            sum_li += s.f * child.li * std::fabs(dot_nv(s.wi, si.sh_n));
            ray_count += child.rays;
        }
    }
    out.li = sum_li;
    out.rays = ray_count;
    return out;
}

// path.rs:49-178
inline RadianceResult path_li(const RenderCtx& c, Ray ray, Sampler& sampler, int32_t* primary_id, RayLog* rays = nullptr) {
    Spec L = spec1(0.0f), beta = spec1(1.0f);
    uint32_t bounces = 0;
    bool specular_bounce = false;
    uint64_t ray_count = 0;
    if (primary_id) *primary_id = -1;
    uint32_t ray_type = RAY_DIRECT;  // only used when collecting into `rays`
    while (bounces < c.integ.max_depth) {
        if (rays) {  // :71-86: bounce rays are drawn up to the scene bounds until a hit shortens them
            float t_max = ray.t_max;
            if (ray_type != RAY_DIRECT && !bounds_intersections_tmax(c.scene.bounds(), ray, &t_max)) t_max = min_debug_ray_length(c.scene);
            rays->push_back({Ray{ray.o, ray.d, t_max}, ray_type});
        }
        ray_count += 1;
        IntersectionResult ir = c.scene.intersect(ray, &c.st->ts);
        if (bounces == 0 && primary_id && ir.has_hit) *primary_id = (int32_t)c.scene.shapes[ir.hit.shape].orig_id;
        if (ir.has_hit) {
            const SurfaceInteraction& si = ir.hit.si;
            const Triangle& tri = c.scene.shapes[ir.hit.shape];
            if (rays) {  // :91-98
                rays->back().ray.t_max = ir.hit.t;
                rays->push_back({Ray{si.p, si.n, min_debug_ray_length(c.scene)}, RAY_NORMAL});
            }
            Bsdf bsdf = compute_scattering_functions(c.scene, c.scene.materials[tri.material], si);
            Spec radiance = light_fold(c, si, bsdf, sampler, rays);
            // :121-123 — beta is applied here AND again below (reference quirk, reproduced)
            if (bounces == 0 || specular_bounce) radiance += beta * emitted_radiance(c.scene, si, -ray.d);
            if (bounces > 0 && c.integ.has_clamp) radiance = smin(radiance, spec1(1.0f) * c.integ.indirect_clamp);
            L += beta * radiance;
            V3 wo = -ray.d;
            BxdfSample s = bsdf.sample_f(wo, sampler.get_2d(), BXDF_ALL);
            if (is_black(s.f) || s.pdf == 0.0f) break;
            specular_bounce = (s.sample_type & BXDF_SPECULAR) != 0;
            beta *= s.f * std::fabs(dot_nv(s.wi, si.sh_n)) / s.pdf;
            ray = spawn_ray(si.p, si.n, s.wi);
            ray_type = (s.sample_type & BXDF_REFLECTION) ? RAY_REFLECTION : RAY_REFRACTION;  // :146-153 (anything else panics there)
        } else {
            L += beta * c.scene.background;
            break;
        }
        if (bounces > 3) {  // :163-169 Russian roulette
            // Deviation: q == 1 (beta.g == 0) breaks even when the stratified draw rounds up to exactly 1.0f, where the
            // reference goes on with beta * 1 / 0 and returns NaN for the pixel. The draw is still taken.
            float q = fmax_(1.0f - beta.g, 0.05f);
            if (sampler.get_1d() < q || q >= 1.0f) break;
            beta *= spec1(1.0f) / (1.0f - q);
        }
        bounces += 1;
    }
    return {L, ray_count};
}

// Integrator::li_debug (integrators/mod.rs:103-118): Whitted and Path collect rays, the debug integrators keep the trait's
// default (zero radiance, no rays, zero ray count).
inline RadianceResult integrator_li_debug(const RenderCtx& c, Ray ray, Sampler& sampler, RayLog* rays) {
    switch (c.integ.kind) {
        case INTEGRATOR_WHITTED: return whitted_li(c, ray, 0, sampler, false, nullptr, rays);
        case INTEGRATOR_PATH: return path_li(c, ray, sampler, nullptr, rays);
        default: return RadianceResult{};
    }
}

inline RadianceResult integrator_li(const RenderCtx& c, Ray ray, Sampler& sampler, int32_t* primary_id) {
    switch (c.integ.kind) {
        case INTEGRATOR_WHITTED: return whitted_li(c, ray, 0, sampler, false, primary_id);
        case INTEGRATOR_PATH: return path_li(c, ray, sampler, primary_id);
        default: break;
    }
    IntersectionResult ir = c.scene.intersect(ray, &c.st->ts);
    if (primary_id) *primary_id = ir.has_hit ? (int32_t)c.scene.shapes[ir.hit.shape].orig_id : -1;
    RadianceResult out;
    out.rays = 1;
    switch (c.integ.kind) {
        case INTEGRATOR_BVH_INTERSECTIONS:  // bvh_heatmap.rs:17-46
            out.li = spec((float)ir.intersection_test_count, (float)ir.intersection_count,
                          ir.has_hit ? (float)ir.intersection_count : 0.0f);
            break;
        case INTEGRATOR_GEOMETRY_NORMALS:  // geometry_normals.rs:15-39
            if (ir.has_hit) { V3 n = ir.hit.si.n / 2.0f + v3(0.5f, 0.5f, 0.5f); out.li = spec(n.x, n.y, n.z); }
            break;
        case INTEGRATOR_SHADING_NORMALS:  // shading_normals.rs:15-43
            if (ir.has_hit) { V3 n = ir.hit.si.sh_n / 2.0f + v3(0.5f, 0.5f, 0.5f); out.li = spec(n.x, n.y, n.z); }
            break;
        case INTEGRATOR_SHADING_UVS:  // shading_uvs.rs:15-40
            if (ir.has_hit) out.li = spec(ir.hit.si.uv.x, ir.hit.si.uv.y, 0.0f);
            break;
        default: break;
    }
    return out;
}

// ------------------------------------------------------------------------------------------------
// Film tiles, film.rs:299-376
struct FilmTile {
    uint16_t x0, y0, x1, y1;
    uint16_t sample;
    uint32_t index;  // flat row-major tile index
};

inline std::vector<FilmTile> film_tiles(uint32_t res_x, uint32_t res_y, uint32_t tile_dim) {
    // generate_tiles :299-331
    int h_tiles = (int)std::ceil((float)res_x / (float)tile_dim);
    int v_tiles = (int)std::ceil((float)res_y / (float)tile_dim);
    std::vector<FilmTile> grid((size_t)h_tiles * v_tiles);
    uint32_t flat = 0;
    for (uint32_t j = 0; j < res_y; j += tile_dim)
        for (uint32_t i = 0; i < res_x; i += tile_dim) {
            FilmTile t{(uint16_t)i, (uint16_t)j, (uint16_t)std::min(i + tile_dim, res_x),
                       (uint16_t)std::min(j + tile_dim, res_y), 0, flat};
            grid[(size_t)(j / tile_dim) * h_tiles + (i / tile_dim)] = t;
            flat += 1;
        }
    // outward_spiral :333-376
    int center_x = (h_tiles / 2) - (1 - h_tiles % 2);
    int center_y = (v_tiles / 2) - (1 - v_tiles % 2);
    int max_dim = std::max(h_tiles, v_tiles);
    int x = 0, y = 0, dx = 0, dy = -1;
    std::vector<FilmTile> queue;
    queue.reserve(grid.size());
    for (int k = 0; k < max_dim * max_dim; ++k) {
        int tx = center_x + x, ty = center_y + y;
        if (tx >= 0 && tx < h_tiles && ty >= 0 && ty < v_tiles) queue.push_back(grid[(size_t)ty * h_tiles + tx]);
        if (x == y || (x < 0 && x == -y) || (x > 0 && x == 1 - y)) {
            std::swap(dx, dy);
            dx *= -1;
        }
        x += dx;
        y += dy;
    }
    return queue;
}

struct RenderOutputs {
    float* film;          // res_y * res_x * 3
    int32_t* hit_ids;     // optional, res_y*res_x: primary hit original triangle id of sample `aux_sample`
    uint32_t aux_sample;
};

struct RenderTotals {
    uint64_t ray_count = 0;      // closest-hit rays, the reference's ray_scene_intersections
    uint64_t shadow_rays = 0;
    uint64_t samples = 0;
    TraversalStats ts;
    uint64_t primary_hit_hash = 0;
    double seconds = 0;
    uint32_t threads = 0;
};

// Integrator::render, integrators/mod.rs:120-185, for one tile (non-accumulating or accumulating).
inline uint64_t render_tile(const Scene& scene, const Camera& cam, const Sampler& proto, const Integrator& integ,
                            bool accumulating, const FilmTile& tile, std::vector<Spec>& tile_pixels,
                            std::vector<int32_t>* tile_ids, uint32_t aux_sample, ThreadStats* st) {
    Sampler sampler = proto;  // per-tile clone, :142
    RenderCtx ctx{scene, integ, st};
    uint32_t tile_w = tile.x1 - tile.x0;
    uint64_t ray_count = 0;
    for (uint32_t y = tile.y0; y < tile.y1; ++y)
        for (uint32_t x = tile.x0; x < tile.x1; ++x) {
            Spec color = spec1(0.0f);
            uint32_t sample_count = accumulating ? 1 : sampler.samples_per_pixel();
            for (uint32_t si = 0; si < sample_count; ++si) {
                uint32_t global = accumulating ? tile.sample : si;
                sampler.start_pixel_sample((uint16_t)x, (uint16_t)y, global, 0);
                V2 j = sampler.get_2d();
                V2 p_film{(float)x + j.x, (float)y + j.y};
                Ray ray = camera_ray(cam, p_film);
                int32_t pid = -1;
                RadianceResult r = integrator_li(ctx, ray, sampler, &pid);
                st->primary_hit_hash += mix_hit(x, y, global, (uint32_t)pid);
                if (tile_ids && global == aux_sample) (*tile_ids)[(y - tile.y0) * tile_w + (x - tile.x0)] = pid;
                color += r.li;
                ray_count += r.rays;
            }
            color = color / (float)sample_count;
            tile_pixels[(y - tile.y0) * tile_w + (x - tile.x0)] = color;
        }
    return ray_count;
}

// Tile-queue worker model: render_manager.rs:78,135-143 + render_worker.rs:172-198 + film.rs:210-282.
// `tiles_in` is the tile list; with `replicate_samples` the manager's accumulate-mode replication (one copy of
// every tile per sample index) is applied, otherwise the caller's list (with its own `sample` fields) is used as is.
inline RenderTotals render(const Scene& scene, const Camera& cam, const Sampler& sampler, const Integrator& integ,
                           uint32_t res_x, uint32_t /*res_y*/, bool accumulate, bool replicate_samples,
                           const std::vector<FilmTile>& tiles_in, uint32_t n_threads, RenderOutputs out) {
    std::deque<FilmTile> queue(tiles_in.begin(), tiles_in.end());
    if (accumulate && replicate_samples) {  // render_manager.rs:135-143
        std::vector<FilmTile> cur(tiles_in.begin(), tiles_in.end());
        for (uint32_t s = 1; s < sampler.samples_per_pixel(); ++s)
            for (auto& t : cur) {
                t.sample += 1;
                queue.push_back(t);
            }
    }
    std::mutex queue_mutex, film_mutex;
    if (n_threads == 0) {
        unsigned hc = std::thread::hardware_concurrency();
        n_threads = hc > 1 ? hc - 1 : 1;  // num_cpus::get() - 1
    }
    std::vector<ThreadStats> stats(n_threads);
    std::vector<uint64_t> rays(n_threads, 0), samples(n_threads, 0);
    auto t0 = std::chrono::steady_clock::now();
    auto worker = [&](uint32_t tid) {
        std::vector<Spec> tile_pixels(64 * 64);  // render_worker.rs:71
        std::vector<int32_t> tile_ids(64 * 64);
        for (;;) {
            FilmTile tile;
            {
                std::lock_guard<std::mutex> g(queue_mutex);
                if (queue.empty()) return;
                tile = queue.front();
                queue.pop_front();
            }
            uint32_t w = tile.x1 - tile.x0, h = tile.y1 - tile.y0;
            if ((size_t)w * h > tile_pixels.size()) { tile_pixels.resize((size_t)w * h); tile_ids.resize((size_t)w * h); }
            rays[tid] += render_tile(scene, cam, sampler, integ, accumulate, tile, tile_pixels,
                                     out.hit_ids ? &tile_ids : nullptr, out.aux_sample, &stats[tid]);
            samples[tid] += (uint64_t)w * h * (accumulate ? 1 : sampler.samples_per_pixel());
            std::lock_guard<std::mutex> g(film_mutex);  // Film::update_tile
            for (uint32_t r = 0; r < h; ++r)
                for (uint32_t cx = 0; cx < w; ++cx) {
                    size_t fi = ((size_t)(tile.y0 + r) * res_x + tile.x0 + cx);
                    Spec c = tile_pixels[r * w + cx];
                    if (accumulate) {
                        out.film[fi * 3 + 0] += c.r; out.film[fi * 3 + 1] += c.g; out.film[fi * 3 + 2] += c.b;
                    } else {
                        out.film[fi * 3 + 0] = c.r; out.film[fi * 3 + 1] = c.g; out.film[fi * 3 + 2] = c.b;
                    }
                    if (out.hit_ids && (!accumulate || tile.sample == out.aux_sample)) out.hit_ids[fi] = tile_ids[r * w + cx];
                }
        }
    };
    std::vector<std::thread> pool;
    for (uint32_t t = 1; t < n_threads; ++t) pool.emplace_back(worker, t);
    worker(0);
    for (auto& th : pool) th.join();
    RenderTotals tot;
    tot.seconds = std::chrono::duration<double>(std::chrono::steady_clock::now() - t0).count();
    tot.threads = n_threads;
    for (uint32_t t = 0; t < n_threads; ++t) {
        tot.ray_count += rays[t];
        tot.samples += samples[t];
        tot.shadow_rays += stats[t].shadow_rays;
        tot.primary_hit_hash += stats[t].primary_hit_hash;
        tot.ts.closest_nodes += stats[t].ts.closest_nodes;
        tot.ts.closest_tris += stats[t].ts.closest_tris;
        tot.ts.any_nodes += stats[t].ts.any_nodes;
        tot.ts.any_tris += stats[t].ts.any_tris;
    }
    return tot;
}

}  // namespace yko
