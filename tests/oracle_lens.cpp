// TEST INFRASTRUCTURE ONLY: the CPU oracle's render (yko_render) with a thin-lens camera, the reference
// tests/test_thin_lens.py compares yk_render's YK_RENDER_THIN_LENS renders with. The test compiles this file with the
// oracle's flags (oracle/Makefile) into a library of its own: it includes the oracle's C entry points, so scenes, samplers,
// integrators and tiles are the very code liboracle.so runs, and only the camera sample differs. The oracle itself stays
// the pinhole reference.
#include "yk_oracle.cpp"

namespace {

// pbrt-v3's PerspectiveCamera::GenerateRay thin lens (include/yuki_gpu.h, yk_thin_lens): the film jitter was drawn first, the
// lens sample `u` is the next get_2d.
Ray camera_ray_lens(const Camera& cam, V2 p_film, V2 u, float lens_radius, float focal_distance) {
    const V3 p_camera = xf_point(cam.raster_to_camera, v3(p_film.x, p_film.y, 0.0f));
    const V3 d = normalized(p_camera);
    const V2 l = concentric_sample_disk(u);
    const float lx = lens_radius * l.x, ly = lens_radius * l.y;
    const float ft = focal_distance / d.z;
    const V3 f = d * ft;
    const V3 o = v3(lx, ly, 0.0f);
    return xf_ray(cam.camera_to_world, Ray{o, normalized(f - o), INFINITY});
}

// yko_render.h's render_tile with the lens camera (lens_radius > 0)
uint64_t render_tile_lens(const Scene& scene, const Camera& cam, const Sampler& proto, const Integrator& integ, bool accumulating,
                          const FilmTile& tile, std::vector<Spec>& tile_pixels, std::vector<int32_t>* tile_ids, uint32_t aux_sample,
                          ThreadStats* st, float lens_radius, float focal_distance) {
    Sampler sampler = proto;
    RenderCtx ctx{scene, integ, st};
    const uint32_t tile_w = tile.x1 - tile.x0;
    uint64_t ray_count = 0;
    for (uint32_t y = tile.y0; y < tile.y1; ++y)
        for (uint32_t x = tile.x0; x < tile.x1; ++x) {
            Spec color = spec1(0.0f);
            const uint32_t sample_count = accumulating ? 1 : sampler.samples_per_pixel();
            for (uint32_t si = 0; si < sample_count; ++si) {
                const uint32_t global = accumulating ? tile.sample : si;
                sampler.start_pixel_sample((uint16_t)x, (uint16_t)y, global, 0);
                const V2 j = sampler.get_2d();
                const V2 u = sampler.get_2d();
                const Ray ray = camera_ray_lens(cam, V2{(float)x + j.x, (float)y + j.y}, u, lens_radius, focal_distance);
                int32_t pid = -1;
                const RadianceResult r = integrator_li(ctx, ray, sampler, &pid);
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

// yko_render.h's render (the tile-queue worker model) over render_tile_lens
RenderTotals render_lens(const Scene& scene, const Camera& cam, const Sampler& sampler, const Integrator& integ, uint32_t res_x,
                         bool accumulate, bool replicate_samples, const std::vector<FilmTile>& tiles_in, uint32_t n_threads,
                         RenderOutputs out, float lens_radius, float focal_distance) {
    std::deque<FilmTile> queue(tiles_in.begin(), tiles_in.end());
    if (accumulate && replicate_samples) {
        std::vector<FilmTile> cur(tiles_in.begin(), tiles_in.end());
        for (uint32_t s = 1; s < sampler.samples_per_pixel(); ++s)
            for (auto& t : cur) {
                t.sample += 1;
                queue.push_back(t);
            }
    }
    std::mutex queue_mutex, film_mutex;
    if (n_threads == 0) {
        const unsigned hc = std::thread::hardware_concurrency();
        n_threads = hc > 1 ? hc - 1 : 1;
    }
    std::vector<ThreadStats> stats(n_threads);
    std::vector<uint64_t> rays(n_threads, 0), samples(n_threads, 0);
    const auto t0 = std::chrono::steady_clock::now();
    auto worker = [&](uint32_t tid) {
        std::vector<Spec> tile_pixels(64 * 64);
        std::vector<int32_t> tile_ids(64 * 64);
        for (;;) {
            FilmTile tile;
            {
                std::lock_guard<std::mutex> g(queue_mutex);
                if (queue.empty()) return;
                tile = queue.front();
                queue.pop_front();
            }
            const uint32_t w = tile.x1 - tile.x0, h = tile.y1 - tile.y0;
            if ((size_t)w * h > tile_pixels.size()) { tile_pixels.resize((size_t)w * h); tile_ids.resize((size_t)w * h); }
            rays[tid] += render_tile_lens(scene, cam, sampler, integ, accumulate, tile, tile_pixels, out.hit_ids ? &tile_ids : nullptr,
                                          out.aux_sample, &stats[tid], lens_radius, focal_distance);
            samples[tid] += (uint64_t)w * h * (accumulate ? 1 : sampler.samples_per_pixel());
            std::lock_guard<std::mutex> g(film_mutex);
            for (uint32_t r = 0; r < h; ++r)
                for (uint32_t cx = 0; cx < w; ++cx) {
                    const size_t fi = ((size_t)(tile.y0 + r) * res_x + tile.x0 + cx);
                    const Spec c = tile_pixels[r * w + cx];
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

}  // namespace

extern "C" {

// yko_render with a thin lens of radius lens_radius > 0 focused at focal_distance; lens_radius 0 is yko_render itself.
int yko_render_lens(const yko_scene* sc, const yko_camera_params* cp, const yko_film_settings* fs, const yko_sampler_desc* sd,
                    const yko_integrator_desc* id, const yko_tile* tiles, uint32_t n_tiles, uint32_t n_threads, float* film,
                    int32_t* hit_ids, uint32_t aux_sample, yko_stats* stats, float lens_radius, float focal_distance) {
    if (lens_radius == 0.0f) return yko_render(sc, cp, fs, sd, id, tiles, n_tiles, n_threads, film, hit_ids, aux_sample, stats);
    Camera cam;
    if (!make_camera(cp, fs->res_x, fs->res_y, &cam)) return -1;
    Sampler sampler{};
    sampler.kind = (SamplerKind)sd->kind;
    sampler.nx = sd->nx;
    sampler.ny = sd->kind == SAMPLER_UNIFORM ? 1 : sd->ny;
    sampler.jitter = sd->jitter != 0;
    sampler.seed = sd->seed;
    const Integrator integ{(IntegratorKind)id->kind, id->max_depth, id->has_clamp != 0, id->indirect_clamp};
    std::vector<FilmTile> tl;
    if (tiles) {
        for (uint32_t i = 0; i < n_tiles; ++i)
            tl.push_back({tiles[i].x0, tiles[i].y0, tiles[i].x1, tiles[i].y1, tiles[i].sample, tiles[i].index});
    } else {
        tl = film_tiles(fs->res_x, fs->res_y, fs->tile_dim);
    }
    const RenderTotals t = render_lens(sc->s, cam, sampler, integ, fs->res_x, fs->accumulate != 0, tiles == nullptr, tl, n_threads,
                                       {film, hit_ids, aux_sample}, lens_radius, focal_distance);
    if (stats) {
        stats->ray_count = t.ray_count; stats->shadow_rays = t.shadow_rays; stats->samples = t.samples;
        stats->closest_nodes = t.ts.closest_nodes; stats->closest_tris = t.ts.closest_tris;
        stats->any_nodes = t.ts.any_nodes; stats->any_tris = t.ts.any_tris;
        stats->primary_hit_hash = t.primary_hit_hash;
        stats->seconds = t.seconds; stats->threads = t.threads; stats->_pad = 0;
    }
    return 0;
}

}  // extern "C"
