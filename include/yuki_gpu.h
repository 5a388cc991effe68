/* yuki_gpu.h — C ABI of the B200 (sm_100a) backend for yuki's per-pixel rendering hot path.
 *
 * This is the drop-in boundary: everything between `render_worker::render_tile` calling
 * `Integrator::render(...)` (yuki/src/renderer/render_worker.rs:229-250, integrators/mod.rs:120-185)
 * and `Film::update_tile` (yuki/src/film.rs:210-282) is replaced by `yk_render`. A Rust host
 * binds this header unchanged with bindgen (see INTEGRATION.md); there are no C++ or torch types in
 * any signature. All matrices are row-major f32[16] (math/matrix.rs:10-18), all colours RGB f32.
 *
 * Two levels:
 *   Level 1 (device path)  yk_context_*, yk_scene_create, yk_render — what the FFI crate calls.
 *   Level 2 (host helpers) yk_host_scene_*, yk_bvh_build, yk_camera_make, yk_film_tiles, yk_xf_* —
 *                          restatements of the host-side steps either side of the path (BVH build,
 *                          camera matrices, spiral tile order) for hosts that do not bring their own.
 *
 * Error convention: every fallible entry point returns 0 (YK_OK) or a negative yk_status; the
 * message is available from yk_last_error() (thread-local). Nothing throws or aborts across the ABI
 * (the reference panics instead: integrators/mod.rs:131,141, bvh.rs:174,368).
 * There is NO CPU fallback: without a CUDA device yk_context_create fails with YK_ERR_CUDA.
 */
#ifndef YUKI_GPU_H
#define YUKI_GPU_H
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef enum {
    YK_OK = 0,
    YK_ERR_INVALID = -1,   /* bad argument / descriptor */
    YK_ERR_CUDA = -2,      /* CUDA runtime error (message holds cudaGetErrorString) */
    YK_ERR_NOMEM = -3,
    YK_ERR_BVH = -4,       /* BVH build failed (bvh.rs:368 "Split failed") or depth > 64 (bvh.rs:172-174) */
    YK_ERR_CANCELLED = -5, /* progress callback asked to stop (render_worker.rs:240-249) */
    YK_ERR_SINGULAR = -6   /* matrix.rs:170 "Can't invert, singular matrix" */
} yk_status;

/* ---- enums mirroring the reference's serde enums ------------------------------------------- */
typedef enum { YK_SPLIT_SAH = 0, YK_SPLIT_MIDDLE = 1, YK_SPLIT_EQUAL_COUNTS = 2 } yk_split_method;      /* bvh.rs:16-21 */
typedef enum {                                                                                           /* integrators/mod.rs:33-40 */
    YK_INTEGRATOR_WHITTED = 0, YK_INTEGRATOR_PATH = 1, YK_INTEGRATOR_BVH_INTERSECTIONS = 2,
    YK_INTEGRATOR_GEOMETRY_NORMALS = 3, YK_INTEGRATOR_SHADING_NORMALS = 4, YK_INTEGRATOR_SHADING_UVS = 5
} yk_integrator_kind;
typedef enum { YK_SAMPLER_UNIFORM = 0, YK_SAMPLER_STRATIFIED = 1 } yk_sampler_kind;                      /* sampling/mod.rs:15-19 */
typedef enum { YK_MAT_MATTE = 0, YK_MAT_GLASS = 1, YK_MAT_METAL = 2, YK_MAT_GLOSSY = 3 } yk_material_kind; /* materials/mod.rs */
typedef enum { YK_LIGHT_POINT = 0, YK_LIGHT_SPOT = 1, YK_LIGHT_RECT = 2, YK_LIGHT_DISTANT = 3 } yk_light_kind; /* lights/mod.rs */
typedef enum { YK_TEX_CONSTANT = 0, YK_TEX_IMAGE = 1 } yk_texture_kind;                                  /* textures/mod.rs */
typedef enum { YK_FOV_X = 0, YK_FOV_Y = 1 } yk_fov_axis;                                                 /* camera.rs:44-48 */

/* ---- small value types --------------------------------------------------------------------- */
typedef struct { float m[16]; float m_inv[16]; } yk_transform;                /* math/transform.rs:12-19 */
typedef struct { float position[3]; float target[3]; float up[3]; uint32_t fov_axis; float fov_deg; } yk_camera_params; /* camera.rs:23-29 */
typedef struct { float camera_to_world[16]; float raster_to_camera[16]; } yk_camera;                    /* camera.rs:17-21 */
typedef struct { uint32_t res_x, res_y, tile_dim, accumulate; } yk_film_settings;                       /* film.rs:13-38 */
/* Stratified: nx*ny strata (stratified.rs:17-34). Uniform: nx = pixel_samples, ny ignored (uniform.rs:13-21).
 * `seed` is explicit; the reference draws it from thread_rng (uniform.rs:37, stratified.rs:51). */
typedef struct { uint32_t kind; uint32_t nx, ny; uint32_t jitter; uint64_t seed; } yk_sampler;
/* whitted.rs:17-25, path.rs:20-32 (defaults: max_depth 3, no clamp) */
typedef struct { uint32_t kind; uint32_t max_depth; uint32_t has_clamp; float indirect_clamp; } yk_integrator;
/* film.rs:42-53 FilmTile: pixel bounds [x0,x1) x [y0,y1), accumulate-mode sample index, flat tile index */
typedef struct { uint16_t x0, y0, x1, y1; uint16_t sample; uint16_t _pad; uint32_t index; } yk_tile;

/* bvh.rs:536-588 — the 32-byte linear node. `offset` = second_child_index (interior, first child is
 * self+1) or first_shape_index (leaf). */
typedef struct {
    float p_min[3];
    float p_max[3];
    uint32_t offset;
    uint16_t shape_count;
    uint8_t split_axis;
    uint8_t is_leaf;
} yk_bvh_node;

/* ---- scene description, host level (what a loader produces) ------------------------------- */
typedef struct {
    uint32_t kind;            /* yk_texture_kind */
    float value[3];           /* constant value; f32 textures use value[0] (textures/constant.rs) */
    uint32_t width, height;   /* image (textures/image_texture.rs:64-72) */
    const float* texels;      /* width*height*3 f32, first row = top row of the file; point-sampled, no gamma */
} yk_texture_desc;

typedef struct {
    uint32_t kind;            /* yk_material_kind */
    int32_t tex[3];           /* matte: kd, sigma | glass: r, t | metal: eta, k, roughness | glossy: rs, roughness */
    float eta;                /* glass.rs:12-16 */
    uint32_t remap_roughness; /* metal.rs:15, glossy.rs:14 */
} yk_material_desc;

typedef struct {
    uint32_t kind;                 /* yk_light_kind */
    yk_transform light_to_world;   /* point_light.rs:19, spot_light.rs:23-36, rectangular_light.rs:27-43 */
    float intensity[3];            /* I (point/spot), L (rect), radiance (distant) */
    float total_width_deg, falloff_start_deg;  /* spot */
    float size[2];                 /* rect, metres */
    float direction[3];            /* distant: w (distant_light.rs:17-21) */
} yk_light_desc;

typedef struct {                   /* shapes/mesh.rs:8-18 + the per-Triangle material/area light (triangle.rs:16-21) */
    yk_transform object_to_world;
    uint32_t n_points;
    uint32_t n_indices;
    const float* points;           /* object space, n_points*3 */
    const float* normals;          /* NULL or n_points*3 */
    const float* uvs;              /* NULL or n_points*2 */
    const uint32_t* indices;       /* n_indices (triplets, CCW) */
    int32_t material;
    int32_t area_light;            /* index of a rect light in `lights`, or -1 */
} yk_mesh_desc;

typedef struct {                   /* Sphere::new, shapes/sphere.rs:23-33 */
    yk_transform object_to_world;
    float radius;
    int32_t material;
} yk_sphere_desc;

typedef struct {                   /* scene/mod.rs:41-49 + SceneLoadSettings :25-39 */
    uint32_t n_meshes, n_textures, n_materials, n_lights;
    const yk_mesh_desc* meshes;
    const yk_texture_desc* textures;
    const yk_material_desc* materials;
    const yk_light_desc* lights;
    float background[3];
    uint32_t max_shapes_in_node;   /* default 1 */
    uint32_t split_method;         /* yk_split_method, default SAH */
    uint32_t n_spheres;            /* shapes are the meshes' triangles in order, then the spheres (scene/mod.rs:497) ... */
    const yk_sphere_desc* spheres;
    uint32_t n_objects;            /* ... unless `objects` gives the declaration order: mesh index, or -1 - sphere index */
    const int32_t* objects;        /* (file order of the pbrt loader, pbrt/mod.rs:797-809); NULL = meshes then spheres */
} yk_host_scene_desc;

/* ---- scene description, device level (flattened; what the FFI crate passes) ---------------- */
typedef struct {                   /* light with its constructor already evaluated */
    uint32_t kind;
    float p[3];                    /* point/spot position; distant: w */
    float i[3];                    /* I / L / radiance */
    float cos_total_width, cos_falloff_start;
    float world_to_light[16];      /* spot: m of the world-to-light transform */
    float sample_to_world[16];     /* rect: m */
    float sample_to_world_inv[16]; /* rect: m_inv (normals use its transpose, transform.rs:144-162) */
    float area;
} yk_light;

#define YK_TRI_SWAPS_HANDEDNESS 1u
#define YK_TRI_HAS_NORMALS 2u
#define YK_TRI_HAS_UVS 4u
#define YK_TRI_IS_SPHERE 8u        /* the leaf slot is a sphere: tri_sphere[i] indexes `spheres`, the vertex slot is unused */

typedef struct {                   /* shapes/sphere.rs:15-21 with both transforms evaluated */
    float object_to_world[16];
    float world_to_object[16];
    float radius;
    uint32_t swaps_handedness;     /* Transform::swaps_handedness, math/transform.rs:84-90 */
} yk_sphere;

typedef struct {
    uint32_t n_nodes;
    const yk_bvh_node* nodes;       /* pre-order, bvh.rs:396-419 */
    uint32_t n_tris;                /* arrays below are in BVH leaf order (the reordered `shapes`, bvh.rs:95) */
    const float* tri_vertices;      /* n_tris*9 world-space positions */
    const float* tri_normals;       /* NULL or n_tris*9 world-space vertex normals */
    const float* tri_uvs;           /* NULL or n_tris*6 */
    const uint32_t* tri_orig_id;    /* index of the triangle before BVH reordering */
    const uint32_t* tri_material;
    const int32_t* tri_area_light;  /* -1 = none */
    const uint8_t* tri_flags;       /* YK_TRI_* */
    uint32_t n_textures, n_materials, n_lights;
    const yk_texture_desc* textures;
    const yk_material_desc* materials;
    const yk_light* lights;
    float background[3];
    uint32_t n_spheres;             /* shapes/sphere.rs; 0 for triangle-only scenes */
    const yk_sphere* spheres;
    const int32_t* tri_sphere;      /* NULL, or per leaf slot: index into `spheres`, -1 for triangles */
} yk_scene_desc;

/* integrators/mod.rs:76-89 */
typedef enum { YK_RAY_DIRECT = 0, YK_RAY_REFLECTION = 1, YK_RAY_REFRACTION = 2, YK_RAY_NORMAL = 3, YK_RAY_SHADOW = 4 } yk_ray_type;
typedef struct {
    float o[3], d[3];
    float t_max;
    uint32_t ray_type;             /* yk_ray_type */
} yk_integrator_ray;

/* ---- render options / statistics ------------------------------------------------------------ */
#define YK_RENDER_FILM_ON_DEVICE 1u  /* film_rgb (and opts.hit_ids) are device pointers on the context's GPU */
#define YK_RENDER_KEEP_FILM 2u       /* non-accumulating render: pixels outside `tiles` are left untouched (default) */
#define YK_RENDER_AOVS 4u            /* read opts.aovs: companion films of the same render (Path / Whitted only; not yk_multi_render) */
#define YK_RENDER_ADAPTIVE 8u        /* read opts.adaptive: stop each pixel once its mean is precise enough (Path / Whitted, averaging
                                        films only; not yk_multi_render) */
#define YK_RENDER_THIN_LENS 32u      /* read opts.lens: depth of field through a thin lens (yk_thin_lens) */
#define YK_RAY_SORT_TRACE_ONLY 16u   /* yk_render_opts.ray_sort flag: only the closest-hit kernel walks the sorted order (default: the
                                        material sort does too, so shading and shadow rays run in the same order) */

/* Companion films of a Path or Whitted render (YK_RENDER_AOVS). Each pointer is optional (NULL = not produced) and, like film_rgb,
 * res_y*res_x*3 f32 on the host, or on the device with YK_RENDER_FILM_ON_DEVICE. They follow film_rgb's semantics: the mean
 * over the samples summed in ascending sample order, or (accumulating films) one add per tile sample in tile-list order;
 * pixels outside `tiles` are left untouched. The four views are the films of the debug integrators from the same camera rays:
 * each equals, bit for bit, what yk_render returns with that integrator. */
typedef struct {
    float* bvh_intersections;  /* BVHIntersections film (bvh_heatmap.rs): (tests, hits, hits if the ray hit, else 0) */
    float* geometry_normals;   /* GeometryNormals film (geometry_normals.rs): n / 2 + 0.5, 0 on a miss */
    float* shading_normals;    /* ShadingNormals film (shading_normals.rs) */
    float* shading_uvs;        /* ShadingUVs film (shading_uvs.rs): (u, v, 0) */
    float* radiance_sq;        /* per pixel and channel: the sum of li * li over the samples, in the film's order, / spp */
} yk_aov_films;

/* Adaptive sampling (YK_RENDER_ADAPTIVE). The sampler's samples_per_pixel becomes each pixel's maximum. After n = min_samples,
 * min_samples + step, ... samples (every such n below spp), a pixel stops when, for all three channels, with its float32 sums
 * S = sum li and Q = sum li * li in ascending sample order and n as a float:
 *     m = S / n;  v = Q / n - m * m;  v = max(v, 0);  e2 = v / (n - 1);  t = rel_error * m + abs_error;  e2 <= t * t
 * (the squared standard error of the mean within the tolerance; every op un-fused IEEE float32, so a NaN never stops). A pixel
 * that stops, or reaches spp, gets film = S / n and the companion films their sums / n. */
typedef struct {
    uint32_t min_samples;      /* first convergence check after this many samples; >= 2 */
    uint32_t step;             /* then a check every `step` samples; >= 1 */
    float rel_error, abs_error;  /* >= 0, finite */
    uint32_t* sample_counts;   /* optional res_y*res_x out: samples taken per pixel; host, or device with YK_RENDER_FILM_ON_DEVICE */
} yk_adaptive;

/* Thin-lens camera (YK_RENDER_THIN_LENS): pbrt-v3's PerspectiveCamera::GenerateRay with lensradius R and focaldistance F. Camera
 * space looks down +z. With R > 0 a camera sample draws the film jitter j = get_2d() (dimensions 0-1) and then the lens sample
 * u = get_2d() (dimensions 2-3), so every later draw of the integrator moves up by 2 dimensions; every op un-fused IEEE float32,
 * in this order:
 *     p_cam = xf_point(raster_to_camera, (x + j.x, y + j.y, 0));  d = unit(p_cam)
 *     l = concentric_sample_disk(u);  lx = R * l.x;  ly = R * l.y      (sampling/mod.rs:68-87, glibc-exact sinf / cosf)
 *     ft = F / d.z;  f = d * ft                                        (the point on the plane of focus)
 *     o_cam = (lx, ly, 0);  d_cam = unit(f - o_cam)
 *     ray = (xf_point(camera_to_world, o_cam), xf_vec(camera_to_world, d_cam)), t_max = inf
 * Points at depth F are sharp; a point at depth z is spread over a disk of radius R * |1 - z / F| around its pinhole image.
 * R = 0 is the pinhole: no lens sample is drawn and the render is the plain one, bit for bit. Works with every integrator,
 * accumulating films, YK_RENDER_AOVS, YK_RENDER_ADAPTIVE and yk_multi_render. yk_debug_ray has no options and stays pinhole. */
typedef struct {
    float lens_radius;         /* >= 0 and finite */
    float focal_distance;      /* > 0 and finite (pbrt-v3's default: 1e6) */
} yk_thin_lens;

typedef int (*yk_progress_fn)(void* user, uint64_t samples_done, uint64_t samples_total); /* return !=0 to cancel */

typedef struct {
    uint32_t flags;
    uint32_t wavefront_paths;   /* paths in flight per batch; 0 = default: what ~24 GB of device memory per pipe hold (~360 B per
                                 * path with one light), at most 64 Mi, never more than a sixth of the free memory */
    int32_t* hit_ids;           /* optional res_x*res_y out: original triangle id of the primary hit of sample `aux_sample` (-1 miss) */
    uint32_t aux_sample;
    uint32_t pipes;             /* wavefront batches in flight on separate CUDA streams: 1 or 2; 0 = default (2; 1 for Whitted) */
    yk_progress_fn progress;
    void* progress_user;
    uint32_t ray_sort;          /* path tracing: order bounce rays for coherence before they are traced (a counting sort over the ray
                                   queue, csrc/wf_sort.cuh). 0 = default (by scene size), 1 = off, 2 = key = leaf slot of the shape the ray
                                   leaves + direction octant, 3 = key = Morton cell of the ray origin + direction octant. The film does
                                   not depend on it (bit-identical either way). */
    uint32_t _reserved;
    const yk_aov_films* aovs;   /* read only when flags & YK_RENDER_AOVS (callers built against the shorter struct never set it) */
    const yk_adaptive* adaptive;  /* read only when flags & YK_RENDER_ADAPTIVE */
    const yk_thin_lens* lens;     /* read only when flags & YK_RENDER_THIN_LENS */
} yk_render_opts;

typedef struct {
    uint64_t ray_count;         /* closest-hit rays: the reference's ray_scene_intersections (path.rs:87) */
    uint64_t shadow_rays;       /* any-hit rays (not counted by the reference) */
    uint64_t samples;
    uint64_t closest_nodes, closest_tris;   /* sum of N_node / N_tri over closest-hit rays */
    uint64_t any_nodes, any_tris;           /* same for shadow rays */
    uint64_t primary_hit_hash;  /* order-independent digest of every (pixel, sample, primary hit id) */
    double seconds;             /* wall time of the call */
    double device_ms;           /* CUDA-event time of the device work */
    double trace_closest_ms;    /* CUDA-event time summed over trace_closest launches */
    double trace_any_ms;        /* shadow-ray and shading kernels: only timed when YK_STAGE_TIMING=2 is set in the environment */
    double shade_ms;            /* (the extra events cost ~1.5 % of a render), else 0 */
    uint64_t kernel_launches;
    uint64_t trace_closest_launches;
} yk_stats;

typedef struct yk_context yk_context;
typedef struct yk_scene yk_scene;
typedef struct yk_host_scene yk_host_scene;

/* ---- Level 1 -------------------------------------------------------------------------------- */
const char* yk_last_error(void);
int yk_context_create(int device_id, yk_context** out);
void yk_context_destroy(yk_context*);
/* Copies the flattened scene to device SoA buffers. Host arrays may be freed on return. At most 32 lights (one bit each in
 * the shading kernels' shadow-ray mask); more -> YK_ERR_INVALID. */
int yk_scene_create(yk_context*, const yk_scene_desc*, yk_scene** out);
void yk_scene_destroy(yk_scene*);
/* Renders `tiles` (normally yk_film_tiles' spiral list, or this GPU's share of it) and writes the film.
 * Replaces Integrator::render + Film::update_tile for every tile in the list. Non-accumulating:
 * film[pixel] = mean over all samples_per_pixel (integrators/mod.rs:152-175). Accumulating
 * (film_settings.accumulate): each tile renders the single sample `tile.sample` and is ADDED to the
 * film (film.rs:260-272). `film_rgb` is res_y*res_x*3 f32, row-major (film.rs:72,95).
 * With YK_RENDER_AOVS the same render also writes opts->aovs' films. Refused (YK_ERR_INVALID, nothing launched) when
 * opts->aovs is NULL, for the debug integrators (they are the views themselves) and for Path with max_depth 0 (no primary
 * ray is traced); yk_multi_render refuses the flag. An all-NULL yk_aov_films is a plain render.
 * With YK_RENDER_ADAPTIVE each pixel takes between min_samples and spp samples (yk_adaptive); the film, companion films and
 * counts do not depend on the batch shape, pipes, ray sort or shadow mode. stats.samples is the sum of the counts, the ray and
 * traversal counters count the samples traced, the progress callback reports (done, spp * pixels) and at the end (total,
 * total), and hit_ids holds -1 for a pixel that stopped before `aux_sample`. Refused (YK_ERR_INVALID, nothing launched)
 * when opts->adaptive is NULL, min_samples < 2, step is 0, a tolerance is negative or not finite, the film accumulates or
 * the integrator is a debug one; yk_multi_render refuses the flag. min_samples >= spp is the plain render.
 * With YK_RENDER_THIN_LENS the camera rays leave through opts->lens (yk_thin_lens). Refused (YK_ERR_INVALID, nothing launched)
 * when opts->lens is NULL, the radius is negative or not finite, or the focal distance is not > 0 and finite. */
int yk_render(yk_context*, const yk_scene*, const yk_camera*, const yk_film_settings*, const yk_sampler*,
              const yk_integrator*, const yk_tile* tiles, uint32_t n_tiles, const yk_render_opts* opts,
              float* film_rgb, yk_stats* stats);
/* launch_debug_ray (app/window.rs:812-905) -> Integrator::li_debug (integrators/mod.rs:103-118): traces ONE path through
 * film pixel (film_px_x, film_px_y) with a freshly cloned sampler (pixel (0,0), sample index 0, PCG stream 0, never seeked:
 * window.rs:884) and returns the rays the integrator collects for the ray visualisation (path.rs:71-153,
 * whitted.rs:89-170), in the reference's order. Writes at most `cap` rays; *n_rays is the number collected. `li_rgb`
 * (3 floats) and `ray_count` are li_debug's RadianceResult. The debug integrators keep the trait's default: no rays, zero
 * radiance, zero ray count. The camera is the pinhole: yk_debug_ray takes no yk_render_opts, hence no yk_thin_lens. */
int yk_debug_ray(yk_context*, const yk_scene*, const yk_camera*, const yk_sampler*, const yk_integrator*,
                 uint32_t film_px_x, uint32_t film_px_y, yk_integrator_ray* rays, uint32_t cap, uint32_t* n_rays,
                 float* li_rgb, uint64_t* ray_count);
/* BoundingVolumeHierarchy::intersect (bvh.rs:160-232) for n caller rays (xyz triples; t_max NULL = infinity): closest
 * hit distance (inf on a miss), the hit shape's original id (-1 on a miss) and, when counts_out (2 per ray) is given, the
 * traversal's (intersection_test_count, intersection_count) of bvh.rs:177-179. Replaces the reference's direct
 * Scene::intersect callers outside the integrators. */
int yk_trace(yk_context*, const yk_scene*, const float* o_xyz, const float* d_xyz, const float* t_max, uint32_t n,
             float* t_out, int32_t* orig_id_out, uint32_t* counts_out);
/* VisibilityTester::unoccluded's traversal (visibility.rs:6-23 -> any_intersect, bvh.rs:235-302) for n segments
 * o -> o + d (d unnormalised, cut at t_max = 0.9999 as interaction.rs:57-58 spawns every shadow ray):
 * occluded_out[i] = 1 when anything lies in between. */
int yk_occluded(yk_context*, const yk_scene*, const float* o_xyz, const float* d_xyz, uint32_t n, uint8_t* occluded_out);
/* Ray queries with the hit's surface (Scene::intersect's Hit { t, si, shape }), on host or device-resident arrays.
 * Host arrays (opts NULL or flags 0) are staged through the context's buffers like yk_trace. With YK_QUERY_ON_DEVICE the
 * rays and every output are device memory (cudaMalloc'd or managed) of the context's GPU, 4-byte aligned: the call reads and
 * writes them in place, starts its device work after the work already queued on opts->stream and returns when its outputs
 * are written. Buffer sizes are the caller's contract. A NaN t_max is refused (YK_ERR_INVALID); on the device path this is
 * found by the kernel that reads t_max, and the outputs are then unspecified. */
#define YK_QUERY_ON_DEVICE 1u   /* rays and every output array are device memory of the context's GPU */
typedef struct {
    uint32_t flags;             /* YK_QUERY_ON_DEVICE or 0 (host arrays) */
    uint32_t _reserved;         /* must be 0 */
    void* stream;               /* ON_DEVICE: the caller's cudaStream_t (NULL = legacy default stream). The call's device
                                   work starts after the work already queued on it; the call returns when its outputs are
                                   written (blocking, like yk_render). Ignored for host arrays. */
} yk_query_opts;
typedef struct {                /* each array optional: NULL = not produced */
    float* t;                   /* n: hit distance, inf on a miss */
    int32_t* orig_id;           /* n: original shape id, -1 on a miss */
    uint32_t* counts;           /* 2n: (intersection_test_count, intersection_count), bvh.rs:177-179 */
    int32_t* material;          /* n: material index of the hit shape, -1 on a miss */
    int32_t* area_light;        /* n: SurfaceInteraction::area_light, -1 for none or a miss */
    float* p;                   /* 3n: SurfaceInteraction::p */
    float* n;                   /* 3n: geometric normal (after set_shading_geometry's faceforward) */
    float* uv;                  /* 2n */
    float* shading_n;           /* 3n: shading.n */
    float* shading_dpdu;        /* 3n: shading.dpdu (what Bsdf::new normalises into its frame's s) */
} yk_hits;                      /* on a miss p, n, uv, shading_n and shading_dpdu are 0 */
/* BoundingVolumeHierarchy::intersect (bvh.rs:160-232) for n rays (t_max NULL = infinity), writing the requested fields of
 * `out`. The geometric dpdu / dpdv and shading.dpdv are not produced. */
int yk_query_intersect(yk_context*, const yk_scene*, const float* o_xyz, const float* d_xyz, const float* t_max,
                       uint32_t n, const yk_query_opts* opts /* NULL = host arrays */, const yk_hits* out);
/* yk_occluded's semantics (segments o -> o + d, cut at 0.9999, no target light) with yk_query_intersect's options. */
int yk_query_occluded(yk_context*, const yk_scene*, const float* o_xyz, const float* d_xyz, uint32_t n,
                      const yk_query_opts* opts, uint8_t* occluded_out);
/* Sampler::{start_pixel_sample(p, index, 0), get_1d, get_2d} (sampling/mod.rs:46-57, uniform.rs:72-94, stratified.rs:90-143)
 * on the device, for n (pixel x, pixel y, sample index) triples: every triple starts a sampler the way Integrator::render
 * does (integrators/mod.rs:163) and performs the draws of `pattern` (1 = get_1d: one float, 2 = get_2d: two floats);
 * `out` receives sum(pattern) floats per triple. The component-level view of what the kernels draw per path. */
int yk_sampler_draws(yk_context*, const yk_sampler*, const uint32_t* pixel_index_xyi, uint32_t n, const uint8_t* pattern,
                     uint32_t n_pattern, float* out);
/* ---- several GPUs of one process (csrc/multi.inl) ------------------------------------------------------------------
 * The reference drives all of its workers from one RenderManager and one shared tile queue
 * (renderer/render_manager.rs:78-97,197-236; render_worker.rs:172-198). yk_multi is that for G devices: one context and
 * one host worker thread per device, the scene replicated, the tile list consumed through one shared cursor in list
 * (spiral) order, and the film assembled on the first device by direct peer (NVLink) stores from the other devices'
 * film kernels — no gather step (devices without a peer mapping are gathered with peer copies at the end). */
typedef struct yk_multi yk_multi;
typedef struct yk_multi_scene yk_multi_scene;
int yk_multi_create(const int* device_ids, int n_devices, yk_multi** out);
void yk_multi_destroy(yk_multi*);
int yk_multi_device_count(const yk_multi*);
yk_context* yk_multi_context(yk_multi*, int i);      /* the i-th device's context (owned by the group) */
int yk_multi_peer_stores(const yk_multi*, int i);    /* 1: device i stores into the first device's film directly */
/* yk_scene_create on every device: the first device validates, uploads and repacks the caller's host arrays; devices with a
 * peer mapping of it copy the repacked scene over NVLink, the others upload for themselves. */
int yk_multi_scene_create(yk_multi*, const yk_scene_desc*, yk_multi_scene** out);
void yk_multi_scene_destroy(yk_multi_scene*);
/* yk_render over all devices of the group. Same arguments and film semantics; `film_rgb` / opts->hit_ids are host
 * buffers, or (YK_RENDER_FILM_ON_DEVICE) buffers on the FIRST device. Non-accumulating renders hand out runs of tiles
 * dynamically (guided self-scheduling: remaining / 2G tiles per pop; jobs below ~256 Mi paths per device are split evenly); accumulating renders send a tile to device `tile.index mod G`, so that a pixel's per-sample adds keep the
 * tile-list order (film.rs:260-272) and the film equals the single-device one bit for bit. `stats` = sums over the
 * devices with device_ms = the busiest device's; `per_device` (NULL or G entries) = each device's own sums, device_ms
 * being its busy time. */
int yk_multi_render(yk_multi*, const yk_multi_scene*, const yk_camera*, const yk_film_settings*, const yk_sampler*,
                    const yk_integrator*, const yk_tile* tiles, uint32_t n_tiles, const yk_render_opts* opts, float* film_rgb,
                    yk_stats* stats, yk_stats* per_device);

/* Device synchronisation helpers for callers that time with their own CUDA events. */
void* yk_context_stream(yk_context*);   /* cudaStream_t the renderer launches on */

/* ---- Level 2: host helpers ------------------------------------------------------------------ */
/* BoundingVolumeHierarchy::new (bvh.rs:39-115) over n_tris world-space triangles. Outputs: `nodes`
 * (capacity 2*n_tris-1), the node count, and `order[i]` = original index of the i-th triangle in leaf
 * order. */
int yk_bvh_build(const float* tri_vertices, uint32_t n_tris, uint32_t max_shapes_in_node, uint32_t split_method,
                 yk_bvh_node* nodes, uint32_t* n_nodes, uint32_t* order);
/* Mesh::new + Triangle::new + BVH build + flattening (scene/mod.rs, mesh.rs:21-43). */
int yk_host_scene_build(const yk_host_scene_desc*, yk_host_scene** out);
void yk_host_scene_destroy(yk_host_scene*);
/* View of the flattened arrays owned by the host scene (valid until it is destroyed). */
void yk_host_scene_flat(const yk_host_scene*, yk_scene_desc* out);
/* Camera::new (camera.rs:52-102) */
int yk_camera_make(const yk_camera_params*, uint32_t res_x, uint32_t res_y, yk_camera* out);
/* film_tiles = generate_tiles + outward_spiral (film.rs:299-376, 409-475). Returns the tile count;
 * writes at most `cap` tiles. */
uint32_t yk_film_tiles(uint32_t res_x, uint32_t res_y, uint32_t tile_dim, yk_tile* out, uint32_t cap);
/* math/transforms.rs + math/transform.rs */
void yk_xf_identity(yk_transform* out);
void yk_xf_translation(const float* delta3, yk_transform* out);
void yk_xf_scale(float x, float y, float z, yk_transform* out);
void yk_xf_rotation(float theta_rad, const float* axis3, yk_transform* out);
int yk_xf_new(const float* m16, yk_transform* out);
int yk_xf_look_at(const float* pos3, const float* target3, const float* up3, yk_transform* out);
void yk_xf_mul(const yk_transform* a, const yk_transform* b, yk_transform* out);
void yk_xf_inverted(const yk_transform* a, yk_transform* out);
void yk_xf_point(const yk_transform*, const float* p3, float* out3);
void yk_xf_vec(const yk_transform*, const float* v3, float* out3);
void yk_xf_normal(const yk_transform*, const float* n3, float* out3);
/* Light constructors (`new` in lights/point_light.rs, spot_light.rs, rectangular_light.rs, distant_light.rs) */
int yk_light_make(const yk_light_desc*, yk_light* out);
/* ---- after the path: film output ---------------------------------------------------------------- */
/* app/util.rs:89-110 `write_exr`: the film as an OpenEXR file with float R, G, B channels (uncompressed scanlines). */
int yk_write_exr(const char* path, uint32_t width, uint32_t height, const float* rgb);
/* app/renderpasses/tonemap.rs:318-399: divide by the tile's sample count (accumulating films; `tile_samples` may be
 * NULL), exposure, ACES filmic fit, clamp to [0,1]. Host buffers; runs on the context's GPU. */
int yk_tonemap_filmic(yk_context*, const float* film_rgb, uint32_t res_x, uint32_t res_y, const float* tile_samples, uint32_t n_tiles,
                      uint32_t tile_dim, float exposure, float* out_rgb);
/* app/renderpasses/tonemap.rs:401-432, 447-472: blue->green->red heat map of one channel (0 R, 1 G, 2 B, 3 luminance;
 * as in the shader, channel 0 displays luminance). auto_range != 0: [min,max] come from `find_min_max` over the film and
 * are written back; otherwise the given values are used. */
int yk_heatmap(yk_context*, const float* film_rgb, uint32_t res_x, uint32_t res_y, uint32_t channel, int auto_range, float* min_val,
               float* max_val, float* out_rgb);
/* Denoising of an averaging Path / Whitted film (no counterpart in the reference): an edge-avoiding a-trous wavelet filter
 * (Dammertz et al., HPG 2010) whose colour weights are scaled by each pixel's variance (SVGF, Schied et al., HPG 2017), from
 * the render's own companion films. Per pixel with n >= 2 samples (n = sample_counts[p], or samples_per_pixel), every op
 * un-fused IEEE float32 in the order written:
 *     v = sq - c * c; if (v < 0) v = 0; v = v / (n - 1)  (per channel);   var = (v.r + v.g) + v.b
 *     guide: d = g * 2 - 1;  l2 = (d.x * d.x + d.y * d.y) + d.z * d.z;  nh = l2 > 0 ? d / sqrtf(l2) : 0
 * Iteration i = 0 .. iterations-1 (step s = 2^i) visits the 5x5 taps q = p + s * (kx - 2, ky - 2), ky outer, skipping taps
 * outside the film or with n < 2. With h = (1/16, 1/4, 3/8, 1/4, 1/16): the centre tap weighs h[2] * h[2]; another tap
 *     num = (dr * dr + dg * dg) + db * db  (d = c_i(p) - c_i(q));   den = (sigma * sigma) * (var_i(p) + var_i(q)) + eps
 *     wc = den / (den + num); wc = wc * wc;   wn = 1, or with a guide t = nh(p) . nh(q), wn = max(t, 0)^128 (7 squarings)
 *     w = ((h[ky] * h[kx]) * wn) * wc
 * and a tap counts only when w > 0 (a NaN or infinite neighbour is skipped): W += w, C += w * c_i(q), V += (w * w) * var_i(q).
 * Then c_i+1 = C / W and var_i+1 = V / (W * W). Pixels with n < 2 are copied through unchanged and are never a tap. The
 * output is c_iterations. Refused (YK_ERR_INVALID, nothing launched): a NULL context, film_rgb, radiance_sq or out_rgb, a zero
 * resolution, unknown flags, iterations outside 1 .. 10, a sigma or eps that is not > 0 and finite, no sample_counts and samples_per_pixel
 * < 2. Host arrays are staged through the device; with YK_DENOISE_ON_DEVICE every array is device memory of the context's
 * GPU and the call's work starts after the work already queued on `stream`. Returns when out_rgb is written. */
#define YK_DENOISE_ON_DEVICE 1u
typedef struct {
    uint32_t flags;                 /* YK_DENOISE_ON_DEVICE or 0 (host arrays) */
    uint32_t iterations;            /* 1 ... 10 */
    float sigma, eps;               /* > 0 and finite */
    uint32_t samples_per_pixel;     /* every pixel's n when sample_counts is NULL; >= 2 */
    uint32_t _reserved;
    const uint32_t* sample_counts;  /* optional res_y*res_x: yk_adaptive.sample_counts of the render */
    const float* normals;           /* optional guide: a geometry_normals / shading_normals companion film */
    void* stream;                   /* ON_DEVICE: the caller's cudaStream_t, as yk_query_opts.stream */
} yk_denoise_params;
/* film_rgb, radiance_sq, normals and out_rgb are res_y*res_x*3 f32; out_rgb may equal film_rgb. */
int yk_denoise(yk_context*, uint32_t res_x, uint32_t res_y, const float* film_rgb, const float* radiance_sq,
               const yk_denoise_params*, float* out_rgb);

/* pbrt-v3 scene file -> host scene description, camera parameters and film resolution: the subset and defaults of
 * scene/pbrt/{lexer,mod,param_set,cie}.rs (see csrc/host_pbrt.cpp for the directive list and the kept quirks).
 * The result's pointers stay owned by the handle. */
typedef struct yk_pbrt_scene yk_pbrt_scene;
typedef struct {
    yk_host_scene_desc scene;
    yk_camera_params camera;
    uint32_t res_x, res_y;
    float lens_radius, focal_distance;  /* Camera "perspective" lensradius (default 0) / focaldistance (default 1e6); Mitsuba: 0 / 1e6 */
} yk_pbrt_result;
int yk_pbrt_load(const char* path, uint32_t max_shapes_in_node, uint32_t split_method, yk_pbrt_scene** out);
/* Mitsuba 2.1.0 XML scene file -> the same result type (read with yk_pbrt_view, freed with yk_pbrt_destroy): the
 * elements, defaults, X-axis mirroring and error cases of scene/mitsuba/{mod,sensor,transform,emitter,material,shape}.rs
 * — sensor, twosided / diffuse / dielectric bsdfs, constant / point / spot emitters, PLY shapes (see
 * csrc/host_mitsuba.cpp). The camera target is moved into the scene bounds as mod.rs:185-197 does. */
int yk_mitsuba_load(const char* path, uint32_t max_shapes_in_node, uint32_t split_method, yk_pbrt_scene** out);
const yk_pbrt_result* yk_pbrt_view(const yk_pbrt_scene*);
void yk_pbrt_destroy(yk_pbrt_scene*);

/* PLY mesh file -> vertex / index arrays: what scene/ply.rs:19-156 takes from a file (vertex x y z [nx ny nz] [u v]
 * as float properties, faces as int/uint lists, fan-triangulated). ASCII and both binary byte orders. The arrays stay
 * owned by the handle. The fit-to-unit transform and the Scene::ply defaults are applied by the caller. */
typedef struct yk_ply yk_ply;
typedef struct {
    uint32_t n_points, n_indices;
    const float* points;      /* n_points * 3 */
    const float* normals;     /* n_points * 3 or NULL */
    const float* uvs;         /* n_points * 2 or NULL */
    const uint32_t* indices;  /* n_indices = 3 * triangles */
} yk_ply_data;
int yk_ply_load(const char* path, yk_ply** out);
void yk_ply_view(const yk_ply*, yk_ply_data* out);
void yk_ply_destroy(yk_ply*);
/* Diagnostic: number of numerators for which the kernels' division-by-invariant (csrc/yk_fastdiv.h; stands in for the
   `/` and `%` of stratified.rs:127-128,177 and the batch index arithmetic) differs from n / d. Must return 0. */
uint64_t yk_selftest_fastdiv(uint32_t d, const uint32_t* numerators, uint64_t count);

#ifdef __cplusplus
}
#endif
#endif /* YUKI_GPU_H */
