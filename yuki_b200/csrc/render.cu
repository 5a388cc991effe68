// B200 (sm_100a) wavefront renderer behind yk_render: replaces Integrator::render + Film::update_tile
// (yuki/src/integrators/mod.rs:120-185, film.rs:210-282) for a list of film tiles.
//
// Pipeline per batch of (pixel, sample) paths, all state in HBM as SoA (kernels in the wf_*.cuh headers of this
// translation unit):
//   jobs_expand / dim_hashes / sample_jumps -> raygen -> [ trace_closest -> classify (sort by material)
//       -> shade_{matte,glass,metal,glossy} (+ compaction of the survivors) -> trace_shadow (+ radiance fold) ]* -> film
// Nothing here is a dense contraction, so no tensor cores: the hot kernel (trace_closest) is a
// dependent-load graph walk bounded by instruction issue / L2 latency (DESIGN.md §4).
// This file holds the host side: context, scene upload (yk_scene_create), the wavefront driver (yk_render).
//
// Compiled with --fmad=false: every float op is the reference's un-fused IEEE op.
#include <cuda_runtime.h>
#include <cub/device/device_scan.cuh>

#include <algorithm>
#include <atomic>
#include <chrono>
#include <memory>
#include <mutex>
#include <cstdio>
#include <cmath>
#include <cstdlib>
#include <cstring>
#include <functional>
#include <future>
#include <string>
#include <thread>
#include <type_traits>
#include <utility>
#include <vector>

#include "wf_common.cuh"
#include "wf_raygen.cuh"
#include "wf_trace.cuh"
#include "wf_shade.cuh"
#include "wf_film.cuh"
#include "wf_query.cuh"
#include "wf_scene_pack.cuh"

#include <nvtx3/nvToolsExt.h>
#include "yk_guard.h"

// =====================================================================================================
// Host side: context, scene upload, wavefront driver.
// =====================================================================================================
#ifndef YK_MAX_PIPES
#define YK_MAX_PIPES 2
#endif
constexpr int kMaxPipes = YK_MAX_PIPES;   // batches in flight on separate streams (their kernels overlap on the SMs)
constexpr int kRing = 2;       // batches queued per pipe before the host waits for the oldest
constexpr int kTimedStages = 5;  // events per bounce: before/after closest, after classify, after shading, after shadow

// One asynchronous wavefront lane: its own stream, path state, bounce counters and timing events.
struct Pipe {
    cudaStream_t stream = nullptr;
    bool owns_stream = false;
    Wave wave{};
    std::vector<void*> wave_allocs;
    uint32_t wave_cap = 0, wave_lights = 0, wave_stack = 0;
    bool wave_sort = false;          // the ray-sort arrays are allocated
    void* sort_scan_tmp = nullptr;   // cub scan workspace for the sort's bins
    size_t sort_scan_bytes = 0;
    IterCounters* d_ctr = nullptr;   // two entries, alternating per bounce
    IterCounters* h_ctr = nullptr;   // pinned: read-back for the integrators whose bounce count is unbounded (Whitted)
    Totals* h_totals = nullptr;      // pinned
    SampleJump* d_jumps = nullptr;   // sampler seek table of the batch being queued (kMaxBatchSamples entries)
    Job* d_jobs = nullptr;           // the pixel jobs of the pipe's current pixel group
    size_t jobs_cap = 0;
    uint32_t* d_dim_hash = nullptr;  // SamplerCfg::hash_table of the pipe's current pixel group
    size_t dim_hash_cap = 0;
    size_t hash_group = (size_t)-1;
    struct Slot {
        cudaEvent_t done = nullptr;
        std::vector<cudaEvent_t> ev;  // kTimedStages per bounce
        uint32_t n_iters = 0;
        uint64_t n_paths = 0;
        bool busy = false;
    } slot[kRing];
    uint64_t n_batches = 0;
    int timing = 2;  // the context's stage_timing when the queued batches were recorded
};

struct yk_context {
    std::recursive_mutex mu;  // calls that use the context's pipes are serialised (SURVEY.md §8b: one context, many caller threads)
    int device = 0;
    int sm_count = 0;
    cudaStream_t stream = nullptr;
    cudaEvent_t ev[4] = {};
    Pipe pipe[kMaxPipes];
    yk_tile* d_tiles = nullptr;              // the tile list of the current render and the prefix sum of its tile areas
    unsigned long long* d_tile_off = nullptr;
    size_t tiles_cap = 0;
    float* d_accum = nullptr;
    float* d_film = nullptr;
    int32_t* d_hit_ids = nullptr;
    size_t film_cap = 0;
    int occ_trace_closest = 0, occ_trace_any = 0, occ_trace_rays = 0;
    int wide_per_sm = 16;  // grid cap of the grid-stride kernels, blocks per SM (development override: YK_WIDE_PER_SM)
    int n_pipes_env = 0;  // YK_PIPES override (development)
    uint64_t mem_budget = 0;  // bytes of wavefront state per pipe the default batch size may use (set at the first render)
    std::vector<void*> query_allocs;  // yk_trace / yk_occluded staging (rays in, results out), kept between calls
    uint32_t query_cap = 0;
    float *q_o = nullptr, *q_d = nullptr, *q_tm = nullptr, *q_t = nullptr;
    int32_t* q_id = nullptr;
    uint32_t* q_cnt = nullptr;
    uint8_t* q_occ = nullptr;
    std::vector<void*> query_surface_allocs;  // yk_query_intersect staging of the surface fields (host arrays), kept too
    uint32_t query_surface_cap = 0;
    int32_t *q_mat = nullptr, *q_al = nullptr;
    float *q_p = nullptr, *q_n = nullptr, *q_uv = nullptr, *q_sh_n = nullptr, *q_sh_dpdu = nullptr;
    std::vector<void*> query_flag_alloc;
    int* q_nan = nullptr;  // device-resident rays: set by k_query_pack when a t_max is NaN
    // Ray sort between bounces (wf_sort.cuh). key: 0 = off, 1 = leaf slot of the shape the ray leaves + octant, 2 = Morton cell of
    // the origin + octant, -1 = by scene size (render_impl). order: 1 = closest-hit kernel only, 2 = material sort too.
    // Environment: YK_SORT_KEY, YK_SORT_ORDER; yk_render_opts.ray_sort overrides the key per render.
    int sort_key = -1, sort_order = 2;
    // Shadow rays: 1 = one ray per lane (k_trace_shadow_rays + k_shadow_fold), 0 = one path per lane with the fold fused
    // (k_trace_shadow), -1 = by scene: per ray when several lights meet a BVH too large for the caches. Measured, one pipe
    // (profiles/r02/ab_shadow_mode.txt): 10 M-triangle terrain with 3 lights 17.2 -> 14.5 ms of shadow time (render +6 %);
    // material room (6.6 K triangles, 3 lights) 22.7 -> 25.6 ms, Cornell box (1 light) 14.6 -> 18.2 ms: on cache-resident
    // scenes the serial walk was not the limiter and the separate fold costs more than it saves. Environment: YK_SHADOW_MODE.
    int shadow_mode = -1;
    int shade_phased = -1;  // k_shade<.., PHASED>: -1 = by scene (run_batch), 0 / 1 = environment YK_SHADE_PHASED
    int stage_timing = 1;  // CUDA events per bounce: 1 = around the closest-hit kernel (the roofline figure), 2 = every stage
                           // (costs ~1.5 % of a Cornell render), 0 = none; environment variable YK_STAGE_TIMING
};

struct yk_scene {
    yk_context* ctx = nullptr;
    int device = 0;
    uint32_t material_kinds = 0;  // bit k set: some triangle's material has kind k
    DevScene dev{};
    std::vector<void*> allocs;
    // what scene_clone_impl needs to copy the repacked scene to another device: element counts and the texture table as the
    // host built it (its texel pointers are patched per device)
    size_t n_records = 0, n_leaf_entries = 0, n_materials = 0, n_spheres = 0;
    std::vector<DevTexture> host_textures;
};

namespace {

// Device buffers come from the device's stream-ordered memory pool, whose release threshold yk_context_create raises to
// "never": a freed scene / wavefront buffer stays mapped and the next allocation of that size is a pool hit. Measured on the
// 10 M-triangle scene: cudaFree of the ~1 GB upload temporaries took 3 ms ... 970 ms (unmapping), and the next
// yk_scene_create paid for mapping them again (profiles/r02: e2e_probe).
template <class T>
int dev_alloc(std::vector<void*>& bag, T** out, size_t count) {
    void* p = nullptr;
    const size_t bytes = std::max<size_t>(count, 1) * sizeof(T);
    cudaError_t e = cudaMallocAsync(&p, bytes, cudaStreamPerThread);
    if (e == cudaErrorMemoryAllocation) {
        // The pool keeps every freed block (release threshold "never"): blocks of other sizes, left by earlier scenes / batch
        // shapes / contexts of this device, can crowd out a large request. Hand the unused ones back and try once more.
        (void)cudaGetLastError();
        int dev = 0;
        cudaMemPool_t pool = nullptr;
        if (cudaGetDevice(&dev) == cudaSuccess && cudaDeviceSynchronize() == cudaSuccess && cudaDeviceGetDefaultMemPool(&pool, dev) == cudaSuccess)
            (void)cudaMemPoolTrimTo(pool, 0);
        if (getenv("YK_SCENE_TIMING")) fprintf(stderr, "dev_alloc: %zu bytes did not fit, memory pool trimmed, retrying\n", bytes);
        e = cudaMallocAsync(&p, bytes, cudaStreamPerThread);
    }
    CUDA_TRY(e);
    CUDA_TRY(cudaStreamSynchronize(cudaStreamPerThread));  // usable on every stream from here on
    bag.push_back(p);
    *out = (T*)p;
    return YK_OK;
}
template <class T>
int dev_upload(std::vector<void*>& bag, const T** out, const T* src, size_t count) {
    T* p = nullptr;
    int rc = dev_alloc(bag, &p, count);
    if (rc != YK_OK) return rc;
    if (count) CUDA_TRY(cudaMemcpy(p, src, count * sizeof(T), cudaMemcpyHostToDevice));
    *out = p;
    return YK_OK;
}
void free_bag(std::vector<void*>& bag) {
    if (bag.empty()) return;
    cudaDeviceSynchronize();  // what cudaFree did implicitly: nothing in flight may still use the buffers
    for (void* p : bag) cudaFreeAsync(p, cudaStreamPerThread);
    cudaStreamSynchronize(cudaStreamPerThread);
    bag.clear();
}

// ---- staged host -> device upload ----------------------------------------------------------------------------------
// A cudaMemcpy from pageable memory moves the 10 M-triangle scene's 1.04 GB at 6.8 GB/s (the driver stages it through one
// internal buffer on one thread). Here several host threads copy 16 MB chunks into pinned buffers and queue the DMA of each
// chunk behind it, so the page-touching memcpy of one chunk overlaps the PCIe transfer of another. The pinned buffers are kept
// in a process-wide pool (cudaMallocHost costs milliseconds).
struct CopyJob {
    void* dst;
    const void* src;
    size_t bytes;
};
class PinnedPool {
public:
    static constexpr size_t kBytes = 16u << 20;
    static constexpr size_t kKeep = 12;  // six upload threads x two buffers
    static PinnedPool& get() {
        static PinnedPool p;
        return p;
    }
    void* take() {
        {
            std::lock_guard<std::mutex> g(mu_);
            if (!free_.empty()) {
                void* p = free_.back();
                free_.pop_back();
                return p;
            }
        }
        void* p = nullptr;
        if (cudaMallocHost(&p, kBytes) != cudaSuccess) {
            (void)cudaGetLastError();
            return nullptr;
        }
        return p;
    }
    void give(void* p) {
        {
            std::lock_guard<std::mutex> g(mu_);
            if (free_.size() < kKeep) {
                free_.push_back(p);
                return;
            }
        }
        cudaFreeHost(p);  // beyond what one upload's threads use: do not keep page-locked memory for ever
    }

private:
    std::mutex mu_;
    std::vector<void*> free_;
};
int staged_upload(int device, const std::vector<CopyJob>& jobs) {
    struct Chunk {
        char* dst;
        const char* src;
        size_t bytes;
    };
    std::vector<Chunk> chunks;
    for (const CopyJob& j : jobs)
        for (size_t off = 0; off < j.bytes; off += PinnedPool::kBytes)
            chunks.push_back(Chunk{(char*)j.dst + off, (const char*)j.src + off, std::min(PinnedPool::kBytes, j.bytes - off)});
    if (chunks.empty()) return YK_OK;
    size_t total_bytes = 0;
    for (const CopyJob& j : jobs) total_bytes += j.bytes;
    if (total_bytes <= (4u << 20) && !getenv("YK_UPLOAD_STAGED")) {  // small scenes (the Cornell box is 13 KB): threads, streams and events would cost more than the copy
        for (const CopyJob& j : jobs)
            if (cudaMemcpy(j.dst, j.src, j.bytes, cudaMemcpyHostToDevice) != cudaSuccess)
                return yk_set_error(YK_ERR_CUDA, std::string("scene upload failed: ") + cudaGetErrorString(cudaGetLastError()));
        // (a pageable cudaMemcpy may return once the data is staged: wait for the DMA before kernels on other streams read it)
        if (cudaStreamSynchronize(cudaStreamLegacy) != cudaSuccess)
            return yk_set_error(YK_ERR_CUDA, std::string("scene upload failed: ") + cudaGetErrorString(cudaGetLastError()));
        return YK_OK;
    }
    const unsigned n_threads = (unsigned)std::max<size_t>(1, std::min<size_t>({(size_t)6, chunks.size(), (size_t)std::max(1u, std::thread::hardware_concurrency() / 2)}));
    std::atomic<size_t> next{0};
    std::atomic<int> failed{0};
    std::mutex err_mu;
    std::string err_text;
    auto note_error = [&](const char* what) {  // (cudaGetLastError is per thread: read it where the call failed)
        const cudaError_t e = cudaGetLastError();
        std::lock_guard<std::mutex> g(err_mu);
        if (err_text.empty()) err_text = std::string(what) + ": " + cudaGetErrorString(e);
        failed = 1;
    };
    auto worker = [&]() {
        if (cudaSetDevice(device) != cudaSuccess) { note_error("cudaSetDevice"); return; }
        cudaStream_t st = nullptr;
        cudaEvent_t ev[2] = {nullptr, nullptr};
        void* buf[2] = {PinnedPool::get().take(), PinnedPool::get().take()};
        bool ok = buf[0] && buf[1] && cudaStreamCreateWithFlags(&st, cudaStreamNonBlocking) == cudaSuccess &&
                  cudaEventCreateWithFlags(&ev[0], cudaEventDisableTiming) == cudaSuccess &&
                  cudaEventCreateWithFlags(&ev[1], cudaEventDisableTiming) == cudaSuccess;
        bool used[2] = {false, false};
        int k = 0;
        while (ok && !failed) {
            const size_t c = next.fetch_add(1);
            if (c >= chunks.size()) break;
            if (used[k] && cudaEventSynchronize(ev[k]) != cudaSuccess) { ok = false; break; }
            std::memcpy(buf[k], chunks[c].src, chunks[c].bytes);
            if (cudaMemcpyAsync(chunks[c].dst, buf[k], chunks[c].bytes, cudaMemcpyHostToDevice, st) != cudaSuccess ||
                cudaEventRecord(ev[k], st) != cudaSuccess) { ok = false; break; }
            used[k] = true;
            k ^= 1;
        }
        if (st && cudaStreamSynchronize(st) != cudaSuccess) ok = false;
        if (!ok) note_error(buf[0] && buf[1] ? "pinned staging copy" : "cudaMallocHost");
        for (int i = 0; i < 2; ++i) {
            if (ev[i]) cudaEventDestroy(ev[i]);
            if (buf[i]) PinnedPool::get().give(buf[i]);
        }
        if (st) cudaStreamDestroy(st);
    };
    std::vector<std::thread> th;
    for (unsigned i = 1; i < n_threads; ++i) th.emplace_back(worker);
    worker();
    for (auto& t : th) t.join();
    if (failed) return yk_set_error(YK_ERR_CUDA, "staged upload failed: " + err_text);
    return YK_OK;
}

// trowbridge_reitz.rs:22-30 on the host (libm logf, as the reference's f32::ln)
float host_roughness_to_alpha(float r) {
    const float x = logf(fmaxf(r, 0.001f));
    return 1.62142f + 0.819955f * x + 0.1734f * x * x + 0.0171201f * x * x * x + 0.000640711f * x * x * x * x;
}

int ensure_wave(Pipe* p, uint32_t cap, uint32_t n_lights, uint32_t stack_entries, bool sort = false) {
    // (a larger allocation serves a smaller batch: Wave::cap is only the stride of the per-light / per-kind arrays)
    if (p->wave_cap >= cap && p->wave_cap && p->wave_lights == n_lights && p->wave_stack == stack_entries && (p->wave_sort || !sort)) return YK_OK;
    free_bag(p->wave_allocs);
    p->wave_cap = 0;
    p->wave_sort = false;
    p->sort_scan_tmp = nullptr;
    Wave w{};
    w.cap = cap;
    w.n_lights = n_lights;
    w.stack_entries = stack_entries;
    std::vector<void*>& bag = p->wave_allocs;
    const size_t nl = std::max<uint32_t>(n_lights, 1);
    int rc = YK_OK;
#define WAVE_ALLOC(field, count) \
    if ((rc = dev_alloc(bag, &w.field, (size_t)(count))) != YK_OK) { free_bag(bag); return rc; }
    for (int k = 0; k < 2; ++k) {
        WAVE_ALLOC(st[k].ray_o, cap) WAVE_ALLOC(st[k].ray_d, cap) WAVE_ALLOC(st[k].beta, cap) WAVE_ALLOC(st[k].rng, cap)
    }
    WAVE_ALLOC(hit, cap) WAVE_ALLOC(bvh_counts, cap) WAVE_ALLOC(L, cap)
    // (+ one chunk of slack: the shadow kernel prefetches whole 64-path chunks of these arrays without per-line bounds tests)
    WAVE_ALLOC(sh_path, (size_t)cap + 64) WAVE_ALLOC(sh_mask, (size_t)cap + 64) WAVE_ALLOC(pend_beta, (size_t)cap + 64) WAVE_ALLOC(pend_extra, (size_t)cap + 64)
    WAVE_ALLOC(lt_o, cap * nl + 64) WAVE_ALLOC(lt_d, cap * nl + 64) WAVE_ALLOC(lt_c, cap * nl + 64)
    WAVE_ALLOC(q_active[0], cap) WAVE_ALLOC(q_active[1], cap) WAVE_ALLOC(q_mat, (size_t)4 * cap) WAVE_ALLOC(q_mat_tri, (size_t)4 * cap) WAVE_ALLOC(q_mat_slot, (size_t)4 * cap)
    WAVE_ALLOC(totals, 1)
    if (stack_entries) {
        WAVE_ALLOC(stack, (size_t)stack_entries * cap * 5)
        WAVE_ALLOC(tree_rng, cap)
    }
    if (sort) {
        WAVE_ALLOC(sort_key, cap) WAVE_ALLOC(perm, cap) WAVE_ALLOC(sort_bins, (size_t)kSortBins + 1)
        size_t bytes = 0;
        if (cub::DeviceScan::ExclusiveSum(nullptr, bytes, w.sort_bins, w.sort_bins, (int)kSortBins) != cudaSuccess) {
            free_bag(bag);
            return yk_set_error(YK_ERR_CUDA, "ensure_wave: cub scan workspace query failed");
        }
        unsigned char* tmp = nullptr;
        if ((rc = dev_alloc(bag, &tmp, bytes)) != YK_OK) { free_bag(bag); return rc; }
        p->sort_scan_tmp = tmp;
        p->sort_scan_bytes = bytes;
    }
#undef WAVE_ALLOC
    p->wave = w;
    p->wave_cap = cap;
    p->wave_lights = n_lights;
    p->wave_stack = stack_entries;
    p->wave_sort = sort;
    return YK_OK;
}

struct Timers {
    double closest = 0, any = 0, shade = 0;
    uint64_t launches = 0, closest_launches = 0;
};

int grid_for(uint32_t n, int threads, int max_blocks) {
    const uint32_t need = (n + threads - 1) / threads;
    return (int)std::max<uint32_t>(1u, std::min<uint32_t>(need, (uint32_t)max_blocks));
}

// Waits for the batch in ring slot `k` of the pipe and folds its stage timings into `tm`.
int retire_slot(Pipe* p, int k, Timers* tm, uint64_t* done_paths) {
    Pipe::Slot& sl = p->slot[k];
    if (!sl.busy) return YK_OK;
    CUDA_TRY(cudaEventSynchronize(sl.done));
    for (uint32_t i = 0; i < sl.n_iters; ++i) {
        cudaEvent_t* e = &sl.ev[(size_t)i * kTimedStages];
        float ms = 0;
        if (p->timing > 0) { cudaEventElapsedTime(&ms, e[0], e[1]); tm->closest += ms; }
        if (p->timing > 1) {
            cudaEventElapsedTime(&ms, e[2], e[3]); tm->shade += ms;
            cudaEventElapsedTime(&ms, e[3], e[4]); tm->any += ms;
        }
    }
    *done_paths += sl.n_paths;
    sl.busy = false;
    return YK_OK;
}

// One batch on one pipe: raygen, the bounce loop, and the per-batch film step, all asynchronous on the pipe's stream.
// Path tracing runs exactly max_depth bounces (every queue length stays on the device); Whitted's tree walk has no
// such bound, so it reads the next bounce's ray count back once per bounce.
int run_batch(yk_context* c, Pipe* p, const yk_scene* sc, const RenderCfg& cfg, const Batch& bt, uint32_t first_sample, bool accumulate_film,
              float* d_film, Timers* tm, uint64_t* done_paths) {
    cudaStream_t s = p->stream;
    Wave& w = p->wave;
    const int k = (int)(p->n_batches % kRing);
    int rc = retire_slot(p, k, tm, done_paths);
    if (rc != YK_OK) return rc;
    Pipe::Slot& sl = p->slot[k];
    if (!sl.done) CUDA_TRY(cudaEventCreate(&sl.done));
    sl.n_iters = 0;
    sl.n_paths = bt.n_paths;
    p->timing = c->stage_timing;
    auto stage_event = [&](uint32_t iter, int stage) -> cudaEvent_t {
        const size_t idx = (size_t)iter * kTimedStages + stage;
        while (sl.ev.size() <= idx) {
            cudaEvent_t e = nullptr;
            cudaEventCreate(&e);
            sl.ev.push_back(e);
        }
        return sl.ev[idx];
    };

    const int T = 256;
#ifdef YK_CHECKED
    CUDA_TRY(cudaMemcpyToSymbolAsync(g_check_queue_cap, &w.cap, sizeof(uint32_t), 0, cudaMemcpyHostToDevice, s));
#endif
    CUDA_TRY(cudaMemsetAsync(p->d_ctr, 0, 2 * sizeof(IterCounters), s));
    nvtxRangePushA("yk raygen");
    k_sample_jumps<<<1, kMaxBatchSamples, 0, s>>>(first_sample, bt.n_samples, p->d_jumps);
    tm->launches += 1;
    k_raygen<<<(bt.n_paths + T - 1) / T, T, 0, s>>>(w, cfg, bt, first_sample, bt.n_samples, p->d_jumps, &p->d_ctr[0]);
    nvtxRangePop();
    tm->launches += 1;
    const bool debug = cfg.integrator >= YK_INTEGRATOR_BVH_INTERSECTIONS;
    const bool sync_loop = cfg.integrator == YK_INTEGRATOR_WHITTED;
    const int trace_blocks_closest = c->sm_count * std::max(1, c->occ_trace_closest);
    const int trace_blocks_shadow = c->sm_count * std::max(1, c->occ_trace_any);
    const int wide_blocks = c->sm_count * c->wide_per_sm;
    const int classify_items = cfg.integrator == YK_INTEGRATOR_WHITTED ? 1 : YK_CLASSIFY_ITEMS;
    const int classify_blocks = grid_for(bt.n_paths, T * classify_items, c->sm_count * 8);
    const int shade_blocks = grid_for(bt.n_paths, kShadeThreads, wide_blocks);
    const int shade_blocks_plain = grid_for(bt.n_paths, kShadeThreadsPlain, wide_blocks);
    // Phase barriers + 256-thread blocks where the shading code a warp walks is long (several lights and / or material kinds);
    // plain 128-thread blocks for the Cornell-box class. YK_SHADE_PHASED=0/1 overrides.
    int n_kinds = 0;
    for (uint32_t kind = 0; kind < 4; ++kind) n_kinds += (sc->material_kinds >> kind) & 1u;
    const bool phased = c->shade_phased >= 0 ? c->shade_phased != 0 : (sc->dev.n_lights >= 2 || n_kinds >= 3);
    const int closest_blocks = grid_for(bt.n_paths, kTraceThreads, trace_blocks_closest);
    const int shadow_blocks = grid_for(bt.n_paths, kTraceThreads, trace_blocks_shadow);
    const int shadow_rays_blocks = grid_for((uint32_t)std::min<uint64_t>((uint64_t)bt.n_paths * std::max(sc->dev.n_lights, 1u), 0xffffffffu), kTraceThreads,
                                            c->sm_count * std::max(1, c->occ_trace_rays));
    const int fold_blocks = grid_for(bt.n_paths, 256, c->sm_count * 8);
    uint32_t max_iters = 1;
    if (cfg.integrator == YK_INTEGRATOR_PATH) max_iters = cfg.max_depth;
    else if (sync_loop) max_iters = 0xffffffffu;
    uint32_t* q_cur = nullptr;
    int flip = 0;
    // Ray sort (wf_sort.cuh): bounce rays are fetched through `perm`, built after the previous bounce's shading. sort_order
    // 1 = the closest-hit kernel only, 2 = the material sort too (shading and shadow rays then run in sorted order).
    const bool sorting = cfg.integrator == YK_INTEGRATOR_PATH && cfg.sort_key_mode != 0 && p->wave_sort && cfg.max_depth > 1;
    const int sort_blocks = grid_for(bt.n_paths, 256, c->sm_count * 8);
    const uint32_t* perm_trace = nullptr;
    const uint32_t* perm_classify = nullptr;
    for (uint32_t iter = 0; iter < max_iters; ++iter) {
        const int b = (int)(iter & 1);  // this bounce reads stream b and writes stream b ^ 1
        IterCounters* cur = &p->d_ctr[iter & 1];
        IterCounters* nxt = &p->d_ctr[(iter + 1) & 1];
        if (iter > 0) CUDA_TRY(cudaMemsetAsync(nxt, 0, sizeof(IterCounters), s));
        if (c->stage_timing > 0) CUDA_TRY(cudaEventRecord(stage_event(iter, 0), s));
        const bool spheres = sc->dev.spheres != nullptr || sc->dev.leaf_table != nullptr;  // the generic instantiations: sphere slots, leaf table
        nvtxRangePushA("yk closest hit");
        if (cfg.integrator == YK_INTEGRATOR_BVH_INTERSECTIONS) {
            if (spheres) k_trace_closest<true, true><<<closest_blocks, kTraceThreads, 0, s>>>(sc->dev, w, b, cur, perm_trace);
            else k_trace_closest<true, false><<<closest_blocks, kTraceThreads, 0, s>>>(sc->dev, w, b, cur, perm_trace);
        } else {
            if (spheres) k_trace_closest<false, true><<<closest_blocks, kTraceThreads, 0, s>>>(sc->dev, w, b, cur, perm_trace);
            else k_trace_closest<false, false><<<closest_blocks, kTraceThreads, 0, s>>>(sc->dev, w, b, cur, perm_trace);
        }
        nvtxRangePop();
        if (c->stage_timing > 0) CUDA_TRY(cudaEventRecord(stage_event(iter, 1), s));
        tm->launches += 1;
        tm->closest_launches += 1;
        if (cfg.debug_log) {  // yk_debug_ray: log this bounce of the single path before it is shaded
            k_debug_log<<<1, 32, 0, s>>>(sc->dev, w, cfg, bt, b, cur);
            tm->launches += 1;
        }
        uint32_t* q_next = w.q_active[flip];
        if (debug) {
            k_debug_shade<<<(bt.n_paths + T - 1) / T, T, 0, s>>>(sc->dev, w, cfg, bt.n_paths);
            // primary-hit digest / id image for the debug integrators too
            k_classify<YK_CLASSIFY_ITEMS, false><<<classify_blocks, T, 0, s>>>(sc->dev, w, cfg, bt, q_cur, b, cur, nxt, 2, q_next, nullptr);
            tm->launches += 2;
            for (int st = 2; st < kTimedStages; ++st) if (c->stage_timing > 1) CUDA_TRY(cudaEventRecord(stage_event(iter, st), s));
            sl.n_iters = iter + 1;
            break;
        }
        nvtxRangePushA("yk classify (misses, material queues)");
        if (cfg.integrator == YK_INTEGRATOR_WHITTED) k_classify<1, true><<<classify_blocks, T, 0, s>>>(sc->dev, w, cfg, bt, q_cur, b, cur, nxt, iter == 0 ? 1 : 0, q_next, nullptr);
        else k_classify<YK_CLASSIFY_ITEMS, false><<<classify_blocks, T, 0, s>>>(sc->dev, w, cfg, bt, q_cur, b, cur, nxt, iter == 0 ? 1 : 0, q_next, perm_classify);
        nvtxRangePop();
        if (c->stage_timing > 1) CUDA_TRY(cudaEventRecord(stage_event(iter, 2), s));
        tm->launches += 1;
        nvtxRangePushA("yk shade (per material kind)");
        const bool is_path = cfg.integrator == YK_INTEGRATOR_PATH;
        for (uint32_t kind = 0; kind < 4; ++kind) {
            if (!(sc->material_kinds & (1u << kind))) continue;  // no triangle of the scene has this material kind
            uint32_t* q = w.q_mat + (size_t)kind * w.cap;
            uint32_t* qt = w.q_mat_tri + (size_t)kind * w.cap;
            uint32_t* qs = w.q_mat_slot + (size_t)kind * w.cap;
#define YK_LAUNCH_SHADE(K)                                                                                                                        \
    do {                                                                                                                                          \
        if (phased) {                                                                                                                             \
            if (is_path) k_shade<K, true, true><<<shade_blocks, kShadeThreads, 0, s>>>(sc->dev, w, cfg, bt, q, qt, qs, b, cur, nxt, q_next);       \
            else k_shade<K, false, true><<<shade_blocks, kShadeThreads, 0, s>>>(sc->dev, w, cfg, bt, q, qt, qs, b, cur, nxt, q_next);              \
        } else {                                                                                                                                  \
            if (is_path) k_shade<K, true, false><<<shade_blocks_plain, kShadeThreadsPlain, 0, s>>>(sc->dev, w, cfg, bt, q, qt, qs, b, cur, nxt, q_next); \
            else k_shade<K, false, false><<<shade_blocks_plain, kShadeThreadsPlain, 0, s>>>(sc->dev, w, cfg, bt, q, qt, qs, b, cur, nxt, q_next);  \
        }                                                                                                                                         \
    } while (0)
            switch (kind) {
                case YK_MAT_MATTE: YK_LAUNCH_SHADE(YK_MAT_MATTE); break;
                case YK_MAT_GLASS: YK_LAUNCH_SHADE(YK_MAT_GLASS); break;
                case YK_MAT_METAL: YK_LAUNCH_SHADE(YK_MAT_METAL); break;
                default: YK_LAUNCH_SHADE(YK_MAT_GLOSSY); break;
            }
#undef YK_LAUNCH_SHADE
            tm->launches += 1;
        }
        nvtxRangePop();
        if (c->stage_timing > 1) CUDA_TRY(cudaEventRecord(stage_event(iter, 3), s));
        nvtxRangePushA("yk shadow rays + fold");
        if (cfg.shadow_per_ray) {  // one shadow ray per lane, then the fold (wf_trace.cuh)
            if (spheres) k_trace_shadow_rays<true><<<shadow_rays_blocks, kTraceThreads, 0, s>>>(sc->dev, w, sc->dev.n_lights, cur);
            else k_trace_shadow_rays<false><<<shadow_rays_blocks, kTraceThreads, 0, s>>>(sc->dev, w, sc->dev.n_lights, cur);
            k_shadow_fold<<<fold_blocks, 256, 0, s>>>(w, cfg, cur);
            tm->launches += 1;
        } else {  // one path per lane, its lights in order, fold fused
            if (spheres) k_trace_shadow<true><<<shadow_blocks, kTraceThreads, 0, s>>>(sc->dev, w, cfg, cur);
            else k_trace_shadow<false><<<shadow_blocks, kTraceThreads, 0, s>>>(sc->dev, w, cfg, cur);
        }
        nvtxRangePop();
        if (c->stage_timing > 1) CUDA_TRY(cudaEventRecord(stage_event(iter, 4), s));
        tm->launches += 1;
        if (cfg.integrator == YK_INTEGRATOR_WHITTED) {
            k_tree_return<<<shade_blocks_plain, kShadeThreadsPlain, 0, s>>>(w, b, cur, nxt, q_next);
            tm->launches += 1;
        }
        if (sorting && iter + 1 < max_iters) {  // order the next bounce's rays
            nvtxRangePushA("yk ray sort");
            CUDA_TRY(cudaMemsetAsync(w.sort_bins, 0, ((size_t)kSortBins + 1) * sizeof(uint32_t), s));
            k_sort_hist<<<sort_blocks, 256, 0, s>>>(w, nxt);
            CUDA_TRY(cub::DeviceScan::ExclusiveSum(p->sort_scan_tmp, p->sort_scan_bytes, w.sort_bins, w.sort_bins, (int)kSortBins, s));
            k_sort_scatter<<<sort_blocks, 256, 0, s>>>(w, nxt);
            nvtxRangePop();
            tm->launches += 3;
            perm_trace = w.perm;
            perm_classify = cfg.sort_order >= 2 ? w.perm : nullptr;
        }
        sl.n_iters = iter + 1;
        q_cur = q_next;
        flip ^= 1;
        if (sync_loop) {
            CUDA_TRY(cudaMemcpyAsync(p->h_ctr, nxt, sizeof(IterCounters), cudaMemcpyDeviceToHost, s));
            CUDA_TRY(cudaStreamSynchronize(s));
            if (p->h_ctr->n_active == 0) break;
            // one iteration per node of the deepest path's recursion tree: at most 2^max_depth - 1 (whitted.rs:132-170)
            if ((uint64_t)iter + 1 > ((uint64_t)1 << std::min(cfg.max_depth, 40u))) return yk_set_error(YK_ERR_INVALID, "yk_render: bounce loop did not terminate");
        }
    }
    nvtxRangePushA("yk film");
    if (accumulate_film) {
        k_film_add<<<(bt.n_paths + T - 1) / T, T, 0, s>>>(w, bt, d_film, cfg.res_x);
    } else {
        k_film_accumulate<<<(bt.n_jobs + T - 1) / T, T, 0, s>>>(w, bt, c->d_accum, cfg.res_x);
    }
    nvtxRangePop();
    tm->launches += 1;
    CUDA_TRY(cudaEventRecord(sl.done, s));
    CUDA_TRY(cudaGetLastError());
    sl.busy = true;
    p->n_batches += 1;
    return YK_OK;
}

}  // namespace

// Makes the context's device current on the calling thread (post.cu: the display passes may be called from any thread).
int yk_context_activate(yk_context* c) {
    CUDA_TRY(cudaSetDevice(c->device));
    return YK_OK;
}

extern "C" {

int yk_context_create(int device_id, yk_context** out) {
    return yk_guard("yk_context_create", [&]() -> int {
    if (!out) return yk_set_error(YK_ERR_INVALID, "yk_context_create: null output");
    int n_dev = 0;
    cudaError_t e = cudaGetDeviceCount(&n_dev);
    if (e != cudaSuccess || n_dev == 0)
        return yk_set_error(YK_ERR_CUDA, std::string("yk_context_create: no CUDA device (") + cudaGetErrorString(e) +
                                             "); this backend has no CPU fallback");
    if (device_id < 0 || device_id >= n_dev) return yk_set_error(YK_ERR_INVALID, "yk_context_create: device id out of range");
    CUDA_TRY(cudaSetDevice(device_id));
    auto* c = new yk_context();
    c->device = device_id;
    cudaDeviceProp prop;
    CUDA_TRY(cudaGetDeviceProperties(&prop, device_id));
    c->sm_count = prop.multiProcessorCount;
    {   // keep freed device buffers in the pool (dev_alloc)
        cudaMemPool_t pool = nullptr;
        unsigned long long keep = ~0ull;
        if (cudaDeviceGetDefaultMemPool(&pool, device_id) == cudaSuccess) cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &keep);
        (void)cudaGetLastError();
    }
    CUDA_TRY(cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking));
    for (auto& ev : c->ev) CUDA_TRY(cudaEventCreateWithFlags(&ev, cudaEventDisableTiming));
    CUDA_TRY(cudaEventDestroy(c->ev[2]));
    CUDA_TRY(cudaEventDestroy(c->ev[3]));
    CUDA_TRY(cudaEventCreate(&c->ev[2]));  // timing pair around the whole render
    CUDA_TRY(cudaEventCreate(&c->ev[3]));
    if (const char* np = getenv("YK_PIPES")) c->n_pipes_env = std::max(1, std::min(kMaxPipes, atoi(np)));
    if (const char* st = getenv("YK_STAGE_TIMING")) c->stage_timing = std::max(0, std::min(2, atoi(st)));
    if (const char* sp = getenv("YK_SHADE_PHASED")) c->shade_phased = atoi(sp) ? 1 : 0;
    if (const char* sm = getenv("YK_SHADOW_MODE")) c->shadow_mode = std::max(-1, std::min(1, atoi(sm)));
    if (const char* sk = getenv("YK_SORT_KEY")) c->sort_key = std::max(-1, std::min(2, atoi(sk)));
    if (const char* so = getenv("YK_SORT_ORDER")) c->sort_order = std::max(1, std::min(2, atoi(so)));
    for (int i = 0; i < kMaxPipes; ++i) {
        Pipe& p = c->pipe[i];
        if (i == 0) p.stream = c->stream;
        else {
            CUDA_TRY(cudaStreamCreateWithFlags(&p.stream, cudaStreamNonBlocking));
            p.owns_stream = true;
        }
        CUDA_TRY(cudaMalloc((void**)&p.d_ctr, 2 * sizeof(IterCounters)));
        CUDA_TRY(cudaMalloc((void**)&p.d_jumps, kMaxBatchSamples * sizeof(SampleJump)));
        CUDA_TRY(cudaMallocHost((void**)&p.h_ctr, sizeof(IterCounters)));
        CUDA_TRY(cudaMallocHost((void**)&p.h_totals, sizeof(Totals)));
    }
    CUDA_TRY(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&c->occ_trace_closest, k_trace_closest<false, false>, kTraceThreads, 0));
    CUDA_TRY(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&c->occ_trace_any, k_trace_shadow<false>, kTraceThreads, 0));
    CUDA_TRY(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&c->occ_trace_rays, k_trace_shadow_rays<false>, kTraceThreads, 0));
    // development overrides (A/B of co-resident kernels of two pipes): blocks per SM of the persistent / grid-stride kernels
    if (const char* e = getenv("YK_TRACE_PER_SM")) c->occ_trace_closest = c->occ_trace_any = c->occ_trace_rays = std::max(1, atoi(e));
    if (const char* e = getenv("YK_WIDE_PER_SM")) c->wide_per_sm = std::max(1, atoi(e));
    *out = c;
    return YK_OK;
    });
}

void yk_context_destroy(yk_context* c) {
    if (!c) return;
    cudaSetDevice(c->device);
    cudaDeviceSynchronize();
    for (Pipe& p : c->pipe) {
        free_bag(p.wave_allocs);
        cudaFree(p.d_ctr);
        cudaFree(p.d_dim_hash);
        cudaFree(p.d_jobs);
        cudaFree(p.d_jumps);
        cudaFreeHost(p.h_ctr);
        cudaFreeHost(p.h_totals);
        for (auto& sl : p.slot) {
            if (sl.done) cudaEventDestroy(sl.done);
            for (cudaEvent_t e : sl.ev) cudaEventDestroy(e);
        }
        if (p.owns_stream) cudaStreamDestroy(p.stream);
    }
    free_bag(c->query_allocs);
    free_bag(c->query_surface_allocs);
    free_bag(c->query_flag_alloc);
    cudaFree(c->d_tiles);
    cudaFree(c->d_tile_off);
    cudaFree(c->d_accum);
    cudaFree(c->d_film);
    cudaFree(c->d_hit_ids);
    for (auto& ev : c->ev) cudaEventDestroy(ev);
    cudaStreamDestroy(c->stream);
    delete c;
}

void* yk_context_stream(yk_context* c) { return c ? (void*)c->stream : nullptr; }

}  // extern "C"

// What the host-side validation of a flattened scene yields (and what the device repack needs from it). yk_multi_scene_create
// validates once and uploads to every device with the result (`pre`).
struct SceneCheck {
    const char* error = nullptr;
    uint32_t n_interior = 0, kinds = 0;
    bool small_leaves = true;
};
static int scene_create_impl(yk_context* c, const yk_scene_desc* d, const SceneCheck* pre, SceneCheck* check_out, yk_scene** out) {
    if (!c || !d || !out) return yk_set_error(YK_ERR_INVALID, "yk_scene_create: null argument");
    if (!d->n_nodes || !d->nodes || !d->n_tris || !d->tri_vertices || !d->tri_orig_id || !d->tri_material || !d->tri_area_light ||
        !d->tri_flags)
        return yk_set_error(YK_ERR_INVALID, "yk_scene_create: missing node / triangle arrays");
    if (d->n_lights > (uint32_t)kMaxLights) return yk_set_error(YK_ERR_INVALID, "yk_scene_create: more than 32 lights");
    if ((d->n_materials && !d->materials) || (d->n_lights && !d->lights) || (d->n_textures && !d->textures) || (d->n_spheres && !d->spheres))
        return yk_set_error(YK_ERR_INVALID, "yk_scene_create: null material / light / texture / sphere table with a non-zero count");
    if (d->n_materials > 0xffffffu) return yk_set_error(YK_ERR_INVALID, "yk_scene_create: too many materials");
    CUDA_TRY(cudaSetDevice(c->device));
    const bool timing = getenv("YK_SCENE_TIMING") != nullptr;  // development: phase times to stderr
    const auto t_start = std::chrono::steady_clock::now();
    auto lap = [&](const char* what) {
        if (timing) fprintf(stderr, "yk_scene_create: %-28s at %8.2f ms\n", what,
                            1e3 * std::chrono::duration<double>(std::chrono::steady_clock::now() - t_start).count());
    };
    auto sc = std::make_unique<yk_scene>();
    sc->ctx = c;
    sc->device = c->device;
    int rc;
    // The reference-layout arrays go to the device as they are and are repacked there (k_scene_*): no host-side copy of
    // the scene is built. Meanwhile host threads validate the same arrays (indices, ranges, flags).
    using Check = SceneCheck;
    const unsigned n_workers = std::max(1u, std::min(16u, std::thread::hardware_concurrency()));
    auto validate = [d, n_workers](unsigned wi) -> Check {
        Check ck;
        auto fail = [&ck](const char* m) { if (!ck.error) ck.error = m; };
        const uint64_t n0 = (uint64_t)d->n_nodes * wi / n_workers, n1 = (uint64_t)d->n_nodes * (wi + 1) / n_workers;
        for (uint64_t i = n0; i < n1; ++i) {
            const yk_bvh_node& n = d->nodes[i];
            if (!n.is_leaf) {
                ck.n_interior += 1;
                if (n.split_axis > 2) fail("yk_scene_create: split axis out of range");
                // children follow their parent (pre-order, bvh.rs:396-419): the walk cannot cycle
                if (n.offset >= d->n_nodes || i + 1 >= d->n_nodes || n.offset <= i + 1) fail("yk_scene_create: child index out of range");
            } else {
                if ((uint64_t)n.offset + n.shape_count > d->n_tris) fail("yk_scene_create: leaf range out of range");
                if (n.shape_count < 1 || n.shape_count > 16) ck.small_leaves = false;
            }
        }
        const uint64_t t0 = (uint64_t)d->n_tris * wi / n_workers, t1 = (uint64_t)d->n_tris * (wi + 1) / n_workers;
        for (uint64_t i = t0; i < t1; ++i) {
            const uint32_t m = d->tri_material[i];
            if (m >= d->n_materials) { fail("yk_scene_create: material index out of range"); continue; }
            if (d->materials[m].kind <= YK_MAT_GLOSSY) ck.kinds |= 1u << d->materials[m].kind;
            const int32_t al = d->tri_area_light[i];
            if (al >= (int32_t)d->n_lights || al < -1) fail("yk_scene_create: area light out of range");
            else if (al >= 0 && d->lights[al].kind != YK_LIGHT_RECT) fail("yk_scene_create: area light must be rectangular");
            const uint8_t f = d->tri_flags[i];
            if ((f & YK_TRI_HAS_NORMALS) && !d->tri_normals) fail("yk_scene_create: normals flagged but absent");
            if ((f & YK_TRI_HAS_UVS) && !d->tri_uvs) fail("yk_scene_create: uvs flagged but absent");
            if ((f & YK_TRI_IS_SPHERE) && (!d->tri_sphere || !d->spheres || d->tri_sphere[i] < 0 || (uint32_t)d->tri_sphere[i] >= d->n_spheres))
                fail("yk_scene_create: sphere slot without a valid sphere index");
        }
        return ck;
    };
    for (uint32_t i = 0; i < d->n_materials; ++i)
        if (d->materials[i].kind > YK_MAT_GLOSSY) return yk_set_error(YK_ERR_INVALID, "yk_scene_create: unknown material kind");
    for (uint32_t i = 0; i < d->n_lights; ++i)
        if (d->lights[i].kind > YK_LIGHT_DISTANT) return yk_set_error(YK_ERR_INVALID, "yk_scene_create: unknown light kind");
    std::vector<std::future<Check>> checks;
    if (!pre)
        for (unsigned wi = 0; wi < n_workers; ++wi) checks.push_back(std::async(std::launch::async, validate, wi));
    auto join_checks = [&](Check* total) {
        if (pre) *total = *pre;
        for (auto& f : checks) {
            const Check ck = f.get();
            if (ck.error && !total->error) total->error = ck.error;
            total->n_interior += ck.n_interior;
            total->kinds |= ck.kinds;
            total->small_leaves = total->small_leaves && ck.small_leaves;
        }
        checks.clear();
    };
    struct Cleanup {  // on an error return: wait for the validators, release what was uploaded
        std::function<void()> fn;
        bool armed = true;
        ~Cleanup() { if (armed) fn(); }
    };
    std::vector<void*> temps;
    Cleanup cleanup{[&] {
        Check ignore;
        join_checks(&ignore);
        cudaDeviceSynchronize();
        free_bag(temps);
        free_bag(sc->allocs);
    }};
    const yk_bvh_node* r_nodes = nullptr;
    const float* r_verts = nullptr;
    const uint32_t *r_orig = nullptr, *r_mat = nullptr;
    const int32_t *r_alight = nullptr, *r_sphere = nullptr;
    const uint8_t *r_flags = nullptr, *r_kinds = nullptr;
    std::vector<uint8_t> kinds(std::max(d->n_materials, 1u), 0);
    for (uint32_t i = 0; i < d->n_materials; ++i) kinds[i] = (uint8_t)d->materials[i].kind;
    lap("validators started");
    {   // device buffers first, then all arrays through the staged, multi-threaded upload
        std::vector<CopyJob> jobs;
        auto up = [&](std::vector<void*>& bag, auto** out, const auto* src, size_t count) -> int {
            using T = std::remove_const_t<std::remove_pointer_t<std::remove_pointer_t<decltype(out)>>>;
            T* p = nullptr;
            const int r = dev_alloc(bag, &p, count);
            if (r != YK_OK) return r;
            *out = p;
            if (count) jobs.push_back(CopyJob{(void*)p, (const void*)src, count * sizeof(T)});
            return YK_OK;
        };
        if ((rc = up(temps, &r_nodes, d->nodes, d->n_nodes)) != YK_OK) return rc;
        if ((rc = up(temps, &r_verts, d->tri_vertices, (size_t)d->n_tris * 9)) != YK_OK) return rc;
        if ((rc = up(temps, &r_orig, d->tri_orig_id, d->n_tris)) != YK_OK) return rc;
        if ((rc = up(temps, &r_mat, d->tri_material, d->n_tris)) != YK_OK) return rc;
        if ((rc = up(temps, &r_alight, d->tri_area_light, d->n_tris)) != YK_OK) return rc;
        if ((rc = up(temps, &r_flags, d->tri_flags, d->n_tris)) != YK_OK) return rc;
        if (d->tri_sphere && (rc = up(temps, &r_sphere, d->tri_sphere, d->n_tris)) != YK_OK) return rc;
        if ((rc = up(temps, &r_kinds, kinds.data(), kinds.size())) != YK_OK) return rc;
        if (d->tri_normals && (rc = up(sc->allocs, &sc->dev.normals, d->tri_normals, (size_t)d->n_tris * 9)) != YK_OK) return rc;
        if (d->tri_uvs && (rc = up(sc->allocs, &sc->dev.uvs, d->tri_uvs, (size_t)d->n_tris * 6)) != YK_OK) return rc;
        if ((rc = staged_upload(c->device, jobs)) != YK_OK) return rc;
    }
    lap("arrays uploaded");
    Check total;
    join_checks(&total);
    lap("validation joined");
    if (total.error) return yk_set_error(YK_ERR_INVALID, total.error);
    if (check_out) *check_out = total;
    if (total.n_interior > kRefIndexMask) return yk_set_error(YK_ERR_INVALID, "yk_scene_create: more than 2^29 interior nodes");
    sc->material_kinds = total.kinds;
    const uint32_t n_interior = total.n_interior, n_leaves = d->n_nodes - n_interior;
    const bool packed_leaves = total.small_leaves && d->n_tris <= (1u << kLeafFirstBits);

    // Nodes: one 64-byte record per interior node with the boxes of both children (DevScene::nodes2). Interior records are
    // numbered in the reference's pre-order (an exclusive scan of the interior flags), so a first child's record follows
    // its parent's; leaves are numbered the same way for the leaf table.
    {
        cudaStream_t st = c->stream;
        const uint32_t n = d->n_nodes;
        uint32_t *d_flag = nullptr, *d_rec = nullptr;
        float4* d_rec_out = nullptr;
        uint2* d_leaf = nullptr;
        if ((rc = dev_alloc(temps, &d_flag, n)) != YK_OK || (rc = dev_alloc(temps, &d_rec, n)) != YK_OK) return rc;
        if ((rc = dev_alloc(sc->allocs, &d_rec_out, (size_t)std::max(n_interior, 1u) * 4)) != YK_OK) return rc;
        if (!packed_leaves && (rc = dev_alloc(sc->allocs, &d_leaf, n_leaves)) != YK_OK) return rc;
        k_scene_interior_flags<<<(n + 255) / 256, 256, 0, st>>>(r_nodes, n, d_flag);
        size_t scan_bytes = 0;
        CUDA_TRY(cub::DeviceScan::ExclusiveSum(nullptr, scan_bytes, d_flag, d_rec, (int)n, st));
        unsigned char* d_scan = nullptr;
        if ((rc = dev_alloc(temps, &d_scan, scan_bytes)) != YK_OK) return rc;
        CUDA_TRY(cub::DeviceScan::ExclusiveSum(d_scan, scan_bytes, d_flag, d_rec, (int)n, st));
        k_scene_records<<<(n + 255) / 256, 256, 0, st>>>(r_nodes, d_rec, n, packed_leaves ? 1 : 0, d_leaf, d_rec_out);
        sc->dev.nodes2 = d_rec_out;
        sc->dev.leaf_table = d_leaf;
        const yk_bvh_node& root = d->nodes[0];
        if (!root.is_leaf) sc->dev.root_ref = kRefInterior | ((uint32_t)root.split_axis << 29);  // record 0
        else if (packed_leaves) sc->dev.root_ref = ((uint32_t)(root.shape_count - 1) << kLeafFirstBits) | root.offset;
        else {
            sc->dev.root_ref = 0;  // leaf 0 of the table; nobody's child, so it is written here
            const uint2 entry = make_uint2(root.offset, root.shape_count);
            CUDA_TRY(cudaMemcpyAsync(d_leaf, &entry, sizeof entry, cudaMemcpyHostToDevice, st));
        }
        std::memcpy(sc->dev.root_min, root.p_min, 12);
        std::memcpy(sc->dev.root_max, root.p_max, 12);
        // Triangles: three 16-byte words, vertices pre-gathered in leaf order and transposed (x0 x1 x2 | y0 y1 y2 | z0 z1 z2);
        // the w lanes carry the per-triangle ids.
        float4* d_tris = nullptr;
        if ((rc = dev_alloc(sc->allocs, &d_tris, (size_t)d->n_tris * 3)) != YK_OK) return rc;
        k_scene_tris<<<(d->n_tris + 255) / 256, 256, 0, st>>>(r_verts, r_orig, r_mat, r_alight, r_flags, r_sphere, r_kinds, d->n_tris, d_tris);
        sc->dev.tris = d_tris;
        CUDA_TRY(cudaGetLastError());
        CUDA_TRY(cudaStreamSynchronize(st));
        lap("repacked on the device");
        free_bag(temps);
        lap("temporaries freed");
    }

    std::vector<DevTexture> tex(d->n_textures);
    for (uint32_t i = 0; i < d->n_textures; ++i) {
        const yk_texture_desc& t = d->textures[i];
        DevTexture dt{};
        dt.kind = t.kind;
        dt.width = t.width;
        dt.height = t.height;
        std::memcpy(dt.value, t.value, 12);
        if (t.kind == YK_TEX_IMAGE) {
            if (!t.texels || !t.width || !t.height) return yk_set_error(YK_ERR_INVALID, "yk_scene_create: empty image texture");
            if ((rc = dev_upload(sc->allocs, &dt.texels, t.texels, (size_t)t.width * t.height * 3)) != YK_OK) return rc;
        } else if (t.kind != YK_TEX_CONSTANT) {
            return yk_set_error(YK_ERR_INVALID, "yk_scene_create: unknown texture kind");
        }
        tex[i] = dt;
    }
    std::vector<DevMaterial> mats(d->n_materials);
    for (uint32_t i = 0; i < d->n_materials; ++i) {
        const yk_material_desc& m = d->materials[i];
        if (m.kind > YK_MAT_GLOSSY) return yk_set_error(YK_ERR_INVALID, "yk_scene_create: unknown material kind");
        const int n_tex = m.kind == YK_MAT_METAL ? 3 : 2;
        for (int k = 0; k < n_tex; ++k)
            if (m.tex[k] < 0 || (uint32_t)m.tex[k] >= d->n_textures)
                return yk_set_error(YK_ERR_INVALID, "yk_scene_create: texture index out of range");
        DevMaterial dm{};
        dm.kind = m.kind;
        std::memcpy(dm.tex, m.tex, 12);
        dm.eta = m.eta;
        dm.remap = m.remap_roughness;
        dm.const_alpha = -1.0f;
        if (m.kind == YK_MAT_METAL || m.kind == YK_MAT_GLOSSY) {
            const yk_texture_desc& rt = d->textures[m.tex[m.kind == YK_MAT_METAL ? 2 : 1]];
            if (rt.kind == YK_TEX_CONSTANT) {  // metal.rs:41-45 / glossy.rs:39-49 + trowbridge_reitz.rs:16-20
                float r = rt.value[0];
                if (m.remap_roughness) r = host_roughness_to_alpha(r);
                dm.const_alpha = fmaxf(m.kind == YK_MAT_GLOSSY ? r * r : r, 0.001f);
            }
        }
        mats[i] = dm;
    }
    if ((rc = dev_upload(sc->allocs, &sc->dev.textures, tex.data(), tex.size())) != YK_OK) return rc;
    if ((rc = dev_upload(sc->allocs, &sc->dev.materials, mats.data(), mats.size())) != YK_OK) return rc;
    if ((rc = dev_upload(sc->allocs, &sc->dev.lights, d->lights, d->n_lights)) != YK_OK) return rc;
    if (d->n_spheres && (rc = dev_upload(sc->allocs, &sc->dev.spheres, d->spheres, d->n_spheres)) != YK_OK) return rc;
    sc->dev.n_lights = d->n_lights;
    sc->dev.n_tris = d->n_tris;
    sc->dev.n_nodes = d->n_nodes;
    std::memcpy(sc->dev.background, d->background, 12);
    sc->n_records = std::max(n_interior, 1u);
    sc->n_leaf_entries = packed_leaves ? 0 : n_leaves;
    sc->n_materials = mats.size();
    sc->n_spheres = d->n_spheres;
    sc->host_textures = tex;
    cleanup.armed = false;
    lap("done");
    *out = sc.release();
    return YK_OK;
}

// The repacked scene of another device, copied over NVLink (yk_multi_scene_create): device 0 takes the host arrays, validates
// and repacks them once; every other device of the group allocates the same buffers and pulls them with peer copies instead of
// staging, uploading and repacking the same gigabyte again (8 devices, 10 M triangles: 8 x 1 GB through the host's memory
// and 8 PCIe links -> one upload + 7 NVLink copies).
static int scene_clone_impl(yk_context* c, const yk_scene* src, yk_scene** out) {
    if (!c || !src || !out) return yk_set_error(YK_ERR_INVALID, "scene clone: null argument");
    const auto t_start = std::chrono::steady_clock::now();
    CUDA_TRY(cudaSetDevice(c->device));
    auto sc = std::make_unique<yk_scene>();
    sc->ctx = c;
    sc->device = c->device;
    sc->material_kinds = src->material_kinds;
    sc->dev = src->dev;  // scalars, root box, background; the pointers are replaced below
    sc->n_records = src->n_records; sc->n_leaf_entries = src->n_leaf_entries; sc->n_materials = src->n_materials; sc->n_spheres = src->n_spheres;
    sc->host_textures = src->host_textures;
    struct Cleanup {
        yk_scene* s; bool armed = true;
        ~Cleanup() { if (armed) free_bag(s->allocs); }
    } cleanup{sc.get()};
    cudaStream_t st = c->stream;
    int rc = YK_OK;
    auto pull = [&](auto** field, size_t count) -> int {
        using T = std::remove_const_t<std::remove_pointer_t<std::remove_pointer_t<decltype(field)>>>;
        const T* from = *field;
        if (!from || !count) { *field = nullptr; return YK_OK; }
        T* p = nullptr;
        const int r = dev_alloc(sc->allocs, &p, count);
        if (r != YK_OK) return r;
        CUDA_TRY(cudaMemcpyPeerAsync(p, c->device, from, src->device, count * sizeof(T), st));
        *field = p;
        return YK_OK;
    };
    const size_t n_tris = src->dev.n_tris;
    if ((rc = pull(&sc->dev.nodes2, sc->n_records * 4)) != YK_OK) return rc;
    if ((rc = pull(&sc->dev.leaf_table, sc->n_leaf_entries)) != YK_OK) return rc;
    if ((rc = pull(&sc->dev.tris, n_tris * 3)) != YK_OK) return rc;
    if ((rc = pull(&sc->dev.normals, n_tris * 9)) != YK_OK) return rc;
    if ((rc = pull(&sc->dev.uvs, n_tris * 6)) != YK_OK) return rc;
    if ((rc = pull(&sc->dev.materials, sc->n_materials)) != YK_OK) return rc;
    if ((rc = pull(&sc->dev.lights, (size_t)src->dev.n_lights)) != YK_OK) return rc;
    if ((rc = pull(&sc->dev.spheres, sc->n_spheres)) != YK_OK) return rc;
    std::vector<DevTexture> tex = sc->host_textures;
    for (DevTexture& t : tex)
        if (t.kind == YK_TEX_IMAGE && (rc = pull(&t.texels, (size_t)t.width * t.height * 3)) != YK_OK) return rc;
    sc->dev.textures = nullptr;
    if ((rc = dev_upload(sc->allocs, &sc->dev.textures, tex.data(), tex.size())) != YK_OK) return rc;
    CUDA_TRY(cudaStreamSynchronize(st));
    if (getenv("YK_SCENE_TIMING"))
        fprintf(stderr, "scene clone to device %d: %.2f ms\n", c->device,
                1e3 * std::chrono::duration<double>(std::chrono::steady_clock::now() - t_start).count());
    cleanup.armed = false;
    *out = sc.release();
    return YK_OK;
}

extern "C" {

int yk_scene_create(yk_context* c, const yk_scene_desc* d, yk_scene** out) {
    return yk_guard("yk_scene_create", [&]() -> int { return scene_create_impl(c, d, nullptr, nullptr, out); });
}

void yk_scene_destroy(yk_scene* s) {
    if (!s) return;
    cudaSetDevice(s->device);
    free_bag(s->allocs);
    delete s;
}

}  // extern "C"

// Internal yk_render_opts.flags bit (yk_multi_render's workers): the caller initialised the hit-id image, do not refill it.
constexpr uint32_t kRenderAuxInitialised = 0x100u;

// yk_render, and yk_debug_ray's single path (`debug_log` = device ray list, `debug_px` = the film pixel of its camera sample).
static int render_impl(yk_context* c, const yk_scene* sc, const yk_camera* cam, const yk_film_settings* fs, const yk_sampler* sm,
                       const yk_integrator* in, const yk_tile* tiles, uint32_t n_tiles, const yk_render_opts* opts, float* film_rgb,
                       yk_stats* stats, DebugLog* debug_log, const float* debug_px) {
    const auto wall0 = std::chrono::steady_clock::now();
    if (!c || !sc || !cam || !fs || !sm || !in || !film_rgb) return yk_set_error(YK_ERR_INVALID, "yk_render: null argument");
    if (sc->ctx != c) return yk_set_error(YK_ERR_INVALID, "yk_render: scene belongs to another context");
    if (!fs->res_x || !fs->res_y || fs->res_x > 0xffffu || fs->res_y > 0xffffu)
        return yk_set_error(YK_ERR_INVALID, "yk_render: film resolution must fit u16 (integrators/mod.rs:140-141)");
    if (in->kind > YK_INTEGRATOR_SHADING_UVS) return yk_set_error(YK_ERR_INVALID, "yk_render: unknown integrator");
    if (sm->kind > YK_SAMPLER_STRATIFIED) return yk_set_error(YK_ERR_INVALID, "yk_render: unknown sampler");
    const uint32_t spp = sm->kind == YK_SAMPLER_UNIFORM ? sm->nx : sm->nx * sm->ny;
    if (spp == 0 || spp > 0x10000u) return yk_set_error(YK_ERR_INVALID, "yk_render: samples per pixel must be in 1..65536");
    if (in->max_depth > 255) return yk_set_error(YK_ERR_INVALID, "yk_render: max_depth above 255");
    if (in->kind == YK_INTEGRATOR_WHITTED && in->max_depth > 24)
        return yk_set_error(YK_ERR_INVALID, "yk_render: whitted max_depth above 24 is not supported");
    if (n_tiles && !tiles) return yk_set_error(YK_ERR_INVALID, "yk_render: null tile list");
    std::lock_guard<std::recursive_mutex> guard(c->mu);
    CUDA_TRY(cudaSetDevice(c->device));
    (void)cudaGetLastError();  // do not inherit a stale error from an unrelated earlier call
    cudaStream_t s = c->stream;
    const uint32_t flags = opts ? opts->flags : 0u;
    const bool on_device = (flags & YK_RENDER_FILM_ON_DEVICE) != 0;
    const bool accumulate = fs->accumulate != 0;

    // Pixel jobs: tile order, row-major inside a tile. Only the tile list and the prefix sum of the tile areas go to the
    // device; each pixel group's jobs are expanded there (k_jobs_expand).
    std::vector<unsigned long long> tile_off((size_t)n_tiles + 1, 0ull);
    for (uint32_t t = 0; t < n_tiles; ++t) {
        const yk_tile& tl = tiles[t];
        if (tl.x0 >= tl.x1 || tl.y0 >= tl.y1 || tl.x1 > fs->res_x || tl.y1 > fs->res_y)
            return yk_set_error(YK_ERR_INVALID, "yk_render: tile outside the film (film.rs:224-231)");
        tile_off[t + 1] = tile_off[t] + (unsigned long long)(tl.x1 - tl.x0) * (tl.y1 - tl.y0);
    }
    const unsigned long long n_jobs_total = tile_off[n_tiles], area = n_jobs_total;
    const size_t n_pixels = (size_t)fs->res_x * fs->res_y;
    const uint32_t samples_per_job = accumulate ? 1u : spp;

    RenderCfg cfg{};
    cfg.sampler = SamplerCfg{};
    cfg.sampler.kind = sm->kind;
    cfg.sampler.nx = sm->nx;
    cfg.sampler.ny = sm->kind == YK_SAMPLER_UNIFORM ? 1u : sm->ny;
    cfg.sampler.jitter = sm->jitter;
    cfg.sampler.seed = sm->seed;
    cfg.sampler.div_nx = FastDiv::make(cfg.sampler.nx);
    cfg.sampler.div_ny = FastDiv::make(cfg.sampler.ny);
    cfg.sampler.div_n = FastDiv::make(cfg.sampler.nx * cfg.sampler.ny);
    cfg.integrator = in->kind;
    cfg.max_depth = in->max_depth;
    cfg.has_clamp = in->has_clamp;
    cfg.clamp = in->indirect_clamp;
    std::memcpy(cfg.c2w, cam->camera_to_world, 64);
    std::memcpy(cfg.r2c, cam->raster_to_camera, 64);
    cfg.res_x = fs->res_x;
    cfg.res_y = fs->res_y;
    cfg.aux_sample = opts ? opts->aux_sample : 0u;
    cfg.debug_log = debug_log;
    if (debug_log) { cfg.debug_px[0] = debug_px[0]; cfg.debug_px[1] = debug_px[1]; }
    cfg.shadow_per_ray = (sc->dev.n_lights > 0 && (c->shadow_mode == 1 || (c->shadow_mode < 0 && sc->dev.n_lights >= 2 && sc->dev.n_tris >= (1u << 18)))) ? 1u : 0u;
    {   // ray sort between bounces (path tracing only; Whitted's tree walk re-queues rays in DFS order)
        int key = c->sort_key;
        cfg.sort_order = (uint32_t)c->sort_order;
        if (opts && (opts->ray_sort & 0xfu)) key = (int)(opts->ray_sort & 0xfu) - 1;
        if (opts && (opts->ray_sort & YK_RAY_SORT_TRACE_ONLY)) cfg.sort_order = 1;
        if (key < 0) key = 0;  // default
        if (in->kind != YK_INTEGRATOR_PATH || in->max_depth < 2 || debug_log) key = 0;
        cfg.sort_key_mode = (uint32_t)std::min(key, 2);
        uint32_t bits = 0;
        while (bits < 32 && ((uint64_t)1 << bits) < sc->dev.n_tris) ++bits;  // leaf slots fit `bits` bits
        cfg.sort_slot_shift = bits > kSortKeyBits - 3 ? bits - (kSortKeyBits - 3) : 0u;
        for (int a = 0; a < 3; ++a) {
            const float ext = sc->dev.root_max[a] - sc->dev.root_min[a];
            cfg.sort_cell_scale[a] = ext > 0.0f ? 32.0f / ext : 0.0f;
        }
    }

    // Device film / accumulators.
    if (c->film_cap < n_pixels) {
        cudaFree(c->d_accum); cudaFree(c->d_film); cudaFree(c->d_hit_ids);
        c->d_accum = nullptr; c->d_film = nullptr; c->d_hit_ids = nullptr;
        c->film_cap = 0;
        CUDA_TRY(cudaMalloc((void**)&c->d_accum, n_pixels * 3 * sizeof(float)));
        CUDA_TRY(cudaMalloc((void**)&c->d_film, n_pixels * 3 * sizeof(float)));
        CUDA_TRY(cudaMalloc((void**)&c->d_hit_ids, n_pixels * sizeof(int32_t)));
        c->film_cap = n_pixels;
    }
    float* d_film = on_device ? film_rgb : c->d_film;
    const bool full_cover = !accumulate && area == n_pixels;
    if (!on_device) {
        if (full_cover) CUDA_TRY(cudaMemsetAsync(d_film, 0, n_pixels * 3 * sizeof(float), s));
        else CUDA_TRY(cudaMemcpyAsync(d_film, film_rgb, n_pixels * 3 * sizeof(float), cudaMemcpyHostToDevice, s));
    }
    int32_t* d_ids = nullptr;
    if (opts && opts->hit_ids) {
        d_ids = on_device ? opts->hit_ids : c->d_hit_ids;
        if (!(flags & kRenderAuxInitialised)) k_fill_i32<<<(unsigned)((n_pixels + 255) / 256), 256, 0, s>>>(d_ids, n_pixels, -1);
    }
    cfg.hit_ids = d_ids;

    yk_stats st{};
    Timers tm;
    Totals totals{};
    CUDA_TRY(cudaEventRecord(c->ev[2], s));
    if (n_jobs_total) {
        if (c->tiles_cap < n_tiles) {
            cudaFree(c->d_tiles);
            cudaFree(c->d_tile_off);
            c->d_tiles = nullptr;
            c->d_tile_off = nullptr;
            c->tiles_cap = 0;
            CUDA_TRY(cudaMalloc((void**)&c->d_tiles, (size_t)n_tiles * sizeof(yk_tile)));
            CUDA_TRY(cudaMalloc((void**)&c->d_tile_off, ((size_t)n_tiles + 1) * sizeof(unsigned long long)));
            c->tiles_cap = n_tiles;
        }
        CUDA_TRY(cudaMemcpyAsync(c->d_tiles, tiles, (size_t)n_tiles * sizeof(yk_tile), cudaMemcpyHostToDevice, s));
        CUDA_TRY(cudaMemcpyAsync(c->d_tile_off, tile_off.data(), tile_off.size() * sizeof(unsigned long long), cudaMemcpyHostToDevice, s));
        // Wavefront capacity: paths in flight per batch. Fewer, longer launches amortise the persistent kernels' tails and the
        // launch gaps, and HBM is 180 GB: measured 4 Mi -> 8 Mi -> 16 Mi paths = +8 %, +12 % on the Cornell bench (round 1), and
        // 16 Mi -> 32 Mi -> 64 Mi = +0.7 %, +0.8 % there with two pipes (+2.5 %, +3.9 % with one) and +4.1 %, +6.4 % on the
        // 10 M-triangle scene (profiles/r02/capsweep_large_batches.txt). Default: as many as ~24 GB of wavefront state per pipe
        // hold (~360 B per path with one light), at most 64 Mi, and never more than a sixth of the free device memory per pipe.
        const uint32_t stack_entries = in->kind == YK_INTEGRATOR_WHITTED ? std::max(in->max_depth, 1u) : 0u;
        uint32_t cap = opts ? opts->wavefront_paths : 0u;
        if (!cap) {
            const uint64_t bytes_per_path = 320ull + 40ull * std::max(sc->dev.n_lights, 1u) + (80ull * stack_entries + (stack_entries ? 8ull : 0ull));
            if (!c->mem_budget) {  // asked once per context: cudaMemGetInfo can take milliseconds
                size_t free_b = 0, total_b = 0;
                c->mem_budget = 24ull << 30;
                if (cudaMemGetInfo(&free_b, &total_b) == cudaSuccess) c->mem_budget = std::min<uint64_t>(c->mem_budget, (uint64_t)free_b / 6);
            }
            cap = (uint32_t)std::min<uint64_t>(1u << 26, std::max<uint64_t>(1u << 20, c->mem_budget / bytes_per_path));
        }
        const uint64_t total_paths = (uint64_t)n_jobs_total * samples_per_job;
        if (cap > total_paths) cap = (uint32_t)total_paths;
        cap = std::max(cap, 32u);
        // Samples of one pixel per batch: enough to amortise per-batch fixed costs, few enough that many pixels
        // (>= 64 Ki when available) share a batch.
        uint32_t m = std::min(samples_per_job, kMaxBatchSamples);
        if (const char* e = getenv("YK_MAX_BATCH_SAMPLES")) m = std::min<uint32_t>(m, (uint32_t)std::max(1, atoi(e)));  // development: A/B of the batch shape
        while (m > 1 && (uint64_t)m * std::min<uint64_t>(n_jobs_total, 65536) > cap) m >>= 1;
        uint32_t jobs_per_batch = std::max(1u, cap / m);
        // Pipes: pixel groups alternate between the streams, so one group's latency-bound shading overlaps the other's
        // issue-bound traversal. A pixel's samples stay on one pipe, in order (the film sum is order-dependent).
        // The accumulating film adds with atomics across tiles, so it keeps to one stream.
        // Default: two pipes. Measured on one box with the current kernels (profiles/r01/README.md): Cornell +5 %, config-4
        // room +6 %, 1 M-triangle heightfield +10 %, 10 M-triangle terrain +12 %. Whitted's bounce loop waits for the host
        // once per bounce, which would serialise the pipes, so it keeps one. YK_PIPES / opts->pipes override (bench.py
        // times its device-resident leg on one pipe so that the event-bracketed kernel times stay exclusive).
        int n_pipes = c->n_pipes_env > 0 ? c->n_pipes_env : (in->kind == YK_INTEGRATOR_WHITTED ? 1 : 2);
        if (opts && opts->pipes) n_pipes = (int)opts->pipes;
        n_pipes = std::max(1, std::min(kMaxPipes, n_pipes));
        if (accumulate) n_pipes = 1;
        // Pixel groups of equal size, their number a multiple of the pipe count: a ragged tail (a last group of a fraction of a
        // batch, or an odd group that runs on one pipe with nothing beside it) cost a 2-GPU yk_multi_render whose runs are
        // not multiples of a group 8 ms per run. Fewer pixel groups than pipes: split the jobs evenly if that leaves decent
        // batches, else use fewer pipes.
        if (!accumulate) {
            for (;;) {
                unsigned long long n_g = (n_jobs_total + jobs_per_batch - 1) / jobs_per_batch;
                n_g = (n_g + n_pipes - 1) / n_pipes * n_pipes;
                const unsigned long long per = (n_jobs_total + n_g - 1) / n_g;
                if (n_pipes == 1 || per * m >= (1u << 20) || n_g > (unsigned long long)n_pipes) {
                    jobs_per_batch = (uint32_t)std::max<unsigned long long>(1, per);
                    break;
                }
                n_pipes -= 1;
            }
        }
        const uint32_t wave_cap = (uint32_t)std::min<uint64_t>(cap, (uint64_t)jobs_per_batch * m);
        int rc = YK_OK;
        CUDA_TRY(cudaEventRecord(c->ev[0], s));
        for (int pi = 0; pi < n_pipes; ++pi) {
            Pipe& p = c->pipe[pi];
            if ((rc = ensure_wave(&p, wave_cap, sc->dev.n_lights, stack_entries, cfg.sort_key_mode != 0)) != YK_OK) return rc;
            if (pi > 0) CUDA_TRY(cudaStreamWaitEvent(p.stream, c->ev[0], 0));
            CUDA_TRY(cudaMemsetAsync(p.wave.totals, 0, sizeof(Totals), p.stream));
            p.hash_group = (size_t)-1;
        }
        // Pixel groups: consecutive runs of at most jobs_per_batch jobs. The accumulating film adds every batch into the
        // film in stream order, so a group never spans a change of `tile.sample`: within one sample index the reference's
        // tiles are disjoint, each pixel appears once per batch and the per-pixel sum runs in tile-list order exactly
        // like the reference's `*fc += c` (film.rs:260-272).
        struct Group { unsigned long long first; uint32_t count, t_lo, t_hi; };  // jobs [first, first + count) lie in tiles [t_lo, t_hi)
        std::vector<Group> groups;
        {
            uint32_t seg_t0 = 0;
            auto flush = [&](uint32_t seg_t1) {  // the jobs of tiles [seg_t0, seg_t1)
                uint32_t t = seg_t0;
                for (unsigned long long j = tile_off[seg_t0]; j < tile_off[seg_t1]; j += jobs_per_batch) {
                    const unsigned long long end = std::min<unsigned long long>(j + jobs_per_batch, tile_off[seg_t1]);
                    while (tile_off[t + 1] <= j) ++t;
                    uint32_t t_hi = t + 1;
                    while (tile_off[t_hi] < end) ++t_hi;
                    groups.push_back(Group{j, (uint32_t)(end - j), t, t_hi});
                }
                seg_t0 = seg_t1;
            };
            if (accumulate)
                for (uint32_t t = 1; t < n_tiles; ++t)
                    if (tiles[t].sample != tiles[t - 1].sample) flush(t);
            flush(n_tiles);
        }
        const size_t n_groups = groups.size();
        uint64_t done = 0;
        bool cancelled = false;
        for (size_t g0 = 0; g0 < n_groups && !cancelled; g0 += n_pipes) {
            for (uint32_t s0 = 0; s0 < samples_per_job && !cancelled; s0 += m) {
                for (int pi = 0; pi < n_pipes && g0 + pi < n_groups && !cancelled; ++pi) {
                    Pipe& p = c->pipe[pi];
                    const size_t group = g0 + pi;
                    const uint32_t nj = groups[group].count;
                    if (p.hash_group != group) {  // a new pixel group on this pipe: its jobs, and a zeroed accumulator
                        if (p.jobs_cap < nj) {
                            CUDA_TRY(cudaStreamSynchronize(p.stream));
                            cudaFree(p.d_jobs);
                            p.d_jobs = nullptr;
                            p.jobs_cap = 0;
                            CUDA_TRY(cudaMalloc((void**)&p.d_jobs, (size_t)std::max(nj, jobs_per_batch) * sizeof(Job)));
                            p.jobs_cap = std::max(nj, jobs_per_batch);
                        }
                        k_jobs_expand<<<(nj + 255) / 256, 256, 0, p.stream>>>(c->d_tiles, c->d_tile_off, groups[group].t_lo, groups[group].t_hi,
                                                                               groups[group].first, nj, accumulate ? 1u : 0u, p.d_jobs);
                        tm.launches += 1;
                        if (!accumulate) {
                            k_zero_jobs<<<(nj + 255) / 256, 256, 0, p.stream>>>(p.d_jobs, nj, c->d_accum, fs->res_x);
                            tm.launches += 1;
                        }
                        if (debug_log) {
                            k_debug_job<<<1, 1, 0, p.stream>>>(p.d_jobs);
                            tm.launches += 1;
                        }
                    }
                    RenderCfg gcfg = cfg;
                    if (sm->kind == YK_SAMPLER_STRATIFIED) {
                        // tabulate the (pixel, dimension) hashes of this pixel group once for all of its samples
                        uint64_t dims = 2;
                        if (in->kind == YK_INTEGRATOR_PATH) dims = 2 + (uint64_t)in->max_depth * (2ull * sc->dev.n_lights + 3);
                        else if (in->kind == YK_INTEGRATOR_WHITTED)
                            dims = 2 + 2ull * sc->dev.n_lights * ((1ull << std::min(in->max_depth, 8u)) - 1);
                        dims = std::min<uint64_t>(dims, std::min<uint64_t>(4096, (256ull << 20) / (4ull * nj)));  // the rest is hashed on the fly
                        if (p.hash_group != group) {
                            const size_t need = (size_t)dims * nj;
                            if (p.dim_hash_cap < need) {
                                CUDA_TRY(cudaStreamSynchronize(p.stream));
                                cudaFree(p.d_dim_hash);
                                p.d_dim_hash = nullptr;
                                p.dim_hash_cap = 0;
                                CUDA_TRY(cudaMalloc((void**)&p.d_dim_hash, need * sizeof(uint32_t)));
                                p.dim_hash_cap = need;
                            }
                            k_dim_hashes<<<dim3((nj + 255) / 256, (unsigned)std::min<uint64_t>(dims, 64)), 256, 0, p.stream>>>(
                                p.d_jobs, nj, (uint32_t)dims, sm->seed, p.d_dim_hash);
                            tm.launches += 1;
                        }
                        gcfg.sampler.hash_table = p.d_dim_hash;
                        gcfg.sampler.n_hash_dims = (uint32_t)dims;
                        gcfg.sampler.hash_stride = nj;
                    }
                    p.hash_group = group;
                    Batch bt;
                    bt.jobs = p.d_jobs;
                    bt.n_jobs = nj;
                    bt.div_jobs = FastDiv::make(nj);
                    bt.sample_off = s0;
                    bt.n_samples = std::min(m, samples_per_job - s0);
                    bt.n_paths = nj * bt.n_samples;
                    // the batch's first sample index: s0, or the sample of the group's tiles (accumulating films: one per group)
                    const uint32_t first_sample = accumulate ? (uint32_t)tiles[groups[group].t_lo].sample : s0;
                    rc = run_batch(c, &p, sc, gcfg, bt, first_sample, accumulate, d_film, &tm, &done);
                    if (rc != YK_OK) {  // nothing may stay in flight or marked busy behind an error return
                        cudaDeviceSynchronize();
                        for (Pipe& q : c->pipe)
                            for (auto& slot : q.slot) slot.busy = false;
                        return rc;
                    }
                    if (!accumulate && s0 + m >= samples_per_job) {
                        // the group's last samples are queued: `color /= sample_count` + Film::update_tile for its pixels
                        k_film_store<<<(nj + 255) / 256, 256, 0, p.stream>>>(p.d_jobs, nj, c->d_accum, d_film, fs->res_x, (float)spp);
                        tm.launches += 1;
                    }
                    if (opts && opts->progress && opts->progress(opts->progress_user, done, total_paths)) cancelled = true;
                }
            }
        }
        for (int pi = 0; pi < n_pipes; ++pi) {
            Pipe& p = c->pipe[pi];
            CUDA_TRY(cudaMemcpyAsync(p.h_totals, p.wave.totals, sizeof(Totals), cudaMemcpyDeviceToHost, p.stream));
            for (int k = 0; k < kRing; ++k)
                if ((rc = retire_slot(&p, k, &tm, &done)) != YK_OK) return rc;
            CUDA_TRY(cudaStreamSynchronize(p.stream));
            const Totals& t = *p.h_totals;
            totals.closest_nodes += t.closest_nodes; totals.closest_tris += t.closest_tris;
            totals.any_nodes += t.any_nodes; totals.any_tris += t.any_tris;
            totals.hit_hash += t.hit_hash; totals.shadow_rays += t.shadow_rays; totals.closest_rays += t.closest_rays;
        }
        if (cancelled) return yk_set_error(YK_ERR_CANCELLED, "yk_render: cancelled by the progress callback");
        if (opts && opts->progress) opts->progress(opts->progress_user, done, total_paths);
        st.samples = total_paths;
    }
    CUDA_TRY(cudaEventRecord(c->ev[3], s));
    if (!on_device) {
        CUDA_TRY(cudaMemcpyAsync(film_rgb, d_film, n_pixels * 3 * sizeof(float), cudaMemcpyDeviceToHost, s));
        if (opts && opts->hit_ids)
            CUDA_TRY(cudaMemcpyAsync(opts->hit_ids, d_ids, n_pixels * sizeof(int32_t), cudaMemcpyDeviceToHost, s));
    }
    CUDA_TRY(cudaStreamSynchronize(s));
    CUDA_TRY(cudaGetLastError());
    if (stats) {
        st.closest_nodes = totals.closest_nodes;
        st.closest_tris = totals.closest_tris;
        st.any_nodes = totals.any_nodes;
        st.any_tris = totals.any_tris;
        st.primary_hit_hash = totals.hit_hash;
        st.shadow_rays = totals.shadow_rays;
        st.ray_count = totals.closest_rays;
        float ms = 0;
        cudaEventElapsedTime(&ms, c->ev[2], c->ev[3]);
        st.device_ms = ms;
        st.trace_closest_ms = tm.closest;
        st.trace_any_ms = tm.any;
        st.shade_ms = tm.shade;
        st.kernel_launches = tm.launches;
        st.trace_closest_launches = tm.closest_launches;
        st.seconds = std::chrono::duration<double>(std::chrono::steady_clock::now() - wall0).count();
        *stats = st;
    }
    return YK_OK;
}

extern "C" {

int yk_render(yk_context* c, const yk_scene* sc, const yk_camera* cam, const yk_film_settings* fs, const yk_sampler* sm,
              const yk_integrator* in, const yk_tile* tiles, uint32_t n_tiles, const yk_render_opts* opts, float* film_rgb,
              yk_stats* stats) {
    return yk_guard("yk_render", [&]() -> int {
    return render_impl(c, sc, cam, fs, sm, in, tiles, n_tiles, opts, film_rgb, stats, nullptr, nullptr);
    });
}

// launch_debug_ray (app/window.rs:812-905): one path, its rays collected by k_debug_log between the wavefront stages. The
// path is "sample 0 of pixel (0, 0)" of a 1x1 accumulating film — the state of a freshly cloned sampler — except that it
// draws from PCG stream 0 (k_debug_job) and that its camera sample lands on the requested film pixel (k_raygen).
int yk_debug_ray(yk_context* c, const yk_scene* sc, const yk_camera* cam, const yk_sampler* sm, const yk_integrator* in,
                 uint32_t film_px_x, uint32_t film_px_y, yk_integrator_ray* rays, uint32_t cap, uint32_t* n_rays, float* li_rgb,
                 uint64_t* ray_count) {
    return yk_guard("yk_debug_ray", [&]() -> int {
    if (!c || !sc || !cam || !sm || !in || !n_rays || (cap && !rays)) return yk_set_error(YK_ERR_INVALID, "yk_debug_ray: null argument");
    if (film_px_x > 0xffffu || film_px_y > 0xffffu) return yk_set_error(YK_ERR_INVALID, "yk_debug_ray: film pixel must fit u16");
    *n_rays = 0;
    if (li_rgb) li_rgb[0] = li_rgb[1] = li_rgb[2] = 0.0f;
    if (ray_count) *ray_count = 0;
    if (in->kind > YK_INTEGRATOR_SHADING_UVS) return yk_set_error(YK_ERR_INVALID, "yk_debug_ray: unknown integrator");
    if (in->kind != YK_INTEGRATOR_WHITTED && in->kind != YK_INTEGRATOR_PATH) return YK_OK;  // default li_debug, integrators/mod.rs:103-118
    if (sc->ctx != c) return yk_set_error(YK_ERR_INVALID, "yk_debug_ray: scene belongs to another context");
    CUDA_TRY(cudaSetDevice(c->device));
    // min_debug_ray_length (path.rs:58-62): Bounds3::maximum_extent (math/bounds.rs:147-156) of the BVH's bounds
    const float* lo = sc->dev.root_min;
    const float* hi = sc->dev.root_max;
    const float dx = hi[0] - lo[0], dy = hi[1] - lo[1], dz = hi[2] - lo[2];
    const int axis = (dx > dy && dx > dz) ? 0 : (dy > dz ? 1 : 2);
    DebugLog head{};
    head.cap = cap;
    head.min_len = (hi[axis] - lo[axis]) / 10.0f;
    DebugLog* d_log = nullptr;
    yk_integrator_ray* d_rays = nullptr;
    CUDA_TRY(cudaMalloc((void**)&d_log, sizeof(DebugLog)));
    if (cudaMalloc((void**)&d_rays, std::max<size_t>(cap, 1) * sizeof(yk_integrator_ray)) != cudaSuccess) {
        cudaFree(d_log);
        return yk_set_error(YK_ERR_CUDA, "yk_debug_ray: out of device memory");
    }
    head.rays = d_rays;
    int rc = YK_OK;
    auto release = [&]() { cudaFree(d_log); cudaFree(d_rays); };
    if (cudaMemcpy(d_log, &head, sizeof(DebugLog), cudaMemcpyHostToDevice) != cudaSuccess) {
        release();
        return yk_set_error(YK_ERR_CUDA, "yk_debug_ray: upload failed");
    }
    yk_film_settings fs{};
    fs.res_x = 1; fs.res_y = 1; fs.tile_dim = 16; fs.accumulate = 1;  // accumulate: render sample index `tile.sample` = 0 only
    yk_tile tile{};
    tile.x0 = 0; tile.y0 = 0; tile.x1 = 1; tile.y1 = 1; tile.sample = 0; tile.index = 0;
    yk_render_opts opts{};
    opts.pipes = 1;
    float li[3] = {0.0f, 0.0f, 0.0f};
    yk_stats st{};
    const float px[2] = {(float)film_px_x, (float)film_px_y};
    rc = render_impl(c, sc, cam, &fs, sm, in, &tile, 1, &opts, li, &st, d_log, px);
    if (rc == YK_OK) {
        if (cudaMemcpy(&head, d_log, sizeof(DebugLog), cudaMemcpyDeviceToHost) != cudaSuccess ||
            cudaMemcpy(rays, d_rays, (size_t)std::min(head.count, cap) * sizeof(yk_integrator_ray), cudaMemcpyDeviceToHost) != cudaSuccess)
            rc = yk_set_error(YK_ERR_CUDA, "yk_debug_ray: read-back failed");
    }
    release();
    if (rc != YK_OK) return rc;
    *n_rays = head.count;
    if (li_rgb) { li_rgb[0] = li[0]; li_rgb[1] = li[1]; li_rgb[2] = li[2]; }
    if (ray_count) *ray_count = st.ray_count;
    return YK_OK;
    });
}


// ---- ray-batch queries ------------------------------------------------------------------------------------
// yk_trace / yk_occluded / yk_query_intersect / yk_query_occluded share one chunk loop (query_run). Host arrays go through
// the context's staging buffers, one synchronise per chunk; device arrays are read and written in place, and the host waits
// once, at the end of the call.
namespace {
struct QueryCall {
    const char* who;
    const float *o, *d, *t_max;
    uint32_t n;
    bool on_device;
    cudaStream_t caller;    // on_device: the pipe's work starts after what is queued here
    const yk_hits* hits;    // closest-hit query: the outputs wanted
    uint8_t* occluded;      // any-hit query (hits == nullptr)
};

bool wants_surface(const yk_hits& h) {
    return h.material || h.area_light || h.p || h.n || h.uv || h.shading_n || h.shading_dpdu;
}

int query_prepare(yk_context* c, const yk_scene* sc, uint32_t n, bool staged, bool staged_surface, uint32_t* chunk) {
    *chunk = std::min<uint32_t>(std::max<uint32_t>(n, 32u), 1u << 22);
    if (staged && c->query_cap < *chunk) {  // staging grows to the largest chunk asked for and stays
        free_bag(c->query_allocs);
        c->query_cap = 0;
        std::vector<void*>& bag = c->query_allocs;
        int rc = YK_OK;
        if ((rc = dev_alloc(bag, &c->q_o, (size_t)3 * *chunk)) != YK_OK || (rc = dev_alloc(bag, &c->q_d, (size_t)3 * *chunk)) != YK_OK ||
            (rc = dev_alloc(bag, &c->q_tm, *chunk)) != YK_OK || (rc = dev_alloc(bag, &c->q_t, *chunk)) != YK_OK ||
            (rc = dev_alloc(bag, &c->q_id, *chunk)) != YK_OK || (rc = dev_alloc(bag, &c->q_cnt, (size_t)2 * *chunk)) != YK_OK ||
            (rc = dev_alloc(bag, &c->q_occ, *chunk)) != YK_OK) {
            free_bag(bag);
            return rc;
        }
        c->query_cap = *chunk;
    }
    if (staged_surface && c->query_surface_cap < *chunk) {
        free_bag(c->query_surface_allocs);
        c->query_surface_cap = 0;
        std::vector<void*>& bag = c->query_surface_allocs;
        int rc = YK_OK;
        if ((rc = dev_alloc(bag, &c->q_mat, *chunk)) != YK_OK || (rc = dev_alloc(bag, &c->q_al, *chunk)) != YK_OK ||
            (rc = dev_alloc(bag, &c->q_p, (size_t)3 * *chunk)) != YK_OK || (rc = dev_alloc(bag, &c->q_n, (size_t)3 * *chunk)) != YK_OK ||
            (rc = dev_alloc(bag, &c->q_uv, (size_t)2 * *chunk)) != YK_OK || (rc = dev_alloc(bag, &c->q_sh_n, (size_t)3 * *chunk)) != YK_OK ||
            (rc = dev_alloc(bag, &c->q_sh_dpdu, (size_t)3 * *chunk)) != YK_OK) {
            free_bag(bag);
            return rc;
        }
        c->query_surface_cap = *chunk;
    }
    if (!staged && !c->q_nan) {
        int rc = dev_alloc(c->query_flag_alloc, &c->q_nan, 1);
        if (rc != YK_OK) return rc;
    }
    Pipe& p = c->pipe[0];
    if (p.wave_cap >= *chunk && p.wave_lights == sc->dev.n_lights) return YK_OK;  // a render's (larger) wavefront state is reused
    return ensure_wave(&p, *chunk, sc->dev.n_lights, 0);
}

// YK_QUERY_ON_DEVICE: every array must be device (or managed) memory of the context's GPU, 4-byte aligned
int check_device_array(const yk_context* c, const void* ptr, const char* who, const char* name) {
    if (!ptr) return YK_OK;
    if ((uintptr_t)ptr % 4u != 0)
        return yk_set_error(YK_ERR_INVALID, std::string(who) + ": " + name + " is not 4-byte aligned");
    cudaPointerAttributes a{};
    const cudaError_t e = cudaPointerGetAttributes(&a, ptr);
    if (e != cudaSuccess) (void)cudaGetLastError();
    if (e != cudaSuccess || (a.type != cudaMemoryTypeDevice && a.type != cudaMemoryTypeManaged) || a.device != c->device)
        return yk_set_error(YK_ERR_INVALID, std::string(who) + ": " + name + " is not device memory of the context's GPU (device " +
                                                std::to_string(c->device) + ") although YK_QUERY_ON_DEVICE is set");
    return YK_OK;
}

int query_run(yk_context* c, const yk_scene* sc, const QueryCall& q) {
    std::lock_guard<std::recursive_mutex> guard(c->mu);
    if (sc->ctx != c) return yk_set_error(YK_ERR_INVALID, std::string(q.who) + ": scene belongs to another context");
    CUDA_TRY(cudaSetDevice(c->device));
    (void)cudaGetLastError();
    const yk_hits none{};
    const yk_hits& h = q.hits ? *q.hits : none;
    if (q.on_device) {
        const std::pair<const void*, const char*> arrays[] = {
            {q.o, "o_xyz"}, {q.d, "d_xyz"}, {q.t_max, "t_max"}, {q.occluded, "occluded_out"}, {h.t, "t"}, {h.orig_id, "orig_id"},
            {h.counts, "counts"}, {h.material, "material"}, {h.area_light, "area_light"}, {h.p, "p"}, {h.n, "n"}, {h.uv, "uv"},
            {h.shading_n, "shading_n"}, {h.shading_dpdu, "shading_dpdu"}};
        for (const auto& a : arrays) {
            const int rc = check_device_array(c, a.first, q.who, a.second);
            if (rc != YK_OK) return rc;
        }
    }
    const bool surface = q.hits && wants_surface(h);
    uint32_t chunk = 0;
    int rc = query_prepare(c, sc, q.n, !q.on_device, !q.on_device && surface, &chunk);
    if (rc != YK_OK) return rc;
    Pipe& p = c->pipe[0];
    cudaStream_t s = p.stream;
    const bool check_nan = q.on_device && q.t_max;
    if (q.on_device) {
        // The pipe's stream is non-blocking: without this event it would not order after the caller's queued work.
        // (ev[1] is otherwise unused; the context mutex serialises its users.)
        CUDA_TRY(cudaEventRecord(c->ev[1], q.caller));
        CUDA_TRY(cudaStreamWaitEvent(s, c->ev[1], 0));
        if (check_nan) CUDA_TRY(cudaMemsetAsync(c->q_nan, 0, sizeof(int), s));
    }
    const bool generic = sc->dev.spheres != nullptr || sc->dev.leaf_table != nullptr;
    RenderCfg cfg{};
    cfg.integrator = YK_INTEGRATOR_PATH;
    const int T = 256;
    for (size_t first = 0; first < q.n; first += chunk) {
        const uint32_t m = (uint32_t)std::min<size_t>(chunk, q.n - first);
        const float *o = q.o + 3 * first, *d = q.d + 3 * first, *tm = q.t_max ? q.t_max + first : nullptr;
        if (!q.on_device) {
            CUDA_TRY(cudaMemcpyAsync(c->q_o, o, (size_t)3 * m * sizeof(float), cudaMemcpyHostToDevice, s));
            CUDA_TRY(cudaMemcpyAsync(c->q_d, d, (size_t)3 * m * sizeof(float), cudaMemcpyHostToDevice, s));
            if (tm) CUDA_TRY(cudaMemcpyAsync(c->q_tm, tm, (size_t)m * sizeof(float), cudaMemcpyHostToDevice, s));
            o = c->q_o;
            d = c->q_d;
            tm = tm ? c->q_tm : nullptr;
        }
        IterCounters ctr{};
        if (q.hits) ctr.n_active = m;
        else ctr.mat[0] = m;  // all segments in the first material queue's range of shading positions
        CUDA_TRY(cudaMemcpyAsync(&p.d_ctr[0], &ctr, sizeof(ctr), cudaMemcpyHostToDevice, s));
        CUDA_TRY(cudaMemsetAsync(p.wave.totals, 0, sizeof(Totals), s));
        // where an output of this chunk goes: the caller's array itself, or the staging buffer it is copied back from
        auto out = [&](auto* caller, auto* staged, size_t per) -> decltype(caller) {
            if (!caller) return nullptr;
            return q.on_device ? caller + per * first : staged;
        };
        auto back = [&](auto* caller, const void* staged, size_t per) -> int {
            if (!q.on_device && caller)
                CUDA_TRY(cudaMemcpyAsync(caller + per * first, staged, per * m * sizeof(*caller), cudaMemcpyDeviceToHost, s));
            return YK_OK;
        };
        if (q.hits) {
            k_query_pack<<<(m + T - 1) / T, T, 0, s>>>(p.wave, o, d, tm, m, check_nan ? c->q_nan : nullptr);
            const int blocks = grid_for(m, kTraceThreads, c->sm_count * std::max(1, c->occ_trace_closest));
            if (generic) k_trace_closest<true, true><<<blocks, kTraceThreads, 0, s>>>(sc->dev, p.wave, 0, &p.d_ctr[0], nullptr);
            else k_trace_closest<true, false><<<blocks, kTraceThreads, 0, s>>>(sc->dev, p.wave, 0, &p.d_ctr[0], nullptr);
            if (h.t || h.orig_id || h.counts)
                k_query_unpack<<<(m + T - 1) / T, T, 0, s>>>(sc->dev, p.wave, m, out(h.t, c->q_t, 1), out(h.orig_id, c->q_id, 1),
                                                             out(h.counts, c->q_cnt, 2));
            if (surface) {
                QuerySurfaceOut so;
                so.material = out(h.material, c->q_mat, 1);
                so.area_light = out(h.area_light, c->q_al, 1);
                so.p = out(h.p, c->q_p, 3);
                so.n = out(h.n, c->q_n, 3);
                so.uv = out(h.uv, c->q_uv, 2);
                so.sh_n = out(h.shading_n, c->q_sh_n, 3);
                so.sh_dpdu = out(h.shading_dpdu, c->q_sh_dpdu, 3);
                k_query_surface<<<(m + T - 1) / T, T, 0, s>>>(sc->dev, p.wave, m, so);
            }
            if ((rc = back(h.t, c->q_t, 1)) != YK_OK || (rc = back(h.orig_id, c->q_id, 1)) != YK_OK ||
                (rc = back(h.counts, c->q_cnt, 2)) != YK_OK || (rc = back(h.material, c->q_mat, 1)) != YK_OK ||
                (rc = back(h.area_light, c->q_al, 1)) != YK_OK || (rc = back(h.p, c->q_p, 3)) != YK_OK ||
                (rc = back(h.n, c->q_n, 3)) != YK_OK || (rc = back(h.uv, c->q_uv, 2)) != YK_OK ||
                (rc = back(h.shading_n, c->q_sh_n, 3)) != YK_OK || (rc = back(h.shading_dpdu, c->q_sh_dpdu, 3)) != YK_OK)
                return rc;
        } else {
            k_query_pack_segments<<<(m + T - 1) / T, T, 0, s>>>(p.wave, o, d, m);
            const bool per_ray = c->shadow_mode != 0;  // one segment per lane either way; the per-ray kernel needs no fold
            if (per_ray) {
                const int blocks = grid_for(m, kTraceThreads, c->sm_count * std::max(1, c->occ_trace_rays));
                if (generic) k_trace_shadow_rays<true><<<blocks, kTraceThreads, 0, s>>>(sc->dev, p.wave, 1u, &p.d_ctr[0]);
                else k_trace_shadow_rays<false><<<blocks, kTraceThreads, 0, s>>>(sc->dev, p.wave, 1u, &p.d_ctr[0]);
            } else {
                const int blocks = grid_for(m, kTraceThreads, c->sm_count * std::max(1, c->occ_trace_any));
                if (generic) k_trace_shadow<true><<<blocks, kTraceThreads, 0, s>>>(sc->dev, p.wave, cfg, &p.d_ctr[0]);
                else k_trace_shadow<false><<<blocks, kTraceThreads, 0, s>>>(sc->dev, p.wave, cfg, &p.d_ctr[0]);
            }
            k_query_unpack_segments<<<(m + T - 1) / T, T, 0, s>>>(p.wave, m, per_ray ? 1 : 0, out(q.occluded, c->q_occ, 1));
            if ((rc = back(q.occluded, c->q_occ, 1)) != YK_OK) return rc;
        }
        if (!q.on_device) CUDA_TRY(cudaStreamSynchronize(s));
    }
    if (q.on_device) {
        int nan_seen = 0;
        if (check_nan) CUDA_TRY(cudaMemcpyAsync(&nan_seen, c->q_nan, sizeof(int), cudaMemcpyDeviceToHost, s));
        CUDA_TRY(cudaStreamSynchronize(s));
        if (nan_seen) return yk_set_error(YK_ERR_INVALID, std::string(q.who) + ": NaN t_max (Ray::new, math/ray.rs)");
    }
    CUDA_TRY(cudaGetLastError());
    return YK_OK;
}

// opts of yk_query_intersect / yk_query_occluded -> (on_device, caller stream)
int query_options(const yk_query_opts* opts, const char* who, bool* on_device, cudaStream_t* stream) {
    *on_device = false;
    *stream = nullptr;
    if (!opts) return YK_OK;
    if (opts->flags & ~YK_QUERY_ON_DEVICE) return yk_set_error(YK_ERR_INVALID, std::string(who) + ": unknown flag bits");
    if (opts->_reserved != 0) return yk_set_error(YK_ERR_INVALID, std::string(who) + ": _reserved must be 0");
    *on_device = (opts->flags & YK_QUERY_ON_DEVICE) != 0;
    *stream = *on_device ? (cudaStream_t)opts->stream : nullptr;
    return YK_OK;
}
}  // namespace

// BoundingVolumeHierarchy::intersect (bvh.rs:160-232) for n caller rays.
int yk_trace(yk_context* c, const yk_scene* sc, const float* o_xyz, const float* d_xyz, const float* t_max, uint32_t n, float* t_out,
             int32_t* orig_id_out, uint32_t* counts_out) {
    return yk_guard("yk_trace", [&]() -> int {
    if (!c || !sc || (n && (!o_xyz || !d_xyz || !t_out || !orig_id_out))) return yk_set_error(YK_ERR_INVALID, "yk_trace: null argument");
    if (n == 0) return YK_OK;
    for (size_t i = 0; t_max && i < n; ++i)
        if (t_max[i] != t_max[i]) return yk_set_error(YK_ERR_INVALID, "yk_trace: NaN t_max (Ray::new, math/ray.rs)");
    yk_hits hits{};
    hits.t = t_out;
    hits.orig_id = orig_id_out;
    hits.counts = counts_out;
    return query_run(c, sc, QueryCall{"yk_trace", o_xyz, d_xyz, t_max, n, false, nullptr, &hits, nullptr});
    });
}

// VisibilityTester::unoccluded's traversal (visibility.rs:6-23 -> any_intersect, bvh.rs:235-302) for n caller segments
// o -> o + d, cut at t_max = 0.9999 like every shadow ray of the reference (interaction.rs:57-58).
int yk_occluded(yk_context* c, const yk_scene* sc, const float* o_xyz, const float* d_xyz, uint32_t n, uint8_t* occluded_out) {
    return yk_guard("yk_occluded", [&]() -> int {
    if (!c || !sc || (n && (!o_xyz || !d_xyz || !occluded_out))) return yk_set_error(YK_ERR_INVALID, "yk_occluded: null argument");
    if (n == 0) return YK_OK;
    return query_run(c, sc, QueryCall{"yk_occluded", o_xyz, d_xyz, nullptr, n, false, nullptr, nullptr, occluded_out});
    });
}

// Scene::intersect (bvh.rs:160-232 + the hit's SurfaceInteraction) for n caller rays, on host or device arrays.
int yk_query_intersect(yk_context* c, const yk_scene* sc, const float* o_xyz, const float* d_xyz, const float* t_max, uint32_t n,
                       const yk_query_opts* opts, const yk_hits* out) {
    return yk_guard("yk_query_intersect", [&]() -> int {
    if (!c || !sc || !out || (n && (!o_xyz || !d_xyz))) return yk_set_error(YK_ERR_INVALID, "yk_query_intersect: null argument");
    bool on_device = false;
    cudaStream_t stream = nullptr;
    int rc = query_options(opts, "yk_query_intersect", &on_device, &stream);
    if (rc != YK_OK || n == 0) return rc;
    for (size_t i = 0; !on_device && t_max && i < n; ++i)  // device arrays: k_query_pack raises c->q_nan instead
        if (t_max[i] != t_max[i]) return yk_set_error(YK_ERR_INVALID, "yk_query_intersect: NaN t_max (Ray::new, math/ray.rs)");
    return query_run(c, sc, QueryCall{"yk_query_intersect", o_xyz, d_xyz, t_max, n, on_device, stream, out, nullptr});
    });
}

// yk_occluded on host or device arrays.
int yk_query_occluded(yk_context* c, const yk_scene* sc, const float* o_xyz, const float* d_xyz, uint32_t n, const yk_query_opts* opts,
                      uint8_t* occluded_out) {
    return yk_guard("yk_query_occluded", [&]() -> int {
    if (!c || !sc || (n && (!o_xyz || !d_xyz || !occluded_out))) return yk_set_error(YK_ERR_INVALID, "yk_query_occluded: null argument");
    bool on_device = false;
    cudaStream_t stream = nullptr;
    int rc = query_options(opts, "yk_query_occluded", &on_device, &stream);
    if (rc != YK_OK || n == 0) return rc;
    return query_run(c, sc, QueryCall{"yk_query_occluded", o_xyz, d_xyz, nullptr, n, on_device, stream, nullptr, occluded_out});
    });
}


// Sampler::{start_pixel_sample, get_1d, get_2d} evaluated on the device for n (pixel x, pixel y, sample index) triples.
int yk_sampler_draws(yk_context* c, const yk_sampler* sm, const uint32_t* pixel_index_xyi, uint32_t n, const uint8_t* pattern,
                     uint32_t n_pattern, float* out) {
    return yk_guard("yk_sampler_draws", [&]() -> int {
    if (!c || !sm || (n && (!pixel_index_xyi || !out)) || (n_pattern && !pattern)) return yk_set_error(YK_ERR_INVALID, "yk_sampler_draws: null argument");
    if (sm->kind > YK_SAMPLER_STRATIFIED) return yk_set_error(YK_ERR_INVALID, "yk_sampler_draws: unknown sampler");
    const uint32_t spp = sm->kind == YK_SAMPLER_UNIFORM ? sm->nx : sm->nx * sm->ny;
    if (spp == 0 || spp > 0x10000u) return yk_set_error(YK_ERR_INVALID, "yk_sampler_draws: samples per pixel must be in 1..65536");
    uint32_t floats = 0;
    for (uint32_t k = 0; k < n_pattern; ++k) {
        if (pattern[k] != 1 && pattern[k] != 2) return yk_set_error(YK_ERR_INVALID, "yk_sampler_draws: pattern entries are 1 (get_1d) or 2 (get_2d)");
        floats += pattern[k];
    }
    for (size_t i = 0; i < n; ++i)
        if (pixel_index_xyi[3 * i] > 0xffffu || pixel_index_xyi[3 * i + 1] > 0xffffu || pixel_index_xyi[3 * i + 2] > 0xffffu)
            return yk_set_error(YK_ERR_INVALID, "yk_sampler_draws: pixel coordinates and sample index must fit u16 (integrators/mod.rs:140-141)");
    if (n == 0 || floats == 0) return YK_OK;
    std::lock_guard<std::recursive_mutex> guard(c->mu);
    CUDA_TRY(cudaSetDevice(c->device));
    SamplerCfg cfg{};
    cfg.kind = sm->kind;
    cfg.nx = sm->nx;
    cfg.ny = sm->kind == YK_SAMPLER_UNIFORM ? 1u : sm->ny;
    cfg.jitter = sm->jitter;
    cfg.seed = sm->seed;
    cfg.div_nx = FastDiv::make(cfg.nx);
    cfg.div_ny = FastDiv::make(cfg.ny);
    cfg.div_n = FastDiv::make(cfg.nx * cfg.ny);
    std::vector<void*> bag;
    uint32_t* d_in = nullptr;
    uint8_t* d_pat = nullptr;
    float* d_out = nullptr;
    int rc = YK_OK;
    if ((rc = dev_alloc(bag, &d_in, (size_t)3 * n)) != YK_OK || (rc = dev_alloc(bag, &d_pat, n_pattern)) != YK_OK ||
        (rc = dev_alloc(bag, &d_out, (size_t)n * floats)) != YK_OK) {
        free_bag(bag);
        return rc;
    }
    cudaStream_t s = c->stream;
    cudaError_t e = cudaMemcpyAsync(d_in, pixel_index_xyi, (size_t)3 * n * sizeof(uint32_t), cudaMemcpyHostToDevice, s);
    if (e == cudaSuccess) e = cudaMemcpyAsync(d_pat, pattern, n_pattern, cudaMemcpyHostToDevice, s);
    if (e == cudaSuccess) {
        k_sampler_draws<<<(n + 127) / 128, 128, 0, s>>>(cfg, d_in, n, d_pat, n_pattern, floats, d_out);
        e = cudaGetLastError();
    }
    if (e == cudaSuccess) e = cudaMemcpyAsync(out, d_out, (size_t)n * floats * sizeof(float), cudaMemcpyDeviceToHost, s);
    if (e == cudaSuccess) e = cudaStreamSynchronize(s);
    free_bag(bag);
    if (e != cudaSuccess) return yk_set_error(YK_ERR_CUDA, std::string("yk_sampler_draws: ") + cudaGetErrorString(e));
    return YK_OK;
    });
}

}  // extern "C"

#include "multi.inl"
