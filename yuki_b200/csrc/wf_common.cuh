// Types shared by the wavefront kernels and the host driver of render.cu: the device-resident scene, the per-bounce
// counters, the SoA path state, and the block-aggregated queue append.
// Part of the single translation unit render.cu (compiled --fmad=false: every float op is the reference's un-fused IEEE op).
#pragma once
#include <cuda_runtime.h>

#include <cstdint>
#include <string>

#include "yk_device.cuh"
#include "yuki_gpu.h"

int yk_set_error(int code, const std::string& msg);  // host_scene.cpp

using namespace ykd;

namespace {


constexpr int kMaxLights = 32;  // one bit per light in the shading kernels' shadow-ray mask
constexpr int kStackDepth = 64;  // bvh.rs:172
constexpr uint32_t kMiss = 0xffffffffu;
constexpr int kTraceThreads = 128;
#ifndef YK_SHADE_THREADS
// 256 threads with the phase barriers of shade_item (k_shade<.., PHASED = true>): the blocks' warps stay inside the same part of
// the ~100 KB kernel, whose top stall at 128 unsynchronised threads was `no_instruction` (32 KB instruction cache). Measured (one
// pipe, profiles/r02/ab_shade_phased.txt): shading time of the material room 29.0 -> 23.9 ms (render +5 %), terrain 6.9 -> 6.6 ms,
// Cornell box unchanged; 512 threads = 256, 1024 threads and barriers without larger blocks are slower.
#define YK_SHADE_THREADS 256
#endif
constexpr int kShadeThreads = YK_SHADE_THREADS;
constexpr int kShadeThreadsPlain = 128;  // the barrier-free instantiation (k_shade<.., PHASED = false>)
#ifndef YK_TRACE_MIN_BLOCKS
// Closest hit: a bound of 6 (cap 80 registers) instead of 8 (cap 64). The path-tracing instantiation still settles on 64
// registers and runs 8 blocks per SM, but without squeezing under a hard cap its schedule is ~2 % faster; the counting /
// sphere instantiations take 72-76 registers (measured 5 = 6, 7 slower than both 6 and 8).
#define YK_TRACE_MIN_BLOCKS 6
#endif
#ifndef YK_SHADOW_MIN_BLOCKS
#define YK_SHADOW_MIN_BLOCKS 8
#endif
#ifndef YK_SHADE_MIN_BLOCKS
#define YK_SHADE_MIN_BLOCKS (1024 / YK_SHADE_THREADS)
#endif

// Wavefront state is written once and read once per bounce, several GB per batch: with YK_STREAM_HINTS its loads and stores
// carry the evict-first policy (ld/st.global.cs), so that they do not push the scene, the pixel-job table and the sampler's
// hash table out of the L2. The shadow / fold kernel reads its inputs twice (the light mask, then the pending terms) and keeps
// plain loads. Measured: +0.5 % (Cornell) ... +1.4 % (1 M-triangle heightfield) render throughput.
#ifndef YK_STREAM_HINTS
#define YK_STREAM_HINTS 1
#endif
template <class T>
__device__ __forceinline__ T ld_once(const T* p) {
#if YK_STREAM_HINTS
    return __ldcs(p);
#else
    return *p;
#endif
}
template <class T>
__device__ __forceinline__ void st_once(T* p, T v) {
#if YK_STREAM_HINTS
    __stcs(p, v);
#else
    *p = v;
#endif
}

// Checked build (-DYK_CHECKED, scripts/checked_build.sh): device-side bounds assertions on every hand-computed index — the
// traversal stack pointer, leaf / record / queue / hand-over indices, sort bins. compute-sanitizer is closed on this GPU pool
// ("runs under it have left GPUs needing a reset"), so the GPU test-suite is run against this build instead; a violated
// assertion surfaces as cudaErrorAssert from the call that launched the kernel.
#ifdef YK_CHECKED
#include <cassert>
#define YK_ASSERT(x) assert(x)
#else
#define YK_ASSERT(x) ((void)0)
#endif

#define CUDA_TRY(expr)                                                                                          \
    do {                                                                                                        \
        cudaError_t e_ = (expr);                                                                                \
        if (e_ != cudaSuccess)                                                                                  \
            return yk_set_error(YK_ERR_CUDA, std::string(#expr) + ": " + cudaGetErrorString(e_));              \
    } while (0)

// ---- device-resident scene ------------------------------------------------------------------------
struct DevTexture {
    uint32_t kind, width, height, _pad;
    float value[3];
    float _pad2;
    const float* texels;
};
struct DevMaterial {
    uint32_t kind;
    int32_t tex[3];
    float eta;
    uint32_t remap;
    float const_alpha;  // >= 0: roughness texture is constant, alpha fully evaluated on the host
    uint32_t _pad;
};
struct DevScene {
    // One 64-byte record per *interior* node holding the boxes of its two children (DESIGN.md §3):
    //   (p_min child0, ref0) (p_max child0, -) (p_min child1, ref1) (p_max child1, -)
    // child0 = the node after its parent in the reference's pre-order array, child1 = second_child_index (bvh.rs:396-419).
    // A visit loads both boxes with one request; leaves have no record of their own (their shape range is in the ref).
    const float4* nodes2;
    const uint2* leaf_table;  // null: leaf refs are packed (count - 1) << 27 | first; else ref = index of (first, count)
    const float4* tris;    // 3 x float4 per triangle: (x0 x1 x2, area_light) (y0 y1 y2, material | flags<<24) (z0 z1 z2, orig_id)
    const float* normals;  // 9 per triangle or null
    const float* uvs;      // 6 per triangle or null
    const DevTexture* textures;
    const DevMaterial* materials;
    const yk_light* lights;
    const yk_sphere* spheres;  // sphere slots of `tris`: vertex lanes are NaN (so the triangle test "accepts" them and the
                               // rare hit path takes over), row 0's w = -2 - sphere index
    uint32_t n_lights, n_tris, n_nodes;
    float background[3];
    float root_min[3], root_max[3];  // the root's own box (tested once per ray)
    uint32_t root_ref;
};
// Child refs: interior = kRefInterior | split_axis << 29 | record index (the axis picks the near child before the record is
// loaded); leaf = bit 31 clear, see leaf_table. kNoNode (all ones) is the stack sentinel / "no node".
constexpr uint32_t kRefInterior = 0x80000000u;
constexpr uint32_t kRefIndexMask = 0x1fffffffu;
constexpr uint32_t kLeafFirstBits = 27;

// ---- per-iteration device counters ----------------------------------------------------------------
// Queue lengths never leave the device: every kernel of a bounce reads its element count from `cur` and appends to
// `nxt`, so a batch is one asynchronous launch sequence (no host round trip per bounce).
struct IterCounters {
    uint32_t n_active;      // rays of this bounce (length of the active queue)
    uint32_t mat[4];        // material queue lengths
    uint32_t work_closest;  // dynamic ray fetch cursors
    uint32_t work_shadow;
    uint32_t _pad;
};
struct Totals {
    unsigned long long closest_nodes, closest_tris, any_nodes, any_tris, hit_hash, shadow_rays, closest_rays;
};

struct Job {  // + the pixel's PCG stream, (SipHash13(x, y) << 1) | 1 (uniform.rs:77-81): one hash per pixel, not per sample
    uint16_t x, y;
    uint32_t sample_begin;
    unsigned long long rng_inc;
};
// Path i of a batch is sample (sample_begin + sample_off + i / n_jobs) of pixel jobs[i % n_jobs]: a warp holds
// 32 neighbouring pixels of one tile row at the same sample index.
struct Batch {
    const Job* jobs;
    uint32_t n_jobs, sample_off, n_samples, n_paths;
    FastDiv div_jobs;  // by n_jobs
};

// ---- wavefront state (SoA, capacity `cap` paths) --------------------------------------------------
// Per bounce a path touches: ray (32 B) + hit (8 B) in the traversal; ray, hit, rng state (8 B), beta (16 B) in
// shading, which writes the next ray / beta / rng state, the pending radiance terms (32 B) and 40 B per light that
// needs a shadow ray; the shadow kernel reads those back and does the one read-modify-write of L (DESIGN.md §3).
struct Wave {
    uint32_t cap, n_lights, stack_entries;
    // Per-bounce path state, streamed: bounce b reads st[b & 1] at the ray's queue slot and the shading kernels write the
    // survivors' state to st[(b + 1) & 1] at their position in the next queue. Every kernel therefore reads and writes
    // dense, (near-)coalesced arrays; nothing is gathered through a path index except L and the Whitted stack.
    struct Stream {
        float4* ray_o;   // o.xyz, t_max
        float4* ray_d;   // d.xyz, -
        // path: throughput, w = flags | sampler dimension << kDimShift. whitted: x = sampler dimension (uint bits), y, z = 1,
        // w = flags: a Whitted sample draws 2 * lights dimensions per tree node, and its trees outgrow the 21 bits of w
        float4* beta;
        unsigned long long* rng;
    } st[2];
    uint2* hit;         // per queue slot: t bits, shape slot (kMiss = none)
    uint2* bvh_counts;  // BVHIntersections: tests, hits
    float4* L;       // accumulated radiance
    // The five arrays below are the shading kernels' hand-over to the shadow kernel. They are indexed by the *shading
    // position* g (position in the concatenation of this bounce's four material queues), not by path: the shading
    // kernels write them fully coalesced and the shadow kernel streams them with no dependent gather.
    uint32_t* sh_path;   // path of shading position g
    uint32_t* sh_mask;   // bit k: light k's shadow ray of shading position g is to be traced / (after k_trace_shadow_rays) is unoccluded
    float4* pend_beta;   // path: weight to apply to this bounce's radiance; w = clamp flag. whitted: node depth | has-children << 8, sampler dimension, -, -1
    float4* pend_extra;  // emitted term of this bounce; w = bit mask of the lights whose shadow ray must be traced
    float4* lt_o;        // cap * n_lights: shadow ray o.xyz | contribution.r   (contribution = f * li * cos / pdf)
    float4* lt_d;        //                 shadow ray d.xyz | contribution.g
    float2* lt_c;        //                 contribution.b   | area light id of the sampled light (int bits, -1 = none)
    float4* stack;       // whitted: recursion frames, stack_entries * cap * 5 float4 (wf_shade.cuh)
    unsigned long long* tree_rng;  // whitted: sampler state after shading position g (nodes without children)
    uint32_t* q_active[2];
    uint32_t* q_mat;     // 4 * cap: paths per material kind
    uint32_t* q_mat_tri; // 4 * cap: the hit shape slot of each entry
    uint32_t* q_mat_slot; // 4 * cap: the entry's slot in this bounce's active queue (index of st[] / hit[])
    // Ray sort (wf_sort.cuh): the shading kernels leave a coherence key per survivor, a counting sort turns the keys into
    // `perm` (sorted position -> queue slot), and the next bounce's traversal (and optionally its material sort) walks the
    // queue through it. Null when the render does not sort.
    uint32_t* sort_key;  // cap
    uint32_t* perm;      // cap
    uint32_t* sort_bins; // kSortBins + 1: histogram, then the bins' write cursors
    Totals* totals;
};
constexpr uint32_t kSortKeyBits = 18;  // 15 spatial bits (major) + 3 direction-octant bits
constexpr uint32_t kSortBins = 1u << kSortKeyBits;
// beta.w flag word
constexpr uint32_t kFlagSpecular = 0x100u;   // path: specular_bounce / whitted: is_specular
constexpr uint32_t kFlagAlive = 0x200u;
constexpr uint32_t kFlagTransmission = 0x400u;  // the ray left a TRANSMISSION lobe (ray type of li_debug, path.rs:146-153)
constexpr uint32_t kDepthMask = 0xffu;       // path: bounces / whitted: depth
constexpr uint32_t kDimShift = 11;           // path: sampler dimension (stratified.rs:40) in the upper 21 bits
constexpr uint32_t kFlagMask = (1u << kDimShift) - 1u;

// Ray list of Integrator::li_debug (integrators/mod.rs:76-118), filled by k_debug_log for the one path of yk_debug_ray.
struct DebugLog {
    uint32_t count, cap;
    float min_len;  // min_debug_ray_length: a tenth of the scene bounds' largest extent (path.rs:58-62, whitted.rs:84-88)
    uint32_t _pad;
    yk_integrator_ray* rays;
};

struct RenderCfg {
    SamplerCfg sampler;
    uint32_t integrator, max_depth, has_clamp;
    float clamp;
    float c2w[16], r2c[16];
    uint32_t res_x, res_y;
    uint32_t aux_sample;
    int32_t* hit_ids;  // device, or null
    DebugLog* debug_log;  // yk_debug_ray only: the single path's rays; the camera sample lands on film pixel debug_px
    float debug_px[2];
    // ray sort: 0 = none; 1 = key from the hit shape's leaf slot (BVH order is a spatial order) + direction octant;
    // 2 = key from the Morton cell of the ray origin inside the scene bounds + direction octant
    uint32_t shadow_per_ray;      // the shadow rays of this render are traced one per lane (k_trace_shadow_rays): the shading kernels fill sh_mask
    uint32_t sort_key_mode;
    uint32_t sort_order;          // 1 = the closest-hit kernel walks the sorted order; 2 = the material sort (hence shading, shadow rays) too
    uint32_t sort_slot_shift;     // mode 1: leaf slot >> shift gives the 15 spatial key bits
    float sort_cell_scale[3];     // mode 2: (o - root_min) * scale = cell coordinate in [0, 32)
};

// ---- helpers --------------------------------------------------------------------------------------
__device__ __forceinline__ V3 f4v(float4 a) { return {a.x, a.y, a.z}; }

__device__ __forceinline__ unsigned long long warp_sum(unsigned long long v) {
    for (int o = 16; o > 0; o >>= 1) v += __shfl_down_sync(0xffffffffu, v, o);
    return v;
}
// Block-aggregated append to one of NQ queues: one global atomic per queue per block (same-address atomics were the
// bottleneck of classify / resolve with one atomic per warp, profiles/r01). `key` in [0, NQ) selects the queue, any
// other value appends nothing. Must be reached by every thread of the block (blockDim.x <= 1024).
// Returns the slot the value was written to (undefined when nothing was appended).
// `K` items per thread share the block's atomics: K * blockDim.x items per global atomic and queue.
#ifdef YK_CHECKED
__device__ uint32_t g_check_queue_cap = 0xffffffffu;  // set by the host driver to the wavefront capacity before each batch
#define YK_CHECK_QUEUE_CAP g_check_queue_cap
#endif
template <int NQ, int K>
__device__ __forceinline__ void block_scatter_multi(const int (&key)[K], const uint32_t (&value)[K], uint32_t* const (&queues)[NQ],
                                                    uint32_t* const (&counters)[NQ], uint32_t (&pos)[K]) {
    __shared__ uint32_t s_cnt[32][NQ];
    __shared__ uint32_t s_base[NQ];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, n_warps = (blockDim.x + 31) >> 5;
    const unsigned lt = (1u << lane) - 1u;
    uint32_t run[NQ];  // warp-uniform: entries of this warp per queue so far
    uint32_t my_rank[K];
#pragma unroll
    for (int q = 0; q < NQ; ++q) run[q] = 0;
#pragma unroll
    for (int k = 0; k < K; ++k) {
        my_rank[k] = 0;
#pragma unroll
        for (int q = 0; q < NQ; ++q) {
            const unsigned votes = __ballot_sync(0xffffffffu, key[k] == q);
            if (key[k] == q) my_rank[k] = run[q] + __popc(votes & lt);
            run[q] += __popc(votes);
        }
    }
    if (lane == 0) {
#pragma unroll
        for (int q = 0; q < NQ; ++q) s_cnt[warp][q] = run[q];
    }
    __syncthreads();
    if (threadIdx.x < NQ) {
        uint32_t total = 0;
        for (int wi = 0; wi < n_warps; ++wi) {
            const uint32_t c = s_cnt[wi][threadIdx.x];
            s_cnt[wi][threadIdx.x] = total;  // exclusive prefix over the block's warps
            total += c;
        }
        s_base[threadIdx.x] = total ? atomicAdd(counters[threadIdx.x], total) : 0u;
    }
    __syncthreads();
#pragma unroll
    for (int k = 0; k < K; ++k) {
        pos[k] = 0;
        if (key[k] >= 0 && key[k] < NQ) {
            pos[k] = s_base[key[k]] + s_cnt[warp][key[k]] + my_rank[k];
            YK_ASSERT(pos[k] < YK_CHECK_QUEUE_CAP);
            queues[key[k]][pos[k]] = value[k];
        }
    }
    __syncthreads();  // the shared arrays are reused by the next call
}
template <int NQ>
__device__ __forceinline__ uint32_t block_scatter(int key, uint32_t value, uint32_t* const (&queues)[NQ], uint32_t* const (&counters)[NQ]) {
    const int keys[1] = {key};
    const uint32_t values[1] = {value};
    uint32_t pos[1];
    block_scatter_multi<NQ, 1>(keys, values, queues, counters, pos);
    return pos[0];
}
__device__ __forceinline__ unsigned long long mix_hit(uint32_t x, uint32_t y, uint32_t sample, uint32_t id) {
    unsigned long long h = ((unsigned long long)x << 48) ^ ((unsigned long long)y << 32) ^ ((unsigned long long)sample << 8) ^
                           (unsigned long long)id * 0x9E3779B97F4A7C15ULL;
    h ^= h >> 31; h *= 0xBF58476D1CE4E5B9ULL; h ^= h >> 29;
    return h;
}

}  // namespace
