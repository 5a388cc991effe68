// yk_denoise: an edge-avoiding a-trous wavelet filter (Dammertz et al., HPG 2010) whose colour weights are scaled by each
// pixel's own variance estimate (SVGF, Schied et al., HPG 2017). Every input comes from the render that made the film: the
// mean, the mean of li * li (`radiance_sq`), the per-pixel sample count and optionally a normal companion film as the edge
// guide. The rule (include/yuki_gpu.h) uses only un-fused + - * /, sqrtf and comparisons, written in the header's order: the
// library is compiled --fmad=false -prec-div=true -prec-sqrt=true, so the numpy float32 restatement in tests/denoise_reference.py gives the
// same bits.
//
// k_denoise_setup packs each pixel into two float4: (colour, variance) and (unit guide normal, 1 when the pixel is filtered,
// i.e. n >= 2). One k_denoise_step launch per iteration then reads a tap as two 16-byte loads, through L1 / L2, ping-ponging
// the (colour, variance) buffers; the last one writes the RGB output.
#include <cuda_runtime.h>

#include <algorithm>
#include <cfloat>
#include <mutex>
#include <string>
#include <utility>

#include "yuki_gpu.h"
#include "yk_guard.h"

int yk_set_error(int code, const std::string& msg);  // host_scene.cpp
int yk_context_activate(yk_context* c);                 // render.cu
std::recursive_mutex& yk_context_mutex(yk_context* c);  // render.cu
int yk_context_follow(yk_context* c, void* caller_stream);

namespace {

#define DN_TRY(expr)                                                                                \
    do {                                                                                            \
        cudaError_t e_ = (expr);                                                                    \
        if (e_ != cudaSuccess)                                                                      \
            return yk_set_error(YK_ERR_CUDA, std::string(#expr) + ": " + cudaGetErrorString(e_));   \
    } while (0)

constexpr int kBlockX = 32, kBlockY = 8;
constexpr uint32_t kMaxIterations = 10;

__global__ void k_denoise_setup(const float* film, const float* sq, const uint32_t* counts, uint32_t spp, const float* normals,
                                size_t n_px, float4* cv, float4* guide) {
    for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < n_px; i += (size_t)gridDim.x * blockDim.x) {
        const uint32_t n = counts ? counts[i] : spp;
        const float r = film[3 * i], g = film[3 * i + 1], b = film[3 * i + 2];
        float var = 0.0f;
        float4 nh = make_float4(0.0f, 0.0f, 0.0f, 0.0f);
        if (n >= 2) {
            const float nf = (float)n;
            float v[3];
            for (int ch = 0; ch < 3; ++ch) {
                const float c = film[3 * i + ch];
                float e = sq[3 * i + ch] - c * c;
                if (e < 0.0f) e = 0.0f;  // (a NaN stays NaN)
                v[ch] = e / (nf - 1.0f);
            }
            var = (v[0] + v[1]) + v[2];
            nh.w = 1.0f;
            if (normals) {
                const float dx = normals[3 * i] * 2.0f - 1.0f, dy = normals[3 * i + 1] * 2.0f - 1.0f, dz = normals[3 * i + 2] * 2.0f - 1.0f;
                const float l2 = (dx * dx + dy * dy) + dz * dz;
                if (l2 > 0.0f) {
                    const float l = sqrtf(l2);
                    nh.x = dx / l;
                    nh.y = dy / l;
                    nh.z = dz / l;
                }
            }
        }
        cv[i] = make_float4(r, g, b, var);
        guide[i] = nh;
    }
}

// One a-trous iteration at step `step`: one thread per pixel, the 5x5 taps ky outer, kx inner. LAST writes RGB to `rgb_out`,
// otherwise (colour, variance) to `cv_out`.
template <bool GUIDE, bool LAST>
__global__ void __launch_bounds__(kBlockX * kBlockY) k_denoise_step(const float4* __restrict__ cv, const float4* __restrict__ guide,
                                                                    uint32_t res_x, uint32_t res_y, int step, float sigma2, float eps,
                                                                    float4* __restrict__ cv_out, float* __restrict__ rgb_out) {
    const float h[5] = {1.0f / 16.0f, 1.0f / 4.0f, 3.0f / 8.0f, 1.0f / 4.0f, 1.0f / 16.0f};
    const int x = (int)(blockIdx.x * kBlockX + threadIdx.x);
    if (x >= (int)res_x) return;
    for (int y = (int)(blockIdx.y * kBlockY + threadIdx.y); y < (int)res_y; y += (int)(gridDim.y * kBlockY)) {
        const size_t p = (size_t)y * res_x + x;
        const float4 cp = cv[p];
        float4 res = cp;
        const float4 np = guide[p];
        if (np.w != 0.0f) {  // n >= 2: filtered; otherwise copied through
            float W = 0.0f, cr = 0.0f, cg = 0.0f, cb = 0.0f, V = 0.0f;
#pragma unroll
            for (int ky = 0; ky < 5; ++ky) {
                const int qy = y + step * (ky - 2);
                if (qy < 0 || qy >= (int)res_y) continue;
#pragma unroll
                for (int kx = 0; kx < 5; ++kx) {
                    const int qx = x + step * (kx - 2);
                    if (qx < 0 || qx >= (int)res_x) continue;
                    float w;
                    float4 cq = cp;
                    if (ky == 2 && kx == 2) {
                        w = h[2] * h[2];
                    } else {
                        const size_t q = (size_t)qy * res_x + qx;
                        const float4 nq = GUIDE ? guide[q] : make_float4(0.0f, 0.0f, 0.0f, __ldg(&guide[q].w));
                        if (nq.w == 0.0f) continue;  // n < 2: never a tap
                        cq = cv[q];
                        const float dr = cp.x - cq.x, dg = cp.y - cq.y, db = cp.z - cq.z;
                        const float num = (dr * dr + dg * dg) + db * db;
                        const float den = sigma2 * (cp.w + cq.w) + eps;
                        float wc = den / (den + num);
                        wc = wc * wc;
                        float wn = 1.0f;
                        if (GUIDE) {
                            const float t = (np.x * nq.x + np.y * nq.y) + np.z * nq.z;
                            wn = t > 0.0f ? t : 0.0f;
#pragma unroll
                            for (int k = 0; k < 7; ++k) wn = wn * wn;  // t^128
                        }
                        w = ((h[ky] * h[kx]) * wn) * wc;
                        if (!(w > 0.0f)) continue;  // zero, or NaN from a NaN / infinite neighbour: skipped, nothing spreads
                    }
                    W = W + w;
                    cr = cr + w * cq.x;
                    cg = cg + w * cq.y;
                    cb = cb + w * cq.z;
                    V = V + (w * w) * cq.w;
                }
            }
            res = make_float4(cr / W, cg / W, cb / W, V / (W * W));
        }
        if (LAST) {
            rgb_out[3 * p] = res.x;
            rgb_out[3 * p + 1] = res.y;
            rgb_out[3 * p + 2] = res.z;
        } else {
            cv_out[p] = res;
        }
    }
}

template <bool GUIDE>
void launch_step(bool last, dim3 grid, cudaStream_t s, const float4* cv, const float4* guide, uint32_t res_x, uint32_t res_y, int step,
                 float sigma2, float eps, float4* cv_out, float* rgb_out) {
    const dim3 block(kBlockX, kBlockY);
    if (last) k_denoise_step<GUIDE, true><<<grid, block, 0, s>>>(cv, guide, res_x, res_y, step, sigma2, eps, cv_out, rgb_out);
    else k_denoise_step<GUIDE, false><<<grid, block, 0, s>>>(cv, guide, res_x, res_y, step, sigma2, eps, cv_out, rgb_out);
}

bool finite_positive(float v) { return v > 0.0f && v <= FLT_MAX; }

// YK_DENOISE_ON_DEVICE: an array must be device (or managed) memory of the current (the context's) device, 4-byte aligned
int check_device_array(const void* ptr, const char* name) {
    if (!ptr) return YK_OK;
    int dev = -1;
    DN_TRY(cudaGetDevice(&dev));
    cudaPointerAttributes a{};
    const cudaError_t e = cudaPointerGetAttributes(&a, ptr);
    if (e != cudaSuccess) (void)cudaGetLastError();
    if ((uintptr_t)ptr % 4u != 0 || e != cudaSuccess || (a.type != cudaMemoryTypeDevice && a.type != cudaMemoryTypeManaged) ||
        a.device != dev)
        return yk_set_error(YK_ERR_INVALID, std::string("yk_denoise: ") + name + " is not 4-byte aligned device memory of the context's GPU "
                                                "(device " + std::to_string(dev) + ") although YK_DENOISE_ON_DEVICE is set");
    return YK_OK;
}

// Work buffers from the device's stream-ordered pool (whose release threshold yk_context_create raises to "never", so a
// repeated call of the same size is a pool hit), returned to it on the same stream on every exit path.
struct StreamBuffers {
    cudaStream_t s;
    void* p[8] = {};
    int n = 0;
    explicit StreamBuffers(cudaStream_t st) : s(st) {}
    ~StreamBuffers() {
        for (int i = 0; i < n; ++i) cudaFreeAsync(p[i], s);
    }
    template <class T>
    cudaError_t alloc(T** out, size_t count) {
        void* q = nullptr;
        const cudaError_t e = cudaMallocAsync(&q, count * sizeof(T), s);
        if (e == cudaSuccess) p[n++] = q;
        *out = (T*)q;
        return e;
    }
};

}  // namespace

extern "C" int yk_denoise(yk_context* c, uint32_t res_x, uint32_t res_y, const float* film_rgb, const float* radiance_sq,
                          const yk_denoise_params* prm, float* out_rgb) {
    return yk_guard("yk_denoise", [&]() -> int {
    if (!c || !film_rgb || !radiance_sq || !out_rgb || !prm) return yk_set_error(YK_ERR_INVALID, "yk_denoise: null argument");
    if (!res_x || !res_y) return yk_set_error(YK_ERR_INVALID, "yk_denoise: zero resolution");
    if (prm->flags & ~YK_DENOISE_ON_DEVICE) return yk_set_error(YK_ERR_INVALID, "yk_denoise: unknown flags");
    if (prm->iterations < 1 || prm->iterations > kMaxIterations)
        return yk_set_error(YK_ERR_INVALID, "yk_denoise: iterations must be 1 ... 10, got " + std::to_string(prm->iterations));
    if (!finite_positive(prm->sigma) || !finite_positive(prm->eps))
        return yk_set_error(YK_ERR_INVALID, "yk_denoise: sigma and eps must be > 0 and finite");
    if (!prm->sample_counts && prm->samples_per_pixel < 2)
        return yk_set_error(YK_ERR_INVALID, "yk_denoise: without sample_counts, samples_per_pixel must be >= 2");
    std::lock_guard<std::recursive_mutex> guard(yk_context_mutex(c));
    if (int rc = yk_context_activate(c)) return rc;
    (void)cudaGetLastError();
    const bool on_device = prm->flags & YK_DENOISE_ON_DEVICE;
    if (on_device) {
        const std::pair<const void*, const char*> arrays[] = {{film_rgb, "film_rgb"}, {radiance_sq, "radiance_sq"}, {out_rgb, "out_rgb"},
                                                              {prm->sample_counts, "sample_counts"}, {prm->normals, "normals"}};
        for (const auto& a : arrays)
            if (int rc = check_device_array(a.first, a.second)) return rc;
    }
    cudaStream_t s = (cudaStream_t)yk_context_stream(c);
    if (on_device)
        if (int rc = yk_context_follow(c, prm->stream)) return rc;
    const size_t n = (size_t)res_x * res_y, rgb_bytes = n * 3 * sizeof(float);
    StreamBuffers buf(s);
    float4 *cv[2] = {nullptr, nullptr}, *guide = nullptr;
    DN_TRY(buf.alloc(&cv[0], n));
    if (prm->iterations > 1) DN_TRY(buf.alloc(&cv[1], n));
    DN_TRY(buf.alloc(&guide, n));
    const float *film = film_rgb, *sq = radiance_sq, *normals = prm->normals;
    const uint32_t* counts = prm->sample_counts;
    float* out = out_rgb;
    if (!on_device) {  // staged: the film's staging buffer also receives the output (k_denoise_setup has read it by then)
        float *d_film = nullptr, *d_sq = nullptr;
        DN_TRY(buf.alloc(&d_film, 3 * n));
        DN_TRY(buf.alloc(&d_sq, 3 * n));
        DN_TRY(cudaMemcpyAsync(d_film, film_rgb, rgb_bytes, cudaMemcpyHostToDevice, s));
        DN_TRY(cudaMemcpyAsync(d_sq, radiance_sq, rgb_bytes, cudaMemcpyHostToDevice, s));
        if (normals) {
            float* d_n = nullptr;
            DN_TRY(buf.alloc(&d_n, 3 * n));
            DN_TRY(cudaMemcpyAsync(d_n, prm->normals, rgb_bytes, cudaMemcpyHostToDevice, s));
            normals = d_n;
        }
        if (counts) {
            uint32_t* d_c = nullptr;
            DN_TRY(buf.alloc(&d_c, n));
            DN_TRY(cudaMemcpyAsync(d_c, prm->sample_counts, n * sizeof(uint32_t), cudaMemcpyHostToDevice, s));
            counts = d_c;
        }
        film = d_film;
        sq = d_sq;
        out = d_film;
    }
    int dev = 0, sms = 0;
    DN_TRY(cudaGetDevice(&dev));
    DN_TRY(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
    const unsigned setup_blocks = (unsigned)std::min<size_t>((n + 255) / 256, (size_t)sms * 16);
    k_denoise_setup<<<setup_blocks, 256, 0, s>>>(film, sq, counts, prm->samples_per_pixel, normals, n, cv[0], guide);
    DN_TRY(cudaGetLastError());
    const dim3 grid((res_x + kBlockX - 1) / kBlockX, (unsigned)std::min<uint32_t>((res_y + kBlockY - 1) / kBlockY, 65535u));
    const float sigma2 = prm->sigma * prm->sigma;
    for (uint32_t i = 0; i < prm->iterations; ++i) {
        const bool last = i + 1 == prm->iterations;
        const float4* in = cv[i & 1];
        float4* next = cv[(i + 1) & 1];
        // (a step beyond the film is allowed: every tap but the centre then falls outside and is skipped)
        const int step = 1 << i;
        if (normals) launch_step<true>(last, grid, s, in, guide, res_x, res_y, step, sigma2, prm->eps, next, out);
        else launch_step<false>(last, grid, s, in, guide, res_x, res_y, step, sigma2, prm->eps, next, out);
        DN_TRY(cudaGetLastError());
    }
    if (!on_device) DN_TRY(cudaMemcpyAsync(out_rgb, out, rgb_bytes, cudaMemcpyDeviceToHost, s));
    DN_TRY(cudaStreamSynchronize(s));
    return YK_OK;
    });
}
