// VM (3 planes x 3 lines) field: mip maintenance and the plain feature gather / scatter.
// Replaces the six nvdiffrast dr.texture calls per field query of the reference
// (network/fields.py:272-293, :786-806; network/flow.py:719-740).
#include <stdarg.h>
#include "common.cuh"
#include "internal.cuh"

// ---- error plumbing (thread-local; see include/tensoflow_b200.h) -------------
static thread_local char g_err[512] = "";
void tf_set_error(const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
}
extern "C" TF_API const char* tf_last_error(void) { return g_err; }
extern "C" TF_API int tf_abi_version(void) { return TF_ABI_VERSION; }

#include <atomic>
static std::atomic<long long> g_launches{0};
void tf_count_launches(int n) { g_launches.fetch_add(n, std::memory_order_relaxed); }
extern "C" TF_API long long tf_launch_count(void) { return g_launches.load(std::memory_order_relaxed); }

// ---- optional per-kernel timing (CUDA events on the launching stream; bench.py reads it for the roofline) ----
#include <map>
#include <mutex>
#include <string>
#include <vector>
namespace {
struct KernelEvents { std::vector<std::pair<cudaEvent_t, cudaEvent_t>> ev; };
std::mutex g_timing_mu;
std::map<std::string, KernelEvents> g_timing;
std::atomic<int> g_timing_on{0};
}  // namespace
TfKernelTimer::TfKernelTimer(const char* name, cudaStream_t stream) : name_(name), stream_(stream), start_(nullptr), stop_(nullptr) {
    if (!g_timing_on.load(std::memory_order_relaxed)) return;
    cudaEventCreate(&start_);
    cudaEventCreate(&stop_);
    cudaEventRecord(start_, stream_);
}
TfKernelTimer::~TfKernelTimer() {
    if (!start_) return;
    cudaEventRecord(stop_, stream_);
    std::lock_guard<std::mutex> lk(g_timing_mu);
    g_timing[name_].ev.emplace_back(start_, stop_);
}
extern "C" TF_API void tf_kernel_timing_enable(int32_t on) {
    g_timing_on.store(on ? 1 : 0);
    if (on) return;
}
extern "C" TF_API void tf_kernel_timing_reset(void) {
    std::lock_guard<std::mutex> lk(g_timing_mu);
    for (auto& kv : g_timing)
        for (auto& e : kv.second.ev) { cudaEventDestroy(e.first); cudaEventDestroy(e.second); }
    g_timing.clear();
}
extern "C" TF_API int tf_kernel_timing_read(const char* name, double* total_ms, int32_t* launches) {
    std::lock_guard<std::mutex> lk(g_timing_mu);
    auto it = g_timing.find(name ? name : "");
    *total_ms = 0.0; *launches = 0;
    if (it == g_timing.end()) return 1;
    for (auto& e : it->second.ev) {
        cudaEventSynchronize(e.second);
        float ms = 0.f;
        if (cudaEventElapsedTime(&ms, e.first, e.second) == cudaSuccess) { *total_ms += ms; *launches += 1; }
    }
    return 0;
}

int tf_check_field(const tf_vm_field_t* f, bool need_mips) {
    TF_REQUIRE(f != nullptr, "field descriptor is NULL");
    TF_REQUIRE(f->n_comp > 0 && f->n_comp % 4 == 0, "n_comp must be a positive multiple of 4 (got %d)", f->n_comp);
    TF_REQUIRE(f->n_levels >= 1 && f->n_levels <= 8, "n_levels out of range (%d)", f->n_levels);
    for (int i = 0; i < 3; ++i) {
        TF_REQUIRE(f->plane[i] && f->line[i], "plane/line %d is NULL", i);
        TF_REQUIRE(((uintptr_t)f->plane[i] & 15) == 0 && ((uintptr_t)f->line[i] & 15) == 0, "plane/line %d not 16-byte aligned", i);
        TF_REQUIRE(f->plane_h[i] > 0 && f->plane_w[i] > 0 && f->line_g[i] > 0, "bad extent on texture %d", i);
        if (f->n_levels > 1) {
            const int m = 1 << (f->n_levels - 1);
            TF_REQUIRE(f->plane_h[i] % m == 0 && f->plane_w[i] % m == 0 && f->line_g[i] % m == 0,
                       "extents of texture %d must be divisible by 2^(n_levels-1)", i);
            if (need_mips) TF_REQUIRE(f->plane_mip[i] && f->line_mip[i], "mip buffers of texture %d are NULL", i);
        }
        TF_REQUIRE(f->aabb_max[i] > f->aabb_min[i], "empty aabb on axis %d", i);
    }
    return 0;
}

// ---- mip build: dst[y][x][c] = mean of the 2x2 (or 2x1) block of src -------------
__global__ void mip_down_kernel(const float* __restrict__ src, float* __restrict__ dst, int Hd, int Wd, int Ws, int C4,
                                int halve_w) {
    const int64_t total = (int64_t)Hd * Wd * C4;
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
        const int c = (int)(i % C4);
        const int x = (int)((i / C4) % Wd);
        const int y = (int)(i / ((int64_t)C4 * Wd));
        const float4* s = reinterpret_cast<const float4*>(src);
        float4 r;
        if (halve_w) {
            float4 a = s[((size_t)(2 * y) * Ws + 2 * x) * C4 + c], b = s[((size_t)(2 * y) * Ws + 2 * x + 1) * C4 + c];
            float4 d = s[((size_t)(2 * y + 1) * Ws + 2 * x) * C4 + c], e = s[((size_t)(2 * y + 1) * Ws + 2 * x + 1) * C4 + c];
            r = make_float4(0.25f * (a.x + b.x + d.x + e.x), 0.25f * (a.y + b.y + d.y + e.y),
                            0.25f * (a.z + b.z + d.z + e.z), 0.25f * (a.w + b.w + d.w + e.w));
        } else {
            float4 a = s[((size_t)(2 * y) * Ws + x) * C4 + c], d = s[((size_t)(2 * y + 1) * Ws + x) * C4 + c];
            r = make_float4(0.5f * (a.x + d.x), 0.5f * (a.y + d.y), 0.5f * (a.z + d.z), 0.5f * (a.w + d.w));
        }
        reinterpret_cast<float4*>(dst)[i] = r;
    }
}

// ---- mip grad fold: fine[2y+dy][2x+dx] += w * coarse[y][x] --------------------------
__global__ void mip_fold_kernel(float* __restrict__ fine, const float* __restrict__ coarse, int Hf, int Wf, int Wc, int C4,
                                int halve_w) {
    const int64_t total = (int64_t)Hf * Wf * C4;
    const float w = halve_w ? 0.25f : 0.5f;
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
        const int c = (int)(i % C4);
        const int x = (int)((i / C4) % Wf);
        const int y = (int)(i / ((int64_t)C4 * Wf));
        const int xc = halve_w ? (x >> 1) : x;
        float4 g = reinterpret_cast<const float4*>(coarse)[((size_t)(y >> 1) * Wc + xc) * C4 + c];
        float4* d = reinterpret_cast<float4*>(fine) + i;
        float4 v = *d;
        v.x += w * g.x; v.y += w * g.y; v.z += w * g.z; v.w += w * g.w;
        *d = v;
    }
}

static inline int grid_for(int64_t total, int block) {
    int64_t g = (total + block - 1) / block;
    int64_t cap = (int64_t)tf_num_sms() * 16;
    return (int)(g < 1 ? 1 : (g > cap ? cap : g));
}

extern "C" TF_API int tf_vm_build_mips(const tf_vm_field_t* f, const tf_vm_mut_t* out, tf_stream_t stream_) {
    if (int e = tf_check_field(f, false)) return e;
    cudaStream_t stream = (cudaStream_t)stream_;
    if (f->n_levels == 1) return 0;
    TF_REQUIRE(out != nullptr, "mip output descriptor is NULL");
    const int C4 = f->n_comp / 4;
    for (int i = 0; i < 3; ++i) {
        TF_REQUIRE(out->plane_mip[i] && out->line_mip[i], "mip output %d is NULL", i);
        const float* src = f->plane[i];
        float* dst = out->plane_mip[i];
        int H = f->plane_h[i], W = f->plane_w[i];
        for (int l = 1; l < f->n_levels; ++l) {
            const int Hd = H >> 1, Wd = W >> 1;
            const int64_t total = (int64_t)Hd * Wd * C4;
            mip_down_kernel<<<grid_for(total, 256), 256, 0, stream>>>(src, dst, Hd, Wd, W, C4, 1);
            tf_count_launches(1);
            src = dst;
            dst += (size_t)Hd * Wd * f->n_comp;
            H = Hd; W = Wd;
        }
        src = f->line[i];
        dst = out->line_mip[i];
        int G = f->line_g[i];
        for (int l = 1; l < f->n_levels; ++l) {
            const int Gd = G >> 1;
            mip_down_kernel<<<grid_for((int64_t)Gd * C4, 256), 256, 0, stream>>>(src, dst, Gd, 1, 1, C4, 0);
            tf_count_launches(1);
            src = dst;
            dst += (size_t)Gd * f->n_comp;
            G = Gd;
        }
    }
    TF_CHECK_LAUNCH("tf_vm_build_mips");
    return 0;
}

extern "C" TF_API int tf_vm_fold_mip_grads(const tf_vm_field_t* f, const tf_vm_mut_t* g, tf_stream_t stream_) {
    if (int e = tf_check_field(f, false)) return e;
    cudaStream_t stream = (cudaStream_t)stream_;
    if (f->n_levels == 1) return 0;
    TF_REQUIRE(g != nullptr, "gradient descriptor is NULL");
    const int C = f->n_comp, C4 = C / 4;
    for (int i = 0; i < 3; ++i) {
        TF_REQUIRE(g->plane[i] && g->line[i] && g->plane_mip[i] && g->line_mip[i], "gradient buffer %d is NULL", i);
        // level pointers, coarse to fine
        float* lp[8]; int lh[8], lw[8];
        lp[0] = g->plane[i]; lh[0] = f->plane_h[i]; lw[0] = f->plane_w[i];
        float* p = g->plane_mip[i];
        for (int l = 1; l < f->n_levels; ++l) {
            lh[l] = lh[l - 1] >> 1; lw[l] = lw[l - 1] >> 1;
            lp[l] = p;
            p += (size_t)lh[l] * lw[l] * C;
        }
        for (int l = f->n_levels - 1; l >= 1; --l) {
            const int64_t total = (int64_t)lh[l - 1] * lw[l - 1] * C4;
            mip_fold_kernel<<<grid_for(total, 256), 256, 0, stream>>>(lp[l - 1], lp[l], lh[l - 1], lw[l - 1], lw[l], C4, 1);
            tf_count_launches(1);
        }
        float* q[8]; int qg[8];
        q[0] = g->line[i]; qg[0] = f->line_g[i];
        p = g->line_mip[i];
        for (int l = 1; l < f->n_levels; ++l) {
            qg[l] = qg[l - 1] >> 1;
            q[l] = p;
            p += (size_t)qg[l] * C;
        }
        for (int l = f->n_levels - 1; l >= 1; --l) {
            mip_fold_kernel<<<grid_for((int64_t)qg[l - 1] * C4, 256), 256, 0, stream>>>(q[l - 1], q[l], qg[l - 1], 1, 1, C4, 0);
            tf_count_launches(1);
        }
    }
    TF_CHECK_LAUNCH("tf_vm_fold_mip_grads");
    return 0;
}

// ---- plain feature gather: feat[n][i*C + c] = plane_i(x)[c] * line_i(x)[c] ----------
__global__ void __launch_bounds__(256) vm_feature_fwd_kernel(tf_vm_field_t f, const float* __restrict__ xyz,
                                                             const float* __restrict__ level, int64_t n,
                                                             float* __restrict__ feat) {
    const int C = f.n_comp, C4 = C / 4;
    const int64_t total = n * 3 * C4;
    for (int64_t it = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; it < total; it += (int64_t)gridDim.x * blockDim.x) {
        const int c = (int)(it % C4) * 4;
        const int i = (int)((it / C4) % 3);
        const int64_t r = it / (3 * C4);
        const float q[3] = {xyz[r * 3 + 0], xyz[r * 3 + 1], xyz[r * 3 + 2]};
        float4 P, L;
        vm_sample(f, q, level ? level[r] : 0.f, level != nullptr, i, c, P, L);
        *reinterpret_cast<float4*>(feat + r * (3 * C) + i * C + c) = f4_mul(P, L);
    }
}

__global__ void __launch_bounds__(256) vm_feature_bwd_kernel(tf_vm_field_t f, tf_vm_mut_t g, const float* __restrict__ xyz,
                                                             const float* __restrict__ level, int64_t n,
                                                             const float* __restrict__ d_feat) {
    const int C = f.n_comp, C4 = C / 4;
    const int64_t total = n * 3 * C4;
    for (int64_t it = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; it < total; it += (int64_t)gridDim.x * blockDim.x) {
        const int c = (int)(it % C4) * 4;
        const int i = (int)((it / C4) % 3);
        const int64_t r = it / (3 * C4);
        const float q[3] = {xyz[r * 3 + 0], xyz[r * 3 + 1], xyz[r * 3 + 2]};
        const float lv = level ? level[r] : 0.f;
        float4 P, L;
        vm_sample(f, q, lv, level != nullptr, i, c, P, L);
        const float4 d = *reinterpret_cast<const float4*>(d_feat + r * (3 * C) + i * C + c);
        vm_scatter(f, g, q, lv, level != nullptr, i, c, f4_mul(d, L), f4_mul(d, P));
    }
}

extern "C" TF_API int tf_vm_feature_fwd(const tf_vm_field_t* f, const float* xyz, const float* level, int64_t n, float* feat,
                                 tf_stream_t stream) {
    if (int e = tf_check_field(f, level != nullptr)) return e;
    if (n == 0) return 0;
    TF_REQUIRE(xyz && feat, "xyz/feat is NULL");
    TF_REQUIRE(((uintptr_t)feat & 15) == 0, "feat not 16-byte aligned");
    const int64_t total = n * 3 * (f->n_comp / 4);
    vm_feature_fwd_kernel<<<grid_for(total, 256), 256, 0, (cudaStream_t)stream>>>(*f, xyz, level, n, feat);
    tf_count_launches(1);
    TF_CHECK_LAUNCH("tf_vm_feature_fwd");
    return 0;
}

extern "C" TF_API int tf_vm_feature_bwd(const tf_vm_field_t* f, const float* xyz, const float* level, int64_t n,
                                 const float* d_feat, const tf_vm_mut_t* g, tf_stream_t stream) {
    if (int e = tf_check_field(f, level != nullptr)) return e;
    if (n == 0) return 0;
    TF_REQUIRE(xyz && d_feat && g, "xyz/d_feat/grad descriptor is NULL");
    for (int i = 0; i < 3; ++i) {
        TF_REQUIRE(g->plane[i] && g->line[i], "gradient buffer %d is NULL", i);
        if (f->n_levels > 1 && level) TF_REQUIRE(g->plane_mip[i] && g->line_mip[i], "mip gradient buffer %d is NULL", i);
    }
    const int64_t total = n * 3 * (f->n_comp / 4);
    vm_feature_bwd_kernel<<<grid_for(total, 256), 256, 0, (cudaStream_t)stream>>>(*f, *g, xyz, level, n, d_feat);
    tf_count_launches(1);
    TF_CHECK_LAUNCH("tf_vm_feature_bwd");
    return 0;
}
