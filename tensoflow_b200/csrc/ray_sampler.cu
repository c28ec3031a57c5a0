// Hierarchical NeuS ray sampler of the shape stage (reference network/shapeRenderer.py:820-932: sample_ray / upsample /
// cat_z_vals; utils/network_utils.py:117-147: sample_pdf with det=True) as four small kernels around the SDF-only field
// queries, replacing the sort / searchsorted / cumprod / gather tensor arithmetic of the reference:
//   sampler_init     : thread per (ray, coarse sample): box clipping of [near, far], stratified depths, query points + mip levels
//   sampler_upsample : warp per ray: [merge the previous round's samples into the sorted list] -> NeuS section alphas ->
//                      transmittance prefix product (warp scan) -> pdf / cdf -> inverse-CDF samples -> their query points
//   sampler_merge    : warp per ray: the last merge (the reference skips the SDF of the last round)
//   sampler_finalize : warp per ray: interval ends, mid points, inside-box mask -> per-ray counts, then (second call) the
//                      packed t_starts / t_ends / ray_indices in ray order
// Depth lists live in [R, S_max] rows (first n valid), ascending after every merge.  Before the first merge a ray that misses
// the box holds a descending coarse list (tmin > tmax after the [near, far] clip), as the reference does; round 0 upsamples
// it in that order.  HBM-bound: ~ (8 n + 100) B per ray and round.
#include "common.cuh"

namespace {

constexpr int SMAX = 256;          // capacity of a ray's depth list (n_samples + n_importance <= 256)
constexpr int WARPS = 4;           // warps (= rays) per CTA

__device__ __forceinline__ float sigmoidf_(float x) { return 1.f / (1.f + expf(-x)); }

// compute_ball_radii (shapeRenderer.py:966-970) and the mip level log2(ball / base_radii)
__device__ __forceinline__ float mip_level(float z, float radii, float cosv, float base_radii) {
    const float inv_cos = 1.f / cosv;
    const float tmp = sqrtf(inv_cos * inv_cos - 1.f) - radii;
    const float ball = z * radii * cosv / sqrtf(tmp * tmp + 1.f);
    return log2f(ball / base_radii);
}

struct InitParams {
    const float* rays_o; const float* dirs; const float* near; const float* far; const float* radiis; const float* rays_cos;
    const float* lin;            // torch.linspace(0, 1, n_samples)
    const float* t_rand;         // [R] or NULL (no perturbation)
    float aabb[6]; float base_radii;
    int R, n, stride;
    float* z; float* pts; float* level;
};

__global__ void __launch_bounds__(256) sampler_init_kernel(InitParams p) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= (int64_t)p.R * p.n) return;
    const int r = (int)(i / p.n), j = (int)(i % p.n);
    float o[3], d[3];
    float tmin = -INFINITY, tmax = INFINITY;
#pragma unroll
    for (int k = 0; k < 3; ++k) {
        o[k] = p.rays_o[r * 3 + k]; d[k] = p.dirs[r * 3 + k];
        const float vec = d[k] == 0.f ? 1e-6f : d[k];
        const float ra = (p.aabb[3 + k] - o[k]) / vec, rb = (p.aabb[k] - o[k]) / vec;
        tmin = fmaxf(tmin, fminf(ra, rb));
        tmax = fminf(tmax, fmaxf(ra, rb));
    }
    const float nr = p.near[r], fr = p.far[r];
    tmin = fminf(fmaxf(tmin, nr), fr);
    tmax = fminf(fmaxf(tmax, nr), fr);
    float z = tmin + (tmax - tmin) * p.lin[j];
    if (p.t_rand) z = z + (p.t_rand[r] - 0.5f) * 2.0f / (float)p.n;
    p.z[(size_t)r * p.stride + j] = z;
    p.pts[i * 3 + 0] = o[0] + d[0] * z; p.pts[i * 3 + 1] = o[1] + d[1] * z; p.pts[i * 3 + 2] = o[2] + d[2] * z;
    p.level[i] = mip_level(z, p.radiis[r], p.rays_cos[r], p.base_radii);
}

// ---- merge of two monotone lists held in shared memory into one ascending list (stable: ties keep the old sample first) --
// zs / ss [0, n) old, zn / sn [0, m) new -> out_z / out_s [0, n + m), n >= 1, m >= 1.  Each input may ascend or descend
// (first > last): a ray that misses the box has tmin > tmax once both are clipped to [near, far], so its coarse list
// descends, and so do the importance samples drawn from it in round 0.  A descending list is read from its end; the
// output is what torch.sort gives the reference.
__device__ __forceinline__ void warp_merge(const float* zs, const float* ss, int n, const float* zn, const float* sn, int m, float* out_z,
                                           float* out_s, int lane) {
    const bool old_desc = zs[0] > zs[n - 1], new_desc = zn[0] > zn[m - 1];
    auto old_at = [&](int k) { return old_desc ? n - 1 - k : k; };       // storage index of the k-th smallest
    auto new_at = [&](int j) { return new_desc ? m - 1 - j : j; };
    for (int k = lane; k < n; k += 32) {
        const int i = old_at(k);
        const float v = zs[i];
        int lo = 0, hi = m;                       // #(new < v)
        while (lo < hi) { const int mid = (lo + hi) >> 1; if (zn[new_at(mid)] < v) lo = mid + 1; else hi = mid; }
        out_z[k + lo] = v;
        if (out_s) out_s[k + lo] = ss[i];
    }
    for (int j = lane; j < m; j += 32) {
        const int i = new_at(j);
        const float v = zn[i];
        int lo = 0, hi = n;                       // #(old <= v)
        while (lo < hi) { const int mid = (lo + hi) >> 1; if (zs[old_at(mid)] <= v) lo = mid + 1; else hi = mid; }
        out_z[j + lo] = v;
        if (out_s) out_s[j + lo] = sn ? sn[i] : 0.f;
    }
}

struct UpParams {
    const float* rays_o; const float* dirs; const float* radiis; const float* rays_cos;
    float* z; float* sdf;        // [R, stride] lists (n valid), updated in place by the merge (ascending afterwards)
    const float* new_z_in;       // [R, m_in] samples of the previous round (NULL: nothing to merge)
    const float* new_sdf_in;     // [R * m_in] their SDF values
    const float* u;              // [m] = linspace(0.5/m, 1-0.5/m, m)
    const float* variance;       // device scalar (inv_s = exp(10 variance), clipped) or NULL
    float inv_s_cap, base_radii;
    int R, n, m_in, m, stride;
    float* new_z; float* new_pts; float* new_level;    // [R, m], [R*m, 3], [R*m]
};

__global__ void __launch_bounds__(32 * WARPS) sampler_upsample_kernel(UpParams p) {
    __shared__ float s_z[WARPS][SMAX], s_s[WARPS][SMAX], s_a[WARPS][SMAX], s_b[WARPS][SMAX];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int r = blockIdx.x * WARPS + warp;
    if (r >= p.R) return;
    float* zs = s_z[warp]; float* ss = s_s[warp]; float* ta = s_a[warp]; float* tb = s_b[warp];
    int n = p.n;
    // ---- sorted list of the ray (merging the previous round first: cat_z_vals, shapeRenderer.py:851-869) ----------
    if (p.new_z_in) {
        for (int k = lane; k < n; k += 32) { ta[k] = p.z[(size_t)r * p.stride + k]; tb[k] = p.sdf[(size_t)r * p.stride + k]; }
        float* nz = ta + n; float* ns = tb + n;         // the tails of the scratch rows hold the new samples
        for (int j = lane; j < p.m_in; j += 32) { nz[j] = p.new_z_in[(size_t)r * p.m_in + j]; ns[j] = p.new_sdf_in ? p.new_sdf_in[(size_t)r * p.m_in + j] : 0.f; }
        __syncwarp();
        warp_merge(ta, tb, n, nz, ns, p.m_in, zs, ss, lane);
        n += p.m_in;
        __syncwarp();
        for (int k = lane; k < n; k += 32) { p.z[(size_t)r * p.stride + k] = zs[k]; p.sdf[(size_t)r * p.stride + k] = ss[k]; }
    } else {
        for (int k = lane; k < n; k += 32) { zs[k] = p.z[(size_t)r * p.stride + k]; ss[k] = p.sdf[(size_t)r * p.stride + k]; }
    }
    __syncwarp();
    if (p.m == 0) return;
    // ---- NeuS section alphas of the n - 1 intervals (upsample, shapeRenderer.py:822-849) ----------------------------
    const float o0 = p.rays_o[r * 3], o1 = p.rays_o[r * 3 + 1], o2 = p.rays_o[r * 3 + 2];
    const float d0 = p.dirs[r * 3], d1 = p.dirs[r * 3 + 1], d2 = p.dirs[r * 3 + 2];
    float inv_s = p.inv_s_cap;
    if (p.variance) inv_s = fminf(expf(__ldg(p.variance) * 10.f), p.inv_s_cap);
    const int ni = n - 1;
    auto radius = [&](int k) {
        const float x = o0 + d0 * zs[k], y = o1 + d1 * zs[k], w = o2 + d2 * zs[k];
        return sqrtf(x * x + y * y + w * w);
    };
    auto raw_cos = [&](int k) { return (ss[k + 1] - ss[k]) / (zs[k + 1] - zs[k] + 1e-5f); };
    for (int k = lane; k < ni; k += 32) {
        const bool inside = (radius(k) < 1.0f) || (radius(k + 1) < 1.0f);
        const float mid = (ss[k] + ss[k + 1]) * 0.5f;
        const float c = raw_cos(k), pc = k == 0 ? 0.f : raw_cos(k - 1);
        float cv = fminf(pc, c);
        cv = fminf(fmaxf(cv, -1e3f), 0.0f) * (inside ? 1.f : 0.f);
        const float dist = zs[k + 1] - zs[k];
        const float prev_cdf = sigmoidf_((mid - cv * dist * 0.5f) * inv_s), next_cdf = sigmoidf_((mid + cv * dist * 0.5f) * inv_s);
        ta[k] = (prev_cdf - next_cdf + 1e-5f) / (prev_cdf + 1e-5f);          // alpha
    }
    __syncwarp();
    // ---- weights = alpha * exclusive cumprod(1 - alpha + 1e-7); blocked over the lanes + warp scan ---------------------
    const int per = (ni + 31) / 32;
    const int k0 = lane * per, k1 = min(k0 + per, ni);
    float prod = 1.f;
    for (int k = k0; k < k1; ++k) prod *= (1.f - ta[k] + 1e-7f);
    float excl = prod;                                   // inclusive scan of the lane products
#pragma unroll
    for (int off = 1; off < 32; off <<= 1) {
        const float t = __shfl_up_sync(0xffffffffu, excl, off);
        if (lane >= off) excl *= t;
    }
    excl = __shfl_up_sync(0xffffffffu, excl, 1);
    if (lane == 0) excl = 1.f;
    float wsum = 0.f;
    {
        float T = excl;
        for (int k = k0; k < k1; ++k) {
            const float w = ta[k] * T + 1e-5f;          // sample_pdf: weights + 1e-5
            T *= (1.f - ta[k] + 1e-7f);
            tb[k] = w;
            wsum += w;
        }
    }
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) wsum += __shfl_xor_sync(0xffffffffu, wsum, off);
    // ---- cdf = [0, cumsum(w / sum)] (length n) ------------------------------------------------------------------------------
    float part = 0.f;
    for (int k = k0; k < k1; ++k) part += tb[k] / wsum;
    float incl = part;
#pragma unroll
    for (int off = 1; off < 32; off <<= 1) {
        const float t = __shfl_up_sync(0xffffffffu, incl, off);
        if (lane >= off) incl += t;
    }
    float run = incl - part;
    __syncwarp();
    for (int k = k0; k < k1; ++k) { run += tb[k] / wsum; ta[k + 1] = run; }     // ta becomes the cdf (alpha no longer needed)
    if (lane == 0) ta[0] = 0.f;
    __syncwarp();
    // ---- inverse CDF at the m fixed quantiles (sample_pdf, det=True) -----------------------------------------------------
    for (int j = lane; j < p.m; j += 32) {
        const float u = p.u[j];
        int lo = 0, hi = n;                              // searchsorted(cdf, u, right=True) = #(cdf <= u)
        while (lo < hi) { const int mid = (lo + hi) >> 1; if (ta[mid] <= u) lo = mid + 1; else hi = mid; }
        const int below = max(lo - 1, 0), above = min(lo, n - 1);
        float denom = ta[above] - ta[below];
        if (denom < 1e-5f) denom = 1.f;
        const float t = (u - ta[below]) / denom;
        const float z = zs[below] + t * (zs[above] - zs[below]);
        const size_t q = (size_t)r * p.m + j;
        p.new_z[q] = z;
        p.new_pts[q * 3 + 0] = o0 + d0 * z; p.new_pts[q * 3 + 1] = o1 + d1 * z; p.new_pts[q * 3 + 2] = o2 + d2 * z;
        p.new_level[q] = mip_level(z, p.radiis[r], p.rays_cos[r], p.base_radii);
    }
}

struct FinalParams {
    const float* rays_o; const float* dirs;
    const float* z;              // [R, stride], n valid
    float aabb[6];
    int R, n, stride;
    int32_t* counts;             // [R] (count pass)
    const int64_t* offsets;      // [R + 1] exclusive prefix sums (write pass)
    float* t_starts; float* t_ends; int64_t* ray_indices;
};

template <bool WRITE>
__global__ void __launch_bounds__(32 * WARPS) sampler_finalize_kernel(FinalParams p) {
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int r = blockIdx.x * WARPS + warp;
    if (r >= p.R) return;
    const float* z = p.z + (size_t)r * p.stride;
    const float o0 = p.rays_o[r * 3], o1 = p.rays_o[r * 3 + 1], o2 = p.rays_o[r * 3 + 2];
    const float d0 = p.dirs[r * 3], d1 = p.dirs[r * 3 + 1], d2 = p.dirs[r * 3 + 2];
    const int n = p.n;
    int64_t base = WRITE ? p.offsets[r] : 0;
    int total = 0;
    for (int k0 = 0; k0 < n; k0 += 32) {
        const int k = k0 + lane;
        bool inner = false;
        float zk = 0.f, dist = 0.f;
        if (k < n) {
            zk = z[k];
            dist = k + 1 < n ? z[k + 1] - zk : (n >= 2 ? z[n - 1] - z[n - 2] : 0.f);       // last interval repeats the previous one
            const float mid = zk + dist * 0.5f;
            const float x = o0 + d0 * mid, y = o1 + d1 * mid, w = o2 + d2 * mid;
            inner = !((p.aabb[0] > x) || (x > p.aabb[3]) || (p.aabb[1] > y) || (y > p.aabb[4]) || (p.aabb[2] > w) || (w > p.aabb[5]));
        }
        const unsigned m = __ballot_sync(0xffffffffu, inner);
        if (WRITE && inner) {
            const int64_t q = base + __popc(m & ((1u << lane) - 1u));
            p.t_starts[q] = zk; p.t_ends[q] = zk + dist; p.ray_indices[q] = r;
        }
        base += __popc(m);
        total += __popc(m);
    }
    if (!WRITE && lane == 0) p.counts[r] = total;
}

// ---- secondary-ray probes (reference utils/network_utils.py:149-202 get_weights / get_intersection and
// ---- network/materialRenderer.py:281-313 get_intersection_around_mesh): NeuS weights of a short depth list, either
// ---- resampled at fixed quantiles (first stage) or returned with the section mid points and SDF (second stage)
struct ProbeInitParams {
    const float* o; const float* d; const float* t0; const float* t1; const float* lin;
    int pn, sn; float* z; float* pts;
};
__global__ void __launch_bounds__(256) probe_init_kernel(ProbeInitParams p) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= (int64_t)p.pn * p.sn) return;
    const int r = (int)(i / p.sn), j = (int)(i % p.sn);
    const float a = p.t0 ? p.t0[r] : 0.f, b = p.t1[r];
    const float z = p.t0 ? a + (b - a) * p.lin[j] : b * p.lin[j];
    p.z[i] = z;
#pragma unroll
    for (int k = 0; k < 3; ++k) p.pts[i * 3 + k] = z * p.d[r * 3 + k] + p.o[r * 3 + k];
}

struct ProbeParams {
    const float* o; const float* d; const float* z; const float* sdf; const float* variance; const float* u;
    int pn, sn, m;
    float* new_z; float* new_pts;                       // m > 0
    float* weights; float* mid_sdf; float* z_mid;       // m == 0
};
__global__ void __launch_bounds__(32 * WARPS) probe_weights_kernel(ProbeParams p) {
    __shared__ float s_z[WARPS][SMAX], s_s[WARPS][SMAX], s_a[WARPS][SMAX], s_b[WARPS][SMAX];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int r = blockIdx.x * WARPS + warp;
    if (r >= p.pn) return;
    float* zs = s_z[warp]; float* ss = s_s[warp]; float* ta = s_a[warp]; float* tb = s_b[warp];
    const int n = p.sn, ni = n - 1;
    for (int k = lane; k < n; k += 32) { zs[k] = p.z[(size_t)r * n + k]; ss[k] = p.sdf[(size_t)r * n + k]; }
    __syncwarp();
    const float inv_s = expf(__ldg(p.variance) * 10.f);
    for (int k = lane; k < ni; k += 32) {
        const float mid = (ss[k] + ss[k + 1]) * 0.5f;
        float cv = (ss[k + 1] - ss[k]) / (zs[k + 1] - zs[k] + 1e-5f);
        const bool surface = cv < 0.f;
        cv = fminf(cv, 0.f);
        const float dist = zs[k + 1] - zs[k];
        const float prev_cdf = sigmoidf_((mid - cv * dist * 0.5f) * inv_s), next_cdf = sigmoidf_((mid + cv * dist * 0.5f) * inv_s);
        ta[k] = (prev_cdf - next_cdf + 1e-5f) / (prev_cdf + 1e-5f) * (surface ? 1.f : 0.f);
        if (p.m == 0) {
            p.mid_sdf[(size_t)r * ni + k] = surface ? mid : -1.0f;
            p.z_mid[(size_t)r * ni + k] = (zs[k + 1] + zs[k]) * 0.5f;
        }
    }
    __syncwarp();
    const int per = (ni + 31) / 32;
    const int k0 = lane * per, k1 = min(k0 + per, ni);
    float prod = 1.f;
    for (int k = k0; k < k1; ++k) prod *= (1.f - ta[k] + 1e-7f);
    float excl = prod;
#pragma unroll
    for (int off = 1; off < 32; off <<= 1) {
        const float t = __shfl_up_sync(0xffffffffu, excl, off);
        if (lane >= off) excl *= t;
    }
    excl = __shfl_up_sync(0xffffffffu, excl, 1);
    if (lane == 0) excl = 1.f;
    float wsum = 0.f;
    {
        float T = excl;
        for (int k = k0; k < k1; ++k) {
            const float w = ta[k] * T;
            T *= (1.f - ta[k] + 1e-7f);
            if (p.m == 0) p.weights[(size_t)r * ni + k] = w;
            tb[k] = w + 1e-5f;
            wsum += w + 1e-5f;
        }
    }
    if (p.m == 0) return;
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) wsum += __shfl_xor_sync(0xffffffffu, wsum, off);
    float part = 0.f;
    for (int k = k0; k < k1; ++k) part += tb[k] / wsum;
    float incl = part;
#pragma unroll
    for (int off = 1; off < 32; off <<= 1) {
        const float t = __shfl_up_sync(0xffffffffu, incl, off);
        if (lane >= off) incl += t;
    }
    float run = incl - part;
    __syncwarp();
    for (int k = k0; k < k1; ++k) { run += tb[k] / wsum; ta[k + 1] = run; }
    if (lane == 0) ta[0] = 0.f;
    __syncwarp();
    for (int j = lane; j < p.m; j += 32) {
        const float u = p.u[j];
        int lo = 0, hi = n;
        while (lo < hi) { const int mid = (lo + hi) >> 1; if (ta[mid] <= u) lo = mid + 1; else hi = mid; }
        const int below = max(lo - 1, 0), above = min(lo, n - 1);
        float denom = ta[above] - ta[below];
        if (denom < 1e-5f) denom = 1.f;
        const float t = (u - ta[below]) / denom;
        const float z = zs[below] + t * (zs[above] - zs[below]);
        const size_t q = (size_t)r * p.m + j;
        p.new_z[q] = z;
#pragma unroll
        for (int k = 0; k < 3; ++k) p.new_pts[q * 3 + k] = z * p.d[r * 3 + k] + p.o[r * 3 + k];
    }
}

int check_common(const void* a, const void* b, int R, int n, int stride) {
    TF_REQUIRE(a && b, "ray sampler: NULL pointer");
    TF_REQUIRE(R >= 0 && n >= 2 && n <= stride && stride <= SMAX, "ray sampler: 2 <= n <= stride <= %d required (n=%d, stride=%d)", SMAX, n, stride);
    return 0;
}

}  // namespace

extern "C" TF_API int tf_sampler_init(const float* rays_o, const float* dirs, const float* near, const float* far, const float* radiis,
                                      const float* rays_cos, const float* lin, const float* t_rand, const float aabb[6], float base_radii,
                                      int32_t R, int32_t n, int32_t stride, float* z, float* pts, float* level, tf_stream_t stream) {
    if (int e = check_common(rays_o, dirs, R, n, stride)) return e;
    TF_REQUIRE(near && far && radiis && rays_cos && lin && aabb && z && pts && level, "tf_sampler_init: NULL pointer");
    if (R == 0) return 0;
    InitParams p = {rays_o, dirs, near, far, radiis, rays_cos, lin, t_rand, {aabb[0], aabb[1], aabb[2], aabb[3], aabb[4], aabb[5]}, base_radii,
                    R, n, stride, z, pts, level};
    const int64_t total = (int64_t)R * n;
    sampler_init_kernel<<<(unsigned)((total + 255) / 256), 256, 0, (cudaStream_t)stream>>>(p);
    tf_count_launches(1);
    TF_CHECK_LAUNCH("tf_sampler_init");
    return 0;
}

extern "C" TF_API int tf_sampler_upsample(const float* rays_o, const float* dirs, const float* radiis, const float* rays_cos, float* z, float* sdf,
                                          const float* new_z_in, const float* new_sdf_in, int32_t m_in, const float* u, int32_t m,
                                          const float* variance, float inv_s_cap, float base_radii, int32_t R, int32_t n, int32_t stride,
                                          float* new_z, float* new_pts, float* new_level, tf_stream_t stream) {
    if (int e = check_common(rays_o, dirs, R, n, stride)) return e;
    TF_REQUIRE(z && sdf && radiis && rays_cos, "tf_sampler_upsample: NULL pointer");
    TF_REQUIRE(m >= 0 && m_in >= 0 && n + m_in <= stride, "tf_sampler_upsample: n + m_in must fit the row stride");
    TF_REQUIRE(!new_z_in || (new_sdf_in || m == 0), "tf_sampler_upsample: merged samples need their SDF values before another round");
    TF_REQUIRE(m == 0 || (u && new_z && new_pts && new_level), "tf_sampler_upsample: NULL output pointer");
    if (R == 0) return 0;
    UpParams p = {rays_o, dirs, radiis, rays_cos, z, sdf, m_in > 0 ? new_z_in : nullptr, new_sdf_in, u, variance, inv_s_cap, base_radii,
                  R, n, m_in, m, stride, new_z, new_pts, new_level};
    // m == 0 with new_sdf_in == NULL is the last merge (the reference skips the SDF of the last round: cat_z_vals(last=True)):
    // the merged SDF entries of those samples are zero-filled and nobody reads them afterwards
    sampler_upsample_kernel<<<(unsigned)((R + WARPS - 1) / WARPS), 32 * WARPS, 0, (cudaStream_t)stream>>>(p);
    tf_count_launches(1);
    TF_CHECK_LAUNCH("tf_sampler_upsample");
    return 0;
}

extern "C" TF_API int tf_sampler_finalize(const float* rays_o, const float* dirs, const float* z, const float aabb[6], int32_t R, int32_t n,
                                          int32_t stride, int32_t* counts, const int64_t* offsets, float* t_starts, float* t_ends,
                                          int64_t* ray_indices, tf_stream_t stream) {
    if (int e = check_common(rays_o, dirs, R, n, stride)) return e;
    TF_REQUIRE(z && aabb, "tf_sampler_finalize: NULL pointer");
    TF_REQUIRE((counts != nullptr) != (offsets != nullptr), "tf_sampler_finalize: pass counts (count pass) or offsets (write pass)");
    if (R == 0) return 0;
    FinalParams p = {rays_o, dirs, z, {aabb[0], aabb[1], aabb[2], aabb[3], aabb[4], aabb[5]}, R, n, stride, counts, offsets, t_starts, t_ends,
                     ray_indices};
    const unsigned grid = (unsigned)((R + WARPS - 1) / WARPS);
    if (counts) {
        sampler_finalize_kernel<false><<<grid, 32 * WARPS, 0, (cudaStream_t)stream>>>(p);
    } else {
        TF_REQUIRE(t_starts && t_ends && ray_indices, "tf_sampler_finalize: NULL output pointer");
        sampler_finalize_kernel<true><<<grid, 32 * WARPS, 0, (cudaStream_t)stream>>>(p);
    }
    tf_count_launches(1);
    TF_CHECK_LAUNCH("tf_sampler_finalize");
    return 0;
}

extern "C" TF_API int tf_probe_init(const float* origins, const float* dirs, const float* t0, const float* t1, const float* lin, int32_t pn,
                                    int32_t sn, float* z, float* pts, tf_stream_t stream) {
    TF_REQUIRE(origins && dirs && t1 && lin && z && pts, "tf_probe_init: NULL pointer");
    TF_REQUIRE(pn >= 0 && sn >= 2 && sn <= SMAX, "tf_probe_init: 2 <= sn <= %d required", SMAX);
    if (pn == 0) return 0;
    ProbeInitParams p = {origins, dirs, t0, t1, lin, pn, sn, z, pts};
    const int64_t total = (int64_t)pn * sn;
    probe_init_kernel<<<(unsigned)((total + 255) / 256), 256, 0, (cudaStream_t)stream>>>(p);
    tf_count_launches(1);
    TF_CHECK_LAUNCH("tf_probe_init");
    return 0;
}

extern "C" TF_API int tf_probe_weights(const float* origins, const float* dirs, const float* z, const float* sdf, const float* variance,
                                       int32_t pn, int32_t sn, const float* u, int32_t m, float* new_z, float* new_pts, float* weights,
                                       float* mid_sdf, float* z_mid, tf_stream_t stream) {
    TF_REQUIRE(origins && dirs && z && sdf && variance, "tf_probe_weights: NULL pointer");
    TF_REQUIRE(pn >= 0 && sn >= 2 && sn <= SMAX && m >= 0, "tf_probe_weights: 2 <= sn <= %d required", SMAX);
    TF_REQUIRE(m > 0 ? (u && new_z && new_pts) : (weights && mid_sdf && z_mid), "tf_probe_weights: NULL output pointer");
    if (pn == 0) return 0;
    ProbeParams p = {origins, dirs, z, sdf, variance, u, pn, sn, m, new_z, new_pts, weights, mid_sdf, z_mid};
    probe_weights_kernel<<<(unsigned)((pn + WARPS - 1) / WARPS), 32 * WARPS, 0, (cudaStream_t)stream>>>(p);
    tf_count_launches(1);
    TF_CHECK_LAUNCH("tf_probe_weights");
    return 0;
}
