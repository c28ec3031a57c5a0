// Seamless (tri)linear cubemap lookup, differentiable in the textures, the direction and the mip level: the
// `dr.texture(..., boundary_mode='cube')` calls of the shape-stage split-sum light (reference network/light.py:95-122:
// diffuse lookup at the normal, specular lookup at the reflected direction with `mip_level_bias` from the roughness over the
// user-supplied prefiltered stack).  One thread per sample:
//   forward   out = (1-f) S_l0(d) + f S_l1(d),  lv = clamp(level, 0, L-1), l0 = floor(lv), f = lv - l0, l1 = min(l0+1, L-1)
//             S_l(d) = sum_k w_k T_l[idx_k] / sum_k w_k over the 4 bilinear taps of the face footprint; taps that leave the face
//             fold onto the neighbouring face, the tap leaving in both axes (cube corner) is dropped
//   backward  d T_l[idx_k] += g w_k / W  (atomics; the textures are <= 128^2 x 6 texels: L2 resident)
//             d d       through the bilinear fractions (d S / d fu = sum_k dw_k/dfu (T_k - S) / W), u = (x/m + 1) R/2 - 1/2
//             d level   = g . (S_l1 - S_l0) inside the clamp range
// In round 1 this was ~150 tensor ops per lookup and level (about 3000 launches per ShapeRenderer step).
#include "shading.cuh"

namespace {

constexpr int CS_MAX_LEVELS = 8;

struct CubeStack {
    const float* tex[CS_MAX_LEVELS];
    float* d_tex[CS_MAX_LEVELS];
    int res[CS_MAX_LEVELS];
    int n;
};

__device__ __forceinline__ void cs_levels(const float* level, int64_t i, int n, int& l0, int& l1, float& f, bool& inside) {
    l0 = 0; l1 = 0; f = 0.f; inside = false;
    if (!level || n <= 1) return;
    const float raw = level[i];
    const float lv = fminf(fmaxf(raw, 0.f), (float)(n - 1));
    inside = raw >= 0.f && raw <= (float)(n - 1);
    const float fl = floorf(lv);
    l0 = (int)fl;
    f = lv - fl;
    l1 = min(l0 + 1, n - 1);
}

__device__ __forceinline__ void cs_fetch(const float* tex, const CubeTaps& t, float s[3]) {
    s[0] = s[1] = s[2] = 0.f;
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        const float* px = tex + (size_t)t.idx[k] * 3;
        s[0] = fmaf(t.w[k], __ldg(px), s[0]); s[1] = fmaf(t.w[k], __ldg(px + 1), s[1]); s[2] = fmaf(t.w[k], __ldg(px + 2), s[2]);
    }
    const float inv = 1.f / t.wsum;
    s[0] *= inv; s[1] *= inv; s[2] *= inv;
}

__global__ void __launch_bounds__(256) cube_sample_fwd_kernel(const CubeStack st, const float* __restrict__ dirs,
                                                              const float* __restrict__ level, int64_t n, float* __restrict__ out) {
    const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (i >= n) return;
    const float d[3] = {dirs[i * 3], dirs[i * 3 + 1], dirs[i * 3 + 2]};
    const CubeFace fm = cube_face(d);
    int l0, l1; float f; bool inside;
    cs_levels(level, i, st.n, l0, l1, f, inside);
    float s0[3];
    cs_fetch(st.tex[l0], cube_taps(fm, st.res[l0]), s0);
    if (l1 != l0 && f != 0.f) {
        float s1[3];
        cs_fetch(st.tex[l1], cube_taps(fm, st.res[l1]), s1);
#pragma unroll
        for (int c = 0; c < 3; ++c) s0[c] = (1.f - f) * s0[c] + f * s1[c];
    }
    out[i * 3] = s0[0]; out[i * 3 + 1] = s0[1]; out[i * 3 + 2] = s0[2];
}

// adjoint of one level's lookup: scatters g * scale into d_tex, returns S and accumulates (dS/dx, dS/dy) . g * scale
__device__ __forceinline__ void cs_level_bwd(const float* tex, float* d_tex, const CubeFace& fm, int R, const float g[3], float scale,
                                             float s[3], float& gx, float& gy) {
    const CubeTaps t = cube_taps(fm, R);
    cs_fetch(tex, t, s);
    const float inv = 1.f / t.wsum;
    float gu = 0.f, gv = 0.f;
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        const float* px = tex + (size_t)t.idx[k] * 3;
        const float dot = g[0] * (__ldg(px) - s[0]) + g[1] * (__ldg(px + 1) - s[1]) + g[2] * (__ldg(px + 2) - s[2]);
        gu = fmaf(t.dwu[k], dot, gu);
        gv = fmaf(t.dwv[k], dot, gv);
        if (d_tex && t.w[k] != 0.f && scale != 0.f) {
            const float w = t.w[k] * inv * scale;
            float* q = d_tex + (size_t)t.idx[k] * 3;
            atomicAdd(q, w * g[0]); atomicAdd(q + 1, w * g[1]); atomicAdd(q + 2, w * g[2]);
        }
    }
    // d fu / d x = R / 2
    gx += gu * inv * scale * 0.5f * R;
    gy += gv * inv * scale * 0.5f * R;
}

__global__ void __launch_bounds__(256) cube_sample_bwd_kernel(const CubeStack st, const float* __restrict__ dirs,
                                                              const float* __restrict__ level, int64_t n, const float* __restrict__ g_out,
                                                              float* __restrict__ d_dirs, float* __restrict__ d_level) {
    const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (i >= n) return;
    const float d[3] = {dirs[i * 3], dirs[i * 3 + 1], dirs[i * 3 + 2]};
    const float g[3] = {g_out[i * 3], g_out[i * 3 + 1], g_out[i * 3 + 2]};
    const CubeFace fm = cube_face(d);
    int l0, l1; float f; bool inside;
    cs_levels(level, i, st.n, l0, l1, f, inside);
    float gx = 0.f, gy = 0.f, s0[3], s1[3] = {0.f, 0.f, 0.f};
    cs_level_bwd(st.tex[l0], st.d_tex[l0], fm, st.res[l0], g, 1.f - f, s0, gx, gy);
    const bool two = l1 != l0;
    if (two) cs_level_bwd(st.tex[l1], st.d_tex[l1], fm, st.res[l1], g, f, s1, gx, gy);
    if (d_level) {
        // out = (1-f) S_l0 + [l1 != l0] f S_l1 (the formulation of the tensor version this kernel replaces)
        float gl = 0.f;
        if (level && st.n > 1 && inside)
            gl = g[0] * ((two ? s1[0] : 0.f) - s0[0]) + g[1] * ((two ? s1[1] : 0.f) - s0[1]) + g[2] * ((two ? s1[2] : 0.f) - s0[2]);
        d_level[i] = gl;
    }
    if (d_dirs) {
        // x = sx d[ax] / m, y = sy d[ay] / m, m = sm d[am]
        float dd[3] = {0.f, 0.f, 0.f};
        const bool live = fabsf(d[fm.am]) >= 1e-30f;          // clamp_min(1e-30) passes no gradient below the bound
        dd[fm.ax] += gx * fm.sx / fm.m;
        dd[fm.ay] += gy * fm.sy / fm.m;
        if (live) dd[fm.am] += -(gx * fm.x + gy * fm.y) * fm.sm / fm.m;
        d_dirs[i * 3] = dd[0]; d_dirs[i * 3 + 1] = dd[1]; d_dirs[i * 3 + 2] = dd[2];
    }
}

int cs_fill(CubeStack& st, const float* const* tex, float* const* d_tex, const int32_t* res, int32_t n_levels) {
    TF_REQUIRE(tex && res && n_levels >= 1 && n_levels <= CS_MAX_LEVELS, "cube sample: 1..%d levels required", CS_MAX_LEVELS);
    st.n = n_levels;
    for (int l = 0; l < CS_MAX_LEVELS; ++l) {
        st.tex[l] = l < n_levels ? tex[l] : nullptr;
        st.d_tex[l] = (l < n_levels && d_tex) ? d_tex[l] : nullptr;
        st.res[l] = l < n_levels ? res[l] : 1;
        if (l < n_levels) TF_REQUIRE(tex[l] && res[l] > 0, "cube sample: NULL texture / bad resolution at level %d", l);
    }
    return 0;
}

}  // namespace

extern "C" TF_API int tf_cube_sample_fwd(const float* const* tex, const int32_t* res, int32_t n_levels, const float* dirs,
                                         const float* level, int64_t n, float* out, tf_stream_t stream) {
    if (n == 0) return 0;
    TF_REQUIRE(dirs && out, "tf_cube_sample_fwd: NULL pointer");
    CubeStack st;
    if (int rc = cs_fill(st, tex, nullptr, res, n_levels)) return rc;
    cube_sample_fwd_kernel<<<(unsigned)((n + 255) / 256), 256, 0, (cudaStream_t)stream>>>(st, dirs, level, n, out);
    tf_count_launches(1);
    TF_CHECK_LAUNCH("tf_cube_sample_fwd");
    return 0;
}

extern "C" TF_API int tf_cube_sample_bwd(const float* const* tex, const int32_t* res, int32_t n_levels, const float* dirs,
                                         const float* level, int64_t n, const float* g_out, float* const* d_tex, float* d_dirs,
                                         float* d_level, tf_stream_t stream) {
    if (n == 0) return 0;
    TF_REQUIRE(dirs && g_out, "tf_cube_sample_bwd: NULL pointer");
    CubeStack st;
    if (int rc = cs_fill(st, tex, d_tex, res, n_levels)) return rc;
    cube_sample_bwd_kernel<<<(unsigned)((n + 255) / 256), 256, 0, (cudaStream_t)stream>>>(st, dirs, level, n, g_out, d_dirs, d_level);
    tf_count_launches(1);
    TF_CHECK_LAUNCH("tf_cube_sample_bwd");
    return 0;
}
