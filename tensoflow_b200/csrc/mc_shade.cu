// Material-stage Monte-Carlo integral (reference MCShadingNetwork.shade_mixed,
// network/fields.py:1075-1335):
//   mc_directions : flow / cosine / GGX direction sets with their pdfs      (fields.py:824-903,1085-1108)
//   cube_light    : exp(seamless bilinear cube lookup) of the env light      (light.py:125-162) fwd + bwd
//   mc_estimate   : Cook-Torrance BRDF weights + diffuse / specular estimators (fields.py:977-1033,1146-1234) fwd + bwd
// One thread per (point, direction) pair for the first two, one warp per point for the estimator.
#include "shading.cuh"

namespace {

constexpr float PI_F = 3.14159265358979323846f;
constexpr float EPSF = 1e-6f;   // fields.py:18

__device__ __forceinline__ float clamp01(float x) { return fminf(fmaxf(x, 0.f), 1.f); }

// tangent frame of fields.py:812-822 (x), y = z cross x
__device__ __forceinline__ void tangent_frame(V3 n, V3& x, V3& y) {
    const V3 o0 = v3(n.y, -n.x, 0.f), o1 = v3(-n.z, 0.f, n.x);
    x = normalize12(sqrtf(dot(o0, o0)) > sqrtf(dot(o1, o1)) ? o0 : o1);
    y = cross(n, x);
}

// ---- direction sets -----------------------------------------------------------------------
// mode 0: flow samples, half-vector parametrisation; src = angles [pn,sn,2], aux = logj [pn,sn]
// mode 1: cosine set; src = table [sn,2] (az/2pi, el), aux = az_shift [pn] or NULL
// mode 2: GGX set;    src = table [sn,2],             aux = az_shift [pn] or NULL, rough [pn]
__global__ void __launch_bounds__(128) mc_directions_kernel(int mode, const float* __restrict__ normals, const float* __restrict__ view,
                                                            const float* __restrict__ src, const float* __restrict__ aux,
                                                            const float* __restrict__ rough, int64_t pn, int sn,
                                                            float* __restrict__ dirs, float* __restrict__ prob, int out_stride,
                                                            int out_offset) {
    const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (i >= pn * sn) return;
    const int64_t p = i / sn;
    const int s = (int)(i % sn);
    const V3 n = ld3(normals, p), v = ld3(view, p);
    V3 tx, ty;
    tangent_frame(n, tx, ty);
    V3 d;
    float pr;
    if (mode == 0) {
        const float phi = src[i * 2] * (2.f * PI_F), theta = src[i * 2 + 1] * (0.5f * PI_F);
        const float st = sinf(theta), ct = cosf(theta);
        const V3 H = (st * cosf(phi)) * tx + (st * sinf(phi)) * ty + ct * n;
        const float hov = clamp01(dot(v, H));
        d = (hov * 2.f) * H - v;
        const float lj = fminf(fmaxf(aux[i], -8.f), 8.f);
        pr = expf(-lj) / fmaxf(4.f * PI_F * PI_F * hov * st, EPSF);
    } else {
        float az = src[s * 2] * (2.f * PI_F);
        const float el = src[s * 2 + 1];
        if (aux) az = fmodf(az + aux[p] * (2.f * PI_F), 2.f * PI_F);
        const float jac = cosf((1.f - el) * PI_F * 0.5f) * PI_F * 0.5f;
        if (mode == 1) {
            const float es = sqrtf(el + 1e-7f), cz = sqrtf(1.f - el + 1e-7f);
            d = (es * cosf(az)) * tx + (es * sinf(az)) * ty + cz * n;
            pr = clamp01(dot(d, n)) / PI_F * jac;
        } else {
            const float a = rough[p];
            const float ctm = sqrtf(fmaxf((1.f - el) / fmaxf(1.f + (a * a - 1.f) * el, EPSF), EPSF));
            const float stm = sqrtf(fmaxf(1.f - ctm * ctm, EPSF));
            const V3 H = (cosf(az) * stm) * tx + (sinf(az) * stm) * ty + ctm * n;
            const float voh = clamp01(dot(v, H));
            d = (voh * 2.f) * H - v;
            const float noh = fmaxf(ctm, 0.f);
            const float a2 = a * a, den = noh * noh * (a2 - 1.f) + 1.f;
            const float D = a2 / fmaxf(PI_F * den * den, EPSF);
            pr = D * noh / fmaxf(4.f * voh, EPSF) * jac;
        }
    }
    const int64_t o = p * out_stride + out_offset + s;
    dirs[o * 3] = d.x; dirs[o * 3 + 1] = d.y; dirs[o * 3 + 2] = d.z;
    prob[o] = pr;
}

// ---- cube map --------------------------------------------------------------------------------
// the footprint of dirs[i] with each weight normalised on its own (w_k / W) before the weighted sum; cube_sample.cu divides the
// sum instead, which rounds differently
__device__ __forceinline__ CubeTaps light_taps(const float* dirs, int64_t i, int R) {
    const float d[3] = {dirs[i * 3], dirs[i * 3 + 1], dirs[i * 3 + 2]};
    CubeTaps t = cube_taps(cube_face(d), R);
#pragma unroll
    for (int k = 0; k < 4; ++k) t.w[k] /= t.wsum;
    return t;
}

// out[p] = exp(bilinear(base, dir[p])) where mask[p] != 0 (mask NULL = everywhere), else 0
__global__ void __launch_bounds__(256) cube_light_fwd_kernel(const float* __restrict__ base, int R, const float* __restrict__ dirs,
                                                             const uint8_t* __restrict__ mask, int64_t P, float* __restrict__ out) {
    const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (i >= P) return;
    float r = 0.f, g = 0.f, b = 0.f;
    if (!mask || mask[i]) {
        const CubeTaps t = light_taps(dirs, i, R);
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            const float* px = base + (size_t)t.idx[k] * 3;
            r = fmaf(t.w[k], __ldg(px), r); g = fmaf(t.w[k], __ldg(px + 1), g); b = fmaf(t.w[k], __ldg(px + 2), b);
        }
        r = expf(r); g = expf(g); b = expf(b);
    }
    out[i * 3] = r; out[i * 3 + 1] = g; out[i * 3 + 2] = b;
}

__global__ void __launch_bounds__(256) cube_light_bwd_kernel(int R, const float* __restrict__ dirs, const uint8_t* __restrict__ mask,
                                                             int64_t P, const float* __restrict__ out, const float* __restrict__ g_out,
                                                             float* __restrict__ d_base) {
    const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (i >= P) return;
    if (mask && !mask[i]) return;
    const float gr = g_out[i * 3] * out[i * 3], gg = g_out[i * 3 + 1] * out[i * 3 + 1], gb = g_out[i * 3 + 2] * out[i * 3 + 2];
    if (gr == 0.f && gg == 0.f && gb == 0.f) return;
    const CubeTaps t = light_taps(dirs, i, R);
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        if (t.w[k] == 0.f) continue;
        float* px = d_base + (size_t)t.idx[k] * 3;
        atomicAdd(px, t.w[k] * gr); atomicAdd(px + 1, t.w[k] * gg); atomicAdd(px + 2, t.w[k] * gb);
    }
}

// ---- BRDF + estimators, one warp per point ------------------------------------------------------
struct Brdf {   // specular weight terms of one direction (fields.py:1216-1224)
    float q, F0[3], Fr[3], G, gv, gl, Dg, den2, noh, nov, nol, den4, hov;
    bool dclamped;
};
__device__ __forceinline__ float g1(float c, float k) { return c / (c * (1.f - k) + k + 1e-5f); }

__device__ __forceinline__ Brdf brdf_terms(V3 n, V3 v, V3 d, const float alb[3], float m, float a) {
    Brdf b;
    const V3 H = normalize12(v + d);
    const float hov = clamp01(dot(H, v));
    b.hov = hov;
    const float t = clamp01(1.f - hov);
    b.q = t * t * t * t * t;
#pragma unroll
    for (int c = 0; c < 3; ++c) { b.F0[c] = 0.04f * (1.f - m) + m * alb[c]; b.Fr[c] = b.F0[c] + (1.f - b.F0[c]) * b.q; }
    b.nov = clamp01(dot(n, v));
    b.nol = clamp01(dot(n, d));
    const float k = a * 0.5f;
    b.gv = g1(b.nov, k); b.gl = g1(b.nol, k);
    b.G = b.gv * b.gl;
    b.noh = clamp01(dot(n, H));
    const float a2 = a * a;
    b.den2 = b.noh * b.noh * (a2 - 1.f) + 1.f;
    const float dd = PI_F * b.den2 * b.den2;
    b.dclamped = dd < EPSF;
    b.Dg = a2 / fmaxf(dd, EPSF);
    b.den4 = fmaxf(4.f * b.nov, EPSF);
    return b;
}

__device__ __forceinline__ float wsum(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

// per point outputs: [0:3] diffuse estimate, [3:6] specular estimate, [6:9] mean diffuse light,
// [9:12] mean specular light (valid dirs), [12] visibility, [13:16] indirect light,
// neural-importance-sampling loss terms (fields.py:1254-1333): [16] sum over the nd flow-sampled diffuse directions and rgb of
// f(x) log q(x) / p(x), [17] the same over the N.L > 0 flow-sampled specular directions, [18] their count   (19 floats)
constexpr int EST_OUT = 19;

// log of the direction pdf of a flow sample in the half-vector parametrisation: log q(x) - log(max(4 pi^2 H.V sin(theta), EPS))
__device__ __forceinline__ float nis_logq(float logq_x, float hov, float theta_unit) {
    return logq_x - logf(fmaxf(4.f * PI_F * PI_F * hov * sinf(theta_unit * (0.5f * PI_F)), EPSF));
}
struct NisArgs {
    const float* logq_d; const float* ang_d; int nd;     // [pn, nd], [pn, nd, 2]: the first nd diffuse directions (NULL: no term)
    const float* logq_s; const float* ang_s;             // [pn, Ds], [pn, Ds, 2]: every specular direction (NULL: no term)
};

__global__ void __launch_bounds__(256) mc_estimate_fwd_kernel(const float* __restrict__ normals, const float* __restrict__ view,
                                                              const float* __restrict__ albedo, const float* __restrict__ metallic,
                                                              const float* __restrict__ rough, const float* __restrict__ dirs,
                                                              const float* __restrict__ prob, const float* __restrict__ lights,
                                                              const uint8_t* __restrict__ hit, int64_t pn, int Dd, int Ds,
                                                              NisArgs nis, float* __restrict__ out) {
    const int lane = threadIdx.x & 31;
    const int64_t p = (blockIdx.x * (int64_t)blockDim.x + threadIdx.x) >> 5;
    if (p >= pn) return;
    const V3 n = ld3(normals, p), v = ld3(view, p);
    const float alb[3] = {albedo[p * 3], albedo[p * 3 + 1], albedo[p * 3 + 2]};
    const float m = metallic[p], a = rough[p];
    const int D = Dd + Ds;
    float acc[EST_OUT];
#pragma unroll
    for (int k = 0; k < EST_OUT; ++k) acc[k] = 0.f;
    for (int j = lane; j < D; j += 32) {
        const int64_t o = p * D + j;
        const V3 d = ld3(dirs, o);
        const float L[3] = {lights[o * 3], lights[o * 3 + 1], lights[o * 3 + 2]};
        const float ip = 1.f / fmaxf(prob[o], EPSF);
        if (j < Dd) {
            const float c = clamp01(dot(d, n)) / PI_F * (1.f - m);
#pragma unroll
            for (int k = 0; k < 3; ++k) { acc[k] += alb[k] * c * L[k] * ip; acc[6 + k] += L[k]; }
            if (nis.logq_d && j < nis.nd) {
                const int64_t q = p * nis.nd + j;
                const float hov = clamp01(dot(normalize12(v + d), v));
                const float A = nis_logq(nis.logq_d[q], hov, nis.ang_d[q * 2 + 1]) * ip;
#pragma unroll
                for (int k = 0; k < 3; ++k) acc[16] += alb[k] * c * L[k] * A;
            }
        } else if (dot(d, n) > 0.f) {
            const Brdf b = brdf_terms(n, v, d, alb, m, a);
            const float h = hit[o] ? 1.f : 0.f;
            float A = 0.f;
            if (nis.logq_s) {
                const int64_t q = p * Ds + (j - Dd);
                A = nis_logq(nis.logq_s[q], b.hov, nis.ang_s[q * 2 + 1]) * ip;
                acc[18] += 1.f;
            }
#pragma unroll
            for (int k = 0; k < 3; ++k) {
                const float sw = b.Dg * b.Fr[k] * b.G / b.den4 * L[k];
                acc[3 + k] += sw * ip;
                acc[17] += sw * A;
                acc[9 + k] += L[k];
                acc[13 + k] += L[k] * h;
            }
            acc[12] += h;
        }
    }
#pragma unroll
    for (int k = 0; k < EST_OUT; ++k) acc[k] = wsum(acc[k]);
    if (lane == 0) {
        const float id = 1.f / (float)Dd, is = 1.f / (float)Ds;
#pragma unroll
        for (int k = 0; k < 3; ++k) {
            out[p * EST_OUT + k] = acc[k] * id;
            out[p * EST_OUT + 3 + k] = acc[3 + k] * is;
            out[p * EST_OUT + 6 + k] = acc[6 + k] * id;
            out[p * EST_OUT + 9 + k] = acc[9 + k] * is;
            out[p * EST_OUT + 13 + k] = acc[13 + k] * is;
        }
        out[p * EST_OUT + 12] = 1.f - acc[12] * is;
        out[p * EST_OUT + 16] = acc[16]; out[p * EST_OUT + 17] = acc[17]; out[p * EST_OUT + 18] = acc[18];
    }
}

// g_out [pn,16] -> d_albedo [pn,3], d_metallic [pn], d_rough [pn], d_lights [pn,D,3]
__global__ void __launch_bounds__(256) mc_estimate_bwd_kernel(const float* __restrict__ normals, const float* __restrict__ view,
                                                              const float* __restrict__ albedo, const float* __restrict__ metallic,
                                                              const float* __restrict__ rough, const float* __restrict__ dirs,
                                                              const float* __restrict__ prob, const float* __restrict__ lights,
                                                              const uint8_t* __restrict__ hit, int64_t pn, int Dd, int Ds,
                                                              NisArgs nis, const float* __restrict__ g_out, float* __restrict__ d_albedo,
                                                              float* __restrict__ d_metallic, float* __restrict__ d_rough,
                                                              float* __restrict__ d_lights, float* __restrict__ d_logq_d,
                                                              float* __restrict__ d_logq_s) {
    const int lane = threadIdx.x & 31;
    const int64_t p = (blockIdx.x * (int64_t)blockDim.x + threadIdx.x) >> 5;
    if (p >= pn) return;
    const V3 n = ld3(normals, p), v = ld3(view, p);
    const float alb[3] = {albedo[p * 3], albedo[p * 3 + 1], albedo[p * 3 + 2]};
    const float m = metallic[p], a = rough[p];
    const int D = Dd + Ds;
    const float id = 1.f / (float)Dd, is = 1.f / (float)Ds;
    float g[EST_OUT];
#pragma unroll
    for (int k = 0; k < EST_OUT; ++k) g[k] = g_out[p * EST_OUT + k];
    float da[3] = {0.f, 0.f, 0.f}, dm = 0.f, dr = 0.f;
    for (int j = lane; j < D; j += 32) {
        const int64_t o = p * D + j;
        const V3 d = ld3(dirs, o);
        const float L[3] = {lights[o * 3], lights[o * 3 + 1], lights[o * 3 + 2]};
        const float ip = 1.f / fmaxf(prob[o], EPSF);
        float dL[3] = {0.f, 0.f, 0.f};
        if (j < Dd) {
            const float c0 = clamp01(dot(d, n)) / PI_F;
            const float c = c0 * (1.f - m);
            // the NIS term of the pair: g16 * sum_k albedo_k c L_k * A with A = log q / p  (same shape as the estimator's 1 / p)
            float A = 0.f;
            if (nis.logq_d && j < nis.nd) {
                const int64_t q = p * nis.nd + j;
                const float hov = clamp01(dot(normalize12(v + d), v));
                A = nis_logq(nis.logq_d[q], hov, nis.ang_d[q * 2 + 1]) * ip;
                d_logq_d[q] = g[16] * (alb[0] * L[0] + alb[1] * L[1] + alb[2] * L[2]) * c * ip;
            }
#pragma unroll
            for (int k = 0; k < 3; ++k) {
                const float gk = g[k] * id * ip + g[16] * A;
                da[k] += gk * c * L[k];
                dm -= gk * alb[k] * c0 * L[k];
                dL[k] = gk * alb[k] * c + g[6 + k] * id;
            }
        } else if (dot(d, n) > 0.f) {
            const Brdf b = brdf_terms(n, v, d, alb, m, a);
            const float h = hit[o] ? 1.f : 0.f;
            float dDg = 0.f, dG = 0.f;
            float A = 0.f;
            if (nis.logq_s) {
                const int64_t q = p * Ds + (j - Dd);
                A = nis_logq(nis.logq_s[q], b.hov, nis.ang_s[q * 2 + 1]) * ip;
                d_logq_s[q] = g[17] * b.Dg * b.G / b.den4 * (b.Fr[0] * L[0] + b.Fr[1] * L[1] + b.Fr[2] * L[2]) * ip;
            }
#pragma unroll
            for (int k = 0; k < 3; ++k) {
                const float gsw = (g[3 + k] * is * ip + g[17] * A) * L[k];   // d / d specular weight (estimator + NIS term)
                const float dF = gsw * b.Dg * b.G / b.den4;
                dDg += gsw * b.Fr[k] * b.G / b.den4;
                dG += gsw * b.Fr[k] * b.Dg / b.den4;
                const float dF0 = dF * (1.f - b.q);
                dm += dF0 * (alb[k] - 0.04f);
                da[k] += dF0 * m;
                dL[k] = (g[3 + k] * is * ip + g[17] * A) * b.Dg * b.Fr[k] * b.G / b.den4 + g[9 + k] * is + g[13 + k] * is * h;
            }
            // D_ggx wrt a (fields.py:1019-1024)
            const float a2 = a * a;
            if (b.dclamped) dr += dDg * 2.f * a / EPSF;
            else dr += dDg * (2.f * a / (PI_F * b.den2 * b.den2) - 4.f * a2 * a * b.noh * b.noh / (PI_F * b.den2 * b.den2 * b.den2));
            // G wrt k = a/2 (fields.py:987-998)
            const float k = a * 0.5f;
            const float dv = b.nov * (1.f - k) + k + 1e-5f, dl = b.nol * (1.f - k) + k + 1e-5f;
            const float dgv = -b.nov * (1.f - b.nov) / (dv * dv), dgl = -b.nol * (1.f - b.nol) / (dl * dl);
            dr += dG * (dgv * b.gl + b.gv * dgl) * 0.5f;
        } else if (nis.logq_s && j >= Dd) {
            d_logq_s[p * Ds + (j - Dd)] = 0.f;                       // N.L <= 0: the pair is not part of the loss
        }
        d_lights[o * 3] = dL[0]; d_lights[o * 3 + 1] = dL[1]; d_lights[o * 3 + 2] = dL[2];
    }
#pragma unroll
    for (int k = 0; k < 3; ++k) da[k] = wsum(da[k]);
    dm = wsum(dm); dr = wsum(dr);
    if (lane == 0) {
        d_albedo[p * 3] = da[0]; d_albedo[p * 3 + 1] = da[1]; d_albedo[p * 3 + 2] = da[2];
        d_metallic[p] = dm;
        d_rough[p] = dr;
    }
}

// ---- hit records -> inner-light MLP input (fields.py:951-975) ---------------------------------------------------------
// X[i, 0:51] = posenc(p, 8), X[i, 51:123] = IDE(reflect(v, n)) with kappa_inv = 0 (utils/ref_utils.py:53-117, degree 5: 36 (m, l)
// pairs), X[i, 123:ldx] = 0, for the i-th occluded (point, direction) pair: p = inters[idx[i]], v = -dirs[idx[i]],
// n = normalize(hit_normals[idx[i]]).  One thread per hit; the IDE polynomial table mat[17, 36] sits in shared memory.
constexpr int PE_L = 8;
__global__ void __launch_bounds__(128) hit_encode_kernel(const float* __restrict__ inters, const float* __restrict__ dirs,
                                                         const float* __restrict__ hit_normals, const int64_t* __restrict__ idx, int64_t M,
                                                         const float* __restrict__ ide_mat, const int32_t* __restrict__ ide_m, int ldx,
                                                         float* __restrict__ X) {
    __shared__ float s_mat[IDE_NP * IDE_N];
    __shared__ int s_m[IDE_N];
    ide_load(ide_mat, ide_m, nullptr, s_mat, s_m, nullptr);
    const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (i >= M) return;
    const int64_t o = idx[i];
    const V3 p = ld3(inters, o), v = -1.f * ld3(dirs, o), n = normalize12(ld3(hit_normals, o));
    const V3 r = (dot(v, n) * 2.f) * n - v;
    float* x = X + i * ldx;
    posenc3(x, p, PE_L);
    ide_encode(x + 51, r, s_mat, s_m, nullptr, 0.f);
    for (int c = 51 + 2 * IDE_N; c < ldx; ++c) x[c] = 0.f;
}

}  // namespace

extern "C" TF_API int tf_mc_directions(int32_t mode, const float* normals, const float* view_dirs, const float* src, const float* aux,
                                       const float* roughness, int64_t n_points, int32_t n_dirs, float* dirs, float* prob,
                                       int32_t out_stride, int32_t out_offset, tf_stream_t stream) {
    if (n_points == 0 || n_dirs == 0) return 0;
    TF_REQUIRE(mode >= 0 && mode <= 2, "tf_mc_directions: bad mode %d", mode);
    TF_REQUIRE(normals && view_dirs && src && dirs && prob, "tf_mc_directions: NULL pointer");
    TF_REQUIRE(mode != 0 || aux, "tf_mc_directions: flow mode needs logj");
    TF_REQUIRE(mode != 2 || roughness, "tf_mc_directions: GGX mode needs roughness");
    TF_REQUIRE(out_stride >= out_offset + n_dirs, "tf_mc_directions: bad output stride");
    const int64_t total = n_points * n_dirs;
    mc_directions_kernel<<<(unsigned)((total + 127) / 128), 128, 0, (cudaStream_t)stream>>>(mode, normals, view_dirs, src, aux, roughness,
                                                                                            n_points, n_dirs, dirs, prob, out_stride,
                                                                                            out_offset);
    tf_count_launches(1);
    TF_CHECK_LAUNCH("tf_mc_directions");
    return 0;
}

extern "C" TF_API int tf_cube_light_fwd(const float* base, int32_t res, const float* dirs, const uint8_t* mask, int64_t n, float* out,
                                        tf_stream_t stream) {
    if (n == 0) return 0;
    TF_REQUIRE(base && dirs && out && res > 0, "tf_cube_light_fwd: NULL pointer / bad res");
    cube_light_fwd_kernel<<<(unsigned)((n + 255) / 256), 256, 0, (cudaStream_t)stream>>>(base, res, dirs, mask, n, out);
    tf_count_launches(1);
    TF_CHECK_LAUNCH("tf_cube_light_fwd");
    return 0;
}

extern "C" TF_API int tf_cube_light_bwd(int32_t res, const float* dirs, const uint8_t* mask, int64_t n, const float* out,
                                        const float* g_out, float* d_base, tf_stream_t stream) {
    if (n == 0) return 0;
    TF_REQUIRE(dirs && out && g_out && d_base && res > 0, "tf_cube_light_bwd: NULL pointer / bad res");
    cube_light_bwd_kernel<<<(unsigned)((n + 255) / 256), 256, 0, (cudaStream_t)stream>>>(res, dirs, mask, n, out, g_out, d_base);
    tf_count_launches(1);
    TF_CHECK_LAUNCH("tf_cube_light_bwd");
    return 0;
}

extern "C" TF_API int tf_mc_estimate_fwd(const float* normals, const float* view_dirs, const float* albedo, const float* metallic,
                                         const float* roughness, const float* dirs, const float* prob, const float* lights,
                                         const uint8_t* hit, int64_t n_points, int32_t n_diffuse, int32_t n_specular,
                                         const float* logq_diffuse, const float* angles_diffuse, int32_t n_nis_diffuse,
                                         const float* logq_specular, const float* angles_specular, float* out, tf_stream_t stream) {
    if (n_points == 0) return 0;
    TF_REQUIRE(normals && view_dirs && albedo && metallic && roughness && dirs && prob && lights && hit && out, "tf_mc_estimate_fwd: NULL pointer");
    TF_REQUIRE(n_diffuse > 0 && n_specular > 0, "tf_mc_estimate_fwd: need diffuse and specular directions");
    TF_REQUIRE(!logq_diffuse || (angles_diffuse && n_nis_diffuse > 0 && n_nis_diffuse <= n_diffuse), "tf_mc_estimate_fwd: bad diffuse NIS arguments");
    TF_REQUIRE(!logq_specular || angles_specular, "tf_mc_estimate_fwd: bad specular NIS arguments");
    const NisArgs nis = {logq_diffuse, angles_diffuse, logq_diffuse ? n_nis_diffuse : 0, logq_specular, angles_specular};
    const int64_t threads = n_points * 32;
    mc_estimate_fwd_kernel<<<(unsigned)((threads + 255) / 256), 256, 0, (cudaStream_t)stream>>>(normals, view_dirs, albedo, metallic, roughness,
                                                                                                dirs, prob, lights, hit, n_points, n_diffuse,
                                                                                                n_specular, nis, out);
    tf_count_launches(1);
    TF_CHECK_LAUNCH("tf_mc_estimate_fwd");
    return 0;
}

extern "C" TF_API int tf_mc_estimate_bwd(const float* normals, const float* view_dirs, const float* albedo, const float* metallic,
                                         const float* roughness, const float* dirs, const float* prob, const float* lights,
                                         const uint8_t* hit, int64_t n_points, int32_t n_diffuse, int32_t n_specular,
                                         const float* logq_diffuse, const float* angles_diffuse, int32_t n_nis_diffuse,
                                         const float* logq_specular, const float* angles_specular, const float* g_out,
                                         float* d_albedo, float* d_metallic, float* d_roughness, float* d_lights, float* d_logq_diffuse,
                                         float* d_logq_specular, tf_stream_t stream) {
    if (n_points == 0) return 0;
    TF_REQUIRE(normals && view_dirs && albedo && metallic && roughness && dirs && prob && lights && hit && g_out, "tf_mc_estimate_bwd: NULL input");
    TF_REQUIRE(d_albedo && d_metallic && d_roughness && d_lights, "tf_mc_estimate_bwd: NULL output");
    TF_REQUIRE(!logq_diffuse || (angles_diffuse && d_logq_diffuse && n_nis_diffuse > 0 && n_nis_diffuse <= n_diffuse), "tf_mc_estimate_bwd: bad diffuse NIS arguments");
    TF_REQUIRE(!logq_specular || (angles_specular && d_logq_specular), "tf_mc_estimate_bwd: bad specular NIS arguments");
    const NisArgs nis = {logq_diffuse, angles_diffuse, logq_diffuse ? n_nis_diffuse : 0, logq_specular, angles_specular};
    const int64_t threads = n_points * 32;
    mc_estimate_bwd_kernel<<<(unsigned)((threads + 255) / 256), 256, 0, (cudaStream_t)stream>>>(normals, view_dirs, albedo, metallic, roughness,
                                                                                                dirs, prob, lights, hit, n_points, n_diffuse,
                                                                                                n_specular, nis, g_out, d_albedo, d_metallic,
                                                                                                d_roughness, d_lights, d_logq_diffuse,
                                                                                                d_logq_specular);
    tf_count_launches(1);
    TF_CHECK_LAUNCH("tf_mc_estimate_bwd");
    return 0;
}

extern "C" TF_API int tf_hit_encode(const float* inters, const float* dirs, const float* hit_normals, const int64_t* idx, int64_t n_hits,
                                    const float* ide_mat, const int32_t* ide_m, int32_t ldx, float* X, tf_stream_t stream) {
    if (n_hits == 0) return 0;
    TF_REQUIRE(inters && dirs && hit_normals && idx && ide_mat && ide_m && X, "tf_hit_encode: NULL pointer");
    TF_REQUIRE(ldx >= 123, "tf_hit_encode: rows need at least 123 columns");
    hit_encode_kernel<<<(unsigned)((n_hits + 127) / 128), 128, 0, (cudaStream_t)stream>>>(inters, dirs, hit_normals, idx, n_hits, ide_mat, ide_m,
                                                                                          ldx, X);
    tf_count_launches(1);
    TF_CHECK_LAUNCH("tf_hit_encode");
    return 0;
}
