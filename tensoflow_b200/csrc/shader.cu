// Per-sample part of the shape-stage shader (reference network/fields.py:448-567 ShapeShadingNetwork.forward,
// utils/ref_utils.py:53-117 integrated directional encoding, utils/network_utils.py:38-50 positional encoding,
// utils/raw_utils.py:4-10 linear_to_srgb) around the MLP heads and the environment-light lookups:
//   shader_encode  : normal / view normalisation, mirror direction, N.V, roughness, and the three MLP input matrices written
//                    directly in their zero-padded tensor-core layouts:
//                      X_rad = [features | points | PE(view, 4) | normals]                       (radiance head)
//                      X_il  = [PE(points, 8) | IDE(mirror direction, roughness)]               (indirect-light head)
//                      X_iw  = [PE(points, 8) | PE(mirror direction, 6)]                         (occlusion head, no gradient)
//   shader_combine : material affine maps, split-sum FG LUT (bilinear, clamp), diffuse + specular combination with the
//                    occlusion blend, linear -> sRGB, clamp
// each with a hand-derived backward.  One thread per sample; HBM-bound (the encode writes ~1.6 KB per sample).
#include "shading.cuh"

namespace {

constexpr int PE_PTS = 8, PE_VIEW = 4, PE_REFL = 6;

struct IdeTables { const float* mat; const int32_t* m; const float* sigma; };   // [17,36], [36], [36] (device)

struct Geo { V3 n, v, r; float nov, rough, nlen; bool bad; };
__device__ __forceinline__ Geo shader_geo(const float* normals, const float* view, const float* mat, int64_t i) {
    Geo g;
    g.n = normalize12(ld3(normals, i), g.nlen);
    g.bad = (g.n.x + g.n.y) == 0.f;                              // fields.py:455-456
    if (g.bad) g.n = v3(0.f, 1e-6f, 1.f);
    float vl;
    g.v = normalize12(ld3(view, i), vl);
    g.nov = dot(g.v, g.n);
    const float s = g.nov * 2.f;
    g.r = v3(g.nov * g.n.x * 2.f - g.v.x, g.nov * g.n.y * 2.f - g.v.y, g.nov * g.n.z * 2.f - g.v.z);
    (void)s;
    g.rough = mat[i * 5 + 3] * 0.9f + 0.09f;                     // fields.py:463
    return g;
}

struct EncParams {
    const float* points; const float* normals; const float* view; const float* mat; const float* feat;
    int fd, ld_rad; int64_t n;
    IdeTables ide;
    float* nrm; float* vdir; float* refl; float* nov; float* rough;
    float* X_rad; float* X_il; float* X_iw;       // ld 128 / 96
};
constexpr int LD_IL = 128, LD_IW = 96;

constexpr int ENC_TS = 129;      // row stride of the per-warp staging tile (conflict-free row writes and row reads)

// rows [base, base + 32) x ncols of the warp's staging tile -> global rows of ld floats at column col0 (coalesced: lane = column)
__device__ __forceinline__ void warp_store_rows(const float* tile, float* __restrict__ dst, int ld, int col0, int ncols, int64_t base, int64_t n, int lane) {
    for (int r = 0; r < 32 && base + r < n; ++r)
        for (int c = lane; c < ncols; c += 32) dst[(base + r) * ld + col0 + c] = tile[r * ENC_TS + c];
}

__global__ void __launch_bounds__(128) shader_encode_fwd_kernel(EncParams p) {
    extern __shared__ float enc_sm[];
    __shared__ float s_mat[IDE_NP * IDE_N];
    __shared__ float s_sig[IDE_N];
    __shared__ int s_m[IDE_N];
    ide_load(p.ide.mat, p.ide.m, p.ide.sigma, s_mat, s_m, s_sig);
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    float* tile = enc_sm + warp * 32 * ENC_TS;
    float* x = tile + lane * ENC_TS;                 // this sample's staging row
    const int64_t base = (blockIdx.x * (int64_t)blockDim.x + threadIdx.x) - lane;
    const int64_t i = base + lane;
    if (base >= p.n) return;
    const bool live = i < p.n;
    Geo g;
    V3 pt = v3(0.f, 0.f, 0.f);
    if (live) {
        g = shader_geo(p.normals, p.view, p.mat, i);
        pt = ld3(p.points, i);
        p.nrm[i * 3] = g.n.x; p.nrm[i * 3 + 1] = g.n.y; p.nrm[i * 3 + 2] = g.n.z;
        p.vdir[i * 3] = g.v.x; p.vdir[i * 3 + 1] = g.v.y; p.vdir[i * 3 + 2] = g.v.z;
        p.refl[i * 3] = g.r.x; p.refl[i * 3 + 1] = g.r.y; p.refl[i * 3 + 2] = g.r.z;
        p.nov[i] = g.nov;
        p.rough[i] = g.rough;
        // ---- [PE(points, 8) | IDE(mirror direction, roughness) | 0] into the staging row -------------------------------
        posenc3(x, pt, PE_PTS);
        ide_encode(x + 51, g.r, s_mat, s_m, s_sig, g.rough);
        for (int c = 51 + 2 * IDE_N; c < LD_IL; ++c) x[c] = 0.f;
    }
    __syncwarp();
    warp_store_rows(tile, p.X_il, LD_IL, 0, LD_IL, base, p.n, lane);
    __syncwarp();
    if (live) {                                     // [PE(points, 8) (kept) | PE(mirror direction, 6) | 0]
        posenc3(x + 51, g.r, PE_REFL);
        for (int c = 51 + 39; c < LD_IW; ++c) x[c] = 0.f;
    }
    __syncwarp();
    warp_store_rows(tile, p.X_iw, LD_IW, 0, LD_IW, base, p.n, lane);
    if (p.X_rad) {                                  // [features | points | PE(view, 4) | normals | 0]
        for (int r = 0; r < 32 && base + r < p.n; ++r) {
            const float4* src = reinterpret_cast<const float4*>(p.feat + (base + r) * p.fd);
            float4* dst = reinterpret_cast<float4*>(p.X_rad + (base + r) * p.ld_rad);
            for (int c = lane; c < p.fd / 4; c += 32) dst[c] = __ldg(src + c);
        }
        __syncwarp();
        const int tail = p.ld_rad - p.fd;
        if (live) {
            x[0] = pt.x; x[1] = pt.y; x[2] = pt.z;
            posenc3(x + 3, g.v, PE_VIEW);
            x[30] = g.n.x; x[31] = g.n.y; x[32] = g.n.z;
            for (int c = 33; c < tail; ++c) x[c] = 0.f;
        }
        __syncwarp();
        warp_store_rows(tile, p.X_rad, p.ld_rad, p.fd, tail, base, p.n, lane);
    }
}

struct EncBwdParams {
    const float* normals; const float* view; const float* mat; int fd, ld_rad; int64_t n;
    IdeTables ide;
    const float* g_nrm; const float* g_refl; const float* g_nov; const float* g_rough; const float* g_Xrad; const float* g_Xil;   // each may be NULL
    float* d_normals; float* d_mat3; float* d_feat;
};

__global__ void __launch_bounds__(128) shader_encode_bwd_kernel(EncBwdParams p) {
    __shared__ float s_mat[IDE_NP * IDE_N];
    __shared__ float s_sig[IDE_N];
    __shared__ int s_m[IDE_N];
    ide_load(p.ide.mat, p.ide.m, p.ide.sigma, s_mat, s_m, s_sig);
    const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (i >= p.n) return;
    const Geo g = shader_geo(p.normals, p.view, p.mat, i);
    V3 dn = p.g_nrm ? ld3(p.g_nrm, i) : v3(0.f, 0.f, 0.f);
    V3 dr = p.g_refl ? ld3(p.g_refl, i) : v3(0.f, 0.f, 0.f);
    float dnov = p.g_nov ? p.g_nov[i] : 0.f;
    float drough = p.g_rough ? p.g_rough[i] : 0.f;
    if (p.g_Xrad) {
        const float* gx = p.g_Xrad + i * p.ld_rad;
        if (p.d_feat) {
            const float4* s4 = reinterpret_cast<const float4*>(gx);
            float4* d4 = reinterpret_cast<float4*>(p.d_feat + i * p.fd);
            for (int c = 0; c < p.fd / 4; ++c) d4[c] = s4[c];
        }
        dn.x += gx[p.fd + 30]; dn.y += gx[p.fd + 31]; dn.z += gx[p.fd + 32];
    }
    if (p.g_Xil) {   // adjoint of the integrated directional encoding wrt the mirror direction and the roughness
        const float* gx = p.g_Xil + i * LD_IL + 51;
        float zk[IDE_NP], re[IDE_NP], im[IDE_NP], dre[IDE_NP], dim_[IDE_NP];
        ide_powers(g.r, zk, re, im);
#pragma unroll
        for (int k = 0; k < IDE_NP; ++k) { dre[k] = 0.f; dim_[k] = 0.f; }
        float dz = 0.f;
        for (int j = 0; j < IDE_N; ++j) {
            float poly = 0.f, dpoly_dz = 0.f;
#pragma unroll
            for (int k = 0; k < IDE_NP; ++k) {
                const float c = s_mat[k * IDE_N + j];
                poly = fmaf(zk[k], c, poly);
                if (k > 0) dpoly_dz = fmaf((float)k * zk[k - 1], c, dpoly_dz);
            }
            const float e = expf(-s_sig[j] * g.rough);
            const float att = poly * e;
            const int m = s_m[j];
            float rm, imm;
            ide_pick(re, im, m, rm, imm);
            const float gre = gx[j], gim = gx[IDE_N + j];
            const float G = gre * rm + gim * imm;                 // d / d att
            dz += G * e * dpoly_dz;
            drough += G * att * (-s_sig[j]);
#pragma unroll
            for (int k = 0; k < IDE_NP; ++k) if (k == m) { dre[k] += gre * att; dim_[k] += gim * att; }
        }
        // (x + i y)^m: d Re / dx = m Re(w^(m-1)), d Re / dy = -m Im(w^(m-1)), d Im / dx = m Im(w^(m-1)), d Im / dy = m Re(w^(m-1))
        float dx = 0.f, dy = 0.f;
#pragma unroll
        for (int k = 1; k < IDE_NP; ++k) {
            dx += (float)k * (dre[k] * re[k - 1] + dim_[k] * im[k - 1]);
            dy += (float)k * (-dre[k] * im[k - 1] + dim_[k] * re[k - 1]);
        }
        dr.x += dx; dr.y += dy; dr.z += dz;
    }
    // mirror direction r = 2 (v.n) n - v and N.V
    const float grn = dot(dr, g.n);
    dn.x += 2.f * (grn * g.v.x + g.nov * dr.x) + dnov * g.v.x;
    dn.y += 2.f * (grn * g.v.y + g.nov * dr.y) + dnov * g.v.y;
    dn.z += 2.f * (grn * g.v.z + g.nov * dr.z) + dnov * g.v.z;
    // F.normalize (no gradient through the replaced degenerate normals)
    V3 out = v3(0.f, 0.f, 0.f);
    if (!g.bad) {
        const float t = dot(g.n, dn);
        out = v3((dn.x - g.n.x * t) / g.nlen, (dn.y - g.n.y * t) / g.nlen, (dn.z - g.n.z * t) / g.nlen);
    }
    p.d_normals[i * 3] = out.x; p.d_normals[i * 3 + 1] = out.y; p.d_normals[i * 3 + 2] = out.z;
    p.d_mat3[i] = drough * 0.9f;
}

// ---- combine ------------------------------------------------------------------------------------------------------
__device__ __forceinline__ float srgb(float x) {           // utils/raw_utils.py:4-10
    const float eps = 1.1920929e-07f;
    return x <= 0.0031308f ? (323.f / 25.f) * x : (211.f * powf(fmaxf(x, eps), 5.f / 12.f) - 11.f) / 200.f;
}
__device__ __forceinline__ float srgb_grad(float x) {
    const float eps = 1.1920929e-07f;
    if (x <= 0.0031308f) return 323.f / 25.f;
    return x >= eps ? (211.f / 200.f) * (5.f / 12.f) * powf(x, -7.f / 12.f) : 0.f;
}
struct Lut { float f0, f1, d0u, d1u, d0v, d1v; };           // values and their u / v derivatives
// dr.texture(FG_LUT, uv, filter_mode='linear', boundary_mode='clamp') (fields.py:522): lut [H,W,2]
__device__ __forceinline__ Lut fg_lookup(const float* __restrict__ lut, int H, int W, float u, float v) {
    const float x = u * W - 0.5f, y = v * H - 0.5f;
    const float x0f = floorf(x), y0f = floorf(y);
    const float fx = x - x0f, fy = y - y0f;
    const int x0 = min(max((int)x0f, 0), W - 1), x1 = min(max((int)x0f + 1, 0), W - 1);
    const int y0 = min(max((int)y0f, 0), H - 1), y1 = min(max((int)y0f + 1, 0), H - 1);
    const float2 t00 = __ldg(reinterpret_cast<const float2*>(lut) + y0 * W + x0), t01 = __ldg(reinterpret_cast<const float2*>(lut) + y0 * W + x1);
    const float2 t10 = __ldg(reinterpret_cast<const float2*>(lut) + y1 * W + x0), t11 = __ldg(reinterpret_cast<const float2*>(lut) + y1 * W + x1);
    Lut r;
    r.f0 = t00.x * (1 - fx) * (1 - fy) + t01.x * fx * (1 - fy) + t10.x * (1 - fx) * fy + t11.x * fx * fy;
    r.f1 = t00.y * (1 - fx) * (1 - fy) + t01.y * fx * (1 - fy) + t10.y * (1 - fx) * fy + t11.y * fx * fy;
    r.d0u = ((t01.x - t00.x) * (1 - fy) + (t11.x - t10.x) * fy) * W;
    r.d1u = ((t01.y - t00.y) * (1 - fy) + (t11.y - t10.y) * fy) * W;
    r.d0v = ((t10.x - t00.x) * (1 - fx) + (t11.x - t01.x) * fx) * H;
    r.d1v = ((t10.y - t00.y) * (1 - fx) + (t11.y - t01.y) * fx) * H;
    return r;
}

struct CombParams {
    const float* mat; const float* diffuse_light; const float* direct_light; const float* indirect_light; const float* w_raw; const float* nov;
    const float* lut; int lut_h, lut_w; int64_t n;
    float* color; float* occ_prob;                              // fwd
    const float* g_color; const float* g_occ;                   // bwd (g_occ may be NULL)
    float* d_mat; float* d_diffuse; float* d_direct; float* d_indirect; float* d_w_raw; float* d_nov;
};

template <bool BWD>
__global__ void __launch_bounds__(256) shader_combine_kernel(CombParams p) {
    const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (i >= p.n) return;
    const float* m = p.mat + i * 5;
    const float alb[3] = {m[0] * 0.77f + 0.03f, m[1] * 0.77f + 0.03f, m[2] * 0.77f + 0.03f};
    const float rough = m[3] * 0.9f + 0.09f, met = m[4];
    const float occ_prob = p.w_raw[i] * 0.5f + 0.5f;
    const float occ = fminf(fmaxf(occ_prob, 0.f), 1.f);
    const float nov = p.nov[i];
    const float u = fminf(fmaxf(nov, 0.f), 1.f), v = fminf(fmaxf(rough, 0.f), 1.f);
    const Lut fg = fg_lookup(p.lut, p.lut_h, p.lut_w, u, v);
    float lin[3], sref[3], slight[3];
#pragma unroll
    for (int c = 0; c < 3; ++c) {
        const float dl = p.diffuse_light[i * 3 + c], ind = p.indirect_light[i * 3 + c], dir = p.direct_light[i * 3 + c];
        const float salb = 0.04f * (1.f - met) + met * alb[c];
        sref[c] = salb * fg.f0 + fg.f1;
        slight[c] = ind * occ + dir * (1.f - occ);
        lin[c] = (1.f - met) * alb[c] * dl + sref[c] * slight[c];
    }
    if (!BWD) {
#pragma unroll
        for (int c = 0; c < 3; ++c) p.color[i * 3 + c] = fminf(fmaxf(srgb(lin[c]), 0.f), 1.f);
        p.occ_prob[i] = occ_prob;
        return;
    }
    float d_alb[3], d_met = 0.f, d_f0 = 0.f, d_f1 = 0.f, d_occ = 0.f;
#pragma unroll
    for (int c = 0; c < 3; ++c) {
        const float s = srgb(lin[c]);
        const float gl = (s >= 0.f && s <= 1.f) ? p.g_color[i * 3 + c] * srgb_grad(lin[c]) : 0.f;      // d / d lin
        const float dl = p.diffuse_light[i * 3 + c], ind = p.indirect_light[i * 3 + c], dir = p.direct_light[i * 3 + c];
        p.d_diffuse[i * 3 + c] = gl * (1.f - met) * alb[c];
        const float d_sref = gl * slight[c], d_sl = gl * sref[c];
        p.d_indirect[i * 3 + c] = d_sl * occ;
        p.d_direct[i * 3 + c] = d_sl * (1.f - occ);
        d_occ += d_sl * (ind - dir);
        const float d_salb = d_sref * fg.f0;
        d_f0 += d_sref * (0.04f * (1.f - met) + met * alb[c]);
        d_f1 += d_sref;
        d_alb[c] = gl * (1.f - met) * dl + d_salb * met;
        d_met += -gl * alb[c] * dl + d_salb * (alb[c] - 0.04f);
    }
    const float d_u = d_f0 * fg.d0u + d_f1 * fg.d1u, d_v = d_f0 * fg.d0v + d_f1 * fg.d1v;
    p.d_nov[i] = (nov >= 0.f && nov <= 1.f) ? d_u : 0.f;
    const float d_rough = (rough >= 0.f && rough <= 1.f) ? d_v : 0.f;
    float d_occp = (occ_prob >= 0.f && occ_prob <= 1.f) ? d_occ : 0.f;
    if (p.g_occ) d_occp += p.g_occ[i];
    p.d_w_raw[i] = d_occp * 0.5f;
    float* dm = p.d_mat + i * 5;
    dm[0] = d_alb[0] * 0.77f; dm[1] = d_alb[1] * 0.77f; dm[2] = d_alb[2] * 0.77f;
    dm[3] = d_rough * 0.9f;
    dm[4] = d_met;
}

int ide_check(const float* a, const int32_t* b, const float* c) {
    TF_REQUIRE(a && b && c, "shader: IDE tables are NULL");
    return 0;
}

}  // namespace

extern "C" TF_API int tf_shader_encode_fwd(const float* points, const float* normals, const float* view_dirs, const float* mat, const float* feat,
                                           int32_t feat_dim, int32_t ld_rad, int64_t n, const float* ide_mat, const int32_t* ide_m,
                                           const float* ide_sigma, float* nrm, float* vdir, float* refl, float* nov, float* rough, float* X_rad,
                                           float* X_il, float* X_iw, tf_stream_t stream) {
    if (n == 0) return 0;
    if (int e = ide_check(ide_mat, ide_m, ide_sigma)) return e;
    TF_REQUIRE(points && normals && view_dirs && mat && nrm && vdir && refl && nov && rough && X_il && X_iw, "tf_shader_encode_fwd: NULL pointer");
    TF_REQUIRE(!X_rad || (feat && feat_dim > 0 && feat_dim % 4 == 0 && ld_rad >= feat_dim + 33 && ((uintptr_t)feat & 15) == 0 && ld_rad % 4 == 0),
               "tf_shader_encode_fwd: radiance input needs features (feat_dim %% 4 == 0, 16-byte aligned) and ld_rad >= feat_dim + 33");
    EncParams p = {points, normals, view_dirs, mat, feat, feat_dim, ld_rad, n, {ide_mat, ide_m, ide_sigma}, nrm, vdir, refl, nov, rough, X_rad, X_il, X_iw};
    TF_REQUIRE(!X_rad || ld_rad - feat_dim <= 128, "tf_shader_encode_fwd: ld_rad - feat_dim must be <= 128");
    const size_t smem = (size_t)4 * 32 * ENC_TS * sizeof(float);
    cudaFuncSetAttribute(shader_encode_fwd_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    shader_encode_fwd_kernel<<<(unsigned)((n + 127) / 128), 128, smem, (cudaStream_t)stream>>>(p);
    tf_count_launches(1);
    TF_CHECK_LAUNCH("tf_shader_encode_fwd");
    return 0;
}

extern "C" TF_API int tf_shader_encode_bwd(const float* normals, const float* view_dirs, const float* mat, int32_t feat_dim, int32_t ld_rad, int64_t n,
                                           const float* ide_mat, const int32_t* ide_m, const float* ide_sigma, const float* g_nrm,
                                           const float* g_refl, const float* g_nov, const float* g_rough, const float* g_X_rad, const float* g_X_il,
                                           float* d_normals, float* d_mat3, float* d_feat, tf_stream_t stream) {
    if (n == 0) return 0;
    if (int e = ide_check(ide_mat, ide_m, ide_sigma)) return e;
    TF_REQUIRE(normals && view_dirs && mat && d_normals && d_mat3, "tf_shader_encode_bwd: NULL pointer");
    TF_REQUIRE(!g_X_rad || (feat_dim % 4 == 0 && ld_rad % 4 == 0), "tf_shader_encode_bwd: bad radiance layout");
    EncBwdParams p = {normals, view_dirs, mat, feat_dim, ld_rad, n, {ide_mat, ide_m, ide_sigma}, g_nrm, g_refl, g_nov, g_rough, g_X_rad, g_X_il,
                      d_normals, d_mat3, d_feat};
    shader_encode_bwd_kernel<<<(unsigned)((n + 127) / 128), 128, 0, (cudaStream_t)stream>>>(p);
    tf_count_launches(1);
    TF_CHECK_LAUNCH("tf_shader_encode_bwd");
    return 0;
}

extern "C" TF_API int tf_shader_combine_fwd(const float* mat, const float* diffuse_light, const float* direct_light, const float* indirect_light,
                                            const float* w_raw, const float* nov, const float* lut, int32_t lut_h, int32_t lut_w, int64_t n,
                                            float* color, float* occ_prob, tf_stream_t stream) {
    if (n == 0) return 0;
    TF_REQUIRE(mat && diffuse_light && direct_light && indirect_light && w_raw && nov && lut && color && occ_prob, "tf_shader_combine_fwd: NULL pointer");
    CombParams p = {};
    p.mat = mat; p.diffuse_light = diffuse_light; p.direct_light = direct_light; p.indirect_light = indirect_light; p.w_raw = w_raw; p.nov = nov;
    p.lut = lut; p.lut_h = lut_h; p.lut_w = lut_w; p.n = n; p.color = color; p.occ_prob = occ_prob;
    shader_combine_kernel<false><<<(unsigned)((n + 255) / 256), 256, 0, (cudaStream_t)stream>>>(p);
    tf_count_launches(1);
    TF_CHECK_LAUNCH("tf_shader_combine_fwd");
    return 0;
}

extern "C" TF_API int tf_shader_combine_bwd(const float* mat, const float* diffuse_light, const float* direct_light, const float* indirect_light,
                                            const float* w_raw, const float* nov, const float* lut, int32_t lut_h, int32_t lut_w, int64_t n,
                                            const float* g_color, const float* g_occ, float* d_mat, float* d_diffuse, float* d_direct,
                                            float* d_indirect, float* d_w_raw, float* d_nov, tf_stream_t stream) {
    if (n == 0) return 0;
    TF_REQUIRE(mat && diffuse_light && direct_light && indirect_light && w_raw && nov && lut && g_color, "tf_shader_combine_bwd: NULL input");
    TF_REQUIRE(d_mat && d_diffuse && d_direct && d_indirect && d_w_raw && d_nov, "tf_shader_combine_bwd: NULL output");
    CombParams p = {};
    p.mat = mat; p.diffuse_light = diffuse_light; p.direct_light = direct_light; p.indirect_light = indirect_light; p.w_raw = w_raw; p.nov = nov;
    p.lut = lut; p.lut_h = lut_h; p.lut_w = lut_w; p.n = n; p.g_color = g_color; p.g_occ = g_occ;
    p.d_mat = d_mat; p.d_diffuse = d_diffuse; p.d_direct = d_direct; p.d_indirect = d_indirect; p.d_w_raw = d_w_raw; p.d_nov = d_nov;
    shader_combine_kernel<true><<<(unsigned)((n + 255) / 256), 256, 0, (cudaStream_t)stream>>>(p);
    tf_count_launches(1);
    TF_CHECK_LAUNCH("tf_shader_combine_bwd");
    return 0;
}
