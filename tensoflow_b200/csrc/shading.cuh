// Shading geometry shared by the cube-map lookups (cube_sample.cu, mc_shade.cu) and the per-sample encoders (mc_shade.cu,
// shader.cu): 3-vectors, the positional encoding, the basis of the integrated directional encoding and the seamless cube-map
// footprint.  The expressions are written as whole trees on purpose: nvcc contracts them into FMAs, so regrouping one changes
// the last bits of every kernel that uses it.
#pragma once
#include "common.cuh"

// ---- 3-vectors --------------------------------------------------------------------------------------------------------------
struct V3 { float x, y, z; };
__device__ __forceinline__ V3 v3(float x, float y, float z) { return V3{x, y, z}; }
__device__ __forceinline__ V3 operator+(V3 a, V3 b) { return v3(a.x + b.x, a.y + b.y, a.z + b.z); }
__device__ __forceinline__ V3 operator-(V3 a, V3 b) { return v3(a.x - b.x, a.y - b.y, a.z - b.z); }
__device__ __forceinline__ V3 operator*(float s, V3 a) { return v3(s * a.x, s * a.y, s * a.z); }
__device__ __forceinline__ float dot(V3 a, V3 b) { return a.x * b.x + a.y * b.y + a.z * b.z; }
__device__ __forceinline__ V3 cross(V3 a, V3 b) { return v3(a.y * b.z - a.z * b.y, a.z * b.x - a.x * b.z, a.x * b.y - a.y * b.x); }
__device__ __forceinline__ V3 ld3(const float* p, int64_t i) { return v3(p[i * 3], p[i * 3 + 1], p[i * 3 + 2]); }
__device__ __forceinline__ V3 normalize12(V3 a, float& len) {   // F.normalize: x / max(|x|, 1e-12)
    len = fmaxf(sqrtf(dot(a, a)), 1e-12f);
    return v3(a.x / len, a.y / len, a.z / len);
}
__device__ __forceinline__ V3 normalize12(V3 a) {
    float len;
    return normalize12(a, len);
}

// [v, sin(2^k v), cos(2^k v)]_{k < L} -> 3 + 6 L floats (utils/network_utils.py:38-50)
__device__ __forceinline__ void posenc3(float* x, V3 v, int L) {
    const float c[3] = {v.x, v.y, v.z};
#pragma unroll
    for (int a = 0; a < 3; ++a) x[a] = c[a];
    for (int k = 0; k < L; ++k) {
        const float f = (float)(1 << k);
#pragma unroll
        for (int a = 0; a < 3; ++a) { x[3 + k * 6 + a] = sinf(c[a] * f); x[3 + k * 6 + 3 + a] = cosf(c[a] * f); }
    }
}

// ---- integrated directional encoding, degree 5 (utils/ref_utils.py:53-117) ----------------------------------------------------
// entry j of the 36 (m, l) pairs: (x + i y)^m * sum_k z^k mat[k, j] * exp(-sigma_j kappa_inv), sigma_j = l (l + 1) / 2
constexpr int IDE_NP = 17, IDE_N = 36;          // powers of z, (m, l) entries

// mat [17,36], m [36] and sigma [36] (may be NULL) into shared memory, then a block barrier
__device__ __forceinline__ void ide_load(const float* mat, const int32_t* m, const float* sigma, float* s_mat, int* s_m, float* s_sig) {
    for (int i = threadIdx.x; i < IDE_NP * IDE_N; i += blockDim.x) s_mat[i] = mat[i];
    for (int i = threadIdx.x; i < IDE_N; i += blockDim.x) {
        s_m[i] = m[i];
        if (sigma) s_sig[i] = sigma[i];
    }
    __syncthreads();
}

// z^k and (x + i y)^k for k < IDE_NP
__device__ __forceinline__ void ide_powers(V3 r, float zk[IDE_NP], float re[IDE_NP], float im[IDE_NP]) {
    zk[0] = 1.f; re[0] = 1.f; im[0] = 0.f;
#pragma unroll
    for (int k = 1; k < IDE_NP; ++k) {
        zk[k] = zk[k - 1] * r.z;
        re[k] = re[k - 1] * r.x - im[k - 1] * r.y;
        im[k] = re[k - 1] * r.y + im[k - 1] * r.x;
    }
}

// sum_k z^k mat[k, j]
__device__ __forceinline__ float ide_poly(const float zk[IDE_NP], const float* s_mat, int j) {
    float poly = 0.f;
#pragma unroll
    for (int k = 0; k < IDE_NP; ++k) poly = fmaf(zk[k], s_mat[k * IDE_N + j], poly);
    return poly;
}

// (x + i y)^m for a run-time m, without indexing the power arrays at run time (they stay in registers)
__device__ __forceinline__ void ide_pick(const float re[IDE_NP], const float im[IDE_NP], int m, float& rm, float& imm) {
    rm = 0.f; imm = 0.f;
#pragma unroll
    for (int k = 0; k < IDE_NP; ++k) if (k == m) { rm = re[k]; imm = im[k]; }
}

// x[0:36] = Re, x[36:72] = Im of the encoding of the direction r; s_sig NULL: kappa_inv = 0 (no attenuation factor)
__device__ __forceinline__ void ide_encode(float* x, V3 r, const float* s_mat, const int* s_m, const float* s_sig, float kappa_inv) {
    float zk[IDE_NP], re[IDE_NP], im[IDE_NP];
    ide_powers(r, zk, re, im);
    for (int j = 0; j < IDE_N; ++j) {
        const float poly = ide_poly(zk, s_mat, j);
        const float att = s_sig ? poly * expf(-s_sig[j] * kappa_inv) : poly;
        float rm, imm;
        ide_pick(re, im, s_m[j], rm, imm);
        x[j] = rm * att;
        x[IDE_N + j] = imm * att;
    }
}

// ---- seamless cube-map footprint --------------------------------------------------------------------------------------------
// face convention of network/light_utils.py:24-31 / renderutils/c_src/cubemap.cu:32-60
__device__ __forceinline__ void cube_to_dir(int s, float x, float y, float c[3]) {
    switch (s) {
        case 0: c[0] = 1.f; c[1] = -y; c[2] = -x; break;
        case 1: c[0] = -1.f; c[1] = -y; c[2] = x; break;
        case 2: c[0] = x; c[1] = 1.f; c[2] = y; break;
        case 3: c[0] = x; c[1] = -1.f; c[2] = -y; break;
        case 4: c[0] = x; c[1] = -y; c[2] = 1.f; break;
        default: c[0] = -x; c[1] = -y; c[2] = -1.f; break;
    }
}

// x = sx d[ax] / m, y = sy d[ay] / m, m = sm d[am] > 0
struct CubeFace { int face, ax, ay, am; float sx, sy, sm, m, x, y; };

__device__ __forceinline__ CubeFace cube_face(const float d[3]) {
    CubeFace f;
    const float a0 = fabsf(d[0]), a1 = fabsf(d[1]), a2 = fabsf(d[2]);
    float am, dx, dy;          // |d[am]|, d[ax], d[ay] picked per branch: indexing d by a run-time axis would put it on the stack
    if (a0 >= a1 && a0 >= a2) {
        f.am = 0; f.ax = 2; f.ay = 1; f.sy = -1.f; am = a0; dx = d[2]; dy = d[1];
        if (d[0] >= 0.f) { f.face = 0; f.sx = -1.f; f.sm = 1.f; } else { f.face = 1; f.sx = 1.f; f.sm = -1.f; }
    } else if (a1 >= a2) {
        f.am = 1; f.ax = 0; f.ay = 2; f.sx = 1.f; am = a1; dx = d[0]; dy = d[2];
        if (d[1] >= 0.f) { f.face = 2; f.sy = 1.f; f.sm = 1.f; } else { f.face = 3; f.sy = -1.f; f.sm = -1.f; }
    } else {
        f.am = 2; f.ax = 0; f.ay = 1; f.sy = -1.f; am = a2; dx = d[0]; dy = d[1];
        if (d[2] >= 0.f) { f.face = 4; f.sx = 1.f; f.sm = 1.f; } else { f.face = 5; f.sx = -1.f; f.sm = -1.f; }
    }
    f.m = fmaxf(am, 1e-30f);
    f.x = f.sx * dx / f.m;
    f.y = f.sy * dy / f.m;
    return f;
}

// the 4 bilinear taps of a face footprint on a [6,R,R] texture: taps that leave the face fold onto the neighbouring face, the tap
// leaving in both axes (cube corner) is dropped.  The weights are raw: a lookup divides by wsum.
struct CubeTaps {
    int idx[4];
    float w[4];             // raw bilinear weights (0 for the dropped corner tap)
    float dwu[4], dwv[4];   // d w / d fu, d w / d fv
    float wsum;
};

__device__ __forceinline__ CubeTaps cube_taps(const CubeFace& f, int R) {
    const float u = (f.x + 1.f) * 0.5f * R - 0.5f, v = (f.y + 1.f) * 0.5f * R - 0.5f;
    const float u0f = floorf(u), v0f = floorf(v);
    const float fu = u - u0f, fv = v - v0f;
    const int u0 = (int)u0f, v0 = (int)v0f;
    CubeTaps t;
    t.wsum = 0.f;
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        const int du = k & 1, dv = k >> 1;
        int iu = u0 + du, iv = v0 + dv;
        const float a = du ? fu : 1.f - fu, b = dv ? fv : 1.f - fv;
        float w = a * b, dwu = (du ? 1.f : -1.f) * b, dwv = (dv ? 1.f : -1.f) * a;
        const bool ou = iu < 0 || iu >= R, ov = iv < 0 || iv >= R;
        int f2 = f.face;
        if (ou && ov) {
            w = 0.f; dwu = 0.f; dwv = 0.f;
            iu = min(max(iu, 0), R - 1); iv = min(max(iv, 0), R - 1);
        } else if (ou || ov) {
            const float fx = 2.f * ((float)iu + 0.5f) / R - 1.f, fy = 2.f * ((float)iv + 0.5f) / R - 1.f;
            float c[3];
            cube_to_dir(f.face, fx, fy, c);
            const int major = f.face >> 1;
            float e = 0.f;
            int over = -1;
#pragma unroll
            for (int a3 = 0; a3 < 3; ++a3)
                if (a3 != major && fabsf(c[a3]) > 1.f) { e = fabsf(c[a3]) - 1.f; over = a3; }
#pragma unroll
            for (int a3 = 0; a3 < 3; ++a3) {
                if (a3 == over) c[a3] = c[a3] > 0.f ? 1.f : -1.f;
                if (a3 == major) c[a3] = (c[a3] > 0.f ? 1.f : -1.f) * (1.f - e);
            }
            const CubeFace g = cube_face(c);
            f2 = g.face;
            iu = min(max((int)floorf((g.x + 1.f) * 0.5f * R), 0), R - 1);
            iv = min(max((int)floorf((g.y + 1.f) * 0.5f * R), 0), R - 1);
        }
        t.idx[k] = (f2 * R + iv) * R + iu;
        t.w[k] = w; t.dwu[k] = dwu; t.dwv[k] = dwv;
        t.wsum += w;
    }
    return t;
}
