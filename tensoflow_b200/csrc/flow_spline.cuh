// Piecewise-quadratic coupling transform of the TensoFlow sampler (reference network/flow.py:314-525,
// ElementWisePWQuadraticTransform, K = 10 bins: st = 11 vertex heights + 10 widths): device functions shared by the
// element-wise kernels (flow.cu) and the fused coupling-block kernels (flow_tc.cu).
#pragma once
#include <float.h>
#include "common.cuh"

namespace flowsp {

constexpr int NB = 10;       // bins
constexpr int NV = NB + 1;   // vertices
constexpr int NST = NB + NV; // conditioner outputs per coordinate (21)

// torch.lerp(a, b, w)
__device__ __forceinline__ float lerp_t(float a, float b, float w) { return w < 0.5f ? a + w * (b - a) : b - (b - a) * (1.f - w); }

struct Spline {
    float e[NB], w[NB], ws[NB], u[NV], v[NV], wr[NB], vr[NV];
    float S, Z;
};

// clamp_w = true for the forward spline (flow.py:343-346), false for the inverse (flow.py:427-431)
template <bool CLAMP_W>
__device__ __forceinline__ void spline_params(const float* __restrict__ st, Spline& s) {
    float cum = 0.f;
    float c[NB];
#pragma unroll
    for (int i = 0; i < NB; ++i) {
        float ei = expf(st[NV + i]);
        if (CLAMP_W) ei = fmaxf(ei, 1e-6f);
        s.e[i] = ei;
        cum += ei;
        c[i] = cum;
    }
    s.S = cum;
#pragma unroll
    for (int i = 0; i < NB; ++i) {
        s.wr[i] = s.e[i] / s.S;
        s.w[i] = CLAMP_W ? fmaxf(s.wr[i], 1e-6f) : s.wr[i];
        s.ws[i] = c[i] / s.S;
    }
#pragma unroll
    for (int j = 0; j < NV; ++j) s.u[j] = expf(st[j]);
    float Z = 0.f;
#pragma unroll
    for (int i = 0; i < NB; ++i) Z += (s.u[i] + s.u[i + 1]) * 0.5f * s.w[i];
    s.Z = Z;
#pragma unroll
    for (int j = 0; j < NV; ++j) {
        s.vr[j] = s.u[j] / Z;
        s.v[j] = fmaxf(s.vr[j], 1e-6f);
    }
}

// forward spline of one element (flow.py:343-412): x, log|dx/dy|
__device__ __forceinline__ void pwquad_eval_forward(const float* sr, float yy, float& x, float& lj) {
    const float eps = FLT_EPSILON;
    Spline s;
    spline_params<true>(sr, s);
    int m = 0;
#pragma unroll
    for (int i = 0; i < NB; ++i) m += (s.ws[i] <= yy) ? 1 : 0;   // number of cumulated widths <= x (flow.py:355-370)
    m = min(m, NB - 1);
    float wm = 0.f, vm = 0.f, vm1 = 0.f, wsh = 0.f, vw = 0.f;
#pragma unroll
    for (int i = 0; i < NB; ++i) {
        if (i == m) { wm = s.w[i]; vm = s.v[i]; vm1 = s.v[i + 1]; wsh = i == 0 ? 0.f : s.ws[i > 0 ? i - 1 : 0]; }
        if (i < m) vw += (s.v[i] + s.v[i + 1]) * 0.5f * s.w[i];
    }
    const float a = fminf(fmaxf((yy - wsh) / wm, 0.f), 1.f);
    float out = a * a * 0.5f * ((vm1 - vm) * wm) + a * vm * wm + vw;
    x = fminf(fmaxf(out, eps), 1.f - eps);
    lj = logf(lerp_t(vm, vm1, a));
}

// inverse spline (the sampling direction, flow.py:415-525)
__device__ __forceinline__ void pwquad_eval_inverse(const float* sr, float yy, float& x, float& lj) {
    const float eps = FLT_EPSILON;
    Spline s;
    spline_params<false>(sr, s);
    float vwc[NV];
    vwc[0] = 0.f;
#pragma unroll
    for (int i = 0; i < NB; ++i) vwc[i + 1] = vwc[i] + (s.v[i] + s.v[i + 1]) * 0.5f * s.w[i];
    int cnt = 0;
#pragma unroll
    for (int j = 0; j < NV; ++j) cnt += (vwc[j] <= yy) ? 1 : 0;  // last vertex whose cumulated area <= y (flow.py:443-457)
    int e = min(max(cnt - 1, 0), NB - 1);
    float we = 0.f, ve = 0.f, ve1 = 0.f, wsh = 0.f, vwe = 0.f;
#pragma unroll
    for (int i = 0; i < NB; ++i)
        if (i == e) { we = s.w[i]; ve = s.v[i]; ve1 = s.v[i + 1]; wsh = i == 0 ? 0.f : s.ws[i > 0 ? i - 1 : 0]; vwe = vwc[i]; }
    float a = (ve1 - ve) * we;
    const float b = ve * we;
    const float c = vwe - yy;
    if (fabsf(a) < eps) a = eps;
    const float d = fmaxf(b * b - 2.f * a * c, 0.f);
    const float sq = sqrtf(d);
    const float sol1 = (-b - sq) / a, sol2 = (-b + sq) / a;
    float sol = (sol1 >= 0.f && sol1 < 1.f) ? sol1 : sol2;
    sol = fminf(fmaxf(sol, eps), 1.f - eps);
    x = fminf(fmaxf(we * sol + wsh, eps), 1.f - eps);
    lj = -logf(lerp_t(ve, ve1, sol));
}

// adjoint of the forward spline: upstream (g_x, g_logj) -> d_y and d_st[21]  (derivation: DESIGN.md, "pwquad adjoint")
__device__ __forceinline__ void pwquad_adjoint(const float* sr, float yy, float gx, float gl, float& d_y, float* d_st) {
    const float eps = FLT_EPSILON;
    Spline s;
    spline_params<true>(sr, s);
    int m = 0;
#pragma unroll
    for (int i = 0; i < NB; ++i) m += (s.ws[i] <= yy) ? 1 : 0;
    m = min(m, NB - 1);
    float wm = 0.f, vm = 0.f, vm1 = 0.f, wsh = 0.f, vw = 0.f, cum_m1 = 0.f;
    {
        float cum = 0.f;
#pragma unroll
        for (int i = 0; i < NB; ++i) {
            if (i == m) { wm = s.w[i]; vm = s.v[i]; vm1 = s.v[i + 1]; wsh = i == 0 ? 0.f : s.ws[i > 0 ? i - 1 : 0]; cum_m1 = cum; }
            if (i < m) vw += (s.v[i] + s.v[i + 1]) * 0.5f * s.w[i];
            cum += s.e[i];
        }
    }
    const float a_raw = (yy - wsh) / wm;
    const float a = fminf(fmaxf(a_raw, 0.f), 1.f);
    const float dv = vm1 - vm;
    const float L = lerp_t(vm, vm1, a);
    const float out_raw = a * a * 0.5f * (dv * wm) + a * vm * wm + vw;
    const float go = (out_raw >= eps && out_raw <= 1.f - eps) ? gx : 0.f;
    // d/d alpha
    float ga = go * wm * (vm + a * dv) + gl * dv / L;
    if (!(a_raw >= 0.f && a_raw <= 1.f)) ga = 0.f;
    float gv[NV], gw[NB];
#pragma unroll
    for (int j = 0; j < NV; ++j) gv[j] = 0.f;
#pragma unroll
    for (int i = 0; i < NB; ++i) gw[i] = 0.f;
    const float gvm = go * (a * wm - a * a * 0.5f * wm) + gl * (1.f - a) / L;
    const float gvm1 = go * (a * a * 0.5f * wm) + gl * a / L;
    const float gwm = go * (a * a * 0.5f * dv + a * vm) - ga * a_raw / wm;
    const float gwsh = -ga / wm;
#pragma unroll
    for (int i = 0; i < NB; ++i) {
        if (i == m) { gv[i] += gvm; gv[i + 1] += gvm1; gw[i] += gwm; }
        if (i < m) { gv[i] += go * 0.5f * s.w[i]; gv[i + 1] += go * 0.5f * s.w[i]; gw[i] += go * (s.v[i] + s.v[i + 1]) * 0.5f; }
    }
    d_y = ga / wm;
    // v = max(u / Z, 1e-6)
    float gu[NV];
    float gZ = 0.f;
#pragma unroll
    for (int j = 0; j < NV; ++j) {
        const float g = s.vr[j] >= 1e-6f ? gv[j] : 0.f;
        gu[j] = g / s.Z;
        gZ -= g * s.vr[j] / s.Z;
    }
#pragma unroll
    for (int i = 0; i < NB; ++i) {
        gu[i] += gZ * 0.5f * s.w[i];
        gu[i + 1] += gZ * 0.5f * s.w[i];
        gw[i] += gZ * (s.u[i] + s.u[i + 1]) * 0.5f;
    }
#pragma unroll
    for (int j = 0; j < NV; ++j) d_st[j] = gu[j] * s.u[j];
    // w = max(e / S, 1e-6), wshift_m = cum_{m-1} / S
    float ge[NB];
    float gS = 0.f;
#pragma unroll
    for (int i = 0; i < NB; ++i) {
        const float g = s.wr[i] >= 1e-6f ? gw[i] : 0.f;
        ge[i] = g / s.S;
        gS -= g * s.wr[i] / s.S;
    }
    if (m > 0) {
        gS -= gwsh * cum_m1 / (s.S * s.S);
#pragma unroll
        for (int i = 0; i < NB; ++i)
            if (i < m) ge[i] += gwsh / s.S;
    }
#pragma unroll
    for (int i = 0; i < NB; ++i) {
        const float ex = expf(sr[NV + i]);
        d_st[NV + i] = ex >= 1e-6f ? (ge[i] + gS) * ex : 0.f;
    }
}


}  // namespace flowsp
