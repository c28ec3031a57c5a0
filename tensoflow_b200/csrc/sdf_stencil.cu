// Fused TensoSDF query: VM gather (3 trilinear plane x 3 line fetches) -> decoder MLP
// (Linear -> Softplus(beta=100) -> Linear) for the sample and its six finite-difference
// taps, in one kernel, with no [N,F] intermediate in HBM.
// Replaces TensoSDF.forward + TensoSDF.gradient of the reference
// (network/fields.py:262-299, :227-260), i.e. 7 x (6 dr.texture + 2 GEMM) launches.
//
// v1 arithmetic: fp32 FFMA register-tiled GEMMs out of shared memory (parity first;
// see DESIGN.md for the tcgen05 plan).  Tiling:
//   CTA = 256 threads, tile = TS=16 samples -> R = 7*16 = 112 query rows (row = q*16 + s)
//   A tile   : [R][KP] features (+ raw xyz, zero padded), gathered once per tile
//   hidden   : processed in chunks of NC=32 units; thread (s = tid/16, tx = tid%16) owns
//              the 7 stencil rows of sample s x 2 hidden units -> the stencil is thread local
//   GEMM2    : centre rows only ([16][NC] x [NC][A]); taps need output 0 only (a dot product)
#include "common.cuh"
#include "internal.cuh"

namespace {

constexpr int TS = 16;       // samples per tile (stencil mode)
constexpr int NQ = 7;        // stencil queries
constexpr int R = TS * NQ;   // rows per tile
constexpr int NC = 32;       // hidden units per chunk
constexpr int NT = 256;      // threads per CTA
constexpr int HCS = NC + 2;  // row stride of the centre-hidden tile

__host__ __device__ inline int round_up4(int x) { return (x + 3) & ~3; }

// ---- weight re-layout (tiny, once per call) ------------------------------------------
//   W0T [KP][H]  : k-major copy of W0 (zero padded rows K..KP-1)     -> GEMM1 B operand
//   W0P [H][KP]  : row-major padded copy of W0                        -> dA = dPre . W0
//   W1T [H][A]   : h-major copy of W1 rows 1..A                       -> GEMM2 B operand
__global__ void prep_weights_kernel(const float* __restrict__ W0, const float* __restrict__ W1, int K, int KP, int H, int A,
                                    float* __restrict__ W0T, float* __restrict__ W0P, float* __restrict__ W1T) {
    const int tid = blockIdx.x * blockDim.x + threadIdx.x, nth = gridDim.x * blockDim.x;
    for (int i = tid; i < KP * H; i += nth) {
        const int k = i / H, h = i % H;
        W0T[i] = k < K ? W0[h * K + k] : 0.f;
    }
    for (int i = tid; i < H * KP; i += nth) {
        const int h = i / KP, k = i % KP;
        W0P[i] = k < K ? W0[h * K + k] : 0.f;
    }
    for (int i = tid; i < H * A; i += nth) {
        const int h = i / A, o = i % A;
        W1T[i] = W1[(1 + o) * H + h];
    }
}

struct StencilParams {
    tf_vm_field_t f;
    const float* xyz;
    const float* level;
    int64_t n;        // samples in this launch
    const float* W0T; const float* W0P; const float* W1T;
    const float* b0; const float* W1; const float* b1;
    int K, KP, KS, H, A;
    float units[3];
    // forward outputs
    float* sdf7; float* feat; float* grad; float* hess; float* sdf1;
    // backward inputs
    const float* sdf7_in; const float* g_sdf; const float* g_feat; const float* g_grad; const float* g_hess;
    // backward outputs
    tf_vm_mut_t g;
    float* dpre;   // [tiles*R][H]
    float* arow;   // [tiles*R][KP]
    float* spc;    // [tiles*TS][H]  softplus hidden of the centre rows
    float* db0; float* dW1r0; float* db1;   // accumulated atomically
};

// gather the feature rows of one tile into shared memory.
// MODE 0: stencil rows (row = q*TS + s, sample = tile*TS + s); MODE 1: R plain rows (sample = tile*R + row)
template <int MODE>
__device__ __forceinline__ void gather_tile(const StencilParams& p, int64_t tile, float* As) {
    const int C = p.f.n_comp, C4 = C / 4, KS = p.KS, F = 3 * C;
    const bool has_level = p.level != nullptr;
    for (int it = threadIdx.x; it < R * 3 * C4; it += NT) {
        const int c = (it % C4) * 4;
        const int i = (it / C4) % 3;
        const int row = it / (3 * C4);
        const int64_t n = MODE == 0 ? tile * TS + (row % TS) : tile * R + row;
        float4 v = f4_zero();
        if (n < p.n) {
            const float x[3] = {p.xyz[n * 3 + 0], p.xyz[n * 3 + 1], p.xyz[n * 3 + 2]};
            float q[3];
            stencil_point(x, p.units, MODE == 0 ? row / TS : 0, q);
            float4 P, L;
            vm_sample(p.f, q, has_level ? p.level[n] : 0.f, has_level, i, c, P, L);
            v = f4_mul(P, L);
        }
        *reinterpret_cast<float4*>(As + row * KS + i * C + c) = v;
    }
    const int tail = p.KP - F;   // raw xyz (fields.py:265,298) + zero padding
    for (int it = threadIdx.x; it < R * tail; it += NT) {
        const int row = it / tail, c = it % tail;
        const int64_t n = MODE == 0 ? tile * TS + (row % TS) : tile * R + row;
        float v = 0.f;
        if (n < p.n && c < 3) {
            v = p.xyz[n * 3 + c];
            if (MODE == 0) {
                const int qi = row / TS;
                if (qi > 0 && ((qi - 1) >> 1) == c) v = v + (((qi - 1) & 1) ? -p.units[c] : p.units[c]);
            }
        }
        As[row * KS + F + c] = v;
    }
}

// acc[r][c] = sum_k As[row_r][k] * W0s[k][tx*2+c]   for the thread's 7 rows
__device__ __forceinline__ void gemm1_chunk(const float* __restrict__ As, const float* __restrict__ W0s, int KP, int KS, int s,
                                            int tx, float acc[NQ][2]) {
#pragma unroll
    for (int r = 0; r < NQ; ++r) { acc[r][0] = 0.f; acc[r][1] = 0.f; }
    for (int k = 0; k < KP; k += 4) {
        float4 a[NQ];
#pragma unroll
        for (int r = 0; r < NQ; ++r) a[r] = *reinterpret_cast<const float4*>(As + (r * TS + s) * KS + k);
        const float2 w0 = *reinterpret_cast<const float2*>(W0s + (k + 0) * NC + tx * 2);
        const float2 w1 = *reinterpret_cast<const float2*>(W0s + (k + 1) * NC + tx * 2);
        const float2 w2 = *reinterpret_cast<const float2*>(W0s + (k + 2) * NC + tx * 2);
        const float2 w3 = *reinterpret_cast<const float2*>(W0s + (k + 3) * NC + tx * 2);
#pragma unroll
        for (int r = 0; r < NQ; ++r) {
            acc[r][0] = fmaf(a[r].x, w0.x, acc[r][0]); acc[r][1] = fmaf(a[r].x, w0.y, acc[r][1]);
            acc[r][0] = fmaf(a[r].y, w1.x, acc[r][0]); acc[r][1] = fmaf(a[r].y, w1.y, acc[r][1]);
            acc[r][0] = fmaf(a[r].z, w2.x, acc[r][0]); acc[r][1] = fmaf(a[r].z, w2.y, acc[r][1]);
            acc[r][0] = fmaf(a[r].w, w3.x, acc[r][0]); acc[r][1] = fmaf(a[r].w, w3.y, acc[r][1]);
        }
    }
}

__device__ __forceinline__ void load_w0_chunk(const float* __restrict__ W0T, int H, int KP, int n0, float* W0s) {
    for (int i = threadIdx.x; i < KP * (NC / 4); i += NT) {
        const int k = i / (NC / 4), j = (i % (NC / 4)) * 4;
        *reinterpret_cast<float4*>(W0s + k * NC + j) = ldg4(W0T + (size_t)k * H + n0 + j);
    }
}

__device__ __forceinline__ float half_warp_sum(float v) {
    v += __shfl_xor_sync(0xffffffffu, v, 8);
    v += __shfl_xor_sync(0xffffffffu, v, 4);
    v += __shfl_xor_sync(0xffffffffu, v, 2);
    v += __shfl_xor_sync(0xffffffffu, v, 1);
    return v;
}

// ---- forward ---------------------------------------------------------------------------
// MODE 0: full stencil (sdf7 + feat + grad + hess).  MODE 1: SDF only, R samples per tile.
template <int MODE>
__global__ void __launch_bounds__(NT, 2) sdf_stencil_fwd_kernel(StencilParams p) {
    extern __shared__ __align__(16) float smem[];
    const int KP = p.KP, KS = p.KS, H = p.H, A = p.A;
    float* As = smem;                       // [R][KS]
    float* W0s = As + R * KS;               // [KP][NC]
    float* W1s = W0s + KP * NC;             // [NC][A]      (MODE 0)
    float* Hc = W1s + NC * A;               // [TS][HCS]    (MODE 0)
    const int s = threadIdx.x / 16, tx = threadIdx.x % 16;
    const int64_t per_tile = MODE == 0 ? TS : R;
    const int64_t ntiles = (p.n + per_tile - 1) / per_tile;

    for (int64_t tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
        gather_tile<MODE>(p, tile, As);
        float psum[NQ];
#pragma unroll
        for (int r = 0; r < NQ; ++r) psum[r] = 0.f;
        float acc2[2][4];
#pragma unroll
        for (int g = 0; g < 2; ++g) { acc2[g][0] = acc2[g][1] = acc2[g][2] = acc2[g][3] = 0.f; }

        for (int n0 = 0; n0 < H; n0 += NC) {
            load_w0_chunk(p.W0T, H, KP, n0, W0s);
            if (MODE == 0 && p.feat) {
                for (int i = threadIdx.x; i < NC * (A / 4); i += NT) {
                    const int j = i / (A / 4), o = (i % (A / 4)) * 4;
                    *reinterpret_cast<float4*>(W1s + j * A + o) = ldg4(p.W1T + (size_t)(n0 + j) * A + o);
                }
            }
            __syncthreads();   // A tile + weight chunks visible
            float acc[NQ][2];
            gemm1_chunk(As, W0s, KP, KS, s, tx, acc);
            const float2 b = *reinterpret_cast<const float2*>(p.b0 + n0 + tx * 2);
            const float2 w1 = *reinterpret_cast<const float2*>(p.W1 + n0 + tx * 2);   // row 0 of W1
#pragma unroll
            for (int r = 0; r < NQ; ++r) {
                const float h0 = softplus100(acc[r][0] + b.x), h1 = softplus100(acc[r][1] + b.y);
                psum[r] = fmaf(h0, w1.x, fmaf(h1, w1.y, psum[r]));
                if (MODE == 0 && r == 0 && p.feat) *reinterpret_cast<float2*>(Hc + s * HCS + tx * 2) = make_float2(h0, h1);
            }
            if (MODE == 0 && p.feat) {
                __syncthreads();   // centre hidden visible
#pragma unroll 4
                for (int j = 0; j < NC; ++j) {
                    const float h = Hc[s * HCS + j];
#pragma unroll
                    for (int g = 0; g < 2; ++g) {
                        const int o = (tx + 16 * g) * 4;
                        if (o < A) {
                            const float4 w = *reinterpret_cast<const float4*>(W1s + j * A + o);
                            acc2[g][0] = fmaf(h, w.x, acc2[g][0]); acc2[g][1] = fmaf(h, w.y, acc2[g][1]);
                            acc2[g][2] = fmaf(h, w.z, acc2[g][2]); acc2[g][3] = fmaf(h, w.w, acc2[g][3]);
                        }
                    }
                }
            }
            __syncthreads();   // everyone done with this chunk's shared tiles
        }

        // reduce the W1[0,:] dot over the 16 threads that share the rows
#pragma unroll
        for (int r = 0; r < NQ; ++r) psum[r] = half_warp_sum(psum[r]) + __ldg(p.b1);

        if (MODE == 0) {
            const int64_t n = tile * TS + s;
            if (n < p.n) {
                if (tx == 0) {
#pragma unroll
                    for (int r = 0; r < NQ; ++r) p.sdf7[n * NQ + r] = psum[r];
                    float g[3], h[3];
#pragma unroll
                    for (int k = 0; k < 3; ++k) {
                        const float e = p.units[k];
                        g[k] = (psum[1 + 2 * k] - psum[2 + 2 * k]) / (2.f * e);
                        h[k] = (psum[1 + 2 * k] + psum[2 + 2 * k] - 2.f * psum[0]) / (e * e);
                    }
                    if (p.grad) { p.grad[n * 3 + 0] = g[0]; p.grad[n * 3 + 1] = g[1]; p.grad[n * 3 + 2] = g[2]; }
                    if (p.hess) p.hess[n] = (g[0] * h[0] + g[1] * h[1] + g[2] * h[2]) / (g[0] * g[0] + g[1] * g[1] + g[2] * g[2] + 1e-5f);
                }
                if (p.feat) {
#pragma unroll
                    for (int g = 0; g < 2; ++g) {
                        const int o = (tx + 16 * g) * 4;
                        if (o < A) {
                            float4 v = make_float4(acc2[g][0] + __ldg(p.b1 + 1 + o), acc2[g][1] + __ldg(p.b1 + 2 + o),
                                                   acc2[g][2] + __ldg(p.b1 + 3 + o), acc2[g][3] + __ldg(p.b1 + 4 + o));
                            *reinterpret_cast<float4*>(p.feat + n * A + o) = v;
                        }
                    }
                }
            }
        } else {
            if (tx == 0) {
#pragma unroll
                for (int r = 0; r < NQ; ++r) {
                    const int64_t n = tile * R + r * TS + s;
                    if (n < p.n) p.sdf1[n] = psum[r];
                }
            }
        }
        // the next tile's gather overwrites As: all reads of As ended before the last __syncthreads
    }
}

// ---- backward, activation side -----------------------------------------------------------
// Per tile: regather A, recompute hidden chunk by chunk, form dPre, accumulate
// dA = dPre . W0 in registers, then scatter dA into the plane/line gradients.
// dPre, A and the centre hidden activations are streamed to the workspace for the
// weight-gradient GEMMs (tf_internal_xty, mlp.cu).
constexpr int DSS = NC + 4;   // row stride of the dPre chunk tile (float4 aligned)

__global__ void __launch_bounds__(NT, 1) sdf_stencil_bwd_kernel(StencilParams p) {
    extern __shared__ __align__(16) float smem[];
    const int KP = p.KP, KS = p.KS, H = p.H, A = p.A, C = p.f.n_comp;
    float* As = smem;                       // [R][KS]   (reused for dA at the end)
    float* W0s = As + R * KS;               // [KP][NC]  k-major chunk (GEMM1)
    float* W0c = W0s + KP * NC;             // [NC][KS]  row-major chunk (dA)
    float* Ds = W0c + NC * KS;              // [R][DSS]  dPre chunk
    float* Gs = Ds + R * DSS;               // [TS][A]   upstream feature grads
    float* W1c = Gs + TS * A;               // [1+A][NC] W1 columns n0..n0+NC
    float* gs7 = W1c + (1 + A) * NC;        // [NQ][TS]  upstream grads of the 7 sdf values
    float* accb0 = gs7 + NQ * TS;           // [H]       per-CTA db0
    float* accw1 = accb0 + H;               // [H]       per-CTA dW1[0,:]
    float* accb1 = accw1 + H;               // [1]
    const int s = threadIdx.x / 16, tx = threadIdx.x % 16;
    const int64_t ntiles = (p.n + TS - 1) / TS;
    const int NKI = (KP + 15) / 16;         // k values per thread in the dA tile (k = tx + 16*i)

    for (int i = threadIdx.x; i < 2 * H + 1; i += NT) accb0[i] = 0.f;

    for (int64_t tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
        __syncthreads();   // previous tile's scatter finished reading As/dA
        gather_tile<0>(p, tile, As);
        // upstream grads -> per-query sdf grads (adjoint of fields.py:245-256)
        if (threadIdx.x < TS) {
            const int ss = threadIdx.x;
            const int64_t n = tile * TS + ss;
            float gq[NQ];
#pragma unroll
            for (int r = 0; r < NQ; ++r) gq[r] = 0.f;
            if (n < p.n) {
                float sd[NQ];
#pragma unroll
                for (int r = 0; r < NQ; ++r) sd[r] = p.sdf7_in[n * NQ + r];
                float g[3], h[3];
#pragma unroll
                for (int k = 0; k < 3; ++k) {
                    const float e = p.units[k];
                    g[k] = (sd[1 + 2 * k] - sd[2 + 2 * k]) / (2.f * e);
                    h[k] = (sd[1 + 2 * k] + sd[2 + 2 * k] - 2.f * sd[0]) / (e * e);
                }
                const float D = g[0] * g[0] + g[1] * g[1] + g[2] * g[2] + 1e-5f;
                const float nh = (g[0] * h[0] + g[1] * h[1] + g[2] * h[2]) / D;
                const float gh = p.g_hess ? p.g_hess[n] : 0.f;
                gq[0] = p.g_sdf ? p.g_sdf[n] : 0.f;
#pragma unroll
                for (int k = 0; k < 3; ++k) {
                    const float e = p.units[k];
                    const float Gk = (p.g_grad ? p.g_grad[n * 3 + k] : 0.f) + gh * (h[k] / D - 2.f * g[k] * nh / D);
                    const float Hk = gh * g[k] / D;
                    gq[1 + 2 * k] = Gk / (2.f * e) + Hk / (e * e);
                    gq[2 + 2 * k] = -Gk / (2.f * e) + Hk / (e * e);
                    gq[0] -= 2.f * Hk / (e * e);
                }
            }
            float tot = 0.f;
#pragma unroll
            for (int r = 0; r < NQ; ++r) { gs7[r * TS + ss] = gq[r]; tot += gq[r]; }
            if (tot != 0.f) atomicAdd(accb1, tot);
        }
        for (int i = threadIdx.x; i < TS * (A / 4); i += NT) {
            const int ss = i / (A / 4), o = (i % (A / 4)) * 4;
            const int64_t n = tile * TS + ss;
            float4 v = f4_zero();
            if (n < p.n && p.g_feat) v = ldg4(p.g_feat + n * A + o);
            *reinterpret_cast<float4*>(Gs + ss * A + o) = v;
        }
        __syncthreads();
        // stream the A tile to the workspace for dW0 = dPre^T A
        for (int i = threadIdx.x; i < R * (KP / 4); i += NT) {
            const int row = i / (KP / 4), k = (i % (KP / 4)) * 4;
            *reinterpret_cast<float4*>(p.arow + ((size_t)tile * R + row) * KP + k) = *reinterpret_cast<const float4*>(As + row * KS + k);
        }

        float dA[NQ][7];
#pragma unroll
        for (int r = 0; r < NQ; ++r)
#pragma unroll
            for (int i = 0; i < 7; ++i) dA[r][i] = 0.f;
        float gq[NQ];
#pragma unroll
        for (int r = 0; r < NQ; ++r) gq[r] = gs7[r * TS + s];

        for (int n0 = 0; n0 < H; n0 += NC) {
            load_w0_chunk(p.W0T, H, KP, n0, W0s);
            for (int i = threadIdx.x; i < NC * (KP / 4); i += NT) {
                const int j = i / (KP / 4), k = (i % (KP / 4)) * 4;
                *reinterpret_cast<float4*>(W0c + j * KS + k) = ldg4(p.W0P + (size_t)(n0 + j) * KP + k);
            }
            for (int i = threadIdx.x; i < (1 + A) * (NC / 4); i += NT) {
                const int o = i / (NC / 4), j = (i % (NC / 4)) * 4;
                *reinterpret_cast<float4*>(W1c + o * NC + j) = ldg4(p.W1 + (size_t)o * H + n0 + j);
            }
            __syncthreads();
            float acc[NQ][2];
            gemm1_chunk(As, W0s, KP, KS, s, tx, acc);
            const float2 b = *reinterpret_cast<const float2*>(p.b0 + n0 + tx * 2);
            const float2 w1 = *reinterpret_cast<const float2*>(W1c + tx * 2);   // W1[0, n0 + tx*2 ..]
            // centre rows: dPost = gq0 * W1[0,:] + g_feat . W1[1:,:]
            float dpc0 = gq[0] * w1.x, dpc1 = gq[0] * w1.y;
            if (p.g_feat) {
                for (int o = 0; o < A; o += 4) {
                    const float4 gf = *reinterpret_cast<const float4*>(Gs + s * A + o);
                    const float2 u0 = *reinterpret_cast<const float2*>(W1c + (1 + o) * NC + tx * 2);
                    const float2 u1 = *reinterpret_cast<const float2*>(W1c + (2 + o) * NC + tx * 2);
                    const float2 u2 = *reinterpret_cast<const float2*>(W1c + (3 + o) * NC + tx * 2);
                    const float2 u3 = *reinterpret_cast<const float2*>(W1c + (4 + o) * NC + tx * 2);
                    dpc0 = fmaf(gf.x, u0.x, fmaf(gf.y, u1.x, fmaf(gf.z, u2.x, fmaf(gf.w, u3.x, dpc0))));
                    dpc1 = fmaf(gf.x, u0.y, fmaf(gf.y, u1.y, fmaf(gf.z, u2.y, fmaf(gf.w, u3.y, dpc1))));
                }
            }
            float sb0 = 0.f, sb1 = 0.f, sw0 = 0.f, sw1 = 0.f;
#pragma unroll
            for (int r = 0; r < NQ; ++r) {
                const float pre0 = acc[r][0] + b.x, pre1 = acc[r][1] + b.y;
                const float h0 = softplus100(pre0), h1 = softplus100(pre1);
                const float dp0 = (r == 0 ? dpc0 : gq[r] * w1.x) * softplus100_grad(pre0);
                const float dp1 = (r == 0 ? dpc1 : gq[r] * w1.y) * softplus100_grad(pre1);
                *reinterpret_cast<float2*>(Ds + (r * TS + s) * DSS + tx * 2) = make_float2(dp0, dp1);
                *reinterpret_cast<float2*>(p.dpre + ((size_t)tile * R + r * TS + s) * H + n0 + tx * 2) = make_float2(dp0, dp1);
                sb0 += dp0; sb1 += dp1;
                sw0 = fmaf(gq[r], h0, sw0); sw1 = fmaf(gq[r], h1, sw1);
                if (r == 0) *reinterpret_cast<float2*>(p.spc + ((size_t)tile * TS + s) * H + n0 + tx * 2) = make_float2(h0, h1);
            }
            // db0 / dW1[0,:] partials: combine the two samples of this warp, then shared atomics
            sb0 += __shfl_xor_sync(0xffffffffu, sb0, 16); sb1 += __shfl_xor_sync(0xffffffffu, sb1, 16);
            sw0 += __shfl_xor_sync(0xffffffffu, sw0, 16); sw1 += __shfl_xor_sync(0xffffffffu, sw1, 16);
            if ((threadIdx.x & 16) == 0) {
                atomicAdd(accb0 + n0 + tx * 2, sb0); atomicAdd(accb0 + n0 + tx * 2 + 1, sb1);
                atomicAdd(accw1 + n0 + tx * 2, sw0); atomicAdd(accw1 + n0 + tx * 2 + 1, sw1);
            }
            __syncthreads();   // dPre chunk visible
            // dA[row][k] += sum_j Ds[row][j] * W0c[j][k],  k = tx + 16*i
            for (int j = 0; j < NC; j += 4) {
                float4 d[NQ];
#pragma unroll
                for (int r = 0; r < NQ; ++r) d[r] = *reinterpret_cast<const float4*>(Ds + (r * TS + s) * DSS + j);
#pragma unroll
                for (int i = 0; i < 7; ++i) {
                    if (i < NKI) {
                        const int k = tx + 16 * i;
                        if (k < KP) {
                            const float wa = W0c[(j + 0) * KS + k], wb = W0c[(j + 1) * KS + k];
                            const float wc = W0c[(j + 2) * KS + k], wd = W0c[(j + 3) * KS + k];
#pragma unroll
                            for (int r = 0; r < NQ; ++r)
                                dA[r][i] = fmaf(d[r].x, wa, fmaf(d[r].y, wb, fmaf(d[r].z, wc, fmaf(d[r].w, wd, dA[r][i]))));
                        }
                    }
                }
            }
            __syncthreads();   // chunk tiles free
        }

        // dA -> shared (over the A tile), then scatter into plane / line gradients
#pragma unroll
        for (int r = 0; r < NQ; ++r)
#pragma unroll
            for (int i = 0; i < 7; ++i) {
                const int k = tx + 16 * i;
                if (i < NKI && k < KP) As[(r * TS + s) * KS + k] = dA[r][i];
            }
        __syncthreads();
        const int C4 = C / 4;
        const bool has_level = p.level != nullptr;
        for (int it = threadIdx.x; it < R * 3 * C4; it += NT) {
            const int c = (it % C4) * 4;
            const int i = (it / C4) % 3;
            const int row = it / (3 * C4);
            const int64_t n = tile * TS + (row % TS);
            if (n >= p.n) continue;
            const float x[3] = {p.xyz[n * 3 + 0], p.xyz[n * 3 + 1], p.xyz[n * 3 + 2]};
            float q[3];
            stencil_point(x, p.units, row / TS, q);
            const float lv = has_level ? p.level[n] : 0.f;
            float4 P, L;
            vm_sample(p.f, q, lv, has_level, i, c, P, L);
            const float4 d = *reinterpret_cast<const float4*>(As + row * KS + i * C + c);
            vm_scatter(p.f, p.g, q, lv, has_level, i, c, f4_mul(d, L), f4_mul(d, P));
        }
    }
    __syncthreads();
    for (int i = threadIdx.x; i < H; i += NT) {
        if (accb0[i] != 0.f) atomicAdd(p.db0 + i, accb0[i]);
        if (accw1[i] != 0.f) atomicAdd(p.dW1r0 + i, accw1[i]);
    }
    if (threadIdx.x == 0 && accb1[0] != 0.f) atomicAdd(p.db1, accb1[0]);
}

struct Dims { int C, K, KP, KS, KT, H, A; };   // KT: K rounded up to the tensor-core K slice (16)

int check_mlp(const tf_vm_field_t* f, const tf_sdf_mlp_t* m, Dims& d) {
    TF_REQUIRE(m && m->W0 && m->b0 && m->W1 && m->b1, "MLP descriptor / weights are NULL");
    TF_REQUIRE(m->hidden > 0 && m->hidden % NC == 0, "hidden must be a multiple of %d (got %d)", NC, m->hidden);
    TF_REQUIRE(m->app_dim >= 4 && m->app_dim % 4 == 0 && m->app_dim <= 128, "app_dim must be a multiple of 4 in [4,128] (got %d)", m->app_dim);
    TF_REQUIRE(f->n_comp <= 36, "n_comp <= 36 supported by the fused stencil (got %d)", f->n_comp);
    d.C = f->n_comp; d.K = 3 * d.C + 3; d.KP = round_up4(d.K); d.KS = d.KP + 4; d.KT = (d.K + 15) / 16 * 16;
    d.H = m->hidden; d.A = m->app_dim;
    return 0;
}

size_t weights_ws_floats(const Dims& d) { return (size_t)2 * d.KP * d.H + (size_t)d.H * d.A; }

size_t fwd_smem(const Dims& d, bool feat) {
    return sizeof(float) * ((size_t)R * d.KS + (size_t)d.KP * NC + (feat ? (size_t)NC * d.A + TS * HCS : 0));
}
size_t bwd_smem(const Dims& d) {
    return sizeof(float) * ((size_t)R * d.KS + (size_t)d.KP * NC + (size_t)NC * d.KS + (size_t)R * DSS + (size_t)TS * d.A +
                            (size_t)(1 + d.A) * NC + NQ * TS + 2 * d.H + 4);
}

void fill_common(StencilParams& p, const tf_vm_field_t* f, const tf_sdf_mlp_t* m, const Dims& d, const float* xyz,
                 const float* level, int64_t n, const float units[3], float* ws) {
    p.f = *f; p.xyz = xyz; p.level = level; p.n = n;
    p.W0T = ws; p.W0P = ws + (size_t)d.KP * d.H; p.W1T = ws + (size_t)2 * d.KP * d.H;
    p.b0 = m->b0; p.W1 = m->W1; p.b1 = m->b1;
    p.K = d.K; p.KP = d.KP; p.KS = d.KS; p.H = d.H; p.A = d.A;
    p.units[0] = units ? units[0] : 0.f; p.units[1] = units ? units[1] : 0.f; p.units[2] = units ? units[2] : 0.f;
}

}  // namespace

// Which decoder shapes run on the tcgen05 kernels; the FFMA kernels above take the others (hidden > 256).  check_mlp and
// tf_check_field already bound the rest: hidden % 32 == 0, n_comp % 4 == 0 and n_comp <= 36, so KT <= 112.
static bool fwd_on_tc(const Dims& d) { return tf_internal_stencil_fwd_tc_ok(d.KT, d.H); }
// the tcgen05 backward reads the centre hidden activations that the tcgen05 forward kept
static bool bwd_on_tc(const Dims& d) { return fwd_on_tc(d) && tf_internal_bwd_tc_smem(d.KT, d.H) <= 227 * 1024; }

static size_t fwd_ws_floats(const Dims& d, int64_t n, bool with_feat) {
    if (!fwd_on_tc(d)) return weights_ws_floats(d);
    return tf_internal_tc_w0_floats(d.KT, d.H) + (with_feat ? (size_t)(n < 1 ? 1 : n) * d.H + tf_internal_linear_tc_ws_floats(d.H, d.A) : 0);
}

extern "C" TF_API size_t tf_sdf_stencil_fwd_workspace(const tf_vm_field_t* f, const tf_sdf_mlp_t* m, int64_t n, int32_t with_feat) {
    Dims d;
    if (!f || !m || check_mlp(f, m, d)) return 0;
    return fwd_ws_floats(d, n, with_feat != 0) * sizeof(float);
}

static int stencil_fwd_impl(int mode, const tf_vm_field_t* f, const tf_sdf_mlp_t* m, const float* xyz, const float* level,
                            int64_t n, const float units[3], float* sdf7, float* feat, float* grad, float* hess, float* sdf1,
                            void* workspace, size_t ws_bytes, tf_stream_t stream_) {
    if (int e = tf_check_field(f, level != nullptr)) return e;
    Dims d;
    if (int e = check_mlp(f, m, d)) return e;
    if (n == 0) return 0;
    TF_REQUIRE(xyz, "xyz is NULL");
    TF_REQUIRE(workspace && ws_bytes >= fwd_ws_floats(d, n, feat != nullptr) * sizeof(float), "workspace too small (%zu bytes)", ws_bytes);
    TF_REQUIRE(((uintptr_t)workspace & 15) == 0, "workspace not 16-byte aligned");
    if (feat) TF_REQUIRE(((uintptr_t)feat & 15) == 0, "feat not 16-byte aligned");
    cudaStream_t stream = (cudaStream_t)stream_;
    if (fwd_on_tc(d)) {
        // tcgen05 path: first layer on the tensor cores, appearance head as one more linear layer
        float* w0tc = (float*)workspace;
        float* spc = feat ? w0tc + tf_internal_tc_w0_floats(d.KT, d.H) : nullptr;
        if (mode == 0) TF_REQUIRE(sdf7, "sdf7 is NULL"); else TF_REQUIRE(sdf1, "sdf is NULL");
        if (int e = tf_internal_stencil_fwd_tc(f, m, xyz, level, n, units, mode == 0 ? 7 : 1, sdf7, grad, hess, sdf1, spc, w0tc, stream)) return e;
        if (feat) {
            // appearance head: feat = hidden(centre) W1[1:,:]^T + b1[1:]
            float* wlin = spc + (size_t)n * d.H;
            // tf_internal_linear_tc_ok holds: K = H <= 256 (fwd_on_tc), N = A <= 128 (check_mlp)
            tf_internal_linear_tc(spc, m->W1 + d.H, d.H, 0, m->b1 + 1, n, d.H, d.A, 0, 0.f, feat, wlin, stream);
        }
        TF_CHECK_LAUNCH("tf_sdf_stencil_fwd (tcgen05)");
        return 0;
    }
    StencilParams p = {};
    fill_common(p, f, m, d, xyz, level, n, units, (float*)workspace);
    p.sdf7 = sdf7; p.feat = feat; p.grad = grad; p.hess = hess; p.sdf1 = sdf1;
    prep_weights_kernel<<<64, 256, 0, stream>>>(m->W0, m->W1, d.K, d.KP, d.H, d.A, (float*)p.W0T, (float*)p.W0P, (float*)p.W1T);
    const int64_t per_tile = mode == 0 ? TS : R;
    const int64_t ntiles = (n + per_tile - 1) / per_tile;
    const int64_t cap = (int64_t)tf_num_sms() * 2;
    const int grid = (int)(ntiles < cap ? ntiles : cap);
    if (mode == 0) {
        TF_REQUIRE(sdf7, "sdf7 is NULL");
        const size_t smem = fwd_smem(d, feat != nullptr);
        cudaFuncSetAttribute(sdf_stencil_fwd_kernel<0>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        sdf_stencil_fwd_kernel<0><<<grid, NT, smem, stream>>>(p);
    } else {
        TF_REQUIRE(sdf1, "sdf is NULL");
        const size_t smem = fwd_smem(d, false);
        cudaFuncSetAttribute(sdf_stencil_fwd_kernel<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        sdf_stencil_fwd_kernel<1><<<grid, NT, smem, stream>>>(p);
    }
    tf_count_launches(2);
    TF_CHECK_LAUNCH("tf_sdf_stencil_fwd");
    return 0;
}

extern "C" TF_API int tf_sdf_stencil_fwd(const tf_vm_field_t* f, const tf_sdf_mlp_t* m, const float* xyz, const float* level,
                                  int64_t n, const float units[3], float* sdf7, float* feat, float* grad, float* hess,
                                  void* workspace, size_t ws_bytes, tf_stream_t stream) {
    TF_REQUIRE(units, "units is NULL");
    return stencil_fwd_impl(0, f, m, xyz, level, n, units, sdf7, feat, grad, hess, nullptr, workspace, ws_bytes, stream);
}

extern "C" TF_API int tf_sdf_only_fwd(const tf_vm_field_t* f, const tf_sdf_mlp_t* m, const float* xyz, const float* level, int64_t n,
                               float* sdf, void* workspace, size_t ws_bytes, tf_stream_t stream) {
    return stencil_fwd_impl(1, f, m, xyz, level, n, nullptr, nullptr, nullptr, nullptr, nullptr, sdf, workspace, ws_bytes, stream);
}

// one query per point with the appearance features (TensoSDF.forward, network/fields.py:262-299, without the FD taps)
extern "C" TF_API int tf_sdf_point_fwd(const tf_vm_field_t* f, const tf_sdf_mlp_t* m, const float* xyz, const float* level, int64_t n,
                                       float* sdf, float* feat, void* workspace, size_t ws_bytes, tf_stream_t stream) {
    Dims d;
    if (!f || !m) { tf_set_error("tf_sdf_point_fwd: NULL descriptor"); return 1; }
    if (int e = check_mlp(f, m, d)) return e;
    TF_REQUIRE(feat, "tf_sdf_point_fwd: feat is NULL (use tf_sdf_only_fwd for the SDF alone)");
    TF_REQUIRE(fwd_on_tc(d), "tf_sdf_point_fwd: only the tensor-core path evaluates single queries with features "
                             "(hidden <= 256); use tf_sdf_stencil_fwd");
    return stencil_fwd_impl(1, f, m, xyz, level, n, nullptr, nullptr, feat, nullptr, nullptr, sdf, workspace, ws_bytes, stream);
}

static size_t bwd_slice_floats(const Dims& d, int64_t n_slice) {
    const int64_t tiles = (n_slice + TS - 1) / TS;
    return (size_t)tiles * ((size_t)R * d.H + (size_t)R * d.KP + (size_t)TS * d.H);
}

// tensor-core backward workspace: [W slices | dW0/db0 staging | per tile of 18 samples: dPre [128,H], A rows [128,KT],
// dHidden(centre) [18,H]]
static size_t bwd_tc_fixed_floats(const Dims& d) {
    return tf_internal_bwd_tc_wtc_floats(d.KT, d.H) + (size_t)d.H * d.KT + tf_internal_linear_tc_ws_floats(d.A, d.H) +
           tf_internal_bwd_tc_scratch_floats(d.KT);
}
static size_t bwd_tc_tile_floats(const Dims& d) {
    return (size_t)128 * (d.H + d.KT) + (size_t)tf_internal_bwd_tc_samples_per_tile() * d.H;
}

extern "C" TF_API size_t tf_sdf_stencil_bwd_workspace(const tf_vm_field_t* f, const tf_sdf_mlp_t* m, int64_t n_slice) {
    Dims d;
    if (!f || !m || check_mlp(f, m, d)) return 0;
    if (n_slice < 1) n_slice = 1;
    if (bwd_on_tc(d)) {
        const int spt = tf_internal_bwd_tc_samples_per_tile();
        return (bwd_tc_fixed_floats(d) + (size_t)((n_slice + spt - 1) / spt) * bwd_tc_tile_floats(d)) * sizeof(float);
    }
    return (weights_ws_floats(d) + bwd_slice_floats(d, n_slice)) * sizeof(float);
}

static int stencil_bwd_tc(const tf_vm_field_t* f, const tf_sdf_mlp_t* m, const Dims& d, const float* xyz, const float* level, int64_t n,
                          const float units[3], const float* sdf7, const float* g_sdf, const float* g_feat, const float* g_grad,
                          const float* g_hess, const tf_vm_mut_t* g_field, const tf_sdf_mlp_grad_t* g_mlp, float* ws, size_t ws_floats,
                          const float* hidden_c, cudaStream_t stream) {
    const int KT = d.KT, H = d.H;
    const int spt = tf_internal_bwd_tc_samples_per_tile();
    const size_t fixed = bwd_tc_fixed_floats(d), per_tile = bwd_tc_tile_floats(d);
    TF_REQUIRE(ws_floats >= fixed + per_tile, "workspace too small (%zu bytes)", ws_floats * sizeof(float));
    int64_t tiles_fit = (int64_t)((ws_floats - fixed) / per_tile);
    const int64_t ntiles_all = (n + spt - 1) / spt;
    if (tiles_fit > ntiles_all) tiles_fit = ntiles_all;
    float* wtc = ws;
    float* tmp = wtc + tf_internal_bwd_tc_wtc_floats(KT, H);
    float* wlin = tmp + (size_t)H * KT;
    float* da_scratch = wlin + tf_internal_linear_tc_ws_floats(d.A, H);
    float* dpre = da_scratch + tf_internal_bwd_tc_scratch_floats(KT);
    float* arow = dpre + (size_t)tiles_fit * 128 * H;
    float* dHc = arow + (size_t)tiles_fit * 128 * KT;
    tf_internal_bwd_tc_prep(m->W0, d.K, KT, H, wtc, stream);
    cudaMemsetAsync(tmp, 0, (size_t)H * KT * sizeof(float), stream);
    for (int64_t t0 = 0; t0 < ntiles_all; t0 += tiles_fit) {
        const int64_t nt = t0 + tiles_fit < ntiles_all ? tiles_fit : ntiles_all - t0;
        const int64_t s0 = t0 * spt;
        const int64_t ns = s0 + nt * spt < n ? nt * spt : n - s0;
        const float* gf = g_feat ? g_feat + s0 * d.A : nullptr;
        // dHidden(centre) = g_feat W1[1:, :]; tf_internal_linear_tc_ok holds: K = A <= 128 (check_mlp), N = H <= 256 (bwd_on_tc)
        if (gf) tf_internal_linear_tc(gf, m->W1 + H, H, 1, nullptr, ns, d.A, H, 0, 0.f, dHc, wlin, stream);
        if (int e = tf_internal_stencil_bwd_tc(f, g_field, m, wtc, xyz + s0 * 3, level ? level + s0 : nullptr, ns, units, sdf7 + s0 * NQ,
                                               g_sdf ? g_sdf + s0 : nullptr, g_grad ? g_grad + s0 * 3 : nullptr,
                                               g_hess ? g_hess + s0 : nullptr, gf ? dHc : nullptr, dpre, arow,
                                               da_scratch, g_mlp->W1, g_mlp->b1, stream))
            return e;
        // [dW0 | db0] staging += dPre^T [A | 1]; the kernel wrote dPre per tile as [H][128] (row fastest: coalesced stores there,
        // no register transpose here)
        TF_REQUIRE(tf_internal_xty_tc_ok(dpre, arow, H, KT), "tensor-core X^T Y does not take this decoder shape (H=%d, KT=%d)", H, KT);
        if (int e = tf_internal_xty_tc_tiled(dpre, arow, nt * 128, H, KT, tmp, KT, d.K + 1, 1, stream)) return e;
        if (gf) {
            // dW1[1:, :] += g_feat^T hidden(centre), from the centre hidden activations kept by the forward call
            tf_internal_xty_auto(gf, hidden_c + s0 * H, ns, d.A, H, g_mlp->W1 + H, stream);
            tf_internal_colsum(gf, d.A, ns, d.A, g_mlp->b1 + 1, stream);
        }
    }
    tf_internal_bwd_tc_fold(tmp, H, d.K, KT, g_mlp->W0, g_mlp->b0, stream);
    TF_CHECK_LAUNCH("tf_sdf_stencil_bwd (tcgen05)");
    return 0;
}

// byte offset of the centre hidden activations [n, hidden] inside the workspace of tf_sdf_stencil_fwd(.., feat != NULL);
// (size_t)-1 exactly when the tcgen05 forward does not apply to this shape (the FFMA forward does not keep them)
extern "C" TF_API size_t tf_sdf_stencil_fwd_hidden_offset(const tf_vm_field_t* f, const tf_sdf_mlp_t* m) {
    Dims d;
    if (!f || !m || check_mlp(f, m, d) || !fwd_on_tc(d)) return (size_t)-1;
    return tf_internal_tc_w0_floats(d.KT, d.H) * sizeof(float);
}

extern "C" TF_API int tf_sdf_stencil_bwd(const tf_vm_field_t* f, const tf_sdf_mlp_t* m, const float* xyz, const float* level,
                                  int64_t n, const float units[3], const float* sdf7, const float* hidden_centre, const float* g_sdf,
                                  const float* g_feat, const float* g_grad, const float* g_hess, const tf_vm_mut_t* g_field,
                                  const tf_sdf_mlp_grad_t* g_mlp, void* workspace, size_t ws_bytes, tf_stream_t stream_) {
    if (int e = tf_check_field(f, level != nullptr)) return e;
    Dims d;
    if (int e = check_mlp(f, m, d)) return e;
    if (n == 0) return 0;
    TF_REQUIRE(xyz && units && sdf7, "xyz/units/sdf7 is NULL");
    TF_REQUIRE(g_field && g_mlp && g_mlp->W0 && g_mlp->b0 && g_mlp->W1 && g_mlp->b1, "gradient descriptors are NULL");
    for (int i = 0; i < 3; ++i) {
        TF_REQUIRE(g_field->plane[i] && g_field->line[i], "gradient buffer %d is NULL", i);
        if (f->n_levels > 1 && level) TF_REQUIRE(g_field->plane_mip[i] && g_field->line_mip[i], "mip gradient buffer %d is NULL", i);
    }
    TF_REQUIRE(((uintptr_t)workspace & 15) == 0, "workspace not 16-byte aligned");
    if (g_feat) TF_REQUIRE(((uintptr_t)g_feat & 15) == 0, "g_feat not 16-byte aligned");
    cudaStream_t stream = (cudaStream_t)stream_;
    float* ws = (float*)workspace;
    TF_REQUIRE(workspace, "workspace is NULL");
    if (bwd_on_tc(d)) {
        TF_REQUIRE(hidden_centre || !g_feat, "tf_sdf_stencil_bwd: hidden_centre is NULL (keep the forward workspace: "
                                             "tf_sdf_stencil_fwd_hidden_offset)");
        TF_REQUIRE(((uintptr_t)hidden_centre & 15) == 0, "hidden_centre not 16-byte aligned");
        return stencil_bwd_tc(f, m, d, xyz, level, n, units, sdf7, g_sdf, g_feat, g_grad, g_hess, g_field, g_mlp, ws,
                              ws_bytes / sizeof(float), hidden_centre, stream);
    }
    const size_t wfl = weights_ws_floats(d);
    TF_REQUIRE(ws_bytes >= (wfl + bwd_slice_floats(d, TS)) * sizeof(float), "workspace too small (%zu bytes)", ws_bytes);
    // samples per slice that fit the workspace (multiple of TS)
    const size_t per_tile = (size_t)R * d.H + (size_t)R * d.KP + (size_t)TS * d.H;
    int64_t tiles_fit = (int64_t)((ws_bytes / sizeof(float) - wfl) / per_tile);
    const int64_t ntiles_all = (n + TS - 1) / TS;
    if (tiles_fit > ntiles_all) tiles_fit = ntiles_all;
    const size_t smem = bwd_smem(d);
    cudaFuncSetAttribute(sdf_stencil_bwd_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    StencilParams p = {};
    fill_common(p, f, m, d, xyz, level, n, units, ws);
    prep_weights_kernel<<<64, 256, 0, stream>>>(m->W0, m->W1, d.K, d.KP, d.H, d.A, (float*)p.W0T, (float*)p.W0P, (float*)p.W1T);
    tf_count_launches(1);
    float* dpre = ws + wfl;
    float* arow = dpre + (size_t)tiles_fit * R * d.H;
    float* spc = arow + (size_t)tiles_fit * R * d.KP;
    for (int64_t t0 = 0; t0 < ntiles_all; t0 += tiles_fit) {
        const int64_t nt = t0 + tiles_fit < ntiles_all ? tiles_fit : ntiles_all - t0;
        const int64_t s0 = t0 * TS;
        const int64_t ns = (s0 + nt * TS < n ? nt * TS : n - s0);
        StencilParams q = p;
        q.xyz = xyz + s0 * 3; q.level = level ? level + s0 : nullptr; q.n = ns;
        q.sdf7_in = sdf7 + s0 * NQ;
        q.g_sdf = g_sdf ? g_sdf + s0 : nullptr; q.g_feat = g_feat ? g_feat + s0 * d.A : nullptr;
        q.g_grad = g_grad ? g_grad + s0 * 3 : nullptr; q.g_hess = g_hess ? g_hess + s0 : nullptr;
        q.g = *g_field;
        q.dpre = dpre; q.arow = arow; q.spc = spc;
        q.db0 = g_mlp->b0; q.dW1r0 = g_mlp->W1; q.db1 = g_mlp->b1;
        const int64_t cap = tf_num_sms();
        const int grid = (int)(nt < cap ? nt : cap);
        sdf_stencil_bwd_kernel<<<grid, NT, smem, stream>>>(q);
        tf_count_launches(1);
        // dW0[h][k] += sum_rows dPre[row][h] * A[row][k]
        tf_internal_xty(dpre, d.H, arow, d.KP, nt * R, d.H, d.K, g_mlp->W0, d.K, stream);
        if (g_feat) {
            // dW1[1+o][h] += sum_n g_feat[n][o] * softplus(hidden_centre)[n][h];  db1[1+o] += sum_n g_feat[n][o]
            tf_internal_xty(q.g_feat, d.A, spc, d.H, ns, d.A, d.H, g_mlp->W1 + d.H, d.H, stream);
            tf_internal_colsum(q.g_feat, d.A, ns, d.A, g_mlp->b1 + 1, stream);
        }
    }
    TF_CHECK_LAUNCH("tf_sdf_stencil_bwd");
    return 0;
}
