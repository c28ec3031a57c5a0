// Fused coupling block of the TensoFlow sampler on the 5th-gen tensor cores (tcgen05 + TMEM), sm_100a.
//
// Contract: tf_flow_block_fwd / tf_flow_block_bwd (include/tensoflow_b200.h, reference network/flow.py:549-641).  The conditioner
// chain [PE(y_c) | feature] -> 64 -> 64 -> 64 -> 21 of a tile of 128 (point, direction) pairs runs as four small GEMMs whose A operand
// never leaves the SM: thread t owns pair t = TMEM lane t; after each layer the accumulator D [128 x 64] is read back
// (tcgen05.ld), bias + LeakyReLU applied, split into tf32 hi | lo and written to TENSOR MEMORY (tcgen05.st) as the A
// operand of the next layer's TS-mode MMAs (3xTF32: hi.hi + hi.lo + lo.hi, fp32-level accuracy).  The weights sit in shared
// memory pre-split in the K-major no-swizzle UMMA layout for the whole kernel (84 KB), the per-point feature part of the first
// layer is added as a per-row bias, the spline runs on the 21 outputs of the last layer in registers.
// Two CTAs share an SM (256 TMEM columns each) so that one CTA's epilogue overlaps the other's MMAs.
#include "common.cuh"
#include "tc_common.cuh"
#include "flow_spline.cuh"
#include "internal.cuh"

namespace {

using namespace flowsp;

constexpr int FH = 64, FPE = 7, FSTP = 24, FTILE = 128, FMAXP = 10, FMAXF = 40;
constexpr int K1 = 8;        // first-layer K: 7 positional-encoding inputs + one zero column
constexpr int N4 = 32;       // last-layer N: 21 spline parameters padded to 32

struct FlowTcParams {
    const float *W1, *b1, *W2, *b2, *W3, *b3, *W4, *b4;
    int F; float scale, offset;
    const float* y_in; const float* logj_in; const float* feat;
    int sn, cond, inverse; int64_t M;
    float* y_out; float* logj_out;
    float* save_h;           // [M][3][64] post-activation h1, h2, h3 (NULL: not kept)
    float* save_st;          // [M][24] spline parameters (NULL: not kept)
};

// W[n][koff + k] (n < n_valid, k < k_valid, row stride ldw) -> K-major no-swizzle B tile [N][K], split hi | lo
__device__ __forceinline__ void fill_b_tile(float* hi, float* lo, const float* __restrict__ W, int ldw, int koff, int N, int K, int n_valid,
                                            int k_valid, int tid, int nth) {
    for (int i = tid; i < N * K; i += nth) {
        const int n = i / K, k = i % K;
        const float v = (n < n_valid && k < k_valid) ? W[(size_t)n * ldw + koff + k] : 0.f;
        const float h = tc::tf32_rn(v);
        const uint32_t off = tc::tile_off_b32(n, k, K / 4) / 4;
        hi[off] = h;
        lo[off] = tc::tf32_rn(v - h);
    }
}

// D[128 x N] = A[128 x K] (TMEM, hi at a_hi, lo at a_lo) * B[N x K]^T (shared memory, hi | lo): 3 * K / 8 MMAs by one thread
__device__ __forceinline__ void issue_layer(uint32_t d, uint32_t a_hi, uint32_t a_lo, const float* b_hi, const float* b_lo, int K, int N) {
    const uint32_t idesc = tc::make_idesc(2, 2, FTILE, N);
    const uint32_t sbo = (uint32_t)(K / 4) * 128;
    const uint64_t bdh = tc::make_smem_desc(tc::smem_u32(b_hi), 128, sbo), bdl = tc::make_smem_desc(tc::smem_u32(b_lo), 128, sbo);
    for (int ks = 0; ks < K / 8; ++ks) {
        const uint64_t h = tc::desc_add(bdh, ks * 256), l = tc::desc_add(bdl, ks * 256);
        tc::mma_tf32_ts(d, a_hi + ks * 8, h, idesc, ks > 0);
        tc::mma_tf32_ts(d, a_hi + ks * 8, l, idesc, 1);
        tc::mma_tf32_ts(d, a_lo + ks * 8, h, idesc, 1);
    }
}

__device__ __forceinline__ float leaky(float x) { return x > 0.f ? x : 0.01f * x; }

__global__ void __launch_bounds__(FTILE, 2) flow_block_fwd_tc_kernel(FlowTcParams p) {
    extern __shared__ __align__(1024) uint8_t fsm_raw[];
    float* sp = reinterpret_cast<float*>(fsm_raw);
    auto carve = [&](int n) { float* r = sp; sp += n; return r; };
    float* b1_hi = carve(FH * K1); float* b1_lo = carve(FH * K1);
    float* b2_hi = carve(FH * FH); float* b2_lo = carve(FH * FH);
    float* b3_hi = carve(FH * FH); float* b3_lo = carve(FH * FH);
    float* b4_hi = carve(N4 * FH); float* b4_lo = carve(N4 * FH);
    float* bias1 = carve(FH); float* bias2 = carve(FH); float* bias3 = carve(FH); float* bias4 = carve(N4);
    float* h1p = carve(FMAXP * FH);
    float* w1b = carve(FMAXF * FH);          // feature part of the first layer, [k][j]
    float* xfs = carve(FMAXP * FMAXF);       // Reshift(feature) of the tile's points
    uint64_t* bar = reinterpret_cast<uint64_t*>(carve(2));
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(carve(2));

    const int tid = threadIdx.x, warp = tid >> 5;
    const int F = p.F, KW1 = FPE + F;
    for (int i = tid; i < F * FH; i += FTILE) { const int k = i / FH, j = i % FH; w1b[i] = p.W1[(size_t)j * KW1 + FPE + k]; }
    fill_b_tile(b1_hi, b1_lo, p.W1, KW1, 0, FH, K1, FH, FPE, tid, FTILE);
    fill_b_tile(b2_hi, b2_lo, p.W2, FH, 0, FH, FH, FH, FH, tid, FTILE);
    fill_b_tile(b3_hi, b3_lo, p.W3, FH, 0, FH, FH, FH, FH, tid, FTILE);
    fill_b_tile(b4_hi, b4_lo, p.W4, FH, 0, N4, FH, NST, FH, tid, FTILE);
    for (int i = tid; i < FH; i += FTILE) { bias1[i] = p.b1[i]; bias2[i] = p.b2[i]; bias3[i] = p.b3[i]; }
    for (int i = tid; i < N4; i += FTILE) bias4[i] = i < NST ? p.b4[i] : 0.f;
    if (warp == 0) tc::tmem_alloc<256>(tmem_slot);
    if (tid == 0) { tc::mbar_init(bar, 1); tc::mbar_fence_init(); }
    tc::fence_async_smem();
    tc::fence_before_sync();
    __syncthreads();
    tc::fence_after_sync();
    const uint32_t tmem = *tmem_slot;
    const uint32_t d_col = tmem, a_hi = tmem + 64, a_lo = tmem + 128;
    const uint32_t lane_base = (uint32_t)(warp * 32) << 16;
    uint32_t parity = 0;

    const int64_t ntiles = (p.M + FTILE - 1) / FTILE;
    for (int64_t tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
        const int64_t i0 = tile * FTILE;
        const int64_t i_last = (i0 + FTILE - 1 < p.M ? i0 + FTILE - 1 : p.M - 1);
        const int64_t p_first = i0 / p.sn;
        const int np = (int)(i_last / p.sn - p_first) + 1;
        // per-point part of the first layer: h1p[lp][j] = b1[j] + sum_k W1[j][7 + k] (scale feat[p][k] + offset)
        for (int e = tid; e < np * F; e += FTILE) xfs[(e / F) * FMAXF + e % F] = __ldg(p.feat + (p_first + e / F) * F + e % F) * p.scale + p.offset;
        __syncthreads();
        for (int e = tid; e < np * FH; e += FTILE) {
            const int lp = e / FH, j = e % FH;
            float acc = bias1[j];
            for (int k = 0; k < F; ++k) acc = fmaf(w1b[k * FH + j], xfs[lp * FMAXF + k], acc);
            h1p[lp * FH + j] = acc;
        }
        const int64_t i = i0 + tid;
        const bool live = i < p.M;
        float yc = 0.f, yt = 0.f;
        {   // ---- layer-1 A operand: Reshift(PE(y_c)) (7 columns + zeros) -> tensor memory ---------------------------
            float xh[16], xl[16];
#pragma unroll
            for (int k = 0; k < 16; ++k) { xh[k] = 0.f; xl[k] = 0.f; }
            if (live) {
                const float y0 = p.y_in[i * 2], y1 = p.y_in[i * 2 + 1];
                yc = p.cond ? y1 : y0; yt = p.cond ? y0 : y1;
                float x[FPE];
                x[0] = yc; x[1] = sinf(yc); x[2] = cosf(yc); x[3] = sinf(yc * 2.f); x[4] = cosf(yc * 2.f); x[5] = sinf(yc * 4.f); x[6] = cosf(yc * 4.f);
#pragma unroll
                for (int k = 0; k < FPE; ++k) { const float v = x[k] * p.scale + p.offset; xh[k] = tc::tf32_rn(v); xl[k] = tc::tf32_rn(v - xh[k]); }
            }
            tc::tmem_st16(a_hi + lane_base, xh);
            tc::tmem_st16(a_lo + lane_base, xl);
            tc::tmem_st_wait();
        }
        tc::fence_before_sync();
        __syncthreads();                                        // A operand + h1p visible
        if (tid == 0) { tc::fence_after_sync(); issue_layer(d_col, a_hi, a_lo, b1_hi, b1_lo, K1, FH); tc::mma_commit(bar); }
        const float* hb = h1p + (live ? (int)(i / p.sn - p_first) : 0) * FH;
        // ---- layers 1-3: D -> bias + LeakyReLU -> A operand of the next layer ------------------------------------------
#pragma unroll 1
        for (int layer = 0; layer < 3; ++layer) {
            tc::mbar_wait(bar, parity); parity ^= 1;
            tc::fence_after_sync();
            const float* bias = layer == 0 ? hb : (layer == 1 ? bias2 : bias3);
#pragma unroll
            for (int c0 = 0; c0 < FH; c0 += 16) {
                float v[16], lo[16];
                tc::tmem_ld16(d_col + lane_base + c0, v);
#pragma unroll
                for (int j = 0; j < 16; ++j) v[j] = live ? leaky(v[j] + bias[c0 + j]) : 0.f;
                if (p.save_h && live) {
                    float4* dst = reinterpret_cast<float4*>(p.save_h + ((size_t)i * 3 + layer) * FH + c0);
#pragma unroll
                    for (int j = 0; j < 4; ++j) dst[j] = make_float4(v[4 * j], v[4 * j + 1], v[4 * j + 2], v[4 * j + 3]);
                }
#pragma unroll
                for (int j = 0; j < 16; ++j) { const float h = tc::tf32_rn(v[j]); lo[j] = tc::tf32_rn(v[j] - h); v[j] = h; }
                tc::tmem_st16(a_hi + lane_base + c0, v);
                tc::tmem_st16(a_lo + lane_base + c0, lo);
            }
            tc::tmem_st_wait();
            tc::fence_before_sync();
            __syncthreads();
            if (tid == 0) {
                tc::fence_after_sync();
                if (layer == 0) issue_layer(d_col, a_hi, a_lo, b2_hi, b2_lo, FH, FH);
                else if (layer == 1) issue_layer(d_col, a_hi, a_lo, b3_hi, b3_lo, FH, FH);
                else issue_layer(d_col, a_hi, a_lo, b4_hi, b4_lo, FH, N4);
                tc::mma_commit(bar);
            }
        }
        // ---- layer 4 -> spline -------------------------------------------------------------------------------------------
        tc::mbar_wait(bar, parity); parity ^= 1;
        tc::fence_after_sync();
        {
            float st[FSTP];
            tc::tmem_ld16(d_col + lane_base, st);
            tc::tmem_ld8(d_col + lane_base + 16, st + 16);
            if (live) {
#pragma unroll
                for (int j = 0; j < FSTP; ++j) st[j] += bias4[j];
                if (p.save_st) {
                    float4* dst = reinterpret_cast<float4*>(p.save_st + (size_t)i * FSTP);
#pragma unroll
                    for (int j = 0; j < FSTP / 4; ++j) dst[j] = make_float4(st[4 * j], st[4 * j + 1], st[4 * j + 2], st[4 * j + 3]);
                }
                float xt, lj;
                if (p.inverse) pwquad_eval_inverse(st, yt, xt, lj);
                else pwquad_eval_forward(st, yt, xt, lj);
                p.y_out[i * 2 + p.cond] = yc;
                p.y_out[i * 2 + 1 - p.cond] = xt;
                p.logj_out[i] = (p.logj_in ? p.logj_in[i] : 0.f) + lj;
            }
        }
        tc::fence_before_sync();
        __syncthreads();                                        // D and h1p are free for the next tile
    }
    tc::fence_before_sync();
    __syncthreads();
    if (warp == 0) tc::tmem_dealloc<256>(tmem);
}

// =====================================================================================================================
// Backward of the coupling block (density direction) with the activations kept by the forward (h1, h2, h3, spline parameters):
//   adjoint chain   d_st -> dh3 -> dpre3 -> dh2 -> dpre2 -> dh1 -> dpre1 -> d x_in : four TS-mode GEMMs against W^T tiles in shared
//                   memory, the running adjoint written to tensor memory by the epilogues (x LeakyReLU' of the kept activation)
//   weight gradients dW_l += dpre_l^T h_(l-1) over the 128 rows of the tile: register-tiled FP32 products from two row-major
//                   shared-memory tiles while the tensor core runs the next chain GEMM; every thread owns a patch of the
//                   per-CTA accumulators (no atomics until the final flush)
//   feature part     per-point sums of dpre1 -> dW1[:, 7:], d feature
// =====================================================================================================================
constexpr int FLD = FH + 4;          // row stride of the fp32 tiles (bank spread for per-thread rows)
constexpr int FLDS = FSTP + 4;

struct FlowTcBwdParams {
    const float *W1, *W2, *W3, *W4;
    int F; float scale, offset;
    const float* y_in; const float* feat; const float* saved_h; const float* saved_st;
    int sn, cond; int64_t M;
    const float* g_y_out; const float* g_logj;
    float* g_y_in; float* d_feat;
    float *dW1, *db1, *dW2, *db2, *dW3, *db3, *dW4, *db4;
};

// acc[j][k] += sum_p D[p][j] H[p][k] over the 128 rows of a tile; every thread owns a JP x KP patch (JP, KP multiples of 4 use
// 16-byte shared-memory loads; rows are FLD = 68 floats apart, so the patch origins must be multiples of 4)
template <int JP, int KP>
__device__ __forceinline__ void tile_xty(const float* __restrict__ D, int ldd, const float* __restrict__ H, int ldh, float* __restrict__ acc, int ldacc,
                                         int j0, int k0) {
    float a[JP][KP];
#pragma unroll
    for (int x = 0; x < JP; ++x)
#pragma unroll
        for (int y = 0; y < KP; ++y) a[x][y] = 0.f;
#pragma unroll 4
    for (int r = 0; r < FTILE; ++r) {
        float d[JP], h[KP];
        if (JP % 4 == 0) {
#pragma unroll
            for (int x = 0; x < JP; x += 4) { const float4 v = *reinterpret_cast<const float4*>(D + r * ldd + j0 + x); d[x] = v.x; d[x + 1] = v.y; d[x + 2] = v.z; d[x + 3] = v.w; }
        } else {
#pragma unroll
            for (int x = 0; x < JP; ++x) d[x] = D[r * ldd + j0 + x];
        }
#pragma unroll
        for (int y = 0; y < KP; y += 4) { const float4 v = *reinterpret_cast<const float4*>(H + r * ldh + k0 + y); h[y] = v.x; h[y + 1] = v.y; h[y + 2] = v.z; h[y + 3] = v.w; }
#pragma unroll
        for (int x = 0; x < JP; ++x)
#pragma unroll
            for (int y = 0; y < KP; ++y) a[x][y] = fmaf(d[x], h[y], a[x][y]);
    }
#pragma unroll
    for (int x = 0; x < JP; ++x)
#pragma unroll
        for (int y = 0; y < KP; ++y) acc[(j0 + x) * ldacc + k0 + y] += a[x][y];
}
__device__ __forceinline__ void tile_colsum(const float* __restrict__ D, int ldd, int ncols, float* __restrict__ acc, int tid) {
    if (tid < ncols) {
        float s = 0.f;
        for (int r = 0; r < FTILE; ++r) s += D[r * ldd + tid];
        acc[tid] += s;
    }
}
// rows [i0, i0 + 128) of the kept activation `layer` -> shared-memory tile (coalesced: 16 threads per 256-byte row)
__device__ __forceinline__ void load_h_tile(float* T, const float* __restrict__ saved_h, int layer, int64_t i0, int64_t M, int tid) {
    for (int e = tid; e < FTILE * (FH / 4); e += FTILE) {
        const int r = e / (FH / 4), c4 = e % (FH / 4);
        float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
        if (i0 + r < M) v = __ldg(reinterpret_cast<const float4*>(saved_h + ((size_t)(i0 + r) * 3 + layer) * FH) + c4);
        *reinterpret_cast<float4*>(T + r * FLD + 4 * c4) = v;
    }
}

__global__ void __launch_bounds__(FTILE, 1) flow_block_bwd_tc_kernel(FlowTcBwdParams p) {
    extern __shared__ __align__(1024) uint8_t fsm_raw[];
    float* sp = reinterpret_cast<float*>(fsm_raw);
    auto carve = [&](int n) { float* r = sp; sp += n; return r; };
    // B tiles of the adjoint chain: B[n = input unit][k = output unit] = W[k][n]
    float* t4_hi = carve(FH * N4); float* t4_lo = carve(FH * N4);      // [64][32]: W4^T
    float* t3_hi = carve(FH * FH); float* t3_lo = carve(FH * FH);
    float* t2_hi = carve(FH * FH); float* t2_lo = carve(FH * FH);
    float* t1_hi = carve(K1 * FH); float* t1_lo = carve(K1 * FH);      // [8][64]: W1[:, :7]^T
    float* aW1a = carve(FH * 8); float* aW1b = carve(FH * FMAXF); float* aW2 = carve(FH * FH); float* aW3 = carve(FH * FH); float* aW4 = carve(FSTP * FH);
    float* ab1 = carve(FH); float* ab2 = carve(FH); float* ab3 = carve(FH); float* ab4 = carve(FSTP);
    float* Th = carve(FTILE * FLD);          // kept activation of the previous layer (row-major fp32)
    float* Td = carve(FTILE * FLD);          // adjoint of the current layer's pre-activation (row-major fp32)
    float* Sp = carve(FMAXP * FH);
    int* row_lp = reinterpret_cast<int*>(carve(FTILE));       // local point index of every row of the tile
    float* w1b = carve(FH * FMAXF);          // feature part of the first layer, [j][k]
    float* xfs = carve(FMAXP * FMAXF);       // Reshift(feature) of the tile's points
    uint64_t* bar = reinterpret_cast<uint64_t*>(carve(2));
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(carve(2));

    const int tid = threadIdx.x, warp = tid >> 5;
    const int F = p.F, KW1 = FPE + F;
    // transposed weight tiles: element (n, k) = W[k][n]
    for (int i = tid; i < FH * N4; i += FTILE) {
        const int n = i / N4, k = i % N4;
        const float v = k < NST ? p.W4[(size_t)k * FH + n] : 0.f;
        const float h = tc::tf32_rn(v); const uint32_t off = tc::tile_off_b32(n, k, N4 / 4) / 4;
        t4_hi[off] = h; t4_lo[off] = tc::tf32_rn(v - h);
    }
    for (int i = tid; i < FH * FH; i += FTILE) {
        const int n = i / FH, k = i % FH;
        const uint32_t off = tc::tile_off_b32(n, k, FH / 4) / 4;
        float v = p.W3[(size_t)k * FH + n]; float h = tc::tf32_rn(v);
        t3_hi[off] = h; t3_lo[off] = tc::tf32_rn(v - h);
        v = p.W2[(size_t)k * FH + n]; h = tc::tf32_rn(v);
        t2_hi[off] = h; t2_lo[off] = tc::tf32_rn(v - h);
    }
    for (int i = tid; i < K1 * FH; i += FTILE) {
        const int n = i / FH, k = i % FH;
        const float v = n < FPE ? p.W1[(size_t)k * KW1 + n] : 0.f;
        const float h = tc::tf32_rn(v); const uint32_t off = tc::tile_off_b32(n, k, FH / 4) / 4;
        t1_hi[off] = h; t1_lo[off] = tc::tf32_rn(v - h);
    }
    for (int i = tid; i < FH * 8 + FH * FMAXF + 2 * FH * FH + FSTP * FH + 3 * FH + FSTP; i += FTILE) aW1a[i] = 0.f;      // contiguous accumulators
    for (int i = tid; i < FH * F; i += FTILE) { const int j = i / F, k = i % F; w1b[j * FMAXF + k] = p.W1[(size_t)j * KW1 + FPE + k]; }
    if (warp == 0) tc::tmem_alloc<256>(tmem_slot);
    if (tid == 0) { tc::mbar_init(bar, 1); tc::mbar_fence_init(); }
    tc::fence_async_smem();
    tc::fence_before_sync();
    __syncthreads();
    tc::fence_after_sync();
    const uint32_t tmem = *tmem_slot;
    const uint32_t d_col = tmem, a_hi = tmem + 64, a_lo = tmem + 128;
    const uint32_t lane_base = (uint32_t)(warp * 32) << 16;
    uint32_t parity = 0;

    const int64_t ntiles = (p.M + FTILE - 1) / FTILE;
    for (int64_t tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
        const int64_t i0 = tile * FTILE;
        const int64_t i_last = (i0 + FTILE - 1 < p.M ? i0 + FTILE - 1 : p.M - 1);
        const int64_t p_first = i0 / p.sn;
        const int np = (int)(i_last / p.sn - p_first) + 1;
        const int64_t i = i0 + tid;
        const bool live = i < p.M;
        float yc = 0.f, d_yt = 0.f;
        row_lp[tid] = live ? (int)(i / p.sn - p_first) : np - 1;
        for (int e = tid; e < np * F; e += FTILE) xfs[(e / F) * FMAXF + e % F] = __ldg(p.feat + (p_first + e / F) * F + e % F) * p.scale + p.offset;
        {   // ---- spline adjoint -> d_st: A operand (tensor memory) + row-major tile --------------------------------------
            float dst[N4], lo[N4];
#pragma unroll
            for (int k = 0; k < N4; ++k) dst[k] = 0.f;
            if (live) {
                float st[FSTP];
                const float4* s4 = reinterpret_cast<const float4*>(p.saved_st + (size_t)i * FSTP);
#pragma unroll
                for (int j = 0; j < FSTP / 4; ++j) { const float4 v = __ldg(s4 + j); st[4 * j] = v.x; st[4 * j + 1] = v.y; st[4 * j + 2] = v.z; st[4 * j + 3] = v.w; }
                const float y0 = p.y_in[i * 2], y1 = p.y_in[i * 2 + 1];
                yc = p.cond ? y1 : y0;
                const float yt = p.cond ? y0 : y1;
                const float gx = p.g_y_out ? p.g_y_out[i * 2 + 1 - p.cond] : 0.f;
                const float gl = p.g_logj ? p.g_logj[i] : 0.f;
                pwquad_adjoint(st, yt, gx, gl, d_yt, dst);
            }
#pragma unroll
            for (int k = 0; k < FLDS; ++k) Td[tid * FLD + k] = k < FSTP ? dst[k] : 0.f;
#pragma unroll
            for (int k = 0; k < N4; ++k) { const float h = tc::tf32_rn(dst[k]); lo[k] = tc::tf32_rn(dst[k] - h); dst[k] = h; }
            tc::tmem_st16(a_hi + lane_base, dst); tc::tmem_st16(a_hi + lane_base + 16, dst + 16);
            tc::tmem_st16(a_lo + lane_base, lo); tc::tmem_st16(a_lo + lane_base + 16, lo + 16);
            tc::tmem_st_wait();
        }
        load_h_tile(Th, p.saved_h, 2, i0, p.M, tid);                      // h3
        tc::fence_before_sync();
        __syncthreads();
        if (tid == 0) { tc::fence_after_sync(); issue_layer(d_col, a_hi, a_lo, t4_hi, t4_lo, N4, FH); tc::mma_commit(bar); }    // dh3 = d_st W4
        tile_xty<3, 4>(Td, FLD, Th, FLD, aW4, FH, 3 * (tid >> 4), 4 * (tid & 15));                                             // dW4 += d_st^T h3
        tile_colsum(Td, FLD, FSTP, ab4, tid);
        // ---- layers 3, 2, 1: epilogue (x LeakyReLU') -> next chain GEMM on the tensor core || weight-gradient products ------
#pragma unroll 1
        for (int layer = 2; layer >= 0; --layer) {
            tc::mbar_wait(bar, parity); parity ^= 1;
            tc::fence_after_sync();
            __syncthreads();                                            // every thread is done reading Td / Th of the previous products
#pragma unroll
            for (int c0 = 0; c0 < FH; c0 += 16) {
                float v[16], lo[16];
                tc::tmem_ld16(d_col + lane_base + c0, v);
#pragma unroll
                for (int j4 = 0; j4 < 4; ++j4) {
                    const float4 h = *reinterpret_cast<const float4*>(Th + tid * FLD + c0 + 4 * j4);       // own row of the kept activation
                    v[4 * j4] *= h.x > 0.f ? 1.f : 0.01f; v[4 * j4 + 1] *= h.y > 0.f ? 1.f : 0.01f;
                    v[4 * j4 + 2] *= h.z > 0.f ? 1.f : 0.01f; v[4 * j4 + 3] *= h.w > 0.f ? 1.f : 0.01f;
                    *reinterpret_cast<float4*>(Td + tid * FLD + c0 + 4 * j4) = make_float4(v[4 * j4], v[4 * j4 + 1], v[4 * j4 + 2], v[4 * j4 + 3]);
                }
#pragma unroll
                for (int j = 0; j < 16; ++j) { const float h = tc::tf32_rn(v[j]); lo[j] = tc::tf32_rn(v[j] - h); v[j] = h; }
                tc::tmem_st16(a_hi + lane_base + c0, v);
                tc::tmem_st16(a_lo + lane_base + c0, lo);
            }
            tc::tmem_st_wait();
            tc::fence_before_sync();
            __syncthreads();                                            // dpre tile + A operand complete, Th free
            if (tid == 0) {
                tc::fence_after_sync();
                if (layer == 2) issue_layer(d_col, a_hi, a_lo, t3_hi, t3_lo, FH, FH);          // dh2 = dpre3 W3
                else if (layer == 1) issue_layer(d_col, a_hi, a_lo, t2_hi, t2_lo, FH, FH);     // dh1 = dpre2 W2
                else issue_layer(d_col, a_hi, a_lo, t1_hi, t1_lo, FH, K1);                     // d x_in = dpre1 W1[:, :7]
                tc::mma_commit(bar);
            }
            if (layer > 0) {
                load_h_tile(Th, p.saved_h, layer - 1, i0, p.M, tid);    // h2 / h1: input of this layer, also the next epilogue's LeakyReLU'
            } else {                                                    // layer 1: the input is Reshift(PE(y_c)), recomputed
                float x[8];
                x[0] = yc; x[1] = sinf(yc); x[2] = cosf(yc); x[3] = sinf(yc * 2.f); x[4] = cosf(yc * 2.f); x[5] = sinf(yc * 4.f); x[6] = cosf(yc * 4.f);
#pragma unroll
                for (int k = 0; k < 8; ++k) Th[tid * FLD + k] = (live && k < FPE) ? x[k] * p.scale + p.offset : 0.f;
            }
            __syncthreads();
            if (layer == 2) { tile_xty<4, 8>(Td, FLD, Th, FLD, aW3, FH, 4 * (tid >> 3), 8 * (tid & 7)); tile_colsum(Td, FLD, FH, ab3, tid); }
            else if (layer == 1) { tile_xty<4, 8>(Td, FLD, Th, FLD, aW2, FH, 4 * (tid >> 3), 8 * (tid & 7)); tile_colsum(Td, FLD, FH, ab2, tid); }
            else {
                tile_xty<1, 4>(Td, FLD, Th, FLD, aW1a, 8, tid >> 1, 4 * (tid & 1));
                tile_colsum(Td, FLD, FH, ab1, tid);
                if (tid >= FH) {                                        // S[lp][j]: dpre1 summed over the tile's rows of point lp
                    const int j = tid - FH;
                    float sacc = 0.f;
                    int cur = 0;
                    for (int r = 0; r < FTILE; ++r) {
                        const int lr = row_lp[r];
                        if (lr != cur) { Sp[cur * FH + j] = sacc; sacc = 0.f; cur = lr; }
                        sacc += Td[r * FLD + j];
                    }
                    Sp[cur * FH + j] = sacc;
                }
            }
        }
        // ---- d y_c from d x_in, feature part of the first layer -----------------------------------------------------------
        tc::mbar_wait(bar, parity); parity ^= 1;
        tc::fence_after_sync();
        {
            float dx[8];
            tc::tmem_ld8(d_col + lane_base, dx);
            if (live) {
                const float dyc = p.scale * (dx[0] + dx[1] * cosf(yc) - dx[2] * sinf(yc) + 2.f * (dx[3] * cosf(2.f * yc) - dx[4] * sinf(2.f * yc)) +
                                             4.f * (dx[5] * cosf(4.f * yc) - dx[6] * sinf(4.f * yc)));
                p.g_y_in[i * 2 + p.cond] = (p.g_y_out ? p.g_y_out[i * 2 + p.cond] : 0.f) + dyc;
                p.g_y_in[i * 2 + 1 - p.cond] = d_yt;
            }
        }
        __syncthreads();                                                // Sp complete
        // feature part: d_feat[p][k] += scale sum_j W1[j][7 + k] S[lp][j] (threads <-> (point, k));  dW1[j][7 + k] += S[lp][j] xf[lp][k]
        // (threads <-> j: every accumulator row has one owner, no atomics)
        for (int e = tid; e < np * F; e += FTILE) {
            const int l = e / F, k = e % F;
            float g = 0.f;
            for (int j = 0; j < FH; ++j) g = fmaf(w1b[j * FMAXF + k], Sp[l * FH + j], g);
            atomicAdd(p.d_feat + (p_first + l) * F + k, g * p.scale);
        }
        if (tid < FH) {
            for (int l = 0; l < np; ++l) {
                const float sj = Sp[l * FH + tid];
                for (int k = 0; k < F; ++k) aW1b[tid * FMAXF + k] = fmaf(sj, xfs[l * FMAXF + k], aW1b[tid * FMAXF + k]);
            }
        }
        tc::fence_before_sync();
        __syncthreads();
    }
    // ---- flush the CTA's weight-gradient partials ------------------------------------------------------------------------
    for (int i = tid; i < FH * FPE; i += FTILE) { const int j = i / FPE, k = i % FPE; const float v = aW1a[j * 8 + k]; if (v != 0.f) atomicAdd(p.dW1 + (size_t)j * KW1 + k, v); }
    for (int i = tid; i < FH * F; i += FTILE) { const int j = i / F, k = i % F; const float v = aW1b[j * FMAXF + k]; if (v != 0.f) atomicAdd(p.dW1 + (size_t)j * KW1 + FPE + k, v); }
    for (int i = tid; i < FH * FH; i += FTILE) {
        if (aW2[i] != 0.f) atomicAdd(p.dW2 + i, aW2[i]);
        if (aW3[i] != 0.f) atomicAdd(p.dW3 + i, aW3[i]);
    }
    for (int i = tid; i < NST * FH; i += FTILE) if (aW4[i] != 0.f) atomicAdd(p.dW4 + i, aW4[i]);
    for (int i = tid; i < FH; i += FTILE) {
        if (ab1[i] != 0.f) atomicAdd(p.db1 + i, ab1[i]);
        if (ab2[i] != 0.f) atomicAdd(p.db2 + i, ab2[i]);
        if (ab3[i] != 0.f) atomicAdd(p.db3 + i, ab3[i]);
    }
    for (int i = tid; i < NST; i += FTILE) if (ab4[i] != 0.f) atomicAdd(p.db4 + i, ab4[i]);
    tc::fence_before_sync();
    __syncthreads();
    if (warp == 0) tc::tmem_dealloc<256>(tmem);
}

size_t flow_tc_bwd_smem() {
    return sizeof(float) * (size_t)(2 * FH * N4 + 4 * FH * FH + 2 * K1 * FH + FH * 8 + FH * FMAXF + 2 * FH * FH + FSTP * FH + 3 * FH + FSTP +
                                    2 * FTILE * FLD + FMAXP * FH + FTILE + FH * FMAXF + FMAXP * FMAXF + 4) + 1024;
}

size_t flow_tc_smem() {
    return sizeof(float) * (size_t)(2 * FH * K1 + 4 * FH * FH + 2 * N4 * FH + 3 * FH + N4 + FMAXP * FH + FMAXF * FH + FMAXP * FMAXF + 4) + 1024;
}

}  // namespace

// tensor-core forward of one coupling block (arguments as tf_flow_block_fwd; save_h / save_st keep the activations for the backward)
int tf_internal_flow_block_fwd_tc(const float* y_in, const float* logj_in, const float* feat, int feat_dim, int sn, const float* W1,
                                  const float* b1, const float* W2, const float* b2, const float* W3, const float* b3, const float* W4,
                                  const float* b4, float scale, float offset, int cond, int inverse, int64_t M, float* y_out, float* logj_out,
                                  float* save_h, float* save_st, cudaStream_t stream) {
    FlowTcParams p = {W1, b1, W2, b2, W3, b3, W4, b4, feat_dim, scale, offset, y_in, logj_in, feat, sn, cond, inverse, M, y_out, logj_out,
                      save_h, save_st};
    const size_t smem = flow_tc_smem();
    cudaFuncSetAttribute(flow_block_fwd_tc_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    const int64_t ntiles = (M + FTILE - 1) / FTILE;
    const int64_t cap = (int64_t)tf_num_sms() * 2;
    const int grid = (int)(ntiles < cap ? ntiles : cap);
    {
        TfKernelTimer timer("flow_block_fwd_tc", stream);
        flow_block_fwd_tc_kernel<<<grid, FTILE, smem, stream>>>(p);
    }
    tf_count_launches(1);
    return 0;
}

// tensor-core backward of one coupling block from the activations kept by tf_internal_flow_block_fwd_tc
int tf_internal_flow_block_bwd_tc(const float* y_in, const float* feat, int feat_dim, int sn, const float* W1, const float* W2, const float* W3,
                                  const float* W4, float scale, float offset, int cond, int64_t M, const float* saved_h, const float* saved_st,
                                  const float* g_y_out, const float* g_logj, float* g_y_in, float* d_feat, float* dW1, float* db1, float* dW2,
                                  float* db2, float* dW3, float* db3, float* dW4, float* db4, cudaStream_t stream) {
    FlowTcBwdParams p = {W1, W2, W3, W4, feat_dim, scale, offset, y_in, feat, saved_h, saved_st, sn, cond, M, g_y_out, g_logj, g_y_in, d_feat,
                         dW1, db1, dW2, db2, dW3, db3, dW4, db4};
    const size_t smem = flow_tc_bwd_smem();
    if (smem > 227 * 1024) { tf_set_error("flow block backward: shared-memory budget exceeded (%zu bytes)", smem); return 1; }
    cudaFuncSetAttribute(flow_block_bwd_tc_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    const int64_t ntiles = (M + FTILE - 1) / FTILE;
    const int grid = (int)(ntiles < tf_num_sms() ? ntiles : tf_num_sms());
    {
        TfKernelTimer timer("flow_block_bwd_tc", stream);
        flow_block_bwd_tc_kernel<<<grid, FTILE, smem, stream>>>(p);
    }
    tf_count_launches(1);
    return 0;
}
