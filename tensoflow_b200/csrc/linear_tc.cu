// Dense layer on the tensor cores: Y[M,N] = act(X[M,K] Wt[N,K]^T + b)   (3xTF32: fp32-level accuracy).
//
// BWD mode computes the data gradient of a layer: the A operand is dPre = dY * act'(Y), formed on load (and written
// back for the weight-gradient pass), contracted with the transposed weights: dX[M,K] = dPre[M,N] W[N,K].
// The output width is padded to a multiple of 16 inside the kernel (zero weight rows, masked stores) and X rows of
// any length are accepted (scalar loads when a row is not float4-aligned).
// Used for the appearance head of the SDF decoder (hidden [n,H] -> feat [n,A], reference network/fields.py:192-198)
// and its input gradient (g_feat [n,A] -> dHidden [n,H], Wt = W1[1:,:]^T).  X rows stream from HBM once:
// one persistent CTA per SM walks 128-row tiles; per K-chunk of 32 the threads load the X chunk (coalesced
// float4 reads), split it into tf32 hi/lo and store it in the K-major no-swizzle UMMA layout (padded K-chunk
// stride -> conflict-free stores) while the matching pre-split weight chunk arrives by cp.async.bulk; one
// thread issues the tcgen05.mma's (accumulator [128 x N] fp32 in TMEM, double buffered across tiles) and the
// epilogue of tile t-1 (bias, activation, 64-byte row stores) overlaps the loads / MMAs of tile t.
#include "common.cuh"
#include "tc_common.cuh"
#include "act.cuh"
#include "internal.cuh"

namespace {

constexpr int TM = 128;
constexpr int KC = 32;                 // K chunk per pipeline stage
constexpr int NSTG = 2;
constexpr int NTH = 512;
constexpr int NWORK = NTH - 32;        // staging warps 1..15; warp 0 streams the weight chunks and issues the MMAs (a thread that issues a
                                       // dozen MMAs back to back is blocked while the tensor queue drains: no staging warp may wait for it)
constexpr int XPT = (1024 + NWORK - 1) / NWORK;   // float4 loads per worker and stage (128 rows x 8 chunks = 1024)
constexpr uint32_t X_LBO = 144;        // K-chunk (16 B) stride of the X operand, padded for bank spread
constexpr uint32_t X_SBO = (KC / 4) * X_LBO;
constexpr uint32_t X_PART = 16 * X_SBO;      // bytes of one X part (hi or lo) of a stage

// pre-split weights: chunk kc -> [N rows x 32] K-major hi | lo
__global__ void linear_tc_prep_kernel(const float* __restrict__ W, int ldw, int trans, int N, int NP, int K, int KP, float* __restrict__ Wtc) {
    const int nchunks = KP / KC;
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < nchunks * NP * KC; i += gridDim.x * blockDim.x) {
        const int kl = i % KC, n = (i / KC) % NP, kc = i / (KC * NP);
        const int k = kc * KC + kl;
        // trans == 0: Wt[n][k] = W[n*ldw + k];  trans == 1: Wt[n][k] = W[k*ldw + n]
        const float v = (k < K && n < N) ? (trans ? W[(size_t)k * ldw + n] : W[(size_t)n * ldw + k]) : 0.f;
        const float hi = tc::tf32_rn(v);
        float* base = Wtc + (size_t)kc * 2 * NP * KC;
        const uint32_t off = tc::tile_off_b32(n, kl, KC / 4) / 4;
        base[off] = hi;
        base[(size_t)NP * KC + off] = tc::tf32_rn(v - hi);
    }
}

__device__ __forceinline__ void bulk_copy_g2s(void* dst, const void* src, uint32_t bytes, uint64_t* bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(tc::smem_u32(dst)),
                 "l"(src), "r"(bytes), "r"(tc::smem_u32(bar))
                 : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(tc::smem_u32(bar)), "r"(bytes) : "memory");
}

struct XRegs { float4 v[XPT]; };     // one stage of X per worker: 128 rows x 8 chunks = 1024 float4 over 480 workers

// one stage of the A operand: X[m][k0 .. k0+32) for the tile's 128 rows.  BWD: element = dY * act'(Y), also stored to dpre
template <bool BWD>
__device__ __forceinline__ void x_load(const float* __restrict__ X, const float* __restrict__ Yact, float* __restrict__ dpre, int act,
                                       float act_p, bool vec, int64_t M, int K, int64_t row0, int k0, XRegs& r) {
#pragma unroll
    for (int j = 0; j < XPT; ++j) {
        const int it = (int)threadIdx.x - 32 + j * NWORK;
        const int row = it >> 3, ch = it & 7;
        const int64_t m = row0 + row;
        const int k = k0 + ch * 4;
        float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
        if (it < 1024 && m < M && k < K) {
            const size_t o = (size_t)m * K + k;
            if (vec) {
                v = ldg4(X + o);
                if (BWD) {
                    const float4 y = ldg4(Yact + o);
                    v.x *= act_bwd(y.x, act, act_p); v.y *= act_bwd(y.y, act, act_p); v.z *= act_bwd(y.z, act, act_p); v.w *= act_bwd(y.w, act, act_p);
                    *reinterpret_cast<float4*>(dpre + o) = v;
                }
            } else {
                float e[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
                for (int i = 0; i < 4; ++i)
                    if (k + i < K) {
                        e[i] = __ldg(X + o + i);
                        if (BWD) { e[i] *= act_bwd(__ldg(Yact + o + i), act, act_p); dpre[o + i] = e[i]; }
                    }
                v = make_float4(e[0], e[1], e[2], e[3]);
            }
        }
        r.v[j] = v;
    }
}
__device__ __forceinline__ void x_store(const XRegs& r, uint8_t* hi, uint8_t* lo) {
#pragma unroll
    for (int j = 0; j < XPT; ++j) {
        const int it = (int)threadIdx.x - 32 + j * NWORK;
        if (it >= 1024) continue;
        const int row = it >> 3, ch = it & 7;
        const uint32_t off = (uint32_t)(row >> 3) * X_SBO + ch * X_LBO + (row & 7) * 16;
        const float4 v = r.v[j];
        const float4 h = make_float4(tc::tf32_rn(v.x), tc::tf32_rn(v.y), tc::tf32_rn(v.z), tc::tf32_rn(v.w));
        *reinterpret_cast<float4*>(hi + off) = h;
        *reinterpret_cast<float4*>(lo + off) =
            make_float4(tc::tf32_rn(v.x - h.x), tc::tf32_rn(v.y - h.y), tc::tf32_rn(v.z - h.z), tc::tf32_rn(v.w - h.w));
    }
}

template <bool BWD>
__global__ void __launch_bounds__(NTH, 1) linear_tc_kernel(const float* __restrict__ X, const float* __restrict__ Yact, float* __restrict__ dpre,
                                                           const float* __restrict__ Wtc, const float* __restrict__ bias, int64_t M, int K, int KP,
                                                           int N, int NP, int act, float act_p, float* __restrict__ Y) {
    extern __shared__ __align__(1024) uint8_t smem[];
    const uint32_t w_part = (uint32_t)NP * KC * 4;
    const bool vec = (K % 4 == 0) && (((uintptr_t)X & 15) == 0) && (!BWD || ((((uintptr_t)Yact | (uintptr_t)dpre) & 15) == 0));
    const bool vec_out = (N % 4 == 0) && (((uintptr_t)Y & 15) == 0);
    const bool bias_vec = bias != nullptr && (((uintptr_t)bias & 15) == 0);
    // shared memory: NSTG X stages (hi | lo) + 2 weight-chunk buffers (hi | lo); TMEM: one accumulator per tile of a group
    uint8_t* wbuf0 = smem + (size_t)NSTG * 2 * X_PART;
    uint64_t* bars = reinterpret_cast<uint64_t*>(wbuf0 + (size_t)2 * 2 * w_part);
    uint64_t* wfull = bars;              // [2] weight chunk landed
    uint64_t* wfree = bars + 2;          // [2] weight chunk consumed by the last MMA that reads it
    uint64_t* sfree = bars + 4;          // [NSTG] X stage consumed by its MMAs
    uint64_t* sready = sfree + NSTG;     // [NSTG] X stage written by the staging warps
    uint64_t* dfull = sready + NSTG;     // accumulators of the group complete
    uint64_t* tfree = dfull + 1;         // accumulators of the group read out by the staging warps
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tfree + 1);
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int nchunks = KP / KC;
    const int cstride = NP <= 128 ? 128 : 256;         // TMEM columns per accumulator
    const int G = 512 / cstride;                       // row tiles per group: they share every weight chunk
    const int64_t ntiles = (M + TM - 1) / TM;
    const int64_t my_tiles = blockIdx.x < ntiles ? (ntiles - blockIdx.x + gridDim.x - 1) / gridDim.x : 0;
    const int64_t ngroups = (my_tiles + G - 1) / G;
    const int64_t total_w = ngroups * nchunks;         // weight chunks this CTA streams

    if (warp == 0) tc::tmem_alloc<512>(tmem_slot);
    if (tid == 0) {
        for (int i = 0; i < 2; ++i) { tc::mbar_init(&wfull[i], 1); tc::mbar_init(&wfree[i], 1); }
        for (int i = 0; i < NSTG; ++i) { tc::mbar_init(&sfree[i], 1); tc::mbar_init(&sready[i], NWORK); }
        tc::mbar_init(dfull, 1); tc::mbar_init(tfree, NWORK);
        tc::mbar_fence_init();
    }
    tc::fence_before_sync();
    __syncthreads();
    tc::fence_after_sync();
    const uint32_t tmem_base = *tmem_slot;
    const uint32_t idesc = tc::make_idesc(2, 2, TM, NP);
    const uint32_t w_sbo = (KC / 4) * 128;

    auto epilogue = [&](int64_t local_tile, int j) {
        const int64_t tile = blockIdx.x + local_tile * gridDim.x;
        const int lq = warp & 3, half = warp >> 2;
        const int64_t m = tile * TM + lq * 32 + lane;
        const uint32_t d = tmem_base + (uint32_t)j * cstride + ((uint32_t)(lq * 32) << 16);
        for (int c0 = half * 16; c0 < NP; c0 += 16 * (NTH / 128)) {
            float v[16];
            tc::tmem_ld16(d + c0, v);
            if (m < M) {
                if (!BWD) {
                    // bias: four 16-byte reads per 16 columns when the row of biases allows it; the activation switch is hoisted
                    // out of the element loop (the appearance head and the dHidden pass have none: a plain add)
                    float b[16];
                    if (bias_vec && c0 + 16 <= N) {
#pragma unroll
                        for (int jj = 0; jj < 4; ++jj) {
                            const float4 t = ldg4(bias + c0 + 4 * jj);
                            b[4 * jj] = t.x; b[4 * jj + 1] = t.y; b[4 * jj + 2] = t.z; b[4 * jj + 3] = t.w;
                        }
                    } else {
#pragma unroll
                        for (int jj = 0; jj < 16; ++jj) b[jj] = (bias && c0 + jj < N) ? __ldg(bias + c0 + jj) : 0.f;
                    }
                    if (act == ACT_NONE) {
#pragma unroll
                        for (int jj = 0; jj < 16; ++jj) v[jj] += b[jj];
                    } else if (act == ACT_RELU) {
#pragma unroll
                        for (int jj = 0; jj < 16; ++jj) v[jj] = fmaxf(v[jj] + b[jj], 0.f);
                    } else if (act == ACT_LEAKY) {
#pragma unroll
                        for (int jj = 0; jj < 16; ++jj) { const float x = v[jj] + b[jj]; v[jj] = x > 0.f ? x : 0.01f * x; }
                    } else {
#pragma unroll
                        for (int jj = 0; jj < 16; ++jj) v[jj] = act_fwd(v[jj] + b[jj], act, act_p);
                    }
                }
                if (vec_out) {
                    float4* dst = reinterpret_cast<float4*>(Y + (size_t)m * N + c0);
#pragma unroll
                    for (int jj = 0; jj < 4; ++jj)
                        if (c0 + 4 * jj < N) dst[jj] = make_float4(v[4 * jj], v[4 * jj + 1], v[4 * jj + 2], v[4 * jj + 3]);
                } else {
#pragma unroll
                    for (int jj = 0; jj < 16; ++jj)
                        if (c0 + jj < N) Y[(size_t)m * N + c0 + jj] = v[jj];
                }
            }
        }
    };
    // weight chunk w of the CTA's stream -> buffer w & 1 (thread 0)
    auto issue_w = [&](int64_t w) {
        const int buf = (int)(w & 1);
        if (w >= 2) tc::mbar_wait(&wfree[buf], (uint32_t)(((w >> 1) - 1) & 1));
        mbar_expect_tx(&wfull[buf], 2 * w_part);
        bulk_copy_g2s(wbuf0 + (size_t)buf * 2 * w_part, Wtc + (size_t)(w % nchunks) * 2 * NP * KC, 2 * w_part, &wfull[buf]);
    };
    // step = (group, weight chunk, tile of the group)
    struct Step { int64_t grp; int kc, j; };
    auto group_size = [&](int64_t grp) { return (int)(my_tiles - grp * G < G ? my_tiles - grp * G : G); };
    auto advance = [&](Step& s) {
        if (++s.j == group_size(s.grp)) { s.j = 0; if (++s.kc == nchunks) { s.kc = 0; ++s.grp; } }
    };
    if (warp == 0) {
        // ======================= driver warp: weight chunks + MMAs (lane 0), then its share of the group's epilogue ==============
        if (lane == 0 && total_w > 0) issue_w(0);
        int64_t q = 0;
        for (int64_t grp = 0; grp < ngroups; ++grp) {
            const int Gc = group_size(grp);
            if (lane == 0) {
                if (grp > 0) { tc::mbar_wait(tfree, (uint32_t)((grp - 1) & 1)); tc::fence_after_sync(); }    // accumulators read out
                for (int kc = 0; kc < nchunks; ++kc) {
                    const int64_t w = grp * nchunks + kc;
                    if (w + 1 < total_w) issue_w(w + 1);
                    tc::mbar_wait(&wfull[w & 1], (uint32_t)((w >> 1) & 1));
                    tc::fence_after_sync();
                    const uint32_t wh = tc::smem_u32(wbuf0 + (size_t)(w & 1) * 2 * w_part);
                    const uint64_t wdh0 = tc::make_smem_desc(wh, 128, w_sbo), wdl0 = tc::make_smem_desc(wh + w_part, 128, w_sbo);
                    for (int j = 0; j < Gc; ++j, ++q) {
                        const int st = (int)(q % NSTG);
                        uint8_t* x_hi = smem + (size_t)st * 2 * X_PART;
                        uint8_t* x_lo = x_hi + X_PART;
                        tc::mbar_wait(&sready[st], (uint32_t)((q / NSTG) & 1));
                        tc::fence_after_sync();
                        const uint32_t d = tmem_base + (uint32_t)j * cstride;
                        const uint64_t xdh = tc::make_smem_desc(tc::smem_u32(x_hi), X_LBO, X_SBO), xdl = tc::make_smem_desc(tc::smem_u32(x_lo), X_LBO, X_SBO);
#pragma unroll
                        for (int ks = 0; ks < KC / 8; ++ks) {
                            const uint64_t adh = tc::desc_add(xdh, ks * 2 * X_LBO), adl = tc::desc_add(xdl, ks * 2 * X_LBO);
                            const uint64_t wdh = tc::desc_add(wdh0, ks * 256), wdl = tc::desc_add(wdl0, ks * 256);
                            tc::mma_tf32_ss(d, adh, wdh, idesc, (kc | ks) != 0);
                            tc::mma_tf32_ss(d, adh, wdl, idesc, 1);
                            tc::mma_tf32_ss(d, adl, wdh, idesc, 1);
                        }
                        tc::mma_commit(&sfree[st]);
                    }
                    tc::mma_commit(&wfree[w & 1]);
                }
                tc::mma_commit(dfull);
            }
            __syncwarp();
            tc::mbar_wait(dfull, (uint32_t)(grp & 1));
            tc::fence_after_sync();
            for (int jj = 0; jj < Gc; ++jj) epilogue(grp * G + jj, jj);
            tc::fence_before_sync();
            __syncwarp();
        }
    } else {
        // ======================= staging warps: X rows -> registers PF steps ahead -> tf32 hi | lo in shared memory ================
        auto load_step = [&](const Step& s, XRegs& r) {
            if (s.grp < ngroups) x_load<BWD>(X, Yact, dpre, act, act_p, vec, M, K, (blockIdx.x + (s.grp * G + s.j) * gridDim.x) * TM, s.kc * KC, r);
        };
        constexpr int PF = 4;
        XRegs xr[PF];
        Step ahead = {0, 0, 0};
#pragma unroll
        for (int i = 0; i < PF; ++i) { load_step(ahead, xr[i]); if (ahead.grp < ngroups) advance(ahead); }
        Step cur = {0, 0, 0};
        int64_t q = 0;                                     // X stage counter
        auto do_step = [&](XRegs& r) {
            const int64_t grp = cur.grp;
            const int kc = cur.kc, j = cur.j, Gc = group_size(grp);
            const int st = (int)(q % NSTG);
            uint8_t* x_hi = smem + (size_t)st * 2 * X_PART;
            uint8_t* x_lo = x_hi + X_PART;
            if (q >= NSTG) tc::mbar_wait(&sfree[st], (uint32_t)(((q / NSTG) - 1) & 1));
            x_store(r, x_hi, x_lo);
            load_step(ahead, r);
            if (ahead.grp < ngroups) advance(ahead);
            tc::fence_async_smem();
            tc::mbar_arrive(&sready[st]);
            ++q;
            if (j == Gc - 1 && kc == nchunks - 1) {
                // the group's accumulators: bias + activation + store, then TMEM is free for the next group
                tc::mbar_wait(dfull, (uint32_t)(grp & 1));
                tc::fence_after_sync();
                for (int jj = 0; jj < Gc; ++jj) epilogue(grp * G + jj, jj);
                tc::fence_before_sync();
                tc::mbar_arrive(tfree);
            }
            advance(cur);
        };
        while (cur.grp < ngroups) {
#pragma unroll
            for (int i = 0; i < PF; ++i)
                if (cur.grp < ngroups) do_step(xr[i]);
        }
    }
    tc::fence_before_sync();
    __syncthreads();
    if (warp == 0) tc::tmem_dealloc<512>(tmem_base);
}

size_t linear_tc_smem(int NP) { return (size_t)NSTG * 2 * X_PART + (size_t)2 * 2 * NP * KC * 4 + (6 + 2 * NSTG) * 8 + 16; }
int pad16(int n) { return (n + 15) / 16 * 16; }

}  // namespace

// shapes the tensor-core dense layer takes: contraction widths up to 1024, output widths up to 256
bool tf_internal_linear_tc_ok(int K, int N) {
    if (N < 1 || N > 256 || K < 1 || K > 1024) return false;
    return linear_tc_smem(pad16(N)) <= 227 * 1024;
}
size_t tf_internal_linear_tc_ws_floats(int K, int N) { return (size_t)2 * pad16(N) * ((K + KC - 1) / KC * KC); }

// Y = act(X Wt^T + b); Wt[n][k] = trans ? W[k*ldw + n] : W[n*ldw + k]; `wtc` = scratch of tf_internal_linear_tc_ws_floats floats
int tf_internal_linear_tc(const float* X, const float* W, int ldw, int trans, const float* bias, int64_t M, int K, int N, int act, float act_p,
                          float* Y, float* wtc, cudaStream_t stream) {
    if (M == 0) return 0;
    const int KP = (K + KC - 1) / KC * KC, NP = pad16(N);
    linear_tc_prep_kernel<<<64, 256, 0, stream>>>(W, ldw, trans, N, NP, K, KP, wtc);
    const size_t smem = linear_tc_smem(NP);
    cudaFuncSetAttribute(linear_tc_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    const int64_t ntiles = (M + TM - 1) / TM;
    const int grid = (int)(ntiles < tf_num_sms() ? ntiles : tf_num_sms());
    {
        TfKernelTimer timer("linear_tc", stream);
        linear_tc_kernel<false><<<grid, NTH, smem, stream>>>(X, nullptr, nullptr, wtc, bias, M, K, KP, N, NP, act, act_p, Y);
    }
    tf_count_launches(2);
    return 0;
}

// data gradient of Y = act(X W^T + b), W [N,K]: dPre = dY * act'(Y) (written to `dpre`), dX[M,K] = dPre W
int tf_internal_linear_tc_bwd(const float* dY, const float* Yact, float* dpre, const float* W, int64_t M, int K, int N, int act, float act_p,
                              float* dX, float* wtc, cudaStream_t stream) {
    if (M == 0) return 0;
    // contraction over the layer's N outputs, K output columns: Wt[k][n] = W[n*K + k]
    const int KP = (N + KC - 1) / KC * KC, NP = pad16(K);
    linear_tc_prep_kernel<<<64, 256, 0, stream>>>(W, K, 1, K, NP, N, KP, wtc);
    const size_t smem = linear_tc_smem(NP);
    cudaFuncSetAttribute(linear_tc_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    const int64_t ntiles = (M + TM - 1) / TM;
    const int grid = (int)(ntiles < tf_num_sms() ? ntiles : tf_num_sms());
    {
        TfKernelTimer timer("linear_tc_bwd", stream);
        linear_tc_kernel<true><<<grid, NTH, smem, stream>>>(dY, Yact, dpre, wtc, nullptr, M, N, KP, K, NP, act, act_p, dX);
    }
    tf_count_launches(2);
    return 0;
}
