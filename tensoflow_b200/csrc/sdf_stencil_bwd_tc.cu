// Fused TensoSDF stencil backward (activation side) on the 5th-gen tensor cores, sm_100a.
//
// One persistent CTA per SM, 16 warps in two groups that work on different tiles at the same time
// (MMA tile = 128 rows = 18 samples x 7 stencil queries, sample-major: stencil_site.cuh):
//   memory group (8 warps, LSU-bound): gather of tile t+1 (features -> A operand hi/lo in shared memory + fp32 rows
//       to the workspace) and shared-stencil scatter of tile t-1 (dA from the CTA's L2 scratch tile -> RED.v4 into plane / line grads)
//   math group (8 warps, ALU-bound) on tile t: GEMM1 pre = A W0^T (3xTF32, accumulator D1 in TMEM), then per
//       32-column hidden chunk: tcgen05.ld -> Softplus / sigmoid -> dPre = (gq W1[0,:] + [centre] g_feat W1[1:]) * sigmoid
//       -> workspace (per tile [H][128], row fastest: one store wavefront per warp and column; X^T Y reads it as K-major
//       units) + TENSOR MEMORY (tcgen05.st, tf32 hi | lo), which the driver thread turns into
//       dA += dPre[:,chunk] W0[chunk,:] MMAs with the A operand read from TMEM (no shared-memory round trip and no
//       4 KB A read per instruction), accumulator D2; finally D2 -> the CTA's scratch tile in L2 for the memory group
// Hand-offs are mbarriers (A ready / GEMM1 done / dA ready / dA consumed); weight slices (W0 by 8 features for GEMM1,
// W0^T by 16 hidden units for GEMM-dA) stream through one 4-stage cp.async.bulk ring, each stage refilled by its own
// issuing lane (bulk copies of one warp execute one after the other).  Weight gradients are finished by X^T Y passes
// over the workspace (xty_tc.cu); the centre hidden activations come from the forward call, which kept them.
#include <stdio.h>
#include <stdlib.h>
#include "common.cuh"
#include "tc_common.cuh"
#include "stencil_site.cuh"
#include "internal.cuh"

namespace {

constexpr int TM = 128;
constexpr int NQ7 = 7;
constexpr int KSL = 16;     // KT granularity (shared with the forward kernel)
constexpr int KS1 = 8;      // K slice of GEMM1 streamed per ring slot (one tf32 k-step)
constexpr int HHC = 16;     // hidden units of a W0^T ring slot (half a chunk)
constexpr int HCH = 32;     // hidden chunk of epilogue-1 / GEMM-dA
constexpr int NST = 4;      // ring stages (16 KB each) = issuing lanes
constexpr int NGRP = 256;             // threads per group
constexpr int NTH = 2 * NGRP;         // math group (warps 0-7) + memory group (warps 8-15)

struct TcBwdParams {
    tf_vm_field_t f;
    tf_vm_mut_t g;
    const float* xyz; const float* level;
    int64_t n;
    const float* Wtc;        // [S + NCH] slots of slot_floats
    const float* b0; const float* w1r0;
    const float* sdf7; const float* g_sdf; const float* g_grad; const float* g_hess;
    const float* dHc;        // [n][H] = g_feat . W1[1:,:]  (NULL when there is no feature gradient)
    int K, KT, H, slot_floats;
    float units[3];
    float* da_scratch;       // [gridDim][128][KT+4]: dA tiles handed from the math to the memory group through L2
    float* dpre;             // [tiles][H][128] (per tile: column-major, rows fastest)
    float* arow;             // [tiles*128][KT]
    float* dW1r0; float* db1;
#ifdef TF_TC_DEBUG_SWITCHES
    long long* prof;         // [3 roles][16] phase cycle totals of CTA 0 (TF_TC_BWD_PROF=1)
    int debug;               // timing experiments only (never compiled into the product library): 1 no gather, 2 no workspace stores,
                             // 4 no scatter, 8 no dW1 reduction, 16 no chunk loop
#endif
};

#ifdef TF_TC_DEBUG_SWITCHES
#define TF_DBG(p, bit) ((p).debug & (bit))
#define PROF_DECL long long pt_[16] = {0}; long long pl_ = clock64();
#define PROF(i) { const long long now_ = clock64(); pt_[i] += now_ - pl_; pl_ = now_; }
#define PROF_DUMP(role) if (p.prof && blockIdx.x == 0) { for (int i_ = 0; i_ < 16; ++i_) p.prof[(role) * 16 + i_] = pt_[i_]; }
#else
#define TF_DBG(p, bit) 0
#define PROF_DECL
#define PROF(i)
#define PROF_DUMP(role)
#endif

// slots 0..S-1        : W0 K-slices      [H rows x 8]   hi | lo   (GEMM1 B operand)
// slots S..S+2*NCH-1   : W0^T half-chunks [KT rows x 16] hi | lo   (GEMM-dA B operand: B[n = feature][k = hidden])
__global__ void tc_prep_bwd_kernel(const float* __restrict__ W0, int K, int KT, int H, int slot_floats, float* __restrict__ Wtc) {
    const int S = KT / KS1, NHC = H / HHC;
    const int tid = blockIdx.x * blockDim.x + threadIdx.x, nth = gridDim.x * blockDim.x;
    for (int i = tid; i < S * H * KS1; i += nth) {
        const int kl = i % KS1, h = (i / KS1) % H, s = i / (KS1 * H);
        const int k = s * KS1 + kl;
        const float v = k < K ? W0[(size_t)h * K + k] : 0.f;
        const float hi = tc::tf32_rn(v);
        float* base = Wtc + (size_t)s * slot_floats;
        const uint32_t off = tc::tile_off_b32(h, kl, KS1 / 4) / 4;
        base[off] = hi;
        base[(size_t)H * KS1 + off] = tc::tf32_rn(v - hi);
    }
    for (int i = tid; i < NHC * KT * HHC; i += nth) {
        const int kk = i % HHC, kf = (i / HHC) % KT, c = i / (HHC * KT);
        const float v = kf < K ? W0[(size_t)(c * HHC + kk) * K + kf] : 0.f;
        const float hi = tc::tf32_rn(v);
        float* base = Wtc + (size_t)(S + c) * slot_floats;
        const uint32_t off = tc::tile_off_b32(kf, kk, HHC / 4) / 4;
        base[off] = hi;
        base[(size_t)KT * HHC + off] = tc::tf32_rn(v - hi);
    }
}

// out[h][k] (k < K) += tmp[h][k];  db0[h] += tmp[h][K]
__global__ void tc_fold_wgrad_kernel(const float* __restrict__ tmp, int H, int K, int KT, float* __restrict__ dW0, float* __restrict__ db0) {
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < H * KT; i += gridDim.x * blockDim.x) {
        const int h = i / KT, k = i % KT;
        const float v = tmp[i];
        if (k < K) dW0[(size_t)h * K + k] += v;
        else if (k == K) db0[h] += v;
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

__global__ void __launch_bounds__(NTH, 1) sdf_stencil_bwd_tc_kernel(TcBwdParams p) {
    extern __shared__ __align__(1024) uint8_t smem[];
    __shared__ site::LevelTab s_tab;
    const int H = p.H, KT = p.KT, S = KT / KS1, NCH = H / HCH, J = S + H / HHC;
    constexpr int SPT = site::SPT;
    const uint32_t a_part = site::a_part_bytes(KT);
    const uint32_t slot_bytes = (uint32_t)p.slot_floats * 4;
    const int DAS = KT + 4;                                        // row stride of the dA tile
    uint8_t* a_hi = smem;
    uint8_t* a_lo = a_hi + a_part;
    float* dAs = p.da_scratch + (size_t)blockIdx.x * TM * DAS;     // [TM][DAS] fp32, math group -> memory group (global / L2:
                                                                   // shared memory goes to the A operand and a deep weight ring)
    uint8_t* wst = a_lo + a_part;
    float* b0s = reinterpret_cast<float*>(wst + (size_t)NST * slot_bytes);
    float* w1s = b0s + H;
    float* accw1 = w1s + H;                                        // per-CTA dW1[0,:]
    float* gqs = accw1 + H;                                        // [TM] upstream gradient of each row's SDF value
    uint64_t* bars = reinterpret_cast<uint64_t*>(gqs + TM);
    uint64_t* full = bars;
    uint64_t* empty = bars + NST;
    uint64_t* dfull1 = bars + 2 * NST;                             // GEMM1 accumulator complete (= A operand consumed)
    uint64_t* dfull2 = dfull1 + 1;                                 // dA accumulator complete
    uint64_t* cfree = dfull2 + 1;                                  // [2] dPre chunk (TMEM) consumed by its MMAs
    uint64_t* aready = cfree + 2;                                  // A operand of the next tile gathered
    uint64_t* daready = aready + 1;                                // dA tile in shared memory
    uint64_t* dafree = daready + 1;                                // dA tile scattered
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(dafree + 1);
    float* accb1 = reinterpret_cast<float*>(tmem_slot + 1);

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int64_t ntiles = (p.n + SPT - 1) / SPT;
    const int64_t my_tiles = blockIdx.x < ntiles ? (ntiles - blockIdx.x + gridDim.x - 1) / gridDim.x : 0;

    if (warp == 0) tc::tmem_alloc<512>(tmem_slot);
    if (tid == 0) {
        for (int i = 0; i < NST; ++i) { tc::mbar_init(&full[i], 1); tc::mbar_init(&empty[i], 1); }
        tc::mbar_init(dfull1, 1); tc::mbar_init(dfull2, 1); tc::mbar_init(&cfree[0], 1); tc::mbar_init(&cfree[1], 1);
        tc::mbar_init(aready, NGRP); tc::mbar_init(daready, NGRP); tc::mbar_init(dafree, NGRP);
        tc::mbar_fence_init();
        *accb1 = 0.f;
    }
    for (int i = tid; i < H; i += NTH) { b0s[i] = p.b0[i]; w1s[i] = p.w1r0[i]; accw1[i] = 0.f; }
    site::build_level_tab(p.f, &s_tab);
    tc::fence_before_sync();
    __syncthreads();
    tc::fence_after_sync();
    const uint32_t tmem_base = *tmem_slot;

    if (tid >= NGRP) {
        // ======================= memory group: gather tile t+1, scatter tile t-1 ========================================
        // the batched texel fetches want registers, the math group needs few: rebalance the 64K register file
        asm volatile("setmaxnreg.inc.sync.aligned.u32 160;");
        const int mtid = tid - NGRP;
        PROF_DECL
        for (int64_t lt = 0; lt < my_tiles; ++lt) {
            const int64_t tile = blockIdx.x + lt * gridDim.x;
            if (lt > 0) tc::mbar_wait(dfull1, (uint32_t)((lt - 1) & 1));       // GEMM1 of the previous tile has consumed A
            PROF(0)
            if (!TF_DBG(p, 1))
                site::gather_tile_lean(p.f, s_tab, p.xyz, p.level, p.n, p.units, tile * SPT, KT, a_hi, a_lo,
                                  TF_DBG(p, 2) ? nullptr : p.arow + (size_t)tile * TM * KT, NGRP, mtid);
            tc::fence_async_smem();
            tc::mbar_arrive(aready);
            PROF(1)
            if (lt > 0) {
                tc::mbar_wait(daready, (uint32_t)((lt - 1) & 1));
                PROF(2)
                if (!TF_DBG(p, 4))
                    site::scatter_tile_lean(p.f, s_tab, p.g, p.xyz, p.level, p.n, p.units, (blockIdx.x + (lt - 1) * gridDim.x) * SPT, dAs, DAS, NGRP, mtid, true);
                tc::mbar_arrive(dafree);
                PROF(3)
            }
        }
        if (mtid == 0) { PROF_DUMP(2) }
        if (my_tiles > 0) {
            tc::mbar_wait(daready, (uint32_t)((my_tiles - 1) & 1));
            if (!TF_DBG(p, 4))
                site::scatter_tile_lean(p.f, s_tab, p.g, p.xyz, p.level, p.n, p.units, (blockIdx.x + (my_tiles - 1) * gridDim.x) * SPT, dAs, DAS, NGRP, mtid, true);
        }
    } else {
        // ======================= math group: GEMM1, chunked dPre epilogue, GEMM-dA ======================================
        asm volatile("setmaxnreg.dec.sync.aligned.u32 96;");
        const int lq = warp & 3, half = warp >> 2;
        const int row = lq * 32 + lane;
        const int row_s = row / NQ7, row_q = row - row_s * NQ7;
        const uint32_t d1 = tmem_base, d2 = tmem_base + 256, chunk_a = tmem_base + 384;   // chunk_a: 2 x (hi 32 | lo 32) columns
        const uint32_t idesc1 = tc::make_idesc(2, 2, TM, H), idesc2 = tc::make_idesc(2, 2, TM, KT);
        const uint32_t a_sbo = site::a_sbo(KT), w1_sbo = (KS1 / 4) * 128, w2_sbo = (HHC / 4) * 128;
        const uint64_t a_desc_hi = tc::make_smem_desc(tc::smem_u32(a_hi), site::A_LBO, a_sbo), a_desc_lo = tc::make_smem_desc(tc::smem_u32(a_lo), site::A_LBO, a_sbo);

        int64_t g_mma = 0;                         // driver (thread 0): ring slot counter
        const int64_t total_slots = my_tiles * J;
        uint32_t cf_commits[2] = {0, 0};           // commits issued on cfree[buf] so far
        // W ring refills: cp.async.bulk copies issued by ONE warp execute one after the other (~800-900 cycles each
        // whatever their size: tests/probes/bulk_probe.cu), copies of different warps overlap.  So every ring stage has
        // its own issuing lane (lane 0 of warps 4..7: stages 0..3) and the MMA thread only posts the byte count.  A slot is
        // refilled NST slots ahead of the MMAs that consume it, at points where the MMAs that free its stage were issued
        // at least one chunk earlier, so the issuing lanes (which are epilogue warps too) rarely wait.
        const int fill_k = (lane == 0 && warp >= 4 && warp < 4 + NST) ? warp - 4 : -1;
        int64_t g_fill = fill_k;                   // next slot of this issuer (slots g = k, k + NST, ...)
        auto pump_to = [&](int64_t limit) {        // refill this issuer's slots below `limit`
            if (fill_k < 0) return;
            while (g_fill < limit && g_fill < total_slots) {
                tc::mbar_wait(&empty[fill_k], (uint32_t)(((g_fill / NST) & 1) ^ 1));   // MMAs of slot g_fill - NST are complete
                bulk_copy_g2s(wst + (size_t)fill_k * slot_bytes, p.Wtc + (size_t)(g_fill % J) * p.slot_floats, slot_bytes, &full[fill_k]);
                g_fill += NST;
            }
        };
        pump_to(NST);
        const float inv2e[3] = {1.f / (2.f * p.units[0]), 1.f / (2.f * p.units[1]), 1.f / (2.f * p.units[2])};
        const float inve2[3] = {1.f / (p.units[0] * p.units[0]), 1.f / (p.units[1] * p.units[1]), 1.f / (p.units[2] * p.units[2])};
        PROF_DECL

        for (int64_t lt = 0; lt < my_tiles; ++lt) {
            const int64_t tile = blockIdx.x + lt * gridDim.x;
            const int64_t s_base = tile * SPT;
            const int64_t tile_row0 = tile * TM;
            const uint32_t tpar = (uint32_t)(lt & 1);
            PROF(0)
            // upstream gradients -> per-query SDF gradients of the tile's samples (adjoint of fields.py:245-256); done by warp 1
            // while thread 0 (warp 0) already issues GEMM1: the HBM reads of this block are not on the MMA thread's path
            if (tid >= 32 && tid < 32 + SPT) {
                const int ts = tid - 32;
                const int64_t n = s_base + ts;
                float gq[NQ7];
#pragma unroll
                for (int r = 0; r < NQ7; ++r) gq[r] = 0.f;
                if (n < p.n) {
                    float sd[NQ7], gg[3] = {0.f, 0.f, 0.f}, gh = 0.f, gs = 0.f;
#pragma unroll
                    for (int r = 0; r < NQ7; ++r) sd[r] = __ldg(p.sdf7 + n * NQ7 + r);      // all reads first: one round trip
                    if (p.g_hess) gh = __ldg(p.g_hess + n);
                    if (p.g_sdf) gs = __ldg(p.g_sdf + n);
                    if (p.g_grad) { gg[0] = __ldg(p.g_grad + n * 3); gg[1] = __ldg(p.g_grad + n * 3 + 1); gg[2] = __ldg(p.g_grad + n * 3 + 2); }
                    // (short on purpose: this block runs once per tile in one warp, so its instructions are fetched cold every
                    // time; the reciprocals of the finite-difference steps are loop constants)
                    float g[3], h[3];
#pragma unroll
                    for (int k = 0; k < 3; ++k) {
                        g[k] = (sd[1 + 2 * k] - sd[2 + 2 * k]) * inv2e[k];
                        h[k] = (sd[1 + 2 * k] + sd[2 + 2 * k] - 2.f * sd[0]) * inve2[k];
                    }
                    const float rD = 1.f / (g[0] * g[0] + g[1] * g[1] + g[2] * g[2] + 1e-5f);
                    const float nh = (g[0] * h[0] + g[1] * h[1] + g[2] * h[2]) * rD;
                    gq[0] = gs;
#pragma unroll
                    for (int k = 0; k < 3; ++k) {
                        const float Gk = gg[k] + gh * (h[k] * rD - 2.f * g[k] * nh * rD);
                        const float Hk = gh * g[k] * rD;
                        gq[1 + 2 * k] = Gk * inv2e[k] + Hk * inve2[k];
                        gq[2 + 2 * k] = -Gk * inv2e[k] + Hk * inve2[k];
                        gq[0] -= 2.f * Hk * inve2[k];
                    }
                }
                float tot = 0.f;
#pragma unroll
                for (int r = 0; r < NQ7; ++r) { gqs[ts * NQ7 + r] = gq[r]; tot += gq[r]; }
                if (tot != 0.f) atomicAdd(accb1, tot);
            } else if (tid >= 32 + SPT && tid < 32 + SPT + 2) {
                gqs[SPT * NQ7 + tid - 32 - SPT] = 0.f;
            }
            // ---- GEMM1 (thread 0): pre = A W0^T ----------------------------------------------------------------------
            if (tid == 0) {
                PROF(14)
                tc::mbar_wait(aready, tpar);
                tc::fence_after_sync();
                PROF(13)
                for (int s = 0; s < S; ++s) {
                    const int st = (int)(g_mma % NST);
                    mbar_expect_tx(&full[st], slot_bytes);
                    tc::mbar_wait(&full[st], (uint32_t)((g_mma / NST) & 1));
                    tc::fence_after_sync();
                    PROF(11)
                    const uint32_t w_hi = tc::smem_u32(wst + (size_t)st * slot_bytes);
                    const uint64_t wdh0 = tc::make_smem_desc(w_hi, 128, w1_sbo), wdl0 = tc::make_smem_desc(w_hi + (uint32_t)H * KS1 * 4, 128, w1_sbo);
#pragma unroll
                    for (int ks = 0; ks < KS1 / 8; ++ks) {
                        const uint32_t koff = (uint32_t)(s * (KS1 / 8) + ks) * 2 * site::A_LBO;
                        const uint64_t adh = tc::desc_add(a_desc_hi, koff), adl = tc::desc_add(a_desc_lo, koff);
                        const uint64_t wdh = tc::desc_add(wdh0, ks * 256), wdl = tc::desc_add(wdl0, ks * 256);
                        tc::mma_tf32_ss(d1, adh, wdh, idesc1, (s | ks) != 0);
                        tc::mma_tf32_ss(d1, adh, wdl, idesc1, 1);
                        tc::mma_tf32_ss(d1, adl, wdh, idesc1, 1);
                    }
                    tc::mma_commit(&empty[st]);
                    ++g_mma;
                    PROF(12)
                }
                tc::mma_commit(dfull1);
            }
            const int64_t n = s_base + row_s;
            const bool centre = row_q == 0 && row_s < SPT && n < p.n;
            const bool has_hc = centre && p.dHc;
            // dHidden(centre) of the next chunk is fetched one chunk ahead (the first one under the GEMM1 wait)
            float4 hc[4] = {f4_zero(), f4_zero(), f4_zero(), f4_zero()};
            if (has_hc) {
                const float4* src = reinterpret_cast<const float4*>(p.dHc + (size_t)n * H + half * 16);
#pragma unroll
                for (int j = 0; j < 4; ++j) hc[j] = __ldg(src + j);
            }
            PROF(1)
            pump_to(lt * J + S + NST);                 // the GEMM1 slices of this tile and the slots of chunks 0 and 1
            tc::bar_sync(1, NGRP);                     // gqs visible to the group
            PROF(2)
            tc::mbar_wait(dfull1, tpar);
            tc::fence_after_sync();
            PROF(3)
            // ---- epilogue-1 + GEMM-dA, chunk by chunk over the hidden units -----------------------------------
            const float gq = gqs[row];
            for (int c = 0; c < (TF_DBG(p, 16) ? 0 : NCH); ++c) {
                const int buf = c & 1;
                if (c >= 2) { tc::mbar_wait(&cfree[buf], (cf_commits[buf] - 1) & 1); tc::fence_after_sync(); }
                PROF(4)
                const int col0 = c * HCH + half * 16;
                float v[16];
                tc::tmem_ld16(d1 + ((uint32_t)(lq * 32) << 16) + col0, v);
                if (tid != 0) { PROF(11) }
                float sp[16];
                const float hcv[16] = {hc[0].x, hc[0].y, hc[0].z, hc[0].w, hc[1].x, hc[1].y, hc[1].z, hc[1].w,
                                       hc[2].x, hc[2].y, hc[2].z, hc[2].w, hc[3].x, hc[3].y, hc[3].z, hc[3].w};
                if (has_hc && c + 1 < NCH) {
                    const float4* src = reinterpret_cast<const float4*>(p.dHc + (size_t)n * H + col0 + HCH);
#pragma unroll
                    for (int j = 0; j < 4; ++j) hc[j] = __ldg(src + j);
                }
#pragma unroll
                for (int j = 0; j < 16; j += 4) {
                    const float4 bb = *reinterpret_cast<const float4*>(b0s + col0 + j);
                    const float4 ww = *reinterpret_cast<const float4*>(w1s + col0 + j);
                    float sg[4];
                    float pre0, pre1, pre2, pre3;
                    unpack2(fadd2(pack2(v[j], v[j + 1]), pack2(bb.x, bb.y)), pre0, pre1);
                    unpack2(fadd2(pack2(v[j + 2], v[j + 3]), pack2(bb.z, bb.w)), pre2, pre3);
                    softplus100_fast_both2(pre0, pre1, sp[j], sp[j + 1], sg[0], sg[1]);
                    softplus100_fast_both2(pre2, pre3, sp[j + 2], sp[j + 3], sg[2], sg[3]);
                    // dPre = dPost * sigmoid, dPost = gq W1[0,:] + [centre] g_feat W1[1:]
                    const uint64_t gg = bcast2(gq);
                    unpack2(fmul2(ffma2(gg, pack2(ww.x, ww.y), pack2(hcv[j], hcv[j + 1])), pack2(sg[0], sg[1])), v[j], v[j + 1]);
                    unpack2(fmul2(ffma2(gg, pack2(ww.z, ww.w), pack2(hcv[j + 2], hcv[j + 3])), pack2(sg[2], sg[3])), v[j + 2], v[j + 3]);
                }
                if (tid != 0) { PROF(12) }
                // dPre of the tile is stored [H][128] (row fastest): a warp's 32 rows of one column are one 128-byte store wavefront
                // (row-major 16-byte pieces cost 8), and X^T Y reads 4 rows of a column as one K-major unit without transposing
                float* dst = p.dpre + (size_t)tile_row0 * H + (size_t)col0 * TM + row;
#pragma unroll
                for (int j = 0; j < 16; ++j)
                    if (!TF_DBG(p, 2)) dst[j * TM] = v[j];
                {   // the chunk becomes the A operand of the dA MMAs straight in tensor memory (tf32 hi | lo, lane = row)
                    float lo[16];
#pragma unroll
                    for (int j = 0; j < 16; ++j) { const float h = tc::tf32_rn(v[j]); lo[j] = tc::tf32_rn(v[j] - h); v[j] = h; }
                    const uint32_t ca = chunk_a + (uint32_t)buf * 64 + ((uint32_t)(lq * 32) << 16) + half * 16;
                    tc::tmem_st16(ca, v);
                    tc::tmem_st16(ca + 32, lo);
                    tc::tmem_st_wait();
                }
                if (tid != 0) { PROF(13) }
                if (!TF_DBG(p, 8)) {
                    // 16 column sums over the warp's 32 rows with 16 shuffles: every exchange halves the columns a lane owns
                    float w8[8], w4[4], w2[2];
                    const bool b16 = lane & 16, b8 = lane & 8, b4 = lane & 4, b2 = lane & 2;
#pragma unroll
                    for (int j = 0; j < 8; ++j) {
                        const float lo_v = gq * sp[j], hi_v = gq * sp[j + 8];
                        w8[j] = (b16 ? hi_v : lo_v) + __shfl_xor_sync(0xffffffffu, b16 ? lo_v : hi_v, 16);
                    }
#pragma unroll
                    for (int j = 0; j < 4; ++j) w4[j] = (b8 ? w8[j + 4] : w8[j]) + __shfl_xor_sync(0xffffffffu, b8 ? w8[j] : w8[j + 4], 8);
#pragma unroll
                    for (int j = 0; j < 2; ++j) w2[j] = (b4 ? w4[j + 2] : w4[j]) + __shfl_xor_sync(0xffffffffu, b4 ? w4[j] : w4[j + 2], 4);
                    float w1 = (b2 ? w2[1] : w2[0]) + __shfl_xor_sync(0xffffffffu, b2 ? w2[0] : w2[1], 2);
                    w1 += __shfl_xor_sync(0xffffffffu, w1, 1);
                    const int col = (b16 ? 8 : 0) + (b8 ? 4 : 0) + (b4 ? 2 : 0) + (b2 ? 1 : 0);
                    if (!(lane & 1) && w1 != 0.f) atomicAdd(&accw1[col0 + col], w1);
                }
                PROF(5)
                tc::fence_before_sync();
                tc::bar_sync(1, NGRP);
                tc::fence_after_sync();
                PROF(6)
                pump_to(lt * J + S + (HCH / HHC) * c + NST);   // slots of the next chunk (after the last one: first slices of the next tile)
                if (tid == 0) {
                    const uint32_t ah = chunk_a + (uint32_t)buf * 64, al = ah + 32;
#pragma unroll
                    for (int hh = 0; hh < HCH / HHC; ++hh) {
                        const int st = (int)(g_mma % NST);
                        mbar_expect_tx(&full[st], slot_bytes);
                        tc::mbar_wait(&full[st], (uint32_t)((g_mma / NST) & 1));
                        tc::fence_after_sync();
                        const uint32_t w_hi = tc::smem_u32(wst + (size_t)st * slot_bytes);
                        const uint64_t wdh0 = tc::make_smem_desc(w_hi, 128, w2_sbo), wdl0 = tc::make_smem_desc(w_hi + (uint32_t)KT * HHC * 4, 128, w2_sbo);
#pragma unroll
                        for (int ks = 0; ks < HHC / 8; ++ks) {
                            const uint64_t wdh = tc::desc_add(wdh0, ks * 256), wdl = tc::desc_add(wdl0, ks * 256);
                            const uint32_t kc = hh * HHC + ks * 8;
                            tc::mma_tf32_ts(d2, ah + kc, wdh, idesc2, (c | hh | ks) != 0);
                            tc::mma_tf32_ts(d2, ah + kc, wdl, idesc2, 1);
                            tc::mma_tf32_ts(d2, al + kc, wdh, idesc2, 1);
                        }
                        tc::mma_commit(&empty[st]);
                        ++g_mma;
                    }
                    tc::mma_commit(&cfree[buf]);
                    if (c == NCH - 1) tc::mma_commit(dfull2);
                }
                ++cf_commits[buf];
                PROF(7)
            }
            if (TF_DBG(p, 16)) {
                for (int c = 0; c < NCH; ++c) {           // timing experiments: the skipped slots still rotate through the ring
                    pump_to(lt * J + S + (HCH / HHC) * c + NST);
                    if (tid == 0) {
                        for (int hh = 0; hh < HCH / HHC; ++hh) {
                            const int st = (int)(g_mma % NST);
                            mbar_expect_tx(&full[st], slot_bytes);
                            tc::mbar_wait(&full[st], (uint32_t)((g_mma / NST) & 1));
                            tc::mma_commit(&empty[st]);
                            ++g_mma;
                        }
                    }
                }
            } else {
                tc::mbar_wait(dfull2, tpar);
            }
            tc::fence_after_sync();
            PROF(8)
            // ---- dA: TMEM -> shared memory (fp32, row-major) once the memory group has scattered the previous tile ----
            if (lt > 0) tc::mbar_wait(dafree, (uint32_t)((lt - 1) & 1));
            PROF(9)
            for (int c0 = half * 16; c0 < KT; c0 += 32) {
                float v[16];
                tc::tmem_ld16(d2 + ((uint32_t)(lq * 32) << 16) + c0, v);
                float4* dst = reinterpret_cast<float4*>(dAs + (size_t)row * DAS + c0);
#pragma unroll
                for (int j = 0; j < 4; ++j) dst[j] = make_float4(v[4 * j], v[4 * j + 1], v[4 * j + 2], v[4 * j + 3]);
            }
            tc::fence_before_sync();
            tc::mbar_arrive(daready);
            PROF(10)
        }
        if (tid == 0) { PROF_DUMP(1) }
        if (tid == 32) { PROF_DUMP(0) }
    }
    __syncthreads();
    for (int i = tid; i < H; i += NTH)
        if (accw1[i] != 0.f) atomicAdd(p.dW1r0 + i, accw1[i]);
    if (tid == 0 && *accb1 != 0.f) atomicAdd(p.db1, *accb1);
    tc::fence_before_sync();
    __syncthreads();
    if (warp == 0) tc::tmem_dealloc<512>(tmem_base);
}

}  // namespace

int tf_internal_bwd_tc_slot_floats(int KT, int H) {
    const int a = 2 * H * KS1, b = 2 * KT * HHC;
    return a > b ? a : b;
}
size_t tf_internal_bwd_tc_wtc_floats(int KT, int H) { return (size_t)(KT / KS1 + H / HHC) * tf_internal_bwd_tc_slot_floats(KT, H); }
size_t tf_internal_bwd_tc_smem(int KT, int H) {
    return (size_t)2 * 16 * (KT / 4) * site::A_LBO + (size_t)NST * tf_internal_bwd_tc_slot_floats(KT, H) * 4 +
           (size_t)3 * H * 4 + (size_t)TM * 4 + (2 * NST + 9) * 8 + 32;
}

int tf_internal_bwd_tc_prep(const float* W0, int K, int KT, int H, float* wtc, cudaStream_t stream) {
    tc_prep_bwd_kernel<<<64, 256, 0, stream>>>(W0, K, KT, H, tf_internal_bwd_tc_slot_floats(KT, H), wtc);
    tf_count_launches(1);
    return 0;
}

int tf_internal_bwd_tc_fold(const float* tmp, int H, int K, int KT, float* dW0, float* db0, cudaStream_t stream) {
    tc_fold_wgrad_kernel<<<32, 256, 0, stream>>>(tmp, H, K, KT, dW0, db0);
    tf_count_launches(1);
    return 0;
}

int tf_internal_bwd_tc_samples_per_tile() { return site::SPT; }
size_t tf_internal_bwd_tc_scratch_floats(int KT) { return (size_t)tf_num_sms() * TM * (KT + 4); }

// one slice of samples (n <= workspace capacity): activation-side backward
int tf_internal_stencil_bwd_tc(const tf_vm_field_t* f, const tf_vm_mut_t* g, const tf_sdf_mlp_t* m, const float* wtc, const float* xyz,
                               const float* level, int64_t n, const float units[3], const float* sdf7, const float* g_sdf,
                               const float* g_grad, const float* g_hess, const float* dHc, float* dpre, float* arow,
                               float* da_scratch, float* dW1r0, float* db1, cudaStream_t stream) {
    const int C = f->n_comp, K = 3 * C + 3, KT = (K + KSL - 1) / KSL * KSL, H = m->hidden;
    TcBwdParams p = {};
    p.f = *f; p.g = *g; p.xyz = xyz; p.level = level; p.n = n;
    p.Wtc = wtc; p.b0 = m->b0; p.w1r0 = m->W1;
    p.sdf7 = sdf7; p.g_sdf = g_sdf; p.g_grad = g_grad; p.g_hess = g_hess; p.dHc = dHc;
    p.K = K; p.KT = KT; p.H = H; p.slot_floats = tf_internal_bwd_tc_slot_floats(KT, H);
    for (int k = 0; k < 3; ++k) p.units[k] = units[k];
    p.dpre = dpre; p.arow = arow; p.da_scratch = da_scratch; p.dW1r0 = dW1r0; p.db1 = db1;
#ifdef TF_TC_DEBUG_SWITCHES
    { const char* e = getenv("TF_TC_BWD_DEBUG"); p.debug = e ? atoi(e) : 0; }
    static long long* prof_dev = nullptr;
    if (getenv("TF_TC_BWD_PROF")) {
        if (!prof_dev) cudaMalloc(&prof_dev, 48 * sizeof(long long));
        cudaMemsetAsync(prof_dev, 0, 48 * sizeof(long long), stream);
        p.prof = prof_dev;
    }
#endif
    const size_t smem = tf_internal_bwd_tc_smem(KT, H);
    cudaFuncSetAttribute(sdf_stencil_bwd_tc_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    const int64_t ntiles = (n + site::SPT - 1) / site::SPT;
    const int grid = (int)(ntiles < tf_num_sms() ? ntiles : tf_num_sms());
    {
        TfKernelTimer timer("sdf_stencil_bwd_tc", stream);
        sdf_stencil_bwd_tc_kernel<<<grid, NTH, smem, stream>>>(p);
    }
    tf_count_launches(1);
#ifdef TF_TC_DEBUG_SWITCHES
    if (p.prof) {
        long long h[48];
        cudaMemcpy(h, p.prof, sizeof(h), cudaMemcpyDeviceToHost);
        const double tiles = (double)((ntiles + grid - 1) / grid);
        const char* roles[3] = {"math worker (warp 1)", "math driver (thread 0)", "memory (warp 8)"};
        for (int r = 0; r < 3; ++r) {
            fprintf(stderr, "[bwd prof] %-22s cycles/tile:", roles[r]);
            for (int i = 0; i < 15; ++i) fprintf(stderr, " %d:%.0f", i, (double)h[r * 16 + i] / tiles);
            fprintf(stderr, "\n");
        }
    }
#endif
    return 0;
}
