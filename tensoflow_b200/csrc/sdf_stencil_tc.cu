// Fused TensoSDF stencil forward on the 5th-gen tensor cores (tcgen05 + TMEM), sm_100a.
//
// Same contract as the SIMT kernel in sdf_stencil.cu (reference network/fields.py:262-299, 227-260)
// but the decoder's first layer -- 7 x [N,K] x [K,H], 85 % of the decoder FLOPs -- runs as
// tcgen05.mma kind::tf32 with fp32-level accuracy from operand splitting
// (x = hi + lo, D = A_hi W_hi + A_hi W_lo + A_lo W_hi: "3xTF32").
//
// One persistent CTA per SM (16 worker warps + a driver warp) walks MMA tiles of M = 128 rows.  In stencil mode a
// tile is sample-major: 18 samples x 7 queries (centre, +-x, +-y, +-z) so that the queries of a sample share
// their plane / line fetches (stencil_site.cuh); in SDF-only mode it is 128 samples:
//   gather  : workers; one (sample, plane, channel group) site per thread and pass, texel reads are 144-byte
//             runs per site; fp32 rows go to a staging tile in shared memory (padded K-chunk stride:
//             conflict-free stores and reads)
//   A       : the staging tile moves to TENSOR MEMORY split into tf32 hi | lo (thread = row, tcgen05.st), so the
//             MMAs of tile t read A from TMEM while the workers already gather tile t+1 into the staging tile
//   W0      : pre-split / pre-tiled once per call into K-slices of 16 (prep kernel); slices stream
//             L2 -> shared memory through a 3-stage ring with cp.async.bulk + mbarrier, one issuing warp per stage
//   MMA     : driver thread issues 6 tcgen05.mma per slice (2 k-steps x 3 passes, A from TMEM), accumulator
//             [128 x H] fp32 in TMEM (256 columns) next to A hi | lo (2 x KT columns)
//   epilogue: tcgen05.ld -> +b0 -> Softplus(beta=100) -> dot with W1[0,:] (the SDF output; taps need nothing
//             else); the centre rows also stream their hidden activations to HBM for the appearance head
//             (second layer, [N,H] x [H,A])
//   finalize: per tile, the 7 SDF values of a sample -> sdf7, central-difference gradient, hessian term.
#include <stdlib.h>
#include "common.cuh"
#include "tc_common.cuh"
#include "stencil_site.cuh"
#include "internal.cuh"

namespace {

constexpr int TM = 128;     // rows per MMA tile = samples per block
constexpr int NQ7 = 7;
constexpr int KSL = 16;     // K-slice (2 tf32 MMA k-steps)
constexpr int NST = 3;      // W ring stages = issuing warps of the driver group (see the W ring comment in the kernel)
constexpr int NWORK = 512;  // 16 worker warps: the gather is latency-bound, thread-level parallelism hides it
constexpr int NTH = NWORK + 128; // + the driver warpgroup (one lane of its first warp: W ring + MMA issue); register
                                // rebalancing (setmaxnreg) is per warpgroup, hence a whole one
constexpr int NCG = NWORK / 128; // column groups of the epilogue (warps sharing a TMEM lane quarter)

struct TcParams {
    tf_vm_field_t f;
    const float* xyz;
    const float* level;
    int64_t n;
    const float* W0tc;   // [S][2][H*16] pre-tiled hi/lo slices
    const float* b0;
    const float* w1r0;   // W1 row 0
    const float* b1;
    int K, KT, H, nq;    // nq = 7 (stencil) or 1 (sdf only)
    float units[3];
    float* sdf7; float* grad; float* hess; float* sdf1;
    float* spc;          // [n][H] centre hidden activations (NULL = not needed)
#ifdef TF_TC_DEBUG_SWITCHES
    int debug;           // timing experiments only (never compiled into the product library): 1 skip gathers, 2 skip MMAs, 4 skip epilogue math, 8 skip the per-sample finalize
#endif
};

// timing-experiment switches exist only in builds made with -DTF_TC_DEBUG_SWITCHES; the product library has none
#ifdef TF_TC_DEBUG_SWITCHES
#define TF_DBG(p, bit) ((p).debug & (bit))
#else
#define TF_DBG(p, bit) 0
#endif

__global__ void tc_prep_w0_kernel(const float* __restrict__ W0, int K, int KT, int H, float* __restrict__ W0tc) {
    const int S = KT / KSL;
    const int total = S * H * KSL;
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < total; i += gridDim.x * blockDim.x) {
        const int kl = i % KSL, h = (i / KSL) % H, s = i / (KSL * H);
        const int k = s * KSL + kl;
        const float v = k < K ? W0[(size_t)h * K + k] : 0.f;
        const float hi = tc::tf32_rn(v);
        const float lo = tc::tf32_rn(v - hi);
        const uint32_t off = tc::tile_off_b32(h, kl, KSL / 4) / 4;
        float* base = W0tc + (size_t)s * 2 * H * KSL;
        base[off] = hi;
        base[(size_t)H * KSL + off] = lo;
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

// SDF-only mode: gather the feature rows of 128 samples (one query each) into the fp32 staging tile
__device__ __forceinline__ void tc_gather_rows(const TcParams& p, int64_t s_base, uint8_t* a_st) {
    const int C = p.f.n_comp, C4 = C / 4, G = p.KT / 4;
    const bool has_level = p.level != nullptr;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    // unit = (8-row group, plane): lane -> (row = lane%8, channel groups lane/8, lane/8+4, ...); the
    // sampling plan of the (row, plane) pair is computed once and reused for its channel groups
    const int n_units = (TM / 8) * 3;
    for (int u = warp; u < n_units; u += NWORK / 32) {
        const int rg = u / 3, i = u % 3;
        const int row = rg * 8 + (lane & 7);
        const int64_t n = s_base + row;
        const bool valid = n < p.n;
        VmTaps taps;
        if (valid) {
            const float x[3] = {p.xyz[n * 3 + 0], p.xyz[n * 3 + 1], p.xyz[n * 3 + 2]};
            taps = vm_taps(p.f, x, has_level ? p.level[n] : 0.f, has_level, i);
        }
        for (int c4 = lane >> 3; c4 < C4; c4 += 4) {
            float4 v = f4_zero();
            if (valid) {
                float4 P, L;
                vm_fetch(taps, C, c4 * 4, P, L);
                v = f4_mul(P, L);
            }
            site::put(a_st, nullptr, site::a_off(row, i * C4 + c4, p.KT), v);
        }
    }
    // raw xyz (fields.py:265,298) + zero padding groups
    const int tail_g = G - 3 * C4;
    for (int it = threadIdx.x; it < TM * tail_g; it += NWORK) {
        const int row = it % TM, g = 3 * C4 + it / TM;
        const int64_t n = s_base + row;
        float4 v = f4_zero();
        if (g == 3 * C4 && n < p.n) v = make_float4(p.xyz[n * 3 + 0], p.xyz[n * 3 + 1], p.xyz[n * 3 + 2], 0.f);
        site::put(a_st, nullptr, site::a_off(row, g, p.KT), v);
    }
}

__device__ __forceinline__ void tc_gather(const TcParams& p, const site::LevelTab& s_tab, int64_t tile, uint8_t* a_st) {
    if (p.nq == NQ7) site::gather_tile_lean(p.f, s_tab, p.xyz, p.level, p.n, p.units, tile * site::SPT, p.KT, a_st, nullptr, nullptr, NWORK, threadIdx.x);
    else tc_gather_rows(p, tile * TM, a_st);
}

// staging tile (fp32, shared memory) -> A operand in tensor memory, split into tf32 hi | lo: thread = row (lane of its
// warp's TMEM quarter), the four warps of a quarter share the 16-column units
__device__ __forceinline__ void tc_stage_to_tmem(const uint8_t* a_st, int KT, uint32_t a_tmem, int lq, int chh, int lane) {
    const int row = lq * 32 + lane;
    const uint32_t lane_sel = (uint32_t)(lq * 32) << 16;
    for (int u = chh; u < KT / 16; u += NCG) {
        float hi[16], lo[16];
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const float4 v = *reinterpret_cast<const float4*>(a_st + site::a_off(row, u * 4 + j, KT));
            const float4 h = site::tf32_hi(v), l = site::tf32_lo(v, h);
            hi[4 * j] = h.x; hi[4 * j + 1] = h.y; hi[4 * j + 2] = h.z; hi[4 * j + 3] = h.w;
            lo[4 * j] = l.x; lo[4 * j + 1] = l.y; lo[4 * j + 2] = l.z; lo[4 * j + 3] = l.w;
        }
        tc::tmem_st16(a_tmem + lane_sel + u * 16, hi);
        tc::tmem_st16(a_tmem + lane_sel + KT + u * 16, lo);
    }
    tc::tmem_st_wait();
}

__global__ void __launch_bounds__(NTH, 1) sdf_stencil_fwd_tc_kernel(TcParams p) {
    extern __shared__ __align__(1024) uint8_t smem[];
    __shared__ site::LevelTab s_tab;
    const int H = p.H, KT = p.KT, S = KT / KSL, nq = p.nq;
    const int spt = nq == NQ7 ? site::SPT : TM;               // samples per tile
    const uint32_t a_part = site::a_part_bytes(KT);           // bytes of the fp32 staging tile
    const uint32_t w_part = (uint32_t)H * KSL * 4;            // bytes of one W slice part
    uint8_t* a_st = smem;
    uint8_t* wst = a_st + a_part;                             // NST stages x (hi, lo)
    float* b0s = reinterpret_cast<float*>(wst + (size_t)NST * 2 * w_part);
    float* w1s = b0s + H;
    float* sdfs = w1s + H;                                    // [2 tiles][NCG column groups][TM]
    uint64_t* bars = reinterpret_cast<uint64_t*>(sdfs + 2 * NCG * TM);
    uint64_t* full = bars;                                    // [NST]
    uint64_t* empty = bars + NST;                             // [NST]
    uint64_t* dfull = bars + 2 * NST;                         // accumulator of the tile complete (= A operand consumed)
    uint64_t* aready = dfull + 1;                             // A operand of the tile is in tensor memory, accumulator drained
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(aready + 1);

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int64_t ntiles = (p.n + spt - 1) / spt;
    // tiles of this CTA: blockIdx.x, blockIdx.x + gridDim.x, ...
    const int64_t my_tiles = blockIdx.x < ntiles ? (ntiles - blockIdx.x + gridDim.x - 1) / gridDim.x : 0;

    if (warp == 0) tc::tmem_alloc<512>(tmem_slot);
    if (tid == 0) {
        for (int i = 0; i < NST; ++i) { tc::mbar_init(&full[i], 1); tc::mbar_init(&empty[i], 1); }
        tc::mbar_init(dfull, 1); tc::mbar_init(aready, NWORK);
        tc::mbar_fence_init();
    }
    for (int i = tid; i < H; i += NTH) { b0s[i] = p.b0[i]; w1s[i] = p.w1r0[i]; }
    site::build_level_tab(p.f, &s_tab);
    tc::fence_before_sync();
    __syncthreads();
    tc::fence_after_sync();
    const uint32_t tmem_base = *tmem_slot;
    const uint32_t d_tmem = tmem_base, a_tmem = tmem_base + 256;          // D [128 x H] | A hi [128 x KT] | A lo [128 x KT]

    if (tid >= NWORK) {
        // ======================= driver: stream the W slices, issue the MMAs (A from tensor memory) ===================
        asm volatile("setmaxnreg.dec.sync.aligned.u32 24;");
        const int dw = warp - NWORK / 32;                     // warp of the driver group
        const uint32_t w_sbo = (KSL / 4) * 128;
        const int64_t total_slices = my_tiles * S;
        if (dw == 0 && lane == 0) {
            // ---- MMA thread: A from tensor memory, W slices from the ring ------------------------------------------
            const uint32_t idesc = tc::make_idesc(2, 2, TM, H);
            int64_t g_mma = 0;
            for (int64_t t = 0; t < my_tiles; ++t) {
                tc::mbar_wait(aready, (uint32_t)(t & 1));
                tc::fence_after_sync();
                for (int s = 0; s < S; ++s) {
                    const int st = (int)(g_mma % NST);
                    mbar_expect_tx(&full[st], 2 * w_part);
                    tc::mbar_wait(&full[st], (uint32_t)((g_mma / NST) & 1));
                    tc::fence_after_sync();
                    const uint32_t w_hi = tc::smem_u32(wst + (size_t)st * 2 * w_part);
                    const uint64_t wdh0 = tc::make_smem_desc(w_hi, 128, w_sbo), wdl0 = tc::make_smem_desc(w_hi + w_part, 128, w_sbo);
#pragma unroll
                    for (int ks = 0; ks < KSL / 8; ++ks) {
                        if (TF_DBG(p, 2)) break;
                        const uint32_t kc = (uint32_t)(s * KSL + ks * 8);
                        const uint64_t wdh = tc::desc_add(wdh0, ks * 256), wdl = tc::desc_add(wdl0, ks * 256);
                        tc::mma_tf32_ts(d_tmem, a_tmem + kc, wdh, idesc, (s | ks) != 0);
                        tc::mma_tf32_ts(d_tmem, a_tmem + kc, wdl, idesc, 1);
                        tc::mma_tf32_ts(d_tmem, a_tmem + KT + kc, wdh, idesc, 1);
                    }
                    tc::mma_commit(&empty[st]);
                    ++g_mma;
                }
                tc::mma_commit(dfull);
            }
        } else if (dw >= 1 && lane == 0) {
            // ---- W ring: cp.async.bulk copies issued by ONE warp execute one after the other (~800-900 cycles each whatever
            // their size: tests/probes/bulk_probe.cu), copies of different warps overlap: one issuing warp per ring stage
            const int k = dw - 1;
            for (int64_t g = k; g < total_slices; g += NST) {
                tc::mbar_wait(&empty[k], (uint32_t)(((g / NST) & 1) ^ 1));
                bulk_copy_g2s(wst + (size_t)k * 2 * w_part, p.W0tc + (size_t)(g % S) * 2 * H * KSL, 2 * w_part, &full[k]);
            }
        }
    } else {
        // ======================= workers: gather tile t+1 while the MMAs of tile t run, then epilogue of tile t ========
        asm volatile("setmaxnreg.inc.sync.aligned.u32 112;");
        const int lq = warp & 3, chh = warp >> 2;
        const int row = lq * 32 + lane;
        const float inv2e[3] = {1.f / (2.f * p.units[0]), 1.f / (2.f * p.units[1]), 1.f / (2.f * p.units[2])};
        const float inve2[3] = {1.f / (p.units[0] * p.units[0]), 1.f / (p.units[1] * p.units[1]), 1.f / (p.units[2] * p.units[2])};
        tc_gather(p, s_tab, blockIdx.x, a_st);
        tc::bar_sync(1, NWORK);
        tc_stage_to_tmem(a_st, KT, a_tmem, lq, chh, lane);
        tc::fence_before_sync();
        tc::mbar_arrive(aready);
        for (int64_t t = 0; t < my_tiles; ++t) {
            const int64_t tile = blockIdx.x + t * gridDim.x;
            tc::bar_sync(1, NWORK);                              // every warp has read the staging tile: it is free again
            if (t + 1 < my_tiles && !TF_DBG(p, 1)) tc_gather(p, s_tab, blockIdx.x + (t + 1) * gridDim.x, a_st);
            // ---- epilogue of tile t --------------------------------------------------------------------------------
            tc::mbar_wait(dfull, (uint32_t)(t & 1));
            tc::fence_after_sync();
            const int s = row / nq, q = row - s * nq;
            const int64_t n = tile * spt + s;
            const bool centre = q == 0 && s < spt && n < p.n;
            const uint32_t dcol = d_tmem + ((uint32_t)(lq * 32) << 16);
            uint64_t psum2 = pack2(0.f, 0.f);                 // two interleaved partial sums (packed FFMA2)
            for (int c0 = chh * 32; c0 < H; c0 += 32 * NCG) {
                if (TF_DBG(p, 4)) break;
#pragma unroll
                for (int hh = 0; hh < 2; ++hh) {            // two 16-column reads keep the register footprint small
                    const int cc = c0 + hh * 16;
                    float v[16];
                    tc::tmem_ld16(dcol + cc, v);
#pragma unroll
                    for (int j = 0; j < 16; j += 4) {
                        const float4 bb = *reinterpret_cast<const float4*>(b0s + cc + j);
                        const float4 ww = *reinterpret_cast<const float4*>(w1s + cc + j);
                        float pre0, pre1, pre2, pre3;
                        unpack2(fadd2(pack2(v[j], v[j + 1]), pack2(bb.x, bb.y)), pre0, pre1);
                        unpack2(fadd2(pack2(v[j + 2], v[j + 3]), pack2(bb.z, bb.w)), pre2, pre3);
                        softplus100_fast2(pre0, pre1, v[j], v[j + 1]);
                        softplus100_fast2(pre2, pre3, v[j + 2], v[j + 3]);
                        psum2 = ffma2(pack2(v[j], v[j + 1]), pack2(ww.x, ww.y), psum2);
                        psum2 = ffma2(pack2(v[j + 2], v[j + 3]), pack2(ww.z, ww.w), psum2);
                    }
                    if (centre && p.spc) {
                        float4* dst = reinterpret_cast<float4*>(p.spc + (size_t)n * H + cc);
#pragma unroll
                        for (int j = 0; j < 4; ++j) dst[j] = make_float4(v[4 * j], v[4 * j + 1], v[4 * j + 2], v[4 * j + 3]);
                    }
                }
            }
            float psum, psum_b;
            unpack2(psum2, psum, psum_b);
            sdfs[((t & 1) * NCG + chh) * TM + row] = psum + psum_b;
            tc::fence_before_sync();
            tc::bar_sync(1, NWORK);                              // staging tile of t+1 complete, partial sums of t visible
            // ---- A operand of tile t+1 -> tensor memory (the accumulator and the A region are free: MMAs of t are done)
            if (t + 1 < my_tiles) {
                tc_stage_to_tmem(a_st, KT, a_tmem, lq, chh, lane);
                tc::fence_before_sync();
                tc::mbar_arrive(aready);
            }
            // ---- finalize the samples of tile t ---------------------------------------------------------------------
            if (tid < spt && !TF_DBG(p, 8)) {
                const int64_t ns = tile * spt + tid;
                const float* sp = &sdfs[(t & 1) * NCG * TM + tid * nq];
                if (ns < p.n) {
                    const float b1 = __ldg(p.b1);
                    if (nq == 1) {
                        float v = b1;
#pragma unroll
                        for (int g = 0; g < NCG; ++g) v += sp[g * TM];
                        p.sdf1[ns] = v;
                    } else {
                        float sd[NQ7];
#pragma unroll
                        for (int r = 0; r < NQ7; ++r) {
                            float v = b1;
#pragma unroll
                            for (int g = 0; g < NCG; ++g) v += sp[g * TM + r];
                            sd[r] = v; p.sdf7[ns * NQ7 + r] = v;
                        }
                        float g[3], h[3];              // (reciprocal FD steps: this block is fetched cold once per tile; keep it short)
#pragma unroll
                        for (int k = 0; k < 3; ++k) {
                            g[k] = (sd[1 + 2 * k] - sd[2 + 2 * k]) * inv2e[k];
                            h[k] = (sd[1 + 2 * k] + sd[2 + 2 * k] - 2.f * sd[0]) * inve2[k];
                        }
                        if (p.grad) { p.grad[ns * 3 + 0] = g[0]; p.grad[ns * 3 + 1] = g[1]; p.grad[ns * 3 + 2] = g[2]; }
                        if (p.hess) p.hess[ns] = (g[0] * h[0] + g[1] * h[1] + g[2] * h[2]) / (g[0] * g[0] + g[1] * g[1] + g[2] * g[2] + 1e-5f);
                    }
                }
            }
        }
    }
    tc::fence_before_sync();
    __syncthreads();
    if (warp == 0) tc::tmem_dealloc<512>(tmem_base);
}

size_t tc_fwd_smem(int KT, int H) {
    return (size_t)16 * (KT / 4) * site::A_LBO + (size_t)NST * 2 * H * KSL * 4 + (size_t)2 * H * 4 + (size_t)2 * NCG * TM * 4 + (2 * NST + 2) * 8 + 16;
}
}  // namespace

// the decoder shapes this kernel takes: the GEMM1 accumulator holds at most 256 hidden columns of TMEM, and the tile must fit
// shared memory.  sdf_stencil.cu dispatches on this predicate; the launcher below re-checks it.
bool tf_internal_stencil_fwd_tc_ok(int KT, int H) { return H <= 256 && tc_fwd_smem(KT, H) <= 227 * 1024; }

// workspace floats needed in front of spc: the pre-tiled W0
size_t tf_internal_tc_w0_floats(int KT, int H) { return (size_t)KT * H * 2; }

int tf_internal_stencil_fwd_tc(const tf_vm_field_t* f, const tf_sdf_mlp_t* m, const float* xyz, const float* level, int64_t n,
                               const float units[3], int nq, float* sdf7, float* grad, float* hess, float* sdf1, float* spc,
                               float* w0tc, cudaStream_t stream) {
    const int C = f->n_comp, K = 3 * C + 3, KT = (K + KSL - 1) / KSL * KSL, H = m->hidden;
    TcParams p = {};
    p.f = *f; p.xyz = xyz; p.level = level; p.n = n;
    p.W0tc = w0tc; p.b0 = m->b0; p.w1r0 = m->W1; p.b1 = m->b1;
    p.K = K; p.KT = KT; p.H = H; p.nq = nq;
    for (int k = 0; k < 3; ++k) p.units[k] = units ? units[k] : 0.f;
    p.sdf7 = sdf7; p.grad = grad; p.hess = hess; p.sdf1 = sdf1; p.spc = spc;
#ifdef TF_TC_DEBUG_SWITCHES
    { const char* e = getenv("TF_TC_DEBUG"); p.debug = e ? atoi(e) : 0; }
#endif
    if (!tf_internal_stencil_fwd_tc_ok(KT, H) || f->n_levels > site::MAXL) {
        tf_set_error("tensor-core stencil: tile does not fit shared / tensor memory (KT=%d, H=%d)", KT, H);
        return 1;
    }
    tc_prep_w0_kernel<<<64, 256, 0, stream>>>(m->W0, K, KT, H, w0tc);
    const size_t smem = tc_fwd_smem(KT, H);
    cudaFuncSetAttribute(sdf_stencil_fwd_tc_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    const int spt = nq == NQ7 ? site::SPT : TM;
    const int64_t ntiles = (n + spt - 1) / spt;
    const int grid = (int)(ntiles < tf_num_sms() ? ntiles : tf_num_sms());
    {
        TfKernelTimer timer("sdf_stencil_fwd_tc", stream);
        sdf_stencil_fwd_tc_kernel<<<grid, NTH, smem, stream>>>(p);
    }
    tf_count_launches(2);
    return 0;
}
