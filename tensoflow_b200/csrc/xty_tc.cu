// Weight-gradient GEMM on the tensor cores: out[m][n] += sum_r X[r][m] * Y[r][n]   (X^T Y over a long row axis).
//
// X [rows][M] and Y [rows][N] are row-major fp32 in HBM (dPre and the gathered feature rows of the stencil
// backward; g_feat and the centre hidden activations of the appearance head).  The GEMM-K axis (rows) is the
// slow axis in memory, the tensor core wants it fastest (K-major operands; tf32 MN-major operands read back
// as zeros on this part), so the staging step transposes in registers: a thread loads the same 4-column group
// of 4 consecutive rows (coalesced float4 reads), which is a 4x4 block = four 16-byte K-major units, splits
// them into tf32 hi/lo (3xTF32, fp32-level accuracy) and stores them conflict-free (row-group stride padded
// by 16 bytes).  One persistent CTA per SM streams its row range through a 2-stage shared-memory pipeline
// (32 rows per stage) and accumulates [M x N] fp32 in TMEM; the kernel is HBM-bound (one pass over X and Y).
// Partial sums are added to `out` with atomics at the end.
#include <stdlib.h>
#include "common.cuh"
#include "tc_common.cuh"
#include "internal.cuh"

namespace {

// RS = rows (GEMM K) per stage: 32, or 16 when both operands are 256 wide (shared-memory budget)
constexpr int NTH = 512;
constexpr int NWORK = NTH - 32;     // staging warps 1..15; warp 0 only issues the MMAs (a thread that issues a dozen MMAs back to back
                                    // is blocked while the tensor queue drains: it must not be one the staging warps wait for)
constexpr int TPT = 2;              // staging tasks per worker and stage (X and Y tasks share one list: <= 960 per stage)
constexpr uint32_t LBO = 144;       // K-chunk (4 rows = 16 bytes per column) stride of a staged operand: 128 + 16 so that stores whose lanes
                                    // walk the K chunks (tiled operands) spread over the banks like those whose lanes walk the columns
template <int RS> struct Stage { static constexpr uint32_t SBO = (RS / 4) * LBO + 16; };   // 8-column-group stride (padded: bank spread)

__device__ __forceinline__ float4 hi4(float4 v) { return make_float4(tc::tf32_rn(v.x), tc::tf32_rn(v.y), tc::tf32_rn(v.z), tc::tf32_rn(v.w)); }
__device__ __forceinline__ float4 lo4(float4 v, float4 h) {
    return make_float4(tc::tf32_rn(v.x - h.x), tc::tf32_rn(v.y - h.y), tc::tf32_rn(v.z - h.z), tc::tf32_rn(v.w - h.w));
}

// One staging task = the 4x4 block (rows 4c..4c+3, columns 4g..4g+3) of X [rows][M] or Y [rows][N].  The global loads
// of stage it+2 are issued into registers before stage it+1 is converted and stored, so HBM latency overlaps the
// staging and MMA work.
struct Prefetch { float4 v[TPT][4]; };
// per-worker staging plan (fixed for the whole kernel: only the row base advances): task list = Y tasks then X tasks
struct StagePlan { int src_off[TPT]; int row[TPT]; int ld[TPT]; uint32_t smem_off[TPT]; bool on[TPT], is_x[TPT], tiled[TPT]; };

// y_tiled: the Y operand is stored per 128-row tile as [tile][N][128] (row fastest): 4 consecutive rows of one column are one
// 16-byte K-major unit already, so its tasks need no register transpose (the stencil backward writes dPre this way: one
// 128-byte store wavefront per warp and column instead of 8 for row-major 16-byte pieces)
template <int RS>
__device__ __forceinline__ StagePlan make_stage_plan(int M, int N, int wtid, bool x_tiled, bool y_tiled) {
    constexpr uint32_t SBO = Stage<RS>::SBO;
    StagePlan p;
    const int ty = (RS / 4) * (N / 4), tx = (RS / 4) * (M / 4);
#pragma unroll
    for (int k = 0; k < TPT; ++k) {
        int it = wtid + k * NWORK;
        p.is_x[k] = it >= ty;
        if (p.is_x[k]) it -= ty;
        const int W = p.is_x[k] ? M : N, G = W / 4;
        p.on[k] = wtid >= 0 && it < (p.is_x[k] ? tx : ty);
        p.tiled[k] = p.is_x[k] ? x_tiled : y_tiled;
        // row-major operand: lanes walk the column groups (coalesced float4 reads along a row); tiled operand: lanes walk the
        // K chunks (8 chunks x 16 bytes = the 128 contiguous bytes of one column in the tile)
        const int g = p.tiled[k] ? it / (RS / 4) : it % G, c = p.tiled[k] ? it % (RS / 4) : it / G;
        p.row[k] = c * 4;
        p.ld[k] = p.tiled[k] ? 128 : W;                   // stride between the task's four 16-byte loads
        p.src_off[k] = p.tiled[k] ? g * 4 * 128 + c * 4 : c * 4 * W + g * 4;
        const int w = g * 4;                              // first of the task's 4 columns (w & 7 is 0 or 4)
        p.smem_off[k] = (uint32_t)(w >> 3) * SBO + c * LBO + (w & 7) * 16;
    }
    return p;
}
__device__ __forceinline__ void stage_load(const float* __restrict__ X, const float* __restrict__ Y, int64_t r0, int64_t r_end, int M, int N,
                                           const StagePlan& sp, Prefetch& pf) {
#pragma unroll
    for (int k = 0; k < TPT; ++k) {
        if (sp.tiled[k]) {
            // tile = r0 / 128 (stages never straddle tiles: 128 % RS == 0 and the CTA's row range starts at a tile); whole tiles only
            const float* base = (sp.is_x[k] ? X + (size_t)(r0 >> 7) * 128 * M : Y + (size_t)(r0 >> 7) * 128 * N) + (r0 & 127) + sp.src_off[k];
#pragma unroll
            for (int i = 0; i < 4; ++i) pf.v[k][i] = (sp.on[k] && r0 + sp.row[k] < r_end) ? ldg4(base + i * 128) : make_float4(0.f, 0.f, 0.f, 0.f);
        } else {
            const float* base = (sp.is_x[k] ? X : Y) + (size_t)r0 * sp.ld[k] + sp.src_off[k];
#pragma unroll
            for (int i = 0; i < 4; ++i)
                pf.v[k][i] = (sp.on[k] && r0 + sp.row[k] + i < r_end) ? ldg4(base + i * sp.ld[k]) : make_float4(0.f, 0.f, 0.f, 0.f);
        }
    }
}
// transpose the 4x4 blocks in registers (four 16-byte K-major units each), split into tf32 hi / lo, store
__device__ __forceinline__ void stage_store(const Prefetch& pf, const StagePlan& sp, uint8_t* xs_hi, uint8_t* xs_lo, uint8_t* ys_hi, uint8_t* ys_lo) {
#pragma unroll
    for (int k = 0; k < TPT; ++k) {
        if (!sp.on[k]) continue;
        uint8_t* hi = sp.is_x[k] ? xs_hi : ys_hi;
        uint8_t* lo = sp.is_x[k] ? xs_lo : ys_lo;
        const float4* v = pf.v[k];
        float4 t[4];
        if (sp.tiled[k]) {                                    // already K-major units (4 rows of one column each)
            t[0] = v[0]; t[1] = v[1]; t[2] = v[2]; t[3] = v[3];
        } else {
            t[0] = make_float4(v[0].x, v[1].x, v[2].x, v[3].x); t[1] = make_float4(v[0].y, v[1].y, v[2].y, v[3].y);
            t[2] = make_float4(v[0].z, v[1].z, v[2].z, v[3].z); t[3] = make_float4(v[0].w, v[1].w, v[2].w, v[3].w);
        }
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const uint32_t off = sp.smem_off[k] + j * 16;     // columns 4g..4g+3 stay inside one 8-row group
            const float4 h = hi4(t[j]);
            *reinterpret_cast<float4*>(hi + off) = h;
            *reinterpret_cast<float4*>(lo + off) = lo4(t[j], h);
        }
    }
}

// D[i][j] = sum_r X[r][i] Y[r][j]: X (width M, a multiple of 4; padded to MP = 128 or 256 MMA rows) is the MMA M side,
// Y (width N, a multiple of 16) the MMA N side.  An SS-mode tf32 MMA costs ~130 cycles whatever its N (the 4 KB A-operand
// read), so the host puts the wider operand on the N side; `tr` then writes the result transposed.
template <int RS>
__global__ void __launch_bounds__(NTH, 1) xty_tc_kernel(const float* __restrict__ X, const float* __restrict__ Y, int64_t rows, int M, int MP, int N,
                                                        float* __restrict__ out, int ldo, int x_valid, int y_valid, int tr, int64_t rows_per_cta,
                                                        int x_tiled, int y_tiled) {
    extern __shared__ __align__(1024) uint8_t smem[];
    constexpr uint32_t SBO = Stage<RS>::SBO;
    const uint32_t x_part = (uint32_t)(MP / 8) * SBO, y_part = (uint32_t)(N / 8) * SBO;
    const uint32_t stage_bytes = 2 * (x_part + y_part);
    uint64_t* bars = reinterpret_cast<uint64_t*>(smem + 2 * stage_bytes);
    uint64_t* empty = bars;          // [2] stage consumed by its MMAs
    uint64_t* ready = bars + 2;      // [2] stage written by the staging warps
    uint64_t* done = bars + 4;
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 5);
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int MT = MP / 128;
    const int ncol_tile = N <= 128 ? 128 : 256;      // TMEM column stride between the M tiles

    if (warp == 0) tc::tmem_alloc<512>(tmem_slot);
    if (tid == 0) {
        tc::mbar_init(&empty[0], 1); tc::mbar_init(&empty[1], 1); tc::mbar_init(&ready[0], NWORK); tc::mbar_init(&ready[1], NWORK);
        tc::mbar_init(done, 1);
        tc::mbar_fence_init();
    }
    // the padding rows of the M side (MP > M) are never written by a staging task: clear both stages once
    for (uint32_t i = tid * 16; i < 2 * stage_bytes; i += NTH * 16) *reinterpret_cast<float4*>(smem + i) = make_float4(0.f, 0.f, 0.f, 0.f);
    tc::fence_async_smem();
    tc::fence_before_sync();
    __syncthreads();
    tc::fence_after_sync();
    const uint32_t tmem_base = *tmem_slot;
    const uint32_t idesc = tc::make_idesc(2, 2, 128, N);

    const int64_t r_begin = (int64_t)blockIdx.x * rows_per_cta;
    const int64_t r_end = r_begin + rows_per_cta < rows ? r_begin + rows_per_cta : rows;
    const int64_t n_stages = r_begin < r_end ? (r_end - r_begin + RS - 1) / RS : 0;

    if (warp == 0) {
        // ---- MMA warp: one lane issues the MMAs of a stage as soon as the staging warps have written it ------------------
        if (lane == 0) {
            for (int64_t it = 0; it < n_stages; ++it) {
                const int buf = (int)(it & 1);
                uint8_t* xs_hi = smem + (size_t)buf * stage_bytes;
                uint8_t* xs_lo = xs_hi + x_part;
                uint8_t* ys_hi = xs_lo + x_part;
                uint8_t* ys_lo = ys_hi + y_part;
                tc::mbar_wait(&ready[buf], (uint32_t)((it >> 1) & 1));
                tc::fence_after_sync();
                // one descriptor per operand part and stage; the MMAs only advance its start address
                const uint64_t xdh = tc::make_smem_desc(tc::smem_u32(xs_hi), LBO, SBO), xdl = tc::make_smem_desc(tc::smem_u32(xs_lo), LBO, SBO);
                const uint64_t ydh = tc::make_smem_desc(tc::smem_u32(ys_hi), LBO, SBO), ydl = tc::make_smem_desc(tc::smem_u32(ys_lo), LBO, SBO);
#pragma unroll
                for (int ks = 0; ks < RS / 8; ++ks) {
                    const uint64_t bdh = tc::desc_add(ydh, ks * 2 * LBO), bdl = tc::desc_add(ydl, ks * 2 * LBO);
#pragma unroll
                    for (int mt = 0; mt < 2; ++mt) {
                        if (mt >= MT) break;
                        const uint32_t d = tmem_base + (uint32_t)mt * ncol_tile;
                        const uint64_t adh = tc::desc_add(xdh, mt * 16 * SBO + ks * 2 * LBO), adl = tc::desc_add(xdl, mt * 16 * SBO + ks * 2 * LBO);
                        tc::mma_tf32_ss(d, adh, bdh, idesc, (it | ks) != 0);
                        tc::mma_tf32_ss(d, adh, bdl, idesc, 1);
                        tc::mma_tf32_ss(d, adl, bdh, idesc, 1);
                    }
                }
                tc::mma_commit(&empty[buf]);
                if (it == n_stages - 1) tc::mma_commit(done);
            }
        }
    } else {
        // ---- staging warps: register prefetch two stages ahead (sets p0 / p1 alternate) ------------------------------------
        Prefetch p0, p1;
        const StagePlan sp = make_stage_plan<RS>(M, N, tid - 32, x_tiled != 0, y_tiled != 0);
        if (n_stages > 0) stage_load(X, Y, r_begin, r_end, M, N, sp, p0);
        if (n_stages > 1) stage_load(X, Y, r_begin + RS, r_end, M, N, sp, p1);
        auto do_stage = [&](int64_t it, Prefetch& pf) {
            const int buf = (int)(it & 1);
            uint8_t* xs_hi = smem + (size_t)buf * stage_bytes;
            uint8_t* xs_lo = xs_hi + x_part;
            uint8_t* ys_hi = xs_lo + x_part;
            uint8_t* ys_lo = ys_hi + y_part;
            if (it >= 2) tc::mbar_wait(&empty[buf], (uint32_t)(((it >> 1) - 1) & 1));
            stage_store(pf, sp, xs_hi, xs_lo, ys_hi, ys_lo);
            if (it + 2 < n_stages) stage_load(X, Y, r_begin + (it + 2) * RS, r_end, M, N, sp, pf);
            tc::fence_async_smem();
            tc::mbar_arrive(&ready[buf]);
        };
        for (int64_t it = 0; it < n_stages; it += 2) {
            do_stage(it, p0);
            if (it + 1 < n_stages) do_stage(it + 1, p1);
        }
    }
    __syncwarp();
    if (n_stages > 0) {
        tc::mbar_wait(done, 0);
        tc::fence_after_sync();
        const int lq = warp & 3, half = warp >> 2;
        for (int mt = 0; mt < MT; ++mt) {
            const int m = mt * 128 + lq * 32 + lane;
            for (int c0 = half * 16; c0 < N; c0 += 16 * (NTH / 128)) {
                float v[16];
                tc::tmem_ld16(tmem_base + (uint32_t)mt * ncol_tile + ((uint32_t)(lq * 32) << 16) + c0, v);
#pragma unroll
                for (int j = 0; j < 16; ++j)
                    if (m < x_valid && c0 + j < y_valid && v[j] != 0.f)
                        atomicAdd(tr ? out + (size_t)(c0 + j) * ldo + m : out + (size_t)m * ldo + c0 + j, v[j]);
            }
        }
    }
    tc::fence_before_sync();
    __syncthreads();
    if (warp == 0) tc::tmem_dealloc<512>(tmem_base);
}

size_t xty_tc_smem(int MP, int N, int rs) { return (size_t)2 * 2 * ((MP / 8) + (N / 8)) * ((rs / 4) * LBO + 16) + 64; }
int xty_tc_stage_rows(int MP, int N) { return xty_tc_smem(MP, N, 32) <= 227 * 1024 ? 32 : 16; }

}  // namespace

// true when the shapes suit the tensor-core kernel (otherwise callers use the SIMT X^T Y kernel)
bool tf_internal_xty_tc_ok(const float* X, const float* Y, int M, int N) {
    if (M % 16 != 0 || N % 16 != 0 || M < 16 || N < 16 || M > 256 || N > 256) return false;
    if (((uintptr_t)X & 15) || ((uintptr_t)Y & 15)) return false;
    const int mw = M > N ? N : M, nw = M > N ? M : N;
    return xty_tc_smem((mw + 127) / 128 * 128, nw, 16) <= 227 * 1024;
}

// X [rows][M] (ld = M), Y [rows][N] (ld = N); out[m][n] (ld = ldo) += X^T Y for n < n_valid
// x_tiled: X is stored per 128-row tile as [tile][M][128] (rows must then be a multiple of 128)
int tf_internal_xty_tc_tiled(const float* X, const float* Y, int64_t rows, int M, int N, float* out, int ldo, int n_valid, int x_tiled,
                             cudaStream_t stream) {
    if (rows == 0) return 0;
    // MMA N side = the wider operand; the M side is padded to whole 128-row MMAs (its extra rows are never read back)
    const bool tr = M > N;
    const float* xs = tr ? Y : X;
    const float* ys = tr ? X : Y;
    const int mw = tr ? N : M, nw = tr ? M : N;
    const int mp = (mw + 127) / 128 * 128;
    const int x_valid = tr ? n_valid : M, y_valid = tr ? M : n_valid;
    const int RS = xty_tc_stage_rows(mp, nw);
    const size_t smem = xty_tc_smem(mp, nw, RS);
    int64_t grid = (rows + 4 * RS - 1) / (4 * RS);
    if (grid > tf_num_sms()) grid = tf_num_sms();
    int64_t rpc = (rows + grid - 1) / grid;
    const int64_t rgran = x_tiled ? 128 : RS;          // tiled operand: every CTA starts at a tile
    rpc = (rpc + rgran - 1) / rgran * rgran;
    grid = (rows + rpc - 1) / rpc;
    if (x_tiled && rows % 128 != 0) { tf_set_error("xty_tc: a tiled operand needs rows to be a multiple of 128"); return 1; }
    const int kx_tiled = (x_tiled && !tr) ? 1 : 0, ky_tiled = (x_tiled && tr) ? 1 : 0;      // which kernel-side operand the caller's X became
    {
        TfKernelTimer timer("xty_tc", stream);
        if (RS == 32) {
            cudaFuncSetAttribute(xty_tc_kernel<32>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
            xty_tc_kernel<32><<<(int)grid, NTH, smem, stream>>>(xs, ys, rows, mw, mp, nw, out, ldo, x_valid, y_valid, tr ? 1 : 0, rpc, kx_tiled, ky_tiled);
        } else {
            cudaFuncSetAttribute(xty_tc_kernel<16>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
            xty_tc_kernel<16><<<(int)grid, NTH, smem, stream>>>(xs, ys, rows, mw, mp, nw, out, ldo, x_valid, y_valid, tr ? 1 : 0, rpc, kx_tiled, ky_tiled);
        }
    }
    tf_count_launches(1);
    return 0;
}

int tf_internal_xty_auto(const float* X, const float* Y, int64_t rows, int M, int N, float* out, cudaStream_t stream) {
    return tf_internal_xty_tc_ok(X, Y, M, N) ? tf_internal_xty_tc_tiled(X, Y, rows, M, N, out, N, N, 0, stream)
                                             : tf_internal_xty(X, M, Y, N, rows, M, N, out, N, stream);
}

extern "C" TF_API int tf_xty_accumulate(const float* X, const float* Y, int64_t rows, int32_t M, int32_t N, float* out,
                                        tf_stream_t stream) {
    if (rows == 0) return 0;
    TF_REQUIRE(X && Y && out && M > 0 && N > 0, "tf_xty_accumulate: NULL pointer or bad shape (%d,%d)", M, N);
    if (int e = tf_internal_xty_auto(X, Y, rows, M, N, out, (cudaStream_t)stream)) return e;
    TF_CHECK_LAUNCH("tf_xty_accumulate");
    return 0;
}
