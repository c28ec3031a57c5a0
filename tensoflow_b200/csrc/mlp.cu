// Tall-skinny fused linear layers (M = 10^5..10^7 rows, K,N <= 256): the small MLPs of the
// hot path -- coupling-layer conditioners (network/flow.py:577-598), indirect-light and
// material predictors (network/other_field.py:20-121), shading heads (network/fields.py:395-417).
//   fwd      : Y = act(X W^T + b)                       (nn.Linear + activation, one pass)
//   bwd-data : dPre = dY * act'(Y);  dX = dPre W        (dPre is written back for bwd-weight)
//   bwd-wgt  : dW += dPre^T X (xty),  db += colsum(dPre)
// v1 arithmetic is fp32 FFMA (128x64 CTA tile, 8x4 register tile); see DESIGN.md.
#include "common.cuh"
#include "act.cuh"
#include "internal.cuh"

namespace {

constexpr int BM = 128, BN = 64, BK = 16, BMP = BM + 4, BNP = BN + 4;

// out[M][Nout] = epi( A[M][Kred] * B ),  B[kk][j] = TRANS_W ? W[kk*ldw + j] : W[j*ldw + kk]
// BWD: A element = dY * act'(Y) (and stored to dpre by the blockIdx.y == 0 column of CTAs)
template <bool TRANS_W, bool BWD>
__global__ void __launch_bounds__(256, 2) linear_kernel(const float* __restrict__ A, int lda, const float* __restrict__ Yact,
                                                        float* __restrict__ dpre, const float* __restrict__ W, int ldw,
                                                        const float* __restrict__ bias, int64_t M, int Kred, int Nout, int act,
                                                        float act_p, float* __restrict__ out, int ldo) {
    __shared__ __align__(16) float As[BK][BMP];
    __shared__ __align__(16) float Bs[BK][BNP];
    const int64_t r0 = (int64_t)blockIdx.x * BM;
    const int c0 = blockIdx.y * BN;
    const int ty = threadIdx.x / 16, tx = threadIdx.x % 16;
    float acc[8][4];
#pragma unroll
    for (int i = 0; i < 8; ++i) acc[i][0] = acc[i][1] = acc[i][2] = acc[i][3] = 0.f;
    for (int k0 = 0; k0 < Kred; k0 += BK) {
        // A tile -> As[k][row]
#pragma unroll
        for (int i = 0; i < BM / 16; ++i) {
            const int row = ty + 16 * i, k = tx;
            const int64_t r = r0 + row;
            float v = 0.f;
            if (r < M && k0 + k < Kred) {
                v = A[r * lda + k0 + k];
                if (BWD) {
                    v *= act_bwd(Yact[r * lda + k0 + k], act, act_p);
                    if (blockIdx.y == 0) dpre[r * lda + k0 + k] = v;
                }
            }
            As[k][row] = v;
        }
        // B tile -> Bs[k][col]
#pragma unroll
        for (int i = 0; i < (BK * BN) / 256; ++i) {
            const int idx = threadIdx.x + 256 * i;
            int k, j;
            if (TRANS_W) { k = idx / BN; j = idx % BN; } else { j = idx / BK; k = idx % BK; }
            float v = 0.f;
            if (k0 + k < Kred && c0 + j < Nout) v = TRANS_W ? __ldg(W + (size_t)(k0 + k) * ldw + c0 + j) : __ldg(W + (size_t)(c0 + j) * ldw + k0 + k);
            Bs[k][j] = v;
        }
        __syncthreads();
#pragma unroll
        for (int k = 0; k < BK; ++k) {
            const float4 a0 = *reinterpret_cast<const float4*>(&As[k][ty * 8]);
            const float4 a1 = *reinterpret_cast<const float4*>(&As[k][ty * 8 + 4]);
            const float4 b = *reinterpret_cast<const float4*>(&Bs[k][tx * 4]);
            const float a[8] = {a0.x, a0.y, a0.z, a0.w, a1.x, a1.y, a1.z, a1.w};
#pragma unroll
            for (int i = 0; i < 8; ++i) {
                acc[i][0] = fmaf(a[i], b.x, acc[i][0]); acc[i][1] = fmaf(a[i], b.y, acc[i][1]);
                acc[i][2] = fmaf(a[i], b.z, acc[i][2]); acc[i][3] = fmaf(a[i], b.w, acc[i][3]);
            }
        }
        __syncthreads();
    }
#pragma unroll
    for (int i = 0; i < 8; ++i) {
        const int64_t r = r0 + ty * 8 + i;
        if (r >= M) continue;
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const int c = c0 + tx * 4 + j;
            if (c >= Nout) continue;
            float v = acc[i][j];
            if (!BWD) {
                if (bias) v += __ldg(bias + c);
                v = act_fwd(v, act, act_p);
            }
            out[r * ldo + c] = v;
        }
    }
}

// ---- weight-gradient GEMM: out[m][n] (ld = ldo) += sum_r X[r][m] * Y[r][n] ---------------
constexpr int XT_M = 128, XT_N = 128, XT_R = 16;
__global__ void __launch_bounds__(256) xty_kernel(const float* __restrict__ X, int ldx, const float* __restrict__ Y, int ldy,
                                                  int64_t rows, int M, int N, float* __restrict__ out, int ldo,
                                                  int64_t rows_per_cta) {
    __shared__ __align__(16) float Xs[XT_R][XT_M];
    __shared__ __align__(16) float Ys[XT_R][XT_N];
    const int m0 = blockIdx.x * XT_M, n0 = blockIdx.y * XT_N;
    const int64_t r_begin = (int64_t)blockIdx.z * rows_per_cta;
    const int64_t r_end = r_begin + rows_per_cta < rows ? r_begin + rows_per_cta : rows;
    const int ty = threadIdx.x / 16, tx = threadIdx.x % 16;
    const bool vec = (ldx % 4 == 0) && (ldy % 4 == 0) && (((uintptr_t)X & 15) == 0) && (((uintptr_t)Y & 15) == 0);
    float acc[8][8];
#pragma unroll
    for (int a = 0; a < 8; ++a)
#pragma unroll
        for (int b = 0; b < 8; ++b) acc[a][b] = 0.f;
    for (int64_t r0 = r_begin; r0 < r_end; r0 += XT_R) {
        for (int i = threadIdx.x; i < XT_R * (XT_M / 4); i += 256) {
            const int rr = i / (XT_M / 4), m = (i % (XT_M / 4)) * 4;
            float4 v = f4_zero();
            if (r0 + rr < r_end) {
                const float* src = X + (size_t)(r0 + rr) * ldx + m0 + m;
                if (vec && m0 + m + 3 < ldx) { if (m0 + m < M) v = ldg4(src); }
                else {
                    if (m0 + m + 0 < M) v.x = __ldg(src + 0);
                    if (m0 + m + 1 < M) v.y = __ldg(src + 1);
                    if (m0 + m + 2 < M) v.z = __ldg(src + 2);
                    if (m0 + m + 3 < M) v.w = __ldg(src + 3);
                }
            }
            *reinterpret_cast<float4*>(&Xs[rr][m]) = v;
        }
        for (int i = threadIdx.x; i < XT_R * (XT_N / 4); i += 256) {
            const int rr = i / (XT_N / 4), nn = (i % (XT_N / 4)) * 4;
            float4 v = f4_zero();
            if (r0 + rr < r_end) {
                const float* src = Y + (size_t)(r0 + rr) * ldy + n0 + nn;
                if (vec && n0 + nn + 3 < ldy) { if (n0 + nn < N) v = ldg4(src); }
                else {
                    if (n0 + nn + 0 < N) v.x = __ldg(src + 0);
                    if (n0 + nn + 1 < N) v.y = __ldg(src + 1);
                    if (n0 + nn + 2 < N) v.z = __ldg(src + 2);
                    if (n0 + nn + 3 < N) v.w = __ldg(src + 3);
                }
            }
            *reinterpret_cast<float4*>(&Ys[rr][nn]) = v;
        }
        __syncthreads();
#pragma unroll
        for (int rr = 0; rr < XT_R; ++rr) {
            const float4 xa = *reinterpret_cast<const float4*>(&Xs[rr][ty * 4]);
            const float4 xb = *reinterpret_cast<const float4*>(&Xs[rr][64 + ty * 4]);
            const float4 ya = *reinterpret_cast<const float4*>(&Ys[rr][tx * 4]);
            const float4 yb = *reinterpret_cast<const float4*>(&Ys[rr][64 + tx * 4]);
            const float xv[8] = {xa.x, xa.y, xa.z, xa.w, xb.x, xb.y, xb.z, xb.w};
            const float yv[8] = {ya.x, ya.y, ya.z, ya.w, yb.x, yb.y, yb.z, yb.w};
#pragma unroll
            for (int a = 0; a < 8; ++a)
#pragma unroll
                for (int b = 0; b < 8; ++b) acc[a][b] = fmaf(xv[a], yv[b], acc[a][b]);
        }
        __syncthreads();
    }
#pragma unroll
    for (int a = 0; a < 8; ++a) {
        const int m = m0 + (a < 4 ? ty * 4 + a : 64 + ty * 4 + a - 4);
        if (m >= M) continue;
#pragma unroll
        for (int b = 0; b < 8; ++b) {
            const int nn = n0 + (b < 4 ? tx * 4 + b : 64 + tx * 4 + b - 4);
            if (nn < N && acc[a][b] != 0.f) atomicAdd(out + (size_t)m * ldo + nn, acc[a][b]);
        }
    }
}

// column sums: out[c] += sum_r X[r][c]
// (threads along the columns: coalesced rows; 8 independent loads in flight per thread, the kernel is HBM-bound)
__global__ void colsum_kernel(const float* __restrict__ X, int ldx, int64_t rows, int cols, float* __restrict__ out) {
    const int c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= cols) return;
    float acc[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
    const int64_t stride = gridDim.y;
    int64_t r = blockIdx.y;
    for (; r + 7 * stride < rows; r += 8 * stride) {
#pragma unroll
        for (int u = 0; u < 8; ++u) acc[u] += __ldg(X + (r + u * stride) * ldx + c);
    }
    for (; r < rows; r += stride) acc[0] += __ldg(X + r * ldx + c);
    const float t = ((acc[0] + acc[1]) + (acc[2] + acc[3])) + ((acc[4] + acc[5]) + (acc[6] + acc[7]));
    if (t != 0.f) atomicAdd(out + c, t);
}

// ---- narrow layers (K, N <= 64): the whole backward of one layer in one pass -----------------------------------
// The coupling-layer conditioners (44 -> 64 -> 64 -> 64 -> 21 on 10^5..10^6 rows) are far below any GEMM roofline; what
// they cost is HBM passes and launches.  One persistent kernel reads dY, Y, X once, forms dPre = dY * act'(Y) in shared
// memory, writes dX = dPre W, and keeps the CTA's share of dW = dPre^T X and db in registers until the end.
constexpr int SL_ROWS = 128, SL_MAX = 64, SL_DS = SL_MAX + 1, SL_XS = SL_MAX + 4;
__global__ void __launch_bounds__(256, 2) small_linear_bwd_kernel(const float* __restrict__ X, const float* __restrict__ W, const float* __restrict__ Y,
                                                                  const float* __restrict__ dY, int64_t M, int K, int N, int act, float act_p,
                                                                  float* __restrict__ dX, float* __restrict__ dW, float* __restrict__ db) {
    extern __shared__ __align__(16) float sl_smem[];
    float* Ds = sl_smem;                         // [128][65]  dPre tile
    float* Xs = Ds + SL_ROWS * SL_DS;            // [128][68]  X tile
    float* Ws = Xs + SL_ROWS * SL_XS;            // [64][68]   W
    const int tid = threadIdx.x;
    for (int i = tid; i < SL_MAX * SL_XS; i += 256) {
        const int n = i / SL_XS, k = i % SL_XS;
        Ws[i] = (n < N && k < K) ? W[(size_t)n * K + k] : 0.f;
    }
    // dW / db ownership: thread -> (n = tid / 4, 16 consecutive k)
    const int wn = tid >> 2, wk0 = (tid & 3) * 16;
    float accw[16];
#pragma unroll
    for (int j = 0; j < 16; ++j) accw[j] = 0.f;
    float accb = 0.f;
    // dX ownership: thread -> (row = tid / 2, 32 consecutive k)
    const int xr = tid >> 1, xk0 = (tid & 1) * 32;
    const int64_t ntiles = (M + SL_ROWS - 1) / SL_ROWS;
    for (int64_t t = blockIdx.x; t < ntiles; t += gridDim.x) {
        const int64_t r0 = t * SL_ROWS;
        const int rows = (int)(M - r0 < SL_ROWS ? M - r0 : SL_ROWS);
        __syncthreads();                         // previous tile fully consumed (also covers the W load)
        for (int i = tid; i < SL_ROWS * N; i += 256) {
            const int r = i / N, n = i % N;
            float v = 0.f;
            if (r < rows) { const size_t o = (size_t)(r0 + r) * N + n; v = __ldg(dY + o) * act_bwd(__ldg(Y + o), act, act_p); }
            Ds[r * SL_DS + n] = v;
        }
        for (int i = tid; i < SL_ROWS * K; i += 256) {
            const int r = i / K, k = i % K;
            Xs[r * SL_XS + k] = r < rows ? __ldg(X + (size_t)(r0 + r) * K + k) : 0.f;
        }
        __syncthreads();
        if (dX && xr < rows && xk0 < K) {
            float acc[32];
#pragma unroll
            for (int j = 0; j < 32; ++j) acc[j] = 0.f;
            for (int n = 0; n < N; ++n) {
                const float d = Ds[xr * SL_DS + n];
                const float4* w4 = reinterpret_cast<const float4*>(Ws + n * SL_XS + xk0);
#pragma unroll
                for (int j = 0; j < 8; ++j) {
                    const float4 w = w4[j];
                    acc[4 * j] = fmaf(d, w.x, acc[4 * j]); acc[4 * j + 1] = fmaf(d, w.y, acc[4 * j + 1]);
                    acc[4 * j + 2] = fmaf(d, w.z, acc[4 * j + 2]); acc[4 * j + 3] = fmaf(d, w.w, acc[4 * j + 3]);
                }
            }
            float* dst = dX + (size_t)(r0 + xr) * K + xk0;
#pragma unroll
            for (int j = 0; j < 32; ++j)
                if (xk0 + j < K) dst[j] = acc[j];
        }
        if (wn < N) {
            for (int r = 0; r < rows; ++r) {
                const float d = Ds[r * SL_DS + wn];
                const float4* x4 = reinterpret_cast<const float4*>(Xs + r * SL_XS + wk0);
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    const float4 x = x4[j];
                    accw[4 * j] = fmaf(d, x.x, accw[4 * j]); accw[4 * j + 1] = fmaf(d, x.y, accw[4 * j + 1]);
                    accw[4 * j + 2] = fmaf(d, x.z, accw[4 * j + 2]); accw[4 * j + 3] = fmaf(d, x.w, accw[4 * j + 3]);
                }
                accb += d;
            }
        }
    }
    if (wn < N) {
        if (dW) {
#pragma unroll
            for (int j = 0; j < 16; ++j)
                if (wk0 + j < K && accw[j] != 0.f) atomicAdd(dW + (size_t)wn * K + wk0 + j, accw[j]);
        }
        if (db && (tid & 3) == 0 && accb != 0.f) atomicAdd(db + wn, accb);
    }
}

}  // namespace

int tf_internal_xty(const float* X, int ldx, const float* Y, int ldy, int64_t rows, int M, int N, float* out, int ldo,
                    cudaStream_t stream) {
    if (rows == 0 || M == 0 || N == 0) return 0;
    dim3 grid((M + XT_M - 1) / XT_M, (N + XT_N - 1) / XT_N, 1);
    const int tiles = grid.x * grid.y;
    int64_t slices = (2 * (int64_t)tf_num_sms() + tiles - 1) / tiles;
    int64_t rpc = (rows + slices - 1) / slices;
    rpc = ((rpc + XT_R - 1) / XT_R) * XT_R;
    if (rpc < 256) rpc = 256;
    grid.z = (unsigned)((rows + rpc - 1) / rpc);
    xty_kernel<<<grid, 256, 0, stream>>>(X, ldx, Y, ldy, rows, M, N, out, ldo, rpc);
    tf_count_launches(1);
    return 0;
}

int tf_internal_colsum(const float* X, int ldx, int64_t rows, int cols, float* out, cudaStream_t stream) {
    if (rows == 0 || cols == 0) return 0;
    int gy = (int)(rows < 1184 ? rows : 1184);          // 8 x 148 row slices
    dim3 cg((cols + 127) / 128, gy);
    colsum_kernel<<<cg, 128, 0, stream>>>(X, ldx, rows, cols, out);
    tf_count_launches(1);
    return 0;
}

// ---- output heads: wide input, N <= 8 outputs (albedo / roughness / metallic / light / weight heads: K = 128 or 256, N = 1..5) --------
// The generic tiles waste their N side here and the X^T dPre product becomes a tall-skinny reduction at a fraction of the
// memory bandwidth.  One warp per row instead: a lane owns 4 consecutive k per 128-column chunk (one coalesced 512-byte row
// segment per load), the N weight rows live in registers.
//   forward   y[m][n] = act(sum_k x[m][k] W[n][k] + b[n])                       (N butterfly reductions per row)
//   backward  dpre = dY act'(Y);  dX[m][:] = sum_n dpre[n] W[n][:];  dW[n][:] += dpre[n] x[m][:];  db[n] += dpre[n]
//             in ONE pass over X (read once) and dX (written once); per-warp partial dW / db are reduced through shared
//             memory and added to the zero-initialised outputs with one atomic per element and CTA.
constexpr int HEAD_NMAX = 8, HEAD_KMAX = 256;
bool head_shape(int64_t M, int K, int N, const void* a, const void* b) {
    return M >= 4096 && N <= HEAD_NMAX && K % 4 == 0 && K > SL_MAX && K <= HEAD_KMAX && (((uintptr_t)a | (uintptr_t)b) & 15) == 0;
}

template <int CH>   // 128-column chunks per row
__global__ void __launch_bounds__(256) head_fwd_kernel(const float* __restrict__ X, const float* __restrict__ W, const float* __restrict__ b,
                                                       int64_t M, int K, int N, int act, float act_p, float* __restrict__ Y) {
    const int lane = threadIdx.x & 31, wpb = blockDim.x >> 5;
    float4 w[HEAD_NMAX][CH];
#pragma unroll
    for (int n = 0; n < HEAD_NMAX; ++n)
#pragma unroll
        for (int c = 0; c < CH; ++c) {
            const int k = c * 128 + lane * 4;
            w[n][c] = (n < N && k < K) ? *reinterpret_cast<const float4*>(W + (size_t)n * K + k) : f4_zero();
        }
    const float bias = (b && lane < N) ? b[lane] : 0.f;
    for (int64_t m = (int64_t)blockIdx.x * wpb + (threadIdx.x >> 5); m < M; m += (int64_t)gridDim.x * wpb) {
        float4 x[CH];
#pragma unroll
        for (int c = 0; c < CH; ++c) {
            const int k = c * 128 + lane * 4;
            x[c] = k < K ? ldg4(X + (size_t)m * K + k) : f4_zero();
        }
        float mine = 0.f;
#pragma unroll
        for (int n = 0; n < HEAD_NMAX; ++n) {
            if (n >= N) break;
            float a = 0.f;
#pragma unroll
            for (int c = 0; c < CH; ++c) a += (x[c].x * w[n][c].x + x[c].y * w[n][c].y) + (x[c].z * w[n][c].z + x[c].w * w[n][c].w);
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) a += __shfl_xor_sync(0xffffffffu, a, o);
            if (lane == n) mine = a;
        }
        if (lane < N) Y[(size_t)m * N + lane] = act_fwd(mine + bias, act, act_p);
    }
}

template <int CH>
__global__ void __launch_bounds__(256) head_bwd_kernel(const float* __restrict__ X, const float* __restrict__ W, const float* __restrict__ Y,
                                                       const float* __restrict__ dY, int64_t M, int K, int N, int act, float act_p,
                                                       float* __restrict__ dX, float* __restrict__ dW, float* __restrict__ db) {
    __shared__ float red[8][HEAD_NMAX][HEAD_KMAX / 2 + 4];     // two passes of 128 columns keep it at 33 KB
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, wpb = blockDim.x >> 5;
    float4 w[HEAD_NMAX][CH], acc[HEAD_NMAX][CH];
#pragma unroll
    for (int n = 0; n < HEAD_NMAX; ++n)
#pragma unroll
        for (int c = 0; c < CH; ++c) {
            const int k = c * 128 + lane * 4;
            w[n][c] = (n < N && k < K) ? *reinterpret_cast<const float4*>(W + (size_t)n * K + k) : f4_zero();
            acc[n][c] = f4_zero();
        }
    float accb = 0.f;                                           // lane n < N owns db[n]
    for (int64_t m = (int64_t)blockIdx.x * wpb + warp; m < M; m += (int64_t)gridDim.x * wpb) {
        float dp = 0.f;
        if (lane < N) { const size_t o = (size_t)m * N + lane; dp = __ldg(dY + o) * act_bwd(__ldg(Y + o), act, act_p); }
        accb += dp;
        float4 x[CH], dx[CH];
#pragma unroll
        for (int c = 0; c < CH; ++c) {
            const int k = c * 128 + lane * 4;
            x[c] = k < K ? ldg4(X + (size_t)m * K + k) : f4_zero();
            dx[c] = f4_zero();
        }
#pragma unroll
        for (int n = 0; n < HEAD_NMAX; ++n) {
            if (n >= N) break;
            const float d = __shfl_sync(0xffffffffu, dp, n);
#pragma unroll
            for (int c = 0; c < CH; ++c) { dx[c] = f4_fma(d, w[n][c], dx[c]); acc[n][c] = f4_fma(d, x[c], acc[n][c]); }
        }
        if (dX) {
#pragma unroll
            for (int c = 0; c < CH; ++c) {
                const int k = c * 128 + lane * 4;
                if (k < K) *reinterpret_cast<float4*>(dX + (size_t)m * K + k) = dx[c];
            }
        }
    }
    // CTA reduction of dW (one 128-column chunk at a time) and db
#pragma unroll
    for (int c = 0; c < CH; ++c) {
        __syncthreads();
#pragma unroll
        for (int n = 0; n < HEAD_NMAX; ++n) *reinterpret_cast<float4*>(&red[warp][n][lane * 4]) = acc[n][c];
        __syncthreads();
        for (int i = threadIdx.x; i < N * 128; i += blockDim.x) {
            const int n = i >> 7, kk = i & 127, k = c * 128 + kk;
            if (k >= K) continue;
            float sum = 0.f;
            for (int wv = 0; wv < wpb; ++wv) sum += red[wv][n][kk];
            if (dW && sum != 0.f) atomicAdd(dW + (size_t)n * K + k, sum);
        }
    }
    if (db) {
        __syncthreads();
        if (lane < N) red[warp][lane][0] = accb;
        __syncthreads();
        if (threadIdx.x < N) {
            float sum = 0.f;
            for (int wv = 0; wv < wpb; ++wv) sum += red[wv][threadIdx.x][0];
            if (sum != 0.f) atomicAdd(db + threadIdx.x, sum);
        }
    }
}

int head_grid(int64_t M) {
    const int64_t want = (M + 127) / 128, cap = (int64_t)tf_num_sms() * 4;     // >= 16 rows per warp: few, well-filled partial sums
    return (int)(want < cap ? want : cap);
}

// Tensor-core dispatch: at least 8192 rows and both widths >= 96.  Narrow layers (the coupling-layer conditioners,
// 44 -> 64 -> 64 -> 21, and 1..3-wide heads) stay on the FFMA kernels: the tensor core would run mostly padding
// there, and the spline parameters they produce are the one place where 3xTF32's ~22-bit products (vs 24) showed
// up in the gradient tolerances.
static const int64_t TC_MIN_ROWS = 8192;
static bool tc_shape(int64_t M, int K, int N) { return M >= TC_MIN_ROWS && K >= 96 && N >= 96; }
// Workspace bytes of the tcgen05 dense layer that contracts K into N outputs over M rows; 0 when that product runs on FFMA.
// The forward is that product at (K, N), the data gradient at (N, K).
static size_t tc_ws_bytes(int64_t M, int K, int N) {
    return tc_shape(M, K, N) && tf_internal_linear_tc_ok(K, N) ? tf_internal_linear_tc_ws_floats(K, N) * sizeof(float) : 0;
}
static bool ws_ok(const void* workspace, size_t ws_bytes, size_t need) {
    return workspace && ((uintptr_t)workspace & 15) == 0 && ws_bytes >= need;
}

extern "C" TF_API size_t tf_linear_workspace(int64_t M, int32_t K, int32_t N) {
    const size_t fwd = tc_ws_bytes(M, K, N), bwd = tc_ws_bytes(M, N, K);
    return fwd > bwd ? fwd : bwd;
}

extern "C" TF_API int tf_linear_fwd(const float* X, const float* W, const float* b, int64_t M, int32_t K, int32_t N, int32_t act,
                                    float act_param, float* Y, void* workspace, size_t ws_bytes, tf_stream_t stream) {
    if (M == 0) return 0;
    TF_REQUIRE(X && W && Y, "tf_linear_fwd: NULL pointer");
    TF_REQUIRE(K > 0 && N > 0 && act >= 0 && act <= 5, "tf_linear_fwd: bad K/N/act (%d,%d,%d)", K, N, act);
    if (head_shape(M, K, N, X, W)) {
        if (K <= 128) head_fwd_kernel<1><<<head_grid(M), 256, 0, (cudaStream_t)stream>>>(X, W, b, M, K, N, act, act_param, Y);
        else head_fwd_kernel<2><<<head_grid(M), 256, 0, (cudaStream_t)stream>>>(X, W, b, M, K, N, act, act_param, Y);
        tf_count_launches(1);
        TF_CHECK_LAUNCH("tf_linear_fwd (head)");
        return 0;
    }
    if (const size_t need = tc_ws_bytes(M, K, N)) {
        TF_REQUIRE(ws_ok(workspace, ws_bytes, need), "tf_linear_fwd: the tcgen05 path needs a 16-byte aligned workspace of %zu bytes "
                                                     "(tf_linear_workspace), got %zu at %p", need, ws_bytes, workspace);
        tf_internal_linear_tc(X, W, K, 0, b, M, K, N, act, act_param, Y, (float*)workspace, (cudaStream_t)stream);
        TF_CHECK_LAUNCH("tf_linear_fwd (tcgen05)");
        return 0;
    }
    dim3 grid((unsigned)((M + BM - 1) / BM), (N + BN - 1) / BN);
    linear_kernel<false, false><<<grid, 256, 0, (cudaStream_t)stream>>>(X, K, nullptr, nullptr, W, K, b, M, K, N, act, act_param, Y, N);
    tf_count_launches(1);
    TF_CHECK_LAUNCH("tf_linear_fwd");
    return 0;
}

extern "C" TF_API int tf_linear_bwd(const float* X, const float* W, const float* Y, const float* dY, float* dpre, int64_t M,
                                    int32_t K, int32_t N, int32_t act, float act_param, float* dX, float* dW, float* db,
                                    void* workspace, size_t ws_bytes, tf_stream_t stream_) {
    if (M == 0) return 0;
    TF_REQUIRE(X && W && Y && dY && dpre && dY != dpre, "tf_linear_bwd: NULL pointer (or dY aliases dpre)");
    TF_REQUIRE(K > 0 && N > 0 && act >= 0 && act <= 5, "tf_linear_bwd: bad K/N/act (%d,%d,%d)", K, N, act);
    cudaStream_t stream = (cudaStream_t)stream_;
    if (K <= SL_MAX && N <= SL_MAX && M >= 4096) {
        // narrow layer: fused one-pass backward (dPre stays in shared memory; the `dpre` buffer is left untouched)
        const size_t smem = sizeof(float) * ((size_t)SL_ROWS * SL_DS + (size_t)SL_ROWS * SL_XS + (size_t)SL_MAX * SL_XS);
        cudaFuncSetAttribute(small_linear_bwd_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        const int64_t ntiles = (M + SL_ROWS - 1) / SL_ROWS;
        const int grid = (int)(ntiles < 2 * tf_num_sms() ? ntiles : 2 * tf_num_sms());
        small_linear_bwd_kernel<<<grid, 256, smem, stream>>>(X, W, Y, dY, M, K, N, act, act_param, dX, dW, db);
        tf_count_launches(1);
        TF_CHECK_LAUNCH("tf_linear_bwd (narrow)");
        return 0;
    }
    if (head_shape(M, K, N, X, W) && (!dX || ((uintptr_t)dX & 15) == 0)) {
        // output head: one pass for dX, dW and db (the `dpre` buffer is left untouched)
        if (K <= 128) head_bwd_kernel<1><<<head_grid(M), 256, 0, stream>>>(X, W, Y, dY, M, K, N, act, act_param, dX, dW, db);
        else head_bwd_kernel<2><<<head_grid(M), 256, 0, stream>>>(X, W, Y, dY, M, K, N, act, act_param, dX, dW, db);
        tf_count_launches(1);
        TF_CHECK_LAUNCH("tf_linear_bwd (head)");
        return 0;
    }
    // dPre = dY * act'(Y) and dX = dPre W.  dX may be NULL (first layer): then a one-column
    // launch still materialises dPre.
    const size_t need = dX ? tc_ws_bytes(M, N, K) : 0;
    if (need) {
        TF_REQUIRE(ws_ok(workspace, ws_bytes, need), "tf_linear_bwd: the tcgen05 path needs a 16-byte aligned workspace of %zu bytes "
                                                     "(tf_linear_workspace), got %zu at %p", need, ws_bytes, workspace);
        tf_internal_linear_tc_bwd(dY, Y, dpre, W, M, K, N, act, act_param, dX, (float*)workspace, stream);
    } else if (dX) {
        dim3 grid((unsigned)((M + BM - 1) / BM), (K + BN - 1) / BN);
        linear_kernel<true, true><<<grid, 256, 0, stream>>>(dY, N, Y, dpre, W, K, nullptr, M, N, K, act, act_param, dX, K);
        tf_count_launches(1);
    } else {
        dim3 grid((unsigned)((M + BM - 1) / BM), 1);
        linear_kernel<true, true><<<grid, 256, 0, stream>>>(dY, N, Y, dpre, W, K, nullptr, M, N, 0, act, act_param, nullptr, K);
        tf_count_launches(1);
    }
    if (dW) {
        // dW[n][k] += sum_m dPre[m][n] X[m][k]
        if (tc_shape(M, K, N)) tf_internal_xty_auto(dpre, X, M, N, K, dW, stream);
        else tf_internal_xty(dpre, N, X, K, M, N, K, dW, K, stream);
    }
    if (db) tf_internal_colsum(dpre, N, M, N, db, stream);
    TF_CHECK_LAUNCH("tf_linear_bwd");
    return 0;
}
