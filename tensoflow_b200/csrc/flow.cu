// Piecewise-quadratic coupling transform of the TensoFlow sampler, one thread per
// (surface point, direction) pair.  Restates ElementWisePWQuadraticTransform
// (reference network/flow.py:314-525) for K = 10 bins: st = 11 vertex heights + 10 widths.
#include "common.cuh"
#include "flow_spline.cuh"
#include "internal.cuh"

namespace {

using namespace flowsp;

__global__ void __launch_bounds__(128) pwquad_fwd_kernel(const float* __restrict__ y, const float* __restrict__ st, int64_t M,
                                                         int inverse, float* __restrict__ x, float* __restrict__ logj) {
    const int64_t r = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (r >= M) return;
    float sr[NST];
#pragma unroll
    for (int i = 0; i < NST; ++i) sr[i] = st[r * NST + i];
    float xo, lj;
    if (!inverse) pwquad_eval_forward(sr, y[r], xo, lj);
    else pwquad_eval_inverse(sr, y[r], xo, lj);
    x[r] = xo;
    logj[r] = lj;
}

__global__ void __launch_bounds__(128) pwquad_bwd_kernel(const float* __restrict__ y, const float* __restrict__ st, int64_t M,
                                                         const float* __restrict__ g_x, const float* __restrict__ g_logj,
                                                         float* __restrict__ d_y, float* __restrict__ d_st) {
    const int64_t r = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (r >= M) return;
    float sr[NST], ds[NST];
#pragma unroll
    for (int i = 0; i < NST; ++i) sr[i] = st[r * NST + i];
    float dy;
    pwquad_adjoint(sr, y[r], g_x[r], g_logj[r], dy, ds);
    d_y[r] = dy;
#pragma unroll
    for (int i = 0; i < NST; ++i) d_st[r * NST + i] = ds[i];
}

// Fused coupling block (reference network/flow.py:549-641): input checks shared by both directions; the kernels are in flow_tc.cu
constexpr int FMAXF = 40;          // widest per-point feature the tensor-core kernels take (their shared-memory tiles)

struct FlowW { const float *W1, *b1, *W2, *b2, *W3, *b3, *W4, *b4; int F; };

int flow_check(const FlowW& w, int sn, int cond, int64_t M) {
    TF_REQUIRE(w.W1 && w.b1 && w.W2 && w.b2 && w.W3 && w.b3 && w.W4 && w.b4, "flow block: NULL weight pointer");
    TF_REQUIRE(w.F >= 1 && w.F <= FMAXF, "flow block: feature width must be in [1, %d] (got %d)", FMAXF, w.F);
    TF_REQUIRE(sn >= 16 && M % sn == 0, "flow block: directions per point must be >= 16 and divide the pair count (sn=%d)", sn);
    TF_REQUIRE(cond == 0 || cond == 1, "flow block: cond must be 0 or 1");
    return 0;
}

}  // namespace

extern "C" TF_API int tf_pwquad_fwd(const float* y, const float* st, int64_t M, int32_t inverse, float* x, float* logj,
                                    tf_stream_t stream) {
    if (M == 0) return 0;
    TF_REQUIRE(y && st && x && logj, "tf_pwquad_fwd: NULL pointer");
    pwquad_fwd_kernel<<<(unsigned)((M + 127) / 128), 128, 0, (cudaStream_t)stream>>>(y, st, M, inverse, x, logj);
    tf_count_launches(1);
    TF_CHECK_LAUNCH("tf_pwquad_fwd");
    return 0;
}

extern "C" TF_API int tf_pwquad_bwd(const float* y, const float* st, int64_t M, const float* g_x, const float* g_logj, float* d_y,
                                    float* d_st, tf_stream_t stream) {
    if (M == 0) return 0;
    TF_REQUIRE(y && st && g_x && g_logj && d_y && d_st, "tf_pwquad_bwd: NULL pointer");
    pwquad_bwd_kernel<<<(unsigned)((M + 127) / 128), 128, 0, (cudaStream_t)stream>>>(y, st, M, g_x, g_logj, d_y, d_st);
    tf_count_launches(1);
    TF_CHECK_LAUNCH("tf_pwquad_bwd");
    return 0;
}

extern "C" TF_API int tf_flow_block_fwd(const float* y_in, const float* logj_in, const float* feat, int32_t feat_dim, int32_t sn,
                                        const float* W1, const float* b1, const float* W2, const float* b2, const float* W3, const float* b3,
                                        const float* W4, const float* b4, float scale, float offset, int32_t cond, int32_t inverse, int64_t M,
                                        float* y_out, float* logj_out, float* save_h, float* save_st, tf_stream_t stream) {
    if (M == 0) return 0;
    if (int e = flow_check({W1, b1, W2, b2, W3, b3, W4, b4, feat_dim}, sn, cond, M)) return e;
    TF_REQUIRE(y_in && feat && y_out && logj_out, "tf_flow_block_fwd: NULL pointer");
    TF_REQUIRE((save_h == nullptr) == (save_st == nullptr), "tf_flow_block_fwd: pass both activation buffers or none");
    if (int e = tf_internal_flow_block_fwd_tc(y_in, logj_in, feat, feat_dim, sn, W1, b1, W2, b2, W3, b3, W4, b4, scale, offset, cond, inverse, M,
                                              y_out, logj_out, save_h, save_st, (cudaStream_t)stream)) return e;
    TF_CHECK_LAUNCH("tf_flow_block_fwd (tcgen05)");
    return 0;
}

extern "C" TF_API int tf_flow_block_bwd(const float* y_in, const float* feat, int32_t feat_dim, int32_t sn, const float* W1, const float* b1,
                                        const float* W2, const float* b2, const float* W3, const float* b3, const float* W4, const float* b4,
                                        float scale, float offset, int32_t cond, int64_t M, const float* saved_h, const float* saved_st,
                                        const float* g_y_out, const float* g_logj, float* g_y_in, float* d_feat, float* dW1, float* db1,
                                        float* dW2, float* db2, float* dW3, float* db3, float* dW4, float* db4, tf_stream_t stream) {
    if (M == 0) return 0;
    if (int e = flow_check({W1, b1, W2, b2, W3, b3, W4, b4, feat_dim}, sn, cond, M)) return e;
    TF_REQUIRE(y_in && feat && g_y_in && d_feat && dW1 && db1 && dW2 && db2 && dW3 && db3 && dW4 && db4, "tf_flow_block_bwd: NULL pointer");
    TF_REQUIRE(saved_h && saved_st, "tf_flow_block_bwd: saved_h / saved_st are NULL (keep the activations in tf_flow_block_fwd)");
    if (int e = tf_internal_flow_block_bwd_tc(y_in, feat, feat_dim, sn, W1, W2, W3, W4, scale, offset, cond, M, saved_h, saved_st, g_y_out, g_logj,
                                              g_y_in, d_feat, dW1, db1, dW2, db2, dW3, db3, dW4, db4, (cudaStream_t)stream)) return e;
    TF_CHECK_LAUNCH("tf_flow_block_bwd (tcgen05)");
    return 0;
}
