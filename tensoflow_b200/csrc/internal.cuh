// Entry points shared between the library's translation units (not part of the C ABI).  Every .cu that defines or calls
// one of them includes this header, so a definition that drifts from its declaration fails to compile or link.
#pragma once
#include <cuda_runtime.h>
#include <stddef.h>
#include <stdint.h>
#include "../../include/tensoflow_b200.h"

// ---- vm_field.cu ----
int tf_check_field(const tf_vm_field_t* f, bool need_mips);

// ---- mlp.cu: FFMA weight-gradient product and column sums ----
// out[m][n] (ld = ldo) += sum_r X[r][m] * Y[r][n]
int tf_internal_xty(const float* X, int ldx, const float* Y, int ldy, int64_t rows, int M, int N, float* out, int ldo, cudaStream_t stream);
// out[c] += sum_r X[r][c]
int tf_internal_colsum(const float* X, int ldx, int64_t rows, int cols, float* out, cudaStream_t stream);

// ---- linear_tc.cu: tensor-core dense layer ----
bool tf_internal_linear_tc_ok(int K, int N);
size_t tf_internal_linear_tc_ws_floats(int K, int N);
int tf_internal_linear_tc(const float* X, const float* W, int ldw, int trans, const float* bias, int64_t M, int K, int N, int act, float act_p,
                          float* Y, float* wtc, cudaStream_t stream);
int tf_internal_linear_tc_bwd(const float* dY, const float* Yact, float* dpre, const float* W, int64_t M, int K, int N, int act, float act_p,
                              float* dX, float* wtc, cudaStream_t stream);

// ---- xty_tc.cu: tensor-core weight-gradient product ----
bool tf_internal_xty_tc_ok(const float* X, const float* Y, int M, int N);
int tf_internal_xty_tc_tiled(const float* X, const float* Y, int64_t rows, int M, int N, float* out, int ldo, int n_valid, int x_tiled,
                             cudaStream_t stream);
// out[M][N] += X^T Y for packed X [rows][M], Y [rows][N]: tcgen05 when tf_internal_xty_tc_ok, FFMA otherwise
int tf_internal_xty_auto(const float* X, const float* Y, int64_t rows, int M, int N, float* out, cudaStream_t stream);

// ---- sdf_stencil_tc.cu: tensor-core stencil forward ----
bool tf_internal_stencil_fwd_tc_ok(int KT, int H);
size_t tf_internal_tc_w0_floats(int KT, int H);
int tf_internal_stencil_fwd_tc(const tf_vm_field_t* f, const tf_sdf_mlp_t* m, const float* xyz, const float* level, int64_t n,
                               const float units[3], int nq, float* sdf7, float* grad, float* hess, float* sdf1, float* spc,
                               float* w0tc, cudaStream_t stream);

// ---- sdf_stencil_bwd_tc.cu: tensor-core stencil backward ----
int tf_internal_bwd_tc_slot_floats(int KT, int H);
size_t tf_internal_bwd_tc_wtc_floats(int KT, int H);
size_t tf_internal_bwd_tc_smem(int KT, int H);
int tf_internal_bwd_tc_prep(const float* W0, int K, int KT, int H, float* wtc, cudaStream_t stream);
int tf_internal_bwd_tc_fold(const float* tmp, int H, int K, int KT, float* dW0, float* db0, cudaStream_t stream);
int tf_internal_bwd_tc_samples_per_tile();
size_t tf_internal_bwd_tc_scratch_floats(int KT);
int tf_internal_stencil_bwd_tc(const tf_vm_field_t* f, const tf_vm_mut_t* g, const tf_sdf_mlp_t* m, const float* wtc, const float* xyz,
                               const float* level, int64_t n, const float units[3], const float* sdf7, const float* g_sdf,
                               const float* g_grad, const float* g_hess, const float* dHc, float* dpre, float* arow,
                               float* da_scratch, float* dW1r0, float* db1, cudaStream_t stream);

// ---- flow_tc.cu: tensor-core coupling block ----
int tf_internal_flow_block_fwd_tc(const float* y_in, const float* logj_in, const float* feat, int feat_dim, int sn, const float* W1,
                                  const float* b1, const float* W2, const float* b2, const float* W3, const float* b3, const float* W4,
                                  const float* b4, float scale, float offset, int cond, int inverse, int64_t M, float* y_out, float* logj_out,
                                  float* save_h, float* save_st, cudaStream_t stream);
int tf_internal_flow_block_bwd_tc(const float* y_in, const float* feat, int feat_dim, int sn, const float* W1, const float* W2, const float* W3,
                                  const float* W4, float scale, float offset, int cond, int64_t M, const float* saved_h, const float* saved_st,
                                  const float* g_y_out, const float* g_logj, float* g_y_in, float* d_feat, float* dW1, float* db1, float* dW2,
                                  float* db2, float* dW3, float* db3, float* dW4, float* db4, cudaStream_t stream);

// ---- bvh.cu: BVH handles ----
struct tf_bvh;
// a handle with room for n_nodes nodes and n_tris triangles (perm included) on the current device; NULL after
// tf_set_error("<who>: ...") when an allocation fails
tf_bvh* tf_internal_bvh_alloc(int64_t n_nodes, int64_t n_tris, const char* who);
