/*
 * tensoflow_b200 -- C ABI of the B200-native TensoFlow hot path.
 *
 * The reference (fudan-zvg/tensoflow) has no plugin registry: its operator
 * boundary is a set of third-party native ops called from PyTorch modules.
 * Each entry point below names the reference call site(s) it replaces
 * (paths relative to the reference tree).  Conventions (SURVEY.md 8b):
 *   - every pointer is a DEVICE pointer to contiguous fp32 (int32 where said),
 *     owned by the caller; the library never allocates, frees or retains them
 *     (exception: the BVH handle, created/destroyed explicitly);
 *   - gradient outputs are ACCUMULATED into (caller zero-initialises);
 *   - all work is enqueued on `stream` (a cudaStream_t); no implicit syncs;
 *   - return 0 on success, non-zero otherwise, message via tf_last_error();
 *   - re-entrant: backward entry points are called from autograd worker threads.
 *   - there is no CPU fallback.
 */
#ifndef TENSOFLOW_B200_H
#define TENSOFLOW_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define TF_ABI_VERSION 1

#if defined(__GNUC__)
#define TF_API __attribute__((visibility("default")))
#else
#define TF_API
#endif

typedef void* tf_stream_t; /* cudaStream_t */

/* A VM-decomposed (3 planes x 3 lines) tensorial field.
 * Reference storage: nn.Parameter [1,C,H,W] / [1,C,G,1] (network/fields.py:101-111).
 * Here the same logical tensors are held channels-last, i.e. plane i is
 * [H][W][C] and line i is [G][C] in memory, so one texel's C channels are
 * contiguous (16-byte vector loads / reductions).  Mip levels 1..L-1 (2x2 box
 * filter, what nvdiffrast builds internally) live in one buffer per texture,
 * level after level.  plane i is addressed with u = x[m0] along W and
 * v = x[m1] along H, (m0,m1) = (0,1),(0,2),(1,2); line i with x[2-i] along G
 * (network/fields.py:28-29,268-288). */
typedef struct {
    const float* plane[3];
    const float* plane_mip[3]; /* may be NULL when n_levels == 1 */
    const float* line[3];
    const float* line_mip[3];
    int32_t plane_h[3], plane_w[3], line_g[3];
    int32_t n_comp;   /* C, multiple of 4 */
    int32_t n_levels; /* L >= 1 */
    float aabb_min[3], aabb_max[3];
} tf_vm_field_t;

/* Mutable twin (mip outputs / gradient accumulators), same layouts. */
typedef struct {
    float* plane[3];
    float* plane_mip[3];
    float* line[3];
    float* line_mip[3];
} tf_vm_mut_t;

/* Decoder MLP of TensoSDF: Linear(3C+3,H) -> Softplus(beta=100) -> Linear(H,1+A)
 * (network/fields.py:78-91).  PyTorch layouts: W0 [H][3C+3], W1 [1+A][H]. */
typedef struct {
    const float* W0; const float* b0; const float* W1; const float* b1;
    int32_t hidden;  /* H, multiple of 32 */
    int32_t app_dim; /* A, multiple of 4, <= 128 */
} tf_sdf_mlp_t;

typedef struct { float* W0; float* b0; float* W1; float* b1; } tf_sdf_mlp_grad_t;

TF_API int tf_abi_version(void);
TF_API const char* tf_last_error(void);
/* number of kernels this library has launched in this process (bench.py reports it) */
TF_API long long tf_launch_count(void);

/* ---- VM field ------------------------------------------------------------ */

/* Rebuild mip levels 1..L-1 from level 0 (nvdiffrast does this inside every
 * dr.texture call: network/fields.py:276-288). */
TF_API int tf_vm_build_mips(const tf_vm_field_t* f, const tf_vm_mut_t* out, tf_stream_t stream);

/* Fold gradients accumulated on levels 1..L-1 into level 0 (x1/4 per level,
 * x1/2 for lines) -- the mip part of dr.texture's backward. */
TF_API int tf_vm_fold_mip_grads(const tf_vm_field_t* f, const tf_vm_mut_t* g, tf_stream_t stream);

/* feat[n, 3C] = concat_i plane_i(x) * line_i(x): the 6 dr.texture calls + product of
 * network/fields.py:272-293, :786-806 and network/flow.py:719-740.
 * level may be NULL (level 0 only). */
TF_API int tf_vm_feature_fwd(const tf_vm_field_t* f, const float* xyz, const float* level, int64_t n,
                      float* feat, tf_stream_t stream);
TF_API int tf_vm_feature_bwd(const tf_vm_field_t* f, const float* xyz, const float* level, int64_t n,
                      const float* d_feat, const tf_vm_mut_t* g, tf_stream_t stream);

/* ---- fused TensoSDF stencil ------------------------------------------------
 * One call = TensoSDF.forward (network/fields.py:262-299) at the sample plus the
 * six finite-difference taps of TensoSDF.gradient (network/fields.py:227-260):
 *   sdf7[n,7] : SDF at (centre, +x, -x, +y, -y, +z, -z), taps at +-units[k]
 *   feat[n,A] : appearance features (decoder outputs 1..A) at the centre
 *   grad[n,3] : central differences          hess[n] : (g.h)/(|g|^2+1e-5)
 * feat / grad / hess may be NULL.  level may be NULL. */
TF_API size_t tf_sdf_stencil_fwd_workspace(const tf_vm_field_t* f, const tf_sdf_mlp_t* m, int64_t n,
                                           int32_t with_feat);
TF_API int tf_sdf_stencil_fwd(const tf_vm_field_t* f, const tf_sdf_mlp_t* m, const float* xyz,
                       const float* level, int64_t n, const float units[3], float* sdf7,
                       float* feat, float* grad, float* hess, void* workspace, size_t ws_bytes,
                       tf_stream_t stream);

/* SDF only (TensoSDF.sdf, network/fields.py:148) -- the hierarchical sampler's query. */
TF_API int tf_sdf_only_fwd(const tf_vm_field_t* f, const tf_sdf_mlp_t* m, const float* xyz,
                    const float* level, int64_t n, float* sdf, void* workspace, size_t ws_bytes,
                    tf_stream_t stream);

/* One query per point WITH the appearance features: sdf[n], feat[n, app_dim] = TensoSDF.forward (network/fields.py:262-299)
 * without the six finite-difference taps (forward only: inference, probes).  Workspace as tf_sdf_stencil_fwd_workspace(.., 1).
 * Needs the tensor-core path (hidden % 32 == 0, hidden <= 256); otherwise an error is returned and tf_sdf_stencil_fwd applies. */
TF_API int tf_sdf_point_fwd(const tf_vm_field_t* f, const tf_sdf_mlp_t* m, const float* xyz, const float* level,
                            int64_t n, float* sdf, float* feat, void* workspace, size_t ws_bytes, tf_stream_t stream);

/* Backward of tf_sdf_stencil_fwd.  g_sdf[n], g_feat[n,A], g_grad[n,3], g_hess[n] are the
 * upstream gradients (each may be NULL = zero); sdf7 is the forward output.
 * Any workspace size >= tf_sdf_stencil_bwd_workspace(.., 1) works; larger is faster
 * (the call processes the n samples in slices that fit). */
TF_API size_t tf_sdf_stencil_bwd_workspace(const tf_vm_field_t* f, const tf_sdf_mlp_t* m, int64_t n_slice);
TF_API int tf_sdf_stencil_bwd(const tf_vm_field_t* f, const tf_sdf_mlp_t* m, const float* xyz,
                       const float* level, int64_t n, const float units[3], const float* sdf7,
                       const float* g_sdf, const float* g_feat, const float* g_grad,
                       const float* g_hess, const tf_vm_mut_t* g_field,
                       const tf_sdf_mlp_grad_t* g_mlp, void* workspace, size_t ws_bytes,
                       tf_stream_t stream);

/* The same with the centre hidden activations KEPT from the forward call: hidden_centre[n, hidden] = the block at byte offset
 * tf_sdf_stencil_fwd_hidden_offset(f, m) of the workspace that was passed to tf_sdf_stencil_fwd (with feat != NULL), which the
 * caller then has to keep alive until the backward call.  The backward kernel does not recompute / store them (they feed the
 * weight gradient of the appearance head).  hidden_centre == NULL behaves like tf_sdf_stencil_bwd; the offset is (size_t)-1
 * when the forward path for this decoder shape does not produce the block. */
TF_API size_t tf_sdf_stencil_fwd_hidden_offset(const tf_vm_field_t* f, const tf_sdf_mlp_t* m);
TF_API int tf_sdf_stencil_bwd_kept(const tf_vm_field_t* f, const tf_sdf_mlp_t* m, const float* xyz,
                       const float* level, int64_t n, const float units[3], const float* sdf7, const float* hidden_centre,
                       const float* g_sdf, const float* g_feat, const float* g_grad,
                       const float* g_hess, const tf_vm_mut_t* g_field,
                       const tf_sdf_mlp_grad_t* g_mlp, void* workspace, size_t ws_bytes,
                       tf_stream_t stream);

/* ---- NeuS alpha + compositing ------------------------------------------------
 * Replaces ShapeRenderer.compute_sdf_alpha's tail (network/shapeRenderer.py:1004-1024),
 * nerfacc.render_weight_from_alpha and the nerfacc.accumulate_along_rays calls
 * (network/shapeRenderer.py:1166-1206).  Samples are packed ray after ray;
 * ray_offsets[r]..ray_offsets[r+1] (int32, n_rays+1 entries) replaces int64 ray_indices.
 *   variance : device scalar, inv_s = clip(exp(10*variance),1e-6,1e6)
 *   vals[n,D]: per-sample values to accumulate (colour, gradient, radiance, ...), D <= 16
 * outputs: alpha[n], weights[n], acc[r], out[r,D] = sum_i w_i vals_i. */
TF_API int tf_neus_composite_fwd(const float* sdf, const float* grad, const float* dists,
                          const float* dirs, const int32_t* ray_offsets, int32_t n_rays,
                          const float* variance, float cos_anneal, const float* vals, int32_t D,
                          float* alpha, float* weights, float* acc, float* out,
                          tf_stream_t stream);
/* alpha, weights, acc, out are the forward's outputs (acc / out give sum_i u_i w_i without a pass over the samples).
 * g_acc, g_out, g_weights may each be NULL (no upstream gradient on that output).  d_variance is a device scalar
 * accumulated atomically (pass NULL when inv_s is frozen: network/shapeRenderer.py:1007-1008). */
TF_API int tf_neus_composite_bwd(const float* sdf, const float* grad, const float* dists,
                          const float* dirs, const int32_t* ray_offsets, int32_t n_rays,
                          const float* variance, float cos_anneal, const float* vals, int32_t D,
                          const float* alpha, const float* weights, const float* acc, const float* out,
                          const float* g_acc, const float* g_out, const float* g_weights, float* d_sdf,
                          float* d_grad, float* d_vals, float* d_variance, tf_stream_t stream);

/* ---- small MLP layers (tall-skinny fused linear) -------------------------------
 * Y[M,N] = act(X[M,K] W[N,K]^T + b[N]) -- one nn.Linear + activation of the reference's
 * predictor stacks (network/other_field.py:20-121), coupling-layer conditioners
 * (network/flow.py:577-598) and TensoFlow.nis_mat (network/flow.py:694-697).
 * act: 0 none, 1 ReLU, 2 LeakyReLU(0.01), 3 Softplus(beta=100), 4 Sigmoid,
 *      5 exp(min(x, act_param)) (ExpActivation, network/other_field.py:12-18).
 * Row-major contiguous X, W, Y.  b may be NULL.
 * `workspace` (tf_linear_workspace(K, N) bytes, 16-byte aligned, may be NULL) holds the pre-split weights of the
 * tensor-core path: with it, layers of >= 8192 rows and 96 <= K <= 1024, 96 <= N <= 256 run on tcgen05 (3xTF32,
 * fp32-level accuracy; K / N need not be aligned, padded inside); without it, for small batches and for narrow
 * layers the FFMA kernels run. */
TF_API size_t tf_linear_workspace(int32_t K, int32_t N);
TF_API int tf_linear_fwd(const float* X, const float* W, const float* b, int64_t M, int32_t K,
                         int32_t N, int32_t act, float act_param, float* Y, void* workspace,
                         size_t ws_bytes, tf_stream_t stream);
/* dpre[M,N] = dY * act'(Y) (scratch: written except by the fused narrow-layer path, K,N <= 64; must not alias dY);
 * dX[M,K] = dpre W (dX may be NULL); dW[N,K] += dpre^T X and db[N] += colsum(dpre) (each may be NULL). */
TF_API int tf_linear_bwd(const float* X, const float* W, const float* Y, const float* dY,
                         float* dpre, int64_t M, int32_t K, int32_t N, int32_t act,
                         float act_param, float* dX, float* dW, float* db, void* workspace,
                         size_t ws_bytes, tf_stream_t stream);

/* ---- TensoFlow sampler: piecewise-quadratic coupling transform -------------------
 * ElementWisePWQuadraticTransform of the reference (network/flow.py:314-525), one
 * coordinate per row, K = 10 bins from st[M,21] = (11 vertex heights, 10 bin widths).
 *   inverse = 0: forward spline (`flow_inv`, density evaluation, flow.py:332-413)
 *   inverse = 1: inverse spline (`flow`, sampling, flow.py:415-525)
 * y[M] in (0,1) -> x[M], logj[M]. */
TF_API int tf_pwquad_fwd(const float* y, const float* st, int64_t M, int32_t inverse, float* x,
                         float* logj, tf_stream_t stream);
/* Backward of the forward spline (inverse = 0 only: the sampling copies are frozen,
 * network/fields.py:1050-1065): given g_x[M], g_logj[M] -> d_y[M], d_st[M,21]. */
TF_API int tf_pwquad_bwd(const float* y, const float* st, int64_t M, const float* g_x,
                         const float* g_logj, float* d_y, float* d_st, tf_stream_t stream);

/* ---- triangle-mesh ray tracer ---------------------------------------------------------
 * Replaces the un-vendored `_raytracing` extension behind raytracing/raytracer.py:8-54
 * (`create_raytracer(vertices, triangles)` / `impl.trace(o, d, positions, normals, depth)`).
 * tf_bvh_create takes HOST arrays (like the reference, which builds from numpy) and uploads a
 * BVH to the current device; the handle owns that device memory until tf_bvh_destroy.
 * trace: closest hit with t > 0; writes position = o + t d, UNIT face normal (e1 x e2, the
 * reference renderer flips it: network/materialRenderer.py:256-257) and depth = t;
 * a miss writes depth = 10 (the sentinel of materialRenderer.py:261), normal = 0. */
typedef struct tf_bvh_opaque tf_bvh_t;
TF_API int tf_bvh_create(const float* vertices_host, int64_t n_vertices, const int32_t* triangles_host,
                         int64_t n_triangles, tf_bvh_t** out);
TF_API void tf_bvh_destroy(tf_bvh_t* handle);
TF_API int tf_bvh_trace(const tf_bvh_t* handle, const float* rays_o, const float* rays_d, int64_t n,
                        float* positions, float* face_normals, float* depth, tf_stream_t stream);

/* ---- material-stage Monte-Carlo integral (network/fields.py:1075-1335) -----------------
 * tf_mc_directions builds one direction set per surface point and its pdf:
 *   mode 0: flow samples in the half-vector parametrisation (fields.py:1085-1108,1164-1188)
 *           src = angles [pn,sn,2] in (0,1)^2, aux = logj [pn,sn]
 *   mode 1: fixed cosine set (fields.py:824-847): src = table [sn,2] (az/2pi, el),
 *           aux = per-point azimuth shift in [0,1) [pn] or NULL
 *   mode 2: fixed GGX set (fields.py:858-895): as mode 1 plus roughness [pn]
 * Outputs go to dirs[(p*out_stride + out_offset + s)*3], prob[p*out_stride + out_offset + s]
 * so several sets can share one [pn, D] buffer.  normals / view_dirs must be unit length. */
TF_API int tf_mc_directions(int32_t mode, const float* normals, const float* view_dirs, const float* src,
                            const float* aux, const float* roughness, int64_t n_points, int32_t n_dirs,
                            float* dirs, float* prob, int32_t out_stride, int32_t out_offset,
                            tf_stream_t stream);
/* EnvLight.direct_light (network/light.py:125-162): out[n,3] = exp(seamless bilinear lookup of the
 * log-radiance cubemap base[6,R,R,3]) where mask[n] != 0 (NULL = all), 0 elsewhere; bwd scatters
 * g_out * out into d_base (accumulated). */
TF_API int tf_cube_light_fwd(const float* base, int32_t res, const float* dirs, const uint8_t* mask,
                             int64_t n, float* out, tf_stream_t stream);
TF_API int tf_cube_light_bwd(int32_t res, const float* dirs, const uint8_t* mask, int64_t n,
                             const float* out, const float* g_out, float* d_base, tf_stream_t stream);
/* Fused coupling block of the TensoFlow sampler (reference network/flow.py:549-641): for each of the M = pn * sn (point,
 * direction) pairs, conditioner MLP [Reshift(PE(y_c, 3 octaves)) (7) | Reshift(feat[p]) (feat_dim)] -> 64 -> 64 -> 64 -> 21
 * with LeakyReLU(0.01) between the layers, then the piecewise-quadratic spline (10 bins) of the other coordinate y_t:
 *   y_out[c] = y_in[c], y_out[t] = spline(y_in[t]) (inverse != 0: the inverse spline = sampling direction),
 *   logj_out = logj_in + log|d y_out[t] / d y_in[t]|   (logj_in == NULL: 0)
 * c = cond (0 / 1), t = 1 - c; feat[pn, feat_dim] holds one conditioning vector per point (sn >= 16 consecutive pairs share
 * it; feat_dim <= 40); W1[64, 7 + feat_dim], W2/W3[64, 64], W4[21, 64] are the nn.Linear weights (row-major [out, in]);
 * scale / offset are the Reshift constants (2, -1).  The [M, 64] activations stay on chip.
 * save_h[M, 3, 64] / save_st[M, 24] (both or none; NULL = not kept): the tensor-core forward stores the three hidden activations
 * and the spline parameters there, and tf_flow_block_bwd given them (saved_h / saved_st) runs its adjoint chain on the tensor
 * cores without recomputing the forward; with NULL it recomputes on the FP32 pipe.  tf_flow_block_uses_tensor_cores() tells
 * which forward kernel is active (TF_FLOW_SIMT=1 in the environment selects the FP32-pipe kernels for A/B runs).
 * bwd (forward spline only): g_y_out[M,2] / g_logj[M] (each may be NULL) -> g_y_in[M,2]; d_feat[pn, feat_dim] and the weight
 * / bias gradients are ACCUMULATED (atomics; the caller zero-initialises).  The gradient of logj_in equals g_logj. */
TF_API int tf_flow_block_fwd(const float* y_in, const float* logj_in, const float* feat, int32_t feat_dim, int32_t sn,
                             const float* W1, const float* b1, const float* W2, const float* b2, const float* W3,
                             const float* b3, const float* W4, const float* b4, float scale, float offset, int32_t cond,
                             int32_t inverse, int64_t M, float* y_out, float* logj_out, float* save_h, float* save_st,
                             tf_stream_t stream);
TF_API int tf_flow_block_uses_tensor_cores(void);
TF_API int tf_flow_block_bwd(const float* y_in, const float* feat, int32_t feat_dim, int32_t sn, const float* W1,
                             const float* b1, const float* W2, const float* b2, const float* W3, const float* b3,
                             const float* W4, const float* b4, float scale, float offset, int32_t cond, int64_t M,
                             const float* saved_h, const float* saved_st, const float* g_y_out, const float* g_logj,
                             float* g_y_in, float* d_feat, float* dW1,
                             float* db1, float* dW2, float* db2, float* dW3, float* db3, float* dW4, float* db4,
                             tf_stream_t stream);
/* Input rows of the inner-light MLP for the occluded (point, direction) pairs (fields.py:951-975): for the pair idx[i]
 * (flat index into the [pn*D] arrays) X[i, 0:51] = positional encoding (8 octaves) of the hit point inters[idx[i]],
 * X[i, 51:123] = integrated directional encoding (utils/ref_utils.py:53-117, degree 5, kappa_inv = 0) of the view direction
 * -dirs[idx[i]] mirrored at normalize(hit_normals[idx[i]]), X[i, 123:ldx] = 0.  ide_mat [17, 36] fp32 and ide_m [36] int32 are
 * the device copies of the IDE polynomial table and the order m of each of its 36 (m, l) entries.  No gradient: the hit
 * records are geometry. */
TF_API int tf_hit_encode(const float* inters, const float* dirs, const float* hit_normals, const int64_t* idx,
                         int64_t n_hits, const float* ide_mat, const int32_t* ide_m, int32_t ldx, float* X,
                         tf_stream_t stream);
/* BRDF weights + estimators per surface point over D = n_diffuse + n_specular directions
 * (fields.py:1146-1157, 1208-1234) and the neural-importance-sampling loss terms (fields.py:1254-1333).
 * out[pn,19] = diffuse estimate (3), specular estimate (3), mean diffuse light (3), mean specular light (3), visibility (1),
 * indirect light (3), then the NIS sums: [16] sum_{j < n_nis_diffuse} sum_rgb f(x_j) log q(x_j) / p(x_j) over the flow-sampled
 * diffuse directions (the first n_nis_diffuse of the diffuse set), [17] the same over the specular directions with N.L > 0,
 * [18] their number, with log q(x) = logq[p,j] - log(max(4 pi^2 H.V sin(theta), 1e-6)), theta = angles[p,j,1] * pi/2 (the
 * half-vector parametrisation).  logq_* / angles_* may be NULL (no NIS term; [16:19] = 0): logq_diffuse [pn, n_nis_diffuse],
 * angles_diffuse [pn, n_nis_diffuse, 2], logq_specular [pn, n_specular], angles_specular [pn, n_specular, 2].
 * The host forms loss_nis_diffuse = -sum_p out[p,16] / (pn n_nis_diffuse 3), loss_nis_specular = -sum_p out[p,17] /
 * max(3 sum_p out[p,18], 1).
 * bwd: g_out[pn,19] -> d_albedo[pn,3], d_metallic[pn], d_roughness[pn], d_lights[pn,D,3], d_logq_diffuse, d_logq_specular. */
TF_API int tf_mc_estimate_fwd(const float* normals, const float* view_dirs, const float* albedo,
                              const float* metallic, const float* roughness, const float* dirs, const float* prob,
                              const float* lights, const uint8_t* hit, int64_t n_points, int32_t n_diffuse,
                              int32_t n_specular, const float* logq_diffuse, const float* angles_diffuse,
                              int32_t n_nis_diffuse, const float* logq_specular, const float* angles_specular,
                              float* out, tf_stream_t stream);
TF_API int tf_mc_estimate_bwd(const float* normals, const float* view_dirs, const float* albedo,
                              const float* metallic, const float* roughness, const float* dirs, const float* prob,
                              const float* lights, const uint8_t* hit, int64_t n_points, int32_t n_diffuse,
                              int32_t n_specular, const float* logq_diffuse, const float* angles_diffuse,
                              int32_t n_nis_diffuse, const float* logq_specular, const float* angles_specular,
                              const float* g_out, float* d_albedo, float* d_metallic, float* d_roughness,
                              float* d_lights, float* d_logq_diffuse, float* d_logq_specular, tf_stream_t stream);

/* ---- cubemap prefilter (EnvLight.build_mips, network/light.py:52-64) -----------------------
 * The reference's diffuse / specular prefilter kernels (network/renderutils/c_src/cubemap.cu:
 * 110-350) are linear maps of the cubemap with weights that depend only on (resolution,
 * roughness, cutoff).  The host builds that operator once as CSR and these entry points apply
 * it to a 3-channel cubemap x[n_cols,3]: y[n_rows,3] = W x, and gx[n_cols,3] += W^T gy. */
TF_API int tf_csr_spmm3_fwd(const int32_t* rowptr, const int32_t* col, const float* val, const float* x,
                            int32_t n_rows, float* y, tf_stream_t stream);
TF_API int tf_csr_spmm3_bwd(const int32_t* rowptr, const int32_t* col, const float* val, const float* gy,
                            int32_t n_rows, float* gx, tf_stream_t stream);

/* ---- total-variation regulariser ---------------------------------------------------------------
 * TVLoss of the reference (network/other_field.py:170-191; TensoSDF.TV_loss_sdf network/fields.py:133-138,
 * MCShadingNetwork.TV_loss :1525-1530) on one channels-last texture x[H,W,C] (C % 4 == 0; lines are W = 1):
 *   sums[0] += sum_{h<H-1} (x[h+1,w,c] - x[h,w,c])^2,  sums[1] += sum_{w<W-1} (x[h,w+1,c] - x[h,w,c])^2
 *   g[h,w,c] += u * (scale_h * d sums[0] / dx + scale_w * d sums[1] / dx),  u = *upstream (device scalar) or 1 if NULL
 * (the host applies weight * 2 / (batch * count_h|w) as in the reference). */
TF_API int tf_tv_fwd(const float* x, int32_t H, int32_t W, int32_t C, float* sums, tf_stream_t stream);
TF_API int tf_tv_bwd(const float* x, int32_t H, int32_t W, int32_t C, float scale_h, float scale_w,
                     const float* upstream, float* g, tf_stream_t stream);

/* ---- Gaussian-smoothness regulariser ------------------------------------------------------------
 * grid_gaussian_loss of the reference (TensoSDF network/fields.py:301-309, MCShadingNetwork :1537-1545; GaussianBlur2D /
 * GaussianBlur1D network/other_field.py:121-168: F.conv2d / F.conv1d, stride 1, zero padding) on one channels-last
 * texture x[H,W,C] (C % 4 == 0; lines are W = 1, KW = 1).  taps is a HOST array [KH*KW] (odd KH, KW; KH*KW <= 81):
 *   r[h,w,c] = x[h,w,c] - sum_{a,b} taps[a,b] x[h+a-KH/2, w+b-KW/2, c]   on the interior KH/2 <= h < H-KH/2, KW/2 <= w < W-KW/2,
 *   r = 0 elsewhere;  *sum += sum r^2
 *   g[h,w,c] += 2 u (r[h,w,c] - sum_{a,b} taps[a,b] r[h-(a-KH/2), w-(b-KW/2), c]),  u = *upstream (device scalar) or 1 if NULL */
TF_API int tf_gauss_residual_fwd(const float* x, int32_t H, int32_t W, int32_t C, const float* taps, int32_t KH,
                                 int32_t KW, float* r, float* sum, tf_stream_t stream);
TF_API int tf_gauss_residual_bwd(const float* r, int32_t H, int32_t W, int32_t C, const float* taps, int32_t KH,
                                 int32_t KW, const float* upstream, float* g, tf_stream_t stream);

/* ---- hierarchical ray sampler ----------------------------------------------------------------------
 * ShapeRenderer.sample_ray / upsample / cat_z_vals (reference network/shapeRenderer.py:820-932) and sample_pdf(det=True)
 * (utils/network_utils.py:117-147) around the SDF-only field queries (tf_sdf_only_fwd).  Depth lists are rows of
 * z[R, stride] / sdf[R, stride] (sorted, the first n entries valid; stride <= 256).
 *   tf_sampler_init     : z[r, j] = clip(box entry / exit, near, far) stratified by lin[j] (= torch.linspace(0, 1, n)) and
 *                         shifted by (t_rand[r] - 0.5) * 2 / n when t_rand != NULL; pts[R*n, 3], level[R*n] = the query points
 *                         and their mip levels log2(ball radius / base_radii) (shapeRenderer.py:966-970).  aabb = HOST
 *                         {min xyz, max xyz}.
 *   tf_sampler_upsample : per ray: merge the m_in samples of the previous round (new_z_in[R, m_in] with their SDF
 *                         new_sdf_in[R*m_in]; NULL / 0 = nothing to merge) into the lists (n -> n + m_in, in place), then
 *                         m new depths from the NeuS section weights of the merged list at the quantiles u[m]
 *                         (= linspace(0.5/m, 1 - 0.5/m, m)) with inv_s = min(exp(10 * *variance), inv_s_cap) (variance == NULL:
 *                         inv_s_cap): new_z[R, m], new_pts[R*m, 3], new_level[R*m].  m == 0 only merges (new_sdf_in may
 *                         then be NULL: the last round's samples carry no SDF).
 *   tf_sampler_finalize : intervals [z_k, z_k + dist_k) (the last one repeats the previous length) whose mid point lies
 *                         inside the box.  Count pass (counts != NULL): counts[r]; write pass (offsets[R+1] = exclusive
 *                         prefix sums of the counts): packed t_starts, t_ends, ray_indices (int64) in ray order. */
TF_API int tf_sampler_init(const float* rays_o, const float* dirs, const float* near, const float* far, const float* radiis,
                           const float* rays_cos, const float* lin, const float* t_rand, const float aabb[6],
                           float base_radii, int32_t R, int32_t n, int32_t stride, float* z, float* pts, float* level,
                           tf_stream_t stream);
TF_API int tf_sampler_upsample(const float* rays_o, const float* dirs, const float* radiis, const float* rays_cos, float* z,
                               float* sdf, const float* new_z_in, const float* new_sdf_in, int32_t m_in, const float* u,
                               int32_t m, const float* variance, float inv_s_cap, float base_radii, int32_t R, int32_t n,
                               int32_t stride, float* new_z, float* new_pts, float* new_level, tf_stream_t stream);
TF_API int tf_sampler_finalize(const float* rays_o, const float* dirs, const float* z, const float aabb[6], int32_t R,
                               int32_t n, int32_t stride, int32_t* counts, const int64_t* offsets, float* t_starts,
                               float* t_ends, int64_t* ray_indices, tf_stream_t stream);

/* ---- secondary-ray SDF probes ----------------------------------------------------------------------
 * get_weights / get_intersection (reference utils/network_utils.py:149-202) and get_intersection_around_mesh
 * (network/materialRenderer.py:281-313) around the SDF-only field queries: NeuS weights of sn depths per ray with
 * inv_s = exp(10 * *variance).
 *   tf_probe_init    : z[r, j] = t0[r] + (t1[r] - t0[r]) * lin[j]  (t0 == NULL: t1[r] * lin[j]), pts = z * dirs + origins
 *   tf_probe_weights : m > 0: m depths resampled at the quantiles u[m] (sample_pdf, det=True) -> new_z[pn, m], new_pts;
 *                      m == 0: weights[pn, sn-1], mid_sdf[pn, sn-1] (-1 where the SDF rises), z_mid[pn, sn-1]. */
TF_API int tf_probe_init(const float* origins, const float* dirs, const float* t0, const float* t1, const float* lin,
                         int32_t pn, int32_t sn, float* z, float* pts, tf_stream_t stream);
TF_API int tf_probe_weights(const float* origins, const float* dirs, const float* z, const float* sdf, const float* variance,
                            int32_t pn, int32_t sn, const float* u, int32_t m, float* new_z, float* new_pts,
                            float* weights, float* mid_sdf, float* z_mid, tf_stream_t stream);

/* ---- alpha-mask lookup ---------------------------------------------------------------------------
 * AlphaGridMask.sample_alpha (reference network/shapeRenderer.py:79-97): out[i] = trilinear sample of volume[D,H,W] at
 * g = (xyz[i] - aabb_min) * inv_half_size - 1 with F.grid_sample's align_corners=True mapping and zero padding
 * (x -> W, y -> H, z -> D).  aabb_min / inv_half_size (= 2 / aabb size) are HOST arrays of 3 floats.  No gradient: the
 * reference only thresholds the result. */
TF_API int tf_alpha_mask_sample(const float* volume, int32_t D, int32_t H, int32_t W, const float aabb_min[3],
                                const float inv_half_size[3], const float* xyz, int64_t n, float* out, tf_stream_t stream);

/* ---- per-sample shape shader ------------------------------------------------------------------------
 * The per-sample arithmetic of ShapeShadingNetwork.forward (reference network/fields.py:448-567) around its MLP heads and
 * environment-light lookups.  ide_mat [17,36] fp32, ide_m [36] int32, ide_sigma [36] fp32 (= l (l + 1) / 2) are device copies of
 * the degree-5 integrated-directional-encoding tables (utils/ref_utils.py:53-117).
 *   tf_shader_encode_fwd: n = normalize(normals) (degenerate n.x + n.y == 0 -> (0, 1e-6, 1)), v = normalize(view_dirs),
 *       nov = n.v, refl = 2 (n.v) n - v, rough = 0.9 mat[:,3] + 0.09 (mat [n,5] = sigmoid outputs of the material head), and the
 *       zero-padded MLP inputs  X_rad[n, ld_rad] = [feat (feat_dim) | points | PE(v, 4 octaves) | n]  (X_rad == NULL: skipped),
 *       X_il[n, 128] = [PE(points, 8) | IDE(refl, rough)],  X_iw[n, 96] = [PE(points, 8) | PE(refl, 6)].
 *   tf_shader_encode_bwd: upstream gradients of nrm, refl, nov, rough, X_rad, X_il (each may be NULL; X_iw carries none, the
 *       reference detaches it) -> d_normals[n,3], d_mat3[n] (gradient of mat[:,3]), d_feat[n, feat_dim] (NULL: skipped).
 *   tf_shader_combine_fwd: albedo = 0.77 mat[:,0:3] + 0.03, metallic = mat[:,4], occ_prob = 0.5 w_raw + 0.5,
 *       specular light = indirect * occ + direct * (1 - occ) (occ = clamp(occ_prob, 0, 1)), split-sum terms from the bilinear
 *       clamp lookup of lut[lut_h, lut_w, 2] at (clamp(nov), clamp(rough)), color = clamp(linear_to_srgb(diffuse + specular), 0, 1).
 *   tf_shader_combine_bwd: g_color[n,3], g_occ[n] (may be NULL) -> d_mat[n,5], d_diffuse, d_direct, d_indirect [n,3],
 *       d_w_raw[n], d_nov[n]. */
TF_API int tf_shader_encode_fwd(const float* points, const float* normals, const float* view_dirs, const float* mat,
                                const float* feat, int32_t feat_dim, int32_t ld_rad, int64_t n, const float* ide_mat,
                                const int32_t* ide_m, const float* ide_sigma, float* nrm, float* vdir, float* refl,
                                float* nov, float* rough, float* X_rad, float* X_il, float* X_iw, tf_stream_t stream);
TF_API int tf_shader_encode_bwd(const float* normals, const float* view_dirs, const float* mat, int32_t feat_dim,
                                int32_t ld_rad, int64_t n, const float* ide_mat, const int32_t* ide_m,
                                const float* ide_sigma, const float* g_nrm, const float* g_refl, const float* g_nov,
                                const float* g_rough, const float* g_X_rad, const float* g_X_il, float* d_normals,
                                float* d_mat3, float* d_feat, tf_stream_t stream);
TF_API int tf_shader_combine_fwd(const float* mat, const float* diffuse_light, const float* direct_light,
                                 const float* indirect_light, const float* w_raw, const float* nov, const float* lut,
                                 int32_t lut_h, int32_t lut_w, int64_t n, float* color, float* occ_prob,
                                 tf_stream_t stream);
TF_API int tf_shader_combine_bwd(const float* mat, const float* diffuse_light, const float* direct_light,
                                 const float* indirect_light, const float* w_raw, const float* nov, const float* lut,
                                 int32_t lut_h, int32_t lut_w, int64_t n, const float* g_color, const float* g_occ,
                                 float* d_mat, float* d_diffuse, float* d_direct, float* d_indirect, float* d_w_raw,
                                 float* d_nov, tf_stream_t stream);

/* ---- differentiable cubemap lookup ---------------------------------------------------------------
 * dr.texture(tex, dirs, [mip=stack, mip_level_bias=level,] filter_mode='linear[-mipmap-linear]', boundary_mode='cube') of the
 * shape-stage light (reference network/light.py:95-122, 135; network/light_utils.py:46-63): seamless bilinear footprint per
 * level (edge taps fold onto the neighbouring face, the corner tap is dropped, weights renormalised), linear blend of the two
 * levels around clamp(level, 0, n_levels-1).  tex[l] is [6,res[l],res[l],3] fp32; `tex`, `d_tex`, `res` are HOST arrays of
 * n_levels (<= 8) entries; level == NULL reads level 0 only.  Backward accumulates into d_tex[l] (atomics, zero-initialised
 * by the caller; entries / the array may be NULL) and writes d_dirs[n,3], d_level[n] (each may be NULL). */
TF_API int tf_cube_sample_fwd(const float* const* tex, const int32_t* res, int32_t n_levels, const float* dirs,
                              const float* level, int64_t n, float* out, tf_stream_t stream);
TF_API int tf_cube_sample_bwd(const float* const* tex, const int32_t* res, int32_t n_levels, const float* dirs,
                              const float* level, int64_t n, const float* g_out, float* const* d_tex, float* d_dirs,
                              float* d_level, tf_stream_t stream);

/* ---- occupancy-grid marcher ---------------------------------------------------------------------
 * nerfacc.OccGridEstimator.sampling as the reference calls it (network/shapeRenderer.py:950-959, 1065-1072): fixed
 * render_step_size, no cone angle, no visibility filter.  nerfacc is not vendored; the rule restated here:
 *   t_k = near[r] + k * step;  interval [t_k, t_k + step] is kept iff its mid-point m satisfies m < far, o + d m lies
 *   inside aabb = {lo xyz, hi xyz} and binaries[(cx * res[1] + cy) * res[2] + cz] != 0, c = floor((p - lo) / (hi - lo) * res).
 * Two passes around a host-side exclusive prefix sum: counts[r] = kept intervals of ray r; then, with offsets[R+1],
 * ray_indices / t_starts / t_ends [offsets[R]] are written ray after ray in marching order (nerfacc's packed format).
 * `aabb` (6 floats) and `res` (3 ints) are HOST arrays; binaries is the device bool / uint8 grid. */
TF_API int tf_occ_march_count(const float* rays_o, const float* rays_d, const float* near, int32_t n_rays, float far,
                              float step, const float* aabb, const int32_t* res, const uint8_t* binaries, int32_t* counts,
                              tf_stream_t stream);
TF_API int tf_occ_march_write(const float* rays_o, const float* rays_d, const float* near, int32_t n_rays, float far,
                              float step, const float* aabb, const int32_t* res, const uint8_t* binaries,
                              const int32_t* offsets, int64_t* ray_indices, float* t_starts, float* t_ends,
                              tf_stream_t stream);

/* ---- isosurface extraction (marching cubes) ---------------------------------------------------------
 * mcubes.marching_cubes(u, threshold) as extract_mesh.py calls it on the shape stage's SDF lattice, GPU-resident.
 * u [nx][ny][nz] fp32, z fastest, nx, ny, nz >= 2, nx*ny*nz < 2^31; a point is inside iff u < threshold.  Rows are the
 * nx*ny (i, j) lines of points.
 *   vertices: one per crossed lattice edge, owned by the edge's lower point p = (i*ny + j)*nz + k, ordered by (p, axis x/y/z),
 *             at index coordinate a_axis + (threshold - u_a) / (u_b - u_a) (each op one fp32 rounding);
 *   triangles int32 [T,3]: cells in order (i*ny + j)*nz + k, then in the order of the generated case table
 *             (tensoflow_b200/isosurface_table.py); (v1 - v0) x (v2 - v0) points toward increasing u.
 * tf_iso_count writes per row the owned crossed edges (vert_count[nx*ny]) and the triangles of the row's cells
 * (tri_count[nx*ny]).  The caller takes the exclusive prefix sums (int64, totals < 2^31), then tf_iso_vertices writes
 * vertices [V,3] and index_volume [nx*ny*nz] (int32 vertices owned by the points before p, every p), and
 * tf_iso_triangles reads index_volume and writes triangles [T,3].  No atomics: the output is bit-reproducible. */
TF_API int tf_iso_count(const float* u, int32_t nx, int32_t ny, int32_t nz, float threshold, int32_t* vert_count,
                        int32_t* tri_count, tf_stream_t stream);
TF_API int tf_iso_vertices(const float* u, int32_t nx, int32_t ny, int32_t nz, float threshold, const int64_t* vert_offsets,
                           float* vertices, int32_t* index_volume, tf_stream_t stream);
TF_API int tf_iso_triangles(const float* u, int32_t nx, int32_t ny, int32_t nz, float threshold, const int64_t* tri_offsets,
                            const int32_t* index_volume, int32_t* triangles, tf_stream_t stream);

/* ---- optimizer step ------------------------------------------------------------------------------
 * torch.optim.Adam(grad_vars, betas=(0.9, 0.99)).step() of the reference trainer (train/trainer_inv.py:112,212; one
 * learning rate per parameter group, :247-248) as ONE streaming pass: for tensor t (numel[t] fp32 elements in any
 * memory order, the four buffers laid out alike) and step k >= 1
 *   m = m + (1-beta1)(g - m);  v = beta2 v + (1-beta2) g^2;
 *   p = p - lr[t] / (1-beta1^k) * m / (sqrt(v) / sqrt(1-beta2^k) + eps)
 * The pointer / numel / lr tables are HOST arrays of n_tensors entries (device pointers inside); launches cover 32
 * tensors each.  28 B of HBM traffic per element. */
TF_API int tf_adam_step(int32_t n_tensors, float* const* params, const float* const* grads, float* const* exp_avg,
                        float* const* exp_avg_sq, const int64_t* numel, const float* lr, float beta1, float beta2,
                        float eps, int32_t step, tf_stream_t stream);

/* ---- per-kernel timing ------------------------------------------------------------------------
 * While enabled, the fused decoder kernels (sdf_stencil_fwd_tc, sdf_stencil_bwd_tc, xty_tc, linear_tc) are
 * bracketed by CUDA events on their launching stream.  tf_kernel_timing_read sums the recorded launches of
 * one kernel (it synchronises on their events); returns 1 when nothing was recorded under that name. */
TF_API void tf_kernel_timing_enable(int32_t on);
TF_API void tf_kernel_timing_reset(void);
TF_API int tf_kernel_timing_read(const char* name, double* total_ms, int32_t* launches);

/* ---- weight-gradient accumulate --------------------------------------------------------------
 * out[m][n] += sum_r X[r][m] * Y[r][n]  (X [rows,M], Y [rows,N], out [M,N], all row-major fp32).
 * This is the dW = dPre^T X product every nn.Linear backward of the path ends with
 * (torch autograd's addmm in the reference: network/fields.py:192-198 decoder, other/material MLPs).
 * Shapes with M in {128,256}, N % 16 == 0, N <= 256 run on tcgen05 (3xTF32, fp32-level accuracy);
 * anything else on the FFMA kernel.  force_simt != 0 selects the FFMA kernel (A/B testing). */
TF_API int tf_xty_accumulate(const float* X, const float* Y, int64_t rows, int32_t M, int32_t N, float* out,
                             int32_t force_simt, tf_stream_t stream);

#ifdef __cplusplus
}
#endif
#endif /* TENSOFLOW_B200_H */
