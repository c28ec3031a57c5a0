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

#define TF_ABI_VERSION 3

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

/* Byte offset of the centre hidden activations [n, hidden] inside the workspace that was passed to tf_sdf_stencil_fwd (with
 * feat != NULL); (size_t)-1 exactly when the tensor-core forward does not apply to this decoder shape (then neither
 * tf_sdf_point_fwd nor the block exists). */
TF_API size_t tf_sdf_stencil_fwd_hidden_offset(const tf_vm_field_t* f, const tf_sdf_mlp_t* m);

/* Backward of tf_sdf_stencil_fwd.  g_sdf[n], g_feat[n,A], g_grad[n,3], g_hess[n] are the
 * upstream gradients (each may be NULL = zero); sdf7 is the forward output.
 * hidden_centre[n, hidden] is the block at tf_sdf_stencil_fwd_hidden_offset(f, m) of the forward's workspace, which the caller
 * keeps alive until this call (it feeds the weight gradient of the appearance head and is not recomputed).  It is required when
 * g_feat != NULL and the offset is not (size_t)-1 (tensor-core path): the call returns an error without it.  Otherwise it is
 * ignored and may be NULL.
 * Any workspace size >= tf_sdf_stencil_bwd_workspace(.., 1) works; larger is faster
 * (the call processes the n samples in slices that fit). */
TF_API size_t tf_sdf_stencil_bwd_workspace(const tf_vm_field_t* f, const tf_sdf_mlp_t* m, int64_t n_slice);
TF_API int tf_sdf_stencil_bwd(const tf_vm_field_t* f, const tf_sdf_mlp_t* m, const float* xyz,
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
 * The shape picks the kernel.  Layers of >= 8192 rows with 96 <= K <= 1024, 96 <= N <= 256 run the forward on
 * tcgen05 (3xTF32, fp32-level accuracy; K / N need not be aligned, padded inside), and layers of >= 8192 rows with
 * 96 <= K <= 256, 96 <= N <= 1024 run the data gradient dX there; smaller batches and narrower layers run on FFMA.
 * tf_linear_workspace(M, K, N) is the size in bytes of the 16-byte aligned `workspace` that holds the pre-split
 * weights of the tcgen05 path at that shape, for either direction, and 0 when neither direction uses it.  When a
 * call takes the tcgen05 path, a NULL, smaller or unaligned workspace is an error. */
TF_API size_t tf_linear_workspace(int64_t M, int32_t K, int32_t N);
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
 * tf_bvh_create takes HOST arrays (like the reference, which builds from numpy), builds the BVH on the
 * host and uploads it to the current device; the handle owns that device memory until tf_bvh_destroy.
 * It rejects an index out of range and a non-finite coordinate on a referenced vertex.
 * trace: closest hit with t > 0; writes position = o + t d, UNIT face normal (e1 x e2, the
 * reference renderer flips it: network/materialRenderer.py:256-257) and depth = t;
 * a miss writes depth = 10 (the sentinel of materialRenderer.py:261), normal = 0. */
typedef struct tf_bvh_opaque tf_bvh_t;
TF_API int tf_bvh_create(const float* vertices_host, int64_t n_vertices, const int32_t* triangles_host,
                         int64_t n_triangles, tf_bvh_t** out);
TF_API void tf_bvh_destroy(tf_bvh_t* handle);
TF_API int tf_bvh_trace(const tf_bvh_t* handle, const float* rays_o, const float* rays_d, int64_t n,
                        float* positions, float* face_normals, float* depth, tf_stream_t stream);

/* ---- BVH build on the device -----------------------------------------------------------
 * The same tree as tf_bvh_create, node for node: nodes (32 B: bmin[3], first, bmax[3], count), triangles (48 B: v0, e1 = b - a,
 * e2 = c - a, each padded with a 0) and perm [n_triangles] (caller index of each triangle slot) are byte-equal to the host
 * build's.  The rule both follow: ranges split at lo + cnt/2 until cnt <= 4; the axis is that of the largest fp32 centroid
 * extent, ties preferring x then y; the left half holds the cnt/2 smallest triangles by (centroid on that axis, caller index);
 * centroids are ((a + b) + c) * (1/3) rounded per operation; -0 counts as +0; a leaf lists its triangles by caller index; the
 * k-th inner node in right-first preorder has its children at 1 + 2k and 2 + 2k.
 * tf_bvh_build_sizes: for 0 < n_triangles < 2^31, the node count of the tree and the bytes of scratch tf_bvh_build needs (this
 *   includes the radix sort's temporary storage as CUB sizes it on the current device).
 * tf_bvh_build: vertices [n_vertices,3] fp32 and triangles [n_triangles,3] int32 on the current device; every index must be in
 *   [0, n_vertices) and every referenced coordinate finite (the kernels do not check: mc_ops.RayTracer validates with one host
 *   read first).  workspace (>= the bytes above, 16-byte aligned) is caller-owned scratch; outputs nodes [n_nodes], tris
 *   [n_triangles] (both 16-byte aligned) and perm [n_triangles].  Level by level: a segmented min / max, one kernel writing
 *   64-bit keys, and one CUB radix sort, about ceil(log2(n / 4)) + 1 levels; everything on `stream`, no allocation, no host
 *   synchronisation.  tf_launch_count counts the build's own kernels, not the sort's.
 * tf_bvh_create_from_device: a handle from device nodes / tris / perm (layouts as above) on the current device.  It COPIES them
 *   (cudaMemcpyAsync on `stream`) into memory the handle owns, so the sources may be released once those copies are ordered
 *   before their reuse (the same stream); tf_bvh_destroy frees the handle's memory and never the sources.
 * tf_bvh_export: the sizes of any handle (NULL to skip) and, for each non-NULL destination, a copy of its nodes [n_nodes]
 *   (32 B each), tris [n_triangles] (48 B each) and perm [n_triangles] to host or device memory.  It synchronises the handle's
 *   device first (so copies enqueued by tf_bvh_create_from_device on any stream are complete) and returns when the copies are.
 * The first three return non-zero with tf_last_error() on a NULL pointer, an empty mesh or n_triangles >= 2^31;
 * tf_bvh_export on a NULL handle or a failed copy. */
TF_API int tf_bvh_build_sizes(int64_t n_triangles, int64_t* n_nodes, size_t* workspace_bytes);
TF_API int tf_bvh_build(const float* vertices, int64_t n_vertices, const int32_t* triangles, int64_t n_triangles,
                        void* workspace, size_t workspace_bytes, void* nodes, void* tris, int32_t* perm, tf_stream_t stream);
TF_API int tf_bvh_create_from_device(const void* nodes, int64_t n_nodes, const void* tris, const int32_t* perm,
                                     int64_t n_triangles, tf_stream_t stream, tf_bvh_t** out);
TF_API int tf_bvh_export(const tf_bvh_t* handle, int64_t* n_nodes, int64_t* n_triangles, void* nodes, void* tris,
                         int32_t* perm);

/* ---- geometry evaluation (point-to-mesh distances, surface samples) ----------------------------
 * tf_bvh_closest_point: for each of the n query points [n,3], the nearest point of the mesh behind `handle`:
 *   out_points [n,3] (fp32), out_dist [n] (Euclidean, fp32), out_tri [n] (int64 index into the triangles given to
 *   tf_bvh_create, in the caller's order).  Branch-and-bound over the BVH; per triangle Ericson's 7-region test
 *   (Real-Time Collision Detection 5.1.5) in fp32; a triangle whose height is below 2^-24 of its longest edge (zero area,
 *   collinear) is measured through its edges and vertices.  The smaller squared distance wins, an exact tie goes to the
 *   smaller triangle index; no atomics, so two runs are bit-identical.  A query point with a NaN coordinate gives out_tri = -1.
 * tf_mesh_sample_surface: n area-weighted samples of the mesh vertices [V,3] fp32 / triangles [n_tris,3] int32 (indices in
 *   range, the caller checks).  cdf [n_tris] fp64 is the inclusive, normalised cumulative triangle area (last element 1);
 *   uniforms [n,3] fp64 in [0,1): triangle t = the first with cdf[t] > u0 (binary search), point
 *   (1 - sqrt(u1)) a + sqrt(u1)(1 - u2) b + sqrt(u1) u2 c evaluated in fp64 and rounded once; out_points [n,3] fp32,
 *   out_tri [n] int64, out_normals [n,3] fp32 = unit (b - a) x (c - a).
 * Both: n == 0 launches nothing; no allocation, no synchronisation. */
TF_API int tf_bvh_closest_point(const tf_bvh_t* handle, const float* points, int64_t n, float* out_points, float* out_dist,
                                int64_t* out_tri, tf_stream_t stream);
TF_API int tf_mesh_sample_surface(const float* vertices, const int32_t* triangles, int64_t n_tris, const double* cdf,
                                  const double* uniforms, int64_t n, float* out_points, int64_t* out_tri, float* out_normals,
                                  tf_stream_t stream);

/* ---- mesh clean-up: connected components ------------------------------------------------------------
 * tf_mesh_components: connected components of the graph whose nodes are the n_vertices vertices and whose edges are the
 *   edges of the n_tris triangles [n_tris,3] int32 (every index in [0, n_vertices): precondition, checked by the caller;
 *   geometry.mesh_components does it with one host read).
 *   root[v]      = the smallest vertex index in v's component (a vertex no triangle references is its own component);
 *   tri_count[r] = the number of triangles whose vertices have root r (zero for every non-root v).
 *   root and tri_count are [n_vertices] int32 outputs; tri_count is zeroed by the call.  0 < n_vertices < 2^31,
 *   0 <= n_tris < 2^31.  Lock-free union-find (ECL-CC: hooks by atomicCAS of the larger root under the smaller, path halving),
 *   then a flatten pass and integer atomics for the counts.  No workspace, no host synchronisation; the result does not
 *   depend on scheduling.  Returns non-zero with tf_last_error() on a NULL pointer or a count out of range, before any launch. */
TF_API int tf_mesh_components(const int32_t* triangles, int64_t n_tris, int64_t n_vertices, int32_t* root, int32_t* tri_count,
                              tf_stream_t stream);

/* ---- mesh simplification: quadric-error edge collapse in rounds -------------------------------------------
 * Garland-Heckbert edge collapse, run in rounds of collapses whose closed 1-rings are vertex-disjoint.  The result is
 * deterministic and bit-equal to oracle/torch_oracle_simplify.py, which restates every rule below in numpy.
 *   quadrics   fp64, per vertex the sum of the unit-normal plane quadrics p p^T of its faces (no area weight, so sqrt(cost) is a
 *              length), summed in face order; a face of zero-length cross product (b - a) x (c - a) adds nothing.  A collapse
 *              gives the survivor Q_a + Q_b.  fp64 operations are rounded one by one (no FMA contraction).
 *   placement  v minimises v^T Q v: with A the 3x3 block of Q, v = -A^-1 (Q_xd, Q_yd, Q_zd) from the adjugate when det(A) >
 *              1e-6 trace(A)^3, else the cheapest of a, b and their midpoint (ties in that order).  v is rounded to fp32 and the
 *              cost max(0, v^T Q v) is taken there; positions are fp32 throughout.  The survivor is the smaller index a.
 *   validity   an edge {a, b} may collapse iff it has exactly two faces, with different apexes c0, c1; neither a nor b is locked
 *              (a vertex is locked when an edge with a face count other than 2 ends there, or a face with a repeated index
 *              holds it: open boundaries and non-manifold vertices stay bit-identical); c0 and c1 each have more than 3 faces;
 *              a and b have no common neighbour but c0 and c1 (link condition); every other face of the two stars whose old
 *              normal is not zero keeps a new normal at a positive dot product with it (no fold-over, no new degenerate face);
 *              and sqrt(cost) <= max_error.
 *   selection  valid edges are ranked by (fp32 cost, a, b); the first k = min(max(1, n_valid / 16), (T - target) / 2) are
 *              candidates.  Candidate i has priority (splitmix64(a << 32 | b) >> 32) << 32 | i and wins iff it holds the minimum
 *              priority claimed by every vertex of its closed 1-ring (the vertices of the faces of a and of b).  Priorities are
 *              hashed, not costs: smooth costs have few local minima, so cost priorities would let a handful of edges win.
 *   stopping   when T <= target + 1 or a round collapses nothing.  Each collapse removes two faces, so T' >= target.
 *   output     surviving faces keep their relative order, referenced vertices keep theirs, indices are renumbered; with no
 *              collapse and every vertex referenced the output equals the input byte for byte.
 * tf_mesh_simplify_sizes: the bytes of scratch tf_mesh_simplify needs for n_vertices and n_triangles (including CUB's temporary
 *   storage as sized on the current device), about 310 bytes per triangle.
 * tf_mesh_simplify: vertices [n_vertices,3] fp32 and triangles [n_triangles,3] int32 on the current device (every index in
 *   [0, n_vertices): precondition, geometry.simplify_mesh checks it with one host read), target >= 0 triangles, max_error >= 0
 *   (+inf for no bound).  Writes out_vertices [V',3] and out_triangles [T',3] (buffers of the input sizes) and V', T' and the
 *   number of rounds that collapsed something to the host pointers.  It runs every round on `stream` and, at the end of each
 *   round, reads one count (the surviving faces) to the host with cudaMemcpyAsync and a stream synchronise; it returns after a
 *   last such read of V'.  Each round re-sorts the (vertex, face) pairs and the half-edges with CUB radix sorts.
 * Both return non-zero with tf_last_error() before any launch on a NULL pointer, 0 or >= 2^31 vertices, 0 or >= 2^31 triangles
 * or 3 n_triangles >= 2^31 (the half-edge sorts count in int; at about 310 B of workspace per triangle no device holds that
 * many), target < 0, max_error negative or NaN, or a workspace smaller than the sizes call gives. */
TF_API int tf_mesh_simplify_sizes(int64_t n_vertices, int64_t n_triangles, size_t* workspace_bytes);
TF_API int tf_mesh_simplify(const float* vertices, int64_t n_vertices, const int32_t* triangles, int64_t n_triangles, int64_t target,
                            double max_error, void* workspace, size_t workspace_bytes, float* out_vertices, int32_t* out_triangles,
                            int64_t* out_n_vertices, int64_t* out_n_triangles, int32_t* out_rounds, tf_stream_t stream);

/* ---- UV atlas of box-projection charts and texture baking -------------------------------------------------
 * Deterministic and bit-equal to oracle/torch_oracle_atlas.py, which restates every rule below in numpy.  fp64 operations are
 * rounded one by one (no FMA contraction) and summed in a fixed order; the only atomics are integer ones.
 *   classes    n = (b - a) x (c - a) in fp64, len = |n|.  Class 2k + (n_k < 0), k the axis of the largest |n_k| (ties to the lower
 *              axis).  Class c (axis c / 2, + for even c) is allowed iff +-n_k >= len / 2, i.e. |n^ . axis| >= 1/2 on the front
 *              side.  4 Jacobi passes: per class, len of the face and of its edge neighbours (for each of its edges k = 0, 1, 2,
 *              the other faces of that edge, ascending) summed in that order; the face takes the allowed class of the largest
 *              sum, its own on ties, then the lower class.
 *   charts     faces sharing an edge (two vertex indices) and a class, neither marked solo, are joined (union-find over faces as
 *              in tf_mesh_components); a chart's root is its smallest face and charts are numbered by root.
 *   projection chart axis k: (u, w) = (p[(k+1)%3], p[(k+2)%3]) for +k, swapped for -k (front faces stay counter-clockwise);
 *              one density s (texels per world unit) for all charts.
 *   packing    rect = max(1, ceil(extent * s)) + 2 padding per axis; rects sorted by (h desc, w desc, chart asc), next-fit
 *              decreasing height into shelves of width R.  s0 = R / sqrt(projected area), the area summed in fixed point
 *              (rint(|n_k| / max |n_k| * 2^32) in uint64); s = s0 if it fits, else the lo of 20 bisection steps on (0, s0].
 *   texels     corner x = fp32((x0 + padding) + (u - umin) s), y likewise, in [0, R]; uv = (x / R, y / R) and texture row j spans
 *              v in [j/R, (j+1)/R] (image writers with row 0 at the top flip v).  Texel (i, j) is covered when its centre
 *              (i + 1/2, j + 1/2) is inside the triangle: fp64 edge functions taken from the endpoint smaller in (x, y) order
 *              (so both faces of an edge see one value), > 0 or = 0 on a top-left edge; a face of negative signed area is taken
 *              reversed, one of zero covers nothing.  Coverage runs over 8x8 tiles of each face's box (a prefix sum of tile
 *              counts, one thread per tile), so a few huge faces do not stall.
 *   conflicts  every face covering a centre that another face covers is marked solo (a chart of its own) and charts, density,
 *              packing and coverage run again, until no centre is covered twice (single triangles never overlap, and rects are
 *              disjoint).  A chart covering no centre gets the texel under its root face's texel centroid, clamped into its rect.
 *   output     vertices are the unique (source vertex, chart) pairs in (vertex, chart) order (split along seams); triangles
 *              keep their order.
 * tf_uv_atlas_sizes: the scratch bytes of tf_uv_atlas (CUB temporary storage sized on the current device), about 250 B per
 *   triangle.
 * tf_uv_atlas: vertices [n_vertices,3] fp32, triangles [n_triangles,3] int32 (indices in range: precondition, geometry.uv_atlas
 *   checks it), 16 <= resolution R <= 16384, 1 <= padding <= 16.  Writes out_chart [T] int32, out_triangles [T,3] int32 (output
 *   vertex ids), out_vertex_index [V'] int64 and out_xy [V',2] fp32 (buffers of 3T rows), out_texel_tri [R,R] int32 (owner
 *   face, -1 for none), out_rects [C,4] int32 (x0, y0, w, h; buffer of T rows), and to host pointers s, V', C, the conflict
 *   rounds and the density trials.  Host reads: the chart count once, one (conflicts, next chart count) read per round and
 *   V' at the end; the density search keeps its state on the device.  Returns 3 with tf_last_error() when the charts do not
 *   fit at any density tried.
 * tf_uv_texel_points: for n texels (j R + i) owned in texel_tri, the point at the barycentrics of the centre in the owner of
 *   triangles [T,3] over vertices [V',3] and xy [V',2] (fp64, clamped at 0 and renormalised; the centroid for a zero-area
 *   face), rounded once to fp32 -> out_points [n,3].
 * tf_uv_fill_sizes / tf_uv_fill: values [n,channels] fp32 scattered to their texels of texture [R,R,channels] (zeroed), then
 *   `padding` dilation passes: an empty texel inside the rect of a filled 8-neighbour's chart takes the fp32 mean of those
 *   neighbours, summed in row order (dy, then dx, from -1).  Rects are disjoint, so bilinear lookups never mix charts.
 * All return non-zero with tf_last_error() before any launch on a NULL pointer, 0 or >= 2^31 vertices or triangles, 3 T >= 2^31,
 * R or padding out of range, or a workspace smaller than the sizes call gives. */
TF_API int tf_uv_atlas_sizes(int64_t n_vertices, int64_t n_triangles, int32_t resolution, size_t* workspace_bytes);
TF_API int tf_uv_atlas(const float* vertices, int64_t n_vertices, const int32_t* triangles, int64_t n_triangles, int32_t resolution,
                       int32_t padding, void* workspace, size_t workspace_bytes, int32_t* out_chart, int32_t* out_triangles,
                       int64_t* out_vertex_index, float* out_xy, int32_t* out_texel_tri, int32_t* out_rects, double* out_scale,
                       int64_t* out_n_vertices, int64_t* out_n_charts, int32_t* out_rounds, int32_t* out_steps, tf_stream_t stream);
TF_API int tf_uv_texel_points(const float* vertices, const int32_t* triangles, const float* xy, const int32_t* texel_tri,
                              int32_t resolution, const int64_t* texels, int64_t n, float* out_points, tf_stream_t stream);
TF_API int tf_uv_fill_sizes(int32_t resolution, int32_t channels, size_t* workspace_bytes);
TF_API int tf_uv_fill(const float* values, const int64_t* texels, int64_t n, int32_t channels, const int32_t* texel_tri,
                      const int32_t* chart, const int32_t* rects, int32_t resolution, int32_t padding, void* workspace,
                      size_t workspace_bytes, float* out_texture, tf_stream_t stream);

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
 * Both directions run on the tensor cores (tcgen05).
 * save_h[M, 3, 64] / save_st[M, 24] (both or none; NULL = not kept): the forward stores the three hidden activations and the
 * spline parameters there.  tf_flow_block_bwd requires them (saved_h / saved_st, from a forward with inverse = 0): its adjoint
 * chain reads them and does not recompute the forward; without them it returns an error and launches nothing.
 * bwd (forward spline only): g_y_out[M,2] / g_logj[M] (each may be NULL) -> g_y_in[M,2]; d_feat[pn, feat_dim] and the weight
 * / bias gradients are ACCUMULATED (atomics; the caller zero-initialises).  The gradient of logj_in equals g_logj. */
TF_API int tf_flow_block_fwd(const float* y_in, const float* logj_in, const float* feat, int32_t feat_dim, int32_t sn,
                             const float* W1, const float* b1, const float* W2, const float* b2, const float* W3,
                             const float* b3, const float* W4, const float* b4, float scale, float offset, int32_t cond,
                             int32_t inverse, int64_t M, float* y_out, float* logj_out, float* save_h, float* save_st,
                             tf_stream_t stream);
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

/* ---- narrow-band isosurface extraction -------------------------------------------------------------
 * The mesh of tf_iso_* (same vertex order, interpolation, triangle order and winding) on a lattice of nx, ny, nz points
 * (2..4096 each; point, edge and cell indices are int64) whose values are known only in bricks around the surface.
 * Bricks are 8^3 cells, brick (I, J, K) has id (I*by + J)*bz + K (bx = ceil((nx-1)/8), ...), covers the points 8I ..
 * min(8I + 8, nx-1) per axis, and owns its cells and the points 8I .. 8I + 7 (the last brick on an axis also its end point).
 * Band rule (tensoflow_b200.isosurface.marching_cubes_narrowband drives it):
 *   1. coarse values u on the points min(8I, n-1) per axis, [bx+1][by+1][bz+1];
 *   2. tf_iso_nb_classify: flags[brick] = 1 iff its 8 coarse corners straddle the threshold or one has
 *      |u - threshold| < band (band = sqrt(3)*8*h_max rounded to fp32, h_max the largest axis spacing), else 0;
 *   3. the values of the active bricks, values[slot][9][9][9] (z fastest; positions past the lattice's end are never read),
 *      at the xyz tf_iso_nb_points writes ([n][729][3], from the axis tables; positions past the end repeat the last point);
 *   4. tf_iso_nb_grow: for each crossed lattice edge in the closure of a listed brick, sets flags = 2 on every brick with
 *      flag 0 whose closure holds the edge (face and edge neighbours).  The caller activates them and repeats from 3
 *      until a round adds none.
 * For a 1-Lipschitz field no brick holding a crossing is missed.  Otherwise every surface component that one active brick
 * touches is still extracted whole; a component that no coarse corner sees (a steep, tiny closed surface between coarse
 * points) is absent.  With the final active bricks in any slot order:
 *   tf_iso_nb_count      per segment (slot*81 + 9*x + y: the row of local points (x, y, *)) the owned crossed edges, the
 *                        triangles of its cells and the key (i*ny + j)*bz + K (INT64_MAX for a row the brick does not own);
 *   the caller sorts the keys and takes exclusive int64 prefix sums of both counts in key order (totals < 2^31);
 *   tf_iso_nb_vertices   vertices [V,3] and index[slot][729] (int32 id of the first vertex of each owned point);
 *   tf_iso_nb_triangles  triangles [T,3] through slot_map[brick id] (int32 slot of every active brick).
 * No atomics: the output is bit-reproducible.  It equals tf_iso_* on the dense lattice when every cell with a crossing lies
 * in an active brick. */
TF_API int tf_iso_nb_classify(const float* coarse, int32_t nx, int32_t ny, int32_t nz, float threshold, float band, uint8_t* flags,
                              tf_stream_t stream);
TF_API int tf_iso_nb_points(const float* ax, const float* ay, const float* az, int32_t nx, int32_t ny, int32_t nz,
                            const int64_t* bricks, int64_t n_bricks, float* xyz, tf_stream_t stream);
TF_API int tf_iso_nb_grow(const float* values, const int64_t* bricks, int64_t n_bricks, int32_t nx, int32_t ny, int32_t nz,
                          float threshold, uint8_t* flags, tf_stream_t stream);
TF_API int tf_iso_nb_count(const float* values, const int64_t* bricks, int64_t n_bricks, int32_t nx, int32_t ny, int32_t nz,
                           float threshold, int32_t* vert_count, int32_t* tri_count, int64_t* keys, tf_stream_t stream);
TF_API int tf_iso_nb_vertices(const float* values, const int64_t* bricks, int64_t n_bricks, int32_t nx, int32_t ny, int32_t nz,
                              float threshold, const int64_t* vert_offsets, float* vertices, int32_t* index, tf_stream_t stream);
TF_API int tf_iso_nb_triangles(const float* values, const int64_t* bricks, int64_t n_bricks, int32_t nx, int32_t ny, int32_t nz,
                               float threshold, const int32_t* slot_map, const int64_t* tri_offsets, const int32_t* index,
                               int32_t* triangles, tf_stream_t stream);

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
 * Shapes with M % 16 == 0, N % 16 == 0, both in [16, 256], and 16-byte aligned X / Y run on tcgen05 (3xTF32, fp32-level
 * accuracy); anything else on the FFMA kernel. */
TF_API int tf_xty_accumulate(const float* X, const float* Y, int64_t rows, int32_t M, int32_t N, float* out,
                             tf_stream_t stream);

#ifdef __cplusplus
}
#endif
#endif /* TENSOFLOW_B200_H */
