// Geometry evaluation queries on a triangle mesh: closest point on the mesh (branch-and-bound over the BVH of bvh.cu) and
// area-weighted surface sampling.
#include <climits>
#include "bvh.cuh"

namespace {

__device__ __forceinline__ float3 sub3(float3 a, float3 b) { return make_float3(a.x - b.x, a.y - b.y, a.z - b.z); }
__device__ __forceinline__ float3 axpy3(float s, float3 x, float3 y) { return make_float3(y.x - s * x.x, y.y - s * x.y, y.z - s * x.z); }
__device__ __forceinline__ float dot3(float3 a, float3 b) { return a.x * b.x + a.y * b.y + a.z * b.z; }
__device__ __forceinline__ float3 cross3(float3 a, float3 b) {
    return make_float3(a.y * b.z - a.z * b.y, a.z * b.x - a.x * b.z, a.x * b.y - a.y * b.x);
}
// a*b - c*d with one rounding's worth of error (Kahan): the face normal of a thin triangle keeps its direction, where the
// plain difference of products loses it to cancellation
__device__ __forceinline__ float dop(float a, float b, float c, float d) {
    const float w = c * d;
    return fmaf(a, b, -w) + fmaf(-c, d, w);
}
// fmaxf returns the non-NaN operand, so 0/0 becomes 0
__device__ __forceinline__ float clamp01(float x) { return fminf(fmaxf(x, 0.f), 1.f); }

// Closest point of the triangle (v0, v0 + e1, v0 + e2) to p = v0 + ap: returns the squared distance and r = p - closest.
// The 7-region test of Ericson, Real-Time Collision Detection 5.1.5, with a = v0, ab = e1, ac = e2.  The edge-region
// discriminants are the book's triple products vc = n.(ap x bp), vb = n.(cp x ap), va = n.(bp x cp), the edge parameters
// use |e|^2 for the book's d1 - d3, d2 - d6, (d4 - d3) + (d5 - d6), and the face region takes the plane offset
// (ap.n / n.n) n: the same formula, conditioned by the distance instead of by the triangle's area.
// A triangle whose height is below 2^-24 of its longest edge (zero area, collinear, repeated vertices) is the union of its
// edges to fp32 precision and is measured as such: the nearest of the three segments, a zero-length one being its vertex.
__device__ __forceinline__ float tri_closest(const float3 ap, const float3 e1, const float3 e2, float3& r) {
    const float3 n = make_float3(dop(e1.y, e2.z, e1.z, e2.y), dop(e1.z, e2.x, e1.x, e2.z), dop(e1.x, e2.y, e1.y, e2.x));
    const float nn = dot3(n, n);
    const float3 e3 = sub3(e2, e1);
    const float l1 = dot3(e1, e1), l2 = dot3(e2, e2), l3 = dot3(e3, e3);
    const float lmax = fmaxf(l1, fmaxf(l2, l3));
    const float3 bp = sub3(ap, e1), cp = sub3(ap, e2);
    if (nn > 0x1p-48f * lmax * lmax) {
        const float d1 = dot3(e1, ap), d2 = dot3(e2, ap);
        if (d1 <= 0.f && d2 <= 0.f) { r = ap; return dot3(r, r); }                                  // vertex a
        const float d3 = dot3(e1, bp), d4 = dot3(e2, bp);
        if (d3 >= 0.f && d4 <= d3) { r = bp; return dot3(r, r); }                                   // vertex b
        const float vc = dot3(n, cross3(e1, ap));
        if (vc <= 0.f && d1 >= 0.f && d3 <= 0.f) { r = axpy3(clamp01(d1 / l1), e1, ap); return dot3(r, r); }   // edge ab
        const float d5 = dot3(e1, cp), d6 = dot3(e2, cp);
        if (d6 >= 0.f && d5 <= d6) { r = cp; return dot3(r, r); }                                   // vertex c
        const float vb = dot3(n, cross3(ap, e2));
        if (vb <= 0.f && d2 >= 0.f && d6 <= 0.f) { r = axpy3(clamp01(d2 / l2), e2, ap); return dot3(r, r); }   // edge ac
        const float va = dot3(n, cross3(bp, cp));
        if (va <= 0.f && d4 - d3 >= 0.f && d5 - d6 >= 0.f) {                                        // edge bc
            r = axpy3(clamp01(dot3(e3, bp) / l3), e3, bp);
            return dot3(r, r);
        }
        const float s = dot3(ap, n) / nn;                                                          // face
        r = make_float3(s * n.x, s * n.y, s * n.z);
        return dot3(r, r);
    }
    float3 rs = axpy3(l1 > 0.f ? clamp01(dot3(ap, e1) / l1) : 0.f, e1, ap);
    float best = dot3(rs, rs);
    r = rs;
    rs = axpy3(l2 > 0.f ? clamp01(dot3(ap, e2) / l2) : 0.f, e2, ap);
    float d = dot3(rs, rs);
    if (d < best) { best = d; r = rs; }
    rs = axpy3(l3 > 0.f ? clamp01(dot3(bp, e3) / l3) : 0.f, e3, bp);
    d = dot3(rs, rs);
    if (d < best) { best = d; r = rs; }
    return best;
}

// squared distance from p to the box of a node (0 inside)
__device__ __forceinline__ float box_d2(const float3 p, const float4 lo, const float4 hi) {
    const float dx = fmaxf(fmaxf(lo.x - p.x, p.x - hi.x), 0.f);
    const float dy = fmaxf(fmaxf(lo.y - p.y, p.y - hi.y), 0.f);
    const float dz = fmaxf(fmaxf(lo.z - p.z, p.z - hi.z), 0.f);
    return dx * dx + dy * dy + dz * dz;
}

__global__ void __launch_bounds__(128) bvh_closest_point_kernel(BvhView b, const int32_t* __restrict__ perm, const float* __restrict__ pts,
                                                                int64_t n, float* __restrict__ out_pts, float* __restrict__ out_dist,
                                                                int64_t* __restrict__ out_tri) {
    const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (i >= n) return;
    const float3 p = make_float3(pts[i * 3], pts[i * 3 + 1], pts[i * 3 + 2]);
    // Each level pushes at most one far child, and the median-split build has depth <= ceil(log2(n_tris / 4)) + 1 <= 30 for
    // int32 triangle counts, so 64 entries cannot overflow.
    int stack_node[64];
    float stack_d2[64];
    int sp = 0;
    int node = 0;
    float best = INFINITY;
    int best_tri = INT_MAX;
    float3 best_r = make_float3(0.f, 0.f, 0.f);
    while (true) {
        const float4* np = reinterpret_cast<const float4*>(b.nodes + node);
        const int first = __float_as_int(__ldg(np).w), count = __float_as_int(__ldg(np + 1).w);
        bool descend = false;
        if (count > 0) {
            for (int k = 0; k < count; ++k) {
                const float4* tp = reinterpret_cast<const float4*>(b.tris + first + k);
                const float4 v0 = __ldg(tp), e1 = __ldg(tp + 1), e2 = __ldg(tp + 2);
                float3 r;
                const float d2 = tri_closest(make_float3(p.x - v0.x, p.y - v0.y, p.z - v0.z), make_float3(e1.x, e1.y, e1.z),
                                             make_float3(e2.x, e2.y, e2.z), r);
                if (d2 <= best) {
                    const int t = __ldg(perm + first + k);
                    if (d2 < best || t < best_tri) { best = d2; best_tri = t; best_r = r; }
                }
            }
        } else {
            const float4* cp = reinterpret_cast<const float4*>(b.nodes + first);
            const float dl = box_d2(p, __ldg(cp), __ldg(cp + 1));
            const float dr = box_d2(p, __ldg(cp + 2), __ldg(cp + 3));
            const int near = dl <= dr ? first : first + 1;
            const float dn = fminf(dl, dr), df = fmaxf(dl, dr);
            // a child whose bound equals the best so far is still visited: it may hold an exactly tied triangle with a
            // smaller index
            if (dn <= best) {
                if (df <= best) { stack_node[sp] = near == first ? first + 1 : first; stack_d2[sp] = df; ++sp; }
                node = near;
                descend = true;
            }
        }
        if (!descend) {
            while (sp > 0 && stack_d2[sp - 1] > best) --sp;
            if (sp == 0) break;
            node = stack_node[--sp];
        }
    }
    out_pts[i * 3 + 0] = p.x - best_r.x;
    out_pts[i * 3 + 1] = p.y - best_r.y;
    out_pts[i * 3 + 2] = p.z - best_r.z;
    out_dist[i] = sqrtf(best);
    out_tri[i] = best_tri == INT_MAX ? -1 : best_tri;
}

__global__ void __launch_bounds__(256) mesh_sample_surface_kernel(const float* __restrict__ verts, const int32_t* __restrict__ tris, int64_t n_tris,
                                                                  const double* __restrict__ cdf, const double* __restrict__ uni, int64_t n,
                                                                  float* __restrict__ out_pts, int64_t* __restrict__ out_tri,
                                                                  float* __restrict__ out_nrm) {
    const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (i >= n) return;
    const double u0 = uni[i * 3], u1 = uni[i * 3 + 1], u2 = uni[i * 3 + 2];
    int64_t lo = 0, hi = n_tris - 1;                 // first triangle whose inclusive CDF exceeds u0
    while (lo < hi) {
        const int64_t mid = (lo + hi) >> 1;
        if (__ldg(cdf + mid) > u0) hi = mid; else lo = mid + 1;
    }
    double a[3], e1[3], e2[3];
    const float* va = verts + 3 * (int64_t)__ldg(tris + 3 * lo);
    const float* vb = verts + 3 * (int64_t)__ldg(tris + 3 * lo + 1);
    const float* vc = verts + 3 * (int64_t)__ldg(tris + 3 * lo + 2);
    for (int k = 0; k < 3; ++k) {
        a[k] = __ldg(va + k);
        e1[k] = (double)__ldg(vb + k) - a[k];
        e2[k] = (double)__ldg(vc + k) - a[k];
    }
    const double s = sqrt(u1), w1 = s * (1.0 - u2), w2 = s * u2;
    for (int k = 0; k < 3; ++k) out_pts[i * 3 + k] = (float)(a[k] + w1 * e1[k] + w2 * e2[k]);
    const double nx = e1[1] * e2[2] - e1[2] * e2[1], ny = e1[2] * e2[0] - e1[0] * e2[2], nz = e1[0] * e2[1] - e1[1] * e2[0];
    const double len = sqrt(nx * nx + ny * ny + nz * nz);
    const double il = len > 0.0 ? 1.0 / len : 0.0;
    out_nrm[i * 3 + 0] = (float)(nx * il);
    out_nrm[i * 3 + 1] = (float)(ny * il);
    out_nrm[i * 3 + 2] = (float)(nz * il);
    out_tri[i] = lo;
}

}  // namespace

extern "C" TF_API int tf_bvh_closest_point(const tf_bvh_t* handle, const float* points, int64_t n, float* out_points, float* out_dist,
                                           int64_t* out_tri, tf_stream_t stream) {
    const tf_bvh* h = reinterpret_cast<const tf_bvh*>(handle);
    TF_REQUIRE(h, "tf_bvh_closest_point: NULL handle");
    TF_REQUIRE(h->n_tris > 0 && h->perm, "tf_bvh_closest_point: empty mesh");
    if (n == 0) return 0;
    TF_REQUIRE(points && out_points && out_dist && out_tri, "tf_bvh_closest_point: NULL pointer");
    BvhView v{h->nodes, h->tris};
    bvh_closest_point_kernel<<<(unsigned)((n + 127) / 128), 128, 0, (cudaStream_t)stream>>>(v, h->perm, points, n, out_points, out_dist, out_tri);
    tf_count_launches(1);
    TF_CHECK_LAUNCH("tf_bvh_closest_point");
    return 0;
}

extern "C" TF_API int tf_mesh_sample_surface(const float* vertices, const int32_t* triangles, int64_t n_tris, const double* cdf,
                                             const double* uniforms, int64_t n, float* out_points, int64_t* out_tri, float* out_normals,
                                             tf_stream_t stream) {
    TF_REQUIRE(n_tris > 0, "tf_mesh_sample_surface: empty mesh");
    if (n == 0) return 0;
    TF_REQUIRE(vertices && triangles && cdf && uniforms && out_points && out_tri && out_normals, "tf_mesh_sample_surface: NULL pointer");
    mesh_sample_surface_kernel<<<(unsigned)((n + 255) / 256), 256, 0, (cudaStream_t)stream>>>(vertices, triangles, n_tris, cdf, uniforms, n,
                                                                                             out_points, out_tri, out_normals);
    tf_count_launches(1);
    TF_CHECK_LAUNCH("tf_mesh_sample_surface");
    return 0;
}
