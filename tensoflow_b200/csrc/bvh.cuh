// Triangle-mesh BVH shared by the stand-alone tracer (bvh.cu) and the fused MC kernels.
#pragma once
#include "common.cuh"

struct __align__(16) BvhNode {
    float bmin[3];
    int first;     // inner: index of the left child (right = first+1); leaf: first triangle
    float bmax[3];
    int count;     // 0 = inner node, >0 = number of triangles in the leaf
};

struct __align__(16) BvhTri {
    float v0[3]; float pad0;
    float e1[3]; float pad1;
    float e2[3]; float pad2;
};

struct tf_bvh {
    BvhNode* nodes;
    BvhTri* tris;
    int32_t* perm;   // perm[slot] = the caller's index of the triangle stored at tris[slot] (the build reorders them)
    int n_nodes, n_tris;
    int device;
};

// BVH build rule shared by the host build (bvh.cu) and the device build (bvh_build.cu): ranges split at lo + cnt/2 until
// cnt <= TF_BVH_LEAF; values are compared and reduced with -0 mapped to +0.
constexpr int TF_BVH_LEAF = 4;
__host__ __device__ __forceinline__ float bvh_canon_zero(float x) { return x == 0.f ? 0.f : x; }

struct BvhView {
    const BvhNode* nodes;
    const BvhTri* tris;
};

constexpr float TF_MISS_DEPTH = 10.0f;   // miss sentinel (reference materialRenderer.py:261: depth >= 10)

// closest hit along o + t d, t > 0.  Returns triangle index (-1 = miss) and t.
__device__ __forceinline__ int bvh_closest_hit(const BvhView& b, const float o[3], const float d[3], float& t_hit) {
    const float inv[3] = {1.f / (d[0] != 0.f ? d[0] : 1e-20f), 1.f / (d[1] != 0.f ? d[1] : 1e-20f), 1.f / (d[2] != 0.f ? d[2] : 1e-20f)};
    int stack[64];
    int sp = 0;
    int node = 0;
    int best = -1;
    float tbest = 3.0e38f;
    while (true) {
        const float4 n0 = __ldg(reinterpret_cast<const float4*>(b.nodes + node));
        const float4 n1 = __ldg(reinterpret_cast<const float4*>(b.nodes + node) + 1);
        // slab test
        float t0x = (n0.x - o[0]) * inv[0], t1x = (n1.x - o[0]) * inv[0];
        float t0y = (n0.y - o[1]) * inv[1], t1y = (n1.y - o[1]) * inv[1];
        float t0z = (n0.z - o[2]) * inv[2], t1z = (n1.z - o[2]) * inv[2];
        const float tn = fmaxf(fmaxf(fminf(t0x, t1x), fminf(t0y, t1y)), fmaxf(fminf(t0z, t1z), 0.f));
        const float tf = fminf(fminf(fmaxf(t0x, t1x), fmaxf(t0y, t1y)), fminf(fmaxf(t0z, t1z), tbest));
        bool descend = false;
        if (tn <= tf) {
            const int first = __float_as_int(n0.w), count = __float_as_int(n1.w);
            if (count > 0) {
                for (int k = 0; k < count; ++k) {
                    const float4* tp = reinterpret_cast<const float4*>(b.tris + first + k);
                    const float4 v0 = __ldg(tp), e1 = __ldg(tp + 1), e2 = __ldg(tp + 2);
                    // Moeller-Trumbore, two sided
                    const float px = d[1] * e2.z - d[2] * e2.y, py = d[2] * e2.x - d[0] * e2.z, pz = d[0] * e2.y - d[1] * e2.x;
                    const float det = e1.x * px + e1.y * py + e1.z * pz;
                    if (fabsf(det) < 1e-12f) continue;
                    const float idet = 1.f / det;
                    const float sx = o[0] - v0.x, sy = o[1] - v0.y, sz = o[2] - v0.z;
                    const float u = (sx * px + sy * py + sz * pz) * idet;
                    if (u < 0.f || u > 1.f) continue;
                    const float qx = sy * e1.z - sz * e1.y, qy = sz * e1.x - sx * e1.z, qz = sx * e1.y - sy * e1.x;
                    const float v = (d[0] * qx + d[1] * qy + d[2] * qz) * idet;
                    if (v < 0.f || u + v > 1.f) continue;
                    const float t = (e2.x * qx + e2.y * qy + e2.z * qz) * idet;
                    if (t > 0.f && t < tbest) { tbest = t; best = first + k; }
                }
            } else {
                // push the far child, continue with the near one (ordered by split-axis direction is
                // approximated by box entry distance of the children on the next iterations)
                if (sp < 63) stack[sp++] = first + 1;
                node = first;
                descend = true;
            }
        }
        if (!descend) {
            if (sp == 0) break;
            node = stack[--sp];
        }
    }
    t_hit = tbest;
    return best;
}
