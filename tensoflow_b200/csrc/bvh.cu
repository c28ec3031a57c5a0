// BVH build (host) + closest-hit trace (device): replaces the un-vendored `_raytracing`
// extension behind raytracing/raytracer.py:8-54 (create_raytracer / RayTracer.trace).
// The host build is the reference of the device build in bvh_build.cu: both give the same nodes, triangles and perm.
#include <algorithm>
#include <cmath>
#include <vector>
#include "bvh.cuh"
#include "internal.cuh"

namespace {

struct BuildTri {
    float c[3];
    float lo[3], hi[3];
    int idx;
};

void build_bvh(const float* verts, const int32_t* tris, int64_t nt, std::vector<BvhNode>& nodes, std::vector<BvhTri>& out_tris,
               std::vector<int32_t>& perm) {
    std::vector<BuildTri> bt((size_t)nt);
    for (int64_t i = 0; i < nt; ++i) {
        const float* a = verts + 3 * (int64_t)tris[3 * i + 0];
        const float* b = verts + 3 * (int64_t)tris[3 * i + 1];
        const float* c = verts + 3 * (int64_t)tris[3 * i + 2];
        // -0 becomes +0 here, so that the min / max below and the split order do not depend on the visiting order
        for (int k = 0; k < 3; ++k) {
            bt[i].lo[k] = bvh_canon_zero(std::min(a[k], std::min(b[k], c[k])));
            bt[i].hi[k] = bvh_canon_zero(std::max(a[k], std::max(b[k], c[k])));
            bt[i].c[k] = bvh_canon_zero((a[k] + b[k] + c[k]) * (1.f / 3.f));
        }
        bt[i].idx = (int)i;
    }
    nodes.clear();
    nodes.reserve((size_t)nt);
    nodes.push_back(BvhNode{});
    struct Job { int node; int64_t lo, hi; };
    std::vector<Job> jobs;
    jobs.push_back({0, 0, nt});
    while (!jobs.empty()) {
        Job j = jobs.back();
        jobs.pop_back();
        float bmin[3] = {3e38f, 3e38f, 3e38f}, bmax[3] = {-3e38f, -3e38f, -3e38f};
        float cmin[3] = {3e38f, 3e38f, 3e38f}, cmax[3] = {-3e38f, -3e38f, -3e38f};
        for (int64_t i = j.lo; i < j.hi; ++i)
            for (int k = 0; k < 3; ++k) {
                bmin[k] = std::min(bmin[k], bt[i].lo[k]); bmax[k] = std::max(bmax[k], bt[i].hi[k]);
                cmin[k] = std::min(cmin[k], bt[i].c[k]);  cmax[k] = std::max(cmax[k], bt[i].c[k]);
            }
        BvhNode& n = nodes[j.node];
        for (int k = 0; k < 3; ++k) { n.bmin[k] = bmin[k]; n.bmax[k] = bmax[k]; }
        const int64_t cnt = j.hi - j.lo;
        if (cnt <= TF_BVH_LEAF) {
            n.first = (int)j.lo;
            n.count = (int)cnt;
            std::sort(bt.begin() + j.lo, bt.begin() + j.hi, [](const BuildTri& x, const BuildTri& y) { return x.idx < y.idx; });
            continue;
        }
        int ax = 0;
        if (cmax[1] - cmin[1] > cmax[ax] - cmin[ax]) ax = 1;
        if (cmax[2] - cmin[2] > cmax[ax] - cmin[ax]) ax = 2;
        const int64_t mid = j.lo + cnt / 2;
        // ties on the centroid go by caller index: the halves are then a function of the mesh alone
        std::nth_element(bt.begin() + j.lo, bt.begin() + mid, bt.begin() + j.hi, [ax](const BuildTri& x, const BuildTri& y) {
            return x.c[ax] < y.c[ax] || (x.c[ax] == y.c[ax] && x.idx < y.idx);
        });
        const int left = (int)nodes.size();
        nodes[j.node].first = left;
        nodes[j.node].count = 0;
        nodes.push_back(BvhNode{});
        nodes.push_back(BvhNode{});
        jobs.push_back({left, j.lo, mid});
        jobs.push_back({left + 1, mid, j.hi});
    }
    out_tris.resize((size_t)nt);
    perm.resize((size_t)nt);
    for (int64_t i = 0; i < nt; ++i) {
        const int t = bt[i].idx;
        perm[i] = t;
        const float* a = verts + 3 * (int64_t)tris[3 * t + 0];
        const float* b = verts + 3 * (int64_t)tris[3 * t + 1];
        const float* c = verts + 3 * (int64_t)tris[3 * t + 2];
        BvhTri& o = out_tris[i];
        for (int k = 0; k < 3; ++k) { o.v0[k] = a[k]; o.e1[k] = b[k] - a[k]; o.e2[k] = c[k] - a[k]; }
        o.pad0 = o.pad1 = o.pad2 = 0.f;
    }
}

__global__ void __launch_bounds__(128) bvh_trace_kernel(BvhView b, const float* __restrict__ ro, const float* __restrict__ rd, int64_t n,
                                                        float* __restrict__ pos, float* __restrict__ nrm, float* __restrict__ depth) {
    const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (i >= n) return;
    const float o[3] = {ro[i * 3], ro[i * 3 + 1], ro[i * 3 + 2]};
    const float d[3] = {rd[i * 3], rd[i * 3 + 1], rd[i * 3 + 2]};
    float t;
    const int tri = bvh_closest_hit(b, o, d, t);
    float nx = 0.f, ny = 0.f, nz = 0.f;
    if (tri >= 0) {
        const BvhTri& T = b.tris[tri];
        nx = T.e1[1] * T.e2[2] - T.e1[2] * T.e2[1];
        ny = T.e1[2] * T.e2[0] - T.e1[0] * T.e2[2];
        nz = T.e1[0] * T.e2[1] - T.e1[1] * T.e2[0];
        const float il = rsqrtf(fmaxf(nx * nx + ny * ny + nz * nz, 1e-30f));
        nx *= il; ny *= il; nz *= il;
    } else {
        t = TF_MISS_DEPTH;
    }
    depth[i] = t;
    pos[i * 3 + 0] = o[0] + t * d[0]; pos[i * 3 + 1] = o[1] + t * d[1]; pos[i * 3 + 2] = o[2] + t * d[2];
    nrm[i * 3 + 0] = nx; nrm[i * 3 + 1] = ny; nrm[i * 3 + 2] = nz;
}

}  // namespace

tf_bvh* tf_internal_bvh_alloc(int64_t n_nodes, int64_t n_tris, const char* who) {
    tf_bvh* h = new tf_bvh();
    h->n_nodes = (int)n_nodes;
    h->n_tris = (int)n_tris;
    cudaGetDevice(&h->device);
    cudaError_t e1 = cudaMalloc(&h->nodes, n_nodes * sizeof(BvhNode));
    cudaError_t e2 = cudaMalloc(&h->tris, n_tris * sizeof(BvhTri));
    cudaError_t e3 = cudaMalloc(&h->perm, n_tris * sizeof(int32_t));
    if (e1 != cudaSuccess || e2 != cudaSuccess || e3 != cudaSuccess) {
        tf_set_error("%s: cudaMalloc failed", who);
        if (e1 == cudaSuccess) cudaFree(h->nodes);
        if (e2 == cudaSuccess) cudaFree(h->tris);
        if (e3 == cudaSuccess) cudaFree(h->perm);
        delete h;
        return nullptr;
    }
    return h;
}

extern "C" TF_API int tf_bvh_create(const float* vertices_host, int64_t n_vertices, const int32_t* triangles_host, int64_t n_triangles,
                                    tf_bvh_t** out) {
    TF_REQUIRE(vertices_host && triangles_host && out, "tf_bvh_create: NULL pointer");
    TF_REQUIRE(n_triangles > 0 && n_vertices > 0, "tf_bvh_create: empty mesh");
    TF_REQUIRE(n_triangles < (int64_t(1) << 31), "tf_bvh_create: %lld triangles, the BVH holds fewer than 2^31", (long long)n_triangles);
    for (int64_t i = 0; i < 3 * n_triangles; ++i)
        TF_REQUIRE(triangles_host[i] >= 0 && triangles_host[i] < n_vertices, "tf_bvh_create: triangle index out of range");
    for (int64_t i = 0; i < 3 * n_triangles; ++i) {
        const float* p = vertices_host + 3 * (int64_t)triangles_host[i];
        TF_REQUIRE(std::isfinite(p[0]) && std::isfinite(p[1]) && std::isfinite(p[2]), "tf_bvh_create: non-finite vertex coordinate");
    }
    std::vector<BvhNode> nodes;
    std::vector<BvhTri> tris;
    std::vector<int32_t> perm;
    build_bvh(vertices_host, triangles_host, n_triangles, nodes, tris, perm);
    tf_bvh* h = tf_internal_bvh_alloc((int64_t)nodes.size(), (int64_t)tris.size(), "tf_bvh_create");
    if (!h) return 2;
    cudaMemcpy(h->nodes, nodes.data(), nodes.size() * sizeof(BvhNode), cudaMemcpyHostToDevice);
    cudaMemcpy(h->tris, tris.data(), tris.size() * sizeof(BvhTri), cudaMemcpyHostToDevice);
    cudaMemcpy(h->perm, perm.data(), perm.size() * sizeof(int32_t), cudaMemcpyHostToDevice);
    *out = reinterpret_cast<tf_bvh_t*>(h);
    return 0;
}

extern "C" TF_API int tf_bvh_create_from_device(const void* nodes, int64_t n_nodes, const void* tris, const int32_t* perm,
                                                int64_t n_triangles, tf_stream_t stream, tf_bvh_t** out) {
    TF_REQUIRE(nodes && tris && perm && out, "tf_bvh_create_from_device: NULL pointer");
    TF_REQUIRE(n_triangles > 0 && n_nodes > 0, "tf_bvh_create_from_device: empty BVH");
    TF_REQUIRE(n_triangles < (int64_t(1) << 31) && n_nodes < (int64_t(1) << 31), "tf_bvh_create_from_device: BVH too large");
    tf_bvh* h = tf_internal_bvh_alloc(n_nodes, n_triangles, "tf_bvh_create_from_device");
    if (!h) return 2;
    const cudaStream_t s = (cudaStream_t)stream;
    cudaError_t e = cudaMemcpyAsync(h->nodes, nodes, n_nodes * sizeof(BvhNode), cudaMemcpyDeviceToDevice, s);
    if (e == cudaSuccess) e = cudaMemcpyAsync(h->tris, tris, n_triangles * sizeof(BvhTri), cudaMemcpyDeviceToDevice, s);
    if (e == cudaSuccess) e = cudaMemcpyAsync(h->perm, perm, n_triangles * sizeof(int32_t), cudaMemcpyDeviceToDevice, s);
    if (e != cudaSuccess) {
        tf_bvh_destroy(reinterpret_cast<tf_bvh_t*>(h));
        tf_set_error("tf_bvh_create_from_device: copy failed: %s", cudaGetErrorString(e));
        return 2;
    }
    *out = reinterpret_cast<tf_bvh_t*>(h);
    return 0;
}

extern "C" TF_API void tf_bvh_destroy(tf_bvh_t* handle) {
    tf_bvh* h = reinterpret_cast<tf_bvh*>(handle);
    if (!h) return;
    cudaFree(h->nodes);
    cudaFree(h->tris);
    cudaFree(h->perm);
    delete h;
}

extern "C" TF_API int tf_bvh_export(const tf_bvh_t* handle, int64_t* n_nodes, int64_t* n_triangles, void* nodes, void* tris,
                                    int32_t* perm) {
    const tf_bvh* h = reinterpret_cast<const tf_bvh*>(handle);
    TF_REQUIRE(h, "tf_bvh_export: NULL handle");
    if (n_nodes) *n_nodes = h->n_nodes;
    if (n_triangles) *n_triangles = h->n_tris;
    int prev = 0;
    cudaGetDevice(&prev);
    cudaSetDevice(h->device);
    // the handle may have been filled by copies on a caller's (possibly non-blocking) stream: wait for all work on its device
    cudaError_t e = cudaDeviceSynchronize();
    if (nodes && e == cudaSuccess) e = cudaMemcpy(nodes, h->nodes, (size_t)h->n_nodes * sizeof(BvhNode), cudaMemcpyDefault);
    if (tris && e == cudaSuccess) e = cudaMemcpy(tris, h->tris, (size_t)h->n_tris * sizeof(BvhTri), cudaMemcpyDefault);
    if (perm && e == cudaSuccess) e = cudaMemcpy(perm, h->perm, (size_t)h->n_tris * sizeof(int32_t), cudaMemcpyDefault);
    cudaSetDevice(prev);
    TF_REQUIRE(e == cudaSuccess, "tf_bvh_export: copy failed: %s", cudaGetErrorString(e));
    return 0;
}

extern "C" TF_API int tf_bvh_trace(const tf_bvh_t* handle, const float* rays_o, const float* rays_d, int64_t n, float* positions,
                                   float* face_normals, float* depth, tf_stream_t stream) {
    const tf_bvh* h = reinterpret_cast<const tf_bvh*>(handle);
    TF_REQUIRE(h, "tf_bvh_trace: NULL handle");
    if (n == 0) return 0;
    TF_REQUIRE(rays_o && rays_d && positions && face_normals && depth, "tf_bvh_trace: NULL pointer");
    BvhView v{h->nodes, h->tris};
    bvh_trace_kernel<<<(unsigned)((n + 127) / 128), 128, 0, (cudaStream_t)stream>>>(v, rays_o, rays_d, n, positions, face_normals, depth);
    tf_count_launches(1);
    TF_CHECK_LAUNCH("tf_bvh_trace");
    return 0;
}
