// Connected components of a triangle mesh: the graph whose nodes are the vertices and whose edges are the triangles' edges.
// Lock-free union-find in the style of ECL-CC (Jaiganesh and Burtscher, "A High-Performance Connected Components
// Implementation for GPUs", HPDC 2018): init, link (a thread per triangle), flatten, count.
//
// root[] is the parent array; the find / unite rules and why they need no locks are in union_find.cuh.  The final root of a
// component is its minimum vertex index whatever the scheduling.
//
// HBM per vertex: init writes root and tri_count (8 B), flatten reads and writes root (8 B); per triangle: link reads 12 B of
// indices plus the parent loads of two unions, count reads 4 B of index and one gathered root (then one atomic per warp and
// component).  The parent array is 4 B per vertex (128 MB at 32 M vertices), so the finds of the link pass hit L2 when it fits.
#include <algorithm>
#include "common.cuh"
#include "union_find.cuh"

namespace {

constexpr unsigned FULL = 0xffffffffu;

using tf_uf::find;
using tf_uf::set_parent;
using tf_uf::unite;

__global__ void __launch_bounds__(256) mesh_cc_init(int32_t* __restrict__ root, int32_t* __restrict__ tri_count, int64_t n_vertices) {
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (int64_t v = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; v < n_vertices; v += stride) {
        root[v] = (int32_t)v;
        tri_count[v] = 0;
    }
}

__global__ void __launch_bounds__(256) mesh_cc_link(const int32_t* __restrict__ tris, int64_t n_tris, int32_t* root) {
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (int64_t t = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; t < n_tris; t += stride) {
        const int32_t a = __ldg(tris + 3 * t), b = __ldg(tris + 3 * t + 1), c = __ldg(tris + 3 * t + 2);
        unite(root, a, b);
        unite(root, a, c);
    }
}

// the root a vertex gets is the smallest vertex of its tree, so this store never raises a parent either
__global__ void __launch_bounds__(256) mesh_cc_flatten(int32_t* root, int64_t n_vertices) {
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (int64_t v = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; v < n_vertices; v += stride)
        set_parent(root, (int32_t)v, find(root, (int32_t)v));
}

// A warp adds once per distinct root among its 32 triangles (consecutive triangles of a mesh mostly share one).  The loop
// runs while the warp's first triangle is in range, so all 32 lanes take part in every match.
__global__ void __launch_bounds__(256) mesh_cc_count(const int32_t* __restrict__ tris, int64_t n_tris, const int32_t* __restrict__ root,
                                                int32_t* __restrict__ tri_count) {
    const int lane = threadIdx.x & 31;
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (int64_t t = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; t - lane < n_tris; t += stride) {
        const bool valid = t < n_tris;
        const int32_t r = valid ? __ldg(root + __ldg(tris + 3 * t)) : -1;
        const unsigned peers = __match_any_sync(FULL, r);
        if (valid && lane == __ffs(peers) - 1) atomicAdd(tri_count + r, __popc(peers));
    }
}

unsigned grid_for(int64_t n) {
    const int64_t cap = (int64_t)tf_num_sms() * 8;          // 8 blocks of 256 threads fill an SM's 2048 threads
    return (unsigned)std::max<int64_t>(1, std::min<int64_t>((n + 255) / 256, cap));
}

}  // namespace

extern "C" TF_API int tf_mesh_components(const int32_t* triangles, int64_t n_tris, int64_t n_vertices, int32_t* root,
                                         int32_t* tri_count, tf_stream_t stream) {
    TF_REQUIRE(root && tri_count && (triangles || n_tris == 0), "tf_mesh_components: NULL pointer");
    TF_REQUIRE(n_vertices > 0 && n_vertices < (int64_t(1) << 31), "tf_mesh_components: %lld vertices, need 0 < V < 2^31",
               (long long)n_vertices);
    TF_REQUIRE(n_tris >= 0 && n_tris < (int64_t(1) << 31), "tf_mesh_components: %lld triangles, need 0 <= T < 2^31",
               (long long)n_tris);
    const cudaStream_t s = (cudaStream_t)stream;
    mesh_cc_init<<<grid_for(n_vertices), 256, 0, s>>>(root, tri_count, n_vertices);
    int launches = 1;
    if (n_tris > 0) {
        mesh_cc_link<<<grid_for(n_tris), 256, 0, s>>>(triangles, n_tris, root);
        mesh_cc_flatten<<<grid_for(n_vertices), 256, 0, s>>>(root, n_vertices);
        mesh_cc_count<<<grid_for(n_tris), 256, 0, s>>>(triangles, n_tris, root, tri_count);
        launches += 3;
    }
    tf_count_launches(launches);
    TF_CHECK_LAUNCH("tf_mesh_components");
    return 0;
}
