// BVH build on the device: node for node, triangle for triangle the tree of the host build in bvh.cu (build_bvh).
//
// The host build is a top-down median split.  A range [lo, lo + cnt) with cnt > TF_BVH_LEAF splits at lo + cnt/2 on the axis
// of largest fp32 centroid extent (ties prefer x, then y); the left half holds the cnt/2 smallest triangles by (centroid on
// that axis, caller index); a leaf lists its triangles by caller index.  The k-th inner node in right-first preorder (the host's
// LIFO job stack) has its children at 1 + 2k (left) and 2 + 2k (right).  So ranges, topology and numbering depend on n alone,
// and only the split axis and the membership of each half depend on the data.
//
// Here the build runs level by level over the slot order (slot i = position in the final triangle array):
//   reduce  per node of the level: min / max of the triangle boxes and centroids (canonical values, so atomics are exact);
//   split   per slot: the axis of its node, the key (node's lo, orderable centroid bits) written at the caller index, and the
//           node the slot belongs to on the next level (the first slot of each child writes the child's range and rank);
//   sort    a stable CUB radix sort of the keys with the caller indices as values: ties go by caller index, and leaves (key
//           (lo, 0)) stay sorted by caller index.
// After the last level each leaf is put in caller-index order, the nodes are written from the reductions, and the triangles
// (v0, e1 = b - a, e2 = c - a) and perm from the final slot order.
//
// Per level and triangle: a gathered 36 B record and one gathered centroid, 8 B of order and 12 B of node id read or written,
// 12 B of key and value scattered, and one radix sort of (32 + bit width of n - 1)-bit keys with 4-byte values.
#include <cub/device/device_radix_sort.cuh>
#include <map>
#include "bvh.cuh"

namespace {

constexpr int MAX_LEVELS = 32;        // depth <= ceil(log2(ceil(n / 4))) + 1 <= 30 for n < 2^31
constexpr int RED_TILES = 16;         // slots per warp in the reduction: 32 * RED_TILES
constexpr unsigned FULL = 0xffffffffu;

struct BuildRec {
    float c[3], lo[3], hi[3];
};

// inner-node counts of subtrees: at depth d the ranges have size[d] = floor(n / 2^d) or size[d] + 1 triangles
struct LevelTab {
    int32_t size[MAX_LEVELS];
    int32_t inner[MAX_LEVELS][2];
};

int64_t inner_count(int64_t m, std::map<int64_t, int64_t>& memo) {
    if (m <= TF_BVH_LEAF) return 0;
    auto it = memo.find(m);
    if (it != memo.end()) return it->second;
    const int64_t v = 1 + inner_count(m / 2, memo) + inner_count(m - m / 2, memo);
    memo[m] = v;
    return v;
}

struct Plan {
    LevelTab tab;
    int levels;            // levels that split: depths 0 .. levels-1
    int64_t n_nodes;
    int end_bit;           // key bits: lo << 32 | centroid
};

Plan make_plan(int64_t n) {
    Plan p{};
    std::map<int64_t, int64_t> memo;
    for (int d = 0; d < MAX_LEVELS; ++d) {
        const int64_t s = n >> d;
        p.tab.size[d] = (int32_t)s;
        p.tab.inner[d][0] = (int32_t)inner_count(s, memo);
        p.tab.inner[d][1] = (int32_t)inner_count(s + 1, memo);
    }
    p.levels = 0;
    while (((n + (int64_t(1) << p.levels) - 1) >> p.levels) > TF_BVH_LEAF) ++p.levels;
    p.n_nodes = 1 + 2 * inner_count(n, memo);
    int bits = 1;
    while ((int64_t(1) << bits) < n) ++bits;
    p.end_bit = 32 + bits;
    return p;
}

// orderable encoding: unsigned order of the codes = float order (no NaN here)
__device__ __forceinline__ uint32_t ord_bits(float x) {
    const uint32_t u = __float_as_uint(x);
    return u ^ ((u >> 31) ? 0xffffffffu : 0x80000000u);
}
__device__ __forceinline__ float ord_float(uint32_t u) { return __uint_as_float(u ^ ((u >> 31) ? 0x80000000u : 0xffffffffu)); }

// acc[12 * node]: box min (3), ~box max (3), centroid min (3), ~centroid max (3), all reduced with atomicMin from 0xffffffff
__device__ __forceinline__ void rec_codes(const BuildRec& r, uint32_t e[12]) {
#pragma unroll
    for (int k = 0; k < 3; ++k) {
        e[k] = ord_bits(r.lo[k]);
        e[3 + k] = ~ord_bits(r.hi[k]);
        e[6 + k] = ord_bits(r.c[k]);
        e[9 + k] = ~ord_bits(r.c[k]);
    }
}

// the host's reductions start from +-3e38
__device__ __forceinline__ float acc_min(const uint32_t* a, int k) { return fminf(ord_float(a[k]), 3e38f); }
__device__ __forceinline__ float acc_max(const uint32_t* a, int k) { return fmaxf(ord_float(~a[k]), -3e38f); }

__global__ void __launch_bounds__(256) bvh_build_prep(const float* __restrict__ verts, const int32_t* __restrict__ tris, int n,
                                                      BuildRec* __restrict__ rec, int32_t* __restrict__ order, int32_t* __restrict__ nid,
                                                      int32_t* __restrict__ node_lo, int32_t* __restrict__ node_cnt,
                                                      int32_t* __restrict__ node_rank) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const float* a = verts + 3 * (int64_t)tris[3 * (int64_t)i + 0];
    const float* b = verts + 3 * (int64_t)tris[3 * (int64_t)i + 1];
    const float* c = verts + 3 * (int64_t)tris[3 * (int64_t)i + 2];
    BuildRec r;
#pragma unroll
    for (int k = 0; k < 3; ++k) {
        const float x = a[k], y = b[k], z = c[k];
        r.lo[k] = bvh_canon_zero(fminf(x, fminf(y, z)));
        r.hi[k] = bvh_canon_zero(fmaxf(x, fmaxf(y, z)));
        r.c[k] = bvh_canon_zero(__fmul_rn(__fadd_rn(__fadd_rn(x, y), z), 1.f / 3.f));   // the host's ((a + b) + c) * (1/3)
    }
    rec[i] = r;
    order[i] = i;
    nid[i] = 0;
    if (i == 0) {
        node_lo[0] = 0;
        node_cnt[0] = n;
        node_rank[0] = n > TF_BVH_LEAF ? 0 : -1;
    }
}

// Per node of the level: min / max of the records of its slots.  A warp takes 32 * RED_TILES consecutive slots; when they all
// belong to one node (upper levels) it reduces them in registers and issues 12 atomics, otherwise it runs a segmented reduction
// per 32 slots (a node's slots are contiguous) and the first lane of each node's run issues them.
__global__ void __launch_bounds__(256, 4) bvh_build_reduce(const BuildRec* __restrict__ rec, const int32_t* __restrict__ order,
                                                        const int32_t* __restrict__ nid, int n, uint32_t* __restrict__ acc) {
    const int lane = threadIdx.x & 31;
    const int64_t base = ((blockIdx.x * (int64_t)blockDim.x + threadIdx.x) >> 5) * (32 * RED_TILES);
    if (base >= n) return;
    const int64_t last = min(base + 32 * RED_TILES, (int64_t)n) - 1;
    const int node0 = nid[base];
    if (nid[last] == node0) {
        uint32_t v[12];
#pragma unroll
        for (int k = 0; k < 12; ++k) v[k] = FULL;
        for (int64_t i = base + lane; i <= last; i += 32) {
            uint32_t e[12];
            rec_codes(rec[order[i]], e);
#pragma unroll
            for (int k = 0; k < 12; ++k) v[k] = min(v[k], e[k]);
        }
#pragma unroll
        for (int off = 16; off > 0; off >>= 1)
#pragma unroll
            for (int k = 0; k < 12; ++k) v[k] = min(v[k], __shfl_xor_sync(FULL, v[k], off));
        if (lane < 12) {
            uint32_t mine = v[0];
#pragma unroll
            for (int k = 1; k < 12; ++k) if (lane == k) mine = v[k];
            atomicMin(acc + 12 * (int64_t)node0 + lane, mine);
        }
        return;
    }
    for (int64_t t0 = base; t0 <= last; t0 += 32) {
        const int64_t i = t0 + lane;
        const bool valid = i <= last;
        const int node = valid ? nid[i] : -1;
        uint32_t e[12];
        if (valid) {
            rec_codes(rec[order[i]], e);
        } else {
#pragma unroll
            for (int k = 0; k < 12; ++k) e[k] = FULL;
        }
        // after the step with offset `off`, lane l holds the minimum over [l, l + 2 off) cut to its node's run
#pragma unroll
        for (int off = 1; off < 32; off <<= 1) {
            const int nb = __shfl_down_sync(FULL, node, off);
            const bool take = lane + off < 32 && nb == node;
#pragma unroll
            for (int k = 0; k < 12; ++k) {
                const uint32_t o = __shfl_down_sync(FULL, e[k], off);
                if (take) e[k] = min(e[k], o);
            }
        }
        const int prev = __shfl_up_sync(FULL, node, 1);
        if (valid && (lane == 0 || prev != node)) {
            uint32_t* a = acc + 12 * (int64_t)node;
#pragma unroll
            for (int k = 0; k < 12; ++k) atomicMin(a + k, e[k]);
        }
    }
}

__device__ __forceinline__ int32_t inner_of(const LevelTab& tab, int d, int32_t m) {
    return m == tab.size[d] ? tab.inner[d][0] : tab.inner[d][1];
}

// Slot i of a node at depth `level`: key (lo, centroid bits on the node's split axis; 0 in a leaf) at the caller index, and the
// node of slot i on the next level.
__global__ void __launch_bounds__(256) bvh_build_split(const BuildRec* __restrict__ rec, const int32_t* __restrict__ order,
                                                       int32_t* __restrict__ nid, int n, const uint32_t* __restrict__ acc,
                                                       int32_t* __restrict__ node_lo, int32_t* __restrict__ node_cnt,
                                                       int32_t* __restrict__ node_rank, const LevelTab tab, int level,
                                                       uint64_t* __restrict__ keys, int32_t* __restrict__ vals) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const int node = nid[i];
    const int t = order[i];
    const int32_t lo = node_lo[node], cnt = node_cnt[node];
    uint32_t cb = 0;
    if (cnt > TF_BVH_LEAF) {
        const uint32_t* a = acc + 12 * (int64_t)node;
        const float ex = __fsub_rn(acc_max(a, 9), acc_min(a, 6));
        const float ey = __fsub_rn(acc_max(a, 10), acc_min(a, 7));
        const float ez = __fsub_rn(acc_max(a, 11), acc_min(a, 8));
        int ax = 0;
        float best = ex;
        if (ey > best) { ax = 1; best = ey; }
        if (ez > best) ax = 2;
        cb = ord_bits(rec[t].c[ax]);
        const int32_t half = cnt / 2, mid = lo + half, k = node_rank[node];
        int32_t child, clo, ccnt, crank;
        if (i < mid) {
            child = 1 + 2 * k; clo = lo; ccnt = half; crank = k + 1 + inner_of(tab, level + 1, cnt - half);
        } else {
            child = 2 + 2 * k; clo = mid; ccnt = cnt - half; crank = k + 1;
        }
        nid[i] = child;
        if (i == clo) {
            node_lo[child] = clo;
            node_cnt[child] = ccnt;
            node_rank[child] = ccnt > TF_BVH_LEAF ? crank : -1;
        }
    }
    keys[t] = ((uint64_t)(uint32_t)lo << 32) | cb;
    vals[t] = t;
}

// Node j from its range and reductions; a leaf's slots are put in caller-index order.
__global__ void __launch_bounds__(256) bvh_build_nodes(const uint32_t* __restrict__ acc, const int32_t* __restrict__ node_lo,
                                                       const int32_t* __restrict__ node_cnt, const int32_t* __restrict__ node_rank,
                                                       int n_nodes, int32_t* __restrict__ order, BvhNode* __restrict__ nodes) {
    const int j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= n_nodes) return;
    const uint32_t* a = acc + 12 * (int64_t)j;
    const int32_t lo = node_lo[j], cnt = node_cnt[j], rank = node_rank[j];
    float4 n0, n1;
    n0.x = acc_min(a, 0); n0.y = acc_min(a, 1); n0.z = acc_min(a, 2);
    n1.x = acc_max(a, 3); n1.y = acc_max(a, 4); n1.z = acc_max(a, 5);
    if (rank >= 0) {
        n0.w = __int_as_float(1 + 2 * rank);
        n1.w = __int_as_float(0);
    } else {
        n0.w = __int_as_float(lo);
        n1.w = __int_as_float(cnt);
        static_assert(TF_BVH_LEAF == 4, "the sorting network below orders 4 slots");
        int32_t s[4];
#pragma unroll
        for (int q = 0; q < 4; ++q) s[q] = q < cnt ? order[lo + q] : INT32_MAX;
        auto cswap = [&](int x, int y) { const int32_t l = min(s[x], s[y]), h = max(s[x], s[y]); s[x] = l; s[y] = h; };
        cswap(0, 1); cswap(2, 3); cswap(0, 2); cswap(1, 3); cswap(1, 2);
#pragma unroll
        for (int q = 0; q < 4; ++q) if (q < cnt) order[lo + q] = s[q];
    }
    float4* o = reinterpret_cast<float4*>(nodes + j);
    o[0] = n0;
    o[1] = n1;
}

__global__ void __launch_bounds__(256) bvh_build_tris(const float* __restrict__ verts, const int32_t* __restrict__ tris,
                                                      const int32_t* __restrict__ order, int n, BvhTri* __restrict__ out,
                                                      int32_t* __restrict__ perm) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const int t = order[i];
    perm[i] = t;
    const float* a = verts + 3 * (int64_t)tris[3 * (int64_t)t + 0];
    const float* b = verts + 3 * (int64_t)tris[3 * (int64_t)t + 1];
    const float* c = verts + 3 * (int64_t)tris[3 * (int64_t)t + 2];
    float4* o = reinterpret_cast<float4*>(out + i);
    o[0] = make_float4(a[0], a[1], a[2], 0.f);
    o[1] = make_float4(__fsub_rn(b[0], a[0]), __fsub_rn(b[1], a[1]), __fsub_rn(b[2], a[2]), 0.f);
    o[2] = make_float4(__fsub_rn(c[0], a[0]), __fsub_rn(c[1], a[1]), __fsub_rn(c[2], a[2]), 0.f);
}

constexpr size_t ALIGN = 256;
size_t up(size_t b) { return (b + ALIGN - 1) / ALIGN * ALIGN; }

struct Layout {
    size_t rec, keys0, keys1, ord0, ord1, nid, node_lo, node_cnt, node_rank, acc, sort, sort_bytes, total;
};

// scratch layout of the workspace for n triangles; sort_bytes from CUB on the current device
int make_layout(int64_t n, const Plan& p, Layout& L, const char* who) {
    cub::DoubleBuffer<uint64_t> kb(nullptr, nullptr);
    cub::DoubleBuffer<int32_t> vb(nullptr, nullptr);
    size_t sort_bytes = 0;
    const cudaError_t e = cub::DeviceRadixSort::SortPairs(nullptr, sort_bytes, kb, vb, (int)n, 0, p.end_bit);
    TF_REQUIRE(e == cudaSuccess, "%s: radix sort sizing failed: %s", who, cudaGetErrorString(e));
    size_t off = 0;
    auto take = [&](size_t bytes) { const size_t o = off; off += up(bytes); return o; };
    L.rec = take(n * sizeof(BuildRec));
    L.keys0 = take(n * sizeof(uint64_t));
    L.keys1 = take(n * sizeof(uint64_t));
    L.ord0 = take(n * sizeof(int32_t));
    L.ord1 = take(n * sizeof(int32_t));
    L.nid = take(n * sizeof(int32_t));
    L.node_lo = take(p.n_nodes * sizeof(int32_t));
    L.node_cnt = take(p.n_nodes * sizeof(int32_t));
    L.node_rank = take(p.n_nodes * sizeof(int32_t));
    L.acc = take(p.n_nodes * 12 * sizeof(uint32_t));
    L.sort_bytes = sort_bytes;
    L.sort = take(sort_bytes);
    L.total = off;
    return 0;
}

}  // namespace

extern "C" TF_API int tf_bvh_build_sizes(int64_t n_triangles, int64_t* n_nodes, size_t* workspace_bytes) {
    TF_REQUIRE(n_nodes && workspace_bytes, "tf_bvh_build_sizes: NULL pointer");
    TF_REQUIRE(n_triangles > 0, "tf_bvh_build_sizes: empty mesh");
    TF_REQUIRE(n_triangles < (int64_t(1) << 31), "tf_bvh_build_sizes: %lld triangles, the BVH holds fewer than 2^31",
               (long long)n_triangles);
    const Plan p = make_plan(n_triangles);
    Layout L;
    if (make_layout(n_triangles, p, L, "tf_bvh_build_sizes")) return 1;
    *n_nodes = p.n_nodes;
    *workspace_bytes = L.total;
    return 0;
}

extern "C" TF_API int tf_bvh_build(const float* vertices, int64_t n_vertices, const int32_t* triangles, int64_t n_triangles,
                                   void* workspace, size_t workspace_bytes, void* nodes, void* tris, int32_t* perm, tf_stream_t stream) {
    TF_REQUIRE(vertices && triangles && workspace && nodes && tris && perm, "tf_bvh_build: NULL pointer");
    TF_REQUIRE(n_triangles > 0 && n_vertices > 0, "tf_bvh_build: empty mesh");
    TF_REQUIRE(n_triangles < (int64_t(1) << 31), "tf_bvh_build: %lld triangles, the BVH holds fewer than 2^31", (long long)n_triangles);
    TF_REQUIRE((reinterpret_cast<uintptr_t>(workspace) | reinterpret_cast<uintptr_t>(nodes) | reinterpret_cast<uintptr_t>(tris)) % 16 == 0,
               "tf_bvh_build: workspace, nodes and tris must be 16-byte aligned");
    const int n = (int)n_triangles;
    const Plan p = make_plan(n_triangles);
    Layout L;
    if (make_layout(n_triangles, p, L, "tf_bvh_build")) return 1;
    TF_REQUIRE(workspace_bytes >= L.total, "tf_bvh_build: workspace of %zu bytes, %zu needed", workspace_bytes, L.total);
    char* ws = static_cast<char*>(workspace);
    BuildRec* rec = reinterpret_cast<BuildRec*>(ws + L.rec);
    uint64_t* keys0 = reinterpret_cast<uint64_t*>(ws + L.keys0);
    uint64_t* keys1 = reinterpret_cast<uint64_t*>(ws + L.keys1);
    int32_t* ord = reinterpret_cast<int32_t*>(ws + L.ord0);
    int32_t* alt = reinterpret_cast<int32_t*>(ws + L.ord1);
    int32_t* nid = reinterpret_cast<int32_t*>(ws + L.nid);
    int32_t* node_lo = reinterpret_cast<int32_t*>(ws + L.node_lo);
    int32_t* node_cnt = reinterpret_cast<int32_t*>(ws + L.node_cnt);
    int32_t* node_rank = reinterpret_cast<int32_t*>(ws + L.node_rank);
    uint32_t* acc = reinterpret_cast<uint32_t*>(ws + L.acc);
    void* sort_tmp = ws + L.sort;
    const cudaStream_t s = (cudaStream_t)stream;
    const unsigned slot_blocks = (unsigned)((n + 255) / 256);
    const unsigned red_blocks = (unsigned)((n + 32 * RED_TILES * 8 - 1) / (32 * RED_TILES * 8));
    int launches = 0;

    cudaError_t e = cudaMemsetAsync(acc, 0xff, (size_t)p.n_nodes * 12 * sizeof(uint32_t), s);
    TF_REQUIRE(e == cudaSuccess, "tf_bvh_build: memset failed: %s", cudaGetErrorString(e));
    bvh_build_prep<<<slot_blocks, 256, 0, s>>>(vertices, triangles, n, rec, ord, nid, node_lo, node_cnt, node_rank);
    ++launches;
    for (int d = 0; d < p.levels; ++d) {
        bvh_build_reduce<<<red_blocks, 256, 0, s>>>(rec, ord, nid, n, acc);
        bvh_build_split<<<slot_blocks, 256, 0, s>>>(rec, ord, nid, n, acc, node_lo, node_cnt, node_rank, p.tab, d, keys0, alt);
        launches += 2;
        cub::DoubleBuffer<uint64_t> kb(keys0, keys1);
        cub::DoubleBuffer<int32_t> vb(alt, ord);
        size_t sort_bytes = L.sort_bytes;
        e = cub::DeviceRadixSort::SortPairs(sort_tmp, sort_bytes, kb, vb, n, 0, p.end_bit, s);
        if (e != cudaSuccess) {
            tf_count_launches(launches);
            tf_set_error("tf_bvh_build: radix sort failed: %s", cudaGetErrorString(e));
            return 2;
        }
        ord = vb.Current();
        alt = vb.Alternate();
    }
    bvh_build_reduce<<<red_blocks, 256, 0, s>>>(rec, ord, nid, n, acc);
    bvh_build_nodes<<<(unsigned)((p.n_nodes + 255) / 256), 256, 0, s>>>(acc, node_lo, node_cnt, node_rank, (int)p.n_nodes, ord,
                                                                         static_cast<BvhNode*>(nodes));
    bvh_build_tris<<<slot_blocks, 256, 0, s>>>(vertices, triangles, ord, n, static_cast<BvhTri*>(tris), perm);
    launches += 3;
    tf_count_launches(launches);
    TF_CHECK_LAUNCH("tf_bvh_build");
    return 0;
}
