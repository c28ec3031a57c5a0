// Lock-free union-find in the style of ECL-CC (Jaiganesh and Burtscher, "A High-Performance Connected Components Implementation
// for GPUs", HPDC 2018), shared by mesh_components.cu (over vertices) and uv_atlas.cu (over faces).
//
// root[] is the parent array.  Parents only ever decrease and stay inside their tree, so root[v] <= v, with equality exactly
// for the roots:
//   - a hook sets a root's parent to a smaller root with atomicCAS(&root[hi], hi, lo), so a node stops being a root once
//     and never becomes one again;
//   - path halving lowers a non-root's parent to what it read as its grandparent with atomicMin: smaller than the node, in
//     its tree, and not its descendant (descendants have larger indices), so the write cannot form a cycle or split a tree.
//     A plain store would not do: a halving store that read the parent before another thread flattened the node could land
//     after it and raise the parent again, leaving a node of the flattened output pointing at an ancestor below its root.
// Trees only ever merge, every finished union leaves both ends in one tree, and each tree's root is its smallest node.  So
// concurrent halving needs no locks, and the final root of a component is its minimum index whatever the scheduling.
// Parents are read through relaxed device-scope atomic references: a plain load may be served from a stale L1 line written by
// another SM.
#pragma once
#include <cuda/atomic>
#include <cstdint>

namespace tf_uf {

using ParentRef = cuda::atomic_ref<int32_t, cuda::thread_scope_device>;

__device__ __forceinline__ int32_t parent_of(int32_t* root, int32_t v) { return ParentRef(root[v]).load(cuda::memory_order_relaxed); }
__device__ __forceinline__ void set_parent(int32_t* root, int32_t v, int32_t p) { ParentRef(root[v]).store(p, cuda::memory_order_relaxed); }

// the root of v's tree; on the way every other node is pointed at its grandparent (path halving)
__device__ __forceinline__ int32_t find(int32_t* root, int32_t v) {
    int32_t p = parent_of(root, v);
    while (p != v) {
        const int32_t gp = parent_of(root, p);
        if (gp == p) return p;
        atomicMin(root + v, gp);
        v = gp;
        p = parent_of(root, v);
    }
    return v;
}

// hook the larger root under the smaller; a failed CAS returns the new parent of the node that is no longer a root, and the
// loop carries on from there
__device__ __forceinline__ void unite(int32_t* root, int32_t a, int32_t b) {
    int32_t ra = find(root, a), rb = find(root, b);
    while (ra != rb) {
        const int32_t lo = min(ra, rb), hi = max(ra, rb);
        const int32_t old = atomicCAS(root + hi, hi, lo);
        if (old == hi) return;
        if (ra == hi) ra = old; else rb = old;
    }
}

}  // namespace tf_uf
