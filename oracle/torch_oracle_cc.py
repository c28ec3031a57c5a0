"""TEST INFRASTRUCTURE ONLY (never imported by tensoflow_b200/).  Host restatement of the mesh clean-up of include/tensoflow_b200.h
and tensoflow_b200/geometry.py: tf_mesh_components from scipy.sparse.csgraph.connected_components, and
remove_small_components in numpy.

Conventions shared with the kernels:
  * the graph's nodes are the V vertices, its edges those of the triangles (a vertex no triangle references is a component of
    its own; repeated indices in a triangle add no edge);
  * root[v] = the smallest vertex index of v's component; tri_count[r] = the number of triangles whose vertices have root r,
    0 for every vertex that is not a root;
  * a triangle is kept iff tri_count[its root] >= min_fraction * max(tri_count) in fp64; kept triangles and the vertices they
    reference keep their order, indices are renumbered, unreferenced vertices are dropped."""
import numpy as np
from scipy.sparse import coo_matrix
from scipy.sparse.csgraph import connected_components


def mesh_components(n_vertices, triangles):
    """-> (root [V] int32, tri_count [V] int32) for triangles [T,3] (any integer array-like, indices in [0, V))."""
    V = int(n_vertices)
    t = np.asarray(triangles, dtype=np.int64).reshape(-1, 3)
    rows = np.concatenate([t[:, 0], t[:, 0]])
    cols = np.concatenate([t[:, 1], t[:, 2]])
    # fp64 weights: repeated edges are summed, and a narrow integer sum could wrap to an explicit zero
    graph = coo_matrix((np.ones(rows.shape[0], np.float64), (rows, cols)), shape=(V, V)).tocsr()
    n, labels = connected_components(graph, directed=False)
    smallest = np.full(n, V, np.int64)
    np.minimum.at(smallest, labels, np.arange(V, dtype=np.int64))
    root = smallest[labels]
    tri_count = np.zeros(V, np.int64)
    np.add.at(tri_count, root[t[:, 0]], 1)
    return root.astype(np.int32), tri_count.astype(np.int32)


def remove_small_components(vertices, triangles, min_fraction):
    """-> (vertices [V',3] of the input dtype, triangles [T',3] int32)."""
    v = np.asarray(vertices)
    t = np.asarray(triangles, dtype=np.int64).reshape(-1, 3)
    root, tri_count = mesh_components(v.shape[0], t)
    kept = t[tri_count[root[t[:, 0]]].astype(np.float64) >= float(min_fraction) * np.float64(tri_count.max())]
    used = np.unique(kept)                                       # sorted: the referenced vertices in input order
    new_index = np.full(v.shape[0], -1, np.int64)
    new_index[used] = np.arange(used.shape[0])
    return v[used], new_index[kept].astype(np.int32)
