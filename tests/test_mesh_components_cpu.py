"""CPU checks of the mesh clean-up: the connected-components oracle (scipy) against a plain breadth-first search on small
hand-made graphs, its remove_small_components against hand-worked answers, and the refusals of geometry.mesh_components /
remove_small_components / ShapeRenderer.extract_geometry and of tf_mesh_components, none of which launches anything."""
import ctypes
from collections import deque

import numpy as np
import pytest
import torch

from oracle import torch_oracle_cc as O


@pytest.fixture(scope="module")
def lib():
    from tensoflow_b200 import build, _lib
    build.build()
    return _lib.load()


def bfs_components(V, triangles):
    """root = smallest vertex of each component, by breadth-first search over adjacency lists"""
    adj = [[] for _ in range(V)]
    for a, b, c in triangles:
        for x, y in ((a, b), (b, c), (a, c)):
            adj[x].append(y)
            adj[y].append(x)
    root = [-1] * V
    for s in range(V):                       # increasing s: the first vertex reached of a component is its smallest
        if root[s] >= 0:
            continue
        root[s] = s
        q = deque([s])
        while q:
            x = q.popleft()
            for y in adj[x]:
                if root[y] < 0:
                    root[y] = s
                    q.append(y)
    count = [0] * V
    for a, _, _ in triangles:
        count[root[a]] += 1
    return np.array(root, np.int32), np.array(count, np.int32)


def _graphs():
    g = {}
    n = 50
    g["chain"] = (n, [(i, i + 1, i + 1) for i in range(n - 1)])
    g["chain-reversed"] = (n, [(i + 1, i, i) for i in reversed(range(n - 1))])
    g["chain-of-triangles"] = (n, [(i, i + 1, i + 2) for i in range(0, n - 2, 2)])
    g["star"] = (n, [(0, i, i) for i in range(1, n)])
    g["star-at-the-end"] = (n, [(n - 1, i, (i * 7) % (n - 1)) for i in range(n - 1)])
    g["duplicates-and-degenerate"] = (12, [(3, 4, 5)] * 5 + [(5, 5, 5), (7, 7, 8), (8, 7, 7), (10, 10, 10), (4, 3, 5)])
    g["unreferenced"] = (20, [(2, 9, 15), (15, 17, 2), (4, 6, 6)])    # 0, 1, 3, 5, 7, ... reference nothing
    g["one-edge-300-times"] = (6, [(0, 1, 1)] * 300 + [(2, 3, 4)] * 256)
    g["one-triangle"] = (3, [(2, 1, 0)])
    g["no-triangles"] = (4, [])
    rng = np.random.default_rng(0)
    for k in range(6):                        # sparse random soups: many components of all sizes
        V = int(rng.integers(5, 200))
        T = int(rng.integers(1, V))
        g[f"random{k}"] = (V, [tuple(int(x) for x in row) for row in rng.integers(0, V, (T, 3))])
    perm = rng.permutation(n)
    g["chain-permuted"] = (n, [(int(perm[i]), int(perm[i + 1]), int(perm[i + 1])) for i in range(n - 1)])
    return g


GRAPHS = _graphs()


@pytest.mark.parametrize("name", sorted(GRAPHS))
def test_oracle_equals_breadth_first_search(name):
    V, tris = GRAPHS[name]
    root, count = O.mesh_components(V, np.array(tris, np.int64).reshape(-1, 3))
    want_root, want_count = bfs_components(V, tris)
    assert root.dtype == np.int32 and count.dtype == np.int32
    np.testing.assert_array_equal(root, want_root)
    np.testing.assert_array_equal(count, want_count)
    assert count.sum() == len(tris)
    assert (count[root != np.arange(V)] == 0).all()


def test_oracle_remove_small_components_by_hand():
    # components (by triangles): {0,1,2,3}: 2, {5,6,7}: 1, {8,9,10}: 2 (tied with the first); 4 and 11 unreferenced
    v = np.arange(12 * 3, dtype=np.float32).reshape(12, 3)
    t = np.array([[8, 9, 10], [0, 1, 2], [7, 6, 5], [3, 2, 1], [10, 9, 8]])
    kv, kt = O.remove_small_components(v, t, 1.0)
    np.testing.assert_array_equal(kv, v[[0, 1, 2, 3, 8, 9, 10]])
    np.testing.assert_array_equal(kt, [[4, 5, 6], [0, 1, 2], [3, 2, 1], [6, 5, 4]])
    assert kt.dtype == np.int32 and kv.dtype == np.float32
    kv, kt = O.remove_small_components(v, t, 0.5)                   # 1 >= 0.5 * 2: everything referenced stays
    np.testing.assert_array_equal(kv, v[[0, 1, 2, 3, 5, 6, 7, 8, 9, 10]])
    np.testing.assert_array_equal(kt, [[7, 8, 9], [0, 1, 2], [6, 5, 4], [3, 2, 1], [9, 8, 7]])
    kv, kt = O.remove_small_components(v, t, 0.5000001)
    np.testing.assert_array_equal(kv, v[[0, 1, 2, 3, 8, 9, 10]])


def _mesh():
    from tensoflow_b200.synthetic import bumpy_sphere
    return bumpy_sphere(16, 8)


@pytest.mark.parametrize("frac", [0.0, -0.1, 1.5, float("nan")])
def test_min_fraction_out_of_range_raises_first(lib, frac):
    """ValueError before any tensor check: the CPU mesh would be refused next"""
    from tensoflow_b200.geometry import remove_small_components
    from tensoflow_b200.shape_renderer import ShapeRenderer
    v, t = _mesh()
    n0 = lib.tf_launch_count()
    with pytest.raises(ValueError, match="min_fraction"):
        remove_small_components(v, t, frac)
    shape = ShapeRenderer.__new__(ShapeRenderer)                  # no field: the argument is refused before it is needed
    with pytest.raises(ValueError, match="min_component_fraction"):
        shape.extract_geometry([-1.0] * 3, [1.0] * 3, 64, min_component_fraction=frac)
    assert lib.tf_launch_count() == n0


@pytest.mark.parametrize("case,match", [
    ("cpu", "CUDA"), ("shape", "CUDA"), ("empty", "CUDA"), ("float-triangles", "integer triangles"),
    ("2^31-vertices", "2\\^31"),
])
def test_mesh_refusals_launch_nothing(lib, case, match):
    """what can be refused without a device: CPU tensors (before shapes and emptiness, which the GPU tests check on CUDA
    tensors), non-integer triangles and 2^31 vertices (an expanded view: no memory behind it)"""
    from tensoflow_b200.geometry import mesh_components, remove_small_components
    v, t = _mesh()
    if case == "shape":
        t = t.reshape(-1, 6)
    elif case == "empty":
        t = t[:0]
    elif case == "float-triangles":
        t = t.float()
    elif case == "2^31-vertices":
        v = torch.zeros(1, 3).expand(1 << 31, 3)
    n0 = lib.tf_launch_count()
    with pytest.raises(RuntimeError, match=match):
        mesh_components(v, t)
    with pytest.raises(RuntimeError, match=match):
        remove_small_components(v, t, 0.5)
    assert lib.tf_launch_count() == n0


def test_entry_point_refuses_bad_arguments(lib):
    fake = ctypes.c_void_p(1 << 20)
    n0 = lib.tf_launch_count()
    for args, match in (((None, 10, 30, fake, fake, None), b"NULL pointer"), ((fake, 10, 30, None, fake, None), b"NULL pointer"),
                        ((fake, 10, 30, fake, None, None), b"NULL pointer"), ((fake, 10, 0, fake, fake, None), b"vertices"),
                        ((fake, 10, 1 << 31, fake, fake, None), b"vertices"), ((fake, -1, 30, fake, fake, None), b"triangles"),
                        ((fake, 1 << 31, 30, fake, fake, None), b"triangles")):
        assert lib.tf_mesh_components(*args) != 0
        assert match in lib.tf_last_error()
    assert lib.tf_launch_count() == n0
