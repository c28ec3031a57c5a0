"""CPU checks of mesh simplification: the numpy oracle (oracle/torch_oracle_simplify.py) on marching-cubes spheres and tori, an
open bumpy sphere, two spheres with a lone tetrahedron, a flat grid with a boundary and a lattice with zero-area faces: closed
2-manifolds stay closed 2-manifolds, Euler characteristic and components are kept, boundaries come out bit-identical, T' meets
the target, max_error = 0 keeps a plane exact, each round's winners have disjoint closed 1-rings and pass every check when it
is recomputed by brute force.  Also the refusals of tf_mesh_simplify / tf_mesh_simplify_sizes, geometry.simplify_mesh and
ShapeRenderer.extract_geometry, none of which launches anything."""
import ctypes
import math

import numpy as np
import pytest
import torch

from oracle import torch_oracle_cc as CC
from oracle import torch_oracle_simplify as O
from oracle.torch_oracle_iso import marching_cubes


@pytest.fixture(scope="module")
def lib():
    from tensoflow_b200 import build, _lib
    build.build()
    return _lib.load()


def _lattice(R):
    ax = torch.linspace(-1, 1, R)
    x, y, z = torch.meshgrid(ax, ax, ax, indexing="ij")
    return torch.stack([x, y, z], -1)


def mc_sphere(R, r=0.5):
    return marching_cubes(_lattice(R).norm(dim=-1) - r)


def mc_torus(R):
    p = _lattice(R)
    q = torch.stack([p[..., :2].norm(dim=-1) - 0.5, p[..., 2]], -1)
    return marching_cubes(q.norm(dim=-1) - 0.2)


def two_spheres_and_tetrahedron():
    p = _lattice(40)
    u = torch.minimum((p - torch.tensor([-0.4, 0.0, 0.0])).norm(dim=-1) - 0.35, (p - torch.tensor([0.45, 0.0, 0.0])).norm(dim=-1) - 0.3)
    v, t = marching_cubes(u)
    tet_v = torch.tensor([[0, 0, 50], [1, 0, 50], [0, 1, 50], [0, 0, 51]], dtype=torch.float32)
    tet_t = torch.tensor([[0, 2, 1], [0, 1, 3], [1, 2, 3], [0, 3, 2]], dtype=torch.int32) + v.shape[0]
    return torch.cat([v, tet_v]), torch.cat([t, tet_t])


def flat_grid(n=64):
    i, j = torch.meshgrid(torch.arange(n), torch.arange(n), indexing="ij")
    v = torch.stack([i.float() / (n - 1), j.float() / (n - 1), torch.zeros(n, n)], -1).reshape(-1, 3)
    a = (i[:-1, :-1] * n + j[:-1, :-1]).reshape(-1)
    t = torch.cat([torch.stack([a, a + n, a + 1], -1), torch.stack([a + 1, a + n, a + n + 1], -1)])
    return v, t.to(torch.int32)


def exact_threshold_lattice():
    """integer-valued field: many lattice values are exactly the threshold, so marching cubes emits zero-area faces"""
    p = _lattice(33) * 16
    return marching_cubes(torch.round(p.norm(dim=-1)) - 9.0)


def bumpy():
    from tensoflow_b200.synthetic import bumpy_sphere
    return bumpy_sphere(40, 21)


MESHES = {"mc-sphere-40": lambda: mc_sphere(40), "mc-torus-48": lambda: mc_torus(48), "bumpy-40x21": bumpy,
          "two-spheres-tetrahedron": two_spheres_and_tetrahedron, "flat-grid-64": flat_grid,
          "exact-threshold": exact_threshold_lattice}
CLOSED = ("mc-sphere-40", "mc-torus-48", "two-spheres-tetrahedron")


def _np(mesh):
    v, t = mesh
    return v.numpy(), t.numpy().astype(np.int64)


def directed_edges(t):
    t = np.asarray(t, np.int64)
    return np.concatenate([t[:, [0, 1]], t[:, [1, 2]], t[:, [2, 0]]])


def edge_counts(t):
    e = np.sort(directed_edges(t), 1)
    keys, counts = np.unique(e[:, 0] * (1 << 32) + e[:, 1], return_counts=True)
    return keys, counts


def is_closed_manifold(t):
    _, counts = edge_counts(t)
    d = directed_edges(t)
    return bool((counts == 2).all()) and np.unique(d[:, 0] * (1 << 32) + d[:, 1]).shape[0] == d.shape[0]


def euler(v, t):
    used = np.unique(t)
    return used.shape[0] - edge_counts(t)[0].shape[0] + t.shape[0]


def n_components(v, t):
    root, cnt = CC.mesh_components(v.shape[0], t)
    return int((cnt > 0).sum())


def boundary(v, t):
    """boundary edges as sorted pairs of position tuples, and the positions of their vertices"""
    keys, counts = edge_counts(t)
    b = keys[counts == 1]
    a, c = b >> 32, b & 0xFFFFFFFF
    pairs = {tuple(sorted((tuple(v[x].tolist()), tuple(v[y].tolist())))) for x, y in zip(a, c)}
    verts = {tuple(v[x].tolist()) for x in np.concatenate([a, c])}
    return pairs, verts


@pytest.fixture(scope="module", params=sorted(MESHES))
def mesh(request):
    return request.param, _np(MESHES[request.param]())


@pytest.mark.parametrize("frac", [0.5, 0.1, 0.01])
def test_oracle_properties(mesh, frac):
    name, (v, t) = mesh
    target = int(frac * t.shape[0])
    vo, to, rounds = O.simplify(v, t, target)
    assert vo.dtype == np.float32 and to.dtype == np.int32
    assert to.shape[0] >= target
    if frac >= 0.1 and name in CLOSED:                                    # the open meshes run out of valid edges first
        assert to.shape[0] in (target, target + 1), (name, to.shape[0], target)
    assert np.unique(to).shape[0] == vo.shape[0]                           # every output vertex is referenced
    if name in CLOSED:
        assert is_closed_manifold(t) and is_closed_manifold(to)
    assert euler(vo, to) == euler(v, t)
    assert n_components(vo, to) == n_components(v, t)
    if name == "two-spheres-tetrahedron":
        tet = v[-4:]
        assert all(any((vo == p).all(1)) for p in tet)                      # the tetrahedron survives, bit for bit
    bp, bv = boundary(v, t)
    bpo, bvo = boundary(vo, to)
    assert bp == bpo and bv <= {tuple(p) for p in vo.tolist()}


def test_flat_grid_with_zero_error_stays_exact():
    v, t = _np(flat_grid())
    vo, to, rounds = O.simplify(v, t, 0, max_error=0.0)
    assert rounds > 0 and to.shape[0] < t.shape[0] // 4
    assert (vo[:, 2] == 0).all()

    def area(v, t):
        p = v.astype(np.float64)[t]
        return float(np.abs(np.cross(p[:, 1] - p[:, 0], p[:, 2] - p[:, 0])[:, 2]).sum() / 2)
    assert abs(area(vo, to) - area(v, t)) <= 1e-12 * area(v, t)


@pytest.mark.parametrize("name", sorted(MESHES))
def test_target_at_least_t_is_identity(name):
    v, t = _np(MESHES[name]())
    for target in (t.shape[0], t.shape[0] - 1, 10 * t.shape[0]):
        vo, to, rounds = O.simplify(v, t, target)
        assert rounds == 0
        used = np.unique(t)
        np.testing.assert_array_equal(vo, v[used])
        if used.shape[0] == v.shape[0]:
            assert vo.tobytes() == v.tobytes() and to.tobytes() == t.astype(np.int32).tobytes()


def _brute_adjacency(F):
    """faces as tuples, star per vertex and the locked vertices, with Python sets and loops"""
    faces = [tuple(int(x) for x in f) for f in F]
    star = {}
    for i, f in enumerate(faces):
        for x in f:
            star.setdefault(x, []).append(i)
    locked = set()
    count = {}
    for f in faces:
        if len(set(f)) < 3:
            locked.update(f)
        for x, y in ((f[0], f[1]), (f[1], f[2]), (f[2], f[0])):
            count[(min(x, y), max(x, y))] = count.get((min(x, y), max(x, y)), 0) + 1
    for (x, y), c in count.items():
        if c != 2:
            locked.update((x, y))
    return faces, star, locked


def _brute_valid(adj, P, Q, a, b, v, max_error):
    """every rule of one collapse recomputed by hand, the placement included"""
    faces, star, locked = adj
    edge_faces = [i for i in star[a] if b in faces[i]]
    if len(edge_faces) != 2 or a in locked or b in locked:
        return False
    c0, c1 = (sum(faces[i]) - a - b for i in edge_faces)
    if c0 == c1 or len(star[c0]) <= 3 or len(star[c1]) <= 3:
        return False
    nbr = lambda x: {y for i in star[x] for y in faces[i]} - {x}
    if nbr(a) & nbr(b) != {c0, c1}:
        return False
    pv, cost = O.placement((Q[a] + Q[b])[None], P[a][None], P[b][None])
    if not np.array_equal(pv[0], v):
        return False
    if max_error is not None and not math.sqrt(cost[0]) <= max_error:
        return False
    for i in set(star[a]) | set(star[b]):
        if i in edge_faces:
            continue
        n0 = O._normal(*[P[x].astype(np.float64) for x in faces[i]])
        if not n0.any():
            continue
        n1 = O._normal(*[v.astype(np.float64) if x in (a, b) else P[x].astype(np.float64) for x in faces[i]])
        if not (n0[0] * n1[0] + n0[1] * n1[1]) + n0[2] * n1[2] > 0:
            return False
    return True


@pytest.mark.parametrize("name,max_error", [("bumpy-40x21", None), ("mc-sphere-40", None), ("exact-threshold", None),
                                            ("flat-grid-64", 0.0), ("mc-torus-48", 0.05)])
def test_each_round_winners_are_independent_and_valid(name, max_error):
    v, t = _np(MESHES[name]())
    if name == "flat-grid-64":
        v, t = _np(flat_grid(16))
    seen = []

    def on_round(F, P, Q, R, w):
        adj = _brute_adjacency(F)
        faces, star, _ = adj
        ring = [set(r[r >= 0].tolist()) for r in w["ring"]]
        assert len(set().union(*ring)) == sum(len(r) for r in ring), "closed 1-rings of two winners overlap"
        for k in range(w["a"].shape[0]):
            a, b = int(w["a"][k]), int(w["b"][k])
            assert ring[k] == {x for i in star[a] + star[b] for x in faces[i]}
            assert _brute_valid(adj, P, Q, a, b, w["v"][k], max_error), (len(seen), a, b)
        seen.append(w["a"].shape[0])

    O.simplify(v, t, t.shape[0] // 20, max_error=max_error, on_round=on_round)
    assert len(seen) > 0 and min(seen) >= 1


def _fake():
    return ctypes.c_void_p(1 << 20)


def test_entry_points_refuse_bad_arguments(lib):
    f = _fake()
    nv, nt, nr = ctypes.c_int64(), ctypes.c_int64(), ctypes.c_int32()
    good = [f, 30, f, 10, 0, float("inf"), f, 1 << 30, f, f, ctypes.byref(nv), ctypes.byref(nt), ctypes.byref(nr), None]
    cases = []
    for i in (0, 2, 6, 8, 9, 10, 11, 12):
        a = list(good)
        a[i] = None
        cases.append((a, b"NULL pointer"))
    for i, val, match in ((1, 0, b"vertices"), (1, 1 << 31, b"vertices"), (3, 0, b"triangles"), (3, 1 << 31, b"triangles"),
                          (4, -1, b"target"), (5, -1e-3, b"max_error"), (5, float("nan"), b"max_error")):
        a = list(good)
        a[i] = val
        cases.append((a, match))
    ws = ctypes.c_size_t()
    n0 = lib.tf_launch_count()
    for a, match in cases:
        assert lib.tf_mesh_simplify(*a) != 0
        assert match in lib.tf_last_error(), (a, lib.tf_last_error())
    for args, match in (((30, 10, None), b"NULL pointer"), ((0, 10, ctypes.byref(ws)), b"vertices"),
                        ((1 << 31, 10, ctypes.byref(ws)), b"vertices"), ((30, 0, ctypes.byref(ws)), b"triangles"),
                        ((30, 1 << 31, ctypes.byref(ws)), b"triangles")):
        assert lib.tf_mesh_simplify_sizes(*args) != 0
        assert match in lib.tf_last_error()
    assert lib.tf_launch_count() == n0


@pytest.mark.parametrize("kw,match", [({"target_triangles": -1}, "target_triangles"), ({"target_triangles": 2.5}, "target_triangles"),
                                      ({"target_triangles": 10, "max_error": -0.1}, "max_error"),
                                      ({"target_triangles": 10, "max_error": float("nan")}, "max_error"),
                                      ({"target_triangles": 10, "max_error": float("inf")}, "max_error")])
def test_limits_are_refused_first(lib, kw, match):
    """ValueError before any tensor check: the CPU mesh would be refused next"""
    from tensoflow_b200.geometry import simplify_mesh
    from tensoflow_b200.shape_renderer import ShapeRenderer
    v, t = bumpy()
    n0 = lib.tf_launch_count()
    with pytest.raises(ValueError, match=match):
        simplify_mesh(v, t, **kw)
    shape = ShapeRenderer.__new__(ShapeRenderer)                  # no field: the arguments are refused before it is needed
    with pytest.raises(ValueError, match=match):
        shape.extract_geometry([-1.0] * 3, [1.0] * 3, 64, **kw)
    assert lib.tf_launch_count() == n0


@pytest.mark.parametrize("case,match", [("cpu", "CUDA"), ("shape", "CUDA"), ("float-triangles", "integer triangles"),
                                        ("2^31-vertices", "2\\^31")])
def test_mesh_refusals_launch_nothing(lib, case, match):
    from tensoflow_b200.geometry import simplify_mesh
    v, t = bumpy()
    if case == "shape":
        t = t.reshape(-1, 6)
    elif case == "float-triangles":
        t = t.float()
    elif case == "2^31-vertices":
        v = torch.zeros(1, 3).expand(1 << 31, 3)
    n0 = lib.tf_launch_count()
    with pytest.raises(RuntimeError, match=match):
        simplify_mesh(v, t, 10)
    assert lib.tf_launch_count() == n0
