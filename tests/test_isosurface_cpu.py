"""Isosurface extraction without a GPU: the generated case table (header in sync, invariants of the rule), the CPU oracle's
meshes (watertight away from the lattice boundary, right topology and geometry on analytic fields) and the GPU entry points'
refusal of CPU tensors."""
import math
from pathlib import Path

import numpy as np
import pytest
import torch

from oracle.torch_oracle_iso import marching_cubes as oracle_mc
from tensoflow_b200 import isosurface_table as T

ROOT = Path(__file__).resolve().parents[1]


# ---- helpers shared with tests/test_isosurface_gpu.py ----------------------------------------------------------------------
def random_volume(shape, kind, seed):
    g = torch.Generator().manual_seed(seed)
    if kind == "normal":
        return torch.randn(shape, generator=g)
    if kind == "exact":                       # many values exactly at the threshold 0 (they count as outside)
        return torch.randint(-2, 3, shape, generator=g).float()
    if kind == "checker":                     # every face of every cell is ambiguous
        i, j, k = torch.meshgrid(*(torch.arange(n) for n in shape), indexing="ij")
        return torch.where((i + j + k) % 2 == 0, 1.0, -1.0) * (1 + torch.rand(shape, generator=g))
    raise ValueError(kind)


RANDOM_CASES = [(s, kind, seed) for seed, s in enumerate([(2, 2, 2), (3, 5, 7), (17, 9, 33)]) for kind in ("normal", "exact", "checker")]


def lattice(n, centre=None):
    g = torch.arange(n, dtype=torch.float64)
    x, y, z = torch.meshgrid(g, g, g, indexing="ij")
    return x, y, z


def sphere_sdf(n, centre, r):
    x, y, z = lattice(n)
    return ((x - centre[0]) ** 2 + (y - centre[1]) ** 2 + (z - centre[2]) ** 2).sqrt() - r


def torus_sdf(n, centre, R, r):
    x, y, z = lattice(n)
    q = ((x - centre[0]) ** 2 + (y - centre[1]) ** 2).sqrt() - R
    return (q ** 2 + (z - centre[2]) ** 2).sqrt() - r


def edge_uses(tris):
    """directed edges [3T,2] int64 of a triangle list"""
    t = tris.long()
    return torch.cat([t[:, [0, 1]], t[:, [1, 2]], t[:, [2, 0]]], 0)


def check_mesh_edges(verts, tris, shape):
    """Away from the lattice's boundary faces every mesh edge is used by exactly two triangles in opposite directions; an edge
    used once lies on a boundary face (both ends on the same boundary plane).  No directed edge is used twice."""
    assert tris.dtype == torch.int32 and verts.dtype == torch.float32
    t = tris.long()
    assert bool((t[:, 0] != t[:, 1]).all() and (t[:, 1] != t[:, 2]).all() and (t[:, 2] != t[:, 0]).all())
    assert t.numel() == 0 or (int(t.min()) >= 0 and int(t.max()) < verts.shape[0])
    e = edge_uses(tris)
    assert torch.unique(e, dim=0).shape[0] == e.shape[0], "a directed edge is used twice"
    und, counts = torch.unique(torch.sort(e, 1)[0], dim=0, return_counts=True)
    once = und[counts == 1]
    v0, v1 = verts[once[:, 0]], verts[once[:, 1]]
    hi = torch.tensor([n - 1 for n in shape], dtype=torch.float32)
    on_plane = (v0 == v1) & ((v0 == 0) | (v0 == hi))
    assert bool(on_plane.any(-1).all()), "an edge used by one triangle lies inside the lattice"
    return int((counts == 2).sum()), int(once.shape[0])


def euler_characteristic(verts, tris):
    und = torch.unique(torch.sort(edge_uses(tris), 1)[0], dim=0)
    return verts.shape[0] - und.shape[0] + tris.shape[0]


def n_components(verts, tris):
    from scipy.sparse import coo_matrix
    from scipy.sparse.csgraph import connected_components
    e = edge_uses(tris).numpy()
    a = coo_matrix((np.ones(e.shape[0]), (e[:, 0], e[:, 1])), shape=(verts.shape[0],) * 2)
    return connected_components(a, directed=False)[0]


def signed_volume(verts, tris):
    v = verts.double()[tris.long()]
    return float((v[:, 0] * torch.cross(v[:, 1], v[:, 2], dim=-1)).sum() / 6)


# ---- the case table ------------------------------------------------------------------------------------------------------
def test_table_header_is_generated():
    assert (ROOT / "tensoflow_b200" / "csrc" / "isosurface_table.cuh").read_text() == T.render_header()


def test_table_invariants():
    table, count = T.build_table()
    hist = {}
    for case in range(256):
        row = [int(v) for v in table[case]]
        n = int(count[case])
        assert n <= T.MAX_TRIS and row[3 * n] == -1 and all(v == -1 for v in row[3 * n:]), case
        used = row[:3 * n]
        assert sorted(set(used)) == T.crossed_edges(case), case        # exactly the crossed edges, each at least once
        # a triangle side joining two edges of one face is that face's segment (no fan diagonal in a face plane)
        segs = {frozenset(s) for s in T._face_segments(case)}
        for tri in zip(used[0::3], used[1::3], used[2::3]):
            for e, f in ((tri[0], tri[1]), (tri[1], tri[2]), (tri[2], tri[0])):
                assert not T.share_face(e, f) or frozenset((e, f)) in segs, (case, tri)
        hist[n] = hist.get(n, 0) + 1
    assert hist == {0: 2, 1: 16, 2: 50, 3: 80, 4: 76, 5: 32}


def test_table_winding_follows_the_field():
    """With vertices at the edge mid-points, every triangle's normal has a positive component along the gradient of the trilinear
    interpolant of the corner signs (outside +1, inside -1) at its centroid: triangles face toward increasing u."""
    for case in range(256):
        val = [-1.0 if case >> c & 1 else 1.0 for c in range(8)]
        for tri in T.case_triangles(case):
            v = [T._edge_mid(e) for e in tri]
            n = np.cross(v[1] - v[0], v[2] - v[0])
            x = np.mean(v, 0)
            g = np.zeros(3)
            for c in range(8):
                p = T.corner_pos(c)
                w = [x[a] if p[a] else 1 - x[a] for a in range(3)]
                for a in range(3):
                    g[a] += val[c] * np.prod([(1 if p[a] else -1) if b == a else w[b] for b in range(3)])
            assert float(np.dot(n, g)) > 0, (case, tri)


# ---- the oracle ----------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("shape,kind,seed", RANDOM_CASES, ids=[f"{'x'.join(map(str, s))}-{k}" for s, k, _ in RANDOM_CASES])
def test_oracle_random_fields_are_crack_free(shape, kind, seed):
    u = random_volume(shape, kind, seed)
    v, t = oracle_mc(u, 0.0)
    assert v.shape[1] == 3 and t.shape[1] == 3
    inside = u < 0
    n_crossed = int((inside[1:] != inside[:-1]).sum() + (inside[:, 1:] != inside[:, :-1]).sum() + (inside[:, :, 1:] != inside[:, :, :-1]).sum())
    assert v.shape[0] == n_crossed
    assert sorted(set(t.reshape(-1).tolist())) == list(range(v.shape[0]))      # every vertex is used
    check_mesh_edges(v, t, shape)


def test_oracle_sphere():
    n, c, r = 64, (31.3, 30.7, 32.1), 20.4
    v, t = oracle_mc(sphere_sdf(n, c, r), 0.0)
    assert check_mesh_edges(v, t, (n,) * 3)[1] == 0                              # closed
    assert n_components(v, t) == 1 and euler_characteristic(v, t) == 2
    # inscribed polyhedron: the volume comes out a little small (0.14 % measured); 1 % bar
    assert abs(signed_volume(v, t) / (4 / 3 * math.pi * r ** 3) - 1) < 1e-2
    # linear interpolation of |x| - r along a unit edge errs by at most ~1 / (8 r) ~ 0.006 voxel; 0.02 voxel bar
    rad = (v.double() - torch.tensor(c, dtype=torch.float64)).norm(dim=-1) - r
    assert float(rad.abs().max()) < 0.02


def test_oracle_torus():
    v, t = oracle_mc(torus_sdf(64, (31.6, 32.3, 31.2), 18.0, 6.5), 0.0)
    assert check_mesh_edges(v, t, (64,) * 3)[1] == 0
    assert n_components(v, t) == 1 and euler_characteristic(v, t) == 0
    assert signed_volume(v, t) > 0


def test_oracle_linear_field():
    """u = a.x + b with dyadic coefficients (exact in fp32): vertices sit on the plane a.x + b = threshold up to the rounding of
    t and of a_axis + t (a few ulp of the coordinate)."""
    a = torch.tensor([0.25, 0.5, -0.75], dtype=torch.float64)
    x, y, z = lattice(64)
    u = a[0] * x + a[1] * y + a[2] * z + 0.125
    thr = 0.3
    v, t = oracle_mc(u, thr)
    assert v.shape[0] > 1000
    resid = (v.double() @ a + 0.125 - float(np.float32(thr))).abs()
    assert float(resid.max()) <= 4 * 2.0 ** -23 * 64 * float(a.abs().sum())
    check_mesh_edges(v, t, (64,) * 3)
    n = torch.cross(v[t[:, 1].long()] - v[t[:, 0].long()], v[t[:, 2].long()] - v[t[:, 0].long()], dim=-1).double()
    assert bool(((n @ a) > 0).all())                                             # facing toward increasing u


# ---- no CPU path ---------------------------------------------------------------------------------------------------------
def test_cpu_tensors_raise_before_any_launch():
    from tensoflow_b200 import _lib
    from tensoflow_b200.isosurface import marching_cubes
    from tensoflow_b200.shape_renderer import ShapeRenderer
    n0 = _lib.launch_count()
    with pytest.raises(RuntimeError):
        marching_cubes(torch.zeros(4, 4, 4))
    shape = ShapeRenderer(dict(device='cpu', gridSize=[16] * 3, sdf_n_comp=4, sdf_dim=32, app_dim=16,
                               shader_config=dict(env_res=16, env_min_res=4)))
    with pytest.raises(RuntimeError):
        shape.extract_geometry([-1.0] * 3, [1.0] * 3, 8)
    assert _lib.launch_count() == n0
