"""Geometry evaluation without a GPU: the fp64 oracle of the closest-point query (oracle/torch_oracle_geom.py) against a dense
barycentric search on single triangles in every region of Ericson's test and on degenerate triangles, the oracle's sampling
is area-weighted, and the GPU entry points refuse CPU tensors before any launch."""
import pytest
import torch

from oracle import torch_oracle_geom as G

A, B, C = [0.0, 0.0, 0.0], [2.0, 0.0, 0.0], [0.5, 1.5, 0.0]


def _grid_search(points, tri, m=400):
    """min over the barycentric grid (i, j) / m, i + j <= m of the distance: an upper bound on the true distance that exceeds it
    by at most the grid's covering radius (the longest edge / m)."""
    i, j = torch.meshgrid(torch.arange(m + 1, dtype=torch.float64), torch.arange(m + 1, dtype=torch.float64), indexing="ij")
    keep = (i + j) <= m
    v, w = i[keep] / m, j[keep] / m
    a, b, c = tri.double()
    grid = a + v[:, None] * (b - a) + w[:, None] * (c - a)
    return torch.cdist(points.double(), grid).min(1)[0]


def _longest_edge(tri):
    a, b, c = tri.double()
    return float(max((b - a).norm(), (c - a).norm(), (c - b).norm()))


def _check_against_grid(points, tri, expected=None):
    q, d, t, second = G.closest_point(points, tri, torch.tensor([[0, 1, 2]]))
    assert torch.equal(t, torch.zeros_like(t)) and bool(torch.isinf(second).all())
    assert bool(torch.isfinite(q).all() and torch.isfinite(d).all())
    assert torch.allclose((points.double() - q).norm(dim=-1), d, rtol=0, atol=1e-12)
    g = _grid_search(points, tri)
    h = _longest_edge(tri) / 400
    assert bool((d <= g + 1e-12).all()), (d - g).max()              # never farther than a point of the triangle
    assert bool((d >= g - h - 1e-12).all()), (g - d).max()         # and the grid comes within its spacing
    if expected is not None:
        assert torch.allclose(q, expected.double(), rtol=0, atol=1e-12)


def test_closest_point_in_each_region():
    """Query points chosen in each of the 7 regions (vertex a, b, c; edge ab, ac, bc; face, above and below), with their
    closest point known analytically; then points exactly on the vertices and edges."""
    tri = torch.tensor([A, B, C], dtype=torch.float64)
    a, b, c = tri
    pts, exp = [], []
    for vtx, out in ((a, torch.tensor([-1.0, -0.5, 0.3])), (b, torch.tensor([1.0, -0.5, -0.2])), (c, torch.tensor([0.1, 1.0, 0.4]))):
        pts.append(vtx + out.double())
        exp.append(vtx)
    for p0, p1 in ((a, b), (a, c), (b, c)):
        e = p1 - p0
        inplane_out = torch.cross(e, torch.tensor([0, 0, 1.0], dtype=torch.float64), dim=0)
        inplane_out = inplane_out / inplane_out.norm()
        if float(torch.dot(inplane_out, (a + b + c) / 3 - p0)) > 0:
            inplane_out = -inplane_out
        foot = p0 + 0.3 * e
        pts.append(foot + 0.7 * inplane_out + torch.tensor([0, 0, 0.25], dtype=torch.float64))
        exp.append(foot)
    for z in (0.6, -0.45):
        foot = 0.5 * a + 0.3 * b + 0.2 * c
        pts.append(foot + torch.tensor([0, 0, z], dtype=torch.float64))
        exp.append(foot)
    on = [a, b, c, 0.5 * (a + b), 0.25 * a + 0.75 * c, 0.6 * b + 0.4 * c, (a + b + c) / 3]
    _check_against_grid(torch.stack(pts + on), tri, torch.stack(exp + on))


def test_closest_point_random_triangles():
    g = torch.Generator().manual_seed(0)
    for _ in range(4):
        tri = torch.randn(3, 3, generator=g, dtype=torch.float64)
        _check_against_grid(torch.randn(200, 3, generator=g, dtype=torch.float64) * 1.5, tri)


@pytest.mark.parametrize("kind", ["collinear", "collinear-outer", "repeated-vertex", "point"])
def test_closest_point_degenerate_triangles(kind):
    """Zero-area triangles are measured through their edges and vertices: the grid search (which covers the union of the edges
    there) agrees, and nothing is NaN, including for query points on the segment and on the vertices."""
    a = torch.tensor([0.2, -0.1, 0.3], dtype=torch.float64)
    d = torch.tensor([1.0, 0.5, -0.25], dtype=torch.float64)
    tri = {"collinear": torch.stack([a, a + 2 * d, a + 0.7 * d]),                    # c between a and b
           "collinear-outer": torch.stack([a, a + d, a - 1.5 * d]),                 # a between b and c
           "repeated-vertex": torch.stack([a, a, a + d]),
           "point": torch.stack([a, a, a])}[kind]
    g = torch.Generator().manual_seed(1)
    pts = torch.cat([torch.randn(100, 3, generator=g, dtype=torch.float64) * 2, tri, a + 0.5 * d[None]])
    _check_against_grid(pts, tri)


def test_closest_point_ties_go_to_the_smaller_index():
    """Two copies of a triangle: every query ties exactly and reports the first copy; the second-best distance equals the best."""
    v = torch.tensor([A, B, C, A, B, C], dtype=torch.float64)
    t = torch.tensor([[3, 4, 5], [0, 1, 2]])
    pts = torch.randn(50, 3, generator=torch.Generator().manual_seed(2), dtype=torch.float64)
    _, d, tri, second = G.closest_point(pts, v, t, tri_chunk=1)
    assert torch.equal(tri, torch.zeros_like(tri)) and torch.equal(second, d)


def test_oracle_sampling_is_area_weighted():
    """Two triangles of areas 1 and 3: triangle counts of 40000 samples pass a chi-square test against 1:3 at p = 1e-3 (fixed seed),
    every point lies on its triangle (z = 0 plane, barycentric inside) and the normals are the unit face normals."""
    from scipy.stats import chisquare
    v = torch.tensor([[0, 0, 0], [1, 0, 0], [0, 2, 0], [5, 0, 0], [8, 0, 0], [5, 2, 0]], dtype=torch.float32)
    t = torch.tensor([[0, 1, 2], [3, 4, 5]], dtype=torch.int32)
    cdf = G.area_cdf(v, t)
    assert torch.allclose(cdf, torch.tensor([0.25, 1.0], dtype=torch.float64), rtol=0, atol=0)
    n = 40000
    u = torch.rand(n, 3, generator=torch.Generator().manual_seed(3), dtype=torch.float64)
    p, tri, nrm = G.sample_surface(v, t, cdf, u)
    counts = torch.bincount(tri, minlength=2).double()
    assert chisquare(counts.numpy(), (torch.tensor([0.25, 0.75]) * n).numpy()).pvalue > 1e-3
    assert float(p[:, 2].abs().max()) == 0.0
    first = tri == 0
    assert bool((p[first, 0] >= 0).all() and (p[first, 1] >= 0).all() and (2 * p[first, 0] + p[first, 1] <= 2 + 1e-12).all())
    assert bool((p[~first, 0] >= 5).all() and (p[~first, 1] >= 0).all() and (2 * (p[~first, 0] - 5) / 3 + p[~first, 1] <= 2 + 1e-12).all())
    assert torch.equal(nrm, torch.tensor([0, 0, 1.0], dtype=torch.float64).expand(n, 3))
    # uniform within a triangle: the mean of the samples of each is its centroid
    assert torch.allclose(p[first].mean(0), torch.tensor([1 / 3, 2 / 3, 0], dtype=torch.float64), atol=0.02)


def test_cpu_tensors_raise_before_any_launch():
    from tensoflow_b200 import _lib
    from tensoflow_b200.geometry import evaluate_mesh, sample_surface
    from tensoflow_b200.mc_ops import RayTracer
    from tensoflow_b200.synthetic import bumpy_sphere
    v, t = bumpy_sphere(16, 8)
    n0 = _lib.launch_count()
    rt = RayTracer.__new__(RayTracer)           # no BVH: building one needs a device, and the refusal comes first
    rt._h = None
    with pytest.raises(RuntimeError, match="CUDA"):
        rt.closest_point(torch.zeros(4, 3))
    with pytest.raises(RuntimeError, match="CUDA"):
        sample_surface(v, t, 16)
    with pytest.raises(RuntimeError, match="CUDA"):
        evaluate_mesh(v, t, v, t, n_samples=16)
    assert _lib.launch_count() == n0
