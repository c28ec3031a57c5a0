"""Geometry evaluation on the GPU: tf_bvh_closest_point against the fp64 brute-force oracle (oracle/torch_oracle_geom.py) on
triangle soups with degenerate triangles and on marching-cubes meshes, at 10^6 points against a 10^6-triangle mesh,
tf_mesh_sample_surface against the oracle from the same CDF and uniforms, known answers of geometry.evaluate_mesh, the shape
stage's extracted mesh against the fp64 field's, and the error paths of the C ABI."""
import ctypes
import math

import pytest
import torch

from oracle import torch_oracle_geom as G
from oracle.torch_oracle_iso import marching_cubes as oracle_mc
from test_isosurface_cpu import sphere_sdf, torus_sdf

pytestmark = pytest.mark.gpu

ULP = 2.0 ** -23


def _cuda():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    return torch.device("cuda:0")


def _soup(n_tris, seed):
    """random triangles of size ~0.2 in [-1, 1]^3; a tenth each collinear, with a repeated vertex, and collapsed to a point"""
    g = torch.Generator().manual_seed(seed)
    c = torch.rand(n_tris, 1, 3, generator=g) * 2 - 1
    tri = c + 0.2 * torch.randn(n_tris, 3, 3, generator=g)
    k = n_tris // 10
    tri[:k, 2] = tri[:k, 0] + 0.37 * (tri[:k, 1] - tri[:k, 0])
    tri[k:2 * k, 1] = tri[k:2 * k, 0]
    tri[2 * k:3 * k, 1:] = tri[2 * k:3 * k, :1]
    perm = torch.randperm(n_tris, generator=g)                 # degenerate ones spread through the caller's order
    return tri[perm].reshape(-1, 3).float(), torch.arange(3 * n_tris, dtype=torch.int32).reshape(-1, 3)


MESHES = {
    "soup": lambda: _soup(2000, 0),
    "mc-sphere": lambda: oracle_mc(sphere_sdf(96, (47.3, 46.6, 48.2), 30.5), 0.0),
    "mc-torus": lambda: oracle_mc(torus_sdf(96, (47.6, 48.3, 47.2), 28.0, 9.5), 0.0),
}


def _queries(v, t, n, seed):
    """n points, a quarter each: far (within 1x the box beyond it), near the surface, on the surface, exactly on vertices"""
    g = torch.Generator().manual_seed(seed)
    m = [n // 4 + (1 if i < n % 4 else 0) for i in range(4)]
    lo, hi = v.min(0)[0], v.max(0)[0]
    far = lo + (hi - lo) * (torch.rand(m[0], 3, generator=g) * 3 - 1)
    ti = torch.randint(0, t.shape[0], (m[1] + m[2],), generator=g)
    w = torch.rand(ti.shape[0], 2, generator=g)
    w = torch.where(w.sum(1, keepdim=True) > 1, 1 - w, w)
    a, b, c = (v[t[ti, k].long()] for k in range(3))
    on = a + w[:, :1] * (b - a) + w[:, 1:] * (c - a)
    near = on[:m[1]] + 1e-3 * float((hi - lo).max()) * torch.randn(m[1], 3, generator=g)
    vert = v[torch.randint(0, v.shape[0], (m[3],), generator=g)]
    return torch.cat([far, near, on[m[1]:], vert]).float()


def _tolerance(d_ref, extent):
    """fp32 bound on a distance: 4 ulp of the scene extent (the rounding of p - v0, of the edges and of the few operations on
    them) plus 2^-22 relative (the squared distance's rounding and the square root)"""
    return 4 * ULP * extent + 2.0 ** -22 * d_ref


def _check_closest(rt, v, t, q, dev):
    from tensoflow_b200 import _lib
    n0 = _lib.launch_count()
    cp, d, tri = rt.closest_point(q.to(dev))
    assert _lib.launch_count() - n0 == 1
    assert cp.shape == q.shape and d.shape == q.shape[:1] and tri.dtype == torch.int64
    assert bool(torch.isfinite(cp).all() and torch.isfinite(d).all()) and int(tri.min()) >= 0 and int(tri.max()) < t.shape[0]
    ref_q, ref_d, ref_t, second = G.closest_point(q.to(dev), v.to(dev), t.to(dev))
    extent = float(torch.cat([v, q]).abs().max())
    tol = _tolerance(ref_d, extent)
    err = (d.double() - ref_d).abs()
    assert bool((err <= tol).all()), float((err / tol).max())
    separated = second - ref_d > tol
    assert torch.equal(tri[separated], ref_t[separated])
    # the reported point is at the reported distance and lies on the reported triangle
    assert bool(((q.to(dev).double() - cp.double()).norm(dim=-1) - d.double()).abs().le(tol).all())
    a = v.to(dev).double()[t.to(dev).long()[tri]]
    on_tri, _ = G.triangle_closest(cp.double() - a[:, 0], a[:, 1] - a[:, 0], a[:, 2] - a[:, 0])
    assert bool((on_tri.sqrt() <= tol).all())


@pytest.mark.parametrize("n", [1, 31, 4099])
@pytest.mark.parametrize("mesh", list(MESHES))
def test_closest_point_matches_oracle(mesh, n):
    from tensoflow_b200.mc_ops import RayTracer
    dev = _cuda()
    v, t = MESHES[mesh]()
    rt = RayTracer(v, t)
    q = _queries(v, t, n, seed=n)
    _check_closest(rt, v, t, q, dev)
    # queries shaped [..., 3] come back in that shape
    cp, d, tri = rt.closest_point(q.to(dev).reshape(1, n, 1, 3))
    assert cp.shape == (1, n, 1, 3) and d.shape == (1, n, 1) and tri.shape == (1, n, 1)


def test_closest_point_at_scale_is_reproducible():
    """10^6 points against the 10^6-triangle bumpy sphere (the config-3 mesh): a fixed 4096-point subset against the oracle,
    and two runs bit for bit."""
    from tensoflow_b200.mc_ops import RayTracer
    from tensoflow_b200.synthetic import bumpy_sphere
    dev = _cuda()
    v, t = bumpy_sphere(1000, 500)
    rt = RayTracer(v, t)
    g = torch.Generator().manual_seed(5)
    n = 1_000_000
    q = torch.cat([torch.rand(n // 2, 3, generator=g) * 1.6 - 0.8,                         # inside, outside, around
                   v[torch.randint(0, v.shape[0], (n - n // 2,), generator=g)] * (1 + 0.02 * torch.randn(n - n // 2, 1, generator=g))])
    qd = q.to(dev)
    cp1, d1, t1 = rt.closest_point(qd)
    cp2, d2, t2 = rt.closest_point(qd)
    torch.cuda.synchronize()
    assert torch.equal(cp1.view(torch.int32), cp2.view(torch.int32)) and torch.equal(d1.view(torch.int32), d2.view(torch.int32))
    assert torch.equal(t1, t2)
    sub = torch.randperm(n, generator=g)[:4096]
    ref_q, ref_d, ref_t, second = G.closest_point(qd[sub], v.to(dev), t.to(dev), point_chunk=1024, tri_chunk=8192)
    extent = float(torch.cat([v, q]).abs().max())
    tol = _tolerance(ref_d, extent)
    assert bool(((d1[sub].double() - ref_d).abs() <= tol).all())
    sep = second - ref_d > tol
    assert torch.equal(t1[sub][sep], ref_t[sep])


@pytest.mark.parametrize("mesh", ["soup", "bumpy"])
def test_sampling_matches_oracle(mesh):
    from tensoflow_b200 import _lib
    from tensoflow_b200.geometry import _sample_surface_from, sample_surface
    from tensoflow_b200.synthetic import bumpy_sphere
    dev = _cuda()
    v, t = _soup(2000, 1) if mesh == "soup" else bumpy_sphere(200, 100)
    vd, td = v.to(dev), t.to(dev)
    cdf = G.area_cdf(vd, td)
    n = 100_003
    u = torch.rand(n, 3, device=dev, dtype=torch.float64, generator=torch.Generator(device=dev).manual_seed(4))
    n0 = _lib.launch_count()
    p, tri, nrm = _sample_surface_from(vd, td, cdf, u)
    assert _lib.launch_count() - n0 == 1
    ref_p, ref_t, ref_n = G.sample_surface(vd, td, cdf, u)
    assert torch.equal(tri, ref_t)
    scale = ref_p.abs().max(-1, keepdim=True)[0]
    assert bool(((p.double() - ref_p).abs() <= 2e-7 * scale).all())
    a = vd.double()[td.long()[tri]]
    on_tri, _ = G.triangle_closest(p.double() - a[:, 0], a[:, 1] - a[:, 0], a[:, 2] - a[:, 0])
    assert float(on_tri.sqrt().max()) <= 1e-6
    assert float((nrm.double().norm(dim=-1) - 1).abs().max()) <= 1e-6
    assert torch.allclose(nrm.double(), ref_n, rtol=0, atol=1e-7)
    area = 0.5 * torch.cross(a[:, 1] - a[:, 0], a[:, 2] - a[:, 0], dim=-1).norm(dim=-1)
    assert bool((area > 0).all())                                 # zero-area triangles are never drawn
    # the public entry point: seeded, reproducible
    s1, s2 = sample_surface(vd, td, 1000, seed=7), sample_surface(vd, td, 1000, seed=7)
    assert all(torch.equal(x, y) for x, y in zip(s1, s2))
    assert not torch.equal(s1[0], sample_surface(vd, td, 1000, seed=8)[0])


def _plane(n, z):
    g = torch.linspace(-1, 1, n + 1)
    x, y = torch.meshgrid(g, g, indexing="ij")
    v = torch.stack([x, y, torch.full_like(x, z)], -1).reshape(-1, 3)
    i, j = torch.meshgrid(torch.arange(n), torch.arange(n), indexing="ij")
    a = (i * (n + 1) + j).reshape(-1)
    b, c, d = a + n + 1, a + 1, a + n + 2
    return v, torch.cat([torch.stack([a, b, c], -1), torch.stack([c, b, d], -1)]).to(torch.int32)


def test_evaluate_mesh_known_answers():
    from tensoflow_b200.geometry import evaluate_mesh
    from tensoflow_b200.synthetic import bumpy_sphere
    dev = _cuda()
    v, t = (x.to(dev) for x in bumpy_sphere(200, 100))
    r = evaluate_mesh(v, t, v, t, n_samples=200_000)
    assert set(r) == {"accuracy", "completeness", "chamfer", "normal_consistency", "precision", "recall", "fscore"}
    assert r["chamfer"] <= 1e-7 and r["normal_consistency"] >= 1 - 1e-6
    assert all(f == 1.0 for f in r["fscore"].values()) and sorted(r["fscore"]) == [0.005, 0.01, 0.02]

    delta = 0.01
    pv, pt = _plane(20, 0.0)
    gv, gt = _plane(20, delta)
    r = evaluate_mesh(pv.to(dev), pt.to(dev), gv.to(dev), gt.to(dev), n_samples=100_000, thresholds=(0.005, 0.02))
    d32 = float(torch.tensor(delta, dtype=torch.float32))
    for k in ("accuracy", "completeness", "chamfer"):
        assert abs(r[k] - d32) <= 4 * ULP + 2.0 ** -22 * d32, (k, r[k])
    assert r["normal_consistency"] >= 1 - 1e-6
    assert r["precision"][0.005] == r["recall"][0.005] == r["fscore"][0.005] == 0.0
    assert r["fscore"][0.02] == 1.0


def _uv_sphere(n_lon, n_lat, r, centre):
    """closed lat-long sphere: n_lat - 1 rings of n_lon vertices plus the two poles"""
    th = torch.arange(1, n_lat, dtype=torch.float64) * math.pi / n_lat
    ph = torch.arange(n_lon, dtype=torch.float64) * 2 * math.pi / n_lon
    T, P = torch.meshgrid(th, ph, indexing="ij")
    ring = torch.stack([T.sin() * P.cos(), T.sin() * P.sin(), T.cos()], -1).reshape(-1, 3)
    v = torch.cat([ring, torch.tensor([[0, 0, 1.0], [0, 0, -1.0]], dtype=torch.float64)]) * r + torch.tensor(centre, dtype=torch.float64)
    i = torch.arange(n_lat - 2)[:, None]
    j = torch.arange(n_lon)[None, :]
    a, b = i * n_lon + j, i * n_lon + (j + 1) % n_lon
    c, d = a + n_lon, b + n_lon
    north, south = (n_lat - 1) * n_lon, (n_lat - 1) * n_lon + 1
    j = torch.arange(n_lon)
    last = (n_lat - 2) * n_lon
    tris = torch.cat([torch.stack([a, c, b], -1).reshape(-1, 3), torch.stack([b, c, d], -1).reshape(-1, 3),
                      torch.stack([torch.full_like(j, north), j, (j + 1) % n_lon], -1),
                      torch.stack([torch.full_like(j, south), last + (j + 1) % n_lon, last + j], -1)])
    edge = 2 * r * math.sin(0.5 * max(2 * math.pi / n_lon, math.pi / n_lat)) * math.sqrt(2)    # >= the longest edge (a diagonal)
    return v.float(), tris.to(torch.int32), edge


def test_marching_cubes_sphere_against_fine_sphere():
    """Marching cubes of |x - c| - r (lattice spacing h = 1, r = 30) against the same sphere tessellated finely.  Bound on every
    distance, hence on the chamfer: a marching-cubes vertex interpolates the radial function linearly along an edge of length
    h, off by at most h^2 / (8 r); a point inside a triangle is further in by at most the sagitta of a chord <= sqrt(3) h
    (a cell's diagonal), 3 h^2 / (8 r); together h^2 / (2 r).  The fine mesh is inscribed, off by the sagitta of its longest
    edge, L^2 / (8 r)."""
    from tensoflow_b200.geometry import evaluate_mesh
    from tensoflow_b200.isosurface import marching_cubes
    dev = _cuda()
    centre, r, h = (35.3, 36.1, 35.7), 30.0, 1.0
    mv, mt = marching_cubes(sphere_sdf(72, centre, r).to(dev))
    fv, ft, edge = _uv_sphere(1024, 512, r, centre)
    bound = h * h / (2 * r) + edge * edge / (8 * r)
    res = evaluate_mesh(mv, mt, fv.to(dev), ft.to(dev), n_samples=500_000)
    assert res["chamfer"] < bound, (res, bound)
    assert res["normal_consistency"] > 0.999


def test_extracted_mesh_against_fp64_field_mesh():
    """ShapeRenderer.extract_geometry (fp32 field kernels + GPU marching cubes) against the oracle marching cubes of the same field
    evaluated in fp64 on the same lattice: the chamfer is within the vertex tolerance of tests/test_isosurface_gpu.py (0.1 voxel)."""
    from tensoflow_b200.geometry import evaluate_mesh
    from test_isosurface_gpu import HI, LO, R, _oracle_field, _shape
    dev = _cuda()
    shape = _shape(dev)
    verts, tris = shape.extract_geometry(LO, HI, R)
    ax = torch.linspace(-1.0, 1.0, R, device=dev).cpu()
    x, y, z = torch.meshgrid(ax, ax, ax, indexing="ij")
    pts = torch.stack([x, y, z], -1).reshape(-1, 3)
    inside = (torch.norm(pts.to(dev), dim=-1) < 1.0).cpu()
    u = torch.ones(pts.shape[0], dtype=torch.float64)
    with torch.no_grad():
        u[inside] = _oracle_field(shape).sdf(pts[inside].double(), None).reshape(-1)
    ref_v, ref_t = oracle_mc(u.reshape(R, R, R), 0.0)
    ref_v = ref_v / (R - 1.0) * 2.0 - 1.0
    res = evaluate_mesh(verts, tris, ref_v.to(dev), ref_t.to(dev), n_samples=200_000)
    voxel = 2.0 / (R - 1)
    assert res["chamfer"] < 0.1 * voxel, res
    assert res["normal_consistency"] > 0.99


def test_abi_errors_launch_nothing():
    from tensoflow_b200 import _lib
    from tensoflow_b200.geometry import sample_surface
    from tensoflow_b200.mc_ops import RayTracer
    from tensoflow_b200.synthetic import bumpy_sphere
    dev = _cuda()
    lib = _lib.load()
    v, t = bumpy_sphere(16, 8)
    rt = RayTracer(v, t)
    vd, td = v.to(dev), t.to(dev)
    p = torch.zeros(5, 3, device=dev)
    out = torch.empty(5, 3, device=dev)
    d = torch.empty(5, device=dev)
    ti = torch.empty(5, device=dev, dtype=torch.int64)
    cdf = torch.linspace(0.1, 1.0, t.shape[0], device=dev, dtype=torch.float64)
    u = torch.rand(5, 3, device=dev, dtype=torch.float64)
    P = lambda x: ctypes.c_void_p(x.data_ptr())
    s = _lib.stream_ptr()
    n0 = lib.tf_launch_count()
    # NULL handle / buffers, an empty mesh
    assert lib.tf_bvh_closest_point(None, P(p), 5, P(out), P(d), P(ti), s) != 0 and b"NULL handle" in lib.tf_last_error()
    assert lib.tf_bvh_closest_point(rt._h, None, 5, P(out), P(d), P(ti), s) != 0 and b"NULL pointer" in lib.tf_last_error()
    assert lib.tf_bvh_closest_point(rt._h, P(p), 5, P(out), P(d), None, s) != 0
    assert lib.tf_mesh_sample_surface(P(vd), P(td), 0, P(cdf), P(u), 5, P(out), P(ti), P(out), s) != 0
    assert b"empty mesh" in lib.tf_last_error()
    assert lib.tf_mesh_sample_surface(P(vd), P(td), t.shape[0], None, P(u), 5, P(out), P(ti), P(out), s) != 0
    h = ctypes.c_void_p()
    assert lib.tf_bvh_create(v.numpy().ctypes.data_as(ctypes.c_void_p), v.shape[0], t.numpy().ctypes.data_as(ctypes.c_void_p), 0,
                             ctypes.byref(h)) != 0 and b"empty mesh" in lib.tf_last_error()
    # n = 0 succeeds without a launch, even with NULL buffers
    assert lib.tf_bvh_closest_point(rt._h, None, 0, None, None, None, s) == 0
    assert lib.tf_mesh_sample_surface(None, None, t.shape[0], None, None, 0, None, None, None, s) == 0
    e = rt.closest_point(torch.zeros(0, 3, device=dev))
    assert e[0].shape == (0, 3) and e[1].shape == (0,) and e[2].shape == (0,)
    assert sample_surface(vd, td, 0)[0].shape == (0, 3)
    # mismatched shapes, out-of-range indices, zero area: the Python layer raises first
    with pytest.raises(RuntimeError, match=r"\[\.\.\., 3\]"):
        rt.closest_point(torch.zeros(4, 2, device=dev))
    with pytest.raises(RuntimeError, match="out of range"):
        sample_surface(vd, td + v.shape[0], 10)
    with pytest.raises(RuntimeError, match="area"):
        sample_surface(torch.zeros(4, 3, device=dev), torch.tensor([[0, 1, 2]], device=dev, dtype=torch.int32), 10)
    with pytest.raises(RuntimeError, match="empty mesh"):
        sample_surface(vd, td[:0], 10)
    assert lib.tf_launch_count() == n0
