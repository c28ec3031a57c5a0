"""Mesh simplification on the GPU (tf_mesh_simplify through geometry.simplify_mesh and ShapeRenderer.extract_geometry): vertex
bits, triangles, V', T' and the round count equal to the numpy oracle on every CPU-test mesh, a 150 k-triangle marching-cubes
sphere and bumpy_sphere(400, 201), at 50 %, 10 % and 1 % targets with and without max_error; two runs bit-identical; the
mesh properties on a 16 M-triangle bumpy sphere and a narrow-band 2048^3 torus; the max_error bound against the input mesh;
extract_geometry's simplification; rays that hit the full and the simplified sphere at depths within 2 max_error; and the
refusals that need a device."""
import concurrent.futures as cf
import functools
import multiprocessing as mp
import os

import pytest
import torch
import torch.nn.functional as F

from oracle import torch_oracle_simplify as O
from test_mesh_simplify_cpu import MESHES, boundary, euler, is_closed_manifold, mc_sphere

pytestmark = pytest.mark.gpu

FRACS = (0.5, 0.1, 0.01)


def _cuda():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    return torch.device("cuda:0")


def _bits(t):
    return t.contiguous().view(torch.int32)


@functools.lru_cache(maxsize=None)
def _sphere256():
    return mc_sphere(256)


def _bumpy400():
    from tensoflow_b200.synthetic import bumpy_sphere
    return bumpy_sphere(400, 201)


ALL = dict(MESHES, **{"mc-sphere-256": _sphere256, "bumpy-400x201": _bumpy400})


def _error_bound(v, t):
    """a quarter of the median edge length (0 on the flat grid, where every collapse is exact)"""
    p = v.double()[t.long()]
    return 0.25 * float((p[:, 1] - p[:, 0]).norm(dim=-1).median())


@pytest.fixture(scope="module")
def cases(request):
    """the oracle result of every selected (mesh, fraction, bound) case, computed in parallel processes (the oracle is numpy,
    one core each): a dict of futures of ((v, t, target, max_error), oracle output)"""
    wanted = sorted({(it.callspec.params["name"], it.callspec.params["frac"], it.callspec.params["bounded"])
                     for it in request.session.items if getattr(it, "originalname", "") == "test_equals_oracle"})
    inputs = {}
    for name in sorted({w[0] for w in wanted}):
        v, t = ALL[name]()
        inputs[name] = (v, t, 0.0 if name.startswith("flat-grid") else _error_bound(v, t))
    ex = cf.ProcessPoolExecutor(max_workers=max(1, min(len(wanted), os.cpu_count() or 1)), mp_context=mp.get_context("spawn"))
    out = {}
    for name, frac, bounded in wanted:
        v, t, e = inputs[name]
        args = (v, t, int(frac * t.shape[0]), e if bounded else None)
        out[(name, frac, bounded)] = (args, ex.submit(O.simplify, v.numpy(), t.numpy(), args[2], args[3]))
    yield out
    ex.shutdown(wait=True, cancel_futures=True)


@pytest.mark.parametrize("bounded", [False, True])
@pytest.mark.parametrize("frac", FRACS)
@pytest.mark.parametrize("name", sorted(ALL))
def test_equals_oracle(cases, name, frac, bounded):
    from tensoflow_b200.geometry import _simplify
    dev = _cuda()
    (v, t, target, err), fut = cases[(name, frac, bounded)]
    want_v, want_t, want_rounds = fut.result()
    got_v, got_t, rounds = _simplify(v.to(dev), t.to(dev), target, err)
    assert got_v.dtype == torch.float32 and got_t.dtype == torch.int32 and got_v.device == dev
    assert (got_v.shape[0], got_t.shape[0], rounds) == (want_v.shape[0], want_t.shape[0], want_rounds)
    assert torch.equal(got_t.cpu(), torch.from_numpy(want_t))
    assert torch.equal(_bits(got_v.cpu()), _bits(torch.from_numpy(want_v)))


def test_two_runs_bit_identical():
    from tensoflow_b200.geometry import _simplify
    dev = _cuda()
    v, t = _bumpy400()
    v, t = v.to(dev), t.to(dev)
    a = _simplify(v, t, t.shape[0] // 20, None)
    b = _simplify(v, t, t.shape[0] // 20, None)
    assert a[2] == b[2] and torch.equal(a[1], b[1]) and torch.equal(_bits(a[0]), _bits(b[0]))


def test_workspace_too_small_is_refused():
    import ctypes
    from tensoflow_b200 import _lib
    dev = _cuda()
    lib = _lib.load()
    v, t = _bumpy400()
    v, t = v.to(dev), t.to(dev)
    ws = ctypes.c_size_t()
    assert lib.tf_mesh_simplify_sizes(v.shape[0], t.shape[0], ctypes.byref(ws)) == 0
    buf = torch.empty(ws.value, device=dev, dtype=torch.uint8)
    ov, ot = torch.empty_like(v), torch.empty_like(t)
    nv, nt, nr = ctypes.c_int64(), ctypes.c_int64(), ctypes.c_int32()
    n0 = lib.tf_launch_count()
    p = lambda x: ctypes.c_void_p(x.data_ptr())
    assert lib.tf_mesh_simplify(p(v), v.shape[0], p(t), t.shape[0], 100, float("inf"), p(buf), ws.value - 1, p(ov), p(ot),
                                ctypes.byref(nv), ctypes.byref(nt), ctypes.byref(nr), None) != 0
    assert b"workspace" in lib.tf_last_error()
    assert lib.tf_launch_count() == n0


def test_index_out_of_range_is_refused():
    from tensoflow_b200 import _lib
    from tensoflow_b200.geometry import simplify_mesh
    dev = _cuda()
    v, t = _bumpy400()
    t = t.clone()
    t[7, 1] = v.shape[0]
    n0 = _lib.launch_count()
    with pytest.raises(RuntimeError, match="out of range"):
        simplify_mesh(v.to(dev), t.to(dev), 100)
    with pytest.raises(RuntimeError, match="empty"):
        simplify_mesh(v.to(dev), t[:0].to(dev), 100)
    assert _lib.launch_count() == n0


def _properties(v0, t0, v1, t1, target, closed):
    """the oracle-free checks on large meshes: T' at the target, Euler characteristic, components, manifoldness, boundary"""
    from tensoflow_b200.geometry import mesh_components
    assert t1.shape[0] in (target, target + 1)
    a, b = (x.cpu().numpy() for x in (t0, t1))
    assert euler(None, b) == euler(None, a)
    assert int((mesh_components(v1, t1)[1] > 0).sum()) == int((mesh_components(v0, t0)[1] > 0).sum())
    if closed:
        assert is_closed_manifold(b)
    else:
        bp0, bv0 = boundary(v0.cpu().numpy(), a)
        bp1, _ = boundary(v1.cpu().numpy(), b)
        assert bp0 == bp1


def _torus_2048(dev):
    """narrow-band marching cubes of an analytic torus (tube radius 0.2 around a circle of radius 0.5) on a 2048^3 lattice"""
    from tensoflow_b200.isosurface import marching_cubes_narrowband

    def fn(p):
        q = torch.stack([p[:, :2].norm(dim=-1) - 0.5, p[:, 2]], -1)
        return q.norm(dim=-1) - 0.2
    ax = torch.linspace(-1, 1, 2048, device=dev)
    v, t = marching_cubes_narrowband(fn, (ax, ax, ax))
    return v / 2047.0 * 2.0 - 1.0, t


def test_large_meshes_keep_their_properties():
    """16 M-triangle bumpy sphere (open: pole holes) and a narrow-band 2048^3 torus to 1 %"""
    from tensoflow_b200.geometry import simplify_mesh
    from tensoflow_b200.synthetic import bumpy_sphere
    dev = _cuda()
    v, t = bumpy_sphere(4000, 2001)
    v, t = v.to(dev), t.to(dev)
    assert t.shape[0] >= 16_000_000
    target = t.shape[0] // 100
    sv, st = simplify_mesh(v, t, target)
    _properties(v, t, sv, st, target, closed=False)
    del v, t, sv, st
    v, t = _torus_2048(dev)
    assert t.shape[0] > 5_000_000
    target = t.shape[0] // 100
    sv, st = simplify_mesh(v, t, target)
    _properties(v, t, sv, st, target, closed=True)


def _bounded_meshes(dev):
    v, t = _sphere256()
    yield "sphere", v.to(dev) / 255.0 * 2.0 - 1.0, t.to(dev)
    yield "torus", *_torus_2048(dev)


def test_max_error_bounds_the_distance_to_the_input():
    """every output vertex lies within max_error of the input mesh (closest point on its BVH); evaluate_mesh is reported"""
    from tensoflow_b200.geometry import evaluate_mesh, simplify_mesh
    from tensoflow_b200.mc_ops import RayTracer
    dev = _cuda()
    for name, v, t in _bounded_meshes(dev):
        e = 2.0 / (255.0 if name == "sphere" else 2047.0) / 2                 # half a voxel
        sv, st = simplify_mesh(v, t, 0, max_error=e)
        assert st.shape[0] < t.shape[0] // 4, (name, st.shape[0], t.shape[0])
        _, dist, _ = RayTracer(v, t).closest_point(sv)
        assert float(dist.max()) <= e * (1 + 1e-5), (name, float(dist.max()), e)
        stats = evaluate_mesh(sv, st, v, t, n_samples=200_000)
        print(f"{name}: {t.shape[0]} -> {st.shape[0]} triangles at max_error {e:.3g}: chamfer {stats['chamfer']:.3g}, "
              f"normal consistency {stats['normal_consistency']:.6f}")
        assert stats["chamfer"] < e


def test_rays_hit_the_full_and_the_simplified_sphere_alike():
    """rays from radius 1.5 towards the centre of the radius-0.5 sphere: near-side depths about 1, far side about 2.  The
    tracer's fp32 Moller-Trumbore test is not watertight, so a ray through a shared edge can slip to the far side of either
    mesh; such rays are counted (a handful in 5e5) and left out of the depth comparison"""
    from tensoflow_b200.geometry import simplify_mesh
    from tensoflow_b200.mc_ops import RayTracer
    dev = _cuda()
    v, t = _sphere256()
    v, t = v.to(dev) / 255.0 * 2.0 - 1.0, t.to(dev)
    e = 1.0 / 255.0
    sv, st = simplify_mesh(v, t, 0, max_error=e)
    g = torch.Generator().manual_seed(3)
    o = F.normalize(torch.randn(500_000, 3, generator=g), dim=-1).to(dev) * 1.5
    d = F.normalize(-o, dim=-1)
    full = RayTracer(v, t).trace(o, d)[2]
    simple = RayTracer(sv, st).trace(o, d)[2]
    assert bool((full < 10).all()) and bool((simple < 10).all())
    near = (full < 1.5) & (simple < 1.5)
    print(f"rays through a crack: full {int((full >= 1.5).sum())}, simplified {int((simple >= 1.5).sum())} of {o.shape[0]}")
    assert int((~near).sum()) <= 20
    assert float((full - simple)[near].abs().max()) <= 2 * e


def _analytic_shape(dev):
    from test_isosurface_narrowband_gpu import _small_shape
    shape = _small_shape(dev)

    def fn(p):
        big = (p - torch.tensor([0.02, -0.03, 0.01], device=p.device)).norm(dim=-1) - 0.5
        small = (p - torch.tensor([0.0, 0.0, 0.82], device=p.device)).norm(dim=-1) - 0.05
        return torch.minimum(big, small)
    shape.sdf_network.sdf = lambda p, lvl: fn(p)[:, None]
    return shape


@pytest.mark.parametrize("R", [256, 1291])
def test_extract_geometry_simplifies_after_the_floaters_go(R):
    """R = 256 runs the dense path, 1291 the narrow band"""
    from tensoflow_b200.geometry import simplify_mesh
    shape = _analytic_shape(_cuda())
    lo, hi = [-1.0] * 3, [1.0] * 3
    v, t = shape.extract_geometry(lo, hi, R, min_component_fraction=0.5)
    for kw in ({"target_triangles": t.shape[0] // 10}, {"max_error": 1.0 / R}, {"target_triangles": 1000, "max_error": 1.0 / R}):
        got_v, got_t = shape.extract_geometry(lo, hi, R, min_component_fraction=0.5, **kw)
        want_v, want_t = simplify_mesh(v, t, kw.get("target_triangles", 0), kw.get("max_error"))
        assert torch.equal(got_t, want_t) and torch.equal(_bits(got_v), _bits(want_v)), kw
        assert got_t.shape[0] < t.shape[0]
    v0, t0 = shape.extract_geometry(lo, hi, R, min_component_fraction=0.5, target_triangles=None, max_error=None)
    assert torch.equal(t0, t) and torch.equal(_bits(v0), _bits(v))
