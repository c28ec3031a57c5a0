"""Connected components of meshes on the GPU (tf_mesh_components through geometry.mesh_components) and the clean-up built on
them (geometry.remove_small_components, ShapeRenderer.extract_geometry(min_component_fraction=...)): root and tri_count equal
to the scipy oracle exactly on marching-cubes meshes and on adversarial soups for union-find, two runs bit-identical, the
filter byte-equal to the oracle and to the mesh of the large component's volume alone, extract_geometry unchanged without the
argument and on single-component fields, a BVH on the cleaned mesh that traces what the large sphere alone traces, and the
refusals before any launch."""
import numpy as np
import pytest
import torch
import torch.nn.functional as F

from oracle import torch_oracle_cc as O

pytestmark = pytest.mark.gpu

LO, HI = [-1.0, -1.0, -1.0], [1.0, 1.0, 1.0]
BIG_C, BIG_R = (0.02, -0.03, 0.01), 0.5


def _cuda():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    return torch.device("cuda:0")


def _bits(t):
    return t.contiguous().view(torch.int32)


def _check(v, t, what):
    """mesh_components on the device == the oracle, exactly; returns (root, tri_count) on the device"""
    from tensoflow_b200.geometry import mesh_components
    dev = _cuda()
    v, t = v.to(dev), t.to(dev)
    root, cnt = mesh_components(v, t)
    assert root.dtype == torch.int32 and cnt.dtype == torch.int32 and root.device == dev
    want_root, want_cnt = O.mesh_components(v.shape[0], t.cpu().numpy())
    got_root, got_cnt = root.cpu().numpy(), cnt.cpu().numpy()
    bad = np.nonzero(got_root != want_root)[0]
    assert bad.size == 0, f"{what}: root differs at {bad.size} vertices, first {bad[:4].tolist()}"
    bad = np.nonzero(got_cnt != want_cnt)[0]
    assert bad.size == 0, f"{what}: tri_count differs at {bad.size} vertices, first {bad[:4].tolist()}"
    return root, cnt


def _sphere(p, c, r):
    return (p - torch.tensor(c, device=p.device, dtype=p.dtype)).norm(dim=-1) - r


def _floater_spheres(n=100, seed=0):
    """n tiny spheres (radius 0.025-0.04) in the shell 0.72 <= |c| <= 0.9, at least 0.18 from the big sphere's surface and
    0.05 apart from each other (so each is a component of its own)"""
    g = torch.Generator().manual_seed(seed)
    out = []
    while len(out) < n:
        c = torch.rand(3, generator=g) * 1.8 - 0.9
        r = 0.025 + 0.015 * float(torch.rand(1, generator=g))
        if 0.72 <= float(c.norm()) <= 0.9 and all(float((c - torch.tensor(q)).norm()) > r + s + 0.05 for q, s in out):
            out.append((tuple(float(x) for x in c), r))
    return out


FLOATERS = _floater_spheres()


def _field(kind):
    """value of an analytic field at points [N,3] (fp32, running minimum over spheres: where the big sphere's value is the
    smallest, the union's value is that value bit for bit)"""
    def fn(p):
        if kind == "two-spheres":
            return torch.minimum(_sphere(p, BIG_C, BIG_R), _sphere(p, (0.0, 0.0, 0.82), 0.1))
        if kind == "nested-shells":
            r = _sphere(p, (0.0, 0.0, 0.0), 0.0)
            return torch.minimum((r - 0.6).abs() - 0.05, r - 0.3)
        if kind == "torus":
            q = torch.stack([p[:, :2].norm(dim=-1) - 0.5, p[:, 2]], -1)
            return q.norm(dim=-1) - 0.2
        u = _sphere(p, BIG_C, BIG_R)
        if kind == "big":
            return u
        if kind == "floaters":
            for c, r in FLOATERS:
                u = torch.minimum(u, _sphere(p, c, r))
            return u
        if kind == "big-and-far":
            return torch.minimum(u, _sphere(p, (0.8, 0.8, 0.0), 0.12))
        raise KeyError(kind)
    return fn


def _mc(kind, R=128):
    """marching-cubes mesh of the field on the lattice linspace(-1, 1, R)^3, vertices in those coordinates"""
    from tensoflow_b200.isosurface import marching_cubes
    dev = _cuda()
    x = torch.linspace(-1, 1, R, device=dev)
    p = torch.stack(torch.meshgrid(x, x, x, indexing="ij"), -1).reshape(-1, 3)
    v, t = marching_cubes(_field(kind)(p).reshape(R, R, R), 0.0)
    return v / (R - 1.0) * 2.0 - 1.0, t


@pytest.mark.parametrize("kind,n_comp", [("two-spheres", 2), ("nested-shells", 3), ("torus", 1), ("floaters", 101)])
def test_marching_cubes_meshes_equal_oracle(kind, n_comp):
    v, t = _mc(kind)
    root, cnt = _check(v, t, kind)
    assert int((cnt > 0).sum()) == n_comp                              # every sphere, shell and floater is a component


def _path(n, order, seed=0):
    if order == "in-order":
        p = torch.arange(n)
    elif order == "reversed":
        p = torch.arange(n).flip(0)
    else:
        p = torch.randperm(n, generator=torch.Generator().manual_seed(seed))
    p = p.to(torch.int32)
    return torch.stack([p[:-1], p[1:], p[1:]], -1).contiguous()


def _soup(name):
    n = 1 << 20
    v = torch.zeros(n, 3)
    if name.startswith("path-"):
        return v, _path(n, name[5:])
    if name in ("star-first", "star-last"):
        c = 0 if name == "star-first" else n - 1
        leaves = torch.arange(1, n, dtype=torch.int32) - (0 if c == 0 else 1)
        leaves = leaves[torch.randperm(n - 1, generator=torch.Generator().manual_seed(1))]
        return v, torch.stack([torch.full_like(leaves, c), leaves, leaves], -1).contiguous()
    if name == "one-triangle-1e5":
        return v[:10], torch.tensor([[5, 1, 3]], dtype=torch.int32).repeat(100_000, 1)
    if name == "random":
        g = torch.Generator().manual_seed(2)
        return v, torch.randint(0, n, (n // 2, 3), generator=g, dtype=torch.int32)   # a giant component and many small ones
    raise KeyError(name)


SOUPS = ["path-in-order", "path-reversed", "path-permuted", "star-first", "star-last", "one-triangle-1e5", "random"]


@pytest.mark.parametrize("name", SOUPS)
def test_union_find_soups_equal_oracle(name):
    v, t = _soup(name)
    root, cnt = _check(v, t, name)
    if name.startswith(("path", "star")):
        assert int(root.max()) == 0 and int(cnt[0]) == t.shape[0]      # one component rooted at vertex 0
    if name == "one-triangle-1e5":
        assert root.cpu().tolist() == [0, 1, 2, 1, 4, 1, 6, 7, 8, 9] and int(cnt[1]) == 100_000


def test_above_2_24_triangles_equals_oracle():
    """a bumpy sphere of 16.8 M triangles with its vertices relabelled at random, beside a copy with the labels as built"""
    from tensoflow_b200.synthetic import bumpy_sphere
    v, t = bumpy_sphere(4200, 2000)
    V = v.shape[0]
    perm = torch.randperm(V, generator=torch.Generator().manual_seed(3)).to(torch.int32)
    t2 = torch.cat([t, perm[t.long()] + V])
    assert t2.shape[0] > 1 << 24
    root, cnt = _check(torch.cat([v, v]), t2, "bumpy4200x2000 twice")
    assert int((cnt > 0).sum()) == 2


def test_two_runs_bit_identical():
    from tensoflow_b200.geometry import mesh_components
    dev = _cuda()
    for v, t in (_mc("floaters"), _soup("path-permuted"), _soup("random")):
        v, t = v.to(dev), t.to(dev)
        a, b = mesh_components(v, t), mesh_components(v, t)
        assert torch.equal(a[0], b[0]) and torch.equal(a[1], b[1])


@pytest.mark.parametrize("frac", [1.0, 0.5, 0.01, 1e-9])
def test_remove_small_components_equals_oracle(frac):
    from tensoflow_b200.geometry import remove_small_components
    dev = _cuda()
    for name, (v, t) in (("floaters", _mc("floaters")), ("random", _soup("random"))):
        v, t = v.to(dev), t.to(dev)
        if name == "random":
            v = torch.randn(v.shape, generator=torch.Generator().manual_seed(4)).to(dev)
        kv, kt = remove_small_components(v, t, frac)
        wv, wt = O.remove_small_components(v.cpu().numpy(), t.cpu().numpy(), frac)
        assert kv.dtype == torch.float32 and kt.dtype == torch.int32
        assert kv.cpu().numpy().tobytes() == wv.tobytes(), (name, frac)
        assert kt.cpu().numpy().tobytes() == wt.tobytes(), (name, frac)


def test_largest_component_is_the_large_sphere_alone():
    """min_fraction = 1.0 on the union of two distant spheres, and on the big sphere with 100 floaters, is the marching-cubes
    mesh of the big sphere's volume alone: same vertices, triangles and order"""
    from tensoflow_b200.geometry import remove_small_components
    bv, bt = _mc("big")
    for kind in ("big-and-far", "floaters"):
        v, t = _mc(kind)
        assert t.shape[0] > bt.shape[0]
        kv, kt = remove_small_components(v, t, 1.0)
        assert torch.equal(kt, bt) and torch.equal(_bits(kv), _bits(bv)), kind


def _analytic_shape(kind):
    from test_isosurface_narrowband_gpu import _small_shape
    shape = _small_shape(_cuda())
    fn = _field(kind)
    shape.sdf_network.sdf = lambda p, lvl: fn(p)[:, None]
    return shape


def test_extract_geometry_without_the_argument_is_unchanged():
    from test_isosurface_narrowband_gpu import _small_shape
    from tensoflow_b200.isosurface import marching_cubes
    shape = _small_shape(_cuda())
    R = 192
    with torch.no_grad():
        dv, dt = marching_cubes(shape.extract_fields(LO, HI, R))
    v0, t0 = shape.extract_geometry(LO, HI, R)
    v1, t1 = shape.extract_geometry(LO, HI, R, 0.0, None)
    v2, t2 = shape.extract_geometry(LO, HI, R, min_component_fraction=None)
    assert dt.shape[0] > 1000
    for v, t in ((v0, t0), (v1, t1), (v2, t2)):
        assert torch.equal(t, dt) and torch.equal(_bits(v), _bits(dv / (R - 1.0) * 2.0 - 1.0))


@pytest.mark.parametrize("R", [256, 1291])
def test_extract_geometry_filters_on_dense_and_narrow_band(R):
    """R = 256 runs the dense path, 1291 the narrow band.  A single-component field comes back unchanged at 0.01; the big
    sphere with floaters comes back at 1.0 as the big sphere's mesh alone, vertices rescaled the same way"""
    single = _analytic_shape("big")
    v, t = single.extract_geometry(LO, HI, R)
    _, cnt = _check(v, t, f"big {R}")
    assert int((cnt > 0).sum()) == 1
    fv, ft = single.extract_geometry(LO, HI, R, min_component_fraction=0.01)
    assert torch.equal(ft, t) and torch.equal(_bits(fv), _bits(v))
    floaters = _analytic_shape("floaters")
    raw_v, raw_t = floaters.extract_geometry(LO, HI, R)
    assert raw_t.shape[0] > t.shape[0]
    fv, ft = floaters.extract_geometry(LO, HI, R, min_component_fraction=1.0)
    assert torch.equal(ft, t) and torch.equal(_bits(fv), _bits(v))


def test_ray_tracer_on_the_cleaned_mesh_traces_the_large_sphere():
    from tensoflow_b200.geometry import remove_small_components
    from tensoflow_b200.mc_ops import RayTracer
    dev = _cuda()
    bv, bt = _mc("big")
    v, t = _mc("floaters")
    kv, kt = remove_small_components(v, t, 0.5)
    g = torch.Generator().manual_seed(5)
    n = 200_000
    o = F.normalize(torch.randn(n, 3, generator=g), dim=-1) * 1.5
    d = F.normalize(torch.randn(n, 3, generator=g) * 0.3 - o, dim=-1)
    o, d = o.to(dev), d.to(dev)
    big = RayTracer(bv, bt).trace(o, d)
    clean = RayTracer(kv, kt).trace(o, d)
    raw = RayTracer(v, t).trace(o, d)
    for x, y in zip(big, clean):
        assert torch.equal(x, y)
    assert float((big[2] < 10).float().mean()) > 0.3
    assert int((raw[2] != big[2]).sum()) > 100                          # the floaters do intercept rays


def test_refusals_launch_nothing():
    from tensoflow_b200 import _lib
    from tensoflow_b200.geometry import mesh_components, remove_small_components
    dev = _cuda()
    v, t = (x.to(dev) for x in _mc("two-spheres", R=32))
    n0 = _lib.launch_count()
    t64 = t.long()
    t64[3, 1] = (1 << 32) + 1                                           # int32 would wrap it into range
    for bad_v, bad_t, match in ((v, t + 1, "out of range"), (v, t - 1, "out of range"), (v, t64, "out of range"),
                                (v, t.reshape(-1, 6), r"\[T,3\]"), (v[:, :2], t, r"\[V,3\]"), (v[:0], t, "empty mesh"),
                                (v, t[:0], "empty mesh"), (v, t.float(), "integer triangles"),
                                (torch.zeros(1, 3, device=dev).expand(1 << 31, 3), t, "2\\^31")):
        with pytest.raises(RuntimeError, match=match):
            mesh_components(bad_v, bad_t)
        with pytest.raises(RuntimeError, match=match):
            remove_small_components(bad_v, bad_t, 1.0)
    for frac in (0.0, -0.1, 1.5):
        with pytest.raises(ValueError, match="min_fraction"):
            remove_small_components(v, t, frac)
    assert _lib.launch_count() == n0
    mesh_components(v, t)
    assert _lib.launch_count() == n0 + 4
