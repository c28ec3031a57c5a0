"""BVH build on the device (tf_bvh_build, what mc_ops.RayTracer runs for CUDA meshes) against the host build (tf_bvh_create,
for numpy arrays and CPU tensors): byte-equal nodes, triangles and perm on meshes full of tied centroids and on every small
triangle count, identical trace / closest_point / MaterialRenderer.nvs / evaluate_mesh results from the two handles,
determinism, the refusals before any launch, and placement on a second device."""
import ctypes

import numpy as np
import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu


def _cuda():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    return torch.device("cuda:0")


def _export(rt):
    """(nodes [N,8] fp32, tris [T,12] fp32, perm [T] int32) of a handle, through tf_bvh_export"""
    from tensoflow_b200 import _lib
    lib = _lib.load()
    nn, nt = ctypes.c_int64(), ctypes.c_int64()
    _lib.check(lib.tf_bvh_export(rt._h, ctypes.byref(nn), ctypes.byref(nt), None, None, None), "tf_bvh_export")
    nodes = np.empty((nn.value, 8), np.float32)
    tris = np.empty((nt.value, 12), np.float32)
    perm = np.empty(nt.value, np.int32)
    P = lambda a: a.ctypes.data_as(ctypes.c_void_p)
    _lib.check(lib.tf_bvh_export(rt._h, None, None, P(nodes), P(tris), P(perm)), "tf_bvh_export")
    return nodes, tris, perm


def _assert_same(a, b, what):
    for x, y, name in zip(a, b, ("nodes", "tris", "perm")):
        assert x.shape == y.shape, (what, name, x.shape, y.shape)
        if x.tobytes() != y.tobytes():
            bad = np.nonzero((x.view(np.uint32) != y.view(np.uint32)).reshape(x.shape[0], -1).any(1))[0]
            raise AssertionError(f"{what}: {name} differ in {bad.size} rows, first {bad[:4].tolist()}")


def _both_builds(v, t):
    from tensoflow_b200.mc_ops import RayTracer
    dev = _cuda()
    host = RayTracer(v.cpu(), t.cpu())
    devb = RayTracer(v.to(dev), t.to(dev))
    assert host._device is None and devb._device == dev
    return host, devb


def _check_tree(v, t, what):
    host, devb = _both_builds(v, t)
    _assert_same(_export(host), _export(devb), what)


def _soup(n, seed):
    g = torch.Generator().manual_seed(seed)
    c = torch.rand(n, 1, 3, generator=g) * 2 - 1
    tri = c + 0.1 * torch.randn(n, 3, 3, generator=g)
    return tri.reshape(-1, 3).float(), torch.arange(3 * n, dtype=torch.int32).reshape(-1, 3)


def _mc_mesh(kind, R=128):
    from tensoflow_b200.isosurface import marching_cubes
    dev = _cuda()
    x = torch.linspace(-1, 1, R, device=dev)
    X, Y, Z = torch.meshgrid(x, x, x, indexing="ij")
    u = (X ** 2 + Y ** 2 + Z ** 2).sqrt() - 0.6 if kind == "sphere" else Z - 0.1037
    return marching_cubes(u, 0.0)


def _named_mesh(name):
    from tensoflow_b200.synthetic import bumpy_sphere
    from test_mesh_query_gpu import _soup as query_soup
    if name.startswith("bumpy"):
        nu, nv = (int(s) for s in name[5:].split("x"))
        return bumpy_sphere(nu, nv)
    if name == "query-soup":
        return query_soup(2000, 0)
    if name in ("mc-sphere", "mc-plane"):
        return _mc_mesh(name[3:])
    if name == "identical":
        v = torch.tensor([[0.1, 0.2, 0.3], [0.5, -0.2, 0.1], [-0.3, 0.4, 0.9]])
        return v.repeat(777, 1), torch.arange(3 * 777, dtype=torch.int32).reshape(-1, 3)
    if name == "degenerate":
        # zero-area triangles (collinear, a repeated vertex, a point) and each triangle twice, in scattered order
        v, t = _soup(600, 3)
        v = v.reshape(-1, 3, 3)
        v[:100, 2] = v[:100, 0] + 0.25 * (v[:100, 1] - v[:100, 0])
        v[100:200, 1] = v[100:200, 0]
        v[200:300, 1:] = v[200:300, :1]
        v = v.reshape(-1, 3)
        t = torch.cat([t, t.flip(1), t])[torch.randperm(1800, generator=torch.Generator().manual_seed(4))]
        return v, t.contiguous()
    if name == "signed-zeros":
        # coordinates on a coarse lattice with a third of the zeros negative: ties between -0 and +0 everywhere
        g = torch.Generator().manual_seed(5)
        v = torch.randint(-2, 3, (3000, 3), generator=g).float() * 0.5
        v = torch.where((v == 0) & (torch.rand(v.shape, generator=g) < 0.33), torch.tensor(-0.0), v)
        return v, torch.randint(0, 3000, (2000, 3), generator=g, dtype=torch.int32)
    raise KeyError(name)


@pytest.mark.parametrize("name", ["bumpy40x20", "bumpy200x100", "bumpy1000x500", "query-soup", "mc-sphere", "mc-plane",
                                  "identical", "degenerate", "signed-zeros"])
def test_device_build_equals_host_build(name):
    v, t = _named_mesh(name)
    _check_tree(v, t, name)


def test_device_build_equals_host_build_every_small_n():
    """every n from 9 to 70: all the shapes of the top of a tree (leaves of 2 to 4 beside inner nodes of 5 on one level)"""
    v, t = _soup(70, 6)
    for n in range(9, 71):
        _check_tree(v, t[:n], f"n={n}")


def test_device_build_equals_host_build_around_powers_of_two():
    """n = 4 * 2^k +- 1 up to 2^20: the sizes where a level starts or stops holding leaves beside inner nodes"""
    v, t = _soup((1 << 20) + 1, 7)
    for k in range(1, 19):
        for n in (4 * 2 ** k - 1, 4 * 2 ** k + 1):
            if n > 8:
                _check_tree(v, t[:n], f"n={n}")


def test_device_build_equals_host_build_above_2_24_triangles():
    from tensoflow_b200.synthetic import bumpy_sphere
    v, t = bumpy_sphere(4200, 2000)
    assert t.shape[0] > 1 << 24
    _check_tree(v, t, "bumpy4200x2000")


def test_device_build_is_deterministic():
    from tensoflow_b200.mc_ops import RayTracer
    dev = _cuda()
    v, t = (x.to(dev) for x in _mc_mesh("sphere"))
    _assert_same(_export(RayTracer(v, t)), _export(RayTracer(v, t)), "two device builds")


def test_trace_identical_from_both_builds():
    """the ray family of test_mc_gpu.test_bvh_trace_matches_brute_force"""
    from test_mc_gpu import bumpy_sphere
    dev = _cuda()
    verts, tris = bumpy_sphere()
    host, devb = _both_builds(verts, tris)
    g = torch.Generator().manual_seed(0)
    n = 4000
    o = F.normalize(torch.randn(n, 3, generator=g), dim=-1) * 1.5
    tgt = torch.randn(n, 3, generator=g) * 0.35
    d = F.normalize(tgt - o, dim=-1)
    o[: n // 4] = F.normalize(torch.randn(n // 4, 3, generator=g), dim=-1) * 0.2
    a = host.trace(o.to(dev), d.to(dev))
    b = devb.trace(o.to(dev), d.to(dev))
    assert float((a[2] < 10).float().mean()) > 0.3
    for x, y in zip(a, b):
        assert torch.equal(x, y)


def test_closest_point_identical_from_both_builds():
    """10^6 queries against the 10^6-triangle bumpy sphere"""
    from tensoflow_b200.synthetic import bumpy_sphere
    from test_mesh_query_gpu import _queries
    dev = _cuda()
    v, t = bumpy_sphere(1000, 501)
    host, devb = _both_builds(v, t)
    q = _queries(v, t, 1_000_000, 11).to(dev)
    for x, y in zip(host.closest_point(q), devb.closest_point(q)):
        assert torch.equal(x, y)


def test_material_nvs_identical_from_both_builds():
    from test_nvs_gpu import SHAPE_CFG, MAT_SHADER
    from tensoflow_b200.material import MaterialRenderer
    from tensoflow_b200.shape_renderer import ShapeRenderer
    from tensoflow_b200.synthetic import bumpy_sphere, perturb_field
    dev = _cuda()
    torch.manual_seed(0)
    shape = ShapeRenderer(dict(device=dev, shader_config=dict(env_res=16, env_min_res=4), **SHAPE_CFG))
    perturb_field(shape.sdf_network, seed=2, noise=5e-3)
    verts, tris = bumpy_sphere(48, 24, r=0.22, bump=0.05)
    h, w = 12, 14
    K = np.array([[18.0, 0, w / 2], [0, 18.0, h / 2], [0, 0, 1]], np.float32)
    pose = np.array([[1, 0, 0, 0.02], [0, 1, 0, -0.03], [0, 0, 1, 1.5]], np.float32)

    def noise_fn(r0, n):
        g = torch.Generator().manual_seed(100 + r0)
        return dict(az_diffuse=torch.rand(n, 1, 1, generator=g).to(dev), az_specular=torch.rand(n, 1, 1, generator=g).to(dev))

    imgs = []
    for vt in ((verts, tris), (verts.to(dev), tris.to(dev))):
        torch.manual_seed(1)
        mat = MaterialRenderer(dict(device=dev, shader_cfg=dict(MAT_SHADER), gridSize=SHAPE_CFG['gridSize']), *vt)
        mat.init_sdf(shape.ckpt_to_save())
        mat.shader_network.outer_light.build_mips_direct()
        torch.manual_seed(2)
        imgs.append(mat.nvs(pose, K, h, w, noise_fn=noise_fn))
    assert imgs[0].keys() == imgs[1].keys()
    hit = np.abs(imgs[0]['normal'] - np.array([0, 0, 1.0])).max(-1) > 1e-6
    assert hit.sum() > 10
    for k in imgs[0]:
        assert imgs[0][k].tobytes() == imgs[1][k].tobytes(), k


def test_evaluate_mesh_identical_from_both_builds(monkeypatch):
    from tensoflow_b200 import mc_ops
    from tensoflow_b200.geometry import evaluate_mesh
    from tensoflow_b200.synthetic import bumpy_sphere
    dev = _cuda()
    pv, pt = (x.to(dev) for x in _mc_mesh("sphere"))
    pv = pv / 127 * 2 - 1
    gv, gt = (x.to(dev) for x in bumpy_sphere(200, 100, r=0.6, bump=0.02))
    on_device = evaluate_mesh(pv, pt, gv, gt, n_samples=200_000)

    class HostBuilt(mc_ops.RayTracer):
        def __init__(self, vertices, triangles):
            super().__init__(vertices.cpu(), triangles.cpu())

    monkeypatch.setattr(mc_ops, "RayTracer", HostBuilt)
    on_host = evaluate_mesh(pv, pt, gv, gt, n_samples=200_000)
    assert on_device == on_host
    assert 0 < on_device["chamfer"] < 0.05


def test_refusals_launch_nothing():
    from tensoflow_b200 import _lib
    from tensoflow_b200.mc_ops import RayTracer
    from tensoflow_b200.synthetic import bumpy_sphere
    dev = _cuda()
    lib = _lib.load()
    v, t = bumpy_sphere(16, 8)
    vd, td = v.to(dev), t.to(dev)
    n0 = lib.tf_launch_count()
    nan, inf = vd.clone(), vd.clone()
    nan[int(t[5, 1]), 2] = float("nan")
    inf[int(t[7, 0]), 0] = float("-inf")
    for bad_v, bad_t, match in ((vd, td + 1, "out of range"), (vd, td - 1, "out of range"), (nan, td, "non-finite"),
                                (inf, td, "non-finite"), (vd[:0], td[:0], "empty mesh"), (vd, td[:0], "empty mesh"),
                                (vd, td[:8], "at least 8")):
        with pytest.raises(RuntimeError, match=match):
            RayTracer(bad_v, bad_t)
    # a non-finite vertex no triangle references is not an error
    unused = torch.cat([vd, torch.full((1, 3), float("nan"), device=dev)])
    RayTracer(unused, td)
    n1 = lib.tf_launch_count()
    assert n1 > n0
    # the raw entry points: NULL pointers and empty meshes return an error without a launch
    P = lambda x: ctypes.c_void_p(x.data_ptr())
    nn, wsb, h = ctypes.c_int64(), ctypes.c_size_t(), ctypes.c_void_p()
    assert lib.tf_bvh_build_sizes(td.shape[0], None, ctypes.byref(wsb)) != 0 and b"NULL" in lib.tf_last_error()
    assert lib.tf_bvh_build_sizes(0, ctypes.byref(nn), ctypes.byref(wsb)) != 0 and b"empty mesh" in lib.tf_last_error()
    assert lib.tf_bvh_build_sizes(1 << 31, ctypes.byref(nn), ctypes.byref(wsb)) != 0 and b"2^31" in lib.tf_last_error()
    assert lib.tf_bvh_build_sizes(td.shape[0], ctypes.byref(nn), ctypes.byref(wsb)) == 0
    ws = torch.empty(wsb.value, device=dev, dtype=torch.uint8)
    nodes = torch.empty(nn.value, 8, device=dev)
    tris = torch.empty(td.shape[0], 12, device=dev)
    perm = torch.empty(td.shape[0], device=dev, dtype=torch.int32)
    s = _lib.stream_ptr()
    args = [P(vd), vd.shape[0], P(td), td.shape[0], P(ws), wsb.value, P(nodes), P(tris), P(perm), s]
    for i in (0, 2, 4, 6, 7, 8):
        a = list(args)
        a[i] = None
        assert lib.tf_bvh_build(*a) != 0 and b"NULL pointer" in lib.tf_last_error()
    a = list(args)
    a[5] = wsb.value - 1
    assert lib.tf_bvh_build(*a) != 0 and b"workspace" in lib.tf_last_error()
    assert lib.tf_bvh_create_from_device(None, nn.value, P(tris), P(perm), td.shape[0], s, ctypes.byref(h)) != 0
    assert b"NULL pointer" in lib.tf_last_error()
    assert lib.tf_bvh_create_from_device(P(nodes), nn.value, P(tris), P(perm), td.shape[0], s, None) != 0
    assert lib.tf_bvh_export(None, ctypes.byref(nn), None, None, None, None) != 0 and b"NULL handle" in lib.tf_last_error()
    assert lib.tf_launch_count() == n1
    # the host build refuses a referenced non-finite vertex too
    with pytest.raises(RuntimeError, match="non-finite"):
        RayTracer(nan.cpu(), t)


def test_build_and_trace_on_second_device():
    from tensoflow_b200.mc_ops import RayTracer
    from tensoflow_b200.synthetic import bumpy_sphere
    _cuda()
    if torch.cuda.device_count() < 2:
        pytest.skip("needs a second CUDA device")
    d1 = torch.device("cuda:1")
    v, t = bumpy_sphere(64, 32)
    host = RayTracer(v, t)
    rt = RayTracer(v.to(d1), t.to(d1))
    assert rt._device == d1
    _assert_same(_export(host), _export(rt), "cuda:1")
    g = torch.Generator().manual_seed(2)
    o = F.normalize(torch.randn(500, 3, generator=g), dim=-1) * 1.5
    d = F.normalize(torch.randn(500, 3, generator=g) * 0.2 - o, dim=-1)
    a = host.trace(o.to("cuda:0"), d.to("cuda:0"))
    b = rt.trace(o.to(d1), d.to(d1))
    assert all(y.device == d1 for y in b)
    for x, y in zip(a, b):
        assert torch.equal(x.cpu(), y.cpu())
