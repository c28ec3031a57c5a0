"""GPU checks of the UV atlas (tf_uv_atlas, tf_uv_texel_points, tf_uv_fill): bit-equality with oracle/torch_oracle_atlas.py on
7 meshes x 3 resolutions (a helicoid that forces conflict rounds, a simplified and an open mesh among them), determinism,
single ownership and rectangles inside the atlas at 16 M triangles, affine reproduction of baked textures under bilinear
lookup, MaterialRenderer.predict_materials / bake_materials against the material network, and refusals before any launch."""
import math

import numpy as np
import pytest
import torch

from oracle import torch_oracle_atlas as O
from oracle.torch_oracle_iso import marching_cubes

pytestmark = pytest.mark.gpu


def _cuda():
    if not torch.cuda.is_available():
        pytest.skip("needs a GPU")
    from tensoflow_b200 import build
    build.build()
    return torch.device("cuda")


def _lattice(R):
    ax = torch.linspace(-1, 1, R)
    x, y, z = torch.meshgrid(ax, ax, ax, indexing="ij")
    return torch.stack([x, y, z], -1)


def helicoid(nu=80, nv=20, turns=3.0):
    u = np.linspace(0, 2 * np.pi * turns, nu)
    v = np.linspace(0.1, 1.0, nv)
    uu, vv = np.meshgrid(u, v, indexing="ij")
    P = np.stack([vv * np.cos(uu), vv * np.sin(uu), 0.3 * uu], -1).reshape(-1, 3).astype(np.float32)
    i, j = np.arange(nu - 1)[:, None], np.arange(nv - 1)[None, :]
    a = i * nv + j
    F = np.concatenate([np.stack([a, a + nv, a + 1], -1).reshape(-1, 3), np.stack([a + 1, a + nv, a + nv + 1], -1).reshape(-1, 3)])
    return torch.from_numpy(P), torch.from_numpy(F.astype(np.int32))


def bumpy(nu, nv):
    from tensoflow_b200.synthetic import bumpy_sphere
    return bumpy_sphere(nu, nv)


def mc_sphere(R):
    return marching_cubes(_lattice(R).norm(dim=-1) - 0.5)


def mc_torus(R):
    p = _lattice(R)
    q = torch.stack([p[..., :2].norm(dim=-1) - 0.5, p[..., 2]], -1)
    return marching_cubes(q.norm(dim=-1) - 0.2)


def exact_threshold():
    return marching_cubes(torch.round(_lattice(33).norm(dim=-1) * 16) - 9.0)


def simplified():
    from tensoflow_b200.geometry import simplify_mesh
    v, t = mc_sphere(96)
    vo, to = simplify_mesh(v.cuda(), t.cuda(), t.shape[0] // 20)
    return vo.cpu(), to.cpu()


MESHES = {"helicoid": helicoid, "bumpy-open-400x201": lambda: bumpy(400, 201), "bumpy-60x31": lambda: bumpy(60, 31),
          "mc-sphere-64": lambda: mc_sphere(64), "mc-torus-80": lambda: mc_torus(80), "exact-threshold": exact_threshold,
          "simplified-sphere-96": simplified}


def _np(A):
    return {k: (v.cpu().numpy() if torch.is_tensor(v) else v) for k, v in vars(A).items()}


@pytest.fixture(scope="module", params=sorted(MESHES))
def mesh(request):
    _cuda()
    v, t = MESHES[request.param]()
    return request.param, v.float(), t.int()


@pytest.mark.parametrize("R", [256, 1024, 2048])
def test_atlas_equals_oracle(mesh, R):
    from tensoflow_b200.geometry import bake_texture, texel_points, uv_atlas
    name, v, t = mesh
    dev = _cuda()
    A = uv_atlas(v.to(dev), t.to(dev), R, 2)
    ref = O.atlas(v.numpy(), t.numpy().astype(np.int64), R, 2)
    got = _np(A)
    assert got["scale"] == ref["scale"] and got["rounds"] == ref["rounds"] and got["steps"] == ref["steps"], name
    for k in ("chart", "rects", "vertex_index", "triangles", "xy", "uv", "texel_tri", "vertices"):
        np.testing.assert_array_equal(got[k], ref[k], err_msg=f"{name} {k}")
    if name == "helicoid":
        assert ref["rounds"] >= 1
    texels, pts = texel_points(A)
    rt, rp, _ = O.texel_points(ref)
    np.testing.assert_array_equal(texels.cpu().numpy(), rt)
    np.testing.assert_array_equal(pts.cpu().numpy(), rp)
    fn = lambda p: torch.cat([torch.sin(3 * p), p[:, :1] * p[:, 1:2]], -1)
    tex, mask = bake_texture(A, fn, 4, chunk=1 << 12)
    ref_tex = O.fill(ref, rt, fn(pts).cpu().numpy(), 2)                        # the same fn values as the bake
    np.testing.assert_array_equal(tex.cpu().numpy(), ref_tex)
    np.testing.assert_array_equal(mask.cpu().numpy(), ref["texel_tri"] >= 0)


def test_two_runs_are_bit_identical():
    from tensoflow_b200.geometry import uv_atlas
    dev = _cuda()
    v, t = helicoid()
    a, b = _np(uv_atlas(v.to(dev), t.to(dev), 512)), _np(uv_atlas(v.to(dev), t.to(dev), 512))
    for k in a:
        assert np.array_equal(a[k], b[k]), k


def _check_invariants(A):
    R = A.resolution
    r = A.rects.long()
    assert int(r[:, 0].min()) >= 0 and int(r[:, 1].min()) >= 0
    assert int((r[:, 0] + r[:, 2]).max()) <= R and int((r[:, 1] + r[:, 3]).max()) <= R
    paint = torch.zeros(R + 1, R + 1, device=r.device, dtype=torch.int32)   # 2-D difference array of the rectangles
    x0, y0, x1, y1 = r[:, 0], r[:, 1], r[:, 0] + r[:, 2], r[:, 1] + r[:, 3]
    for ys, xs, s in ((y0, x0, 1), (y0, x1, -1), (y1, x0, -1), (y1, x1, 1)):
        paint.index_put_((ys, xs), torch.full_like(ys, s, dtype=torch.int32), accumulate=True)
    assert int(paint.cumsum(0).cumsum(1).max()) == 1                          # disjoint
    xy = A.xy[A.triangles.long()]                                             # [T,3,2]
    rc = r[A.chart.long()].float()
    p = float(A.padding)
    assert bool((xy[..., 0] >= (rc[:, 0:1] + p)).all()) and bool((xy[..., 0] <= (rc[:, 0:1] + rc[:, 2:3] - p)).all())
    assert bool((xy[..., 1] >= (rc[:, 1:2] + p)).all()) and bool((xy[..., 1] <= (rc[:, 1:2] + rc[:, 3:4] - p)).all())


def test_invariants_at_16m_triangles():
    from tensoflow_b200.geometry import uv_atlas
    from tensoflow_b200.synthetic import bumpy_sphere
    dev = _cuda()
    v, t = bumpy_sphere(4000, 2001)
    A = uv_atlas(v.to(dev), t.to(dev), 4096)
    assert t.shape[0] >= 16_000_000
    _check_invariants(A)
    # every owned texel lies in the rectangle of its owner's chart (rectangles are disjoint, so no texel has two charts)
    R = A.resolution
    idx = torch.nonzero(A.texel_tri.reshape(-1) >= 0)[:, 0]
    own = A.texel_tri.reshape(-1)[idx].long()
    assert idx.numel() > 0 and int(own.max()) < t.shape[0]
    rc = A.rects.long()[A.chart.long()[own]]
    i, j = idx % R, idx // R
    assert bool(((i >= rc[:, 0]) & (i < rc[:, 0] + rc[:, 2]) & (j >= rc[:, 1]) & (j < rc[:, 1] + rc[:, 3])).all())


def _bilinear(tex, x, y):
    R = tex.shape[0]
    xf, yf = x - 0.5, y - 0.5
    i0, j0 = torch.floor(xf).long(), torch.floor(yf).long()
    fx, fy = (xf - i0).unsqueeze(-1), (yf - j0).unsqueeze(-1)
    i1, j1 = (i0 + 1).clamp(0, R - 1), (j0 + 1).clamp(0, R - 1)
    i0, j0 = i0.clamp(0, R - 1), j0.clamp(0, R - 1)
    val = (tex[j0, i0] * (1 - fx) + tex[j0, i1] * fx) * (1 - fy) + (tex[j1, i0] * (1 - fx) + tex[j1, i1] * fx) * fy
    return val, (i0, i1, j0, j1)


def test_affine_reproduction():
    from tensoflow_b200.geometry import bake_texture, sample_surface, uv_atlas
    dev = _cuda()
    v, t = bumpy(200, 101)
    v, t = v.to(dev), t.to(dev)
    A = uv_atlas(v, t, 1024)
    G = torch.tensor([[0.3, -1.2], [0.7, 0.4], [-0.5, 0.9]], device=dev, dtype=torch.float64)
    b = torch.tensor([0.25, -0.5], device=dev, dtype=torch.float64)
    fn = lambda p: torch.cat([(p.double() @ G + b).float(), torch.ones(p.shape[0], 1, device=dev)], -1)
    tex, _ = bake_texture(A, fn, 3)
    pts, tri, _ = sample_surface(v, t, 200_000, seed=3)
    # texel-space position of each sample from its barycentrics in its triangle
    P = v.double()[t.long()[tri]]
    xy = A.xy.double()[A.triangles.long()[tri]]
    e0, e1, q = P[:, 1] - P[:, 0], P[:, 2] - P[:, 0], pts.double() - P[:, 0]
    d00, d01, d11 = (e0 * e0).sum(-1), (e0 * e1).sum(-1), (e1 * e1).sum(-1)
    d20, d21 = (q * e0).sum(-1), (q * e1).sum(-1)
    den = d00 * d11 - d01 * d01
    lb, lc = (d11 * d20 - d01 * d21) / den, (d00 * d21 - d01 * d20) / den
    la = 1 - lb - lc
    x = la * xy[:, 0, 0] + lb * xy[:, 1, 0] + lc * xy[:, 2, 0]
    y = la * xy[:, 0, 1] + lb * xy[:, 1, 1] + lc * xy[:, 2, 1]
    val, (i0, i1, j0, j1) = _bilinear(tex.double(), x, y)
    want = pts.double() @ G + b
    tt = A.texel_tri
    one = (tt[j0, i0] == tri) & (tt[j0, i1] == tri) & (tt[j1, i0] == tri) & (tt[j1, i1] == tri)
    filled = val[:, 2] > 1 - 1e-6                                             # all four texels filled (after dilation)
    err = (val[:, :2] - want).abs().amax(-1)
    assert float(one.double().mean()) > 0.1                                 # the exact case is not vacuous
    assert float(err[one].max()) <= 1e-5
    grad = float(G.abs().sum(0).max())
    bound = grad * 2.0 / A.scale + 1e-5
    assert float(filled.double().mean()) > 0.99
    assert float(err[filled].max()) <= bound


MAT_CFG = dict(train_ray_num=64, gridSize=[16] * 3, shader_cfg=dict(gridSize=[16, 16, 16], light_reso=16, mat_grid=24))


def _material_renderer(dev):
    from tensoflow_b200.material import MaterialRenderer
    torch.manual_seed(0)
    v, t = bumpy(120, 61)
    r = MaterialRenderer(dict(MAT_CFG, device=dev), v.to(dev), t.to(dev))
    with torch.no_grad():                                                   # materials that vary over the surface
        for p in r.shader_network.mat_plane:
            p.copy_(torch.randn_like(p) * 0.3)
    return r, v.to(dev), t.to(dev)


def test_predict_materials_per_vertex():
    dev = _cuda()
    r, v, t = _material_renderer(dev)
    m = r.predict_materials(batch_size=1000)
    with torch.no_grad():
        metallic, rough2, albedo = r.shader_network.predict_materials(v)
    assert m['metallic'].shape == (v.shape[0], 1) and m['roughness'].shape == (v.shape[0], 1) and m['albedo'].shape == (v.shape[0], 3)
    torch.testing.assert_close(m['metallic'], metallic, rtol=0, atol=1e-5)
    torch.testing.assert_close(m['roughness'], torch.sqrt(rough2), rtol=0, atol=1e-5)
    torch.testing.assert_close(m['albedo'], albedo, rtol=0, atol=1e-5)


def test_bake_materials_matches_texel_points():
    from tensoflow_b200.geometry import texel_points
    dev = _cuda()
    r, v, t = _material_renderer(dev)
    out = r.bake_materials(resolution=512, padding=2)
    A = out['atlas']
    texels, pts = texel_points(A)
    with torch.no_grad():
        metallic, rough2, albedo = r.shader_network.predict_materials(pts)
    R = A.resolution
    flat = lambda x: x.reshape(R * R, -1)[texels]
    assert bool(out['mask'].reshape(-1)[texels].all()) and int(out['mask'].sum()) == texels.shape[0]
    torch.testing.assert_close(flat(out['albedo']), albedo, rtol=0, atol=1e-5)
    torch.testing.assert_close(flat(out['roughness']), torch.sqrt(rough2), rtol=0, atol=1e-5)
    torch.testing.assert_close(flat(out['metallic']), metallic, rtol=0, atol=1e-5)
    np.testing.assert_array_equal(A.vertices.cpu().numpy(), v.cpu().numpy()[A.vertex_index.cpu().numpy()])


@pytest.mark.parametrize("case,match", [("index-range", "out of range"), ("negative-index", "out of range"),
                                        ("nan-vertex", "non-finite"), ("inf-vertex", "non-finite"), ("zero-area", "total area"),
                                        ("2^31-triangles", "2\\^31")])
def test_refusals_launch_nothing(case, match):
    from tensoflow_b200 import _lib
    from tensoflow_b200.geometry import uv_atlas
    dev = _cuda()
    v, t = bumpy(40, 21)
    v, t = v.to(dev), t.to(dev)
    if case == "index-range":
        t = t.clone(); t[5, 1] = v.shape[0]
    elif case == "negative-index":
        t = t.clone(); t[0, 0] = -1
    elif case == "nan-vertex":
        v = v.clone(); v[3, 2] = float("nan")
    elif case == "inf-vertex":
        v = v.clone(); v[3, 0] = float("inf")
    elif case == "zero-area":
        v = torch.zeros_like(v)
    elif case == "2^31-triangles":
        t = torch.zeros(1, 3, device=dev, dtype=torch.int32).expand(1 << 31, 3)
    n0 = _lib.launch_count()
    with pytest.raises(RuntimeError, match=match):
        uv_atlas(v, t, 256)
    assert _lib.launch_count() == n0


def test_charts_that_do_not_fit_are_refused():
    from tensoflow_b200.geometry import uv_atlas
    dev = _cuda()
    n = 2000
    base = torch.tensor([[0, 0, 0], [1, 0, 0], [0, 1, 0]], dtype=torch.float32) * 0.01
    v = (base[None] + torch.rand(n, 1, 3, generator=torch.Generator().manual_seed(0)) * 10).reshape(-1, 3)
    t = torch.arange(3 * n, dtype=torch.int32).reshape(n, 3)
    with pytest.raises(RuntimeError, match="do not fit"):
        uv_atlas(v.to(dev), t.to(dev), 32)
