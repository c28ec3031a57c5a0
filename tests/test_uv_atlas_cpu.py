"""CPU checks of the UV atlas: the numpy oracle (oracle/torch_oracle_atlas.py) on a bumpy lat-long sphere (open at the poles), a
marching-cubes sphere, a lattice with zero-area faces, a helicoid whose charts fold, a single triangle and 10^4 disjoint
components: every texel centre has at most one owner, every chart's triangles lie in its rectangle, rectangles are disjoint and
inside the atlas, seam duplicates share their position, baked points lie on their triangles, the stretch is at most 2 and
dilation stays inside each chart's rectangle.  Also the refusals of the entry points and of geometry.uv_atlas / bake_texture,
none of which launches anything."""
import ctypes

import numpy as np
import pytest
import torch

from oracle import torch_oracle_atlas as O
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


def helicoid(nu=40, nv=10, turns=2.0):
    u = np.linspace(0, 2 * np.pi * turns, nu)
    v = np.linspace(0.1, 1.0, nv)
    uu, vv = np.meshgrid(u, v, indexing="ij")
    P = np.stack([vv * np.cos(uu), vv * np.sin(uu), 0.3 * uu], -1).reshape(-1, 3).astype(np.float32)
    i, j = np.arange(nu - 1)[:, None], np.arange(nv - 1)[None, :]
    a = i * nv + j
    F = np.concatenate([np.stack([a, a + nv, a + 1], -1).reshape(-1, 3), np.stack([a + 1, a + nv, a + nv + 1], -1).reshape(-1, 3)])
    return P, F.astype(np.int64)


def bumpy(nu=60, nv=31):
    from tensoflow_b200.synthetic import bumpy_sphere
    v, t = bumpy_sphere(nu, nv)
    return v.numpy(), t.numpy().astype(np.int64)


def mc_sphere(R=40):
    v, t = marching_cubes(_lattice(R).norm(dim=-1) - 0.5)
    return v.numpy(), t.numpy().astype(np.int64)


def exact_threshold():
    v, t = marching_cubes(torch.round(_lattice(25).norm(dim=-1) * 12) - 7.0)
    return v.numpy(), t.numpy().astype(np.int64)


def single_triangle():
    return np.array([[0, 0, 0], [1, 0, 0], [0.2, 1, 0.3]], np.float32), np.array([[0, 1, 2]], np.int64)


def many_components(n=10000):
    rng = np.random.default_rng(0)
    base = np.array([[0, 0, 0], [1, 0, 0], [0, 1, 0]], np.float32) * 0.01
    off = (rng.random((n, 1, 3)) * 10).astype(np.float32)
    return (base[None] + off).reshape(-1, 3).astype(np.float32), np.arange(3 * n, dtype=np.int64).reshape(n, 3)


MESHES = {"bumpy-60x31": (bumpy, 256), "mc-sphere-40": (mc_sphere, 256), "exact-threshold": (exact_threshold, 128),
          "helicoid": (helicoid, 128), "single-triangle": (single_triangle, 16), "components-1e4": (many_components, 512)}


@pytest.fixture(scope="module", params=sorted(MESHES))
def case(request):
    make, R = MESHES[request.param]
    P, F = make()
    pad = 1 if request.param == "components-1e4" else 2
    return request.param, P, F, R, pad, O.atlas(P, F, R, pad)


def test_single_owner_per_texel(case):
    _, P, F, R, pad, A = case
    xy = A["xy"][A["triangles"]]
    f, t = O.coverage(xy, R)
    assert np.bincount(t, minlength=R * R).max() <= 1
    tt = A["texel_tri"].reshape(-1)
    assert (tt[t] == f).all()
    assert ((tt >= 0).sum() - t.shape[0]) <= A["rects"].shape[0]           # the rest are one fallback texel per chart at most


def test_charts_inside_disjoint_rects(case):
    _, P, F, R, pad, A = case
    r = A["rects"].astype(np.int64)
    assert (r[:, 0] >= 0).all() and (r[:, 1] >= 0).all() and (r[:, 0] + r[:, 2] <= R).all() and (r[:, 1] + r[:, 3] <= R).all()
    paint = np.zeros((R, R), np.int64)
    for x0, y0, w, h in r:
        paint[y0:y0 + h, x0:x0 + w] += 1
    assert paint.max() == 1
    xy = A["xy"][A["triangles"]].astype(np.float64)                       # [T,3,2]
    rc = r[A["chart"]]
    assert (xy[..., 0] >= (rc[:, 0] + pad)[:, None]).all() and (xy[..., 0] <= (rc[:, 0] + rc[:, 2] - pad)[:, None]).all()
    assert (xy[..., 1] >= (rc[:, 1] + pad)[:, None]).all() and (xy[..., 1] <= (rc[:, 1] + rc[:, 3] - pad)[:, None]).all()
    tt = A["texel_tri"]
    for c in range(r.shape[0]):                                           # every chart owns a texel inside its rectangle
        x0, y0, w, h = r[c]
        own = tt[y0:y0 + h, x0:x0 + w]
        assert (own >= 0).any() and (A["chart"][own[own >= 0]] == c).all()


def test_seams_share_positions(case):
    _, P, F, R, pad, A = case
    np.testing.assert_array_equal(A["vertices"], P[A["vertex_index"]])
    np.testing.assert_array_equal(A["vertex_index"][A["triangles"]], F)
    pairs = np.unique(np.stack([A["vertex_index"][A["triangles"]].reshape(-1), np.repeat(A["chart"], 3)], 1), axis=0)
    assert pairs.shape[0] == A["vertices"].shape[0]
    np.testing.assert_array_equal(A["uv"], A["xy"] / np.float32(R))


def test_baked_points_lie_on_their_triangles(case):
    _, P, F, R, pad, A = case
    texels, pts, bary = O.texel_points(A)
    assert (bary >= 0).all() and (bary <= 1).all()
    np.testing.assert_allclose(bary.sum(1), 1.0, rtol=0, atol=1e-12)
    tri = P[F[A["texel_tri"].reshape(-1)[texels]]].astype(np.float64)
    exact = (bary[:, 0:1] * tri[:, 0] + bary[:, 1:2] * tri[:, 1]) + bary[:, 2:3] * tri[:, 2]
    scale = np.abs(tri).max(axis=(1, 2))[:, None]
    assert (np.abs(pts - exact) <= np.spacing(np.float32(1)) * scale + 1e-30).all()


def test_stretch_at_most_two(case):
    _, P, F, R, pad, A = case
    p = P.astype(np.float64)[F]
    e1, e2 = p[:, 1] - p[:, 0], p[:, 2] - p[:, 0]
    n = np.cross(e1, e2)
    ln = np.linalg.norm(n, axis=1)
    ok = ln > 1e-9 * ln.max()
    # the projection onto the chart plane only shrinks (singular values <= 1); the smaller one is |n^ . axis| >= 1/2
    k = A["classes"][ok] // 2
    cos = np.abs(n[ok][np.arange(ok.sum()), k]) / ln[ok]
    assert (cos >= 0.5 - 1e-12).all()
    xy = A["xy"][A["triangles"]].astype(np.float64)[ok]
    d1, d2 = xy[:, 1] - xy[:, 0], xy[:, 2] - xy[:, 0]
    area2 = np.abs(d1[:, 0] * d2[:, 1] - d1[:, 1] * d2[:, 0])
    ratio = area2 / (ln[ok] * A["scale"] ** 2)
    big = ln[ok] * A["scale"] ** 2 > 100.0                                   # fp32 texel rounding is negligible there
    assert (ratio[big] >= 0.5 * (1 - 1e-3)).all() and (ratio[big] <= 1 + 1e-3).all()


def test_dilation_stays_in_rects(case):
    _, P, F, R, pad, A = case
    texels, pts, _ = O.texel_points(A)
    vals = np.concatenate([pts, np.ones((pts.shape[0], 1), np.float32)], 1)
    tex = O.fill(A, texels, vals, pad)
    filled = tex[..., 3] > 0
    inside = np.zeros((R, R), bool)
    for x0, y0, w, h in A["rects"]:
        inside[y0:y0 + h, x0:x0 + w] = True
    assert not (filled & ~inside).any()
    assert filled.sum() >= texels.shape[0]
    np.testing.assert_array_equal(tex[..., 3][filled], 1.0)


def test_helicoid_forces_a_conflict_round():
    P, F = helicoid()
    A = O.atlas(P, F, 128, 2)
    assert A["rounds"] >= 1
    f, t = O.coverage(A["xy"][A["triangles"]], 128)
    assert np.bincount(t, minlength=128 * 128).max() <= 1


def test_bumpy_sphere_charts_are_few():
    P, F = bumpy()
    A = O.atlas(P, F, 256, 2)
    assert A["rounds"] == 0 and A["rects"].shape[0] < F.shape[0] // 20


def test_too_many_charts_do_not_fit():
    P, F = many_components(2000)
    with pytest.raises(O.AtlasError, match="do not fit"):
        O.atlas(P, F, 32, 2)


def _fake():
    return ctypes.c_void_p(1 << 20)


def test_entry_points_refuse_bad_arguments(lib):
    f = _fake()
    scale, nv, nc = ctypes.c_double(), ctypes.c_int64(), ctypes.c_int64()
    rounds, steps = ctypes.c_int32(), ctypes.c_int32()
    good = [f, 30, f, 10, 256, 2, f, 1 << 30, f, f, f, f, f, f, ctypes.byref(scale), ctypes.byref(nv), ctypes.byref(nc),
            ctypes.byref(rounds), ctypes.byref(steps), None]
    cases = []
    for i in (0, 2, 6, 8, 9, 10, 11, 12, 13, 14, 15, 16, 17, 18):
        a = list(good)
        a[i] = None
        cases.append((a, b"NULL pointer"))
    for i, val, match in ((1, 0, b"vertices"), (1, 1 << 31, b"vertices"), (3, 0, b"triangles"), (3, 1 << 31, b"triangles"),
                          (4, 15, b"resolution"), (4, 16385, b"resolution"), (5, 0, b"padding"), (5, 17, b"padding")):
        a = list(good)
        a[i] = val
        cases.append((a, match))
    n0 = lib.tf_launch_count()
    for a, match in cases:
        assert lib.tf_uv_atlas(*a) != 0
        assert match in lib.tf_last_error(), (a, lib.tf_last_error())
    ws = ctypes.c_size_t()
    for args, match in (((30, 10, 256, None), b"NULL pointer"), ((0, 10, 256, ctypes.byref(ws)), b"vertices"),
                        ((30, 0, 256, ctypes.byref(ws)), b"triangles"), ((30, 10, 8, ctypes.byref(ws)), b"resolution")):
        assert lib.tf_uv_atlas_sizes(*args) != 0
        assert match in lib.tf_last_error()
    assert lib.tf_uv_texel_points(f, f, f, f, 8, f, 4, f, None) != 0 and b"resolution" in lib.tf_last_error()
    assert lib.tf_uv_texel_points(None, f, f, f, 64, f, 4, f, None) != 0 and b"NULL" in lib.tf_last_error()
    assert lib.tf_uv_fill_sizes(64, 0, ctypes.byref(ws)) != 0 and b"channels" in lib.tf_last_error()
    assert lib.tf_uv_fill(f, f, 4, 3, f, f, f, 64, 2, f, 1, f, None) != 0 and b"workspace" in lib.tf_last_error()
    assert lib.tf_uv_fill(f, f, 4, 3, f, f, f, 64, 17, f, 1 << 30, f, None) != 0 and b"padding" in lib.tf_last_error()
    assert lib.tf_launch_count() == n0


@pytest.mark.parametrize("kw,exc,match", [({"resolution": 15}, ValueError, "resolution"), ({"resolution": 16385}, ValueError, "resolution"),
                                          ({"resolution": 64.5}, ValueError, "resolution"), ({"padding": 0}, ValueError, "padding"),
                                          ({"padding": 17}, ValueError, "padding")])
def test_limits_are_refused_first(lib, kw, exc, match):
    from tensoflow_b200.geometry import uv_atlas
    v, t = (torch.from_numpy(x) for x in bumpy())
    n0 = lib.tf_launch_count()
    with pytest.raises(exc, match=match):
        uv_atlas(v, t.int(), **kw)
    assert lib.tf_launch_count() == n0


@pytest.mark.parametrize("case,match", [("cpu", "CUDA"), ("shape", "CUDA"), ("float-triangles", "integer triangles"),
                                        ("2^31-vertices", "2\\^31")])
def test_mesh_refusals_launch_nothing(lib, case, match):
    from tensoflow_b200.geometry import uv_atlas
    v, t = (torch.from_numpy(x) for x in bumpy())
    t = t.int()
    if case == "shape":
        t = t.reshape(-1, 6)
    elif case == "float-triangles":
        t = t.float()
    elif case == "2^31-vertices":
        v = torch.zeros(1, 3).expand(1 << 31, 3)
    n0 = lib.tf_launch_count()
    with pytest.raises(RuntimeError, match=match):
        uv_atlas(v, t)
    assert lib.tf_launch_count() == n0
