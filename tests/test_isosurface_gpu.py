"""Isosurface extraction on the GPU (`tf_iso_*` kernels): bit-exact against the CPU oracle (oracle/torch_oracle_iso.py), a
closed mesh at 512^3, the shape stage's extract_geometry against the fp64 field oracle, and the hand-over of the extracted mesh
to the material stage."""
import pytest
import torch

from conftest import rel_err
from oracle import torch_oracle as O
from oracle import torch_oracle_renderer as RR
from oracle.torch_oracle_iso import marching_cubes as oracle_mc
from test_isosurface_cpu import RANDOM_CASES, random_volume, sphere_sdf, torus_sdf

pytestmark = pytest.mark.gpu

SHAPE_CFG = dict(gridSize=[32, 32, 32], sdf_n_comp=8, sdf_dim=32, app_dim=128, max_levels=1, has_radiance_field=False,
                 n_samples=16, n_importance=16, sdf_multires=0)
MAT_SHADER = dict(gridSize=[16, 16, 16], light_reso=16, mat_grid=24)


def _cuda():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    return torch.device("cuda:0")


def _planes(n):
    k = torch.arange(n, dtype=torch.float32).reshape(1, 1, n).expand(n, n, n)
    return (k - n // 2).contiguous()                     # the plane k = n/2 sits exactly at the threshold 0


VOLUMES = {
    **{f"{'x'.join(map(str, s))}-{kind}": (lambda s=s, kind=kind, seed=seed: random_volume(s, kind, seed)) for s, kind, seed in RANDOM_CASES},
    "130-random": lambda: random_volume((130, 130, 130), "normal", 7),
    "sphere": lambda: sphere_sdf(96, (47.3, 46.6, 48.2), 30.5),
    "torus": lambda: torus_sdf(96, (47.6, 48.3, 47.2), 28.0, 9.5),
    "all-inside": lambda: -torch.ones(9, 10, 11),
    "all-outside": lambda: torch.ones(9, 10, 11),
    "exact-planes": lambda: _planes(40),
}


def _bits(t):
    return t.contiguous().view(torch.int32)


@pytest.mark.parametrize("name", list(VOLUMES))
def test_marching_cubes_matches_oracle_bit_for_bit(name):
    from tensoflow_b200 import _lib
    from tensoflow_b200.isosurface import marching_cubes
    dev = _cuda()
    vol = VOLUMES[name]()
    ref_v, ref_t = oracle_mc(vol, 0.0)
    n0 = _lib.launch_count()
    v, t = marching_cubes(vol.to(dev), 0.0)                 # fp64 volumes (sphere, torus) are converted to fp32 once
    launches = _lib.launch_count() - n0
    assert v.device == dev and t.device == dev and v.dtype == torch.float32 and t.dtype == torch.int32
    assert v.shape == ref_v.shape and t.shape == ref_t.shape
    assert torch.equal(t.cpu(), ref_t)
    assert torch.equal(_bits(v.cpu()), _bits(ref_v))
    v2, t2 = marching_cubes(vol.to(dev), 0.0)
    assert torch.equal(_bits(v2), _bits(v)) and torch.equal(t2, t)
    if ref_t.shape[0] == 0:
        assert v.shape == (0, 3) and t.shape == (0, 3)
        assert launches == 1                                 # the count kernel only
    else:
        assert launches == 3


def test_marching_cubes_threshold_and_strided_input():
    from tensoflow_b200.isosurface import marching_cubes
    dev = _cuda()
    vol = random_volume((20, 24, 28), "normal", 11)
    ref_v, ref_t = oracle_mc(vol.permute(2, 0, 1), 0.3)
    v, t = marching_cubes(vol.to(dev).permute(2, 0, 1), 0.3)   # non-contiguous view
    assert torch.equal(t.cpu(), ref_t) and torch.equal(_bits(v.cpu()), _bits(ref_v))


def test_sphere_512_is_closed():
    from tensoflow_b200.isosurface import marching_cubes
    dev = _cuda()
    n = 512
    g = torch.arange(n, device=dev, dtype=torch.float32)
    c, r = (255.3, 254.6, 256.2), 200.5
    u = ((g[:, None, None] - c[0]) ** 2 + (g[None, :, None] - c[1]) ** 2 + (g[None, None, :] - c[2]) ** 2).sqrt() - r
    v, t = marching_cubes(u)
    del u
    assert 0 < v.shape[0] < 2 ** 31 and 0 < t.shape[0] < 2 ** 31
    assert bool(torch.isfinite(v).all()) and int(t.min()) >= 0 and int(t.max()) < v.shape[0]
    tl = t.long()
    e = torch.cat([tl[:, [0, 1]], tl[:, [1, 2]], tl[:, [2, 0]]], 0)
    V = v.shape[0]
    fwd = torch.sort(e[:, 0] * V + e[:, 1])[0]
    rev = torch.sort(e[:, 1] * V + e[:, 0])[0]
    assert bool((fwd[1:] != fwd[:-1]).all())                # no directed edge twice
    assert torch.equal(fwd, rev)                            # every directed edge has its twin: closed, consistently wound
    rad = (v.double() - torch.tensor(c, device=dev, dtype=torch.float64)).norm(dim=-1) - r
    assert float(rad.abs().max()) < 0.02                    # fraction of a voxel (see the CPU sphere test)


def test_non_finite_volume_raises():
    from tensoflow_b200 import _lib
    from tensoflow_b200.isosurface import marching_cubes
    dev = _cuda()
    for bad in (float("nan"), float("inf")):
        vol = random_volume((8, 9, 10), "normal", 3).to(dev)
        vol[3, 4, 5] = bad
        n0 = _lib.launch_count()
        with pytest.raises(RuntimeError, match="non-finite"):
            marching_cubes(vol)
        assert _lib.launch_count() - n0 == 1                # no vertex / triangle kernel ran


def _shape(dev):
    from tensoflow_b200.shape_renderer import ShapeRenderer
    from tensoflow_b200.synthetic import perturb_field
    torch.manual_seed(0)
    shape = ShapeRenderer(dict(device=dev, shader_config=dict(env_res=16, env_min_res=4), **SHAPE_CFG))
    perturb_field(shape.sdf_network, seed=2, noise=5e-3)           # the field of tests/test_nvs_gpu.py
    return shape


def _oracle_field(shape, dtype=torch.float64):
    f = O.TensoSDF([32] * 3, torch.tensor([[-1., -1, -1], [1, 1, 1]]), sdf_n_comp=8, sdf_dim=32, app_dim=128, init_n_levels=1)
    f.load_state_dict({k: v.detach().cpu() for k, v in shape.sdf_network.state_dict().items()}, strict=False)
    return f.to(dtype)


R = 64
LO, HI = [-1.0, -1.0, -1.0], [1.0, 1.0, 1.0]


def test_extract_geometry_matches_oracle():
    from tensoflow_b200.isosurface import marching_cubes
    dev = _cuda()
    shape = _shape(dev)
    u = shape.extract_fields(LO, HI, R)
    assert u.shape == (R, R, R) and u.device.type == "cuda"
    ax = torch.linspace(-1.0, 1.0, R)
    x, y, z = torch.meshgrid(ax, ax, ax, indexing="ij")
    pts = torch.stack([x, y, z], -1).reshape(-1, 3)
    inside_ball = (torch.norm(pts.to(dev), dim=-1) < 1.0).cpu()   # the product's own test of the outside mask
    assert 0.4 < float(inside_ball.float().mean()) < 0.6
    assert torch.equal(u.reshape(-1).cpu()[~inside_ball], torch.ones(int((~inside_ball).sum())))
    got = u.reshape(-1)[inside_ball.to(dev)]
    with torch.no_grad():
        r64 = _oracle_field(shape).sdf(pts[inside_ball].double(), None).reshape(-1)
        r32 = _oracle_field(shape, torch.float32).sdf(pts[inside_ball], None).reshape(-1)
    # the bar of the SDF-only kernel tests (tests/test_shape_gpu.py close_as_fp32): 1e-5, floating with 4x the fp32 oracle's
    # own error, never above 1e-4
    assert rel_err(got, r64) <= min(1e-4, max(1e-5, 4 * rel_err(r32, r64)))

    verts, tris = shape.extract_geometry(LO, HI, R)
    ref_v, ref_t = oracle_mc(u.cpu(), 0.0)
    assert tris.shape[0] > 500 and torch.equal(tris.cpu(), ref_t)
    assert torch.allclose(verts.cpu(), ref_v / (R - 1.0) * 2.0 - 1.0, rtol=0, atol=1e-6)
    v_idx, _ = marching_cubes(u)
    assert torch.equal(_bits(v_idx.cpu()), _bits(ref_v))
    # The field is smooth at the lattice scale (its factor grid has 31 cells across the box, the lattice 63), so linear
    # interpolation along a voxel edge errs by ~h^2 |f''| / 8, a small fraction of a voxel h: 0.04 h measured on the fp64 oracle.
    # Bar: 0.1 voxel.
    with torch.no_grad():
        s = shape.sdf_network.sdf(verts, None).reshape(-1)
    voxel = 2.0 / (R - 1)
    assert float(s.abs().max()) < 0.1 * voxel


def test_extracted_mesh_hands_over_to_material_stage():
    """MaterialRenderer(cfg, *shape.extract_geometry(...)) + init_sdf(shape.ckpt_to_save()): surface points refined on the frozen
    SDF match the fp64 oracle fed with the mesh depths (the rule of tests/test_nvs_gpu.py::test_surface_points_match_oracle)."""
    from tensoflow_b200.material import MaterialRenderer
    from tensoflow_b200.synthetic import make_rays
    dev = _cuda()
    shape = _shape(dev)
    verts, tris = shape.extract_geometry(LO, HI, R)
    mat = MaterialRenderer(dict(device=dev, shader_cfg=dict(MAT_SHADER), gridSize=SHAPE_CFG['gridSize']), verts, tris)
    mat.init_sdf(shape.ckpt_to_save())
    rays = make_rays(600, seed=3, device=dev, radii_jitter=False)
    o, d = rays['rays_o'], rays['dirs']
    _, face_n, _ = mat.tracer.ray_tracer.trace(o, d)
    _, _, depth0, hit0 = mat.trace(o, d)
    inters, normals, depth, hit = mat.trace_sdf_with_mesh(o, d, 32, 9)
    hit = hit.squeeze(-1)
    assert torch.equal(hit, hit0.squeeze(-1)) and 50 < int(hit.sum()) < 600
    # face normals of the extracted mesh point out of the object: against rays arriving from outside
    assert float((face_n[hit] * d[hit]).sum(-1).max()) < 0

    f64 = _oracle_field(shape)
    oh, dh, m_depth = o[hit].cpu().double(), d[hit].cpu().double(), depth0[hit].cpu().double()
    inv_s = float(mat.deviation_net(torch.zeros(1, 3, device=dev))[0, 0])
    dep, pts, n = RR.surface_refine(f64, inv_s, oh, dh, m_depth, float(mat.unit_size), float(mat.radius), 32, 9)
    assert rel_err(depth[hit], dep) < 1e-4
    assert rel_err(inters[hit], pts) < 1e-4
    assert float((normals[hit].cpu().double() - n).abs().max()) < 2e-3
    assert float(((normals[hit] * d[hit]).sum(-1)).max()) <= 0
