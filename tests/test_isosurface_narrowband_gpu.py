"""Narrow-band marching cubes on the GPU (`tf_iso_nb_*`): bit-exact against the CPU restatement of the band rule round by
round, field values independent of the batch they are evaluated in, the dense mesh of extract_geometry at 256^3 and 512^3 on
trained-like fields, a closed sphere and the dense 1024^3 mesh's geometry at 2048^3, and error paths that launch nothing."""
import ctypes

import pytest
import torch

from oracle.torch_oracle_iso_nb import marching_cubes_narrowband as oracle_nb
from test_isosurface_narrowband_cpu import (FIELDS, NORMAL, STEEP_GROW, STEEP_TINY, axes_of, lattice_values, union)

pytestmark = pytest.mark.gpu

LO, HI = [-1.0, -1.0, -1.0], [1.0, 1.0, 1.0]


def _cuda():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    return torch.device("cuda:0")


def _bits(t):
    return t.contiguous().view(torch.int32)


def _lookup_fn(u, axes, dev):
    """fn on the GPU that returns the CPU lattice values u at lattice points: the kernels see exactly the oracle's values"""
    ud = u.to(dev).reshape(-1)
    ad = [a.to(dev) for a in axes]
    n = [a.shape[0] for a in axes]

    def fn(p):
        i = [torch.searchsorted(ad[a], p[:, a].contiguous()) for a in range(3)]
        for a in range(3):
            assert bool((ad[a][i[a]] == p[:, a]).all())
        return ud[(i[0] * n[1] + i[1]) * n[2] + i[2]]
    return fn


CASES = {**{f"{f}-{lat}": (FIELDS[f], lat) for f in FIELDS for lat in ("65-aniso", "70", "33x70x65")},
         "sphere-129-aniso": (FIELDS["sphere"], "129-aniso"), "steep-grow": (STEEP_GROW, "33"),
         "steep-tiny": (union(NORMAL, STEEP_TINY), "33")}


@pytest.mark.parametrize("name", list(CASES))
def test_kernels_match_oracle_round_by_round(name):
    from tensoflow_b200 import _lib
    from tensoflow_b200.isosurface import marching_cubes_narrowband
    dev = _cuda()
    fn, lat = CASES[name]
    axes = axes_of(lat)
    u = lattice_values(fn, axes)
    ref_v, ref_t, ref_active, ref_rounds = oracle_nb(fn, axes)
    stats = {}
    v, t = marching_cubes_narrowband(_lookup_fn(u, axes, dev), [a.to(dev) for a in axes], 0.0, stats=stats)
    assert v.dtype == torch.float32 and t.dtype == torch.int32 and v.device == dev
    assert len(stats["rounds"]) == len(ref_rounds) and stats["grow_rounds"] == len(ref_rounds) - 1
    for got, ref in zip(stats["rounds"], ref_rounds):
        assert torch.equal(got.cpu(), ref)
    assert stats["bricks"] == ref_active.shape[0]
    assert torch.equal(t.cpu(), ref_t) and torch.equal(_bits(v.cpu()), _bits(ref_v))
    if name == "steep-grow":
        assert stats["grow_rounds"] >= 1
    n0 = _lib.launch_count()
    v2, t2 = marching_cubes_narrowband(_lookup_fn(u, axes, dev), [a.to(dev) for a in axes])
    assert torch.equal(_bits(v2), _bits(v)) and torch.equal(t2, t)                    # bit-reproducible
    assert _lib.launch_count() > n0


def _small_shape(dev):
    from tensoflow_b200.shape_renderer import ShapeRenderer
    from tensoflow_b200.synthetic import perturb_field
    torch.manual_seed(0)
    shape = ShapeRenderer(dict(device=dev, shader_config=dict(env_res=16, env_min_res=4), gridSize=[32, 32, 32], sdf_n_comp=8,
                               sdf_dim=32, app_dim=128, max_levels=1, has_radiance_field=False, n_samples=16, n_importance=16,
                               sdf_multires=0))
    perturb_field(shape.sdf_network, seed=2, noise=5e-3)           # the field of tests/test_isosurface_gpu.py
    return shape


def _config2_shape(dev):
    """G 512, C 36, H 256, A 128, 3 mip levels, perturbed: the field of scripts/bench_extract_mesh.py"""
    from tensoflow_b200 import synthetic
    from tensoflow_b200.shape_renderer import ShapeRenderer
    torch.manual_seed(6033)
    G0 = 128
    m = ShapeRenderer(dict(device=dev, gridSize=[G0] * 3, sdf_n_comp=36, sdf_dim=256, app_dim=128, max_levels=1,
                           shader_config=dict(env_res=16, env_min_res=4)))
    for lv in (1, 2):
        m.sdf_network.upsample_volume_grid(torch.tensor([G0 << lv] * 3))
        m.update_stepSize(torch.tensor([G0 << lv] * 3), lv + 1)
    synthetic.perturb_field(m.sdf_network, seed=1, noise=1e-2)
    return m


def test_field_values_do_not_depend_on_the_batch():
    """Every value fn returns for a brick or coarse point equals extract_fields' value at that lattice point, bit for bit"""
    from tensoflow_b200.isosurface import marching_cubes_narrowband
    dev = _cuda()
    for shape in (_small_shape(dev), _config2_shape(dev)):
        R = 96
        u = shape.extract_fields(LO, HI, R).reshape(-1)
        axes = shape._extract_axes(LO, HI, R)
        seen = []

        def fn(p):
            val = shape._extract_values(p)
            seen.append((p.clone(), val.clone()))
            return val
        with torch.no_grad():
            marching_cubes_narrowband(fn, axes)
        assert len(seen) >= 2
        for p, val in seen:
            i = [torch.searchsorted(axes[a], p[:, a].contiguous()) for a in range(3)]
            assert all(bool((axes[a][i[a]] == p[:, a]).all()) for a in range(3))
            assert torch.equal(_bits(val), _bits(u[(i[0] * R + i[1]) * R + i[2]]))


@pytest.mark.parametrize("R", [256, 512])
@pytest.mark.parametrize("which", ["perturbed", "config2"])
def test_narrowband_equals_dense_extract_geometry(which, R):
    from tensoflow_b200.isosurface import marching_cubes, marching_cubes_narrowband
    dev = _cuda()
    shape = _small_shape(dev) if which == "perturbed" else _config2_shape(dev)
    with torch.no_grad():
        dv, dt = marching_cubes(shape.extract_fields(LO, HI, R))
        v, t = marching_cubes_narrowband(shape._extract_values, shape._extract_axes(LO, HI, R))
    assert dt.shape[0] > 1000
    assert torch.equal(t, dt) and torch.equal(_bits(v), _bits(dv))
    gv, gt = shape.extract_geometry(LO, HI, R)                       # extract_geometry's rescale of the same index-space mesh
    assert torch.equal(gt, dt) and torch.equal(_bits(gv), _bits(v / (R - 1.0) * 2.0 - 1.0))


# peak device memory of a 2048^3 extraction, far below the 34 GB of a dense fp32 volume: 6 GiB
PEAK_2048 = 6 << 30


def test_sphere_2048_is_closed():
    """extract_geometry at 2048^3 on an analytic sphere (the SDF query replaced by |x - c| - r): closed, genus 0, every vertex
    within 0.05 voxel of the sphere, peak memory below PEAK_2048, and the mesh builds a BVH that rays hit."""
    from tensoflow_b200.material import MaterialRenderer
    from tensoflow_b200.synthetic import make_rays
    dev = _cuda()
    shape = _small_shape(dev)
    c = torch.tensor([0.031, -0.047, 0.022], device=dev)
    r = 0.61
    shape.sdf_network.sdf = lambda p, lvl: ((p - c) ** 2).sum(-1).sqrt()[:, None] - r
    R = 2048
    torch.cuda.synchronize()
    torch.cuda.reset_peak_memory_stats(dev)
    base = torch.cuda.memory_allocated(dev)
    v, t = shape.extract_geometry(LO, HI, R)
    torch.cuda.synchronize()
    peak = torch.cuda.max_memory_allocated(dev) - base
    assert peak < PEAK_2048, peak
    assert t.shape[0] > 10 ** 6 and bool(torch.isfinite(v).all()) and int(t.min()) >= 0 and int(t.max()) < v.shape[0]
    tl = t.long()
    e = torch.cat([tl[:, [0, 1]], tl[:, [1, 2]], tl[:, [2, 0]]], 0)
    V = v.shape[0]
    fwd = torch.sort(e[:, 0] * V + e[:, 1])[0]
    rev = torch.sort(e[:, 1] * V + e[:, 0])[0]
    assert bool((fwd[1:] != fwd[:-1]).all()) and torch.equal(fwd, rev)      # closed, consistently wound
    n_edges = fwd.shape[0] // 2
    assert V - n_edges + t.shape[0] == 2                                     # Euler characteristic of a sphere
    voxel = 2.0 / (R - 1)
    rad = (v.double() - c.double()).norm(dim=-1) - r
    assert float(rad.abs().max()) < 0.05 * voxel
    mat = MaterialRenderer(dict(device=dev, shader_cfg=dict(gridSize=[16, 16, 16], light_reso=16, mat_grid=24),
                                gridSize=[32, 32, 32]), v, t)
    rays = make_rays(600, seed=3, device=dev, radii_jitter=False)
    o, d = rays['rays_o'], rays['dirs']
    pos, face_n, depth = mat.tracer.ray_tracer.trace(o, d)
    hit = face_n.abs().sum(-1) > 0                                       # a miss has a zero normal
    assert int(hit.sum()) > 500                                              # the rays aim at [-0.3, 0.3]^3
    assert float((face_n[hit] * d[hit]).sum(-1).max()) < 0                   # faces point out, against the incoming rays
    assert float(((pos[hit].double() - c.double()).norm(dim=-1) - r).abs().max()) < voxel


def test_config2_2048_matches_dense_1024():
    """The trained-like field at 2048^3 through extract_geometry lies within one 1024^3 voxel (Chamfer, evaluate_mesh) of
    the dense 1024^3 mesh; peak memory below PEAK_2048."""
    from tensoflow_b200.geometry import evaluate_mesh
    dev = _cuda()
    shape = _config2_shape(dev)
    dense = shape.extract_geometry(LO, HI, 1024)
    torch.cuda.synchronize()
    torch.cuda.reset_peak_memory_stats(dev)
    base = torch.cuda.memory_allocated(dev)
    fine = shape.extract_geometry(LO, HI, 2048)
    torch.cuda.synchronize()
    peak = torch.cuda.max_memory_allocated(dev) - base
    assert peak < PEAK_2048, peak
    assert fine[1].shape[0] > 3 * dense[1].shape[0]
    m = evaluate_mesh(fine[0], fine[1], dense[0], dense[1], n_samples=1_000_000)
    assert m["chamfer"] < 2.0 / 1023, m


def test_errors_launch_nothing():
    from tensoflow_b200 import _lib
    from tensoflow_b200.isosurface import marching_cubes_narrowband
    dev = _cuda()
    lib = _lib.load()
    P = lambda x: ctypes.c_void_p(x.data_ptr())
    s = _lib.stream_ptr()
    f = torch.zeros(8 * 729, device=dev)
    b = torch.zeros(8, device=dev, dtype=torch.int64)
    i32 = torch.zeros(8 * 81, device=dev, dtype=torch.int32)
    i64 = torch.zeros(8 * 81, device=dev, dtype=torch.int64)
    u8 = torch.zeros(64, device=dev, dtype=torch.uint8)
    shape = _small_shape(dev)
    n0 = lib.tf_launch_count()
    assert lib.tf_iso_nb_classify(P(f), 4097, 9, 9, 0.0, 1.0, P(u8), s) != 0 and b"4096" in lib.tf_last_error()
    assert lib.tf_iso_nb_classify(P(f), 9, 1, 9, 0.0, 1.0, P(u8), s) != 0
    assert lib.tf_iso_nb_classify(None, 9, 9, 9, 0.0, 1.0, P(u8), s) != 0 and b"NULL" in lib.tf_last_error()
    assert lib.tf_iso_nb_points(P(f), P(f), None, 9, 9, 9, P(b), 1, P(f), s) != 0
    assert lib.tf_iso_nb_grow(P(f), P(b), -1, 9, 9, 9, 0.0, P(u8), s) != 0
    assert lib.tf_iso_nb_grow(P(f), None, 1, 9, 9, 9, 0.0, P(u8), s) != 0
    assert lib.tf_iso_nb_count(P(f), P(b), 1, 9, 9, 4097, 0.0, P(i32), P(i32), P(i64), s) != 0
    assert lib.tf_iso_nb_vertices(P(f), P(b), 1, 9, 9, 9, 0.0, None, P(f), P(i32), s) != 0
    assert lib.tf_iso_nb_triangles(P(f), P(b), 1, 9, 9, 9, 0.0, None, P(i64), P(i32), P(i32), s) != 0
    # no bricks: nothing to do, even with NULL buffers
    assert lib.tf_iso_nb_count(None, None, 0, 9, 9, 9, 0.0, None, None, None, s) == 0
    assert lib.tf_iso_nb_triangles(None, None, 0, 9, 9, 9, 0.0, None, None, None, None, s) == 0
    # the Python layer: oversized lattices, including extract_geometry above 4096
    fn = lambda p: p[:, 0]
    with pytest.raises(RuntimeError, match="4096"):
        marching_cubes_narrowband(fn, [torch.linspace(-1, 1, 4097, device=dev)] + [torch.linspace(-1, 1, 9, device=dev)] * 2)
    with pytest.raises(RuntimeError, match="4096"):
        shape.extract_geometry(LO, HI, 4097)
    assert lib.tf_launch_count() == n0
    # a non-finite value: raises before the vertex and triangle kernels
    axes = [torch.linspace(-1, 1, 33, device=dev)] * 3
    for bad in (float("nan"), float("inf")):
        def fn_bad(p):
            val = (p.norm(dim=-1) - 0.5)
            return torch.where((p - 0.125).abs().max(-1).values < 1e-6, torch.full_like(val, bad), val)
        n1 = lib.tf_launch_count()
        with pytest.raises(RuntimeError, match="non-finite"):
            marching_cubes_narrowband(fn_bad, axes)
        assert lib.tf_launch_count() - n1 <= 3                          # classify, points, grow at most
