"""Narrow-band marching cubes without a GPU: the CPU restatement of the band rule (oracle/torch_oracle_iso_nb.py
marching_cubes_narrowband) gives the dense oracle's mesh bit for bit on true SDFs and on the capped field of extract_fields,
grows through bricks the coarse test misses on a steep field, misses an isolated steep component as documented, and the GPU
entry points refuse CPU tensors and oversized lattices before any launch."""
import math

import pytest
import torch

from oracle.torch_oracle_iso import marching_cubes as oracle_mc
from oracle.torch_oracle_iso_nb import marching_cubes_narrowband as oracle_nb


# ---- analytic fields on world points [N,3] (fp64 arithmetic, fp32 values); shared with tests/test_isosurface_narrowband_gpu.py
def sphere(c, r, slope=1.0):
    c = torch.tensor(c, dtype=torch.float64)
    return lambda p: (slope * ((p.double() - c).norm(dim=-1) - r)).float()


def torus(c, R, r):
    c = torch.tensor(c, dtype=torch.float64)

    def f(p):
        d = p.double() - c
        q = d[:, :2].norm(dim=-1) - R
        return ((q * q + d[:, 2] * d[:, 2]).sqrt() - r).float()
    return f


def union(*fs):
    return lambda p: torch.stack([f(p) for f in fs]).min(0).values


def plane(nrm, d):
    n = torch.tensor(nrm, dtype=torch.float64)
    n = n / n.norm()
    return lambda p: (p.double() @ n + d).float()


def capped(f):
    """the outside value of ShapeRenderer.extract_fields: +1.0 where ||x|| >= 1"""
    return lambda p: torch.where(p.norm(dim=-1) >= 1.0, torch.ones(p.shape[0]), f(p))


FIELDS = {
    "sphere": sphere((0.07, -0.11, 0.05), 0.61),
    "torus": torus((0.03, 0.02, -0.04), 0.55, 0.2),
    "two-spheres": union(sphere((-0.45, -0.4, -0.38), 0.3), sphere((0.42, 0.37, 0.4), 0.35)),
    "plane": plane((0.3, -0.5, 0.8), 0.07),
    "capped-sphere": capped(sphere((0.25, 0.0, -0.1), 0.9)),          # cut open by the ball: a jump from < 0 to +1
}

LATTICES = {                                                            # (points per axis), (bound_min), (bound_max)
    "33": ((33, 33, 33), (-1.0, -1.0, -1.0), (1.0, 1.0, 1.0)),
    "65-aniso": ((65, 65, 65), (-1.0, -0.9, -1.1), (1.05, 0.95, 1.0)),
    "70": ((70, 70, 70), (-1.0, -1.0, -1.0), (1.0, 1.0, 1.0)),
    "129-aniso": ((129, 129, 129), (-1.1, -1.0, -0.95), (1.0, 1.1, 1.05)),
    "33x70x65": ((33, 70, 65), (-1.0, -1.2, -1.0), (1.0, 1.0, 1.3)),
}


def axes_of(name):
    n, lo, hi = LATTICES[name]
    return [torch.linspace(lo[a], hi[a], n[a]) for a in range(3)]


def lattice_values(fn, axes):
    x, y, z = torch.meshgrid(*axes, indexing="ij")
    return fn(torch.stack([x, y, z], -1).reshape(-1, 3)).reshape(x.shape)


def bits(t):
    return t.contiguous().view(torch.int32)


def assert_same_mesh(a, b):
    assert a[0].shape == b[0].shape and a[1].shape == b[1].shape
    assert torch.equal(a[1], b[1])
    assert torch.equal(bits(a[0]), bits(b[0]))


# steep fields: u = 8 (|x - c| - r) on the 33^3 lattice of [-1, 1]^3 (h = 1/16, coarse spacing 8h = 0.5).  The band is
# sqrt(3) 8 h in u, sqrt(3) h in distance: a sphere of radius 4.5h centred 0.45h off a brick's centre toward one coarse
# corner reaches that corner's band, and pokes through the brick's three far faces into bricks none of whose corners is in
# the band.  Centred on the brick's centre, the same sphere is 1.9h from all eight corners: no coarse test sees it.
H33 = 2.0 / 32
STEEP_GROW = sphere([-1.0 + 12.45 * H33] * 3, 4.5 * H33, 8.0)
STEEP_TINY = sphere([-1.0 + 28.0 * H33] * 3, 4.5 * H33, 8.0)
NORMAL = sphere((-0.45, -0.4, -0.42), 0.35)


@pytest.mark.parametrize("lat", list(LATTICES))
@pytest.mark.parametrize("field", list(FIELDS))
def test_oracle_narrowband_equals_dense(field, lat):
    axes = axes_of(lat)
    fn = FIELDS[field]
    v, t, active, rounds = oracle_nb(fn, axes)
    ref = oracle_mc(lattice_values(fn, axes))
    assert t.shape[0] > 100
    assert_same_mesh((v, t), ref)
    nb = [(a.shape[0] - 2) // 8 + 1 for a in axes]
    if min(nb) >= 8:
        assert active.shape[0] < nb[0] * nb[1] * nb[2]              # the band is narrower than the lattice
    assert torch.equal(torch.sort(torch.cat(rounds)).values, active)


def test_oracle_steep_sphere_grows_and_equals_dense():
    """The coarse test misses bricks that hold crossings; one grow round adds them (a single sphere this small reaches no
    brick that only a brick of the grow round touches), and the result is the dense mesh."""
    axes = [torch.linspace(-1.0, 1.0, 33)] * 3
    v, t, active, rounds = oracle_nb(STEEP_GROW, axes)
    assert len(rounds) - 1 >= 1 and rounds[1].shape[0] > 0
    assert_same_mesh((v, t), oracle_mc(lattice_values(STEEP_GROW, axes)))


def test_oracle_isolated_steep_component_is_missed():
    """The documented gap: a steep, tiny closed surface between coarse points is absent; the rest is the dense mesh."""
    axes = [torch.linspace(-1.0, 1.0, 33)] * 3
    both = union(NORMAL, STEEP_TINY)
    v, t, _, _ = oracle_nb(both, axes)
    dense_both = oracle_mc(lattice_values(both, axes))
    dense_normal = oracle_mc(lattice_values(NORMAL, axes))
    tiny = oracle_mc(lattice_values(STEEP_TINY, axes))
    assert tiny[1].shape[0] > 100 and dense_both[1].shape[0] == dense_normal[1].shape[0] + tiny[1].shape[0]
    assert oracle_nb(STEEP_TINY, axes)[1].shape[0] == 0
    assert_same_mesh((v, t), dense_normal)


def test_oracle_band_constant():
    """band = sqrt(3) * 8 * h_max in fp32, h_max the largest spacing of any axis"""
    from tensoflow_b200.isosurface import narrowband_band
    axes = axes_of("33x70x65")
    h = max(float((a[1:] - a[:-1]).max()) for a in axes)
    assert narrowband_band(axes) == float(torch.tensor(math.sqrt(3.0) * 8 * h, dtype=torch.float32))


# ---- no CPU path, no lattice above 4096 points per axis ---------------------------------------------------------------
def test_cpu_tensors_and_oversized_lattices_raise_before_any_launch():
    from tensoflow_b200 import _lib
    from tensoflow_b200.isosurface import marching_cubes_narrowband
    from tensoflow_b200.shape_renderer import ShapeRenderer
    n0 = _lib.launch_count()
    fn = FIELDS["sphere"]
    with pytest.raises(RuntimeError, match="CUDA"):
        marching_cubes_narrowband(fn, axes_of("33"))
    with pytest.raises(RuntimeError, match="4096"):
        marching_cubes_narrowband(fn, [torch.linspace(-1, 1, 4097), torch.linspace(-1, 1, 8), torch.linspace(-1, 1, 8)])
    with pytest.raises(RuntimeError, match="4096"):
        marching_cubes_narrowband(fn, [torch.linspace(-1, 1, 8)] * 2)
    with pytest.raises(RuntimeError, match="4096"):
        marching_cubes_narrowband(fn, [torch.linspace(-1, 1, 8), torch.linspace(-1, 1, 1), torch.linspace(-1, 1, 8)])
    shape = ShapeRenderer(dict(device='cpu', gridSize=[16] * 3, sdf_n_comp=4, sdf_dim=32, app_dim=16,
                               shader_config=dict(env_res=16, env_min_res=4)))
    with pytest.raises(RuntimeError):
        shape.extract_geometry([-1.0] * 3, [1.0] * 3, 2048)                 # the narrow-band branch
    assert _lib.launch_count() == n0
