"""CPU tests of the TensoFlow oracle: self-consistency identities (the reference's only
known-answer material for the flow, SURVEY 8c), values pinned to stored outputs of seeded inputs
(tests/golden/pins_oracle_flow_cpu.npz, oracle/golden_pins.py) and, where the original project's source tree is present,
exact agreement with its own network/flow.py through the shim."""
import pytest
import torch

from oracle import golden_pins, torch_oracle_mat as OM, ref_shim


def test_spline_round_trip_and_unit_mass():
    torch.manual_seed(0)
    st = torch.randn(2000, 21, dtype=torch.float64)
    y = torch.rand(2000, dtype=torch.float64).clamp(1e-6, 1 - 1e-6)
    x, lj = OM.pwquad_inverse(y, st)
    back, lj2 = OM.pwquad_forward(x, st)
    assert float((back - y).abs().max()) < 1e-7          # reference measured 9.9e-8 in fp32
    assert float((lj + lj2).abs().max()) < 1e-5
    # the forward spline is a CDF: F(0+)=0, F(1-)=1, monotone
    g = torch.linspace(1e-6, 1 - 1e-6, 257, dtype=torch.float64)
    F = torch.stack([OM.pwquad_forward(g, st[i:i + 1].expand(257, -1))[0] for i in range(8)])
    assert float(F[:, 0].max()) < 1e-4 and float((1 - F[:, -1]).max()) < 1e-4
    assert bool((F[:, 1:] >= F[:, :-1]).all())


def test_prior_angles():
    a = OM.sphere_prior_angles(64)
    assert a.shape == (64, 2) and float(a.min()) >= 0 and float(a.max()) <= 1
    a32 = OM.sphere_prior_angles(32)
    assert a32.shape == (32, 2)


def test_sample_density_consistency():
    torch.manual_seed(0)
    f = OM.TensoFlow(torch.tensor([[-1., -1, -1], [1, 1, 1]]), gridSize=(16, 16, 16))
    pts, va, r = torch.rand(40, 3) - 0.5, torch.rand(40, 2), torch.rand(40, 1)
    with torch.no_grad():
        x, lj = f.sample(pts, va, r, 64, None)
        z, lq = f(pts, va, r, x)
    assert float((lj + lq).abs().max()) < 2e-2           # reference: <= 8e-3 (SURVEY appendix D-5)


def test_oracle_matches_reference_tensoflow():
    golden_pins.check("test_oracle_flow_cpu", "tensoflow", PINS["tensoflow"]())
    if not ref_shim.available():
        return
    ref_shim.install()
    import network.flow as RFL
    torch.manual_seed(0)
    aabb = torch.tensor([[-1., -1, -1], [1, 1, 1]])
    ref = RFL.TensoFlow(d=2, aabb=aabb, device='cpu', gridSize=[16, 16, 16])
    mine = OM.TensoFlow(aabb, gridSize=(16, 16, 16))
    with torch.no_grad():
        for p in ref.nis_plane:
            p.mul_(1000)
    res = mine.load_state_dict(ref.state_dict(), strict=False)
    assert not res.unexpected_keys
    pn, sn = 30, 64
    pts, va, rough = torch.rand(pn, 3) * 1.8 - 0.9, torch.rand(pn, 2), torch.rand(pn, 1)
    ref.eval()
    a, la = ref.sample(pts, va, rough, sn, return_jacobian=True)
    b, lb = mine.sample(pts, va, rough, sn, None)
    assert torch.equal(a, b) and torch.equal(la, lb)
    ref.train()
    shift = torch.rand(pn, sn, 1)
    orig = torch.rand_like
    torch.rand_like = lambda x, *a_, **k: shift
    try:
        a, la = ref.sample(pts, va, rough, sn, return_jacobian=True)
    finally:
        torch.rand_like = orig
    b, lb = mine.sample(pts, va, rough, sn, shift)
    assert torch.equal(a, b) and torch.equal(la, lb)
    rid = torch.sort(torch.randint(0, pn, (200,)))[0]
    xr = torch.rand(200, 2)
    z, lq = ref(pts, va, rough, xr, return_jacobian=True, rays_id=rid)
    z2, lq2 = mine(pts, va, rough, xr, rays_id=rid)
    assert torch.equal(z, z2) and torch.equal(lq, lq2)
    lq.sum().backward()
    lq2.sum().backward()
    gm = dict(mine.named_parameters())
    for n, p in ref.named_parameters():
        if p.grad is not None:
            assert torch.allclose(p.grad, gm[n].grad, rtol=0, atol=0), n


@pytest.mark.parametrize("version", ["direction", "sphere_direction"])
def test_oracle_outer_mlp_lights_match_reference(version):
    """MLP outer lights (reference fields.py:716-721, 913-928; `outer_light_version: direction` is the reference default and the
    setting of 8 shipped material configs): oracle predict_outer_lights == the reference class's, same weights."""
    import torch.nn.functional as F
    from conftest import rel_err
    golden_pins.check("test_oracle_flow_cpu", f"outer_lights_{version}", PINS[f"outer_lights_{version}"]())
    if not ref_shim.available():
        return
    ref_shim.install()
    import network.fields as RF
    from oracle import torch_oracle_mc as MC
    torch.manual_seed(3)
    aabb = torch.tensor([[-1., -1, -1], [1, 1, 1]])
    tracer = MC.analytic_sphere_tracer(0.45)
    ref = RF.MCShadingNetwork(dict(outer_light_version=version, light_exp_max=5.0, inner_light_exp_max=5.0, human_lights=False,
                                   gridSize=[16, 16, 16]), tracer, aabb)
    mine = MC.MCShadingNetwork(tracer, aabb, gridSize=(8, 8, 8), flow_grid=(16, 16, 16), outer_light_version=version)
    with torch.no_grad():
        for p in ref.outer_light.parameters():
            p.add_(0.1 * torch.randn_like(p))
    mine.outer_light.load_state_dict(ref.outer_light.state_dict())
    n = 500
    pts = F.normalize(torch.randn(n, 3), dim=-1) * torch.rand(n, 1)
    pts[:20] = F.normalize(pts[:20], dim=-1) * (0.999 + 0.0019 * torch.rand(20, 1))    # the `> 0.999 -> shrink` branch (the reference asserts beyond ~1.001)
    dirs = F.normalize(torch.randn(n, 3), dim=-1)
    a = ref.predict_outer_lights(pts, dirs)
    b = mine.predict_outer_lights(pts, dirs)
    assert a.shape == (n, 3) and rel_err(b, a) < 1e-6


# ------------------------------------------------------------------ pinned values (seeded oracle modules and inputs)
def _tensoflow_values():
    torch.manual_seed(0)
    f = OM.TensoFlow(torch.tensor([[-1., -1, -1], [1, 1, 1]]), gridSize=(16, 16, 16))
    with torch.no_grad():
        for p in f.nis_plane:
            p.mul_(1000)
    pn, sn = 30, 64
    pts, va, rough = torch.rand(pn, 3) * 1.8 - 0.9, torch.rand(pn, 2), torch.rand(pn, 1)
    a_eval, la_eval = f.sample(pts, va, rough, sn, None)
    shift = torch.rand(pn, sn, 1)
    a, la = f.sample(pts, va, rough, sn, shift)
    rid = torch.sort(torch.randint(0, pn, (200,)))[0]
    z, lq = f(pts, va, rough, torch.rand(200, 2), rays_id=rid)
    lq.sum().backward()
    return ([("angles_eval", a_eval, 0), ("logj_eval", la_eval, 0), ("angles", a, 0), ("logj", la, 0), ("z", z, 0), ("logq", lq, 0)]
            + [(f"d_{n}", p.grad, 0) for n, p in f.named_parameters() if p.grad is not None])


def _outer_light_values(version):
    import torch.nn.functional as F
    from oracle import torch_oracle_mc as MC
    torch.manual_seed(3)
    m = MC.MCShadingNetwork(MC.analytic_sphere_tracer(0.45), torch.tensor([[-1., -1, -1], [1, 1, 1]]), gridSize=(8, 8, 8),
                            flow_grid=(16, 16, 16), outer_light_version=version)
    with torch.no_grad():
        for p in m.outer_light.parameters():
            p.add_(0.1 * torch.randn_like(p))
    n = 500
    pts = F.normalize(torch.randn(n, 3), dim=-1) * torch.rand(n, 1)
    pts[:20] = F.normalize(pts[:20], dim=-1) * (0.999 + 0.0019 * torch.rand(20, 1))
    dirs = F.normalize(torch.randn(n, 3), dim=-1)
    return [("lights", m.predict_outer_lights(pts, dirs), 1e-6)]


PINS = {"tensoflow": _tensoflow_values, "outer_lights_direction": lambda: _outer_light_values("direction"),
        "outer_lights_sphere_direction": lambda: _outer_light_values("sphere_direction")}
