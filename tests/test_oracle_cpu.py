"""CPU tests of the oracle itself: texture semantics, autograd consistency, values pinned to stored outputs of seeded inputs
(tests/golden/pins_oracle_cpu.npz, oracle/golden_pins.py) and, where the original project's source tree is present,
agreement with its own classes through the shim."""
import torch
import torch.nn.functional as F

from oracle import golden_pins, torch_oracle as O, ref_shim
from conftest import rel_err


def test_texture2d_matches_grid_sample():
    """Level-0 clamp-mode bilinear == grid_sample(align_corners=False, border)."""
    torch.manual_seed(0)
    tex = torch.randn(12, 20, 5, dtype=torch.float64)
    uv = torch.rand(500, 2, dtype=torch.float64) * 1.4 - 0.2
    a = O.texture2d(tex, uv, None, 1)
    b = F.grid_sample(tex.permute(2, 0, 1)[None], (uv * 2 - 1)[None, :, None, :], mode="bilinear",
                      padding_mode="border", align_corners=False)[0, :, :, 0].T
    assert rel_err(a, b) < 1e-12


def test_texture2d_mip_levels():
    torch.manual_seed(1)
    tex = torch.randn(16, 16, 3, dtype=torch.float64)
    uv = torch.rand(200, 2, dtype=torch.float64)
    chain = O.build_mip_chain(tex, 3)
    assert chain[1].shape == (8, 8, 3) and chain[2].shape == (4, 4, 3)
    assert torch.allclose(chain[1][0, 0], tex[:2, :2].mean((0, 1)))
    for lv, (l0, l1, f) in {-1.0: (0, 0, 0.0), 0.25: (0, 1, 0.25), 1.0: (1, 1, 0.0), 1.5: (1, 2, 0.5), 7.0: (2, 2, 0.0)}.items():
        got = O.texture2d(tex, uv, torch.full((200,), lv, dtype=torch.float64), 3)
        want = (1 - f) * O._bilinear_clamp(chain[l0], uv) + f * O._bilinear_clamp(chain[l1], uv)
        assert rel_err(got, want) < 1e-12, lv
    line = torch.randn(16, 1, 3, dtype=torch.float64)
    lc = O.build_mip_chain(line, 3)
    assert lc[2].shape == (4, 1, 3)
    assert torch.allclose(lc[1][0, 0], line[:2, 0].mean(0))


def test_weights_and_accumulate():
    torch.manual_seed(2)
    alpha = torch.rand(10, dtype=torch.float64)
    idx = torch.tensor([0, 0, 0, 2, 2, 3, 3, 3, 3, 3])
    w, T = O.render_weight_from_alpha(alpha, idx, 5)
    assert torch.allclose(T[0], torch.tensor(1.0, dtype=torch.float64)) and torch.allclose(T[3], torch.tensor(1.0, dtype=torch.float64))
    assert torch.allclose(T[2], (1 - alpha[0]) * (1 - alpha[1]))
    acc = O.accumulate_along_rays(w, None, idx, 5)
    assert acc.shape == (5, 1) and float(acc[1]) == 0.0 and float(acc[4]) == 0.0


def test_sphere_init_is_a_sphere():
    """Known-answer from the reference's deterministic initialisers (SURVEY 8c): eikonal ~ 1."""
    torch.manual_seed(0)
    f = O.TensoSDF([128] * 3, [[-1.0] * 3, [1.0] * 3], sdf_n_comp=16, sdf_dim=128, app_dim=128, init_n_levels=1)
    x = torch.rand(4096, 3) * 1.6 - 0.8
    out = f(x, None)
    g, _ = f.gradient(x, None)
    assert abs(float(out[:, 0].mean()) - 0.587) < 0.05
    assert abs(float(g.norm(dim=-1).mean()) - 0.99) < 0.05


def test_oracle_matches_reference_tensosdf():
    golden_pins.check("test_oracle_cpu", "tensosdf", PINS["tensosdf"]())
    if not ref_shim.available():
        return
    ref_shim.install()
    import network.fields as RF
    torch.manual_seed(0)
    G = torch.tensor([16, 16, 16]); aabb = torch.tensor([[-1., -1, -1], [1, 1, 1]])
    ref = RF.TensoSDF(G, aabb, device='cpu', sdf_n_comp=8, sdf_dim=32, app_dim=16, init_n_levels=1, sdf_multires=0)
    ref.upsample_volume_grid(torch.tensor([33, 33, 33]))
    ref.upsample_volume_grid(torch.tensor([66, 66, 66]))
    mine = O.TensoSDF(G, aabb, sdf_n_comp=8, sdf_dim=32, app_dim=16, init_n_levels=1)
    mine.upsample_volume_grid(torch.tensor([33, 33, 33])); mine.upsample_volume_grid(torch.tensor([66, 66, 66]))
    assert list(mine.gridSize) == list(ref.gridSize) and mine.n_levels == ref.n_levels == 3
    with torch.no_grad():
        for p in list(ref.sdf_plane) + list(ref.sdf_line):
            p.add_(0.05 * torch.randn_like(p))
    mine.load_state_dict({k: v for k, v in ref.state_dict().items() if 'gaussian' not in k}, strict=False)
    x = torch.rand(777, 3) * 2.2 - 1.1
    lv = torch.rand(777, 1) * 4 - 1
    a, b = ref(x, lv), mine(x, lv)
    assert rel_err(b, a) < 1e-6
    ga, ha = ref.gradient(x, lv, training=True, sdf=a[:, :1])
    gb, hb = mine.gradient(x, lv, training=True, sdf=b[:, :1])
    assert rel_err(gb, ga) < 1e-5 and rel_err(hb, ha) < 1e-4
    (a.sum() + ga.sum()).backward(); (b.sum() + gb.sum()).backward()
    for (n, p), (_, q) in zip(ref.named_parameters(), mine.named_parameters()):
        assert rel_err(q.grad, p.grad) < 1e-5, n


def test_surface_refine_matches_reference_material_renderer():
    """oracle surface_refine == the reference's own MaterialRenderer.trace_sdf_with_mesh (materialRenderer.py:315-343) driven by
    a stand-in tracer (the mesh depth is an input of both)."""
    import types
    golden_pins.check("test_oracle_cpu", "surface_refine", PINS["surface_refine"]())
    if not ref_shim.available():
        return
    ref_shim.install()
    import network.fields as RF
    import network.materialRenderer as MR
    from oracle import torch_oracle_renderer as RR
    torch.manual_seed(0)
    G = torch.tensor([32, 32, 32]); aabb = torch.tensor([[-1., -1, -1], [1, 1, 1]])
    ref_field = RF.TensoSDF(G, aabb, device='cpu', sdf_n_comp=8, sdf_dim=32, app_dim=16, init_n_levels=1, sdf_multires=0)
    with torch.no_grad():
        for p in list(ref_field.sdf_plane) + list(ref_field.sdf_line):
            p.add_(5e-3 * torch.randn_like(p))
    mine = O.TensoSDF(G, aabb, sdf_n_comp=8, sdf_dim=32, app_dim=16, init_n_levels=1)
    mine.load_state_dict({k: v for k, v in ref_field.state_dict().items() if 'gaussian' not in k}, strict=False)
    pn = 200
    o = torch.nn.functional.normalize(torch.randn(pn, 3), dim=-1) * 2.0
    d = torch.nn.functional.normalize((torch.rand(pn, 3) - 0.5) * 0.2 - o, dim=-1)
    m_depth = 2.0 - 0.22 + 0.05 * torch.randn(pn, 1)                 # a bumpy sphere of radius ~0.22 seen from distance 2
    hit = torch.rand(pn) < 0.8
    inv_s = 20.0
    unit = torch.mean((aabb[1] - aabb[0]) / (G - 1))
    radius = (aabb[1] - aabb.mean(0)).mean()

    fake = types.SimpleNamespace()
    fake.radius, fake.unit_size, fake.sdf_network = radius, unit, ref_field
    fake.sdf_inter_fun = lambda x: ref_field.sdf(x, None)
    fake.deviation_net = lambda x: torch.full_like(x[..., :1], inv_s)
    fake.near_far_from_sphere = types.MethodType(MR.MaterialRenderer.near_far_from_sphere, fake)
    fake.get_intersection_around_mesh = types.MethodType(MR.MaterialRenderer.get_intersection_around_mesh, fake)
    fake.trace = lambda ro, rd: (ro + m_depth * rd, -rd.clone(), torch.where(hit[:, None], m_depth, torch.full_like(m_depth, 10.0)).clone(),
                                 hit[:, None].clone())
    inters, normals, depth, hit_out = MR.MaterialRenderer.trace_sdf_with_mesh(fake, o, d, 32, 9)
    dep, pts, n = RR.surface_refine(mine, inv_s, o[hit], d[hit], m_depth[hit], float(unit), float(radius), 32, 9)
    assert torch.equal(hit_out.squeeze(-1), hit)
    assert rel_err(dep, depth[hit]) < 1e-6
    assert rel_err(pts, inters[hit]) < 1e-6
    assert float((n - normals[hit]).abs().max()) < 1e-4


# ------------------------------------------------------------------ pinned values (seeded oracle fields and inputs)
def _tensosdf_values():
    torch.manual_seed(0)
    G = torch.tensor([16, 16, 16]); aabb = torch.tensor([[-1., -1, -1], [1, 1, 1]])
    f = O.TensoSDF(G, aabb, sdf_n_comp=8, sdf_dim=32, app_dim=16, init_n_levels=1)
    f.upsample_volume_grid(torch.tensor([33, 33, 33])); f.upsample_volume_grid(torch.tensor([66, 66, 66]))
    with torch.no_grad():
        for p in list(f.sdf_plane) + list(f.sdf_line):
            p.add_(0.05 * torch.randn_like(p))
    x = torch.rand(777, 3) * 2.2 - 1.1
    lv = torch.rand(777, 1) * 4 - 1
    out = f(x, lv)
    g, h = f.gradient(x, lv, training=True, sdf=out[:, :1])
    (out.sum() + g.sum()).backward()
    return [("out", out, 1e-6), ("grad", g, 1e-5), ("hess", h, 1e-4)] + [(f"d_{n}", p.grad, 1e-5) for n, p in f.named_parameters()]


def _surface_refine_values():
    from oracle import torch_oracle_renderer as RR
    torch.manual_seed(0)
    G = torch.tensor([32, 32, 32]); aabb = torch.tensor([[-1., -1, -1], [1, 1, 1]])
    f = O.TensoSDF(G, aabb, sdf_n_comp=8, sdf_dim=32, app_dim=16, init_n_levels=1)
    with torch.no_grad():
        for p in list(f.sdf_plane) + list(f.sdf_line):
            p.add_(5e-3 * torch.randn_like(p))
    pn = 200
    o = F.normalize(torch.randn(pn, 3), dim=-1) * 2.0
    d = F.normalize((torch.rand(pn, 3) - 0.5) * 0.2 - o, dim=-1)
    m_depth = 2.0 - 0.22 + 0.05 * torch.randn(pn, 1)
    hit = torch.rand(pn) < 0.8
    unit = torch.mean((aabb[1] - aabb[0]) / (G - 1))
    radius = (aabb[1] - aabb.mean(0)).mean()
    dep, pts, n = RR.surface_refine(f, 20.0, o[hit], d[hit], m_depth[hit], float(unit), float(radius), 32, 9)
    return [("depth", dep, 1e-6), ("points", pts, 1e-6), ("normals", n, 1e-4)]


PINS = {"tensosdf": _tensosdf_values, "surface_refine": _surface_refine_values}
