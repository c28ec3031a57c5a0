"""The pure-tensor host logic of the product (sampler helpers of tensoflow_b200/shape_renderer.py, losses, encodings) and the
oracle restatements that check its kernels: pinned to stored values of seeded inputs (tests/golden/pins_host_logic_cpu.npz,
oracle/golden_pins.py) and, where the original project's source tree is present, to its own functions through the shim."""
import pytest
import torch
import torch.nn.functional as F

from conftest import rel_err
from oracle import golden_pins, ref_shim


def _sdf_sphere(x):
    return (x.norm(dim=-1, keepdim=True) - 0.45) + 0.02 * torch.sin(7 * x[..., :1])


def test_sample_pdf_and_weights_match_reference():
    """The product runs these on the tf_sampler_* / tf_probe_* kernels (GPU tests: tests/test_renderer.py); here their checker --
    the oracle's restatements of sample_pdf(det=True), get_sphere_intersection, get_weights and get_intersection -- is pinned to
    the reference's own functions (utils/network_utils.py:108-202), bit for bit."""
    golden_pins.check("test_host_logic_cpu", "sampler", PINS["sampler"]())
    if not ref_shim.available():
        return
    ref_shim.install()
    import utils.network_utils as RU
    from tensoflow_b200 import shape_renderer as P
    from oracle import torch_oracle_renderer as OR
    torch.manual_seed(0)
    pn, sn = 64, 33
    z = torch.sort(torch.rand(pn, sn) * 2.0, dim=-1).values
    w = torch.rand(pn, sn - 1) ** 3
    w[:5] = 0.0                                                       # rays without any surface: uniform fallback
    assert torch.equal(OR.sample_pdf_det(z, w, 9), RU.sample_pdf(z, w, 9, True))
    o = torch.nn.functional.normalize(torch.randn(pn, 3), dim=-1) * 0.9
    d = torch.nn.functional.normalize(-o + 0.3 * torch.randn(pn, 3), dim=-1)
    inv = lambda p: torch.full_like(p[..., :1], 37.0)
    zz = P.get_sphere_intersection(o, d) * torch.linspace(0, 1, 24)[None]
    assert torch.equal(P.get_sphere_intersection(o, d), RU.get_sphere_intersection(o, d))
    assert torch.equal(OR.sphere_exit(o, d), RU.get_sphere_intersection(o, d))
    wa = OR.probe_weights(lambda x: _sdf_sphere(x).reshape(-1), 37.0, zz, o, d)
    wb, _ = RU.get_weights(_sdf_sphere, inv, zz, o, d)
    assert torch.equal(wa, wb)
    pa = OR.occlusion_probability(lambda x: _sdf_sphere(x).reshape(-1), 37.0, o, d, sn0=32, sn1=9)
    _, hw, _ = RU.get_intersection(_sdf_sphere, inv, o, d, sn0=32, sn1=9)
    assert torch.equal(pa, hw.sum(-1, keepdim=True))


def test_upsample_and_ball_radii_match_reference():
    golden_pins.check("test_host_logic_cpu", "upsample", PINS["upsample"]())
    if not ref_shim.available():
        return
    ref_shim.install()
    import network.shapeRenderer as RS
    from tensoflow_b200 import shape_renderer as P
    torch.manual_seed(1)
    pn, sn = 48, 40
    o = torch.nn.functional.normalize(torch.randn(pn, 3), dim=-1) * 2.0
    d = torch.nn.functional.normalize(-o + 0.2 * torch.randn(pn, 3), dim=-1)
    near, far = P.near_far_from_sphere(o, d, 1.0)
    z = near + (far - near) * torch.linspace(0, 1, sn)[None]
    sdf = _sdf_sphere(o[:, None, :] + d[:, None, :] * z[..., None])[..., 0]
    inv_s = torch.full((pn, sn - 1), 64.0)
    # the product's sampler is the tf_sampler_* kernels (GPU test: tests/test_renderer.py); their checker, the oracle's
    # restatement of upsample + sample_pdf, is pinned here to the reference's own function
    from oracle import torch_oracle_renderer as OR
    a = OR.ShapeRenderer._upsample(None, o, d, z, sdf, 16, inv_s)
    b = RS.ShapeRenderer.upsample(o, d, z, sdf, 16, inv_s)
    assert torch.equal(a, b)
    dist, radiis, cos = torch.rand(pn, 1) * 3 + 0.5, torch.rand(pn, 1) * 2e-3 + 1e-4, torch.rand(pn, 1) * 0.5 + 0.5
    assert torch.equal(P.compute_ball_radii(dist, radiis, cos), RS.ShapeRenderer.compute_ball_radii(dist, radiis, cos))


def test_surface_refinement_helpers_match_reference():
    """MaterialRenderer.near_far_from_sphere == the reference's, and the checker of the kernel-backed
    get_intersection_around_mesh (oracle surface_refine's depth; GPU test tests/test_nvs_gpu.py) == the reference's
    get_intersection_around_mesh + the depth reduction of trace_sdf_with_mesh (materialRenderer.py:281-343)."""
    import types
    golden_pins.check("test_host_logic_cpu", "surface", PINS["surface"]())
    if not ref_shim.available():
        return
    ref_shim.install()
    import network.materialRenderer as RM
    from tensoflow_b200.material import MaterialRenderer as PM
    from oracle import torch_oracle_renderer as OR
    torch.manual_seed(2)
    pn = 80
    o = torch.nn.functional.normalize(torch.randn(pn, 3), dim=-1) * 2.0
    d = torch.nn.functional.normalize(-o + 0.15 * torch.randn(pn, 3), dim=-1)
    m_depth = 2.0 - 0.45 + 0.03 * torch.randn(pn, 1)
    inv = lambda p: torch.full_like(p[..., :1], 25.0)
    unit, radius = torch.tensor(2.0 / 63), torch.tensor(1.0)
    ref, mine = types.SimpleNamespace(radius=radius, unit_size=unit), types.SimpleNamespace(radius=radius, unit_size=unit)
    ref.near_far_from_sphere = types.MethodType(RM.MaterialRenderer.near_far_from_sphere, ref)
    mine.near_far_from_sphere = types.MethodType(PM.near_far_from_sphere, mine)
    for a, b in zip(mine.near_far_from_sphere(o, d), ref.near_far_from_sphere(o, d)):
        assert torch.equal(a, b)
    z, w, _ = RM.MaterialRenderer.get_intersection_around_mesh(ref, _sdf_sphere, inv, o, d, m_depth, 32, 9)
    w = w / torch.sum(w, dim=-1, keepdim=True)
    w = torch.where(torch.isnan(w), torch.full_like(w, 1. / 8), w)
    want = torch.sum(w * z, -1, keepdim=True)
    field = types.SimpleNamespace(sdf=lambda x, lvl: _sdf_sphere(x), gradient=lambda x, lvl: (torch.nn.functional.normalize(x, dim=-1), None))
    got, _, _ = OR.surface_refine(field, 25.0, o, d, m_depth, unit, radius, 32, 9)
    assert torch.equal(got, want)


def test_alpha_mask_encodings_and_losses_match_reference():
    golden_pins.check("test_host_logic_cpu", "encodings", PINS["encodings"]())
    if not ref_shim.available():
        return
    ref_shim.install()
    import network.shapeRenderer as RS
    import utils.network_utils as RU
    import utils.ref_utils as RR
    from tensoflow_b200 import shape_renderer as P
    from tensoflow_b200.flow import posenc
    from tensoflow_b200.material import ide_encode
    from tensoflow_b200.shape_shader import ide_encode_rough
    torch.manual_seed(3)
    aabb = torch.tensor([[-1.0, -0.8, -1.2], [1.0, 0.9, 1.1]])
    vol = (torch.rand(12, 10, 14) > 0.6).float()
    x = (torch.rand(500, 3) * 2.4 - 1.2)
    from oracle import torch_oracle_renderer as OR         # the product's lookup is a CUDA kernel (tests/test_renderer.py); here
    a = OR.alpha_mask_sample(vol, aabb, x)                  # the oracle restatement is pinned to the reference class
    b = RS.AlphaGridMask('cpu', aabb, vol).sample_alpha(x)
    assert torch.equal(a, b)
    for multires in (3, 4, 6, 8):                                      # get_embedder (utils/network_utils.py:6-50)
        emb, dim = RU.get_embedder(multires, 3)
        assert torch.equal(posenc(x, multires), emb(x)) and dim == 3 + 6 * multires
    d = torch.nn.functional.normalize(torch.randn(400, 3), dim=-1)
    ide = RR.generate_ide_fn(5)                                        # complex arithmetic in the reference, real recurrences here
    rough = torch.rand(400, 1)
    from oracle import torch_oracle_mc as MC                            # the reference function is fp32-only: fp64 arbiter = oracle
    want0, want1 = MC.ide_encode(d.double(), 0), MC.ide_encode(d.double(), rough.double())
    # fp32 evaluation of the degree-16 harmonics carries ~4e-3 of rounding in the reference as well
    assert rel_err(ide_encode(d), want0) < 4 * max(rel_err(ide(d, torch.zeros(400, 1)), want0), 1e-4)
    assert rel_err(ide_encode_rough(d, rough), want1) < 4 * max(rel_err(ide(d, rough), want1), 1e-4)
    pr, gt = torch.rand(64, 3), torch.rand(64, 3)
    assert torch.equal(P.charbonnier(pr, gt), torch.sqrt(torch.sum((gt - pr) ** 2, dim=-1) + 0.001))   # shapeRenderer.py:803-805


def test_loss_variants_and_schedules_match_reference():
    import types
    golden_pins.check("test_host_logic_cpu", "losses", PINS["losses"]())
    from tensoflow_b200.shape_renderer import ShapeRenderer
    with pytest.raises(NotImplementedError):
        ShapeRenderer.compute_rgb_loss(types.SimpleNamespace(cfg={'rgb_loss': 'huber'}), torch.rand(4, 3), torch.rand(4, 3))
    if not ref_shim.available():
        return
    ref_shim.install()
    import network.shapeRenderer as RS
    import network.materialRenderer as RM
    from tensoflow_b200.shape_renderer import ShapeRenderer as PS
    from tensoflow_b200.material import MaterialRenderer as PM
    torch.manual_seed(4)
    pr, gt = torch.rand(100, 3), torch.rand(100, 3)
    for kind in ('l2', 'l1', 'smooth_l1', 'charbonier'):
        s = types.SimpleNamespace(cfg={'rgb_loss': kind})
        assert torch.equal(PS.compute_rgb_loss(s, pr, gt), RS.ShapeRenderer.compute_rgb_loss(s, pr, gt)), kind
    for kind in ('l1', 'charbonier'):
        s = types.SimpleNamespace(cfg={'rgb_loss': kind, 'reg_diffuse_light_lambda': 0.1})
        assert torch.equal(PM.compute_rgb_loss(s, pr, gt), RM.MaterialRenderer.compute_rgb_loss(s, pr, gt)), kind
        assert torch.equal(PM.compute_diffuse_light_regularization(s, pr), RM.MaterialRenderer.compute_diffuse_light_regularization(s, pr))
    with pytest.raises(NotImplementedError):
        PS.compute_rgb_loss(types.SimpleNamespace(cfg={'rgb_loss': 'huber'}), pr, gt)
    for anneal_end in (-1, 50000):                                     # cos-anneal schedule (shapeRenderer.py get_anneal_val)
        s = types.SimpleNamespace(cfg={'anneal_end': anneal_end})
        for step in (0, 1, 24999, 50000, 300000):
            assert PS.get_anneal_val(s, step) == RS.ShapeRenderer.get_anneal_val(s, step)


# ------------------------------------------------------------------ pinned values (the seeded inputs of the tests above)
def _sampler_values():
    from tensoflow_b200 import shape_renderer as P
    from oracle import torch_oracle_renderer as OR
    torch.manual_seed(0)
    pn, sn = 64, 33
    z = torch.sort(torch.rand(pn, sn) * 2.0, dim=-1).values
    w = torch.rand(pn, sn - 1) ** 3
    w[:5] = 0.0
    o = F.normalize(torch.randn(pn, 3), dim=-1) * 0.9
    d = F.normalize(-o + 0.3 * torch.randn(pn, 3), dim=-1)
    zz = P.get_sphere_intersection(o, d) * torch.linspace(0, 1, 24)[None]
    sdf = lambda x: _sdf_sphere(x).reshape(-1)
    return [("sample_pdf", OR.sample_pdf_det(z, w, 9), 0), ("sphere_exit", P.get_sphere_intersection(o, d), 0),
            ("sphere_exit", OR.sphere_exit(o, d), 0), ("weights", OR.probe_weights(sdf, 37.0, zz, o, d), 0),
            ("occlusion", OR.occlusion_probability(sdf, 37.0, o, d, sn0=32, sn1=9), 0)]


def _upsample_values():
    from tensoflow_b200 import shape_renderer as P
    from oracle import torch_oracle_renderer as OR
    torch.manual_seed(1)
    pn, sn = 48, 40
    o = F.normalize(torch.randn(pn, 3), dim=-1) * 2.0
    d = F.normalize(-o + 0.2 * torch.randn(pn, 3), dim=-1)
    near, far = P.near_far_from_sphere(o, d, 1.0)
    z = near + (far - near) * torch.linspace(0, 1, sn)[None]
    sdf = _sdf_sphere(o[:, None, :] + d[:, None, :] * z[..., None])[..., 0]
    inv_s = torch.full((pn, sn - 1), 64.0)
    up = OR.ShapeRenderer._upsample(None, o, d, z, sdf, 16, inv_s)
    dist, radiis, cos = torch.rand(pn, 1) * 3 + 0.5, torch.rand(pn, 1) * 2e-3 + 1e-4, torch.rand(pn, 1) * 0.5 + 0.5
    return [("upsample", up, 0), ("ball_radii", P.compute_ball_radii(dist, radiis, cos), 0)]


def _surface_values():
    import types
    from tensoflow_b200.material import MaterialRenderer as PM
    from oracle import torch_oracle_renderer as OR
    torch.manual_seed(2)
    pn = 80
    o = F.normalize(torch.randn(pn, 3), dim=-1) * 2.0
    d = F.normalize(-o + 0.15 * torch.randn(pn, 3), dim=-1)
    m_depth = 2.0 - 0.45 + 0.03 * torch.randn(pn, 1)
    unit, radius = torch.tensor(2.0 / 63), torch.tensor(1.0)
    mine = types.SimpleNamespace(radius=radius, unit_size=unit)
    near, far = types.MethodType(PM.near_far_from_sphere, mine)(o, d)
    field = types.SimpleNamespace(sdf=lambda x, lvl: _sdf_sphere(x), gradient=lambda x, lvl: (F.normalize(x, dim=-1), None))
    depth, _, _ = OR.surface_refine(field, 25.0, o, d, m_depth, unit, radius, 32, 9)
    return [("near", near, 0), ("far", far, 0), ("depth", depth, 0)]


def _encoding_values():
    from tensoflow_b200.flow import posenc
    from tensoflow_b200.material import ide_encode
    from tensoflow_b200.shape_shader import ide_encode_rough
    from oracle import torch_oracle_renderer as OR
    torch.manual_seed(3)
    aabb = torch.tensor([[-1.0, -0.8, -1.2], [1.0, 0.9, 1.1]])
    vol = (torch.rand(12, 10, 14) > 0.6).float()
    x = (torch.rand(500, 3) * 2.4 - 1.2)
    out = [("alpha_mask", OR.alpha_mask_sample(vol, aabb, x), 0)]
    out += [(f"posenc{m}", posenc(x, m), 0) for m in (3, 4, 6, 8)]
    d = F.normalize(torch.randn(400, 3), dim=-1)
    rough = torch.rand(400, 1)
    return out + [("ide", ide_encode(d), 0), ("ide_rough", ide_encode_rough(d, rough), 0)]


def _loss_values():
    import types
    from tensoflow_b200.shape_renderer import ShapeRenderer as PS
    from tensoflow_b200.material import MaterialRenderer as PM
    torch.manual_seed(4)
    pr, gt = torch.rand(100, 3), torch.rand(100, 3)
    out = [(f"shape_{k}", PS.compute_rgb_loss(types.SimpleNamespace(cfg={'rgb_loss': k}), pr, gt), 0)
           for k in ('l2', 'l1', 'smooth_l1', 'charbonier')]
    for k in ('l1', 'charbonier'):
        s = types.SimpleNamespace(cfg={'rgb_loss': k, 'reg_diffuse_light_lambda': 0.1})
        out += [(f"material_{k}", PM.compute_rgb_loss(s, pr, gt), 0),
                (f"diffuse_light_reg_{k}", PM.compute_diffuse_light_regularization(s, pr), 0)]
    anneal = [[PS.get_anneal_val(types.SimpleNamespace(cfg={'anneal_end': e}), step) for step in (0, 1, 24999, 50000, 300000)]
              for e in (-1, 50000)]
    return out + [("anneal", torch.tensor(anneal, dtype=torch.float64), 0)]


PINS = {"sampler": _sampler_values, "upsample": _upsample_values, "surface": _surface_values, "encodings": _encoding_values,
        "losses": _loss_values}
