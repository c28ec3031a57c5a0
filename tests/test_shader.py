"""Shape-stage shader + prefiltered env light: oracle vs reference golden (CPU) and the CUDA
product vs the same reference outputs (GPU).  Fixture: tests/golden/shader.npz, produced by
oracle/gen_golden.py from the reference's own ShapeShadingNetwork / EnvLight."""
import pytest
import torch

from conftest import rel_err
from test_golden import load
from oracle import torch_oracle_shader as SH


def _oracle(g, dtype=torch.float32):
    m = SH.ShapeShadingNetwork(has_radiance_field=True, env_res=16, env_min_res=4, dtype=dtype)
    res = m.load_state_dict({k: v.to(dtype) for k, v in g["state"].items()}, strict=False)
    assert not res.unexpected_keys and res.missing_keys == ["FG_LUT"], res
    return m


def _run(m, i, dt, dev="cpu"):
    nrm = i["normals"].detach().clone().to(dev, dt).requires_grad_()
    feat = i["features"].detach().clone().to(dev, dt).requires_grad_()
    return nrm, feat


def test_oracle_shader_golden():
    g = load("shader.npz")
    m = _oracle(g)
    i, o = g["inputs"], g["outputs"]
    m.envlight.build_mips()
    assert rel_err(m.envlight.diffuse, o["diffuse"]) < 1e-6
    for k, s in enumerate(m.envlight.specular):
        assert rel_err(s, o[f"specular{k}"]) < 1e-6
    nrm, feat = _run(m, i, torch.float32)
    color, rad, occ = m(i["points"], nrm, i["view_dirs"], feat, with_radiance=True)
    assert rel_err(color, o["color"]) < 1e-5 and rel_err(rad, o["radiance"]) < 1e-5
    assert rel_err(occ["occ_prob"], o["occ_prob"]) < 1e-5 and rel_err(occ["roughness"], o["roughness"]) < 1e-6
    ((color * i["u"]).sum() + rad.sum() + occ["occ_prob"].sum()).backward()
    assert rel_err(nrm.grad, g["grads"]["__normals"]) < 1e-4
    assert rel_err(feat.grad, g["grads"]["__features"]) < 1e-4
    for n, p in m.named_parameters():
        if n in g["grads"]:
            assert rel_err(p.grad, g["grads"][n]) < 1e-4, n


@pytest.mark.gpu
def test_cuda_shader_golden():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    from tensoflow_b200.shape_shader import ShapeShadingNetwork
    dev = torch.device("cuda:0")
    g = load("shader.npz")
    i, o = g["inputs"], g["outputs"]
    m = ShapeShadingNetwork(dict(has_radiance_field=True, radiance_field_step=0, env_res=16, env_min_res=4, device=dev))
    res = m.load_state_dict(g["state"], strict=False)
    # the fixture was written without the reference's idle `outer_light` head (registered for checkpoint round trips only)
    assert not res.unexpected_keys and [k for k in res.missing_keys if not k.startswith("outer_light")] == ["FG_LUT"], res
    m64 = _oracle(g, torch.float64)
    m.envlight.build_mips()
    m64.envlight.build_mips()
    assert rel_err(m.envlight.diffuse, o["diffuse"]) < 1e-5
    for k, s in enumerate(m.envlight.specular):
        assert rel_err(s, o[f"specular{k}"]) < 1e-5
    nrm, feat = _run(m, i, torch.float32, dev)
    color, rad, occ = m(i["points"].to(dev), nrm, i["view_dirs"].to(dev), feat, None, step=10)
    n64, f64 = _run(m64, i, torch.float64)
    c64, r64, o64 = m64(i["points"].double(), n64, i["view_dirs"].double(), f64, with_radiance=True)

    def close(got, ref32, ref64, tol, what):
        e, e_ref = rel_err(got, ref64), rel_err(ref32, ref64)
        assert e <= max(tol, 4 * e_ref), f"{what}: rel err {e:.3e} (reference fp32 vs fp64 oracle {e_ref:.3e})"

    close(color, o["color"], c64, 1e-4, "color")
    close(rad, o["radiance"], r64, 1e-4, "radiance")
    close(occ["occ_prob"], o["occ_prob"], o64["occ_prob"], 1e-4, "occ_prob")
    close(occ["roughness"], o["roughness"], o64["roughness"], 1e-4, "roughness")
    ((color * i["u"].to(dev)).sum() + rad.sum() + occ["occ_prob"].sum()).backward()
    ((c64 * i["u"].double()).sum() + r64.sum() + o64["occ_prob"].sum()).backward()
    close(nrm.grad, g["grads"]["__normals"], n64.grad, 1e-3, "d normals")
    close(feat.grad, g["grads"]["__features"], f64.grad, 1e-3, "d features")
    p64 = dict(m64.named_parameters())
    for n, p in m.named_parameters():
        if n in g["grads"]:
            assert p.grad is not None, n
            close(p.grad, g["grads"][n], p64[n].grad, 1e-3, f"d {n}")


@pytest.mark.gpu
@pytest.mark.parametrize("with_level", [False, True])
def test_cube_lookup_kernel_matches_oracle_texture_cube(with_level):
    """tf_cube_sample_fwd/bwd against the oracle's texture_cube / texture_cube_mip (the tensor formulation the oracle shader of
    the golden test above runs on) in fp64: values and the gradients wrt every texture level, the direction and the mip level."""
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    import torch.nn.functional as F
    from conftest import rel_err
    from tensoflow_b200 import shape_shader as S
    from oracle import torch_oracle_mat as OM
    dev = torch.device("cuda:0")
    g = torch.Generator().manual_seed(5)
    res = [32, 16, 8, 4] if with_level else [16]
    texs = [torch.randn(6, r, r, 3, generator=g) * 0.5 for r in res]
    d = F.normalize(torch.randn(6000, 3, generator=g), dim=-1)
    # directions within a texel of cube edges / corners exercise the fold and the dropped corner tap
    e = F.normalize(torch.tensor([[1.0, 1.0, 0.3], [1.0, -1.0, 0.99], [0.98, 1.0, 1.0], [-1.0, 0.2, 1.0], [0.1, -1.0, -1.0]]), dim=-1)
    e = F.normalize(e[None] + 0.03 * torch.randn(300, 5, 3, generator=g), dim=-1).reshape(-1, 3)
    d = torch.cat([d, e], 0) * (0.5 + torch.rand(7500, 1, generator=g))          # un-normalised directions are legal inputs
    n = d.shape[0]
    level = torch.rand(n, generator=g) * 4.0 - 0.5 if with_level else None        # below 0 and above L-1: clamped
    if with_level:
        level[:50] = torch.randint(0, 4, (50,), generator=g).float()              # integer levels (f = 0)
    u = torch.randn(n, 3, generator=g)

    def tensor_version(dt):
        tx = [t.detach().clone().to(dt).requires_grad_() for t in texs]
        dd = d.detach().clone().to(dt).requires_grad_()
        lv = None if level is None else level.detach().clone().to(dt).requires_grad_()
        out = OM.texture_cube(tx[0], dd) if lv is None else OM.texture_cube_mip(tx, dd, lv)
        (out * u.to(dt)).sum().backward()
        return out, [t.grad for t in tx], dd.grad, None if lv is None else lv.grad

    o64, gt64, gd64, gl64 = tensor_version(torch.float64)
    o32, gt32, gd32, gl32 = tensor_version(torch.float32)
    tx = [t.detach().clone().to(dev).requires_grad_() for t in texs]
    dd = d.detach().clone().to(dev).requires_grad_()
    lv = None if level is None else level.detach().clone().to(dev).requires_grad_()
    out = S.cube_lookup(tx, dd, lv)
    (out * u.to(dev)).sum().backward()

    def close(a, b32, b64, tol, what):
        e_, e_ref = rel_err(a, b64), rel_err(b32, b64)
        assert e_ <= max(tol, 4 * e_ref), f"{what}: {e_:.3e} (fp32 tensor version {e_ref:.3e})"

    close(out, o32, o64, 1e-5, "out")
    for l in range(len(res)):
        close(tx[l].grad, gt32[l], gt64[l], 1e-4, f"d tex[{l}]")
    close(dd.grad, gd32, gd64, 1e-4, "d dirs")
    if with_level:
        close(lv.grad, gl32, gl64, 1e-4, "d level")
        outside = (level < 0) | (level > 3)
        assert float(lv.grad.cpu()[outside].abs().max()) == 0.0
