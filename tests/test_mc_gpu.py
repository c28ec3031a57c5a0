"""GPU parity tests of the material stage: BVH tracer, env-light cube lookup, and the whole
MCShadingNetwork (direction sets, occlusion, lights, BRDF estimators, NIS losses, gradients)
against reference outputs (tests/golden/mcshade.npz) and the oracle."""
import numpy as np
import pytest
import torch
import torch.nn.functional as F

from conftest import rel_err
from test_golden import load, occluder_tracer, _oracle_mc, MC_KEYS

pytestmark = pytest.mark.gpu

from oracle import torch_oracle_mat as OM, torch_oracle_mc as MC  # noqa: E402


def _cuda():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    return torch.device("cuda:0")


def bumpy_sphere(nu=40, nv=20, r=0.5):
    """lat-long sphere with radial bumps (the synthetic mesh family of BASELINE config 3)."""
    u = torch.linspace(0, 2 * np.pi, nu + 1)[:-1]
    v = torch.linspace(0.05, np.pi - 0.05, nv)
    vv, uu = torch.meshgrid(v, u, indexing="ij")
    rad = r * (1 + 0.1 * torch.sin(5 * uu) * torch.sin(4 * vv))
    verts = torch.stack([rad * torch.sin(vv) * torch.cos(uu), rad * torch.sin(vv) * torch.sin(uu), rad * torch.cos(vv)], -1).reshape(-1, 3)
    tris = []
    for i in range(nv - 1):
        for j in range(nu):
            a, b = i * nu + j, i * nu + (j + 1) % nu
            c, d = (i + 1) * nu + j, (i + 1) * nu + (j + 1) % nu
            tris += [[a, c, b], [b, c, d]]
    return verts.float(), torch.tensor(tris, dtype=torch.int32)


def brute_force_trace(verts, tris, o, d):
    """Moeller-Trumbore over every triangle in fp64 (closest t > 0)."""
    v0, v1, v2 = (verts[tris[:, k].long()].double() for k in range(3))
    e1, e2 = v1 - v0, v2 - v0
    o, d = o.double(), d.double()
    p = torch.cross(d[:, None, :].expand(-1, e2.shape[0], -1), e2[None].expand(o.shape[0], -1, -1), dim=-1)
    det = (e1[None] * p).sum(-1)
    ok = det.abs() > 1e-14
    idet = 1.0 / torch.where(ok, det, torch.ones_like(det))
    s = o[:, None, :] - v0[None]
    u = (s * p).sum(-1) * idet
    q = torch.cross(s, e1[None].expand_as(s), dim=-1)
    v = (d[:, None, :] * q).sum(-1) * idet
    t = (e2[None] * q).sum(-1) * idet
    ok = ok & (u >= 0) & (u <= 1) & (v >= 0) & (u + v <= 1) & (t > 0)
    t = torch.where(ok, t, torch.full_like(t, float("inf")))
    tmin, arg = t.min(-1)
    return tmin, arg


def test_bvh_trace_matches_brute_force():
    from tensoflow_b200.mc_ops import RayTracer
    dev = _cuda()
    verts, tris = bumpy_sphere()
    rt = RayTracer(verts, tris)
    g = torch.Generator().manual_seed(0)
    n = 4000
    o = F.normalize(torch.randn(n, 3, generator=g), dim=-1) * 1.5
    tgt = torch.randn(n, 3, generator=g) * 0.35
    d = F.normalize(tgt - o, dim=-1)
    o[: n // 4] = F.normalize(torch.randn(n // 4, 3, generator=g), dim=-1) * 0.2     # rays starting inside
    pos, nrm, depth = rt.trace(o.to(dev), d.to(dev))
    tmin, arg = brute_force_trace(verts, tris, o, d)
    hit = torch.isfinite(tmin)
    got_hit = depth.cpu() < 10
    assert bool((hit == got_hit).all())
    assert float(hit.float().mean()) > 0.3 and float((~hit).float().mean()) > 0.05
    assert rel_err(depth.cpu()[hit], tmin[hit]) < 1e-4
    assert rel_err(pos.cpu()[hit], (o.double() + tmin[:, None] * d.double())[hit]) < 1e-4
    assert float((depth.cpu()[~hit] - 10.0).abs().max()) == 0.0
    v0, v1, v2 = (verts[tris[arg[hit]][:, k].long()].double() for k in range(3))
    fn = F.normalize(torch.cross(v1 - v0, v2 - v0, dim=-1), dim=-1)
    assert float((nrm.cpu()[hit].double() - fn).abs().max()) < 1e-4
    assert float(nrm.cpu()[~hit].abs().max()) == 0.0


def test_cube_light_forward_backward():
    from tensoflow_b200.mc_ops import CubeLightFunction
    dev = _cuda()
    g = torch.Generator().manual_seed(1)
    R = 16
    base = torch.randn(6, R, R, 3, generator=g) * 0.5
    d = F.normalize(torch.randn(6000, 3, generator=g), dim=-1)
    # directions within one texel of cube edges / corners exercise the seamless path
    e = F.normalize(torch.tensor([[1.0, 1.0, 0.3], [1.0, -1.0, 0.99], [0.98, 1.0, 1.0], [-1.0, 0.2, 1.0], [0.1, -1.0, -1.0]]), dim=-1)
    e = F.normalize(e[None] + 0.02 * torch.randn(200, 5, 3, generator=g), dim=-1).reshape(-1, 3)
    d = torch.cat([d, e], 0)
    mask = torch.rand(d.shape[0], generator=g) > 0.2
    u = torch.randn(d.shape[0], 3, generator=g)

    def ref(dt):
        b = base.detach().clone().to(dt).requires_grad_()
        out = torch.exp(OM.texture_cube(b, d.to(dt))) * mask[:, None].to(dt)
        (out * u.to(dt)).sum().backward()
        return out, b.grad

    o64, g64 = ref(torch.float64)
    o32, g32 = ref(torch.float32)
    b = base.detach().clone().to(dev).requires_grad_()
    out = CubeLightFunction.apply(b, d.to(dev), mask.to(dev))
    (out * u.to(dev)).sum().backward()
    assert rel_err(out, o64) < max(1e-5, 4 * rel_err(o32, o64))
    assert rel_err(b.grad, g64) < max(1e-4, 4 * rel_err(g32, g64))


def test_hit_encode_matches_posenc_and_ide():
    """tf_hit_encode, the inner-light MLP input of the occluded pairs, against fp64 posenc(p, 8) | IDE(reflect(v, n), kappa_inv = 0)
    of the oracle, and the zero padding up to ldx."""
    from tensoflow_b200 import mc_ops
    from tensoflow_b200.flow import posenc
    from tensoflow_b200.material import _ide_device_tables
    dev = _cuda()
    g = torch.Generator().manual_seed(2)
    K, M = 20000, 6000
    inters = torch.rand(K, 3, generator=g) * 2.4 - 1.2
    dirs = F.normalize(torch.randn(K, 3, generator=g), dim=-1)
    hit_normals = torch.randn(K, 3, generator=g) * (0.5 + torch.rand(K, 1, generator=g))     # the kernel normalises them
    idx = torch.randperm(K, generator=g)[:M]
    ide_mat, ide_m, _ = _ide_device_tables(dev)
    X = mc_ops.hit_encode(inters.to(dev), dirs.to(dev), hit_normals.to(dev), idx.to(dev), ide_mat, ide_m, 128)

    def ref(dt):
        p, v, n = inters[idx].to(dt), -dirs[idx].to(dt), F.normalize(hit_normals[idx].to(dt), dim=-1)
        r = 2.0 * (v * n).sum(-1, keepdim=True) * n - v
        return posenc(p, 8), MC.ide_encode(r, 0)

    pe64, ide64 = ref(torch.float64)
    _, ide32 = ref(torch.float32)
    assert rel_err(X[:, :51], pe64) < 1e-5
    # the degree-16 entries lose ~5e-3 to cancellation in any fp32 evaluation, the fp32 oracle's included
    assert rel_err(X[:, 51:123], ide64) < max(1e-5, 4 * rel_err(ide32, ide64))
    assert float(X[:, 123:].abs().max()) == 0.0


def _product_mc(g, dev):
    from tensoflow_b200.material import MCShadingNetwork
    cfg = dict(gridSize=[16, 16, 16], light_reso=16, mat_grid=24, device=dev)
    m = MCShadingNetwork(cfg, occluder_tracer(), torch.tensor([[-1., -1, -1], [1, 1, 1]]))
    res = m.load_state_dict(g["state"], strict=False)
    assert not res.missing_keys, res.missing_keys
    assert all(k.endswith(("scale", "offset")) or True for k in res.unexpected_keys)
    m.use_flow_diffuse_copy = m.use_flow_specular_copy = True
    for f in (m.flow_diffuse_copy, m.flow_specular_copy):
        for p in f.parameters():
            p.requires_grad = False
    return m


def test_mcshade_matches_reference_golden():
    dev = _cuda()
    g = load("mcshade.npz")
    m = _product_mc(g, dev)
    m64 = _oracle_mc(g, torch.float64)
    i = g["inputs"]
    noise = {k: i[k].to(dev) for k in ("az_diffuse", "phi_diffuse", "phi_specular")}
    m.train()
    rgb, out = m(i["pts"].to(dev), i["view_dirs"].to(dev), i["normals"].to(dev), None, 2000, True, noise=noise)
    n64 = {k: i[k].double() for k in ("az_diffuse", "phi_diffuse", "phi_specular")}
    rgb64, out64 = m64(i["pts"].double(), i["view_dirs"].double(), i["normals"].double(), n64, 2000)

    def close(got, key_ref, key64, tol, what):
        e, e_ref = rel_err(got, key64), rel_err(key_ref, key64)
        assert e <= max(tol, 4 * e_ref), f"{what}: rel err {e:.3e} (reference fp32 vs fp64 oracle {e_ref:.3e})"

    close(rgb, g["outputs"]["rgb"], rgb64, 1e-4, "rgb")
    for k in MC_KEYS:
        close(out[k], g["outputs"][k], out64[k], 1e-4, k)
    ((rgb * i["u_rgb"].to(dev)).sum() + 100.0 * out["loss_nis"]).backward()
    ((rgb64 * i["u_rgb"].double()).sum() + 100.0 * out64["loss_nis"]).backward()
    p64 = dict(m64.named_parameters())
    checked = 0
    for n, p in m.named_parameters():
        if not p.requires_grad or n not in g["grads"]:
            continue
        assert p.grad is not None, n
        assert p64[n].grad is not None, n
        close(p.grad, g["grads"][n], p64[n].grad, 1e-3, f"d {n}")
        checked += 1
    assert checked > 60


def test_mcshade_fixed_sets_and_bvh():
    """Before the flows are switched on (step < 1000) the cosine + GGX sets are used; run them
    with a real mesh through the BVH and compare with the oracle driven by the same tracer."""
    from tensoflow_b200.material import MCShadingNetwork, MeshTracer
    dev = _cuda()
    torch.manual_seed(3)
    verts, tris = bumpy_sphere(64, 32)
    aabb = torch.tensor([[-1., -1, -1], [1, 1, 1]])
    tracer = MeshTracer(verts, tris, offset=2 * 2.0 / 512)
    cfg = dict(gridSize=[16, 16, 16], light_reso=16, mat_grid=24, device=dev)
    m = MCShadingNetwork(cfg, tracer, aabb)
    with torch.no_grad():
        for p in m.mat_plane:
            p.mul_(3000)
        m.outer_light.base.add_(0.5 * torch.randn_like(m.outer_light.base))

    def cpu_tracer(o, d):
        r = tracer(o.to(dev).float(), d.to(dev).float())
        return tuple(t.cpu().to(o.dtype) if t.dtype.is_floating_point else t.cpu() for t in r)

    o64 = MC.MCShadingNetwork(cpu_tracer, aabb, gridSize=(24, 24, 24), flow_grid=(16, 16, 16), light_reso=16, dtype=torch.float64)
    o64.load_state_dict({k: v.detach().cpu().double() for k, v in m.state_dict().items()}, strict=False)
    o64.use_flow_diffuse_copy = o64.use_flow_specular_copy = False
    pn = 96
    idx = torch.randint(0, verts.shape[0], (pn,))
    pts = verts[idx] * 1.001
    normals = F.normalize(pts, dim=-1)
    view = F.normalize(F.normalize(torch.randn(pn, 3) + 2 * normals, dim=-1) * 2.0 - pts, dim=-1)
    noise = dict(az_diffuse=torch.rand(pn, 1, 1), az_specular=torch.rand(pn, 1, 1))
    rgb, out = m(pts.to(dev), view.to(dev), normals.to(dev), None, 100, True, noise={k: v.to(dev) for k, v in noise.items()})
    rgb64, out64 = o64(pts.double(), view.double(), normals.double(), {k: v.double() for k, v in noise.items()}, 100)
    # a handful of rays graze triangle edges where fp32 (kernel) and fp64 (oracle inputs) may disagree on hit/miss
    bad = ((rgb.detach().cpu().double() - rgb64).abs().max(-1).values > 1e-3).float().mean()
    assert float(bad) < 0.05
    ok = (rgb.detach().cpu().double() - rgb64).abs().max(-1).values <= 1e-3
    assert rel_err(rgb.detach().cpu()[ok], rgb64[ok]) < 1e-3
    assert float(out["visibility"].mean()) < 0.999        # some occlusion present


@pytest.mark.parametrize("version", ["direction", "sphere_direction"])
def test_mcshade_mlp_outer_lights(version):
    """`outer_light_version: direction / sphere_direction` (reference fields.py:716-721, 913-928; the oracle's restatement is pinned
    to the reference class in tests/test_oracle_flow_cpu.py): whole shading step against the fp64 oracle, outputs and gradients."""
    from tensoflow_b200.material import MCShadingNetwork
    dev = _cuda()
    g = load("mcshade.npz")                                   # materials / flows / inner light of the reference fixture ...
    torch.manual_seed(11)
    cfg = dict(gridSize=[16, 16, 16], light_reso=16, mat_grid=24, device=dev, outer_light_version=version)
    m = MCShadingNetwork(cfg, occluder_tracer(), torch.tensor([[-1., -1, -1], [1, 1, 1]]))
    state = {k: v for k, v in g["state"].items() if not k.startswith("outer_light")}
    m.load_state_dict(state, strict=False)                    # ... with a freshly initialised MLP light
    with torch.no_grad():
        for p in m.outer_light.parameters():
            p.add_(0.05 * torch.randn_like(p))
    m.use_flow_diffuse_copy = m.use_flow_specular_copy = True
    for f in (m.flow_diffuse_copy, m.flow_specular_copy):
        for p in f.parameters():
            p.requires_grad = False
    def oracle(dt):
        o = MC.MCShadingNetwork(occluder_tracer(), torch.tensor([[-1., -1, -1], [1, 1, 1]]), gridSize=(24, 24, 24), flow_grid=(16, 16, 16),
                                light_reso=16, dtype=dt, outer_light_version=version)
        res = o.load_state_dict({k: v.detach().cpu().to(dt) for k, v in m.state_dict().items()}, strict=False)
        assert not [k for k in res.missing_keys if 'outer_light' in k], res.missing_keys
        return o

    i = g["inputs"]
    keys = ("az_diffuse", "phi_diffuse", "phi_specular")
    runs = {}
    for dt in (torch.float64, torch.float32):                  # the fp32 oracle run calibrates what fp32 can reach (hit / miss flips)
        o = oracle(dt)
        rgb_o, out_o = o(i["pts"].to(dt), i["view_dirs"].to(dt), i["normals"].to(dt), {k: i[k].to(dt) for k in keys}, 2000)
        ((rgb_o * i["u_rgb"].to(dt)).sum() + 100.0 * out_o["loss_nis"]).backward()
        runs[dt] = (rgb_o, out_o, {n: p.grad for n, p in o.named_parameters() if p.grad is not None})
    rgb64, out64, g64 = runs[torch.float64]
    rgb32, out32, g32 = runs[torch.float32]

    def close(got, b32, b64, tol, what):
        e, e_ref = rel_err(got, b64), rel_err(b32, b64)
        assert e <= max(tol, 4 * e_ref), f"{what}: rel err {e:.3e} (fp32 oracle vs fp64 oracle {e_ref:.3e})"

    m.train()
    rgb, out = m(i["pts"].to(dev), i["view_dirs"].to(dev), i["normals"].to(dev), None, 2000, True, noise={k: i[k].to(dev) for k in keys})
    close(rgb, rgb32, rgb64, 1e-4, "rgb")
    for k in MC_KEYS:
        close(out[k], out32[k], out64[k], 1e-4, k)
    ((rgb * i["u_rgb"].to(dev)).sum() + 100.0 * out["loss_nis"]).backward()
    n_light = 0
    for n, p in m.named_parameters():
        if not p.requires_grad or p.grad is None or n not in g64:
            continue
        close(p.grad, g32[n], g64[n], 1e-3, f"d {n}")
        n_light += n.startswith("outer_light")
    assert n_light >= 8                                       # weight-norm g / v + bias of the four light layers
    groups = m.get_optparam_groups(0.02, 0.001, 0.1)
    assert groups[2]['lr'] == 0.001                           # MLP lights train at the network rate (reference fields.py:1584)
    m.update_step(999)                                        # no cubemap to upsample (the reference raises here)


def test_material_renderer_train_step_matches_oracle():
    """MaterialRenderer.forward -> train_step (reference network/materialRenderer.py:536-562, 757-762): host-resident surface-point
    pool -> H2D slice -> update_step -> shade (flows on: step 2000, BVH occlusion against a real mesh) -> rgb loss (charbonier),
    psnr, material regulariser (fields.py:1547-1578) and diffuse-light regulariser (materialRenderer.py:506-510); outputs,
    losses and every parameter gradient against the fp64 oracle driven by the same tracer, with the losses restated from the
    reference lines above."""
    from tensoflow_b200.material import MaterialRenderer
    dev = _cuda()
    torch.manual_seed(5)
    verts, tris = bumpy_sphere(64, 32)
    pn = 80
    cfg = dict(train_ray_num=pn, device=dev, gridSize=[16] * 3,
               shader_cfg=dict(gridSize=[16, 16, 16], light_reso=16, mat_grid=24))
    r = MaterialRenderer(cfg, verts, tris)
    sh = r.shader_network
    g = load("mcshade.npz")
    sh.load_state_dict(g["state"], strict=False)          # trained-looking materials / flows / inner light of the reference fixture
    with torch.no_grad():
        sh.outer_light.base.add_(0.5 * torch.randn_like(sh.outer_light.base))
    sh.use_flow_diffuse_copy = sh.use_flow_specular_copy = True
    for f in (sh.flow_diffuse_copy, sh.flow_specular_copy):
        for p in f.parameters():
            p.requires_grad = False
    gen = torch.Generator().manual_seed(6)
    idx = torch.randint(0, verts.shape[0], (pn,), generator=gen)
    pts = verts[idx] * 1.001
    normals = F.normalize(pts, dim=-1)
    cams = F.normalize(torch.randn(pn, 3, generator=gen) + 2 * normals, dim=-1) * 2.0
    rays_d = F.normalize(pts - cams, dim=-1)
    rgb_gt = torch.rand(pn, 3, generator=gen)
    noise = dict(az_diffuse=torch.rand(pn, 1, 1, generator=gen), az_specular=torch.rand(pn, 1, 1, generator=gen),
                 phi_diffuse=torch.rand(pn, 64, 1, generator=gen), phi_specular=torch.rand(pn, 32, 1, generator=gen))
    step = 2000

    def cpu_tracer(o, d):
        res = r.tracer(o.to(dev).float(), d.to(dev).float())
        return tuple(t.cpu().to(o.dtype) if t.dtype.is_floating_point else t.cpu() for t in res)

    def run_oracle(dt):
        o = MC.MCShadingNetwork(cpu_tracer, torch.tensor([[-1., -1, -1], [1, 1, 1]]), gridSize=(24, 24, 24), flow_grid=(16, 16, 16),
                                light_reso=16, dtype=dt)
        o.load_state_dict({k: v.detach().cpu().to(dt) for k, v in sh.state_dict().items()}, strict=False)
        rgb, out = o(pts.to(dt), (-rays_d).to(dt), normals.to(dt), {k: v.to(dt) for k, v in noise.items()}, step)
        loss_rgb = torch.sqrt(torch.sum((rgb_gt.to(dt) - rgb) ** 2, dim=-1) + 0.001)                      # materialRenderer.py:498-504
        tv = sum(OT.tv_loss(o.mat_plane[i]) + OT.tv_loss(o.mat_line[i]) for i in range(3))                # fields.py:1525-1530
        reg = tv * 0.1                                                                                     # fields.py:1568 (step >= 2000)
        dl = out["diffuse_light"]
        loss_dl = torch.sum(torch.abs(dl - torch.mean(dl, dim=-1, keepdim=True)), dim=-1) * 0.1           # materialRenderer.py:506-510
        total = loss_rgb.mean() + reg + loss_dl.mean() + out["loss_nis_diffuse"].mean() + out["loss_nis_specular"].mean()
        total.backward()
        return dict(rgb=rgb, loss_rgb=loss_rgb, reg=reg, loss_dl=loss_dl, total=total, out=out,
                    grads={n: p.grad for n, p in o.named_parameters() if p.grad is not None})

    from oracle import torch_oracle as OT
    o64, o32 = run_oracle(torch.float64), run_oracle(torch.float32)
    r.set_train_batch(dict(inters=pts, normals=normals, rays_d=rays_d, rgb=rgb_gt))
    r.train()
    out = r({"step": step, "noise": {k: v.to(dev) for k, v in noise.items()}})
    total = out["loss_rgb"].mean() + out["loss_mat_reg"] + out["loss_diffuse_light"].mean() + out["loss_nis_diffuse"].mean() \
        + out["loss_nis_specular"].mean()
    total.backward()

    def close(got, b32, b64, tol, what):
        e, e_ref = rel_err(got, b64), rel_err(b32, b64)
        assert e <= max(tol, 4 * e_ref), f"{what}: rel err {e:.3e} (fp32 oracle vs fp64 oracle {e_ref:.3e})"

    # a few occlusion rays graze triangle edges where the fp32 kernel and the fp64 oracle inputs may disagree on hit / miss:
    # per-point outputs are compared on the points whose colour agrees, and those must be nearly all
    ok = (out["rgb_pr"].detach().cpu().double() - o64["rgb"]).abs().max(-1).values <= 1e-3
    assert float(ok.float().mean()) > 0.95
    close(out["rgb_pr"].detach().cpu()[ok], o32["rgb"][ok], o64["rgb"][ok], 1e-4, "rgb_pr")
    close(out["loss_rgb"].detach().cpu()[ok], o32["loss_rgb"][ok], o64["loss_rgb"][ok], 1e-4, "loss_rgb")
    close(out["loss_diffuse_light"].detach().cpu()[ok], o32["loss_dl"][ok], o64["loss_dl"][ok], 1e-4, "loss_diffuse_light")
    close(out["loss_mat_reg"].reshape(()), o32["reg"], o64["reg"], 1e-4, "loss_mat_reg")
    assert torch.equal(out["rgb_gt"].cpu(), rgb_gt)
    mse = F.mse_loss(out["rgb_pr"].detach().cpu().double(), rgb_gt.double())
    assert abs(float(out["psnr"]) - float(20 * torch.log10(1.0 / torch.sqrt(mse)))) < 1e-3
    if bool(ok.all()):
        close(total, o32["total"], o64["total"], 1e-4, "total loss")
        checked = 0
        for n, p in sh.named_parameters():
            if p.requires_grad and p.grad is not None and n in o64["grads"]:
                close(p.grad, o32["grads"][n], o64["grads"][n], 1e-3, f"d {n}")
                checked += 1
        assert checked > 60


def test_bvh_trace_million_triangle_mesh():
    """BASELINE config 3's mesh size: the 1 M-triangle bumpy sphere of scripts/bench_material.py.  Closest hits of the BVH kernel
    against fp64 brute force over ALL triangles (Moeller-Trumbore on the device, in triangle chunks) for 1500 rays: hit / miss,
    depth, position, and the face normal of the reported triangle."""
    from tensoflow_b200.mc_ops import RayTracer
    from tensoflow_b200.synthetic import bumpy_sphere as big_sphere
    dev = _cuda()
    verts, tris = big_sphere(1000, 501)
    assert tris.shape[0] == 1_000_000
    rt = RayTracer(verts, tris)
    g = torch.Generator().manual_seed(3)
    n = 1500
    o = F.normalize(torch.randn(n, 3, generator=g), dim=-1) * 1.5
    d = F.normalize(torch.randn(n, 3, generator=g) * 0.3 - o, dim=-1)
    o[: n // 5] = F.normalize(torch.randn(n // 5, 3, generator=g), dim=-1) * 0.2            # rays starting inside the mesh
    pos, nrm, depth = rt.trace(o.to(dev), d.to(dev))
    # brute force in fp64 on the device, 50 k triangles at a time
    vd, td = verts.to(dev).double(), tris.to(dev).long()
    od, dd = o.to(dev).double(), d.to(dev).double()
    best = torch.full((n,), float("inf"), dtype=torch.float64, device=dev)
    for t0 in range(0, td.shape[0], 50_000):
        tt = td[t0:t0 + 50_000]
        v0, e1, e2 = vd[tt[:, 0]], vd[tt[:, 1]] - vd[tt[:, 0]], vd[tt[:, 2]] - vd[tt[:, 0]]
        p = torch.cross(dd[:, None, :].expand(-1, tt.shape[0], -1), e2[None].expand(n, -1, -1), dim=-1)
        det = (e1[None] * p).sum(-1)
        ok = det.abs() > 1e-14
        idet = 1.0 / torch.where(ok, det, torch.ones_like(det))
        s = od[:, None, :] - v0[None]
        u = (s * p).sum(-1) * idet
        q = torch.cross(s, e1[None].expand_as(s), dim=-1)
        v = (dd[:, None, :] * q).sum(-1) * idet
        t = (e2[None] * q).sum(-1) * idet
        ok = ok & (u >= 0) & (u <= 1) & (v >= 0) & (u + v <= 1) & (t > 0)
        best = torch.minimum(best, torch.where(ok, t, torch.full_like(t, float("inf"))).min(-1).values)
    hit = torch.isfinite(best)
    got_hit = depth < 10
    # a ray through a shared edge / vertex can be won or lost by an ulp of the fp32 barycentrics: allow a handful of flips
    assert int((hit != got_hit).sum()) <= 3, int((hit != got_hit).sum())
    both = hit & got_hit
    assert float(both.float().mean()) > 0.3
    assert rel_err(depth[both], best[both]) < 1e-4
    assert rel_err(pos[both], (od + best[:, None] * dd)[both]) < 1e-4
    assert float((depth[~got_hit] - 10.0).abs().max()) == 0.0


def test_material_stage_parity_at_bench_scale():
    """The configuration scripts/bench_material.py measures (BASELINE config 3: 512^2 x 36 material planes, 512^2 x 12 flow planes,
    128^2 environment cubemap, 512 cosine + 64 + 32 flow-sampled directions, NIS losses on) against a 125 k-triangle mesh, at a point
    count the fp64 oracle finishes in seconds: outputs, both NIS losses and every parameter gradient.  The oracle traces through the
    SAME BVH (wrapped), so hit / miss decisions can only differ by the fp32 / fp64 ray origins."""
    from tensoflow_b200.material import MaterialRenderer
    from tensoflow_b200.synthetic import bumpy_sphere as big_sphere
    dev = _cuda()
    torch.manual_seed(7)
    verts, tris = big_sphere(250, 251)
    assert tris.shape[0] >= 100_000
    pn = 192
    cfg = dict(train_ray_num=pn, device=dev, gridSize=[512] * 3,
               shader_cfg=dict(diffuse_sample_num=512, specular_sample_num=256, nis_diffuse_sample_num=64, nis_specular_sample_num=32,
                               light_reso=128, gridSize=[512] * 3, mat_grid=512))
    r = MaterialRenderer(cfg, verts, tris)
    sh = r.shader_network
    with torch.no_grad():
        for p in list(sh.mat_plane) + list(sh.flow_diffuse.parameters()) + list(sh.flow_specular.parameters()):
            if p.dim() == 4:
                p.add_(1e-2 * torch.randn_like(p))
        sh.outer_light.base.add_(0.5 * torch.randn_like(sh.outer_light.base))
    step = 2000
    sh.update_step(step)
    sh.use_flow_diffuse_copy = sh.use_flow_specular_copy = True
    gen = torch.Generator().manual_seed(8)
    idx = torch.randint(0, verts.shape[0], (pn,), generator=gen)
    pts = verts[idx] * 1.001
    normals = F.normalize(pts, dim=-1)
    cams = F.normalize(torch.randn(pn, 3, generator=gen) + 2 * normals, dim=-1) * 2.0
    view = -F.normalize(pts - cams, dim=-1)
    noise = dict(az_diffuse=torch.rand(pn, 1, 1, generator=gen), az_specular=torch.rand(pn, 1, 1, generator=gen),
                 phi_diffuse=torch.rand(pn, 64, 1, generator=gen), phi_specular=torch.rand(pn, 32, 1, generator=gen))
    u_rgb = torch.randn(pn, 3, generator=gen)

    def cpu_tracer(o, d):
        res = r.tracer(o.to(dev).float(), d.to(dev).float())
        return tuple(t.cpu().to(o.dtype) if t.dtype.is_floating_point else t.cpu() for t in res)

    def run_oracle(dt):
        o = MC.MCShadingNetwork(cpu_tracer, torch.tensor([[-1., -1, -1], [1, 1, 1]]), gridSize=(512, 512, 512), flow_grid=(512, 512, 512),
                                light_reso=128, dtype=dt)
        res = o.load_state_dict({k: v.detach().cpu().to(dt) for k, v in sh.state_dict().items()}, strict=False)
        assert not [k for k in res.missing_keys if not k.endswith("aabb") and "direction_samples" not in k], res.missing_keys
        rgb, out = o(pts.to(dt), view.to(dt), normals.to(dt), {k: v.to(dt) for k, v in noise.items()}, step)
        ((rgb * u_rgb.to(dt)).sum() + 100.0 * out["loss_nis"]).backward()
        return rgb, out, {n: p.grad for n, p in o.named_parameters() if p.grad is not None}

    rgb64, out64, g64 = run_oracle(torch.float64)
    rgb32, out32, g32 = run_oracle(torch.float32)
    sh.train()
    rgb, out = sh(pts.to(dev), view.to(dev), normals.to(dev), None, step, True, noise={k: v.to(dev) for k, v in noise.items()})
    ((rgb * u_rgb.to(dev)).sum() + 100.0 * out["loss_nis"]).backward()

    def close(got, b32, b64, tol, what):
        e, e_ref = rel_err(got, b64), rel_err(b32, b64)
        assert e <= max(tol, 4 * e_ref), f"{what}: rel err {e:.3e} (fp32 oracle vs fp64 oracle {e_ref:.3e})"

    ok = (rgb.detach().cpu().double() - rgb64).abs().max(-1).values <= 1e-3          # points whose occlusion rays agree on hit / miss
    assert float(ok.float().mean()) > 0.95, float(ok.float().mean())
    close(rgb.detach().cpu()[ok], rgb32[ok], rgb64[ok], 1e-4, "rgb")
    for k in ("albedo", "roughness", "metallic", "diffuse_light", "specular_light", "visibility"):
        close(out[k].detach().cpu()[ok], out32[k][ok], out64[k][ok], 1e-4, k)
    if bool(ok.all()):
        close(out["loss_nis_diffuse"], out32["loss_nis_diffuse"], out64["loss_nis_diffuse"], 1e-4, "loss_nis_diffuse")
        close(out["loss_nis_specular"], out32["loss_nis_specular"], out64["loss_nis_specular"], 1e-4, "loss_nis_specular")
        checked = 0
        for n_, p in sh.named_parameters():
            if p.requires_grad and p.grad is not None and n_ in g64:
                close(p.grad, g32[n_], g64[n_], 1e-3, f"d {n_}")
                checked += 1
        assert checked > 60
