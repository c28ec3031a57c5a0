"""Generate tests/golden/*.npz from the REFERENCE's own classes (imported from
/root/reference through oracle/ref_shim.py).  Run in the build container only:

    python -m oracle.gen_golden

Each fixture holds the reference module's state_dict, the seeded inputs (including every
random draw the reference makes) and the reference's outputs and parameter gradients, so the
GPU box -- where /root/reference does not exist -- can check both the oracle and the CUDA path
against reference outputs.  The un-vendored native ops underneath (nvdiffrast / nerfacc /
torch_scatter / raytracing) are the shim's restatements: that part stays "parity unpinned".
"""
from __future__ import annotations

import glob
import os
import sys
import zlib

import numpy as np
import torch
import torch.nn.functional as F

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLD = os.path.join(ROOT, "tests", "golden")


def _np(d):
    return {k: v.detach().cpu().numpy() for k, v in d.items()}


PART_BYTES = 900_000       # a fixture larger than this is written as <stem>.0.npz, <stem>.1.npz, ... (each file below 1 MB)


def _save(name, **groups):
    flat = {}
    for g, d in groups.items():
        for k, v in d.items():
            flat[f"{g}/{k}"] = v
    write_fixture(name, flat)


def write_fixture(name, flat):
    """Compressed arrays in one file, or in parts of at most ~PART_BYTES each (tests/test_golden.py load() joins them)."""
    os.makedirs(GOLD, exist_ok=True)
    stem = os.path.join(GOLD, name[:-4])
    for old in glob.glob(stem + ".npz") + glob.glob(stem + ".[0-9].npz"):
        os.remove(old)
    parts, size = [{}], 0
    for k, v in flat.items():
        n = len(zlib.compress(np.ascontiguousarray(v).tobytes()))
        if parts[-1] and size + n > PART_BYTES:
            parts.append({})
            size = 0
        parts[-1][k] = v
        size += n
    paths = [stem + ".npz"] if len(parts) == 1 else [f"{stem}.{i}.npz" for i in range(len(parts))]
    for path, part in zip(paths, parts):
        np.savez_compressed(path, **part)
        print(os.path.basename(path), f"{os.path.getsize(path) / 1e6:.2f} MB", len(part), "arrays")


def gen_tensosdf():
    import network.fields as RF
    torch.manual_seed(0)
    aabb = torch.tensor([[-1., -1, -1], [1, 1, 1]])
    ref = RF.TensoSDF(torch.tensor([12, 12, 12]), aabb, device='cpu', sdf_n_comp=8, sdf_dim=32, app_dim=16, init_n_levels=1,
                      sdf_multires=0)
    ref.upsample_volume_grid(torch.tensor([24, 24, 24]))
    ref.upsample_volume_grid(torch.tensor([50, 50, 50]))     # -> 48, 3 levels
    with torch.no_grad():
        for p in list(ref.sdf_plane) + list(ref.sdf_line):
            p.add_(0.05 * torch.randn_like(p))
        ref.sdf_mat[0].weight.mul_(0.3)
    n = 301
    xyz = torch.rand(n, 3) * 2.1 - 1.05
    level = torch.rand(n, 1) * 4 - 1
    out = ref(xyz, level)
    grad, hess = ref.gradient(xyz, level, training=True, sdf=out[:, :1])
    u = {"out": torch.randn_like(out), "grad": torch.randn_like(grad), "hess": torch.randn_like(hess) * 1e-2}
    ((out * u["out"]).sum() + (grad * u["grad"]).sum() + (hess * u["hess"]).sum()).backward()
    sd = {k: v for k, v in ref.state_dict().items() if "gaussian" not in k}
    _save("tensosdf.npz", state=_np(sd), inputs=_np({"xyz": xyz, "level": level, **{f"u_{k}": v for k, v in u.items()}}),
          outputs=_np({"out": out, "grad": grad, "hess": hess}),
          grads=_np({k: p.grad for k, p in ref.named_parameters() if p.grad is not None}),
          meta={"gridSize": np.array([48, 48, 48]), "n_levels": np.array(3), "units": ref.units.numpy()})


def gen_tensoflow():
    import network.flow as RFL
    torch.manual_seed(1)
    aabb = torch.tensor([[-1., -1, -1], [1, 1, 1]])
    ref = RFL.TensoFlow(d=2, aabb=aabb, device='cpu', gridSize=[16, 16, 16])
    with torch.no_grad():
        for p in ref.nis_plane:
            p.mul_(2000)
        for blk in ref.flows:
            blk.nn[7].weight.mul_(3.0)
    pn, sn = 40, 64
    pts, va, rough = torch.rand(pn, 3) * 1.9 - 0.95, torch.rand(pn, 2), torch.rand(pn, 1)
    shift = torch.rand(pn, sn, 1)
    ref.train()
    orig = torch.rand_like
    torch.rand_like = lambda x, *a, **k: shift
    try:
        ang, logj = ref.sample(pts, va, rough, sn, return_jacobian=True)
    finally:
        torch.rand_like = orig
    x = torch.rand(pn, sn, 2)
    u = torch.randn(pn, sn, 1)
    z, logq = ref(pts, va, rough, x, return_jacobian=True)
    (logq * u).sum().backward()
    _save("tensoflow.npz", state=_np(ref.state_dict()),
          inputs=_np({"pts": pts, "view_angles": va, "roughness": rough, "phi_shift": shift, "x": x, "u": u}),
          outputs=_np({"angles": ang, "logj": logj, "z": z, "logq": logq}),
          grads=_np({k: p.grad for k, p in ref.named_parameters() if p.grad is not None}))


def occluder_tracer():
    """Analytic stand-in for the BVH callback used by the MC fixture: a sphere of radius 0.45
    centred at (0.9,0,0) next to the shaded sphere (radius 0.5 at the origin)."""
    from oracle import torch_oracle_mc as MC
    base = MC.analytic_sphere_tracer(0.45)

    def trace(o, d):
        c = torch.tensor([0.9, 0.0, 0.0], dtype=o.dtype, device=o.device)
        i, n, dep, h = base(o - c, d)
        return i + c, n, dep, h
    return trace


def gen_mcshade():
    import network.fields as RF
    import torch.nn as nn
    torch.manual_seed(2)
    aabb = torch.tensor([[-1., -1, -1], [1, 1, 1]])
    cfg = dict(diffuse_sample_num=512, specular_sample_num=256, outer_light_version='envlight', light_exp_max=5.0,
               inner_light_exp_max=5.0, human_lights=False, gridSize=[16, 16, 16], light_reso=16)
    ref = RF.MCShadingNetwork(cfg, occluder_tracer(), aabb)
    # the reference hard-codes a 512^2 x 36 material grid (fields.py:676-684); shrink it for the fixture
    G = 24
    ref.mat_plane = nn.ParameterList([nn.Parameter(0.3 * (2 * torch.rand(1, 36, G, G) - 1)) for _ in range(3)])
    ref.mat_line = nn.ParameterList([nn.Parameter(torch.full((1, 36, G, 1), 1. / 108) + 0.01 * torch.randn(1, 36, G, 1)) for _ in range(3)])
    with torch.no_grad():
        ref.outer_light.base.add_(0.5 * torch.randn_like(ref.outer_light.base))
        for f in (ref.flow_diffuse, ref.flow_specular):
            for p in f.nis_plane:
                p.mul_(1000)
    ref.flow_diffuse_copy.load_state_dict(ref.flow_diffuse.state_dict())
    ref.flow_specular_copy.load_state_dict(ref.flow_specular.state_dict())
    for f in (ref.flow_diffuse_copy, ref.flow_specular_copy):
        for p in f.parameters():
            p.requires_grad = False
    ref.use_flow_diffuse_copy = ref.use_flow_specular_copy = True
    pn = 48
    pts = F.normalize(torch.randn(pn, 3), dim=-1) * 0.5
    normals = F.normalize(pts + 0.1 * torch.randn(pn, 3), dim=-1)
    cam = F.normalize(torch.randn(pn, 3) + 2 * pts, dim=-1) * 2.0
    view = F.normalize(cam - pts, dim=-1)
    noise = dict(az_diffuse=torch.rand(pn, 1, 1), phi_diffuse=torch.rand(pn, 64, 1), phi_specular=torch.rand(pn, 32, 1))
    ref.train()
    q_like = [noise['phi_diffuse'], noise['phi_specular']]
    orig_rl, orig_r = torch.rand_like, torch.rand
    torch.rand_like = lambda x, *a, **k: q_like.pop(0)
    torch.rand = lambda *a, **k: noise['az_diffuse']
    try:
        rgb, out = ref(pts, view, normals, None, 2000, True)
    finally:
        torch.rand_like, torch.rand = orig_rl, orig_r
    u = torch.randn_like(rgb)
    ((rgb * u).sum() + 100.0 * out['loss_nis']).backward()
    keep = ['albedo', 'roughness', 'metallic', 'diffuse_light', 'specular_light', 'diffuse_color', 'specular_color', 'visibility',
            'indirect_light', 'loss_nis_diffuse', 'loss_nis_specular', 'loss_nis']
    sd = {k: v for k, v in ref.state_dict().items()
          if not any(s in k for s in ('feats_network', 'mat_n_comp_mat', 'gaussian', 'light_pts'))}
    _save("mcshade.npz", state=_np(sd), inputs=_np({"pts": pts, "view_dirs": view, "normals": normals, "u_rgb": u, **noise}),
          outputs=_np({"rgb": rgb, **{k: out[k] for k in keep}}),
          grads=_np({k: p.grad for k, p in ref.named_parameters() if p.grad is not None and 'feats_network' not in k}))


def gen_shader():
    import network.fields as RF
    import network.light as RL
    torch.manual_seed(3)
    ref = RF.ShapeShadingNetwork(dict(has_radiance_field=True, radiance_field_step=0))
    ref.envlight = RL.EnvLight(trainable=True, max_res=16, min_res=4)     # the shader hard-codes 128 (fields.py:359)
    with torch.no_grad():
        ref.envlight.base.add_(0.5 * torch.randn_like(ref.envlight.base))
    n = 257
    pts = torch.rand(n, 3) * 1.6 - 0.8
    nrm = torch.randn(n, 3, requires_grad=True)
    view = torch.randn(n, 3)
    feat = torch.randn(n, 128, requires_grad=True)
    ref.envlight.build_mips()
    color, rad, occ = ref(pts, nrm, view, feat, None, step=10)
    u = torch.randn_like(color)
    ((color * u).sum() + rad.sum() + occ['occ_prob'].sum()).backward()
    sd = {k: v for k, v in ref.state_dict().items() if not k.startswith('outer_light') and k != 'FG_LUT'}
    grads = {k: p.grad for k, p in ref.named_parameters() if p.grad is not None and not k.startswith('outer_light')}
    grads['__normals'] = nrm.grad
    grads['__features'] = feat.grad
    _save("shader.npz", state=_np(sd), inputs=_np({"points": pts, "normals": nrm, "view_dirs": view, "features": feat, "u": u}),
          outputs=_np({"color": color, "radiance": rad, "occ_prob": occ['occ_prob'], "roughness": occ['roughness'],
                       "reflective": occ['reflective'], "diffuse": ref.envlight.diffuse,
                       **{f"specular{i}": s for i, s in enumerate(ref.envlight.specular)}}),
          grads=_np(grads))


RENDERER_CFG = dict(gridSize=[32, 32, 32], sdf_n_comp=8, sdf_dim=32, app_dim=128, max_levels=1, predict_BG=False,
                    has_radiance_field=True, radiance_field_step=100, occ_loss_step=0, occ_loss_max_pn=100000, n_samples=16,
                    n_importance=16, up_sample_steps=4, sdf_multires=0)


def renderer_total_loss(o):
    return (o['ray_rgb'].sum() + o['radiance'].sum() * 0.5 + o['gradient_error'].mean() * 0.1 + o['loss_sparse']
            + o['loss_hessian'] * 1e-3 + o['loss_tv_sdf'] + o['loss_occ'].sum())


def gen_renderer():
    """ShapeRenderer.render (hierarchical sampler + render_core + shader + losses), train mode."""
    import network.shapeRenderer as RS
    import network.light as RL
    from tensoflow_b200 import synthetic
    torch.manual_seed(4)
    ref = RS.ShapeRenderer(dict(device='cpu', **RENDERER_CFG), training=False)
    ref.color_network.envlight = RL.EnvLight(trainable=True, max_res=16, min_res=4)
    with torch.no_grad():
        ref.color_network.envlight.base.add_(0.5 * torch.randn_like(ref.color_network.envlight.base))
        for p in list(ref.sdf_network.sdf_plane) + list(ref.sdf_network.sdf_line):
            p.add_(0.01 * torch.randn_like(p))
    R = 48
    rays = synthetic.make_rays(R, seed=5)
    batch = dict(rays_o=rays['rays_o'], rays_d=rays['dirs'], dirs=rays['dirs'], radiis=rays['radiis'], rays_cos=rays['rays_cos'])
    near, far = ref.near_far_from_sphere(batch['rays_o'], batch['dirs'])
    t_rand = torch.rand(R, 1)
    orig = torch.rand
    torch.rand = lambda *a, **k: t_rand
    try:
        ref.color_network.envlight.build_mips()
        out = ref.render(batch, near, far, torch.zeros(R, 3, 4), -1, 0.7, is_train=True, step=30000)
    finally:
        torch.rand = orig
    renderer_total_loss(out).backward()
    keys = ['ray_rgb', 'acc', 'normal', 'radiance', 'roughness_weights', 'gradient_error', 'loss_sparse', 'loss_hessian', 'std',
            'loss_tv_sdf', 'loss_occ']
    sd = {k: v for k, v in ref.state_dict().items() if 'gaussian' not in k and 'outer_light' not in k and 'FG_LUT' not in k}
    _save("renderer.npz", state=_np(sd), inputs=_np({**batch, "near": near, "far": far, "t_rand": t_rand}),
          outputs=_np({**{k: torch.as_tensor(out[k]) for k in keys}, "sample_num": torch.tensor(out['sample_num'])}),
          grads=_np({k: p.grad for k, p in ref.named_parameters() if p.grad is not None and 'outer_light' not in k}))


def main():
    sys.path.insert(0, ROOT)
    from oracle import ref_shim
    ref_shim.install()
    which = sys.argv[1:] or ["tensosdf", "tensoflow", "mcshade", "shader", "renderer"]
    for name in which:
        globals()[f"gen_{name}"]()


if __name__ == "__main__":
    main()
