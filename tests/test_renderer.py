"""ShapeRenderer.render end to end (hierarchical NeuS sampler -> fused field stencil -> shader ->
NeuS alpha / compositing -> occlusion, sparse, hessian, TV losses) against the reference's own
ShapeRenderer.render output (tests/golden/renderer.npz, from oracle/gen_golden.py)."""
from types import SimpleNamespace

import pytest
import torch
import torch.nn.functional as F

from conftest import rel_err
from test_golden import load
from oracle import torch_oracle_renderer as RR

KEYS = ['ray_rgb', 'acc', 'normal', 'radiance', 'roughness_weights', 'gradient_error', 'loss_sparse', 'loss_hessian', 'std',
        'loss_tv_sdf', 'loss_occ']
CFG = dict(gridSize=[32, 32, 32], sdf_n_comp=8, sdf_dim=32, app_dim=128, max_levels=1, predict_BG=False, has_radiance_field=True,
           radiance_field_step=100, occ_loss_step=0, occ_loss_max_pn=100000, n_samples=16, n_importance=16, up_sample_steps=4,
           sdf_multires=0)


def total_loss(o):
    return (o['ray_rgb'].sum() + o['radiance'].sum() * 0.5 + o['gradient_error'].mean() * 0.1 + o['loss_sparse']
            + o['loss_hessian'] * 1e-3 + o['loss_tv_sdf'] + o['loss_occ'].sum())


def _oracle(g, dtype=torch.float32):
    m = RR.ShapeRenderer([32] * 3, sdf_n_comp=8, sdf_dim=32, app_dim=128, max_levels=1, has_radiance_field=True,
                         radiance_field_step=100, n_samples=16, n_importance=16, occ_loss_step=0, occ_loss_max_pn=100000,
                         env_res=16, env_min_res=4, dtype=dtype)
    res = m.load_state_dict({k: v.to(dtype) for k, v in g["state"].items()}, strict=False)
    assert not res.unexpected_keys, res.unexpected_keys
    return m


def _render_oracle(m, i, dt):
    m.color_network.envlight.build_mips()
    return m.render(i["rays_o"].to(dt), i["dirs"].to(dt), i["radiis"].to(dt), i["rays_cos"].to(dt), i["near"].to(dt), i["far"].to(dt),
                    0.7, 30000, t_rand=i["t_rand"].to(dt))


def test_oracle_renderer_golden():
    g = load("renderer.npz")
    m = _oracle(g)
    out = _render_oracle(m, g["inputs"], torch.float32)
    assert abs(out["sample_num"] - float(g["outputs"]["sample_num"])) < 1e-6
    for k in KEYS:
        assert rel_err(torch.as_tensor(out[k]), g["outputs"][k]) < 1e-5, k
    total_loss(out).backward()
    for n, p in m.named_parameters():
        if n in g["grads"] and p.grad is not None:
            assert rel_err(p.grad, g["grads"][n]) < 1e-4, n


def test_oracle_sample_ray_rounds():
    """sample_ray(rounds=...) records the depth / SDF lists after the coarse samples and after every round without changing
    what it returns.  A ray that misses the box keeps the descending coarse list of the reference until the first sort."""
    g = load("renderer.npz")
    i = g["inputs"]
    m = _oracle(g, torch.float64)
    o = torch.cat([i["rays_o"][:5], torch.tensor([[2.0, 1.2, 0.0]])]).double()          # last ray: misses the unit box
    d = torch.cat([i["dirs"][:5], F.normalize(torch.tensor([[-1.0, 0.1, 0.05]]), dim=-1)]).double()
    near, far = RR.near_far_from_sphere(o, d)
    args = (o, d, near, far, torch.full((6, 1), 1e-3, dtype=torch.float64), torch.ones(6, 1, dtype=torch.float64),
            torch.rand(6, 1, generator=torch.Generator().manual_seed(2), dtype=torch.float64))
    want = m.sample_ray(*args)
    rounds = []
    got = m.sample_ray(*args, rounds=rounds)
    assert all(torch.equal(a, b) for a, b in zip(got, want))
    steps, n = m.cfg['up_sample_steps'], m.cfg['n_samples']
    assert len(rounds) == steps + 1
    for r, (t, sdf) in enumerate(rounds):
        assert t.shape == (6, n + r * (m.cfg['n_importance'] // steps))
        assert (sdf is None) == (r == steps)
        if r > 0:
            assert bool((t[:, 1:] >= t[:, :-1]).all())
        if sdf is not None:
            pts = o[:, None, :] + d[:, None, :] * t[..., None]
            lvl = torch.log2(RR.O.compute_ball_radii(t[..., None], args[4][:, None, :], args[5][:, None, :]) / m.base_radii)
            assert torch.allclose(sdf, m.sdf_network.sdf(pts.reshape(-1, 3), lvl.reshape(-1, 1)).reshape(t.shape), atol=1e-12)
    t_coarse = rounds[0][0]
    assert bool((t_coarse[-1, 1:] < t_coarse[-1, :-1]).all()) and bool((t_coarse[:5, 1:] > t_coarse[:5, :-1]).all())
    ts, _, idx = got                                   # the packed starts come from the last list of their ray
    assert all(bool(torch.isin(ts[idx == r], rounds[-1][0][r]).all()) for r in range(6))


@pytest.mark.gpu
def test_cuda_renderer_golden():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    from tensoflow_b200.shape_renderer import ShapeRenderer
    dev = torch.device("cuda:0")
    g = load("renderer.npz")
    i = g["inputs"]
    m = ShapeRenderer(dict(device=dev, shader_config=dict(env_res=16, env_min_res=4), **CFG))
    res = m.load_state_dict(g["state"], strict=False)
    assert not res.unexpected_keys, res.unexpected_keys
    m64 = _oracle(g, torch.float64)
    o64 = _render_oracle(m64, i, torch.float64)
    batch = {k: i[k].to(dev) for k in ("rays_o", "rays_d", "dirs", "radiis", "rays_cos")}
    m.color_network.envlight.build_mips()
    out = m.render(batch, i["near"].to(dev), i["far"].to(dev), None, -1, 0.7, is_train=True, step=30000, t_rand=i["t_rand"].to(dev))
    assert abs(out["sample_num"] - float(g["outputs"]["sample_num"])) < 0.05   # a sample on the aabb face may flip

    def close(got, ref32, ref64, tol, what):
        e, e_ref = rel_err(got, ref64), rel_err(ref32, ref64)
        assert e <= max(tol, 4 * e_ref), f"{what}: rel err {e:.3e} (reference fp32 vs fp64 oracle {e_ref:.3e})"

    if abs(out["sample_num"] - float(g["outputs"]["sample_num"])) < 1e-6:
        for k in KEYS:
            close(torch.as_tensor(out[k]), g["outputs"][k], torch.as_tensor(o64[k]), 1e-4 if k != "loss_hessian" else 1e-3, k)
        total_loss(out).backward()
        total_loss(o64).backward()
        p64 = dict(m64.named_parameters())
        for n, p in m.named_parameters():
            if n in g["grads"] and p.grad is not None and n in p64:
                close(p.grad, g["grads"][n], p64[n].grad, 1e-3, f"d {n}")
    else:   # per-ray outputs still have to agree
        for k in ('ray_rgb', 'acc', 'radiance'):
            assert rel_err(out[k], g["outputs"][k]) < 1e-3, k


@pytest.mark.gpu
def test_alpha_mask_and_train_step():
    """updateAlphaMask + a train_step through set_train_batch (host-resident rays, H2D per step)."""
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    from tensoflow_b200.shape_renderer import ShapeRenderer
    from tensoflow_b200 import synthetic
    dev = torch.device("cuda:0")
    torch.manual_seed(0)
    m = ShapeRenderer(dict(device=dev, shader_config=dict(env_res=16, env_min_res=4), train_ray_num=64, **CFG))
    rays = synthetic.make_rays(256, seed=1)
    m.set_train_batch(dict(rays_o=rays["rays_o"], rays_d=rays["dirs"], dirs=rays["dirs"], radiis=rays["radiis"],
                           rays_cos=rays["rays_cos"], rgbs=rays["rgbs"]))
    out = m({'step': 30000})
    loss = out['loss_rgb'].mean() + 0.1 * out['gradient_error'].mean() + out['loss_tv_sdf']
    loss.backward()
    assert torch.isfinite(loss) and m.sdf_network.sdf_plane[0].grad is not None
    n_before = out['sample_num']
    new_aabb = m.updateAlphaMask((32, 32, 32))
    assert new_aabb.shape == (2, 3) and float(m.alphaMask.alpha_volume.mean()) < 1.0
    out2 = m({'step': 30001})
    assert out2['sample_num'] <= n_before + 1e-6       # the mask only removes samples
    assert torch.isfinite(out2['ray_rgb']).all()


@pytest.mark.gpu
def test_nvs_full_image_chunked():
    """ShapeRenderer.nvs (reference shapeRenderer.py:569-668): chunking must not change the image."""
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    import numpy as np
    from tensoflow_b200.shape_renderer import ShapeRenderer
    dev = torch.device("cuda:0")
    torch.manual_seed(0)
    h, w = 10, 12
    K = np.array([[20.0, 0, w / 2], [0, 20.0, h / 2], [0, 0, 1]], np.float32)
    pose = np.array([[1, 0, 0, 0.1], [0, 1, 0, -0.05], [0, 0, 1, 2.0]], np.float32)      # camera at z = 2 looking down -z
    imgs = []
    for trn in (4096, 37):
        torch.manual_seed(0)
        m = ShapeRenderer(dict(device=dev, shader_config=dict(env_res=16, env_min_res=4), test_ray_num=trn, **CFG))
        m.color_network.envlight.build_mips()
        imgs.append(m.nvs(pose, K, h, w, perturb_overwrite=0))
    for k in ('color', 'normal', 'acc', 'radiance'):
        assert imgs[0][k].shape[:2] == (h, w)
        assert np.isfinite(imgs[0][k]).all()
        assert np.abs(imgs[0][k] - imgs[1][k]).max() < 1e-4, k
    assert imgs[0]['acc'].max() > 0.5            # the initial sphere is visible


@pytest.mark.gpu
def test_alpha_mask_kernel_matches_grid_sample():
    """AlphaGridMask.sample_alpha (reference shapeRenderer.py:79-97) on tf_alpha_mask_sample against the reference's
    F.grid_sample formulation (oracle restatement, pinned to the reference class on CPU in test_host_logic_cpu.py):
    values and the `> 0` keep decisions, points outside the box included."""
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    from tensoflow_b200.shape_renderer import AlphaGridMask
    from oracle import torch_oracle_renderer as OR
    dev = torch.device("cuda:0")
    torch.manual_seed(3)
    aabb = torch.tensor([[-1.0, -0.8, -1.2], [1.0, 0.9, 1.1]])
    vol = (torch.rand(12, 10, 14) > 0.6).float()
    x = torch.rand(5000, 3) * 2.4 - 1.2
    x[:8] = torch.tensor([[-1.0, -0.8, -1.2], [1.0, 0.9, 1.1], [0.0, 0.0, 0.0], [1.0, -0.8, 1.1], [-1.0, 0.9, -1.2], [0.3, 0.9, 0.2],
                          [1.0000001, 0.0, 0.0], [-5.0, 0.0, 0.0]])
    want = OR.alpha_mask_sample(vol.double(), aabb.double(), x.double())
    got = AlphaGridMask(dev, aabb, vol.to(dev)).sample_alpha(x.to(dev)).cpu()
    assert float((got.double() - want).abs().max()) < 1e-5
    sure = (want > 1e-5) | (want == 0)                       # away from the fp32 noise floor the keep decision must agree
    assert torch.equal((got > 0)[sure], (want > 0)[sure])


@pytest.mark.gpu
@pytest.mark.parametrize("box,clip_var,perturb", [(1.0, True, True), (0.7, False, True), (1.0, True, False)])
def test_hierarchical_sampler_kernels_match_oracle(box, clip_var, perturb):
    """tensoflow_b200.sampler.hierarchical_sample (tf_sampler_* kernels) against the oracle's restatement of
    ShapeRenderer.sample_ray / upsample / cat_z_vals / sample_pdf (reference shapeRenderer.py:820-932,
    network_utils.py:117-147; pinned to the reference class in tests/test_oracle_cpu.py) driven by the SAME analytic,
    level-dependent SDF, in fp64: packed depths, interval ends, ray indices and CSR offsets."""
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    from tensoflow_b200 import sampler, synthetic
    dev = torch.device("cuda:0")
    R = 257
    rays = synthetic.make_rays(R, seed=5)
    o, d = rays["rays_o"], rays["dirs"]
    near, far = RR.near_far_from_sphere(o, d)
    g = torch.Generator().manual_seed(8)
    t_rand = torch.rand(R, 1, generator=g) if perturb else None

    def sdf_any(p, lvl):        # bumpy sphere whose level set moves a little with the mip level
        r = p.norm(dim=-1)
        return r - 0.45 - 0.05 * torch.sin(6 * p[..., 0]) * torch.cos(5 * p[..., 1]) + 0.003 * lvl.reshape(-1)

    ora = RR.ShapeRenderer([32] * 3, max_levels=1, clip_sample_variance=clip_var, dtype=torch.float64)
    ora.sdf_network.aabb.copy_(torch.tensor([[-box] * 3, [box] * 3], dtype=torch.float64))
    ora.sdf_network.sdf = lambda p, lvl=None: sdf_any(p, lvl)[:, None]
    with torch.no_grad():
        ora.deviation_network.variance.fill_(0.45)            # exp(4.5) = 90: between the caps 64 and 128 of rounds 0 / 1
    t0, t1, idx = ora.sample_ray(o.double(), d.double(), near.double(), far.double(), rays["radiis"].double(), rays["rays_cos"].double(),
                                 None if t_rand is None else t_rand.double())
    aabb = torch.tensor([[-box] * 3, [box] * 3], device=dev)
    base_radii = float(ora.base_radii)
    var = torch.tensor(0.45, device=dev)
    s0, s1, sidx, offs = sampler.hierarchical_sample(lambda p, lvl: sdf_any(p, lvl), aabb, base_radii, o.to(dev), d.to(dev), near.to(dev),
                                                     far.to(dev), rays["radiis"].to(dev), rays["rays_cos"].to(dev), 64, 64, 4,
                                                     1.0 if perturb else 0.0, None if t_rand is None else t_rand.to(dev), var, clip_var)
    cnt_o = torch.bincount(idx, minlength=R)
    cnt_k = torch.bincount(sidx.cpu(), minlength=R)
    assert torch.equal(offs.cpu().long(), torch.cat([torch.zeros(1, dtype=torch.long), torch.cumsum(cnt_k, 0)]))
    same = cnt_o == cnt_k                                     # a mid point within fp32 rounding of the box face may flip
    assert float(same.float().mean()) > 0.99, float(same.float().mean())
    if box == 1.0:                                            # unit sphere inside the box: only the mid point of a ray's LAST interval
        assert int(cnt_k.min()) >= 127                        # (which reaches past the sphere exit) can leave it
    ko = same[idx]
    kk = same[sidx.cpu()]
    assert float((s0.cpu().double()[kk] - t0[ko]).abs().max()) < 2e-5
    assert float((s1.cpu().double()[kk] - t1[ko]).abs().max()) < 2e-5
    # sorted depths per ray
    ds = s0[1:] - s0[:-1]
    assert bool((ds[sidx[1:] == sidx[:-1]] >= 0).all())


@pytest.mark.gpu
@pytest.mark.parametrize("mode", ["occlusion", "around_mesh"])
def test_probe_kernels_match_oracle(mode):
    """tf_probe_* (get_weights / get_intersection, reference utils/network_utils.py:149-202; get_intersection_around_mesh,
    network/materialRenderer.py:281-313) against the oracle restatements (pinned to the reference functions in
    tests/test_host_logic_cpu.py), same analytic SDF, fp64 arbiter: section mid points, weights, mid SDF."""
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    from tensoflow_b200 import sampler
    from tensoflow_b200.shape_renderer import get_intersection
    dev = torch.device("cuda:0")
    torch.manual_seed(4)
    pn = 301
    sdf_any = lambda p: p.norm(dim=-1) - 0.5 - 0.04 * torch.sin(7 * p[..., 0]) * torch.cos(6 * p[..., 2])
    var = torch.tensor(0.33)
    inv_s = float(torch.exp(var * 10.0))
    if mode == "occlusion":
        o = F.normalize(torch.randn(pn, 3), dim=-1) * (0.55 + 0.5 * torch.rand(pn, 1))        # some outside the unit sphere
        d = F.normalize(-o + 0.6 * torch.randn(pn, 3), dim=-1)
        want = RR.occlusion_probability(lambda x: sdf_any(x), inv_s, o.double(), d.double(), sn0=64, sn1=16)
        hz, hw, hs = get_intersection(lambda x: sdf_any(x)[:, None], var.to(dev), o.to(dev), d.to(dev), sn0=64, sn1=16)
        got = hw.sum(-1, keepdim=True).cpu().double()
        assert float((got - want).abs().max()) < 1e-4
        outside = o.norm(dim=-1) >= 0.999
        assert bool(outside.any()) and float(hw.cpu()[outside].abs().max()) == 0.0 and float(hs.cpu()[outside].max()) == -1.0
    else:
        o = F.normalize(torch.randn(pn, 3), dim=-1) * 2.0
        d = F.normalize(-o + 0.1 * torch.randn(pn, 3), dim=-1)
        m_depth = 1.5 + 0.02 * torch.randn(pn, 1)
        unit, radius = 2.0 / 127, 1.0
        field = SimpleNamespace(sdf=lambda x, lvl: sdf_any(x)[:, None], gradient=lambda x, lvl: (F.normalize(x, dim=-1), None))
        want, _, _ = RR.surface_refine(field, inv_s, o.double(), d.double(), m_depth.double(), unit, radius, 32, 9)
        near, far = RR.near_far_from_sphere(o, d, radius)
        t_min = torch.minimum(torch.maximum(m_depth - unit * 4, near), far)
        t_max = torch.minimum(torch.maximum(m_depth + unit * 4, near), far)
        z, w, _ = sampler.probe_sections(lambda x: sdf_any(x), var.to(dev), o.to(dev), d.to(dev), t_min.to(dev), t_max.to(dev), 32, 9)
        w = w / torch.sum(w, dim=-1, keepdim=True)
        w = torch.where(torch.isnan(w), torch.full_like(w, 1. / 8), w)
        got = torch.sum(w * z, -1, keepdim=True).cpu().double()
        assert float((got - want).abs().max()) < 2e-5
