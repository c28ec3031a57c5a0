"""GPU parity tests of the shape-stage kernels (through the C ABI) against the oracle.

Tolerances follow BASELINE.json's north star: colour / SDF / alpha within 1e-4 relative,
parameter gradients within 1e-3 relative, where relative error = max|a-b| / max|b|
(conftest.rel_err).  The fp64 oracle is the arbiter; finite-difference outputs
(normals, hessian) are ill-conditioned in fp32 (division by units ~ 1/G), so for those the
bar is "no worse than a small multiple of the fp32 oracle's own error against fp64".
"""
import ctypes

import pytest
import torch
import torch.nn.functional as F

from conftest import rel_err, record_err

pytestmark = pytest.mark.gpu

from oracle import torch_oracle as O  # noqa: E402


def _cuda():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    return torch.device("cuda:0")


def close_as_fp32(got, o64, o32, tol, what, slack=4.0, fd=False):
    """|got - fp64 oracle| <= tol (relative, conftest.rel_err).  Only finite-difference outputs (`fd=True`: normals,
    hessian, and what is differentiated through them) may instead sit within `slack` x the fp32 oracle's own error:
    they divide fp32 SDF differences by units ~ 2/G, so the fp32 reference itself misses the bar there.
    The achieved errors are recorded (conftest.record_err -> gpurun_out/gpu_test_errors.json)."""
    e_ref = rel_err(o32, o64)
    e_got = record_err(what, got, o64, tol, fp32_oracle_rel_err=e_ref, fd=bool(fd))
    if fd:
        bar = max(tol, slack * e_ref)
    elif tol < 1e-4:          # bars tighter than the north star's 1e-4: may float with the fp32 oracle, never above 1e-4
        bar = min(1e-4, max(tol, slack * e_ref))
    else:
        bar = tol
    assert e_got <= bar, f"{what}: rel err {e_got:.3e} (fp32 oracle {e_ref:.3e}, tol {tol:.1e}, fd={fd})"
    return e_got


def make_fields(C, H, A, G0, ups, seed=0, noise=0.05):
    """Oracle fp32 / fp64 TensoSDF and the CUDA module with identical parameters."""
    from tensoflow_b200.fields import TensoSDF
    from tensoflow_b200 import synthetic
    dev = _cuda()
    torch.manual_seed(seed)
    aabb = [[-1.0, -1.0, -1.0], [1.0, 1.0, 1.0]]
    o32 = O.TensoSDF([G0] * 3, aabb, sdf_n_comp=C, sdf_dim=H, app_dim=A, init_n_levels=1)
    for r in ups:
        o32.upsample_volume_grid(torch.tensor([r] * 3))
    synthetic.perturb_field(o32, seed=seed + 1, noise=noise)
    with torch.no_grad():   # move the hidden pre-activations off the softplus linear branch
        o32.sdf_mat[0].weight.mul_(0.05)
        o32.sdf_mat[0].bias.add_(0.01 * torch.randn_like(o32.sdf_mat[0].bias))
        o32.sdf_mat[2].weight[1:].add_(0.1 * torch.randn_like(o32.sdf_mat[2].weight[1:]))
    o64 = O.TensoSDF([G0] * 3, aabb, sdf_n_comp=C, sdf_dim=H, app_dim=A, init_n_levels=1, dtype=torch.float64)
    for r in ups:
        o64.upsample_volume_grid(torch.tensor([r] * 3))
    synthetic.copy_field_params(o32, o64)
    cu = TensoSDF(torch.tensor([G0] * 3), torch.tensor(aabb), device=dev, sdf_n_comp=C, sdf_dim=H, app_dim=A,
                  init_n_levels=1, sdf_multires=0)
    for r in ups:
        cu.upsample_volume_grid(torch.tensor([r] * 3))
    synthetic.copy_field_params(o32, cu)
    assert cu.n_levels == o32.n_levels and list(cu.gridSize) == list(o32.gridSize)
    return o32, o64, cu


def points(n, seed, with_level, n_levels):
    g = torch.Generator().manual_seed(seed)
    x = torch.rand(n, 3, generator=g) * 2.1 - 1.05          # a few points outside the aabb (clamp)
    lv = (torch.rand(n, 1, generator=g) * (n_levels + 1.5) - 1.0) if with_level else None
    return x, lv


CONFIGS = [
    # C,  H,   A,  G0, ups,        N
    (8, 32, 16, 16, [32, 64], 1003),      # small, 3 mip levels, ragged tile
    (16, 128, 128, 128, [], 4099),         # BASELINE config 1 dims (128^3, 48 comps), L=1
    (36, 256, 128, 16, [32, 64], 2050),    # BASELINE config 2 dims on a small grid, L=3
]
# hidden > 256 is outside the tensor-core stencil: the FFMA kernels run it, and TensoSDF.forward without autograd falls back from
# the single-query kernel to the stencil
FFMA_CONFIG = (8, 288, 16, 16, [32], 1000)


@pytest.mark.parametrize("C,H,A,G0,ups,N", CONFIGS)
@pytest.mark.parametrize("with_level", [True, False])
def test_vm_feature(C, H, A, G0, ups, N, with_level):
    from tensoflow_b200 import ops
    o32, o64, cu = make_fields(C, H, A, G0, ups)
    dev = _cuda()
    x, lv = points(N, 3, with_level, o32.n_levels)
    f64 = O.vm_feature(o64.sdf_plane, o64.sdf_line, x.double(), None if lv is None else lv.double(), o64.aabb, o64.n_levels)
    f32 = O.vm_feature(o32.sdf_plane, o32.sdf_line, x, lv, o32.aabb, o32.n_levels)
    got = ops.VMFeatureFunction.apply(x.to(dev), None if lv is None else lv.to(dev), cu.aabb, cu.n_levels,
                                      *cu.sdf_plane, *cu.sdf_line)
    close_as_fp32(got, f64, f32, 1e-5, "vm feature")
    gup = torch.randn(N, 3 * C, generator=torch.Generator().manual_seed(5))
    (f64 * gup.double()).sum().backward()
    (got * gup.to(dev)).sum().backward()
    for name in ("sdf_plane", "sdf_line"):
        for i in range(3):
            e = rel_err(getattr(cu, name)[i].grad, getattr(o64, name)[i].grad)
            assert e < 1e-4, f"{name}[{i}] grad rel err {e:.3e}"


@pytest.mark.parametrize("C,H,A,G0,ups,N", CONFIGS + [FFMA_CONFIG])
@pytest.mark.parametrize("with_level", [True, False])
def test_stencil_forward(C, H, A, G0, ups, N, with_level):
    o32, o64, cu = make_fields(C, H, A, G0, ups)
    dev = _cuda()
    x, lv = points(N, 7, with_level, o32.n_levels)
    with torch.no_grad():
        r64 = o64(x.double(), None if lv is None else lv.double())
        g64, h64 = o64.gradient(x.double(), None if lv is None else lv.double(), training=True, sdf=r64[:, :1])
        r32 = o32(x, lv)
        g32, h32 = o32.gradient(x, lv, training=True, sdf=r32[:, :1])
        sdf, feat, grad, hess = cu.stencil(x.to(dev), None if lv is None else lv.to(dev))
        only = cu.sdf(x.to(dev), None if lv is None else lv.to(dev))
        full = cu(x.to(dev), None if lv is None else lv.to(dev))
    close_as_fp32(sdf, r64[:, 0], r32[:, 0], 1e-5, "sdf")
    close_as_fp32(only[:, 0], r64[:, 0], r32[:, 0], 1e-5, "sdf (sdf-only kernel)")
    close_as_fp32(feat, r64[:, 1:], r32[:, 1:], 1e-5, "appearance features")
    close_as_fp32(full, r64, r32, 1e-5, "TensoSDF.forward")
    close_as_fp32(grad, g64, g32, 1e-4, "FD gradient", fd=True)
    close_as_fp32(hess, h64, h32, 1e-4, "normal hessian", fd=True)


@pytest.mark.parametrize("C,H,A,G0,ups,N", CONFIGS + [FFMA_CONFIG])
@pytest.mark.parametrize("with_level", [True, False])
def test_stencil_backward(C, H, A, G0, ups, N, with_level, monkeypatch):
    from tensoflow_b200 import ops
    o32, o64, cu = make_fields(C, H, A, G0, ups)
    dev = _cuda()
    if N > 2000:   # force the sliced-workspace path
        monkeypatch.setattr(ops, "BWD_WORKSPACE_BYTES", 48 << 20)
    x, lv = points(N, 11, with_level, o32.n_levels)
    g = torch.Generator().manual_seed(13)
    u_sdf, u_feat = torch.randn(N, generator=g), torch.randn(N, A, generator=g)
    u_grad, u_hess = torch.randn(N, 3, generator=g), torch.randn(N, generator=g) * 1e-2

    def oracle_loss(f, dt):
        r = f(x.to(dt), None if lv is None else lv.to(dt))
        gr, he = f.gradient(x.to(dt), None if lv is None else lv.to(dt), training=True, sdf=r[:, :1])
        return (r[:, 0] * u_sdf.to(dt)).sum() + (r[:, 1:] * u_feat.to(dt)).sum() + (gr * u_grad.to(dt)).sum() + (he * u_hess.to(dt)).sum()

    oracle_loss(o64, torch.float64).backward()
    oracle_loss(o32, torch.float32).backward()
    sdf, feat, grad, hess = cu.stencil(x.to(dev), None if lv is None else lv.to(dev))
    ((sdf * u_sdf.to(dev)).sum() + (feat * u_feat.to(dev)).sum() + (grad * u_grad.to(dev)).sum() + (hess * u_hess.to(dev)).sum()).backward()
    for (name, p64), (_, p32), (_, pc) in zip(o64.named_parameters(), o32.named_parameters(), cu.named_parameters()):
        assert pc.grad is not None, name
        close_as_fp32(pc.grad, p64.grad, p32.grad, 1e-3, f"d {name}", fd=True)    # upstream gradients enter through the FD taps


@pytest.mark.parametrize("N", [1, 5, 18, 19, 37, 2665])
def test_stencil_tiny_and_ragged_batches(N):
    """Edge sizes of the persistent tensor-core kernels: fewer samples than one 18-sample tile, exactly one tile, one sample into the
    second tile, fewer tiles than CTAs, and one tile more than the 148 CTAs (2665 = 148 * 18 + 1): forward values and all parameter
    gradients against the fp64 oracle."""
    C_, H, A, G0, ups, _ = CONFIGS[2]
    o32, o64, cu = make_fields(C_, H, A, G0, ups)
    dev = _cuda()
    x, lv = points(N, 23, True, o32.n_levels)
    g = torch.Generator().manual_seed(29)
    u_sdf, u_feat = torch.randn(N, generator=g), torch.randn(N, A, generator=g)
    u_grad = torch.randn(N, 3, generator=g)

    def oracle_loss(f, dt):
        r = f(x.to(dt), lv.to(dt))
        gr, he = f.gradient(x.to(dt), lv.to(dt), training=True, sdf=r[:, :1])
        return r, gr, (r[:, 0] * u_sdf.to(dt)).sum() + (r[:, 1:] * u_feat.to(dt)).sum() + (gr * u_grad.to(dt)).sum()

    r64, g64, l64 = oracle_loss(o64, torch.float64)
    l64.backward()
    r32, g32, l32 = oracle_loss(o32, torch.float32)
    l32.backward()
    sdf, feat, grad, hess = cu.stencil(x.to(dev), lv.to(dev))
    ((sdf * u_sdf.to(dev)).sum() + (feat * u_feat.to(dev)).sum() + (grad * u_grad.to(dev)).sum()).backward()
    # (max-normalised errors over a handful of samples: the denominator is the largest value of a few rows, not of thousands,
    # so the value bars are 3e-5 here instead of the 1e-5 of the large-batch tests)
    close_as_fp32(sdf, r64[:, 0].detach(), r32[:, 0].detach(), 3e-5, f"sdf (N={N})")
    close_as_fp32(feat, r64[:, 1:].detach(), r32[:, 1:].detach(), 3e-5, f"features (N={N})")
    close_as_fp32(grad, g64.detach(), g32.detach(), 1e-4, f"FD gradient (N={N})", fd=True)
    with torch.no_grad():
        only = cu.sdf(x.to(dev), lv.to(dev))
        full = cu(x.to(dev), lv.to(dev))
    close_as_fp32(only[:, 0], r64[:, 0].detach(), r32[:, 0].detach(), 3e-5, f"sdf-only kernel (N={N})")
    close_as_fp32(full, r64.detach(), r32.detach(), 3e-5, f"single-query forward with features (N={N})")
    for (name, p64), (_, p32), (_, pc) in zip(o64.named_parameters(), o32.named_parameters(), cu.named_parameters()):
        assert pc.grad is not None, name
        close_as_fp32(pc.grad, p64.grad, p32.grad, 1e-3, f"d {name} (N={N})", fd=True)


def _composite_inputs(n_rays, max_s, seed, D=7):
    g = torch.Generator().manual_seed(seed)
    counts = torch.randint(0, max_s + 1, (n_rays,), generator=g)
    counts[0] = 0
    counts[-1] = max_s
    idx = torch.repeat_interleave(torch.arange(n_rays), counts)
    n = int(counts.sum())
    sdf = torch.randn(n, generator=g) * 0.05
    grad = F.normalize(torch.randn(n, 3, generator=g), dim=-1) * (1 + 0.1 * torch.randn(n, 1, generator=g))
    dists = torch.rand(n, generator=g) * 0.02 + 0.002
    dirs = F.normalize(torch.randn(n_rays, 3, generator=g), dim=-1)
    vals = torch.rand(n, D, generator=g)
    return idx, sdf, grad, dists, dirs, vals


@pytest.mark.parametrize("cos_anneal,max_s,D", [(0.0, 100, 7), (0.4, 100, 7), (1.0, 100, 7), (0.7, 700, 6), (0.7, 300, 13), (1.0, 40, 1)])
def test_neus_composite(cos_anneal, max_s, D):
    """ragged rays (0 .. max_s samples: one to several 128- / 64-sample iterations of the kernels' chunk loop), D <= 8 and
    D > 8 accumulated channels (the two template instances)"""
    from tensoflow_b200 import ops
    from tensoflow_b200.shape_renderer import ray_offsets_from_indices
    dev = _cuda()
    n_rays = 333
    idx, sdf, grad, dists, dirs, vals = _composite_inputs(n_rays, max_s, 21, D)
    if max_s > 200:
        sdf = sdf + 0.15                     # long rays: keep the transmittance alive beyond the first chunks
    g = torch.Generator().manual_seed(22)
    u_acc, u_out = torch.randn(n_rays, generator=g), torch.randn(n_rays, D, generator=g)
    u_w = torch.randn(sdf.shape[0], generator=g) * 0.1

    def run_oracle(dt):
        s, gr, va = (t.detach().clone().to(dt).requires_grad_() for t in (sdf, grad, vals))
        var = torch.tensor(0.3, dtype=dt, requires_grad=True)
        alpha, _ = O.neus_alpha(s, gr, dists.to(dt), dirs.to(dt)[idx], var, cos_anneal)
        w, _ = O.render_weight_from_alpha(alpha, idx, n_rays)
        acc = O.accumulate_along_rays(w, None, idx, n_rays)[:, 0]
        out = O.accumulate_along_rays(w, va, idx, n_rays)
        ((acc * u_acc.to(dt)).sum() + (out * u_out.to(dt)).sum() + (w * u_w.to(dt)).sum()).backward()
        return alpha, w, acc, out, s.grad, gr.grad, va.grad, var.grad

    r64, r32 = run_oracle(torch.float64), run_oracle(torch.float32)
    s, gr, va = (t.detach().clone().to(dev).requires_grad_() for t in (sdf, grad, vals))
    var = torch.tensor(0.3, device=dev, requires_grad=True)
    offs = ray_offsets_from_indices(idx.to(dev), n_rays)
    alpha, w, acc, out = ops.NeusCompositeFunction.apply(s, gr, dists.to(dev), dirs.to(dev), offs, var, cos_anneal, va, True)
    ((acc * u_acc.to(dev)).sum() + (out * u_out.to(dev)).sum() + (w * u_w.to(dev)).sum()).backward()
    got = (alpha, w, acc, out, s.grad, gr.grad, va.grad, var.grad)
    names = ("alpha", "weights", "acc", "out", "d sdf", "d grad", "d vals", "d variance")
    tols = (1e-4, 1e-4, 1e-4, 1e-4, 1e-3, 1e-3, 1e-3, 1e-3)
    for a, b64, b32, nm, tol in zip(got, r64, r32, names, tols):
        close_as_fp32(a, b64, b32, tol, nm)


def test_neus_composite_empty():
    from tensoflow_b200 import ops
    dev = _cuda()
    z = torch.zeros(0, device=dev)
    offs = torch.zeros(5, dtype=torch.int32, device=dev)
    alpha, w, acc, out = ops.NeusCompositeFunction.apply(z, torch.zeros(0, 3, device=dev), z, torch.ones(4, 3, device=dev), offs,
                                                         torch.tensor(0.3, device=dev), 1.0, torch.zeros(0, 6, device=dev), True)
    assert acc.shape == (4,) and float(acc.abs().sum()) == 0.0 and float(out.abs().sum()) == 0.0


@pytest.mark.parametrize("C,H,A,G0,ups,R,S", [(16, 128, 128, 128, [], 256, 64), (36, 256, 128, 32, [64, 128], 128, 48)])
def test_render_core_end_to_end(C, H, A, G0, ups, R, S):
    """field -> alpha -> composite -> charbonnier + 0.1 eikonal, fwd + bwd, vs the oracle."""
    from tensoflow_b200 import synthetic
    from tensoflow_b200.shape_renderer import render_core, charbonnier
    o32, o64, cu = make_fields(C, H, A, G0, ups, noise=0.01)
    dev = _cuda()
    rays = synthetic.make_rays(R, seed=0)
    t0, t1, idx = synthetic.uniform_samples(rays["rays_o"], rays["dirs"], o32.aabb, S)

    def run_oracle(f, dt):
        var = torch.tensor(0.3, dtype=dt, requires_grad=True)
        r = O.shape_render_core(f, var, rays["rays_o"].to(dt), rays["dirs"].to(dt), rays["radiis"].to(dt), rays["rays_cos"].to(dt),
                                t0.to(dt), t1.to(dt), idx, synthetic.simple_color_fn, cos_anneal_ratio=0.7)
        loss = O.charbonnier(r["ray_rgb"], rays["rgbs"].to(dt)).mean() + 0.1 * r["gradient_error"].mean() \
            + 0.01 * r["loss_sparse"] + 1e-4 * r["loss_hessian"]
        loss.backward()
        return r, loss, var

    r64, l64, v64 = run_oracle(o64, torch.float64)
    r32, l32, v32 = run_oracle(o32, torch.float32)
    var = torch.tensor(0.3, device=dev, requires_grad=True)
    rc = render_core(cu, var, synthetic.simple_color_fn, rays["rays_o"].to(dev), rays["dirs"].to(dev), rays["radiis"].to(dev),
                     rays["rays_cos"].to(dev), t0.to(dev), t1.to(dev), idx.to(dev), cos_anneal_ratio=0.7)
    loss = charbonnier(rc["ray_rgb"], rays["rgbs"].to(dev)).mean() + 0.1 * rc["gradient_error"].mean() \
        + 0.01 * rc["loss_sparse"] + 1e-4 * rc["loss_hessian"]
    loss.backward()
    close_as_fp32(rc["sdf"], r64["sdf"], r32["sdf"], 1e-4, "sdf")
    for k in ("ray_rgb", "acc", "alpha", "weights"):          # alpha takes the FD normal (cos of the NeuS section)
        close_as_fp32(rc[k], r64[k], r32[k], 1e-4, k, fd=True)
    close_as_fp32(rc["normal"], r64["normal"], r32["normal"], 1e-4, "normal", fd=True)
    close_as_fp32(loss, l64, l32, 1e-4, "loss", fd=True)
    close_as_fp32(var.grad, v64.grad, v32.grad, 1e-3, "d variance", fd=True)
    for (name, p64), (_, p32), (_, pc) in zip(o64.named_parameters(), o32.named_parameters(), cu.named_parameters()):
        close_as_fp32(pc.grad, p64.grad, p32.grad, 1e-3, f"d {name}", fd=True)


def test_bench_configuration_parity(monkeypatch):
    """The configuration bench.py measures (BASELINE.json configs[1]: G = 512, C = 36, H = 256, A = 128, 3 mip levels,
    512 samples per ray, bench.build_shape / bench.shape_step themselves) at a ray count the oracle finishes in seconds:
    288 rays x 512 samples = 147 k samples = 8192 stencil tiles = 55 tiles per persistent CTA (the mbarrier phase
    arithmetic, the W ring and the TMEM double buffers wrap many times), with the stencil-backward workspace forced
    into 2 slices.  Oracle (fp64 arbiter, fp32 for the finite-difference slack) runs on the GPU device in PyTorch."""
    import bench
    from tensoflow_b200 import ops, synthetic
    from tensoflow_b200.shape_renderer import render_core, charbonnier
    dev = _cuda()
    cfg = dict(bench.SHAPE_CFG)
    R = 288
    field, variance = bench.build_shape(cfg, dev)
    assert int(field.gridSize[0]) == 512 and field.n_levels == 3 and field.sdf_n_comp == 36
    rays = synthetic.make_rays(R, seed=0, device=dev)
    t0, t1, idx = synthetic.uniform_samples(rays["rays_o"], rays["dirs"], field.aabb, cfg["samples"])
    n = int(idx.shape[0])
    assert n >= 50 * 148 * 18, n
    monkeypatch.setattr(ops, "BWD_WORKSPACE_BYTES", 1 << 30)       # 8192 tiles x 202 KB = 1.7 GB -> 2 slices
    vm = ops.vm_desc(field.sdf_plane, field.sdf_line, field.aabb, field.n_levels, False)
    m, _ = ops._mlp_desc(field.sdf_mat[0].weight, field.sdf_mat[0].bias, field.sdf_mat[2].weight, field.sdf_mat[2].bias)
    ws_bytes = lambda tiles: ops._lib.load().tf_sdf_stencil_bwd_workspace(ctypes.byref(vm.c), ctypes.byref(m), 18 * tiles)
    per_tile = ws_bytes(2) - ws_bytes(1)
    tiles_fit = ((1 << 30) - (ws_bytes(1) - per_tile)) // per_tile
    n_tiles = -(-n // 18)                                            # 18 samples per stencil tile
    assert -(-n_tiles // tiles_fit) == 2, (n_tiles, tiles_fit)

    def oracle(dt):
        o = O.TensoSDF([128] * 3, [[-1.0] * 3, [1.0] * 3], sdf_n_comp=cfg["C"], sdf_dim=cfg["H"], app_dim=cfg["A"], init_n_levels=1, dtype=dt)
        for r in (256, 512):
            o.upsample_volume_grid(torch.tensor([r] * 3))
        synthetic.copy_field_params(field, o)
        o = o.to(dev)
        o.update_gridSize(o.gridSize, o.n_levels)                    # units follow the aabb buffer onto the device
        var = torch.tensor(0.3, dtype=dt, device=dev, requires_grad=True)
        r = O.shape_render_core(o, var, rays["rays_o"].to(dt), rays["dirs"].to(dt), rays["radiis"].to(dt), rays["rays_cos"].to(dt),
                                t0.to(dt), t1.to(dt), idx, synthetic.simple_color_fn, cos_anneal_ratio=1.0)
        loss = O.charbonnier(r["ray_rgb"], rays["rgbs"].to(dt)).mean() + 0.1 * r["gradient_error"].mean()
        loss.backward()
        keep = {k: r[k].detach() for k in ("ray_rgb", "acc", "sdf", "alpha", "weights", "normal", "levels")}
        return keep, loss.detach(), var.grad, {n_: p.grad for n_, p in o.named_parameters()}

    r64, l64, v64, g64 = oracle(torch.float64)
    r32, l32, v32, g32 = oracle(torch.float32)
    lv = r64["levels"]
    assert float((lv > 0).float().mean()) > 0.3 and float(lv.max()) > 1.0      # the mip chain is really exercised
    for p in field.parameters():
        p.grad = None
    rc = render_core(field, variance, synthetic.simple_color_fn, rays["rays_o"], rays["dirs"], rays["radiis"], rays["rays_cos"],
                     t0, t1, idx, cos_anneal_ratio=1.0)
    loss = charbonnier(rc["ray_rgb"], rays["rgbs"]).mean() + 0.1 * rc["gradient_error"].mean()
    loss.backward()
    close_as_fp32(rc["sdf"], r64["sdf"], r32["sdf"], 1e-4, "sdf")
    for k in ("ray_rgb", "acc", "alpha", "weights", "normal"):
        close_as_fp32(rc[k], r64[k], r32[k], 1e-4, k, fd=True)
    close_as_fp32(loss, l64, l32, 1e-4, "loss", fd=True)
    close_as_fp32(variance.grad, v64, v32, 1e-3, "d variance", fd=True)
    for name, pc in field.named_parameters():
        close_as_fp32(pc.grad, g64[name], g32[name], 1e-3, f"d {name}", fd=True)


@pytest.mark.parametrize("shape", [(1, 8, 33, 47), (1, 36, 64, 1), (1, 16, 5, 5)])
def test_tv_loss_fused_matches_reference_formula(shape):
    """TVLoss (reference other_field.py:170-191) through the fused channels-last kernels: value and gradient."""
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    from tensoflow_b200.fields import TVLoss, _cl
    dev = torch.device("cuda:0")
    torch.manual_seed(sum(shape))
    x0 = torch.randn(*shape)
    tv = TVLoss(1.7)
    xc = torch.nn.Parameter(_cl(x0.to(dev)))
    loss = tv(xc) * 0.3
    loss.backward()
    xr = x0.double().requires_grad_()
    ref = O.tv_loss(xr, 1.7) * 0.3   # the reference formulation (oracle/torch_oracle.py)
    ref.backward()
    assert abs(float(loss.detach()) - float(ref.detach())) <= 1e-5 * abs(float(ref.detach()))
    assert rel_err(xc.grad.cpu(), xr.grad) < 1e-5


@pytest.mark.parametrize("shape,ks,sigma", [((1, 8, 33, 47), 5, 0.5), ((1, 36, 64, 1), 5, 0.5), ((1, 16, 12, 9), 3, 0.8), ((1, 4, 4, 4), 5, 0.5)])
def test_gaussian_residual_loss(shape, ks, sigma):
    """one term of grid_gaussian_loss (reference network/fields.py:301-309; GaussianBlur2D / 1D network/other_field.py:121-168,
    F.conv2d / F.conv1d with zero padding, interior only) through tf_gauss_residual_*: value and gradient against the
    reference formulation in fp64.  (1,4,4,4) with a 5x5 kernel has an empty interior: loss 0, gradient 0."""
    from tensoflow_b200 import ops
    from tensoflow_b200.fields import _cl
    dev = _cuda()
    torch.manual_seed(sum(shape) + ks)
    x0 = torch.randn(*shape)
    line = shape[3] == 1
    k1, k2 = ops.gaussian_taps(ks, sigma)
    xc = torch.nn.Parameter(_cl(x0.to(dev)))
    loss = ops.GaussResidualFunction.apply(xc, k1 if line else k2, ks, 1 if line else ks) * 0.7
    loss.backward()
    xr = x0.double().requires_grad_()
    k = ks // 2
    xs = torch.arange(-ks // 2 + 1.0, ks // 2 + 1.0, dtype=torch.float64)
    if line:
        kern = torch.exp(-xs ** 2 / (2 * sigma ** 2))
        kern = (kern / kern.sum())[None, None]
        blur = F.conv1d(xr.permute(1, 0, 2, 3).squeeze(-1), kern, stride=1, padding=k).unsqueeze(-1).permute(1, 0, 2, 3)
        ref = torch.sum((xr[..., k:-k, :] - blur[..., k:-k, :]).square()) * 0.7
    else:
        xx, yy = torch.meshgrid(xs, xs, indexing="ij")
        kern = torch.exp(-(xx ** 2 + yy ** 2) / (2 * sigma ** 2))
        kern = (kern / kern.sum())[None, None]
        blur = F.conv2d(xr.permute(1, 0, 2, 3), kern, stride=1, padding=k).permute(1, 0, 2, 3)
        ref = torch.sum((xr[..., k:-k, k:-k] - blur[..., k:-k, k:-k]).square()) * 0.7
    ref.backward()
    assert abs(float(loss.detach()) - float(ref.detach())) <= 1e-5 * max(abs(float(ref.detach())), 1e-6)
    if float(ref.detach()) > 0:
        assert rel_err(xc.grad.cpu(), xr.grad) < 1e-5
    else:
        assert float(xc.grad.abs().max()) == 0.0
