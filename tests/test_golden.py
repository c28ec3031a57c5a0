"""Golden-vector tests.  tests/golden/*.npz were produced by oracle/gen_golden.py from the
REFERENCE's own classes (network/fields.py TensoSDF + MCShadingNetwork, network/flow.py
TensoFlow) in the build container.  CPU tests pin the oracle to them; GPU tests pin the CUDA
path (through the C ABI) to the same reference outputs.  Tolerances: outputs 1e-4 relative,
parameter gradients 1e-3 relative (BASELINE.json north star), rel err = max|a-b|/max|b|."""
import glob
import os

import numpy as np
import pytest
import torch

from conftest import rel_err
from oracle import torch_oracle as O, torch_oracle_mat as OM, torch_oracle_mc as MC

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def load(name):
    """name.npz, or its parts name.0.npz, name.1.npz, ... (oracle/gen_golden.py splits fixtures into files below 1 MB)."""
    stem = os.path.join(GOLD, name[:-4])
    out = {}
    for path in sorted(glob.glob(stem + ".[0-9].npz")) or [stem + ".npz"]:
        z = np.load(path)
        for k in z.files:
            g, key = k.split("/", 1)
            out.setdefault(g, {})[key] = torch.from_numpy(z[k])
    return out


def occluder_tracer():
    base = MC.analytic_sphere_tracer(0.45)

    def trace(o, d):
        c = torch.tensor([0.9, 0.0, 0.0], dtype=o.dtype, device=o.device)
        i, n, dep, h = base(o - c, d)
        return i + c, n, dep, h
    return trace


# ------------------------------------------------------------------ oracle vs reference (CPU)
def _oracle_sdf(g, dtype=torch.float32):
    f = O.TensoSDF([12] * 3, [[-1.0] * 3, [1.0] * 3], sdf_n_comp=8, sdf_dim=32, app_dim=16, init_n_levels=1, dtype=dtype)
    f.upsample_volume_grid(torch.tensor([24] * 3))
    f.upsample_volume_grid(torch.tensor([50] * 3))
    f.load_state_dict({k: v.to(dtype) for k, v in g["state"].items()}, strict=False)
    return f


def test_oracle_tensosdf_golden():
    g = load("tensosdf.npz")
    f = _oracle_sdf(g)
    assert torch.allclose(f.units, g["meta"]["units"])
    i = g["inputs"]
    out = f(i["xyz"], i["level"])
    grad, hess = f.gradient(i["xyz"], i["level"], training=True, sdf=out[:, :1])
    assert rel_err(out, g["outputs"]["out"]) < 1e-6
    assert rel_err(grad, g["outputs"]["grad"]) < 1e-5
    assert rel_err(hess, g["outputs"]["hess"]) < 1e-4
    ((out * i["u_out"]).sum() + (grad * i["u_grad"]).sum() + (hess * i["u_hess"]).sum()).backward()
    for n, p in f.named_parameters():
        assert rel_err(p.grad, g["grads"][n]) < 1e-5, n


def _oracle_flow(g, dtype=torch.float32):
    f = OM.TensoFlow(torch.tensor([[-1., -1, -1], [1, 1, 1]]), gridSize=(16, 16, 16), dtype=dtype)
    f.load_state_dict({k: v.to(dtype) for k, v in g["state"].items()}, strict=False)
    return f


def test_oracle_tensoflow_golden():
    g = load("tensoflow.npz")
    f = _oracle_flow(g)
    i = g["inputs"]
    ang, logj = f.sample(i["pts"], i["view_angles"], i["roughness"], 64, i["phi_shift"])
    assert rel_err(ang, g["outputs"]["angles"]) < 1e-6 and rel_err(logj, g["outputs"]["logj"]) < 1e-6
    z, logq = f(i["pts"], i["view_angles"], i["roughness"], i["x"])
    assert rel_err(z, g["outputs"]["z"]) < 1e-6 and rel_err(logq, g["outputs"]["logq"]) < 1e-6
    (logq * i["u"]).sum().backward()
    for n, p in f.named_parameters():
        if n in g["grads"]:
            assert rel_err(p.grad, g["grads"][n]) < 1e-5, n


def _oracle_mc(g, dtype=torch.float32):
    m = MC.MCShadingNetwork(occluder_tracer(), torch.tensor([[-1., -1, -1], [1, 1, 1]]), gridSize=(24, 24, 24),
                            flow_grid=(16, 16, 16), light_reso=16, dtype=dtype)
    res = m.load_state_dict({k: v.to(dtype) for k, v in g["state"].items()}, strict=False)
    assert not res.unexpected_keys, res.unexpected_keys
    return m


MC_KEYS = ['albedo', 'roughness', 'metallic', 'diffuse_light', 'specular_light', 'diffuse_color', 'specular_color', 'visibility',
           'indirect_light', 'loss_nis_diffuse', 'loss_nis_specular', 'loss_nis']


def test_oracle_mcshade_golden():
    g = load("mcshade.npz")
    m = _oracle_mc(g)
    i = g["inputs"]
    noise = {k: i[k] for k in ("az_diffuse", "phi_diffuse", "phi_specular")}
    rgb, out = m(i["pts"], i["view_dirs"], i["normals"], noise, 2000)
    assert rel_err(rgb, g["outputs"]["rgb"]) < 1e-5
    for k in MC_KEYS:
        assert rel_err(out[k], g["outputs"][k]) < 1e-5, k
    ((rgb * i["u_rgb"]).sum() + 100.0 * out["loss_nis"]).backward()
    params = dict(m.named_parameters())
    checked = 0
    for n, gref in g["grads"].items():
        if n in params and params[n].grad is not None:
            assert rel_err(params[n].grad, gref) < 1e-4, n
            checked += 1
    assert checked > 60


# ------------------------------------------------------------------ CUDA vs reference (GPU)
def _cuda():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    return torch.device("cuda:0")


@pytest.mark.gpu
def test_cuda_tensosdf_golden():
    from tensoflow_b200.fields import TensoSDF
    dev = _cuda()
    g = load("tensosdf.npz")
    f = TensoSDF(torch.tensor([12] * 3), torch.tensor([[-1.0] * 3, [1.0] * 3]), device=dev, sdf_n_comp=8, sdf_dim=32, app_dim=16,
                 init_n_levels=1, sdf_multires=0)
    f.upsample_volume_grid(torch.tensor([24] * 3))
    f.upsample_volume_grid(torch.tensor([50] * 3))
    f.load_state_dict(g["state"], strict=True)
    i = {k: v.to(dev) for k, v in g["inputs"].items()}
    sdf, feat, grad, hess = f.stencil(i["xyz"], i["level"])
    out = torch.cat([sdf[:, None], feat], -1)
    f64 = _oracle_sdf(g, torch.float64)
    with torch.no_grad():
        o64 = f64(g["inputs"]["xyz"].double(), g["inputs"]["level"].double())
        g64, h64 = f64.gradient(g["inputs"]["xyz"].double(), g["inputs"]["level"].double(), training=True, sdf=o64[:, :1])
    assert rel_err(out, g["outputs"]["out"]) < 1e-4
    # FD outputs: no worse than 4x the reference's own fp32 error against the fp64 oracle
    assert rel_err(grad, g64) < max(1e-4, 4 * rel_err(g["outputs"]["grad"], g64))
    assert rel_err(hess, h64) < max(1e-4, 4 * rel_err(g["outputs"]["hess"], h64))
    ((out * i["u_out"]).sum() + (grad * i["u_grad"]).sum() + (hess * i["u_hess"]).sum()).backward()
    (o := f64(g["inputs"]["xyz"].double(), g["inputs"]["level"].double()))
    gg, hh = f64.gradient(g["inputs"]["xyz"].double(), g["inputs"]["level"].double(), training=True, sdf=o[:, :1])
    ((o * g["inputs"]["u_out"].double()).sum() + (gg * g["inputs"]["u_grad"].double()).sum() + (hh * g["inputs"]["u_hess"].double()).sum()).backward()
    p64 = dict(f64.named_parameters())
    for n, p in f.named_parameters():
        assert rel_err(p.grad, p64[n].grad) < max(1e-3, 4 * rel_err(g["grads"][n], p64[n].grad)), n


@pytest.mark.gpu
def test_cuda_tensoflow_golden():
    from tensoflow_b200.flow import TensoFlow
    dev = _cuda()
    g = load("tensoflow.npz")
    f = TensoFlow(2, torch.tensor([[-1., -1, -1], [1, 1, 1]]), device=dev, gridSize=[16, 16, 16])
    f.load_state_dict(g["state"], strict=True)
    i = {k: v.to(dev) for k, v in g["inputs"].items()}
    ang, logj = f.sample(i["pts"], i["view_angles"], i["roughness"], 64, return_jacobian=True, phi_shift=i["phi_shift"])
    assert rel_err(ang, g["outputs"]["angles"]) < 1e-4 and rel_err(logj, g["outputs"]["logj"]) < 1e-4
    z, logq = f(i["pts"], i["view_angles"], i["roughness"], i["x"], return_jacobian=True)
    assert rel_err(z, g["outputs"]["z"]) < 1e-4 and rel_err(logq, g["outputs"]["logq"]) < 1e-4
    (logq * i["u"]).sum().backward()
    for n, p in f.named_parameters():
        if n in g["grads"]:
            assert rel_err(p.grad, g["grads"][n]) < 1e-3, n
