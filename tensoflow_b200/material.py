"""Material stage (reference network/fields.py:618-1595 MCShadingNetwork, network/light.py
EnvLight, network/materialRenderer.py) on the sm_100a kernels.

In-scope branches (SURVEY.md 8a): shade_mixed, use_nis_diffuse + use_nis_specular with the
half-vector parametrisation, outer_light_version='envlight' | 'direction' | 'sphere_direction',
geometry_type='schlick', no human lights.  Parameter names follow the reference so its checkpoints load
(`mat_plane.*`, `mat_line.*`, `*_predictor.*`, `outer_light.base`, `inner_light.*`,
`flow_{diffuse,specular}[_copy].*`); the reference's dead weights (`feats_network`,
`mat_n_comp_mat`) are not instantiated.
"""
from __future__ import annotations

import math
from typing import Callable, Dict, Optional

import numpy as np
import torch
import torch.nn as nn
import torch.nn.functional as F

from . import ops, mc_ops
from .fields import _cl, MAT_MODE, VEC_MODE, TVLoss
from .flow import TensoFlow, posenc

EPS = 1e-6   # reference network/fields.py:18


def linear_to_srgb(linear):
    """reference utils/raw_utils.py:4-10"""
    eps = torch.finfo(torch.float32).eps
    srgb0 = 323 / 25 * linear
    srgb1 = (211 * torch.clamp(linear, min=eps) ** (5 / 12) - 11) / 200
    return torch.where(linear <= 0.0031308, srgb0, srgb1)


def saturate_dot(a, b):
    return torch.clamp(torch.sum(a * b, dim=-1, keepdim=True), min=0.0, max=1.0)


def sample_sphere(num_samples, begin_elevation=0):
    """reference utils/base_utils.py:869-882"""
    ratio = (begin_elevation + 90) / 180
    num_points = int(num_samples // (1 - ratio))
    phi = (np.sqrt(5) - 1.0) / 2.
    az, el = [], []
    for n in range(num_points - num_samples, num_points):
        z = 2. * n / num_points - 1.
        az.append(2 * np.pi * n * phi % (2 * np.pi))
        el.append(np.arcsin(z))
    return np.array(az), np.array(el)


# ---- integrated directional encoding (reference utils/ref_utils.py:8-117) ----
def _ide_tables(deg_view=5):
    ml = []
    for i in range(deg_view):
        l = 2 ** i
        for m in range(l + 1):
            ml.append((m, l))
    ml = np.array(ml).T
    l_max = 2 ** (deg_view - 1)

    def gbc(a, k):
        return np.prod(a - np.arange(k)) / math.factorial(k)

    mat = np.zeros((l_max + 1, ml.shape[1]))
    for i, (m, l) in enumerate(ml.T):
        for k in range(l - m + 1):
            alc = ((-1) ** m * 2 ** l * math.factorial(l) / math.factorial(k) / math.factorial(l - k - m)
                   * gbc(0.5 * (l + k + m - 1.0), l))
            mat[k, i] = np.sqrt((2.0 * l + 1.0) * math.factorial(l - m) / (4.0 * np.pi * math.factorial(l + m))) * alc
    return ml, mat.astype(np.float32)


_IDE_DEV = {}


def _ide_device_tables(device):
    """The degree-5 IDE tables on `device`: polynomial table mat [17,36] fp32, the order m of its 36 entries (int32) and
    sigma = l (l + 1) / 2 [36] fp32.  tf_hit_encode takes (mat, m), tf_shader_encode_* all three."""
    key = str(device)
    if key not in _IDE_DEV:
        ml, mat = _ide_tables(5)
        _IDE_DEV[key] = (torch.from_numpy(np.ascontiguousarray(mat, dtype=np.float32)).to(device).contiguous(),
                         torch.from_numpy(ml[0].astype(np.int32)).to(device).contiguous(),
                         torch.from_numpy((0.5 * ml[1] * (ml[1] + 1)).astype(np.float32)).to(device).contiguous())
    return _IDE_DEV[key]


def ide_encode(xyz: torch.Tensor, kappa_inv: Optional[torch.Tensor] = None) -> torch.Tensor:
    """generate_ide_fn(5)(xyz, kappa_inv) -> [N,72] with real arithmetic: (x+iy)^m by recurrence.  kappa_inv [N,1] attenuates
    entry (m, l) by exp(-l (l + 1) / 2 kappa_inv); None is kappa_inv = 0 and skips the multiply."""
    mat, m_idx, sigma = _ide_device_tables(xyz.device)
    x, y, z = xyz[:, 0:1], xyz[:, 1:2], xyz[:, 2:3]
    n_pow = mat.shape[0]
    zs = [torch.ones_like(z)]
    re, im = [torch.ones_like(x)], [torch.zeros_like(x)]
    for _ in range(1, n_pow):
        zs.append(zs[-1] * z)
        re_n = re[-1] * x - im[-1] * y
        im_n = re[-1] * y + im[-1] * x
        re.append(re_n)
        im.append(im_n)
    vmz = torch.cat(zs, -1)
    re, im = torch.cat(re, -1).index_select(1, m_idx), torch.cat(im, -1).index_select(1, m_idx)   # backward = index_add, not a sorted index_put
    att = vmz @ mat
    if kappa_inv is not None:
        att = att * torch.exp(-sigma * kappa_inv)
    return torch.cat([re * att, im * att], -1)


def make_predictor(n_layers, feats_dim, output_dim, run_dim=None):
    """weight-norm Linear stacks of reference network/other_field.py:20-121 (activations are
    applied by the fused linear kernels)."""
    run_dim = run_dim or (256 if n_layers == 4 else 128)
    wn = nn.utils.parametrizations.weight_norm
    layers, last = [], feats_dim
    for _ in range(n_layers - 1):
        layers += [wn(nn.Linear(last, run_dim)), nn.ReLU()]
        last = run_dim
    layers += [wn(nn.Linear(last, output_dim)), nn.Identity()]
    return nn.Sequential(*layers)


def run_predictor_padded(seq: nn.Sequential, x_padded, k_valid: int, final_act: str, act_param: float = 0.0):
    """run_predictor for an input whose rows are already zero-padded from k_valid to x_padded.shape[1] columns: the first
    layer's weight is padded alike (zero columns), so no copy of the activations is made."""
    n = len(seq) // 2
    x = x_padded
    for i in range(n):
        lin = seq[2 * i]
        w = lin.weight
        if i == 0 and x.shape[1] != k_valid:
            w = F.pad(w, (0, x.shape[1] - k_valid))
        x = ops.linear(x, w, lin.bias, "relu" if i < n - 1 else final_act, act_param)
    return x


def run_predictor(seq: nn.Sequential, x, final_act: str, act_param: float = 0.0):
    n = len(seq) // 2
    for i in range(n):
        lin = seq[2 * i]
        x = ops.linear(x, lin.weight, lin.bias, "relu" if i < n - 1 else final_act, act_param)
    return x


class EnvLight(nn.Module):
    """reference network/light.py:8-31: trainable log-radiance cubemap; `direct_light`
    (light.py:125-162) is the lookup the MC shader uses."""

    def __init__(self, path=None, device='cuda', scale=1.0, min_res=16, start_res=16, max_res=512, min_roughness=0.08,
                 max_roughness=0.5, trainable=False):
        super().__init__()
        self.max_res, self.min_res = max_res, min_res
        self.base = nn.Parameter(torch.full((6, max_res, max_res, 3), math.log(0.5), dtype=torch.float32, device=device),
                                 requires_grad=trainable)
        self.level = max(0, int(np.log2(max_res / start_res)) + 0.5)

    def upsample(self):
        if self.level > 0:
            self.level = max(self.level - 1, 0)

    def build_mips_direct(self, cutoff=0.99):
        """reference light.py:66-70 (average-pool chain; unused by direct_light)."""
        self.base_mip = [self.base]
        while self.base_mip[-1].shape[1] > self.min_res:
            self.base_mip.append(F.avg_pool2d(self.base_mip[-1].permute(0, 3, 1, 2), (2, 2)).permute(0, 2, 3, 1).contiguous())

    def direct_light(self, l, roughness=None, mask=None):
        return mc_ops.CubeLightFunction.apply(self.base, l, mask)


def get_orthogonal_directions(d):
    """reference fields.py:812-822"""
    x, y, z = torch.split(d, 1, dim=-1)
    o0 = torch.cat([y, -x, torch.zeros_like(x)], -1)
    o1 = torch.cat([-z, torch.zeros_like(x), x], -1)
    mask0 = (torch.norm(o0, dim=-1) > torch.norm(o1, dim=-1))[:, None]
    return F.normalize(torch.where(mask0, o0, o1), dim=-1)


def direction_to_angle(normals, directions):
    """reference fields.py:1035-1048"""
    z = normals
    x = get_orthogonal_directions(normals)
    y = torch.cross(z, x, dim=-1)
    cx = torch.sum(x.unsqueeze(1) * directions, -1, keepdim=True)
    cy = torch.sum(y.unsqueeze(1) * directions, -1, keepdim=True)
    cz = torch.sum(z.unsqueeze(1) * directions, -1, keepdim=True).clamp(-1 + EPS, 1 - EPS)
    phi = (torch.atan2(cy, cx) + 2 * np.pi) % (2 * np.pi)
    return torch.cat([phi, torch.acos(cz)], dim=-1)


class MCShadingNetwork(nn.Module):
    default_cfg = {
        'diffuse_sample_num': 512, 'specular_sample_num': 256, 'human_lights': False, 'light_exp_max': 5.0,
        'inner_light_exp_max': 5.0, 'outer_light_version': 'envlight', 'geometry_type': 'schlick', 'random_azimuth': True,
        'shade_fn': 'shade_mixed', 'use_nis_diffuse': True, 'use_nis_specular': True, 'gridSize': [512, 512, 512],
        'nis_diffuse_sample_num': 64, 'nis_specular_sample_num': 32, 'nis_start_iter_diffuse': 1000,
        'nis_start_iter_specular': 1000, 'nis_loss_iter_diffuse': 500, 'nis_loss_iter_specular': 500,
        'nis_update_interval_diffuse': 1000, 'nis_update_interval_specular': 1000, 'flow_diffuse': 'pwquad',
        'flow_specular': 'pwquad', 'use_half_diffuse': True, 'use_half_specular': True, 'light_upsample_interval': 1000,
        'light_reso': 128, 'reg_min_max': True, 'mat_grid': 512, 'device': 'cuda',
    }

    def __init__(self, cfg, ray_trace_fun: Callable, aabb):
        super().__init__()
        self.cfg = {**self.default_cfg, **cfg}
        c = self.cfg
        if c['outer_light_version'] not in ('envlight', 'direction', 'sphere_direction') or c['human_lights'] \
                or c['shade_fn'] != 'shade_mixed' or c['geometry_type'] != 'schlick' \
                or not (c['use_half_diffuse'] and c['use_half_specular']):
            raise NotImplementedError("tensoflow_b200 implements the shipped material configurations "
                                      "(envlight / direction / sphere_direction outer light, shade_mixed, half-vector flows, "
                                      "schlick geometry, no human lights)")
        dev = c['device']
        self.aabb = torch.as_tensor(aabb, dtype=torch.float32).to(dev)
        self.use_nis = True
        self.mat_n_comp, self.n_levels, self.nplane = 36, 3, 3
        G = int(c['mat_grid'])      # the reference hard-codes 512 (fields.py:676-684)
        self.gridSize = torch.tensor([G, G, G])
        planes, lines = [], []
        for i in range(3):          # reference fields.py:765-774
            planes.append(nn.Parameter(_cl((1e-4 * (2 * torch.rand(1, self.mat_n_comp, G, G) - 1)).to(dev))))
            lines.append(nn.Parameter(_cl(torch.full((1, self.mat_n_comp, G, 1), 1. / (self.mat_n_comp * 3), device=dev))))
        self.mat_plane, self.mat_line = nn.ParameterList(planes), nn.ParameterList(lines)
        self.mat_feature_dim = self.mat_n_comp * self.n_levels
        self.tv_reg = TVLoss()
        self.metallic_predictor = make_predictor(2, self.mat_feature_dim, 1).to(dev)
        self.roughness_predictor = make_predictor(2, self.mat_feature_dim, 1).to(dev)
        self.albedo_predictor = make_predictor(2, self.mat_feature_dim, 3).to(dev)
        if c['outer_light_version'] == 'envlight':              # reference fields.py:716-723
            self.outer_light = EnvLight(trainable=True, max_res=c['light_reso'], device=dev)
        else:                                                    # 4-layer MLP on the IDE of the direction (+ of the sphere exit point)
            self.outer_light = make_predictor(4, 72 if c['outer_light_version'] == 'direction' else 144, 3).to(dev)
            nn.init.constant_(self.outer_light[-2].bias, np.log(0.5))
        self.inner_light = make_predictor(4, 51 + 72, 3).to(dev)
        nn.init.constant_(self.inner_light[-2].bias, np.log(0.5))
        for name, n in (('diffuse_direction_samples', c['diffuse_sample_num']), ('specular_direction_samples', c['specular_sample_num'])):
            az, el = sample_sphere(n, 0)            # reference fields.py:734-742
            az, el = az * 0.5 / np.pi, 1 - 2 * el / np.pi
            setattr(self, name, torch.from_numpy(np.stack([az, el], -1).astype(np.float32)).to(dev))
        self.ray_trace_fun = ray_trace_fun
        self.use_flow_diffuse_copy = False
        self.use_flow_specular_copy = False
        mk = lambda: TensoFlow(d=2, aabb=self.aabb, gridSize=c['gridSize'], device=dev, flow='pwquad')
        self.flow_diffuse, self.flow_diffuse_copy = mk(), mk()
        self.flow_specular, self.flow_specular_copy = mk(), mk()

    # ---- bookkeeping --------------------------------------------------------------------
    def get_optparam_groups(self, lr_init_spatialxyz=0.02, lr_init_network=0.001, lr_init_env=0.1):
        g = [{'params': self.mat_line, 'lr': lr_init_spatialxyz}, {'params': self.mat_plane, 'lr': lr_init_spatialxyz},
             {'params': self.outer_light.parameters(), 'lr': lr_init_env if self.cfg['outer_light_version'] == 'envlight' else lr_init_network},
             {'params': list(self.albedo_predictor.parameters()) + list(self.metallic_predictor.parameters())
              + list(self.roughness_predictor.parameters()) + list(self.inner_light.parameters()), 'lr': lr_init_network}]
        g += self.flow_diffuse.get_optparam_groups(lr_init_spatialxyz, lr_init_network)
        g += self.flow_specular.get_optparam_groups(lr_init_spatialxyz, lr_init_network)
        return g

    def update_step(self, step):
        """reference fields.py:1050-1068: periodic refresh of the frozen sampling copies."""
        c = self.cfg
        for kind in ('diffuse', 'specular'):
            if (step + 1) >= c[f'nis_start_iter_{kind}'] and (step + 1 - c[f'nis_start_iter_{kind}']) % c[f'nis_update_interval_{kind}'] == 0:
                setattr(self, f'use_flow_{kind}_copy', True)
                copy = getattr(self, f'flow_{kind}_copy')
                copy.load_state_dict(getattr(self, f'flow_{kind}').state_dict())
                for p in copy.parameters():
                    p.requires_grad = False
        if (step + 1) % c['light_upsample_interval'] == 0 and c['outer_light_version'] == 'envlight':
            # (the reference calls .upsample() on the MLP lights too and raises there: fields.py:1067-1068)
            self.outer_light.upsample()

    # ---- materials (reference fields.py:776-810, 1010-1017) ------------------------------------
    def tenso_feature(self, xyz_sampled, level_vol=None):
        return ops.VMFeatureFunction.apply(xyz_sampled, level_vol, self.aabb, self.n_levels, *self.mat_plane, *self.mat_line)

    def predict_materials(self, pts):
        feats = self.tenso_feature(pts)
        metallic = run_predictor(self.metallic_predictor, feats, "sigmoid")
        roughness = run_predictor(self.roughness_predictor, feats, "sigmoid") * (1.0 - 0.04 ** 2) + 0.04 ** 2
        albedo = run_predictor(self.albedo_predictor, feats, "sigmoid")
        return metallic, roughness, albedo

    def TV_loss(self):
        total = 0
        for i in range(3):
            total = total + self.tv_reg(self.mat_plane[i]) + self.tv_reg(self.mat_line[i])
        return total

    def material_regularization(self, pts, normals, metallic, roughness, albedo, step):
        """reference fields.py:1547-1578"""
        reg = self.TV_loss() * 0.1
        if self.cfg['reg_min_max'] and step is not None and step < 2000:
            reg = reg + torch.sum(torch.clamp(roughness - 0.9 ** 2, min=0)) + torch.sum(torch.clamp(0.1 ** 2 - roughness, min=0))
            reg = reg + torch.sum(torch.clamp(metallic - 0.98, min=0)) + torch.sum(torch.clamp(0.02 - metallic, min=0))
        return reg

    # ---- lights (reference fields.py:905-975) -----------------------------------------------------
    def get_lights(self, pts, dirs):
        """pts [pn,3], dirs [pn,D,3] -> lights [pn,D,3] (autograd), hit [pn,D] bool, inters [pn,D,3]"""
        pn, D, _ = dirs.shape
        eps = 1e-5
        with torch.no_grad():
            o = (pts[:, None, :] + dirs * eps).reshape(-1, 3)
            inters, hit_normals, depth, hit = self.ray_trace_fun(o, dirs.reshape(-1, 3))
            hit = hit.reshape(-1)
            near = (depth.reshape(-1, 1) > eps).to(torch.float32)
        flat_dirs = dirs.reshape(-1, 3)
        if self.cfg['outer_light_version'] == 'envlight':
            lights = self.outer_light.direct_light(flat_dirs, None, ~hit)
        else:                                                    # reference fields.py:913-928, on the directions that miss
            lights = torch.zeros(pn * D, 3, device=pts.device)
            midx = torch.nonzero(~hit)[:, 0]
            if midx.numel() > 0:
                d = flat_dirs[midx]
                enc = ide_encode(d)
                if self.cfg['outer_light_version'] == 'sphere_direction':
                    p = pts[torch.div(midx, D, rounding_mode='floor')]
                    p = torch.where((torch.norm(p, dim=-1) > 0.999)[:, None], p * 0.999, p)
                    dtx = torch.sum(p * d, dim=-1, keepdim=True)             # get_sphere_intersection, utils/network_utils.py:108-114
                    dist = -dtx + torch.sqrt(dtx ** 2 - torch.sum(p ** 2, dim=-1, keepdim=True) + 1 + 1e-6)
                    enc = torch.cat([enc, ide_encode(p + d * dist)], -1)
                lights = lights.index_add(0, midx, run_predictor(self.outer_light, enc, "exp", self.cfg['light_exp_max']))
        idx = torch.nonzero(hit)[:, 0]
        if idx.numel() > 0:                                           # occluded directions: indirect-light MLP
            # [posenc(hit point, 8) | IDE(view mirrored at the hit normal)] of the hit records in one kernel, already padded to
            # the 128 columns the tensor-core first layer wants
            ide_mat, ide_m, _ = _ide_device_tables(pts.device)
            enc = mc_ops.hit_encode(inters, dirs, hit_normals, idx, ide_mat, ide_m, 128)
            inner = run_predictor_padded(self.inner_light, enc, 123, "exp", self.cfg['inner_light_exp_max'])
            lights = lights.index_add(0, idx, inner)
        lights = lights * near
        return lights.reshape(pn, D, 3), hit.reshape(pn, D), inters.reshape(pn, D, 3)

    # ---- shade_mixed (reference fields.py:1075-1335) -------------------------------------------------
    def shade_mixed(self, pts, normals, view_dirs, reflections, metallic, roughness, albedo, human_poses, is_train, step=None,
                    nis_sample=None, noise: Optional[Dict[str, torch.Tensor]] = None):
        c = self.cfg
        noise = noise or {}
        pn, dev = pts.shape[0], pts.device
        use_fd = c['use_nis_diffuse'] and ((nis_sample is not None and nis_sample) or (nis_sample is None and self.use_flow_diffuse_copy))
        use_fs = c['use_nis_specular'] and ((nis_sample is not None and nis_sample) or (nis_sample is None and self.use_flow_specular_copy))
        nd, ns = c['nis_diffuse_sample_num'], c['nis_specular_sample_num']
        Dd = c['diffuse_sample_num'] + (nd if use_fd else 0)
        Ds = ns if use_fs else c['specular_sample_num']
        rand_az = is_train and c['random_azimuth']
        with torch.no_grad():
            view_angles = direction_to_angle(normals, view_dirs.unsqueeze(1)).squeeze(1)
            view_angles = view_angles / torch.tensor([2 * np.pi, 0.5 * np.pi], device=dev)
            dirs = torch.empty(pn, Dd + Ds, 3, device=dev)
            prob = torch.empty(pn, Dd + Ds, device=dev)
            rough_d = roughness.detach()
            ang_d = ang_s = None
            off = 0
            if use_fd:
                self.flow_diffuse_copy.train(is_train)
                ang_d, lj = self.flow_diffuse_copy.sample(pts, view_angles, rough_d, nd, return_jacobian=True, phi_shift=noise.get('phi_diffuse'))
                mc_ops.mc_directions(0, normals, view_dirs, ang_d, lj.reshape(pn, nd), None, nd, dirs, prob, 0)
                off = nd
            az = noise.get('az_diffuse')
            if az is None and rand_az:
                az = torch.rand(pn, 1, 1, device=dev)
            mc_ops.mc_directions(1, normals, view_dirs, self.diffuse_direction_samples, None if az is None else az.reshape(pn), None,
                                 c['diffuse_sample_num'], dirs, prob, off)
            if use_fs:
                self.flow_specular_copy.train(is_train)
                ang_s, lj = self.flow_specular_copy.sample(pts, view_angles, rough_d, ns, return_jacobian=True, phi_shift=noise.get('phi_specular'))
                mc_ops.mc_directions(0, normals, view_dirs, ang_s, lj.reshape(pn, ns), None, ns, dirs, prob, Dd)
            else:
                az = noise.get('az_specular')
                if az is None and rand_az:
                    az = torch.rand(pn, 1, 1, device=dev)
                mc_ops.mc_directions(2, normals, view_dirs, self.specular_direction_samples, None if az is None else az.reshape(pn),
                                     rough_d.reshape(pn), Ds, dirs, prob, Dd)
        lights, hit, inters = self.get_lights(pts, dirs)
        # ---- flow densities of the flow-sampled directions (reference fields.py:1254-1333): log q(x) enters the estimator
        # ---- kernel, which also accumulates the two neural-importance-sampling loss sums per point --------------------
        nis_d = use_fd and step is not None and step >= c['nis_loss_iter_diffuse']
        nis_s = use_fs and step is not None and step >= c['nis_loss_iter_specular']
        logq_d = logq_s = None
        def flow_input(ang):            # fields.py:1272-1273: the angles go through radians and back before the clamp
            phi, theta = ang[..., :1] * (2 * np.pi), ang[..., 1:2] * (0.5 * np.pi)
            return torch.cat([phi / (2 * np.pi), theta / (0.5 * np.pi)], -1).clamp(EPS, 1 - EPS)
        if nis_d:
            _, logq_d = self.flow_diffuse(pts, view_angles, roughness, flow_input(ang_d), return_jacobian=True)
        if nis_s:
            _, logq_s = self.flow_specular(pts, view_angles, roughness, flow_input(ang_s), return_jacobian=True)
        est = mc_ops.McEstimateFunction.apply(normals, view_dirs, albedo, metallic, roughness, dirs, prob, lights, hit, Dd,
                                              logq_d, ang_d if nis_d else None, logq_s, ang_s if nis_s else None)
        diffuse_colors, specular_colors = est[:, 0:3], est[:, 3:6]
        colors = linear_to_srgb(diffuse_colors + specular_colors)
        outputs = {
            'albedo': albedo, 'normal': (normals + 1) / 2, 'roughness': roughness, 'metallic': metallic,
            'diffuse_light': torch.clamp(linear_to_srgb(est[:, 6:9]), min=0, max=1),
            'specular_light': torch.clamp(linear_to_srgb(est[:, 9:12]), min=0, max=1),
            'diffuse_color': torch.clamp(linear_to_srgb(diffuse_colors), min=0, max=1),
            'specular_color': torch.clamp(linear_to_srgb(specular_colors), min=0, max=1),
            'visibility': est[:, 12:13], 'indirect_light': est[:, 13:16],
            'human_lights': torch.zeros(1, 3, device=dev),
        }
        zero = torch.zeros((), device=dev)
        outputs['loss_nis_diffuse'] = -est[:, 16].sum() / float(pn * nd * 3) if nis_d else zero
        # the reference compacts the N.L > 0 pairs and takes the mean over them (fields.py:1209-1214,1321)
        outputs['loss_nis_specular'] = -est[:, 17].sum() / (est[:, 18].sum().detach() * 3).clamp_min(1.0) if nis_s else zero
        outputs['loss_nis'] = outputs['loss_nis_diffuse'] + outputs['loss_nis_specular']
        return colors, outputs

    def forward(self, pts, view_dirs, normals, human_poses, step, is_train, noise=None):
        """reference fields.py:1453-1473"""
        view_dirs, normals = F.normalize(view_dirs, dim=-1), F.normalize(normals, dim=-1)
        metallic, roughness, albedo = self.predict_materials(pts)
        reflections = torch.sum(view_dirs * normals, -1, keepdim=True) * normals * 2 - view_dirs
        if step is not None:
            return self.shade_mixed(pts, normals, view_dirs, reflections, metallic, roughness, albedo, human_poses, is_train, step,
                                    noise=noise)
        colors, outputs = self.shade_mixed(pts, normals, view_dirs, reflections, metallic, roughness, albedo, human_poses, is_train,
                                           step, nis_sample=False, noise=noise)
        colors_nis, outputs_nis = self.shade_mixed(pts, normals, view_dirs, reflections, metallic, roughness, albedo, human_poses,
                                                   is_train, nis_sample=True, noise=noise)
        outputs_nis['rgb_pr'] = colors_nis
        outputs.update({k + '_nis': v for k, v in outputs_nis.items()})
        return colors, outputs


class MeshTracer:
    """MaterialRenderer.trace (reference network/materialRenderer.py:253-263) over the BVH kernel:
    flipped + normalised face normals, hit = depth < 10.  `offset` is the 2*unit_size push the
    renderer applies to secondary rays (materialRenderer.py:223)."""

    def __init__(self, vertices, triangles, offset: float = 0.0):
        self.ray_tracer = mc_ops.RayTracer(vertices, triangles)
        self.offset = float(offset)

    def trace(self, rays_o, rays_d):
        inters, normals, depth = self.ray_tracer.trace(rays_o, rays_d)
        depth = depth.reshape(*depth.shape, 1)
        normals = F.normalize(-normals, dim=-1)
        hit_mask = ~(depth >= 10)
        return inters, normals, depth, hit_mask

    def __call__(self, o, d):
        return self.trace(o + self.offset * d, d)


class MaterialRenderer(nn.Module):
    """Material-stage orchestration (reference network/materialRenderer.py:98-887), per-step part:
    gather the precomputed surface points of the batch -> MCShadingNetwork -> rgb / regulariser
    losses (materialRenderer.py:518-564).  Mesh / image IO and the one-off surface-point
    precompute are out of scope (SURVEY.md 8): the caller supplies the mesh arrays and the
    surface-point batch (`inters`, `normals`, `rays_d`, `rgb`) as tensors."""
    default_cfg = {'train_ray_num': 2048, 'test_ray_num': 8192, 'rgb_loss': 'charbonier', 'shader_cfg': {}, 'reg_mat': True,
                   'reg_diffuse_light': True, 'reg_diffuse_light_lambda': 0.1, 'device': 'cuda',
                   'aabb': [[-1.0, -1.0, -1.0], [1.0, 1.0, 1.0]], 'gridSize': [512, 512, 512], 'nvs_ray_num': 512,
                   'std_act': 'exp', 'inv_s_init': 0.3, 'direct_sn0': 128, 'direct_sn1': 9}

    def __init__(self, cfg, vertices, triangles, training=True):
        super().__init__()
        self.cfg = {**self.default_cfg, **cfg}
        dev = self.cfg['device']
        self.vertices, self.triangles = vertices, triangles      # the mesh predict_materials / bake_materials export onto
        self.aabb = torch.tensor(self.cfg['aabb'], device=dev)
        grid = torch.tensor(self.cfg['gridSize'], device=dev)
        self.unit_size = torch.mean((self.aabb[1] - self.aabb[0]) / (grid - 1))
        self.tracer = MeshTracer(vertices, triangles, offset=float(2 * self.unit_size))    # materialRenderer.py:223
        self.shader_network = MCShadingNetwork({**self.cfg['shader_cfg'], 'device': dev}, self.tracer, self.aabb)
        self.train_batch = None
        self.sdf_network = None                 # set by init_sdf (frozen shape-stage geometry)
        self.radius = (self.aabb[1] - torch.mean(self.aabb, 0)).mean().float()

    # ---- frozen geometry from the shape stage (reference materialRenderer.py:148-179) -----------------------------
    def init_sdf(self, ckpt):
        """Builds the frozen TensoSDF + deviation network from a shape-stage checkpoint (`ShapeRenderer.ckpt_to_save()` here or
        the reference's: keys 'kwargs', 'network_state_dict')."""
        from .fields import TensoSDF, SingleVarianceNetwork
        dev = self.cfg['device']
        kw = ckpt['kwargs']
        self.aabb = torch.as_tensor(kw['aabb'], dtype=torch.float32, device=dev)
        grid = torch.tensor(kw['gridSize'], device=dev)
        self.radius = (self.aabb[1] - torch.mean(self.aabb, 0)).mean().float()
        self.unit_size = torch.mean((self.aabb[1] - self.aabb[0]) / (grid - 1))
        self.tracer.offset = float(2 * self.unit_size)
        self.sdf_network = TensoSDF(grid, self.aabb, device=dev, init_n_levels=kw['max_levels'], sdf_n_comp=kw['sdf_n_comp'],
                                    sdf_dim=kw['sdf_dim'], app_dim=kw['app_dim'], sdf_multires=kw.get('sdf_multires', 0))
        self.deviation_net = SingleVarianceNetwork(init_val=self.cfg['inv_s_init'], activation=self.cfg['std_act']).to(dev)
        sd = ckpt['network_state_dict']
        self.sdf_network.load_state_dict({k.split('.', 1)[1]: v for k, v in sd.items() if k.startswith('sdf_network.')}, strict=False)
        self.deviation_net.load_state_dict({k.split('.', 1)[1]: v for k, v in sd.items() if k.startswith('deviation')})
        for p in list(self.sdf_network.parameters()) + list(self.deviation_net.parameters()):
            p.requires_grad = False
        self.sdf_inter_fun = lambda x: self.sdf_network.sdf(x, None)

    # ---- surface points: mesh hit refined on the SDF (reference materialRenderer.py:265-357) ----------------------
    def near_far_from_sphere(self, rays_o, rays_d):
        a = torch.sum(rays_d ** 2, dim=-1, keepdim=True)
        b = 2.0 * torch.sum(rays_o * rays_d, dim=-1, keepdim=True)
        mid = 0.5 * (-b) / a
        return torch.clamp(mid - self.radius, min=1e-3), mid + self.radius

    @torch.no_grad()
    def get_intersection_around_mesh(self, sdf_fun, inv_fun, rays_o, rays_d, m_depth, sn0=128, sn1=9):
        """reference materialRenderer.py:281-313: NeuS weights on sn0 samples within +-4 voxels of the mesh depth, sn1 importance
        samples from them (deterministic), weights again -> (z_mid, weights, mid_sdf) [pn, sn1-1]."""
        from . import sampler
        near, far = self.near_far_from_sphere(rays_o, rays_d)
        t_min = torch.minimum(torch.maximum(m_depth - self.unit_size * 4, near), far)
        t_max = torch.minimum(torch.maximum(m_depth + self.unit_size * 4, near), far)
        return sampler.probe_sections(lambda x: sdf_fun(x).reshape(-1), inv_fun.variance, rays_o, rays_d, t_min, t_max, sn0, sn1)

    @torch.no_grad()
    def trace_sdf_with_mesh(self, rays_o, rays_d, sn0, sn1):
        """reference materialRenderer.py:315-343: BVH closest hit, depth refined as the NeuS-weighted mean of sn1-1 mid-points,
        normal = normalised finite-difference SDF gradient (fused stencil kernel) flipped towards the camera."""
        inters, normals, depth, hit_mask = self.trace(rays_o, rays_d)
        hit = hit_mask.squeeze(-1)
        if self.sdf_network is not None and bool(hit.any()):
            o, d = rays_o[hit], rays_d[hit]
            z, w, _ = self.get_intersection_around_mesh(self.sdf_inter_fun, self.deviation_net, o, d, depth[hit], sn0, sn1)
            w = w / torch.sum(w, dim=-1, keepdim=True)
            w = torch.where(torch.isnan(w), torch.full_like(w, 1. / (sn1 - 1)), w)
            dep = torch.sum(w * z, -1, keepdim=True)
            pts = o + dep * d
            g, _ = self.sdf_network.gradient(pts, None)
            n = F.normalize(g, dim=-1)
            n = torch.where((n * d).sum(-1, keepdim=True) >= 0, -n, n)
            depth, inters, normals = depth.clone(), inters.clone(), normals.clone()
            depth[hit], inters[hit], normals[hit] = dep, pts, n
        return inters, normals, depth, hit.unsqueeze(-1)

    def trace_sdf_in_batch(self, rays_o, rays_d, batch_size=10240 * 5):
        """reference materialRenderer.py:265-279 (sn0 = 32, sn1 = 9 as there)"""
        outs = [self.trace_sdf_with_mesh(rays_o[i:i + batch_size], rays_d[i:i + batch_size], 32, 9)
                for i in range(0, rays_o.shape[0], batch_size)]
        return tuple(torch.cat(x, 0) for x in zip(*outs))

    def _get_trace_ray_batch_info(self, ray_batch_infos, is_train=True):
        """reference materialRenderer.py:481-504"""
        rays_o, rays_d = ray_batch_infos['rays_o'], ray_batch_infos['rays_d']
        pn = rays_o.shape[0]
        inters, normals, depth, hit_mask = self.trace_sdf_in_batch(rays_o, rays_d)
        inters, normals, depth, hit_mask = inters.reshape(pn, 3), normals.reshape(pn, 3), depth.reshape(pn, 1), hit_mask.reshape(pn)
        if is_train:
            out = {k: v[hit_mask] for k, v in ray_batch_infos.items()}
            out.update({'inters': inters[hit_mask], 'normals': normals[hit_mask], 'depth': depth[hit_mask]})
        else:
            out = dict(ray_batch_infos)
            out.update({'inters': inters, 'normals': normals, 'depth': depth, 'hit_mask': hit_mask})
        return out

    # ---- full-image relighting / novel-view inference (reference materialRenderer.py:641-752) --------------------
    NVS_KEYS = {'color': 3, 'normal': 3, 'spec_light': 3, 'diff_light': 3, 'indirect_light': 3, 'spec_color': 3, 'diff_color': 3,
                'albedo': 3, 'roughness': 1, 'metallic': 1, 'occ_trace': 1}

    @staticmethod
    def image_rays(pose, K, h, w, device):
        """`construct_ray_dirs_nerf` of reference materialRenderer.py:647-672: OpenGL pixel directions rotated by the
        camera-to-world pose [3,4] and normalised; origin = pose translation."""
        K = torch.as_tensor(np.asarray(K, np.float32), device=device)
        pose = torch.as_tensor(np.asarray(pose, np.float32), device=device)
        i, j = torch.meshgrid(torch.linspace(0, w - 1, w, device=device), torch.linspace(0, h - 1, h, device=device), indexing='ij')
        i, j = i.t(), j.t()
        d = torch.stack([(i - K[0][2]) / K[0][0], -(j - K[1][2]) / K[1][1], -torch.ones_like(i)], -1).reshape(-1, 3)
        rays_d = F.normalize(d @ pose[:3, :3].t(), dim=-1)
        rays_o = pose[:3, 3].expand(h * w, 3).contiguous()
        return {'rays_o': rays_o, 'rays_d': rays_d}

    @torch.no_grad()
    def nvs(self, pose, K, h, w, rank=0, world=1, noise_fn=None):
        """Forward-only shading of a full h x w view in `nvs_ray_num`-ray chunks (512 in the reference, :705): trace + SDF
        refinement -> MCShadingNetwork with is_train=False, step=None (both the plain and the NIS estimators run, the plain one is
        the image).  With world > 1 (BASELINE config 5) rank r shades pixels r, r+world, ... and the results are
        all-gathered back into pixel order.  `noise_fn(r0, n)` may supply the per-chunk random draws (tests)."""
        from .dist import interleaved_ids, gather_interleaved
        dev = self.cfg['device']
        rays = self.image_rays(pose, K, h, w, dev)
        if world > 1:
            ids = interleaved_ids(h * w, rank, world, dev)
            rays = {k: v[ids] for k, v in rays.items()}
        n_loc = rays['rays_o'].shape[0]
        trn = self.cfg['nvs_ray_num']
        chunks = {k: [] for k in self.NVS_KEYS}
        for r0 in range(0, n_loc, trn):
            cur = self._get_trace_ray_batch_info({k: v[r0:r0 + trn] for k, v in rays.items()}, is_train=False)
            hit = cur['hit_mask']
            out = {k: torch.zeros(hit.shape[0], d, device=dev) for k, d in self.NVS_KEYS.items()}
            out['color'][:] = 1.0
            out['normal'][:, 2] = 1.0
            if bool(hit.any()):
                nrm = cur['normals'][hit]
                so = self.shade(cur['inters'][hit], -cur['rays_d'][hit], nrm, None, False,
                                noise=None if noise_fn is None else noise_fn(r0, int(hit.sum())))
                for k, src in (('color', 'rgb_pr'), ('spec_light', 'specular_light'), ('diff_light', 'diffuse_light'),
                               ('indirect_light', 'indirect_light'), ('occ_trace', 'visibility'), ('spec_color', 'specular_color'),
                               ('diff_color', 'diffuse_color'), ('albedo', 'albedo'), ('metallic', 'metallic')):
                    out[k][hit] = so[src]
                out['normal'][hit] = nrm
                out['roughness'][hit] = torch.sqrt(so['roughness'])          # predictions are roughness squared (:738)
            for k in self.NVS_KEYS:
                chunks[k].append(out[k])
        res = {}
        for k, d in self.NVS_KEYS.items():
            local = torch.cat(chunks[k], 0) if chunks[k] else torch.zeros(0, d, device=dev)
            full = gather_interleaved(local, h * w) if world > 1 else local
            res[k] = full.reshape(h, w, -1).cpu().numpy()
        return res

    def trace(self, rays_o, rays_d):
        return self.tracer.trace(rays_o, rays_d)

    # ---- material export onto the mesh ------------------------------------------------------------------------------
    def _materials_at(self, pts, batch_size):
        """[n,3] -> [n,5] fp32: albedo (3), roughness (sqrt of the predicted roughness squared), metallic"""
        out = []
        for i in range(0, pts.shape[0], batch_size):
            metallic, roughness, albedo = self.shader_network.predict_materials(pts[i:i + batch_size])
            out.append(torch.cat([albedo, torch.sqrt(roughness), metallic], -1).float())
        return torch.cat(out, 0) if out else torch.zeros(0, 5, device=pts.device)

    @torch.no_grad()
    def predict_materials(self, batch_size: int = 8192):
        """Per-vertex materials of the mesh the renderer was built with -> {'metallic' [V,1], 'roughness' [V,1], 'albedo' [V,3]}
        on the device, from the material stage at the vertex positions in batches of `batch_size`.  Roughness is reported as
        sqrt of the network's squared roughness, as `nvs` reports it.  This is the export behind relighting with vertex colours;
        the reference renderer has a method of this name, but its source is not part of this repository, so whether its return
        form (keys, shapes, roughness convention) matches this one is unverified."""
        dev = self.cfg['device']
        v = torch.as_tensor(self.vertices).to(device=dev, dtype=torch.float32).contiguous()
        m = self._materials_at(v, int(batch_size))
        return {'metallic': m[:, 4:5], 'roughness': m[:, 3:4], 'albedo': m[:, 0:3]}

    @torch.no_grad()
    def bake_materials(self, resolution: int = 2048, padding: int = 2, batch_size: int = 8192):
        """Materials baked into textures over a UV atlas of the renderer's mesh (geometry.uv_atlas, geometry.bake_texture) ->
        {'atlas': UVAtlas (split vertices, triangles, uv, ...), 'albedo' [R,R,3], 'roughness' [R,R,1] (sqrt convention, as
        predict_materials), 'metallic' [R,R,1] fp32, 'mask' [R,R] bool (texels covered before dilation)}.  Texture row j spans
        v in [j/R, (j+1)/R]."""
        from .geometry import bake_texture, uv_atlas
        dev = self.cfg['device']
        atlas = uv_atlas(torch.as_tensor(self.vertices).to(dev), torch.as_tensor(self.triangles).to(dev), resolution, padding)
        tex, mask = bake_texture(atlas, lambda p: self._materials_at(p, int(batch_size)), 5)
        return {'atlas': atlas, 'albedo': tex[..., 0:3], 'roughness': tex[..., 3:4], 'metallic': tex[..., 4:5], 'mask': mask}

    def get_train_opt_params(self, learning_rate_xyz, learning_rate_net, learning_rate_env):
        return self.shader_network.get_optparam_groups(learning_rate_xyz, learning_rate_net, learning_rate_env)

    def ckpt_to_save(self):
        return {'network_state_dict': self.state_dict()}

    def set_train_batch(self, batch: Dict[str, torch.Tensor]):
        self.train_batch, self.train_batch_i, self.tbn = batch, 0, batch['inters'].shape[0]

    def shade(self, pts, view_dirs, normals, human_poses, is_train, step=None, noise=None):
        rgb_pr, outputs = self.shader_network(pts, view_dirs, normals, human_poses, step, is_train, noise=noise)
        outputs['rgb_pr'] = rgb_pr
        return outputs

    def compute_rgb_loss(self, rgb_pr, rgb_gt):
        if self.cfg['rgb_loss'] == 'l1':
            return torch.sum(F.l1_loss(rgb_pr, rgb_gt, reduction='none'), -1)
        if self.cfg['rgb_loss'] == 'charbonier':
            return torch.sqrt(torch.sum((rgb_gt - rgb_pr) ** 2, dim=-1) + 0.001)
        raise NotImplementedError

    def compute_diffuse_light_regularization(self, diffuse_lights):
        return torch.sum(torch.abs(diffuse_lights - torch.mean(diffuse_lights, dim=-1, keepdim=True)), dim=-1) * self.cfg['reg_diffuse_light_lambda']

    def _shuffle_train_batch(self):
        """reference materialRenderer.py:472-476: a new host-side permutation of the surface-point pool at every wrap"""
        self.train_batch_i = 0
        idx = torch.randperm(self.tbn, device='cpu')
        for k, v in self.train_batch.items():
            pinned = v.is_pinned()
            v = v[idx]
            self.train_batch[k] = v.pin_memory() if pinned else v

    def train_step(self, step, noise=None):
        rn = self.cfg['train_ray_num']
        dev = self.cfg['device']
        b = {k: v[self.train_batch_i:self.train_batch_i + rn].to(dev, non_blocking=True) for k, v in self.train_batch.items()}
        self.train_batch_i += rn
        if self.train_batch_i + rn >= self.tbn:
            self._shuffle_train_batch()
        self.shader_network.update_step(step)
        out = self.shade(b['inters'], -b['rays_d'], b['normals'], None, True, step, noise=noise)
        out['rgb_gt'] = b['rgb']
        out['loss_rgb'] = self.compute_rgb_loss(out['rgb_pr'], b['rgb'])
        out['psnr'] = 20 * torch.log10(1.0 / torch.sqrt(F.mse_loss(out['rgb_pr'], b['rgb'])))
        if self.cfg['reg_mat']:
            out['loss_mat_reg'] = self.shader_network.material_regularization(b['inters'], b['normals'], out['metallic'], out['roughness'],
                                                                              out['albedo'], step)
        if self.cfg['reg_diffuse_light']:
            out['loss_diffuse_light'] = self.compute_diffuse_light_regularization(out['diffuse_light'])
        return out

    def forward(self, data):
        if self.shader_network.cfg['outer_light_version'] == 'envlight':
            self.shader_network.outer_light.build_mips_direct()      # materialRenderer.py:760-761
        return self.train_step(data['step'], data.get('noise'))
