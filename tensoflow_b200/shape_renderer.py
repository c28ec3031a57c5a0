"""Shape-stage per-ray work (reference network/shapeRenderer.py) on the sm_100a kernels.

`render_core` mirrors ShapeRenderer.render_core (reference shapeRenderer.py:1105-1277):
packed samples in, per-ray colour / acc / normal and the sample-level loss terms out.
Two kernels do the work: the fused TensoSDF stencil (field + FD normals + hessian) and
the NeuS alpha + compositing kernel; the few remaining elementwise ops are index
plumbing.
"""
from __future__ import annotations

from typing import Callable, Dict, Optional

import torch
import torch.nn.functional as F

from . import ops


def near_far_from_sphere(rays_o, dirs, radius=1.0):
    """reference shapeRenderer.py:676-684"""
    a = torch.sum(dirs ** 2, dim=-1, keepdim=True)
    b = 2.0 * torch.sum(rays_o * dirs, dim=-1, keepdim=True)
    mid = 0.5 * (-b) / a
    return torch.clamp(mid - radius, min=1e-3), mid + radius


def compute_ball_radii(distance, radiis, cos):
    """reference shapeRenderer.py:966-970"""
    inverse_cos = 1.0 / cos
    tmp = (inverse_cos * inverse_cos - 1).sqrt() - radiis
    return distance * radiis * cos / (tmp * tmp + 1.0).sqrt()


def ray_offsets_from_indices(ray_indices: torch.Tensor, n_rays: int) -> torch.Tensor:
    """sorted int64 ray_indices [N] (nerfacc packing) -> CSR offsets int32 [n_rays+1]"""
    bounds = torch.arange(n_rays + 1, device=ray_indices.device, dtype=ray_indices.dtype)
    return torch.searchsorted(ray_indices.contiguous(), bounds).to(torch.int32)


def charbonnier(rgb_pr, rgb_gt, epsilon=0.001):
    """reference shapeRenderer.py:803-805"""
    return torch.sqrt(torch.sum((rgb_gt - rgb_pr) ** 2, dim=-1) + epsilon)


def render_core(field, variance: torch.Tensor, color_fn: Callable, rays_o, dirs, radiis, rays_cos, t_starts, t_ends,
                ray_indices, cos_anneal_ratio: float = 1.0, base_radii: Optional[float] = None, is_train: bool = True,
                train_variance: bool = True, white_bg: bool = True) -> Dict[str, torch.Tensor]:
    """reference shapeRenderer.py:1105-1206.  `field` is a tensoflow_b200.fields.TensoSDF,
    `color_fn(points, normals, view_dirs, feature_vectors) -> [N,3]` stands for the shading network."""
    n_rays = rays_o.shape[0]
    mid = (t_starts + t_ends) * 0.5
    dists = t_ends - t_starts
    viewdir = dirs[ray_indices]
    pts = rays_o[ray_indices] + viewdir * mid[:, None]
    if base_radii is None:
        base_radii = float(field.aabbSize[0] / 2 / field.gridSize[0])          # reference shapeRenderer.py:251
    ball = compute_ball_radii(mid[:, None], radiis[ray_indices], rays_cos[ray_indices])
    levels = torch.log2(ball / base_radii)
    sdf, feat, grads, hess = field.stencil(pts, levels)
    normals = F.normalize(grads, dim=-1)
    colors = color_fn(pts, normals, -viewdir, feat)
    offsets = ray_offsets_from_indices(ray_indices, n_rays)
    vals = torch.cat([colors, grads], -1)
    alpha, weights, acc, out = ops.NeusCompositeFunction.apply(sdf, grads, dists, dirs, offsets, variance,
                                                               float(cos_anneal_ratio), vals, train_variance)
    acc = acc[:, None]
    rgb = out[:, :3]
    if white_bg:
        rgb = rgb + (1 - acc)
    up = torch.tensor([0.0, 0.0, 1.0], device=rgb.device)
    normal = F.normalize(out[:, 3:6] * acc + (1.0 - acc) * up, dim=-1)
    res = {
        'ray_rgb': rgb, 'acc': acc, 'normal': normal,
        'gradient_error': (torch.linalg.norm(grads, ord=2, dim=-1) - 1.0) ** 2,
        'sample_num': pts.shape[0] / max(n_rays, 1),
        'sdf': sdf, 'alpha': alpha, 'weights': weights, 'gradients': grads, 'feat': feat, 'levels': levels,
        'points': pts,
    }
    if is_train and pts.shape[0] > 0:
        res['loss_sparse'] = torch.exp(-20.0 * sdf.abs()).mean()
        res['loss_hessian'] = hess.abs().mean()
        res['hessian'] = hess
        res['std'] = torch.mean(1 / torch.exp(variance * 10.0).clip(1e-6, 1e6))
    return res


# ======================================================================================
# Full shape-stage orchestration (reference network/shapeRenderer.py:79-1326).  Dataset /
# image IO is out of scope (SURVEY.md 8): ray batches are handed in as tensors.
# ======================================================================================
def get_sphere_intersection(pts, dirs):
    """reference utils/network_utils.py:108-114"""
    dtx = torch.sum(pts * dirs, dim=-1, keepdim=True)
    xtx = torch.sum(pts ** 2, dim=-1, keepdim=True)
    dist = dtx ** 2 - xtx + 1
    return -dtx + torch.sqrt(dist + 1e-6)


def get_intersection(sdf_fun, variance, pts, dirs, sn0=128, sn1=9):
    """reference utils/network_utils.py:172-202 (secondary-ray occlusion probe, no_grad) on the `tf_probe_*` kernels
    (tensoflow_b200/sampler.py): `variance` is the SingleVarianceNetwork parameter (inv_s = exp(10 variance)),
    sdf_fun(points [N,3]) -> [N,1]."""
    from . import sampler
    dev = pts.device
    inside = torch.norm(pts, dim=-1) < 0.999
    pn = pts.shape[0]
    hit_z = torch.zeros([pn, sn1 - 1], device=dev)
    hit_w = torch.zeros([pn, sn1 - 1], device=dev)
    hit_sdf = -torch.ones([pn, sn1 - 1], device=dev)
    if torch.sum(inside) > 0:
        p, d = pts[inside], dirs[inside]
        max_dist = get_sphere_intersection(p, d)
        z_mid, w, mid_sdf = sampler.probe_sections(lambda x: sdf_fun(x).reshape(-1), variance, p, d, None, max_dist, sn0, sn1)
        hit_z[inside], hit_w[inside], hit_sdf[inside] = z_mid, w, mid_sdf
    return hit_z, hit_w, hit_sdf


class AlphaGridMask(torch.nn.Module):
    """reference shapeRenderer.py:79-97"""

    def __init__(self, device, aabb, alpha_volume):
        super().__init__()
        self.device = device
        self.aabb = aabb.to(device)
        self.aabbSize = self.aabb[1] - self.aabb[0]
        self.invgridSize = 1.0 / self.aabbSize * 2
        self.alpha_volume = alpha_volume.view(1, 1, *alpha_volume.shape[-3:])
        self._a0 = [float(v) for v in self.aabb[0].cpu()]
        self._inv = [float(v) for v in self.invgridSize.cpu()]

    def sample_alpha(self, xyz_sampled):
        """trilinear lookup on `tf_alpha_mask_sample` (the reference's F.grid_sample(..., align_corners=True))"""
        import ctypes as C
        from . import _lib
        from ._lib import check, ptr, stream_ptr
        xyz = xyz_sampled.detach().reshape(-1, 3).float().contiguous()
        vol = self.alpha_volume.float().contiguous()
        out = torch.empty(xyz.shape[0], device=xyz.device, dtype=torch.float32)
        _, _, D, H, W = vol.shape
        check(_lib.load().tf_alpha_mask_sample(ptr(vol), D, H, W, (C.c_float * 3)(*self._a0), (C.c_float * 3)(*self._inv), ptr(xyz),
                                               xyz.shape[0], ptr(out), stream_ptr()), "tf_alpha_mask_sample")
        return out


class ShapeRenderer(torch.nn.Module):
    default_cfg = {
        'std_act': 'exp', 'inv_s_init': 0.3, 'freeze_inv_s_step': None, 'n_samples': 64, 'n_importance': 64, 'up_sample_steps': 4,
        'perturb': 1.0, 'anneal_end': 50000, 'train_ray_num': 1024, 'test_ray_num': 2048, 'clip_sample_variance': True,
        'rgb_loss': 'charbonier', 'apply_occ_loss': True, 'apply_tv_loss': True, 'apply_sparse_loss': True, 'apply_hessian_loss': True,
        'apply_gaussian_loss': False, 'occ_loss_step': 20000, 'occ_loss_max_pn': 2048, 'occ_sdf_thresh': 0.01, 'gaussianLoss_step': 20000,
        'device': 'cuda', 'gridSize': [512, 512, 512], 'aabb': [[-1.0, -1.0, -1.0], [1.0, 1.0, 1.0]], 'step_ratio': 0.5,
        'alphaMask_thres': 0.0001, 'sdf_n_comp': 16, 'sdf_dim': 128, 'app_dim': 128, 'sdf_multires': 0, 'max_levels': 1,
        'has_radiance_field': False, 'radiance_field_step': 0, 'predict_BG': False, 'isBGWhite': True, 'apply_mask_loss': False,
        'mul_length': 10, 'use_occ_grid': False, 'occ_grid_reso': 128, 'shader_config': {},
    }

    def __init__(self, cfg, training=True):
        super().__init__()
        from .fields import TensoSDF, SingleVarianceNetwork, TVLoss
        from .shape_shader import ShapeShadingNetwork
        self.cfg = {**self.default_cfg, **cfg}
        c = self.cfg
        if c['predict_BG']:
            raise NotImplementedError("predict_BG raises in the reference too (shapeRenderer.py:1109-1110)")
        self.device = c['device']
        self.aabb = torch.tensor(c['aabb'].cpu().tolist() if isinstance(c['aabb'], torch.Tensor) else c['aabb'], device=self.device)
        self.radius = (self.aabb[1] - torch.mean(self.aabb, axis=0)).mean().float()
        self.alphaMask = None
        self.occ_grid = None
        if c['use_occ_grid']:                                   # reference shapeRenderer.py:211-215
            from .occ_grid import OccGridEstimator
            self.occ_grid = OccGridEstimator(self.aabb.reshape(-1), resolution=c['occ_grid_reso']).to(self.device)
        self.update_stepSize(torch.tensor(c['gridSize']), c['max_levels'])
        self.sdf_network = TensoSDF(self.gridSize, self.aabb, device=self.device, init_n_levels=self.max_levels, sdf_n_comp=c['sdf_n_comp'],
                                    sdf_dim=c['sdf_dim'], app_dim=c['app_dim'], sdf_multires=c['sdf_multires'])
        self.tv_reg = TVLoss()
        self.deviation_network = SingleVarianceNetwork(init_val=c['inv_s_init'], activation=c['std_act']).to(self.device)
        shader_cfg = {'has_radiance_field': c['has_radiance_field'], 'radiance_field_step': c['radiance_field_step'],
                      'app_feats_dim': c['app_dim'], 'device': self.device, **c['shader_config']}
        self.color_network = ShapeShadingNetwork(shader_cfg)
        self.sdf_inter_fun = lambda x: self.sdf_network.sdf(x, None)
        self.train_batch = None

    # ---- bookkeeping ------------------------------------------------------------------------
    def update_stepSize(self, gridSize, max_levels):
        """reference shapeRenderer.py:243-254"""
        self.aabbSize = self.aabb[1] - self.aabb[0]
        self.gridSize = torch.tensor(gridSize.cpu().tolist(), dtype=torch.int32).to(self.device)
        self.max_levels = max_levels
        self.units = self.aabbSize / (self.gridSize - 1)
        self.stepSize = torch.mean(self.units) * self.cfg['step_ratio']
        self.base_radii = self.aabbSize[0] / 2.0 / self.gridSize[0]
        self._base_radii_f = float(self.base_radii)              # host copy: the sampler kernels take it by value

    def get_train_opt_params(self, lr_xyz, lr_net, lr_env=0.01):
        g = self.sdf_network.get_optparam_groups(lr_xyz, lr_net)
        g += [{'params': self.deviation_network.parameters(), 'lr': lr_net}]
        g += self.color_network.get_optparam_groups(lr_net, lr_env)
        return g

    def get_kwargs(self):
        """reference shapeRenderer.py:326-341 (the keys MaterialRenderer.init_sdf reads back)"""
        c = self.cfg
        return {'aabb': self.aabb, 'gridSize': self.gridSize.tolist(), 'sdf_n_comp': c['sdf_n_comp'], 'sdf_dim': c['sdf_dim'],
                'app_dim': c['app_dim'], 'sdf_multires': c['sdf_multires'], 'alphaMask_thres': c['alphaMask_thres'],
                'step_ratio': c['step_ratio'], 'max_levels': self.max_levels,
                # carried by the reference dictionary as well (shapeRenderer.py:332,338); unused by this package
                'appearance_n_comp': c.get('app_n_comp', c.get('appearance_n_comp', 0)),
                'marched_weights_thres': c.get('marched_weights_thres', 0.0001)}

    def ckpt_to_save(self):
        """reference shapeRenderer.py:343-354: same dictionary layout (kwargs, state dict, bit-packed alpha mask)"""
        import numpy as np
        ckpt = {'kwargs': self.get_kwargs(), 'network_state_dict': self.state_dict()}
        if self.alphaMask is not None:
            vol = self.alphaMask.alpha_volume.bool().cpu().numpy()
            ckpt.update({'alphaMask.shape': vol.shape, 'alphaMask.mask': np.packbits(vol.reshape(-1)),
                         'alphaMask.aabb': self.alphaMask.aabb.cpu()})
        if self.occ_grid is not None:
            ckpt['occ_grid_state_dict'] = self.occ_grid.state_dict()
        return ckpt

    def load_ckpt(self, ckpt):
        """reference shapeRenderer.py:356-363; a checkpoint saved at a finer grid than this module was built with is followed:
        the factors take the stored shapes and `gridSize` / `max_levels` / step sizes are updated (the reference trainer replays its
        upsampling schedule before loading instead)."""
        import numpy as np
        if 'alphaMask.aabb' in ckpt:
            length = int(np.prod(ckpt['alphaMask.shape']))
            vol = torch.from_numpy(np.unpackbits(ckpt['alphaMask.mask'])[:length].reshape(ckpt['alphaMask.shape']))
            self.alphaMask = AlphaGridMask(self.device, ckpt['alphaMask.aabb'].to(self.device), vol.float().to(self.device))
        if 'occ_grid_state_dict' in ckpt and self.occ_grid is not None:
            self.occ_grid.load_state_dict(ckpt['occ_grid_state_dict'], strict=False)
        self.load_state_dict(ckpt['network_state_dict'], strict=False)       # TensoSDF adopts the stored factor shapes
        kw = ckpt.get('kwargs')
        if kw is not None and (list(kw['gridSize']) != self.gridSize.tolist() or kw['max_levels'] != self.max_levels):
            res = torch.tensor(kw['gridSize'])
            self.sdf_network.update_gridSize_aabb(res.long().cpu(), self.sdf_network.aabb, kw['max_levels'])
            self.update_stepSize(res, kw['max_levels'])

    def upsample_sdf_grid(self, res_target):
        res, n_levels = self.sdf_network.upsample_volume_grid(torch.as_tensor(res_target))
        self.update_stepSize(res, n_levels)

    def get_anneal_val(self, step):
        return 1.0 if self.cfg['anneal_end'] < 0 else float(min(1.0, step / self.cfg['anneal_end']))

    def set_train_batch(self, batch: Dict[str, torch.Tensor]):
        """rays_o, rays_d, dirs, radiis, rays_cos, rgbs, human_poses (host tensors, like the reference's CPU-resident batch)"""
        self.train_batch, self.train_batch_i, self.tbn = batch, 0, batch['rays_o'].shape[0]

    def _shuffle_train_batch(self):
        """reference shapeRenderer.py:411-415: a new host-side permutation of the ray pool at every wrap"""
        self.train_batch_i = 0
        idx = torch.randperm(self.tbn, device='cpu')
        for k, v in self.train_batch.items():
            pinned = v.is_pinned()
            v = v[idx]
            self.train_batch[k] = v.pin_memory() if pinned else v

    # ---- sampling (reference shapeRenderer.py:820-932) -----------------------------------------
    def sample_ray(self, rays_o, dirs, near, far, perturb, radiis=None, rays_cos=None, t_rand=None):
        """Coarse + hierarchical importance depths on the `tf_sampler_*` kernels (tensoflow_b200/sampler.py); the SDF of the
        query points comes from the SDF-only field kernel.  Returns the packed (t_starts, t_ends, ray_indices)."""
        from . import sampler
        c = self.cfg
        net = self.sdf_network
        sdf_fn = lambda pts, level: net.sdf(pts, level.reshape(-1, 1)).reshape(-1)
        t_starts, t_ends, ray_indices, offsets = sampler.hierarchical_sample(
            sdf_fn, self.aabb, self._base_radii_f, rays_o, dirs, near, far, radiis, rays_cos, c['n_samples'], c['n_importance'],
            c['up_sample_steps'], perturb, t_rand, self.deviation_network.variance, c['clip_sample_variance'])
        self._last_ray_offsets = (ray_indices, offsets)          # the compositor's CSR offsets come for free
        return t_starts, t_ends, ray_indices

    # ---- occlusion loss (reference shapeRenderer.py:1027-1103) ------------------------------------
    def compute_occ_loss(self, occ_info, points, sdf, gradients, dirs, step, perm=None):
        c = self.cfg
        if step < c['occ_loss_step']:
            return torch.zeros(1, device=points.device)
        occ_prob, reflective = occ_info['occ_prob'], occ_info['reflective']
        inner = ~((self.aabb[0] > points) | (points > self.aabb[1])).any(dim=-1)
        mask = inner & (torch.sum(gradients * dirs, -1) < 0) & (torch.abs(sdf) < c['occ_sdf_thresh'])
        if torch.sum(mask) > c['occ_loss_max_pn']:
            indices = torch.nonzero(mask)[:, 0]
            idx = torch.randperm(indices.shape[0], device=points.device) if perm is None else perm
            indices = indices[idx[:c['occ_loss_max_pn']]]
            mask = torch.zeros_like(mask)
            mask[indices] = 1
        if torch.sum(mask) > 0:
            if self.occ_grid is None:
                _, inter_prob, _ = get_intersection(self.sdf_inter_fun, self.deviation_network.variance, points[mask], reflective[mask], sn0=64, sn1=16)
                return F.l1_loss(occ_prob[mask], torch.sum(inter_prob, -1, keepdim=True))
            return F.l1_loss(occ_prob[mask], self.occ_grid_hit_probability(points[mask], reflective[mask]))
        return torch.zeros(1, device=points.device)

    @torch.no_grad()
    def occ_grid_hit_probability(self, pts, dirs):
        """Occlusion probability of the secondary rays (pts, dirs) marched through the occupancy grid with the fixed step
        (reference shapeRenderer.py:1055-1100) -> [pn,1]."""
        occ_prob_gt = torch.zeros(pts.shape[0], 1, device=pts.device)
        inside = torch.norm(pts, dim=-1) < 0.999
        if torch.sum(inside) == 0:
            return occ_prob_gt
        pts, dirs = pts[inside].contiguous(), dirs[inside].contiguous()
        pn = pts.shape[0]
        step = float(self.stepSize)
        max_dist = get_sphere_intersection(pts, dirs)
        ray_indices, t0, t1 = self.occ_grid.sampling(pts, dirs, near_plane=step, far_plane=max_dist.max().item(), render_step_size=step,
                                                     stratified=False)
        if ray_indices.shape[0] == 0:
            return occ_prob_gt
        prev_points = pts[ray_indices] + dirs[ray_indices] * t0.unsqueeze(-1)
        next_points = pts[ray_indices] + dirs[ray_indices] * t1.unsqueeze(-1)
        prev_sdf = self.sdf_network.sdf(prev_points)[..., 0]
        next_sdf = self.sdf_network.sdf(next_points)[..., 0]
        mid_sdf = (prev_sdf + next_sdf) * 0.5
        cos_val = (next_sdf - prev_sdf) / (t1 - t0 + 1e-5)
        surface_mask = (cos_val < 0)
        cos_val = torch.clamp(cos_val, max=0)
        inv_s = self.deviation_network(prev_points).clip(1e-6, 1e6)[..., 0]
        prev_cdf = torch.sigmoid((mid_sdf - cos_val * step * 0.5) * inv_s)
        next_cdf = torch.sigmoid((mid_sdf + cos_val * step * 0.5) * inv_s)
        alpha = (prev_cdf - next_cdf + 1e-5) / (prev_cdf + 1e-5) * surface_mask.float()
        # nerfacc.render_weight_from_alpha + accumulate_along_rays(values=None): 1 - prod(1 - alpha) per ray, here through a
        # segmented sum of log(1 - alpha) over the packed samples (no_grad target of an L1 loss)
        log_t = torch.zeros(pn, device=pts.device).index_add_(0, ray_indices, torch.log1p(-alpha.clamp(max=1.0 - 1e-7)))
        occ_prob_gt[inside] = (1.0 - torch.exp(log_t))[:, None]
        return occ_prob_gt

    @torch.no_grad()
    def compute_alpha(self, points):
        """reference shapeRenderer.py:972-993: opacity of one fixed-size step at `points` (the occupancy-grid refresh criterion)"""
        if points.shape[0] == 0:
            return torch.zeros(0, device=self.device)
        sdf = self.sdf_network.sdf(points).squeeze(-1)
        inv_s = self.deviation_network(points).clip(1e-6, 1e6)[..., 0]
        prev_cdf = torch.sigmoid((sdf + self.stepSize * 0.5) * inv_s)
        next_cdf = torch.sigmoid((sdf - self.stepSize * 0.5) * inv_s)
        return ((prev_cdf - next_cdf + 1e-5) / (prev_cdf + 1e-5)).clip(0.0, 1.0)

    # ---- render (reference shapeRenderer.py:934-963, 1105-1277) --------------------------------------
    def render(self, ray_batch, near, far, human_poses=None, perturb_overwrite=-1, cos_anneal_ratio=0.0, is_train=True, step=None,
               t_rand=None):
        perturb = self.cfg['perturb'] if perturb_overwrite < 0 else perturb_overwrite
        rays_o, rays_d, dirs, radiis, rays_cos = (ray_batch[k] for k in ('rays_o', 'rays_d', 'dirs', 'radiis', 'rays_cos'))
        if self.occ_grid is not None:                           # reference shapeRenderer.py:950-959
            ray_indices, t_starts, t_ends = self.occ_grid.sampling(rays_o, dirs, near_plane=near.min().item(), far_plane=far.max().item(),
                                                                   render_step_size=float(self.stepSize), stratified=is_train, noise=t_rand)
        else:
            t_starts, t_ends, ray_indices = self.sample_ray(rays_o, dirs, near, far, perturb, radiis=radiis, rays_cos=rays_cos, t_rand=t_rand)
        return self.render_core(rays_o, rays_d, dirs, radiis, rays_cos, t_starts, t_ends, ray_indices, human_poses,
                                cos_anneal_ratio=cos_anneal_ratio, step=step, is_train=is_train)

    def render_core(self, rays_o, rays_d, viewdirs, radiis, rays_cos, t_starts, t_ends, ray_indices, human_poses=None,
                    cos_anneal_ratio=0.0, step=None, is_train=True):
        c = self.cfg
        batch_size = rays_o.shape[0]
        dev = rays_o.device
        mid_t = (t_starts + t_ends) * 0.5
        dists = t_ends - t_starts
        points = rays_o[ray_indices] + viewdirs[ray_indices] * mid_t[:, None]
        if self.occ_grid is None and self.alphaMask is not None:                  # reference shapeRenderer.py:1119
            keep = self.alphaMask.sample_alpha(points) > 0
            ray_indices, mid_t, points, dists = ray_indices[keep], mid_t[keep], points[keep], dists[keep]
        N = ray_indices.shape[0]
        viewdir = viewdirs[ray_indices]
        ball = compute_ball_radii(mid_t[:, None], radiis[ray_indices], rays_cos[ray_indices])
        levels = torch.log2(ball / self.base_radii)
        variance = self.deviation_network.variance
        train_var = not (c['freeze_inv_s_step'] is not None and step < c['freeze_inv_s_step'])
        sdf, feature_vector, gradients, hessian = self.sdf_network.stencil(points, levels)
        valid_normals = F.normalize(gradients, dim=-1)
        with_rad = c['has_radiance_field'] and step > c['radiance_field_step']
        sampled_color, sampled_radiance, occ_info = self.color_network(points, valid_normals, -viewdir, feature_vector, None, step=step)
        vals = [sampled_color, gradients]
        if with_rad:
            vals += [sampled_radiance, occ_info['roughness']]
        last = getattr(self, '_last_ray_offsets', None)
        if last is not None and last[0] is ray_indices and N == ray_indices.shape[0]:
            offsets = last[1]                                     # CSR offsets of the sampler (no sample was culled since)
        else:
            offsets = ray_offsets_from_indices(ray_indices, batch_size)
        alpha, weights, acc, out = ops.NeusCompositeFunction.apply(sdf, gradients, dists, viewdirs, offsets, variance,
                                                                   float(cos_anneal_ratio), torch.cat(vals, -1), train_var)
        acc_map = acc[:, None]
        color = out[:, :3] + (1 - acc_map) if c['isBGWhite'] else out[:, :3]
        outputs = {'ray_rgb': color, 'gradient_error': (torch.linalg.norm(gradients, ord=2, dim=-1) - 1.0) ** 2, 'acc': acc_map,
                   'sample_num': N / batch_size}
        up = torch.tensor([0.0, 0.0, 1.0], device=dev)
        outputs['normal'] = F.normalize(out[:, 3:6] * acc_map + (1. - acc_map) * up, dim=-1)
        if with_rad:
            outputs['radiance'] = out[:, 6:9] + (1 - acc_map) if c['isBGWhite'] else out[:, 6:9]
            outputs['roughness_weights'] = out[:, 9].clone().detach()
        inv_s = torch.exp(variance * 10.0).clip(1e-6, 1e6)
        outputs['std'] = torch.mean(1 / inv_s).reshape(()) if N > 0 else torch.zeros(1, device=dev)
        if step is not None and step < 1000:
            outputs['sdf_pts'], outputs['sdf_vals'] = (points, sdf) if N > 0 else (torch.zeros(1, device=dev), torch.zeros(1, device=dev))
        if c['apply_occ_loss']:
            outputs['loss_occ'] = self.compute_occ_loss(occ_info, points, sdf, valid_normals, viewdir, step) if N > 0 else torch.zeros(1, device=dev)
        if c['apply_gaussian_loss'] and step > c['gaussianLoss_step']:
            outputs['loss_gaussian'] = self.sdf_network.grid_gaussian_loss() if N > 0 else torch.zeros(1, device=dev)
        if c['apply_tv_loss']:
            outputs['loss_tv_sdf'] = self.sdf_network.TV_loss_sdf(self.tv_reg)
        if c['apply_sparse_loss']:
            outputs['loss_sparse'] = torch.exp(-20. * sdf.abs()).mean() if N > 0 else torch.zeros(1, device=dev)
        if c['apply_hessian_loss']:
            outputs['loss_hessian'] = hessian.abs().mean() if (is_train and N > 0) else torch.zeros(1, device=dev)
        outputs.update({'_sdf': sdf, '_alpha': alpha, '_weights': weights})
        return outputs

    def compute_rgb_loss(self, rgb_pr, rgb_gt):
        """reference shapeRenderer.py:796-808"""
        kind = self.cfg['rgb_loss']
        if kind == 'l2':
            return torch.sum((rgb_pr - rgb_gt) ** 2, -1)
        if kind == 'l1':
            return torch.sum(F.l1_loss(rgb_pr, rgb_gt, reduction='none'), -1)
        if kind == 'smooth_l1':
            return torch.sum(F.smooth_l1_loss(rgb_pr, rgb_gt, reduction='none', beta=0.25), -1)
        if kind == 'charbonier':
            return charbonnier(rgb_pr, rgb_gt)
        raise NotImplementedError

    def train_step(self, step):
        """reference shapeRenderer.py:777-794: slice the host batch, H2D, render, losses."""
        rn = self.cfg['train_ray_num']
        b = {k: v[self.train_batch_i:self.train_batch_i + rn].to(self.device, non_blocking=True) for k, v in self.train_batch.items()}
        self.train_batch_i += rn
        if self.train_batch_i + rn >= self.tbn:
            self._shuffle_train_batch()
        near, far = near_far_from_sphere(b['rays_o'], b['dirs'], self.radius)
        outputs = self.render(b, near, far, b.get('human_poses'), -1, self.get_anneal_val(step), is_train=True, step=step)
        outputs['loss_rgb'] = self.compute_rgb_loss(outputs['ray_rgb'], b['rgbs'])
        outputs['psnr'] = 20 * torch.log10(1.0 / torch.sqrt(F.mse_loss(outputs['ray_rgb'], b['rgbs'])))
        if self.cfg['has_radiance_field'] and step > self.cfg['radiance_field_step']:
            outputs['loss_radiance'] = self.compute_rgb_loss(outputs['radiance'], b['rgbs']) * outputs['roughness_weights']
            outputs['loss_rgb'] = outputs['loss_rgb'] * (1.0 - outputs['roughness_weights'])
        if self.cfg['apply_mask_loss']:
            outputs['loss_mask'] = F.binary_cross_entropy(outputs['acc'].clip(1e-3, 1.0 - 1e-3), (b['masks'] > 0.5).float())
        return outputs

    def forward(self, data):
        """reference shapeRenderer.py:1279-1306 (training branch)"""
        if self.occ_grid is not None:                           # reference shapeRenderer.py:1285-1290
            self.occ_grid.update_every_n_steps(step=data['step'], occ_eval_fn=self.compute_alpha, n=100, warmup_steps=10000)
        self.color_network.envlight.build_mips()
        return self.train_step(data['step'])

    # ---- full-image inference (reference shapeRenderer.py:569-668) ------------------------------------------------
    @staticmethod
    def image_rays(pose, K, h, w, device):
        """nerfDataType ray construction of the reference (`construct_ray_dirs_nerf` shapeRenderer.py:592-621 and
        `_process_ray_batch_nerf` :708-719): pixel directions in the OpenGL camera frame, tri-mip pixel radii, rays_cos,
        rotated by the camera-to-world pose [3,4]."""
        K = torch.as_tensor(K, dtype=torch.float32, device=device)
        pose = torch.as_tensor(pose, dtype=torch.float32, device=device)
        i, j = torch.meshgrid(torch.linspace(0, w - 1, w, device=device), torch.linspace(0, h - 1, h, device=device), indexing='ij')
        i, j = i.t(), j.t()
        rays_d = torch.stack([(i - K[0][2]) / K[0][0], -(j - K[1][2]) / K[1][1], -torch.ones_like(i)], -1)      # h,w,3
        dx = (rays_d[:, :-1, :] - rays_d[:, 1:, :]).norm(dim=-1, keepdim=True)
        dx = torch.cat([dx, dx[:, -2:-1, :]], 1)
        dy = (rays_d[:-1, :, :] - rays_d[1:, :, :]).norm(dim=-1, keepdim=True)
        dy = torch.cat([dy, dy[-2:-1, :, :]], 0)
        radiis = torch.sqrt(dx * dy / torch.pi).reshape(-1, 1)
        rays_d = rays_d.reshape(-1, 3)
        rays_cos = 1 / rays_d.norm(dim=-1, keepdim=True)
        rays_o = pose[:3, -1].expand(rays_d.shape[0], 3).contiguous()
        rays_d = torch.sum(rays_d[..., None, :] * pose[:3, :3], -1)
        return {'rays_o': rays_o, 'rays_d': rays_d, 'dirs': F.normalize(rays_d, dim=-1), 'radiis': radiis, 'rays_cos': rays_cos}

    @torch.no_grad()
    def nvs(self, pose, K, h, w, step=300000, rank=0, world=1, perturb_overwrite=-1):
        """Forward-only rendering of a full h x w image in `test_ray_num` chunks (reference shapeRenderer.py:569-668).
        With world > 1 (BASELINE config 5) rank r renders pixels r, r+world, ... (a strided split balances object and
        background pixels over the ranks) and the results are all-gathered back into pixel order; every rank returns the full image.  Returns [h,w,C] numpy arrays
        'color', 'normal', 'acc' (+ 'radiance' when the radiance field is on): the channels the fused compositor produces."""
        from .dist import interleaved_ids, gather_interleaved
        rays = self.image_rays(pose, K, h, w, self.device)
        rn = h * w
        if world > 1:
            ids = interleaved_ids(rn, rank, world, self.device)
            rays = {k: v[ids] for k, v in rays.items()}
        n_loc = rays['rays_o'].shape[0]
        trn = self.cfg['test_ray_num']
        keys = {'color': 'ray_rgb', 'normal': 'normal', 'acc': 'acc'}
        if self.cfg['has_radiance_field'] and step > self.cfg['radiance_field_step']:
            keys['radiance'] = 'radiance'
        chunks = {k: [] for k in keys}
        for r0 in range(0, n_loc, trn):
            cur = {k: v[r0:r0 + trn] for k, v in rays.items()}
            near, far = near_far_from_sphere(cur['rays_o'], cur['rays_d'], float(self.radius))
            out = self.render(cur, near, far, None, perturb_overwrite=perturb_overwrite, is_train=False, step=step)   # as :646
            for k, src in keys.items():
                chunks[k].append(out[src])
        res = {}
        for k in keys:
            local = torch.cat(chunks[k], 0) if chunks[k] else torch.zeros(0, 1, device=self.device)
            full = gather_interleaved(local, rn) if world > 1 else local
            res[k] = full.reshape(h, w, -1).cpu().numpy()
        return res

    # ---- mesh export (the reference's NeRO-derived extract_fields / extract_geometry, used by extract_mesh.py) ---------------
    EXTRACT_SLAB_POINTS = 1 << 24          # lattice points per field-evaluation slab (bounds the temporary xyz to 192 MB)

    def _extract_axes(self, bound_min, bound_max, R: int):
        lo = torch.as_tensor(bound_min, dtype=torch.float32).reshape(3).cpu()
        hi = torch.as_tensor(bound_max, dtype=torch.float32).reshape(3).cpu()
        return [torch.linspace(float(lo[a]), float(hi[a]), R).to(self.device) for a in range(3)]

    def _extract_values(self, pts: torch.Tensor) -> torch.Tensor:
        """the lattice value at points [N,3]: the SDF-only query, +1.0 where ||x|| >= 1"""
        val = self.sdf_network.sdf(pts, None).reshape(-1)
        return torch.where(torch.norm(pts, dim=-1) >= 1.0, torch.ones_like(val), val)

    @torch.no_grad()
    def extract_fields(self, bound_min, bound_max, resolution: int) -> torch.Tensor:
        """u [R,R,R] fp32 on the device: TensoSDF.sdf(x, None) on the lattice linspace(bound_min[a], bound_max[a], R) per axis
        (z fastest), +1.0 (the outside value) where ||x|| >= 1.  Evaluated in slabs of x-planes."""
        if torch.device(self.device).type != 'cuda':
            raise RuntimeError("extract_fields runs on the CUDA kernels (tensoflow_b200 has no CPU path)")
        R = int(resolution)
        axes = self._extract_axes(bound_min, bound_max, R)
        yy, zz = torch.meshgrid(axes[1], axes[2], indexing='ij')
        yz = torch.stack([yy, zz], -1).reshape(1, R * R, 2)
        u = torch.empty(R, R, R, device=self.device, dtype=torch.float32)
        planes = max(1, self.EXTRACT_SLAB_POINTS // (R * R))
        for i0 in range(0, R, planes):
            xs = axes[0][i0:i0 + planes]
            pts = torch.cat([xs[:, None, None].expand(-1, R * R, 1), yz.expand(xs.shape[0], -1, -1)], -1).reshape(-1, 3)
            u[i0:i0 + xs.shape[0]] = self._extract_values(pts).reshape(xs.shape[0], R, R)
        return u

    @torch.no_grad()
    def extract_geometry(self, bound_min, bound_max, resolution: int, threshold: float = 0.0):
        """Zero level set of the SDF as a triangle mesh -> (vertices [V,3] world fp32, triangles [T,3] int32) on the device,
        winding out of the object, vertices rescaled as v / (R - 1) * (bound_max - bound_min) + bound_min.
        `MaterialRenderer(cfg, *shape.extract_geometry(...))` takes it.  Below 2^31 lattice points (R <= 1290): marching
        cubes (tensoflow_b200.isosurface) on extract_fields.  From there up to R = 4096, where the dense volume no longer fits
        the kernels' indices: the narrow band (marching_cubes_narrowband) on the same lattice values, which evaluates the
        field only in bricks around the surface and gives the dense mesh wherever its band rule captures the surface."""
        from .isosurface import marching_cubes, marching_cubes_narrowband
        R = int(resolution)
        if R ** 3 < 2 ** 31:
            verts, tris = marching_cubes(self.extract_fields(bound_min, bound_max, R), threshold)
        else:
            if torch.device(self.device).type != 'cuda':
                raise RuntimeError("extract_geometry runs on the CUDA kernels (tensoflow_b200 has no CPU path)")
            verts, tris = marching_cubes_narrowband(self._extract_values, self._extract_axes(bound_min, bound_max, R), threshold)
        lo = torch.as_tensor(bound_min, dtype=torch.float32).reshape(1, 3).to(verts.device)
        hi = torch.as_tensor(bound_max, dtype=torch.float32).reshape(1, 3).to(verts.device)
        return verts / (R - 1.0) * (hi - lo) + lo, tris

    # ---- alpha mask (reference shapeRenderer.py:257-325) --------------------------------------------
    @torch.no_grad()
    def compute_grid_alpha(self, xyz_locs, length):
        if self.alphaMask is not None:
            alpha_mask = self.alphaMask.sample_alpha(xyz_locs) > 0
        else:
            alpha_mask = torch.ones_like(xyz_locs[:, 0], dtype=bool)
        alpha = torch.zeros(xyz_locs.shape[:-1], device=xyz_locs.device)
        if alpha_mask.any():
            x = xyz_locs[alpha_mask]
            sdfs = self.sdf_inter_fun(x)[..., 0]
            near_surf = torch.abs(sdfs) < self.cfg['mul_length'] * length
            inv_s = self.deviation_network(x).clip(1e-6, 1e6)[..., 0]
            prev_cdf = torch.sigmoid((sdfs + length * 0.5) * inv_s)
            next_cdf = torch.sigmoid((sdfs - length * 0.5) * inv_s)
            a = ((prev_cdf - next_cdf + 1e-5) / (prev_cdf + 1e-5)).clip(min=0.0, max=1.0)
            a[near_surf] = 1
            alpha[alpha_mask] = a
        return alpha

    @torch.no_grad()
    def updateAlphaMask(self, gridSize=(128, 128, 128)):
        g = torch.LongTensor(list(gridSize)).to(self.device)
        samples = torch.stack(torch.meshgrid(torch.linspace(0, 1, int(g[0]), device=self.device), torch.linspace(0, 1, int(g[1]), device=self.device),
                                             torch.linspace(0, 1, int(g[2]), device=self.device), indexing='ij'), -1)
        grid_xyz = self.aabb[0] * (1 - samples) + self.aabb[1] * samples
        step_len = torch.mean(self.aabbSize / (g - 1))
        alpha = torch.zeros_like(grid_xyz[..., 0])
        for i in range(int(g[0])):
            alpha[i] = self.compute_grid_alpha(grid_xyz[i].view(-1, 3), step_len).view((int(g[1]), int(g[2])))
        grid_xyz = grid_xyz.transpose(0, 2).contiguous()
        alpha = alpha.clamp(0, 1).transpose(0, 2).contiguous()[None, None]
        alpha = F.max_pool3d(alpha, kernel_size=3, padding=1, stride=1).view(list(gridSize)[::-1])
        alpha = (alpha >= self.cfg['alphaMask_thres']).float()
        self.alphaMask = AlphaGridMask(self.device, self.aabb, alpha)
        valid = grid_xyz[alpha > 0.5]
        return torch.stack((valid.amin(0), valid.amax(0)))
