"""Pure-PyTorch restatement of the shape-stage orchestration: hierarchical NeuS sampling,
render_core with the shading network, occlusion / sparse / hessian / TV losses
(reference network/shapeRenderer.py:676-684, 820-1025, 1027-1103, 1105-1277;
utils/network_utils.py:108-202).

TEST INFRASTRUCTURE ONLY (see oracle/__init__.py).  Pinned to the reference's own
ShapeRenderer.render by tests/test_renderer.py (through oracle/ref_shim.py) and
tests/golden/renderer.npz.
"""
from __future__ import annotations

import torch
import torch.nn as nn
import torch.nn.functional as F

from . import torch_oracle as O
from . import torch_oracle_shader as SH


def near_far_from_sphere(rays_o, dirs, radius=1.0):                          # shapeRenderer.py:676-684
    a = torch.sum(dirs ** 2, dim=-1, keepdim=True)
    b = 2.0 * torch.sum(rays_o * dirs, dim=-1, keepdim=True)
    mid = 0.5 * (-b) / a
    return torch.clamp(mid - radius, min=1e-3), mid + radius


def sample_pdf_det(bins, weights, n_samples):                                # network_utils.py:117-147, det=True
    weights = weights + 1e-5
    pdf = weights / torch.sum(weights, -1, keepdim=True)
    cdf = torch.cat([torch.zeros_like(pdf[..., :1]), torch.cumsum(pdf, -1)], -1)
    u = torch.linspace(0. + 0.5 / n_samples, 1. - 0.5 / n_samples, steps=n_samples, dtype=bins.dtype)
    u = u.expand(list(cdf.shape[:-1]) + [n_samples]).contiguous()
    inds = torch.searchsorted(cdf, u, right=True)
    below = (inds - 1).clamp_min(0)
    above = inds.clamp_max(cdf.shape[-1] - 1)
    cdf_b, cdf_a = torch.gather(cdf, 1, below), torch.gather(cdf, 1, above)
    bin_b, bin_a = torch.gather(bins, 1, below), torch.gather(bins, 1, above)
    denom = cdf_a - cdf_b
    denom = torch.where(denom < 1e-5, torch.ones_like(denom), denom)
    return bin_b + (u - cdf_b) / denom * (bin_a - bin_b)


def sphere_exit(pts, dirs):                                                   # network_utils.py:108-114
    dtx = torch.sum(pts * dirs, dim=-1, keepdim=True)
    xtx = torch.sum(pts ** 2, dim=-1, keepdim=True)
    return -dtx + torch.sqrt(dtx ** 2 - xtx + 1 + 1e-6)


def probe_weights(sdf_fun, inv_s, z, o, d):                                   # network_utils.py:149-170
    pts = z.unsqueeze(-1) * d.unsqueeze(-2) + o.unsqueeze(-2)
    pn, sn = pts.shape[:2]
    sdf = sdf_fun(pts.reshape(-1, 3)).reshape(pn, sn)
    ps, ns, pz, nz = sdf[:, :-1], sdf[:, 1:], z[:, :-1], z[:, 1:]
    mid = (ps + ns) * 0.5
    cosv = (ns - ps) / (nz - pz + 1e-5)
    surf = cosv < 0
    cosv = torch.clamp(cosv, max=0)
    dist = nz - pz
    pc = torch.sigmoid((mid - cosv * dist * 0.5) * inv_s)
    nc = torch.sigmoid((mid + cosv * dist * 0.5) * inv_s)
    alpha = (pc - nc + 1e-5) / (pc + 1e-5) * surf.to(z.dtype)
    w = alpha * torch.cumprod(torch.cat([torch.ones_like(alpha[:, :1]), 1. - alpha + 1e-7], -1), -1)[:, :-1]
    return w


def occlusion_probability(sdf_fun, inv_s, pts, dirs, sn0=64, sn1=16):        # network_utils.py:172-202 + shapeRenderer.py:1052-1053
    out = torch.zeros(pts.shape[0], 1, dtype=pts.dtype)
    inside = torch.norm(pts, dim=-1) < 0.999
    if inside.any():
        p, d = pts[inside], dirs[inside]
        with torch.no_grad():
            z = sphere_exit(p, d) * torch.linspace(0, 1, sn0, dtype=pts.dtype).unsqueeze(0)
            w = probe_weights(sdf_fun, inv_s, z, p, d)
            z_new = sample_pdf_det(z, w, sn1)
            w = probe_weights(sdf_fun, inv_s, z_new, p, d)
        out[inside] = w.sum(-1, keepdim=True)
    return out


def surface_refine(field, inv_s, rays_o, rays_d, m_depth, unit_size, radius, sn0=32, sn1=9):
    """MaterialRenderer.get_intersection_around_mesh + the tail of trace_sdf_with_mesh (materialRenderer.py:281-343) for rays
    that hit the mesh at depth m_depth [pn,1]: NeuS weights on sn0 samples within +-4 voxels, sn1 deterministic importance samples,
    depth = weighted mean of their mid-points, normal = normalised FD gradient flipped against the ray.
    -> (depth [pn,1], points [pn,3], normals [pn,3])"""
    with torch.no_grad():
        sdf_fun = lambda x: field.sdf(x, None).reshape(-1)
        near, far = near_far_from_sphere(rays_o, rays_d, radius)
        t_min = torch.minimum(torch.maximum(m_depth - unit_size * 4, near), far)
        t_max = torch.minimum(torch.maximum(m_depth + unit_size * 4, near), far)
        z = t_min + (t_max - t_min) * torch.linspace(0.0, 1.0, sn0, dtype=rays_o.dtype)[None, :]
        w = probe_weights(sdf_fun, inv_s, z, rays_o, rays_d)
        z_new = sample_pdf_det(z, w, sn1)
        w = probe_weights(sdf_fun, inv_s, z_new, rays_o, rays_d)
        z_mid = (z_new[:, 1:] + z_new[:, :-1]) * 0.5
        w = w / torch.sum(w, dim=-1, keepdim=True)
        w = torch.where(torch.isnan(w), torch.full_like(w, 1.0 / (sn1 - 1)), w)
        depth = torch.sum(w * z_mid, -1, keepdim=True)
        pts = rays_o + depth * rays_d
    g, _ = field.gradient(pts, None)
    n = F.normalize(g.detach(), dim=-1)
    n = torch.where((n * rays_d).sum(-1, keepdim=True) >= 0, -n, n)
    return depth, pts, n


class ShapeRenderer(nn.Module):
    def __init__(self, gridSize, sdf_n_comp=16, sdf_dim=128, app_dim=128, max_levels=1, has_radiance_field=False,
                 radiance_field_step=0, n_samples=64, n_importance=64, up_sample_steps=4, clip_sample_variance=True,
                 occ_loss_step=20000, occ_loss_max_pn=2048, occ_sdf_thresh=0.01, inv_s_init=0.3, env_res=128, env_min_res=16,
                 dtype=torch.float32):
        super().__init__()
        aabb = [[-1.0] * 3, [1.0] * 3]
        self.sdf_network = O.TensoSDF(gridSize, aabb, sdf_n_comp=sdf_n_comp, sdf_dim=sdf_dim, app_dim=app_dim,
                                      init_n_levels=max_levels, dtype=dtype)
        self.deviation_network = nn.Module()
        self.deviation_network.register_parameter('variance', nn.Parameter(torch.tensor(inv_s_init, dtype=dtype)))
        self.color_network = SH.ShapeShadingNetwork(app_dim, has_radiance_field, env_res=env_res, env_min_res=env_min_res, dtype=dtype)
        self.cfg = dict(n_samples=n_samples, n_importance=n_importance, up_sample_steps=up_sample_steps,
                        clip_sample_variance=clip_sample_variance, occ_loss_step=occ_loss_step, occ_loss_max_pn=occ_loss_max_pn,
                        occ_sdf_thresh=occ_sdf_thresh, has_radiance_field=has_radiance_field, radiance_field_step=radiance_field_step)

    @property
    def aabb(self):
        return self.sdf_network.aabb

    @property
    def base_radii(self):                                                     # shapeRenderer.py:251
        f = self.sdf_network
        return (f.aabb[1, 0] - f.aabb[0, 0]) / 2.0 / f.gridSize[0]

    def inv_s(self):
        return torch.exp(self.deviation_network.variance * 10.0)

    def _upsample(self, o, d, z, sdf, n_imp, inv_s):                          # shapeRenderer.py:820-849
        pts = o[:, None, :] + d[:, None, :] * z[..., :, None]
        radius = torch.linalg.norm(pts, ord=2, dim=-1)
        inside = (radius[:, :-1] < 1.0) | (radius[:, 1:] < 1.0)
        ps, ns, pz, nz = sdf[:, :-1], sdf[:, 1:], z[:, :-1], z[:, 1:]
        mid = (ps + ns) * 0.5
        cosv = (ns - ps) / (nz - pz + 1e-5)
        prev = torch.cat([torch.zeros_like(cosv[:, :1]), cosv[:, :-1]], dim=-1)
        cosv = torch.minimum(prev, cosv).clip(-1e3, 0.0) * inside
        dist = nz - pz
        pc = torch.sigmoid((mid - cosv * dist * 0.5) * inv_s)
        nc = torch.sigmoid((mid + cosv * dist * 0.5) * inv_s)
        alpha = (pc - nc + 1e-5) / (pc + 1e-5)
        w = alpha * torch.cumprod(torch.cat([torch.ones_like(alpha[:, :1]), 1. - alpha + 1e-7], -1), -1)[:, :-1]
        return sample_pdf_det(z, w, n_imp).detach()

    def sample_ray(self, o, d, near, far, radiis, rays_cos, t_rand=None, rounds=None):     # shapeRenderer.py:871-932
        """rounds: optional list; (t, sdf) of the depth lists is appended to it after the coarse samples and after every
        upsampling round (sdf None after the last round, whose SDF the reference does not query).  The return value does
        not depend on it."""
        c = self.cfg
        f = self.sdf_network
        ns = c['n_samples']
        vec = torch.where(d == 0, torch.full_like(d, 1e-6), d)
        ra, rb = (f.aabb[1] - o) / vec, (f.aabb[0] - o) / vec
        t_min = torch.minimum(ra, rb).amax(-1).clamp(min=near[..., 0], max=far[..., 0]).unsqueeze(-1)
        t_max = torch.maximum(ra, rb).amin(-1).clamp(min=near[..., 0], max=far[..., 0]).unsqueeze(-1)
        t = t_min + (t_max - t_min) * torch.linspace(0.0, 1.0, ns, dtype=o.dtype)[None, :]
        if t_rand is not None:
            t = t + (t_rand - 0.5) * 2.0 / ns
        with torch.no_grad():
            pts = o[:, None, :] + d[:, None, :] * t[..., :, None]
            lvl = torch.log2(O.compute_ball_radii(t[..., :, None], radiis[:, None, :], rays_cos[:, None, :]) / self.base_radii)
            sdf = f.sdf(pts.reshape(-1, 3), lvl.reshape(-1, 1)).reshape(t.shape)
            if rounds is not None:
                rounds.append((t.detach().clone(), sdf.clone()))
            for i in range(c['up_sample_steps']):
                if c['clip_sample_variance']:
                    inv_s = torch.clamp(self.inv_s(), max=64 * 2 ** i)
                else:
                    inv_s = 64.0 * 2 ** i
                new_t = self._upsample(o, d, t, sdf, c['n_importance'] // c['up_sample_steps'], inv_s)
                t_all, index = torch.sort(torch.cat([t, new_t], dim=-1), dim=-1)
                if i + 1 != c['up_sample_steps']:
                    pts = o[:, None, :] + d[:, None, :] * new_t[..., :, None]
                    lvl = torch.log2(O.compute_ball_radii(new_t[..., None], radiis[..., None, :], rays_cos[..., None, :]) / self.base_radii)
                    new_sdf = f.sdf(pts.reshape(-1, 3), lvl.reshape(-1, 1)).reshape(new_t.shape)
                    sdf = torch.gather(torch.cat([sdf, new_sdf], dim=-1), 1, index)
                t = t_all
                if rounds is not None:
                    rounds.append((t.detach().clone(), sdf.clone() if i + 1 != c['up_sample_steps'] else None))
        dists = t[..., 1:] - t[..., :-1]
        dists = torch.cat([dists, dists[..., -1:]], -1)
        mid = t + dists * 0.5
        idx = torch.arange(o.shape[0])[:, None].expand(-1, t.shape[1])
        pts = o.unsqueeze(-2) + d.unsqueeze(-2) * mid.unsqueeze(-1)
        inner = ~((f.aabb[0] > pts) | (pts > f.aabb[1])).any(dim=-1)
        return t[inner], (t + dists)[inner], idx[inner]

    def render(self, rays_o, dirs, radiis, rays_cos, near, far, cos_anneal_ratio, step, t_rand=None):
        c = self.cfg
        f = self.sdf_network
        ts, te, idx = self.sample_ray(rays_o, dirs, near, far, radiis, rays_cos, t_rand)
        n_rays = rays_o.shape[0]
        mid, dists = (ts + te) * 0.5, te - ts
        vd = dirs[idx]
        pts = rays_o[idx] + vd * mid[:, None]
        lvl = torch.log2(O.compute_ball_radii(mid[:, None], radiis[idx], rays_cos[idx]) / self.base_radii)
        out = f(pts, lvl)
        sdf, feat = out[..., 0], out[..., 1:]
        grads, hess = f.gradient(pts, lvl, training=True, sdf=sdf[..., None])
        alpha, inv_s = O.neus_alpha(sdf, grads, dists, vd, self.deviation_network.variance, cos_anneal_ratio)
        normals = F.normalize(grads, dim=-1)
        with_rad = c['has_radiance_field'] and step > c['radiance_field_step']
        color, radiance, occ = self.color_network(pts, normals, -vd, feat, with_radiance=with_rad)
        w, _ = O.render_weight_from_alpha(alpha, idx, n_rays)
        acc = O.accumulate_along_rays(w, None, idx, n_rays)
        res = {
            'ray_rgb': O.accumulate_along_rays(w, color, idx, n_rays) + (1 - acc), 'acc': acc,
            'gradient_error': (torch.linalg.norm(grads, ord=2, dim=-1) - 1.0) ** 2,
            'loss_sparse': torch.exp(-20. * sdf.abs()).mean(), 'loss_hessian': hess.abs().mean(),
            'std': torch.mean(1 / inv_s.clip(1e-6, 1e6)), 'sample_num': idx.shape[0] / n_rays,
            'loss_tv_sdf': f.TV_loss_sdf(O.tv_loss),
        }
        nrm = O.accumulate_along_rays(w, grads, idx, n_rays)
        res['normal'] = F.normalize(nrm * acc + (1. - acc) * torch.tensor([0.0, 0.0, 1.0], dtype=nrm.dtype), dim=-1)
        if with_rad:
            res['radiance'] = O.accumulate_along_rays(w, radiance, idx, n_rays) + (1 - acc)
            res['roughness_weights'] = O.accumulate_along_rays(w, occ['roughness'], idx, n_rays).squeeze(-1).detach()
        # occlusion loss (shapeRenderer.py:1027-1103, non-occ-grid branch)
        if step >= c['occ_loss_step']:
            inner = ~((f.aabb[0] > pts) | (pts > f.aabb[1])).any(dim=-1)
            mask = inner & (torch.sum(normals * vd, -1) < 0) & (torch.abs(sdf) < c['occ_sdf_thresh'])
            assert int(mask.sum()) <= c['occ_loss_max_pn'], "oracle has no random subsampling: raise occ_loss_max_pn"
            if mask.any():
                gt = occlusion_probability(lambda x: f.sdf(x, None)[..., 0], self.inv_s(), pts[mask].detach(),
                                           occ['reflective'][mask].detach())
                res['loss_occ'] = F.l1_loss(occ['occ_prob'][mask], gt)
            else:
                res['loss_occ'] = torch.zeros(1, dtype=pts.dtype)
        else:
            res['loss_occ'] = torch.zeros(1, dtype=pts.dtype)
        res.update({'_sdf': sdf, '_alpha': alpha, '_weights': w})
        return res


def alpha_mask_sample(alpha_volume, aabb, xyz_sampled):
    """AlphaGridMask.sample_alpha (network/shapeRenderer.py:79-97): alpha_volume [D,H,W], aabb [2,3], xyz [N,3] -> [N]."""
    aabb_size = aabb[1] - aabb[0]
    inv = 1.0 / aabb_size * 2
    xyz = (xyz_sampled - aabb[0]) * inv - 1
    vol = alpha_volume.view(1, 1, *alpha_volume.shape[-3:])
    return F.grid_sample(vol, xyz.view(1, -1, 1, 1, 3), align_corners=True).view(-1)
