"""Shape-stage shader (reference network/fields.py:320-575 ShapeShadingNetwork) and its
prefiltered environment light (reference network/light.py:8-122).

The MLP heads (material / indirect light / occlusion / radiance) run on the fused linear kernels, the cubemap prefilter on
the cached CSR operator kernel, the per-sample encodings and the combine on the tf_shader_* kernels, and the
(direction- and level-differentiable) cube lookups on tf_cube_sample_*.
"""
from __future__ import annotations

import ctypes as C
import math
import os
from typing import Dict, List, Optional, Tuple

import numpy as np
import torch
import torch.nn as nn
import torch.nn.functional as F

from . import _lib, ops
from ._lib import check, ptr, stream_ptr
from .flow import posenc
from .material import make_predictor, run_predictor, run_predictor_padded, linear_to_srgb, _ide_device_tables


# ---- cube geometry (reference network/light_utils.py:24-31, renderutils/c_src/cubemap.cu:32-60) ----
def cube_to_dir_t(face: torch.Tensor, x: torch.Tensor, y: torch.Tensor) -> torch.Tensor:
    one = torch.ones_like(x)
    opts = [(one, -y, -x), (-one, -y, x), (x, one, y), (x, -one, -y), (x, -y, one), (-x, -y, -one)]
    out = torch.stack(opts[5], -1)
    for s in range(4, -1, -1):
        out = torch.where((face == s).unsqueeze(-1), torch.stack(opts[s], -1), out)
    return out


class CubeSampleFunction(torch.autograd.Function):
    """Seamless (tri)linear cube lookup on `tf_cube_sample_fwd/bwd`, differentiable in the textures, the direction and the level:
    (d [N,3], level [N] or None, *texs [6,R_l,R_l,3]) -> [N,3]."""

    @staticmethod
    def forward(ctx, d, level, *texs):
        import ctypes as C
        lib = _lib.load()
        d_c = d.detach().float().contiguous()
        lv = None if level is None else level.detach().float().contiguous().reshape(-1)
        tex_c = [t.detach().float().contiguous() for t in texs]
        n, L = d_c.shape[0], len(tex_c)
        out = torch.empty(n, 3, device=d_c.device, dtype=torch.float32)
        ptrs = (C.c_void_p * L)(*[t.data_ptr() for t in tex_c])
        res = (C.c_int32 * L)(*[int(t.shape[1]) for t in tex_c])
        check(lib.tf_cube_sample_fwd(ptrs, res, L, ptr(d_c), ptr(lv), n, ptr(out), stream_ptr()), "tf_cube_sample_fwd")
        ctx.save_for_backward(d_c, lv, *tex_c)
        ctx.has_level = level is not None
        return out

    @staticmethod
    def backward(ctx, g):
        import ctypes as C
        lib = _lib.load()
        d_c, lv, *tex_c = ctx.saved_tensors
        n, L = d_c.shape[0], len(tex_c)
        g_c = g.detach().float().contiguous()
        need_tex = [ctx.needs_input_grad[2 + l] for l in range(L)]
        d_tex = [torch.zeros_like(t) if need else None for t, need in zip(tex_c, need_tex)]
        d_d = torch.empty_like(d_c) if ctx.needs_input_grad[0] else None
        d_lv = torch.empty(n, device=d_c.device, dtype=torch.float32) if (ctx.has_level and ctx.needs_input_grad[1]) else None
        ptrs = (C.c_void_p * L)(*[t.data_ptr() for t in tex_c])
        dptrs = (C.c_void_p * L)(*[(t.data_ptr() if t is not None else None) for t in d_tex])
        res = (C.c_int32 * L)(*[int(t.shape[1]) for t in tex_c])
        check(lib.tf_cube_sample_bwd(ptrs, res, L, ptr(d_c), ptr(lv), n, ptr(g_c), dptrs, ptr(d_d), ptr(d_lv), stream_ptr()),
              "tf_cube_sample_bwd")
        return (d_d, d_lv, *d_tex)


def cube_lookup(texs: List[torch.Tensor], d: torch.Tensor, level: Optional[torch.Tensor] = None) -> torch.Tensor:
    """The product path of the cube lookups (CUDA kernel; no CPU fallback)."""
    if d.shape[0] == 0:
        return torch.zeros(0, 3, device=d.device)
    return CubeSampleFunction.apply(d, level, *texs)


def texture2d_linear_clamp(tex: torch.Tensor, uv: torch.Tensor) -> torch.Tensor:
    """dr.texture(tex[None], uv, filter_mode='linear', boundary_mode='clamp') (reference fields.py:522):
    tex [H,W,C], uv [N,2]; differentiable in uv."""
    H, W, _ = tex.shape
    x, y = uv[:, 0] * W - 0.5, uv[:, 1] * H - 0.5
    x0, y0 = torch.floor(x), torch.floor(y)
    fx, fy = (x - x0).unsqueeze(-1), (y - y0).unsqueeze(-1)
    x0i, x1i = x0.long().clamp(0, W - 1), (x0.long() + 1).clamp(0, W - 1)
    y0i, y1i = y0.long().clamp(0, H - 1), (y0.long() + 1).clamp(0, H - 1)
    return (tex[y0i, x0i] * (1 - fx) * (1 - fy) + tex[y0i, x1i] * fx * (1 - fy)
            + tex[y1i, x0i] * (1 - fx) * fy + tex[y1i, x1i] * fx * fy)


# ---- cubemap prefilter operators (reference renderutils/c_src/cubemap.cu:17-60,110-350) ----------------
def _texel_dirs(N, device):
    c = 2.0 * ((torch.arange(N, device=device, dtype=torch.float32) + 0.5) / N) - 1.0
    fy, fx = torch.meshgrid(c, c, indexing="ij")
    face = torch.arange(6, device=device)[:, None, None].expand(6, N, N)
    return F.normalize(cube_to_dir_t(face, fx.expand(6, N, N), fy.expand(6, N, N)), dim=-1).reshape(-1, 3)


def _pixel_area(N, device):
    if N <= 1:
        return torch.ones(6, device=device)
    H = N // 2
    i = (torch.arange(N, device=device) - H).abs().float()
    dx = torch.atan((i + 1) / H) - torch.atan(i / H)
    return (dx[None, :] * dx[:, None]).reshape(1, -1).repeat(6, 1).reshape(-1)


def _ndf_cutoff(roughness: float, cutoff: float) -> float:
    """reference renderutils/ops.py:427-438"""
    a2 = roughness ** 4
    ct = np.cos(np.linspace(0, np.pi / 2.0, 1000000))
    c = np.clip(ct, 0.0, 1.0)
    dd = (c * a2 - c) * c + 1.0
    D = np.cumsum(a2 / (dd * dd * np.pi))
    return float(ct[np.argmax(D >= D[-1] * cutoff)])


class PrefilterOp:
    """CSR operator of one prefilter pass, built once per (res, kind, roughness, cutoff)."""
    _cache: Dict[Tuple, "PrefilterOp"] = {}

    def __init__(self, res: int, kind: str, roughness: float, cutoff: float, device, chunk: int = 4096):
        dirs = _texel_dirs(res, device)
        area = _pixel_area(res, device)
        rows, cols, vals = [], [], []
        if kind == "specular":
            cos_cut = _ndf_cutoff(roughness, cutoff)
            a2 = (roughness * roughness) ** 2
        for i in range(0, dirs.shape[0], chunk):
            V = dirs[i:i + chunk]
            LdV = V @ dirs.T
            if kind == "diffuse":
                w = LdV.clamp(0.0, 0.999) * area[None, :] / 3.141592
                keep = w > 0
            else:
                Hh = F.normalize(dirs[None, :, :] + V[:, None, :], dim=-1, eps=1e-20)
                VdH = (Hh * V[:, None, :]).sum(-1).clamp(0.0, 1.0)
                dd = (VdH * a2 - VdH) * VdH + 1.0
                w = LdV.clamp_min(0.0) * (a2 / (dd * dd * math.pi)) * area[None, :] / 4.0
                keep = LdV >= cos_cut
                w = torch.where(keep, w, torch.zeros_like(w))
                w = w / w.sum(-1, keepdim=True)
            r, c = torch.nonzero(keep, as_tuple=True)
            rows.append(r + i); cols.append(c); vals.append(w[r, c])
        rows, cols, vals = torch.cat(rows), torch.cat(cols), torch.cat(vals)
        n = dirs.shape[0]
        counts = torch.bincount(rows, minlength=n)
        self.rowptr = torch.cat([torch.zeros(1, dtype=torch.long, device=device), torch.cumsum(counts, 0)]).to(torch.int32)
        self.col = cols.to(torch.int32).contiguous()
        self.val = vals.float().contiguous()
        self.n = n

    @classmethod
    def get(cls, res, kind, roughness, cutoff, device):
        key = (res, kind, float(roughness), float(cutoff), str(device))
        if key not in cls._cache:
            cls._cache[key] = PrefilterOp(res, kind, roughness, cutoff, device)
        return cls._cache[key]


class PrefilterFunction(torch.autograd.Function):
    @staticmethod
    def forward(ctx, cubemap, op: PrefilterOp):
        x = cubemap.detach().contiguous().reshape(-1, 3)
        y = torch.empty_like(x)
        check(_lib.load().tf_csr_spmm3_fwd(ptr(op.rowptr), ptr(op.col), ptr(op.val), ptr(x), op.n, ptr(y), stream_ptr()), "tf_csr_spmm3_fwd")
        ctx.op = op
        return y.reshape(cubemap.shape)

    @staticmethod
    def backward(ctx, g):
        op = ctx.op
        gy = g.contiguous().reshape(-1, 3)
        gx = torch.zeros_like(gy)
        check(_lib.load().tf_csr_spmm3_bwd(ptr(op.rowptr), ptr(op.col), ptr(op.val), ptr(gy), op.n, ptr(gx), stream_ptr()), "tf_csr_spmm3_bwd")
        return gx.reshape(g.shape), None


def diffuse_cubemap(cubemap):
    return PrefilterFunction.apply(cubemap, PrefilterOp.get(cubemap.shape[1], "diffuse", 0.0, 0.0, cubemap.device))


def specular_cubemap(cubemap, roughness, cutoff=0.99):
    return PrefilterFunction.apply(cubemap, PrefilterOp.get(cubemap.shape[1], "specular", roughness, cutoff, cubemap.device))


class CubemapMip(torch.autograd.Function):
    """reference network/light_utils.py:66-82: 2x2 average pool forward; the backward is a seamless
    bilinear cube lookup of dout/4 at the fine texel centres (kept as the reference defines it)."""

    @staticmethod
    def forward(ctx, cubemap):
        return F.avg_pool2d(cubemap.permute(0, 3, 1, 2), (2, 2)).permute(0, 2, 3, 1).contiguous()

    _dirs = {}      # res, device -> the normalised fine texel centre directions: constant geometry, built once

    @staticmethod
    def backward(ctx, dout):
        res = dout.shape[1] * 2
        key = (res, str(dout.device))
        if key not in CubemapMip._dirs:
            CubemapMip._dirs[key] = _texel_dirs(res, dout.device)
        return cube_lookup([dout * 0.25], CubemapMip._dirs[key]).reshape(6, res, res, -1)


class ShadingEnvLight(nn.Module):
    """reference network/light.py:8-122 (the prefiltered split-sum light of the shape stage)"""

    def __init__(self, device='cuda', min_res=16, max_res=128, min_roughness=0.08, max_roughness=0.5, trainable=True):
        super().__init__()
        self.min_res, self.max_res = min_res, max_res
        self.min_roughness, self.max_roughness = min_roughness, max_roughness
        self.base = nn.Parameter(torch.full((6, max_res, max_res, 3), math.log(0.5), dtype=torch.float32, device=device),
                                 requires_grad=trainable)

    def build_mips(self, cutoff=0.99):
        self.specular = [self.base]
        while self.specular[-1].shape[1] > self.min_res:
            self.specular.append(CubemapMip.apply(self.specular[-1]))
        self.diffuse = diffuse_cubemap(self.specular[-1])
        n = len(self.specular)
        for idx in range(n - 1):
            r = (idx / (n - 2)) * (self.max_roughness - self.min_roughness) + self.min_roughness
            self.specular[idx] = specular_cubemap(self.specular[idx], r, cutoff)
        self.specular[-1] = specular_cubemap(self.specular[-1], 1.0, cutoff)

    def get_mip(self, roughness):
        n = len(self.specular)
        lo = (torch.clamp(roughness, self.min_roughness, self.max_roughness) - self.min_roughness) / \
            (self.max_roughness - self.min_roughness) * (n - 2)
        hi = (torch.clamp(roughness, self.max_roughness, 1.0) - self.max_roughness) / (1.0 - self.max_roughness) + n - 2
        return torch.where(roughness < self.max_roughness, lo, hi)

    def forward(self, l, roughness=None):
        if roughness is None:
            return torch.exp(cube_lookup([self.diffuse], l))
        return torch.exp(cube_lookup(self.specular, l, self.get_mip(roughness)[..., 0]))


class ShaderEncodeFunction(torch.autograd.Function):
    """Normalised normal / view, mirror direction, N.V, roughness and the zero-padded inputs of the radiance, indirect-light
    and occlusion heads (reference fields.py:453-501) in one kernel; backward in one kernel (IDE / mirror / normalisation
    adjoints).  (points, normals, view_dirs, mat [N,5], feat [N,fd] or None) ->
    (nrm [N,3], vdir [N,3], refl [N,3], nov [N], rough [N], X_rad [N,ld] or None, X_il [N,128], X_iw [N,96])"""

    @staticmethod
    def forward(ctx, points, normals, view_dirs, mat, feat):
        lib = _lib.load()
        pc, nc, vc, mc, fc = (ops._f32c(t) for t in (points, normals, view_dirs, mat, feat))
        n, dev = pc.shape[0], pc.device
        fd = 0 if fc is None else int(fc.shape[1])
        ld_rad = 0 if fc is None else (fd + 33 + 15) // 16 * 16
        ide = _ide_device_tables(dev)
        f32 = dict(device=dev, dtype=torch.float32)
        nrm, vdir, refl = torch.empty(n, 3, **f32), torch.empty(n, 3, **f32), torch.empty(n, 3, **f32)
        nov, rough = torch.empty(n, **f32), torch.empty(n, **f32)
        X_rad = None if fc is None else torch.empty(n, ld_rad, **f32)
        X_il, X_iw = torch.empty(n, 128, **f32), torch.empty(n, 96, **f32)
        with ops._timed("shader_encode_fwd"):
            check(lib.tf_shader_encode_fwd(ptr(pc), ptr(nc), ptr(vc), ptr(mc), ptr(fc), fd, ld_rad, n, ptr(ide[0]), ptr(ide[1]), ptr(ide[2]),
                                           ptr(nrm), ptr(vdir), ptr(refl), ptr(nov), ptr(rough), ptr(X_rad), ptr(X_il), ptr(X_iw), stream_ptr()),
                  "tf_shader_encode_fwd")
        ctx.save_for_backward(nc, vc, mc)
        ctx.dims = (fd, ld_rad, feat is not None)
        ctx.mark_non_differentiable(vdir, X_iw)
        ctx.set_materialize_grads(False)
        return nrm, vdir, refl, nov, rough, X_rad, X_il, X_iw

    @staticmethod
    def backward(ctx, g_nrm, _g_vdir, g_refl, g_nov, g_rough, g_Xrad, g_Xil, _g_Xiw):
        lib = _lib.load()
        nc, vc, mc = ctx.saved_tensors
        fd, ld_rad, has_feat = ctx.dims
        n, dev = nc.shape[0], nc.device
        ide = _ide_device_tables(dev)
        gs = [ops._f32c(g) for g in (g_nrm, g_refl, g_nov, g_rough, g_Xrad, g_Xil)]
        d_normals = torch.empty(n, 3, device=dev, dtype=torch.float32)
        d_mat = torch.zeros(n, 5, device=dev, dtype=torch.float32)
        d_mat3 = torch.empty(n, device=dev, dtype=torch.float32)
        d_feat = None
        if has_feat:
            d_feat = torch.empty(n, fd, device=dev, dtype=torch.float32) if gs[4] is not None else torch.zeros(n, fd, device=dev, dtype=torch.float32)
        with ops._timed("shader_encode_bwd"):
            check(lib.tf_shader_encode_bwd(ptr(nc), ptr(vc), ptr(mc), fd, ld_rad, n, ptr(ide[0]), ptr(ide[1]), ptr(ide[2]), *(ptr(g) for g in gs),
                                           ptr(d_normals), ptr(d_mat3), ptr(d_feat) if gs[4] is not None else None, stream_ptr()),
                  "tf_shader_encode_bwd")
        d_mat[:, 3] = d_mat3
        return None, d_normals, None, d_mat, d_feat


class ShaderCombineFunction(torch.autograd.Function):
    """Material affine maps + split-sum FG LUT + diffuse / specular combination with the occlusion blend + linear->sRGB + clamp
    (reference fields.py:463-531) in one kernel each way.
    (mat [N,5], diffuse_light, direct_light, indirect_light [N,3], w_raw [N], nov [N], lut [H,W,2]) -> color [N,3], occ_prob [N]"""

    @staticmethod
    def forward(ctx, mat, diffuse_light, direct_light, indirect_light, w_raw, nov, lut):
        lib = _lib.load()
        t = [ops._f32c(x) for x in (mat, diffuse_light, direct_light, indirect_light, w_raw.reshape(-1), nov.reshape(-1), lut)]
        n, dev = t[0].shape[0], t[0].device
        color = torch.empty(n, 3, device=dev, dtype=torch.float32)
        occ = torch.empty(n, device=dev, dtype=torch.float32)
        with ops._timed("shader_combine_fwd"):
            check(lib.tf_shader_combine_fwd(*(ptr(x) for x in t), int(t[6].shape[0]), int(t[6].shape[1]), n, ptr(color), ptr(occ), stream_ptr()),
                  "tf_shader_combine_fwd")
        ctx.save_for_backward(*t)
        ctx.shapes = (w_raw.shape, nov.shape)
        ctx.set_materialize_grads(False)
        return color, occ

    @staticmethod
    def backward(ctx, g_color, g_occ):
        lib = _lib.load()
        t = list(ctx.saved_tensors)
        n, dev = t[0].shape[0], t[0].device
        gc = ops._f32c(g_color) if g_color is not None else torch.zeros(n, 3, device=dev, dtype=torch.float32)
        go = None if g_occ is None else ops._f32c(g_occ.reshape(-1))
        f32 = dict(device=dev, dtype=torch.float32)
        d_mat, d_dif, d_dir, d_ind = torch.empty(n, 5, **f32), torch.empty(n, 3, **f32), torch.empty(n, 3, **f32), torch.empty(n, 3, **f32)
        d_w, d_nov = torch.empty(n, **f32), torch.empty(n, **f32)
        with ops._timed("shader_combine_bwd"):
            check(lib.tf_shader_combine_bwd(*(ptr(x) for x in t), int(t[6].shape[0]), int(t[6].shape[1]), n, ptr(gc), ptr(go), ptr(d_mat), ptr(d_dif),
                                            ptr(d_dir), ptr(d_ind), ptr(d_w), ptr(d_nov), stream_ptr()), "tf_shader_combine_bwd")
        return d_mat, d_dif, d_dir, d_ind, d_w.reshape(ctx.shapes[0]), d_nov.reshape(ctx.shapes[1]), None


def load_fg_lut(device):
    p = os.path.join(os.path.dirname(os.path.abspath(__file__)), "assets", "fg_lut_256.npz")
    return torch.from_numpy(np.load(p)["fg"]).to(device)


class ShapeShadingNetwork(nn.Module):
    default_cfg = {'human_light': False, 'sphere_direction': False, 'light_pos_freq': 8, 'inner_init': -0.95, 'light_exp_max': 0.0,
                   'app_feats_dim': 128, 'has_radiance_field': False, 'radiance_field_step': 0, 'mat_pos_multires': -1,
                   'device': 'cuda', 'env_res': 128, 'env_min_res': 16}

    def __init__(self, cfg):
        super().__init__()
        self.cfg = {**self.default_cfg, **cfg}
        c = self.cfg
        if c['human_light'] or c['mat_pos_multires'] != -1 or c['light_pos_freq'] != 8:
            raise NotImplementedError("tensoflow_b200 implements the shipped shape-shader configuration")
        dev, fd = c['device'], c['app_feats_dim']
        if c['has_radiance_field']:
            self.rad_mlp = make_predictor(3, fd + 3 + 27 + 3, 3, run_dim=128).to(dev)
        self.mat_mlp = make_predictor(3, fd, 5, run_dim=128).to(dev)
        self.register_buffer('FG_LUT', load_fg_lut(dev)[None])
        self.envlight = ShadingEnvLight(device=dev, max_res=c['env_res'], min_res=c['env_min_res'])
        # the reference registers `outer_light` (fields.py:352-358) but its forward never calls it (:422, :444 are commented
        # out): kept as an idle module so that state dicts round-trip with the reference's strict load_state_dict
        self.outer_light = make_predictor(3, 72 * 2 if c['sphere_direction'] else 72, 3, run_dim=128).to(dev)
        nn.init.constant_(self.outer_light[-2].bias, np.log(0.5))
        for p_ in self.outer_light.parameters():
            p_.requires_grad_(False)
        self.inner_light = make_predictor(3, 51 + 72, 3, run_dim=128).to(dev)
        nn.init.constant_(self.inner_light[-2].bias, np.log(0.5))
        self.inner_weight = make_predictor(3, 51 + 39, 1, run_dim=128).to(dev)
        nn.init.constant_(self.inner_weight[-2].bias, c['inner_init'])

    def get_optparam_groups(self, lr_init_network, lr_init_envlight):
        return [{'params': self.envlight.parameters(), 'lr': lr_init_envlight},
                {'params': [p for n, p in self.named_parameters() if 'envlight' not in n], 'lr': lr_init_network}]

    def predict_materials(self, points, feature_vectors):
        mat = run_predictor(self.mat_mlp, feature_vectors, "sigmoid")
        return mat[..., 4:], mat[..., 3:4], mat[..., :3]

    def forward(self, points, normals, view_dirs, feature_vectors, human_poses=None, inter_results=False, step=None):
        c = self.cfg
        with_rad = c['has_radiance_field'] and step is not None and step > c['radiance_field_step']
        dev = points.device
        if points.shape[0] == 0:
            occ_info = {'reflective': torch.zeros(0, 1, device=dev), 'occ_prob': torch.zeros(0, 1, device=dev), 'roughness': torch.zeros(0, 1, device=dev)}
            return torch.zeros(0, 3, device=dev), (torch.zeros(0, 3, device=dev) if with_rad else None), occ_info
        # material head, then the per-sample kernels: encode (normalisation, mirror direction, N.V, roughness, the padded inputs of
        # the three remaining heads) -> heads + environment lookups -> combine (FG LUT, occlusion blend, sRGB)
        fd = feature_vectors.shape[1]
        mat = run_predictor(self.mat_mlp, feature_vectors, "sigmoid")
        normals, view_dirs, reflective, nov, rough, X_rad, X_il, X_iw = ShaderEncodeFunction.apply(
            points, normals, view_dirs, mat, feature_vectors if with_rad else None)
        roughness = rough[:, None]
        radiance = run_predictor_padded(self.rad_mlp, X_rad, fd + 33, "sigmoid") if with_rad else None
        diffuse_light = self.envlight(normals)
        direct_light = self.envlight(reflective, roughness)
        indirect_light = run_predictor_padded(self.inner_light, X_il, 123, "exp", c['light_exp_max'])
        w_raw = run_predictor_padded(self.inner_weight, X_iw, 90, "none")
        color, occ = ShaderCombineFunction.apply(mat, diffuse_light, direct_light, indirect_light, w_raw, nov, self.FG_LUT[0])
        occ_prob = occ[:, None]
        if inter_results:                                        # visualisation outputs of the inference path: plain tensor arithmetic
            albedo, metallic = mat[..., :3] * 0.77 + 0.03, mat[..., 4:]
            NoV = nov[:, None]
            diffuse_albedo = (1 - metallic) * albedo
            diffuse_color = diffuse_albedo * diffuse_light
            specular_albedo = 0.04 * (1 - metallic) + metallic * albedo
            occ_ = torch.clamp(occ_prob, min=0, max=1)
            specular_light = indirect_light * occ_ + direct_light * (1 - occ_)
            indirect = indirect_light * occ_
            fg_uv = torch.cat([torch.clamp(NoV, min=0.0, max=1.0), torch.clamp(roughness, min=0.0, max=1.0)], -1)
            fg = texture2d_linear_clamp(self.FG_LUT[0], fg_uv)
            specular_ref = specular_albedo * fg[:, 0:1] + fg[:, 1:2]
            specular_color = specular_ref * specular_light
        occ_info = {'reflective': reflective, 'occ_prob': occ_prob, 'roughness': roughness}
        if inter_results:
            inter = {
                'specular_albedo': specular_albedo, 'specular_ref': torch.clamp(specular_ref, min=0.0, max=1.0),
                'specular_direct_light': direct_light,
                'specular_light': torch.clamp(linear_to_srgb(specular_light), min=0.0, max=1.0),
                'specular_color': torch.clamp(linear_to_srgb(specular_color), min=0.0, max=1.0),
                'diffuse_albedo': diffuse_albedo, 'diffuse_light': torch.clamp(linear_to_srgb(diffuse_light), min=0.0, max=1.0),
                'diffuse_color': torch.clamp(linear_to_srgb(diffuse_color), min=0.0, max=1.0),
                'metallic': metallic, 'roughness': roughness, 'albedo': albedo,
                'occ_prob': torch.clamp(occ_prob, max=1.0, min=0.0), 'indirect_light': indirect,
            }
            return color, occ_info, inter
        return color, radiance, occ_info
