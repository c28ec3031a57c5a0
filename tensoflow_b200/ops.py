"""torch.autograd.Function layer over the C ABI (include/tensoflow_b200.h).

PyTorch is plumbing here: it owns device memory and streams; all arithmetic of the
hot path runs in the hand-written sm_100a kernels of libtensoflow_b200.so.
"""
from __future__ import annotations

import ctypes as C
from typing import List, Optional, Sequence

import torch

from . import _lib
from ._lib import VMField, VMMut, SdfMlp, SdfMlpGrad, check, ptr, stream_ptr

BWD_WORKSPACE_BYTES = int(__import__('os').environ.get('TF_BWD_WORKSPACE_GIB', '4')) << 30   # upper bound for the stencil-backward scratch


class KernelTimers:
    """Optional CUDA-event timing of the C-ABI calls (bench.py turns it on for the timed
    region; events are recorded on the launching stream)."""
    enabled = False
    events = {}

    @classmethod
    def reset(cls, enabled: bool):
        cls.enabled = enabled
        cls.events = {}

    @classmethod
    def totals_ms(cls):
        return {k: (sum(a.elapsed_time(b) for a, b in v), len(v)) for k, v in cls.events.items()}


class _timed:
    def __init__(self, name):
        self.name = name

    def __enter__(self):
        if KernelTimers.enabled:
            self.a = torch.cuda.Event(enable_timing=True)
            self.b = torch.cuda.Event(enable_timing=True)
            self.a.record()
        return self

    def __exit__(self, *exc):
        if KernelTimers.enabled:
            self.b.record()
            KernelTimers.events.setdefault(self.name, []).append((self.a, self.b))
        return False


def _nhwc(p: torch.Tensor) -> torch.Tensor:
    """[1,C,H,W] parameter -> contiguous [H,W,C] tensor (a view when the parameter is
    stored channels-last, which is how tensoflow_b200 modules hold it)."""
    v = p.detach()[0].permute(1, 2, 0)
    return v if v.is_contiguous() else v.contiguous()


def mip_sizes(h: int, w: int, n_levels: int):
    out = []
    for _ in range(1, n_levels):
        h = h // 2 if h > 1 else 1
        w = w // 2 if w > 1 else 1
        out.append((h, w))
    return out


_GRAD_ALLOCATOR = None


def set_grad_allocator(fn):
    """fn(tensor aliasing a parameter's storage) -> zeroed gradient buffer with the parameter's shape and strides, or None.
    dist.FlatGradBucket installs it for the duration of a backward pass so that the kernels scatter parameter gradients
    straight into the flat allreduce buffer."""
    global _GRAD_ALLOCATOR
    _GRAD_ALLOCATOR = fn


def _grad_zeros(param_like: torch.Tensor) -> torch.Tensor:
    """Zero-initialised gradient buffer shaped / strided like this parameter."""
    if _GRAD_ALLOCATOR is not None:
        v = _GRAD_ALLOCATOR(param_like)
        if v is not None:
            return v
    return torch.zeros_like(param_like, memory_format=torch.preserve_format)


_AABB_CACHE: dict = {}
_VMDESC_CACHE: dict = {}
_PARAM_EPOCH = 0


def bump_param_epoch():
    """Invalidate every cached descriptor / mip chain.  Called by code that rewrites parameters through raw device pointers
    (optim.FusedAdam, which cannot bump the autograd version counters the cache keys rely on)."""
    global _PARAM_EPOCH
    _PARAM_EPOCH += 1
    _VMDESC_CACHE.clear()


def _aabb_floats(aabb: torch.Tensor):
    """The 6 aabb bounds as Python floats; cached per (storage, version) so that a CUDA aabb costs one D2H sync, not one per
    call.  The entry keeps the tensor alive: its storage cannot be freed and handed to another tensor (with another box)
    while the key is live."""
    key = (aabb.data_ptr(), aabb._version, str(aabb.device))
    hit = _AABB_CACHE.get(key)
    if hit is None:
        if len(_AABB_CACHE) > 64:
            _AABB_CACHE.clear()
        ab = aabb.detach().float().cpu()
        hit = (aabb, ([float(ab[0, i]) for i in range(3)], [float(ab[1, i]) for i in range(3)]))
        _AABB_CACHE[key] = hit
    return hit[1]


def vm_desc(planes, lines, aabb, n_levels, build_mips):
    """VMDesc for these factors, reused while none of them has been modified (same storage, same autograd version, same
    parameter epoch): the forward / backward / SDF-only calls of one training step share one descriptor and ONE mip-chain
    build.  The descriptor holds references to the factor tensors and the aabb, so a key cannot outlive its storage."""
    key = tuple((t.data_ptr(), t._version) for t in (*planes, *lines)) + (aabb.data_ptr(), aabb._version, int(n_levels), bool(build_mips),
                                                                         torch.cuda.current_stream().cuda_stream, _PARAM_EPOCH)
    if not (build_mips and int(n_levels) > 1):
        return VMDesc(planes, lines, aabb, n_levels, build_mips)      # nothing expensive to share
    d = _VMDESC_CACHE.get(key)
    if d is None:
        _VMDESC_CACHE.clear()                             # one live entry per call site pattern is enough; mips are large
        d = VMDesc(planes, lines, aabb, n_levels, build_mips)
        _VMDESC_CACHE[key] = d
    return d


class VMDesc:
    """Owns the C descriptor of a VM field plus the tensors it points to."""

    def __init__(self, planes: Sequence[torch.Tensor], lines: Sequence[torch.Tensor], aabb: torch.Tensor,
                 n_levels: int, build_mips: bool):
        self.param_planes, self.param_lines = list(planes), list(lines)
        self.planes = [_nhwc(p) for p in planes]          # [H,W,C]
        self.lines = [_nhwc(l)[:, 0, :] for l in lines]   # [G,C]
        self.lines = [l if l.is_contiguous() else l.contiguous() for l in self.lines]
        self.n_levels = int(n_levels)
        self.aabb = aabb                                  # keeps the storage behind the cache key alive
        self.C = int(self.planes[0].shape[-1])
        dev = self.planes[0].device
        self.device = dev
        f = VMField()
        self.plane_mips: List[Optional[torch.Tensor]] = [None] * 3
        self.line_mips: List[Optional[torch.Tensor]] = [None] * 3
        ab_min, ab_max = _aabb_floats(aabb)
        for i in range(3):
            H, W, _ = self.planes[i].shape
            G = self.lines[i].shape[0]
            f.plane[i] = self.planes[i].data_ptr()
            f.line[i] = self.lines[i].data_ptr()
            f.plane_h[i], f.plane_w[i], f.line_g[i] = H, W, G
            f.aabb_min[i] = ab_min[i]
            f.aabb_max[i] = ab_max[i]
            if self.n_levels > 1 and build_mips:
                npl = sum(h * w for h, w in mip_sizes(H, W, self.n_levels))
                nln = sum(h for h, _ in mip_sizes(G, 1, self.n_levels))
                self.plane_mips[i] = torch.empty(npl * self.C, device=dev, dtype=torch.float32)
                self.line_mips[i] = torch.empty(nln * self.C, device=dev, dtype=torch.float32)
                f.plane_mip[i] = self.plane_mips[i].data_ptr()
                f.line_mip[i] = self.line_mips[i].data_ptr()
        f.n_comp = self.C
        f.n_levels = self.n_levels
        self.c = f
        if self.n_levels > 1 and build_mips:
            out = VMMut()
            for i in range(3):
                out.plane_mip[i] = self.plane_mips[i].data_ptr()
                out.line_mip[i] = self.line_mips[i].data_ptr()
            check(_lib.load().tf_vm_build_mips(C.byref(f), C.byref(out), stream_ptr()), "tf_vm_build_mips")

    def new_grads(self, with_mips: bool):
        """Zeroed gradient accumulators with the same layouts; returns (VMMut, tensors)."""
        g = VMMut()
        gp, gl = [], []
        for p, l, pv, lv in zip(self.param_planes, self.param_lines, self.planes, self.lines):
            if pv.data_ptr() == p.data_ptr() and lv.data_ptr() == l.data_ptr():     # channels-last parameters (no staging copy)
                gp.append(_nhwc(_grad_zeros(p.detach())))
                gl.append(_nhwc(_grad_zeros(l.detach()))[:, 0, :])
            else:
                gp.append(torch.zeros_like(pv))
                gl.append(torch.zeros_like(lv))
        gpm: List[Optional[torch.Tensor]] = [None] * 3
        glm: List[Optional[torch.Tensor]] = [None] * 3
        for i in range(3):
            g.plane[i] = gp[i].data_ptr()
            g.line[i] = gl[i].data_ptr()
            if with_mips and self.n_levels > 1:
                gpm[i] = torch.zeros_like(self.plane_mips[i])
                glm[i] = torch.zeros_like(self.line_mips[i])
                g.plane_mip[i] = gpm[i].data_ptr()
                g.line_mip[i] = glm[i].data_ptr()
        return g, gp, gl, gpm, glm

    def finish_grads(self, g, gp, gl, with_mips: bool):
        """Fold mip gradients into level 0 and return grads shaped like the parameters."""
        if with_mips and self.n_levels > 1:
            check(_lib.load().tf_vm_fold_mip_grads(C.byref(self.c), C.byref(g), stream_ptr()), "tf_vm_fold_mip_grads")
        planes = [t.permute(2, 0, 1).unsqueeze(0) for t in gp]                 # [1,C,H,W] (channels-last strides)
        lines = [t.permute(1, 0).unsqueeze(0).unsqueeze(-1) for t in gl]       # [1,C,G,1]
        return planes, lines


def _f32c(t: Optional[torch.Tensor]) -> Optional[torch.Tensor]:
    if t is None:
        return None
    t = t.detach()
    if t.dtype != torch.float32:
        t = t.float()
    return t if t.is_contiguous() else t.contiguous()


def _mlp_desc(W0, b0, W1, b1):
    m = SdfMlp()
    ws = [_f32c(W0), _f32c(b0), _f32c(W1), _f32c(b1)]
    m.W0, m.b0, m.W1, m.b1 = (w.data_ptr() for w in ws)
    m.hidden = int(W0.shape[0])
    m.app_dim = int(W1.shape[0]) - 1
    return m, ws


def _units_arr(units) -> C.Array:
    u = [float(x) for x in units]
    return (C.c_float * 3)(*u)


class SdfStencilFunction(torch.autograd.Function):
    """TensoSDF.forward at x plus the six FD taps of TensoSDF.gradient
    (reference network/fields.py:262-299, 227-260) in one fused kernel.

    inputs : xyz [N,3], level [N] or None, units (3 floats), aabb [2,3], n_levels,
             W0,b0,W1,b1, plane0..2, line0..2
    outputs: sdf [N], feat [N,A], grad [N,3], hess [N]
    No gradient flows to xyz / level (the reference detaches uv and never asks for d level).
    """

    @staticmethod
    def forward(ctx, xyz, level, units, aabb, n_levels, W0, b0, W1, b1, *factors):
        lib = _lib.load()
        planes, lines = factors[:3], factors[3:6]
        xyz_c = _f32c(xyz.reshape(-1, 3))
        lvl_c = None if level is None else _f32c(level.reshape(-1))
        n = xyz_c.shape[0]
        vm = vm_desc(planes, lines, aabb, n_levels, lvl_c is not None)
        m, mlp_keep = _mlp_desc(W0, b0, W1, b1)
        A = m.app_dim
        dev = xyz_c.device
        sdf7 = torch.empty(n, 7, device=dev, dtype=torch.float32)
        feat = torch.empty(n, A, device=dev, dtype=torch.float32)
        grad = torch.empty(n, 3, device=dev, dtype=torch.float32)
        hess = torch.empty(n, device=dev, dtype=torch.float32)
        wsb = lib.tf_sdf_stencil_fwd_workspace(C.byref(vm.c), C.byref(m), n, 1)
        if wsb == 0:
            check(1, "tf_sdf_stencil_fwd_workspace")
        ws = torch.empty(wsb // 4, device=dev, dtype=torch.float32)
        u = _units_arr(units)
        with _timed("sdf_stencil_fwd"):
            check(lib.tf_sdf_stencil_fwd(C.byref(vm.c), C.byref(m), ptr(xyz_c), ptr(lvl_c), n, u, ptr(sdf7), ptr(feat),
                                         ptr(grad), ptr(hess), ptr(ws), wsb, stream_ptr()), "tf_sdf_stencil_fwd")
        ctx.save_for_backward(xyz_c, lvl_c, sdf7, aabb, W0, b0, W1, b1, *factors)
        ctx.units = [float(x) for x in units]
        ctx.n_levels = n_levels
        # the centre hidden activations sit in the forward workspace: keep it for the backward (4 n H bytes), which reads them
        # (they feed the weight gradient of the appearance head)
        ctx.hidden = None
        if any(ctx.needs_input_grad):
            off = lib.tf_sdf_stencil_fwd_hidden_offset(C.byref(vm.c), C.byref(m))
            if off != C.c_size_t(-1).value:
                ctx.hidden = (ws, off)
        sdf = sdf7[:, 0].contiguous()
        return sdf, feat, grad, hess

    @staticmethod
    def backward(ctx, g_sdf, g_feat, g_grad, g_hess):
        lib = _lib.load()
        xyz_c, lvl_c, sdf7, aabb, W0, b0, W1, b1, *factors = ctx.saved_tensors
        planes, lines = factors[:3], factors[3:6]
        n = xyz_c.shape[0]
        with_mips = lvl_c is not None
        vm = vm_desc(planes, lines, aabb, ctx.n_levels, with_mips)
        m, mlp_keep = _mlp_desc(W0, b0, W1, b1)
        g, gp, gl, gpm, glm = vm.new_grads(with_mips)
        dW0, db0, dW1, db1 = (_grad_zeros(w) for w in mlp_keep)
        mg = SdfMlpGrad()
        mg.W0, mg.b0, mg.W1, mg.b1 = dW0.data_ptr(), db0.data_ptr(), dW1.data_ptr(), db1.data_ptr()
        need_all = lib.tf_sdf_stencil_bwd_workspace(C.byref(vm.c), C.byref(m), max(n, 1))
        wsb = min(need_all, max(BWD_WORKSPACE_BYTES, lib.tf_sdf_stencil_bwd_workspace(C.byref(vm.c), C.byref(m), 16)))
        ws = torch.empty(wsb // 4, device=xyz_c.device, dtype=torch.float32)
        gs, gf, gg, gh = _f32c(g_sdf), _f32c(g_feat), _f32c(g_grad), _f32c(g_hess)
        hid = None if ctx.hidden is None else ctx.hidden[0].data_ptr() + ctx.hidden[1]
        with _timed("sdf_stencil_bwd"):
            check(lib.tf_sdf_stencil_bwd(C.byref(vm.c), C.byref(m), ptr(xyz_c), ptr(lvl_c), n, _units_arr(ctx.units), ptr(sdf7), hid,
                                         ptr(gs), ptr(gf), ptr(gg), ptr(gh), C.byref(g), C.byref(mg), ptr(ws), wsb, stream_ptr()),
                  "tf_sdf_stencil_bwd")
        ctx.hidden = None
        d_planes, d_lines = vm.finish_grads(g, gp, gl, with_mips)
        return (None, None, None, None, None, dW0, db0, dW1, db1, *d_planes, *d_lines)


def sdf_only(xyz, level, aabb, n_levels, W0, b0, W1, b1, planes, lines) -> torch.Tensor:
    """TensoSDF.sdf (reference network/fields.py:148) without autograd -> [N]."""
    lib = _lib.load()
    xyz_c = _f32c(xyz.reshape(-1, 3))
    lvl_c = None if level is None else _f32c(level.reshape(-1))
    n = xyz_c.shape[0]
    vm = vm_desc(planes, lines, aabb, n_levels, lvl_c is not None)
    m, keep = _mlp_desc(W0, b0, W1, b1)
    out = torch.empty(n, device=xyz_c.device, dtype=torch.float32)
    wsb = lib.tf_sdf_stencil_fwd_workspace(C.byref(vm.c), C.byref(m), n, 0)
    if wsb == 0:
        check(1, "tf_sdf_stencil_fwd_workspace")
    ws = torch.empty(wsb // 4, device=xyz_c.device, dtype=torch.float32)
    check(lib.tf_sdf_only_fwd(C.byref(vm.c), C.byref(m), ptr(xyz_c), ptr(lvl_c), n, ptr(out), ptr(ws), wsb, stream_ptr()),
          "tf_sdf_only_fwd")
    return out


def sdf_point(xyz, level, aabb, n_levels, W0, b0, W1, b1, planes, lines):
    """TensoSDF.forward (reference network/fields.py:262-299) without autograd and without the FD taps -> (sdf [N], feat [N,A]);
    None when the decoder shape is outside the tensor-core path (the caller then uses the stencil)."""
    lib = _lib.load()
    xyz_c = _f32c(xyz.reshape(-1, 3))
    lvl_c = None if level is None else _f32c(level.reshape(-1))
    n = xyz_c.shape[0]
    vm = vm_desc(planes, lines, aabb, n_levels, lvl_c is not None)
    m, keep = _mlp_desc(W0, b0, W1, b1)
    if lib.tf_sdf_stencil_fwd_hidden_offset(C.byref(vm.c), C.byref(m)) == C.c_size_t(-1).value:
        return None
    sdf = torch.empty(n, device=xyz_c.device, dtype=torch.float32)
    feat = torch.empty(n, m.app_dim, device=xyz_c.device, dtype=torch.float32)
    if n == 0:
        return sdf, feat
    wsb = lib.tf_sdf_stencil_fwd_workspace(C.byref(vm.c), C.byref(m), n, 1)
    if wsb == 0:
        check(1, "tf_sdf_stencil_fwd_workspace")
    ws = torch.empty(wsb // 4, device=xyz_c.device, dtype=torch.float32)
    check(lib.tf_sdf_point_fwd(C.byref(vm.c), C.byref(m), ptr(xyz_c), ptr(lvl_c), n, ptr(sdf), ptr(feat), ptr(ws), wsb, stream_ptr()),
          "tf_sdf_point_fwd")
    return sdf, feat


class VMFeatureFunction(torch.autograd.Function):
    """feat[N,3C] = concat_i plane_i(x)*line_i(x) (reference network/fields.py:776-806,
    network/flow.py:709-740).  inputs: xyz, level|None, aabb, n_levels, plane0..2, line0..2."""

    @staticmethod
    def forward(ctx, xyz, level, aabb, n_levels, *factors):
        lib = _lib.load()
        planes, lines = factors[:3], factors[3:6]
        xyz_c = _f32c(xyz.reshape(-1, 3))
        lvl_c = None if level is None else _f32c(level.reshape(-1))
        n = xyz_c.shape[0]
        vm = vm_desc(planes, lines, aabb, n_levels, lvl_c is not None)
        feat = torch.empty(n, 3 * vm.C, device=xyz_c.device, dtype=torch.float32)
        check(lib.tf_vm_feature_fwd(C.byref(vm.c), ptr(xyz_c), ptr(lvl_c), n, ptr(feat), stream_ptr()), "tf_vm_feature_fwd")
        ctx.save_for_backward(xyz_c, lvl_c, aabb, *factors)
        ctx.n_levels = n_levels
        return feat

    @staticmethod
    def backward(ctx, g_feat):
        lib = _lib.load()
        xyz_c, lvl_c, aabb, *factors = ctx.saved_tensors
        planes, lines = factors[:3], factors[3:6]
        with_mips = lvl_c is not None
        vm = vm_desc(planes, lines, aabb, ctx.n_levels, with_mips)
        g, gp, gl, gpm, glm = vm.new_grads(with_mips)
        gf = _f32c(g_feat)
        check(lib.tf_vm_feature_bwd(C.byref(vm.c), ptr(xyz_c), ptr(lvl_c), xyz_c.shape[0], ptr(gf), C.byref(g), stream_ptr()),
              "tf_vm_feature_bwd")
        d_planes, d_lines = vm.finish_grads(g, gp, gl, with_mips)
        return (None, None, None, None, *d_planes, *d_lines)


class NeusCompositeFunction(torch.autograd.Function):
    """NeuS alpha + transmittance + per-ray accumulation (reference
    network/shapeRenderer.py:1004-1024, 1166-1206).

    inputs : sdf [N], grad [N,3], dists [N], dirs [R,3], ray_offsets int32 [R+1],
             variance (0-d), cos_anneal (float), vals [N,D], train_variance (bool)
    outputs: alpha [N], weights [N], acc [R], out [R,D]
    """

    @staticmethod
    def forward(ctx, sdf, grad, dists, dirs, ray_offsets, variance, cos_anneal, vals, train_variance=True):
        lib = _lib.load()
        sdf_c, grad_c, dists_c, dirs_c = _f32c(sdf), _f32c(grad), _f32c(dists), _f32c(dirs)
        vals_c = _f32c(vals)
        var_c = _f32c(variance.reshape(1))
        offs = ray_offsets.contiguous()
        assert offs.dtype == torch.int32
        n, R = sdf_c.shape[0], dirs_c.shape[0]
        D = 0 if vals_c is None else int(vals_c.shape[1])
        dev = sdf_c.device
        alpha = torch.empty(n, device=dev, dtype=torch.float32)
        weights = torch.empty(n, device=dev, dtype=torch.float32)
        acc = torch.empty(R, device=dev, dtype=torch.float32)
        out = torch.empty(R, D, device=dev, dtype=torch.float32)
        if n == 0:   # no samples at all: every ray composites to zero
            acc.zero_(); out.zero_()
            ctx.save_for_backward(sdf_c, grad_c, dists_c, dirs_c, offs, var_c, vals_c, alpha, weights, acc, out)
            ctx.cos_anneal, ctx.train_variance, ctx.var_shape = float(cos_anneal), bool(train_variance), variance.shape
            ctx.mark_non_differentiable(alpha)
            ctx.set_materialize_grads(False)
            return alpha, weights, acc, out
        with _timed("neus_composite_fwd"):
          check(lib.tf_neus_composite_fwd(ptr(sdf_c), ptr(grad_c), ptr(dists_c), ptr(dirs_c), ptr(offs), R, ptr(var_c),
                                        float(cos_anneal), ptr(vals_c), D, ptr(alpha), ptr(weights), ptr(acc), ptr(out),
                                        stream_ptr()), "tf_neus_composite_fwd")
        ctx.save_for_backward(sdf_c, grad_c, dists_c, dirs_c, offs, var_c, vals_c, alpha, weights, acc, out)
        ctx.cos_anneal = float(cos_anneal)
        ctx.train_variance = bool(train_variance)
        ctx.var_shape = variance.shape
        ctx.mark_non_differentiable(alpha)
        ctx.set_materialize_grads(False)       # an unused output (usually `weights`) reaches backward as None, not as zeros [N]
        return alpha, weights, acc, out

    @staticmethod
    def backward(ctx, _g_alpha, g_weights, g_acc, g_out):
        lib = _lib.load()
        sdf_c, grad_c, dists_c, dirs_c, offs, var_c, vals_c, alpha, weights, acc, out = ctx.saved_tensors
        n, R = sdf_c.shape[0], dirs_c.shape[0]
        D = 0 if vals_c is None else int(vals_c.shape[1])
        dev = sdf_c.device
        d_sdf = torch.zeros(n, device=dev, dtype=torch.float32)
        d_grad = torch.zeros(n, 3, device=dev, dtype=torch.float32)
        d_vals = torch.zeros(n, D, device=dev, dtype=torch.float32) if D > 0 else None
        d_var = torch.zeros(1, device=dev, dtype=torch.float32) if ctx.train_variance else None
        if n == 0:
            dv = None if d_var is None else d_var.reshape(ctx.var_shape)
            return d_sdf, d_grad, None, None, None, dv, None, d_vals, None
        ga, go, gw = _f32c(g_acc), _f32c(g_out), _f32c(g_weights)      # converted copies must outlive the launch
        with _timed("neus_composite_bwd"):
          check(lib.tf_neus_composite_bwd(ptr(sdf_c), ptr(grad_c), ptr(dists_c), ptr(dirs_c), ptr(offs), R, ptr(var_c),
                                        ctx.cos_anneal, ptr(vals_c), D, ptr(alpha), ptr(weights), ptr(acc), ptr(out),
                                        ptr(ga), ptr(go), ptr(gw), ptr(d_sdf), ptr(d_grad), ptr(d_vals),
                                        ptr(d_var), stream_ptr()), "tf_neus_composite_bwd")
        dv = None if d_var is None else d_var.reshape(ctx.var_shape)
        return d_sdf, d_grad, None, None, None, dv, None, d_vals, None


ACT = {"none": 0, "relu": 1, "leaky": 2, "softplus100": 3, "sigmoid": 4, "exp": 5}


class LinearFunction(torch.autograd.Function):
    """Y = act(X W^T + b): one nn.Linear + activation of the reference's small MLPs
    (network/other_field.py:20-121, network/flow.py:577-598) as one fused kernel.
    X [M,K], W [N,K], b [N] or None, act in ACT, act_param (max for 'exp')."""

    @staticmethod
    def forward(ctx, X, W, b, act, act_param=0.0):
        lib = _lib.load()
        Xc, Wc, bc = _f32c(X), _f32c(W), _f32c(b)
        M, K = Xc.shape
        N = Wc.shape[0]
        Y = torch.empty(M, N, device=Xc.device, dtype=torch.float32)
        wsb = int(lib.tf_linear_workspace(M, K, N))
        ws = torch.empty(wsb // 4, device=Xc.device, dtype=torch.float32) if wsb else None
        with _timed(f"linear_fwd[{K}->{N}]"):
            check(lib.tf_linear_fwd(ptr(Xc), ptr(Wc), ptr(bc), M, K, N, ACT[act], float(act_param), ptr(Y), ptr(ws), wsb,
                                    stream_ptr()), "tf_linear_fwd")
        ctx.save_for_backward(Xc, Wc, Y)
        ctx.act, ctx.act_param, ctx.has_bias = act, float(act_param), b is not None
        return Y

    @staticmethod
    def backward(ctx, gY):
        lib = _lib.load()
        Xc, Wc, Y = ctx.saved_tensors
        M, K = Xc.shape
        N = Wc.shape[0]
        gYc = _f32c(gY)
        dpre = torch.empty_like(Y)
        need_x, need_w, need_b = ctx.needs_input_grad[0], ctx.needs_input_grad[1], ctx.has_bias and ctx.needs_input_grad[2]
        dX = torch.empty(M, K, device=Xc.device, dtype=torch.float32) if need_x else None
        dW = torch.zeros_like(Wc) if need_w else None
        db = torch.zeros(N, device=Xc.device, dtype=torch.float32) if need_b else None
        wsb = int(lib.tf_linear_workspace(M, K, N))
        ws = torch.empty(wsb // 4, device=Xc.device, dtype=torch.float32) if wsb else None
        with _timed(f"linear_bwd[{K}->{N}]"):
            check(lib.tf_linear_bwd(ptr(Xc), ptr(Wc), ptr(Y), ptr(gYc), ptr(dpre), M, K, N, ACT[ctx.act], ctx.act_param,
                                    ptr(dX), ptr(dW), ptr(db), ptr(ws), wsb, stream_ptr()), "tf_linear_bwd")
        return dX, dW, db, None, None


def linear(X, W, b=None, act="none", act_param=0.0):
    if X.shape[0] == 0:
        return X.new_zeros(0, W.shape[0])
    K = X.shape[1]
    pad = -K % 16
    if pad and _lib.load().tf_linear_workspace(X.shape[0], K + pad, W.shape[0]) > 0:
        # ragged input width (the shader heads read 90 / 123 / 161 concatenated features) of a layer that the tensor-core
        # kernels take once it is padded: zero columns up to the next multiple of 16 put the layer, its data gradient and its
        # weight gradient there (16-byte aligned rows); the result is unchanged and autograd slices the padding off both gradients
        X = torch.nn.functional.pad(X, (0, pad))
        W = torch.nn.functional.pad(W, (0, pad))
    return LinearFunction.apply(X, W, b, act, act_param)


class TVFunction(torch.autograd.Function):
    """TVLoss (reference network/other_field.py:170-191) of one [1,C,H,W] texture stored channels-last: two sums of
    squared neighbour differences in one pass, gradient in one pass.  Returns weight * 2 * (sum_h/count_h + sum_w/count_w)."""

    @staticmethod
    def forward(ctx, x, weight):
        lib = _lib.load()
        v = _nhwc(x)                                     # [H,W,C] contiguous view of the channels-last parameter
        H, W, C = v.shape
        sums = torch.zeros(2, device=x.device, dtype=torch.float32)
        with _timed("tv_fwd"):
            check(lib.tf_tv_fwd(ptr(v), H, W, C, ptr(sums), stream_ptr()), "tf_tv_fwd")
        count_h, count_w = C * (H - 1) * W, C * H * (W - 1)
        ctx.save_for_backward(x)
        ctx.scales = (float(weight) * 2.0 / count_h if count_h else 0.0, float(weight) * 2.0 / count_w if count_w else 0.0)
        return sums[0] * ctx.scales[0] + sums[1] * ctx.scales[1]

    @staticmethod
    def backward(ctx, g_out):
        lib = _lib.load()
        (x,) = ctx.saved_tensors
        v = _nhwc(x)
        H, W, C = v.shape
        g = torch.zeros_like(v)
        go = _f32c(g_out.reshape(1))                     # stays on the device: no host sync in backward
        with _timed("tv_bwd"):
            check(lib.tf_tv_bwd(ptr(v), H, W, C, ctx.scales[0], ctx.scales[1], ptr(go), ptr(g), stream_ptr()), "tf_tv_bwd")
        return g.permute(2, 0, 1)[None], None            # logical [1,C,H,W], channels-last memory like the parameter


def gaussian_taps(kernel_size: int, sigma: float):
    """Normalised 1-D and 2-D taps of the reference's GaussianBlur1D / GaussianBlur2D (network/other_field.py:121-135),
    evaluated in fp32 like the reference buffers.  Returns (taps1d [KS], taps2d [KS*KS]) as Python float lists."""
    xs = torch.arange(-kernel_size // 2 + 1.0, kernel_size // 2 + 1.0)
    k1 = torch.exp(-xs ** 2 / (2 * sigma ** 2))
    k1 = k1 / k1.sum()
    xx, yy = torch.meshgrid(xs, xs, indexing='ij')
    k2 = torch.exp(-(xx ** 2 + yy ** 2) / (2 * sigma ** 2))
    k2 = k2 / k2.sum()
    return [float(v) for v in k1], [float(v) for v in k2.reshape(-1)]


class GaussResidualFunction(torch.autograd.Function):
    """sum over the interior of (x - GaussianBlur(x))^2 for one [1,C,H,W] texture stored channels-last (one term of
    grid_gaussian_loss, reference network/fields.py:301-309): one kernel for the residual + its squared sum, one for the
    gradient.  `taps` is the row-major [KH*KW] kernel (KW = 1 for the [1,C,G,1] lines)."""

    @staticmethod
    def forward(ctx, x, taps, KH, KW):
        lib = _lib.load()
        v = _nhwc(x)
        H, W, Cc = v.shape
        r = torch.empty_like(v)
        total = torch.zeros(1, device=x.device, dtype=torch.float32)
        tp = (C.c_float * len(taps))(*taps)
        with _timed("gauss_fwd"):
            check(lib.tf_gauss_residual_fwd(ptr(v), H, W, Cc, tp, KH, KW, ptr(r), ptr(total), stream_ptr()), "tf_gauss_residual_fwd")
        ctx.save_for_backward(r)
        ctx.taps, ctx.k = tp, (KH, KW)
        return total[0]

    @staticmethod
    def backward(ctx, g_out):
        lib = _lib.load()
        (r,) = ctx.saved_tensors
        H, W, Cc = r.shape
        g = torch.zeros_like(r)
        go = _f32c(g_out.reshape(1))
        with _timed("gauss_bwd"):
            check(lib.tf_gauss_residual_bwd(ptr(r), H, W, Cc, ctx.taps, ctx.k[0], ctx.k[1], ptr(go), ptr(g), stream_ptr()),
                  "tf_gauss_residual_bwd")
        return g.permute(2, 0, 1)[None], None, None, None


class PwquadFunction(torch.autograd.Function):
    """Piecewise-quadratic coupling transform (reference network/flow.py:314-525).
    y [M], st [M,21] -> x [M], logj [M].  inverse=True is the sampling direction (no grad)."""

    @staticmethod
    def forward(ctx, y, st, inverse):
        lib = _lib.load()
        yc, stc = _f32c(y), _f32c(st)
        M = yc.shape[0]
        x = torch.empty_like(yc)
        logj = torch.empty_like(yc)
        with _timed("pwquad_fwd"):
            check(lib.tf_pwquad_fwd(ptr(yc), ptr(stc), M, 1 if inverse else 0, ptr(x), ptr(logj), stream_ptr()), "tf_pwquad_fwd")
        ctx.save_for_backward(yc, stc)
        ctx.inverse = bool(inverse)
        return x, logj

    @staticmethod
    def backward(ctx, g_x, g_logj):
        if ctx.inverse:
            raise RuntimeError("the inverse (sampling) spline has no backward: the reference samples from frozen flow copies")
        lib = _lib.load()
        yc, stc = ctx.saved_tensors
        M = yc.shape[0]
        d_y = torch.empty_like(yc)
        d_st = torch.empty_like(stc)
        gx, gl = _f32c(g_x), _f32c(g_logj)                           # converted copies must outlive the launch
        with _timed("pwquad_bwd"):
            check(lib.tf_pwquad_bwd(ptr(yc), ptr(stc), M, ptr(gx), ptr(gl), ptr(d_y), ptr(d_st), stream_ptr()),
                  "tf_pwquad_bwd")
        return d_y, d_st, None


class FlowBlockFunction(torch.autograd.Function):
    """One coupling block of the TensoFlow sampler (reference network/flow.py:549-641) as ONE kernel per direction of
    differentiation: conditioner MLP + spline for every (point, direction) pair, the per-point feature part of the first
    layer evaluated once per point.  y [M,2], logj [M] or None, feat [pn,F] (M = pn * sn), the eight nn.Linear tensors of the
    conditioner, Reshift constants.  inverse=True is the sampling direction (no backward)."""

    @staticmethod
    def forward(ctx, y, logj, feat, sn, cond, inverse, scale, offset, W1, b1, W2, b2, W3, b3, W4, b4):
        lib = _lib.load()
        yc, fc = _f32c(y.reshape(-1, 2)), _f32c(feat)
        lc = None if logj is None else _f32c(logj.reshape(-1))
        ws = [_f32c(w) for w in (W1, b1, W2, b2, W3, b3, W4, b4)]
        M = yc.shape[0]
        y_out = torch.empty_like(yc)
        lj_out = torch.empty(M, device=yc.device, dtype=torch.float32)
        # density direction with gradients: the tensor-core forward keeps h1, h2, h3 and the spline parameters (864 B per pair),
        # so that the backward is the adjoint chain alone
        keep = (not inverse) and any(ctx.needs_input_grad)
        sh = torch.empty(M, 3, 64, device=yc.device, dtype=torch.float32) if keep else None
        sst = torch.empty(M, 24, device=yc.device, dtype=torch.float32) if keep else None
        with _timed("flow_block_fwd"):
            check(lib.tf_flow_block_fwd(ptr(yc), ptr(lc), ptr(fc), int(fc.shape[1]), int(sn), *(ptr(w) for w in ws), float(scale), float(offset),
                                        int(cond), 1 if inverse else 0, M, ptr(y_out), ptr(lj_out), ptr(sh), ptr(sst), stream_ptr()),
                  "tf_flow_block_fwd")
        ctx.save_for_backward(yc, fc, *ws)
        ctx.kept = (sh, sst)
        ctx.cfg = (int(sn), int(cond), bool(inverse), float(scale), float(offset), None if logj is None else logj.shape)
        return y_out, lj_out

    @staticmethod
    def backward(ctx, g_y, g_lj):
        sn, cond, inverse, scale, offset, logj_shape = ctx.cfg
        if inverse:
            raise RuntimeError("the inverse (sampling) coupling block has no backward: the reference samples from frozen flow copies")
        lib = _lib.load()
        yc, fc, *ws = ctx.saved_tensors
        M = yc.shape[0]
        gy = None if g_y is None else _f32c(g_y.reshape(-1, 2))
        gl = None if g_lj is None else _f32c(g_lj.reshape(-1))
        g_in = torch.empty_like(yc)
        d_feat = torch.zeros_like(fc)
        dws = [_grad_zeros(w) for w in ws]
        with _timed("flow_block_bwd"):
            check(lib.tf_flow_block_bwd(ptr(yc), ptr(fc), int(fc.shape[1]), sn, *(ptr(w) for w in ws), scale, offset, cond, M, ptr(ctx.kept[0]),
                                        ptr(ctx.kept[1]), ptr(gy), ptr(gl), ptr(g_in), ptr(d_feat), *(ptr(d) for d in dws), stream_ptr()),
                  "tf_flow_block_bwd")
        ctx.kept = (None, None)
        g_logj_in = None if (logj_shape is None or gl is None) else gl.reshape(logj_shape)
        return (g_in, g_logj_in, d_feat, None, None, None, None, None, *dws)
