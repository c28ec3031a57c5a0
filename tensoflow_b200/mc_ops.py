"""Material-stage operators over the C ABI: mesh ray tracer, direction sets, env-light
lookup and the BRDF / Monte-Carlo estimator (reference network/fields.py:824-1335,
network/light.py:125-162, raytracing/raytracer.py)."""
from __future__ import annotations

import contextlib
import ctypes as C

import numpy as np
import torch

from . import _lib
from ._lib import check, ptr, stream_ptr
from .ops import _f32c, _timed


class _TooFewTriangles(RuntimeError, AssertionError):
    """A mesh of at most 8 triangles: a RuntimeError like every other refusal of the device build, and still the
    AssertionError the host build raises for it."""


class RayTracer:
    """Drop-in for the reference's raytracing.RayTracer (raytracing/raytracer.py:8-54):
    RayTracer(vertices, triangles).trace(rays_o, rays_d) -> positions, face_normals, depth.

    CUDA tensors (both on one device) are built into a BVH on that device (tf_bvh_build, no host copy); numpy arrays and CPU
    tensors by the host build (tf_bvh_create).  Both builds give the same BVH node for node, so trace and closest_point return
    the same bits either way.  A mesh of at most 8 triangles raises _TooFewTriangles on the device path: a RuntimeError like the
    device path's other refusals, and also the AssertionError that callers of the host path (and of the reference) catch."""

    def __init__(self, vertices, triangles):
        self._device = None
        if torch.is_tensor(vertices) and torch.is_tensor(triangles) and vertices.is_cuda and vertices.device == triangles.device:
            self._build_on_device(vertices.detach(), triangles.detach())
            return
        if torch.is_tensor(vertices):
            vertices = vertices.detach().cpu().numpy()
        if torch.is_tensor(triangles):
            triangles = triangles.detach().cpu().numpy()
        assert triangles.shape[0] > 8, "BVH needs at least 8 triangles."
        v = np.ascontiguousarray(vertices, dtype=np.float32)
        t = np.ascontiguousarray(triangles, dtype=np.int32)
        self._h = C.c_void_p()
        lib = _lib.load()
        check(lib.tf_bvh_create(v.ctypes.data_as(C.c_void_p), v.shape[0], t.ctypes.data_as(C.c_void_p), t.shape[0],
                                C.byref(self._h)), "tf_bvh_create")
        self.n_triangles = int(t.shape[0])

    def _build_on_device(self, vertices, triangles):
        """tf_bvh_build on the tensors' device after the checks below, which read back one small tensor and raise before any
        launch of the library."""
        self._h = None
        nt, nv = validate_device_mesh(vertices, triangles)
        dev = vertices.device
        with torch.cuda.device(dev):
            v = _f32c(vertices)
            t = triangles.to(torch.int32).contiguous()
            lib = _lib.load()
            n_nodes, ws_bytes = C.c_int64(), C.c_size_t()
            check(lib.tf_bvh_build_sizes(nt, C.byref(n_nodes), C.byref(ws_bytes)), "tf_bvh_build_sizes")
            ws = torch.empty(ws_bytes.value, device=dev, dtype=torch.uint8)
            nodes = torch.empty(n_nodes.value, 8, device=dev, dtype=torch.float32)
            tris = torch.empty(nt, 12, device=dev, dtype=torch.float32)
            perm = torch.empty(nt, device=dev, dtype=torch.int32)
            s = stream_ptr()
            with _timed("bvh_build"):
                check(lib.tf_bvh_build(ptr(v), nv, ptr(t), nt, ptr(ws), ws_bytes.value, ptr(nodes), ptr(tris), ptr(perm), s),
                      "tf_bvh_build")
            h = C.c_void_p()
            check(lib.tf_bvh_create_from_device(ptr(nodes), n_nodes.value, ptr(tris), ptr(perm), nt, s, C.byref(h)),
                  "tf_bvh_create_from_device")
        self._h = h
        self._device = dev
        self.n_triangles = nt

    def _on_device(self):
        return torch.cuda.device(self._device) if self._device is not None else contextlib.nullcontext()

    def __del__(self):
        try:
            if getattr(self, "_h", None):
                _lib.load().tf_bvh_destroy(self._h)
                self._h = None
        except Exception:
            pass

    def trace(self, rays_o, rays_d, inplace=False):
        rays_o = _f32c(rays_o)
        rays_d = _f32c(rays_d)
        prefix = rays_o.shape[:-1]
        o, d = rays_o.reshape(-1, 3), rays_d.reshape(-1, 3)
        n = o.shape[0]
        positions = torch.empty_like(o)
        normals = torch.empty_like(d)
        depth = torch.empty(n, device=o.device, dtype=torch.float32)
        with self._on_device(), _timed("bvh_trace"):
            check(_lib.load().tf_bvh_trace(self._h, ptr(o), ptr(d), n, ptr(positions), ptr(normals), ptr(depth), stream_ptr()),
                  "tf_bvh_trace")
        return positions.reshape(*prefix, 3), normals.reshape(*prefix, 3), depth.reshape(*prefix)

    def closest_point(self, points):
        """Nearest point of the mesh to each of `points` [..., 3] -> (closest [..., 3] fp32, distance [...] fp32, triangle [...]
        int64 indexing the constructor's `triangles`).  The smaller squared distance wins, an exact tie the smaller triangle
        index; the result is bit-reproducible.  CUDA tensors only."""
        if not torch.is_tensor(points) or not points.is_cuda:
            raise RuntimeError("RayTracer.closest_point needs CUDA tensors (tensoflow_b200 has no CPU path)")
        if points.shape[-1] != 3:
            raise RuntimeError(f"RayTracer.closest_point needs points [..., 3], got {list(points.shape)}")
        p = _f32c(points)
        prefix = p.shape[:-1]
        q = p.reshape(-1, 3)
        n = q.shape[0]
        closest = torch.empty_like(q)
        dist = torch.empty(n, device=q.device, dtype=torch.float32)
        tri = torch.empty(n, device=q.device, dtype=torch.int64)
        with self._on_device(), _timed("bvh_closest_point"):
            check(_lib.load().tf_bvh_closest_point(self._h, ptr(q), n, ptr(closest), ptr(dist), ptr(tri), stream_ptr()),
                  "tf_bvh_closest_point")
        return closest.reshape(*prefix, 3), dist.reshape(prefix), tri.reshape(prefix)


def validate_device_mesh(vertices, triangles):
    """The checks RayTracer makes before building on the device: vertices [V,3] floating point, triangles [T,3] integer,
    8 < T < 2^31, every index in [0, min(V, 2^31)) and every coordinate of a referenced vertex finite once rounded to fp32 (the
    build's precision, so a float64 coordinate beyond the fp32 range is refused as the host build refuses it).  Reads one small tensor
    back to the host and launches nothing of the library.  Returns (T, V); raises RuntimeError."""
    if vertices.ndim != 2 or vertices.shape[1] != 3 or triangles.ndim != 2 or triangles.shape[1] != 3:
        raise RuntimeError(f"RayTracer needs vertices [V, 3] and triangles [T, 3], got {list(vertices.shape)} and "
                           f"{list(triangles.shape)}")
    if not vertices.is_floating_point() or triangles.is_floating_point() or triangles.dtype in (torch.bool, torch.uint8):
        raise RuntimeError(f"RayTracer needs floating-point vertices and int32 / int64 triangles, got {vertices.dtype} and "
                           f"{triangles.dtype}")
    nt, nv = int(triangles.shape[0]), int(vertices.shape[0])
    if nt == 0 or nv == 0:
        raise RuntimeError("RayTracer: empty mesh")
    if nt <= 8:
        raise _TooFewTriangles("BVH needs at least 8 triangles.")
    if nt >= 1 << 31:
        raise RuntimeError(f"RayTracer: {nt} triangles, the BVH holds fewer than 2^31")
    flat = triangles.reshape(-1)
    bad_vertex = ~torch.isfinite(vertices.to(torch.float32)).all(1)
    idx = flat.clamp(0, nv - 1)
    referenced = torch.index_select(bad_vertex, 0, idx if idx.dtype in (torch.int32, torch.int64) else idx.long())
    tmin, tmax, n_bad = torch.stack([flat.min().to(torch.int64), flat.max().to(torch.int64),
                                     referenced.sum().to(torch.int64)]).tolist()
    if tmin < 0 or tmax >= min(nv, 1 << 31):
        raise RuntimeError(f"RayTracer: triangle index out of range (indices span [{tmin}, {tmax}], {nv} vertices)")
    if n_bad:
        raise RuntimeError("RayTracer: non-finite vertex coordinate on a referenced vertex")
    return nt, nv


def mc_directions(mode: int, normals, view_dirs, src, aux, roughness, n_dirs: int, dirs_out, prob_out, offset: int):
    """Fill dirs_out[:, offset:offset+n_dirs], prob_out[:, offset:offset+n_dirs] (no autograd:
    direction sets are geometry + frozen-flow samples in the reference)."""
    pn, D = prob_out.shape
    with _timed("mc_directions"):
        check(_lib.load().tf_mc_directions(mode, ptr(_f32c(normals)), ptr(_f32c(view_dirs)), ptr(_f32c(src)), ptr(_f32c(aux)),
                                           ptr(_f32c(roughness)), pn, n_dirs, ptr(dirs_out), ptr(prob_out), D, offset, stream_ptr()),
              "tf_mc_directions")


def hit_encode(inters, dirs, hit_normals, idx, ide_mat, ide_m, ldx: int = 128):
    """[posenc(hit point, 8) | IDE(mirrored view direction)] rows of the occluded pairs `idx`, zero-padded to ldx columns
    (the inner-light MLP input of reference fields.py:951-975) in one kernel; no autograd (hit records are geometry)."""
    M = int(idx.shape[0])
    X = torch.empty(M, ldx, device=inters.device, dtype=torch.float32)
    with _timed("hit_encode"):
        check(_lib.load().tf_hit_encode(ptr(_f32c(inters.reshape(-1, 3))), ptr(_f32c(dirs.reshape(-1, 3))), ptr(_f32c(hit_normals.reshape(-1, 3))),
                                        ptr(idx.contiguous()), M, ptr(ide_mat), ptr(ide_m), ldx, ptr(X), stream_ptr()), "tf_hit_encode")
    return X


class CubeLightFunction(torch.autograd.Function):
    """EnvLight.direct_light: exp(cube bilinear(base, dirs)) on the masked pairs, 0 elsewhere."""

    @staticmethod
    def forward(ctx, base, dirs, mask):
        basec, dirsc = _f32c(base), _f32c(dirs.reshape(-1, 3))
        maskc = None if mask is None else mask.reshape(-1).to(torch.uint8).contiguous()
        n = dirsc.shape[0]
        out = torch.empty(n, 3, device=dirsc.device, dtype=torch.float32)
        with _timed("cube_light_fwd"):
            check(_lib.load().tf_cube_light_fwd(ptr(basec), int(basec.shape[1]), ptr(dirsc), ptr(maskc), n, ptr(out), stream_ptr()),
                  "tf_cube_light_fwd")
        ctx.save_for_backward(dirsc, maskc, out)
        ctx.base_shape = basec.shape
        return out.reshape(*dirs.shape)

    @staticmethod
    def backward(ctx, g):
        dirsc, maskc, out = ctx.saved_tensors
        d_base = torch.zeros(ctx.base_shape, device=out.device, dtype=torch.float32)
        gc = _f32c(g.reshape(-1, 3))
        with _timed("cube_light_bwd"):
            check(_lib.load().tf_cube_light_bwd(int(ctx.base_shape[1]), ptr(dirsc), ptr(maskc), dirsc.shape[0], ptr(out), ptr(gc),
                                                ptr(d_base), stream_ptr()), "tf_cube_light_bwd")
        return d_base, None, None


class McEstimateFunction(torch.autograd.Function):
    """BRDF weights + diffuse / specular Monte-Carlo estimators per surface point, plus the per-point sums of the two
    neural-importance-sampling losses (reference fields.py:1254-1333) when the flows' log q are given.
    returns out [pn,19]: diffuse(3) specular(3) mean diffuse light(3) mean specular light(3) visibility(1) indirect(3)
    nis_diffuse_sum(1) nis_specular_sum(1) nis_specular_count(1)."""

    @staticmethod
    def forward(ctx, normals, view_dirs, albedo, metallic, roughness, dirs, prob, lights, hit, n_diffuse,
                logq_d=None, ang_d=None, logq_s=None, ang_s=None):
        t = [_f32c(x) for x in (normals, view_dirs, albedo, metallic.reshape(-1), roughness.reshape(-1), dirs, prob, lights)]
        hitc = hit.to(torch.uint8).contiguous()
        pn, D = t[6].shape
        nis = [None if x is None else _f32c(x) for x in (logq_d, ang_d, logq_s, ang_s)]
        nd = 0 if nis[0] is None else int(nis[0].numel() // max(pn, 1))
        out = torch.empty(pn, 19, device=t[0].device, dtype=torch.float32)
        with _timed("mc_estimate_fwd"):
            check(_lib.load().tf_mc_estimate_fwd(*(ptr(x) for x in t), ptr(hitc), pn, int(n_diffuse), int(D - n_diffuse), ptr(nis[0]),
                                                 ptr(nis[1]), nd, ptr(nis[2]), ptr(nis[3]), ptr(out), stream_ptr()), "tf_mc_estimate_fwd")
        ctx.save_for_backward(*t, hitc, *[x for x in nis if x is not None])
        ctx.has_nis = [x is not None for x in nis]
        ctx.n_diffuse, ctx.nd = int(n_diffuse), nd
        ctx.m_shape, ctx.r_shape = metallic.shape, roughness.shape
        ctx.q_shapes = (None if logq_d is None else logq_d.shape, None if logq_s is None else logq_s.shape)
        return out

    @staticmethod
    def backward(ctx, g_out):
        saved = list(ctx.saved_tensors)
        t, hitc, rest = saved[:8], saved[8], saved[9:]
        nis = [rest.pop(0) if h else None for h in ctx.has_nis]
        pn, D = t[6].shape
        dev = t[0].device
        d_alb = torch.empty(pn, 3, device=dev, dtype=torch.float32)
        d_met = torch.empty(pn, device=dev, dtype=torch.float32)
        d_rgh = torch.empty(pn, device=dev, dtype=torch.float32)
        d_lights = torch.empty(pn, D, 3, device=dev, dtype=torch.float32)
        d_qd = None if nis[0] is None else torch.empty_like(nis[0])
        d_qs = None if nis[2] is None else torch.empty_like(nis[2])
        go = _f32c(g_out)
        with _timed("mc_estimate_bwd"):
            check(_lib.load().tf_mc_estimate_bwd(*(ptr(x) for x in t), ptr(hitc), pn, ctx.n_diffuse, D - ctx.n_diffuse, ptr(nis[0]),
                                                 ptr(nis[1]), ctx.nd, ptr(nis[2]), ptr(nis[3]), ptr(go), ptr(d_alb), ptr(d_met), ptr(d_rgh),
                                                 ptr(d_lights), ptr(d_qd), ptr(d_qs), stream_ptr()), "tf_mc_estimate_bwd")
        return (None, None, d_alb, d_met.reshape(ctx.m_shape), d_rgh.reshape(ctx.r_shape), None, None, d_lights, None, None,
                None if d_qd is None else d_qd.reshape(ctx.q_shapes[0]), None, None if d_qs is None else d_qs.reshape(ctx.q_shapes[1]), None)
