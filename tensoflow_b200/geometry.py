"""Geometry evaluation of a mesh against a reference mesh on the GPU: area-weighted surface samples (`tf_mesh_sample_surface`)
and exact point-to-mesh distances on the BVH (`tf_bvh_closest_point`, through mc_ops.RayTracer), reduced in fp64.  There is
no CPU path."""
from __future__ import annotations

import torch

from . import _lib
from ._lib import check, ptr, stream_ptr
from .ops import _f32c


def _mesh(vertices, triangles, what):
    """-> (vertices [V,3] fp32, triangles [T,3] int32), contiguous CUDA tensors; raises before any launch otherwise."""
    if not (torch.is_tensor(vertices) and torch.is_tensor(triangles) and vertices.is_cuda and triangles.is_cuda):
        raise RuntimeError(f"{what} needs CUDA tensors (tensoflow_b200 has no CPU path)")
    if vertices.dim() != 2 or vertices.shape[1] != 3 or triangles.dim() != 2 or triangles.shape[1] != 3:
        raise RuntimeError(f"{what} needs vertices [V,3] and triangles [T,3], got {list(vertices.shape)} and {list(triangles.shape)}")
    if triangles.shape[0] == 0 or vertices.shape[0] == 0:
        raise RuntimeError(f"{what}: empty mesh")
    if vertices.device != triangles.device:
        raise RuntimeError(f"{what}: vertices and triangles are on different devices")
    return _f32c(vertices), triangles.detach().to(torch.int32).contiguous()


def _face_cross(v, t):
    """(b - a) x (c - a) per triangle, fp64 [T,3] (twice the area times the unit normal)"""
    v = v.double()
    t = t.long()
    return torch.cross(v[t[:, 1]] - v[t[:, 0]], v[t[:, 2]] - v[t[:, 0]], dim=-1)


def _sample_surface_from(v, t, cdf, uniforms):
    """tf_mesh_sample_surface on prepared inputs: v [V,3] fp32, t [T,3] int32 (indices in range), cdf [T] fp64 inclusive and
    normalised, uniforms [n,3] fp64 in [0,1) -> (points [n,3] fp32, tri [n] int64, unit normals [n,3] fp32)."""
    n = uniforms.shape[0]
    pts = torch.empty(n, 3, device=v.device, dtype=torch.float32)
    tri = torch.empty(n, device=v.device, dtype=torch.int64)
    nrm = torch.empty(n, 3, device=v.device, dtype=torch.float32)
    check(_lib.load().tf_mesh_sample_surface(ptr(v), ptr(t), t.shape[0], ptr(cdf), ptr(uniforms), n, ptr(pts), ptr(tri), ptr(nrm),
                                             stream_ptr()), "tf_mesh_sample_surface")
    return pts, tri, nrm


def sample_surface(vertices, triangles, n: int, seed: int = 0):
    """n area-weighted samples of the mesh surface -> (points [n,3] fp32, triangle [n] int64, unit face normal [n,3] fp32), on the
    mesh's device.  Triangle areas and their fp64 cumulative sum are computed on the device; the uniforms are drawn from a
    torch.Generator seeded with `seed`, so a seed gives the same samples every run.  Raises RuntimeError on CPU tensors, an
    empty mesh, a triangle index out of range, or a mesh of zero or non-finite total area."""
    v, t = _mesh(vertices, triangles, "sample_surface")
    dev = v.device
    with torch.cuda.device(dev):
        cdf = torch.cumsum(0.5 * _face_cross(v, t.clamp(0, v.shape[0] - 1)).norm(dim=-1), 0)
        total, lo, hi = torch.stack([cdf[-1], t.min().double(), t.max().double()]).tolist()   # the one host read
        if lo < 0 or hi >= v.shape[0]:
            raise RuntimeError(f"sample_surface: triangle index out of range [0, {v.shape[0]})")
        if not (0.0 < total < float("inf")):
            raise RuntimeError(f"sample_surface: total area {total} is not positive and finite")
        cdf = cdf / cdf[-1]                                            # last element exactly 1
        g = torch.Generator(device=dev).manual_seed(int(seed))
        uniforms = torch.rand(int(n), 3, device=dev, dtype=torch.float64, generator=g)
        return _sample_surface_from(v, t, cdf, uniforms)


def evaluate_mesh(pred_vertices, pred_triangles, gt_vertices, gt_triangles, n_samples: int = 1_000_000,
                  thresholds=(0.005, 0.01, 0.02), seed: int = 0) -> dict:
    """Distance of a predicted mesh to a ground-truth mesh, from `n_samples` area-weighted samples of each (seeds `seed` for the
    prediction, `seed + 1` for the ground truth) and the exact distance of each sample to the OTHER mesh (closest point on
    its BVH).  Distances are point-to-mesh: the only sampling is that of the query points, so there is no second floor set by
    the spacing of a sampled reference set.  Reductions are in fp64.  Returns floats:

      accuracy            mean distance of the predicted samples to the ground-truth mesh
      completeness        mean distance of the ground-truth samples to the predicted mesh
      chamfer             (accuracy + completeness) / 2
      normal_consistency  mean over both directions of |n_sample . n_closest_face| (a closest face of zero area counts 0)
      precision, recall, fscore
                          dicts keyed by threshold tau (default 0.005, 0.01, 0.02, in the meshes' units): the fraction of
                          predicted (precision) / ground-truth (recall) samples at distance < tau, and 2PR / (P + R), 0 when
                          both are 0.

    The reference's eval_geo.py is not part of this repository, so these point-to-mesh definitions have not been checked
    against its formula (it may use sampled-set nearest neighbours and clip outliers); numbers may differ from it for that
    reason.  CUDA tensors only; each mesh needs more than 8 triangles (mc_ops.RayTracer)."""
    from .mc_ops import RayTracer
    pv, pt = _mesh(pred_vertices, pred_triangles, "evaluate_mesh (prediction)")
    gv, gt = _mesh(gt_vertices, gt_triangles, "evaluate_mesh (ground truth)")
    if pv.device != gv.device:
        raise RuntimeError("evaluate_mesh: the two meshes are on different devices")
    ps, _, pn = sample_surface(pv, pt, n_samples, seed)
    gs, _, gn = sample_surface(gv, gt, n_samples, seed + 1)
    with torch.cuda.device(pv.device):
        _, d_acc, t_acc = RayTracer(gv, gt).closest_point(ps)
        _, d_comp, t_comp = RayTracer(pv, pt).closest_point(gs)

    def unit_normals(v, t):
        c = _face_cross(v, t)
        ln = c.norm(dim=-1, keepdim=True)
        return torch.where(ln > 0, c / torch.where(ln > 0, ln, torch.ones_like(ln)), torch.zeros_like(c))

    nc = torch.cat([(pn.double() * unit_normals(gv, gt)[t_acc]).sum(-1).abs(),
                    (gn.double() * unit_normals(pv, pt)[t_comp]).sum(-1).abs()])
    d_acc, d_comp = d_acc.double(), d_comp.double()
    taus = [float(x) for x in thresholds]
    tau = torch.tensor(taus, device=pv.device, dtype=torch.float64)[:, None]
    stats = torch.cat([torch.stack([d_acc.mean(), d_comp.mean(), nc.mean()]),
                       (d_acc[None] < tau).double().mean(1), (d_comp[None] < tau).double().mean(1)]).tolist()
    acc, comp, normal = stats[:3]
    prec, rec = stats[3:3 + len(taus)], stats[3 + len(taus):]
    fscore = [2 * p * r / (p + r) if p + r > 0 else 0.0 for p, r in zip(prec, rec)]
    return {"accuracy": acc, "completeness": comp, "chamfer": 0.5 * (acc + comp), "normal_consistency": normal,
            "precision": dict(zip(taus, prec)), "recall": dict(zip(taus, rec)), "fscore": dict(zip(taus, fscore))}
