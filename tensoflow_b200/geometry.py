"""Mesh geometry on the GPU: evaluation against a reference mesh (area-weighted surface samples, `tf_mesh_sample_surface`, and
exact point-to-mesh distances on the BVH, `tf_bvh_closest_point` through mc_ops.RayTracer, reduced in fp64), connected
components (`tf_mesh_components`) and quadric-error simplification (`tf_mesh_simplify`).  There is no CPU path."""
from __future__ import annotations

import ctypes

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


def _components(vertices, triangles, what):
    """Checks, then tf_mesh_components -> (triangles [T,3] int32, root [V] int32, tri_count [V] int32) on the mesh's device.
    Every refusal comes before any launch; the index range costs one host read."""
    if torch.is_tensor(triangles) and (triangles.is_floating_point() or triangles.is_complex() or triangles.dtype == torch.bool):
        raise RuntimeError(f"{what} needs integer triangles, got {triangles.dtype}")
    if torch.is_tensor(vertices) and vertices.dim() == 2 and vertices.shape[0] >= 2 ** 31:
        raise RuntimeError(f"{what}: {vertices.shape[0]} vertices, the kernel indexes fewer than 2^31")
    v, t = _mesh(vertices, triangles, what)
    V = v.shape[0]
    with torch.cuda.device(v.device):
        flat = triangles.detach().reshape(-1)
        lo, hi = torch.stack([flat.min(), flat.max()]).to(torch.int64).tolist()           # the one host read
        if lo < 0 or hi >= V:
            raise RuntimeError(f"{what}: triangle index out of range (indices span [{lo}, {hi}], {V} vertices)")
        root = torch.empty(V, device=v.device, dtype=torch.int32)
        tri_count = torch.empty(V, device=v.device, dtype=torch.int32)
        check(_lib.load().tf_mesh_components(ptr(t), t.shape[0], V, ptr(root), ptr(tri_count), stream_ptr()), "tf_mesh_components")
    return t, root, tri_count


def mesh_components(vertices, triangles):
    """Connected components of a mesh (vertices joined by triangle edges) -> (root [V] int32, tri_count [V] int32) on the mesh's
    device: root[v] is the smallest vertex index of v's component (a vertex no triangle references is a component of its own),
    tri_count[r] the number of triangles of the component whose root is r, 0 for every vertex that is not a root.  Lock-free
    union-find on the GPU (tf_mesh_components); the result does not depend on scheduling.  Raises RuntimeError, before any
    launch, on CPU tensors, shapes other than [V,3] / [T,3], an empty mesh, non-integer triangles, 2^31 or more vertices, or a
    triangle index out of range (one host read)."""
    _, root, tri_count = _components(vertices, triangles, "mesh_components")
    return root, tri_count


def remove_small_components(vertices, triangles, min_fraction: float):
    """Drop the small connected components of a mesh ("floaters") -> (vertices [V',3], triangles [T',3] int32) on its device.
    A triangle is kept iff its component has tri_count >= min_fraction * (the largest component's tri_count), compared in
    fp64; min_fraction = 1.0 keeps the largest component and every component tied with it.  Kept triangles keep their order,
    the vertices they reference keep theirs (and their dtype), and the indices are renumbered.  Vertices that no triangle
    references are dropped.  Raises ValueError for min_fraction outside (0, 1], and what mesh_components raises, before any
    launch.  Two host reads: the index range before the union-find, the output sizes after it."""
    f = float(min_fraction)
    if not 0.0 < f <= 1.0:
        raise ValueError(f"remove_small_components: min_fraction must lie in (0, 1], got {min_fraction}")
    t, root, tri_count = _components(vertices, triangles, "remove_small_components")
    with torch.cuda.device(t.device):
        # an unreferenced vertex has tri_count 0 < f * max, so it goes; a component's vertices and triangles go together
        keep_v = tri_count[root.long()].double() >= f * tri_count.max().double()
        keep_t = keep_v[t[:, 0].long()]
        new_index = torch.cumsum(keep_v, 0, dtype=torch.int32) - 1
        n_v, n_t = torch.stack([keep_v.sum(), keep_t.sum()]).tolist()                      # the second host read
        vi = torch.nonzero_static(keep_v, size=n_v).reshape(-1)
        ti = torch.nonzero_static(keep_t, size=n_t).reshape(-1)
        return vertices.detach()[vi], new_index[t[ti].long()]


def _simplify_limits(target_triangles, max_error, what):
    """-> (target int, max_error float, +inf for None); ValueError on a negative target or a negative / non-finite bound"""
    if isinstance(target_triangles, bool) or int(target_triangles) != target_triangles or int(target_triangles) < 0:
        raise ValueError(f"{what}: target_triangles must be an integer >= 0, got {target_triangles}")
    err = float("inf") if max_error is None else float(max_error)
    if max_error is not None and not (0.0 <= err < float("inf")):
        raise ValueError(f"{what}: max_error must be finite and >= 0 (None for no bound), got {max_error}")
    return int(target_triangles), err


def simplify_mesh(vertices, triangles, target_triangles: int, max_error: float | None = None):
    """Quadric-error edge collapse on the GPU (tf_mesh_simplify) -> (vertices [V',3] fp32, triangles [T',3] int32) on the mesh's
    device.  Collapses run in rounds of edges with vertex-disjoint closed 1-rings until T' <= target_triangles + 1 or no edge
    may collapse; T' is never below the target.  max_error (None: no bound) bounds sqrt of each collapse's quadric cost, which
    bounds the distance of the new vertex to the plane of every input face merged into it.  Open boundaries and non-manifold
    vertices are kept bit for bit, surviving triangles keep their order, and the referenced vertices keep theirs.  The result
    is deterministic (bit-equal to oracle/torch_oracle_simplify.py).  Raises ValueError on a negative target or a negative or
    non-finite max_error, and RuntimeError on CPU tensors, shapes other than [V,3] / [T,3], an empty mesh, non-integer
    triangles, 2^31 or more vertices or triangles, or a triangle index out of range (one host read), all before any launch.
    The rounds read one count each to the host."""
    return _simplify(vertices, triangles, target_triangles, max_error)[:2]


def _simplify(vertices, triangles, target_triangles, max_error):
    """simplify_mesh -> (vertices, triangles, the number of rounds that collapsed something)"""
    what = "simplify_mesh"
    target, max_error = _simplify_limits(target_triangles, max_error, what)
    if torch.is_tensor(triangles) and (triangles.is_floating_point() or triangles.is_complex() or triangles.dtype == torch.bool):
        raise RuntimeError(f"{what} needs integer triangles, got {triangles.dtype}")
    for x, name in ((vertices, "vertices"), (triangles, "triangles")):
        if torch.is_tensor(x) and x.dim() == 2 and x.shape[0] >= 2 ** 31:
            raise RuntimeError(f"{what}: {x.shape[0]} {name}, the kernel indexes fewer than 2^31")
    v, t = _mesh(vertices, triangles, what)
    V, T = v.shape[0], t.shape[0]
    lib = _lib.load()
    with torch.cuda.device(v.device):
        flat = triangles.detach().reshape(-1)
        lo, hi = torch.stack([flat.min(), flat.max()]).to(torch.int64).tolist()           # the one host read before the rounds
        if lo < 0 or hi >= V:
            raise RuntimeError(f"{what}: triangle index out of range (indices span [{lo}, {hi}], {V} vertices)")
        ws_bytes = ctypes.c_size_t()
        check(lib.tf_mesh_simplify_sizes(V, T, ctypes.byref(ws_bytes)), "tf_mesh_simplify_sizes")
        ws = torch.empty(ws_bytes.value, device=v.device, dtype=torch.uint8)
        out_v = torch.empty(V, 3, device=v.device, dtype=torch.float32)
        out_t = torch.empty(T, 3, device=v.device, dtype=torch.int32)
        n_v, n_t, rounds = ctypes.c_int64(), ctypes.c_int64(), ctypes.c_int32()
        check(lib.tf_mesh_simplify(ptr(v), V, ptr(t), T, target, max_error, ptr(ws), ws_bytes.value, ptr(out_v), ptr(out_t),
                                   ctypes.byref(n_v), ctypes.byref(n_t), ctypes.byref(rounds), stream_ptr()), "tf_mesh_simplify")
        del ws
        return out_v[:n_v.value].clone(), out_t[:n_t.value].clone(), rounds.value


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
