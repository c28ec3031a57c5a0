"""Mesh geometry on the GPU: evaluation against a reference mesh (area-weighted surface samples, `tf_mesh_sample_surface`, and
exact point-to-mesh distances on the BVH, `tf_bvh_closest_point` through mc_ops.RayTracer, reduced in fp64), connected
components (`tf_mesh_components`), quadric-error simplification (`tf_mesh_simplify`), and UV atlases with texture baking
(`tf_uv_atlas`, `tf_uv_texel_points`, `tf_uv_fill`).  There is no CPU path."""
from __future__ import annotations

import ctypes
from dataclasses import dataclass

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


@dataclass
class UVAtlas:
    """A UV atlas from `uv_atlas`, on the mesh's device.  Vertices are split along chart seams: output vertex i is the pair
    (vertex_index[i], chart) and sits at vertices[i] = the input position.

      vertices [V',3] fp32, triangles [T,3] int32 (input order), uv [V',2] fp32 in [0,1], vertex_index [V'] int64
      xy [V',2] fp32        texel-space coordinates in [0, R]: uv = xy / R; texture row j spans v in [j/R, (j+1)/R], column i
                            spans u in [i/R, (i+1)/R] (row 0 at v = 0: image writers that put row 0 at the top flip v)
      chart [T] int32       chart of each triangle, numbered by its smallest triangle
      texel_tri [R,R] int32 the triangle owning each texel (its centre lies inside it), -1 for none; [j, i] is row j, column i
      rects [C,4] int32     each chart's rectangle (x0, y0, w, h) in texels, padding included; rectangles are disjoint
      scale                 texels per world unit, the same for every chart
      resolution, padding, rounds (conflict rounds), steps (density trials)"""
    vertices: torch.Tensor
    triangles: torch.Tensor
    uv: torch.Tensor
    xy: torch.Tensor
    vertex_index: torch.Tensor
    chart: torch.Tensor
    texel_tri: torch.Tensor
    rects: torch.Tensor
    scale: float
    resolution: int
    padding: int
    rounds: int
    steps: int


def uv_atlas(vertices, triangles, resolution: int = 2048, padding: int = 2) -> UVAtlas:
    """A UV atlas of box-projection charts on the GPU (tf_uv_atlas; rules in include/tensoflow_b200.h) -> UVAtlas.

    Each triangle takes the axis direction (+-x, +-y, +-z) of its largest normal component, smoothed over edge neighbours in 4
    passes among the directions within 60 degrees of its normal; a chart is an edge-connected set of triangles of one
    direction, projected orthographically along it at one density for all charts (so stretch is at most 2 in one direction).
    Charts are packed as rectangles with `padding` texels on every side into an R x R atlas, next-fit decreasing height, at
    the largest density a bisection finds to fit.  A chart whose projection folds over itself (a texel centre covered twice)
    is split into single triangles and the atlas is laid out again, until every texel centre has at most one triangle.  The
    result is deterministic (bit-equal to oracle/torch_oracle_atlas.py).

    Raises ValueError for resolution outside [16, 16384] or padding outside [1, 16], and RuntimeError on CPU tensors, shapes
    other than [V,3] / [T,3], an empty mesh, non-integer triangles, 2^31 or more vertices or triangles, a triangle index out of
    range, non-finite vertices or a zero total area (one host read), all before any launch; RuntimeError when the charts do
    not fit in the atlas at any density (more charts than R x R holds)."""
    what = "uv_atlas"
    if isinstance(resolution, bool) or int(resolution) != resolution or not 16 <= int(resolution) <= 16384:
        raise ValueError(f"{what}: resolution must be an integer in [16, 16384], got {resolution}")
    if isinstance(padding, bool) or int(padding) != padding or not 1 <= int(padding) <= 16:
        raise ValueError(f"{what}: padding must be an integer in [1, 16], got {padding}")
    R, pad = int(resolution), int(padding)
    if torch.is_tensor(triangles) and (triangles.is_floating_point() or triangles.is_complex() or triangles.dtype == torch.bool):
        raise RuntimeError(f"{what} needs integer triangles, got {triangles.dtype}")
    for x, name in ((vertices, "vertices"), (triangles, "triangles")):
        if torch.is_tensor(x) and x.dim() == 2 and x.shape[0] >= 2 ** 31:
            raise RuntimeError(f"{what}: {x.shape[0]} {name}, the kernel indexes fewer than 2^31")
    if torch.is_tensor(triangles) and triangles.dim() == 2 and 3 * triangles.shape[0] >= 2 ** 31:
        raise RuntimeError(f"{what}: {triangles.shape[0]} triangles, the sorts need 3 T < 2^31")
    v, t = _mesh(vertices, triangles, what)
    V, T = v.shape[0], t.shape[0]
    lib = _lib.load()
    dev = v.device
    with torch.cuda.device(dev):
        flat = triangles.detach().reshape(-1)
        lo, hi = flat.min().to(torch.int64), flat.max().to(torch.int64)
        finite = torch.isfinite(v).all()
        area = 0.5 * _face_cross(v, t.clamp(0, V - 1)).norm(dim=-1).sum()
        lo, hi, finite, area = torch.stack([lo.double(), hi.double(), finite.double(), area]).tolist()   # the one host read
        if lo < 0 or hi >= V:
            raise RuntimeError(f"{what}: triangle index out of range (indices span [{int(lo)}, {int(hi)}], {V} vertices)")
        if not finite:
            raise RuntimeError(f"{what}: non-finite vertex coordinates")
        if not area > 0:
            raise RuntimeError(f"{what}: total area {area} is not positive")
        ws_bytes = ctypes.c_size_t()
        check(lib.tf_uv_atlas_sizes(V, T, R, ctypes.byref(ws_bytes)), "tf_uv_atlas_sizes")
        ws = torch.empty(ws_bytes.value, device=dev, dtype=torch.uint8)
        chart = torch.empty(T, device=dev, dtype=torch.int32)
        tri = torch.empty(T, 3, device=dev, dtype=torch.int32)
        vidx = torch.empty(3 * T, device=dev, dtype=torch.int64)
        xy = torch.empty(3 * T, 2, device=dev, dtype=torch.float32)
        texel_tri = torch.empty(R, R, device=dev, dtype=torch.int32)
        rects = torch.empty(T, 4, device=dev, dtype=torch.int32)
        scale, n_v, n_c = ctypes.c_double(), ctypes.c_int64(), ctypes.c_int64()
        rounds, steps = ctypes.c_int32(), ctypes.c_int32()
        check(lib.tf_uv_atlas(ptr(v), V, ptr(t), T, R, pad, ptr(ws), ws_bytes.value, ptr(chart), ptr(tri), ptr(vidx), ptr(xy),
                              ptr(texel_tri), ptr(rects), ctypes.byref(scale), ctypes.byref(n_v), ctypes.byref(n_c),
                              ctypes.byref(rounds), ctypes.byref(steps), stream_ptr()), "tf_uv_atlas")
        del ws
        vidx, xy = vidx[:n_v.value].clone(), xy[:n_v.value].clone()
        return UVAtlas(vertices=v[vidx], triangles=tri, uv=xy / R, xy=xy, vertex_index=vidx, chart=chart, texel_tri=texel_tri,
                       rects=rects[:n_c.value].clone(), scale=scale.value, resolution=R, padding=pad, rounds=rounds.value,
                       steps=steps.value)


def texel_points(atlas: UVAtlas):
    """-> (texels [n] int64, the covered texels j * R + i in row order, and points [n,3] fp32 on their owning triangles): the
    point at the barycentric coordinates of each texel centre, evaluated in fp64 and rounded once (tf_uv_texel_points).  One
    host read (the count)."""
    R = atlas.resolution
    with torch.cuda.device(atlas.texel_tri.device):
        texels = torch.nonzero(atlas.texel_tri.reshape(-1) >= 0)[:, 0]
        pts = torch.empty(texels.shape[0], 3, device=texels.device, dtype=torch.float32)
        check(_lib.load().tf_uv_texel_points(ptr(atlas.vertices), ptr(atlas.triangles), ptr(atlas.xy), ptr(atlas.texel_tri), R,
                                             ptr(texels), texels.shape[0], ptr(pts), stream_ptr()), "tf_uv_texel_points")
    return texels, pts


def bake_texture(atlas: UVAtlas, fn, channels: int, chunk: int = 2 ** 20):
    """Bake fn over the atlas -> (texture [R,R,channels] fp32, mask [R,R] bool of the texels covered before dilation).

    fn(points [n,3] fp32 CUDA) -> [n, channels] runs on the texel points of `texel_points`, at most `chunk` at a time.  The
    values are scattered to their texels, then `atlas.padding` dilation passes fill each empty texel of a chart's rectangle
    that touches filled ones with the mean of its filled 8-neighbours of that chart (tf_uv_fill), so bilinear lookups inside a
    chart never read another chart.  Row j of the texture spans v in [j/R, (j+1)/R] (see UVAtlas).  Raises RuntimeError when
    fn returns another shape or non-finite values, and ValueError for channels < 1 or chunk < 1."""
    if isinstance(channels, bool) or int(channels) != channels or int(channels) < 1:
        raise ValueError(f"bake_texture: channels must be an integer >= 1, got {channels}")
    if int(chunk) < 1:
        raise ValueError(f"bake_texture: chunk must be >= 1, got {chunk}")
    C, R = int(channels), atlas.resolution
    lib = _lib.load()
    texels, pts = texel_points(atlas)
    dev = pts.device
    with torch.cuda.device(dev):
        values = torch.empty(pts.shape[0], C, device=dev, dtype=torch.float32)
        for s in range(0, pts.shape[0], int(chunk)):
            out = fn(pts[s:s + int(chunk)])
            if not torch.is_tensor(out) or tuple(out.shape) != (min(int(chunk), pts.shape[0] - s), C):
                raise RuntimeError(f"bake_texture: fn must return [n, {C}], got "
                                   f"{list(out.shape) if torch.is_tensor(out) else type(out).__name__}")
            values[s:s + out.shape[0]] = out.detach()
        if not bool(torch.isfinite(values).all()):
            raise RuntimeError("bake_texture: fn returned a non-finite value")
        ws_bytes = ctypes.c_size_t()
        check(lib.tf_uv_fill_sizes(R, C, ctypes.byref(ws_bytes)), "tf_uv_fill_sizes")
        ws = torch.empty(ws_bytes.value, device=dev, dtype=torch.uint8)
        tex = torch.empty(R, R, C, device=dev, dtype=torch.float32)
        check(lib.tf_uv_fill(ptr(values), ptr(texels), texels.shape[0], C, ptr(atlas.texel_tri), ptr(atlas.chart), ptr(atlas.rects),
                             R, atlas.padding, ptr(ws), ws_bytes.value, ptr(tex), stream_ptr()), "tf_uv_fill")
        return tex, atlas.texel_tri >= 0


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
