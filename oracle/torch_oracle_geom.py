"""TEST INFRASTRUCTURE ONLY (never imported by tensoflow_b200/).  fp64, device-agnostic restatement of the geometry-evaluation
kernels of include/tensoflow_b200.h: tf_bvh_closest_point as a brute force over every triangle (no BVH) and
tf_mesh_sample_surface from the same CDF and uniforms.

Conventions shared with the kernels:
  * per triangle (a, b, c), Ericson's 7-region closest-point test (Real-Time Collision Detection 5.1.5) with ab = b - a,
    ac = c - a; a triangle whose height is below 2^-24 of its longest edge (|ab x ac|^2 <= 2^-48 max|edge|^4) is measured
    through its three edges, a zero-length edge being its vertex;
  * the smaller squared distance wins, an exact tie goes to the smaller triangle index;
  * sampling: triangle = first t with cdf[t] > u0, point (1 - sqrt(u1)) a + sqrt(u1)(1 - u2) b + sqrt(u1) u2 c, normal the unit
    (b - a) x (c - a)."""
import torch


def _dot(x, y):
    return (x * y).sum(-1)


def _sdiv(num, den):
    return torch.where(den > 0, num / torch.where(den > 0, den, torch.ones_like(den)), torch.zeros_like(num))


def _clamp01(x):
    return x.clamp(0.0, 1.0)


def triangle_closest(ap, e1, e2):
    """ap [..., 3] = p - a, e1 = b - a, e2 = c - a (broadcast together) -> (squared distance [...], r [..., 3] = p - closest point)."""
    ap, e1, e2 = torch.broadcast_tensors(ap, e1, e2)
    n = torch.cross(e1, e2, dim=-1)
    nn = _dot(n, n)
    e3 = e2 - e1
    l1, l2, l3 = _dot(e1, e1), _dot(e2, e2), _dot(e3, e3)
    lmax = torch.maximum(l1, torch.maximum(l2, l3))
    bp, cp = ap - e1, ap - e2
    d1, d2 = _dot(e1, ap), _dot(e2, ap)
    d3, d4 = _dot(e1, bp), _dot(e2, bp)
    d5, d6 = _dot(e1, cp), _dot(e2, cp)
    vc = _dot(n, torch.cross(e1, ap, dim=-1))
    vb = _dot(n, torch.cross(ap, e2, dim=-1))
    va = _dot(n, torch.cross(bp, cp, dim=-1))

    def along(s, e, l):
        return s - _clamp01(_sdiv(_dot(s, e), l))[..., None] * e

    # regions in increasing priority: each later assignment overrides the earlier ones where its condition holds
    r = _sdiv(_dot(ap, n), nn)[..., None] * n                                                   # face
    r = torch.where(((va <= 0) & (d4 - d3 >= 0) & (d5 - d6 >= 0))[..., None], along(bp, e3, l3), r)   # edge bc
    r = torch.where(((vb <= 0) & (d2 >= 0) & (d6 <= 0))[..., None], along(ap, e2, l2), r)        # edge ac
    r = torch.where(((d6 >= 0) & (d5 <= d6))[..., None], cp, r)                                  # vertex c
    r = torch.where(((vc <= 0) & (d1 >= 0) & (d3 <= 0))[..., None], along(ap, e1, l1), r)        # edge ab
    r = torch.where(((d3 >= 0) & (d4 <= d3))[..., None], bp, r)                                  # vertex b
    r = torch.where(((d1 <= 0) & (d2 <= 0))[..., None], ap, r)                                   # vertex a
    # degenerate: nearest of the edges ab, ac, bc (a later one only when strictly nearer)
    seg = [along(ap, e1, l1), along(ap, e2, l2), along(bp, e3, l3)]
    rs = seg[0]
    for s in seg[1:]:
        rs = torch.where((_dot(s, s) < _dot(rs, rs))[..., None], s, rs)
    r = torch.where((nn > 2.0 ** -48 * lmax * lmax)[..., None], r, rs)
    return _dot(r, r), r


def closest_point(points, vertices, triangles, point_chunk=4096, tri_chunk=4096):
    """Brute force over every triangle, fp64 on the points' device -> (closest [n,3], dist [n], tri [n] int64, second [n]), where
    `second` is the distance to the nearest OTHER triangle (inf for a one-triangle mesh)."""
    dev = points.device
    p = points.detach().to(torch.float64).reshape(-1, 3)
    v = vertices.detach().to(device=dev, dtype=torch.float64)
    t = triangles.detach().to(device=dev, dtype=torch.int64)
    a, b, c = v[t[:, 0]], v[t[:, 1]], v[t[:, 2]]
    e1, e2 = b - a, c - a
    T = t.shape[0]
    out_q = torch.empty_like(p)
    out_d = torch.empty(p.shape[0], dtype=torch.float64, device=dev)
    out_t = torch.empty(p.shape[0], dtype=torch.int64, device=dev)
    out_s = torch.empty(p.shape[0], dtype=torch.float64, device=dev)
    for i0 in range(0, p.shape[0], point_chunk):
        pc = p[i0:i0 + point_chunk]
        m = pc.shape[0]
        best = torch.full((m,), float("inf"), dtype=torch.float64, device=dev)
        second = best.clone()
        best_t = torch.zeros(m, dtype=torch.int64, device=dev)
        best_r = torch.zeros(m, 3, dtype=torch.float64, device=dev)
        for j0 in range(0, T, tri_chunk):
            sl = slice(j0, j0 + tri_chunk)
            d2, r = triangle_closest(pc[:, None, :] - a[None, sl], e1[None, sl], e2[None, sl])
            k = min(2, d2.shape[1])
            vals, idx = torch.topk(d2, k, dim=1, largest=False, sorted=True)
            cmin = vals[:, 0]
            carg = torch.argmin(d2, dim=1)                      # first (smallest index) of an exact tie
            c2 = vals[:, 1] if k > 1 else torch.full_like(cmin, float("inf"))
            upd = cmin < best                                   # earlier chunks hold smaller indices: they keep ties
            second = torch.where(upd, torch.minimum(best, c2), torch.minimum(second, cmin))
            best_r = torch.where(upd[:, None], r[torch.arange(m, device=dev), carg], best_r)
            best_t = torch.where(upd, carg + j0, best_t)
            best = torch.where(upd, cmin, best)
        out_q[i0:i0 + m] = pc - best_r
        out_d[i0:i0 + m] = best.sqrt()
        out_t[i0:i0 + m] = best_t
        out_s[i0:i0 + m] = second.sqrt()
    return out_q, out_d, out_t, out_s


def area_cdf(vertices, triangles):
    """Inclusive normalised cumulative triangle area [T] fp64 (the computation tensoflow_b200.geometry.sample_surface makes)."""
    v = vertices.detach().to(torch.float64)
    t = triangles.detach().to(device=v.device, dtype=torch.int64)
    area = 0.5 * torch.cross(v[t[:, 1]] - v[t[:, 0]], v[t[:, 2]] - v[t[:, 0]], dim=-1).norm(dim=-1)
    cdf = torch.cumsum(area, 0)
    return cdf / cdf[-1]


def sample_surface(vertices, triangles, cdf, uniforms):
    """-> (points [n,3] fp64, tri [n] int64, unit normals [n,3] fp64) from the inclusive CDF [T] and uniforms [n,3] in [0,1)."""
    v = vertices.detach().to(torch.float64)
    t = triangles.detach().to(device=v.device, dtype=torch.int64)
    u = uniforms.detach().to(device=v.device, dtype=torch.float64)
    cdf = cdf.detach().to(device=v.device, dtype=torch.float64)
    tri = torch.searchsorted(cdf, u[:, 0].contiguous(), right=True).clamp_max(t.shape[0] - 1)
    a, b, c = v[t[tri, 0]], v[t[tri, 1]], v[t[tri, 2]]
    e1, e2 = b - a, c - a
    s = u[:, 1:2].sqrt()
    pts = a + (s * (1 - u[:, 2:3])) * e1 + (s * u[:, 2:3]) * e2
    n = torch.cross(e1, e2, dim=-1)
    ln = n.norm(dim=-1, keepdim=True)
    return pts, tri, torch.where(ln > 0, n / torch.where(ln > 0, ln, torch.ones_like(ln)), torch.zeros_like(n))
