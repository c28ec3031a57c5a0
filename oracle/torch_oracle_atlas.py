"""TEST INFRASTRUCTURE ONLY (never imported by tensoflow_b200/).  numpy restatement of tf_uv_atlas, tf_uv_texel_points and tf_uv_fill
(include/tensoflow_b200.h, tensoflow_b200/csrc/uv_atlas.cu): a UV atlas of box-projection charts and texture baking.  Every
floating-point operation below is an elementwise numpy op in the kernels' order (no `@`, einsum or BLAS, no fused multiply-add),
so the results are bit-equal to the device's.

The rules, on positions P [V,3] fp32 and faces F [T,3]:

  * normal n = (b - a) x (c - a) in fp64, len = sqrt((nx nx + ny ny) + nz nz) (twice the area).  Class 2k + (n_k < 0) with k the
    axis of the largest |n_k|, ties to the lower axis.  Class c (axis c // 2, sign + for even c) is allowed for the face iff
    sign n_k >= len / 2 (|n^ . axis| >= 1/2 on the front side; a face of zero length allows every class).
  * half-edges (min(a, b) << 32 | max(a, b), 3 f + k) for corner k -> k + 1, stably sorted by key: each edge's run lists its faces
    in ascending order.  The neighbours of f are, for k = 0, 1, 2, the other members of the run of its half-edge k, in run order.
  * 4 Jacobi smoothing passes: acc[c] = len_f added to the own class, then len_g of every neighbour g (in the order above) added
    to g's class; the new class is the allowed class of the largest acc, the own class on ties, then the lower index.
  * charts: faces joined when they share an edge and a class and neither is "solo"; the root of a chart is its smallest face and
    charts are numbered by root.  Solo faces (those found in a conflict, below) are charts of their own.
  * projection of a corner of chart class c, axis k: (u, w) = (p[(k+1)%3], p[(k+2)%3]) for even c, (p[(k+2)%3], p[(k+1)%3]) for
    odd c.  Chart bounding boxes in fp32.
  * density: q_f = rint(|n_k| / max |n_k| * 2^32) (k the face's class axis) summed in uint64; A = (S * max) * 2^-33 (the
    projected area); s0 = R / sqrt(A).  rect_in = max(1, ceil((umax - umin) * s)) (capped at R + 1) per axis, rect = rect_in +
    2 padding.  Rects sorted by (h desc, w desc, chart asc) and packed next-fit decreasing height into shelves of width R; they
    fit when no w exceeds R and the last shelf ends at y <= R.  s = s0 if it fits, else 20 bisection steps on (0, s0] from lo = 0,
    hi = s0 with mid = (lo + hi) * 0.5, keeping lo.  lo = 0 means the charts do not fit.
  * texel coordinates of a corner: x = fp32((x0 + padding) + (u - umin) * s), y likewise with w, fp64 before the one rounding.
  * coverage of texel (i, j): the centre (i + 1/2, j + 1/2) inside the triangle.  Edge functions are evaluated from the endpoint
    that is smaller in (x, y) order (negated for the other direction), so a shared edge gives both faces the same value.  A face
    of signed area E_ab(c) < 0 is taken as (a, c, b); area 0 covers nothing.  Inside: E > 0 on all three edges, or E = 0 on a
    top-left edge (dy < 0, or dy = 0 and dx < 0).
  * conflict: a centre covered twice makes every face covering it solo; the charts, density, packing and coverage are redone
    until no centre is covered twice.  A chart covering no centre gets the texel floor of its root face's texel centroid ((x0 + x1)
    + x2) * fp64(1/3), clamped into its rectangle's interior, owned by the root face.
  * output vertices: the unique (vertex, chart) pairs in (vertex, chart) order; uv = fp32(x / R), fp32(y / R).
  * texel points: barycentrics of the centre from fp64 edge functions over the signed area, clamped at 0 and renormalised (1/3
    each when the area or their sum is 0), point = (la Pa + lb Pb) + lc Pc rounded once to fp32.
  * fill: values scattered to their texels; `padding` dilation passes in which an empty texel inside the rectangle of a filled
    8-neighbour's chart takes the fp32 mean of those neighbours, summed in row order (dy, then dx, from -1), divided by their
    count."""
import numpy as np

SMOOTH_PASSES = 4
BISECTION_STEPS = 20
NEIGHBOURS = [(dx, dy) for dy in (-1, 0, 1) for dx in (-1, 0, 1) if (dx, dy) != (0, 0)]


class AtlasError(RuntimeError):
    pass


def _cross(e1, e2):
    return np.stack([e1[..., 1] * e2[..., 2] - e1[..., 2] * e2[..., 1],
                     e1[..., 2] * e2[..., 0] - e1[..., 0] * e2[..., 2],
                     e1[..., 0] * e2[..., 1] - e1[..., 1] * e2[..., 0]], -1)


def face_normals(P, F):
    p = P.astype(np.float64)[F]
    n = _cross(p[:, 1] - p[:, 0], p[:, 2] - p[:, 0])
    ln = np.sqrt((n[:, 0] * n[:, 0] + n[:, 1] * n[:, 1]) + n[:, 2] * n[:, 2])
    return n, ln


def initial_classes(n):
    a = np.abs(n)
    k = np.zeros(n.shape[0], np.int64)
    k = np.where(a[:, 1] > a[np.arange(len(k)), k], 1, k)
    k = np.where(a[:, 2] > a[np.arange(len(k)), k], 2, k)
    return 2 * k + (n[np.arange(len(k)), k] < 0)


def allowed_classes(n, ln):
    cols = []
    for c in range(6):
        comp = n[:, c // 2] if c % 2 == 0 else -n[:, c // 2]
        cols.append(comp >= ln * 0.5)
    return np.stack(cols, 1)


def half_edges(F):
    """-> (sorted keys [3T], sorted half-edge ids [3T], position of each half-edge [3T], run start, run end per position)"""
    T = F.shape[0]
    a = F.astype(np.int64)
    b = a[:, [1, 2, 0]]
    key = ((np.minimum(a, b) << 32) | np.maximum(a, b)).reshape(-1)
    order = np.argsort(key, kind="stable")
    sk = key[order]
    pos = np.empty(3 * T, np.int64)
    pos[order] = np.arange(3 * T)
    head = np.ones(3 * T, bool)
    head[1:] = sk[1:] != sk[:-1]
    start = np.maximum.accumulate(np.where(head, np.arange(3 * T), 0))
    tail = np.ones(3 * T, bool)
    tail[:-1] = sk[1:] != sk[:-1]
    end = np.minimum.accumulate(np.where(tail, np.arange(3 * T), 3 * T)[::-1])[::-1] + 1
    return sk, order, pos, start, end


def smooth(cls, ln, allowed, he):
    _, order, pos, start, end = he
    T = cls.shape[0]
    face = order // 3
    maxrun = int((end - start).max())
    f_all = np.arange(T)
    for _ in range(SMOOTH_PASSES):
        acc = np.zeros((T, 6))
        acc[f_all, cls] = acc[f_all, cls] + ln
        for k in range(3):
            p = pos[3 * f_all + k]
            for j in range(maxrun):
                q = start[p] + j
                ok = (q < end[p]) & (q != p)
                f, g = f_all[ok], face[q[ok]]
                acc[f, cls[g]] = acc[f, cls[g]] + ln[g]
        best = cls.copy()
        bv = acc[f_all, cls]
        for c in range(6):
            take = allowed[:, c] & (acc[:, c] > bv)
            best = np.where(take, c, best)
            bv = np.where(take, acc[:, c], bv)
        cls = best
    return cls


def charts(cls, solo, he):
    """-> chart index per face (numbered by root), root face per chart"""
    from scipy.sparse import coo_matrix
    from scipy.sparse.csgraph import connected_components
    _, order, _, start, end = he
    T = cls.shape[0]
    face = order // 3
    rows, cols = [], []
    maxrun = int((end - start).max())
    p = np.arange(face.shape[0])
    for j in range(1, maxrun):
        q = p + j
        ok = q < end
        f, g = face[p[ok]], face[q[ok]]
        keep = (cls[f] == cls[g]) & ~solo[f] & ~solo[g] & (f != g)
        rows.append(f[keep])
        cols.append(g[keep])
    r = np.concatenate(rows) if rows else np.zeros(0, np.int64)
    c = np.concatenate(cols) if cols else np.zeros(0, np.int64)
    g = coo_matrix((np.ones(r.shape[0]), (r, c)), shape=(T, T))
    _, lab = connected_components(g, directed=False)
    root_of_label = np.full(lab.max() + 1, T, np.int64)
    np.minimum.at(root_of_label, lab, np.arange(T))
    root = root_of_label[lab]
    roots = np.unique(root)
    chart = np.searchsorted(roots, root)
    return chart, roots


def project(P, F, chart_cls_of_face):
    c = chart_cls_of_face
    k = c // 2
    i1, i2 = (k + 1) % 3, (k + 2) % 3
    iu = np.where(c % 2 == 0, i1, i2)[:, None]
    iw = np.where(c % 2 == 0, i2, i1)[:, None]
    pf = P[F]                                                       # [T,3,3] fp32
    u = np.take_along_axis(pf, iu[:, :, None].repeat(3, 1), 2)[..., 0]
    w = np.take_along_axis(pf, iw[:, :, None].repeat(3, 1), 2)[..., 0]
    return u, w                                                     # [T,3] fp32


def density_bound(n, cls, R):
    k = cls // 2
    a = np.abs(n[np.arange(n.shape[0]), k])
    amax = a.max()
    if not amax > 0:
        raise AtlasError("zero projected area")
    q = np.rint((a / amax) * 4294967296.0).astype(np.uint64)
    S = np.uint64(0)
    for x in np.array_split(q, max(1, q.shape[0] // 65536)):      # exact in uint64
        S = S + x.sum(dtype=np.uint64)
    A = (np.float64(S) * amax) * 2.0 ** -33
    return np.float64(R) / np.sqrt(A)


def rect_dims(bb, s, R, pad):
    """bb [C,4] fp32 (umin, umax, wmin, wmax) -> (w, h) int64 with padding"""
    out = []
    for lo, hi in ((0, 1), (2, 3)):
        t = (bb[:, hi].astype(np.float64) - bb[:, lo].astype(np.float64)) * s
        d = np.ceil(np.minimum(t, R + 1.0)).astype(np.int64)
        out.append(np.maximum(d, 1) + 2 * pad)
    return out[0], out[1]


def nfdh(w, h, R):
    """-> (fits, x0 [C], y0 [C])"""
    C = w.shape[0]
    order = np.lexsort((np.arange(C), -w, -h))
    x0 = np.zeros(C, np.int64)
    y0 = np.zeros(C, np.int64)
    x = y = shelf = 0
    fits = True
    for c in order.tolist():
        wc, hc = int(w[c]), int(h[c])
        if wc > R:
            fits = False
            break
        if x + wc > R:
            y += shelf
            x = 0
            shelf = 0
        if shelf == 0:
            shelf = hc
        x0[c], y0[c] = x, y
        x += wc
        if y + shelf > R:
            fits = False
            break
    return fits, x0, y0


def choose_density(bb, s0, R, pad):
    steps = 1
    w, h = rect_dims(bb, s0, R, pad)
    if nfdh(w, h, R)[0]:
        return s0, steps
    lo, hi = 0.0, s0
    for _ in range(BISECTION_STEPS):
        mid = (lo + hi) * 0.5
        w, h = rect_dims(bb, mid, R, pad)
        steps += 1
        if nfdh(w, h, R)[0]:
            lo = mid
        else:
            hi = mid
    if lo == 0.0:
        raise AtlasError(f"the charts do not fit in a {R}x{R} atlas")
    return np.float64(lo), steps


def _edge(px_, py_, qx, qy, cx, cy):
    """canonical edge function of the directed edge p -> q at (cx, cy) -> (E, dx, dy), fp64 arrays"""
    base_p = (px_ < qx) | ((px_ == qx) & (py_ <= qy))
    bx, by = np.where(base_p, px_, qx), np.where(base_p, py_, qy)
    ox, oy = np.where(base_p, qx, px_), np.where(base_p, qy, py_)
    ex, ey = ox - bx, oy - by
    e = ex * (cy - by) - ey * (cx - bx)
    sg = np.where(base_p, 1.0, -1.0)
    return sg * e, sg * ex, sg * ey


def _inside(e, dx, dy):
    return (e > 0) | ((e == 0) & ((dy < 0) | ((dy == 0) & (dx < 0))))


def coverage(xy, R, chunk=1 << 22):
    """xy [T,3,2] fp32 texel-space corners -> (face [m], texel [m]) of every covered centre, face-major"""
    x = xy[..., 0].astype(np.float64)
    y = xy[..., 1].astype(np.float64)
    i0 = np.clip(np.ceil(x.min(1) - 0.5), 0, R - 1).astype(np.int64)
    i1 = np.clip(np.floor(x.max(1) - 0.5), -1, R - 1).astype(np.int64)
    j0 = np.clip(np.ceil(y.min(1) - 0.5), 0, R - 1).astype(np.int64)
    j1 = np.clip(np.floor(y.max(1) - 0.5), -1, R - 1).astype(np.int64)
    ni, nj = np.maximum(i1 - i0 + 1, 0), np.maximum(j1 - j0 + 1, 0)
    cnt = ni * nj
    area, _, _ = _edge(x[:, 0], y[:, 0], x[:, 1], y[:, 1], x[:, 2], y[:, 2])
    flip = area < 0
    bxs = np.where(flip, x[:, 2], x[:, 1]); bys = np.where(flip, y[:, 2], y[:, 1])
    cxs = np.where(flip, x[:, 1], x[:, 2]); cys = np.where(flip, y[:, 1], y[:, 2])
    faces, texels = [], []
    f_all = np.repeat(np.arange(x.shape[0]), cnt)
    off = np.concatenate([[0], np.cumsum(cnt)])
    for s in range(0, f_all.shape[0], chunk):
        f = f_all[s:s + chunk]
        r = np.arange(s, s + f.shape[0]) - off[f]
        ii = i0[f] + r % ni[f]
        jj = j0[f] + r // ni[f]
        cx, cy = ii + 0.5, jj + 0.5
        ax_, ay_ = x[f, 0], y[f, 0]
        ok = area[f] != 0
        for (p, q) in (((ax_, ay_), (bxs[f], bys[f])), ((bxs[f], bys[f]), (cxs[f], cys[f])), ((cxs[f], cys[f]), (ax_, ay_))):
            e, dx, dy = _edge(p[0], p[1], q[0], q[1], cx, cy)
            ok &= _inside(e, dx, dy)
        faces.append(f[ok])
        texels.append(jj[ok] * R + ii[ok])
    if not faces:
        return np.zeros(0, np.int64), np.zeros(0, np.int64)
    return np.concatenate(faces), np.concatenate(texels)


def atlas(P, F, R=2048, padding=2):
    """-> dict(vertices, triangles, uv, xy, vertex_index, chart, texel_tri, rects [C,4] (x0, y0, w, h), scale, rounds, steps)"""
    P = np.ascontiguousarray(P, np.float32)
    F = np.asarray(F, np.int64)
    T = F.shape[0]
    n, ln = face_normals(P, F)
    he = half_edges(F)
    cls = smooth(initial_classes(n), ln, allowed_classes(n, ln), he)
    s0 = density_bound(n, cls, R)
    solo = np.zeros(T, bool)
    rounds = steps = 0
    while True:
        chart, roots = charts(cls, solo, he)
        C = roots.shape[0]
        u, w = project(P, F, cls)
        bb = np.zeros((C, 4), np.float32)
        bb[:, 0] = np.inf; bb[:, 2] = np.inf; bb[:, 1] = -np.inf; bb[:, 3] = -np.inf
        cf = np.repeat(chart, 3)
        np.minimum.at(bb[:, 0], cf, u.reshape(-1)); np.maximum.at(bb[:, 1], cf, u.reshape(-1))
        np.minimum.at(bb[:, 2], cf, w.reshape(-1)); np.maximum.at(bb[:, 3], cf, w.reshape(-1))
        s, st = choose_density(bb, s0, R, padding)
        steps += st
        rw, rh = rect_dims(bb, s, R, padding)
        _, x0, y0 = nfdh(rw, rh, R)
        xy = np.empty((T, 3, 2), np.float32)
        xy[..., 0] = ((x0[chart] + padding).astype(np.float64)[:, None]
                      + (u.astype(np.float64) - bb[chart, 0:1].astype(np.float64)) * s).astype(np.float32)
        xy[..., 1] = ((y0[chart] + padding).astype(np.float64)[:, None]
                      + (w.astype(np.float64) - bb[chart, 2:3].astype(np.float64)) * s).astype(np.float32)
        f, t = coverage(xy, R)
        cnt = np.bincount(t, minlength=R * R)
        bad = cnt[t] > 1
        if not bad.any():
            break
        solo[f[bad]] = True
        rounds += 1
    texel_tri = np.full(R * R, -1, np.int32)
    texel_tri[t] = f
    hit = np.zeros(C, bool)
    hit[chart[f]] = True
    for c in np.nonzero(~hit)[0]:
        r = roots[c]
        cx = ((xy[r, 0, 0].astype(np.float64) + xy[r, 1, 0]) + xy[r, 2, 0]) * (1.0 / 3.0)
        cy = ((xy[r, 0, 1].astype(np.float64) + xy[r, 1, 1]) + xy[r, 2, 1]) * (1.0 / 3.0)
        i = int(min(max(np.floor(cx), x0[c] + padding), x0[c] + rw[c] - padding - 1))
        j = int(min(max(np.floor(cy), y0[c] + padding), y0[c] + rh[c] - padding - 1))
        texel_tri[j * R + i] = r
    key = (np.repeat(F, 1, 0) << 32 | chart[:, None]).reshape(-1)
    uk, inv = np.unique(key, return_inverse=True)
    vid = uk >> 32
    vxy = np.empty((uk.shape[0], 2), np.float32)
    vxy[inv] = xy.reshape(-1, 2)
    return dict(vertices=P[vid], triangles=inv.reshape(T, 3).astype(np.int32), uv=vxy / np.float32(R), xy=vxy,
                vertex_index=vid.astype(np.int64), chart=chart.astype(np.int32), texel_tri=texel_tri.reshape(R, R),
                rects=np.stack([x0, y0, rw, rh], 1).astype(np.int32), scale=float(s), rounds=rounds, steps=steps,
                classes=cls)


def texel_points(A, texels=None):
    """-> (texels [n] int64 (the covered ones in row order unless given), points [n,3] fp32, barycentrics [n,3] fp64)"""
    R = A["texel_tri"].shape[0]
    tt = A["texel_tri"].reshape(-1)
    if texels is None:
        texels = np.nonzero(tt >= 0)[0]
    f = tt[texels].astype(np.int64)
    tri = A["triangles"][f].astype(np.int64)
    xy = A["xy"][tri].astype(np.float64)                                    # [n,3,2]
    Pv = A["vertices"][tri].astype(np.float64)                              # [n,3,3]
    px, py = (texels % R) + 0.5, (texels // R) + 0.5
    (xa, ya), (xb, yb), (xc, yc) = [(xy[:, k, 0], xy[:, k, 1]) for k in range(3)]
    area = (xb - xa) * (yc - ya) - (yb - ya) * (xc - xa)
    ok = area != 0
    safe = np.where(ok, area, 1.0)
    la = ((xc - xb) * (py - yb) - (yc - yb) * (px - xb)) / safe
    lb = ((xa - xc) * (py - yc) - (ya - yc) * (px - xc)) / safe
    lc = ((xb - xa) * (py - ya) - (yb - ya) * (px - xa)) / safe
    la, lb, lc = np.maximum(la, 0.0), np.maximum(lb, 0.0), np.maximum(lc, 0.0)
    sm = (la + lb) + lc
    ok &= sm > 0
    ssafe = np.where(ok, sm, 1.0)
    third = 1.0 / 3.0
    la, lb, lc = (np.where(ok, l / ssafe, third) for l in (la, lb, lc))
    pts = (la[:, None] * Pv[:, 0] + lb[:, None] * Pv[:, 1]) + lc[:, None] * Pv[:, 2]
    return texels, pts.astype(np.float32), np.stack([la, lb, lc], 1)


def fill(A, texels, values, padding):
    """values [n,C] fp32 at texels -> texture [R,R,C] fp32 after `padding` dilation passes"""
    R = A["texel_tri"].shape[0]
    C = values.shape[1]
    tex = np.zeros((R * R, C), np.float32)
    tex[texels] = values.astype(np.float32)
    ch = np.full(R * R, -1, np.int64)
    ch[texels] = A["chart"][A["texel_tri"].reshape(-1)[texels]]
    rects = A["rects"].astype(np.int64)
    ii, jj = np.arange(R * R) % R, np.arange(R * R) // R
    for _ in range(padding):
        acc = np.zeros((R * R, C), np.float32)
        num = np.zeros(R * R, np.int64)
        newc = np.full(R * R, -1, np.int64)
        for dx, dy in NEIGHBOURS:
            ni, nj = ii + dx, jj + dy
            inb = (ni >= 0) & (ni < R) & (nj >= 0) & (nj < R)
            nt = np.where(inb, nj * R + ni, 0)
            c = np.where(inb, ch[nt], -1)
            rc = rects[np.maximum(c, 0)]
            ok = (ch < 0) & (c >= 0) & (ii >= rc[:, 0]) & (ii < rc[:, 0] + rc[:, 2]) & (jj >= rc[:, 1]) & (jj < rc[:, 1] + rc[:, 3])
            acc = np.where(ok[:, None], acc + tex[nt], acc)
            num += ok
            newc = np.where(ok, c, newc)
        grow = num > 0
        tex = np.where(grow[:, None], acc / np.maximum(num, 1).astype(np.float32)[:, None], tex).astype(np.float32)
        ch = np.where(grow, newc, ch)
    return tex.reshape(R, R, C)
