"""TEST INFRASTRUCTURE ONLY (never imported by tensoflow_b200/).  numpy restatement of tf_mesh_simplify (include/tensoflow_b200.h,
tensoflow_b200/csrc/mesh_simplify.cu): Garland-Heckbert quadric-error edge collapse in rounds of independent collapses.  Every
floating-point operation below is an elementwise numpy op in the kernel's order (no `@`, einsum or BLAS), so the result is
bit-equal to the device's.

The rules, per round, on the current faces F [T,3] (input order, collapsed faces removed) and positions P [V,3] fp32:

  * quadrics (fp64, 10 entries xx xy xz xd yy yz yd zz zd dd of p p^T): at the start, each vertex sums the unit-normal plane
    quadric of its faces in face order, starting from 0; a face whose cross product (b - a) x (c - a) has zero length adds
    nothing.  A collapse gives the survivor Q_a + Q_b.
  * star(v): the faces referencing v, ascending.  deg(v) = |star(v)|.  An edge {a, b}, a < b, is the pair of two consecutive
    corners of a face; its faces are the faces having it, ascending.
  * locked vertices: both ends of every edge with a face count other than 2, and the vertices of a face with a repeated index.
  * an edge is valid iff it has exactly two faces f0 < f1, with apexes c0 != c1; a and b are not locked; deg(c0) > 3 and
    deg(c1) > 3 (an apex of valence 3 would leave two coincident faces); N(a) and N(b) have no common vertex but c0 and c1
    (link condition); every face of star(a) + star(b) other than f0, f1 whose old normal is not zero has a new normal n' with
    n . n' > 0 (no fold-over, no new degenerate face); and sqrt(cost) <= max_error.
  * placement: A = the 3x3 block of Q = Q_a + Q_b, t = xx + yy + zz.  If det(A) > 1e-6 t^3 (products left to right), v =
    -A^-1 (xd, yd, zd) from the adjugate, rounded to fp32.  Otherwise v is the cheapest of P[a], P[b] and the fp32 midpoint,
    ties in that order.  cost = max(0, v^T Q v) at the fp32 v, rows of Q summed left to right.  The survivor is a.
  * selection: valid edges ranked by (fp32(cost), a, b); the first k are candidates, k = min(max(1, n_valid >> BAND_SHIFT),
    (T - target) // 2) (0 with no valid edge).  Candidate i has priority (hash(a << 32 | b) >> 32) << 32 | i (splitmix64
    finaliser).  It wins iff its priority is the minimum claimed by every vertex of its closed 1-ring (the vertices of star(a)
    and star(b)); winners have vertex-disjoint closed 1-rings.
  * apply: P[a] = v, Q[a] = Q[a] + Q[b], f0 and f1 are removed, b becomes a in the other faces of star(b).
  * stop when T <= target + 1 or a round collapses nothing.  Output: surviving faces in order, referenced vertices in order,
    indices renumbered."""
import numpy as np

BAND_SHIFT = 4                 # candidates: the cheapest sixteenth of the valid edges
COND = 1e-6                    # det(A) > COND * trace(A)^3: closed-form placement


def edge_hash(key):
    """splitmix64 finaliser of uint64 keys (wrapping arithmetic)"""
    z = np.asarray(key, np.uint64)
    with np.errstate(over="ignore"):
        z = (z ^ (z >> np.uint64(30))) * np.uint64(0xBF58476D1CE4E5B9)
        z = (z ^ (z >> np.uint64(27))) * np.uint64(0x94D049BB133111EB)
    return z ^ (z >> np.uint64(31))


def _cross(e1, e2):
    return np.stack([e1[..., 1] * e2[..., 2] - e1[..., 2] * e2[..., 1],
                     e1[..., 2] * e2[..., 0] - e1[..., 0] * e2[..., 2],
                     e1[..., 0] * e2[..., 1] - e1[..., 1] * e2[..., 0]], -1)


def _normal(p0, p1, p2):
    """(p1 - p0) x (p2 - p0), fp64 inputs"""
    return _cross(p1 - p0, p2 - p0)


def face_quadrics(P, F):
    """unit-normal plane quadric per face [T,10] fp64 (zeros for a zero-length cross product)"""
    p = P.astype(np.float64)[F]
    n = _normal(p[:, 0], p[:, 1], p[:, 2])
    ln = np.sqrt((n[:, 0] * n[:, 0] + n[:, 1] * n[:, 1]) + n[:, 2] * n[:, 2])
    ok = ln > 0
    u = n / np.where(ok, ln, 1.0)[:, None]
    d = -((u[:, 0] * p[:, 0, 0] + u[:, 1] * p[:, 0, 1]) + u[:, 2] * p[:, 0, 2])
    x, y, z = u[:, 0], u[:, 1], u[:, 2]
    q = np.stack([x * x, x * y, x * z, x * d, y * y, y * z, y * d, z * z, z * d, d * d], -1)
    return np.where(ok[:, None], q, 0.0)


def quad_cost(Q, v):
    """max(0, v^T Q v) for v [...,3] fp64, Q [...,10]"""
    xx, xy, xz, xd, yy, yz, yd, zz, zd, dd = (Q[..., k] for k in range(10))
    x, y, z = v[..., 0], v[..., 1], v[..., 2]
    r0 = ((xx * x + xy * y) + xz * z) + xd
    r1 = ((xy * x + yy * y) + yz * z) + yd
    r2 = ((xz * x + yz * y) + zz * z) + zd
    r3 = ((xd * x + yd * y) + zd * z) + dd
    c = ((x * r0 + y * r1) + z * r2) + r3
    return np.where(c < 0, 0.0, c)


def placement(Q, pa, pb):
    """-> (v [E,3] fp32, cost [E] fp64) for Q [E,10] fp64 and endpoint positions pa, pb [E,3] fp32"""
    xx, xy, xz, xd, yy, yz, yd, zz, zd = (Q[:, k] for k in range(9))
    i00 = yy * zz - yz * yz
    i01 = xz * yz - xy * zz
    i02 = xy * yz - xz * yy
    i11 = xx * zz - xz * xz
    i12 = xy * xz - xx * yz
    i22 = xx * yy - xy * xy
    det = (xx * i00 + xy * i01) + xz * i02
    tr = (xx + yy) + zz
    solve = det > ((COND * tr) * tr) * tr
    sdet = np.where(solve, det, 1.0)
    vs = np.stack([-(((i00 * xd + i01 * yd) + i02 * zd) / sdet),
                   -(((i01 * xd + i11 * yd) + i12 * zd) / sdet),
                   -(((i02 * xd + i12 * yd) + i22 * zd) / sdet)], -1)
    with np.errstate(over="ignore", invalid="ignore"):
        vs = vs.astype(np.float32)
    mid = ((pa.astype(np.float64) + pb.astype(np.float64)) * 0.5).astype(np.float32)
    best, cbest = pa, quad_cost(Q, pa.astype(np.float64))
    for cand in (pb, mid):
        c = quad_cost(Q, cand.astype(np.float64))
        take = c < cbest
        best = np.where(take[:, None], cand, best)
        cbest = np.where(take, c, cbest)
    v = np.where(solve[:, None], vs, best).astype(np.float32)
    return v, quad_cost(Q, v.astype(np.float64))


class _Round:
    """adjacency of the current mesh"""

    def __init__(self, F, V):
        T = F.shape[0]
        flat = F.reshape(-1)
        order = np.argsort(flat, kind="stable")
        self.deg = np.bincount(flat, minlength=V)
        start = np.concatenate([[0], np.cumsum(self.deg)])
        D = int(self.deg.max())
        self.star = np.full((V, D), -1, np.int64)                 # star[v, j]: j-th face of v, ascending
        sv = flat[order]
        self.star[sv, np.arange(3 * T) - start[sv]] = order // 3
        a = np.concatenate([F[:, 0], F[:, 1], F[:, 2]])
        b = np.concatenate([F[:, 1], F[:, 2], F[:, 0]])
        he_face = np.concatenate([np.arange(T)] * 3)
        he_id = np.concatenate([3 * np.arange(T), 3 * np.arange(T) + 1, 3 * np.arange(T) + 2])
        lo, hi = np.minimum(a, b), np.maximum(a, b)
        key = lo * (1 << 32) + hi
        o = np.lexsort((he_id, key))                                # the device's stable sort of the half-edges 3f + k
        key, he_face = key[o], he_face[o]
        first = np.concatenate([[True], key[1:] != key[:-1]])
        starts = np.nonzero(first)[0]
        count = np.diff(np.concatenate([starts, [3 * T]]))
        self.ekey = key[starts]
        self.ea, self.eb = self.ekey >> 32, self.ekey & 0xFFFFFFFF
        self.count = count
        self.f0 = he_face[starts]
        self.f1 = he_face[np.minimum(starts + 1, 3 * T - 1)]
        locked = np.zeros(V, bool)
        locked[self.ea[count != 2]] = True
        locked[self.eb[count != 2]] = True
        rep = (F[:, 0] == F[:, 1]) | (F[:, 1] == F[:, 2]) | (F[:, 0] == F[:, 2])
        locked[F[rep].reshape(-1)] = True
        self.locked = locked
        # neighbour lists (both directions of every edge), to test the link condition
        na = np.concatenate([self.ea, self.eb])
        nb = np.concatenate([self.eb, self.ea])
        o = np.argsort(na, kind="stable")
        self.nb_of, self.nb_start = nb[o], np.concatenate([[0], np.cumsum(np.bincount(na, minlength=V))])


def _check_edges(F, P, Q, R, idx, max_error):
    """validity, placement and cost of the edges idx (count 2) -> (valid [n] bool, v [n,3] fp32, cost [n] fp64)"""
    a, b, f0, f1 = R.ea[idx], R.eb[idx], R.f0[idx], R.f1[idx]
    c0 = F[f0].sum(1) - a - b
    c1 = F[f1].sum(1) - a - b
    ok = ~R.locked[a] & ~R.locked[b] & (c0 != c1) & (R.deg[c0] > 3) & (R.deg[c1] > 3)
    # link condition: the common neighbours of a and b are c0 and c1 only
    n_a = R.nb_start[a + 1] - R.nb_start[a]
    rows = np.repeat(np.arange(idx.shape[0]), n_a)
    w = R.nb_of[np.repeat(R.nb_start[a], n_a) + (np.arange(rows.shape[0]) - np.repeat(np.cumsum(n_a) - n_a, n_a))]
    bb = b[rows]
    k = np.minimum(bb, w) * (1 << 32) + np.maximum(bb, w)
    pos = np.minimum(np.searchsorted(R.ekey, k), R.ekey.shape[0] - 1)
    extra = (R.ekey[pos] == k) & (w != c0[rows]) & (w != c1[rows])
    ok &= np.bincount(rows[extra], minlength=idx.shape[0]) == 0
    Qe = Q[a] + Q[b]
    v, cost = placement(Qe, P[a], P[b])
    if max_error is not None:
        ok &= np.sqrt(cost) <= max_error
    # fold-over over the faces of star(a) and star(b) other than f0, f1
    for s in range(0, idx.shape[0], 1 << 15):
        e = np.arange(s, min(s + (1 << 15), idx.shape[0]))
        e = e[ok[e]]
        if e.size == 0:
            continue
        g = np.concatenate([R.star[a[e]], R.star[b[e]]], 1)                   # [n, 2D]
        live = (g >= 0) & (g != f0[e][:, None]) & (g != f1[e][:, None])
        gv = F[np.where(live, g, 0)]                                         # [n, 2D, 3]
        p_old = P.astype(np.float64)[gv]
        moved = (gv == a[e][:, None, None]) | (gv == b[e][:, None, None])
        p_new = np.where(moved[..., None], v[e].astype(np.float64)[:, None, None, :], p_old)
        n_old = _normal(p_old[..., 0, :], p_old[..., 1, :], p_old[..., 2, :])
        n_new = _normal(p_new[..., 0, :], p_new[..., 1, :], p_new[..., 2, :])
        dot = (n_old[..., 0] * n_new[..., 0] + n_old[..., 1] * n_new[..., 1]) + n_old[..., 2] * n_new[..., 2]
        flat = (n_old[..., 0] == 0) & (n_old[..., 1] == 0) & (n_old[..., 2] == 0)
        ok[e] &= ~(live & ~flat & ~(dot > 0)).any(1)
    return ok, v, cost


def ring_vertices(F, R, a, b):
    """closed 1-ring of each edge: vertices of star(a) and star(b), [n, 6D] with -1 padding"""
    g = np.concatenate([R.star[a], R.star[b]], 1)
    return np.where((g >= 0)[..., None], F[np.where(g >= 0, g, 0)], -1).reshape(g.shape[0], -1)


def simplify(vertices, triangles, target, max_error=None, band_shift=BAND_SHIFT, on_round=None):
    """-> (vertices [V',3] fp32, triangles [T',3] int32, rounds).  on_round(F, P, Q, R, winners) is called after each round's
    selection, before the collapses are applied: winners is a dict of arrays a, b, f0, f1, v, cost, ring (edge order)."""
    P = np.array(vertices, np.float32).reshape(-1, 3)
    F = np.asarray(triangles, np.int64).reshape(-1, 3)
    V = P.shape[0]
    target = int(target)
    Q = None
    rounds = 0
    while F.shape[0] > target + 1:
        T = F.shape[0]
        R = _Round(F, V)
        if Q is None:
            fq = face_quadrics(P, F)
            Q = np.zeros((V, 10))
            for j in range(R.star.shape[1]):                             # per vertex, faces in face order
                g = R.star[:, j]
                Q = Q + np.where((g >= 0)[:, None], fq[np.where(g >= 0, g, 0)], 0.0)
        idx = np.nonzero(R.count == 2)[0]
        ok, v, cost = _check_edges(F, P, Q, R, idx, max_error)
        idx, v, cost = idx[ok], v[ok], cost[ok]
        n_valid = idx.shape[0]
        if n_valid == 0:
            break
        k = min(max(1, n_valid >> band_shift), (T - target) // 2)
        order = np.argsort(cost.astype(np.float32), kind="stable")[:k]       # ties: edge order = (a, b)
        e, v, cost = idx[order], v[order], cost[order]
        a, b = R.ea[e], R.eb[e]
        prio = ((edge_hash(R.ekey[e].astype(np.uint64)) >> np.uint64(32)) << np.uint64(32)) | np.arange(k, dtype=np.uint64)
        ring = ring_vertices(F, R, a, b)
        claim = np.full(V, np.iinfo(np.uint64).max, np.uint64)
        m = ring >= 0
        np.minimum.at(claim, ring[m], np.broadcast_to(prio[:, None], ring.shape)[m])
        win = ((claim[np.where(m, ring, 0)] == prio[:, None]) | ~m).all(1)
        if on_round is not None:
            on_round(F, P, Q, R, {"a": a[win], "b": b[win], "f0": R.f0[e][win], "f1": R.f1[e][win], "v": v[win],
                                  "cost": cost[win], "ring": ring[win]})
        a, b = a[win], b[win]
        P[a] = v[win]
        Q[a] = Q[a] + Q[b]
        dead = np.zeros(T, bool)
        dead[R.f0[e][win]] = True
        dead[R.f1[e][win]] = True
        remap = np.arange(V)
        remap[b] = a
        F = remap[F[~dead]]
        rounds += 1
    used = np.zeros(V, bool)
    used[F.reshape(-1)] = True
    new_index = np.cumsum(used) - 1
    return P[used], new_index[F].astype(np.int32), rounds
