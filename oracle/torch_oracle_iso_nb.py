"""TEST INFRASTRUCTURE ONLY (never imported by tensoflow_b200/).  The narrow-band rule of include/tensoflow_b200.h
(tf_iso_nb_*, tensoflow_b200.isosurface.marching_cubes_narrowband) restated on the CPU on top of the dense marching-cubes oracle
(oracle/torch_oracle_iso.py): the coarse brick test, the grow loop until closed, and the dense mesh cut to the active bricks."""
import math

import torch

from oracle.torch_oracle_iso import _COUNT, marching_cubes

BRICK = 8                                                     # cells per brick edge of the narrow band


def marching_cubes_narrowband(fn, axes, threshold: float = 0.0):
    """The narrow-band rule of include/tensoflow_b200.h (tf_iso_nb_*, tensoflow_b200.isosurface.marching_cubes_narrowband)
    restated on the CPU.  fn(points [N,3] fp32) -> [N] values; axes: three 1-D fp32 tensors (nx, ny, nz points).  The dense
    lattice is evaluated here (small lattices only); the result depends only on the values in the active bricks.
    -> (vertices [V,3] fp32, triangles [T,3] int32, active brick ids (I*by + J)*bz + K sorted, rounds), where rounds[0] holds
    the bricks of the coarse test and rounds[r] those added by grow round r (len(rounds) - 1 grow rounds added bricks).
    The mesh is the dense oracle's, cut to the cells of the active bricks and the vertices those cells use (renumbered in
    order); it equals marching_cubes of the dense lattice when every cell with a crossing lies in an active brick."""
    ax = [torch.as_tensor(a).detach().cpu().to(torch.float32) for a in axes]
    n = [a.shape[0] for a in ax]
    assert all(2 <= m <= 4096 for m in n), n
    x, y, z = torch.meshgrid(*ax, indexing="ij")
    u = torch.as_tensor(fn(torch.stack([x, y, z], -1).reshape(-1, 3))).to(torch.float32).reshape(n)
    thr = torch.tensor(threshold, dtype=torch.float32)
    nb = [(m - 1 + BRICK - 1) // BRICK for m in n]
    strides = [nb[1] * nb[2], nb[2], 1]

    # 1-2. coarse test: corners straddle the threshold, or one within sqrt(3) * 8 * h_max of it (fp32 compare)
    h = max(float((a[1:] - a[:-1]).abs().max()) for a in ax)
    band = torch.tensor(math.sqrt(3.0) * BRICK * h, dtype=torch.float32)
    ci = [torch.clamp(torch.arange(b + 1) * BRICK, max=m - 1) for b, m in zip(nb, n)]
    cu = u[ci[0]][:, ci[1]][:, :, ci[2]]
    n_in = torch.zeros(nb, dtype=torch.int64)
    near = torch.zeros(nb, dtype=torch.bool)
    for c in range(8):
        b0, b1, b2 = c & 1, c >> 1 & 1, c >> 2 & 1
        corner = cu[b0:nb[0] + b0, b1:nb[1] + b1, b2:nb[2] + b2]
        n_in += corner < thr
        near |= (corner - thr).abs() < band
    active = (((n_in > 0) & (n_in < 8)) | near).reshape(-1)

    # 4. bricks whose closure holds each crossed lattice edge: the cell-range brick along the edge; across it, the brick of
    # the point and, on a brick boundary, the one before it
    inside = u < thr
    hold = []                                                 # per crossed edge, its 4 possible holders (-1: none)
    for a in range(3):
        e = torch.nonzero(inside.narrow(a, 0, n[a] - 1) != inside.narrow(a, 1, n[a] - 1))
        opts = []
        for b in range(3):
            if b == a:
                opts.append([e[:, b] // BRICK])
            else:
                opts.append([torch.where(e[:, b] // BRICK < nb[b], e[:, b] // BRICK, -1),
                             torch.where((e[:, b] % BRICK == 0) & (e[:, b] > 0), e[:, b] // BRICK - 1, -1)])
        hold.append(torch.stack([torch.where((c0 >= 0) & (c1 >= 0) & (c2 >= 0), c0 * strides[0] + c1 * strides[1] + c2, -1)
                                 for c0 in opts[0] for c1 in opts[1] for c2 in opts[2]], 1))
    hold = torch.cat(hold, 0)                                 # [M, 4]
    rounds = [torch.nonzero(active)[:, 0]]
    new = active.clone()
    while True:
        touched = ((hold >= 0) & new[hold.clamp_min(0)]).any(1)
        cand = hold[touched].reshape(-1)
        mark = torch.zeros_like(active)
        mark[cand[cand >= 0]] = True
        mark &= ~active
        if not bool(mark.any()):
            break
        active |= mark
        new = mark
        rounds.append(torch.nonzero(mark)[:, 0])

    # 5. the dense mesh cut to the active bricks' cells
    verts, tris = marching_cubes(u, threshold)
    ins = inside.to(torch.int64)
    case = torch.zeros(n[0] - 1, n[1] - 1, n[2] - 1, dtype=torch.int64)
    for c in range(8):
        b0, b1, b2 = c & 1, c >> 1 & 1, c >> 2 & 1
        case |= ins[b0:n[0] - 1 + b0, b1:n[1] - 1 + b1, b2:n[2] - 1 + b2] << c
    cnt = _COUNT[case]
    cells = torch.nonzero(cnt)
    brick_of_cell = (cells[:, 0] // BRICK) * strides[0] + (cells[:, 1] // BRICK) * strides[1] + cells[:, 2] // BRICK
    keep = torch.repeat_interleave(active[brick_of_cell], cnt[cnt > 0])
    kept = tris[keep].long()
    used = torch.zeros(verts.shape[0], dtype=torch.bool)
    used[kept.reshape(-1)] = True
    renum = torch.cumsum(used, 0) - 1
    return verts[used], renum[kept].to(torch.int32).reshape(-1, 3), torch.nonzero(active)[:, 0], rounds
