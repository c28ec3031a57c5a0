"""TEST INFRASTRUCTURE ONLY (never imported by tensoflow_b200/).  Vectorised CPU marching cubes under the conventions of
include/tensoflow_b200.h (tf_iso_*): the stand-in for the reference's `mcubes.marching_cubes(u, threshold)`
(extract_mesh.py), which PyMCubes provides there and which is absent here.

Conventions (the kernels reproduce them bit for bit):
  * u [nx, ny, nz] fp32, z fastest; a lattice point is inside iff u < threshold (fp32 compare);
  * one vertex per crossed lattice edge, ordered by (p, axis) with p = (i * ny + j) * nz + k the edge's lower point and axis
    order x, y, z; it lies at index coordinate a_axis + t, t = (threshold - u_a) / (u_b - u_a), each op one fp32 rounding;
  * triangles int32, ordered by cell (i * ny + j) * nz + k, then in the order of the case table
    (tensoflow_b200/isosurface_table.py)."""
import torch

from tensoflow_b200.isosurface_table import EDGES, build_table

_TABLE, _COUNT = (torch.from_numpy(a.astype("int64")) for a in build_table())


def marching_cubes(volume, threshold: float = 0.0):
    """volume [nx, ny, nz] (any float dtype, converted to fp32 once) -> (vertices [V,3] fp32 index space, triangles [T,3] int32)"""
    u = torch.as_tensor(volume).detach().cpu().to(torch.float32).contiguous()
    assert u.dim() == 3 and min(u.shape) >= 2, u.shape
    nx, ny, nz = u.shape
    thr = torch.tensor(threshold, dtype=torch.float32)
    inside = u < thr

    crossed = torch.zeros(nx, ny, nz, 3, dtype=torch.bool)
    crossed[:-1, :, :, 0] = inside[:-1] != inside[1:]
    crossed[:, :-1, :, 1] = inside[:, :-1] != inside[:, 1:]
    crossed[:, :, :-1, 2] = inside[:, :, :-1] != inside[:, :, 1:]
    flat = crossed.reshape(-1)
    vid = torch.cumsum(flat, 0) - 1                          # vertex id of the owned edge (p, axis) where crossed
    sel = torch.nonzero(flat)[:, 0]
    axis = sel % 3
    p = sel // 3
    ijk = torch.stack([p // (ny * nz), p // nz % ny, p % nz], -1)
    rows = torch.arange(sel.shape[0])
    q = ijk.clone()
    q[rows, axis] += 1
    ua = u[ijk[:, 0], ijk[:, 1], ijk[:, 2]]
    ub = u[q[:, 0], q[:, 1], q[:, 2]]
    t = (thr - ua) / (ub - ua)
    verts = ijk.to(torch.float32)
    verts[rows, axis] = verts[rows, axis] + t

    ins = inside.to(torch.int64)
    case = torch.zeros(nx - 1, ny - 1, nz - 1, dtype=torch.int64)
    for c in range(8):
        b0, b1, b2 = c & 1, c >> 1 & 1, c >> 2 & 1
        case |= ins[b0:nx - 1 + b0, b1:ny - 1 + b1, b2:nz - 1 + b2] << c
    cells = torch.nonzero((_COUNT[case] > 0).reshape(-1))[:, 0]
    if cells.numel() == 0:
        return verts, torch.zeros(0, 3, dtype=torch.int32)
    cc = case.reshape(-1)[cells]
    ci, cj, ck = cells // ((ny - 1) * (nz - 1)), cells // (nz - 1) % (ny - 1), cells % (nz - 1)
    edge_vid = torch.stack([vid[(((ci + (c0 & 1)) * ny + cj + (c0 >> 1 & 1)) * nz + ck + (c0 >> 2 & 1)) * 3 + e // 4]
                            for e, (c0, _) in enumerate(EDGES)], -1)                       # [M, 12]
    tri_edges = _TABLE[cc, :15].reshape(-1, 5, 3)
    valid = torch.arange(5)[None, :] < _COUNT[cc][:, None]
    tris = edge_vid.gather(1, tri_edges.clamp_min(0).reshape(-1, 15)).reshape(-1, 5, 3)[valid]
    return verts, tris.to(torch.int32)
