"""Mesh simplification on the GPU (geometry.simplify_mesh, tf_mesh_simplify) on bumpy spheres of 1 M, 4 M, 16 M and 64 M
triangles (the meshes of bench_bvh_build.py) and on marching-cubes spheres (radius 0.5 in [-1, 1]^3) at 1024^3 (dense) and at
2048^3 and 4096^3 (narrow band), each to 10 % and 1 % of its triangles and with max_error = half a voxel and no target.

Per row: T, T', V' and the rounds; tf_mesh_simplify alone (CUDA events around the call, workspace allocated outside, best of
--reps after a warm-up) and simplify_mesh end to end (wall time to a device synchronise, best of --reps); peak device bytes per
input triangle (torch's peak over the mesh already resident); evaluate_mesh of the output against the input (chamfer and
normal consistency, 10^6 samples each way); the device BVH build and a 4.98 M-ray trace (bench_bvh_build.config3_rays) on the
input and on the output.  Bumpy-sphere voxels are 2 / 1023.

The band constant (the cheapest sixteenth of the valid edges are candidates each round) was chosen from the numpy restatement
(oracle/torch_oracle_simplify.py) run with a quarter and a sixteenth on the marching-cubes sphere at 128^3 to 1 %: rounds
and quality are reported under "band".  The restatement is a plain numpy transcription for testing, not an optimized host library; its
time per round is reported on the 1 M-triangle sphere, where a full run would take hours.  GPU name and power limit go with
the numbers.

    python scripts/bench_mesh_simplify.py [--spheres 1 4 16 64] [--res 1024 2048 4096] [--reps 2] [--out results.json]
"""
import argparse
import ctypes
import json
import os
import sys
import time

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))

SPHERES = {1: (1000, 501), 4: (2000, 1001), 16: (4000, 2001), 64: (8000, 4001)}     # 2 nu (nv - 1) triangles


def sync_wall(fn):
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    out = fn()
    torch.cuda.synchronize()
    return time.perf_counter() - t0, out


def entry_point_ms(v, t, target, max_error, reps):
    """tf_mesh_simplify alone between CUDA events, outputs and workspace allocated outside"""
    from tensoflow_b200 import _lib
    lib = _lib.load()
    ws = ctypes.c_size_t()
    _lib.check(lib.tf_mesh_simplify_sizes(v.shape[0], t.shape[0], ctypes.byref(ws)), "tf_mesh_simplify_sizes")
    buf = torch.empty(ws.value, device=v.device, dtype=torch.uint8)
    ov, ot = torch.empty_like(v), torch.empty_like(t)
    nv, nt, nr = ctypes.c_int64(), ctypes.c_int64(), ctypes.c_int32()
    best = float("inf")
    for _ in range(reps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        _lib.check(lib.tf_mesh_simplify(_lib.ptr(v), v.shape[0], _lib.ptr(t), t.shape[0], target, max_error, _lib.ptr(buf), ws.value,
                                        _lib.ptr(ov), _lib.ptr(ot), ctypes.byref(nv), ctypes.byref(nt), ctypes.byref(nr),
                                        _lib.stream_ptr()), "tf_mesh_simplify")
        b.record()
        torch.cuda.synchronize()
        best = min(best, a.elapsed_time(b))
    return best


def bvh_and_trace(v, t, rays, reps):
    from bench_bvh_build import time_trace
    from tensoflow_b200.mc_ops import RayTracer
    RayTracer(v, t)
    build = min(sync_wall(lambda: RayTracer(v, t))[0] for _ in range(reps))
    rt = RayTracer(v, t)
    return {"bvh_build_ms": round(build * 1e3, 3), "trace_ms": round(time_trace([rt], *rays, reps)[0], 3)}


def measure(name, v, t, voxel, reps):
    from bench_bvh_build import config3_rays
    from tensoflow_b200.geometry import _simplify, evaluate_mesh
    T = int(t.shape[0])
    rays = config3_rays(v, t)
    before = bvh_and_trace(v, t, rays, reps)
    rows = []
    for label, target, err in (("10%", T // 10, None), ("1%", T // 100, None), ("half voxel", 0, voxel / 2)):
        torch.cuda.synchronize()
        torch.cuda.empty_cache()
        base = torch.cuda.memory_allocated()
        torch.cuda.reset_peak_memory_stats()
        _, (sv, st, rounds) = sync_wall(lambda: _simplify(v, t, target, err))           # warm-up, and the peak
        peak = torch.cuda.max_memory_allocated() - base
        wall = min(sync_wall(lambda: _simplify(v, t, target, err))[0] for _ in range(reps))
        ep = entry_point_ms(v, t, target, float("inf") if err is None else err, reps)
        ev = evaluate_mesh(sv, st, v, t, n_samples=1_000_000)
        row = {"mesh": name, "T": T, "target": label, "target_triangles": target, "max_error": err, "T_out": int(st.shape[0]),
               "V_out": int(sv.shape[0]), "rounds": rounds, "entry_point_ms": round(ep, 3),
               "simplify_mesh_wall_ms": round(wall * 1e3, 3), "peak_bytes_per_triangle": round(peak / T, 1),
               "chamfer": ev["chamfer"], "normal_consistency": ev["normal_consistency"],
               "before": before, "after": bvh_and_trace(sv, st, rays, reps)}
        print(json.dumps(row), flush=True)
        rows.append(row)
        del sv, st
    return rows


def band_comparison():
    """the numpy restatement with a quarter and a sixteenth of the valid edges as candidates, on one mesh to 1 %"""
    import numpy as np
    from oracle import torch_oracle_simplify as O
    from tensoflow_b200.geometry import evaluate_mesh
    v, t = (x.cpu() for x in sphere_mesh(128, torch.device("cuda:0")))
    out = {"mesh": "mc_sphere 128^3", "T": int(t.shape[0]), "target": int(t.shape[0]) // 100}
    for shift, label in ((2, "1/4"), (4, "1/16")):
        t0 = time.perf_counter()
        sv, st, rounds = O.simplify(v.numpy(), t.numpy(), out["target"], band_shift=shift)
        sec = time.perf_counter() - t0
        ev = evaluate_mesh(torch.from_numpy(sv).cuda(), torch.from_numpy(np.ascontiguousarray(st)).cuda(), v.cuda(), t.cuda(),
                           n_samples=1_000_000)
        out[label] = {"rounds": rounds, "T_out": int(st.shape[0]), "chamfer": ev["chamfer"],
                      "normal_consistency": ev["normal_consistency"], "numpy_restatement_seconds": round(sec, 2)}
    print(json.dumps({"band": out}), flush=True)
    return out


def oracle_per_round(v, t):
    """seconds of one round of the numpy restatement on the full mesh (the target two triangles below T stops it after one)"""
    from oracle import torch_oracle_simplify as O
    t0 = time.perf_counter()
    _, _, rounds = O.simplify(v.cpu().numpy(), t.cpu().numpy(), int(t.shape[0]) - 2)
    return {"rounds": rounds, "seconds_per_round": round((time.perf_counter() - t0) / max(rounds, 1), 2)}


def sphere_mesh(R, dev):
    """marching cubes of |p| - 0.5 on an R^3 lattice of [-1, 1]^3, world coordinates: dense below 2^31 points, else narrow band"""
    from tensoflow_b200.isosurface import marching_cubes, marching_cubes_narrowband
    ax = torch.linspace(-1, 1, R, device=dev)
    if R ** 3 < 2 ** 31:
        x, y, z = torch.meshgrid(ax, ax, ax, indexing="ij")
        u = (x * x + y * y + z * z).sqrt_() - 0.5
        del x, y, z
        v, t = marching_cubes(u)
        del u
    else:
        v, t = marching_cubes_narrowband(lambda p: p.norm(dim=-1) - 0.5, (ax, ax, ax))
    return v / (R - 1.0) * 2.0 - 1.0, t


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--spheres", type=int, nargs="*", default=[1, 4, 16, 64], help="bumpy spheres, millions of triangles")
    ap.add_argument("--res", type=int, nargs="*", default=[1024, 2048, 4096], help="marching-cubes sphere resolutions")
    ap.add_argument("--reps", type=int, default=2)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_mesh_simplify.py measures the device path: no CUDA device")
    from bench_extract_mesh import gpu_info
    from tensoflow_b200.synthetic import bumpy_sphere
    dev = torch.device("cuda:0")
    result = {"info": gpu_info(), "rows": []}
    result["band"] = band_comparison()
    for m in args.spheres:
        v, t = (x.to(dev) for x in bumpy_sphere(*SPHERES[m]))
        if m == 1:
            result["numpy_restatement_1M"] = oracle_per_round(v, t)
            print(json.dumps({"numpy_restatement_1M": result["numpy_restatement_1M"]}), flush=True)
        result["rows"] += measure(f"bumpy_sphere{SPHERES[m]}", v, t, 2.0 / 1023, args.reps)
        del v, t
        torch.cuda.empty_cache()
    for R in args.res:
        v, t = sphere_mesh(R, dev)
        torch.cuda.empty_cache()
        result["rows"] += measure(f"mc_sphere {R}^3", v, t, 2.0 / (R - 1), args.reps)
        del v, t
        torch.cuda.empty_cache()
    if args.out:
        with open(args.out, "w") as f:
            json.dump(result, f, indent=1)


if __name__ == "__main__":
    main()
