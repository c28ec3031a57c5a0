"""BVH build of mc_ops.RayTracer: the host build (tf_bvh_create, what a CPU mesh gets, timed from a CUDA mesh including its copy
to the host) against the device build (tf_bvh_build, what a CUDA mesh gets), on bumpy spheres of 1 M, 4 M, 16 M and 64 M
triangles and on ShapeRenderer.extract_geometry meshes of a config-2-shaped field (the field of bench_extract_mesh.py) at
1024^3, 2048^3 and 4096^3.

Per mesh: T; host build seconds; device build seconds (wall time to a device synchronise, sorts included, best of --reps after
a warm-up build); peak device memory of the device build (torch's peak over the mesh already resident, plus the handle's
own copy of the tree); the two trees compared byte for byte; and bvh_trace of a config-3-shaped ray batch (8192 surface points x
608 directions, scripts/bench_material.py) with each handle, alternating, best of --reps.  Then geometry.evaluate_mesh end to
end at 10^6 samples on the 2048^3 mesh against bumpy_sphere(1000, 500).  GPU name and power limit go with the numbers.

    python scripts/bench_bvh_build.py [--spheres 1 4 16 64] [--res 1024 2048 4096] [--reps 3] [--out results.json]
"""
import argparse
import ctypes
import json
import math
import os
import sys
import time

import numpy as np
import torch
import torch.nn.functional as F

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))

SPHERES = {1: (1000, 501), 4: (2000, 1001), 16: (4000, 2001), 64: (8000, 4001)}     # 2 nu (nv - 1) triangles


def export(rt):
    from tensoflow_b200 import _lib
    lib = _lib.load()
    nn, nt = ctypes.c_int64(), ctypes.c_int64()
    _lib.check(lib.tf_bvh_export(rt._h, ctypes.byref(nn), ctypes.byref(nt), None, None, None), "tf_bvh_export")
    out = [np.empty(nn.value * 32, np.uint8), np.empty(nt.value * 48, np.uint8), np.empty(nt.value * 4, np.uint8)]
    _lib.check(lib.tf_bvh_export(rt._h, None, None, *(a.ctypes.data_as(ctypes.c_void_p) for a in out)), "tf_bvh_export")
    return out, nn.value


def config3_rays(v, t, n_points=8192, n_dirs=608, seed=0):
    """rays leaving n_points surface points (triangle centroids pushed 1e-4 along the normal) in n_dirs random directions of
    the outer hemisphere each: the secondary-ray batch of one config-3 step"""
    g = torch.Generator(device=v.device).manual_seed(seed)
    ti = torch.randint(0, t.shape[0], (n_points,), device=v.device, generator=g)
    a, b, c = (v[t[ti, k].long()] for k in range(3))
    n = F.normalize(torch.cross(b - a, c - a, dim=-1), dim=-1)
    p = (a + b + c) / 3 + 1e-4 * n
    d = F.normalize(torch.randn(n_points, n_dirs, 3, device=v.device, generator=g), dim=-1)
    d = torch.where(((d * n[:, None]).sum(-1, keepdim=True) < 0), -d, d)
    return p[:, None].expand(-1, n_dirs, -1).reshape(-1, 3).contiguous(), d.reshape(-1, 3).contiguous()


def time_trace(rts, o, d, reps):
    ms = [[] for _ in rts]
    for rt in rts:
        rt.trace(o, d)
    for _ in range(reps):
        for i, rt in enumerate(rts):
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            rt.trace(o, d)
            b.record()
            torch.cuda.synchronize()
            ms[i].append(a.elapsed_time(b))
    return [min(x) for x in ms]


def measure(name, v, t, reps, host_build=True):
    from tensoflow_b200.mc_ops import RayTracer
    T = int(t.shape[0])
    row = {"mesh": name, "T": T}
    torch.cuda.synchronize()
    dev_rt = RayTracer(v, t)                         # warm-up
    del dev_rt
    times = []
    for _ in range(reps):
        torch.cuda.synchronize()
        base = torch.cuda.memory_allocated()
        torch.cuda.reset_peak_memory_stats()
        t0 = time.perf_counter()
        dev_rt = RayTracer(v, t)
        torch.cuda.synchronize()
        times.append(time.perf_counter() - t0)
        peak = torch.cuda.max_memory_allocated() - base
    dev_tree, n_nodes = export(dev_rt)
    row["device_build_s"] = min(times)
    row["device_build_peak_bytes"] = int(peak + 32 * n_nodes + 52 * T)
    row["device_build_bytes_per_triangle"] = round(row["device_build_peak_bytes"] / T, 1)
    rts = [dev_rt]
    if host_build:
        t0 = time.perf_counter()
        host_rt = RayTracer(v.cpu(), t.cpu())
        torch.cuda.synchronize()
        row["host_build_s"] = time.perf_counter() - t0
        row["trees_byte_equal"] = all(x.tobytes() == y.tobytes() for x, y in zip(export(host_rt)[0], dev_tree))
        row["speedup"] = row["host_build_s"] / row["device_build_s"]
        rts.append(host_rt)
    else:
        row["host_build_s"] = "not measured"
    o, d = config3_rays(v, t)
    tr = time_trace(rts, o, d, reps)
    row["trace_rays"] = int(o.shape[0])
    row["bvh_trace_ms_device_built"] = tr[0]
    row["bvh_trace_ms_host_built"] = tr[1] if host_build else "not measured"
    print(json.dumps(row), flush=True)
    return row


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--spheres", type=int, nargs="*", default=[1, 4, 16, 64], help="bumpy spheres, millions of triangles")
    ap.add_argument("--res", type=int, nargs="*", default=[1024, 2048, 4096], help="extract_geometry resolutions")
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--no-host-above", type=int, default=1 << 31, help="skip the host build above this many triangles")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_bvh_build.py measures the device build: no CUDA device")
    from bench_extract_mesh import gpu_info, make_shape
    from tensoflow_b200.geometry import evaluate_mesh
    from tensoflow_b200.synthetic import bumpy_sphere
    dev = torch.device("cuda:0")
    result = {"info": gpu_info(), "rows": []}
    for m in args.spheres:
        v, t = (x.to(dev) for x in bumpy_sphere(*SPHERES[m]))
        result["rows"].append(measure(f"bumpy_sphere{SPHERES[m]}", v, t, args.reps, t.shape[0] <= args.no_host_above))
        del v, t
        torch.cuda.empty_cache()
    if args.res:
        shape = make_shape(dev)
        lo, hi = [-1.0] * 3, [1.0] * 3
        for R in args.res:
            with torch.no_grad():
                v, t = shape.extract_geometry(lo, hi, R)
            torch.cuda.empty_cache()
            result["rows"].append(measure(f"extract_geometry {R}^3", v, t, args.reps, t.shape[0] <= args.no_host_above))
            if R == 2048:
                gv, gt = (x.to(dev) for x in bumpy_sphere(1000, 500))
                evaluate_mesh(v, t, gv, gt, n_samples=1_000_000)           # warm-up
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                ev = evaluate_mesh(v, t, gv, gt, n_samples=1_000_000)
                torch.cuda.synchronize()
                result["evaluate_mesh_2048"] = {"seconds": time.perf_counter() - t0, "T_pred": int(t.shape[0]),
                                                "T_gt": int(gt.shape[0]), "n_samples": 1_000_000, "chamfer": ev["chamfer"]}
                print(json.dumps({"evaluate_mesh_2048": result["evaluate_mesh_2048"]}), flush=True)
            del v, t
            torch.cuda.empty_cache()
    if args.out:
        with open(args.out, "w") as f:
            json.dump(result, f, indent=1)


if __name__ == "__main__":
    main()
