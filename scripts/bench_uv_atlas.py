"""UV atlas and texture baking on the GPU (geometry.uv_atlas, geometry.bake_texture) on bumpy spheres of 1 M, 16 M and 64 M
triangles, the marching-cubes sphere at 4096^3 (narrow band, world coordinates) and that mesh simplified to half a voxel of
error, each at R = 2048, 4096 and 8192.

Per row: T, the charts, conflict rounds and density trials; uv_atlas end to end (wall time to a device synchronise, best of
--reps after a warm-up); bake_texture of a 5-channel fn (the texel points' sin / cos and |p|, standing in for albedo,
roughness and metallic) likewise; occupancy (covered texels / R^2); peak device bytes over the mesh already resident; and,
from one run under torch.profiler, the device time of the sequential next-fit packing kernel (one thread) summed over all
its launches.  GPU name and power limit go with the numbers.

    python scripts/bench_uv_atlas.py [--spheres 1 16 64] [--res 2048 4096 8192] [--reps 2] [--out profiles/bench_uv_atlas_1gpu.json]
"""
import argparse
import json
import os
import sys
import time

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))

SPHERES = {1: (1000, 501), 16: (4000, 2001), 64: (8000, 4001)}     # 2 nu (nv - 1) triangles


def sync_wall(fn):
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    out = fn()
    torch.cuda.synchronize()
    return time.perf_counter() - t0, out


def fn5(p):
    return torch.cat([torch.sin(p), torch.cos(p[:, :1]), p.norm(dim=-1, keepdim=True)], -1)


def nfdh_ms(v, t, R):
    from torch.profiler import ProfilerActivity, profile
    from tensoflow_b200.geometry import uv_atlas
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        uv_atlas(v, t, R)
        torch.cuda.synchronize()
    total = sum(e.device_time_total for e in prof.key_averages() if "ua_nfdh" in e.key)
    return round(total / 1e3, 3)


def measure(name, v, t, res, reps):
    from tensoflow_b200.geometry import bake_texture, uv_atlas
    rows = []
    for R in res:
        uv_atlas(v, t, R)                                                    # warm-up
        torch.cuda.synchronize()
        torch.cuda.empty_cache()
        base = torch.cuda.memory_allocated()
        torch.cuda.reset_peak_memory_stats()
        best_a, A = min((sync_wall(lambda: uv_atlas(v, t, R)) for _ in range(reps)), key=lambda x: x[0])
        peak_atlas = torch.cuda.max_memory_allocated() - base
        bake_texture(A, fn5, 5)
        best_b, (tex, mask) = min((sync_wall(lambda: bake_texture(A, fn5, 5)) for _ in range(reps)), key=lambda x: x[0])
        peak = torch.cuda.max_memory_allocated() - base
        row = {"mesh": name, "T": int(t.shape[0]), "R": R, "charts": int(A.rects.shape[0]), "rounds": A.rounds, "steps": A.steps,
               "V_out": int(A.vertices.shape[0]), "scale": A.scale, "atlas_ms": round(best_a * 1e3, 3), "bake_ms": round(best_b * 1e3, 3),
               "occupancy": round(float(mask.double().mean()), 4), "peak_atlas_bytes": int(peak_atlas), "peak_bytes": int(peak),
               "nfdh_ms": nfdh_ms(v, t, R)}
        print(json.dumps(row), flush=True)
        rows.append(row)
        del A, tex, mask
        torch.cuda.empty_cache()
    return rows


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--spheres", type=int, nargs="*", default=[1, 16, 64], help="bumpy spheres, millions of triangles")
    ap.add_argument("--res", type=int, nargs="*", default=[2048, 4096, 8192])
    ap.add_argument("--mc", type=int, default=4096, help="marching-cubes sphere resolution (0: skip)")
    ap.add_argument("--reps", type=int, default=2)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "bench_uv_atlas_1gpu.json"))
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_uv_atlas.py measures the device path: no CUDA device")
    from bench_extract_mesh import gpu_info
    from bench_mesh_simplify import sphere_mesh
    from tensoflow_b200.geometry import simplify_mesh
    from tensoflow_b200.synthetic import bumpy_sphere
    dev = torch.device("cuda:0")
    result = {"info": gpu_info(), "rows": []}
    for m in args.spheres:
        v, t = (x.to(dev) for x in bumpy_sphere(*SPHERES[m]))
        result["rows"] += measure(f"bumpy_sphere{SPHERES[m]}", v, t, args.res, args.reps)
        del v, t
        torch.cuda.empty_cache()
    if args.mc:
        v, t = sphere_mesh(args.mc, dev)
        torch.cuda.empty_cache()
        result["rows"] += measure(f"mc_sphere {args.mc}^3", v, t, args.res, args.reps)
        vs, ts = simplify_mesh(v, t, 0, max_error=0.5 * 2.0 / (args.mc - 1))
        del v, t
        torch.cuda.empty_cache()
        result["rows"] += measure(f"mc_sphere {args.mc}^3 simplified to half a voxel", vs, ts, args.res, args.reps)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(result, f, indent=1)


if __name__ == "__main__":
    main()
