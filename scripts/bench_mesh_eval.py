"""Geometry evaluation on one GPU: closest-point queries (tf_bvh_closest_point) and geometry.evaluate_mesh.

Reports, with CUDA events after a warm-up of every shape:
  * closest-point queries per second for 10^6 points against synthetic.bumpy_sphere(1000, 500) (10^6 triangles, the config-3
    mesh) and against the extract_geometry mesh at 512^3 of a config-2-shaped field (G 512, C 36, H 256, A 128, 3 mip levels,
    seeded perturbation; the field of scripts/bench_extract_mesh.py).  Half the queries are uniform in the mesh's box grown by
    20 %, half are surface samples pushed off the surface by 1 % of the box;
  * evaluate_mesh end to end (sampling, two BVH builds on the host, two query passes, fp64 reductions) between the two meshes'
    normalised copies at the default 10^6 samples, by a host clock around a synchronised call;
  * the fp64 brute-force oracle (oracle/torch_oracle_geom.py) on the host for a small subset of the queries against the
    bumpy sphere, scaled to 10^6 queries and labelled as such;
  * the GPU name and power limit, read in the same run.
The BVH of a 10^6-triangle mesh (48 MB of triangles, about 17 MB of nodes, 4 MB of index map) fits in the 126 MB L2.

    python scripts/bench_mesh_eval.py [--reps 5] [--host-points 16] [--out results.json]
"""
import argparse
import json
import os
import subprocess
import sys
import time

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "scripts"))


def gpu_info():
    name = torch.cuda.get_device_name(0)
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30)
        power = q.stdout.strip() or "unknown"
    except (OSError, subprocess.SubprocessError):
        power = "unknown"
    return {"gpu": name, "power_limit_and_max_sm_clock": power}


def queries(v, t, n, seed):
    from tensoflow_b200.geometry import sample_surface
    g = torch.Generator(device=v.device).manual_seed(seed)
    lo, hi = v.min(0)[0], v.max(0)[0]
    span = hi - lo
    box = lo - 0.1 * span + 1.2 * span * torch.rand(n // 2, 3, device=v.device, generator=g)
    s, _, nrm = sample_surface(v, t, n - n // 2, seed=seed)
    off = s + 0.01 * float(span.max()) * torch.randn(s.shape[0], 1, device=v.device, generator=g) * nrm
    return torch.cat([box, off])


def time_queries(rt, q, reps):
    rt.closest_point(q)
    torch.cuda.synchronize()
    ms = []
    for _ in range(reps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        rt.closest_point(q)
        b.record()
        torch.cuda.synchronize()
        ms.append(a.elapsed_time(b))
    return min(ms), ms


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--points", type=int, default=1_000_000)
    ap.add_argument("--res", type=int, default=512)
    ap.add_argument("--host-points", type=int, default=16)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_mesh_eval.py measures the GPU path: no CUDA device")
    from bench_extract_mesh import make_shape
    from oracle import torch_oracle_geom as G
    from tensoflow_b200 import synthetic
    from tensoflow_b200.geometry import evaluate_mesh
    from tensoflow_b200.mc_ops import RayTracer
    dev = torch.device("cuda:0")
    result = {"info": gpu_info(), "points": args.points, "gpu": [], "host": []}

    bv, bt = (x.to(dev) for x in synthetic.bumpy_sphere(1000, 500))
    shape = make_shape(dev)
    t0 = time.perf_counter()
    ev, et = shape.extract_geometry([-1.0] * 3, [1.0] * 3, args.res)
    torch.cuda.synchronize()
    result["extract_geometry_s"] = time.perf_counter() - t0
    del shape
    torch.cuda.empty_cache()

    for name, (v, t) in {"bumpy_sphere(1000, 500)": (bv, bt), f"extract_geometry {args.res}^3": (ev, et)}.items():
        t0 = time.perf_counter()
        rt = RayTracer(v, t)
        build_s = time.perf_counter() - t0
        q = queries(v, t, args.points, seed=1)
        best, ms = time_queries(rt, q, args.reps)
        row = {"mesh": name, "triangles": int(t.shape[0]), "bvh_build_host_s": build_s, "query_ms": best, "query_ms_all": ms,
               "queries_per_s": args.points / (best * 1e-3)}
        result["gpu"].append(row)
        print(json.dumps(row), flush=True)
        if name.startswith("bumpy"):
            sub = q[:args.host_points // 2].cpu()
            sub = torch.cat([sub, q[args.points // 2:args.points // 2 + args.host_points - sub.shape[0]].cpu()])
            t0 = time.perf_counter()
            G.closest_point(sub, v.cpu(), t.cpu(), point_chunk=16, tri_chunk=65536)
            s = time.perf_counter() - t0
            result["host"].append({"mesh": name, "oracle_points": sub.shape[0], "oracle_cpu_s": s,
                                   "oracle_cpu_s_scaled_to_points (extrapolated, not run)": s * args.points / sub.shape[0],
                                   "threads": torch.get_num_threads()})
            print(json.dumps(result["host"][-1]), flush=True)
        del rt

    # evaluate_mesh end to end: the bumpy sphere (radius 0.5) and the extracted surface, each normalised into the unit box
    def normalised(v):
        lo, hi = v.min(0)[0], v.max(0)[0]
        return ((v - 0.5 * (lo + hi)) / float((hi - lo).max())).contiguous()
    pv, gv = normalised(ev), normalised(bv)
    evaluate_mesh(pv, et, gv, bt, n_samples=10_000)                     # warm-up
    torch.cuda.synchronize()
    runs = []
    for _ in range(max(1, args.reps // 2)):
        t0 = time.perf_counter()
        res = evaluate_mesh(pv, et, gv, bt)
        torch.cuda.synchronize()
        runs.append(time.perf_counter() - t0)
    result["evaluate_mesh"] = {"n_samples": 1_000_000, "s": min(runs), "s_all": runs, "result": {k: v for k, v in res.items()}}
    print(json.dumps(result["evaluate_mesh"], default=str), flush=True)
    print(json.dumps(result, default=str))
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(result, f, indent=1, default=str)


if __name__ == "__main__":
    main()
