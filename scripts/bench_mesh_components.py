"""Mesh clean-up on the GPU (geometry.mesh_components / remove_small_components, tf_mesh_components) against the host path a
user would otherwise take (copy the mesh to the host, then scipy.sparse.csgraph.connected_components and the numpy filter of
oracle/torch_oracle_cc.py), on bumpy spheres of 1 M, 4 M, 16 M and 64 M triangles (the meshes of bench_bvh_build.py), each
without and with 1000 floaters (small closed spheres around it), and on ShapeRenderer.extract_geometry meshes of a
config-2-shaped field (the field of bench_extract_mesh.py) at 2048^3 and 4096^3.

Per mesh: V, T, components; tf_mesh_components alone (CUDA events around the call, best of --reps after a warm-up);
mesh_components and remove_small_components(min_fraction) end to end (wall time to a device synchronise, host reads
included, best of --reps); the host path once (copy to the host included); the device results compared with the host's
exactly.  GPU name and power limit go with the numbers.  The index and parent arrays of the larger meshes (12 B per triangle,
4 B per vertex) are above the 126 MB L2.

    python scripts/bench_mesh_components.py [--spheres 1 4 16 64] [--res 2048 4096] [--reps 5] [--out results.json]
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

SPHERES = {1: (1000, 501), 4: (2000, 1001), 16: (4000, 2001), 64: (8000, 4001)}     # 2 nu (nv - 1) triangles
N_FLOATERS = 1000


def with_floaters(v, t, n=N_FLOATERS, seed=0):
    """the mesh plus n small bumpy spheres (r = 0.004 .. 0.012, 224 triangles each) centred at 0.65 <= |c| <= 0.95, appended"""
    from tensoflow_b200.synthetic import bumpy_sphere
    g = torch.Generator().manual_seed(seed)
    sv, st = bumpy_sphere(16, 8, r=1.0, bump=0.1)
    vs, ts = [v], [t]
    base = v.shape[0]
    while len(vs) <= n:
        c = torch.rand(3, generator=g) * 2 - 1
        if not 0.65 <= float(c.norm()) <= 0.95:
            continue
        r = 0.004 + 0.008 * float(torch.rand(1, generator=g))
        vs.append(sv * r + c)
        ts.append(st + base)
        base += sv.shape[0]
    return torch.cat(vs), torch.cat(ts)


def best_wall(fn, reps):
    fn()
    out = []
    for _ in range(reps):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        fn()
        torch.cuda.synchronize()
        out.append(time.perf_counter() - t0)
    return min(out)


def kernel_ms(t, V, reps):
    """tf_mesh_components alone between CUDA events (init, link, flatten, count)"""
    from tensoflow_b200 import _lib
    from tensoflow_b200._lib import check, ptr, stream_ptr
    lib = _lib.load()
    root = torch.empty(V, device=t.device, dtype=torch.int32)
    cnt = torch.empty(V, device=t.device, dtype=torch.int32)
    call = lambda: check(lib.tf_mesh_components(ptr(t), t.shape[0], V, ptr(root), ptr(cnt), stream_ptr()), "tf_mesh_components")
    call()
    ms = []
    for _ in range(reps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        call()
        b.record()
        torch.cuda.synchronize()
        ms.append(a.elapsed_time(b))
    return min(ms)


def measure(name, v, t, reps, min_fraction, host):
    from oracle import torch_oracle_cc as O
    from tensoflow_b200.geometry import mesh_components, remove_small_components
    V, T = int(v.shape[0]), int(t.shape[0])
    t = t.to(torch.int32).contiguous()
    row = {"mesh": name, "V": V, "T": T, "min_fraction": min_fraction}
    root, cnt = mesh_components(v, t)
    kv, kt = remove_small_components(v, t, min_fraction)
    row["components"] = int((cnt > 0).sum())
    row["T_kept"], row["V_kept"] = int(kt.shape[0]), int(kv.shape[0])
    row["kernel_ms"] = kernel_ms(t, V, reps)
    # compulsory HBM traffic: 16 B per vertex (init and flatten) and 16 B per triangle (12 B of indices in the link pass, 4 B in
    # the count pass); the gathered parent loads of the finds come on top
    row["compulsory_GB_per_s"] = (16 * V + 16 * T) / (row["kernel_ms"] * 1e-3) / 1e9
    row["mesh_components_s"] = best_wall(lambda: mesh_components(v, t), reps)
    row["remove_small_components_s"] = best_wall(lambda: remove_small_components(v, t, min_fraction), reps)
    if host:
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        hv, ht = v.cpu().numpy(), t.cpu().numpy()
        h_root, h_cnt = O.mesh_components(V, ht)
        row["host_components_s"] = time.perf_counter() - t0
        t0 = time.perf_counter()
        hv, ht = v.cpu().numpy(), t.cpu().numpy()
        wv, wt = O.remove_small_components(hv, ht, min_fraction)
        row["host_remove_small_components_s"] = time.perf_counter() - t0
        row["equal_to_host"] = bool((root.cpu().numpy() == h_root).all() and (cnt.cpu().numpy() == h_cnt).all()
                                    and kv.cpu().numpy().tobytes() == wv.tobytes() and kt.cpu().numpy().tobytes() == wt.tobytes())
        row["speedup_components"] = row["host_components_s"] / row["mesh_components_s"]
        row["speedup_remove_small_components"] = row["host_remove_small_components_s"] / row["remove_small_components_s"]
    else:
        row["host_components_s"] = row["host_remove_small_components_s"] = "not measured"
    print(json.dumps(row), flush=True)
    return row


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--spheres", type=int, nargs="*", default=[1, 4, 16, 64], help="bumpy spheres, millions of triangles")
    ap.add_argument("--res", type=int, nargs="*", default=[2048, 4096], help="extract_geometry resolutions")
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--min-fraction", type=float, default=0.01)
    ap.add_argument("--no-host-above", type=int, default=1 << 31, help="skip the host path above this many triangles")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_mesh_components.py measures the device path: no CUDA device")
    from bench_extract_mesh import gpu_info, make_shape
    from tensoflow_b200.synthetic import bumpy_sphere
    dev = torch.device("cuda:0")
    result = {"info": gpu_info(), "rows": []}
    for m in args.spheres:
        v, t = bumpy_sphere(*SPHERES[m])
        for floaters in (False, True):
            vv, tt = with_floaters(v, t) if floaters else (v, t)
            name = f"bumpy_sphere{SPHERES[m]}" + (f" + {N_FLOATERS} floaters" if floaters else "")
            vv, tt = vv.to(dev), tt.to(dev)
            result["rows"].append(measure(name, vv, tt, args.reps, args.min_fraction, tt.shape[0] <= args.no_host_above))
            del vv, tt
            torch.cuda.empty_cache()
    if args.res:
        shape = make_shape(dev)
        lo, hi = [-1.0] * 3, [1.0] * 3
        for R in args.res:
            with torch.no_grad():
                v, t = shape.extract_geometry(lo, hi, R)
                cleaned_s = best_wall(lambda: shape.extract_geometry(lo, hi, R, min_component_fraction=args.min_fraction), 1)
                plain_s = best_wall(lambda: shape.extract_geometry(lo, hi, R), 1)
            row = measure(f"extract_geometry {R}^3", v, t, args.reps, args.min_fraction, t.shape[0] <= args.no_host_above)
            row["extract_geometry_s"] = plain_s
            row["extract_geometry_with_clean_up_s"] = cleaned_s
            print(json.dumps({"extract_geometry": R, "plain_s": plain_s, "with_clean_up_s": cleaned_s}), flush=True)
            result["rows"].append(row)
            del v, t
            torch.cuda.empty_cache()
    if args.out:
        with open(args.out, "w") as f:
            json.dump(result, f, indent=1)


if __name__ == "__main__":
    main()
