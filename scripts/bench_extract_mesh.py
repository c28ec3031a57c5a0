"""Mesh extraction of the shape stage (ShapeRenderer.extract_geometry = extract_mesh.py's extract_fields + marching cubes) on a
config-2-shaped field (G 512, C 36, H 256, A 128, 3 mip levels, seeded perturbation): the dense path at lattice resolutions
512 and 1024 (--res) and the narrow band (isosurface.marching_cubes_narrowband, --nb-res) at 512, 1024, 2048 and 4096.  Where
both run at one resolution their repetitions alternate, so the two paths see the same machine state; 512 and 1024 are the two
sizes on the dense side of extract_geometry's switch at 2^31 lattice points.

Times, with CUDA events after a warm-up of every shape: the field evaluation (extract_fields) and each isosurface kernel
(tf_iso_count, tf_iso_vertices, tf_iso_triangles; the host prefix sum + size read between count and vertices is reported as
`scan_ms`).  Reports cells/s, the bytes each kernel must move (from the shapes: compulsory traffic only, see `bytes`), the share
of the 7.7 TB/s HBM bound, V and T, the GPU name and power limit, and the CPU oracle (oracle/torch_oracle_iso.py) at 128^3 and
256^3 as the host figure.  The 256^3 volume (64 MB) fits in the 126 MB L2; the 512^3 and 1024^3 volumes do not.

Narrow band, per phase with CUDA events (best of --reps): coarse (coarse lattice queries + brick test), fine (brick-point
queries, all rounds), grow (grow kernel + one host read per round), kernels (count, vertices, triangles), ordering (segment
key sort, prefix sums, size read, slot map); SDF queries against R^3, grow rounds, active bricks, peak memory, V and T.

    python scripts/bench_extract_mesh.py [--res 512 1024] [--nb-res 512 1024 2048 4096] [--reps 3] [--out results.json]
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

HBM_BYTES_PER_S = 7.7e12          # HGX B200 data sheet, one GPU


def gpu_info():
    name = torch.cuda.get_device_name(0)
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30)
        power = q.stdout.strip() or "unknown"
    except (OSError, subprocess.SubprocessError):
        power = "unknown"
    return {"gpu": name, "power_limit_and_max_sm_clock": power}


def make_shape(dev):
    from tensoflow_b200 import synthetic
    from tensoflow_b200.shape_renderer import ShapeRenderer
    torch.manual_seed(6033)
    G0 = 128
    m = ShapeRenderer(dict(device=dev, gridSize=[G0] * 3, sdf_n_comp=36, sdf_dim=256, app_dim=128, max_levels=1,
                           shader_config=dict(env_res=16, env_min_res=4)))
    for l in (1, 2):                      # the reference's upsampling schedule: 128 -> 256 -> 512, one more mip level each time
        m.sdf_network.upsample_volume_grid(torch.tensor([G0 << l] * 3))
        m.update_stepSize(torch.tensor([G0 << l] * 3), l + 1)
    synthetic.perturb_field(m.sdf_network, seed=1, noise=1e-2)
    return m


def timed_iso(u, thr=0.0):
    """marching_cubes (tensoflow_b200/isosurface.py) with CUDA events around each launch -> (ms per phase, V, T)"""
    from tensoflow_b200 import _lib
    from tensoflow_b200._lib import check, ptr, stream_ptr
    lib = _lib.load()
    nx, ny, nz = u.shape
    dev = u.device
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(5)]
    counts = torch.empty(2, nx * ny, device=dev, dtype=torch.int32)
    ev[0].record()
    check(lib.tf_iso_count(ptr(u), nx, ny, nz, thr, ptr(counts[0]), ptr(counts[1]), stream_ptr()), "tf_iso_count")
    ev[1].record()
    incl = torch.cumsum(counts, 1, dtype=torch.int64)
    n_verts, n_tris = incl[:, -1].tolist()
    offsets = incl - counts
    verts = torch.empty(n_verts, 3, device=dev)
    tris = torch.empty(n_tris, 3, device=dev, dtype=torch.int32)
    index = torch.empty(nx, ny, nz, device=dev, dtype=torch.int32)
    ev[2].record()
    check(lib.tf_iso_vertices(ptr(u), nx, ny, nz, thr, ptr(offsets[0]), ptr(verts), ptr(index), stream_ptr()), "tf_iso_vertices")
    ev[3].record()
    check(lib.tf_iso_triangles(ptr(u), nx, ny, nz, thr, ptr(offsets[1]), ptr(index), ptr(tris), stream_ptr()), "tf_iso_triangles")
    ev[4].record()
    torch.cuda.synchronize()
    ms = {"count_ms": ev[0].elapsed_time(ev[1]), "scan_ms": ev[1].elapsed_time(ev[2]), "vertices_ms": ev[2].elapsed_time(ev[3]),
          "triangles_ms": ev[3].elapsed_time(ev[4])}
    return ms, n_verts, n_tris


def best_scan(phases):
    return min(p["scan_ms"] for p in phases)


def kernel_bytes(R, V, T):
    """Compulsory HBM traffic per kernel: the volume is read once per kernel (4 B/point), row counts / offsets move 8 B per row,
    the index volume is written in full (4 B/point) and read back only around surface cells (not counted), vertices are 12 B,
    triangles 12 B."""
    N, rows = R ** 3, R ** 2
    return {"count": 4 * N + 8 * rows, "vertices": 4 * N + 4 * N + 8 * rows + 12 * V, "triangles": 4 * N + 8 * rows + 12 * T}


def timed_narrowband(shape, lo, hi, R):
    """ShapeRenderer.extract_geometry's narrow band at resolution R -> row of phase times (ms), counts, peak memory"""
    from tensoflow_b200.isosurface import marching_cubes_narrowband
    torch.cuda.synchronize()
    torch.cuda.reset_peak_memory_stats()
    base = torch.cuda.memory_allocated()
    stats = {}
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    with torch.no_grad():
        v, t = marching_cubes_narrowband(shape._extract_values, shape._extract_axes(lo, hi, R), 0.0, stats=stats)
    b.record()
    torch.cuda.synchronize()
    ms = {}
    for name, e0, e1 in stats["events"]:
        ms[f"{name}_ms"] = ms.get(f"{name}_ms", 0.0) + e0.elapsed_time(e1)
    row = {"total_ms": a.elapsed_time(b), **ms, "grow_rounds": stats["grow_rounds"], "bricks": stats["bricks"],
           "queries": stats["queries"], "queries_over_R3": stats["queries"] / R ** 3,
           "peak_bytes": torch.cuda.max_memory_allocated() - base, "V": v.shape[0], "T": t.shape[0]}
    del v, t
    return row


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--res", type=int, nargs="+", default=[512, 1024])
    ap.add_argument("--nb-res", type=int, nargs="+", default=[512, 1024, 2048, 4096])
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--host-res", type=int, nargs="+", default=[128, 256])
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_extract_mesh.py measures the GPU path: no CUDA device")
    from oracle.torch_oracle_iso import marching_cubes as oracle_mc
    from tensoflow_b200.isosurface import marching_cubes
    dev = torch.device("cuda:0")
    shape = make_shape(dev)
    lo, hi = [-1.0] * 3, [1.0] * 3
    result = {"info": gpu_info(), "field": "G 512, C 36, H 256, A 128, 3 levels, perturbed (seed 1, 1e-2)", "gpu": [], "host": [],
              "narrowband": []}
    for R in sorted(set(args.res) | set(args.nb_res)):
        if R in args.nb_res:
            timed_narrowband(shape, lo, hi, R)                          # warm-up
            nb_rows = []
        if R not in args.res:
            for _ in range(args.reps):
                nb_rows.append(timed_narrowband(shape, lo, hi, R))
            best = {k: min(r[k] for r in nb_rows) for k in nb_rows[0] if k.endswith("_ms")}
            row = {"res": R, **nb_rows[0], **best}
            result["narrowband"].append(row)
            print(json.dumps({"narrowband": row}), flush=True)
            torch.cuda.empty_cache()
            continue
        shape.extract_geometry(lo, hi, R)                              # warm-up of every shape of this resolution
        u = shape.extract_fields(lo, hi, R)
        timed_iso(u)
        torch.cuda.synchronize()
        field_ms, phases = [], []
        for _ in range(args.reps):
            if R in args.nb_res:                                       # alternate with the dense repetitions
                del u
                torch.cuda.empty_cache()
                nb_rows.append(timed_narrowband(shape, lo, hi, R))
                u = torch.empty(0)
            del u
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            u = shape.extract_fields(lo, hi, R)
            b.record()
            torch.cuda.synchronize()
            field_ms.append(a.elapsed_time(b))
            ms, V, T = timed_iso(u)
            phases.append(ms)
        v_ref, t_ref = marching_cubes(u)                               # the public entry point gives the same mesh
        assert v_ref.shape[0] == V and t_ref.shape[0] == T
        best = {k: min(p[k] for p in phases) for k in phases[0]}
        nbytes = kernel_bytes(R, V, T)
        iso_ms = best["count_ms"] + best["vertices_ms"] + best["triangles_ms"]
        row = {"res": R, "V": V, "T": T, "field_ms": min(field_ms), "field_points_per_s": R ** 3 / (min(field_ms) * 1e-3),
               **best, "iso_kernels_ms": iso_ms, "cells_per_s": (R - 1) ** 3 / (iso_ms * 1e-3), "bytes": nbytes,
               "hbm_share": {k: nbytes[k] / HBM_BYTES_PER_S / (best[f"{k}_ms"] * 1e-3) for k in nbytes}}
        result["gpu"].append(row)
        print(json.dumps(row), flush=True)
        if R in args.nb_res:
            best = {k: min(r[k] for r in nb_rows) for k in nb_rows[0] if k.endswith("_ms")}
            nrow = {"res": R, **nb_rows[0], **best, "dense_total_ms": min(field_ms) + iso_ms + best_scan(phases)}
            result["narrowband"].append(nrow)
            print(json.dumps({"narrowband": nrow}), flush=True)
        if R in args.host_res:
            uc = u.cpu()
            t0 = time.perf_counter()
            oracle_mc(uc)
            result["host"].append({"res": R, "oracle_cpu_s": time.perf_counter() - t0, "threads": torch.get_num_threads()})
        del u
        torch.cuda.empty_cache()
    for R in args.host_res:
        if R in args.res:
            continue
        uc = shape.extract_fields(lo, hi, R).cpu()
        t0 = time.perf_counter()
        oracle_mc(uc)
        result["host"].append({"res": R, "oracle_cpu_s": time.perf_counter() - t0, "threads": torch.get_num_threads()})
    print(json.dumps(result))
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(result, f, indent=1)


if __name__ == "__main__":
    main()
