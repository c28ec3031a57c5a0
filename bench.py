#!/usr/bin/env python
"""Benchmark of the TensoFlow hot path on B200 (see the contract in DESIGN.md).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]

Default workload = BASELINE.json configs[1]: shape stage, VM field 512^3 (C=36, H=256,
A=128, 3 mip levels), 8192-ray batch x 512 samples, forward + backward
(field stencil -> NeuS alpha -> compositing -> charbonnier + eikonal loss).
One "step" = one such pass over one synthetic ray batch.  Under torchrun every rank runs
its own 8192-ray batch (weak scaling) and the VM-factor / MLP gradients are summed with one
flat-bucket NCCL allreduce inside the timed region.

Prints ONE JSON line on rank 0.

The other BASELINE.json configurations have their own scripts (same timing rules, one JSON line each):
scripts/bench_material.py (config 3), scripts/bench_joint.py (config 4, torchrun), scripts/bench_relight.py (config 5,
torchrun), scripts/bench_shape_renderer.py (the full ShapeRenderer.forward module path), scripts/bench_adam.py (optimizer step).
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import torch  # noqa: E402

SHAPE_CFG = dict(G=512, C=36, H=256, A=128, L=3, rays=8192, samples=512)


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return dict(hbm=d["hbm_gbs"], tf=d["bf16_tflops_sustained"], tf_burst=d["bf16_tflops"], src="measured")
    return dict(hbm=6650.0, tf=1400.0, tf_burst=1590.0, src="fallback")


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled during the timed region."""
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.rows = []
        self.proc = None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-i", str(index), "-lms", "100"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        for r in self.rows:
            f = [x.strip() for x in r.split(",")]
            if len(f) < 6:
                continue
            try:
                sm.append(float(f[0])); mx.append(float(f[1]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[2:6]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def profiled_traffic(kernel):
    """dram__bytes_read.sum + dram__bytes_write.sum of one launch of `kernel`, from the committed `ncu --set full` summary
    (profiles/r<round>_<kernel>_ncu_full_summary.txt, newest round first; the capture's launch is one 4 GiB-workspace slice of
    this same command, the same size as the bench's)."""
    path = None
    for rnd in ("r2", "r1"):
        cand = os.path.join(ROOT, "profiles", f"{rnd}_{kernel.replace('sdf_', '')}_ncu_full_summary.txt")
        if os.path.exists(cand):
            path = cand
            break
    if path is None:
        return None
    tot, scale = 0.0, {"byte": 1.0, "Kbyte": 1e3, "Mbyte": 1e6, "Gbyte": 1e9, "Tbyte": 1e12}
    for line in open(path):
        f = line.split()
        if len(f) >= 3 and f[0] in ("dram__bytes_read.sum", "dram__bytes_write.sum") and f[2] in scale:
            tot += float(f[1]) * scale[f[2]]
    return tot or None


def shape_algorithmic(cfg, n_samples, n_rays):
    """SURVEY.md 8d: algorithmic bytes and decoder FLOPs of one shape-stage step."""
    C, H, A, G, L = cfg["C"], cfg["H"], cfg["A"], cfg["G"], cfg["L"]
    K = 3 * C + 3
    p_vm = 3 * C * 4 * sum((G >> l) ** 2 + (G >> l) for l in range(L))
    by = n_samples * 1128 + n_rays * 120 + 3 * p_vm
    fwd_flops = n_samples * (2 * (K * H + H * (1 + A)) + 6 * 2 * (K * H + H))
    return by, fwd_flops


def build_shape(cfg, device, seed=0):
    from tensoflow_b200.fields import TensoSDF
    from tensoflow_b200 import synthetic
    torch.manual_seed(6033)   # reference trainer seed (train/trainer_inv.py:42)
    aabb = torch.tensor([[-1.0] * 3, [1.0] * 3])
    G0 = cfg["G"] >> (cfg["L"] - 1)
    field = TensoSDF(torch.tensor([G0] * 3), aabb, device=device, sdf_n_comp=cfg["C"], sdf_dim=cfg["H"], app_dim=cfg["A"],
                     init_n_levels=1, sdf_multires=0)
    for l in range(1, cfg["L"]):   # bilinear upsampling exactly as the reference schedule does
        field.upsample_volume_grid(torch.tensor([G0 << l] * 3))
    synthetic.perturb_field(field, seed=seed + 1, noise=1e-2)
    variance = torch.nn.Parameter(torch.tensor(0.3, device=device))
    return field, variance


def shape_step(field, variance, rays, cfg, loss_scale=1.0):
    """fwd + bwd of the shape-stage hot path on one ray batch (already on the device): (loss, samples, render outputs)."""
    from tensoflow_b200 import synthetic
    from tensoflow_b200.shape_renderer import render_core, charbonnier
    t0, t1, idx = synthetic.uniform_samples(rays["rays_o"], rays["dirs"], field.aabb, cfg["samples"])
    out = render_core(field, variance, synthetic.simple_color_fn, rays["rays_o"], rays["dirs"], rays["radiis"], rays["rays_cos"],
                      t0, t1, idx, cos_anneal_ratio=1.0)
    loss = charbonnier(out["ray_rgb"], rays["rgbs"]).mean() + 0.1 * out["gradient_error"].mean()
    (loss * loss_scale).backward()
    return loss.detach(), int(idx.shape[0]), out


DUMP_SAMPLE = 1 << 18      # elements written of a larger array


def dump_array(t):
    """`t` as a float32 host array: whole when it has at most DUMP_SAMPLE elements, otherwise DUMP_SAMPLE elements of its
    flattened values at sorted indices drawn from a fixed seed (the same indices in every run of the same configuration)."""
    t = t.detach()
    if t.numel() > DUMP_SAMPLE:
        idx = torch.randint(t.numel(), (DUMP_SAMPLE,), generator=torch.Generator().manual_seed(0)).sort().values
        t = t.reshape(-1)[idx.to(t.device)]
    return t.float().cpu().numpy()


def step_outputs(loss, out, field, variance):
    """What one training step hands its caller: the loss, the render outputs and the parameter gradients (host arrays)."""
    arrays = {"loss": dump_array(loss)}
    arrays.update({k: dump_array(v) for k, v in out.items() if torch.is_tensor(v)})
    arrays.update({f"grad.{n}": dump_array(p.grad) for n, p in field.named_parameters() if p.grad is not None})
    arrays["grad.variance"] = dump_array(variance.grad)
    return arrays


def cpu_baseline_shape(cfg, n_rays, iters, threads):
    """The oracle port of the reference path, timed on the host cores (fwd + bwd)."""
    from oracle import torch_oracle as O
    from tensoflow_b200 import synthetic
    torch.set_num_threads(threads)
    torch.manual_seed(6033)
    aabb = [[-1.0] * 3, [1.0] * 3]
    G0 = cfg["G"] >> (cfg["L"] - 1)
    f = O.TensoSDF([G0] * 3, aabb, sdf_n_comp=cfg["C"], sdf_dim=cfg["H"], app_dim=cfg["A"], init_n_levels=1)
    for l in range(1, cfg["L"]):
        f.upsample_volume_grid(torch.tensor([G0 << l] * 3))
    synthetic.perturb_field(f, seed=1, noise=1e-2)
    var = torch.tensor(0.3, requires_grad=True)
    rays = synthetic.make_rays(n_rays, seed=0)
    times = []
    for it in range(iters + 1):
        t = time.perf_counter()
        t0, t1, idx = synthetic.uniform_samples(rays["rays_o"], rays["dirs"], f.aabb, cfg["samples"])
        r = O.shape_render_core(f, var, rays["rays_o"], rays["dirs"], rays["radiis"], rays["rays_cos"], t0, t1, idx,
                                synthetic.simple_color_fn, cos_anneal_ratio=1.0)
        loss = O.charbonnier(r["ray_rgb"], rays["rgbs"]).mean() + 0.1 * r["gradient_error"].mean()
        for p in f.parameters():
            p.grad = None
        loss.backward()
        if it > 0:
            times.append(time.perf_counter() - t)
    return n_rays / statistics.median(times), times


def parity_check(field, variance, cfg, dev, n_rays):
    """The benchmarked field and step on a ray subset against the oracle (fp64, PyTorch on the same device; checker only):
    max|a-b| / max|b| of the rendered colour / SDF / alpha and of the parameter gradients."""
    from oracle import torch_oracle as O
    from tensoflow_b200 import synthetic
    from tensoflow_b200.shape_renderer import render_core, charbonnier
    rays = synthetic.make_rays(n_rays, seed=4242, device=dev)
    t0, t1, idx = synthetic.uniform_samples(rays["rays_o"], rays["dirs"], field.aabb, cfg["samples"])
    dt = torch.float64
    G0 = cfg["G"] >> (cfg["L"] - 1)
    o = O.TensoSDF([G0] * 3, [[-1.0] * 3, [1.0] * 3], sdf_n_comp=cfg["C"], sdf_dim=cfg["H"], app_dim=cfg["A"], init_n_levels=1, dtype=dt)
    for l in range(1, cfg["L"]):
        o.upsample_volume_grid(torch.tensor([G0 << l] * 3))
    synthetic.copy_field_params(field, o)
    o = o.to(dev)
    o.update_gridSize(o.gridSize, o.n_levels)
    var_o = variance.detach().to(dt).clone().requires_grad_()
    ro = O.shape_render_core(o, var_o, rays["rays_o"].to(dt), rays["dirs"].to(dt), rays["radiis"].to(dt), rays["rays_cos"].to(dt),
                             t0.to(dt), t1.to(dt), idx, synthetic.simple_color_fn, cos_anneal_ratio=1.0)
    (O.charbonnier(ro["ray_rgb"], rays["rgbs"].to(dt)).mean() + 0.1 * ro["gradient_error"].mean()).backward()
    for p in list(field.parameters()) + [variance]:
        p.grad = None
    rc = render_core(field, variance, synthetic.simple_color_fn, rays["rays_o"], rays["dirs"], rays["radiis"], rays["rays_cos"],
                     t0, t1, idx, cos_anneal_ratio=1.0)
    (charbonnier(rc["ray_rgb"], rays["rgbs"]).mean() + 0.1 * rc["gradient_error"].mean()).backward()

    def rel(a, b):
        return float((a.detach().double() - b.detach().double()).abs().max() / b.detach().double().abs().max().clamp_min(1e-30))

    errs = {"rays": n_rays, "samples": int(idx.shape[0]), "rgb": rel(rc["ray_rgb"], ro["ray_rgb"]), "sdf": rel(rc["sdf"], ro["sdf"]),
            "alpha": rel(rc["alpha"], ro["alpha"]), "d_variance": rel(variance.grad, var_o.grad)}
    og = dict(o.named_parameters())
    for name, p in field.named_parameters():
        errs["d_" + name] = rel(p.grad, og[name].grad)
    errs["max_output"] = max(errs["rgb"], errs["sdf"], errs["alpha"])
    errs["max_grad"] = max(v for k, v in errs.items() if k.startswith("d_"))
    errs["within_tolerance"] = bool(errs["max_output"] < 1e-4 and errs["max_grad"] < 1e-3)
    for p in list(field.parameters()) + [variance]:
        p.grad = None
    return errs


def secondary_lines():
    """Config 3 (material stage) and the module-level shape step (ShapeRenderer.forward), measured in this same run by their
    own scripts in child processes (same box, same clocks): so that they are driver-visible, not builder-only, numbers."""
    out = {}
    for key, script, extra in (("material_stage_config3", "bench_material.py", ["--steps", "5"]),
                               ("shape_renderer_forward_4096x128", "bench_shape_renderer.py", ["--steps", "5"])):
        try:
            r = subprocess.run([sys.executable, os.path.join(ROOT, "scripts", script), *extra], capture_output=True, text=True, timeout=600)
            line = [l for l in r.stdout.splitlines() if l.startswith("{")]
            d = json.loads(line[-1]) if line else {"error": (r.stderr or "no output")[-300:]}
            out[key] = {k: d[k] for k in ("metric", "value", "unit", "ms_per_step", "gpu_launches_per_step", "config", "rays", "error") if k in d}
        except Exception as e:  # noqa: BLE001
            out[key] = {"error": repr(e)[:300]}
    return out


def config1_line(dev, steps):
    """BASELINE.json configs[0] (the reference's CPU-runnable case): VM field 128^3, 48 feature components (C = 16), H = 128,
    4096 rays x 128 samples, fwd + bwd, device-resident rays, CUDA events."""
    from tensoflow_b200 import synthetic
    cfg = dict(G=128, C=16, H=128, A=128, L=1, rays=4096, samples=128)
    field, variance = build_shape(cfg, dev)
    params = list(field.parameters()) + [variance]
    rays = [synthetic.make_rays(cfg["rays"], seed=50 + b, device=dev) for b in range(2)]
    for i in range(3):
        for p in params:
            p.grad = None
        shape_step(field, variance, rays[i % 2], cfg)
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for i in range(steps):
        for p in params:
            p.grad = None
        shape_step(field, variance, rays[i % 2], cfg)
    b.record()
    torch.cuda.synchronize()
    ms = a.elapsed_time(b) / steps
    return {"metric": "train rays/sec (fwd+bwd)", "value": cfg["rays"] / (ms / 1e3), "unit": "rays/s", "ms_per_step": ms,
            "config": {"workload": workload_name(cfg)}}


def workload_name(cfg):
    return (f"shape stage: TensoSDF VM field {cfg['G']}^3 (C={cfg['C']}, H={cfg['H']}, A={cfg['A']}, {cfg['L']} mip levels), "
            f"{cfg['rays']}-ray batch x {cfg['samples']} samples, fwd+bwd")


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cfg = dict(SHAPE_CFG)
    threads = len(os.sched_getaffinity(0))
    n_rays = args.ref_rays
    from oracle import torch_oracle as O  # noqa: F401
    t_all = time.perf_counter()
    # a 512-ray step of the port costs 10-25 s on the host cores: the arm times a BOUNDED number of steps (<= 3 after one
    # warm-up step) whatever K / W say, so that the run ends within a few minutes; the line says how many
    timed = max(1, min(args.steps, args.ref_steps))
    rps, times = cpu_baseline_shape(cfg, n_rays, timed, threads)
    ms = 1e3 * statistics.median(times)
    val = n_rays / (ms / 1e3)
    line = {
        "impl": "reference", "metric": "train rays/sec (fwd+bwd)", "value": val, "unit": "rays/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": workload_name(cfg),
                   "sample": f"{n_rays} of {cfg['rays']} rays (BASELINE.md 3: 1/16 subset) x {cfg['samples']} samples per step; "
                             f"{len(times)} timed steps after 1 warm-up step (bounded sample, not K / W)"},
        "cpu_baseline": {"value": val, "unit": "rays/s", "cores": threads, "kind": "port",
                         "sample": f"oracle/torch_oracle.py (PyTorch CPU restatement of the reference path, pinned bit for bit to the "
                                   f"reference classes), {n_rays} rays x {cfg['samples']} samples per step, median of {len(times)} steps",
                         "step_seconds": [round(t, 2) for t in times]},
        "e2e": {"value": val, "unit": "rays/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "wall_s": time.perf_counter() - t_all,
    }
    print(json.dumps(line), flush=True)


def run_ours(args):
    import torch.distributed as dist
    from tensoflow_b200 import build as tb
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise RuntimeError("bench.py needs a CUDA device: tensoflow_b200 has no CPU fallback (use --impl reference for the CPU arm)")
    if rank == 0:
        tb.build()
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
        dist.barrier()
    from tensoflow_b200 import _lib, ops, synthetic
    _lib.load()
    cfg = dict(SHAPE_CFG)
    if args.rays:
        cfg["rays"] = args.rays
    if args.samples:
        cfg["samples"] = args.samples
    field, variance = build_shape(cfg, dev)
    params = list(field.parameters()) + [variance]
    # rank-specific synthetic ray batches in pinned host memory (the reference keeps its rays on the CPU too,
    # network/shapeRenderer.py:780)
    n_batches = 4
    host = [{k: v.pin_memory() for k, v in synthetic.make_rays(cfg["rays"], seed=1000 * rank + b).items()} for b in range(n_batches)]
    h2d = sum(v.numel() * v.element_size() for v in host[0].values())
    bucket = None
    if world > 1:
        from tensoflow_b200.dist import FlatGradBucket
        bucket = FlatGradBucket(params)

    def zero_grads():
        if bucket is not None:
            bucket.begin_step()        # one memset of the flat buffer; the backward kernels scatter straight into its views
        else:
            for p in params:
                p.grad = None

    def allreduce_grads():
        # one in-place sum-allreduce of the flat fp32 gradient buffer (VM planes / lines, MLP weights, variance) on NCCL's
        # stream; p.grad of every parameter is a view into it afterwards, as an optimizer step would consume them
        if bucket is not None:
            bucket.allreduce(async_op=True)
            bucket.finish()

    def step_device(b):
        rays = {k: v.to(dev, non_blocking=True) for k, v in host[b % n_batches].items()}
        return rays

    resident = [{k: v.to(dev) for k, v in h.items()} for h in host]
    n_samples = 0
    # ---- warm-up ----
    for i in range(max(args.warmup, 3)):
        zero_grads()
        _, n_samples, _ = shape_step(field, variance, resident[i % n_batches], cfg, 1.0 / world)
        allreduce_grads()
    torch.cuda.synchronize()

    def timed(run_step, timers):
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        ops.KernelTimers.reset(timers)
        lib = _lib.load()
        lib.tf_kernel_timing_reset()
        lib.tf_kernel_timing_enable(1 if timers else 0)
        l0 = _lib.launch_count()
        sampler = ClockSampler(local) if rank == 0 else None
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        prof = timers and bool(os.environ.get('TF_PROFILE_RANGE'))      # ncu --profile-from-start off: only the timed steps
        if prof:
            torch.cuda.profiler.start()
        a.record()
        for i in range(args.steps):
            run_step(i)
        b.record()
        torch.cuda.synchronize()
        if prof:
            torch.cuda.profiler.stop()
        if world > 1:
            dist.barrier()
        ms = a.elapsed_time(b)
        clocks = sampler.stop() if sampler else None
        launches = _lib.launch_count() - l0
        tot = ops.KernelTimers.totals_ms()
        ops.KernelTimers.reset(False)
        kern = {}
        if timers:
            import ctypes as C
            for name in ("sdf_stencil_fwd_tc", "sdf_stencil_bwd_tc", "xty_tc", "linear_tc"):
                t_ms, n = C.c_double(0.0), C.c_int32(0)
                if lib.tf_kernel_timing_read(name.encode(), C.byref(t_ms), C.byref(n)) == 0 and n.value:
                    kern[name] = (t_ms.value, n.value)
        lib.tf_kernel_timing_enable(0)
        lib.tf_kernel_timing_reset()
        if world > 1:
            t = torch.tensor([ms], device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t)
        return ms, clocks, launches, tot, kern

    # ---- device-resident timing (value) ----
    last = {}

    def step_resident(i):
        zero_grads()
        loss, _, out = shape_step(field, variance, resident[i % n_batches], cfg, 1.0 / world)
        allreduce_grads()
        if args.dump_outputs and i == args.steps - 1:     # only the last step's outputs are kept alive past their step
            last.update(loss=loss, out=out)

    ms, clocks, launches, ktimes, kern = timed(step_resident, True)
    # copied out before the next timed window overwrites the gradients (in place in the flat bucket when world > 1)
    dumped = step_outputs(last["loss"], last["out"], field, variance) if (args.dump_outputs and rank == 0) else None
    last.clear()

    # ---- end-to-end timing: pinned host rays -> H2D -> step -> D2H loss ----
    losses = []

    def step_e2e(i):
        zero_grads()
        rays = step_device(i)
        loss, _, _ = shape_step(field, variance, rays, cfg, 1.0 / world)
        allreduce_grads()
        losses.append(float(loss.cpu()))   # D2H read of the step's result

    ms_e2e, _, _, _, _ = timed(step_e2e, False)

    # ---- config 4 (joint shape + material step, strong scaling over the same ranks), so that it is in the driver's record ----
    joint = None
    if world > 1 and not args.no_secondary:
        try:
            sys.path.insert(0, os.path.join(ROOT, "scripts"))
            import bench_joint
            joint = bench_joint.run_joint(bench_joint.parse_args([]), own_process_group=False)
        except Exception as e:  # noqa: BLE001
            joint = {"metric": "joint shape+material train rays/sec (fwd+bwd)", "error": repr(e)[:300]} if rank == 0 else None
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    pk = peaks()
    rays_total = cfg["rays"] * world
    value = rays_total * args.steps / (ms / 1e3)
    e2e = rays_total * args.steps / (ms_e2e / 1e3)
    by, fwd_flops = shape_algorithmic(cfg, n_samples, cfg["rays"])
    # dominant kernel: per-kernel CUDA-event times recorded inside the library on the launching stream
    # (fwd: 1x, bwd: 2x the minimal decoder FLOPs; SURVEY 8d)
    kt = {k: v[0] / max(v[1], 1) for k, v in ktimes.items()}
    roof = None
    if kern:
        dom = max(kern, key=lambda k: kern[k][0])
        dom_ms, dom_n = kern[dom]
        per_step_ms = dom_ms / args.steps
        flops = fwd_flops * (2 if "bwd" in dom else 1) if "stencil" in dom else 0
        ach = flops / (per_step_ms / 1e3) / 1e12
        roof = {"bound": "tensor", "kernel": dom + "_kernel", "achieved": ach, "peak": pk["tf"], "unit": "TFLOP/s", "frac": ach / pk["tf"],
                "traffic": profiled_traffic(dom), "traffic_unit": "bytes per launch (dram read + write, ncu --set full, profiles/)",
                "peak_source": f"{pk['src']} dense bf16 sustained (cuBLAS)",
                "ms_per_launch": dom_ms / max(dom_n, 1), "launches_per_step": dom_n / args.steps, "ms_per_step": per_step_ms,
                "share_of_step": dom_ms / ms,
                "note": ("achieved = algorithmic fp32 decoder FLOPs of the step's samples / the kernel's summed launch time; the MMAs run "
                         "as 3xTF32 (fp32-level accuracy), i.e. 3 tensor-core passes at the tf32 rate (1/2 of bf16) per algorithmic FLOP, "
                         "so the tensor pipe itself is ~6x busier than `frac`; the kernel is bound by the L2 gather of plane/line texels, "
                         "the RED.v4 scatter of their gradients and the softplus epilogue, not by the MMAs (profiles/)"),
                "kernels_ms_per_step": {k: round(v[0] / args.steps, 3) for k, v in kern.items()},
                "calls_ms": {k: round(v, 3) for k, v in kt.items()},
                "hbm_algorithmic": {"bytes_per_step": by, "GBps_at_step_rate": by / (ms / args.steps / 1e3) / 1e9,
                                    "frac_of_hbm_peak": by / (ms / args.steps / 1e3) / 1e9 / pk["hbm"]}}
    cpu = None
    if world == 1 and not args.no_cpu_baseline:
        threads = len(os.sched_getaffinity(0))
        rps, times = cpu_baseline_shape(cfg, args.ref_rays, 1, threads)
        cpu = {"value": rps, "unit": "rays/s", "cores": threads, "kind": "port",
               "sample": f"oracle port, {args.ref_rays} of {cfg['rays']} rays x {cfg['samples']} samples, fwd+bwd, "
                         f"{len(times)} timed step after 1 warm-up step ({times[0]:.1f} s)"}
    check = parity_check(field, variance, cfg, dev, args.check_rays) if (world == 1 and args.check_rays > 0) else None
    secondary = None
    if world == 1 and not args.no_secondary:
        secondary = secondary_lines()
        secondary["config1_128cube_4096x128"] = config1_line(dev, args.steps)
    if joint is not None:
        secondary = {"joint_config4": {k: joint[k] for k in ("metric", "value", "unit", "ms_per_step", "n_gpus", "scaling", "config") if k in joint}}
    line = {
        "metric": "train rays/sec (fwd+bwd)", "value": value, "unit": "rays/s", "n_gpus": world, "steps": args.steps,
        "warmup": max(args.warmup, 3), "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": workload_name(cfg), "samples_per_step_per_gpu": n_samples,
                   "colour": "synthetic.simple_color_fn (shading network not in this workload)",
                   "l2": "working set per step (>= 2 GB of per-sample tensors) exceeds the 126 MB L2; no explicit flush",
                   "parallelism": f"dp{world} (ray sharding + flat fp32 gradient allreduce)" if world > 1 else "single GPU"},
        "roofline": roof, "cpu_baseline": cpu,
        "e2e": {"value": e2e, "unit": "rays/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": 4, "ms_per_step": ms_e2e / args.steps},
        "gpu_launches": launches, "clocks": clocks, "loss": losses[-1] if losses else None,
        "check": check, "secondary": secondary,
    }
    if dumped is not None:
        import numpy as np
        os.makedirs(args.dump_outputs, exist_ok=True)
        for name, a in dumped.items():
            np.save(os.path.join(args.dump_outputs, name + ".npy"), a)
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--rays", type=int, default=0, help="override rays per GPU per step (parity/debug only)")
    ap.add_argument("--samples", type=int, default=0, help="override samples per ray (parity/debug only)")
    ap.add_argument("--ref-rays", type=int, default=512, help="rays per CPU-baseline step (BASELINE.md 3: 1/16 of the batch)")
    ap.add_argument("--ref-steps", type=int, default=3, help="upper bound on the timed steps of the CPU arm")
    ap.add_argument("--check-rays", type=int, default=64, help="rays of the parity check against the oracle (0 = off)")
    ap.add_argument("--no-secondary", action="store_true", help="skip the config-3 / module-path lines of `secondary`")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write the loss, render outputs and parameter gradients of the last timed step "
                         "as DIR/<name>.npy (float32; an array of more than 2^18 elements as a fixed seeded sample of them)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the outputs of the CUDA path (--impl ours)")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
