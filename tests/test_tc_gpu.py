"""tcgen05 self-test: the tensor-core GEMM primitive (TMEM accumulator, smem descriptors, mbarrier
commit) against an fp64 matmul; tf32 operand splitting must reach fp32-level accuracy."""
import pytest
import torch

pytestmark = pytest.mark.gpu


def _probe(N, K, passes, a_mode=0, b_mode=0, a_lbo=128, mn_sbo=128, swap_mn=0, reps=1):
    """tests/probes/_bin/tc_probe (standalone executable built by tensoflow_b200.build.build_probes): D = A B^T for one layout
    configuration against an fp64 host product -> parsed JSON line."""
    import json
    import subprocess
    from tensoflow_b200 import build
    exe = build.build_probes()
    out = subprocess.run([str(exe)] + [str(x) for x in (N, K, passes, reps, a_mode, b_mode, a_lbo, mn_sbo, swap_mn)], capture_output=True,
                         text=True, timeout=120)
    assert out.returncode == 0, out.stdout + out.stderr
    return json.loads(out.stdout.strip().splitlines()[-1])


@pytest.mark.parametrize("N,K", [(128, 8), (128, 64), (256, 32), (256, 56), (112, 32)])
@pytest.mark.parametrize("a_mode,a_lbo", [(0, 128), (0, 144), (3, 128)])
def test_tcgen05_gemm_matches_fp64(N, K, a_mode, a_lbo):
    """the operand layouts the fused kernels use: K-major no-swizzle A (dense and 144-byte padded K chunks) and A from tensor
    memory, K-major no-swizzle B; plain tf32 and the 3xTF32 split"""
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    if a_mode == 3 and K % 16:
        pytest.skip("the TS-mode probe stores A in 16-column pieces")
    e1 = _probe(N, K, 1, a_mode=a_mode, a_lbo=a_lbo)["rel_err"]
    e3 = _probe(N, K, 3, a_mode=a_mode, a_lbo=a_lbo)["rel_err"]
    print(f"N={N} K={K} a_mode={a_mode} lbo={a_lbo}: tf32 {e1:.2e}  3xtf32 {e3:.2e}")
    assert e1 < 5e-3, e1          # plain tf32: ~1e-3
    assert e3 < 2e-6, e3          # split: fp32 level


@pytest.mark.parametrize("rows,M,N", [(1000, 256, 112), (4099, 128, 256), (31, 128, 16), (20000, 256, 64), (9000, 256, 256), (5000, 48, 240),
                                      (5000, 40, 240), (3001, 96, 300)])
def test_xty_tensor_core_matches_fp64(rows, M, N):
    """dW = X^T Y on tcgen05 with MN-major operands straight from row-major HBM tensors; the last two shapes (M % 16 != 0,
    N > 256) run on the FFMA kernel."""
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    from tensoflow_b200 import _lib
    from tensoflow_b200._lib import check, ptr, stream_ptr
    dev = torch.device("cuda:0")
    g = torch.Generator().manual_seed(rows + M + N)
    X = torch.randn(rows, M, generator=g).to(dev)
    Y = torch.randn(rows, N, generator=g).to(dev)
    ref = X.double().T @ Y.double()
    out = torch.ones(M, N, device=dev)
    check(_lib.load().tf_xty_accumulate(ptr(X), ptr(Y), rows, M, N, ptr(out), stream_ptr()), "tf_xty_accumulate")
    torch.cuda.synchronize()
    e = float((out.double() - 1 - ref).abs().max() / ref.abs().max())
    print(f"rows={rows} M={M} N={N}: {e:.2e}")
    assert e < 5e-6, e


@pytest.mark.parametrize("M,K,N,act", [(20000, 123, 256, "relu"), (9000, 256, 99, "exp"), (10000, 108, 128, "sigmoid"),
                                       (8200, 256, 256, "relu"), (8192, 97, 101, "none"), (9000, 256, 3, "exp"),
                                       (10000, 44, 64, "leaky"), (5000, 64, 21, "none"), (4099, 57, 64, "leaky"), (9000, 16, 3, "sigmoid")])
def test_linear_tensor_core_fwd_bwd(M, K, N, act):
    """ops.linear on the tcgen05 path (M >= 8192, wide layers) and on the fused narrow-layer backward (K, N <= 64):
    padded N, unaligned K, activation epilogue, data and weight gradients."""
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    from tensoflow_b200 import ops
    dev = torch.device("cuda:0")
    g = torch.Generator().manual_seed(M + K + N)
    X = torch.randn(M, K, generator=g)
    W = torch.randn(N, K, generator=g) / K ** 0.5
    b = 0.1 * torch.randn(N, generator=g)
    gY = torch.randn(M, N, generator=g)

    def run(dt, device, fn):
        x, w, bb = (t.detach().clone().to(device=device, dtype=dt).requires_grad_() for t in (X, W, b))
        y = fn(x, w, bb)
        y.backward(gY.to(device=device, dtype=dt))
        return [t.detach().cpu().double() for t in (y, x.grad, w.grad, bb.grad)]

    def torch_fn(x, w, bb):
        z = x @ w.T + bb
        return {"relu": torch.relu, "sigmoid": torch.sigmoid, "none": lambda t: t, "exp": lambda t: torch.exp(t.clamp(max=5.0)),
                "leaky": lambda t: torch.nn.functional.leaky_relu(t, 0.01)}[act](z)

    ref = run(torch.float64, "cpu", torch_fn)
    f32 = run(torch.float32, "cpu", torch_fn)
    ours = run(torch.float32, dev, lambda x, w, bb: ops.linear(x, w, bb, act, 5.0))
    for name, o, r, f in zip(("y", "dX", "dW", "db"), ours, ref, f32):
        e = float((o - r).abs().max() / r.abs().max())
        e32 = float((f - r).abs().max() / r.abs().max())
        print(f"{name}: ours {e:.2e} torch-fp32 {e32:.2e}")
        # 3xTF32 keeps ~22 mantissa bits per product; exp() turns the absolute error of its argument into a relative one
        assert e <= max(2e-5 if act == "exp" else 3e-6, 4 * e32), (name, e, e32)
