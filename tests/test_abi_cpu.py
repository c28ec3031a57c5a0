"""CPU checks of the C-ABI boundary: the library builds, loads without a GPU, and exports
every symbol include/tensoflow_b200.h declares.  No compute calls."""
import ctypes
import re
from pathlib import Path

import pytest

ROOT = Path(__file__).resolve().parents[1]


@pytest.fixture(scope="module")
def lib():
    from tensoflow_b200 import build, _lib
    build.build()
    return _lib.load()


def test_header_symbols_exported(lib):
    from tensoflow_b200 import _lib
    header = (ROOT / "include" / "tensoflow_b200.h").read_text()
    declared = set(re.findall(r"TF_API\s+[\w\s\*]+?\b(tf_[a-z0-9_]+)\s*\(", header))
    assert declared, "no declarations parsed"
    raw = ctypes.CDLL(str(_lib.lib_path()))
    for name in sorted(declared):
        assert hasattr(raw, name), f"{name} declared in the header but not exported"
    assert declared == set(_lib.exported_symbols()), declared ^ set(_lib.exported_symbols())


def test_abi_version_3_and_error_string(lib):
    """ABI 3: tf_linear_workspace takes the row count, and the tcgen05 dense layer refuses to run without its workspace."""
    assert lib.tf_abi_version() == 3
    assert isinstance(lib.tf_last_error(), bytes)


def _linear_tc_bytes(K, N):
    """Pre-split weights of the tcgen05 dense layer contracting K into N outputs: hi | lo, N padded to 16, K to 32."""
    return 4 * 2 * (-(-N // 16) * 16) * (-(-K // 32) * 32)


@pytest.mark.parametrize("M,K,N,fwd,bwd", [
    (8191, 128, 128, False, False), (8192, 128, 128, True, True),       # rows
    (8192, 95, 128, False, False), (8192, 96, 128, True, True),         # K >= 96
    (8192, 1024, 128, True, False), (8192, 1025, 128, False, False),    # forward K <= 1024 (backward K <= 256)
    (8192, 128, 95, False, False), (8192, 128, 96, True, True),         # N >= 96
    (8192, 512, 256, True, False), (8192, 512, 257, False, False),      # forward N <= 256 (backward K <= 256)
    (8192, 128, 512, False, True),                                      # only the data gradient (N into K) runs on tcgen05
    (1 << 20, 64, 64, False, False),                                    # narrow layer: FFMA at any row count
])
def test_linear_workspace_follows_the_dispatch(lib, M, K, N, fwd, bwd):
    """tf_linear_workspace(M, K, N) is what the tcgen05 forward (K into N) or data gradient (N into K) needs, 0 when neither runs."""
    want = max(_linear_tc_bytes(K, N) if fwd else 0, _linear_tc_bytes(N, K) if bwd else 0)
    assert lib.tf_linear_workspace(M, K, N) == want


@pytest.mark.parametrize("bad", ["null", "small", "unaligned"])
def test_linear_tc_requires_workspace(lib, bad):
    """On a tcgen05 shape tf_linear_fwd / tf_linear_bwd return an error before any launch when the workspace is NULL, too
    small or not 16-byte aligned, instead of falling back to the FFMA kernels.  The addresses are fake: the check fires before
    anything is dereferenced."""
    M, K, N = 8192, 128, 128
    fake = lambda i: ctypes.c_void_p((1 << 20) * (i + 1))
    need = lib.tf_linear_workspace(M, K, N)
    ws, wsb = {"null": (None, need), "small": (fake(9), need - 4), "unaligned": (ctypes.c_void_p((1 << 20) * 10 + 4), need)}[bad]
    launches = lib.tf_launch_count()
    rc = lib.tf_linear_fwd(fake(0), fake(1), None, M, K, N, 0, 0.0, fake(2), ws, wsb, None)
    assert rc != 0
    assert b"workspace" in lib.tf_last_error()
    rc = lib.tf_linear_bwd(fake(0), fake(1), fake(2), fake(3), fake(4), M, K, N, 0, 0.0, fake(5), fake(6), fake(7), ws, wsb, None)
    assert rc != 0
    assert b"workspace" in lib.tf_last_error()
    assert lib.tf_launch_count() == launches


def test_flow_block_bwd_requires_kept_activations(lib):
    """tf_flow_block_bwd without the activations kept by the forward (saved_h / saved_st) returns an error before any launch.
    The addresses are fake: the check fires before anything is dereferenced."""
    fake, M, sn, F = ctypes.c_void_p(1 << 20), 64, 16, 8
    launches = lib.tf_launch_count()
    rc = lib.tf_flow_block_bwd(*(fake,) * 2, F, sn, *(fake,) * 8, 2.0, -1.0, 0, M, None, None, None, None, *(fake,) * 10, None)
    assert rc != 0
    assert b"saved_h" in lib.tf_last_error()
    assert lib.tf_launch_count() == launches


def test_no_cpu_fallback():
    """Product ops refuse CPU tensors instead of silently computing elsewhere."""
    import torch
    from tensoflow_b200 import _lib
    with pytest.raises(RuntimeError):
        _lib.ptr(torch.zeros(4))


def test_product_does_not_import_oracle():
    for p in (ROOT / "tensoflow_b200").glob("*.py"):
        src = p.read_text()
        assert "import oracle" not in src and "from oracle" not in src, p


def test_new_entry_points_refuse_cpu_tensors():
    """FusedAdam, the occupancy marcher and the cube lookup have no CPU path either: CPU tensors raise before any launch."""
    import torch
    from tensoflow_b200.optim import FusedAdam
    from tensoflow_b200.occ_grid import OccGridEstimator
    from tensoflow_b200.shape_shader import cube_lookup
    p = torch.nn.Parameter(torch.zeros(4))
    p.grad = torch.ones(4)
    with pytest.raises(RuntimeError):
        FusedAdam([p]).step()
    est = OccGridEstimator([-1, -1, -1, 1, 1, 1], resolution=4)
    est.mark_all_occupied()
    with pytest.raises(RuntimeError):
        est.sampling(torch.zeros(2, 3), torch.ones(2, 3), near_plane=0.1, far_plane=2.0, render_step_size=0.1)
    with pytest.raises(RuntimeError):
        cube_lookup([torch.zeros(6, 4, 4, 3)], torch.ones(5, 3))


def test_occ_grid_refresh_host_logic():
    """OccGridEstimator._update / update_every_n_steps / state_dict are tensor logic: check them on CPU (nerfacc semantics:
    occs = max(occs * decay, occ), binaries = occs > min(mean, thre); refresh only when step % n == 0 in training mode)."""
    import torch
    from tensoflow_b200.occ_grid import OccGridEstimator
    est = OccGridEstimator([-1, -1, -1, 1, 1, 1], resolution=8)
    ball = lambda x: (x.norm(dim=-1) < 0.6).float()
    est._update(0, ball, warmup_steps=10, jitter=torch.full((512, 3), 0.5))
    centres = (est.grid_coords.float() + 0.5) / 8 * 2 - 1
    assert torch.equal(est.binaries.reshape(-1), centres.norm(dim=-1) < 0.6)
    before = est.occs.clone()
    est._update(0, lambda x: torch.zeros(x.shape[0]), ema_decay=0.5, warmup_steps=10)
    assert torch.allclose(est.occs, before * 0.5)                    # decay only
    est.eval()
    est.update_every_n_steps(100, ball, n=100, warmup_steps=0)        # not training: untouched
    assert torch.allclose(est.occs, before * 0.5)
    est.train()
    est.update_every_n_steps(101, ball, n=100, warmup_steps=0)        # not a multiple of n: untouched
    assert torch.allclose(est.occs, before * 0.5)
    est.update_every_n_steps(200, ball, n=100, warmup_steps=0)        # partial refresh (a quarter + the occupied cells)
    assert float(est.occs.max()) == 1.0
    sd = est.state_dict()
    assert set(sd) == {"resolution", "aabbs", "occs", "binaries"}
    est2 = OccGridEstimator([-1, -1, -1, 1, 1, 1], resolution=8)
    est2.load_state_dict(sd)
    assert torch.equal(est2.binaries, est.binaries) and torch.equal(est2.occs, est.occs)
