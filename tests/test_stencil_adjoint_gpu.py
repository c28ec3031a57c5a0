"""The fused SDF stencil (tf_sdf_stencil_fwd / tf_sdf_stencil_bwd), the SDF-only and single-query forwards and the VM feature
op on anisotropic fields, against an fp64 reference conditioned on the kernel's own finite-difference taps.

The hessian term divides sums of tap SDFs by units^2, so rounding the seven tap values to fp32 moves its adjoint far more than
any kernel arithmetic does; a bar that floats with the fp32 oracle's error hides kernel errors of that size.  Two choices
remove the input rounding, so that what is left is the kernel's own arithmetic:
  * exact taps: dyadic units, distinct per axis, an aabb with power-of-two extents, positions on a 2^-12 lattice (2^-13 on the
    half-extent axis) and levels on a 2^-8 lattice.  Then x +- e, the normalised coordinate and u N - 0.5 are exact in fp32 for
    every plane, line and mip size, and the kernel picks the same texels with the same 1-D weights as the fp64 oracle
    (test_taps_exact_in_fp32 asserts it).
  * conditioned adjoint: a[n, k] = d/d s7[n, k] (u_sdf s0 + u_grad . g(s7) + u_hess nh(s7)) is formed in fp64 from the
    kernel's sdf7 output, with s+ + s- taking its fp32 value as in the kernel: that is the one step whose rounding is amplified,
    by |s| / (e^2 |h|).
The reference gradient is ref = grad_theta [sum_{n,k} a[n,k] S64[n,k] + sum u_feat . feat64], with S64[:, k] the fp64 oracle's
SDF at tap k, and M = sum_k |grad_theta sum_n a[n,k] S64[n,k]| + |grad_theta sum u_feat . feat64| is the size of the terms the
kernel adds up.  Gradient errors are max|got - ref| / max M, which stays meaningful where ref cancels to about 0 (d b1[0] under a
hessian-only upstream is analytically 0).  A correct fp32 kernel sits near 1e-7 on that scale; the bar is 1e-5.

Fields are anisotropic (distinct grid, units and aabb extent per axis, non-square planes), so an axis mix-up in units, plane
extents, plane axes or the aabb changes the result.  The fp64 reference runs on the device.
"""
import ctypes as C

import pytest
import torch

from conftest import record_err

from oracle import torch_oracle as O  # noqa: E402

AABB = [[-1.0, -0.5, -1.0], [1.0, 0.5, 1.0]]          # extents 2, 1, 2: powers of two
UNITS = (2.0 ** -5, 2.0 ** -6, 3 * 2.0 ** -8)          # dyadic finite-difference steps, distinct per axis
BWD_BAR = 1e-5                                          # max|got - ref| / max M of every parameter gradient
FWD_BAR = 1e-5                                          # sdf: max|got - ref| / max|ref|; features: / max of their term sizes
GRAD_BAR, HESS_BAR = 1e-6, 1e-5                         # grad / hess against the FD formula on the kernel's own sdf7
VM_BAR = 1e-6                                           # VM feature op: no decoder, exact taps
ZERO_VS_NULL_BAR = 5e-6     # NULL upstreams against zero tensors: atomic-order noise only (a line texel sums thousands of
                            # terms; measured up to 1.3e-6 of max M on a B200)

# name: (C, H, A, G0, grid, levels)
SHAPES = {
    "aniso": (8, 32, 16, (20, 12, 24), (40, 24, 48), 2),
    "bench": (36, 256, 128, (128, 96, 64), (512, 384, 256), 3),       # bench.py decoder dims on a non-cubic grid
    "ffma": (8, 288, 16, (20, 12, 24), (40, 24, 48), 2),              # hidden > 256: the FFMA stencil kernels
}
UPSTREAMS = ("sdf", "feat", "grad", "hess", "all")


def _cuda():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    return torch.device("cuda:0")


def tap_offsets(units, dtype=torch.float64, device="cpu"):
    """[7, 3]: centre, +-x, +-y, +-z (the kernel's query order, reference network/fields.py:239-244)."""
    offs = torch.zeros(7, 3, dtype=dtype, device=device)
    for k in range(3):
        offs[1 + 2 * k, k] = units[k]
        offs[2 + 2 * k, k] = -units[k]
    return offs


# ---- sample sets (fp64 on the host, exact in fp32) ----------------------------------------------------------------------
def lattice_points(n, seed, n_levels):
    """Positions on the 2^-12 lattice scaled by the half extents (up to ~5 % beyond every face: clamp addressing), levels on
    the 2^-8 lattice from -0.25 to L - 0.75."""
    g = torch.Generator().manual_seed(seed)
    half = torch.tensor([(b - a) / 2 for a, b in zip(*AABB)], dtype=torch.float64)
    x = torch.randint(-4300, 4301, (n, 3), generator=g).double() * 2.0 ** -12 * half
    lv = torch.randint(-64, 256 * (n_levels - 1) + 64, (n,), generator=g).double() * 2.0 ** -8
    return x, lv


def edge_points(grid, n_levels, seed=5):
    """Every combination of special per-axis coordinates: texel centres and texel edges at level 0 (the dyadic ones), the
    aabb faces, and 1-3 texels outside the box; levels cycle through 0, L-1, values below 0 and above L-1, and lattice values."""
    vals = []
    for ax in range(3):
        N, lo, ext = grid[ax], AABB[0][ax], AABB[1][ax] - AABB[0][ax]
        a = (N & -N).bit_length() - 1                        # N = 2^a * odd: u = j / 2^a is a texel edge, (2j+1) / 2^(a+1) a centre
        p = (N - 1).bit_length()                             # 2^p >= N: k / 2^p is k * N / 2^p texels
        us = [(2 * j + 1) / 2 ** (a + 1) for j in (0, 1, 2 ** a - 1)] + [j / 2 ** a for j in (1, 2 ** (a - 1))]
        us += [0.0, 1.0] + [-k / 2 ** p for k in (2, 3, 4)] + [1 + k / 2 ** p for k in (2, 3, 4)]
        vals.append(torch.tensor([lo + u * ext for u in us], dtype=torch.float64))
    x = torch.cartesian_prod(*vals)
    L1 = n_levels - 1
    special = torch.tensor([0.0, L1, -0.5, -3.0, L1 + 0.25, L1 + 2.0, 0.5, L1 - 2.0 ** -8], dtype=torch.float64)
    g = torch.Generator().manual_seed(seed)
    rnd = torch.randint(0, 256 * L1 + 1, (x.shape[0],), generator=g).double() * 2.0 ** -8
    idx = torch.arange(x.shape[0])
    lv = torch.where(idx % 2 == 0, special[(idx // 2) % special.numel()], rnd)
    return x, lv


def tap_exactness(x, lv, grid, n_levels, units):
    """Names of the fp32 steps of the kernel's sampling plan that are not exact for these samples (empty = all exact):
    tap positions, normalised coordinates, u N - 0.5 for every texture extent and mip size, and the levels."""
    bad = []
    exact = lambda t: bool((t.float().double() == t).all())   # noqa: E731
    lo = torch.tensor(AABB[0], dtype=torch.float64)
    ext = torch.tensor(AABB[1], dtype=torch.float64) - lo
    for q, e in enumerate(tap_offsets(units)):
        p = x + e
        if not exact(p):
            bad.append(f"position of tap {q}")
        u = (p - lo) / ext
        if not exact(u):
            bad.append(f"coordinate of tap {q}")
        for ax in range(3):
            for l in range(n_levels):
                if not exact(u[:, ax] * (grid[ax] >> l) - 0.5):
                    bad.append(f"texel coordinate of tap {q}, axis {ax}, level {l}")
    if lv is not None and not exact(lv):
        bad.append("levels")
    return bad


# ---- fields --------------------------------------------------------------------------------------------------------------
class Field:
    """The fp64 oracle (on the device) and the fp32 CUDA-side tensors of one anisotropic TensoSDF with identical values."""

    def __init__(self, shape, dev):
        from tensoflow_b200 import synthetic
        from tensoflow_b200.fields import _cl
        C_, H, A, G0, grid, L = SHAPES[shape]
        torch.manual_seed(0)
        o = O.TensoSDF(list(G0), AABB, sdf_n_comp=C_, sdf_dim=H, app_dim=A, init_n_levels=L - 1, dtype=torch.float64)
        o.upsample_volume_grid(torch.tensor(grid))
        assert [int(v) for v in o.gridSize] == list(grid) and o.n_levels == L
        synthetic.perturb_field(o, seed=1, noise=0.05)
        g = torch.Generator().manual_seed(2)
        with torch.no_grad():   # hidden pre-activations off the softplus linear branch, appearance rows distinct
            o.sdf_mat[0].weight.mul_(0.05)
            o.sdf_mat[0].bias.add_(0.01 * torch.randn(o.sdf_mat[0].bias.shape, generator=g, dtype=torch.float64))
            o.sdf_mat[2].weight[1:].add_(0.1 * torch.randn(o.sdf_mat[2].weight[1:].shape, generator=g, dtype=torch.float64))
            for p in o.parameters():                 # fp32 values: the kernel reads exactly the oracle's parameters
                p.copy_(p.float().double())
        self.o64 = o.to(dev)
        self.o64.update_gridSize(self.o64.gridSize, L)
        for i in range(3):                           # non-square planes: [grid[m1], grid[m0]]
            m0, m1 = O.MAT_MODE[i]
            assert tuple(o.sdf_plane[i].shape[2:]) == (grid[m1], grid[m0])
        self.planes = [_cl(p.detach().float()) for p in self.o64.sdf_plane]
        self.lines = [_cl(p.detach().float()) for p in self.o64.sdf_line]
        self.mlp = [p.detach().float().contiguous() for p in self.o64.sdf_mat.parameters()]   # W0, b0, W1, b1
        self.aabb = torch.tensor(AABB, device=dev)
        self.grid, self.L, self.A, self.H = grid, L, A, H
        self.dev = dev


_FIELDS = {}


def field(shape):
    dev = _cuda()
    if shape not in _FIELDS:
        _FIELDS[shape] = Field(shape, dev)
    return _FIELDS[shape]


# ---- the kernels through the C ABI -----------------------------------------------------------------------------------------
def kernel_fwd(F, x, lv):
    """tf_sdf_stencil_fwd -> sdf7, feat, grad, hess, and the forward workspace + hidden offset (the backward reads the centre
    hidden activations there)."""
    from tensoflow_b200 import _lib, ops
    from tensoflow_b200._lib import check, ptr, stream_ptr
    lib = _lib.load()
    vm = ops.vm_desc(F.planes, F.lines, F.aabb, F.L, lv is not None)
    m, _keep = ops._mlp_desc(*F.mlp)
    n = x.shape[0]
    sdf7 = torch.empty(n, 7, device=F.dev)
    feat = torch.empty(n, F.A, device=F.dev)
    grad = torch.empty(n, 3, device=F.dev)
    hess = torch.empty(n, device=F.dev)
    wsb = lib.tf_sdf_stencil_fwd_workspace(C.byref(vm.c), C.byref(m), n, 1)
    ws = torch.empty(wsb // 4, device=F.dev)
    check(lib.tf_sdf_stencil_fwd(C.byref(vm.c), C.byref(m), ptr(x), ptr(lv), n, ops._units_arr(UNITS), ptr(sdf7), ptr(feat),
                                 ptr(grad), ptr(hess), ptr(ws), wsb, stream_ptr()), "tf_sdf_stencil_fwd")
    off = lib.tf_sdf_stencil_fwd_hidden_offset(C.byref(vm.c), C.byref(m))
    hidden = None if off == C.c_size_t(-1).value else ws.data_ptr() + off
    return sdf7, feat, grad, hess, (ws, hidden)


def kernel_bwd(F, x, lv, sdf7, hidden, ups, n_slice=None):
    """tf_sdf_stencil_bwd with the upstreams ups = (g_sdf, g_feat, g_grad, g_hess) (None = NULL); mip gradients folded by
    tf_vm_fold_mip_grads.  n_slice: size the workspace for that many samples (the call then runs in slices).
    -> ({parameter name: gradient}, number of workspace slices of the tensor-core path)."""
    from tensoflow_b200 import _lib, ops
    from tensoflow_b200._lib import SdfMlpGrad, check, ptr, stream_ptr
    lib = _lib.load()
    with_mips = lv is not None
    vm = ops.vm_desc(F.planes, F.lines, F.aabb, F.L, with_mips)
    m, _keep = ops._mlp_desc(*F.mlp)
    g, gp, gl, _gpm, _glm = vm.new_grads(with_mips)
    dmlp = [torch.zeros_like(w) for w in F.mlp]
    mg = SdfMlpGrad()
    mg.W0, mg.b0, mg.W1, mg.b1 = (t.data_ptr() for t in dmlp)
    n = x.shape[0]
    ws_of = lambda k: lib.tf_sdf_stencil_bwd_workspace(C.byref(vm.c), C.byref(m), k)   # noqa: E731
    wsb = ws_of(n if n_slice is None else n_slice)
    ws = torch.empty(wsb // 4, device=F.dev)
    gs, gf, gg, gh = ups
    check(lib.tf_sdf_stencil_bwd(C.byref(vm.c), C.byref(m), ptr(x), ptr(lv), n, ops._units_arr(UNITS), ptr(sdf7), hidden,
                                 ptr(gs), ptr(gf), ptr(gg), ptr(gh), C.byref(g), C.byref(mg), ptr(ws), wsb, stream_ptr()),
          "tf_sdf_stencil_bwd")
    d_planes, d_lines = vm.finish_grads(g, gp, gl, with_mips)
    out = {f"sdf_plane.{i}": d_planes[i] for i in range(3)}
    out.update({f"sdf_line.{i}": d_lines[i] for i in range(3)})
    out.update(dict(zip(("sdf_mat.0.weight", "sdf_mat.0.bias", "sdf_mat.2.weight", "sdf_mat.2.bias"), dmlp)))
    per_tile = ws_of(36) - ws_of(18)            # tensor-core path: 18 samples per tile
    tiles_fit = (wsb - (ws_of(18) - per_tile)) // per_tile
    return out, -(-(-(-n // 18)) // tiles_fit)


# ---- the conditioned fp64 reference --------------------------------------------------------------------------------------
def fd_terms(s7, units, fp32_sum):
    """(g [n,3], nh [n]) of the finite-difference formula (reference network/fields.py:245-256) in fp64 at s7, differentiable
    in s7.  fp32_sum: s+ + s- takes its fp32 value (what the kernel forms) and keeps the derivative of the exact sum."""
    gs, hs = [], []
    for k in range(3):
        sp, sm = s7[:, 1 + 2 * k], s7[:, 2 + 2 * k]
        ssum = sp + sm
        if fp32_sum:
            ssum = ssum + ((sp.float() + sm.float()).double() - ssum).detach()
        gs.append((sp - sm) / (2 * units[k]))
        hs.append((ssum - 2 * s7[:, 0]) / units[k] ** 2)
    g, h = torch.stack(gs, 1), torch.stack(hs, 1)
    return g, (g * h).sum(1) / ((g * g).sum(1) + 1e-5)


def adjoint(s7, units, u_sdf, u_grad, u_hess, fp32_sum=True):
    """a[n, 7] = d/d s7 (u_sdf s0 + u_grad . g(s7) + u_hess nh(s7)) in fp64 (None upstreams are zero)."""
    s = s7.detach().double().requires_grad_()
    g, nh = fd_terms(s, units, fp32_sum)
    loss = s.new_zeros(())
    if u_sdf is not None:
        loss = loss + (s[:, 0] * u_sdf.double()).sum()
    if u_grad is not None:
        loss = loss + (g * u_grad.double()).sum()
    if u_hess is not None:
        loss = loss + (nh * u_hess.double()).sum()
    if not loss.requires_grad:
        return torch.zeros_like(s)
    return torch.autograd.grad(loss, s)[0]


def reference_grads(o, x, lv, units, a, u_feat):
    """ref and M (see the module docstring) for every parameter of the oracle o, at samples x [n,3] / lv [n] or None."""
    names = [n for n, _ in o.named_parameters()]
    params = [p for _, p in o.named_parameters()]
    ref = {n: torch.zeros_like(p) for n, p in zip(names, params)}
    M = {n: torch.zeros_like(p) for n, p in zip(names, params)}
    offs = tap_offsets(units, x.dtype, x.device)
    lvl = None if lv is None else lv[:, None]
    terms = [(o.sdf(x + offs[k], lvl)[:, 0] * a[:, k]).sum() for k in range(7) if bool((a[:, k] != 0).any())]
    if u_feat is not None:
        terms.append((o(x, lvl)[:, 1:] * u_feat.double()).sum())
    for t in terms:
        for n, gv in zip(names, torch.autograd.grad(t, params, allow_unused=True)):
            if gv is not None:
                ref[n] += gv
                M[n] += gv.abs()
    return ref, M


def oracle_taps(o, x, lv):
    """S64 [n, 7] and feat64 [n, A] of the fp64 oracle at the kernel's taps."""
    offs = tap_offsets(UNITS, x.dtype, x.device)
    lvl = None if lv is None else lv[:, None]
    with torch.no_grad():
        S = torch.stack([o.sdf(x + offs[k], lvl)[:, 0] for k in range(7)], 1)
        feat = o(x, lvl)[:, 1:]
    return S, feat


def upstreams(n, A, which, seed, dev):
    g = torch.Generator().manual_seed(seed)
    full = (torch.randn(n, generator=g), torch.randn(n, A, generator=g), torch.randn(n, 3, generator=g), torch.randn(n, generator=g))
    keep = {"sdf": (0,), "feat": (1,), "grad": (2,), "hess": (3,), "all": (0, 1, 2, 3)}[which]
    return tuple(t.to(dev) if i in keep else None for i, t in enumerate(full))


def check_grads(got, ref, M, label, bar=BWD_BAR):
    """max|got - ref| / max M <= bar for every parameter; recorded with M."""
    for name in ref:
        m = float(M[name].max())
        d = float((got[name].double() - ref[name]).abs().max())
        if m == 0.0:
            assert d == 0.0, f"{label} d {name}: {d:.3e} where every term is 0"
            continue
        e = d / m
        record_err(f"{label} d {name} (err / max M)", got[name], ref[name], bar, max_M=m, err_M=e)
        assert e <= bar, f"{label} d {name}: max|got - ref| / max M = {e:.3e} > {bar:.0e}"


def check_values(got, ref, what, bar):
    e = record_err(what, got, ref, bar)
    assert e <= bar, f"{what}: rel err {e:.3e} > {bar:.0e}"


def feat_term_size(o, x, lvl):
    """[n, A]: sum_h |hidden_h W1[1 + o, h]| + |b1[1 + o]|, the size of the terms the appearance head adds up.  The features
    are sums of H terms of both signs that cancel to a fraction of that size, so their rounding floor is stated against it."""
    with torch.no_grad():
        f = O.vm_feature(o.sdf_plane, o.sdf_line, x, lvl, o.aabb, o.n_levels)
        hid = o.sdf_mat[1](o.sdf_mat[0](torch.cat([f, x], -1)))
        return hid.abs() @ o.sdf_mat[2].weight[1:].abs().T + o.sdf_mat[2].bias[1:].abs()


def check_feat(got, ref, scale, what):
    m = float(scale.max())
    e = float((got.double() - ref).abs().max()) / m
    record_err(what + " (err / max term size)", got, ref, FWD_BAR, max_M=m, err_M=e)
    assert e <= FWD_BAR, f"{what}: max|got - ref| / max term size = {e:.3e} > {FWD_BAR:.0e}"


def to_dev(F, x, lv):
    return x.float().to(F.dev), None if lv is None else lv.float().to(F.dev)


def forward_checks(F, x, lv, label):
    """sdf7 (all 7 taps), feat, grad and hess of the stencil forward; the SDF-only and single-query forwards."""
    from tensoflow_b200 import ops
    xd, ld = to_dev(F, x, lv)
    x64, l64 = xd.double(), None if ld is None else ld.double()
    sdf7, feat, grad, hess, keep = kernel_fwd(F, xd, ld)
    S64, f64 = oracle_taps(F.o64, x64, l64)
    for k in range(7):
        check_values(sdf7[:, k], S64[:, k], f"{label} sdf7[:, {k}]", FWD_BAR)
    fscale = feat_term_size(F.o64, x64, None if l64 is None else l64[:, None])
    check_feat(feat, f64, fscale, f"{label} feat")
    g_ref, nh_ref = fd_terms(sdf7.double(), UNITS, fp32_sum=True)
    check_values(grad, g_ref, f"{label} grad (FD formula on the kernel's sdf7)", GRAD_BAR)
    check_values(hess, nh_ref, f"{label} hess (FD formula on the kernel's sdf7)", HESS_BAR)
    planes, lines = F.planes, F.lines
    only = ops.sdf_only(xd, ld, F.aabb, F.L, *F.mlp, planes, lines)
    check_values(only, S64[:, 0], f"{label} tf_sdf_only_fwd", FWD_BAR)
    point = ops.sdf_point(xd, ld, F.aabb, F.L, *F.mlp, planes, lines)
    if F.H <= 256:
        assert point is not None
        check_values(point[0], S64[:, 0], f"{label} tf_sdf_point_fwd sdf", FWD_BAR)
        check_feat(point[1], f64, fscale, f"{label} tf_sdf_point_fwd feat")
    else:
        assert point is None          # outside the tensor-core path: the caller falls back to the stencil
    return xd, ld, sdf7, keep


def backward_checks(F, xd, ld, sdf7, keep, which, label, seed, n_slice=None, min_slices=1):
    """One upstream path (or all four): NULL for the others, then zero tensors for the others; both against the reference."""
    n = xd.shape[0]
    ups = upstreams(n, F.A, which, seed, F.dev)
    hidden = keep[1] if ups[1] is not None else None           # hidden_centre = NULL whenever g_feat is NULL
    got, slices = kernel_bwd(F, xd, ld, sdf7, hidden, ups, n_slice)
    assert slices >= min_slices, slices
    a = adjoint(sdf7, UNITS, ups[0], ups[2], ups[3])
    ref, M = reference_grads(F.o64, xd.double(), None if ld is None else ld.double(), UNITS, a, ups[1])
    check_grads(got, ref, M, f"{label} [{which}, others NULL]")
    if which != "all":
        shapes = ((n,), (n, F.A), (n, 3), (n,))
        zeros = tuple(torch.zeros(shp, device=F.dev) if u is None else u for shp, u in zip(shapes, ups))
        got_z, _ = kernel_bwd(F, xd, ld, sdf7, keep[1], zeros, n_slice)
        check_grads(got_z, ref, M, f"{label} [{which}, others zero]")
        check_grads(got_z, got, M, f"{label} [{which}, zeros vs NULL]", ZERO_VS_NULL_BAR)


# ---- GPU tests --------------------------------------------------------------------------------------------------------------
# (shape, N, with_level, workspace slice): the bench-dims case runs its backward in >= 2 workspace slices
CASES = {
    "aniso": ("aniso", 3001, True, None),
    "aniso-level-NULL": ("aniso", 3001, False, None),
    "ffma": ("ffma", 1003, True, None),
    "bench": ("bench", 4099, True, 1500),
}


@pytest.mark.gpu
@pytest.mark.parametrize("case", list(CASES))
def test_stencil_forward_exact_taps(case):
    shape, n, with_level, _ = CASES[case]
    F = field(shape)
    x, lv = lattice_points(n, 3, F.L)
    forward_checks(F, x, lv if with_level else None, case)


@pytest.mark.gpu
@pytest.mark.parametrize("which", UPSTREAMS)
@pytest.mark.parametrize("case", list(CASES))
def test_stencil_backward_per_upstream(case, which):
    shape, n, with_level, n_slice = CASES[case]
    F = field(shape)
    x, lv = lattice_points(n, 3, F.L)
    xd, ld = to_dev(F, x, lv if with_level else None)
    sdf7, _feat, _grad, _hess, keep = kernel_fwd(F, xd, ld)
    backward_checks(F, xd, ld, sdf7, keep, which, case, seed=11 + UPSTREAMS.index(which), n_slice=n_slice,
                    min_slices=2 if n_slice else 1)


@pytest.mark.gpu
@pytest.mark.parametrize("n", [1, 17, 18, 19])
def test_stencil_around_one_tile(n):
    """Fewer samples than the 18-sample tile of the tensor-core kernels, exactly one tile, one sample into the second."""
    F = field("aniso")
    x, lv = lattice_points(n, 29, F.L)
    xd, ld, sdf7, keep = forward_checks(F, x, lv, f"N={n}")
    backward_checks(F, xd, ld, sdf7, keep, "all", f"N={n}", seed=31)
    backward_checks(F, xd, ld, sdf7, keep, "hess", f"N={n}", seed=37)


@pytest.mark.gpu
@pytest.mark.parametrize("shape", ["aniso", "ffma"])
def test_stencil_edge_band(shape):
    """Samples on texel centres, on texel edges, on the aabb faces and 1-3 texels outside the box (clamp addressing), at levels
    0 and L-1, below 0 and above L-1."""
    F = field(shape)
    x, lv = edge_points(F.grid, F.L)
    xd, ld, sdf7, keep = forward_checks(F, x, lv, f"edge band {shape}")
    for which in ("all", "hess"):
        backward_checks(F, xd, ld, sdf7, keep, which, f"edge band {shape}", seed=41)


@pytest.mark.gpu
@pytest.mark.parametrize("with_level", [True, False])
@pytest.mark.parametrize("shape", ["aniso", "bench"])
def test_vm_feature_exact_taps(shape, with_level):
    """tf_vm_feature_fwd / _bwd (VMFeatureFunction) on non-square planes, with tf_vm_build_mips / tf_vm_fold_mip_grads when
    levels are given.  Gradients: max|got - ref| / max M with M the gradient of sum |u| . feat(|planes|, |lines|), the sum of
    the magnitudes of the scattered terms."""
    from tensoflow_b200 import ops
    F = field(shape)
    o = F.o64
    x, lv = lattice_points(2053, 43, F.L)
    if not with_level:
        lv = None
    xd, ld = to_dev(F, x, lv)
    x64, l64 = xd.double(), None if ld is None else ld.double()
    planes = [p.detach().requires_grad_() for p in F.planes]
    lines = [p.detach().requires_grad_() for p in F.lines]
    got = ops.VMFeatureFunction.apply(xd, ld, F.aabb, F.L, *planes, *lines)
    ref = O.vm_feature(o.sdf_plane, o.sdf_line, x64, l64, o.aabb, F.L)
    check_values(got, ref, f"vm feature {shape}", VM_BAR)
    u = torch.randn(got.shape, generator=torch.Generator().manual_seed(47)).to(F.dev)
    (got * u).sum().backward()
    fac = list(o.sdf_plane) + list(o.sdf_line)
    gref = torch.autograd.grad((ref * u.double()).sum(), fac)
    absf = [p.detach().abs().requires_grad_() for p in fac]
    gM = torch.autograd.grad((O.vm_feature(absf[:3], absf[3:], x64, l64, o.aabb, F.L) * u.double().abs()).sum(), absf)
    names = [f"sdf_plane.{i}" for i in range(3)] + [f"sdf_line.{i}" for i in range(3)]
    check_grads({nm: p.grad for nm, p in zip(names, planes + lines)}, dict(zip(names, gref)), dict(zip(names, gM)),
                f"vm feature {shape} level={with_level}", VM_BAR)


# ---- CPU checks of the reference ---------------------------------------------------------------------------------------------
def test_taps_exact_in_fp32():
    """Every sample set of the GPU tests has exact taps for every texture and mip size; the oracle's own units (aabb extent /
    (grid - 1)) would not."""
    for shape, n, _, _ in CASES.values():
        grid, L = SHAPES[shape][4], SHAPES[shape][5]
        x, lv = lattice_points(n, 3, L)
        assert tap_exactness(x, lv, grid, L, UNITS) == [], shape
    for shape in ("aniso", "bench"):
        grid, L = SHAPES[shape][4], SHAPES[shape][5]
        assert tap_exactness(*lattice_points(2053, 43, L), grid, L, UNITS) == []
    grid, L = SHAPES["aniso"][4], SHAPES["aniso"][5]
    for n in (1, 17, 18, 19):
        assert tap_exactness(*lattice_points(n, 29, L), grid, L, UNITS) == []
    x, lv = edge_points(grid, L)
    assert tap_exactness(x, lv, grid, L, UNITS) == []
    # the band really holds texel centres, edges, faces and outside samples, and every kind of level
    t = (x[:, 0] + 1) / 2 * grid[0] - 0.5
    assert bool((t == t.round()).any()) and bool((t - t.floor() == 0.5).any())
    assert bool((x[:, 0] == -1).any()) and bool((x[:, 0] == 1).any()) and bool((t < -1.5).any()) and bool((t > grid[0] + 0.5).any())
    assert all(bool((lv == v).any()) for v in (0.0, L - 1.0)) and bool((lv < 0).any()) and bool((lv > L - 1).any())
    own = [(b - a) / (g - 1) for a, b, g in zip(*AABB, grid)]
    assert tap_exactness(x, lv, grid, L, own) != []


def test_conditioned_reference_matches_oracle_gradient():
    """With the oracle's own units and its own fp64 taps (no fp32 rounding of the tap sums), the per-tap reference reproduces
    the autograd gradients of TensoSDF.forward + TensoSDF.gradient(training=True) for all four upstreams to 1e-12."""
    from tensoflow_b200 import synthetic
    torch.manual_seed(0)
    o = O.TensoSDF([10, 6, 12], AABB, sdf_n_comp=4, sdf_dim=32, app_dim=8, init_n_levels=1, dtype=torch.float64)
    o.upsample_volume_grid(torch.tensor([20, 12, 24]))
    synthetic.perturb_field(o, seed=1, noise=0.05)
    with torch.no_grad():
        o.sdf_mat[0].weight.mul_(0.05)
    n = 300
    x, lv = lattice_points(n, 7, o.n_levels)
    units = [float(u) for u in o.units]
    g = torch.Generator().manual_seed(9)
    u_sdf, u_feat, u_grad, u_hess = (torch.randn(n, generator=g, dtype=torch.float64), torch.randn(n, 8, generator=g, dtype=torch.float64),
                                     torch.randn(n, 3, generator=g, dtype=torch.float64), torch.randn(n, generator=g, dtype=torch.float64))
    for with_level in (True, False):
        lvl = lv[:, None] if with_level else None
        r = o(x, lvl)
        gr, nh = o.gradient(x, lvl, training=True, sdf=r[:, :1])
        loss = (r[:, 0] * u_sdf).sum() + (r[:, 1:] * u_feat).sum() + (gr * u_grad).sum() + (nh * u_hess).sum()
        want = torch.autograd.grad(loss, list(o.parameters()))
        with torch.no_grad():
            S = torch.stack([o.sdf(x + e, lvl)[:, 0] for e in tap_offsets(units)], 1)
        a = adjoint(S, units, u_sdf, u_grad, u_hess, fp32_sum=False)
        ref, M = reference_grads(o, x, lv if with_level else None, units, a, u_feat)
        for (name, _), w in zip(o.named_parameters(), want):
            e = float((ref[name] - w).abs().max() / w.abs().max())
            assert e <= 1e-12, (name, with_level, e)
            assert bool((M[name] >= ref[name].abs() * (1 - 1e-12)).all()), name
