"""Hierarchical NeuS sampler (tf_sampler_*, tensoflow_b200/sampler.py) on the rays a renderer meets besides object rays: rays
that miss the box (background pixels) or the unit sphere, rays that graze a box edge, rays whose box interval lies outside
[near, far], origins inside the box and directions with an exactly-zero component, sharing CTAs (4 rays each) with ordinary
rays.  The arbiter is the fp64 oracle restatement of ShapeRenderer.sample_ray (oracle/torch_oracle_renderer.py, pinned to the
reference in tests/test_oracle_cpu.py) driven by the same analytic, level-dependent SDF.

A ray that misses the box has tmin > tmax once both are clipped to its [near, far] window, so its coarse depth list descends;
the reference upsamples it in that order and torch.sort makes every later list ascending.  The row test reads the depth and
SDF rows after every round and holds them to the oracle's lists of the same round."""
import ctypes as C

import pytest
import torch
import torch.nn.functional as F

from conftest import record_err, rel_err
from oracle import torch_oracle_renderer as RR

pytestmark = pytest.mark.gpu

SLAB = ((-0.6, -0.45, -0.7), (0.6, 0.45, 0.7))       # the shape of a shrunk alpha-mask bound: the unit sphere pokes out of it
CUBE = ((-1.0, -1.0, -1.0), (1.0, 1.0, 1.0))         # the default bound: it holds the unit sphere
BOXES = {"slab": SLAB, "cube": CUBE}
VARIANCE = 0.45                                       # inv_s = exp(4.5) = 90: between the caps 64 and 128 of rounds 0 / 1
# (n_samples, n_importance, up_sample_steps); the last one fills the 256-entry depth row of the kernels
CONFIGS = [(64, 64, 4), (64, 0, 0), (16, 16, 1), (33, 27, 3), (128, 128, 4)]
R_FULL = 3001
RAY_COUNTS = (1, 3, 257, R_FULL)                     # one ray, fewer rays than a CTA holds, one ray past a CTA multiple, many
EDGE_KINDS = ("miss_box", "miss_sphere", "graze", "collapsed", "inside", "zero_dir")
TOL = 2e-5


def _cuda():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    return torch.device("cuda:0")


def sdf_any(p, lvl):
    """bumpy sphere whose level set moves a little with the mip level (the SDF of test_renderer's sampler test)"""
    r = p.norm(dim=-1)
    return r - 0.45 - 0.05 * torch.sin(6 * p[..., 0]) * torch.cos(5 * p[..., 1]) + 0.003 * lvl.reshape(-1)


def slab_interval(o, d, box):
    """unclipped box interval of the sampler (the same `d == 0 -> 1e-6` substitution), in fp64"""
    lo, hi = (torch.tensor(b, dtype=torch.float64) for b in box)
    o, d = o.double(), d.double()
    vec = torch.where(d == 0, torch.full_like(d, 1e-6), d)
    ra, rb = (hi - o) / vec, (lo - o) / vec
    return torch.minimum(ra, rb).amax(-1), torch.maximum(ra, rb).amin(-1)


def _unit(g, n):
    return F.normalize(torch.randn(n, 3, generator=g, dtype=torch.float64), dim=-1)


def _pool(kind, box, g, n):
    """n rays of one kind: (origins, directions, explicit [near, far] or None for the sphere window), fp64"""
    lo, hi = (torch.tensor(b, dtype=torch.float64) for b in box)
    if kind in ("ordinary", "collapsed"):
        o = _unit(g, n) * (1.6 + 1.2 * torch.rand(n, 1, generator=g, dtype=torch.float64))
        tgt = lo * 0.5 + (hi - lo) * 0.5 * torch.rand(n, 3, generator=g, dtype=torch.float64)
        d = F.normalize(tgt - o, dim=-1)
        if kind == "ordinary":
            return o, d, None
        # the box interval wholly before `near` (first half) or after `far`; a short gap, so that the t_rand shift of up to
        # 1/n_samples moves some of these one-depth lists back into the box, where they pack n zero-length intervals
        tmin, tmax = slab_interval(o.float(), d.float(), box)
        gap = 0.002 + 0.078 * torch.rand(n, generator=g, dtype=torch.float64)
        before = torch.arange(n) < n // 2
        near = torch.where(before, tmax + gap, (tmin - gap - 1.0).clamp_min(1e-3))
        far = torch.where(before, tmax + gap + 1.0, tmin - gap)
        return o, d, torch.stack([near, far], -1)
    if kind == "miss_box":                          # aimed at points between the box and a sphere of radius 1.5
        o = _unit(g, n) * (1.6 + 1.2 * torch.rand(n, 1, generator=g, dtype=torch.float64))
        tgt = _unit(g, n) * (0.5 + torch.rand(n, 1, generator=g, dtype=torch.float64))
        return o, F.normalize(tgt - o, dim=-1), None
    if kind == "miss_sphere":                       # closest approach to the origin between 1.02 and 1.45
        c = _unit(g, n) * (1.02 + 0.43 * torch.rand(n, 1, generator=g, dtype=torch.float64))
        d = F.normalize(torch.linalg.cross(c, torch.randn(n, 3, generator=g, dtype=torch.float64)), dim=-1)
        return c - d * (1.5 + torch.rand(n, 1, generator=g, dtype=torch.float64)), d, None
    if kind == "graze":                             # through a point within +-4e-5 of a box edge, across the edge
        a = torch.randint(0, 3, (n,), generator=g)
        b = (a + 1 + torch.randint(0, 2, (n,), generator=g)) % 3
        sa, sb = (torch.randint(0, 2, (n, 2), generator=g) * 2 - 1).double().unbind(-1)
        ea, eb = F.one_hot(a, 3).double(), F.one_hot(b, 3).double()
        mid, half = (hi + lo) * 0.5, (hi - lo) * 0.5
        p = mid + half * (torch.rand(n, 3, generator=g, dtype=torch.float64) - 0.5) * 1.2
        p = p * (1 - ea - eb) + ea * (mid + sa[:, None] * half) + eb * (mid + sb[:, None] * half)
        eps = (torch.rand(n, 1, generator=g, dtype=torch.float64) - 0.5) * 8e-5
        p = p + eps * (sa[:, None] * ea + sb[:, None] * eb)
        u = sa[:, None] * ea - sb[:, None] * eb + (1 - ea - eb) * (torch.rand(n, 3, generator=g, dtype=torch.float64) - 0.5)
        d = F.normalize(u, dim=-1)
        return p - d * (1.8 + 0.8 * torch.rand(n, 1, generator=g, dtype=torch.float64)), d, None
    if kind == "inside":
        o = lo * 0.8 + (hi - lo) * 0.8 * torch.rand(n, 3, generator=g, dtype=torch.float64)
        return o, _unit(g, n), None
    if kind == "zero_dir":                          # one or two direction components exactly zero, hitting or missing the box
        zero = torch.rand(n, 3, generator=g) < torch.where(torch.rand(n, 1, generator=g) < 0.5, 1 / 3, 2 / 3)
        zero[zero.all(-1)] = torch.tensor([True, True, False])
        zero[~zero.any(-1)] = torch.tensor([False, True, False])
        d = F.normalize(torch.randn(n, 3, generator=g, dtype=torch.float64).masked_fill(zero, 0.0), dim=-1)
        p = (torch.rand(n, 3, generator=g, dtype=torch.float64) - 0.5) * 1.9
        return p - d * (2.0 + 0.6 * torch.rand(n, 1, generator=g, dtype=torch.float64)), d, None
    raise ValueError(kind)


def edge_rays(box, seed=11, R=R_FULL):
    """R rays, every fourth one (index 1 mod 4) ordinary, the others cycling through EDGE_KINDS, so that each CTA of the
    kernels mixes edge rays with an ordinary one.  Returns fp32 CPU tensors (rays_o, dirs, near, far, radiis, rays_cos, t_rand)
    and `kind` [R] (index into ("ordinary",) + EDGE_KINDS)."""
    g = torch.Generator().manual_seed(seed)
    kinds = ("ordinary",) + EDGE_KINDS
    slot = torch.arange(R)
    kind = torch.where(slot % 4 == 1, 0, 1 + (slot - (slot + 2) // 4) % len(EDGE_KINDS))
    o, d, nf, tr = (torch.zeros(R, 3), torch.zeros(R, 3), torch.zeros(R, 2), torch.zeros(R))
    for ki, name in enumerate(kinds):
        want = int((kind == ki).sum())
        po, pd, pnf, pt, have = [], [], [], [], 0
        while have < want:
            co, cd, cnf = _pool(name, box, g, 4 * want + 64)
            co, cd = co.float(), cd.float()
            if cnf is None:
                cnf = torch.cat(RR.near_far_from_sphere(co.double(), cd.double()), -1)
            cnf = cnf.float()
            ct = torch.rand(co.shape[0], generator=g)
            if name == "inside":             # keep the first depth of a ray from inside the box in front of its origin
                ct = 0.5 + 0.5 * ct         # (a depth behind it has no mip level: log2 of a negative ball radius)
            keep = _keep(name, co, cd, cnf, ct, box)
            po.append(co[keep]); pd.append(cd[keep]); pnf.append(cnf[keep]); pt.append(ct[keep])
            have += int(keep.sum())
        sel = kind == ki
        o[sel], d[sel], nf[sel], tr[sel] = (torch.cat(x)[:want] for x in (po, pd, pnf, pt))
    rays = dict(rays_o=o, dirs=d, near=nf[:, :1].contiguous(), far=nf[:, 1:].contiguous(),
                radiis=1.25e-3 * 2.0 ** (torch.rand(R, 1, generator=g) * 3 - 1), rays_cos=0.7 + 0.3 * torch.rand(R, 1, generator=g),
                t_rand=tr[:, None].contiguous())
    return rays, kind


def _keep(name, o, d, nf, t_rand, box):
    """which candidates belong to the kind; apart from origins inside the box, every depth stays >= 0.1 - 1/16 > 0"""
    tmin, tmax = slab_interval(o, d, box)
    near, far = nf[:, 0].double(), nf[:, 1].double()
    cmin, cmax = tmin.clamp(near, far), tmax.clamp(near, far)
    inside_window = (tmin > near) & (tmin < far) & (tmax > near) & (tmax < far)
    ahead = torch.minimum(cmin, cmax) > 0.1
    if name == "ordinary":
        return (tmax - tmin > 0.05) & ahead
    if name == "miss_box":
        return (tmin - tmax > 0.05) & inside_window & ahead
    if name == "miss_sphere":
        return ahead
    if name == "graze":
        return ((cmax - cmin).abs() <= 1e-4) & inside_window & ahead
    if name == "collapsed":                         # the one depth, shifted by t_rand, keeps 1e-3 off the box faces for all n
        keep = (cmax == cmin) & (tmax - tmin > 0.05) & ahead
        for ns in sorted({c[0] for c in CONFIGS}):
            for z in (cmin, cmin + (t_rand.double() - 0.5) * 2.0 / ns):
                keep &= torch.minimum((z - tmin).abs(), (z - tmax).abs()) > 1e-3
        return keep
    if name == "inside":                            # not a window behind the origin (far < 0: it points away from the sphere)
        return torch.minimum(cmin, cmax) > 0
    if name == "zero_dir":
        return (d == 0).any(-1) & ((tmin - tmax).abs() > 1e-3) & ahead
    raise ValueError(name)


def clipped_span(rays, box):
    tmin, tmax = slab_interval(rays["rays_o"], rays["dirs"], box)
    near, far = rays["near"][:, 0].double(), rays["far"][:, 0].double()
    return tmin.clamp(near, far), tmax.clamp(near, far)


def run_oracle(rays, box, ns, ni, steps, perturb, clip_var, dtype=torch.float64):
    """oracle (fp64: the arbiter; fp32: the same arithmetic at the kernels' precision): the lists after every round
    (ShapeRenderer.sample_ray's `rounds`) and the packed intervals"""
    ora = RR.ShapeRenderer([32] * 3, max_levels=1, n_samples=ns, n_importance=ni, up_sample_steps=steps, clip_sample_variance=clip_var,
                           dtype=dtype)
    ora.sdf_network.aabb.copy_(torch.tensor(box, dtype=dtype))
    ora.sdf_network.sdf = lambda p, lvl=None: sdf_any(p, lvl)[:, None]
    with torch.no_grad():
        ora.deviation_network.variance.fill_(VARIANCE)
    rounds = []
    t0, t1, idx = ora.sample_ray(*(rays[k].to(dtype) for k in ("rays_o", "dirs", "near", "far", "radiis", "rays_cos")),
                                 rays["t_rand"].to(dtype) if perturb else None, rounds=rounds)
    return rounds, (t0, t1, idx), float(ora.base_radii)


def well_conditioned(rays, box, ns, ni, steps, perturb, clip_var, rounds64):
    """Rays whose lists fp32 arithmetic reproduces: adjacent coarse depths more than 1e-4 apart once the +1e-5 guard of the
    section cosine is added (closer ones cancel the raw_cos denominator: grazing rays, one-depth lists), and lists of the
    fp32 oracle within TOL / 4 of the fp64 ones after every round.  The second condition excludes rays that pass the surface
    at a small distance inside the unit sphere without reaching it: there both section sigmoids round near 1, their
    difference (the alpha) carries the rounding of 1.0f, and with little weight on the ray that noise moves the samples by
    up to ~1e-3 in any fp32 implementation."""
    t = rounds64[0][0]
    well = ((t[:, 1:] - t[:, :-1] + 1e-5).abs() > 1e-4).all(-1)
    rounds32, _, _ = run_oracle(rays, box, ns, ni, steps, perturb, clip_var, torch.float32)
    for (z64, s64), (z32, s32) in zip(rounds64, rounds32):
        well &= ((z32.double() - z64).abs() <= TOL / 4).all(-1)
        if s64 is not None:
            well &= ((s32.double() - s64).abs() <= TOL / 4).all(-1)
    return well


def check_well(err, strict, what):
    """err: per-ray largest |kernel - oracle| over the well-conditioned rays.  Every ray in `strict` (the rays that miss the
    box or the unit sphere) is within TOL.  Of the others 99.5 % are, and none is off by more than 10 TOL: in the later,
    sharper rounds the sigmoid rounding described in well_conditioned still moves a sample of about one ray in a thousand by
    a few TOL, more than the fp32 oracle showed on that ray."""
    if bool(strict.any()):
        es = float(err[strict].max())
        assert es <= TOL, f"{what}: a ray that misses the box or the sphere is off by {es:.3e}"
    if err.numel() > 0:
        share = float((err <= TOL).double().mean())
        assert share >= 0.995 and float(err.max()) <= 10 * TOL, \
            f"{what}: {share:.4f} of the well-conditioned rays within {TOL}, largest error {float(err.max()):.3e}"


def kernel_rows(rays, R, box, base_radii, ns, ni, steps, perturb, clip_var):
    """tf_sampler_init / tf_sampler_upsample / tf_sampler_finalize in the call sequence of sampler.hierarchical_sample, keeping
    the (z, sdf) rows after the coarse samples and after every merge (sdf None after the last merge, which carries no SDF)
    and the per-ray counts of the finalize count pass."""
    from tensoflow_b200 import _lib, sampler
    from tensoflow_b200._lib import check, ptr, stream_ptr
    lib = _lib.load()
    dev = _cuda()
    ro, rd, nr, fr, rad, rc = (rays[k][:R].reshape(R, -1).squeeze(-1).contiguous().to(dev)
                               for k in ("rays_o", "dirs", "near", "far", "radiis", "rays_cos"))
    aabb6 = (C.c_float * 6)(*box[0], *box[1])
    S = ns + ni
    z = torch.empty(R, S, device=dev)
    sdf = torch.empty(R, S, device=dev)
    pts = torch.empty(R * ns, 3, device=dev)
    level = torch.empty(R * ns, device=dev)
    tr = rays["t_rand"][:R].reshape(-1).contiguous().to(dev) if perturb else None
    check(lib.tf_sampler_init(ptr(ro), ptr(rd), ptr(nr), ptr(fr), ptr(rad), ptr(rc), ptr(sampler._table("lin", ns, dev)), ptr(tr), aabb6,
                              base_radii, R, ns, S, ptr(z), ptr(pts), ptr(level), stream_ptr()), "tf_sampler_init")
    sdf[:, :ns] = sdf_any(pts, level).reshape(R, ns)
    rows = [(z[:, :ns].clone(), sdf[:, :ns].clone())]
    n = ns
    if ni > 0:
        m = ni // steps
        u = sampler._table("u", m, dev)
        var = torch.tensor([VARIANCE], device=dev) if clip_var else None
        new_z = new_sdf = None
        m_in = 0
        for i in range(steps):
            out_z = torch.empty(R, m, device=dev)
            out_pts = torch.empty(R * m, 3, device=dev)
            out_lv = torch.empty(R * m, device=dev)
            check(lib.tf_sampler_upsample(ptr(ro), ptr(rd), ptr(rad), ptr(rc), ptr(z), ptr(sdf), ptr(new_z), ptr(new_sdf), m_in, ptr(u), m,
                                          ptr(var), float(64 * 2 ** i), base_radii, R, n, S, ptr(out_z), ptr(out_pts), ptr(out_lv),
                                          stream_ptr()), "tf_sampler_upsample")
            n += m_in
            if i > 0:
                rows.append((z[:, :n].clone(), sdf[:, :n].clone()))
            new_z, m_in = out_z, m
            new_sdf = sdf_any(out_pts, out_lv).contiguous() if i + 1 < steps else None
        check(lib.tf_sampler_upsample(ptr(ro), ptr(rd), ptr(rad), ptr(rc), ptr(z), ptr(sdf), ptr(new_z), None, m_in, None, 0, None, 0.0,
                                      base_radii, R, n, S, None, None, None, stream_ptr()), "tf_sampler_upsample (merge)")
        n += m_in
        rows.append((z[:, :n].clone(), None))
    counts = torch.empty(R, device=dev, dtype=torch.int32)
    check(lib.tf_sampler_finalize(ptr(ro), ptr(rd), ptr(z), aabb6, R, n, S, ptr(counts), None, None, None, None, stream_ptr()),
          "tf_sampler_finalize (count)")
    return [(zr.cpu().double(), None if sr is None else sr.cpu().double()) for zr, sr in rows], counts.cpu().long()


@pytest.mark.parametrize("perturb,clip_var", [(True, True), (False, False), (True, False), (False, True)])
@pytest.mark.parametrize("box", sorted(BOXES))
@pytest.mark.parametrize("ns,ni,steps", CONFIGS)
def test_sampler_rows_match_oracle_every_round(ns, ni, steps, box, perturb, clip_var):
    """After the coarse samples and after every merge, every depth row is finite, every merged row ascends, and on
    well-conditioned rays the depth and SDF rows equal the oracle's lists of the same round (check_well); rows of
    ill-conditioned rays stay within the ray's clipped span (widened by the t_rand shift).  Rays that miss the box get no
    samples from the finalize pass."""
    _cuda()
    b = BOXES[box]
    rays, kind = edge_rays(b)
    rounds, (ot0, _, oidx), base_radii = run_oracle(rays, b, ns, ni, steps, perturb, clip_var)
    assert len(rounds) == (steps + 1 if ni > 0 else 1)
    cmin, cmax = clipped_span(rays, b)
    shift = 1.0 / ns if perturb else 0.0
    lo, hi = torch.minimum(cmin, cmax) - shift - 1e-5, torch.maximum(cmin, cmax) + shift + 1e-5
    well = well_conditioned(rays, b, ns, ni, steps, perturb, clip_var, rounds)
    assert bool(well[kind == 1].all()), "every box-missing ray of the set is well-conditioned"
    assert bool((cmin > cmax)[kind == 1].all()), "box-missing rays have descending coarse lists"
    strict = well & ((kind == 1) | (kind == 2))
    o_counts = torch.bincount(oidx, minlength=R_FULL)
    for R in RAY_COUNTS:
        rows, counts = kernel_rows(rays, R, b, base_radii, ns, ni, steps, perturb, clip_var)
        assert len(rows) == len(rounds)
        w, ill = well[:R], ~well[:R]
        for r, ((kz, ks), (oz, osdf)) in enumerate(zip(rows, rounds)):
            oz, what = oz[:R], f"R={R} round {r}"
            assert kz.shape == oz.shape, what
            assert bool(torch.isfinite(kz).all()), f"{what}: non-finite depth"
            if r > 0:
                bad = (kz[:, 1:] < kz[:, :-1]).any(-1)
                assert not bool(bad.any()), f"{what}: rows of rays {bad.nonzero().flatten()[:8].tolist()} are not ascending"
            if bool(w.any()):
                e = (kz[w] - oz[w]).abs().amax(-1)
                if R == R_FULL:
                    record_err(f"depth row, round {r}, well-conditioned rays (abs tol {TOL})", kz[w], oz[w], None,
                               abs_err=float(e.max()), share_within_tol=float((e <= TOL).double().mean()))
                check_well(e, strict[:R][w], f"{what}: depth rows")
                if ks is not None:
                    assert bool(torch.isfinite(ks).all()), f"{what}: non-finite SDF"
                    es = (ks[w] - osdf[:R][w]).abs().amax(-1)
                    if R == R_FULL:
                        record_err(f"SDF row, round {r}, well-conditioned rays (abs tol {TOL})", ks[w], osdf[:R][w], None,
                                   abs_err=float(es.max()), share_within_tol=float((es <= TOL).double().mean()))
                    check_well(es, strict[:R][w], f"{what}: SDF rows")
            if bool(ill.any()):
                out = (kz[ill] < lo[:R][ill, None]) | (kz[ill] > hi[:R][ill, None])
                assert not bool(out.any()), f"{what}: depths of ill-conditioned rays outside their clipped span"
        same = (counts == o_counts[:R])[w]                 # a mid point within fp32 rounding of a box face may flip
        assert float(same.float().mean()) >= (0.99 if R > 100 else 1.0), f"R={R}: per-ray counts of the finalize pass"
        assert int(counts[(kind[:R] == 1)].abs().sum()) == 0, f"R={R}: a box-missing ray got samples"


@pytest.mark.parametrize("perturb", [True, False])
@pytest.mark.parametrize("box", sorted(BOXES))
@pytest.mark.parametrize("ns,ni,steps", CONFIGS)
def test_sampler_packed_edges_match_oracle(ns, ni, steps, box, perturb):
    """sampler.hierarchical_sample: rays that miss the box get no samples, every packed value is finite, counts / t_starts /
    t_ends / CSR offsets match the oracle, and one-depth lists inside the box pack zero-length intervals as the oracle does."""
    from tensoflow_b200 import sampler
    dev = _cuda()
    b = BOXES[box]
    rays, kind = edge_rays(b)
    rounds, (ot0, ot1, oidx), base_radii = run_oracle(rays, b, ns, ni, steps, perturb, True)
    well = well_conditioned(rays, b, ns, ni, steps, perturb, True, rounds)
    tmin, tmax = slab_interval(rays["rays_o"], rays["dirs"], b)
    miss = tmin - tmax > 1e-3
    assert int(miss.sum()) > R_FULL // 8
    cmin, cmax = clipped_span(rays, b)
    shift = 1.0 / ns if perturb else 0.0
    lo, hi = torch.minimum(cmin, cmax) - shift - 1e-5, torch.maximum(cmin, cmax) + shift + 1e-5
    collapsed = kind == 1 + EDGE_KINDS.index("collapsed")
    zero_len_rays = 0
    for R in RAY_COUNTS:
        s0, s1, sidx, offs = sampler.hierarchical_sample(
            lambda p, lvl: sdf_any(p, lvl), torch.tensor(b, device=dev), base_radii,
            *(rays[k][:R].to(dev) for k in ("rays_o", "dirs", "near", "far", "radiis", "rays_cos")), ns, ni, steps,
            1.0 if perturb else 0.0, rays["t_rand"][:R].to(dev) if perturb else None, torch.tensor(VARIANCE, device=dev), True)
        s0, s1, sidx, offs = s0.cpu().double(), s1.cpu().double(), sidx.cpu(), offs.cpu().long()
        assert bool(torch.isfinite(s0).all()) and bool(torch.isfinite(s1).all()), f"R={R}: non-finite packed depths"
        ko = oidx < R
        t0, t1, idx = ot0[ko], ot1[ko], oidx[ko]
        cnt_o = torch.bincount(idx, minlength=R)
        cnt_k = torch.bincount(sidx, minlength=R)
        assert torch.equal(offs, torch.cat([torch.zeros(1, dtype=torch.long), torch.cumsum(cnt_k, 0)])), f"R={R}: CSR offsets"
        assert int(cnt_k[miss[:R]].sum()) == 0, f"R={R}: a ray that misses the box got samples"
        same = cnt_o == cnt_k                                 # a mid point within fp32 rounding of a box face may flip
        share = float(same[well[:R]].float().mean())
        assert share >= (0.99 if R > 100 else 1.0), f"R={R}: equal counts on {share:.4f} of the well-conditioned rays"
        assert bool(same[collapsed[:R]].all()), f"R={R}: one-depth lists packed differently"
        sel = same & well[:R]
        kk, oo = sel[sidx], sel[idx]
        if bool(kk.any()):
            e = torch.zeros(R, dtype=torch.float64)         # per ray: the largest error of its t_starts and t_ends
            e.index_reduce_(0, sidx[kk], torch.maximum((s0[kk] - t0[oo]).abs(), (s1[kk] - t1[oo]).abs()), "amax")
            if R == R_FULL:
                record_err(f"t_starts, well-conditioned rays (abs tol {TOL})", s0[kk], t0[oo], None,
                           abs_err=float(e.max()), share_within_tol=float((e[sel] <= TOL).double().mean()))
                record_err(f"t_ends, well-conditioned rays (abs tol {TOL})", s1[kk], t1[oo], None)
            check_well(e[sel], torch.zeros(int(sel.sum()), dtype=torch.bool), f"R={R}: packed intervals")
        ki = (~well[:R])[sidx]
        assert bool(((s0[ki] >= lo[sidx[ki]]) & (s0[ki] <= hi[sidx[ki]])).all()), f"R={R}: ill-conditioned rays outside their span"
        zk, zo = collapsed[:R][sidx], collapsed[:R][idx]      # equal counts on these rays, so the packed entries line up
        assert bool((t0[zo] == t1[zo]).all())
        assert torch.equal(s0[zk], s1[zk]), f"R={R}: one-depth lists must pack zero-length intervals"
        if bool(zk.any()):
            assert float((s0[zk] - t0[zo]).abs().max()) <= TOL, f"R={R}: zero-length intervals at other depths than the oracle's"
            zero_len_rays = max(zero_len_rays, int(torch.unique(sidx[zk]).numel()))
        ds = s0[1:] - s0[:-1]
        assert bool((ds[sidx[1:] == sidx[:-1]] >= 0).all()), f"R={R}: packed depths of a ray must ascend"
    if perturb:
        assert zero_len_rays > 0, "the ray set has no one-depth list inside the box"


def test_sampler_rejects_rows_past_256():
    """n_samples + n_importance = 257 does not fit a depth row: the library reports it and launches nothing"""
    from tensoflow_b200 import _lib, sampler
    dev = _cuda()
    rays, _ = edge_rays(SLAB, R=8)
    n0 = _lib.launch_count()
    with pytest.raises(RuntimeError, match="ray sampler"):
        sampler.hierarchical_sample(lambda p, lvl: sdf_any(p, lvl), torch.tensor(SLAB, device=dev), 0.01,
                                    *(rays[k].to(dev) for k in ("rays_o", "dirs", "near", "far", "radiis", "rays_cos")), 129, 128, 4,
                                    1.0, rays["t_rand"].to(dev), torch.tensor(VARIANCE, device=dev), True)
    torch.cuda.synchronize()
    assert _lib.launch_count() == n0


@pytest.mark.parametrize("train", [False, True])
def test_render_image_with_background_pixels(train):
    """ShapeRenderer.render of a 16 x 16 image with a wide field of view (focal length 6 pixels, camera 2.6 from the centre),
    most of whose pixels miss the box, against the fp64 oracle's render with the golden renderer state: background pixels get
    acc 0, normal (0, 0, 1) and ray_rgb 1 exactly; the other pixels pass the rule of test_cuda_renderer_golden (calibrated
    against the fp32 oracle on the CPU); nothing is NaN.  Eval mode is unperturbed, train mode uses a fixed t_rand."""
    from tensoflow_b200.shape_renderer import ShapeRenderer
    from test_golden import load
    from test_renderer import CFG, _oracle
    dev = _cuda()
    g = load("renderer.npz")
    h = w = 16
    K = [[6.0, 0.0, 8.0], [0.0, 6.0, 8.0], [0.0, 0.0, 1.0]]
    pose = [[1.0, 0.0, 0.0, 0.2], [0.0, 1.0, 0.0, -0.15], [0.0, 0.0, 1.0, 2.6]]
    rays = ShapeRenderer.image_rays(pose, K, h, w, "cpu")
    rays["rays_d"] = rays["dirs"]
    near, far = RR.near_far_from_sphere(rays["rays_o"], rays["dirs"])
    t_rand = torch.rand(h * w, 1, generator=torch.Generator().manual_seed(21)) if train else None
    tmin, tmax = slab_interval(rays["rays_o"], rays["dirs"], CUBE)
    assert int((tmin > tmax).sum()) >= h * w // 3, "at least a third of the pixels miss the box"
    ref, counts = {}, None
    for dt in (torch.float64, torch.float32):
        mo = _oracle(g, dt)
        mo.color_network.envlight.build_mips()
        args = [rays[k].to(dt) for k in ("rays_o", "dirs", "radiis", "rays_cos")] + [near.to(dt), far.to(dt)]
        ref[dt] = {k: v.detach() for k, v in mo.render(*args, 0.7, 30000, t_rand=None if t_rand is None else t_rand.to(dt)).items()
                   if k in ("ray_rgb", "acc", "normal")}
        if dt == torch.float64:
            with torch.no_grad():
                _, _, idx = mo.sample_ray(args[0], args[1], args[4], args[5], args[2], args[3], None if t_rand is None else t_rand.to(dt))
            counts = torch.bincount(idx, minlength=h * w)
    m = ShapeRenderer(dict(device=dev, shader_config=dict(env_res=16, env_min_res=4), **CFG))
    res = m.load_state_dict(g["state"], strict=False)
    assert not res.unexpected_keys, res.unexpected_keys
    m.color_network.envlight.build_mips()
    batch = {k: rays[k].to(dev) for k in ("rays_o", "rays_d", "dirs", "radiis", "rays_cos")}
    out = m.render(batch, near.to(dev), far.to(dev), None, perturb_overwrite=-1 if train else 0, cos_anneal_ratio=0.7, is_train=train,
                   step=30000, t_rand=None if t_rand is None else t_rand.to(dev))
    got = {k: out[k].detach().cpu() for k in ("ray_rgb", "acc", "normal")}
    cnt_k = torch.bincount(m._last_ray_offsets[0].cpu(), minlength=h * w)
    for k, v in got.items():
        assert bool(torch.isfinite(v).all()), f"{k}: NaN or inf"
    bg = counts == 0
    assert int(bg.sum()) >= h * w // 3 and int((~bg).sum()) >= 16
    assert bool((cnt_k[bg] == 0).all()), "a background pixel got samples"
    assert bool((got["acc"][bg] == 0).all())
    assert bool((got["ray_rgb"][bg] == 1).all())
    assert torch.equal(got["normal"][bg], torch.tensor([0.0, 0.0, 1.0]).expand(int(bg.sum()), 3))
    same = ~bg & (cnt_k == counts)                       # a sample whose mid point sits on a box face may flip
    assert int(same.sum()) >= 0.75 * int((~bg).sum()), f"{int(same.sum())} of {int((~bg).sum())} object pixels with equal counts"
    for k in ("ray_rgb", "acc", "normal"):
        e, e_ref = rel_err(got[k][same], ref[torch.float64][k][same]), rel_err(ref[torch.float32][k][same], ref[torch.float64][k][same])
        record_err(f"{k}, object pixels", got[k][same], ref[torch.float64][k][same], max(1e-4, 4 * e_ref), fp32_oracle_rel_err=e_ref)
        assert e <= max(1e-4, 4 * e_ref), f"{k}: rel err {e:.3e} (fp32 oracle vs fp64 oracle {e_ref:.3e})"
