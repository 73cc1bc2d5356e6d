"""GPU parity tests of the volume-compositing / importance-resampling kernels against the C oracle and the
reference's own CUDA kernels (oracle/_ref where built, their stored outputs elsewhere: tests/ref_golden.py).
Tolerances are written per test; the serial-order recurrences are expected to be bit exact."""
import numpy as np
import pytest
import torch

import ref_golden
import scenes
from oracle import rayops as orc
from oracle import ref_gpu

pytestmark = pytest.mark.gpu
_fresh_generators = pytest.fixture(autouse=True)(ref_golden.fresh_generators)
V = 128


def T(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def N(t):
    return t.detach().cpu().numpy()


def to_oracle(rsp):
    p = orc.Packed(rsp.ray_start_end_idx.shape[0], rsp.samples_z.shape[0])
    p.pos, p.dirs, p.z, p.dt = N(rsp.samples_pos), N(rsp.samples_dirs), N(rsp.samples_z), N(rsp.samples_dt)
    p.fixed_dt, p.start_end = N(rsp.ray_fixed_dt), N(rsp.ray_start_end_idx)
    p.max_nr_samples = rsp.max_nr_samples
    p.equal, p.fixed_n, p.has_sdf = rsp.rays_have_equal_nr_of_samples, rsp.fixed_nr_of_samples_per_ray, rsp.has_sdf
    if rsp.has_sdf:
        p.sdf = N(rsp.samples_sdf)
    return p


def to_ref(rsp):
    p = ref_gpu.Packed(rsp.ray_start_end_idx.shape[0], rsp.samples_z.shape[0])
    p.pos, p.dirs, p.z, p.dt = rsp.samples_pos, rsp.samples_dirs, rsp.samples_z, rsp.samples_dt
    p.fixed_dt, p.start_end = rsp.ray_fixed_dt, rsp.ray_start_end_idx
    p.max_nr_samples = rsp.max_nr_samples
    p.equal, p.fixed_n, p.has_sdf = rsp.rays_have_equal_nr_of_samples, rsp.fixed_nr_of_samples_per_ray, rsp.has_sdf
    if rsp.has_sdf:
        p.sdf = rsp.samples_sdf.contiguous()
    return p


@pytest.fixture(scope="module")
def packed(cuda):
    from permuto_sdf import OccupancyGrid, Sphere
    o, d = scenes.make_rays(384, seed=7)
    values, occ = scenes.analytic_occupancy(V)
    grid = OccupancyGrid(V, 1.0, [0, 0, 0])
    grid.set_grid_occupancy(T(occ.astype(np.uint8)).bool())
    sph = Sphere(0.5, [0, 0, 0])
    pe, te, px, tx, hit = sph.ray_intersection(T(o), T(d))
    rsp = grid.compute_samples_in_occupied_regions(T(o), T(d), te, tx, 1e-3, 96, False).compact_to_valid_samples()
    assert rsp.samples_pos.shape[0] > 5000
    return dict(rsp=rsp, o=T(o), d=T(d), tx=tx)


def eq(a, b, what, tol=0.0):
    a, b = np.asarray(a), np.asarray(b)
    assert a.shape == b.shape, what
    if tol == 0.0:
        assert np.array_equal(a, b), "%s not bit exact (max err %g)" % (what, np.abs(a.astype(np.float64) - b).max())
    else:
        err = np.abs(a.astype(np.float64) - b.astype(np.float64)).max()
        assert err <= tol, "%s: max abs err %g > %g" % (what, err, tol)


def test_scans_and_sums(packed):
    from permuto_sdf import VolumeRendering as VR
    rsp = packed["rsp"]
    Ns, R = rsp.samples_z.shape[0], rsp.ray_start_end_idx.shape[0]
    p = to_oracle(rsp)
    rp = ref_golden.once(lambda: to_ref(rsp))
    g = torch.Generator(device="cuda").manual_seed(0)
    alpha = torch.rand(Ns, 1, device="cuda", generator=g) * 0.2 + 0.8
    Tt, bg = VR.cumprod_alpha2transmittance(rsp, alpha)
    eT, ebg = orc.vr_cumprod(p, N(alpha))
    eq(N(Tt), eT, "transmittance"); eq(N(bg), ebg, "bg_transmittance")
    w = torch.rand(Ns, 1, device="cuda", generator=g)
    rgb = torch.rand(Ns, 3, device="cuda", generator=g)
    eq(N(VR.integrate_with_weights(rsp, rgb, w)), orc.vr_integrate(p, N(rgb), N(w)), "integrate")
    for D in (1, 2, 3, 32):
        v = torch.rand(Ns, D, device="cuda", generator=g)
        sr, ss = VR.sum_over_each_ray(rsp, v)
        er, es = orc.vr_sum(p, N(v))
        eq(N(sr), er, "sum ray D=%d" % D); eq(N(ss), es, "sum sample D=%d" % D)
        ref = ref_golden.once(lambda: ref_gpu.vr_sum(rp(), v))
        ref_golden.equal("volrender.sum_ray.D%d" % D, sr, lambda: ref()[0])
        ref_golden.equal("volrender.sum_sample.D%d" % D, ss, lambda: ref()[1])
        if D <= 3:
            gr, gs = torch.rand(R, D, device="cuda", generator=g), torch.rand(Ns, D, device="cuda", generator=g)
            gb = VR.sum_over_each_ray_backward(gr, gs, rsp, v)
            eq(N(gb), orc.vr_sum_backward(p, N(gr), N(gs)), "sum backward")
            ref_golden.equal("volrender.sum_backward.D%d" % D, gb, lambda: ref_gpu.vr_sum_backward(rp(), gr, gs, v))
    for inv in (False, True):
        eq(N(VR.cumsum_over_each_ray(rsp, w, inv)), orc.vr_cumsum(p, N(w), inv), "cumsum inverse=%s" % inv)
    eq(N(VR.compute_cdf(rsp, w)), orc.vr_cdf(p, N(w)), "cdf")
    eq(N(VR.compute_dt(rsp, packed["tx"], True)), orc.vr_compute_dt(p, N(packed["tx"]), True), "compute_dt")
    ref = ref_golden.once(lambda: ref_gpu.vr_cumprod(rp(), alpha))
    ref_golden.equal("volrender.T", Tt, lambda: ref()[0]); ref_golden.equal("volrender.bg", bg, lambda: ref()[1])
    ref_golden.equal("volrender.integrate", VR.integrate_with_weights(rsp, rgb, w), lambda: ref_gpu.vr_integrate(rp(), rgb, w))
    ref_golden.equal("volrender.rev_cumsum", VR.cumsum_over_each_ray(rsp, w, True), lambda: ref_gpu.vr_cumsum(rp(), w, True))
    ref_golden.equal("volrender.cdf", VR.compute_cdf(rsp, w), lambda: ref_gpu.vr_cdf(rp(), w))
    ref_golden.equal("volrender.dt", VR.compute_dt(rsp, packed["tx"], False), lambda: ref_gpu.vr_compute_dt(rp(), packed["tx"], False))
    # backward kernels
    gT = torch.rand(Ns, 1, device="cuda", generator=g)
    gbg = torch.rand(R, 1, device="cuda", generator=g)
    cs = VR.cumsum_over_each_ray(rsp, gT * Tt, True)
    ga = VR.cumprod_alpha2transmittance_backward(gT, gbg, rsp, alpha, Tt, bg, cs)
    eq(N(ga), orc.vr_cumprod_backward(p, N(gbg), N(alpha), N(bg), N(cs)), "cumprod backward", 1e-6)
    gp = torch.rand(R, 3, device="cuda", generator=g)
    pred = VR.integrate_with_weights(rsp, rgb, w)
    VR.reference_bugs = False
    gv, gw = VR.integrate_with_weights_backward(gp, rsp, rgb, w, pred)
    ev, ew = orc.vr_integrate_backward(p, N(gp), N(rgb), N(w), False)
    eq(N(gv), ev, "integrate backward vals"); eq(N(gw), ew, "integrate backward weights (fixed blue channel)")
    VR.reference_bugs = True
    gv2, gw2 = VR.integrate_with_weights_backward(gp, rsp, rgb, w, pred)
    VR.reference_bugs = False
    eq(N(gw2), orc.vr_integrate_backward(p, N(gp), N(rgb), N(w), True)[1], "integrate backward weights (reference bug mode)")
    ref_golden.close("volrender.cumprod_backward", ga, lambda: ref_gpu.vr_cumprod_backward(rp(), gT, gbg, alpha, Tt, bg, cs), 1e-6)
    ref = ref_golden.once(lambda: ref_gpu.vr_integrate_backward(rp(), gp, rgb, w, pred))
    ref_golden.equal("volrender.integrate_backward.vals", gv2, lambda: ref()[0])
    ref_golden.equal("volrender.integrate_backward.weights_bug_mode", gw2, lambda: ref()[1])


def test_nerf_render(packed):
    from permuto_sdf import VolumeRendering as VR
    rsp = packed["rsp"]
    Ns, R = rsp.samples_z.shape[0], rsp.ray_start_end_idx.shape[0]
    p = to_oracle(rsp)
    g = torch.Generator(device="cuda").manual_seed(1)
    rgb = torch.rand(Ns, 3, device="cuda", generator=g)
    rad = torch.rand(Ns, 1, device="cuda", generator=g) * 200
    pr, dp, bg, w = VR.volume_render_nerf(rsp, rgb, rad, packed["tx"], False)
    er = orc.vr_render_nerf(p, N(rgb), N(rad))
    for a, b, n in zip((pr, dp, bg, w), er, ("rgb", "depth", "bg", "w")):
        eq(N(a), b, "nerf " + n, 2e-5)      # __expf vs expf
    gp, gb = torch.rand(R, 3, device="cuda", generator=g), torch.rand(R, 1, device="cuda", generator=g)
    grgb, grad = VR.volume_render_nerf_backward(gp, gb, torch.zeros(Ns, 1, device="cuda"), pr, rsp, rgb, rad, packed["tx"], False, bg)
    e1, e2 = orc.vr_render_nerf_backward(p, N(gp), N(gb), N(pr), N(bg), N(rgb), N(rad))
    eq(N(grgb), e1, "nerf g_rgb", 2e-5); eq(N(grad), e2, "nerf g_radiance", 2e-4)
    rr = ref_golden.once(lambda: ref_gpu.vr_render_nerf(to_ref(rsp), packed["tx"], rgb, rad))
    for i, (a, n) in enumerate(zip((pr, dp, bg, w), ("rgb", "depth", "bg", "w"))):
        ref_golden.close("volrender.nerf." + n, a, lambda i=i: rr()[i], 1e-6)
    rb = ref_golden.once(lambda: ref_gpu.vr_render_nerf_backward(to_ref(rsp), gp, gb, pr, packed["tx"], bg, rgb, rad))
    ref_golden.close("volrender.nerf.g_rgb", grgb, lambda: rb()[0], 1e-6)
    ref_golden.close("volrender.nerf.g_radiance", grad, lambda: rb()[1], 1e-5)


@pytest.mark.parametrize("jitter", [False, True])
def test_importance_resampling(packed, jitter):
    """sdf2alpha -> cumprod -> weights -> normalise -> cdf -> importance_sample -> combine, as in
    permuto_sdf_py/utils/sdf_utils.py:383-405"""
    from permuto_sdf import VolumeRendering as VR
    rsp = packed["rsp"]
    o, d, tx = packed["o"], packed["d"], packed["tx"]
    sdf = (rsp.samples_pos.norm(dim=1, keepdim=True) - scenes.OBJECT_RADIUS).contiguous()
    rsp.set_sdf(sdf)
    p = to_oracle(rsp)
    alpha = VR.sdf2alpha(rsp, sdf, 512, True, 1.0)
    eq(N(alpha), orc.vr_sdf2alpha(p, N(sdf), 512, True, 1.0), "sdf2alpha", 5e-6)   # expf ulp
    key = "volrender.importance.j%d." % jitter
    ref_golden.close(key + "sdf2alpha", alpha, lambda: ref_gpu.vr_sdf2alpha(to_ref(rsp), sdf, 512, True, 1.0), 2e-6)
    alpha = alpha.clip(0.0, 1.0)
    Tt, _ = VR.cumprod_alpha2transmittance(rsp, 1 - alpha + 1e-7)
    w = alpha * Tt
    _, wsum = VR.sum_over_each_ray(rsp, w)
    w = w / torch.clamp(wsum, min=1e-6)
    cdf = VR.compute_cdf(rsp, w)
    st, inc = VR.m_rng.state, VR.m_rng.inc
    imp = VR.importance_sample(o, d, rsp, cdf, 16, jitter)
    eimp = orc.vr_importance_sample(N(o), N(d), p, N(cdf), 16, jitter, st, inc)
    assert imp.rays_have_equal_nr_of_samples and imp.fixed_nr_of_samples_per_ray == 16
    eq(N(imp.samples_z), eimp.z, "importance z"); eq(N(imp.samples_pos), eimp.pos, "importance pos")
    rimp = ref_golden.once(lambda: ref_gpu.vr_importance_sample(o, d, to_ref(rsp), cdf, 16, jitter, st, inc))
    ref_golden.equal(key + "z", imp.samples_z, lambda: rimp().z)
    ref_golden.equal(key + "pos", imp.samples_pos, lambda: rimp().pos)
    sdf_imp = (imp.samples_pos.norm(dim=1, keepdim=True) - scenes.OBJECT_RADIUS).contiguous()
    imp.set_sdf(sdf_imp)
    eimp.sdf, eimp.has_sdf = N(sdf_imp), True
    comb = VR.combine_uniform_samples_with_imp(o, d, tx, rsp, imp)
    ecomb = orc.vr_combine(N(o), N(d), N(tx), p, eimp)
    se = N(comb.ray_start_end_idx)
    assert np.array_equal(se, ecomb.start_end)
    assert int(comb.cur_nr_samples.item()) == ecomb.cur
    n = ecomb.cur
    for a, b, nm in [(comb.samples_z, ecomb.z, "z"), (comb.samples_dt, ecomb.dt, "dt"), (comb.samples_pos, ecomb.pos, "pos"),
                     (comb.samples_sdf, ecomb.sdf, "sdf"), (comb.samples_dirs, ecomb.dirs, "dirs")]:
        eq(N(a)[:n], b[:n], "combined " + nm)
    eq(N(comb.ray_fixed_dt), ecomb.fixed_dt, "combined fixed_dt")
    zz = N(comb.samples_z)
    for s, e in se:
        assert np.all(np.diff(zz[s:e, 0]) >= 0), "merged samples must be sorted by z"
    cc = comb.compact_to_valid_samples()
    assert cc.samples_pos.shape[0] == n and cc.has_sdf
    def ref_combine():
        r = rimp()
        r.sdf, r.has_sdf = sdf_imp, True
        return ref_gpu.vr_combine(o, d, tx, to_ref(rsp), r)
    rcomb = ref_golden.once(ref_combine)
    ref_golden.equal(key + "combined.counts", ref_golden.counts(se), lambda: ref_golden.counts(rcomb().start_end))
    ours = ref_golden.per_ray(se, comb.samples_z, comb.samples_dt, comb.samples_pos, comb.samples_sdf)
    for i, nm in enumerate(("z", "dt", "pos", "sdf")):
        ref_golden.equal(key + "combined." + nm, ours[i],
                         lambda i=i: ref_golden.per_ray(rcomb().start_end, rcomb().z, rcomb().dt, rcomb().pos, rcomb().sdf)[i])
    rsp.remove_sdf()


@pytest.mark.parametrize("jitter,mult", [(False, 1.0), (True, 2.0)])
def test_importance_round_equals_separate_calls(packed, jitter, mult):
    """the fused importance-sampling round (one launch) reproduces the chain of separate kernels + PyTorch glue bit for bit,
    including the jitter stream of the class-static generator"""
    import permuto_sdf_b200.train as tr
    from permuto_sdf import VolumeRendering
    rsp, o, d = packed["rsp"], packed["o"], packed["d"]
    torch.manual_seed(4)
    sdf = (rsp.samples_pos.norm(dim=1, keepdim=True) - 0.3 + 0.01 * torch.randn(rsp.samples_pos.shape[0], 1, device="cuda")).contiguous()
    state = (VolumeRendering.m_rng.state, VolumeRendering.m_rng.inc)
    out = {}
    for fused in (False, True):
        VolumeRendering.m_rng.state, VolumeRendering.m_rng.inc = state
        tr.FUSED_IMPORTANCE_ROUND = fused
        imp = tr._imp_round(rsp, sdf, 512, mult, o, d, 16, jitter)
        out[fused] = (imp.samples_z.clone(), imp.samples_pos.clone(), imp.samples_dirs.clone(), VolumeRendering.m_rng.state)
    tr.FUSED_IMPORTANCE_ROUND = True
    assert out[True][3] == out[False][3]
    for a, b, name in zip(out[True][:3], out[False][:3], ("z", "pos", "dirs")):
        assert torch.equal(a, b), name
    assert float(out[True][0].max()) > 0
