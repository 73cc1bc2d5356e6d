"""GPU parity tests of the ray-path kernels (through the C ABI / the `permuto_sdf` mirror) against
 (a) the C oracle (oracle/rayops_oracle.c) and
 (b) the reference's own CUDA kernels compiled for sm_100a (oracle/_ref/libpsdf_ref_gpu.so) where built, their stored outputs
     elsewhere (tests/ref_golden.py).
Integer / index results must match bit for bit; float results within the tolerance written in each test
(north star: <= 1e-3 relative; we hold the ray path to <= 1e-6 absolute and report bit-exact fractions)."""
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
FTOL = 2e-6


def T(a, dtype=None):
    t = torch.from_numpy(np.ascontiguousarray(a)).cuda()
    return t if dtype is None else t.to(dtype)


def N(t):
    return t.detach().cpu().numpy()


@pytest.fixture(scope="module")
def scene(cuda):
    from permuto_sdf import OccupancyGrid, Sphere
    o, d = scenes.make_rays(512, seed=3)
    values, occ = scenes.analytic_occupancy(V)
    grid = OccupancyGrid(V, 1.0, [0, 0, 0])
    grid.set_grid_values(T(values))
    grid.set_grid_occupancy(T(occ.astype(np.uint8)).bool())
    sph = Sphere(scenes.SPHERE_RADIUS, [0, 0, 0])
    return dict(o=o, d=d, values=values, occ=occ.astype(np.uint8), grid=grid, sphere=sph)


def close(a, b, tol=FTOL, what=""):
    a, b = np.asarray(a, np.float64), np.asarray(b, np.float64)
    assert a.shape == b.shape, (what, a.shape, b.shape)
    err = np.abs(a - b).max() if a.size else 0.0
    assert err <= tol, "%s: max abs err %g > %g" % (what, err, tol)


# --------------------------------------------------------------------------------------------------- Sphere
def test_sphere_ray_intersection(scene):
    o, d = scene["o"], scene["d"]
    got = scene["sphere"].ray_intersection(T(o), T(d))
    exp = orc.sphere_ray_intersection(scenes.SPHERE_RADIUS, [0, 0, 0], o, d)
    assert np.array_equal(N(got[4]), exp[4])
    for g, e, name in zip(got[:4], exp[:4], ["pts_entry", "t_entry", "pts_exit", "t_exit"]):
        assert np.array_equal(N(g), e), name + " not bit-exact vs oracle"
    ref = ref_golden.once(lambda: ref_gpu.sphere_ray_intersection(scenes.SPHERE_RADIUS, [0, 0, 0], T(o), T(d)))
    for i, (g, name) in enumerate(zip(got, ["pts_entry", "t_entry", "pts_exit", "t_exit", "hit"])):
        ref_golden.equal("rayops.sphere." + name, g, lambda i=i: ref()[i])


def test_sphere_points(scene):
    sph = scene["sphere"]
    torch.manual_seed(0)
    pts = sph.rand_points_inside(4096)
    assert bool(sph.check_point_inside_primitive(pts).all())
    phi = torch.rand(1000, device="cuda") * 6.28; ct = torch.rand(1000, device="cuda") * 2 - 1; u = torch.rand(1000, device="cuda")
    from permuto_sdf_b200 import call
    out = torch.empty(1000, 3, device="cuda")
    call("psdf_sphere_rand_points_inside", 1000, 0.5, phi, ct, u, out)
    close(N(out), orc.sphere_rand_points_inside(0.5, N(phi), N(ct), N(u)), 1e-6, "rand_points_inside")
    ref_golden.close("rayops.rand_points_inside", out, lambda: ref_gpu.sphere_rand_points_inside(0.5, [0, 0, 0], phi, ct, u), 1e-6)


# --------------------------------------------------------------------------------------------------- Occupancy grid
@pytest.mark.parametrize("randomize", [False, True])
def test_grid_points(scene, randomize):
    from permuto_sdf import OccupancyGrid
    g = scene["grid"]
    st, inc = OccupancyGrid.m_rng.state, OccupancyGrid.m_rng.inc
    pts = g.compute_grid_points(randomize)
    exp = orc.occ_grid_points(V, 1.0, [0, 0, 0], None, randomize, st, inc)
    assert np.array_equal(N(pts), exp)
    ref_golden.equal("rayops.grid_points.r%d" % randomize, pts, lambda: ref_gpu.occ_grid_points(V, 1.0, [0, 0, 0], None, randomize, st, inc))
    torch.manual_seed(5)
    st = OccupancyGrid.m_rng.state
    p2, idx = g.compute_random_sample_of_grid_points(5000, randomize)
    assert idx.dtype == torch.int32 and int(idx.max()) < V ** 3
    exp2 = orc.occ_grid_points(V, 1.0, [0, 0, 0], N(idx), randomize, st, inc)
    assert np.array_equal(N(p2), exp2)
    ref_golden.equal("rayops.grid_points_subset.r%d" % randomize, p2, lambda: ref_gpu.occ_grid_points(V, 1.0, [0, 0, 0], idx, randomize, st, inc))


def test_grid_updates_and_lookup(scene):
    from permuto_sdf import OccupancyGrid
    rng = np.random.RandomState(0)
    g = OccupancyGrid(V, 1.0, [0, 0, 0])
    pts = g.compute_grid_points(False)
    sdf = T(scenes.analytic_sdf(N(pts)))          # same float32 sdf values as the oracle scene
    g.update_with_sdf(sdf, 512.0, 1e10, 1e-4)
    assert np.array_equal(N(g.get_grid_occupancy()).astype(np.uint8), scene["occ"]), "occupancy bits differ from oracle"
    assert np.array_equal(N(g.get_grid_values()), scene["values"])
    def ref_occupancy():
        rv, ro = torch.ones(V ** 3, device="cuda"), torch.ones(V ** 3, dtype=torch.bool, device="cuda")
        ref_gpu.occ_update_with_sdf(V, 1.0, sdf, None, 512.0, 1e-4, rv, ro)
        return ro
    ref_golden.equal("rayops.update_with_sdf.occupancy", g.get_grid_occupancy(), ref_occupancy)
    # random-sample sdf update (1.0 half diagonals, inv_s from a tensor)
    idx = torch.from_numpy(rng.permutation(V ** 3)[:20000].astype(np.int32)).cuda()
    s2 = torch.from_numpy(rng.uniform(-0.05, 0.05, (20000, 1)).astype(np.float32)).cuda()
    v0, o0 = N(g.get_grid_values()).copy(), N(g.get_grid_occupancy()).astype(np.uint8)
    g.update_with_sdf_random_sample(idx, s2, torch.tensor([300.0], device="cuda"), 1e-4)
    ev, eo = orc.occ_update_with_sdf(N(s2), N(idx), 1.0, V, 300.0, 1e-4, 1, v0, o0)
    assert np.array_equal(N(g.get_grid_values()), ev)
    mism = int((N(g.get_grid_occupancy()) != eo).sum())
    assert mism <= 2, "occupancy bits differ (expf ulp effects allowed on <=2 voxels): %d" % mism
    # density updates
    g2 = OccupancyGrid(V, 1.0, [0, 0, 0])
    dens = torch.from_numpy(rng.rand(V ** 3, 1).astype(np.float32) * 2).cuda()
    g2.update_with_density(dens, 0.9, 1.2)
    ev, eo = orc.occ_update_with_density(N(dens), None, 0.9, 1.2, np.ones(V ** 3, np.float32), np.ones(V ** 3, np.uint8))
    assert np.array_equal(N(g2.get_grid_values()), ev) and np.array_equal(N(g2.get_grid_occupancy()), eo)
    d3 = torch.from_numpy(rng.rand(20000, 1).astype(np.float32) * 3).cuda()
    g2.update_with_density_random_sample(idx, d3, 0.5, 1.0)
    ev2, eo2 = orc.occ_update_with_density(N(d3), N(idx), 0.5, 1.0, ev, eo)
    assert np.array_equal(N(g2.get_grid_values()), ev2) and np.array_equal(N(g2.get_grid_occupancy()), eo2)
    # lookup, including points outside the grid
    q = torch.from_numpy(rng.uniform(-0.7, 0.7, (50000, 3)).astype(np.float32)).cuda()
    got = scene["grid"].check_occupancy(q)
    assert np.array_equal(N(got), orc.occ_check_occupancy(V, 1.0, [0, 0, 0], scene["occ"], N(q)))
    ref_golden.equal("rayops.check_occupancy", got, lambda: ref_gpu.occ_check_occupancy(V, 1.0, [0, 0, 0], scene["grid"].get_grid_occupancy(), q))


def per_ray(pk_start_end, arrs):
    """canonical per-ray view of packed arrays: list over rays of tuples of numpy slices"""
    out = []
    for s, e in pk_start_end:
        out.append(tuple(a[s:e] for a in arrs))
    return out


@pytest.mark.parametrize("jitter", [False, True])
def test_samples_in_occupied_regions(scene, jitter):
    from permuto_sdf import OccupancyGrid
    o, d = scene["o"], scene["d"]
    pe, te, px, tx, hit = scene["sphere"].ray_intersection(T(o), T(d))
    st, inc = OccupancyGrid.m_rng.state, OccupancyGrid.m_rng.inc
    rsp = scene["grid"].compute_samples_in_occupied_regions(T(o), T(d), te, tx, 1e-3, 64, jitter)
    exp = orc.occ_samples_in_occupied_regions(V, 1.0, [0, 0, 0], o, d, N(te), N(tx), scene["occ"], 1e-3, 64, jitter, st, inc)
    se = N(rsp.ray_start_end_idx)
    assert np.array_equal(se, exp.start_end), "ray_start_end_idx differs from the oracle"
    assert int(rsp.cur_nr_samples.item()) == exp.cur
    assert (se[:, 1] - se[:, 0]).max() > 30, "scene should produce real samples"
    assert np.array_equal(N(rsp.ray_fixed_dt), exp.fixed_dt)
    for a, b, name in [(rsp.samples_z, exp.z, "z"), (rsp.samples_dt, exp.dt, "dt"), (rsp.samples_pos, exp.pos, "pos"),
                       (rsp.samples_dirs, exp.dirs, "dirs")]:
        ga = N(a)
        for (s, e) in se:
            assert np.array_equal(ga[s:e], b[s:e]), name + " not bit exact vs oracle"
    # compaction
    comp = rsp.compact_to_valid_samples()
    ecomp = orc.packed_compact(exp)
    assert comp.samples_pos.shape[0] == ecomp.cur == comp.compute_exact_nr_samples()
    assert np.array_equal(N(comp.ray_start_end_idx), ecomp.start_end)
    for a, b in [(comp.samples_z, ecomp.z), (comp.samples_dt, ecomp.dt), (comp.samples_pos, ecomp.pos), (comp.samples_dirs, ecomp.dirs),
                 (comp.ray_fixed_dt, ecomp.fixed_dt)]:
        assert np.array_equal(N(a), b)
    idx = comp.compute_per_sample_ray_idx(comp.ray_start_end_idx, comp.samples_pos.shape[0])
    assert np.array_equal(N(idx), orc.packed_per_sample_ray_idx(ecomp.start_end, ecomp.cur))
    ref = ref_golden.once(lambda: ref_gpu.occ_samples_in_occupied_regions(V, 1.0, [0, 0, 0], T(o), T(d), te, tx, scene["grid"].get_grid_occupancy(),
                                                                         1e-3, 64, jitter, st, inc))
    key = "rayops.occ_samples.j%d." % jitter
    ref_golden.equal(key + "counts", ref_golden.counts(se), lambda: ref_golden.counts(ref().start_end))
    ref_golden.equal(key + "fixed_dt", rsp.ray_fixed_dt, lambda: ref().fixed_dt)
    ours = ref_golden.per_ray(se, rsp.samples_z, rsp.samples_dt, rsp.samples_pos)
    for i, name in enumerate(("z", "dt", "pos")):
        ref_golden.equal(key + name, ours[i], lambda i=i: ref_golden.per_ray(ref().start_end, ref().z, ref().dt, ref().pos)[i])


def test_first_sample_and_advance(scene):
    o, d = scene["o"], scene["d"]
    pe, te, px, tx, hit = scene["sphere"].ray_intersection(T(o), T(d))
    rsp = scene["grid"].compute_first_sample_start_of_occupied_regions(T(o), T(d), te, tx)
    exp = orc.occ_first_sample_start(V, 1.0, [0, 0, 0], o, d, N(te), N(tx), scene["occ"])
    se = N(rsp.ray_start_end_idx)
    assert np.array_equal(se, exp.start_end)
    for (s, e) in se:
        assert np.array_equal(N(rsp.samples_pos)[s:e], exp.pos[s:e]) and np.array_equal(N(rsp.samples_z)[s:e], exp.z[s:e])
    ref = ref_golden.once(lambda: ref_gpu.occ_first_sample_start(V, 1.0, [0, 0, 0], T(o), T(d), te, tx, scene["grid"].get_grid_occupancy()))
    ref_golden.equal("rayops.first_sample.counts", ref_golden.counts(se), lambda: ref_golden.counts(ref().start_end))
    ref_golden.equal("rayops.first_sample.pos", ref_golden.per_ray(se, rsp.samples_pos)[0], lambda: ref_golden.per_ray(ref().start_end, ref().pos)[0])
    comp = rsp.compact_to_valid_samples()
    pos = comp.samples_pos + comp.samples_dirs * (0.5 / V)
    # move some points into empty space (towards the centre of the object, which is unoccupied inside)
    pos = (pos * 0.2).contiguous()
    expect_pos, expect_within = orc.occ_advance_to_next_occupied(V, 1.0, [0, 0, 0], N(comp.samples_dirs), N(pos), scene["occ"])
    pos_in = pos.clone()                                # ours moves pos in place
    ref = ref_golden.once(lambda: ref_gpu.occ_advance_to_next_occupied(V, 1.0, [0, 0, 0], comp.samples_dirs, pos_in,
                                                                      scene["grid"].get_grid_occupancy()))
    newpos, within = scene["grid"].advance_sample_to_next_occupied_voxel(comp.samples_dirs, pos)
    assert newpos.data_ptr() == pos.data_ptr(), "output must alias the input like the reference"
    assert np.array_equal(N(within), expect_within) and np.array_equal(N(newpos), expect_pos)
    ref_golden.equal("rayops.advance.within", within, lambda: ref()[1])
    ref_golden.equal("rayops.advance.pos", newpos, lambda: ref()[0])


# --------------------------------------------------------------------------------------------------- RaySampler
@pytest.mark.parametrize("jitter", [False, True])
def test_sampler_fg_bg(scene, jitter):
    from permuto_sdf import RaySampler
    o, d = scene["o"], scene["d"]
    pe, te, px, tx, hit = scene["sphere"].ray_intersection(T(o), T(d))
    st, inc = RaySampler.m_rng.state, RaySampler.m_rng.inc
    fg = RaySampler.compute_samples_fg(T(o), T(d), te, tx, 0.01, 48, 0.5, torch.zeros(3, device="cuda"), jitter)
    exp = orc.sampler_fg(o, d, N(te), N(tx), 0.01, 48, jitter, st, inc)
    se = N(fg.ray_start_end_idx)
    assert np.array_equal(se, exp.start_end)
    for (s, e) in se:
        assert np.array_equal(N(fg.samples_z)[s:e], exp.z[s:e]) and np.array_equal(N(fg.samples_pos)[s:e], exp.pos[s:e])
        assert np.array_equal(N(fg.samples_dt)[s:e], exp.dt[s:e])
    ref = ref_golden.once(lambda: ref_gpu.sampler_fg(T(o), T(d), te, tx, 0.5, [0, 0, 0], 0.01, 48, jitter, st, inc))
    ref_golden.equal("rayops.sampler_fg.j%d.counts" % jitter, ref_golden.counts(se), lambda: ref_golden.counts(ref().start_end))
    ref_golden.equal("rayops.sampler_fg.j%d.z" % jitter, ref_golden.per_ray(se, fg.samples_z)[0], lambda: ref_golden.per_ray(ref().start_end, ref().z)[0])
    st, inc = RaySampler.m_rng.state, RaySampler.m_rng.inc
    bg = RaySampler.compute_samples_bg(T(o), T(d), tx, 32, 0.5, [0.0, 0.0, 0.0], jitter, False)
    eb = orc.sampler_bg(o, d, N(tx), 32, 0.5, [0, 0, 0], jitter, False, st, inc)
    assert bg.rays_have_equal_nr_of_samples and bg.fixed_nr_of_samples_per_ray == 32
    assert np.array_equal(N(bg.ray_start_end_idx), eb.start_end)
    hitm = N(hit).reshape(-1)
    sel = np.repeat(hitm, 32)
    close(N(bg.samples_z)[sel], eb.z[sel], 1e-3, "bg z")        # z = t_exit / t can be ~1e3: relative 1e-6
    assert np.allclose(N(bg.samples_z)[sel], eb.z[sel], rtol=2e-6, atol=1e-6)
    assert np.allclose(N(bg.samples_pos_4d)[sel], eb.pos4[sel], rtol=2e-5, atol=2e-6)
    rb = ref_golden.once(lambda: ref_gpu.sampler_bg(T(o), T(d), tx, 32, 0.5, [0, 0, 0], jitter, False, st, inc))
    key = "rayops.sampler_bg.j%d." % jitter
    ref_golden.close(key + "z", N(bg.samples_z)[sel], lambda: N(rb().z)[sel], 1e-6, 2e-6)
    ref_golden.close(key + "pos4", N(bg.samples_pos_4d)[sel], lambda: N(rb().pos4)[sel], 2e-6, 2e-5)
    ref_golden.close(key + "dt", N(bg.samples_dt)[sel], lambda: N(rb().dt)[sel], 1e-5, 1e-4)


# --------------------------------------------------------------------------------------------------- statics
@pytest.mark.parametrize("degree", [1, 2, 3, 4, 5, 6, 7])
def test_spherical_harmonics(cuda, degree):
    from permuto_sdf import PermutoSDF
    rng = np.random.RandomState(degree)
    d = rng.randn(3001, 3).astype(np.float32)
    d /= np.linalg.norm(d, axis=1, keepdims=True)
    got = PermutoSDF.spherical_harmonics(T(d), degree)
    assert got.shape == (3001, degree * degree)
    close(N(got), orc.spherical_harmonics(d, degree), 2e-6, "SH vs oracle")
    ref_golden.close("rayops.sh.deg%d" % degree, got, lambda: ref_gpu.spherical_harmonics(T(d), degree), 2e-6)


def test_random_rays_from_reel(cuda):
    from permuto_sdf import PermutoSDF

    class Reel:
        pass
    rgb, mask, K, tf = scenes.synthetic_reel()
    reel = Reel()
    reel.rgb_reel, reel.mask_reel, reel.K_reel, reel.tf_world_cam_reel = T(rgb), T(mask), T(K), T(tf)
    torch.manual_seed(11)
    o, d, gt, gm, img = PermutoSDF.random_rays_from_reel(reel, 2000)
    assert o.shape == (2000, 3) and gm.shape == (2000, 1) and img.dtype == torch.int32
    torch.manual_seed(11)
    pix = torch.randint(0, rgb.shape[2] * rgb.shape[3], (2000,), dtype=torch.int32, device="cuda")
    img2 = torch.randint(0, rgb.shape[0], (2000,), dtype=torch.int32, device="cuda")
    assert torch.equal(img, img2)
    eo, ed, egt, egm = orc.random_rays_from_reel(rgb, mask, K, tf, N(pix), N(img))
    close(N(o), eo, 0, "origins"); close(N(d), ed, 1e-6, "dirs"); close(N(gt), egt, 0, "gt rgb"); close(N(gm), egm, 0, "mask")
    ref = ref_golden.once(lambda: ref_gpu.random_rays_from_reel(T(rgb), T(mask), T(K), T(tf), pix, img))
    ref_golden.close("rayops.reel.dirs", d, lambda: ref()[1], 1e-6)
    for i, (g, name) in enumerate(((o, "origins"), (gt, "gt"), (gm, "mask"))):
        ref_golden.equal("rayops.reel." + name, g, lambda i=i: ref()[(0, 2, 3)[i]])
