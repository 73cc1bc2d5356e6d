"""Ray-path parity at the sizes bench.py runs (VERDICT r1: the other ray-path tests use V = 128 / 64 samples): 256^3 occupancy grid,
512 rays, 96 grid samples per ray at min distance 1e-4, then the two importance-sampling rounds with 16 samples each (128 samples per
ray in total), jitter off and on. Ours (through the `permuto_sdf` mirror / C ABI) against the reference's own kernels compiled for
sm_100a (oracle/_ref/libpsdf_ref_gpu.so where built, their stored outputs elsewhere: tests/ref_golden.py) and, for the grid samples,
against the C oracle: per-ray sample counts, z, dt and positions must be bit-identical."""
import numpy as np
import pytest
import torch

import ref_golden
import scenes
from oracle import rayops as orc
from oracle import ref_gpu

pytestmark = pytest.mark.gpu
_fresh_generators = pytest.fixture(autouse=True)(ref_golden.fresh_generators)
V, R, MAX_PER_RAY, NR_IMP, MIN_DIST = 256, 512, 96, 16, 1e-4


def T(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def N(t):
    return t.detach().cpu().numpy()


@pytest.fixture(scope="module")
def scene(cuda):
    from permuto_sdf import OccupancyGrid, Sphere
    o, d = scenes.make_rays(R, seed=5, miss_fraction=0.05)
    values, occ = scenes.analytic_occupancy(V)
    grid = OccupancyGrid(V, 1.0, [0, 0, 0])
    grid.set_grid_values(T(values))
    grid.set_grid_occupancy(T(occ.astype(np.uint8)).bool())
    return dict(o=o, d=d, occ=occ.astype(np.uint8), grid=grid, sphere=Sphere(scenes.SPHERE_RADIUS, [0, 0, 0]))


def _per_ray_equal(se_a, arrs_a, se_b, arrs_b, what):
    assert np.array_equal(se_a[:, 1] - se_a[:, 0], se_b[:, 1] - se_b[:, 0]), what + ": per-ray sample counts differ"
    for (s, e), (rs, re) in zip(se_a, se_b):
        for a, b in zip(arrs_a, arrs_b):
            assert np.array_equal(a[s:e], b[rs:re]), what + ": samples not bit-identical"


def _per_ray_equal_ref(key, ours, theirs):
    """ours: packed container; theirs: callable -> the reference's packed container"""
    ref_golden.equal(key + ".counts", ref_golden.counts(ours.ray_start_end_idx), lambda: ref_golden.counts(theirs().start_end))
    arrs = ref_golden.per_ray(ours.ray_start_end_idx, ours.samples_z, ours.samples_dt, ours.samples_pos)
    for i, nm in enumerate(("z", "dt", "pos")):
        ref_golden.equal(key + "." + nm, arrs[i], lambda i=i: ref_golden.per_ray(theirs().start_end, theirs().z, theirs().dt, theirs().pos)[i])


@pytest.mark.parametrize("jitter", [False, True])
def test_grid_sampling_and_importance_rounds_at_bench_size(scene, jitter):
    from permuto_sdf import OccupancyGrid, VolumeRendering
    o, d = T(scene["o"]), T(scene["d"])
    _, te, _, tx, _ = scene["sphere"].ray_intersection(o, d)
    st, inc = OccupancyGrid.m_rng.state, OccupancyGrid.m_rng.inc
    uni = scene["grid"].compute_samples_in_occupied_regions(o, d, te, tx, MIN_DIST, MAX_PER_RAY, jitter)
    se = N(uni.ray_start_end_idx)
    assert (se[:, 1] - se[:, 0]).max() == MAX_PER_RAY, "the bench scene fills the per-ray budget"
    # (a) the C oracle
    exp = orc.occ_samples_in_occupied_regions(V, 1.0, [0, 0, 0], scene["o"], scene["d"], N(te), N(tx), scene["occ"], MIN_DIST, MAX_PER_RAY, jitter, st, inc)
    _per_ray_equal(se, [N(uni.samples_z), N(uni.samples_dt), N(uni.samples_pos)], exp.start_end, [exp.z, exp.dt, exp.pos], "grid samples vs C oracle")
    # (b) the reference kernel
    key = "benchsize.j%d" % jitter
    ref = ref_golden.once(lambda: ref_gpu.occ_samples_in_occupied_regions(V, 1.0, [0, 0, 0], o, d, te, tx, scene["grid"].get_grid_occupancy(),
                                                                         MIN_DIST, MAX_PER_RAY, jitter, st, inc))
    _per_ray_equal_ref(key + ".grid_samples", uni, ref)
    # importance sampling on the analytic SDF (identical sdf values on both sides), two rounds like sdf_utils.py:383-423
    ours = uni.compact_to_valid_samples()
    theirs = ref_golden.once(lambda: ref().compact())

    def sdf_of(pos):
        return (torch.sqrt((pos * pos).sum(1, keepdim=True)) - scenes.OBJECT_RADIUS).contiguous()

    for rnd, mult in enumerate((1.0, 2.0)):
        so = sdf_of(ours.samples_pos)
        ours.set_sdf(so)
        st, inc = VolumeRendering.m_rng.state, VolumeRendering.m_rng.inc
        # ours: the fused round (one launch) ...
        imp_o = VolumeRendering.importance_round(o, d, ours, so, 512.0, True, mult, NR_IMP, jitter)

        # ... theirs: the chain of reference kernels
        def ref_round(prev=theirs, mult=mult, st=st, inc=inc):
            p = prev()
            sr = sdf_of(p.pos)
            p.sdf, p.has_sdf = sr, True
            a = ref_gpu.vr_sdf2alpha(p, sr, 512.0, True, mult).clip(0.0, 1.0)
            Tr, _ = ref_gpu.vr_cumprod(p, 1 - a + 1e-7)
            w = a * Tr
            _, wsum = ref_gpu.vr_sum(p, w)
            w = w / torch.clamp(wsum, min=1e-6)
            cdf = ref_gpu.vr_cdf(p, w)
            imp_r = ref_gpu.vr_importance_sample(o, d, p, cdf, NR_IMP, jitter, st, inc)
            imp_r.sdf, imp_r.has_sdf = sdf_of(imp_r.pos), True
            return imp_r, ref_gpu.vr_combine(o, d, tx, p, imp_r).compact()
        ref_r = ref_golden.once(ref_round)
        ref_golden.equal("%s.round%d.importance_z" % (key, rnd), imp_o.samples_z, lambda: ref_r()[0].z)
        imp_o.set_sdf(sdf_of(imp_o.samples_pos))
        ours = VolumeRendering.combine_uniform_samples_with_imp(o, d, tx, ours, imp_o).compact_to_valid_samples()
        theirs = ref_golden.once(lambda ref_r=ref_r: ref_r()[1])
        _per_ray_equal_ref("%s.round%d.merged" % (key, rnd), ours, theirs)
    n = N(ours.ray_start_end_idx)
    assert (n[:, 1] - n[:, 0]).max() == MAX_PER_RAY + 2 * NR_IMP, "128 samples per ray, the bench configuration"
