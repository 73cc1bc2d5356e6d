"""GPU tests of the tcgen05 path: the raw tensor-core GEMM self test (descriptor / layout check) and the fused
encoding+MLP SDF kernel against (a) the CPU oracle and (b) the unfused differentiable model. Tolerance: the
north star's 1e-3 relative; the bf16x2 split keeps it ~1e-5."""
import numpy as np
import pytest
import torch

from oracle import encoding_oracle as eo

pytestmark = pytest.mark.gpu


def rel(a, b):
    a, b = a.detach().cpu().double(), b.detach().cpu().double()
    return float((a - b).abs().max() / (b.abs().max() + 1e-30))


def _probe_call(name, *args):
    """tcgen05 self tests live in the probe library (tests/probe/libumma_probe.so, test infrastructure), not in the product ABI"""
    import ctypes
    import os
    so = os.path.join(os.path.dirname(os.path.abspath(__file__)), "probe", "libumma_probe.so")
    lib = ctypes.CDLL(so)
    conv = [a.data_ptr() if isinstance(a, torch.Tensor) else int(a) for a in args] + [torch.cuda.current_stream().cuda_stream]
    fn = getattr(lib, name)
    fn.argtypes = [ctypes.c_int if isinstance(a, int) else ctypes.c_void_p for a in args] + [ctypes.c_void_p]
    rc = fn(*conv)
    assert rc == 0, "%s failed with %d" % (name, rc)


def _gemm_err(N, K):
    from permuto_sdf_b200 import call
    torch.manual_seed(N * 100 + K)
    A = torch.randn(128, K, device="cuda")
    B = torch.randn(N, K, device="cuda")
    D = torch.zeros(128, N, device="cuda")
    _probe_call("umma_probe_gemm", N, K, A, B, D)
    torch.cuda.synchronize()
    return rel(D, A.double() @ B.double().t())


@pytest.mark.parametrize("N,K", [(64, 64), (48, 64), (64, 48), (16, 16), (33, 36), (64, 63)])
def test_umma_gemm_self_test(cuda, N, K):
    from permuto_sdf_b200 import call
    torch.manual_seed(N * 100 + K)
    A = torch.randn(128, K, device="cuda")
    B = torch.randn(N, K, device="cuda")
    D = torch.zeros(128, N, device="cuda")
    _probe_call("umma_probe_gemm", N, K, A, B, D)
    torch.cuda.synchronize()
    ref = (A.double() @ B.double().t())
    err = rel(D, ref)
    assert err < 5e-5, "tensor-core GEMM mismatch (rel err %g): descriptor/layout problem" % err


@pytest.mark.parametrize("L,hidden,N", [(16, 64, 5000), (8, 32, 1000), (24, 32, 777), (4, 64, 128)])
def test_fused_sdf_matches_oracle_and_model(cuda, L, hidden, N):
    from permuto_sdf import Sphere
    from permuto_sdf_b200.fused import FusedSDF
    from permuto_sdf_b200.models import SDF
    torch.manual_seed(L)
    m = SDF(3, Sphere(0.5, [0, 0, 0]), 32, 10000, nr_levels=L, capacity=2 ** 16, hidden=hidden).to("cuda")
    with torch.no_grad():
        m.encoding.lattice_values.normal_(0, 0.3)          # non-trivial features
    f = FusedSDF(m)
    pos = ((torch.rand(N, 3) - 0.5) * 0.9)
    it = 3000
    sdf, grad, geom = f(pos.cuda(), it, with_gradient=True)
    sdf_v, none_g, geom_v = f(pos.cuda(), it, with_gradient=False)
    assert none_g is None and torch.equal(sdf, sdf_v) or rel(sdf_v, sdf) < 1e-6
    # (b) unfused differentiable model
    s1, g1, f1 = m.get_sdf_and_gradient(pos.cuda().clone(), it)
    assert rel(sdf, s1) < 1e-3 and rel(grad, g1) < 1e-3 and rel(geom, f1) < 1e-3
    # (a) CPU oracle
    enc = m.encoding
    lin = [l for l in m.mlp_sdf if isinstance(l, torch.nn.Linear)]
    W = [l.weight.detach().cpu() for l in lin]; Bs = [l.bias.detach().cpu() for l in lin]
    window = eo.coarse2fine(L, 0.3 + 0.7 * it / 10000)
    s0, g0, f0 = eo.sdf_and_gradient(pos, enc.lattice_values.detach().cpu(), enc.scale_factor.cpu(), enc.random_shift_per_level.detach().cpu(),
                                     window, W, Bs, True, 1e-3)
    e = (rel(sdf, s0), rel(grad, g0), rel(geom, f0))
    assert max(e) < 1e-3, e
    # the blob follows weight updates
    with torch.no_grad():
        lin[3].bias += 0.25
    s2, _, _ = f(pos.cuda(), it)
    assert rel(s2, s0 + 0.25) < 1e-3


@pytest.mark.parametrize("L,hidden,N", [(16, 64, 3000), (8, 32, 500), (24, 32, 129), (16, 64, 65536)])
def test_fused_training_gradients_match_autograd(cuda, L, hidden, N):
    """parameter gradients of a loss on (sdf, d sdf/dx, geom): fused forward+backward kernels vs autograd through the
    modular path (encoding double backward + torch MLP). North-star tolerance 1e-3 relative."""
    from permuto_sdf import Sphere
    from permuto_sdf_b200.models import SDF
    torch.manual_seed(L + N)
    m = SDF(3, Sphere(0.5, [0, 0, 0]), 32, 10000, nr_levels=L, capacity=2 ** 16, hidden=hidden).to("cuda")
    with torch.no_grad():
        m.encoding.lattice_values.normal_(0, 0.3)
    pos = ((torch.rand(N, 3, device="cuda") - 0.5) * 0.9)
    tgt = torch.randn(N, 3, device="cuda")
    wgeom = torch.randn(32, device="cuda")

    def loss_fn(sdf, grad, geom):
        return ((grad.norm(dim=-1) - 1.0) ** 2).mean() + (sdf ** 2).mean() + (grad * tgt).sum(-1).mean() + (torch.tanh(geom) * wgeom).mean()

    params = [m.encoding.lattice_values] + [p for l in m.mlp_sdf if isinstance(l, torch.nn.Linear) for p in (l.weight, l.bias)]
    it = 4000
    sdf0, grad0, geom0 = m.get_sdf_and_gradient(pos.clone(), it)
    l0 = loss_fn(sdf0, grad0, geom0)
    g0 = torch.autograd.grad(l0, params)
    m.enable_fused_training()
    assert m.fused_training
    sdf1, grad1, geom1 = m.get_sdf_and_gradient(pos.clone(), it)
    l1 = loss_fn(sdf1, grad1, geom1)
    g1 = torch.autograd.grad(l1, params)
    assert rel(sdf1, sdf0) < 1e-3 and rel(grad1, grad0) < 1e-3 and rel(geom1, geom0) < 1e-3
    assert abs(float(l1) - float(l0)) < 1e-3 * abs(float(l0))
    names = ["lattice", "W0", "b0", "W1", "b1", "W2", "b2", "W3", "b3"]
    errs = {n: rel(a, b) for n, a, b in zip(names, g1, g0)}
    assert max(errs.values()) < 1e-3, errs
    # a second call accumulates into .grad like any autograd op
    m.zero_grad()
    loss_fn(*m.get_sdf_and_gradient(pos.clone(), it)).backward()
    assert rel(m.encoding.lattice_values.grad, g0[0]) < 1e-3


def test_fused_sdf_large_and_ragged(cuda):
    from permuto_sdf import Sphere
    from permuto_sdf_b200.fused import FusedSDF
    from permuto_sdf_b200.models import SDF
    torch.manual_seed(0)
    m = SDF(3, Sphere(0.5, [0, 0, 0]), 32, 1, nr_levels=16, capacity=2 ** 18, hidden=64).to("cuda")
    f = FusedSDF(m)
    for N in (0, 1, 127, 129, 65536 + 5):
        pos = (torch.rand(N, 3, device="cuda") - 0.5)
        sdf, grad, geom = f(pos, 10, with_gradient=True)
        assert sdf.shape == (N, 1) and grad.shape == (N, 3) and geom.shape == (N, 32)
        if N:
            s1, g1, f1 = m.get_sdf_and_gradient(pos.clone(), 10)
            assert rel(sdf, s1) < 1e-3 and rel(grad, g1) < 1e-3 and rel(geom, f1) < 1e-3


@pytest.mark.parametrize("M,N", [(64, 64), (64, 48), (16, 64), (48, 16)])
def test_umma_transposed_gemm_weight_gradient_layout(cuda, M, N):
    """dW-style product D = A^T B with the sample axis as the MMA K dimension (MN-major operands straight from activation tiles).
    The kernel dumps every TMEM lane; the test also reports where the M = 64 accumulator rows live."""
    from permuto_sdf_b200._lib import call
    torch.manual_seed(M * 100 + N)
    A = torch.randn(128, M, device="cuda")
    B = torch.randn(128, N, device="cuda")
    dump = torch.full((128, 64), float("nan"), device="cuda")
    _probe_call("umma_probe_gemm_tn", M, N, A, B, dump)
    torch.cuda.synchronize()
    want = (A.double().t() @ B.double()).float()
    Mp = (M + 15) // 16 * 16
    # accumulator row m of an M<=64, cta_group::1 instruction: find the lane that holds it
    lanes = []
    for m in range(M):
        err = (dump[:, :N] - want[m][None, :]).abs().max(dim=1).values
        lane = int(err.argmin())
        assert float(err[lane]) < 2e-3 * float(want.abs().max()), "row %d not found in TMEM (best lane %d, err %g)" % (m, lane, float(err[lane]))
        lanes.append(lane)
    print("M=%d N=%d accumulator row -> TMEM lane: %s" % (M, N, lanes))
    assert lanes == list(range(M)) or lanes == [(m // 16) * 32 + (m % 16) for m in range(M)], lanes


@pytest.mark.parametrize("L,N,it", [(16, 5000, 20000), (8, 129, 0), (24, 2000, 20000), (16, 65536, 20000)])
def test_fused_rgb_forward_matches_model(cuda, L, N, it):
    """fused colour network (encoding + SH + normal + geom -> Lipschitz MLP on tcgen05) against the modular RGB model"""
    from permuto_sdf import Sphere
    from permuto_sdf_b200.fused import FusedRGB
    from permuto_sdf_b200.models import RGB
    torch.manual_seed(L + N)
    m = RGB(3, Sphere(0.5, [0, 0, 0]), 32, 1, nr_levels=L, capacity=2 ** 16).to("cuda")
    with torch.no_grad():
        m.encoding.lattice_values.normal_(0, 0.3)
        for l in m.mlp.layers:
            l.bias.normal_(0, 0.1)
        m.mlp.lipshitz_bound_per_layer[1].fill_(1.0)          # make the Lipschitz clamp active on one layer
    pts = (torch.rand(N, 3, device="cuda") - 0.5) * 0.8
    dirs = torch.nn.functional.normalize(torch.randn(N, 3, device="cuda"), dim=-1)
    grads = torch.randn(N, 3, device="cuda") * 2.0
    geom = torch.randn(N, 32, device="cuda")
    with torch.no_grad():
        m.fused_head = False
        want = m(pts, dirs, grads, geom, it)                 # sigmoid(MLP(...))
        x = FusedRGB(m)(pts, dirs, grads, geom, it)
    got = torch.sigmoid(x)
    assert float((got - want).abs().max()) < 1e-4, float((got - want).abs().max())
    # and on the linear output itself, relative to its scale
    want_lin = torch.logit(want.double().clamp(1e-9, 1 - 1e-9)).float()
    assert float((x - want_lin).abs().max() / want_lin.abs().max()) < 1e-3


@pytest.mark.parametrize("L,N,it", [(16, 3000, 20000), (8, 129, 0), (24, 1000, 20000), (16, 40000, 20000)])
def test_fused_rgb_training_gradients_match_autograd(cuda, L, N, it):
    """fused colour-network backward (reverse sweep + tensor-core dW + lattice scatter + normal / geom gradients) against autograd
    through the modular RGB model"""
    from permuto_sdf import Sphere
    from permuto_sdf_b200.models import RGB
    torch.manual_seed(L * 7 + N)
    m = RGB(3, Sphere(0.5, [0, 0, 0]), 32, 1, nr_levels=L, capacity=2 ** 14).to("cuda")
    with torch.no_grad():
        m.encoding.lattice_values.normal_(0, 0.3)
        for l in m.mlp.layers:
            l.bias.normal_(0, 0.1)
        m.mlp.lipshitz_bound_per_layer[1].fill_(1.0)
    pts = (torch.rand(N, 3, device="cuda") - 0.5) * 0.8
    dirs = torch.nn.functional.normalize(torch.randn(N, 3, device="cuda"), dim=-1)
    grads0 = torch.randn(N, 3, device="cuda") * 2.0
    geom0 = torch.randn(N, 32, device="cuda")
    coef = torch.randn(N, 3, device="cuda")
    m.fused_head = False
    res = {}
    for mode in ("modular", "fused"):
        if mode == "fused":
            m.enable_fused()
        m.zero_grad()
        g = grads0.clone().requires_grad_(True)
        f = geom0.clone().requires_grad_(True)
        out = m(pts, dirs, g, f, it)                      # sigmoid(MLP(...)), no calibration
        loss = (out * coef).sum() + (out ** 2).sum()
        loss.backward()
        res[mode] = dict(loss=float(loss), g=g.grad.clone(), f=f.grad.clone(), lat=m.encoding.lattice_values.grad.clone(),
                         W=[l.weight.grad.clone() for l in m.mlp.layers], b=[l.bias.grad.clone() for l in m.mlp.layers],
                         c=[c.grad.clone() for c in m.mlp.lipshitz_bound_per_layer])
    a, b = res["fused"], res["modular"]
    rel = lambda x, y: float((x - y).abs().max() / (y.abs().max() + 1e-20))
    assert abs(a["loss"] - b["loss"]) < 1e-4 * abs(b["loss"])
    assert rel(a["g"], b["g"]) < 1e-3, ("sdf gradient", rel(a["g"], b["g"]))
    assert rel(a["f"], b["f"]) < 1e-3, ("geom", rel(a["f"], b["f"]))
    assert rel(a["lat"], b["lat"]) < 1e-3, ("lattice", rel(a["lat"], b["lat"]))
    for l in range(4):
        assert rel(a["W"][l], b["W"][l]) < 1e-3, ("W", l, rel(a["W"][l], b["W"][l]))
        assert rel(a["b"][l], b["b"][l]) < 1e-3, ("b", l, rel(a["b"][l], b["b"][l]))
        assert float((a["c"][l] - b["c"][l]).abs().max()) < 1e-3 * max(1e-6, float(b["c"][l].abs().max())) + 1e-7, ("c", l)


@pytest.mark.parametrize("N", [1, 127, 128, 130])
def test_fused_kernels_tile_boundaries(cuda, N):
    """sample counts around the 128-row tile size (and a single sample) through every fused kernel pair: values and parameter
    gradients agree with the modular autograd path"""
    from permuto_sdf import Sphere
    from permuto_sdf_b200.models import RGB, SDF
    torch.manual_seed(N)
    sph = Sphere(0.5, [0, 0, 0])
    pts = (torch.rand(N, 3, device="cuda") - 0.5) * 0.8
    rel = lambda x, y: float((x - y).abs().max() / (y.abs().max() + 1e-20))
    # ---- SDF
    m = SDF(3, sph, 32, 10000, nr_levels=8, capacity=2 ** 12, hidden=32).to("cuda")
    with torch.no_grad():
        m.encoding.lattice_values.normal_(0, 0.3)
    res = {}
    for fused in (False, True):
        if fused:
            m.enable_fused_training()
        m.zero_grad()
        sdf, grad, geom = m.get_sdf_and_gradient(pts.clone(), 20000)
        ((grad.norm(dim=-1) - 1) ** 2).sum().add(sdf.sum()).add(geom.pow(2).sum()).backward()
        lin = [l for l in m.mlp_sdf if isinstance(l, torch.nn.Linear)]
        res[fused] = (sdf.detach(), grad.detach(), m.encoding.lattice_values.grad.clone(), [l.weight.grad.clone() for l in lin])
    assert rel(res[True][0], res[False][0]) < 1e-3 and rel(res[True][1], res[False][1]) < 1e-3
    assert rel(res[True][2], res[False][2]) < 1e-3
    for a, b in zip(res[True][3], res[False][3]):
        assert rel(a, b) < 1e-3
    # ---- colour network
    c = RGB(3, sph, 32, 1, nr_levels=8, capacity=2 ** 12).to("cuda")
    with torch.no_grad():
        c.encoding.lattice_values.normal_(0, 0.3)
    c.fused_head = False
    dirs = torch.nn.functional.normalize(torch.randn(N, 3, device="cuda"), dim=-1)
    g0, f0 = torch.randn(N, 3, device="cuda"), torch.randn(N, 32, device="cuda")
    res = {}
    for fused in (False, True):
        if fused:
            c.enable_fused()
        c.zero_grad()
        g, f = g0.clone().requires_grad_(True), f0.clone().requires_grad_(True)
        out = c(pts, dirs, g, f, 20000)
        out.pow(2).sum().backward()
        res[fused] = (out.detach(), g.grad.clone(), f.grad.clone(), c.encoding.lattice_values.grad.clone(),
                      [l.weight.grad.clone() for l in c.mlp.layers])
    assert float((res[True][0] - res[False][0]).abs().max()) < 1e-4
    for i in (1, 2, 3):
        assert rel(res[True][i], res[False][i]) < 1e-3, i
    for a, b in zip(res[True][4], res[False][4]):
        assert rel(a, b) < 1e-3


@pytest.mark.parametrize("n", [1000, 128 * 37 + 5, 65536])
def test_dual_group_forward_equals_lock_step_forward(cuda, n):
    """k_sdf_fused_dual (two independent 64-sample groups per CTA, M = 64 MMAs, 16x256b TMEM loads) against k_sdf_fused<true> (one
    128-sample tile per CTA): same arithmetic per sample -> identical sdf, gradient and geometric feature"""
    from permuto_sdf import Sphere
    from permuto_sdf_b200 import call
    from permuto_sdf_b200.models import SDF
    torch.manual_seed(3)
    m = SDF(3, Sphere(0.5, [0, 0, 0]), 32, 10000, nr_levels=16, capacity=2 ** 18, hidden=64).to("cuda")
    with torch.no_grad():
        m.encoding.lattice_values.mul_(1e4)          # default init is 1e-5: make the lattice matter
    f = m.enable_fused_inference()
    pos = ((torch.rand(n, 3) - 0.5) * 0.9).cuda()
    res = {}
    try:
        for variant in (0, 1):
            assert call("psdf_sdf_forward_variant", variant) == variant
            res[variant] = f(pos, 4000, with_gradient=True)
    finally:
        call("psdf_sdf_forward_variant", 1)
    for a, b in zip(res[0], res[1]):
        assert torch.isfinite(b).all()
        assert float((a - b).abs().max()) <= 1e-6 * float(a.abs().max()), float((a - b).abs().max())
