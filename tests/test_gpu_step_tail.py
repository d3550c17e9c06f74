"""The tail of the batched step: the Chamfer loss head with the weighted batch mean inside (vpn_chamfer_loss_mean_fwd /
_bwd), and the small-first-cloud Chamfer (P <= 256, VP-diverse) as one cluster launch forward and one gather launch
backward (csrc/chamfer_simple.cu).  The mean's gradients must be the bits of torch's `each_batch.mean() * weight`
composition; the small-P forward must be the CPU oracle's bits; the small-P backward must agree with a float64 oracle
and repeat its bits across calls and between a sample alone and the same sample in a batch."""
import ctypes
import os
import subprocess

import numpy as np
import pytest
import torch

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PKG = os.path.join(REPO, "volumetric-primitives-net_b200")
VPN_ERR_SHAPE, VPN_ERR_ARG = -2, -3

gpu = pytest.mark.gpu


@pytest.fixture(scope="module")
def vpn():
    if not os.path.isfile(os.path.join(PKG, "lib", "libvpn_b200.so")):
        subprocess.check_call(["make", "-C", os.path.join(PKG, "csrc"), "-j8"])
    import vpn_b200
    return vpn_b200


@pytest.fixture(scope="module")
def O():
    from oracle import vpn_oracle
    return vpn_oracle


def clouds(gen, b, p, m, ties=False):
    p1, p2 = torch.rand(b, p, 3, generator=gen) - 0.5, torch.rand(b, m, 3, generator=gen) - 0.5
    if ties:                                    # coarse lattice: exact ties in d and in sqrt(d), duplicate targets
        p1, p2 = torch.floor(p1 * 6) / 4, torch.floor(p2 * 6) / 4 + 0.125
    return p1.contiguous(), p2.contiguous()


def test_mean_entry_points_reject_bad_arguments_without_a_device(vpn):
    from vpn_b200 import _lib
    lib = _lib.load()
    d = ctypes.c_void_p(16)                     # never dereferenced: every call below fails its argument checks first

    def fwd(min1=d, min2=d, loss=d, scratch=d, b=2, p=16, m=64):
        return lib.vpn_chamfer_loss_mean_fwd(min1, min2, 1.0, 1.0, 0.1, loss, scratch, b, p, m, None)

    for bad in ({"b": 0}, {"b": -1}, {"b": 65536}, {"p": 0}, {"m": 0}):
        assert fwd(**bad) == VPN_ERR_SHAPE, bad
    for name in ("min1", "min2", "loss", "scratch"):
        assert fwd(**{name: None}) == VPN_ERR_ARG, name

    def bwd(p1=d, p2=d, min1=d, idx1=d, min2=d, idx2=d, g=d, gp1=d, b=2, p=16, m=64):
        return lib.vpn_chamfer_loss_mean_bwd(p1, p2, min1, idx1, min2, idx2, g, 1.0, 1.0, 0.1, gp1, None, b, p, m, None)

    for bad in ({"b": 0}, {"b": 65536}, {"p": -2}, {"m": 0}):
        assert bwd(**bad) == VPN_ERR_SHAPE, bad
    for name in ("p1", "p2", "min1", "idx1", "min2", "idx2", "g", "gp1"):
        assert bwd(**{name: None}) == VPN_ERR_ARG, name


@gpu
@pytest.mark.parametrize("shape", [(32, 16, 8192), (3, 16, 2048), (1, 128, 1000), (8, 128, 16384), (3, 300, 200)])
@pytest.mark.parametrize("weight", [1.0, 0.1])
def test_weighted_mean_matches_torch_composition(vpn, shape, weight):
    b, p, m = shape
    gen = torch.Generator().manual_seed(b * 7 + p + m)
    p1, p2 = (x.cuda() for x in clouds(gen, b, p, m))
    a, c = p1.clone().requires_grad_(), p1.clone().requires_grad_()
    t2a, t2c = p2.clone().requires_grad_(), p2.clone().requires_grad_()
    fused = vpn.chamfer_distance(a, t2a, w1=0.5, w2=1.0, weight=weight)
    ref = vpn.chamfer_distance(c, t2c, each_batch=True, w1=0.5, w2=1.0).mean() * weight
    assert fused.shape == ref.shape == ()
    rel = abs(fused.item() - ref.item()) / abs(ref.item())
    print(f"{shape} weight={weight}: loss {fused.item():.9g} vs {ref.item():.9g}, relative difference {rel:.3g}")
    assert rel <= 1e-6
    g1, g2 = torch.autograd.grad(fused, (a, t2a))
    r1, r2 = torch.autograd.grad(ref, (c, t2c))
    if p <= 256:                                # fixed-order gather backward: the same bits
        assert torch.equal(g1, r1) and torch.equal(g2, r2)
    else:                                       # the column pass scatters with atomics: order-dependent last bits
        torch.testing.assert_close(g1, r1, rtol=1e-6, atol=1e-9)
        torch.testing.assert_close(g2, r2, rtol=1e-6, atol=1e-9)


@gpu
@pytest.mark.parametrize("shape,ties", [((32, 16, 8192), False), ((8, 128, 16384), False), ((1, 16, 2048), False),
                                        ((4, 16, 8192), True), ((2, 200, 5000), True), ((3, 256, 20000), False)])
def test_small_first_cloud_forward_bit_exact(vpn, c_oracle, shape, ties):
    b, p, m = shape
    assert vpn.chamfer_main_kernel_name(b, p, m) == "chamfer_smallp_fwd_kernel"
    gen = torch.Generator().manual_seed(p + m + int(ties))
    p1, p2 = clouds(gen, b, p, m, ties)
    ref = c_oracle(p1.numpy(), p2.numpy())
    got = vpn.chamfer_nn(p1.cuda(), p2.cuda())
    for name, r, g in zip(("min1", "idx1", "min2", "idx2"), ref, got):
        g = g.cpu().numpy()
        if name.startswith("min"):
            assert np.array_equal(g.view(np.uint32), r.view(np.uint32)), name
        else:
            assert np.array_equal(g.astype(np.int64), r), name


@gpu
@pytest.mark.parametrize("shape,ties", [((32, 16, 8192), False), ((8, 128, 16384), False), ((1, 16, 2048), False),
                                        ((3, 256, 20000), False), ((4, 16, 8192), True)])
def test_small_first_cloud_backward(vpn, O, shape, ties):
    b, p, m = shape
    gen = torch.Generator().manual_seed(3 * p + m)
    p1, p2 = clouds(gen, b, p, m, ties)
    if ties:
        p2 = p2 + 0.01                           # no pair at distance 0 (its gradient is NaN, as in the reference)
    g1, g2 = torch.rand(b, p, generator=gen), torch.rand(b, m, generator=gen)

    def run(x1, x2, u1, u2):
        a, c = x1.cuda().requires_grad_(), x2.cuda().requires_grad_()
        o1, _, o2, _ = vpn.chamfer_nn(a, c)
        return torch.autograd.grad((o1 * u1.cuda()).sum() + (o2 * u2.cuda()).sum(), (a, c))

    gp1, gp2 = run(p1, p2, g1, g2)
    m1, i1, m2, i2 = O.chamfer_nn(p1, p2)
    r1, r2 = O.chamfer_grad_from_nn(p1.double(), p2.double(), m1.double(), i1, m2.double(), i2, g1.double(), g2.double())
    for got, want in ((gp1, r1), (gp2, r2)):
        got = got.cpu().double()
        err = (got - want).abs().max().item()
        print(f"{shape} ties={ties}: max |float32 - float64| = {err:.3g} (max |grad| {want.abs().max().item():.3g})")
        torch.testing.assert_close(got, want, rtol=1e-4, atol=1e-5 * want.abs().max().item())
    for _ in range(2):                          # the same bits on every call
        again = run(p1, p2, g1, g2)
        assert torch.equal(again[0], gp1) and torch.equal(again[1], gp2)
    k = b // 2                                  # and a sample alone gives the bits it gives inside the batch
    alone = run(p1[k:k + 1], p2[k:k + 1], g1[k:k + 1], g2[k:k + 1])
    assert torch.equal(alone[0], gp1[k:k + 1]) and torch.equal(alone[1], gp2[k:k + 1])


@gpu
def test_graph_replay_equals_eager_step(vpn):
    """c2's step at B = 4: view Chamfer (tensor-core filter, large P) + VP-diverse (small P) through the weighted-mean
    heads, with the graphed step seeded by a preallocated scalar."""
    import bench
    d = bench.synthetic("c2", "cpu", batch=4)[0]
    dev = torch.device("cuda")
    v, q, t, tgt = (d[k].to(dev) for k in ("v", "q", "t", "target"))
    cfg = vpn.PrimitiveLossConfig(kind="cuboid")
    n = 4096
    gr = vpn.GraphedPrimitiveLoss(cfg, v, q, t, tgt, n_samples=n)
    for i in range(2):
        torch.cuda.manual_seed(500 + i)
        loss, gv, gq, gt = (x.clone() for x in gr(v, q, t, tgt))
        torch.cuda.manual_seed(500 + i)
        u = torch.rand((4, 16, n, 3), device=dev)
        vc, qc, tc = (x.clone().requires_grad_() for x in (v, q, t))
        out = vpn.PrimitiveLoss(cfg)(vc, qc, tc, u, tgt)
        out["total"].backward()
        assert torch.equal(loss, out["total"].detach())           # the forward and both loss heads are fixed-order
        torch.testing.assert_close(gv, vc.grad, rtol=1e-5, atol=1e-9)
        torch.testing.assert_close(gq, qc.grad, rtol=1e-5, atol=1e-9)
        torch.testing.assert_close(gt, tc.grad, rtol=1e-5, atol=1e-9)
