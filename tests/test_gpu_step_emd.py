"""The EMD loss term (train.py:188-195, train_gcn.py:91-95): the fused loss head and backward of vpn_b200.emd_distance
against the composition it replaces (ops.emd_auction + torch.sqrt(dist).mean(1) * weight) and against the CPU oracle,
its independence of the batch and of the auction's cluster size, and the term inside PrimitiveLoss, eager and replayed
from a CUDA graph."""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def vpn():
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    import vpn_b200
    return vpn_b200


@pytest.fixture(scope="module")
def O():
    from oracle import vpn_oracle
    return vpn_oracle


def C(a):
    return torch.as_tensor(np.asarray(a)).cuda()


def close(a, b, rtol, atol=0.0, what=""):
    a = a.detach().cpu().numpy() if isinstance(a, torch.Tensor) else np.asarray(a)
    b = b.detach().cpu().numpy() if isinstance(b, torch.Tensor) else np.asarray(b)
    np.testing.assert_allclose(a, b, rtol=rtol, atol=atol, err_msg=what)


def on_target_clouds(vpn, b, n, seed, eps, iters):
    """Uniform clouds in [0,1] in which prediction 5 of sample 0 sits exactly on the target the auction assigns it."""
    g = torch.Generator().manual_seed(seed)
    x1 = torch.rand(b, n, 3, generator=g); x2 = torch.rand(b, n, 3, generator=g)
    for _ in range(4):                                     # moving the prediction can change the assignment: repeat
        _, a = vpn.emd_auction(C(x1), C(x2), eps, iters)
        on = x2[0, int(a[0, 5])]
        if torch.equal(x1[0, 5], on):
            break
        x1[0, 5] = on
    return C(x1), C(x2)


@pytest.mark.parametrize("b,n,weight", [(4, 2048, 1.0), (3, 1536, 0.7), (2, 1000, 2.5)])
def test_loss_head_matches_composition(vpn, b, n, weight):
    eps, iters = 0.005, 50
    x1, x2 = on_target_clouds(vpn, b, n, 10 + n, eps, iters)
    up = C(torch.rand(b, generator=torch.Generator().manual_seed(n)) + 0.5)
    xr = x1.clone().requires_grad_()
    dist, _ = vpn.emd_auction(xr, x2, eps, iters)
    assert float(dist[0, 5].detach()) == 0.0, "the test cloud must put one prediction on its assigned target"
    ref = torch.sqrt(dist).mean(1) * weight
    (ref * up).sum().backward()
    xo = x1.clone().requires_grad_()
    loss = vpn.emd_distance(xo, x2, eps, iters, weight=weight, each_batch=True)
    assert loss.shape == (b,)
    (loss * up).sum().backward()
    close(loss, ref, rtol=1e-6, what="per-sample loss")
    nan = torch.isnan(xr.grad)
    assert bool(nan[0, 5].all()) and int(nan.sum()) == 3, "dist == 0 gives NaN, as in the reference"
    assert torch.equal(torch.isnan(xo.grad), nan), "NaN in different places"
    close(xo.grad, xr.grad, rtol=1e-6, atol=1e-12, what="gradient")
    mean = vpn.emd_distance(x1, x2, eps, iters, weight=weight)
    assert mean.dim() == 0
    close(mean, loss.mean(), rtol=1e-6)


def test_targets_get_zero_gradient(vpn):
    g = torch.Generator().manual_seed(2)
    x1 = C(torch.rand(2, 1024, 3, generator=g)).requires_grad_()
    x2 = C(torch.rand(2, 1024, 3, generator=g)).requires_grad_()
    vpn.emd_distance(x1, x2).backward()
    assert torch.equal(x2.grad, torch.zeros_like(x2)) and torch.isfinite(x1.grad).all()


@pytest.mark.parametrize("b,n", [(2, 2048), (2, 1536)])
def test_loss_matches_oracle(vpn, O, b, n):
    eps, iters = 0.005, 50
    g = torch.Generator().manual_seed(300 + n)
    x1 = torch.rand(b, n, 3, generator=g); x2 = torch.rand(b, n, 3, generator=g)
    dist, _ = vpn.emd_auction(C(x1), C(x2), eps, iters)
    loss = vpn.emd_distance(C(x1), C(x2), eps, iters, each_batch=True)
    for i in range(b):
        d_ref, _ = O.emd_auction(x1[i].numpy(), x2[i].numpy(), eps, iters)
        np.testing.assert_array_equal(dist[i].cpu().numpy(), d_ref, err_msg=f"dist sample {i}")
        close(loss[i], np.sqrt(d_ref.astype(np.float64)).mean(), rtol=1e-6, what=f"loss sample {i}")


def test_loss_independent_of_batch_and_cluster_size(vpn):
    """A sample's loss is the same bits in a batch of 8, alone, and for every cluster size of the auction, so a batch
    split over GPUs gives what one GPU gives."""
    from vpn_b200 import _lib
    lib = _lib.load()
    g = torch.Generator().manual_seed(21)
    x1 = C(torch.rand(8, 2048, 3, generator=g)); x2 = C(torch.rand(8, 2048, 3, generator=g))
    full = vpn.emd_distance(x1, x2, each_batch=True).cpu()
    try:
        for c in (0, 1, 2, 4, 8):
            assert lib.vpn_set_tuning(b"emd_cluster", c) == 0
            batch = vpn.emd_distance(x1, x2, each_batch=True).cpu()
            assert torch.equal(batch, full), f"batch of 8, cluster {c}"
            for i in (0, 3, 7):
                alone = vpn.emd_distance(x1[i:i + 1], x2[i:i + 1], each_batch=True).cpu()
                assert torch.equal(alone[0], full[i]), f"sample {i} alone, cluster {c}"
    finally:
        lib.vpn_set_tuning(b"emd_cluster", 0)


def scene(O, b, k, m, seed):
    g = torch.Generator().manual_seed(seed)
    v, q, t = O.synthetic_primitives(b, k, seed=seed)
    t = t * 0.3
    tgt = (torch.rand(b, m, 3, generator=g) - 0.5) * 0.8
    return v, q, t, tgt, g


@pytest.mark.parametrize("vertex", [False, True])
def test_step_emd_term_matches_public_ops(vpn, O, vertex):
    """PrimitiveLoss(l_view_cd=1, l_vp_div=0.1, l_emd=1) against the same terms composed from public ops on the same
    uniforms: sampled points (train.py) and composed mesh vertices (train_gcn.py)."""
    from vpn_b200 import templates
    b, k, n = 2, 16, 128
    nv = templates.template("sphere", "cpu")[0].shape[0]
    per = nv if vertex else n
    v, q, t, tgt, g = scene(O, b, k, k * per, 41 + vertex)
    u = None if vertex else C(torch.rand(b, k, n, 2, generator=g))
    cfg = vpn.PrimitiveLossConfig(kind="sphere", l_view_cd=1.0, l_vp_div=0.1, l_emd=1.0, vertex_chamfer=vertex)
    vc, qc, tc = (C(x).requires_grad_() for x in (v, q, t))
    out = vpn.PrimitiveLoss(cfg)(vc, qc, tc, u, C(tgt))
    out["total"].backward()
    vr, qr, tr = (C(x).requires_grad_() for x in (v, q, t))
    tv, _ = templates.template("sphere", "cuda")
    pts = vpn.mesh_vertices(tv, vr, qr, tr) if vertex else vpn.sample_primitives("sphere", vr, qr, tr, u)
    terms = {"view_cd": vpn.chamfer_distance(pts, C(tgt)) * 1.0,
             "vp_div": vpn.chamfer_distance(tr.contiguous(), C(tgt), w1=0.5, w2=1.0) * 0.1,
             "emd": vpn.emd_distance(pts, C(tgt), 0.005, 50) * 1.0}
    total = terms["view_cd"] + terms["vp_div"] + terms["emd"]
    total.backward()
    for name, want in terms.items():
        close(out[name], want, rtol=1e-6, what=name)
    close(out["total"], total, rtol=1e-6, what="total")
    assert float(out["emd"].detach()) > 0
    for got, want, nm in ((vc.grad, vr.grad, "v"), (qc.grad, qr.grad, "q"), (tc.grad, tr.grad, "t")):
        close(got, want, rtol=1e-5, atol=1e-7, what=f"grad {nm}")


def test_graphed_step_with_emd_matches_eager(vpn, O):
    """train_gcn.py's vertex path (no random draw) with the EMD term and the silhouette, both on their own streams:
    captured once, replayed twice (new inputs the second time), equal to the eager step."""
    b, k, res = 2, 16, 32
    v, q, t, tgt, g = scene(O, b, k, k * 128, 57)
    gt = (torch.rand(b, 1, res, res, generator=g) > 0.5).float()
    cfg = vpn.PrimitiveLossConfig(kind="sphere", l_sil=1.0, l_emd=1.0, vertex_chamfer=True)
    gr = vpn.GraphedPrimitiveLoss(cfg, C(v), C(q), C(t), C(tgt), C(gt))
    no_emd = vpn.GraphedPrimitiveLoss(vpn.PrimitiveLossConfig(kind="sphere", l_sil=1.0, vertex_chamfer=True),
                                      C(v), C(q), C(t), C(tgt), C(gt))
    assert gr.launches_per_step == no_emd.launches_per_step + 4           # auction, loss head (2), backward
    for scale, shift in ((1.0, 0.0), (0.7, 0.05)):
        vc, qc, tc = C(v * scale).requires_grad_(), C(q).requires_grad_(), C(t + shift).requires_grad_()
        tg = C(tgt * scale)
        loss, gv, gq, gtt = gr(vc.detach(), qc.detach(), tc.detach(), tg, C(gt))
        out = vpn.PrimitiveLoss(cfg)(vc, qc, tc, None, tg, silhouettes=C(gt))
        out["total"].backward()
        assert float(out["emd"].detach()) > 0
        close(loss, out["total"], rtol=1e-6)
        close(gv, vc.grad, rtol=1e-5, atol=1e-7); close(gq, qc.grad, rtol=1e-5, atol=1e-7); close(gtt, tc.grad, rtol=1e-5, atol=1e-7)
