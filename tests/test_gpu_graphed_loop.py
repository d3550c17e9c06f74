"""The graphed steps as a complete replacement for the training loop's eager step: per-term losses read from the graph
(GraphedPrimitiveLoss.terms / GraphedMeshLoss.terms), the silhouette rendered from the dataset's cameras (sil_cameras=,
train.py with IS_VIEW_CENTER = False), the epoch's short last batch (a graph per smaller batch size, captured on first
use into the full-size graph's pool), and HostPipeline carrying the terms and the short batch.  Each against the eager
PrimitiveLoss / MeshLoss on the same inputs; sampled steps under the same device seed."""
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


def close(a, b, rtol=1e-4, atol=0.0, what=""):
    a = a.detach().cpu().numpy() if isinstance(a, torch.Tensor) else np.asarray(a)
    b = b.detach().cpu().numpy() if isinstance(b, torch.Tensor) else np.asarray(b)
    np.testing.assert_allclose(a, b, rtol=rtol, atol=atol, err_msg=what)


def launches():
    from vpn_b200 import _lib
    torch.cuda.synchronize()
    return int(_lib.load().vpn_launch_count())


def scene(O, b, k, m, res, seed):
    g = torch.Generator().manual_seed(seed)
    v, q, t = O.synthetic_primitives(b, k, seed=seed)
    tgt = (torch.rand(b, m, 3, generator=g) - 0.5) * 0.8
    gt = (torch.rand(b, 1, res, res, generator=g) > 0.5).float()
    return v.cuda(), q.cuda(), (t * 0.3).cuda(), tgt.cuda(), gt.cuda(), g


def view_params(b, g):
    """dists, elevs, azims, angles of train.py's dataset: a camera off the view-centred one."""
    return ((1.2 + 0.6 * torch.rand(b, generator=g)).cuda(), (10.0 + 30.0 * torch.rand(b, generator=g)).cuda(),
            (360.0 * torch.rand(b, generator=g)).cuda(), (360.0 * torch.rand(b, generator=g)).cuda())


def eager(vpn, cfg, v, q, t, u, tgt, **kw):
    vc, qc, tc = (x.detach().clone().requires_grad_() for x in (v, q, t))
    out = vpn.PrimitiveLoss(cfg)(vc, qc, tc, u, tgt, **kw)
    out["total"].backward()
    return out, (vc.grad, qc.grad, tc.grad)


def check_step(got, terms, out, grads, what):
    """Graphed results against the eager step: the tolerances of test_graphed_step_matches_eager."""
    loss, *g = got
    close(loss, out["total"], rtol=1e-6, what=f"{what} loss")
    for a, b_, nm in zip(g, grads, "vqt"):
        assert a.shape == b_.shape, f"{what} grad {nm} shape"
        close(a, b_, rtol=1e-5, atol=1e-7, what=f"{what} grad {nm}")
    names = [k for k in out if k in ("view_cd", "obj_cd", "vp_div", "emd", "sil", "cd")]
    assert list(terms) == names, f"{what} term keys"
    for k in names:
        close(terms[k], out[k], rtol=1e-6, what=f"{what} term {k}")


def test_primitive_terms_match_eager_and_sum_to_the_loss(vpn, O):
    """Every term on (vertex Chamfer: no random draw): the graphed step's terms are the eager dict's, and summed in the
    eager step's order they give the returned loss bit for bit."""
    b, k, res = 2, 16, 32
    v, q, t, tgt, gt, g = scene(O, b, k, k * 128, res, 5)
    cams = view_params(b, g)
    canon = tgt * cams[0][:, None, None]
    cfg = vpn.PrimitiveLossConfig(kind="sphere", vertex_chamfer=True, l_view_cd=1.0, l_can_cd=0.5, l_vp_div=0.1,
                                  l_sil=1.0, l_emd=1.0)
    gr = vpn.GraphedPrimitiveLoss(cfg, v, q, t, tgt, gt, canonical_points=canon, cameras=cams)
    for scale, shift in ((1.0, 0.0), (0.8, 0.03)):
        vi, ti, tg = v * scale, t + shift, tgt * scale
        got = gr(vi, q, ti, tg, gt, canonical_points=canon * scale, cameras=cams)
        assert len(got) == 4
        out, grads = eager(vpn, cfg, vi, q, ti, None, tg, silhouettes=gt, canonical_points=canon * scale, dists=cams[0],
                           elevs=cams[1], azims=cams[2], angles=cams[3])
        assert list(gr.terms) == ["view_cd", "obj_cd", "vp_div", "emd", "sil"]
        assert all(gr.terms[x].dim() == 0 for x in gr.terms)
        check_step(got, gr.terms, out, grads, f"scale {scale}")
        total = None
        for x in vpn.PrimitiveLoss.TERMS:
            total = gr.terms[x] if total is None else total + gr.terms[x]
        assert torch.equal(total, got[0]), "terms summed in the eager order"


def test_mesh_terms_match_eager_and_sum_to_the_loss(vpn):
    b, res = 2, 32
    g = torch.Generator().manual_seed(9)
    faces = vpn.PrimitiveLoss().composed_faces(16, "cuda")
    verts = (torch.rand(b, 2048, 3, generator=g) * 0.6 + 0.2).cuda()
    target = (torch.rand(b, 2048, 3, generator=g) * 0.8 + 0.1).cuda()
    gt = (torch.rand(b, 1, res, res, generator=g) > 0.5).float().cuda()
    cfg = vpn.MeshLossConfig(n_samples=0, l_sil=1.0, l_emd=1.0)
    gr = vpn.GraphedMeshLoss(cfg, verts, faces, target, gt)
    for scale, shift in ((1.0, 0.0), (0.9, 0.03)):
        vin, tin = verts * scale + shift, target * scale + shift
        got = gr(vin, tin, gt)
        assert len(got) == 2
        vc = vin.clone().requires_grad_()
        out = vpn.MeshLoss(cfg)(vc, faces, tin, silhouettes=gt)
        out["total"].backward()
        assert list(gr.terms) == ["cd", "emd", "sil"]
        check_step(got, gr.terms, out, (vc.grad,), f"mesh scale {scale}")
        assert torch.equal(gr.terms["cd"] + gr.terms["emd"] + gr.terms["sil"], got[0])


def test_sil_cameras_match_eager(vpn, O):
    """train.py with IS_VIEW_CENTER = False: the silhouette rendered from the dataset's (dists, elevs, azims), copied in
    at every call; equal to eager PrimitiveLoss(..., sil_cameras=), and different from the view-centred render."""
    b, k, res = 2, 8, 32
    v, q, t, tgt, gt, g = scene(O, b, k, 1024, res, 13)
    cfg = vpn.PrimitiveLossConfig(kind="sphere", vertex_chamfer=True, l_sil=1.0)
    cams = [view_params(b, g)[:3] for _ in range(2)]
    gr = vpn.GraphedPrimitiveLoss(cfg, v, q, t, tgt, gt, sil_cameras=cams[0])
    centred = vpn.GraphedPrimitiveLoss(cfg, v, q, t, tgt, gt)
    for i, sc in enumerate(cams):
        vi = v * (1.0 - 0.1 * i)
        got = [x.clone() for x in gr(vi, q, t, tgt, gt, sil_cameras=sc)]
        terms = {x: y.clone() for x, y in gr.terms.items()}
        out, grads = eager(vpn, cfg, vi, q, t, None, tgt, silhouettes=gt, sil_cameras=sc)
        check_step(got, terms, out, grads, f"cameras {i}")
        assert float(out["sil"]) > 0
        c_loss = centred(vi, q, t, tgt, gt)[0]
        c_sil = centred.terms["sil"].clone()
        assert not torch.equal(c_sil, terms["sil"]) and abs(float(c_sil) - float(terms["sil"])) > 1e-4 * float(c_sil)
        assert not torch.equal(c_loss, got[0])


SHORT = {
    "vertex": dict(cfg=dict(kind="sphere", vertex_chamfer=True, l_sil=1.0, l_emd=1.0), k=8, n=0),
    "sphere": dict(cfg=dict(kind="sphere", l_sil=1.0), k=8, n=128),
    "mixed": dict(cfg=dict(kind="mixed", n_cuboids=3, l_sil=1.0), k=8, n=128),
}


@pytest.mark.parametrize("path", list(SHORT))
def test_short_batches_primitive(vpn, O, path):
    """Captured at B = 4, called with b = 3, 4, 3 on fresh inputs, each against the eager step (the sampled paths under
    the same device seed; a replay draws afresh).  The full-size results after a short replay are still right (the
    shared pool corrupts nothing), later b = 3 calls capture nothing, b = 5 is refused before any copy or launch."""
    p = SHORT[path]
    big, k, n = 4, p["k"], p["n"]
    cfg = vpn.PrimitiveLossConfig(**p["cfg"])
    m = k * 128 if n == 0 else 1024
    v, q, t, tgt, gt, _ = scene(O, big, k, m, 32, 20)
    gr = vpn.GraphedPrimitiveLoss(cfg, v, q, t, tgt, gt, n_samples=n)
    full_graph = gr.graph

    def uniforms(b):
        if n == 0:
            return None
        if path == "mixed":
            kc = cfg.n_cuboids
            return torch.rand((b, kc, n, 3), device="cuda"), torch.rand((b, k - kc, n, 2), device="cuda")
        return torch.rand((b, k, n, 2), device="cuda")

    for i, b in enumerate((3, 4, 3)):
        v, q, t, tgt, gt, _ = scene(O, b, k, m, 32, 30 + i)
        if i == 0:
            # the first b = 3 call captures; its eager warm-up steps advance the device generator, so the comparison
            # under a fresh seed is made on the next call
            n0 = launches()
            gr(v, q, t, tgt, gt)
            assert launches() > n0
        n0 = launches()
        torch.cuda.manual_seed(500 + i)
        got = [x.clone() for x in gr(v, q, t, tgt, gt)]
        terms = {x: y.clone() for x, y in gr.terms.items()}
        assert launches() == n0, f"call {i}: a replay launches nothing from the host"
        torch.cuda.manual_seed(500 + i)
        out, grads = eager(vpn, cfg, v, q, t, uniforms(b), tgt, silhouettes=gt)
        assert all(torch.isfinite(x).all() for x in got)
        check_step(got, terms, out, grads, f"{path} b={b}")
        if n:
            again = gr(v, q, t, tgt, gt)[0]
            assert float(again) != float(got[0]), "a replay draws fresh uniforms"
    assert gr.graph is full_graph and gr.launches_per_step > 5
    before = [x.detach().clone() for x in (gr.v, gr.q, gr.t, gr.targets, gr.sil)]
    v, q, t, tgt, gt, _ = scene(O, 5, k, m, 32, 40)
    n0 = launches()
    with pytest.raises(AssertionError):
        gr(v, q, t, tgt, gt)
    assert launches() == n0
    for x, y in zip(before, (gr.v, gr.q, gr.t, gr.targets, gr.sil)):
        assert torch.equal(x, y.detach())


@pytest.mark.parametrize("n_samples", [2048, 0])
def test_short_batches_mesh(vpn, n_samples):
    big, res = 4, 32
    faces = vpn.PrimitiveLoss().composed_faces(16, "cuda")

    def data(b, seed):
        g = torch.Generator().manual_seed(seed)
        return ((torch.rand(b, 2048, 3, generator=g) * 0.6 + 0.2).cuda(), (torch.rand(b, 2048, 3, generator=g) * 0.8 + 0.1).cuda(),
                (torch.rand(b, 1, res, res, generator=g) > 0.5).float().cuda())

    cfg = vpn.MeshLossConfig(n_samples=n_samples, l_sil=1.0, l_emd=1.0)
    gr = vpn.GraphedMeshLoss(cfg, *data(big, 1)[:1], faces, *data(big, 1)[1:])
    for i, b in enumerate((3, 4, 3)):
        verts, tgt, gt = data(b, 10 + i)
        if i == 0:
            n0 = launches()
            gr(verts, tgt, gt)                                  # captures (test_short_batches_primitive)
            assert launches() > n0
        n0 = launches()
        torch.cuda.manual_seed(700 + i)
        got = [x.clone() for x in gr(verts, tgt, gt)]
        terms = {x: y.clone() for x, y in gr.terms.items()}
        assert launches() == n0, f"call {i}: a replay launches nothing from the host"
        torch.cuda.manual_seed(700 + i)
        vc = verts.clone().requires_grad_()
        out = vpn.MeshLoss(cfg)(vc, faces, tgt, silhouettes=gt)
        out["total"].backward()
        check_step(got, terms, out, (vc.grad,), f"mesh n={n_samples} b={b}")
    n0 = launches()
    before = gr.verts.detach().clone()
    with pytest.raises(AssertionError):
        gr(*data(5, 3))
    assert launches() == n0 and torch.equal(before, gr.verts.detach())


def test_host_pipeline_with_terms_and_a_short_last_batch(vpn, O):
    """Five full batches and a last one of 2 out of 3 through HostPipeline, the terms returned with the results: equal
    to direct graphed calls, with the tolerances of test_host_pipeline_matches_direct_steps."""
    big, k, m, res = 3, 8, 1024, 32
    cfg = vpn.PrimitiveLossConfig(kind="sphere", l_sil=1.0, vertex_chamfer=True)
    batches = []
    for i, b in enumerate((big,) * 5 + (2,)):
        v, q, t, tgt, gt, _ = scene(O, b, k, m, res, 80 + i)
        batches.append({"v": v.cpu().pin_memory(), "q": q.cpu().pin_memory(), "t": t.cpu().pin_memory(),
                        "target": tgt.cpu().pin_memory(), "sil": gt.cpu().pin_memory(), "unused": None})
    d0 = {key: (x.cuda() if x is not None else None) for key, x in batches[0].items()}
    gr = vpn.GraphedPrimitiveLoss(cfg, d0["v"], d0["q"], d0["t"], d0["target"], d0["sil"])
    fn = lambda s: (*gr(s["v"], s["q"], s["t"], s["target"], s["sil"]), *gr.terms.values())
    want = []
    for bt in batches:
        d = {key: (x.cuda() if x is not None else None) for key, x in bt.items()}
        want.append([x.detach().cpu().clone() for x in fn(d)])
    pipe = vpn.HostPipeline(fn, batches[0], "cuda")
    got = []
    pipe.submit(batches[0])
    for bt in batches[1:]:
        pipe.submit(bt)
        got.append([x.clone() for x in pipe.result()])
    got.append([x.clone() for x in pipe.result()])
    assert len(got) == 6 and all(len(x) == 4 + 3 for x in got)                 # loss, 3 grads, view_cd / vp_div / sil
    assert tuple(got[-1][1].shape) == (2, k, 3)
    for i, (w, gg) in enumerate(zip(want, got)):                # the backward scatters with atomics: not bitwise repeatable
        close(gg[0], w[0], rtol=1e-6, what=f"batch {i} loss")
        for a, c in zip(w[1:4], gg[1:4]):
            close(c, a, rtol=1e-5, atol=1e-7, what=f"batch {i} grad")
        for a, c in zip(w[4:], gg[4:]):
            close(c, a, rtol=1e-6, what=f"batch {i} term")
