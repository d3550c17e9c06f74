"""Mixed cuboid + sphere assemblies (train.py: CUBOID_NUM cuboids, then SPHERE_NUM spheres): the one-launch mixed pose
kernels against the single-kind kernels bit for bit, forward and backward, sampled and template; PrimitiveLoss(kind=
"mixed") against the CPU oracle and the train.py helpers run on the drop-in modules; the vertex + EMD path against the
public ops; and GraphedPrimitiveLoss(kind="mixed") replayed against the eager step, also fed through HostPipeline."""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

# (B, Kc, Ks, N): N = 1001 takes the unvectorised tail path, N = 4096 two slices per primitive; Kc = 0 and Ks = 0 are
# the single-kind assemblies
CASES = [(2, 1, 1, 128), (3, 5, 3, 1001), (8, 8, 8, 128), (2, 16, 16, 4096), (2, 0, 7, 300), (3, 6, 0, 2500)]


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


def same_bits(a, b, what):
    assert a.shape == b.shape, f"{what}: shape {tuple(a.shape)} vs {tuple(b.shape)}"
    assert torch.equal(a.detach().view(torch.int32), b.detach().view(torch.int32)), f"{what}: bits differ"


def assembly(O, b, k, seed, spread=0.3):
    v, q, t = O.synthetic_primitives(b, k, seed=seed)
    return v.cuda(), q.cuda(), (t * spread).cuda()


def leaves(*xs):
    return [x.detach().clone().requires_grad_() for x in xs]


@pytest.mark.parametrize("b,kc,ks,n", CASES)
def test_sampled_forward_and_backward_bits(vpn, O, b, kc, ks, n):
    k = kc + ks
    v, q, t = assembly(O, b, k, seed=100 + n + kc)
    g = torch.Generator(device="cuda").manual_seed(n + k)
    uc = torch.rand(b, kc, n, 3, device="cuda", generator=g)
    us = torch.rand(b, ks, n, 2, device="cuda", generator=g)
    vm, qm, tm = leaves(v, q, t)
    pts = vpn.sample_mixed_primitives(kc, vm, qm, tm, uc, us)
    assert pts.shape == (b, k * n, 3)
    grad = torch.randn(b, k * n, 3, device="cuda", generator=g)
    pts.backward(grad)
    for kind, sl, u in (("cuboid", slice(0, kc), uc), ("sphere", slice(kc, k), us)):
        if sl.stop == sl.start:
            continue
        vs, qs, ts = leaves(v[:, sl], q[:, sl], t[:, sl])
        ref = vpn.sample_primitives(kind, vs, qs, ts, u)
        same_bits(pts.view(b, k, n, 3)[:, sl], ref.view(b, -1, n, 3), f"{kind} points")
        ref.backward(grad.view(b, k, n, 3)[:, sl].reshape(b, -1, 3))
        for got, want, nm in ((vm.grad, vs.grad, "v"), (qm.grad, qs.grad, "q"), (tm.grad, ts.grad, "t")):
            same_bits(got[:, sl], want, f"{kind} grad {nm}")


@pytest.mark.parametrize("b,kc,ks", [(2, 1, 1), (3, 5, 3), (8, 8, 8), (2, 16, 16), (2, 0, 7), (3, 6, 0)])
def test_template_vertices_and_gradients_bits(vpn, O, b, kc, ks):
    from vpn_b200 import templates
    k = kc + ks
    tc, ts_ = templates.template("cuboid", "cuda")[0], templates.template("sphere", "cuda")[0]
    nvc, nvs = tc.shape[0], ts_.shape[0]
    v, q, t = assembly(O, b, k, seed=7 + k)
    vm, qm, tm = leaves(v, q, t)
    verts = vpn.mesh_vertices_mixed(kc, tc, ts_, vm, qm, tm)
    assert verts.shape == (b, kc * nvc + ks * nvs, 3)
    grad = torch.randn(verts.shape, device="cuda", generator=torch.Generator(device="cuda").manual_seed(k))
    verts.backward(grad)
    rows = {"cuboid": slice(0, kc * nvc), "sphere": slice(kc * nvc, kc * nvc + ks * nvs)}
    for kind, sl, tpl in (("cuboid", slice(0, kc), tc), ("sphere", slice(kc, k), ts_)):
        if sl.stop == sl.start:
            continue
        vs, qs, tt = leaves(v[:, sl], q[:, sl], t[:, sl])
        ref = vpn.mesh_vertices(tpl, vs, qs, tt)
        same_bits(verts[:, rows[kind]], ref, f"{kind} vertices")
        ref.backward(grad[:, rows[kind]])
        for got, want, nm in ((vm.grad, vs.grad, "v"), (qm.grad, qs.grad, "q"), (tm.grad, tt.grad, "t")):
            same_bits(got[:, sl], want, f"{kind} grad {nm}")


def oracle_mesh(O, kc, v, q, t):
    """The mixed assembly's composed mesh on the CPU oracle: per-primitive meshing, then compose_meshes."""
    from vpn_b200 import templates
    k = v.shape[1]
    tpl = [templates.template("cuboid" if i < kc else "sphere", "cpu") for i in range(k)]
    verts = torch.cat([O.mesh_vertices(tpl[i][0], v[:, i], q[:, i], t[:, i]) for i in range(k)], dim=1)
    _, faces = O.compose_meshes([tv for tv, _ in tpl], [tf.long() for _, tf in tpl])
    return verts, faces


@pytest.mark.parametrize("b,kc,ks,res", [(2, 2, 3, 48), (1, 8, 8, 64)])
def test_mixed_silhouette_vs_oracle(vpn, O, b, kc, ks, res):
    """Tolerances of test_gpu_parity.py::test_silhouette_vs_oracle, on the mixed mesh and its composed faces."""
    k = kc + ks
    v, q, t = O.synthetic_primitives(b, k, seed=21)
    v, t = v * 1.5, t * 0.25
    step = vpn.PrimitiveLoss(vpn.PrimitiveLossConfig(kind="mixed", n_cuboids=kc))
    _, faces_ref = oracle_mesh(O, kc, v, q, t)
    faces = step.composed_faces(k, "cuda")
    assert torch.equal(faces.cpu().long(), faces_ref)
    verts = step._vertices(v.cuda(), q.cuda(), t.cuda()).detach().requires_grad_()
    verts_ref = verts.detach().cpu().clone().requires_grad_()
    cams = [O.look_at_camera(0.0, 0.0, 1.0) for _ in range(b)]
    rot, pos = torch.stack([c[0] for c in cams]), torch.stack([c[1] for c in cams])
    ref = O.soft_silhouette(verts_ref, faces_ref, rot, pos, res, res)
    w = torch.rand(b, res, res, generator=torch.Generator().manual_seed(4))
    (ref * w).sum().backward()
    r_c, p_c = vpn.look_at_cameras(torch.zeros(b).cuda(), torch.zeros(b).cuda(), torch.ones(b).cuda())
    alpha, _, _ = vpn.soft_silhouette(verts, faces, r_c, p_c, res, res)
    close(alpha, ref, rtol=1e-4, atol=2e-6)
    assert ((alpha.detach().cpu() == 1.0) == (ref.detach() == 1.0)).all()
    assert float(alpha.detach().max()) > 0.5
    (alpha * w.cuda()).sum().backward()
    close(verts.grad, verts_ref.grad, rtol=1e-3, atol=1e-4 * float(verts_ref.grad.abs().max()))


def uniforms_in_reference_order(seed, b, kc, ks, n):
    """The draws Sampling.cuboid_sampling / sphere_sampling make for primitives 0..K-1 of train.py's loop (cuboid.py:66:
    one (B,N,3) draw; sphere.py:26-27: elev, then azim), regrouped as (u_cuboid, u_sphere)."""
    torch.manual_seed(seed)
    uc = torch.empty(b, kc, n, 3, device="cuda")
    us = torch.empty(b, ks, n, 2, device="cuda")
    for i in range(kc + ks):
        if i < kc:
            uc[:, i] = torch.rand((b, n, 3), device="cuda")
        else:
            us[:, i - kc, :, 0:1] = torch.rand((b, n, 1), device="cuda")
            us[:, i - kc, :, 1:2] = torch.rand((b, n, 1), device="cuda")
    return uc, us


@pytest.mark.parametrize("kc,ks", [(8, 8), (3, 13)])
def test_step_vs_oracle_and_train_py_helpers(vpn, O, kc, ks):
    """PrimitiveLoss(kind="mixed") with l_view_cd, l_vp_div and l_sil against the CPU oracle and against train.py's
    helpers restated on the drop-in modules with CUBOID_NUM = kc, SPHERE_NUM = ks, on the same uniforms."""
    from test_gpu_train_loop_integration import helpers
    b, n, m, res, seed = 4, 128, 2048, 64, 31
    k = kc + ks
    v, q, t = O.synthetic_primitives(b, k, seed=seed)
    t = t * 0.3
    g = torch.Generator().manual_seed(seed)
    target = (torch.rand(b, m, 3, generator=g) - 0.5) * 0.8
    gt = (torch.rand(b, 1, res, res, generator=g) > 0.5).float()
    cfg = vpn.PrimitiveLossConfig(kind="mixed", n_cuboids=kc, l_sil=1.0, l_vp_div=0.1)
    uc, us = uniforms_in_reference_order(seed, b, kc, ks, n)
    vc, qc, tc = (x.cuda().requires_grad_() for x in (v, q, t))
    out = vpn.PrimitiveLoss(cfg)(vc, qc, tc, (uc, us), target.cuda(), silhouettes=gt.cuda())
    out["total"].backward()

    # train.py's helpers on the drop-in modules: the same draws from the same seed
    ns = helpers("train", CUBOID_NUM=kc, SPHERE_NUM=ks, L_SIL=1.0, L_VP_DIV=0.1, L_VIEW_CD=1.0, SAMPLE_NUM=n)
    vd, qd, td = (x.cuda().requires_grad_() for x in (v, q, t))
    vols, rots, trs = ([x[:, i] for i in range(k)] for x in (vd, qd, td))
    torch.manual_seed(seed)
    pts_d = ns["sample_predict_points"](vols, rots, trs)
    same_bits(out["points"], pts_d, "points vs train.py helpers")
    zero, one = torch.zeros(b).cuda(), torch.ones(b).cuda()
    view_cd, _ = ns["calculate_cd_loss"](pts_d, target.cuda(), target.cuda(), one, zero, zero, zero)
    meshes = ns["compose_vp_meshes"](ns["get_vp_meshes"](vols, rots, trs))
    sil = ns["calculate_silhouette_loss"](meshes, gt.cuda(), one, zero, zero)
    div = ns["calculate_vp_div_loss"](trs, target.cuda())
    total_d = view_cd + sil + div
    total_d.backward()
    for name, want in (("view_cd", view_cd), ("sil", sil), ("vp_div", div), ("total", total_d)):
        close(out[name], want, rtol=1e-6, what=f"{name} vs train.py helpers")
    for got, want, nm in ((vc.grad, vd.grad, "v"), (qc.grad, qd.grad, "q"), (tc.grad, td.grad, "t")):
        close(got, want, rtol=0, atol=1e-4 * float(want.abs().max()), what=f"grad {nm} vs train.py helpers")

    # CPU oracle on the same uniforms
    vo, qo, to = (x.clone().requires_grad_() for x in (v, q, t))
    pts_o = torch.cat([O.sample_predict_points("cuboid", vo[:, :kc], qo[:, :kc], to[:, :kc], uc.cpu()),
                       O.sample_predict_points("sphere", vo[:, kc:], qo[:, kc:], to[:, kc:], us.cpu())], dim=1)
    close(out["points"], pts_o, rtol=0, atol=1e-6, what="points vs oracle (libm ulps)")
    verts_o, faces_o = oracle_mesh(O, kc, vo, qo, to)
    ref = (O.chamfer_dense(pts_o, target) + O.chamfer_dense(to, target, w1=0.5, w2=1.0) * 0.1
           + O.silhouette_loss(verts_o, faces_o, gt, torch.ones(b), torch.zeros(b), torch.zeros(b)) * 1.0)
    ref.backward()
    close(out["total"], ref, rtol=1e-4, what="loss vs oracle")
    for got, want, nm in ((vc.grad, vo.grad, "v"), (qc.grad, qo.grad, "q"), (tc.grad, to.grad, "t")):
        close(got, want, rtol=0, atol=1e-4 * float(want.abs().max()), what=f"grad {nm} vs oracle")


def test_vertex_chamfer_emd_path_matches_public_ops(vpn, O):
    """train_gcn.py-style vertex path (Chamfer + VP-diverse + EMD on the composed mesh vertices) on a mixed assembly."""
    from vpn_b200 import templates
    b, kc, ks = 2, 6, 10
    k = kc + ks
    tc, ts_ = templates.template("cuboid", "cuda")[0], templates.template("sphere", "cuda")[0]
    m = kc * tc.shape[0] + ks * ts_.shape[0]
    v, q, t = O.synthetic_primitives(b, k, seed=43)
    t = t * 0.3
    tgt = ((torch.rand(b, m, 3, generator=torch.Generator().manual_seed(43)) - 0.5) * 0.8).cuda()
    cfg = vpn.PrimitiveLossConfig(kind="mixed", n_cuboids=kc, l_view_cd=1.0, l_vp_div=0.1, l_emd=1.0, vertex_chamfer=True)
    vc, qc, tcc = (x.cuda().requires_grad_() for x in (v, q, t))
    out = vpn.PrimitiveLoss(cfg)(vc, qc, tcc, None, tgt)
    out["total"].backward()
    vr, qr, tr = (x.cuda().requires_grad_() for x in (v, q, t))
    pts = vpn.mesh_vertices_mixed(kc, tc, ts_, vr, qr, tr)
    same_bits(out["points"], pts, "vertices")
    terms = {"view_cd": vpn.chamfer_distance(pts, tgt) * 1.0,
             "vp_div": vpn.chamfer_distance(tr.contiguous(), tgt, w1=0.5, w2=1.0) * 0.1,
             "emd": vpn.emd_distance(pts, tgt, 0.005, 50) * 1.0}
    total = terms["view_cd"] + terms["vp_div"] + terms["emd"]
    total.backward()
    for name, want in terms.items():
        close(out[name], want, rtol=1e-6, what=name)
    close(out["total"], total, rtol=1e-6, what="total")
    assert float(out["emd"].detach()) > 0
    for got, want, nm in ((vc.grad, vr.grad, "v"), (qc.grad, qr.grad, "q"), (tcc.grad, tr.grad, "t")):
        close(got, want, rtol=1e-5, atol=1e-7, what=f"grad {nm}")


@pytest.mark.parametrize("kc", [5, 0, 16])
def test_graphed_mixed_step_matches_eager(vpn, O, kc):
    """Uniforms drawn in the graph (u_cuboid, then u_sphere), silhouette on its own stream: captured once, replayed twice
    with new inputs the second time, equal to the eager step under the same device seed.  The mixed step launches as many
    of our kernels as a single-kind step with the same K and terms."""
    b, k, n, m, res = 2, 16, 128, 2048, 32
    v, q, t = O.synthetic_primitives(b, k, seed=61)
    t = t * 0.3
    g = torch.Generator().manual_seed(61)
    tgt = (torch.rand(b, m, 3, generator=g) - 0.5) * 0.8
    gt = (torch.rand(b, 1, res, res, generator=g) > 0.5).float()
    C = lambda x: x.cuda()
    cfg = vpn.PrimitiveLossConfig(kind="mixed", n_cuboids=kc, l_sil=1.0)
    gr = vpn.GraphedPrimitiveLoss(cfg, C(v), C(q), C(t), C(tgt), C(gt), n_samples=n)
    single = vpn.GraphedPrimitiveLoss(vpn.PrimitiveLossConfig(kind="cuboid", l_sil=1.0), C(v), C(q), C(t), C(tgt), C(gt),
                                      n_samples=n)
    assert gr.launches_per_step == single.launches_per_step
    for i, (scale, shift) in enumerate(((1.0, 0.0), (0.8, 0.04))):
        vc, qc, tc = C(v * scale).requires_grad_(), C(q).requires_grad_(), C(t + shift).requires_grad_()
        tg = C(tgt * scale)
        torch.cuda.manual_seed(300 + i)
        loss, gv, gq, gtt = (x.clone() for x in gr(vc.detach(), qc.detach(), tc.detach(), tg, C(gt)))
        torch.cuda.manual_seed(300 + i)
        u = (torch.rand((b, kc, n, 3), device="cuda"), torch.rand((b, k - kc, n, 2), device="cuda"))
        out = vpn.PrimitiveLoss(cfg)(vc, qc, tc, u, tg, silhouettes=C(gt))
        out["total"].backward()
        assert float(out["sil"].detach()) > 0
        close(loss, out["total"], rtol=1e-6)
        close(gv, vc.grad, rtol=1e-5, atol=1e-7); close(gq, qc.grad, rtol=1e-5, atol=1e-7); close(gtt, tc.grad, rtol=1e-5, atol=1e-7)


def test_host_pipeline_feeds_the_graphed_mixed_step(vpn, O):
    """HostPipeline needs nothing mixed-specific: pinned host batches through the graphed mixed vertex step come back in
    order and equal to direct calls (to the repeatability of the silhouette backward's atomics)."""
    b, kc, k, res = 2, 6, 16, 32
    m = kc * 128 + (k - kc) * 128
    cfg = vpn.PrimitiveLossConfig(kind="mixed", n_cuboids=kc, l_sil=1.0, vertex_chamfer=True)
    batches = []
    for s in range(4):
        v, q, t = O.synthetic_primitives(b, k, seed=70 + s)
        g = torch.Generator().manual_seed(70 + s)
        batches.append({"v": v.pin_memory(), "q": q.pin_memory(), "t": (t * 0.3).pin_memory(),
                        "target": ((torch.rand(b, m, 3, generator=g) - 0.5) * 0.8).pin_memory(),
                        "sil": (torch.rand(b, 1, res, res, generator=g) > 0.5).float().pin_memory()})
    d0 = {key: x.cuda() for key, x in batches[0].items()}
    gr = vpn.GraphedPrimitiveLoss(cfg, d0["v"], d0["q"], d0["t"], d0["target"], d0["sil"])
    want = []
    for bt in batches:
        d = {key: x.cuda() for key, x in bt.items()}
        want.append([x.cpu().clone() for x in gr(d["v"], d["q"], d["t"], d["target"], d["sil"])])
    pipe = vpn.HostPipeline(lambda s: gr(s["v"], s["q"], s["t"], s["target"], s["sil"]), d0, "cuda")
    got = []
    pipe.submit(batches[0])
    for bt in batches[1:]:
        pipe.submit(bt)
        got.append([x.clone() for x in pipe.result()])
    got.append([x.clone() for x in pipe.result()])
    for gw, ww in zip(got, want):                                 # the backward scatters with atomics: not bitwise repeatable
        close(gw[0], ww[0], rtol=1e-6)
        for x, y in zip(gw[1:], ww[1:]):
            close(x, y, rtol=1e-5, atol=1e-7)
