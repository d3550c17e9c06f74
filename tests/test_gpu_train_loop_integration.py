"""The training scripts' loop helpers, restated, run against the drop-in `modules` package and compared with the CPU oracle.

The helpers of train.py:105-195, train_sphere.py:62-80 and train_gcn.py:56-95 call the hot-path modules in the order and
with the arguments SURVEY.md section 3 records.  The scripts are not part of this repository, so `helpers()` restates
those calls from that record, reading the same `config` constants, and every result and gradient is compared with the
CPU oracle.  A call in the real scripts that differs from the record (another keyword or argument order) is not caught.
"""
import os
import sys

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
RTOL = 1e-4


def close(a, b, rtol=RTOL, atol=1e-6, what=""):
    a = a.detach().cpu().numpy() if isinstance(a, torch.Tensor) else np.asarray(a)
    b = b.detach().cpu().numpy() if isinstance(b, torch.Tensor) else np.asarray(b)
    np.testing.assert_allclose(a, b, rtol=rtol, atol=atol, err_msg=what)


@pytest.fixture(scope="module")
def O():
    from oracle import vpn_oracle
    return vpn_oracle


def helpers(script, **overrides):
    """Namespace of one training script's helpers, bound to the drop-in modules (what the script's imports resolve to
    when volumetric-primitives-net_b200/ is first on sys.path); `overrides` replace config constants."""
    import config
    from modules.loss import ChamferDistanceLoss, EarthMoverDistanceLoss, SilhouetteLoss, VPDiverseLoss
    from modules.meshing import Meshing
    from modules.sampling import Sampling
    from modules.transform import view_to_obj_points
    c = {k: getattr(config, k) for k in dir(config) if k.isupper()}
    c.update(overrides)
    spheres_only = script == "train_gcn"                          # train_gcn.py: 16 spheres, hard-coded

    def sample_predict_points(volumes, rotates, translates):      # train.py:105-120: per primitive, then cat
        points = []
        for i in range(len(volumes)):
            cuboid = not spheres_only and i < c["CUBOID_NUM"]
            sampling = Sampling.cuboid_sampling if cuboid else Sampling.sphere_sampling
            points.append(sampling(volumes[i], rotates[i], translates[i], c["SAMPLE_NUM"]))
        return torch.cat(points, dim=1)

    def get_vp_meshes(volumes, rotates, translates):              # train.py:123-136: per primitive, B meshes each
        meshes = []
        for i in range(len(volumes)):
            cuboid = not spheres_only and i < c["CUBOID_NUM"]
            meshing = Meshing.cuboid_meshing if cuboid else Meshing.sphere_meshing
            meshes.append(meshing(volumes[i], rotates[i], translates[i]))
        return meshes

    def compose_vp_meshes(vp_meshes):                             # train.py:139-149: one mesh per sample
        return [Meshing.compose_meshes([m[b] for m in vp_meshes]) for b in range(len(vp_meshes[0]))]

    def calculate_cd_loss(predict_points, canonical_points, view_center_points, dists, elevs, azims, angles):
        # train.py:152-163: the canonical-frame term is computed even at its default weight L_CAN_CD = 0
        predict_canonical = view_to_obj_points(predict_points, dists, elevs, azims, angles)
        view_cd = ChamferDistanceLoss()(predict_points, view_center_points) * c["L_VIEW_CD"]
        obj_cd = ChamferDistanceLoss()(predict_canonical, canonical_points) * c["L_CAN_CD"]
        return view_cd, obj_cd

    def calculate_silhouette_loss(predict_meshes, silhouettes, dists, elevs, azims):   # train.py:166-176
        if c["L_SIL"] == 0:
            return 0
        if c["IS_VIEW_CENTER"]:                                   # the view-centred camera for every sample
            dists, elevs, azims = torch.ones_like(dists), torch.zeros_like(elevs), torch.zeros_like(azims)
        return SilhouetteLoss()(predict_meshes, silhouettes, dists, elevs, azims) * c["L_SIL"]

    def calculate_vp_div_loss(translates, gt_points):             # train.py:179-185
        return VPDiverseLoss()(translates, gt_points) * c["L_VP_DIV"]

    def calculate_emd_loss(predict_points, gt_points):            # train.py:188-195, train_gcn.py:91-95
        dist, _ = EarthMoverDistanceLoss()(predict_points, gt_points, 0.005, 50)
        return torch.sqrt(dist).mean() * c["L_EMD"]

    def deform_meshes(meshes, vertices_offset):                   # train_sphere.py:62-68
        for b in range(len(meshes)):
            meshes[b].vertices += vertices_offset[b]
        return meshes

    def sample_points(meshes):                                    # train_sphere.py:71-80
        n = c["SAMPLE_NUM"] * (c["CUBOID_NUM"] + c["SPHERE_NUM"] + c["CONE_NUM"])
        return torch.stack([m.sample(n)[0] for m in meshes])

    return dict(locals())


def prim_lists(O, b, k, seed, spread=0.3):
    v, q, t = O.synthetic_primitives(b, k, seed=seed)
    t = t * spread
    leaves = [x.cuda().requires_grad_() for x in (v, q, t)]
    lists = [[x[:, i] for i in range(k)] for x in leaves]          # the network emits per-primitive lists (train.py:240)
    return (v, q, t), leaves, lists


def sphere_uniforms_in_reference_order(seed, b, k, n):
    """The draws Sampling.sphere_sampling makes for primitives 0..K-1 (sphere.py:26-27: elev draw, then azim draw)."""
    torch.manual_seed(seed)
    u = torch.empty(b, k, n, 2)
    for i in range(k):
        u[:, i, :, 0:1] = torch.rand((b, n, 1), device="cuda").cpu()
        u[:, i, :, 1:2] = torch.rand((b, n, 1), device="cuda").cpu()
    return u


def test_train_py_helpers_run_unmodified(O):
    """train.py:243-258 with the reference's default config (16 spheres x 128 samples, B = 8) plus L_SIL switched on."""
    import config
    from vpn_b200 import templates
    b, k, n = config.BATCH_SIZE, config.SPHERE_NUM, config.SAMPLE_NUM
    assert (b, k, n) == (8, 16, 128)
    ns = helpers("train", L_SIL=1.0)
    (v, q, t), (vc, qc, tc), (volumes, rotates, translates) = prim_lists(O, b, k, seed=3)
    g = torch.Generator().manual_seed(5)
    m, res = 2048, 32
    view_center = (torch.rand(b, m, 3, generator=g) - 0.5) * 0.8
    dists = 1.0 + 0.5 * torch.rand(b, generator=g); elevs = 20 + 20.0 * torch.rand(b, generator=g)
    azims = 360.0 * torch.rand(b, generator=g); angles = 360.0 * torch.rand(b, generator=g)
    canonical = view_center * dists[:, None, None]
    sil = (torch.rand(b, 1, res, res, generator=g) > 0.5).float()
    C = lambda x: x.cuda()

    torch.manual_seed(1234)
    predict_points = ns["sample_predict_points"](volumes, rotates, translates)                 # train.py:243
    view_cd, obj_cd = ns["calculate_cd_loss"](predict_points, C(canonical), C(view_center), C(dists), C(elevs), C(azims), C(angles))
    vp_meshes = ns["get_vp_meshes"](volumes, rotates, translates)                              # train.py:249
    predict_meshes = ns["compose_vp_meshes"](vp_meshes)
    sil_loss = ns["calculate_silhouette_loss"](predict_meshes, C(sil), C(dists), C(elevs), C(azims))
    vp_div = ns["calculate_vp_div_loss"](translates, C(view_center))
    emd = ns["calculate_emd_loss"](predict_points, C(view_center))
    total = view_cd + obj_cd + sil_loss + vp_div + emd                                         # train.py:260
    total.backward()

    # oracle on the same uniforms
    u = sphere_uniforms_in_reference_order(1234, b, k, n)
    vo, qo, to = (x.clone().requires_grad_() for x in (v, q, t))
    pts = O.sample_predict_points("sphere", vo, qo, to, u)
    assert predict_points.shape == (b, k * n, 3)
    close(predict_points, pts, atol=1e-6, what="sample_predict_points")
    ref_view = O.chamfer_dense(pts, view_center) * config.L_VIEW_CD
    close(view_cd, ref_view, what="view_cd")
    assert float(obj_cd) == 0.0                                     # L_CAN_CD = 0: computed, weighted by 0 (train.py:160-161)
    tv, tf = templates.template("sphere", "cpu")
    verts, faces = O.compose_primitive_meshes(tv, tf.long(), vo, qo, to)
    assert len(predict_meshes) == b and predict_meshes[0].faces.dtype == torch.int64
    close(torch.stack([mm.vertices for mm in predict_meshes]), verts, atol=1e-6, what="composed vertices")
    assert (predict_meshes[0].faces.cpu() == faces).all()
    # IS_VIEW_CENTER: the silhouette camera is dist 1, elev 0, azim 0 whatever the view parameters are (train.py:172-174)
    ref_sil = O.silhouette_loss(verts, faces, sil, torch.ones(b), torch.zeros(b), torch.zeros(b))
    close(sil_loss, ref_sil, what="silhouette loss", atol=1e-7)
    ref_div = O.chamfer_dense(to, view_center, w1=0.5, w2=1.0) * config.L_VP_DIV
    close(vp_div, ref_div, what="vp_div")
    assert torch.isfinite(emd) and 0.0 < float(emd) < 1.0
    # gradients of everything but the (non-deterministic in the reference) EMD term against autograd through the oracle
    (ref_view + ref_sil + ref_div).backward()
    import vpn_b200
    ve, qe, te = (x.detach().clone().requires_grad_() for x in (vc, qc, tc))
    pe = vpn_b200.sample_primitives("sphere", ve, qe, te, u.cuda())
    d_e, _ = vpn_b200.emd_auction(pe, C(view_center), 0.005, 50)
    torch.sqrt(d_e).mean().backward()
    for got, emd_part, want, nm in ((vc.grad, ve.grad, vo.grad, "v"), (qc.grad, qe.grad, qo.grad, "q"), (tc.grad, te.grad, to.grad, "t")):
        close(got - emd_part, want, rtol=2e-3, atol=3e-4 * float(want.abs().max()), what=f"grad {nm}")


def test_train_gcn_helpers_run_unmodified(O):
    """train_gcn.py:127-132: 16 sphere primitives (hard-coded), any batch size; meshes composed to (B, 2048, 3) vertices."""
    from vpn_b200 import templates
    ns = helpers("train_gcn")
    b, k = 3, 16
    (v, q, t), _, (volumes, rotates, translates) = prim_lists(O, b, k, seed=12)
    torch.manual_seed(99)
    pts = ns["sample_predict_points"](volumes, rotates, translates)
    u = sphere_uniforms_in_reference_order(99, b, k, 128)
    close(pts, O.sample_predict_points("sphere", v, q, t, u), atol=1e-6)
    meshes = ns["compose_vp_meshes"](ns["get_vp_meshes"](volumes, rotates, translates))
    tv, tf = templates.template("sphere", "cpu")
    verts, faces = O.compose_primitive_meshes(tv, tf.long(), v, q, t)
    assert len(meshes) == b and meshes[0].vertices.shape == (2048, 3) and meshes[0].faces.shape == (4032, 3)
    close(torch.stack([m.vertices for m in meshes]), verts, atol=1e-6)
    gt = torch.rand(b, 2048, 3, generator=torch.Generator().manual_seed(1)).cuda()
    vert_batch = torch.stack([m.vertices for m in meshes])
    vert_batch = (vert_batch - vert_batch.min()) / (vert_batch.max() - vert_batch.min())      # EMD wants [0, 1] (emd_module.py:8)
    e = ns["calculate_emd_loss"](vert_batch, gt)
    assert torch.isfinite(e) and float(e) > 0


def test_train_sphere_helpers_run_unmodified(O, golden_templates):
    """train_sphere.py:111-121: deform the 386-vertex sphere by the network's offsets, sample SAMPLE_NUM * vp_num surface
    points per mesh with TriangleMesh.sample, Chamfer to the targets, gradient back to the offsets."""
    import config
    from modules.meshing import TriangleMesh
    ns = helpers("train_sphere")
    b = config.BATCH_SIZE
    n = config.SAMPLE_NUM * (config.CUBOID_NUM + config.SPHERE_NUM + config.CONE_NUM)
    tv = torch.tensor(golden_templates["sphere386_vertices"]); tf = torch.tensor(golden_templates["sphere386_faces"]).long()
    g = torch.Generator().manual_seed(8)
    offsets = (torch.tanh(torch.randn(b, 386, 3, generator=g)) * 0.05)
    target = (torch.rand(b, 1024, 3, generator=g) - 0.5) * 0.9
    off_c = offsets.cuda().requires_grad_()
    meshes = [TriangleMesh.from_tensors(tv.clone().cuda(), tf.cuda()) for _ in range(b)]      # load_sphere_meshes
    meshes = ns["deform_meshes"](meshes, off_c)
    torch.manual_seed(4321)
    pts = ns["sample_points"](meshes)
    assert pts.shape == (b, n, 3)
    from modules.loss import ChamferDistanceLoss
    loss = ChamferDistanceLoss()(pts, target.cuda())
    loss.backward()
    # oracle: the same draws (one torch.rand((1, n, 3)) per mesh, in batch order)
    torch.manual_seed(4321)
    us = [torch.rand((1, n, 3), device="cuda").cpu()[0] for _ in range(b)]
    off_o = offsets.clone().requires_grad_()
    ref_pts = torch.stack([O.mesh_sample(tv + off_o[i], tf, us[i])[0] for i in range(b)])
    close(pts, ref_pts, atol=1e-6, what="sampled surface points")
    ref = O.chamfer_dense(ref_pts, target)
    close(loss, ref, what="train_sphere Chamfer loss")
    ref.backward()
    close(off_c.grad, off_o.grad, rtol=1e-3, atol=1e-4 * float(off_o.grad.abs().max()), what="offset gradient")
