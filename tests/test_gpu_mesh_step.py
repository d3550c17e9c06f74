"""The mesh-loss step of train_sphere.py / train_gcn.py and the mesh sampler's gather backward under it: the backward against
the atomic kernel (vpn_mesh_sample_bwd) and autograd through the CPU oracle, its fixed summation order, and MeshLoss /
GraphedMeshLoss against the oracle and the public ops they compose, eager and replayed from a CUDA graph."""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

RTOL = 1e-4


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


def close(a, b, rtol=RTOL, atol=1e-6, what=""):
    a = a.detach().cpu().numpy() if isinstance(a, torch.Tensor) else np.asarray(a)
    b = b.detach().cpu().numpy() if isinstance(b, torch.Tensor) else np.asarray(b)
    np.testing.assert_allclose(a, b, rtol=rtol, atol=atol, err_msg=what)


def sphere386(golden_templates, b, seed):
    """train_sphere.py's mesh: the 386-vertex sphere deformed by tanh(N) * 0.05 offsets."""
    g = torch.Generator().manual_seed(seed)
    tv = torch.from_numpy(golden_templates["sphere386_vertices"]).float()
    tf = torch.from_numpy(golden_templates["sphere386_faces"]).long()
    offs = torch.tanh(torch.randn(b, tv.shape[0], 3, generator=g)) * 0.05
    return tv, tf, offs, g


def wavy_grid(b, r, seed):
    """An r x r vertex sheet with 2 (r - 1)^2 faces and per-mesh heights: a mesh with many faces."""
    g = torch.Generator().manual_seed(seed)
    y, x = torch.meshgrid(torch.linspace(-0.5, 0.5, r), torch.linspace(-0.5, 0.5, r), indexing="ij")
    base = torch.stack([x, y, 0.1 * torch.sin(6 * x) * torch.cos(5 * y)], -1).reshape(-1, 3)
    verts = base[None] + 0.01 * torch.randn(b, r * r, 3, generator=g)
    i = torch.arange(r - 1)
    q = (i[:, None] * r + i[None, :]).reshape(-1)
    faces = torch.cat([torch.stack([q, q + 1, q + r], 1), torch.stack([q + 1, q + r + 1, q + r], 1)])
    return verts, faces, g


def atomic_bwd(faces, u, fidx, gpoints, nv):
    """The atomic kernel vpn_mesh_sample_bwd, the reference of the gather form."""
    from vpn_b200 import _lib
    from vpn_b200._lib import check, ptr, stream_ptr
    b, n = fidx.shape
    gv = torch.empty((b, nv, 3), device="cuda")
    check(_lib.load().vpn_mesh_sample_bwd(ptr(faces), ptr(u), ptr(fidx), ptr(gpoints), ptr(gv), b, nv, faces.shape[0], n,
                                          stream_ptr(gv.device)), "vpn_mesh_sample_bwd")
    return gv


def sampled_grad(vpn, verts, faces, u, up):
    vd = verts.detach().clone().requires_grad_()
    pts, fidx = vpn.sample_mesh_surface(vd, faces, u)
    (pts * up).sum().backward()
    return vd.grad, fidx


@pytest.mark.parametrize("case", ["sphere-1x16384", "sphere-3x1000", "sphere-2x1", "grid-50", "grid-60"])
def test_sampler_backward_matches_atomic_and_oracle(vpn, O, golden_templates, case):
    """(B, n) of test_mesh_sample_matches_oracle, and meshes of 4802 and 6962 faces (histogram in shared memory / in the
    workspace)."""
    if case.startswith("sphere"):
        b, n = (int(x) for x in case.split("-")[1].split("x"))
        tv, tf, offs, g = sphere386(golden_templates, b, 3)
        verts, faces = tv[None] + offs, tf
    else:
        b, n = 2, 20000
        verts, faces, g = wavy_grid(b, int(case.split("-")[1]), 4)
        assert faces.shape[0] > 4096
    u = torch.rand(b, n, 3, generator=g)
    up = torch.rand(b, n, 3, generator=g)
    fc = C(faces).int()
    gv, fidx = sampled_grad(vpn, C(verts), fc, C(u), C(up))
    ref = atomic_bwd(fc, C(u), fidx, C(up), verts.shape[1])
    close(gv, ref, rtol=RTOL, atol=1e-5 * float(ref.abs().max()), what="vs atomic kernel")
    for i in range(b):
        vo = verts[i].clone().requires_grad_()
        po, fo = O.mesh_sample(vo, faces, u[i])
        assert torch.equal(fidx[i].long().cpu(), fo)
        (po * up[i]).sum().backward()
        close(gv[i], vo.grad, rtol=RTOL, atol=1e-5 * float(vo.grad.abs().max()), what=f"vs oracle, mesh {i}")


def test_sampler_backward_is_fixed_order(vpn, golden_templates):
    """Two calls give the same bits, and a mesh alone gives the bits it gets at position 2 of a batch of 4."""
    tv, tf, offs, g = sphere386(golden_templates, 4, 7)
    n = 16384
    verts, faces = C(tv[None] + offs), C(tf).int()
    u, up = C(torch.rand(4, n, 3, generator=g)), C(torch.rand(4, n, 3, generator=g))
    first, _ = sampled_grad(vpn, verts, faces, u, up)
    again, _ = sampled_grad(vpn, verts, faces, u, up)
    assert torch.equal(first, again)
    alone, _ = sampled_grad(vpn, verts[2:3], faces, u[2:3], up[2:3])
    assert torch.equal(alone[0], first[2])


def test_face_without_samples_contributes_zero(vpn, golden_templates):
    """With 3 samples, every vertex outside the sampled faces gets exactly 0 (the output is fully written, not
    accumulated into memory the caller zeroed)."""
    tv, tf, offs, g = sphere386(golden_templates, 2, 11)
    faces = C(tf).int()
    u, up = C(torch.rand(2, 3, 3, generator=g)), C(torch.rand(2, 3, 3, generator=g) + 0.5)
    gv, fidx = sampled_grad(vpn, C(tv[None] + offs), faces, u, up)
    for i in range(2):
        touched = torch.zeros(tv.shape[0], dtype=torch.bool)
        touched[tf[fidx[i].long().cpu()].reshape(-1)] = True
        assert torch.count_nonzero(gv[i].cpu()[~touched]) == 0
        assert bool((gv[i].cpu()[touched].abs().sum(1) > 0).all())


@pytest.mark.parametrize("l_sil", [0.0, 1.0])
def test_sampled_path_matches_oracle_and_public_ops(vpn, O, golden_templates, l_sil):
    """train_sphere.py: verts = template + offsets, n area-weighted samples, Chamfer (+ the silhouette) - against the CPU
    oracle (tolerances of test_train_sphere_helpers_run_unmodified) and against the public ops on the same draws."""
    b, n, m, res = 2, 2048, 1024, 32
    tv, tf, offs, g = sphere386(golden_templates, b, 8)
    target = (torch.rand(b, m, 3, generator=g) - 0.5) * 0.9
    gt = (torch.rand(b, 1, res, res, generator=g) > 0.5).float()
    u = torch.rand(b, n, 3, generator=g)
    cfg = vpn.MeshLossConfig(n_samples=n, l_sil=l_sil)
    faces = C(tf).int()
    off_c = C(offs).requires_grad_()
    out = vpn.MeshLoss(cfg)(C(tv)[None] + off_c, faces, C(target), uniforms=C(u), silhouettes=C(gt) if l_sil else None)
    out["total"].backward()
    assert set(out) == {"points", "cd", "total"} | ({"sil", "alpha"} if l_sil else set())
    # oracle
    off_o = offs.clone().requires_grad_()
    vo = tv[None] + off_o
    ref_pts = torch.stack([O.mesh_sample(vo[i], tf, u[i])[0] for i in range(b)])
    close(out["points"], ref_pts, atol=1e-6, what="sampled surface points")
    ref = O.chamfer_dense(ref_pts, target)
    if l_sil:
        ref = ref + O.silhouette_loss(vo, tf, gt, torch.ones(b), torch.zeros(b), torch.zeros(b)) * l_sil
    close(out["total"], ref, what="loss vs oracle")
    ref.backward()
    close(off_c.grad, off_o.grad, rtol=1e-3, atol=1e-4 * float(off_o.grad.abs().max()), what="offset gradient")
    # the same terms from the public ops
    vr = C(tv)[None] + C(offs)
    pts, _ = vpn.sample_mesh_surface(vr, faces, C(u))
    want = vpn.chamfer_distance(pts, C(target))
    if l_sil:
        rot, pos = vpn.look_at_cameras(torch.zeros(b, device="cuda"), torch.zeros(b, device="cuda"), torch.ones(b, device="cuda"))
        alpha = vpn.soft_silhouette(vr, faces, rot, pos, res, res)[0]
        close(out["alpha"], alpha, rtol=0, atol=0, what="alpha")
        want = want + (alpha[:, None] - C(gt)).abs().mean() * l_sil
    close(out["total"], want, rtol=1e-6, atol=0, what="loss vs public ops")


def composed_spheres(vpn, b, seed):
    """train_gcn.py's output: 2048 vertices of 16 composed spheres (4032 faces), coordinates in [0, 1]."""
    g = torch.Generator().manual_seed(seed)
    faces = vpn.PrimitiveLoss().composed_faces(16, "cuda")
    verts = torch.rand(b, 2048, 3, generator=g) * 0.6 + 0.2
    target = torch.rand(b, 2048, 3, generator=g) * 0.8 + 0.1
    return verts, faces, target, g


def test_vertex_path_matches_public_ops(vpn):
    """train_gcn.py: Chamfer + EMD on the predicted vertices; `points` is the vertex tensor itself."""
    b = 2
    verts, faces, target, _ = composed_spheres(vpn, b, 5)
    cfg = vpn.MeshLossConfig(n_samples=0, l_emd=1.0)
    vc = C(verts).requires_grad_()
    out = vpn.MeshLoss(cfg)(vc, faces, C(target))
    out["total"].backward()
    assert out["points"] is vc
    vr = C(verts).requires_grad_()
    terms = {"cd": vpn.chamfer_distance(vr, C(target)), "emd": vpn.emd_distance(vr, C(target), 0.005, 50)}
    total = terms["cd"] + terms["emd"]
    total.backward()
    for name, want in terms.items():
        close(out[name], want, rtol=1e-6, atol=0, what=name)
    close(out["total"], total, rtol=1e-6, atol=0, what="total")
    close(vc.grad, vr.grad, rtol=1e-5, atol=1e-7, what="grad verts")


@pytest.mark.parametrize("n_samples", [2048, 0])
def test_graphed_step_matches_eager(vpn, n_samples):
    """Silhouette and EMD forked onto their streams; captured once, replayed twice with new inputs the second time; equal
    to the eager step.  The sampled path draws its uniforms in the graph: the device RNG is seeded the same for both."""
    b, res = 2, 32
    verts, faces, target, g = composed_spheres(vpn, b, 9)
    gt = (torch.rand(b, 1, res, res, generator=g) > 0.5).float()
    cfg = vpn.MeshLossConfig(n_samples=n_samples, l_sil=1.0, l_emd=1.0)
    gr = vpn.GraphedMeshLoss(cfg, C(verts), faces, C(target), C(gt))
    no_emd = vpn.GraphedMeshLoss(vpn.MeshLossConfig(n_samples=n_samples, l_sil=1.0), C(verts), faces, C(target), C(gt))
    assert gr.launches_per_step == no_emd.launches_per_step + 4           # auction, loss head (2), backward
    if n_samples:
        vertex = vpn.GraphedMeshLoss(vpn.MeshLossConfig(n_samples=0, l_sil=1.0, l_emd=1.0), C(verts), faces, C(target), C(gt))
        assert gr.launches_per_step == vertex.launches_per_step + 5       # sampler: forward 2, backward 3
    for i, (scale, shift) in enumerate(((1.0, 0.0), (0.9, 0.03))):
        vin, tin = C(verts * scale + shift), C(target * scale + shift)
        torch.cuda.manual_seed(100 + i)
        loss, gv = gr(vin, tin, C(gt))
        loss, gv = loss.clone(), gv.clone()
        torch.cuda.manual_seed(100 + i)
        vc = vin.clone().requires_grad_()
        out = vpn.MeshLoss(cfg)(vc, faces, tin, silhouettes=C(gt))
        out["total"].backward()
        assert float(out["emd"].detach()) > 0 and float(out["sil"].detach()) > 0
        close(loss, out["total"], rtol=1e-6, atol=0)
        close(gv, vc.grad, rtol=1e-5, atol=1e-7)
