"""The soft-silhouette rasteriser (csrc/silhouette.cu) at its edges, against the DIB-R restatement
oracle.vpn_oracle.soft_silhouette: ragged, rectangular and tiny images (partial 16 x 16 tiles, H != W), the knum cut-off
at knum 1..32, face indices above 32767 in the 16-bit candidate lists and the F limit, poisoned samples (NaN vertex,
vertex on the camera plane) and batch isolation, sparse upstream gradients, and the six distance cases plus the
foot-off-segment constant one at a time (with a float64 check of the backward's closed form).

Bars as in test_gpu_render_parity.py: alpha rtol 1e-4 / atol 2e-6 with the alpha == 1 set identical, `covered`
bit-exact, vertex gradients rtol 1e-3 / atol 1e-4 max|g_ref|; exact properties (fixed-order forward, zero gradients)
are asserted bit for bit.  The scenes are built in screen space for the default camera (dist 1, elev 0, azim 0), and
each scene's premise (what it is meant to exercise) is asserted with the oracle's own selection logic; the premises
that need no GPU also run in test_raster_edges_premises.py."""
import ctypes
import math

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

RTOL = 1e-4
VPN_ERR_SHAPE, VPN_ERR_ARG = -2, -3
RAGGED = [(48, 80, "sphere"), (80, 48, "cuboid"), (17, 33, "cuboid"), (137, 137, "sphere"), (1, 1, "cuboid"),
          (5, 3, "sphere"), (1, 37, "cuboid"), (130, 16, "sphere")]


def _oracle():
    from oracle import vpn_oracle
    return vpn_oracle


@pytest.fixture(scope="module")
def vpn():
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    import vpn_b200
    return vpn_b200


@pytest.fixture(scope="module")
def O():
    return _oracle()


def C(a):
    return torch.as_tensor(np.asarray(a)).cuda()


def close(a, b, rtol=RTOL, atol=1e-6, what=""):
    a = a.detach().cpu().numpy() if isinstance(a, torch.Tensor) else np.asarray(a)
    b = b.detach().cpu().numpy() if isinstance(b, torch.Tensor) else np.asarray(b)
    np.testing.assert_allclose(a, b, rtol=rtol, atol=atol, err_msg=what)


def same(a, b, what=""):
    a = a.detach().cpu().numpy() if isinstance(a, torch.Tensor) else np.asarray(a)
    b = b.detach().cpu().numpy() if isinstance(b, torch.Tensor) else np.asarray(b)
    np.testing.assert_array_equal(a, b, err_msg=what)


# ------------------------------------------------------------------------------------------------
# scenes (CPU, oracle only)
# ------------------------------------------------------------------------------------------------
def _screen_scale():
    """Scaled screen units per world unit on the plane x = 0 of the default camera: (0, y, z) -> (-z, y) * this."""
    return float(_oracle().projection_vector()[0]) * 1000.0


def default_camera(b):
    rot, pos = _oracle().look_at_camera(0.0, 0.0, 1.0)
    return rot[None].repeat(b, 1, 1).contiguous(), pos[None].repeat(b, 1).contiguous()


def to_world(sxy):
    """(..., 2) scaled screen coordinates -> (..., 3) points on the plane x = 0 that project there (to rounding)."""
    p = _screen_scale()
    sxy = torch.as_tensor(sxy, dtype=torch.float64)
    return torch.stack([torch.zeros_like(sxy[..., 0]), sxy[..., 1] / p, -sxy[..., 0] / p], -1).float()


# Primitive centres and radii in scaled screen units (the image spans [-1000, 1000] in X and Y): silhouettes that
# cross the last, partial tile row and column of every ragged size, the image centre, and the one row of 1 x 37.
SPOTS = [(880.0, -880.0, 260.0), (930.0, 250.0, 160.0), (-350.0, -930.0, 180.0), (0.0, 0.0, 330.0),
         (-650.0, 620.0, 120.0), (790.0, -30.0, 110.0)]


def spot_scene(kind, b=2, seed=3):
    """Sample i: the SPOTS primitives of one template, radii x (1 - 0.15 i), random orientations."""
    O = _oracle()
    from vpn_b200 import templates
    tv, tf = templates.template(kind, "cpu")
    p = _screen_scale()
    k = len(SPOTS)
    _, q, _ = O.synthetic_primitives(b, k, seed=seed)
    v = torch.stack([torch.tensor([[r * (1 - 0.15 * i) / p] * 3 for _, _, r in SPOTS]) for i in range(b)])
    t = torch.stack([to_world(torch.tensor([[x, y] for x, y, _ in SPOTS]))] * b)
    verts, faces = O.compose_primitive_meshes(tv, tf.long(), v, q, t)
    return verts.detach().contiguous(), faces


def ragged_mask(h, w):
    """Pixels of the partial tiles (the last tile row / column when H or W is not a multiple of 16)."""
    m = torch.zeros(h, w, dtype=torch.bool)
    m[(h // 16) * 16:, :] = True
    m[:, (w // 16) * 16:] = True
    return m


def ragged_pixels(h, w, n_other=600, seed=0):
    """137 x 137: every partial-tile pixel and a random sample of the rest (keeps the dense oracle small)."""
    rag = ragged_mask(h, w).flatten()
    other = (~rag).nonzero().flatten()
    gen = torch.Generator().manual_seed(seed)
    return torch.cat([rag.nonzero().flatten(), other[torch.randperm(other.numel(), generator=gen)[:n_other]]]).sort()[0]


def ragged_premise(ref, h, w, pixels=None):
    """Every sample has covered pixels in the partial tiles (anywhere, for the whole-tile sizes), and from 37 pixels up
    soft ones too: a partial tile left out, or pixel centres misplaced, changes what is compared."""
    rag = ragged_mask(h, w).flatten()
    if pixels is not None:
        rag = rag[pixels]
    if not rag.any():
        rag = torch.ones_like(rag)
    a = ref.reshape(ref.shape[0], -1)
    assert ((a == 1) & rag).any(1).all(), "premise: covered pixels in the partial tiles of every sample"
    if h * w >= 37:
        assert ((a > 0) & (a < 1) & rag).any(), "premise: soft pixels in the partial tiles"


# Fans for the knum cut-off: around each chosen pixel centre, FAN_N small triangles that all hold the pixel in their
# expanded box and none contains it.  Distances grow with the face index, so the first knum and the last knum differ;
# every fourth triangle is wound the other way (a back face), so the two back-face rules keep different sets.  Each
# points its apex at the pixel (a vertex case): an edge of 5 units ~500 units from the origin cancels too much in
# float32 (C = x2 y1 - x1 y2) for the kernel's closed form and the oracle's autograd to agree to 1e-3.
KNUM_HW = (40, 24)
KNUM_PIXELS = [(5, 3), (20, 17), (37, 22)]        # (h, w); the last one lies in a partial tile
FAN_N = 48


def pixel_centre(h, w, H, W):
    X, Y = _oracle()._sil_pixel_centres(H, W)
    return float(X[h * W + w]), float(Y[h * W + w])


def knum_scene(reverse=False):
    tris = []
    for (h, w) in KNUM_PIXELS:
        cx, cy = pixel_centre(h, w, *KNUM_HW)
        for i in range(FAN_N):
            th = 2 * math.pi * (i * 7 % FAN_N) / FAN_N + 0.05 * (h % 3)
            r = 11.0 + 7.5 * i / FAN_N
            u, n = np.array([math.cos(th), math.sin(th)]), np.array([-math.sin(th), math.cos(th)])
            c = np.array([cx, cy])
            tri = [c + r * u, c + (r + 5) * u + 2.5 * n, c + (r + 5) * u - 2.5 * n]
            if i % 4 != 3:
                tri = [tri[0], tri[2], tri[1]]
            tris.append(tri)
    verts = to_world(torch.tensor(np.array(tris)).reshape(-1, 2))[None].contiguous()
    faces = torch.arange(verts.shape[1]).reshape(-1, 3)
    return verts, (faces.flip(0) if reverse else faces).contiguous()


# 16-bit candidate lists: the live faces (one sphere, F = 252) at the end of a 65535-face array; the padding faces
# lie in front of the camera far outside the image, so their 32-face groups are culled whole.
WIDE_F = 65535
WIDE_HW = (40, 56)


def wide_scene():
    O = _oracle()
    from vpn_b200 import templates
    tv, tf = templates.template("sphere", "cpu")
    p = _screen_scale()
    _, q, _ = O.synthetic_primitives(1, 1, seed=11)
    live_v, live_f = O.compose_primitive_meshes(tv, tf.long(), torch.full((1, 1, 3), 420.0 / p), q,
                                                to_world(torch.tensor([[[60.0, -40.0]]])))
    pad_v = to_world(torch.tensor([[5000.0, 5000.0], [5100.0, 5000.0], [5000.0, 5100.0]]))[None]
    nv, n_live = live_v.shape[1], live_f.shape[0]
    verts = torch.cat([live_v.detach(), pad_v], 1).contiguous()
    pad_f = torch.tensor([nv, nv + 1, nv + 2]).repeat(WIDE_F - n_live, 1)
    faces = torch.cat([pad_f, live_f]).contiguous()
    return verts, faces, nv, WIDE_F - n_live


# Distance cases: sample 0 is one large triangle whose neighbourhood holds all six cases; sample 1 is a needle
# (one edge of 600 000 units at a slope of 1/250) whose expanded box reaches pixels more than 2000 units (d2 > 4 mult^2)
# from every vertex with every perpendicular foot off its segment: the foot-off constant wins there.
CASES_HW = (256, 256)


def cases_scene():
    tri = torch.tensor([[[-600.0, -500.0], [700.0, -300.0], [-100.0, 650.0]],
                        [[-500.0, -1500.0], [500.0, -2000.0], [599500.0, 920.0]]])
    return to_world(tri).contiguous(), torch.tensor([[0, 1, 2]])


def case_pixels(sel, alpha, b):
    """Per case 0..5 (edge 0-2 with the foot on the segment, vertex 0-2) and 6 (foot-off constant): the uncovered
    candidate pixel of sample b where that case wins, from the oracle's own selection, -1 where it does not occur.
    With one face alpha is that face's probability: the pixel with alpha nearest 1/2 (about 10 units from the
    feature) is taken, so that the gradient is large and the edge term A X + B Y + C does not cancel to a few units."""
    use, case, const = sel["use"][b][:, 0], sel["case"][b][:, 0], sel["const"][b][:, 0]
    kind = torch.where(const, torch.full_like(case, 6), case)
    out = []
    for c in range(7):
        idx = (use & (kind == c)).nonzero().flatten()
        out.append(int(idx[torch.argmin((alpha[b].flatten()[idx] - 0.5).abs())]) if idx.numel() else -1)
    return out


# ------------------------------------------------------------------------------------------------
# device calls
# ------------------------------------------------------------------------------------------------
def abi_fwd(vpn, verts, faces, rot, pos, h, w, cull, knum):
    """vpn_silhouette_fwd at any knum; returns (rc, alpha, covered, workspace)."""
    from vpn_b200 import _lib, ops
    from vpn_b200._lib import check, ptr, stream_ptr
    lib = _lib.load()
    verts, faces, rot, pos = (x.cuda().contiguous() for x in (verts, faces.int(), rot, pos))
    b, v, _ = verts.shape
    f = faces.shape[0]
    nb = ctypes.c_size_t(0)
    check(lib.vpn_silhouette_workspace_bytes(b, v, f, ctypes.byref(nb)), "workspace")
    ws = torch.empty(nb.value, dtype=torch.uint8, device="cuda")
    alpha = torch.empty(b, h, w, device="cuda")
    covered = torch.empty(b, h, w, dtype=torch.uint8, device="cuda")
    px, py, pz = ops.projection_vector()
    rc = lib.vpn_silhouette_fwd(ptr(verts), ptr(faces), ptr(rot), ptr(pos), px, py, pz, ops.DIBR_EXPAND, knum,
                                ops.DIBR_MULTIPLIER, ops.DIBR_DELTA, int(cull), ptr(alpha), ptr(covered), None, ptr(ws),
                                nb.value, b, v, f, h, w, stream_ptr("cuda"))
    return rc, alpha, covered, (ws, faces, rot, b, v, f)


def abi_bwd(vpn, state, galpha, covered, h, w, cull, knum, grad_verts=None):
    from vpn_b200 import _lib, ops
    from vpn_b200._lib import ptr, stream_ptr
    lib = _lib.load()
    ws, faces, rot, b, v, f = state
    gv = torch.empty(b, v, 3, device="cuda") if grad_verts is None else grad_verts
    galpha = galpha.cuda().contiguous()
    px, py, pz = ops.projection_vector()
    rc = lib.vpn_silhouette_bwd(ptr(faces), ptr(rot), px, py, pz, ops.DIBR_EXPAND, knum, ops.DIBR_MULTIPLIER,
                                ops.DIBR_DELTA, int(cull), ptr(galpha), ptr(covered), ptr(gv),
                                ptr(ws), ws.numel(), b, v, f, h, w, stream_ptr("cuda"))
    assert rc == 0, rc
    return gv


def device_camera(vpn, b):
    """The default camera computed on the device (the oracle is given the same fp32 values)."""
    zero = torch.zeros(b, device="cuda")
    return vpn.look_at_cameras(zero, zero, zero + 1.0)


def render(vpn, verts, faces, h, w, cull):
    """ops.soft_silhouette with the device's default cameras; returns (alpha, covered, verts leaf, rot, pos)."""
    r_c, p_c = device_camera(vpn, verts.shape[0])
    vg = verts.cuda().clone().requires_grad_()
    alpha, covered, _ = vpn.soft_silhouette(vg, faces.cuda().int(), r_c, p_c, h, w, soft_cull_backfaces=cull)
    return alpha, covered, vg, r_c, p_c


def oracle_alpha_grad(O, verts, faces, rot, pos, h, w, cull, upstream, pixels=None, knum=30):
    """Oracle alpha (B,H,W) or (B,P), the vertex gradient of sum(alpha * upstream) and the coverage flags."""
    vr = verts.detach().cpu().clone().requires_grad_()
    args = (faces.long().cpu(), rot.cpu(), pos.cpu(), h, w, cull)
    ref = O.soft_silhouette(vr, *args, pixels=pixels, knum=knum)
    (ref * upstream.reshape(ref.shape)).sum().backward()
    cov = torch.stack(O.soft_silhouette_selection(verts.detach().cpu(), *args, pixels=pixels, knum=knum)["covered"])
    return ref.detach(), vr.grad, cov.reshape(ref.shape)


def check_alpha(alpha, covered, ref, ref_cov, what):
    """alpha to the bar, the alpha == 1 set identical, `covered` bit-exact (a soft alpha can round to 1 too)."""
    close(alpha, ref, rtol=RTOL, atol=2e-6, what=f"{what}: alpha")
    assert ((alpha.detach().cpu() == 1.0) == (ref == 1.0)).all(), f"{what}: alpha == 1 set differs"
    same(covered.cpu().bool(), ref_cov, f"{what}: covered")


def check_grad(got, ref, what):
    close(got, ref, rtol=1e-3, atol=1e-4 * float(ref.abs().max()), what=f"{what}: vertex gradient")


# ------------------------------------------------------------------------------------------------
# 2. ragged, rectangular and tiny images
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("cull", [False, True])
@pytest.mark.parametrize("h,w,kind", RAGGED, ids=[f"{h}x{w}-{k}" for h, w, k in RAGGED])
def test_ragged_rectangular_tiny(vpn, O, h, w, kind, cull):
    """alpha, covered and vertex gradients (random upstream over every compared pixel) at sizes that are not multiples
    of 16, not square, or smaller than one tile; the silhouettes cross the partial tiles."""
    verts, faces = spot_scene(kind)
    b = verts.shape[0]
    alpha, covered, vg, r_c, p_c = render(vpn, verts, faces, h, w, cull)
    pixels = ragged_pixels(h, w) if (h, w) == (137, 137) else None
    n = h * w if pixels is None else pixels.numel()
    up = torch.rand(b, n, generator=torch.Generator().manual_seed(h * 1000 + w))
    ref, gref, rcov = oracle_alpha_grad(O, verts, faces, r_c, p_c, h, w, cull, up, pixels=pixels)
    got_a, got_c = alpha.reshape(b, -1), covered.reshape(b, -1)
    if pixels is not None:
        got_a, got_c = got_a[:, pixels.cuda()], got_c[:, pixels.cuda()]
    check_alpha(got_a, got_c, ref.reshape(b, -1), rcov.reshape(b, -1), f"{h}x{w}")
    ragged_premise(ref, h, w, pixels)
    wg = torch.zeros(b, h * w)
    wg[:, slice(None) if pixels is None else pixels] = up
    (alpha * wg.view(b, h, w).cuda()).sum().backward()
    check_grad(vg.grad, gref, f"{h}x{w}")


def test_step_rectangular_silhouette(vpn, O):
    """PrimitiveLoss(l_sil, vertex_chamfer) with 48 x 80 ground-truth silhouettes: the step takes H and W from them."""
    from vpn_b200 import templates
    b, k, (h, w) = 2, 4, (48, 80)
    v, q, t = O.synthetic_primitives(b, k, seed=9); t = t * 0.25; v = v * 1.5
    g = torch.Generator().manual_seed(2)
    tgt = (torch.rand(b, 256, 3, generator=g) - 0.5) * 0.8
    gt = (torch.rand(b, 1, h, w, generator=g) > 0.5).float()
    cfg = vpn.PrimitiveLossConfig(kind="sphere", l_sil=1.0, l_view_cd=0.0, l_vp_div=0.0, vertex_chamfer=True)
    vc, qc, tc = (C(x).requires_grad_() for x in (v, q, t))
    out = vpn.PrimitiveLoss(cfg)(vc, qc, tc, None, C(tgt), silhouettes=C(gt))
    out["total"].backward()
    tv, tf = templates.template("sphere", "cpu")
    vo, qo, to = (x.clone().requires_grad_() for x in (v, q, t))
    verts, faces = O.compose_primitive_meshes(tv, tf.long(), vo, qo, to)
    ref = O.silhouette_loss(verts, faces, gt, torch.ones(b), torch.zeros(b), torch.zeros(b))
    ref.backward()
    close(out["total"], ref, rtol=RTOL, atol=1e-7)
    for got, want, nm in ((vc.grad, vo.grad, "v"), (qc.grad, qo.grad, "q"), (tc.grad, to.grad, "t")):
        close(got, want, rtol=2e-3, atol=3e-4 * float(want.abs().max()), what=f"48x80 grad {nm}")


# ------------------------------------------------------------------------------------------------
# 3. the knum cut-off
# ------------------------------------------------------------------------------------------------
def knum_premise(O, reverse, cull):
    """The fan pixels are uncovered, hold more than 32 soft candidates, and reversing the face order changes alpha."""
    h, w = KNUM_HW
    verts, faces = knum_scene(reverse)
    rot, pos = default_camera(1)
    pix = torch.tensor([hh * w + ww for hh, ww in KNUM_PIXELS])
    sel = O.soft_silhouette_selection(verts, faces, rot, pos, h, w, cull, pixels=pix)
    assert not sel["covered"][0].any(), "premise: fan pixels uncovered"
    n_cand = sel["in_soft"][0].sum(1)
    assert (n_cand > 32).all(), f"premise: more than 32 soft candidates per fan pixel, got {n_cand.tolist()}"
    a = O.soft_silhouette(verts, faces, rot, pos, h, w, cull, pixels=pix)
    ar = O.soft_silhouette(*knum_scene(not reverse), rot, pos, h, w, cull, pixels=pix)
    assert (a != ar).all(), "premise: the face order matters at every fan pixel"
    assert ((a > 0) & (a < 1)).all(), "premise: fan pixels are soft"
    return verts, faces


@pytest.mark.parametrize("cull", [False, True])
@pytest.mark.parametrize("reverse", [False, True])
def test_knum_cutoff(vpn, O, reverse, cull):
    """vpn_silhouette_fwd / _bwd at knum 1, 7, 30, 32 on pixels with more than 32 candidates, both face orders and
    both back-face rules, against the oracle at the same knum."""
    h, w = KNUM_HW
    verts, faces = knum_premise(O, reverse, cull)
    rot, pos = default_camera(1)
    r_c, p_c = device_camera(vpn, 1)
    up = torch.rand(1, h, w, generator=torch.Generator().manual_seed(7))
    alphas = {}
    for knum in (1, 7, 30, 32):
        rc, alpha, covered, state = abi_fwd(vpn, verts, faces, r_c, p_c, h, w, cull, knum)
        assert rc == 0, rc
        ref, gref, rcov = oracle_alpha_grad(O, verts, faces, r_c, p_c, h, w, cull, up, knum=knum)
        check_alpha(alpha, covered, ref, rcov, f"knum {knum}")
        gv = abi_bwd(vpn, state, up, covered, h, w, cull, knum)
        check_grad(gv, gref, f"knum {knum}")
        alphas[knum] = alpha
    fan = torch.tensor([hh * w + ww for hh, ww in KNUM_PIXELS], device="cuda")
    for lo, hi in ((1, 7), (7, 30), (30, 32)):
        assert (alphas[lo].flatten()[fan] < alphas[hi].flatten()[fan]).all(), f"knum {lo} -> {hi} adds factors"


# ------------------------------------------------------------------------------------------------
# 4. 16-bit face indices and the F limit
# ------------------------------------------------------------------------------------------------
def wide_premise(O):
    """Live faces' candidates have indices above 65000 in the padded numbering, reaching into the last group; the
    padding face is no pixel's candidate, so the oracle on the live faces alone is the padded scene's result."""
    h, w = WIDE_HW
    verts, faces, nv, first_live = wide_scene()
    rot, pos = default_camera(1)
    sel = O.soft_silhouette_selection(verts[:, :nv], faces[first_live:], rot, pos, h, w)
    used = sel["use"][0].any(0).nonzero().flatten() + first_live
    assert used.numel() > 32 and used.min() > 65000 and used.max() >= WIDE_F - 32, "premise: candidate indices"
    pad = O.soft_silhouette_selection(verts, faces[:1], rot, pos, h, w)
    assert not pad["in_soft"][0].any() and not pad["covered"][0].any(), "premise: padding faces hold no pixel"
    soft = sel["use"][0].any(1)
    assert soft.sum() > 20, "premise: uncovered pixels with candidates"
    return verts, faces, nv, first_live


@pytest.mark.parametrize("cull", [False, True])
def test_face_indices_above_32767(vpn, O, cull):
    h, w = WIDE_HW
    verts, faces, nv, first_live = wide_premise(O)
    alpha, covered, vg, r_c, p_c = render(vpn, verts, faces, h, w, cull)
    up = torch.rand(1, h, w, generator=torch.Generator().manual_seed(13))
    ref, gref, rcov = oracle_alpha_grad(O, verts[:, :nv], faces[first_live:], r_c, p_c, h, w, cull, up)
    check_alpha(alpha, covered, ref, rcov, "F = 65535")
    (alpha * up.cuda()).sum().backward()
    check_grad(vg.grad[:, :nv], gref, "F = 65535")
    assert (vg.grad[:, nv:] == 0).all(), "padding vertices get no gradient"


def test_face_limit_raises(vpn):
    """F = 65536 does not fit the 16-bit candidate lists: VpnError through ops (the C ABI code is checked on the CPU)."""
    verts = torch.rand(1, 3, 3, device="cuda")
    faces = torch.tensor([[0, 1, 2]], dtype=torch.int32, device="cuda").repeat(65536, 1)
    r_c, p_c = device_camera(vpn, 1)
    with pytest.raises(vpn.VpnError, match="65535"):
        vpn.soft_silhouette(verts, faces, r_c, p_c, 16, 16)
    rc, _, _, _ = abi_fwd(vpn, verts, faces, r_c, p_c, 16, 16, False, 30)
    assert rc == VPN_ERR_SHAPE


# ------------------------------------------------------------------------------------------------
# 5. poisoned samples and batch isolation
# ------------------------------------------------------------------------------------------------
POISON_HW = (40, 56)


def poison_scene(mode):
    """B = 3 spot scenes; sample 1's rightmost vertex of the centre sphere is NaN ('nan') or on the camera plane
    ('plane': x = 1, so cam.z = 0 and its projection is infinite).  Returns verts, faces, the vertex index."""
    verts, faces = spot_scene("sphere", b=3, seed=5)
    nv = 128
    centre = verts[1, 3 * nv:4 * nv]
    j = 3 * nv + int(torch.argmin(centre[:, 2]))            # screen x = -z * scale: the rim vertex on the right
    if mode == "nan":
        verts[1, j] = float("nan")
    else:
        verts[1, j, 0] = 1.0
    return verts, faces, j


def poison_premise(O, mode):
    """Under a box rule that drops the non-finite coordinates (fminf / fmaxf), the poisoned faces would hold uncovered
    pixels of sample 1: the test sees whether they are skipped."""
    h, w = POISON_HW
    verts, faces, j = poison_scene(mode)
    rot, pos = default_camera(3)
    _, xy = O.project_vertices(verts, rot, pos)
    s = xy[1] * O.DIBR_MULTIPLIER
    assert not torch.isfinite(s[j]).all(), "premise: the vertex's projection is not finite"
    X, Y = O._sil_pixel_centres(h, w)
    sel = O.soft_silhouette_selection(verts, faces, rot, pos, h, w)
    hit = torch.zeros(h * w, dtype=torch.bool)
    for f in (faces == j).any(1).nonzero().flatten():
        c = s[faces[f]]
        c = c[torch.isfinite(c).all(1)]
        lo, hi = c.min(0)[0] - 20.0, c.max(0)[0] + 20.0
        hit |= (X >= lo[0]) & (X < hi[0]) & (Y >= lo[1]) & (Y < hi[1])
    assert (hit & ~sel["covered"][1]).any(), "premise: the poisoned faces' finite corners reach uncovered pixels"
    return verts, faces, j


@pytest.mark.parametrize("mode", ["nan", "plane"])
def test_poisoned_sample_isolated(vpn, O, mode):
    """A face with a non-finite screen coordinate takes part in neither pass, in the kernel and the oracle alike: the
    other samples keep the bits they have alone, every gradient is finite, the poisoned vertex's is zero."""
    h, w = POISON_HW
    verts, faces, j = poison_scene(mode)
    poison_premise(O, mode)
    alpha, covered, vg, r_c, p_c = render(vpn, verts, faces, h, w, False)
    up = torch.rand(3, h, w, generator=torch.Generator().manual_seed(17))
    (alpha * up.cuda()).sum().backward()
    assert torch.isfinite(alpha).all() and torch.isfinite(vg.grad).all()
    for i in (0, 2):
        a1, c1, v1, _, _ = render(vpn, verts[i:i + 1], faces, h, w, False)
        same(alpha[i], a1[0], f"sample {i}: alpha alone vs in the batch"); same(covered[i], c1[0], f"sample {i}: covered")
        (a1 * up[i:i + 1].cuda()).sum().backward()
        close(vg.grad[i], v1.grad[0], rtol=1e-5, atol=1e-6 * float(v1.grad.abs().max()), what=f"sample {i}: gradient")
    ref, gref, rcov = oracle_alpha_grad(O, verts[1:2], faces, r_c[1:2], p_c[1:2], h, w, False, up[1:2])
    check_alpha(alpha[1:2], covered[1:2], ref, rcov, f"poisoned sample ({mode})")
    assert (vg.grad[1, j] == 0).all(), "the poisoned vertex gets no gradient"
    keep = torch.ones(verts.shape[1], dtype=torch.bool); keep[j] = False
    assert torch.isfinite(gref[0, keep]).all()
    check_grad(vg.grad[1, keep.cuda()], gref[0, keep], f"poisoned sample ({mode})")


def test_batch_matches_alone_and_repeats(vpn):
    """The forward is fixed-order with no atomics: each sample of a batch of 4 gives the bits it gives alone, and two
    calls give the same bits."""
    h, w = 48, 80
    verts, faces = spot_scene("cuboid", b=4, seed=8)
    a, c, _, _, _ = render(vpn, verts, faces, h, w, False)
    a2, c2, _, _, _ = render(vpn, verts, faces, h, w, False)
    same(a, a2, "alpha, two calls"); same(c, c2, "covered, two calls")
    for i in range(4):
        ai, ci, _, _, _ = render(vpn, verts[i:i + 1], faces, h, w, False)
        same(a[i], ai[0], f"sample {i}: alpha"); same(c[i], ci[0], f"sample {i}: covered")


# ------------------------------------------------------------------------------------------------
# 6. sparse upstream gradients
# ------------------------------------------------------------------------------------------------
def test_sparse_upstream(vpn, O):
    h, w = 48, 80
    verts, faces = spot_scene("sphere", b=2, seed=4)
    rot, pos = default_camera(2)
    alpha, covered, vg, r_c, p_c = render(vpn, verts, faces, h, w, False)
    a = alpha.detach().cpu()
    # one soft pixel of sample 1
    soft = ((a[1] > 0.05) & (a[1] < 0.95)).flatten().nonzero().flatten()
    assert soft.numel() > 0
    p = int(soft[soft.numel() // 2])
    up = torch.zeros(2, h, w); up.view(2, -1)[1, p] = 1.0
    (alpha * up.cuda()).sum().backward(retain_graph=True)
    _, gref, _ = oracle_alpha_grad(O, verts, faces, r_c, p_c, h, w, False, up)
    check_grad(vg.grad, gref, "single soft pixel")
    sel = O.soft_silhouette_selection(verts[1:2], faces, rot[1:2], pos[1:2], h, w, pixels=torch.tensor([p]))
    recorded = faces[sel["use"][0][0]].flatten().unique()
    assert recorded.numel() >= 3
    mask = torch.zeros(verts.shape[1], dtype=torch.bool); mask[recorded] = True
    g = vg.grad.cpu()
    assert (g[0] == 0).all() and (g[1, ~mask] == 0).all() and (g[1, mask] != 0).any(), "only the recorded faces' vertices"
    # covered pixels only: exactly zero
    vg.grad = None
    cov = (covered == 1).float()
    assert cov.sum() > 100
    (alpha * cov * torch.rand(2, h, w, device="cuda")).sum().backward(retain_graph=True)
    assert (vg.grad == 0).all(), "covered pixels carry no gradient"
    # all zero: exactly zero, and the output buffer is overwritten
    rc, _, cv, state = abi_fwd(vpn, verts, faces, r_c, p_c, h, w, False, 30)
    assert rc == 0
    gv = torch.full((2, verts.shape[1], 3), float("nan"), device="cuda")
    abi_bwd(vpn, state, torch.zeros(2, h, w), cv, h, w, False, 30, grad_verts=gv)
    assert (gv == 0).all(), "zero upstream: zero gradient over a garbage-filled buffer"


# ------------------------------------------------------------------------------------------------
# 7. the distance cases one at a time
# ------------------------------------------------------------------------------------------------
def cases_premise(O):
    h, w = CASES_HW
    verts, faces = cases_scene()
    rot, pos = default_camera(2)
    sel = O.soft_silhouette_selection(verts, faces, rot, pos, h, w)
    alpha = O.soft_silhouette(verts, faces, rot, pos, h, w)
    pix0, pix1 = case_pixels(sel, alpha, 0), case_pixels(sel, alpha, 1)
    assert all(p >= 0 for p in pix0[:6]), f"premise: every edge and vertex case occurs on the triangle, {pix0}"
    assert pix1[6] >= 0, "premise: the foot-off constant wins on a pixel of the needle"
    return verts, faces, pix0[:6], pix1[6]


def grad64(O, verts, faces, rot, pos, h, w, pixel, case):
    """d alpha / d verts of one pixel with one candidate (alpha = prob) in float64, from the kernel's float32 inputs
    (vertices, camera, projection constants, pixel centre) and the case the oracle selects."""
    from vpn_b200 import ops
    v = verts.double().clone().requires_grad_()
    proj = torch.tensor(ops.projection_vector(), dtype=torch.float32).double()
    d = v - pos.double()[:, None]
    cam = torch.einsum("bkj,bvj->bvk", rot.double(), d)
    xy = cam[..., :2] * proj[:2] / (cam[..., 2:] * proj[2])
    s = xy[0, faces[0]] * 1000.0                           # (3,2)
    X, Y = (c.double()[0] for c in O._sil_pixel_centres(h, w, torch.tensor([pixel])))
    if case < 3:
        (x1, y1), (x2, y2) = s[case], s[(case + 1) % 3]
        A, Bc, C_ = y2 - y1, x1 - x2, x2 * y1 - x1 * y2
        up = A * X + Bc * Y + C_
        d2 = up * up / (A * A + Bc * Bc + 1e-15)
    else:
        d2 = (X - s[case - 3, 0]) ** 2 + (Y - s[case - 3, 1]) ** 2
    prob = torch.exp(-(7000.0 * d2 / 1e6))
    prob.backward()
    return v.grad


def test_distance_cases_one_at_a_time(vpn, O):
    """Each of edge 0/1/2 (foot on the segment), vertex 0/1/2 and the foot-off constant from a single pixel: the vertex
    gradient against the oracle, and the closed form of the backward against float64 on the same float32 inputs (the
    constant case: exactly zero)."""
    h, w = CASES_HW
    verts, faces, pixels, p_const = cases_premise(O)
    rot, pos = default_camera(2)
    r_c, p_c = device_camera(vpn, 2)
    rc, alpha, covered, state = abi_fwd(vpn, verts, faces, r_c, p_c, h, w, False, 30)
    assert rc == 0
    up = torch.zeros(2, h, w)
    ref_a, _, rcov = oracle_alpha_grad(O, verts, faces, r_c, p_c, h, w, False, up)
    check_alpha(alpha, covered, ref_a, rcov, "cases")
    for case, (b, p) in enumerate([(0, q) for q in pixels] + [(1, p_const)]):
        up = torch.zeros(2, h, w); up.view(2, -1)[b, p] = 1.0
        gv = abi_bwd(vpn, state, up, covered, h, w, False, 30).cpu()
        _, gref, _ = oracle_alpha_grad(O, verts, faces, r_c, p_c, h, w, False, up)
        assert (gv[1 - b] == 0).all()
        if case == 6:
            assert (gv == 0).all() and (gref == 0).all(), "the foot-off constant carries no gradient"
            continue
        assert gv.abs().max() > 0
        check_grad(gv, gref, f"case {case}")
        g64 = grad64(O, verts[b:b + 1], faces, r_c[b:b + 1].cpu(), p_c[b:b + 1].cpu(), h, w, p, case)
        close(gv[b], g64[0].float(), rtol=1e-4, atol=1e-5 * float(g64.abs().max()), what=f"case {case}: float64 closed form")
