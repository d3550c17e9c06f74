"""torch.autograd.Functions over the C ABI (include/vpn_b200.h).

Each Function follows the ownership convention of the reference's only native op
(modules/loss/emd/emd_module.py:32-59): Python allocates outputs and scratch with torch, the native
call fills them on the current CUDA stream.  No CPU path exists; CPU tensors raise VpnError.
"""
from __future__ import annotations

import ctypes
import math
from typing import Optional, Tuple

import torch

from . import _lib
from ._lib import VpnError, check, ptr, require, stream_ptr

KIND_SPHERE, KIND_CUBOID, KIND_TEMPLATE, KIND_POINTS = 0, 1, 2, 3
CHAMFER_AUTO, CHAMFER_GENERIC, CHAMFER_TILED_EXACT, CHAMFER_TILED_FMA, CHAMFER_TILED_EXPAND, CHAMFER_TILED_TC = 0, 1, 2, 3, 4, 5

f32 = torch.float32


def _scratch_bytes(nbytes: int, device) -> torch.Tensor:
    return torch.empty(max(int(nbytes), 16), dtype=torch.uint8, device=device)


# --------------------------------------------------------------------------------------
# primitive instantiation
# --------------------------------------------------------------------------------------
class _PosePoints(torch.autograd.Function):
    """out[p, n] = R(q[p]) (canonical(kind, src)[p, n] * v[p]) + t[p]   for nprim primitives."""

    @staticmethod
    def forward(ctx, kind, v, q, t, src, n_points):
        lib = _lib.load()
        q = require(q, f32, "q")
        nprim = q.shape[0]
        dev = q.device
        if kind != KIND_POINTS:
            v = require(v, f32, "v")
        if t is not None:
            t = require(t, f32, "t")
        src = require(src, f32, "src")
        out = torch.empty((nprim, n_points, 3), dtype=f32, device=dev)
        check(lib.vpn_pose_points_fwd(kind, ptr(v) if kind != KIND_POINTS else None, ptr(q), ptr(t), ptr(src),
                                      ptr(out), nprim, n_points, stream_ptr(dev)), "vpn_pose_points_fwd")
        ctx.kind, ctx.n_points, ctx.has_t = kind, n_points, t is not None
        ctx.save_for_backward(v if kind != KIND_POINTS else q, q, src)
        return out

    @staticmethod
    def backward(ctx, grad_out):
        lib = _lib.load()
        v, q, src = ctx.saved_tensors
        kind, n = ctx.kind, ctx.n_points
        nprim, dev = q.shape[0], q.device
        grad_out = grad_out.contiguous()
        need_v = kind != KIND_POINTS and ctx.needs_input_grad[1]
        need_q, need_t = ctx.needs_input_grad[2], ctx.has_t and ctx.needs_input_grad[3]
        need_p = kind == KIND_POINTS and ctx.needs_input_grad[4]
        gv = torch.empty((nprim, 3), dtype=f32, device=dev) if need_v else None
        gq = torch.empty((nprim, 4), dtype=f32, device=dev) if need_q else None
        gt = torch.empty((nprim, 3), dtype=f32, device=dev) if need_t else None
        gp = torch.empty((nprim, n, 3), dtype=f32, device=dev) if need_p else None
        nfl = ctypes.c_size_t(0)
        check(lib.vpn_pose_bwd_workspace_floats(nprim, n, ctypes.byref(nfl)), "vpn_pose_bwd_workspace_floats")
        ws = torch.empty(max(nfl.value, 16), dtype=f32, device=dev)
        check(lib.vpn_pose_points_bwd(kind, ptr(v) if kind != KIND_POINTS else None, ptr(q), ptr(src), ptr(grad_out),
                                      ptr(gv), ptr(gq), ptr(gt), ptr(gp), ptr(ws), nfl.value, nprim, n,
                                      stream_ptr(dev)), "vpn_pose_points_bwd")
        return None, gv, gq, gt, gp, None


def _flat_prims(v, q, t):
    if q.dim() != 3 or q.size(-1) != 4:
        raise AssertionError("q must be (B, K, 4)")
    b, k = q.shape[:2]
    assert v.shape == (b, k, 3) and t.shape == (b, k, 3), "v, t must be (B, K, 3)"
    return b, k, v.reshape(b * k, 3).contiguous(), q.reshape(b * k, 4).contiguous(), t.reshape(b * k, 3).contiguous()


def sample_primitives(kind: str, v: torch.Tensor, q: torch.Tensor, t: torch.Tensor, u: torch.Tensor) -> torch.Tensor:
    """Fused sampling + pose of K primitives per sample (train.py:105-120 in one launch).

    v (B,K,3), q (B,K,4), t (B,K,3); u uniforms in [0,1): sphere (B,K,N,2) = [elev draw, azim draw]
    (sampling/sphere.py:26-27), cuboid (B,K,N,3) (sampling/cuboid.py:66).  Returns (B, K*N, 3),
    primitive-major along dim 1 exactly like the reference's torch.cat(dim=1)."""
    b, k, vf, qf, tf = _flat_prims(v, q, t)
    kid = {"sphere": KIND_SPHERE, "cuboid": KIND_CUBOID}[kind]
    width = 2 if kid == KIND_SPHERE else 3
    assert u.dim() == 4 and u.shape[:2] == (b, k) and u.size(-1) == width, "bad uniforms shape"
    n = u.size(2)
    out = _PosePoints.apply(kid, vf, qf, tf, u.reshape(b * k, n, width).contiguous(), n)
    return out.view(b, k * n, 3)


def mesh_vertices(template: torch.Tensor, v: torch.Tensor, q: torch.Tensor, t: torch.Tensor) -> torch.Tensor:
    """Template vertices (V,3) scaled by v and posed per primitive: (B, K*V, 3)
    (meshing/sphere.py:8-27, cuboid.py:8-27, then compose order of meshing.py:28-46)."""
    b, k, vf, qf, tf = _flat_prims(v, q, t)
    assert template.dim() == 2 and template.size(1) == 3
    nv = template.size(0)
    out = _PosePoints.apply(KIND_TEMPLATE, vf, qf, tf, template.contiguous(), nv)
    return out.view(b, k * nv, 3)


def transform_points(points: torch.Tensor, q: torch.Tensor, t: Optional[torch.Tensor]) -> torch.Tensor:
    """translate(rotate(points, q), t)  (transform/transform.py:6-9); t=None -> rotate only."""
    assert points.dim() == 3 and points.size(-1) == 3
    b, n = points.shape[:2]
    assert q.shape == (b, 4) and (t is None or t.shape == (b, 3))
    if n == 0:
        return points.clone()
    return _PosePoints.apply(KIND_POINTS, None, q.contiguous(), None if t is None else t.contiguous(),
                             points.contiguous(), n)


def cuboid_face_counts(v: torch.Tensor, num_points: int) -> torch.Tensor:
    """get_faces_points (sampling/cuboid.py:30-53): (..., 6) int32."""
    lib = _lib.load()
    vf = require(v.reshape(-1, 3).contiguous(), f32, "v")
    out = torch.empty((vf.shape[0], 6), dtype=torch.int32, device=vf.device)
    check(lib.vpn_cuboid_face_counts(ptr(vf), ptr(out), vf.shape[0], int(num_points), stream_ptr(vf.device)),
          "vpn_cuboid_face_counts")
    return out.view(*v.shape[:-1], 6)


# --------------------------------------------------------------------------------------
# camera frame changes
# --------------------------------------------------------------------------------------
class _ViewPoints(torch.autograd.Function):
    @staticmethod
    def forward(ctx, mode, points, dists, elevs, azims, angles):
        out = _ViewPoints._run(mode, 0, points, dists, elevs, azims, angles)
        ctx.mode = mode
        ctx.save_for_backward(dists, elevs, azims, angles if angles is not None else dists)
        return out

    @staticmethod
    def _run(mode, transpose, x, dists, elevs, azims, angles):
        lib = _lib.load()
        x = require(x.contiguous(), f32, "points")
        b, n = x.shape[:2]
        dev = x.device
        args = [require(a.contiguous(), f32, nm) for a, nm in ((dists, "dists"), (elevs, "elevs"), (azims, "azims"))]
        ang = require(angles.contiguous(), f32, "angles") if mode == 0 else None
        out = torch.empty_like(x)
        nb = ctypes.c_size_t(0)
        check(lib.vpn_view_workspace_bytes(b, ctypes.byref(nb)), "vpn_view_workspace_bytes")
        ws = _scratch_bytes(nb.value, dev)
        check(lib.vpn_view_points(mode, transpose, ptr(x), ptr(args[0]), ptr(args[1]), ptr(args[2]), ptr(ang), ptr(out),
                                  ptr(ws), nb.value, b, n, stream_ptr(dev)), "vpn_view_points")
        return out

    @staticmethod
    def backward(ctx, grad_out):
        dists, elevs, azims, angles = ctx.saved_tensors
        g = _ViewPoints._run(ctx.mode, 1, grad_out, dists, elevs, azims, angles)
        return None, g, None, None, None, None


def view_to_obj_points(points, dists, elevs, azims, angles):
    """transform/transform.py:21-47."""
    assert points.dim() == 3
    assert dists.dim() == elevs.dim() == azims.dim() == 1
    return _ViewPoints.apply(0, points, dists, elevs, azims, angles)


def obj_to_view_points(points, dists, elevs, azims):
    """transform/transform.py:50-73."""
    assert points.dim() == 3
    assert dists.dim() == elevs.dim() == azims.dim() == 1
    return _ViewPoints.apply(1, points, dists, elevs, azims, None)


# --------------------------------------------------------------------------------------
# Chamfer
# --------------------------------------------------------------------------------------
class _ChamferNN(torch.autograd.Function):
    @staticmethod
    def forward(ctx, p1, p2, impl):
        lib = _lib.load()
        p1 = require(p1.contiguous(), f32, "points1")
        p2 = require(p2.contiguous(), f32, "points2")
        b, p, _ = p1.shape
        m = p2.shape[1]
        dev = p1.device
        min1 = torch.empty((b, p), dtype=f32, device=dev); idx1 = torch.empty((b, p), dtype=torch.int32, device=dev)
        min2 = torch.empty((b, m), dtype=f32, device=dev); idx2 = torch.empty((b, m), dtype=torch.int32, device=dev)
        nb = ctypes.c_size_t(0)
        check(lib.vpn_chamfer_workspace_bytes(b, p, m, impl, ctypes.byref(nb)), "vpn_chamfer_workspace_bytes")
        ws = _scratch_bytes(nb.value, dev)
        check(lib.vpn_chamfer_fwd(ptr(p1), ptr(p2), ptr(min1), ptr(idx1), ptr(min2), ptr(idx2), b, p, m,
                                  ptr(ws), nb.value, impl, stream_ptr(dev)), "vpn_chamfer_fwd")
        ctx.save_for_backward(p1, p2, min1, idx1, min2, idx2)
        ctx.mark_non_differentiable(idx1, idx2)
        return min1, idx1, min2, idx2

    @staticmethod
    def backward(ctx, g1, _gi1, g2, _gi2):
        lib = _lib.load()
        p1, p2, min1, idx1, min2, idx2 = ctx.saved_tensors
        b, p, _ = p1.shape
        m = p2.shape[1]
        dev = p1.device
        g1 = torch.zeros_like(min1) if g1 is None else g1.contiguous()
        g2 = torch.zeros_like(min2) if g2 is None else g2.contiguous()
        gp1 = torch.empty_like(p1)
        gp2 = torch.empty_like(p2) if ctx.needs_input_grad[1] else None
        check(lib.vpn_chamfer_bwd(ptr(p1), ptr(p2), ptr(min1), ptr(idx1), ptr(min2), ptr(idx2), ptr(g1), ptr(g2),
                                  ptr(gp1), ptr(gp2), b, p, m, stream_ptr(dev)), "vpn_chamfer_bwd")
        return (gp1 if ctx.needs_input_grad[0] else None), gp2, None


def chamfer_nn(points1: torch.Tensor, points2: torch.Tensor, impl: int = CHAMFER_AUTO):
    """Nearest neighbours in both directions: (min1 (B,P), idx1 (B,P) int32, min2 (B,M), idx2 (B,M) int32).
    min* are differentiable w.r.t. both clouds; arithmetic and tie rule of chamfer_distance.py:14-23."""
    assert points1.dim() == 3 and points1.size(-1) == 3          # chamfer_distance.py:33-35
    assert points2.dim() == 3 and points2.size(-1) == 3
    assert points1.size(0) == points2.size(0)
    return _ChamferNN.apply(points1, points2, impl)


def chamfer_nn_stage_ms(points1: torch.Tensor, points2: torch.Tensor, impl: int = CHAMFER_AUTO, reps: int = 5):
    """Device time (ms, mean of `reps`) of the forward's stages, measured with CUDA events on the launch stream:
    {'main', 'fallback', 'rows', 'cols', 'total'}.  Measurement helper for bench.py."""
    lib = _lib.load()
    p1 = require(points1.contiguous(), f32, "points1"); p2 = require(points2.contiguous(), f32, "points2")
    b, p, _ = p1.shape
    m = p2.shape[1]
    dev = p1.device
    min1 = torch.empty((b, p), dtype=f32, device=dev); idx1 = torch.empty((b, p), dtype=torch.int32, device=dev)
    min2 = torch.empty((b, m), dtype=f32, device=dev); idx2 = torch.empty((b, m), dtype=torch.int32, device=dev)
    nb = ctypes.c_size_t(0)
    check(lib.vpn_chamfer_workspace_bytes(b, p, m, impl, ctypes.byref(nb)), "vpn_chamfer_workspace_bytes")
    ws = _scratch_bytes(nb.value, dev)
    ms = (ctypes.c_float * 4)()
    check(lib.vpn_chamfer_fwd_timed(ptr(p1), ptr(p2), ptr(min1), ptr(idx1), ptr(min2), ptr(idx2), b, p, m, ptr(ws),
                                    nb.value, impl, reps, ms, stream_ptr(dev)), "vpn_chamfer_fwd_timed")
    out = dict(zip(("main", "fallback", "rows", "cols"), [float(x) for x in ms]))
    out["total"] = sum(out.values())
    stages, skipped = ctypes.c_ulonglong(0), ctypes.c_ulonglong(0)
    check(lib.vpn_chamfer_prune_stats(ptr(ws), b, p, m, impl, ctypes.byref(stages), ctypes.byref(skipped), stream_ptr(dev)),
          "vpn_chamfer_prune_stats")
    out["stages"], out["stages_skipped"] = int(stages.value), int(skipped.value)
    cnt = (ctypes.c_ulonglong * 16)()
    check(lib.vpn_chamfer_tc_counters(ptr(ws), b, p, m, impl, cnt, stream_ptr(dev)), "vpn_chamfer_tc_counters")
    out["tc_counters"] = [int(x) for x in cnt[:16]]
    return out


class _ChamferLoss(torch.autograd.Function):
    """Per-sample loss w1*mean(min1) + w2*mean(min2) with the nearest-neighbour search, the two means and the
    whole backward as vpn_b200 kernels (no (B,P)/(B,M) gradient tensors, no elementwise torch launches)."""

    @staticmethod
    def forward(ctx, p1, p2, w1, w2, impl):
        lib = _lib.load()
        p1 = require(p1.contiguous(), f32, "points1")
        p2 = require(p2.contiguous(), f32, "points2")
        b, p, _ = p1.shape
        m = p2.shape[1]
        dev = p1.device
        min1 = torch.empty((b, p), dtype=f32, device=dev); idx1 = torch.empty((b, p), dtype=torch.int32, device=dev)
        min2 = torch.empty((b, m), dtype=f32, device=dev); idx2 = torch.empty((b, m), dtype=torch.int32, device=dev)
        nb = ctypes.c_size_t(0)
        check(lib.vpn_chamfer_workspace_bytes(b, p, m, impl, ctypes.byref(nb)), "vpn_chamfer_workspace_bytes")
        ws = _scratch_bytes(nb.value, dev)
        st = stream_ptr(dev)
        check(lib.vpn_chamfer_fwd(ptr(p1), ptr(p2), ptr(min1), ptr(idx1), ptr(min2), ptr(idx2), b, p, m,
                                  ptr(ws), nb.value, impl, st), "vpn_chamfer_fwd")
        loss = torch.empty((b,), dtype=f32, device=dev)
        part = torch.empty((b * 64,), dtype=f32, device=dev)
        check(lib.vpn_chamfer_loss_fwd(ptr(min1), ptr(min2), float(w1), float(w2), ptr(loss), ptr(part), b, p, m, st),
              "vpn_chamfer_loss_fwd")
        ctx.save_for_backward(p1, p2, min1, idx1, min2, idx2)
        ctx.w = (float(w1), float(w2))
        return loss

    @staticmethod
    def backward(ctx, gloss):
        lib = _lib.load()
        p1, p2, min1, idx1, min2, idx2 = ctx.saved_tensors
        b, p, _ = p1.shape
        m = p2.shape[1]
        dev = p1.device
        gloss = gloss.contiguous()
        gp1 = torch.empty_like(p1)
        gp2 = torch.empty_like(p2) if ctx.needs_input_grad[1] else None
        check(lib.vpn_chamfer_loss_bwd(ptr(p1), ptr(p2), ptr(min1), ptr(idx1), ptr(min2), ptr(idx2), ptr(gloss),
                                       ctx.w[0], ctx.w[1], ptr(gp1), ptr(gp2), b, p, m, stream_ptr(dev)),
              "vpn_chamfer_loss_bwd")
        return (gp1 if ctx.needs_input_grad[0] else None), gp2, None, None, None


def chamfer_distance(points1, points2, each_batch=False, w1=1.0, w2=1.0, impl: int = CHAMFER_AUTO):
    """ChamferDistanceLoss.forward (chamfer_distance.py:10-30)."""
    assert points1.dim() == 3 and points1.size(-1) == 3          # chamfer_distance.py:33-35
    assert points2.dim() == 3 and points2.size(-1) == 3
    assert points1.size(0) == points2.size(0)
    loss = _ChamferLoss.apply(points1, points2, w1, w2, impl)
    return loss if each_batch else loss.mean()


# --------------------------------------------------------------------------------------
# soft silhouette
# --------------------------------------------------------------------------------------
DIBR_FOVY_DEG = 49.13434207744484
DIBR_EXPAND, DIBR_KNUM, DIBR_MULTIPLIER, DIBR_DELTA = 0.02, 30, 1000.0, 7000.0


def projection_vector() -> Tuple[float, float, float]:
    tf = math.tan(math.radians(DIBR_FOVY_DEG) / 2.0)
    return 1.0 / tf, 1.0 / tf, -1.0


def look_at_cameras(azims: torch.Tensor, elevs: torch.Tensor, dists: torch.Tensor):
    """kaolin compute_camera_params for a batch, on the tensors' device, no host sync:
    rot (B,3,3) rows = unit X = Y0 x Z, Y = Z x X, Z = cam_pos; pos (B,3)."""
    theta, phi = torch.deg2rad(azims.double()), torch.deg2rad(elevs.double())
    d = dists.double()
    pos = torch.stack([d * torch.cos(phi) * torch.cos(theta), d * torch.sin(phi), d * torch.cos(phi) * torch.sin(theta)], 1)
    az = pos
    # Y0 = (0, 1, 0) built on the device without a host-to-device copy (safe inside CUDA-graph capture)
    ay0 = torch.zeros_like(pos)
    ay0[:, 1] = 1.0
    ax = torch.cross(ay0, az, dim=1)
    ay = torch.cross(az, ax, dim=1)
    unit = lambda x: x / torch.linalg.norm(x, dim=1, keepdim=True)
    rot = torch.stack([unit(ax), unit(ay), unit(az)], dim=1)
    return rot.float().contiguous(), pos.float().contiguous()


class _SoftSilhouette(torch.autograd.Function):
    @staticmethod
    def forward(ctx, verts, faces, rot, pos, height, width, want_normals, soft_cull):
        lib = _lib.load()
        verts = require(verts.contiguous(), f32, "verts")
        faces = require(faces.contiguous(), torch.int32, "faces")
        rot = require(rot.contiguous(), f32, "cam_rot")
        pos = require(pos.contiguous(), f32, "cam_pos")
        b, v, _ = verts.shape
        f = faces.shape[0]
        dev = verts.device
        alpha = torch.empty((b, height, width), dtype=f32, device=dev)
        covered = torch.empty((b, height, width), dtype=torch.uint8, device=dev)
        normals = torch.empty((b, f, 3), dtype=f32, device=dev) if want_normals else None
        nb = ctypes.c_size_t(0)
        check(lib.vpn_silhouette_workspace_bytes(b, v, f, ctypes.byref(nb)), "vpn_silhouette_workspace_bytes")
        ws = _scratch_bytes(nb.value, dev)
        px, py, pz = projection_vector()
        check(lib.vpn_silhouette_fwd(ptr(verts), ptr(faces), ptr(rot), ptr(pos), px, py, pz, DIBR_EXPAND, DIBR_KNUM,
                                     DIBR_MULTIPLIER, DIBR_DELTA, int(soft_cull), ptr(alpha), ptr(covered), ptr(normals), ptr(ws),
                                     nb.value, b, v, f, height, width, stream_ptr(dev)), "vpn_silhouette_fwd")
        ctx.save_for_backward(faces, rot, covered, ws)
        ctx.dims = (b, v, f, height, width, nb.value, int(soft_cull))
        ctx.mark_non_differentiable(covered)
        if normals is None:
            normals = torch.empty(0, device=dev)
        ctx.mark_non_differentiable(normals)
        return alpha, covered, normals

    @staticmethod
    def backward(ctx, galpha, _gc, _gn):
        lib = _lib.load()
        faces, rot, covered, ws = ctx.saved_tensors
        b, v, f, h, w, nbytes, soft_cull = ctx.dims
        dev = rot.device
        galpha = galpha.contiguous()
        gverts = torch.empty((b, v, 3), dtype=f32, device=dev)
        px, py, pz = projection_vector()
        check(lib.vpn_silhouette_bwd(ptr(faces), ptr(rot), px, py, pz, DIBR_EXPAND, DIBR_KNUM, DIBR_MULTIPLIER, DIBR_DELTA,
                                     soft_cull, ptr(galpha), ptr(covered), ptr(gverts), ptr(ws), nbytes, b, v, f, h, w,
                                     stream_ptr(dev)), "vpn_silhouette_bwd")
        return gverts, None, None, None, None, None, None, None


def soft_silhouette(verts, faces, rot, pos, height: int, width: int, want_normals: bool = False,
                    soft_cull_backfaces: bool = False):
    """Batched DIB-R soft alpha: verts (B,V,3), faces (F,3) int32 (shared topology), cameras (B,3,3)/(B,3).
    Returns (alpha (B,H,W), covered (B,H,W) uint8, face_normals (B,F,3) or empty).
    soft_cull_backfaces=False is DIB-R's rule as recalled in SURVEY.md 8(a-R): the coverage pass skips back faces, the
    soft (probability) pass does not; True skips them in both (DESIGN.md section 2)."""
    assert verts.dim() == 3 and verts.size(-1) == 3 and faces.dim() == 2 and faces.size(-1) == 3
    _check_face_indices(faces, verts.size(1))
    return _SoftSilhouette.apply(verts, faces, rot, pos, int(height), int(width), bool(want_normals), bool(soft_cull_backfaces))


_FACES_CHECKED = {}


def _check_face_indices(faces: torch.Tensor, n_verts: int):
    """The kernels index vertex arrays with the caller's face indices: validate each faces tensor ONCE (keyed by storage
    pointer, shape and version; one device-to-host read the first time, none afterwards, nothing during graph capture)."""
    key = (faces.data_ptr(), tuple(faces.shape), faces._version, int(n_verts), str(faces.device))
    if key in _FACES_CHECKED:
        return
    if faces.is_cuda and torch.cuda.is_current_stream_capturing():
        return                                   # cannot read back while capturing; the eager warm-up call has checked
    if faces.numel():
        lo, hi = int(faces.min()), int(faces.max())
        if lo < 0 or hi >= n_verts:
            raise VpnError(f"faces index vertices outside [0, {n_verts}): min {lo}, max {hi}")
    if len(_FACES_CHECKED) > 256:
        _FACES_CHECKED.clear()
    _FACES_CHECKED[key] = True


# --------------------------------------------------------------------------------------
# mesh surface sampling
# --------------------------------------------------------------------------------------
class _MeshSample(torch.autograd.Function):
    @staticmethod
    def forward(ctx, verts, faces, u):
        lib = _lib.load()
        verts = require(verts.contiguous(), f32, "verts")
        faces = require(faces.contiguous(), torch.int32, "faces")
        u = require(u.contiguous(), f32, "uniforms")
        b, v, _ = verts.shape
        f, n, dev = faces.shape[0], u.shape[1], verts.device
        points = torch.empty((b, n, 3), dtype=f32, device=dev)
        face_idx = torch.empty((b, n), dtype=torch.int32, device=dev)
        cdf = torch.empty((b, f), dtype=f32, device=dev)
        check(lib.vpn_mesh_sample_fwd(ptr(verts), ptr(faces), ptr(u), ptr(points), ptr(face_idx), ptr(cdf), b, v, f, n,
                                      stream_ptr(dev)), "vpn_mesh_sample_fwd")
        ctx.save_for_backward(faces, u, face_idx)
        ctx.dims = (b, v, f, n)
        ctx.mark_non_differentiable(face_idx)
        return points, face_idx

    @staticmethod
    def backward(ctx, gpoints, _gidx):
        lib = _lib.load()
        faces, u, face_idx = ctx.saved_tensors
        b, v, f, n = ctx.dims
        dev = u.device
        offsets, entries = mesh_adjacency(faces, v)
        gverts = torch.empty((b, v, 3), dtype=f32, device=dev)
        nb = ctypes.c_size_t(0)
        check(lib.vpn_mesh_sample_bwd_workspace_bytes(b, f, n, ctypes.byref(nb)), "vpn_mesh_sample_bwd_workspace_bytes")
        ws = _scratch_bytes(nb.value, dev)
        check(lib.vpn_mesh_sample_bwd_sorted(ptr(faces), ptr(u), ptr(face_idx), ptr(gpoints.contiguous()), ptr(gverts),
                                             ptr(offsets), ptr(entries), ptr(ws), nb.value, b, v, f, n, stream_ptr(dev)),
              "vpn_mesh_sample_bwd_sorted")
        return gverts, None, None


_ADJACENCY = {}


def mesh_adjacency(faces: torch.Tensor, n_verts: int):
    """Vertex -> (face, corner) CSR of a faces tensor (F,3) int32: (offsets (V+1,) int32, entries (3F,) int32 = 3 * face +
    corner), a vertex's entries in increasing order.  It fixes the order in which the sampler's backward sums a vertex's
    gradient.  Built on the device with torch, without a host read, and cached once per faces tensor outside graph
    capture; the cache holds the tensor, so its storage cannot be reused under a cached key."""
    key = (faces.data_ptr(), tuple(faces.shape), faces._version, int(n_verts), str(faces.device))
    hit = _ADJACENCY.get(key)
    if hit is not None:
        return hit[1], hit[2]
    flat = faces.reshape(-1).long()
    entries = torch.argsort(flat, stable=True)
    offsets = torch.searchsorted(flat[entries], torch.arange(n_verts + 1, device=faces.device))
    if torch.cuda.is_current_stream_capturing():
        return offsets.int(), entries.int()          # filled in only when the graph replays: not for eager callers
    if len(_ADJACENCY) >= 64:
        _ADJACENCY.clear()
    _ADJACENCY[key] = (faces, offsets.int(), entries.int())
    return _ADJACENCY[key][1], _ADJACENCY[key][2]


def sample_mesh_surface(verts, faces, uniforms):
    """Batched TriangleMesh.sample (train_sphere.py:71-80): verts (B,V,3), faces (F,3) int32 shared topology,
    uniforms (B,n,3) in [0,1) = [face draw, u1, u2].  Returns (points (B,n,3), face_idx (B,n) int32); the gradient
    flows to the vertices through the barycentric weights."""
    assert verts.dim() == 3 and verts.size(-1) == 3 and faces.dim() == 2 and faces.size(-1) == 3
    assert uniforms.dim() == 3 and uniforms.size(-1) == 3 and uniforms.size(0) == verts.size(0)
    _check_face_indices(faces, verts.size(1))
    return _MeshSample.apply(verts, faces, uniforms)


# --------------------------------------------------------------------------------------
# EMD auction
# --------------------------------------------------------------------------------------
class _EmdAuction(torch.autograd.Function):
    @staticmethod
    def forward(ctx, xyz1, xyz2, eps, iters):
        lib = _lib.load()
        xyz1 = require(xyz1.contiguous(), f32, "xyz1"); xyz2 = require(xyz2.contiguous(), f32, "xyz2")
        b, n, _ = xyz1.shape
        dev = xyz1.device
        dist = torch.empty((b, n), dtype=f32, device=dev)
        assignment = torch.empty((b, n), dtype=torch.int32, device=dev)
        nb = ctypes.c_size_t(0)
        check(lib.vpn_emd_workspace_bytes(b, n, ctypes.byref(nb)), "vpn_emd_workspace_bytes")
        ws = _scratch_bytes(nb.value, dev)
        check(lib.vpn_emd_fwd(ptr(xyz1), ptr(xyz2), ptr(dist), ptr(assignment), ptr(ws), nb.value, b, n, float(eps), int(iters),
                              stream_ptr(dev)), "vpn_emd_fwd")
        ctx.save_for_backward(xyz1, xyz2, assignment)
        ctx.mark_non_differentiable(assignment)
        return dist, assignment

    @staticmethod
    def backward(ctx, gdist, _gidx):
        lib = _lib.load()
        xyz1, xyz2, assignment = ctx.saved_tensors
        b, n, _ = xyz1.shape
        g1 = torch.empty_like(xyz1)
        check(lib.vpn_emd_bwd(ptr(xyz1), ptr(xyz2), ptr(assignment), ptr(gdist.contiguous()), ptr(g1), b, n,
                              stream_ptr(xyz1.device)), "vpn_emd_bwd")
        g2 = torch.zeros_like(xyz2) if ctx.needs_input_grad[1] else None      # emd_module.py:66-67: zeros for xyz2
        return g1, g2, None, None


def emd_auction(xyz1, xyz2, eps: float, iters: int):
    """emdFunction.apply (emd_module.py:29-79): (dist (B,n) squared distance to the assigned point, assignment (B,n) int32)."""
    assert xyz1.dim() == 3 and xyz1.size(-1) == 3 and xyz2.shape == xyz1.shape        # emd_module.py:37-38: n == m, same batch
    return _EmdAuction.apply(xyz1, xyz2, eps, iters)


class _EmdLoss(torch.autograd.Function):
    """Per-sample loss weight * mean(sqrt(dist)) with the auction, the mean and the whole backward as vpn_b200 kernels
    (no (B,n) gradient tensor, no elementwise torch launches)."""

    @staticmethod
    def forward(ctx, xyz1, xyz2, eps, iters, weight):
        lib = _lib.load()
        xyz1 = require(xyz1.contiguous(), f32, "xyz1"); xyz2 = require(xyz2.contiguous(), f32, "xyz2")
        b, n, _ = xyz1.shape
        dev = xyz1.device
        dist = torch.empty((b, n), dtype=f32, device=dev)
        assignment = torch.empty((b, n), dtype=torch.int32, device=dev)
        nb = ctypes.c_size_t(0)
        check(lib.vpn_emd_workspace_bytes(b, n, ctypes.byref(nb)), "vpn_emd_workspace_bytes")
        ws = _scratch_bytes(nb.value, dev)
        st = stream_ptr(dev)
        check(lib.vpn_emd_fwd(ptr(xyz1), ptr(xyz2), ptr(dist), ptr(assignment), ptr(ws), nb.value, b, n, float(eps), int(iters),
                              st), "vpn_emd_fwd")
        loss = torch.empty((b,), dtype=f32, device=dev)
        part = torch.empty((b * 32,), dtype=f32, device=dev)
        check(lib.vpn_emd_loss_fwd(ptr(dist), float(weight), ptr(loss), ptr(part), b, n, st), "vpn_emd_loss_fwd")
        ctx.save_for_backward(xyz1, xyz2, assignment, dist)
        ctx.weight = float(weight)
        return loss

    @staticmethod
    def backward(ctx, gloss):
        lib = _lib.load()
        xyz1, xyz2, assignment, dist = ctx.saved_tensors
        b, n, _ = xyz1.shape
        g1 = torch.empty_like(xyz1)
        check(lib.vpn_emd_loss_bwd(ptr(xyz1), ptr(xyz2), ptr(assignment), ptr(dist), ptr(gloss.contiguous()), ctx.weight,
                                   ptr(g1), b, n, stream_ptr(xyz1.device)), "vpn_emd_loss_bwd")
        g2 = torch.zeros_like(xyz2) if ctx.needs_input_grad[1] else None      # emd_module.py:66-67: zeros for xyz2
        return g1, g2, None, None, None


def emd_distance(points1, points2, eps: float = 0.005, iters: int = 50, weight: float = 1.0, each_batch: bool = False):
    """EMD loss term of train.py:188-195 / train_gcn.py:91-95, weight * torch.sqrt(dist).mean(), with the auction of
    emd_auction (same preconditions: (B,n,3) clouds of equal shape, coordinates in [0,1]).  Returns the per-sample values
    (B,) when each_batch, else their mean.  points2 receives a zero gradient, as in the reference."""
    assert points1.dim() == 3 and points1.size(-1) == 3 and points2.shape == points1.shape     # emd_module.py:37-38
    loss = _EmdLoss.apply(points1, points2, eps, iters, weight)
    return loss if each_batch else loss.mean()


def sample_primitives_ms(kind: str, v, q, t, uniform_sets, reps: int = 32) -> float:
    """Mean device time (ms) of one fused sample+pose launch over a stream of `reps` launches that rotate through
    `uniform_sets` (list of (B,K,N,2|3) tensors; make their total size exceed L2 for cold reads).  Measurement helper."""
    lib = _lib.load()
    kid = {"sphere": KIND_SPHERE, "cuboid": KIND_CUBOID}[kind]
    b, k, vf, qf, tf = _flat_prims(v.detach(), q.detach(), t.detach())
    n = uniform_sets[0].shape[2]
    dev = qf.device
    srcs = [require(u.contiguous(), f32, "uniforms") for u in uniform_sets]
    arr = (ctypes.c_void_p * len(srcs))(*[u.data_ptr() for u in srcs])
    out = torch.empty((b * k, n, 3), dtype=f32, device=dev)
    ms = ctypes.c_float(0)
    check(lib.vpn_pose_points_fwd_timed(kid, ptr(vf), ptr(qf), ptr(tf), arr, len(srcs), ptr(out), b * k, n, reps,
                                        ctypes.byref(ms), stream_ptr(dev)), "vpn_pose_points_fwd_timed")
    return float(ms.value)


def chamfer_main_kernel_name(b: int, p: int, m: int, impl: int = CHAMFER_AUTO) -> str:
    """Name of the kernel vpn_chamfer_fwd spends its time in for this shape / impl (bench.py's roofline label)."""
    lib = _lib.load()
    return lib.vpn_chamfer_main_kernel(b, p, m, impl).decode()


def fp32_peak_tflops(device=None, reps: int = 3):
    """Achieved FP32 FMA throughput (TFLOP/s) of scalar FFMA and packed FFMA2 streams on this GPU."""
    lib = _lib.load()
    dev = torch.device("cuda" if device is None else device)
    scratch = torch.ones(64, dtype=f32, device=dev)
    a, b = ctypes.c_double(0), ctypes.c_double(0)
    check(lib.vpn_fp32_peak_probe(ptr(scratch), reps, ctypes.byref(a), ctypes.byref(b), stream_ptr(dev)),
          "vpn_fp32_peak_probe")
    return {"ffma": a.value, "ffma2": b.value}


# --------------------------------------------------------------------------------------
# GCN vertex-feature pooling (modules/network/gcn.py:84-164)
# --------------------------------------------------------------------------------------
def image_bounds(imgs: torch.Tensor, threshold: float = 0.03) -> torch.Tensor:
    """GCNModel.get_bound_of_images (gcn.py:90-133): (B,C,H,W) -> (B,4) normalised [x lo, x hi, y lo, y hi].  One launch;
    the reference walks columns and rows in Python and reads device scalars at every step."""
    assert imgs.ndimension() == 4
    imgs = require(imgs.contiguous(), f32, "imgs")
    b, c, h, w = imgs.shape
    out = torch.empty((b, 4), dtype=f32, device=imgs.device)
    check(_lib.load().vpn_image_bounds(ptr(imgs), ptr(out), b, c, h, w, float(threshold), stream_ptr(imgs.device)),
          "vpn_image_bounds")
    return out


class _FeaturePool(torch.autograd.Function):
    """pooled (B, N, sum C) = bilinear samples of every feature map at the vertices' image positions."""

    @staticmethod
    def forward(ctx, points, bounds, *features):
        lib = _lib.load()
        points = require(points.contiguous(), f32, "points")
        bounds = require(bounds.contiguous(), f32, "bounds")
        feats = [require(f.contiguous(), f32, "features") for f in features]
        b, n = points.shape[:2]
        dev = points.device
        ctot = sum(f.shape[1] for f in feats)
        out = torch.empty((b, n, ctot), dtype=f32, device=dev)
        rng = torch.empty((b, 4), dtype=f32, device=dev)
        arg = torch.empty((b, 4), dtype=torch.int32, device=dev)
        if b > 0 and n > 0:
            check(lib.vpn_points_yz_range(ptr(points), ptr(rng), ptr(arg), b, n, stream_ptr(dev)), "vpn_points_yz_range")
            coff = 0
            for f in feats:
                assert f.dim() == 4 and f.shape[0] == b, "feature maps must be (B, C, H, W)"
                check(lib.vpn_feature_pool_fwd(ptr(f), ptr(points), ptr(bounds), ptr(rng), ptr(out), b, f.shape[1], f.shape[2],
                                               f.shape[3], n, ctot, coff, stream_ptr(dev)), "vpn_feature_pool_fwd")
                coff += f.shape[1]
        ctx.save_for_backward(points, bounds, rng, arg, *feats)
        return out

    @staticmethod
    def backward(ctx, grad_out):
        lib = _lib.load()
        points, bounds, rng, arg, *feats = ctx.saved_tensors
        b, n = points.shape[:2]
        dev = points.device
        grad_out = grad_out.contiguous()
        ctot = grad_out.shape[2]
        ggrid = torch.zeros((b, n, 2), dtype=f32, device=dev)
        gfeats = []
        coff = 0
        ws, nws = None, ctypes.c_size_t(0)
        if b > 0 and n > 0:
            check(lib.vpn_feature_pool_bwd_workspace_bytes(b, n, ctypes.byref(nws)), "vpn_feature_pool_bwd_workspace_bytes")
            ws = _scratch_bytes(nws.value, dev)
        for f in feats:
            gf = torch.empty_like(f)
            if b > 0 and n > 0:
                check(lib.vpn_feature_pool_bwd_sorted(ptr(f), ptr(points), ptr(bounds), ptr(rng), ptr(grad_out), ptr(gf), ptr(ggrid),
                                                      ptr(ws), nws.value, b, f.shape[1], f.shape[2], f.shape[3], n, ctot, coff,
                                                      stream_ptr(dev)), "vpn_feature_pool_bwd_sorted")
            else:
                gf.zero_()
            gfeats.append(gf)
            coff += f.shape[1]
        gp = None
        if ctx.needs_input_grad[0]:
            gp = torch.zeros_like(points)
            if b > 0 and n > 0:
                check(lib.vpn_feature_pool_points_bwd(ptr(points), ptr(bounds), ptr(rng), ptr(arg), ptr(ggrid), ptr(gp), b, n,
                                                      stream_ptr(dev)), "vpn_feature_pool_points_bwd")
        return (gp, None, *gfeats)


def perceptual_feature_pooling(perceptual_features, points: torch.Tensor, bounds: torch.Tensor) -> torch.Tensor:
    """GCNModel.perceptual_feature_pooling (gcn.py:135-164): list of (B,C_l,H_l,W_l) maps, points (B,N,3), bounds (B,4)
    -> (B, N, sum C_l).  Differentiable w.r.t. the maps and the points (through the grid and the per-sample range)."""
    assert points.ndimension() == 3
    assert bounds.ndimension() == 2
    return _FeaturePool.apply(points, bounds, *perceptual_features)
