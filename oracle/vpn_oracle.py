"""CPU oracle for the primitive-assembly + loss hot path.  TEST INFRASTRUCTURE ONLY.

This module restates, in plain torch-CPU / numpy, the arithmetic of the reference
(hank-kuo-cs/Volumetric-Primitives-Net) for the path SURVEY.md section 8 scopes:
transform -> sampling -> Chamfer / VP-diverse, meshing -> soft silhouette -> image loss.
Only `tests/`, `__graft_entry__.smoke()` and `bench.py`'s cpu_baseline / `--impl reference`
legs may import it, and only as the checker or the timed CPU baseline.  The product package
never imports anything from `oracle/`.

Parity status
-------------
* transform / sampling / Chamfer / VP-diverse: PINNED.  `oracle/make_golden.py` imports the
  reference's own modules from /root/reference (package-__init__ bypass, CPU patch of
  rotate.py:34) and stores inputs + outputs under tests/golden/; tests/test_oracle_golden.py
  checks every function below against those vectors.
* meshing (template scale + transform + compose): PINNED through the same vectors, with the
  OBJ parsing restated here because kaolin's TriangleMesh.from_obj is not available.
* soft-silhouette renderer (kaolin v0.1 DIB-R, a third-party dependency that is neither
  vendored nor pinned by the reference and is not installed here): PARITY UNPINNED.  The
  functions in the "render" section restate the published DIB-R algorithm (Chen et al.,
  NeurIPS 2019) with kaolin v0.1's default constants as recalled in SURVEY.md section 8(a-R).

* mesh surface sampling (kaolin v0.1 TriangleMesh.sample, call sites train_sphere.py:71-80 and
  dataset/dataset.py:162-165; same absent dependency): PARITY UNPINNED.  `mesh_sample` restates
  kaolin v0.1's published formula (area-weighted face choice, sqrt-u barycentric point) with the
  three random draws made explicit inputs; kaolin's own RNG stream (Categorical.sample + two
  Uniform.sample) cannot be replayed, so parity beyond "same distribution" is not claimed.

* EMD auction loss (modules/loss/emd, SURVEY.md section 8f "next" #1): the reference implementation is
  non-deterministic by construction (racing writes decide which of several equal bidders wins,
  emd_cuda.cu:181-194, and its value arithmetic mixes double and contracted fp32, :141,219) and cannot be
  run here (no GPU in the build container; the extension does not compile against current ATen).
  `emd_auction` restates its algorithm with the races resolved deterministically (lowest index wins) and
  plain separately-rounded fp32 arithmetic: PARITY IS STATISTICAL - same auction, same eps / iteration
  schedule; tests check validity and near-optimality of the assignment against scipy's exact solver.

Every function cites the reference file:line it follows (paths relative to /root/reference).
"""
from __future__ import annotations

import math
from typing import List, Optional, Sequence, Tuple

import numpy as np
import torch

# rotate.py:4 and sphere.py:7 both hard-code this float32-rounded value of pi.
PI = 3.1415927410125732

# config.py:12-13
CD_W1 = 1.0
CD_W2 = 1.0


# --------------------------------------------------------------------------------------
# transform  (modules/transform/rotate.py, translate.py, transform.py)
# --------------------------------------------------------------------------------------
def refine_quaternions(q: torch.Tensor) -> torch.Tensor:
    """rotate.py:59-72.  (axis, turn-fraction) -> unit quaternion (x, y, z, w).

    half_angle = ((q3 mod 1) * 2 * PI) / 2 ; raw = (axis * sin(half_angle), cos(half_angle));
    result = raw / ||raw||_2.  The axis is NOT normalised first.
    """
    half = torch.div((q[:, 3] % 1) * 2 * PI, 2)
    s = torch.sin(half)
    raw = torch.cat([q[:, :3] * s[:, None], torch.cos(half)[:, None]], dim=1)
    return raw / torch.norm(raw, dim=1)[:, None]


def rotation_matrices(qn: torch.Tensor) -> torch.Tensor:
    """rotate.py:28-46.  Unit quaternion -> (B,3,3), entry order and signs as the reference."""
    x, y, z, w = qn[:, 0], qn[:, 1], qn[:, 2], qn[:, 3]
    x2, y2, z2, w2 = x * x, y * y, z * z, w * w
    xy, zw, xz, yw, yz, xw = x * y, z * w, x * z, y * w, y * z, x * w
    r0 = torch.stack([x2 - y2 - z2 + w2, 2 * (xy - zw), 2 * (xz + yw)], dim=1)
    r1 = torch.stack([2 * (xy + zw), -x2 + y2 - z2 + w2, 2 * (yz - xw)], dim=1)
    r2 = torch.stack([2 * (xz - yw), 2 * (yz + xw), -x2 - y2 + z2 + w2], dim=1)
    return torch.stack([r0, r1, r2], dim=1)


def _fma(a: torch.Tensor, b: torch.Tensor, c: torch.Tensor) -> torch.Tensor:
    """a * b + c rounded once to fp32: the product of two fp32 values is exact in fp64, and the fp64 sum rounds to the
    same fp32 value as the exact sum unless it lands exactly halfway between two fp32 values."""
    return (a.double() * b.double() + c.double()).float()


def rotate_points(points: torch.Tensor, q: torch.Tensor) -> torch.Tensor:
    """rotate.py:7-25.  out[b,n,:] = R(q[b]) @ points[b,n,:] (torch.bmm with k = 3).

    torch.bmm's rounding depends on the host: below 400 multiply-adds per matrix ATen sums the products itself,
    ((r0 x + r1 y) + r2 z) with every operation rounded; above, the CPU BLAS does, and whether its kernel fuses the
    multiply-adds depends on the instruction set.  tests/golden/ was recorded where it evaluated
    fma(r2, z, fma(r1, y, r0 x)).  Both orders are written out so that the oracle gives the same bits on every host,
    except where _fma's fp64 sum lands exactly halfway between two fp32 values and rounds twice (rare).  With torch.bmm,
    MKL_ENABLE_INSTRUCTIONS=AVX2 alone fails four golden tests of tests/test_oracle_golden.py."""
    assert points.ndimension() == 3 and points.size(-1) == 3      # rotate.py:49-51
    assert q.ndimension() == 2 and q.size(-1) == 4                # rotate.py:54-56
    mats = rotation_matrices(refine_quaternions(q))
    x, y, z = points[..., 0], points[..., 1], points[..., 2]
    rows = []
    for i in range(3):
        r0, r1, r2 = (mats[:, i, j, None] for j in range(3))
        if 9 * points.size(1) < 400:
            rows.append((r0 * x + r1 * y) + r2 * z)
        else:
            rows.append(_fma(r2, z, _fma(r1, y, r0 * x)))
    return torch.stack(rows, dim=2)


def translate_points(points: torch.Tensor, t: torch.Tensor) -> torch.Tensor:
    """translate.py:4-8."""
    assert points.ndimension() == 3 and points.size(-1) == 3
    assert t.ndimension() == 2 and t.size(-1) == 3
    return points + t[:, None, :]


def transform_points(points: torch.Tensor, q: torch.Tensor, t: torch.Tensor) -> torch.Tensor:
    """transform.py:6-18.  translate(rotate(points, q), t) with the reference's shape checks."""
    assert points.ndimension() == 3 and points.size(-1) == 3
    b = points.size(0)
    assert q.size() == (b, 4) and t.size() == (b, 3)
    return translate_points(rotate_points(points, q), t)


def _axis_quat(axis: Sequence[float], turns: torch.Tensor) -> torch.Tensor:
    b = turns.numel()
    ax = torch.tensor([list(axis)], dtype=torch.float32).repeat(b, 1)
    return torch.cat([ax, turns.reshape(-1, 1)], dim=1)


def rotate_points_forward_x_axis(points: torch.Tensor, angles: torch.Tensor) -> torch.Tensor:
    """transform.py:76-94.  Rotate about +x by angles/360 turns."""
    assert points.ndimension() == 3 and angles.ndimension() == 1
    return rotate_points(points, _axis_quat((1, 0, 0), angles.reshape(-1, 1) / 360))


def view_to_obj_points(points, dists, elevs, azims, angles) -> torch.Tensor:
    """transform.py:21-47.  Undo the camera: x-rotation by -angle, then y' (y rotated about -z by
    elev) by -azim, then -z by -elev, then scale by dist."""
    assert points.ndimension() == 3
    assert dists.ndimension() == elevs.ndimension() == azims.ndimension() == 1
    b = points.size(0)
    d, e, a = dists.view(-1, 1), elevs.view(-1, 1) / 360, azims.view(-1, 1) / 360
    pts = rotate_points_forward_x_axis(points, -angles)
    y = torch.tensor([[0.0, 1.0, 0.0]]).repeat(b, 1)
    y = rotate_points(y[:, None, :], _axis_quat((0, 0, -1), e)).squeeze(1)
    pts = rotate_points(pts, torch.cat([y, -a], dim=1))
    pts = rotate_points(pts, _axis_quat((0, 0, -1), -e))
    return pts * d[:, :, None]


def obj_to_view_points(points, dists, elevs, azims) -> torch.Tensor:
    """transform.py:50-73.  Forward camera transform, divide by dist."""
    assert points.ndimension() == 3
    assert dists.ndimension() == elevs.ndimension() == azims.ndimension() == 1
    b = points.size(0)
    d, e, a = dists.view(-1, 1), elevs.view(-1, 1) / 360, azims.view(-1, 1) / 360
    q = _axis_quat((0, 0, -1), e)
    pts = rotate_points(points, q)
    y = torch.tensor([[0.0, 1.0, 0.0]]).repeat(b, 1)
    y = rotate_points(y[:, None, :], q).squeeze(1)
    pts = rotate_points(pts, torch.cat([y, a], dim=1))
    return pts / d[:, :, None]


# --------------------------------------------------------------------------------------
# sampling  (modules/sampling/sphere.py, cuboid.py, sampling.py)
# The reference draws its uniforms with torch.rand on DEVICE; here they are explicit inputs,
# in the reference's draw order, so that oracle and kernels consume identical numbers.
# --------------------------------------------------------------------------------------
def sphere_canonical(v: torch.Tensor, u_elev: torch.Tensor, u_azim: torch.Tensor) -> torch.Tensor:
    """sphere.py:22-43.  v (B,3); u_elev,u_azim (B,N,1) in [0,1) (elev is drawn first, :26-27)."""
    elev = -torch.acos(1 - 2 * u_elev) + PI * 0.5
    azim = u_azim * 2 * PI
    dist = torch.ones_like(u_elev)
    xs = dist * torch.cos(elev) * torch.sin(azim)
    ys = dist * torch.sin(elev)
    zs = dist * torch.cos(elev) * torch.cos(azim)
    return torch.cat([xs, ys, zs], dim=2) * v[:, None, :]


def cuboid_face_counts(v: torch.Tensor, num_points: int) -> torch.Tensor:
    """cuboid.py:30-53.  (B,6) int32 points per face in order +w,-w,+h,-h,+d,-d.  Faces 0..4 are
    round-half-even of N*area/total; face 5 takes the remainder (may be <= 0)."""
    w, h, d = v[:, 0:1], v[:, 1:2], v[:, 2:3]
    hd, dw, wh = h * d, d * w, w * h
    area = torch.cat([hd, hd, dw, dw, wh, wh], dim=1)
    total = (hd + dw + wh) * 2
    counts = (torch.full_like(area, num_points) * (area / total)).round().int()
    counts[:, 5] = num_points - counts[:, :5].sum(dim=1).int()
    return counts


def cuboid_canonical(v: torch.Tensor, u: torch.Tensor) -> torch.Tensor:
    """cuboid.py:8-22,56-101.  v (B,3); u (B,N,3) in [0,1).  Volume sample (-1+2u)*v, then the
    points of the contiguous index range owned by face i get coordinate i//2 pinned to +-v."""
    b, n, _ = u.shape
    counts = cuboid_face_counts(v, n)
    pts = (-1 + 2 * u) * v[:, None, :]
    start = torch.zeros(b, dtype=torch.int64)
    idx = torch.arange(n)[None, :]
    for face in range(6):
        axis, sign = face // 2, (-1.0 if face % 2 else 1.0)
        cnt = counts[:, face].to(torch.int64)
        lo = start[:, None]
        hi = (start + cnt)[:, None]
        # python slice [lo:hi] on a length-n axis; lo, hi >= 0 here except hi < lo (empty)
        sel = (idx >= lo) & (idx < hi)
        pinned = (sign * v[:, axis])[:, None].expand(b, n)
        coord = torch.where(sel, pinned, pts[:, :, axis])
        pts = torch.cat([pts[:, :, :axis], coord[:, :, None], pts[:, :, axis + 1:]], dim=2)
        start = start + cnt
    return pts


def sphere_sampling(v, q, t, u_elev, u_azim) -> torch.Tensor:
    """sampling.py:26-38 with explicit uniforms."""
    b = v.size(0)
    assert v.size() == (b, 3) and q.size() == (b, 4) and t.size() == (b, 3)   # sampling.py:48-52
    return transform_points(sphere_canonical(v, u_elev, u_azim), q, t)


def cuboid_sampling(v, q, t, u) -> torch.Tensor:
    """sampling.py:12-24 with explicit uniforms."""
    b = v.size(0)
    assert v.size() == (b, 3) and q.size() == (b, 4) and t.size() == (b, 3)
    return transform_points(cuboid_canonical(v, u), q, t)


def sample_predict_points(kind: str, volumes, rotates, translates, uniforms) -> torch.Tensor:
    """train.py:105-120.  K primitives, each sampled then concatenated along dim 1 (primitive-major).
    volumes/rotates/translates: (B,K,3|4|3).  uniforms: sphere (B,K,N,2) [elev, azim]; cuboid (B,K,N,3)."""
    k = volumes.size(1)
    out = []
    for i in range(k):
        if kind == "sphere":
            out.append(sphere_sampling(volumes[:, i], rotates[:, i], translates[:, i],
                                       uniforms[:, i, :, 0:1], uniforms[:, i, :, 1:2]))
        else:
            out.append(cuboid_sampling(volumes[:, i], rotates[:, i], translates[:, i], uniforms[:, i]))
    return torch.cat(out, dim=1)


# --------------------------------------------------------------------------------------
# Chamfer / VP-diverse  (modules/loss/chamfer_distance.py, vp_diverse.py)
# --------------------------------------------------------------------------------------
def chamfer_dense(p1: torch.Tensor, p2: torch.Tensor, each_batch: bool = False,
                  w1: float = CD_W1, w2: float = CD_W2) -> torch.Tensor:
    """chamfer_distance.py:10-30, op for op (dense (B,P,M,3) broadcast).  Differentiable; this is
    also the CPU baseline that bench.py times, because it is the reference's own formulation."""
    assert p1.ndimension() == 3 and p1.size(-1) == 3
    assert p2.ndimension() == 3 and p2.size(-1) == 3
    diff = p1[:, :, None, :] - p2[:, None, :, :]
    dist = torch.sum(diff * diff, dim=3)
    d1 = torch.sqrt(dist)
    d2 = torch.sqrt(torch.transpose(dist, 1, 2))
    m1, _ = torch.min(d1, dim=2)
    m2, _ = torch.min(d2, dim=2)
    loss = w1 * m1.mean(1) + w2 * m2.mean(1)
    return loss if each_batch else loss.mean()


def _ieee_sqrt(x: torch.Tensor) -> torch.Tensor:
    """Correctly rounded fp32 sqrt.  torch.sqrt on large contiguous CPU tensors goes through MKL VML
    and is 1 ulp off for ~0.7% of inputs (measured here); the reference's own device is 'cuda'
    (config.py:2) where torch.sqrt is the IEEE sqrt.rn.f32, so the oracle pins the IEEE value."""
    return torch.from_numpy(np.sqrt(x.detach().numpy()))


def chamfer_nn(p1: torch.Tensor, p2: torch.Tensor, row_block: int = 2048):
    """Chunked evaluation of the same per-pair arithmetic as chamfer_distance.py:14-23:
    d = fl(fl(fl(dx*dx)+fl(dy*dy))+fl(dz*dz)), v = sqrt(d), min over the other cloud with the FIRST
    index on ties (torch.min semantics).  Returns (min1 (B,P), idx1 (B,P) int64, min2 (B,M), idx2)."""
    b, p, _ = p1.shape
    m = p2.size(1)
    min1 = torch.empty(b, p); idx1 = torch.empty(b, p, dtype=torch.int64)
    min2 = torch.full((b, m), float("inf")); idx2 = torch.zeros(b, m, dtype=torch.int64)
    for s in range(0, p, row_block):
        e = min(p, s + row_block)
        diff = p1[:, s:e, None, :] - p2[:, None, :, :]
        dist = _ieee_sqrt(torch.sum(diff * diff, dim=3))
        mv, mi = torch.min(dist, dim=2)
        min1[:, s:e], idx1[:, s:e] = mv, mi
        cv, ci = torch.min(dist, dim=1)
        better = cv < min2            # strict: earlier row block keeps ties (first index)
        min2 = torch.where(better, cv, min2)
        idx2 = torch.where(better, ci + s, idx2)
    return min1, idx1, min2, idx2


def chamfer_from_nn(min1, min2, each_batch=False, w1=CD_W1, w2=CD_W2) -> torch.Tensor:
    """chamfer_distance.py:25-30."""
    loss = w1 * min1.mean(1) + w2 * min2.mean(1)
    return loss if each_batch else loss.mean()


def chamfer_grad_from_nn(p1, p2, min1, idx1, min2, idx2, g1, g2):
    """Closed form of what autograd does through chamfer_distance.py:14-23 given the arg-mins.
    g1 (B,P), g2 (B,M): upstream grads of min1/min2.  Returns (grad_p1, grad_p2).  A selected pair at
    distance 0 yields NaN exactly as sqrt's backward does in the reference (inf * 0)."""
    b, p, _ = p1.shape
    m = p2.size(1)
    gp1 = torch.zeros_like(p1); gp2 = torch.zeros_like(p2)
    bi = torch.arange(b)[:, None]
    d1 = p1 - p2[bi, idx1]                               # (B,P,3)
    c1 = (g1 / (2 * min1))[:, :, None] * (2 * d1)
    gp1 += c1
    gp2.index_put_((bi.expand(b, p), idx1), -c1, accumulate=True)
    d2 = p1[bi, idx2] - p2                               # (B,M,3)
    c2 = (g2 / (2 * min2))[:, :, None] * (2 * d2)
    gp2 -= c2
    gp1.index_put_((bi.expand(b, m), idx2), c2, accumulate=True)
    return gp1, gp2


def vp_diverse(translates: Sequence[torch.Tensor], gt_points: torch.Tensor) -> torch.Tensor:
    """vp_diverse.py:12-18.  Chamfer between the K primitive centres and the target, w1=.5, w2=1."""
    assert isinstance(translates, list)
    centres = torch.cat([t[:, None, :] for t in translates], dim=1)
    return chamfer_dense(centres, gt_points, w1=0.5, w2=1.0)


# --------------------------------------------------------------------------------------
# EMD auction  (modules/loss/emd/emd_cuda.cu, emd_module.py)
# --------------------------------------------------------------------------------------
def emd_auction(xyz1: np.ndarray, xyz2: np.ndarray, eps: float, iters: int, row_block: int = 512):
    """emd_cuda_forward (emd_cuda.cu:227-281) for one sample: xyz1 (n,3) bidders, xyz2 (n,3) objects, fp32.
    Returns (dist (n,) fp32 squared distance to the assigned object, assignment (n,) int32).

    Per iteration (emd_cuda.cu:257-269): the unassigned bidders each find the object maximising
    value = 3 - |x2 - x1| - price (Bid, :95-179; best = first maximum, better = second largest value),
    bid increment = best - better + eps, per-object maximum increment; the bidder whose increment is within
    1e-6 of the object's maximum wins it (GetMax, :181-194; here the LOWEST such bidder - the reference lets
    racing writes decide), evicts the previous owner, and the price rises by its increment (Assign, :196-216).
    In the last iteration every still unassigned bidder takes its preferred object unconditionally, so the
    result need not be a bijection.  dist = |x1 - x2[assignment]|^2 (CalcDist, :218-226).
    Arithmetic: fp32, every operation rounded separately ((dx^2 + dy^2) + dz^2, IEEE sqrt, (3 - s) - price)."""
    f32 = np.float32
    x1 = np.ascontiguousarray(xyz1, dtype=f32)
    x2 = np.ascontiguousarray(xyz2, dtype=f32)
    n = x1.shape[0]
    assert x2.shape[0] == n and iters >= 1
    assignment = np.full(n, -1, dtype=np.int32)
    assignment_inv = np.full(n, -1, dtype=np.int32)
    price = np.zeros(n, dtype=f32)
    max_inc = np.full(n, f32(-1e9), dtype=f32)
    epsf = f32(eps)
    for it in range(iters):
        last = it == iters - 1
        un = np.nonzero(assignment == -1)[0]
        if un.size == 0:
            continue
        best = np.empty(un.size, dtype=f32); better = np.empty(un.size, dtype=f32)
        best_i = np.empty(un.size, dtype=np.int64)
        for r0 in range(0, un.size, row_block):
            rows = un[r0:r0 + row_block]
            d = x2[None, :, :] - x1[rows, None, :]
            d2 = (d[..., 0] * d[..., 0] + d[..., 1] * d[..., 1]) + d[..., 2] * d[..., 2]
            val = (f32(3.0) - np.sqrt(d2)) - price[None, :]
            bi = np.argmax(val, axis=1)                                 # first maximum
            ar = np.arange(rows.size)
            bv = val[ar, bi]
            val[ar, bi] = -np.inf
            sv = np.maximum(val.max(axis=1), f32(-1e9)) if n > 1 else np.full(rows.size, f32(-1e9), dtype=f32)
            best[r0:r0 + rows.size] = bv; better[r0:r0 + rows.size] = sv; best_i[r0:r0 + rows.size] = bi
        inc = ((best - better).astype(f32) + epsf).astype(f32)
        np.maximum.at(max_inc, best_i, inc)
        # winner of an object: lowest bidder whose increment is within 1e-6 (compared in double) of the maximum
        mx = max_inc[best_i].astype(np.float64)
        ok = (inc.astype(np.float64) - 1e-6 <= mx) & (mx <= inc.astype(np.float64) + 1e-6)
        winner = np.full(n, np.iinfo(np.int32).max, dtype=np.int64)
        np.minimum.at(winner, best_i[ok], un[ok])
        for u, j in enumerate(un):                                       # ascending bidder order
            t = best_i[u]
            if last or winner[t] == j:
                old = assignment_inv[t]
                if not last and old != -1:
                    assignment[old] = -1
                assignment_inv[t] = j
                assignment[j] = t
                price[t] = f32(price[t] + inc[u])
                max_inc[t] = f32(-1e9)
    d = x1 - x2[assignment]
    dist = (d[:, 0] * d[:, 0] + d[:, 1] * d[:, 1]) + d[:, 2] * d[:, 2]
    return dist.astype(f32), assignment


def emd_backward(xyz1: np.ndarray, xyz2: np.ndarray, assignment: np.ndarray, grad_dist: np.ndarray) -> np.ndarray:
    """NmDistanceGradKernel (emd_cuda.cu:283-300): d dist / d xyz1 = 2 g (x1 - x2[assignment]); xyz2 gets no
    gradient (emd_module.py:66-67 returns zeros)."""
    g = (grad_dist.astype(np.float32) * np.float32(2.0))[:, None]
    return (g * (xyz1.astype(np.float32) - xyz2.astype(np.float32)[assignment])).astype(np.float32)


# --------------------------------------------------------------------------------------
# meshing  (modules/meshing/sphere.py, cuboid.py, meshing.py)
# --------------------------------------------------------------------------------------
def parse_obj(text: str) -> Tuple[np.ndarray, np.ndarray]:
    """What TriangleMesh.from_obj yields for the reference's templates (meshing/sphere.py:32,
    meshing/cuboid.py:31, train_sphere.py:53): 'v x y z' rows -> float32 (V,3); 'f a b c' or
    'f a//n b//n c//n' rows -> int64 (F,3), 1-based -> 0-based."""
    vs, fs = [], []
    for line in text.splitlines():
        tok = line.split()
        if not tok:
            continue
        if tok[0] == "v":
            vs.append([float(x) for x in tok[1:4]])
        elif tok[0] == "f":
            fs.append([int(x.split("/")[0]) - 1 for x in tok[1:4]])
    return np.asarray(vs, dtype=np.float32), np.asarray(fs, dtype=np.int64)


def sphere_template(raw_vertices: torch.Tensor) -> torch.Tensor:
    """meshing/sphere.py:30-36.  Zero-centre, divide by the mean vertex radius."""
    v = raw_vertices - torch.mean(raw_vertices, 0)
    return v / torch.mean(torch.norm(v, dim=1))


def mesh_vertices(template: torch.Tensor, v, q, t) -> torch.Tensor:
    """meshing/sphere.py:8-27 / cuboid.py:8-27.  (V,3) template scaled by v[b] then posed: (B,V,3)."""
    b = v.size(0)
    assert v.size() == (b, 3) and q.size() == (b, 4) and t.size() == (b, 3)   # meshing.py:49-55
    return transform_points(template[None, :, :] * v[:, None, :], q, t)


def compose_meshes(vertices: List[torch.Tensor], faces: List[torch.Tensor]):
    """meshing/meshing.py:28-46.  Concatenate vertices; faces get a running vertex offset."""
    off, fo = 0, []
    for vtx, f in zip(vertices, faces):
        fo.append(f + off)
        off += vtx.size(0)
    return torch.cat(vertices), torch.cat(fo)


def mesh_face_cdf(verts: np.ndarray, faces: np.ndarray, lanes: int = 256, eps: float = 1e-10) -> np.ndarray:
    """Cumulative area shares of the faces, fp32, as kaolin v0.1 TriangleMesh.sample computes the areas
    (call site train_sphere.py:76): edge vectors x = v0 - v1, y = v1 - v2, area = sqrt(a + b + c) / 2 with
    a, b, c the squared cross-product components, shares = area / (sum(area) + eps).  Every operation is
    rounded to fp32 separately (a chain of torch ops).  The summation order is fixed: `lanes` consecutive
    chunks of ceil(F / lanes) faces, running sum inside a chunk, chunk totals added in order (kaolin's
    torch.sum / Categorical normalisation order is unspecified)."""
    f32 = np.float32
    v = verts.astype(f32)
    x = v[faces[:, 0]] - v[faces[:, 1]]
    y = v[faces[:, 1]] - v[faces[:, 2]]
    a = x[:, 1] * y[:, 2] - x[:, 2] * y[:, 1]
    b = x[:, 2] * y[:, 0] - x[:, 0] * y[:, 2]
    c = x[:, 0] * y[:, 1] - x[:, 1] * y[:, 0]
    area = np.sqrt((a * a + b * b) + c * c) / f32(2.0)
    nf = faces.shape[0]
    per = (nf + lanes - 1) // lanes
    local = np.zeros(nf, dtype=f32)
    totals = np.zeros(lanes, dtype=f32)
    for lane in range(lanes):
        run = f32(0.0)
        for f in range(lane * per, min(nf, (lane + 1) * per)):
            run = f32(run + area[f])
            local[f] = run
        totals[lane] = run
    base = np.zeros(lanes, dtype=f32)
    acc = f32(0.0)
    for lane in range(lanes):
        base[lane] = acc
        acc = f32(acc + totals[lane])
    denom = f32(acc + f32(eps))
    lane_of = np.minimum(np.arange(nf) // per, lanes - 1)
    return ((local + base[lane_of]).astype(f32) / denom).astype(f32)


def mesh_sample(verts: torch.Tensor, faces: torch.Tensor, u: torch.Tensor):
    """kaolin v0.1 TriangleMesh.sample(n) (train_sphere.py:71-80) with explicit draws u (n,3) in [0,1):
    face = first face whose cumulative area share exceeds u[:,0] (inverse CDF in place of Categorical.sample),
    su = sqrt(u[:,1]), p = (1 - su) v0 + su (1 - u2) v1 + su u2 v2.  Differentiable w.r.t. verts through the
    barycentric weights, as kaolin's index_select chain is.  Returns (points (n,3), face_idx (n,) int64)."""
    cdf = torch.from_numpy(mesh_face_cdf(verts.detach().numpy(), faces.numpy()))
    nf = faces.shape[0]
    face = torch.searchsorted(cdf, u[:, 0].contiguous(), right=True).clamp(max=nf - 1)
    sel = faces[face]
    v0, v1, v2 = verts[sel[:, 0]], verts[sel[:, 1]], verts[sel[:, 2]]
    su = _ieee_sqrt(u[:, 1:2])          # torch-CPU sqrt (MKL VML) is 1 ulp off for some inputs; the reference's device is IEEE
    vv = u[:, 2:3]
    pts = ((1.0 - su) * v0 + (su * (1.0 - vv)) * v1) + (su * vv) * v2
    return pts, face


def compose_primitive_meshes(template, faces, volumes, rotates, translates):
    """train.py:123-149.  K primitives of one template -> per-sample composed mesh.
    Returns vertices (B, K*V, 3) and faces (K*F, 3) int64 (identical topology for every sample)."""
    k = volumes.size(1)
    vs = [mesh_vertices(template, volumes[:, i], rotates[:, i], translates[:, i]) for i in range(k)]
    v_all = torch.cat(vs, dim=1)
    nv = template.size(0)
    f_all = torch.cat([faces + i * nv for i in range(k)], dim=0)
    return v_all, f_all


# --------------------------------------------------------------------------------------
# render: soft silhouette (kaolin v0.1 DIBRenderer, VertexColor mode).  PARITY UNPINNED.
# Call sites: render/vertex_renderer.py:7,18,24 ; loss/silhouette.py:13-23.
# --------------------------------------------------------------------------------------
DIBR_FOVY_DEG = 49.13434207744484
DIBR_EXPAND = 0.02
DIBR_KNUM = 30
DIBR_MULTIPLIER = 1000.0
DIBR_DELTA = 7000.0
DIBR_EPS = 1e-15


def look_at_camera(azim_deg: float, elev_deg: float, dist: float):
    """kaolin compute_camera_params: camera position on a sphere, rows of the rotation are the unit
    X = Y0 x Z, Y = Z x X, Z = cam_pos axes (Y0 = +y).  Returns (rot (3,3), pos (3,)) float32."""
    theta, phi = np.deg2rad(azim_deg), np.deg2rad(elev_deg)
    cam_y = dist * np.sin(phi)
    tmp = dist * np.cos(phi)
    pos = np.array([tmp * np.cos(theta), cam_y, tmp * np.sin(theta)], dtype=np.float64)
    az = pos.copy()
    ay = np.array([0.0, 1.0, 0.0])
    ax = np.cross(ay, az)
    ay = np.cross(az, ax)
    rot = np.stack([ax / np.linalg.norm(ax), ay / np.linalg.norm(ay), az / np.linalg.norm(az)])
    return torch.tensor(rot, dtype=torch.float32), torch.tensor(pos, dtype=torch.float32)


def projection_vector() -> torch.Tensor:
    """kaolin perspectiveprojectionnp(fovy, ratio=1): (1/tan(fovy/2), 1/tan(fovy/2), -1)."""
    tf = np.tan(np.deg2rad(DIBR_FOVY_DEG) / 2.0)
    return torch.tensor([1.0 / tf, 1.0 / tf, -1.0], dtype=torch.float32)


def project_vertices(verts: torch.Tensor, rot: torch.Tensor, pos: torch.Tensor):
    """kaolin perspective_projection: camera-space points and their screen xy.
    verts (B,V,3); rot (B,3,3); pos (B,3).  Returns cam (B,V,3), xy (B,V,2)."""
    # kaolin: torch.matmul (cuBLAS batched GEMM, accumulation order unspecified).  The restatement pins ONE order,
    # (dx r_k0 + dy r_k1) + dz r_k2 with every operation rounded separately: the rasteriser works on coordinates x 1000
    # and cancels, so a 1-ulp difference in a projected vertex moves alpha by ~1e-4 and can flip a nearest-edge choice.
    d = verts - pos[:, None, :]
    cam = torch.stack([(d[..., 0] * rot[:, k, 0, None] + d[..., 1] * rot[:, k, 1, None]) + d[..., 2] * rot[:, k, 2, None]
                       for k in range(3)], dim=-1)
    proj = projection_vector()
    xyz = cam * proj[None, None, :]
    return cam, xyz[:, :, :2] / xyz[:, :, 2:3]


def soft_silhouette(verts: torch.Tensor, faces: torch.Tensor, rot: torch.Tensor, pos: torch.Tensor,
                    height: int, width: int, soft_cull_backfaces: bool = False, pixels=None) -> torch.Tensor:
    """Soft alpha channel of DIB-R's VertexColor renderer: (B,H,W).  Differentiable w.r.t. verts.
    `pixels` (1-D LongTensor of flat pixel indices h*W+w) restricts the evaluation to those pixels and returns
    (B, len(pixels)) - used to check BASELINE-size meshes (F = 16 128 / 32 256) on a pixel subset.

    Back faces (normal.z < 0): the hard pass skips them (`if (direction < 0) continue;` in DIB-R's render kernel); the
    soft pass does NOT (its kernel receives only the 2-D points, the expanded boxes and the coverage index - SURVEY.md
    8(a-R) lists the back-face skip for the hard pass only).  soft_cull_backfaces=True is the other reading (skip
    them in both passes), kept selectable because Kaolin v0.1 cannot be run here to settle it.

    Hard pass: a pixel centre strictly inside (barycentrics >= 0) the tight bbox of any front face
    (normal.z >= 0) is covered -> alpha 1.  Soft pass, uncovered pixels only: faces are visited in
    index order; a face whose bbox expanded by `expand` contains the pixel contributes
    prob = exp(-delta * d2 / mult^2) with d2 the squared screen distance (x mult) to the triangle
    (min over 3 edge-perpendicular distances whose foot lies on the segment, else 4 mult^2, and 3
    vertex distances); at most `knum` faces are recorded; alpha = 1 - prod(1 - prob).
    The selections (coverage, bbox, first-knum, min case, foot test) carry no gradient.
    """
    b, v, _ = verts.shape
    f = faces.size(0)
    cam, xy = project_vertices(verts, rot, pos)
    mult = DIBR_MULTIPLIER
    # per-face data
    p0c, p1c, p2c = cam[:, faces[:, 0]], cam[:, faces[:, 1]], cam[:, faces[:, 2]]       # (B,F,3)
    normal_z = torch.cross(p1c - p0c, p2c - p0c, dim=2)[:, :, 2]                          # (B,F)
    s = torch.stack([xy[:, faces[:, 0]], xy[:, faces[:, 1]], xy[:, faces[:, 2]]], dim=2) * mult  # (B,F,3,2)
    bmin = s.min(dim=2)[0]
    bmax = s.max(dim=2)[0]
    bmin2 = bmin - DIBR_EXPAND * mult
    bmax2 = bmax + DIBR_EXPAND * mult
    # pixel centres
    wi = torch.arange(width, dtype=torch.float32)
    hi = torch.arange(height, dtype=torch.float32)
    x0 = (mult / width) * (2 * wi + 1 - width)            # (W,)
    y0 = (mult / height) * (height - 2 * hi - 1)          # (H,)
    X = x0[None, :].expand(height, width).reshape(-1)     # (HW,)
    Y = y0[:, None].expand(height, width).reshape(-1)
    if pixels is not None:
        X, Y = X[pixels], Y[pixels]
    out = torch.zeros(b, X.numel())
    front = (normal_z >= 0)                                # direction < 0 -> skipped
    for bi in range(b):
        sb = s[bi]                                         # (F,3,2)
        ax, ay = sb[:, 0, 0][None], sb[:, 0, 1][None]      # (1,F)
        bx, by = sb[:, 1, 0][None], sb[:, 1, 1][None]
        cx, cy = sb[:, 2, 0][None], sb[:, 2, 1][None]
        Xp, Yp = X[:, None], Y[:, None]                    # (HW,1)
        with torch.no_grad():
            in_tight = (Xp >= bmin[bi, :, 0][None]) & (Xp < bmax[bi, :, 0][None]) & \
                       (Yp >= bmin[bi, :, 1][None]) & (Yp < bmax[bi, :, 1][None])
            m_, p_, n_, q_ = bx - ax, by - ay, cx - ax, cy - ay
            s_, t_ = Xp - ax, Yp - ay
            k1 = s_ * q_ - n_ * t_
            k2 = m_ * t_ - s_ * p_
            k3 = m_ * q_ - n_ * p_
            w1 = k1 / (k3 + DIBR_EPS)
            w2 = k2 / (k3 + DIBR_EPS)
            w0 = 1 - w1 - w2
            inside = in_tight & front[bi][None] & (w0 >= 0) & (w1 >= 0) & (w2 >= 0)
            covered = inside.any(dim=1)                    # (HW,)
            in_soft = (Xp >= bmin2[bi, :, 0][None]) & (Xp < bmax2[bi, :, 0][None]) & \
                      (Yp >= bmin2[bi, :, 1][None]) & (Yp < bmax2[bi, :, 1][None])
            if soft_cull_backfaces:
                in_soft = in_soft & front[bi][None]
            rank = torch.cumsum(in_soft.to(torch.int32), dim=1)
            use = in_soft & (rank <= DIBR_KNUM) & (~covered)[:, None]
        # squared distance pixel -> triangle, 6 cases
        pd = []
        vx = [ax, bx, cx]
        vy = [ay, by, cy]
        for i in range(3):
            x1, y1, x2, y2 = vx[i], vy[i], vx[(i + 1) % 3], vy[(i + 1) % 3]
            A = y2 - y1
            Bc = x1 - x2
            C = x2 * y1 - x1 * y2
            up = A * Xp + Bc * Yp + C
            down = A * A + Bc * Bc
            with torch.no_grad():
                x3 = (Bc * Bc * Xp - A * Bc * Yp - A * C) / (down + DIBR_EPS)
                y3 = (A * A * Yp - A * Bc * Xp - Bc * C) / (down + DIBR_EPS)
                bad = ((x3 - x1) * (x3 - x2) + (y3 - y1) * (y3 - y2)) > 0
            perp = up * up / (down + DIBR_EPS)
            pd.append(torch.where(bad, torch.full_like(perp, 4 * mult * mult), perp))
        for i in range(3):
            pd.append((Xp - vx[i]) ** 2 + (Yp - vy[i]) ** 2)
        pd = torch.stack(pd, dim=2)                         # (HW,F,6)
        with torch.no_grad():
            case = torch.argmin(pd, dim=2, keepdim=True)    # first minimum, like the `>` scan
        d2 = torch.gather(pd, 2, case).squeeze(2)
        prob = torch.exp(-(DIBR_DELTA * d2 / mult / mult))
        one_minus = torch.where(use, 1 - prob, torch.ones_like(prob))
        alpha = 1 - torch.prod(one_minus, dim=1)
        out[bi] = torch.where(covered, torch.ones_like(alpha), alpha)
    return out if pixels is not None else out.view(b, height, width)


def silhouette_loss(verts, faces, gt, dists, elevs, azims, loss_func: str = "L1", soft_cull_backfaces: bool = False) -> torch.Tensor:
    """loss/silhouette.py:13-23 + render/vertex_renderer.py:15-26: per-sample look-at camera,
    soft alpha (B,1,H,W), then L1Loss / MSELoss (mean over B*H*W) vs gt (B,1,H,W)."""
    b = verts.size(0)
    h, w = gt.shape[-2:]
    cams = [look_at_camera(float(azims[i]), float(elevs[i]), float(dists[i])) for i in range(b)]
    rot = torch.stack([c[0] for c in cams])
    pos = torch.stack([c[1] for c in cams])
    alpha = soft_silhouette(verts, faces, rot, pos, h, w, soft_cull_backfaces=soft_cull_backfaces)[:, None]
    if loss_func == "L1":
        return (alpha - gt).abs().mean()
    return ((alpha - gt) ** 2).mean()


# --------------------------------------------------------------------------------------
# synthetic inputs (SURVEY.md section 8d) shared by tests, smoke() and bench.py
# --------------------------------------------------------------------------------------
# ------------------------------------------------------------------------------------------------
# GCN vertex-feature pooling (modules/network/gcn.py:84-164; SURVEY.md section 8f-4)
# ------------------------------------------------------------------------------------------------
def image_bounds(imgs: torch.Tensor, threshold: float = 0.03) -> torch.Tensor:
    """gcn.py:90-133 (get_bound_of_images) without the per-pixel Python loops.  mask = channel sum > 0.03; the scan sets
    the lower bound at the first occupied column/row whose index is NOT 0 (`bounds == 0` also means "unset", gcn.py:107,
    :119: an occupied column 0 leaves it unset and the next occupied column overwrites it) and the upper bound at the
    last occupied one; unset bounds stay 0 and w (h).  Normalised to [-1, 1] as x / w * 2 - 1."""
    assert imgs.ndimension() == 4
    b, _, h, w = imgs.shape
    out = torch.zeros(b, 4)
    for i in range(b):
        mask = imgs[i].sum(0) > threshold
        for k, (occ, size) in enumerate(((mask.any(0), w), (mask.any(1), h))):
            idx = torch.nonzero(occ).flatten()
            lo_c = idx[idx > 0]
            out[i, 2 * k] = float(lo_c[0]) if lo_c.numel() else 0.0
            out[i, 2 * k + 1] = float(idx[-1]) if idx.numel() else float(size)
    out[:, :2] = out[:, :2] / w * 2 - 1
    out[:, 2:4] = out[:, 2:4] / h * 2 - 1
    return out


def bilinear_sample(feat: torch.Tensor, gx: torch.Tensor, gy: torch.Tensor) -> torch.Tensor:
    """torch.nn.functional.grid_sample(feat (B,C,H,W), grid (B,1,N,2), mode='bilinear', padding_mode='zeros',
    align_corners=True) -> (B,C,N), restated: ix = (x+1)/2 (W-1); taps nw, ne, sw, se with weights
    (ix_se-ix)(iy_se-iy), (ix-ix_sw)(iy_sw-iy), (ix_ne-ix)(iy-iy_ne), (ix-ix_nw)(iy-iy_nw); out-of-range taps add 0."""
    b, c, h, w = feat.shape
    ix = ((gx + 1) / 2) * (w - 1)
    iy = ((gy + 1) / 2) * (h - 1)
    x0, y0 = torch.floor(ix), torch.floor(iy)
    x1, y1 = x0 + 1, y0 + 1
    out = torch.zeros(b, c, gx.shape[1], dtype=feat.dtype)
    flat = feat.reshape(b, c, h * w)
    for xx, yy, wgt in ((x0, y0, (x1 - ix) * (y1 - iy)), (x1, y0, (ix - x0) * (y1 - iy)),
                        (x0, y1, (x1 - ix) * (iy - y0)), (x1, y1, (ix - x0) * (iy - y0))):
        ok = (xx >= 0) & (xx <= w - 1) & (yy >= 0) & (yy <= h - 1)
        lin = (yy.clamp(0, h - 1) * w + xx.clamp(0, w - 1)).long()
        tap = torch.gather(flat, 2, lin[:, None, :].expand(b, c, -1))
        out = out + tap * (wgt * ok)[:, None, :]
    return out


def perceptual_feature_pooling(features: Sequence[torch.Tensor], points: torch.Tensor, bounds: torch.Tensor) -> torch.Tensor:
    """gcn.py:135-164.  grid x from z, grid y from y, both flipped and rescaled by the sample's own min / max into the
    image bounds; every feature map sampled bilinearly there; channels of all maps concatenated -> (B, N, sum C)."""
    assert points.ndimension() == 3 and bounds.ndimension() == 2
    mx, mn = points.max(1)[0], points.min(1)[0]                      # (B,3): differentiable through the arg-max / arg-min
    sz = (points[..., 2] - mn[:, None, 2]) / (mx[:, None, 2] - mn[:, None, 2])
    sy = (points[..., 1] - mn[:, None, 1]) / (mx[:, None, 1] - mn[:, None, 1])
    gx = bounds[:, None, 0] + (1 - sz) * (bounds[:, None, 1] - bounds[:, None, 0])
    gy = bounds[:, None, 2] + (1 - sy) * (bounds[:, None, 3] - bounds[:, None, 2])
    pooled = [bilinear_sample(f, gx, gy) for f in features]
    return torch.cat(pooled, 1).permute(0, 2, 1)


def synthetic_primitives(b: int, k: int, seed: int = 1234):
    """Network-output-shaped (v, q, t): vpnet_one_resnet.py:69-85 with IS_SIGMOID and
    VOLUME_RESTRICT = [8, 10, 10] (config.py:25-26)."""
    g = torch.Generator().manual_seed(seed)
    v = (torch.sigmoid(torch.randn(b, k, 3, generator=g)) + 0.1) / torch.tensor([8.0, 10.0, 10.0])
    q = torch.sigmoid(torch.randn(b, k, 4, generator=g))
    t = torch.tanh(torch.randn(b, k, 3, generator=g))
    return v, q, t
