"""One primitive-loss step: the per-iteration primitive assembly + loss of train.py:243-260, batched over all K
primitives and all B samples, every stage a vpn_b200 kernel.

    points   = sample + pose of K primitives            (train.py:105-120 -> one launch)
    view_cd  = Chamfer(points, view_center_points)       (train.py:152-163)
    obj_cd   = Chamfer(view_to_obj(points), canonical)   (only when L_CAN_CD != 0; the reference computes
                                                          it even when its weight is 0, train.py:160-161)
    vp_div   = Chamfer(centres, targets, w1=.5, w2=1)    (train.py:179-185, vp_diverse.py:12-18)
    sil      = L1/MSE(soft_silhouette(mesh), gt)         (train.py:123-149,166-176; silhouette.py:13-23)
    emd      = mean sqrt(auction dist)(points, targets)  (only when l_emd != 0; train.py:188-195, train_gcn.py:91-95)
"""
from __future__ import annotations

from dataclasses import dataclass
from typing import Dict, Optional

import torch

from . import ops, templates


@dataclass
class PrimitiveLossConfig:
    kind: str = "sphere"              # 'sphere' | 'cuboid'   (config.py:32-35 SPHERE_NUM / CUBOID_NUM)
    l_view_cd: float = 1.0            # config.py:14-17
    l_can_cd: float = 0.0
    l_sil: float = 0.0
    l_vp_div: float = 0.1
    cd_w1: float = 1.0                # config.py:12-13
    cd_w2: float = 1.0
    silhouette_loss: str = "L1"       # config.py:27
    img_size: int = 128               # config.py:46
    chamfer_impl: int = ops.CHAMFER_AUTO
    vertex_chamfer: bool = False      # train_gcn.py:127-130: the Chamfer term scores the composed mesh vertices, not samples
    soft_cull_backfaces: bool = False  # rasteriser soft pass: False = DIB-R (back faces culled by the coverage pass only)
    overlap_silhouette: bool = True   # run mesh -> silhouette -> image loss on a second stream, concurrently with the Chamfer terms
    # EMD term (train.py:188-195, train_gcn.py:91-95).  The reference's config.py:17 sets L_EMD = 1.0; the default here is
    # 0 so that every caller written before the term existed (bench.py's workloads among them) computes what it did.
    # Pass l_emd=1.0 for the reference's training loss.  It needs as many points as targets (P == M).
    l_emd: float = 0.0
    emd_eps: float = 0.005            # train.py:188-195
    emd_iters: int = 50


class _LossStep:
    """What the batched steps share: the view-centred silhouette cameras, the side streams their independent branches are
    forked onto, and the EMD term.  Subclasses have a `cfg` with l_emd / emd_eps / emd_iters and say whether they compute
    any other term (_has_other_terms)."""

    def default_cameras(self, b: int, device):
        """IS_VIEW_CENTER cameras: dist = 1, elev = azim = 0 for every sample (train.py:172-174); built once per batch size."""
        key = ("cam", b, str(device))
        cache = self.__dict__.setdefault("_cams", {})
        if key not in cache:
            cache[key] = ops.look_at_cameras(torch.zeros(b, device=device), torch.zeros(b, device=device),
                                             torch.ones(b, device=device))
        return cache[key]

    def _side_stream(self, device, name="side"):
        key = (name, str(device))
        cache = self.__dict__.setdefault("_streams", {})
        if key not in cache:
            cache[key] = torch.cuda.Stream(device=device)
        return cache[key]

    def _forked(self, device, name, fn, uses=()):
        """fn() -> tuple of tensors, run on side stream `name` after the work queued so far on the caller's stream.
        `uses`: tensors made by the step that the branch reads.  Returns (outputs, side stream); pass the stream to _join
        before the outputs are used on the caller's stream.  Autograd runs the branch's backward on the same side stream;
        under CUDA-graph capture the fork / join becomes two parallel branches of the graph."""
        cur = torch.cuda.current_stream(device)
        side = self._side_stream(device, name)
        side.wait_stream(cur)
        with torch.cuda.stream(side):
            for x in uses:
                x.record_stream(side)
            outs = fn()
            for o in outs:
                o.record_stream(cur)
        return outs, side

    @staticmethod
    def _join(device, side):
        if side is not None:
            torch.cuda.current_stream(device).wait_stream(side)

    def _has_other_terms(self) -> bool:
        raise NotImplementedError

    def _fork_emd(self, points) -> bool:
        """Run the EMD term on its own stream whenever another term can use the SMs the auction leaves free
        (tools/bench_step_emd.py overrides this to time both placements)."""
        return points.is_cuda and self._has_other_terms()

    def _emd_term(self, points, targets):
        """l_emd * mean over the batch of mean sqrt(dist) (train.py:188-195; train_gcn.py:91-95)."""
        cfg = self.cfg
        return ops.emd_distance(points, targets, eps=cfg.emd_eps, iters=cfg.emd_iters, weight=cfg.l_emd)

    def _emd_branch(self, points, targets):
        """(EMD term, its side stream or None).  The auction is one cluster launch that holds its SMs for milliseconds and
        shares nothing with the other terms but the points: forked, the other terms run on the SMs it leaves free.
        Measured faster than running it inline on every workload of tools/bench_step_emd.py (DESIGN.md section 4.6)."""
        if self._fork_emd(points):
            (term,), side = self._forked(points.device, "emd", lambda: (self._emd_term(points, targets),), uses=(points,))
            return term, side
        return self._emd_term(points, targets), None


def _image_loss(alpha, silhouettes, kind: str, weight: float):
    """weight * L1Loss | MSELoss of the soft alpha (B,H,W) against the ground truth (B,1,H,W) (silhouette.py:13-23)."""
    diff = alpha[:, None] - silhouettes
    sil = diff.abs().mean() if kind == "L1" else (diff * diff).mean()
    return sil * weight


def _capture(run, device, warmup: int):
    """Run `run` `warmup` times on a side stream (caches, function attributes, allocator), then capture one call into a
    CUDA graph.  Returns (graph, what the captured call returned, our kernel launches in one replay)."""
    from . import _lib
    side = torch.cuda.Stream(device=device)
    side.wait_stream(torch.cuda.current_stream(device))
    with torch.cuda.stream(side):
        for _ in range(warmup):
            run()
    torch.cuda.current_stream(device).wait_stream(side)
    torch.cuda.synchronize(device)
    lib = _lib.load()
    n0 = lib.vpn_launch_count()
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        outs = run()
    return graph, outs, int(lib.vpn_launch_count() - n0)


class PrimitiveLoss(_LossStep):
    def __init__(self, config: Optional[PrimitiveLossConfig] = None):
        self.cfg = config or PrimitiveLossConfig()
        assert self.cfg.kind in ("sphere", "cuboid")

    def composed_faces(self, k: int, device) -> torch.Tensor:
        """Faces of K composed template meshes (meshing.py:28-46 running vertex offset), int32 (K*F,3)."""
        key = (k, str(device))
        cache = self.__dict__.setdefault("_faces", {})
        if key not in cache:
            tv, tf = templates.template(self.cfg.kind, device)
            nv = tv.shape[0]
            cache[key] = torch.cat([tf + i * nv for i in range(k)], dim=0).contiguous()
        return cache[key]

    def __call__(self, v: torch.Tensor, q: torch.Tensor, t: torch.Tensor, uniforms: torch.Tensor,
                 view_center_points: torch.Tensor, silhouettes: Optional[torch.Tensor] = None,
                 canonical_points: Optional[torch.Tensor] = None, dists=None, elevs=None, azims=None,
                 angles=None, sil_cameras=None) -> Dict[str, torch.Tensor]:
        """dists / elevs / azims / angles (B,) are the view parameters of view_to_obj_points (train.py:152-163) and are
        used by the canonical-frame Chamfer ONLY.  The silhouette is always rendered from the view-centred camera
        dist = 1, elev = azim = 0, as the reference does under IS_VIEW_CENTER (train.py:166-176: the predicted meshes
        live in the view-centred frame), unless sil_cameras = (dists, elevs, azims) is passed explicitly."""
        cfg = self.cfg
        out: Dict[str, torch.Tensor] = {}
        b, k = q.shape[:2]
        if cfg.l_emd:
            # the auction pairs every point with one target (emd_module.py:37-38): checked from the shapes before any launch
            per_prim = templates.template(cfg.kind, v.device)[0].shape[0] if cfg.vertex_chamfer else uniforms.shape[2]
            assert view_center_points.dim() == 3 and tuple(view_center_points.shape) == (b, k * per_prim, 3), (
                f"l_emd needs as many points as targets: {k} x {per_prim} points, targets {tuple(view_center_points.shape)}")
        verts = None
        if cfg.vertex_chamfer:
            tv, _ = templates.template(cfg.kind, v.device)
            points = verts = ops.mesh_vertices(tv, v, q, t)
        else:
            points = ops.sample_primitives(cfg.kind, v, q, t, uniforms)
        out["points"] = points
        total = None

        def add(name, val):
            nonlocal total
            out[name] = val
            total = val if total is None else total + val

        # The silhouette branch (mesh vertices -> rasteriser -> image loss) shares nothing with the Chamfer terms but the
        # primitives: it is forked onto a second stream and joined before the sum.  The rasteriser is latency bound and
        # leaves most of every SM idle (one 131 KB Chamfer CTA + raster CTAs fit an SM together), so the two overlap almost
        # completely, forward and backward (autograd runs a node's backward on the stream of its forward).  Under CUDA-graph
        # capture the fork / join becomes two parallel branches of the graph.
        sil_term, side = None, None
        if cfg.l_sil:
            fork = cfg.overlap_silhouette and v.is_cuda and (cfg.l_view_cd or cfg.l_can_cd or cfg.l_vp_div)
            if sil_cameras is None:
                self.default_cameras(b, v.device)          # cached constants are created on the caller's stream, before the fork
            self.composed_faces(k, v.device)
            sil = lambda: self._silhouette_term(v, q, t, verts, silhouettes, sil_cameras)
            if fork:
                (sil_term, out["alpha"]), side = self._forked(v.device, "side", sil)
            else:
                sil_term, out["alpha"] = sil()
        emd_term, emd_side = None, None
        if cfg.l_emd:
            emd_term, emd_side = self._emd_branch(points, view_center_points)
        if cfg.l_view_cd:
            add("view_cd", ops.chamfer_distance(points, view_center_points, w1=cfg.cd_w1, w2=cfg.cd_w2,
                                                impl=cfg.chamfer_impl) * cfg.l_view_cd)
        if cfg.l_can_cd:
            can = ops.view_to_obj_points(points, dists, elevs, azims, angles)
            add("obj_cd", ops.chamfer_distance(can, canonical_points, w1=cfg.cd_w1, w2=cfg.cd_w2,
                                               impl=cfg.chamfer_impl) * cfg.l_can_cd)
        if cfg.l_vp_div:
            add("vp_div", ops.chamfer_distance(t.contiguous(), view_center_points, w1=0.5, w2=1.0,
                                               impl=cfg.chamfer_impl) * cfg.l_vp_div)
        if emd_term is not None:
            self._join(v.device, emd_side)
            add("emd", emd_term)
        if sil_term is not None:
            self._join(v.device, side)
            add("sil", sil_term)
        out["total"] = total
        return out

    def _has_other_terms(self) -> bool:
        cfg = self.cfg
        return bool(cfg.l_view_cd or cfg.l_can_cd or cfg.l_vp_div or cfg.l_sil)

    def _silhouette_term(self, v, q, t, verts, silhouettes, sil_cameras):
        """l_sil * L1|MSE(soft alpha, gt) and alpha (train.py:123-149,166-176; silhouette.py:13-23)."""
        cfg = self.cfg
        b, k = q.shape[:2]
        if verts is None:
            tv, _ = templates.template(cfg.kind, v.device)
            verts = ops.mesh_vertices(tv, v, q, t)
        faces = self.composed_faces(k, v.device)
        h, w = silhouettes.shape[-2:]
        if sil_cameras is None:
            rot, pos = self.default_cameras(b, v.device)
        else:
            sd, se, sa = sil_cameras
            rot, pos = ops.look_at_cameras(sa, se, sd)
        alpha, _, _ = ops.soft_silhouette(verts, faces, rot, pos, h, w, soft_cull_backfaces=cfg.soft_cull_backfaces)
        return _image_loss(alpha, silhouettes, cfg.silhouette_loss, cfg.l_sil), alpha


class GraphedPrimitiveLoss:
    """The same step - draw uniforms, forward, backward to (v, q, t) - captured once into a CUDA graph and replayed.

    The step is ~20 of our launches plus torch's bookkeeping kernels; at small batch sizes (BASELINE config 1: B = 1) and
    in the end-to-end loop, where a device-to-host read forces a synchronisation every step, the host's launch latency is
    what is being timed.  Replaying removes it.  Shapes are fixed at construction; inputs are copied into static buffers
    (device-to-device or pinned-host-to-device, stream ordered), results are read from static buffers.

        g = GraphedPrimitiveLoss(cfg, v, q, t, targets, silhouettes)      # example tensors give the shapes
        loss, gv, gq, gt = g(v, q, t, targets, silhouettes)               # static output buffers, overwritten by the next call
    """

    def __init__(self, config: PrimitiveLossConfig, v, q, t, targets, silhouettes=None, n_samples: int = 0, warmup: int = 3,
                 canonical_points=None, cameras=None, after_backward=None):
        """after_backward: optional callable queued on the step's stream after the backward pass and captured with it -
        e.g. GradientAllReduce.launch(inline=True) when the all-reduce is our own self-synchronising kernel, so that no
        host launch sits between the step's tail and the collective.  It also runs in each of the `warmup` eager steps
        (every rank makes the same number of calls)."""
        self.cfg = config
        self.step = PrimitiveLoss(config)
        dev = v.device
        self.v = v.detach().clone().requires_grad_()
        self.q = q.detach().clone().requires_grad_()
        self.t = t.detach().clone().requires_grad_()
        self.targets = targets.detach().clone()
        self.sil = None if silhouettes is None else silhouettes.detach().clone()
        # canonical-frame Chamfer of train.py:152-163: targets in the object frame + (dists, elevs, azims, angles)
        self.canonical = None if canonical_points is None else canonical_points.detach().clone()
        self.cameras = None if cameras is None else tuple(c.detach().clone() for c in cameras)
        b, k = q.shape[:2]
        self.ushape = None if config.vertex_chamfer else (b, k, n_samples, 2 if config.kind == "sphere" else 3)
        assert config.vertex_chamfer or n_samples > 0, "n_samples (points per primitive) is required unless vertex_chamfer"

        def run():
            u = None if self.ushape is None else torch.rand(self.ushape, device=dev)      # drawn on the device, as the reference does
            cams = self.cameras or (None, None, None, None)
            out = self.step(self.v, self.q, self.t, u, self.targets, silhouettes=self.sil, canonical_points=self.canonical,
                            dists=cams[0], elevs=cams[1], azims=cams[2], angles=cams[3])
            gv, gq, gt = torch.autograd.grad(out["total"], (self.v, self.q, self.t))
            if after_backward is not None:
                after_backward()
            return out["total"], gv, gq, gt

        self.graph, (self.loss, self.gv, self.gq, self.gt), self.launches_per_step = _capture(run, dev, warmup)

    def __call__(self, v, q, t, targets, silhouettes=None, canonical_points=None, cameras=None):
        if self.canonical is not None and canonical_points is not None:
            self.canonical.copy_(canonical_points, non_blocking=True)
        if self.cameras is not None and cameras is not None:
            for dst, src in zip(self.cameras, cameras):
                dst.copy_(src, non_blocking=True)
        self.v.data.copy_(v, non_blocking=True)
        self.q.data.copy_(q, non_blocking=True)
        self.t.data.copy_(t, non_blocking=True)
        self.targets.copy_(targets, non_blocking=True)
        if self.sil is not None and silhouettes is not None:
            self.sil.copy_(silhouettes, non_blocking=True)
        self.graph.replay()
        return self.loss, self.gv, self.gq, self.gt


@dataclass
class MeshLossConfig:
    """Loss of the two loops whose free variable is a mesh's vertex tensor (one topology for the whole batch):
    train_sphere.py (n_samples > 0: area-weighted surface samples of the deformed sphere, train_sphere.py:71-80) and
    train_gcn.py (n_samples = 0: the predicted vertices themselves)."""
    n_samples: int = 2048             # train_sphere.py: SAMPLE_NUM * VP_NUM = 128 * 16 per mesh; 0 = score the vertices
    l_cd: float = 1.0                 # config.py:14 (L_VIEW_CD)
    cd_w1: float = 1.0                # config.py:12-13
    cd_w2: float = 1.0
    l_sil: float = 0.0                # config.py:16; silhouette of the mesh from the view-centred camera (train_sphere.py:125-128)
    silhouette_loss: str = "L1"       # config.py:27
    # EMD term: off by default for the reason given at PrimitiveLossConfig.l_emd; train_gcn.py adds it with weight 1.
    # It needs as many points (n_samples, or V) as targets.
    l_emd: float = 0.0
    emd_eps: float = 0.005
    emd_iters: int = 50
    chamfer_impl: int = ops.CHAMFER_AUTO
    soft_cull_backfaces: bool = False


class MeshLoss(_LossStep):
    """One loss step on a batch of meshes, every stage a vpn_b200 kernel; the gradient goes to `verts`.

        points = verts                                      (n_samples == 0: train_gcn.py)
               | area-weighted samples of the surface       (n_samples > 0: train_sphere.py, TriangleMesh.sample)
        cd     = Chamfer(points, targets, cd_w1, cd_w2)
        sil    = L1/MSE(soft_silhouette(verts, faces), gt)  (only when l_sil != 0; own stream when cd is on)
        emd    = mean sqrt(auction dist)(points, targets)   (only when l_emd != 0; own stream when another term is on)

    train_sphere.py passes verts = template + offsets (the offsets' gradient is the vertices'); train_gcn.py passes the
    network's vertices.  The branches are placed on streams as in PrimitiveLoss."""

    def __init__(self, config: Optional[MeshLossConfig] = None):
        self.cfg = config or MeshLossConfig()
        assert self.cfg.n_samples >= 0

    def _has_other_terms(self) -> bool:
        return bool(self.cfg.l_cd or self.cfg.l_sil)

    def __call__(self, verts: torch.Tensor, faces: torch.Tensor, targets: torch.Tensor, uniforms: Optional[torch.Tensor] = None,
                 silhouettes: Optional[torch.Tensor] = None) -> Dict[str, torch.Tensor]:
        """verts (B,V,3), faces (F,3) int32, targets (B,M,3); uniforms (B,n_samples,3) in [0,1) = [face draw, u1, u2],
        drawn on the device when None; silhouettes (B,1,H,W) when l_sil != 0.  Every check below reads shapes only, so
        a failing call raises AssertionError before any launch (and the checks are safe under graph capture)."""
        cfg = self.cfg
        n = cfg.n_samples
        assert verts.dim() == 3 and verts.size(-1) == 3, "verts must be (B, V, 3)"
        assert faces.dim() == 2 and faces.size(-1) == 3, "faces must be (F, 3)"
        b, nv = verts.shape[:2]
        assert n > 0 or uniforms is None, "n_samples = 0 scores the vertices: uniforms have nothing to draw"
        assert uniforms is None or tuple(uniforms.shape) == (b, n, 3), (
            f"uniforms must be (B, n_samples, 3) = {(b, n, 3)}, got {tuple(uniforms.shape)}")
        if cfg.l_emd:
            # the auction pairs every point with one target (emd_module.py:37-38)
            assert targets.dim() == 3 and tuple(targets.shape) == (b, n or nv, 3), (
                f"l_emd needs as many points as targets: {n or nv} points per mesh, targets {tuple(targets.shape)}")
        assert not cfg.l_sil or silhouettes is not None, "l_sil needs the ground-truth silhouettes"
        ops._check_face_indices(faces, nv)
        out: Dict[str, torch.Tensor] = {}
        if n:
            if uniforms is None:
                uniforms = torch.rand((b, n, 3), device=verts.device)       # drawn on the device, as TriangleMesh.sample_batch does
            points = ops.sample_mesh_surface(verts, faces, uniforms)[0]
        else:
            points = verts
        out["points"] = points
        total = None

        def add(name, val):
            nonlocal total
            out[name] = val
            total = val if total is None else total + val

        sil_term, side = None, None
        if cfg.l_sil:
            self.default_cameras(b, verts.device)            # cached constants are created on the caller's stream, before the fork
            sil = lambda: self._silhouette_term(verts, faces, silhouettes)
            if verts.is_cuda and cfg.l_cd:
                (sil_term, out["alpha"]), side = self._forked(verts.device, "side", sil)
            else:
                sil_term, out["alpha"] = sil()
        emd_term, emd_side = None, None
        if cfg.l_emd:
            emd_term, emd_side = self._emd_branch(points, targets)
        if cfg.l_cd:
            add("cd", ops.chamfer_distance(points, targets, w1=cfg.cd_w1, w2=cfg.cd_w2, impl=cfg.chamfer_impl) * cfg.l_cd)
        if emd_term is not None:
            self._join(verts.device, emd_side)
            add("emd", emd_term)
        if sil_term is not None:
            self._join(verts.device, side)
            add("sil", sil_term)
        out["total"] = total
        return out

    def _silhouette_term(self, verts, faces, silhouettes):
        cfg = self.cfg
        rot, pos = self.default_cameras(verts.size(0), verts.device)
        h, w = silhouettes.shape[-2:]
        alpha, _, _ = ops.soft_silhouette(verts, faces, rot, pos, h, w, soft_cull_backfaces=cfg.soft_cull_backfaces)
        return _image_loss(alpha, silhouettes, cfg.silhouette_loss, cfg.l_sil), alpha


class GraphedMeshLoss:
    """MeshLoss - draw the uniforms, forward, backward to the vertices - captured once into a CUDA graph and replayed,
    as GraphedPrimitiveLoss does for the primitive step.  The topology is fixed at construction; vertices, targets and
    silhouettes are copied into static buffers, results are read from static buffers.

        g = GraphedMeshLoss(cfg, verts, faces, targets, silhouettes)   # example tensors give the shapes
        loss, grad_verts = g(verts, targets, silhouettes)             # overwritten by the next call
        offsets.backward(grad_verts)                                  # train_sphere.py: verts = template + offsets
    """

    def __init__(self, config: MeshLossConfig, verts, faces, targets, silhouettes=None, warmup: int = 3):
        self.cfg = config
        self.step = MeshLoss(config)
        dev = verts.device
        self.verts = verts.detach().clone().requires_grad_()
        self.faces = faces.detach().clone()
        self.targets = targets.detach().clone()
        self.sil = None if silhouettes is None else silhouettes.detach().clone()

        def run():
            out = self.step(self.verts, self.faces, self.targets, silhouettes=self.sil)
            (gv,) = torch.autograd.grad(out["total"], (self.verts,))
            return out["total"], gv

        # the sampler's backward reads the cached vertex CSR of these faces: build it before the capture and keep it
        # alive as long as the graph
        self._adjacency = ops.mesh_adjacency(self.faces, verts.size(1)) if config.n_samples and verts.is_cuda else None
        self.graph, (self.loss, self.gv), self.launches_per_step = _capture(run, dev, warmup)

    def __call__(self, verts, targets, silhouettes=None):
        self.verts.data.copy_(verts, non_blocking=True)
        self.targets.copy_(targets, non_blocking=True)
        if self.sil is not None and silhouettes is not None:
            self.sil.copy_(silhouettes, non_blocking=True)
        self.graph.replay()
        return self.loss, self.gv


class HostPipeline:
    """Feeds a step with batches that live in (pinned) HOST memory and hands the results back in host memory, with the
    transfers overlapped with the computation - what a training loop with a pinned-memory loader does.

        pipe = HostPipeline(step, example_batch, device)       # step(device_batch: dict) -> tuple of device tensors
        pipe.submit(batch0)
        for batch in batches[1:]:
            pipe.submit(batch)            # host -> device copy of THIS batch runs while the previous step computes
            outs = pipe.result()          # results of the PREVIOUS batch (pinned host tensors, valid until two submits later)
        outs = pipe.result()

    Every batch is copied host -> device and every result device -> host, once per step; nothing is cached.  Two staging
    slots on the device: the copy stream fills slot i % 2 while the compute stream works on the other; the step for a
    batch is queued as soon as it is submitted (behind the previous one), so the device never waits for the host between
    steps, and the host synchronises once per step, on the oldest outstanding result.  `pre_step` (optional) is queued
    on the compute stream before every step (the bench's L2 flush).  On a CPU device everything runs synchronously (the
    ordering logic is the same; used by the tests)."""

    def __init__(self, step, example_batch: Dict[str, Optional[torch.Tensor]], device, pre_step=None):
        self.step, self.pre_step = step, pre_step
        self.device = torch.device(device)
        self.cuda = self.device.type == "cuda"
        self.staging = [{k: (None if v is None else torch.empty(v.shape, dtype=v.dtype, device=self.device))
                         for k, v in example_batch.items()} for _ in range(2)]
        self.host_out: list = [None, None]
        self.submitted = 0
        self.returned = 0
        if self.cuda:
            self.copy_stream = torch.cuda.Stream(device=self.device)
            self.staged = [torch.cuda.Event(), torch.cuda.Event()]
            self.free = [torch.cuda.Event(), torch.cuda.Event()]
            self.done = [torch.cuda.Event(), torch.cuda.Event()]
            self.pre_done = None                                     # end of the most recent submit's pre_step
            cur = torch.cuda.current_stream(self.device)
            for e in self.free:
                e.record(cur)

    def submit(self, batch: Dict[str, Optional[torch.Tensor]]) -> None:
        assert self.submitted - self.returned < 2, "two batches are already in flight: call result() first"
        slot = self.submitted % 2
        st = self.staging[slot]
        if self.cuda:
            cur = torch.cuda.current_stream(self.device)
            with torch.cuda.stream(self.copy_stream):
                self.copy_stream.wait_event(self.free[slot])          # the step that last read this slot has finished
                if self.pre_done is not None:
                    # start after the running step's pre_step: a host-to-device copy that overlaps the bench's 256 MB
                    # flush kernel slowed the loop by 0.14 ms per step (measured, tools/e2e_probe.py)
                    self.copy_stream.wait_event(self.pre_done)
                for k, v in batch.items():
                    if v is not None:
                        st[k].copy_(v, non_blocking=True)
                self.staged[slot].record(self.copy_stream)
            cur.wait_event(self.staged[slot])
        else:
            for k, v in batch.items():
                if v is not None:
                    st[k].copy_(v)
        if self.pre_step is not None:
            self.pre_step()
            if self.cuda:
                self.pre_done = torch.cuda.Event()
                self.pre_done.record(cur)
        outs = self.step(st)
        if self.cuda:
            self.free[slot].record(cur)
        if self.host_out[slot] is None:
            self.host_out[slot] = [torch.empty(o.shape, dtype=o.dtype, pin_memory=self.cuda) for o in outs]
        for h, o in zip(self.host_out[slot], outs):
            h.copy_(o.detach(), non_blocking=True)
        if self.cuda:
            self.done[slot].record(cur)
        self.submitted += 1

    def result(self):
        assert self.returned < self.submitted, "nothing in flight"
        slot = self.returned % 2
        if self.cuda:
            self.done[slot].synchronize()
        self.returned += 1
        return self.host_out[slot]
