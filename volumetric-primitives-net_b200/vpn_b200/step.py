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


class PrimitiveLoss:
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

    def default_cameras(self, b: int, device):
        """IS_VIEW_CENTER cameras: dist = 1, elev = azim = 0 for every sample (train.py:172-174); built once per batch size."""
        key = ("cam", b, str(device))
        cache = self.__dict__.setdefault("_cams", {})
        if key not in cache:
            cache[key] = ops.look_at_cameras(torch.zeros(b, device=device), torch.zeros(b, device=device),
                                             torch.ones(b, device=device))
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
            if fork:
                cur = torch.cuda.current_stream(v.device)
                side = self._side_stream(v.device)
                side.wait_stream(cur)
                with torch.cuda.stream(side):
                    sil_term, out["alpha"] = self._silhouette_term(v, q, t, verts, silhouettes, sil_cameras)
                    sil_term.record_stream(cur); out["alpha"].record_stream(cur)
            else:
                sil_term, out["alpha"] = self._silhouette_term(v, q, t, verts, silhouettes, sil_cameras)
        # The EMD auction is one cluster launch that holds its SMs for milliseconds and shares nothing with the Chamfer
        # terms but the points: forked like the silhouette branch, the other terms run on the SMs it leaves free.  Measured
        # faster than running it inline on every workload of tools/bench_step_emd.py (DESIGN.md section 4.6).
        emd_term, emd_side = None, None
        if cfg.l_emd:
            if self._fork_emd(points):
                cur = torch.cuda.current_stream(v.device)
                emd_side = self._side_stream(v.device, "emd")
                emd_side.wait_stream(cur)
                with torch.cuda.stream(emd_side):
                    points.record_stream(emd_side)
                    emd_term = self._emd_term(points, view_center_points)
                    emd_term.record_stream(cur)
            else:
                emd_term = self._emd_term(points, view_center_points)
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
            if emd_side is not None:
                torch.cuda.current_stream(v.device).wait_stream(emd_side)
            add("emd", emd_term)
        if sil_term is not None:
            if side is not None:
                torch.cuda.current_stream(v.device).wait_stream(side)
            add("sil", sil_term)
        out["total"] = total
        return out

    def _side_stream(self, device, name="side"):
        key = (name, str(device))
        cache = self.__dict__.setdefault("_streams", {})
        if key not in cache:
            cache[key] = torch.cuda.Stream(device=device)
        return cache[key]

    def _fork_emd(self, points) -> bool:
        """Run the EMD term on its own stream whenever another term can use the SMs the auction leaves free
        (tools/bench_step_emd.py overrides this to time both placements)."""
        cfg = self.cfg
        return points.is_cuda and bool(cfg.l_view_cd or cfg.l_can_cd or cfg.l_vp_div or cfg.l_sil)

    def _emd_term(self, points, targets):
        """l_emd * mean over the batch of mean sqrt(dist) (train.py:188-195; train_gcn.py:91-95)."""
        cfg = self.cfg
        return ops.emd_distance(points, targets, eps=cfg.emd_eps, iters=cfg.emd_iters, weight=cfg.l_emd)

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
        diff = alpha[:, None] - silhouettes
        sil = diff.abs().mean() if cfg.silhouette_loss == "L1" else (diff * diff).mean()
        return sil * cfg.l_sil, alpha


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
        from . import _lib
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

        side = torch.cuda.Stream(device=dev)
        side.wait_stream(torch.cuda.current_stream(dev))
        with torch.cuda.stream(side):                      # warm-up off the capture: caches, function attributes, allocator
            for _ in range(warmup):
                run()
        torch.cuda.current_stream(dev).wait_stream(side)
        torch.cuda.synchronize(dev)
        lib = _lib.load()
        n0 = lib.vpn_launch_count()
        self.graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(self.graph):
            self.loss, self.gv, self.gq, self.gt = run()
        self.launches_per_step = int(lib.vpn_launch_count() - n0)      # our kernels inside one replay

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
