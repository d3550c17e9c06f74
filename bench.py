#!/usr/bin/env python
"""Headline benchmark: primitive-loss forward+backward samples/s (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload c2|c3|c1] [--dump-outputs DIR]

A step = one pass of the hot path over one synthetic batch: draw uniforms -> fused sample+pose of K
primitives -> Chamfer NN (both directions) vs the targets (+ VP-diverse Chamfer, + mesh vertices ->
soft silhouette -> L1 when the workload has a render term) -> backward to (v, q, t).
Default workload = BASELINE.json configs[1] ("c2": B=32/GPU, 16 cuboids x 4096 samples, 8192 targets).
Multi-GPU: one process per GPU under torchrun, batch sharded (weak scaling, 32 samples per GPU), plus one
NCCL all-reduce of a VPNetOneRes-sized gradient buffer (22 875 848 fp32) per step.
Prints ONE JSON line on rank 0.
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import threading
import time

REPO = os.path.dirname(os.path.abspath(__file__))
PKG = os.path.join(REPO, "volumetric-primitives-net_b200")
for p in (REPO, PKG):
    if p not in sys.path:
        sys.path.insert(0, p)

import torch  # noqa: E402

WORKLOADS = {
    # name: (kind, B per GPU, K, N, M, render resolution or 0)          BASELINE.json configs[0..4]
    "c1": ("sphere", 1, 16, 1024, 2048, 64),
    "c2": ("cuboid", 32, 16, 4096, 8192, 0),
    "c3": ("cuboid", 32, 32, 4096, 8192, 128),
    "c4": ("cuboid", 256, 32, 4096, 8192, 128),       # B = 256 in TOTAL, split over the ranks (strong scaling)
    "c5": ("sphere", 8, 128, 128, 16384, 256),        # train_gcn.py shape: the K*128 mesh vertices are the predicted points
    # c2 as train.py:152-163 runs it: BOTH big Chamfers (view frame + canonical frame through view_to_obj_points; the
    # reference computes the second even at its default weight L_CAN_CD = 0) + VP-diverse
    "c2f": ("cuboid", 32, 16, 4096, 8192, 0),
}
STRONG = {"c4"}            # workloads whose B is the global batch
VERTEX_MODE = {"c5"}       # Chamfer on the composed mesh vertices (train_gcn.py:127-130) instead of surface samples
FAITHFUL = {"c2f"}         # canonical-frame Chamfer included (l_can_cd = 1 so that it is computed AND differentiated)


def per_gpu_batch(workload, world):
    b = WORKLOADS[workload][1]
    return max(1, b // world) if workload in STRONG else b

GRAD_NUMEL = 22_875_848          # VPNetOneRes parameters at K = 16 (SURVEY.md section 8c)
METRIC = "primitive-loss fwd+bwd samples/sec"


def synthetic(workload, device, seed=1234, sets=1, batch=None):
    """Network-output-shaped primitives + ShapeNet-shaped targets (SURVEY.md section 8d), fp32."""
    kind, b, k, n, m, res = WORKLOADS[workload]
    b = batch or b
    g = torch.Generator().manual_seed(seed)
    out = []
    for _ in range(sets):
        v = (torch.sigmoid(torch.randn(b, k, 3, generator=g)) + 0.1) / torch.tensor([8.0, 10.0, 10.0])
        q = torch.sigmoid(torch.randn(b, k, 4, generator=g))
        t = torch.tanh(torch.randn(b, k, 3, generator=g)) * 0.4
        # targets: points on the surface of a random union of boxes inside [-0.5, 0.5]^3
        centre = (torch.rand(b, 8, 3, generator=g) - 0.5) * 0.7
        half = torch.rand(b, 8, 3, generator=g) * 0.12 + 0.03
        which = torch.randint(0, 8, (b, m), generator=g)
        p = (torch.rand(b, m, 3, generator=g) * 2 - 1)
        axis = torch.randint(0, 3, (b, m), generator=g)
        sign = torch.randint(0, 2, (b, m), generator=g).float() * 2 - 1
        p.scatter_(2, axis[..., None], sign[..., None])
        bi = torch.arange(b)[:, None]
        tgt = centre[bi, which] + p * half[bi, which]
        sil = (torch.rand(b, 1, res, res, generator=g) > 0.5).float() if res else None
        d = dict(v=v, q=q, t=t, target=tgt.contiguous(), sil=sil)
        if workload in FAITHFUL:
            # object-frame copy of the targets + the view parameters that map one frame to the other (dataset.py ranges)
            d["dists"] = 1.0 + 0.5 * torch.rand(b, generator=g)
            d["elevs"] = 20.0 + 20.0 * torch.rand(b, generator=g)
            d["azims"] = 360.0 * torch.rand(b, generator=g)
            d["angles"] = 360.0 * torch.rand(b, generator=g)
            d["canon"] = (tgt * d["dists"][:, None, None]).contiguous()
        out.append(d)
    return out


class ClockSampler(threading.Thread):
    """nvidia-smi-equivalent clock / throttle sampling (NVML) during the timed region, on rank 0 only; arm() starts it.
    In a multi-rank job, sampling a GPU makes that rank reach the following all-reduces late and every other rank waits
    for it; a single process on one GPU shows no cost at all (profiles/r02_nvml_cost_probe_1gpu.txt).  Measured, ms per
    C2 step (2.94 without any sampling on 2 or 8 GPUs with the NVLS all-reduce; single runs, different boxes):
      all ranks, every 10 ms, from before the loop   8 GPUs 3.22 - 3.72     (2 GPUs, NCCL: 2.87 vs 2.86 unsampled)
      rank 0,    every 20 ms, from before the loop   8 GPUs 3.16, 3.16      <- what bench.py does
      rank 0,    every 20 ms, once the steps are enqueued      8 GPUs 3.45; 2 GPUs 3.15
      rank 0,    every 200 ms, once enqueued (one sample)      2 GPUs 3.17; with NVML warmed up first 3.34 / 4.13
    (profiles/r01w_scale_8gpu.txt, r01y_*, r02_scale_2gpu_sampling_variants.txt).  The delay does not scale with the
    number of samples and its mechanism is not understood; VPN_BENCH_NO_CLOCKS=1 switches the sampling off."""

    def __init__(self, index, enabled=True, period_s=0.03):
        super().__init__(daemon=True)
        self.index, self.samples, self.reasons, self.stop_flag, self.max_mhz = index, [], set(), False, None
        self.period_s, self.nv = period_s, None
        self.armed, self.ready = threading.Event(), threading.Event()
        if not enabled:
            return
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self.nv = None

    def run(self):
        if self.nv is None:
            self.ready.set()
            return
        nv = self.nv
        names = {nv.nvmlClocksThrottleReasonHwSlowdown: "hw_slowdown",
                 nv.nvmlClocksThrottleReasonHwThermalSlowdown: "hw_thermal_slowdown",
                 nv.nvmlClocksThrottleReasonSwThermalSlowdown: "sw_thermal_slowdown",
                 nv.nvmlClocksThrottleReasonSwPowerCap: "sw_power_cap"}
        self.ready.set()
        self.armed.wait()
        while True:                                  # at least one sample, taken right after arm()
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for bit, name in names.items():
                    if r & bit:
                        self.reasons.add(name)
            except Exception:
                pass
            if self.stop_flag:
                break
            time.sleep(self.period_s)

    def arm(self):
        self.armed.set()

    def stop(self):
        self.stop_flag = True
        self.armed.set()

    def summary(self):
        s = sorted(self.samples)
        return {"sm_mhz": (s[len(s) // 2] if s else None), "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons),
                "samples": len(s)}


def cpu_reference_step(workload, rows_per_sample, threads, rows_per_slice=8192):
    """The reference's own formulation on the host (oracle port, op for op: dense (B,P,M,3) broadcast,
    modules/loss/chamfer_distance.py:14-23), fwd + bwd to (v,q,t), on a bounded sample of the workload:
    one sample, `rows_per_sample` of its K*N predicted points, taken as slices of whole primitives (the dense
    temporaries of one slice are ~1 GB each; a whole C2 sample at once needs 15 GB)."""
    from oracle import vpn_oracle as O
    kind, b, k, n, m, res = WORKLOADS[workload]
    per = max(1, rows_per_slice // n)                    # primitives per slice
    kk = min(k, max(per, (rows_per_sample // n) // per * per))
    torch.set_num_threads(threads)
    data = synthetic(workload, "cpu")[0]
    tgt = data["target"][:1]
    g = torch.Generator().manual_seed(1)
    dt = 0.0
    for k0 in range(0, kk, per):
        v, q, t = (data[x][:1, k0:k0 + per].clone().requires_grad_() for x in ("v", "q", "t"))
        u = torch.rand(1, v.shape[1], n, 2 if kind == "sphere" else 3, generator=g)
        t0 = time.perf_counter()
        pts = O.sample_predict_points(kind, v, q, t, u)
        loss = O.chamfer_dense(pts, tgt) + 0.1 * O.chamfer_dense(t, tgt, w1=0.5, w2=1.0)
        loss.backward()
        dt += time.perf_counter() - t0
    frac = (kk * n) / float(k * n)          # share of one sample's pair work that was timed
    return dt, frac, kk * n


CPU_SAMPLE_ROWS = 32768      # ONE method for both CPU legs (cpu_baseline of our arm and --impl reference): one sample, this many
                             # of its predicted points (whole primitives), scaled linearly to a full sample


def cpu_sample_rows(workload):
    kind, b, k, n, m, res = WORKLOADS[workload]
    return min(k * n, CPU_SAMPLE_ROWS)


def cpu_sample_text(workload, used, dt=None):
    kind, b, k, n, m, res = WORKLOADS[workload]
    t = f", {dt:.1f} s" if dt is not None else ""
    return (f"1 sample, {used} of {k * n} predicted points x {m} targets per step (dense torch-CPU formulation of the "
            f"reference, fwd+bwd, no render term){t}, scaled linearly to a full sample")


def run_reference(args):
    """`--impl reference`: the reference's CPU path (oracle port) on this box's host cores."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    threads = os.cpu_count() or 1
    kind, b, k, n, m, res = WORKLOADS[args.workload]
    rows = cpu_sample_rows(args.workload)
    for _ in range(args.warmup):
        cpu_reference_step(args.workload, min(rows, 8192), threads)
    times = []
    for _ in range(args.steps):
        dt, frac, used = cpu_reference_step(args.workload, rows, threads)
        times.append(dt)
    mean = sum(times) / len(times)
    per_sample = mean / frac
    value = 1.0 / per_sample
    sample = cpu_sample_text(args.workload, used)
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": "samples/s", "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": mean * 1e3, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": describe(args.workload)},
            "cpu_baseline": {"value": value, "unit": "samples/s", "cores": threads, "kind": "port", "sample": sample},
            "e2e": {"value": value, "unit": "samples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)


def describe(workload, world=1):
    kind, b, k, n, m, res = WORKLOADS[workload]
    b = per_gpu_batch(workload, world)
    what = "template vertices" if workload in VERTEX_MODE else "samples"
    s = f"{workload}: B={b}/GPU, {k} {kind} primitives x {n} {what} (P={k * n}), Chamfer vs M={m} targets + VP-diverse"
    if workload in FAITHFUL:
        s += " + canonical-frame Chamfer through view_to_obj_points (train.py:152-163)"
    if res:
        s += f" + {res}x{res} soft-silhouette L1"
    return s + ", fwd+bwd to (v,q,t)"


class Bench:
    """Shared state of one bench.py process: device, process group, flush buffer, gradient all-reduce."""

    def __init__(self, args):
        import vpn_b200
        from vpn_b200 import _lib, dist as vdist
        import torch.distributed as dist
        self.vpn, self.dist, self.args = vpn_b200, dist, args
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        self.rank = int(os.environ.get("RANK", "0"))
        self.local = int(os.environ.get("LOCAL_RANK", "0"))
        assert torch.cuda.is_available(), "bench.py needs a CUDA device (no CPU fallback)"
        torch.cuda.set_device(self.local)
        self.dev = torch.device("cuda", self.local)
        if self.world > 1:
            dist.init_process_group("nccl", device_id=self.dev)
        self.lib = _lib.load()
        self.flush = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device=self.dev)      # > 126 MB L2
        self.sync = vdist.GradientAllReduce(GRAD_NUMEL, self.dev) if self.world > 1 else None
        self.do_flush = os.environ.get("VPN_BENCH_FLUSH", "1") != "0"
        self.clocks_on = os.environ.get("VPN_BENCH_NO_CLOCKS", "0") != "1"

    def barrier(self):
        torch.cuda.synchronize()
        if self.world > 1:
            self.dist.barrier()
            torch.cuda.synchronize()

    def new_sampler(self):
        """NVML clock sampler thread for rank 0, fully initialised (nvmlInit, handle, first query) BEFORE the barrier that
        starts a timed region: its set-up cost on rank 0 used to make rank 0 enter the timed loop milliseconds after the
        other ranks, which then waited for it in their first all-reduce (the 'inter-rank skew' of round 1)."""
        s = ClockSampler(self.local, enabled=(self.rank == 0 and self.clocks_on), period_s=0.02)
        s.start()
        s.ready.wait(timeout=10.0)
        return s


def measure_workload(B, workload, steps, warmup, chamfer_impl=0, graph="auto", with_rooflines=True, cpu_baseline=False,
                     keep_outputs=False):
    """value (device-resident inputs), e2e (pinned host inputs, copies inside the timed region) and, on rank 0, the
    rooflines of one workload.  Both timed regions run under the same conditions: 256 MB L2 flush before every step,
    NVML clock sampling on rank 0, gradient all-reduce (N > 1) inside the step.  Returns a dict (rank 0) or None.
    keep_outputs: the result also holds, as numpy arrays under "outputs", what the last timed step returned."""
    vpn, dist, dev, world, rank, lib = B.vpn, B.dist, B.dev, B.world, B.rank, B.lib
    kind, b, k, n, m, res = WORKLOADS[workload]
    b = per_gpu_batch(workload, world)
    vertex_mode = workload in VERTEX_MODE
    faithful = workload in FAITHFUL
    width = 2 if kind == "sphere" else 3
    nsets = 4
    torch.manual_seed(1234 + rank)            # the step's uniforms are drawn on the device: the same draws in every run
    host = synthetic(workload, "cpu", seed=1234 + rank, sets=nsets, batch=b)
    devsets = [{kk: (vv.to(dev) if vv is not None else None) for kk, vv in s.items()} for s in host]
    pinned = [{kk: (vv.pin_memory() if vv is not None else None) for kk, vv in s.items()} for s in host]
    cfg = vpn.PrimitiveLossConfig(kind=kind, l_sil=(1.0 if res else 0.0), chamfer_impl=chamfer_impl,
                                  vertex_chamfer=vertex_mode, l_can_cd=(1.0 if faithful else 0.0),
                                  overlap_silhouette=os.environ.get("VPN_BENCH_NO_SIL_OVERLAP", "0") != "1")

    def cams_of(s):
        return (s["dists"], s["elevs"], s["azims"], s["angles"]) if faithful else None
    step_fn = vpn.PrimitiveLoss(cfg)
    sync, flush = B.sync, B.flush
    # the bench joins the all-reduce right after launching it (nothing of this path can overlap it), so it is queued on the
    # step's own stream; when it is our self-synchronising NVLS kernel it is captured INSIDE the step's CUDA graph
    ar_inline = os.environ.get("VPN_BENCH_AR_STREAM", "inline") != "side"
    ar_in_graph = (sync is not None and ar_inline and sync.graph_capturable and os.environ.get("VPN_BENCH_AR_IN_GRAPH", "1") != "0")
    graphed, graph_error = None, None
    if graph != "off":
        try:
            d0 = devsets[0]
            graphed = vpn.GraphedPrimitiveLoss(cfg, d0["v"], d0["q"], d0["t"], d0["target"], d0["sil"], n_samples=n,
                                               canonical_points=d0.get("canon"), cameras=cams_of(d0),
                                               after_backward=(lambda: sync.launch(inline=True)) if ar_in_graph else None)
        except Exception as e:                               # noqa: BLE001 - eager launches are always available
            graph_error = repr(e)[:200]
            ar_in_graph = False
            if graph == "on":
                raise
    if world > 1:                                            # every rank must take the same path (graph or eager)
        flag = torch.tensor([1 if graphed is not None else 0], dtype=torch.int32, device=dev)
        dist.all_reduce(flag, op=dist.ReduceOp.MIN)
        if int(flag.item()) == 0 and graphed is not None:
            raise RuntimeError("CUDA-graph capture succeeded on this rank but failed on another")

    def one_step(s):
        if graphed is not None:
            out = graphed(s["v"], s["q"], s["t"], s["target"], s["sil"], canonical_points=s.get("canon"), cameras=cams_of(s))
            if sync is not None and not ar_in_graph:
                sync.launch(inline=ar_inline)
            return out
        v, q, t = (s[x].detach().requires_grad_() for x in ("v", "q", "t"))
        u = None if vertex_mode else torch.rand((b, k, n, width), device=dev)      # drawn on device, like the reference
        c4 = cams_of(s) or (None, None, None, None)
        out = step_fn(v, q, t, u, s["target"], silhouettes=s["sil"], canonical_points=s.get("canon"),
                      dists=c4[0], elevs=c4[1], azims=c4[2], angles=c4[3])
        out["total"].backward()
        if sync is not None:
            sync.launch(inline=ar_inline)
        return out["total"], v.grad, q.grad, t.grad

    # ---- device-resident throughput ("value") ---------------------------------------------------
    for i in range(warmup):
        one_step(devsets[i % nsets])
    if sync is not None:
        sync.join()
    evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
    mids = [torch.cuda.Event(enable_timing=True) for _ in range(steps)]      # end of the rank's own compute, before the join
    sampler = B.new_sampler()
    launches0 = lib.vpn_launch_count()
    B.barrier()                                   # barrier + synchronize immediately before the timed steps, on every rank
    sampler.arm()
    wall0 = time.perf_counter()
    for i in range(steps):
        if B.do_flush:
            flush.zero_()                                           # L2 flush between timed iterations
        evs[i][0].record()
        last = one_step(devsets[i % nsets])
        mids[i].record()
        if sync is not None:
            sync.join()
        evs[i][1].record()
    torch.cuda.synchronize()
    wall = time.perf_counter() - wall0
    launches = (lib.vpn_launch_count() - launches0) // steps
    if graphed is not None:
        launches = graphed.launches_per_step + (0 if (ar_in_graph or sync is None) else (lib.vpn_launch_count() - launches0) // steps)
    sampler.stop()
    sampler.join(timeout=5.0)
    B.barrier()
    # copied now: the graphed step returns static buffers, which the e2e loop below overwrites
    outputs = ({name: x.detach().cpu().numpy() for name, x in zip(("loss", "grad_v", "grad_q", "grad_t"), last)}
               if keep_outputs else None)
    step_ms = [a.elapsed_time(bb) for a, bb in evs]
    total_ms = torch.tensor([sum(step_ms)], dtype=torch.float64, device=dev)
    # per rank: mean step time and the part of it spent before the all-reduce's completion is awaited
    own_ms = sum(a.elapsed_time(m_) for (a, _), m_ in zip(evs, mids)) / steps
    rank_ms = torch.tensor([sum(step_ms) / steps, own_ms], dtype=torch.float64, device=dev)
    rank_all = [rank_ms]
    if world > 1:
        dist.all_reduce(total_ms, op=dist.ReduceOp.MAX)
        rank_all = [torch.zeros_like(rank_ms) for _ in range(world)]
        dist.all_gather(rank_all, rank_ms)
    rank_all = [[round(float(x), 4) for x in r_.tolist()] for r_ in rank_all]
    total_ms = float(total_ms.item())
    value = world * b * steps / (total_ms * 1e-3)

    # ---- end to end through the public API with host buffers ("e2e") ------------------------------
    # same conditions as above (flush before every step, clock sampling); every step's inputs are copied from pinned host
    # memory and its results land in pinned host buffers, through vpn_b200.HostPipeline - the package's loop for host
    # batches: the copy of batch i + 1 runs on a copy stream while step i computes, and the host synchronises once per
    # step, on the oldest outstanding result.  Timed over the whole loop (first submit to last result), flushes included.
    def e2e_fn(s):
        out = one_step(s)
        if sync is not None:
            sync.join()
        return out

    def e2e_flush():
        if B.do_flush:
            flush.zero_()

    pipe = vpn.HostPipeline(e2e_fn, pinned[0], dev, pre_step=e2e_flush)

    def e2e_loop(count):
        pipe.submit(pinned[0])
        for i in range(1, count):
            pipe.submit(pinned[i % nsets])
            pipe.result()
        return pipe.result()

    e2e_loop(3)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e2e_steps = max(3, steps // 2)
    sampler2 = B.new_sampler()
    B.barrier()
    sampler2.arm()
    t0 = time.perf_counter()
    e0.record()
    e2e_loop(e2e_steps)
    e1.record()
    torch.cuda.synchronize()
    e2e_wall = time.perf_counter() - t0
    sampler2.stop()
    sampler2.join(timeout=5.0)
    e2e_ms = torch.tensor([max(e0.elapsed_time(e1), e2e_wall * 1e3)], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(e2e_ms, op=dist.ReduceOp.MAX)
    e2e_value = world * b * e2e_steps / (float(e2e_ms.item()) * 1e-3)
    h2d = sum(vv.numel() * vv.element_size() for vv in pinned[0].values() if vv is not None)
    d2h = 4 + b * k * 10 * 4
    ar_timeout = bool(sync.nvls_timed_out()) if sync is not None else False
    if rank != 0:
        return None

    out = {"workload": describe(workload, world), "value": value, "unit": "samples/s", "ms_per_step": total_ms / steps,
           "steps": steps, "scaling": "strong" if workload in STRONG else "weak", "global_batch": world * b,
           "gpu_launches": int(launches), "cuda_graph": graphed is not None, "cuda_graph_error": graph_error,
           "allreduce_in_graph": bool(ar_in_graph), "allreduce_wait_timed_out": ar_timeout,
           "wall_ms_per_step_incl_flush": wall * 1e3 / steps, "rank_ms_step_and_own_kernels": rank_all,
           "clocks": sampler.summary(),
           "e2e": {"value": e2e_value, "unit": "samples/s", "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h),
                   "steps": e2e_steps, "clocks": sampler2.summary(),
                   "conditions": "same as value: 256 MB L2 flush before every step (inside the timed region here), NVML "
                                 "clock sampling on rank 0, all-reduce inside the step; one host synchronisation per step; "
                                 "vpn_b200.HostPipeline: the host-to-device copy of batch i + 1 overlaps step i, every "
                                 "batch and every result is copied every step"}}
    if outputs is not None:
        out["outputs"] = outputs
    if not with_rooflines:
        return out

    # ---- roofline of the dominant kernel group: Chamfer forward (FP32 pipe) ----------------------
    s = devsets[0]
    with torch.no_grad():
        if vertex_mode:
            from vpn_b200 import templates as _tpl
            pts = vpn.mesh_vertices(_tpl.template(kind, dev)[0], s["v"], s["q"], s["t"])
        else:
            pts = vpn.sample_primitives(kind, s["v"], s["q"], s["t"], torch.rand((b, k, n, width), device=dev))
        reps = 10
        vpn.chamfer_nn_stage_ms(pts, s["target"], chamfer_impl, reps=3)
        stage = vpn.chamfer_nn_stage_ms(pts, s["target"], chamfer_impl, reps=reps)
        cham_ms = stage["total"]
        # sampling kernel: a stream of launches over rotating uniform buffers larger than L2 in total (every
        # launch reads cold inputs; no write-flush, whose dirty lines would be written back during the launch)
        sbytes = b * k * n * (12 + 4 * width)
        nrot = min(64, max(2, -(-300_000_000 // sbytes)))
        nl = 4 * nrot
        us = [torch.rand((b, k, n, width), device=dev) for _ in range(nrot)]
        samp_ms = vpn.sample_primitives_ms(kind, s["v"], s["q"], s["t"], us, reps=nl)
        del us
    peak = vpn.fp32_peak_tflops(dev)
    flops = 8.0 * b * (k * n) * m                      # 8 flop per (predicted, target) pair, both directions
    main_ms = stage["main"] if stage["main"] > 0 else cham_ms
    achieved = flops / (main_ms * 1e-3) / 1e12
    sm_mhz_max = sampler.summary()["sm_max_mhz"] or 1965
    nominal = 148 * 128 * 2 * sm_mhz_max * 1e6 / 1e12
    peak_tf = max(peak["ffma2"], peak["ffma"])
    main_kernel = vpn.chamfer_main_kernel_name(b, k * n, m, chamfer_impl)
    traffic_db = {}
    try:
        traffic_db = json.load(open(os.path.join(REPO, "profiles", "traffic.json"))).get(workload, {})
    except Exception:
        pass
    traffic = traffic_db.get(main_kernel)
    tsrc = "profiles/traffic.json (dram__bytes_read.sum + dram__bytes_write.sum per launch, ncu --set full capture of the same launch)"
    skipped_share = (stage.get("stages_skipped", 0) / stage["stages"]) if stage.get("stages") else 0.0
    executed_tf = achieved * (1.0 - skipped_share)      # 8 flop per pair the filter actually evaluates
    roofline = {"kernel": main_kernel + " (main kernel of vpn_chamfer_fwd; both Chamfer directions in one launch"
                          + (", preceded by the target sort, pruning-bounds and plan kernels, which are inside `ms`" if skipped_share else "") + ")",
                "bound": "fp32", "achieved": executed_tf, "peak": peak_tf, "unit": "TFLOP/s", "frac": executed_tf / peak_tf,
                "peak_source": "live FFMA2 stream probe (vpn_fp32_peak_probe), burst; MEASURED_PEAKS.json has no FP32 "
                               "entry; nominal 148 SM x 128 lanes x 2 x max clock given beside it",
                "peak_nominal": nominal, "frac_of_nominal": executed_tf / nominal, "ms": main_ms,
                "algorithmic_flops": flops * (1.0 - skipped_share), "traffic": traffic, "traffic_source": tsrc if traffic else None,
                "pairs_skipped_share": skipped_share,
                "pairs_skipped_note": "share of the 128 x 128 distance blocks (both directions) the spatial pruning proves "
                                      "irrelevant and never evaluates (csrc/chamfer_prep.cu).  `achieved` / `frac` count 8 flop "
                                      "for the EVALUATED pairs only (the kernel's own work over its time, prep kernels included "
                                      "in the time); `all_pairs` is the same time against the reference's full pair count",
                "all_pairs": {"flops": flops, "tflops": achieved, "x_peak": achieved / peak_tf,
                              "note": "8 flop x B x P x M / ms: what a kernel evaluating every pair would have to sustain to "
                                      "finish in this time; above the FP32 peak because most pairs are never evaluated"},
                "note": "achieved = 8 flop per (predicted, target) pair / kernel time, against the FP32 FMA peak the "
                        "north star names; chamfer_tc_kernel evaluates the pairs on the tensor cores (fp16-split "
                        "operands, the fp32 sum rounded once into an fp16 accumulator) and is bounded by the packed integer mins of its epilogue on the ALU pipe, see DESIGN.md 4.1",
                "forward_total": {"ms": cham_ms, "stages_ms": stage,
                                  "achieved": flops * (1.0 - skipped_share) / (cham_ms * 1e-3) / 1e12,
                                  "frac": flops * (1.0 - skipped_share) / (cham_ms * 1e-3) / 1e12 / peak_tf,
                                  "all_pairs_tflops": flops / (cham_ms * 1e-3) / 1e12,
                                  "note": "main kernel + exact recovery kernels: the time to the final min / arg-min; "
                                          "achieved / frac count the evaluated pairs only"}}
    hbm_peak, tensor_peak = 6536.7, None
    try:
        mp = json.load(open(os.path.join(REPO, "MEASURED_PEAKS.json")))
        hbm_peak, hbm_src = mp["hbm_gbs"], "MEASURED_PEAKS.json"
        tensor_peak = mp.get("bf16_tflops")
    except Exception:
        hbm_peak, hbm_src = 6650.0, "fallback"
    if main_kernel == "chamfer_tc_kernel":
        # what the tensor pipe actually executes: a 16-term fp16 dot product per pair and direction (2 x 16 MACs = 64 flop)
        executed = 64.0 * b * (k * n) * m * (1.0 - skipped_share) / (main_ms * 1e-3) / 1e12
        roofline["tensor_executed"] = {"tflops": executed, "peak_dense_16bit": tensor_peak,
                                       "frac": (executed / tensor_peak) if tensor_peak else None,
                                       "note": "fp16 operands, fp16 accumulator (fp32 sum rounded once), K = 16; padded tiles not counted"}
    out["roofline"] = roofline
    if not vertex_mode:
        pk = "pose_fwd_kernel"
        out["roofline_sampling"] = {
            "kernel": "pose_fwd_kernel (fused sample+pose)", "bound": "hbm",
            "achieved": sbytes / (samp_ms * 1e-3) / 1e9, "peak": hbm_peak, "unit": "GB/s",
            "frac": sbytes / (samp_ms * 1e-3) / 1e9 / hbm_peak, "peak_source": hbm_src, "ms": samp_ms,
            "algorithmic_bytes": sbytes, "traffic": traffic_db.get(pk), "traffic_source": tsrc if traffic_db.get(pk) else None,
            "how": f"{nl} back-to-back launches over {nrot} rotating uniform buffers ({nrot * sbytes // 2 >> 20} MB of inputs > L2), "
                   "one CUDA-event pair around the stream (vpn_pose_points_fwd_timed)"}
    if res:
        from vpn_b200 import templates
        with torch.no_grad():
            tv, tf = templates.template(kind, dev)
            verts = vpn.mesh_vertices(tv, s["v"], s["q"], s["t"])
            faces = step_fn.composed_faces(k, dev)
            rot, pos = vpn.look_at_cameras(torch.zeros(b, device=dev), torch.zeros(b, device=dev), torch.ones(b, device=dev))
            for _ in range(2):
                vpn.soft_silhouette(verts, faces, rot, pos, res, res)
            re_ = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(reps)]
            for i in range(reps):
                flush.zero_()
                re_[i][0].record()
                vpn.soft_silhouette(verts, faces, rot, pos, res, res)
                re_[i][1].record()
            torch.cuda.synchronize()
            r_ms = sum(a.elapsed_time(bb) for a, bb in re_) / reps
        rbytes = 12 * b * verts.shape[1] + 12 * faces.shape[0] + 4 * b * res * res
        rt = [traffic_db.get(kn) for kn in ("sil_project_kernel", "sil_faces_kernel", "sil_raster_fwd_kernel")]
        out["roofline_raster"] = {
            "kernel": "sil_project_kernel + sil_faces_kernel + sil_raster_fwd_kernel (vpn_silhouette_fwd, whole batch)",
            "bound": "hbm", "achieved": rbytes / (r_ms * 1e-3) / 1e9, "peak": hbm_peak, "unit": "GB/s",
            "frac": rbytes / (r_ms * 1e-3) / 1e9 / hbm_peak, "peak_source": hbm_src, "ms": r_ms,
            "algorithmic_bytes": rbytes, "traffic": (sum(rt) if all(x is not None for x in rt) else None),
            "traffic_source": tsrc if all(x is not None for x in rt) else None, "faces": int(faces.shape[0]),
            "pixel_face_tests_per_s": b * res * res * float(faces.shape[0]) / (r_ms * 1e-3),
            "note": "algorithmic bytes are ~1 us of HBM time: the rasteriser is latency / ALU bound (DESIGN.md 4.4)"}
    out["fp32_peak_probe_tflops"] = peak
    if cpu_baseline:
        threads = os.cpu_count() or 1
        rows = cpu_sample_rows(workload)
        cpu_reference_step(workload, min(rows, n), threads)      # warm-up on one primitive
        dt, frac, used = cpu_reference_step(workload, rows, threads)
        out["cpu_baseline"] = {"value": 1.0 / (dt / frac), "unit": "samples/s", "cores": threads, "kind": "port",
                               "sample": cpu_sample_text(workload, used, dt)}
    return out


def compact(r):
    """One entry of the `configs` block: what the verdict asked for per extra workload (value, ms, roofline, launches)."""
    c = {kk: r[kk] for kk in ("workload", "value", "unit", "ms_per_step", "steps", "scaling", "global_batch", "gpu_launches",
                              "cuda_graph", "allreduce_in_graph")}
    c["e2e"] = {kk: r["e2e"][kk] for kk in ("value", "h2d_bytes_per_step", "d2h_bytes_per_step")}
    c["clocks"] = r["clocks"]
    if "roofline" in r:
        rf = r["roofline"]
        c["roofline"] = {"kernel": rf["kernel"].split(" ")[0], "bound": rf["bound"], "achieved": rf["achieved"], "peak": rf["peak"],
                         "unit": rf["unit"], "frac": rf["frac"], "ms": rf["ms"], "traffic": rf["traffic"],
                         "pairs_skipped_share": rf.get("pairs_skipped_share"), "all_pairs_tflops": rf["all_pairs"]["tflops"],
                         "forward_total_frac": rf["forward_total"]["frac"], "forward_total_ms": rf["forward_total"]["ms"]}
    for key in ("roofline_sampling", "roofline_raster"):
        if key in r:
            rr = r[key]
            c[key] = {kk: rr[kk] for kk in ("bound", "achieved", "peak", "unit", "frac", "ms", "algorithmic_bytes", "traffic")}
    return c


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20,
                    help="timed steps of the headline value (the JSON `value` and `ms_per_step`); the e2e loop times "
                         "max(3, steps // 2) steps and each extra workload of --configs max(5, min(10, steps))")
    ap.add_argument("--warmup", type=int, default=5, help="untimed steps before timing (at least 3)")
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="c2", choices=sorted(WORKLOADS))
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--chamfer-impl", type=int, default=0)
    ap.add_argument("--graph", default="auto", choices=["auto", "on", "off"],
                    help="replay the step from a CUDA graph (vpn_b200.GraphedPrimitiveLoss); auto falls back to eager launches")
    ap.add_argument("--configs", default="auto",
                    help="extra workloads measured after the headline one and reported in the `configs` block of the same JSON "
                         "line: 'auto' = c3,c5,c2f,c4 when the headline is c2, 'none', or a comma-separated list")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the last timed step of the headline workload returned (loss and the gradients to "
                         "v, q, t; rank 0) as DIR/<name>.npy, to compare two builds output for output")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.impl == "reference":
        if args.dump_outputs:
            ap.error("--dump-outputs applies to --impl ours")
        return run_reference(args)
    B = Bench(args)
    world, rank = B.world, B.rank
    warm = max(3, args.warmup)
    head = measure_workload(B, args.workload, args.steps, warm, args.chamfer_impl, args.graph, with_rooflines=True,
                            cpu_baseline=(world == 1 and not args.no_cpu_baseline),
                            keep_outputs=bool(args.dump_outputs))
    if rank == 0 and args.dump_outputs:
        import numpy as np
        os.makedirs(args.dump_outputs, exist_ok=True)
        for name, arr in head.pop("outputs").items():
            np.save(os.path.join(args.dump_outputs, name + ".npy"), arr)
    extras = []
    if args.configs == "auto":
        extras = ["c3", "c5", "c2f", "c4"] if args.workload == "c2" else []
    elif args.configs != "none":
        extras = [w for w in args.configs.split(",") if w in WORKLOADS and w != args.workload]
    configs = {}
    for w in extras:
        try:
            r = measure_workload(B, w, max(5, min(10, args.steps)), 3, args.chamfer_impl, args.graph, with_rooflines=True)
            if rank == 0:
                configs[w] = compact(r)
        except Exception as e:                               # noqa: BLE001 - an extra workload must not cost the headline line
            if world > 1:
                raise                                        # ranks must stay in lock step: fail loudly
            configs[w] = {"error": repr(e)[:200]}
    if rank == 0:
        sync = B.sync
        line = {"metric": METRIC, "value": head["value"], "unit": "samples/s", "n_gpus": world, "steps": args.steps,
                "warmup": warm, "ms_per_step": head["ms_per_step"], "higher_is_better": True,
                "scaling": head["scaling"], "vs_baseline": None, "dtype": "f32", "data": "synthetic",
                "config": {"workload": head["workload"], "global_batch": head["global_batch"],
                           "parallelism": f"dp{world}", "l2": "256 MB L2 flush before every timed step (value: outside the "
                           "per-step CUDA-event pairs; e2e: inside the timed loop); 4 rotating input sets",
                           "cuda_graph": head["cuda_graph"], "cuda_graph_error": head["cuda_graph_error"],
                           "allreduce_numel": GRAD_NUMEL if world > 1 else 0,
                           "allreduce": (sync.mode if sync is not None else None),
                           "allreduce_in_graph": head["allreduce_in_graph"],
                           "allreduce_wait_timed_out": head["allreduce_wait_timed_out"],
                           "allreduce_trial_ms": (sync.trial_ms if sync is not None else None),
                           "wall_ms_per_step_incl_flush": head["wall_ms_per_step_incl_flush"],
                           "rank_ms_step_and_own_kernels": head["rank_ms_step_and_own_kernels"], "l2_flush": B.do_flush,
                           "timed_region": "barrier + synchronize on every rank immediately before the first timed step "
                                           "(after all per-rank set-up, incl. NVML init on rank 0) and after the last"},
                "clocks": head["clocks"], "gpu_launches": head["gpu_launches"], "e2e": head["e2e"],
                "roofline": head.get("roofline"), "roofline_sampling": head.get("roofline_sampling"),
                "roofline_raster": head.get("roofline_raster"), "cpu_baseline": head.get("cpu_baseline"),
                "fp32_peak_probe_tflops": head.get("fp32_peak_probe_tflops"),
                "configs": configs}
        print(json.dumps(line), flush=True)
    if world > 1:
        B.dist.barrier()
        B.dist.destroy_process_group()


if __name__ == "__main__":
    main()
