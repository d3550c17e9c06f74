"""Cost of one mesh-loss step (vpn_b200.MeshLoss / GraphedMeshLoss) on the shapes of train_sphere.py and train_gcn.py,
against the drop-in composition those loops run without it, and the sampler's gather backward against the atomic one.

    a0 train_sphere.py defaults: B = 8, the 386-vertex sphere + tanh(N) * 0.05 offsets, n = 2048 samples, M = 2048, l_sil 0
    a1 the same with l_sil = 1 at 128 x 128
    b  BASELINE config 1, script-faithful: B = 1, n = 16384, M = 2048, l_sil = 1 at 64 x 64
    c  train_gcn.py: B = 8, 2048 vertices of 16 composed spheres (4032 faces), M = 2048, Chamfer + EMD, no silhouette

Each step computes the loss and its gradient to the vertices (train_sphere.py: the offsets'), in four forms:
    dropin    modules.meshing.TriangleMesh.sample_batch + modules.loss.{ChamferDistanceLoss, SilhouetteLoss,
              EarthMoverDistanceLoss + sqrt + mean}, eager - what a user of either loop runs today
    eager     MeshLoss
    graphed   GraphedMeshLoss
    e2e       GraphedMeshLoss through HostPipeline: vertices and targets from pinned host memory, results back to it

Timing: CUDA events around every step; a 256 MB write flushes the 126 MB L2 before every step, outside the timed interval
(e2e: the flush is HostPipeline's pre_step, inside the timed loop, and the loop is timed first submit to last result).
Each form runs warm-up steps, then enough steps to last --seconds per round; forms alternate within a round; the median
over rounds is reported.  The sampler backward alone (vpn_mesh_sample_bwd_sorted against vpn_mesh_sample_bwd, memset
included) is timed the same way at the sample counts of a and b.  The card's name and power limit are read in the same
run.  Writes one JSON file (--out)."""
import argparse
import ctypes
import json
import math
import os
import statistics
import sys
import time

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (REPO, os.path.join(REPO, "volumetric-primitives-net_b200"), os.path.join(REPO, "tools")):
    if p not in sys.path:
        sys.path.insert(0, p)

import numpy as np  # noqa: E402
import torch  # noqa: E402

import vpn_b200  # noqa: E402
from vpn_b200 import _lib, ops  # noqa: E402
from vpn_b200._lib import check, ptr, stream_ptr  # noqa: E402
from bench_step_emd import card, time_steps  # noqa: E402

WORKLOADS = {
    "a0_sphere_b8": dict(b=8, n=2048, m=2048, res=0, mesh="sphere386", l_emd=0.0),
    "a1_sphere_b8_sil128": dict(b=8, n=2048, m=2048, res=128, mesh="sphere386", l_emd=0.0),
    "b_c1_b1_sil64": dict(b=1, n=16384, m=2048, res=64, mesh="sphere386", l_emd=0.0),
    "c_gcn_b8_emd": dict(b=8, n=0, m=2048, res=0, mesh="gcn", l_emd=1.0),
}
FORMS = ("dropin", "eager", "graphed", "e2e")


def inputs(w, dev, seed=1234):
    """(verts (B,V,3), faces (F,3) int32, targets (B,M,3), silhouettes (B,1,H,W) or None) on the device.  The sphere's
    vertices are template + offsets; their gradient is the offsets'."""
    g = torch.Generator().manual_seed(seed)
    b = w["b"]
    if w["mesh"] == "sphere386":
        t = np.load(os.path.join(REPO, "tests", "golden", "templates.npz"))
        tv = torch.from_numpy(t["sphere386_vertices"]).float()
        faces = torch.from_numpy(t["sphere386_faces"]).int()
        offs = torch.tanh(torch.randn(b, tv.shape[0], 3, generator=g)) * 0.05
        verts = tv[None] + offs
        tgt = (torch.rand(b, w["m"], 3, generator=g) - 0.5) * 0.9
    else:
        faces = vpn_b200.PrimitiveLoss().composed_faces(16, "cpu")
        verts = torch.rand(b, 2048, 3, generator=g) * 0.6 + 0.2                     # EMD wants coordinates in [0, 1]
        tgt = torch.rand(b, w["m"], 3, generator=g) * 0.8 + 0.1
    sil = (torch.rand(b, 1, w["res"], w["res"], generator=g) > 0.5).float() if w["res"] else None
    return verts.to(dev), faces.to(dev), tgt.to(dev), None if sil is None else sil.to(dev)


def config(w):
    return vpn_b200.MeshLossConfig(n_samples=w["n"], l_sil=1.0 if w["res"] else 0.0, l_emd=w["l_emd"])


def count_launches(fn):
    lib = _lib.load()
    torch.cuda.synchronize()
    n0 = lib.vpn_launch_count()
    fn()
    torch.cuda.synchronize()
    return int(lib.vpn_launch_count() - n0)


class Runner:
    def __init__(self, w, form, data, flush):
        verts, faces, tgt, sil = data
        cfg = config(w)
        self.form = form
        if form == "dropin":
            from modules.loss import ChamferDistanceLoss, EarthMoverDistanceLoss, SilhouetteLoss
            from modules.meshing import TriangleMesh
            cd, sl, emd = ChamferDistanceLoss(), SilhouetteLoss(), EarthMoverDistanceLoss()
            vl = verts.clone().requires_grad_()
            f64 = faces.long()
            ones, zeros = torch.ones(w["b"], device=verts.device), torch.zeros(w["b"], device=verts.device)

            def fn():
                meshes = [TriangleMesh.from_tensors(vl[i], f64) for i in range(w["b"])]
                pts = TriangleMesh.sample_batch(meshes, w["n"]) if w["n"] else vl
                loss = cd(pts, tgt)
                if w["l_emd"]:
                    d, _ = emd(pts, tgt, 0.005, 50)
                    loss = loss + torch.sqrt(d).mean() * w["l_emd"]
                if sil is not None:
                    loss = loss + sl(meshes, sil, ones, zeros, zeros)
                return torch.autograd.grad(loss, (vl,))
            self.fn = fn
        elif form == "eager":
            step = vpn_b200.MeshLoss(cfg)
            vl = verts.clone().requires_grad_()

            def fn():
                out = step(vl, faces, tgt, silhouettes=sil)
                return torch.autograd.grad(out["total"], (vl,))
            self.fn = fn
        else:
            g = vpn_b200.GraphedMeshLoss(cfg, verts, faces, tgt, sil)
            self.graph_launches = g.launches_per_step
            if form == "graphed":
                self.fn = lambda: g(verts, tgt, sil)
            else:
                pinned = [{"verts": verts.cpu().pin_memory(), "targets": tgt.cpu().pin_memory()} for _ in range(2)]
                pipe = vpn_b200.HostPipeline(lambda st: g(st["verts"], st["targets"], sil), pinned[0], verts.device,
                                             pre_step=flush.zero_)
                self.pipe, self.pinned = pipe, pinned
        if form != "e2e":
            for _ in range(3):
                self.fn()
        # a replay launches nothing from the host: the graphed forms report the kernels captured in the graph
        self.launches = count_launches(self.fn) if form in ("dropin", "eager") else self.graph_launches

    def e2e_loop(self, count):
        self.pipe.submit(self.pinned[0])
        for i in range(1, count):
            self.pipe.submit(self.pinned[i % 2])
            self.pipe.result()
        return self.pipe.result()

    def time(self, steps, flush):
        if self.form != "e2e":
            return time_steps(self.fn, steps, flush)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        self.e2e_loop(steps)
        torch.cuda.synchronize()
        return (time.perf_counter() - t0) * 1e3 / steps


def sampler_bwd_ms(b, n, flush, seconds, rounds):
    """vpn_mesh_sample_bwd_sorted against vpn_mesh_sample_bwd (its memset included) on the sphere at (b, n): device ms per
    call, median over alternated rounds, and the largest relative difference of their results."""
    dev = torch.device("cuda")
    t = np.load(os.path.join(REPO, "tests", "golden", "templates.npz"))
    g = torch.Generator().manual_seed(77)
    tv = torch.from_numpy(t["sphere386_vertices"]).float()
    faces = torch.from_numpy(t["sphere386_faces"]).int().to(dev)
    verts = (tv[None] + torch.tanh(torch.randn(b, tv.shape[0], 3, generator=g)) * 0.05).to(dev)
    u = torch.rand(b, n, 3, generator=g).to(dev)
    _, fidx = vpn_b200.sample_mesh_surface(verts, faces, u)
    gp = torch.rand(b, n, 3, generator=g).to(dev)
    nv, nf = verts.shape[1], faces.shape[0]
    offsets, entries = ops.mesh_adjacency(faces, nv)
    lib = _lib.load()
    nb = ctypes.c_size_t(0)
    check(lib.vpn_mesh_sample_bwd_workspace_bytes(b, nf, n, ctypes.byref(nb)), "workspace")
    ws = torch.empty(nb.value, dtype=torch.uint8, device=dev)
    out = {"atomic": torch.empty(b, nv, 3, device=dev), "sorted": torch.empty(b, nv, 3, device=dev)}
    calls = {
        "atomic": lambda: check(lib.vpn_mesh_sample_bwd(ptr(faces), ptr(u), ptr(fidx), ptr(gp), ptr(out["atomic"]), b, nv, nf, n,
                                                        stream_ptr(dev)), "atomic"),
        "sorted": lambda: check(lib.vpn_mesh_sample_bwd_sorted(ptr(faces), ptr(u), ptr(fidx), ptr(gp), ptr(out["sorted"]),
                                                               ptr(offsets), ptr(entries), ptr(ws), nb.value, b, nv, nf, n,
                                                               stream_ptr(dev)), "sorted"),
    }
    steps = {}
    for k, fn in calls.items():
        time_steps(fn, 20, flush)
        steps[k] = max(200, math.ceil(seconds * 1e3 / time_steps(fn, 50, flush)))
    ms = {k: [] for k in calls}
    for _ in range(rounds):
        for k, fn in calls.items():
            ms[k].append(time_steps(fn, steps[k], flush))
    med = {k: statistics.median(x) for k, x in ms.items()}
    rel = float(((out["sorted"] - out["atomic"]).abs().max() / out["atomic"].abs().max()).item())
    return {"b": b, "n": n, "ms": {k: round(v, 5) for k, v in med.items()}, "ms_rounds": {k: [round(x, 5) for x in v] for k, v in ms.items()},
            "sorted_over_atomic": round(med["sorted"] / med["atomic"], 3), "max_abs_diff_over_max_abs": rel}


def main():
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("--workloads", default=",".join(WORKLOADS), help="comma-separated subset of " + ", ".join(WORKLOADS))
    ap.add_argument("--rounds", type=int, default=3, help="rounds; each times every form once, in turn")
    ap.add_argument("--seconds", type=float, default=1.5, help="device time per form per round")
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--out", default=None, help="JSON file to write (default: print only)")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("bench_mesh_step.py measures on the GPU and found none")
    dev = torch.device("cuda:0")
    torch.cuda.set_device(dev)
    torch.manual_seed(0)
    flush = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device=dev)
    result = {"card": card(), "l2": "256 MB write before every step, outside the timed interval (e2e: inside, as pre_step)",
              "timing": f"CUDA events around each step (e2e: host clock over the loop, ending in a synchronise); median over "
                        f"{args.rounds} rounds of >= {args.seconds} s per form, forms alternated within a round",
              "sampler_backward": [sampler_bwd_ms(b, n, flush, args.seconds, args.rounds) for b, n in ((8, 2048), (1, 16384))],
              "workloads": {}}
    print(json.dumps({"sampler_backward": result["sampler_backward"]}), flush=True)
    for name in args.workloads.split(","):
        w = WORKLOADS[name]
        data = inputs(w, dev)
        runners = {f: Runner(w, f, data, flush) for f in FORMS}
        steps = {}
        for f, r in runners.items():
            r.time(args.warmup, flush)
            steps[f] = max(50, math.ceil(args.seconds * 1e3 / r.time(20, flush)))
        ms = {f: [] for f in FORMS}
        for _ in range(args.rounds):
            for f, r in runners.items():
                ms[f].append(r.time(steps[f], flush))
        med = {f: statistics.median(x) for f, x in ms.items()}
        res = {"shape": w, "ms_per_step": {f: round(med[f], 4) for f in FORMS},
               "ms_per_step_rounds": {f: [round(x, 4) for x in ms[f]] for f in FORMS}, "steps_per_round": steps,
               "launches_per_step": {f: runners[f].launches for f in FORMS},
               "e2e_samples_per_s": round(w["b"] * 1e3 / med["e2e"], 1),
               "graphed_speedup_over_dropin": round(med["dropin"] / med["graphed"], 2)}
        print(json.dumps({name: res}), flush=True)
        result["workloads"][name] = res
        del runners
        torch.cuda.synchronize()
    text = json.dumps(result, indent=1)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as fh:
            fh.write(text + "\n")
    print(text)


if __name__ == "__main__":
    main()
