"""The tail of bench.py's c2 step: what one replay of the CUDA graph launches with each kernel's device time, and the time
of the VP-diverse Chamfer term (16 centres against 8192 targets per sample).  Prints one JSON line.  Run on the GPU:

    python tools/bench_step_tail.py [--replays 20] [--reps 7] [--inner 50]

- `replay`: every kernel and memset of one replay, from torch.profiler in a run of its own over --replays replays:
  the count per replay and the mean device time per replay by kernel name, with the loss heads summed apart
  (the Chamfer loss kernels plus the torch reductions, multiplies and fills around them).
- `vp_div`: CUDA-event time of the term's eager forward and of its backward (launch gaps included, so mostly what the
  host takes to issue them), each the mean of --inner calls, median and range over --reps repetitions.

Written to run on older trees too: where ops.chamfer_distance has no `weight` argument it times the composition the
step used then, chamfer_distance(...) * weight.
"""
import argparse
import inspect
import json
import os
import subprocess
import sys
from collections import defaultdict

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(REPO, "volumetric-primitives-net_b200")); sys.path.insert(0, REPO)

import torch  # noqa: E402
import vpn_b200  # noqa: E402
from vpn_b200 import ops  # noqa: E402
from bench import synthetic, WORKLOADS  # noqa: E402

LOSS_HEAD = ("chamfer_loss", "reduce_kernel", "elementwise_kernel", "fill", "FillFunctor", "MulFunctor", "mean")


def c2_step(dev):
    kind, b, k, n, m, _ = WORKLOADS["c2"]
    s = synthetic("c2", "cpu")[0]
    v, q, t, tgt = (s[x].to(dev) for x in ("v", "q", "t", "target"))
    return vpn_b200.GraphedPrimitiveLoss(vpn_b200.PrimitiveLossConfig(kind=kind), v, q, t, tgt, n_samples=n), (v, q, t, tgt)


def profile_replay(g, inputs, replays):
    from torch.profiler import ProfilerActivity, profile
    for _ in range(5):
        g(*inputs)
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(replays):
            g.graph.replay()
        torch.cuda.synchronize()
    names, kernels, memsets = defaultdict(float), 0, 0
    for e in prof.events():
        if e.device_type != torch.autograd.DeviceType.CUDA:
            continue
        low = e.name.lower()
        if "memset" in low:
            memsets += 1
        elif "memcpy" not in low:
            kernels += 1
        names[e.name] += e.device_time_total if hasattr(e, "device_time_total") else e.cuda_time_total
    per = {k: round(v / replays, 2) for k, v in sorted(names.items(), key=lambda kv: -kv[1])}
    head = sum(v for k, v in per.items() if any(s in k for s in LOSS_HEAD))
    return {"kernels_per_replay": kernels / replays, "memsets_per_replay": memsets / replays,
            "loss_heads_us": round(head, 2), "us_by_name": per}


def time_vp_div(dev, reps, inner):
    s = synthetic("c2", "cpu")[0]
    t = s["t"].to(dev).contiguous().requires_grad_()
    tgt = s["target"].to(dev)
    w = vpn_b200.PrimitiveLossConfig().l_vp_div
    native = "weight" in inspect.signature(ops.chamfer_distance).parameters
    fwd = (lambda: ops.chamfer_distance(t, tgt, w1=0.5, w2=1.0, weight=w)) if native else \
        (lambda: ops.chamfer_distance(t, tgt, w1=0.5, w2=1.0) * w)
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(4)]
    f_ms, b_ms = [], []
    for r in range(reps + 1):
        ef = eb = 0.0
        for _ in range(inner):
            ev[0].record()
            loss = fwd()
            ev[1].record()
            ev[2].record()
            torch.autograd.grad(loss, (t,))
            ev[3].record()
            torch.cuda.synchronize()
            ef += ev[0].elapsed_time(ev[1]); eb += ev[2].elapsed_time(ev[3])
        if r:                                   # the first repetition warms up
            f_ms.append(ef / inner); b_ms.append(eb / inner)
    stat = lambda v: {"median": sorted(v)[len(v) // 2], "min": min(v), "max": max(v)}
    return {"native_weighted_mean": native, "fwd_ms": stat(f_ms), "bwd_ms": stat(b_ms)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--replays", type=int, default=20)
    ap.add_argument("--reps", type=int, default=7)
    ap.add_argument("--inner", type=int, default=50)
    args = ap.parse_args()
    dev = torch.device("cuda")
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()
    g, inputs = c2_step(dev)
    out = {"gpu": smi[0] if smi else torch.cuda.get_device_name(dev),
           "our_launches_per_replay": g.launches_per_step,
           "replay": profile_replay(g, inputs, args.replays),
           "vp_div": time_vp_div(dev, args.reps, args.inner)}
    print(json.dumps(out), flush=True)


if __name__ == "__main__":
    main()
