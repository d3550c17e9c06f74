"""Cost of one primitive-loss step on a mixed cuboid + sphere assembly (PrimitiveLoss / GraphedPrimitiveLoss with
kind="mixed"), against the single-kind steps of the same K and the drop-in composition train.py runs without it.

    a0 train.py defaults with CUBOID_NUM = SPHERE_NUM = 8: B = 8, 16 primitives x 128 samples, M = 2048, l_vp_div = 0.1
    a1 the same with l_sil = 1 at 128 x 128
    b  C2 size: B = 32, 8 + 8 primitives x 4096 samples, M = 8192

Each step draws the uniforms and computes the loss and its gradient to (v, q, t), in five forms:
    mixed_graphed   GraphedPrimitiveLoss(kind="mixed", n_cuboids=8)
    mixed_eager     PrimitiveLoss(kind="mixed", n_cuboids=8)
    cuboid_graphed  GraphedPrimitiveLoss(kind="cuboid"), all 16 primitives cuboids
    sphere_graphed  GraphedPrimitiveLoss(kind="sphere"), all 16 primitives spheres
    dropin          train.py's helpers on the drop-in modules: Sampling / Meshing per primitive, torch.cat,
                    modules.loss.{ChamferDistanceLoss, VPDiverseLoss, SilhouetteLoss}, eager

Timing: CUDA events around every step; a 256 MB write flushes the 126 MB L2 before every step, outside the timed interval.
Each form runs warm-up steps, then enough steps to last --seconds per round; forms alternate within a round; the median
over rounds is reported.  The mixed pose forward (vpn_pose_mixed_fwd, sampled) is timed alone the same way at each
workload's shape and reported as GB/s on its algorithmic bytes B*N*(Kc*24 + Ks*20) (12 or 8 bytes of uniforms read and
12 bytes of points written per point), next to a device-to-device copy moving as many bytes in the same run.  The card's
name and power limit are read in the same run.  Writes one JSON file (--out)."""
import argparse
import json
import math
import os
import statistics
import sys

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (REPO, os.path.join(REPO, "volumetric-primitives-net_b200"), os.path.join(REPO, "tools")):
    if p not in sys.path:
        sys.path.insert(0, p)

import torch  # noqa: E402

import vpn_b200  # noqa: E402
from vpn_b200 import _lib  # noqa: E402
from bench_step_emd import card, time_steps  # noqa: E402

WORKLOADS = {
    "a0_train_b8": dict(b=8, kc=8, ks=8, n=128, m=2048, res=0),
    "a1_train_b8_sil128": dict(b=8, kc=8, ks=8, n=128, m=2048, res=128),
    "b_c2_b32": dict(b=32, kc=8, ks=8, n=4096, m=8192, res=0),
}
FORMS = ("mixed_graphed", "mixed_eager", "cuboid_graphed", "sphere_graphed", "dropin")


def inputs(w, dev, seed=1234):
    from oracle import vpn_oracle as O
    b, k = w["b"], w["kc"] + w["ks"]
    g = torch.Generator().manual_seed(seed)
    v, q, t = O.synthetic_primitives(b, k, seed=seed)
    tgt = (torch.rand(b, w["m"], 3, generator=g) - 0.5) * 0.8
    sil = (torch.rand(b, 1, w["res"], w["res"], generator=g) > 0.5).float() if w["res"] else None
    return v.to(dev), q.to(dev), (t * 0.3).to(dev), tgt.to(dev), None if sil is None else sil.to(dev)


def config(w, kind):
    return vpn_b200.PrimitiveLossConfig(kind=kind, n_cuboids=w["kc"] if kind == "mixed" else 0,
                                        l_sil=1.0 if w["res"] else 0.0, l_vp_div=0.1)


def count_launches(fn):
    lib = _lib.load()
    torch.cuda.synchronize()
    n0 = lib.vpn_launch_count()
    fn()
    torch.cuda.synchronize()
    return int(lib.vpn_launch_count() - n0)


def runner(w, form, data):
    """(step function, our kernel launches per step)."""
    v, q, t, tgt, sil = data
    b, kc, ks, n = w["b"], w["kc"], w["ks"], w["n"]
    if form == "dropin":
        from test_gpu_train_loop_integration import helpers
        ns = helpers("train", CUBOID_NUM=kc, SPHERE_NUM=ks, SAMPLE_NUM=n, L_SIL=1.0 if w["res"] else 0.0, L_VP_DIV=0.1,
                     L_CAN_CD=0.0)
        leaves = [x.clone().requires_grad_() for x in (v, q, t)]
        zero, one = torch.zeros(b, device=v.device), torch.ones(b, device=v.device)

        def fn():
            vols, rots, trs = ([x[:, i] for i in range(kc + ks)] for x in leaves)
            pts = ns["sample_predict_points"](vols, rots, trs)
            view_cd, obj_cd = ns["calculate_cd_loss"](pts, tgt, tgt, one, zero, zero, zero)
            loss = view_cd + obj_cd + ns["calculate_vp_div_loss"](trs, tgt)
            if sil is not None:
                meshes = ns["compose_vp_meshes"](ns["get_vp_meshes"](vols, rots, trs))
                loss = loss + ns["calculate_silhouette_loss"](meshes, sil, one, zero, zero)
            return torch.autograd.grad(loss, leaves)
    elif form == "mixed_eager":
        step = vpn_b200.PrimitiveLoss(config(w, "mixed"))
        leaves = [x.clone().requires_grad_() for x in (v, q, t)]

        def fn():
            u = (torch.rand((b, kc, n, 3), device=v.device), torch.rand((b, ks, n, 2), device=v.device))
            out = step(*leaves, u, tgt, silhouettes=sil)
            return torch.autograd.grad(out["total"], leaves)
    else:
        kind = form.split("_")[0]
        g = vpn_b200.GraphedPrimitiveLoss(config(w, kind), v, q, t, tgt, sil, n_samples=n)
        fn = lambda: g(v, q, t, tgt, sil)
        for _ in range(3):
            fn()
        return fn, g.launches_per_step          # a replay launches nothing from the host: the kernels captured in the graph
    for _ in range(3):
        fn()
    return fn, count_launches(fn)


def pose_fwd_gbs(w, data, flush, seconds, rounds):
    """vpn_pose_mixed_fwd (sampled) alone, and a device-to-device copy moving its algorithmic bytes: GB/s, medians."""
    v, q, t = data[:3]
    b, kc, ks, n = w["b"], w["kc"], w["ks"], w["n"]
    g = torch.Generator(device=v.device).manual_seed(5)
    uc = torch.rand((b, kc, n, 3), device=v.device, generator=g)
    us = torch.rand((b, ks, n, 2), device=v.device, generator=g)
    nbytes = b * n * (kc * 24 + ks * 20)
    src = torch.empty(nbytes // 2, dtype=torch.uint8, device=v.device)
    dst = torch.empty_like(src)
    calls = {"pose_mixed_fwd": lambda: vpn_b200.sample_mixed_primitives(kc, v, q, t, uc, us),
             "d2d_copy": lambda: dst.copy_(src)}
    steps = {}
    for k, fn in calls.items():
        time_steps(fn, 20, flush)
        steps[k] = max(200, math.ceil(seconds * 1e3 / time_steps(fn, 50, flush)))
    ms = {k: [] for k in calls}
    for _ in range(rounds):
        for k, fn in calls.items():
            ms[k].append(time_steps(fn, steps[k], flush))
    med = {k: statistics.median(x) for k, x in ms.items()}
    return {"algorithmic_bytes": nbytes, "ms": {k: round(x, 5) for k, x in med.items()},
            "gb_per_s": {k: round(nbytes / (x * 1e6), 1) for k, x in med.items()},
            "pose_over_copy": round(med["d2d_copy"] / med["pose_mixed_fwd"], 3)}


def main():
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("--workloads", default=",".join(WORKLOADS), help="comma-separated subset of " + ", ".join(WORKLOADS))
    ap.add_argument("--rounds", type=int, default=3, help="rounds; each times every form once, in turn")
    ap.add_argument("--seconds", type=float, default=1.5, help="device time per form per round")
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--out", default=None, help="JSON file to write (default: print only)")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("bench_mixed_step.py measures on the GPU and found none")
    sys.path.insert(0, os.path.join(REPO, "tests"))           # the restated train.py helpers of the integration tests
    dev = torch.device("cuda:0")
    torch.cuda.set_device(dev)
    torch.manual_seed(0)
    flush = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device=dev)
    result = {"card": card(), "l2": "256 MB write before every step, outside the timed interval",
              "timing": f"CUDA events around each step; median over {args.rounds} rounds of >= {args.seconds} s per form, "
                        f"forms alternated within a round", "workloads": {}}
    for name in args.workloads.split(","):
        w = WORKLOADS[name]
        data = inputs(w, dev)
        runners = {f: runner(w, f, data) for f in FORMS}
        steps = {}
        for f, (fn, _) in runners.items():
            time_steps(fn, args.warmup, flush)
            steps[f] = max(50, math.ceil(args.seconds * 1e3 / time_steps(fn, 20, flush)))
        ms = {f: [] for f in FORMS}
        for _ in range(args.rounds):
            for f, (fn, _) in runners.items():
                ms[f].append(time_steps(fn, steps[f], flush))
        med = {f: statistics.median(x) for f, x in ms.items()}
        res = {"shape": w, "ms_per_step": {f: round(med[f], 4) for f in FORMS},
               "ms_per_step_rounds": {f: [round(x, 4) for x in ms[f]] for f in FORMS}, "steps_per_round": steps,
               "launches_per_step": {f: runners[f][1] for f in FORMS},
               "mixed_graphed_speedup_over_dropin": round(med["dropin"] / med["mixed_graphed"], 2),
               "pose_forward": pose_fwd_gbs(w, data, flush, args.seconds, args.rounds)}
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
