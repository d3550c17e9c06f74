"""Cost of the EMD term in the batched step (train.py:188-195, train_gcn.py:91-95), and where it should run.

For each workload, CUDA-graphed and eager, it times one step (draw uniforms, forward, backward to v, q, t) in three
variants, alternated round by round: without the EMD term (l_emd = 0), with it on the caller's stream (inline), and with
it forked onto its own stream (forked).  PrimitiveLoss._fork_emd is what chooses between the two; this script overrides
it to time both sides, and reports which one the step picks for the workload.

    (a) train.py defaults: B = 8, 16 spheres x 128 samples (P = 2048), M = 2048, l_view_cd 1, l_vp_div 0.1, l_emd 1
    (b) the same at B = 32
    (c) train_gcn.py's vertex path: vertex_chamfer, 16 spheres x 128 template vertices, M = 2048, B = 32

Timing: CUDA events around every step; a 256 MB write flushes the 126 MB L2 before every step, outside the timed
interval.  Each variant runs warm-up steps first, then enough steps to last --seconds per round.  The auction alone is
timed the same way, on the step's points and on uniform clouds of the same shape.  The card's name and power limit are
read in the same run.  Writes one JSON file (--out)."""
import argparse
import contextlib
import json
import math
import os
import statistics
import subprocess
import sys

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (REPO, os.path.join(REPO, "volumetric-primitives-net_b200")):
    if p not in sys.path:
        sys.path.insert(0, p)

import torch  # noqa: E402

import vpn_b200  # noqa: E402
from vpn_b200 import _lib, step as step_mod  # noqa: E402

WORKLOADS = {
    "a_train_b8": dict(b=8, k=16, n=128, m=2048, vertex=False),
    "b_train_b32": dict(b=32, k=16, n=128, m=2048, vertex=False),
    "c_gcn_vertex_b32": dict(b=32, k=16, n=0, m=2048, vertex=True),
}
VARIANTS = ("no_emd", "inline", "forked")
orig_fork = step_mod.PrimitiveLoss._fork_emd


@contextlib.contextmanager
def emd_placement(fork):
    """fork None: the step's own choice; True / False: force the EMD term onto its own stream / the caller's."""
    orig = step_mod.PrimitiveLoss._fork_emd
    if fork is not None:
        step_mod.PrimitiveLoss._fork_emd = lambda self, points: fork
    try:
        yield
    finally:
        step_mod.PrimitiveLoss._fork_emd = orig


def inputs(w, dev, seed=1234):
    from oracle import vpn_oracle as O
    g = torch.Generator().manual_seed(seed)
    v, q, t = O.synthetic_primitives(w["b"], w["k"], seed=seed)
    tgt = 0.5 + (torch.rand(w["b"], w["m"], 3, generator=g) - 0.5) * 0.8         # EMD wants coordinates in [0, 1]
    return [x.to(dev).contiguous() for x in (v, q, t * 0.3 + 0.5, tgt)]


def config(w, variant):
    return vpn_b200.PrimitiveLossConfig(kind="sphere", l_view_cd=1.0, l_vp_div=0.1, l_emd=0.0 if variant == "no_emd" else 1.0,
                                        vertex_chamfer=w["vertex"])


class Runner:
    """One step of one variant, eager or graphed, and the number of our kernel launches in it."""

    def __init__(self, w, variant, graphed, data):
        self.fork = {"no_emd": None, "inline": False, "forked": True}[variant]
        cfg = config(w, variant)
        v, q, t, tgt = data
        lib = _lib.load()
        with emd_placement(self.fork):
            if graphed:
                g = vpn_b200.GraphedPrimitiveLoss(cfg, v, q, t, tgt, None, n_samples=w["n"])
                self.fn = lambda: g(v, q, t, tgt)
                self.launches = g.launches_per_step
            else:
                step = vpn_b200.PrimitiveLoss(cfg)
                vl, ql, tl = (x.clone().requires_grad_() for x in (v, q, t))
                ushape = (w["b"], w["k"], w["n"], 2)

                def fn():
                    u = None if w["vertex"] else torch.rand(ushape, device=v.device)
                    out = step(vl, ql, tl, u, tgt)
                    return torch.autograd.grad(out["total"], (vl, ql, tl))
                self.fn = fn
                for _ in range(3):
                    fn()
                torch.cuda.synchronize()
                n0 = lib.vpn_launch_count()
                fn()
                self.launches = int(lib.vpn_launch_count() - n0)
            self.picks_fork = None
            if variant != "no_emd":
                pts = torch.empty((w["b"], w["m"], 3), device=v.device)
                self.picks_fork = orig_fork(step_mod.PrimitiveLoss(cfg), pts)

    def time(self, steps, flush):
        with emd_placement(self.fork):
            return time_steps(self.fn, steps, flush)


def time_steps(fn, steps, flush):
    """Mean device ms of fn over `steps` calls, each after an L2 flush that is not timed."""
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
    for e0, e1 in ev:
        flush.zero_()
        e0.record()
        fn()
        e1.record()
    torch.cuda.synchronize()
    return sum(e0.elapsed_time(e1) for e0, e1 in ev) / steps


def auction_ms(x1, x2, flush, seconds):
    """The auction alone (vpn_b200.emd_auction forward at eps 0.005, 50 iterations): its time depends on the clouds,
    through the number of iterations until every point is assigned."""
    fn = lambda: vpn_b200.emd_auction(x1, x2, 0.005, 50)
    time_steps(fn, 3, flush)
    per = time_steps(fn, 5, flush)
    return round(time_steps(fn, max(20, math.ceil(seconds * 1e3 / per)), flush), 4)


def card():
    props = torch.cuda.get_device_properties(torch.cuda.current_device())
    info = {"torch_name": props.name, "sm_count": props.multi_processor_count}
    try:
        rows = subprocess.run(["nvidia-smi", "--query-gpu=pci.bus_id,name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                              capture_output=True, text=True, timeout=60).stdout.strip().splitlines()
    except (OSError, subprocess.SubprocessError) as e:
        return dict(info, nvidia_smi_error=str(e))
    bus = getattr(props, "pci_bus_id", None)
    dev = getattr(props, "pci_device_id", None)
    mine = [r for r in rows if bus is not None and dev is not None and f"{bus:02X}:{dev:02X}.0" in r.split(",")[0].upper()]
    if mine:
        _, name, power, clock = (x.strip() for x in mine[0].split(","))
        info.update(name=name, power_limit=power, max_sm_clock=clock)
    else:
        info["nvidia_smi_rows"] = rows
    return info


def main():
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("--workloads", default=",".join(WORKLOADS), help="comma-separated subset of " + ", ".join(WORKLOADS))
    ap.add_argument("--rounds", type=int, default=3, help="rounds; each times every variant once, in turn")
    ap.add_argument("--seconds", type=float, default=1.5, help="device time per variant per round")
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--out", default=None, help="JSON file to write (default: print only)")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("bench_step_emd.py measures on the GPU and found none")
    dev = torch.device("cuda:0")
    torch.cuda.set_device(dev)
    torch.manual_seed(0)
    flush = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device=dev)
    result = {"card": card(), "l2": "256 MB write before every step, outside the timed interval",
              "timing": f"CUDA events around each step; median over {args.rounds} rounds of >= {args.seconds} s per variant, "
                        "variants alternated within a round", "workloads": {}}
    for name in args.workloads.split(","):
        w = WORKLOADS[name]
        data = inputs(w, dev)
        res = {"shape": w}
        v, q, t, tgt = data
        with torch.no_grad():
            u = None if w["vertex"] else torch.rand((w["b"], w["k"], w["n"], 2), device=dev)
            pts = vpn_b200.PrimitiveLoss(config(w, "no_emd"))(v, q, t, u, tgt)["points"].contiguous()
        res["auction_only_ms"] = {"step_points_vs_targets": auction_ms(pts, tgt, flush, args.seconds),
                                  "uniform_clouds": auction_ms(torch.rand_like(tgt), torch.rand_like(tgt), flush, args.seconds)}
        print(json.dumps({name: res}), flush=True)
        for graphed in (True, False):
            mode = "graphed" if graphed else "eager"
            runners = {v: Runner(w, v, graphed, data) for v in VARIANTS}
            steps = {}
            for v, r in runners.items():
                r.time(args.warmup, flush)
                per = r.time(20, flush)
                steps[v] = max(50, math.ceil(args.seconds * 1e3 / per))
            ms = {v: [] for v in VARIANTS}
            for _ in range(args.rounds):
                for v, r in runners.items():
                    ms[v].append(r.time(steps[v], flush))
            med = {v: statistics.median(x) for v, x in ms.items()}
            best = min(("inline", "forked"), key=lambda v: med[v])
            res[mode] = {
                "ms_per_step": {v: round(med[v], 4) for v in VARIANTS},
                "ms_per_step_rounds": {v: [round(x, 4) for x in ms[v]] for v in VARIANTS},
                "steps_per_round": steps,
                "launches_per_step": {v: runners[v].launches for v in VARIANTS},
                "emd_ms": {v: round(med[v] - med["no_emd"], 4) for v in ("inline", "forked")},
                "emd_share": {v: round((med[v] - med["no_emd"]) / med[v], 4) for v in ("inline", "forked")},
                "faster": best,
                "forked_saves_ms": round(med["inline"] - med["forked"], 4),
                "step_picks": "forked" if runners["inline"].picks_fork else "inline",
            }
            print(json.dumps({name: {mode: res[mode]}}), flush=True)
            del runners
            torch.cuda.synchronize()
        result["workloads"][name] = res
    text = json.dumps(result, indent=1)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as fh:
            fh.write(text + "\n")
    print(text)


if __name__ == "__main__":
    main()
