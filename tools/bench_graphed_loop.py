"""What the training-loop features of the graphed primitive step cost: per-term losses read back through HostPipeline,
the replay of a short last batch, and the lazy capture of its graph.

    a   train.py defaults: B = 8, 16 spheres x 128 samples, M = 2048, l_vp_div = 0.1, l_emd = 1.0
    c2  C2 size: B = 32, 16 cuboids x 4096 samples, M = 8192, l_vp_div = 0.1

Per workload:
    pipe / pipe_terms   GraphedPrimitiveLoss through HostPipeline from pinned host batches, returning (loss, gv, gq, gt),
                        or that plus g.terms: the difference is the per-step cost of reading the terms back.  The 256 MB
                        L2 flush is HostPipeline's pre_step, inside the loop; host clock over the loop, first submit to
                        last result, divided by the steps (the method of tools/bench_mesh_step.py's e2e form).
    full / short        the replay at B and at b = B - 3 on device inputs: CUDA events around each step, 256 MB L2 flush
                        before every step outside the timed interval.
Forms alternate within a round; the median over rounds is reported.  Then, on fresh step objects, the host clock around
the first call at b = B - 3 (warm-up steps + capture + replay, ending in a synchronise), and torch.cuda.memory_reserved()
before and after that call (and after empty_cache, which leaves what the graphs hold), next to the same numbers for the
construction (the full-size capture).  The card's name and power limit are read in the same run.  Writes one JSON file
(--out)."""
import argparse
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

import torch  # noqa: E402

import vpn_b200  # noqa: E402
from bench_step_emd import card, time_steps  # noqa: E402

WORKLOADS = {
    "a_train_b8": dict(b=8, kind="sphere", k=16, n=128, m=2048, l_emd=1.0),
    "c2_b32": dict(b=32, kind="cuboid", k=16, n=4096, m=8192, l_emd=0.0),
}
FORMS = ("pipe", "pipe_terms", "full", "short")
SHORT = 3                      # b = B - SHORT


def config(w):
    return vpn_b200.PrimitiveLossConfig(kind=w["kind"], l_vp_div=0.1, l_emd=w["l_emd"])


def inputs(w, b, dev, seed):
    from oracle import vpn_oracle as O
    g = torch.Generator().manual_seed(seed)
    v, q, t = O.synthetic_primitives(b, w["k"], seed=seed)
    tgt = (torch.rand(b, w["m"], 3, generator=g) - 0.5) * 0.8
    return {"v": v.to(dev), "q": q.to(dev), "t": (t * 0.3).to(dev), "target": tgt.to(dev)}


def graphed(w, d):
    return vpn_b200.GraphedPrimitiveLoss(config(w), d["v"], d["q"], d["t"], d["target"], None, n_samples=w["n"])


def pipe_runner(g, pinned, flush, terms):
    fn = ((lambda s: (*g(s["v"], s["q"], s["t"], s["target"]), *g.terms.values())) if terms
          else (lambda s: g(s["v"], s["q"], s["t"], s["target"])))
    pipe = vpn_b200.HostPipeline(fn, pinned[0], "cuda", pre_step=flush.zero_)

    def run(steps):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        pipe.submit(pinned[0])
        for i in range(1, steps):
            pipe.submit(pinned[i % len(pinned)])
            pipe.result()
        pipe.result()
        torch.cuda.synchronize()
        return (time.perf_counter() - t0) * 1e3 / steps
    return run


def lazy_capture(w, d_full, d_short, rounds):
    """Host ms of the first short call on a fresh object, and memory_reserved around it and around the construction."""
    res = []
    for _ in range(rounds):
        torch.cuda.synchronize()
        torch.cuda.empty_cache()
        m0 = torch.cuda.memory_reserved()
        g = graphed(w, d_full)
        torch.cuda.synchronize()
        m1 = torch.cuda.memory_reserved()
        torch.cuda.empty_cache()
        m1e = torch.cuda.memory_reserved()
        t0 = time.perf_counter()
        g(d_short["v"], d_short["q"], d_short["t"], d_short["target"])
        torch.cuda.synchronize()
        ms = (time.perf_counter() - t0) * 1e3
        m2 = torch.cuda.memory_reserved()
        torch.cuda.empty_cache()
        m2e = torch.cuda.memory_reserved()
        t0 = time.perf_counter()
        g(d_short["v"], d_short["q"], d_short["t"], d_short["target"])
        torch.cuda.synchronize()
        again = (time.perf_counter() - t0) * 1e3
        mb = lambda x: round(x / 2**20, 1)
        res.append({"first_short_call_ms": round(ms, 2), "second_short_call_ms": round(again, 3),
                    "reserved_mb": {"before_construction": mb(m0), "after_construction": mb(m1),
                                    "after_construction_empty_cache": mb(m1e), "after_first_short_call": mb(m2),
                                    "after_first_short_call_empty_cache": mb(m2e)}})
        del g
    return {"rounds": res, "first_short_call_ms_median": statistics.median(r["first_short_call_ms"] for r in res)}


def main():
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("--workloads", default=",".join(WORKLOADS), help="comma-separated subset of " + ", ".join(WORKLOADS))
    ap.add_argument("--rounds", type=int, default=3, help="rounds; each times every form once, in turn")
    ap.add_argument("--seconds", type=float, default=1.5, help="time per form per round")
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--out", default=None, help="JSON file to write (default: print only)")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("bench_graphed_loop.py measures on the GPU and found none")
    dev = torch.device("cuda:0")
    torch.cuda.set_device(dev)
    torch.manual_seed(0)
    flush = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device=dev)
    result = {"card": card(), "short_batch": f"B - {SHORT}",
              "timing": f"median over {args.rounds} rounds of >= {args.seconds} s per form, forms alternated within a "
                        "round; full / short: CUDA events per step, 256 MB L2 flush before every step outside the timed "
                        "interval; pipe / pipe_terms: host clock over the HostPipeline loop, the flush its pre_step",
              "workloads": {}}
    for name in args.workloads.split(","):
        w = WORKLOADS[name]
        b, bs = w["b"], w["b"] - SHORT
        d_full, d_short = inputs(w, b, dev, 1), inputs(w, bs, dev, 2)
        pinned = [{k: x.cpu().pin_memory() for k, x in inputs(w, b, "cpu", 10 + i).items()} for i in range(2)]
        lazy = lazy_capture(w, d_full, d_short, args.rounds)
        g = graphed(w, d_full)
        g(d_short["v"], d_short["q"], d_short["t"], d_short["target"])          # capture the short graph
        runners = {
            "pipe": pipe_runner(g, pinned, flush, False),
            "pipe_terms": pipe_runner(g, pinned, flush, True),
            "full": lambda steps: time_steps(lambda: g(d_full["v"], d_full["q"], d_full["t"], d_full["target"]), steps, flush),
            "short": lambda steps: time_steps(lambda: g(d_short["v"], d_short["q"], d_short["t"], d_short["target"]), steps,
                                              flush),
        }
        steps = {}
        for f, run in runners.items():
            run(args.warmup)
            steps[f] = max(50, math.ceil(args.seconds * 1e3 / run(20)))
        ms = {f: [] for f in FORMS}
        for _ in range(args.rounds):
            for f, run in runners.items():
                ms[f].append(run(steps[f]))
        med = {f: statistics.median(x) for f, x in ms.items()}
        res = {"shape": dict(w, b_short=bs), "terms": list(g.terms), "launches_per_step": g.launches_per_step,
               "launches_per_short_step": g._graphs[bs].launches,
               "ms_per_step": {f: round(med[f], 4) for f in FORMS},
               "ms_per_step_rounds": {f: [round(x, 4) for x in ms[f]] for f in FORMS}, "steps_per_round": steps,
               "terms_readback_ms": round(med["pipe_terms"] - med["pipe"], 4),
               "short_over_full": round(med["short"] / med["full"], 3), "lazy_capture": lazy}
        print(json.dumps({name: res}), flush=True)
        result["workloads"][name] = res
        del runners, g
        torch.cuda.synchronize()
    text = json.dumps(result, indent=1)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as fh:
            fh.write(text + "\n")
    print(text)


if __name__ == "__main__":
    main()
