"""Stage times of the Chamfer forward (vpn_b200.chamfer_nn_stage_ms: main, fallback, rows, cols, total, in ms) at the
C2, C3 and C5 shapes of bench.py, over several repetitions, with their spread.  `total - main` is the exact recovery the
step waits for after the filter.  Prints one JSON line.  Run on the GPU:

    python tools/bench_recovery.py [--reps 7] [--workloads c2,c3,c5]
"""
import argparse
import json
import os
import subprocess
import sys

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(REPO, "volumetric-primitives-net_b200")); sys.path.insert(0, REPO)

import torch  # noqa: E402
import vpn_b200  # noqa: E402
from bench import synthetic, WORKLOADS, VERTEX_MODE  # noqa: E402


def chamfer_inputs(wl, dev):
    kind, b, k, n, m, res = WORKLOADS[wl]
    torch.manual_seed(0)
    s = {kk: (vv.to(dev) if vv is not None else None) for kk, vv in synthetic(wl, "cpu")[0].items()}
    if wl in VERTEX_MODE:
        from vpn_b200 import templates as _tpl
        pts = vpn_b200.mesh_vertices(_tpl.template(kind, dev)[0], s["v"], s["q"], s["t"])
    else:
        pts = vpn_b200.sample_primitives(kind, s["v"], s["q"], s["t"],
                                         torch.rand((b, k, n, 2 if kind == "sphere" else 3), device=dev))
    return pts.contiguous(), s["target"].contiguous()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=7, help="repetitions, each the mean of --inner forwards")
    ap.add_argument("--inner", type=int, default=20)
    ap.add_argument("--workloads", default="c2,c3,c5")
    args = ap.parse_args()
    dev = torch.device("cuda")
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()
    out = {"gpu": smi[0] if smi else torch.cuda.get_device_name(dev), "reps": args.reps, "inner": args.inner, "workloads": {}}
    for wl in args.workloads.split(","):
        p1, p2 = chamfer_inputs(wl, dev)
        vpn_b200.chamfer_nn_stage_ms(p1, p2, reps=3)
        runs = []
        for _ in range(args.reps):
            st = vpn_b200.chamfer_nn_stage_ms(p1, p2, reps=args.inner)
            runs.append({k: st[k] for k in ("main", "fallback", "rows", "cols", "total")})
        res = {"shape": {"B": p1.shape[0], "P": p1.shape[1], "M": p2.shape[1]}}
        for key in ("main", "rows", "cols", "total", "recovery"):
            v = sorted((r["total"] - r["main"]) if key == "recovery" else r[key] for r in runs)
            res[key] = {"median": v[len(v) // 2], "min": v[0], "max": v[-1]}
        out["workloads"][wl] = res
    print(json.dumps(out), flush=True)


if __name__ == "__main__":
    main()
