"""TEST INFRASTRUCTURE.  Writes tests/golden/emd_golden.npz, what tests/test_gpu_emd_reference.py compares the EMD kernels with.

The reference's own EMD kernels (oracle/_ref/libemd_ref.so) need the reference's source tree to build; the suite must run
without it.  So the values the tests compare with are frozen here, on the tests' own seeded clouds, from
oracle.emd_auction / oracle.emd_backward: the deterministic restatement that vpn_emd_fwd / vpn_emd_bwd reproduce bit for
bit (tests/test_gpu_parity.py) and whose results were measured against the reference's kernels with the tolerances the
tests keep (batch-mean EMD within 0.1-0.6 %, DESIGN.md section 2).  Runs on the CPU in about a minute:

    python -m oracle.make_emd_golden
"""
import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
REPO = os.path.dirname(HERE)
sys.path[:0] = [REPO, os.path.join(REPO, "tests")]

from oracle import vpn_oracle as O                                       # noqa: E402
from test_gpu_emd_reference import BACKWARD, CASES, NEAR_OPTIMAL, case_key, clouds, seeded_clouds   # noqa: E402

OUT = os.path.join(REPO, "tests", "golden", "emd_golden.npz")


def auction(x1, x2, eps, iters):
    out = [O.emd_auction(x1[i].numpy(), x2[i].numpy(), eps, iters) for i in range(x1.shape[0])]
    return np.stack([d for d, _ in out]), np.stack([a for _, a in out])


def main():
    d = {}
    for kind, b, n, eps, iters, _ in CASES:
        key = case_key(kind, b, n, eps, iters)
        x1, x2 = seeded_clouds(kind, b, n, iters)
        dist, ass = auction(x1, x2, eps, iters)
        d[key + "_head"] = x1[:, :4].numpy()
        d[key + "_emd"] = np.sqrt(dist).mean(1).astype(np.float32)                       # per sample, what train.py:194 averages
        d[key + "_uniq"] = np.array([np.unique(a).size for a in ass], np.float64) / n     # distinct assigned objects
    kind, b, n, seed = NEAR_OPTIMAL
    x1, x2 = clouds(kind, b, n, torch.Generator().manual_seed(seed))
    dist, _ = auction(x1, x2, 0.005, 50)
    d["near_optimal_head"] = x1[:, :4].numpy()
    d["near_optimal_emd"] = np.sqrt(dist).mean(1).astype(np.float32)
    kind, b, n, seed = BACKWARD
    gen = torch.Generator().manual_seed(seed)
    x1, x2 = clouds(kind, b, n, gen)
    _, ass = auction(x1, x2, 0.005, 50)
    up = torch.rand(b, n, generator=gen).numpy()
    d["backward_head"] = x1[:, :4].numpy()
    d["backward_assignment"] = ass.astype(np.int32)
    d["backward_grad"] = np.stack([O.emd_backward(x1[i].numpy(), x2[i].numpy(), ass[i], up[i]) for i in range(b)])
    np.savez_compressed(OUT, **d)
    print(f"make_emd_golden: wrote {OUT} ({os.path.getsize(OUT)} bytes)")


if __name__ == "__main__":
    main()
