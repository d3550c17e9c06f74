"""vpn_emd_fwd / vpn_emd_bwd against the reference's EMD auction (modules/loss/emd/emd_cuda.cu:23-226, :284-300).

The reference auction is racy by construction (GetMax / Assign, emd_cuda.cu:181-215: among bidders within 1e-6 of an
object's maximum increment the last writer wins; calc_unass_idx orders the unassigned list with atomics); this kernel
resolves the races deterministically (lowest index), so parity is STATISTICAL, at the training setting of
train.py:188-195 (eps 0.005, 50 iterations) and train_gcn.py:91-95:
  * mean sqrt(dist) - the EMD loss value the training loop uses - within 1 % of the reference's over the batch;
  * the share of distinct assigned objects (how far the assignment is from a bijection) within 1 % absolute;
  * both at or above the exact optimum (scipy) and within the same bound above it;
  * the backward kernel, which is deterministic given the assignment, equal to 1e-6.
The reference's kernels need its source tree to build (oracle/build_ref_emd.sh -> oracle/_ref/libemd_ref.so), which is
not part of this repository.  The values compared with are therefore frozen in tests/golden/emd_golden.npz
(oracle/make_emd_golden.py), on these tests' seeded clouds: the results of the deterministic auction that was measured
against the reference's kernels with these tolerances (batch means 0.1-0.6 % apart, DESIGN.md section 2).  They pin the
kernel independently of oracle.emd_auction, which test_gpu_parity.py matches bit for bit.
test_reference_emd_run_to_run_spread measures the reference's own kernels and skips where they are not built.
"""
import ctypes
import os

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REF_SO = os.path.join(REPO, "oracle", "_ref", "libemd_ref.so")

CASES = [
    # kind, b, n, eps, iters, per-sample tolerance
    ("uniform", 32, 2048, 0.005, 50, 0.03),          # train.py:188-195 / train_gcn.py:91-95 setting, B = 32
    ("surface", 32, 2048, 0.005, 50, 0.03),
    # degenerate start of training (every prediction within 0.05 of the centre: all bidders want the same objects and the
    # 50 iterations end far from convergence).  The reference moves by up to 3 % between two runs on the SAME sample
    # here; single samples of this kernel land up to 6 % from the reference's mean, the batch mean within 1 %.
    ("clustered", 8, 2048, 0.005, 50, 0.08),
    ("uniform", 4, 1024, 0.002, 100, 0.03),
    ("uniform", 2, 8192, 0.05, 30, 0.03),            # emd_module.py:81-86 smoke shape (shorter)
]
NEAR_OPTIMAL = ("uniform", 2, 1024, 11)              # kind, b, n, seed
BACKWARD = ("surface", 3, 2048, 3)


def case_key(kind, b, n, eps, iters):
    return f"{kind}_{b}_{n}_{eps}_{iters}"


@pytest.fixture(scope="module")
def golden_emd():
    return dict(np.load(os.path.join(REPO, "tests", "golden", "emd_golden.npz")))


def check_head(golden_emd, key, x1):
    """The seeded clouds are the ones the golden values were computed on."""
    np.testing.assert_array_equal(x1[:, :4].cpu().numpy(), golden_emd[key + "_head"])


@pytest.fixture(scope="module")
def ref_emd_binary():
    """forward of the reference's own kernels (oracle/_ref/libemd_ref.so), built only where the reference's source is."""
    if not os.path.isfile(REF_SO):
        pytest.skip("oracle/_ref/libemd_ref.so not built: run `make -C oracle` with VPN_REFERENCE_ROOT set to the "
                    "reference's source tree")
    lib = ctypes.CDLL(REF_SO)
    lib.ref_emd_workspace_bytes.restype = ctypes.c_size_t
    lib.ref_emd_workspace_bytes.argtypes = [ctypes.c_int, ctypes.c_int]
    lib.ref_emd_forward.restype = ctypes.c_int
    lib.ref_emd_forward.argtypes = [ctypes.c_void_p] * 5 + [ctypes.c_int, ctypes.c_int, ctypes.c_float, ctypes.c_int]

    def forward(x1, x2, eps, iters):
        b, n, _ = x1.shape
        dist = torch.empty(b, n, device="cuda")
        ass = torch.empty(b, n, dtype=torch.int32, device="cuda")
        ws = torch.empty(lib.ref_emd_workspace_bytes(b, n), dtype=torch.uint8, device="cuda")
        torch.cuda.synchronize()
        rc = lib.ref_emd_forward(x1.data_ptr(), x2.data_ptr(), dist.data_ptr(), ass.data_ptr(), ws.data_ptr(), b, n, eps, iters)
        assert rc == 1, f"reference emd_cuda_forward status {rc}"
        return dist, ass

    return forward


def clouds(kind, b, n, gen):
    """xyz1 = predicted, xyz2 = ground truth, normalised to [0, 1] as emd_module.py:8 requires."""
    if kind == "uniform":
        return torch.rand(b, n, 3, generator=gen), torch.rand(b, n, 3, generator=gen)
    if kind == "surface":                     # points on a box surface vs a noisy, shifted copy: what training sees late
        p = torch.rand(b, n, 3, generator=gen)
        axis = torch.randint(0, 3, (b, n), generator=gen)
        side = torch.randint(0, 2, (b, n), generator=gen).float()
        p.scatter_(2, axis[..., None], side[..., None])
        p = 0.25 + 0.5 * p
        perm = torch.stack([torch.randperm(n, generator=gen) for _ in range(b)])
        q = torch.gather(p, 1, perm[..., None].expand(-1, -1, 3)) + 0.02 * torch.randn(b, n, 3, generator=gen)
        return q.clamp(0, 1), p
    if kind == "clustered":                   # early training: predictions collapsed near the centre, targets spread out
        return 0.5 + 0.05 * torch.randn(b, n, 3, generator=gen), torch.rand(b, n, 3, generator=gen)
    raise KeyError(kind)


def seeded_clouds(kind, b, n, iters):
    return clouds(kind, b, n, torch.Generator().manual_seed(4242 + n + iters))


@pytest.mark.parametrize("kind,b,n,eps,iters,per_sample", CASES)
def test_emd_matches_reference_kernels(golden_emd, kind, b, n, eps, iters, per_sample):
    import vpn_b200
    key = case_key(kind, b, n, eps, iters)
    x1, x2 = (t.cuda().contiguous() for t in seeded_clouds(kind, b, n, iters))
    check_head(golden_emd, key, x1)
    d_our, a_our = vpn_b200.emd_auction(x1, x2, eps, iters)
    torch.cuda.synchronize()
    # the assignment indexes valid objects and dist is the squared distance to it
    assert int(a_our.min()) >= 0 and int(a_our.max()) < n
    chk = ((x1 - torch.gather(x2, 1, a_our.long()[..., None].expand(-1, -1, 3))) ** 2).sum(-1)
    np.testing.assert_allclose(d_our.cpu().numpy(), chk.cpu().numpy(), rtol=1e-5, atol=1e-9)
    emd_ref = golden_emd[key + "_emd"].astype(np.float64)
    emd_our = torch.sqrt(d_our).mean(1).double().cpu().numpy()
    # The loss value (mean over the batch): within 1 %.
    np.testing.assert_allclose(emd_our.mean(), emd_ref.mean(), rtol=0.01)
    # Single samples: within `per_sample` (3 % for the training-like clouds).  The auction's tie races, which the
    # reference leaves to the hardware, decide individual assignments.
    assert (np.abs(emd_our - emd_ref) <= per_sample * emd_ref).all(), (emd_our, emd_ref)
    uniq_ref = golden_emd[key + "_uniq"]
    uniq_our = np.array([a.unique().numel() for a in a_our]) / n
    assert abs(uniq_our.mean() - uniq_ref.mean()) <= 0.01, (uniq_our, uniq_ref)


def test_reference_emd_run_to_run_spread(ref_emd_binary):
    """How far the reference is from itself on identical input (documents the tolerance above): <= 1 % per sample."""
    fwd = ref_emd_binary
    gen = torch.Generator().manual_seed(7)
    x1, x2 = (t.cuda().contiguous() for t in clouds("uniform", 8, 2048, gen))
    runs = np.stack([torch.sqrt(fwd(x1, x2, 0.005, 50)[0]).mean(1).cpu().numpy() for _ in range(3)])
    assert (np.abs(runs - runs[0]) / runs[0]).max() <= 0.01


def test_emd_both_near_optimal(golden_emd):
    """Exact optimum by scipy on n = 1024: both auctions are >= it and within the same distance of it."""
    from scipy.optimize import linear_sum_assignment
    import vpn_b200
    kind, b, n, seed = NEAR_OPTIMAL
    x1, x2 = clouds(kind, b, n, torch.Generator().manual_seed(seed))
    check_head(golden_emd, "near_optimal", x1)
    d_our, a_our = vpn_b200.emd_auction(x1.cuda(), x2.cuda(), 0.005, 50)
    for i in range(b):
        cost = torch.cdist(x1[i].double(), x2[i].double()).numpy()
        r, c = linear_sum_assignment(cost)
        opt = cost[r, c].mean()
        e_ref = float(golden_emd["near_optimal_emd"][i]); e_our = float(torch.sqrt(d_our[i]).mean())
        # Upper bound: the auction's eps-optimality slack.  No tight lower bound exists: in the last iteration every still
        # unassigned bidder takes its favourite object (emd_cuda.cu:196-215, `last`), the result is not a bijection and
        # undercuts the bijective optimum (the reference lands ~13 % below it here) - both must undercut it alike.
        for e in (e_ref, e_our):
            assert 0.5 * opt <= e <= opt + 3 * 0.005 + 0.02 * opt, (e, opt)
        assert abs(e_our - e_ref) <= 0.02 * e_ref, (e_our, e_ref, opt)


def test_emd_backward_equals_reference_kernel(golden_emd):
    """NmDistanceGradKernel (emd_cuda.cu:284-300) on the same assignment: deterministic, equal to 1e-6."""
    from vpn_b200 import _lib
    from vpn_b200._lib import check, ptr, stream_ptr
    kind, b, n, seed = BACKWARD
    gen = torch.Generator().manual_seed(seed)
    x1, x2 = (t.cuda().contiguous() for t in clouds(kind, b, n, gen))
    check_head(golden_emd, "backward", x1)
    up = torch.rand(b, n, generator=gen).cuda()
    ass = torch.from_numpy(golden_emd["backward_assignment"]).cuda()
    g = torch.empty_like(x1)
    check(_lib.load().vpn_emd_bwd(ptr(x1), ptr(x2), ptr(ass), ptr(up), ptr(g), b, n, stream_ptr(x1.device)), "vpn_emd_bwd")
    torch.cuda.synchronize()
    np.testing.assert_allclose(g.cpu().numpy(), golden_emd["backward_grad"], rtol=1e-6, atol=1e-7)
