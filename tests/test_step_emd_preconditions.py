"""CPU-side checks of the EMD term of PrimitiveLoss: with l_emd != 0 the step refuses point / target clouds of different
sizes with AssertionError, from the shapes, before any kernel is called.  The tensors are CPU tensors, so a call that got
as far as a kernel would raise VpnError (no CPU path) instead; the matching-shape cases show that it does."""
import os
import subprocess

import pytest
import torch

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PKG = os.path.join(REPO, "volumetric-primitives-net_b200")


@pytest.fixture(scope="module")
def vpn():
    if not os.path.isfile(os.path.join(PKG, "lib", "libvpn_b200.so")):
        subprocess.check_call(["make", "-C", os.path.join(PKG, "csrc"), "-j8"])
    import vpn_b200
    return vpn_b200


def prims(b, k):
    return torch.ones(b, k, 3), torch.tensor([0.0, 0.0, 1.0, 0.1]).repeat(b, k, 1), torch.zeros(b, k, 3)


@pytest.mark.parametrize("m", [1000, 1025])
def test_emd_term_rejects_unequal_clouds_before_any_kernel(vpn, m):
    b, k, n = 2, 4, 256                                                  # P = 1024 sampled points
    v, q, t = prims(b, k)
    step = vpn.PrimitiveLoss(vpn.PrimitiveLossConfig(kind="sphere", l_emd=1.0))
    with pytest.raises(AssertionError, match="as many points as targets"):
        step(v, q, t, torch.rand(b, k, n, 2), torch.rand(b, m, 3))
    with pytest.raises(vpn.VpnError):                                    # P == M: on to the first kernel
        step(v, q, t, torch.rand(b, k, n, 2), torch.rand(b, k * n, 3))


def test_emd_term_vertex_path_rejects_unequal_clouds(vpn):
    from vpn_b200 import templates
    b, k = 2, 4
    nv = templates.template("sphere", "cpu")[0].shape[0]
    v, q, t = prims(b, k)
    step = vpn.PrimitiveLoss(vpn.PrimitiveLossConfig(kind="sphere", l_emd=1.0, vertex_chamfer=True))
    with pytest.raises(AssertionError, match="as many points as targets"):
        step(v, q, t, None, torch.rand(b, k * nv + 1, 3))
    with pytest.raises(AssertionError, match="as many points as targets"):
        step(v, q, t, None, torch.rand(b + 1, k * nv, 3))                 # batch sizes differ
    with pytest.raises(vpn.VpnError):
        step(v, q, t, None, torch.rand(b, k * nv, 3))


def test_emd_term_is_off_by_default(vpn):
    """l_emd defaults to 0: existing callers keep their loss, and unequal clouds stay legal without the EMD term."""
    assert vpn.PrimitiveLossConfig().l_emd == 0.0
    b, k = 1, 2
    v, q, t = prims(b, k)
    with pytest.raises(vpn.VpnError):
        vpn.PrimitiveLoss()(v, q, t, torch.rand(b, k, 8, 2), torch.rand(b, 100, 3))
