"""CPU-side checks of MeshLoss: the shape preconditions raise AssertionError from the shapes alone, before any kernel is
called.  The tensors are CPU tensors, so a call that got as far as a kernel would raise VpnError (no CPU path) instead;
the well-formed cases show that it does."""
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


def mesh(b, v=12):
    faces = torch.tensor([[0, 1, 2], [2, 3, 0], [4, 5, 6], [8, 9, 11]], dtype=torch.int32)
    return torch.rand(b, v, 3), faces


@pytest.mark.parametrize("n,m", [(64, 63), (64, 65), (0, 11), (0, 13)])
def test_emd_needs_as_many_points_as_targets(vpn, n, m):
    b = 2
    verts, faces = mesh(b)
    step = vpn.MeshLoss(vpn.MeshLossConfig(n_samples=n, l_emd=1.0))
    with pytest.raises(AssertionError, match="as many points as targets"):
        step(verts, faces, torch.rand(b, m, 3))
    with pytest.raises(AssertionError, match="as many points as targets"):
        step(verts, faces, torch.rand(b + 1, n or verts.shape[1], 3))            # batch sizes differ
    with pytest.raises(vpn.VpnError):                                            # P == M: on to the first kernel
        step(verts, faces, torch.rand(b, n or verts.shape[1], 3))


def test_vertex_path_takes_no_uniforms(vpn):
    b = 2
    verts, faces = mesh(b)
    step = vpn.MeshLoss(vpn.MeshLossConfig(n_samples=0))
    with pytest.raises(AssertionError, match="n_samples = 0"):
        step(verts, faces, torch.rand(b, 20, 3), uniforms=torch.rand(b, 8, 3))
    with pytest.raises(vpn.VpnError):
        step(verts, faces, torch.rand(b, 20, 3))


def test_uniforms_shape_is_checked(vpn):
    b = 2
    verts, faces = mesh(b)
    step = vpn.MeshLoss(vpn.MeshLossConfig(n_samples=16))
    with pytest.raises(AssertionError, match="uniforms must be"):
        step(verts, faces, torch.rand(b, 20, 3), uniforms=torch.rand(b, 15, 3))
    with pytest.raises(vpn.VpnError):
        step(verts, faces, torch.rand(b, 20, 3), uniforms=torch.rand(b, 16, 3))


def test_defaults(vpn):
    cfg = vpn.MeshLossConfig()
    assert (cfg.n_samples, cfg.l_cd, cfg.l_sil, cfg.l_emd, cfg.emd_eps, cfg.emd_iters) == (2048, 1.0, 0.0, 0.0, 0.005, 50)
