"""CPU side of test_gpu_raster_edges.py: the premises of its scenes, checked with the oracle's own selection logic (each
scene really exercises what its GPU test is for), the oracle's knum and non-finite-face rules, and the rasteriser's C ABI
argument checks, which reject knum outside [1, 32] and F > 65535 before any CUDA call."""
import os
import subprocess

import pytest
import torch

import test_gpu_raster_edges as T
from oracle import vpn_oracle as O

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PKG = os.path.join(REPO, "volumetric-primitives-net_b200")


@pytest.mark.parametrize("h,w,kind", T.RAGGED, ids=[f"{h}x{w}-{k}" for h, w, k in T.RAGGED])
def test_ragged_scene_reaches_partial_tiles(h, w, kind):
    verts, faces = T.spot_scene(kind)
    rot, pos = T.default_camera(2)
    pixels = T.ragged_pixels(h, w) if (h, w) == (137, 137) else None
    T.ragged_premise(O.soft_silhouette(verts, faces, rot, pos, h, w, pixels=pixels), h, w, pixels)


@pytest.mark.parametrize("cull", [False, True])
@pytest.mark.parametrize("reverse", [False, True])
def test_knum_scene_premise(reverse, cull):
    T.knum_premise(O, reverse, cull)


def test_wide_scene_premise():
    T.wide_premise(O)


@pytest.mark.parametrize("mode", ["nan", "plane"])
def test_poison_scene_premise(mode):
    T.poison_premise(O, mode)


def test_cases_scene_premise():
    T.cases_premise(O)


def test_oracle_knum_keyword():
    """knum = 30 is the default; fewer candidates give a smaller alpha on the fan pixels."""
    verts, faces = T.knum_scene()
    rot, pos = T.default_camera(1)
    h, w = T.KNUM_HW
    a30 = O.soft_silhouette(verts, faces, rot, pos, h, w)
    assert torch.equal(a30, O.soft_silhouette(verts, faces, rot, pos, h, w, knum=30))
    fan = torch.tensor([hh * w + ww for hh, ww in T.KNUM_PIXELS])
    prev = torch.zeros(fan.numel())
    for knum in (1, 7, 30, 32):
        a = O.soft_silhouette(verts, faces, rot, pos, h, w, knum=knum).flatten()[fan]
        assert (a > prev).all()
        prev = a


@pytest.mark.parametrize("mode", ["nan", "plane"])
def test_oracle_skips_nonfinite_faces(mode):
    """A face with a non-finite screen coordinate is in neither pass: the poisoned sample renders as the same mesh
    without those faces (to the rounding of the longer product), and every other vertex's gradient is finite."""
    verts, faces, j = T.poison_scene(mode)
    rot, pos = T.default_camera(3)
    h, w = T.POISON_HW
    v = verts[1:2].clone().requires_grad_()
    a = O.soft_silhouette(v, faces, rot[1:2], pos[1:2], h, w)
    keep = ~(faces == j).any(1)
    b = O.soft_silhouette(verts[1:2], faces[keep], rot[1:2], pos[1:2], h, w)
    assert torch.isfinite(a).all()
    torch.testing.assert_close(a, b, rtol=1e-6, atol=1e-7)
    a.sum().backward()
    others = torch.ones(verts.shape[1], dtype=torch.bool)
    others[j] = False
    assert torch.isfinite(v.grad[0, others]).all() and v.grad[0, others].abs().sum() > 0


@pytest.fixture(scope="module")
def lib():
    if not os.path.isfile(os.path.join(PKG, "lib", "libvpn_b200.so")):
        subprocess.check_call(["make", "-C", os.path.join(PKG, "csrc"), "-j8"])
    from vpn_b200 import _lib
    return _lib.load()


def _fwd_bwd_rc(lib, knum, f):
    """Return codes of vpn_silhouette_fwd / _bwd for an empty batch (B = 0, NULL buffers): the argument checks run,
    then an empty batch returns VPN_OK without touching the device."""
    fwd = lib.vpn_silhouette_fwd(None, None, None, None, 1.0, 1.0, -1.0, 0.02, knum, 1000.0, 7000.0, 0, None, None, None,
                                 None, 0, 0, 3, f, 16, 16, None)
    bwd = lib.vpn_silhouette_bwd(None, None, 1.0, 1.0, -1.0, 0.02, knum, 1000.0, 7000.0, 0, None, None, None, None, 0,
                                 0, 3, f, 16, 16, None)
    return fwd, bwd


def test_abi_rejects_knum_and_face_count(lib):
    for knum in (0, 33, -1):
        assert _fwd_bwd_rc(lib, knum, 1) == (T.VPN_ERR_ARG, T.VPN_ERR_ARG), knum
    assert _fwd_bwd_rc(lib, 30, 65536) == (T.VPN_ERR_SHAPE, T.VPN_ERR_SHAPE)
    assert b"65535" in lib.vpn_last_error_string()
    for knum, f in ((1, 1), (32, 65535)):
        assert _fwd_bwd_rc(lib, knum, f) == (0, 0), (knum, f)
