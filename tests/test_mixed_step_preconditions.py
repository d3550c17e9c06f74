"""CPU-side checks of mixed cuboid + sphere assemblies: the config, shape and argument preconditions of
PrimitiveLoss(kind="mixed"), ops.sample_mixed_primitives / mesh_vertices_mixed and the vpn_pose_mixed_* C entry points
fail before any kernel is called.  The tensors are CPU tensors, so a call that got as far as a kernel would raise
VpnError (no CPU path) instead; the well-formed cases show that it does."""
import ctypes
import os
import subprocess

import pytest
import torch

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PKG = os.path.join(REPO, "volumetric-primitives-net_b200")
VPN_ERR_SHAPE, VPN_ERR_ARG, VPN_ERR_WORKSPACE = -2, -3, -4


@pytest.fixture(scope="module")
def vpn():
    if not os.path.isfile(os.path.join(PKG, "lib", "libvpn_b200.so")):
        subprocess.check_call(["make", "-C", os.path.join(PKG, "csrc"), "-j8"])
    import vpn_b200
    return vpn_b200


def prims(b, k):
    return torch.ones(b, k, 3), torch.tensor([0.0, 0.0, 1.0, 0.1]).repeat(b, k, 1), torch.zeros(b, k, 3)


def test_defaults_unchanged(vpn):
    cfg = vpn.PrimitiveLossConfig()
    assert (cfg.kind, cfg.n_cuboids) == ("sphere", 0)


def test_config_rejects_n_cuboids_with_a_single_kind(vpn):
    for kind in ("sphere", "cuboid"):
        with pytest.raises(AssertionError, match="kind='mixed' only"):
            vpn.PrimitiveLossConfig(kind=kind, n_cuboids=2)
    with pytest.raises(AssertionError):
        vpn.PrimitiveLossConfig(kind="cone")
    with pytest.raises(AssertionError):
        vpn.PrimitiveLossConfig(kind="mixed", n_cuboids=-1)
    vpn.PrimitiveLossConfig(kind="mixed", n_cuboids=3)


@pytest.mark.parametrize("vertex", [False, True])
def test_n_cuboids_above_k_is_rejected(vpn, vertex):
    b, k, n = 2, 4, 16
    v, q, t = prims(b, k)
    step = vpn.PrimitiveLoss(vpn.PrimitiveLossConfig(kind="mixed", n_cuboids=k + 1, vertex_chamfer=vertex))
    u = None if vertex else (torch.rand(b, k + 1, n, 3), torch.rand(b, 0, n, 2))
    with pytest.raises(AssertionError, match="exceeds"):
        step(v, q, t, u, torch.rand(b, 64, 3))
    with pytest.raises(AssertionError, match="n_cuboids must be in"):
        vpn.sample_mixed_primitives(k + 1, v, q, t, torch.rand(b, k + 1, n, 3), torch.rand(b, 0, n, 2))


@pytest.mark.parametrize("case", ["n_mismatch", "sphere_width_3", "cuboid_width_2", "kc_mismatch", "not_a_pair"])
def test_wrong_uniform_shapes_are_rejected(vpn, case):
    b, k, kc, n = 2, 5, 2, 16
    v, q, t = prims(b, k)
    uc, us = {"n_mismatch": (torch.rand(b, kc, n, 3), torch.rand(b, k - kc, n + 4, 2)),
              "sphere_width_3": (torch.rand(b, kc, n, 3), torch.rand(b, k - kc, n, 3)),
              "cuboid_width_2": (torch.rand(b, kc, n, 2), torch.rand(b, k - kc, n, 2)),
              "kc_mismatch": (torch.rand(b, kc + 1, n, 3), torch.rand(b, k - kc - 1, n, 2)),
              "not_a_pair": (None, None)}[case]
    step = vpn.PrimitiveLoss(vpn.PrimitiveLossConfig(kind="mixed", n_cuboids=kc))
    u = torch.rand(b, k, n, 2) if case == "not_a_pair" else (uc, us)
    with pytest.raises(AssertionError):
        step(v, q, t, u, torch.rand(b, 64, 3))
    if case != "not_a_pair":
        with pytest.raises(AssertionError):
            vpn.sample_mixed_primitives(kc, v, q, t, uc, us)


@pytest.mark.parametrize("kc", [0, 2, 5])
def test_valid_shapes_reach_the_kernel(vpn, kc):
    b, k, n = 2, 5, 16
    v, q, t = prims(b, k)
    u = (torch.rand(b, kc, n, 3), torch.rand(b, k - kc, n, 2))
    with pytest.raises(vpn.VpnError):
        vpn.PrimitiveLoss(vpn.PrimitiveLossConfig(kind="mixed", n_cuboids=kc))(v, q, t, u, torch.rand(b, 64, 3))
    with pytest.raises(vpn.VpnError):
        vpn.sample_mixed_primitives(kc, v, q, t, *u)
    with pytest.raises(vpn.VpnError):
        vpn.mesh_vertices_mixed(kc, torch.rand(8, 3), torch.rand(12, 3), v, q, t)


@pytest.mark.parametrize("vertex", [False, True])
def test_emd_counts_the_mixed_points(vpn, vertex):
    from vpn_b200 import templates
    b, k, kc, n = 2, 5, 2, 16
    v, q, t = prims(b, k)
    nvc, nvs = (templates.template(name, "cpu")[0].shape[0] for name in ("cuboid", "sphere"))
    m = kc * nvc + (k - kc) * nvs if vertex else k * n
    u = None if vertex else (torch.rand(b, kc, n, 3), torch.rand(b, k - kc, n, 2))
    step = vpn.PrimitiveLoss(vpn.PrimitiveLossConfig(kind="mixed", n_cuboids=kc, l_emd=1.0, vertex_chamfer=vertex))
    for bad in ((b, m + 1, 3), (b, m - 1, 3), (b + 1, m, 3)):
        with pytest.raises(AssertionError, match="as many points as targets"):
            step(v, q, t, u, torch.rand(*bad))
    with pytest.raises(vpn.VpnError):                                    # P == M: on to the first kernel
        step(v, q, t, u, torch.rand(b, m, 3))


def test_composed_faces_order(vpn):
    """Cuboid faces for the first n_cuboids primitives, then sphere faces, with running vertex offsets."""
    from vpn_b200 import templates
    kc, k = 2, 5
    (cv, cf), (sv, sf) = templates.template("cuboid", "cpu"), templates.template("sphere", "cpu")
    faces = vpn.PrimitiveLoss(vpn.PrimitiveLossConfig(kind="mixed", n_cuboids=kc)).composed_faces(k, "cpu")
    want, off = [], 0
    for i in range(k):
        tv, tf = (cv, cf) if i < kc else (sv, sf)
        want.append(tf + off)
        off += tv.shape[0]
    assert faces.dtype == torch.int32 and torch.equal(faces, torch.cat(want))
    assert int(faces.max()) == kc * cv.shape[0] + (k - kc) * sv.shape[0] - 1


def test_c_entry_points_reject_bad_arguments_without_a_device(vpn):
    from vpn_b200 import _lib
    lib = _lib.load()
    dummy = ctypes.c_void_p(16)                  # never dereferenced: every call below fails its argument checks first
    B, K, Kc, N = 2, 4, 1, 128

    def fwd(mode=0, v=dummy, q=dummy, src_c=dummy, src_s=dummy, out=dummy, b=B, k=K, kc=Kc, nc=N, ns=N):
        return lib.vpn_pose_mixed_fwd(mode, v, q, None, src_c, src_s, out, b, k, kc, nc, ns, None)

    assert fwd(kc=-1) == VPN_ERR_SHAPE
    assert fwd(kc=K + 1) == VPN_ERR_SHAPE
    for bad in ({"b": 0}, {"k": 0}, {"nc": 0, "ns": 0}, {"ns": -3, "mode": 1}, {"nc": N, "ns": N + 4}):
        assert fwd(**bad) == VPN_ERR_SHAPE, bad
    assert fwd(mode=2) == VPN_ERR_ARG
    assert fwd(src_c=None) == VPN_ERR_ARG                               # cuboids present
    assert fwd(src_s=None) == VPN_ERR_ARG                               # spheres present
    assert fwd(q=None) == VPN_ERR_ARG and fwd(out=None) == VPN_ERR_ARG and fwd(v=None) == VPN_ERR_ARG
    assert fwd(kc=0, src_c=None, q=None) == VPN_ERR_ARG                 # a kind without primitives may be NULL; q may not
    assert fwd(kc=K, src_s=None, out=None) == VPN_ERR_ARG

    floats = ctypes.c_size_t(0)
    assert lib.vpn_pose_mixed_bwd_workspace_floats(B, K, K + 1, N, N, ctypes.byref(floats)) == VPN_ERR_SHAPE
    assert lib.vpn_pose_mixed_bwd_workspace_floats(B, K, Kc, N, N, None) == VPN_ERR_ARG
    assert lib.vpn_pose_mixed_bwd_workspace_floats(B, K, Kc, N, N, ctypes.byref(floats)) == 0
    assert floats.value == B * K * 1 * 16                               # one 2048-point slice per primitive
    assert lib.vpn_pose_mixed_bwd_workspace_floats(B, K, Kc, 100, 4097, ctypes.byref(floats)) == 0
    assert floats.value == B * K * 3 * 16                               # slots sized for the larger kind

    def bwd(mode=0, src_c=dummy, src_s=dummy, gout=dummy, ws=dummy, nws=B * K * 16, kc=Kc, nc=N, ns=N):
        return lib.vpn_pose_mixed_bwd(mode, dummy, dummy, src_c, src_s, gout, None, None, None, ws, nws, B, K, kc, nc, ns,
                                      None)

    assert bwd(kc=K + 1) == VPN_ERR_SHAPE and bwd(nc=0) == VPN_ERR_SHAPE and bwd(ns=N + 1) == VPN_ERR_SHAPE
    assert bwd(mode=-1) == VPN_ERR_ARG
    assert bwd(src_c=None) == VPN_ERR_ARG and bwd(src_s=None) == VPN_ERR_ARG
    assert bwd(gout=None) == VPN_ERR_ARG and bwd(ws=None) == VPN_ERR_ARG
    assert bwd(nws=B * K * 16 - 1) == VPN_ERR_WORKSPACE
