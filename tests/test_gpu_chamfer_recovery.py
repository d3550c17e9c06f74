"""Per-block row recovery of the Chamfer forward over sorted clouds (csrc/chamfer_tiled.cu,
chamfer_recover_rows_sorted_kernel): min, arg-min and the first-original-index tie rule must match the CPU oracle bit
for bit on the inputs that take its less common branches - block unions wider than one staged page, target clouds of
more than 64 column chunks (several splits of the filter's records), and a flagged sample inside a batch.  The kernel
runs when the batch has at least one 128-row block per resident CTA slot of the GPU (8 per SM), so every case here has
B * ceil(P / 128) >= 1500."""
import ctypes

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

TILED_TC = 5


@pytest.fixture(scope="module")
def lib():
    assert torch.cuda.is_available()
    from vpn_b200 import _lib
    return _lib


def scene(gen, b, k, n, m, step=None):
    """K cuboid-surface patches of N rows each against M targets on a few box surfaces, in random order; with `step`
    every coordinate is rounded to that lattice (exact ties, duplicate points)."""
    centres = (torch.rand(b, k, 1, 3, generator=gen) - 0.5) * 0.8
    ext = torch.rand(b, k, 1, 3, generator=gen) * 0.1 + 0.02
    u = torch.rand(b, k, n, 3, generator=gen) * 2 - 1
    axis = torch.arange(n)[None, None, :] * 3 // n
    u.scatter_(3, axis[..., None].expand(b, k, n, 1), 1.0)
    p1 = (centres + u * ext).reshape(b, k * n, 3)
    tc = (torch.rand(b, 6, 3, generator=gen) - 0.5) * 0.7
    th = torch.rand(b, 6, 3, generator=gen) * 0.12 + 0.03
    w = torch.randint(0, 6, (b, m), generator=gen)
    t = torch.rand(b, m, 3, generator=gen) * 2 - 1
    ax = torch.randint(0, 3, (b, m), generator=gen)
    t.scatter_(2, ax[..., None], (torch.randint(0, 2, (b, m, 1), generator=gen).float() * 2 - 1))
    bi = torch.arange(b)[:, None]
    p2 = tc[bi, w] + t * th[bi, w]
    if step is not None:
        p1 = torch.round(p1 / step) * step
        p2 = torch.round(p2 / step) * step
    return p1.contiguous(), p2.contiguous()


def nn(lib, p1, p2, impl):
    dl = lib.load()
    b, p, _ = p1.shape
    m = p2.shape[1]
    p1, p2 = p1.cuda(), p2.cuda()
    nb = ctypes.c_size_t(0)
    lib.check(dl.vpn_chamfer_workspace_bytes(b, p, m, impl, ctypes.byref(nb)), "ws")
    ws = torch.empty(nb.value, dtype=torch.uint8, device="cuda")
    out = [torch.empty(b, p, device="cuda"), torch.empty(b, p, dtype=torch.int32, device="cuda"),
           torch.empty(b, m, device="cuda"), torch.empty(b, m, dtype=torch.int32, device="cuda")]
    lib.check(dl.vpn_chamfer_fwd(lib.ptr(p1), lib.ptr(p2), *[lib.ptr(o) for o in out], b, p, m, lib.ptr(ws), nb.value, impl,
                                 lib.stream_ptr(p1.device)), "fwd")
    return [o.cpu().numpy() for o in out]


def assert_exact(got, want):
    m1, i1, m2, i2 = got
    np.testing.assert_array_equal(i1.astype(np.int64), want[1], err_msg="idx1")
    np.testing.assert_array_equal(i2.astype(np.int64), want[3], err_msg="idx2")
    np.testing.assert_array_equal(m1.view(np.int32), want[0].view(np.int32), err_msg="min1")
    np.testing.assert_array_equal(m2.view(np.int32), want[2].view(np.int32), err_msg="min2")


@pytest.mark.parametrize("case", ["coarse_lattice", "duplicate_targets"])
def test_wide_block_unions_take_several_pages(lib, c_oracle, case):
    """A coarse lattice makes rows tie with many targets; a target cloud of one repeated point makes every unit a
    candidate of every row.  Either way a block's candidate units exceed one staged page."""
    gen = torch.Generator().manual_seed(31)
    p1, p2 = scene(gen, 4, 48, 1000, 4096, step=0.25 if case == "coarse_lattice" else None)
    if case == "duplicate_targets":
        p2 = p2[:, :1].expand_as(p2).contiguous()
    assert_exact(nn(lib, p1, p2, TILED_TC), c_oracle(p1.numpy(), p2.numpy()))


@pytest.mark.parametrize("m", [8193, 16500, 40000])
def test_target_clouds_past_64_chunks(lib, c_oracle, m):
    """More than 64 column chunks: unit indices past 256 and several splits of the row records."""
    gen = torch.Generator().manual_seed(m)
    p1, p2 = scene(gen, 4, 48, 1000, m)
    assert_exact(nn(lib, p1, p2, TILED_TC), c_oracle(p1.numpy(), p2.numpy()))


def test_flagged_sample_inside_a_batch(lib, c_oracle):
    """A sample whose coordinates are too large for the filter is redone by the brute-force kernel; the row recovery
    skips it and still serves its neighbours in the batch."""
    gen = torch.Generator().manual_seed(44)
    p1, p2 = scene(gen, 4, 48, 1000, 4096)
    p1[1, 100] = torch.tensor([3e18, -2e18, 1e18])
    assert_exact(nn(lib, p1, p2, TILED_TC), c_oracle(p1.numpy(), p2.numpy()))
