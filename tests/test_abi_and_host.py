"""CPU-side checks: the C-ABI library loads and exports every symbol include/vpn_b200.h declares, the
product refuses to run without CUDA (no CPU fallback), never touches oracle/, and the drop-ins keep the
reference's AssertionError behaviour.  No compute calls are made here."""
import ctypes
import os
import re
import subprocess

import pytest
import torch

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PKG = os.path.join(REPO, "volumetric-primitives-net_b200")


@pytest.fixture(scope="module")
def lib_path():
    path = os.path.join(PKG, "lib", "libvpn_b200.so")
    if not os.path.isfile(path):
        subprocess.check_call(["make", "-C", os.path.join(PKG, "csrc"), "-j8"])
    return path


def header_functions():
    text = open(os.path.join(REPO, "include", "vpn_b200.h")).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(vpn_[a-z0-9_]+)\s*\(", text)))


def test_library_exports_every_declared_symbol(lib_path):
    lib = ctypes.CDLL(lib_path)
    names = header_functions()
    assert len(names) >= 15
    for n in names:
        assert hasattr(lib, n), f"{n} declared in include/vpn_b200.h but not exported"
    lib.vpn_abi_version.restype = ctypes.c_int
    assert lib.vpn_abi_version() == 2


def test_python_binding_covers_header(lib_path):
    from vpn_b200 import _lib
    assert _lib.exported_symbols() == header_functions()
    _lib.load()


def test_library_is_sm100a_only(lib_path):
    out = subprocess.run(["cuobjdump", "-lelf", lib_path], capture_output=True, text=True).stdout
    archs = set(re.findall(r"sm_(\d+a?)", out))
    assert archs == {"100a"}, archs


def test_no_cpu_fallback(lib_path):
    import vpn_b200
    with pytest.raises(vpn_b200.VpnError):
        vpn_b200.chamfer_nn(torch.zeros(1, 4, 3), torch.zeros(1, 4, 3))
    with pytest.raises(vpn_b200.VpnError):
        vpn_b200.sample_primitives("sphere", torch.zeros(1, 1, 3), torch.zeros(1, 1, 4), torch.zeros(1, 1, 3),
                                   torch.zeros(1, 1, 8, 2))


def test_missing_library_fails_loudly(lib_path, monkeypatch):
    from vpn_b200 import _lib
    monkeypatch.setattr(_lib, "_lib", None)
    monkeypatch.setattr(_lib, "LIB_PATH", "/nonexistent/libvpn_b200.so")
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        _lib.load()


def test_product_never_imports_oracle():
    bad = []
    for root, _, files in os.walk(PKG):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h")):
                txt = open(os.path.join(root, f)).read()
                if re.search(r"^\s*(from|import)\s+oracle\b", txt, flags=re.M) or "vpn_oracle" in txt:
                    bad.append(os.path.join(root, f))
    assert not bad, bad


def test_dropin_shape_asserts_match_reference(lib_path):
    """transform.py:12-18, sampling.py:48-52, chamfer_distance.py:33-35, meshing.py:49-55 raise AssertionError."""
    import modules.loss as ml
    import modules.meshing as mm
    import modules.sampling as ms
    import modules.transform as mt
    z = torch.zeros
    with pytest.raises(AssertionError):
        mt.transform_points(z(2, 5, 3), z(2, 3), z(2, 3))
    with pytest.raises(AssertionError):
        mt.transform_points(z(2, 5, 2), z(2, 4), z(2, 3))
    with pytest.raises(AssertionError):
        mt.rotate_points(z(2, 5), z(2, 4))
    with pytest.raises(AssertionError):
        mt.view_to_obj_points(z(2, 5, 3), z(2, 1), z(2), z(2), z(2))
    with pytest.raises(AssertionError):
        ms.Sampling.cuboid_sampling(z(2, 3), z(2, 4), z(3, 3), 10)
    with pytest.raises(AssertionError):
        ms.Sampling.sphere_sampling(z(2, 3), z(2, 4), z(2, 3), 0)
    with pytest.raises(AssertionError):
        ml.ChamferDistanceLoss()(z(2, 5, 2), z(2, 5, 3))
    with pytest.raises(AssertionError):
        ml.VPDiverseLoss()([z(2, 3)] * 3, z(2, 5, 3))          # len != VP_NUM
    with pytest.raises(AssertionError):
        mm.Meshing.sphere_meshing(z(2, 3), z(2, 4), z(3, 3))
    assert ms.Sampling.cone_sampling(z(2, 3), z(2, 4), z(2, 3)) is None


def test_templates_match_reference_assets(golden_templates):
    from vpn_b200 import templates
    from oracle import vpn_oracle as O
    for name in ("sphere", "cuboid", "sphere386"):
        v, f = templates.raw_template(name)
        assert (v == golden_templates[name + "_vertices"]).all() and (f == golden_templates[name + "_faces"]).all()
    tv, _ = templates.template("sphere", "cpu")
    ref = O.sphere_template(torch.from_numpy(golden_templates["sphere_vertices"]))
    assert torch.equal(tv, ref)


def test_pooling_dropin_asserts_and_no_cpu_path(lib_path):
    """gcn.py:91,137-138 raise AssertionError on the wrong rank; CPU tensors are refused (no fallback)."""
    import vpn_b200
    from modules import GCNFeaturePooling as P
    z = torch.zeros
    with pytest.raises(AssertionError):
        P.get_bound_of_images(z(3, 8, 8))
    with pytest.raises(AssertionError):
        P.perceptual_feature_pooling([z(1, 2, 4, 4)], z(5, 3), z(1, 4))
    with pytest.raises(AssertionError):
        P.perceptual_feature_pooling([z(1, 2, 4, 4)], z(1, 5, 3), z(4))
    with pytest.raises(vpn_b200.VpnError):
        P.get_bound_of_images(z(1, 3, 8, 8))
    with pytest.raises(vpn_b200.VpnError):
        P.perceptual_feature_pooling([z(1, 2, 4, 4)], z(1, 5, 3), z(1, 4))


def test_bench_host_logic():
    """Workload table, synthetic inputs and the clock sampler's state machine (no GPU, no NVML needed)."""
    import bench
    for name, (kind, b, k, n, m, res) in bench.WORKLOADS.items():
        d = bench.synthetic(name, "cpu", batch=2)[0]
        assert d["v"].shape == (2, k, 3) and d["q"].shape == (2, k, 4) and d["t"].shape == (2, k, 3)
        assert d["target"].shape == (2, m, 3) and (d["sil"] is None) == (res == 0)
        assert ("canon" in d) == (name in bench.FAITHFUL)
        assert name in bench.describe(name) and str(k * n) in bench.describe(name)
    # network-output-shaped ranges (vpnet_one_resnet.py:69-85): v in (0.0125, 0.1375) x (0.01, 0.11)^2, q in (0, 1)
    d = bench.synthetic("c2", "cpu", batch=4)[0]
    assert 0.0125 < float(d["v"][..., 0].min()) and float(d["v"][..., 0].max()) < 0.1375
    assert 0.0 < float(d["q"].min()) and float(d["q"].max()) < 1.0
    assert bench.per_gpu_batch("c2", 8) == 32 and bench.per_gpu_batch("c4", 8) == 32 and bench.per_gpu_batch("c4", 1) == 256
    same = bench.synthetic("c2", "cpu", seed=7, batch=1)[0]["target"]
    assert torch.equal(same, bench.synthetic("c2", "cpu", seed=7, batch=1)[0]["target"])
    s = bench.ClockSampler(0, enabled=False)                     # disabled sampler: starts, arms, stops, reports nothing
    s.start(); assert s.ready.wait(5.0)
    s.arm(); s.stop(); s.join(5.0)
    assert not s.is_alive() and s.summary()["samples"] == 0 and s.summary()["reasons"] == []


def test_clock_sampler_with_fake_nvml(monkeypatch):
    """The sampling thread against a stand-in NVML: samples only after arm(), median / reasons reported, always stops."""
    import sys
    import time
    import types
    import bench
    fake = types.ModuleType("pynvml")
    fake.NVML_CLOCK_SM = 1
    fake.nvmlClocksThrottleReasonHwSlowdown, fake.nvmlClocksThrottleReasonHwThermalSlowdown = 0x8, 0x40
    fake.nvmlClocksThrottleReasonSwThermalSlowdown, fake.nvmlClocksThrottleReasonSwPowerCap = 0x20, 0x4
    calls = {"n": 0}
    fake.nvmlInit = lambda: None
    fake.nvmlDeviceGetHandleByIndex = lambda i: ("gpu", i)
    fake.nvmlDeviceGetMaxClockInfo = lambda h, c: 1965
    def clock(h, c):
        calls["n"] += 1
        return 1965 if calls["n"] % 2 else 1900
    fake.nvmlDeviceGetClockInfo = clock
    fake.nvmlDeviceGetCurrentClocksThrottleReasons = lambda h: 0x4
    monkeypatch.setitem(sys.modules, "pynvml", fake)
    s = bench.ClockSampler(0, enabled=True, period_s=0.005)
    s.start(); assert s.ready.wait(5.0)
    time.sleep(0.03)
    assert s.samples == []                                        # nothing before arm()
    s.arm(); time.sleep(0.06); s.stop(); s.join(5.0)
    out = s.summary()
    assert not s.is_alive() and out["samples"] >= 3 and out["sm_max_mhz"] == 1965
    assert out["sm_mhz"] in (1900, 1965) and out["reasons"] == ["sw_power_cap"]
    s2 = bench.ClockSampler(0, enabled=True, period_s=10.0)       # stop() before arm(): still takes its one sample and exits
    s2.start(); s2.stop(); s2.join(5.0)
    assert not s2.is_alive() and s2.summary()["samples"] == 1


def test_reference_derived_test_binaries_build_here():
    """oracle/_ref/libemd_ref.so holds the reference's own EMD kernels, compiled from its source tree (VPN_REFERENCE_ROOT)
    where that tree is at hand; nothing of the reference's text is tracked."""
    import subprocess
    from oracle import ref_import
    if not os.path.isfile(os.path.join(ref_import.REFERENCE_ROOT, "modules", "loss", "emd", "emd_cuda.cu")):
        pytest.skip("the reference's source tree is not present")
    subprocess.check_call(["make", "-C", os.path.join(REPO, "oracle")])
    assert os.path.isfile(os.path.join(REPO, "oracle", "_ref", "libemd_ref.so"))
    # nothing of the reference's text is tracked by git: _ref is ignored
    tracked = subprocess.run(["git", "-C", REPO, "ls-files", "oracle/_ref"], capture_output=True, text=True).stdout.strip()
    assert tracked == ""


def test_host_pipeline_orders_results_and_bounds_in_flight():
    """vpn_b200.HostPipeline (CPU path: same ordering logic, synchronous copies): results come back in submission order,
    one step late; a third submit without a result() is refused; host outputs of a slot stay valid until two submits later."""
    import torch
    import vpn_b200
    seen = []

    def step(batch):
        seen.append(float(batch["x"][0]))
        return batch["x"].sum(), batch["x"] * 2

    pipe = vpn_b200.HostPipeline(step, {"x": torch.zeros(4), "unused": None}, "cpu", pre_step=lambda: seen.append("pre"))
    batches = [{"x": torch.full((4,), float(i)), "unused": None} for i in range(5)]
    got = []
    pipe.submit(batches[0])
    for b in batches[1:]:
        pipe.submit(b)
        got.append([t.clone() for t in pipe.result()])
    with pytest.raises(AssertionError):
        pipe.submit(batches[0]); pipe.submit(batches[1])
    got.append([t.clone() for t in pipe.result()])
    assert [float(g[0]) for g in got] == [0.0, 4.0, 8.0, 12.0, 16.0]
    assert [float(g[1][0]) for g in got] == [0.0, 2.0, 4.0, 6.0, 8.0]
    assert seen[:4] == ["pre", 0.0, "pre", 1.0]
