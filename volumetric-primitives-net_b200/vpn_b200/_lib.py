"""ctypes binding of libvpn_b200.so (include/vpn_b200.h).

There is no CPU fallback: if the shared library is missing, or a tensor is not a contiguous CUDA
tensor of the expected dtype, the call raises.  torch is used for device memory and streams only.
"""
from __future__ import annotations

import ctypes
import os
from ctypes import c_char_p, c_double, c_float, c_int, c_size_t, c_void_p, POINTER

import torch

_PKG_ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LIB_PATH = os.environ.get("VPN_B200_LIB", os.path.join(_PKG_ROOT, "lib", "libvpn_b200.so"))

_lib = None

_SIGNATURES = {
    "vpn_last_error_string": (c_char_p, []),
    "vpn_abi_version": (c_int, []),
    "vpn_launch_count": (ctypes.c_ulonglong, []),
    "vpn_set_tuning": (c_int, [c_char_p, c_int]),
    "vpn_device_info": (c_int, [POINTER(c_int)] * 4),
    "vpn_pose_points_fwd": (c_int, [c_int, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_void_p]),
    "vpn_pose_points_fwd_timed": (c_int, [c_int, c_void_p, c_void_p, c_void_p, POINTER(c_void_p), c_int, c_void_p, c_int, c_int,
                                          c_int, POINTER(c_float), c_void_p]),
    "vpn_pose_bwd_workspace_floats": (c_int, [c_int, c_int, POINTER(c_size_t)]),
    "vpn_pose_points_bwd": (c_int, [c_int] + [c_void_p] * 9 + [c_size_t, c_int, c_int, c_void_p]),
    "vpn_pose_mixed_fwd": (c_int, [c_int] + [c_void_p] * 6 + [c_int] * 5 + [c_void_p]),
    "vpn_pose_mixed_bwd_workspace_floats": (c_int, [c_int] * 5 + [POINTER(c_size_t)]),
    "vpn_pose_mixed_bwd": (c_int, [c_int] + [c_void_p] * 9 + [c_size_t] + [c_int] * 5 + [c_void_p]),
    "vpn_cuboid_face_counts": (c_int, [c_void_p, c_void_p, c_int, c_int, c_void_p]),
    "vpn_view_workspace_bytes": (c_int, [c_int, POINTER(c_size_t)]),
    "vpn_view_points": (c_int, [c_int, c_int] + [c_void_p] * 7 + [c_size_t, c_int, c_int, c_void_p]),
    "vpn_chamfer_workspace_bytes": (c_int, [c_int, c_int, c_int, c_int, POINTER(c_size_t)]),
    "vpn_chamfer_fwd": (c_int, [c_void_p] * 6 + [c_int, c_int, c_int, c_void_p, c_size_t, c_int, c_void_p]),
    "vpn_chamfer_main_kernel": (c_char_p, [c_int, c_int, c_int, c_int]),
    "vpn_chamfer_fwd_timed": (c_int, [c_void_p] * 6 + [c_int, c_int, c_int, c_void_p, c_size_t, c_int, c_int,
                                      POINTER(c_float), c_void_p]),
    "vpn_chamfer_bwd": (c_int, [c_void_p] * 10 + [c_int, c_int, c_int, c_void_p]),
    "vpn_chamfer_tc_counters": (c_int, [c_void_p, c_int, c_int, c_int, c_int, POINTER(ctypes.c_ulonglong), c_void_p]),
    "vpn_chamfer_prune_stats": (c_int, [c_void_p, c_int, c_int, c_int, c_int, POINTER(ctypes.c_ulonglong), POINTER(ctypes.c_ulonglong),
                                        c_void_p]),
    "vpn_chamfer_loss_fwd": (c_int, [c_void_p, c_void_p, c_float, c_float, c_void_p, c_void_p, c_int, c_int, c_int,
                                     c_void_p]),
    "vpn_chamfer_loss_bwd": (c_int, [c_void_p] * 7 + [c_float, c_float, c_void_p, c_void_p, c_int, c_int, c_int, c_void_p]),
    "vpn_silhouette_workspace_bytes": (c_int, [c_int, c_int, c_int, POINTER(c_size_t)]),
    "vpn_silhouette_fwd": (c_int, [c_void_p] * 4 + [c_float] * 4 + [c_int, c_float, c_float, c_int] + [c_void_p] * 4
                           + [c_size_t] + [c_int] * 5 + [c_void_p]),
    "vpn_silhouette_bwd": (c_int, [c_void_p] * 2 + [c_float] * 4 + [c_int, c_float, c_float, c_int] + [c_void_p] * 4
                           + [c_size_t] + [c_int] * 5 + [c_void_p]),
    "vpn_mesh_sample_fwd": (c_int, [c_void_p] * 6 + [c_int] * 4 + [c_void_p]),
    "vpn_mesh_sample_bwd": (c_int, [c_void_p] * 5 + [c_int] * 4 + [c_void_p]),
    "vpn_mesh_sample_bwd_workspace_bytes": (c_int, [c_int, c_int, c_int, POINTER(c_size_t)]),
    "vpn_mesh_sample_bwd_sorted": (c_int, [c_void_p] * 8 + [c_size_t] + [c_int] * 4 + [c_void_p]),
    "vpn_emd_workspace_bytes": (c_int, [c_int, c_int, POINTER(c_size_t)]),
    "vpn_emd_fwd": (c_int, [c_void_p] * 5 + [c_size_t, c_int, c_int, c_float, c_int, c_void_p]),
    "vpn_emd_bwd": (c_int, [c_void_p] * 5 + [c_int, c_int, c_void_p]),
    "vpn_emd_loss_fwd": (c_int, [c_void_p, c_float, c_void_p, c_void_p, c_int, c_int, c_void_p]),
    "vpn_emd_loss_bwd": (c_int, [c_void_p] * 5 + [c_float, c_void_p, c_int, c_int, c_void_p]),
    "vpn_image_bounds": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_float, c_void_p]),
    "vpn_points_yz_range": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_int, c_void_p]),
    "vpn_feature_pool_fwd": (c_int, [c_void_p] * 5 + [c_int] * 7 + [c_void_p]),
    "vpn_feature_pool_bwd": (c_int, [c_void_p] * 7 + [c_int] * 7 + [c_void_p]),
    "vpn_feature_pool_bwd_workspace_bytes": (c_int, [c_int, c_int, POINTER(c_size_t)]),
    "vpn_feature_pool_bwd_sorted": (c_int, [c_void_p] * 8 + [c_size_t] + [c_int] * 7 + [c_void_p]),
    "vpn_feature_pool_points_bwd": (c_int, [c_void_p] * 6 + [c_int, c_int, c_void_p]),
    "vpn_allreduce_nvls": (c_int, [c_void_p, c_size_t, c_int, c_int, c_void_p]),
    "vpn_allreduce_nvls_flag_floats": (c_int, [POINTER(c_size_t)]),
    "vpn_allreduce_nvls_error_word": (c_int, []),
    "vpn_allreduce_nvls_sync": (c_int, [c_void_p, c_void_p, c_size_t, c_int, c_int, c_void_p]),
    "vpn_fp32_peak_probe": (c_int, [c_void_p, c_int, POINTER(c_double), POINTER(c_double), c_void_p]),
}


def exported_symbols():
    """Names include/vpn_b200.h declares (tests check that the library exports each one)."""
    return sorted(_SIGNATURES)


def load():
    global _lib
    if _lib is None:
        if not os.path.isfile(LIB_PATH):
            raise RuntimeError(
                f"vpn_b200: CUDA library not found at {LIB_PATH}. Build it with "
                "`make -C volumetric-primitives-net_b200/csrc` (or __graft_entry__.build()). "
                "There is no CPU fallback.")
        lib = ctypes.CDLL(LIB_PATH)
        for name, (res, args) in _SIGNATURES.items():
            fn = getattr(lib, name)
            fn.restype, fn.argtypes = res, args
        _lib = _DeviceGuardedLib(lib)
    return _lib


class _StreamArg(c_void_p):
    """cudaStream_t of torch's current stream on `device_index` (what stream_ptr returns)."""
    device_index = -1


class _DeviceGuardedLib:
    """The C ABI launches on the calling thread's CURRENT device.  Calls whose stream argument belongs to another
    device (tensors on cuda:1 while cuda:0 is current) are made with that device current, so multi-GPU single-process
    callers work; the common case costs one integer comparison."""

    def __init__(self, lib):
        self._raw = lib

    def __getattr__(self, name):
        fn = getattr(self._raw, name)

        def call(*args):
            st = args[-1] if args else None
            if isinstance(st, _StreamArg) and st.device_index >= 0 and st.device_index != torch.cuda.current_device():
                with torch.cuda.device(st.device_index):
                    return fn(*args)
            return fn(*args)

        call.__name__ = name
        setattr(self, name, call)
        return call


class VpnError(RuntimeError):
    pass


def check(rc: int, what: str):
    if rc != 0:
        msg = load().vpn_last_error_string()
        raise VpnError(f"{what} failed (status {rc}): {msg.decode() if msg else ''}")


def ptr(t):
    return None if t is None else c_void_p(t.data_ptr())


def stream_ptr(device):
    s = _StreamArg(torch.cuda.current_stream(device).cuda_stream)
    idx = torch.device(device).index
    s.device_index = torch.cuda.current_device() if idx is None else idx
    return s


def require(t: torch.Tensor, dtype, name: str):
    if not isinstance(t, torch.Tensor) or not t.is_cuda:
        raise VpnError(f"{name}: expected a CUDA tensor (vpn_b200 has no CPU path), got "
                       f"{type(t).__name__ if not isinstance(t, torch.Tensor) else t.device}")
    if t.dtype != dtype:
        raise VpnError(f"{name}: expected dtype {dtype}, got {t.dtype}")
    if not t.is_contiguous():
        raise VpnError(f"{name}: expected a contiguous tensor")
    return t
