"""ctypes binding of libkplanes_b200.so (the C-ABI declared in include/kplanes_b200.h).

There is deliberately NO fallback: if the shared library is missing or a call fails, a RuntimeError is
raised.  Tensors are handed over as raw device pointers; the current torch CUDA stream is passed as the
``void* stream`` argument so kernels are ordered with the surrounding PyTorch work.
"""
from __future__ import annotations

import ctypes
import os
from ctypes import POINTER, Structure, c_char_p, c_double, c_float, c_int, c_int32, c_int64, c_uint32, c_void_p
from typing import Optional, Sequence

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libkplanes_b200.so")
ABI_VERSION = 4

_lib = None
LAUNCH_COUNT = 0  # number of C-ABI kernel-launching calls made (bench.py reports it as gpu_launches evidence)


class KpPoints(Structure):
    _fields_ = [
        ("pts", c_void_p), ("origins", c_void_p), ("directions", c_void_p), ("starts", c_void_p), ("ends", c_void_p),
        ("times", c_void_p), ("D", c_int32), ("S", c_int32), ("norm_mode", c_int32), ("aabb", c_float * 6),
        ("ray_tile", c_int32),
    ]


# name -> argtypes.  Must list every symbol include/kplanes_b200.h declares (tests/test_abi.py checks this).
_P = c_void_p
SIGNATURES = {
    "kp_abi_version": ([], c_int),
    "kp_last_error": ([], c_char_p),
    "kp_launch_count": ([], ctypes.c_longlong),
    "kp_hexplane_fwd": ([_P, _P, c_int, c_int, c_int, POINTER(KpPoints), c_int64, c_int, c_uint32, _P, _P], c_int),
    "kp_hexplane_fwd_dyn": ([_P, _P, c_int, c_int, c_int, POINTER(KpPoints), c_int64, c_int, c_uint32, _P, _P, _P], c_int),
    "kp_hexplane_bwd": ([_P, _P, _P, c_int, c_int, c_int, POINTER(KpPoints), c_int64, c_int, c_uint32, _P, _P], c_int),
    "kp_hexplane_bwd_flags": ([_P, _P, _P, _P, c_int, c_int, c_int, POINTER(KpPoints), c_int64, c_int, c_uint32, _P, _P], c_int),
    "kp_density_field_fwd": ([_P, _P, c_int, c_int, _P, _P, c_int, c_int, POINTER(KpPoints), c_int64, c_uint32, _P, _P], c_int),
    "kp_density_field_bwd": ([_P, _P, _P, c_int, c_int, _P, _P, c_int, c_int, POINTER(KpPoints), c_int64, c_uint32, _P, _P, _P, _P], c_int),
    "kp_sigma_net_fwd": ([_P, _P, _P, c_int64, c_int, c_int, _P, _P, _P, _P], c_int),
    "kp_sigma_net_bwd": ([_P, _P, _P, c_int64, c_int, c_int, _P, _P, _P, _P, _P, _P, _P, _P, _P], c_int),
    "kp_color_net_fwd": ([_P, c_int, _P, c_int, _P, _P, _P, c_int64, c_int, _P, _P, _P, _P, _P], c_int),
    "kp_color_net_bwd": ([c_int, _P, _P, _P, _P, _P, _P, _P, c_int64, c_int, _P, _P, _P, _P, _P, _P, _P, _P], c_int),
    "kp_tc_linear_fwd": ([_P, c_int64, _P, c_int64, _P, c_int64, c_int64, c_int, c_int, c_int, _P], c_int),
    "kp_tc_linear_bwd_data": ([_P, c_int64, _P, c_int64, _P, c_int64, c_int64, c_int, c_int, _P, c_int64, _P], c_int),
    "kp_tc_linear_bwd_weight": ([_P, c_int64, _P, c_int64, _P, c_int64, c_int64, c_int, c_int, _P], c_int),
    "kp_tc_supported": ([c_int, c_int], c_int),
    "kp_decoder_fused_supported": ([c_int, c_int, c_int], c_int),
    "kp_decoder_fwd_fused": ([_P, c_int, _P, c_int, _P, _P, _P, _P, _P, c_int64, c_int, c_int, _P, _P, _P, _P, _P, _P, _P, _P], c_int),
    "kp_aabb_intersect": ([_P, _P, c_int64, POINTER(c_float), c_float, _P, _P, _P], c_int),
    "kp_intersect_aabb": ([_P, _P, c_int64, POINTER(c_float), _P, _P, _P], c_int),
    "kp_uniform_bins": ([_P, _P, c_int, _P, _P, c_int64, c_int, c_int, _P, _P, _P, _P, _P, _P], c_int),
    "kp_pdf_resample": ([_P, _P, c_int, _P, _P, c_int, _P, _P, c_int64, c_int, c_float, c_float, c_int, _P, _P, _P, _P, _P, c_float,
                         _P, _P, _P, _P], c_int),
    "kp_weights_fwd": ([_P, _P, c_int64, c_int, _P, _P], c_int),
    "kp_weights_bwd": ([_P, _P, _P, c_int64, c_int, _P, _P], c_int),
    "kp_render_fwd": ([_P, _P, _P, _P, c_int, c_int, c_int64, c_int, _P, _P, _P, _P, _P, _P, _P, _P], c_int),
    "kp_render_bwd": ([_P, _P, _P, c_int, c_int64, c_int, _P, _P, _P, _P, _P], c_int),
    "kp_distortion_fwd": ([_P, _P, c_int64, c_int, _P, _P], c_int),
    "kp_distortion_bwd": ([_P, _P, _P, c_int64, c_int, _P, _P], c_int),
    "kp_interlevel_fwd": ([_P, _P, _P, _P, c_int64, c_int, c_int, _P, _P], c_int),
    "kp_interlevel_bwd": ([_P, _P, _P, _P, _P, c_int64, c_int, c_int, _P, _P], c_int),
    "kp_plane_reg_fused": ([_P, _P, _P, _P, c_int, _P, c_int, _P, _P], c_int),
    "kp_plane_reg_fused_range": ([_P, _P, _P, _P, c_int, _P, c_int, _P, _P, _P], c_int),
    "kp_plane_reg_fused_shard": ([_P, _P, _P, _P, c_int, _P, c_int, _P, _P, _P], c_int),
    "kp_plane_reg_adam_supported": ([c_int], c_int),
    "kp_plane_reg_adam_scratch_bytes": ([_P, c_int], c_int64),
    "kp_plane_reg_adam": ([_P, _P, _P, _P, _P, _P, c_int, _P, c_float, c_float, c_float, c_float, c_float, c_int64, c_float, _P, _P,
                          _P, c_int64, c_int, _P], c_int),
    "kp_step_scalars": ([_P, _P, _P, c_int64, c_int, POINTER(c_float), c_float, _P, _P, _P], c_int),
    "kp_adam_multi": ([_P, _P, _P, _P, _P, c_int, c_float, c_float, c_float, c_float, c_float, c_int64, c_float, _P, _P], c_int),
    "kp_generate_rays": ([_P, _P, _P, _P, _P, c_int, _P, c_int, c_int, c_int64, c_int64, c_float, _P, _P, _P, _P, _P, _P], c_int),
    "kp_ist_map": ([_P, c_int, c_int64, _P, _P, c_float, _P, _P], c_int),
    "kp_isg_map": ([_P, c_int, c_int64, _P, _P, _P, c_int, c_int, c_float, _P, _P, _P], c_int),
    "kp_importance_pixels_scratch_bytes": ([c_int, c_int], c_int64),
    "kp_importance_pixels": ([_P, c_int, c_int64, c_int, _P, c_int, c_int, ctypes.c_uint64, _P, _P, _P], c_int),
    "kp_image_metrics_scratch_bytes": ([c_int, c_int, c_int], c_int64),
    "kp_image_metrics": ([_P, _P, c_int, c_int, c_int, _P, _P, _P], c_int),
    "kp_image_metrics_masked_scratch_bytes": ([c_int, c_int, c_int], c_int64),
    "kp_image_metrics_masked": ([_P, _P, _P, c_int, c_int, c_int, _P, _P, _P], c_int),
    "kp_depth_metrics_scratch_bytes": ([c_int, c_int64, c_int], c_int64),
    "kp_depth_metrics": ([_P, _P, _P, _P, c_int, c_int64, _P, _P, _P], c_int),
    "kp_eval_maps_scratch_bytes": ([c_int, c_int, c_int], c_int64),
    "kp_eval_maps": ([_P, _P, _P, _P, _P, c_int, c_int, c_int, _P, _P, _P, _P, _P], c_int),
    "kp_compose_frame_scratch_bytes": ([c_int, c_int, c_int], c_int64),
    "kp_compose_frame": ([_P, POINTER(c_int), c_int, c_int, c_int, _P, _P, _P, _P, _P, _P], c_int),
    "kp_compose_frame_accs": ([_P, POINTER(c_int), _P, c_int, c_int, c_int, _P, _P, _P, _P, _P], c_int),
    "kp_jpeg_encode_capacity": ([c_int, c_int], c_int64),
    "kp_jpeg_encode_scratch_bytes": ([c_int, c_int], c_int64),
    "kp_jpeg_header": ([c_int, c_int, c_int, _P], c_int),
    "kp_jpeg_encode": ([_P, c_int, c_int, _P, _P, _P, _P, _P], c_int),
    "kp_loss_head_fwd": ([_P, _P, c_int64, _P, _P, _P, c_int, c_float, c_float, c_float, _P, c_int, _P, _P, _P, _P, _P], c_int),
    "kp_loss_head_bwd": ([_P, _P, c_int64, _P, c_int, c_float, c_float, c_float, _P, _P, _P, _P, _P, _P], c_int),
    "kp_peer_alloc": ([c_int64, POINTER(c_void_p), _P], c_int),
    "kp_peer_open": ([_P, POINTER(c_void_p)], c_int),
    "kp_peer_close": ([_P], c_int),
    "kp_peer_free": ([_P], c_int),
    "kp_peer_error": ([_P, POINTER(c_uint32)], c_int),
    "kp_peer_allreduce": ([_P, c_int, c_int, c_int64, c_int64, c_int, _P], c_int),
    "kp_peer_sharded_adam": ([_P, c_int, c_int, c_int64, c_int64, c_int64, _P, _P, c_float, c_float, c_float, c_float, c_float,
                             c_int64, c_float, _P, c_int, _P], c_int),
    "kp_peer_sharded_adam_sparse": ([_P, c_int, c_int, c_int64, c_int64, c_int64, c_int64, _P, _P, c_float, c_float, c_float, c_float,
                                    c_float, c_int64, c_float, _P, c_int, _P], c_int),
    "kp_line_probe": ([_P, c_int64, c_int, c_int, c_int, c_uint32, _P, POINTER(c_int64), _P], c_int),
    "kp_repack_nchw_to_hwc": ([_P, _P, c_int, c_int, c_int, _P], c_int),
    "kp_repack_hwc_to_nchw": ([_P, _P, c_int, c_int, c_int, _P], c_int),
}


def load() -> ctypes.CDLL:
    """dlopen the library (once) and declare argument types.  Raises if it is missing: no CPU fallback."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(
            f"{LIB_PATH} not found: build it with `python __graft_entry__.py` (nvcc, sm_100a). "
            "soccernerfs_b200 has no CPU or PyTorch fallback path."
        )
    lib = ctypes.CDLL(LIB_PATH)
    for name, (argtypes, restype) in SIGNATURES.items():
        fn = getattr(lib, name)  # AttributeError if the .so does not export a declared symbol
        fn.argtypes = argtypes
        fn.restype = restype
    got = lib.kp_abi_version()
    if got != ABI_VERSION:
        raise RuntimeError(f"libkplanes_b200 ABI version {got} != expected {ABI_VERSION}; rebuild")
    _lib = lib
    return lib


# bench.py's live per-kernel timing: names in TIMED get a CUDA-event pair recorded around the call on the
# launching (current) stream; (name, start, end) tuples are appended to EVENTS.
TIMED = set()
EVENTS = []


def call(name: str, *args) -> None:
    """Invoke a C-ABI entry point and raise RuntimeError(kp_last_error()) on a non-zero status."""
    global LAUNCH_COUNT
    lib = load()
    if name in TIMED:
        start, end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        start.record()
        status = getattr(lib, name)(*args)
        end.record()
        EVENTS.append((name, start, end))
    else:
        status = getattr(lib, name)(*args)
    LAUNCH_COUNT += 1
    if status != 0:
        raise RuntimeError(f"{name} failed ({status}): {lib.kp_last_error().decode()}")


def launch_count() -> int:
    """Kernels launched through the library so far (counted inside the .so)."""
    return int(load().kp_launch_count())


def stream_ptr() -> c_void_p:
    return c_void_p(torch.cuda.current_stream().cuda_stream)


def ptr(t: Optional[torch.Tensor]) -> c_void_p:
    """Device pointer of a contiguous fp32/int64/fp64 CUDA tensor (None -> NULL)."""
    if t is None:
        return c_void_p(0)
    if not t.is_cuda:
        raise RuntimeError("soccernerfs_b200 kernels need CUDA tensors (there is no CPU path)")
    if not t.is_contiguous():
        raise RuntimeError("tensor passed to the C-ABI must be contiguous")
    return c_void_p(t.data_ptr())


def f32c(t: torch.Tensor) -> torch.Tensor:
    """contiguous fp32 view/copy (AMP: inputs are promoted to fp32 like _TruncExp's custom_fwd does)."""
    if t.dtype != torch.float32:
        t = t.float()
    return t if t.is_contiguous() else t.contiguous()


def ptr_array(tensors: Sequence[Optional[torch.Tensor]]):
    arr = (c_void_p * len(tensors))()
    for i, t in enumerate(tensors):
        arr[i] = 0 if t is None else ptr(t).value
    return arr


def hw_array(planes: Sequence[torch.Tensor]):
    """planes are channel-last [H,W,C]."""
    arr = (c_int32 * (2 * len(planes)))()
    for i, p in enumerate(planes):
        arr[2 * i], arr[2 * i + 1] = p.shape[0], p.shape[1]
    return arr


def make_points(*, pts=None, origins=None, directions=None, starts=None, ends=None, times=None, D=4, S=1,
                norm_mode=1, aabb=None, ray_tile=0) -> KpPoints:
    kp = KpPoints()
    kp.pts = ptr(pts).value
    kp.origins = ptr(origins).value
    kp.directions = ptr(directions).value
    kp.starts = ptr(starts).value
    kp.ends = ptr(ends).value
    kp.times = ptr(times).value
    kp.D, kp.S, kp.norm_mode = D, S, norm_mode
    kp.ray_tile = int(ray_tile)
    vals = [0.0] * 6 if aabb is None else [float(v) for v in aabb]
    for i in range(6):
        kp.aabb[i] = vals[i]
    return kp


c_float_p = POINTER(c_float)
__all__ = ["load", "call", "ptr", "ptr_array", "hw_array", "make_points", "stream_ptr", "f32c", "KpPoints", "SIGNATURES",
           "c_float", "c_double", "c_int", "c_int64", "c_uint32", "LIB_PATH"]
