"""ctypes binding of liby5obb.so — the C ABI declared in include/y5obb.h.

There is no CPU fallback and no alternative backend: if the library is missing or a call fails this
module raises.  PyTorch is used only for device memory and streams.
"""
import ctypes
from ctypes import c_void_p, c_int, c_int64, c_float, c_size_t, c_char_p
from pathlib import Path

import torch

_PKG = Path(__file__).resolve().parent
_LIBPATH = _PKG / "liby5obb.so"
_lib = None

_ERR = {1: "Y5OBB_EINVAL (bad argument)", 2: "Y5OBB_EWORKSPACE (workspace too small)",
        3: "Y5OBB_ECUDA (CUDA call failed)", 4: "Y5OBB_EARCH (device is not sm_100)"}

# name -> (restype, argtypes); mirrors include/y5obb.h one to one (tests/test_abi.py checks the set)
PROTOTYPES = {
    "y5obb_abi_version": (c_int, []),
    "y5obb_last_cuda_error": (c_int, []),
    "y5obb_build_info": (c_char_p, []),
    "y5obb_nms_workspace_bytes": (c_size_t, [c_int64, c_int64, c_int64]),
    "y5obb_nms_rotated_f32": (c_int, [c_void_p, c_void_p, c_int64, c_float, c_int, c_void_p, c_void_p,
                                      c_void_p, c_size_t, c_void_p]),
    "y5obb_nms_rotated_batched_f32": (c_int, [c_void_p, c_void_p, c_void_p, c_int64, c_int64, c_int64, c_float,
                                              c_int, c_int64, c_void_p, c_void_p, c_void_p, c_void_p, c_size_t,
                                              c_void_p]),
    "y5obb_nms_debug_stage_timing": (c_int, [c_int]),
    "y5obb_nms_debug_stage_ms": (c_int, [ctypes.POINTER(c_float)]),
    "y5obb_rbox_iou_pairs_f32": (c_int, [c_void_p, c_void_p, c_void_p, c_int64, c_void_p]),
    "y5obb_nms_obb_workspace_bytes": (c_size_t, [c_int64, c_int64, c_int64, c_int64]),
    "y5obb_nms_obb_f32": (c_int, [c_void_p, c_int64, c_int64, c_int, c_int, c_float, c_float, ctypes.c_uint64, c_int,
                                  c_int, c_int, c_int, c_float, c_int, c_int64, c_void_p, c_void_p, c_void_p, c_size_t,
                                  c_void_p]),
    "y5obb_conv_tiling": (c_int, [c_int, c_int, c_int, c_int] + [ctypes.POINTER(c_int)] * 5),
    "y5obb_conv_create": (c_int, [c_void_p, ctypes.POINTER(c_void_p)]),
    "y5obb_conv_run": (c_int, [c_void_p, c_void_p]),
    "y5obb_conv_info": (c_int, [c_void_p, ctypes.POINTER(ctypes.c_double), ctypes.POINTER(ctypes.c_double)]
                        + [ctypes.POINTER(c_int)] * 4),
    "y5obb_conv_destroy": (None, [c_void_p]),
    "y5obb_conv_debug_timestamps": (c_int, [c_void_p, c_void_p]),
    "y5obb_loss_workspace_bytes": (c_size_t, [c_void_p]),
    "y5obb_loss_forward": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_size_t, c_void_p]),
    "y5obb_loss_backward": (c_int, [c_void_p, c_void_p, c_void_p, c_size_t, c_void_p]),
    "y5obb_rbox2poly_f32": (c_int, [c_void_p, c_void_p, c_int64, c_void_p]),
    "y5obb_poly2hbb_f32": (c_int, [c_void_p, c_void_p, c_int64, c_void_p]),
    "y5obb_scale_polys_f32": (c_int, [c_void_p, c_int64, c_float, c_float, c_float, c_void_p]),
    "y5obb_poly2rbox": (c_int, [c_void_p, c_void_p, c_int64, c_int, c_void_p]),
    "y5obb_gaussian_label": (c_int, [c_void_p, c_void_p, c_int64, c_int, ctypes.c_double, c_void_p]),
    "y5obb_bn_scratch_floats": (c_int64, [c_int]),
    "y5obb_bn_batch_stats": (c_int, [c_void_p, c_int64, c_int64, c_int, c_void_p, c_void_p, c_float, c_float, c_void_p, c_void_p,
                                     c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int64, c_void_p]),
    "y5obb_bn_stats": (c_int, [c_void_p, c_int64, c_int64, c_int, c_void_p, c_void_p, c_void_p, c_int64, c_void_p]),
    "y5obb_bn_finalize": (c_int, [c_void_p, c_void_p, c_int64, c_int, c_void_p, c_void_p, c_float, c_float, c_void_p,
                                  c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p]),
    "y5obb_bn_silu_apply": (c_int, [c_void_p, c_int64, c_int64, c_int, c_int, c_void_p, c_void_p, c_int, c_void_p,
                                    c_int64, c_void_p, c_int64, c_void_p, c_int64, c_void_p]),
    "y5obb_bn_silu_bwd": (c_int, [c_void_p, c_int64, c_void_p, c_int64, c_int64, c_int, c_void_p, c_void_p, c_void_p,
                                  c_void_p, c_int, c_void_p, c_void_p, c_void_p, c_int64, c_void_p, c_int64, c_int,
                                  c_void_p, c_void_p, c_int, c_void_p, c_int64, c_void_p]),
    "y5obb_wgrad_create": (c_int, [c_void_p, ctypes.POINTER(c_void_p)]),
    "y5obb_wgrad_run": (c_int, [c_void_p, c_void_p]),
    "y5obb_wgrad_destroy": (None, [c_void_p]),
    "y5obb_sgd_ema_plan_create": (c_int, [c_void_p, c_int, ctypes.POINTER(c_void_p)]),
    "y5obb_sgd_ema_plan_run": (c_int, [c_void_p, c_void_p, c_float, c_float, c_int, c_void_p]),
    "y5obb_sgd_ema_plan_destroy": (None, [c_void_p]),
    "y5obb_poly_nms_workspace_bytes": (c_size_t, [c_int64]),
    "y5obb_poly_nms_f64": (c_int, [c_void_p, c_int64, ctypes.c_double, c_void_p, c_void_p, c_void_p, c_size_t, c_void_p]),
    "y5obb_poly_iou_pairs_f64": (c_int, [c_void_p, c_void_p, c_void_p, c_int64, c_void_p]),
    "y5obb_tiles_to_scene_workspace_bytes": (c_size_t, [c_int]),
    "y5obb_tiles_to_scene_f64": (c_int, [c_void_p, c_void_p, c_int, c_int, c_void_p, c_void_p, c_int, c_int, c_void_p, c_void_p,
                                         c_void_p, c_void_p, c_void_p, c_size_t, c_void_p]),
    "y5obb_poly_nms_segmented_workspace_bytes": (c_size_t, [c_void_p, c_int64]),
    "y5obb_poly_nms_segmented_f64": (c_int, [c_void_p, c_void_p, c_int64, c_void_p, c_int64, ctypes.c_double, c_void_p,
                                             c_void_p, c_void_p, c_size_t, c_void_p]),
    "y5obb_poly_nms_f32_workspace_bytes": (c_size_t, [c_int64]),
    "y5obb_poly_nms_f32": (c_int, [c_void_p, c_int64, c_float, c_int, c_void_p, c_void_p, c_void_p, c_size_t, c_void_p]),
    "y5obb_poly_overlaps_f32": (c_int, [c_void_p, c_void_p, c_int64, c_int64, c_void_p, c_void_p]),
    "y5obb_poly_iou_pairs_f32": (c_int, [c_void_p, c_void_p, c_void_p, c_int64, c_void_p]),
    "y5obb_devkit_poly_nms": (None, [c_void_p, c_void_p, c_void_p, c_int, c_int, c_float, c_int]),
    "y5obb_devkit_overlaps": (None, [c_void_p, c_void_p, c_void_p, c_int, c_int, c_int]),
    "y5obb_val_match_f32": (c_int, [c_void_p, c_void_p, c_int, c_int, c_void_p, c_int, c_void_p, c_void_p, c_int, c_void_p,
                                    c_void_p, c_void_p, c_void_p, c_void_p]),
    "y5obb_pack_plan_create": (c_int, [c_void_p, c_int, ctypes.POINTER(c_void_p)]),
    "y5obb_pack_plan_run": (c_int, [c_void_p, c_void_p]),
    "y5obb_pack_plan_destroy": (None, [c_void_p]),
    "y5obb_upsample2x_bwd": (c_int, [c_void_p, c_int64, c_void_p, c_int64, c_int64, c_int, c_int, c_int, c_void_p]),
    "y5obb_zero_stuff2x": (c_int, [c_void_p, c_int64, c_void_p, c_int64, c_int64, c_int, c_int, c_void_p]),
    "y5obb_maxpool5_bwd": (c_int, [c_void_p, c_int64, c_void_p, c_void_p, c_int64, c_void_p, c_int, c_int, c_int, c_int,
                                   c_void_p]),
    "y5obb_add_f32_to_bf16": (c_int, [c_void_p, c_void_p, c_int64, c_int64, c_int, c_int, c_void_p]),
    "y5obb_detect_grad_pack": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int, c_int, c_void_p]),
    "y5obb_stem_s2d": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_void_p]),
    "y5obb_stem_s2d_u8": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_void_p]),
    "y5obb_stem_s2d_scene_u8": (c_int, [c_void_p, c_int, c_int, c_void_p, c_int, c_int, c_int, c_void_p, c_int, c_void_p]),
    "y5obb_sppf_pool": (c_int, [c_void_p, c_int64, c_int, c_int, c_int, c_int, c_void_p]),
}

NMS_STRICT_GT = 1
NMS_DROP_SMALL = 2
NMS_NO_CLASS_SPLIT = 4
NMS_COMPACT_PRED = 8


def lib() -> ctypes.CDLL:
    """Load liby5obb.so (built in-tree by yolov5_obb_b200.build / __graft_entry__.build)."""
    global _lib
    if _lib is None:
        if not _LIBPATH.exists():
            raise RuntimeError(f"{_LIBPATH} is missing: run `python -m yolov5_obb_b200.build` "
                               "(there is no CPU or PyTorch fallback for this path)")
        L = ctypes.CDLL(str(_LIBPATH))
        for name, (res, args) in PROTOTYPES.items():
            fn = getattr(L, name)  # AttributeError if the ABI and this table disagree
            fn.restype, fn.argtypes = res, args
        _lib = L
    return _lib


def check(rc: int, what: str) -> None:
    if rc != 0:
        extra = ""
        if rc == 3:
            extra = f" cudaError={lib().y5obb_last_cuda_error()}"
        raise RuntimeError(f"{what} failed: {_ERR.get(rc, rc)}{extra}")


def ptr(t) -> int:
    return 0 if t is None else t.data_ptr()


def stream_ptr(device=None) -> int:
    return torch.cuda.current_stream(device).cuda_stream


_WS = {}


def workspace(nbytes: int, device, tag: str = "default") -> torch.Tensor:
    """Grow-only cached byte buffer per (device, tag).  Stream-ordered reuse: callers on the same
    stream may share a tag; different streams must use different tags."""
    key = (torch.device(device).index or 0, tag)
    buf = _WS.get(key)
    if buf is None or buf.numel() < nbytes:
        buf = torch.empty(int(nbytes * 1.25) + 4096, dtype=torch.uint8, device=device)
        _WS[key] = buf
    return buf


def require_cuda(t: torch.Tensor, name: str) -> None:
    if not t.is_cuda:
        raise RuntimeError(f"{name} must be a CUDA tensor: yolov5_obb_b200 has no CPU path "
                           "(the CPU restatement lives in oracle/ and is test infrastructure)")
