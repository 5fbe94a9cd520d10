"""ctypes binding of libcf_b200.so (include/cf_b200.h).  No CPU fallback: a missing library or a device
that is not sm_100 raises RuntimeError from every op."""
from __future__ import annotations

import ctypes as C
import os
import subprocess

_PKG = os.path.dirname(os.path.abspath(__file__))
SO_PATH = os.path.join(_PKG, "libcf_b200.so")
CSRC = os.path.join(_PKG, "csrc")

MODE_FP32, MODE_BF16, MODE_SIMT, MODE_BF16_TABLES = 0, 1, 2, 3
BWD_DETERMINISTIC = 0x100   # CF_BWD_DETERMINISTIC: OR-ed into the mode of cf_fusion_bwd
IO_BF16 = 0x200             # CF_IO_BF16: OR-ed into the mode of cf_fusion_fwd / cf_fusion_bwd for bf16 BEV maps
IO_NHWC = 0x400             # CF_IO_NHWC: OR-ed into the mode of cf_fusion_fwd / cf_fusion_bwd for (B,H,W,C) (channels_last) BEV maps
# "bf16t" = CF_MODE_BF16_TABLES: bf16 operands AND bf16 layer-1 tables (inference only)
MODES = {"fp32": MODE_FP32, "bf16": MODE_BF16, "simt": MODE_SIMT, "bf16t": MODE_BF16_TABLES}
MAX_K = 16
MAX_CAMERAS = 8             # CF_MAX_CAMERAS: cameras of a rig (cf_point_gather_multi, cf_point_gather_rig)
ABI_VERSION = 2

_vp, _i32, _i64, _f32, _sz = C.c_void_p, C.c_int32, C.c_int64, C.c_float, C.c_size_t


class CameraMap(C.Structure):
    """cf_camera_map: one camera of a cf_point_gather_rig* call (its map, ELEMENT strides, extent and image size)."""
    _fields_ = [("d_map", _vp), ("sb", _i64), ("sc", _i64), ("sh", _i64), ("sw", _i64), ("Hf", _i32), ("Wf", _i32),
                ("img_w", _f32), ("img_h", _f32)]


_cams = C.POINTER(CameraMap)

# name -> (restype, argtypes); mirrors include/cf_b200.h one to one
SIGNATURES = {
    "cf_abi_version": (C.c_int, []),
    "cf_last_error": (C.c_char_p, []),
    "cf_device_check": (C.c_int, []),
    "cf_launch_count": (C.c_longlong, []),
    "cf_bucket_workspace_bytes": (_sz, [_i32, _i32, _i32]),
    "cf_bucket_points": (C.c_int, [_vp, _vp, _i32, _i32, _f32, _f32, _f32, _i32, _i32, _vp, _vp, _vp, _vp]),
    "cf_knn_query": (C.c_int, [_vp, _vp, _i32, _i32, _f32, _f32, _f32, _i32, _i32, _i32, _i32, _f32, _f32, _f32, _f32,
                               _f32, _i32, _vp, _vp]),
    "cf_knn_subsample": (C.c_int, [_vp, _i32, _i32, _i32, _i32, _vp, _i32, _i32, _i32, _vp]),
    "cf_gather_workspace_bytes": (_sz, [_i32, _i32, _i32, _i32, _i64]),
    "cf_point_gather": (C.c_int, [_vp, _i64, _i64, _i64, _i64, _i32, _i32, _i32, _i32, _vp, _vp, C.POINTER(C.c_float),
                                  _vp, _i32, _f32, _f32, _vp, _vp, _vp]),
    "cf_point_gather_bf16": (C.c_int, [_vp, _i64, _i64, _i64, _i64, _i32, _i32, _i32, _i32, _vp, _vp, C.POINTER(C.c_float),
                                       _vp, _i32, _f32, _f32, _vp, _vp, _vp]),
    "cf_gather_multi_workspace_bytes": (_sz, [_i32, _i32, _i32, _i32, _i32, _i64]),
    "cf_point_gather_multi": (C.c_int, [_vp, _i64, _i64, _i64, _i64, _i64, _i32, _i32, _i32, _i32, _i32, _vp, _vp, _vp, _i32,
                                        _f32, _f32, _vp, _vp, _vp]),
    "cf_point_gather_multi_bf16": (C.c_int, [_vp, _i64, _i64, _i64, _i64, _i64, _i32, _i32, _i32, _i32, _i32, _vp, _vp, _vp,
                                             _i32, _f32, _f32, _vp, _vp, _vp]),
    "cf_point_gather_multi_bwd": (C.c_int, [_vp, _vp, _i64, _i64, _i64, _i64, _i64, _i32, _i32, _i32, _i32, _i32, _vp, _vp,
                                            _vp, _i32, _f32, _f32, _vp]),
    "cf_point_gather_multi_bwd_det_workspace_bytes": (_sz, [_i32, _i32, _i32, _i32, _i32]),
    "cf_point_gather_multi_bwd_det": (C.c_int, [_vp, _vp, _i64, _i64, _i64, _i64, _i64, _i32, _i32, _i32, _i32, _i32, _vp,
                                                _vp, _vp, _i32, _f32, _f32, _vp, _vp]),
    "cf_gather_rig_workspace_bytes": (_sz, [_i32, _i32, _i32, _cams]),
    "cf_point_gather_rig": (C.c_int, [_cams, _i32, _i32, _i32, _vp, _vp, _vp, _i32, _vp, _vp, _vp]),
    "cf_point_gather_rig_bf16": (C.c_int, [_cams, _i32, _i32, _i32, _vp, _vp, _vp, _i32, _vp, _vp, _vp]),
    "cf_point_gather_rig_bwd": (C.c_int, [_vp, C.POINTER(_vp), _cams, _i32, _i32, _i32, _vp, _vp, _vp, _i32, _vp]),
    "cf_point_gather_rig_bwd_det_workspace_bytes": (_sz, [_i32, _i32, _i32, _cams]),
    "cf_point_gather_rig_bwd_det": (C.c_int, [_vp, C.POINTER(_vp), _cams, _i32, _i32, _i32, _vp, _vp, _vp, _i32, _vp, _vp]),
    "cf_point_mlp1_workspace_bytes": (_sz, [_i32, _i32, _i32]),
    "cf_point_mlp1": (C.c_int, [_vp, _vp, _vp, _i32, _i32, _i32, _i32, _vp, _vp, _vp, _i32, _vp, _vp, _vp]),
    "cf_point_mlp1_pack_weights": (C.c_int, [_vp, _i32, _i32, _i32, _vp, _vp]),
    "cf_point_mlp1_multi": (C.c_int, [_vp, _vp, _vp, _i32, _i32, _i32, _i32, C.POINTER(_i32), C.POINTER(_vp), C.POINTER(_vp),
                                      C.POINTER(_vp), _i32, C.POINTER(_vp), _vp]),
    "cf_fusion_packed_bytes": (_sz, [_i32, _i32]),
    "cf_fusion_pack_weights": (C.c_int, [_vp, _vp, _i32, _i32, _vp, _vp]),
    "cf_fusion_workspace_bytes": (_sz, [_i32, _i32, _i32, _i32, _i32]),
    "cf_fusion_fwd": (C.c_int, [_vp, _vp, _vp, _i32, _i32, _i32, _i32, _i32, _i32, _f32, _f32, _f32, _f32, _vp, _i32,
                                _vp, _vp, _vp, _vp, _vp, _i32, _vp, _vp, _vp]),
    "cf_fusion_bwd_workspace_bytes": (_sz, [_i32, _i32, _i32, _i32, _i32, _i32, _i32]),
    "cf_fusion_bwd": (C.c_int, [_vp, _vp, _vp, _vp, _vp, _i32, _i32, _i32, _i32, _i32, _i32, _f32, _f32, _f32, _f32,
                                _vp, _vp, _i32, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _i32, _vp, _vp]),
    "cf_point_gather_bwd": (C.c_int, [_vp, _vp, _i64, _i64, _i64, _i64, _i32, _i32, _i32, _i32, _vp, _vp,
                                      C.POINTER(C.c_float), _vp, _i32, _f32, _f32, _vp]),
    "cf_fusion_bwd_det_workspace_bytes": (_sz, [_i32, _i32, _i32, _i32, _i32, _i32, _i32]),
    "cf_point_gather_bwd_det_workspace_bytes": (_sz, [_i32, _i32, _i32, _i32]),
    "cf_point_gather_bwd_det": (C.c_int, [_vp, _vp, _i64, _i64, _i64, _i64, _i32, _i32, _i32, _i32, _vp, _vp,
                                          C.POINTER(C.c_float), _vp, _i32, _f32, _f32, _vp, _vp]),
    "cf_voxelize_workspace_bytes": (_sz, [_i32, _i32, _i32, _i32, _i32]),
    "cf_voxelize_project": (C.c_int, [_vp, _vp, _i32, _i32, C.POINTER(C.c_float), C.POINTER(C.c_float), _i32, _i32, _i32,
                                      C.POINTER(C.c_float), _f32, _f32, _i32, _vp, _vp, _vp, _vp, _vp, _vp]),
    "cf_loss_targets": (C.c_int, [_vp, _vp, _i32, _i32, _i32, _i32, _i32, _f32, _f32, _f32, _f32, _f32, _i32, _i32, _i32, _i32,
                                  _vp, _vp, _i32, _vp, _vp, _vp, _vp, _vp, _vp]),
    "cf_get_bboxes": (C.c_int, [_vp, _vp, _i32, _i32, _i32, _f32, _i32, _vp, _vp, _vp, _vp]),
    "cf_nms_workspace_bytes": (_sz, [_i32, _i32]),
    "cf_nms_sat": (C.c_int, [_vp, _vp, _i32, _i32, _vp, _vp, _vp, _vp]),
    "cf_nms_iou": (C.c_int, [_vp, _vp, _i32, _i32, _f32, _vp, _vp, _vp, _vp]),
    "cf_sat_matrix": (C.c_int, [_vp, _i32, _vp, _vp]),
    "cf_box_iou": (C.c_int, [_vp, _i32, _vp, _i32, _f32, _vp, _vp, _vp]),
    "cf_debug_umma_gemm": (C.c_int, [_vp, _vp, _i32, _i32, _i32, _vp, _vp]),
    "cf_debug_bwd_packed_bytes": (_sz, [_i32, _i32]),
    "cf_debug_bwd_gemm_nn": (C.c_int, [_vp, _i64, _vp, _i32, _i32, _vp, _i32, _vp, _i32, _vp, _vp, _vp]),
    "cf_debug_bwd_gemm_tn": (C.c_int, [_vp, _i32, _vp, _i32, _vp, _i32, _vp, _i64, _vp, _vp, _vp, _vp]),
}

_lib = None


def build(verbose: bool = False) -> str:
    """nvcc -gencode arch=compute_100a,code=sm_100a ... -> libcf_b200.so, in-tree (cross-compiles without a GPU)."""
    cmd = ["make", "-C", CSRC, "-j8"]
    res = subprocess.run(cmd, capture_output=True, text=True)
    if verbose or res.returncode != 0:
        print(res.stdout[-4000:])
        print(res.stderr[-4000:])
    if res.returncode != 0:
        raise RuntimeError("building libcf_b200.so failed")
    return SO_PATH


def load():
    """The loaded library.  Raises RuntimeError if it has not been built -- there is no fallback."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(SO_PATH):
        raise RuntimeError(
            f"{SO_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "(this package has no CPU or PyTorch fallback)")
    lib = C.CDLL(SO_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)  # AttributeError here means header and library disagree
        fn.restype, fn.argtypes = res, args
    ver = lib.cf_abi_version()
    if ver != ABI_VERSION:
        raise RuntimeError(f"libcf_b200.so ABI {ver} != expected {ABI_VERSION}; rebuild")
    _lib = lib
    return lib


def check(rc: int, what: str = ""):
    if rc != 0:
        msg = load().cf_last_error().decode("utf-8", "replace")
        raise RuntimeError(f"libcf_b200 error {rc} {what}: {msg}")


def stream_ptr():
    import torch
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def ptr(t):
    """Device pointer of a tensor (None -> NULL)."""
    return C.c_void_p(0 if t is None else t.data_ptr())
