"""Geometry of the hot path: reference config values, camera calibration, BEV cell centres, bucket grid.

Everything here is host-side scalar arithmetic done in float64 and rounded once to float32, so the
CUDA kernels and the CPU oracle receive bit-identical float32 scalars.
"""
from __future__ import annotations

import copy
import math

import numpy as np

# the values of config/config_carla.yaml in the reference (plain facts; the YAML itself is the user's)
_CARLA = {
    "batch_size": 8, "dataset_name": "carla", "cuda_visible_id": "0", "port_number": "12233",
    "saved_model_name": "model_", "num_epoch": 60, "learning_rate": 0.0001, "beta1": 0.9, "plot_AP_graph": False,
    "max_num_pc": 20000, "max_num_bbox": 20,
    "lidar_x_min": 0.0, "lidar_x_max": 70.0, "lidar_y_min": -30.0, "lidar_y_max": 30.0,
    "lidar_z_min": -2.4, "lidar_z_max": 0.8, "delta": 0.2,
    "voxel_length": 384, "voxel_width": 256, "voxel_channel": 32,
    "image_height": 480, "image_width": 640,
    "regress_type": 0, "regress_loss_gain": 3, "positive_range": 5, "pos_sample_threshold": 128,
    "neg_sample_threshold": 128,
    "anchor_bbox_feature": {"width": 2.0, "length": 4.0, "height": 1.5, "reduced_scale": 4},
    "lidar_module": {"out_feature1": 32, "out_feature2": 64, "out_feature3": 128, "out_feature4": 192,
                     "out_feature5": 256, "num_res_block1": 1, "num_res_block2": 2, "num_res_block3": 4,
                     "num_res_block4": 6, "num_res_block5": 6},
    "nms_iou_score_theshold": 0.01, "score_threshold": 0.8,
}

# additive keys of this implementation (SURVEY Appendix A); absent keys take these defaults
FUSION_DEFAULTS = {
    "fusion_k": 3,                 # neighbours per BEV cell (A4/A5)
    "fusion_radius": 2.0,          # metres (A4)
    "fusion_scales": (1,),         # residual groups after which the layer is applied, 1..5 (A11)
    "fusion_image_channels": 128,  # C_img of the camera feature map
    "fusion_image_stride": 4,      # camera map is (image_height/stride, image_width/stride)
    "fusion_mlp_mode": "fp32",     # "fp32" | "bf16" | "bf16t" (bf16 + bf16 tables, inference only) | "simt" (A12)
    "fusion_bucket_size": 0.5,     # metres, K-1 grid pitch
    "fusion_camera_yaws": None,    # degrees, one per camera of a rig (geometry.camera_rig); None = the single camera
    "fusion_camera_image_sizes": None,   # [[w, h], ...] one per camera of the rig; None = image_width x image_height each
}


def carla_config(**overrides) -> dict:
    cfg = copy.deepcopy(_CARLA)
    cfg.update(overrides)
    return cfg


def fusion_option(config: dict, key: str):
    return config.get(key, FUSION_DEFAULTS[key])


def voxel_scales(config: dict):
    """(x_scale, y_scale, x_offset, y_offset) exactly as data_import_carla.py:35-39 computes them."""
    x_scale = int(config["voxel_length"] / (config["lidar_x_max"] - config["lidar_x_min"]))
    y_scale = int(config["voxel_width"] / (config["lidar_y_max"] - config["lidar_y_min"]))
    x_offset = int(-config["lidar_x_min"] * x_scale)
    y_offset = int(-config["lidar_y_min"] * y_scale)
    return x_scale, y_scale, x_offset, y_offset


def voxel_matrix(config: dict):
    """(x_scale, y_scale, z_scale, x_off, y_off, z_off) of pc_to_voxel_indice, data_import_carla.py:35-43 (Python-float
    arithmetic, truncated to int exactly as the reference does)."""
    xs, ys, xo, yo = voxel_scales(config)
    zs = int(config["voxel_channel"] / (config["lidar_z_max"] - config["lidar_z_min"]))
    return xs, ys, zs, xo, yo, int(-config["lidar_z_min"] * zs)


def lidar_range(config: dict):
    """(x_lo, x_hi, y_lo, y_hi, z_lo, z_hi) float32 thresholds of the range filter, data_import_carla.py:214-226:
    keep lo < v < hi with hi = max - delta evaluated in double and then compared in float32."""
    d = config["delta"]
    return tuple(float(np.float32(v)) for v in (config["lidar_x_min"], config["lidar_x_max"] - d, config["lidar_y_min"],
                                                config["lidar_y_max"] - d, config["lidar_z_min"], config["lidar_z_max"] - d))


def scale_geometry(config: dict, stride: int):
    """BEV cell centres at a backbone scale (SURVEY Appendix A3).

    Cell (i, j) of the stride-`stride` feature map sits on input voxel (i*stride, j*stride), whose
    metric centre is ((i*stride + 0.5 - x_offset)/x_scale, (j*stride + 0.5 - y_offset)/y_scale).
    Returns float32 scalars (x0, y0, dx, dy): cx = x0 + float(i)*dx, cy = y0 + float(j)*dy.
    """
    xs, ys, xo, yo = voxel_scales(config)
    return (np.float32((0.5 - xo) / xs), np.float32((0.5 - yo) / ys), np.float32(stride / xs), np.float32(stride / ys))


def bucket_grid(config: dict, cell: float | None = None):
    """(gx0, gy0, cell, nbx, nby) of the K-1 bucket grid covering the LiDAR range of the config."""
    cell = float(fusion_option(config, "fusion_bucket_size") if cell is None else cell)
    gx0, gy0 = float(config["lidar_x_min"]), float(config["lidar_y_min"])
    # cover the voxel grid extent too (it can overshoot lidar_*_max because the scales are truncated ints)
    xs, ys, _, _ = voxel_scales(config)
    x_hi = max(float(config["lidar_x_max"]), gx0 + config["voxel_length"] / xs)
    y_hi = max(float(config["lidar_y_max"]), gy0 + config["voxel_width"] / ys)
    nbx = max(1, int(math.ceil((x_hi - gx0) / cell)))
    nby = max(1, int(math.ceil((y_hi - gy0) / cell)))
    return np.float32(gx0), np.float32(gy0), np.float32(cell), nbx, nby


def _projection64(yaw: float = 0.0, width: float = 640.0, height: float = 480.0) -> np.ndarray:
    """(3,4) float64 projection Cm [R | 0] of the reference camera turned by `yaw` radians about the LiDAR z axis, its
    intrinsics scaled to a width x height image (fx, cx by width/640, fy, cy by height/480: the same field of view).

    The reference builds R with numpy-quaternion's from_euler_angles(v_cam - v_lidar) (:180-188), i.e. the
    Z-Y-Z Euler convention R = Rz(alpha) Ry(beta) Rz(gamma); translation 0; intrinsics from :190-194.  A camera turned by
    yaw sees the point p where the reference camera sees Rz(-yaw) p, so its rotation is R Rz(-yaw) (yaw 0 leaves R as it is).
    """
    a, b, g = (np.array([-3.13498819, 1.59196951, 1.56942932]) - np.array([-1.57079633, 3.12042851, -1.57079633]))

    def rz(t):
        return np.array([[math.cos(t), -math.sin(t), 0.0], [math.sin(t), math.cos(t), 0.0], [0.0, 0.0, 1.0]])

    def ry(t):
        return np.array([[math.cos(t), 0.0, math.sin(t)], [0.0, 1.0, 0.0], [-math.sin(t), 0.0, math.cos(t)]])

    R = rz(a) @ ry(b) @ rz(g)
    if yaw != 0.0:
        R = R @ rz(-yaw)
    RT = np.concatenate([R, np.zeros((3, 1))], axis=1)
    sx, sy = width / 640.0, height / 480.0
    Cm = np.array([[268.51188197672957 * sx, 0.0, 320.0 * sx], [0.0, 268.51188197672957 * sy, 240.0 * sy], [0.0, 0.0, 1.0]])
    return Cm @ RT


def calibration_crt() -> np.ndarray:
    """CRT_tensor of data_import_carla.py:31-34 as a (4,3) float32 array: [x y z 1] @ CRT = (u*w, v*w, w), w < 0 for points
    in front of the camera (the reference's orientation)."""
    return np.ascontiguousarray(_projection64().T.astype(np.float32))


MAX_CAMERAS = 8   # CF_MAX_CAMERAS of include/cf_b200.h


def camera_rig(yaws_deg, image_sizes=None) -> np.ndarray:
    """(M,4,3) float32 calibrations of a rig of M reference cameras, camera m turned by yaws_deg[m] degrees about the LiDAR
    z axis (positive toward +y, i.e. to the left), for cf_point_gather_multi / cf_point_gather_rig: [x y z 1] @ CRT_m =
    (u*w, v*w, w) with w > 0 in front of the camera.  Computed in float64, rounded once to float32 and negated (exact), so
    yaw 0 is exactly -calibration_crt() and every camera's (u, v) is the reference camera's (u, v) of the point turned by
    -yaw.  `image_sizes`: M (w, h) image sizes; camera m's intrinsics are scaled (in float64) to its image, so it keeps the
    reference camera's field of view and projects to (u * w/640, v * h/480).  None, or 640 x 480 everywhere, is the
    reference image."""
    yaws = [float(y) for y in np.asarray(yaws_deg, dtype=np.float64).reshape(-1)]
    if not 1 <= len(yaws) <= MAX_CAMERAS:
        raise ValueError(f"camera_rig: {len(yaws)} cameras, expected 1..{MAX_CAMERAS}")
    sizes = [(640.0, 480.0)] * len(yaws) if image_sizes is None else [tuple(float(v) for v in s) for s in image_sizes]
    if len(sizes) != len(yaws) or any(len(s) != 2 or not (s[0] > 0 and s[1] > 0) for s in sizes):
        raise ValueError(f"camera_rig: image_sizes must be {len(yaws)} positive (w, h) pairs, got {image_sizes}")
    crt = np.stack([_projection64(math.radians(y), w, h).T.astype(np.float32) for y, (w, h) in zip(yaws, sizes)])
    return np.ascontiguousarray(-crt)
