"""CPU: the camera-rig surface that needs no GPU -- the C ABI of cf_point_gather_multi* is declared, exported and bound,
geometry.camera_rig turns the reference camera exactly, argument errors are raised before anything is launched, and a
rig model keeps the single-camera module tree and state-dict keys."""
import ctypes
import math
import os
import re

import numpy as np
import pytest
import torch

import dcf_b200 as dcf

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
NEW = ("cf_gather_multi_workspace_bytes", "cf_point_gather_multi", "cf_point_gather_multi_bf16", "cf_point_gather_multi_bwd",
       "cf_point_gather_multi_bwd_det_workspace_bytes", "cf_point_gather_multi_bwd_det")


def _header():
    return open(os.path.join(ROOT, "include", "cf_b200.h")).read()


def test_rig_entry_points_declared_exported_and_bound():
    h = _header()
    assert re.search(r"#define CF_ABI_VERSION 2\b", h) and dcf._lib.ABI_VERSION == 2
    m = re.search(r"#define CF_MAX_CAMERAS (\d+)\b", h)
    assert m and int(m.group(1)) == dcf._lib.MAX_CAMERAS == dcf.geometry.MAX_CAMERAS == 8
    lib = ctypes.CDLL(dcf.SO_PATH)
    for name in NEW:
        assert re.search(rf"CF_API\s+[\w\s\*]+?\b{name}\s*\(", h), name
        assert hasattr(lib, name) and name in dcf._lib.SIGNATURES, name
    # the bf16 map variant takes the fp32 variant's arguments
    assert dcf._lib.SIGNATURES["cf_point_gather_multi_bf16"] == dcf._lib.SIGNATURES["cf_point_gather_multi"]
    L = dcf.load()
    assert L.cf_abi_version() == 2
    assert L.cf_gather_multi_workspace_bytes(2, 3, 128, 120, 160, 1) == 0           # channels_last: read in place
    assert L.cf_gather_multi_workspace_bytes(2, 3, 128, 120, 160, 19200) == 2 * 3 * 128 * 120 * 160 * 4
    assert (L.cf_point_gather_multi_bwd_det_workspace_bytes(2, 3, 1000, 30, 40)
            == L.cf_point_gather_bwd_det_workspace_bytes(6, 1000, 30, 40))          # the single-camera lists over B*M maps


def test_rig_yaw_zero_is_the_negated_reference_camera():
    G = dcf.geometry
    rig = G.camera_rig([0])
    assert rig.shape == (1, 4, 3) and rig.dtype == np.float32
    assert np.array_equal(rig[0].view(np.uint32), (-G.calibration_crt()).view(np.uint32))
    three = G.camera_rig([-60.0, 0.0, 60.0])
    assert np.array_equal(three[1].view(np.uint32), rig[0].view(np.uint32))
    with pytest.raises(ValueError):
        G.camera_rig([0.0] * 9)
    with pytest.raises(ValueError):
        G.camera_rig([])


@pytest.mark.parametrize("yaw", [-60.0, 0.0, 45.0, 60.0, 120.0])
def test_rig_camera_sees_the_turned_point(yaw):
    """(u, v) of camera m at point p == (u, v) of the reference camera at Rz(-yaw) p; w > 0 in front of camera m."""
    G = dcf.geometry
    crt = G.camera_rig([yaw])[0].astype(np.float64)
    ref = G.calibration_crt().astype(np.float64)
    rng = np.random.default_rng(3)
    n = 4000
    az = np.deg2rad(yaw) + rng.uniform(-0.7, 0.7, n)           # within the camera's ~+-50 deg horizontal view
    r = rng.uniform(3.0, 70.0, n)
    p = np.stack([r * np.cos(az), r * np.sin(az), rng.uniform(-2.3, 0.7, n)], axis=1)
    t = -math.radians(yaw)
    rot = np.array([[math.cos(t), -math.sin(t), 0.0], [math.sin(t), math.cos(t), 0.0], [0.0, 0.0, 1.0]])
    q = np.concatenate([p, np.ones((n, 1))], axis=1) @ crt
    q_ref = np.concatenate([p @ rot.T, np.ones((n, 1))], axis=1) @ ref
    assert (q[:, 2] > 0).all() and (q_ref[:, 2] < 0).all()
    uv, uv_ref = q[:, :2] / q[:, 2:], q_ref[:, :2] / q_ref[:, 2:]
    assert np.abs(uv - uv_ref).max() <= 1e-3
    # a point behind the camera has w < 0
    back = np.concatenate([-p[:, :2], p[:, 2:], np.ones((n, 1))], axis=1) @ crt
    assert (back[:, 2] < 0).all()


def _cpu_rig(B=2, M=3, Ci=8, N=16):
    return torch.zeros(B, M, Ci, 6, 8), torch.zeros(B, N, 3), torch.tensor([N] * B), torch.zeros(M, 4, 3)


def test_rig_argument_errors_before_any_launch():
    ops = dcf.ops
    img, pts, cnt, cal = _cpu_rig()
    before = dcf.load().cf_launch_count()
    with pytest.raises(ValueError, match="cameras"):
        ops.point_gather_multi(torch.zeros(2, 9, 8, 6, 8), pts, cnt, torch.zeros(9, 4, 3))
    with pytest.raises(ValueError, match="calib"):
        ops.point_gather_multi(img, pts, cnt, torch.zeros(2, 4, 4, 3))          # 4 calibrations for 3 cameras
    with pytest.raises(ValueError, match="calib"):
        ops.point_gather_multi(img, pts, cnt, torch.zeros(3, 4, 3, 3))          # not (4,3) per camera
    with pytest.raises(ValueError, match="points"):
        ops.point_gather_multi(img, torch.zeros(3, 16, 3), cnt, cal)            # batch mismatch
    with pytest.raises(ValueError, match="B,M,Ci,Hf,Wf"):
        ops.point_gather_multi(img[:, 0], pts, cnt, cal)
    with pytest.raises(ValueError, match="multiple of 4"):
        ops.point_gather_multi(torch.zeros(2, 3, 6, 6, 8), pts, cnt, cal)
    with pytest.raises(TypeError):
        ops.point_gather_multi(img, pts, cnt, dcf.geometry.camera_rig([0, 10, 20]))   # a host array: calib lives on the device
    with pytest.raises(TypeError):
        ops.point_gather_multi(img, pts, cnt, cal.double())
    with pytest.raises(ValueError, match="cameras"):
        ops.point_gather_multi_bwd(torch.zeros(2, 16, 8), torch.zeros(2, 9, 8, 6, 8), pts, cnt, torch.zeros(9, 4, 3))
    # precomputed uv cannot serve a rig: FrameContext.gather refuses it before touching its state
    with pytest.raises(ValueError, match="uv"):
        dcf.FrameContext.gather(object(), img, calib=cal, uv=torch.zeros(2, 16, 2))
    with pytest.raises(ValueError, match="calib"):
        dcf.FrameContext.gather(object(), img)
    assert dcf.load().cf_launch_count() == before


def _rig_cfg(**kw):
    return dcf.geometry.carla_config(fusion_scales=(1, 3), fusion_camera_yaws=(-60.0, 0.0, 60.0), **kw)


def test_rig_model_keeps_the_state_dict_and_loads_single_camera_checkpoints():
    torch.manual_seed(0)
    single = dcf.ObjectDetection_DCF(dcf.geometry.carla_config(fusion_scales=(1, 3)))
    rig = dcf.ObjectDetection_DCF(_rig_cfg())
    assert list(single.state_dict().keys()) == list(rig.state_dict().keys())
    assert [n for n, _ in single.named_modules()] == [n for n, _ in rig.named_modules()]
    assert rig.cameras == 3 and single.cameras is None
    assert torch.equal(rig.rig_calib, torch.from_numpy(dcf.geometry.camera_rig((-60.0, 0.0, 60.0))))
    rig.load_state_dict(single.state_dict(), strict=True)
    assert all(torch.equal(a, b) for a, b in zip(single.state_dict().values(), rig.state_dict().values()))


def test_rig_model_input_errors():
    m = dcf.ObjectDetection_DCF(_rig_cfg()).eval()
    x_lidar = torch.zeros(1, 32, 384, 256)
    pts, cnt = torch.zeros(1, 16, 3), torch.tensor([16])
    with pytest.raises(ValueError, match="projected_loc_uv"):
        m(x_lidar, torch.zeros(1, 3, 3, 480, 640, dtype=torch.uint8), pointcloud_raw=pts, num_points_raw=cnt,
          projected_loc_uv=torch.zeros(1, 16, 2))
    with pytest.raises(ValueError, match="x_image"):
        m(x_lidar, torch.zeros(1, 3, 480, 640, dtype=torch.uint8), pointcloud_raw=pts, num_points_raw=cnt)
    single = dcf.ObjectDetection_DCF(dcf.geometry.carla_config(fusion_scales=(1,))).eval()
    with pytest.raises(ValueError, match="camera_calib"):
        single(x_lidar, None, camera_calib=torch.zeros(1, 3, 4, 3))
