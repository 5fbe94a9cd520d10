"""CPU: the surface of camera rigs whose cameras differ in map and image size that needs no GPU -- cf_camera_map and the
cf_point_gather_rig* entry points are declared, exported and bound with the C layout, malformed camera lists are refused
before anything is launched, and geometry.camera_rig scales each camera's intrinsics to its image."""
import ctypes
import os
import re

import numpy as np
import pytest
import torch

import dcf_b200 as dcf

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
NEW = ("cf_gather_rig_workspace_bytes", "cf_point_gather_rig", "cf_point_gather_rig_bf16", "cf_point_gather_rig_bwd",
       "cf_point_gather_rig_bwd_det_workspace_bytes", "cf_point_gather_rig_bwd_det")
YAWS = (-60.0, 0.0, 60.0)


def _header():
    return open(os.path.join(ROOT, "include", "cf_b200.h")).read()


def test_header_declares_the_descriptor_and_the_entry_points():
    h = _header()
    m = re.search(r"typedef struct cf_camera_map \{(.*?)\} cf_camera_map;", h, flags=re.S)
    assert m, "cf_camera_map is not declared"
    body = re.sub(r"/\*.*?\*/", "", m.group(1), flags=re.S)
    fields = re.findall(r"(\w+)\s*;", body.replace(",", "; "))
    assert fields == ["d_map", "sb", "sc", "sh", "sw", "Hf", "Wf", "img_w", "img_h"], fields
    lib = ctypes.CDLL(dcf.SO_PATH)
    for name in NEW:
        assert re.search(rf"CF_API\s+[\w\s\*]+?\b{name}\s*\(", h), name
        assert hasattr(lib, name) and name in dcf._lib.SIGNATURES, name
    # descriptors go in by pointer, never by value
    for name in NEW:
        assert any(t is ctypes.POINTER(dcf._lib.CameraMap) for t in dcf._lib.SIGNATURES[name][1]), name
    assert dcf._lib.SIGNATURES["cf_point_gather_rig_bf16"] == dcf._lib.SIGNATURES["cf_point_gather_rig"]


def test_ctypes_structure_has_the_c_layout():
    S = dcf._lib.CameraMap
    # void* (8), 4 x int64 (32), 2 x int32 (8), 2 x float (8): 56 bytes, no padding on LP64
    assert ctypes.sizeof(S) == 56 and ctypes.alignment(S) == 8
    offsets = {f: getattr(S, f).offset for f, _ in S._fields_}
    assert offsets == dict(d_map=0, sb=8, sc=16, sh=24, sw=32, Hf=40, Wf=44, img_w=48, img_h=52)


def _cams(*shapes, sc_one=False, Ci=8, B=2):
    out = []
    for Hf, Wf in shapes:
        stride = (Hf * Wf * Ci, 1, Wf * Ci, Ci) if sc_one else (Ci * Hf * Wf, Hf * Wf, Wf, 1)
        out.append(dcf._lib.CameraMap(0, *stride, Hf, Wf, 640.0, 480.0))
    return (dcf._lib.CameraMap * len(out))(*out)


def test_workspace_sizes():
    L = dcf.load()
    # channel-major cameras are re-laid one after the other (fp32 size); channels_last cameras are read in place
    cams = _cams((120, 160), (88, 160), (160, 120))
    assert L.cf_gather_rig_workspace_bytes(2, 3, 8, cams) == 2 * 8 * 4 * (120 * 160 + 88 * 160 + 160 * 120)
    assert L.cf_gather_rig_workspace_bytes(2, 3, 8, _cams((120, 160), (88, 160), (160, 120), sc_one=True)) == 0
    # equal cameras: the workspace of the (B,M,Ci,Hf,Wf) rig
    assert (L.cf_gather_rig_workspace_bytes(2, 3, 8, _cams((30, 40), (30, 40), (30, 40)))
            == L.cf_gather_multi_workspace_bytes(2, 3, 8, 30, 40, 1200))
    assert (L.cf_point_gather_rig_bwd_det_workspace_bytes(2, 3, 1000, _cams((30, 40), (30, 40), (30, 40)))
            == L.cf_point_gather_multi_bwd_det_workspace_bytes(2, 3, 1000, 30, 40))
    # a larger camera needs more list space than the smaller ones
    assert (L.cf_point_gather_rig_bwd_det_workspace_bytes(2, 3, 1000, _cams((60, 80), (30, 40), (30, 40)))
            > L.cf_point_gather_multi_bwd_det_workspace_bytes(2, 3, 1000, 30, 40))


def _lists():
    maps = [torch.zeros(2, 8, 6, 8), torch.zeros(2, 8, 4, 8), torch.zeros(2, 8, 8, 6)]
    return maps, torch.zeros(2, 16, 3), torch.tensor([16, 16]), torch.zeros(3, 4, 3), [(640, 480), (640, 352), (480, 640)]


def test_malformed_camera_lists_raise_before_any_launch():
    ops = dcf.ops
    maps, pts, cnt, cal, sizes = _lists()
    before = dcf.load().cf_launch_count()
    for fn, extra in ((ops.point_gather_rig, ()), (ops.point_gather_rig_bwd, None)):
        def call(m, c=cal, s=sizes):
            if extra is None:
                return fn(torch.zeros(2, 16, 8), m, pts, cnt, c, s)
            return fn(m, pts, cnt, c, s)
        with pytest.raises(ValueError, match="cameras"):
            call([])
        with pytest.raises(ValueError, match="cameras"):
            call([maps[0]] * 9, torch.zeros(9, 4, 3), sizes * 3)
        with pytest.raises(ValueError, match="calib"):
            call(maps[:2], s=sizes[:2])                                       # 3 calibrations for 2 cameras
        with pytest.raises(ValueError, match="Ci"):
            call([maps[0], torch.zeros(2, 12, 4, 8), maps[2]])              # Ci mismatch
        with pytest.raises(ValueError, match="B=2"):
            call([maps[0], torch.zeros(1, 8, 4, 8), maps[2]])               # batch mismatch
        with pytest.raises(TypeError, match="one dtype"):
            call([maps[0], maps[1].to(torch.bfloat16), maps[2]])            # mixed dtypes
        with pytest.raises(TypeError):
            call([maps[0], maps[1].half(), maps[2]])                        # not a map dtype
        with pytest.raises(ValueError, match="img_sizes"):
            call(maps, s=sizes[:2])                                         # one image size short
        with pytest.raises(ValueError, match="img_sizes"):
            call(maps, s=[(640, 480), (640, 0), (480, 640)])
        with pytest.raises(ValueError, match="multiple of 4"):
            call([torch.zeros(2, 6, 4, 4)] * 3)
        with pytest.raises(ValueError, match=r"\(B,Ci,Hf,Wf\)"):
            call([maps[0], maps[1][0], maps[2]])
        with pytest.raises(TypeError, match="list"):
            call(torch.zeros(2, 3, 8, 6, 8))
    # FrameContext.gather refuses a list with uv, or without calib, before touching its state
    with pytest.raises(ValueError, match="uv"):
        dcf.FrameContext.gather(object(), maps, calib=cal, uv=torch.zeros(2, 16, 2))
    with pytest.raises(ValueError, match="calib"):
        dcf.FrameContext.gather(object(), maps)
    assert dcf.load().cf_launch_count() == before


def test_camera_rig_at_the_reference_size_is_unchanged():
    G = dcf.geometry
    for yaws in ((0.0,), YAWS, (-150.0, -90.0, -30.0, 30.0, 90.0, 150.0)):
        ref = G.camera_rig(yaws)
        got = G.camera_rig(yaws, [(640, 480)] * len(yaws))
        assert got.dtype == np.float32 and np.array_equal(got.view(np.uint32), ref.view(np.uint32))
    with pytest.raises(ValueError, match="image_sizes"):
        G.camera_rig(YAWS, [(640, 480)] * 2)
    with pytest.raises(ValueError, match="image_sizes"):
        G.camera_rig(YAWS, [(640, 480), (0, 480), (640, 480)])


@pytest.mark.parametrize("size", [(640, 352), (480, 640), (1920, 1280), (1920, 886), (320, 240)])
def test_scaled_camera_projects_to_its_image(size):
    """Camera m at w_m x h_m sees point p at (u * w_m/640, v * h_m/480), (u, v) the 640 x 480 camera's projection."""
    G = dcf.geometry
    w, h = size
    rng = np.random.default_rng(7)
    n = 2000
    az = np.deg2rad(60.0) + rng.uniform(-0.7, 0.7, n)
    r = rng.uniform(3.0, 70.0, n)
    p = np.stack([r * np.cos(az), r * np.sin(az), rng.uniform(-2.3, 0.7, n)], axis=1).astype(np.float32)
    ref = G.camera_rig(YAWS)[2]
    got = G.camera_rig(YAWS, [(640, 480), (640, 480), size])[2]
    assert np.array_equal(G.camera_rig(YAWS, [(640, 480), (640, 480), size])[:2], G.camera_rig(YAWS)[:2])

    def proj(crt):
        q = np.concatenate([p, np.ones((n, 1), np.float32)], axis=1) @ crt   # float32 throughout
        return q[:, :2] / q[:, 2:], q[:, 2]

    (uv_ref, w_ref), (uv, w_) = proj(ref), proj(got)
    assert (w_ > 0).all() and np.array_equal(w_.view(np.uint32), w_ref.view(np.uint32))   # the depth row is not scaled
    want = uv_ref * np.array([w / 640.0, h / 480.0], np.float32)
    # float32 rounding of the scaled entries and of the projection: a few ulps of the pixel coordinate
    assert np.abs(uv - want).max() <= 8 * np.finfo(np.float32).eps * max(1.0, float(np.abs(want).max()))


def test_rig_model_with_image_sizes_keeps_the_state_dict():
    torch.manual_seed(0)
    sizes = [[640, 480], [640, 352], [480, 640]]
    single = dcf.ObjectDetection_DCF(dcf.geometry.carla_config(fusion_scales=(1, 3)))
    rig = dcf.ObjectDetection_DCF(dcf.geometry.carla_config(fusion_scales=(1, 3), fusion_camera_yaws=YAWS,
                                                            fusion_camera_image_sizes=sizes))
    assert list(single.state_dict().keys()) == list(rig.state_dict().keys())
    assert torch.equal(rig.rig_calib, torch.from_numpy(dcf.geometry.camera_rig(YAWS, sizes)))
    assert rig.camera_sizes == [(640.0, 480.0), (640.0, 352.0), (480.0, 640.0)]
    rig.load_state_dict(single.state_dict(), strict=True)
    plain = dcf.ObjectDetection_DCF(dcf.geometry.carla_config(fusion_scales=(1,), fusion_camera_yaws=YAWS))
    assert torch.equal(plain.rig_calib, torch.from_numpy(dcf.geometry.camera_rig(YAWS)))
    with pytest.raises(ValueError, match="fusion_camera_image_sizes"):
        dcf.ObjectDetection_DCF(dcf.geometry.carla_config(fusion_camera_yaws=YAWS, fusion_camera_image_sizes=sizes[:2]))
    with pytest.raises(ValueError, match="x_image"):
        rig.eval()(torch.zeros(1, 32, 384, 256), [torch.zeros(1, 3, 480, 640, dtype=torch.uint8)] * 2,
                   pointcloud_raw=torch.zeros(1, 16, 3), num_points_raw=torch.tensor([16]))
