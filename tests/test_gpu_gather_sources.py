"""GPU: where the camera gather takes its map coordinates (uv, the host CRT_tensor, a rig of device calibrations).

Points BEHIND the reference camera (w > 0 under CRT_tensor) whose mirrored projection lands inside the map tell the
sources apart: the reference's projection divides by w whatever its sign, so cf_point_gather with h_calib, or with those
points' uv, gathers them exactly as the oracle's project_points + gather_points do, while a rig camera, which sees only
w > 0 under its own (negated) calibration, gives them zeros.  The same holds for both adjoints."""
import numpy as np
import pytest
import torch

from _util import dev, rel_err

pytestmark = pytest.mark.gpu
BF = torch.bfloat16
SIZE = (640.0, 480.0)


def _w(pts, crt):
    """Third projected component in fp32, in the kernels' operation order."""
    f = np.float32
    return ((pts[..., 0] * f(crt[0, 2]) + pts[..., 1] * f(crt[1, 2])) + pts[..., 2] * f(crt[2, 2])) + f(crt[3, 2])


@pytest.fixture(scope="module")
def mirrored(dcf, oracle):
    """The standard workload with every other point reflected through the camera centre: w changes sign, u and v stay."""
    wl = dcf.synthetic.make_workload(dict(dcf.synthetic.workload("yaml"), batch=2, scales=(1,)), seed=11, c_img=64,
                                     img_hw=(30, 41))
    crt = wl["calib"]
    R, t = crt[:3].astype(np.float64), crt[3].astype(np.float64)
    centre = -t @ np.linalg.inv(R)
    pts = wl["points"].copy()
    pts[:, 1::2] = (2.0 * centre - pts[:, 1::2].astype(np.float64)).astype(np.float32)
    img = wl["img_feat"]
    Hf, Wf = img.shape[2:]
    uv = np.zeros(pts.shape[:2] + (2,), np.float32)
    behind = np.zeros(pts.shape[:2], bool)
    for b in range(pts.shape[0]):
        n = int(wl["num_points"][b])
        uv[b, :n] = oracle.project_points(pts[b, :n], crt)
        uf = (uv[b, :n, 0] + np.float32(0.5)) * (np.float32(Wf) / np.float32(SIZE[0])) - np.float32(0.5)
        vf = (uv[b, :n, 1] + np.float32(0.5)) * (np.float32(Hf) / np.float32(SIZE[1])) - np.float32(0.5)
        behind[b, :n] = (_w(pts[b, :n], crt) > 0) & (uf > -1) & (uf < Wf) & (vf > -1) & (vf < Hf)
        assert behind[b].sum() > 100 and behind[b, 1:n:2].mean() > 0.9, "mirrored points project into the map"
        assert not (_w(pts[b, 0:n:2], crt) > 0).any(), "the other points are in front of the camera"
    return dict(points=pts, num_points=wl["num_points"], img=img, calib=crt, uv=uv, behind=behind)


def _oracle_gather(oracle, d, img):
    out = np.zeros(d["points"].shape[:2] + (img.shape[1],), np.float32)
    for b in range(out.shape[0]):
        n = int(d["num_points"][b])
        out[b, :n] = oracle.gather_points(img[b], d["uv"][b, :n], SIZE[0], SIZE[1])
    return out


@pytest.mark.parametrize("channels_last", (False, True))
@pytest.mark.parametrize("dtype", (torch.float32, BF))
def test_points_behind_the_reference_camera_are_gathered_from_crt_and_uv(dcf, oracle, mirrored, dtype, channels_last):
    d, ops = mirrored, dcf.ops
    img = dev(d["img"]).to(dtype)
    if channels_last:
        img = img.contiguous(memory_format=torch.channels_last)
    ref = _oracle_gather(oracle, d, img.float().cpu().numpy())
    assert np.abs(ref[d["behind"]]).sum(axis=-1).min() > 0
    pts, cnt = dev(d["points"]), dev(d["num_points"])
    by_crt, _ = ops.point_gather(img, pts, cnt, calib=d["calib"], img_size=SIZE)
    by_uv, _ = ops.point_gather(img, pts, cnt, uv=dev(d["uv"]), img_size=SIZE)
    assert rel_err(by_crt.cpu().numpy(), ref) <= 1e-6
    assert rel_err(by_uv.cpu().numpy(), ref) <= 1e-6
    # a rig camera sees w > 0 under its own calibration only: nothing behind the reference camera
    rig = torch.from_numpy(-d["calib"]).cuda().reshape(1, 4, 3)
    by_rig, _ = ops.point_gather_multi(img.unsqueeze(1), pts, cnt, rig, img_size=SIZE)
    behind = torch.from_numpy(d["behind"]).cuda()
    assert not by_rig[behind].any()
    assert torch.equal(by_rig[~behind], by_crt[~behind])


@pytest.mark.parametrize("deterministic", (False, True))
def test_adjoints_reach_the_map_through_crt_and_uv_only(dcf, mirrored, deterministic):
    d, ops = mirrored, dcf.ops
    img = dev(d["img"])
    pts, cnt = dev(d["points"]), dev(d["num_points"])
    behind = torch.from_numpy(d["behind"]).cuda()
    gen = torch.Generator(device="cuda").manual_seed(7)
    g = torch.randn(pts.shape[:2] + (img.shape[1],), device="cuda", generator=gen) * behind[..., None]
    feat, _ = ops.point_gather(img, pts, cnt, calib=d["calib"], img_size=SIZE)
    lhs = float((feat.double() * g.double()).sum())
    for kw in (dict(calib=d["calib"]), dict(uv=dev(d["uv"]))):
        dimg = ops.point_gather_bwd(g, img, pts, cnt, img_size=SIZE, deterministic=deterministic, **kw)
        assert float(dimg.abs().sum()) > 0
        rhs = float((img.double() * dimg.double()).sum())
        assert abs(lhs - rhs) <= 1e-5 * max(abs(lhs), 1.0), (kw.keys(), lhs, rhs)
    rig = torch.from_numpy(-d["calib"]).cuda().reshape(1, 4, 3)
    dimg = ops.point_gather_multi_bwd(g, img.unsqueeze(1), pts, cnt, rig, img_size=SIZE, deterministic=deterministic)
    assert not dimg.any()
