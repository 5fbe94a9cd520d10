"""GPU: multi-camera continuous fusion (cf_point_gather_multi*, FrameContext with a 5-D map, FusionRunner(cameras=M), the
rig model).

One camera with the negated reference calibration gives the bits of the single-camera path; three cameras match a
restatement built from the CPU oracle's projection and gather; per-frame calibrations equal single-frame calls; the
backward is the adjoint (fixed-order path reproducible bit for bit); a CUDA-graph replay reads calibrations from the
device."""
import math

import numpy as np
import pytest
import torch

from _util import dev, rel_err

pytestmark = pytest.mark.gpu
BF = torch.bfloat16
YAWS = (-60.0, 0.0, 60.0)
SIZE = (640.0, 480.0)


def _sweep_points(seed, cfg, batch=2, n_beams=32, n_az=1800, sensor_h=2.2):
    """Full-azimuth LiDAR sweep (ground rings, returns above the ground, near-field returns) through the range filter only:
    no camera filter, so points lie beside the front camera's view and below every camera's view too."""
    N = int(cfg["max_num_pc"])
    pts = np.zeros((batch, N, 3), np.float32)
    cnt = np.zeros((batch,), np.int64)
    d = np.float32(cfg["delta"])
    for b in range(batch):
        rng = np.random.default_rng(seed * 100 + b)
        elev = np.deg2rad(np.linspace(-24.8, -1.0, n_beams))[:, None] + rng.normal(0.0, 2e-4, (n_beams, n_az))
        az = rng.uniform(-math.pi, math.pi, (n_beams, n_az))
        r = sensor_h / np.tan(-elev) * (1.0 + rng.normal(0.0, 2e-3, elev.shape))
        near = rng.random(elev.shape) < 0.05     # near-field returns, below every camera's vertical view
        r = np.where(near, rng.uniform(0.5, 2.0, elev.shape), r)
        z = -sensor_h + np.where(rng.random(elev.shape) < 0.2, rng.uniform(0.0, 2.5, elev.shape), 0.0)
        p = np.stack([(r * np.cos(az)).ravel(), (r * np.sin(az)).ravel(), z.ravel()], axis=1).astype(np.float32)
        keep = ((p[:, 0] > np.float32(cfg["lidar_x_min"])) & (p[:, 0] < np.float32(cfg["lidar_x_max"]) - d) &
                (p[:, 1] > np.float32(cfg["lidar_y_min"])) & (p[:, 1] < np.float32(cfg["lidar_y_max"]) - d) &
                (p[:, 2] > np.float32(cfg["lidar_z_min"])) & (p[:, 2] < np.float32(cfg["lidar_z_max"]) - d))
        p = p[keep]
        if p.shape[0] > N:
            p = p[np.sort(rng.choice(p.shape[0], N, replace=False))]
        pts[b, :p.shape[0]], cnt[b] = p, p.shape[0]
    return pts, cnt


def _w(pts, crt):
    """Third projected component in fp32, in the kernels' operation order."""
    f = np.float32
    return ((pts[:, 0] * f(crt[0, 2]) + pts[:, 1] * f(crt[1, 2])) + pts[:, 2] * f(crt[2, 2])) + f(crt[3, 2])


def _restated_rig_gather(O, img, pts, n, rig):
    """Mean over the visible cameras, in camera order, of the oracle's projection + bilinear gather.  img (M,Ci,Hf,Wf)."""
    M, Ci, Hf, Wf = img.shape
    acc = np.zeros((n, Ci), np.float32)
    nvis = np.zeros((n,), np.int64)
    for m in range(M):
        uv = O.project_points(pts[:n], rig[m])
        uf = (uv[:, 0] + np.float32(0.5)) * (np.float32(Wf) / np.float32(SIZE[0])) - np.float32(0.5)
        vf = (uv[:, 1] + np.float32(0.5)) * (np.float32(Hf) / np.float32(SIZE[1])) - np.float32(0.5)
        vis = (_w(pts[:n], rig[m]) > 0) & (uf > -1) & (uf < Wf) & (vf > -1) & (vf < Hf)
        g = O.gather_points(img[m], uv, SIZE[0], SIZE[1])
        acc += np.where(vis[:, None], g, np.float32(0))
        nvis += vis
    return acc / np.maximum(nvis, 1)[:, None].astype(np.float32), nvis


@pytest.fixture(scope="module")
def std(dcf):
    """The standard synthetic workload (camera-filtered points) with a 64-channel map."""
    return dcf.synthetic.make_workload(dict(dcf.synthetic.workload("yaml"), batch=2, scales=(1,)), seed=11, c_img=64,
                                       img_hw=(30, 41))


@pytest.fixture(scope="module")
def sweep(dcf):
    cfg = dcf.geometry.carla_config(voxel_length=384, voxel_width=256, max_num_pc=20000)
    pts, cnt = _sweep_points(5, cfg)
    rng = np.random.default_rng(17)
    img = rng.standard_normal((2, 3, 32, 120, 160), dtype=np.float32)   # the camera stream's stride-4 map of a 640x480 image
    return dict(config=cfg, points=pts, num_points=cnt, img=img)


def _layout(x, channels_last):
    """(B,M,Ci,Hf,Wf) view of per-camera channels_last maps (what the model's camera stream emits) or a dense NCHW stack."""
    if not channels_last:
        return x.contiguous()
    B, M = x.shape[:2]
    return x.flatten(0, 1).contiguous(memory_format=torch.channels_last).unflatten(0, (B, M))


# ---------------------------------------------------------------------------------------------------- 1. M = 1
@pytest.mark.parametrize("channels_last", (False, True))
@pytest.mark.parametrize("dtype", (torch.float32, BF))
def test_one_camera_gives_the_bits_of_the_single_camera_path(dcf, std, dtype, channels_last):
    ops, wl = dcf.ops, std
    crt = wl["calib"]
    for b in range(2):
        n = int(wl["num_points"][b])
        assert (_w(wl["points"][b, :n], -crt) > 0).all(), "every point of the standard workload is in front of the camera"
    pts, cnt = dev(wl["points"]), dev(wl["num_points"])
    img4 = dev(wl["img_feat"]).to(dtype)
    if channels_last:
        img4 = img4.contiguous(memory_format=torch.channels_last)
    img5 = img4.unsqueeze(1)
    rig = torch.from_numpy(-crt).cuda().reshape(1, 4, 3)
    ref, _ = ops.point_gather(img4, pts, cnt, calib=crt, img_size=SIZE)
    got, _ = ops.point_gather_multi(img5, pts, cnt, rig, img_size=SIZE)
    assert torch.equal(got, ref)
    g = torch.randn(ref.shape, device="cuda", generator=torch.Generator(device="cuda").manual_seed(3))
    ref_d = ops.point_gather_bwd(g, img4, pts, cnt, calib=crt, img_size=SIZE, deterministic=True)
    got_d = ops.point_gather_multi_bwd(g, img5, pts, cnt, rig, img_size=SIZE, deterministic=True)
    assert got_d.dtype == dtype and got_d.stride() == img5.stride() and torch.equal(got_d[:, 0], ref_d)
    # float atomics sum in arrival order: the atomic paths agree to rounding in general ...
    ref_a = ops.point_gather_bwd(g, img4, pts, cnt, calib=crt, img_size=SIZE)
    got_a = ops.point_gather_multi_bwd(g, img5, pts, cnt, rig, img_size=SIZE)
    assert rel_err(got_a[:, 0].float().cpu(), ref_a.float().cpu()) <= (1e-6 if dtype == torch.float32 else 1e-2)
    # ... and bit for bit where every pixel receives at most one product (one point per frame)
    one = torch.ones(2, dtype=torch.int64, device="cuda")
    assert torch.equal(ops.point_gather_multi_bwd(g, img5, pts, one, rig, img_size=SIZE)[:, 0],
                       ops.point_gather_bwd(g, img4, pts, one, calib=crt, img_size=SIZE))


# ---------------------------------------------------------------------------------------------------- 2. M = 3
@pytest.mark.parametrize("channels_last", (False, True))
def test_three_cameras_match_the_restatement(dcf, oracle, sweep, channels_last):
    rig = dcf.geometry.camera_rig(YAWS)
    img = _layout(dev(sweep["img"]), channels_last)
    got, _ = dcf.ops.point_gather_multi(img, dev(sweep["points"]), dev(sweep["num_points"]), torch.from_numpy(rig).cuda(),
                                        img_size=SIZE)
    got = got.cpu().numpy()
    seen = np.zeros(4, np.int64)
    for b in range(2):
        n = int(sweep["num_points"][b])
        ref, nvis = _restated_rig_gather(oracle, sweep["img"][b], sweep["points"][b], n, rig)
        assert rel_err(got[b, :n], ref) <= 1e-6
        assert not got[b, n:].any() and not got[b, :n][nvis == 0].any()
        seen += np.bincount(nvis, minlength=4)[:4]
    assert seen[0] > 0 and seen[1] > 0 and seen[2] > 0, seen


# ---------------------------------------------------------------------------------------------------- 3. per frame
def test_per_frame_calibration_equals_single_frame_calls(dcf, sweep):
    G, ops = dcf.geometry, dcf.ops
    rigs = torch.from_numpy(np.stack([G.camera_rig(YAWS), G.camera_rig((-30.0, 20.0, 90.0))])).cuda()
    for dtype, cl in ((torch.float32, False), (BF, True)):
        img = _layout(dev(sweep["img"]).to(dtype), cl)
        pts, cnt = dev(sweep["points"]), dev(sweep["num_points"])
        got, _ = ops.point_gather_multi(img, pts, cnt, rigs, img_size=SIZE)
        for b in range(2):
            one, _ = ops.point_gather_multi(img[b:b + 1], pts[b:b + 1], cnt[b:b + 1], rigs[b], img_size=SIZE)
            assert torch.equal(got[b:b + 1], one)
        # an (M,4,3) rig is every frame's calibration
        shared, _ = ops.point_gather_multi(img, pts, cnt, rigs[0], img_size=SIZE)
        assert torch.equal(shared, ops.point_gather_multi(img, pts, cnt, rigs[0].expand(2, 3, 4, 3).contiguous(),
                                                          img_size=SIZE)[0])


# ---------------------------------------------------------------------------------------------------- 4. backward
@pytest.mark.parametrize("channels_last", (False, True))
def test_backward_is_the_adjoint_and_reproducible(dcf, sweep, channels_last):
    ops = dcf.ops
    rig = torch.from_numpy(dcf.geometry.camera_rig(YAWS)).cuda()
    x = _layout(dev(sweep["img"]), channels_last)
    pts, cnt = dev(sweep["points"]), dev(sweep["num_points"])
    g = torch.randn((2, pts.shape[1], 32), device="cuda", generator=torch.Generator(device="cuda").manual_seed(9))
    d1 = ops.point_gather_multi_bwd(g, x, pts, cnt, rig, img_size=SIZE, deterministic=True)
    d2 = ops.point_gather_multi_bwd(g, x, pts, cnt, rig, img_size=SIZE, deterministic=True)
    assert torch.equal(d1, d2) and d1.stride() == x.stride()
    a = ops.point_gather_multi_bwd(g, x, pts, cnt, rig, img_size=SIZE)
    assert float((a - d1).double().norm() / d1.double().norm()) <= 1e-6
    f, _ = ops.point_gather_multi(x, pts, cnt, rig, img_size=SIZE)
    lhs = float((f.double() * g.double()).sum())
    rhs = float((x.double() * d1.double()).sum())
    assert abs(lhs - rhs) <= 1e-5 * max(abs(lhs), 1.0), (lhs, rhs)
    # bf16 maps: the fp32 gradient of the widened map, rounded once
    x16 = x.to(BF)
    d16 = ops.point_gather_multi_bwd(g, x16, pts, cnt, rig, img_size=SIZE, deterministic=True)
    assert d16.dtype == BF and d16.stride() == x16.stride()
    assert torch.equal(d16, ops.point_gather_multi_bwd(g, x16.float(), pts, cnt, rig, img_size=SIZE, deterministic=True).to(BF))


# ---------------------------------------------------------------------------------------------------- 5. layer, model
@pytest.fixture
def deterministic():
    before = torch.are_deterministic_algorithms_enabled()
    torch.use_deterministic_algorithms(True)
    yield
    torch.use_deterministic_algorithms(before)


def _frames(dcf, sweep):
    grid = dcf.ops.BucketGrid(*dcf.geometry.bucket_grid(sweep["config"]))
    return dcf.FrameContext(dev(sweep["points"]), dev(sweep["num_points"]), grid)


def test_layer_on_a_rig_trains_reproducibly(dcf, sweep, deterministic):
    G = dcf.geometry
    geom = G.scale_geometry(sweep["config"], 1)
    rig = torch.from_numpy(G.camera_rig(YAWS)).cuda()
    torch.manual_seed(4)
    layer = dcf.ContinuousFusion(32, 32, k=3, radius=2.0, geom=geom, mode="fp32").cuda()
    bev0 = torch.randn(2, 32, 384, 256, device="cuda")
    grads = []
    for _ in range(2):
        layer.zero_grad(set_to_none=True)
        img = _layout(dev(sweep["img"]), True).requires_grad_(True)
        bev = bev0.clone().requires_grad_(True)
        frames = _frames(dcf, sweep)
        with pytest.raises(ValueError, match="uv"):
            frames.gather(img, calib=rig, uv=torch.zeros(2, frames.N, 2, device="cuda"))
        frames.gather(img, calib=rig, img_size=SIZE)
        out = layer(bev, frames=frames)
        (out * out).sum().backward()
        grads.append([img.grad.clone(), bev.grad.clone()] + [p.grad.clone() for p in layer.parameters()])
    assert grads[0][0].abs().sum() > 0
    assert all(torch.equal(a, b) for a, b in zip(*grads))


def test_points_outside_the_front_camera_get_features_from_the_rig(dcf, sweep):
    G = dcf.geometry
    crt = G.calibration_crt()
    img = dev(sweep["img"])
    with torch.no_grad():
        single = _frames(dcf, sweep).gather(img[:, 1].contiguous(), calib=crt, img_size=SIZE).cpu().numpy()
        rig = _frames(dcf, sweep).gather(img, calib=torch.from_numpy(G.camera_rig(YAWS)).cuda(), img_size=SIZE).cpu().numpy()
    total = 0
    for b in range(2):
        n = int(sweep["num_points"][b])
        p = sweep["points"][b, :n].astype(np.float64)
        q = np.concatenate([p, np.ones((n, 1))], axis=1) @ crt.astype(np.float64)
        u = q[:, 0] / q[:, 2]
        out = (q[:, 2] >= 0) | (u < -8.0) | (u > 648.0)     # behind the front camera, or beside its image by a margin
        assert out.sum() > 100
        assert not single[b, :n][out].any()
        nz = np.abs(rig[b, :n][out]).sum(axis=1) > 0
        assert nz.mean() > 0.5, nz.mean()
        total += nz.sum()
    assert total > 0


def _rig_model(dcf, **kw):
    cfg = dcf.geometry.carla_config(fusion_scales=(1, 3), fusion_k=3, fusion_camera_yaws=YAWS, **kw)
    torch.manual_seed(0)
    return cfg, dcf.ObjectDetection_DCF(cfg).cuda().eval()


@pytest.mark.parametrize("amp", (False, True))
def test_rig_model_inference_and_train_step(dcf, sweep, amp):
    cfg, model = _rig_model(dcf)
    x_lidar = torch.rand(2, 32, 384, 256, device="cuda")
    x_image = torch.randint(0, 255, (2, 3, 3, 480, 640), device="cuda", dtype=torch.uint8)
    kw = dict(pointcloud_raw=dev(sweep["points"]), num_points_raw=dev(sweep["num_points"]))
    with torch.no_grad(), torch.autocast("cuda", dtype=BF, enabled=amp):
        pred = model(x_lidar, x_image, **kw)
        pred2 = model(x_lidar, x_image, camera_calib=model.rig_calib.expand(2, 3, 4, 3), **kw)
    assert pred.shape == (2, 32, 96, 64) and bool(torch.isfinite(pred.float()).all())
    assert torch.equal(pred, pred2)
    model.zero_grad(set_to_none=True)
    with torch.autocast("cuda", dtype=BF, enabled=amp):
        loss = model(x_lidar, x_image, **kw).float().square().mean()
    loss.backward()
    assert bool(torch.isfinite(loss))
    grads = {n: p.grad for n, p in model.named_parameters()}
    assert all(g is None or bool(torch.isfinite(g).all()) for g in grads.values())
    for n in ("fusion.group1.fc1.weight", "fusion.group3.fc1.weight", "image_backbone.stem.0.weight"):
        assert grads[n] is not None and float(grads[n].abs().sum()) > 0, n


def test_single_camera_checkpoint_loads_strictly(dcf):
    single = dcf.ObjectDetection_DCF(dcf.geometry.carla_config(fusion_scales=(1, 3), fusion_k=3)).cuda()
    _, rig = _rig_model(dcf)
    rig.load_state_dict(single.state_dict(), strict=True)


# ---------------------------------------------------------------------------------------------------- 6. FusionRunner
def test_fusion_runner_with_a_rig_reads_calibrations_from_the_device(dcf, sweep):
    G = dcf.geometry
    cfg = sweep["config"]
    shapes = dcf.synthetic.scale_shapes(cfg)[:2]
    torch.manual_seed(5)
    layers = [dcf.ContinuousFusion(32, C, k=3, radius=2.0, geom=G.scale_geometry(cfg, s), mode="fp32").cuda().eval()
              for (C, _, _), s in zip(shapes, (1, 2))]
    grid = dcf.ops.BucketGrid(*G.bucket_grid(cfg))
    runner = dcf.FusionRunner(layers, grid, 2, sweep["points"].shape[1], (32, 120, 160), shapes, calib=G.camera_rig(YAWS),
                              img_size=SIZE, inplace=False, cameras=3)
    assert tuple(runner.img_feat.shape) == (2, 3, 32, 120, 160) and tuple(runner.calib.shape) == (2, 3, 4, 3)
    runner.points.copy_(dev(sweep["points"]))
    runner.num_points.copy_(dev(sweep["num_points"]))
    runner.img_feat.copy_(dev(sweep["img"]))
    gen = torch.Generator(device="cuda").manual_seed(6)
    bevs = [torch.randn((2,) + tuple(s), device="cuda", generator=gen) for s in shapes]
    for d, b in zip(runner.bevs, bevs):
        d.copy_(b)
    for yaws in (YAWS, (-90.0, -20.0, 45.0)):
        rig = torch.from_numpy(G.camera_rig(yaws)).cuda()
        runner.calib.copy_(rig.expand(2, 3, 4, 3))          # no recapture
        outs = [o.clone() for o in runner()]
        frames = _frames(dcf, sweep)
        with torch.no_grad():
            frames.gather(dev(sweep["img"]), calib=rig, img_size=SIZE)
            ref = dcf.fuse_scales(frames, layers, bevs)
        torch.cuda.synchronize()
        assert all(torch.equal(o, r) for o, r in zip(outs, ref)), yaws
