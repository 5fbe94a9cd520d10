"""GPU: camera rigs whose cameras differ in map and image size (cf_point_gather_rig*, FrameContext with a list of maps,
FusionRunner with per-camera shapes, the rig model with fusion_camera_image_sizes).

Equal descriptors give the bits of the (B,M,Ci,Hf,Wf) rig; three different cameras match a restatement built from the CPU
oracle; a smaller camera does not count points outside its own map (a zero-padded rig does); the backward is the adjoint
for every map (fixed-order path reproducible bit for bit)."""
import numpy as np
import pytest
import torch
import torch.nn.functional as F

from _util import dev, rel_err
from test_gpu_multicam import _sweep_points, _w

pytestmark = pytest.mark.gpu
BF = torch.bfloat16
YAWS = (-60.0, 0.0, 60.0)
SIZES = [(640.0, 480.0), (640.0, 352.0), (480.0, 640.0)]   # stride-4 maps 120x160, 88x160, 160x120
SHAPES = [(120, 160), (88, 160), (160, 120)]


@pytest.fixture(scope="module")
def sweep(dcf):
    cfg = dcf.geometry.carla_config(voxel_length=384, voxel_width=256, max_num_pc=20000)
    pts, cnt = _sweep_points(7, cfg)
    rng = np.random.default_rng(23)
    maps = [rng.standard_normal((2, 32, h, w), dtype=np.float32) for h, w in SHAPES]
    img5 = rng.standard_normal((2, 3, 32, 120, 160), dtype=np.float32)
    return dict(config=cfg, points=pts, num_points=cnt, maps=maps, img5=img5)


def _layout(t, channels_last):
    return t.contiguous(memory_format=torch.channels_last) if channels_last else t.contiguous()


def _restated(O, maps, pts, n, rig, sizes):
    """Mean over the visible cameras, in camera order, of the oracle's projection + bilinear gather, camera m in its own
    map and image.  maps: M (Ci,Hf_m,Wf_m)."""
    Ci = maps[0].shape[0]
    acc = np.zeros((n, Ci), np.float32)
    nvis = np.zeros((n,), np.int64)
    for m, (img, (iw, ih)) in enumerate(zip(maps, sizes)):
        _, Hf, Wf = img.shape
        uv = O.project_points(pts[:n], rig[m])
        uf = (uv[:, 0] + np.float32(0.5)) * (np.float32(Wf) / np.float32(iw)) - np.float32(0.5)
        vf = (uv[:, 1] + np.float32(0.5)) * (np.float32(Hf) / np.float32(ih)) - np.float32(0.5)
        vis = (_w(pts[:n], rig[m]) > 0) & (uf > -1) & (uf < Wf) & (vf > -1) & (vf < Hf)
        g = O.gather_points(img, uv, iw, ih)
        acc += np.where(vis[:, None], g, np.float32(0))
        nvis += vis
    return acc / np.maximum(nvis, 1)[:, None].astype(np.float32), nvis


# ------------------------------------------------------------------------------------------- 1. equal descriptors
@pytest.mark.parametrize("channels_last", (False, True))
@pytest.mark.parametrize("dtype", (torch.float32, BF))
def test_equal_descriptors_give_the_bits_of_the_rig(dcf, sweep, dtype, channels_last):
    ops = dcf.ops
    rig = torch.from_numpy(dcf.geometry.camera_rig(YAWS)).cuda()
    pts, cnt = dev(sweep["points"]), dev(sweep["num_points"])
    x = dev(sweep["img5"]).to(dtype)
    img5 = x.flatten(0, 1).contiguous(memory_format=torch.channels_last).unflatten(0, (2, 3)) if channels_last else x
    views = [img5[:, m] for m in range(3)]                      # one tensor: the single re-layout launch
    apart = [_layout(img5[:, m].clone(), channels_last) for m in range(3)]   # three tensors: one re-layout per camera
    size = SIZES[0]
    ref, _ = ops.point_gather_multi(img5, pts, cnt, rig, img_size=size)
    for maps in (views, apart):
        got, _ = ops.point_gather_rig(maps, pts, cnt, rig, [size] * 3)
        assert torch.equal(got, ref)
    g = torch.randn(ref.shape, device="cuda", generator=torch.Generator(device="cuda").manual_seed(3))
    ref_d = ops.point_gather_multi_bwd(g, img5, pts, cnt, rig, img_size=size, deterministic=True)
    ref_a = ops.point_gather_multi_bwd(g, img5, pts, cnt, rig, img_size=size)
    for maps in (views, apart):
        got_d = ops.point_gather_rig_bwd(g, maps, pts, cnt, rig, [size] * 3, deterministic=True)
        got_a = ops.point_gather_rig_bwd(g, maps, pts, cnt, rig, [size] * 3)
        for m in range(3):
            assert got_d[m].dtype == dtype and got_d[m].stride() == maps[m].contiguous(
                memory_format=torch.channels_last if channels_last else torch.contiguous_format).stride()
            assert torch.equal(got_d[m], ref_d[:, m])
            # float atomics sum in arrival order: the two atomic results agree to rounding
            a, r = got_a[m].double(), ref_a[:, m].double()
            assert float((a - r).norm() / r.norm()) <= (1e-6 if dtype == torch.float32 else 1e-2)


# ------------------------------------------------------------------------------------------- 2. three sizes
@pytest.mark.parametrize("channels_last", (False, True))
def test_three_sizes_match_the_restatement(dcf, oracle, sweep, channels_last):
    rig = dcf.geometry.camera_rig(YAWS, SIZES)
    maps = [_layout(dev(m), channels_last) for m in sweep["maps"]]
    got, _ = dcf.ops.point_gather_rig(maps, dev(sweep["points"]), dev(sweep["num_points"]), torch.from_numpy(rig).cuda(),
                                      SIZES)
    got = got.cpu().numpy()
    seen = np.zeros(4, np.int64)
    for b in range(2):
        n = int(sweep["num_points"][b])
        ref, nvis = _restated(oracle, [m[b] for m in sweep["maps"]], sweep["points"][b], n, rig, SIZES)
        assert rel_err(got[b, :n], ref) <= 1e-6
        assert not got[b, n:].any() and not got[b, :n][nvis == 0].any()
        seen += np.bincount(nvis, minlength=4)[:4]
    assert seen[0] > 0 and seen[1] > 0 and seen[2] > 0, seen


# ------------------------------------------------------------------------------------------- 3. no padding
def test_a_smaller_camera_does_not_count_points_outside_its_map(dcf, oracle, sweep):
    """Two cameras looking the same way with the same lens: 640x480 (map 120x160) and a 640x352 crop of it (the top 352
    rows, map 88x160).  Zero-padding the crop's map to 120x160 and projecting into a 640x480 image keeps its scale, but
    lets it 'see' the points that land in the padding rows: they are counted in n_vis and zeros are averaged in."""
    sizes = [(640.0, 480.0), (640.0, 352.0)]
    crt = dcf.geometry.camera_rig((0.0, 0.0))                   # the crop keeps the lens and the principal point
    rig = torch.from_numpy(crt).cuda()
    big, small = dev(sweep["maps"][0]), dev(sweep["maps"][1])
    pts, cnt = dev(sweep["points"]), dev(sweep["num_points"])
    got, _ = dcf.ops.point_gather_rig([big, small], pts, cnt, rig, sizes)
    padded = torch.stack([big, F.pad(small, (0, 0, 0, 120 - 88))], 1)
    pad, _ = dcf.ops.point_gather_multi(padded, pts, cnt, rig, img_size=(640.0, 480.0))
    got, pad = got.cpu().numpy(), pad.cpu().numpy()
    total = 0
    for b in range(2):
        n = int(sweep["num_points"][b])
        p = sweep["points"][b, :n]
        ref, _ = _restated(oracle, [big[b].cpu().numpy(), small[b].cpu().numpy()], p, n, crt, sizes)
        assert rel_err(got[b, :n], ref) <= 1e-6
        uv = oracle.project_points(p, crt[1])
        uf = (uv[:, 0] + np.float32(0.5)) * np.float32(0.25) - np.float32(0.5)
        vf = (uv[:, 1] + np.float32(0.5)) * np.float32(0.25) - np.float32(0.5)
        in_pad = (_w(p, crt[1]) > 0) & (uf > -1) & (uf < 160) & (vf >= 88) & (vf < 120)   # the padding rows only
        differ = np.abs(got[b, :n] - pad[b, :n]).max(axis=1) > 0
        # the big camera sees those points too: the padded rig averages its feature with zeros; elsewhere both rigs agree
        assert differ[in_pad].mean() > 0.99, differ[in_pad].mean()
        assert not differ[~in_pad].any()
        total += int(in_pad.sum())
    assert total > 100, total


# ------------------------------------------------------------------------------------------- 4. adjoint
def test_backward_is_the_adjoint_for_every_map(dcf, sweep):
    ops = dcf.ops
    rig = torch.from_numpy(dcf.geometry.camera_rig(YAWS, SIZES)).cuda()
    pts, cnt = dev(sweep["points"]), dev(sweep["num_points"])
    for cl in (False, True):
        xs = [_layout(dev(m), cl) for m in sweep["maps"]]
        g = torch.randn((2, pts.shape[1], 32), device="cuda", generator=torch.Generator(device="cuda").manual_seed(9))
        d1 = ops.point_gather_rig_bwd(g, xs, pts, cnt, rig, SIZES, deterministic=True)
        d2 = ops.point_gather_rig_bwd(g, xs, pts, cnt, rig, SIZES, deterministic=True)
        a = ops.point_gather_rig_bwd(g, xs, pts, cnt, rig, SIZES)
        f, _ = ops.point_gather_rig(xs, pts, cnt, rig, SIZES)
        lhs = float((f.double() * g.double()).sum())
        rhs = 0.0
        for m in range(3):
            assert torch.equal(d1[m], d2[m]) and d1[m].stride() == xs[m].stride()
            assert float(d1[m].abs().sum()) > 0, m
            assert float((a[m] - d1[m]).double().norm() / d1[m].double().norm()) <= 1e-6
            rhs += float((xs[m].double() * d1[m].double()).sum())
            # each map on its own: <g, J_m x_m> = <J_m^T g, x_m>
            only = [xs[k] if k == m else torch.zeros_like(xs[k]) for k in range(3)]
            fm, _ = ops.point_gather_rig(only, pts, cnt, rig, SIZES)
            lm, rm = float((fm.double() * g.double()).sum()), float((xs[m].double() * d1[m].double()).sum())
            assert abs(lm - rm) <= 1e-5 * max(abs(lm), 1.0), (m, lm, rm)
        assert abs(lhs - rhs) <= 1e-5 * max(abs(lhs), 1.0), (lhs, rhs)
        d16 = ops.point_gather_rig_bwd(g, [x.to(BF) for x in xs], pts, cnt, rig, SIZES, deterministic=True)
        assert all(torch.equal(h, d.to(BF)) and h.dtype == BF for h, d in zip(d16, d1))


# ------------------------------------------------------------------------------------------- 5. layer
@pytest.fixture
def deterministic():
    before = torch.are_deterministic_algorithms_enabled()
    torch.use_deterministic_algorithms(True)
    yield
    torch.use_deterministic_algorithms(before)


def _frames(dcf, sweep):
    grid = dcf.ops.BucketGrid(*dcf.geometry.bucket_grid(sweep["config"]))
    return dcf.FrameContext(dev(sweep["points"]), dev(sweep["num_points"]), grid)


def test_layer_on_a_mixed_rig_sends_gradients_to_every_map(dcf, sweep, deterministic):
    G = dcf.geometry
    rig = torch.from_numpy(G.camera_rig(YAWS, SIZES)).cuda()
    torch.manual_seed(4)
    layer = dcf.ContinuousFusion(32, 32, k=3, radius=2.0, geom=G.scale_geometry(sweep["config"], 1), mode="fp32").cuda()
    bev0 = torch.randn(2, 32, 384, 256, device="cuda")
    grads = []
    for _ in range(2):
        layer.zero_grad(set_to_none=True)
        maps = [_layout(dev(m), True).requires_grad_(True) for m in sweep["maps"]]
        frames = _frames(dcf, sweep)
        frames.gather(maps, calib=rig, img_size=SIZES)
        out = layer(bev0, frames=frames)
        (out * out).sum().backward()
        assert all(m.grad is not None and float(m.grad.abs().sum()) > 0 for m in maps)
        grads.append([m.grad.clone() for m in maps] + [p.grad.clone() for p in layer.parameters()])
    assert all(torch.equal(a, b) for a, b in zip(*grads))


# ------------------------------------------------------------------------------------------- 6. FusionRunner
def test_fusion_runner_with_mixed_shapes(dcf, sweep):
    G = dcf.geometry
    cfg = sweep["config"]
    shapes = dcf.synthetic.scale_shapes(cfg)[:2]
    torch.manual_seed(5)
    layers = [dcf.ContinuousFusion(32, C, k=3, radius=2.0, geom=G.scale_geometry(cfg, s), mode="fp32").cuda().eval()
              for (C, _, _), s in zip(shapes, (1, 2))]
    grid = dcf.ops.BucketGrid(*G.bucket_grid(cfg))
    runner = dcf.FusionRunner(layers, grid, 2, sweep["points"].shape[1], [(32,) + s for s in SHAPES], shapes,
                              calib=G.camera_rig(YAWS, SIZES), img_size=SIZES, inplace=False, cameras=3)
    assert [tuple(t.shape) for t in runner.img_feat] == [(2, 32) + s for s in SHAPES]
    runner.points.copy_(dev(sweep["points"]))
    runner.num_points.copy_(dev(sweep["num_points"]))
    for t, m in zip(runner.img_feat, sweep["maps"]):
        t.copy_(dev(m))
    gen = torch.Generator(device="cuda").manual_seed(6)
    bevs = [torch.randn((2,) + tuple(s), device="cuda", generator=gen) for s in shapes]
    for d, b in zip(runner.bevs, bevs):
        d.copy_(b)
    prev = None
    for yaws in (YAWS, (-90.0, -20.0, 45.0)):
        rig = torch.from_numpy(G.camera_rig(yaws, SIZES)).cuda()
        runner.calib.copy_(rig.expand(2, 3, 4, 3))          # no recapture
        outs = [o.clone() for o in runner()]
        frames = _frames(dcf, sweep)
        with torch.no_grad():
            frames.gather([dev(m) for m in sweep["maps"]], calib=rig, img_size=SIZES)
            ref = dcf.fuse_scales(frames, layers, bevs)
        torch.cuda.synchronize()
        assert all(torch.equal(o, r) for o, r in zip(outs, ref)), yaws
        assert prev is None or not torch.equal(prev[0], outs[0])
        prev = outs


# ------------------------------------------------------------------------------------------- 7. model
def _model(dcf, sizes=SIZES):
    cfg = dcf.geometry.carla_config(fusion_scales=(1, 3), fusion_k=3, fusion_camera_yaws=YAWS,
                                    fusion_camera_image_sizes=[list(s) for s in sizes])
    torch.manual_seed(0)
    return dcf.ObjectDetection_DCF(cfg).cuda().eval()


def _images(sizes, seed=1):
    gen = torch.Generator(device="cuda").manual_seed(seed)
    return [torch.randint(0, 255, (2, 3, int(h), int(w)), device="cuda", dtype=torch.uint8, generator=gen) for w, h in sizes]


def test_model_with_mixed_image_sizes(dcf, sweep):
    model = _model(dcf)
    x_lidar = torch.rand(2, 32, 384, 256, device="cuda")
    x_image = _images(SIZES)
    kw = dict(pointcloud_raw=dev(sweep["points"]), num_points_raw=dev(sweep["num_points"]))
    with torch.no_grad():
        pred = model(x_lidar, x_image, **kw)
    assert pred.shape == (2, 32, 96, 64) and bool(torch.isfinite(pred).all())
    with pytest.raises(ValueError, match="list"):
        with torch.no_grad():
            model(x_lidar, torch.zeros(2, 3, 3, 480, 640, dtype=torch.uint8, device="cuda"), **kw)
    model.train()
    model.zero_grad(set_to_none=True)
    loss = model(x_lidar, x_image, **kw).float().square().mean()
    loss.backward()
    assert bool(torch.isfinite(loss))
    grads = {n: p.grad for n, p in model.named_parameters()}
    assert all(g is None or bool(torch.isfinite(g).all()) for g in grads.values())
    for n in ("fusion.group1.fc1.weight", "fusion.group3.fc1.weight", "image_backbone.stem.0.weight",
              "image_backbone.out.weight"):
        assert grads[n] is not None and float(grads[n].abs().sum()) > 0, n


def test_model_equal_size_list_gives_the_bits_of_the_5d_input(dcf, sweep):
    model = _model(dcf, [(640.0, 480.0)] * 3)
    x_lidar = torch.rand(2, 32, 384, 256, device="cuda")
    x_image = _images([(640.0, 480.0)] * 3)
    kw = dict(pointcloud_raw=dev(sweep["points"]), num_points_raw=dev(sweep["num_points"]))
    with torch.no_grad():
        a = model(x_lidar, x_image, **kw)
        b = model(x_lidar, torch.stack(x_image, 1), **kw)
    assert torch.equal(a, b)


def test_single_camera_checkpoint_loads_strictly(dcf):
    single = dcf.ObjectDetection_DCF(dcf.geometry.carla_config(fusion_scales=(1, 3), fusion_k=3)).cuda()
    _model(dcf).load_state_dict(single.state_dict(), strict=True)
