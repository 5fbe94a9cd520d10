"""GPU: bf16 feature maps through the continuous-fusion layer (CF_IO_BF16, cf_point_gather_bf16).

The contract: a bf16 map is widened exactly to fp32, the layer computes in fp32 as it does for an fp32 map, and a bf16
output is rounded once when stored.  So every bf16 result equals the fp32 path run on the widened map, then rounded --
compared bit for bit here (torch.equal), for every MLP mode and width, in place and out of place, on compacted and
uncompacted scales, odd planes and empty frames; then the autograd Functions, the drop-in model under torch.autocast and
FusionRunner."""
import os
import sys

import numpy as np
import pytest
import torch

from _util import dev

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BF = torch.bfloat16
WIDTHS = (32, 64, 96, 128, 192, 256)
CASES = [(m, C) for m in ("fp32", "bf16", "bf16t", "simt") for C in WIDTHS] + [("simt", 48)]
_CACHE = {}


def _setup(dcf, size, C, num_points=None, c_img=32):
    """Inputs of one scale: `size` "full" = the YAML grid's scale 1 at batch 2 (many tiles: compacted cell lists), "small" =
    the tiny workload's scale 1 (few tiles: not compacted)."""
    key = (size, C, tuple(num_points) if num_points else None)
    if key not in _CACHE:
        base = dcf.synthetic.workload("yaml" if size == "full" else "tiny")
        wl = dcf.synthetic.make_workload(dict(base, batch=2, scales=(1,)), seed=40 + C, c_img=c_img,
                                         img_hw=(24, 32), channels=[C, 64, 128, 192, 256])
        sc = wl["scales"][0]
        cnt = dev(wl["num_points"]) if num_points is None else torch.tensor(num_points, dtype=torch.int64, device="cuda")
        frames = dcf.FrameContext(dev(wl["points"]), cnt, dcf.ops.BucketGrid(*dcf.geometry.bucket_grid(wl["config"])))
        frames.gather(dev(wl["img_feat"]), calib=wl["calib"])
        _CACHE[key] = (wl, sc, frames, [dev(x) for x in sc["weights"]])
    return _CACHE[key]


def _bev16(shape, seed):
    gen = torch.Generator(device="cuda").manual_seed(seed)
    return (torch.randn(shape, device="cuda", generator=gen) * 4).to(BF)


def _check_fwd(dcf, frames, knn, geom, w, bev16, mode):
    w1, b1, w2, b2, w3, b3 = w
    T = dcf.ops.point_mlp1(frames.feat, frames.points, frames.num_points, w1, b1, mode=mode)
    ref = dcf.ops.fusion_fwd(bev16.float(), T, knn, geom, w1, w2, b2, w3, b3, mode=mode)[0].to(BF)
    got = dcf.ops.fusion_fwd(bev16, T, knn, geom, w1, w2, b2, w3, b3, mode=mode)[0]
    assert got.dtype == BF and torch.equal(got, ref), "out of place"
    io = bev16.clone()
    res = dcf.ops.fusion_fwd(io, T, knn, geom, w1, w2, b2, w3, b3, mode=mode, out=io)[0]
    assert res.data_ptr() == io.data_ptr() and torch.equal(io, ref), "in place"


@pytest.mark.parametrize("size", ("full", "small"))
@pytest.mark.parametrize("mode, C", CASES)
def test_fused_forward_equals_widened_fp32_rounded(dcf, mode, C, size):
    wl, sc, frames, w = _setup(dcf, size, C)
    knn = frames.knn(sc["H"], sc["W"], sc["geom"], wl["radius"], wl["k"])
    _check_fwd(dcf, frames, knn, sc["geom"], w, _bev16((2, C, sc["H"], sc["W"]), C), mode)


@pytest.mark.parametrize("mode, C", [(m, C) for m in ("fp32", "bf16", "bf16t", "simt") for C in (32, 64, 256)] + [("simt", 48)])
@pytest.mark.parametrize("size", ("full", "small"))
def test_fused_forward_odd_plane_and_empty_frame(dcf, mode, C, size):
    """An odd H*W (37 x 53: no vector alignment of the planes) and a frame without points (every cell a plain copy)."""
    wl, sc, frames, w = _setup(dcf, size, C, num_points=[int(_setup(dcf, size, C)[0]["num_points"][0]), 0])
    knn = frames.knn(37, 53, sc["geom"], wl["radius"], wl["k"])
    assert bool((knn[1] < 0).all())
    _check_fwd(dcf, frames, knn, sc["geom"], w, _bev16((2, C, 37, 53), 7), mode)


@pytest.mark.parametrize("channels_last", (False, True))
@pytest.mark.parametrize("use_uv", (False, True))
def test_gather_equals_widened_map(dcf, use_uv, channels_last):
    wl = dcf.synthetic.make_workload("tiny", seed=5, c_img=64, img_hw=(30, 41))
    img16 = dev(wl["img_feat"]).to(BF)
    if channels_last:
        img16 = img16.contiguous(memory_format=torch.channels_last)
    kw = dict(uv=dev(wl["uv"])) if use_uv else dict(calib=wl["calib"])
    pts, cnt = dev(wl["points"]), dev(wl["num_points"])
    got, _ = dcf.ops.point_gather(img16, pts, cnt, **kw)
    ref, _ = dcf.ops.point_gather(img16.float(), pts, cnt, **kw)
    assert got.dtype == torch.float32 and torch.equal(got, ref)


def _bwd(dcf, frames, knn, sc, w, gout, mode, det):
    w1, b1, w2, b2, w3, _ = w
    table = dcf.ops.point_mlp1(frames.feat, frames.points, frames.num_points, w1, b1, mode=mode)
    return dcf.ops.fusion_bwd(gout, frames.feat, frames.points, frames.num_points, knn, sc["geom"], w1, b1, w2, b2, w3,
                              table=table, mode=mode, deterministic=det)


@pytest.mark.parametrize("mode, C", [(m, C) for m in ("fp32", "bf16", "simt") for C in WIDTHS] + [("simt", 48)])
def test_fusion_bwd_with_bf16_grad_out(dcf, mode, C):
    wl, sc, frames, w = _setup(dcf, "full", C)
    knn = frames.knn(sc["H"], sc["W"], sc["geom"], wl["radius"], wl["k"])
    g16 = _bev16((2, C, sc["H"], sc["W"]), 100 + C)
    got = _bwd(dcf, frames, knn, sc, w, g16, mode, True)
    ref = _bwd(dcf, frames, knn, sc, w, g16.float(), mode, True)
    for a, b in zip(got, ref):
        assert a.dtype == torch.float32 and torch.equal(a, b)
    got = _bwd(dcf, frames, knn, sc, w, g16, mode, False)
    for a, b in zip(got, ref):
        assert (a.double() - b.double()).norm().item() <= 1e-5 * max(b.double().norm().item(), 1e-30)


@pytest.mark.parametrize("channels_last", (False, True))
@pytest.mark.parametrize("use_uv", (False, True))
def test_point_gather_bwd_bf16_map(dcf, use_uv, channels_last):
    wl = dcf.synthetic.make_workload("tiny", seed=6, c_img=32, img_hw=(30, 41))
    img16 = dev(wl["img_feat"]).to(BF)
    if channels_last:
        img16 = img16.contiguous(memory_format=torch.channels_last)
    kw = dict(uv=dev(wl["uv"])) if use_uv else dict(calib=wl["calib"])
    pts, cnt = dev(wl["points"]), dev(wl["num_points"])
    gfeat = torch.randn((pts.shape[0], pts.shape[1], 32), device="cuda")
    got = dcf.ops.point_gather_bwd(gfeat, img16, pts, cnt, deterministic=True, **kw)
    ref = dcf.ops.point_gather_bwd(gfeat, img16.float(), pts, cnt, deterministic=True, **kw)
    assert got.dtype == BF and got.stride() == img16.stride()
    assert torch.equal(got, ref.to(BF))
    fast = dcf.ops.point_gather_bwd(gfeat, img16, pts, cnt, **kw)
    assert fast.dtype == BF and fast.stride() == img16.stride()


@pytest.mark.parametrize("mode", ("fp32", "bf16", "simt"))
def test_autograd_bf16_maps(dcf, mode):
    wl = dcf.synthetic.make_workload("tiny", seed=8, c_img=32, img_hw=(24, 32))
    sc = wl["scales"][0]

    def run(dtype):
        torch.manual_seed(3)
        layer = dcf.ContinuousFusion(32, sc["C"], k=wl["k"], radius=wl["radius"], geom=sc["geom"], mode=mode).cuda()
        img = dev(wl["img_feat"]).to(BF).to(dtype).contiguous(memory_format=torch.channels_last).requires_grad_(True)
        bev = dev(sc["bev"]).to(BF).to(dtype).requires_grad_(True)
        frames = dcf.prepare_frames(dev(wl["points"]), dev(wl["num_points"]), img, config=wl["config"], calib=wl["calib"])
        out = layer(bev, frames=frames)
        assert out.dtype == dtype
        gout = torch.randn(out.shape, device="cuda", generator=torch.Generator(device="cuda").manual_seed(4)).to(BF).to(dtype)
        out.backward(gout)
        return bev.grad, gout, img.grad, [p.grad for p in layer.parameters()]

    before = torch.are_deterministic_algorithms_enabled()
    torch.use_deterministic_algorithms(True)
    try:
        gb16, gout16, gi16, gw16 = run(BF)
        _, _, gi32, gw32 = run(torch.float32)
    finally:
        torch.use_deterministic_algorithms(before)
    assert gb16.dtype == BF and torch.equal(gb16, gout16)
    assert gi16.dtype == BF and torch.equal(gi16, gi32.to(BF))
    for a, b in zip(gw16, gw32):
        assert a.dtype == torch.float32 and torch.equal(a, b)


def _model_inputs(dcf, B=2):
    dev_ = torch.device("cuda")
    wl = dcf.synthetic.make_workload(dict(dcf.synthetic.workload("yaml"), batch=B), seed=7)
    to = lambda x: torch.from_numpy(np.ascontiguousarray(x)).to(dev_)
    x_lidar = torch.rand(B, 32, 384, 256, device=dev_)
    x_image = torch.randint(0, 255, (B, 3, 480, 640), device=dev_, dtype=torch.uint8)
    return x_lidar, x_image, dict(pointcloud_raw=to(wl["points"]), num_points_raw=to(wl["num_points"]),
                                  projected_loc_uv=to(wl["uv"]))


def test_model_under_autocast_infers_in_place_and_trains(dcf):
    sys.path.insert(0, os.path.join(ROOT, "scripts"))
    from train_step_bench import synthetic_labels
    torch.manual_seed(0)
    cfg = dcf.geometry.carla_config(fusion_scales=(1, 2, 3, 4, 5), fusion_k=3)
    model = dcf.ObjectDetection_DCF(cfg).cuda().eval()
    x_lidar, x_image, extra = _model_inputs(dcf)
    seen, busy = [], [False]

    def pre(mod, args, kwargs):
        if not busy[0]:
            mod._map_in = args[0].detach().clone()

    def post(mod, args, kwargs, out):
        if busy[0]:
            return
        busy[0] = True
        try:
            with torch.no_grad():
                ref = mod(mod._map_in.float(), frames=kwargs["frames"]).to(mod._map_in.dtype)
        finally:
            busy[0] = False
        seen.append((mod._map_in.dtype, out.dtype, torch.equal(out, ref), out.data_ptr() == args[0].data_ptr()))

    hooks = []
    for layer in model.fusion.values():
        hooks.append(layer.register_forward_pre_hook(pre, with_kwargs=True))
        hooks.append(layer.register_forward_hook(post, with_kwargs=True))
    with torch.no_grad(), torch.autocast("cuda", dtype=BF):
        pred = model(x_lidar, x_image, **extra)
    for h in hooks:
        h.remove()
    # Group 1 ends in an identity shortcut that adds the fp32 input voxels to a bf16 conv branch, so autocast's type promotion
    # hands its fusion layer an fp32 map; every later group starts with a projection shortcut and its map is bf16.  Each layer
    # returns the dtype it was given, equal to the fp32 layer on the widened input, rounded to that dtype.
    assert len(seen) == 5
    assert [s[0] for s in seen] == [torch.float32] + [BF] * 4, [s[0] for s in seen]
    for g, (din, dt, eq, inplace) in enumerate(seen, start=1):
        assert dt == din and eq and inplace, f"group {g}: in {din}, out {dt}, equal {eq}, in place {inplace}"
    assert bool(torch.isfinite(pred.float()).all())
    boxes = dcf.PostProcess().get_bboxes(pred[:, :4].float(), pred[:, 4:18].float(), 0.5)
    assert len(boxes) == 2

    crit = dcf.LossTotal(cfg, batch_reduction="sum", generator=torch.Generator(device="cuda").manual_seed(1)).cuda()
    opt = torch.optim.Adam(model.parameters(), lr=1e-4)
    ref, num = synthetic_labels(2, 11, torch.device("cuda"))
    opt.zero_grad(set_to_none=True)
    with torch.autocast("cuda", dtype=BF):
        pred = model(x_lidar, x_image, **extra)
        pred_cls, pred_reg, _ = torch.split(pred, [4, 14, 14], dim=1)
        loss = crit(ref, num, pred_cls, pred_reg).sum()
    loss.backward()
    opt.step()
    assert bool(torch.isfinite(loss))
    fusion_grads = [p.grad for n, p in model.named_parameters() if n.startswith("fusion.")]
    assert fusion_grads and all(g is not None and g.dtype == torch.float32 and bool(torch.isfinite(g).all()) for g in fusion_grads)
    assert all(p.grad is None or bool(torch.isfinite(p.grad).all()) for p in model.parameters())


def test_fusion_runner_bf16_replay_equals_eager(dcf):
    wl = dcf.synthetic.make_workload(dict(dcf.synthetic.workload("yaml"), batch=2, k=3), seed=31)
    torch.manual_seed(2)
    layers = [dcf.ContinuousFusion(wl["img_feat"].shape[1], sc["C"], k=wl["k"], radius=wl["radius"], geom=sc["geom"],
                                   mode="fp32").cuda().eval() for sc in wl["scales"]]
    grid = dcf.ops.BucketGrid(*dcf.geometry.bucket_grid(wl["config"], None))
    size = (float(wl["config"]["image_width"]), float(wl["config"]["image_height"]))
    runner = dcf.FusionRunner(layers, grid, 2, wl["points"].shape[1], wl["img_feat"].shape[1:],
                              [sc["bev"].shape[1:] for sc in wl["scales"]], calib=wl["calib"], img_size=size, dtype=BF)
    assert runner.img_feat.dtype == BF and all(b.dtype == BF for b in runner.bevs)
    runner.points.copy_(dev(wl["points"]))
    runner.num_points.copy_(dev(wl["num_points"]))
    runner.img_feat.copy_(dev(wl["img_feat"]).to(BF))
    bevs = [dev(sc["bev"]).to(BF) for sc in wl["scales"]]
    for d, b in zip(runner.bevs, bevs):
        d.copy_(b)
    outs = runner()
    frames = dcf.prepare_frames(dev(wl["points"]), dev(wl["num_points"]), dev(wl["img_feat"]).to(BF), config=wl["config"],
                                calib=wl["calib"])
    ref = dcf.fuse_scales(frames, layers, bevs)
    torch.cuda.synchronize()
    for o, r in zip(outs, ref):
        assert o.dtype == BF and torch.equal(o, r)


def test_errors(dcf):
    wl, sc, frames, w = _setup(dcf, "small", 32)
    knn = frames.knn(sc["H"], sc["W"], sc["geom"], wl["radius"], wl["k"])
    w1, b1, w2, b2, w3, b3 = w
    T = dcf.ops.point_mlp1(frames.feat, frames.points, frames.num_points, w1, b1)
    bev = dev(sc["bev"])
    with pytest.raises(TypeError, match="bfloat16"):
        dcf.ops.fusion_fwd(bev.half(), T, knn, sc["geom"], w1, w2, b2, w3, b3)
    with pytest.raises(TypeError, match="bfloat16"):
        dcf.ops.point_gather(dev(wl["img_feat"]).half(), frames.points, frames.num_points, calib=wl["calib"])
    with pytest.raises(ValueError, match="dtype"):
        dcf.ops.fusion_fwd(bev.to(BF), T, knn, sc["geom"], w1, w2, b2, w3, b3, out=torch.empty_like(bev))
    with pytest.raises(ValueError, match="dtype"):
        dcf.ops.fusion_fwd(bev, T, knn, sc["geom"], w1, w2, b2, w3, b3, out=torch.empty_like(bev, dtype=BF))
    layer = dcf.ContinuousFusion(32, 32, k=wl["k"], radius=wl["radius"], geom=sc["geom"], mode="bf16t").cuda()
    with pytest.raises(RuntimeError, match="inference only"):
        layer(bev.to(BF).requires_grad_(True), frames=frames)
