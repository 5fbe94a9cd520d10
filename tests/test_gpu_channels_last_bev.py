"""GPU: channels_last BEV maps through the continuous-fusion layer (CF_IO_NHWC).

The contract: the layout changes only where the maps are read and written.  So every NHWC result equals the NCHW call on
the same values bit for bit (torch.equal) -- for every MLP mode, width and map dtype, K = 3 / 10 / 16, in place and out of
place, on compacted and uncompacted scales, odd planes and empty frames -- and the output keeps the channels_last format.
Then the backward, the autograd Function, the drop-in model converted with .to(memory_format=torch.channels_last), CUDA
graphs and the launch count."""
import os
import sys

import numpy as np
import pytest
import torch

from _util import dev

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BF = torch.bfloat16
CL = torch.channels_last
WIDTHS = (32, 64, 96, 128, 192, 256)
CASES = [(m, C) for m in ("fp32", "bf16", "bf16t", "simt") for C in WIDTHS] + [("simt", 48)]
_CACHE = {}


def _setup(dcf, size, C, num_points=None):
    """Inputs of one scale: `size` "full" = the YAML grid's scale 1 at batch 2 (many tiles: compacted cell lists), "small" =
    the tiny workload's scale 1 (few tiles: not compacted)."""
    key = (size, C, tuple(num_points) if num_points else None)
    if key not in _CACHE:
        base = dcf.synthetic.workload("yaml" if size == "full" else "tiny")
        wl = dcf.synthetic.make_workload(dict(base, batch=2, scales=(1,)), seed=60 + C, c_img=32,
                                         img_hw=(24, 32), channels=[C, 64, 128, 192, 256])
        sc = wl["scales"][0]
        cnt = dev(wl["num_points"]) if num_points is None else torch.tensor(num_points, dtype=torch.int64, device="cuda")
        frames = dcf.FrameContext(dev(wl["points"]), cnt, dcf.ops.BucketGrid(*dcf.geometry.bucket_grid(wl["config"])))
        frames.gather(dev(wl["img_feat"]), calib=wl["calib"])
        _CACHE[key] = (wl, sc, frames, [dev(x) for x in sc["weights"]])
    return _CACHE[key]


def _bev(shape, seed, dtype):
    gen = torch.Generator(device="cuda").manual_seed(seed)
    return (torch.randn(shape, device="cuda", generator=gen) * 4).to(dtype)


def _is_nhwc(t):
    return t.is_contiguous(memory_format=CL) and not t.is_contiguous()


def _check_fwd(dcf, frames, knn, geom, w, bev, mode):
    """NHWC out of place and in place against the NCHW call on the same map."""
    w1, b1, w2, b2, w3, b3 = w
    T = dcf.ops.point_mlp1(frames.feat, frames.points, frames.num_points, w1, b1, mode=mode)
    ref = dcf.ops.fusion_fwd(bev, T, knn, geom, w1, w2, b2, w3, b3, mode=mode)[0]
    cl = bev.contiguous(memory_format=CL)
    keep = cl.clone()
    got = dcf.ops.fusion_fwd(cl, T, knn, geom, w1, w2, b2, w3, b3, mode=mode, memory_format=CL)[0]
    assert got.dtype == bev.dtype and _is_nhwc(got), got.stride()
    assert torch.equal(got, ref), "out of place"
    assert torch.equal(cl, keep), "bev is unchanged out of place"
    io = cl.clone()
    res = dcf.ops.fusion_fwd(io, T, knn, geom, w1, w2, b2, w3, b3, mode=mode, out=io, memory_format=CL)[0]
    assert res.data_ptr() == io.data_ptr() and torch.equal(io, ref), "in place"


@pytest.mark.parametrize("dtype", (torch.float32, BF), ids=("fp32map", "bf16map"))
@pytest.mark.parametrize("size", ("full", "small"))
@pytest.mark.parametrize("mode, C", CASES)
def test_forward_nhwc_equals_nchw(dcf, mode, C, size, dtype):
    wl, sc, frames, w = _setup(dcf, size, C)
    knn = frames.knn(sc["H"], sc["W"], sc["geom"], wl["radius"], wl["k"])
    _check_fwd(dcf, frames, knn, sc["geom"], w, _bev((2, C, sc["H"], sc["W"]), C, dtype), mode)


@pytest.mark.parametrize("K", (10, 16))
@pytest.mark.parametrize("dtype", (torch.float32, BF), ids=("fp32map", "bf16map"))
@pytest.mark.parametrize("mode, C", [(m, C) for m in ("fp32", "bf16", "bf16t") for C in WIDTHS] + [("simt", 32), ("simt", 48)])
def test_forward_nhwc_equals_nchw_more_neighbours(dcf, mode, C, dtype, K):
    wl, sc, frames, w = _setup(dcf, "full", C)
    knn = frames.knn(sc["H"], sc["W"], sc["geom"], wl["radius"], K)
    _check_fwd(dcf, frames, knn, sc["geom"], w, _bev((2, C, sc["H"], sc["W"]), C + K, dtype), mode)


@pytest.mark.parametrize("dtype", (torch.float32, BF), ids=("fp32map", "bf16map"))
@pytest.mark.parametrize("mode, C", [(m, C) for m in ("fp32", "bf16", "bf16t", "simt") for C in (32, 64, 128, 256)] + [("simt", 48)])
@pytest.mark.parametrize("size", ("full", "small"))
def test_forward_nhwc_odd_plane_and_empty_frame(dcf, mode, C, size, dtype):
    """An odd H*W (37 x 53) and a frame without points (every cell a plain copy)."""
    wl, sc, frames, w = _setup(dcf, size, C, num_points=[int(_setup(dcf, size, C)[0]["num_points"][0]), 0])
    knn = frames.knn(37, 53, sc["geom"], wl["radius"], wl["k"])
    assert bool((knn[1] < 0).all())
    _check_fwd(dcf, frames, knn, sc["geom"], w, _bev((2, C, 37, 53), 7, dtype), mode)


@pytest.mark.parametrize("dtype", (torch.float32, BF), ids=("fp32map", "bf16map"))
def test_sk_and_tc_kernels_agree_in_nhwc(dcf, dtype):
    """C = 128 in fp32 mode: K = 3 runs k_fusion_sk, the same table padded with empty slots to K = 16 runs k_fusion_tc."""
    wl, sc, frames, w = _setup(dcf, "full", 128)
    knn3 = frames.knn(sc["H"], sc["W"], sc["geom"], wl["radius"], 3)
    knn16 = torch.cat([knn3, torch.full(knn3.shape[:3] + (13,), -1, dtype=torch.int32, device="cuda")], dim=3).contiguous()
    w1, b1, w2, b2, w3, b3 = w
    T = dcf.ops.point_mlp1(frames.feat, frames.points, frames.num_points, w1, b1, mode="fp32")
    bev = _bev((2, 128, sc["H"], sc["W"]), 5, dtype).contiguous(memory_format=CL)
    a = dcf.ops.fusion_fwd(bev, T, knn3, sc["geom"], w1, w2, b2, w3, b3, mode="fp32", memory_format=CL)[0]
    b = dcf.ops.fusion_fwd(bev, T, knn16, sc["geom"], w1, w2, b2, w3, b3, mode="fp32", memory_format=CL)[0]
    assert _is_nhwc(a) and _is_nhwc(b) and torch.equal(a, b)


@pytest.mark.parametrize("mode, C", (("fp32", 64), ("fp32", 128), ("simt", 48)))
@pytest.mark.parametrize("dtype", (torch.float32, BF), ids=("fp32map", "bf16map"))
def test_backward_nhwc_grad_out(dcf, mode, C, dtype):
    wl, sc, frames, w = _setup(dcf, "full", C)
    knn = frames.knn(sc["H"], sc["W"], sc["geom"], wl["radius"], wl["k"])
    w1, b1, w2, b2, w3, b3 = w
    g = _bev((2, C, sc["H"], sc["W"]), 11, dtype)
    gcl = g.contiguous(memory_format=CL)
    args = (frames.feat, frames.points, frames.num_points, knn, sc["geom"], w1, b1, w2, b2, w3)
    for det in (True, False):
        ref = dcf.ops.fusion_bwd(g, *args, mode=mode, deterministic=det)
        got = dcf.ops.fusion_bwd(gcl, *args, mode=mode, deterministic=det)
        for name, a, b in zip(("gW1", "gb1", "gW2", "gb2", "gW3", "gb3", "gfeat"), got, ref):
            if det:
                assert torch.equal(a, b), name
            else:
                err = (a.double() - b.double()).norm().item() / max(b.double().norm().item(), 1e-30)
                assert err <= 1e-5, (name, err)


@pytest.mark.parametrize("dtype", (torch.float32, BF), ids=("fp32map", "bf16map"))
@pytest.mark.parametrize("mode", ("fp32", "bf16", "simt"))
def test_autograd_channels_last_bev(dcf, mode, dtype):
    wl = dcf.synthetic.make_workload("tiny", seed=8, c_img=32, img_hw=(24, 32))
    sc = wl["scales"][0]

    def run(fmt):
        torch.manual_seed(3)
        layer = dcf.ContinuousFusion(32, sc["C"], k=wl["k"], radius=wl["radius"], geom=sc["geom"], mode=mode).cuda()
        img = dev(wl["img_feat"]).contiguous(memory_format=CL).requires_grad_(True)
        bev = dev(sc["bev"]).to(dtype).contiguous(memory_format=fmt).requires_grad_(True)
        frames = dcf.prepare_frames(dev(wl["points"]), dev(wl["num_points"]), img, config=wl["config"], calib=wl["calib"])
        out = layer(bev, frames=frames)
        gout = _bev(out.shape, 4, dtype).contiguous(memory_format=fmt)
        out.backward(gout)
        return out, bev.grad, gout, img.grad, [p.grad for p in layer.parameters()]

    before = torch.are_deterministic_algorithms_enabled()
    torch.use_deterministic_algorithms(True)
    try:
        o_cl, gb_cl, gout_cl, gi_cl, gw_cl = run(CL)
        o_ref, _, _, gi_ref, gw_ref = run(torch.contiguous_format)
    finally:
        torch.use_deterministic_algorithms(before)
    assert _is_nhwc(o_cl) and o_ref.is_contiguous() and torch.equal(o_cl, o_ref)
    assert torch.equal(gb_cl, gout_cl)
    assert torch.equal(gi_cl, gi_ref)
    for a, b in zip(gw_cl, gw_ref):
        assert torch.equal(a, b)


def _model_inputs(dcf, B=2):
    dev_ = torch.device("cuda")
    wl = dcf.synthetic.make_workload(dict(dcf.synthetic.workload("yaml"), batch=B), seed=7)
    to = lambda x: torch.from_numpy(np.ascontiguousarray(x)).to(dev_)
    x_lidar = torch.rand(B, 32, 384, 256, device=dev_).contiguous(memory_format=CL)
    x_image = torch.randint(0, 255, (B, 3, 480, 640), device=dev_, dtype=torch.uint8).contiguous(memory_format=CL)
    return x_lidar, x_image, dict(pointcloud_raw=to(wl["points"]), num_points_raw=to(wl["num_points"]),
                                  projected_loc_uv=to(wl["uv"]))


def test_channels_last_model_fuses_in_place_and_trains(dcf):
    sys.path.insert(0, os.path.join(ROOT, "scripts"))
    from train_step_bench import synthetic_labels
    torch.manual_seed(0)
    cfg = dcf.geometry.carla_config(fusion_scales=(1, 2, 3, 4, 5), fusion_k=3)
    model = dcf.ObjectDetection_DCF(cfg).cuda().eval().to(memory_format=CL)
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
                ref = mod(mod._map_in.contiguous(), frames=kwargs["frames"])
        finally:
            busy[0] = False
        seen.append((_is_nhwc(mod._map_in), _is_nhwc(out), torch.equal(out, ref), out.data_ptr() == args[0].data_ptr()))

    hooks = []
    for layer in model.fusion.values():
        hooks.append(layer.register_forward_pre_hook(pre, with_kwargs=True))
        hooks.append(layer.register_forward_hook(post, with_kwargs=True))
    with torch.no_grad():
        pred = model(x_lidar, x_image, **extra)
    for h in hooks:
        h.remove()
    assert len(seen) == 5
    for g, (cl_in, cl_out, eq, inplace) in enumerate(seen, start=1):
        assert cl_in and cl_out and eq and inplace, f"group {g}: NHWC in {cl_in}, out {cl_out}, equal {eq}, in place {inplace}"
    assert bool(torch.isfinite(pred).all())

    crit = dcf.LossTotal(cfg, batch_reduction="sum", generator=torch.Generator(device="cuda").manual_seed(1)).cuda()
    opt = torch.optim.Adam(model.parameters(), lr=1e-4)
    ref, num = synthetic_labels(2, 11, torch.device("cuda"))
    model.train()
    for amp in (False, True):
        opt.zero_grad(set_to_none=True)
        with torch.autocast("cuda", dtype=BF, enabled=amp):
            pred = model(x_lidar, x_image, **extra)
            pred_cls, pred_reg, _ = torch.split(pred, [4, 14, 14], dim=1)
            loss = crit(ref, num, pred_cls, pred_reg).sum()
        loss.backward()
        opt.step()
        assert bool(torch.isfinite(loss)), amp
        fusion_grads = [p.grad for n, p in model.named_parameters() if n.startswith("fusion.")]
        assert fusion_grads and all(g is not None and bool(torch.isfinite(g).all()) for g in fusion_grads), amp


def _scales_setup(dcf):
    wl = dcf.synthetic.make_workload(dict(dcf.synthetic.workload("yaml"), batch=2, k=3), seed=31)
    torch.manual_seed(2)
    layers = [dcf.ContinuousFusion(wl["img_feat"].shape[1], sc["C"], k=wl["k"], radius=wl["radius"], geom=sc["geom"],
                                   mode="fp32").cuda().eval() for sc in wl["scales"]]
    return wl, layers


def _frames(dcf, wl):
    return dcf.prepare_frames(dev(wl["points"]), dev(wl["num_points"]), dev(wl["img_feat"]), config=wl["config"],
                              calib=wl["calib"])


def test_fuse_scales_graph_replay_equals_eager(dcf):
    wl, layers = _scales_setup(dcf)
    pts, cnt, img = dev(wl["points"]), dev(wl["num_points"]), dev(wl["img_feat"])   # static inputs of the capture
    frames = lambda: dcf.prepare_frames(pts, cnt, img, config=wl["config"], calib=wl["calib"])
    bevs = [dev(sc["bev"]).contiguous(memory_format=CL) for sc in wl["scales"]]
    eager = dcf.fuse_scales(frames(), layers, bevs)
    nchw = dcf.fuse_scales(frames(), layers, [b.contiguous() for b in bevs])
    torch.cuda.synchronize()
    for e, r in zip(eager, nchw):
        assert _is_nhwc(e) and torch.equal(e, r)
    static = [b.clone() for b in bevs]
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):   # warm-up outside the capture
        for _ in range(2):
            dcf.fuse_scales(frames(), layers, [b.clone() for b in bevs], inplace=True)
    torch.cuda.current_stream().wait_stream(side)
    torch.cuda.synchronize()
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        outs = dcf.fuse_scales(frames(), layers, static, inplace=True)
    for s, b in zip(static, bevs):
        s.copy_(b)
    graph.replay()
    torch.cuda.synchronize()
    for o, s, e in zip(outs, static, eager):
        assert o.data_ptr() == s.data_ptr() and _is_nhwc(o) and torch.equal(o, e)


def test_fusion_runner_channels_last_replay_equals_eager(dcf):
    wl, layers = _scales_setup(dcf)
    grid = dcf.ops.BucketGrid(*dcf.geometry.bucket_grid(wl["config"], None))
    size = (float(wl["config"]["image_width"]), float(wl["config"]["image_height"]))
    for inplace in (True, False):
        runner = dcf.FusionRunner(layers, grid, 2, wl["points"].shape[1], wl["img_feat"].shape[1:],
                                  [sc["bev"].shape[1:] for sc in wl["scales"]], calib=wl["calib"], img_size=size,
                                  inplace=inplace, memory_format=CL)
        assert all(_is_nhwc(b) for b in runner.bevs)
        runner.points.copy_(dev(wl["points"]))
        runner.num_points.copy_(dev(wl["num_points"]))
        runner.img_feat.copy_(dev(wl["img_feat"]))
        bevs = [dev(sc["bev"]) for sc in wl["scales"]]
        for d, b in zip(runner.bevs, bevs):
            d.copy_(b)
        outs = runner()
        ref = dcf.fuse_scales(_frames(dcf, wl), layers, bevs)
        torch.cuda.synchronize()
        for o, r in zip(outs, ref):
            assert _is_nhwc(o) and torch.equal(o, r), inplace


@pytest.mark.parametrize("mode", ("fp32", "simt"))
def test_nhwc_call_launches_what_the_nchw_call_launches(dcf, mode):
    wl, sc, frames, w = _setup(dcf, "full", 64)
    knn = frames.knn(sc["H"], sc["W"], sc["geom"], wl["radius"], wl["k"])
    w1, b1, w2, b2, w3, b3 = w
    T = dcf.ops.point_mlp1(frames.feat, frames.points, frames.num_points, w1, b1, mode=mode)
    lib = dcf.load()
    bev = _bev((2, 64, sc["H"], sc["W"]), 3, torch.float32)
    counts = []
    for b, fmt in ((bev, torch.contiguous_format), (bev.contiguous(memory_format=CL), CL)):
        out = torch.empty_like(b)
        n0 = lib.cf_launch_count()
        dcf.ops.fusion_fwd(b, T, knn, sc["geom"], w1, w2, b2, w3, b3, mode=mode, out=out, memory_format=fmt)
        counts.append(lib.cf_launch_count() - n0)
    assert counts[0] == counts[1] > 0


def test_errors(dcf):
    wl, sc, frames, w = _setup(dcf, "small", 32)
    knn = frames.knn(sc["H"], sc["W"], sc["geom"], wl["radius"], wl["k"])
    w1, b1, w2, b2, w3, b3 = w
    T = dcf.ops.point_mlp1(frames.feat, frames.points, frames.num_points, w1, b1)
    bev = dev(sc["bev"])
    cl = bev.contiguous(memory_format=CL)
    args = (T, knn, sc["geom"], w1, w2, b2, w3, b3)
    with pytest.raises(ValueError, match="channels_last"):
        dcf.ops.fusion_fwd(bev, *args, memory_format=CL)                               # an NCHW bev
    with pytest.raises(ValueError, match="out must be"):
        dcf.ops.fusion_fwd(cl, *args, out=torch.empty_like(bev), memory_format=CL)    # an NCHW out
    with pytest.raises(ValueError, match="out must be"):
        dcf.ops.fusion_fwd(bev, *args, out=torch.empty_like(cl))                       # a channels_last out, NCHW call
    layer = dcf.ContinuousFusion(32, 32, k=wl["k"], radius=wl["radius"], geom=sc["geom"]).cuda()
    with torch.no_grad(), pytest.raises(ValueError, match="out must be"):
        layer(cl, frames=frames, out=torch.empty_like(bev))
