"""GPU: the deterministic backward (cf_fusion_bwd | CF_BWD_DETERMINISTIC, cf_point_gather_bwd_det) and the drop-in model
under torch.use_deterministic_algorithms(True).

Repeated calls give bit-identical gradients whatever else runs on the GPU; they agree with the default (atomic) path to
rounding, and with float64 autograd as tightly as the default path does; a CUDA-graph replay gives the eager result bit for
bit; two fresh processes training the drop-in model for three steps end with the same bytes."""
import hashlib
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

from _util import dev
from test_gpu_backward import torch_layer

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
NAMES = ("gW1", "gb1", "gW2", "gb2", "gW3", "gb3", "gfeat")


@pytest.fixture
def deterministic():
    before = torch.are_deterministic_algorithms_enabled()
    torch.use_deterministic_algorithms(True)
    yield
    torch.use_deterministic_algorithms(before)


def _scale1(dcf, C, seed=31, batch=4, c_img=128, num_points=None):
    """configs[3]-sized scale 1 (YAML grid 384x256, batch 4, K = 3): inputs of one cf_fusion_bwd call."""
    wl = dcf.synthetic.make_workload(dict(dcf.synthetic.workload("yaml"), batch=batch, scales=(1,)), seed=seed, c_img=c_img,
                                     channels=[C, 64, 128, 192, 256])
    sc = wl["scales"][0]
    pts, cnt = dev(wl["points"]), dev(wl["num_points"])
    if num_points is not None:
        cnt = torch.tensor(num_points, dtype=torch.int64, device="cuda")
    frames = dcf.FrameContext(pts, cnt, dcf.ops.BucketGrid(*dcf.geometry.bucket_grid(wl["config"])))
    frames.gather(dev(wl["img_feat"]), calib=wl["calib"])
    knn = frames.knn(sc["H"], sc["W"], sc["geom"], wl["radius"], wl["k"])
    w = [dev(x) for x in sc["weights"]]
    gen = torch.Generator(device="cuda").manual_seed(seed)
    gout = torch.randn((batch, C, sc["H"], sc["W"]), device="cuda", generator=gen)
    return wl, sc, frames, knn, w, gout


def _bwd(dcf, frames, knn, sc, w, gout, mode, deterministic):
    w1, b1, w2, b2, w3, _ = w
    table = dcf.ops.point_mlp1(frames.feat, frames.points, frames.num_points, w1, b1, mode=mode)
    return dcf.ops.fusion_bwd(gout, frames.feat, frames.points, frames.num_points, knn, sc["geom"], w1, b1, w2, b2, w3,
                              table=table, mode=mode, deterministic=deterministic)


def _perturb(side, a):
    with torch.cuda.stream(side):      # unrelated work that competes for the SMs while the next call runs
        for _ in range(4):
            a = a @ a
            a = a / a.norm()
    return a


def _rel(a, b):
    return (a.double() - b.double()).norm().item() / max(b.double().norm().item(), 1e-30)


CASES = [(C, m) for C in (32, 64, 256) for m in ("fp32", "bf16", "simt")] + [(48, "simt")]


@pytest.mark.parametrize("C, mode", CASES)
def test_fusion_bwd_repeatable_and_within_rounding_of_atomic_path(dcf, C, mode):
    wl, sc, frames, knn, w, gout = _scale1(dcf, C)
    side = torch.cuda.Stream()
    a = torch.randn(2048, 2048, device="cuda")
    first = None
    for _ in range(5):
        a = _perturb(side, a)
        got = _bwd(dcf, frames, knn, sc, w, gout, mode, True)
        torch.cuda.synchronize()
        if first is None:
            first = [g.clone() for g in got]
        else:
            for name, x, y in zip(NAMES, got, first):
                assert torch.equal(x, y), f"C={C} {mode}: {name} differs between two deterministic calls"
    atomic = _bwd(dcf, frames, knn, sc, w, gout, mode, False)
    for name, x, y in zip(NAMES, first, atomic):
        assert torch.isfinite(x).all(), name
        assert _rel(x, y) <= 1e-5, f"C={C} {mode}: {name} rel L2 {_rel(x, y):.3e} against the atomic path"


@pytest.mark.parametrize("use_uv", [False, True])
@pytest.mark.parametrize("channels_last", [False, True])
def test_point_gather_bwd_repeatable_and_within_rounding(dcf, use_uv, channels_last):
    wl = dcf.synthetic.make_workload(dict(dcf.synthetic.workload("yaml"), batch=4, scales=(1,)), seed=33, c_img=128)
    pts, cnt = dev(wl["points"]), dev(wl["num_points"])
    img = dev(wl["img_feat"])
    if channels_last:
        img = img.contiguous(memory_format=torch.channels_last)
    gfeat = torch.randn((4, pts.shape[1], 128), device="cuda", generator=torch.Generator(device="cuda").manual_seed(2))
    kw = dict(uv=dev(wl["uv"])) if use_uv else dict(calib=wl["calib"])
    side = torch.cuda.Stream()
    a = torch.randn(2048, 2048, device="cuda")
    first = None
    for _ in range(5):
        a = _perturb(side, a)
        g = dcf.ops.point_gather_bwd(gfeat, img, pts, cnt, deterministic=True, **kw)
        torch.cuda.synchronize()
        assert g.stride() == img.stride()
        if first is None:
            first = g.clone()
        else:
            assert torch.equal(g, first)
    atomic = dcf.ops.point_gather_bwd(gfeat, img, pts, cnt, **kw)
    assert first.abs().sum() > 0
    assert _rel(first, atomic) <= 1e-6


@pytest.mark.parametrize("mode", ["fp32", "simt"])
def test_deterministic_gradients_match_float64_autograd(dcf, deterministic, mode):
    """Through the autograd Functions with the flag on (the layer picks the deterministic kernels by itself), against the
    float64 reference of test_gpu_backward.py with its tolerances."""
    wl = dcf.synthetic.make_workload(dict(dcf.synthetic.workload("tiny"), scales=(1, 2)), seed=21, c_img=32, img_hw=(24, 32))
    img = dev(wl["img_feat"]).requires_grad_(True)
    pts, cnt = dev(wl["points"]), dev(wl["num_points"])
    frames = dcf.FrameContext(pts, cnt, dcf.ops.BucketGrid(*dcf.geometry.bucket_grid(wl["config"])))
    frames.gather(img, calib=wl["calib"])
    gen = torch.Generator(device="cuda").manual_seed(5)
    sets, loss = [], 0.0
    for sc in wl["scales"]:
        layer = dcf.ContinuousFusion(32, sc["C"], k=wl["k"], radius=wl["radius"], geom=sc["geom"], mode=mode).cuda()
        with torch.no_grad():
            for p_, w_ in zip(layer.parameters(), sc["weights"]):
                p_.copy_(dev(w_))
        bev = dev(sc["bev"]).requires_grad_(True)
        out, knn = layer(bev, frames=frames, return_knn=True)
        s = torch.randn(out.shape, device="cuda", generator=gen)
        loss = loss + (out * s).sum()
        sets.append((sc, layer, bev, knn, s))
    loss.backward()
    torch.use_deterministic_algorithms(False)   # the float64 reference uses grid_sample's (atomic) backward
    img64 = dev(wl["img_feat"]).double().requires_grad_(True)
    ref_loss, refs = 0.0, []
    for sc, layer, bev, knn, s in sets:
        w64 = [p_.detach().double().requires_grad_(True) for p_ in layer.parameters()]
        b64 = dev(sc["bev"]).double().requires_grad_(True)
        ro = torch_layer(b64, img64, pts.double(), wl["num_points"], knn, sc["geom"], dev(wl["calib"]).double(), w64)
        ref_loss = ref_loss + (ro * s.double()).sum()
        refs.append((w64, b64))
    ref_loss.backward()
    tol = 2e-3 if mode == "simt" else 5e-3
    bad = []

    def close(a, b, name, t=tol):
        l2, mx = _rel(a, b), (a.double() - b).abs().max().item() / max(b.abs().max().item(), 1e-12)
        if not (l2 < t and mx < 10 * t):
            bad.append(f"{name}: rel L2 {l2:.3e}, rel max {mx:.3e}")

    close(img.grad, img64.grad, "d img_feat")
    for (sc, layer, bev, _, _), (w64, b64) in zip(sets, refs):
        close(bev.grad, b64.grad, f"C={sc['C']} d bev", 1e-6)
        for name, p_, r_ in zip(["W1", "b1", "W2", "b2", "W3", "b3"], layer.parameters(), w64):
            close(p_.grad, r_.grad, f"C={sc['C']} d {name}")
    assert not bad, bad


def test_edge_cases_empty_frame_no_neighbours_taps_outside(dcf):
    # a frame without points (its rows, cells and camera taps vanish)
    wl, sc, frames, knn, w, gout = _scale1(dcf, 64, seed=35, num_points=[0, 9000, 0, 12000])
    for mode in ("fp32", "simt"):
        det = _bwd(dcf, frames, knn, sc, w, gout, mode, True)
        ref = _bwd(dcf, frames, knn, sc, w, gout, mode, False)
        for name, x, y in zip(NAMES, det, ref):
            assert torch.isfinite(x).all() and _rel(x, y) <= 1e-5, (mode, name)
        assert det[6][0].abs().max() == 0 and det[6][2].abs().max() == 0
    # no cell has a neighbour: every weight gradient is zero (b3 too: n_valid = 0 everywhere)
    empty = torch.full_like(knn, -1)
    for mode in ("fp32", "simt"):
        det = _bwd(dcf, frames, empty, sc, w, gout, mode, True)
        torch.cuda.synchronize()
        for name, x in zip(NAMES, det):
            assert x.abs().max() == 0, (mode, name)
    # camera taps: points far outside the map, on its border (two of four taps inside) and past num_points contribute
    # nothing / only their inside taps, exactly as in the atomic path
    B, N, Ci, Hf, Wf = 2, 4096, 64, 30, 40
    gen = torch.Generator(device="cuda").manual_seed(8)
    uv = torch.rand((B, N, 2), device="cuda", generator=gen) * torch.tensor([640.0, 480.0], device="cuda")
    uv[:, :512] = uv[:, :512] * 3 - 640        # mostly outside
    uv[:, 512:640, 0] = 639.9                  # right border: two taps outside
    uv[:, 640:768, 1] = -7.0                   # above the map: one row of taps outside
    pts = torch.zeros((B, N, 3), device="cuda")
    cnt = torch.tensor([N, N - 1000], dtype=torch.int64, device="cuda")
    gfeat = torch.randn((B, N, Ci), device="cuda", generator=gen)
    img = torch.empty((B, Ci, Hf, Wf), device="cuda")
    det = dcf.ops.point_gather_bwd(gfeat, img, pts, cnt, uv=uv, img_size=(640.0, 480.0), deterministic=True)
    ref = dcf.ops.point_gather_bwd(gfeat, img, pts, cnt, uv=uv, img_size=(640.0, 480.0))
    assert torch.isfinite(det).all() and _rel(det, ref) <= 1e-6
    # rows at or beyond num_points add nothing: changing their gradient changes nothing
    gfeat2 = gfeat.clone()
    gfeat2[1, N - 1000:] = 1e6
    assert torch.equal(dcf.ops.point_gather_bwd(gfeat2, img, pts, cnt, uv=uv, deterministic=True), det)


def test_cuda_graph_replay_equals_eager(dcf, deterministic):
    wl = dcf.synthetic.make_workload(dict(dcf.synthetic.workload("yaml"), batch=2, scales=(1,)), seed=37, c_img=128,
                                     channels=[64, 64, 128, 192, 256])
    sc = wl["scales"][0]
    pts, cnt = dev(wl["points"]), dev(wl["num_points"])
    frames = dcf.FrameContext(pts, cnt, dcf.ops.BucketGrid(*dcf.geometry.bucket_grid(wl["config"])))
    frames.gather(dev(wl["img_feat"]), calib=wl["calib"])
    frames.knn(sc["H"], sc["W"], sc["geom"], wl["radius"], wl["k"])
    layer = dcf.ContinuousFusion(128, 64, k=wl["k"], radius=wl["radius"], geom=sc["geom"], mode="fp32").cuda()
    with torch.no_grad():
        for p_, w_ in zip(layer.parameters(), sc["weights"]):
            p_.copy_(dev(w_))
    bev = dev(sc["bev"])
    seed = torch.randn(bev.shape, device="cuda", generator=torch.Generator(device="cuda").manual_seed(3))
    feat = frames.feat.detach().clone().requires_grad_(True)
    frames.feat = feat

    def step():
        for p_ in list(layer.parameters()) + [feat]:
            p_.grad = None
        (layer(bev, frames=frames) * seed).sum().backward()
        return [p_.grad for p_ in list(layer.parameters()) + [feat]]

    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        eager = [g.clone() for g in step()]
        step()
    torch.cuda.current_stream().wait_stream(side)
    torch.cuda.synchronize()
    graph = torch.cuda.CUDAGraph()
    for p_ in list(layer.parameters()) + [feat]:
        p_.grad = None
    with torch.cuda.graph(graph):
        (layer(bev, frames=frames) * seed).sum().backward()
    static = [p_.grad for p_ in list(layer.parameters()) + [feat]]
    graph.replay()
    torch.cuda.synchronize()
    r1 = [g.clone() for g in static]
    graph.replay()
    torch.cuda.synchronize()
    for a, b, c in zip(r1, static, eager):
        assert torch.equal(a, b) and torch.equal(a, c)


_CHILD = r"""
import hashlib, os, sys
import numpy as np, torch
torch.use_deterministic_algorithms(True)
sys.path.insert(0, sys.argv[1]); sys.path.insert(0, os.path.join(sys.argv[1], "scripts"))
import dcf_b200 as dcf
from train_step_bench import synthetic_labels
dev = torch.device("cuda")
torch.manual_seed(0)
cfg = dcf.geometry.carla_config(fusion_scales=(1, 2, 3, 4, 5), fusion_k=3)
model = dcf.ObjectDetection_DCF(cfg).to(dev).eval()
crit = dcf.LossTotal(cfg, batch_reduction="sum", generator=torch.Generator(device=dev).manual_seed(1)).to(dev)
opt = torch.optim.Adam(model.parameters(), lr=1e-4, betas=(0.9, 0.999))
B = 2
wl = dcf.synthetic.make_workload(dict(dcf.synthetic.workload("yaml"), batch=B), seed=7)
to = lambda x: torch.from_numpy(np.ascontiguousarray(x)).to(dev)
x_lidar = torch.rand(B, 32, 384, 256, device=dev)
x_image = torch.randint(0, 255, (B, 3, 480, 640), device=dev, dtype=torch.uint8)
ref, num = synthetic_labels(B, 11, dev)
h = hashlib.sha256()
for _ in range(3):
    opt.zero_grad(set_to_none=True)
    pred = model(x_lidar, x_image, pointcloud_raw=to(wl["points"]), num_points_raw=to(wl["num_points"]),
                 projected_loc_uv=to(wl["uv"]))
    pred_cls, pred_reg, _ = torch.split(pred, [4, 14, 14], dim=1)
    loss = crit(ref, num, pred_cls, pred_reg).sum()
    loss.backward()
    opt.step()
    h.update(loss.detach().cpu().numpy().tobytes())
for n, p in model.named_parameters():
    h.update(n.encode()); h.update(p.detach().cpu().numpy().tobytes())
print("DIGEST", h.hexdigest())
"""


def test_two_processes_train_to_the_same_bytes():
    env = dict(os.environ, CUBLAS_WORKSPACE_CONFIG=":4096:8")
    digests = []
    for _ in range(2):
        res = subprocess.run([sys.executable, "-c", _CHILD, ROOT], env=env, capture_output=True, text=True, timeout=900)
        assert res.returncode == 0, res.stderr[-3000:]
        line = [l for l in res.stdout.splitlines() if l.startswith("DIGEST ")]
        assert line, res.stdout[-2000:]
        digests.append(line[-1].split()[1])
    assert digests[0] == digests[1]
