"""GPU: the whole fused layer (K-1..K-4) through ContinuousFusion / the C ABI against the brute-force,
naive-formulation CPU oracle.  Tolerance (Appendix A13): ||out-ref||_inf / max(||ref||_inf, 1e-6) <= 1e-4 in
fp32 modes, 1e-2 in bf16 mode; additionally the fusion DELTA (out - bev) must meet the same bound, so the
N(0,1) BEV input cannot mask an error in the MLP."""
import numpy as np
import pytest
import torch

from _util import cuda_fusion, dev, oracle_fusion, rel_err

pytestmark = pytest.mark.gpu

TOL = {"simt": 1e-4, "fp32": 1e-4, "bf16": 1e-2}


def _compare(wl, outs, knns, ref_outs, ref_knns, tol):
    for sc, o, k, ro, rk in zip(wl["scales"], outs, knns, ref_outs, ref_knns):
        assert np.array_equal(k, rk), f"group {sc['group']}: knn mismatch"
        assert o.shape == ro.shape and o.dtype == np.float32
        assert rel_err(o, ro) <= tol, f"group {sc['group']}: rel err {rel_err(o, ro):.3e}"
        d, rd = o - sc["bev"], ro - sc["bev"]
        assert np.abs(rd).max() > 1e-2                      # the layer actually contributes
        assert rel_err(d, rd) <= tol * 2, f"group {sc['group']}: delta rel err {rel_err(d, rd):.3e}"


@pytest.mark.parametrize("mode", ["simt", "fp32", "bf16"])
@pytest.mark.parametrize("name,seed,use_uv", [("tiny", 11, False), ("tiny", 12, True)])
def test_fusion_matches_oracle_small(dcf, oracle, mode, name, seed, use_uv):
    wl = dcf.synthetic.make_workload(name, seed=seed, c_img=32, img_hw=(24, 32))
    outs, knns = cuda_fusion(dcf, wl, mode, use_uv=use_uv)
    ref_outs, ref_knns = oracle_fusion(oracle, wl, use_uv=use_uv)
    _compare(wl, outs, knns, ref_outs, ref_knns, TOL[mode])


@pytest.mark.parametrize("mode", ["simt", "fp32", "bf16"])
def test_fusion_all_five_scales_yaml_grid(dcf, oracle, mode):
    """The reference YAML's 384x256 grid, all five residual groups (C = 32..256), 128-channel camera map."""
    wl = dcf.synthetic.make_workload(dict(dcf.synthetic.workload("yaml"), batch=1, k=5), seed=13)
    outs, knns = cuda_fusion(dcf, wl, mode)
    ref_outs, ref_knns = oracle_fusion(oracle, wl)
    _compare(wl, outs, knns, ref_outs, ref_knns, TOL[mode])


@pytest.mark.parametrize("mode", ["fp32", "bf16"])
def test_fusion_in_place_equals_out_of_place(dcf, mode):
    """out may alias bev (inference): same bits as the out-of-place call, on the compacted and the plain tile path."""
    wl = dcf.synthetic.make_workload(dict(dcf.synthetic.workload("yaml"), batch=2, k=5), seed=17)
    a, _ = cuda_fusion(dcf, wl, mode)
    b, _ = cuda_fusion(dcf, wl, mode, inplace=True)
    for x, y in zip(a, b):
        assert np.array_equal(x, y)


def test_fuse_scales_matches_per_layer_calls(dcf):
    """fuse_scales (side streams, memcpy + in-place layer) returns what the layers return one by one, and leaves bev intact."""
    wl = dcf.synthetic.make_workload(dict(dcf.synthetic.workload("yaml"), batch=2, k=3), seed=18)
    ref, _ = cuda_fusion(dcf, wl, "fp32")
    pts, cnt, img = dev(wl["points"]), dev(wl["num_points"]), dev(wl["img_feat"])
    frames = dcf.prepare_frames(pts, cnt, img, config=wl["config"], calib=wl["calib"])
    layers, bevs = [], []
    for sc in wl["scales"]:
        layer = dcf.ContinuousFusion(img.shape[1], sc["C"], k=wl["k"], radius=wl["radius"], geom=sc["geom"], mode="fp32").cuda()
        with torch.no_grad():
            for prm, w in zip((layer.fc1.weight, layer.fc1.bias, layer.fc2.weight, layer.fc2.bias, layer.fc3.weight,
                               layer.fc3.bias), sc["weights"]):
                prm.copy_(dev(w))
        layers.append(layer.eval())
        bevs.append(dev(sc["bev"]))
    outs = dcf.fuse_scales(frames, layers, bevs)
    torch.cuda.synchronize()
    for sc, o, r, bv in zip(wl["scales"], outs, ref, bevs):
        assert np.array_equal(o.cpu().numpy(), r)
        assert np.array_equal(bv.cpu().numpy(), sc["bev"])


@pytest.mark.parametrize("mode", ["fp32", "bf16"])
def test_point_mlp1_multi_equals_per_scale_calls(dcf, mode):
    """cf_point_mlp1_multi (one launch, A operand packed once) == cf_point_mlp1 per scale, bit for bit, incl. ragged frames."""
    torch.manual_seed(19)
    B, N, Ci = 3, 1000, 128
    feat = torch.randn(B, N, Ci, device="cuda")
    pts = torch.randn(B, N, 3, device="cuda") * 20
    cnt = torch.tensor([1000, 0, 517], dtype=torch.int64, device="cuda")
    Cs = [32, 64, 128, 192, 256]
    W1s = [torch.randn(c, Ci + 3, device="cuda") * 0.1 for c in Cs]
    b1s = [torch.randn(c, device="cuda") for c in Cs]
    pks = [dcf.ops.PackedWeights().w1(w, mode) for w in W1s]
    multi = dcf.ops.point_mlp1_multi(feat, pts, cnt, W1s, b1s, pks, mode=mode,
                                     outs=[torch.zeros(B, N, c, device="cuda") for c in Cs])
    for w, b, pk, tm, c in zip(W1s, b1s, pks, multi, Cs):
        one = dcf.ops.point_mlp1(feat, pts, cnt, w, b, mode=mode, packed=pk, out=torch.zeros(B, N, c, device="cuda"))
        torch.cuda.synchronize()
        assert torch.equal(one, tm)
        assert one[0].abs().max() > 0 and float(tm[1].abs().max()) == 0.0 and float(tm[2, 517:].abs().max()) == 0.0


@pytest.mark.parametrize("mode", ["fp32", "bf16"])
@pytest.mark.parametrize("Ci", [16, 48, 96])
def test_point_mlp1_camera_widths(dcf, mode, Ci):
    """cf_point_mlp1 with and without a packed image, incl. ragged frames, at camera widths the other tests do not use.
    Ci % 32 == 16 has no tensor-core operand layout: the FFMA kernel runs, bit-equal to "simt".  Ci = 96 is a one-scale
    call of the tensor-core kernel: bit-equal to cf_point_mlp1_multi, and within the mode's tolerance of "simt".  Rows past
    num_points stay untouched."""
    torch.manual_seed(43)
    B, N, C = 3, 1000, 64
    feat = torch.randn(B, N, Ci, device="cuda")
    pts = torch.randn(B, N, 3, device="cuda") * 20
    cnt = torch.tensor([N, 0, 517], dtype=torch.int64, device="cuda")
    W1 = torch.randn(C, Ci + 3, device="cuda") * 0.1
    b1 = torch.randn(C, device="cuda")
    untouched = lambda t: bool((t[1] == 7.0).all()) and bool((t[2, 517:] == 7.0).all())
    live = lambda t: torch.cat([t[0], t[2, :517]]).cpu().numpy()
    ref = dcf.ops.point_mlp1(feat, pts, cnt, W1, b1, mode="simt", out=torch.full((B, N, C), 7.0, device="cuda"))
    pk = dcf.ops.PackedWeights().w1(W1, mode)
    for packed in (None, pk):
        got = dcf.ops.point_mlp1(feat, pts, cnt, W1, b1, mode=mode, packed=packed, out=torch.full((B, N, C), 7.0, device="cuda"))
        torch.cuda.synchronize()
        assert untouched(ref) and untouched(got)
        if Ci % 32:
            assert torch.equal(got, ref), f"packed={packed is not None}"
        else:
            multi, = dcf.ops.point_mlp1_multi(feat, pts, cnt, [W1], [b1], [pk], mode=mode,
                                              outs=[torch.full((B, N, C), 7.0, device="cuda")])
            assert torch.equal(got, multi), f"packed={packed is not None}"
            assert rel_err(live(got), live(ref)) <= TOL[mode], f"packed={packed is not None}: {rel_err(live(got), live(ref)):.3e}"


def test_bf16_tables_layer1_is_the_rounded_fp32_table(dcf):
    """CF_MODE_BF16_TABLES ("bf16t"): cf_point_mlp1_multi writes exactly round-to-nearest-even bf16 of the CF_MODE_BF16 table
    (full tiles leave through TMA stores, the partial tile of a frame through direct stores), rows past num_points stay
    untouched, and the single-scale entry point gives the same rows."""
    torch.manual_seed(23)
    B, N, Ci = 3, 1000, 128
    feat = torch.randn(B, N, Ci, device="cuda")
    pts = torch.randn(B, N, 3, device="cuda") * 20
    cnt = torch.tensor([1000, 0, 517], dtype=torch.int64, device="cuda")
    Cs = [32, 64, 128, 192, 256]
    W1s = [torch.randn(c, Ci + 3, device="cuda") * 0.1 for c in Cs]
    b1s = [torch.randn(c, device="cuda") for c in Cs]
    pk = [dcf.ops.PackedWeights().w1(w, "bf16") for w in W1s]
    pkt = [dcf.ops.PackedWeights().w1(w, "bf16t") for w in W1s]
    ref = dcf.ops.point_mlp1_multi(feat, pts, cnt, W1s, b1s, pk, mode="bf16", outs=[torch.zeros(B, N, c, device="cuda") for c in Cs])
    got = dcf.ops.point_mlp1_multi(feat, pts, cnt, W1s, b1s, pkt, mode="bf16t",
                                   outs=[torch.zeros(B, N, c, device="cuda", dtype=torch.bfloat16) for c in Cs])
    torch.cuda.synchronize()
    for r, g, w, b, p, c in zip(ref, got, W1s, b1s, pkt, Cs):
        assert g.dtype == torch.bfloat16 and torch.equal(g, r.to(torch.bfloat16)), f"C={c}"
        assert float(g[1].abs().max()) == 0.0 and float(g[2, 517:].abs().max()) == 0.0 and float(g[0].abs().max()) > 0
        one = dcf.ops.point_mlp1(feat, pts, cnt, w, b, mode="bf16t", packed=p, out=torch.zeros(B, N, c, device="cuda", dtype=torch.bfloat16))
        assert torch.equal(one, g), f"C={c}: single-scale entry point"
    with pytest.raises(ValueError, match="bfloat16"):
        dcf.ops.point_mlp1_multi(feat, pts, cnt, W1s, b1s, pkt, mode="bf16t", outs=[torch.zeros(B, N, c, device="cuda") for c in Cs])


def test_layer1_direct_store_path_equals_tma_store_path():
    """CF_NO_TMA_STORE=1 (read once per process, hence the child process) makes the layer-1 kernel store every tile directly,
    the path it takes when the driver has no tensor maps: same bits as the staged TMA stores, in "bf16" and "bf16t"."""
    import os
    import subprocess
    import sys
    code = r"""
import sys, torch
sys.path.insert(0, %r)
import dcf_b200 as dcf
torch.manual_seed(41)
B, N, Ci = 2, 700, 128
feat = torch.randn(B, N, Ci, device="cuda"); pts = torch.randn(B, N, 3, device="cuda") * 20
cnt = torch.tensor([700, 389], dtype=torch.int64, device="cuda")
Cs = [32, 64, 128, 192, 256]
W1s = [torch.randn(c, Ci + 3, device="cuda") * 0.1 for c in Cs]; b1s = [torch.randn(c, device="cuda") for c in Cs]
for mode in ("bf16", "bf16t"):
    pk = [dcf.ops.PackedWeights().w1(w, mode) for w in W1s]
    outs = dcf.ops.point_mlp1_multi(feat, pts, cnt, W1s, b1s, pk, mode=mode,
                                    outs=[torch.zeros(B, N, c, device="cuda", dtype=dcf.ops.table_dtype(mode)) for c in Cs])
    torch.cuda.synchronize()
    torch.save([o.cpu() for o in outs], sys.argv[1] + mode + ".pt")
""" % os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    import tempfile
    with tempfile.TemporaryDirectory() as d:
        logs = {}
        for tag, env in (("tma_", {}), ("direct_", {"CF_NO_TMA_STORE": "1"})):
            r = subprocess.run([sys.executable, "-c", code, os.path.join(d, tag)], capture_output=True, text=True, timeout=300,
                               env=dict(os.environ, CF_DEBUG_LAUNCH="1", **env))
            assert r.returncode == 0, r.stderr[-2000:]
            logs[tag] = r.stderr
        assert "staged TMA stores 1" in logs["tma_"] and "staged TMA stores 0" in logs["direct_"] and "staged TMA stores 1" not in logs["direct_"]
        for mode in ("bf16", "bf16t"):
            a = torch.load(os.path.join(d, "tma_" + mode + ".pt"))
            b = torch.load(os.path.join(d, "direct_" + mode + ".pt"))
            for x, y in zip(a, b):
                assert torch.equal(x, y) and float(x[1, 389:].abs().max()) == 0.0 and float(x[0].abs().max()) > 0


@pytest.mark.parametrize("name,seed", [("tiny", 31), ("yaml", 32)])
def test_bf16_tables_fused_layer_equals_bf16_mode_on_the_rounded_table(dcf, name, seed):
    """The fused kernels of "bf16t" differ from "bf16" only in how a table row is loaded: fed the same (bf16-representable)
    rows they must give the same bits, at every scale width, out of place and in place."""
    wl = dcf.synthetic.make_workload(name, seed=seed)
    pts, cnt, img = dev(wl["points"]), dev(wl["num_points"]), dev(wl["img_feat"])
    frames = dcf.prepare_frames(pts, cnt, img, config=wl["config"], calib=wl["calib"])
    for sc in wl["scales"]:
        w1, b1, w2, b2, w3, b3 = [dev(w) for w in sc["weights"]]
        bev = dev(sc["bev"])
        knn = frames.knn(sc["H"], sc["W"], sc["geom"], wl["radius"], wl["k"])
        Th = dcf.ops.point_mlp1(frames.feat, pts, cnt, w1, b1, mode="bf16t")
        assert Th.dtype == torch.bfloat16
        a, _ = dcf.ops.fusion_fwd(bev, Th, knn, sc["geom"], w1, w2, b2, w3, b3, mode="bf16t")
        b, _ = dcf.ops.fusion_fwd(bev, Th.float(), knn, sc["geom"], w1, w2, b2, w3, b3, mode="bf16")
        assert torch.equal(a, b), f"C={sc['C']}"
        io = bev.clone()
        dcf.ops.fusion_fwd(io, Th, knn, sc["geom"], w1, w2, b2, w3, b3, mode="bf16t", out=io)
        assert torch.equal(io, a), f"C={sc['C']} in place"
        with pytest.raises(TypeError, match="bfloat16"):
            dcf.ops.fusion_fwd(bev, Th.float(), knn, sc["geom"], w1, w2, b2, w3, b3, mode="bf16t")


def test_bf16_tables_mode_is_inference_only(dcf):
    wl = dcf.synthetic.make_workload("tiny", seed=33, c_img=32, img_hw=(24, 32))
    sc = wl["scales"][0]
    layer = dcf.ContinuousFusion(32, sc["C"], k=wl["k"], radius=wl["radius"], geom=sc["geom"], mode="bf16t").cuda()
    frames = dcf.prepare_frames(dev(wl["points"]), dev(wl["num_points"]), dev(wl["img_feat"]), config=wl["config"], calib=wl["calib"])
    with torch.no_grad():
        out = layer(dev(sc["bev"]), frames=frames)
    assert out.shape == sc["bev"].shape and bool(torch.isfinite(out).all())
    with pytest.raises(RuntimeError, match="inference only"):
        layer(dev(sc["bev"]), frames=frames)


def test_fusion_channels_last_map_equals_nchw(dcf):
    wl = dcf.synthetic.make_workload("tiny", seed=14, c_img=64, img_hw=(30, 40))
    a, _ = cuda_fusion(dcf, wl, "simt", channels_last=False)
    b, _ = cuda_fusion(dcf, wl, "simt", channels_last=True)
    for x, y in zip(a, b):
        assert np.array_equal(x, y)


def test_fusion_empty_frame_is_identity(dcf):
    """A frame with no points (or no point within the radius) must return bev unchanged (A4/A10)."""
    wl = dcf.synthetic.make_workload("tiny", seed=15, c_img=32, img_hw=(24, 32))
    wl["num_points"][:] = 0
    for mode in ("simt", "fp32", "bf16"):
        outs, knns = cuda_fusion(dcf, wl, mode)
        for sc, o, k in zip(wl["scales"], outs, knns):
            assert (k == -1).all()
            assert np.array_equal(o, sc["bev"])


def test_fusion_linearity_in_last_layer(dcf):
    """Property (size independent): the layer is affine in (W3, b3): f(2*W3, 2*b3) - bev = 2 (f(W3,b3) - bev)."""
    wl = dcf.synthetic.make_workload("tiny", seed=16, c_img=32, img_hw=(24, 32))
    a, _ = cuda_fusion(dcf, wl, "fp32")
    for sc in wl["scales"]:
        w = list(sc["weights"])
        w[4], w[5] = w[4] * 2, w[5] * 2
        sc["weights"] = tuple(w)
    b, _ = cuda_fusion(dcf, wl, "fp32")
    for sc, x, y in zip(wl["scales"], a, b):
        assert rel_err(y - sc["bev"], 2 * (x - sc["bev"])) < 1e-5


def test_module_rejects_bad_inputs(dcf):
    layer = dcf.ContinuousFusion(32, 32, geom=(0.0, 0.0, 1.0, 1.0)).cuda()
    with pytest.raises(ValueError):
        layer(torch.zeros(1, 16, 4, 4, device="cuda"), torch.zeros(1, 32, 4, 4, device="cuda"),
              torch.zeros(1, 8, 3, device="cuda"), torch.tensor([3]))
    with pytest.raises(ValueError):
        dcf.ContinuousFusion(32, 40)
    for c in (48, 160, 224):       # multiples of 16 without a tensor-core instantiation: rejected at construction ...
        with pytest.raises(ValueError, match="tensor-core"):
            dcf.ContinuousFusion(32, c, mode="fp32")
        dcf.ContinuousFusion(32, c, mode="simt")   # ... but fine on the CUDA-core path
    bev = torch.zeros(1, 32, 4, 4, device="cuda")
    T = torch.zeros(1, 8, 32, device="cuda")
    knn = torch.full((1, 4, 4, 3), -1, dtype=torch.int32, device="cuda")
    w = [torch.zeros(32, 35, device="cuda"), torch.zeros(32, 32, device="cuda"), torch.zeros(32, device="cuda"),
         torch.zeros(32, 32, device="cuda"), torch.zeros(32, device="cuda")]
    with pytest.raises(ValueError, match="out must be"):   # a strided / wrongly shaped output is never written through
        dcf.ops.fusion_fwd(bev, T, knn, (0.0, 0.0, 1.0, 1.0), *w, out=torch.zeros(1, 32, 4, 8, device="cuda")[..., ::2])
    cl = torch.zeros(1, 32, 4, 4, device="cuda").contiguous(memory_format=torch.channels_last)
    with pytest.raises(ValueError, match="out must be|in-place"):
        dcf.ops.fusion_fwd(cl, T, knn, (0.0, 0.0, 1.0, 1.0), *w, out=cl)
    with pytest.raises(ValueError):
        dcf.ContinuousFusion(32, 32, k=17)


def test_config2_density_k10_bf16_properties(dcf, oracle):
    """BASELINE configs[2] shape at reduced batch: 64-beam density (~110k points, max_num_pc = 131072), K = 10, bf16
    MLP, all five scales of the 700x800 BEV.  Full-size checks: KNN bit-exact against the oracle on sampled rows of
    cells at scale 1 and on every cell of scales 4-5; fused features within 1e-2 (A12) of the oracle on scale 5, and
    size-independent properties elsewhere (cells without a neighbour are untouched; delta is finite and bounded)."""
    wl = dcf.synthetic.make_workload(dict(dcf.synthetic.workload("cfg2"), batch=1), seed=31)
    n = int(wl["num_points"][0])
    assert 90000 < n <= 131072 and wl["k"] == 10
    outs, knns = cuda_fusion(dcf, wl, "bf16")
    pts = wl["points"][0]
    r2 = np.float32(wl["radius"]) ** 2
    for sc, out, knn in zip(wl["scales"], outs, knns):
        H, W = sc["H"], sc["W"]
        x0, y0, dx, dy = sc["geom"]
        rows = range(H) if sc["group"] >= 4 else np.sort(np.random.default_rng(sc["group"]).choice(H, 3, replace=False))
        for r in rows:
            ref = oracle.knn_bruteforce(pts, n, H, W, x0, y0, dx, dy, r2, 10, cell_range=(int(r) * W, (int(r) + 1) * W))
            assert np.array_equal(knn[0, r], ref), f"group {sc['group']} row {r}"
        empty = (knn[0] < 0).all(-1)
        assert np.array_equal(out[0][:, empty], sc["bev"][0][:, empty])          # untouched where nothing is in reach
        delta = out[0] - sc["bev"][0]
        assert np.isfinite(delta).all() and np.abs(delta[:, ~empty]).max() > 1e-3
    sc = wl["scales"][4]
    feat = oracle.gather_points(wl["img_feat"][0], oracle.project_points(pts[:n], wl["calib"]))
    ref = oracle.fusion_mlp(sc["bev"][0], feat, pts, knns[4][0], sc["geom"], sc["weights"])
    assert rel_err(outs[4][0], ref) <= 1e-2
    assert rel_err(outs[4][0] - sc["bev"][0], ref - sc["bev"][0]) <= 2e-2


def test_fusion_runner_graph_replay_matches_eager(dcf):
    """FusionRunner (fixed-shape pipeline replayed as one CUDA graph on static buffers, in place) == the eager modules,
    for two different batches pushed through the same runner."""
    cfg = dict(dcf.synthetic.workload("yaml"), batch=2, k=3)
    layers = None
    runner = None
    for seed in (31, 32):
        wl = dcf.synthetic.make_workload(cfg, seed=seed)
        ref, _ = cuda_fusion(dcf, wl, "fp32")
        if layers is None:
            layers = []
            for sc in wl["scales"]:
                layer = dcf.ContinuousFusion(wl["img_feat"].shape[1], sc["C"], k=wl["k"], radius=wl["radius"], geom=sc["geom"],
                                             mode="fp32").cuda()
                layers.append(layer.eval())
            grid = dcf.ops.BucketGrid(*dcf.geometry.bucket_grid(wl["config"], None))
            size = (float(wl["config"]["image_width"]), float(wl["config"]["image_height"]))
            runner = dcf.FusionRunner(layers, grid, 2, wl["points"].shape[1], wl["img_feat"].shape[1:],
                                      [sc["bev"].shape[1:] for sc in wl["scales"]], calib=wl["calib"], img_size=size)
        with torch.no_grad():
            for layer, sc in zip(layers, wl["scales"]):
                for prm, w in zip((layer.fc1.weight, layer.fc1.bias, layer.fc2.weight, layer.fc2.bias, layer.fc3.weight,
                                   layer.fc3.bias), sc["weights"]):
                    prm.copy_(dev(w))
        # weights changed in place: the packed operand images must be refreshed before the graph is replayed
        runner.refresh_weights()
        runner.points.copy_(dev(wl["points"]))
        runner.num_points.copy_(dev(wl["num_points"]))
        runner.img_feat.copy_(dev(wl["img_feat"]))
        for d, sc in zip(runner.bevs, wl["scales"]):
            d.copy_(dev(sc["bev"]))
        outs = runner()
        torch.cuda.synchronize()
        for o, r in zip(outs, ref):
            assert np.array_equal(o.cpu().numpy(), r)
