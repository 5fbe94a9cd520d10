"""CPU: host-side logic -- geometry, synthetic generator, the drop-in nn.Module tree, reference parity of the
untouched LiDAR-only path, and post-process plumbing."""
import numpy as np
import pytest
import torch

from oracle import ref_shims


def test_scale_geometry_follows_voxel_mapping(dcf):
    G = dcf.geometry
    cfg = G.carla_config()
    assert G.voxel_scales(cfg) == (5, 4, 0, 120)                 # data_import_carla.py:35-40 with the YAML values
    x0, y0, dx, dy = G.scale_geometry(cfg, 1)
    assert (x0, y0, dx, dy) == (np.float32(0.1), np.float32(-29.875), np.float32(0.2), np.float32(0.25))
    x0, y0, dx, dy = G.scale_geometry(cfg, 4)
    assert (dx, dy) == (np.float32(0.8), np.float32(1.0)) and x0 == np.float32(0.1)
    gx0, gy0, cell, nbx, nby = G.bucket_grid(cfg)
    assert gx0 == 0.0 and gy0 == -30.0 and nbx * cell >= 76.8 and nby * cell >= 64.0


def test_calibration_constants(dcf):
    crt = dcf.geometry.calibration_crt()
    assert crt.shape == (4, 3) and crt.dtype == np.float32
    expect_T = np.array([[-319.42096068, -268.94292664, 11.77212178, 0], [-228.41786897, -2.08561481, 278.42334332, 0],
                         [-0.99910298, -0.00136578, 0.04232468, 0]])
    assert np.allclose(crt.T, expect_T, atol=1e-4)               # SURVEY 8a row I-4
    q = np.array([10, 0, 0, 1.0]) @ crt.astype(np.float64)
    assert np.allclose(q[:2] / q[2], [319.7, 228.6], atol=0.1)


@pytest.mark.parametrize("name", ["tiny", "yaml", "cfg0"])
def test_workloads_have_reference_layout(dcf, name):
    wl = dcf.synthetic.make_workload(name, seed=3)
    pts, uv, cnt = wl["points"], wl["uv"], wl["num_points"]
    B, N, _ = pts.shape
    assert N == wl["config"]["max_num_pc"] and uv.shape == (B, N, 2) and cnt.dtype == np.int64
    for b in range(B):
        n = int(cnt[b])
        assert 0 < n < N
        assert not pts[b, n:].any() and not uv[b, n:].any()      # zero padding rows (data_import_carla.py:263-266)
        assert (pts[b, :n, 0] > 0).all() and (uv[b, :n, 0] > 0).all() and (uv[b, :n, 0] < 480).all()
    # determinism
    wl2 = dcf.synthetic.make_workload(name, seed=3)
    assert np.array_equal(wl2["points"], pts) and np.array_equal(wl2["scales"][0]["bev"], wl["scales"][0]["bev"])
    shapes = dcf.synthetic.scale_shapes(dcf.geometry.carla_config(voxel_length=700, voxel_width=800))
    assert shapes == [(32, 700, 800), (64, 350, 400), (128, 175, 200), (192, 88, 100), (256, 44, 50)]


def test_dropin_module_tree_and_lidar_only_path(dcf):
    cfg = dcf.geometry.carla_config(fusion_scales=(1, 3))
    m = dcf.ObjectDetection_DCF(cfg).eval()
    keys = set(m.state_dict().keys())
    for k in ["lidar_backbone.backbone.layer1.sequential.resblock_0.conv1.weight",
              "lidar_backbone.backbone.layer5.sequential.resblock_5.bn2.running_var",
              "lidar_backbone.backbone.layer2.sequential.resblock_0.down_conv.weight", "lidar_backbone.latconv1.weight",
              "lidar_backbone.bbox3dconv.weight", "fusion.group1.fc1.weight", "fusion.group3.fc3.bias"]:
        assert k in keys, k
    assert m.fusion["group3"].fc1.weight.shape == (128, 131)
    with torch.no_grad():
        y = m(torch.randn(1, 32, 384, 256), None)               # forward(x_lidar, x_image): LiDAR-only, CPU is fine
    assert y.shape == (1, 32, 96, 64)                            # cls4 | reg14 | bbox14 at H/4 x W/4 (model.py:204)
    cls = y[:, :4]
    assert torch.allclose(cls[:, 0] + cls[:, 1], torch.ones_like(cls[:, 0]), atol=1e-5)


@pytest.mark.skipif(not ref_shims.available(), reason="needs the original project: set CF_REFERENCE_DIR to its checkout")
def test_lidar_only_path_equals_reference_model(dcf):
    """Same weights -> same output as the reference's LidarBackboneNetwork, and its checkpoints load."""
    ref = ref_shims.load()
    torch.manual_seed(0)
    ref_net = ref.model.LidarBackboneNetwork().eval()
    cfg = dcf.geometry.carla_config()
    mine = dcf.ObjectDetection_DCF(cfg).eval()
    sd = {"lidar_backbone." + k: v for k, v in ref_net.state_dict().items()}
    missing, unexpected = mine.load_state_dict(sd, strict=False)
    assert not unexpected
    assert all(k.startswith(("image_backbone.", "fusion.")) for k in missing)
    x = torch.randn(1, 32, 384, 256)
    with torch.no_grad():
        rc, rr = ref_net(x.clone())
        y = mine(x.clone(), None)
    assert torch.allclose(y[:, :4], rc, atol=1e-5) and torch.allclose(y[:, 4:18], rr, atol=1e-5)
    # decoded boxes against the reference's OffsettoBbox arithmetic (model.py:121-137), restated on CPU
    assert torch.allclose(ref.model.AnchorBoundingBoxFeature(cfg)(), dcf.model.AnchorBoundingBoxFeature(cfg)(), atol=1e-6)
    # OffsettoBbox hard-codes .cuda() in the reference (model.py:125); restate its arithmetic on CPU for one anchor
    anc = ref.model.AnchorBoundingBoxFeature(cfg)().unsqueeze(0)
    xy = rr[:, :2] * torch.sqrt(anc[:, 3:4] ** 2 + anc[:, 4:5] ** 2) + anc[:, :2]
    whl = torch.exp(rr[:, 3:6]) * anc[:, 3:6]
    assert torch.allclose(y[:, 18:20], xy, atol=1e-5) and torch.allclose(y[:, 21:24], whl, atol=1e-5)


def test_pad_boxes_and_reference_shaped_outputs(dcf):
    a, b = torch.randn(5, 7), torch.zeros(0, 7)
    boxes, counts = dcf.postprocess.pad_boxes([a, b], device="cpu")
    assert boxes.shape == (2, 64, 7) and counts.tolist() == [5, 0]
    assert torch.equal(boxes[0, :5], a) and not boxes[0, 5:].any()
    rows = dcf.PostProcess._rows([a, b], [torch.tensor([0, 3]), torch.tensor([], dtype=torch.int64)])
    assert len(rows[0]) == 2 and rows[1] == [] and torch.equal(rows[0][1], a[3])
