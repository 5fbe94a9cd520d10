"""Generate tests/golden/*.npz by running the UNMODIFIED reference (imported from $CF_REFERENCE_DIR through
oracle/ref_shims.py) on seeded inputs:

    CF_REFERENCE_DIR=<checkout of the original project> python oracle/gen_golden.py

Each fixture stores the inputs and the reference's outputs; tests compare the CPU oracle (CPU suite) and
the CUDA path (GPU suite) against them.  numpy 2.3.5 / torch 2.11 / scipy 1.18.1 (SURVEY 8c: the reference's
SAT arithmetic depends on numpy >= 2 scalar promotion).
"""
from __future__ import annotations

import math
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[0] = ROOT  # replace the script directory so that `oracle` is the package, not oracle.py
from oracle import ref_shims as R  # noqa: E402
import dcf_b200  # noqa: E402

OUT = os.path.join(ROOT, "tests", "golden")


def car_boxes(rng, n, x=(0, 70), y=(-30, 30), z=(-2.0, -1.0)):
    c = np.stack([rng.uniform(*x, n), rng.uniform(*y, n), rng.uniform(*z, n)], axis=1)
    s = np.array([4.0, 2.0, 1.5]) * np.exp(0.1 * rng.normal(size=(n, 3)))
    yaw = rng.uniform(-math.pi, math.pi, (n, 1))
    return np.concatenate([c, s, yaw], axis=1).astype(np.float32)


def edge_case_boxes():
    b = [
        [10, 0, -1, 4, 2, 1.5, 0.0],
        [14, 0, -1, 4, 2, 1.5, 0.0],          # shares an edge with box 0 (closed-interval SAT -> overlap)
        [18.0001, 0, -1, 4, 2, 1.5, 0.0],     # 1e-4 gap from box 1 -> separate
        [10, 0, -1, 4, 2, 1.5, 0.0],          # identical to box 0
        [30, 5, -1, 4, 2, 1.5, math.pi / 4],
        [30, 5, -1, 2, 1, 1.0, math.pi / 4],  # nested in box 4
        [32.5, 7.5, -1, 4, 2, 1.5, -math.pi / 4],  # corner region of box 4
        [50, -10, -1, 4, 2, 1.5, math.pi / 2],
        [50, -7, -1, 4, 2, 1.5, 0.0],         # T-junction touching box 7
        [60, 20, -1, 4, 2, 1.5, 3.0],
        [0.5, -29.5, -1, 4, 2, 1.5, 1.0],
    ]
    return np.array(b, dtype=np.float32)


def chain_fixture():
    """The evaluator's chain on a decoded prediction map (test.py:79-85): split -> get_bboxes -> NMS_SAT.  The box
    channels hold decoded car-sized boxes (model.py:129 guarantees l, w > 0), ~3 % of the anchors pass the score."""
    rng = np.random.default_rng(19)
    B, H, W = 3, 44, 50
    cls = rng.random((B, 4, H, W)).astype(np.float32) * 0.7
    for a in (1, 3):
        cls[:, a] = np.where(rng.random((B, H, W)) < 0.035, 0.8 + 0.2 * rng.random((B, H, W)), cls[:, a]).astype(np.float32)
    cls[2, 1] = 0.1
    cls[2, 3] = 0.2                                  # a frame without detections
    box = np.zeros((B, 14, H, W), np.float32)
    for a in range(2):
        bx = car_boxes(rng, B * H * W, x=(0, 70), y=(-30, 30)).reshape(B, H, W, 7)
        box[:, 7 * a:7 * a + 7] = bx.transpose(0, 3, 1, 2)
    boxes = R.get_bboxes(torch.from_numpy(cls), torch.from_numpy(box), 0.8)
    keep = R.nms_sat(boxes)
    data = dict(cls=cls, box=box, thr=np.float32(0.8), counts=np.array([b.shape[0] for b in boxes]))
    for b in range(B):
        data[f"boxes_{b}"] = boxes[b].numpy().reshape(-1, 7)
        data[f"keep_{b}"] = keep[b]
        print("chain frame", b, boxes[b].shape[0], "->", len(keep[b]))
    np.savez_compressed(os.path.join(OUT, "postprocess_chain.npz"), **data)


def loss_fixture(regress_type, seed):
    """LossTotal (loss.py:33-189) of the unmodified reference on a seeded batch: boxes inside, on the border and outside the
    map, overlapping windows, a frame with the maximum of 20 boxes (more positives than the 128 kept) and one with 2."""
    cfg = dcf_b200.geometry.carla_config(regress_type=regress_type)
    rng = np.random.default_rng(seed)
    B, M, H, W = 4, 20, 96, 64
    ref = np.zeros((B, M, 8), np.float32)
    num = np.array([6, 20, 2, 11], np.int64)
    for b in range(B):
        n = int(num[b])
        ref[b, :n, 0] = rng.uniform(-3, 74, n)      # a few centres fall outside 0..70 m / -30..30 m
        ref[b, :n, 1] = rng.uniform(-33, 33, n)
        ref[b, :n, 2] = rng.uniform(-2, -1, n)
        ref[b, :n, 3:6] = np.array([4, 2, 1.5]) * np.exp(0.1 * rng.normal(size=(n, 3)))
        ref[b, :n, 6] = rng.uniform(-math.pi, math.pi, n)
        ref[b, :n, 7] = 1
    ref[3, 0, :2] = (0.1, -29.9)                    # corner cell: the window is clipped on two sides
    ref[3, 1, :2] = (0.5, -29.5)                    # overlaps the window of box 0
    ref[3, 2, :2] = (-0.1, 0.0)                     # int() truncates -0.125 to cell 0: counted as inside (loss.py:86,88)
    pred_cls = rng.normal(size=(B, 4, H, W)).astype(np.float32)
    pred_reg = (0.3 * rng.normal(size=(B, 14, H, W))).astype(np.float32)
    R_ = cfg["positive_range"]
    L = 4 * (cfg["neg_sample_threshold"] + 1)
    keys = rng.random((B, M * R_ * R_)).astype(np.float32)
    cand = np.stack([rng.integers(0, H, (B, L)), rng.integers(0, W, (B, L))], axis=2).astype(np.int32)
    losses, pos, neg = R.loss_total(cfg, ref, num, pred_cls, pred_reg, keys, cand)
    pos_a = -np.ones((B, cfg["pos_sample_threshold"]), np.int32)
    neg_a = -np.ones((B, cfg["neg_sample_threshold"] + 1), np.int32)
    for b in range(B):
        pos_a[b, :len(pos[b])] = pos[b]
        neg_a[b, :len(neg[b])] = neg[b]
    return dict(ref=ref, num=num, pred_cls=pred_cls, pred_reg=pred_reg, keys=keys, cand=cand, losses=losses, pos=pos_a,
                npos=np.array([len(x) for x in pos], np.int32), neg=neg_a, nneg=np.array([len(x) for x in neg], np.int32),
                regress_type=np.int32(regress_type))


def main():
    os.makedirs(OUT, exist_ok=True)
    ref = R.load()
    if "--only-chain" in sys.argv:
        return chain_fixture()
    chain_fixture()
    # ---- NMS_SAT keep lists (test.py:142-175)
    frames = {}
    for n in (0, 1, 2, 50, 200, 600, 2000):
        frames[f"uniform_{n}"] = dcf_b200.synthetic.nms_boxes(n, n) if n else np.zeros((0, 7), np.float32)
    rng = np.random.default_rng(11)
    frames["dense_300"] = car_boxes(rng, 300, x=(10, 30), y=(-8, 8))   # heavy overlap
    frames["edge_cases"] = edge_case_boxes()
    data = {}
    for name, boxes in frames.items():
        keep = R.nms_sat([torch.from_numpy(boxes)])[0]
        data[f"{name}__boxes"] = boxes
        data[f"{name}__keep"] = keep
        print("nms_sat", name, boxes.shape[0], "->", len(keep))
    np.savez_compressed(os.path.join(OUT, "nms_sat.npz"), **data)

    # ---- pairwise SAT on the edge cases + a random set (separation_axis_theorem.py:66-94)
    boxes = np.concatenate([edge_case_boxes(), car_boxes(np.random.default_rng(12), 53, x=(5, 40), y=(-10, 10))])
    n = boxes.shape[0]
    m = np.zeros((n, n), np.uint8)
    verts = []
    for i in range(n):
        t = torch.from_numpy(boxes[i])
        verts.append(ref.sat.get_vertice_rect(t[:3].numpy(), t[3:6].numpy(), t[6].numpy()))
    for i in range(n):
        for j in range(n):
            m[i, j] = ref.sat.separating_axis_theorem(verts[i], verts[j])
    np.savez_compressed(os.path.join(OUT, "sat_pairs.npz"), boxes=boxes, overlap=m,
                        vertices=np.array(verts, dtype=np.float32))
    print("sat_pairs", n, int(m.sum()))

    # ---- rotated IoU (IOU.py:91-155 as called from test.py:185-196)
    rng = np.random.default_rng(13)
    a = np.concatenate([edge_case_boxes(), car_boxes(rng, 40, x=(0, 12), y=(-1, 1), z=(-6, 6))])
    b = np.concatenate([edge_case_boxes()[::-1].copy(), car_boxes(rng, 40, x=(0, 12), y=(-1, 1), z=(-6, 6))])
    i3 = np.zeros((a.shape[0], b.shape[0]))
    i2 = np.zeros_like(i3)
    bad = np.zeros(i3.shape, np.uint8)
    for i in range(a.shape[0]):
        ta = torch.from_numpy(a[i])
        ca = ref.IOU.get_3d_box(ta[:3].numpy(), ta[3:6].numpy(), ta[6].numpy())
        for j in range(b.shape[0]):
            tb = torch.from_numpy(b[j])
            cb = ref.IOU.get_3d_box(tb[:3].numpy(), tb[3:6].numpy(), tb[6].numpy())
            try:
                i3[i, j], i2[i, j] = ref.IOU.box3d_iou(ca, cb)
            except Exception:  # Qhull refuses degenerate clip polygons; the reference would crash here
                bad[i, j] = 1
    np.savez_compressed(os.path.join(OUT, "box_iou.npz"), boxes_a=a, boxes_b=b, iou3d=i3, iou2d=i2, qhull_error=bad)
    print("box_iou", i3.shape, "overlapping pairs", int((i2 > 0).sum()), "qhull errors", int(bad.sum()))
    # known answer of IOU.py:161-168 with its float64 corners
    c1 = ref.IOU.get_3d_box((2.882992, 1.698800, 20.785644), (1.497255, 1.644981, 3.628938), -1.531692)
    c2 = ref.IOU.get_3d_box((2.756923, 1.661275, 20.943280), (1.458242, 1.604773, 3.707947), -1.549553)
    ka = ref.IOU.box3d_iou(c2, c1)
    np.savez_compressed(os.path.join(OUT, "box_iou_known.npz"), corners_pred=c2, corners_gt=c1, iou=np.array(ka))
    print("known answer", ka)

    # ---- NMS_IOU (test.py:110-140)
    bx = car_boxes(np.random.default_rng(14), 120, x=(0, 40), y=(-1, 1), z=(-15, 15))
    keep = R.nms_iou([torch.from_numpy(bx)], 0.01)[0]
    np.savez_compressed(os.path.join(OUT, "nms_iou.npz"), boxes=bx, keep=keep, thr=np.float32(0.01))
    print("nms_iou", bx.shape[0], "->", len(keep))

    # ---- get_bboxes (test.py:88-108)
    g = torch.Generator().manual_seed(15)
    cls = torch.rand(3, 4, 24, 16, generator=g)
    box = torch.randn(3, 14, 24, 16, generator=g)
    out = R.get_bboxes(cls, box, 0.8)
    np.savez_compressed(os.path.join(OUT, "get_bboxes.npz"), cls=cls.numpy(), box=box.numpy(), thr=np.float32(0.8),
                        counts=np.array([o.shape[0] for o in out]), boxes=torch.cat(out).numpy())
    print("get_bboxes", [o.shape[0] for o in out])

    # ---- dataset-side projection / filter / padding (data_import_carla.py:196-267) on synthetic returns
    cfg = dcf_b200.geometry.carla_config()
    ds = R.carla_dataset_stub(cfg)
    raw = dcf_b200.synthetic.lidar_sweep(np.random.default_rng(16), 32, 700)
    _, pc, uv, num, _ = ds.Voxelization_Projection(torch.from_numpy(raw))
    np.savez_compressed(os.path.join(OUT, "projection.npz"), raw=raw, pointcloud_raw=pc.numpy()[:num + 8],
                        projected_loc_uv=uv.numpy()[:num + 8], num_points_raw=np.int64(num),
                        crt=ds.CRT_tensor.numpy())
    print("projection", raw.shape[0], "->", num)

    # ---- voxelisation + projection (data_import_carla.py:212-267), the reference's own tensors on two sweeps.
    # `voxel[idx] += w` with repeated indices is an index_put_ without accumulation: on several threads the winner among
    # the points that share a voxel depends on torch's intra-op scheduling (8 threads here: ~0.3 % of the nonzero voxels
    # differ from run to run / from the sequential result).  The fixture pins the SEQUENTIAL semantics (last point wins).
    torch.set_num_threads(1)
    for tag, seed, beams, az in (("a", 17, 32, 700), ("b", 18, 64, 400)):
        raw = dcf_b200.synthetic.lidar_sweep(np.random.default_rng(seed), beams, az)
        vox, pc, uv, num, _ = ds.Voxelization_Projection(torch.from_numpy(raw))
        vox = vox.numpy()
        nzi = np.flatnonzero(vox).astype(np.int32)
        np.savez_compressed(os.path.join(OUT, f"voxelize_{tag}.npz"), raw=raw, vox_shape=np.array(vox.shape),
                            vox_idx=nzi, vox_val=vox.ravel()[nzi], pointcloud_raw=pc.numpy()[:num + 8],
                            projected_loc_uv=uv.numpy()[:num + 8], num_points_raw=np.int64(num), crt=ds.CRT_tensor.numpy())
        print("voxelize", tag, raw.shape[0], "->", num, "nonzero voxels", nzi.size)

    # ---- LossTotal (loss.py:33-189): target lists and per-frame values of the unmodified reference, both regress types
    for rt, seed in ((0, 19), (1, 20)):
        fx = loss_fixture(rt, seed)
        np.savez_compressed(os.path.join(OUT, f"loss_total_rt{rt}.npz"), **fx)
        print("loss_total regress_type", rt, "losses", fx["losses"], "positives", fx["npos"], "negatives", fx["nneg"])


if __name__ == "__main__":
    main()
