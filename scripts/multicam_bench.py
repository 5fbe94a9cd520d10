"""Camera-rig gather (cf_point_gather_multi*) on the GPU, at BASELINE.json configs[1] sizes: batch 4, up to 20 000 points per
frame, 128-channel stride-4 camera maps (120 x 160) of 640 x 480 images.

Reports, as JSON lines (CUDA events; the L2 is overwritten before every timed call, so maps are read from HBM):
  * gather forward, atomic backward and fixed-order backward for M = 1, 3 and 6 cameras (channels_last maps, as the
    model's camera stream emits them) on a LiDAR sweep through the range filter only;
  * the same for a 5-camera rig whose cameras differ in image and map size (cf_point_gather_rig, Waymo-like sizes);
  * the rig path at M = 1 (calib = -CRT) against cf_point_gather on the standard camera-filtered points, NCHW and
    channels_last (the outputs are checked bit for bit);
  * one fuse_scales step (bucket, gather, tables, KNN, fused layer of the five scales) with 3 cameras against the single
    camera.
Usage: python scripts/multicam_bench.py [--reps 30] [--out FILE]"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

RIGS = {1: (0.0,), 3: (-60.0, 0.0, 60.0), 6: (-150.0, -90.0, -30.0, 30.0, 90.0, 150.0)}


def gpu_label():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
        return q[0] if q else "unknown"
    except (OSError, subprocess.SubprocessError):
        return "unknown"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=30)
    ap.add_argument("--out", default=None, help="also append the JSON lines to this file")
    args = ap.parse_args()
    import torch
    import dcf_b200 as dcf
    G, ops, syn = dcf.geometry, dcf.ops, dcf.synthetic
    if not torch.cuda.is_available():
        raise SystemExit("multicam_bench.py measures on the GPU; no CUDA device found")
    torch.cuda.set_device(0)
    label = dict(gpu=torch.cuda.get_device_name(0), nvidia_smi=gpu_label())
    lines = []

    def emit(rec):
        rec = dict(rec, **label)
        lines.append(json.dumps(rec))
        print(lines[-1], flush=True)

    flush_buf = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")   # twice the L2

    def timed(fn, reps=args.reps, warm=3):
        for _ in range(warm):
            fn()
        ts = []
        for _ in range(reps):
            flush_buf.zero_()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            fn()
            b.record()
            ts.append((a, b))
        torch.cuda.synchronize()
        ms = sorted(a.elapsed_time(b) for a, b in ts)
        return dict(median_ms=round(ms[len(ms) // 2], 4), min_ms=round(ms[0], 4), max_ms=round(ms[-1], 4), reps=reps)

    wl = syn.make_workload("cfg1", seed=0)
    cfg, B, N, size = wl["config"], wl["points"].shape[0], wl["points"].shape[1], (640.0, 480.0)
    gen = torch.Generator(device="cuda").manual_seed(0)

    # points of a rig: a LiDAR sweep through the range filter only (no camera filter)
    x_lo, x_hi, y_lo, y_hi, z_lo, z_hi = G.lidar_range(cfg)
    sweep = np.zeros((B, N, 3), np.float32)
    counts = np.zeros((B,), np.int64)
    for b in range(B):
        raw = syn.lidar_sweep(np.random.default_rng(1000 + b), 32, 3000)
        keep = ((raw[:, 0] > x_lo) & (raw[:, 0] < x_hi) & (raw[:, 1] > y_lo) & (raw[:, 1] < y_hi) & (raw[:, 2] > z_lo) &
                (raw[:, 2] < z_hi))
        raw = raw[keep][:N]
        sweep[b, :len(raw)], counts[b] = raw, len(raw)
    pts, cnt = torch.from_numpy(sweep).cuda(), torch.from_numpy(counts).cuda()
    Ci, Hf, Wf = wl["img_feat"].shape[1:]
    for M, yaws in RIGS.items():
        img = torch.randn((B * M, Ci, Hf, Wf), device="cuda", generator=gen).contiguous(
            memory_format=torch.channels_last).unflatten(0, (B, M))
        rig = torch.from_numpy(G.camera_rig(yaws)).cuda().expand(B, M, 4, 3).contiguous()
        feat, ws = ops.point_gather_multi(img, pts, cnt, rig, img_size=size)
        g = torch.randn(feat.shape, device="cuda", generator=gen)
        rec = dict(what="gather_multi", cameras=M, yaws=yaws, batch=B, points=counts.tolist(), c_img=Ci, map=[Hf, Wf],
                   layout="channels_last")
        rec["fwd"] = timed(lambda: ops.point_gather_multi(img, pts, cnt, rig, img_size=size, out=feat, workspace=ws))
        rec["bwd_atomic"] = timed(lambda: ops.point_gather_multi_bwd(g, img, pts, cnt, rig, img_size=size))
        rec["bwd_deterministic"] = timed(lambda: ops.point_gather_multi_bwd(g, img, pts, cnt, rig, img_size=size,
                                                                           deterministic=True))
        emit(rec)

    # a rig whose cameras differ in size (cf_point_gather_rig): Waymo-like, three 1920x1280 front cameras and two 1920x886
    # side cameras, stride-4 maps (320 x 480 and 222 x 480), channels_last as the camera stream emits them
    het_yaws, het_sizes = (0.0, 45.0, -45.0, 90.0, -90.0), [(1920.0, 1280.0)] * 3 + [(1920.0, 886.0)] * 2
    maps = [torch.randn((B, Ci, int(h) // 4 + (int(h) % 4 > 0), int(w) // 4), device="cuda", generator=gen).contiguous(
        memory_format=torch.channels_last) for w, h in het_sizes]
    rig = torch.from_numpy(G.camera_rig(het_yaws, het_sizes)).cuda().expand(B, 5, 4, 3).contiguous()
    feat, ws = ops.point_gather_rig(maps, pts, cnt, rig, het_sizes)
    g = torch.randn(feat.shape, device="cuda", generator=gen)
    rec = dict(what="gather_rig_mixed_sizes", cameras=5, yaws=het_yaws, image_sizes=het_sizes,
               maps=[list(m.shape[2:]) for m in maps], batch=B, points=counts.tolist(), c_img=Ci, layout="channels_last")
    rec["fwd"] = timed(lambda: ops.point_gather_rig(maps, pts, cnt, rig, het_sizes, out=feat, workspace=ws))
    rec["bwd_atomic"] = timed(lambda: ops.point_gather_rig_bwd(g, maps, pts, cnt, rig, het_sizes))
    rec["bwd_deterministic"] = timed(lambda: ops.point_gather_rig_bwd(g, maps, pts, cnt, rig, het_sizes, deterministic=True))
    emit(rec)

    # M = 1 against the single-camera kernel, on the standard (camera-filtered) points
    spts, scnt = torch.from_numpy(wl["points"]).cuda(), torch.from_numpy(wl["num_points"]).cuda()
    crt = wl["calib"]
    neg = torch.from_numpy(-crt).cuda().reshape(1, 1, 4, 3).expand(B, 1, 4, 3).contiguous()
    for layout in ("nchw", "channels_last"):
        img4 = torch.from_numpy(wl["img_feat"]).cuda()
        if layout == "channels_last":
            img4 = img4.contiguous(memory_format=torch.channels_last)
        img5 = img4.unsqueeze(1)
        f1, ws1 = ops.point_gather(img4, spts, scnt, calib=crt, img_size=size)
        fm, wsm = ops.point_gather_multi(img5, spts, scnt, neg, img_size=size)
        same = bool(torch.equal(f1, fm))
        single, multi = [], []
        for _ in range(3):   # alternate the two, so drift in the shared machine hits both
            single.append(timed(lambda: ops.point_gather(img4, spts, scnt, calib=crt, img_size=size, out=f1, workspace=ws1)))
            multi.append(timed(lambda: ops.point_gather_multi(img5, spts, scnt, neg, img_size=size, out=fm, workspace=wsm)))
        s = float(np.median([r["median_ms"] for r in single]))
        m = float(np.median([r["median_ms"] for r in multi]))
        emit(dict(what="gather_m1_vs_single", layout=layout, batch=B, points=wl["num_points"].tolist(), c_img=Ci,
                  map=[Hf, Wf], bit_identical=same, single_ms=s, multi_ms=m, ratio=round(m / s, 4), single_runs=single,
                  multi_runs=multi))

    # one fuse_scales step: 3 cameras against the single camera (eager, inference)
    layers = []
    for sc in wl["scales"]:
        layer = dcf.ContinuousFusion(Ci, sc["C"], k=wl["k"], radius=wl["radius"], geom=sc["geom"], mode="fp32").cuda().eval()
        with torch.no_grad():
            for p, w in zip((layer.fc1.weight, layer.fc1.bias, layer.fc2.weight, layer.fc2.bias, layer.fc3.weight,
                             layer.fc3.bias), sc["weights"]):
                p.copy_(torch.from_numpy(w))
        layers.append(layer)
    bevs = [torch.from_numpy(sc["bev"]).cuda() for sc in wl["scales"]]
    grid = ops.BucketGrid(*G.bucket_grid(cfg))
    img1 = torch.from_numpy(wl["img_feat"]).cuda().contiguous(memory_format=torch.channels_last)
    img3 = torch.randn((B * 3, Ci, Hf, Wf), device="cuda", generator=gen).contiguous(
        memory_format=torch.channels_last).unflatten(0, (B, 3))
    rig3 = torch.from_numpy(G.camera_rig(RIGS[3])).cuda()

    def step(img, calib, points, num):
        with torch.no_grad():
            frames = dcf.FrameContext(points, num, grid)
            frames.gather(img, calib=calib, img_size=size)
            return dcf.fuse_scales(frames, layers, bevs)

    t1 = timed(lambda: step(img1, crt, spts, scnt), reps=max(10, args.reps // 2))
    t3 = timed(lambda: step(img3, rig3, pts, cnt), reps=max(10, args.reps // 2))
    emit(dict(what="fuse_scales_step", batch=B, scales=len(layers), k=wl["k"], single_camera=t1, rig_3_cameras=t3,
              note="single camera: camera-filtered points; rig: range-filtered sweep"))
    if args.out:
        with open(args.out, "a") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
