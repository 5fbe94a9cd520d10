#!/usr/bin/env python
"""Developer micro-benchmark: cf_fusion_fwd per scale of a bench workload, out of place and in place,
each call timed alone with CUDA events after a 256 MB L2 flush (median of --reps, and the min..max spread).
`--io bf16` times bf16 BEV maps (CF_IO_BF16), `--io both` alternates fp32 and bf16 maps call by call.
`--layout nhwc` times channels_last BEV maps (CF_IO_NHWC); `--layout both` alternates NCHW, NHWC and `nhwc-copy` call by
call, where `nhwc-copy` is what a channels_last map costs without the NHWC kernels: copy to NCHW, the NCHW call, copy back.
Not part of the bench contract."""
import argparse
import os
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import dcf_b200 as dcf  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--workload", default="cfg1")
    ap.add_argument("--mode", default=None)
    ap.add_argument("--reps", type=int, default=15)
    ap.add_argument("--groups", default="")
    ap.add_argument("--empty", action="store_true", help="no LiDAR points: every cell is a pure bev -> out copy")
    ap.add_argument("--io", choices=("fp32", "bf16", "both"), default="fp32", help="element type of the BEV maps")
    ap.add_argument("--layout", choices=("nchw", "nhwc", "both"), default="nchw", help="memory format of the BEV maps")
    a = ap.parse_args()
    wl = dcf.synthetic.make_workload(a.workload, seed=100)
    mode = a.mode or wl["workload"]["mode"]
    dev = torch.device("cuda")
    ops = dcf.ops
    to = lambda x: torch.from_numpy(np.ascontiguousarray(x)).to(dev)
    if a.empty:
        wl["num_points"][:] = 0
    points, counts, img = to(wl["points"]), to(wl["num_points"]), to(wl["img_feat"])
    grid = ops.BucketGrid(*dcf.geometry.bucket_grid(wl["config"], None))
    size = (float(wl["config"]["image_width"]), float(wl["config"]["image_height"]))
    start, srt, _ = ops.bucket_points(points, counts, grid)
    feat, _ = ops.point_gather(img, points, counts, calib=wl["calib"], img_size=size)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    fine = None
    want = set(int(g) for g in a.groups.split(",") if g)
    for sc in wl["scales"]:
        w = [to(x) for x in sc["weights"]]
        T = ops.point_mlp1(feat, points, counts, w[0], w[1], mode=mode)
        if fine is None:
            knn = ops.knn_query(start, srt, grid, sc["H"], sc["W"], sc["geom"], wl["radius"], wl["k"])
            fine, fs = knn, sc["stride"]
        else:
            knn = ops.knn_subsample(fine, sc["stride"] // fs, sc["H"], sc["W"])
        if want and sc["group"] not in want:
            continue
        pk = ops.PackedWeights()
        packed = pk.w23(w[2], w[4], mode)
        dtypes = {"fp32": [torch.float32], "bf16": [torch.bfloat16], "both": [torch.float32, torch.bfloat16]}[a.io]
        layouts = {"nchw": ["nchw"], "nhwc": ["nhwc"], "both": ["nchw", "nhwc", "nhwc-copy"]}[a.layout]
        arms = [(dt, lay) for dt in dtypes for lay in layouts]
        fmt = lambda lay: torch.contiguous_format if lay == "nchw" else torch.channels_last
        bevs = {(dt, lay): to(sc["bev"]).to(dt).contiguous(memory_format=fmt(lay)) for dt, lay in arms}
        live = float((knn[..., 0] >= 0).float().mean())
        args = (T, knn, sc["geom"], w[0], w[2], w[3], w[4], w[5])
        for name, inplace in (("out_of_place", False), ("in_place", True)):
            outs = {k: b.clone() if inplace else torch.empty_like(b) for k, b in bevs.items()}
            ts = {k: [] for k in arms}
            for _ in range(a.reps + 3):
                for k in arms:   # --io / --layout both: the arms alternate call by call
                    out = outs[k]
                    src = out if inplace else bevs[k]
                    flush.zero_()
                    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    e0.record()
                    if k[1] == "nhwc-copy":
                        x = src.contiguous()
                        y = ops.fusion_fwd(x, *args, mode=mode, packed=packed, out=x if inplace else None)[0]
                        out.copy_(y)
                    else:
                        ops.fusion_fwd(src, *args, mode=mode, packed=packed, out=out, memory_format=fmt(k[1]))
                    e1.record()
                    torch.cuda.synchronize()
                    ts[k].append(e0.elapsed_time(e1))
            for dt, lay in arms:
                t = np.array(ts[(dt, lay)][3:]) * 1e3
                es = torch.empty((), dtype=dt).element_size()
                # algorithmic BEV bytes: read bev + write out for every cell; in place, only the cells with a neighbour
                nbytes = 2 * es * bevs[(dt, lay)].numel() * (live if inplace else 1.0)
                print(f"g{sc['group']} C={sc['C']} {sc['H']}x{sc['W']} live={live:.3f} {name:12s} {str(dt)[6:]:8s} {lay:9s} "
                      f"median {np.median(t):.1f} us  spread {t.min():.1f}..{t.max():.1f} us  "
                      f"bev bytes {nbytes / 1e6:.1f} MB ({es} B/element)", flush=True)


if __name__ == "__main__":
    main()
