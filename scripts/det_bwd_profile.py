#!/usr/bin/env python
"""Kernel time of the fusion backward (cf_fusion_bwd + cf_point_gather_bwd, every scale) in the BASELINE.json configs[3]
train step (YAML grid 384x256, batch 4, five fusion scales, K = 3), default (atomic) path against the deterministic path,
from torch.profiler.  The two paths alternate, one profiled eager step each, `--rounds` times; prints one JSON line with the
per-step medians and the GPU's name and power limit.  `--trace-dir` also writes the Chrome traces there."""
import argparse
import json
import os
import re
import subprocess
import sys

os.environ.setdefault("CUBLAS_WORKSPACE_CONFIG", ":4096:8")   # before CUDA initialises (matmuls of the deterministic step)

import numpy as np  # noqa: E402
import torch  # noqa: E402
from torch.profiler import ProfilerActivity, profile  # noqa: E402

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import dcf_b200 as dcf  # noqa: E402
from train_step_bench import synthetic_labels  # noqa: E402

# kernels of csrc/cf_bwd.cu, cf_bwd_tc.cu and cf_bwd_det.cu (the backward of the fused layer and of the camera gather)
BWD = re.compile(r"\bk_(bwd_\w+|sgemm_nn|sgemm_tn|colsum|transpose_sq_b|point_gather_bwd|det_\w+|gdet_\w+)\b")


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                             text=True, timeout=30).stdout.strip().splitlines()
        return out[0] if out else torch.cuda.get_device_name()
    except Exception:
        return torch.cuda.get_device_name()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--trace-dir", default=None)
    a = ap.parse_args()
    dev = torch.device("cuda")
    torch.manual_seed(0)
    cfg = dcf.geometry.carla_config(fusion_scales=(1, 2, 3, 4, 5), fusion_k=3)
    model = dcf.ObjectDetection_DCF(cfg).to(dev).eval()
    opt = torch.optim.Adam(model.parameters(), lr=1e-4)
    B = 4
    wl = dcf.synthetic.make_workload(dict(dcf.synthetic.workload("yaml"), batch=B), seed=200)
    to = lambda x: torch.from_numpy(np.ascontiguousarray(x)).to(dev)
    x_lidar = torch.rand(B, 32, 384, 256, device=dev)
    x_image = torch.randint(0, 255, (B, 3, 480, 640), device=dev, dtype=torch.uint8)
    ref, num = synthetic_labels(B, 300, dev)
    crit = dcf.LossTotal(cfg, batch_reduction="sum").to(dev)
    extra = dict(pointcloud_raw=to(wl["points"]), num_points_raw=to(wl["num_points"]), projected_loc_uv=to(wl["uv"]))

    def step():
        opt.zero_grad(set_to_none=True)
        pred = model(x_lidar, x_image, **extra)
        pred_cls, pred_reg, _ = torch.split(pred, [4, 14, 14], dim=1)
        crit(ref, num, pred_cls, pred_reg).sum().backward()
        opt.step()

    res = {"default": [], "deterministic": []}
    fills = {"default": [], "deterministic": []}
    for det in (False, True):          # warm both paths
        torch.use_deterministic_algorithms(det)
        for _ in range(3):
            step()
    torch.cuda.synchronize()
    for r in range(a.rounds):
        for det in (False, True):
            torch.use_deterministic_algorithms(det)
            with profile(activities=[ProfilerActivity.CUDA]) as prof:
                step()
                torch.cuda.synchronize()
            key = "deterministic" if det else "default"
            us = sum(e.device_time_total for e in prof.key_averages() if BWD.search(e.key))
            fill = sum(e.device_time_total for e in prof.key_averages() if "fill" in e.key.lower())
            res[key].append(us / 1e3)
            fills[key].append(fill / 1e3)
            if a.trace_dir:
                os.makedirs(a.trace_dir, exist_ok=True)
                prof.export_chrome_trace(os.path.join(a.trace_dir, f"train_step_{key}_{r}.json"))
    torch.use_deterministic_algorithms(False)
    print(json.dumps({"what": "fusion backward kernels per train step (cf_fusion_bwd x5 scales + cf_point_gather_bwd), "
                      "configs[3]: YAML grid 384x256, batch 4, K=3, eager step, torch.profiler",
                      "gpu": gpu_info(),
                      "bwd_kernel_ms_default": round(float(np.median(res["default"])), 3),
                      "bwd_kernel_ms_deterministic": round(float(np.median(res["deterministic"])), 3),
                      "fill_kernel_ms_default": round(float(np.median(fills["default"])), 3),
                      "fill_kernel_ms_deterministic": round(float(np.median(fills["deterministic"])), 3),
                      "rounds": a.rounds}), flush=True)


if __name__ == "__main__":
    main()
