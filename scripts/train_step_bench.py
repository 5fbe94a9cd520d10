#!/usr/bin/env python
"""BASELINE.json configs[3]: a full train step of the drop-in ObjectDetection_DCF (LiDAR backbone + camera trunk +
continuous fusion at every residual group, forward + backward + Adam) on synthetic CARLA-shaped inputs (reference YAML
grid 384x256, batch 4 per GPU), closed with the drop-in LossTotal (loss.py of the reference with its target assignment on the
device, SURVEY 8 f-4) on synthetic ground-truth boxes in the dataset's label layout (B, 20, 8); `--mse` closes it with an MSE
on the prediction tensor instead (the loss-free step of round 1).
Single process, or `torchrun --nproc-per-node N` (one process per GPU, DDP all-reduce over NCCL).  `bench.py --workload train`
runs the same step under the bench contract; this script prints one JSON line on rank 0."""
import argparse
import json
import os
import sys
import time

import numpy as np
import torch
import torch.nn.functional as F

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import dcf_b200 as dcf  # noqa: E402


def synthetic_labels(batch, seed, dev, max_boxes=20):
    """object_data (B, 20, 8) = [x, y, z, l, w, h, yaw, flag] and num_ref (B) as the CARLA reader collates them."""
    rng = np.random.default_rng(seed)
    ref = np.zeros((batch, max_boxes, 8), np.float32)
    num = rng.integers(3, max_boxes + 1, batch)
    for b in range(batch):
        n = int(num[b])
        ref[b, :n, 0], ref[b, :n, 1], ref[b, :n, 2] = rng.uniform(2, 68, n), rng.uniform(-28, 28, n), rng.uniform(-2, -1, n)
        ref[b, :n, 3:6] = np.array([4.0, 2.0, 1.5]) * np.exp(0.1 * rng.normal(size=(n, 3)))
        ref[b, :n, 6] = rng.uniform(-np.pi, np.pi, n)
        ref[b, :n, 7] = 1
    return torch.from_numpy(ref).to(dev), torch.from_numpy(num.astype(np.int64)).to(dev)


def main(argv=None):
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, default=4)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--no-fusion", action="store_true", help="LiDAR-only model (the reference as it is) for comparison")
    ap.add_argument("--mse", action="store_true", help="close the step with an MSE instead of LossTotal")
    ap.add_argument("--graph", action="store_true", help="capture forward + backward + Adam as ONE CUDA graph and replay it "
                    "(single process only): the step time without the host's launch overhead")
    ap.add_argument("--deterministic", action="store_true", help="torch.use_deterministic_algorithms(True): bit-reproducible "
                    "gradients (the fusion layer's fixed-order backward, the trunk's matmul adjoint of the bilinear resizes)")
    ap.add_argument("--amp", action="store_true", help="forward and loss under torch.autocast('cuda', dtype=torch.bfloat16): "
                    "bf16 convolutions, bf16 BEV / camera maps through the fusion layer (fp32 weights and gradients)")
    a = ap.parse_args(argv)
    if a.deterministic:
        # before CUDA initialises: cuBLAS reads its workspace setting when the first handle is created
        os.environ.setdefault("CUBLAS_WORKSPACE_CONFIG", ":4096:8")
        torch.use_deterministic_algorithms(True)
    rank, world, local = dcf.dist_util.env_rank_world()
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    dcf.dist_util.init("nccl", dev)
    cfg = dcf.geometry.carla_config(fusion_scales=(1, 2, 3, 4, 5), fusion_k=3)
    torch.manual_seed(rank)
    model = dcf.ObjectDetection_DCF(cfg).to(dev).eval()      # BatchNorm in eval mode, as in the reference (test.py:37)
    if world > 1:
        model = torch.nn.parallel.DistributedDataParallel(model, device_ids=[local], find_unused_parameters=True)
    opt = torch.optim.Adam(model.parameters(), lr=1e-4, betas=(0.9, 0.999), capturable=a.graph)
    wl = dcf.synthetic.make_workload(dict(dcf.synthetic.workload("yaml"), batch=a.batch), seed=200 + rank)
    to = lambda x: torch.from_numpy(np.ascontiguousarray(x)).to(dev)
    x_lidar = torch.rand(a.batch, 32, 384, 256, device=dev)
    x_image = torch.randint(0, 255, (a.batch, 3, 480, 640), device=dev, dtype=torch.uint8)
    target = torch.randn(a.batch, 32, 96, 64, device=dev)
    ref_boxes, num_ref = synthetic_labels(a.batch, 300 + rank, dev)
    # every frame of the batch contributes ("sum"); the reference keeps the last frame only (loss.py:71, LossTotal's default)
    # (draws from the default CUDA generator, seeded per rank above: its Philox offset is graph-safe under capture)
    criterion = dcf.LossTotal(cfg, batch_reduction="sum").to(dev)

    def closing_loss(pred):
        if a.mse:
            return F.mse_loss(pred[:, :18], target[:, :18])
        pred_cls, pred_reg, _ = torch.split(pred, [4, 14, 14], dim=1)      # train.py:32
        return criterion(ref_boxes, num_ref, pred_cls, pred_reg).sum()
    extra = {} if a.no_fusion else dict(pointcloud_raw=to(wl["points"]), num_points_raw=to(wl["num_points"]),
                                        projected_loc_uv=to(wl["uv"]))

    # the autocast weight cache would hold casts made during a graph capture outside the graph's pool: off under --graph
    amp = lambda: torch.autocast("cuda", dtype=torch.bfloat16, enabled=a.amp, cache_enabled=not a.graph)

    def step():
        opt.zero_grad(set_to_none=True)
        with amp():
            pred = model(x_lidar, x_image, **extra)
            loss = closing_loss(pred)
        loss.backward()
        opt.step()
        return loss

    if a.graph:
        if world > 1:
            raise SystemExit("--graph is a single-process measurement")
        side = torch.cuda.Stream(dev)
        side.wait_stream(torch.cuda.current_stream(dev))
        with torch.cuda.stream(side):
            for _ in range(3):
                step()
        torch.cuda.current_stream(dev).wait_stream(side)
        torch.cuda.synchronize()
        graph = torch.cuda.CUDAGraph()
        opt.zero_grad(set_to_none=True)
        with torch.cuda.graph(graph):
            with amp():
                pred = model(x_lidar, x_image, **extra)
                static_loss = closing_loss(pred)
            static_loss.backward()
            opt.step()

        def step():  # noqa: F811  (gradients are overwritten in place by the replay, nothing to zero)
            graph.replay()
            return static_loss
    for _ in range(max(a.warmup, 3)):
        step()
    dcf.dist_util.barrier()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0 = time.perf_counter()
    e0.record()
    for _ in range(a.steps):
        loss = step()
    e1.record()
    host_ms = (time.perf_counter() - t0) * 1e3 / a.steps      # time the host needs to ENQUEUE a step (no synchronisation)
    dcf.dist_util.barrier()
    torch.cuda.synchronize()
    ms = dcf.dist_util.max_over_ranks([e0.elapsed_time(e1) / a.steps], device=dev)[0]
    res = {"what": "train step (fwd + bwd + Adam), ObjectDetection_DCF, YAML grid 384x256",
           "fusion": not a.no_fusion, "loss": "mse" if a.mse else "LossTotal (device target assignment)",
           "launch": "cuda_graph_replay" if a.graph else "eager", "deterministic": a.deterministic,
           "amp": "bf16" if a.amp else None,
           "batch_per_gpu": a.batch, "n_gpus": world, "steps": a.steps, "ms_per_step": round(ms, 3),
           "host_enqueue_ms_per_step": round(host_ms, 3),
           "frames_per_sec": round(a.batch * world / ms * 1e3, 1), "loss_value": float(loss)}
    if rank == 0 and argv is None:
        print(json.dumps(res), flush=True)
    if world > 1:
        torch.distributed.destroy_process_group()
    return res if rank == 0 else None


if __name__ == "__main__":
    main()
