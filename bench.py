#!/usr/bin/env python
"""bench.py -- fusion-layer frames/s on N B200s (BASELINE.json metric), one JSON line on rank 0.

A "step" is one pass of the continuous-fusion hot path over one batch of synthetic frames:
K-1 bucket points, K-3 project + gather camera features, then per backbone scale K-4a per-point MLP half,
K-2 KNN per BEV cell, K-4 fused MLP + K-sum-pool + BEV add.  Workload = BASELINE.json configs[1]
(batch 4, K=5, fusion after every residual group, 700x800 BEV, fp32 parity mode) per GPU; frames are
independent, so N GPUs run N disjoint batches with no collective on the data path (weak scaling).

  value  frames/s, inputs resident in HBM, CUDA-event timed, max over ranks
  e2e    same through the public nn.Module API with HOST buffers: pinned H2D of every input and D2H of every
         fused BEV map inside the timed region
  roofline      the dominant kernel against the measured HBM peak (MEASURED_PEAKS.json); roofline_per_scale: every fused
                launch against the HBM peak and, from the flops it executes, against the sustained bf16 tensor peak
  cpu_baseline  the CPU oracle (a port: the reference has no fusion layer to time) on WHOLE frames of the workload
  cfg2 / e2e_model / steady_200_replays / nms_sat.cpu_baseline / box_iou   side records (single GPU only)

`--impl reference` times that CPU port alone with all host threads (rank 0 only): one step = one whole frame.
`--dump-outputs DIR` saves the fused BEV maps of the last timed step of rank 0 as DIR/fused_g<group>.npy (float32), so that
two builds run with the same arguments (hence the same seeded inputs) can be compared output for output.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

CONFIG_OF = {"cfg0": "configs[0]", "cfg1": "configs[1]", "cfg2": "configs[2]", "yaml": "reference YAML grid"}
METRIC = "fusion_layer_frames_per_sec"
UNIT = "frames/s"


# ------------------------------------------------------------------------------------------ helpers
def algorithmic_bytes_per_frame(wl, c_img, img_hw, n_valid_mean):
    """SURVEY 8(d): sum_s [2*4*C_s*cells_s + 4*K*cells_s + weights_s] + 4*C_img*Hf*Wf + 12*n_b."""
    K = wl["k"]
    total = 4 * c_img * img_hw[0] * img_hw[1] + 12 * n_valid_mean
    for sc in wl["scales"]:
        cells = sc["H"] * sc["W"]
        C = sc["C"]
        total += 2 * 4 * C * cells + 4 * K * cells + 4 * (C * (c_img + 3) + 2 * C * C + 3 * C)
    return float(total)


def fusion_kernel_bytes(sc, B, K, live_frac=1.0):
    """Algorithmic bytes of ONE cf_fusion_fwd launch (out of place): BEV read + write of every cell, 4 B per cell for
    the liveness test, the K neighbour indices of the `live_frac` of the cells that have a neighbour, layer weights."""
    cells = sc["H"] * sc["W"]
    C = sc["C"]
    return float(B * cells * (2 * 4 * C + 4 + live_frac * 4 * K) + 4 * (2 * C * C + 4 * C))


def recorded_traffic(workload, mode, kernel):
    """DRAM bytes per launch of `kernel` from the committed ncu capture (profiles/traffic.json), or None."""
    path = os.path.join(ROOT, "profiles", "traffic.json")
    try:
        with open(path) as f:
            e = json.load(f).get(f"{workload}/{mode}/{kernel}")
        return (float(e["dram_bytes_per_launch"]), e["source"]) if e else (None, None)
    except Exception:
        return None, None


def measured_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            p = json.load(f)
        return float(p["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


def measured_tensor_peak():
    """Dense bf16 TFLOP/s a kernel inside a long step can sustain (MEASURED_PEAKS.json), else the guide's fallback."""
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            p = json.load(f)
        return float(p.get("bf16_tflops_sustained", p.get("bf16_tflops", 1390.0))), "measured (MEASURED_PEAKS.json, sustained)"
    return 1390.0, "fallback (B200_PROFILING.md)"


DUMP_BUDGET_BYTES = 60 * 2 ** 20   # all dumped arrays together, under 64 MB with the .npy headers


def dump_outputs(dirname, named, budget=DUMP_BUDGET_BYTES, seed=0):
    """Writes every (name, tensor) as dirname/<name>.npy in float32.  The budget is split evenly between the tensors; one
    with more elements than its share is saved as a 1-D sample of that many elements, taken at the sorted flat indices
    `sample_indices(numel, share, seed)`, the same positions on every run with the same shapes."""
    import torch
    os.makedirs(dirname, exist_ok=True)
    share = budget // 4 // max(1, len(named))
    for name, t in named:
        t = t.detach()
        if t.numel() > share:
            idx = torch.from_numpy(sample_indices(t.numel(), share, seed)).to(t.device)
            t = t.reshape(-1)[idx]
        np.save(os.path.join(dirname, f"{name}.npy"), t.float().cpu().numpy())


def sample_indices(numel, n, seed=0):
    """n distinct flat indices out of numel, increasing: [0, numel) is cut into n equal strata and each gives one index at
    an offset drawn from a generator seeded with `seed` (O(n) time and memory, the whole map covered evenly)."""
    edges = np.arange(n + 1, dtype=np.int64) * numel // n
    offsets = (np.random.default_rng(seed).random(n) * (edges[1:] - edges[:-1])).astype(np.int64)
    return edges[:-1] + offsets


class ClockSampler:
    """SM clock / throttle reasons sampled during the timed region: NVML polled every 2 ms from a thread
    (pynvml), or `nvidia-smi -lms` when NVML is not importable."""

    def __init__(self, index=0):
        self.index, self.samples, self.proc, self.thread = index, [], None, None
        self.stop_flag = threading.Event()
        self.nvml = None

    def start(self):
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nvml = pynvml
            self.handle = pynvml.nvmlDeviceGetHandleByIndex(self.index)
            self.max_sm = float(pynvml.nvmlDeviceGetMaxClockInfo(self.handle, pynvml.NVML_CLOCK_SM))
            self.thread = threading.Thread(target=self._poll, daemon=True)
            self.thread.start()
            return
        except Exception:
            self.nvml = None
        q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={q}",
                                          "--format=csv,noheader,nounits", "-lms", "20"], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
        except Exception:
            self.proc = None
            return
        self.thread = threading.Thread(target=self._read, daemon=True)
        self.thread.start()

    def _poll(self):
        n = self.nvml
        bits = {"hw_slowdown": n.nvmlClocksEventReasonHwSlowdown if hasattr(n, "nvmlClocksEventReasonHwSlowdown") else 0x8,
                "hw_thermal_slowdown": 0x40, "sw_thermal_slowdown": 0x20, "sw_power_cap": 0x4}
        while not self.stop_flag.is_set():
            try:
                sm = float(n.nvmlDeviceGetClockInfo(self.handle, n.NVML_CLOCK_SM))
                try:
                    r = int(n.nvmlDeviceGetCurrentClocksEventReasons(self.handle))
                except Exception:
                    r = int(n.nvmlDeviceGetCurrentClocksThrottleReasons(self.handle))
                self.samples.append((sm, self.max_sm, [k for k, b in bits.items() if r & b]))
            except Exception:
                pass
            time.sleep(0.002)

    def _read(self):
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for line in self.proc.stdout:
            parts = [p.strip() for p in line.strip().split(",")]
            if len(parts) < 6:
                continue
            try:
                self.samples.append((float(parts[0]), float(parts[1]),
                                     [n for n, v in zip(names, parts[2:6]) if v.lower().startswith("active")]))
            except ValueError:
                continue

    def mark(self):
        """Index of the next sample: samples[mark_start:mark_end] are the ones taken inside the timed region."""
        return len(self.samples)

    def stop(self, lo=0, hi=None):
        if self.nvml is None and self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["clock sampling unavailable"]}
        time.sleep(0.01)
        self.stop_flag.set()
        if self.proc is not None:
            time.sleep(0.05)
            self.proc.terminate()
            try:
                self.proc.wait(timeout=2)
            except Exception:
                self.proc.kill()
        window = self.samples[lo:hi] or self.samples
        sm = [s[0] for s in window]
        mx = [s[1] for s in window]
        reasons = set(r for s in window for r in s[2])
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm), "source": "nvml" if self.nvml is not None else "nvidia-smi"}


# ------------------------------------------------------------------------------------------ CPU port
def cpu_port_frame(O, wl, f):
    """One WHOLE frame of the workload through the CPU port (projection, per-point gather, and for every scale the
    brute-force KNN of every cell + the per-neighbour MLP, pool and BEV add); returns seconds."""
    pts, n = wl["points"][f], int(wl["num_points"][f])
    r2 = np.float32(wl["radius"]) ** 2
    t0 = time.perf_counter()
    uv = O.project_points(pts[:n], wl["calib"])
    feat = O.gather_points(wl["img_feat"][f], uv)
    for sc in wl["scales"]:
        x0, y0, dx, dy = sc["geom"]
        knn = O.knn_bruteforce(pts, n, sc["H"], sc["W"], x0, y0, dx, dy, r2, wl["k"])
        O.fusion_mlp(sc["bev"][f], feat, pts, knn, sc["geom"], sc["weights"])
    return time.perf_counter() - t0


def cpu_port_frames(wl, max_frames, budget_s, warm_frames=0, threads=None):
    """Runs whole frames of the workload (cycling through its batch) until `max_frames` are done or `budget_s` seconds of
    timed CPU work have passed (at least one frame); returns (seconds per frame list, threads)."""
    from oracle import oracle as O
    O.build()
    threads = O.set_threads(threads or os.cpu_count())   # torchrun exports OMP_NUM_THREADS=1: ask for every host core
    B = wl["points"].shape[0]
    for i in range(warm_frames):
        cpu_port_frame(O, wl, i % B)
    ts = []
    while len(ts) < max_frames and (not ts or sum(ts) + ts[-1] <= budget_s):
        ts.append(cpu_port_frame(O, wl, (warm_frames + len(ts)) % B))
    return ts, threads


def cpu_postprocess_baselines(dcf, B):
    """The CPU port of the rotated-box post-process on the bench's boxes (1 core: the reference's Test.NMS_SAT and box3d_iou
    are single-threaded Python; the port is single-threaded C): ms per 2 000-box frame of NMS_SAT, box3d_iou pairs/s."""
    from oracle import oracle as O
    O.build()
    boxes = dcf.synthetic.nms_boxes(500, 2000)
    O.nms_sat(boxes[:200])
    t0 = time.perf_counter()
    reps = 0
    while reps < 3 or time.perf_counter() - t0 < 1.0:
        keep = O.nms_sat(boxes)
        reps += 1
    t_nms = (time.perf_counter() - t0) / reps
    a, b = boxes[:300], boxes[300:600]
    O.box3d_iou_matrix(a[:20], b[:20])
    t0 = time.perf_counter()
    O.box3d_iou_matrix(a, b)
    t_iou = time.perf_counter() - t0
    return {"nms_sat_ms_per_frame": round(t_nms * 1e3, 3), "nms_sat_kept": int(len(keep)), "box3d_iou_pairs_per_sec": round(len(a) * len(b) / t_iou, 1),
            "cores": 1, "kind": "port"}


# ------------------------------------------------------------------------------------------ GPU arm
class GpuPipeline:
    """Device-resident buffers + the op sequence of one step (through the package's public ops / modules)."""

    def __init__(self, dcf, wl, mode, device, bucket_size=None):
        import torch
        self.torch, self.dcf, self.wl, self.mode = torch, dcf, wl, mode
        self.device = device
        self.grid = dcf.ops.BucketGrid(*dcf.geometry.bucket_grid(wl["config"], bucket_size))
        dev = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(device)
        self.points, self.counts = dev(wl["points"]), dev(wl["num_points"])
        self.img = dev(wl["img_feat"])
        self.calib = wl["calib"]
        self.layers, self.bev, self.out = [], [], []
        c_img = self.img.shape[1]
        for sc in wl["scales"]:
            layer = dcf.ContinuousFusion(c_img, sc["C"], k=wl["k"], radius=wl["radius"], geom=sc["geom"], mode=mode).to(device)
            with torch.no_grad():
                for p, w in zip((layer.fc1.weight, layer.fc1.bias, layer.fc2.weight, layer.fc2.bias, layer.fc3.weight,
                                 layer.fc3.bias), sc["weights"]):
                    p.copy_(dev(w))
            self.layers.append(layer.eval())
            self.bev.append(dev(sc["bev"]))
        self.size = (float(wl["config"]["image_width"]), float(wl["config"]["image_height"]))
        self.live_frac, self.valid_rows = {}, {}

    def step(self, bev=None, points=None, counts=None, img=None, inplace=False):
        torch = self.torch
        bev = self.bev if bev is None else bev
        with torch.no_grad():
            frames = self.dcf.FrameContext(self.points if points is None else points,
                                           self.counts if counts is None else counts, self.grid)
            frames.gather(self.img if img is None else img, calib=self.calib, img_size=self.size)
            return self.dcf.fuse_scales(frames, self.layers, bev, inplace=inplace)

    def timed_ops(self):
        """One step with a CUDA-event pair around every C-ABI call -> {op name: ms}, per-launch list."""
        torch, ops = self.torch, self.dcf.ops
        ev = []

        def timed(name, fn):
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            r = fn()
            b.record()
            ev.append((name, a, b))
            return r

        with torch.no_grad():
            start, srt, _ = timed("cf_bucket_points", lambda: ops.bucket_points(self.points, self.counts, self.grid))
            feat, _ = timed("cf_point_gather", lambda: ops.point_gather(self.img, self.points, self.counts, calib=self.calib,
                                                                        img_size=self.size))
            fine, fine_stride = None, 1
            packed1 = [l._packed.w1(l.fc1.weight, self.mode) for l in self.layers]
            Ts = timed("cf_point_mlp1_multi", lambda: ops.point_mlp1_multi(feat, self.points, self.counts,
                                                                           [l.fc1.weight for l in self.layers],
                                                                           [l.fc1.bias for l in self.layers], packed1,
                                                                           mode=self.mode))
            for sc, layer, bev, T in zip(self.wl["scales"], self.layers, self.bev, Ts):
                g = sc["group"]
                if fine is None:
                    knn = timed(f"cf_knn_query[g{g}]", lambda: ops.knn_query(start, srt, self.grid, sc["H"], sc["W"],
                                                                             sc["geom"], self.wl["radius"], self.wl["k"]))
                    fine, fine_stride = knn, sc["stride"]
                else:   # nested scales: strided copy of the finest table (what FrameContext.knn does)
                    knn = timed(f"cf_knn_subsample[g{g}]", lambda: ops.knn_subsample(fine, sc["stride"] // fine_stride,
                                                                                     sc["H"], sc["W"]))
                timed(f"cf_fusion_fwd[g{g}]", lambda: ops.fusion_fwd(bev, T, knn, sc["geom"], layer.fc1.weight,
                                                                     layer.fc2.weight, layer.fc2.bias, layer.fc3.weight,
                                                                     layer.fc3.bias, mode=self.mode,
                                                                     packed=layer._packed.w23(layer.fc2.weight, layer.fc3.weight, self.mode)))
                self.live_frac[g] = float((knn[..., 0] >= 0).float().mean())
                self.valid_rows[g] = float((knn >= 0).sum())
        torch.cuda.synchronize()
        return [(n, a.elapsed_time(b)) for n, a, b in ev]


def run_gpu(args):
    import torch
    import dcf_b200 as dcf
    rank, world, local = dcf.dist_util.env_rank_world()
    if not torch.cuda.is_available():
        raise RuntimeError("bench.py needs a CUDA device: the product path has no CPU fallback")
    torch.cuda.set_device(local)
    device = torch.device("cuda", local)
    import torch.distributed as dist
    dcf.dist_util.init("nccl", device)
    # N ranks share one host: give every rank its own slice of the cores, so that its launch thread and its pinned-buffer
    # traffic do not migrate between the ranks' cores (the end-to-end arm is bound by the host side at N > 1)
    affinity = None
    if world > 1 and hasattr(os, "sched_setaffinity"):
        try:
            cores = sorted(os.sched_getaffinity(0))
            per = max(1, len(cores) // world)
            mine = cores[local * per:(local + 1) * per] or cores
            os.sched_setaffinity(0, mine)
            affinity = [mine[0], mine[-1]]
        except OSError:
            affinity = None

    def barrier():
        dcf.dist_util.barrier()
        torch.cuda.synchronize()

    wl = dcf.synthetic.make_workload(args.workload, seed=dcf.dist_util.rank_seed(100, rank))   # disjoint frames per rank
    B = wl["points"].shape[0]
    mode = args.mode or wl["workload"]["mode"]
    pipe = GpuPipeline(dcf, wl, mode, device, args.bucket_size)
    lib = dcf.load()

    # ---- device-resident throughput -------------------------------------------------------------------
    # The step is ~25 short launches on several streams; its host-side launch cost would otherwise be on the critical
    # path, so after eager warm-up it is captured once into a CUDA graph and the timed region replays the graph.
    for _ in range(max(args.warmup, 3)):
        pipe.step()
    torch.cuda.synchronize()
    launches0 = lib.cf_launch_count()
    pipe.step()
    launches_per_step = lib.cf_launch_count() - launches0
    graph = None
    if not args.no_graph:
        torch.cuda.synchronize()
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph):
            graph_outs = pipe.step()      # every replay rewrites these tensors
        for _ in range(3):
            graph.replay()
    run_step = graph.replay if graph is not None else pipe.step
    barrier()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    c_lo = sampler.mark()
    e0.record()
    for _ in range(args.steps):
        last_outs = run_step()
    e1.record()
    barrier()
    c_hi = sampler.mark()
    ms = e0.elapsed_time(e1)
    if args.dump_outputs and rank == 0:
        last_outs = graph_outs if graph is not None else last_outs
        dump_outputs(args.dump_outputs, [(f"fused_g{sc['group']}", o) for sc, o in zip(wl["scales"], last_outs)])
    launches = launches_per_step * args.steps
    clocks = sampler.stop(c_lo, c_hi) if rank == 0 else None
    # the same step over a longer region (the contract's K steps are ~20 ms: one hiccup would move them)
    n_steady = 200
    g0, g1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    g0.record()
    for _ in range(n_steady):
        run_step()
    g1.record()
    barrier()
    ms_steady = g0.elapsed_time(g1)

    # ---- the same step writing into its input maps (cf_fusion_fwd with d_out == d_bev) -----------------
    # How the drop-in model (inference) and the end-to-end runner below call the layer: cells without a LiDAR point in
    # reach then cost no memory traffic.  The headline `value` above stays out of place (the reference allocates a new map,
    # model.py:74-78).  Every replay adds the fused term to the same maps again; the kernels' work does not depend on the
    # map values, and 3 + K additions of O(1) terms stay far from overflow.
    ms_inplace = None
    if graph is not None:
        bev_io = [b.clone() for b in pipe.bev]
        for _ in range(2):
            pipe.step(bev=bev_io, inplace=True)
        torch.cuda.synchronize()
        graph_ip = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph_ip):
            pipe.step(bev=bev_io, inplace=True)
        graph_ip.replay()
        i0, i1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        i0.record()
        for _ in range(args.steps):
            graph_ip.replay()
        i1.record()
        barrier()
        ms_inplace = i0.elapsed_time(i1)
        del graph_ip, bev_io

    # ---- end to end: host buffers in, host buffers out ------------------------------------------------
    pin = lambda a: torch.from_numpy(np.ascontiguousarray(a)).pin_memory()
    h_points, h_counts, h_img = pin(wl["points"]), pin(wl["num_points"]), pin(wl["img_feat"])
    h_bev = [pin(sc["bev"]) for sc in wl["scales"]]
    h_out = [torch.empty_like(b).pin_memory() for b in h_bev]
    h2d = sum(t.numel() * t.element_size() for t in [h_points, h_counts, h_img] + h_bev)
    d2h = sum(t.numel() * t.element_size() for t in h_out)

    # Public API for this arm: dcf.FusionRunner = the fixed-shape pipeline (bucket, gather, tables, KNN, fused layer of every
    # scale, in place) captured once as a CUDA graph on static device buffers.  Frames are independent, so they stream
    # through two single-frame runners: frame f+1 uploads (pinned host -> the runner's input buffers) while frame f
    # computes and frame f-1 downloads; PCIe is full duplex and the three streams keep both directions busy.
    s_in, s_out = torch.cuda.Stream(device), torch.cuda.Stream(device)
    s_main = torch.cuda.current_stream(device)
    bev_shapes = [tuple(b.shape[1:]) for b in pipe.bev]
    runners = [dcf.FusionRunner(pipe.layers, pipe.grid, 1, h_points.shape[1], tuple(h_img.shape[1:]), bev_shapes,
                                calib=pipe.calib, img_size=pipe.size, inplace=True, device=device) for _ in range(2)]
    free_ev = [None, None]     # the runner's buffers may be overwritten once its previous download has finished

    def e2e_step():
        for f in range(B):
            r = runners[f % 2]
            if free_ev[f % 2] is not None:
                s_in.wait_event(free_ev[f % 2])
            with torch.cuda.stream(s_in):
                r.points.copy_(h_points[f:f + 1], non_blocking=True)
                r.num_points.copy_(h_counts[f:f + 1], non_blocking=True)
                r.img_feat.copy_(h_img[f:f + 1], non_blocking=True)
                for d, hb in zip(r.bevs, h_bev):
                    d.copy_(hb[f:f + 1], non_blocking=True)
                up = torch.cuda.Event()
                up.record(s_in)
            s_main.wait_event(up)
            outs = r()                                   # one graph replay on the current stream
            done = torch.cuda.Event()
            done.record(s_main)
            s_out.wait_event(done)
            with torch.cuda.stream(s_out):
                for o, h in zip(outs, h_out):
                    h[f:f + 1].copy_(o, non_blocking=True)
                fe = torch.cuda.Event()
                fe.record(s_out)
            free_ev[f % 2] = fe
        s_main.wait_stream(s_out)

    e2e_steps = max(2, min(args.steps, 10))
    for _ in range(3):
        e2e_step()
    barrier()
    f0, f1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    f0.record()
    for _ in range(e2e_steps):
        e2e_step()
    f1.record()
    barrier()
    ms_e2e = f0.elapsed_time(f1)
    # the two PCIe directions on their own (same pinned buffers, same per-frame copies): what one rank's link gives when the
    # other direction is idle; with N ranks on one host the ratio to the N = 1 figure is the host-side ceiling
    def copy_rate(direction):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        reps = 3
        torch.cuda.synchronize()
        a.record()
        for _ in range(reps):
            for f in range(B):
                r = runners[f % 2]
                if direction == "h2d":
                    r.points.copy_(h_points[f:f + 1], non_blocking=True)
                    r.img_feat.copy_(h_img[f:f + 1], non_blocking=True)
                    for d, hb in zip(r.bevs, h_bev):
                        d.copy_(hb[f:f + 1], non_blocking=True)
                else:
                    for o, h in zip(r.bevs, h_out):
                        h[f:f + 1].copy_(o, non_blocking=True)
        b.record()
        torch.cuda.synchronize()
        return (h2d if direction == "h2d" else d2h) * reps / (a.elapsed_time(b) * 1e-3) / 1e9
    barrier()
    h2d_gbs = copy_rate("h2d")
    barrier()
    d2h_gbs = copy_rate("d2h")
    barrier()

    # ---- max over ranks ---------------------------------------------------------------------------------
    ms, ms_e2e, ms_steady, inv_h2d, inv_d2h, ms_inplace = dcf.dist_util.max_over_ranks(
        [ms, ms_e2e, ms_steady, 1.0 / h2d_gbs, 1.0 / d2h_gbs, ms_inplace if ms_inplace is not None else -1.0], device=device)
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    # ---- per-kernel times + roofline of the dominant kernel (rank 0) -------------------------------------
    reps = 7
    acc = {}
    pipe.timed_ops()   # untimed: the graph capture emptied the allocator cache, the first pass re-populates it
    for _ in range(reps):
        for name, t_ms in pipe.timed_ops():
            acc.setdefault(name, []).append(t_ms)
    per_op = {k: float(np.median(v)) for k, v in acc.items()}
    step_ms = ms / args.steps
    dom = max((k for k in per_op if k.startswith("cf_")), key=per_op.get)
    peak, peak_src = measured_peaks()
    K = wl["k"]
    roof = None
    if dom.startswith("cf_fusion_fwd"):
        g = int(dom.split("[g")[1].rstrip("]"))
        sc = [s for s in wl["scales"] if s["group"] == g][0]
        nbytes = fusion_kernel_bytes(sc, B, K, pipe.live_frac[g])
        ach = nbytes / (per_op[dom] * 1e-3) / 1e9
        traffic, traffic_src = recorded_traffic(args.workload, mode, dom)
        roof = {"bound": "hbm", "kernel": dom, "achieved": round(ach, 1), "peak": peak, "unit": "GB/s",
                "frac": round(ach / peak, 4), "traffic": traffic, "traffic_source": traffic_src, "peak_source": peak_src,
                "bytes_per_launch": nbytes, "ms_per_launch": round(per_op[dom], 4),
                "share_of_step": round(per_op[dom] / sum(per_op.values()), 3),
                "cells_with_neighbour": round(pipe.live_frac[g], 4)}
    else:
        roof = {"bound": "hbm", "kernel": dom, "achieved": None, "peak": peak, "unit": "GB/s", "frac": None,
                "traffic": None, "peak_source": peak_src, "ms_per_launch": round(per_op[dom], 4),
                "share_of_step": round(per_op[dom] / sum(per_op.values()), 3),
                "note": "dominant kernel is compute/latency bound; see DESIGN.md"}
    # ---- every fused launch against both roofs -------------------------------------------------------------------------
    # HBM: the launch's algorithmic bytes.  Tensor: the flops the launch EXECUTES (layer 2 on every (cell, k) row that holds a
    # neighbour, layer 3 on every cell that has one; x3 MMA passes in fp32 mode, SURVEY 7.5) against the sustained bf16 peak.
    tpeak, tpeak_src = measured_tensor_peak()
    passes = 3 if mode == "fp32" else 1
    per_scale = []
    for sc in wl["scales"]:
        g = sc["group"]
        name = f"cf_fusion_fwd[g{g}]"
        if name not in per_op:
            continue
        C, cells = sc["C"], sc["H"] * sc["W"]
        rows, live = pipe.valid_rows[g], pipe.live_frac[g] * B * cells
        flops = passes * (2.0 * rows * C * C + 2.0 * live * C * C)
        t = per_op[name] * 1e-3
        nb = fusion_kernel_bytes(sc, B, K, pipe.live_frac[g])
        per_scale.append({"kernel": name, "C": C, "cells": cells, "ms": round(per_op[name], 4),
                          "hbm_gbs": round(nb / t / 1e9, 1), "hbm_frac": round(nb / t / 1e9 / peak, 4),
                          "tensor_tflops_executed": round(flops / t / 1e12, 2), "tensor_frac": round(flops / t / 1e12 / tpeak, 4),
                          "mma_passes": passes})
    # ---- rotated-box post-process beside it: Test.NMS_SAT semantics on 2 000 boxes per frame (SURVEY 8d) ----------------
    nms = None
    try:
        boxes_h = np.stack([dcf.synthetic.nms_boxes(500 + f, 2000) for f in range(B)])
        boxes_d = torch.zeros((B, 2048, 7), device=device)
        boxes_d[:, :2000] = torch.from_numpy(boxes_h).to(device)
        counts_d = torch.full((B,), 2000, dtype=torch.int32, device=device)
        for _ in range(3):
            keep, kcnt = dcf.ops.nms_sat(boxes_d, counts_d)
        n0, n1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        n0.record()
        for _ in range(10):
            keep, kcnt = dcf.ops.nms_sat(boxes_d, counts_d)
        n1.record()
        torch.cuda.synchronize()
        nms_ms = n0.elapsed_time(n1) / 10
        nms = {"boxes_per_frame": 2000, "frames": B, "ms_per_call": round(nms_ms, 4),
               "frames_per_sec": round(B / (nms_ms * 1e-3), 1), "kept_per_frame": [int(x) for x in kcnt.tolist()]}
        # rotated IoU (Test.box3d_iou of every pred x GT pair, SURVEY P-8): 2 000 x 64 pairs per call
        ba, bb = boxes_d[0, :2000].contiguous(), boxes_d[1, :64].contiguous()
        for _ in range(3):
            dcf.ops.box_iou(ba, bb)
        n0.record()
        for _ in range(10):
            dcf.ops.box_iou(ba, bb)
        n1.record()
        torch.cuda.synchronize()
        box_iou = {"pairs_per_call": 2000 * 64, "ms_per_call": round(n0.elapsed_time(n1) / 10, 4),
                   "pairs_per_sec": round(2000 * 64 / (n0.elapsed_time(n1) / 10 * 1e-3), 1)}
        if world == 1 and not args.no_cpu_baseline:
            cb = cpu_postprocess_baselines(dcf, B)
            nms["cpu_baseline"] = {"value": round(1e3 / cb["nms_sat_ms_per_frame"], 3), "unit": "frames/s", "ms_per_frame": cb["nms_sat_ms_per_frame"],
                                   "kept": cb["nms_sat_kept"], "cores": 1, "kind": "port",
                                   "note": "the reference's own Test.NMS_SAT (pure Python, test.py:142-175) took 5.15 s on such a frame (SURVEY 8a P-4)"}
            box_iou["cpu_baseline"] = {"value": cb["box3d_iou_pairs_per_sec"], "unit": "pairs/s", "cores": 1, "kind": "port"}
    except Exception as e:  # never let the side measurement break the bench line
        nms = {"error": str(e)[:200]}
        box_iou = None
    n_valid = float(np.mean(wl["num_points"]))
    layer_bytes = algorithmic_bytes_per_frame(wl, wl["img_feat"].shape[1], wl["img_feat"].shape[2:], n_valid)
    layer_gbs = layer_bytes * B / (step_ms * 1e-3) / 1e9

    # ---- CPU port beside it: whole frames, about args.cpu_budget seconds of CPU work ------------------------
    cpu = None
    if world == 1 and not args.no_cpu_baseline:
        ts, nthr = cpu_port_frames(wl, max_frames=64, budget_s=args.cpu_budget, warm_frames=0)
        cpu = {"value": round(len(ts) / sum(ts), 6), "unit": UNIT, "cores": nthr, "kind": "port",
               "sample": f"{len(ts)} whole frame(s) of the workload, every cell of every scale, nothing extrapolated ({sum(ts):.1f} s of CPU work)"}
    # ---- side records (single GPU): BASELINE configs[2], the drop-in model end to end -----------------------
    cfg2 = e2e_model = None
    if world == 1 and not args.no_extras and args.workload == "cfg1":
        try:
            cfg2 = side_workload(dcf, "cfg2", device, peak)
        except Exception as e:
            cfg2 = {"error": str(e)[:200]}
        try:
            e2e_model = model_e2e(dcf, device)
        except Exception as e:
            e2e_model = {"error": str(e)[:200]}

    line = {
        "metric": METRIC, "value": round(dcf.dist_util.aggregate_rate(B, world, args.steps, ms), 2), "unit": UNIT, "n_gpus": world,
        "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": round(step_ms, 4), "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32" if mode in ("fp32", "simt") else "bf16",
        "data": "synthetic",
        "config": {"workload": workload_label(args.workload, wl)},
        "run": {"mlp_mode": mode, "frames_per_step_per_gpu": B, "launch": "eager" if graph is None else "cuda_graph_replay",
                "l2_policy": f"inputs_exceed_l2 (BEV in+out {2 * sum(b.numel() * 4 for b in pipe.bev) / 1e6:.0f} MB per step vs 126 MB L2)"},
        "in_place": None if ms_inplace < 0 else {
            "ms_per_step": round(ms_inplace / args.steps, 4), "value": round(dcf.dist_util.aggregate_rate(B, world, args.steps, ms_inplace), 2),
            "unit": UNIT, "note": "same step, same protocol, the fused layer writing into its input maps (d_out == d_bev), as the "
                                  "drop-in model at inference and the e2e runner call it"},
        "steady_200_replays": {"replays": n_steady, "ms_per_step": round(ms_steady / n_steady, 4),
                               "value": round(dcf.dist_util.aggregate_rate(B, world, n_steady, ms_steady), 2), "unit": UNIT},
        "e2e": {"value": round(dcf.dist_util.aggregate_rate(B, world, e2e_steps, ms_e2e), 2), "unit": UNIT, "h2d_bytes_per_step": h2d,
                "d2h_bytes_per_step": d2h, "steps": e2e_steps, "ms_per_step": round(ms_e2e / e2e_steps, 3),
                "per_rank_gbs": {"h2d_alone_min_over_ranks": round(1.0 / inv_h2d, 1), "d2h_alone_min_over_ranks": round(1.0 / inv_d2h, 1),
                                 "both_directions_in_e2e": round((h2d + d2h) / (ms_e2e / e2e_steps * 1e-3) / 1e9, 1)},
                "host_affinity_cores_rank0": affinity},
        "gpu_launches": int(launches),
        "roofline": roof,
        "roofline_per_scale": {"tensor_peak_tflops": tpeak, "tensor_peak_source": tpeak_src, "hbm_peak_gbs": peak, "launches": per_scale},
        "layer": {"algorithmic_bytes_per_frame": layer_bytes, "achieved_gbs": round(layer_gbs, 1),
                  "frac_of_hbm_peak": round(layer_gbs / peak, 4)},
        "kernel_ms": {k: round(v, 4) for k, v in per_op.items()},
        "nms_sat": nms,
        "box_iou": box_iou,
        "cfg2": cfg2,
        "e2e_model": e2e_model,
        "cpu_baseline": cpu,
        "clocks": clocks,
    }
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def side_workload(dcf, name, device, peak, replays=60):
    """A second workload through the same device-resident pipeline (CUDA-graph replay, CUDA events): BASELINE configs[2]
    = batch 8, ~119 k points/frame, K = 10, bf16 MLP on tcgen05 -- the largest single-GPU configuration."""
    import torch
    wl = dcf.synthetic.make_workload(name, seed=100)
    mode = wl["workload"]["mode"]
    B = wl["points"].shape[0]
    pipe = GpuPipeline(dcf, wl, mode, device)
    for _ in range(3):
        pipe.step()
    torch.cuda.synchronize()
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        pipe.step()
    for _ in range(3):
        graph.replay()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    a.record()
    for _ in range(replays):
        graph.replay()
    b.record()
    torch.cuda.synchronize()
    ms = a.elapsed_time(b) / replays
    acc = {}
    pipe.timed_ops()
    for _ in range(3):
        for n, t in pipe.timed_ops():
            acc.setdefault(n, []).append(t)
    per_op = {k: round(float(np.median(v)), 4) for k, v in acc.items()}
    n_valid = float(np.mean(wl["num_points"]))
    layer_bytes = algorithmic_bytes_per_frame(wl, wl["img_feat"].shape[1], wl["img_feat"].shape[2:], n_valid)
    out = {"workload": workload_label(name, wl), "mlp_mode": mode, "value": round(B / (ms * 1e-3), 2), "unit": UNIT, "ms_per_step": round(ms, 4),
           "replays": replays, "layer_frac_of_hbm_peak": round(layer_bytes * B / (ms * 1e-3) / 1e9 / peak, 4), "kernel_ms": per_op}
    del graph, pipe
    torch.cuda.empty_cache()
    if mode == "bf16":
        # the same workload with the layer-1 tables stored as bf16 too (CF_MODE_BF16_TABLES, inference only; same 1e-2 tolerance,
        # tests/test_gpu_fullsize.py): half the table bytes written by K-4a and gathered by K-4
        pipe = GpuPipeline(dcf, wl, "bf16t", device)
        for _ in range(3):
            pipe.step()
        torch.cuda.synchronize()
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph):
            pipe.step()
        for _ in range(3):
            graph.replay()
        torch.cuda.synchronize()
        a.record()
        for _ in range(replays):
            graph.replay()
        b.record()
        torch.cuda.synchronize()
        ms_t = a.elapsed_time(b) / replays
        out["bf16_tables"] = {"mlp_mode": "bf16t", "value": round(B / (ms_t * 1e-3), 2), "unit": UNIT, "ms_per_step": round(ms_t, 4), "replays": replays}
        del graph, pipe
        torch.cuda.empty_cache()
    return out


def model_e2e(dcf, device, batch=4, steps=10):
    """The drop-in model end to end through its public API (the reference's call, test.py:78-79): ObjectDetection_DCF(config)
    on the reference YAML grid, inputs in pinned HOST memory (voxel grid, uint8 camera image, raw points, counts, uv), the
    prediction tensor read back to the host, inside the timed region; the LiDAR-only model (the reference as it is) beside it."""
    import torch
    cfg = dcf.geometry.carla_config(fusion_scales=(1, 2, 3, 4, 5), fusion_k=3)
    torch.manual_seed(0)
    wl = dcf.synthetic.make_workload(dict(dcf.synthetic.workload("yaml"), batch=batch), seed=300)
    pin = lambda t: t.pin_memory()
    h = {"x_lidar": pin(torch.rand(batch, 32, 384, 256)), "x_image": pin(torch.randint(0, 255, (batch, 3, 480, 640), dtype=torch.uint8)),
         "pointcloud_raw": pin(torch.from_numpy(np.ascontiguousarray(wl["points"]))),
         "num_points_raw": pin(torch.from_numpy(np.ascontiguousarray(wl["num_points"]))),
         "projected_loc_uv": pin(torch.from_numpy(np.ascontiguousarray(wl["uv"])))}
    out = {"model": "ObjectDetection_DCF, reference YAML grid 384x256, fusion at all five groups, K=3", "frames_per_step": batch}
    for tag, keys in (("fused", list(h)), ("lidar_only", ["x_lidar", "x_image"])):
        model = dcf.ObjectDetection_DCF(cfg).to(device).eval()
        h_pred = torch.empty(batch, 32, 96, 64).pin_memory()

        def step():
            d = {k: h[k].to(device, non_blocking=True) for k in keys}
            with torch.no_grad():
                pred = model(d["x_lidar"], d["x_image"], **{k: d[k] for k in keys[2:]})
            h_pred.copy_(pred, non_blocking=True)

        for _ in range(3):
            step()
        torch.cuda.synchronize()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(steps):
            step()
        b.record()
        torch.cuda.synchronize()
        ms = a.elapsed_time(b) / steps
        out[tag] = {"value": round(batch / (ms * 1e-3), 2), "unit": "frames/s", "ms_per_step": round(ms, 3),
                    "h2d_bytes_per_step": int(sum(h[k].numel() * h[k].element_size() for k in keys)),
                    "d2h_bytes_per_step": int(h_pred.numel() * 4)}
        del model
    torch.cuda.empty_cache()
    return out


def workload_label(name, wl):
    """One string for both arms: the workload's key, the BASELINE.json entry it stands for, and its sizes."""
    ci, hf, wf = wl["img_feat"].shape[1:]
    return (f"{name}: BASELINE.json {CONFIG_OF.get(name, 'custom')} (batch {wl['points'].shape[0]}/GPU, K={wl['k']}, "
            f"{len(wl['scales'])} scales of a {wl['workload']['bev'][0]}x{wl['workload']['bev'][1]} BEV, "
            f"~{int(float(np.mean(wl['num_points'])))} LiDAR points/frame, {ci}x{hf}x{wf} camera map)")


# ------------------------------------------------------------------------------------------ reference arm
def run_reference(args):
    """The CPU implementation of the same path on the host cores (rank 0 only).  The upstream repository has no
    fusion layer (model.py:199-203 is a TODO), so the arm is the oracle PORT, all host threads."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import dcf_b200 as dcf
    wl = dcf.synthetic.make_workload(args.workload, seed=100)
    B = wl["points"].shape[0]
    # One step of this arm = ONE whole frame (every cell of every scale, nothing sampled or extrapolated); frames cycle through
    # the workload's batch.  `steps` in the line = the frames actually timed: all of --steps unless they would not fit in
    # ~150 s of CPU work, which the line then says.
    warm = min(max(args.warmup, 0), 3)
    ts, nthr = cpu_port_frames(wl, max_frames=max(1, args.steps), budget_s=150.0, warm_frames=warm)
    v = len(ts) / sum(ts)
    desc = (f"{len(ts)} whole frame(s) of the workload after {warm} warm-up frame(s), every cell of every scale, nothing extrapolated "
            f"({sum(ts):.1f} s of CPU work); one step = one frame")
    line = {"impl": "reference", "metric": METRIC, "value": round(v, 6), "unit": UNIT,
            "n_gpus": int(os.environ.get("WORLD_SIZE", "1")), "steps": len(ts), "steps_requested": max(1, args.steps), "warmup": warm,
            "ms_per_step": round(1e3 * sum(ts) / len(ts), 1), "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic",
            "config": {"workload": workload_label(args.workload, wl)},
            "run": {"frames_per_step": 1, "threads": nthr},
            "cpu_baseline": {"value": round(v, 6), "unit": UNIT, "cores": nthr, "kind": "port", "sample": desc},
            "e2e": {"value": round(v, 6), "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)


def run_train(args):
    """BASELINE.json configs[3] under the bench contract: the full train step of the drop-in model (LiDAR backbone + camera
    trunk + continuous fusion at every residual group + LossTotal with device-side target assignment, forward + backward +
    Adam), batch-partitioned over the ranks with DDP's gradient all-reduce over NCCL (the path's only collective).
    `--impl reference`: the reference has no fusion layer and its train.py needs a private dataset, so there is nothing to run."""
    if args.impl == "reference":
        if int(os.environ.get("RANK", "0")) == 0:
            print(json.dumps({"impl": "reference", "unavailable": "train.py of the reference needs its private CARLA dataset and has no fusion layer"}), flush=True)
        return
    sys.path.insert(0, os.path.join(ROOT, "scripts"))
    import train_step_bench
    argv = ["--steps", str(args.steps), "--warmup", str(max(args.warmup, 3))]
    if not args.no_graph and int(os.environ.get("WORLD_SIZE", "1")) == 1:
        argv.append("--graph")
    res = train_step_bench.main(argv)
    if res is None:
        return
    line = {"metric": "train_step_frames_per_sec", "value": res["frames_per_sec"], "unit": UNIT, "n_gpus": res["n_gpus"],
            "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": res["ms_per_step"], "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": "train: BASELINE.json configs[3] (ObjectDetection_DCF on the reference YAML grid 384x256, batch 4/GPU, "
                                   "fusion at all five groups K=3, LossTotal, Adam; DDP all-reduce over NCCL for N > 1)"},
            "run": {k: res[k] for k in ("launch", "loss", "host_enqueue_ms_per_step", "loss_value")}}
    print(json.dumps(line), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="cfg1")
    ap.add_argument("--mode", default=None, help="fp32 | bf16 | bf16t (bf16 with bf16 tables) | simt (default: the workload's)")
    ap.add_argument("--cpu-budget", type=float, default=15.0, help="seconds of CPU work for the cpu_baseline sample")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="skip the side records (cfg2 sub-record, model end to end)")
    ap.add_argument("--no-graph", action="store_true", help="time eager launches instead of a CUDA-graph replay")
    ap.add_argument("--bucket-size", type=float, default=None, help="K-1 bucket pitch in metres (default: config)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, save the fused BEV maps of the last one (rank 0) as DIR/fused_g<group>.npy, "
                         "float32, 60 MiB in all: a map larger than its share is saved as a seeded sample (see dump_outputs)")
    args = ap.parse_args()
    if args.dump_outputs is not None:
        if args.workload == "train" or args.impl == "reference":
            ap.error("--dump-outputs saves the fused maps of the GPU fusion path; "
                     "it cannot be used with --workload train or --impl reference")
        if args.steps < 1:
            ap.error("--dump-outputs needs at least one timed step (--steps >= 1)")
    if args.workload == "train":
        run_train(args)
    elif args.impl == "reference":
        run_reference(args)
    else:
        run_gpu(args)


if __name__ == "__main__":
    main()
