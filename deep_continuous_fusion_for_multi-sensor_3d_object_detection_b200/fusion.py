"""The continuous-fusion layer as an nn.Module -- the layer the reference leaves as a TODO at
model.py:199-203, inserted after residual groups of ResnetCustomed.forward (model.py:74-78).

Per batch (shared by all scales, `FrameContext`):   K-1 bucket the LiDAR points, K-3 project + gather the
camera features per point.   Per scale (`ContinuousFusion`):   K-4a per-point half of MLP layer 1, K-2 KNN
per BEV cell, K-4 fused MLP + K-sum-pool + BEV add.   All arithmetic is in libcf_b200.so.
"""
from __future__ import annotations

import numpy as np
import torch
import torch.nn as nn

from . import geometry as G
from . import ops


TENSOR_CORE_WIDTHS = (32, 64, 96, 128, 192, 256)   # C with a tcgen05 instantiation of cf_fusion_fwd (cf_mlp_tc.cu)
MAX_FRAMES_PER_CALL = 64                            # cf_fusion_fwd: frames per call on the tensor-core path

_STREAM_POOL = {}   # device index -> side streams, shared by every FrameContext (creating streams per frame is not free)


def rig_image_sizes(img_size, M):
    """M (w, h) image sizes from one pair (every camera) or M pairs."""
    if np.ndim(img_size) == 1:
        return [tuple(float(v) for v in img_size)] * M
    return [tuple(float(v) for v in s) for s in img_size]


class FrameContext:
    """Per-batch state shared by every fusion scale: bucketed points and gathered camera features."""

    def __init__(self, points, num_points, grid: ops.BucketGrid):
        if points.dim() != 3 or points.shape[-1] != 3:
            raise ValueError(f"pointcloud_raw: expected (B,N,3), got {tuple(points.shape)}")
        self.points = ops._contig(points, "pointcloud_raw", torch.float32, 3)
        self.B, self.N = self.points.shape[:2]
        if self.B > MAX_FRAMES_PER_CALL:
            raise ValueError(f"FrameContext: {self.B} frames per call; the fused kernels take at most {MAX_FRAMES_PER_CALL} "
                             f"(split the batch)")
        self.num_points = ops.as_counts(num_points, self.B, self.points.device)
        self.grid = grid
        self.feat = None
        self._gather_ws = None
        self._knn_cache = {}
        self._tables = {}      # id(layer) -> (T, ready event): per-scale point tables computed ahead on side streams
        # K-1 runs on a side stream: the camera-feature gather (K-3) does not depend on it, only the KNN search does
        main = torch.cuda.current_stream(self.points.device)
        st = self._side_streams(1)[0]
        st.wait_stream(main)
        self.points.record_stream(st)       # read by the bucketing stream
        self.num_points.record_stream(st)
        with torch.cuda.stream(st):
            self.bucket_start, self.sorted_pts, self._bucket_ws = ops.bucket_points(self.points, self.num_points, grid)
            self._bucket_done = torch.cuda.Event()
            self._bucket_done.record(st)
        for t in (self.bucket_start, self.sorted_pts, self._bucket_ws):
            t.record_stream(main)

    def gather(self, img_feat, calib=None, uv=None, img_size=(640.0, 480.0)):
        """K-3.  A (B,Ci,Hf,Wf) map: one camera, `calib` the reference's (4,3) CRT_tensor or `uv` the projected points.
        A (B,M,Ci,Hf,Wf) map: a rig of M cameras, `calib` a (B,M,4,3) or (M,4,3) CUDA tensor with w > 0 in front
        (geometry.camera_rig), read on the device; each point gets the mean feature of the cameras that see it.
        A list of M (B,Ci,Hf_m,Wf_m) maps: the same rig with cameras that differ in map and image size; `img_size` is one
        (w, h) for every camera or M of them."""
        if isinstance(img_feat, (list, tuple)):
            if uv is not None:
                raise ValueError("gather: precomputed uv cannot be used with a camera rig (list of maps); pass the rig's calib")
            if calib is None:
                raise ValueError("gather: a camera rig (list of maps) needs calib (B,M,4,3) or (M,4,3)")
            sizes = rig_image_sizes(img_size, len(img_feat))
            if torch.is_grad_enabled() and any(isinstance(m, torch.Tensor) and m.requires_grad for m in img_feat):
                self.feat = _GatherRigFunction.apply(self.points, self.num_points, calib, sizes, *img_feat)
            else:
                self.feat, self._gather_ws = ops.point_gather_rig(img_feat, self.points, self.num_points, calib, sizes,
                                                                  workspace=self._gather_ws)
            return self.feat
        if isinstance(img_feat, torch.Tensor) and img_feat.dim() == 5:
            if uv is not None:
                raise ValueError("gather: precomputed uv cannot be used with a camera rig (5-D map); pass the rig's calib")
            if calib is None:
                raise ValueError("gather: a camera rig (5-D map) needs calib (B,M,4,3) or (M,4,3)")
            if torch.is_grad_enabled() and img_feat.requires_grad:
                self.feat = _GatherMultiFunction.apply(img_feat, self.points, self.num_points, calib, tuple(img_size))
            else:
                self.feat, self._gather_ws = ops.point_gather_multi(img_feat, self.points, self.num_points, calib,
                                                                    img_size=img_size, workspace=self._gather_ws)
            return self.feat
        if torch.is_grad_enabled() and img_feat.requires_grad:
            self.feat = _GatherFunction.apply(img_feat, self.points, self.num_points, calib, uv, tuple(img_size))
        else:
            self.feat, self._gather_ws = ops.point_gather(img_feat, self.points, self.num_points, calib=calib, uv=uv,
                                                          img_size=img_size, workspace=self._gather_ws)
        return self.feat

    def knn(self, H, W, geom, radius, K):
        """(B,H,W,K) int32 neighbour table of one scale, computed once per batch.

        The backbone's scales are nested: with the voxel-consistent centres of geometry.scale_geometry the centre
        of coarse cell (i,j) is bit-identical to fine cell (i*2^m, j*2^m) (same x0,y0; dx,dy scaled by 2^m, an exact
        fp32 scaling), so a coarser table is a strided copy of an already computed finer one (cf_knn_subsample)
        instead of a second search."""
        geom = tuple(float(g) for g in geom)
        key = (H, W, geom, float(radius), int(K))
        if key in self._knn_cache:
            return self._knn_cache[key]
        for (Hf, Wf, gf, rf, Kf), fine in self._knn_cache.items():
            if rf != float(radius) or Kf != int(K) or gf[0] != geom[0] or gf[1] != geom[1]:
                continue
            for m in (2, 4, 8, 16, 32):
                if (float(np.float32(gf[2]) * np.float32(m)) == geom[2] and float(np.float32(gf[3]) * np.float32(m)) == geom[3]
                        and (H - 1) * m < Hf and (W - 1) * m < Wf):
                    self._knn_cache[key] = ops.knn_subsample(fine, m, H, W)
                    return self._knn_cache[key]
        torch.cuda.current_stream(self.points.device).wait_event(self._bucket_done)
        self._knn_cache[key] = ops.knn_query(self.bucket_start, self.sorted_pts, self.grid, H, W, geom, radius, K)
        return self._knn_cache[key]


    # ------------------------------------------------------------------------------------------------------------
    # Scheduling.  The per-scale point tables (K-4a) and the KNN tables (K-2) depend only on the frame, not on the BEV
    # features, and the fusion of different scales is independent once its BEV map exists.  None of these launches
    # fills the GPU on its own, so they are issued on side streams and joined with events: in the detector they run
    # under the backbone's convolutions, in a stand-alone multi-scale call (fuse_scales) they overlap each other.
    # ------------------------------------------------------------------------------------------------------------
    def _side_streams(self, n):
        dev = self.points.device
        pool = _STREAM_POOL.setdefault(dev.index if dev.index is not None else torch.cuda.current_device(), [])
        while len(pool) < n:
            pool.append(torch.cuda.Stream(dev))
        return pool[:n]

    def precompute(self, layers, shapes=None):
        """Launch the point tables of `layers` (and, if `shapes` = [(H,W)] is given, their KNN tables) ahead of use.
        The tables carry no autograd graph: a layer that needs gradients treats its table as an intermediate of its own
        autograd Function (which differentiates through feat / W1 / b1 itself)."""
        if self.feat is None:
            raise ValueError("FrameContext.precompute: call gather() first")
        main = torch.cuda.current_stream(self.points.device)
        streams = self._side_streams(len(layers) + 1)
        dev = self.points.device
        Ci = self.feat.shape[2]
        multi = (len(layers) <= 8 and Ci % 32 == 0 and Ci <= 128 and len({l.mode for l in layers}) == 1
                 and layers[0].mode in ("fp32", "bf16", "bf16t") and all(l.c_bev % 32 == 0 for l in layers)
                 and sum(-(-l.c_bev // 128) for l in layers) <= 16)
        if multi:
            # one launch for every scale: the point features are packed into the tensor-core operand once
            Ts = [torch.empty((self.B, self.N, l.c_bev), dtype=ops.table_dtype(l.mode), device=dev) for l in layers]
            packed = [l._packed.w1(l.fc1.weight.detach(), l.mode) for l in layers]   # packs on the current (main) stream if stale
            st = streams[1]
            st.wait_stream(main)
            with torch.cuda.stream(st), torch.no_grad():
                ops.point_mlp1_multi(self.feat, self.points, self.num_points, [l.fc1.weight for l in layers],
                                     [l.fc1.bias for l in layers], packed, mode=layers[0].mode, outs=Ts)
                ev = torch.cuda.Event()
                ev.record(st)
            for l, T in zip(layers, Ts):
                T.record_stream(st)   # allocated on main's pool, written on st: the block must not be reused before st is done
                self._tables[id(l)] = (T, ev)
        for layer, st in zip([] if multi else layers, streams[1:]):
            T = torch.empty((self.B, self.N, layer.c_bev), dtype=ops.table_dtype(layer.mode), device=dev)
            packed = layer._packed.w1(layer.fc1.weight, layer.mode)   # packs on the current (main) stream if stale
            st.wait_stream(main)
            with torch.cuda.stream(st), torch.no_grad():
                ops.point_mlp1(self.feat, self.points, self.num_points, layer.fc1.weight, layer.fc1.bias, mode=layer.mode,
                               out=T, packed=packed)
                ev = torch.cuda.Event()
                ev.record(st)
            T.record_stream(st)
            self._tables[id(layer)] = (T, ev)
        if shapes is not None:
            # The search runs on the bucketing stream (it only needs K-1, not the gather).  Only the largest map is
            # searched here; tables of nested coarser scales are strided copies of it, made by each layer on its own
            # stream (FrameContext.knn), so they run side by side instead of one after the other.
            st = streams[0]
            with torch.cuda.stream(st):
                big = max(range(len(layers)), key=lambda i: shapes[i][0] * shapes[i][1])
                knn = self.knn(shapes[big][0], shapes[big][1], layers[big].geom, layers[big].radius, layers[big].k)
                knn.record_stream(main)
                ev = torch.cuda.Event()
                ev.record(st)
            self._knn_ready = ev
        return self

    def table_for(self, layer):
        """Precomputed point table of `layer` (waits for it on the current stream) or None."""
        hit = self._tables.get(id(layer))
        if hit is None:
            return None
        torch.cuda.current_stream(self.points.device).wait_event(hit[1])
        return hit[0]

    def wait_knn(self):
        ev = getattr(self, "_knn_ready", None)
        if ev is not None:
            torch.cuda.current_stream(self.points.device).wait_event(ev)


def fuse_scales(frames, layers, bevs, inplace=False):
    """Fuse several backbone scales of one batch at once (inference): tables and KNN ahead on side streams, then one
    stream per scale, joined before returning.  Returns the fused maps in order (`inplace=True`: the inputs, updated
    in place -- the cells without a LiDAR point in reach then cost no memory traffic at all)."""
    dev = frames.points.device
    main = torch.cuda.current_stream(dev)
    with torch.no_grad():
        frames.precompute(layers, [tuple(b.shape[-2:]) for b in bevs])
        frames.wait_knn()
        outs = list(bevs) if inplace else [torch.empty_like(b) for b in bevs]
        streams = frames._side_streams(len(layers) + 1)[1:]
        # Launch order.  The coarse scales' kernels are short latency-bound chains on few CTAs, the fine scales' kernels fill
        # the machine: with several frames per batch, launching the small ones first lets them run beside the tail of the
        # tables / KNN and of each other instead of queueing behind the big ones (batch 4: 3350 -> 3430 frames/s, batch 8:
        # 3764 -> 3868); with one or two frames nothing fills the machine and the longest chain should start first
        # (batch 1: 2087 vs 2118).
        small_first = bevs[0].shape[0] >= 3
        order = sorted(range(len(layers)), key=lambda i: bevs[i].numel(), reverse=not small_first)
        for i in order:
            layer, bev, out, st = layers[i], bevs[i], outs[i], streams[i]
            st.wait_stream(main)
            with torch.cuda.stream(st):
                layer(bev, frames=frames, out=out)
        for st in streams:
            main.wait_stream(st)
    return outs


class FusionRunner:
    """Fixed-shape inference pipeline replayed as ONE CUDA graph: K-1 bucket, K-3 gather, K-4a tables, K-2 KNN and the
    fused layer of every scale (fuse_scales) on static device buffers.

    A serving loop copies a batch into `.points (B,N,3)`, `.num_points (B,) int64`, `.img_feat (B,Ci,Hf,Wf)` and
    `.bevs[s] (B,C_s,H_s,W_s)` (e.g. straight from pinned host memory), calls the runner, and reads `.outs[s]`
    (the same tensors as `.bevs` when `inplace=True`).  Replaying the graph costs one launch on the host instead of the
    ~20 launches and several stream hand-offs of the eager path, which matters when the host is the slow side.
    `dtype=torch.bfloat16`: `.img_feat`, `.bevs` and `.outs` are bf16 maps (half the bytes to copy in and out).
    `memory_format=torch.channels_last`: `.bevs` and `.outs` are channels_last maps, fused by the NHWC kernels.
    `cameras=M`: a camera rig.  `.img_feat` is (B,M,Ci,Hf,Wf) and `.calib` a static (B,M,4,3) float32 device buffer
    (initialised from `calib`, an (M,4,3) or (B,M,4,3) rig such as geometry.camera_rig, if given): calibrations written into
    it between replays take effect without a new capture.  With `img_shape` given as M (Ci, Hf_m, Wf_m) tuples (cameras that
    differ in map size; `img_size` one (w, h) or M of them), `.img_feat` is a list of M static (B,Ci,Hf_m,Wf_m) buffers."""

    def __init__(self, layers, grid, batch, max_points, img_shape, bev_shapes, calib=None, img_size=(640.0, 480.0),
                 inplace=True, device=None, dtype=torch.float32, cameras=None, memory_format=torch.contiguous_format):
        dev = torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)
        self.layers, self.grid, self.calib, self.img_size, self.inplace = list(layers), grid, calib, tuple(img_size), inplace
        self.points = torch.zeros((batch, max_points, 3), dtype=torch.float32, device=dev)
        self.num_points = torch.zeros((batch,), dtype=torch.int64, device=dev)
        if dtype not in ops.MAP_DTYPES:
            raise TypeError(f"FusionRunner: dtype must be torch.float32 or torch.bfloat16, got {dtype}")
        img_feat = None
        if cameras is not None:
            cameras = int(cameras)
            if not 1 <= cameras <= G.MAX_CAMERAS:
                raise ValueError(f"FusionRunner: cameras={cameras}, expected 1..{G.MAX_CAMERAS}")
            self.calib = torch.zeros((batch, cameras, 4, 3), dtype=torch.float32, device=dev)
            if calib is not None:
                self.calib.copy_(torch.as_tensor(calib, dtype=torch.float32, device=dev).expand(batch, cameras, 4, 3))
            if np.ndim(img_shape) == 2:   # one (Ci, Hf_m, Wf_m) per camera
                if len(img_shape) != cameras:
                    raise ValueError(f"FusionRunner: {len(img_shape)} image shapes for {cameras} cameras")
                self.img_size = rig_image_sizes(img_size, cameras)
                img_feat = [torch.zeros((batch,) + tuple(sh), dtype=dtype, device=dev) for sh in img_shape]
            else:
                img_shape = (cameras,) + tuple(img_shape)
        self.img_feat = torch.zeros((batch,) + tuple(img_shape), dtype=dtype, device=dev) if img_feat is None else img_feat
        self.bevs = [torch.zeros((batch,) + tuple(sh), dtype=dtype, device=dev).contiguous(memory_format=memory_format)
                     for sh in bev_shapes]
        self.outs = None
        self.graph = None
        side = torch.cuda.Stream(dev)
        side.wait_stream(torch.cuda.current_stream(dev))
        with torch.cuda.stream(side):            # warm-up outside the capture: packs weights, sizes the allocator
            for _ in range(2):
                self._step()
        torch.cuda.current_stream(dev).wait_stream(side)
        torch.cuda.synchronize(dev)
        self.graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(self.graph):
            self.outs = self._step()

    def _step(self):
        with torch.no_grad():
            frames = FrameContext(self.points, self.num_points, self.grid)
            frames.gather(self.img_feat, calib=self.calib, img_size=self.img_size)
            return fuse_scales(frames, self.layers, self.bevs, inplace=self.inplace)

    def refresh_weights(self):
        """Re-pack the tensor-core operand images of every layer from its current weights (in place: the captured graph
        reads the same buffers).  Call after an optimizer step / load_state_dict and before the next replay -- a replay never
        re-packs by itself unless the pack kernels were part of the capture."""
        with torch.no_grad():
            for l in self.layers:
                l._packed.refresh(l.fc1.weight, l.fc2.weight, l.fc3.weight, l.mode)

    def __call__(self):
        self.graph.replay()
        return self.outs


def prepare_frames(points, num_points, img_feat, config=None, calib=None, uv=None, grid=None, img_size=None):
    """Build the per-batch context: bucket points (K-1) and gather camera features (K-3)."""
    if grid is None:
        config = G.carla_config() if config is None else config
        grid = ops.BucketGrid(*G.bucket_grid(config))
    if img_size is None:
        img_size = (float(config["image_width"]), float(config["image_height"])) if config else (640.0, 480.0)
    ctx = FrameContext(points, num_points, grid)
    ctx.gather(img_feat, calib=calib, uv=uv, img_size=img_size)
    return ctx


class _GatherFunction(torch.autograd.Function):
    """K-3 with its adjoint: the camera map's gradient is the bilinear scatter-add of the per-point gradients."""

    @staticmethod
    def forward(ctx, img_feat, points, num_points, calib, uv, img_size):
        feat, _ = ops.point_gather(img_feat, points, num_points, calib=calib, uv=uv, img_size=img_size)
        ctx.save_for_backward(points, num_points, uv if uv is not None else points.new_empty(0))
        ctx.calib, ctx.has_uv, ctx.img_size, ctx.img_like = calib, uv is not None, img_size, img_feat
        return feat

    @staticmethod
    def backward(ctx, grad_feat):
        points, num_points, uv = ctx.saved_tensors
        gimg = ops.point_gather_bwd(grad_feat, ctx.img_like, points, num_points, calib=None if ctx.has_uv else ctx.calib,
                                    uv=uv if ctx.has_uv else None, img_size=ctx.img_size,
                                    deterministic=torch.are_deterministic_algorithms_enabled())
        return gimg, None, None, None, None, None


class _GatherMultiFunction(torch.autograd.Function):
    """K-3 of a camera rig with its adjoint; the deterministic kernel under torch.use_deterministic_algorithms(True)."""

    @staticmethod
    def forward(ctx, img_feats, points, num_points, calib, img_size):
        feat, _ = ops.point_gather_multi(img_feats, points, num_points, calib, img_size=img_size)
        ctx.save_for_backward(points, num_points, calib)
        ctx.img_size, ctx.img_like = img_size, img_feats
        return feat

    @staticmethod
    def backward(ctx, grad_feat):
        points, num_points, calib = ctx.saved_tensors
        det = torch.are_deterministic_algorithms_enabled()
        gimg = ops.point_gather_multi_bwd(grad_feat, ctx.img_like, points, num_points, calib, img_size=ctx.img_size,
                                          deterministic=det)
        return gimg, None, None, None, None


class _GatherRigFunction(torch.autograd.Function):
    """K-3 of a rig whose cameras differ in map and image size, with its adjoint: one gradient per camera map; the
    deterministic kernel under torch.use_deterministic_algorithms(True)."""

    @staticmethod
    def forward(ctx, points, num_points, calib, img_sizes, *maps):
        feat, _ = ops.point_gather_rig(list(maps), points, num_points, calib, img_sizes)
        ctx.save_for_backward(points, num_points, calib)
        ctx.img_sizes, ctx.maps_like = img_sizes, maps
        return feat

    @staticmethod
    def backward(ctx, grad_feat):
        points, num_points, calib = ctx.saved_tensors
        det = torch.are_deterministic_algorithms_enabled()
        gimgs = ops.point_gather_rig_bwd(grad_feat, list(ctx.maps_like), points, num_points, calib, ctx.img_sizes,
                                         deterministic=det)
        return (None, None, None, None) + tuple(gimgs)


class _FusionFunction(torch.autograd.Function):
    """Forward = cf_point_mlp1 + cf_fusion_fwd.  Saves indices, inputs and weights, never the gathered rows."""

    @staticmethod
    def forward(ctx, bev, feat, points, num_points, knn_idx, geom, mode, w1, b1, w2, b2, w3, b3, packed=None, table=None,
                out=None):
        p23 = packed.w23(w2, w3, mode) if packed is not None else None
        if table is None:
            p1 = packed.w1(w1, mode) if packed is not None else None
            table = ops.point_mlp1(feat, points, num_points, w1, b1, mode=mode, packed=p1)
        out, _ = ops.fusion_fwd(bev, table, knn_idx, geom, w1, w2, b2, w3, b3, mode=mode, packed=p23, out=out,
                                memory_format=ops.map_format(bev))
        # the table is kept for the backward (B*N*C floats: far smaller than the activations autograd keeps for one conv)
        ctx.save_for_backward(feat, points, num_points, knn_idx, w1, b1, w2, b2, w3, b3, table)
        ctx.geom, ctx.mode = geom, mode
        return out

    @staticmethod
    def backward(ctx, grad_out):
        feat, points, num_points, knn_idx, w1, b1, w2, b2, w3, b3, table = ctx.saved_tensors
        gw1, gb1, gw2, gb2, gw3, gb3, gfeat = ops.fusion_bwd(grad_out, feat, points, num_points, knn_idx, ctx.geom, w1, b1,
                                                             w2, b2, w3, table=table, mode=ctx.mode,
                                                             deterministic=torch.are_deterministic_algorithms_enabled())
        # d out / d bev is the identity
        return grad_out, gfeat, None, None, None, None, None, gw1, gb1, gw2, gb2, gw3, gb3, None, None, None


class ContinuousFusion(nn.Module):
    """out = bev + sum_{k in KNN(cell)} MLP([camera feature of point k, offset of point k to the cell]).

    Parameters follow SURVEY Appendix A9: Linear(c_img+3, c_bev) - ReLU - Linear(c_bev, c_bev) - ReLU -
    Linear(c_bev, c_bev), input order [image feature | offset].
    `geom` = (x0, y0, dx, dy) float32 scalars of the BEV cell centres at this scale (geometry.scale_geometry).
    """

    def __init__(self, c_img: int, c_bev: int, k: int = 3, radius: float = 2.0, geom=None, mode: str = "fp32"):
        super().__init__()
        if not (1 <= k <= 16):
            raise ValueError("k must be in [1, 16]")
        if mode not in ("fp32", "bf16", "simt", "bf16t"):
            raise ValueError(f"mode must be 'fp32', 'bf16', 'bf16t' (bf16 with bf16 tables, inference only) or 'simt', got {mode!r}")
        if c_bev % 16 or not (16 <= c_bev <= 256):
            raise ValueError("c_bev must be a multiple of 16 in [16, 256]")
        if mode != "simt" and c_bev not in TENSOR_CORE_WIDTHS:
            # the tcgen05 kernels are instantiated for the backbone's widths; anything else would only fail at the first forward
            raise ValueError(f"c_bev={c_bev} has no tensor-core instantiation (modes 'fp32' / 'bf16' support {TENSOR_CORE_WIDTHS}); "
                             f"use mode='simt' for other multiples of 16")
        if c_img % 4:
            raise ValueError("c_img must be a multiple of 4")
        self.c_img, self.c_bev, self.k, self.radius, self.mode = c_img, c_bev, int(k), float(radius), mode
        self.geom = tuple(float(g) for g in geom) if geom is not None else None
        self.fc1 = nn.Linear(c_img + 3, c_bev)
        self.fc2 = nn.Linear(c_bev, c_bev)
        self.fc3 = nn.Linear(c_bev, c_bev)
        self._packed = ops.PackedWeights()   # operand images of the weights, re-packed only when they change

    def extra_repr(self):
        return f"c_img={self.c_img}, c_bev={self.c_bev}, k={self.k}, radius={self.radius}, mode={self.mode}"

    def forward(self, bev, img_feat=None, points=None, num_points=None, calib=None, uv=None, frames: FrameContext = None,
                geom=None, return_knn: bool = False, out=None):
        """Returns a map of bev's dtype: fp32, or bf16 (under torch.autocast the maps arrive in bf16; autocast does not cast
        the inputs of this layer, which widens bf16 maps exactly and computes in fp32 with fp32 weights).
        A channels_last-dense bev (a backbone converted with .to(memory_format=torch.channels_last)) is fused by the NHWC
        kernels without a layout copy and gives a channels_last map; `out`, if given, must then be channels_last too.
        Any other bev is fused as an NCHW map."""
        geom = tuple(float(g) for g in geom) if geom is not None else self.geom
        if geom is None:
            raise ValueError("ContinuousFusion: BEV geometry (x0,y0,dx,dy) not set")
        if bev.dim() != 4 or bev.shape[1] != self.c_bev:
            raise ValueError(f"bev: expected (B,{self.c_bev},H,W), got {tuple(bev.shape)}")
        if frames is None:
            if img_feat is None or points is None or num_points is None:
                raise ValueError("ContinuousFusion: pass either frames= or img_feat/points/num_points")
            frames = prepare_frames(points, num_points, img_feat, calib=calib, uv=uv)
        if frames.feat is None:
            raise ValueError("ContinuousFusion: FrameContext has no gathered camera features (call .gather)")
        if frames.feat.shape[2] != self.c_img:
            raise ValueError(f"camera feature width {frames.feat.shape[2]} != c_img {self.c_img}")
        B, _, H, W = bev.shape
        knn_idx = frames.knn(H, W, geom, self.radius, self.k)
        args = (bev, frames.feat, frames.points, frames.num_points, knn_idx, geom, self.mode, self.fc1.weight,
                self.fc1.bias, self.fc2.weight, self.fc2.bias, self.fc3.weight, self.fc3.bias, self._packed)
        needs_grad = torch.is_grad_enabled() and (bev.requires_grad or frames.feat.requires_grad or
                                                  any(p.requires_grad for p in self.parameters()))
        if needs_grad and self.mode == "bf16t":
            raise RuntimeError("ContinuousFusion: mode 'bf16t' stores the layer-1 tables as bf16 and is inference only; "
                               "train in 'fp32' or 'bf16' (same weights) and switch layer.mode for deployment")
        if needs_grad:
            # a table launched ahead by FrameContext.precompute is only an intermediate of this Function: its gradient
            # path (feat, W1, b1) is the Function's own backward, so it can be used here as well
            out = _FusionFunction.apply(*args, frames.table_for(self), None)
        else:
            with torch.no_grad():
                out = _FusionFunction.forward(_NullCtx(), *[a.detach() if isinstance(a, torch.Tensor) else a for a in args],
                                              table=frames.table_for(self), out=out)
        return (out, knn_idx) if return_knn else out


class _NullCtx:
    def save_for_backward(self, *a):
        pass
