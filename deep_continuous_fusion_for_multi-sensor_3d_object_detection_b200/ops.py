"""Thin torch-tensor wrappers, one per C-ABI entry point of include/cf_b200.h.

PyTorch is plumbing here: it owns device memory and the current stream; all arithmetic happens in
libcf_b200.so.  Every wrapper validates device / dtype / contiguity and raises instead of falling back.
"""
from __future__ import annotations

import ctypes as C

import numpy as np
import torch

from . import _lib
from ._lib import check, load, ptr, stream_ptr


def _req(t: torch.Tensor, name: str, dtype, ndim=None):
    if not isinstance(t, torch.Tensor):
        raise TypeError(f"{name}: expected a torch.Tensor, got {type(t).__name__}")
    if not t.is_cuda:
        raise RuntimeError(f"{name}: must be a CUDA tensor (this package has no CPU path)")
    if t.dtype != dtype:
        raise TypeError(f"{name}: expected dtype {dtype}, got {t.dtype}")
    if ndim is not None and t.dim() != ndim:
        raise ValueError(f"{name}: expected {ndim} dims, got shape {tuple(t.shape)}")
    return t


def _contig(t: torch.Tensor, name: str, dtype, ndim=None):
    _req(t, name, dtype, ndim)
    return t if t.is_contiguous() else t.contiguous()


def _scratch(nbytes: int, device) -> torch.Tensor:
    """Workspace that the kernels write before they read it.  torch.use_deterministic_algorithms(True) makes torch.empty fill
    new memory (hundreds of MB per backward call here); scratch needs no fill, so it is allocated without one."""
    import torch.utils.deterministic as det
    prev = det.fill_uninitialized_memory
    det.fill_uninitialized_memory = False
    try:
        return torch.empty((max(int(nbytes), 16),), dtype=torch.uint8, device=device)
    finally:
        det.fill_uninitialized_memory = prev


def as_counts(num_points, B: int, device) -> torch.Tensor:
    """sample["num_points_raw"] after collation is a (B,) int64 CPU tensor (data_import_carla.py:262)."""
    if not isinstance(num_points, torch.Tensor):
        num_points = torch.as_tensor(np.asarray(num_points), dtype=torch.int64)
    num_points = num_points.reshape(-1).to(device=device, dtype=torch.int64, non_blocking=True)
    if num_points.numel() != B:
        raise ValueError(f"num_points: expected {B} entries, got {num_points.numel()}")
    return num_points.contiguous()


_CALIB_CACHE = {}


def _calib_host(calib):
    """(4,3) CRT_tensor -> ctypes float[12].  A device tensor (the drop-in model registers it as a buffer that .cuda()
    moves) is copied to the host ONCE per (storage, version): the calls stay free of host synchronisation afterwards and
    remain capturable in a CUDA graph."""
    if isinstance(calib, torch.Tensor):
        key = (calib.data_ptr(), calib._version, calib.device)
        hit = _CALIB_CACHE.get(key)
        if hit is not None:
            return hit
        if calib.is_cuda and torch.cuda.is_current_stream_capturing():
            raise RuntimeError("calib: first use of a device-resident CRT_tensor inside CUDA-graph capture; call the layer "
                               "once before capturing (or pass a host array)")
        arr = calib.detach().to("cpu", torch.float32).numpy()
    else:
        key = None
        arr = np.asarray(calib, dtype=np.float32)
    arr = np.ascontiguousarray(arr, dtype=np.float32)
    if arr.shape != (4, 3):
        raise ValueError(f"calib: expected (4,3) CRT_tensor, got {arr.shape}")
    out = (C.c_float * 12)(*arr.reshape(-1).tolist())
    if key is not None:
        if len(_CALIB_CACHE) > 64:
            _CALIB_CACHE.clear()
        _CALIB_CACHE[key] = out
    return out


class BucketGrid:
    """Uniform BEV bucket grid (K-1) + the per-batch sorted point storage."""

    def __init__(self, gx0, gy0, cell, nbx, nby):
        self.gx0, self.gy0, self.cell = float(gx0), float(gy0), float(cell)
        self.nbx, self.nby = int(nbx), int(nby)


def bucket_points(points: torch.Tensor, num_points: torch.Tensor, grid: BucketGrid, out=None):
    """K-1.  points (B,N,3) f32, num_points (B,) i64 -> bucket_start (B,G+1) i32, sorted (B,N,4) f32."""
    lib = load()
    points = _contig(points, "points", torch.float32, 3)
    B, N, three = points.shape
    if three != 3:
        raise ValueError(f"points: last dim must be 3, got {three}")
    num_points = _req(num_points, "num_points", torch.int64, 1)
    G = grid.nbx * grid.nby
    if out is None:
        start = torch.empty((B, G + 1), dtype=torch.int32, device=points.device)
        srt = torch.empty((B, N, 4), dtype=torch.float32, device=points.device)
        ws = torch.empty((max(lib.cf_bucket_workspace_bytes(B, grid.nbx, grid.nby), 16),), dtype=torch.uint8,
                         device=points.device)
    else:
        start, srt, ws = out
    check(lib.cf_bucket_points(ptr(points), ptr(num_points), B, N, grid.gx0, grid.gy0, grid.cell, grid.nbx, grid.nby,
                               ptr(start), ptr(srt), ptr(ws), stream_ptr()), "cf_bucket_points")
    return start, srt, ws


def voxelize_project(raw, num_raw, config, calib, max_num_pc=None, workspace=None):
    """Dataset side on the device: CarlaDataset.Voxelization_Projection (data_import_carla.py:212-267) for a batch.

    raw (B,Nraw,3) f32 LiDAR xyz, num_raw (B,) valid rows -> (lidar_voxel (B,Z,X,Y), pointcloud_raw (B,max_num_pc,3),
    projected_loc_uv (B,max_num_pc,2), num_points_raw (B,) int64): the sample[...] tensors of the reference dataset."""
    import ctypes as C
    from . import geometry as G
    lib = load()
    raw = _contig(raw, "raw", torch.float32, 3)
    B, Nraw, three = raw.shape
    if three != 3:
        raise ValueError(f"raw: last dim must be 3, got {three}")
    num_raw = as_counts(num_raw, B, raw.device)
    Z, X, Y = int(config["voxel_channel"]), int(config["voxel_length"]), int(config["voxel_width"])
    N = int(config["max_num_pc"] if max_num_pc is None else max_num_pc)
    f6 = lambda v: (C.c_float * 6)(*[float(x) for x in v])
    crt = _calib_host(calib)
    need = lib.cf_voxelize_workspace_bytes(B, Nraw, Z, X, Y)
    if workspace is None or workspace.numel() < need:
        workspace = torch.empty((need,), dtype=torch.uint8, device=raw.device)
    vox = torch.empty((B, Z, X, Y), dtype=torch.float32, device=raw.device)
    pts = torch.empty((B, N, 3), dtype=torch.float32, device=raw.device)
    uv = torch.empty((B, N, 2), dtype=torch.float32, device=raw.device)
    num = torch.empty((B,), dtype=torch.int64, device=raw.device)
    check(lib.cf_voxelize_project(ptr(raw), ptr(num_raw), B, Nraw, f6(G.lidar_range(config)), f6(G.voxel_matrix(config)), Z, X, Y,
                                  crt, float(config["image_height"]),
                                  float(config["image_width"]), N, ptr(vox), ptr(pts), ptr(uv), ptr(num), ptr(workspace),
                                  stream_ptr()), "cf_voxelize_project")
    return vox, pts, uv, num


def knn_query(bucket_start, sorted_pts, grid: BucketGrid, H, W, geom, radius, K, out=None):
    """K-2.  -> knn_idx (B,H,W,K) int32, -1 = empty slot."""
    lib = load()
    _req(bucket_start, "bucket_start", torch.int32, 2)
    _req(sorted_pts, "sorted_pts", torch.float32, 3)
    B, N, _ = sorted_pts.shape
    x0, y0, dx, dy = [float(g) for g in geom]
    if out is None:
        out = torch.empty((B, H, W, K), dtype=torch.int32, device=sorted_pts.device)
    check(lib.cf_knn_query(ptr(bucket_start), ptr(sorted_pts), B, N, grid.gx0, grid.gy0, grid.cell, grid.nbx, grid.nby,
                           H, W, x0, y0, dx, dy, float(radius), int(K), ptr(out), stream_ptr()), "cf_knn_query")
    return out


def knn_subsample(knn_fine, step, Hc, Wc):
    """KNN table of a `step`-times coarser scale whose cell centres coincide with every step-th fine centre."""
    lib = load()
    knn_fine = _contig(knn_fine, "knn_fine", torch.int32, 4)
    B, Hf, Wf, K = knn_fine.shape
    out = torch.empty((B, Hc, Wc, K), dtype=torch.int32, device=knn_fine.device)
    check(lib.cf_knn_subsample(ptr(knn_fine), B, Hf, Wf, int(step), ptr(out), Hc, Wc, K, stream_ptr()), "cf_knn_subsample")
    return out


def point_gather(img_feat, points, num_points, calib=None, uv=None, img_size=(640.0, 480.0), out=None, workspace=None):
    """K-3.  img_feat logical (B,Ci,Hf,Wf) (any strides; channels_last avoids the re-layout pass),
    points (B,N,3), exactly one of calib ((4,3) array, host) / uv ((B,N,2) device) -> feat (B,N,Ci)."""
    lib = load()
    _req(img_feat, "img_feat", torch.float32, 4)
    points = _contig(points, "points", torch.float32, 3)
    B, Ci, Hf, Wf = img_feat.shape
    N = points.shape[1]
    sb, sc, sh, sw = img_feat.stride()
    if (calib is None) == (uv is None):
        raise ValueError("pass exactly one of calib / uv")
    calib_arr = None
    if calib is not None:
        calib_arr = _calib_host(calib)
    else:
        uv = _contig(uv, "uv", torch.float32, 3)
        if uv.shape != (B, N, 2):
            raise ValueError(f"uv: expected {(B, N, 2)}, got {tuple(uv.shape)}")
    if out is None:
        out = torch.empty((B, N, Ci), dtype=torch.float32, device=points.device)
    need = lib.cf_gather_workspace_bytes(B, Ci, Hf, Wf, sc)
    if need and (workspace is None or workspace.numel() < need):
        workspace = torch.empty((need,), dtype=torch.uint8, device=points.device)
    check(lib.cf_point_gather(ptr(img_feat), sb, sc, sh, sw, B, Ci, Hf, Wf, ptr(points), ptr(uv), calib_arr,
                              ptr(num_points), N, float(img_size[0]), float(img_size[1]), ptr(out), ptr(workspace),
                              stream_ptr()), "cf_point_gather")
    return out, workspace


class PackedWeights:
    """Cache of the UMMA operand images of one layer's weights.  Re-packs only when a weight tensor was modified
    in place (optimizer step -> Tensor._version changes) or replaced; in inference the weights are packed once."""

    def __init__(self):
        self._key1, self._buf1, self._key23, self._buf23 = None, None, None, None

    def invalidate(self):
        """Forget the cached keys: the next w1() / w23() re-packs (in place, so buffers captured by a CUDA graph see it)."""
        self._key1 = self._key23 = None

    def refresh(self, W1, W2, W3, mode):
        """Re-pack every operand image now, on the current stream.  Call after the weights changed and before replaying a
        CUDA graph that captured the layer (FusionRunner.refresh_weights does): replays read the images, they do not re-pack."""
        self.invalidate()
        return self.w1(W1, mode), self.w23(W2, W3, mode)

    @staticmethod
    def _repack_in_capture(W):
        """While a TRAINING step is being captured (autograd on) the pack kernels are always emitted, so that every replay
        re-packs from the weights the optimizer just updated, whatever ran between the last step and the capture.  An
        inference capture (torch.no_grad, FusionRunner) keeps the images static: call refresh() when the weights change."""
        return W.is_cuda and torch.is_grad_enabled() and torch.cuda.is_current_stream_capturing()

    @staticmethod
    def _key(*tensors, mode):
        return tuple((t.data_ptr(), t._version, tuple(t.shape)) for t in tensors) + (mode,)

    def w1(self, W1, mode):
        lib = load()
        m = _lib.MODES[mode]
        if m == _lib.MODE_SIMT:
            return None
        C_out, Ci = W1.shape[0], W1.shape[1] - 3
        if Ci % 16 or Ci > 256 or C_out % 32:
            return None
        key = self._key(W1, mode=m)
        if key != self._key1 or self._repack_in_capture(W1):
            need = lib.cf_point_mlp1_workspace_bytes(Ci, C_out, m)
            if self._buf1 is None or self._buf1.numel() != need or self._buf1.device != W1.device:
                self._buf1 = torch.empty((need,), dtype=torch.uint8, device=W1.device)   # else: repack in place, so a
                # CUDA graph that captured this buffer (FusionRunner) sees the refreshed image
            check(lib.cf_point_mlp1_pack_weights(ptr(W1.detach().contiguous()), Ci, C_out, m, ptr(self._buf1), stream_ptr()),
                  "cf_point_mlp1_pack_weights")
            self._key1 = key
        return self._buf1

    def w23(self, W2, W3, mode):
        lib = load()
        m = _lib.MODES[mode]
        Cc = W2.shape[0]
        if m == _lib.MODE_SIMT or Cc % 32:
            return None
        key = self._key(W2, W3, mode=m)
        if key != self._key23 or self._repack_in_capture(W2):
            need = lib.cf_fusion_packed_bytes(Cc, m)
            if self._buf23 is None or self._buf23.numel() != need or self._buf23.device != W2.device:
                self._buf23 = torch.empty((need,), dtype=torch.uint8, device=W2.device)
            check(lib.cf_fusion_pack_weights(ptr(W2.detach().contiguous()), ptr(W3.detach().contiguous()), Cc, m,
                                             ptr(self._buf23), stream_ptr()), "cf_fusion_pack_weights")
            self._key23 = key
        return self._buf23


def _table_check(t, name, m, shape):
    """A caller-supplied table must have the mode's dtype: the kernels take raw pointers."""
    want = table_dtype(m)
    if t.dtype != want or tuple(t.shape) != tuple(shape) or not t.is_contiguous() or not t.is_cuda:
        raise ValueError(f"{name}: expected a contiguous CUDA {want} tensor of shape {tuple(shape)}, got {t.dtype} {tuple(t.shape)}")


def table_dtype(mode):
    """dtype of the layer-1 tables T in `mode`: bf16 in "bf16t" (CF_MODE_BF16_TABLES), fp32 otherwise."""
    m = _lib.MODES[mode] if isinstance(mode, str) else int(mode)
    return torch.bfloat16 if m == _lib.MODE_BF16_TABLES else torch.float32


def point_mlp1(feat, points, num_points, W1, b1, mode="fp32", out=None, workspace=None, packed=None):
    """K-4a.  T (B,N,C) = feat W1[:, :Ci]^T + points W1[:, Ci:]^T + b1  (fp32; bf16 rows in mode "bf16t")."""
    lib = load()
    feat = _contig(feat, "feat", torch.float32, 3)
    points = _contig(points, "points", torch.float32, 3)
    W1 = _contig(W1, "W1", torch.float32, 2)
    b1 = _contig(b1, "b1", torch.float32, 1)
    B, N, Ci = feat.shape
    C_out = W1.shape[0]
    if W1.shape[1] != Ci + 3 or b1.shape[0] != C_out:
        raise ValueError(f"W1/b1: expected ({C_out},{Ci + 3})/({C_out},), got {tuple(W1.shape)}/{tuple(b1.shape)}")
    m = _lib.MODES[mode] if isinstance(mode, str) else int(mode)
    need = 0 if packed is not None else lib.cf_point_mlp1_workspace_bytes(Ci, C_out, m)
    if need and (workspace is None or workspace.numel() < need):
        workspace = torch.empty((need,), dtype=torch.uint8, device=feat.device)
    if out is None:
        out = torch.empty((B, N, C_out), dtype=table_dtype(m), device=feat.device)
    _table_check(out, "point_mlp1: out", m, (B, N, C_out))
    check(lib.cf_point_mlp1(ptr(feat), ptr(points), ptr(num_points), B, N, Ci, C_out, ptr(W1), ptr(b1), ptr(out), m,
                            ptr(packed), ptr(workspace) if need else None, stream_ptr()), "cf_point_mlp1")
    return out


def point_mlp1_multi(feat, points, num_points, W1s, b1s, packeds, mode="fp32", outs=None):
    """K-4a for several scales in ONE launch (cf_point_mlp1_multi): the point features are packed into the tensor-core
    operand once and multiplied by every scale's W1.  `packeds` = the scales' packed W1 images (PackedWeights.w1).
    Returns the list of T (B,N,C_s), identical to per-scale point_mlp1 calls."""
    import ctypes as C
    lib = load()
    feat = _contig(feat, "feat", torch.float32, 3)
    points = _contig(points, "points", torch.float32, 3)
    B, N, Ci = feat.shape
    n = len(W1s)
    W1s = [_contig(w, "W1", torch.float32, 2) for w in W1s]
    b1s = [_contig(b, "b1", torch.float32, 1) for b in b1s]
    for w, b in zip(W1s, b1s):
        if w.shape[1] != Ci + 3 or b.shape[0] != w.shape[0]:
            raise ValueError(f"W1/b1: expected (C,{Ci + 3})/(C,), got {tuple(w.shape)}/{tuple(b.shape)}")
    if len(b1s) != n or len(packeds) != n or any(pk is None for pk in packeds):
        raise ValueError("point_mlp1_multi: one W1, b1 and packed image per scale")
    m = _lib.MODES[mode] if isinstance(mode, str) else int(mode)
    if outs is None:
        outs = [torch.empty((B, N, w.shape[0]), dtype=table_dtype(m), device=feat.device) for w in W1s]
    for t, w in zip(outs, W1s):
        _table_check(t, "point_mlp1_multi: outs", m, (B, N, w.shape[0]))
    arr = lambda ts: (C.c_void_p * n)(*[t.data_ptr() for t in ts])
    hC = (C.c_int32 * n)(*[int(w.shape[0]) for w in W1s])
    check(lib.cf_point_mlp1_multi(ptr(feat), ptr(points), ptr(num_points), B, N, Ci, n, hC, arr(W1s), arr(b1s), arr(outs), m,
                                  arr(packeds), stream_ptr()), "cf_point_mlp1_multi")
    return outs


def fusion_fwd(bev, T, knn_idx, geom, W1, W2, b2, W3, b3, mode="fp32", out=None, workspace=None, packed=None):
    """K-4.  out = bev + W3 sum_k relu(W2 relu(T[idx_k] - e_cell) + b2) + n_valid b3."""
    lib = load()
    _req(bev, "bev", torch.float32, 4)
    if out is not None:
        _req(out, "out", torch.float32, 4)
        if out.shape != bev.shape or out.device != bev.device or not out.is_contiguous():
            raise ValueError(f"fusion_fwd: out must be a contiguous (dense NCHW) tensor of bev's shape {tuple(bev.shape)} on "
                             f"{bev.device}, got shape {tuple(out.shape)}, strides {out.stride()}, device {out.device}")
        if out.data_ptr() == bev.data_ptr() and not bev.is_contiguous():
            raise ValueError("fusion_fwd: in-place operation (out is bev) needs a contiguous (dense NCHW) map")
    bev = _contig(bev, "bev", torch.float32, 4)
    T = _contig(T, "T", table_dtype(mode), 3)
    knn_idx = _contig(knn_idx, "knn_idx", torch.int32, 4)
    B, Cc, H, W = bev.shape
    N = T.shape[1]
    K = knn_idx.shape[3]
    if T.shape[0] != B or T.shape[2] != Cc or tuple(knn_idx.shape[:3]) != (B, H, W):
        raise ValueError("fusion_fwd: inconsistent shapes")
    W1 = _contig(W1, "W1", torch.float32, 2)
    W2 = _contig(W2, "W2", torch.float32, 2)
    W3 = _contig(W3, "W3", torch.float32, 2)
    b2 = _contig(b2, "b2", torch.float32, 1)
    b3 = _contig(b3, "b3", torch.float32, 1)
    Ci = W1.shape[1] - 3
    m = _lib.MODES[mode] if isinstance(mode, str) else int(mode)
    need = max(lib.cf_fusion_workspace_bytes(Cc, m, B, H, W), 16)
    if workspace is None or workspace.numel() < need:
        workspace = torch.empty((need,), dtype=torch.uint8, device=bev.device)
    if out is None:
        out = torch.empty_like(bev)
    x0, y0, dx, dy = [float(g) for g in geom]
    check(lib.cf_fusion_fwd(ptr(bev), ptr(T), ptr(knn_idx), B, N, Cc, H, W, K, x0, y0, dx, dy, ptr(W1), Ci, ptr(W2),
                            ptr(b2), ptr(W3), ptr(b3), ptr(out), m, ptr(packed), ptr(workspace), stream_ptr()),
          "cf_fusion_fwd")
    return out, workspace


def fusion_bwd(grad_out, feat, points, num_points, knn_idx, geom, W1, b1, W2, b2, W3, grad_feat=None, table=None,
               mode="fp32", deterministic=False):
    """K-4b.  Returns (gW1, gb1, gW2, gb2, gW3, gb3, gfeat); d bev is grad_out itself.
    `table`: the forward's point_mlp1 output (B,N,C) if it was kept (else it is recomputed); `mode` "simt" keeps every
    GEMM on CUDA cores, any other mode runs them on tcgen05 with fp32-accurate split operands.
    `deterministic`: fixed summation order everywhere (CF_BWD_DETERMINISTIC): identical inputs give bit-identical gradients."""
    lib = load()
    grad_out = _contig(grad_out, "grad_out", torch.float32, 4)
    feat = _contig(feat, "feat", torch.float32, 3)
    points = _contig(points, "points", torch.float32, 3)
    knn_idx = _contig(knn_idx, "knn_idx", torch.int32, 4)
    W1, W2, W3 = [_contig(w, "W", torch.float32, 2) for w in (W1, W2, W3)]
    b1, b2 = _contig(b1, "b1", torch.float32, 1), _contig(b2, "b2", torch.float32, 1)
    B, Cc, H, W = grad_out.shape
    N, Ci, K = feat.shape[1], feat.shape[2], knn_idx.shape[3]
    dev = grad_out.device
    gW1, gb1 = torch.zeros_like(W1), torch.zeros_like(b1)
    gW2, gb2 = torch.zeros_like(W2), torch.zeros_like(b2)
    gW3, gb3 = torch.zeros_like(W3), torch.zeros((Cc,), dtype=torch.float32, device=dev)
    gfeat = torch.zeros_like(feat) if grad_feat is None else grad_feat
    if table is not None:
        table = _contig(table, "table", torch.float32, 3)
        if tuple(table.shape) != (B, N, Cc):
            raise ValueError("fusion_bwd: table must be (B, N, C)")
    ws_bytes = (lib.cf_fusion_bwd_det_workspace_bytes if deterministic else lib.cf_fusion_bwd_workspace_bytes)(B, N, Cc, Ci, H, W, K)
    ws = _scratch(ws_bytes, dev)
    m = _lib.MODES[mode] if isinstance(mode, str) else int(mode)
    if deterministic:
        m |= _lib.BWD_DETERMINISTIC
    x0, y0, dx, dy = [float(g) for g in geom]
    check(lib.cf_fusion_bwd(ptr(grad_out), ptr(feat), ptr(points), ptr(num_points), ptr(knn_idx), B, N, Cc, H, W, K, x0, y0,
                            dx, dy, ptr(W1), ptr(b1), Ci, ptr(W2), ptr(b2), ptr(W3), ptr(table), ptr(gW1), ptr(gb1), ptr(gW2),
                            ptr(gb2), ptr(gW3), ptr(gb3), ptr(gfeat), m, ptr(ws), stream_ptr()), "cf_fusion_bwd")
    return gW1, gb1, gW2, gb2, gW3, gb3, gfeat


def point_gather_bwd(grad_feat, img_like, points, num_points, calib=None, uv=None, img_size=(640.0, 480.0),
                     deterministic=False):
    """Adjoint of point_gather: gradient w.r.t. the camera feature map (same shape / memory format as img_like).
    `deterministic`: each pixel sums its (point, tap) contributions in a fixed order (cf_point_gather_bwd_det)."""
    lib = load()
    grad_feat = _contig(grad_feat, "grad_feat", torch.float32, 3)
    points = _contig(points, "points", torch.float32, 3)
    gimg = torch.zeros_like(img_like)
    B, Ci, Hf, Wf = gimg.shape
    sb, sc, sh, sw = gimg.stride()
    calib_arr = None
    if calib is not None:
        calib_arr = _calib_host(calib)
    else:
        uv = _contig(uv, "uv", torch.float32, 3)
    N = points.shape[1]
    if deterministic:
        ws = _scratch(lib.cf_point_gather_bwd_det_workspace_bytes(B, N, Hf, Wf), gimg.device)
        check(lib.cf_point_gather_bwd_det(ptr(grad_feat), ptr(gimg), sb, sc, sh, sw, B, Ci, Hf, Wf, ptr(points), ptr(uv),
                                          calib_arr, ptr(num_points), N, float(img_size[0]), float(img_size[1]), ptr(ws),
                                          stream_ptr()), "cf_point_gather_bwd_det")
        return gimg
    check(lib.cf_point_gather_bwd(ptr(grad_feat), ptr(gimg), sb, sc, sh, sw, B, Ci, Hf, Wf, ptr(points), ptr(uv), calib_arr,
                                  ptr(num_points), N, float(img_size[0]), float(img_size[1]), stream_ptr()),
          "cf_point_gather_bwd")
    return gimg


# ------------------------------------------------------------------------------------------ post-process
def loss_targets(ref_boxes, num_ref, H, W, scales, reduced_scale, positive_range, regress_type, pos_threshold, neg_threshold,
                 shuffle_keys, candidates):
    """SURVEY 8(f-4): LossTotal's target assignment (loss.py:74-127) for the whole batch in one launch.
    ref_boxes (B,M,>=2) fp32, num_ref (B) int; scales = (x_scale, y_scale, x_offset, y_offset) of loss.py:80-83;
    shuffle_keys (B, M*R*R) fp32 and candidates (B,L,2) int32 are the random draws (RNG contract: include/cf_b200.h).
    Returns pos_cells (B,pos_threshold), pos_count (B), neg_cells (B,neg_threshold+1), neg_count (B), reg_cells (B,M,R*R):
    int32 linear cells x*W+y, -1 padded."""
    ref_boxes = _contig(ref_boxes, "ref_boxes", torch.float32, 3)
    B, M, stride = ref_boxes.shape
    num_ref = as_counts(num_ref, B, ref_boxes.device)
    R = int(positive_range)
    shuffle_keys = _contig(shuffle_keys, "shuffle_keys", torch.float32, 2)
    candidates = _contig(candidates, "candidates", torch.int32, 3)
    if tuple(shuffle_keys.shape) != (B, M * R * R) or candidates.shape[0] != B or candidates.shape[2] != 2:
        raise ValueError("loss_targets: shuffle_keys must be (B, M*R*R), candidates (B, L, 2)")
    dev = ref_boxes.device
    pos = torch.empty((B, int(pos_threshold)), dtype=torch.int32, device=dev)
    neg = torch.empty((B, int(neg_threshold) + 1), dtype=torch.int32, device=dev)
    npos = torch.empty((B,), dtype=torch.int32, device=dev)
    nneg = torch.empty((B,), dtype=torch.int32, device=dev)
    reg = torch.empty((B, M, R * R), dtype=torch.int32, device=dev)
    xs, ys, xo, yo = (float(v) for v in scales)
    check(load().cf_loss_targets(ptr(ref_boxes), ptr(num_ref), B, M, stride, int(H), int(W), xs, ys, xo, yo, float(reduced_scale), R,
                                 int(regress_type), int(pos_threshold), int(neg_threshold), ptr(shuffle_keys), ptr(candidates),
                                 int(candidates.shape[1]), ptr(pos), ptr(npos), ptr(neg), ptr(nneg), ptr(reg), stream_ptr()),
          "cf_loss_targets")
    return pos, npos, neg, nneg, reg


def get_bboxes(pred_cls, pred_box, thr=0.8, cap=4096):
    """P-1.  (B,4,H,W), (B,14,H,W) -> boxes (B,cap,7), counts (B,) i32 (clamped), counts_raw (B,) i32."""
    lib = load()
    pred_cls = _contig(pred_cls, "pred_cls", torch.float32, 4)
    pred_box = _contig(pred_box, "pred_box", torch.float32, 4)
    B, c4, H, W = pred_cls.shape
    if c4 != 4 or tuple(pred_box.shape) != (B, 14, H, W):
        raise ValueError("get_bboxes: expected (B,4,H,W) and (B,14,H,W)")
    boxes = torch.zeros((B, cap, 7), dtype=torch.float32, device=pred_cls.device)
    counts = torch.empty((B,), dtype=torch.int32, device=pred_cls.device)
    raw = torch.empty((B,), dtype=torch.int32, device=pred_cls.device)
    check(lib.cf_get_bboxes(ptr(pred_cls), ptr(pred_box), B, H, W, float(thr), cap, ptr(boxes), ptr(counts), ptr(raw),
                            stream_ptr()), "cf_get_bboxes")
    return boxes, counts, raw


def _nms(fn_name, boxes, counts, extra=()):
    lib = load()
    boxes = _contig(boxes, "boxes", torch.float32, 3)
    counts = _contig(counts, "counts", torch.int32, 1)
    B, cap, seven = boxes.shape
    if seven != 7 or counts.shape[0] != B:
        raise ValueError("nms: expected boxes (B,cap,7) and counts (B,)")
    keep = torch.empty((B, cap), dtype=torch.int32, device=boxes.device)
    kcnt = torch.empty((B,), dtype=torch.int32, device=boxes.device)
    ws = torch.empty((max(lib.cf_nms_workspace_bytes(B, cap), 16),), dtype=torch.uint8, device=boxes.device)
    fn = getattr(lib, fn_name)
    check(fn(ptr(boxes), ptr(counts), B, cap, *extra, ptr(keep), ptr(kcnt), ptr(ws), stream_ptr()), fn_name)
    return keep, kcnt


def nms_sat(boxes, counts):
    """P-2..P-4.  boxes (B,cap,7), counts (B,) i32 -> keep_idx (B,cap) i32 (-1 padded), keep_count (B,) i32."""
    return _nms("cf_nms_sat", boxes, counts)


def nms_iou(boxes, counts, thr=0.01):
    """P-7."""
    return _nms("cf_nms_iou", boxes, counts, (float(thr),))


def sat_matrix(boxes):
    lib = load()
    boxes = _contig(boxes, "boxes", torch.float32, 2)
    n = boxes.shape[0]
    m = torch.empty((n, n), dtype=torch.uint8, device=boxes.device)
    check(lib.cf_sat_matrix(ptr(boxes), n, ptr(m), stream_ptr()), "cf_sat_matrix")
    return m


def box_iou(boxes_a, boxes_b, nudge_b=0.0):
    """P-5/P-6.  (na,7), (nb,7) -> iou3d, iou2d (na,nb) float64."""
    lib = load()
    boxes_a = _contig(boxes_a, "boxes_a", torch.float32, 2)
    boxes_b = _contig(boxes_b, "boxes_b", torch.float32, 2)
    na, nb = boxes_a.shape[0], boxes_b.shape[0]
    i3 = torch.empty((na, nb), dtype=torch.float64, device=boxes_a.device)
    i2 = torch.empty((na, nb), dtype=torch.float64, device=boxes_a.device)
    if na and nb:
        check(lib.cf_box_iou(ptr(boxes_a), na, ptr(boxes_b), nb, float(nudge_b), ptr(i3), ptr(i2), stream_ptr()),
              "cf_box_iou")
    return i3, i2


def debug_umma_gemm(A, Bm, split=False):
    """Self-test: D (128,N) = A (128,K) @ B (N,K)^T through the library's tcgen05 building blocks."""
    lib = load()
    A = _contig(A, "A", torch.float32, 2)
    Bm = _contig(Bm, "B", torch.float32, 2)
    if A.shape[0] != 128 or A.shape[1] != Bm.shape[1]:
        raise ValueError("debug_umma_gemm: A must be (128,K) and B (N,K)")
    D = torch.empty((128, Bm.shape[0]), dtype=torch.float32, device=A.device)
    check(lib.cf_debug_umma_gemm(ptr(A), ptr(Bm), Bm.shape[0], A.shape[1], int(bool(split)), ptr(D), stream_ptr()),
          "cf_debug_umma_gemm")
    return D


def debug_bwd_gemm_nn(X, Wm, transpose=False, epi=0, aux=None, out=None, row_count=None):
    """Self-test of the NN GEMM of the backward: epi(X @ B.T), B = Wm (N,Kd) or Wm.T with Wm (Kd,N)."""
    lib = load()
    X = _contig(X, "X", torch.float32, 2)
    Wm = _contig(Wm, "W", torch.float32, 2)
    R, Kd = X.shape
    N = Wm.shape[1] if transpose else Wm.shape[0]
    out = torch.zeros((R, N), dtype=torch.float32, device=X.device) if out is None else out
    packed = torch.empty((lib.cf_debug_bwd_packed_bytes(N, Kd),), dtype=torch.uint8, device=X.device)
    check(lib.cf_debug_bwd_gemm_nn(ptr(X), R, ptr(row_count), Kd, N, ptr(Wm), int(bool(transpose)), ptr(out), int(epi),
                                   ptr(aux), ptr(packed), stream_ptr()), "cf_debug_bwd_gemm_nn")
    return out


def debug_bwd_gemm_tn(X, Y=None, Y2=None, wcol=None, bias=False, row_count=None):
    """Self-test of the TN GEMM of the backward: (X.T @ [Y | Y2], X.T @ (wcol or 1))."""
    lib = load()
    X = _contig(X, "X", torch.float32, 2)
    R, M = X.shape
    N = 0 if Y is None else Y.shape[1]
    n2 = 0 if Y2 is None else Y2.shape[1]
    dW = torch.zeros((M, N + n2), dtype=torch.float32, device=X.device)
    db = torch.zeros((M,), dtype=torch.float32, device=X.device) if bias else None
    check(lib.cf_debug_bwd_gemm_tn(ptr(X), M, ptr(Y), N, ptr(Y2), n2, ptr(wcol), R, ptr(row_count), ptr(dW), ptr(db),
                                   stream_ptr()), "cf_debug_bwd_gemm_tn")
    return dW, db
