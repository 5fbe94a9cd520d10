"""Drop-in `ObjectDetection_DCF(config)` (model.py:176-204 of the reference) with the continuous-fusion
layer filled in.

Boundary contract (SURVEY 8b):
  * same constructor, `.cuda()`, DDP-wrappable; `forward(x_lidar, x_image)` still returns the
    (B, 4+14+14, H/4, W/4) tensor that train.py:32 / test.py:79 split, and with no extra inputs the
    computation is the reference's LiDAR-only path;
  * `state_dict` keys of the reference's modules are unchanged (`lidar_backbone.backbone.layerN.sequential.
    resblock_i.*`, `lidar_backbone.latconv1.weight`, ...), the camera stream and fusion MLPs only ADD keys,
    so checkpoints written by train.py:79 load with strict=False;
  * the three dataset tensors the reference already produces but never forwards
    (data_import_carla.py:67-82) are optional keyword inputs:
        forward(x_lidar, x_image, pointcloud_raw=None, num_points_raw=None, projected_loc_uv=None).

The BEV backbone / heads are ordinary PyTorch (cuDNN) modules -- they are outside the hot path -- written
here only so that the module tree and parameter names match.
"""
from __future__ import annotations

import numpy as np
import torch
import torch.nn as nn
import torch.nn.functional as F

from . import geometry as G
from . import ops
from .fusion import ContinuousFusion, FrameContext


def _conv(cin, cout, k, stride=1):
    return nn.Conv2d(cin, cout, kernel_size=(k, k), stride=(stride, stride), padding=(k // 2, k // 2), bias=False)


_INTERP_MATS = {}   # (n_in, n_out, align_corners, device, dtype) -> (n_out, n_in) interpolation matrix


def _interp_matrix(n_in, n_out, align_corners, device, dtype):
    """The (n_out, n_in) matrix of 1-D linear interpolation along one axis of F.interpolate(mode="bilinear"), built once
    per shape and device (a CUDA-graph capture of the step finds it cached from the eager warm-up)."""
    key = (int(n_in), int(n_out), bool(align_corners), device, dtype)
    m = _INTERP_MATS.get(key)
    if m is None:
        # the weights in fp32, as PyTorch's kernels compute them (scale, source coordinate, fraction)
        f = np.float32
        dst = np.arange(n_out, dtype=f)
        if align_corners:
            src = dst * (f(n_in - 1) / f(n_out - 1) if n_out > 1 else f(0))
        else:
            src = np.maximum((dst + f(0.5)) * (f(n_in) / f(n_out)) - f(0.5), f(0))
        i0 = np.minimum(src.astype(np.int64), n_in - 1)
        i1 = np.minimum(i0 + 1, n_in - 1)
        l1 = (src - i0.astype(f)).astype(f)
        a = np.zeros((n_out, n_in), np.float64)
        np.add.at(a, (np.arange(n_out), i0), f(1) - l1)
        np.add.at(a, (np.arange(n_out), i1), l1)
        m = _INTERP_MATS[key] = torch.from_numpy(a).to(device=device, dtype=dtype)
    return m


class _BilinearDeterministic(torch.autograd.Function):
    """F.interpolate(mode="bilinear") whose backward is the separable adjoint  Ry^T g Rx  (two matmuls) instead of
    PyTorch's atomic scatter, which torch.use_deterministic_algorithms(True) rejects.  The forward is the same call."""

    @staticmethod
    def forward(ctx, x, size, scale_factor, align_corners):
        ctx.hw_in, ctx.align_corners = tuple(x.shape[-2:]), align_corners
        return F.interpolate(x, size, scale_factor, "bilinear", align_corners)

    @staticmethod
    def backward(ctx, g):
        (hi, wi), (ho, wo) = ctx.hw_in, g.shape[-2:]
        ry = _interp_matrix(hi, ho, ctx.align_corners, g.device, g.dtype)
        rx = _interp_matrix(wi, wo, ctx.align_corners, g.device, g.dtype)
        return ry.t() @ (g @ rx), None, None, None


def bilinear(x, size=None, scale_factor=None, align_corners=False):
    """F.interpolate(x, size, scale_factor, mode="bilinear", align_corners).  Under torch.use_deterministic_algorithms(True)
    the backward is a fixed-order pair of matmuls (on CUDA these need CUBLAS_WORKSPACE_CONFIG=:4096:8, as PyTorch itself
    requires for cuBLAS in that mode); otherwise it is exactly the PyTorch call."""
    if torch.are_deterministic_algorithms_enabled():
        return _BilinearDeterministic.apply(x, size, scale_factor, align_corners)
    return F.interpolate(x, size, scale_factor, "bilinear", align_corners)


def _upsample(module: nn.UpsamplingBilinear2d, x):
    """`module(x)`, routed through `bilinear` in deterministic mode (same forward, fixed-order backward)."""
    if torch.are_deterministic_algorithms_enabled():
        return _BilinearDeterministic.apply(x, module.size, module.scale_factor, module.align_corners)
    return module(x)


class ResidualBlock(nn.Module):
    """3x3-3x3 residual block; a channel change implies stride 2 and a 1x1 projection shortcut (model.py:10-45)."""

    def __init__(self, in_channels, out_channels):
        super().__init__()
        self.in_channels, self.out_channels = in_channels, out_channels
        down = in_channels != out_channels
        self.conv1 = _conv(in_channels, out_channels, 3, 2 if down else 1)
        self.bn1 = nn.BatchNorm2d(out_channels)
        self.relu1 = nn.ReLU(inplace=True)
        self.conv2 = _conv(out_channels, out_channels, 3)
        self.bn2 = nn.BatchNorm2d(out_channels)
        self.relu2 = nn.ReLU(inplace=True)
        if down:
            self.down_conv = nn.Conv2d(in_channels, out_channels, kernel_size=(1, 1), stride=(2, 2), bias=False)
            self.down_bn = nn.BatchNorm2d(out_channels)

    @property
    def should_apply_shortcut(self):
        return self.in_channels != self.out_channels

    def forward(self, x):
        skip = self.down_bn(self.down_conv(x)) if self.should_apply_shortcut else x
        y = self.bn2(self.conv2(self.relu1(self.bn1(self.conv1(x)))))
        return self.relu2(y + skip)


class ResidualBlockModule(nn.Module):
    def __init__(self, first_in_channel, last_out_channel, num_resblock):
        super().__init__()
        self.sequential = nn.Sequential()
        for i in range(num_resblock):
            cin = first_in_channel if i == 0 else last_out_channel
            self.sequential.add_module(f"resblock_{i}", ResidualBlock(cin, last_out_channel))

    def forward(self, x):
        return self.sequential(x)


class ResnetCustomed(nn.Module):
    """Five residual groups (model.py:64-79).  `fuse(group, x)` is applied after each group (Appendix A11)."""

    def __init__(self, out_feature=(32, 64, 128, 192, 256), num_res_block=(1, 2, 4, 6, 6)):
        super().__init__()
        cin = out_feature[0]
        for g, (cout, n) in enumerate(zip(out_feature, num_res_block), start=1):
            setattr(self, f"layer{g}", ResidualBlockModule(cin, cout, n))
            cin = cout

    def forward(self, x, fuse=None):
        feats = []
        for g in range(1, 6):
            x = getattr(self, f"layer{g}")(x)
            if fuse is not None:
                x = fuse(g, x)
            feats.append(x)
        return feats[4], feats[3], feats[2]


class AnchorBoundingBoxFeature(nn.Module):
    """Two anchors per cell (yaw 0 and pi/2) on a linspace grid (model.py:82-113)."""

    def __init__(self, config):
        super().__init__()
        self.config = config
        a = config["anchor_bbox_feature"]
        self.f_height = int(config["voxel_length"] / a["reduced_scale"])
        self.f_width = int(config["voxel_width"] / a["reduced_scale"])
        self.width, self.length, self.height = a["width"], a["length"], a["height"]

    def forward(self):
        c, fh, fw = self.config, self.f_height, self.f_width
        ax = torch.linspace(c["lidar_x_min"], c["lidar_x_max"], fh).view(1, fh, 1).expand(1, fh, fw)
        ay = torch.linspace(c["lidar_y_min"], c["lidar_y_max"], fw).view(1, 1, fw).expand(1, fh, fw)
        one = torch.ones(1, fh, fw)
        base = [ax, ay, one * (-4.5), one * self.length, one * self.width, one * self.height]
        return torch.cat(base + [one * 0] + base + [one * 3.1415926 / 2], dim=0)


class OffsettoBbox(nn.Module):
    """Decode regression offsets against the anchors (model.py:116-137)."""

    def __init__(self, config):
        super().__init__()
        self.anchor_bbox_feature = AnchorBoundingBoxFeature(config)
        self._anchors = {}   # device -> (1,14,fh,fw): the anchors are constants of the config; the reference rebuilds
                             # them on the CPU and copies them every forward (model.py:125), which a CUDA-graph
                             # capture of the step cannot contain

    def forward(self, x):
        anc = self._anchors.get(x.device)
        if anc is None:
            anc = self._anchors[x.device] = self.anchor_bbox_feature().to(x.device).unsqueeze(0)
        outs = []
        for a in (0, 7):
            diag = torch.sqrt(anc[:, a + 3:a + 4] ** 2 + anc[:, a + 4:a + 5] ** 2)
            xy = x[:, a:a + 2] * diag + anc[:, a:a + 2]
            z = x[:, a + 2:a + 3] * anc[:, a + 5:a + 6] + anc[:, a + 2:a + 3]
            lwh = torch.exp(x[:, a + 3:a + 6]) * anc[:, a + 3:a + 6]
            ang = x[:, a + 6:a + 7] + anc[:, a + 6:a + 7]
            outs += [xy, z, lwh, torch.atan2(torch.sin(ang), torch.cos(ang))]
        return torch.cat(outs, dim=1)


class LidarBackboneNetwork(nn.Module):
    """BEV ResNet + FPN + heads (model.py:140-173)."""

    def __init__(self, out_feature=(32, 64, 128, 192, 256), num_res_block=(1, 2, 4, 6, 6), Num_anchor=2):
        super().__init__()
        self.backbone = ResnetCustomed(out_feature, num_res_block)
        self.num_anchor = Num_anchor
        c5, c4, c3 = out_feature[-1], out_feature[-2], out_feature[-3]
        self.latconv1 = _conv(c4, c4, 1)
        self.downconv1 = _conv(c5, c4, 1)
        self.upscale1 = nn.UpsamplingBilinear2d(scale_factor=2)
        self.latconv2 = _conv(c3, c4, 1)
        self.upscale2 = nn.UpsamplingBilinear2d(scale_factor=2)
        self.conv3 = _conv(c4, c4, 3)
        self.classconv = _conv(c4, Num_anchor * 2, 1)
        self.softmax1 = nn.Softmax(dim=1)
        self.softmax2 = nn.Softmax(dim=1)
        self.bbox3dconv = _conv(c4, Num_anchor * 7, 1)

    def forward(self, x, fuse=None):
        x4, x3, x2 = self.backbone(x, fuse)
        x3 = self.latconv1(x3) + _upsample(self.upscale1, self.downconv1(x4))
        x2 = self.latconv2(x2) + _upsample(self.upscale2, x3)
        x_pred = self.conv3(x2)
        x_cls = self.classconv(x_pred)
        x_cls = torch.cat((self.softmax1(x_cls[:, :2]), self.softmax2(x_cls[:, 2:4])), dim=1)
        return x_cls, self.bbox3dconv(x_pred)


class ImageBackbone(nn.Module):
    """Camera stream: a ResNet-18-shaped trunk whose stride-4/8/16 maps are merged top-down into ONE
    (B, c_img, H/4, W/4) map (the "multi-scale fusion" box of the paper's figure; the reference only has
    the commented-out `models.resnet18` at model.py:192).  Emits channels_last so that the gather kernel
    reads pixel-major rows without a re-layout pass."""

    def __init__(self, c_img=128):
        super().__init__()

        def stage(cin, cout, stride):
            return nn.Sequential(_conv(cin, cout, 3, stride), nn.BatchNorm2d(cout), nn.ReLU(inplace=True),
                                 _conv(cout, cout, 3), nn.BatchNorm2d(cout), nn.ReLU(inplace=True))

        self.stem = nn.Sequential(nn.Conv2d(3, 64, 7, 2, 3, bias=False), nn.BatchNorm2d(64), nn.ReLU(inplace=True),
                                  nn.MaxPool2d(3, 2, 1))
        self.stage1, self.stage2, self.stage3 = stage(64, 64, 1), stage(64, 128, 2), stage(128, 256, 2)
        self.lat1, self.lat2, self.lat3 = _conv(64, c_img, 1), _conv(128, c_img, 1), _conv(256, c_img, 1)
        self.out = _conv(c_img, c_img, 3)

    def forward(self, image):
        x = image.float() / 255.0 if image.dtype == torch.uint8 else image
        f1 = self.stage1(self.stem(x))
        f2 = self.stage2(f1)
        f3 = self.stage3(f2)
        t = self.lat2(f2) + bilinear(self.lat3(f3), size=f2.shape[-2:], align_corners=False)
        t = self.lat1(f1) + bilinear(t, size=f1.shape[-2:], align_corners=False)
        return self.out(t).contiguous(memory_format=torch.channels_last)


class ObjectDetection_DCF(nn.Module):
    def __init__(self, config):
        super().__init__()
        self.config = config
        self.offset_to_bbox = OffsettoBbox(config)
        lm = config["lidar_module"]
        feats = tuple(lm[f"out_feature{i}"] for i in range(1, 6))
        blocks = tuple(lm[f"num_res_block{i}"] for i in range(1, 6))
        self.lidar_backbone = LidarBackboneNetwork(feats, blocks)
        # ---- additive: camera stream + continuous fusion (SURVEY Appendix A) ----
        self.fusion_scales = tuple(int(s) for s in G.fusion_option(config, "fusion_scales"))
        c_img = int(G.fusion_option(config, "fusion_image_channels"))
        self.image_backbone = ImageBackbone(c_img)
        self.fusion = nn.ModuleDict()
        for g in self.fusion_scales:
            self.fusion[f"group{g}"] = ContinuousFusion(c_img, feats[g - 1], k=int(G.fusion_option(config, "fusion_k")),
                                                        radius=float(G.fusion_option(config, "fusion_radius")),
                                                        geom=G.scale_geometry(config, 2 ** (g - 1)),
                                                        mode=str(G.fusion_option(config, "fusion_mlp_mode")))
        self._grid = ops.BucketGrid(*G.bucket_grid(config))
        self.register_buffer("calib", torch.from_numpy(G.calibration_crt()), persistent=False)
        # optional camera rig (additive key): M reference cameras turned about the LiDAR z axis, one shared camera stream
        yaws = G.fusion_option(config, "fusion_camera_yaws")
        self.cameras = None if yaws is None else len(yaws)
        if yaws is not None:
            # per-camera image sizes (additive key): each camera's intrinsics are scaled to its own image
            sizes = G.fusion_option(config, "fusion_camera_image_sizes")
            if sizes is not None and len(sizes) != len(yaws):
                raise ValueError(f"fusion_camera_image_sizes: {len(sizes)} sizes for {len(yaws)} cameras")
            self.camera_sizes = ([(float(config["image_width"]), float(config["image_height"]))] * len(yaws) if sizes is None
                                 else [(float(w), float(h)) for w, h in sizes])
            self.register_buffer("rig_calib", torch.from_numpy(G.camera_rig(yaws, sizes)), persistent=False)

    def _camera_stream(self, x_image):
        """Camera maps of a rig.  (B,M,3,H,W): the one camera stream runs on all B*M images and its channels_last output is
        viewed as (B,M,Ci,Hf,Wf).  A list of M (B,3,H_m,W_m) images: the stream runs once per distinct image size, on the
        cameras of that size batched together, and gives the list of M maps (one size: the (B,M,3,H,W) call)."""
        if isinstance(x_image, torch.Tensor):
            return self.image_backbone(x_image.flatten(0, 1)).unflatten(0, tuple(x_image.shape[:2]))
        groups = {}
        for m, x in enumerate(x_image):
            groups.setdefault(tuple(x.shape[-2:]), []).append(m)
        if len(groups) == 1:
            return self._camera_stream(torch.stack(list(x_image), 1))
        maps = [None] * len(x_image)
        for ms in groups.values():
            f = self.image_backbone(torch.stack([x_image[m] for m in ms], 1).flatten(0, 1)).unflatten(0, (-1, len(ms)))
            for j, m in enumerate(ms):
                maps[m] = f[:, j]
        return maps

    def forward(self, x_lidar, x_image, pointcloud_raw=None, num_points_raw=None, projected_loc_uv=None, camera_calib=None):
        """With `fusion_camera_yaws` in the config, x_image is (B,M,3,H,W) (one image per camera) or a list of M (B,3,H_m,W_m)
        images (cameras of different image sizes, `fusion_camera_image_sizes`), and `camera_calib` (B,M,4,3) float32,
        w > 0 in front (geometry.camera_rig), optionally replaces the rig built from the yaws."""
        fuse = None
        if self.cameras is None and camera_calib is not None:
            raise ValueError("camera_calib needs a camera rig (config key fusion_camera_yaws)")
        if self.cameras is not None and pointcloud_raw is not None:
            if projected_loc_uv is not None:
                raise ValueError("projected_loc_uv cannot be used with a camera rig (fusion_camera_yaws): the rig projects "
                                 "every point on the device")
            if isinstance(x_image, (list, tuple)):
                if len(x_image) != self.cameras or any(not isinstance(x, torch.Tensor) or x.dim() != 4 for x in x_image):
                    raise ValueError(f"x_image: expected {self.cameras} (B,3,H_m,W_m) images for the {self.cameras}-camera "
                                     f"rig, got {len(x_image)} entries")
            elif x_image.dim() != 5 or x_image.shape[1] != self.cameras:
                raise ValueError(f"x_image: expected (B,{self.cameras},3,H,W) for the {self.cameras}-camera rig, got "
                                 f"{tuple(x_image.shape)}")
        if pointcloud_raw is not None:
            if num_points_raw is None:
                raise ValueError("num_points_raw is required with pointcloud_raw")
            # K-1 (point bucketing) is launched first, on its side stream: it runs under the camera trunk
            frames = FrameContext(pointcloud_raw.to(x_lidar.device), num_points_raw, self._grid)
            img_feat = self.image_backbone(x_image) if self.cameras is None else self._camera_stream(x_image)
            size = (float(self.config["image_width"]), float(self.config["image_height"]))
            if self.cameras is not None:
                if isinstance(img_feat, torch.Tensor) and len(set(self.camera_sizes)) > 1:
                    raise ValueError("x_image: the cameras of fusion_camera_image_sizes differ in size; pass a list of "
                                     "M (B,3,H_m,W_m) images")
                frames.gather(img_feat, calib=self.rig_calib if camera_calib is None else camera_calib,
                              img_size=self.camera_sizes if isinstance(img_feat, list) else self.camera_sizes[0])
            elif projected_loc_uv is not None:
                frames.gather(img_feat, uv=projected_loc_uv.to(x_lidar.device), img_size=size)
            else:
                frames.gather(img_feat, calib=self.calib, img_size=size)

            # K-4a of every scale in one launch, on a side stream (training too: the tables are intermediates of each
            # layer's autograd Function, not autograd leaves)
            frames.precompute([self.fusion[f"group{g}"] for g in self.fusion_scales])

            inplace = not torch.is_grad_enabled()   # inference: the group's output map is fused in place (no copy of the
                                                    # ~2/3 of the cells that have no LiDAR point in reach)

            def fuse(group, x):
                key = f"group{group}"
                if key not in self.fusion:
                    return x
                dense = x.is_contiguous() or x.is_contiguous(memory_format=torch.channels_last)   # NCHW or NHWC kernels
                return self.fusion[key](x, frames=frames, out=x if inplace and dense else None)

        cls, reg = self.lidar_backbone(x_lidar, fuse)
        return torch.cat((cls, reg, self.offset_to_bbox(reg)), dim=1)
