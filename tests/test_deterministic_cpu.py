"""CPU: the deterministic-mode pieces that do not need a GPU.  The camera trunk's and the FPN's bilinear resizes under
torch.use_deterministic_algorithms(True): the forward is the PyTorch call bit for bit, the backward (the separable
adjoint Ry^T g Rx) matches autograd through F.interpolate.  The C ABI and the host layer expose the deterministic backward."""
import os
import re

import pytest
import torch
import torch.nn as nn
import torch.nn.functional as F

import dcf_b200 as dcf

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture
def deterministic():
    before = torch.are_deterministic_algorithms_enabled()
    torch.use_deterministic_algorithms(True)
    yield
    torch.use_deterministic_algorithms(before)


@pytest.mark.parametrize("hw_in, hw_out", [((30, 40), (60, 80)), ((60, 80), (120, 160)), ((31, 41), (61, 81))])
def test_bilinear_helper_forward_and_adjoint(deterministic, hw_in, hw_out):
    gen = torch.Generator().manual_seed(3)
    x = torch.randn(2, 5, *hw_in, generator=gen)
    g = torch.randn(2, 5, *hw_out, generator=gen)
    ref_x = x.clone().requires_grad_(True)
    torch.use_deterministic_algorithms(False)     # the reference: PyTorch's own backward
    ref = F.interpolate(ref_x, size=hw_out, mode="bilinear", align_corners=False)
    ref.backward(g)
    torch.use_deterministic_algorithms(True)
    xx = x.clone().requires_grad_(True)
    out = dcf.model.bilinear(xx, size=hw_out, align_corners=False)
    assert out.grad_fn is not None and "Bilinear" in type(out.grad_fn).__name__   # the helper's own Function
    assert torch.equal(out, ref.detach())
    out.backward(g)
    err = (xx.grad - ref_x.grad).abs().max().item()
    assert err <= 1e-6 * max(ref_x.grad.abs().max().item(), 1.0), err


@pytest.mark.parametrize("hw_in", [(12, 8), (13, 9)])
def test_fpn_upsampling_adjoint(deterministic, hw_in):
    """nn.UpsamplingBilinear2d (align_corners=True) of the LiDAR FPN goes through the same Function."""
    up = nn.UpsamplingBilinear2d(scale_factor=2)
    gen = torch.Generator().manual_seed(4)
    x = torch.randn(1, 3, *hw_in, generator=gen)
    torch.use_deterministic_algorithms(False)
    ref_x = x.clone().requires_grad_(True)
    ref = up(ref_x)
    g = torch.randn(ref.shape, generator=gen)
    ref.backward(g)
    torch.use_deterministic_algorithms(True)
    xx = x.clone().requires_grad_(True)
    out = dcf.model._upsample(up, xx)
    assert torch.equal(out, ref.detach())
    out.backward(g)
    assert (xx.grad - ref_x.grad).abs().max().item() <= 1e-6 * max(ref_x.grad.abs().max().item(), 1.0)


def test_helper_is_the_plain_call_without_the_flag():
    assert not torch.are_deterministic_algorithms_enabled()
    x = torch.randn(1, 2, 7, 9, requires_grad=True)
    out = dcf.model.bilinear(x, size=(14, 18))
    assert "Deterministic" not in type(out.grad_fn).__name__      # PyTorch's own UpsampleBilinear2D backward
    assert torch.equal(out, F.interpolate(x, size=(14, 18), mode="bilinear", align_corners=False))


def test_state_dict_keys_unchanged_by_the_helper():
    cfg = dcf.geometry.carla_config(fusion_scales=(1, 2), fusion_k=3)
    keys = set(dcf.ObjectDetection_DCF(cfg).state_dict())
    assert not any("interp" in k or "bilinear" in k.lower() for k in keys)
    assert "image_backbone.out.weight" in keys and "lidar_backbone.latconv1.weight" in keys


def test_abi_declares_the_deterministic_entry_points():
    header = open(os.path.join(ROOT, "include", "cf_b200.h")).read()
    assert re.search(r"#define CF_BWD_DETERMINISTIC 0x100\b", header)
    assert re.search(r"#define CF_ABI_VERSION 2\b", header)
    for name in ("cf_fusion_bwd_det_workspace_bytes", "cf_point_gather_bwd_det_workspace_bytes", "cf_point_gather_bwd_det"):
        assert name in dcf._lib.SIGNATURES and name + "(" in header
    assert dcf._lib.BWD_DETERMINISTIC == 0x100


def test_host_layer_takes_the_flag():
    import inspect
    assert inspect.signature(dcf.ops.fusion_bwd).parameters["deterministic"].default is False
    assert inspect.signature(dcf.ops.point_gather_bwd).parameters["deterministic"].default is False
    src = inspect.getsource(dcf.fusion)
    assert src.count("deterministic=torch.are_deterministic_algorithms_enabled()") == 2
