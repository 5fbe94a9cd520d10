"""GPU: the two tensor-core fused kernels, k_fusion_tc and k_fusion_sk, give the same bits.

At C = 128 in fp32 mode the library runs the double-buffered k_fusion_sk while its shared memory fits (K <= 14) and
k_fusion_tc from K = 15 on.  The same neighbour sets as a K = 3 table and padded to K = 16 with -1 therefore run the two
kernels on one problem: trailing -1 slots change neither a tile's round count nor any cell's neighbour count, so the
outputs must be equal bit for bit."""
import os
import subprocess
import sys

import pytest
import torch

from _util import dev

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BF = torch.bfloat16
_CACHE = {}


def _setup(dcf, size, C):
    """Inputs of one scale: "full" = the YAML grid's scale 1 at batch 2 (compacted cell lists), "small" = the tiny
    workload's scale 1 (not compacted)."""
    key = (size, C)
    if key not in _CACHE:
        base = dcf.synthetic.workload("yaml" if size == "full" else "tiny")
        wl = dcf.synthetic.make_workload(dict(base, batch=2, scales=(1,)), seed=60 + C, c_img=32, img_hw=(24, 32),
                                         channels=[C, 64, 128, 192, 256])
        sc = wl["scales"][0]
        frames = dcf.FrameContext(dev(wl["points"]), dev(wl["num_points"]),
                                  dcf.ops.BucketGrid(*dcf.geometry.bucket_grid(wl["config"])))
        frames.gather(dev(wl["img_feat"]), calib=wl["calib"])
        _CACHE[key] = (wl, sc, frames, [dev(x) for x in sc["weights"]])
    return _CACHE[key]


def _pad(knn, K):
    pad = torch.full(knn.shape[:3] + (K - knn.shape[3],), -1, dtype=knn.dtype, device=knn.device)
    return torch.cat([knn, pad], dim=3).contiguous()


@pytest.mark.parametrize("inplace", (False, True))
@pytest.mark.parametrize("map_dtype", (torch.float32, BF))
@pytest.mark.parametrize("size", ("full", "small"))
def test_sk_and_tc_kernels_give_the_same_bits(dcf, size, map_dtype, inplace):
    wl, sc, frames, w = _setup(dcf, size, 128)
    w1, b1, w2, b2, w3, b3 = w
    knn3 = frames.knn(sc["H"], sc["W"], sc["geom"], wl["radius"], 3)
    assert bool((knn3[..., 0] >= 0).any())
    knn16 = _pad(knn3, 16)
    T = dcf.ops.point_mlp1(frames.feat, frames.points, frames.num_points, w1, b1, mode="fp32")
    gen = torch.Generator(device="cuda").manual_seed(11)
    bev = (torch.randn((2, 128, sc["H"], sc["W"]), device="cuda", generator=gen) * 4).to(map_dtype)
    outs = []
    for knn in (knn3, knn16):
        io = bev.clone() if inplace else None
        outs.append(dcf.ops.fusion_fwd(bev if io is None else io, T, knn, sc["geom"], w1, w2, b2, w3, b3, mode="fp32",
                                       out=io)[0])
    assert outs[0].dtype == map_dtype
    assert not torch.equal(outs[0], bev)
    assert torch.equal(outs[0], outs[1])


_CHILD = r"""
import sys
import torch
sys.path.insert(0, sys.argv[1])
import dcf_b200 as dcf
B, N, H, W = 1, 512, 20, 24
for C in (96, 128):
    for K in (3, 16):
        g = torch.Generator(device="cuda").manual_seed(C + K)
        knn = torch.randint(0, N, (B, H, W, K), device="cuda", generator=g, dtype=torch.int32)
        knn[..., 3:] = -1
        T = torch.randn((B, N, C), device="cuda", generator=g)
        w1 = torch.randn((C, 35), device="cuda", generator=g)
        w2, w3 = torch.randn((C, C), device="cuda", generator=g), torch.randn((C, C), device="cuda", generator=g)
        b2, b3 = torch.randn((C,), device="cuda", generator=g), torch.randn((C,), device="cuda", generator=g)
        bev = torch.randn((B, C, H, W), device="cuda", generator=g)
        print(f"CASE C={C} K={K}", file=sys.stderr, flush=True)
        dcf.ops.fusion_fwd(bev, T, knn, (0.0, 0.0, 0.5, 0.5), w1, w2, b2, w3, b3, mode="fp32")
        torch.cuda.synchronize()
"""


def test_kernel_choice_follows_width_and_k():
    """C = 128 fp32: k_fusion_sk at K = 3, k_fusion_tc at K = 16 (the pairing above); C = 96: k_fusion_sk at both."""
    env = dict(os.environ, CF_DEBUG_LAUNCH="1")   # read once per process
    res = subprocess.run([sys.executable, "-c", _CHILD, ROOT], env=env, capture_output=True, text=True, timeout=600)
    assert res.returncode == 0, res.stderr[-3000:]
    launched, case = {}, None
    for line in res.stderr.splitlines():
        if line.startswith("CASE "):
            case = line[5:]
        elif line.startswith("k_fusion_"):
            launched[case] = line.split(":")[0]
    assert launched == {"C=96 K=3": "k_fusion_sk<96,2>", "C=96 K=16": "k_fusion_sk<96,2>",
                        "C=128 K=3": "k_fusion_sk<128,2>", "C=128 K=16": "k_fusion_tc<128,2>"}, res.stderr[-3000:]
