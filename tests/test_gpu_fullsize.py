"""GPU: the BASELINE.json shapes at FULL size against the brute-force CPU oracle (VERDICT round 1, item 1).

configs[1]: whole 700x800 frames, K = 5, all five scales (700x800x32 ... 44x50x256): KNN indices bit-exact on EVERY
cell of every scale, fused features within 1e-4 (Appendix A13) in fp32 mode, out of place and in place -- this is
where the strip / tile sequencing, the cells without a neighbour and the multi-wave persistent grids engage.
configs[2]: one 64-beam frame (~110 k points), K = 10, bf16 MLP: KNN bit-exact on every cell, features within 1e-2.
The oracle is the naive formulation (brute-force KNN, per-neighbour three-layer MLP) on all host cores; a frame takes
a few seconds."""
import os

import numpy as np
import pytest

from _util import cuda_fusion, oracle_fusion, rel_err

pytestmark = pytest.mark.gpu


def _check(wl, outs, knns, ref_outs, ref_knns, tol, what):
    for sc, o, k, ro, rk in zip(wl["scales"], outs, knns, ref_outs, ref_knns):
        tag = f"{what} group {sc['group']} ({sc['C']}x{sc['H']}x{sc['W']})"
        assert k.shape == rk.shape and np.array_equal(k, rk), f"{tag}: KNN differs from brute force"
        assert o.shape == ro.shape and o.dtype == np.float32
        e = rel_err(o, ro)
        assert e <= tol, f"{tag}: rel err {e:.3e} > {tol}"
        d, rd = o - sc["bev"], ro - sc["bev"]
        assert np.abs(rd).max() > 1e-2
        e = rel_err(d, rd)
        assert e <= 2 * tol, f"{tag}: delta rel err {e:.3e} > {2 * tol}"
        empty = (rk < 0).all(-1)                       # (B,H,W): cells nothing reaches keep their bits
        for b in range(o.shape[0]):
            assert np.array_equal(o[b][:, empty[b]], sc["bev"][b][:, empty[b]]), f"{tag}: untouched cells changed"


def test_cfg1_full_frames_fp32(dcf, oracle):
    """BASELINE configs[1] at full size, two frames (ragged point counts), fp32 mode (split bf16 x 3 on tcgen05)."""
    oracle.set_threads(os.cpu_count() or 1)
    wl = dcf.synthetic.make_workload(dict(dcf.synthetic.workload("cfg1"), batch=2), seed=41)
    wl["num_points"][1] = int(wl["num_points"][1]) * 2 // 3       # ragged: frame 1 uses two thirds of its rows
    ref_outs, ref_knns = oracle_fusion(oracle, wl)
    outs, knns = cuda_fusion(dcf, wl, "fp32")
    _check(wl, outs, knns, ref_outs, ref_knns, 1e-4, "out of place")
    outs_ip, _ = cuda_fusion(dcf, wl, "fp32", inplace=True)
    for sc, a, b in zip(wl["scales"], outs, outs_ip):
        assert np.array_equal(a, b), f"group {sc['group']}: in place != out of place"


def test_cfg1_full_frame_bf16(dcf, oracle):
    oracle.set_threads(os.cpu_count() or 1)
    wl = dcf.synthetic.make_workload(dict(dcf.synthetic.workload("cfg1"), batch=1), seed=42)
    ref_outs, ref_knns = oracle_fusion(oracle, wl)
    outs, knns = cuda_fusion(dcf, wl, "bf16")
    _check(wl, outs, knns, ref_outs, ref_knns, 1e-2, "bf16")


def test_cfg2_full_frame_bf16(dcf, oracle):
    """BASELINE configs[2], one frame: ~110 k points, K = 10, bf16 MLP, all five scales, every cell."""
    oracle.set_threads(os.cpu_count() or 1)
    wl = dcf.synthetic.make_workload(dict(dcf.synthetic.workload("cfg2"), batch=1), seed=43)
    assert wl["k"] == 10 and int(wl["num_points"][0]) > 90000
    ref_outs, ref_knns = oracle_fusion(oracle, wl)
    outs, knns = cuda_fusion(dcf, wl, "bf16")
    _check(wl, outs, knns, ref_outs, ref_knns, 1e-2, "cfg2")
    # the same frame with the layer-1 tables stored as bf16 (CF_MODE_BF16_TABLES): same tolerance, out of place and in place
    outs_t, knns_t = cuda_fusion(dcf, wl, "bf16t")
    _check(wl, outs_t, knns_t, ref_outs, ref_knns, 1e-2, "cfg2 bf16 tables")
    outs_ti, _ = cuda_fusion(dcf, wl, "bf16t", inplace=True)
    for sc, x, y in zip(wl["scales"], outs_t, outs_ti):
        assert np.array_equal(x, y), f"group {sc['group']}: bf16 tables, in place != out of place"

