"""GPU: `bench.py --dump-outputs` saves what the timed path computed -- the fused BEV maps of the last timed step, equal to
the CPU oracle on the same seeded inputs -- with the CUDA-graph replay and with eager launches, and the JSON line reports
the number of timed steps that was asked for."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

from _util import oracle_fusion, rel_err

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.mark.parametrize("graph", [True, False])
def test_dumped_outputs_are_the_fused_maps(dcf, oracle, tmp_path, graph):
    args = ["--workload", "tiny", "--steps", "3", "--warmup", "1", "--no-cpu-baseline", "--no-extras",
            "--dump-outputs", str(tmp_path)] + ([] if graph else ["--no-graph"])
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *args], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    line = json.loads([l for l in r.stdout.splitlines() if l.startswith("{")][-1])
    assert line["steps"] == 3 and line["run"]["launch"] == ("cuda_graph_replay" if graph else "eager")
    wl = dcf.synthetic.make_workload("tiny", seed=dcf.dist_util.rank_seed(100, 0))   # rank 0's frames in bench.py
    ref_outs, _ = oracle_fusion(oracle, wl)
    assert sorted(os.listdir(tmp_path)) == sorted(f"fused_g{sc['group']}.npy" for sc in wl["scales"])
    for sc, ro in zip(wl["scales"], ref_outs):
        o = np.load(tmp_path / f"fused_g{sc['group']}.npy")
        assert o.dtype == np.float32 and o.shape == ro.shape      # small maps are saved whole
        assert rel_err(o, ro) <= 1e-4, f"group {sc['group']}: rel err {rel_err(o, ro):.3e}"
        assert rel_err(o - sc["bev"], ro - sc["bev"]) <= 2e-4      # the fused term itself, not only the copied input
