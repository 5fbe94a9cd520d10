"""bench.py contract, CPU side: the reference arm (the CPU port, rank 0 only) prints ONE JSON line whose `config` equals what
the GPU arm prints for the same workload, whose `steps` are the whole frames it really timed, and which carries the keys the
driver reads; `--workload train --impl reference` reports that there is nothing to run."""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _run(*args, env=None):
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *args], capture_output=True, text=True, timeout=600,
                       env=dict(os.environ, **(env or {})))
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [l for l in r.stdout.splitlines() if l.startswith("{")]
    return [json.loads(l) for l in lines]


def test_reference_arm_line():
    lines = _run("--impl", "reference", "--workload", "tiny", "--steps", "3", "--warmup", "1")
    assert len(lines) == 1
    l = lines[0]
    assert l["impl"] == "reference" and l["metric"] == "fusion_layer_frames_per_sec" and l["unit"] == "frames/s"
    assert l["higher_is_better"] is True and l["vs_baseline"] is None
    assert l["steps"] == 3 and l["steps_requested"] == 3 and l["warmup"] == 1
    # steps x ms_per_step is CPU time that was really spent: value = frames / that time, one step = one whole frame
    assert abs(l["value"] - 1e3 / l["ms_per_step"]) <= 1e-2 * l["value"]
    assert l["cpu_baseline"]["kind"] == "port" and l["cpu_baseline"]["cores"] >= 1 and "nothing extrapolated" in l["cpu_baseline"]["sample"]
    assert l["e2e"] == {"value": l["value"], "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    # the identical config dict in both arms: only the workload label (arm-specific settings live under "run")
    sys.path.insert(0, ROOT)
    import bench
    import dcf_b200 as dcf
    wl = dcf.synthetic.make_workload("tiny", seed=100)
    assert l["config"] == {"workload": bench.workload_label("tiny", wl)}


def test_reference_arm_is_silent_on_other_ranks():
    assert _run("--impl", "reference", "--workload", "tiny", "--steps", "1", "--warmup", "0", env={"RANK": "1", "WORLD_SIZE": "2"}) == []


def test_train_workload_has_no_reference():
    lines = _run("--workload", "train", "--impl", "reference")
    assert len(lines) == 1 and lines[0]["impl"] == "reference" and "unavailable" in lines[0]


def test_dump_outputs_keeps_small_maps_whole_and_samples_large_ones(tmp_path):
    """--dump-outputs: float32 files within the budget; a tensor over its share of the budget is saved at the same seeded
    positions on every run, so that two builds are compared value for value."""
    import numpy as np
    import torch
    sys.path.insert(0, ROOT)
    import bench
    small = torch.arange(12, dtype=torch.float64).reshape(3, 4)
    big = torch.randn(2, 500, generator=torch.Generator().manual_seed(1))
    budget = 2 * 100 * 4                                                   # 100 float32 values per tensor
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), [("small", small), ("big", big)], budget=budget)
    a_small, a_big = np.load(tmp_path / "a" / "small.npy"), np.load(tmp_path / "a" / "big.npy")
    assert a_small.dtype == a_big.dtype == np.float32
    assert np.array_equal(a_small, small.float().numpy())
    idx = bench.sample_indices(1000, 100)
    assert idx.shape == (100,) and np.unique(idx).size == 100 and (np.diff(idx) > 0).all() and idx[-1] < 1000
    assert np.array_equal(a_big, big.numpy().reshape(-1)[idx])
    assert a_small.nbytes + a_big.nbytes <= budget
    assert np.array_equal(np.load(tmp_path / "b" / "big.npy"), a_big)
    # the full-size workload: five maps of up to 287 MB fit the 64 MB the option promises, .npy headers included
    assert bench.DUMP_BUDGET_BYTES + 5 * 128 <= 64e6
    idx = bench.sample_indices(71_680_000, 3_145_728)                      # scale 1 of configs[1]
    assert (np.diff(idx) > 0).all() and idx[0] >= 0 and idx[-1] < 71_680_000 and idx[-1] > 71_000_000


def test_dump_outputs_is_refused_where_it_cannot_be_honoured(tmp_path):
    """The reference arm and the train workload compute no fused maps, and zero timed steps have no last step: asking for
    a dump there is an error, not a run that silently writes nothing."""
    for args in (["--impl", "reference", "--workload", "tiny"], ["--workload", "train"], ["--steps", "0"]):
        r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *args, "--dump-outputs", str(tmp_path / "d")],
                           capture_output=True, text=True, timeout=120)
        assert r.returncode == 2 and "--dump-outputs" in r.stderr, (args, r.stderr[-500:])
        assert not (tmp_path / "d").exists()
