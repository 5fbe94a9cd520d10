"""Import the UNMODIFIED reference from the directory named by the environment variable CF_REFERENCE_DIR
(a checkout of the original project; it is not part of this repository).

TEST INFRASTRUCTURE ONLY.  Nothing on the product path (``-m gpu`` tests, smoke(), bench.py) imports
this module; it is used by oracle/gen_golden.py (fixture generation) and by two CPU tests that skip
when the reference is not available.  The fixtures it produced are stored under tests/golden/.

Shims (harness-side only, the reference files are never edited or copied):
  * empty stand-ins for matplotlib / h5py / numpy-quaternion, which the container lacks and which
    the post-process functions never touch (test.py:13-15, data_import_carla.py:3,9);
  * ``IOU.min/IOU.max = builtins.min/max``: ``from numpy import *`` (IOU.py:6) shadows the
    built-ins under numpy >= 2 and ``min(a, b)`` at IOU.py:112-113 would raise TypeError.
"""
from __future__ import annotations

import builtins
import importlib
import os
import sys
import types

REFERENCE_DIR = os.environ.get("CF_REFERENCE_DIR", "")


def available() -> bool:
    return bool(REFERENCE_DIR) and os.path.isfile(os.path.join(REFERENCE_DIR, "separation_axis_theorem.py"))


_loaded = {}


def load():
    """Returns a namespace with the reference modules: test, IOU, sat, data_import_carla, model."""
    if _loaded:
        return types.SimpleNamespace(**_loaded)
    if not available():
        raise RuntimeError("reference tree not present: set CF_REFERENCE_DIR to a checkout of the original project")
    for name in ("matplotlib", "matplotlib.pyplot", "h5py", "quaternion"):
        if name not in sys.modules:
            sys.modules[name] = types.ModuleType(name)
    sys.modules["matplotlib"].use = lambda *a, **k: None
    sys.modules["matplotlib"].pyplot = sys.modules["matplotlib.pyplot"]
    saved_test = sys.modules.pop("test", None)
    sys.path.insert(0, REFERENCE_DIR)
    try:
        _loaded["sat"] = importlib.import_module("separation_axis_theorem")
        iou = importlib.import_module("IOU")
        iou.min, iou.max = builtins.min, builtins.max
        _loaded["IOU"] = iou
        _loaded["test"] = importlib.import_module("test")  # the reference's test.py, not the stdlib package
        _loaded["data_import_carla"] = importlib.import_module("data_import_carla")
        _loaded["model"] = importlib.import_module("model")
    finally:
        sys.path.remove(REFERENCE_DIR)
        if saved_test is not None:
            sys.modules["test"] = saved_test
    return types.SimpleNamespace(**_loaded)


def nms_sat(boxes_list):
    """Test.NMS_SAT (test.py:142-175) on a list of (n,7) float32 torch tensors -> list of index arrays.

    The reference returns the kept *rows*; indices are recovered by identity of the row objects'
    storage offsets (each kept entry is pred_bboxes[b][i], a view at offset 7*i)."""
    import numpy as np
    ref = load()
    out = ref.test.Test.NMS_SAT(None, boxes_list)
    res = []
    for kept in out:
        res.append(np.array([k.storage_offset() // 7 for k in kept], dtype=np.int32))
    return res


def nms_iou(boxes_list, thr=0.01):
    import contextlib
    import io
    import numpy as np
    ref = load()
    with contextlib.redirect_stdout(io.StringIO()):  # test.py:116 prints
        out = ref.test.Test.NMS_IOU(None, boxes_list, thr)
    return [np.array([k.storage_offset() // 7 for k in kept], dtype=np.int32) for kept in out]


def get_bboxes(pred_cls, pred_box, thr=0.8):
    ref = load()
    return ref.test.Test.get_bboxes(None, pred_cls, pred_box, thr)


def carla_dataset_stub(config):
    """A CarlaDataset instance without HDF5 / quaternion: enough state for Projection and
    Voxelization_Projection (data_import_carla.py:196-267) to run on synthetic points."""
    import numpy as np
    import torch
    ref = load()
    ds = object.__new__(ref.data_import_carla.CarlaDataset)
    ds.config = config
    # restate get_extrinsic_parameter (:180-188) without numpy-quaternion: from_euler_angles is the
    # Z-Y-Z convention R = Rz(alpha) Ry(beta) Rz(gamma)
    a, b, g = (np.array([-3.13498819, 1.59196951, 1.56942932]) - np.array([-1.57079633, 3.12042851, -1.57079633]))

    def rz(t):
        return np.array([[np.cos(t), -np.sin(t), 0], [np.sin(t), np.cos(t), 0], [0, 0, 1.0]])

    def ry(t):
        return np.array([[np.cos(t), 0, np.sin(t)], [0, 1.0, 0], [-np.sin(t), 0, np.cos(t)]])

    R = rz(a) @ ry(b) @ rz(g)
    RT = np.concatenate((R, np.zeros((3, 1))), axis=-1)
    Cm = ds.get_intrinsic_parameter()
    ds.CRT_tensor = torch.tensor(Cm @ RT).permute(1, 0).type(torch.float)
    x_scale = int(config["voxel_length"] / (config["lidar_x_max"] - config["lidar_x_min"]))
    y_scale = int(config["voxel_width"] / (config["lidar_y_max"] - config["lidar_y_min"]))
    z_scale = int(config["voxel_channel"] / (config["lidar_z_max"] - config["lidar_z_min"]))
    x_offset = int(-config["lidar_x_min"] * x_scale)
    y_offset = int(-config["lidar_y_min"] * y_scale)
    z_offset = int(-config["lidar_z_min"] * z_scale)
    ds.pc_to_voxel_indice = torch.tensor([[x_scale, 0, 0, x_offset], [0, y_scale, 0, y_offset],
                                          [0, 0, z_scale, z_offset]], dtype=torch.float).permute(1, 0)
    return ds


def loss_total(config, ref_boxes, num_ref, pred_cls, pred_reg, keys, cand):
    """The reference's LossTotal (loss.py:33-189), UNMODIFIED, run on the CPU for every frame of the batch with the random
    draws of the RNG contract (oracle.loss_targets).  Harness-side stubs only: torchvision (loss.py:3 imports save_image
    for a __main__ block), Tensor.cuda -> identity (loss.py:40,51 call .cuda() unconditionally; the container has no GPU),
    np.random.shuffle / randint -> the supplied draws.  loss.py:71 keeps only the LAST frame of a batch, so frame b's value
    is obtained by calling the reference on the batch cut after frame b.
    Returns (losses (B,), positives per frame, negatives per frame) -- the lists are the reference's own, captured from
    getPositionOfPositive / getPositionOfNegative."""
    import contextlib
    import numpy as np
    import torch
    load()
    for name in ("torchvision", "torchvision.utils"):
        if name not in sys.modules:
            sys.modules[name] = types.ModuleType(name)
    sys.modules["torchvision.utils"].save_image = lambda *a, **k: None
    sys.modules["torchvision"].utils = sys.modules["torchvision.utils"]
    saved_cuda = torch.Tensor.cuda
    torch.Tensor.cuda = lambda self, *a, **k: self
    sys.path.insert(0, REFERENCE_DIR)
    try:
        loss_mod = importlib.import_module("loss")
        state = {"frame": -1, "c": 0}
        W = pred_cls.shape[3]

        def shuffle(lst):
            state["frame"] += 1
            state["c"] = 0
            order = np.argsort(np.asarray(keys[state["frame"]][:len(lst)], dtype=np.float32), kind="stable")
            lst[:] = [lst[j] for j in order]

        def randint(n):
            b, c = state["frame"], state["c"]
            state["c"] += 1
            return int(cand[b][c // 2][c % 2])

        captured = {"pos": [], "neg": []}
        LT = loss_mod.LossTotal
        orig_pos, orig_neg = LT.getPositionOfPositive, LT.getPositionOfNegative

        def cap_pos(self, *a, **k):
            r = orig_pos(self, *a, **k)
            captured["pos"].append([p[0] * W + p[1] for p in r[2]])
            return r

        def cap_neg(self, *a, **k):
            r = orig_neg(self, *a, **k)
            captured["neg"].append([p[0] * W + p[1] for p in r])
            return r

        saved = np.random.shuffle, np.random.randint
        np.random.shuffle, np.random.randint = shuffle, randint
        LT.getPositionOfPositive, LT.getPositionOfNegative = cap_pos, cap_neg
        try:
            lt = LT(config)
            B = ref_boxes.shape[0]
            losses, pos, neg = [], [], []
            with torch.no_grad():
                for b in range(B):
                    state["frame"] = -1
                    captured["pos"].clear()
                    captured["neg"].clear()
                    v = lt(torch.as_tensor(ref_boxes[:b + 1]), torch.as_tensor(num_ref[:b + 1]), torch.as_tensor(pred_cls[:b + 1]),
                           torch.as_tensor(pred_reg[:b + 1]))
                    losses.append(float(v))
                    pos.append(list(captured["pos"][-1]))
                    neg.append(list(captured["neg"][-1]))
        finally:
            np.random.shuffle, np.random.randint = saved
            LT.getPositionOfPositive, LT.getPositionOfNegative = orig_pos, orig_neg
    finally:
        torch.Tensor.cuda = saved_cuda
        sys.path.remove(REFERENCE_DIR)
    return np.asarray(losses), pos, neg
