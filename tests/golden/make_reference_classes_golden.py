#!/usr/bin/env python
"""Generates tests/golden/reference_classes.json with two of the REFERENCE's own Python classes, unmodified, run here on CPU:

  replay_buffer     Modules.ReplayBuffer(size, simple=True) (Modules.py:28-55) driven the agent's way (tests/test_replay_buffer.py
                    `_drive`): every sampled batch, as the pushed step indices, for three (size, batch, pushes) settings.
  grasping_dataset  `Offline RL/grasping_dataset.py` Grasping_Dataset on a file written by mujoco_rl_ur5_b200.offline_data
                    (tests/test_offline_data.py `_batch(3, seed=5)`): length, item 1's action, reward and shape, and its depth
                    channel (np.random.seed(0) before the item) at 256 fixed pixels.  The RGB channels go through an unseeded
                    ColorJitter and are not recorded.

`prettytable` is stubbed for Modules.py and `Modules` for grasping_dataset.py; nothing else is touched.
Run:  python tests/golden/make_reference_classes_golden.py [reference dir]"""
import importlib.util
import json
import os
import sys
import tempfile
import types
from collections import namedtuple

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))
from mujoco_rl_ur5_b200 import offline_data as od  # noqa: E402
from tests.test_offline_data import _batch  # noqa: E402
from tests.test_replay_buffer import REPLAY_SETTINGS, _drive  # noqa: E402

REF = sys.argv[1] if len(sys.argv) > 1 else os.environ["GRASP_REFERENCE_DIR"]


def _load(name, path):
    spec = importlib.util.spec_from_file_location(name, path)
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


sys.modules["prettytable"] = types.SimpleNamespace(PrettyTable=object)
modules = _load("ref_modules", os.path.join(REF, "Modules.py"))
replay = []
for size, B, n in REPLAY_SETTINGS:
    rb = modules.ReplayBuffer(size, simple=True)  # seeds the global `random` with 20
    replay.append(_drive(lambda k: rb.push(torch.full((1, 1, 2, 2), float(k)), torch.tensor([[k * 3]]), torch.tensor([[k % 2]])),
                         lambda B_: [int(t.state[0, 0, 0, 0]) for t in rb.sample(B_)], lambda: len(rb), n, size, B))

sys.modules["Modules"] = types.SimpleNamespace(simple_Transition=namedtuple("simple_Transition", ("state", "action", "reward")))
dataset = _load("ref_grasping_dataset", os.path.join(REF, "Offline RL", "grasping_dataset.py"))
rgb, depth, act, rew = _batch(3, seed=5)
with tempfile.TemporaryDirectory() as d:
    p = os.path.join(d, "grasping_data_1.pt")
    od.save_transitions(p, rgb, depth, od.flat_action(act), rew)
    _orig = torch.load
    torch.load = lambda f, *a, **k: _orig(f, *a, **{**k, "weights_only": False})  # the reference predates the weights_only default
    ds = dataset.Grasping_Dataset(p)
    torch.load = _orig
    np.random.seed(0)
    state, a, r = ds[1]
pix = np.random.RandomState(7).choice(200 * 200, 256, replace=False)
item = dict(length=len(ds), shape=list(state.shape), action=int(a), reward=int(r), pixels=pix.tolist(),
            depth=[float(v) for v in state[3].reshape(-1)[pix]])

path = os.path.join(HERE, "reference_classes.json")
json.dump(dict(replay_buffer=dict(settings=REPLAY_SETTINGS, samples=replay), grasping_dataset=item), open(path, "w"), separators=(",", ":"))
print("wrote", path, "replay batches", [len(s) for s in replay], "dataset item", item["shape"], item["action"], item["reward"])
