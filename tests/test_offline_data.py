"""Offline-RL wire format (SURVEY 8f.3): files written from batched observations are what the reference's own loader
(`Offline RL/grasping_dataset.py`) and scripts (`generate_data.py`, `unite_data.py`, `extract_positives.py`) read and write."""
import json
import os
import sys

import numpy as np
import pytest

from mujoco_rl_ur5_b200 import offline_data as od

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference_classes.json")


def _batch(n, seed=0, H=200, W=200):
    rng = np.random.RandomState(seed)
    rgb = rng.randint(0, 256, (n, H, W, 3)).astype(np.uint8)
    depth = (1.0 + 0.2 * rng.rand(n, H, W)).astype(np.float32)
    act = np.stack([rng.randint(0, H * W, n), rng.randint(0, 6, n)], axis=1)
    rew = rng.randint(0, 2, n)
    return rgb, depth, act, rew


def test_flat_action_is_the_inverse_of_transform_action():
    # Grasp_Agent.transform_action (Grasping_Agent_multidiscrete.py:381-386): rot = a // (H*W), pixel = a % (H*W)
    a = np.array([[0, 0], [39999, 5], [12345, 3]])
    f = od.flat_action(a)
    assert f.tolist() == [0, 5 * 40000 + 39999, 3 * 40000 + 12345]
    assert (od.env_action(f) == a).all()


def test_round_trip_and_python_types(tmp_path):
    import torch

    rgb, depth, act, rew = _batch(7)
    p = str(tmp_path / "Data" / "grasping_data_1.pt")
    assert od.save_transitions(p, rgb, depth, od.flat_action(act), rew) == 7
    raw = torch.load(p, weights_only=False)
    assert set(raw.keys()) == {"states", "actions", "rewards"}
    assert isinstance(raw["states"], list) and isinstance(raw["actions"][0], int) and isinstance(raw["rewards"][0], int)
    s = raw["states"][3]
    assert s["rgb"].dtype == np.uint8 and s["rgb"].shape == (200, 200, 3) and s["depth"].dtype == np.float32 and s["depth"].shape == (200, 200)
    r2, d2, a2, w2 = od.load_transitions(p)
    assert (r2 == rgb).all() and (d2 == depth).all() and (a2 == od.flat_action(act)).all() and (w2 == rew).all()


def test_recorder_writes_files_of_twelve(tmp_path):
    rec = od.TransitionRecorder(str(tmp_path), file_size=12)
    allr, alla = [], []
    for k in range(5):
        rgb, depth, act, rew = _batch(5, seed=k, H=20, W=20)
        rec.W = rec.H = 20
        rec.add({"rgb": rgb, "depth": depth}, act, rew)
        allr.append(rew); alla.append(od.flat_action(act, 20, 20))
    files = rec.close()
    assert [os.path.basename(f) for f in files] == ["grasping_data_1.pt", "grasping_data_2.pt", "grasping_data_3.pt"]
    sizes = [len(od.load_transitions(f)[2]) for f in files]
    assert sizes == [12, 12, 1]
    u = od.unite(files)
    assert u["rewards"] == np.concatenate(allr).tolist() and u["actions"] == np.concatenate(alla).tolist()
    pos = od.extract_positives(u)
    assert len(pos["rewards"]) == int(np.concatenate(allr).sum()) and all(r == 1 for r in pos["rewards"])
    assert sum(rec.reward_counter.values()) == 25


def test_ragged_reference_file_is_cut_to_the_common_prefix(tmp_path):
    import torch

    rgb, depth, act, rew = _batch(4, H=8, W=8)
    d = od.pack_transitions(rgb, depth, od.flat_action(act, 8, 8), rew)
    d["states"].append({"rgb": rgb[0], "depth": depth[0]})  # a state whose action was never taken (generate_data.py:96-100)
    p = str(tmp_path / "x.pt")
    torch.save(d, p)
    assert len(od.load_transitions(p)[0]) == 4


def test_reference_dataset_class_reads_our_file(tmp_path):
    """the unmodified Grasping_Dataset (Offline RL/grasping_dataset.py:12-74) on a file written by this module, frozen in
    tests/golden/reference_classes.json (tests/golden/make_reference_classes_golden.py): the same file read the way that class reads
    it (torch.load, then states[i]["rgb"/"depth"], actions[i], rewards[i]) gives its length, action, reward and depth channel"""
    import torch

    g = json.load(open(GOLD))["grasping_dataset"]
    rgb, depth, act, rew = _batch(3, seed=5)
    p = str(tmp_path / "grasping_data_1.pt")
    od.save_transitions(p, rgb, depth, od.flat_action(act), rew)
    data = torch.load(p, weights_only=False)
    assert len(data["states"]) == g["length"] == 3
    assert data["actions"][1] == g["action"] == int(od.flat_action(act)[1]) and data["rewards"][1] == g["reward"] == int(rew[1])
    s = data["states"][1]
    assert g["shape"] == [4, 200, 200] and s["rgb"].shape == (200, 200, 3) and s["rgb"].dtype == np.uint8  # HWC uint8: what ToPILImage takes
    # transform_observation's depth channel (grasping_dataset.py:42-56), in float32 like the file: clip at 1.1, add N(0, 1e-3) noise,
    # negate, min-max normalise
    np.random.seed(0)
    d = np.minimum(s["depth"], np.float32(1.1))
    d += np.random.normal(loc=0, scale=0.001, size=d.shape)
    d = -d
    d = (d - d.min()) / (d.max() - d.min())
    assert float(d.min()) == 0.0 and float(d.max()) == 1.0
    assert np.abs(d.reshape(-1)[g["pixels"]].astype(np.float32) - np.array(g["depth"], np.float32)).max() <= 1e-6


@pytest.mark.gpu
def test_batched_data_generation_on_the_gpu(tmp_path):
    """SURVEY 8f.3 end to end on the device: tools/generate_data_batched.py (epsilon-greedy Q-net actions over batched environments)
    writes files in the reference's layout that load back with the right shapes and reward range"""
    import subprocess

    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    out = str(tmp_path / "Data")
    r = subprocess.run([sys.executable, os.path.join(root, "tools", "generate_data_batched.py"), "--envs", "12", "--episodes", "1", "--steps", "2", "--out", out],
                       capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stderr[-2000:]
    files = sorted(os.listdir(out))
    assert len(files) == 2  # 24 transitions, 12 per file (generate_data.py:19,83)
    rgb, depth, actions, rewards = od.load_transitions(os.path.join(out, files[0]))
    assert rgb.shape == (12, 200, 200, 3) and depth.shape == (12, 200, 200) and actions.shape == (12,)
    assert set(rewards.tolist()) <= {0, 1} and 0 <= actions.min() and actions.max() < 6 * 200 * 200
    assert 0.5 < float(depth.min()) and rgb.std() > 1
