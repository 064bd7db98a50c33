"""The north star's acceptance replay: "grasp-success flag bit-exact on a fixed 256-action replay, joint angles within 1e-4".

tests/golden/replay_256.json + replay_256_states.npz hold 16 environments x 16 consecutive GraspEnv.step calls run on the fp64
CPU oracle (tests/golden/make_replay_golden.py: the reference's step(), GraspingEnv.py:62-156, restated on the oracle) together
with the oracle's full state before every action.  Here the same frozen actions go through the product's public batched API
(BatchedGraspEnv.step: host actions -> depth lookup in the device-rendered observation -> pixel_2_world -> gate -> whole grasp
attempt on the device -> re-render), every step starting from the stored state (re-synchronised replay: contact dynamics is
chaotic, a free-running 16-attempt sequence of two fp64 implementations that differ in summation order separates after 9-14
attempts - measured on the B200, gpurun of r01h - so the 256 attempts are compared one by one along the oracle's trajectory).
Compared per record: the depth read at the action pixel (1e-4 m), the executed / skipped decision (exact), the reward
(bit-exact), the per-phase sub-step counts of the grasp program (identical on >= 98 % of the attempts) and the arm joint angles
after the attempt (1e-4 rad).
"""
import json
import os

import numpy as np
import pytest

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "replay_256.json")


def _load():
    return json.load(open(GOLD))


def test_replay_fixture_is_what_the_oracle_produces_today():
    """CPU: re-run the first 3 steps of two environments on the oracle and compare with the committed fixture."""
    import sys

    sys.path.insert(0, os.path.dirname(GOLD))
    import make_replay_golden as mk

    g = _load()
    st = np.load(GOLD.replace(".json", "_states.npz"))
    assert g["n_envs"] * g["n_steps"] == 256 and len(g["envs"]) == 16 and all(len(e) == 16 for e in g["envs"])
    old_steps = mk.N_STEPS
    mk.N_STEPS = 3
    try:
        for i in (0, 11):
            rec = mk.replay_env(i, [s["action"] for s in g["envs"][i][:3]], (st["qpos0"][i], st["qvel0"][i]))
            for sn, so in zip(rec, g["envs"][i]):
                assert (sn["executed"], sn["reward"], sn["info"]) == (so["executed"], so["reward"], so["info"])
                assert abs(sn["depth"] - so["depth"]) < 1e-7
                assert np.abs(np.array(sn["arm_qpos"]) - np.array(so["arm_qpos"])).max() < 1e-9
    finally:
        mk.N_STEPS = old_steps


def test_replay_fixture_exercises_every_outcome():
    """the replay is only a parity statement if it contains skipped actions, failed attempts and successful grasps"""
    flat = [s for e in _load()["envs"] for s in e]
    assert sum(not s["executed"] for s in flat) >= 10
    assert sum(s["reward"] for s in flat) >= 5
    assert sum(s["info"][11] for s in flat) >= 20       # fingers closed on something at the table
    assert sum(s["info"][3] == 2 for s in flat) >= 1    # grasp height not reached within 300 sub-steps
    assert sum(s["substeps"] for s in flat) > 400_000


@pytest.mark.gpu
def test_fixed_256_action_replay_matches_oracle(tmp_path):
    from mujoco_rl_ur5_b200.batched_env import BatchedGraspEnv

    g = _load()
    st = np.load(GOLD.replace(".json", "_states.npz"))
    n, T = g["n_envs"], g["n_steps"]
    env = BatchedGraspEnv(n, "A", 0, seed_base=20000, settle_ms=1000)
    bad = []
    n_reward, n_exec = 0, 0
    worst_q, worst_d, worst_obj = 0.0, 0.0, 0.0
    from oracle.oracle_py import OracleEnv

    orc = OracleEnv(env.blob)  # renders the oracle's image of the oracle's state AFTER every attempt (the checker, not the product)
    post_frac = np.zeros((n, T))   # fraction of the 40 000 pixels of the post-attempt depth image within 1e-4 m of the oracle's
    post_worst_px = 0
    for k in range(T):
        env.engine.set_state(st["qpos0"][:, k], st["qvel0"][:, k])  # synchronisation point (the oracle did reset(qpos, qvel) here)
        env.current_observation = None                               # -> step() renders the observation of this state
        actions = np.array([g["envs"][i][k]["action"] for i in range(n)], dtype=np.int32)
        depth_before = env.get_observation()["depth"].cpu().numpy()
        obs, reward, done, info = env.step(actions)
        executed = info["executed"].cpu().numpy().astype(bool)
        ginfo = env.engine.grasp_info().cpu().numpy()
        qpos = env.engine.get_state()[0].cpu().numpy()
        depth_after = obs["depth"].cpu().numpy()
        for i in range(n):
            orc.reset(st["qpos1"][i, k])
            _, od = orc.render(env.cam, 200, 200)
            close = np.abs(depth_after[i] - od) <= 1e-4
            post_frac[i, k] = close.mean()
            post_worst_px = max(post_worst_px, int((~close).sum()))
        for i in range(n):
            s = g["envs"][i][k]
            x, y = s["action"][0] % 200, s["action"][0] // 200
            dd = abs(float(depth_before[i, y, x]) - s["depth"])
            worst_d = max(worst_d, dd)
            if dd > 1e-4:
                bad.append(("depth", i, k, float(depth_before[i, y, x]), s["depth"]))
            if bool(executed[i]) != s["executed"]:
                bad.append(("executed", i, k, bool(executed[i]), s["executed"]))
                continue
            if int(reward[i]) != s["reward"]:
                bad.append(("reward", i, k, int(reward[i]), s["reward"], ginfo[i].tolist(), s["info"]))
            if s["executed"]:
                n_exec += 1
                if ginfo[i].tolist() != s["info"]:
                    bad.append(("phase steps", i, k, ginfo[i].tolist(), s["info"]))
            dq = float(np.abs(qpos[i][:8] - np.array(s["arm_qpos"])).max())
            worst_q = max(worst_q, dq)
            if dq > 1e-4:
                bad.append(("arm_qpos", i, k, dq))
            worst_obj = max(worst_obj, float(np.abs(qpos[i] - st["qpos1"][i, k]).max()))  # reported, not gated: objects may tumble differently
            n_reward += int(reward[i])
        assert not done.any()
    env.close()
    orc.close()
    report = {"actions": n * T, "executed": n_exec, "successful_grasps": n_reward, "max_abs_arm_angle_diff": worst_q,
              "max_abs_depth_diff_at_action_pixel": worst_d, "max_abs_qpos_diff_incl_objects": worst_obj,
              "post_attempt_depth_image": {"compared_with": "oracle render of the oracle's post-attempt state, 200x200, tolerance 1e-4 m",
                                           "records_with_every_pixel_within_tol": int((post_frac == 1.0).sum()),
                                           "records_with_99.9pct_pixels_within_tol": int((post_frac >= 0.999).sum()),
                                           "mean_fraction_within_tol": float(post_frac.mean()), "min_fraction_within_tol": float(post_frac.min()),
                                           "most_pixels_off_in_one_image": post_worst_px},
              "mismatches": [list(map(str, b)) for b in bad]}
    json.dump(report, open(tmp_path / "replay_256_report.json", "w"), indent=1)
    print("replay:", {k: v for k, v in report.items() if k != "mismatches"})
    # gates: depth / executed / reward / arm angles on every one of the 256 records; the per-phase sub-step counts must agree on
    # >= 98 % of the executed attempts (a tolerance test that falls one sub-step later on one side is rounding, not a different
    # outcome - the count is reported)
    hard = [b for b in bad if b[0] != "phase steps"]
    soft = [b for b in bad if b[0] == "phase steps"]
    assert not hard, hard[:10]
    assert len(soft) <= 0.02 * n_exec, soft[:10]
    # post-attempt image (what the agent sees next): an object that came to rest a few mm elsewhere moves its silhouette by a pixel
    # column, so the gate is on the fraction of pixels - measured r02: see profiles/r02*_replay_256_report.json
    assert post_frac.mean() >= 0.999 and (post_frac >= 0.99).mean() >= 0.97, (post_frac.mean(), (post_frac >= 0.99).mean(), post_frac.min())


@pytest.mark.gpu
@pytest.mark.parametrize("build", ["default", "nofma"])
def test_free_running_replay_agreement(build, tmp_path):
    """The same 256 actions WITHOUT re-synchronisation (every env continues from its own state).  Contact dynamics amplifies
    rounding: the CPU oracle replaying its own fixture with ONE coordinate moved by one unit in the last place reproduces 250 of
    256 records (4 of 16 envs leave the trajectory, first at step 7), the oracle built with -O3 -ffp-contract=fast 249 of 256
    (tools/free_run_replay.py; numbers in DESIGN.md).  The CUDA engine must do no worse than that class of perturbation: both the
    default build and the -fmad=false test build.  Gate = the measured agreement minus slack, so that it cannot regress silently."""
    import subprocess
    import sys

    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    out = str(tmp_path / f"free_run_gpu_{build}.json")
    envv = dict(os.environ)
    if build == "nofma":
        lib = os.path.join(root, "mujoco_rl_ur5_b200", "csrc", "libgrasp_engine_nofma.so")
        assert os.path.exists(lib), "build it with __graft_entry__.build()"
        envv["GE_LIB"] = lib
    r = subprocess.run([sys.executable, os.path.join(root, "tools", "free_run_replay.py"), "--backend", "gpu", "--out", out],
                       env=envv, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    rep = json.loads(r.stdout.strip().splitlines()[-1])
    print("free-running replay:", {k: rep[k] for k in ("replayer", "records_identical", "rewards_identical", "envs_identical_to_the_end",
                                                       "first_differing_step_per_env")})
    assert rep["records"] == 256
    assert rep["rewards_identical"] >= 248 and rep["records_identical"] >= 236, rep
    assert rep["envs_identical_to_the_end"] >= 9, rep
    assert rep["max_state_diff_before_step"][1] < 1e-6, rep  # after ONE attempt the trajectories are still rounding-close


def test_oracle_free_run_is_sensitive_to_one_ulp():
    """CPU: the rounding-sensitivity baseline quoted above, checked on 4 environments (the full 16 take ~10 s on 8 cores)"""
    import sys

    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    sys.path.insert(0, os.path.join(root, "tools"))
    sys.path.insert(0, os.path.dirname(GOLD))
    import make_replay_golden as mk

    g = _load()
    i = 4  # the env whose trajectory separates first under a one-ulp perturbation
    rec = mk.replay_env(i, [s["action"] for s in g["envs"][i]], None, perturb_ulp=1)
    same = [(r["executed"], r["reward"], r["info"]) == (s["executed"], s["reward"], s["info"]) for r, s in zip(rec, g["envs"][i])]
    assert all(same[:5]) and not all(same), same
