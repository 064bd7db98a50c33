#!/usr/bin/env python
"""bench.py — MuJoCo-equivalent sub-steps/s of the batched grasp engine (BASELINE.json metric).

A "step" is one pass of the hot path over one batch: every busy environment advances `--chunk` iterations of the
reference control loop (7 PID evaluations + one mj_step, MujocoController.py:318-382) while running the grasp program
(GraspingEnv.py:205-386); environments whose attempt finished get the next synthetic waypoint before the next step.
Headline workload: scene A (UR5gripper_2_finger.xml), 4096 envs per GPU, physics + control only in the timed `value`
(BASELINE configs[1]/[2] scene and env count); `e2e` goes through BatchedGraspEnv.step (host actions in, pixel_2_world,
whole attempts, 200x200 RGB-D render, host rewards AND the observation copied to pinned host memory, as the reference's API
hands it to its caller).  Extra objects on the same JSON line (not the headline): `configs` = BASELINE configs 3, 4, 5 as
specified (SURVEY 8d; config 5 runs in a child process per rank), `qnet` = the a16 forward alone, `learner` = one learn() update.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--legs 3,4,5,qnet,learn] [--dump-outputs DIR]
Under torchrun every rank owns one GPU and its own envs (weak scaling, no data-path collective).
--dump-outputs DIR writes what the last timed step left for a caller of the engine (rank 0's environments) as DIR/<name>.npy; the
inputs are seeded and the engine's result does not depend on timing, so two runs with the same arguments write the same arrays
and two builds can be compared array by array.
Nothing is written into the source tree: the fast oracle build goes to a temporary directory.
"""
import argparse
import atexit
import hashlib
import json
import os
import shutil
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True  # the tree may be read-only, and the benchmark leaves nothing in it

METRIC = "mujoco_substeps_per_sec"
UNIT = "substeps/s"
STATE_BYTES_PER_SUBSTEP = 2 * (50 + 44 + 44 + 14) * 8  # fp64 read+write of qpos, qvel, qacc_warmstart, 7 PID inputs, 7 targets (scene A)
ENGINE_SO = os.path.join(ROOT, "mujoco_rl_ur5_b200", "csrc", "libgrasp_engine.so")
DUMP_MAX_BYTES = 60 * 10**6  # --dump-outputs stays under 64 MB with the .npy headers


def measured_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured"
        except Exception:
            pass
    return 6650.0, "fallback"


def host_cores():
    """what this process may actually use: the scheduler affinity mask and the cgroup CPU quota (a box can show 128 logical CPUs
    and grant ~9 of them, r01) next to os.cpu_count()"""
    out = {"os_cpu_count": os.cpu_count() or 1}
    try:
        out["affinity"] = len(os.sched_getaffinity(0))
    except Exception:
        out["affinity"] = out["os_cpu_count"]
    quota = None
    try:
        q, per = open("/sys/fs/cgroup/cpu.max").read().split()
        if q != "max":
            quota = float(q) / float(per)
    except Exception:
        try:
            q = float(open("/sys/fs/cgroup/cpu/cpu.cfs_quota_us").read())
            per = float(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
            if q > 0:
                quota = q / per
        except Exception:
            pass
    out["cgroup_quota_cpus"] = quota
    usable = out["affinity"]
    if quota:
        usable = max(1, min(usable, int(round(quota))))
    out["usable"] = usable
    return out


def lib_sha16(path=ENGINE_SO):
    try:
        return hashlib.sha256(open(path, "rb").read()).hexdigest()[:16]
    except Exception:
        return None


def build_fast_oracle():
    """-O3 -march=native -ffp-contract=fast build of the oracle, compiled on THIS machine (the optimistic CPU baseline) in a temporary
    directory that is removed at exit; returns the library's path, or None if it does not build"""
    try:
        d = tempfile.mkdtemp(prefix="grasp_oracle_fast_")
        atexit.register(shutil.rmtree, d, True)
        for f in ("Makefile", "grasp_oracle.c", "orc_math.h"):
            shutil.copy(os.path.join(ROOT, "oracle", f), d)
        subprocess.check_call(["make", "-s", "-C", d, "fast"], stdout=subprocess.DEVNULL, stderr=subprocess.DEVNULL)
        so = os.path.join(d, "libgrasp_oracle_fast.so")
        return so if os.path.exists(so) else None
    except Exception:
        return None


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""

    Q = "index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, gpu_index):
        self.gpu = gpu_index
        self.proc = None
        self.path = None

    def start(self):
        try:
            f = tempfile.NamedTemporaryFile("w", suffix=".csv", delete=False)
            self.path = f.name
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "200", "-i", str(self.gpu)],
                                         stdout=f, stderr=subprocess.DEVNULL)
        except Exception:
            self.proc = None

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": []}
        if not self.proc:
            return out
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        try:
            for line in open(self.path):
                c = [x.strip() for x in line.split(",")]
                if len(c) < 8:
                    continue
                try:
                    sm.append(float(c[1]))
                    mx.append(float(c[2]))
                except ValueError:
                    continue
                for name, v in zip(["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"], c[4:8]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
            os.unlink(self.path)
        except Exception:
            pass
        if sm:
            out = {"sm_mhz": float(np.median(sm)), "sm_max_mhz": float(max(mx)), "reasons": sorted(reasons)}
        return out


# ------------------------------------------------------------------------------------------------ CPU oracle legs
def _oracle_worker(args):
    seed, n_attempts, budget_s = args
    from mujoco_rl_ur5_b200.batched_env import scene_a_reset_qpos
    from mujoco_rl_ur5_b200.model.scene import load_scene, load_scene_blob
    from oracle.oracle_py import OracleEnv

    blob = load_scene_blob("A")
    A, _ = load_scene("A")
    o = OracleEnv(blob)
    o.reset(scene_a_reset_qpos(A, seed))
    o.stay(1000)
    rng = np.random.RandomState(30000 + seed)
    s0, t0 = o.substeps, time.perf_counter()
    for _ in range(n_attempts):
        xyz = [rng.uniform(-0.2, 0.2), rng.uniform(-0.75, -0.45), 0.92]
        o.move_and_grasp(xyz, int(rng.randint(0, 6)), 0.91)
        if time.perf_counter() - t0 > budget_s:
            break
    dt = time.perf_counter() - t0
    n = o.substeps - s0
    o.close()
    return n, dt


def _oracle_leg_subprocess(so, budget_s):
    """times one single-env oracle in a fresh process with the given build of the library"""
    env = dict(os.environ)
    if so:
        env["GRASP_ORACLE_SO"] = so
    r = subprocess.run([sys.executable, os.path.abspath(__file__), "--oracle-leg", str(budget_s)], env=env, capture_output=True, text=True)
    n, dt = json.loads(r.stdout.strip().splitlines()[-1])
    return n, dt


def cpu_baseline_single(budget_s=10.0):
    """the oracle on ONE host core (the reference is single-threaded Python), two builds: the -O2 no-FMA checker build every parity test
    uses, and -O3 -march=native -ffp-contract=fast compiled on this machine; `value` is the faster one (the more honest baseline)"""
    half = max(budget_s / 2, 1.0)
    n2, dt2 = _oracle_leg_subprocess(None, half)
    v2 = n2 / dt2
    v3, n3, dt3 = None, 0, 0.0
    fast = build_fast_oracle()
    if fast:
        try:
            n3, dt3 = _oracle_leg_subprocess(fast, half)
            v3 = n3 / dt3
        except Exception:
            v3 = None
    best = max(v2, v3 or 0.0)
    return {"value": best, "unit": UNIT, "cores": 1, "kind": "port",
            "builds": {"O2_no_fma_checker": v2, "O3_march_native_fma": v3},
            "sample": f"oracle restatement (not mujoco_py), 1 env, synthetic-waypoint grasp attempts: {dt2:.1f} s = {n2} sub-steps (-O2 checker build)"
                      + (f", {dt3:.1f} s = {n3} sub-steps (-O3 -march=native build, compiled on this host)" if v3 else "")}


_W = {}


def _ref_init():
    from mujoco_rl_ur5_b200.model.scene import load_scene, load_scene_blob
    from oracle.oracle_py import OracleEnv

    _W["blob"] = load_scene_blob("A")
    _W["A"] = load_scene("A")[0]
    _W["env"] = OracleEnv(_W["blob"])
    _W["episode"] = 0


def _ref_work(args):
    """one worker = one oracle env (one host thread): reset + settle + grasp attempts until `budget_s` of wall time is used"""
    worker, budget_s = args
    from mujoco_rl_ur5_b200.batched_env import scene_a_reset_qpos

    o = _W["env"]
    t0 = time.perf_counter()
    s0 = o.substeps
    seed = 20000 + worker + 1000 * _W["episode"]
    _W["episode"] += 1
    o.reset(scene_a_reset_qpos(_W["A"], seed))
    o.stay(1000)
    rng = np.random.RandomState(30000 + seed)
    while time.perf_counter() - t0 < budget_s:
        xyz = [rng.uniform(-0.2, 0.2), rng.uniform(-0.75, -0.45), 0.92]
        o.move_and_grasp(xyz, int(rng.randint(0, 6)), 0.91)
    return o.substeps - s0


def run_reference(args):
    """--impl reference: the reference's own mujoco_py path cannot be installed (SURVEY 8c), so this arm times the CPU oracle
    restatement (the -O3 -march=native build when it compiles here) with one single-env process per USABLE host thread (affinity mask
    and cgroup quota, not os.cpu_count()) — every worker resets, settles and runs grasp attempts for a bounded wall-time budget per
    step; value = sub-steps of all workers / wall time."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import multiprocessing as mp

    hc = host_cores()
    cores = hc["usable"]
    fast = build_fast_oracle()
    if fast:
        os.environ["GRASP_ORACLE_SO"] = fast  # inherited by the spawned workers
    budget = args.ref_step_seconds
    ctx = mp.get_context("spawn")
    with ctx.Pool(cores, initializer=_ref_init) as pool:
        total_n, total_t = 0, 0.0
        for step in range(args.warmup + args.steps):
            t0 = time.perf_counter()
            res = pool.map(_ref_work, [(w, budget) for w in range(cores)], chunksize=1)
            dt = time.perf_counter() - t0
            if step >= args.warmup:
                total_n += sum(res)
                total_t += dt
    value = total_n / total_t
    sample = (f"{cores} single-env oracle processes ({'-O3 -march=native' if fast else '-O2'} build; host: {json.dumps(hc)}), each step = reset + settle + "
              f"grasp attempts for >= {budget:.1f} s wall per worker, {args.steps} steps")
    print(json.dumps({
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": 1e3 * total_t / max(args.steps, 1), "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64",
        "data": "synthetic", "config": {"workload": "scene A (UR5gripper_2_finger.xml) grasp attempts, synthetic waypoints; CPU oracle restatement of the reference path (not mujoco_py)"},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample, "host": hc},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }))


# ------------------------------------------------------------------------------------------------ GPU arm
def run_config5_child(args):
    """BASELINE config 5 on one GPU: N scene-B envs, reset + settle, then whole grasp attempts at random table pixels; one JSON line"""
    import torch

    from mujoco_rl_ur5_b200.batched_env import BatchedGraspEnv

    dev_i, n5 = args.config5_child, args.scene_b_envs
    torch.cuda.set_device(dev_i)
    rng = np.random.RandomState(args.config5_seed)
    e5 = BatchedGraspEnv(n5, "B", dev_i, env_index_offset=args.config5_offset, settle_ms=1000)
    t0 = time.perf_counter()
    e5.reset()
    torch.cuda.synchronize()
    reset_s = time.perf_counter() - t0
    n0 = e5.total_substeps()
    t0 = time.perf_counter()
    for _ in range(args.scene_b_steps):
        px, py = rng.randint(40, 160, n5), rng.randint(60, 140, n5)
        e5.step(np.stack([py * 200 + px, rng.randint(0, 6, n5)], axis=1))
    torch.cuda.synchronize()
    dt = time.perf_counter() - t0
    out = {"substeps": int(e5.total_substeps() - n0), "seconds": dt, "reset_s": reset_s, "flagged": int((e5.engine.status() != 0).sum().item()),
           "workspace": "shared memory, CTA per env" if e5.engine.size(9) else "shared memory, warp per env"}
    e5.close()
    print(json.dumps(out), flush=True)


def dump_outputs(directory, arrays):
    """writes each [N, ...] tensor as <directory>/<name>.npy, float32 kept, everything else as float64; above DUMP_MAX_BYTES in all, the
    same seeded sample of environments (rows) from every array, with their indices in env_index.npy"""
    arrays = {k: v.detach().cpu().numpy() for k, v in arrays.items()}
    arrays = {k: v.astype(np.float32 if v.dtype == np.float32 else np.float64) for k, v in arrays.items()}
    n = len(next(iter(arrays.values())))
    row_bytes = sum(v.nbytes for v in arrays.values()) // max(n, 1)
    if n * row_bytes > DUMP_MAX_BYTES:
        keep = np.sort(np.random.RandomState(0).choice(n, DUMP_MAX_BYTES // (row_bytes + 8), replace=False))
        arrays = {k: v[keep] for k, v in arrays.items()}
        arrays["env_index"] = keep.astype(np.float64)
    os.makedirs(directory, exist_ok=True)
    for k, v in arrays.items():
        np.save(os.path.join(directory, k + ".npy"), v)


def run_ours(args):
    import torch
    import torch.distributed as dist

    from mujoco_rl_ur5_b200.batched_env import BatchedGraspEnv

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    N = args.envs
    legs = set(x for x in args.legs.split(",") if x)
    env = BatchedGraspEnv(N, "A", local, env_index_offset=rank * N)
    eng = env.engine
    env.reset()
    gen = torch.Generator(device=dev)
    gen.manual_seed(30000 + rank)
    flush = torch.empty(256 * 1024 * 1024 // 4, dtype=torch.float32, device=dev)  # > 126 MB L2

    def assign_idle():
        idle = (eng.busy() == 0)
        u = torch.rand((N, 3), generator=gen, device=dev, dtype=torch.float64)
        coords = torch.stack([-0.2 + 0.4 * u[:, 0], -0.75 + 0.3 * u[:, 1], torch.full((N,), 0.92, device=dev, dtype=torch.float64)], dim=1)
        rot = torch.randint(0, 6, (N,), generator=gen, device=dev, dtype=torch.int32)
        eng.grasp(coords, rot, 0.91, env_mask=idle.to(torch.uint8))

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def aggregate(n_local, seconds_local):
        """whole-job units / max-over-ranks time"""
        tt = torch.tensor([seconds_local], dtype=torch.float64, device=dev)
        tn = torch.tensor([float(n_local)], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
            dist.all_reduce(tn, op=dist.ReduceOp.SUM)
        return float(tn[0]), float(tt[0])

    # ---- value: device-resident stepping
    for _ in range(args.warmup):
        assign_idle()
        eng.run_async(args.chunk)
    barrier()
    sub0 = env.total_substeps()
    l0, s0 = eng.counters()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    barrier()
    evs = []
    kern_evs = []
    for _ in range(args.steps):
        flush.fill_(1.0)  # L2 flush between timed iterations (outside the event pairs)
        a, b, c = torch.cuda.Event(True), torch.cuda.Event(True), torch.cuda.Event(True)
        a.record()
        assign_idle()
        b.record()
        eng.run_async(args.chunk)
        c.record()
        evs.append((a, c))
        kern_evs.append((b, c))
    barrier()
    clocks = sampler.stop() if rank == 0 else None
    if args.dump_outputs and rank == 0:
        qpos, qvel = eng.get_state()
        result, steps, reward, total = eng.results()
        dump_outputs(args.dump_outputs, {"qpos": qpos, "qvel": qvel, "targets": eng.get_targets(), "ctrl": eng.get_ctrl(), "result": result,
                                         "steps": steps, "reward": reward, "total_substeps": total, "grasp_info": eng.grasp_info(),
                                         "busy": eng.busy(), "status": eng.status()})
    ms = sum(a.elapsed_time(c) for a, c in evs)
    kern_ms = sum(b.elapsed_time(c) for b, c in kern_evs)
    sub1 = env.total_substeps()
    l1, s1 = eng.counters()
    nsub = sub1 - sub0
    nsub_all, sec_max = aggregate(nsub, ms * 1e-3)
    value = nsub_all / sec_max
    ms_max = sec_max * 1e3

    # ---- e2e: the public batched gym API with HOST buffers: actions from pinned host memory, rewards AND observations back to it
    env.reset()
    rng = np.random.RandomState(30000 + rank)

    def table_actions(n=N):
        # random pixels over the table region of the image (the agent's random-action filter, Grasping_Agent_multidiscrete.py:267-279)
        px = rng.randint(40, 160, n)
        py = rng.randint(60, 140, n)
        return np.stack([py * 200 + px, rng.randint(0, 6, n)], axis=1)

    env.step(table_actions(), obs_to_host=True)  # warm-up attempt (allocates the pinned observation buffers)
    barrier()
    e_sub0 = env.total_substeps()
    t0 = time.perf_counter()
    for _ in range(args.e2e_steps):
        env.step(table_actions(), obs_to_host=True)
    torch.cuda.synchronize()
    e_dt = time.perf_counter() - t0
    e_n_all, e_sec = aggregate(env.total_substeps() - e_sub0, e_dt)
    e2e_value = e_n_all / e_sec
    status = eng.status()
    status_or = int(torch.bitwise_or(status[0], status.max()).item()) if N else 0
    n_flag = int((status != 0).sum().item())
    h2d, d2h = env.h2d_bytes_per_step, env.d2h_bytes_per_step + env.obs_bytes
    env.close()
    del env, eng
    torch.cuda.empty_cache()

    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass

    # ---- a16: Q-network forward (bf16 tcgen05) alone; extra object, not the headline
    qinfo = None
    qf = None
    if "qnet" in legs or "4" in legs:
        from mujoco_rl_ur5_b200.qnet import QNetForward, make_torch_qnet

        torch.manual_seed(0)
        qf = QNetForward(make_torch_qnet(6).state_dict(), local, max_batch=args.qnet_chunk)
    if "qnet" in legs:
        envq = BatchedGraspEnv(args.qnet_images, "A", local, env_index_offset=rank * args.qnet_images)
        sub = envq.reset()
        nimg = args.qnet_images
        for _ in range(2):
            act, _ = qf.greedy(qf.forward(qf.obs_to_state(sub, 1.1)))
        barrier()
        l_q0 = qf.launches
        q0, q1 = torch.cuda.Event(True), torch.cuda.Event(True)
        q0.record()
        for _ in range(args.qnet_reps):
            act, _ = qf.greedy(qf.forward(qf.obs_to_state(sub, 1.1)))
        q1.record()
        barrier()
        qms = q0.elapsed_time(q1) / args.qnet_reps
        tf = nimg * 41.99424e9 / (qms * 1e-3) / 1e12
        pk = float(peaks.get("bf16_tflops_sustained", 1400.0))
        qinfo = {"images": nimg, "chunk": args.qnet_chunk, "ms_per_batch": qms, "images_per_s": nimg / (qms * 1e-3), "tflops": tf,
                 "roofline": {"bound": "tensor", "achieved": tf, "peak": pk, "unit": "TFLOP/s", "frac": tf / pk,
                              "note": "41.99 GFLOP per 200x200 image (SURVEY 8d); peak = " + ("measured sustained cuBLAS bf16" if peaks else "fallback")},
                 "kernels_per_batch": (qf.launches - l_q0) // max(args.qnet_reps, 1)}
        envq.close()
        del envq, sub

    # ---- f2: the learner's update (Grasping_Agent_multidiscrete.py:388-446: BATCH_SIZE 12 transitions, BN in train mode over the batch,
    # gather-BCE, Adam with weight decay); under torchrun the fp32 gradient all-reduce over the default process group is inside the step
    linfo = None
    if "learn" in legs:
        from mujoco_rl_ur5_b200.qnet_learn import QNetLearner

        lb = 12
        g = torch.Generator(device="cpu").manual_seed(7 + rank)
        st = torch.rand(lb, 4, 200, 200, generator=g).to(dev)
        ac = torch.randint(0, 6 * 200 * 200, (lb, 1), generator=g).to(dev)
        rw = (torch.rand(lb, 1, generator=g) < 0.3).float().to(dev)
        import torch.distributed as dist

        # the per-group gradient all-reduce (NCCL) is part of the step only on request: it is checked by tools/learner_2gpu_check.py, and the
        # default multi-rank bench line must not depend on it
        use_pg = world > 1 and os.environ.get("BENCH_LEARN_ALLREDUCE", "0") == "1"
        learner = QNetLearner(seed=0, device=local, process_group=dist.group.WORLD if use_pg else None)
        for _ in range(2):
            learner.learn_step(st, ac, rw)
        barrier()
        l_l0 = learner.launches
        e0, e1 = torch.cuda.Event(True), torch.cuda.Event(True)
        e0.record()
        for _ in range(args.qnet_reps):
            loss_l = learner.learn_step(st, ac, rw)
        e1.record()
        barrier()
        lms = e0.elapsed_time(e1) / args.qnet_reps
        ltf = lb * 3 * 41.99424e9 / (lms * 1e-3) / 1e12  # forward + dgrad + wgrad ~ 3x the forward MACs
        linfo = {"batch_per_gpu": lb, "ms_per_update": lms, "updates_per_s": 1e3 / lms, "transitions_per_s": world * lb * 1e3 / lms, "tflops_per_gpu": ltf,
                 "kernels_per_update": (learner.launches - l_l0) // max(args.qnet_reps, 1), "loss": loss_l,
                 "collective": ("all_reduce of %.1f MB fp32 gradients over %d ranks (NCCL)" % (learner.grad.numel() * 4 / 1e6, world)) if use_pg else None,
                 "note": "QNetLearner.learn_step: forward (tcgen05) with batch-statistics BN, gather-BCE, dgrad (tcgen05), wgrad (CUDA-core tiles), Adam; "
                         "includes the loss .item() read like the reference"}
        del learner, st, ac, rw

    configs = {}
    # ---- BASELINE config 3: 4096 envs + 200x200 RGB-D raster, fixed-size objects (scene A1 = iteration 1, README.md:20), render every
    # attempt, actions through the depth image like GraspEnv.step
    if "3" in legs:
        e3 = BatchedGraspEnv(N, "A1", local, env_index_offset=rank * N)
        e3.reset()
        e3.step(table_actions())
        barrier()
        n0 = e3.total_substeps()
        t0 = time.perf_counter()
        for _ in range(args.leg_steps):
            e3.step(table_actions())
        torch.cuda.synchronize()
        n3, s3 = aggregate(e3.total_substeps() - n0, time.perf_counter() - t0)
        configs["3"] = {"workload": f"BASELINE config 3: {N} envs/GPU, scene A1 (six 4 cm cubes), {args.leg_steps} BatchedGraspEnv.step calls = whole grasp "
                                    "attempts at random table pixels + 200x200 RGB-D render after every attempt",
                        "value": n3 / s3, "unit": UNIT, "attempts_per_s": world * N * args.leg_steps / s3,
                        "envs_flagged": int((e3.engine.status() != 0).sum().item())}
        e3.close()
        del e3
    # ---- BASELINE config 4: full step + Modules.py Q-net forward (bf16) choosing the action, 512 envs per GPU (4096 over 8 GPUs)
    if "4" in legs:
        from mujoco_rl_ur5_b200.batched_agent import BatchedGreedyAgent

        n4 = args.config4_envs
        e4 = BatchedGraspEnv(n4, "A1", local, env_index_offset=rank * n4)
        obs = e4.reset()
        agent = BatchedGreedyAgent.__new__(BatchedGreedyAgent)
        agent.torch, agent.env, agent.qnet, agent.depth_threshold = torch, e4, qf, 1.1
        agent.gen = torch.Generator(device=dev)
        agent.gen.manual_seed(rank)
        act, _ = agent.greedy(obs)
        obs, _, _, _ = e4.step(act)
        barrier()
        n0 = e4.total_substeps()
        t0 = time.perf_counter()
        rew = 0
        for _ in range(args.leg_steps):
            act, _ = agent.greedy(obs)           # obs -> state (device) -> tcgen05 forward of all images -> arg-max; actions stay on the GPU
            obs, r, _, _ = e4.step(act)
            rew += int(r.sum())
        torch.cuda.synchronize()
        n4s, s4 = aggregate(e4.total_substeps() - n0, time.perf_counter() - t0)
        configs["4"] = {"workload": f"BASELINE config 4: {n4} envs/GPU (x{world} GPUs), scene A1, every step = Q-net forward (bf16 tcgen05, random-init "
                                    f"weights torch.manual_seed(0), chunks of {args.qnet_chunk}) over ALL {n4} observations -> greedy pixel/rotation -> whole grasp "
                                    "attempt -> RGB-D render",
                        "value": n4s / s4, "unit": UNIT, "steps": args.leg_steps, "qnet_images_per_step": world * n4,
                        "env_steps_per_s": world * n4 * args.leg_steps / s4, "rewards": rew}
        e4.close()
        del e4, agent
    # ---- BASELINE config 5: the reference's default scene (40-object random pile), 1024 envs per GPU, reset + 500 settle sub-steps, then
    # FULL grasp attempts (~1000-3000 sub-steps each) through the depth image, 6 rotations
    if "5" in legs:
        # The leg runs in a CHILD process on this rank's GPU (bench.py --config5-child): the big-scene build has an open defect (DESIGN.md
        # section 4: an illegal memory access for roughly one in five random action sets of 1024 attempts), and a CUDA fault in this
        # process would take the headline line with it.  The child only computes; the cross-rank reduction stays here.
        n5 = args.scene_b_envs
        cmd = [sys.executable, os.path.abspath(__file__), "--config5-child", str(local), "--scene-b-envs", str(n5), "--scene-b-steps", str(args.scene_b_steps),
               "--config5-offset", str(rank * n5), "--config5-seed", str(40000 + rank)]
        child, err5 = None, None
        try:
            r5 = subprocess.run(cmd, capture_output=True, text=True, timeout=1500)
            lines5 = [l for l in r5.stdout.strip().splitlines() if l.startswith("{")]
            if r5.returncode == 0 and lines5:
                child = json.loads(lines5[-1])
            else:
                tail = [l for l in r5.stderr.strip().splitlines() if "Error" in l or "error" in l]
                err5 = (tail[-1] if tail else "exit code %d" % r5.returncode)[:300]
        except Exception as e:  # timeout
            err5 = repr(e)[:300]
        ok_all, _ = aggregate(1.0 if child else 0.0, 0.0)
        n5s, s5 = aggregate(child["substeps"] if child else 0.0, child["seconds"] if child else 0.0)
        if ok_all == world:
            configs["5"] = {"workload": f"BASELINE config 5: scene B UR5gripper_2_finger_many_objects.xml (40 free objects, condim 6, nv 248), {n5} envs/GPU, "
                                        f"reset by the reference rule + 500 settle sub-steps (untimed: {child['reset_s']:.1f} s), then {args.scene_b_steps} BatchedGraspEnv.step = "
                                        "full grasp attempts at random table pixels (6 rotations) + render; run in a child process per rank",
                            "value": n5s / s5, "unit": UNIT, "envs_per_gpu": n5, "seconds": s5, "substeps_per_attempt": n5s / (world * n5 * args.scene_b_steps),
                            "workspace": child["workspace"], "envs_flagged": child["flagged"]}
        else:
            configs["5"] = {"workload": f"BASELINE config 5: scene B, {n5} envs/GPU, full grasp attempts (child process per rank)", "value": None, "unit": UNIT,
                            "error": err5 or "the child of another rank failed", "ranks_ok": int(ok_all)}
        if rank == 0 and args.cpu_seconds > 0 and "5" in configs:
            from mujoco_rl_ur5_b200.batched_env import HOME, scene_b_reset_qpos
            from mujoco_rl_ur5_b200.model.scene import load_scene, load_scene_blob
            from oracle.oracle_py import OracleEnv  # cpu_baseline leg: the checker timed beside the product, never on its path

            Ab, _ = load_scene("B")
            o = OracleEnv(load_scene_blob("B"))
            o.reset(scene_b_reset_qpos(Ab, 20000))
            o.move_group("All", HOME, 1e-9, 249)
            t0 = time.time()
            o.move_group("All", HOME, 1e-9, 79)
            dtb = time.time() - t0
            o.close()
            configs["5"]["cpu_baseline"] = {"value": 80 / dtb, "unit": UNIT, "cores": 1, "kind": "port",
                                            "sample": "fp64 oracle (-O2 checker build), one env, 80 sub-steps after 250 sub-steps of settling"}

    if rank == 0:
        peak, which = measured_peak()
        per_launch_sub = nsub / max(args.steps, 1)
        achieved = (nsub * STATE_BYTES_PER_SUBSTEP) / (kern_ms * 1e-3) / 1e9 if kern_ms > 0 else 0.0
        # DRAM traffic per launch: only from an ncu capture of THIS build at THIS launch shape (profiles/k_run_traffic.json records the
        # library hash, env count and chunk it was taken with); anything else is unmeasured -> null
        traffic, traffic_note = None, "unmeasured for this build (no matching ncu capture)"
        tp = os.path.join(ROOT, "profiles", "k_run_traffic.json")
        if os.path.exists(tp):
            try:
                tj = json.load(open(tp))
                if tj.get("lib_sha16") == lib_sha16() and tj.get("chunk") == args.chunk and tj.get("envs") == N:
                    traffic = tj.get("dram_bytes_per_launch")
                    traffic_note = f"ncu --set full of this build ({tj.get('capture')}): dram__bytes_read.sum + dram__bytes_write.sum per k_run launch"
            except Exception:
                pass
        cpu = cpu_baseline_single(args.cpu_seconds)
        cpu["host"] = host_cores()
        out = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms_max / max(args.steps, 1), "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64",
            "data": "synthetic",
            "config": {"workload": f"scene A UR5gripper_2_finger.xml, {N} envs/GPU, physics+PID+grasp-program sub-steps, synthetic waypoints; "
                                   f"step = {args.chunk} loop iterations per busy env; L2 flushed (256 MiB fill) between timed steps",
                       "envs_per_gpu": N, "chunk": args.chunk, "substeps_per_step": per_launch_sub, "solver": "newton", "parallelism": f"env-shard x{world}",
                       "engine_lib_sha16": lib_sha16()},
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "traffic": traffic,
                         "traffic_note": traffic_note,
                         "note": f"k_run; algorithmic bytes = {STATE_BYTES_PER_SUBSTEP} B/env-sub-step (fp64 state rows), peak = {which} copy bandwidth; "
                                 "this path is fp64-ALU/latency bound, not HBM bound (DESIGN.md)"},
            "cpu_baseline": cpu,
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                    "steps": args.e2e_steps, "note": "BatchedGraspEnv.step(obs_to_host=True): pinned host actions -> pixel_2_world -> full grasp attempts -> RGB-D "
                                                     "render -> rewards AND the whole observation (rgb u8 + depth f32) copied to pinned host memory, as the reference API "
                                                     "returns it to its caller every step"},
            "gpu_launches": int(l1 - l0), "substep_kernel_launches": int(s1 - s0),
            "clocks": clocks, "env_status_flags": {"envs_flagged": n_flag, "or": status_or}, "qnet": qinfo, "learner": linfo, "configs": configs,
        }
        print(json.dumps(out))
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--envs", type=int, default=4096, help="environments per GPU")
    ap.add_argument("--chunk", type=int, default=256, help="control-loop iterations per busy env and step")
    ap.add_argument("--e2e-steps", type=int, default=2)
    ap.add_argument("--cpu-seconds", type=float, default=10.0)
    ap.add_argument("--legs", default="3,4,5,qnet,learn", help="extra objects: BASELINE configs 3,4,5, the Q-net forward alone, one learner update ('' = none)")
    ap.add_argument("--leg-steps", type=int, default=2, help="timed BatchedGraspEnv.step calls of the config 3 / 4 legs")
    ap.add_argument("--config4-envs", type=int, default=512, help="environments per GPU of the config 4 leg (4096 over 8 GPUs)")
    ap.add_argument("--qnet-images", type=int, default=512, help="images of the Q-net forward leg")
    ap.add_argument("--qnet-chunk", type=int, default=64)
    ap.add_argument("--qnet-reps", type=int, default=3)
    ap.add_argument("--scene-b-envs", type=int, default=1024, help="environments per GPU of the config 5 leg")
    ap.add_argument("--scene-b-steps", type=int, default=1, help="timed BatchedGraspEnv.step calls (full grasp attempts) of the config 5 leg")
    ap.add_argument("--ref-step-seconds", type=float, default=3.0, help="--impl reference: wall-time budget per worker and step")
    ap.add_argument("--dump-outputs", default=None, metavar="DIR",
                    help="write the engine state and results after the last timed step as DIR/<name>.npy (rank 0's environments)")
    ap.add_argument("--oracle-leg", type=float, default=None, help=argparse.SUPPRESS)
    ap.add_argument("--config5-child", type=int, default=None, help=argparse.SUPPRESS)
    ap.add_argument("--config5-offset", type=int, default=0, help=argparse.SUPPRESS)
    ap.add_argument("--config5-seed", type=int, default=40000, help=argparse.SUPPRESS)
    args = ap.parse_args()
    if args.config5_child is not None:  # internal: the config 5 leg on one GPU, in its own process (see run_ours)
        run_config5_child(args)
        return
    if args.oracle_leg is not None:  # internal: one single-env oracle timing in a fresh process (GRASP_ORACLE_SO picks the build)
        print(json.dumps(_oracle_worker((20000, 1000, args.oracle_leg))))
        return
    if args.warmup < 3 and args.impl == "ours":
        args.warmup = 3
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
