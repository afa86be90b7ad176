#!/usr/bin/env python
"""bench.py - env-steps/sec of the batched engine on BASELINE.json's configurations.

One "step" = one control step of every environment on the GPU = 25 x {step1, controller, step2} per environment
(robosuite/environments/base.py:467-521): by default the phase-kernel pipeline, one CUDA graph of 25 x 4 kernel nodes per
environment group (8 groups per task handle, each on its own stream); --mode 2 = one persistent unit-queue kernel per handle
(DESIGN.md section 4).  Device-timed with CUDA events around each step on the launch stream, L2 flushed between timed
iterations, max over ranks; the e2e leg times the public API with host buffers (DESIGN.md section 6).

  python bench.py --gpus N --steps K --warmup W [--config 2|3|4|5]   # this repo's CUDA path
  python bench.py --impl reference --gpus N --steps K ...            # CPU arm: the oracle port of the same path on host cores
  python bench.py --gpus 1 --steps K --warmup W --dump-outputs DIR   # also write the last timed step's outputs as DIR/<name>.npy

--config selects BASELINE.json `configs[i-1]`: 2 = 4096 Panda Lift OSC_POSE (the headline metric, default), 3 = 8192 Sawyer
Stack JOINT_VELOCITY, 4 = 16384 Panda NutAssemblyRound, 5 = mixed Lift/Stack/Door/PickPlace, 8192 per GPU (65536 on 8 GPUs)
with the per-step NCCL observation all-gather.  Prints ONE JSON line (rank 0).
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
# The engine replays one CUDA graph per environment group on its own stream; with the default of 8 hardware work queues per process
# streams beyond the eighth share a queue and serialise falsely.  Must be set before CUDA initialises.
os.environ.setdefault("CUDA_DEVICE_MAX_CONNECTIONS", "32")

N_SUBSTEPS = 25
_SCALE = float(os.environ.get("B2S_BENCH_SCALE", "1"))  # scaling experiments only: multiplies every batch size
CONFIGS = {
    2: dict(parts=[("Lift", "Panda", "OSC_POSE", 4096)],
            metric="env-steps/sec (device-timed) Panda-Lift OSC_POSE @4096 envs per GPU",
            workload="4096 Panda Lift envs, OSC_POSE, fp32, random actions, 1xB200 (BASELINE.json configs[1]); weak-scaled: 4096 envs per GPU"),
    3: dict(parts=[("Stack", "Sawyer", "JOINT_VELOCITY", 8192)],
            metric="env-steps/sec (device-timed) Sawyer-Stack JOINT_VELOCITY @8192 envs per GPU",
            workload="8192 Sawyer Stack envs (contact-rich), JOINT_VELOCITY controller, 1xB200 (BASELINE.json configs[2]); weak-scaled"),
    4: dict(parts=[("NutAssemblyRound", "Panda", "OSC_POSE", 16384)],
            metric="env-steps/sec (device-timed) Panda-NutAssemblyRound OSC_POSE @16384 envs per GPU",
            workload="16384 Panda NutAssemblyRound envs (peg-in-hole), OSC_POSE, 1xB200 (BASELINE.json configs[3]); weak-scaled"),
    5: dict(parts=[("Lift", "Panda", "OSC_POSE", 2048), ("Stack", "Panda", "OSC_POSE", 2048), ("Door", "Panda", "OSC_POSE", 2048),
                   ("PickPlace", "Panda", "OSC_POSE", 2048)],
            metric="env-steps/sec (device-timed) mixed Lift/Stack/Door/PickPlace @8192 envs per GPU, obs all-gather",
            workload="65536 mixed Lift/Stack/Door/PickPlace envs sharded across 8xB200 = 4 x 2048 per GPU, NCCL obs all-gather "
                     "(BASELINE.json configs[4]); weak-scaled: 8192 envs per GPU"),
}
# Static per-environment-substep instruction counts from the ncu captures under profiles/ (warp-level instructions executed),
# and SURVEY.md section 8d's useful-FLOP estimate: the inputs of roofline.compute
INST_COUNTS = os.path.join(ROOT, "profiles", "inst_counts.json")


def _peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            return float(json.load(f)["hbm_gbs"]), "measured"
    return 6650.0, "fallback"


def host_threads():
    """threads this process may really use: the scheduler affinity mask capped by the cgroup CPU quota (a container with a
    2-core quota on a 128-core host reports os.cpu_count() == 128; oversubscribing it 64x is what made round 1's CPU arm
    swing 7.6 k .. 21.7 k env-steps/s between boxes)"""
    try:
        n = len(os.sched_getaffinity(0))
    except Exception:
        n = os.cpu_count() or 1
    quota = None
    for path in ("/sys/fs/cgroup/cpu.max", "/sys/fs/cgroup/cpu/cpu.cfs_quota_us"):
        try:
            with open(path) as f:
                txt = f.read().split()
            if path.endswith("cpu.max"):
                if txt[0] != "max":
                    quota = float(txt[0]) / float(txt[1])
            else:
                q = float(txt[0])
                if q > 0:
                    with open("/sys/fs/cgroup/cpu/cpu.cfs_period_us") as f2:
                        quota = q / float(f2.read().split()[0])
            break
        except Exception:
            continue
    if quota is not None:
        n = max(1, min(n, int(quota + 0.5)))
    return n, quota


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region (started before the warm-up: the first sample
    of `nvidia-smi -lms` takes a few hundred ms to arrive)"""

    Q = "clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
        "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index):
        self.rows = []
        self.p = None
        try:
            self.p = subprocess.Popen(["nvidia-smi", "-i", str(index), f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                       "-lms", "20"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.p = None

    def _read(self):
        for line in self.p.stdout:
            self.rows.append((time.time(), line.strip()))

    def stop(self, t0, t1):
        if self.p is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"], "samples": 0}
        time.sleep(0.1)
        self.p.terminate()

        def parse(rows):
            sm, mx, reasons = [], [], set()
            for ts, line in rows:
                f = [x.strip() for x in line.split(",")]
                try:
                    sm.append(float(f[0])); mx.append(float(f[1]))
                except Exception:
                    continue
                for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[2:6]):
                    if val.lower().startswith("active"):
                        reasons.add(name)
            return sm, mx, reasons

        inside = [r for r in self.rows if t0 <= r[0] <= t1 + 0.03]
        sm, mx, reasons = parse(inside)
        where = "timed region"
        if not sm:  # a sub-100 ms region can fall between two samples: use the samples bracketing it (GPU busy on both sides)
            near = [r for r in self.rows if t0 - 0.5 <= r[0] <= t1 + 0.5]
            sm, mx, reasons = parse(near)
            where = "timed region +-0.5 s (warm-up / e2e loops run on both sides)"
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm), "window": where}


def controller_cfg(ctrl, robot):
    from robosuite_b200 import controller_config as cc

    if ctrl == "OSC_POSE":
        return None  # the robot's default composite config (default_panda.json / default_sawyer.json)
    return cc.refactor_composite_controller_config(cc.load_part_controller_config(ctrl), robot, ["right"])


# ------------------------------------------------------------------------------------------------ CPU arm
class CpuArm:
    """The oracle port (fp64 C, oracle/) of the same path on `threads` host threads; each thread owns independent
    environments (the reference runs one env per process: SURVEY.md section 2.1).  Same measurement protocol as the GPU
    arm: `preroll` untimed control steps of random actions first (steady-state contact load), then timed chunks.
    Environments are built by the SAME host code as the GPU arm (reset samplers, controller config resolution) running
    on the CPU stand-in simulator of the test suite."""

    def __init__(self, parts, n_env, threads, preroll):
        import numpy as np

        import robosuite_b200 as suite
        from tests.oracle_sim import OracleSim

        self.threads = threads
        self.rng = np.random.default_rng(0)
        self.sims = []  # (oracle, action_dim)
        per = max(1, n_env // len(parts))
        for task, robot, ctrl, _ in parts:
            env = suite.make(task, robots=robot, num_envs=per, seed=0, horizon=10 ** 9, sim_cls=OracleSim,
                             controller_configs=controller_cfg(ctrl, robot))
            for e in range(per):
                env.sim._push(e)
                self.sims.append((env.sim.o[e], env.action_dim))
            self._keep = getattr(self, "_keep", []) + [env]
        self.n_env = len(self.sims)
        self.preroll_s = self.run(preroll)[1] if preroll > 0 else 0.0

    def run(self, n_steps):
        """n_steps more control steps on every environment -> (env-steps/s, seconds)"""
        sims, n_env, threads = self.sims, self.n_env, self.threads
        actions = [self.rng.uniform(-1, 1, size=(n_steps, ad)) for _, ad in sims]

        def work(tid):
            for e in range(tid, n_env, threads):
                o = sims[e][0]
                for t in range(n_steps):
                    o.env_step(actions[e][t], N_SUBSTEPS)

        t0 = time.perf_counter()
        ths = [threading.Thread(target=work, args=(i,)) for i in range(threads)]
        for t in ths:
            t.start()
        for t in ths:
            t.join()
        dt = time.perf_counter() - t0
        return n_env * n_steps / dt, dt


# measured in the build container with tools/time_reference_on_shim.py (the unmodified reference Python stack stepping on the
# oracle through oracle/mujoco_shim); /root/reference does not exist on the GPU box, so this row is a recorded number
REFERENCE_STACK_ROW = {"value": 57.0, "unit": "env-steps/s", "cores": 1, "kind": "reference Python stack on the oracle shim",
                       "sample": "200 env.step of Lift/Panda OSC_POSE, 1 process, build container (8 cores), recorded - not re-measured here"}


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cfg = CONFIGS[args.config]
    cores, quota = host_threads()
    n_env = max(cores, 8)
    per_step = 8  # control steps per env per bench "step" (bounded sample of the workload)
    arm = CpuArm(cfg["parts"], n_env, cores, args.preroll)  # same protocol as the GPU arm: untimed pre-roll into the steady-state regime
    rates = []
    for i in range(args.warmup + args.steps):
        r, dt = arm.run(per_step)
        if i >= args.warmup:
            rates.append((r, dt))
    total_steps = sum(arm.n_env * per_step for _ in rates)
    total_t = sum(dt for _, dt in rates)
    value = total_steps / total_t
    sample = (f"{arm.n_env} envs x {per_step} control steps per bench step after {args.preroll} untimed pre-roll steps "
              f"({arm.preroll_s:.1f}s), {cores} threads (affinity {len(os.sched_getaffinity(0))}, cgroup quota {quota}), "
              f"oracle port (fp64 C) incl. controller")
    out = {
        "impl": "reference", "metric": cfg["metric"], "value": value, "unit": "env-steps/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * total_t / max(len(rates), 1),
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": cfg["workload"], "sample": sample},
        "cpu_baseline": {"value": value, "unit": "env-steps/s", "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": value, "unit": "env-steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(out))


# ------------------------------------------------------------------------------------------------ GPU arm
def device_timeline(part, groups):
    """Per-kernel launch durations of the CUDA-graph replay itself, from %globaltimer stamps written by a -DB2S_INSTR build of the
    library (robosuite_b200/variants/libb2s_instr.so) in a child process: events cannot subdivide a graph, and the eager
    timeline round 1 used includes host launch latency."""
    lib = os.path.join(ROOT, "robosuite_b200", "variants", "libb2s_instr.so")
    if not os.path.exists(lib):
        return None
    task, robot, ctrl, n = part
    env = dict(os.environ, B2S_LIB=lib, B2S_GROUPS=str(groups))
    try:
        r = subprocess.run([sys.executable, os.path.join(ROOT, "tools", "probe_instr.py"), task, robot, str(n), ctrl],
                           capture_output=True, text=True, timeout=600, env=env)
        return json.loads(r.stdout.strip().splitlines()[-1])
    except Exception:
        return None


DUMP_LIMIT_BYTES = 64 * 1024 * 1024


def dump_outputs(directory, arrays):
    """arrays {name: [rows, ...] ndarray} -> directory/<name>.npy in float32 / float64.  Above DUMP_LIMIT_BYTES in all, every
    array keeps the same fraction of its rows, chosen by a fixed seed, so that two builds dump the same environments."""
    import numpy as np

    arrays = {k: np.asarray(v, dtype=np.float64 if v.dtype == np.float64 else np.float32) for k, v in arrays.items()}
    total = sum(a.nbytes for a in arrays.values())
    os.makedirs(directory, exist_ok=True)
    for name, a in arrays.items():
        if total > DUMP_LIMIT_BYTES:
            keep = max(1, int(a.shape[0] * DUMP_LIMIT_BYTES / total))
            a = a[np.sort(np.random.default_rng(0).choice(a.shape[0], keep, replace=False))]
        np.save(os.path.join(directory, name + ".npy"), a)


def run_gpu(args):
    import torch
    import torch.distributed as dist

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device (the product path has no CPU fallback)")
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    import robosuite_b200 as suite
    from robosuite_b200.envs.base import load_task_model
    from robosuite_b200.parallel import allgather_obs, broadcast_model
    from robosuite_b200.wrappers import BatchedGymWrapper

    cfg = CONFIGS[args.config]
    parts = [(t, r, c, max(1, int(n * _SCALE))) for t, r, c, n in cfg["parts"]]
    dev = torch.device("cuda", local)
    clocks = ClockSampler(local) if rank == 0 else None
    envs = []
    for task, robot, ctrl, n in parts:
        # model constants: compiled once on rank 0, broadcast to the other ranks over NCCL (SURVEY.md section 8e)
        model = load_task_model(task, robot) if rank == 0 else None
        model = broadcast_model(model, src=0, device=dev) if world > 1 else model
        env = suite.make(task, robots=robot, num_envs=n, device=local, seed=1000 + rank, horizon=500,
                         controller_configs=controller_cfg(ctrl, robot), has_renderer=False, has_offscreen_renderer=False,
                         use_camera_obs=False, model=model, ignore_done=True)
        env.sim.set_mode(args.mode)
        envs.append(env)
    # one stream per task handle: the handles own separate constant-memory descriptor slots, so their graphs run concurrently
    streams = [torch.cuda.Stream(device=dev) for _ in envs] if len(envs) > 1 else [torch.cuda.current_stream(dev)]
    if len(envs) > 1:
        torch.cuda.synchronize()
        for e, st in zip(envs, streams):
            e.sim.set_stream(st)
    main_stream = torch.cuda.current_stream(dev)

    def fork():
        if len(envs) > 1:
            for st in streams:
                st.wait_stream(main_stream)

    def join():
        if len(envs) > 1:
            for st in streams:
                main_stream.wait_stream(st)
    N = sum(e.num_envs for e in envs)
    K, W = args.steps, args.warmup
    dtype = envs[0].dtype
    gen = torch.Generator(device=dev)
    gen.manual_seed(7 + rank)

    def rand_actions(count):
        return [torch.rand((count, e.num_envs, e.action_dim), generator=gen, device=dev, dtype=dtype) * 2 - 1 for e in envs]

    flush = torch.empty(256 * 1024 * 1024 // 4, dtype=torch.float32, device=dev)  # > 126 MB L2

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- pre-roll (untimed): random-action rollouts settle into their steady-state contact load only after ~50
    # control steps (cube lands, arms spread out, link-link hull tests start to fire); time THAT regime
    pre = rand_actions(args.preroll)
    def step_all(acts, i):
        fork()
        for e, a, st in zip(envs, acts, streams):
            with torch.cuda.stream(st):
                e.sim.env_step(a[i], N_SUBSTEPS)
        join()

    for i in range(args.preroll):
        step_all(pre, i)
    torch.cuda.synchronize()
    del pre
    actions = rand_actions(W + K)
    # ---- kernel-only timing (inputs resident in HBM)
    for i in range(W):
        step_all(actions, i)
    barrier()
    l0 = sum(e.sim.launch_count for e in envs)
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(K)]
    t_wall0 = time.time()
    for i in range(K):
        flush.zero_()  # L2 flush between timed iterations (outside the event pair)
        ev[i][0].record()
        step_all(actions, W + i)
        ev[i][1].record()
    barrier()
    t_wall1 = time.time()
    # what the last timed step left for its caller, copied before the e2e loop below steps the same environments again
    outputs = {}
    if args.dump_outputs and rank == 0:
        for (task, robot, _, _), e in zip(parts, envs):
            for k in ("qpos", "qvel", "qacc", "ctrl", "obs", "task_out"):
                outputs[f"{task}_{robot}_{k}"] = getattr(e.sim, k).cpu().numpy()
    launches = sum(e.sim.launch_count for e in envs) - l0
    ms = sum(a.elapsed_time(b) for a, b in ev)
    t = torch.tensor([ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms = float(t.item())
    value = world * N * K / (ms * 1e-3)
    warn = max(int(e.sim.warn.abs().max().item()) for e in envs)

    # ---- end to end through the public API (BatchedGymWrapper.step: the call an RL user makes) with HOST buffers (pinned):
    # action upload, 25-substep control step, reward, horizon-500 episodes with resets of finished environments inside step()
    # (episode phases staggered so that ~N/500 environments finish on every step), observation all-gather over NCCL when N>1,
    # observation + reward download - all inside the timed region
    wraps = [BatchedGymWrapper(e) for e in envs]
    for e in envs:
        e.ignore_done = False
        e.set_episode_steps(torch.randint(0, e.horizon, (e.num_envs,), generator=gen, device=dev))
    obs_dim = max(w.obs_dim for w in wraps)
    esz = 4 if dtype == torch.float32 else 8
    h_act = [torch.empty((K, e.num_envs, e.action_dim), dtype=dtype).pin_memory() for e in envs]
    for h, a in zip(h_act, actions):
        h.copy_(a[W:W + K].cpu())
    d_act = [torch.empty((e.num_envs, e.action_dim), dtype=dtype, device=dev) for e in envs]
    local_obs = torch.zeros((N, obs_dim), dtype=dtype, device=dev)  # task observations padded to the widest (config 5: 106)
    h_obs = torch.empty((N, obs_dim), dtype=dtype).pin_memory()
    h_rew = torch.empty((N,), dtype=dtype).pin_memory()
    d_rew = torch.empty((N,), dtype=dtype, device=dev)
    gathered = torch.empty((world * N, obs_dim), dtype=dtype, device=dev) if world > 1 else None
    h_all = torch.empty((world * N, obs_dim), dtype=dtype).pin_memory() if (world > 1 and rank == 0) else None
    n_resets = 0

    def e2e_step(i):
        """one end-to-end step: L2 flush, pinned-host action upload, wrapper.step (incl. in-step resets), obs all-gather, obs + reward download"""
        nonlocal n_resets
        flush.zero_()
        lo = 0
        fork()
        for w, ha, da, st in zip(wraps, h_act, d_act, streams):
            with torch.cuda.stream(st):
                da.copy_(ha[i], non_blocking=True)
                obs, rew, term, trunc, info = w.step(da)
                n = w.num_envs
                local_obs[lo:lo + n, :obs.shape[1]] = obs
                d_rew[lo:lo + n] = rew
            n_resets += int("final_observation" in info)
            lo += n
        join()
        if world > 1 and args.allgather_obs:
            allgather_obs(local_obs, gathered)  # per-step NCCL all-gather of observations (SURVEY.md section 8e)
            if rank == 0:
                h_all.copy_(gathered, non_blocking=True)
        h_obs.copy_(local_obs, non_blocking=True)
        h_rew.copy_(d_rew, non_blocking=True)

    # warm-up of THIS path (round 2 found the first wrapper / reset calls - lazily uploaded constants, first masked-reset launches -
    # inside the timed region: ~80 ms of one-time work spread over K steps, tools/probe_e2e.py)
    for i in range(W):
        e2e_step(i % K)
    n_resets = 0
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(K):
        e2e_step(i)
    e1.record()
    barrier()
    ms2 = e0.elapsed_time(e1)
    if args.dump_outputs and rank == 0:
        outputs["e2e_obs"], outputs["e2e_reward"] = h_obs.numpy().copy(), h_rew.numpy().copy()
        dump_outputs(args.dump_outputs, outputs)
    t2 = torch.tensor([ms2], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t2, op=dist.ReduceOp.MAX)
    e2e_value = world * N * K / (float(t2.item()) * 1e-3)
    h2d = sum(e.num_envs * e.action_dim for e in envs) * esz
    d2h = N * (obs_dim + 1) * esz + (world * N * obs_dim * esz if (world > 1 and args.allgather_obs) else 0)
    clk = clocks.stop(t_wall0, t_wall1) if clocks else None

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    # ---- roofline of the dominant kernel.  Pipeline mode: the merged tail kernel phase_kernel<R,5>; its launch duration comes
    # from %globaltimer stamps of the graph replay (device_timeline).  Algorithmic bytes of ONE launch = environments per launch
    # x per-substep state round trip (SURVEY.md section 8d), counted from the arrays the kernel really reads/writes in HBM.
    env0 = envs[0]
    m = env0.model
    per_env_in = (m.nq + 3 * m.nv + m.nu + 1 + 3 + 9 + 4 + 8 + env0.action_dim) * esz
    per_env_out = (m.nq + 3 * m.nv + m.nu + 1 + 3 + 9 + 4 + env0.obs_dim + 4 + 8) * esz + 4
    peak, how = _peaks()
    step_bytes = sum(e.num_envs for e in envs) * (per_env_in + per_env_out)
    achieved_step = step_bytes / (ms / K * 1e-3) / 1e9
    groups = int(os.environ.get("B2S_GROUPS", "8"))
    kernel, launch_us, envs_per_launch, launch_src = "step_kernel", ms / K * 1e3, env0.num_envs, "whole step (CUDA events)"
    alg_bytes = step_bytes
    tl = None
    if args.mode == 1 and world == 1 and not args.no_timeline:
        for e in envs[1:]:
            e.close()
        tl = device_timeline(parts[0], groups)
    if args.mode == 2:
        kernel = "unit_kernel<float> (persistent: every environment-substep of the control step as units on a ticket ring)"
    if args.mode == 1:
        envs_per_launch = env0.num_envs // groups
        kernel = "tail_kernel<float> (contact gather, constraint rows, Newton solve, integrate; small tier)"
        sub_in = (m.nq + 2 * m.nv + m.nu + 1 + 3 + 9 + 4) * esz   # qpos qvel qacc_ws ctrl time + controller state
        sub_out = (m.nq + 3 * m.nv + m.nu + 1) * esz                # qpos qvel qacc qacc_ws ctrl time
        alg_bytes = envs_per_launch * (sub_in + sub_out)
        if tl:
            launch_us, launch_src = tl["kernels"]["tail"]["mean_us"], "%globaltimer stamps of the graph replay (-DB2S_INSTR build, child process)"
        else:
            launch_us, launch_src = 0.62 * (ms / K * 1e3) / N_SUBSTEPS / max(1, groups // 2), "estimate: tail share 0.62 of the step (profiles/), 2 groups resident"
    achieved = alg_bytes / (launch_us * 1e-6) / 1e9
    traffic = None
    tp = os.path.join(ROOT, "profiles", "traffic.json")
    if os.path.exists(tp):
        try:
            with open(tp) as f:
                traffic = json.load(f).get("dram_bytes_per_launch")
        except Exception:
            traffic = None
    # ---- compute side (SURVEY.md section 8d "report both fractions"): issue slots and useful FP32 work
    compute = None
    if os.path.exists(INST_COUNTS):
        try:
            with open(INST_COUNTS) as f:
                ic = json.load(f).get(parts[0][0] + "_" + parts[0][1])
            sm_mhz = (clk or {}).get("sm_mhz") or 1965.0
            issue_peak = 148 * 4 * sm_mhz * 1e6                  # warp instructions / s (4 schedulers per SM)
            fp32_peak = 148 * 128 * 2 * sm_mhz * 1e6             # FLOP/s, non-tensor FP32 (128 FMA lanes per SM)
            substeps_s = value / world * N_SUBSTEPS * (parts[0][3] / N)
            compute = {"warp_inst_per_env_substep": ic["warp_inst_per_env_substep"], "issue_slots_frac": ic["warp_inst_per_env_substep"] * substeps_s / issue_peak,
                       "useful_flop_per_env_step": ic["useful_flop_per_env_step"], "fp32_frac": ic["useful_flop_per_env_step"] * (value / world) / fp32_peak,
                       "issue_peak_winst_s": issue_peak, "fp32_peak_flops": fp32_peak, "source": ic.get("source")}
        except Exception:
            compute = None
    # ---- CPU baseline on a bounded sample (rank 0, N=1 only)
    cpu = None
    if world == 1 and not args.no_cpu_baseline:
        cores, quota = host_threads()
        n_env, n_steps = max(cores, 8) * 2, 30
        arm = CpuArm(cfg["parts"], n_env, cores, args.preroll)
        r, dtc = arm.run(n_steps)
        cpu = {"value": r, "unit": "env-steps/s", "cores": cores, "kind": "port",
               "sample": f"{arm.n_env} envs x {n_steps} control steps ({dtc:.1f}s) after {args.preroll} untimed pre-roll steps "
                         f"({arm.preroll_s:.1f}s), oracle port (fp64 C) incl. controller, {cores} threads "
                         f"(affinity {len(os.sched_getaffinity(0))}, cgroup quota {quota})",
               "reference_python_stack": REFERENCE_STACK_ROW}
    out = {
        "metric": cfg["metric"], "value": value, "unit": "env-steps/s", "n_gpus": world, "steps": K, "warmup": W,
        "ms_per_step": ms / K, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32" if esz == 4 else "f64", "data": "synthetic",
        "config": {"workload": cfg["workload"], "baseline_config": args.config, "envs_per_gpu": N,
                   "tasks": [f"{t}/{r}/{c} x{n}" for t, r, c, n in parts], "substeps_per_step": N_SUBSTEPS,
                   "l2": "flushed (256 MiB memset) between timed iterations", "solver_warn_flags": warn,
                   "preroll_steps": args.preroll, "kernel_mode": ["fused", "pipeline", "unit-queue"][args.mode],
                   "e2e": f"BatchedGymWrapper.step, horizon 500 with staggered episode phases ({n_resets} in-step resets during the "
                          f"{K} timed steps), pinned-host action upload and obs+reward download, {W} warm-up steps of the same path, L2 flushed "
                          f"before every step (inside the timed region)",
                   "multi_gpu": "env shards independent; NCCL: model broadcast at start" + (", obs all-gather per step (e2e loop)" if args.allgather_obs else "")},
        "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                     "traffic": traffic, "peak_source": how, "kernel": kernel, "launch_us": launch_us, "launch_us_source": launch_src,
                     "envs_per_launch": envs_per_launch, "alg_bytes_per_launch": alg_bytes,
                     "whole_step": {"achieved": achieved_step, "frac": achieved_step / peak, "alg_bytes": step_bytes},
                     "compute": compute,
                     "timeline": ({"kernels_us": {k: v["mean_us"] for k, v in tl["kernels"].items()}, "gaps_us": tl["gaps_us"],
                                   "phase_kernels_running_hist": tl["phase_kernels_running_hist"],
                                   "solver_mean_niter": tl["solver"]["mean_niter"], "ls_evals_per_solve": tl["solver"]["ls_evals_per_solve"]}
                                  if tl else None),
                     "note": "per-environment state stays in shared memory / L2 between phases: algorithmic HBM traffic is tiny, "
                             "the kernels are latency / issue bound (DESIGN.md section 5): see `compute`"},
        "cpu_baseline": cpu,
        "e2e": {"value": e2e_value, "unit": "env-steps/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h},
        "gpu_launches": int(launches),
        "clocks": clk,
    }
    print(json.dumps(out))
    for e in envs:
        try:
            e.close()
        except Exception:
            pass
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200")
    ap.add_argument("--config", type=int, default=int(os.environ.get("B2S_BENCH_CONFIG", "2")), choices=sorted(CONFIGS))
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-timeline", action="store_true", help="skip the per-kernel device timeline (child process, INSTR build)")
    ap.add_argument("--preroll", type=int, default=100, help="untimed control steps before the timed region")
    ap.add_argument("--mode", type=int, default=int(os.environ.get("B2S_BENCH_MODE", "1")), help="0 fused kernel, 1 phase-kernel pipeline, 2 unit queue (persistent kernel)")
    ap.add_argument("--allgather-obs", type=int, default=1, help="N>1: all-gather observations over NCCL every e2e step")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write what the last timed step computed (rank 0: per task qpos, qvel, qacc, "
                    "ctrl, obs, task_out; the e2e loop's obs and reward) as DIR/<name>.npy")
    args = ap.parse_args()
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs is available for the GPU arm only")
    if args.warmup < 3 and args.impl != "reference":
        args.warmup = 3
    if args.impl == "reference":
        run_reference(args)
    else:
        run_gpu(args)


if __name__ == "__main__":
    main()
