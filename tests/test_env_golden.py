"""Environment-layer parity against the REFERENCE'S OWN Python code.

tests/golden/env_golden.npz was produced by tools/gen_env_golden.py: the unmodified robosuite stack (environments, robots,
composite/part controllers, observables, rewards) stepping on the CPU oracle through oracle/mujoco_shim.  Physics is shared
with the oracle by construction, so these vectors pin everything the reference does AROUND the engine calls: the substep
protocol, controller arithmetic, action scaling, gripper handling, observation layout/order/sampling and rewards.

CPU part: the oracle's C `o_env_step` must reproduce the reference stack's trajectory.
GPU part: robosuite_b200's env API must reproduce the reference stack's observations, rewards and trajectory."""
import os

import numpy as np
import pytest

from tests.util import ROOT, load

TASKS = ["Lift", "Door", "NutAssemblyRound", "PickPlace", "Stack"]


def _golden():
    return np.load(os.path.join(ROOT, "tests", "golden", "env_golden.npz"), allow_pickle=True)


def _model(task, G):
    m = load(task + "_Panda" if "_" not in task else ("Lift_Panda" if ("JOINT" in task or "OSC_" in task) else task))
    m.body_pos[:] = G[task + "/body_pos"]   # the reference writes sampled placements into the model (Door, visual objects)
    m.body_quat[:] = G[task + "/body_quat"]
    return m


@pytest.mark.parametrize("task", TASKS + ["Lift_Sawyer", "Stack_Sawyer", "Lift_JOINT_POSITION", "Lift_JOINT_TORQUE", "Lift_OSC_POSITION"])
def test_oracle_env_step_matches_reference_stack(task):
    """150 substeps of {step1, reference controllers, step2} vs the oracle's C controller + loop: <= 1e-6 on qpos
    (the residual is the reference's float32 round trip in transform_utils.quat2mat)"""
    from oracle.pyoracle import CtrlCfg as OCfg
    from oracle.pyoracle import Oracle
    from robosuite_b200 import controller_config as cc
    from robosuite_b200.mjcf.compiler import pack_model

    G = _golden()
    m = _model(task, G)
    o = Oracle(pack_model(m))
    sawyer = task.endswith("Sawyer")
    cfg = cc.load_composite_controller_config(None, "Sawyer") if sawyer else cc.default_composite_config()
    if "JOINT" in task or "OSC_POSITION" in task:  # part controller selected like demos/demo_control.py:99-103
        cfg = cc.refactor_composite_controller_config(cc.load_part_controller_config(task.split("_", 1)[1]), "Panda", ["right"])
    o.ctrl_setup(cc.resolve(m, cfg, OCfg, gripper="rethink" if sawyer else "panda"))
    o.qpos[:] = G[task + "/qpos0"]
    o.forward()
    o.ctrl_reset()
    for t, a in enumerate(G[task + "/actions"]):
        o.env_step(a, 25)
        assert np.abs(o.qpos - G[task + "/qpos"][t]).max() < 1e-6, (task, t)


@pytest.mark.gpu
@pytest.mark.parametrize("task", TASKS + ["Lift_JOINT_POSITION", "Lift_JOINT_TORQUE"])
def test_env_api_matches_reference_stack(task):
    """observations (layout, order, sampling instant, lagged object-in-gripper poses), rewards and state after every control
    step, fp32 engine vs the reference stack on the fp64 oracle"""
    import torch

    import robosuite_b200 as suite

    G = _golden()
    m = _model(task, G)
    n = 2
    kw = {}
    if "JOINT" in task:
        from robosuite_b200 import controller_config as cc

        kw["controller_configs"] = cc.refactor_composite_controller_config(cc.load_part_controller_config(task.split("_", 1)[1]), "Panda", ["right"])
    env = suite.make(task.split("_")[0], robots="Panda", num_envs=n, seed=0, horizon=1000, reward_shaping=True, model=m, **kw)
    obs = env.reset_to(G[task + "/qpos0"])
    for key, ref in (("object-state", G[task + "/obs0_object"]), ("robot0_proprio-state", G[task + "/obs0_proprio"])):
        got = obs[key].cpu().numpy().astype(np.float64)
        assert got.shape == (n, ref.shape[0]), (task, key, got.shape, ref.shape)
        assert np.abs(got - ref).max() < 2e-5, (task, "reset", key, int(np.abs(got[0] - ref).argmax()), float(np.abs(got - ref).max()))
    worst_o = worst_r = worst_q = 0.0
    for t, a in enumerate(G[task + "/actions"]):
        act = torch.as_tensor(np.tile(a, (n, 1)))
        obs, rew, done, info = env.step(act)
        for key, ref in (("object-state", G[task + "/obs_object"][t]), ("robot0_proprio-state", G[task + "/obs_proprio"][t])):
            got = obs[key].cpu().numpy().astype(np.float64)
            err = np.abs(got - ref)
            if key.startswith("robot0"):
                err[:, 28:35] /= max(1.0, np.abs(ref[28:35]).max())  # joint accelerations: relative
            worst_o = max(worst_o, float(err.max()))
            # (PickPlace: four mesh objects settling on the bin floor amplify fp32 rounding: measured 9.7e-4)
            assert err.max() < (3e-3 if task == "PickPlace" else 1e-3), (task, t, key, int(err[0].argmax()), float(err.max()))
        r = rew.cpu().numpy().astype(np.float64)
        worst_r = max(worst_r, float(np.abs(r - G[task + "/reward"][t]).max()))
        assert np.abs(r - G[task + "/reward"][t]).max() < 2e-4, (task, t, r, G[task + "/reward"][t])
        q = env.sim.qpos.cpu().numpy().astype(np.float64)
        worst_q = max(worst_q, float(np.abs(q - G[task + "/qpos"][t]).max()))
    print(task, "vs reference stack: obs %.2g reward %.2g qpos %.2g" % (worst_o, worst_r, worst_q))
    # PickPlace: four mesh objects settling on the bin floor amplify fp32 rounding (the oracle-vs-device tests show the same)
    assert worst_q < (2e-3 if task == "PickPlace" else 1e-4)
    assert int(env.sim.warn.abs().max()) == 0
    env.close()


CPU_CASES = TASKS + ["Lift_JOINT_POSITION", "Lift_JOINT_TORQUE", "Lift_OSC_POSITION", "Lift_Sawyer", "Stack_Sawyer"]


@pytest.mark.parametrize("task", CPU_CASES)
def test_env_host_layer_matches_reference_stack_on_cpu(task):
    """the HOST side of the environment layer (observation tables incl. the lagged entries, reset_to, reward / success code of
    every task class, action_spec, controller config resolution) driven by tests/oracle_sim.OracleSim instead of the CUDA
    engine: observations, rewards and states must equal what the reference stack produced on the same physics"""
    import torch

    import robosuite_b200 as suite
    from robosuite_b200 import controller_config as cc
    from tests.oracle_sim import OracleSim

    G = _golden()
    m = _model(task, G)
    robot = "Sawyer" if task.endswith("Sawyer") else "Panda"
    kw = {}
    if "JOINT" in task or "OSC_POSITION" in task:
        kw["controller_configs"] = cc.refactor_composite_controller_config(cc.load_part_controller_config(task.split("_", 1)[1]), "Panda", ["right"])
    env = suite.make(task.split("_")[0], robots=robot, num_envs=2, seed=0, horizon=1000, reward_shaping=True, model=m,
                     sim_cls=OracleSim, **kw)
    assert env.action_dim == G[task + "/actions"].shape[1]
    obs = env.reset_to(G[task + "/qpos0"])
    assert np.abs(obs["object-state"].numpy() - G[task + "/obs0_object"]).max() < 1e-6
    assert np.abs(obs["robot0_proprio-state"].numpy() - G[task + "/obs0_proprio"]).max() < 1e-6
    for t, a in enumerate(G[task + "/actions"]):
        obs, rew, done, info = env.step(torch.as_tensor(np.tile(a, (2, 1))))
        eo = np.abs(obs["object-state"].numpy() - G[task + "/obs_object"][t]).max()
        ep = np.abs(obs["robot0_proprio-state"].numpy() - G[task + "/obs_proprio"][t])
        ep[:, 28:35] /= max(1.0, np.abs(G[task + "/obs_proprio"][t][28:35]).max())
        assert eo < 2e-6 and ep.max() < 1e-5, (task, t, eo, ep.max(), int(ep[0].argmax()))
        assert np.abs(rew.numpy() - G[task + "/reward"][t]).max() < 1e-6, (task, t, rew, G[task + "/reward"][t])
        assert np.abs(env.sim.qpos.numpy() - G[task + "/qpos"][t]).max() < 1e-6
    env.close()


@pytest.mark.parametrize("task", ["Lift", "Stack", "NutAssemblyRound", "PickPlace", "Door", "Lift_sparse"])
def test_staged_rewards_grasp_and_success_match_reference_stack_on_cpu(task):
    """scripted reach / descend / close / lift episode recorded from the reference stack (tools/gen_reward_golden.py):
    the task classes' staged rewards, grasp detection (fingerpad-group contacts) and success flags, evaluated on the CPU
    stand-in sim, must follow the reference step by step (70 control steps, 1750 substeps of contact-rich motion)"""
    import torch

    import robosuite_b200 as suite
    from tests.oracle_sim import OracleSim

    G = np.load(os.path.join(ROOT, "tests", "golden", "reward_golden.npz"), allow_pickle=True)
    key = task
    kw = {}
    if task == "Lift_sparse":  # reward_shaping=False, reward_scale=3.0
        task, kw = "Lift", dict(reward_shaping=False, reward_scale=3.0)
    m = load(task + "_Panda")
    if task + "/body_pos" in G.files and key == task:  # Door: the placement the reference drew for this episode
        m.body_pos[:] = G[task + "/body_pos"]; m.body_quat[:] = G[task + "/body_quat"]
    mk = dict(reward_shaping=True)
    mk.update(kw)
    env = suite.make(task, robots="Panda", num_envs=1, seed=0, horizon=1000, model=m, sim_cls=OracleSim, **mk)
    G = {k[len(key) + 1:]: G[k] for k in G.files if k.startswith(key + "/")}
    G = {task + "/" + k: v for k, v in G.items()}
    env.reset_to(G[task + "/qpos0"])
    n_grasp = n_succ = 0
    for t, a in enumerate(G[task + "/actions"]):
        obs, rew, done, info = env.step(torch.as_tensor(a[None]))
        dq = np.abs(env.sim.qpos.numpy()[0] - G[task + "/qpos"][t]).max()
        tol = 1e-4 if task == "Door" else 1e-5
        if task in ("PickPlace", "Door") and dq >= tol:
            # PickPlace: the gripper ploughs through four loose objects; Door: the open gripper slides along the handle.  The
            # 1e-7 residual of the reference's float32 round trip is amplified step by step; the comparison covers the steps
            # before the two trajectories separate (Door: the whole latch rotation)
            assert t >= (15 if task == "PickPlace" else 55), (t, dq)
            break
        assert dq < tol, (task, t, dq)
        assert abs(float(rew[0]) - G[task + "/reward"][t]) < tol, (task, t, float(rew[0]), G[task + "/reward"][t])
        grasped = bool(int(env.sim.task_out[0, 5]) >> 3 & 1) if task == "PickPlace" else bool(env.sim.task_out[0, 2] > 0)  # Can = object 3
        assert task == "Door" or grasped == bool(G[task + "/grasp"][t]), (task, t)
        assert bool(env._check_success()[0]) == bool(G[task + "/success"][t]), (task, t)
        n_grasp += bool(G[task + "/grasp"][t]); n_succ += bool(G[task + "/success"][t])
    assert (n_grasp > 20 or task in ("NutAssemblyRound", "PickPlace", "Door")) and (task != "Lift" or n_succ > 10)
    env.close()


def test_batched_gym_wrapper_autoreset_on_cpu():
    """BatchedGymWrapper (wrappers/gym_wrapper.py:26-180 semantics) on the CPU stand-in sim: key order, 5-tuple, reset inside
    step, per-environment episode counters"""
    import torch

    import robosuite_b200 as suite
    from robosuite_b200.wrappers import BatchedGymWrapper
    from tests.oracle_sim import OracleSim

    n = 3
    env = BatchedGymWrapper(suite.make("Lift", robots="Panda", num_envs=n, seed=2, horizon=2, sim_cls=OracleSim))
    obs, info = env.reset(seed=7)
    assert obs.shape == (n, 60) and info == {} and env.obs_dim == 60
    d = env.env._get_observations()
    assert torch.equal(obs[:, :10], d["object-state"]) and torch.equal(obs[:, 10:], d["robot0_proprio-state"])
    low, high = env.action_low, env.action_high
    assert low.shape == (7,) and np.all(low == -1) and np.all(high == 1)
    # VectorEnv surface: per-environment spaces as gym_wrapper.py:70-85 builds them, batched along the leading axis
    assert env.single_observation_space.shape == (60,) and env.single_action_space.shape == (7,)
    assert env.observation_space.shape == (n, 60) and env.action_space.shape == (n, 7)
    assert np.all(np.isinf(env.single_observation_space.high)) and np.all(env.single_action_space.low == -1)
    assert env.single_action_space.contains(np.zeros(7, dtype=np.float32)) and not env.single_action_space.contains(np.full(7, 2.0, dtype=np.float32))
    assert env.action_space.contains(env.action_space.sample())
    obs, rew, term, trunc, info = env.step(torch.zeros((n, 7)))
    assert not bool(term.any()) and "final_observation" not in info
    obs, rew, term, trunc, info = env.step(torch.zeros((n, 7)))
    assert bool(term.all()) and not bool(trunc.any()) and info["final_observation"].shape == (n, 60)
    assert int(env.env.timestep.max()) == 0 and not bool(env.env.done.any())
    assert torch.allclose(obs[:, 2], torch.full((n,), 0.83, dtype=obs.dtype), atol=5e-3)  # cube back on the table
    obs, rew, term, trunc, info = env.step(torch.zeros((n, 7)))
    assert not bool(term.any())
    env.close()


@pytest.mark.parametrize("task", ["Lift", "Stack", "NutAssemblyRound", "PickPlace", "Door"])
def test_reset_distribution_matches_reference_stack(task):
    """qpos after reset: the batched samplers (torch, one draw per environment) against 250 resets of the reference stack
    (tools/gen_reset_golden.py): coordinates the reference never varies are reproduced exactly, varying ones stay inside the
    reference's observed range (plus a sampling margin) and have matching mean / spread"""
    import robosuite_b200 as suite
    from tests.oracle_sim import OracleSim

    G = np.load(os.path.join(ROOT, "tests", "golden", "reset_golden.npz"), allow_pickle=True)
    lo, hi, mean, std = (G[task + "/" + k] for k in ("min", "max", "mean", "std"))
    n = 400
    env = suite.make(task, robots="Panda", num_envs=n, seed=123, sim_cls=OracleSim)
    q = env._sample_reset_state(n).cpu().numpy()
    env.close()
    if task == "NutAssemblyRound":  # the unused square nut: the reference parks it at (10, 10, 10) after sampling it
        a = env.obj_qadr["SquareNut"]
        assert np.allclose(q[:, a:a + 3], 10.0) and np.allclose(lo[a:a + 3], 10.0)
    fixed = std < 1e-9
    assert np.abs(q[:, fixed] - mean[fixed]).max() < 1e-9, (task, np.nonzero(fixed)[0][np.abs(q[:, fixed] - mean[fixed]).max(0) > 1e-9])
    var = ~fixed
    span = hi - lo
    gauss = np.zeros_like(var)
    gauss[env._ref_joint_pos_indexes] = True  # arm joints: N(init, 0.02^2) - unbounded, compare moments only
    rng_like = var & ~gauss
    margin = 0.08 * span + 1e-6                 # 250 reference draws do not reach the ends of a uniform range exactly
    assert np.all(q[:, rng_like] >= (lo - margin)[rng_like]) and np.all(q[:, rng_like] <= (hi + margin)[rng_like]), task
    # same centre and spread (quaternion components of a uniform yaw included)
    assert np.abs(q[:, var].mean(0) - mean[var]).max() < 0.25 * std[var].max() + 0.15 * span[var].max(), task
    ratio = q[:, var].std(0) / std[var]
    assert np.all(ratio > 0.7) and np.all(ratio < 1.4), (task, ratio)


def test_door_placement_is_drawn_per_environment_and_reset():
    """door.py:303-318, 417-427: x in [0.07, 0.09], y in [-0.01, 0.01], yaw in [-pi/2 - 0.25, -pi/2] relative to table_offset, redrawn at
    every reset of the environment; a masked reset leaves the other environments' doors where they are; the welded frame body follows"""
    import torch

    import robosuite_b200 as suite
    from tests.oracle_sim import OracleSim

    n = 64
    env = suite.make("Door", robots="Panda", num_envs=n, seed=7, sim_cls=OracleSim)
    env.reset()
    P, Q = (t.clone() for t in env.door_pose)
    tx, ty, tz = env.table_offset
    x, y = P[:, 0] - tx, P[:, 1] - ty
    yaw = 2 * torch.atan2(Q[:, 3], Q[:, 0])
    assert float(x.min()) >= 0.07 - 1e-9 and float(x.max()) <= 0.09 + 1e-9 and float(x.std()) > 0.003
    assert float(y.min()) >= -0.01 - 1e-9 and float(y.max()) <= 0.01 + 1e-9 and float(y.std()) > 0.003
    assert float(yaw.min()) >= -np.pi / 2 - 0.25 - 1e-9 and float(yaw.max()) <= -np.pi / 2 + 1e-9 and float(yaw.std()) > 0.04
    assert torch.allclose(P[:, 2], torch.full((n,), tz + 0.3, dtype=P.dtype)) and float(Q[:, 1:3].abs().max()) == 0
    obs = env._get_observations()
    bn = env.model.names["body"]
    off = obs["door_pos"] - P  # Door_door sits at a fixed offset in the (rotated) frame: |offset| is the same everywhere
    assert float((off.norm(dim=1) - off.norm(dim=1)[0]).abs().max()) < 1e-9 and float((off[0] - off[1]).abs().max()) > 1e-4
    mask = torch.zeros(n, dtype=torch.bool); mask[::2] = True
    env.reset(mask=mask, host_mask=mask.numpy())
    P2, _ = env.door_pose
    assert torch.equal(P2[1::2], P[1::2]) and float((P2[::2] - P[::2]).abs().max()) > 1e-4
    env.close()
    pinned = suite.make("Door", robots="Panda", num_envs=2, seed=7, sim_cls=OracleSim, door_placement=(0.08, 0.0, -np.pi / 2 - 0.125))
    assert pinned.door_pose is None
    pinned.close()
