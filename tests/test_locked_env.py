"""Batched dactyl/locked environment (robogym_b200/locked_env.py): goal generation, goal reward, multi-goal
bookkeeping, drop handling and reset -- against the answers of the reference's own LockedEnv driven through the mujoco_py
shim (recorded in tests/golden/ref_locked_*.npz by tools/make_reference_golden.py), by itself on the CPU oracle simulator,
and on the CUDA engine (gpu)."""
import math
import os
import sys

import numpy as np
import pytest

from robogym_b200 import modelblob

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(HERE, "stubs"))


def cpu_env(locked_blob, locked_names, nenv, **kw):
    import torch

    from oracle_batched_sim import OracleBatchedSim
    from robogym_b200.locked_env import BatchedLockedEnv

    m = modelblob.unpack(locked_blob)
    kw.setdefault("pool_size", 2)
    return BatchedLockedEnv(lambda n: OracleBatchedSim(locked_blob, n), m, locked_names, nenv, torch.device("cpu"), **kw)


def golden(name):
    """what robogym's own LockedEnv / wrappers answered on the mujoco_py shim (tools/make_reference_golden.py)"""
    return np.load(os.path.join(HERE, "golden", "ref_%s.npz" % name))


def _start_from(b, g):
    """the batched environment takes the reference environment's state after its reset"""
    import torch

    b.sim.qpos[0] = torch.tensor(g["qpos"]); b.sim.qvel[0] = torch.tensor(g["qvel"]); b.sim.ctrl[0] = torch.tensor(g["ctrl"])
    b.sim.pid[0] = torch.tensor(g["pid"]); b.sim.qacc_warmstart[0] = torch.tensor(g["warm"])
    b.goal_quat[0] = torch.tensor(g["goal_quat"]); b.prev_dist[0] = float(g["prev_dist"])
    tr = [int(x) for x in g["tracker"]]
    b.steps_since_last_goal[0], b.consecutive_success[0], b.successes_so_far[0], b.goals_so_far[0], b.success_pending[0] = tr


def test_parallel_quats_are_the_reference_set():
    from robogym_b200.locked_env import parallel_quats

    mine, ref = parallel_quats(), golden("locked_parallel_quats")["quats"]
    assert mine.shape == ref.shape == (24, 4)
    for q in ref:                       # same set of rotations (q and -q are the same rotation)
        assert min(np.minimum(np.abs(mine - q).max(1), np.abs(mine + q).max(1))) < 1e-9
    assert np.all(mine[:, 0] >= 0) and np.allclose(np.linalg.norm(mine, axis=1), 1.0)


def test_step_logic_matches_reference_env(locked_blob, locked_names):
    """Same state, goal and actions -> same observations, reward terms, done flags and tracker statistics as
    robogym's LockedEnv (no wrappers), through goal successes, a new-goal draw and a per-goal timeout."""
    import torch

    g = golden("locked_step_logic")
    b = cpu_env(locked_blob, locked_names, 1, stop_on_fall=False, auto_reset=False, max_timesteps_per_goal=6, successes_needed=2)
    _start_from(b, g)
    seen = dict(success=0, newgoal=0, timeout=0, trial=0)
    for k in range(len(g["done"])):
        if not np.isnan(g["goal_override"][k]).any():    # the goal put on top of the current orientation: the next step succeeds
            b.goal_quat[0] = torch.tensor(g["goal_override"][k])
        mo, mr, md, mi = b.step(g["action"][k][None], new_goals=g["new_goal"][k][None])
        for key in ("cube_pos", "cube_quat", "hand_angle", "fingertip_pos", "goal_quat", "qpos_goal", "qpos", "qvel"):
            assert np.abs(mo[key][0].numpy().ravel() - g["obs_" + key][k]).max() < 1e-7, (k, key)
        assert float(mo["is_goal_achieved"][0]) == float(g["is_goal_achieved"][k]), k
        assert np.abs(mr[0, :3].numpy() - g["rew"][k]).max() < 1e-7, (k, g["rew"][k], mr)
        assert bool(md[0]) == bool(g["done"][k]), k
        assert abs(float(mi["goal_dist"][0]) - g["goal_dist"][k]) < 1e-7
        for key in ("successes_so_far", "goals_so_far", "steps_since_last_goal"):
            assert int(mi[key][0]) == int(g[key][k]), (k, key)
        for key in ("trial_success", "sub_goal_is_successful"):
            assert bool(mi[key][0]) == bool(g[key][k]), (k, key)
        seen["success"] += bool(g["sub_goal_is_successful"][k]); seen["newgoal"] += bool(g["goal_reset"][k])
        seen["timeout"] += bool(g["done"][k] and not g["trial_success"][k]); seen["trial"] += bool(g["trial_success"][k])
    assert seen["success"] == 2 and seen["newgoal"] == 1 and seen["trial"] == 1, seen


def test_timeout_matches_reference_env(locked_blob, locked_names):
    g = golden("locked_timeout")
    b = cpu_env(locked_blob, locked_names, 1, stop_on_fall=False, auto_reset=False, max_timesteps_per_goal=3, successes_needed=2)
    _start_from(b, g)
    for k in range(3):
        _, mr, md, mi = b.step(np.zeros((1, 20)))
        assert bool(md[0]) == bool(g["done"][k]) and np.abs(mr[0, :3].numpy() - g["rew"][k]).max() < 1e-7
    assert list(g["done"]) == [False, False, True]


def test_reset_randomisation_matches_reference(locked_blob, locked_names):
    """InitialStatePool.randomize with the reference's draws reproduces LockedEnv._randomize_cube_initial_position.
    The random cube pose usually starts in penetration with the fingers, and resolving it amplifies round-off by many
    orders of magnitude per env-step, so the strict comparison uses ONE random-action step; the default ten steps are
    compared through what the reference uses them for (is the cube still on the palm)."""
    import torch

    g = golden("locked_reset_randomisation")
    for nrand, tol in ((1, 1e-6), (10, None)):
        b = cpu_env(locked_blob, locked_names, 1, pool_size=1, n_random_initial_steps=nrand)
        for seed in (3, 4):
            r = np.random.RandomState(seed)
            wig, quat, act = r.randn(3), r.randn(4), r.uniform(-1.0, 1.0, 20)
            ok = b.pool.randomize(torch.tensor(wig[None]), torch.tensor(quat[None]), torch.tensor(act[None]))
            key = "n%d_seed%d_" % (nrand, seed)
            if tol is not None:
                assert np.abs(b.pool.sim.qpos[0].numpy() - g[key + "qpos"]).max() < tol
                assert np.abs(b.pool.sim.qvel[0].numpy() - g[key + "qvel"]).max() < 1e-3
            else:
                assert np.abs(b.pool.sim.qpos[0, 14:].numpy() - g[key + "qpos"][14:]).max() < 5e-3     # hand joints
            assert bool(ok[0]) == bool(g[key + "on_palm"])


def test_cpu_env_success_timeout_and_autoreset(locked_blob, locked_names):
    """No reference needed: the bookkeeping invariants on the CPU oracle simulator."""
    import torch

    b = cpu_env(locked_blob, locked_names, 2, seed=0, max_timesteps_per_goal=3, successes_needed=2, n_random_initial_steps=1)
    obs = b.reset()
    assert obs["qpos"].shape == (2, 38) and b.episodes == 2 and int(b.goals_so_far.min()) == 1
    assert bool(b.fac.on_palm(b.sim.site_xpos).all())
    assert np.allclose(b.goal_quat.norm(dim=1).numpy(), 1.0) and float(b.goal_distance().max()) <= math.pi + 1e-9
    # env 0: goal on top of the current orientation -> success on the next step; env 1 runs into the timeout
    b.goal_quat[0] = b.sim.qpos[0, b.fac.cube_quat_idx]
    tot = torch.zeros(2, 4, dtype=torch.float64)
    for k in range(3):
        if k == 1:
            b.goal_quat[0] = b.sim.qpos[0, b.fac.cube_quat_idx]
        obs, rew, done, info = b.step(torch.zeros(2, 20))
        tot += rew
        if k == 0:
            assert bool(info["sub_goal_is_successful"][0]) and float(rew[0, 2]) == 5.0 and bool(info["goal_reset"][0]) and not bool(done[0])
            assert int(info["goals_so_far"][0]) == 2 and int(b.steps_since_last_goal[0]) == 0
        if k == 1:
            assert bool(info["trial_success"][0]) and bool(done[0])       # second success ends the episode ...
            assert int(b.successes_so_far[0]) == 0 and int(b.t[0]) == 0    # ... and the environment restarted
    assert bool(done[1]) and not bool(info["trial_success"][1])            # per-goal timeout after 3 steps
    assert b.episodes == 4 and float(tot[:, 0].abs().max()) == 0.0 and float(tot[0, 2]) == 10.0
    assert bool(b.fac.on_palm(b.sim.site_xpos).all())


@pytest.mark.gpu
def test_cuda_env_runs_and_autoresets():
    import torch

    from robogym_b200.locked_env import make_cuda_env

    env = make_cuda_env(512, seed=1, max_timesteps_per_goal=8, pool_size=256)
    obs = env.reset()
    assert obs["qpos"].shape == (512, 38) and obs["fingertip_pos"].shape == (512, 15)
    gen = torch.Generator(device=env.device); gen.manual_seed(0)
    ndone = 0
    ret = torch.zeros(512, device=env.device)
    for k in range(20):
        a = torch.rand(512, 20, device=env.device, generator=gen) * 2 - 1
        obs, rew, done, info = env.step(a)
        assert torch.isfinite(rew).all() and all(torch.isfinite(v).all() for v in obs.values())
        ndone += int(done.sum())
        ret += rew.sum(1)
        assert bool(env.fac.on_palm(env.sim.site_xpos)[done].all())      # restarted environments start on the palm
    assert ndone >= 512 and env.episodes == 512 + ndone                  # every environment hit the 8-step goal timeout at least once
    assert int(env.sim.warn.max()) == 0
    assert float(env.goal_distance().max()) <= math.pi + 1e-4


@pytest.mark.gpu
def test_cuda_env_with_domain_randomisation():
    """The locked.py:263-277 randomisation stack sampled per environment on the device: episodes start from pool states
    generated under their own parameters, parameters travel with the state on reset, timestep / wind change per step."""
    import torch

    from robogym_b200.locked_env import make_cuda_env

    env = make_cuda_env(256, seed=3, max_timesteps_per_goal=6, pool_size=128, randomize=True)
    env.reset()
    p = env.sim._params
    assert len(p) == 16 and float(p["dof_damping"].std(dim=0).max()) > 0 and float(p["opt_gravity"].std(dim=0).min()) > 0.1
    gen = torch.Generator(device=env.device); gen.manual_seed(0)
    damp0 = p["dof_damping"].clone()
    seen_ts = []
    for k in range(14):
        obs, rew, done, info = env.step(torch.rand(256, 20, device=env.device, generator=gen) * 2 - 1)
        assert torch.isfinite(rew).all() and all(torch.isfinite(v).all() for v in obs.values())
        seen_ts.append(env.timestep.clone())
    ts = torch.stack(seen_ts)
    assert float(ts.min()) >= 0.004 - 1e-7 and float(ts.max()) < 0.03 and float(ts.std()) > 1e-6
    assert env.episodes > 256 and not torch.equal(env.sim._params["dof_damping"], damp0)    # restarted envs got new parameters
    # randomised friction (up to 5x), gains, limits and timesteps occasionally fill the contact / row buffers (bits 0, 1) or
    # destabilise an environment, which the engine then resets like mj_step does (bit 2) -- MuJoCo warns in the same
    # situations; it must stay rare and nothing else may be flagged
    w = env.sim.warn
    assert float(((w & 4) != 0).float().mean()) < 0.05
    assert float(env.fac.on_palm(env.sim.site_xpos).float().mean()) > 0.8


@pytest.mark.gpu
def test_cuda_env_matches_oracle_env_teacher_forced(locked_blob, locked_names):
    """Rows f1/f2 of SURVEY 8(f) on the GPU tier, as parity rather than smoke: the batched environment on the CUDA engine
    beside the same environment on the fp64 oracle simulator, 60 env-steps, teacher-forced (before every step the CUDA side
    receives the oracle side's simulator state and bookkeeping; both get the same action and the same new goals).
    Observations, the reward terms, done flags and tracker statistics must agree: >= 95 % of the 960 environment-steps within
    2e-3 in every qpos-derived observation and in the goal reward (one env-step of fp32 vs fp64 contact dynamics; the rest
    are contact-mode switches, bounded at 0.1), discrete outcomes exactly except at a decision threshold."""
    import torch

    from robogym_b200.locked_env import STATE_FIELDS, make_cuda_env

    n, steps = 16, 60
    kw = dict(max_timesteps_per_goal=12, successes_needed=3, auto_reset=False, success_threshold=2.0)   # wide threshold: random play reaches goals
    ref = cpu_env(locked_blob, locked_names, n, seed=5, pool_size=n, **kw)
    env = make_cuda_env(n, seed=5, pool_size=n, **kw)
    ref.reset()
    env.reset()
    rng = np.random.RandomState(0)
    book = ("goal_quat", "prev_dist", "t", "steps_since_last_goal", "consecutive_success", "successes_so_far", "goals_so_far", "success_pending", "first_drop")
    worst = dict(qpos=0.0, reward=0.0)
    errs = []
    mism = 0
    for k in range(steps):
        for f in STATE_FIELDS:                       # teacher forcing: oracle state -> CUDA engine
            getattr(env.sim, f).copy_(getattr(ref.sim, f).to(device=env.device, dtype=getattr(env.sim, f).dtype))
        for f in book:
            getattr(env, f).copy_(getattr(ref, f).to(device=env.device, dtype=getattr(env, f).dtype))
        a = rng.uniform(-1, 1, (n, 20))
        g = ref.sample_goals(n)
        o1, r1, d1, i1 = ref.step(torch.as_tensor(a), new_goals=g)
        o2, r2, d2, i2 = env.step(torch.as_tensor(a, dtype=torch.float32, device=env.device), new_goals=g.to(env.device, torch.float32))
        e_obs = torch.stack([(o2[key].cpu().double() - o1[key]).abs().reshape(n, -1).max(1).values for key in ("cube_pos", "cube_quat", "hand_angle", "fingertip_pos", "qpos")]).max(0).values
        e_rew = (r2.cpu().double() - r1).abs().max(1).values
        worst["qpos"] = max(worst["qpos"], float(e_obs.max()))
        near = (i1["goal_dist"] - ref.success_threshold).abs() < 5e-3          # a success decided within fp32 noise of the threshold
        worst["reward"] = max(worst["reward"], float((r2.cpu().double() - r1)[~near].abs().max()) if (~near).any() else 0.0)
        same = (d2.cpu() == d1) & (i2["goal_achieved"].cpu() == i1["goal_achieved"]) & (i2["fell_down"].cpu() == i1["fell_down"]) & \
               (i2["successes_so_far"].cpu() == i1["successes_so_far"]) & (i2["goals_so_far"].cpu() == i1["goals_so_far"])
        big = e_obs > 2e-3                           # a contact-mode switch inside this env-step: its discrete outcomes may differ too
        mism += int((~same & ~near & ~big).sum())
        errs.append(torch.maximum(e_obs, torch.where(near, torch.zeros_like(e_rew), e_rew)))
    errs = torch.cat(errs)
    assert int(env.sim.warn.max()) == 0
    assert float((errs < 2e-3).double().mean()) >= 0.95, float((errs < 2e-3).double().mean())
    assert float(errs.median()) < 1e-4
    # (no bound on the single worst environment-step: without auto-reset a dropped cube keeps tumbling on the floor, and one
    #  env-step of that amplifies fp32/fp64 differences without limit; the 95 % / median statistics above are the claim)
    assert mism == 0
    assert int(ref.successes_so_far.sum()) > 0 and int(ref.goals_so_far.max()) > 1          # the run did exercise successes and goal switches


@pytest.mark.gpu
def test_randomised_env_with_reference_capacities_never_overflows():
    """VERDICT r1 item 4: the randomised stack (friction up to 5x, joint limits, gains, timesteps) used to fill the 32-contact /
    64-row buffers.  With run-time capacities at the reference's sizes for contacts (nconmax=100, assets.xml:6) and 160
    single-row elements, 200 env-steps at 2048 environments must not set the contact-full / rows-full bits at all."""
    import torch

    from robogym_b200 import engine
    from robogym_b200.locked_env import BatchedLockedEnv
    import json

    here = os.path.join(os.path.dirname(HERE), "robogym_b200")
    blob = open(os.path.join(here, "assets", "dactyl_locked.rgm"), "rb").read()
    names = json.load(open(os.path.join(here, "assets", "dactyl_locked.names.json")))
    model = engine.DeviceModel(blob, 0)
    dev = torch.device("cuda", 0)
    factory = lambda n: engine.BatchedSim(model, n, 10, outputs=("site_xpos", "act_force", "ncon", "warn"), contact_capacity=100, row_capacity=160, dofs_per_contact=24)
    env = BatchedLockedEnv(factory, model.host, names, 2048, dev, seed=3, pool_size=512, randomize=True)
    env.reset()
    gen = torch.Generator(device=dev); gen.manual_seed(0)
    worst = 0
    for k in range(200):
        env.step(torch.rand(2048, 20, device=dev, generator=gen) * 2 - 1)
        worst = max(worst, int(env.sim.ncon.max()))
    w = env.sim.warn
    assert int((w & 3).max()) == 0 and int((w & 32).max()) == 0, (int(w.max()), worst)
    assert worst <= 100


def test_action_latency_matches_the_reference_wrapper(locked_blob, locked_names):
    """RandomizedActionLatency (robogym/wrappers/randomizations.py:516-556, first entry of the locked.py:265-277 stack): with
    the same per-coordinate delays, the batched environment hands the simulation the same delayed actions and reports the
    same action_history / action_delay observations as the reference wrapper around the reference env."""
    import torch

    g = golden("locked_action_latency")
    b = cpu_env(locked_blob, locked_names, 2, stop_on_fall=False, auto_reset=False, action_latency=2)
    b.reset()
    assert b.action_delay.shape == (2, 20) and int(b.action_delay.max()) <= 2 and int(b.action_delay.min()) >= 0
    b.action_delay[0] = torch.tensor(g["delay"])
    b.action_delay[1] = 0
    sent = []
    orig = b.fac.denormalize_position_control
    b.fac.denormalize_position_control = lambda a, *args, **kw: (sent.append(a.clone()), orig(a, *args, **kw))[1]
    for k in range(len(g["action"])):
        a = g["action"][k]
        mo, _, _, _ = b.step(np.stack([a, a]))
        assert np.abs(sent[-1][0].numpy() - g["performed"][k]).max() < 1e-6, k      # env 0: the wrapper's delays
        assert np.abs(sent[-1][1].numpy() - a).max() < 1e-6                           # env 1: no delay
        assert np.abs(mo["action_history"][0].numpy() - g["action_history"][k]).max() < 1e-6
        assert np.array_equal(mo["action_delay"][0].numpy(), g["action_delay"][k])
    assert len(set(g["delay"])) > 1, "the fixture drew a single delay: nothing was exercised"
