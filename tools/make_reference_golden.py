"""Generate tests/golden/ref_*.npz: what the tests compare against from the ORIGINAL robogym project, recorded once.

Runs the unmodified robogym code (a checkout named by ROBOGYM_REFERENCE) on the mujoco_py shim with the fp64 oracle as engine
and stores its answers -- states, observations, rewards, wrapper draws, contact queries -- so that the tests replay them
without the original project.  Each function below records the reference side of one test; the test next to its name
holds the batched side.

    ROBOGYM_REFERENCE=<robogym checkout> python tools/make_reference_golden.py [case ...]
"""
import os
import subprocess
import sys
from collections import OrderedDict

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.abspath(os.path.join(HERE, ".."))
GOLDEN = os.path.join(ROOT, "tests", "golden")
ASSETS = os.path.join(ROOT, "robogym_b200", "assets")
MAX_POSITION_CHANGE = float(np.float32(0.1))


def _setup():
    ref = os.environ.get("ROBOGYM_REFERENCE")
    if not ref or not os.path.isdir(os.path.join(ref, "robogym")):
        raise SystemExit("set ROBOGYM_REFERENCE to a checkout of the original robogym project")
    for p in (os.path.join(ROOT, "tests", "stubs"), os.path.join(ROOT, "tests"), ref, ROOT):
        if p not in sys.path:
            sys.path.insert(0, p)
    import robogym_b200.mujoco_py_shim as shim

    shim.install()
    from oracle_engine import OracleEngine

    shim.set_engine_factory(OracleEngine)


def _asset(name):
    return open(os.path.join(ASSETS, name + ".rgm"), "rb").read()


def _same_model(blob, name):
    """the recorded environment runs the committed asset: the tests replay on it"""
    assert blob == _asset(name), "the environment's compiled model is not robogym_b200/assets/%s.rgm" % name


def _state(mj, prefix):
    d = mj.data
    w = len(d.userdata)
    out = {prefix + "qpos": d.qpos, prefix + "qvel": d.qvel, prefix + "ctrl": d.ctrl, prefix + "pid": d.userdata[:w], prefix + "warm": d.qacc_warmstart,
           prefix + "body_xpos": d.body_xpos, prefix + "body_xquat": d.body_xquat}
    if mj.model.nmocap:
        out.update({prefix + "mocap_pos": d.mocap_pos, prefix + "mocap_quat": d.mocap_quat})
    return {k: np.array(v, dtype=np.float64, copy=True) for k, v in out.items()}


# ---------------------------------------------------------------- tests/test_locked_env.py
def locked_parallel_quats():
    from robogym.envs.dactyl.common import cube_utils

    return dict(quats=np.array(cube_utils.PARALLEL_QUATS, dtype=np.float64))


def _locked_start(env):
    d = env.mujoco_simulation.mj_sim.data
    tr = env.multi_goal_tracker
    return dict(qpos=d.qpos.copy(), qvel=d.qvel.copy(), ctrl=d.ctrl.copy(), pid=d.userdata[:60].copy(), warm=d.qacc_warmstart.copy(),
                goal_quat=np.array(env._goal["cube_quat"], dtype=np.float64), prev_dist=float(env._previous_goal_distance["cube_quat"]),
                tracker=np.array([tr._steps_since_last_goal, tr._consecutive_steps_with_success, tr._successes_so_far, tr._goals_so_far,
                                  tr._success_and_no_goal_reset], dtype=np.int64))


LOCKED_OBS = ("cube_pos", "cube_quat", "hand_angle", "fingertip_pos", "goal_quat", "qpos_goal", "qpos", "qvel")
LOCKED_INFO = ("successes_so_far", "goals_so_far", "steps_since_last_goal", "trial_success", "sub_goal_is_successful", "goal_reset")


def locked_step_logic():
    from robogym.envs.dactyl.locked import make_simple_env

    env = make_simple_env(starting_seed=5, constants=dict(max_timesteps_per_goal=6, successes_needed=2))
    env.reset()
    d = env.mujoco_simulation.mj_sim.data
    out = _locked_start(env)
    rng = np.random.RandomState(1)
    rec = {k: [] for k in ("action", "goal_override", "new_goal", "rew", "done", "goal_dist", "is_goal_achieved") + LOCKED_INFO}
    rec.update({"obs_" + k: [] for k in LOCKED_OBS})
    for k in range(16):
        g = np.full(4, np.nan)
        if k in (2, 6):   # put the goal on top of the current orientation: the next step succeeds
            g = d.qpos[env.mujoco_simulation.qpos_idxs["cube_rotation"]].copy()
            env._goal["cube_quat"] = g
            env._goal["qpos_goal"][env.mujoco_simulation.qpos_idxs["cube_rotation"]] = g
        a = rng.uniform(-1, 1, 20)
        obs, rew, done, info = env.step(a)
        rec["action"].append(a); rec["goal_override"].append(g); rec["new_goal"].append(np.array(env._goal["cube_quat"], dtype=np.float64))
        for key in LOCKED_OBS:
            rec["obs_" + key].append(np.array(obs[key], dtype=np.float64).ravel())
        rec["is_goal_achieved"].append(float(np.array(obs["is_goal_achieved"]).ravel()[0]))
        rec["rew"].append(np.array(rew, dtype=np.float64)); rec["done"].append(bool(done)); rec["goal_dist"].append(info["goal_dist"]["cube_quat"])
        for key in LOCKED_INFO:
            rec[key].append(int(info.get(key, False)))
        if done:
            break
    out.update({k: np.array(v) for k, v in rec.items()})
    return out


def locked_timeout():
    from robogym.envs.dactyl.locked import make_simple_env

    env = make_simple_env(starting_seed=2, constants=dict(max_timesteps_per_goal=3, successes_needed=2))
    env.reset()
    out = _locked_start(env)
    rew, done = [], []
    for k in range(3):
        _, r, dn, _ = env.step(np.zeros(20))
        rew.append(np.array(r, dtype=np.float64)); done.append(bool(dn))
    out.update(rew=np.array(rew), done=np.array(done))
    return out


def locked_reset_randomisation():
    from robogym.envs.dactyl.locked import make_simple_env

    env = make_simple_env(starting_seed=11)
    out = {}
    for nrand in (1, 10):
        env.parameters.n_random_initial_steps = nrand
        for seed in (3, 4):
            env._random_state.seed(seed)
            env.mujoco_simulation.reset()
            env._randomize_cube_initial_position()
            d = env.mujoco_simulation.mj_sim.data
            key = "n%d_seed%d_" % (nrand, seed)
            out.update({key + "qpos": d.qpos.copy(), key + "qvel": d.qvel.copy(), key + "on_palm": np.array(bool(env.mujoco_simulation.is_cube_on_palm()))})
    return out


def locked_action_latency():
    from robogym.envs.dactyl.locked import make_simple_env
    from robogym.wrappers import randomizations as rz

    inner = make_simple_env(starting_seed=3)
    performed = []
    real_step = inner.step

    def spy(action):
        performed.append(np.array(action, copy=True))
        return real_step(action)

    inner.step = spy
    w = rz.RandomizedActionLatency(inner, max_delay=2)
    w.reset()
    delay = np.array(w._action_delay).copy()
    rng = np.random.RandomState(0)
    rec = dict(action=[], performed=[], action_history=[], action_delay=[])
    for k in range(6):
        a = rng.uniform(-1, 1, 20)
        obs, _, _, _ = w.step(a)
        rec["action"].append(a); rec["performed"].append(performed[-1])
        rec["action_history"].append(np.array(obs["action_history"], dtype=np.float64)); rec["action_delay"].append(np.array(obs["action_delay"]))
    out = {k: np.array(v) for k, v in rec.items()}
    out["delay"] = delay
    return out


# ---------------------------------------------------------------- tests/test_obs_noise.py
def obs_noise():
    import gym
    from gym.spaces import Box, Dict

    from robogym.wrappers.randomizations import RandomizeObservationWrapper
    from robogym_b200.obs_noise import LOCKED_LEVELS
    from test_obs_noise import NENV, NSTEPS, WIDTHS, clean_observations

    clean = clean_observations()

    class Recorder:
        def __init__(self, seed):
            self.rs, self.log = np.random.RandomState(seed), []

        def randn(self, *shape):
            v = self.rs.randn(*shape); self.log.append(("randn", v.copy())); return v

        def uniform(self, lo, hi, size=None):
            v = self.rs.uniform(lo, hi, size=size); self.log.append(("uniform", v.copy())); return v

    class FakeEnv(gym.Env):
        def __init__(self, e):
            self.e, self.k = e, 0
            self._random_state = Recorder(100 + e)
            self.observation_space = Dict({k: Box(-np.inf, np.inf, (w,), np.float64) for k, w in WIDTHS.items()})
            self.action_space = Box(-1, 1, (1,), np.float64)

        @property
        def unwrapped(self):
            return self

        def reset(self):
            self.k = 0
            return OrderedDict((k, v.copy()) for k, v in clean[0][self.e].items())

        def step(self, a):
            self.k += 1
            return OrderedDict((k, v.copy()) for k, v in clean[self.k][self.e].items()), 0.0, False, {}

    envs = [RandomizeObservationWrapper(FakeEnv(e), levels=LOCKED_LEVELS) for e in range(NENV)]
    ref = [[w.reset() for w in envs]]
    for s in range(NSTEPS):
        ref.append([w.step(np.zeros(1))[0] for w in envs])
    logs = [w.unwrapped._random_state.log for w in envs]
    kinds = [kind for kind, _ in logs[0]]
    assert all([kind for kind, _ in log] == kinds for log in logs)
    out = dict(draw_kind=np.array(kinds), draw_size=np.array([v.size for _, v in logs[0]]),
               draws=np.stack([np.concatenate([v.ravel() for _, v in log]) for log in logs]))
    for k in WIDTHS:
        out["noisy_" + k] = np.array([[ref[s][e]["noisy_" + k] for e in range(NENV)] for s in range(NSTEPS + 1)], dtype=np.float64)
    return out


# ---------------------------------------------------------------- tests/test_batched_facade.py
def facade():
    from robogym.envs.dactyl.locked import make_env
    from robogym.utils.sensor_utils import check_occlusion

    from robogym_b200 import modelblob

    env = make_env(starting_seed=3)
    env.reset()
    env = env.unwrapped
    sim = env.mujoco_simulation.mj_sim
    robot = env.mujoco_simulation.shadow_hand
    # make_env's wrappers randomise the model: store the fields that differ from the committed asset
    mine, asset = modelblob.unpack(sim.model._cm.blob()), modelblob.unpack(_asset("dactyl_locked"))
    assert sim.model._cm.names == modelblob.unpack_names(_asset("dactyl_locked"))
    model = {"model_" + k: np.array(v) for k, v in mine.items() if np.array(v).tobytes() != np.array(asset[k]).tobytes()}
    rng = np.random.RandomState(0)
    keys = ("cube_pos", "cube_quat", "hand_angle", "fingertip_pos")
    rec = {k: [] for k in ("action", "qpos_before", "ctrl_rel", "ctrl_abs", "site_xpos", "qpos", "qvel", "actuator_force", "effort", "on_palm",
                           "contact", "ncon", "occluded") + keys}
    for k in range(12):
        action = rng.uniform(-1, 1, 20)
        rec["action"].append(action); rec["qpos_before"].append(sim.data.qpos.copy())
        want_rel = robot.denormalize_position_control(action, relative_action=True)
        rec["ctrl_rel"].append(want_rel); rec["ctrl_abs"].append(robot.denormalize_position_control(action, relative_action=False))
        robot.set_position_control(want_rel)
        env.mujoco_simulation.step()
        obs = env.observe()
        for key in keys:
            rec[key].append(np.array(obs[key], dtype=np.float64).ravel())
        rec["site_xpos"].append(sim.data.site_xpos.copy()); rec["qpos"].append(sim.data.qpos.copy()); rec["qvel"].append(sim.data.qvel.copy())
        rec["actuator_force"].append(sim.data.actuator_force.copy()); rec["effort"].append(robot.observe().actuator_effort())
        rec["on_palm"].append(bool(env.mujoco_simulation.is_cube_on_palm()))
        con = np.zeros((64, 4))
        for i in range(sim.data.ncon):
            c = sim.data.contact[i]
            con[i] = (c.geom1, c.geom2, c.dist, c.dim)
        rec["contact"].append(con); rec["ncon"].append(sim.data.ncon)
        rec["occluded"].append(np.array(check_occlusion(sim, dist_cutoff=-1e-4)).astype(np.int64))
    return dict({k: np.array(v) for k, v in rec.items()}, **model)


# ---------------------------------------------------------------- tests/test_randomization.py
def range_rules():
    from robogym.envs.dactyl.locked import make_simple_env
    from robogym.wrappers import randomizations as rz

    env = make_simple_env(starting_seed=0)
    sim = env.unwrapped.sim
    jw = rz.RandomizedJointLimitWrapper(env)
    tw = rz.RandomizedTendonRangeWrapper(env)
    jw._orig_value = np.array(jw._get_field(sim), copy=True)
    tw._orig_value = np.array(tw._get_field(sim), copy=True)
    out = {}
    for seed in (0, 1, 2):
        r = np.random.RandomState(seed)
        zj, zt = r.randn(len(sim.model.joint_names), 2), r.randn(sim.model.ntendon, 2)
        jw._random_noises = lambda n, z=zj: z
        jw._set_field(sim)
        env.unwrapped._random_state = type("R", (), {"randn": staticmethod(lambda *s, z=zt: z)})()
        tw._set_field(sim)
        key = "seed%d_" % seed
        out.update({key + "zj": zj, key + "zt": zt, key + "jnt_range": np.array(sim.model.jnt_range, dtype=np.float64).ravel(),
                    key + "actuator_ctrlrange": np.array(sim.model.actuator_ctrlrange, dtype=np.float64).ravel(),
                    key + "tendon_range": np.array(sim.model.tendon_range, dtype=np.float64).ravel()})
    return out


# ---------------------------------------------------------------- tests/test_rearrange_contacts.py, tests/test_rearrange_arm.py
def _rearrange_env(reset_controller_error=True, wrist=False):
    from robogym.envs.rearrange.blocks import make_env
    from robogym.robot.robot_interface import ControlMode, TcpSolverMode

    env = make_env(parameters=dict(n_random_initial_steps=0, simulation_params=dict(num_objects=5),
                                   robot_control_params=dict(control_mode=ControlMode.TCP_WRIST if wrist else ControlMode.TCP_ROLL_YAW,
                                                             tcp_solver_mode=TcpSolverMode.MOCAP_IK, arm_reset_controller_error=reset_controller_error,
                                                             max_position_change=MAX_POSITION_CHANGE)), starting_seed=0)
    env.reset()
    return env.unwrapped


def rearrange_contacts():
    from test_rearrange_contacts import contact_actions

    env = _rearrange_env()
    sim = env.mujoco_simulation
    _same_model(sim.mj_sim.model._cm.blob(), "rearrange_blocks5_tcp")
    tcp = sim.mj_sim.data.get_body_xpos("robot0:gripper_tcp").copy()
    adr = sim.mj_sim.model.get_joint_qpos_addr("object0:joint")[0]
    sim.mj_sim.data.qpos[adr:adr + 2] = tcp[:2]
    sim.forward()
    rec = dict(contact=[], ncon=[], table=[], obj=[])
    cams = None
    for a in contact_actions():
        env.step(a)
        d = sim.mj_sim.data
        con = np.zeros((64, 3))
        con[:, :2] = -1
        for i in range(d.ncon):
            c = d.contact[i]
            con[i] = (c.geom1, c.geom2, c.dist)
        rec["contact"].append(con); rec["ncon"].append(d.ncon)
        rec["table"].append(bool(sim.get_gripper_table_contact())); rec["obj"].append(np.array(sim.get_object_gripper_contact(pad=False)))
        want_cam = sim.get_wrist_cam_collisions()
        cams = cams or {n: [] for n in want_cam}
        for n, v in want_cam.items():
            cams[n].append(bool(v))
    out = {k: np.array(v) for k, v in rec.items()}
    out.update({"cam_" + n: np.array(v) for n, v in cams.items()})
    return out


def arm_wrist():
    env = _rearrange_env(wrist=True)
    main_mj = env.mujoco_simulation.mj_sim
    arm = env.robot.robots[0]
    solver_mj = arm.controller_arm.mj_sim
    assert type(arm.controller_arm).__name__ == "FreeWristTcpArm" and env.action_space.shape[0] == 5
    _same_model(main_mj.model._cm.blob(), "rearrange_blocks5_tcp")
    _same_model(solver_mj.model._cm.blob(), "rearrange_solver_arm")
    out = dict(_state(main_mj, "main0_"), **_state(solver_mj, "solver0_"))
    out.update(nsub_main=main_mj.nsubsteps, nsub_solver=solver_mj.nsubsteps)
    rng = np.random.RandomState(1)
    rec = dict(action=[], main_qpos=[], solver_qpos=[], solver_mocap_quat=[])
    for k in range(8):
        a = rng.uniform(-1, 1, 5).astype(np.float32)
        env.step(a)
        rec["action"].append(a); rec["main_qpos"].append(main_mj.data.qpos.copy()); rec["solver_qpos"].append(solver_mj.data.qpos.copy())
        rec["solver_mocap_quat"].append(np.array(solver_mj.data.mocap_quat, dtype=np.float64))
    out.update({k: np.array(v) for k, v in rec.items()})
    return out


def arm_reset():
    env = _rearrange_env()
    main_mj = env.mujoco_simulation.mj_sim
    solver_mj = env.robot.robots[0].controller_arm.mj_sim
    _same_model(main_mj.model._cm.blob(), "rearrange_blocks5_tcp")
    _same_model(solver_mj.model._cm.blob(), "rearrange_solver_arm")
    out = _state(main_mj, "main0_")
    out.update(nsub_main=main_mj.nsubsteps, nsub_solver=solver_mj.nsubsteps, solver_mocap_pos=np.array(solver_mj.data.mocap_pos, dtype=np.float64))
    return out


def arm_ycb():
    from robogym.envs.rearrange.ycb import make_env
    from robogym.robot.robot_interface import ControlMode, TcpSolverMode

    env = make_env(parameters=dict(n_random_initial_steps=0, simulation_params=dict(num_objects=8, max_num_objects=8),
                                   robot_control_params=dict(control_mode=ControlMode.TCP_ROLL_YAW, tcp_solver_mode=TcpSolverMode.MOCAP_IK,
                                                             max_position_change=MAX_POSITION_CHANGE)),
                   constants=dict(stabilize_objects=False), starting_seed=1)
    env.reset()
    env = env.unwrapped
    main_mj = env.mujoco_simulation.mj_sim
    solver_mj = env.robot.robots[0].controller_arm.mj_sim
    _same_model(main_mj.model._cm.blob(), "rearrange_ycb8_tcp")
    _same_model(solver_mj.model._cm.blob(), "rearrange_solver_arm")
    out = dict(_state(main_mj, "main0_"), **_state(solver_mj, "solver0_"))
    out.update(nsub_main=main_mj.nsubsteps, nsub_solver=solver_mj.nsubsteps)
    rng = np.random.RandomState(2)
    rec = dict(action=[], main_qpos=[], solver_qpos=[])
    for k in range(5):
        a = rng.uniform(-1, 1, 6).astype(np.float32)
        env.step(a)
        rec["action"].append(a); rec["main_qpos"].append(main_mj.data.qpos.copy()); rec["solver_qpos"].append(solver_mj.data.qpos.copy())
    out.update({k: np.array(v) for k, v in rec.items()})
    return out


# ---------------------------------------------------------------- tests/test_full_cube_plumbing.py
def full_cube():
    from robogym.envs.dactyl.full_perpendicular import make_simple_env

    env = make_simple_env(starting_seed=0)
    ms = env.mujoco_simulation
    _same_model(ms.mj_sim.model._cm.blob(), "dactyl_full_perpendicular")
    ms.reset()
    ms.forward()
    d = ms.mj_sim.data
    out = {"start_" + k: np.array(v, dtype=np.float64, copy=True) for k, v in
           (("qpos", d.qpos), ("qvel", d.qvel), ("ctrl", d.ctrl), ("pid", d.userdata), ("warm", d.qacc_warmstart))}
    ctrl = []
    for _ in range(5):
        c = ms.shadow_hand.denormalize_position_control(np.zeros(20))
        ms.shadow_hand.set_position_control(c)
        ms.step()
        ctrl.append(np.array(d.ctrl, dtype=np.float64))
    out.update(ctrl=np.array(ctrl), nsubsteps=ms.mj_sim.nsubsteps, qpos=d.qpos.copy(), qvel=d.qvel.copy(), ncon=d.ncon,
               on_palm=bool(ms.is_cube_on_palm()))
    return out


CASES = [locked_parallel_quats, locked_step_logic, locked_timeout, locked_reset_randomisation, locked_action_latency, obs_noise, facade,
         range_rules, rearrange_contacts, arm_wrist, arm_reset, arm_ycb, full_cube]


def main(names):
    if not names:       # every case in a process of its own: the reference's environments share module-level state
        for f in CASES:
            subprocess.check_call([sys.executable, os.path.abspath(__file__), f.__name__])
        return
    _setup()
    for f in CASES:
        if f.__name__ in names:
            out = f()
            path = os.path.join(GOLDEN, "ref_%s.npz" % f.__name__)
            np.savez_compressed(path, **{k: np.array(v) for k, v in out.items()})
            print("%-28s %7d bytes" % (f.__name__, os.path.getsize(path)), flush=True)


if __name__ == "__main__":
    main(sys.argv[1:])
