"""The batched dual-simulation arm controller (robogym_b200/rearrange_arm.py, SURVEY 8(f) row 4) beside the UNMODIFIED reference
environment: `robogym.envs.rearrange.blocks.make_env` with ControlMode.TCP_ROLL_YAW + TcpSolverMode.MOCAP_IK (the mode SURVEY
8(d) row 4 names: 3 tool translations + roll / yaw + gripper) ran on the mujoco_py shim with the oracle as engine and its states
were recorded (tests/golden/rearrange_arm.json, tests/golden/ref_arm_*.npz); the batched controller runs on oracle-backed
stand-ins of its two BatchedSims built from the SAME compiled models and started from the SAME states.  Both take the same
actions: every env-step must leave the same main-simulation and solver-simulation state
(fp64 on both sides, so the comparison is tight -- any difference is a difference in the control logic).  The GPU test runs the
controller on two real BatchedSims (CUDA) against the oracle stand-ins, teacher-forced."""
import os
import sys

import numpy as np
import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
for p in (os.path.join(HERE, "stubs"),):
    if p not in sys.path:
        sys.path.insert(0, p)

MAX_POSITION_CHANGE = float(np.float32(0.1))    # the reference stores the parameter as a float32
ASSETS = os.path.join(HERE, "..", "robogym_b200", "assets")


def _recorded(name):
    """what the reference environment's two simulations did on the mujoco_py shim (tools/make_reference_golden.py)"""
    return np.load(os.path.join(HERE, "golden", "ref_%s.npz" % name))


def _state_of(g, prefix, sim):
    """one recorded simulation state in the layout _load_state takes"""
    st = {k: g[prefix + k] for k in ("qpos", "qvel", "ctrl", "warm", "body_xpos", "body_xquat")}
    st["pid"] = g[prefix + "pid"][:sim.pid.shape[1]]
    if sim.mocap_pos is not None:
        st.update(mocap_pos=g[prefix + "mocap_pos"], mocap_quat=g[prefix + "mocap_quat"])
    return st


@pytest.mark.parametrize("reset_controller_error", [True, False])
def test_batched_controller_steps_like_the_reference_environment(reset_controller_error):
    """Two environments in one batch from the reference environment's recorded reset state: every env-step reproduces the
    recorded main / solver states and controls (fp64 on both sides), and the batch rows agree bit for bit."""
    import torch

    from oracle_generic_sim import OracleGenericSim
    from robogym_b200.rearrange_arm import BatchedTcpArmController

    fx, blobs = _fixture()
    rec = fx["reset_error_%s" % str(reset_controller_error).lower()]
    assert rec["reset_controller_error"] == reset_controller_error and len(rec["actions"][0]) == 6
    nenv = 2
    main = OracleGenericSim(blobs[0], nenv, rec["nsub_main"])
    solver = OracleGenericSim(blobs[1], nenv, rec["nsub_solver"])
    assert main.model.host["nu"] == 7 and list(main.model.host["actuator_user0"]) == [1, 1, 1, 1, 1, 1, 0]    # cascaded-PI arm, PID gripper
    assert solver.model.host["nmocap"] == 1 and solver.model.host["neq"] == 2        # mocap weld + gripper coupling
    _load_state(main, rec["main0"]); _load_state(solver, rec["solver0"])
    ctl = BatchedTcpArmController(main, solver, MAX_POSITION_CHANGE, reset_controller_error=reset_controller_error)
    assert ctl.action_dim == 6
    worst = 0.0
    for k, a in enumerate(rec["actions"]):
        ctl.step(torch.tensor([a, a], dtype=torch.float32))
        em = np.abs(main.qpos[0].numpy() - rec["main_qpos"][k]).max()
        es = np.abs(solver.qpos[0].numpy() - rec["solver_qpos"][k]).max()
        ec = np.abs(main.ctrl[0].numpy() - rec["main_ctrl"][k]).max()
        emo = np.abs(solver.mocap_pos[0].numpy() - np.asarray(rec["solver_mocap_pos"][k])).max()
        worst = max(worst, em, es, ec, emo)
        assert em < 1e-9 and es < 1e-9 and ec < 1e-9 and emo < 1e-9, (k, em, es, ec, emo)
        assert torch.equal(main.qpos[0], main.qpos[1])
    assert worst < 1e-9 and int(main.warn.max()) == 0


def test_wrist_mode_with_its_alignment_axis_steps_like_the_reference_environment():
    """ControlMode.TCP_WRIST: one tool rotation (about the vertical), the commanded orientation re-aligned with the vertical
    axis every step (MocapSolver.align_axis)."""
    import torch

    from oracle_generic_sim import OracleGenericSim
    from robogym_b200.rearrange_arm import BatchedTcpArmController

    g = _recorded("arm_wrist")
    _, blobs = _fixture()
    main = OracleGenericSim(blobs[0], 1, int(g["nsub_main"]))
    solver = OracleGenericSim(blobs[1], 1, int(g["nsub_solver"]))
    _load_state(main, _state_of(g, "main0_", main))
    _load_state(solver, _state_of(g, "solver0_", solver))
    ctl = BatchedTcpArmController(main, solver, MAX_POSITION_CHANGE, dof_dims=("pitch",), align_axis="pitch")
    assert ctl.action_dim == g["action"].shape[1] == 5
    for k, a in enumerate(g["action"]):
        ctl.step(torch.tensor(a[None]))
        em = np.abs(main.qpos[0].numpy() - g["main_qpos"][k]).max()
        es = np.abs(solver.qpos[0].numpy() - g["solver_qpos"][k]).max()
        eq = np.abs(solver.mocap_quat[0].numpy() - g["solver_mocap_quat"][k]).max()
        assert em < 1e-9 and es < 1e-9 and eq < 1e-9, (k, em, es, eq)


def test_controller_reset_reseats_the_mocap_weld_like_the_reference():
    import torch

    from oracle_generic_sim import OracleGenericSim
    from robogym_b200.rearrange_arm import BatchedTcpArmController

    g = _recorded("arm_reset")
    _, blobs = _fixture()
    main = OracleGenericSim(blobs[0], 1, int(g["nsub_main"]))
    solver = OracleGenericSim(blobs[1], 1, int(g["nsub_solver"]))
    _load_state(main, _state_of(g, "main0_", main))
    # the solver stand-in starts from its MODEL state (qpos0, compiled weld pose); reset() must bring it to the reference's
    solver.model.set_field("eq_data", np.tile([0.1, 0.0, 0.0, 1.0, 0.0, 0.0, 0.0], int(solver.model.host["neq"])))
    ctl = BatchedTcpArmController(main, solver, MAX_POSITION_CHANGE)
    ctl.reset()
    weld = [i for i in range(int(solver.model.host["neq"])) if int(solver.model.host["eq_type"][i]) == 1]
    assert np.allclose(np.asarray(solver.model.host["eq_data"]).reshape(int(solver.model.host["neq"]), -1)[weld, :7], [0, 0, 0, 1, 0, 0, 0])
    assert np.abs(solver.qpos[0, ctl.arm_qadr_solver].numpy() - g["main0_qpos"][ctl.arm_qadr_main]).max() == 0
    tcp = solver.model.name2id("body", "robot0:gripper_tcp")
    assert torch.equal(solver.mocap_pos[0, 0], solver.body_xpos[0, tcp]) and torch.equal(solver.mocap_quat[0, 0], solver.body_xquat[0, tcp])
    assert np.abs(solver.mocap_pos[0, 0].numpy() - g["solver_mocap_pos"][0]).max() < 2e-3   # the reference's helper arm has drifted a little by then


# ---- the same comparison from the committed fixture (tools/make_rearrange_arm_fixture.py): no reference needed, and the GPU tier
def _fixture():
    import json

    fx = json.load(open(os.path.join(HERE, "golden", "rearrange_arm.json")))
    blobs = [open(os.path.join(ASSETS, n + ".rgm"), "rb").read() for n in ("rearrange_blocks5_tcp", "rearrange_solver_arm")]
    return fx, blobs


def _load_state(sim, st, rows=slice(None)):
    t = sim.torch
    f = lambda v: t.as_tensor(np.asarray(v), dtype=sim.qpos.dtype).to(sim.qpos.device)
    sim.qpos[rows] = f(st["qpos"]); sim.qvel[rows] = f(st["qvel"]); sim.ctrl[rows] = f(st["ctrl"]); sim.pid[rows] = f(st["pid"])
    sim.qacc_warmstart[rows] = f(st["warm"])
    if sim.mocap_pos is not None:
        sim.mocap_pos[rows] = f(st["mocap_pos"]); sim.mocap_quat[rows] = f(st["mocap_quat"])
    sim.body_xpos[rows] = f(st["body_xpos"]); sim.body_xquat[rows] = f(st["body_xquat"])


@pytest.mark.parametrize("key", ["reset_error_true", "reset_error_false"])
def test_controller_replays_the_recorded_reference_rollout(key):
    """fp64 stand-ins, free-running for 16 env-steps from the recorded reset state: the reference environment's recorded main /
    solver states are reproduced to 1e-9 at every step."""
    import torch

    from oracle_generic_sim import OracleGenericSim
    from robogym_b200.rearrange_arm import BatchedTcpArmController

    fx, blobs = _fixture()
    rec = fx[key]
    main = OracleGenericSim(blobs[0], 1, rec["nsub_main"])
    solver = OracleGenericSim(blobs[1], 1, rec["nsub_solver"])
    _load_state(main, rec["main0"]); _load_state(solver, rec["solver0"])
    ctl = BatchedTcpArmController(main, solver, rec["max_position_change"], reset_controller_error=rec["reset_controller_error"])
    for k, a in enumerate(rec["actions"]):
        ctl.step(torch.tensor([a], dtype=torch.float32))
        assert np.abs(main.qpos[0].numpy() - rec["main_qpos"][k]).max() < 1e-9, k
        assert np.abs(main.ctrl[0].numpy() - rec["main_ctrl"][k]).max() < 1e-9, k
        assert np.abs(solver.qpos[0].numpy() - rec["solver_qpos"][k]).max() < 1e-9, k
        assert np.abs(solver.mocap_pos[0].numpy() - np.asarray(rec["solver_mocap_pos"][k])).max() < 1e-9, k
    # the policy's actions reached the arm: the tool moved by centimetres, the arm joints by tenths of a radian
    q0, q1 = np.asarray(rec["main0"]["qpos"]), main.qpos[0].numpy()
    assert np.abs(q1[:6] - q0[:6]).max() > 0.05


def _follow(make_sims, key, device="cpu"):
    """shared by the emulation and the CUDA tier: the fp32 engine beside the fp64 stand-ins"""
    import torch

    from oracle_generic_sim import OracleGenericSim
    from robogym_b200.rearrange_arm import BatchedTcpArmController

    fx, blobs = _fixture()
    rec = fx[key]
    main, solver, nenv, sync = make_sims(blobs, rec)
    ctl = BatchedTcpArmController(main, solver, rec["max_position_change"], reset_controller_error=rec["reset_controller_error"])
    omain = OracleGenericSim(blobs[0], 1, rec["nsub_main"])
    osolver = OracleGenericSim(blobs[1], 1, rec["nsub_solver"])
    octl = BatchedTcpArmController(omain, osolver, rec["max_position_change"], reset_controller_error=rec["reset_controller_error"])
    _load_state(omain, rec["main0"]); _load_state(osolver, rec["solver0"])

    def push(dst, src):
        for n in ("qpos", "qvel", "ctrl", "pid", "qacc_warmstart", "mocap_pos", "mocap_quat", "body_xpos", "body_xquat"):
            s = getattr(src, n, None)
            if s is not None:
                getattr(dst, n).copy_(s.to(torch.float32).expand_as(getattr(dst, n)))

    # teacher-forced: every env-step starts from the oracle stand-in's state
    err_arm, err_obj, err_sol = [], [], []
    for k, a in enumerate(rec["actions"]):
        push(main, omain); push(solver, osolver)
        ctl.step(torch.tensor([a] * nenv, dtype=torch.float32, device=device))
        octl.step(torch.tensor([a], dtype=torch.float32))
        sync()
        q, qo = main.qpos.cpu().numpy().astype(np.float64), omain.qpos[0].numpy()
        err_arm.append(np.abs(q[0, :6] - qo[:6]).max()); err_obj.append(np.abs(q[0, 8:] - qo[8:]).max())
        err_sol.append(np.abs(solver.qpos[0].cpu().numpy() - osolver.qpos[0].numpy()).max())
        assert np.array_equal(q[0], q[nenv - 1])
    assert int(main.warn.max()) == 0 and int(solver.warn.max()) == 0
    # free-running from the recorded reset state
    _load_state(omain, rec["main0"]); _load_state(osolver, rec["solver0"])
    push(main, omain); push(solver, osolver)
    err_free = []
    for k, a in enumerate(rec["actions"]):
        ctl.step(torch.tensor([a] * nenv, dtype=torch.float32, device=device))
        sync()
        err_free.append(np.abs(main.qpos[0].cpu().numpy().astype(np.float64)[:6] - np.asarray(rec["main_qpos"][k])[:6]).max())
    return dict(arm=max(err_arm), obj_median=float(np.median(err_obj)), obj_max=max(err_obj), solver=max(err_sol), free=max(err_free)), main


@pytest.mark.parametrize("key", ["reset_error_true"])
def test_emulated_kernels_follow_the_recorded_reference_rollout(key):
    """The kernel source in CPU emulation (fp32) under the same controller: what the CUDA tier asserts, checked without a GPU."""
    from emu_generic_sim import EmuGenericSim

    def make(blobs, rec):
        return (EmuGenericSim(blobs[0], 2, rec["nsub_main"], contact_capacity=64, row_capacity=160), EmuGenericSim(blobs[1], 2, rec["nsub_solver"]), 2, lambda: None)

    err, _ = _follow(make, key)
    assert err["arm"] < 1e-4 and err["solver"] < 2e-4 and err["obj_median"] < 1e-4 and err["obj_max"] < 2e-3 and err["free"] < 2e-3, err


@pytest.mark.gpu
@pytest.mark.parametrize("key", ["reset_error_true", "reset_error_false"])
def test_cuda_controller_follows_the_recorded_reference_rollout(key):
    """Both simulations on the CUDA engine (two BatchedSims, two launches per env-step, the hand-off on the device).
    Teacher-forced: every env-step starts from the oracle stand-in's state; the fp32 engine must land within 1e-4 rad of the
    fp64 arm joints and track the blocks.  Free-running for the 16 recorded steps: the arm stays within 2e-3 rad of the
    reference environment's recorded trajectory (the cascaded-PI loop is contracting), and batch rows agree bit for bit."""
    import torch

    from robogym_b200 import build, engine

    build.build()
    models = {}

    def make(blobs, rec):
        nenv = 4
        mm, ms = engine.DeviceModel(blobs[0], 0), engine.DeviceModel(blobs[1], 0)
        models["main"] = mm
        main = engine.BatchedSim(mm, nenv, rec["nsub_main"], outputs=("body_xpos", "body_xquat", "ncon", "warn", "sensordata", "contact"), contact_capacity=64, row_capacity=160)
        solver = engine.BatchedSim(ms, nenv, rec["nsub_solver"], outputs=("body_xpos", "body_xquat", "warn"))
        return main, solver, nenv, torch.cuda.synchronize

    err, main = _follow(make, key, device="cuda:0")
    assert err["arm"] < 2e-4 and err["solver"] < 4e-4 and err["obj_median"] < 2e-4 and err["obj_max"] < 4e-3 and err["free"] < 4e-3, err
    mm = models["main"]
    # force / torque sensors of the tool flange are live on the device (robot/ur16e/mujoco/joint_controlled_arm.py:35-45)
    sd = main.sensordata[0].cpu().numpy()
    adr = mm.host["sensor_adr"][mm.name2id("sensor", "toolhead_force")]
    assert np.isfinite(sd).all() and 2.0 < np.linalg.norm(sd[adr:adr + 3]) < 100.0      # about the gripper's weight (0.5 kg), give or take its motion
    # contact-based observations from the device's contact list (rearrange_contacts.py; the logic is checked against the reference's
    # functions in tests/test_rearrange_contacts.py): blocks rest on the table, nothing touches the gripper in this rollout
    from robogym_b200.rearrange_contacts import BatchedRearrangeContacts

    qc = BatchedRearrangeContacts(main, num_objects=5)
    assert mm.id2name("geom", qc.table_plane) == "table_collision_plane" and bool(qc.is_robot[qc.wrist_sphere]) and int(qc.is_gripper.sum()) >= 9
    assert int(main.ncon.min()) >= 5                                   # at least the blocks' table contacts
    assert not bool(qc.gripper_table_contact().any()) and qc.object_gripper_contact().shape == (4, 5, 2)
    assert not bool(qc.wrist_cam_collisions()["any"].any())


# ---- the reference's recorded controller response (robogym/envs/rearrange/tests/test_rearrange_sim.py:135-230), on the BATCHED controller
IMPULSE_CASES = [(True, 0.165, 0.036, 5), (False, 0.05, 0.0363, 12), (True, 0.1, 0.022, 5), (False, 0.03, 0.022, 12)]


def _impulse_response(make_sims, device="cpu", sync=lambda: None):
    """test_mocap_ik_impulse_response restated on BatchedTcpArmController: from the environment's reset state (the committed fixture),
    2 zero actions, one full-scale action on one tool axis, 40 zero actions; all 4 parameter sets x 3 axes run as ONE batch of 12
    environments.  Returns the tool trajectories [12, 43, 3] (relative to the first sample)."""
    import torch

    from robogym_b200.rearrange_arm import BatchedTcpArmController

    fx, blobs = _fixture()
    out = []
    for rce, mpc, _, _ in IMPULSE_CASES:
        rec = fx["reset_error_true" if rce else "reset_error_false"]
        main, solver = make_sims(blobs, rec, 3)
        _load_state(main, rec["main0"]); _load_state(solver, rec["solver0"])
        ctl = BatchedTcpArmController(main, solver, float(np.float32(mpc)), reset_controller_error=rce)
        tcp = main.model.name2id("body", "robot0:gripper_tcp")
        traj = []
        # the reference test steps the environment below its action discretisation but THROUGH SmoothActionWrapper(alpha=0.3)
        # (rearrange/common/base.py:987; wrappers/util.py:142-218): a bias-corrected exponential moving average of the actions
        alpha = 0.3 ** ((main.n_substeps * float(main.model.host["opt_timestep"][0])) / 0.08)
        ema, t_ema = np.zeros((3, 6)), 0
        for k in range(43):
            raw = np.zeros((3, 6))
            if k == 2:
                raw[0, 0] = raw[1, 1] = raw[2, 2] = 1.0     # environment d gets the impulse on tool axis d
            ema = ema * alpha + (1.0 - alpha) * raw
            t_ema += 1
            a = torch.tensor((ema / (1.0 - alpha ** t_ema)).astype(np.float32), device=device)
            ctl.step(a)
            sync()
            traj.append(main.body_xpos[:, tcp].detach().cpu().numpy().astype(np.float64).copy())
        traj = np.stack(traj, axis=1)
        out.append(traj - traj[:, :1])
    return np.concatenate(out, axis=0)


def _assert_impulse(traj, tol=1e-3):
    for c, (rce, mpc, want, rise) in enumerate(IMPULSE_CASES):
        for d in range(3):
            x = traj[3 * c + d, :, d]
            assert abs(x[-1] - want) < tol, (rce, mpc, d, x[-1], want)                   # steady-state displacement, the reference's number
            assert abs(x[2 + rise]) > 0.9 * x[-1], (rce, mpc, d, x[2 + rise], x[-1])    # 90 % within `rise` steps of the impulse


def test_recorded_impulse_response_on_the_batched_controller_fp64_and_emulated():
    """The reference's real-MuJoCo numbers for its controller (tool displacement 0.036 / 0.0363 / 0.022 / 0.022 m +- 1e-3, 90 % rise
    within 5 / 12 steps) asserted on the batched dual-simulation controller: on the fp64 stand-ins and on the fp32 kernel logic."""
    from emu_generic_sim import EmuGenericSim
    from oracle_generic_sim import OracleGenericSim

    _assert_impulse(_impulse_response(lambda blobs, rec, n: (OracleGenericSim(blobs[0], n, rec["nsub_main"]), OracleGenericSim(blobs[1], n, rec["nsub_solver"]))))
    _assert_impulse(_impulse_response(lambda blobs, rec, n: (EmuGenericSim(blobs[0], n, rec["nsub_main"], contact_capacity=64, row_capacity=160),
                                                              EmuGenericSim(blobs[1], n, rec["nsub_solver"]))))


@pytest.mark.gpu
def test_recorded_impulse_response_on_cuda():
    """the same on the CUDA engine: the reference's recorded displacements, asserted on the product path"""
    import torch

    from robogym_b200 import build, engine

    build.build()

    def make(blobs, rec, n):
        main = engine.BatchedSim(engine.DeviceModel(blobs[0], 0), n, rec["nsub_main"], outputs=("body_xpos", "body_xquat", "warn"), contact_capacity=64, row_capacity=160)
        solver = engine.BatchedSim(engine.DeviceModel(blobs[1], 0), n, rec["nsub_solver"], outputs=("body_xpos", "body_xquat", "warn"))
        return main, solver

    _assert_impulse(_impulse_response(make, device="cuda:0", sync=torch.cuda.synchronize))


def test_batched_controller_steps_like_the_reference_ycb_environment():
    """BASELINE configs[4]: the reference's ycb environment (8 mesh objects of its own draw, the first starting_seed whose
    placement succeeds; its main simulation is the committed rearrange_ycb8_tcp asset) beside the batched controller."""
    import torch

    from oracle_generic_sim import OracleGenericSim
    from robogym_b200.rearrange_arm import BatchedTcpArmController

    g = _recorded("arm_ycb")
    blob = open(os.path.join(ASSETS, "rearrange_ycb8_tcp.rgm"), "rb").read()
    main = OracleGenericSim(blob, 1, int(g["nsub_main"]))
    solver = OracleGenericSim(_fixture()[1][1], 1, int(g["nsub_solver"]))
    assert (main.model.host["nq"], main.model.host["nv"], main.model.host["nu"]) == (64, 56, 7)
    _load_state(main, _state_of(g, "main0_", main))
    _load_state(solver, _state_of(g, "solver0_", solver))
    ctl = BatchedTcpArmController(main, solver, MAX_POSITION_CHANGE)
    for k, a in enumerate(g["action"]):
        ctl.step(torch.tensor(a[None]))
        em = np.abs(main.qpos[0].numpy() - g["main_qpos"][k]).max()
        es = np.abs(solver.qpos[0].numpy() - g["solver_qpos"][k]).max()
        assert em < 1e-9 and es < 1e-9, (k, em, es)
