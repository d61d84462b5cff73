"""Device-side domain randomisation (robogym_b200/randomization.py): the batched mj_setConst against the host
compiler's, the range-perturbation rules against the reference wrappers' own code, the sampled distributions,
and -- on the GPU -- that the sampled rows reach the engine."""
import os

import numpy as np
import pytest

from robogym_b200 import mjcf, modelblob

HERE = os.path.dirname(os.path.abspath(__file__))


class NumpyRand:
    def __init__(self, seed, torch):
        self.r, self.torch = np.random.RandomState(seed), torch

    def randn(self, n, k):
        return self.torch.tensor(self.r.randn(n, k))

    def uniform(self, lo, hi, n, k):
        return self.torch.tensor(self.r.uniform(lo, hi, (n, k)))

    def randint(self, hi, n):
        return self.torch.tensor(self.r.randint(hi, size=n))


@pytest.fixture(scope="module")
def rnd(locked_blob, locked_names):
    import torch

    from robogym_b200.randomization import LockedRandomizer

    m = modelblob.unpack(locked_blob)
    return m, LockedRandomizer(m, locked_names, NumpyRand(0, torch), torch, torch.device("cpu"), torch.float64)


def test_batched_constants_match_host_set_const(rnd):
    import torch

    m, R = rnd
    rng = np.random.RandomState(1)
    scale = rng.uniform(0.5, 1.5, (3, m["nbody"], 1))
    scale[0] = 1.0
    rows = torch.tensor((m["body_inertia"].reshape(1, -1, 3) * scale).reshape(3, -1))
    got = R.constants.derive(rows)
    for e in range(3):
        mm = {k: (np.array(v, copy=True) if isinstance(v, np.ndarray) else v) for k, v in m.items()}
        mm["body_inertia"] = rows[e].numpy().copy()
        mjcf.set_const(mm)
        for key in ("dof_invweight0", "body_invweight0", "tendon_invweight0", "opt_meaninertia"):
            a, b = got[key][e].numpy().ravel(), np.asarray(mm[key]).ravel()
            assert np.abs(a - b).max() <= 1e-9 * max(1.0, np.abs(b).max()), (e, key)
    # the unscaled row reproduces the constants stored in the compiled model
    for key in ("dof_invweight0", "body_invweight0", "tendon_invweight0", "opt_meaninertia"):
        assert np.allclose(got[key][0].numpy().ravel(), np.asarray(m[key]).ravel(), rtol=1e-6, atol=1e-12), key


def test_sampled_rows_have_the_wrappers_ranges(rnd, locked_names):
    m, R = rnd
    n = 400
    p = R.sample(n)
    assert set(p) == set(R.EPISODE_PARAMS)
    for k, v in p.items():
        assert v.shape == (n, np.asarray(m[k]).size), k
    r = lambda k: (p[k].numpy() / np.where(np.asarray(m[k]).ravel() == 0, 1, np.asarray(m[k]).ravel()))
    bi = r("body_inertia").reshape(n, -1, 3)
    nz = m["body_inertia"].reshape(-1, 3)[:, 0] > 0
    assert bi[:, nz].min() >= 0.5 and bi[:, nz].max() <= 1.5 and np.allclose(bi[:, nz, 0], bi[:, nz, 1])   # one factor per body
    fr = r("geom_friction").reshape(n, -1, 3)
    rg, cg = R.robot_geoms.numpy(), R.cube_geoms.numpy()
    assert 0.7 <= fr[:, rg, 0].min() and fr[:, rg, 0].max() <= 1.3 and 0.5 <= fr[:, rg, 1].min() and fr[:, rg, 2].max() <= 1.5
    assert 0.5 <= fr[:, cg, 0].min() and fr[:, cg, 0].max() <= 1.5 and 0.2 <= fr[:, cg, 1].min() and fr[:, cg, 2].max() <= 5.0
    assert np.ptp(fr[:, rg, 0], axis=1).max() < 1e-12                       # a single multiplier per column and group
    others = np.setdiff1d(np.arange(m["ngeom"]), np.concatenate([rg, cg]))
    assert np.allclose(fr[:, others], 1.0)
    g = p["opt_gravity"].numpy() - m["opt_gravity"]
    assert abs(g.std() - 0.4) < 0.05 and abs(g.mean()) < 0.06
    dd = r("dof_damping")[:, R.robot_dofs.numpy()]
    assert dd.min() >= 1 / 1.5 - 1e-12 and dd.max() <= 1.5 + 1e-12 and abs(np.log(dd).mean()) < 0.03
    kp = r("actuator_gainprm").reshape(n, m["nu"], -1)[:, :, 0]
    assert kp.min() >= 0.5 - 1e-12 and kp.max() <= 2.0 + 1e-12
    jr = p["jnt_range"].numpy().reshape(n, -1, 2)
    assert (jr[:, :, 1] > jr[:, :, 0] - 1e-12).all()
    tr = p["tendon_range"].numpy().reshape(n, -1, 2)
    assert (tr[:, :, 0] >= 0).all() and (tr[:, :, 1] > tr[:, :, 0]).all()
    gs = r("geom_size").reshape(n, -1, 3)[:, R.cube_middle]
    assert gs.min() >= 0.95 and gs.max() <= 1.05
    assert np.allclose(p["geom_rbound"].numpy()[:, R.cube_middle], np.linalg.norm(p["geom_size"].numpy().reshape(n, -1, 3)[:, R.cube_middle], axis=1))
    # per-step samplers
    st = R.timestep_state(n)
    ts = np.stack([R.next_timestep(st).numpy() for _ in range(50)])
    assert ts.min() >= 0.5 * 0.008 - 1e-12 and ts.max() < 0.008 + 0.02 and 5e-5 < np.abs(ts - 0.008).mean() < 1e-3
    import torch
    ws = R.wind_state(n, 0.08)
    x = torch.zeros(n, m["nbody"], 6, dtype=torch.float64)
    hits = 0
    for _ in range(200):
        R.next_wind(ws, x)
        hits += int((x[:, R.cube_body, :3].abs().sum(1) > 0).sum() > 0)
    assert hits > 0 and float(x[:, :, 3:].abs().max()) == 0.0 and float(x[:, :R.cube_body].abs().max()) == 0.0


def test_range_rules_match_reference_wrappers(rnd):
    """joint-limit / control-range and tendon-range perturbation: the reference wrappers' own _set_field, run on the
    shim with given normal draws (tests/golden/ref_range_rules.npz, tools/make_reference_golden.py), against the batched
    rules fed the same draws."""
    import torch

    m, R = rnd
    g = np.load(os.path.join(HERE, "golden", "ref_range_rules.npz"))
    for seed in (0, 1, 2):
        key = "seed%d_" % seed
        zj, zt = g[key + "zj"], g[key + "zt"]
        assert zt.shape == (m["ntendon"], 2)
        got = R.sample(1, noises=dict(joint_limit=torch.tensor(zj[None]), tendon_range=torch.tensor(zt[None])))
        assert np.abs(got["jnt_range"][0].numpy() - g[key + "jnt_range"]).max() < 1e-12
        assert np.abs(got["actuator_ctrlrange"][0].numpy() - g[key + "actuator_ctrlrange"]).max() < 1e-12
        assert np.abs(got["tendon_range"][0].numpy() - g[key + "tendon_range"]).max() < 1e-12


@pytest.mark.gpu
def test_sampled_parameters_reach_the_engine(locked_blob, locked_names):
    """Environments with different sampled parameters evolve differently; an environment whose rows equal the model's
    reproduces the unrandomised step bit for bit; a subset of rows can be re-sampled in place."""
    import torch

    from robogym_b200 import build, engine
    from robogym_b200.locked_env import TorchRand
    from robogym_b200.randomization import LockedRandomizer

    build.build()
    model = engine.DeviceModel(locked_blob, 0)
    dev = torch.device("cuda", 0)
    n = 64
    R = LockedRandomizer(model.host, locked_names, TorchRand(torch, dev, 5), torch, dev, torch.float32)
    base = engine.BatchedSim(model, n, 10)
    sim = engine.BatchedSim(model, n, 10)
    p = R.sample(n)
    for k in p:                     # environment 0 keeps the model's own values
        p[k][0] = R.orig[k][0]
    R.apply(sim, p)
    ctrl = torch.tensor(model.host["actuator_ctrlrange"].reshape(-1, 2).mean(1), dtype=torch.float32, device=dev)
    for s in (base, sim):
        s.ctrl.copy_(ctrl.repeat(n, 1))
        for _ in range(3):
            s.step()
    torch.cuda.synchronize()
    assert int(sim.warn.max()) == 0
    assert torch.equal(sim.qpos[0], base.qpos[0]) and torch.equal(sim.qvel[0], base.qvel[0])
    d = (sim.qpos[1:] - base.qpos[1:]).abs().max(dim=1).values
    assert float(d.min()) > 1e-6
    idx = torch.tensor([3, 7], device=dev)
    q = R.sample(2)
    before = sim._params["dof_damping"].clone()
    R.apply(sim, q, idx)
    after = sim._params["dof_damping"]
    assert torch.equal(after[idx], q["dof_damping"]) and torch.equal(after[0], before[0]) and not torch.equal(after[3], before[3])


def test_full_cube_randomizer_covers_the_cfg3_stack(tmp_path):
    """dactyl/full_perpendicular's wrapper list (full_perpendicular.py:425-440) = the locked list + face damping (+ the mesh-scaling cube
    size wrapper, which is documented as not covered): rows for the nv=168 model, face damping confined to the 66 face / cubelet
    dofs of the manipulated cube with factors in [1/3, 3], robot damping still in [1/1.5, 1.5], cube friction on every cube geom."""
    import json

    import torch

    from robogym_b200 import modelblob
    from robogym_b200.randomization import FullCubeRandomizer

    blob = open(os.path.join(HERE, "..", "robogym_b200", "assets", "dactyl_full_perpendicular.rgm"), "rb").read()
    names = json.load(open(os.path.join(HERE, "..", "robogym_b200", "assets", "dactyl_full_perpendicular.names.json")))
    m = modelblob.unpack(blob)
    R = FullCubeRandomizer(m, names, NumpyRand(3, torch), torch, torch.device("cpu"), torch.float64)
    assert R.cube_middle is None and int(R.face_dofs.numel()) == 66 and int(R.cube_geoms.numel()) == 26
    n = 64
    p = R.sample(n)
    assert "geom_size" not in p and p["dof_damping"].shape == (n, 168)
    d0 = np.asarray(m["dof_damping"])
    ratio = p["dof_damping"].numpy() / np.where(d0 > 0, d0, 1.0)
    face, robot = R.face_dofs.numpy(), R.robot_dofs.numpy()
    other = np.setdiff1d(np.arange(168), np.concatenate([face, robot]))
    assert ratio[:, face].min() >= 1 / 3.0 - 1e-12 and ratio[:, face].max() <= 3.0 + 1e-12 and ratio[:, face].std() > 0.3
    assert ratio[:, robot].min() >= 1 / 1.5 - 1e-12 and ratio[:, robot].max() <= 1.5 + 1e-12
    assert np.all(p["dof_damping"].numpy()[:, other] == d0[other])                # the target cube's joints are left alone
    fr = p["geom_friction"].reshape(n, -1, 3).numpy() / np.asarray(m["geom_friction"]).reshape(1, -1, 3)
    cg = R.cube_geoms.numpy()
    assert np.allclose(fr[:, cg], fr[:, cg[:1]]) and fr[:, cg, 0].min() >= 0.5 and fr[:, cg, 1].max() <= 5.0   # one draw per env, all cube geoms
    assert p["body_inertia"].shape == (n, 3 * m["nbody"]) and p["dof_invweight0"].shape == (n, 168)
