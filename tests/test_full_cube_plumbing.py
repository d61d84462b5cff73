"""BASELINE.json configs[2] (dactyl/full_perpendicular: Rubik's cube with 6 face drivers, nq170/nv168) as PLUMBING: the
committed model is what the reference builds on the mujoco_py shim (tools/compile_models.py), it has the size SURVEY.md
Appendix A predicts, and the fp64 oracle steps it from the reference environment's reset state exactly as the reference
environment did (tests/golden/ref_full_cube.npz, tools/make_reference_golden.py)."""
import os

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))


def test_full_perpendicular_compiles_and_steps_on_the_oracle():
    from helpers import oracle_pair
    from robogym_b200 import modelblob

    blob = open(os.path.join(HERE, "..", "robogym_b200", "assets", "dactyl_full_perpendicular.rgm"), "rb").read()
    m = modelblob.unpack(blob)
    assert (m["nq"], m["nv"], m["nu"]) == (170, 168, 20)
    assert m["njnt"] == 164 and m["ntendon"] == 12 and m["nbody"] == 135
    g = np.load(os.path.join(HERE, "golden", "ref_full_cube.npz"))
    om, d = oracle_pair(blob)
    d.qpos[:] = g["start_qpos"]; d.qvel[:] = g["start_qvel"]; d.ctrl[:] = g["start_ctrl"]
    d.userdata[:] = g["start_pid"]; d.qacc_warmstart[:] = g["start_warm"]
    d.forward()
    for c in g["ctrl"]:                      # the hand held at its zero action, as the reference environment was
        d.ctrl[:] = c
        d.env_step(int(g["nsubsteps"]))
    assert np.isfinite(d.qpos).all() and np.isfinite(d.qvel).all()
    assert np.abs(d.qpos - g["qpos"]).max() < 1e-9 and np.abs(d.qvel - g["qvel"]).max() < 1e-6
    assert int(d.ncon[0]) == int(g["ncon"]) >= 10     # the 26 cubelets rest on each other and on the palm
    assert bool(g["on_palm"])
