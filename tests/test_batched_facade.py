"""Batched host facade (robogym_b200/batched_env.py) against the reference's OWN per-env code: robogym's locked
environment on the mujoco_py shim (oracle engine, CPU) recorded its controls, observations, contacts and occlusion
flags, and the model fields its randomisation wrappers changed (tests/golden/ref_facade.npz, tools/make_reference_golden.py);
the facade must compute the same from the recorded simulator state."""
import os

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))


def test_facade_matches_reference_host_code(locked_blob, locked_names):
    import torch

    from robogym_b200 import modelblob
    from robogym_b200.batched_env import ShadowHandCubeFacade

    g = np.load(os.path.join(HERE, "golden", "ref_facade.npz"))
    m = modelblob.unpack(locked_blob)
    m.update({k[len("model_"):]: g[k] for k in g.files if k.startswith("model_")})    # the recorded environment's randomised model
    fac = ShadowHandCubeFacade(m, locked_names, "cpu", dtype=torch.float64)
    t = lambda k, i: torch.tensor(g[k][i][None])
    for k in range(len(g["action"])):
        # a6: relative and absolute denormalisation
        got_rel = fac.denormalize_position_control(t("action", k), t("qpos_before", k), relative_action=True)[0].numpy()
        got_abs = fac.denormalize_position_control(t("action", k), None, relative_action=False)[0].numpy()
        assert np.abs(got_rel - g["ctrl_rel"][k]).max() < 1e-12 and np.abs(got_abs - g["ctrl_abs"][k]).max() < 1e-12
        # a7: observations
        sx = t("site_xpos", k)
        mine = fac.observe(t("qpos", k), t("qvel", k), sx, t("actuator_force", k))
        for key in ("cube_pos", "cube_quat", "hand_angle", "fingertip_pos"):
            assert np.abs(mine[key][0].numpy().ravel() - g[key][k]).max() < 1e-9, key
        assert np.abs(mine["actuator_force"][0].numpy() - g["effort"][k]).max() < 1e-9
        # a8
        assert bool(fac.on_palm(sx)[0]) == bool(g["on_palm"][k])
        # a9
        got = fac.fingers_occluded(t("contact", k), torch.tensor([int(g["ncon"][k])]))[0].numpy()
        assert np.array_equal(got.astype(int), g["occluded"][k])
    assert (g["ncon"] > 0).any()
