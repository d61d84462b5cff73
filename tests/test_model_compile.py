"""Model compiler + blob format (host logic, CPU only)."""
import os

import numpy as np
import pytest

from robogym_b200 import mjcf, modelblob

HAVE_REF = os.path.isdir("/root/reference/robogym")


def test_blob_roundtrip(locked_blob):
    m = modelblob.unpack(locked_blob)
    assert modelblob.pack(m, modelblob.unpack_names(locked_blob)) == locked_blob
    assert m["nq"] == 38 and m["nv"] == 36 and m["npair"] == 1243


def test_static_tables_are_consistent(locked_blob):
    m = modelblob.unpack(locked_blob)
    parent = m["body_parentid"]
    assert all(parent[b] < b for b in range(1, m["nbody"]))                 # depth-first numbering
    mask = m["body_dofmask"].view(np.uint32).reshape(m["nbody"], -1)
    for d in range(m["nv"]):                                                 # dof moves its own body and its subtree only
        b = m["dof_bodyid"][d]
        assert (mask[b, d // 32] >> (d % 32)) & 1
        assert not (mask[parent[b], d // 32] >> (d % 32)) & 1
    adjadr, adj = m["mesh_adjadr"], m["mesh_adj"]
    for i in range(m["nmesh"]):                                              # hull adjacency is symmetric
        va, vn = m["mesh_vertadr"][i], m["mesh_vertnum"][i]
        nb = [set(adj[adjadr[va + v]:adjadr[va + v + 1]]) for v in range(vn)]
        assert all(v in nb[w] for v in range(vn) for w in nb[v])
        assert all(len(s) >= 3 for s in nb)
    # hill climbing on the hull graph finds the exhaustive support vertex
    rng = np.random.RandomState(0)
    V = m["mesh_vert"].reshape(-1, 3)
    for i in range(m["nmesh"]):
        va, vn = m["mesh_vertadr"][i], m["mesh_vertnum"][i]
        for _ in range(20):
            dl = rng.randn(3)
            cur, best = 0, V[va] @ dl
            while True:
                nbr = adj[adjadr[va + cur]:adjadr[va + cur + 1]]
                dd = V[va + nbr] @ dl
                k = int(dd.argmax())
                if dd[k] > best:
                    best, cur = dd[k], int(nbr[k])
                else:
                    break
            assert abs(best - (V[va:va + vn] @ dl).max()) < 1e-12


def test_mass_matrix_formulations_agree(locked_blob):
    """numpy Jacobian-sum M (mjcf.mass_matrix) == oracle spatial-inertia M at a random pose."""
    from helpers import oracle_pair

    m = modelblob.unpack(locked_blob)
    om, d = oracle_pair(locked_blob)
    rng = np.random.RandomState(3)
    q = m["qpos0"].copy()
    jr = m["jnt_range"].reshape(-1, 2)
    for j in range(m["njnt"]):
        if m["jnt_type"][j] == 3 and m["jnt_limited"][j]:
            q[m["jnt_qposadr"][j]] = rng.uniform(*jr[j])
    quat = rng.randn(4)
    q[3:7] = quat / np.linalg.norm(quat)
    M_np, _ = mjcf.mass_matrix(m, q)
    d.qpos[:] = q
    d.forward()
    assert np.abs(M_np - d.M.reshape(m["nv"], m["nv"])).max() < 1e-12
    L_np, J_np = mjcf.tendon_eval(m, q)
    assert np.abs(L_np - d.ten_length).max() < 1e-12 and np.abs(J_np - d.ten_J.reshape(J_np.shape)).max() < 1e-10


@pytest.mark.needs_reference
@pytest.mark.skipif(not HAVE_REF, reason="needs /root/reference")
def test_committed_blob_is_reproducible(locked_blob):
    """tools/compile_models.py on the reference assets reproduces the committed blob bit for bit."""
    import robogym_b200.mujoco_py_shim as shim

    # the composer falls back to a bare mujoco_py stand-in when none is loaded; the reference modules it imports stay cached
    # for the rest of the process, so they must bind to the shim the later tests drive them through
    shim.install()
    import compose_reference_xml as ref

    cm = mjcf.compile_mjcf(ref.locked_xml())
    cm.m["opt_pid"][0] = 1
    assert cm.blob() == locked_blob


def test_compiler_passes_one_by_one():
    """compile_mjcf is a sequence of passes over one context (mjcf._PASSES): run them one at a time on a small document and
    check what each leaves behind for the next."""
    from robogym_b200 import mjcf
    from toy_models import FREE_BODIES

    c = mjcf._Ctx()
    c.xml_string, c.asset_loader = FREE_BODIES, None
    seen = {}
    for p in mjcf._PASSES:
        p(c)
        seen[p.__name__] = set(vars(c))
    assert [p.__name__ for p in mjcf._PASSES][:4] == ["_pass_document", "_pass_compiler_option_size", "_pass_assets", "_pass_kinematic_tree"]
    assert "root" in seen["_pass_document"] and "angle_scale" in seen["_pass_compiler_option_size"]
    assert "nbody" in seen["_pass_kinematic_tree"] and "nbody" not in seen["_pass_assets"]
    assert c.nbody == 7 and (c.nq, c.nv) == (23, 20)                     # world, floor, box, ball, brick, arm, fore; 3 free joints + 2 hinges
    assert "pair1" in seen["_pass_collision_pair_list"] and "pair1" not in seen["_pass_sites"]
    assert len(c.pair1) == len(c.pair2) > 0
    assert "act_gainprm" in seen["_pass_actuators"] and c.nu == 2
    assert "cm" in seen["_pass_mesh_tables_and_model"]
    assert c.cm.blob() == mjcf.compile_mjcf(FREE_BODIES).blob()
