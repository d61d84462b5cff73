"""Contact-based observations of the rearrange environments, batched (robogym_b200/rearrange_contacts.py), against the
reference's own functions (robogym/robot/ur16e/mujoco/simulation/base.py:142-167, robogym/envs/rearrange/simulation/base.py:562-636)
evaluated on the same contact lists: the unmodified reference environment ran on the shim (oracle engine) while the gripper
was driven down onto a block and the table, and its contact lists and answers after every step were recorded
(tests/golden/ref_rearrange_contacts.npz, tools/make_reference_golden.py); the batched answers computed from a contact tensor
that holds those contacts must equal the reference's."""
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(HERE, "stubs"))


def contact_actions():
    """put block 0 under the tool, open gripper, then push down: finger pads meet the block, later the gripper meets the table plane"""
    out = []
    for k in range(26):
        a = np.zeros(6, dtype=np.float32)
        if k < 8:
            a[2] = -1.0                      # straight down onto the block
            a[5] = 1.0 if k < 4 else -1.0    # open, then close on it
        elif k < 12:
            a[2], a[1], a[5] = 0.6, 1.0, 1.0  # up and away from the blocks, open
        else:
            a[2] = -1.0                      # down until the fingers meet the table
        out.append(a)
    return out


class _ContactView:
    """the slice of BatchedSim that BatchedRearrangeContacts reads, filled from a recorded contact list"""

    def __init__(self, blob, K=64):
        import torch

        from oracle_generic_sim import _Model

        self.torch = torch
        self.model = _Model(blob)
        self.qpos = torch.zeros(1, 1, dtype=torch.float64)
        self.contact = torch.zeros(1, K, 4, dtype=torch.float64)
        self.ncon = torch.zeros(1, dtype=torch.int32)

    def load(self, con, ncon):
        self.contact.zero_()
        self.contact[0, :, :3] = self.torch.tensor(con)
        self.ncon[0] = int(ncon)


def test_batched_contact_queries_equal_the_reference_functions():
    from robogym_b200.rearrange_contacts import BatchedRearrangeContacts

    g = np.load(os.path.join(HERE, "golden", "ref_rearrange_contacts.npz"))
    blob = open(os.path.join(HERE, "..", "robogym_b200", "assets", "rearrange_blocks5_tcp.rgm"), "rb").read()
    view = _ContactView(blob)
    q = BatchedRearrangeContacts(view, num_objects=5)
    cams = sorted(k[4:] for k in g.files if k.startswith("cam_"))
    assert len(g["ncon"]) == len(contact_actions()) and "any" in cams
    seen = dict(table=0, pad=0)
    for k in range(len(g["ncon"])):
        view.load(g["contact"][k], g["ncon"][k])
        want_obj = g["obj"][k]
        assert bool(q.gripper_table_contact()[0]) == bool(g["table"][k]), k
        got_cam = q.wrist_cam_collisions()
        assert {n: bool(v[0]) for n, v in got_cam.items()} == {n: bool(g["cam_" + n][k]) for n in cams}, k
        assert np.array_equal(q.object_gripper_contact()[0].numpy(), want_obj), (k, want_obj)
        seen["table"] += bool(g["table"][k]); seen["pad"] += int(want_obj.sum() > 0)
    assert seen["table"] > 0 and seen["pad"] > 0, seen        # the scenario did exercise the queries
