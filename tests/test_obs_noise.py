"""robogym_b200/obs_noise.py against the reference's RandomizeObservationWrapper (robogym/wrappers/randomizations.py:314-389): the
reference wrapper ran on a minimal fake environment with a random state that RECORDED its draws (tests/golden/ref_obs_noise.npz,
tools/make_reference_golden.py); the batched rule replays exactly those draws and must give the same noisy observations,
episode biases included."""
import os
from collections import OrderedDict

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
WIDTHS = dict(fingertip_pos=15, hand_angle=24, cube_pos=3, cube_quat=4)
NENV, NSTEPS = 3, 4


def clean_observations():
    """[step][env] -> the fake environment's clean observation dict"""
    rng = np.random.RandomState(0)
    clean = []
    for s in range(NSTEPS + 1):
        row = []
        for e in range(NENV):
            q = rng.randn(4); q /= np.linalg.norm(q)
            row.append(OrderedDict(fingertip_pos=rng.randn(15) * 0.05, hand_angle=rng.randn(24) * 0.3, cube_pos=rng.randn(3) * 0.1, cube_quat=q))
        clean.append(row)
    return clean


class _Replay:
    """the batched rule's `rand`: hands the recorded draws out again, one environment per row"""

    def __init__(self, torch, kinds, sizes, draws):
        self.torch, self.kinds, self.sizes, self.draws, self.pos, self.off = torch, kinds, sizes, draws, 0, 0

    def _next(self, kind, k):
        assert self.kinds[self.pos] == kind and self.sizes[self.pos] == k, (self.kinds[self.pos], kind, self.sizes[self.pos], k)
        v = self.draws[:, self.off:self.off + k]
        self.pos += 1
        self.off += k
        return self.torch.tensor(v)

    def randn(self, n, k):
        return self._next("randn", k)

    def uniform(self, lo, hi, n, k):
        return self._next("uniform", k)


def test_batched_rule_replays_the_reference_wrapper():
    import torch

    from robogym_b200.obs_noise import LOCKED_LEVELS, BatchedObservationNoise

    g = np.load(os.path.join(HERE, "golden", "ref_obs_noise.npz"))
    clean = clean_observations()
    rule = BatchedObservationNoise.__new__(BatchedObservationNoise)
    rule.torch, rule.rand, rule.nenv = torch, _Replay(torch, [str(k) for k in g["draw_kind"]], g["draw_size"], g["draws"]), NENV
    rule.levels = dict(LOCKED_LEVELS); rule.widths = {k: (1 if k.endswith("_quat") else w) for k, w in WIDTHS.items()}
    rule.cm = rule.um = 1.0
    rule.additive, rule.multiplicative = {}, {}
    rule.reset()
    for s in range(NSTEPS + 1):
        obs = {k: torch.tensor(np.stack([clean[s][e][k] for e in range(NENV)])) for k in WIDTHS}
        got = rule(obs)
        for k in WIDTHS:
            assert np.abs(got["noisy_" + k].numpy() - g["noisy_" + k][s]).max() < 1e-12, (s, k)
            assert np.array_equal(got[k].numpy(), obs[k].numpy())
    assert rule.rand.pos == len(g["draw_kind"]) and rule.rand.off == g["draws"].shape[1]   # every recorded draw was consumed, in order
    # the noise is of the documented size: cube position within centimetres, the quaternion a few degrees off
    d = got["noisy_cube_pos"].numpy() - obs["cube_pos"].numpy()
    assert 1e-4 < np.abs(d).max() < 0.05
    ang = 2 * np.arccos(np.clip(np.abs((got["noisy_cube_quat"].numpy() * obs["cube_quat"].numpy()).sum(1)), 0, 1))
    assert 0.0 < ang.max() < 1.0
