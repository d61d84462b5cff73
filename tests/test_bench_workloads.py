"""bench.py's dual-simulation rearrange workload (RearrangeTcpWorkload: placement, controller loop, episode ends, resets) on the
CPU emulation of the kernel -- the host logic the GPU bench line runs, checked without a GPU."""
import json
import os
import sys

import numpy as np
import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.join(HERE, "..")
sys.path.insert(0, os.path.join(HERE, "stubs"))
sys.path.insert(0, ROOT)


@pytest.mark.parametrize("config", ["rearrange_blocks_tcp", "rearrange_ycb_tcp"])
def test_dual_simulation_workload_runs_on_the_emulated_kernels(config):
    import torch

    import bench
    from emu_generic_sim import EmuGenericSim

    cfg = bench.CONFIGS[config]
    blob, sblob = bench.load_blob(cfg["asset"]), bench.load_blob(cfg["solver_asset"])
    names = json.load(open(os.path.join(ROOT, "robogym_b200", "assets", cfg["asset"] + ".names.json")))
    n = 3
    main = EmuGenericSim(blob, n, cfg["nsub"], contact_capacity=cfg["caps"][0], row_capacity=cfg["caps"][1])
    solver = EmuGenericSim(sblob, n, cfg["nsub"])
    gen = torch.Generator(device="cpu")
    gen.manual_seed(1)
    wl = bench.RearrangeTcpWorkload(main, main.model, names, torch.device("cpu"), gen, cfg["nobj"], cfg["grid"], solver)
    assert wl.action_dim == 6
    tcp0 = main.body_xpos[:, wl.tcp_main].clone()
    q_arm0 = main.qpos[:, wl.ctl.arm_qadr_main].clone()
    for k in range(6):
        wl.apply_action(wl.sample_action())
        wl.step_timed()
        wl.auto_reset()
    assert int(main.warn.max()) == 0 and int(solver.warn.max()) == 0
    z = torch.stack([main.qpos[:, a + 2] for a in wl.blocks], dim=1)
    assert bool((z > 0.49).all()) and bool((z < 0.56).all())                    # every object still on the table top
    assert float((main.body_xpos[:, wl.tcp_main] - tcp0).abs().max()) > 0.02   # the tool went where the actions sent it
    assert float((main.qpos[:, wl.ctl.arm_qadr_main] - q_arm0).abs().max()) > 0.02
    # a forced episode end re-seats the arm, the objects and both controllers' state
    mask = torch.tensor([False, True, False])
    wl.reset(mask)
    assert torch.allclose(main.qpos[1, wl.ctl.arm_qadr_main], wl.q0[1, wl.ctl.arm_qadr_main]) and not bool(main.pid[1].any())
    assert torch.equal(solver.qpos[1, wl.ctl.arm_qadr_solver], main.qpos[1, wl.ctl.arm_qadr_main]) and not bool(solver.qvel[1].any())
    assert bool(main.qvel[0].any())                                              # the others keep going


@pytest.mark.parametrize("config", ["rearrange_blocks_tcp", "rearrange_ycb_tcp"])
def test_emulated_main_scene_follows_the_oracle_from_workload_states(config):
    """Teacher-forced parity of the scenes the dual-simulation bench lines run: states reached by the workload on the emulated
    kernels, one env-step (40 substeps + 2 forwards, cascaded-PI arm, objects resting on the table) on the fp32 kernel logic
    against the fp64 oracle."""
    import torch

    import bench
    from emu_generic_sim import EmuGenericSim
    from oracle_generic_sim import OracleGenericSim

    cfg = bench.CONFIGS[config]
    blob, sblob = bench.load_blob(cfg["asset"]), bench.load_blob(cfg["solver_asset"])
    names = json.load(open(os.path.join(ROOT, "robogym_b200", "assets", cfg["asset"] + ".names.json")))
    n = 2
    main = EmuGenericSim(blob, n, cfg["nsub"], contact_capacity=cfg["caps"][0], row_capacity=cfg["caps"][1])
    solver = EmuGenericSim(sblob, n, cfg["nsub"])
    gen = torch.Generator(device="cpu")
    gen.manual_seed(7)
    wl = bench.RearrangeTcpWorkload(main, main.model, names, torch.device("cpu"), gen, cfg["nobj"], cfg["grid"], solver)
    for _ in range(3):
        wl.apply_action(wl.sample_action()); wl.step_timed()
    om = OracleGenericSim(blob, n, cfg["nsub"])
    for f in ("qpos", "qvel", "ctrl", "pid", "qacc_warmstart"):
        getattr(om, f).copy_(getattr(main, f).to(torch.float64))
    main.step(final_forward=2)
    om.step(final_forward=2)
    dq = (main.qpos.to(torch.float64) - om.qpos).abs()
    arm = wl.ctl.arm_qadr_main
    assert int(main.warn.max()) == 0 and int(om.warn.max()) == 0
    assert float(dq[:, arm].max()) < 5e-5, float(dq[:, arm].max())                      # the arm under its cascaded-PI controllers
    # objects: resting contacts; a mesh object rocking on a multi-part hull can switch a contact within fp32 noise (tests/test_rearrange_ycb.py)
    assert float(dq.max()) < (5e-4 if "blocks" in config else 3e-3) and float(dq.median()) < 1e-5, (float(dq.max()), float(dq.median()))


def test_reference_arm_prints_the_contract_line():
    """`bench.py --impl reference` (the CPU arm the driver runs beside the GPU arm): one JSON line with the contract's keys, the
    reference-arm extras, and a positive rate -- on a tiny bounded sample."""
    import subprocess

    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "1"],
                         capture_output=True, text=True, timeout=300, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-1500:]
    line = json.loads(out.stdout.strip().splitlines()[-1])
    for k in ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline", "dtype", "data", "config",
              "cpu_baseline", "e2e", "gpu_launches"):
        assert k in line, k
    assert line["impl"] == "reference" and line["value"] > 0 and line["unit"] == "env-steps/s" and line["higher_is_better"] is True
    assert line["cpu_baseline"]["kind"] == "port" and line["cpu_baseline"]["cores"] >= 1
    assert line["e2e"]["h2d_bytes_per_step"] == 0 and line["e2e"]["d2h_bytes_per_step"] == 0 and line["gpu_launches"] == 0
    assert "workload" in line["config"]


def test_dump_outputs_writes_float_arrays_and_samples_environments(tmp_path):
    """bench.py --dump-outputs: float32 outputs stay float32, integer ones become exact float64; above the size limit the same
    seeded sample of environments is taken from every array and its indices are written beside them."""
    import torch

    import bench

    n = 1000
    arrays = dict(qpos=torch.arange(n * 3, dtype=torch.float32).reshape(n, 3), ncon=torch.arange(n, dtype=torch.int32))
    bench.dump_outputs(arrays, str(tmp_path / "all"))
    q, c = np.load(tmp_path / "all" / "qpos.npy"), np.load(tmp_path / "all" / "ncon.npy")
    assert q.dtype == np.float32 and c.dtype == np.float64 and np.array_equal(q, arrays["qpos"].numpy()) and np.array_equal(c, np.arange(n))
    assert not (tmp_path / "all" / "env_index.npy").exists()
    for d in ("a", "b"):
        bench.dump_outputs(arrays, str(tmp_path / d), limit=4000)
    idx = np.load(tmp_path / "a" / "env_index.npy")
    assert np.array_equal(idx, np.load(tmp_path / "b" / "env_index.npy")) and 0 < len(idx) < n
    assert sum(os.path.getsize(tmp_path / "a" / f) for f in os.listdir(tmp_path / "a")) < 4000 + 3 * 128     # + .npy headers
    assert np.array_equal(np.load(tmp_path / "a" / "ncon.npy"), idx) and np.array_equal(np.load(tmp_path / "a" / "qpos.npy")[:, 0], 3 * idx)
