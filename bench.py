#!/usr/bin/env python
"""bench.py -- env-steps/sec of the dactyl/locked step path at batch 8192 per GPU (BASELINE.json).

One "step" = one SimulationInterface.step() for every environment of the batch
(robogym/mujoco/simulation_interface.py:176-189: 10 x mj_step + mj_forward), i.e. one launch of
the fused rg_step kernel per rank.  `value` = whole-job env-steps/s with inputs resident in HBM;
`e2e` = the same through the public API (robogym_b200.engine.BatchedSim + the batched facade's action -> control law)
with HOST buffers: pinned actions -> device, control law, step, qpos/qvel -> pinned host, every step, inside the timed region.

    python bench.py --gpus 1 --steps 20 --warmup 3
    python -m torch.distributed.run --nnodes=1 --nproc-per-node 8 --master-addr 127.0.0.1 \
        --master-port 29500 bench.py --gpus 8 --steps 20 --warmup 3
    python bench.py --impl reference        # the CPU port of the reference path on the host cores
    python bench.py --dump-outputs bench_outputs     # also write what the last timed step computed, bench_outputs/<name>.npy
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

NENV_PER_GPU = 8192
NSUB = 10
ALGO_BYTES_PER_ENV_STEP = 1664       # SURVEY.md 8(d): 784 B read + 680 B written + ~200 B derived outputs
METRIC = "env-steps/sec dactyl/locked batch 8192 @1/2/4/8 B200 vs CPU mujoco-py"


# ---------------------------------------------------------------- host logic shared with tests/test_dist.py
def shard_range(total, rank, world):
    per = total // world
    return rank * per, (rank + 1) * per


def rank_seed(seed, rank):
    return seed * 1000003 + rank


def max_over_ranks(x, dist, device):
    import torch

    t = torch.tensor([x], dtype=torch.float64, device=device)
    if dist is not None and dist.is_initialized():
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return float(t.item())


def sum_over_ranks(x, dist, device):
    import torch

    t = torch.tensor([x], dtype=torch.float64, device=device)
    if dist is not None and dist.is_initialized():
        dist.all_reduce(t, op=dist.ReduceOp.SUM)
    return float(t.item())


def load_blob(asset="dactyl_locked"):
    with open(os.path.join(ROOT, "robogym_b200", "assets", asset + ".rgm"), "rb") as f:
        return f.read()


def measured_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured"
        except Exception:
            pass
    return 6650.0, "fallback"


# ---------------------------------------------------------------- clocks sampler
class ClockSampler:
    """Samples SM clock and throttle reasons of one GPU every 50 ms in a thread (NVML) during the timed region."""

    def __init__(self, index):
        self.index, self.samples, self.reasons, self.smax, self._stop, self._thr = index, [], set(), None, False, None

    def start(self):
        import threading

        try:
            import pynvml

            pynvml.nvmlInit()
            h = pynvml.nvmlDeviceGetHandleByIndex(self.index)
            self.smax = float(pynvml.nvmlDeviceGetMaxClockInfo(h, pynvml.NVML_CLOCK_SM))
        except Exception:
            return
        names = {"hw_slowdown": getattr(pynvml, "nvmlClocksThrottleReasonHwSlowdown", 0x8),
                 "hw_thermal_slowdown": getattr(pynvml, "nvmlClocksThrottleReasonHwThermalSlowdown", 0x40),
                 "sw_thermal_slowdown": getattr(pynvml, "nvmlClocksThrottleReasonSwThermalSlowdown", 0x20),
                 "sw_power_cap": getattr(pynvml, "nvmlClocksThrottleReasonSwPowerCap", 0x4)}

        def run():
            while not self._stop:
                try:
                    self.samples.append(float(pynvml.nvmlDeviceGetClockInfo(h, pynvml.NVML_CLOCK_SM)))
                    r = pynvml.nvmlDeviceGetCurrentClocksThrottleReasons(h)
                    for k, bit in names.items():
                        if r & bit:
                            self.reasons.add(k)
                except Exception:
                    pass
                time.sleep(0.05)

        self._thr = threading.Thread(target=run, daemon=True)
        self._thr.start()

    def stop(self):
        self._stop = True
        if self._thr is not None:
            self._thr.join(timeout=2)
        return {"sm_mhz": statistics.median(self.samples) if self.samples else None, "sm_max_mhz": self.smax,
                "reasons": sorted(self.reasons), "samples": len(self.samples)}


# ---------------------------------------------------------------- CPU arm (oracle port of the reference path)
class _CpuEnv:
    """One dactyl/locked environment on the fp64 CPU port, driven with the GPU arm's workload (SURVEY 8(d) cfg 2: relative
    full-range actions, reset when the cube leaves the palm)."""

    def __init__(self, blob, seed):
        import numpy as np

        from oracle import pyoracle
        from robogym_b200 import modelblob

        self.np = np
        self.om = pyoracle.OracleModel(blob)
        self.d = pyoracle.OracleData(self.om)
        m = modelblob.unpack(blob)
        self.P = control_matrix(m)
        self.cr = self.om.field("actuator_ctrlrange").reshape(-1, 2)
        self.site = json.load(open(os.path.join(ROOT, "robogym_b200", "assets", "dactyl_locked.names.json")))["site"].index("cube:center")
        self.rng = np.random.RandomState(seed)
        self.d.ctrl[:] = self.cr.mean(1)
        for _ in range(20):
            self.d.env_step(NSUB)
        self.q0, self.c0 = self.d.qpos.copy(), self.d.ctrl.copy()
        self.reset()

    def reset(self):
        d, np = self.d, self.np
        d.qpos[:] = self.q0
        d.qpos[0:3] += 0.005 * self.rng.randn(3)
        q = self.rng.randn(4)
        d.qpos[3:7] = q / np.linalg.norm(q)
        d.qvel[:] = 0
        d.userdata[:] = 0
        d.qacc_warmstart[:] = 0
        d.ctrl[:] = self.c0

    def step(self):
        d, np, cr = self.d, self.np, self.cr
        a = self.rng.uniform(-1, 1, len(cr))
        d.ctrl[:] = np.clip(self.P @ d.qpos + a * (cr[:, 1] - cr[:, 0]) / 2, cr[:, 0], cr[:, 1])
        d.env_step(NSUB)
        if d.site_xpos.reshape(-1, 3)[self.site, 2] <= 0.04:
            self.reset()


def _cpu_worker(args):
    blob, seed, n_steps = args
    env = _CpuEnv(blob, seed)
    t0 = time.perf_counter()
    for _ in range(n_steps):
        env.step()
    return time.perf_counter() - t0


def cpu_baseline(blob, seconds=10.0):
    """Single-thread timing of the fp64 CPU port on a bounded sample (about `seconds` of CPU work)."""
    from oracle import pyoracle

    pyoracle.build()
    probe = _cpu_worker((blob, 1, 20))
    n = max(20, int(seconds / (probe / 20)))
    t = _cpu_worker((blob, 2, n))
    return {"value": n / t, "unit": "env-steps/s", "cores": 1, "kind": "port",
            "sample": f"{n} env-steps (x{NSUB} substeps) of one dactyl/locked env, the GPU arm's workload (relative full-range actions, reset on drop), "
                      "fp64 CPU port of the reference path (oracle/: dense, scalar, written for clarity -- NOT mujoco-py, which is not installable here); "
                      "one otherwise idle core: under full load the per-core rate is lower (see --impl reference: value / cores)"}


def cpu_baseline_rearrange(blob, names, seconds=10.0):
    """Single-thread timing of the fp64 CPU port on the rearrange/blocks workload (one environment, bounded sample)."""
    import numpy as np

    from oracle import pyoracle

    pyoracle.build()
    om = pyoracle.OracleModel(blob)
    d = pyoracle.OracleData(om)
    jn = names["joint"]
    d.qpos[:6] = np.deg2rad([135.0, -90.0, 135.0, -100.0, -240.0, 135.0])
    nobj = sum(1 for n in jn if n and n.startswith("object") and n.endswith(":joint"))
    for i in range(nobj):
        a = int(om.field("jnt_qposadr")[jn.index("object%d:joint" % i)])
        d.qpos[a:a + 3] = [1.25 + 0.27 * (i % 3), 0.32 + 0.36 * (i // 3), 0.60] if nobj > 5 else [1.2 + 0.13 * (i % 3), 0.5 + 0.16 * (i // 3), 0.453 + 0.03324 + 0.0254 + 0.001]
    d.forward()
    tcp = names["body"].index("robot0:gripper_tcp")
    om.field("eq_data")[:7] = [0, 0, 0, 1, 0, 0, 0]
    p0 = d.xpos[3 * tcp:3 * tcp + 3].copy()
    d.mocap_pos[:3] = p0
    d.mocap_quat[:4] = d.xquat[4 * tcp:4 * tcp + 4]
    lo, hi = om.field("actuator_ctrlrange")[:2]
    rng = np.random.RandomState(0)

    def run(n):
        t0 = time.perf_counter()
        for _ in range(n):
            a = rng.uniform(-1, 1, 4)
            d.mocap_pos[:3] = np.clip(d.mocap_pos[:3] + 0.01 * a[:3], p0 + [-0.15, -0.05, -0.055], p0 + [0.25, 0.45, 0.10])
            d.ctrl[0] = lo + (hi - lo) * 0.5 * (a[3] + 1)
            d.env_step(20)
        return time.perf_counter() - t0

    probe = run(10)
    n = max(10, int(seconds / (probe / 10)))
    t = run(n)
    return {"value": n / t, "unit": "env-steps/s", "cores": 1, "kind": "port",
            "sample": f"{n} env-steps (x20 substeps) of one rearrange env with {nobj} objects, the GPU arm's workload, fp64 CPU port of the reference path "
                      "(oracle/: dense, scalar -- NOT mujoco-py); one otherwise idle core"}


def cpu_baseline_rearrange_tcp(blob, solver_blob, seconds=10.0):
    """Single-thread timing of the fp64 CPU port on the dual-simulation rearrange loop: the same controller class on oracle-backed
    stand-ins of its two simulations (tests/stubs/oracle_generic_sim.py: checker infrastructure, used here as the CPU arm only)."""
    import numpy as np
    import torch

    from oracle import pyoracle

    pyoracle.build()
    sys.path.insert(0, os.path.join(ROOT, "tests", "stubs"))
    from oracle_generic_sim import OracleGenericSim
    from robogym_b200.rearrange_arm import BatchedTcpArmController

    main, solver = OracleGenericSim(blob, 1, 40), OracleGenericSim(solver_blob, 1, 40)
    ctl = BatchedTcpArmController(main, solver, max_position_change=0.1)
    arm = np.deg2rad([135.0, -90.0, 135.0, -100.0, -240.0, 135.0])
    main.qpos[0, ctl.arm_qadr_main] = torch.tensor(arm)
    main.ctrl[0, ctl.arm_act_main] = torch.tensor(arm)
    jn = main.model.names["joint"]
    for i in range(5):
        a = int(main.model.host["jnt_qposadr"][jn.index("object%d:joint" % i)])
        main.qpos[0, a:a + 3] = torch.tensor([1.2 + 0.13 * (i % 3), 0.5 + 0.16 * (i // 3), 0.453 + 0.03324 + 0.0254 + 0.001])
    main.forward()
    ctl.reset()
    rng = np.random.RandomState(0)

    def run(n):
        t0 = time.perf_counter()
        for _ in range(n):
            ctl.step(torch.tensor(rng.uniform(-1, 1, (1, 6)).astype(np.float32)))
        return time.perf_counter() - t0

    probe = run(5)
    n = max(5, int(seconds / (probe / 5)))
    t = run(n)
    return {"value": n / t, "unit": "env-steps/s", "cores": 1, "kind": "port",
            "sample": f"{n} env-steps (solver arm: forward + 40 substeps; main scene: 40 substeps + 2 forwards) of one rearrange env with 5 blocks, the GPU arm's "
                      "workload, fp64 CPU port of the reference path (oracle/: dense, scalar -- NOT mujoco-py); one otherwise idle core"}


_REF = {}


def _ref_init(blob, base_seed):
    """Pool initializer: one persistent oracle environment per worker process (model loaded and settled once)."""
    _REF.update(env=_CpuEnv(blob, base_seed + os.getpid()))


def _ref_step(n_steps):
    env = _REF["env"]
    for _ in range(n_steps):
        env.step()
    return n_steps


def usable_cores():
    """Host threads this process can really use: affinity mask, capped by the cgroup CPU quota if there is one."""
    n = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    for path in ("/sys/fs/cgroup/cpu.max", "/sys/fs/cgroup/cpu/cpu.cfs_quota_us"):
        try:
            txt = open(path).read().split()
            if path.endswith("cpu.max"):
                if txt[0] != "max":
                    n = min(n, max(1, int(int(txt[0]) / int(txt[1]))))
            else:
                q = int(txt[0])
                if q > 0:
                    n = min(n, max(1, q // int(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())))
            break
        except Exception:
            continue
    return n


def run_reference_arm(args):
    """--impl reference: the CPU implementation of the path on all host cores.  mujoco-py 2.0.2.13 /
    MuJoCo 2.0 (robogym setup.py:16) is a closed binary that is not installable here (no network, not in
    the wheelhouse), so this arm times the fp64 CPU port under oracle/ -- one persistent single-env
    simulation per host core, the way robogym would be vectorised on CPUs."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import multiprocessing as mp

    from oracle import pyoracle

    pyoracle.build()
    blob = load_blob()
    cores = usable_cores()
    per_step = 16                     # env-steps per worker per bench "step" (bounded sample of the 8192-env workload)
    ctx = mp.get_context("fork")
    with ctx.Pool(cores, initializer=_ref_init, initargs=(blob, 1234)) as pool:
        for _ in range(max(args.warmup, 1)):
            pool.map(_ref_step, [per_step] * cores, chunksize=1)
        t0 = time.perf_counter()
        for _ in range(args.steps):
            pool.map(_ref_step, [per_step] * cores, chunksize=1)
        dt = time.perf_counter() - t0
    value = cores * per_step * args.steps / dt
    sample = (f"each bench step = {cores} persistent worker processes x {per_step} env-steps of one dactyl/locked env each "
              f"(fp64 CPU port of the reference path -- dense, scalar, unoptimised, NOT mujoco-py; 10 substeps + forward per env-step; "
              f"per-core rate under this full load: {value / cores:.0f} env-steps/s)")
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": "env-steps/s", "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f64", "data": "synthetic",
            "config": {"workload": CONFIGS["locked"]["label"] + ", 10 substeps of 0.008 s + forward per env-step, relative actions a~U(-1,1): "
                                   "ctrl = clip(P qpos + a*range/2), reset of environments whose cube left the palm; CPU arm = bounded sample of that workload"},
            "cpu_baseline": {"value": value, "unit": "env-steps/s", "cores": cores, "kind": "port", "per_core_under_load": value / cores, "sample": sample},
            "e2e": {"value": value, "unit": "env-steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}, "gpu_launches": 0}
    print(json.dumps(line), flush=True)


# ---------------------------------------------------------------- GPU arm
def newest_profile_metrics():
    """Per-launch counters of rg_step_kernel from the newest ncu capture committed under profiles/ (8192 envs, one launch):
    DRAM bytes and warp instructions.  None when no capture is there."""
    import csv
    import glob

    files = sorted(glob.glob(os.path.join(ROOT, "profiles", "r*_ncu_metrics.csv")), key=lambda f: (os.path.basename(f).split("_")[0][:2], os.path.getmtime(f)))
    latest = os.path.join(ROOT, "profiles", "latest_ncu_metrics.txt")     # names the capture of the current build (file times do not survive a checkout)
    if os.path.exists(latest):
        files.append(os.path.join(ROOT, "profiles", open(latest).read().strip()))
    for f in reversed(files):
        try:
            d = {r[0]: (r[1], float(r[2].replace(",", ""))) for r in csv.reader(open(f)) if len(r) == 3 and r[0] != "metric"}
            unit = {"byte": 1.0, "Kbyte": 1e3, "Mbyte": 1e6, "Gbyte": 1e9}
            rd, wr = d["dram__bytes_read.sum"], d["dram__bytes_write.sum"]
            return {"file": os.path.relpath(f, ROOT), "dram_bytes": rd[1] * unit.get(rd[0], 1.0) + wr[1] * unit.get(wr[0], 1.0),
                    "warp_inst": d["smsp__inst_executed.sum"][1]}
        except Exception:
            continue
    return None


CONFIGS = {
    # BASELINE.json configs[1] (the headline) and configs[2]; capacities per environment = (contacts, single-row elements, dofs per contact), 0 = engine default
    "locked": dict(asset="dactyl_locked", nenv=8192, caps=(0, 0, 0),
                   label="dactyl/locked (BASELINE.json configs[1], SURVEY 8(d) cfg 2): ShadowHand + locked cube, nq38/nv36/nu20"),
    "full_perpendicular": dict(asset="dactyl_full_perpendicular", nenv=4096, caps=(96, 288, 32),
                               label="dactyl/full_perpendicular (BASELINE.json configs[2], SURVEY 8(d) cfg 3 without per-env parameter randomisation): "
                                     "ShadowHand + Rubik's cube (26 cubelets, 6 face drivers), nq170/nv168/nu20"),
    # BASELINE.json configs[3]: the reference's UR16e + Robotiq 2f-85 + table world with 5 blocks (tools/compose_reference_xml.py)
    "rearrange_blocks": dict(asset="rearrange_blocks5", nenv=2048, caps=(64, 128, 16), nsub=20, workload="rearrange", nobj=5, grid=(3, 6, 1.20, 0.50, 0.13, 0.16),
                             label="rearrange/blocks (BASELINE.json configs[3]): UR16e + Robotiq 2f-85 driven through the mocap weld, 5 free "
                                   "blocks (condim 6, elliptic cones, impratio 10) on the table, nq43/nv38/nu1"),
    # BASELINE.json configs[3] with the reference's own two-simulation control loop and 6-D tool actions (SURVEY 8(d) row 4)
    "rearrange_blocks_tcp": dict(asset="rearrange_blocks5_tcp", solver_asset="rearrange_solver_arm", nenv=2048, caps=(64, 160, 16), nsub=40, workload="rearrange_tcp", nobj=5,
                                 grid=(3, 6, 1.20, 0.50, 0.13, 0.16),
                                 label="rearrange/blocks (BASELINE.json configs[3], SURVEY 8(d) cfg 4): UR16e + Robotiq 2f-85 under the reference's dual-simulation "
                                       "MOCAP_IK controller (solver arm with mocap weld nq8 -> joint targets -> main scene with cascaded-PI joint controllers, "
                                       "5 free blocks, condim 6, elliptic cones, impratio 10), nq43/nv38/nu7"),
    # BASELINE.json configs[4] with the reference's control loop: the main simulation of the reference's own ycb environment (its draw of 8 objects)
    "rearrange_ycb_tcp": dict(asset="rearrange_ycb8_tcp", solver_asset="rearrange_solver_arm", nenv=1024, caps=(64, 160, 16), nsub=40, workload="rearrange_tcp", nobj=8,
                              grid=(3, 9, 1.25, 0.32, 0.27, 0.36),
                              label="rearrange/ycb (BASELINE.json configs[4], SURVEY 8(d) cfg 5): the main simulation the reference's ycb environment compiles "
                                    "(8 YCB mesh objects of its own draw) under the dual-simulation MOCAP_IK controller, nq64/nv56/nu7"),
    # BASELINE.json configs[4]: the same world with 8 YCB objects (unions of 1..29 convex meshes each; one fixed draw of the eight)
    "rearrange_ycb": dict(asset="rearrange_ycb8", nenv=1024, caps=(64, 128, 16), nsub=20, workload="rearrange", nobj=8, grid=(3, 9, 1.25, 0.32, 0.27, 0.36),
                          label="rearrange/ycb (BASELINE.json configs[4]): UR16e + Robotiq 2f-85 driven through the mocap weld, 8 YCB mesh objects "
                                "(cracker box, banana, mug, power drill, hammer, soup can, scissors, apple: 59 convex parts) on the table, nq64/nv56/nu1"),
}


def control_matrix(m):
    """ctrl = P qpos for the position actuators (joint -> 1, fixed tendon -> its joint coefficients): what
    robot/shadow_hand/hand_interface.py:245-266 tabulates, read off the compiled transmissions."""
    import numpy as np

    P = np.zeros((m["nu"], m["nq"]))
    for i in range(m["nu"]):
        tid = int(m["actuator_trnid"][i])
        if m["actuator_trntype"][i] == 0:
            P[i, m["jnt_qposadr"][tid]] = 1.0
        else:
            for w in range(m["tendon_adr"][tid], m["tendon_adr"][tid] + m["tendon_num"][tid]):
                P[i, m["jnt_qposadr"][int(m["wrap_objid"][w])]] = m["wrap_prm"][w]
    return P


class Workload:
    """SURVEY.md 8(d) cfg 2: a ~ U(-1,1)^20, ctrl = clip(P qpos_hand + a * range / 2, ctrlrange) (relative actions,
    robogym/robot/robot_interface.py:247-278), held for the 10 substeps of an env-step; an environment whose cube left
    the palm is reset (CubeEnv._reset style: settled hand, cube position jitter N(0, 0.005^2), uniform random cube
    orientation) before the next step, so dropped cubes do not make steps cheaper.  Both dactyl scenes start their qpos
    with the cube's three slide joints and its ball joint."""

    def __init__(self, sim, model, names, dev, gen):
        import torch

        self.torch, self.sim, self.gen, self.dev = torch, sim, gen, dev
        m = model.host
        self.nu = m["nu"]
        N = sim.nenv
        f32 = dict(dtype=torch.float32, device=dev)
        self.P = torch.tensor(control_matrix(m), **f32)
        cr = m["actuator_ctrlrange"].reshape(-1, 2)
        self.ctrl_lo, self.ctrl_hi = torch.tensor(cr[:, 0], **f32), torch.tensor(cr[:, 1], **f32)
        self.cube_site = names["site"].index("cube:center")
        sim.ctrl.copy_((0.5 * (self.ctrl_lo + self.ctrl_hi)).repeat(N, 1))
        for _ in range(20):                              # locked.py:200-205: settle with zero actions
            sim.step()
        self.q0, self.c0 = sim.qpos.clone(), sim.ctrl.clone()
        self.n_resets = 0
        self.reset(torch.ones(N, dtype=torch.bool, device=dev))

    def reset(self, mask):
        t, sim = self.torch, self.sim
        N = sim.nenv
        q = self.q0.clone()
        q[:, 0:3] += 0.005 * t.randn(N, 3, device=self.dev, generator=self.gen)
        quat = t.randn(N, 4, device=self.dev, generator=self.gen)
        q[:, 3:7] = quat / quat.norm(dim=1, keepdim=True)
        mk = mask.unsqueeze(1)
        sim.qpos.copy_(t.where(mk, q, sim.qpos))
        sim.qvel.mul_((~mk).to(sim.qvel.dtype))
        sim.pid.mul_((~mk).to(sim.pid.dtype))
        sim.qacc_warmstart.mul_((~mk).to(sim.qvel.dtype))
        sim.ctrl.copy_(t.where(mk, self.c0, sim.ctrl))

    def ctrl_from_action(self, a):
        """Robot.denormalize_position_control with relative actions (robogym/robot/robot_interface.py:247-278) on the device:
        the formula of robogym_b200.batched_env.ShadowHandCubeFacade.denormalize_position_control"""
        t, sim = self.torch, self.sim
        center = sim.qpos @ self.P.T
        return t.minimum(t.maximum(center + a * 0.5 * (self.ctrl_hi - self.ctrl_lo), self.ctrl_lo), self.ctrl_hi)

    def next_ctrl(self):
        return self.ctrl_from_action(self.sample_action())

    @property
    def action_dim(self):
        return self.nu

    def sample_action(self):
        t, sim = self.torch, self.sim
        return t.rand(sim.nenv, self.nu, device=self.dev, generator=self.gen) * 2 - 1

    def apply_action(self, a):
        self.sim.ctrl.copy_(self.ctrl_from_action(a))

    def on_palm(self):
        return self.sim.site_xpos[:, self.cube_site, 2] > 0.04      # envs/dactyl/common/cube_utils.py:17-23

    def auto_reset(self):
        dropped = ~self.on_palm()
        self.reset(dropped)
        return dropped

    def step_timed(self):
        self.sim.step()


class RearrangeWorkload:
    """BASELINE.json configs[3]: TCP control through the mocap weld.  Action a ~ U(-1,1)^4: the mocap target moves by
    a[:3] * 0.01 m per env-step inside a box over the table (what gym's mocap_set_action does with MocapSolver's scaled action,
    robogym/robot/control/tcp/mocap_solver.py:52-53), a[3] picks the gripper's position target in its control range; 20 substeps
    of 0.002 s + forward per env-step (RearrangeSimulationInterface.build defaults, simulation/base.py:262-265).  Reset as
    the reference does it: arm at TABLETOP_EXPERIMENT_INITIAL_POS (robot/ur16e/arm_interface.py:27), reset_mocap_welds +
    reset_mocap2body_xpos, blocks dropped on random free spots of the table; an environment that lost a block over the
    table's edge is reset before the next step."""

    action_dim = 4

    def __init__(self, sim, model, names, dev, gen, nobj=5, grid=(3, 6, 1.20, 0.50, 0.13, 0.16)):
        import numpy as np
        import torch

        self.torch, self.sim, self.gen, self.dev = torch, sim, gen, dev
        m = model.host
        N = sim.nenv
        f32 = dict(dtype=torch.float32, device=dev)
        self.nobj, self.grid = nobj, grid
        self.tcp = names["body"].index("robot0:gripper_tcp")
        self.blocks = [int(m["jnt_qposadr"][names["joint"].index("object%d:joint" % i)]) for i in range(nobj)]
        rest = self.rest_heights(m, names, nobj)
        self.rest = torch.tensor(rest, **f32)
        cr = m["actuator_ctrlrange"].reshape(-1, 2)
        self.ctrl_lo, self.ctrl_hi = torch.tensor(cr[:, 0], **f32), torch.tensor(cr[:, 1], **f32)
        eq = np.array(m["eq_data"], dtype=np.float64).reshape(-1, 7)
        eq[0] = [0, 0, 0, 1, 0, 0, 0]                               # gym reset_mocap_welds
        model.set_field("eq_data", eq.reshape(-1))
        q0 = torch.tensor(m["qpos0"], **f32).repeat(N, 1)
        q0[:, :6] = torch.tensor(np.deg2rad([135.0, -90.0, 135.0, -100.0, -240.0, 135.0]), **f32)
        for k, a in enumerate(self.blocks):                          # parked far apart for the pose query below
            q0[:, a:a + 3] = torch.tensor([1.0 + 0.25 * (k % 4), 1.1 + 0.3 * (k // 4), 0.75], **f32)
        sim.qpos.copy_(q0)
        sim.forward()
        self.tcp_pos0 = sim.body_xpos[:, self.tcp].clone()
        self.tcp_quat0 = sim.body_xquat[:, self.tcp].clone()
        self.q0 = q0
        self.lo = self.tcp_pos0[0] + torch.tensor([-0.15, -0.05, -0.055], **f32)
        self.hi = self.tcp_pos0[0] + torch.tensor([0.25, 0.45, 0.10], **f32)
        self.reset(torch.ones(N, dtype=torch.bool, device=dev))

    @staticmethod
    def rest_heights(m, names, nobj):
        """resting height of every object: the table top minus the lowest point of its geoms in the body frame"""
        rest = []
        for i in range(nobj):
            b = names["body"].index("object%d" % i)
            zmin = 0.0
            for g in range(m["ngeom"]):
                if m["geom_bodyid"][g] != b:
                    continue
                if m["geom_dataid"][g] >= 0:
                    a, n = int(m["mesh_vertadr"][m["geom_dataid"][g]]), int(m["mesh_vertnum"][m["geom_dataid"][g]])
                    zmin = min(zmin, float((m["mesh_vert"].reshape(-1, 3)[a:a + n, 2] + m["geom_pos"].reshape(-1, 3)[g, 2]).min()))
                else:
                    zmin = min(zmin, float(m["geom_pos"].reshape(-1, 3)[g, 2] - m["geom_size"].reshape(-1, 3)[g, 2]))
            rest.append(0.453 + 0.03324 - zmin + 0.001)
        return rest

    def reset_blocks(self, mask):
        """arm at its start pose, objects re-placed, velocities / controller state / warm start cleared -- for the masked environments"""
        t, sim = self.torch, self.sim
        N = sim.nenv
        q = self.q0.clone()
        # objects on a jittered grid of the table area in front of the arm (one cell stays empty), random yaw
        ncol, ncell, x0, y0, dx, dy = self.grid
        no = self.nobj
        cells = t.argsort(t.rand(N, ncell, device=self.dev, generator=self.gen), dim=1)[:, :no]
        cx = x0 + dx * (cells % ncol).to(q.dtype) + 0.02 * (t.rand(N, no, device=self.dev, generator=self.gen) - 0.5)
        cy = y0 + dy * (cells // ncol).to(q.dtype) + 0.02 * (t.rand(N, no, device=self.dev, generator=self.gen) - 0.5)
        yaw = 3.14159 * t.rand(N, no, device=self.dev, generator=self.gen)
        for k, a in enumerate(self.blocks):
            q[:, a] = cx[:, k]; q[:, a + 1] = cy[:, k]; q[:, a + 2] = self.rest[k]
            q[:, a + 3] = t.cos(0.5 * yaw[:, k]); q[:, a + 4] = 0.0; q[:, a + 5] = 0.0; q[:, a + 6] = t.sin(0.5 * yaw[:, k])
        mk = mask.unsqueeze(1)
        sim.qpos.copy_(t.where(mk, q, sim.qpos))
        sim.qvel.mul_((~mk).to(sim.qvel.dtype))
        sim.pid.mul_((~mk).to(sim.pid.dtype))
        sim.qacc_warmstart.mul_((~mk).to(sim.qvel.dtype))

    def reset(self, mask):
        t, sim = self.torch, self.sim
        self.reset_blocks(mask)
        mk = mask.unsqueeze(1)
        sim.ctrl.copy_(t.where(mk, self.ctrl_hi.expand_as(sim.ctrl), sim.ctrl))
        sim.mocap_pos[:, 0].copy_(t.where(mk, self.tcp_pos0, sim.mocap_pos[:, 0]))       # reset_mocap2body_xpos
        sim.mocap_quat[:, 0].copy_(t.where(mk, self.tcp_quat0, sim.mocap_quat[:, 0]))

    def apply_action(self, a):
        t, sim = self.torch, self.sim
        sim.mocap_pos[:, 0].copy_(t.minimum(t.maximum(sim.mocap_pos[:, 0] + 0.01 * a[:, :3], self.lo), self.hi))
        sim.ctrl.copy_(self.ctrl_lo + (self.ctrl_hi - self.ctrl_lo) * (0.5 * (a[:, 3:4] + 1.0)))

    def sample_action(self):
        return self.torch.rand(self.sim.nenv, 4, device=self.dev, generator=self.gen) * 2 - 1

    def step_timed(self):
        self.sim.step()

    def on_palm(self):
        """healthy = every block still on (or above) the table"""
        z = self.torch.stack([self.sim.qpos[:, a + 2] for a in self.blocks], dim=1)
        return (z > 0.45).all(dim=1)

    def auto_reset(self):
        lost = ~self.on_palm()
        self.reset(lost)
        return lost


class RearrangeTcpWorkload(RearrangeWorkload):
    """BASELINE.json configs[3] with the reference's own control loop (SURVEY 8(d) row 4): a ~ U(-1,1)^6 = tool translation (3) +
    roll / yaw (2) + gripper (1) (ControlMode.TCP_ROLL_YAW, TcpSolverMode.MOCAP_IK, free_dof_tcp_arm.py:161-178).  TWO simulations
    per environment, as robogym/robot/composite/ur_gripper_arm.py:104-150 builds them: the solver arm (mocap weld, 40 substeps of
    0.001 s) turns the tool action into joint angles, the main scene (arm joints under mujoco-py's cascaded-PI controllers, 5
    blocks, 40 substeps + 2 forwards) tracks them -- robogym_b200.rearrange_arm.BatchedTcpArmController, two launches per
    env-step with the hand-off on the device."""

    action_dim = 6

    def __init__(self, sim, model, names, dev, gen, nobj, grid, solver_sim):
        import numpy as np
        import torch

        from robogym_b200.rearrange_arm import BatchedTcpArmController

        self.torch, self.sim, self.gen, self.dev = torch, sim, gen, dev
        self.solver = solver_sim
        m = model.host
        N = sim.nenv
        f32 = dict(dtype=torch.float32, device=dev)
        self.nobj, self.grid = nobj, grid
        self.blocks = [int(m["jnt_qposadr"][names["joint"].index("object%d:joint" % i)]) for i in range(nobj)]
        self.rest = torch.tensor(self.rest_heights(m, names, nobj), **f32)
        self.ctl = BatchedTcpArmController(sim, solver_sim, max_position_change=0.1, reset_controller_error=True)
        q0 = torch.tensor(m["qpos0"], **f32).repeat(N, 1)
        q0[:, self.ctl.arm_qadr_main] = torch.tensor(np.deg2rad([135.0, -90.0, 135.0, -100.0, -240.0, 135.0]), **f32)   # TABLETOP_EXPERIMENT_INITIAL_POS
        self.q0 = q0
        self.ctrl0 = torch.zeros(N, m["nu"], **f32)
        self.ctrl0[:, self.ctl.arm_act_main] = q0[:, self.ctl.arm_qadr_main]
        self.pending = None
        self.tcp_main = names["body"].index("robot0:gripper_tcp")
        self.reset(torch.ones(N, dtype=torch.bool, device=dev))
        sim.forward()
        self.ctl.reset()
        p0 = sim.body_xpos[0, self.tcp_main].clone()
        self.lo = p0 + torch.tensor([-0.25, -0.15, -0.06], **f32)      # episode ends when the tool leaves the table-top workspace
        self.hi = p0 + torch.tensor([0.35, 0.55, 0.25], **f32)

    def reset(self, mask):
        t, sim, sol = self.torch, self.sim, self.solver
        RearrangeWorkload.reset_blocks(self, mask)
        mk = mask.unsqueeze(1)
        sim.ctrl.copy_(t.where(mk, self.ctrl0, sim.ctrl))
        # the helper arm restarts with the main arm (JointControlledTcpArm.reset): joints re-synced every step anyway
        keep = (~mk).to(sol.qvel.dtype)
        sol.qvel.mul_(keep); sol.pid.mul_(keep); sol.qacc_warmstart.mul_(keep)
        sol.qpos[:, self.ctl.arm_qadr_solver] = t.where(mk, sim.qpos[:, self.ctl.arm_qadr_main], sol.qpos[:, self.ctl.arm_qadr_solver])

    def apply_action(self, a):
        self.pending = a

    def step_timed(self):
        self.ctl.step(self.pending)

    def auto_reset(self):
        p = self.sim.body_xpos[:, self.tcp_main]
        out = ((p < self.lo) | (p > self.hi)).any(dim=1) | ~self.on_palm()
        self.reset(out)
        return out

    def sample_action(self):
        return self.torch.rand(self.sim.nenv, 6, device=self.dev, generator=self.gen) * 2 - 1


DUMP_LIMIT_BYTES = 64 << 20


def dump_outputs(arrays, out_dir, limit=DUMP_LIMIT_BYTES, seed=0):
    """Write each [nenv, ...] array as out_dir/<name>.npy: float32 arrays as they are, integer ones as float64 (exact).
    When they would take more than `limit` bytes in all, the same fixed, seeded sample of environments is taken from every
    array and its indices are written as env_index.npy."""
    import numpy as np

    arrays = {k: v.cpu().numpy() for k, v in arrays.items()}
    arrays = {k: v.astype(np.float32 if v.dtype == np.float32 else np.float64) for k, v in arrays.items()}
    nenv = next(iter(arrays.values())).shape[0]
    per_env = sum(v.nbytes // nenv for v in arrays.values())
    if per_env * nenv > limit:
        rows = np.sort(np.random.RandomState(seed).choice(nenv, max(1, (limit - 8 * nenv) // per_env), replace=False))
        arrays = {k: v[rows] for k, v in arrays.items()}
        arrays["env_index"] = rows.astype(np.float64)
    os.makedirs(out_dir, exist_ok=True)
    for k, v in arrays.items():
        np.save(os.path.join(out_dir, k + ".npy"), v)


def run_gpu_arm(args):
    import numpy as np
    import torch

    from robogym_b200 import build, engine

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    dist = None
    if world > 1:
        import torch.distributed as dist

        torch.cuda.set_device(local)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    dev = torch.device("cuda", local)
    torch.cuda.set_device(dev)
    build.build()
    cfg = CONFIGS[args.config]
    blob = load_blob(cfg["asset"])
    names = json.load(open(os.path.join(ROOT, "robogym_b200", "assets", cfg["asset"] + ".names.json")))
    model = engine.DeviceModel(blob, local)
    strong = args.scaling == "strong"
    NBOX = cfg["nenv"]
    N = NBOX // world if strong else NBOX                      # weak: the config's batch per GPU; strong: per box
    if os.environ.get("RG_BENCH_NENV"):                        # experiments only
        N = int(os.environ["RG_BENCH_NENV"])
    lo_env, hi_env = shard_range(N * world, rank, world)
    caps = cfg["caps"]
    if os.environ.get("RG_BENCH_CAPS"):        # experiments: "contacts,rows,dofs" (0 = engine default)
        caps = tuple(int(x) for x in os.environ["RG_BENCH_CAPS"].split(","))
    nsub = cfg.get("nsub", NSUB)
    rearrange = cfg.get("workload") in ("rearrange", "rearrange_tcp")
    tcp = cfg.get("workload") == "rearrange_tcp"
    outputs = ("site_xpos", "act_force", "ncon", "warn") + (("body_xpos", "body_xquat") if rearrange else ())
    sim = engine.BatchedSim(model, N, nsub, outputs=outputs, contact_capacity=caps[0], row_capacity=caps[1], dofs_per_contact=caps[2])
    m = model.host
    nu, nq, nv = m["nu"], m["nq"], m["nv"]
    gen = torch.Generator(device=dev)
    gen.manual_seed(rank_seed(1234, rank))
    solver = None
    if tcp:
        solver_model = engine.DeviceModel(load_blob(cfg["solver_asset"]), local)
        solver = engine.BatchedSim(solver_model, N, nsub, outputs=("body_xpos", "body_xquat", "warn"))
        wl = RearrangeTcpWorkload(sim, model, names, dev, gen, cfg["nobj"], cfg["grid"], solver)
    else:
        wl = RearrangeWorkload(sim, model, names, dev, gen, cfg["nobj"], cfg["grid"]) if rearrange else Workload(sim, model, names, dev, gen)
    nact = wl.action_dim
    rnd = None
    if args.randomize:
        if rearrange:
            raise SystemExit("--randomize: dactyl configs only")
        from robogym_b200.locked_env import TorchRand
        from robogym_b200.randomization import FullCubeRandomizer, LockedRandomizer

        R = (FullCubeRandomizer if args.config == "full_perpendicular" else LockedRandomizer)(m, names, TorchRand(torch, dev, rank_seed(77, rank)), torch, dev, torch.float32)
        R.apply(sim, R.sample(N))                                   # one draw per environment (episode-level re-draws are not part of the timed loop)
        rnd = dict(R=R, ts=R.timestep_state(N), wind=R.wind_state(N, nsub * R.timestep0), timestep=sim.enable_per_env_timestep(),
                   xfrc=sim.xfrc_applied if sim.xfrc_applied is not None else sim.enable_xfrc())

    def randomize_step():
        """RandomizedTimestepWrapper.step / RandomizedWindWrapper.step: the next env-step's timestep and gust (untimed, like the action sampling)"""
        if rnd is not None:
            rnd["timestep"].copy_(rnd["R"].next_timestep(rnd["ts"]))
            rnd["R"].next_wind(rnd["wind"], rnd["xfrc"])
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)   # > L2 (126 MB)
    warmup = max(args.warmup, 3)
    for _ in range(warmup):
        wl.apply_action(wl.sample_action())
        randomize_step()
        wl.step_timed()
        wl.auto_reset()
    torch.cuda.synchronize()

    # ---- timed region 1: device-resident (kernel) throughput
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    if dist is not None:
        dist.barrier()
    torch.cuda.synchronize()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
    resets = torch.zeros((), dtype=torch.int64, device=dev)
    ncon_sum = torch.zeros((), dtype=torch.float64, device=dev)
    warn = torch.zeros((), dtype=torch.int32, device=dev)
    ncon_max = torch.zeros((), dtype=torch.int32, device=dev)
    last = None
    for k in range(args.steps):
        nxt = wl.sample_action()
        flush.zero_()                                   # evict L2 between timed iterations (outside the event pair)
        wl.apply_action(nxt)
        randomize_step()
        ev[k][0].record()
        wl.step_timed()                                 # one launch (two for the dual-simulation rearrange loop, hand-off included)
        ev[k][1].record()
        if args.dump_outputs and k == args.steps - 1:   # what the last timed step handed its caller, before the auto-reset
            last = {n: getattr(sim, n).clone() for n in ("qpos", "qvel", "ctrl") + outputs}
            if solver is not None:
                last.update({"solver_" + n: getattr(solver, n).clone() for n in ("qpos", "qvel", "ctrl")})
        ncon_sum += sim.ncon.double().mean()
        ncon_max = torch.maximum(ncon_max, sim.ncon.max())
        warn |= sim.warn.max() if solver is None else torch.maximum(sim.warn.max(), solver.warn.max())
        resets += wl.auto_reset().sum()                 # in-loop auto-reset (untimed torch ops, like the action sampling)
    torch.cuda.synchronize()
    if dist is not None:
        dist.barrier()
    clocks = sampler.stop() if rank == 0 else None
    step_ms = [a.elapsed_time(b) for a, b in ev]
    t_dev = max_over_ranks(sum(step_ms) / 1e3, dist, dev)
    total_steps = sum_over_ranks(float(N * args.steps), dist, dev)
    value = total_steps / t_dev
    on_palm = float(wl.on_palm().float().mean().item())
    warn = int(warn.item())

    # ---- timed region 2: end to end through the public API with host buffers: every step the policy's ACTIONS come from
    # pinned host memory (H2D), the batched facade turns them into controls on the device (what RobotEnv.step does per
    # environment on the host, robot_interface.py:247-278), the step runs, and the observation (qpos, qvel) is read back (D2H)
    # and waited for, because the next action depends on it
    h_act = [torch.empty(N, nact, dtype=torch.float32).pin_memory() for _ in range(2)]
    d_act = torch.empty(N, nact, dtype=torch.float32, device=dev)
    h_q = torch.empty(N, nq, dtype=torch.float32).pin_memory()
    h_v = torch.empty(N, nv, dtype=torch.float32).pin_memory()
    rng = np.random.RandomState(rank_seed(99, rank) % (2 ** 31))
    acts = [(rng.uniform(-1, 1, (N, nact)).astype(np.float32)) for _ in range(args.steps)]
    if dist is not None:
        dist.barrier()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for k in range(args.steps):
        buf = h_act[k & 1]
        buf.numpy()[:] = acts[k]                        # the policy's output lands in pinned host memory
        flush.zero_()                                   # same cold L2 as the device-timed region (0.05 ms of memset, inside the timing)
        d_act.copy_(buf, non_blocking=True)             # H2D of this step's inputs
        wl.apply_action(d_act)
        randomize_step()
        wl.step_timed()
        h_q.copy_(sim.qpos, non_blocking=True)          # D2H of this step's result
        h_v.copy_(sim.qvel, non_blocking=True)
        wl.auto_reset()                                 # the environment loop restarts dropped cubes (else steps get cheaper)
        torch.cuda.synchronize()                        # the host consumes the observation every step
    e1.record()
    torch.cuda.synchronize()
    t_e2e = max_over_ranks(e0.elapsed_time(e1) / 1e3, dist, dev)
    e2e_value = total_steps / t_e2e

    if rank == 0:
        peak, peak_kind = measured_peak()
        kernel_s = statistics.mean(step_ms) / 1e3
        achieved = ALGO_BYTES_PER_ENV_STEP * N / kernel_s / 1e9
        info = sim.launch_info()
        prof = newest_profile_metrics() if args.config == "locked" else None
        sm_mhz = (clocks or {}).get("sm_mhz") or 1965.0
        roof = {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                "traffic": prof["dram_bytes"] * N / NENV_PER_GPU if prof else None,   # the capture is one 8192-env launch
                "traffic_unit": "bytes per launch (dram__bytes_read+write of rg_step_kernel, ncu --set full; %s)" % (prof["file"] if prof else "no capture"),
                "algorithmic_bytes_per_launch": ALGO_BYTES_PER_ENV_STEP * N,
                "peak_source": peak_kind + " (MEASURED_PEAKS.json hbm_gbs)" if peak_kind == "measured" else "fallback 6.65 TB/s",
                "note": "algorithmic 1664 B/env-step; the path is instruction-issue bound, not HBM bound (DESIGN.md): see fp32_issue_frac"}
        if prof:
            # SURVEY 8(d) asks for both fractions: warp instructions issued per second against 148 SMs x 4 schedulers x clock
            inst_per_env_step = prof["warp_inst"] / NENV_PER_GPU
            per_gpu = value / world
            roof["fp32_issue_frac"] = inst_per_env_step * per_gpu / (148 * 4 * sm_mhz * 1e6)
            roof["warp_inst_per_env_step"] = inst_per_env_step
        line = {
            "metric": METRIC, "value": value, "unit": "env-steps/s", "n_gpus": world, "steps": args.steps, "warmup": warmup,
            "ms_per_step": t_dev / args.steps * 1e3, "higher_is_better": True, "scaling": "strong" if strong else "weak", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic",
            "config": {"workload": cfg["label"] + (", batch %d per GPU, per env-step: solver arm forward + 40 substeps of 0.001 s, main scene 40 substeps + 2 forwards, "
                                                   "a~U(-1,1)^6 relative tool actions (max_position_change 0.1, arm_reset_controller_error); auto-reset of environments that lost an object" % N if tcp else
                                                   ", batch %d per GPU, 20 substeps of 0.002 s + forward per env-step, a~U(-1,1)^4: mocap target += 0.01 a[:3] "
                                                   "(clipped to a box over the table), gripper target from a[3]; auto-reset of environments that lost an object" % N if rearrange else
                                                   ", batch %d per GPU, 10 substeps of 0.008 s + forward per env-step, relative actions a~U(-1,1): "
                                                   "ctrl = clip(P qpos + a*range/2), auto-reset of environments whose cube left the palm" % N),
                       "randomize": bool(args.randomize), "envs_per_gpu": N, "substeps": nsub, "physics_substeps_per_s": value * nsub,
                       "l2": "flushed between timed steps (256 MiB memset outside the per-step event pairs)",
                       "launch": info, "cubes_on_palm_at_end": on_palm, "resets_in_timed_region_rank0": int(resets.item()),
                       "mean_contacts": float(ncon_sum.item()) / args.steps, "max_contacts": int(ncon_max.item()), "warn_bits": warn, "env_shard_rank0": [lo_env, hi_env]},
            "clocks": clocks,
            "e2e": {"value": e2e_value, "unit": "env-steps/s", "h2d_bytes_per_step": N * nact * 4, "d2h_bytes_per_step": N * (nq + nv) * 4},
            # per step and simulation: rg_step_kernel + rg_order_kernel (work-ordered schedule of the next launch); the dual-simulation
            # loop also runs a forward of the solver arm (sync to the main arm) before its step
            "gpu_launches": (5 if tcp else 2) * args.steps * world,
            "roofline": roof,
        }
        if world == 1:
            try:
                if tcp:
                    line["cpu_baseline"] = cpu_baseline_rearrange_tcp(blob, load_blob(cfg["solver_asset"]), seconds=float(os.environ.get("RG_CPU_BASELINE_SECONDS", "10")))
                elif rearrange:
                    line["cpu_baseline"] = cpu_baseline_rearrange(blob, names, seconds=float(os.environ.get("RG_CPU_BASELINE_SECONDS", "10")))
                else:
                    line["cpu_baseline"] = cpu_baseline(blob, seconds=float(os.environ.get("RG_CPU_BASELINE_SECONDS", "10")))
            except Exception as e:  # the baseline is reported, never required for the GPU number
                line["cpu_baseline"] = {"value": None, "unit": "env-steps/s", "cores": 0, "kind": "port", "sample": f"failed: {e}"}
        print(json.dumps(line), flush=True)
        if last is not None:
            dump_outputs(last, args.dump_outputs)
    if dist is not None:
        dist.destroy_process_group()


def model_site(model, name):
    import json as _json

    names = _json.load(open(os.path.join(ROOT, "robogym_b200", "assets", "dactyl_locked.names.json")))
    return names["site"].index(name)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--scaling", default="weak", choices=["weak", "strong"], help="weak: 8192 envs per GPU; strong: 8192 envs per box")
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--randomize", action="store_true", help="dactyl configs: per-environment model parameters drawn with the reference wrappers' distributions "
                                                             "(locked.py:263-277 / full_perpendicular.py:425-440), per-step timestep and wind -- SURVEY 8(d) cfg 3's randomize=True")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write what the last timed step of the device-resident region computed (rank 0's "
                                                           "environments: qpos, qvel, ctrl and the engine's outputs) as DIR/<name>.npy; "
                                                           "the inputs are seeded, so two builds can be compared output for output")
    ap.add_argument("--config", default="locked", choices=sorted(CONFIGS), help="locked = BASELINE.json's headline config; full_perpendicular = configs[2]; rearrange_blocks = configs[3]; rearrange_ycb = configs[4]")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs: the GPU path only")
    if args.impl == "reference":
        run_reference_arm(args)
    else:
        run_gpu_arm(args)


if __name__ == "__main__":
    main()
