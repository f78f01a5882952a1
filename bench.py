#!/usr/bin/env python
"""Headline benchmark: drone-steps/s of the full hot path on synthetic swarms (BASELINE.json).

    python bench.py --gpus N --steps K --warmup W            # this framework (one process per GPU)
    python bench.py --impl reference --gpus N --steps K ...   # the reference's own classes on the host cores

Workload (config.workload): SURVEY.md 8(d) C5 -- per GPU 125 000 independent environments x 8 drones
(1M drones), 240 Hz; every drone-step = Lemniscate reference -> LQR-yank-omega nominal -> order-3
CBF-QP (28 pair rows + 8 obstacle rows + box/force bounds per env) -> YankOmega inner loop ->
DYN_GND_DRAG_DW physics (ground effect, drag, pairwise downwash) -> 20-float observation.

One bench "step" = one ``mds_rollout`` call = ONE kernel launch = ``--fuse`` control steps of every drone with the
observation and body rates in registers from step to step (environments are independent; a lane group owns its env);
every step's observation is also written to HBM (obs log), as the reference's loop keeps every obs.
``value``   : drone-steps/s, state resident in HBM, CUDA events on the launching stream, max over ranks (weak scaling:
              ``--envs`` environments per GPU).
``strong``  : BASELINE.json configs[4] as stated -- the FIXED swarm (``--envs`` environments in total) sharded over the
              N GPUs; efficiency = strong value / (N x the per-GPU rate of the full-size shard).
``e2e``     : the same metric through the per-call API with HOST buffers (multidronesim_b200.HostPipeline): every
              control step copies the step's references host -> device from pinned memory and the new observation
              device -> host, copies overlapped with the neighbouring steps' kernels on their own streams; with
              ``pcie_ceiling`` = plain cudaMemcpyAsync loops of the same sizes on all ranks at once, and ``fused`` =
              the K-step host call (multidronesim_b200.HostRollout: one launch + one large D2H per K steps).
``roofline``: the dominant (only) kernel of the timed region, rollout_loop_kernel.  It is FP32-pipe-bound (the state
              never leaves the registers), so achieved = algorithmic flop per launch / launch duration against the
              non-tensor FP32 peak (FMA-chain microbenchmark measured live; nominal SMs x 128 x 2 x clock if the
              microbenchmark reads < 95 % of it); ``frac_counters`` = the hardware's own fraction (executed fadd + fmul
              + 2 ffma per cycle / 2 x ffma peak) from the committed ncu capture; its HBM view is reported inside.
              ``roofline_ctrl`` / ``roofline_physics``: the per-call kernels (what ``e2e`` launches) against the
              measured HBM copy bandwidth.  No tensor cores on this path: nothing is a dense contraction.
``configs`` : the other BASELINE.json configurations at N = 1 (C2 4096 x 1 geometric, C3 order 2 16 384 x 8, C4 65 536
              fp64 model comparison, C5 in fp64), each with its own roofline fraction and clocks.
``cpu_baseline``: the reference's own trajectories / controllers / CBF builder / QP tracker (oracle/_ref, ``kind:
              "reference"``) around the oracle env step and QP solver on all host cores, bounded sample;
              ``cpu_baseline_port`` = the numpy port of the same algorithms (oracle/pipeline.py).
"""
from __future__ import annotations

import argparse
import json
import multiprocessing as mp
import os
import statistics
import subprocess
import sys
import threading
import time

# one BLAS thread per worker process: the CPU arm parallelises over processes (one env per core)
for _v in ("OMP_NUM_THREADS", "OPENBLAS_NUM_THREADS", "MKL_NUM_THREADS"):
    os.environ.setdefault(_v, "1")

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

N_DRONES = 8
SWARM_OBSTACLES = [[0.2, 0.0, 0.5, 0.1]]  # == multidronesim_b200.scenarios.SWARM_OBSTACLES (checked in run_gpu_arm)
CBF_ORDER = 3
METRIC = "drone-steps/sec (DYN_GND_DRAG_DW + LQR + order-3 CBF-QP, 8 drones/env)"
# Algorithmic work per drone-step of the C5 path (DESIGN.md "Roofline"): FP32 operations of the closed-form math
# (add / mul / compare / min-max = 1, fma = 2, transcendental / div / sqrt = 1), hand-counted per stage.  4.5 barrier rows
# per drone (3.5 pair rows under the half-ownership + 1 obstacle row) at ~105 flop, the per-drone projection and row tests,
# 3.5 downwash pair terms.  Cross-check (profiles/r2_ncu_kernels.txt): ncu's executed fadd + fmul + 2 ffma per drone-step is
# 1114; the table adds the compares / min-max / MUFU ops those counters leave out.
ALGO_FLOP_PER_DRONE_STEP = {"traj": 70, "lqr_yank": 120, "cbf_rows": 475, "projection_and_row_tests": 90, "lowlevel": 150,
                            "physics_gnd_drag_dw_n8": 380, "obs": 60}
ALGO_FLOP_GEOMETRIC = {"traj": 50, "geometric_ctrl_and_mixer": 600, "physics_gnd_drag": 240, "obs": 60}  # C2 (SURVEY 8d: ~0.95 kflop)
# Algorithmic HBM bytes per drone-step (fp32), per kernel of the rollout (DESIGN.md "Roofline"):
ALGO_BYTES_CTRL_F32 = {"read_obs": 80, "read_traj_spec": 48, "read_pid": 24, "write_pid": 24, "write_action": 16}
ALGO_BYTES_PHYS_F32 = {"read_state": 68, "read_action": 16, "write_state": 68, "write_obs": 80}  # SURVEY 8(d): 232 B
# the K-steps-in-one-launch kernel, per drone and per LAUNCH (not per step): initial obs + body rates + trajectory spec,
# PID state in and out, final state + obs + action
ALGO_BYTES_OBS_LOG_PER_STEP_F32 = 80  # the observation of every control step, written to its log slot
ALGO_BYTES_LOOP_PER_LAUNCH_F32 = {"read_obs": 80, "read_body_rates": 12, "read_traj_spec": 48, "read_pid": 24, "write_pid": 24,
                                  "write_state": 68, "write_obs": 80, "write_action": 16}
SM_FP32_LANES, SM_FP64_LANES = 128, 64  # FMA lanes per SM and clock on B200 (ncu: sm__sass_thread_inst_executed_op_{f,d}fma peak_sustained)


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--envs", type=int, default=125000, help="environments per GPU (weak scaling); also the TOTAL of the strong-scaling leg")
    ap.add_argument("--fuse", type=int, default=24, help="control steps per fused launch (one bench step)")
    ap.add_argument("--settle", type=int, default=3024, help="untimed control steps that take the swarm from its start at rest into its steady "
                                                               "lap before warm-up, in both arms (default: one lemniscate period); the start-up "
                                                               "transient has heavy-tailed QP iteration counts")
    ap.add_argument("--e2e-steps", type=int, default=48, help="control steps timed on the host-buffer path")
    ap.add_argument("--cpu-seconds", type=float, default=12.0, help="wall budget of each cpu_baseline sample (reference classes, port)")
    ap.add_argument("--ref-steps-per-step", type=int, default=8, help="control steps per reference-arm step and worker")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-configs", action="store_true", help="skip the secondary configurations (C2, C3 order 2, C4, C5 fp64)")
    ap.add_argument("--no-strong", action="store_true")
    ap.add_argument("--streams", type=int, default=2, help="sub-swarms per GPU, each advanced on its own CUDA stream (multidronesim_b200.SwarmStreams): "
                                                           "the tail wave of one sub-swarm's launch is filled by the next launch of another; 1 = one launch per step")
    ap.add_argument("--dtype", default="f32", choices=["f32", "f64"])
    ap.add_argument("--dump-outputs", metavar="DIR", help="after the timed steps, write what the last one computed to DIR/<name>.npy: obs_log.npy = "
                                                          "the observation after each control step of that launch [T, n, 8, 20] for a fixed, seeded "
                                                          "sample of n <= 2048 of (rank 0's) environments in ascending order (T = fuse unless the log "
                                                          "of one environment exceeds the 48 MB budget; then its last T steps), rollout_stats.npy = "
                                                          "the statistics of the timed steps (MDS_STAT_*, float64)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes the outputs of the b200 arm")
    return args


# ----------------------------------------------------------------------------------------------
# CPU arm: the reference-style loop (per-drone Python loops) on the host cores
# ----------------------------------------------------------------------------------------------
def _lem_specs():
    import numpy as np
    phase = (2 * np.pi / (N_DRONES + 0.25)) * np.arange(N_DRONES)
    return [dict(a=1.0, center=np.array([0, 0, 0.5]), omega=0.5, yaw_rate=0.0, phase_shift=float(p)) for p in phase]


def _oracle_env(env_index, seed=3):
    import numpy as np
    from oracle import trajectories as otj
    from oracle.aviary import OracleCtrlAviary
    from oracle.constants import DroneModel as ODM, Physics as OPH
    N = N_DRONES
    specs = _lem_specs()
    rng = np.random.default_rng(np.random.SeedSequence([seed, 10_000_000 + env_index]))
    init = np.array([otj.Lemniscate(**sp)(0.0)[0] for sp in specs]) + rng.normal(0, 0.02, (N, 3))
    init[:, 2] += 0.04 * np.arange(N)
    env = OracleCtrlAviary(ODM.CF2P, N, initial_xyzs=init, physics=OPH.DYN_GND_DRAG_DW)
    return env, [otj.Lemniscate(**sp) for sp in specs]


_WORKER = {}


def reference_classes_available():
    from oracle import ref_pipeline
    return ref_pipeline.reference_root() is not None


def _cpu_worker_step(args):
    """Advance this worker's private environment by `steps` control steps; returns drone-steps done.
    kind "port": oracle/pipeline.run_cbf (numpy restatement).  kind "reference": the reference's own classes
    (oracle/ref_pipeline.ReferenceLoop), continuing from wherever the port left the same environment."""
    from oracle import pipeline as opl
    env_index, steps, kind = args
    if env_index not in _WORKER:
        env, trajs = _oracle_env(env_index)
        _WORKER[env_index] = dict(env=env, trajs=trajs, ctrls=opl.make_controllers(env, "yank10"), t=0.0, loop=None)
    w = _WORKER[env_index]
    if kind == "reference":
        from oracle import ref_pipeline
        if w["loop"] is None:
            w["loop"] = ref_pipeline.ReferenceLoop(w["env"], CBF_ORDER, _lem_specs(), SWARM_OBSTACLES)
            w["loop"].adopt_inner_loop_state(w["ctrls"])
            w["loop"].t = w["t"]
        w["loop"].run(steps)
        w["t"] = w["loop"].t
        for mine, ref_c in zip(w["ctrls"], w["loop"].ctrl):  # hand the inner-loop state back, should the port continue
            toc = ref_c.yo_controller.thrust_omega_ctrl
            mine.low.inner.last_omega, mine.low.inner.integral = toc.last_omega.copy(), toc.integral_omega_e.copy()
    else:
        if w["loop"] is not None:
            w["loop"] = None
        opl.run_cbf(w["env"], w["trajs"], CBF_ORDER, steps, obstacles=SWARM_OBSTACLES, ctrls=w["ctrls"], t0=w["t"], log=False)
        w["t"] += steps * w["env"].CTRL_TIMESTEP
    return N_DRONES * steps


def _describe(kind):
    if kind == "reference":
        return ("the reference's own Lemniscate / LQRYankOmegaController / YankOmegaController / DroneCBF._build_ineq_const / DroneQPTracker "
                "(oracle/_ref, unmodified) in the loop of simulations/CBFTestOrd3.py:305-360; env.step = oracle/aviary.py and cvxopt.solvers.qp = "
                "oracle/qp.py (neither is in the reference tree)")
    return ("oracle/pipeline.run_cbf (the reference's algorithms restated in numpy; cvxopt -> oracle active-set QP, PyBullet env -> restated "
            "DYN_GND_DRAG_DW step)")


def cpu_baseline(seconds, settle=3024):
    """bounded samples: every host core advances its own C5 environment; first with the reference's own classes (if
    oracle/_ref or /root/reference is there), then with the numpy port; both after `settle` steps of the (faster) port"""
    cores = os.cpu_count() or 1
    ctx = mp.get_context("fork")
    out = {}
    with ctx.Pool(cores) as pool:
        pool.map(_cpu_worker_step, [(i, max(2, settle), "port") for i in range(cores)], chunksize=1)  # imports, gains, settle into steady flight
        kinds = (["reference"] if reference_classes_available() else []) + ["port"]
        for kind in kinds:
            per_task = 4 if kind == "reference" else 24
            pool.map(_cpu_worker_step, [(i, 2, kind) for i in range(cores)], chunksize=1)  # construct / warm
            done, t0, rounds = 0, time.perf_counter(), 0
            while time.perf_counter() - t0 < seconds:
                done += sum(pool.map(_cpu_worker_step, [(i, per_task, kind) for i in range(cores)], chunksize=1))
                rounds += 1
            dt = time.perf_counter() - t0
            out[kind] = {"value": done / dt, "unit": "drone-steps/s", "cores": cores, "kind": kind,
                         "sample": f"{cores} C5 environments x {N_DRONES} drones (one per core), {rounds * per_task} control steps each after {settle} "
                                   f"settling steps; {_describe(kind)}; {dt:.1f} s wall"}
    return out


def run_reference_arm(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cores = os.cpu_count() or 1
    S = args.ref_steps_per_step
    kind = "reference" if reference_classes_available() else "port"
    ctx = mp.get_context("fork")
    with ctx.Pool(cores) as pool:
        pool.map(_cpu_worker_step, [(i, max(1, args.settle), "port") for i in range(cores)], chunksize=1)  # settle into steady flight (fast port)
        for _ in range(max(1, args.warmup)):
            pool.map(_cpu_worker_step, [(i, 2, kind) for i in range(cores)], chunksize=1)
        t0 = time.perf_counter()
        done = 0
        for _ in range(args.steps):
            done += sum(pool.map(_cpu_worker_step, [(i, S, kind) for i in range(cores)], chunksize=1))
        dt = time.perf_counter() - t0
    value = done / dt
    sample = f"each step: {cores} C5 environments x {N_DRONES} drones (one per host core) advance {S} control steps; {_describe(kind)}"
    line = {"impl": "reference", "metric": METRIC, "value": value,
            "unit": "drone-steps/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * dt / args.steps,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": workload_config(args, cores * 1, per_gpu=False),
            "cpu_baseline": {"value": value, "unit": "drone-steps/s", "cores": cores, "kind": kind, "sample": sample},
            "e2e": {"value": value, "unit": "drone-steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    emit(line)


def workload_config(args, envs, per_gpu=True):
    return {"workload": "C5 swarm sweep: envs x 8 drones, Physics.DYN_GND_DRAG_DW 240 Hz, Lemniscate refs, LQR-yank-omega nominal, "
                        "order-3 CBF-QP (r_safe 0.125, zscale 2, poles -3/-3.6/-5.6) + sphere obstacle r=0.1 at (0.2, 0, 0.5), YankOmega inner loop",
            "envs_per_gpu" if per_gpu else "envs": envs, "drones_per_env": N_DRONES, "drone_model": "cf2p", "cbf_order": CBF_ORDER,
            "control_steps_per_step": args.fuse if per_gpu else args.ref_steps_per_step, "settle_steps": args.settle,
            "parallelism": f"env-sharded x{args.gpus}" + (f", {max(1, args.streams)} sub-swarms per GPU on their own CUDA streams" if per_gpu else ""),
            "obs": "every control step's observation is written to HBM (log ring of control_steps_per_step slots)",
            "l2": "working set (state+obs+traj specs+PID+obs log > 2 GB per GPU) exceeds the 126 MB L2; no flush needed"}


# ----------------------------------------------------------------------------------------------
# clocks
# ----------------------------------------------------------------------------------------------
class ClockSampler:
    Q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
        "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index):
        self.rows, self.proc, self.index = [], None, index

    def __enter__(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "50", "-i", str(self.index)],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except OSError:
            self.proc = None
        return self

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.perf_counter(), line.strip()))

    def __exit__(self, *a):
        if self.proc is not None:
            self.proc.terminate()
            try:
                self.proc.wait(timeout=2)
            except subprocess.TimeoutExpired:
                self.proc.kill()

    def summary(self, t0=None, t1=None):
        """clocks over the samples that arrived inside [t0, t1] (the timed region); if the region is too short for two
        samples, over everything since the sampler started (settle + warm-up + timed: the same kernels, same load)"""
        rows, window = self.rows, "all samples"
        if t0 is not None:
            inside = [r for r in self.rows if t0 <= r[0] <= t1 + 0.12]
            if len(inside) >= 2:
                rows, window = inside, "timed region"
            else:
                window = "settle + warm-up + timed region (timed region shorter than two sampling periods)"
        sm, mx, reasons = [], [], set()
        for _, r in rows:
            f = [x.strip() for x in r.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0])); mx.append(float(f[1]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"], "samples": 0}
        return {"sm_mhz": statistics.median(sm), "sm_max_mhz": max(mx), "reasons": sorted(reasons), "samples": len(sm), "window": window}


# ----------------------------------------------------------------------------------------------
# GPU arm
# ----------------------------------------------------------------------------------------------
def measured_peaks():
    try:
        return json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except (OSError, ValueError):
        return None


def snapshot(env, ctrl, ro):
    return (env.state_dict(), ctrl.low_level._a.clone(), ctrl.low_level._b.clone(), ro.t, ro.stats.clone())


def restore(env, ctrl, ro, snap):
    env.load_state_dict(snap[0])
    ctrl.low_level._a.copy_(snap[1])
    ctrl.low_level._b.copy_(snap[2])
    ro.t = snap[3]
    ro.stats.copy_(snap[4])


def ncu_capture(kernel, envs, dtype):
    """Row of the committed ncu --set full capture for this kernel at this size (profiles/ncu_traffic.json, written by
    tools/ncu_traffic.py from the .ncu-rep): DRAM bytes per launch and the executed FP instruction rates; or None."""
    try:
        tab = json.load(open(os.path.join(ROOT, "profiles", "ncu_traffic.json")))
    except (OSError, ValueError):
        return None
    for row in tab.get("kernels", []):
        if row["kernel"].startswith(kernel) and row["envs"] == envs and row["dtype"] == dtype:
            return row
    return None


def fp_peak(mds, sms, clocks, use_f64):
    """Non-tensor FMA peak in TFLOP/s: the live FMA-chain microbenchmark, or the nominal SMs x lanes x 2 x clock when the
    microbenchmark reads below 95 % of it (MEASURED_PEAKS.json carries no non-tensor figure)."""
    measured = mds._lib.fma_peak_tflops(use_f64=use_f64)
    mhz = (clocks or {}).get("sm_mhz") or (measured_peaks() or {}).get("sm_max_mhz") or 1965.0
    nominal = sms * (SM_FP64_LANES if use_f64 else SM_FP32_LANES) * 2 * mhz * 1e6 / 1e12
    if measured >= 0.95 * nominal:
        return measured, nominal, measured, "measured live: mds_fma_peak (16 independent FMA chains per thread, unrolled) on all SMs"
    return nominal, nominal, measured, (f"nominal {sms} SMs x {SM_FP64_LANES if use_f64 else SM_FP32_LANES} lanes x 2 x {mhz:.0f} MHz (the live FMA-chain "
                                        f"microbenchmark read {measured:.1f} TFLOP/s, below 95 % of it)")


DUMP_ENVS, DUMP_BYTES = 2048, 48 << 20  # --dump-outputs: environments sampled from the swarm, and the byte budget of their observation log


def dump_outputs(out_dir, rings, stats):
    """--dump-outputs: the observation log of the last launch (``rings``: one [F, E_p, N, 20] tensor per sub-swarm, in env order) for a
    sample of environments drawn with a fixed seed, so that the same arguments select the same environments in every run, and the
    statistics of the timed steps"""
    import numpy as np
    import torch
    F, _, N, C = rings[0].shape
    offsets = np.cumsum([0] + [r.shape[1] for r in rings])
    slot_bytes = N * C * rings[0].element_size()
    T = min(F, DUMP_BYTES // slot_bytes)  # the last T control steps of one environment fit the budget (all of them unless F is huge)
    n = max(1, min(int(offsets[-1]), DUMP_ENVS, DUMP_BYTES // (T * slot_bytes)))
    envs = np.sort(np.random.default_rng(0).choice(int(offsets[-1]), n, replace=False))
    parts = [r[F - T:, torch.as_tensor(envs[(envs >= b0) & (envs < b1)] - b0, device=r.device)] for r, b0, b1 in zip(rings, offsets[:-1], offsets[1:])]
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "obs_log.npy"), torch.cat(parts, dim=1).cpu().numpy())
    np.save(os.path.join(out_dir, "rollout_stats.npy"), stats.cpu().numpy())


def time_launches(torch, fn, reps, swarm=None):
    """CUDA-event time of ``reps`` calls of ``fn`` on the current stream; with ``swarm`` (SwarmStreams) the sub-swarm streams are
    forked after the first event and joined before the second, as in the headline's timed region"""
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    w0 = time.perf_counter()
    e0.record()
    if swarm is not None:
        swarm.fork()
    for _ in range(reps):
        fn()
    if swarm is not None:
        swarm.join()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1), w0, time.perf_counter()


def run_gpu_arm(args):
    cpu = None
    rank_env = int(os.environ.get("RANK", "0"))
    if rank_env == 0 and args.gpus == 1 and not args.no_cpu_baseline:
        cpu = cpu_baseline(args.cpu_seconds, settle=args.settle)  # before CUDA is initialised in this process (fork-safe)

    import torch
    import torch.distributed as dist

    import multidronesim_b200 as mds
    from multidronesim_b200 import scenarios

    assert scenarios.SWARM_OBSTACLES == SWARM_OBSTACLES
    rank, local_rank, world = mds.dist.init_from_env()
    if world != args.gpus:
        raise SystemExit(f"--gpus {args.gpus} but WORLD_SIZE={world}: launch with torchrun --nproc-per-node {args.gpus}")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    dtype = torch.float32 if args.dtype == "f32" else torch.float64
    esz = 4 if dtype == torch.float32 else 8
    E, N, F, K, W = args.envs, N_DRONES, args.fuse, args.steps, max(3, args.warmup)
    D = E * N
    sms = mds._lib.device_info()["sm_count"]

    P_STREAMS = max(1, args.streams)

    def barrier():
        if world > 1:
            dist.barrier()

    def max_over_ranks(x):
        t = torch.tensor([x], device=dev, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def timed_swarm(n_envs, env_offset, clk=None, dump_dir=None):
        """settle + warm up + time K bench steps of an n_envs-environment swarm cut into P_STREAMS sub-swarms; every control step's
        observation is materialised in HBM (per sub-swarm a ring of F log slots, reused by each launch), as the reference's loop
        does (observations.append(obs)): a drone-step includes its 80 B observation write.  ``dump_dir``: dump_outputs() after timing"""
        swarm, subs = scenarios.cbf_swarm_streams(n_envs, P_STREAMS, N, order=CBF_ORDER, dtype=dtype, device=dev, env_offset=env_offset)
        rings = [torch.empty(F, s_["env"].NUM_ENVS, N, 20, device=dev, dtype=dtype) for s_ in subs]
        step = lambda: swarm.run(F, obs_logs=rings, log_every=1)
        for _ in range(args.settle // F + W):
            step()
        swarm.synchronize()
        swarm.reset_stats()
        torch.cuda.synchronize()
        barrier()
        cur = torch.cuda.current_stream(dev)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        w0 = time.perf_counter()
        e0.record(cur)
        swarm.fork()          # the sub-swarm streams start after e0 ...
        for _ in range(K):
            step()
        swarm.join()          # ... and e1 is recorded after all of them
        e1.record(cur)
        torch.cuda.synchronize()
        w1 = time.perf_counter()
        if dump_dir:
            dump_outputs(dump_dir, rings, swarm.stats())
        barrier()
        if not all(r.plan() == 6 for r in swarm.rollouts):
            raise SystemExit("bench.py assumes the K-steps-in-one-launch plan")
        return e0.elapsed_time(e1), w0, w1, swarm.stats().clone()

    # ---- device-resident headline -------------------------------------------------------------
    with ClockSampler(local_rank) as clk:  # sampling starts with the settle phase: nvidia-smi needs ~0.2 s to deliver its first line
        ms, t_wall0, t_wall1, stats_rank = timed_swarm(E, rank * E, dump_dir=args.dump_outputs if rank == 0 else None)
        time.sleep(0.12)  # let the sample that covers the end of the region arrive
    ms_max = max_over_ranks(ms)
    value = world * D * F * K / (ms_max * 1e-3)
    stats_all = mds.dist.gather_stats(stats_rank)  # the path's only collective (NCCL all-gather of 8 doubles per rank)
    stats = dict(zip(mds._lib.STAT_NAMES, mds.dist.reduce_stats(stats_all).tolist()))
    clocks = clk.summary(t_wall0, t_wall1)
    torch.cuda.empty_cache()

    # one full-size swarm for the per-call replay and the host-buffer path, settled like the headline's
    sc = scenarios.cbf_swarm(E, N, order=CBF_ORDER, dtype=dtype, device=dev, env_offset=rank * E)
    env, ro, ctrl = sc["env"], sc["rollout"], sc["ctrl"]
    obs_ring = torch.empty(F, E, N, 20, device=dev, dtype=dtype)
    for _ in range(args.settle // F + W):
        ro.run(F, obs_log=obs_ring, log_every=1)
    torch.cuda.synchronize()
    ro.reset_stats()
    snap = snapshot(env, ctrl, ro)

    # ---- roofline of the dominant kernel: the K-steps-in-one-launch rollout kernel (this rank) ----------------
    # Every bench step is one launch of rollout_loop_kernel per sub-swarm (F control steps with the state in registers); the
    # launches of the P_STREAMS sub-swarms overlap on the GPU, so the kernel's duration per bench step is the timed region / K.
    n_steps = K * F
    launch_ms = ms / K
    peaks = measured_peaks()
    hbm_peak = peaks["hbm_gbs"] if peaks else 6650.0
    peak_src = "MEASURED_PEAKS.json hbm_gbs, of measured (sustained copy)" if peaks else "fallback 6.65 TB/s, of fallback"
    sfx = "float" if dtype == torch.float32 else "double"
    use_f64 = dtype == torch.float64
    fpk, fpk_nominal, fpk_chain, fpk_src = fp_peak(mds, sms, clocks, use_f64)
    flop_step = sum(ALGO_FLOP_PER_DRONE_STEP.values())
    bytes_launch = (sum(ALGO_BYTES_LOOP_PER_LAUNCH_F32.values()) + F * ALGO_BYTES_OBS_LOG_PER_STEP_F32) * esz // 4
    tf = flop_step * D * F / (launch_ms * 1e-3) / 1e12
    gbs = bytes_launch * D / (launch_ms * 1e-3) / 1e9
    cap = ncu_capture("rollout_loop_kernel", E, args.dtype)
    roofline = {"bound": "fp64" if use_f64 else "fp32", "kernel": f"rollout_loop_kernel<{sfx}, MDS_CTRL_LQR_YANK, true, 8, 1>",
                "launches_per_step": P_STREAMS, "envs_per_launch": E // P_STREAMS, "achieved": tf, "peak": fpk,
                "unit": "TFLOP/s", "frac": tf / fpk, "peak_source": fpk_src, "peak_nominal": fpk_nominal, "peak_fma_chain": fpk_chain,
                "frac_counters": cap.get("fp_frac_counters") if cap else None,
                "frac_counters_scalar_only": cap.get("fp_frac_counters_scalar_only") if cap else None,
                "frac_counters_source": (f"profiles/{cap['report']}: executed (fadd + fmul + 2 ffma + 2 fadd2 + 2 fmul2 + 4 ffma2) per cycle / (2 x ffma peak_sustained); scalar opcodes from the hardware counters, "
                                         "packed fp32 opcodes from the SASS page of the same ncu --set full capture (the counters leave them out)"
                                         if cap and cap.get("fp_frac_counters") is not None else None),
                "algorithmic_flop_per_drone_step": flop_step, "control_steps_per_launch": F, "launch_ms": launch_ms, "share_of_step": 1.0,
                "traffic": cap["dram_bytes_per_launch"] if cap else None,
                "hbm": {"achieved": gbs, "peak": hbm_peak, "unit": "GB/s", "frac": gbs / hbm_peak, "algorithmic_bytes_per_drone_per_launch": bytes_launch,
                        "peak_source": peak_src},
                "note": f"arithmetic intensity {flop_step * F / bytes_launch:.0f} flop/B > ridge {fpk * 1e3 / hbm_peak:.1f} flop/B: the state lives in "
                        "registers for the whole launch and HBM sees the per-step observation log plus one state load/store per launch, so the "
                        "FP pipe (not HBM, not tensor cores: nothing is a dense contraction) bounds it"}

    # ---- the per-call kernels against the HBM roofline: replay with one launch per kernel ----------------------
    # (MdsRolloutCfg.stages 1 = controller kernel, 2 = physics kernel; a CUDA event pair around every launch)
    n_rep = min(n_steps, 240)
    evs = [[torch.cuda.Event(enable_timing=True) for _ in range(3)] for _ in range(n_rep)]
    for k in range(n_rep):
        evs[k][0].record()
        ro.run(1, stages=1)
        evs[k][1].record()
        ro.run(1, stages=2)
        evs[k][2].record()
    torch.cuda.synchronize()
    ctrl_ms = sum(e[0].elapsed_time(e[1]) for e in evs) / n_rep
    phys_ms = sum(e[1].elapsed_time(e[2]) for e in evs) / n_rep
    b_ctrl, b_phys = sum(ALGO_BYTES_CTRL_F32.values()) * esz // 4, sum(ALGO_BYTES_PHYS_F32.values()) * esz // 4

    def roof(kernel, bytes_unit, launch):
        g = bytes_unit * D / (launch * 1e-3) / 1e9
        c = ncu_capture(kernel.split("<")[0], E, args.dtype)
        return {"bound": "hbm", "kernel": kernel, "achieved": g, "peak": hbm_peak, "unit": "GB/s", "frac": g / hbm_peak, "peak_source": peak_src,
                "algorithmic_bytes_per_drone_step": bytes_unit, "launch_ms": launch, "traffic": c["dram_bytes_per_launch"] if c else None,
                "note": "per-call path (two launches per control step); replay of the first %d control steps of the timed region" % n_rep}

    roofline_ctrl = roof(f"ctrl_step_kernel<{sfx}, MDS_CTRL_LQR_YANK, true, 8>", b_ctrl, ctrl_ms)
    roofline_physics = roof(f"physics_step_kernel<{sfx}, 8>", b_phys, phys_ms)

    # ---- end to end through the per-call API with host buffers --------------------------------
    e2e = None
    if not args.no_e2e:
        del obs_ring
        e2e = run_e2e(args, mds, sc, dev, dtype, world, barrier, max_over_ranks)

    # ---- strong scaling: the FIXED swarm (args.envs environments in total) sharded over the ranks ----------------
    strong = None
    if not args.no_strong:
        if world == 1:
            strong = {"value": value, "unit": "drone-steps/s", "total_envs": E, "envs_per_gpu": E, "ms_per_step": ms_max / K, "efficiency": 1.0,
                      "streams_per_gpu": P_STREAMS, "note": "N = 1: the fixed swarm is the weak-scaling shard"}
        else:
            b0, b1 = mds.dist.env_shard(E, rank, world)
            Es = b1 - b0
            ms_s, _, _, _ = timed_swarm(Es, b0)
            ms_s = max_over_ranks(ms_s)
            v_s = E * N * F * K / (ms_s * 1e-3)
            strong = {"value": v_s, "unit": "drone-steps/s", "total_envs": E, "envs_per_gpu": Es, "ms_per_step": ms_s / K,
                      "efficiency": v_s / value, "streams_per_gpu": P_STREAMS,
                      "note": f"{E} environments in total, contiguous shards of {Es} per GPU (dist.env_shard), each cut into {P_STREAMS} sub-swarms on their own "
                              f"streams like `value`; efficiency = strong value / weak value (= N x the rate of one GPU on the full {E}-environment shard, "
                              "measured in this run)"}
            torch.cuda.empty_cache()

    # ---- the other BASELINE.json configurations (N = 1 only; every rank of a multi-GPU run would repeat them) ----------
    configs = None
    if world == 1 and not args.no_configs:
        del sc, env, ro, ctrl
        torch.cuda.empty_cache()
        configs = run_configs(args, mds, scenarios, torch, dev, sms, hbm_peak, local_rank)

    if rank == 0:
        line = {"metric": METRIC, "value": value, "unit": "drone-steps/s",
                "n_gpus": world, "steps": K, "warmup": W, "ms_per_step": ms_max / K, "higher_is_better": True, "scaling": "weak",
                "vs_baseline": None, "dtype": args.dtype, "data": "synthetic", "config": workload_config(args, E),
                "clocks": clocks, "e2e": e2e, "gpu_launches": K * P_STREAMS, "roofline": roofline, "roofline_ctrl": roofline_ctrl,
                "roofline_physics": roofline_physics, "strong": strong, "configs": configs,
                "cpu_baseline": (cpu.get("reference") or cpu.get("port")) if cpu else None,
                "cpu_baseline_port": cpu.get("port") if cpu and "reference" in cpu else None,
                "rollout_stats": stats, "sm_count": sms}
        emit(line)
    if world > 1:
        dist.destroy_process_group()


def run_configs(args, mds, scenarios, torch, dev, sms, hbm_peak, local_rank):
    """C2 / C3 order 2 / C4 / C5 fp64 (BASELINE.json configs[1..3] and the fp64 mode north_star asks for), time-boxed:
    each from rest through a short settling run, then a few timed launches; roofline fraction against the bound that
    applies (FP32 / FP64 pipe for the fused rollouts, HBM for the model-comparison kernels)."""
    out = {}
    with ClockSampler(local_rank) as clk:
        def timed(ro, steps_per_launch, reps, log=None):
            fn = (lambda: ro.run(steps_per_launch, obs_log=log, log_every=1)) if log is not None else (lambda: ro.run(steps_per_launch))
            fn()
            ms, w0, w1 = time_launches(torch, fn, reps)
            return ms / (reps * steps_per_launch), (w0, w1)

        pk32, _, _, src32 = fp_peak(mds, sms, None, False)
        pk64, _, _, src64 = fp_peak(mds, sms, None, True)
        # C2: 4096 envs x 1 drone, geometric SE(3) controller on Circle / Lemniscate, DYN_GND_DRAG_DW (simulations/EnvGeometric.py)
        sw = scenarios.tracking_swarm(4096, dtype=torch.float32, device=dev)
        sw["rollout"].run(240)
        ms, win = timed(sw["rollout"], 240, 20)
        fl = sum(ALGO_FLOP_GEOMETRIC.values())
        out["C2_4096"] = {"workload": "4096 envs x 1 drone, geometric SE(3) tracking of Circle / Lemniscate, DYN_GND_DRAG_DW, fp32, 240 control steps per launch",
                          "value": 4096 / (ms * 1e-3), "unit": "drone-steps/s", "us_per_control_step": ms * 1e3,
                          "roofline": {"bound": "latency", "achieved": fl * 4096 / (ms * 1e-3) / 1e12, "peak": pk32, "unit": "TFLOP/s",
                                       "frac": fl * 4096 / (ms * 1e-3) / 1e12 / pk32,
                                       "note": f"4096 threads = 16 blocks on {sms} SMs: one dependent chain per resident warp, bounded by instruction latency, not by a pipe"},
                          "stats": {"max_pos_err": sw["rollout"].stats_dict()["max_pos_err"]}, "clocks": clk.summary(*win)}
        del sw
        # C3 in its order-2 form: 16 384 envs x 8 drones, LQR-omega nominal + order-2 CBF-QP (simulations/CBFTest.py), sphere beside the crossing
        # two sub-swarm streams as in the headline: 16 384 environments are 1.73 waves of the loop kernel's resident blocks
        ro, subs = scenarios.cbf_swarm_streams(16384, 2, N_DRONES, order=2, dtype=torch.float32, device=dev)
        log = [torch.empty(24, s_["env"].NUM_ENVS, N_DRONES, 20, device=dev) for s_ in subs]
        c3_step = lambda: ro.run(24, obs_logs=log, log_every=1)
        for _ in range(20):
            c3_step()
        ro.synchronize()
        ro.reset_stats()
        c3_step()
        ms, w0, w1 = time_launches(torch, c3_step, 20, swarm=ro)
        ms, win = ms / (20 * 24), (w0, w1)
        ro.synchronize()
        st = ro.stats_dict()
        fl = sum(ALGO_FLOP_PER_DRONE_STEP.values())
        n_env_steps = max(1.0, st["drone_steps"] / N_DRONES)
        out["C3_o2_16384"] = {"workload": "16 384 envs x 8 drones, LQR-omega nominal + order-2 CBF-QP (r_safe 0.1, zscale 1, poles -2.2/-2.4) + sphere, DYN_GND_DRAG_DW, fp32, 2 sub-swarm streams",
                              "value": 16384 * N_DRONES / (ms * 1e-3), "unit": "drone-steps/s", "us_per_control_step": ms * 1e3,
                              "roofline": {"bound": "fp32", "achieved": fl * 16384 * N_DRONES / (ms * 1e-3) / 1e12, "peak": pk32, "unit": "TFLOP/s",
                                           "frac": fl * 16384 * N_DRONES / (ms * 1e-3) / 1e12 / pk32, "peak_source": src32},
                              "qp": {"active_frac": st["qp_solves"] / n_env_steps, "iters_per_solve": st["qp_iters"] / max(1.0, st["qp_solves"]),
                                     "infeasible_frac": st["qp_infeasible"] / n_env_steps, "iter_cap_frac": st["qp_iter_cap"] / n_env_steps,
                                     "note": "infeasible = the reference's own fallback to the nominal input (cbf/qptracker.py:30-34): order-2 rows lose their "
                                             "input coefficient as ez -> 0"},
                              "clocks": clk.summary(*win)}
        del ro, subs, log
        # C4: CompareModels on 65 536 samples, fp64: LinearizedModel.calc_xdot + QuadrotorDynamics.dynamics mapped to the linear order
        E4 = 65536
        env4 = mds.BatchedCtrlAviary(drone_model=mds.DroneModel.CF2P, num_drones=1, num_envs=E4, dtype=torch.float64, device=dev)
        g = torch.Generator(device="cpu").manual_seed(4)
        obs4 = torch.zeros(E4, 1, 20, dtype=torch.float64)
        obs4[..., 0:3] = torch.rand(E4, 1, 3, generator=g) * 4 - 2
        rpy = torch.rand(E4, 1, 3, generator=g) - 0.5
        obs4[..., 7:10] = rpy
        h = rpy * 0.5
        cr, sr, cp, sp, cy, sy = h[..., 0].cos(), h[..., 0].sin(), h[..., 1].cos(), h[..., 1].sin(), h[..., 2].cos(), h[..., 2].sin()
        obs4[..., 3], obs4[..., 4] = sr * cp * cy - cr * sp * sy, cr * sp * cy + sr * cp * sy
        obs4[..., 5], obs4[..., 6] = cr * cp * sy - sr * sp * cy, cr * cp * cy + sr * sp * sy
        obs4[..., 10:16] = torch.randn(E4, 1, 6, generator=g)
        obs4[..., 16:20] = 9440.3 + torch.rand(E4, 1, 4, generator=g) * (env4.MAX_RPM - 9440.3)
        obs4 = obs4.to(dev)
        lin, nl = mds.model.LinearizedModel(env4), mds.model.QuadrotorDynamics(env4.PYB_FREQ)
        nl.load_env_params(env4)
        o_lin, o_nl = torch.empty(E4, 1, 12, device=dev, dtype=torch.float64), torch.empty(E4, 1, 12, device=dev, dtype=torch.float64)
        fn4 = lambda: (lin.calc_xdot_from_obs(obs4, out=o_lin), nl.dynamics_from_obs(obs4, out=o_nl))
        fn4()
        ms4, w0, w1 = time_launches(torch, fn4, 200)
        ms4 /= 200
        b4 = 2 * (20 + 12) * 8  # each kernel: read obs (20), write xdot (12), fp64
        out["C4_65536_f64"] = {"workload": "CompareModels: 65 536 samples, fp64, LinearizedModel.calc_xdot + QuadrotorDynamics.dynamics (two launches per pass)",
                               "value": E4 / (ms4 * 1e-3), "unit": "samples/s", "us_per_pass": ms4 * 1e3,
                               "roofline": {"bound": "hbm", "achieved": b4 * E4 / (ms4 * 1e-3) / 1e9, "peak": hbm_peak, "unit": "GB/s",
                                            "frac": b4 * E4 / (ms4 * 1e-3) / 1e9 / hbm_peak, "algorithmic_bytes_per_sample": b4,
                                            "note": "33 MB working set: L2-resident and launch-bound (two ~3 us kernels per pass)"},
                               "clocks": clk.summary(w0, w1)}
        del env4, obs4, lin, nl, o_lin, o_nl
        # C5 in fp64 (north_star: an fp64 mode, FP64 pipe utilisation)
        E5 = args.envs
        sw = scenarios.cbf_swarm(E5, N_DRONES, order=CBF_ORDER, dtype=torch.float64, device=dev)
        ro = sw["rollout"]
        log = torch.empty(24, E5, N_DRONES, 20, device=dev, dtype=torch.float64)
        for _ in range(480 // 24):
            ro.run(24, obs_log=log, log_every=1)
        ro.reset_stats()
        ms, win = timed(ro, 24, 6, log)
        st = ro.stats_dict()
        fl = sum(ALGO_FLOP_PER_DRONE_STEP.values())
        out["C5_f64"] = {"workload": f"the headline workload in fp64: {E5} envs x 8 drones, after 504 control steps from rest (2.1 s of flight)",
                         "value": E5 * N_DRONES / (ms * 1e-3), "unit": "drone-steps/s", "ms_per_control_step": ms,
                         "roofline": {"bound": "fp64", "achieved": fl * E5 * N_DRONES / (ms * 1e-3) / 1e12, "peak": pk64, "unit": "TFLOP/s",
                                      "frac": fl * E5 * N_DRONES / (ms * 1e-3) / 1e12 / pk64, "peak_source": src64},
                         "qp": {"iters_per_solve": st["qp_iters"] / max(1.0, st["qp_solves"]), "infeasible": st["qp_infeasible"], "iter_cap": st["qp_iter_cap"]},
                         "clocks": clk.summary(*win)}
        del sw, ro, log
        torch.cuda.empty_cache()
    return out


def pcie_ceiling(torch, dev, d2h_bytes, h2d_bytes, reps, barrier, max_over_ranks):
    """Plain copies of the e2e path's sizes and nothing else: one cudaMemcpyAsync per copy (Tensor.copy_ between pinned host
    and device memory), device -> host on one stream and host -> device on another, `reps` times, all ranks at once."""
    hb_out, hb_in = torch.empty(d2h_bytes, dtype=torch.uint8).pin_memory(), torch.empty(h2d_bytes, dtype=torch.uint8).pin_memory()
    db_out, db_in = torch.empty(d2h_bytes, dtype=torch.uint8, device=dev), torch.empty(h2d_bytes, dtype=torch.uint8, device=dev)
    s_out, s_in = torch.cuda.Stream(dev), torch.cuda.Stream(dev)
    res = {}
    for name, do_out, do_in in (("d2h_alone", True, False), ("h2d_alone", False, True), ("both", True, True)):
        for timed in (False, True):
            torch.cuda.synchronize()
            if timed:
                barrier()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            cs = torch.cuda.current_stream(dev)
            e0.record()
            s_out.wait_event(e0); s_in.wait_event(e0)
            for _ in range(reps if timed else 2):
                if do_out:
                    with torch.cuda.stream(s_out):
                        hb_out.copy_(db_out, non_blocking=True)
                if do_in:
                    with torch.cuda.stream(s_in):
                        db_in.copy_(hb_in, non_blocking=True)
            cs.wait_stream(s_out); cs.wait_stream(s_in)
            e1.record()
            torch.cuda.synchronize()
            if timed:
                res[name] = max_over_ranks(e0.elapsed_time(e1)) / reps
    return res


def run_e2e(args, mds, sc, dev, dtype, world, barrier, max_over_ranks):
    """Reference-facing per-call sequence with HOST buffers (multidronesim_b200.HostPipeline), every control step:
       H2D refs (what the reference passes to set_desired_trajectory) -> LQR (skip_low_level) -> caller glue
       (nominal -= mg, xdes) -> CBF-QP -> inner loop -> env.step -> D2H observations; the copies of neighbouring
       steps overlap the kernels on their own streams."""
    import torch
    env, ctrl, trk, trajs = sc["env"], sc["ctrl"], sc["tracker"], sc["trajs"]
    E, N = env.NUM_ENVS, env.NUM_DRONES
    D = E * N
    S = args.e2e_steps
    esz = 4 if dtype == torch.float32 else 8
    # continues from the swarm's current (steady-flight) state; the host owns the references (pre-evaluated for the
    # S steps, as a host-side planner would) and receives the observations
    t_start = sc["rollout"].t
    ref_host = torch.empty(S + 4, D, 11, dtype=dtype).pin_memory()
    for k in range(S + 4):
        ref_host[k].copy_(trajs.eval(t_start + k * env.CTRL_TIMESTEP))
    torch.cuda.synchronize()
    obs_host = [torch.empty(E, N, 20, dtype=dtype).pin_memory() for _ in range(2)]
    pipe = mds.HostPipeline(env, ctrl, trk, sc["obstacles"])
    for k in range(4):
        pipe.step(ref_host[k], obs_host[k & 1])
    pipe.synchronize()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    torch.cuda.synchronize()
    cs = torch.cuda.current_stream(dev)
    ev0.record()
    for k in range(S):
        pipe.step(ref_host[4 + k], obs_host[k & 1])
    cs.wait_stream(pipe.s_out)  # the last observation has landed in host memory
    cs.wait_stream(pipe.s_in)
    ev1.record()
    torch.cuda.synchronize()
    barrier()
    ms = max_over_ranks(ev0.elapsed_time(ev1))
    value = world * D * S / (ms * 1e-3)
    del ref_host, pipe

    # the link's own ceiling for these transfer sizes, all ranks copying at once
    h2d, d2h = D * 11 * esz, D * 20 * esz
    pc = pcie_ceiling(torch, dev, d2h, h2d, 24, barrier, max_over_ranks)
    ceil_ms = pc["both"]
    ceiling = {"d2h_gbs_alone": d2h / pc["d2h_alone"] / 1e6, "h2d_gbs_alone": h2d / pc["h2d_alone"] / 1e6,
               "d2h_gbs_concurrent": d2h / pc["both"] / 1e6, "ms_per_control_step": ceil_ms, "value": world * D / (ceil_ms * 1e-3), "unit": "drone-steps/s",
               "note": f"{d2h} B device->host and {h2d} B host->device per control step per GPU, plain Tensor.copy_ (one cudaMemcpyAsync each) on two streams, "
                       f"{world} rank(s) copying at once; per-GPU GB/s"}

    # K-step host call: one launch of F control steps + ONE device->host copy of the F observations, double-buffered
    F = args.fuse
    hr = mds.HostRollout(sc["rollout"], F)
    big = [torch.empty(F, E, N, 20, dtype=dtype).pin_memory() for _ in range(2)]
    n_calls = max(2, S // F)
    for j in range(2):
        hr.step(big[j & 1])
    hr.synchronize()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    torch.cuda.synchronize()
    ev0.record()
    for j in range(n_calls):
        hr.step(big[j & 1])
    cs.wait_stream(hr.s_out)
    ev1.record()
    torch.cuda.synchronize()
    barrier()
    ms_f = max_over_ranks(ev0.elapsed_time(ev1))
    fused = {"value": world * D * F * n_calls / (ms_f * 1e-3), "unit": "drone-steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": d2h,
             "control_steps": F * n_calls, "ms_per_control_step": ms_f / (F * n_calls), "frac_of_pcie_ceiling": pc["d2h_alone"] / (ms_f / (F * n_calls)),
             "path": f"mds_rollout ({F} control steps in one launch, device-resident trajectories, every observation logged) -> ONE D2H of the {F} observations "
                     "to pinned host memory on a copy stream, two log buffers (the copy of call j overlaps the launch of call j + 1)"}
    return {"value": value, "unit": "drone-steps/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
            "control_steps": S, "ms_per_control_step": ms / S, "kernels_per_control_step": 5,
            "pcie_ceiling": ceiling, "frac_of_pcie_ceiling": ceil_ms / (ms / S), "fused": fused,
            "path": "pinned host refs -> H2D (copy stream) -> mds_lqr_ctrl -> mds_cbf_prepare -> mds_cbf_qp -> mds_lowlevel -> mds_physics_step "
                    "-> D2H obs to pinned host (copy stream); two slots, copies overlap the next step's kernels"}


_JSON_FD = None


def emit(line):
    """the ONE JSON line goes to the process's original stdout; everything else (NCCL banners, warnings) to stderr"""
    data = (json.dumps(line) + "\n").encode()
    os.write(_JSON_FD if _JSON_FD is not None else 1, data)


def main():
    global _JSON_FD
    args = parse_args()
    sys.stdout.flush()
    _JSON_FD = os.dup(1)
    os.dup2(2, 1)  # libraries that print to stdout (e.g. "NCCL version ...") must not pollute the JSON line
    if args.impl == "reference":
        run_reference_arm(args)
    else:
        run_gpu_arm(args)


if __name__ == "__main__":
    main()
