"""Per-call learning loop vs the fused LearningRollout (mds_learning_rollout), decentralised LQR with hover references.
For every (precision, m, K, E x N): warm-up, then the two paths timed with CUDA events, alternating, from the same saved
state; in the same run one pair of runs from identical states is compared (fp64: 1e-9 of each quantity's scale; fp32: 2e-4,
the per-call RLS tests' fp32 tolerance).  Prints the card name and power limit first, then one JSON line per case.
--feedback: the same for closed-loop exploration (run(feedback=True) against the per-call loop with dl.compute and an add;
gains from compute_controller() on the prior models, perturbations: the open-loop draws centred and scaled by 1/4, i.e.
+-0.1 m g and +-0.05 rad/s); at 1 M drones the fused
open-loop call on the open-loop excitation is timed alongside (fused_open_ms), which shows what flying the gain costs.
--torque: the 12-dim torque-level DecentralizedLQR (TorqueLearningRollout, theta_update) against its per-call loop with
utils.input_to_action, open loop (thrust in [0.7, 1.5] m g, torques +-1e-5 N m), under per-drone gains
(compute_controller(force_diagonal=True)) and under the robot-coupled gain (compute_controller(): one host solve, every
environment has the same prior models), the perturbations +-0.1 m g and +-5e-6 N m.
usage: python tools/bench_learning.py [reps=3] [--feedback | --torque]"""
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import multidronesim_b200 as mds  # noqa: E402
from multidronesim_b200 import _lib  # noqa: E402
from multidronesim_b200.control import dlqr  # noqa: E402

ARGS = [a for a in sys.argv[1:] if a not in ("--feedback", "--torque")]
FEEDBACK = "--feedback" in sys.argv[1:]
TORQUE = "--torque" in sys.argv[1:]
REPS = int(ARGS[0]) if ARGS else 3


def card():
    try:
        return subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True,
                              text=True, timeout=30).stdout.strip()
    except Exception as e:  # the measurement itself does not depend on it
        return f"unknown ({e})"


def setup(E, N, dtype, m):
    rng = np.random.default_rng(0)
    init = np.stack(np.meshgrid(np.arange(E, dtype=float), np.arange(N, dtype=float), indexing="ij"), -1)
    init = np.concatenate([init * 3.0, np.ones((E, N, 1)) + rng.uniform(0, 0.5, (E, N, 1))], -1)
    env = mds.BatchedCtrlAviary(drone_model=mds.DroneModel.CF2P, num_drones=N, num_envs=E, dtype=dtype, initial_xyzs=init)
    if m == 9:
        dl = dlqr.DecentralizedLQROmega(env, [mds.model.LinearizedOmegaModel(env) for _ in range(N)])
    elif m == 12:
        dl = dlqr.DecentralizedLQR(env, [mds.model.LinearizedModel(env) for _ in range(N)])
    else:
        dl = dlqr.DecentralizedLQRYankOmega(env, [mds.model.LinearizedYankOmegaModel(env) for _ in range(N)])
    params = np.concatenate([init.reshape(-1, 3), np.zeros((E * N, 1))], 1)  # Wait: position, yaw
    ts = mds.trajectories.TrajectorySet.from_arrays(_lib.TRAJ_WAIT, params, dtype=dtype, drones_per_env=N)
    return env, dl, ts


def snapshot(env, dl):
    return env.state_dict(), dl.theta_planes.clone(), dl.P_planes.clone(), dl.low_level._a.clone(), dl.low_level._b.clone()


def restore(env, dl, s):
    env.load_state_dict(s[0])
    for dst, src in zip((dl.theta_planes, dl.P_planes, dl.low_level._a, dl.low_level._b), s[1:]):
        dst.copy_(src)


def percall(env, dl, ts, us):
    obs = env.obs
    for k in range(us.shape[0]):
        dl.set_reference(ts.eval(k * env.CTRL_TIMESTEP))
        e_t = dl.error_state(obs).clone()
        if FEEDBACK:
            u = dl.compute(obs, skip_low_level=True)[1] + us[k]
        else:
            u = us[k]
        phis = torch.cat([e_t, u], dim=-1)
        obs = env.step(dl.compute_low_level(u, obs))[0]
        dl.theta_update(phis, dl.error_state(obs))


def outputs(env, dl):
    f = lambda t: t.double().cpu().numpy()
    return [f(dl.theta_planes), f(dl.P_planes), f(env.obs)[..., :16], f(dl.low_level._a), f(dl.low_level._b), f(dl.resid)]


def main():
    print(json.dumps({"card": card(), "torch": torch.__version__, "feedback": FEEDBACK}), flush=True)
    for dtype in (torch.float32, torch.float64):
        for m in (9, 10):
            for E, N in ((125000, 8), (1, 2), (1, 7)):
                env, dl, ts = setup(E, N, dtype, m)
                if FEEDBACK:
                    dl.compute_controller()
                ro = mds.LearningRollout(env, ts, dl)
                s0 = snapshot(env, dl)
                for K in (24, 40):
                    mg = env.M * env.G
                    g = torch.Generator(device="cuda").manual_seed(K)
                    thrust = torch.empty(K, E, N, 1, device="cuda", dtype=dtype).uniform_(0.7 * mg, 1.5 * mg, generator=g)
                    us_open = torch.cat([thrust, torch.empty(K, E, N, 3, device="cuda", dtype=dtype).uniform_(-0.2, 0.2, generator=g)], -1).contiguous()
                    us = (us_open - torch.tensor([1.1 * mg, 0, 0, 0], device="cuda", dtype=dtype)) / 4 if FEEDBACK else us_open  # +-0.1 m g
                    # agreement from identical states
                    restore(env, dl, s0); percall(env, dl, ts, us); torch.cuda.synchronize(); want = outputs(env, dl)
                    restore(env, dl, s0); ro.run(us, t0=0.0, feedback=FEEDBACK); torch.cuda.synchronize(); got = outputs(env, dl)
                    tol = 1e-9 if dtype == torch.float64 else 2e-4
                    errs = [float(np.abs(a - b).max()) / max(1.0, float(np.abs(b).max())) for a, b in zip(got, want)]
                    # timing: warm-up, then alternate the two paths, each from the saved state (the restore is outside the events)
                    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    D = E * N
                    times = {"percall": [], "fused": []}
                    if FEEDBACK and D >= 1_000_000:
                        times["fused_open"] = []
                    for rep in range(REPS + 1):
                        for name in times:
                            restore(env, dl, s0)
                            torch.cuda.synchronize()
                            a.record()
                            if name == "percall":
                                percall(env, dl, ts, us)
                            elif name == "fused":
                                ro.run(us, t0=0.0, feedback=FEEDBACK)
                            else:
                                ro.run(us_open, t0=0.0)
                            b.record()
                            torch.cuda.synchronize()
                            if rep > 0:
                                times[name].append(a.elapsed_time(b))
                    tc, tf = float(np.median(times["percall"])), float(np.median(times["fused"]))
                    line = {"dtype": str(dtype).split(".")[1], "m": m, "K": K, "E": E, "N": N, "feedback": FEEDBACK, "percall_ms": round(tc, 4),
                            "fused_ms": round(tf, 4), "speedup": round(tc / tf, 2), "fused_drone_steps_per_s": D * K / (tf * 1e-3),
                            "percall_drone_steps_per_s": D * K / (tc * 1e-3), "max_rel_err": max(errs), "tol": tol,
                            "agree": bool(max(errs) <= tol), "t": time.strftime("%H:%M:%S")}
                    if "fused_open" in times:
                        line["fused_open_ms"] = round(float(np.median(times["fused_open"])), 4)
                    print(json.dumps(line), flush=True)
                del env, dl, ts, ro, s0
                torch.cuda.empty_cache()


def percall_torque(env, dl, ts, us, feedback):
    from multidronesim_b200 import utils as U
    obs = env.obs
    for k in range(us.shape[0]):
        dl.set_reference(ts.eval(k * env.CTRL_TIMESTEP))
        e_t = dl.error_state(obs).clone()
        u = dl.compute(obs, skip_low_level=True)[1] + us[k] if feedback else us[k].clone()
        obs = env.step(U.input_to_action(env, u))[0]
        dl.theta_update(torch.cat([e_t, u], -1), dl.error_state(obs))


def main_torque():
    print(json.dumps({"card": card(), "torch": torch.__version__, "torque": True}), flush=True)
    for dtype in (torch.float32, torch.float64):
        for E, N in ((125000, 8), (1, 2), (1, 7)):
            for gain in ("open", "drone", "coupled"):
                env, dl, ts = setup(E, N, dtype, 12)
                feedback = gain != "open"
                if feedback:
                    dl.compute_controller(force_diagonal=gain == "drone")
                ro = mds.TorqueLearningRollout(env, ts, dl)
                s0 = (env.state_dict(), dl.theta_planes.clone(), dl.P_planes.clone())

                def restore():
                    env.load_state_dict(s0[0])
                    dl.theta_planes.copy_(s0[1])
                    dl.P_planes.copy_(s0[2])

                def outs():
                    f = lambda t: t.double().cpu().numpy()
                    return [f(dl.theta_planes), f(dl.P_planes), f(env.obs)[..., :16], f(dl.resid)]

                for K in (24, 40):
                    mg = env.M * env.G
                    g = torch.Generator(device="cuda").manual_seed(K)
                    if feedback:
                        us = torch.cat([torch.empty(K, E, N, 1, device="cuda", dtype=dtype).uniform_(-0.1 * mg, 0.1 * mg, generator=g),
                                        torch.empty(K, E, N, 3, device="cuda", dtype=dtype).uniform_(-5e-6, 5e-6, generator=g)], -1).contiguous()
                    else:
                        us = torch.cat([torch.empty(K, E, N, 1, device="cuda", dtype=dtype).uniform_(0.7 * mg, 1.5 * mg, generator=g),
                                        torch.empty(K, E, N, 3, device="cuda", dtype=dtype).uniform_(-1e-5, 1e-5, generator=g)], -1).contiguous()
                    restore(); percall_torque(env, dl, ts, us, feedback); torch.cuda.synchronize(); want = outs()
                    restore(); ro.run(us, t0=0.0, feedback=feedback); torch.cuda.synchronize(); got = outs()
                    tol = 1e-9 if dtype == torch.float64 else 2e-4
                    errs = [float(np.abs(a - b).max()) / max(1.0, float(np.abs(b).max())) for a, b in zip(got, want)]
                    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    times = {"percall": [], "fused": []}
                    for rep in range(REPS + 1):
                        for name in times:
                            restore()
                            torch.cuda.synchronize()
                            a.record()
                            if name == "percall":
                                percall_torque(env, dl, ts, us, feedback)
                            else:
                                ro.run(us, t0=0.0, feedback=feedback)
                            b.record()
                            torch.cuda.synchronize()
                            if rep > 0:
                                times[name].append(a.elapsed_time(b))
                    D = E * N
                    tc, tf = float(np.median(times["percall"])), float(np.median(times["fused"]))
                    print(json.dumps({"dtype": str(dtype).split(".")[1], "m": 12, "gain": gain, "coupled": bool(dl._coupled) if feedback else False,
                                      "K": K, "E": E, "N": N, "percall_ms": round(tc, 4), "fused_ms": round(tf, 4), "speedup": round(tc / tf, 2),
                                      "fused_drone_steps_per_s": D * K / (tf * 1e-3), "percall_drone_steps_per_s": D * K / (tc * 1e-3),
                                      "max_rel_err": max(errs), "tol": tol, "agree": bool(max(errs) <= tol), "t": time.strftime("%H:%M:%S")}),
                          flush=True)
                del env, dl, ts, ro, s0
                torch.cuda.empty_cache()


if __name__ == "__main__":
    main_torque() if TORQUE else main()
