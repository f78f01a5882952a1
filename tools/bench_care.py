"""The robot-coupled Riccati solve of the 12-dim DecentralizedLQR: compute_controller(solver="device") (mds_care_gains_coupled)
on distinct perturbed models (the prior scaled entry-wise by 5 % noise, half of the drones with a dense 0.05 perturbation of
A, drawn on the device), timed with CUDA events after a warm-up call, median of the reps.  The host route (scipy on the full
12N-state problem of each environment, compute_controller(solver="host")) is timed on the first min(E, 200) environments and
reported per environment; on those environments the device gain is checked against it in the same run (max |K_dev - K_host|
over max |K_host| of each environment, every entry of the [4N, 12N] gain).  Prints the card name, power limit and max SM
clock first, then one JSON line per case.
usage: python tools/bench_care.py [reps=5]"""
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
from multidronesim_b200.control import dlqr  # noqa: E402

REPS = int(sys.argv[1]) if len(sys.argv) > 1 else 5
CASES = [(125_000, 8), (500_000, 2), (1, 2), (1, 7)]
HOST_ENVS = 200


def card():
    try:
        return subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True,
                              text=True, timeout=30).stdout.strip()
    except Exception as e:  # the measurement itself does not depend on it
        return f"unknown ({e})"


def controller(E, N, dtype):
    env = mds.BatchedCtrlAviary(drone_model=mds.DroneModel.CF2P, num_drones=N, num_envs=E, dtype=dtype)
    return dlqr.DecentralizedLQR(env, [mds.model.LinearizedModel(env) for _ in range(N)])


def perturb(dl, seed):
    g = torch.Generator(device="cuda").manual_seed(seed)
    th = dl.theta_planes                                       # [(16 * 12), D]; planes k < 144 hold A
    th.mul_(1.0 + 0.05 * torch.randn(th.shape, device="cuda", dtype=th.dtype, generator=g))
    half = th.shape[1] // 2
    th[:144, half:] += 0.05 * torch.randn(144, th.shape[1] - half, device="cuda", dtype=th.dtype, generator=g)


def full_gain(dl):
    E, N, m = dl.env.NUM_ENVS, dl.num_robots, dl.m
    planes = dl.K_planes.double().cpu().numpy().reshape(N, 4, m, E, N)
    return planes.transpose(3, 4, 1, 0, 2).reshape(E, 4 * N, m * N)


def main():
    if not torch.cuda.is_available():
        raise SystemExit("bench_care.py needs a CUDA device (there is no CPU path)")
    print("card:", card(), flush=True)
    for dtype in (torch.float32, torch.float64):
        for E, N in CASES:
            dl = controller(E, N, dtype)
            perturb(dl, seed=E + N)
            dl.compute_controller(solver="device")             # warm-up (module load, shared-memory opt-in)
            torch.cuda.synchronize()
            times = []
            for _ in range(REPS):
                a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                a.record()
                dl.compute_controller(solver="device")
                b.record()
                b.synchronize()
                times.append(a.elapsed_time(b))
            failed = int(dl.care_status.sum())
            # the host route on the first environments, and the device gain on the same models
            Es = min(E, HOST_ENVS)
            sub = controller(Es, N, dtype)
            sub.theta_planes.copy_(dl.theta_planes[:, :Es * N])
            t0 = time.perf_counter()
            K_host = np.array(sub.compute_controller(solver="host"))
            torch.cuda.synchronize()
            host_s = time.perf_counter() - t0
            sub.compute_controller(solver="device")
            K_dev = full_gain(sub)
            rel = max(float(np.abs(K_dev[e] - K_host[e]).max() / np.abs(K_host[e]).max()) for e in range(Es))
            print(json.dumps({"dtype": str(dtype).replace("torch.", ""), "E": E, "N": N, "drones": E * N, "device_ms_median": round(float(np.median(times)), 3),
                              "device_ms_min": round(float(np.min(times)), 3), "reps": REPS, "status_failures": failed,
                              "host_envs": Es, "host_ms_per_env": round(1e3 * host_s / Es, 3), "max_rel_err_vs_host": float(f"{rel:.3e}")}), flush=True)
            del dl, sub
            torch.cuda.empty_cache()


if __name__ == "__main__":
    main()
