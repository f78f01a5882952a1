"""Synthetic swarm set-ups of SURVEY.md 8(d): the configurations bench.py / smoke() time and the
parity tests replay in miniature.  Everything here is init-time host work (numpy) that ends in
device tensors; the per-step path never touches it."""
from __future__ import annotations

import math

import numpy as np
import torch

from . import _lib
from .cbf import DroneCBF, DroneQPTracker
from .control import (GeometricControl, LQROmegaController, LQRYankOmegaController, ThrustOmegaController,
                      YankOmegaController)
from .enums import DroneModel, Physics
from .envs import BatchedCtrlAviary
from .model import LinearizedOmegaModel, LinearizedYankOmegaModel
from .rollout import FusedRollout
from .trajectories import TrajectorySet


# Sphere obstacle of the C3 / C5 swarm workload: r = 0.1 m, 0.2 m beside the lemniscate's crossing point, so every
# drone skims its barrier (Ds = r_safe + r = 0.225 m) twice per lap.  The reference's own order-2 main puts the
# sphere ON the crossing point (simulations/CBFTest.py:421-424); with 8 drones and the order-3 filter that makes
# the reference's algorithms (oracle, fp64) infeasible in ~15 % of the steps and sends drones > 10 m off their
# references within 10 s (DESIGN.md "Workload"), so the bench uses the offset sphere: same rows, bounded closed loop.
SWARM_OBSTACLES = [[0.2, 0.0, 0.5, 0.1]]


def lemniscate_pos(a, theta, center):
    """Lemniscate.py:51-53 at phase theta (vectorised)."""
    s, c = np.sin(theta), np.cos(theta)
    den = 1 + s * s
    return np.stack([center[0] + a * s * c / den, center[1] + a * c / den, np.full_like(theta, center[2])], axis=-1)


def counter_normal(seed, env_ids, per_env):
    """Standard normals [len(env_ids), per_env] that depend only on (seed, absolute env index, slot): a splitmix64
    counter hash -> two uniforms -> Box-Muller.  Env e draws the same numbers however the envs are sharded over
    GPUs, so an N-GPU run reproduces the 1-GPU run env for env (SURVEY.md 8e)."""
    def mix(z):
        z = (z + np.uint64(0x9E3779B97F4A7C15))
        z = (z ^ (z >> np.uint64(30))) * np.uint64(0xBF58476D1CE4E5B9)
        z = (z ^ (z >> np.uint64(27))) * np.uint64(0x94D049BB133111EB)
        return z ^ (z >> np.uint64(31))
    with np.errstate(over="ignore"):
        e = np.asarray(env_ids, dtype=np.uint64)[:, None]
        k = np.arange(per_env, dtype=np.uint64)[None, :]
        base = mix(mix(np.uint64(seed) + np.uint64(0x1234567)) ^ (e * np.uint64(0xD1342543DE82EF95))) ^ (k * np.uint64(0x2545F4914F6CDD1D))
        a, b = mix(base), mix(base ^ np.uint64(0xA5A5A5A5A5A5A5A5))
    u1 = ((a >> np.uint64(11)).astype(np.float64) + 1.0) / 9007199254740993.0   # (0, 1)
    u2 = (b >> np.uint64(11)).astype(np.float64) / 9007199254740992.0           # [0, 1)
    return np.sqrt(-2.0 * np.log(u1)) * np.cos(2.0 * np.pi * u2)


def cbf_swarm_init(num_envs, num_drones=8, seed=3, env_offset=0, a=1.0, center=(0.0, 0.0, 0.5), jitter=0.02, z_step=0.04):
    """Initial positions [E, N, 3] of the C3 / C5 swarm for the env range [env_offset, env_offset + E): drone k at
    phase 2 pi k / (N + 0.25) of the lemniscate, N(0, jitter^2) per coordinate, plus k * z_step in z."""
    E, N = int(num_envs), int(num_drones)
    phase = (2 * np.pi / (N + 0.25)) * np.arange(N)
    base = lemniscate_pos(a, phase, np.asarray(center, dtype=float))
    noise = counter_normal(seed, env_offset + np.arange(E), 3 * N).reshape(E, N, 3)
    init = base[None] + jitter * noise
    init[..., 2] += z_step * np.arange(N)[None, :]
    return init


def cbf_swarm(num_envs, num_drones=8, order=3, dtype=torch.float32, device="cuda", seed=3, env_offset=0,
              omega=0.5, obstacle=True, physics=Physics.DYN_GND_DRAG_DW, pyb_freq=240, ctrl_freq=240):
    """C3 / C5: N drones per env on one lemniscate (a=1, centre (0,0,0.5)) with phase shifts
    2 pi k / (N + 0.25) (reference simulations/CBFTestOrd3.py:450), one sphere obstacle r=0.1 beside the
    lemniscate's crossing point (SWARM_OBSTACLES), per-env position jitter N(0, 0.02^2) with a
    distinct z offset per drone (order-2 rows vanish at ez = 0).  LQR nominal -> CBF-QP -> inner loop.
    ``env_offset`` makes per-env random streams independent of how envs are sharded over GPUs."""
    E, N = int(num_envs), int(num_drones)
    center = np.array([0.0, 0.0, 0.5])
    phase = (2 * np.pi / (N + 0.25)) * np.arange(N)
    init = cbf_swarm_init(E, N, seed=seed, env_offset=env_offset)
    env = BatchedCtrlAviary(drone_model=DroneModel.CF2P, num_drones=N, initial_xyzs=init, physics=physics,
                            pyb_freq=pyb_freq, ctrl_freq=ctrl_freq, num_envs=E, device=device, dtype=dtype)
    if order == 3:
        mdl = LinearizedYankOmegaModel(env)
        ctrl = LQRYankOmegaController(env, mdl, YankOmegaController(env))
        cbf = DroneCBF(env, [mdl] * N, safety_radius=0.125, zscale=2, order=3, cbf_poles=np.array([-3.0, -3.6, -5.6]))
        trk = DroneQPTracker(cbf, order=3, num_robots=N, xdim=10, env=env)
    else:
        mdl = LinearizedOmegaModel(env)
        ctrl = LQROmegaController(env, mdl, ThrustOmegaController(env))
        cbf = DroneCBF(env, [mdl] * N, safety_radius=0.1, zscale=1, order=2, cbf_poles=np.array([-2.2, -2.4]))
        trk = DroneQPTracker(cbf, order=2, num_robots=N, xdim=9, env=env)
    params = np.zeros((N, 7))
    params[:, 0], params[:, 1], params[:, 2:5], params[:, 5], params[:, 6] = 1.0, omega, center, 0.0, phase
    trajs = TrajectorySet.from_arrays(_lib.TRAJ_LEMNISCATE, np.tile(params, (E, 1)), device=device, dtype=dtype, drones_per_env=N)
    obstacles = [list(o) for o in SWARM_OBSTACLES] if obstacle else None
    rollout = FusedRollout(env, trajs, ctrl, trk, obstacles)
    return dict(env=env, ctrl=ctrl, cbf=cbf, tracker=trk, trajs=trajs, obstacles=obstacles, rollout=rollout, init=init)


def cbf_swarm_streams(num_envs, parts, num_drones=8, order=3, dtype=torch.float32, device="cuda", seed=3, env_offset=0, **kw):
    """The same swarm as ``cbf_swarm(num_envs, ...)`` cut into ``parts`` contiguous sub-swarms (dist.env_shard), each with its own
    env / controller / rollout, wrapped in ``SwarmStreams``.  Env e has the same initial condition whichever way the swarm is cut
    (counter-hash of the absolute env index).  -> (SwarmStreams, [sub-swarm dicts])"""
    from .dist import env_shard
    from .rollout import SwarmStreams
    subs = []
    for p in range(int(parts)):
        b0, b1 = env_shard(int(num_envs), p, int(parts))
        subs.append(cbf_swarm(b1 - b0, num_drones, order=order, dtype=dtype, device=device, seed=seed, env_offset=env_offset + b0, **kw))
    return SwarmStreams([s["rollout"] for s in subs]), subs


def tracking_swarm(num_envs, dtype=torch.float32, device="cuda", seed=1, env_offset=0, physics=Physics.DYN_GND_DRAG_DW):
    """C2: one drone per env, geometric SE(3) controller; even envs track CircleTrajectory(r=1, v=0.5,
    centre (0,0,1)), odd envs Lemniscate(a=1, omega=1.5, centre (0,0,0.5)) with a random phase shift;
    initial position = traj(0) + N(0, 0.05^2), z >= 0.1."""
    E = int(num_envs)
    ids = env_offset + np.arange(E)
    kind = np.where(ids % 2 == 0, _lib.TRAJ_CIRCLE, _lib.TRAJ_LEMNISCATE)
    # a uniform phase from the same per-env counter stream (Phi of a standard normal)
    phase = 2 * np.pi * 0.5 * (1.0 + np.vectorize(math.erf)(counter_normal(seed + 1000, ids, 1)[:, 0] / math.sqrt(2.0)))
    params = np.zeros((E, 7))
    circ = kind == _lib.TRAJ_CIRCLE
    params[circ, 0:6] = [1.0, 0.5, 0.0, 0.0, 1.0, 0.0]
    params[~circ, 0:5] = [1.0, 1.5, 0.0, 0.0, 0.5]
    params[~circ, 6] = phase[~circ]
    p0 = np.where(circ[:, None], np.array([1.0, 0.0, 1.0])[None], lemniscate_pos(1.0, phase, np.array([0.0, 0.0, 0.5])))
    init = p0 + 0.05 * counter_normal(seed, ids, 3)
    init[:, 2] = np.maximum(init[:, 2], 0.1)
    env = BatchedCtrlAviary(drone_model=DroneModel.CF2P, num_drones=1, initial_xyzs=init.reshape(E, 1, 3), physics=physics,
                            num_envs=E, device=device, dtype=dtype)
    ctrl = GeometricControl(env)
    trajs = TrajectorySet.from_arrays(kind, params, device=device, dtype=dtype)
    return dict(env=env, ctrl=ctrl, trajs=trajs, rollout=FusedRollout(env, trajs, ctrl), init=init, kind=kind, params=params)
