"""The reference table of the fused rollout: when every environment flies the same N trajectories (TrajectorySet.env_period),
rollout_loop_kernel evaluates each reference once per block and step instead of once per drone.  CPU: the periodicity
detection.  GPU: the table path gives the same bits as the per-drone path (FusedRollout(ref_table=False)), across table
refills and in the block that holds the last environments, and a swarm whose environments differ stays on the per-drone path."""
import numpy as np
import pytest
import torch

N = 8


def lem_params(n=N, omega=0.5):
    """Lemniscate rows of the C3 / C5 swarm (scenarios.cbf_swarm)"""
    p = np.zeros((n, 7))
    p[:, 0], p[:, 1], p[:, 2:5], p[:, 6] = 1.0, omega, [0.0, 0.0, 0.5], (2 * np.pi / (n + 0.25)) * np.arange(n)
    return p


def compound_trajs(T):
    """eight trajectories that go through the segment table: compounds (wait, line, rotated circle), a stand-alone rotated
    lemniscate, and two closed-form generators with yaw motion; short segments so that a 77-step run crosses their ends"""
    from multidronesim_b200.scenarios import lemniscate_pos
    base = lemniscate_pos(1.0, lem_params()[:, 6], np.array([0.0, 0.0, 0.5]))
    base[:, 2] += 0.04 * np.arange(N)
    c, s = np.cos(0.3), np.sin(0.3)
    R = np.array([[c, -s, 0.0], [s, c, 0.0], [0.0, 0.0, 1.0]])
    out = []
    for n in range(N):
        p = base[n]
        if n < 5:
            out.append(T.CompoundTrajectory([T.WaitTrajectory(p, 0.04 + 0.01 * n),
                                             T.LineTrajectory(p, p + np.array([0.05, -0.03, 0.02]), speed=0.5),
                                             T.RotateTrajectory(T.CircleTrajectory(r=0.05, v=0.2, center=p - np.array([0.05, 0.0, 0.0])), R, p)]))
        elif n == 5:
            out.append(T.RotateTrajectory(T.Lemniscate(a=0.1, omega=1.0, center=p, phase_shift=0.4), R, p))
        elif n == 6:
            out.append(T.Lemniscate(a=0.1, omega=1.0, center=p, yaw_rate=0.5, phase_shift=1.0))
        else:
            out.append(T.CircleTrajectory(r=0.05, v=0.2, center=p - np.array([0.05, 0.0, 0.0]), yaw_rate=0.3))
    return out


def test_env_period_detection(lib_built):
    from multidronesim_b200 import _lib
    from multidronesim_b200 import trajectories as T
    E = 5
    tiled = np.tile(lem_params(), (E, 1))
    arrays = lambda kind, p, **kw: T.TrajectorySet.from_arrays(kind, p, device="cpu", **kw)
    assert arrays(_lib.TRAJ_LEMNISCATE, tiled, drones_per_env=N).env_period == N
    assert arrays(_lib.TRAJ_LEMNISCATE, tiled).env_period == 0  # drone count not given: no claim
    assert arrays(_lib.TRAJ_LEMNISCATE, tiled, drones_per_env=4).env_period == 0  # environments of 4 drones differ
    assert arrays(_lib.TRAJ_LEMNISCATE, tiled, drones_per_env=3).env_period == 0  # 40 drones are not environments of 3
    bad = tiled.copy()
    bad[3 * N + 5, 6] += 1e-3  # one drone of environment 3
    assert arrays(_lib.TRAJ_LEMNISCATE, bad, drones_per_env=N).env_period == 0
    kinds = np.full(E * N, _lib.TRAJ_LEMNISCATE)
    kinds[2 * N + 1] = _lib.TRAJ_CIRCLE
    assert arrays(kinds, tiled, drones_per_env=N).env_period == 0
    assert arrays(np.full(E * N, _lib.TRAJ_LEMNISCATE), tiled, drones_per_env=N).env_period == N

    ts = T.TrajectorySet(compound_trajs(T), num_envs=E, device="cpu")
    assert ts.env_period == N and ts.num == E * N
    ts.specs = ts.specs.clone()  # replaced descriptors are not known to repeat
    assert ts.env_period == 0
    assert T.TrajectorySet(compound_trajs(T), device="cpu").env_period == N  # one environment of eight drones


def run_swarm(E, K, table, trajs=None, calls=2):
    """C5 swarm of E environments; ``calls`` launches of K steps each (the second starts mid-flight), every observation
    logged -> everything the rollouts wrote"""
    from multidronesim_b200 import FusedRollout, scenarios
    sc = scenarios.cbf_swarm(E, N, order=3)
    ro = sc["rollout"]
    if trajs is not None:
        ro = FusedRollout(sc["env"], trajs, sc["ctrl"], sc["tracker"], sc["obstacles"])
    ro.ref_table = table
    env = sc["env"]
    logs = []
    for _ in range(calls):
        log = torch.zeros(K, E, N, 20, device="cuda")
        ro.run(K, obs_log=log, log_every=1)
        logs.append(log)
    assert ro.cfg.traj_period == (N if table else 0)
    torch.cuda.synchronize()
    pid = sc["ctrl"].low_level
    out = dict(log=torch.stack(logs), pos_wx=env._pos_wx, quat=env._quat, vel_wy=env._vel_wy, rpm=env._rpm, wz=env._wz, obs=env._obs,
               action=env._action, pid_a=pid._a, pid_b=pid._b, stats=ro.stats)
    return {k: v.cpu().clone() for k, v in out.items()}


def assert_same_bits(a, b):
    for k in a:
        assert torch.equal(a[k], b[k]), f"{k}: max |diff| {float((a[k].double() - b[k].double()).abs().max())}"


@pytest.mark.gpu
@pytest.mark.parametrize("K", [24, 77])
def test_cbf_swarm_table_equals_per_drone(K, lib_built):
    """1003 environments (the last block holds 11 of its 32: a part-filled warp and five warps with no environment of their
    own); K = 77 refills the 32-step table twice and ends on a part-filled one"""
    E = 1003
    table, per_drone = run_swarm(E, K, True), run_swarm(E, K, False)
    assert table["stats"][0] == 2 * K * E * N
    assert_same_bits(table, per_drone)


@pytest.mark.gpu
def test_segment_table_swarm_table_equals_per_drone(lib_built):
    from multidronesim_b200 import trajectories as T
    E, K = 67, 77
    runs = []
    for table in (True, False):
        ts = T.TrajectorySet(compound_trajs(T), num_envs=E)
        assert ts.env_period == N
        runs.append(run_swarm(E, K, table, trajs=ts))
    assert_same_bits(*runs)


@pytest.mark.gpu
def test_swarm_with_one_different_environment_matches_oracle(lib_built):
    """one drone of one environment flies a shifted lemniscate: the set is not periodic, the rollout keeps the per-drone
    references, and that environment follows the oracle's closed loop on its own references"""
    from multidronesim_b200 import FusedRollout, _lib, scenarios
    from multidronesim_b200 import trajectories as T
    from oracle import pipeline as opl
    from oracle import trajectories as otj
    from oracle.aviary import OracleCtrlAviary
    from oracle.constants import DroneModel as ODM, Physics as OPH
    E, K, e_bad = 64, 24, 37
    params = np.tile(lem_params(), (E, 1))
    params[e_bad * N + 3, 6] += 0.3
    ts = T.TrajectorySet.from_arrays(_lib.TRAJ_LEMNISCATE, params, drones_per_env=N)
    assert ts.env_period == 0
    sc = scenarios.cbf_swarm(E, N, order=3)
    ro = FusedRollout(sc["env"], ts, sc["ctrl"], sc["tracker"], sc["obstacles"])
    obs = ro.run(K).double().cpu().numpy()
    assert ro.cfg.traj_period == 0
    init = sc["init"].astype(np.float32).astype(np.float64)
    worst = 0.0
    for e in (0, e_bad):
        o = OracleCtrlAviary(ODM.CF2P, N, initial_xyzs=init[e], physics=OPH.DYN_GND_DRAG_DW)
        p = params[e * N:(e + 1) * N]
        trajs = [otj.Lemniscate(a=r[0], omega=r[1], center=r[2:5], yaw_rate=r[5], phase_shift=r[6]) for r in p]
        _, want, _ = opl.run_cbf(o, trajs, 3, K, obstacles=sc["obstacles"], log=False)
        worst = max(worst, float(np.max(np.abs(obs[e, :, 0:3] - want[:, 0:3]))))
    assert worst < 1e-3, worst
