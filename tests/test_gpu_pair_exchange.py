"""GPU: the fused rollout (plan 6) takes the downwash of a control step's first physics sub-step from the CBF stage's pair
exchange.  Plan 4 (ctrl_step_kernel, then physics_step_kernel) sums it in the physics kernel from positions of its own, so
it is an independent check: the two plans agree, and both agree with the oracle, at the edges of that fusion -- a stack of
drones where the downwash is a large share of the thrust, every shape of the pair ownership, environments past the last
full block, two physics sub-steps, physics without downwash, wind, and calls split at the reference table's refill."""
import numpy as np
import pytest
import torch

from helpers import scaled_err
from oracle import pipeline as opl
from oracle import trajectories as otj
from oracle.aviary import OracleCtrlAviary
from oracle.constants import DroneModel as ODM, Physics as OPH

pytestmark = pytest.mark.gpu


def stack_init(E, N, rng):
    """Per env: a vertical stack in hover, neighbours 0.05-0.3 m apart in z with small xy offsets; drone 2 at drone 1's
    height (dz = 0), the last drone beyond 10 m in the plane (N >= 4)."""
    init = np.zeros((E, N, 3))
    for e in range(E):
        init[e, :, 0:2] = rng.normal(0, 0.03, (N, 2))
        init[e, :, 2] = 0.5 + np.concatenate([[0.0], np.cumsum(rng.uniform(0.05, 0.3, N - 1))])
        if N >= 3:
            init[e, 2, 2] = init[e, 1, 2]
            init[e, 2, 0:2] = init[e, 1, 0:2] + np.array([0.3, 0.0])
        if N >= 4:
            init[e, N - 1, 0:2] = np.array([12.0, 0.0])
    return np.float32(init).astype(np.float64)  # representable in both precisions: the oracle starts where the device does


def build(E, N, dtype, order, init, physics="dyn_gnd_drag_dw", shared_refs=False, pyb_freq=240):
    """LQR nominal -> order-2 (LQR_OMEGA) or order-3 (LQR_YANK) CBF-QP -> inner loop; every drone hovers where it starts
    (shared_refs: at environment 0's positions, so that every environment flies the same N references)."""
    import multidronesim_b200 as mds
    import multidronesim_b200.trajectories as T
    env = mds.BatchedCtrlAviary(drone_model=mds.DroneModel.CF2P, num_drones=N, physics=mds.Physics(physics), num_envs=E, dtype=dtype,
                                initial_xyzs=init, pyb_freq=pyb_freq)
    M = mds.model
    if order == 2:
        c = mds.control.LQROmegaController(env, M.LinearizedOmegaModel(env), mds.control.ThrustOmegaController(env))
        cbf = mds.cbf.DroneCBF(env, [M.LinearizedOmegaModel(env) for _ in range(N)], safety_radius=0.1, zscale=1.0, order=2,
                               cbf_poles=np.array([-2.2, -2.4]))
    else:
        c = mds.control.LQRYankOmegaController(env, M.LinearizedYankOmegaModel(env), mds.control.YankOmegaController(env))
        cbf = mds.cbf.DroneCBF(env, [M.LinearizedYankOmegaModel(env) for _ in range(N)], safety_radius=0.125, zscale=2.0, order=3,
                               cbf_poles=np.array([-3.0, -3.6, -5.6]))
    trk = mds.cbf.DroneQPTracker(cbf, order=order, num_robots=N, xdim=cbf.xdim, env=env)
    if shared_refs:
        trajs = [T.WaitTrajectory(init[0, j], 100.0) for j in range(N)] * E
    else:
        trajs = [T.WaitTrajectory(init[e, j], 100.0) for e in range(E) for j in range(N)]
    ts = mds.trajectories.TrajectorySet(trajs, dtype=dtype)
    return env, mds.FusedRollout(env, ts, c, trk, None)


def fused_and_two_launch(E, N, dtype, order, init, K, **kw):
    """observations after K steps in plan 6 and in plan 4, and plan 6's full-step log"""
    out = []
    for plan in (6, 4):
        env, ro = build(E, N, dtype, order, init, **kw)
        log = torch.zeros(K, E, N, 20, device="cuda", dtype=dtype)
        ro.run(K, stages=plan, obs_log=log, log_every=1)
        assert ro.stats_dict()["drone_steps"] == E * N * K
        out.append((env.obs.cpu().numpy().copy(), log.double().cpu().numpy()))
    return out


def check_plans(E, N, dtype, order, init, K, **kw):
    (o6, log6), (o4, log4) = fused_and_two_launch(E, N, dtype, order, init, K, **kw)
    assert np.all(np.isfinite(o6))
    if dtype == torch.float64:
        assert np.max(np.abs(log6 - log4)) < 1e-9 * (1 + np.max(np.abs(log4)))
    else:
        assert scaled_err(log6, log4) < 1e-5, scaled_err(log6, log4)
    return log6


def oracle_positions(init_e, N, order, K, physics=OPH.DYN_GND_DRAG_DW, pyb_freq=240):
    o = OracleCtrlAviary(ODM.CF2P, N, initial_xyzs=init_e, physics=physics, pyb_freq=pyb_freq)
    want, _, _ = opl.run_cbf(o, [otj.Wait(init_e[j], 100.0) for j in range(N)], order, K, log=True)
    return want[:, :, 0:3]


# (N, dtype, order, shared references): N = 8 is the packed pair loop (shared references: the reference-table kernel);
# every other N the run-time-N scalar loop -- odd N has no diameter slot, N = 1 no pairs, 16 two warps' halves
CASES = [(8, torch.float32, 3, True), (8, torch.float32, 3, False), (8, torch.float32, 2, True), (8, torch.float64, 3, False),
         (8, torch.float64, 2, True), (2, torch.float32, 3, False), (3, torch.float64, 2, False), (4, torch.float32, 2, False),
         (7, torch.float32, 3, False), (16, torch.float64, 3, False), (16, torch.float32, 2, False), (1, torch.float32, 3, False)]


@pytest.mark.parametrize("N,dtype,order,shared", CASES)
def test_stack_fused_downwash_equals_two_launch(N, dtype, order, shared, lib_built):
    """37 environments: not a multiple of the 32 environments of an fp32 8-drone block, so the last warps re-run an
    environment (FULLW) -- whose downwash terms must stay in their own lane group."""
    E, K = 37, 12
    rng = np.random.default_rng(100 + N)
    init = stack_init(E, N, rng)
    log6 = check_plans(E, N, dtype, order, init, K, shared_refs=shared)
    if N > 1:  # the stack really is in the downwash: the lower drones sink relative to a lone drone
        env1, ro1 = build(1, 1, dtype, order, init[:1, :1])
        ro1.run(K)
        assert abs(float(env1.obs[0, 0, 2]) - log6[-1, 0, 0, 2]) > 1e-6


@pytest.mark.parametrize("N,dtype,order", [(8, torch.float64, 3), (4, torch.float64, 2), (8, torch.float32, 3)])
def test_stack_fused_downwash_vs_oracle(N, dtype, order, lib_built):
    E, K = 3, 48
    init = stack_init(E, N, np.random.default_rng(7))
    env, ro = build(E, N, dtype, order, init)
    log = torch.zeros(K, E, N, 20, device="cuda", dtype=dtype)
    ro.run(K, obs_log=log, log_every=1)
    got = log.double().cpu().numpy()
    tol = 1e-6 if dtype == torch.float64 else 2e-3
    for e in range(E):
        want = oracle_positions(init[e], N, order, K)
        assert np.max(np.abs(got[:, e, :, 0:3] - want)) < tol, e


@pytest.mark.parametrize("N,dtype", [(8, torch.float32), (3, torch.float64)])
def test_two_physics_substeps(N, dtype, lib_built):
    """pyb_freq = 2 ctrl_freq: sub-step 0 takes the CBF stage's downwash, sub-step 1 exchanges the moved positions"""
    E, K = 37, 12
    init = stack_init(E, N, np.random.default_rng(5))
    check_plans(E, N, dtype, 3, init, K, pyb_freq=480)
    env, ro = build(2, N, dtype, 3, init[:2], pyb_freq=480)
    log = torch.zeros(K, 2, N, 20, device="cuda", dtype=dtype)
    ro.run(K, obs_log=log, log_every=1)
    got = log.double().cpu().numpy()
    tol = 1e-6 if dtype == torch.float64 else 2e-3
    for e in range(2):
        assert np.max(np.abs(got[:, e, :, 0:3] - oracle_positions(init[e], N, 3, K, pyb_freq=480))) < tol


@pytest.mark.parametrize("N,dtype", [(8, torch.float32), (4, torch.float64)])
def test_dyn_physics_with_cbf(N, dtype, lib_built):
    """physics without downwash: the CBF stage sums nothing and the stack falls freely of its neighbours"""
    E, K = 37, 12
    init = stack_init(E, N, np.random.default_rng(9))
    check_plans(E, N, dtype, 3, init, K, physics="dyn")
    env, ro = build(2, N, dtype, 3, init[:2], physics="dyn")
    log = torch.zeros(K, 2, N, 20, device="cuda", dtype=dtype)
    ro.run(K, obs_log=log, log_every=1)
    got = log.double().cpu().numpy()
    tol = 1e-6 if dtype == torch.float64 else 2e-3
    for e in range(2):
        assert np.max(np.abs(got[:, e, :, 0:3] - oracle_positions(init[e], N, 3, K, physics=OPH.DYN))) < tol


@pytest.mark.parametrize("N,dtype", [(8, torch.float32), (3, torch.float64)])
def test_cbf_rollout_with_wind(N, dtype, lib_built):
    """a constant world-frame force beside the fused downwash, in plans 6 and 4"""
    E, K = 6, 12
    init = stack_init(E, N, np.random.default_rng(13))
    wind = np.zeros((E, N, 3))
    wind[..., 0] = 0.0005 * (1 + np.arange(E))[:, None]
    out = {}
    for plan in (6, 4, "calm"):
        env, ro = build(E, N, dtype, 3, init)
        if plan != "calm":
            env.set_external_force(wind)
        out[plan] = ro.run(K, stages=6 if plan == "calm" else plan).double().cpu().numpy().copy()
    if dtype == torch.float64:
        assert np.max(np.abs(out[6] - out[4])) < 1e-9 * (1 + np.max(np.abs(out[4])))
    else:
        assert scaled_err(out[6], out[4]) < 1e-5
    assert np.max(np.abs(out["calm"][..., 0:3] - out[6][..., 0:3])) > 1e-6


def test_c5_split_calls_equal_one_call(lib_built):
    """The bench workload (reference table, one physics sub-step): 200 steps at 2 000 environments as calls of 24 equal
    one call of 200 bit for bit -- the one call refills the table every 32 steps, the calls of 24 never do."""
    from multidronesim_b200 import scenarios
    E, K, chunk = 2000, 200, 24
    runs = []
    for split in (False, True):
        sw = scenarios.cbf_swarm(E, 8, order=3)
        ro = sw["rollout"]
        if split:
            k = 0
            while k < K:
                ro.run(min(chunk, K - k))
                k += chunk
        else:
            ro.run(K)
        runs.append((sw["env"].obs.cpu().numpy().copy(), ro.stats_dict()))
    assert np.array_equal(runs[0][0], runs[1][0])
    for key in ("drone_steps", "qp_solves", "qp_iters", "qp_infeasible", "qp_iter_cap", "min_barrier"):
        assert runs[0][1][key] == runs[1][1][key], key
