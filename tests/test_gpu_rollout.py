"""GPU: the fused K-step rollout equals the per-call API loop, and both track the oracle's reference-style
closed loops (<= 1 mm over 1 s of hover / circle tracking in fp32; CBF closed loop)."""
import numpy as np
import pytest
import torch

from oracle import pipeline as opl
from oracle import trajectories as otj
from oracle.aviary import OracleCtrlAviary
from oracle.constants import DroneModel as ODM, Physics as OPH

pytestmark = pytest.mark.gpu


def build(E, N, dtype, physics, trajs_dev, ctrl, cbf_order=None, obstacles=None, init=None):
    import multidronesim_b200 as mds
    env = mds.BatchedCtrlAviary(drone_model=mds.DroneModel.CF2P, num_drones=N, physics=mds.Physics(physics), num_envs=E, dtype=dtype,
                                initial_xyzs=init)
    M = mds.model
    if ctrl == "geometric":
        c = mds.control.GeometricControl(env)
    elif ctrl == "torque12":
        c = mds.control.LQRController(env, M.LinearizedModel(env))
    elif ctrl == "omega9":
        c = mds.control.LQROmegaController(env, M.LinearizedOmegaModel(env), mds.control.ThrustOmegaController(env))
    else:
        c = mds.control.LQRYankOmegaController(env, M.LinearizedYankOmegaModel(env), mds.control.YankOmegaController(env))
    trk = None
    if cbf_order is not None:
        Mdl = M.LinearizedOmegaModel if cbf_order == 2 else M.LinearizedYankOmegaModel
        poles = np.array([-2.2, -2.4]) if cbf_order == 2 else np.array([-3.0, -3.6, -5.6])
        rs, zs = (0.1, 1.0) if cbf_order == 2 else (0.125, 2.0)
        cbf = mds.cbf.DroneCBF(env, [Mdl(env) for _ in range(N)], safety_radius=rs, zscale=zs, order=cbf_order, cbf_poles=poles,
                               allow_extra_obstacles=obstacles is not None and len(obstacles) > N)
        trk = mds.cbf.DroneQPTracker(cbf, order=cbf_order, num_robots=N, xdim=cbf.xdim, env=env)
    ts = mds.trajectories.TrajectorySet(trajs_dev, dtype=dtype)
    return mds, env, c, trk, ts, mds.FusedRollout(env, ts, c, trk, obstacles)


def percall_loop(mds, env, c, trk, ts, steps, obstacles):
    """the reference's loop structure through the per-call device API"""
    obs = env.obs
    t = 0.0
    obst = None if obstacles is None else torch.as_tensor(obstacles, device="cuda", dtype=env.dtype)
    mg = env.M * env.G
    for _ in range(steps):
        ref = ts.eval(t)
        c.set_reference(ref)
        if trk is None:
            out = c.compute(obs)
            action = out if isinstance(out, torch.Tensor) else out[0]
        else:
            _, u = c.compute(obs, skip_low_level=True)
            unom = u.clone()
            unom[..., 0] -= mg
            r3 = ref.view(env.NUM_ENVS, env.NUM_DRONES, 11)
            z = torch.zeros_like(r3[..., 0:1])
            if trk.order == 2:
                xdes = torch.cat([z, z, r3[..., 9:10], r3[..., 3:6], r3[..., 0:3]], dim=-1).contiguous()
            else:
                xdes = torch.cat([z, z, r3[..., 9:10], z + mg, r3[..., 3:6], r3[..., 0:3]], dim=-1).contiguous()
            us = trk.compute_control(obs, xdes, unom, x_obs=obst).clone()
            if trk.order == 2:
                us[..., 0] += mg
            action = c.compute_low_level(us, obs)
        obs = env.step(action)[0]
        t += env.CTRL_TIMESTEP
    return obs


def lem_params(N, E, rng, a=1.0, omega=0.5, z=0.5, ph0=0.0):
    ph = ph0 + (2 * np.pi / (N + 0.25)) * np.arange(N)
    return [dict(a=a, center=np.array([0, 0, z]), omega=omega, yaw_rate=0.0, phase_shift=float(p)) for p in ph]


@pytest.mark.parametrize("ctrl,cbf_order,physics,N", [("geometric", None, "dyn_gnd_drag_dw", 1), ("torque12", None, "dyn", 2),
                                                      ("omega9", None, "dyn_gnd_drag_dw", 3), ("yank10", None, "dyn", 2),
                                                      ("omega9", 2, "dyn_gnd_drag_dw", 2), ("yank10", 3, "dyn_gnd_drag_dw", 8)])
def test_fused_equals_percall(ctrl, cbf_order, physics, N, lib_built):
    import multidronesim_b200.trajectories as T
    E, steps, dtype = 5, 40, torch.float64
    rng = np.random.default_rng(2)
    specs = lem_params(N, E, rng)
    obstacles = [[0.0, 0.0, 0.5, 0.1]] if cbf_order is not None else None
    init = np.zeros((E, N, 3))
    for e in range(E):
        for j, sp in enumerate(specs):
            init[e, j] = otj.Lemniscate(**sp)(0.0)[0] + rng.normal(0, 0.02, 3) + np.array([0, 0, 0.03 * j])
    runs = []
    for fused in (True, False):
        mds, env, c, trk, ts, ro = build(E, N, dtype, physics, [T.Lemniscate(**sp) for sp in specs] * E, ctrl, cbf_order, obstacles, init)
        obs = ro.run(steps) if fused else percall_loop(mds, env, c, trk, ts, steps, obstacles)
        runs.append(obs.cpu().numpy().copy())
        if fused:
            st = ro.stats_dict()
            assert st["drone_steps"] == E * N * steps
    assert np.max(np.abs(runs[0] - runs[1])) < 1e-9 * (1 + np.max(np.abs(runs[1])))


@pytest.mark.parametrize("dtype,tol", [(torch.float64, 1e-7), (torch.float32, 1e-3)])
def test_c2_tracking_vs_oracle_1s(dtype, tol, lib_built):
    """config C2 in miniature: geometric controller tracking Circle / Lemniscate for 1 s (240 steps),
    DYN_GND_DRAG_DW; fp32 position within 1 mm of the fp64 oracle loop."""
    import multidronesim_b200.trajectories as T
    E, N, steps = 6, 1, 240
    rng = np.random.default_rng(1)
    dev_trajs, ora_trajs, init = [], [], np.zeros((E, N, 3))
    for e in range(E):
        if e % 2 == 0:
            kw = dict(r=1.0, v=0.5, center=np.array([0, 0, 1.0]), yaw_rate=0.0)
            dev_trajs.append(T.CircleTrajectory(**kw)); ora_trajs.append(otj.Circle(**kw))
        else:
            kw = dict(a=1.0, omega=1.5, center=np.array([0, 0, 0.5]), yaw_rate=0.0, phase_shift=float(rng.uniform(0, 2 * np.pi)))
            dev_trajs.append(T.Lemniscate(**kw)); ora_trajs.append(otj.Lemniscate(**kw))
        p0 = ora_trajs[-1](0.0)[0] + rng.normal(0, 0.05, 3)
        p0[2] = max(p0[2], 0.1)
        init[e, 0] = np.float32(p0)
    mds, env, c, trk, ts, ro = build(E, N, dtype, "dyn_gnd_drag_dw", dev_trajs, "geometric", init=init)
    log = torch.zeros(steps, E, N, 20, device="cuda", dtype=dtype)
    ro.run(steps, obs_log=log, log_every=1)
    got = log.double().cpu().numpy()
    worst = 0.0
    for e in range(E):
        o = OracleCtrlAviary(ODM.CF2P, N, initial_xyzs=init[e], physics=OPH.DYN_GND_DRAG_DW)
        want, _ = opl.run_tracking(o, [ora_trajs[e]], "geometric", steps)
        worst = max(worst, float(np.max(np.abs(got[:, e, :, 0:3] - want[:, :, 0:3]))))
    assert worst < tol, worst
    assert ro.stats_dict()["max_pos_err"] < 0.5


@pytest.mark.parametrize("order,N,dtype,tol", [(2, 2, torch.float64, 1e-6), (3, 4, torch.float64, 1e-6), (3, 5, torch.float64, 1e-6), (3, 8, torch.float32, 2e-3)])
def test_cbf_closed_loop_vs_oracle(order, N, dtype, tol, lib_built):
    """config C3 in miniature: LQR nominal -> CBF-QP -> inner loop -> DYN_GND_DRAG_DW, drones on one
    lemniscate through a sphere obstacle at its centre (simulations/CBFTest.py:418-424)."""
    import multidronesim_b200.trajectories as T
    E, steps = 3, 120
    rng = np.random.default_rng(3)
    # drone 0 starts 0.3 rad before the lemniscate's centre crossing, i.e. heading into the obstacle
    specs = lem_params(N, E, rng, omega=0.5, ph0=np.pi / 2 - 0.3)
    obstacles = [[0.0, 0.0, 0.5, 0.1]]
    init = np.zeros((E, N, 3))
    for e in range(E):
        for j, sp in enumerate(specs):
            init[e, j] = np.float32(otj.Lemniscate(**sp)(0.0)[0] + rng.normal(0, 0.02, 3) + np.array([0, 0, 0.04 * j]))
    ctrl = "omega9" if order == 2 else "yank10"
    mds, env, c, trk, ts, ro = build(E, N, dtype, "dyn_gnd_drag_dw", [T.Lemniscate(**sp) for sp in specs] * E, ctrl, order, obstacles, init)
    log = torch.zeros(steps, E, N, 20, device="cuda", dtype=dtype)
    ro.run(steps, obs_log=log, log_every=1)
    got = log.double().cpu().numpy()
    worst, n_active, ora_fail = 0.0, 0, 0
    for e in range(E):
        o = OracleCtrlAviary(ODM.CF2P, N, initial_xyzs=init[e], physics=OPH.DYN_GND_DRAG_DW)
        want, _, info = opl.run_cbf(o, [otj.Lemniscate(**sp) for sp in specs], order, steps, obstacles=obstacles)
        n_active += info["solves"]
        ora_fail += info["status"][1] + info["status"][2]
        # fp64 follows the oracle through infeasible steps too (same nominal fallback); fp32 is compared only
        # where the oracle's QP always solved (a borderline feasibility flip would fork the trajectories)
        if dtype == torch.float64 or info["status"][1] + info["status"][2] == 0:
            worst = max(worst, float(np.max(np.abs(got[:, e, :, 0:3] - want[:, :, 0:3]))))
    st = ro.stats_dict()
    assert worst < tol, worst
    assert st["qp_solves"] > 0 and n_active > 0
    assert st["qp_iter_cap"] == 0                                    # the device never gives up on a QP ...
    if dtype == torch.float64 or ora_fail == 0:
        assert st["qp_infeasible"] == ora_fail, (st, ora_fail)       # ... and falls back to the nominal input exactly where the oracle does


@pytest.mark.parametrize("dtype,tol", [(torch.float64, 1e-6), (torch.float32, 5e-3)])
def test_c5_full_lap_vs_oracle(dtype, tol, lib_built):
    """The bench workload (scenarios.cbf_swarm: 8 drones on one lemniscate, order-3 filter, sphere beside the crossing) over a
    whole lap (3024 control steps) against oracle/pipeline.run_cbf: same positions, and every QP the oracle solves the
    device solves (no iteration-cap or infeasible fallbacks)."""
    import multidronesim_b200 as mds
    from multidronesim_b200 import scenarios
    E, N, steps, every = 3, 8, 3024, 126
    sw = scenarios.cbf_swarm(E, N, order=3, dtype=dtype)
    ro = sw["rollout"]
    log = torch.zeros(steps // every, E, N, 20, device="cuda", dtype=dtype)
    ro.run(steps, obs_log=log, log_every=every)
    got = log.double().cpu().numpy()
    st = ro.stats_dict()
    phase = (2 * np.pi / (N + 0.25)) * np.arange(N)
    worst, fails = 0.0, 0
    for e in range(E):
        o = OracleCtrlAviary(ODM.CF2P, N, initial_xyzs=sw["init"][e], physics=OPH.DYN_GND_DRAG_DW)
        trajs = [otj.Lemniscate(a=1.0, omega=0.5, center=np.array([0, 0, 0.5]), yaw_rate=0.0, phase_shift=float(p)) for p in phase]
        want, _, info = opl.run_cbf(o, trajs, 3, steps, obstacles=scenarios.SWARM_OBSTACLES)
        fails += info["status"][1] + info["status"][2]
        worst = max(worst, float(np.max(np.abs(got[:, e, :, 0:3] - want[every - 1::every, :, 0:3]))))
    assert fails == 0                                   # the bench scenario is feasible all the way in the oracle ...
    assert st["qp_iter_cap"] == 0 and st["qp_infeasible"] == 0, st   # ... and on the device
    assert worst < tol, worst
    assert st["qp_solves"] > 0.5 * E * steps            # the filter is active in most steps of this workload


@pytest.mark.parametrize("ctrl,cbf_order,N,n_obs", [("yank10", 3, 8, 1), ("omega9", 2, 3, 1), ("geometric", None, 1, 0),
                                                    ("yank10", 3, 2, 4)])  # last: more obstacles than drones (SURVEY 8f-4)
def test_remaining_launch_plans_agree(ctrl, cbf_order, N, n_obs, lib_built):
    """MdsRolloutCfg.stages: the two-launch plan (4) and a launch-by-launch replay (1, then 2, per step) are the same
    computation: bit-identical observations, statistics, actions and rate-PID state.  The K-steps-in-one-launch plan (6)
    agrees with them to fp32 rounding, including the observation log.  Plans 4 and 6 run the K steps as two calls, so the
    second call starts from the state, rate-PID state and action the first one stored."""
    import multidronesim_b200.trajectories as T
    E, K, K1, dtype = 5, 9, 3, torch.float32
    rng = np.random.default_rng(11)
    specs = [dict(a=1.0, center=np.array([0, 0, 0.5]), omega=0.5, yaw_rate=0.1, phase_shift=float(2 * np.pi / (N + 0.25) * k)) for k in range(N)]
    init = np.zeros((E, N, 3))
    for e in range(E):
        for j, sp in enumerate(specs):
            init[e, j] = otj.Lemniscate(**sp)(0.0)[0] + rng.normal(0, 0.02, 3) + np.array([0, 0, 0.04 * j])
    obstacles = [[0.2, 0.0, 0.5, 0.1], [-0.3, 0.1, 0.6, 0.08], [0.9, 0.4, 0.45, 0.12], [-0.8, -0.3, 0.5, -0.1]][:n_obs] if cbf_order is not None else None
    outs = []
    for plan in ("two", "replay", "loop"):
        mds, env, c, trk, ts, ro = build(E, N, dtype, "dyn_gnd_drag_dw", [T.Lemniscate(**sp) for sp in specs] * E, ctrl, cbf_order, obstacles, init)
        log = torch.zeros(K // 3, E, N, 20, device="cuda", dtype=dtype)
        if plan == "replay":
            for k in range(K):
                ro.run(1, stages=1)
                ro.run(1, stages=2)
        else:
            if plan == "loop":
                assert ro.plan() == 6  # the default is the K-steps-in-one-launch plan
            # K1 is a whole number of log periods: the two calls fill the log of one K-step call
            ro.run(K1, obs_log=log[:K1 // 3], log_every=3, stages=4 if plan == "two" else 6)
            ro.run(K - K1, obs_log=log[K1 // 3:], log_every=3, stages=4 if plan == "two" else 6)
        assert abs(ro.t - K * env.CTRL_TIMESTEP) < 1e-12
        pid = (c.low_level._a.cpu().numpy().copy(), c.low_level._b.cpu().numpy().copy()) if ctrl in ("yank10", "omega9") else ()
        outs.append((env.obs.cpu().numpy().copy(), log.cpu().numpy().copy(), ro.stats.cpu().numpy().copy(), env._action.cpu().numpy().copy(), pid))
    for s in (3, 5, 7):  # plans that no longer exist
        with pytest.raises(ValueError):
            ro.run(1, stages=s)
    two, replay, loop = outs
    assert np.array_equal(two[0], replay[0]) and np.array_equal(two[2], replay[2]) and np.array_equal(two[3], replay[3])
    assert all(np.array_equal(x, y) for x, y in zip(two[4], replay[4]))
    assert np.abs(two[1]).max() > 0
    # the K-steps-in-one-launch plan is the same arithmetic compiled as one loop body: nvcc may contract a*b+c into
    # an FMA differently there, so it agrees to fp32 rounding (amplified over K closed-loop steps), not bit for bit;
    # its per-thread float accumulation of the error sum rounds differently, the counters are exact
    tol = dict(rtol=2e-4, atol=2e-4)
    assert np.allclose(two[0], loop[0], **tol) and np.allclose(two[1], loop[1], **tol)
    assert np.allclose(two[2], loop[2], rtol=1e-3) and two[2][0] == loop[2][0]
    assert np.allclose(two[3], loop[3], rtol=tol["rtol"], atol=tol["atol"] * 2e4)  # rotor speeds, ~1e4 rpm
    for x, y in zip(two[4], loop[4]):
        assert np.allclose(x, y, rtol=tol["rtol"], atol=tol["atol"] * 10)


def test_full_size_env_independence(lib_built):
    """At the bench size (125 000 envs x 8 drones) there is no oracle to compare with in reasonable time; the domain's
    size-independent property is that environments never interact: any environment rolled out inside the 1M-drone swarm
    must equal, bit for bit, the same environment rolled out in a tiny batch (same shard-invariant initial conditions),
    and the statistics must count every drone-step.  Checks indexing at scale (first, interior, last block, last env)."""
    from multidronesim_b200 import scenarios
    E, K = 125000, 48
    big = scenarios.cbf_swarm(E, 8, order=3)
    big["rollout"].run(K)
    st = big["rollout"].stats_dict()
    assert st["drone_steps"] == E * 8 * K
    assert np.isfinite(st["sum_pos_err"]) and st["max_pos_err"] < 1.0 and st["qp_solves"] > 0
    obs_big = big["env"].obs
    assert bool(torch.isfinite(obs_big).all())
    for e0 in (0, 31, 32, 77777, E - 1):
        small = scenarios.cbf_swarm(1, 8, order=3, env_offset=e0)
        assert np.array_equal(small["init"][0], big["init"][e0])
        small["rollout"].run(K)
        assert torch.equal(small["env"].obs[0], obs_big[e0]), e0


def test_rollout_with_wind_in_plans_6_and_4(lib_built):
    """A constant per-drone world-frame force (the reference's wind, EnvGeometric.py:463-467; set_external_force) acts in
    every launch plan of the rollout exactly as in the per-call loop, and changes the flight."""
    import multidronesim_b200.trajectories as T
    E, N, K, dtype = 4, 2, 30, torch.float64
    specs = [dict(a=0.8, center=np.array([0, 0, 0.8]), omega=0.7, yaw_rate=0.0, phase_shift=float(k)) for k in range(N)]
    init = np.array([[otj.Lemniscate(**sp)(0.0)[0] for sp in specs]] * E)
    wind = np.zeros((E, N, 3)); wind[..., 0] = 0.00025 * (1 + np.arange(E))[:, None]
    outs = {}
    for plan in ("percall", 6, 4, "calm"):
        mds, env, c, trk, ts, ro = build(E, N, dtype, "dyn_gnd_drag_dw", [T.Lemniscate(**sp) for sp in specs] * E, "geometric", init=init)
        if plan != "calm":
            env.set_external_force(wind)
        obs = percall_loop(mds, env, c, trk, ts, K, None) if plan == "percall" else ro.run(K, stages=6 if plan == "calm" else plan)
        outs[plan] = obs.cpu().numpy().copy()
    for plan in (6, 4):
        assert np.max(np.abs(outs[plan] - outs["percall"])) < 1e-9 * (1 + np.max(np.abs(outs["percall"]))), plan
    assert np.max(np.abs(outs["calm"][..., 0:3] - outs[6][..., 0:3])) > 1e-5   # the wind moved the drones


@pytest.mark.parametrize("dtype,tol", [(torch.float64, 1e-7), (torch.float32, 1e-3)])
def test_cf2x_x_frame_mixer_tracking(dtype, tol, lib_built):
    """SURVEY 8f-4 extension: a CF2X under the torque-level geometric controller with the X-frame mixer
    (``x_frame_mixer=True``; the reference's mixer is PLUS-frame whatever the model).  2 s of circle tracking in
    DYN_GND_DRAG_DW: against the oracle loop with the same switch, and the drone really tracks (it does not with
    the PLUS-frame mixer, whose roll / pitch torques land 45 degrees off a CF2X's axes)."""
    import multidronesim_b200 as mds
    import multidronesim_b200.trajectories as T
    E, N, steps = 3, 1, 480
    kw = dict(r=1.0, v=0.5, center=np.array([0, 0, 1.0]), yaw_rate=0.0)
    init = np.zeros((E, N, 3))
    for e in range(E):
        init[e, 0] = np.float32(otj.Circle(**kw)(0.0)[0] + np.array([0.03 * e, -0.02 * e, 0.01 * e]))
    env = mds.BatchedCtrlAviary(drone_model=mds.DroneModel.CF2X, num_drones=N, physics=mds.Physics.DYN_GND_DRAG_DW, num_envs=E, dtype=dtype,
                                initial_xyzs=init, x_frame_mixer=True)
    c = mds.control.GeometricControl(env)
    ts = mds.trajectories.TrajectorySet([T.CircleTrajectory(**kw)] * E, dtype=dtype)
    ro = mds.FusedRollout(env, ts, c, None, None)
    log = torch.zeros(steps, E, N, 20, device="cuda", dtype=dtype)
    ro.run(steps, obs_log=log, log_every=1)
    got = log.double().cpu().numpy()
    worst = 0.0
    for e in range(E):
        o = OracleCtrlAviary(ODM.CF2X, N, initial_xyzs=init[e], physics=OPH.DYN_GND_DRAG_DW, x_frame_mixer=True)
        want, _ = opl.run_tracking(o, [otj.Circle(**kw)], "geometric", steps)
        worst = max(worst, float(np.max(np.abs(got[:, e, :, 0:3] - want[:, :, 0:3]))))
    assert worst < tol, worst
    ref_end = otj.Circle(**kw)((steps - 1) * env.CTRL_TIMESTEP)[0]
    assert np.abs(got[-1, :, 0, 0:3] - ref_end).max() < 0.1           # converging from a standing start: 7-8 cm behind after 2 s
    assert ro.stats_dict()["max_pos_err"] < 0.2                       # (the PLUS-frame mixer loses a CF2X: tests/test_oracle_env.py)


def test_host_pipelines_equal_device_paths(lib_built):
    """HostPipeline (pinned host references in, pinned host observations out, three streams / two slots) delivers, step by step,
    exactly what PerCallPipeline computes with device buffers; its ref-ready event fires before the host reference buffer is
    reused.  HostRollout (K-step host call: one launch + one large D2H, double-buffered) delivers FusedRollout's observation log."""
    import multidronesim_b200 as mds
    import multidronesim_b200.trajectories as T
    E, N, steps, dtype = 7, 4, 12, torch.float32
    rng = np.random.default_rng(4)
    specs = lem_params(N, E, rng)
    obstacles = [[0.2, 0.0, 0.5, 0.1]]
    init = np.zeros((E, N, 3))
    for e in range(E):
        for j, sp in enumerate(specs):
            init[e, j] = otj.Lemniscate(**sp)(0.0)[0] + rng.normal(0, 0.02, 3) + np.array([0, 0, 0.04 * j])
    trajs_dev = [T.Lemniscate(**sp) for sp in specs] * E
    # device-buffer path
    mds_, env, c, trk, ts, ro = build(E, N, dtype, "dyn_gnd_drag_dw", trajs_dev, "yank10", 3, obstacles, init)
    pipe = mds.PerCallPipeline(env, c, trk, obstacles)
    want = []
    for k in range(steps):
        want.append(pipe.step(ts.eval(k * env.CTRL_TIMESTEP)).clone().cpu().numpy())
    # host-buffer path: ONE pinned reference buffer reused every step (legal once last_ref_ready has fired)
    mds_, env2, c2, trk2, ts2, ro2 = build(E, N, dtype, "dyn_gnd_drag_dw", trajs_dev, "yank10", 3, obstacles, init)
    hp = mds.HostPipeline(env2, c2, trk2, obstacles)
    ref_host = torch.empty(E * N, 11, dtype=dtype).pin_memory()
    obs_host = [torch.empty(E, N, 20, dtype=dtype).pin_memory() for _ in range(2)]
    for k in range(steps):
        ref_host.copy_(ts2.eval(k * env2.CTRL_TIMESTEP))
        torch.cuda.synchronize()
        done = hp.step(ref_host, obs_host[k & 1])
        hp.last_ref_ready.synchronize()          # the reference buffer may be overwritten from here on
        ref_host.fill_(float("nan"))
        done.synchronize()
        assert np.array_equal(obs_host[k & 1].numpy(), want[k]), k
    hp.synchronize()
    # K-step host call against the fused rollout's own log
    K = 6
    mds_, env3, c3, trk3, ts3, ro3 = build(E, N, dtype, "dyn_gnd_drag_dw", trajs_dev, "yank10", 3, obstacles, init)
    log = torch.zeros(2 * K, E, N, 20, device="cuda", dtype=dtype)
    ro3.run(2 * K, obs_log=log, log_every=1)
    mds_, env4, c4, trk4, ts4, ro4 = build(E, N, dtype, "dyn_gnd_drag_dw", trajs_dev, "yank10", 3, obstacles, init)
    hr = mds.HostRollout(ro4, K)
    out = [torch.empty(K, E, N, 20, dtype=dtype).pin_memory() for _ in range(2)]
    evs = [hr.step(out[j]) for j in range(2)]
    for j in range(2):
        evs[j].synchronize()
        assert np.array_equal(out[j].numpy(), log[j * K:(j + 1) * K].cpu().numpy()), j
    hr.synchronize()


def test_swarm_streams_equal_one_swarm(lib_built):
    """scenarios.cbf_swarm_streams: the C5 swarm cut into sub-swarms advanced on their own CUDA streams (SwarmStreams) is, env for
    env, the swarm run as one: identical observations (same kernel, same per-env inputs) and the same combined statistics."""
    from multidronesim_b200 import scenarios
    E, K = 90, 30
    one = scenarios.cbf_swarm(E, 8, order=3)
    one["rollout"].run(K); one["rollout"].run(K)
    swarm, subs = scenarios.cbf_swarm_streams(E, 3, 8, order=3)
    swarm.run(K); swarm.run(K)
    swarm.synchronize()
    got = torch.cat([s["env"].obs for s in subs], dim=0)
    assert torch.equal(got, one["env"].obs)
    a, b = one["rollout"].stats_dict(), swarm.stats_dict()
    for k in ("drone_steps", "qp_solves", "qp_iters", "qp_infeasible", "qp_iter_cap", "max_pos_err", "min_barrier"):
        assert a[k] == b[k], k
    assert abs(a["sum_pos_err"] - b["sum_pos_err"]) < 1e-6 * a["sum_pos_err"]


def test_extrema_statistics_across_blocks(lib_built):
    """min_barrier / max_pos_err are folded over the blocks of a launch with integer atomics on the doubles' bit patterns
    (mds_rollout.cuh atomic_min_double / atomic_max_double; the barrier minimum is usually NEGATIVE, the error maximum never).
    A swarm of E environments (several blocks, last warp partly filled: the FULLW re-run groups must not count) has to report
    the extrema of its environments rolled out one by one -- single-block launches whose results are folded here on the host --
    and exact counters."""
    from multidronesim_b200 import scenarios
    E, K = 70, 96
    big = scenarios.cbf_swarm(E, 8, order=3)
    big["rollout"].run(K)
    st = big["rollout"].stats_dict()
    assert st["drone_steps"] == E * 8 * K
    mins, maxs, solves = [], [], 0
    for e0 in range(E):
        one = scenarios.cbf_swarm(1, 8, order=3, env_offset=e0)
        one["rollout"].run(K)
        s1 = one["rollout"].stats_dict()
        assert s1["drone_steps"] == 8 * K
        mins.append(s1["min_barrier"]); maxs.append(s1["max_pos_err"]); solves += s1["qp_solves"]
    assert min(mins) < 0 < max(maxs)           # the sign cases the atomics distinguish are exercised
    assert st["min_barrier"] == min(mins) and st["max_pos_err"] == max(maxs) and st["qp_solves"] == solves


def test_persistent_ctrl_kernel_walks_its_tiles(lib_built):
    """ctrl_step_kernel is persistent (mds_rollout.cuh): its grid is capped at the resident set (2 blocks per SM) and every block
    walks block-sized tiles of the environments with stride gridDim.x.  Small swarms never make a block take a second tile,
    so this runs the two-launch plan on 21 003 environments (657 tiles on at most 296 blocks, last tile partly filled) and
    checks (a) environments first, interior, at tile / grid-stride boundaries and last against the same environments
    rolled out alone -- environments never interact, and a one-environment launch is a single tile -- bit for bit, and
    (b) that the statistics count every drone-step exactly once."""
    from multidronesim_b200 import scenarios
    E, K = 21003, 6
    big = scenarios.cbf_swarm(E, 8, order=3)
    big["rollout"].run(K, stages=4)
    st = big["rollout"].stats_dict()
    assert st["drone_steps"] == E * 8 * K
    # the K-step loop kernel (plan 6) is the same arithmetic compiled as one loop body: its QP counters agree up to the few
    # borderline decisions fp32 rounding can flip among 126 018 environment-steps (the swarm starts from rest: some early QPs
    # are infeasible and fall back, as in the reference)
    ref = scenarios.cbf_swarm(E, 8, order=3)
    ref["rollout"].run(K, stages=6)
    sr = ref["rollout"].stats_dict()
    for k in ("qp_solves", "qp_iters", "qp_infeasible", "qp_iter_cap"):
        assert abs(st[k] - sr[k]) <= 0.02 * max(sr[k], 50.0), (k, st[k], sr[k])
    obs_big = big["env"].obs
    assert bool(torch.isfinite(obs_big).all())
    for e0 in (0, 31, 32, 296 * 32 - 1, 296 * 32, 296 * 32 + 33, 2 * 296 * 32 + 5, E - 4, E - 1):
        small = scenarios.cbf_swarm(1, 8, order=3, env_offset=e0)
        small["rollout"].run(K, stages=4)
        assert torch.equal(small["env"].obs[0], obs_big[e0]), e0
