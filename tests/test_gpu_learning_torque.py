"""TorqueLearningRollout / mds_learning_rollout_torque: the learning loop of the 12-dim torque-level DecentralizedLQR -- open
loop, under each drone's own gain and under the robot-coupled gain -- K steps in one launch, against the per-call loop over
mds_error_state, input_to_action, mds_physics_step (and mds_dlqr_ctrl) and mds_rls_update, and against the oracle.  The
C-argument refusals run without a GPU."""
import ctypes

import numpy as np
import pytest
import torch

from multidronesim_b200 import _lib

gpu = pytest.mark.gpu

# (method, gain, E, N, physics, wind, lemniscate); gain: "open" (no feedback), "drone" (per-drone gains), "coupled"
CASES = {
    "open_theta_update": ("theta_update", "open", 3, 2, "DYN", False, False),
    "open_approx": ("approx_theta_update", "open", 5, 3, "DYN_GND_DRAG_DW", True, True),
    "drone_theta_update": ("theta_update", "drone", 4, 2, "DYN_GND_DRAG_DW", True, False),
    "drone_approx": ("approx_theta_update", "drone", 3, 3, "DYN", False, True),
    "coupled_theta_update": ("theta_update", "coupled", 4, 2, "DYN", True, True),   # DYN: no group sync inside the physics step
    "coupled_approx": ("approx_theta_update", "coupled", 6, 3, "DYN_GND_DRAG_DW", False, False),
}


def make_setup(E, N, dtype, physics="DYN", wind=False, lemniscate=False, gain="open", seed=0):
    """env, DecentralizedLQR (gains as `gain` asks, from the prior models) and TrajectorySet, the same for every dtype"""
    import multidronesim_b200 as mds
    import multidronesim_b200.trajectories as T
    from multidronesim_b200.control import dlqr
    rng = np.random.default_rng(seed)
    if lemniscate:
        specs = [dict(a=1.0, center=np.array([0, 0, 1.0]), omega=0.5, yaw_rate=0.0, phase_shift=float(p)) for p in (2 * np.pi / (N + 0.25)) * np.arange(N)]
        from oracle import trajectories as otj
        init = np.array([[otj.Lemniscate(**sp)(0.0)[0] for sp in specs]] * E) + rng.normal(0, 0.02, (E, N, 3)) + np.array([0, 0, 0.1]) * np.arange(N)[:, None]
        trajs = [T.Lemniscate(**sp) for sp in specs] * E
    else:
        init = rng.uniform(-0.5, 0.5, (E, N, 3)) + np.array([0, 0, 1.0])
        init[..., 2] += 0.15 * np.arange(N)  # drones of an environment stacked: downwash acts where it is on
        trajs = [T.WaitTrajectory(init[e, j], 1000.0) for e in range(E) for j in range(N)]
    env = mds.BatchedCtrlAviary(drone_model=mds.DroneModel.CF2P, num_drones=N, num_envs=E, dtype=dtype, initial_xyzs=init,
                                physics=getattr(mds.Physics, physics))
    if wind:
        env.set_external_force(rng.normal(0, 0.01, (E, N, 3)))
    dl = dlqr.DecentralizedLQR(env, [mds.model.LinearizedModel(env) for _ in range(N)])
    if gain == "drone":
        dl.compute_controller(force_diagonal=True)   # per-drone gains, device Riccati solve
    elif gain == "coupled":
        dl.compute_controller()                      # N >= 2: the robot-coupled gain (host solve); N = 1: per-drone
        assert dl._coupled == (N >= 2)
    return env, dl, mds.trajectories.TrajectorySet(trajs, dtype=dtype)


def inputs_for(gain, K, E, N, seed=1, thrust_lo=0.7):
    """[K, E, N, 4] float64 numpy: open loop, sigma1-like torque-level inputs (thrust in [thrust_lo, 1.5] m g, torques +-1e-5 N m);
    with a gain, perturbations of the law (+-0.1 m g, +-5e-6 N m)"""
    mg = 0.027 * 9.8
    rng = np.random.default_rng(seed)
    if gain == "open":
        return np.concatenate([rng.uniform(thrust_lo * mg, 1.5 * mg, (K, E, N, 1)), rng.uniform(-1e-5, 1e-5, (K, E, N, 3))], axis=-1)
    return np.concatenate([rng.uniform(-0.1 * mg, 0.1 * mg, (K, E, N, 1)), rng.uniform(-5e-6, 5e-6, (K, E, N, 3))], axis=-1)


def percall_loop(env, dl, ts, us, method, learn_from, feedback, t0=0.0, obs_steps=None):
    """the loop TorqueLearningRollout.run replaces; obs_steps (a list) receives every step's observation"""
    from multidronesim_b200 import utils as U
    obs = env.obs
    for k in range(us.shape[0]):
        dl.set_reference(ts.eval(t0 + k * env.CTRL_TIMESTEP))
        e_t = dl.error_state(obs).clone()
        if feedback:
            _, u = dl.compute(obs, skip_low_level=True)
            u = u + us[k]
        else:
            u = us[k].clone()
        obs = env.step(U.input_to_action(env, u))[0]   # clamps u[..., 0] >= 0 in place
        if obs_steps is not None:
            obs_steps.append(obs.double().cpu().numpy().copy())
        if k >= learn_from:
            getattr(dl, method)(torch.cat([e_t, u], -1), dl.error_state(obs).clone())
    return obs


def outputs(env, dl):
    """the quantities the loop leaves behind, float64 numpy"""
    f = lambda t: t.detach().double().cpu().numpy().copy()
    return {"theta": f(dl.theta), "P": f(dl.P), "obs": f(env.obs)[..., :16], "resid": f(dl.resid), "K": f(dl.K_planes),
            "state": np.concatenate([f(env._pos_wx), f(env._quat), f(env._vel_wy), f(env._wz)[:, None]], axis=1)}


def run_both(method, gain, E, N, dtype, physics, wind, lemniscate, K, learn_from, seed=0, phases=1, us_np=None, set_gain=None):
    """per-call and fused from identical setups; `phases` runs of K steps with compute_controller() between them;
    set_gain(dl): installs a gain of the test's own after the setup"""
    import multidronesim_b200 as mds
    if us_np is None:
        us_np = inputs_for(gain, K * phases, E, N, seed + 1)
    feedback = gain != "open"
    res = {}
    for mode in ("percall", "fused"):
        env, dl, ts = make_setup(E, N, dtype, physics, wind, lemniscate, "open" if set_gain else gain, seed)
        if set_gain:
            set_gain(dl)
        us = torch.as_tensor(us_np, device="cuda", dtype=dtype).contiguous()
        ro = mds.TorqueLearningRollout(env, ts, dl)
        res[mode + "_prior_theta"] = dl.theta.double().cpu().numpy().copy()
        for ph in range(phases):
            if ph:
                dl.compute_controller()
            K0 = dl.K_planes.clone()
            part = us[ph * K:(ph + 1) * K]
            if mode == "percall":
                percall_loop(env, dl, ts, part, method, learn_from, feedback, t0=ph * K * env.CTRL_TIMESTEP)
            else:
                ro.run(part, method=method, learn_from=learn_from, feedback=feedback)
                assert torch.equal(dl.K_planes, K0)  # the launch reads the gain, never writes it
        if mode == "fused":
            assert env.step_counter == K * phases * env.PYB_STEPS_PER_CTRL and abs(ro.t - K * phases * env.CTRL_TIMESTEP) < 1e-12
        torch.cuda.synchronize()
        res[mode] = outputs(env, dl)
    return res


def err(a, b):
    return float(np.abs(a - b).max()) / max(1.0, float(np.abs(b).max()))


def check_fp64(got, want, what, keys=("theta", "P", "obs", "resid", "state")):
    for k in keys:
        assert err(got[k], want[k]) <= 1e-9, (what, k, err(got[k], want[k]))


def check_fp32(fused32, percall32, percall64, what):
    for k in ("theta", "P", "obs", "resid", "state"):
        e_fused, e_call = err(fused32[k], percall64[k]), err(percall32[k], percall64[k])
        assert e_fused <= max(2 * e_call, 2e-4), (what, k, e_fused, e_call)


def check_both_dtypes(what, *args, **kw):
    r64 = run_both(*args, dtype=torch.float64, **kw)
    check_fp64(r64["fused"], r64["percall"], what)
    r32 = run_both(*args, dtype=torch.float32, **kw)
    check_fp32(r32["fused"], r32["percall"], r64["percall"], what)
    return r64


@gpu
@pytest.mark.parametrize("tag", list(CASES))
def test_parity_with_percall_loop(tag, lib_built):
    """Both methods x open loop / per-drone gains / coupled gains, K = 40, learn_from = 1: fp64 to 1e-9 of each quantity's
    scale; fp32 no further from the per-call fp64 run than twice the per-call fp32 run (or 2e-4 of the scale).  theta moved."""
    method, gain, E, N, physics, wind, lem = CASES[tag]
    r64 = check_both_dtypes(tag, method, gain, E, N, physics=physics, wind=wind, lemniscate=lem, K=40, learn_from=1)
    assert err(r64["fused"]["theta"], r64["fused_prior_theta"]) > 1e-6  # the models moved


def dense_coupled_gain(seed=3):
    """installs a random dense robot-coupled gain (any gain will do: this tests the law, not the CARE); thrust rows 1e-3,
    torque rows 1e-6, so that 16 steps stay near hover"""
    def install(dl):
        env = dl.env
        E, N, m = env.NUM_ENVS, env.NUM_DRONES, dl.m
        rng = np.random.default_rng(seed)
        Kfull = rng.normal(0, 1.0, (E, N, 4, N * m)) * np.array([1e-3, 1e-6, 1e-6, 1e-6])[None, None, :, None]
        Kfull = Kfull.reshape(E, 4 * N, m * N)
        planes = Kfull.reshape(E, N, 4, N, m).transpose(3, 2, 4, 0, 1).reshape(N * 4 * m, E * N)
        dl._coupled = True
        dl.K_planes = torch.as_tensor(np.ascontiguousarray(planes), device="cuda", dtype=env.dtype)
        dl.K = Kfull
    return install


@gpu
@pytest.mark.parametrize("E,N", [(7, 5), (3, 32)])
def test_coupled_law_odd_sizes(E, N, lib_built):
    """Random dense coupled gains at group sizes that do not fill a warp (N = 5) and the largest group (N = 32; fp64 stages
    93 KB per block, past 48 KB of shared memory), both precisions, against the per-call loop with mds_dlqr_ctrl."""
    check_both_dtypes((E, N), "theta_update", "coupled", E, N, physics="DYN_GND_DRAG_DW", wind=False, lemniscate=False, K=16, learn_from=1,
                      seed=3, set_gain=dense_coupled_gain())


@gpu
def test_thrust_clamp_reaches_phi(lib_built):
    """Open-loop inputs with negative thrusts: input_to_action clamps them to 0 in place and the RLS step must see the clamped
    u in phi (the per-call loop's phi); both precisions."""
    E, N, K = 4, 3, 40
    us = inputs_for("open", K, E, N, seed=12, thrust_lo=-0.5)
    assert (us[..., 0] < 0).mean() > 0.2
    check_both_dtypes("clamp", "approx_theta_update", "open", E, N, physics="DYN_GND_DRAG_DW", wind=True, lemniscate=False, K=K,
                      learn_from=1, us_np=us)


@gpu
def test_certainty_equivalence_phases(lib_built):
    """Three phases of 30 steps under the robot-coupled gain with dl.compute_controller() (host solver) between them, fp64:
    theta, P, K_planes, obs and the state to 1e-9 of their scale."""
    r = run_both("theta_update", "coupled", 3, 2, torch.float64, "DYN_GND_DRAG_DW", True, False, 30, 1, seed=6, phases=3)
    check_fp64(r["fused"], r["percall"], "phases", keys=("theta", "P", "K", "obs", "state"))
    assert err(r["fused"]["theta"], r["fused_prior_theta"]) > 1e-6


@gpu
@pytest.mark.parametrize("dtype", [torch.float64, torch.float32])
def test_split_calls_are_bit_identical(dtype, lib_built):
    """run(K) == run(K1) + run(K - K1) under the coupled gain, bit for bit (state, obs, theta, P)."""
    import multidronesim_b200 as mds
    E, N, K, K1 = 5, 3, 30, 11
    us = torch.as_tensor(inputs_for("coupled", K, E, N, 7), device="cuda", dtype=dtype).contiguous()
    res = []
    for parts in ((K,), (K1, K - K1)):
        env, dl, ts = make_setup(E, N, dtype, "DYN_GND_DRAG_DW", gain="coupled", seed=5)
        ro = mds.TorqueLearningRollout(env, ts, dl)
        k0 = 0
        for p in parts:
            ro.run(us[k0:k0 + p], method="approx_theta_update", feedback=True)
            k0 += p
        res.append(outputs(env, dl))
    for k in ("theta", "P", "obs", "state"):
        assert np.array_equal(res[0][k], res[1][k]), k


@gpu
@pytest.mark.parametrize("dtype", [torch.float64, torch.float32])
@pytest.mark.parametrize("gain", ["open", "drone"])
def test_no_learning_leaves_the_model_alone(gain, dtype, lib_built):
    """learn_from >= K: theta and P come back bit-identical, and the flight equals that of learn_from = 0 bit for bit (the gain
    is fixed within the launch)."""
    import multidronesim_b200 as mds
    E, N, K = 4, 3, 20
    us = torch.as_tensor(inputs_for(gain, K, E, N, 9), device="cuda", dtype=dtype).contiguous()
    res = []
    for learn_from in (K, 0):
        env, dl, ts = make_setup(E, N, dtype, "DYN_GND_DRAG_DW", wind=True, gain=gain, seed=2)
        th0, P0 = dl.theta_planes.clone(), dl.P_planes.clone()
        mds.TorqueLearningRollout(env, ts, dl).run(us, learn_from=learn_from, feedback=gain != "open")
        if learn_from == K:
            assert torch.equal(dl.theta_planes, th0) and torch.equal(dl.P_planes, P0)
        else:
            assert not torch.equal(dl.theta_planes, th0)
        res.append(outputs(env, dl))
    for k in ("obs", "state"):
        assert np.array_equal(res[0][k], res[1][k]), k


@gpu
@pytest.mark.parametrize("dtype", [torch.float64, torch.float32])
@pytest.mark.parametrize("gain", ["open", "coupled"])
def test_odd_sizes(gain, dtype, lib_built):
    """E = 37 (not a multiple of the environments per block) with N = 1, where compute_controller() gives a per-drone gain."""
    r = run_both("theta_update", gain, 37, 1, dtype, "DYN", False, False, 16, 1, seed=3)
    if dtype == torch.float64:
        check_fp64(r["fused"], r["percall"], gain)
    else:
        r64 = run_both("theta_update", gain, 37, 1, torch.float64, "DYN", False, False, 16, 1, seed=3)
        check_fp32(r["fused"], r["percall"], r64["percall"], gain)


@gpu
@pytest.mark.parametrize("dtype", [torch.float64, torch.float32])
def test_obs_log_matches_percall_steps(dtype, lib_built):
    """obs_log / log_every: slot j holds the observation after step (j + 1) * log_every, as the per-call loop saw it (K = 20,
    log_every = 3: six slots, the last two steps unlogged; a spare slot stays untouched)."""
    import multidronesim_b200 as mds
    E, N, K, every = 5, 3, 20, 3
    us = torch.as_tensor(inputs_for("open", K, E, N, 11), device="cuda", dtype=dtype).contiguous()
    env, dl, ts = make_setup(E, N, dtype, "DYN_GND_DRAG_DW", seed=4)
    want = []
    percall_loop(env, dl, ts, us, "theta_update", 0, False, obs_steps=want)
    env2, dl2, ts2 = make_setup(E, N, dtype, "DYN_GND_DRAG_DW", seed=4)
    log = torch.full((K // every + 1, E, N, _lib.OBS_DIM), -7.0, device="cuda", dtype=dtype)
    last = mds.TorqueLearningRollout(env2, ts2, dl2).run(us, obs_log=log, log_every=every)
    got = log.double().cpu().numpy()
    tol = 1e-9 if dtype == torch.float64 else 2e-4
    for j in range(K // every):
        w = want[(j + 1) * every - 1][..., :16]
        assert np.abs(got[j][..., :16] - w).max() <= tol * max(1.0, np.abs(w).max()), j
    assert (got[K // every] == -7.0).all()
    assert np.abs(last.double().cpu().numpy()[..., :16] - want[-1][..., :16]).max() <= tol * max(1.0, np.abs(want[-1][..., :16]).max())


@gpu
def test_learning_loop_vs_oracle(lib_built):
    """40 open-loop steps of the torque-level model in ONE fp64 call against the oracle loop (aviary,
    conversions.input_to_action, sysid theta_update with project_theta after the update), with test_learning_loop_vs_oracle's
    thresholds."""
    import multidronesim_b200 as mds
    import multidronesim_b200.trajectories as T
    from oracle import controllers as oc
    from oracle import conversions as cv
    from oracle import sysid
    from oracle.aviary import OracleCtrlAviary
    from oracle.constants import DroneModel as ODM, Physics as OPH
    E, N, steps, dtype = 3, 2, 40, torch.float64
    rng = np.random.default_rng(21)
    init = rng.uniform(-0.5, 0.5, (E, N, 3)) + np.array([0, 0, 1.0])
    env = mds.BatchedCtrlAviary(drone_model=mds.DroneModel.CF2P, num_drones=N, num_envs=E, dtype=dtype, initial_xyzs=init, physics=mds.Physics.DYN)
    dl = mds.control.DecentralizedLQR(env, [mds.model.LinearizedModel(env) for _ in range(N)])
    ts = mds.trajectories.TrajectorySet([T.WaitTrajectory(init[e, j], 1000.0) for e in range(E) for j in range(N)], dtype=dtype)
    mg = env.M * env.G
    us = np.concatenate([rng.uniform(0.7 * mg, 1.5 * mg, (steps, E, N, 1)), rng.uniform(-1e-5, 1e-5, (steps, E, N, 3))], axis=-1)
    oenvs = [OracleCtrlAviary(ODM.CF2P, N, initial_xyzs=init[e], physics=OPH.DYN) for e in range(E)]
    octl = [[oc.Lqr(oenvs[e], "torque12", K=np.zeros((4, 12))) for _ in range(N)] for e in range(E)]
    th = dl.theta.cpu().numpy().copy().reshape(E, N, 16, 12)
    P = dl.P.cpu().numpy().copy().reshape(E, N, 16, 16)
    codes = sysid.project_codes(12)
    oobs = [o.reset()[0] for o in oenvs]
    obs = mds.TorqueLearningRollout(env, ts, dl).run(torch.as_tensor(us, device="cuda", dtype=dtype).contiguous(), learn_from=1)
    for i in range(steps):
        for e in range(E):
            ophis, act = [], np.zeros((N, 4))
            for j in range(N):
                c = octl[e][j]
                c.set_desired_trajectory(j, init[e, j], np.zeros(3), np.zeros(3), 0.0, 0.0)
                u = us[i, e, j].copy()
                act[j] = cv.input_to_action(oenvs[e], u)     # clamps u[0] in place
                ophis.append(np.hstack([c.error_state(oobs[e][j]), u]))
            oobs[e] = oenvs[e].step(act)[0]
            if i != 0:
                for j in range(N):
                    th[e, j], P[e, j], _ = sysid.rls_update(th[e, j], P[e, j], ophis[j], octl[e][j].error_state(oobs[e][j]), env.CTRL_TIMESTEP,
                                                            sysid.TARGET_PREDICT, False, True, sysid.PROJECT_AFTER, codes)
    got_th = dl.theta.cpu().numpy().reshape(E, N, 16, 12)
    got_P = dl.P.cpu().numpy().reshape(E, N, 16, 16)
    assert np.abs(obs.cpu().numpy() - np.array(oobs))[..., :16].max() < 1e-8
    assert np.abs(got_th - th).max() <= 1e-8 * np.abs(th).max(), np.abs(got_th - th).max()
    assert np.abs(got_P - P).max() <= 1e-8 * np.abs(P).max()
    lm = mds.model.LinearizedModel(env)
    assert np.abs(th - np.hstack([lm.Ahat, lm.Bhat]).T).max() > 1e-3  # the models really moved


@gpu
def test_refusals(lib_built):
    """TorqueLearningRollout refuses, before any launch, other controllers, malformed inputs, methods DecentralizedLQR does
    not define, and feedback=True before compute_controller(); none of them touches any state.  K = 0 does nothing."""
    import multidronesim_b200 as mds
    from multidronesim_b200.control import dlqr
    E, N = 2, 2
    env, dl, ts = make_setup(E, N, torch.float64)
    with pytest.raises(TypeError):
        mds.TorqueLearningRollout(env, ts, dlqr.DecentralizedLQROmega(env, [mds.model.LinearizedOmegaModel(env) for _ in range(N)]))
    with pytest.raises(TypeError):
        mds.TorqueLearningRollout(env, ts, mds.control.LQROmegaController(env, mds.model.LinearizedOmegaModel(env), mds.control.ThrustOmegaController(env)))
    with pytest.raises(_lib.MdsError, match="TorqueLearningRollout"):
        mds.LearningRollout(env, ts, dl)
    ro = mds.TorqueLearningRollout(env, ts, dl)
    good = torch.zeros(3, E, N, 4, device="cuda", dtype=torch.float64)
    th0, P0, obs0 = dl.theta_planes.clone(), dl.P_planes.clone(), env.obs.clone()
    with pytest.raises(ValueError):
        ro.run(good, method="theta_update2")              # the torque model defines theta_update and approx_theta_update
    with pytest.raises(ValueError):
        ro.run(torch.zeros(3, E, N + 1, 4, device="cuda", dtype=torch.float64))
    with pytest.raises(ValueError):
        ro.run(torch.zeros(3, E * N, 4, device="cuda", dtype=torch.float64))
    with pytest.raises(_lib.MdsError):
        ro.run(good.float())
    with pytest.raises(_lib.MdsError):
        ro.run(good.cpu())
    with pytest.raises(TypeError):
        ro.run(good.cpu().numpy())
    with pytest.raises(TypeError):
        ro.run(good, method="approx_theta_update", project=False)   # the 12-dim approx_theta_update takes no options
    with pytest.raises(_lib.MdsError, match="compute_controller"):
        ro.run(good, feedback=True)
    torch.cuda.synchronize()
    assert env.step_counter == 0 and ro.t == 0.0
    assert torch.equal(dl.theta_planes, th0) and torch.equal(dl.P_planes, P0) and torch.equal(env.obs, obs0)
    ro.run(torch.zeros(0, E, N, 4, device="cuda", dtype=torch.float64))   # K = 0: nothing happens
    assert env.step_counter == 0 and ro.t == 0.0 and torch.equal(dl.theta_planes, th0) and torch.equal(env.obs, obs0)


def cfg(m=12, target=0, project=1, dpe=2, code=1, dt=1 / 240):
    """an MdsRlsCfg with every theta_code entry set to `code`"""
    c = _lib.RlsCfg()
    c.m, c.target, c.predict_from_xtp1, c.normalize_gain, c.project, c.drones_per_env, c.dt = m, target, 0, 1, project, dpe, dt
    for k in range(16 * 12):
        c.theta_code[k] = code
    return c


def test_torque_c_argument_errors_do_not_need_a_gpu(lib_built):
    """mds_learning_rollout_torque validates every argument before it launches anything (the non-null dummy pointers are
    never touched); every message starts with "learning_rollout_torque: "."""
    from multidronesim_b200.constants import DroneConstants
    prm = DroneConstants().c_params()
    p = ctypes.c_void_p(64)
    st = _lib.State(64, 64, 64, 64, 64)

    def call(c, K=4, E=3, N=2, null=False, gain=None, coupled=0, every=0, log=p, fn=lib_built.mds_learning_rollout_torque_f32):
        q = None if null else p
        return fn(prm, c, 0, every, st, q, q, p, gain, coupled, p, p, None, p, None, log, 0.0, K, E, N, None)

    f64 = lib_built.mds_learning_rollout_torque_f64
    cases = [
        (dict(c=cfg(), null=True), b"null pointer"),
        (dict(c=cfg(m=9)), b"m must be 12"),
        (dict(c=cfg(m=10), fn=f64), b"m must be 12"),
        (dict(c=cfg(target=2)), b"unknown target"),
        (dict(c=cfg(project=0)), b"project must be AFTER"),
        (dict(c=cfg(project=0), gain=p, fn=f64), b"project must be AFTER"),
        (dict(c=cfg(project=3)), b"unknown projection mode"),
        (dict(c=cfg(), coupled=1), b"coupled law needs a gain"),
        (dict(c=cfg(project=2), coupled=1, K=0, fn=f64), b"coupled law needs a gain"),
        (dict(c=cfg(dpe=3)), b"drones_per_env"),
        (dict(c=cfg(dt=0.0)), b"dt must be positive"),
        (dict(c=cfg(), K=-1), b"bad K, E or N"),
        (dict(c=cfg(), E=0, fn=f64), b"bad K, E or N"),
        (dict(c=cfg(dpe=0), N=0), b"bad K, E or N"),
        (dict(c=cfg(dpe=33), N=33, fn=f64), b"bad K, E or N"),
        (dict(c=cfg(code=3)), b"theta_code"),
        (dict(c=cfg(), every=1, log=None), b"obs_log buffer missing"),
    ]
    for kw, msg in cases:
        rc = call(**kw)
        e = lib_built.mds_last_error()
        assert rc == -1 and e.startswith(b"learning_rollout_torque: ") and msg in e, (kw, e)
    assert call(cfg(), K=0) == 0  # K = 0: nothing to do
    assert call(cfg(project=2), K=0, gain=p, coupled=1, fn=f64) == 0
    # an empty input tensor has no storage: K = 0 takes a NULL inputs pointer, K > 0 does not
    assert lib_built.mds_learning_rollout_torque_f64(prm, cfg(), 0, 0, st, p, p, None, None, 0, p, p, None, p, None, None, 0.0, 0, 3, 2, None) == 0
    rc = lib_built.mds_learning_rollout_torque_f64(prm, cfg(), 0, 0, st, p, p, None, None, 0, p, p, None, p, None, None, 0.0, 1, 3, 2, None)
    assert rc == -1 and b"null pointer" in lib_built.mds_last_error()
