"""LearningRollout / mds_learning_rollout: the decentralised-LQR learning loop (excitation -> inner loop -> physics -> RLS)
for K steps in one launch against the per-call loop over mds_error_state, mds_lowlevel, mds_physics_step and
mds_rls_update, and against the oracle.  The C-argument refusals run without a GPU."""
import ctypes

import numpy as np
import pytest
import torch

from multidronesim_b200 import _lib

gpu = pytest.mark.gpu

# (class, method, method kwargs, E, N, physics, wind, lemniscate)
CASES = {
    "omega_theta_update": ("DecentralizedLQROmega", "theta_update", {}, 3, 2, "DYN", False, False),
    "omega_theta_update2": ("DecentralizedLQROmega", "theta_update2", {}, 5, 3, "DYN_GND_DRAG_DW", False, False),
    "yank_theta_update": ("DecentralizedLQRYankOmega", "theta_update", {}, 4, 2, "DYN_GND_DRAG_DW", True, False),
    "yo_theta_update": ("DecentralizedYOLQRCrazyflie", "theta_update", {}, 7, 3, "DYN", False, True),
    "yo_approx_project": ("DecentralizedYOLQRCrazyflie", "approx_theta_update", {"project": True}, 6, 3, "DYN_GND_DRAG_DW", False, False),
    "yo_approx_noproject": ("DecentralizedYOLQRCrazyflie", "approx_theta_update", {"project": False}, 3, 2, "DYN", False, False),
}


def make_setup(cls_name, E, N, dtype, physics="DYN", wind=False, lemniscate=False, seed=0):
    """env, controller, TrajectorySet and the initial positions, the same for every dtype (seeded)"""
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
    model = mds.model.LinearizedOmegaModel if cls_name == "DecentralizedLQROmega" else mds.model.LinearizedYankOmegaModel
    models = [model(env) for _ in range(N)]
    dl = dlqr.DecentralizedYOLQRCrazyflie(env, models, np.eye(10), np.eye(4)) if cls_name == "DecentralizedYOLQRCrazyflie" else getattr(dlqr, cls_name)(env, models)
    ts = mds.trajectories.TrajectorySet(trajs, dtype=dtype)
    return env, dl, ts


def excitation(K, E, N, seed=1):
    """sigma1-like draws [K, E, N, 4] (float64 numpy): thrust in [0.7, 1.5] m g, body-rate targets in +-0.2"""
    from oracle.constants import drone_params
    mg = drone_params("cf2p", 240, 240).M * 9.8
    rng = np.random.default_rng(seed)
    return np.concatenate([rng.uniform(0.7 * mg, 1.5 * mg, (K, E, N, 1)), rng.uniform(-0.2, 0.2, (K, E, N, 3))], axis=-1)


def percall_loop(env, dl, ts, us, method, learn_from, t0=0.0, **kw):
    obs = env.obs
    for k in range(us.shape[0]):
        dl.set_reference(ts.eval(t0 + k * env.CTRL_TIMESTEP))
        e_t = dl.error_state(obs).clone()
        phis = torch.cat([e_t, us[k]], dim=-1)
        obs = env.step(dl.compute_low_level(us[k], obs))[0]
        e_tp1 = dl.error_state(obs).clone()
        if k >= learn_from:
            getattr(dl, method)(phis, e_tp1, **kw)
    return obs


def outputs(env, dl):
    """the quantities the loop leaves behind, float64 numpy"""
    f = lambda t: t.detach().double().cpu().numpy().copy()
    return {"theta": f(dl.theta), "P": f(dl.P), "obs": f(env.obs)[..., :16], "pid_a": f(dl.low_level._a), "pid_b": f(dl.low_level._b),
            "resid": f(dl.resid), "state": np.concatenate([f(env._pos_wx), f(env._quat), f(env._vel_wy), f(env._wz)[:, None]], axis=1)}


def run_both(cls_name, method, kw, E, N, dtype, physics, wind, lemniscate, K, learn_from, seed=0):
    import multidronesim_b200 as mds
    us_np = excitation(K, E, N, seed + 1)
    res = {}
    for mode in ("percall", "fused"):
        env, dl, ts = make_setup(cls_name, E, N, dtype, physics, wind, lemniscate, seed)
        us = torch.as_tensor(us_np, device="cuda", dtype=dtype).contiguous()
        if mode == "percall":
            percall_loop(env, dl, ts, us, method, learn_from, **kw)
        else:
            ro = mds.LearningRollout(env, ts, dl)
            ro.run(us, method=method, learn_from=learn_from, **kw)
            assert env.step_counter == K * env.PYB_STEPS_PER_CTRL and abs(ro.t - K * env.CTRL_TIMESTEP) < 1e-15
        torch.cuda.synchronize()
        res[mode] = outputs(env, dl)
    return res


def err(a, b):
    return float(np.abs(a - b).max()) / max(1.0, float(np.abs(b).max()))


def check_fp64(got, want, what):
    for k in ("theta", "P", "obs", "pid_a", "pid_b", "resid"):
        assert err(got[k], want[k]) <= 1e-9, (what, k, err(got[k], want[k]))


def check_fp32(fused32, percall32, percall64, what):
    for k in ("theta", "P", "obs", "pid_a", "pid_b", "resid"):
        e_fused, e_call = err(fused32[k], percall64[k]), err(percall32[k], percall64[k])
        assert e_fused <= max(2 * e_call, 2e-4), (what, k, e_fused, e_call)


@gpu
@pytest.mark.parametrize("tag", list(CASES))
def test_parity_with_percall_loop(tag, lib_built):
    """Every (class, method) row, K = 40, learn_from = 1: fp64 to 1e-9 of each quantity's scale; fp32 no further from the
    per-call fp64 run than twice the per-call fp32 run (or 2e-4 of the scale)."""
    cls_name, method, kw, E, N, physics, wind, lem = CASES[tag]
    r64 = run_both(cls_name, method, kw, E, N, torch.float64, physics, wind, lem, 40, 1)
    check_fp64(r64["fused"], r64["percall"], tag)
    assert err(r64["percall"]["theta"], make_prior(cls_name, E, N)) > 1e-6  # the models moved
    r32 = run_both(cls_name, method, kw, E, N, torch.float32, physics, wind, lem, 40, 1)
    check_fp32(r32["fused"], r32["percall"], r64["percall"], tag)


def make_prior(cls_name, E, N):
    _, dl, _ = make_setup(cls_name, E, N, torch.float64)
    return dl.theta.cpu().numpy()


@gpu
@pytest.mark.parametrize("dtype", [torch.float64, torch.float32])
@pytest.mark.parametrize("E,N", [(37, 1), (7, 5), (3, 32)])
def test_odd_sizes(E, N, dtype, lib_built):
    """E not a multiple of the environments per block; N = 32 in fp64 takes more than 48 KB of shared memory per block."""
    physics = "DYN_GND_DRAG_DW" if N > 1 else "DYN"
    r = run_both("DecentralizedLQRYankOmega", "theta_update", {}, E, N, dtype, physics, False, False, 16, 1, seed=3)
    if dtype == torch.float64:
        check_fp64(r["fused"], r["percall"], (E, N))
    else:
        r64 = run_both("DecentralizedLQRYankOmega", "theta_update", {}, E, N, torch.float64, physics, False, False, 16, 1, seed=3)
        check_fp32(r["fused"], r["percall"], r64["percall"], (E, N))


@gpu
def test_learning_loop_vs_oracle(lib_built):
    """The scenario of test_gpu_dlqr.py::test_learning_loop_vs_oracle (warm-up loop of simulations/CBFTestOrd3.py:153-198) in
    ONE fused call against the oracle loop (aviary + controllers + sysid), fp64, with that test's thresholds."""
    import multidronesim_b200 as mds
    import multidronesim_b200.trajectories as T
    from oracle import controllers as oc
    from oracle import sysid
    from oracle.aviary import OracleCtrlAviary
    from oracle.constants import DroneModel as ODM, Physics as OPH
    E, N, steps, dtype = 3, 2, 40, torch.float64
    rng = np.random.default_rng(21)
    init = rng.uniform(-0.5, 0.5, (E, N, 3)) + np.array([0, 0, 1.0])
    env = mds.BatchedCtrlAviary(drone_model=mds.DroneModel.CF2P, num_drones=N, num_envs=E, dtype=dtype, initial_xyzs=init, physics=mds.Physics.DYN)
    dl = mds.control.DecentralizedLQROmega(env, [mds.model.LinearizedOmegaModel(env) for _ in range(N)])
    ts = mds.trajectories.TrajectorySet([T.WaitTrajectory(init[e, j], 1000.0) for e in range(E) for j in range(N)], dtype=dtype)
    mg = env.M * env.G
    us = np.concatenate([rng.uniform(0.7 * mg, 1.5 * mg, (steps, E, N, 1)), rng.uniform(-0.2, 0.2, (steps, E, N, 3))], axis=-1)
    oenvs = [OracleCtrlAviary(ODM.CF2P, N, initial_xyzs=init[e], physics=OPH.DYN) for e in range(E)]
    octl = [[oc.Lqr(oenvs[e], "omega9", low_level=oc.ThrustOmegaPid(oenvs[e]), K=np.zeros((4, 9))) for _ in range(N)] for e in range(E)]
    th = dl.theta.cpu().numpy().copy().reshape(E, N, 13, 9)
    P = dl.P.cpu().numpy().copy().reshape(E, N, 13, 13)
    oobs = [o.reset()[0] for o in oenvs]
    obs = mds.LearningRollout(env, ts, dl).run(torch.as_tensor(us, device="cuda", dtype=dtype).contiguous(), learn_from=1)
    for i in range(steps):
        for e in range(E):
            ophis, act = [], np.zeros((N, 4))
            for j in range(N):
                c = octl[e][j]
                c.set_desired_trajectory(j, init[e, j], np.zeros(3), np.zeros(3), 0.0, 0.0)
                ophis.append(np.hstack([c.error_state(oobs[e][j]), us[i, e, j]]))
                act[j] = c.compute_low_level(us[i, e, j].copy(), oobs[e][j])
            oobs[e] = oenvs[e].step(act)[0]
            if i != 0:
                for j in range(N):
                    th[e, j], P[e, j], _ = sysid.rls_update(th[e, j], P[e, j], ophis[j], octl[e][j].error_state(oobs[e][j]), env.CTRL_TIMESTEP,
                                                            sysid.TARGET_PREDICT, True, True)
    got_th = dl.theta.cpu().numpy().reshape(E, N, 13, 9)
    got_P = dl.P.cpu().numpy().reshape(E, N, 13, 13)
    assert np.abs(obs.cpu().numpy() - np.array(oobs))[..., :16].max() < 1e-8
    assert np.abs(got_th - th).max() <= 1e-8 * np.abs(th).max(), np.abs(got_th - th).max()
    assert np.abs(got_P - P).max() <= 1e-8 * np.abs(P).max()
    prior = np.hstack([mds.model.LinearizedOmegaModel(env).Ahat, mds.model.LinearizedOmegaModel(env).Bhat]).T
    assert np.abs(th - prior).max() > 1e-3


@gpu
@pytest.mark.parametrize("dtype", [torch.float64, torch.float32])
def test_split_calls_are_bit_identical(dtype, lib_built):
    """run(K) == run(K1) + run(K - K1), bit for bit, with hover references (state, PID state, theta, P)."""
    import multidronesim_b200 as mds
    E, N, K, K1 = 5, 3, 30, 11
    us = torch.as_tensor(excitation(K, E, N, 7), device="cuda", dtype=dtype).contiguous()
    res = []
    for parts in ((K,), (K1, K - K1)):
        env, dl, ts = make_setup("DecentralizedYOLQRCrazyflie", E, N, dtype, "DYN_GND_DRAG_DW", seed=5)
        ro = mds.LearningRollout(env, ts, dl)
        k0 = 0
        for p in parts:
            ro.run(us[k0:k0 + p], method="approx_theta_update")
            k0 += p
        res.append(outputs(env, dl))
    for k in ("theta", "P", "obs", "pid_a", "pid_b", "state"):
        assert np.array_equal(res[0][k], res[1][k]), k


@gpu
@pytest.mark.parametrize("dtype", [torch.float64, torch.float32])
def test_no_learning_leaves_the_model_alone(dtype, lib_built):
    """learn_from >= K: theta and P come back bit-identical; the open-loop flight equals that of learn_from = 0 bit for bit."""
    import multidronesim_b200 as mds
    E, N, K = 4, 3, 20
    us = torch.as_tensor(excitation(K, E, N, 9), device="cuda", dtype=dtype).contiguous()
    res = []
    for learn_from in (K, 0):
        env, dl, ts = make_setup("DecentralizedLQROmega", E, N, dtype, "DYN_GND_DRAG_DW", wind=True, seed=2)
        th0, P0 = dl.theta_planes.clone(), dl.P_planes.clone()
        mds.LearningRollout(env, ts, dl).run(us, learn_from=learn_from)
        if learn_from == K:
            assert torch.equal(dl.theta_planes, th0) and torch.equal(dl.P_planes, P0)
        else:
            assert not torch.equal(dl.theta_planes, th0)
        res.append(outputs(env, dl))
    for k in ("obs", "pid_a", "pid_b", "state"):
        assert np.array_equal(res[0][k], res[1][k]), k


@gpu
def test_refusals(lib_built):
    """LearningRollout refuses, before any launch, what the kernel does not run."""
    import multidronesim_b200 as mds
    from multidronesim_b200.control import dlqr
    E, N = 2, 2
    env, dl, ts = make_setup("DecentralizedLQRYankOmega", E, N, torch.float64)
    with pytest.raises(_lib.MdsError):
        mds.LearningRollout(env, ts, dlqr.DecentralizedLQR(env, [mds.model.LinearizedModel(env) for _ in range(N)]))
    with pytest.raises(TypeError):
        mds.LearningRollout(env, ts, mds.control.LQROmegaController(env, mds.model.LinearizedOmegaModel(env), mds.control.ThrustOmegaController(env)))
    ro = mds.LearningRollout(env, ts, dl)
    good = torch.zeros(3, E, N, 4, device="cuda", dtype=torch.float64)
    th0 = dl.theta_planes.clone()
    with pytest.raises(ValueError):
        ro.run(good, method="theta_update2")            # the yank-omega variant defines theta_update only
    with pytest.raises(ValueError):
        ro.run(good, method="approx_theta_update")
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
        ro.run(good, method="theta_update", project=False)   # theta_update takes no options, as the per-call method
    assert env.step_counter == 0 and ro.t == 0.0 and torch.equal(dl.theta_planes, th0)
    obs0 = env.obs.clone()
    ro.run(torch.zeros(0, E, N, 4, device="cuda", dtype=torch.float64))   # K = 0: nothing happens
    assert env.step_counter == 0 and ro.t == 0.0 and torch.equal(dl.theta_planes, th0) and torch.equal(env.obs, obs0)
    yo_env, yo, yo_ts = make_setup("DecentralizedYOLQRCrazyflie", E, N, torch.float64)
    with pytest.raises(TypeError):
        mds.LearningRollout(yo_env, yo_ts, yo).run(good, method="approx_theta_update", projekt=False)


@gpu
@pytest.mark.parametrize("dtype", [torch.float64, torch.float32])
def test_obs_log_matches_percall_steps(dtype, lib_built):
    """obs_log / log_every: slot j holds the observation after step (j + 1) * log_every, as the per-call loop saw it (K = 20,
    log_every = 3: six slots, the last two steps unlogged)."""
    import multidronesim_b200 as mds
    E, N, K, every = 5, 3, 20, 3
    us = torch.as_tensor(excitation(K, E, N, 11), device="cuda", dtype=dtype).contiguous()
    env, dl, ts = make_setup("DecentralizedLQROmega", E, N, dtype, "DYN_GND_DRAG_DW", seed=4)
    want = []
    obs = env.obs
    for k in range(K):  # the per-call loop, keeping every step's observation
        dl.set_reference(ts.eval(k * env.CTRL_TIMESTEP))
        e_t = dl.error_state(obs).clone()
        phis = torch.cat([e_t, us[k]], dim=-1)
        obs = env.step(dl.compute_low_level(us[k], obs))[0]
        dl.theta_update(phis, dl.error_state(obs).clone())
        want.append(obs.double().cpu().numpy().copy())
    env2, dl2, ts2 = make_setup("DecentralizedLQROmega", E, N, dtype, "DYN_GND_DRAG_DW", seed=4)
    log = torch.full((K // every + 1, E, N, _lib.OBS_DIM), -7.0, device="cuda", dtype=dtype)  # one spare slot: must stay untouched
    last = mds.LearningRollout(env2, ts2, dl2).run(us, obs_log=log, log_every=every)
    got = log.double().cpu().numpy()
    tol = 1e-9 if dtype == torch.float64 else 2e-4
    for j in range(K // every):
        w = want[(j + 1) * every - 1][..., :16]
        assert np.abs(got[j][..., :16] - w).max() <= tol * max(1.0, np.abs(w).max()), j
    assert (got[K // every] == -7.0).all()
    assert np.abs(last.double().cpu().numpy()[..., :16] - want[-1][..., :16]).max() <= tol * max(1.0, np.abs(want[-1][..., :16]).max())


def cfg(m=9, target=0, project=0, dpe=2, code=1, dt=1 / 48):
    """an MdsRlsCfg with every theta_code entry set to `code`"""
    c = _lib.RlsCfg()
    c.m, c.target, c.predict_from_xtp1, c.normalize_gain, c.project, c.drones_per_env, c.dt = m, target, 1, 1, project, dpe, dt
    for k in range(16 * 12):
        c.theta_code[k] = code
    return c


def test_c_argument_errors_do_not_need_a_gpu(lib_built):
    """mds_learning_rollout validates every argument before it launches anything (non-null dummy pointers are never touched)."""
    from multidronesim_b200.constants import DroneConstants
    prm = DroneConstants().c_params()
    p = ctypes.c_void_p(64)
    st, pid = _lib.State(64, 64, 64, 64, 64), _lib.PidState(64, 64)

    def call(c, variant=_lib.CTRL_LQR_OMEGA, K=4, E=3, N=2, null=False, fn=lib_built.mds_learning_rollout_f32):
        q = None if null else p
        return fn(prm, c, variant, 0, 0, st, pid, q, q, q, q, q, None, q, None, None, 0.0, K, E, N, None)

    cases = [
        (dict(c=cfg(), null=True), b"null pointer"),
        (dict(c=cfg(), variant=_lib.CTRL_LQR_TORQUE), b"variant"),
        (dict(c=cfg(), variant=_lib.CTRL_GEOMETRIC), b"variant"),
        (dict(c=cfg(m=10)), b"m must be 9 with LQR_OMEGA"),
        (dict(c=cfg(m=9), variant=_lib.CTRL_LQR_YANK), b"m must be 9 with LQR_OMEGA"),
        (dict(c=cfg(m=12), variant=_lib.CTRL_LQR_YANK), b"m must be 9 with LQR_OMEGA"),
        (dict(c=cfg(target=1)), b"est_x_dot"),
        (dict(c=cfg(project=1)), b"project_theta is defined for m = 10 only"),   # the m = 9 kernel carries no projection
        (dict(c=cfg(project=2), fn=lib_built.mds_learning_rollout_f64), b"project_theta is defined for m = 10 only"),
        (dict(c=cfg(), K=-1), b"bad K, E or N"),
        (dict(c=cfg(dpe=3)), b"drones_per_env"),
        (dict(c=cfg(dpe=0), N=0), b"bad K, E or N"),
        (dict(c=cfg(dpe=33), N=33), b"bad K, E or N"),
        (dict(c=cfg(), E=0), b"bad K, E or N"),
        (dict(c=cfg(code=3)), b"theta_code"),
        (dict(c=cfg(m=10, code=3, project=2), variant=_lib.CTRL_LQR_YANK, fn=lib_built.mds_learning_rollout_f64), b"theta_code"),
    ]
    for kw, msg in cases:
        rc = call(**kw)
        assert rc == -1 and msg in lib_built.mds_last_error(), (kw, lib_built.mds_last_error())
    c = cfg()
    assert lib_built.mds_learning_rollout_f64(prm, c, _lib.CTRL_LQR_OMEGA, 0, 0, st, pid, p, p, p, p, p, None, p, None, None, 0.0, 0, 3, 2, None) == 0  # K = 0: nothing to do
    # an empty excitation has no storage: K = 0 takes a NULL inputs pointer, K > 0 does not
    assert lib_built.mds_learning_rollout_f32(prm, c, _lib.CTRL_LQR_OMEGA, 0, 0, st, pid, p, p, None, p, p, None, p, None, None, 0.0, 0, 3, 2, None) == 0
    rc = lib_built.mds_learning_rollout_f32(prm, c, _lib.CTRL_LQR_OMEGA, 0, 0, st, pid, p, p, None, p, p, None, p, None, None, 0.0, 1, 3, 2, None)
    assert rc == -1 and b"null pointer" in lib_built.mds_last_error()


def test_rls_update_c_argument_errors_do_not_need_a_gpu(lib_built):
    """mds_rls_update refuses a bad configuration or argument before it launches anything (the dummy pointers are never touched)."""
    p = ctypes.c_void_p(64)

    def call(c, D=6, null=False, fn=lib_built.mds_rls_update_f32):
        return fn(c, None if null else p, p, p, p, None, D, None)

    cases = [
        (dict(c=cfg(), null=True), b"bad argument"),
        (dict(c=cfg(), D=0), b"bad argument"),
        (dict(c=cfg(m=11)), b"m must be 9, 10 or 12"),
        (dict(c=cfg(target=2), fn=lib_built.mds_rls_update_f64), b"unknown target"),
        (dict(c=cfg(m=9, target=1)), b"est_x_dot"),
        (dict(c=cfg(m=10, project=3)), b"unknown projection mode"),
        (dict(c=cfg(m=12, project=-1), fn=lib_built.mds_rls_update_f64), b"unknown projection mode"),
        (dict(c=cfg(dt=0.0)), b"dt and drones_per_env must be positive"),
        (dict(c=cfg(dt=-1 / 48), fn=lib_built.mds_rls_update_f64), b"dt and drones_per_env must be positive"),
        (dict(c=cfg(dpe=0)), b"dt and drones_per_env must be positive"),
        (dict(c=cfg(m=10, target=1, project=2, code=3)), b"theta_code"),
        (dict(c=cfg(m=12, code=3), fn=lib_built.mds_rls_update_f64), b"theta_code"),
    ]
    for kw, msg in cases:
        rc = call(**kw)
        err = lib_built.mds_last_error()
        assert rc == -1 and err.startswith(b"rls_update: ") and msg in err, (kw, err)
