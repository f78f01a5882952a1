"""CPU: self-tests of the restated env step (oracle/aviary.py) against closed-form cases.  The upstream
simulator is absent (parity unpinned), so these pin the restatement to physics instead."""
import math

import numpy as np
import pytest

from oracle.aviary import OracleCtrlAviary, integrate_q, quat_to_matrix, quat_to_rpy, rpy_to_quat
from oracle.constants import DroneModel, Physics, drone_params


def test_constants():
    p = drone_params("cf2p")
    assert abs(p.HOVER_RPM - 14468.429) < 1e-3 and abs(p.MAX_RPM - 21702.64) < 1e-2 and abs(p.MAX_THRUST - 0.59535) < 1e-5
    assert np.allclose(np.diag(p.J), [2.3951e-5, 2.3951e-5, 3.2347e-5])      # utils/graph_fedce.py:45-47
    assert p.G == 9.8 and p.M == 0.027 and p.KF == 3.16e-10 and p.KM == 7.94e-12


def test_free_fall_semi_implicit_euler():
    env = OracleCtrlAviary(DroneModel.CF2P, 1, initial_xyzs=[[0, 0, 10.0]], physics=Physics.DYN)
    n, dt = 100, 1 / 240
    for _ in range(n):
        obs = env.step(np.zeros((1, 4)))[0]
    # v_k = -g k dt ; z_k = z0 - g dt^2 k(k+1)/2
    assert abs(obs[0, 12] + 9.8 * n * dt) < 1e-12 and abs(obs[0, 2] - (10.0 - 9.8 * dt * dt * n * (n + 1) / 2)) < 1e-12


def test_hover_is_stationary_and_obs_layout():
    env = OracleCtrlAviary(DroneModel.CF2X, 2, initial_xyzs=[[0, 0, 1.0], [1, 0, 1.0]], physics=Physics.DYN)
    for _ in range(240):
        obs, r, term, trunc, info = env.step(np.full((2, 4), env.HOVER_RPM))
    assert np.allclose(obs[:, 0:3], [[0, 0, 1.0], [1, 0, 1.0]], atol=1e-9) and np.allclose(obs[:, 3:7], [0, 0, 0, 1])
    assert np.allclose(obs[:, 16:20], env.HOVER_RPM) and obs.shape == (2, 20)
    assert (r, term, trunc, info) == (-1, False, False, {"answer": 42})


def test_pure_yaw_spin_and_world_rates():
    env = OracleCtrlAviary(DroneModel.CF2P, 1, initial_xyzs=[[0, 0, 1.0]], physics=Physics.DYN)
    env.set_state([[0, 0, 1.0]], [rpy_to_quat([0.3, 0.0, 0.0])], [[0, 0, 0]], [[0, 0, 2.0]])
    q0 = env.quat[0].copy()
    obs = env.step(np.full((1, 4), env.HOVER_RPM))[0]
    assert np.allclose(env.quat[0], integrate_q(q0, env.rpy_rates[0], 1 / 240))
    assert abs(np.linalg.norm(env.quat[0]) - 1) < 1e-14
    assert np.allclose(obs[0, 13:16], quat_to_matrix(q0) @ env.rpy_rates[0])   # world rates = R(old) w(new)


def test_euler_roundtrip_and_clip():
    for rpy in ([0.1, -0.2, 0.3], [1.0, 0.5, -2.5], [0, 0, 0]):
        assert np.allclose(quat_to_rpy(rpy_to_quat(rpy)), rpy, atol=1e-12)
    env = OracleCtrlAviary(DroneModel.CF2P, 1, physics=Physics.DYN)
    obs = env.step(np.array([[-5.0, 1e9, 100.0, env.MAX_RPM]]))[0]
    assert np.allclose(obs[0, 16:20], [0, env.MAX_RPM, 100.0, env.MAX_RPM])


def test_composite_effects_have_the_right_sign():
    prm = dict(physics=Physics.DYN_GND_DRAG_DW)
    low = OracleCtrlAviary(DroneModel.CF2P, 1, initial_xyzs=[[0, 0, 0.05]], **prm)
    high = OracleCtrlAviary(DroneModel.CF2P, 1, initial_xyzs=[[0, 0, 5.0]], **prm)
    a = np.full((1, 4), low.HOVER_RPM)
    assert low.step(a)[0][0, 12] > high.step(a)[0][0, 12] >= -1e-9            # ground effect adds lift near the floor
    pair = OracleCtrlAviary(DroneModel.CF2P, 2, initial_xyzs=[[0, 0, 1.0], [0, 0, 1.4]], **prm)
    o = pair.step(np.full((2, 4), pair.HOVER_RPM))[0]
    assert o[0, 12] < -1e-3 and abs(o[1, 12]) < 1e-4                           # downwash acts on the lower drone only
    drag = OracleCtrlAviary(DroneModel.CF2P, 1, initial_xyzs=[[0, 0, 5.0]], **prm)
    drag.set_state([[0, 0, 5.0]], [[0, 0, 0, 1]], [[1.0, 0, 0]], [[0, 0, 0]], [[drag.HOVER_RPM] * 4])
    assert drag.step(np.full((1, 4), drag.HOVER_RPM))[0][0, 10] < 1.0         # drag opposes velocity
    floor = OracleCtrlAviary(DroneModel.CF2P, 1, initial_xyzs=[[0, 0, 0.02]], **prm)
    for _ in range(60):
        o = floor.step(np.zeros((1, 4)))[0]
    assert o[0, 2] == floor.Z_FLOOR and o[0, 12] == 0.0                         # contact clamp
    dyn = OracleCtrlAviary(DroneModel.CF2P, 1, initial_xyzs=[[0, 0, 0.02]], physics=Physics.DYN)
    for _ in range(60):
        o = dyn.step(np.zeros((1, 4)))[0]
    assert o[0, 2] < 0                                                          # upstream DYN has no ground


def test_dslpid_hover_config1():
    """config C1: 2 CF2X drones under the (halved-gain) DSL PID climb 1 m and hold, 240 Hz, DYN."""
    from oracle.controllers import DslPid
    init = np.array([[1.0, 0, 0], [-1.0, 0, 0]])
    env = OracleCtrlAviary(DroneModel.CF2X, 2, initial_xyzs=init, physics=Physics.DYN)
    ctrls = [DslPid(env, gain_scale=0.5) for _ in range(2)]
    obs = env.step(np.zeros((2, 4)))[0]
    target = init + np.array([0, 0, 1.0])
    for _ in range(240 * 6):
        act = np.array([ctrls[j].compute_from_state(env.CTRL_TIMESTEP, obs[j], target[j])[0] for j in range(2)])
        obs = env.step(act)[0]
    assert np.max(np.abs(obs[:, 0:3] - target)) < 0.05


def test_cf2x_needs_the_x_frame_mixer():
    """SURVEY 8f-4: the reference's input_to_action is PLUS-frame whatever the model (utils/model_conversions.py:74-77).  On a
    CF2X under the DYN dynamics its roll / pitch torques land 45 degrees off the body axes and the geometric controller
    loses the drone; with ``x_frame_mixer=True`` (builder extension) the mixer inverts the allocation the dynamics apply."""
    from oracle import conversions as cv
    from oracle import pipeline as opl
    from oracle import trajectories as otj
    from oracle.aviary import OracleCtrlAviary
    from oracle.constants import DroneModel as ODM, Physics as OPH
    kw = dict(r=1.0, v=0.5, center=np.array([0, 0, 1.0]), yaw_rate=0.0)
    end = {}
    for xf in (True, False):
        o = OracleCtrlAviary(ODM.CF2X, 1, initial_xyzs=otj.Circle(**kw)(0.0)[0][None], physics=OPH.DYN_GND_DRAG_DW, x_frame_mixer=xf)
        if xf:  # the mixer is the exact inverse of the CF2X allocation of the dynamics
            u = np.array([o.M * o.G * 1.1, 2e-4, -1.5e-4, 3e-5])
            rpm = cv.input_to_action(o, u.copy())
            f, l2 = o.KF * rpm ** 2, o.L / np.sqrt(2.0)
            tau = [o.cf2x_torque_sign * (f[0] + f[1] - f[2] - f[3]) * l2, (-f[0] + f[1] + f[2] - f[3]) * l2, o.KM * (-rpm[0] ** 2 + rpm[1] ** 2 - rpm[2] ** 2 + rpm[3] ** 2)]
            assert abs(f.sum() - u[0]) < 1e-15 and np.abs(np.array(tau) - u[1:]).max() < 1e-15
            assert np.abs(cv.action_to_input(o, rpm) - u).max() < 1e-15
        log, _ = opl.run_tracking(o, [otj.Circle(**kw)], "geometric", 480)
        end[xf] = float(np.abs(log[-1, 0, 0:3] - otj.Circle(**kw)(479 / 240)[0]).max())
    assert end[True] < 0.1 and end[False] > 1.0, end


# ---------------------------------------------------------------------------------------------------------------
# What the reference tree DOES hold about the env step: its continuous rigid-body model (model/dynamics.py:83-106) and its
# hover linearisation (model/linearized.py:52-79).  Upstream's explicit DYN update (restated in oracle/aviary.py from the
# published algorithm; gym-pybullet-drones itself is absent) must be a first-order integrator OF that model: its difference
# quotients converge to dynamics() as dt -> 0, and their Jacobian at hover is (A, B).  What the reference's model
# computes comes from tests/golden/models.npz (oracle/make_golden.golden_models, run on the reference's own classes).
# ---------------------------------------------------------------------------------------------------------------
def _fd_xdot(model, pos, quat, vel, w_body, rpm, dt_hz, J=None):
    """((v_new - v) / dt, (w_new - w) / dt, (p_new - p) / dt, R(q_new), R(q)) of ONE explicit Physics.DYN update at 1 / dt_hz,
    with the inertia ``J`` in place of the drone model's if given"""
    from oracle.aviary import quat_to_matrix
    env = OracleCtrlAviary(model, 1, physics=Physics.DYN, pyb_freq=dt_hz, ctrl_freq=dt_hz)
    if J is not None:
        env.J, env.J_INV = np.array(J, float), np.linalg.inv(J)
    env.set_state(pos, quat, vel, w_body, last_rpm=rpm)
    R0 = quat_to_matrix(env.quat[0])
    env.step(np.asarray(rpm, float).reshape(1, 4))
    dt = 1.0 / dt_hz
    return (env.vel[0] - vel) / dt, (env.rpy_rates[0] - w_body) / dt, (env.pos[0] - pos) / dt, quat_to_matrix(env.quat[0]), R0


@pytest.mark.parametrize("model", [DroneModel.CF2P])
def test_dyn_step_converges_to_the_reference_dynamics(golden, model):
    """(state(t + dt) - state(t)) / dt of the restated Physics.DYN step -> QuadrotorDynamics.dynamics (model/dynamics.py:83-106,
    inputs from the reference's own action_to_input) as dt -> 0: first-order convergence at the 128 stored random states, to
    1e-6 relative at dt = 1e-7 s.  The stored xdot was computed with the inertia load_env_params leaves in place (the Hummingbird's,
    quirk B22), so the env step runs with that inertia here."""
    g = golden["models"]
    J = np.diag(g["J_dynamics"])
    for k, (o, want) in enumerate(zip(g["obs"], g["xdot_nonlinear"])):
        # stored in linear order (w, w_dot, v_dot, x_dot) (utils/model_conversions.py:124-135), with obs[13:16] as the body rates;
        # the DYN update does not depend on position, so every state is lifted 3 m to keep it clear of the ground
        pos, quat, vel, w, rpm = o[0:3] + [0, 0, 3], o[3:7], o[10:13], o[13:16], o[16:20]
        errs = []
        for hz in (1e4, 1e5, 1e6, 1e7):
            vdot, wdot, pdot, R1, R0 = _fd_xdot(model, pos, quat, vel, w, rpm, hz, J=J)
            scale = 1.0 + np.abs(want[3:9]).max()
            e = max(np.abs(vdot - want[6:9]).max(), np.abs(wdot - want[3:6]).max()) / scale
            # position uses the NEW velocity (semi-implicit): p_dot -> v; attitude: (R1 - R0) / dt -> R hat(w)
            e = max(e, np.abs(pdot - want[9:12]).max() / (1 + np.abs(vel).max()))
            Rdot = R0 @ np.array([[0, -w[2], w[1]], [w[2], 0, -w[0]], [-w[1], w[0], 0]])
            e = max(e, np.abs((R1 - R0) * hz - Rdot).max() / (1 + np.abs(Rdot).max()))
            errs.append(e)
        assert errs[-1] < 1e-5, (k, errs)
        assert errs[1] < 0.2 * errs[0] + 1e-9 and errs[2] < 0.2 * errs[1] + 1e-9, (k, errs)   # O(dt)


def test_dyn_step_hover_jacobian_is_the_reference_linear_model(golden):
    """Jacobian of the DYN difference quotient at hover, in the reference's linear-model coordinates x = [rpy, w, v, p],
    u = [f, tau] (utils/model_conversions.py:20-58,69-83), equals LinearizedModel's A and B (model/linearized.py:52-79), as
    stored for the CF2P in tests/golden/models.npz."""
    from scipy.spatial.transform import Rotation
    env = OracleCtrlAviary(DroneModel.CF2P, 1, physics=Physics.DYN)
    A_ref, B_ref = golden["models"]["torque12_A"], golden["models"]["torque12_B"]
    hz, eps = 1e7, 1e-4
    mixer = np.array([[1, 1, 1, 1], [0, env.L, 0, -env.L], [-env.L, 0, env.L, 0], [-env.KM / env.KF, env.KM / env.KF, -env.KM / env.KF, env.KM / env.KF]])

    def xdot(x, u):
        """x = [rpy, w, v, p] -> d/dt of the same 12 coordinates from one tiny DYN step"""
        quat = Rotation.from_euler("xyz", x[0:3]).as_quat()
        thrusts = np.linalg.solve(mixer, u)
        rpm = np.sqrt(np.maximum(thrusts, 0) / env.KF)
        vdot, wdot, pdot, R1, R0 = _fd_xdot(DroneModel.CF2P, x[9:12], quat, x[6:9], x[3:6], rpm, hz)
        rpy1 = Rotation.from_matrix(R1).as_euler("xyz")
        return np.hstack([(rpy1 - x[0:3]) * hz, wdot, vdot, pdot])

    x0 = np.zeros(12); x0[11] = 1.0
    u0 = np.array([env.M * env.G, 0, 0, 0])
    f0 = xdot(x0, u0)
    assert np.abs(f0).max() < 1e-6                                       # hover is an equilibrium
    A = np.array([(xdot(x0 + eps * np.eye(12)[k], u0) - xdot(x0 - eps * np.eye(12)[k], u0)) / (2 * eps) for k in range(12)]).T
    du = np.array([1e-3 * env.M * env.G, 1e-6, 1e-6, 1e-7])
    B = np.array([(xdot(x0, u0 + du[k] * np.eye(4)[k]) - xdot(x0, u0 - du[k] * np.eye(4)[k])) / (2 * du[k]) for k in range(4)]).T
    assert np.abs(A - A_ref).max() < 1e-5 * (1 + np.abs(A_ref).max()), np.abs(A - A_ref).max()
    assert np.abs(B - B_ref).max() < 1e-5 * (1 + np.abs(B_ref).max()), np.abs((B - B_ref) / (1 + np.abs(B_ref))).max()
