"""mds_care_gains_coupled / DecentralizedLQR.compute_controller(solver="device") with the robot-coupled Q of the 12-dim model
(decentralized_lqr.py:44-53): the device gain against the full 12N-state scipy solve of every environment, a structured scipy
reference at N = 32, the reference's own coupled gain, failure reporting, the certainty-equivalence loop against the host
solver, and the refusals (the C-ABI ones, of mds_care_gains too, without a GPU)."""
import ctypes

import numpy as np
import pytest
import scipy.linalg as la
import torch

from multidronesim_b200 import _lib

gpu = pytest.mark.gpu
DTYPES = [torch.float64, torch.float32]
TOL = {torch.float64: 1e-9, torch.float32: 1e-5}  # fp32: K is rounded to fp32 on store; theta is the same fp32 copy on both sides


def make_ctrl(E, N, dtype, cls=None):
    import multidronesim_b200 as mds
    from multidronesim_b200.control import dlqr
    env = mds.BatchedCtrlAviary(drone_model=mds.DroneModel("cf2p"), num_drones=N, num_envs=E, dtype=dtype)
    return (cls or dlqr.DecentralizedLQR)(env, [mds.model.LinearizedModel(env) for _ in range(N)])


def perturbed_theta(c, seed):
    """distinct learned models: the prior scaled entry-wise by 5 % noise, the second half with a dense 0.05 perturbation of A"""
    D, m = c.env.NUM_TOTAL, c.m
    rng = np.random.default_rng(seed)
    th = c.theta.double().cpu().numpy() * (1.0 + 0.05 * rng.normal(size=(D, m + 4, m)))
    th[D // 2:, :m, :] += 0.05 * rng.normal(size=(D - D // 2, m, m))
    return th


def set_theta(c, th):
    c.set_theta(torch.as_tensor(np.ascontiguousarray(th), device="cuda", dtype=c.env.dtype))


def full_gain(c):
    """[E, 4N, mN] from the robot-coupled planes: entry (j, i*m + k, e*N + r) = K_e[4r + i, m j + k]"""
    E, N, m = c.env.NUM_ENVS, c.num_robots, c.m
    planes = c.K_planes.double().cpu().numpy().reshape(N, 4, m, E, N)   # j, i, k, e, r
    return planes.transpose(3, 4, 1, 0, 2).reshape(E, 4 * N, m * N)


def in_structure(N, m=12):
    """[4N, mN] mask of the blocks {0, 1} x {0, 1} and {j} x {j}"""
    mask = np.zeros((4 * N, m * N), bool)
    mask[:8, :2 * m] = True
    for j in range(2, N):
        mask[4 * j:4 * j + 4, m * j:m * j + m] = True
    return mask


def care_gain(A, B, Q, R):
    return la.solve(R, B.T @ la.solve_continuous_are(A, B, Q, R, balanced=True))


@gpu
@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("E,N", [(50, 2), (20, 3), (7, 8)])
def test_coupled_device_vs_full_scipy(E, N, dtype, lib_built):
    """every entry of every environment's [4N, 12N] gain within 1e-9 (fp64) / 1e-5 (fp32) of its max |K| of the full 12N-state
    scipy solve (the host route); exact zeros outside the blocks on the device, within the tolerance of zero on the host"""
    c = make_ctrl(E, N, dtype)
    set_theta(c, perturbed_theta(c, 9 + N))
    K_host = np.array(c.compute_controller(solver="host"))               # [E, 4N, 12N], scipy per environment
    c.K_planes.fill_(7.0)
    K = c.compute_controller(solver="device")
    assert K is c.K_planes and c._coupled and tuple(K.shape) == (N * 48, E * N)
    assert int(c.care_status.sum()) == 0
    K_dev = full_gain(c)
    tol, mask = TOL[dtype], in_structure(N)
    for e in range(E):
        scale = np.abs(K_host[e]).max()
        assert np.abs(K_dev[e] - K_host[e]).max() <= tol * scale, (e, np.abs(K_dev[e] - K_host[e]).max() / scale)
        assert np.all(K_dev[e][~mask] == 0.0)
        assert np.abs(K_host[e][~mask]).max(initial=0.0) <= tol * scale   # the decomposition: the full solve has nothing there
        assert np.abs(K_dev[e][0:4, 12:24]).max() > 1e-4 * scale          # robot 0's gain on robot 1's state: the coupling is real


@gpu
@pytest.mark.parametrize("dtype", DTYPES)
def test_coupled_largest_group(dtype, lib_built):
    """N = 32 (E = 2) against a structured scipy reference: the pair problem of robots 0 and 1 plus 30 single problems"""
    E, N, m = 2, 32, 12
    c = make_ctrl(E, N, dtype)
    th = perturbed_theta(c, 31)
    set_theta(c, th)
    th = c.theta.double().cpu().numpy()   # the Real copy the device reads
    Q, R = c._env_weights()
    Qp, Rp = Q[:2 * m, :2 * m], R[:8, :8]
    c.compute_controller(solver="device")
    assert int(c.care_status.sum()) == 0
    K_dev = full_gain(c)
    for e in range(E):
        blk = th[e * N:(e + 1) * N]
        want = np.zeros((4 * N, m * N))
        A = la.block_diag(blk[0][:m].T, blk[1][:m].T)
        B = la.block_diag(blk[0][m:].T, blk[1][m:].T)
        want[:8, :2 * m] = care_gain(A, B, Qp, Rp)
        for j in range(2, N):
            want[4 * j:4 * j + 4, m * j:m * j + m] = care_gain(blk[j][:m].T, blk[j][m:].T, c.ind_Q, c.ind_R)
        scale = np.abs(want).max()
        assert np.abs(K_dev[e] - want).max() <= TOL[dtype] * scale, (e, np.abs(K_dev[e] - want).max() / scale)
        assert np.all(K_dev[e][~in_structure(N)] == 0.0)


@gpu
@pytest.mark.parametrize("dtype", DTYPES)
def test_coupled_reference_gain(golden, dtype, lib_built):
    """the reference's own coupled gain (tests/golden/dlqr.npz, N = 3) from its theta tiled over four environments"""
    g = golden["dlqr"]
    E, Kg = 4, g["ctrl_torque12_K"]
    c = make_ctrl(E, 3, dtype)
    set_theta(c, np.tile(g["ctrl_torque12_theta"], (E, 1, 1)))
    c.compute_controller(solver="device")
    assert int(c.care_status.sum()) == 0
    K = full_gain(c)
    for e in range(E):
        assert np.allclose(K[e], Kg, rtol=1e-6, atol=1e-8 * np.abs(Kg).max()), e
        assert np.abs(K[e][0:4, 12:24]).max() > 1e-5 * np.abs(Kg).max()   # the cross block is there


@gpu
@pytest.mark.parametrize("dtype", DTYPES)
def test_coupled_failures_are_reported(dtype, lib_built):
    """a zero model (no stabilising solution) for drone 0 of environment 0 flags drones 0 and 1 there and leaves their
    entries alone; a zero model for drone 2 of environment 2 flags that drone only; every other drone solves as before"""
    E, N = 4, 3
    c = make_ctrl(E, N, dtype)
    th = perturbed_theta(c, 4)
    set_theta(c, th)
    c.compute_controller(solver="device")
    K_good = c.K_planes.clone()
    bad = th.copy()
    bad[0] = 0.0
    bad[2 * N + 2] = 0.0
    set_theta(c, bad)
    c.K_planes.fill_(7.0)
    c.compute_controller(solver="device")
    st = c.care_status.cpu().numpy()
    flagged = [0, 1, 2 * N + 2]
    assert st[flagged].tolist() == [1, 1, 1] and st.sum() == 3
    keep = np.setdiff1d(np.arange(E * N), flagged)
    assert bool(torch.all(c.K_planes[:, flagged] == 7.0))
    assert torch.equal(c.K_planes[:, keep], K_good[:, keep])


@gpu
@pytest.mark.parametrize("E,N", [(3, 2), (4, 3)])
def test_certainty_equivalence_on_device(E, N, lib_built):
    """three phases of TorqueLearningRollout.run(feedback=True) with compute_controller(solver="device") before each, against
    the same loop with solver="host", fp64: theta, P, the gain planes, obs and state to 1e-9 of their scale"""
    import multidronesim_b200 as mds
    from test_gpu_learning_torque import err, inputs_for, make_setup, outputs
    K, phases = 30, 3
    us_np = inputs_for("coupled", K * phases, E, N, seed=7)
    res = {}
    for solver in ("host", "device"):
        env, dl, ts = make_setup(E, N, torch.float64, "DYN_GND_DRAG_DW", True, False, "open", seed=6)
        us = torch.as_tensor(us_np, device="cuda", dtype=torch.float64).contiguous()
        ro = mds.TorqueLearningRollout(env, ts, dl)
        prior = dl.theta.double().cpu().numpy().copy()
        for ph in range(phases):
            dl.compute_controller(solver=solver)
            assert dl._coupled
            if solver == "device":
                assert int(dl.care_status.sum()) == 0
            ro.run(us[ph * K:(ph + 1) * K], method="theta_update", learn_from=1, feedback=True)
        torch.cuda.synchronize()
        res[solver] = outputs(env, dl)
        assert err(res[solver]["theta"], prior) > 1e-6   # the models moved
    for k in ("theta", "P", "K", "obs", "state"):
        assert err(res["device"][k], res["host"][k]) <= 1e-9, (k, err(res["device"][k], res["host"][k]))


def _subclass(q_extra=None, ind_q_offdiag=False):
    from multidronesim_b200.control import dlqr

    class Variant(dlqr.DecentralizedLQR):
        def _weights(self):
            Q, R = super()._weights()
            if ind_q_offdiag:
                Q = Q.copy()
                Q[0, 1] = Q[1, 0] = 1.0
            return Q, R

        def _env_weights(self):
            Q, R = super()._env_weights()
            if q_extra is not None:
                q_extra(Q)
            return Q, R
    return Variant


def _couple_1_2(Q):
    Q[12 + 9, 24 + 9] = Q[24 + 9, 12 + 9] = -10.0


def _asymmetric(Q):
    Q[9, 12 + 3] = -10.0


def _inside_a_drone(Q):
    Q[12 + 0, 12 + 1] = Q[12 + 1, 12 + 0] = 1.0


@gpu
@pytest.mark.parametrize("case", ["couple_1_2", "asymmetric", "inside_a_drone", "ind_q_offdiag"])
def test_coupled_refusals(case, lib_built):
    """other couplings raise MdsError before anything runs: K_planes and care_status stay as they were"""
    cls = {"couple_1_2": _subclass(_couple_1_2), "asymmetric": _subclass(_asymmetric), "inside_a_drone": _subclass(_inside_a_drone),
           "ind_q_offdiag": _subclass(ind_q_offdiag=True)}[case]
    c = make_ctrl(2, 3, torch.float64, cls)
    if case != "ind_q_offdiag":
        c.compute_controller(force_diagonal=True, solver="device")   # a care_status to watch
    status = getattr(c, "care_status", None)
    status_before = None if status is None else status.clone()
    K_planes = c.K_planes
    K_before = K_planes.clone()
    with pytest.raises(_lib.MdsError, match="solver='host'"):
        c.compute_controller(solver="device")
    torch.cuda.synchronize()
    assert c.K_planes is K_planes and torch.equal(K_planes, K_before)
    assert getattr(c, "care_status", None) is status
    if status is not None:
        assert torch.equal(status, status_before)


def test_coupled_c_argument_errors_do_not_need_a_gpu(lib_built):
    """mds_care_gains_coupled and mds_care_gains validate every argument before they launch anything (the dummy device
    pointers are never touched); every message starts with "care_gains_coupled: " or "care_gains: "."""
    p = ctypes.c_void_p(64)
    arr = lambda vals: (ctypes.c_double * len(vals))(*vals)
    q = [1 / (np.pi / 10) ** 2] * 2 + [1 / (np.pi / 20) ** 2] + [4.0] * 3 + [1 / .15 ** 2] * 3 + [400.0] * 3
    r = [1.0, 1e6, 1e6, 1e6]
    reference_cross = np.zeros((12, 12))
    reference_cross[9:11, 9:11] = -100.0   # decentralized_lqr.py:44-53: Q[9:11, 21:23] = -1 / 0.1**2
    diag_too_big = np.zeros((12, 12))
    diag_too_big[9, 9] = -400.5            # |q_cross_kk| > q_kk
    block_too_big = np.zeros((12, 12))
    block_too_big[9:11, 9:11] = -250.0     # each entry below q_kk, the 2 x 2 block not
    f32, f64 = lib_built.mds_care_gains_coupled_f32, lib_built.mds_care_gains_coupled_f64

    def call(m=12, qq=q, rr=r, cross=reference_cross, theta=p, K=p, E=3, N=2, fn=f32):
        return fn(m, arr(qq) if qq is not None else None, arr(rr), arr(cross.reshape(-1)) if cross is not None else None, theta, K, None, E, N, None)

    cases = [
        (dict(m=9), b"m must be 12"),
        (dict(m=10, fn=f64), b"m must be 12"),
        (dict(N=1), b"bad E or N"),
        (dict(N=33, fn=f64), b"bad E or N"),
        (dict(E=0), b"bad E or N"),
        (dict(theta=None), b"null pointer"),
        (dict(K=None, fn=f64), b"null pointer"),
        (dict(cross=None), b"null pointer"),
        (dict(qq=None), b"null pointer"),
        (dict(qq=q[:11] + [0.0]), b"Q must be diagonal and positive"),
        (dict(rr=[1.0, 1.0, -1.0, 1.0], fn=f64), b"R must be diagonal and positive"),
        (dict(cross=diag_too_big), b"not positive semidefinite"),
        (dict(cross=block_too_big, fn=f64), b"not positive semidefinite"),
        (dict(cross=np.full((12, 12), np.nan)), b"finite"),
    ]
    for kw, msg in cases:
        rc = call(**kw)
        e = lib_built.mds_last_error()
        assert rc == -1 and e.startswith(b"care_gains_coupled: ") and msg in e, (kw, e)

    g32, g64 = lib_built.mds_care_gains_f32, lib_built.mds_care_gains_f64

    def call_per_drone(m=9, qq=q, rr=r, theta=p, K=p, D=6, fn=g32):
        return fn(m, arr(qq[:m]) if qq is not None else None, arr(rr), theta, K, None, D, None)

    cases = [
        (dict(m=11), b"m must be 9, 10 or 12"),
        (dict(m=13, fn=g64), b"m must be 9, 10 or 12"),
        (dict(m=8, fn=g64), b"m must be 9, 10 or 12"),
        (dict(theta=None), b"bad argument"),
        (dict(K=None, fn=g64), b"bad argument"),
        (dict(qq=None), b"bad argument"),
        (dict(D=0), b"bad argument"),
        (dict(D=-4, fn=g64), b"bad argument"),
        (dict(qq=q[:8] + [0.0]), b"Q must be diagonal and positive"),
        (dict(m=10, qq=q[:9] + [float("nan")], fn=g64), b"Q must be diagonal and positive"),
        (dict(m=12, qq=q[:11] + [-1.0]), b"Q must be diagonal and positive"),
        (dict(rr=[1.0, 0.0, 1.0, 1.0], fn=g64), b"R must be diagonal and positive"),
    ]
    for kw, msg in cases:
        rc = call_per_drone(**kw)
        e = lib_built.mds_last_error()
        assert rc == -1 and e.startswith(b"care_gains: ") and msg in e, (kw, e)
