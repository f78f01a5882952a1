"""GPU parity of the CBF stage: device rows vs the REFERENCE's dense G, h (fixtures), device QP vs the
oracle solver on the same rows (CBF-filtered actions within 1e-4, BASELINE.json north_star), per-env
status flags and the nominal fallback."""
import numpy as np
import pytest
import torch

from helpers import scaled_err
from oracle.qp import kkt_residuals, solve_qp

pytestmark = pytest.mark.gpu
CASES = [("o2_n2_obs1", 2, 2), ("o2_n8_obs1", 2, 8), ("o3_n7_obs0", 3, 7), ("o3_n8_obs1", 3, 8), ("o3_n4_obs3", 3, 4)]


def setup(golden, name, order, N, dtype):
    import multidronesim_b200 as mds
    g = golden["cbf_rows"]
    obs, xdes, obst, unom = g[f"{name}_obs"], g[f"{name}_xdes"], g[f"{name}_obstacles"], g[f"{name}_unom"]
    E = obs.shape[0]
    env = mds.BatchedCtrlAviary(drone_model=mds.DroneModel.CF2P, num_drones=N, num_envs=E, dtype=dtype)
    Mdl = mds.model.LinearizedOmegaModel if order == 2 else mds.model.LinearizedYankOmegaModel
    poles = np.array([-2.2, -2.4]) if order == 2 else np.array([-3.0, -3.6, -5.6])
    rs, zs = (0.1, 1.0) if order == 2 else (0.125, 2.0)
    cbf = mds.cbf.DroneCBF(env, [Mdl(env) for _ in range(N)], safety_radius=rs, zscale=zs, order=order, cbf_poles=poles)
    trk = mds.cbf.DroneQPTracker(cbf, order=order, num_robots=N, xdim=cbf.xdim, env=env)
    dev = lambda a: torch.as_tensor(a, device="cuda", dtype=dtype).contiguous()
    return g, env, cbf, trk, dev(obs), dev(xdes), (dev(obst) if len(obst) else None), dev(unom)


@pytest.mark.parametrize("dtype", [torch.float64, torch.float32])
@pytest.mark.parametrize("name,order,N", CASES)
def test_rows_match_reference(golden, name, order, N, dtype, lib_built):
    g, env, cbf, trk, obs, xdes, obst, unom = setup(golden, name, order, N, dtype)
    assert np.allclose(cbf.Kcbf, g[f"{name}_Kcbf"], rtol=1e-12) and np.allclose(cbf.umax, g[f"{name}_umax"], rtol=1e-12)
    G, h = cbf.build_ineq_const(obs, xdes, obst)
    Gr, hr = g[f"{name}_G"], g[f"{name}_h"]
    assert tuple(G.shape) == Gr.shape and tuple(h.shape) == hr.shape
    tol = 1e-9 if dtype == torch.float64 else 2e-5
    G, h = G.double().cpu().numpy(), h.double().cpu().numpy()
    # row-wise: each row against its own magnitude (rows span 1e-3 .. 1e3)
    gs = 1.0 + np.max(np.abs(Gr), axis=2, keepdims=True)
    assert np.max(np.abs(G - Gr) / gs) < tol
    # rhs sums terms of mixed sign: compare against the size of its summands (|h| + K0 * Ds^4 scale)
    assert np.max(np.abs(h - hr) / (1.0 + np.abs(hr))) < (tol if dtype == torch.float64 else 5e-4)


@pytest.mark.parametrize("name,order,N", CASES)
def test_qp_matches_oracle_fp64(golden, name, order, N, lib_built):
    g, env, cbf, trk, obs, xdes, obst, unom = setup(golden, name, order, N, torch.float64)
    u = trk.compute_control(obs, xdes, unom, x_obs=obst).cpu().numpy()
    st = trk.status.cpu().numpy()
    n_solved = 0
    for e in range(obs.shape[0]):
        Gr, hr, un = g[f"{name}_G"][e], g[f"{name}_h"][e], g[f"{name}_unom"][e]
        uo, lam, so, _ = solve_qp(np.eye(4 * N), -un.reshape(-1), Gr, hr)
        if so == 0:
            assert st[e] == 0, (e, int(st[e]))        # the oracle solved it: the device must not fall back to the nominal input
            assert np.max(np.abs(u[e].reshape(-1) - uo)) < 1e-7 * (1 + np.max(np.abs(uo))), e
            n_solved += 1
        elif so == 1:
            assert st[e] != 0, e                      # infeasible must never be reported optimal
        if st[e] != 0:
            assert np.array_equal(u[e], un), e        # nominal fallback (cbf/qptracker.py:30-34)
        else:
            # independent certificate: the device answer is primal feasible and no worse than the oracle's optimum
            x = u[e].reshape(-1)
            assert np.max(Gr @ x - hr) < 1e-7 * (1 + np.max(np.abs(hr)))
            if so == 0:
                assert 0.5 * np.sum((x - un.reshape(-1)) ** 2) <= 0.5 * np.sum((uo - un.reshape(-1)) ** 2) + 1e-7
    assert n_solved >= 2


@pytest.mark.parametrize("name,order,N", CASES)
def test_qp_fp32_within_1e4(golden, name, order, N, lib_built):
    g, env, cbf, trk, obs, xdes, obst, unom = setup(golden, name, order, N, torch.float32)
    u = trk.compute_control(obs, xdes, unom, x_obs=obst).double().cpu().numpy()
    st = trk.status.cpu().numpy()
    checked = 0
    for e in range(obs.shape[0]):
        Gr, hr, un = g[f"{name}_G"][e], g[f"{name}_h"][e], g[f"{name}_unom"][e]
        uo, lam, so, _ = solve_qp(np.eye(4 * N), -un.reshape(-1), Gr, hr)
        if so == 0:
            assert st[e] == 0, (e, int(st[e]))
            # north_star: "CBF-filtered actions must agree to 1e-4": absolute, every column (yank O(1), rates up to 10 rad/s)
            err = np.abs(u[e] - uo.reshape(N, 4))
            assert np.max(err) < 1e-4, (e, np.max(err))
            checked += 1
        if st[e] != 0:
            assert np.allclose(u[e], un.astype(np.float32))
    assert checked >= 2


def test_anchor_and_status_codes(lib_built):
    """SURVEY App. C anchor (u_safe[0,0] = -0.113260464) + an infeasible env + an untouched env."""
    import multidronesim_b200 as mds
    for dtype, tol in ((torch.float64, 1e-8), (torch.float32, 1e-5)):
        env = mds.BatchedCtrlAviary(drone_model=mds.DroneModel.CF2P, num_drones=2, num_envs=3, pyb_freq=100, ctrl_freq=100, dtype=dtype)
        cbf = mds.cbf.DroneCBF(env, [mds.model.LinearizedOmegaModel(env) for _ in range(2)], safety_radius=.1, zscale=1)
        trk = mds.cbf.DroneQPTracker(cbf, num_robots=2)
        obs = torch.zeros(3, 2, 20, device="cuda", dtype=dtype)
        obs[..., 6] = 1.0
        obs[..., 16:20] = env.HOVER_RPM
        obs[0, 0, 0:3] = torch.tensor([0, 0, .75]); obs[0, 0, 12] = -.8
        obs[0, 1, 0:3] = torch.tensor([1, 1, 1.5])
        obs[1, 0, 0:3] = torch.tensor([0, 0, .53])                            # at rest deep inside the safety zone: needs u > umax
        obs[1, 1, 0:3] = torch.tensor([1, 1, 1.5])
        obs[2, 0, 0:3] = torch.tensor([2, 0, 1.0]); obs[2, 1, 0:3] = torch.tensor([-2, 0, 1.5])
        xdes = torch.zeros(3, 2, 9, device="cuda", dtype=dtype)
        xdes[..., 6:9] = obs[..., 0:3]
        unom = torch.zeros(3, 2, 4, device="cuda", dtype=dtype)
        unom[0, 0, 0] = -0.2
        unom[2, 1, 1] = 3.0
        x_obs = np.array([np.array([[0, 0, .5], np.zeros(3)])])
        u = trk.compute_control(obs, xdes, unom, x_obs=x_obs, obs_r_list=[.1])
        assert abs(float(u[0, 0, 0]) - (-0.113260464)) < tol and float(u[0].abs().sum()) == pytest.approx(0.113260464, abs=tol)
        assert trk.status.tolist() == [0, 1, 0] and int(trk.iters[0]) >= 1 and int(trk.iters[2]) == 0
        assert torch.equal(u[1], unom[1]) and torch.equal(u[2], unom[2])
        with pytest.raises(IndexError):  # N_obs > N is refused like the reference (IndexError, quirk B14) unless opted in
            trk.compute_control(obs, xdes, unom, x_obs=torch.zeros(3, 4, device="cuda", dtype=dtype))


@pytest.mark.parametrize("order,dtype,tol", [(2, torch.float64, 1e-9), (3, torch.float64, 1e-9), (3, torch.float32, 1e-4)])
def test_cylinder_obstacles_vs_oracle(golden, order, dtype, tol, lib_built, tmp_path):
    """Builder extension (the reference has spheres only; parity unpinned): a sphere and a vertical cylinder
    (obstacles.Cylinder -> negative radius) in one obstacle set; device rows and QP answers against oracle/cbf.py."""
    import multidronesim_b200 as mds
    from multidronesim_b200.obstacles import Cylinder, Sphere
    from oracle import cbf as ocbf
    from oracle import conversions as cv
    from oracle.aviary import OracleCtrlAviary
    from oracle.constants import DroneModel as ODM, Physics as OPH
    name, N = ("o2_n8_obs1", 8) if order == 2 else ("o3_n8_obs1", 8)
    g, env, cbf, trk, obs, xdes, _, unom = setup(golden, name, order, N, dtype)
    prims = [Sphere((0.0, 0.0, 0.5), 0.1), Cylinder((0.4, -0.3, 0.0), 0.15, height=3.0)]
    obst = torch.tensor([p.as_row() for p in prims], device="cuda", dtype=dtype)
    Gd, hd = cbf.build_ineq_const(obs, xdes, obst)
    u = trk.compute_control(obs, xdes, unom, x_obs=obst).double().cpu().numpy()
    st = trk.status.cpu().numpy()
    oenv = OracleCtrlAviary(ODM.CF2P, N, physics=OPH.DYN)
    prm = ocbf.CbfParams(oenv, order, 1.0 if order == 2 else 2.0, 0.1 if order == 2 else 0.125, (-2.2, -2.4) if order == 2 else (-3.0, -3.6, -5.6))
    obs_h, xdes_h, unom_h = g[f"{name}_obs"], g[f"{name}_xdes"], g[f"{name}_unom"]
    solved = 0
    for e in range(obs_h.shape[0]):
        x = np.array([cv.obs_to_lin_model(obs_h[e, i], prm.xdim, oenv) for i in range(N)])
        Gr, hr = ocbf.build_ineq(prm, x, xdes_h[e], [np.array(p.center) for p in prims], [p.as_row()[3] for p in prims])
        assert scaled_err(Gd[e].double().cpu().numpy(), Gr) < max(tol, 1e-5 if dtype == torch.float32 else 0)
        assert scaled_err(hd[e].double().cpu().numpy(), hr) < max(tol, 1e-5 if dtype == torch.float32 else 0)
        uo, _, so, _ = solve_qp(np.eye(4 * N), -unom_h[e].reshape(-1), Gr, hr)
        if so == 0:
            assert st[e] == 0, (e, int(st[e]))
            err = np.abs(u[e] - uo.reshape(N, 4))
            assert np.max(err) < max(tol, 1e-8) * (1.0 if dtype == torch.float32 else 1 + np.max(np.abs(uo))), (e, np.max(err))
            solved += 1
    assert solved >= (1 if order == 2 else 2)   # order-2 rows vanish at ez = 0: most random order-2 cases are infeasible
    import os
    from multidronesim_b200.obstacles import generate_cylinder
    path = generate_cylinder(0.15, 3.0, folder=str(tmp_path))
    assert os.path.isfile(path) and 'cylinder radius="0.15" length="3.0"' in open(path).read()


@pytest.mark.parametrize("N,n_obs,order", [(5, 2, 3), (16, 1, 3), (32, 2, 3), (3, 0, 2), (1, 1, 3), (6, 3, 2),
                                           (2, 5, 3), (1, 3, 2), (4, 8, 3)])  # the last three: more obstacles than drones (SURVEY 8f-4 extension)
def test_qp_other_group_sizes_vs_oracle(N, n_obs, order, lib_built):
    """Lane-group sizes other than the swarm's 8 (NP = 1, 4, 8 with idle lanes, 16, 32; odd N has no 'diameter' slot):
    dense rows and QP answers in fp64 against oracle/cbf.py + oracle/qp.py on random states."""
    import multidronesim_b200 as mds
    from oracle import cbf as ocbf
    from oracle import conversions as cv
    from oracle.aviary import OracleCtrlAviary
    from oracle.constants import DroneModel as ODM, Physics as OPH
    from scipy.spatial.transform import Rotation
    E, dtype = 9, torch.float64
    rng = np.random.default_rng(100 + N)
    env = mds.BatchedCtrlAviary(drone_model=mds.DroneModel.CF2P, num_drones=N, num_envs=E, dtype=dtype)
    Mdl = mds.model.LinearizedOmegaModel if order == 2 else mds.model.LinearizedYankOmegaModel
    poles = np.array([-2.2, -2.4]) if order == 2 else np.array([-3.0, -3.6, -5.6])
    rs, zs = (0.1, 1.0) if order == 2 else (0.125, 2.0)
    extra = n_obs > N
    cbf = mds.cbf.DroneCBF(env, [Mdl(env) for _ in range(N)], safety_radius=rs, zscale=zs, order=order, cbf_poles=poles, allow_extra_obstacles=extra)
    trk = mds.cbf.DroneQPTracker(cbf, order=order, num_robots=N, xdim=cbf.xdim, env=env)
    if extra:  # without the opt-in the host mirror refuses like the reference's builder does (cbf/cbf.py:388)
        strict = mds.cbf.DroneCBF(env, [Mdl(env) for _ in range(N)], safety_radius=rs, zscale=zs, order=order, cbf_poles=poles)
        with pytest.raises(IndexError):
            strict.check_obstacle_count(n_obs)
    oenv = OracleCtrlAviary(ODM.CF2P, N, physics=OPH.DYN)
    prm = ocbf.CbfParams(oenv, order, zs, rs, tuple(poles))
    spread = 0.6 * N ** (1 / 3)
    rpy = rng.uniform(-0.3, 0.3, (E, N, 3))
    obs = np.concatenate([rng.uniform(-spread, spread, (E, N, 3)), Rotation.from_euler("xyz", rpy.reshape(-1, 3)).as_quat().reshape(E, N, 4), rpy,
                          rng.normal(0, 0.5, (E, N, 3)), rng.normal(0, 0.5, (E, N, 3)), rng.uniform(12000, 17000, (E, N, 4))], axis=-1)
    xdes = np.zeros((E, N, cbf.xdim))
    xdes[..., -3:] = obs[..., 0:3] + rng.normal(0, 0.2, (E, N, 3))
    if order == 3:
        xdes[..., 3] = oenv.M * oenv.G
    unom = rng.normal(0, 1.0, (E, N, 4)) * np.array([0.5, 2.0, 2.0, 2.0])
    obst = np.concatenate([rng.uniform(-spread, spread, (n_obs, 3)), rng.uniform(0.05, 0.2, (n_obs, 1))], axis=1) if n_obs else None
    dev = lambda a: None if a is None else torch.as_tensor(a, device="cuda", dtype=dtype).contiguous()
    Gd, hd = cbf.build_ineq_const(dev(obs), dev(xdes), dev(obst))
    u = trk.compute_control(dev(obs), dev(xdes), dev(unom), x_obs=dev(obst)).cpu().numpy()
    st, solved = trk.status.cpu().numpy(), 0
    for e in range(E):
        x = np.array([cv.obs_to_lin_model(obs[e, i], prm.xdim, oenv) for i in range(N)])
        Gr, hr = ocbf.build_ineq(prm, x, xdes[e], None if obst is None else [o[:3] for o in obst], None if obst is None else [o[3] for o in obst],
                                 allow_extra_obstacles=extra)
        assert scaled_err(Gd[e].cpu().numpy(), Gr) < 1e-9 and scaled_err(hd[e].cpu().numpy(), hr) < 1e-9
        uo, _, so, _ = solve_qp(np.eye(4 * N), -unom[e].reshape(-1), Gr, hr)
        if so == 0:
            assert st[e] == 0, (e, int(st[e]))
            assert np.max(np.abs(u[e].reshape(-1) - uo)) < 1e-7 * (1 + np.max(np.abs(uo))), (e, np.max(np.abs(u[e].reshape(-1) - uo)))
            solved += 1
        elif so == 1:
            assert st[e] != 0
        if st[e] != 0:
            assert np.array_equal(u[e], unom[e])
    assert solved >= (1 if order == 2 else 3), (solved, st.tolist())


def dense_case(N, n_obs, order, E, seed):
    """Random dense swarm (positions in a cube of half-width 0.6 N^(1/3)): many barrier rows active at once."""
    from oracle import cbf as ocbf
    from oracle.aviary import OracleCtrlAviary
    from oracle.constants import DroneModel as ODM, Physics as OPH
    from scipy.spatial.transform import Rotation
    rng = np.random.default_rng(seed)
    oenv = OracleCtrlAviary(ODM.CF2P, N, physics=OPH.DYN)
    poles = (-2.2, -2.4) if order == 2 else (-3.0, -3.6, -5.6)
    rs, zs = (0.1, 1.0) if order == 2 else (0.125, 2.0)
    prm = ocbf.CbfParams(oenv, order, zs, rs, poles)
    spread = 0.6 * N ** (1 / 3)
    rpy = rng.uniform(-0.3, 0.3, (E, N, 3))
    obs = np.concatenate([rng.uniform(-spread, spread, (E, N, 3)), Rotation.from_euler("xyz", rpy.reshape(-1, 3)).as_quat().reshape(E, N, 4), rpy,
                          rng.normal(0, 0.5, (E, N, 3)), rng.normal(0, 0.5, (E, N, 3)), rng.uniform(12000, 17000, (E, N, 4))], axis=-1)
    xdes = np.zeros((E, N, prm.xdim))
    xdes[..., -3:] = obs[..., 0:3] + rng.normal(0, 0.2, (E, N, 3))
    if order == 3:
        xdes[..., 3] = oenv.M * oenv.G
    unom = rng.normal(0, 1.0, (E, N, 4)) * np.array([0.5, 2.0, 2.0, 2.0])
    obst = np.concatenate([rng.uniform(-spread, spread, (n_obs, 3)), rng.uniform(0.05, 0.2, (n_obs, 1))], axis=1) if n_obs else None
    return oenv, prm, poles, rs, zs, obs, xdes, unom, obst


@pytest.mark.parametrize("dtype", [torch.float64, torch.float32])
@pytest.mark.parametrize("N,n_obs,min_active", [(8, 1, 7), (16, 1, 13), (32, 2, 25)])
def test_dense_swarms_never_fall_back(N, n_obs, min_active, dtype, lib_built):
    """The hole VERDICT r1 names: 'oracle solved, device gave up'.  Dense random swarms whose optimal active sets exceed the
    12 slots of the in-shared-memory solver (up to 34 at N = 32): the device must report OPTIMAL wherever the oracle does and
    return the same minimiser (fp64 1e-7 relative, fp32 1e-4 absolute), through the scratch solver where needed."""
    import multidronesim_b200 as mds
    from oracle import cbf as ocbf
    from oracle import conversions as cv
    E, order = 24, 3
    oenv, prm, poles, rs, zs, obs, xdes, unom, obst = dense_case(N, n_obs, order, E, 100 + N)
    env = mds.BatchedCtrlAviary(drone_model=mds.DroneModel.CF2P, num_drones=N, num_envs=E, dtype=dtype)
    cbf = mds.cbf.DroneCBF(env, [mds.model.LinearizedYankOmegaModel(env) for _ in range(N)], safety_radius=rs, zscale=zs, order=order,
                           cbf_poles=np.array(poles))
    trk = mds.cbf.DroneQPTracker(cbf, order=order, num_robots=N, xdim=cbf.xdim, env=env)
    dev = lambda a: None if a is None else torch.as_tensor(a, device="cuda", dtype=dtype).contiguous()
    # Solver parity: both solvers get the SAME problem data.  fp64: the oracle's own rows (the device rows equal them to 1e-9,
    # test_qp_other_group_sizes_vs_oracle).  fp32: the rows the device built in fp32 (mds_cbf_rows, the same row code as the QP
    # kernel) -- a row error of 1e-6 moves the minimiser by 1e-6 / |a|, which is the rows' conditioning, not the solver's.
    Gd, hd = cbf.build_ineq_const(dev(obs), dev(xdes), dev(obst))
    Gd, hd = Gd.double().cpu().numpy(), hd.double().cpu().numpy()
    u = trk.compute_control(dev(obs), dev(xdes), dev(unom), x_obs=dev(obst)).double().cpu().numpy()
    st, it = trk.status.cpu().numpy(), trk.iters.cpu().numpy()
    unom_seen = unom if dtype == torch.float64 else unom.astype(np.float32).astype(np.float64)
    n_opt, most_active, worst, worst_e2e = 0, 0, 0.0, 0.0
    for e in range(E):
        x = np.array([cv.obs_to_lin_model(obs[e, i], prm.xdim, oenv) for i in range(N)])
        Gr, hr = ocbf.build_ineq(prm, x, xdes[e], [o[:3] for o in obst], [o[3] for o in obst])
        if dtype == torch.float64:
            assert scaled_err(Gd[e], Gr) < 1e-9 and scaled_err(hd[e], hr) < 1e-9
        ue, _, se, _ = solve_qp(np.eye(4 * N), -unom[e].reshape(-1), Gr, hr)          # fp64 data end to end
        uo, lam, so, _ = solve_qp(np.eye(4 * N), -unom_seen[e].reshape(-1), Gd[e], hd[e])  # the device's data
        if so == 0:
            assert st[e] == 0, (e, int(st[e]), int(it[e]), int((lam > 0).sum()))
            err = np.max(np.abs(u[e].reshape(-1) - uo))
            worst = max(worst, err)
            assert err < (1e-7 * (1 + np.max(np.abs(uo))) if dtype == torch.float64 else 1e-4), (e, err, int((lam > 0).sum()))
            n_opt += 1
            most_active = max(most_active, int((lam > 0).sum()))
            if se == 0:
                worst_e2e = max(worst_e2e, float(np.max(np.abs(u[e].reshape(-1) - ue))))
        elif so == 1:
            assert st[e] != 0, e
    print(f"dense N={N} {dtype}: solver parity {worst:.2e}, vs fp64 rows end to end {worst_e2e:.2e}, largest active set {most_active}")
    assert worst_e2e < (1e-6 if dtype == torch.float64 else 5e-3)
    assert n_opt >= E // 2 and most_active >= min_active, (n_opt, most_active)


def test_do_state_bounds_false(lib_built):
    """CBF(do_state_bounds=False) (cbf/cbf.py:473-476): no force-bound rows -- 2 N fewer rows, and the 4th input is
    clamped by the +-umax box alone."""
    import multidronesim_b200 as mds
    from oracle import cbf as ocbf
    from oracle import conversions as cv
    N, E, order, dtype = 4, 6, 3, torch.float64
    oenv, prm, poles, rs, zs, obs, xdes, unom, obst = dense_case(N, 1, order, E, 7)
    unom[..., 3] = np.linspace(-12, 12, E * N).reshape(E, N)  # beyond both the box (10) and the force-bound interval
    env = mds.BatchedCtrlAviary(drone_model=mds.DroneModel.CF2P, num_drones=N, num_envs=E, dtype=dtype)
    dev = lambda a: torch.as_tensor(a, device="cuda", dtype=dtype).contiguous()
    outs = {}
    for flag in (True, False):
        cbf = mds.cbf.DroneCBF(env, [mds.model.LinearizedYankOmegaModel(env) for _ in range(N)], safety_radius=rs, zscale=zs, order=order,
                               cbf_poles=np.array(poles))
        cbf.do_state_bounds = flag
        trk = mds.cbf.DroneQPTracker(cbf, order=order, num_robots=N, xdim=cbf.xdim, env=env)
        G, h = cbf.build_ineq_const(dev(obs), dev(xdes), dev(obst))
        assert G.shape[1] == N * (N - 1) // 2 + 8 * N + (2 * N if flag else 0) + N
        u = trk.compute_control(dev(obs), dev(xdes), dev(unom), x_obs=dev(obst)).cpu().numpy()
        st = trk.status.cpu().numpy()
        for e in range(E):
            x = np.array([cv.obs_to_lin_model(obs[e, i], prm.xdim, oenv) for i in range(N)])
            Gr, hr = ocbf.build_ineq(prm, x, xdes[e], [o[:3] for o in obst], [o[3] for o in obst], do_state_bounds=flag)
            assert scaled_err(G[e].cpu().numpy(), Gr) < 1e-9 and scaled_err(h[e].cpu().numpy(), hr) < 1e-9
            uo, _, so, _ = solve_qp(np.eye(4 * N), -unom[e].reshape(-1), Gr, hr)
            if so == 0:
                assert st[e] == 0 and np.max(np.abs(u[e].reshape(-1) - uo)) < 1e-7 * (1 + np.max(np.abs(uo))), (flag, e)
        outs[flag] = u
    assert np.max(np.abs(outs[True][..., 3] - outs[False][..., 3])) > 1e-3   # the force-bound rows do bind in this case


def test_iteration_cap_only_where_the_oracle_has_no_solution(lib_built):
    """From its start at rest the C5 swarm meets QPs the reference cannot solve either (cbf/qptracker.py:30-34 falls back to the
    nominal input); in a 21 003-environment swarm a handful of those end at the device's iteration cap instead of a proof of
    infeasibility (statistics qp_iter_cap = 7 of 126 018 environment-steps, every launch plan).  Both outcomes return the nominal
    input -- what matters is the converse (VERDICT r1): a QP the ORACLE solves must never end at the cap.  The per-call path
    exposes the per-environment status; every capped environment-step is re-solved here by the oracle on the device's own rows."""
    import multidronesim_b200 as mds
    from multidronesim_b200 import scenarios
    E, K = 21003, 6
    sw = scenarios.cbf_swarm(E, 8, order=3)
    env, trk, cbf, trajs = sw["env"], sw["tracker"], sw["cbf"], sw["trajs"]
    pipe = mds.PerCallPipeline(env, sw["ctrl"], trk, sw["obstacles"])
    obst = pipe.obst
    n_cap = n_inf = 0
    for k in range(K):
        ref = trajs.eval(k * env.CTRL_TIMESTEP)
        obs_before = env.obs.clone()
        pipe.step(ref)
        st = trk.status.cpu().numpy()
        n_inf += int((st == 1).sum())
        capped = np.nonzero(st == 2)[0]
        n_cap += len(capped)
        if len(capped) == 0:
            continue
        idx = torch.as_tensor(capped, device="cuda")
        # the nominal input the QP saw: recompute it for the capped environments from the observation the step started from
        env_obs = obs_before[idx].contiguous()
        sub = scenarios.cbf_swarm(len(capped), 8, order=3)   # same parameters; state and reference overwritten below
        sub["env"].obs.copy_(env_obs)
        sub["ctrl"].set_reference(ref.reshape(E, 8, -1)[idx].reshape(-1, ref.shape[-1]).contiguous())
        _, u = sub["ctrl"].compute(sub["env"].obs, skip_low_level=True)
        sp = mds.PerCallPipeline(sub["env"], sub["ctrl"], sub["tracker"], sw["obstacles"])
        mds._lib.call("mds_cbf_prepare", sub["env"].dtype, sub["env"]._prm, 3, sp.mg, mds._lib.ptr(sub["ctrl"]._ref_view), mds._lib.ptr(u), mds._lib.ptr(sp.xdes),
                      sub["env"].NUM_TOTAL, mds._lib.stream_ptr(sub["env"].device))
        G, h = sub["cbf"].build_ineq_const(sub["env"].obs, sp.xdes, obst)
        G, h, un = G.double().cpu().numpy(), h.double().cpu().numpy(), u.double().cpu().numpy().reshape(len(capped), -1)
        us = sub["tracker"].compute_control(sub["env"].obs, sp.xdes, u, x_obs=obst)
        assert (sub["tracker"].status.cpu().numpy() == 2).all()   # the sub-swarm reproduces the capped QPs
        for j in range(len(capped)):
            _, _, so, _ = solve_qp(np.eye(32), -un[j], G[j], h[j])
            assert so != 0, (k, int(capped[j]), "the oracle solves a QP the device gave up on")
    print(f"start-up of {E} envs x {K} steps: {n_inf} infeasible, {n_cap} at the iteration cap, none of them solvable by the oracle")
    assert n_inf > 0
