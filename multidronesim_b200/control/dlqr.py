"""Decentralised LQR with per-drone learned models (reference control/dlqr/decentralized_lqr.py,
decentralized_lqr_omega.py, decentralized_lqr_yank_omega.py, decentralized_yolqr_crazyflie.py), batched on device.

Every drone d carries its own model estimate ``theta_d = [Ahat_d, Bhat_d]^T`` [(m+4), m], its RLS matrix ``P_d``
[(m+4), (m+4)] and its own LQR gain.  The reference stores one block-diagonal theta for the N robots of its single
environment; the blocks never mix in the learning step, hence one small problem per drone here.  The gain is K_d [4, m]
where Q and R are block diagonal (9- and 10-dim variants) and the drone's four rows of the environment's full
[4N, mN] gain where Q couples robots (12-dim variant, decentralized_lqr.py:44-53).  Device layout: PLANES -- entry k of
drone d at ``[k, d]`` -- so that one thread per drone reads and writes coalesced lines (``mds_rls_update``, ``mds_dlqr_ctrl``).

  theta_update / theta_update2 / approx_theta_update : one launch of ``mds_rls_update`` for all E*N drones
  compute                                            : one launch of ``mds_dlqr_ctrl``
  compute_controller                                 : one launch of ``mds_care_gains`` (one warp per drone solves its Riccati
                                                       equation) for diagonal per-drone weights; with ``solver="device"`` the
                                                       robot-coupled 12-dim case through ``mds_care_gains_coupled`` (one warp
                                                       per pair problem of robots 0 and 1, one per other drone); scipy on the
                                                       host, like the reference, for non-diagonal weights and by default for
                                                       the robot-coupled case
"""
from __future__ import annotations

import inspect

import numpy as np
import scipy.linalg as la
import torch

from .. import _lib
from .base_controller import BaseController
from .low_level import ThrustOmegaController, YankOmegaController

RLS_TARGET_PREDICT, RLS_TARGET_XDOT = 0, 1
RLS_PROJECT_NONE, RLS_PROJECT_AFTER, RLS_PROJECT_LOOP = 0, 1, 2


class _DecentralizedBase(BaseController):
    VARIANT = None
    M = None           # model state dimension; n = 4 inputs
    P0_SCALE = 1.0     # initial P = P0_SCALE * I

    def __init__(self, env, lin_models, debug=False):
        super().__init__(env)
        self.m, self.n = self.M, 4
        self.mn = self.m + self.n
        E, N, D = env.NUM_ENVS, env.NUM_DRONES, env.NUM_TOTAL
        if not isinstance(lin_models, (list, tuple)):
            lin_models = [lin_models] * N
        if len(lin_models) != N:
            raise ValueError("lin_models: one linear model per drone of an environment")
        self.lin_models = list(lin_models)
        self.num_robots = N
        self.ind_Q, self.ind_R = self._weights()
        th0 = []
        for agent in self.lin_models:
            if agent.Ahat.shape != (self.m, self.m) or agent.Bhat.shape != (self.m, self.n):
                raise ValueError("linear model dimensions do not match this controller")
            th0.append(np.hstack([agent.Ahat, agent.Bhat]).T)
        th0 = np.stack(th0)                                                     # [N, mn, m]
        planes = np.tile(th0.reshape(N, -1).T, (1, E))                          # [(mn*m), D], d = e*N + n
        self.theta_planes = torch.as_tensor(planes, dtype=env.dtype).to(env.device).contiguous()
        eye = torch.eye(self.mn, dtype=env.dtype, device=env.device).reshape(-1, 1) * self.P0_SCALE
        self.P_planes = eye.repeat(1, D).contiguous()
        self._init_P()
        self.K_planes = torch.zeros(self.n * self.m, D, device=env.device, dtype=env.dtype)
        self.K = None
        self._coupled = False
        self.resid = torch.zeros(D, self.m, device=env.device, dtype=env.dtype)
        self.u = torch.zeros(E, N, 4, device=env.device, dtype=env.dtype)
        self.action = torch.zeros(E, N, 4, device=env.device, dtype=env.dtype)
        self._err = torch.zeros(D, self.m, device=env.device, dtype=env.dtype)
        self.low_level = self._make_low_level()
        self._codes = None

    # ------------------------------------------------------------------ hooks of the variants
    def _weights(self):
        raise NotImplementedError

    def _init_P(self):
        pass

    def _make_low_level(self):
        return None

    def _project_codes(self):
        raise _lib.MdsError("the reference defines project_theta for the 12-dim and the crazyflie 10-dim variants only")

    # ------------------------------------------------------------------ per-drone views
    def _drone(self, i, env_idx=0):
        return env_idx * self.num_robots + i

    def get_thetai(self, i, env_idx=0):
        """[(m+4), m] = [Ahat_i, Bhat_i]^T of robot i in environment env_idx (a copy)."""
        return self.theta_planes[:, self._drone(i, env_idx)].reshape(self.mn, self.m).clone()

    def overwrite_theta(self, theta_new, i, env_idx=0):
        t = torch.as_tensor(np.asarray(theta_new, dtype=np.float64)) if not isinstance(theta_new, torch.Tensor) else theta_new
        self.theta_planes[:, self._drone(i, env_idx)] = t.to(self.theta_planes).reshape(-1)

    @property
    def theta(self):
        """[D, (m+4), m]: every drone's block (the reference's block-diagonal matrix holds the same blocks)."""
        return self.theta_planes.t().reshape(-1, self.mn, self.m)

    @property
    def P(self):
        return self.P_planes.t().reshape(-1, self.mn, self.mn)

    def set_theta(self, theta):
        self.theta_planes.copy_(_lib.require_cuda(theta, "theta", self.env.dtype).reshape(-1, self.mn * self.m).t())

    def set_P(self, P):
        self.P_planes.copy_(_lib.require_cuda(P, "P", self.env.dtype).reshape(-1, self.mn * self.mn).t())

    # ------------------------------------------------------------------ model learning
    # method -> (target, predict_from_xtp1, normalize_gain, project) of its RLS step; the variants fill it in
    RLS_METHODS = {}

    def rls_cfg(self, method, **options):
        """MdsRlsCfg of the RLS step ``method`` defines (the per-call methods and LearningRollout both build it here).
        ``options``: the keyword options the per-call method itself takes, nothing else -- ``project=False``
        (approx_theta_update of the crazyflie variant) is the same step without project_theta."""
        if method not in self.RLS_METHODS:
            raise ValueError(f"{type(self).__name__} defines no RLS method {method!r}; it has {sorted(self.RLS_METHODS)}")
        accepted = [n for n in inspect.signature(getattr(self, method)).parameters if n not in ("phis", "xtp1s")]
        unknown = sorted(set(options) - set(accepted))
        if unknown:
            raise TypeError(f"{type(self).__name__}.{method} takes no option {', '.join(unknown)} (it takes {accepted or 'none'})")
        target, predict_from_xtp1, normalize_gain, proj = self.RLS_METHODS[method]
        if not options.get("project", True):
            proj = RLS_PROJECT_NONE
        env = self.env
        cfg = _lib.RlsCfg()
        cfg.m, cfg.target, cfg.predict_from_xtp1, cfg.normalize_gain = self.m, target, int(predict_from_xtp1), int(normalize_gain)
        cfg.project, cfg.drones_per_env, cfg.dt = proj, env.NUM_DRONES, env.CTRL_TIMESTEP
        codes = self._project_codes() if proj != RLS_PROJECT_NONE else np.ones((self.mn, self.m), dtype=np.uint8)
        for k, v in enumerate(np.asarray(codes, dtype=np.uint8).reshape(-1)):
            cfg.theta_code[k] = int(v)
        return cfg

    def _rls(self, phis, xtp1s, method, **options):
        env = self.env
        D = env.NUM_TOTAL
        phis = _lib.require_cuda(phis, "phis", env.dtype).reshape(D, self.mn)
        xtp1s = _lib.require_cuda(xtp1s, "xtp1s", env.dtype).reshape(D, self.m)
        cfg = self.rls_cfg(method, **options)
        _lib.call("mds_rls_update", env.dtype, cfg, _lib.ptr(phis.contiguous()), _lib.ptr(xtp1s.contiguous()), _lib.ptr(self.theta_planes),
                  _lib.ptr(self.P_planes), _lib.ptr(self.resid), D, _lib.stream_ptr(env.device))
        return self.resid

    def project_theta(self):
        codes = torch.as_tensor(np.asarray(self._project_codes(), dtype=np.int64).reshape(-1, 1), device=self.env.device)
        self.theta_planes.masked_fill_(codes == 0, 0.0)
        self.theta_planes.masked_fill_(codes == 2, 1.0)

    def error_state(self, obs):
        """e [E, N, m] of every drone against the current reference (set_desired_trajectory / set_reference)."""
        env = self.env
        _lib.call("mds_error_state", env.dtype, env._prm, self.VARIANT, _lib.ptr(self._obs(obs)), _lib.ptr(self._ref_view), _lib.ptr(self._err),
                  env.NUM_TOTAL, _lib.stream_ptr(env.device))
        return self._err.view(env.NUM_ENVS, env.NUM_DRONES, self.m)

    # ------------------------------------------------------------------ control
    COUPLED = False    # True: Q couples robots of an environment -> K is a full 4N x mN matrix per environment

    def _env_weights(self):
        """(Q, R) of one whole environment (N robots); block diagonal unless the variant couples robots."""
        N = self.num_robots
        return np.kron(np.eye(N), self.ind_Q), np.kron(np.eye(N), self.ind_R)

    def compute_controller(self, force_diagonal=False, solver="auto"):
        """Gains from the continuous-time Riccati equation of the learned models (decentralized_lqr_omega.py:185-204,
        decentralized_lqr.py:300-317).

        Block-diagonal Q, R (or ``force_diagonal``): one m x m problem per drone, K_d [4, m] -- solved ON DEVICE by
        ``mds_care_gains`` (one warp per drone, matrix sign function in double; <= 2e-12 of scipy's answer) when Q and R are
        diagonal, as all of the reference's Bryson weights are.  ``solver="host"`` forces the reference's own route
        (scipy.linalg.solve_continuous_are per DISTINCT model, ~1 ms each); it is also what non-diagonal weights use.

        The robot-coupled Q of the 12-dim variant with N >= 2 (one mN x mN problem per environment, full K [4N, mN]): by
        default (``"auto"``) and with ``"host"`` scipy solves it per environment and ``self.K`` is the numpy [E, 4N, mN] gain.
        ``solver="device"`` solves it ON DEVICE through ``mds_care_gains_coupled`` when the per-drone Q and R are diagonal and
        the environment's Q is kron(I, Q_d) apart from a cross block between robots 0 and 1 (the reference's weights): the
        stabilising solution is block diagonal over the drones {0, 1}, {2}, ..., {N-1}, so one 24-state problem per
        environment and one 12-state problem per other drone give the whole gain.  ``self.K`` is then ``self.K_planes``, the
        robot-coupled [N][4*m][D] planes (no host copy).  Any other coupling raises MdsError before anything runs.
        ``self.care_status`` [D] (device, int32) after a device solve: 0 ok, 1 no stabilising solution (gain left as it was;
        both drones of a failed pair)."""
        N = self.num_robots
        coupled = bool(self.COUPLED and N >= 2 and not force_diagonal)
        diag_w = np.count_nonzero(self.ind_Q - np.diag(np.diag(self.ind_Q))) == 0 and np.count_nonzero(self.ind_R - np.diag(np.diag(self.ind_R))) == 0
        if solver not in ("auto", "device", "host"):
            raise ValueError("solver must be 'auto', 'device' or 'host'")
        if solver == "device" and coupled:
            cross = self._pair_cross_block() if diag_w else None
            if cross is None:
                raise _lib.MdsError("the device Riccati solver takes diagonal per-drone Q and R, coupled at most through a cross block "
                                    "between robots 0 and 1; use solver='host'")
            return self._compute_controller_device(cross)
        if solver == "device" and not diag_w:
            raise _lib.MdsError("the device Riccati solver takes diagonal, per-drone Q and R; use solver='host'")
        if solver != "host" and not coupled and diag_w:
            return self._compute_controller_device()
        return self._compute_controller_host(force_diagonal)

    def _pair_cross_block(self):
        """C [m, m] when ``_env_weights()`` is (kron(I, ind_Q), kron(I, ind_R)) apart from Q[:m, m:2m] = C and Q[m:2m, :m] = C';
        None for any other coupling."""
        Q, R = self._env_weights()
        N, m = self.num_robots, self.m
        Q0, R0 = np.kron(np.eye(N), self.ind_Q), np.kron(np.eye(N), self.ind_R)
        if Q.shape != Q0.shape or R.shape != R0.shape or not np.array_equal(R, R0):
            return None
        C = np.array(Q[:m, m:2 * m], dtype=np.float64)
        rest = np.array(Q, dtype=np.float64) - Q0
        rest[:m, m:2 * m] -= C
        rest[m:2 * m, :m] -= C.T
        return C if not np.any(rest) else None

    def _compute_controller_device(self, cross=None):
        """One device Riccati solve: per drone (``mds_care_gains``) or, given the pair's cross block ``cross`` [m, m],
        robot-coupled (``mds_care_gains_coupled``).  K_planes and care_status are replaced only after the call succeeds."""
        env = self.env
        E, N, D, m = env.NUM_ENVS, self.num_robots, env.NUM_TOTAL, self.m
        coupled = cross is not None
        rows = (N if coupled else 1) * self.n * m
        K_planes = self.K_planes if self.K_planes.shape[0] == rows else torch.zeros(rows, D, device=env.device, dtype=env.dtype)
        status = getattr(self, "care_status", None)
        if status is None:
            status = torch.zeros(D, device=env.device, dtype=torch.int32)
        q = (_lib.C.c_double * m)(*np.diag(self.ind_Q).tolist())
        r = (_lib.C.c_double * 4)(*np.diag(self.ind_R).tolist())
        theta, K, st, stream = _lib.ptr(self.theta_planes), _lib.ptr(K_planes), _lib.ptr(status), _lib.stream_ptr(env.device)
        if coupled:
            qx = (_lib.C.c_double * (m * m))(*cross.reshape(-1).tolist())
            _lib.call("mds_care_gains_coupled", env.dtype, m, q, r, qx, theta, K, st, E, N, stream)
        else:
            _lib.call("mds_care_gains", env.dtype, m, q, r, theta, K, st, D, stream)
        self.K_planes, self.care_status, self._coupled = K_planes, status, coupled
        # planes [4*m][D] (K_matrix(d) gives one drone's [4, m]) or, coupled, [N][4*m][D]: entry (j, i*m + k, e*N + r) = K_e[4r + i, m j + k]
        self.K = self.K_planes
        return self.K

    def K_matrix(self, i=0, env_idx=0):
        """[4, m] gain of robot i in environment env_idx (uncoupled variants)."""
        if self._coupled:
            raise _lib.MdsError("coupled gain: read self.K_planes [N*4*m, D] (or self.K [E, 4N, mN] after the host solver)")
        return self.K_planes[:, self._drone(i, env_idx)].reshape(self.n, self.m).clone()

    def _compute_controller_host(self, force_diagonal=False):
        th = self.theta.detach().to("cpu", torch.float64).numpy()
        D, N, m, n = th.shape[0], self.num_robots, self.m, self.n
        cache = {}
        self._coupled = bool(self.COUPLED and N >= 2 and not force_diagonal)
        if not self._coupled:
            K = np.zeros((D, n, m))
            for d in range(D):
                key = th[d].tobytes()
                if key not in cache:
                    A, B = th[d][:m].T, th[d][m:].T
                    Pc = la.solve_continuous_are(A, B, self.ind_Q, self.ind_R, e=None, s=None, balanced=True)
                    cache[key] = la.solve(self.ind_R, B.T @ Pc)
                K[d] = cache[key]
            planes = K.reshape(D, -1).T
        else:
            Q, R = self._env_weights()
            E = D // N
            K = np.zeros((E, n * N, m * N))
            for e in range(E):
                blk = th[e * N:(e + 1) * N]
                key = blk.tobytes()
                if key not in cache:
                    A = la.block_diag(*[b[:m].T for b in blk])
                    B = la.block_diag(*[b[m:].T for b in blk])
                    Pc = la.solve_continuous_are(A, B, Q, R, e=None, s=None, balanced=True)
                    cache[key] = la.solve(R, B.T @ Pc)
                K[e] = cache[key]
            # planes [N_src][4*m][D]: entry (j, i*m + k, d = e*N + r) = K[e][4r + i, m j + k]
            Kb = K.reshape(E, N, n, N, m)                      # e, r, i, j, k
            planes = Kb.transpose(3, 2, 4, 0, 1).reshape(N * n * m, D)
        self.K = K
        if self.K_planes.shape[0] != planes.shape[0]:
            self.K_planes = torch.zeros(planes.shape[0], D, device=self.env.device, dtype=self.env.dtype)
        self.K_planes.copy_(torch.as_tensor(np.ascontiguousarray(planes)).to(self.K_planes))
        return K

    def compute(self, obs, skip_low_level=False):
        """-> (action [E,N,4] or None, u [E,N,4]); u_d = -sum_j K_dj e_j (+ hover thrust), capped like the variant's
        reference (the 12-dim reference returns the un-offset flat u, decentralized_lqr.py:336-342; here u is always the
        per-drone input that produced the action)."""
        if self.K is None:
            raise _lib.MdsError("compute_controller() has not been called")
        env = self.env
        run_inner = not skip_low_level
        pid = self.low_level.pid_struct() if self.low_level is not None else _lib.PidState(None, None)
        _lib.call("mds_dlqr_ctrl", env.dtype, env._prm, self.VARIANT, _lib.ptr(self.K_planes), int(self._coupled), _lib.ptr(self._obs(obs)),
                  _lib.ptr(self._ref_view), _lib.ptr(self.u), _lib.ptr(self.action) if run_inner else None, pid, env.NUM_ENVS, env.NUM_DRONES,
                  _lib.stream_ptr(env.device))
        return (self.action if run_inner else None), self.u

    def compute_low_level(self, u, obs, robot_idx=None):
        return self.low_level.compute_from_obs(u, obs)

    def cost(self, x, u):
        """x' Q x + u' R u per drone (decentralized_lqr_omega.py:251-252); x [..., m], u [..., 4]."""
        Q = torch.as_tensor(np.diag(self.ind_Q).copy()).to(x)
        R = torch.as_tensor(np.diag(self.ind_R).copy()).to(u)
        return (x * x * Q).sum(-1) + (u * u * R).sum(-1)

    # exploration inputs (decentralized_lqr_omega.py:140-157): [E, N, 4] draws from a torch generator
    def sigma1(self, generator=None):
        env = self.env
        shp = (env.NUM_ENVS, env.NUM_DRONES)
        mg = env.M * env.G
        thrust = torch.empty(*shp, 1, device=env.device, dtype=env.dtype).uniform_(0.7 * mg, 1.5 * mg, generator=generator)
        ang = torch.empty(*shp, 3, device=env.device, dtype=env.dtype).uniform_(-1e-5, 1e-5, generator=generator)
        return torch.cat([thrust, ang], dim=-1)

    def sigma_explore(self, generator=None):
        env = self.env
        shp = (env.NUM_ENVS, env.NUM_DRONES)
        mg = env.M * env.G
        thrust = mg + 0.005 * mg * torch.randn(*shp, 1, device=env.device, dtype=env.dtype, generator=generator)
        ang = 5e-9 * torch.randn(*shp, 3, device=env.device, dtype=env.dtype, generator=generator)
        return torch.cat([thrust, ang], dim=-1)


class DecentralizedLQROmega(_DecentralizedBase):
    """9-dim thrust + body-rate model (control/dlqr/decentralized_lqr_omega.py)."""
    VARIANT, M = _lib.CTRL_LQR_OMEGA, 9
    RLS_METHODS = {"theta_update": (RLS_TARGET_PREDICT, True, True, RLS_PROJECT_NONE),
                   "theta_update2": (RLS_TARGET_PREDICT, True, False, RLS_PROJECT_NONE)}

    def _weights(self):
        mt = self.env.MAX_THRUST  # decentralized_lqr_omega.py:21-37
        r = [1 / mt ** 2, 100.0, 100.0, 100.0]
        q = [1 / (np.pi / 20) ** 2] * 2 + [1 / (np.pi / 40) ** 2] + [1 / .15 ** 2] * 3 + [1 / .05 ** 2] * 3
        return np.diag(q), np.diag(r)

    def _make_low_level(self):
        return ThrustOmegaController(self.env)

    def theta_update(self, phis, xtp1s):
        """:125-139 -- RLS on x_{t+1} - forward_predict(x_{t+1}, u) (the reference starts the prediction at x_{t+1})."""
        return self._rls(phis, xtp1s, "theta_update")

    def theta_update2(self, phis, xtp1s):
        """:110-123 -- information form: theta += V^-1 phi r, V += phi phi'.  ``P`` holds V^-1 here (V0 = I), kept current
        by the rank-one inverse update, so no 13 x 13 inverse per drone and step."""
        return self._rls(phis, xtp1s, "theta_update2")


class DecentralizedLQRYankOmega(_DecentralizedBase):
    """10-dim yank + body-rate model (control/dlqr/decentralized_lqr_yank_omega.py).  Its ``error_state`` / ``compute``
    index a 9-dim layout and raise in the reference (3 x 3 rotation applied to 4 entries); here they follow the
    LQRYankOmegaController error state (lqr_YO_controller.py:106-116), which is what the crazyflie variant's YOState does."""
    VARIANT, M = _lib.CTRL_LQR_YANK, 10
    RLS_METHODS = {"theta_update": (RLS_TARGET_PREDICT, True, True, RLS_PROJECT_NONE)}

    def _weights(self):
        env = self.env  # decentralized_lqr_yank_omega.py:20-41
        max_yank = (env.MAX_THRUST / env.CTRL_TIMESTEP) / 2
        r = [1 / max_yank ** 2, 100.0, 100.0, 100.0]
        q = [1 / (np.pi / 20) ** 2] * 2 + [1 / (np.pi / 40) ** 2] + [1 / (env.MAX_THRUST - env.M * env.G) ** 2] + [1 / .15 ** 2] * 3 + [1 / .05 ** 2] * 3
        return np.diag(q), np.diag(r)

    def _make_low_level(self):
        return YankOmegaController(self.env)

    def theta_update(self, phis, xtp1s):
        """:112-126"""
        return self._rls(phis, xtp1s, "theta_update")


class DecentralizedYOLQRCrazyflie(DecentralizedLQRYankOmega):
    """control/dlqr/decentralized_yolqr_crazyflie.py: caller-supplied Q / R, P0 = 5 I, x_dot regression with projection."""
    P0_SCALE = 5.0
    RLS_METHODS = dict(DecentralizedLQRYankOmega.RLS_METHODS, approx_theta_update=(RLS_TARGET_XDOT, False, True, RLS_PROJECT_LOOP))

    def __init__(self, env, lin_models, indQ, indR, debug=False, P=None):
        self._qr = (np.asarray(indQ, float), np.asarray(indR, float))
        super().__init__(env, lin_models, debug)
        if P is not None:
            self.set_P(P)
        self.compute_controller()

    def _weights(self):
        return self._qr

    def _project_codes(self):
        if self._codes is None:
            m = self.m  # :164-186, 245-257
            A = np.zeros((m, m), np.uint8)
            B = np.zeros((m, 4), np.uint8)
            A[(4, 5), (1, 0)] = 1
            A[(7, 8, 9), (4, 5, 6)] = 2
            A[6, 3] = 1
            B[(0, 1, 2), (1, 2, 3)] = 1
            B[3, 0] = 1
            self._codes = np.vstack([A.T, B.T])
        return self._codes

    def approx_theta_update(self, phis, xtp1s, project=True):
        """:259-290"""
        return self._rls(phis, xtp1s, "approx_theta_update", project=project)


class DecentralizedLQR(_DecentralizedBase):
    """12-dim torque-level model (control/dlqr/decentralized_lqr.py)."""
    VARIANT, M = _lib.CTRL_LQR_TORQUE, 12
    P0_SCALE = 20.0
    COUPLED = True
    RLS_METHODS = {"theta_update": (RLS_TARGET_PREDICT, False, True, RLS_PROJECT_AFTER),
                   "approx_theta_update": (RLS_TARGET_XDOT, False, True, RLS_PROJECT_LOOP)}

    def _weights(self):
        mt = self.env.MAX_THRUST  # decentralized_lqr.py:16-34
        r = [1 / mt ** 2, 1 / 0.001 ** 2, 1 / 0.001 ** 2, 1 / 0.001 ** 2]
        q = [1 / (np.pi / 10) ** 2] * 2 + [1 / (np.pi / 20) ** 2] + [1 / .5 ** 2] * 3 + [1 / .15 ** 2] * 3 + [1 / .05 ** 2] * 3
        return np.diag(q), np.diag(r)

    def _env_weights(self):
        Q, R = super()._env_weights()  # :44-53: negative weight between the xy positions of robots 0 and 1
        Q[9:11, 21:23] = -1 / 0.1 ** 2
        Q[21:23, 9:11] = -1 / 0.1 ** 2
        return Q, R

    def _init_P(self):
        P = self.P_planes.view(self.mn, self.mn, -1)  # :60-63: the three torque inputs start at 5e6
        for k in range(self.mn - 3, self.mn):
            P[k, k, :] = 5_000_000.0

    def _project_codes(self):
        if self._codes is None:
            A = np.zeros((12, 12), np.uint8)  # :70-87, 230-240
            B = np.zeros((12, 4), np.uint8)
            A[(6, 7), (1, 0)] = 1
            A[(0, 1, 2), (3, 4, 5)] = 2
            A[(9, 10, 11), (6, 7, 8)] = 2
            B[3:6, 1:] = 1
            B[8, 0] = 1
            self._codes = np.vstack([A.T, B.T])
        return self._codes

    def theta_update(self, phis, xtp1s):
        """:157-183 -- prediction from e_t, project_theta once after the robots' loop."""
        return self._rls(phis, xtp1s, "theta_update")

    def approx_theta_update(self, phis, xtp1s):
        """:200-228"""
        return self._rls(phis, xtp1s, "approx_theta_update")
