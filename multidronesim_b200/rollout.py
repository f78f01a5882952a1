"""K-step rollout (``mds_rollout``): by default ONE launch advances every environment K control steps (trajectory ->
tracking controller -> CBF-QP -> inner loop -> physics sub-steps, observation and body rates in registers from step to
step); other launch plans (two launches per step, single kernels) via ``stages``.

It is the device equivalent of the reference's per-step Python loops
(simulations/EnvGeometric.py:434-479, simulations/CBFTest.py:302-358,
simulations/CBFTestOrd3.py:305-360) including what those callers do around the library calls
(``nominal_us[:,0] -= M*G`` before the QP, ``+= M*G`` after it for order 2 only)."""
from __future__ import annotations

import torch

from . import _lib
from .control.dslpid import DSLPIDControl
from .control.geometric import GeometricControl
from .control.lqr import LQRController, LQROmegaController, LQRYankOmegaController
from .control.dlqr import DecentralizedLQR, _DecentralizedBase


class FusedRollout:
    def __init__(self, env, trajs, controller, qp_tracker=None, obstacles=None, ref_table=True):
        """env: BatchedCtrlAviary; trajs: TrajectorySet (one per drone); controller: GeometricControl |
        LQRController | LQROmegaController | LQRYankOmegaController; qp_tracker: DroneQPTracker or None;
        obstacles: tensor/list [N_obs, 4] = cx, cy, cz, r (shared by all envs).
        ref_table: when every environment flies the same trajectories (``trajs.env_period == N``), let the kernel
        evaluate each reference once per block and step (MdsRolloutCfg.traj_period; same results).  False (or the attribute
        of the same name) keeps the per-drone evaluation."""
        self.env, self.trajs, self.controller, self.qp = env, trajs, controller, qp_tracker
        self.ref_table = ref_table
        if trajs.num != env.NUM_TOTAL:
            raise ValueError("need one trajectory per drone")
        cfg = _lib.RolloutCfg()
        if isinstance(controller, GeometricControl):
            cfg.ctrl = _lib.CTRL_GEOMETRIC
        elif isinstance(controller, DSLPIDControl):
            cfg.ctrl = _lib.CTRL_DSLPID
        elif isinstance(controller, _DecentralizedBase):
            # the reference's `--controller dlqr` (simulations/CBFTest.py:319-321): every drone under its own learned gain
            if controller.K is None or controller._coupled:
                raise _lib.MdsError("FusedRollout takes a decentralised LQR with per-drone gains: call compute_controller() first "
                                    "(the robot-coupled 12-dim gain runs through PerCallPipeline)")
            cfg.ctrl = controller.VARIANT
        elif isinstance(controller, LQROmegaController):
            cfg.ctrl = _lib.CTRL_LQR_OMEGA
        elif isinstance(controller, LQRYankOmegaController):
            cfg.ctrl = _lib.CTRL_LQR_YANK
        elif isinstance(controller, LQRController):
            cfg.ctrl = _lib.CTRL_LQR_TORQUE
        else:
            raise TypeError("unsupported controller type")
        cfg.use_cbf = int(qp_tracker is not None)
        rows = [] if obstacles is None else (obstacles.tolist() if isinstance(obstacles, torch.Tensor) else list(obstacles))
        if len(rows) > _lib.MAX_OBSTACLES:
            raise ValueError("too many obstacles")
        cfg.num_obstacles = len(rows) if qp_tracker is not None else 0
        if qp_tracker is not None:
            qp_tracker.cbf.check_obstacle_count(cfg.num_obstacles)
        for i, r in enumerate(rows):
            for k in range(4):
                cfg.obstacles[4 * i + k] = float(r[k])
        cfg.write_obs_every = 0
        self.cfg = cfg
        self.stats = torch.zeros(_lib.STAT_COUNT, device=env.device, dtype=torch.float64)
        self.reset_stats()
        self.t = 0.0

    def reset_stats(self):
        self.stats.zero_()
        self.stats[3] = 1e30  # MDS_STAT_MIN_BARRIER

    def plan(self):
        """launch plan ``run`` uses by default (6: all K steps in one launch)"""
        return _lib.load_library().mds_rollout_plan(self.env.NUM_ENVS, self.env.NUM_DRONES)

    def run(self, K, t0=None, obs_log=None, log_every=0, stages=0):
        """Advance every environment K control steps.  ``obs_log`` [K//log_every, E, N, 20] receives the
        observation after every ``log_every``-th step (the reference's ``observations.append(obs)``).
        ``stages`` (MdsRolloutCfg.stages): 0 = whole steps with the default plan (``plan()``: 6 = all K steps in ONE
        launch, observation and body rates in registers from step to step; 6 selects it explicitly);
        4 = whole steps as two launches each; 1 = controller kernel only (fills the env's action buffer, time does
        not advance); 2 = physics kernel only (consumes that action buffer).  ``run(1, stages=1)`` then
        ``run(1, stages=2)`` is one step of plan 4: K such pairs replay a rollout launch by launch.
        Returns the env's obs buffer (observation after the last step)."""
        env = self.env
        if t0 is None:
            t0 = self.t
        if stages not in (0, 1, 2, 4, 6):
            raise ValueError("stages must be 0, 1, 2, 4 or 6")
        self.cfg.stages = int(stages)
        self.cfg.write_obs_every = int(log_every) if obs_log is not None else 0
        N = env.NUM_DRONES
        self.cfg.traj_period = N if (self.ref_table and self.trajs.env_period == N) else 0
        if obs_log is not None:
            _lib.require_cuda(obs_log, "obs_log", env.dtype)
            if obs_log.numel() < (K // max(1, log_every)) * env.NUM_TOTAL * _lib.OBS_DIM:
                raise ValueError("obs_log too small")
        is_lqr = self.cfg.ctrl in (_lib.CTRL_LQR_TORQUE, _lib.CTRL_LQR_OMEGA, _lib.CTRL_LQR_YANK)
        geo = self.controller.c_gains() if self.cfg.ctrl == _lib.CTRL_GEOMETRIC else None
        per_drone = isinstance(self.controller, _DecentralizedBase)
        if per_drone:  # gains: the controller's K planes (re-read every call: compute_controller() may have run since)
            if self.controller._coupled:
                raise _lib.MdsError("robot-coupled gains cannot run in the fused rollout")
            self.cfg.lqr_gain_planes_dev = self.controller.K_planes.data_ptr()
            lqr = _lib.LqrGains()
            lqr.dim = self.controller.m
            pid = self.controller.low_level.pid_struct() if self.controller.low_level is not None else _lib.PidState(None, None)
        else:
            self.cfg.lqr_gain_planes_dev = None
            lqr = self.controller.c_gains() if is_lqr else None
            pid = self.controller._pid() if is_lqr else _lib.PidState(None, None)
        dsl = self.controller.c_gains() if self.cfg.ctrl == _lib.CTRL_DSLPID else None
        dsl_state = self.controller.state_struct() if self.cfg.ctrl == _lib.CTRL_DSLPID else _lib.DslPidState(None, None, None)
        cbf = self.qp.cbf.c_params() if self.qp is not None else None
        _lib.call("mds_rollout", env.dtype, env._prm, self.cfg, geo, lqr, cbf, env._state_struct(), pid, dsl, dsl_state,
                  _lib.ptr(self.trajs.specs), _lib.ptr(self.trajs.segs), _lib.ptr(env._obs), _lib.ptr(env._action), _lib.ptr(env._ext_force), _lib.ptr(obs_log),
                  _lib.ptr(self.stats), float(t0), int(K), env.NUM_ENVS, env.NUM_DRONES, _lib.stream_ptr(env.device))
        if stages != 1:
            env.step_counter += K * env.PYB_STEPS_PER_CTRL
            self.t = t0 + K * env.CTRL_TIMESTEP
        return env._obs

    def stats_dict(self):
        v = self.stats.tolist()
        return dict(zip(_lib.STAT_NAMES, v))


class LearningRollout:
    """The system-identification loop of the decentralised LQR (the warm-up / learning phases of the reference's
    simulations/CBFTest.py:150-265 and CBFTestOrd3.py:150-270) for K control steps in ONE launch (``mds_learning_rollout``).
    Every drone flies the caller's excitation inputs through its inner loop while its RLS model learns from the
    transitions; theta and P stay in shared memory for the whole launch.  ``run`` equals this per-call loop::

        for k in range(K):
            dl.set_reference(trajs.eval(t0 + k * dt))
            e_t = dl.error_state(obs); action = dl.compute_low_level(inputs[k], obs); obs = env.step(action)[0]
            if k >= learn_from: getattr(dl, method)(torch.cat([e_t, inputs[k]], -1), dl.error_state(obs), **method_kwargs)

    ``run(..., feedback=True)`` is closed-loop exploration (``mds_learning_rollout_feedback``): every drone flies its own
    learned gain ``dl.K_planes`` plus the perturbation ``inputs[k]`` while its model learns -- the certainty-equivalence loop
    ``compute_controller() -> run(feedback=True) -> compute_controller() -> ...``.  It equals this per-call loop::

        for k in range(K):
            dl.set_reference(trajs.eval(t0 + k * dt))
            e_t = dl.error_state(obs).clone()
            _, u = dl.compute(obs, skip_low_level=True)   # u = -K_d e_t (+ m g unless yank-omega); LQR_OMEGA: cap_u
            u = u + inputs[k]                              # exploration perturbation
            obs = env.step(dl.compute_low_level(u, obs))[0]
            if k >= learn_from: getattr(dl, method)(torch.cat([e_t, u], -1), dl.error_state(obs), **method_kwargs)

    The gain is read once per launch and stays constant within it (the loop above does not recompute it either), and the
    feedback acts from step 0 whatever ``learn_from`` is.

    controller: DecentralizedLQROmega, DecentralizedLQRYankOmega or DecentralizedYOLQRCrazyflie (the variants with an inner
    loop); trajs: TrajectorySet with one trajectory per drone (the references of the error states)."""

    def __init__(self, env, trajs, controller):
        if isinstance(controller, DecentralizedLQR):
            raise _lib.MdsError("LearningRollout takes the decentralised LQR variants with an inner loop; the 12-dim torque model "
                                "has none and a robot-coupled gain")
        if not isinstance(controller, _DecentralizedBase):
            raise TypeError("LearningRollout needs a decentralised LQR controller (control.dlqr)")
        if trajs.num != env.NUM_TOTAL:
            raise ValueError("need one trajectory per drone")
        if controller.env is not env:
            raise ValueError("the controller belongs to another env")
        self.env, self.trajs, self.controller = env, trajs, controller
        self.t = 0.0

    def run(self, inputs, method="theta_update", learn_from=0, t0=None, obs_log=None, log_every=0, feedback=False, **method_kwargs):
        """inputs [K, E, N, 4] (device, the env's dtype): the excitation of every step (``dl.sigma1()`` draws, say); with
        ``feedback=True`` the perturbations added to the law's output (entry 0 perturbs the yank of the yank-omega variants).
        method: the controller's RLS method (``theta_update``, ``theta_update2``, ``approx_theta_update``), method_kwargs its
        options (``project``).  The first RLS step is step ``learn_from`` (1 reproduces the reference's ``if i != 0``).
        ``obs_log`` [K//log_every, E, N, 20] receives the observation after every ``log_every``-th step.  Leaves the env state
        and obs, the inner loop's PID state, theta, P and ``resid`` (of the last update) as the loop does.  Returns the obs."""
        env, dl = self.env, self.controller
        if not isinstance(inputs, torch.Tensor):
            raise TypeError("inputs must be a torch tensor [K, E, N, 4]")
        if inputs.dim() != 4 or tuple(inputs.shape[1:]) != (env.NUM_ENVS, env.NUM_DRONES, 4):
            raise ValueError(f"inputs must have shape [K, {env.NUM_ENVS}, {env.NUM_DRONES}, 4], got {tuple(inputs.shape)}")
        _lib.require_cuda(inputs, "inputs", env.dtype)
        cfg = dl.rls_cfg(method, **method_kwargs)
        if feedback and dl.K is None:
            raise _lib.MdsError("feedback=True flies the learned gain: call compute_controller() first")
        K = int(inputs.shape[0])
        if t0 is None:
            t0 = self.t
        if K == 0:  # nothing to run (the C entry point takes K = 0 as well; an empty tensor has no storage to point at)
            return env._obs
        write_every = int(log_every) if obs_log is not None else 0
        if obs_log is not None:
            _lib.require_cuda(obs_log, "obs_log", env.dtype)
            if write_every < 1 or obs_log.numel() < (K // write_every) * env.NUM_TOTAL * _lib.OBS_DIM:
                raise ValueError("obs_log too small or log_every < 1")
        name, gain = ("mds_learning_rollout_feedback", [_lib.ptr(dl.K_planes)]) if feedback else ("mds_learning_rollout", [])
        _lib.call(name, env.dtype, env._prm, cfg, dl.VARIANT, int(learn_from), write_every, env._state_struct(), dl.low_level.pid_struct(),
                  _lib.ptr(self.trajs.specs), _lib.ptr(self.trajs.segs), _lib.ptr(inputs), *gain, _lib.ptr(dl.theta_planes), _lib.ptr(dl.P_planes),
                  _lib.ptr(dl.resid), _lib.ptr(env._obs), _lib.ptr(env._ext_force), _lib.ptr(obs_log), float(t0), K, env.NUM_ENVS,
                  env.NUM_DRONES, _lib.stream_ptr(env.device))
        env.step_counter += K * env.PYB_STEPS_PER_CTRL
        dl.low_level.control_counter += K
        self.t = t0 + K * env.CTRL_TIMESTEP
        return env._obs


class PerCallPipeline:
    """One control step through the per-call device API in the reference's call order
    (simulations/CBFTest.py:302-350): references in -> ctrl.compute(skip_low_level) -> caller glue
    (mds_cbf_prepare) -> qp_tracker.compute_control -> ctrl.compute_low_level -> env.step."""

    def __init__(self, env, controller, qp_tracker=None, obstacles=None):
        self.env, self.ctrl, self.qp = env, controller, qp_tracker
        self.obst = None
        if qp_tracker is not None and obstacles is not None and len(obstacles):
            self.obst = torch.as_tensor(obstacles, device=env.device, dtype=env.dtype).reshape(-1, 4).contiguous()
        if qp_tracker is not None:
            self.xdes = torch.zeros(env.NUM_ENVS, env.NUM_DRONES, qp_tracker.xdim, device=env.device, dtype=env.dtype)
        self.mg = env.M * env.G
        self.launches_per_step = 5 if qp_tracker is not None else 2

    def step(self, ref, obs_out=None):
        """ref: device tensor [D, 11] (pos, vel, acc, yaw, yaw_rate per drone).  Returns the new observation
        (written to ``obs_out`` when given, see BatchedCtrlAviary.step)."""
        env, c = self.env, self.ctrl
        c.set_reference(ref)
        obs = env.obs
        if self.qp is None:
            out = c.compute(obs)
            action = out if isinstance(out, torch.Tensor) else out[0]
        else:
            _, u = c.compute(obs, skip_low_level=True)
            _lib.call("mds_cbf_prepare", env.dtype, env._prm, self.qp.order, self.mg, _lib.ptr(ref), _lib.ptr(u), _lib.ptr(self.xdes),
                      env.NUM_TOTAL, _lib.stream_ptr(env.device))
            us = self.qp.compute_control(obs, self.xdes, u, x_obs=self.obst)
            if self.qp.order == 2:
                us[..., 0] += self.mg
            action = c.compute_low_level(us, obs)
        return env.step(action, obs_out)[0]


class HostPipeline:
    """Host-buffer form of the per-call path: every control step takes that step's references from PINNED host
    memory and delivers the new observation into PINNED host memory, as a host-side caller of the reference's
    loop would see it (obs out of ``env.step``, set-points in through ``set_desired_trajectory``).

    Three streams, two slots: the H2D copy of step k+1's references and the D2H copy of step k's observation
    run on their own streams while the kernels of step k+1 run on the caller's stream; events order the reuse
    of the two device reference buffers and the two device observation buffers.  ``step`` is asynchronous;
    the returned event fires when ``obs_host`` holds the step's observation."""

    def __init__(self, env, controller, qp_tracker=None, obstacles=None):
        self.env = env
        self.pipe = PerCallPipeline(env, controller, qp_tracker, obstacles)
        dev, dt = env.device, env.dtype
        self.s_in, self.s_out = torch.cuda.Stream(dev), torch.cuda.Stream(dev)
        self.ref_dev = [torch.empty(env.NUM_TOTAL, _lib.REF_DIM, device=dev, dtype=dt) for _ in range(2)]
        self.obs_dev = [torch.empty(env.NUM_ENVS, env.NUM_DRONES, _lib.OBS_DIM, device=dev, dtype=dt) for _ in range(2)]
        mk = lambda: [torch.cuda.Event() for _ in range(2)]
        self.ref_ready, self.ref_free, self.obs_ready, self.obs_free = mk(), mk(), mk(), mk()
        self.k = 0
        self.launches_per_step = self.pipe.launches_per_step

    def step(self, ref_host, obs_host):
        env, slot = self.env, self.k & 1
        cs = torch.cuda.current_stream(env.device)
        first = self.k < 2
        with torch.cuda.stream(self.s_in):
            if not first:
                self.s_in.wait_event(self.ref_free[slot])
            self.ref_dev[slot].copy_(ref_host.reshape(self.ref_dev[slot].shape), non_blocking=True)
            self.ref_ready[slot].record(self.s_in)
        cs.wait_event(self.ref_ready[slot])
        if not first:
            cs.wait_event(self.obs_free[slot])
        self.pipe.step(self.ref_dev[slot], obs_out=self.obs_dev[slot])
        self.ref_free[slot].record(cs)
        self.obs_ready[slot].record(cs)
        with torch.cuda.stream(self.s_out):
            self.s_out.wait_event(self.obs_ready[slot])
            obs_host.copy_(self.obs_dev[slot].reshape(obs_host.shape), non_blocking=True)
            self.obs_free[slot].record(self.s_out)
        self.k += 1
        self.last_ref_ready = self.ref_ready[slot]   # fires when ``ref_host`` has been read: the caller may overwrite it then
        return self.obs_free[slot]

    def synchronize(self):
        self.s_in.synchronize()
        self.s_out.synchronize()
        torch.cuda.current_stream(self.env.device).synchronize()


class HostRollout:
    """K-step host call: ``step`` advances every environment K control steps in ONE launch (``FusedRollout``: trajectories,
    controllers, CBF-QP, inner loop and physics on device, every step's observation written to a device log), then moves
    the K observations to PINNED host memory with one large D2H copy on a copy stream.  Two device log buffers: the copy of
    call j overlaps the launch of call j + 1.  The returned event fires when ``obs_host`` [K, E, N, 20] is complete.
    The device-resident form of the reference's ``observations.append(obs)`` + ``np.save`` (simulations/EnvGeometric.py:470-473,553-556)."""

    def __init__(self, rollout, K):
        env = rollout.env
        self.ro, self.K, self.env = rollout, int(K), env
        self.s_out = torch.cuda.Stream(env.device)
        self.log = [torch.empty(self.K, env.NUM_ENVS, env.NUM_DRONES, _lib.OBS_DIM, device=env.device, dtype=env.dtype) for _ in range(2)]
        self.ready = [torch.cuda.Event() for _ in range(2)]
        self.free = [torch.cuda.Event() for _ in range(2)]
        self.j = 0

    def step(self, obs_host):
        slot = self.j & 1
        cs = torch.cuda.current_stream(self.env.device)
        if self.j >= 2:
            cs.wait_event(self.free[slot])
        self.ro.run(self.K, obs_log=self.log[slot], log_every=1)
        self.ready[slot].record(cs)
        with torch.cuda.stream(self.s_out):
            self.s_out.wait_event(self.ready[slot])
            obs_host.copy_(self.log[slot].reshape(obs_host.shape), non_blocking=True)
            self.free[slot].record(self.s_out)
        self.j += 1
        return self.free[slot]

    def synchronize(self):
        self.s_out.synchronize()
        torch.cuda.current_stream(self.env.device).synchronize()


class SwarmStreams:
    """P independent sub-swarms, each a ``FusedRollout`` over its own ``BatchedCtrlAviary``, advanced on P CUDA streams.

    Environments never interact, so a swarm can be cut into sub-swarms that progress independently.  One ``mds_rollout``
    launch of E environments occupies the GPU in waves of equal blocks (148 SMs x 2 blocks x 32 environments on B200), and
    its last wave is rarely full: 15 625 environments (BASELINE.json configs[4] on one of 8 GPUs) are 1.65 waves and cost 2.
    With the sub-swarms on separate streams the block scheduler fills the tail of one sub-swarm's launch with the blocks of
    the next launch of another, across calls: measured 1.18e10 -> 1.43e10 drone-steps/s at 15 625 environments, 1.42e10 ->
    1.46e10 at 125 000 (tools/exp_streams.py).  ``run`` is asynchronous and does NOT join the streams -- that is the point;
    call ``synchronize()`` (or ``join()`` to order the caller's stream after them) before reading any sub-swarm's tensors."""

    def __init__(self, rollouts):
        self.rollouts = list(rollouts)
        dev = self.rollouts[0].env.device
        self.device = dev
        self.streams = [torch.cuda.Stream(dev) for _ in self.rollouts]
        cur = torch.cuda.current_stream(dev)
        for st in self.streams:   # the sub-swarms' tensors were initialised on the caller's stream
            st.wait_stream(cur)

    @property
    def num_envs(self):
        return sum(r.env.NUM_ENVS for r in self.rollouts)

    def run(self, K, obs_logs=None, log_every=0):
        """Advance every sub-swarm K control steps (one launch each, on its own stream).  ``obs_logs``: one log tensor per sub-swarm."""
        for i, (ro, st) in enumerate(zip(self.rollouts, self.streams)):
            with torch.cuda.stream(st):
                ro.run(K, obs_log=None if obs_logs is None else obs_logs[i], log_every=log_every)

    def fork(self):
        """order the sub-swarm streams after the caller's stream (e.g. after an event recorded there)"""
        cur = torch.cuda.current_stream(self.device)
        for st in self.streams:
            st.wait_stream(cur)

    def join(self):
        """order the caller's stream after everything queued on the sub-swarm streams"""
        cur = torch.cuda.current_stream(self.device)
        for st in self.streams:
            cur.wait_stream(st)

    def synchronize(self):
        for st in self.streams:
            st.synchronize()

    def reset_stats(self):
        self.join()
        for ro in self.rollouts:
            ro.reset_stats()
        self.fork()

    def stats(self):
        """the sub-swarms' statistics combined (layout include/mds_b200.h MDS_STAT_*)"""
        from .dist import reduce_stats
        self.join()
        return reduce_stats(torch.stack([ro.stats for ro in self.rollouts], dim=0))

    def stats_dict(self):
        return dict(zip(_lib.STAT_NAMES, self.stats().tolist()))
