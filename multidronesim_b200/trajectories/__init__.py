"""Reference trajectory generators, evaluated on device.

Same constructors and call contract as the reference's ``trajectories`` package
(``traj(t) -> (pos, vel, acc, yaw, omega)``; Circle.py:5-45, Lemniscate.py:3-63,
LineTrajectory.py:4-14,16-103, CompoundTrajectory.py:5-40, RotateTrajectory.py:5-24),
but a trajectory object is only a *description*: ``TrajectorySet`` packs one description
per drone into the device tables ``MdsTrajSpec`` / ``MdsTrajSeg`` (include/mds_b200.h) and
``TrajectorySet(t)`` evaluates all of them with one launch of ``mds_traj_eval``.  Init-time
scalar set-up (Line's trapezoid timings) runs on the host exactly like the reference's
constructors; nothing per-step runs on the CPU.
"""
from __future__ import annotations

import math

import numpy as np
import torch

from .. import _lib


class TrajectoryBase:
    def get_total_time(self):
        raise NotImplementedError

    def segments(self):
        """List of (kind, dur, p[<=24], rot[12] or None) segment descriptions."""
        raise NotImplementedError

    def simple_spec(self):
        """(kind, p[<=8]) if the generator fits a per-drone MdsTrajSpec, else None."""
        return None


class CircleTrajectory(TrajectoryBase):
    def __init__(self, r=1.0, v=.5, center=np.array([0, 0, 0]), yaw_rate=0, revolutions=None, duration=None):
        self.r, self.v, self.yaw_rate = float(r), float(v), float(yaw_rate)
        self.center = np.asarray(center, dtype=float)
        if revolutions is not None:
            self.total_time = 2 * r * np.pi * revolutions / self.v
        elif duration is not None:
            self.total_time = duration
        else:
            self.total_time = 2 * np.pi * self.r / self.v

    def get_total_time(self):
        return self.total_time

    def _p(self):
        return [self.r, self.v, *self.center, self.yaw_rate]

    def simple_spec(self):
        return _lib.TRAJ_CIRCLE, self._p()

    def segments(self):
        return [(_lib.SEG_CIRCLE, self.total_time, self._p(), None)]


class Lemniscate(TrajectoryBase):
    def __init__(self, a=1, omega=.5, center=np.array([0, 0, 0]), yaw_rate=0, revolutions=None, duration=None, phase_shift=0):
        self.a, self.omega, self.yaw_rate, self.phase_shift = float(a), float(omega), float(yaw_rate), float(phase_shift)
        self.center = np.asarray(center, dtype=float)
        if revolutions is not None:
            self.total_time = 2 * np.pi * revolutions / omega
        elif duration is not None:
            self.total_time = duration
        else:
            self.total_time = 2 * np.pi / omega

    def get_total_time(self):
        return self.total_time

    def _p(self):
        return [self.a, self.omega, *self.center, self.yaw_rate, self.phase_shift]

    def simple_spec(self):
        return _lib.TRAJ_LEMNISCATE, self._p()

    def segments(self):
        return [(_lib.SEG_LEMNISCATE, self.total_time, self._p(), None)]


class WaitTrajectory(TrajectoryBase):
    def __init__(self, position, duration, yaw=0):
        self.position, self.duration, self.yaw = np.asarray(position, dtype=float), float(duration), float(yaw)

    def get_total_time(self):
        return self.duration

    def _p(self):
        return [*self.position, self.yaw]

    def simple_spec(self):
        return _lib.TRAJ_WAIT, self._p()

    def segments(self):
        return [(_lib.SEG_WAIT, self.duration, self._p(), None)]


class LineTrajectory(TrajectoryBase):
    """Trapezoidal speed profile with a_max = 1 (LineTrajectory.py:16-103, quirk B20 kept:
    ``speed`` is required, ``dist_end`` uses |v0|, the ramps accelerate by sign() per axis)."""

    def __init__(self, start, end, speed=None, duration=None, s0=0, sf=0):
        assert speed > 0, "Speed must be positive"
        if duration is not None:
            assert duration > 0, "Duration must be positive"
        self.start, self.end = np.asarray(start, dtype=float), np.asarray(end, dtype=float)
        delta = self.end - self.start
        dist = float(np.linalg.norm(delta))
        self.max_acc = 1.0
        self.speed = float(speed)
        self.dir = delta / dist
        self.v0, self.vf = s0 * self.dir, sf * self.dir

        def ramps():
            dvi, dve = self.speed * self.dir - self.v0, self.vf - self.speed * self.dir
            ti, te = np.linalg.norm(dvi) / self.max_acc, np.linalg.norm(dve) / self.max_acc
            n0 = np.linalg.norm(self.v0)
            return dvi, dve, ti, te, n0 * ti + .5 * self.max_acc * ti ** 2, n0 * te + .5 * self.max_acc * te ** 2

        dvi, dve, ti, te, di, de = ramps()
        if di + de > dist:
            self.time_middle = 0.0
            self.speed = sf + math.sqrt(dist * self.max_acc) + 0.5 * s0 ** 2 - 0.5 * sf ** 2
            dvi, dve, ti, te, di, de = ramps()
        else:
            self.time_middle = (dist - di - de) / self.speed
        self.delta_v_init, self.delta_v_end, self.time_init, self.time_end = dvi, dve, float(ti), float(te)
        self.total_time = self.time_init + self.time_middle + self.time_end

    def get_total_time(self):
        return self.total_time

    def segments(self):
        p = [*self.start, *self.v0, *np.sign(self.delta_v_init), *(self.speed * self.dir), *np.sign(self.delta_v_end),
             *self.end, *self.vf, self.time_init, self.time_middle, self.total_time]
        return [(_lib.SEG_LINE, self.total_time, p, None)]


class CompoundTrajectory(TrajectoryBase):
    """Piecewise dispatcher (CompoundTrajectory.py:5-40).  The device evaluates it statelessly
    (segment = first k with t <= cumulative end); identical to the reference's cursor for a
    forward-running clock, see DESIGN.md."""

    def __init__(self, trajectories):
        self.trajectories = list(trajectories)
        self.total_time = sum(t.get_total_time() for t in self.trajectories)

    def get_total_time(self):
        return self.total_time

    def segments(self):
        out = []
        for t in self.trajectories:
            out.extend(t.segments())
        return out


class RotateTrajectory(TrajectoryBase):
    def __init__(self, trajectory, R, center):
        self.trajectory, self.R, self.center = trajectory, np.asarray(R, dtype=float), np.asarray(center, dtype=float)

    def get_total_time(self):
        return self.trajectory.get_total_time()

    def segments(self):
        out = []
        for kind, dur, p, rot in self.trajectory.segments():
            if rot is not None:
                raise NotImplementedError("nested RotateTrajectory is not supported on device")
            else:
                out.append((kind, dur, p, [*self.R.reshape(-1), *self.center]))
        return out


class TrajectorySet:
    """One trajectory per drone, packed for the device.  ``trajs`` is a list of D = E*N
    descriptions, or N descriptions repeated over ``num_envs`` environments.

    ``env_period`` is N when every environment flies the same N trajectories (descriptor d equals descriptor d mod N), else 0.
    ``FusedRollout`` passes it to the kernel, which then evaluates each reference once per block instead of once per drone.
    Assigning ``specs`` clears it; code that edits the ``specs`` tensor in place must set it to 0 itself."""

    def __init__(self, trajs, num_envs=1, device="cuda", dtype=torch.float32):
        _lib.load_library()
        self.device, self.dtype = torch.device(device), dtype
        real = "f4" if dtype == torch.float32 else "f8"
        trajs = list(trajs)
        n_unique = len(trajs)
        specs = np.zeros(n_unique, dtype=_lib.traj_spec_dtype(real))
        segs = []
        for d, tr in enumerate(trajs):
            simple = tr.simple_spec()
            if simple is not None:
                kind, p = simple
                specs[d]["kind"] = kind
                specs[d]["p"][:len(p)] = p
            else:
                sg = tr.segments()
                specs[d]["kind"] = _lib.TRAJ_TABLE
                specs[d]["seg_begin"], specs[d]["seg_count"] = len(segs), len(sg)
                # a generator used on its own keeps its own behaviour past total_time (e.g. Line returns
                # (end, vf, 0); Rotate(Lemniscate) stays periodic); only CompoundTrajectory clamps at the end
                specs[d]["pad"] = 0 if isinstance(tr, CompoundTrajectory) else 1
                t_end = 0.0
                for kind, dur, p, rot in sg:
                    t_end += dur
                    segs.append((kind, rot is not None, t_end, dur, p, rot))
        seg_arr = np.zeros(max(1, len(segs)), dtype=_lib.traj_seg_dtype(real))
        for k, (kind, has_rot, t_end, dur, p, rot) in enumerate(segs):
            seg_arr[k]["kind"], seg_arr[k]["has_rot"], seg_arr[k]["t_end"], seg_arr[k]["dur"] = kind, int(has_rot), t_end, dur
            seg_arr[k]["p"][:len(p)] = p
            if rot is not None:
                seg_arr[k]["rot"][:] = rot
        if num_envs > 1:
            specs = np.tile(specs, num_envs)
        self._finish(specs, seg_arr, n_unique)

    def _finish(self, specs, seg_arr, env_period):
        self.num = len(specs)
        self.specs = torch.from_numpy(specs.view(np.uint8).copy()).to(self.device)
        self.segs = torch.from_numpy(seg_arr.view(np.uint8).copy()).to(self.device)
        self.ref = torch.zeros(self.num, _lib.REF_DIM, device=self.device, dtype=self.dtype)
        self.env_period = env_period

    @property
    def specs(self):
        return self._specs

    @specs.setter
    def specs(self, value):
        self._specs = value
        self.env_period = 0  # new descriptors are not known to repeat per environment

    @classmethod
    def from_arrays(cls, kind, params, device="cuda", dtype=torch.float32, drones_per_env=None):
        """Vectorised constructor for large swarms: ``kind`` int or [D] array of MDS_TRAJ_*,
        ``params`` [D, <=8] (layout of include/mds_b200.h).  With ``drones_per_env`` = N the descriptors are
        checked for repeating per environment (``env_period``)."""
        self = cls.__new__(cls)
        _lib.load_library()
        self.device, self.dtype = torch.device(device), dtype
        real = "f4" if dtype == torch.float32 else "f8"
        params = np.asarray(params, dtype=float)
        specs = np.zeros(params.shape[0], dtype=_lib.traj_spec_dtype(real))
        specs["kind"] = kind
        specs["p"][:, :params.shape[1]] = params
        period = 0
        if drones_per_env and len(specs) % int(drones_per_env) == 0:
            envs = specs.view(np.uint8).reshape(len(specs) // int(drones_per_env), -1)  # one row of bytes per environment
            period = int(drones_per_env) if bool((envs == envs[0]).all()) else 0
        self._finish(specs, np.zeros(1, dtype=_lib.traj_seg_dtype(real)), period)
        return self

    def eval(self, t, out=None):
        """All references at time t -> [D, 11] = pos3, vel3, acc3, yaw, yaw_rate (library-owned buffer)."""
        out = self.ref if out is None else out
        _lib.call("mds_traj_eval", self.dtype, _lib.ptr(self.specs), _lib.ptr(self.segs), float(t), _lib.ptr(out),
                  self.num, _lib.stream_ptr(self.device))
        return out

    def __call__(self, t):
        r = self.eval(t)
        return r[:, 0:3], r[:, 3:6], r[:, 6:9], r[:, 9], r[:, 10]
