"""ctypes binding of the C-ABI library ``csrc/libmds_b200.so`` (include/mds_b200.h).

There is NO CPU fallback: if the shared library is missing or a call fails, an
exception is raised.  Device pointers are ``torch.Tensor.data_ptr()`` values;
PyTorch is used only for device memory, streams and ``torch.distributed``.
"""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("MDS_B200_LIB") or os.path.join(_HERE, "csrc", "libmds_b200.so")  # override: kernel-variant experiments

MAX_DRONES_PER_ENV = 32
MAX_OBSTACLES = 8
OBS_DIM = 20
REF_DIM = 11
STAT_COUNT = 8
STAT_NAMES = ("drone_steps", "sum_pos_err", "max_pos_err", "min_barrier",
              "qp_solves", "qp_iters", "qp_infeasible", "qp_iter_cap")

DRONE_CF2X, DRONE_CF2P = 0, 1
PHYSICS_DYN, PHYSICS_DYN_GND_DRAG_DW = 0, 1
QP_OPTIMAL, QP_INFEASIBLE, QP_ITER_CAP = 0, 1, 2
CTRL_GEOMETRIC, CTRL_LQR_TORQUE, CTRL_LQR_OMEGA, CTRL_LQR_YANK, CTRL_DSLPID = 0, 1, 2, 3, 4
TRAJ_WAIT, TRAJ_CIRCLE, TRAJ_LEMNISCATE, TRAJ_TABLE = 0, 1, 2, 3
SEG_WAIT, SEG_CIRCLE, SEG_LEMNISCATE, SEG_LINE = 0, 1, 2, 3


class MdsError(RuntimeError):
    pass


class DroneParams(C.Structure):
    _fields_ = [(n, C.c_double) for n in (
        "m", "g", "kf", "km", "arm_l", "ixx", "iyy", "izz", "max_rpm", "max_thrust",
        "gnd_eff_coeff", "prop_radius", "gnd_eff_h_clip", "drag_xy", "drag_z", "dw1", "dw2", "dw3", "dw_dz_clip")] + [
        ("prop_x", C.c_double * 4), ("prop_y", C.c_double * 4),
        ("z_floor", C.c_double), ("dt_phys", C.c_double), ("dt_ctrl", C.c_double),
        ("substeps", C.c_int), ("drone_model", C.c_int), ("physics", C.c_int),
        ("cf2x_torque_sign", C.c_int), ("renormalize_quat", C.c_int), ("ground_clamp", C.c_int), ("x_frame_mixer", C.c_int)]


class State(C.Structure):
    _fields_ = [(n, C.c_void_p) for n in ("pos_wx", "quat", "vel_wy", "rpm", "wz")]


class PidState(C.Structure):
    _fields_ = [("a", C.c_void_p), ("b", C.c_void_p)]


class DslPidState(C.Structure):
    _fields_ = [("a", C.c_void_p), ("b", C.c_void_p), ("c", C.c_void_p)]


class DslPidGains(C.Structure):
    _fields_ = [(n, C.c_double * 3) for n in ("p_for", "i_for", "d_for", "p_tor", "i_tor", "d_tor")]


class GeoGains(C.Structure):
    _fields_ = [(n, C.c_double) for n in ("kp", "kv", "kr", "kw", "g_ctrl", "max_tilt")]


class LqrGains(C.Structure):
    _fields_ = [("K", C.c_double * 48), ("dim", C.c_int)]


class CbfParams(C.Structure):
    _fields_ = [("order", C.c_int), ("zscale", C.c_double), ("safety_radius", C.c_double),
                ("kcbf", C.c_double * 3), ("umax", C.c_double * 4), ("fmin", C.c_double),
                ("fmax", C.c_double), ("max_iter", C.c_int), ("no_state_bounds", C.c_int)]


class RlsCfg(C.Structure):
    _fields_ = [("m", C.c_int), ("target", C.c_int), ("predict_from_xtp1", C.c_int), ("normalize_gain", C.c_int),
                ("project", C.c_int), ("drones_per_env", C.c_int), ("dt", C.c_double), ("theta_code", C.c_ubyte * (16 * 12))]


class RolloutCfg(C.Structure):
    _fields_ = [("ctrl", C.c_int), ("use_cbf", C.c_int), ("num_obstacles", C.c_int),
                ("write_obs_every", C.c_int), ("stages", C.c_int), ("obstacles", C.c_double * (MAX_OBSTACLES * 4)),
                ("lqr_gain_planes_dev", C.c_void_p), ("traj_period", C.c_int)]


# numpy dtypes of the device-side trajectory tables (must match the C structs)
def traj_spec_dtype(real):
    import numpy as np
    return np.dtype([("kind", "i4"), ("seg_begin", "i4"), ("seg_count", "i4"), ("pad", "i4"), ("p", real, (8,))], align=True)


def traj_seg_dtype(real):
    import numpy as np
    return np.dtype([("kind", "i4"), ("has_rot", "i4"), ("t_end", real), ("dur", real),
                     ("p", real, (24,)), ("rot", real, (12,))], align=True)


_P = C.c_void_p
_I = C.c_int
_D = C.c_double
_PRM = C.POINTER(DroneParams)

# name -> argtypes (suffix-less); each exists as _f32 and _f64
_SIGS = {
    "mds_physics_step": [_PRM, State, _P, _P, _P, _I, _I, _P],
    "mds_physics_step_host": [_PRM, State, _P, _P, _P, _P, _I, _I, _P],
    "mds_obs_from_state": [_PRM, State, _P, _I, _P],
    "mds_traj_eval": [_P, _P, _D, _P, _I, _P],
    "mds_geometric_ctrl": [_PRM, C.POINTER(GeoGains), _P, _P, _P, _P, _I, _P],
    "mds_dslpid_ctrl": [_PRM, C.POINTER(DslPidGains), _P, _P, DslPidState, _P, _P, _I, _P],
    "mds_lqr_ctrl": [_PRM, C.POINTER(LqrGains), _I, _P, _P, _P, _P, PidState, _I, _P],
    "mds_lowlevel": [_PRM, _I, _P, _P, PidState, _P, _I, _P],
    "mds_rls_update": [C.POINTER(RlsCfg), _P, _P, _P, _P, _P, _I, _P],
    "mds_care_gains": [_I, C.POINTER(_D), C.POINTER(_D), _P, _P, _P, _I, _P],
    "mds_error_state": [_PRM, _I, _P, _P, _P, _I, _P],
    "mds_state_feedback": [_I, _P, _P, _P, _P, _P, _I, _P],
    "mds_dlqr_ctrl": [_PRM, _I, _P, _I, _P, _P, _P, _P, PidState, _I, _I, _P],
    "mds_cbf_qp": [_PRM, C.POINTER(CbfParams), _P, _P, _P, _P, _I, _P, _P, _P, _I, _I, _P],
    "mds_cbf_rows": [_PRM, C.POINTER(CbfParams), _P, _P, _P, _I, _P, _P, _I, _I, _P],
    "mds_cbf_prepare": [_PRM, _I, _D, _P, _P, _P, _I, _P],
    "mds_xdot_linear": [_PRM, _I, _P, _P, _I, _P],
    "mds_xdot_nonlinear": [_PRM, _D, _D, _D, _P, _P, _I, _P],
    "mds_linear_rollout": [_PRM, _P, _D, _P, _I, _I, _P],
    "mds_rollout": [_PRM, C.POINTER(RolloutCfg), C.POINTER(GeoGains), C.POINTER(LqrGains), C.POINTER(CbfParams),
                    State, PidState, C.POINTER(DslPidGains), DslPidState, _P, _P, _P, _P, _P, _P, _P, _D, _I, _I, _I, _P],
    "mds_learning_rollout": [_PRM, C.POINTER(RlsCfg), _I, _I, _I, State, PidState, _P, _P, _P, _P, _P, _P, _P, _P, _P, _D, _I, _I, _I, _P],
    "mds_learning_rollout_feedback": [_PRM, C.POINTER(RlsCfg), _I, _I, _I, State, PidState, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _D, _I, _I,
                                      _I, _P],
}
_PLAIN = {
    "mds_abi_version": ([], _I),
    "mds_last_error": ([], C.c_char_p),
    "mds_device_info": ([C.POINTER(_I)] * 4, _I),
    "mds_cbf_num_rows": ([_I, _I, _I], _I),
    "mds_rollout_plan": ([_I, _I], _I),
    "mds_fma_peak": ([_I, _I, C.POINTER(_D), _P], _I),
    "mds_device_alloc": ([C.c_size_t, C.POINTER(C.c_void_p)], _I),
    "mds_device_free": ([_P], _I),
    "mds_copy_to_device": ([_P, _P, C.c_size_t, _P], _I),
    "mds_copy_to_host": ([_P, _P, C.c_size_t, _P], _I),
    "mds_stream_synchronize": ([_P], _I),
}

EXPORTED_SYMBOLS = tuple(sorted([f"{k}_{s}" for k in _SIGS for s in ("f32", "f64")] + list(_PLAIN)))

_lib = None


def load_library():
    """Load (once) and return the ctypes handle; raises MdsError if it is not built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.isfile(LIB_PATH):
        raise MdsError(
            f"{LIB_PATH} not found: build it with `make -C {os.path.dirname(LIB_PATH)}` or "
            "`python -c 'import __graft_entry__ as g; g.build()'` (there is no CPU fallback)")
    lib = C.CDLL(LIB_PATH)
    for name, args in _SIGS.items():
        for suf in ("f32", "f64"):
            fn = getattr(lib, f"{name}_{suf}")
            fn.argtypes = args
            fn.restype = _I
    for name, (args, res) in _PLAIN.items():
        fn = getattr(lib, name)
        fn.argtypes = args
        fn.restype = res
    _lib = lib
    return lib


def suffix(dtype) -> str:
    import torch
    if dtype == torch.float32:
        return "f32"
    if dtype == torch.float64:
        return "f64"
    raise MdsError(f"unsupported dtype {dtype}: the kernels compute in float32 or float64")


def call(name, dtype, *args):
    """Invoke ``<name>_<f32|f64>`` and raise on a non-zero status."""
    lib = load_library()
    rc = getattr(lib, f"{name}_{suffix(dtype)}")(*args)
    if rc != 0:
        raise MdsError(f"{name}: status {rc}: {lib.mds_last_error().decode()}")


def ptr(t):
    """Device pointer of a tensor (None -> NULL)."""
    return None if t is None else C.c_void_p(t.data_ptr())


def stream_ptr(device=None):
    import torch
    return C.c_void_p(torch.cuda.current_stream(device).cuda_stream)


def require_cuda(t, name, dtype=None, shape=None):
    import torch
    if not isinstance(t, torch.Tensor) or not t.is_cuda:
        raise MdsError(f"{name} must be a CUDA tensor (no CPU path exists)")
    if not t.is_contiguous():
        raise MdsError(f"{name} must be contiguous")
    if dtype is not None and t.dtype != dtype:
        raise MdsError(f"{name} must have dtype {dtype}, got {t.dtype}")
    if shape is not None and tuple(t.shape) != tuple(shape):
        raise MdsError(f"{name} must have shape {tuple(shape)}, got {tuple(t.shape)}")
    return t


def device_info():
    lib = load_library()
    v = [_I(0) for _ in range(4)]
    rc = lib.mds_device_info(*[C.byref(x) for x in v])
    if rc != 0:
        raise MdsError(lib.mds_last_error().decode())
    return {"sm_count": v[0].value, "cc": (v[1].value, v[2].value), "l2_bytes": v[3].value}


def fma_peak_tflops(use_f64=False, iters=1 << 16):
    lib = load_library()
    out = _D(0)
    rc = lib.mds_fma_peak(int(use_f64), int(iters), C.byref(out), stream_ptr())
    if rc != 0:
        raise MdsError(lib.mds_last_error().decode())
    return out.value
