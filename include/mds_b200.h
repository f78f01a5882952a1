/*
 * mds_b200.h -- C ABI of the B200-native batched multi-drone hot path.
 *
 * Drop-in boundary for the per-step loop of JasonTStanley/MultiDroneSim
 *   traj(t) -> ctrl.compute(obs) -> qpTracker.compute_control(...) ->
 *   ctrl.compute_low_level(...) -> env.step(action)
 * (reference simulations/EnvGeometric.py:434-479, simulations/CBFTest.py:302-358).
 *
 * Conventions
 *   - Every entry point returns int: 0 = ok, < 0 = error (see MDS_ERR_*); nothing
 *     throws across the boundary; mds_last_error() gives a thread-local message.
 *   - Every pointer named *_dev / inside MdsState / MdsPidState is a DEVICE pointer
 *     (e.g. torch.Tensor.data_ptr()); structs of parameters are HOST pointers,
 *     copied by value into the launch.  No global / __constant__ state is kept.
 *   - `stream` is a cudaStream_t passed as void* (NULL = legacy default stream).
 *   - Suffix _f32 / _f64 selects the arithmetic type `Real` (float / double).
 *   - D = E * N drones, index d = e * N + n (env-major).  N <= MDS_MAX_DRONES_PER_ENV.
 *
 * State layout in HBM (structure of arrays, 128-bit planes, 17 Real per drone):
 *   pos_wx [D] Real4 = (px, py, pz, wx)      world position, body rate x
 *   quat   [D] Real4 = (qx, qy, qz, qw)      PyBullet xyzw order
 *   vel_wy [D] Real4 = (vx, vy, vz, wy)      world velocity, body rate y
 *   rpm    [D] Real4 = last clipped motor RPM
 *   wz     [D] Real  = body rate z
 * Observation layout (reference layout, array of 20 Real per drone; consumed at
 * reference utils/model_conversions.py:34-45,109-113):
 *   [0:3] pos, [3:7] quat xyzw, [7:10] rpy, [10:13] vel world, [13:16] ang vel WORLD,
 *   [16:20] last clipped RPM.
 */
#ifndef MDS_B200_H
#define MDS_B200_H

#ifdef __cplusplus
extern "C" {
#endif

#define MDS_ABI_VERSION 9
#define MDS_MAX_DRONES_PER_ENV 32
#define MDS_MAX_OBSTACLES 8
#define MDS_OBS_DIM 20
#define MDS_REF_DIM 11 /* pos3 vel3 acc3 yaw yaw_rate */

#define MDS_OK 0
#define MDS_ERR_ARG (-1)    /* bad argument (null pointer, size, enum) */
#define MDS_ERR_LAUNCH (-2) /* CUDA launch / runtime error */
#define MDS_ERR_UNSUPPORTED (-3)

/* gym-pybullet-drones DroneModel / Physics (reference simulations/EnvGeometric.py:9,21-22) */
enum { MDS_DRONE_CF2X = 0, MDS_DRONE_CF2P = 1 };
enum { MDS_PHYSICS_DYN = 0, MDS_PHYSICS_DYN_GND_DRAG_DW = 1 };

/* per-env QP status written by mds_cbf_qp / mds_rollout (SURVEY.md 8b) */
enum { MDS_QP_OPTIMAL = 0, MDS_QP_INFEASIBLE = 1, MDS_QP_ITER_CAP = 2 };

/* controller stack selected in mds_rollout */
enum {
  MDS_CTRL_GEOMETRIC = 0,   /* control/geometric.py -> input_to_action              */
  MDS_CTRL_LQR_TORQUE = 1,  /* control/lqr/lqr_controller.py (12-dim) -> mixer     */
  MDS_CTRL_LQR_OMEGA = 2,   /* lqr_omega_controller.py (9-dim) + ThrustOmega PID   */
  MDS_CTRL_LQR_YANK = 3,    /* lqr_YO_controller.py (10-dim) + YankOmega PID       */
  MDS_CTRL_DSLPID = 4       /* upstream DSLPIDControl (MultiDroneExample.py:85-114): target = reference pos / vel / yaw / yaw rate */
};

/* trajectory generator kinds (reference trajectories/ package) */
enum {
  MDS_TRAJ_WAIT = 0,       /* LineTrajectory.py:4-14   p = {x,y,z,yaw}                              */
  MDS_TRAJ_CIRCLE = 1,     /* Circle.py:5-45           p = {r,v,cx,cy,cz,yaw_rate}                  */
  MDS_TRAJ_LEMNISCATE = 2, /* Lemniscate.py:3-63       p = {a,omega,cx,cy,cz,yaw_rate,phase_shift}  */
  MDS_TRAJ_TABLE = 3       /* CompoundTrajectory.py:5-40 over a segment table (Line/Wait/Circle/...) */
};
enum { MDS_SEG_WAIT = 0, MDS_SEG_CIRCLE = 1, MDS_SEG_LEMNISCATE = 2, MDS_SEG_LINE = 3 };

/* Drone + integrator constants: upstream BaseAviary attributes the reference reads
 * (env.M, env.J, env.G, env.KF, env.KM, env.L, env.MAX_RPM, env.MAX_THRUST, ...). */
typedef struct MdsDroneParams {
  double m, g, kf, km, arm_l;
  double ixx, iyy, izz;
  double max_rpm, max_thrust;
  double gnd_eff_coeff, prop_radius, gnd_eff_h_clip;
  double drag_xy, drag_z;
  double dw1, dw2, dw3;
  double dw_dz_clip;           /* lower clip of the vertical separation in the downwash magnitude (0 = upstream-exact, singular at dz -> 0+) */
  double prop_x[4], prop_y[4]; /* prop link offsets, body frame */
  double z_floor;              /* ground-plane contact clamp height */
  double dt_phys;              /* PYB_TIMESTEP  */
  double dt_ctrl;              /* CTRL_TIMESTEP */
  int substeps;                /* PYB_STEPS_PER_CTRL */
  int drone_model;             /* MDS_DRONE_*   */
  int physics;                 /* MDS_PHYSICS_* */
  int cf2x_torque_sign;        /* sign applied to the CF2X roll torque (SURVEY A.2 switch) */
  int renormalize_quat;        /* 0 = upstream (no renormalisation) */
  int ground_clamp;            /* 1 = clamp z at z_floor (composite mode default) */
  int x_frame_mixer;           /* 0 = the reference's PLUS-frame mixer for every model (utils/model_conversions.py:74-77,90-93);
                                  1 = for CF2X use the X-frame allocation the CF2X dynamics apply (SURVEY 8f-4 extension) */
} MdsDroneParams;

typedef struct MdsState {
  void* pos_wx; void* quat; void* vel_wy; void* rpm; void* wz;
} MdsState;

/* ThrustOmegaController state: control/low_level/thrust_omega_ctrl.py:65-75 */
typedef struct MdsPidState {
  void* a; /* Real4[D] = (last_wx, last_wy, last_wz, integral_x) */
  void* b; /* Real2[D] = (integral_y, integral_z) */
} MdsPidState;

/* upstream DSLPIDControl state (SURVEY.md App. A.5): integral_pos_e, last_rpy, integral_rpy_e */
typedef struct MdsDslPidState {
  void* a; /* Real4[D] = (integral_pos_e xyz, last_roll)                              */
  void* b; /* Real4[D] = (last_pitch, last_yaw, integral_rpy_e x, integral_rpy_e y)   */
  void* c; /* Real [D] = integral_rpy_e z                                             */
} MdsDslPidState;
/* upstream DSLPIDControl gains (P/I/D of the position loop "FOR" and the attitude loop "TOR"; MultiDroneExample.py:87-92
 * overrides them with half of the upstream defaults) */
typedef struct MdsDslPidGains {
  double p_for[3], i_for[3], d_for[3], p_tor[3], i_tor[3], d_tor[3];
} MdsDslPidGains;

/* control/geometric.py:14-23 */
typedef struct MdsGeoGains {
  double kp, kv, kr, kw, g_ctrl, max_tilt;
} MdsGeoGains;

/* LQR gain K (4 x dim row-major, dim in {12, 9, 10}); control/lqr/ package */
typedef struct MdsLqrGains {
  double K[48];
  int dim;
} MdsLqrGains;

/* cbf/cbf.py:545-580 (DroneCBF) */
typedef struct MdsCbfParams {
  int order;             /* 2 (xdim 9) or 3 (xdim 10) */
  double zscale;         /* c */
  double safety_radius;
  double kcbf[3];        /* place_poles gain, order entries */
  double umax[4];
  double fmin, fmax;     /* order-3 force-bound rows (cbf.py:446-464) */
  int max_iter;          /* iteration cap of the in-shared-memory active-set solver (0 = default 64); a solve that exceeds it, or
                          * whose active set outgrows its 12 slots, is repeated by the scratch solver (no cap on the active set) */
  int no_state_bounds;   /* 0 = CBF(do_state_bounds=True), the reference's default: order-3 force-bound rows on column 4i+3
                          * (cbf.py:446-476); 1 = do_state_bounds=False: those rows are not emitted */
} MdsCbfParams;

/* per-drone trajectory descriptor, 48 B (f32) / 80 B (f64).  MDS_TRAJ_TABLE: segments
 * [seg_begin, seg_begin + seg_count); pad != 0 marks a stand-alone single segment (no compound end clamp) */
typedef struct MdsTrajSpecF32 { int kind, seg_begin, seg_count, pad; float p[8]; } MdsTrajSpecF32;
typedef struct MdsTrajSpecF64 { int kind, seg_begin, seg_count, pad; double p[8]; } MdsTrajSpecF64;
/* shared segment table entry for MDS_TRAJ_TABLE.  t_end = cumulative end time.
 * LINE p[]: start3, v0 3, sgn_init3, cruise3, sgn_end3, end3, vf3, time_init, time_middle, total_time */
typedef struct MdsTrajSegF32 { int kind; int has_rot; float t_end; float dur; float p[24]; float rot[12]; } MdsTrajSegF32;
typedef struct MdsTrajSegF64 { int kind; int has_rot; double t_end; double dur; double p[24]; double rot[12]; } MdsTrajSegF64;

/* rollout statistics (one block of doubles, accumulated with atomics) */
enum {
  MDS_STAT_DRONE_STEPS = 0, MDS_STAT_SUM_POS_ERR = 1, MDS_STAT_MAX_POS_ERR = 2,
  MDS_STAT_MIN_BARRIER = 3, MDS_STAT_QP_SOLVES = 4, MDS_STAT_QP_ITERS = 5,
  MDS_STAT_QP_INFEASIBLE = 6, MDS_STAT_QP_ITER_CAP = 7, MDS_STAT_COUNT = 8
};

typedef struct MdsRolloutCfg {
  int ctrl;            /* MDS_CTRL_*                                       */
  int use_cbf;         /* 0/1; requires ctrl LQR_OMEGA (order 2) or LQR_YANK (order 3) */
  int num_obstacles;   /* obstacles shared by all envs, <= MDS_MAX_OBSTACLES (the reference itself fails beyond N, quirk B14) */
  int write_obs_every; /* 0 = only after the last step; k>0 = log obs every k steps     */
  int stages;          /* launch plan for the K control steps:
                          0      whole steps, plan chosen by mds_rollout_plan(E, N) (currently always 6)
                          6      all K steps in ONE launch: observation and body rates stay in registers from step to
                                 step (environments are independent and a lane group owns its environment)
                          4      whole steps as two launches each (controller kernel, physics kernel)
                          1      controller kernel only (action_dev <- controller stack at obs_dev; env does not advance)
                          2      physics kernel only (env advances under action_dev)
                          A call with 1 then a call with 2 (K = 1 each) is one step of plan 4: repeated K times, they let
                          a caller replay a rollout launch by launch with its own CUDA events.  Any other value is an error. */
  double obstacles[MDS_MAX_OBSTACLES * 4]; /* cx, cy, cz, r (r < 0: vertical cylinder of radius |r|) */
  const void* lqr_gain_planes_dev; /* optional, LQR controllers: a gain per drone, [4*dim][D] planes of Real (DecentralizedLQR*.K,
                                      simulations/CBFTest.py:319-321 `--controller dlqr`); NULL = MdsLqrGains.K for every drone */
  int traj_period;     /* 0 = one trajectory descriptor per drone (no assumption); N (the drone count) = every environment flies
                          the references of environment 0: specs_dev[d] equals specs_dev[d mod N] for every drone d.  The caller
                          guarantees it; plan 6 then evaluates each reference once per block and step instead of once per drone
                          (fp32, N = 8, LQR_OMEGA / LQR_YANK; the results are the same bits) */
} MdsRolloutCfg;

/* ---- library ------------------------------------------------------------------ */
int mds_abi_version(void);
const char* mds_last_error(void);
int mds_device_info(int* sm_count, int* cc_major, int* cc_minor, int* l2_bytes);

/* ---- plain-host helpers (for callers without a CUDA-aware array library; the reference is numpy-only) ---- */
#include <stddef.h>
int mds_device_alloc(size_t bytes, void** out_dev); /* zero-filled device buffer */
int mds_device_free(void* dev);
int mds_copy_to_device(void* dst_dev, const void* src_host, size_t bytes, void* stream);
int mds_copy_to_host(void* dst_host, const void* src_dev, size_t bytes, void* stream);
int mds_stream_synchronize(void* stream);

/* ---- env step: replaces CtrlAviary.step (call sites EnvGeometric.py:431,469) ----- */
/* clip RPM to [0, max_rpm]; `substeps` explicit DYN / DYN_GND_DRAG_DW updates; write obs.
 * ext_force_dev: optional [D*3] world-frame force per drone (wind, EnvGeometric.py:463-467). */
int mds_physics_step_f32(const MdsDroneParams* prm, MdsState st, const float* action_dev,
                         const float* ext_force_dev, float* obs_dev, int E, int N, void* stream);
int mds_physics_step_f64(const MdsDroneParams* prm, MdsState st, const double* action_dev,
                         const double* ext_force_dev, double* obs_dev, int E, int N, void* stream);
/* HOST-array form of the same call, the literal `obs = env.step(action)` of the reference's loops
 * (EnvGeometric.py:469): action_host [D*4] -> H2D -> step -> D2H -> obs_host [D*20]; synchronous on `stream`.
 * action_dev / obs_dev are the library-side device staging buffers (caller-owned). */
int mds_physics_step_host_f32(const MdsDroneParams* prm, MdsState st, const float* action_host, float* action_dev,
                              float* obs_dev, float* obs_host, int E, int N, void* stream);
int mds_physics_step_host_f64(const MdsDroneParams* prm, MdsState st, const double* action_host, double* action_dev,
                              double* obs_dev, double* obs_host, int E, int N, void* stream);
/* (re)build obs from state without stepping (reset(); ang vel = R w) */
int mds_obs_from_state_f32(const MdsDroneParams* prm, MdsState st, float* obs_dev, int D, void* stream);
int mds_obs_from_state_f64(const MdsDroneParams* prm, MdsState st, double* obs_dev, int D, void* stream);

/* ---- trajectories: replaces trajs[j](t) (EnvGeometric.py:437) -------------------- */
int mds_traj_eval_f32(const MdsTrajSpecF32* specs_dev, const MdsTrajSegF32* segs_dev, double t,
                      float* ref_dev, int D, void* stream);
int mds_traj_eval_f64(const MdsTrajSpecF64* specs_dev, const MdsTrajSegF64* segs_dev, double t,
                      double* ref_dev, int D, void* stream);

/* ---- controllers: replace ctrl[j].compute(obs[j]) -------------------------------- */
/* GeometricControl.compute (control/geometric.py:59-115) + input_to_action.  u_out optional. */
int mds_geometric_ctrl_f32(const MdsDroneParams* prm, const MdsGeoGains* gains, const float* obs_dev,
                           const float* ref_dev, float* action_dev, float* u_dev, int D, void* stream);
int mds_geometric_ctrl_f64(const MdsDroneParams* prm, const MdsGeoGains* gains, const double* obs_dev,
                           const double* ref_dev, double* action_dev, double* u_dev, int D, void* stream);
/* upstream DSLPIDControl.computeControlFromState (call site MultiDroneExample.py:111-114), one drone per thread.
 * target_dev [D*12] = target_pos3, target_rpy3, target_vel3, target_rpy_rates3; pos_e_dev optional [D*3]. */
int mds_dslpid_ctrl_f32(const MdsDroneParams* prm, const MdsDslPidGains* gains, const float* obs_dev, const float* target_dev,
                        MdsDslPidState state, float* action_dev, float* pos_e_dev, int D, void* stream);
int mds_dslpid_ctrl_f64(const MdsDroneParams* prm, const MdsDslPidGains* gains, const double* obs_dev, const double* target_dev,
                        MdsDslPidState state, double* action_dev, double* pos_e_dev, int D, void* stream);
/* LQR*.compute(obs, skip_low_level): u = -K e (+ hover), capped as each variant does.
 * variant = MDS_CTRL_LQR_*; action_dev may be NULL (skip_low_level=True).  For LQR_TORQUE the
 * action is the mixer output; for LQR_OMEGA / LQR_YANK it runs the inner PID (pid required). */
int mds_lqr_ctrl_f32(const MdsDroneParams* prm, const MdsLqrGains* gains, int variant, const float* obs_dev,
                     const float* ref_dev, float* u_dev, float* action_dev, MdsPidState pid, int D, void* stream);
int mds_lqr_ctrl_f64(const MdsDroneParams* prm, const MdsLqrGains* gains, int variant, const double* obs_dev,
                     const double* ref_dev, double* u_dev, double* action_dev, MdsPidState pid, int D, void* stream);
/* ctrl.compute_low_level(u, obs, idx): ThrustOmega / YankOmega inner loop -> RPM */
int mds_lowlevel_f32(const MdsDroneParams* prm, int variant, const float* u_dev, const float* obs_dev,
                     MdsPidState pid, float* action_dev, int D, void* stream);
int mds_lowlevel_f64(const MdsDroneParams* prm, int variant, const double* u_dev, const double* obs_dev,
                     MdsPidState pid, double* action_dev, int D, void* stream);

/* ---- CBF-QP: replaces DroneQPTracker.compute_control (cbf/qptracker.py:22-34) ------ */
/* xdes_dev [E*N*xdim]; u_nom_dev / u_safe_dev [E*N*4]; obstacles_dev [n_obs*4] = cx,cy,cz,r
 * (shared by all envs; r > 0: sphere as cbf/cbf.py:380-383; r < 0: vertical cylinder of radius |r|, unbounded
 * height, through (cx, cy) -- builder extension, the reference has spheres only) ; status_dev [E] int32 ; iters_dev [E] int32 (may be NULL).
 * status: MDS_QP_OPTIMAL -> u_safe is the QP's minimiser; MDS_QP_INFEASIBLE / MDS_QP_ITER_CAP -> u_safe = u_nom (the reference's
 * except branch, cbf/qptracker.py:30-34,105-114).  The solve has three tiers: (1) every drone projects onto its most violated
 * single-drone row (obstacle rows, +-umax box) in registers and the step ends there if no row is violated at the projected
 * point; (2) otherwise the environment's lane group runs a dual active-set solve in shared memory (<= 12 active rows,
 * MdsCbfParams.max_iter iterations); (3) a solve that outgrows (2), or whose factor breaks down, is repeated in a per-device
 * scratch pool with room for 3 N active rows, the number of coupled variables (no cap), scalar part in double.  ITER_CAP is
 * therefore only ever the scratch solver's own iteration limit (16 * 3N + 64).  The pool is allocated at the first CBF call
 * on a device (make that call outside any stream capture). */
int mds_cbf_qp_f32(const MdsDroneParams* prm, const MdsCbfParams* cbf, const float* obs_dev,
                   const float* xdes_dev, const float* u_nom_dev, const float* obstacles_dev, int n_obs,
                   float* u_safe_dev, int* status_dev, int* iters_dev, int E, int N, void* stream);
int mds_cbf_qp_f64(const MdsDroneParams* prm, const MdsCbfParams* cbf, const double* obs_dev,
                   const double* xdes_dev, const double* u_nom_dev, const double* obstacles_dev, int n_obs,
                   double* u_safe_dev, int* status_dev, int* iters_dev, int E, int N, void* stream);
/* dense G [E*m*4N], h [E*m] exactly as CBF._build_ineq_const (cbf/cbf.py:308-367); parity aid */
int mds_cbf_rows_f32(const MdsDroneParams* prm, const MdsCbfParams* cbf, const float* obs_dev,
                     const float* xdes_dev, const float* obstacles_dev, int n_obs, float* G_dev, float* h_dev,
                     int E, int N, void* stream);
int mds_cbf_rows_f64(const MdsDroneParams* prm, const MdsCbfParams* cbf, const double* obs_dev,
                     const double* xdes_dev, const double* obstacles_dev, int n_obs, double* G_dev, double* h_dev,
                     int E, int N, void* stream);
int mds_cbf_num_rows(int order, int N, int n_obs);
/* the glue the reference's callers do around the QP (simulations/CBFTest.py:339-343, CBFTestOrd3.py:344-347):
 * u[:,0] -= u0_offset (in place) and xdes = [0, 0, yaw, (m g,) vel, pos] from the reference samples */
int mds_cbf_prepare_f32(const MdsDroneParams* prm, int order, double u0_offset, const float* ref_dev, float* u_inout_dev,
                        float* xdes_dev, int D, void* stream);
int mds_cbf_prepare_f64(const MdsDroneParams* prm, int order, double u0_offset, const double* ref_dev, double* u_inout_dev,
                        double* xdes_dev, int D, void* stream);

/* ---- model comparison: replaces the loop of simulations/CompareModels.py:48-55 ------ */
/* kind 12: LinearizedModel.calc_xdot_from_obs; 9 / 10: builder-defined (quirk B23) */
int mds_xdot_linear_f32(const MdsDroneParams* prm, int kind, const float* obs_dev, float* xdot_dev, int D, void* stream);
int mds_xdot_linear_f64(const MdsDroneParams* prm, int kind, const double* obs_dev, double* xdot_dev, int D, void* stream);
/* roll_out_linear_system (simulations/CompareModels.py:82-95): the 12-dim linear model driven by the logged RPMs as
 * zero-order-hold inputs, advanced exactly over each log interval dt (the reference uses scipy RK45).
 * obs_log_dev [T][D*20] (e.g. the obs_log of mds_rollout) -> x_dev [T][D*12], x_dev[0] = first logged state. */
int mds_linear_rollout_f32(const MdsDroneParams* prm, const float* obs_log_dev, double dt, float* x_dev, int T, int D, void* stream);
int mds_linear_rollout_f64(const MdsDroneParams* prm, const double* obs_log_dev, double dt, double* x_dev, int T, int D, void* stream);
/* QuadrotorDynamics.dynamics via action_to_input / obs_to_geo_model / geo_x_dot_to_linear; J = diag(jx,jy,jz) */
int mds_xdot_nonlinear_f32(const MdsDroneParams* prm, double jx, double jy, double jz, const float* obs_dev, float* xdot_dev, int D, void* stream);
int mds_xdot_nonlinear_f64(const MdsDroneParams* prm, double jx, double jy, double jz, const double* obs_dev, double* xdot_dev, int D, void* stream);

/* ---- K-step rollout.  Default plan: ONE launch for all K control steps -- every lane group runs its own environment
 * forward (reference -> tracking controller -> CBF-QP -> inner loop -> physics sub-steps) with the observation and
 * the body rates in registers; HBM sees the initial load, the PID state, the log slots that are due and the final
 * store.  Other plans (MdsRolloutCfg.stages): two launches per step, single kernels.
 * Everything is enqueued on `stream` with no host synchronisation.
 * obs_dev [D*20] in/out (observation before the first / after the last step); action_dev [D*4] scratch;
 * ext_force_dev optional [D*3] constant world-frame force per drone (wind, EnvGeometric.py:463-467);
 * obs_log_dev optional [K/write_obs_every][D*20]; stats_dev optional [MDS_STAT_COUNT] doubles (accumulated).
 * With the CBF filter the library keeps a per-device scratch pool for QPs whose active set outgrows the in-kernel
 * workspace (allocated at the first such call: make that call outside any stream capture). */
int mds_rollout_f32(const MdsDroneParams* prm, const MdsRolloutCfg* cfg, const MdsGeoGains* geo,
                    const MdsLqrGains* lqr, const MdsCbfParams* cbf, MdsState st, MdsPidState pid,
                    const MdsDslPidGains* dsl, MdsDslPidState dsl_state, const MdsTrajSpecF32* specs_dev, const MdsTrajSegF32* segs_dev, float* obs_dev, float* action_dev,
                    const float* ext_force_dev, float* obs_log_dev, double* stats_dev, double t0, int K, int E, int N, void* stream);
int mds_rollout_f64(const MdsDroneParams* prm, const MdsRolloutCfg* cfg, const MdsGeoGains* geo,
                    const MdsLqrGains* lqr, const MdsCbfParams* cbf, MdsState st, MdsPidState pid,
                    const MdsDslPidGains* dsl, MdsDslPidState dsl_state, const MdsTrajSpecF64* specs_dev, const MdsTrajSegF64* segs_dev, double* obs_dev, double* action_dev,
                    const double* ext_force_dev, double* obs_log_dev, double* stats_dev, double t0, int K, int E, int N, void* stream);

/* ---- decentralised LQR with per-drone learned models (SURVEY 8(f)3): control/dlqr/ ------------------------- */
/* regression target of one recursive-least-squares step */
enum {
  MDS_RLS_TARGET_PREDICT = 0, /* x_{t+1} - forward_predict(...)   (theta_update / theta_update2, decentralized_lqr_omega.py:110-139) */
  MDS_RLS_TARGET_XDOT = 1     /* est_x_dot(x_{t+1}, phi) - theta' phi (approx_theta_update, decentralized_lqr.py:185-228)             */
};
/* project_theta (decentralized_lqr.py:230-240): never / once after the update (12-dim theta_update :183) / inside the
 * per-robot loop (approx_theta_update :216: robots after the first of an env are also projected BEFORE their update) */
enum { MDS_RLS_PROJECT_NONE = 0, MDS_RLS_PROJECT_AFTER = 1, MDS_RLS_PROJECT_LOOP = 2 };
typedef struct MdsRlsCfg {
  int m;                  /* model state dimension: 9 (omega), 10 (yank-omega), 12 (torque); inputs n = 4            */
  int target;             /* MDS_RLS_TARGET_*                                                                        */
  int predict_from_xtp1;  /* PREDICT: start the prediction at x_{t+1} (omega / yank-omega variants, :134) not phi[:m] */
  int normalize_gain;     /* 1: L = P phi / (1 + phi' P phi); 0: L = P phi with P = V^-1 (theta_update2, :119-122)    */
  int project;            /* MDS_RLS_PROJECT_*                                                                       */
  int drones_per_env;     /* N (only read by MDS_RLS_PROJECT_LOOP)                                                   */
  double dt;              /* env.CTRL_TIMESTEP                                                                       */
  unsigned char theta_code[16 * 12]; /* project_theta per entry of theta [(m+4)][m] row-major: 0 zero, 1 keep, 2 one */
} MdsRlsCfg;
/* One RLS step for every drone.  phi_dev [D][m+4] = [e_t, u_t], xtp1_dev [D][m] = e_{t+1} (row-major per drone);
 * theta_dev [(m+4)*m][D] and P_dev [(m+4)*(m+4)][D] are PLANES (entry k of drone d at [k*D + d]), updated in place;
 * resid_dev optional [D][m] receives the regression residual. */
int mds_rls_update_f32(const MdsRlsCfg* cfg, const float* phi_dev, const float* xtp1_dev, float* theta_dev, float* P_dev,
                       float* resid_dev, int D, void* stream);
int mds_rls_update_f64(const MdsRlsCfg* cfg, const double* phi_dev, const double* xtp1_dev, double* theta_dev, double* P_dev,
                       double* resid_dev, int D, void* stream);
/* error_state of the LQR family (decentralized_lqr_omega.py:174-183, lqr_omega_controller.py:97-110): obs + reference
 * sample -> e_dev [D][dim], dim = 12 / 9 / 10 for variant MDS_CTRL_LQR_TORQUE / _OMEGA / _YANK */
int mds_error_state_f32(const MdsDroneParams* prm, int variant, const float* obs_dev, const float* ref_dev, float* e_dev, int D, void* stream);
int mds_error_state_f64(const MdsDroneParams* prm, int variant, const double* obs_dev, const double* ref_dev, double* e_dev, int D, void* stream);
/* The same error state on model STATE vectors x_dev, xdes_dev [D][dim] (decentralized_lqr_omega.py:174-183 as called with
 * states, YOState.error_state decentralized_yolqr_crazyflie.py:88-102; attitude error in closed form, |pitch| <= pi/2) ->
 * e_dev [D][dim] (optional) and, with K_dev [4*dim][D] planes, u_dev [D*4] = -K_d e_d (optional; no hover offset:
 * DecentralizedYOLQRCrazyflie.compute :350-362, the FedCE wrapper's lqr_control). */
int mds_state_feedback_f32(int variant, const float* K_dev, const float* x_dev, const float* xdes_dev, float* e_dev, float* u_dev, int D, void* stream);
int mds_state_feedback_f64(int variant, const double* K_dev, const double* x_dev, const double* xdes_dev, double* e_dev, double* u_dev, int D, void* stream);
/* mds_lqr_ctrl with a gain per drone (DecentralizedLQR*.compute).  coupled = 0: u_d = -K_d e_d, K_dev [4*dim][D] planes.
 * coupled = 1: u_d = -sum_j K_{d,j} e_j over the N drones j of d's environment, K_dev [N][4*dim][D] (source-major):
 * the 12-dim reference couples robots 0 and 1 through off-diagonal blocks of Q (decentralized_lqr.py:44-53), so its K
 * is a full 4N x 12N matrix.  Same outputs and inner loop as mds_lqr_ctrl. */
int mds_dlqr_ctrl_f32(const MdsDroneParams* prm, int variant, const float* K_dev, int coupled, const float* obs_dev, const float* ref_dev,
                      float* u_dev, float* action_dev, MdsPidState pid, int E, int N, void* stream);
int mds_dlqr_ctrl_f64(const MdsDroneParams* prm, int variant, const double* K_dev, int coupled, const double* obs_dev, const double* ref_dev,
                      double* u_dev, double* action_dev, MdsPidState pid, int E, int N, void* stream);

/* The system-identification loop of the decentralised LQR (learning phases of simulations/CBFTest.py:150-265,
 * CBFTestOrd3.py:150-270) for K control steps in ONE launch.  Step k of every drone: ref_k = trajectory at t0 + k*dt_ctrl,
 * e_t = error state against ref_k, inner loop (variant MDS_CTRL_LQR_OMEGA: ThrustOmega, _YANK: YankOmega) on the caller's
 * excitation inputs_dev[k] [D*4], physics step (ext_force_dev optional [D*3], as mds_physics_step), e_t+1 against the same
 * ref_k, and -- if k >= learn_from -- one RLS step of `rls` with phi = [e_t, u_k], x1 = e_t+1 (rls->m = 9 with OMEGA, 10
 * with YANK; project_theta at m = 10 only; drones_per_env = N).  The same results as that loop over mds_traj_eval,
 * mds_error_state, mds_lowlevel, mds_physics_step and mds_rls_update.  theta_dev / P_dev planes as mds_rls_update, updated in place; resid_dev optional
 * [D][m] (the residual of the last update, untouched when none ran); obs_dev [D*20] in/out; PID state in/out;
 * obs_log_dev optional [K/write_obs_every][D*20].  K = 0 launches nothing (inputs_dev may then be NULL). */
int mds_learning_rollout_f32(const MdsDroneParams* prm, const MdsRlsCfg* rls, int variant, int learn_from, int write_obs_every, MdsState st,
                             MdsPidState pid, const MdsTrajSpecF32* specs_dev, const MdsTrajSegF32* segs_dev, const float* inputs_dev,
                             float* theta_dev, float* P_dev, float* resid_dev, float* obs_dev, const float* ext_force_dev, float* obs_log_dev,
                             double t0, int K, int E, int N, void* stream);
int mds_learning_rollout_f64(const MdsDroneParams* prm, const MdsRlsCfg* rls, int variant, int learn_from, int write_obs_every, MdsState st,
                             MdsPidState pid, const MdsTrajSpecF64* specs_dev, const MdsTrajSegF64* segs_dev, const double* inputs_dev,
                             double* theta_dev, double* P_dev, double* resid_dev, double* obs_dev, const double* ext_force_dev, double* obs_log_dev,
                             double t0, int K, int E, int N, void* stream);
/* mds_learning_rollout under each drone's own gain (closed-loop exploration): the inner loop flies
 * u_k = -K_d e_t (+ m g unless MDS_CTRL_LQR_YANK; MDS_CTRL_LQR_OMEGA caps the thrust as mds_dlqr_ctrl does) + inputs_dev[k],
 * and the RLS step takes phi = [e_t, u_k] with that applied u_k.  inputs_dev[k] [D*4] are perturbations of the law (with
 * LQR_YANK, entry 0 perturbs the yank).  gain_dev [4*m][D]: the uncoupled planes of mds_dlqr_ctrl, non-NULL, read once
 * per launch (constant for its K steps).  The same results as the mds_learning_rollout loop with mds_dlqr_ctrl (no
 * action) and an add before mds_lowlevel; every other argument and check is mds_learning_rollout's. */
int mds_learning_rollout_feedback_f32(const MdsDroneParams* prm, const MdsRlsCfg* rls, int variant, int learn_from, int write_obs_every,
                                      MdsState st, MdsPidState pid, const MdsTrajSpecF32* specs_dev, const MdsTrajSegF32* segs_dev,
                                      const float* inputs_dev, const float* gain_dev, float* theta_dev, float* P_dev, float* resid_dev,
                                      float* obs_dev, const float* ext_force_dev, float* obs_log_dev, double t0, int K, int E, int N, void* stream);
int mds_learning_rollout_feedback_f64(const MdsDroneParams* prm, const MdsRlsCfg* rls, int variant, int learn_from, int write_obs_every,
                                      MdsState st, MdsPidState pid, const MdsTrajSpecF64* specs_dev, const MdsTrajSegF64* segs_dev,
                                      const double* inputs_dev, const double* gain_dev, double* theta_dev, double* P_dev, double* resid_dev,
                                      double* obs_dev, const double* ext_force_dev, double* obs_log_dev, double t0, int K, int E, int N,
                                      void* stream);
/* The same loop for the 12-dim torque-level model (MDS_CTRL_LQR_TORQUE error state, decentralized_lqr.py), which has no inner
 * loop and no PID state: step k flies input_to_action(u_k), which clamps u_k[0] >= 0 in place, and the RLS step takes
 * phi = [e_t, u_k] with the clamped u_k.  gain_dev NULL: open loop, u_k = inputs_dev[k] [D*4] = [f, tx, ty, tz].  Otherwise
 * u_k = max(-sum_j K_dj e_j + m g, 0 on the thrust) + inputs_dev[k] (mds_dlqr_ctrl's law and clamp, then the perturbation),
 * the gain read once per launch: coupled = 0: K_dj = 0 for j != d, gain_dev [48][D] planes (staged with theta and P);
 * coupled = 1: the robot-coupled gain_dev [N][48][D] planes of mds_dlqr_ctrl (read from device memory every step).
 * rls->m = 12, rls->project AFTER (theta_update) or LOOP (approx_theta_update): both methods project theta.  Every other
 * argument and check is mds_learning_rollout's; error messages start with "learning_rollout_torque: ". */
int mds_learning_rollout_torque_f32(const MdsDroneParams* prm, const MdsRlsCfg* rls, int learn_from, int write_obs_every, MdsState st,
                                    const MdsTrajSpecF32* specs_dev, const MdsTrajSegF32* segs_dev, const float* inputs_dev, const float* gain_dev,
                                    int coupled, float* theta_dev, float* P_dev, float* resid_dev, float* obs_dev, const float* ext_force_dev,
                                    float* obs_log_dev, double t0, int K, int E, int N, void* stream);
int mds_learning_rollout_torque_f64(const MdsDroneParams* prm, const MdsRlsCfg* rls, int learn_from, int write_obs_every, MdsState st,
                                    const MdsTrajSpecF64* specs_dev, const MdsTrajSegF64* segs_dev, const double* inputs_dev, const double* gain_dev,
                                    int coupled, double* theta_dev, double* P_dev, double* resid_dev, double* obs_dev, const double* ext_force_dev,
                                    double* obs_log_dev, double t0, int K, int E, int N, void* stream);

/* compute_controller (decentralized_lqr_omega.py:185-204): K_d = R^-1 B_d' X_d, X_d the stabilising solution of the
 * continuous-time algebraic Riccati equation of drone d's learned model theta_d = [A_d, B_d]^T, for diagonal Q (q_diag [m])
 * and R (r_diag [4], host arrays).  One warp per drone, double precision inside (matrix sign function; the reference calls
 * scipy.linalg.solve_continuous_are on the host).  theta_dev [(m+4)*m][D] planes -> K_dev [4*m][D] planes;
 * status_dev optional [D]: 0 ok, 1 no stabilising solution found (K_d left untouched). */
int mds_care_gains_f32(int m, const double* q_diag, const double* r_diag, const float* theta_dev, float* K_dev, int* status_dev, int D, void* stream);
int mds_care_gains_f64(int m, const double* q_diag, const double* r_diag, const double* theta_dev, double* K_dev, int* status_dev, int D, void* stream);

/* compute_controller of the 12-dim model when Q couples robots 0 and 1 of every environment (decentralized_lqr.py:44-53,
 * 300-317): the environment's Q is kron(I_N, diag(q_diag)) plus the cross block q_cross [m*m] (row-major, host array;
 * Q[k][m + l] = Q[m + l][k] = q_cross[k*m + l], robot 0's state k against robot 1's state l), R = kron(I_N, diag(r_diag)).
 * The environment's stabilising solution is block diagonal over the drones {0, 1}, {2}, ..., {N-1}: one warp solves each
 * 24-state pair problem and each 12-state single problem in double.  theta_dev [(m+4)*m][D] planes -> K_dev the robot-coupled
 * [N][4*m][D] planes that mds_dlqr_ctrl (coupled = 1) and mds_learning_rollout_torque read (entry (j, i*m + k, d = e*N + r) =
 * K_e[4r + i][m j + k]); a solved drone's entries for source drones outside its problem are written as zeros.
 * status_dev optional [D]: 0 ok, 1 the drone's problem has no stabilising solution found (its entries left untouched; both
 * drones of a failed pair).  Refuses (MDS_ERR_ARG) m != 12, N outside [2, MDS_MAX_DRONES_PER_ENV], E < 1, null pointers,
 * non-positive q or r, and a cross block for which the pair's Q is not positive semidefinite. */
int mds_care_gains_coupled_f32(int m, const double* q_diag, const double* r_diag, const double* q_cross, const float* theta_dev, float* K_dev,
                               int* status_dev, int E, int N, void* stream);
int mds_care_gains_coupled_f64(int m, const double* q_diag, const double* r_diag, const double* q_cross, const double* theta_dev, double* K_dev,
                               int* status_dev, int E, int N, void* stream);

/* launch plan (a MdsRolloutCfg.stages value) that stages == 0 selects for E envs of N drones */
int mds_rollout_plan(int E, int N);

/* ---- measurement aid: dependent-FMA-chain peak of the FP32 / FP64 pipes (TFLOP/s) ---- */
int mds_fma_peak(int use_f64, int iters, double* tflops_out, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* MDS_B200_H */
