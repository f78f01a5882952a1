// mds_kernels.cu -- __global__ kernels of the batched drone hot path and their C ABI
// (include/mds_b200.h).  Built for sm_100a only.  One thread per drone; the drones of
// an environment always share a thread block (blockDim = envs_per_block * N) so that
// downwash neighbours and CBF rows are staged through shared memory.
#include <cuda_runtime.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <mutex>

#include "mds_cbf.cuh"
#include "mds_common.cuh"
#include "mds_ctrl.cuh"
#include "mds_physics.cuh"
#include "mds_sysid.cuh"
#include "mds_traj.cuh"

using namespace mds;

// ------------------------------------------------------------------ error plumbing
static thread_local char g_err[512] = "";
static int fail(int code, const char* fmt, const char* a = "") {
  snprintf(g_err, sizeof(g_err), fmt, a);
  return code;
}
static int check_launch(const char* what) {
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) {
    snprintf(g_err, sizeof(g_err), "%s: %s", what, cudaGetErrorString(e));
    return MDS_ERR_LAUNCH;
  }
  return MDS_OK;
}
// a failed runtime call leaves its error for the next cudaGetLastError(): report it and clear it
static int cuda_fail(const char* what, cudaError_t e) {
  (void)cudaGetLastError();
  snprintf(g_err, sizeof(g_err), "%s: %s", what, cudaGetErrorString(e));
  return MDS_ERR_LAUNCH;
}
#define MDS_REQUIRE(cond, msg) \
  if (!(cond)) return fail(MDS_ERR_ARG, "%s", msg)

#include "mds_rollout.cuh"
#include "mds_rollout_launch.cuh"
#include "mds_learn_launch.cuh"
#include "mds_care_launch.cuh"

template <typename Real>
__global__ void obs_from_state_kernel(DroneP<Real> P, StateP<Real> st, Real* __restrict__ obs, int D) {
  int d = blockIdx.x * blockDim.x + threadIdx.x;
  if (d >= D) return;
  Drone<Real> s = load_drone(st, d);
  M3<Real> R = quat_to_mat(s.qx, s.qy, s.qz, s.qw);
  store_obs(obs, d, make_obs(s, mul(R, s.w)));
}

// ------------------------------------------------------------------ kernels: trajectories / controllers
template <typename Real> MDS_DEV Ref<Real> load_ref(const Real* __restrict__ ref, int d) {
  const Real* r = ref + (size_t)d * MDS_REF_DIM;
  Ref<Real> o;
  o.p = {r[0], r[1], r[2]}; o.v = {r[3], r[4], r[5]}; o.a = {r[6], r[7], r[8]}; o.yaw = r[9]; o.yaw_rate = r[10];
  return o;
}
template <typename Real>
__global__ void traj_eval_kernel(const typename TrajSpecT<Real>::spec* __restrict__ specs,
                                 const typename TrajSpecT<Real>::seg* __restrict__ segs, double t, Real* __restrict__ ref, int D) {
  int d = blockIdx.x * blockDim.x + threadIdx.x;
  if (d >= D) return;
  Ref<Real> o = eval_traj<Real>(specs[d], segs, t);
  Real* r = ref + (size_t)d * MDS_REF_DIM;
  r[0] = o.p.x; r[1] = o.p.y; r[2] = o.p.z; r[3] = o.v.x; r[4] = o.v.y; r[5] = o.v.z;
  r[6] = o.a.x; r[7] = o.a.y; r[8] = o.a.z; r[9] = o.yaw; r[10] = o.yaw_rate;
}
template <typename Real>
__global__ void geometric_ctrl_kernel(DroneP<Real> P, GeoP<Real> G, const Real* __restrict__ obs, const Real* __restrict__ ref,
                                      Real* __restrict__ action, Real* __restrict__ u_out, int D) {
  int d = blockIdx.x * blockDim.x + threadIdx.x;
  if (d >= D) return;
  Real u[4], rpm[4];
  geometric_input(P, G, load_obs(obs, d), load_ref(ref, d), u);
  input_to_action(P, u, rpm);
  store4(action, d, rpm);
  if (u_out) store4(u_out, d, u);
}
template <typename Real>
__global__ void lqr_ctrl_kernel(DroneP<Real> P, LqrP<Real> L, int variant, const Real* __restrict__ obs, const Real* __restrict__ ref,
                                Real* __restrict__ u_out, Real* __restrict__ action, PidP<Real> pid, int D) {
  int d = blockIdx.x * blockDim.x + threadIdx.x;
  if (d >= D) return;
  Obs<Real> o = load_obs(obs, d);
  Real u[4], rpm[4];
  lqr_input(P, L, variant, o, load_ref(ref, d), u);
  if (variant == MDS_CTRL_LQR_TORQUE) {
    input_to_action(P, u, rpm);  // clamps u[0] >= 0 in place, like the reference
    if (action) store4(action, d, rpm);
  } else {
    if (action) {  // inner loop sees the un-capped u (quirk B9)
      Pid<Real> ps = load_pid(pid, d);
      low_level(P, variant, ps, u, o, rpm);
      store_pid(pid, d, ps);
      store4(action, d, rpm);
      if (variant == MDS_CTRL_LQR_OMEGA) u[0] = max_(u[0], Real(0));
    }
    if (variant == MDS_CTRL_LQR_OMEGA) u[0] = cap_thrust(P, u[0]);
  }
  store4(u_out, d, u);
}
// DecentralizedLQR*.compute: lqr_ctrl_kernel with a gain per drone (K planes).  coupled = 0: u_d = -K_d e_d, K [4*dim][D].
// coupled = 1: u_d = -sum_j K_{d,j} e_j over the N drones j of d's environment, K [N][4*dim][D] (source-major) -- the
// 12-dim reference couples robots 0 and 1 through off-diagonal blocks of Q (decentralized_lqr.py:44-53), so its K is
// a full 4N x 12N matrix.  blockDim is a multiple of N: an environment never straddles two blocks.
template <typename Real>
__global__ void dlqr_ctrl_kernel(DroneP<Real> P, int variant, const Real* __restrict__ K, int coupled, const Real* __restrict__ obs,
                                 const Real* __restrict__ ref, Real* __restrict__ u_out, Real* __restrict__ action, PidP<Real> pid, int D, int N) {
  extern __shared__ __align__(16) unsigned char dlqr_smem[];
  Real* e_sh = reinterpret_cast<Real*>(dlqr_smem);  // [blockDim][12]
  const int d = blockIdx.x * blockDim.x + threadIdx.x;
  const bool valid = d < D;
  Obs<Real> o;
  Real e[12], u[4], rpm[4];
  int dim = 0;
  if (valid) {
    o = load_obs(obs, d);
    dim = lqr_error_state(P, variant, o, load_ref(ref, d), e);
  }
  if (coupled) {
    if (valid)
      for (int k = 0; k < dim; ++k) e_sh[threadIdx.x * 12 + k] = e[k];
    __syncthreads();
  }
  if (!valid) return;
  const size_t Ds = (size_t)D;
#pragma unroll
  for (int i = 0; i < 4; ++i) u[i] = Real(0);
  if (coupled) {
    const int n = d % N;
    for (int j = 0; j < N; ++j) {
      const Real* ej = e_sh + (threadIdx.x - n + j) * 12;
      const Real* Kj = K + (size_t)j * 4 * dim * Ds;
#pragma unroll
      for (int i = 0; i < 4; ++i)
        for (int k = 0; k < dim; ++k) u[i] -= Kj[(size_t)(i * dim + k) * Ds + d] * ej[k];
    }
  } else {
#pragma unroll
    for (int i = 0; i < 4; ++i)
      for (int k = 0; k < dim; ++k) u[i] -= K[(size_t)(i * dim + k) * Ds + d] * e[k];
  }
  if (variant != MDS_CTRL_LQR_YANK) u[0] += P.m * P.g;
  if (variant == MDS_CTRL_LQR_TORQUE) {
    input_to_action(P, u, rpm);
    if (action) store4(action, d, rpm);
  } else {
    if (action) {
      Pid<Real> ps = load_pid(pid, d);
      low_level(P, variant, ps, u, o, rpm);
      store_pid(pid, d, ps);
      store4(action, d, rpm);
      if (variant == MDS_CTRL_LQR_OMEGA) u[0] = max_(u[0], Real(0));
    }
    if (variant == MDS_CTRL_LQR_OMEGA) u[0] = cap_thrust(P, u[0]);
  }
  store4(u_out, d, u);
}
// error_state on model STATE vectors (not observations) and, optionally, the feedback u = -K_d e_d:
// decentralized_lqr_omega.py:174-183, decentralized_lqr.py:288-298, YOState.error_state decentralized_yolqr_crazyflie.py:88-102
// and DecentralizedYOLQRCrazyflie.compute (:350-362), whose states come from outside the simulator (FedCE).
// x, x_des [D][dim]; attitude error in closed form (roll, pitch, wrap(yaw - yaw_des)), valid for |pitch| <= pi/2.
template <typename Real>
__global__ void state_feedback_kernel(int variant, const Real* __restrict__ K, const Real* __restrict__ x, const Real* __restrict__ xdes,
                                      Real* __restrict__ e_out, Real* __restrict__ u_out, int D) {
  const int d = blockIdx.x * blockDim.x + threadIdx.x;
  if (d >= D) return;
  const int dim = variant == MDS_CTRL_LQR_TORQUE ? 12 : (variant == MDS_CTRL_LQR_OMEGA ? 9 : 10);
  Real xs[12], xd[12], e[12];
  for (int k = 0; k < dim; ++k) { xs[k] = x[(size_t)d * dim + k]; xd[k] = xdes[(size_t)d * dim + k]; }
  Real sy, cy;
  sincos_(xd[2], &sy, &cy);
  const Real two_pi = Real(6.283185307179586476925286766559), inv_two_pi = Real(0.15915494309189533576888376337251);
  e[0] = xs[0]; e[1] = xs[1];
  const Real dy = xs[2] - xd[2];
  e[2] = dy - two_pi * rint_(dy * inv_two_pi);
  int first = 3;
  if (variant == MDS_CTRL_LQR_YANK) { e[3] = xs[3] - xd[3]; first = 4; }
  for (int b = first; b < dim; b += 3) {  // every remaining 3-vector (rates, velocity, position) rotated by R_eq^T (yaw only)
    const Real ax = xs[b] - xd[b], ay = xs[b + 1] - xd[b + 1];
    e[b] = cy * ax + sy * ay; e[b + 1] = -sy * ax + cy * ay; e[b + 2] = xs[b + 2] - xd[b + 2];
  }
  if (e_out)
    for (int k = 0; k < dim; ++k) e_out[(size_t)d * dim + k] = e[k];
  if (u_out) {
    Real u[4] = {Real(0), Real(0), Real(0), Real(0)};
    for (int i = 0; i < 4; ++i)
      for (int k = 0; k < dim; ++k) u[i] -= K[(size_t)(i * dim + k) * (size_t)D + d] * e[k];
    store4(u_out, d, u);
  }
}
template <typename Real>
__global__ void error_state_kernel(DroneP<Real> P, int variant, const Real* __restrict__ obs, const Real* __restrict__ ref, Real* __restrict__ e_out, int D) {
  int d = blockIdx.x * blockDim.x + threadIdx.x;
  if (d >= D) return;
  Real e[12];
  const int dim = lqr_error_state(P, variant, load_obs(obs, d), load_ref(ref, d), e);
  for (int k = 0; k < dim; ++k) e_out[(size_t)d * dim + k] = e[k];
}
template <typename Real>
__global__ void dslpid_ctrl_kernel(DroneP<Real> P, DslP<Real> G, const Real* __restrict__ obs, const Real* __restrict__ target,
                                   DslStateP<Real> st, Real* __restrict__ action, Real* __restrict__ pos_e, int D) {
  int d = blockIdx.x * blockDim.x + threadIdx.x;
  if (d >= D) return;
  const Real* t = target + (size_t)d * 12;
  DslState<Real> s = load_dsl(st, d);
  Real rpm[4];
  V3<Real> pe;
  dslpid_control(P, G, s, load_obs(obs, d), v3(t[0], t[1], t[2]), v3(t[3], t[4], t[5]), v3(t[6], t[7], t[8]), v3(t[9], t[10], t[11]), rpm, &pe);
  store_dsl(st, d, s);
  store4(action, d, rpm);
  if (pos_e) { pos_e[3 * d] = pe.x; pos_e[3 * d + 1] = pe.y; pos_e[3 * d + 2] = pe.z; }
}
template <typename Real>
__global__ void lowlevel_kernel(DroneP<Real> P, int variant, const Real* __restrict__ u_in, const Real* __restrict__ obs,
                                PidP<Real> pid, Real* __restrict__ action, int D) {
  int d = blockIdx.x * blockDim.x + threadIdx.x;
  if (d >= D) return;
  Real u[4], rpm[4];
  load4(u_in, d, u);
  Pid<Real> ps = load_pid(pid, d);
  low_level(P, variant, ps, u, load_obs(obs, d), rpm);
  store_pid(pid, d, ps);
  store4(action, d, rpm);
}

// ------------------------------------------------------------------ kernels: CBF
template <typename Real, int ORD>
__global__ void __launch_bounds__(MDS_BLOCK) cbf_qp_kernel(DroneP<Real> P, CbfP<Real> C, const Real* __restrict__ obs, const Real* __restrict__ xdes,
                                                            const Real* __restrict__ unom_g, const Real* __restrict__ obstacles, int n_obs,
                                                            Real* __restrict__ usafe_g, int* __restrict__ status, int* __restrict__ iters,
                                                            int E, int N, int NP) {
  extern __shared__ __align__(32) unsigned char smem_raw[];
  CbfSmem<Real> S = cbf_smem_carve<Real>(smem_raw, NP, N, n_obs);
  const GroupMap g = group_map(N, NP, E);
  if (!g.env_valid) return;
  const int xdim = C.order == 2 ? 9 : 10;
  CbfAgent<Real> ag;
  ag.p = {Real(0), Real(0), Real(0)}; ag.dv = ag.p; ag.da = ag.p;
  Real F = Real(0), unom[4] = {Real(0), Real(0), Real(0), Real(0)}, usafe[4];
  if (g.valid) {
    Obs<Real> o = load_obs(obs, g.d);
    Real xd[10];
    for (int k = 0; k < xdim; ++k) xd[k] = xdes[(size_t)g.d * xdim + k];
    ag = cbf_agent<ORD>(P, C, o, xd, &F);
    load4(unom_g, g.d, unom);
  }
  Real min_h = Real(1e30);
  int it = 0;
  int st = cbf_filter_group<ORD>(P, C, S, obstacles, n_obs, g, N, NP, ag, F, unom, usafe, &min_h, &it);
  if (g.valid) {
    store4(usafe_g, g.d, usafe);
    if (g.n == 0) {
      status[g.e] = st;
      if (iters) iters[g.e] = it;
    }
  }
}

template <typename Real>
__global__ void cbf_prepare_kernel(DroneP<Real> P, int order, Real u0_offset, const Real* __restrict__ ref, Real* __restrict__ u,
                                   Real* __restrict__ xdes, int D) {
  int d = blockIdx.x * blockDim.x + threadIdx.x;
  if (d >= D) return;
  Ref<Real> r = load_ref(ref, d);
  u[(size_t)d * 4] -= u0_offset;
  const int xdim = order == 2 ? 9 : 10;
  Real* x = xdes + (size_t)d * xdim;
  x[0] = Real(0); x[1] = Real(0); x[2] = r.yaw;
  int o = 3;
  if (order == 3) x[o++] = P.g * P.m;
  x[o] = r.v.x; x[o + 1] = r.v.y; x[o + 2] = r.v.z; x[o + 3] = r.p.x; x[o + 4] = r.p.y; x[o + 5] = r.p.z;
}

// dense G, h in the reference's row order (parity aid; one thread per env)
template <typename Real>
__global__ void cbf_rows_kernel(DroneP<Real> P, CbfP<Real> C, const Real* __restrict__ obs, const Real* __restrict__ xdes,
                                const Real* __restrict__ obstacles, int n_obs, Real* __restrict__ Gm, Real* __restrict__ hv, int E, int N) {
  int e = blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= E) return;
  const int xdim = C.order == 2 ? 9 : 10;
  const int n_pairs = N * (N - 1) / 2, W = 4 * N;
  const bool force_rows = C.order == 3 && C.state_bounds;
  const int m = n_pairs + 8 * N + (force_rows ? 2 * N : 0) + N * n_obs;
  Real* G = Gm + (size_t)e * m * W;
  Real* h = hv + (size_t)e * m;
  for (size_t k = 0; k < (size_t)m * W; ++k) G[k] = Real(0);
  auto agent = [&](int i, Real* F) {
    Obs<Real> o = load_obs(obs, e * N + i);
    Real xd[10];
    for (int k = 0; k < xdim; ++k) xd[k] = xdes[(size_t)(e * N + i) * xdim + k];
    return cbf_agent<0>(P, C, o, xd, F);
  };
  int row = 0;
  Real F, a3[3], rhs, h0;
  for (int i = 0; i < N - 1; ++i)
    for (int j = i + 1; j < N; ++j) {
      CbfAgent<Real> ai = agent(i, &F), aj = agent(j, &F);
      cbf_row<0>(P, C, ai, aj, C.ds4_pair, C.c4inv, a3, &rhs, &h0);
      for (int c = 0; c < 3; ++c) { G[(size_t)row * W + 4 * i + c] = -a3[c]; G[(size_t)row * W + 4 * j + c] = a3[c]; }
      h[row++] = rhs;
    }
  for (int k = 0; k < W; ++k) { G[(size_t)row * W + k] = Real(1); h[row++] = C.umax[k & 3]; }
  for (int k = 0; k < W; ++k) { G[(size_t)row * W + k] = Real(-1); h[row++] = C.umax[k & 3]; }
  if (force_rows)
    for (int i = 0; i < N; ++i) {
      agent(i, &F);
      G[(size_t)row * W + 4 * i + 3] = Real(1); h[row++] = C.k2 * (C.fmax - F);
      G[(size_t)row * W + 4 * i + 3] = Real(-1); h[row++] = C.k2 * (F - C.fmin);
    }
  for (int i = 0; i < N; ++i)
    for (int o = 0; o < n_obs; ++o) {
      CbfAgent<Real> ai = agent(i, &F), aj;
      aj.p = {obstacles[4 * o], obstacles[4 * o + 1], obstacles[4 * o + 2]};
      aj.dv = {Real(0), Real(0), Real(0)}; aj.da = aj.dv;
      Real Ds, c4inv;
      obstacle_shape(C, obstacles[4 * o + 3], &Ds, &c4inv);
      cbf_row<0>(P, C, ai, aj, (Ds * Ds) * (Ds * Ds), c4inv, a3, &rhs, &h0);
      for (int c = 0; c < 3; ++c) G[(size_t)row * W + 4 * i + c] = -a3[c];
      h[row++] = rhs;
    }
}

// ------------------------------------------------------------------ kernels: model comparison
template <typename Real>
__global__ void xdot_linear_kernel(DroneP<Real> P, int kind, const Real* __restrict__ obs, Real* __restrict__ xdot, int D) {
  int d = blockIdx.x * blockDim.x + threadIdx.x;
  if (d >= D) return;
  Obs<Real> o = load_obs(obs, d);
  Real* out = xdot + (size_t)d * kind;
  if (kind == 12) {  // model/linearized.py:83-104: x = [rpy, w(obs 13:16), v, p], u from action_to_input
    Real u[4];
    action_to_input(P, o.rpm, u);
    out[0] = o.av.x; out[1] = o.av.y; out[2] = o.av.z;
    out[3] = u[1] / P.ixx; out[4] = u[2] / P.iyy; out[5] = u[3] / P.izz;
    out[6] = P.g * o.rpy.y; out[7] = -P.g * o.rpy.x; out[8] = (u[0] - P.m * P.g) / P.m;
    out[9] = o.v.x; out[10] = o.v.y; out[11] = o.v.z;
    return;
  }
  // builder-defined 9 / 10-dim (quirk B23): u = [f | yank = 0, body rates]
  M3<Real> R = quat_to_rot_scipy(o.qx, o.qy, o.qz, o.qw);
  V3<Real> wb = mulT(R, o.av);
  Real F = z_thrust(P, o.rpm);
  out[0] = wb.x; out[1] = wb.y; out[2] = wb.z;
  if (kind == 9) {
    out[3] = P.g * o.rpy.y; out[4] = -P.g * o.rpy.x; out[5] = (F - P.m * P.g) / P.m;
    out[6] = o.v.x; out[7] = o.v.y; out[8] = o.v.z;
  } else {
    out[3] = Real(0);
    out[4] = P.g * o.rpy.y; out[5] = -P.g * o.rpy.x; out[6] = (F - P.m * P.g) / P.m;
    out[7] = o.v.x; out[8] = o.v.y; out[9] = o.v.z;
  }
}
template <typename Real>
__global__ void xdot_nonlinear_kernel(DroneP<Real> P, Real jx, Real jy, Real jz, const Real* __restrict__ obs, Real* __restrict__ xdot, int D) {
  int d = blockIdx.x * blockDim.x + threadIdx.x;
  if (d >= D) return;
  Obs<Real> o = load_obs(obs, d);
  Real u[4];
  action_to_input(P, o.rpm, u);
  M3<Real> R = quat_to_rot_scipy(o.qx, o.qy, o.qz, o.qw);
  V3<Real> w = o.av;
  V3<Real> Jw = {jx * w.x, jy * w.y, jz * w.z};
  V3<Real> g = cross(w, Jw);
  Real* out = xdot + (size_t)d * 12;  // geo_x_dot_to_linear order: (w, wdot, vdot, v)
  out[0] = w.x; out[1] = w.y; out[2] = w.z;
  out[3] = (u[1] - g.x) / jx; out[4] = (u[2] - g.y) / jy; out[5] = (u[3] - g.z) / jz;
  Real a = u[0] / P.m;
  out[6] = R.m[2] * a; out[7] = R.m[5] * a; out[8] = R.m[8] * a - P.g;
  out[9] = o.v.x; out[10] = o.v.y; out[11] = o.v.z;
}

// Roll-out of the 12-dim hover-linearised model along a logged flight (simulations/CompareModels.py:82-95): the reference
// integrates x' = A (x - x_eq) + B (u(t) - u_eq) with scipy's RK45 and the logged RPMs as zero-order-hold inputs.  With a
// constant input the chain  u -> w -> rpy -> (vx, vy) -> (px, py)  integrates to polynomials in t, so each log interval
// is advanced EXACTLY (to rounding); one thread per drone walks its T samples.  obs_log [T, D, 20] -> x_out [T, D, 12],
// x = [rpy, w, v, p] (utils/model_conversions.py:41-45), x_out[0] = the first logged state.
template <typename Real>
__global__ void linear_rollout_kernel(DroneP<Real> P, const Real* __restrict__ obs_log, Real dt, Real* __restrict__ x_out, int T, int D) {
  int d = blockIdx.x * blockDim.x + threadIdx.x;
  if (d >= D) return;
  Obs<Real> o = load_obs(obs_log, d);
  V3<Real> rpy = o.rpy, w = o.av, v = o.v, p = o.p;
  const Real t = dt, t2 = t * t * Real(0.5), t3 = t * t * t / Real(6), t4 = t * t * t * t / Real(24);
  for (int k = 0;; ++k) {
    Real* x = x_out + ((size_t)k * D + d) * 12;
    x[0] = rpy.x; x[1] = rpy.y; x[2] = rpy.z; x[3] = w.x; x[4] = w.y; x[5] = w.z;
    x[6] = v.x; x[7] = v.y; x[8] = v.z; x[9] = p.x; x[10] = p.y; x[11] = p.z;
    if (k == T - 1) break;
    Real u[4];
    action_to_input(P, o.rpm, u);  // the input logged with sample k holds until sample k + 1
    const V3<Real> al = {u[1] / P.ixx, u[2] / P.iyy, u[3] / P.izz};
    const Real az = (u[0] - P.m * P.g) / P.m;
    p = {p.x + v.x * t + P.g * (rpy.y * t2 + w.y * t3 + al.y * t4), p.y + v.y * t - P.g * (rpy.x * t2 + w.x * t3 + al.x * t4), p.z + v.z * t + az * t2};
    v = {v.x + P.g * (rpy.y * t + w.y * t2 + al.y * t3), v.y - P.g * (rpy.x * t + w.x * t2 + al.x * t3), v.z + az * t};
    rpy = {rpy.x + w.x * t + al.x * t2, rpy.y + w.y * t + al.y * t2, rpy.z + w.z * t + al.z * t2};
    w = {w.x + al.x * t, w.y + al.y * t, w.z + al.z * t};
    o = load_obs(obs_log + (size_t)(k + 1) * D * MDS_OBS_DIM, d);  // only its RPMs are used
  }
}

// ------------------------------------------------------------------ FMA-chain peak microbenchmark
// 16 independent dependent-FMA chains per thread, unrolled 16 x: 256 FMAs per loop trip against one counter update and
// one branch, 16 chains against the FMA pipe's 4-cycle latency (r1's 8-chain, un-unrolled loop reached 86 % of nominal).
template <typename Real> __global__ void fma_peak_kernel(Real* out, int iters) {
  Real a[16];
#pragma unroll
  for (int j = 0; j < 16; ++j) a[j] = Real(threadIdx.x) * Real(1e-3) + Real(j);
  const Real b = Real(0.999), c = Real(1e-3);
  for (int i = 0; i < iters; i += 16) {
#pragma unroll
    for (int u = 0; u < 16; ++u) {
#pragma unroll
      for (int j = 0; j < 16; ++j) a[j] = fma_(a[j], b, c);
    }
  }
  Real s = Real(0);
#pragma unroll
  for (int j = 0; j < 16; ++j) s += a[j];
  out[blockIdx.x * blockDim.x + threadIdx.x] = s;
}

// ================================================================== C ABI
template <typename Real>
static int physics_step_impl(const MdsDroneParams* prm, MdsState st, const Real* action, const Real* fext, Real* obs, int E, int N, void* stream) {
  MDS_REQUIRE(prm && st.pos_wx && st.quat && st.vel_wy && st.rpm && st.wz && action, "physics_step: null pointer");
  MDS_REQUIRE(E > 0 && N > 0 && N <= MDS_MAX_DRONES_PER_ENV, "physics_step: bad E or N");
  MDS_REQUIRE(prm->substeps >= 1, "physics_step: substeps must be >= 1");
  MDS_REQUIRE(prm->physics == MDS_PHYSICS_DYN || prm->physics == MDS_PHYSICS_DYN_GND_DRAG_DW, "physics_step: unknown physics mode");
  int NP = next_pow2(N), epb = MDS_BLOCK / NP, blocks = (E + epb - 1) / epb;
  if (N == 8) physics_step_kernel<Real, 8><<<blocks, MDS_BLOCK, 0, (cudaStream_t)stream>>>(to_dev<Real>(*prm), to_dev<Real>(st), action, fext, obs, E, N, NP);
  else physics_step_kernel<Real, 0><<<blocks, MDS_BLOCK, 0, (cudaStream_t)stream>>>(to_dev<Real>(*prm), to_dev<Real>(st), action, fext, obs, E, N, NP);
  return check_launch("physics_step");
}
template <typename Real> static int obs_from_state_impl(const MdsDroneParams* prm, MdsState st, Real* obs, int D, void* stream) {
  MDS_REQUIRE(prm && st.pos_wx && st.quat && st.vel_wy && st.rpm && st.wz && obs && D > 0, "obs_from_state: bad argument");
  obs_from_state_kernel<Real><<<(D + 255) / 256, 256, 0, (cudaStream_t)stream>>>(to_dev<Real>(*prm), to_dev<Real>(st), obs, D);
  return check_launch("obs_from_state");
}
template <typename Real>
static int traj_eval_impl(const typename TrajSpecT<Real>::spec* specs, const typename TrajSpecT<Real>::seg* segs, double t, Real* ref, int D, void* stream) {
  MDS_REQUIRE(specs && ref && D > 0, "traj_eval: bad argument");
  traj_eval_kernel<Real><<<(D + 255) / 256, 256, 0, (cudaStream_t)stream>>>(specs, segs, t, ref, D);
  return check_launch("traj_eval");
}
template <typename Real>
static int geometric_impl(const MdsDroneParams* prm, const MdsGeoGains* g, const Real* obs, const Real* ref, Real* action, Real* u, int D, void* stream) {
  MDS_REQUIRE(prm && g && obs && ref && action && D > 0, "geometric_ctrl: bad argument");
  geometric_ctrl_kernel<Real><<<(D + 127) / 128, 128, 0, (cudaStream_t)stream>>>(to_dev<Real>(*prm), to_dev<Real>(*g), obs, ref, action, u, D);
  return check_launch("geometric_ctrl");
}
template <typename Real>
static int dslpid_impl(const MdsDroneParams* prm, const MdsDslPidGains* g, const Real* obs, const Real* target, MdsDslPidState st, Real* action,
                       Real* pos_e, int D, void* stream) {
  MDS_REQUIRE(prm && g && obs && target && st.a && st.b && st.c && action && D > 0, "dslpid_ctrl: bad argument");
  dslpid_ctrl_kernel<Real><<<(D + 127) / 128, 128, 0, (cudaStream_t)stream>>>(to_dev<Real>(*prm), to_dev<Real>(*g), obs, target, to_dev<Real>(st), action,
                                                                                pos_e, D);
  return check_launch("dslpid_ctrl");
}
static bool lqr_dim_ok(int variant, int dim) {
  return (variant == MDS_CTRL_LQR_TORQUE && dim == 12) || (variant == MDS_CTRL_LQR_OMEGA && dim == 9) || (variant == MDS_CTRL_LQR_YANK && dim == 10);
}
template <typename Real>
static int lqr_impl(const MdsDroneParams* prm, const MdsLqrGains* g, int variant, const Real* obs, const Real* ref, Real* u, Real* action,
                    MdsPidState pid, int D, void* stream) {
  MDS_REQUIRE(prm && g && obs && ref && u && D > 0, "lqr_ctrl: bad argument");
  MDS_REQUIRE(lqr_dim_ok(variant, g->dim), "lqr_ctrl: variant / gain dimension mismatch");
  MDS_REQUIRE(!(action && variant != MDS_CTRL_LQR_TORQUE) || (pid.a && pid.b), "lqr_ctrl: inner loop needs PID state");
  lqr_ctrl_kernel<Real><<<(D + 127) / 128, 128, 0, (cudaStream_t)stream>>>(to_dev<Real>(*prm), to_dev<Real>(*g), variant, obs, ref, u, action,
                                                                             to_dev<Real>(pid), D);
  return check_launch("lqr_ctrl");
}
// The MdsRlsCfg checks that mds_rls_update and mds_learning_rollout share, and its translation to the kernels' RlsP
// (theta_code packed into 2-bit row codes).  cfg->m must already be checked: it sizes the theta_code walk.
static int rls_params(const MdsRlsCfg* cfg, const char* who, RlsP* out) {
  if (cfg->target != MDS_RLS_TARGET_PREDICT && cfg->target != MDS_RLS_TARGET_XDOT) return fail(MDS_ERR_ARG, "%s: unknown target", who);
  if (cfg->target == MDS_RLS_TARGET_XDOT && cfg->m == 9)
    return fail(MDS_ERR_ARG, "%s: the reference defines est_x_dot for m = 10 and 12 only", who);
  if (cfg->project < MDS_RLS_PROJECT_NONE || cfg->project > MDS_RLS_PROJECT_LOOP) return fail(MDS_ERR_ARG, "%s: unknown projection mode", who);
  RlsP c;
  c.target = cfg->target; c.predict_from_xtp1 = cfg->predict_from_xtp1; c.normalize_gain = cfg->normalize_gain;
  c.project = cfg->project; c.drones_per_env = cfg->drones_per_env; c.dt = cfg->dt;
  for (int i = 0; i < 16; ++i) c.row_code[i] = 0x55555555u;
  for (int i = 0; i < cfg->m + 4; ++i)
    for (int j = 0; j < cfg->m; ++j) {
      const unsigned code = cfg->theta_code[i * cfg->m + j];
      if (code > 2) return fail(MDS_ERR_ARG, "%s: theta_code entries must be 0, 1 or 2", who);
      c.row_code[i] = (c.row_code[i] & ~(3u << (2 * j))) | (code << (2 * j));
    }
  *out = c;
  return MDS_OK;
}
template <typename Real>
static int rls_impl(const MdsRlsCfg* cfg, const Real* phi, const Real* xtp1, Real* theta, Real* Pm, Real* resid, int D, void* stream) {
  MDS_REQUIRE(cfg && phi && xtp1 && theta && Pm && D > 0, "rls_update: bad argument");
  MDS_REQUIRE(cfg->m == 9 || cfg->m == 10 || cfg->m == 12, "rls_update: m must be 9, 10 or 12");
  RlsP c;
  if (const int rc = rls_params(cfg, "rls_update", &c)) return rc;
  MDS_REQUIRE(cfg->dt > 0.0 && cfg->drones_per_env >= 1, "rls_update: dt and drones_per_env must be positive");
  cudaStream_t cs = (cudaStream_t)stream;
  cudaError_t ae = cudaSuccess;
  // One thread per drone, one warp (f32) / half a warp (f64) per block; P is read from its upper triangle (mds_sysid.cuh).  Round 1's
  // two-lanes-per-drone variant for the 12-dim x_dot form lost to this kernel once the triangle halved its staging footprint
  // (1.14 vs 1.26 ms per 1 M drones) and is gone.
#define MDS_LAUNCH_RLS(MM)                                                                                                    \
  do {                                                                                                                        \
    const int threads = rls_threads<Real, MM>(), blocks = (D + threads - 1) / threads;                                       \
    const size_t smem = (size_t)rls_words_per_thread<Real, MM>() * threads * sizeof(Real);                                    \
    auto kern = cfg->project != MDS_RLS_PROJECT_NONE ? rls_update_kernel<Real, MM, true> : rls_update_kernel<Real, MM, false>; \
    ae = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);                                  \
    if (ae == cudaSuccess) kern<<<blocks, threads, smem, cs>>>(c, phi, xtp1, theta, Pm, resid, D);                            \
  } while (0)
  if (cfg->m == 9) MDS_LAUNCH_RLS(9);
  else if (cfg->m == 10) MDS_LAUNCH_RLS(10);
  else MDS_LAUNCH_RLS(12);
#undef MDS_LAUNCH_RLS
  if (ae != cudaSuccess) return cuda_fail("rls_update: shared-memory opt-in", ae);
  return check_launch("rls_update");
}
// The weights of both Riccati solves (mds_care_tu.cu): diagonal Q [m] and R [4], every entry positive; c gets sqrt(q) and 1 / r.
static int care_weights(const char* what, int m, const double* q, const double* r, CareP* c) {
  for (int i = 0; i < m; ++i) {
    if (!(q[i] > 0.0)) return fail(MDS_ERR_ARG, "%s: Q must be diagonal and positive", what);
    c->sq[i] = sqrt(q[i]);
  }
  for (int i = 0; i < 4; ++i) {
    if (!(r[i] > 0.0)) return fail(MDS_ERR_ARG, "%s: R must be diagonal and positive", what);
    c->rinv[i] = 1.0 / r[i];
  }
  return MDS_OK;
}
template <typename Real>
static int care_impl(int m, const double* q, const double* r, const Real* theta, Real* K, int* status, int D, void* stream) {
  MDS_REQUIRE(q && r && theta && K && D > 0, "care_gains: bad argument");
  MDS_REQUIRE(m == 9 || m == 10 || m == 12, "care_gains: m must be 9, 10 or 12");
  CareP c{};
  if (const int rc = care_weights("care_gains", m, q, r, &c)) return rc;
  const cudaError_t ae = launch_care<Real>(c, m, false, theta, K, status, D, 1, (cudaStream_t)stream);
  if (ae != cudaSuccess) return cuda_fail("care_gains: shared-memory opt-in", ae);
  return check_launch("care_gains");
}
// The robot-coupled solve: Q = kron(I_N, diag(q)) plus the cross block q_cross [m][m] between robots 0 and 1
template <typename Real>
static int care_coupled_impl(int m, const double* q, const double* r, const double* q_cross, const Real* theta, Real* K, int* status, int E, int N,
                             void* stream) {
  MDS_REQUIRE(q && r && q_cross && theta && K, "care_gains_coupled: null pointer");
  MDS_REQUIRE(m == 12, "care_gains_coupled: m must be 12 (the robot-coupled weights are the torque-level model's)");
  MDS_REQUIRE(E >= 1 && N >= 2 && N <= MDS_MAX_DRONES_PER_ENV && (long long)E * N <= 0x7fffffffLL, "care_gains_coupled: bad E or N (N in [2, 32])");
  CareP c{};
  if (const int rc = care_weights("care_gains_coupled", m, q, r, &c)) return rc;
  for (int k = 0; k < 12; ++k)
    for (int l = 0; l < 12; ++l) {
      MDS_REQUIRE(isfinite(q_cross[k * 12 + l]), "care_gains_coupled: q_cross must be finite");
      c.cross[k * 12 + l] = q_cross[k * 12 + l] / (c.sq[k] * c.sq[l]);
    }
  // the pair's scaled Q~ = [[I, C], [C', I]] is positive semidefinite iff I - C'C is: Cholesky with a tolerance for the
  // semidefinite case (a diagonal C needs |q_cross_kk| <= q_kk)
  double S[12][12];
  for (int k = 0; k < 12; ++k)
    for (int l = 0; l < 12; ++l) {
      double v = k == l ? 1.0 : 0.0;
      for (int i = 0; i < 12; ++i) v -= c.cross[i * 12 + k] * c.cross[i * 12 + l];
      S[k][l] = v;
    }
  const double tol = 1e-12;
  for (int k = 0; k < 12; ++k) {
    MDS_REQUIRE(S[k][k] >= -tol, "care_gains_coupled: the pair's Q is not positive semidefinite");
    if (S[k][k] <= tol) {
      for (int i = k + 1; i < 12; ++i) MDS_REQUIRE(fabs(S[i][k]) <= 1e-6, "care_gains_coupled: the pair's Q is not positive semidefinite");
      continue;
    }
    for (int i = k + 1; i < 12; ++i)
      for (int j = k + 1; j < 12; ++j) S[i][j] -= S[i][k] * S[k][j] / S[k][k];
  }
  const cudaError_t ae = launch_care<Real>(c, m, true, theta, K, status, E, N, (cudaStream_t)stream);
  if (ae != cudaSuccess) return cuda_fail("care_gains_coupled: shared-memory opt-in", ae);
  return check_launch("care_gains_coupled");
}
static bool lqr_variant_ok(int v) { return v == MDS_CTRL_LQR_TORQUE || v == MDS_CTRL_LQR_OMEGA || v == MDS_CTRL_LQR_YANK; }
template <typename Real>
static int error_state_impl(const MdsDroneParams* prm, int variant, const Real* obs, const Real* ref, Real* e, int D, void* stream) {
  MDS_REQUIRE(prm && obs && ref && e && D > 0, "error_state: bad argument");
  MDS_REQUIRE(lqr_variant_ok(variant), "error_state: unknown variant");
  error_state_kernel<Real><<<(D + 127) / 128, 128, 0, (cudaStream_t)stream>>>(to_dev<Real>(*prm), variant, obs, ref, e, D);
  return check_launch("error_state");
}
template <typename Real>
static int state_feedback_impl(int variant, const Real* K, const Real* x, const Real* xdes, Real* e, Real* u, int D, void* stream) {
  MDS_REQUIRE(x && xdes && (e || u) && D > 0, "state_feedback: bad argument");
  MDS_REQUIRE(lqr_variant_ok(variant), "state_feedback: unknown variant");
  MDS_REQUIRE(!u || K, "state_feedback: u requested without gains");
  state_feedback_kernel<Real><<<(D + 127) / 128, 128, 0, (cudaStream_t)stream>>>(variant, K, x, xdes, e, u, D);
  return check_launch("state_feedback");
}
template <typename Real>
static int dlqr_impl(const MdsDroneParams* prm, int variant, const Real* K, int coupled, const Real* obs, const Real* ref, Real* u, Real* action,
                     MdsPidState pid, int E, int N, void* stream) {
  MDS_REQUIRE(prm && K && obs && ref && u && E > 0 && N > 0 && N <= MDS_MAX_DRONES_PER_ENV, "dlqr_ctrl: bad argument");
  MDS_REQUIRE(lqr_variant_ok(variant), "dlqr_ctrl: unknown variant");
  MDS_REQUIRE(!(action && variant != MDS_CTRL_LQR_TORQUE) || (pid.a && pid.b), "dlqr_ctrl: inner loop needs PID state");
  const int D = E * N, threads = (128 / N) * N, blocks = (D + threads - 1) / threads;
  const size_t smem = coupled ? (size_t)threads * 12 * sizeof(Real) : 0;
  dlqr_ctrl_kernel<Real><<<blocks, threads, smem, (cudaStream_t)stream>>>(to_dev<Real>(*prm), variant, K, coupled ? 1 : 0, obs, ref, u, action,
                                                                          to_dev<Real>(pid), D, N);
  return check_launch("dlqr_ctrl");
}
template <typename Real>
static int lowlevel_impl(const MdsDroneParams* prm, int variant, const Real* u, const Real* obs, MdsPidState pid, Real* action, int D, void* stream) {
  MDS_REQUIRE(prm && u && obs && pid.a && pid.b && action && D > 0, "lowlevel: bad argument");
  MDS_REQUIRE(variant == MDS_CTRL_LQR_OMEGA || variant == MDS_CTRL_LQR_YANK, "lowlevel: variant must be LQR_OMEGA or LQR_YANK");
  lowlevel_kernel<Real><<<(D + 255) / 256, 256, 0, (cudaStream_t)stream>>>(to_dev<Real>(*prm), variant, u, obs, to_dev<Real>(pid), action, D);
  return check_launch("lowlevel");
}
// Scratch of the large-active-set QP solver (mds_cbf.cuh qp_solve_group_big): one pool per device, owned by the library,
// allocated at the first CBF launch (so that call must not sit inside a stream capture) and regrown when a larger
// drone count shows up.  MDS_QP_SCRATCH_SLOTS solves can be in flight at once; further ones wait for a slot.
#ifndef MDS_QP_SCRATCH_SLOTS
#define MDS_QP_SCRATCH_SLOTS 1024
#endif
#define MDS_MAX_DEVICES 64
static QpScratch g_qp_scratch[MDS_MAX_DEVICES];
static std::mutex g_qp_scratch_mutex;
static long long qp_slot_doubles(int qmax) {  // act | lam | d | r | y (qmax each) + Lc | Lm (qmax (qmax + 1) / 2 each) + hdr (4)
  return 5LL * qmax + (long long)qmax * (qmax + 1) + 4;
}
static int qp_scratch_for(int N, QpScratch* out) {
  int dev = 0;
  cudaError_t e = cudaGetDevice(&dev);
  if (e != cudaSuccess) return cuda_fail("qp scratch", e);
  if (dev < 0 || dev >= MDS_MAX_DEVICES) return fail(MDS_ERR_ARG, "%s", "qp scratch: device index out of range");
  std::lock_guard<std::mutex> lock(g_qp_scratch_mutex);
  QpScratch& S = g_qp_scratch[dev];
  const int qmax = 3 * N;  // the coupled variables of an environment: an active set cannot be larger
  if (S.base == nullptr || S.qmax < qmax) {
    if (S.base) { cudaFree(S.base); cudaFree(S.flags); S.base = nullptr; S.flags = nullptr; }  // cudaFree waits for kernels in flight
    const long long sd = qp_slot_doubles(qmax);
    e = cudaMalloc((void**)&S.base, (size_t)MDS_QP_SCRATCH_SLOTS * (size_t)sd * sizeof(double));
    if (e == cudaSuccess) e = cudaMalloc((void**)&S.flags, MDS_QP_SCRATCH_SLOTS * sizeof(int));
    if (e == cudaSuccess) e = cudaMemset(S.flags, 0, MDS_QP_SCRATCH_SLOTS * sizeof(int));
    if (e != cudaSuccess) { S.base = nullptr; S.flags = nullptr; return cuda_fail("qp scratch allocation", e); }
    S.slots = MDS_QP_SCRATCH_SLOTS; S.qmax = qmax; S.slot_doubles = sd;
  }
  *out = S;
  return MDS_OK;
}
static int cbf_args_ok(const MdsCbfParams* c, int N, int n_obs) {
  if (!c) return fail(MDS_ERR_ARG, "%s", "cbf: null params");
  if (c->order != 2 && c->order != 3) return fail(MDS_ERR_ARG, "%s", "cbf: order must be 2 or 3");
  if (N < 1 || N > MDS_MAX_DRONES_PER_ENV) return fail(MDS_ERR_ARG, "%s", "cbf: bad N");
  // The reference fails for n_obs > N (it indexes agent blocks by obstacle id, cbf.py:388, quirk B14) although nothing in
  // the barrier needs it: every obstacle row uses only drone i's own model.  The library takes up to MDS_MAX_OBSTACLES for
  // any N (SURVEY 8f-4); the host mirror keeps the reference's refusal unless asked (DroneCBF(allow_extra_obstacles=True)).
  if (n_obs < 0 || n_obs > MDS_MAX_OBSTACLES) return fail(MDS_ERR_ARG, "%s", "cbf: n_obs must be in [0, MDS_MAX_OBSTACLES]");
  return MDS_OK;
}
template <typename Real>
static int cbf_qp_impl(const MdsDroneParams* prm, const MdsCbfParams* c, const Real* obs, const Real* xdes, const Real* unom, const Real* obstacles,
                       int n_obs, Real* usafe, int* status, int* iters, int E, int N, void* stream) {
  int rc = cbf_args_ok(c, N, n_obs);
  if (rc) return rc;
  MDS_REQUIRE(prm && obs && xdes && unom && usafe && status && E > 0, "cbf_qp: bad argument");
  MDS_REQUIRE(n_obs == 0 || obstacles, "cbf_qp: obstacles pointer is null");
  const int NP = next_pow2(N), threads = cbf_block_threads<Real>(NP, N, n_obs), epb = threads / NP, blocks = (E + epb - 1) / epb;
  size_t smem = cbf_smem_bytes<Real>(threads, NP, N, n_obs);
  CbfP<Real> C = to_dev<Real>(*c);
  rc = qp_scratch_for(N, &C.scr);
  if (rc) return rc;
  auto kern = c->order == 2 ? cbf_qp_kernel<Real, 2> : cbf_qp_kernel<Real, 3>;
  cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (e != cudaSuccess) return cuda_fail("cbf_qp: shared memory opt-in failed", e);
  kern<<<blocks, threads, smem, (cudaStream_t)stream>>>(to_dev<Real>(*prm), C, obs, xdes, unom, obstacles, n_obs, usafe, status, iters, E, N, NP);
  return check_launch("cbf_qp");
}
template <typename Real>
static int cbf_rows_impl(const MdsDroneParams* prm, const MdsCbfParams* c, const Real* obs, const Real* xdes, const Real* obstacles, int n_obs,
                         Real* Gm, Real* h, int E, int N, void* stream) {
  int rc = cbf_args_ok(c, N, n_obs);
  if (rc) return rc;
  MDS_REQUIRE(prm && obs && xdes && Gm && h && E > 0, "cbf_rows: bad argument");
  cbf_rows_kernel<Real><<<(E + 63) / 64, 64, 0, (cudaStream_t)stream>>>(to_dev<Real>(*prm), to_dev<Real>(*c), obs, xdes, obstacles, n_obs, Gm, h, E, N);
  return check_launch("cbf_rows");
}
template <typename Real>
static int cbf_prepare_impl(const MdsDroneParams* prm, int order, double u0, const Real* ref, Real* u, Real* xdes, int D, void* stream) {
  MDS_REQUIRE(prm && ref && u && xdes && D > 0, "cbf_prepare: bad argument");
  MDS_REQUIRE(order == 2 || order == 3, "cbf_prepare: order must be 2 or 3");
  cbf_prepare_kernel<Real><<<(D + 255) / 256, 256, 0, (cudaStream_t)stream>>>(to_dev<Real>(*prm), order, Real(u0), ref, u, xdes, D);
  return check_launch("cbf_prepare");
}
template <typename Real> static int xdot_linear_impl(const MdsDroneParams* prm, int kind, const Real* obs, Real* xdot, int D, void* stream) {
  MDS_REQUIRE(prm && obs && xdot && D > 0, "xdot_linear: bad argument");
  MDS_REQUIRE(kind == 12 || kind == 9 || kind == 10, "xdot_linear: kind must be 12, 9 or 10");
  xdot_linear_kernel<Real><<<(D + 255) / 256, 256, 0, (cudaStream_t)stream>>>(to_dev<Real>(*prm), kind, obs, xdot, D);
  return check_launch("xdot_linear");
}
template <typename Real> static int linear_rollout_impl(const MdsDroneParams* prm, const Real* obs_log, double dt, Real* x_out, int T, int D, void* stream) {
  MDS_REQUIRE(prm && obs_log && x_out && T > 0 && D > 0 && dt > 0, "linear_rollout: bad argument");
  linear_rollout_kernel<Real><<<(D + 127) / 128, 128, 0, (cudaStream_t)stream>>>(to_dev<Real>(*prm), obs_log, Real(dt), x_out, T, D);
  return check_launch("linear_rollout");
}
template <typename Real>
static int xdot_nonlinear_impl(const MdsDroneParams* prm, double jx, double jy, double jz, const Real* obs, Real* xdot, int D, void* stream) {
  MDS_REQUIRE(prm && obs && xdot && D > 0 && jx > 0 && jy > 0 && jz > 0, "xdot_nonlinear: bad argument");
  xdot_nonlinear_kernel<Real><<<(D + 255) / 256, 256, 0, (cudaStream_t)stream>>>(to_dev<Real>(*prm), Real(jx), Real(jy), Real(jz), obs, xdot, D);
  return check_launch("xdot_nonlinear");
}
extern "C" int mds_rollout_plan(int E, int N);
extern "C" int mds_device_info(int* sm_count, int* cc_major, int* cc_minor, int* l2_bytes);
// PhysSpec<1> (mds_common.cuh): the swarm configuration of the reference's CBF mains, compiled without its mode switches
static int phys_spec_of(const MdsDroneParams& p) {
  return (p.physics == MDS_PHYSICS_DYN_GND_DRAG_DW && p.drone_model == MDS_DRONE_CF2P && p.substeps == 1 && !p.renormalize_quat && p.ground_clamp &&
          !p.x_frame_mixer) ? 1 : 0;
}
template <typename Real>
static int rollout_impl(const MdsDroneParams* prm, const MdsRolloutCfg* cfg, const MdsGeoGains* geo, const MdsLqrGains* lqr, const MdsCbfParams* cbf,
                        MdsState st, MdsPidState pid, const MdsDslPidGains* dsl, MdsDslPidState dsl_state,
                        const typename TrajSpecT<Real>::spec* specs, const typename TrajSpecT<Real>::seg* segs,
                        Real* obs, Real* action, const Real* fext, Real* obs_log, double* stats, double t0, int K, int E, int N, void* stream) {
  MDS_REQUIRE(prm && cfg && st.pos_wx && st.quat && st.vel_wy && st.rpm && st.wz && specs && obs && action, "rollout: null pointer");
  MDS_REQUIRE(E > 0 && N > 0 && N <= MDS_MAX_DRONES_PER_ENV && K > 0, "rollout: bad E, N or K");
  MDS_REQUIRE(cfg->ctrl >= MDS_CTRL_GEOMETRIC && cfg->ctrl <= MDS_CTRL_DSLPID, "rollout: unknown controller");
  MDS_REQUIRE(cfg->stages == 0 || cfg->stages == 1 || cfg->stages == 2 || cfg->stages == 4 || cfg->stages == 6,
              "rollout: stages must be 0, 1, 2, 4 or 6");
  RolloutP<Real> R;
  memset(&R, 0, sizeof(R));
  R.ctrl = cfg->ctrl; R.use_cbf = cfg->use_cbf; R.n_obs = cfg->num_obstacles; R.write_obs_every = cfg->write_obs_every;
  R.lqr_planes = (const Real*)cfg->lqr_gain_planes_dev; R.lqr_D = E * N;
  MDS_REQUIRE(!R.lqr_planes || lqr_variant_ok(cfg->ctrl), "rollout: per-drone gains need an LQR controller");
  GeoP<Real> G;
  memset(&G, 0, sizeof(G));
  LqrP<Real> L;
  memset(&L, 0, sizeof(L));
  CbfP<Real> C;
  memset(&C, 0, sizeof(C));
  C.order = 2;
  DslP<Real> Dg;
  memset(&Dg, 0, sizeof(Dg));
  DslStateP<Real> Ds = to_dev<Real>(dsl_state);
  if (cfg->ctrl == MDS_CTRL_GEOMETRIC) {
    MDS_REQUIRE(geo, "rollout: geometric gains missing");
    G = to_dev<Real>(*geo);
  } else if (cfg->ctrl == MDS_CTRL_DSLPID) {
    MDS_REQUIRE(dsl && dsl_state.a && dsl_state.b && dsl_state.c, "rollout: DSL PID gains or state missing");
    MDS_REQUIRE(!cfg->use_cbf, "rollout: the CBF filter needs an LQR_OMEGA / LQR_YANK nominal controller");
    Dg = to_dev<Real>(*dsl);
  } else {
    MDS_REQUIRE(lqr && lqr_dim_ok(cfg->ctrl, lqr->dim), "rollout: LQR gains missing or of the wrong dimension");
    L = to_dev<Real>(*lqr);
    if (cfg->ctrl != MDS_CTRL_LQR_TORQUE) MDS_REQUIRE(pid.a && pid.b, "rollout: PID state missing");
  }
  if (cfg->use_cbf) {
    int rc = cbf_args_ok(cbf, N, cfg->num_obstacles);
    if (rc) return rc;
    MDS_REQUIRE((cfg->ctrl == MDS_CTRL_LQR_OMEGA && cbf->order == 2) || (cfg->ctrl == MDS_CTRL_LQR_YANK && cbf->order == 3),
                "rollout: CBF order 2 needs LQR_OMEGA, order 3 needs LQR_YANK");
    C = to_dev<Real>(*cbf);
    rc = qp_scratch_for(N, &C.scr);
    if (rc) return rc;
    for (int i = 0; i < cfg->num_obstacles * 4; ++i) R.obstacles[i] = Real(cfg->obstacles[i]);
    // reference caller: nominal_us[:,0] -= M*G before the QP (CBFTest.py:339, CBFTestOrd3.py:344);
    // added back only for order 2 (CBFTest.py:346 vs CBFTestOrd3.py:350)
    R.u0_pre = Real(prm->m * prm->g);
    R.u0_post = cbf->order == 2 ? Real(prm->m * prm->g) : Real(0);
  } else {
    R.n_obs = 0;
  }
  MDS_REQUIRE(!(cfg->write_obs_every > 0) || obs_log, "rollout: obs_log buffer missing");
  MDS_REQUIRE(cfg->write_obs_every <= 32767, "rollout: write_obs_every must be <= 32767");
  MDS_REQUIRE(cfg->traj_period == 0 || cfg->traj_period == N, "rollout: traj_period must be 0 or the drone count N");
  const int NP = next_pow2(N), threads = R.use_cbf ? cbf_block_threads<Real>(NP, N, R.n_obs) : MDS_BLOCK, epb = threads / NP;
  const int blocks = (E + epb - 1) / epb;
  size_t smem = R.use_cbf ? cbf_smem_bytes<Real>(threads, NP, N, R.n_obs) : 32;
  cudaStream_t cs = (cudaStream_t)stream;
  const DroneP<Real> Pd = to_dev<Real>(*prm);
  const StateP<Real> Sd = to_dev<Real>(st);
  const PidP<Real> Pi = to_dev<Real>(pid);
  const size_t obs_elems = (size_t)E * N * MDS_OBS_DIM;
  // launch plan.  stages 0: mds_rollout_plan(E, N) (= 6, K steps in one launch); 4: two launches (ctrl, physics) per step;
  // 1: controller kernel only; 2: physics kernel only -- 1 then 2 per step lets a caller replay a rollout launch by launch.
  const int mode = cfg->stages == 0 ? mds_rollout_plan(E, N) : cfg->stages;
  auto obs_slot = [&](int j) -> Real* {  // where the observation after physics step j (1-based) goes
    if (R.write_obs_every > 0 && (j % R.write_obs_every) == 0) return obs_log + (size_t)(j / R.write_obs_every - 1) * obs_elems;
    return obs;
  };
  cudaError_t attr_err = cudaSuccess;
  RolloutLaunch<Real> RL{Pd, R, G, L, C, Dg, Ds, Sd, Pi, specs, segs, action, fext, obs, obs_log, stats, E, N, NP, blocks, threads, phys_spec_of(*prm), smem, cs,
                         cfg->traj_period};
  auto keep = [&](cudaError_t e) { if (e != cudaSuccess) attr_err = e; };
  // the loop kernel packs two rare-event counters into 16 bits each: longer runs go out as several launches (whole log periods each)
  auto launch_loop = [&]() {
    RolloutLaunch<Real> RLL = RL;  // the loop kernel has its own block size (MDS_LOOP_BLOCK)
    RLL.threads = R.use_cbf ? cbf_block_threads<Real>(NP, N, R.n_obs, loop_block<Real>()) : loop_block<Real>();
    if (RLL.threads < NP) RLL.threads = NP;
    const int epb_l = RLL.threads / NP;
    RLL.blocks = (E + epb_l - 1) / epb_l;
    RLL.smem = R.use_cbf ? cbf_smem_bytes<Real>(RLL.threads, NP, N, R.n_obs) : 32;
    const int every = R.write_obs_every;
    int chunk = 16384;
    if (every > 0) chunk = every >= 16384 ? every : (16384 / every) * every;
    for (int k0 = 0; k0 < K; k0 += chunk) {
      RolloutLaunch<Real> part = RLL;
      if (every > 0) part.obs_log = obs_log + (size_t)(k0 / every) * obs_elems;
      keep(launch_loop_kernel<Real>(part, t0 + k0 * prm->dt_ctrl, prm->dt_ctrl, K - k0 < chunk ? K - k0 : chunk));
    }
  };
  bool first_ctrl = true;
  auto launch_ctrl = [&](double t, Real* obs_ptr) {
    keep(launch_ctrl_kernel<Real>(RL, t, obs_ptr, first_ctrl));
    first_ctrl = false;
  };
  auto launch_phys = [&](Real* obs_out) {
    if (N == 8) physics_step_kernel<Real, 8><<<blocks, threads, 0, cs>>>(Pd, Sd, action, fext, obs_out, E, N, NP);
    else physics_step_kernel<Real, 0><<<blocks, threads, 0, cs>>>(Pd, Sd, action, fext, obs_out, E, N, NP);
  };
  const double dt = prm->dt_ctrl;
  Real* obs_last = obs;  // buffer holding the newest observation
  if (mode == 1) {
    for (int k = 0; k < K; ++k) launch_ctrl(t0 + k * dt, obs);
  } else if (mode == 2) {
    for (int k = 0; k < K; ++k) { obs_last = obs_slot(k + 1); launch_phys(obs_last); }
  } else if (mode == 4) {
    for (int k = 0; k < K; ++k) {
      launch_ctrl(t0 + k * dt, obs_last);
      obs_last = obs_slot(k + 1);
      launch_phys(obs_last);
    }
  } else {
    launch_loop();  // writes the final observation to `obs` itself
  }
  if (attr_err != cudaSuccess) return cuda_fail("rollout: shared memory opt-in failed", attr_err);
  if (obs_last != obs) {
    cudaError_t e = cudaMemcpyAsync(obs, obs_last, obs_elems * sizeof(Real), cudaMemcpyDeviceToDevice, cs);
    if (e != cudaSuccess) return fail(MDS_ERR_LAUNCH, "rollout: %s", cudaGetErrorString(e));
  }
  return check_launch("rollout");
}

// The checks of the fused learning rollouts after their model checks: sizes, physics and the observation log
static int learn_shape_checks(const MdsDroneParams* prm, const MdsRlsCfg* rls, int write_obs_every, const void* obs_log, int K, int E, int N,
                              const char* who) {
  if (!(rls->dt > 0.0 && rls->drones_per_env == N)) return fail(MDS_ERR_ARG, "%s: dt must be positive and drones_per_env equal to N", who);
  if (!(K >= 0 && E > 0 && N >= 1 && N <= MDS_MAX_DRONES_PER_ENV)) return fail(MDS_ERR_ARG, "%s: bad K, E or N", who);
  if (prm->substeps < 1) return fail(MDS_ERR_ARG, "%s: substeps must be >= 1", who);
  if (prm->physics != MDS_PHYSICS_DYN && prm->physics != MDS_PHYSICS_DYN_GND_DRAG_DW) return fail(MDS_ERR_ARG, "%s: unknown physics mode", who);
  if (write_obs_every > 0 && !obs_log) return fail(MDS_ERR_ARG, "%s: obs_log buffer missing", who);
  return MDS_OK;
}
template <typename Real>
static int learning_rollout_impl(const MdsDroneParams* prm, const MdsRlsCfg* rls, int variant, int learn_from, int write_obs_every, MdsState st,
                                 MdsPidState pid, const typename TrajSpecT<Real>::spec* specs, const typename TrajSpecT<Real>::seg* segs,
                                 const Real* inputs, const Real* gain, Real* theta, Real* Pm, Real* resid, Real* obs, const Real* fext, Real* obs_log,
                                 double t0, int K, int E, int N, void* stream) {
  // inputs [K][D*4] may be NULL when K = 0 (an empty excitation tensor has no storage); gain: NULL flies the inputs open loop
  MDS_REQUIRE(prm && rls && st.pos_wx && st.quat && st.vel_wy && st.rpm && st.wz && pid.a && pid.b && specs && (inputs || K == 0) && theta && Pm &&
                  obs,
              "learning_rollout: null pointer");
  MDS_REQUIRE(variant == MDS_CTRL_LQR_OMEGA || variant == MDS_CTRL_LQR_YANK, "learning_rollout: variant must be LQR_OMEGA or LQR_YANK");
  MDS_REQUIRE((variant == MDS_CTRL_LQR_OMEGA && rls->m == 9) || (variant == MDS_CTRL_LQR_YANK && rls->m == 10),
              "learning_rollout: m must be 9 with LQR_OMEGA and 10 with LQR_YANK");
  RlsP c;
  if (const int rc = rls_params(rls, "learning_rollout", &c)) return rc;
  // project_theta exists for the 10-dim crazyflie model only (decentralized_yolqr_crazyflie.py:245-257); the m = 9 kernel carries none
  MDS_REQUIRE(!(rls->m == 9 && rls->project != MDS_RLS_PROJECT_NONE), "learning_rollout: project_theta is defined for m = 10 only");
  if (const int rc = learn_shape_checks(prm, rls, write_obs_every, obs_log, K, E, N, "learning_rollout")) return rc;
  if (K == 0) return MDS_OK;
  LearnLaunch<Real> a{to_dev<Real>(*prm), c, rls->m, rls->project != MDS_RLS_PROJECT_NONE, learn_from, write_obs_every > 0 ? write_obs_every : 0,
                      to_dev<Real>(st), to_dev<Real>(pid), specs, segs, inputs, gain, 0, theta, Pm, resid, obs, fext, obs_log, t0, prm->dt_ctrl, K, E,
                      N, (cudaStream_t)stream};
  const cudaError_t e = launch_learn_kernel<Real>(a);
  if (e != cudaSuccess) return cuda_fail("learning_rollout: shared-memory opt-in", e);
  return check_launch("learning_rollout");
}

// The 12-dim torque-level model: no inner loop and no PID state; both of its reference methods project theta.  gain NULL: open
// loop; coupled: gain holds the robot-coupled [N][48][D] planes, otherwise the per-drone [48][D] planes.
template <typename Real>
static int learning_rollout_torque_impl(const MdsDroneParams* prm, const MdsRlsCfg* rls, int learn_from, int write_obs_every, MdsState st,
                                        const typename TrajSpecT<Real>::spec* specs, const typename TrajSpecT<Real>::seg* segs, const Real* inputs,
                                        const Real* gain, int coupled, Real* theta, Real* Pm, Real* resid, Real* obs, const Real* fext, Real* obs_log,
                                        double t0, int K, int E, int N, void* stream) {
  MDS_REQUIRE(prm && rls && st.pos_wx && st.quat && st.vel_wy && st.rpm && st.wz && specs && (inputs || K == 0) && theta && Pm && obs,
              "learning_rollout_torque: null pointer");
  MDS_REQUIRE(rls->m == 12, "learning_rollout_torque: m must be 12");
  RlsP c;
  if (const int rc = rls_params(rls, "learning_rollout_torque", &c)) return rc;
  MDS_REQUIRE(rls->project != MDS_RLS_PROJECT_NONE,
              "learning_rollout_torque: project must be AFTER (theta_update) or LOOP (approx_theta_update): both methods project theta");
  MDS_REQUIRE(!coupled || gain, "learning_rollout_torque: a coupled law needs a gain");
  if (const int rc = learn_shape_checks(prm, rls, write_obs_every, obs_log, K, E, N, "learning_rollout_torque")) return rc;
  if (K == 0) return MDS_OK;
  LearnLaunch<Real> a{to_dev<Real>(*prm), c, 12, 1, learn_from, write_obs_every > 0 ? write_obs_every : 0, to_dev<Real>(st), PidP<Real>{nullptr, nullptr},
                      specs, segs, inputs, gain, coupled ? 1 : 0, theta, Pm, resid, obs, fext, obs_log, t0, prm->dt_ctrl, K, E, N,
                      (cudaStream_t)stream};
  const cudaError_t e = launch_learn_torque_kernel<Real>(a);
  if (e != cudaSuccess) return cuda_fail("learning_rollout_torque: shared-memory opt-in", e);
  return check_launch("learning_rollout_torque");
}

extern "C" {

int mds_abi_version(void) { return MDS_ABI_VERSION; }
const char* mds_last_error(void) { return g_err; }
int mds_device_info(int* sm_count, int* cc_major, int* cc_minor, int* l2_bytes) {
  int dev = 0;
  cudaError_t e = cudaGetDevice(&dev);
  if (e != cudaSuccess) return fail(MDS_ERR_LAUNCH, "device_info: %s", cudaGetErrorString(e));
  cudaDeviceProp p;
  e = cudaGetDeviceProperties(&p, dev);
  if (e != cudaSuccess) return fail(MDS_ERR_LAUNCH, "device_info: %s", cudaGetErrorString(e));
  if (sm_count) *sm_count = p.multiProcessorCount;
  if (cc_major) *cc_major = p.major;
  if (cc_minor) *cc_minor = p.minor;
  if (l2_bytes) *l2_bytes = p.l2CacheSize;
  return MDS_OK;
}
// ---- plain-host helpers: let a caller without a CUDA-aware array library (the reference is numpy-only) own
// device buffers and move host arrays across the boundary
int mds_device_alloc(size_t bytes, void** out_dev) {
  MDS_REQUIRE(out_dev && bytes > 0, "device_alloc: bad argument");
  cudaError_t e = cudaMalloc(out_dev, bytes);
  if (e != cudaSuccess) return fail(MDS_ERR_LAUNCH, "device_alloc: %s", cudaGetErrorString(e));
  e = cudaMemset(*out_dev, 0, bytes);
  if (e != cudaSuccess) return fail(MDS_ERR_LAUNCH, "device_alloc: %s", cudaGetErrorString(e));
  return MDS_OK;
}
int mds_device_free(void* dev) {
  cudaError_t e = cudaFree(dev);
  if (e != cudaSuccess) return fail(MDS_ERR_LAUNCH, "device_free: %s", cudaGetErrorString(e));
  return MDS_OK;
}
int mds_copy_to_device(void* dst_dev, const void* src_host, size_t bytes, void* stream) {
  MDS_REQUIRE(dst_dev && src_host, "copy_to_device: null pointer");
  cudaError_t e = cudaMemcpyAsync(dst_dev, src_host, bytes, cudaMemcpyHostToDevice, (cudaStream_t)stream);
  if (e != cudaSuccess) return fail(MDS_ERR_LAUNCH, "copy_to_device: %s", cudaGetErrorString(e));
  return MDS_OK;
}
int mds_copy_to_host(void* dst_host, const void* src_dev, size_t bytes, void* stream) {
  MDS_REQUIRE(dst_host && src_dev, "copy_to_host: null pointer");
  cudaError_t e = cudaMemcpyAsync(dst_host, src_dev, bytes, cudaMemcpyDeviceToHost, (cudaStream_t)stream);
  if (e != cudaSuccess) return fail(MDS_ERR_LAUNCH, "copy_to_host: %s", cudaGetErrorString(e));
  return MDS_OK;
}
int mds_stream_synchronize(void* stream) {
  cudaError_t e = cudaStreamSynchronize((cudaStream_t)stream);
  if (e != cudaSuccess) return fail(MDS_ERR_LAUNCH, "stream_synchronize: %s", cudaGetErrorString(e));
  return MDS_OK;
}
// Measured on B200 (tools/exp_plans.py, tools/exp_c2.py): the K-steps-in-one-launch plan (6) is the fastest at every
// size and precision -- C2 4096 envs 1.8 us per step vs 8.3 (one fused launch per step, a plan since removed) / 11.3 (two
// launches); C5 1M drones fp32 0.127 ms vs 0.140 / 0.132; fp64 0.305 ms vs 0.50 / 0.44 -- so stages == 0 always selects it.
// 4 remains as the per-call reference with the observation in HBM after every step, 1 / 2 for launch-by-launch replays.
int mds_rollout_plan(int E, int N) { (void)E; (void)N; return 6; }
int mds_cbf_num_rows(int order, int N, int n_obs) { return N * (N - 1) / 2 + 8 * N + (order == 3 ? 2 * N : 0) + N * n_obs; }

#define MDS_DEFINE(SUF, REAL, SPEC, SEG)                                                                                                          \
  int mds_physics_step_##SUF(const MdsDroneParams* prm, MdsState st, const REAL* action, const REAL* fext, REAL* obs, int E, int N, void* stream) { \
    return physics_step_impl<REAL>(prm, st, action, fext, obs, E, N, stream);                                                                      \
  }                                                                                                                                                \
  int mds_physics_step_host_##SUF(const MdsDroneParams* prm, MdsState st, const REAL* action_host, REAL* action_dev, REAL* obs_dev,              \
                                  REAL* obs_host, int E, int N, void* stream) {                                                                   \
    MDS_REQUIRE(action_host && action_dev && obs_dev && obs_host && E > 0 && N > 0, "physics_step_host: bad argument");                             \
    const size_t D = (size_t)E * N;                                                                                                                \
    int rc = mds_copy_to_device(action_dev, action_host, D * 4 * sizeof(REAL), stream);                                                            \
    if (rc) return rc;                                                                                                                             \
    rc = physics_step_impl<REAL>(prm, st, action_dev, (const REAL*)nullptr, obs_dev, E, N, stream);                                                \
    if (rc) return rc;                                                                                                                             \
    rc = mds_copy_to_host(obs_host, obs_dev, D * MDS_OBS_DIM * sizeof(REAL), stream);                                                              \
    if (rc) return rc;                                                                                                                             \
    return mds_stream_synchronize(stream);                                                                                                         \
  }                                                                                                                                                \
  int mds_obs_from_state_##SUF(const MdsDroneParams* prm, MdsState st, REAL* obs, int D, void* stream) {                                           \
    return obs_from_state_impl<REAL>(prm, st, obs, D, stream);                                                                                     \
  }                                                                                                                                                \
  int mds_traj_eval_##SUF(const SPEC* specs, const SEG* segs, double t, REAL* ref, int D, void* stream) {                                          \
    return traj_eval_impl<REAL>(specs, segs, t, ref, D, stream);                                                                                   \
  }                                                                                                                                                \
  int mds_geometric_ctrl_##SUF(const MdsDroneParams* prm, const MdsGeoGains* g, const REAL* obs, const REAL* ref, REAL* action, REAL* u, int D,    \
                               void* stream) {                                                                                                     \
    return geometric_impl<REAL>(prm, g, obs, ref, action, u, D, stream);                                                                           \
  }                                                                                                                                                \
  int mds_dslpid_ctrl_##SUF(const MdsDroneParams* prm, const MdsDslPidGains* g, const REAL* obs, const REAL* target, MdsDslPidState st,          \
                            REAL* action, REAL* pos_e, int D, void* stream) {                                                                    \
    return dslpid_impl<REAL>(prm, g, obs, target, st, action, pos_e, D, stream);                                                                  \
  }                                                                                                                                                \
  int mds_lqr_ctrl_##SUF(const MdsDroneParams* prm, const MdsLqrGains* g, int variant, const REAL* obs, const REAL* ref, REAL* u, REAL* action,    \
                         MdsPidState pid, int D, void* stream) {                                                                                   \
    return lqr_impl<REAL>(prm, g, variant, obs, ref, u, action, pid, D, stream);                                                                   \
  }                                                                                                                                                \
  int mds_rls_update_##SUF(const MdsRlsCfg* cfg, const REAL* phi, const REAL* xtp1, REAL* theta, REAL* Pm, REAL* resid, int D, void* stream) {          \
    return rls_impl<REAL>(cfg, phi, xtp1, theta, Pm, resid, D, stream);                                                                            \
  }                                                                                                                                                \
  int mds_care_gains_##SUF(int m, const double* q, const double* r, const REAL* theta, REAL* K, int* status, int D, void* stream) {                 \
    return care_impl<REAL>(m, q, r, theta, K, status, D, stream);                                                                                  \
  }                                                                                                                                                \
  int mds_care_gains_coupled_##SUF(int m, const double* q, const double* r, const double* q_cross, const REAL* theta, REAL* K, int* status, int E, \
                                   int N, void* stream) {                                                                                         \
    return care_coupled_impl<REAL>(m, q, r, q_cross, theta, K, status, E, N, stream);                                                            \
  }                                                                                                                                                \
  int mds_state_feedback_##SUF(int variant, const REAL* K, const REAL* x, const REAL* xdes, REAL* e, REAL* u, int D, void* stream) {                \
    return state_feedback_impl<REAL>(variant, K, x, xdes, e, u, D, stream);                                                                        \
  }                                                                                                                                                \
  int mds_error_state_##SUF(const MdsDroneParams* prm, int variant, const REAL* obs, const REAL* ref, REAL* e, int D, void* stream) {              \
    return error_state_impl<REAL>(prm, variant, obs, ref, e, D, stream);                                                                           \
  }                                                                                                                                                \
  int mds_dlqr_ctrl_##SUF(const MdsDroneParams* prm, int variant, const REAL* K, int coupled, const REAL* obs, const REAL* ref, REAL* u,           \
                          REAL* action, MdsPidState pid, int E, int N, void* stream) {                                                             \
    return dlqr_impl<REAL>(prm, variant, K, coupled, obs, ref, u, action, pid, E, N, stream);                                                      \
  }                                                                                                                                                \
  int mds_lowlevel_##SUF(const MdsDroneParams* prm, int variant, const REAL* u, const REAL* obs, MdsPidState pid, REAL* action, int D,             \
                         void* stream) {                                                                                                           \
    return lowlevel_impl<REAL>(prm, variant, u, obs, pid, action, D, stream);                                                                      \
  }                                                                                                                                                \
  int mds_cbf_qp_##SUF(const MdsDroneParams* prm, const MdsCbfParams* c, const REAL* obs, const REAL* xdes, const REAL* unom,                      \
                       const REAL* obstacles, int n_obs, REAL* usafe, int* status, int* iters, int E, int N, void* stream) {                       \
    return cbf_qp_impl<REAL>(prm, c, obs, xdes, unom, obstacles, n_obs, usafe, status, iters, E, N, stream);                                       \
  }                                                                                                                                                \
  int mds_cbf_rows_##SUF(const MdsDroneParams* prm, const MdsCbfParams* c, const REAL* obs, const REAL* xdes, const REAL* obstacles, int n_obs,    \
                         REAL* Gm, REAL* h, int E, int N, void* stream) {                                                                          \
    return cbf_rows_impl<REAL>(prm, c, obs, xdes, obstacles, n_obs, Gm, h, E, N, stream);                                                          \
  }                                                                                                                                                \
  int mds_cbf_prepare_##SUF(const MdsDroneParams* prm, int order, double u0, const REAL* ref, REAL* u, REAL* xdes, int D, void* stream) {        \
    return cbf_prepare_impl<REAL>(prm, order, u0, ref, u, xdes, D, stream);                                                                        \
  }                                                                                                                                                \
  int mds_xdot_linear_##SUF(const MdsDroneParams* prm, int kind, const REAL* obs, REAL* xdot, int D, void* stream) {                               \
    return xdot_linear_impl<REAL>(prm, kind, obs, xdot, D, stream);                                                                                \
  }                                                                                                                                                \
  int mds_linear_rollout_##SUF(const MdsDroneParams* prm, const REAL* obs_log, double dt, REAL* x_out, int T, int D, void* stream) {               \
    return linear_rollout_impl<REAL>(prm, obs_log, dt, x_out, T, D, stream);                                                                       \
  }                                                                                                                                                \
  int mds_xdot_nonlinear_##SUF(const MdsDroneParams* prm, double jx, double jy, double jz, const REAL* obs, REAL* xdot, int D, void* stream) {     \
    return xdot_nonlinear_impl<REAL>(prm, jx, jy, jz, obs, xdot, D, stream);                                                                       \
  }                                                                                                                                                \
  int mds_rollout_##SUF(const MdsDroneParams* prm, const MdsRolloutCfg* cfg, const MdsGeoGains* geo, const MdsLqrGains* lqr,                       \
                        const MdsCbfParams* cbf, MdsState st, MdsPidState pid, const MdsDslPidGains* dsl, MdsDslPidState dsl_state,                \
                        const SPEC* specs, const SEG* segs, REAL* obs, REAL* action, const REAL* fext, REAL* obs_log, double* stats, double t0,    \
                        int K, int E, int N, void* stream) {                                                                                       \
    return rollout_impl<REAL>(prm, cfg, geo, lqr, cbf, st, pid, dsl, dsl_state, specs, segs, obs, action, fext, obs_log, stats, t0, K, E, N,      \
                              stream);                                                                                                             \
  }                                                                                                                                                \
  int mds_learning_rollout_##SUF(const MdsDroneParams* prm, const MdsRlsCfg* rls, int variant, int learn_from, int write_obs_every, MdsState st,     \
                                 MdsPidState pid, const SPEC* specs, const SEG* segs, const REAL* inputs, REAL* theta, REAL* Pm, REAL* resid,      \
                                 REAL* obs, const REAL* fext, REAL* obs_log, double t0, int K, int E, int N, void* stream) {                       \
    return learning_rollout_impl<REAL>(prm, rls, variant, learn_from, write_obs_every, st, pid, specs, segs, inputs, (const REAL*)nullptr, theta,  \
                                       Pm, resid, obs, fext, obs_log, t0, K, E, N, stream);                                                        \
  }                                                                                                                                                \
  int mds_learning_rollout_feedback_##SUF(const MdsDroneParams* prm, const MdsRlsCfg* rls, int variant, int learn_from, int write_obs_every,       \
                                          MdsState st, MdsPidState pid, const SPEC* specs, const SEG* segs, const REAL* inputs,                    \
                                          const REAL* gain, REAL* theta, REAL* Pm, REAL* resid, REAL* obs, const REAL* fext, REAL* obs_log,        \
                                          double t0, int K, int E, int N, void* stream) {                                                          \
    MDS_REQUIRE(gain, "learning_rollout: null gain pointer");                                                                                      \
    return learning_rollout_impl<REAL>(prm, rls, variant, learn_from, write_obs_every, st, pid, specs, segs, inputs, gain, theta, Pm, resid, obs,  \
                                       fext, obs_log, t0, K, E, N, stream);                                                                        \
  }                                                                                                                                                \
  int mds_learning_rollout_torque_##SUF(const MdsDroneParams* prm, const MdsRlsCfg* rls, int learn_from, int write_obs_every, MdsState st,         \
                                        const SPEC* specs, const SEG* segs, const REAL* inputs, const REAL* gain, int coupled, REAL* theta, REAL* Pm, \
                                        REAL* resid, REAL* obs, const REAL* fext, REAL* obs_log, double t0, int K, int E, int N, void* stream) {     \
    return learning_rollout_torque_impl<REAL>(prm, rls, learn_from, write_obs_every, st, specs, segs, inputs, gain, coupled, theta, Pm, resid, obs, \
                                              fext, obs_log, t0, K, E, N, stream);                                                                 \
  }

MDS_DEFINE(f32, float, MdsTrajSpecF32, MdsTrajSegF32)
MDS_DEFINE(f64, double, MdsTrajSpecF64, MdsTrajSegF64)

int mds_fma_peak(int use_f64, int iters, double* tflops_out, void* stream) {
  MDS_REQUIRE(tflops_out && iters > 0, "fma_peak: bad argument");
  int sms = 0;
  int rc = mds_device_info(&sms, nullptr, nullptr, nullptr);
  if (rc) return rc;
  const int threads = 512, blocks = sms * 4;
  iters = (iters + 15) & ~15;
  void* buf = nullptr;
  cudaError_t e = cudaMalloc(&buf, (size_t)threads * blocks * sizeof(double));
  if (e != cudaSuccess) return fail(MDS_ERR_LAUNCH, "fma_peak: %s", cudaGetErrorString(e));
  cudaEvent_t a, b;
  cudaEventCreate(&a);
  cudaEventCreate(&b);
  cudaStream_t s = (cudaStream_t)stream;
  float best = 1e30f;
  for (int rep = 0; rep < 4; ++rep) {
    cudaEventRecord(a, s);
    if (use_f64) fma_peak_kernel<double><<<blocks, threads, 0, s>>>((double*)buf, iters);
    else fma_peak_kernel<float><<<blocks, threads, 0, s>>>((float*)buf, iters);
    cudaEventRecord(b, s);
    cudaEventSynchronize(b);
    float ms = 0.f;
    cudaEventElapsedTime(&ms, a, b);
    if (rep > 0 && ms < best) best = ms;
  }
  cudaEventDestroy(a);
  cudaEventDestroy(b);
  cudaFree(buf);
  rc = check_launch("fma_peak");
  if (rc) return rc;
  double flops = 2.0 * 16.0 * (double)iters * (double)threads * (double)blocks;
  *tflops_out = flops / ((double)best * 1e-3) / 1e12;
  return MDS_OK;
}

}  // extern "C"
