// mds_learn.cuh -- the system-identification loop of the decentralised LQR (the warm-up / learning phases of the reference's
// simulations/CBFTest.py:150-265, CBFTestOrd3.py:150-270) as ONE launch for K control steps:
//   ref_k = eval(t0 + k dt);  e_t = error_state(obs, ref_k);  action = low_level(u[k], obs);  obs = env.step(action);
//   e_t+1 = error_state(obs, ref_k);  if k >= learn_from: RLS step with phi = [e_t, u[k]], x1 = e_t+1
// which is what the per-call loop does with mds_error_state, mds_lowlevel, mds_physics_step and mds_rls_update.
// One thread per drone in env lane groups (mds_rollout.cuh), so the downwash exchange of the physics step is the rollout's.
// Each thread stages its drone's theta and packed upper triangle of P in shared memory once ([entry][thread], as
// rls_update_kernel does), keeps them there for all K steps and writes theta and both triangles of P back at the end;
// state, observation, PID state and trajectory descriptor stay in registers.  Per step HBM sees u[k] (16 or 32 B per
// drone) and the observation-log slot when one is due.
#pragma once
#include <cuda_runtime.h>
#include "mds_learn_launch.cuh"
#include "mds_rollout.cuh"

// ---- the sweeps of one RLS step over a thread's staged columns: the arithmetic of rls_update_kernel (mds_sysid.cuh) in the
// same order, with a run-time thread stride T.  Shared memory is [entry][thread]; sP is the packed upper triangle of P, sT
// theta, s_phi / s_w / s_term scratch columns (MN, MN, M entries), all already offset to the calling thread.
// (rls_update_kernel keeps its own copy: calling these from it changed its fp64 SASS by 16-24 instructions per variant.)

// project_theta before the update (MDS_RLS_PROJECT_LOOP, robots after the first of an env): s_code holds the codes per theta row
template <typename Real, int M> MDS_DEV void rls_pre_project(Real* sT, const unsigned* s_code, int T) {
  constexpr int MN = M + 4;
#pragma unroll 1
  for (int i = 0; i < MN; ++i) {
    const unsigned word = s_code[i];
#pragma unroll
    for (int j = 0; j < M; ++j) {
      const unsigned code = (word >> (2 * j)) & 3u;
      if (code != 1u) sT[(i * M + j) * T] = code == 0u ? Real(0) : Real(1);
    }
  }
}

// gain: w = P phi (= v'), s = 1 + phi' P phi; returns s.  v[] must be zero on entry and holds w on return (also in s_w).
// Row i of the triangle holds P(i, j >= i): it contributes P(i,j) phi_j to w_i and, for j > i, P(i,j) phi_i to w_j.  The
// run-time row loop of the fp64 RLS kernel in both precisions (the fully unrolled fp32 form takes 255 registers on its own):
// the row's own part of w_i goes to shared memory, the transposed contributions to v[j] with static j.
template <typename Real, int MN>
MDS_DEV Real rls_gain(const Real* sP, const Real* s_phi, Real* s_w, const Real (&phi)[MN], Real (&v)[MN], int T) {
  Real s = Real(1);
#pragma unroll 2
  for (int i = 0; i < MN; ++i) {
    const Real phi_i = s_phi[i * T];
    Real wi = Real(0);
    const int row0 = i * MN - i * (i - 1) / 2 - i;  // rls_tri(i, j) = row0 + j
#pragma unroll
    for (int j = 0; j < MN; ++j) {
      if (j >= i) {
        const Real p = sP[(row0 + j) * T];
        wi += p * phi[j];
        if (j > i) v[j] += p * phi_i;
      }
    }
    s_w[i * T] = wi;
  }
#pragma unroll
  for (int i = 0; i < MN; ++i) v[i] += s_w[i * T];
#pragma unroll
  for (int i = 0; i < MN; ++i) { s_w[i * T] = v[i]; s += phi[i] * v[i]; }
  return s;
}

// regression residual r (m) of the staged theta: est_x_dot - theta' phi (XDOT) or x1 - forward_predict (PREDICT)
template <typename Real, int M>
MDS_DEV void rls_residual(const RlsP& c, const Real (&phi)[M + 4], const Real (&x1)[M], const Real* s_phi, const Real* sT, Real* s_term,
                          Real (&r)[M], int T) {
  constexpr int MN = M + 4;
  if (c.target == MDS_RLS_TARGET_XDOT) {
    // est_x_dot, then x_dot - theta' phi
    const Real inv_dt = Real(1.0 / c.dt);
    if (M == 12) {  // decentralized_lqr.py:185-198
#pragma unroll
      for (int k = 0; k < 3; ++k) {
        r[k] = x1[3 + k];
        r[3 + k] = (x1[3 + k] - phi[3 + k]) * inv_dt;
        r[6 + k] = (x1[6 + k] - phi[6 + k]) * inv_dt;
        r[9 + k] = x1[6 + k];
      }
    } else {  // decentralized_yolqr_crazyflie.py:228-243 (m = 10; m = 9 is rejected on the host)
#pragma unroll
      for (int k = 0; k < 3; ++k) {
        r[k] = phi[M + 1 + k];
        r[4 + k] = (x1[4 + k] - phi[4 + k]) * inv_dt;
        r[7 + k] = x1[4 + k];
      }
      r[3] = phi[M];
    }
#pragma unroll kRlsRowUnroll
    for (int i = 0; i < MN; ++i) {
      const Real phi_i = s_phi[i * T];
#pragma unroll
      for (int j = 0; j < M; ++j) r[j] -= sT[(i * M + j) * T] * phi_i;
    }
  } else {
    // forward_predict: e' = Ahat e + Bhat u over dt from e0, Ahat = theta[:m]^T, Bhat = theta[m:]^T.  The reference runs
    // scipy RK45 (its error over one 1/240 s step is far below its 1e-3 tolerance); here the exact solution
    // e(dt) = e0 + sum_{k>=1} dt^k / k! A^(k-1) (A e0 + B u), summed until the terms vanish in Real.
    Real acc[M], nt[M];
#pragma unroll
    for (int j = 0; j < M; ++j) {
      acc[j] = c.predict_from_xtp1 ? x1[j] : phi[j];
      s_term[j * T] = acc[j];
      nt[j] = Real(0);
    }
#pragma unroll kRlsRowUnroll
    for (int i = 0; i < MN; ++i) {  // A e0 + B u = theta' [e0; u]
      const Real zi = i < M ? s_term[i * T] : s_phi[i * T];
#pragma unroll
      for (int j = 0; j < M; ++j) nt[j] += sT[(i * M + j) * T] * zi;
    }
    Real coef = Real(c.dt);
    const Real eps = sizeof(Real) == 4 ? Real(1e-9) : Real(1e-18);
#pragma unroll 1
    for (int k = 1; k <= 16; ++k) {
      Real big = Real(0), mag = Real(0);
#pragma unroll
      for (int j = 0; j < M; ++j) {
        const Real inc = coef * nt[j];
        acc[j] += inc;
        big = max_(big, abs_(inc)); mag = max_(mag, abs_(acc[j]));
        s_term[j * T] = nt[j]; nt[j] = Real(0);
      }
      if (big <= eps * mag) break;  // the series has converged in Real (|A| dt ~ 0.05: 5-7 terms)
      coef *= Real(c.dt) / Real(k + 1);
#pragma unroll kRlsRowUnroll
      for (int i = 0; i < M; ++i) {
        const Real ti = s_term[i * T];
#pragma unroll
        for (int j = 0; j < M; ++j) nt[j] += sT[(i * M + j) * T] * ti;
      }
    }
#pragma unroll
    for (int j = 0; j < M; ++j) r[j] = x1[j] - acc[j];
  }
}

// Threads per block: the RLS kernel's (one warp in fp32, half a warp in fp64; the staged columns set the occupancy),
// raised to the lane-group size NP where that is larger.  Both are at most 32.
template <typename Real, int M> static int learn_threads(int NP) { return rls_threads<Real, M>() > NP ? rls_threads<Real, M>() : NP; }

// M = 9: DecentralizedLQROmega (LQR_OMEGA error state, ThrustOmega inner loop); M = 10: the yank-omega variants (LQR_YANK,
// YankOmega inner loop).  PROJECT: project_theta is applied (approx_theta_update(project=True)), compile-time like the RLS kernel.
template <typename Real, int M, bool PROJECT>
__global__ void __launch_bounds__(32) learn_rollout_kernel(DroneP<Real> P, RlsP c, StateP<Real> st, PidP<Real> pid,
                                                           const typename TrajSpecT<Real>::spec* __restrict__ specs,
                                                           const typename TrajSpecT<Real>::seg* __restrict__ segs,
                                                           const Real* __restrict__ inputs, Real* __restrict__ theta, Real* __restrict__ Pm,
                                                           Real* __restrict__ resid_out, Real* __restrict__ obs, const Real* __restrict__ fext,
                                                           Real* __restrict__ obs_log, double t0, double dt_ctrl, int learn_from, int write_obs_every,
                                                           int K, int E, int N, int NP) {
  constexpr int MN = M + 4, TRI = MN * (MN + 1) / 2;
  constexpr int CTRL = M == 9 ? MDS_CTRL_LQR_OMEGA : MDS_CTRL_LQR_YANK;
  using R4 = typename Vec4T<Real>::type;
  extern __shared__ __align__(16) unsigned char learn_smem[];
  __shared__ R4 sm_pos[32];  // downwash positions of the block's lane groups
  __shared__ unsigned s_code[16];
  const int T = blockDim.x, tid = threadIdx.x;
  if (PROJECT && tid == 0) {
#pragma unroll
    for (int i = 0; i < MN; ++i) s_code[i] = c.row_code[i];
  }
  if (PROJECT) __syncthreads();  // the only block barrier, before any thread leaves
  const GroupMap g = group_map(N, NP, E);
  if (!g.env_valid) return;  // whole lane groups leave together
  Real* sP = reinterpret_cast<Real*>(learn_smem) + tid;  // packed upper triangle of P: entry (i, j >= i) at sP[rls_tri<MN>(i, j) * T]
  Real* sT = sP + TRI * T;
  Real* s_phi = sT + MN * M * T;
  Real* s_w = s_phi + MN * T;
  Real* s_term = s_w + MN * T;
  const size_t D = (size_t)E * N, d = (size_t)g.d;
  Drone<Real> s;
  Pid<Real> ps;
  Obs<Real> o;
  typename TrajSpecT<Real>::spec spec;
  V3<Real> fx = {Real(0), Real(0), Real(0)};
  if (g.valid) {
#pragma unroll 1
    for (int i = 0; i < MN; ++i)
#pragma unroll 1
      for (int j = i; j < MN; ++j) cp_async_real(sP + rls_tri<MN>(i, j) * T, Pm + (size_t)(i * MN + j) * D + d);
#pragma unroll 1
    for (int k = 0; k < MN * M; ++k) cp_async_real(sT + k * T, theta + (size_t)k * D + d);
    s = load_drone(st, g.d);
    ps = load_pid(pid, g.d);
    o = load_obs(obs, g.d);
    spec = specs[g.d];
    if (fext) fx = {fext[3 * d], fext[3 * d + 1], fext[3 * d + 2]};
    cp_async_wait_all();
  }
  // robots after the first of an env see the projection of the earlier robots' loop iterations before their own update
  const bool pre_project = PROJECT && c.project == MDS_RLS_PROJECT_LOOP && (g.n != 0);
  const size_t obs_elems = D * MDS_OBS_DIM;
  int log_countdown = write_obs_every;  // steps until the next log slot is due
  Real* log_slot = obs_log;
  for (int k = 0; k < K; ++k) {
    Real e0[12], u[4], rpm[4] = {Real(0), Real(0), Real(0), Real(0)};
    Ref<Real> ref;
    if (g.valid) {
      ref = eval_traj<Real>(spec, segs, t0 + (double)k * dt_ctrl);  // the time expression of the rollout kernel and its host plans
      lqr_error_state(P, CTRL, o, ref, e0);
      load4(inputs + (size_t)k * D * 4, g.d, u);
      low_level(P, CTRL, ps, u, o, rpm);
    }
    o = physics_core<0>(P, s, rpm, fx, sm_pos + (tid - g.n), g, N, NP);
    if (write_obs_every > 0 && --log_countdown == 0) {
      if (g.valid) store_obs(log_slot, g.d, o, true);  // streaming stores: the log is write-once
      log_slot += obs_elems;
      log_countdown = write_obs_every;
    }
    if (!g.valid || k < learn_from) continue;
    // ---- one RLS step in the staged columns: phi = [e_t, u], x1 = e_t+1 against the same reference sample
    Real e1[12], phi[MN], x1[M], v[MN];
    lqr_error_state(P, CTRL, o, ref, e1);
#pragma unroll
    for (int i = 0; i < MN; ++i) { phi[i] = i < M ? e0[i] : u[i - M]; s_phi[i * T] = phi[i]; v[i] = Real(0); }
#pragma unroll
    for (int i = 0; i < M; ++i) x1[i] = e1[i];
    if (pre_project) rls_pre_project<Real, M>(sT, s_code, T);
    const Real inv_s = Real(1) / rls_gain<Real, MN>(sP, s_phi, s_w, phi, v, T);
    Real r[M];
    rls_residual<Real, M>(c, phi, x1, s_phi, sT, s_term, r, T);
    if (resid_out && k == K - 1) {  // the residual of the last update
#pragma unroll
      for (int j = 0; j < M; ++j) resid_out[d * M + j] = r[j];
    }
    // theta += L r' (then project_theta), P -= (w / s) w' -- in place (run-time row loops: the step's physics and inner loop
    // share the registers)
#pragma unroll kRlsRowUnroll
    for (int i = 0; i < MN; ++i) {
      const Real wi = s_w[i * T];
      const Real Li = c.normalize_gain ? wi * inv_s : wi;
      const unsigned word = PROJECT ? s_code[i] : 0x55555555u;
#pragma unroll
      for (int j = 0; j < M; ++j) {
        const Real val = sT[(i * M + j) * T] + Li * r[j];
        if (!PROJECT) sT[(i * M + j) * T] = val;
        else {
          const unsigned code = (word >> (2 * j)) & 3u;
          sT[(i * M + j) * T] = code == 1u ? val : (code == 0u ? Real(0) : Real(1));
        }
      }
    }
#pragma unroll 2
    for (int i = 0; i < MN; ++i) {
      const Real Li = s_w[i * T] * inv_s;
      const int row0 = i * MN - i * (i - 1) / 2 - i;  // rls_tri(i, j) = row0 + j
#pragma unroll
      for (int j = 0; j < MN; ++j)
        if (j >= i) sP[(row0 + j) * T] -= Li * v[j];
    }
  }
  if (!g.valid) return;
  // ---- write back: state, observation, PID state; theta and both triangles of P (the planes keep the full square)
  store_drone(st, g.d, s);
  store_obs(obs, g.d, o);
  store_pid(pid, g.d, ps);
#pragma unroll 1
  for (int k = 0; k < MN * M; ++k) theta[(size_t)k * D + d] = sT[k * T];
#pragma unroll 1
  for (int i = 0; i < MN; ++i)
#pragma unroll 1
    for (int j = i; j < MN; ++j) {
      const Real pij = sP[rls_tri<MN>(i, j) * T];
      Pm[(size_t)(i * MN + j) * D + d] = pij;
      if (j > i) Pm[(size_t)(j * MN + i) * D + d] = pij;
    }
}
