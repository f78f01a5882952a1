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
// FEEDBACK: closed-loop exploration -- every drone flies its own learned gain plus the caller's perturbation,
//   u = -K_d e_t (+ m g unless yank-omega; LQR_OMEGA: cap_thrust) + u[k],  phi = [e_t, u]
// which is the per-call loop with mds_dlqr_ctrl(skip_low_level) and an add before mds_lowlevel.  The gain [4*m][D] planes
// (mds_dlqr_ctrl's uncoupled layout) are read once per launch and staged next to theta and P: constant within the launch.
// M = 12: the torque-level model (decentralized_lqr.py), no inner loop and no PID state: the action is input_to_action(u),
// which clamps u[0] >= 0 in place, so phi carries the clamped u.  Its law is
//   u = max(-sum_j K_dj e_j + m g, 0 on the thrust) + u[k]
// with K_dj the drone's own gain (FEEDBACK) or, COUPLED, the robot-coupled gain [N][48][D] planes of mds_dlqr_ctrl.  The
// coupled gain is not staged (N * 48 words per thread would not fit beside theta and P at N = 32 in fp64): it is read from
// HBM every step, as dlqr_ctrl_kernel does.  The partners' error states come through shared memory: each lane publishes
// e_t in its s_phi column (where the RLS step puts phi[:12] = e_t anyway), the lane group syncs, sums over its N sources and
// syncs again before any lane writes s_phi -- in every physics mode, DYN included, whose physics step has no group sync.
#pragma once
#include <cuda_runtime.h>
#include "mds_learn_launch.cuh"
#include "mds_rollout.cuh"

// Threads per block: the RLS kernel's (one warp in fp32, half a warp in fp64; the staged columns set the occupancy),
// raised to the lane-group size NP where that is larger.  Both are at most 32.
template <typename Real, int M> static int learn_threads(int NP) { return rls_threads<Real, M>() > NP ? rls_threads<Real, M>() : NP; }
// Staged words per thread: the RLS kernel's columns, plus the 4*M gain entries when FEEDBACK
template <typename Real, int M, bool FEEDBACK> constexpr int learn_words_per_thread() { return rls_words_per_thread<Real, M>() + (FEEDBACK ? 4 * M : 0); }
// COUPLED stages no gain
template <typename Real, int M, bool FEEDBACK, bool COUPLED> constexpr int learn_words_per_thread() { return learn_words_per_thread<Real, M, FEEDBACK && !COUPLED>(); }

// M = 9: DecentralizedLQROmega (LQR_OMEGA error state, ThrustOmega inner loop); M = 10: the yank-omega variants (LQR_YANK,
// YankOmega inner loop); M = 12: DecentralizedLQR (LQR_TORQUE error state, input_to_action, pid unused; PROJECT only).
// PROJECT: project_theta is applied (approx_theta_update(project=True)), compile-time like the RLS kernel.
// FEEDBACK: inputs are perturbations of the law u = -K_d e_t (gain: [4*M][D] planes; the last parameter, so that the open-loop
// kernels keep their parameter layout); otherwise inputs are the inner loop's inputs and gain is unused.
// COUPLED (M = 12, with FEEDBACK): gain holds the robot-coupled [N][4*M][D] planes, read from HBM every step.
template <typename Real, int M, bool PROJECT, bool FEEDBACK, bool COUPLED>
__global__ void __launch_bounds__(32) learn_rollout_kernel(DroneP<Real> P, RlsP c, StateP<Real> st, PidP<Real> pid,
                                                           const typename TrajSpecT<Real>::spec* __restrict__ specs,
                                                           const typename TrajSpecT<Real>::seg* __restrict__ segs,
                                                           const Real* __restrict__ inputs, Real* __restrict__ theta, Real* __restrict__ Pm,
                                                           Real* __restrict__ resid_out, Real* __restrict__ obs, const Real* __restrict__ fext,
                                                           Real* __restrict__ obs_log, double t0, double dt_ctrl, int learn_from, int write_obs_every,
                                                           int K, int E, int N, int NP, const Real* __restrict__ gain) {
  constexpr int MN = M + 4, TRI = MN * (MN + 1) / 2;
  constexpr int CTRL = M == 9 ? MDS_CTRL_LQR_OMEGA : (M == 10 ? MDS_CTRL_LQR_YANK : MDS_CTRL_LQR_TORQUE);
  static_assert(M != 12 || PROJECT, "both 12-dim reference methods project theta");
  static_assert(!COUPLED || (M == 12 && FEEDBACK), "the robot-coupled law is the 12-dim model's");
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
  Real* sK = s_term + M * T;  // FEEDBACK, not COUPLED: gain entry (i, k) of u_i = -sum_k K_ik e_k at sK[(i * M + k) * T]
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
    if (FEEDBACK && !COUPLED) {
#pragma unroll 1
      for (int k = 0; k < 4 * M; ++k) cp_async_real(sK + k * T, gain + (size_t)k * D + d);
    }
    s = load_drone(st, g.d);
    if constexpr (M != 12) ps = load_pid(pid, g.d);
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
      if (FEEDBACK && !COUPLED) {  // dlqr_ctrl_kernel's law and order of operations (skip_low_level: capped, no max(u, 0)), then + u[k]
        Real uf[4] = {Real(0), Real(0), Real(0), Real(0)};
#pragma unroll
        for (int i = 0; i < 4; ++i)
#pragma unroll
          for (int j = 0; j < M; ++j) uf[i] -= sK[(i * M + j) * T] * e0[j];
        if (CTRL != MDS_CTRL_LQR_YANK) uf[0] += P.m * P.g;
        if (CTRL == MDS_CTRL_LQR_OMEGA) uf[0] = cap_thrust(P, uf[0]);
        if (CTRL == MDS_CTRL_LQR_TORQUE) uf[0] = max_(uf[0], Real(0));  // dlqr_ctrl_kernel's input_to_action clamp
#pragma unroll
        for (int i = 0; i < 4; ++i) u[i] = uf[i] + u[i];
      }
      if constexpr (M == 12) {
        if (!COUPLED) input_to_action(P, u, rpm);  // clamps u[0] >= 0 in place: phi carries the clamped u
      } else {
        low_level(P, CTRL, ps, u, o, rpm);
      }
    }
    if constexpr (COUPLED) {  // u = -sum_j K_dj e_j over the env's N drones: publish e_t, sync, sum, sync (s_phi is reused below)
      if (g.valid) {
#pragma unroll
        for (int i = 0; i < M; ++i) s_phi[i * T] = e0[i];
      }
      __syncwarp(g.gmask);
      if (g.valid) {
        Real uf[4] = {Real(0), Real(0), Real(0), Real(0)};
        for (int j = 0; j < N; ++j) {  // dlqr_ctrl_kernel's order: source j, then row i, then column k
          const Real* ej = s_phi + (j - g.n);
          const Real* Kj = gain + (size_t)j * 4 * M * D + d;
#pragma unroll
          for (int i = 0; i < 4; ++i)
#pragma unroll
            for (int k = 0; k < M; ++k) uf[i] -= Kj[(size_t)(i * M + k) * D] * ej[k * T];
        }
        uf[0] = max_(uf[0] + P.m * P.g, Real(0));
#pragma unroll
        for (int i = 0; i < 4; ++i) u[i] = uf[i] + u[i];
        input_to_action(P, u, rpm);
      }
      __syncwarp(g.gmask);  // every lane of the group has read its partners' e_t
    }
    o = physics_core<0>(P, s, rpm, fx, sm_pos + (tid - g.n), g, N, NP);
    if (write_obs_every > 0 && --log_countdown == 0) {
      if (g.valid) store_obs(log_slot, g.d, o, true);  // streaming stores: the log is write-once
      log_slot += obs_elems;
      log_countdown = write_obs_every;
    }
    if (!g.valid || k < learn_from) continue;
    // ---- one RLS step in the staged columns (the sweeps of mds_sysid.cuh): phi = [e_t, u], x1 = e_t+1 against the same
    // reference sample
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
  if constexpr (M != 12) store_pid(pid, g.d, ps);
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

// Shared-memory opt-in and launch of one instantiation (mds_learn_tu.cu, mds_learn_torque_tu.cu)
template <typename Real, int M, bool PROJECT, bool FEEDBACK, bool COUPLED> static cudaError_t launch_learn(const LearnLaunch<Real>& a) {
  const int NP = next_pow2(a.N), threads = learn_threads<Real, M>(NP);
  const size_t smem = (size_t)learn_words_per_thread<Real, M, FEEDBACK, COUPLED>() * threads * sizeof(Real);
  auto kern = learn_rollout_kernel<Real, M, PROJECT, FEEDBACK, COUPLED>;
  // N = 32 in fp64 stages 61-105 KB per block: past the default 48 KB of dynamic shared memory (so does m = 12 feedback in fp32)
  const cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (e != cudaSuccess) return e;
  const int epb = threads / NP, blocks = (a.E + epb - 1) / epb;
  kern<<<blocks, threads, smem, a.cs>>>(a.Pd, a.c, a.Sd, a.Pi, a.specs, a.segs, a.inputs, a.theta, a.Pm, a.resid, a.obs, a.fext, a.obs_log, a.t0,
                                        a.dt_ctrl, a.learn_from, a.write_obs_every, a.K, a.E, a.N, NP, a.gain);
  return cudaSuccess;
}
template <typename Real, int M, bool PROJECT> static cudaError_t launch_learn(const LearnLaunch<Real>& a) {
  return a.gain ? launch_learn<Real, M, PROJECT, true, false>(a) : launch_learn<Real, M, PROJECT, false, false>(a);
}
