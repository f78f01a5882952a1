// mds_learn_launch.cuh -- host-side launchers of the fused learning rollout (mds_learn.cuh).  Declared here, defined in
// mds_learn_tu.cu (m = 9, 10) and mds_learn_torque_tu.cu (m = 12), translation units of their own: mds_kernels.cu (the C
// ABI) validates the arguments and calls them.
#pragma once
#include <cuda_runtime.h>
#include "mds_common.cuh"
#include "mds_ctrl.cuh"
#include "mds_sysid.cuh"
#include "mds_traj.cuh"

using namespace mds;

template <typename Real> struct LearnLaunch {
  DroneP<Real> Pd;
  RlsP c;
  int m, project;  // model dimension (9: LQR_OMEGA, 10: LQR_YANK, 12: LQR_TORQUE); whether project_theta is applied at all
  int learn_from, write_obs_every;
  StateP<Real> Sd;
  PidP<Real> Pi;
  const typename TrajSpecT<Real>::spec* specs;
  const typename TrajSpecT<Real>::seg* segs;
  const Real* inputs;  // [K][D*4]
  const Real* gain;    // [4*m][D] gain planes of the closed-loop law; NULL: inputs are the inner loop's inputs (open loop)
  int coupled;         // m = 12 with a gain: gain holds the robot-coupled [N][4*m][D] planes
  Real *theta, *Pm, *resid, *obs;
  const Real* fext;
  Real* obs_log;
  double t0, dt_ctrl;
  int K, E, N;
  cudaStream_t cs;
};

// Returns the error of the shared-memory opt-in (cudaSuccess otherwise); launch errors are picked up by the caller's
// cudaGetLastError().
template <typename Real> cudaError_t launch_learn_kernel(const LearnLaunch<Real>& a);
template <typename Real> cudaError_t launch_learn_torque_kernel(const LearnLaunch<Real>& a);
