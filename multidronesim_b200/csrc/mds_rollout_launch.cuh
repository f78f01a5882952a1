// mds_rollout_launch.cuh -- host-side launchers of the two heavy rollout kernels.  Declared here, defined in
// mds_rollout_tu.cu, which the Makefile compiles once per (precision, kernel kind): the ~110 instantiations build in
// parallel instead of inside one translation unit.
#pragma once
#include <cuda_runtime.h>
#include "mds_rollout.cuh"

template <typename Real> struct RolloutLaunch {
  DroneP<Real> Pd;
  RolloutP<Real> R;
  GeoP<Real> G;
  LqrP<Real> L;
  CbfP<Real> C;
  DslP<Real> Dg;
  DslStateP<Real> Ds;
  StateP<Real> Sd;
  PidP<Real> Pi;
  const typename TrajSpecT<Real>::spec* specs;
  const typename TrajSpecT<Real>::seg* segs;
  Real* action;
  const Real* fext;
  Real* obs;
  Real* obs_log;
  double* stats;
  int E, N, NP, blocks, threads;
  int spec;  // PhysSpec instantiation the parameter block qualifies for (0 = none: run-time switches)
  size_t smem;
  cudaStream_t cs;
  int traj_period;  // MdsRolloutCfg.traj_period: 0, or N when every environment flies the references of environment 0
};

// Each returns the error of the shared-memory opt-in (cudaSuccess when it was not needed); launch errors are
// picked up by the caller's cudaGetLastError().
template <typename Real> cudaError_t launch_loop_kernel(const RolloutLaunch<Real>& a, double t0, double dt_ctrl, int K);
template <typename Real> cudaError_t launch_ctrl_kernel(const RolloutLaunch<Real>& a, double t, const Real* obs_in, bool set_attr);
