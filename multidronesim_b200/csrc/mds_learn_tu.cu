// mds_learn_tu.cu -- the fused learning rollout's kernels (mds_learn.cuh) and their launcher, in a translation unit of their
// own: <Real in {float, double}, M in {9, 10}, PROJECT (M = 10 only), FEEDBACK>, twelve kernels.  mds_kernels.cu (the C ABI)
// calls the launcher.  The 12-dim kernels are in mds_learn_torque_tu.cu.
#include "mds_learn.cuh"

template <typename Real> cudaError_t launch_learn_kernel(const LearnLaunch<Real>& a) {
  if (a.m == 9) return launch_learn<Real, 9, false>(a);
  return a.project ? launch_learn<Real, 10, true>(a) : launch_learn<Real, 10, false>(a);
}

template cudaError_t launch_learn_kernel<float>(const LearnLaunch<float>& a);
template cudaError_t launch_learn_kernel<double>(const LearnLaunch<double>& a);
