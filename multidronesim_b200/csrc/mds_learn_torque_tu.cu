// mds_learn_torque_tu.cu -- the 12-dim torque-level instantiations of the fused learning rollout (mds_learn.cuh) and their
// launcher: <Real in {float, double}, M = 12, PROJECT, open loop / FEEDBACK / FEEDBACK + COUPLED>, six kernels.  A translation
// unit of their own: in mds_learn_tu.cu's object, the fp64 m = 9 / 10 kernels would be scheduled differently around the
// calls they share with them.
#include "mds_learn.cuh"

template <typename Real> cudaError_t launch_learn_torque_kernel(const LearnLaunch<Real>& a) {
  return a.gain && a.coupled ? launch_learn<Real, 12, true, true, true>(a) : launch_learn<Real, 12, true>(a);
}

template cudaError_t launch_learn_torque_kernel<float>(const LearnLaunch<float>& a);
template cudaError_t launch_learn_torque_kernel<double>(const LearnLaunch<double>& a);
