// mds_learn_tu.cu -- the fused learning rollout's kernels (mds_learn.cuh) and their launcher, in a translation unit of their
// own: <Real in {float, double}, M in {9, 10}, PROJECT (M = 10 only), FEEDBACK>, twelve kernels.  mds_kernels.cu (the C ABI)
// calls the launcher.
#include "mds_learn.cuh"

template <typename Real, int M, bool PROJECT, bool FEEDBACK> static cudaError_t launch_learn(const LearnLaunch<Real>& a) {
  const int NP = next_pow2(a.N), threads = learn_threads<Real, M>(NP);
  const size_t smem = (size_t)learn_words_per_thread<Real, M, FEEDBACK>() * threads * sizeof(Real);
  auto kern = learn_rollout_kernel<Real, M, PROJECT, FEEDBACK>;
  // N = 32 in fp64 stages 61-83 KB per block: past the default 48 KB of dynamic shared memory
  const cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (e != cudaSuccess) return e;
  const int epb = threads / NP, blocks = (a.E + epb - 1) / epb;
  kern<<<blocks, threads, smem, a.cs>>>(a.Pd, a.c, a.Sd, a.Pi, a.specs, a.segs, a.inputs, a.theta, a.Pm, a.resid, a.obs, a.fext, a.obs_log, a.t0,
                                        a.dt_ctrl, a.learn_from, a.write_obs_every, a.K, a.E, a.N, NP, a.gain);
  return cudaSuccess;
}
template <typename Real, int M, bool PROJECT> static cudaError_t launch_learn(const LearnLaunch<Real>& a) {
  return a.gain ? launch_learn<Real, M, PROJECT, true>(a) : launch_learn<Real, M, PROJECT, false>(a);
}

template <typename Real> cudaError_t launch_learn_kernel(const LearnLaunch<Real>& a) {
  if (a.m == 9) return launch_learn<Real, 9, false>(a);
  return a.project ? launch_learn<Real, 10, true>(a) : launch_learn<Real, 10, false>(a);
}

template cudaError_t launch_learn_kernel<float>(const LearnLaunch<float>& a);
template cudaError_t launch_learn_kernel<double>(const LearnLaunch<double>& a);
