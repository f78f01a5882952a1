// mds_learn_tu.cu -- the fused learning rollout's kernels (mds_learn.cuh) and their launcher, in a translation unit of their
// own: <Real in {float, double}, M in {9, 10}, PROJECT (M = 10 only)>, six kernels.  mds_kernels.cu (the C ABI) calls the launcher.
#include "mds_learn.cuh"

template <typename Real> cudaError_t launch_learn_kernel(const LearnLaunch<Real>& a) {
  const int NP = next_pow2(a.N);
  auto go = [&](auto kern, int threads, size_t smem) -> cudaError_t {
    // N = 32 in fp64 stages 50-72 KB per block: past the default 48 KB of dynamic shared memory
    const cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
    const int epb = threads / NP, blocks = (a.E + epb - 1) / epb;
    kern<<<blocks, threads, smem, a.cs>>>(a.Pd, a.c, a.Sd, a.Pi, a.specs, a.segs, a.inputs, a.theta, a.Pm, a.resid, a.obs, a.fext, a.obs_log, a.t0,
                                          a.dt_ctrl, a.learn_from, a.write_obs_every, a.K, a.E, a.N, NP);
    return cudaSuccess;
  };
  if (a.m == 9) {
    const int threads = learn_threads<Real, 9>(NP);
    return go(learn_rollout_kernel<Real, 9, false>, threads, (size_t)rls_words_per_thread<Real, 9>() * threads * sizeof(Real));
  }
  const int threads = learn_threads<Real, 10>(NP);
  const size_t smem = (size_t)rls_words_per_thread<Real, 10>() * threads * sizeof(Real);
  return a.project ? go(learn_rollout_kernel<Real, 10, true>, threads, smem) : go(learn_rollout_kernel<Real, 10, false>, threads, smem);
}

template cudaError_t launch_learn_kernel<float>(const LearnLaunch<float>& a);
template cudaError_t launch_learn_kernel<double>(const LearnLaunch<double>& a);
