// mds_rollout_tu.cu -- one translation unit per (precision, kernel kind) of the rollout kernels:
//   nvcc -DMDS_TU_REAL=float|double -DMDS_TU_KIND=0 (rollout_loop_kernel) | 1 (ctrl_step_kernel)
// Each defines the matching launcher of mds_rollout_launch.cuh; mds_kernels.cu (the C ABI) calls them.
#include "mds_rollout_launch.cuh"

#ifndef MDS_TU_REAL
#error "compile with -DMDS_TU_REAL=float or double"
#endif
#if !defined(MDS_TU_KIND) || (MDS_TU_KIND != 0 && MDS_TU_KIND != 1)
#error "compile with -DMDS_TU_KIND=0 or 1"
#endif
using Real = MDS_TU_REAL;

// controller / filter dispatch shared by the two launchers: calls F.template run<CTRL, USE_CBF, PDKC>()
template <typename F> static void dispatch_ctrl(int ctrl, int use_cbf, F&& f) {
  switch (ctrl) {
    case MDS_CTRL_GEOMETRIC: f.template run<MDS_CTRL_GEOMETRIC, false, false>(); break;
    case MDS_CTRL_LQR_TORQUE: f.template run<MDS_CTRL_LQR_TORQUE, false, true>(); break;
    case MDS_CTRL_DSLPID: f.template run<MDS_CTRL_DSLPID, false, false>(); break;
    case MDS_CTRL_LQR_OMEGA:
      if (use_cbf) f.template run<MDS_CTRL_LQR_OMEGA, true, true>();
      else f.template run<MDS_CTRL_LQR_OMEGA, false, true>();
      break;
    default:
      if (use_cbf) f.template run<MDS_CTRL_LQR_YANK, true, true>();
      else f.template run<MDS_CTRL_LQR_YANK, false, true>();
      break;
  }
}

#if MDS_TU_KIND == 0
struct LoopLauncher {
  const RolloutLaunch<Real>& a;
  double t0, dt_ctrl;
  int K;
  cudaError_t err;
  template <int CT, bool CB, bool PDKC> void run() {
    const bool pdk = a.R.lqr_planes != nullptr;  // per-drone gains: the run-time-N instantiation compiled with PDK (NT = -1)
    auto kern = pdk ? rollout_loop_kernel<Real, CT, CB, (PDKC ? -1 : 0), 0>
                    : (a.spec == 1 ? ((a.N == 8) ? rollout_loop_kernel<Real, CT, CB, 8, 1> : rollout_loop_kernel<Real, CT, CB, 0, 1>)
                                   : ((a.N == 8) ? rollout_loop_kernel<Real, CT, CB, 8, 0> : rollout_loop_kernel<Real, CT, CB, 0, 0>));
    // every environment flies the same 8 references: the instantiation that evaluates them once per block into a table
    if constexpr (sizeof(Real) == 4 && (CT == MDS_CTRL_LQR_OMEGA || CT == MDS_CTRL_LQR_YANK)) {
      if (!pdk && a.N == 8 && a.traj_period == 8)
        kern = a.spec == 1 ? rollout_loop_kernel<Real, CT, CB, 8, 1, true> : rollout_loop_kernel<Real, CT, CB, 8, 0, true>;
    }
    err = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)a.smem);
    kern<<<a.blocks, a.threads, a.smem, a.cs>>>(a.Pd, a.R, a.G, a.L, a.C, a.Dg, a.Ds, a.Sd, a.Pi, a.specs, a.segs, a.action, a.fext, a.obs, a.obs_log,
                                                 a.stats, t0, dt_ctrl, K, a.E, a.N, a.NP);
  }
};
template <> cudaError_t launch_loop_kernel<Real>(const RolloutLaunch<Real>& a, double t0, double dt_ctrl, int K) {
  LoopLauncher l{a, t0, dt_ctrl, K, cudaSuccess};
  dispatch_ctrl(a.R.ctrl, a.R.use_cbf, l);
  return l.err;
}
#else
struct CtrlLauncher {
  const RolloutLaunch<Real>& a;
  double t;
  const Real* obs_in;
  bool set_attr;
  cudaError_t err;
  template <int CT, bool CB, bool PDKC> void run() {
    const bool pdk = a.R.lqr_planes != nullptr;
    auto kern = pdk ? ctrl_step_kernel<Real, CT, CB, (PDKC ? -1 : 0)>
                    : ((a.N == 8) ? ctrl_step_kernel<Real, CT, CB, 8> : ctrl_step_kernel<Real, CT, CB, 0>);
    if (set_attr) err = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)a.smem);
    // persistent grid: the resident set (the kernel walks the tiles); small swarms keep one block per tile
    int grid = a.blocks;
#if MDS_CTRL_PERSISTENT
    static int resident_blocks = 0;  // per process: every device of a box is the same part
    if (resident_blocks == 0) {
      int dev = 0, sms = 0;
      cudaGetDevice(&dev);
      cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
      resident_blocks = 2 * (sms > 0 ? sms : 148);
    }
    if (grid > resident_blocks) grid = resident_blocks;
#endif
    kern<<<grid, a.threads, a.smem, a.cs>>>(a.Pd, a.R, a.G, a.L, a.C, a.Dg, a.Ds, a.Pi, a.specs, a.segs, obs_in, a.action, a.stats, t, a.E, a.N, a.NP);
  }
};
template <> cudaError_t launch_ctrl_kernel<Real>(const RolloutLaunch<Real>& a, double t, const Real* obs_in, bool set_attr) {
  CtrlLauncher l{a, t, obs_in, set_attr, cudaSuccess};
  dispatch_ctrl(a.R.ctrl, a.R.use_cbf, l);
  return l.err;
}
#endif
