// mds_care_launch.cuh -- host-side launcher of the batched Riccati solve (mds_care_tu.cu, a translation unit of its own):
// mds_kernels.cu (the C ABI) validates the arguments and calls it.
#pragma once
#include <cuda_runtime.h>

namespace mds {

struct CareP {
  double sq[12];          // sqrt(q_kk) of a drone's diagonal Q (the first m entries)
  double rinv[4];         // 1 / r_ii
  double cross[12 * 12];  // robot-coupled only, the pair's scaled cross block: Q[k][12 + l] / (sq_k sq_l), robot 0's state k
                          // against robot 1's state l
};

}  // namespace mds

// coupled = false: one m x m problem per drone of the E x N drones, K planes [4m][E N] (the per-drone solve passes E = D,
// N = 1).  coupled = true (m = 12): one launch for the pair problems (drones 0 and 1 of every environment), one for the single
// problems of drones 2 .. N-1 (N > 2), K planes [N][48][E N].  Returns the error of a shared-memory opt-in (cudaSuccess
// otherwise); launch errors are picked up by the caller's cudaGetLastError().
template <typename Real>
cudaError_t launch_care(const mds::CareP& c, int m, bool coupled, const Real* theta, Real* K, int* status, int E, int N, cudaStream_t cs);
