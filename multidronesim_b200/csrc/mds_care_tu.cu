// mds_care_tu.cu -- the batched continuous-time Riccati solve of the decentralised LQR, both kinds, and its launcher: one m x m
// problem per drone (mds_care_gains), and the 12-dim case whose Q couples robots 0 and 1 of every environment
// (mds_care_gains_coupled).
//
// compute_controller (decentralized_lqr_omega.py:185-204): K_d = R^-1 B_d' X_d with X_d the stabilising solution of
// A'X + XA - X B R^-1 B' X + Q = 0 for every drone's learned (A_d, B_d) = theta_d.  The reference calls scipy
// (solve_continuous_are: QZ on the balanced extended pencil) once per learning phase on the host; a swarm of distinct
// learned models needs one solve per drone, so here ONE WARP solves one problem in shared memory, in double:
//   * state scaling z = sqrt(Q) x (Q diagonal) -> Q~ = I, which equalises the Hamiltonian's blocks (the reference's
//     Bryson weights span 1e-6 .. 1e6);
//   * matrix sign function of H = [[A~, -G~], [-Q~, -A~']] by the determinant-scaled Newton iteration
//     Z <- (c Z + (c Z)^-1) / 2, c = |det Z|^(-1/2n), each inverse a Gauss-Jordan sweep with partial pivoting over
//     [Z | I]; 7-9 iterations to 1e-13;
//   * X~ from W12 X~ = -(W11 + I) (W = sign H), symmetrised, scaled back, then K = R^-1 B' X.
// Agreement with scipy on the reference's three parametrisations with perturbed / dense learned models: <= 2e-12 of max |K|.
//
// Robot-coupled Q (decentralized_lqr.py:44-53: a cross block between the xy positions of robots 0 and 1): A, B and R are block
// diagonal per drone and Q is kron(I_N, Q_d) apart from that cross block, so the block-diagonal X with blocks {0, 1}, {2}, ...,
// {N-1} satisfies the environment's Riccati equation block by block; its closed loop is block diagonal and Hurwitz, so it is
// THE stabilising solution.  The 12N-state problem of an environment splits into one 24-state pair problem (drones 0 and 1,
// Q~ = I plus the scaled cross block) and N - 2 independent 12-state problems; the gain is zero outside the blocks
// {0, 1} x {0, 1} and {j} x {j}.  Results go straight to the robot-coupled [N][48][D] planes that mds_dlqr_ctrl (coupled = 1)
// and the fused learning rollout read; a solved drone's entries for sources outside its problem are written as exact zeros.
// The per-drone planes [4m][D] are that layout with a single source block (N = 1).
#include "mds_care_launch.cuh"
#include "mds_common.cuh"

namespace mds {

// S drones per problem: 1 (single) or 2 (pair).  One warp per problem; lane l owns the Hamiltonian rows l + 32 t (the 48 rows
// of the pair problem do not fit lane = row).  Shared memory per problem: Z [2n][2n], [Z | I] [2n][4n + 1] and B~ [n][4]
// doubles, n = M S: 14 400 B at M = 12 (single; four problems per block) / 56 448 B (pair; one per block).
template <int S> constexpr int care_warps() { return S == 1 ? 4 : 1; }
template <int M, int S> constexpr int care_doubles() { return (2 * M * S) * (2 * M * S) + (2 * M * S) * (4 * M * S + 1) + M * S * 4; }

// Gauss-Jordan elimination with partial pivoting of the leading rows x rows block of a (row stride ld) to the identity, lane l
// owning rows l + 32 t (t < R).  Columns left of the pivot are already zero in the rows that take part, so every sweep starts
// at the pivot column.  Returns false on a vanishing pivot; *logdet += sum log |pivot|.
template <int R> MDS_DEV bool warp_gauss_jordan(double* a, int rows, int cols, int ld, int lane, double* logdet) {
  const unsigned full = 0xffffffffu;
  for (int k = 0; k < rows; ++k) {
    double best = -1.0;
    int who = lane;
#pragma unroll
    for (int t = 0; t < R; ++t) {
      const int row = lane + 32 * t;
      if (row >= k && row < rows) {
        const double v = fabs(a[row * ld + k]);
        if (v > best) { best = v; who = row; }
      }
    }
    for (int off = 16; off > 0; off >>= 1) {
      const double ob = __shfl_xor_sync(full, best, off);
      const int ow = __shfl_xor_sync(full, who, off);
      if (ob > best || (ob == best && ow < who)) { best = ob; who = ow; }
    }
    if (!(best > 1e-300)) return false;
    *logdet += log(best);
    if (who != k)
      for (int c = k + lane; c < cols; c += 32) { const double t = a[k * ld + c]; a[k * ld + c] = a[who * ld + c]; a[who * ld + c] = t; }
    __syncwarp(full);
    const double inv = 1.0 / a[k * ld + k];
    __syncwarp(full);
    for (int c = k + lane; c < cols; c += 32) a[k * ld + c] *= inv;
    __syncwarp(full);
#pragma unroll
    for (int t = 0; t < R; ++t) {
      const int row = lane + 32 * t;
      if (row < rows && row != k) {
        const double f = a[row * ld + k];
        for (int c = k; c < cols; ++c) a[row * ld + c] -= f * a[k * ld + c];
      }
    }
    __syncwarp(full);
  }
  return true;
}

// M states per drone.  Problem p: S == 2 -> environment p, drones 0 and 1; S == 1 -> environment p / (N - first), drone
// first + p % (N - first).  K is [N][4M][D], D = E N.
// Register budget 72 (single) / 68 (pair): shared memory bounds residency (at most six 128-thread blocks per SM, at M = 9),
// so neither costs occupancy.  Left to ptxas's own choice the M = 9, 10 kernels are held to 64 registers and the single
// problems lose the schedule of the elimination sweep that loads a row's next element before storing the current one
// (3 % slower at M = 12 on a B200); at 72 the fp64 pair kernel is 0.2 % slower than at 68.
template <typename Real, int M, int S>
__global__ void __maxnreg__(S == 1 ? 72 : 68) care_kernel(CareP c, const Real* __restrict__ theta, Real* __restrict__ K,
                                                          int* __restrict__ status, int E, int N, int first) {
  static_assert(S == 1 || M == 12, "the robot-coupled pair problem is the 12-dim model's");
  constexpr int n = M * S, N2 = 2 * n, LD = 2 * N2 + 1, R = (N2 + 31) / 32, W = care_warps<S>();
  extern __shared__ __align__(16) unsigned char care_smem[];
  __shared__ double s_sq[M], s_rinv[4], s_cross[S == 2 ? M * M : 1];
  if (threadIdx.x == 0) {
#pragma unroll
    for (int i = 0; i < M; ++i) s_sq[i] = c.sq[i];
#pragma unroll
    for (int i = 0; i < 4; ++i) s_rinv[i] = c.rinv[i];
    if (S == 2)
      for (int i = 0; i < M * M; ++i) s_cross[i] = c.cross[i];
  }
  __syncthreads();
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int per_env = S == 2 ? 1 : N - first;
  const size_t p = (size_t)blockIdx.x * W + warp;
  if (p >= (size_t)E * per_env) return;  // whole warps leave together
  const size_t e = p / per_env;
  const unsigned D = (unsigned)E * N;  // < 2^31 (the C ABI checks it); a 64-bit D costs the M = 9 kernels a spill
  const int n0 = S == 2 ? 0 : first + (int)(p % per_env);  // the problem's first drone in its environment
  const size_t d0 = e * N + n0;
  const unsigned full = 0xffffffffu;
  double* Z = reinterpret_cast<double*>(care_smem) + (size_t)warp * care_doubles<M, S>();
  double* Ag = Z + N2 * N2;
  double* Bs = Ag + N2 * LD;  // B~ [n][4] = sqrt(Q) B
  // theta[i][j] of the problem's drone a: A[j][i] for i < M, B[j][i-M] above
  auto th = [&](int a, int i, int j) { return (double)theta[(size_t)(i * M + j) * D + d0 + a]; };
  // state s of the problem: drone s / M within the problem (0 for S == 1), its state s % M
  auto drone = [](int s) { return S == 1 ? 0 : s / M; };
  for (int s = lane; s < n; s += 32) {
    const int a = drone(s), k = s - a * M;
    for (int i = 0; i < 4; ++i) Bs[s * 4 + i] = th(a, M + i, k) * s_sq[k];
  }
  __syncwarp(full);
#pragma unroll
  for (int t = 0; t < R; ++t) {
    const int row = lane + 32 * t;
    if (row < n) {  // rows [A~, -G~]: zero between the two drones of a pair
      const int a = drone(row), k = row - a * M;
      for (int cc = 0; cc < n; ++cc) {
        const int b = drone(cc), l = cc - b * M;
        double z = 0.0, g = 0.0;
        if (a == b) {
          z = th(a, l, k) * s_sq[k] / s_sq[l];
          for (int i = 0; i < 4; ++i) g += Bs[row * 4 + i] * s_rinv[i] * Bs[cc * 4 + i];
        }
        Z[row * N2 + cc] = z;
        Z[row * N2 + n + cc] = -g;
      }
    } else if (row < N2) {  // rows [-Q~, -A~']
      const int rr = row - n, a = drone(rr), k = rr - a * M;
      for (int cc = 0; cc < n; ++cc) {
        const int b = drone(cc), l = cc - b * M;
        double q = cc == rr ? 1.0 : 0.0;
        if (S == 2 && a != b) q = a == 0 ? s_cross[k * M + l] : s_cross[l * M + k];
        Z[row * N2 + cc] = -q;
        Z[row * N2 + n + cc] = a == b ? -th(a, k, l) * s_sq[l] / s_sq[k] : 0.0;
      }
    }
  }
  __syncwarp(full);
  bool ok = true;
  int it = 0;
  for (; it < 60; ++it) {
#pragma unroll
    for (int t = 0; t < R; ++t) {
      const int row = lane + 32 * t;
      if (row < N2)
        for (int cc = 0; cc < N2; ++cc) { Ag[row * LD + cc] = Z[row * N2 + cc]; Ag[row * LD + N2 + cc] = cc == row ? 1.0 : 0.0; }
    }
    __syncwarp(full);
    double logdet = 0.0;
    if (!warp_gauss_jordan<R>(Ag, N2, 2 * N2, LD, lane, &logdet)) { ok = false; break; }
    const double sc = exp(-logdet / (double)N2), isc = 1.0 / sc;
    double diff = 0.0, mx = 0.0;
#pragma unroll
    for (int t = 0; t < R; ++t) {
      const int row = lane + 32 * t;
      if (row < N2)
        for (int cc = 0; cc < N2; ++cc) {
          const double z = Z[row * N2 + cc], zn = 0.5 * (sc * z + isc * Ag[row * LD + N2 + cc]);
          diff = fmax(diff, fabs(zn - z)); mx = fmax(mx, fabs(zn));
          Z[row * N2 + cc] = zn;
        }
    }
    for (int off = 16; off > 0; off >>= 1) { diff = fmax(diff, __shfl_xor_sync(full, diff, off)); mx = fmax(mx, __shfl_xor_sync(full, mx, off)); }
    __syncwarp(full);
    if (diff <= 1e-13 * mx) break;
  }
  if (ok && it < 60) {  // W12 X~ = -(W11 + I): n <= 24 rows, lane = row
    constexpr int LD2 = 2 * n + 1;
    if (lane < n)
      for (int cc = 0; cc < n; ++cc) {
        Ag[lane * LD2 + cc] = Z[lane * N2 + n + cc];
        Ag[lane * LD2 + n + cc] = -(Z[lane * N2 + cc] + (cc == lane ? 1.0 : 0.0));
      }
    __syncwarp(full);
    double ld = 0.0;
    ok = warp_gauss_jordan<1>(Ag, n, 2 * n, LD2, lane, &ld);
    if (ok && lane < n) {  // column `lane` of the problem's K = R^-1 B' X, X[r][c] = sq_r (X~[r][c] + X~[c][r]) / 2 sq_c
      const int b = drone(lane), l = lane - b * M;
      for (int a = 0; a < S; ++a) {  // drone a's four rows, source drone b, its state l
        double kc[4] = {0.0, 0.0, 0.0, 0.0};
        for (int k = 0; k < M; ++k) {
          const int r = M * a + k;
          const double x = 0.5 * (Ag[r * LD2 + n + lane] + Ag[lane * LD2 + n + r]) * s_sq[l];  // times sq_r below, inside B~
          for (int i = 0; i < 4; ++i) kc[i] += Bs[r * 4 + i] * x;
        }
        for (int i = 0; i < 4; ++i) K[(size_t)((n0 + b) * 4 * M + i * M + l) * D + d0 + a] = (Real)(s_rinv[i] * kc[i]);
      }
    }
    if (ok)  // the entries of the other source drones: plane (j * 4M + i * M + k), j outside the problem
      for (int a = 0; a < S; ++a)
        for (int q = lane; q < N * 4 * M; q += 32)
          if (q < n0 * 4 * M || q >= (n0 + S) * 4 * M) K[(size_t)q * D + d0 + a] = Real(0);
  } else {
    ok = false;
  }
  if (lane == 0 && status)
    for (int a = 0; a < S; ++a) status[d0 + a] = ok ? 0 : 1;
}

template <typename Real, int M, int S>
static cudaError_t launch_care_problems(const CareP& c, const Real* theta, Real* K, int* status, int E, int N, int first, cudaStream_t cs) {
  constexpr int W = care_warps<S>();
  const size_t problems = (size_t)E * (S == 2 ? 1 : N - first);
  const size_t smem = (size_t)care_doubles<M, S>() * W * sizeof(double);
  const cudaError_t ae = cudaFuncSetAttribute(care_kernel<Real, M, S>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (ae != cudaSuccess) return ae;
  care_kernel<Real, M, S><<<(unsigned)((problems + W - 1) / W), 32 * W, smem, cs>>>(c, theta, K, status, E, N, first);
  return cudaSuccess;
}

}  // namespace mds

template <typename Real>
cudaError_t launch_care(const mds::CareP& c, int m, bool coupled, const Real* theta, Real* K, int* status, int E, int N, cudaStream_t cs) {
  using namespace mds;
  if (coupled) {
    cudaError_t e = launch_care_problems<Real, 12, 2>(c, theta, K, status, E, N, 0, cs);
    if (e == cudaSuccess && N > 2) e = launch_care_problems<Real, 12, 1>(c, theta, K, status, E, N, 2, cs);
    return e;
  }
  if (m == 9) return launch_care_problems<Real, 9, 1>(c, theta, K, status, E, N, 0, cs);
  if (m == 10) return launch_care_problems<Real, 10, 1>(c, theta, K, status, E, N, 0, cs);
  return launch_care_problems<Real, 12, 1>(c, theta, K, status, E, N, 0, cs);
}

template cudaError_t launch_care<float>(const mds::CareP&, int, bool, const float*, float*, int*, int, int, cudaStream_t);
template cudaError_t launch_care<double>(const mds::CareP&, int, bool, const double*, double*, int*, int, int, cudaStream_t);
