// mds_sysid.cuh -- per-drone recursive-least-squares model learning and the per-drone-gain LQR law of the
// reference's decentralised LQR (SURVEY.md 8(f)3):
//   control/dlqr/decentralized_lqr_omega.py:125-139 (theta_update), :110-123 (theta_update2), :212-231 (compute)
//   control/dlqr/decentralized_lqr_yank_omega.py:112-126
//   control/dlqr/decentralized_lqr.py:132-183 (theta_update2 / theta_update), :185-240 (est_x_dot, approx_theta_update,
//   project_theta), control/dlqr/decentralized_yolqr_crazyflie.py:228-290 (same for the 10-dim yank model)
// One thread per drone.  theta [(m+4) x m] and P [(m+4) x (m+4)] live in HBM as planes of D Reals (element k of drone d at
// [k * D + d]): every access of a warp is one coalesced line.  Each thread stages its own columns in shared memory
// (cp.async), so HBM sees each matrix once in and once out although the algorithm sweeps them twice.
#pragma once
#include "mds_common.cuh"

namespace mds {

struct RlsP {
  int target;             // MDS_RLS_TARGET_PREDICT / MDS_RLS_TARGET_XDOT
  int predict_from_xtp1;  // PREDICT: integrate from x_{t+1} (omega / yank-omega quirk) instead of phi[:m]
  int normalize_gain;     // 1: L = P phi / (1 + phi' P phi) (RLS); 0: L = P phi (information form, P holds V^-1)
  int project;            // MDS_RLS_PROJECT_*
  int drones_per_env;
  double dt;
  unsigned row_code[16];  // project_theta: 2 bits per entry of theta row i (bits 2j, 2j+1 for column j): 0 -> zero, 1 -> keep, 2 -> one
};

// 4- / 8-byte asynchronous global -> shared copy (LDGSTS): the whole theta / P column of a thread is in flight at once
// without passing through registers.
template <typename Real> MDS_DEV void cp_async_real(Real* smem_dst, const Real* gmem_src) {
  const unsigned dst = (unsigned)__cvta_generic_to_shared(smem_dst);
  if (sizeof(Real) == 4) asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"(dst), "l"(gmem_src) : "memory");
  else asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"(dst), "l"(gmem_src) : "memory");
}
MDS_DEV void cp_async_wait_all() { asm volatile("cp.async.commit_group;\ncp.async.wait_group 0;" ::: "memory"); }

// P is symmetric (identity-scaled prior, rank-one updates), so only its upper triangle is read and staged
template <typename Real, int M> constexpr int rls_words_per_thread() { return (M + 4) * (M + 5) / 2 + (M + 4) * M + 2 * (M + 4) + M; }
// index of entry (i, j), i <= j, in the row-major packed upper triangle of an MN x MN matrix
template <int MN> MDS_DEV constexpr int rls_tri(int i, int j) { return i * MN - i * (i - 1) / 2 + (j - i); }
// Threads per block: ONE warp (f32) / half a warp (f64).  A staged block is 40-63 KB, so 3-5 blocks share an SM and their
// load / compute / store phases overlap; measured at 1 M drones, m = 9 f32: 0.61 ms at 32 threads, 0.80 ms at 64 or 128.
// Row loops over the staged columns: unrolled by 4 so that several rows' shared-memory loads are in flight (registers are
// free here: occupancy is set by the staging footprint, not by registers).
constexpr int kRlsRowUnroll = 4;  // (#pragma unroll takes a constant expression, not a macro)
template <typename Real, int M> constexpr int rls_threads() { return sizeof(Real) == 4 ? 32 : 16; }

// ---- the sweeps of one RLS step over a thread's staged columns, shared by rls_update_kernel and learn_rollout_kernel
// (mds_learn.cuh).  Shared memory is [entry][thread] with thread stride T (a constant in rls_update_kernel, the block size
// in learn_rollout_kernel); sP is the packed upper triangle of P, sT theta, s_phi / s_w / s_term scratch columns (MN, MN,
// M entries), all already offset to the calling thread.

// project_theta before the update (MDS_RLS_PROJECT_LOOP, robots after the first of an env): s_code holds the codes per theta row
template <typename Real, int M> MDS_DEV void rls_pre_project(Real* sT, const unsigned* s_code, int T) {
  constexpr int MN = M + 4;
#pragma unroll 1
  for (int i = 0; i < MN; ++i) {
    const unsigned word = s_code[i];
#pragma unroll
    for (int j = 0; j < M; ++j) {
      const unsigned code = (word >> (2 * j)) & 3u;
      if (code != 1u) sT[(i * M + j) * T] = code == 0u ? Real(0) : Real(1);
    }
  }
}

// gain: w = P phi (= v'), s = 1 + phi' P phi; returns s.  v[] must be zero on entry and holds w on return (also in s_w).
// Row i of the triangle holds P(i, j >= i): it contributes P(i,j) phi_j to w_i and, for j > i, P(i,j) phi_i to w_j.  The
// fp64 RLS kernel's run-time row loop, used by learn_rollout_kernel in both precisions (the fully unrolled fp32 form takes
// 255 registers on its own): the row's own part of w_i goes to shared memory, the transposed contributions to v[j] with
// static j; the two halves are joined afterwards.
template <typename Real, int MN>
MDS_DEV Real rls_gain(const Real* sP, const Real* s_phi, Real* s_w, const Real (&phi)[MN], Real (&v)[MN], int T) {
  Real s = Real(1);
#pragma unroll 2
  for (int i = 0; i < MN; ++i) {
    const Real phi_i = s_phi[i * T];
    Real wi = Real(0);
    const int row0 = i * MN - i * (i - 1) / 2 - i;  // rls_tri(i, j) = row0 + j
#pragma unroll
    for (int j = 0; j < MN; ++j) {
      if (j >= i) {
        const Real p = sP[(row0 + j) * T];
        wi += p * phi[j];
        if (j > i) v[j] += p * phi_i;
      }
    }
    s_w[i * T] = wi;
  }
#pragma unroll
  for (int i = 0; i < MN; ++i) v[i] += s_w[i * T];
#pragma unroll
  for (int i = 0; i < MN; ++i) { s_w[i * T] = v[i]; s += phi[i] * v[i]; }
  return s;
}

// regression residual r (m) of the staged theta: est_x_dot - theta' phi (XDOT) or x1 - forward_predict (PREDICT)
template <typename Real, int M>
MDS_DEV void rls_residual(const RlsP& c, const Real (&phi)[M + 4], const Real (&x1)[M], const Real* s_phi, const Real* sT, Real* s_term,
                          Real (&r)[M], int T) {
  constexpr int MN = M + 4;
  if (c.target == MDS_RLS_TARGET_XDOT) {
    // est_x_dot, then x_dot - theta' phi
    const Real inv_dt = Real(1.0 / c.dt);
    if (M == 12) {  // decentralized_lqr.py:185-198
#pragma unroll
      for (int k = 0; k < 3; ++k) {
        r[k] = x1[3 + k];
        r[3 + k] = (x1[3 + k] - phi[3 + k]) * inv_dt;
        r[6 + k] = (x1[6 + k] - phi[6 + k]) * inv_dt;
        r[9 + k] = x1[6 + k];
      }
    } else {  // decentralized_yolqr_crazyflie.py:228-243 (m = 10; m = 9 is rejected on the host)
#pragma unroll
      for (int k = 0; k < 3; ++k) {
        r[k] = phi[M + 1 + k];
        r[4 + k] = (x1[4 + k] - phi[4 + k]) * inv_dt;
        r[7 + k] = x1[4 + k];
      }
      r[3] = phi[M];
    }
#pragma unroll kRlsRowUnroll
    for (int i = 0; i < MN; ++i) {
      const Real phi_i = s_phi[i * T];
#pragma unroll
      for (int j = 0; j < M; ++j) r[j] -= sT[(i * M + j) * T] * phi_i;
    }
  } else {
    // forward_predict: e' = Ahat e + Bhat u over dt from e0, Ahat = theta[:m]^T, Bhat = theta[m:]^T.  The reference runs
    // scipy RK45 (its error over one 1/240 s step is far below its 1e-3 tolerance); here the exact solution
    // e(dt) = e0 + sum_{k>=1} dt^k / k! A^(k-1) (A e0 + B u), summed until the terms vanish in Real.
    Real acc[M], nt[M];
#pragma unroll
    for (int j = 0; j < M; ++j) {
      acc[j] = c.predict_from_xtp1 ? x1[j] : phi[j];
      s_term[j * T] = acc[j];
      nt[j] = Real(0);
    }
#pragma unroll kRlsRowUnroll
    for (int i = 0; i < MN; ++i) {  // A e0 + B u = theta' [e0; u]
      const Real zi = i < M ? s_term[i * T] : s_phi[i * T];
#pragma unroll
      for (int j = 0; j < M; ++j) nt[j] += sT[(i * M + j) * T] * zi;
    }
    Real coef = Real(c.dt);
    const Real eps = sizeof(Real) == 4 ? Real(1e-9) : Real(1e-18);
#pragma unroll 1
    for (int k = 1; k <= 16; ++k) {
      Real big = Real(0), mag = Real(0);
#pragma unroll
      for (int j = 0; j < M; ++j) {
        const Real inc = coef * nt[j];
        acc[j] += inc;
        big = max_(big, abs_(inc)); mag = max_(mag, abs_(acc[j]));
        s_term[j * T] = nt[j]; nt[j] = Real(0);
      }
      if (big <= eps * mag) break;  // the series has converged in Real (|A| dt ~ 0.05: 5-7 terms)
      coef *= Real(c.dt) / Real(k + 1);
#pragma unroll kRlsRowUnroll
      for (int i = 0; i < M; ++i) {
        const Real ti = s_term[i * T];
#pragma unroll
        for (int j = 0; j < M; ++j) nt[j] += sT[(i * M + j) * T] * ti;
      }
    }
#pragma unroll
    for (int j = 0; j < M; ++j) r[j] = x1[j] - acc[j];
  }
}

// One RLS step for drone d.  phi = [e_t (m), u_t (4)], x1 = e_{t+1} (m).
// Both matrices are needed twice (gain / prediction over the WHOLE matrix first, rank-one update second), and a swarm's
// in-flight footprint (1.1 KB per drone) exceeds L2, so a second sweep over HBM planes would double the traffic.  Each
// thread therefore stages its own columns of P and theta in shared memory ([entry][thread]: conflict-free) with cp.async,
// works there (run-time row loops, register-resident column vectors) and writes the updated entries straight back:
// HBM sees every entry once in and once out.  A thread only ever touches its own shared column.
// PROJECT: whether project_theta is applied at all (compile-time: the unprojected variants carry none of its code)
template <typename Real, int M, bool PROJECT>
__global__ void __launch_bounds__(rls_threads<Real, M>()) rls_update_kernel(RlsP c, const Real* __restrict__ phi_in, const Real* __restrict__ x1_in,
                                                                         Real* __restrict__ theta, Real* __restrict__ Pm, Real* __restrict__ resid_out,
                                                                         int D_) {
  constexpr int MN = M + 4, T = rls_threads<Real, M>();
  extern __shared__ __align__(16) unsigned char rls_smem[];
  const int tid = threadIdx.x;
  constexpr int TRI = MN * (MN + 1) / 2;
  Real* sP = reinterpret_cast<Real*>(rls_smem) + tid;  // packed upper triangle of P: entry (i, j >= i) at sP[rls_tri<MN>(i, j) * T]
  Real* sT = sP + TRI * T;
  Real* s_phi = sT + MN * M * T;
  Real* s_w = s_phi + MN * T;
  Real* s_term = s_w + MN * T;
  // project_theta codes per theta row, block-shared (a parameter array indexed by the run-time row would be copied to
  // local memory); the only block barrier of the kernel, before any thread leaves
  __shared__ unsigned s_code[16];
  if (PROJECT && tid == 0) {
#pragma unroll
    for (int i = 0; i < MN; ++i) s_code[i] = c.row_code[i];
  }
  if (PROJECT) __syncthreads();
  const size_t d = (size_t)blockIdx.x * T + tid, D = (size_t)D_;
  if (d >= D) return;
#pragma unroll 1
  for (int i = 0; i < MN; ++i)
#pragma unroll 1
    for (int j = i; j < MN; ++j) cp_async_real(sP + rls_tri<MN>(i, j) * T, Pm + (size_t)(i * MN + j) * D + d);
#pragma unroll 1
  for (int k = 0; k < MN * M; ++k) cp_async_real(sT + k * T, theta + (size_t)k * D + d);
  Real x1[M], phi[MN], v[MN];  // v = phi' P = (P phi)' = w' by symmetry: accumulated from both halves of the triangle
#pragma unroll
  for (int i = 0; i < MN; ++i) { phi[i] = phi_in[d * MN + i]; s_phi[i * T] = phi[i]; v[i] = Real(0); }
#pragma unroll
  for (int i = 0; i < M; ++i) x1[i] = x1_in[d * M + i];
  cp_async_wait_all();
  // robots after the first of an env see the projection of the earlier robots' loop iterations before their own update
  const bool pre_project = PROJECT && c.project == MDS_RLS_PROJECT_LOOP && (d % (size_t)c.drones_per_env) != 0;
  if (pre_project) rls_pre_project<Real, M>(sT, s_code, T);
  // ---- gain: w = P phi (= v'), s = 1 + phi' P phi
  Real s = Real(1);
  if (sizeof(Real) == 4) {  // fully unrolled: every index is static, w lives in v[] (255 registers in fp32, no spills)
#pragma unroll
    for (int i = 0; i < MN; ++i) {
      Real wi = v[i];
#pragma unroll
      for (int j = i; j < MN; ++j) {
        const Real p = sP[rls_tri<MN>(i, j) * T];
        wi += p * phi[j];
        if (j > i) v[j] += p * phi[i];
      }
      v[i] = wi;
    }
  } else {  // fp64: rls_gain's row loop, inline (rls_gain itself costs this kernel 16-24 more instructions per variant, all
            // address arithmetic: the loads lose their shared base register with immediate offsets)
#pragma unroll 2
    for (int i = 0; i < MN; ++i) {
      const Real phi_i = s_phi[i * T];
      Real wi = Real(0);
      const int row0 = i * MN - i * (i - 1) / 2 - i;  // rls_tri(i, j) = row0 + j
#pragma unroll
      for (int j = 0; j < MN; ++j) {
        if (j >= i) {
          const Real p = sP[(row0 + j) * T];
          wi += p * phi[j];
          if (j > i) v[j] += p * phi_i;
        }
      }
      s_w[i * T] = wi;
    }
#pragma unroll
    for (int i = 0; i < MN; ++i) v[i] += s_w[i * T];
  }
#pragma unroll
  for (int i = 0; i < MN; ++i) { s_w[i * T] = v[i]; s += phi[i] * v[i]; }
  const Real inv_s = Real(1) / s;
  Real r[M];
  rls_residual<Real, M>(c, phi, x1, s_phi, sT, s_term, r, T);
  if (resid_out) {
#pragma unroll
    for (int j = 0; j < M; ++j) resid_out[d * M + j] = r[j];
  }
  // ---- theta += L r' (then project_theta), P -= (w / s) v: straight from the staged columns back to the HBM planes
#pragma unroll kRlsRowUnroll
  for (int i = 0; i < MN; ++i) {
    const Real wi = s_w[i * T];
    const Real Li = c.normalize_gain ? wi * inv_s : wi;
    if (!PROJECT) {
#pragma unroll
      for (int j = 0; j < M; ++j) theta[(size_t)(i * M + j) * D + d] = sT[(i * M + j) * T] + Li * r[j];
    } else {
      const unsigned word = s_code[i];
#pragma unroll
      for (int j = 0; j < M; ++j) {
        const unsigned code = (word >> (2 * j)) & 3u;
        const Real val = sT[(i * M + j) * T] + Li * r[j];
        theta[(size_t)(i * M + j) * D + d] = code == 1u ? val : (code == 0u ? Real(0) : Real(1));
      }
    }
  }
  // P -= (w / s) w': both triangles are written (the planes keep the full square), exactly symmetric
  if (sizeof(Real) == 4) {
#pragma unroll
    for (int i = 0; i < MN; ++i) {
      const Real Li = v[i] * inv_s;
#pragma unroll
      for (int j = i; j < MN; ++j) {
        const Real pij = sP[rls_tri<MN>(i, j) * T] - Li * v[j];
        Pm[(size_t)(i * MN + j) * D + d] = pij;
        if (j > i) Pm[(size_t)(j * MN + i) * D + d] = pij;
      }
    }
  } else {
#pragma unroll 2
    for (int i = 0; i < MN; ++i) {
      const Real Li = s_w[i * T] * inv_s;
      const int row0 = i * MN - i * (i - 1) / 2 - i;
#pragma unroll
      for (int j = 0; j < MN; ++j) {
        if (j >= i) {
          const Real pij = sP[(row0 + j) * T] - Li * v[j];
          Pm[(size_t)(i * MN + j) * D + d] = pij;
          if (j > i) Pm[(size_t)(j * MN + i) * D + d] = pij;
        }
      }
    }
  }
}

}  // namespace mds

// ================================================================== batched continuous-time Riccati solve
// compute_controller (decentralized_lqr_omega.py:185-204): K_d = R^-1 B_d' X_d with X_d the stabilising solution of
// A'X + XA - X B R^-1 B' X + Q = 0 for every drone's learned (A_d, B_d) = theta_d.  The reference calls scipy
// (solve_continuous_are: QZ on the balanced extended pencil) once per learning phase on the host; a swarm of distinct
// learned models needs one solve per drone, so here ONE WARP solves one drone's equation in shared memory, in double:
//   * state scaling z = sqrt(Q) x (Q diagonal) -> Q~ = I, which equalises the Hamiltonian's blocks (the reference's
//     Bryson weights span 1e-6 .. 1e6);
//   * matrix sign function of H = [[A~, -G~], [-I, -A~']] by the determinant-scaled Newton iteration
//     Z <- (c Z + (c Z)^-1) / 2, c = |det Z|^(-1/2m), each inverse a Gauss-Jordan sweep with partial pivoting over
//     [Z | I] (lane = row); 7-9 iterations to 1e-13;
//   * X~ from W12 X~ = -(W11 + I) (W = sign H), symmetrised, scaled back, then K = R^-1 B' X.
// Agreement with scipy on the reference's three parametrisations with perturbed / dense learned models: <= 2e-12 of max |K|.
namespace mds {

struct CareP {
  double sq[12];    // sqrt(q_ii)
  double rinv[4];   // 1 / r_ii
};

// Gauss-Jordan elimination with partial pivoting on the rows x cols matrix a (row stride ld, rows <= 32, lane = row) until
// its leading rows x rows block is the identity.  Returns false on a vanishing pivot; *logdet += sum log |pivot|.
MDS_DEV bool warp_gauss_jordan(double* a, int rows, int cols, int ld, int lane, double* logdet) {
  const unsigned full = 0xffffffffu;
  for (int k = 0; k < rows; ++k) {
    double best = (lane >= k && lane < rows) ? fabs(a[lane * ld + k]) : -1.0;
    int who = lane;
    for (int off = 16; off > 0; off >>= 1) {
      const double ob = __shfl_xor_sync(full, best, off);
      const int ow = __shfl_xor_sync(full, who, off);
      if (ob > best || (ob == best && ow < who)) { best = ob; who = ow; }
    }
    if (!(best > 1e-300)) return false;
    *logdet += log(best);
    if (who != k)
      for (int c = lane; c < cols; c += 32) { const double t = a[k * ld + c]; a[k * ld + c] = a[who * ld + c]; a[who * ld + c] = t; }
    __syncwarp(full);
    const double inv = 1.0 / a[k * ld + k];
    __syncwarp(full);
    for (int c = lane; c < cols; c += 32) a[k * ld + c] *= inv;
    __syncwarp(full);
    if (lane < rows && lane != k) {
      const double f = a[lane * ld + k];
      for (int c = 0; c < cols; ++c) a[lane * ld + c] -= f * a[k * ld + c];
    }
    __syncwarp(full);
  }
  return true;
}

#define MDS_CARE_WARPS 4
template <int M> constexpr int care_doubles_per_warp() { return (2 * M) * (2 * M) + (2 * M) * (4 * M + 1) + M * 4; }

template <typename Real, int M>
__global__ void __launch_bounds__(32 * MDS_CARE_WARPS) care_gain_kernel(CareP c, const Real* __restrict__ theta, Real* __restrict__ K,
                                                                        int* __restrict__ status, int D_) {
  constexpr int N2 = 2 * M, LD = 2 * N2 + 1;
  extern __shared__ __align__(16) unsigned char care_smem[];
  __shared__ double s_sq[12], s_rinv[4];
  if (threadIdx.x == 0) {
#pragma unroll
    for (int i = 0; i < M; ++i) s_sq[i] = c.sq[i];
#pragma unroll
    for (int i = 0; i < 4; ++i) s_rinv[i] = c.rinv[i];
  }
  __syncthreads();
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const size_t d = (size_t)blockIdx.x * MDS_CARE_WARPS + warp, D = (size_t)D_;
  if (d >= D) return;  // whole warps leave together
  const unsigned full = 0xffffffffu;
  double* Z = reinterpret_cast<double*>(care_smem) + (size_t)warp * care_doubles_per_warp<M>();
  double* Ag = Z + N2 * N2;
  double* Bs = Ag + N2 * LD;  // B~ [M][4] = sqrt(Q) B
  auto th = [&](int i, int j) { return (double)theta[(size_t)(i * M + j) * D + d]; };  // theta[i][j]: A[j][i] for i < M, B[j][i-M] above
  if (lane < M)
    for (int k = 0; k < 4; ++k) Bs[lane * 4 + k] = th(M + k, lane) * s_sq[lane];
  __syncwarp(full);
  if (lane < M) {  // rows [A~, -G~]
    const int r = lane;
    for (int cc = 0; cc < M; ++cc) {
      Z[r * N2 + cc] = th(cc, r) * s_sq[r] / s_sq[cc];
      double g = 0.0;
      for (int k = 0; k < 4; ++k) g += Bs[r * 4 + k] * s_rinv[k] * Bs[cc * 4 + k];
      Z[r * N2 + M + cc] = -g;
    }
  } else if (lane < N2) {  // rows [-I, -A~']
    const int r = lane - M;
    for (int cc = 0; cc < M; ++cc) {
      Z[lane * N2 + cc] = cc == r ? -1.0 : 0.0;
      Z[lane * N2 + M + cc] = -th(r, cc) * s_sq[cc] / s_sq[r];
    }
  }
  __syncwarp(full);
  bool ok = true;
  int it = 0;
  for (; it < 60; ++it) {
    if (lane < N2)
      for (int cc = 0; cc < N2; ++cc) { Ag[lane * LD + cc] = Z[lane * N2 + cc]; Ag[lane * LD + N2 + cc] = cc == lane ? 1.0 : 0.0; }
    __syncwarp(full);
    double logdet = 0.0;
    if (!warp_gauss_jordan(Ag, N2, 2 * N2, LD, lane, &logdet)) { ok = false; break; }
    const double sc = exp(-logdet / (double)N2), isc = 1.0 / sc;
    double diff = 0.0, mx = 0.0;
    if (lane < N2)
      for (int cc = 0; cc < N2; ++cc) {
        const double z = Z[lane * N2 + cc], zn = 0.5 * (sc * z + isc * Ag[lane * LD + N2 + cc]);
        diff = fmax(diff, fabs(zn - z)); mx = fmax(mx, fabs(zn));
        Z[lane * N2 + cc] = zn;
      }
    for (int off = 16; off > 0; off >>= 1) { diff = fmax(diff, __shfl_xor_sync(full, diff, off)); mx = fmax(mx, __shfl_xor_sync(full, mx, off)); }
    __syncwarp(full);
    if (diff <= 1e-13 * mx) break;
  }
  if (ok && it < 60) {  // W12 X~ = -(W11 + I)
    constexpr int LD2 = 2 * M + 1;
    if (lane < M)
      for (int cc = 0; cc < M; ++cc) {
        Ag[lane * LD2 + cc] = Z[lane * N2 + M + cc];
        Ag[lane * LD2 + M + cc] = -(Z[lane * N2 + cc] + (cc == lane ? 1.0 : 0.0));
      }
    __syncwarp(full);
    double ld = 0.0;
    ok = warp_gauss_jordan(Ag, M, 2 * M, LD2, lane, &ld);
    if (ok && lane < M) {  // column `lane` of K = R^-1 B' X, X[r][c] = sq_r (X~[r][c] + X~[c][r]) / 2 sq_c
      double kc[4] = {0.0, 0.0, 0.0, 0.0};
      for (int r = 0; r < M; ++r) {
        const double x = 0.5 * (Ag[r * LD2 + M + lane] + Ag[lane * LD2 + M + r]) * s_sq[lane];  // times sq_r below, inside B~
        for (int i = 0; i < 4; ++i) kc[i] += Bs[r * 4 + i] * x;
      }
      for (int i = 0; i < 4; ++i) K[(size_t)(i * M + lane) * D + d] = (Real)(s_rinv[i] * kc[i]);
    }
  } else {
    ok = false;
  }
  if (lane == 0 && status) status[d] = ok ? 0 : 1;
}

}  // namespace mds
