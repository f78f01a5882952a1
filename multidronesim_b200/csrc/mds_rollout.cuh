// mds_rollout.cuh -- the lane-group machinery and the two heavy kernels of the fused control step
// (ctrl_step_kernel, rollout_loop_kernel) + physics_step_kernel.  Header so that every
// (precision, kernel kind) pair compiles in its own translation unit (mds_rollout_tu.cu; `make -j`).
#pragma once
#include <cuda_runtime.h>
#include "mds_cbf.cuh"
#include "mds_common.cuh"
#include "mds_ctrl.cuh"
#include "mds_physics.cuh"
#include "mds_traj.cuh"

using namespace mds;

// ------------------------------------------------------------------ thread mapping
// An environment's drones occupy NP = next_pow2(N) consecutive lanes of ONE warp ("lane group"; lanes
// n >= N idle), so every cross-drone exchange (downwash neighbours, CBF rows, the QP) needs only
// group-level synchronisation: shared memory + __syncwarp(gmask) / shuffles.  No block barriers.
#ifndef MDS_BLOCK
#define MDS_BLOCK 256
#endif
#ifndef MDS_CTRL_MINB
#define MDS_CTRL_MINB 4  // resident blocks per SM of the NON-persistent controller kernel (64 registers; MDS_CTRL_PERSISTENT=0 builds it)
#endif
#ifndef MDS_LOOP_MINB
#define MDS_LOOP_MINB 2  // the K-step loop kernel serves small swarms: registers before occupancy
#endif
#ifndef MDS_LOOP_BLOCK
#define MDS_LOOP_BLOCK 256  // threads per block of the K-step loop kernel (a multiple of 32, <= MDS_BLOCK); with MDS_LOOP_MINB it sets the register cap
#endif
#ifndef MDS_LOOP_BLOCK_F64
#define MDS_LOOP_BLOCK_F64 192  // fp64: 2 x 192 threads = 168 registers (2 x 256 = 128 spills 59 loads + 26 stores per warp-step: 0.184 -> 0.167 ms)
#endif
// threads per block of the loop kernels for a precision
template <typename Real> constexpr int loop_block() { return sizeof(Real) == 4 ? MDS_LOOP_BLOCK : MDS_LOOP_BLOCK_F64; }
#ifndef MDS_PHYS_MINB
#define MDS_PHYS_MINB 5
#endif
static inline int next_pow2(int n) { int p = 1; while (p < n) p <<= 1; return p; }
struct GroupMap {
  int el, n, e, d;   // env slot in block, drone in env, global env, global drone
  bool valid;        // lane maps to a real drone
  bool env_valid;    // group maps to a real env
  unsigned gmask;    // lanes of this group within the warp
  unsigned cmask;    // mask for the synchronising calls at the stage boundaries every lane group of the warp reaches together:
                     // gmask, or the full warp where a kernel guarantees 32 live lanes (rollout_loop_kernel FULLW)
};
// tile: which block-sized slice of the environments this block works on (blockIdx.x, or the iteration of a persistent kernel)
MDS_DEV GroupMap group_map(int N, int NP, int E, int tile) {
  GroupMap g;
  const int tid = threadIdx.x, lg = __ffs(NP) - 1;  // NP is a power of two
  g.el = tid >> lg;
  g.n = tid & (NP - 1);
  g.e = tile * (blockDim.x >> lg) + g.el;  // blockDim.x <= MDS_BLOCK (launch_geometry)
  g.env_valid = g.e < E;
  g.valid = g.env_valid && g.n < N;
  g.d = g.e * N + g.n;
  const int lane0 = (tid & 31) & ~(NP - 1);
  g.gmask = NP >= 32 ? 0xffffffffu : (((1u << NP) - 1u) << lane0);
  g.cmask = g.gmask;
  return g;
}

MDS_DEV GroupMap group_map(int N, int NP, int E) { return group_map(N, NP, E, (int)blockIdx.x); }

// OR over the lane group.  __reduce_or_sync with a partial run-time mask makes the lane groups of a warp take turns
// (WARPSYNC.EXCLUSIVE: 6 instructions per group, 24 per warp); log2(NP) butterfly shuffles serve all groups at once.
MDS_DEV unsigned group_or(unsigned gmask, int NP, unsigned v) {
#ifndef MDS_NO_OR_SHFL
  if (NP < 32) {
#pragma unroll
    for (int w = 1; w < 32; w <<= 1)
      if (w < NP) v |= __shfl_xor_sync(gmask, v, w);
    return v;
  }
#endif
  return __reduce_or_sync(gmask, v);
}

// Compile-time drone count that fills its lane group (N == NP, e.g. the swarm's 8): every lane of a valid environment
// maps to a drone, so `valid` is a compile-time `true` inside the env_valid region and the per-stage `if (g.valid)`
// guards fold away (uniform branches: fewer instructions, no measurable change in time).
template <int NT> MDS_DEV void full_group_hint(GroupMap& g) {
  if (NT > 0 && (NT & (NT - 1)) == 0) g.valid = true;
}

// Downwash sum for this lane's drone over its env mates, whose positions the group has already published in shared memory:
// drone m's position is the (x, y, z) of pos[STRIDE m].  Called by every lane of the group (shuffles, no sync).  Only the
// LOWER drone of a pair feels the other's downwash, so each unordered pair is evaluated once, by the lane that owns it under
// the CBF stage's ownership (mds_cbf.cuh: lane n owns (n, n+s+1 mod N) for s < (N-1)/2, and the "diameter" (n, n+N/2) for
// n < N/2 when N is even); the owner keeps the term if it is the lower one and otherwise hands it to its partner with one
// shuffle per slot.
template <int STRIDE, typename Real>
MDS_DEV Real downwash_exchange(const DroneP<Real>& P, const typename Vec4T<Real>::type* pos, V3<Real> p, const GroupMap& g, int N, int NP) {
  Real dw = Real(0);
  const int n = g.n, lane0 = (threadIdx.x & 31) - n;
  const int K1 = (N - 1) >> 1, half = (N & 1) ? 0 : (N >> 1), S0 = K1 + (half ? 1 : 0);
#pragma unroll
  for (int s = 0; s < S0; ++s) {
    int m = n, src = n;  // partner of the pair this lane owns in slot s; lane whose slot-s pair has this lane as partner
    bool own = false, recv = false;
    if (g.valid) {
      if (s < K1) {
        m = n + s + 1; m = m >= N ? m - N : m;
        src = n - s - 1; src = src < 0 ? src + N : src;
        own = true; recv = true;
      } else if (n < half) { m = n + half; own = true; }
      else { src = n - half; recv = true; }
    }
    Real give = Real(0);
    if (own) {
      const auto q = pos[STRIDE * m];
      const Real dz = q.z - p.z, dx = q.x - p.x, dy = q.y - p.y;  // dz > 0: the partner is above, this drone is pushed down
      const Real dxy2 = dx * dx + dy * dy;
      Real v = Real(0);
      if (dz != Real(0) && dxy2 < Real(100)) v = downwash_pair(P, abs_(dz), dxy2);
      if (dz > Real(0)) dw += v;
      else give = v;
    }
    const Real got = __shfl_sync(g.cmask, give, lane0 + src);
    if (recv) dw += got;
  }
  return dw;
}

// fp32: two slots per pass with packed fp32 arithmetic (mds_common.cuh F2) -- slot s in the low halves, slot s + 1 in the
// high halves; a slot this lane does not own is evaluated against the lane's own position (dz = 0: no force).  Per pair of
// slots ~30 instructions instead of 2 x 25, and the half-populated "diameter" slot rides along for free.
#ifndef MDS_NO_DW_PACK
template <int STRIDE>
MDS_DEV float downwash_exchange(const DroneP<float>& P, const float4* pos, V3<float> p, const GroupMap& g, int N, int NP) {
  float dw = 0.f;
  const int n = g.n;
  const int K1 = (N - 1) >> 1, half = (N & 1) ? 0 : (N >> 1), S0 = K1 + (half ? 1 : 0);
#pragma unroll
  for (int s = 0; s < S0; s += 2) {
    int m[2] = {n, n}, src[2] = {n, n};
    bool recv[2] = {false, false};
#pragma unroll
    for (int h = 0; h < 2; ++h) {
      const int sl = s + h;
      if (g.valid && sl < S0) {
        if (sl < K1) {
          m[h] = wrap_n(n + sl + 1, N);
          src[h] = wrap_n(n - sl - 1, N);
          recv[h] = true;
        } else if (n < half) m[h] = n + half;
        else { src[h] = n - half; recv[h] = true; }
      }
    }
    const float4 q0 = pos[STRIDE * m[0]], q1 = pos[STRIDE * m[1]];
    const F2 dz(q0.z - p.z, q1.z - p.z), dx(q0.x - p.x, q1.x - p.x), dy(q0.y - p.y, q1.y - p.y);  // dz > 0: the partner is above
    const F2 dxy2 = fma_(dy, dy, dx * dx);
    const F2 v = downwash_pair2(P, F2(abs_(dz.v.x), abs_(dz.v.y)), dxy2);
    const float v0 = (dz.v.x != 0.f && dxy2.v.x < 100.f) ? v.v.x : 0.f, v1 = (dz.v.y != 0.f && dxy2.v.y < 100.f) ? v.v.y : 0.f;
    dw += dz.v.x > 0.f ? v0 : 0.f;
    dw += dz.v.y > 0.f ? v1 : 0.f;
    const float got0 = __shfl_sync(g.cmask, dz.v.x > 0.f ? 0.f : v0, src[0], NP);  // width NP: the source is relative to the lane group
    if (recv[0]) dw += got0;
    if (s + 1 < S0) {
      const float got1 = __shfl_sync(g.cmask, dz.v.y > 0.f ? 0.f : v1, src[1], NP);
      if (recv[1]) dw += got1;
    }
  }
  return dw;
}
#endif

// The same with the positions staged here: env_pos is the environment's NP slots -- a slice of a per-block array, or the
// head of the environment's CBF block, which is idle during the physics.  Two group syncs.
template <typename Real>
MDS_DEV Real downwash_group(const DroneP<Real>& P, typename Vec4T<Real>::type* env_pos, V3<Real> p, const GroupMap& g, int N, int NP) {
  typename Vec4T<Real>::type me;
  me.x = p.x; me.y = p.y; me.z = p.z; me.w = Real(0);
  env_pos[g.n] = me;
  __syncwarp(g.cmask);
  const Real dw = downwash_exchange<1>(P, env_pos, p, g, N, NP);
  __syncwarp(g.cmask);
  return dw;
}

// per-env shared-memory block of the CBF stage (in Reals; every part is a multiple of 4 so that the Vec4
// accesses stay aligned):
//   head  max(12 NP, WS)  agents (p, dv, da per drone; 3 Vec4 each) -- overlaid by the QP workspace once the rows exist
//   rows  4 NP RPL        one Vec4 (a0, a1, a2, rhs) per row, owner-major (mds_cbf.cuh "Row ownership")
//   x     4 NP            the QP iterate, one Vec4 per drone
//   xnom  4 NP            u_nom, kept for the fp32 polish of long solves
template <typename Real> struct CbfSmem {
  Real* env0;
  int stride, off_rows, off_x;
};
static inline int cbf_env_stride(int NP, int N, int n_obs) {
  int rpl = (N - 1) / 2 + ((N & 1) ? 0 : 1) + n_obs;
  int head = 12 * NP > MDS_QP_WS_WORDS ? 12 * NP : ((MDS_QP_WS_WORDS + 3) & ~3);
  return head + 4 * NP * rpl + 8 * NP;
}
template <typename Real> static size_t cbf_smem_bytes(int threads, int NP, int N, int n_obs) {
  return (size_t)(threads / NP) * cbf_env_stride(NP, N, n_obs) * sizeof(Real) + 32;
}
// Threads per block (a power of two in [NP or 32, MDS_BLOCK]) such that the CBF stage's shared memory stays under
// ~100 KB per block (two blocks per SM): only small lane groups in fp64 (many envs per block, each with its own QP
// workspace) and 32-drone groups with many obstacles ever need fewer than MDS_BLOCK threads.
template <typename Real> static int cbf_block_threads(int NP, int N, int n_obs, int max_threads = MDS_BLOCK) {
  int threads = max_threads;
  const int floor_threads = NP > 32 ? NP : 32;
  while (threads > floor_threads && cbf_smem_bytes<Real>(threads, NP, N, n_obs) > 100 * 1024) {
    threads = (threads >> 1) & ~31;  // whole warps (the loop kernel may start from 224 or 192)
    if (threads < floor_threads) threads = floor_threads;
  }
  return threads;
}
template <typename Real> MDS_DEV CbfSmem<Real> cbf_smem_carve(unsigned char* raw, int NP, int N, int n_obs) {
  CbfSmem<Real> s;
  s.env0 = reinterpret_cast<Real*>(raw);
  const RowMap M = row_map(N, n_obs);
  int head = 12 * NP > MDS_QP_WS_WORDS ? 12 * NP : ((MDS_QP_WS_WORDS + 3) & ~3);
  s.off_rows = head; s.off_x = head + 4 * NP * M.RPL;
  s.stride = s.off_x + 8 * NP;  // x, then the untouched copy of u_nom
  return s;
}

// CBF safety filter for one env by its lane group: u_nom -> u_safe for this lane's drone.
// Every lane of a valid group calls it; returns the env's QP status, *iters_out its iteration count.
//
// Flow.  Constraints that touch ONE drone's inputs (its obstacle rows and its +-umax box) are orthogonal between
// drones, so each lane first handles its own in registers: it finds its most violated one at u_nom and projects onto
// it (one closed-form Goldfarb-Idnani step).  The lanes then publish their agents and projected inputs, build their pair
// rows and test them -- and their other single-drone rows -- at the projected point.  If nothing is violated the point is
// the QP's minimiser (it minimises |u - u_nom|^2 on an active set with positive multipliers and is feasible for every
// other row), and the step is over without any group-wide argmin, workspace or second scan: in the swarm workloads that
// is nearly every step.  Otherwise the group runs the cooperative active-set solver from u_nom (qp_solve_group), and if
// that one runs out of workspace / iterations or its factor breaks down, the scratch solver (qp_solve_group_big).
// NT > 0 (compile-time drone count) in fp32: the pair rows are evaluated two at a time with packed fp32 instructions
// (cbf_row2) and stay in registers -- they are written to shared memory only if the cooperative solver is needed.
// dw_out (optional): receives this lane's downwash sum (downwash_group's value) when dw_on -- the agents the stage exchanges
// carry the positions the physics starts from, and the pair rows have the downwash's pair ownership, so the physics' own
// publication of the positions and its two group syncs are not needed.  The packed path takes each slot's downwash from the
// partner it has just loaded for the row; the scalar path runs downwash_exchange over the published agents.
template <int ORD, typename Real, int NT = 0>
MDS_DEV int cbf_filter_group(const DroneP<Real>& P, const CbfP<Real>& C, const CbfSmem<Real>& S, const Real* obstacles, int n_obs,
                             const GroupMap& g, int N, int NP, const CbfAgent<Real>& ag, Real F, const Real unom[4], Real usafe[4],
                             Real* min_h, int* iters_out, Real* dw_out = nullptr, bool dw_on = false) {
  using R4 = typename Vec4T<Real>::type;
  const bool fuse_dw = dw_out != nullptr && dw_on;  // uniform over the group
  Real dw = Real(0);
  const int n = g.n;
  const RowMap M = row_map(N, n_obs);
  Real* env = S.env0 + (size_t)g.el * S.stride;
  R4* agents = reinterpret_cast<R4*>(env);
  R4* rows = reinterpret_cast<R4*>(env + S.off_rows);
  R4* x = reinterpret_cast<R4*>(env + S.off_x);
  R4* xnom = x + NP;
  int fl = 0, escalate = 0, touched = 0;
  Real lo = Real(0), hi = Real(0);
  Real xn[3] = {unom[0], unom[1], unom[2]};
  if (g.valid) {
    // ---- own single-drone rows: obstacle rows (built here), box bounds; most violated one at u_nom.  Written without
    // branches: in the swarm workloads a quarter of the drones project at any step, so a branch would run its body for a
    // few lanes of nearly every warp (ncu: 8 of 32 threads) -- selects cost less than the partial-warp passes.
    Real wv = Real(0);  // normalised slack of the most violated row so far (negative)
    int wobs = -1;      // the most violated obstacle row, kept in registers: (a, rhs), |a|^2
    Real w0 = Real(0), w1 = Real(0), w2 = Real(0), w3 = Real(0), wa2 = Real(1);
    const CbfAgent<Real> zero = {{Real(0), Real(0), Real(0)}, {Real(0), Real(0), Real(0)}, {Real(0), Real(0), Real(0)}};
    auto obstacle_row = [&](int o) {
      CbfAgent<Real> other = zero;
      other.p = {obstacles[4 * o], obstacles[4 * o + 1], obstacles[4 * o + 2]};
      Real a3[3], rhs, h0, Ds, c4inv;
      obstacle_shape(C, obstacles[4 * o + 3], &Ds, &c4inv);
      const Real Ds2 = Ds * Ds;
      cbf_row<ORD>(P, C, ag, other, Ds2 * Ds2, c4inv, a3, &rhs, &h0);
      *min_h = min_(*min_h, h0);
      R4 row;
      row.x = a3[0]; row.y = a3[1]; row.z = a3[2]; row.w = rhs;
      rows[n * M.RPL + M.S0 + o] = row;
      // G u = -a . u_n <= rhs
      const Real sl = rhs + (a3[0] * xn[0] + a3[1] * xn[1] + a3[2] * xn[2]);
      const Real mag = abs_(a3[0] * xn[0]) + abs_(a3[1] * xn[1]) + abs_(a3[2] * xn[2]);
      const bool viol = sl < -qp_tol<Real>() * (abs_(rhs) + mag + Real(1e-12));
      const Real a2 = a3[0] * a3[0] + a3[1] * a3[1] + a3[2] * a3[2];
      if (viol && !(a2 > Real(0))) escalate = 1;  // zero row with negative rhs: the cooperative path reports it as infeasible
      const Real v = sl * rsqrt_(max_(a2, Real(1e-30)));
      const bool worse = viol && v < wv;
      wv = worse ? v : wv; wobs = worse ? o : wobs;
      w0 = worse ? a3[0] : w0; w1 = worse ? a3[1] : w1; w2 = worse ? a3[2] : w2; w3 = worse ? rhs : w3; wa2 = worse ? a2 : wa2;
    };
    // first obstacle peeled (the usual count is one): its "worst so far" state is the constants above, and the loop
    // bookkeeping stays off the common path
    if (n_obs > 0) obstacle_row(0);
    for (int o = 1; o < n_obs; ++o) obstacle_row(o);
    // box bounds: |u| > umax_hi  <=>  umax - |u| < -tol (umax + |u|); a later component wins only if strictly worse.
    // (Literal indices: a component INDEX would let nvcc turn the selects into dynamically indexed accesses, i.e. move u_n
    // and the whole parameter block C into local memory.)
    const Real ax0 = abs_(xn[0]), ax1 = abs_(xn[1]), ax2 = abs_(xn[2]);
    const Real v0 = C.umax[0] - ax0, v1 = C.umax[1] - ax1, v2 = C.umax[2] - ax2;
    const bool b0 = ax0 > C.umax_hi[0] && v0 < wv;
    wv = b0 ? v0 : wv;
    const bool b1 = ax1 > C.umax_hi[1] && v1 < wv;
    wv = b1 ? v1 : wv;
    const bool b2 = ax2 > C.umax_hi[2] && v2 < wv;
    const bool wb2 = b2, wb1 = b1 && !b2, wb0 = b0 && !b1 && !b2, isbox = b0 || b1 || b2;
    // one projection: u_n <- u_n - t g (g = -a),  t = -slack / |g|^2 (t = 0 unless an obstacle row is the worst); or the box face
    const Real t = (wobs >= 0 && !isbox) ? -(w3 + (w0 * xn[0] + w1 * xn[1] + w2 * xn[2])) / wa2 : Real(0);
    xn[0] += t * w0; xn[1] += t * w1; xn[2] += t * w2;
    xn[0] = wb0 ? (xn[0] < Real(0) ? -C.umax[0] : C.umax[0]) : xn[0];
    xn[1] = wb1 ? (xn[1] < Real(0) ? -C.umax[1] : C.umax[1]) : xn[1];
    xn[2] = wb2 ? (xn[2] < Real(0) ? -C.umax[2] : C.umax[2]) : xn[2];
    touched = (wobs >= 0 || isbox) ? 1 : 0;
    // the other single-drone rows at the projected point (the projected row itself holds with equality: skipped); only
    // when there is another obstacle row than the projected one -- a rare branch
    if (touched && n_obs > (isbox ? 0 : 1)) {
      const int wcon = isbox ? -1 : wobs;
      for (int o = 0; o < n_obs; ++o) {
        if (o == wcon) continue;
        const R4 row = rows[n * M.RPL + M.S0 + o];
        const Real sl = row.w + (row.x * xn[0] + row.y * xn[1] + row.z * xn[2]);
        if (sl < Real(0)) {
          const Real mag = abs_(row.x * xn[0]) + abs_(row.y * xn[1]) + abs_(row.z * xn[2]);
          if (sl < -qp_tol<Real>() * (abs_(row.w) + mag + Real(1e-12))) escalate = 1;
        }
      }
    }
    // the box at the projected point (an untouched u_n is inside it)
    const bool out0 = abs_(xn[0]) > C.umax_hi[0], out1 = abs_(xn[1]) > C.umax_hi[1], out2 = abs_(xn[2]) > C.umax_hi[2];
    escalate |= (int)((!wb0 & out0) | (!wb1 & out1) | (!wb2 & out2));  // bitwise: no short-circuit branches
    if (!cbf_wz_bounds<ORD>(C, F, &lo, &hi)) fl = 1;
    // ---- publish the agent and the projected inputs
    R4 a0, a1, a2, xv;
    a0.x = ag.p.x; a0.y = ag.p.y; a0.z = ag.p.z; a0.w = ag.dv.x;
    a1.x = ag.dv.y; a1.y = ag.dv.z; a1.z = ag.da.x; a1.w = ag.da.y;
    a2.x = ag.da.z; a2.y = Real(0); a2.z = Real(0); a2.w = Real(0);
    agents[3 * n] = a0; agents[3 * n + 1] = a1; agents[3 * n + 2] = a2;
    xv.x = xn[0]; xv.y = xn[1]; xv.z = xn[2]; xv.w = unom[3];
    x[n] = xv;
  }
  __syncwarp(g.cmask);
  constexpr bool PACK = (NT > 1) && sizeof(Real) == 4;
  constexpr int S0C = PACK ? (NT - 1) / 2 + ((NT & 1) ? 0 : 1) : 1, NPAIR = (S0C + 1) / 2;
  F2 pa[NPAIR][3], prhs[NPAIR];  // packed path: the pair rows, slot 2q in the low halves and 2q + 1 in the high halves
  if constexpr (PACK) {
    // the downwash shuffles below need every lane of the group: `valid` must be the compile-time true of full_group_hint
    static_assert((NT & (NT - 1)) == 0, "the packed pair loop needs a drone count that fills its lane group");
    if (g.valid) {
#pragma unroll
      for (int q = 0; q < NPAIR; ++q) {
        const int s0 = 2 * q, s1 = 2 * q + 1;
        // a slot below K1 always has a partner (compile-time); the "diameter" slot only for the lower half of the drones
        const bool ok0 = s0 < M.K1 || n < M.half, ok1 = s1 < S0C && (s1 < M.K1 || n < M.half);
        const int m0 = ok0 ? row_partner(M, N, n, s0) : n, m1 = ok1 ? row_partner(M, N, n, s1) : n;
        CbfAgent<float> o0, o1;
        const R4 b0 = agents[3 * m0], b1 = agents[3 * m0 + 1], b2 = agents[3 * m0 + 2], xm0 = x[m0];
        const R4 c0 = agents[3 * m1], c1 = agents[3 * m1 + 1], c2 = agents[3 * m1 + 2], xm1 = x[m1];
        o0.p = {b0.x, b0.y, b0.z}; o0.dv = {b0.w, b1.x, b1.y}; o0.da = {b1.z, b1.w, b2.x};
        o1.p = {c0.x, c0.y, c0.z}; o1.dv = {c0.w, c1.x, c1.y}; o1.da = {c1.z, c1.w, c2.x};
        F2 rhs, h0;
        cbf_row2<ORD>(P, C, ag, o0, o1, C.ds4_pair, C.c4inv, pa[q], &rhs, &h0);  // owner - partner (mds_cbf.cuh "Row ownership")
        if (ok0) *min_h = min_(*min_h, h0.v.x);
        else { pa[q][0].v.x = 0.f; pa[q][1].v.x = 0.f; pa[q][2].v.x = 0.f; rhs.v.x = 1e30f; }  // unused slot: a never-violated row
        if (ok1) *min_h = min_(*min_h, h0.v.y);
        else { pa[q][0].v.y = 0.f; pa[q][1].v.y = 0.f; pa[q][2].v.y = 0.f; rhs.v.y = 1e30f; }
        prhs[q] = rhs;
        if (fuse_dw) {
          // The two slots' downwash: packed downwash_exchange, the same operations in the same order, from the partners just
          // loaded.  It reads the row's differences e = own - partner where downwash_exchange forms d = partner - own: IEEE
          // subtraction is sign-symmetric (flushed denormals included), so |dz| = |ez|, dz > 0 <=> ez < 0, and
          // dxy2 = fma(dy, dy, dx dx) is bit for bit the row's rho = fma(ey, ey, ex ex) -- the same instructions as the row's.
          const F2 ex(ag.p.x - o0.p.x, ag.p.x - o1.p.x), ey(ag.p.y - o0.p.y, ag.p.y - o1.p.y), ez(ag.p.z - o0.p.z, ag.p.z - o1.p.z);
          const F2 dxy2 = fma_(ey, ey, ex * ex);
          const F2 v = downwash_pair2(P, F2(abs_(ez.v.x), abs_(ez.v.y)), dxy2);
          const float v0 = (ez.v.x != 0.f && dxy2.v.x < 100.f) ? v.v.x : 0.f, v1 = (ez.v.y != 0.f && dxy2.v.y < 100.f) ? v.v.y : 0.f;
          dw += ez.v.x < 0.f ? v0 : 0.f;  // the partner is above: this drone is pushed down
          dw += ez.v.y < 0.f ? v1 : 0.f;
          // the lane that owns the slot's pair with this lane as its partner (none: the lower half's diameter slot)
          const bool recv0 = s0 < M.K1 || n >= M.half, recv1 = s1 < M.K1 || n >= M.half;
          const int src0 = s0 < M.K1 ? wrap_n(n - s0 - 1, N) : (recv0 ? n - M.half : n);
          const int src1 = s1 < M.K1 ? wrap_n(n - s1 - 1, N) : (recv1 ? n - M.half : n);
          const float got0 = __shfl_sync(g.cmask, ez.v.x < 0.f ? 0.f : v0, src0, NP);
          if (recv0) dw += got0;
          if (s1 < S0C) {
            const float got1 = __shfl_sync(g.cmask, ez.v.y < 0.f ? 0.f : v1, src1, NP);
            if (recv1) dw += got1;
          }
        }
        // G u = -a . u_n + a . u_m <= rhs  <=>  slack = rhs + a . (u_n - u_m) >= 0
        const F2 sl = fma_(pa[q][2], F2(xn[2] - xm0.z, xn[2] - xm1.z),
                           fma_(pa[q][1], F2(xn[1] - xm0.y, xn[1] - xm1.y), fma_(pa[q][0], F2(xn[0] - xm0.x, xn[0] - xm1.x), rhs)));
        if (sl.v.x < 0.f) {
          const float a0 = pa[q][0].v.x, a1 = pa[q][1].v.x, a2 = pa[q][2].v.x;
          const float mag = abs_(a0 * xn[0]) + abs_(a1 * xn[1]) + abs_(a2 * xn[2]) + abs_(a0 * xm0.x) + abs_(a1 * xm0.y) + abs_(a2 * xm0.z);
          if (sl.v.x < -qp_tol<float>() * (abs_(rhs.v.x) + mag + 1e-12f)) escalate = 1;
        }
        if (sl.v.y < 0.f) {
          const float a0 = pa[q][0].v.y, a1 = pa[q][1].v.y, a2 = pa[q][2].v.y;
          const float mag = abs_(a0 * xn[0]) + abs_(a1 * xn[1]) + abs_(a2 * xn[2]) + abs_(a0 * xm1.x) + abs_(a1 * xm1.y) + abs_(a2 * xm1.z);
          if (sl.v.y < -qp_tol<float>() * (abs_(rhs.v.y) + mag + 1e-12f)) escalate = 1;
        }
      }
    }
  } else if (g.valid) {
    // ---- own pair rows (compile-time count when N is), each tested at the projected point as it is built
#pragma unroll
    for (int s = 0; s < M.S0; ++s) {
      const int m = row_partner(M, N, n, s);
      R4 row;
      row.x = Real(0); row.y = Real(0); row.z = Real(0); row.w = Real(1e30);
      if (m >= 0) {
        CbfAgent<Real> other;
        R4 b0 = agents[3 * m], b1 = agents[3 * m + 1], b2 = agents[3 * m + 2], xm = x[m];
        other.p = {b0.x, b0.y, b0.z}; other.dv = {b0.w, b1.x, b1.y}; other.da = {b1.z, b1.w, b2.x};
        Real a3[3], rhs, h0;
        cbf_row<ORD>(P, C, ag, other, C.ds4_pair, C.c4inv, a3, &rhs, &h0);  // owner - partner (mds_cbf.cuh "Row ownership")
        *min_h = min_(*min_h, h0);
        row.x = a3[0]; row.y = a3[1]; row.z = a3[2]; row.w = rhs;
        // G u = -a . u_n + a . u_m <= rhs
        const Real d0 = xm.x - xn[0], d1 = xm.y - xn[1], d2 = xm.z - xn[2];
        const Real sl = rhs - (a3[0] * d0 + a3[1] * d1 + a3[2] * d2);
        if (sl < Real(0)) {
          const Real mag = abs_(a3[0] * xn[0]) + abs_(a3[1] * xn[1]) + abs_(a3[2] * xn[2]) + abs_(a3[0] * xm.x) + abs_(a3[1] * xm.y) + abs_(a3[2] * xm.z);
          if (sl < -qp_tol<Real>() * (abs_(rhs) + mag + Real(1e-12))) escalate = 1;
        }
      }
      rows[n * M.RPL + s] = row;
    }
  }
  if constexpr (!PACK) {
    if (fuse_dw) dw = downwash_exchange<3>(P, agents, ag.p, g, N, NP);  // before the QP workspace overlays the agents
  }
  if (dw_out != nullptr) *dw_out = dw;
  // one group-wide OR of (escalate, infeasible 4th-input interval, projected) -- the step's only collective in the common case
  const unsigned any = group_or(g.cmask, NP, (unsigned)(escalate | (fl << 1) | (touched << 2)));
  int status = MDS_QP_OPTIMAL, iters = (any & 4u) ? 1 : 0;
  if (any & 2u) {
    status = MDS_QP_INFEASIBLE;
  } else if (any & 1u) {
    // ---- cooperative solve from u_nom (agents are no longer needed: their storage becomes the QP workspace)
    if constexpr (PACK) {  // the solver reads the rows from shared memory
      if (g.valid) {
#pragma unroll
        for (int q = 0; q < NPAIR; ++q) {
          R4 r0, r1;
          r0.x = pa[q][0].v.x; r0.y = pa[q][1].v.x; r0.z = pa[q][2].v.x; r0.w = prhs[q].v.x;
          r1.x = pa[q][0].v.y; r1.y = pa[q][1].v.y; r1.z = pa[q][2].v.y; r1.w = prhs[q].v.y;
          rows[n * M.RPL + 2 * q] = r0;
          if (2 * q + 1 < S0C) rows[n * M.RPL + 2 * q + 1] = r1;
        }
      }
    }
    __syncwarp(g.gmask);  // every lane has read its partners' agents and projected inputs
    if (g.valid) {
      R4 xv;
      xv.x = unom[0]; xv.y = unom[1]; xv.z = unom[2]; xv.w = unom[3];
      x[n] = xv; xnom[n] = xv;
    }
    __syncwarp(g.gmask);
    const Real un3[3] = {unom[0], unom[1], unom[2]};
    const int p0 = qp_scan(C, rows, x, un3, M, N, NP, n, g.valid, 0u, 0u, g.gmask);
    if (p0 == -2) status = MDS_QP_INFEASIBLE;
    else if (p0 >= 0) {
      status = qp_solve_group<Real, Real, false>(C, rows, x, xnom, env, 0, M, N, NP, n, g.valid, g.gmask, p0, &iters);
      if (status == MDS_QP_ITER_CAP) {
        __syncwarp(g.gmask);
        if (g.valid) { R4 xv = xnom[n]; x[n] = xv; }
        __syncwarp(g.gmask);
        const int big = qp_solve_group_big<Real>(C.umax[0], C.umax[1], C.umax[2], C.scr, rows, x, xnom, M, N, NP, n, g.valid, g.gmask, p0);
        status = big & 0xff;
        iters += big >> 8;
      }
    }
    if (g.valid) { R4 xv = x[n]; xn[0] = xv.x; xn[1] = xv.y; xn[2] = xv.z; }
  }
  if (g.valid) {
    if (status == MDS_QP_OPTIMAL) {
      usafe[0] = xn[0]; usafe[1] = xn[1]; usafe[2] = xn[2];
      usafe[3] = clamp_(unom[3], lo, hi);
    } else {  // reference falls back to the nominal input (cbf/qptracker.py:30-34)
      usafe[0] = unom[0]; usafe[1] = unom[1]; usafe[2] = unom[2]; usafe[3] = unom[3];
    }
  }
  __syncwarp(g.cmask);  // the env block may be reused by the next step
  *iters_out = iters;
  return status;
}

// ------------------------------------------------------------------ kernels: env step
// NT > 0: drones per env as a compile-time constant (the rollout's specialisation for the 8-drone swarms: partner
// loops unroll, lane maps fold to shifts); NT == 0: run-time N.
template <int NT> MDS_DEV int ct_n(int n_rt) { return NT > 0 ? NT : n_rt; }
template <int NT> MDS_DEV int ct_np(int np_rt) {
  if (NT <= 0) return np_rt;
  int p = 1;
  while (p < NT) p <<= 1;
  return p;
}
template <typename Real> MDS_DEV void store4(Real* p, int d, const Real v[4]) {
  typename Vec4T<Real>::type o;
  o.x = v[0]; o.y = v[1]; o.z = v[2]; o.w = v[3];
  reinterpret_cast<typename Vec4T<Real>::type*>(p)[d] = o;
}
template <typename Real> MDS_DEV void load4(const Real* p, int d, Real v[4]) {
  auto o = reinterpret_cast<const typename Vec4T<Real>::type*>(p)[d];
  v[0] = o.x; v[1] = o.y; v[2] = o.z; v[3] = o.w;
}
// One control period of the env for this lane's drone with the state in registers (every lane of a valid group
// calls it): clips the action, runs the sub-steps, returns the new observation.  R0 (optional): the rotation matrix of the
// attitude the period starts from, when the caller already has it (the inner loop of the controller stack builds it).
// dw0 (optional): the downwash of the first sub-step, when the caller has summed it from the positions the period starts
// from (cbf_filter_group's dw_out); later sub-steps exchange their moved positions.
template <int SPEC, typename Real>
MDS_DEV Obs<Real> physics_core(const DroneP<Real>& P, Drone<Real>& s, const Real action[4], V3<Real> fx, typename Vec4T<Real>::type* env_pos,
                               const GroupMap& g, int N, int NP, const M3<Real>* R0 = nullptr, const Real* dw0 = nullptr) {
  using S = PhysSpec<SPEC>;
  Real rpm[4];
#pragma unroll
  for (int i = 0; i < 4; ++i) rpm[i] = clamp_(action[i], Real(0), P.max_rpm);
  V3<Real> av = {Real(0), Real(0), Real(0)};
  const bool dwash = (S::physics(P) == MDS_PHYSICS_DYN_GND_DRAG_DW) && (N > 1);
  const int substeps = S::substeps(P);
  for (int k = 0; k < substeps; ++k) {
    Real dw = Real(0);
    if (dwash) dw = (dw0 != nullptr && k == 0) ? *dw0 : downwash_group(P, env_pos, s.p, g, N, NP);
    if (g.valid) {
      const M3<Real> R = (R0 != nullptr && k == 0) ? *R0 : quat_to_mat(s.qx, s.qy, s.qz, s.qw);
      av = physics_substep<SPEC>(P, s, rpm, dw, fx, R);
#pragma unroll
      for (int i = 0; i < 4; ++i) s.rpm[i] = rpm[i];
    }
  }
  Obs<Real> o;
  if (g.valid) o = make_obs(s, av);
  return o;
}

// The same through HBM: loads the state and the action, stores the state and (if obs != nullptr) the observation,
// and returns the observation in registers.
template <typename Real>
MDS_DEV Obs<Real> physics_body(const DroneP<Real>& P, const StateP<Real>& st, const Real* __restrict__ action, const Real* __restrict__ fext,
                               Real* __restrict__ obs, typename Vec4T<Real>::type* env_pos, const GroupMap& g, int N, int NP) {
  Drone<Real> s;
  s.p = {Real(0), Real(0), Real(0)};
  Real act[4] = {Real(0), Real(0), Real(0), Real(0)};
  V3<Real> fx = {Real(0), Real(0), Real(0)};
  if (g.valid) {
    s = load_drone(st, g.d);
    load4(action, g.d, act);
    if (fext) fx = {fext[3 * g.d], fext[3 * g.d + 1], fext[3 * g.d + 2]};
  }
  Obs<Real> o = physics_core<0>(P, s, act, fx, env_pos, g, N, NP);
  if (g.valid) {
    store_drone(st, g.d, s);
    if (obs) store_obs(obs, g.d, o);
  }
  return o;
}

template <typename Real, int NT>
__global__ void __launch_bounds__(MDS_BLOCK, sizeof(Real) == 4 ? MDS_PHYS_MINB : 2) physics_step_kernel(DroneP<Real> P, StateP<Real> st, const Real* __restrict__ action,
                                                                  const Real* __restrict__ fext, Real* __restrict__ obs, int E, int N_rt, int NP_rt) {
  __shared__ typename Vec4T<Real>::type sm_pos[MDS_BLOCK];
  const int N = ct_n<NT>(N_rt), NP = ct_np<NT>(NP_rt);
  GroupMap g = group_map(N, NP, E);
  if (!g.env_valid) return;  // whole groups leave together
  full_group_hint<NT>(g);
  physics_body(P, st, action, fext, obs, sm_pos + (threadIdx.x - g.n), g, N, NP);
}

// ------------------------------------------------------------------ kernel: fused K-step rollout
template <typename Real> struct RolloutP {
  int ctrl, use_cbf, n_obs, write_obs_every;
  Real u0_pre, u0_post;
  Real obstacles[MDS_MAX_OBSTACLES * 4];
  const Real* lqr_planes;  // per-drone LQR gains [4*dim][D] (decentralised LQR), or null: the shared gain of LqrP
  int lqr_D;
};

// min / max of doubles by ONE integer atomic each, no compare-and-swap loop (thousands of blocks hit the same two words):
// IEEE doubles of one sign order like their bit patterns -- non-negative ones as signed integers ascending, negative ones as
// unsigned integers descending -- and a negative double is "less than" any non-negative one in the signed view and "greater"
// in the unsigned view.  NaNs never reach these (the statistics are sums / extrema of finite fp32 values).
MDS_DEV void atomic_min_double(double* addr, double v) {
  v += 0.0;  // -0.0 -> +0.0
  if (v >= 0.0) atomicMin(reinterpret_cast<long long*>(addr), __double_as_longlong(v));
  else atomicMax(reinterpret_cast<unsigned long long*>(addr), (unsigned long long)__double_as_longlong(v));
}
MDS_DEV void atomic_max_double(double* addr, double v) {
  v += 0.0;
  if (v >= 0.0) atomicMax(reinterpret_cast<long long*>(addr), __double_as_longlong(v));
  else atomicMin(reinterpret_cast<unsigned long long*>(addr), (unsigned long long)__double_as_longlong(v));
}

// L1 prefetch of the lines a thread will load much later (PID state after the QP, trajectory spec after the
// physics step): the three global-load latencies of a thread then overlap instead of adding up.
MDS_DEV void prefetch_l1(const void* p) { asm volatile("prefetch.global.L1 [%0];" ::"l"(p)); }

// per-lane contributions to the rollout statistics
struct StepStats {
  float err, min_h;
  int qp_solves, qp_iters, qp_infeas, qp_cap;
};

// One control step of the controller stack for this lane's drone (every lane of a valid group calls it):
// reference -> tracking controller -> (CBF-QP) -> inner loop -> RPM action.  CTRL / USE_CBF are compile-time so
// that each instantiation carries only its own stage code (one kernel with run-time switches overflowed the
// instruction cache: 55 % of the stall samples were "no instruction").
// PDK: a gain per drone (Rc.lqr_planes) instead of LqrP's; SPEC: compile-time parameter switches (PhysSpec); R_out (optional)
// receives the rotation matrix of the observation's attitude when the inner loop built it (HAS_PID controllers).
// REFTAB: the reference is read from ref_slot (a slot of rollout_loop_kernel's reference table) instead of evaluated from
// (spec, segs, t), which are then unused.  dw_out (optional, with USE_CBF): receives the downwash of the physics sub-step that
// follows from the observation's positions, summed by the CBF stage (physics_core's dw0).
template <typename Real, int CTRL, bool USE_CBF, bool PDK = false, int SPEC = 0, int NT = 0, bool REFTAB = false>
MDS_DEV void ctrl_body(const DroneP<Real>& P, const RolloutP<Real>& Rc, const GeoP<Real>& G, const LqrP<Real>& L, const CbfP<Real>& C,
                       const DslP<Real>& Dg, const DslStateP<Real>& dst, const CbfSmem<Real>& S, const PidP<Real>& pid,
                       const typename TrajSpecT<Real>::spec& spec,
                       const typename TrajSpecT<Real>::seg* __restrict__ segs, const Obs<Real>& o, const GroupMap& g, int N, int NP,
                       double t, Real rpm[4], StepStats& ss, int pid_idx, M3<Real>* R_out = nullptr,
                       const typename Vec4T<Real>::type* ref_slot = nullptr, Real* dw_out = nullptr) {
  constexpr bool HAS_PID = (CTRL == MDS_CTRL_LQR_OMEGA || CTRL == MDS_CTRL_LQR_YANK);
  constexpr int ORD = CTRL == MDS_CTRL_LQR_OMEGA ? 2 : 3;  // rollout_impl pairs the order-2 filter with LQR_OMEGA, order 3 with LQR_YANK
  Real u[4] = {Real(0), Real(0), Real(0), Real(0)};
  Ref<Real> ref;
  if (g.valid) {
    if constexpr (REFTAB) ref = load_ref<Real>(ref_slot);
    else ref = eval_traj<Real>(spec, segs, t);
    ss.err = (float)norm(o.p - ref.p);
    if (CTRL == MDS_CTRL_GEOMETRIC) {
      geometric_input(P, G, o, ref, u);
      input_to_action<SPEC>(P, u, rpm);
    } else if (CTRL == MDS_CTRL_DSLPID) {
      DslState<Real> ds = load_dsl(dst, g.d);
      V3<Real> pe;
      dslpid_control(P, Dg, ds, o, ref.p, v3(Real(0), Real(0), ref.yaw), ref.v, v3(Real(0), Real(0), ref.yaw_rate), rpm, &pe);
      store_dsl(dst, g.d, ds);
    } else {
      if (PDK) dlqr_input(P, Rc.lqr_planes, (size_t)Rc.lqr_D, (size_t)g.d, CTRL, o, ref, u);
      else lqr_input(P, L, CTRL, o, ref, u);
      if (CTRL == MDS_CTRL_LQR_TORQUE) input_to_action<SPEC>(P, u, rpm);
    }
  }
  if (HAS_PID) {
    if (USE_CBF) {
      CbfAgent<Real> ag;
      ag.p = {Real(0), Real(0), Real(0)}; ag.dv = ag.p; ag.da = ag.p;
      Real F = Real(0), unom[4] = {Real(0), Real(0), Real(0), Real(0)}, usafe[4] = {Real(0), Real(0), Real(0), Real(0)};
      if (g.valid) {
        if (CTRL == MDS_CTRL_LQR_OMEGA) u[0] = cap_thrust(P, u[0]);  // skip_low_level=True returns cap_u(u)
        Real xd[10];
        xd[0] = Real(0); xd[1] = Real(0); xd[2] = ref.yaw;
        if (CTRL == MDS_CTRL_LQR_OMEGA) { xd[3] = ref.v.x; xd[4] = ref.v.y; xd[5] = ref.v.z; }
        else { xd[3] = P.g * P.m; xd[4] = ref.v.x; xd[5] = ref.v.y; xd[6] = ref.v.z; }
        ag = cbf_agent<ORD>(P, C, o, xd, &F);
        unom[0] = u[0] - Rc.u0_pre; unom[1] = u[1]; unom[2] = u[2]; unom[3] = u[3];
      }
      Real mh = Real(1e30);
      int it = 0;
      const bool dwash = (PhysSpec<SPEC>::physics(P) == MDS_PHYSICS_DYN_GND_DRAG_DW) && (N > 1);  // physics_core's condition
      int stt = cbf_filter_group<ORD, Real, NT>(P, C, S, Rc.obstacles, Rc.n_obs, g, N, NP, ag, F, unom, usafe, &mh, &it, dw_out, dwash);
      if (g.valid) {
        ss.min_h = (float)mh;
        if (g.n == 0) {
          ss.qp_solves = (it > 0 || stt != MDS_QP_OPTIMAL);
          ss.qp_iters = it;
          ss.qp_infeas = (stt == MDS_QP_INFEASIBLE);
          ss.qp_cap = (stt == MDS_QP_ITER_CAP);
        }
        u[0] = usafe[0] + Rc.u0_post; u[1] = usafe[1]; u[2] = usafe[2]; u[3] = usafe[3];
      }
    }
    if (g.valid) {
      Pid<Real> ps = load_pid(pid, pid_idx);  // pid_idx: g.d for HBM-resident state, the thread index when the caller staged it
      low_level<SPEC>(P, CTRL, ps, u, o, rpm, R_out);
      store_pid(pid, pid_idx, ps);
    }
  }
}

// Block-wide accumulation of the statistics (called by EVERY thread of the block).
// Per-warp reduction with redux.sync on integer images (counters; non-negative float bits order like unsigned
// ints; the barrier minimum goes through an order-preserving float -> int map) and five float shuffles for the
// error sum, then shared memory and ONE set of atomics per block: same-address atomics from every warp cost
// more than the whole step (1.6 ms vs 0.4 ms per step at 1M drones).
template <bool USE_CBF> MDS_DEV void stats_block_reduce(double* __restrict__ stats, int drone_steps, const StepStats& ss, float max_err) {
  __shared__ float sm_f[MDS_BLOCK / 32][2];
  __shared__ int sm_i[MDS_BLOCK / 32][6];
  const int n_warps = blockDim.x >> 5;
  const unsigned full = 0xffffffffu;
  int mh_i = __float_as_int(ss.min_h);
  mh_i = mh_i >= 0 ? mh_i : (mh_i ^ 0x7fffffff);
  const int w_steps = __reduce_add_sync(full, drone_steps), w_solves = __reduce_add_sync(full, ss.qp_solves);
  const int w_iters = __reduce_add_sync(full, ss.qp_iters), w_inf = __reduce_add_sync(full, ss.qp_infeas), w_cap = __reduce_add_sync(full, ss.qp_cap);
  const unsigned w_maxe = __reduce_max_sync(full, __float_as_uint(max_err));
  const int w_minh = __reduce_min_sync(full, mh_i);
  float w_sum = ss.err;
  for (int off = 16; off > 0; off >>= 1) w_sum += __shfl_xor_sync(full, w_sum, off);
  const int w = threadIdx.x >> 5;
  if ((threadIdx.x & 31) == 0) {
    sm_f[w][0] = w_sum; sm_f[w][1] = __uint_as_float(w_maxe);
    sm_i[w][0] = w_steps; sm_i[w][1] = w_solves; sm_i[w][2] = w_iters; sm_i[w][3] = w_inf; sm_i[w][4] = w_cap; sm_i[w][5] = w_minh;
  }
  __syncthreads();
  if (threadIdx.x < MDS_STAT_COUNT) {
    const int k = threadIdx.x;
    double acc = 0.0;
    if (k == MDS_STAT_SUM_POS_ERR) {
      for (int i = 0; i < n_warps; ++i) acc += (double)sm_f[i][0];
    } else if (k == MDS_STAT_MAX_POS_ERR) {
      for (int i = 0; i < n_warps; ++i) acc = fmax(acc, (double)sm_f[i][1]);
    } else if (k == MDS_STAT_MIN_BARRIER) {
      int m = sm_i[0][5];
      for (int i = 1; i < n_warps; ++i) m = min(m, sm_i[i][5]);
      acc = (double)__int_as_float(m >= 0 ? m : (m ^ 0x7fffffff));
    } else {
      const int col = k == MDS_STAT_DRONE_STEPS ? 0 : (k == MDS_STAT_QP_SOLVES ? 1 : (k == MDS_STAT_QP_ITERS ? 2 : (k == MDS_STAT_QP_INFEASIBLE ? 3 : 4)));
      long long t = 0;
      for (int i = 0; i < n_warps; ++i) t += sm_i[i][col];
      acc = (double)t;
    }
    if (k == MDS_STAT_MAX_POS_ERR) atomic_max_double(&stats[k], acc);
    else if (k == MDS_STAT_MIN_BARRIER) { if (USE_CBF) atomic_min_double(&stats[k], acc); }
    else if (acc != 0.0) atomicAdd(&stats[k], acc);
  }
}

// controller stack alone: obs (HBM) -> action (HBM).
// PERSISTENT: the grid is the resident set (2 blocks per SM; fewer for small swarms) and every block walks the
// block-sized tiles of the environments with stride gridDim.x.  One block per tile at 64 registers (4 resident blocks, 182 KB of
// shared memory, 41 KB of L1 left for 960-byte frames) ran at IPC 1.6, latency-bound on its first loads and its spills, with a
// statistics reduction + block barrier per tile (9 % of the instructions, 20 % of the stall samples).  The same stack inside
// the K-step loop kernel reaches IPC 2.8 with 16 warps at 128 registers -- so this kernel now runs in that configuration,
// prefetches the NEXT tile's observation / trajectory descriptor / PID state into L1 while it works on the current one,
// accumulates its statistics in registers and reduces them once.
#ifndef MDS_CTRL_PERSISTENT
#define MDS_CTRL_PERSISTENT 1
#endif
template <typename Real, int CTRL, bool USE_CBF, int NT>
__global__ void __launch_bounds__(MDS_BLOCK, MDS_CTRL_PERSISTENT ? 2 : (sizeof(Real) == 4 ? MDS_CTRL_MINB : 2))
    ctrl_step_kernel(DroneP<Real> P, RolloutP<Real> Rc, GeoP<Real> G, LqrP<Real> L, CbfP<Real> C,
                     DslP<Real> Dg, DslStateP<Real> dst, PidP<Real> pid, const typename TrajSpecT<Real>::spec* __restrict__ specs,
                     const typename TrajSpecT<Real>::seg* __restrict__ segs,
                     const Real* __restrict__ obs, Real* __restrict__ action,
                     double* __restrict__ stats, double t, int E, int N_rt, int NP_rt) {
  extern __shared__ __align__(32) unsigned char smem_raw[];
  const int N = ct_n<NT>(N_rt), NP = ct_np<NT>(NP_rt);
  CbfSmem<Real> S = cbf_smem_carve<Real>(smem_raw, NP, N, Rc.n_obs);
  constexpr bool HAS_PID = (CTRL == MDS_CTRL_LQR_OMEGA || CTRL == MDS_CTRL_LQR_YANK);
  const int epb = blockDim.x / NP, n_tiles = (E + epb - 1) / epb;
  StepStats acc = {0.f, 1e30f, 0, 0, 0, 0};
  float max_err = 0.f;
  int n_done = 0;
  for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
    GroupMap g = group_map(N, NP, E, tile);
    if (!g.env_valid) continue;  // whole lane groups skip together (only in the last tile)
    full_group_hint<NT>(g);
    Real rpm[4] = {Real(0), Real(0), Real(0), Real(0)};
    Obs<Real> o;
    typename TrajSpecT<Real>::spec spec;
    spec.kind = MDS_TRAJ_WAIT;
    if (g.valid) {  // every global load of this thread is issued here, before the first dependent instruction
      o = load_obs(obs, g.d);
      spec = specs[g.d];
      if (HAS_PID) { prefetch_l1(pid.a + g.d); prefetch_l1(pid.b + g.d); }
      const int e_next = g.e + (int)gridDim.x * epb;  // this lane's environment in the block's next tile
      if (e_next < E) {
        const size_t d_next = (size_t)e_next * N + g.n;
        const char* on = reinterpret_cast<const char*>(obs + d_next * MDS_OBS_DIM);
        prefetch_l1(on); prefetch_l1(on + 16 * sizeof(Real));
        prefetch_l1(specs + d_next); prefetch_l1(reinterpret_cast<const char*>(specs + d_next) + 32);
        if (HAS_PID) { prefetch_l1(pid.a + d_next); prefetch_l1(pid.b + d_next); }
      }
    }
    StepStats ss = {0.f, 1e30f, 0, 0, 0, 0};
    ctrl_body<Real, CTRL, USE_CBF, (NT < 0), 0, NT>(P, Rc, G, L, C, Dg, dst, S, pid, spec, segs, o, g, N, NP, t, rpm, ss, g.d);
    if (g.valid) {
      store4(action, g.d, rpm);
      ++n_done;
      acc.err += ss.err; max_err = fmaxf(max_err, ss.err); acc.min_h = fminf(acc.min_h, ss.min_h);
      acc.qp_solves += ss.qp_solves; acc.qp_iters += ss.qp_iters; acc.qp_infeas += ss.qp_infeas; acc.qp_cap += ss.qp_cap;
    }
  }
  if (stats) stats_block_reduce<USE_CBF>(stats, n_done, acc, max_err);
}

// Reference table of rollout_loop_kernel<..., REFTAB = true>: the references of MDS_REF_STEPS consecutive control steps for
// the NT drones of an environment, slot (j, n) = 3 words at 3 (j NT + n).  A power of two (the step loop picks the row by a
// mask); 32 steps x 8 drones = 12 KB in fp32.
#ifndef MDS_REF_STEPS
#define MDS_REF_STEPS 32
#endif
// Fills rows [0, steps) with the references of steps k0 + j of drones [0, NT) of environment 0 -- of every environment when the
// trajectory set repeats with period NT -- one slot per thread of the block.  The time is formed exactly as the per-drone path
// forms it (t0 + (double)k * dt_ctrl), so the slots hold the same bits as eval_traj there.  Out of line: the fp64 time and
// phase arithmetic stays out of the step loop's instruction stream.
template <typename Real, int NT>
__device__ __noinline__ void build_ref_table(typename Vec4T<Real>::type* tab, const typename TrajSpecT<Real>::spec* __restrict__ specs,
                                             const typename TrajSpecT<Real>::seg* __restrict__ segs, double t0, double dt_ctrl, int k0, int steps) {
  for (int i = threadIdx.x; i < steps * NT; i += blockDim.x) {
    const int j = i / NT, n = i - j * NT;
    const typename TrajSpecT<Real>::spec sp = specs[n];
    store_ref<Real>(tab + 3 * i, eval_traj<Real>(sp, segs, t0 + (double)(k0 + j) * dt_ctrl));
  }
}

// K control steps in ONE launch.  Environments never interact, and everything that couples the drones of an
// environment (downwash, CBF rows, QP) is exchanged inside its lane group, so a group can run its env forward on its
// own: the observation and the body rates stay in registers from step to step, HBM sees the initial load, the log slots
// that are due and the final store.  No launch per step, no grid-wide barrier.
// SPEC: compile-time parameter switches (PhysSpec); K <= 32767 (rollout_impl splits longer runs): the rare-event counters
// share one register.
// REFTAB (fp32, compile-time N, rate-PID controllers; the host selects it when every environment flies the same N references,
// MdsRolloutCfg.traj_period): the block evaluates the references of the next MDS_REF_STEPS steps once into a shared-memory
// table and the lanes read their slot, instead of every lane evaluating its own drone's reference every step (fp64 time and
// phase, sincos, a 48-byte descriptor staged per thread).  The table is refilled every MDS_REF_STEPS steps between two block
// barriers; K <= MDS_REF_STEPS (the swarm workloads' 24-step launches) fills it once, before the loop.
template <typename Real, int CTRL, bool USE_CBF, int NT, int SPEC, bool REFTAB = false>
__global__ void __launch_bounds__(loop_block<Real>(), MDS_LOOP_MINB) rollout_loop_kernel(DroneP<Real> P, RolloutP<Real> Rc, GeoP<Real> G, LqrP<Real> L, CbfP<Real> C,
                                                                  DslP<Real> Dg, DslStateP<Real> dst, StateP<Real> st, PidP<Real> pid,
                                                                  const typename TrajSpecT<Real>::spec* __restrict__ specs,
                                                                  const typename TrajSpecT<Real>::seg* __restrict__ segs,
                                                                  Real* __restrict__ action, const Real* __restrict__ fext, Real* __restrict__ obs,
                                                                  Real* __restrict__ obs_log, double* __restrict__ stats, double t0, double dt_ctrl, int K, int E,
                                                                  int N_rt, int NP_rt) {
  extern __shared__ __align__(32) unsigned char smem_raw[];
  using R4 = typename Vec4T<Real>::type;
  // downwash positions (with the CBF stage only those of the sub-steps after the first: FUSE_DW below): with the CBF stage
  // they live in the head of the environment's CBF block (idle during the physics; the stage's closing group sync orders the
  // reuse), otherwise in a per-block array.  Every KB of shared memory the kernel does not take is L1 for its spill slots
  // (L1 = 228 KB - shared memory in use).
  __shared__ R4 sm_pos[USE_CBF ? 1 : loop_block<Real>()];
  // fp32 stages the per-step read-mostly data (trajectory descriptor, rate-PID state) in shared memory for the launch;
  // fp64 does not: with the CBF stage's 91 KB that would leave one resident block per SM instead of two (0.41 vs 0.31 ms)
  constexpr bool STAGE = sizeof(Real) == 4;
  __shared__ __align__(16) typename TrajSpecT<Real>::spec sm_spec[(STAGE && !REFTAB) ? loop_block<Real>() : 1];
  __shared__ R4 sm_ref[REFTAB ? 3 * MDS_REF_STEPS * NT : 1];
  constexpr bool HAS_PID = (CTRL == MDS_CTRL_LQR_OMEGA || CTRL == MDS_CTRL_LQR_YANK);
  constexpr bool FUSE_DW = USE_CBF && HAS_PID;  // the CBF stage runs (ctrl_body) and sums the downwash of the physics
  __shared__ R4 sm_pid_a[(STAGE && HAS_PID) ? loop_block<Real>() : 1];
  __shared__ typename Vec2T<Real>::type sm_pid_b[(STAGE && HAS_PID) ? loop_block<Real>() : 1];
  const PidP<Real> pid_s = STAGE ? PidP<Real>{sm_pid_a, sm_pid_b} : pid;
  const int N = ct_n<NT>(N_rt), NP = ct_np<NT>(NP_rt);
  CbfSmem<Real> S = cbf_smem_carve<Real>(smem_raw, NP, N, Rc.n_obs);
  GroupMap g = group_map(N, NP, E);
  R4* const env_pos = USE_CBF ? reinterpret_cast<R4*>(S.env0 + (size_t)g.el * S.stride) : sm_pos + (threadIdx.x - g.n);
  StepStats acc = {0.f, 1e30f, 0, 0, 0, 0};  // qp_infeas holds infeasible | iteration-cap << 16
  float max_err = 0.f;
  int steps_done = 0;
  // FULLW (fp32 swarms whose drones fill their lane groups, per-thread state staged in shared memory): every warp that holds
  // a live environment runs with all 32 lanes -- the lane groups past the last environment re-run environment E - 1 without
  // storing anything -- so the synchronising calls at the stage boundaries take the constant full-warp mask.  A group mask
  // only known at run time costs a MATCH.ANY / REDUX / VOTE / BRA.DIV preamble per call (8 calls per step).
#ifndef MDS_NO_FULLW
  constexpr bool FULLW = STAGE && HAS_PID && NT > 1 && NT < 32 && (NT & (NT - 1)) == 0;
#else
  constexpr bool FULLW = false;
#endif
  static_assert(!REFTAB || (FULLW && NT * MDS_REF_STEPS <= 8 * 32 && (MDS_REF_STEPS & (MDS_REF_STEPS - 1)) == 0),
                "the reference table needs the full-warp instantiation and at most 12 KB of shared memory");
  const bool live = g.env_valid;
  if (FULLW) {
    const int first_env = g.e - (int)((threadIdx.x & 31) / NP);  // lane group 0 of this warp
    // REFTAB: warps past the last environment re-run it too, so that every warp of the block reaches the table's barriers
    g.env_valid = REFTAB || first_env < E;
    if (g.env_valid && !live) { g.e = E - 1; g.d = g.e * N + g.n; }
    g.cmask = 0xffffffffu;
  }
  if (g.env_valid) {
    full_group_hint<NT>(g);
    Obs<Real> o;
    V3<Real> wb = {Real(0), Real(0), Real(0)};  // body rates: the one part of the state the observation does not carry
    // The trajectory descriptor is read every step; its address escapes into the out-of-line table walk, so as an
    // automatic it would live in local memory (LDL, L1-missing under this kernel's local footprint): stage it in
    // shared memory instead (12-word lane stride: 128-bit reads are conflict-free per quarter warp).
    typename TrajSpecT<Real>::spec spec_reg;
    typename TrajSpecT<Real>::spec& spec = (STAGE && !REFTAB) ? sm_spec[threadIdx.x] : spec_reg;
    spec.kind = MDS_TRAJ_WAIT;
    V3<Real> fx_reg = {Real(0), Real(0), Real(0)};  // constant world-frame force on this drone (wind), if any
    const bool has_fx = fext != nullptr;
    if (g.valid) {
      o = load_obs(obs, g.d);
      if (!REFTAB) spec = specs[g.d];
      wb = {st.pos_wx[g.d].w, st.vel_wy[g.d].w, st.wz[g.d]};
      if (has_fx && !STAGE) fx_reg = {fext[3 * g.d], fext[3 * g.d + 1], fext[3 * g.d + 2]};
      if (STAGE && HAS_PID) { sm_pid_a[threadIdx.x] = pid.a[g.d]; sm_pid_b[threadIdx.x] = pid.b[g.d]; }
    }
    if constexpr (REFTAB) {
      build_ref_table<Real, NT>(sm_ref, specs, segs, t0, dt_ctrl, 0, min(K, MDS_REF_STEPS));
      __syncthreads();
    }
    Real rpm[4] = {Real(0), Real(0), Real(0), Real(0)};
    const size_t obs_elems = (size_t)E * N * MDS_OBS_DIM;
    int log_countdown = Rc.write_obs_every;  // steps until the next log slot is due (no division in the loop)
    Real* log_slot = obs_log;
    for (int k = 0; k < K; ++k) {
      const int row = k & (MDS_REF_STEPS - 1);
      if constexpr (REFTAB) {
        if (k > 0 && row == 0) {  // every lane has read the table's last row
          __syncthreads();
          build_ref_table<Real, NT>(sm_ref, specs, segs, t0, dt_ctrl, k, min(K - k, MDS_REF_STEPS));
          __syncthreads();
        }
      }
      StepStats ss = {0.f, 1e30f, 0, 0, 0, 0};
      M3<Real> R;
      Real dw = Real(0);  // with the CBF stage: the downwash of the step's first physics sub-step, summed by the stage
      ctrl_body<Real, CTRL, USE_CBF, (NT < 0), SPEC, NT, REFTAB>(P, Rc, G, L, C, Dg, dst, S, pid_s, spec, segs, o, g, N, NP, t0 + (double)k * dt_ctrl,
                                                             rpm, ss, STAGE ? (int)threadIdx.x : g.d, HAS_PID ? &R : nullptr,  // the host plans form t exactly like this
                                                             REFTAB ? sm_ref + 3 * (row * NT + g.n) : nullptr, FUSE_DW ? &dw : nullptr);
      acc.err += ss.err; max_err = fmaxf(max_err, ss.err); acc.min_h = fminf(acc.min_h, ss.min_h);
      acc.qp_solves += ss.qp_solves; acc.qp_iters += ss.qp_iters; acc.qp_infeas += ss.qp_infeas + (ss.qp_cap << 16);
      Drone<Real> s;
      s.p = o.p; s.qx = o.qx; s.qy = o.qy; s.qz = o.qz; s.qw = o.qw; s.v = o.v; s.w = wb;
#pragma unroll
      for (int i = 0; i < 4; ++i) s.rpm[i] = o.rpm[i];
      V3<Real> fx = fx_reg;
      if (STAGE) {  // fp32 is short of registers: the wind (rarely set) is re-read every step, 12 B per drone from L1
        fx = {Real(0), Real(0), Real(0)};
        if (has_fx && g.valid) fx = {__ldg(fext + 3 * g.d), __ldg(fext + 3 * g.d + 1), __ldg(fext + 3 * g.d + 2)};
      }
      o = physics_core<SPEC>(P, s, rpm, fx, env_pos, g, N, NP, HAS_PID ? &R : nullptr, FUSE_DW ? &dw : nullptr);
      wb = s.w;
      if (Rc.write_obs_every > 0 && --log_countdown == 0) {
        if (g.valid && live) store_obs(log_slot, g.d, o, true);  // streaming stores: the log is write-once
        log_slot += obs_elems;
        log_countdown = Rc.write_obs_every;
      }
    }
    if (g.valid && live) {
      Drone<Real> s;
      s.p = o.p; s.qx = o.qx; s.qy = o.qy; s.qz = o.qz; s.qw = o.qw; s.v = o.v; s.w = wb;
#pragma unroll
      for (int i = 0; i < 4; ++i) s.rpm[i] = o.rpm[i];
      store_drone(st, g.d, s);
      store_obs(obs, g.d, o);
      store4(action, g.d, rpm);
      if (STAGE && HAS_PID) { pid.a[g.d] = sm_pid_a[threadIdx.x]; pid.b[g.d] = sm_pid_b[threadIdx.x]; }
      steps_done = K;
    }
  }
  if (FULLW && !live) { acc = {0.f, 1e30f, 0, 0, 0, 0}; max_err = 0.f; }  // a re-run environment counts nowhere
  acc.qp_cap = acc.qp_infeas >> 16;
  acc.qp_infeas &= 0xffff;
  if (stats) stats_block_reduce<USE_CBF>(stats, steps_done, acc, max_err);
}
