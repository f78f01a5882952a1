// mds_traj.cuh -- closed-form reference generators evaluated on device.
// Replaces the reference's trajectories/*.py (Circle.py:24-45, Lemniscate.py:32-63,
// LineTrajectory.py:4-14,69-103, CompoundTrajectory.py:26-40, RotateTrajectory.py:19-24).
// The phase (angle) is formed in double and range-reduced before the Real sincos so
// that fp32 rollouts do not lose the reference's fp64 time accumulation.
#pragma once
#include "mds_common.cuh"

namespace mds {

template <typename Real> struct TrajSpecT;
template <> struct TrajSpecT<float> { using spec = MdsTrajSpecF32; using seg = MdsTrajSegF32; };
template <> struct TrajSpecT<double> { using spec = MdsTrajSpecF64; using seg = MdsTrajSegF64; };

template <typename Real> struct Ref {
  V3<Real> p, v, a;
  Real yaw, yaw_rate;
};

MDS_DEV double reduce_2pi(double th) {
  const double two_pi = 6.283185307179586476925286766559, inv_two_pi = 0.15915494309189533576888376337251;
  return th - two_pi * floor(th * inv_two_pi);  // multiply: the fp64 divide is a ~40-instruction subroutine
}

// Circle.py:24-45.  p = {r, v, cx, cy, cz, yaw_rate}.  Quirk B18: yaw in [pi, 3pi).
template <typename Real> MDS_DEV Ref<Real> eval_circle(const Real* p, double t) {
  const double pi = 3.14159265358979323846, two_pi = 2.0 * pi;
  Real r = p[0], v = p[1];
  double wt = (double)v / (double)r * t;
  Real s, c;
  sincos_(Real(reduce_2pi(wt)), &s, &c);
  Real cen = v * v / r;
  Ref<Real> o;
  o.p = {p[2] + r * c, p[3] + r * s, p[4]};
  o.v = {-v * s, v * c, Real(0)};
  o.a = {-cen * c, -cen * s, Real(0)};
  double y = (double)p[5] * t - pi;
  o.yaw = Real(y - two_pi * floor(y / two_pi) + pi);
  o.yaw_rate = p[5];
  return o;
}

// Lemniscate.py:32-63.  p = {a, omega, cx, cy, cz, yaw_rate, phase_shift}.
template <typename Real> MDS_DEV Ref<Real> eval_lemniscate(const Real* p, double t) {
  const Real pi = Real(3.14159265358979323846);
  Real a = p[0], om = p[1];
  double th = reduce_2pi(t * (double)om + (double)p[6]);
  Real s, c;
  sincos_(Real(th), &s, &c);
  Real s2 = s * s, c2 = c * c;
  Real cos2 = c2 - s2, sin2 = Real(2) * s * c;          // cos 2th, sin 2th
  Real cos4 = Real(2) * cos2 * cos2 - Real(1);         // cos 4th
  Real den = Real(1) + s2, inv = rcp_(den), inv2 = inv * inv;
  Real k3 = cos2 - Real(3);
  Real ik3 = rcp_(k3 * k3 * k3);
  Ref<Real> o;
  o.p = {p[2] + a * s * c * inv, p[3] + a * c * inv, p[4]};
  o.v = {-a * om * (s2 * s2 + s2 + (s2 - Real(1)) * c2) * inv2, -a * om * s * (s2 + Real(2) * c2 + Real(1)) * inv2, Real(0)};
  o.a = {Real(4) * a * om * om * sin2 * (Real(3) * cos2 + Real(7)) * ik3,
         a * om * om * c * (Real(44) * cos2 + cos4 - Real(21)) * ik3, Real(0)};
  if (p[5] == Real(0)) {            // no yaw motion (the reference's mains): sin(0) = 0, cos(0) = 1 without the sincos
    o.yaw = Real(0);
    o.yaw_rate = Real(0);
    return o;
  }
  Real sy, cy;
  sincos_(Real(reduce_2pi((double)p[5] * t)), &sy, &cy);
  o.yaw = pi * sy;                  // quirk B19
  o.yaw_rate = pi * p[5] * cy;
  return o;
}

// LineTrajectory.py:4-14.  p = {x, y, z, yaw}
template <typename Real> MDS_DEV Ref<Real> eval_wait(const Real* p) {
  Ref<Real> o;
  o.p = {p[0], p[1], p[2]};
  o.v = {Real(0), Real(0), Real(0)};
  o.a = o.v;
  o.yaw = p[3];
  o.yaw_rate = Real(0);
  return o;
}

// LineTrajectory.py:69-103 (trapezoid, per-axis sign() acceleration -- quirk B20).
// p = start3, v0 3, sgn_init3, cruise3, sgn_end3, end3, vf3, time_init, time_middle, total_time
template <typename Real> MDS_DEV Ref<Real> eval_line(const Real* p, Real t) {
  const Real a_max = Real(1);
  V3<Real> start = {p[0], p[1], p[2]}, v0 = {p[3], p[4], p[5]}, sgi = {p[6], p[7], p[8]};
  V3<Real> cruise = {p[9], p[10], p[11]}, sge = {p[12], p[13], p[14]};
  Real t_init = p[21], t_mid = p[22], t_tot = p[23];
  Ref<Real> o;
  o.yaw = Real(0);
  o.yaw_rate = Real(0);
  if (t > t_tot) {
    o.p = {p[15], p[16], p[17]};
    o.v = {p[18], p[19], p[20]};
    o.a = {Real(0), Real(0), Real(0)};
    return o;
  }
  if (t < t_init) {
    o.p = start + t * v0 + (Real(0.5) * a_max * t * t) * sgi;
    o.v = v0 + (a_max * t) * sgi;
    o.a = a_max * sgi;
    return o;
  }
  V3<Real> d_init = t_init * v0 + (Real(0.5) * a_max * t_init * t_init) * sgi;
  if (t < t_mid + t_init) {
    Real tau = t - t_init;
    o.p = start + d_init + tau * cruise;
    o.v = cruise;
    o.a = {Real(0), Real(0), Real(0)};
    return o;
  }
  Real tau = t - t_mid - t_init;
  V3<Real> d_mid = d_init + t_mid * cruise;
  o.p = start + d_mid + tau * cruise + (Real(0.5) * a_max * tau * tau) * sge;
  o.v = cruise + (a_max * tau) * sge;
  o.a = a_max * sge;
  return o;
}

template <typename Real, typename Seg> MDS_DEV Ref<Real> eval_segment(const Seg& sg, double t_local) {
  Ref<Real> o;
  switch (sg.kind) {
    case MDS_SEG_CIRCLE: o = eval_circle<Real>(sg.p, t_local); break;
    case MDS_SEG_LEMNISCATE: o = eval_lemniscate<Real>(sg.p, t_local); break;
    case MDS_SEG_LINE: o = eval_line<Real>(sg.p, Real(t_local)); break;
    default: o = eval_wait<Real>(sg.p); break;
  }
  if (sg.has_rot) {  // RotateTrajectory.py:19-24: rot = R (9, row-major) + centre (3)
    M3<Real> R;
#pragma unroll
    for (int i = 0; i < 9; ++i) R.m[i] = sg.rot[i];
    V3<Real> c = {sg.rot[9], sg.rot[10], sg.rot[11]};
    o.p = mul(R, o.p - c) + c;
    o.v = mul(R, o.v);
    o.a = mul(R, o.a);
  }
  return o;
}

// Stateless equivalent of CompoundTrajectory.__call__ for a forward-running clock:
// segment = first k with t <= t_end[k]; past the end -> last segment at its own end.
// Out of line: the closed-form generators are the hot path of the swarm workloads, and keeping the segment-table
// walk (and the Line / Rotate code it pulls in) out of the callers' instruction stream keeps their hot loop compact.
template <typename Real>
__device__ __noinline__ Ref<Real> eval_traj_table(const typename TrajSpecT<Real>::spec& sp, const typename TrajSpecT<Real>::seg* __restrict__ segs, double t) {
  int b = sp.seg_begin, n = sp.seg_count;
  if (sp.pad) return eval_segment<Real>(segs[b], t);  // stand-alone generator: no compound end clamp
  double total = (double)segs[b + n - 1].t_end;
  if (t >= total) return eval_segment<Real>(segs[b + n - 1], (double)segs[b + n - 1].dur);
  int k = 0;
  double t0 = 0.0;
  while (k < n - 1 && t > (double)segs[b + k].t_end) {
    t0 = (double)segs[b + k].t_end;
    ++k;
  }
  return eval_segment<Real>(segs[b + k], t - t0);
}

template <typename Real>
MDS_DEV Ref<Real> eval_traj(const typename TrajSpecT<Real>::spec& sp, const typename TrajSpecT<Real>::seg* __restrict__ segs, double t) {
  switch (sp.kind) {
    case MDS_TRAJ_CIRCLE: return eval_circle<Real>(sp.p, t);
    case MDS_TRAJ_LEMNISCATE: return eval_lemniscate<Real>(sp.p, t);
    case MDS_TRAJ_WAIT: return eval_wait<Real>(sp.p);
    default: break;
  }
  // the out-of-line walk gets its OWN copy: passing `sp` itself would let its address escape and pin the caller's
  // descriptor (read by every closed-form generator above) in local memory
  const typename TrajSpecT<Real>::spec table_spec = sp;
  return eval_traj_table<Real>(table_spec, segs, t);
}

// A reference sample in three 128-bit words (11 Reals + 1 pad): (p, v.x) (v.y, v.z, a.x, a.y) (a.z, yaw, yaw_rate, -)
template <typename Real> MDS_DEV void store_ref(typename Vec4T<Real>::type* w, const Ref<Real>& r) {
  typename Vec4T<Real>::type w0, w1, w2;
  w0.x = r.p.x; w0.y = r.p.y; w0.z = r.p.z; w0.w = r.v.x;
  w1.x = r.v.y; w1.y = r.v.z; w1.z = r.a.x; w1.w = r.a.y;
  w2.x = r.a.z; w2.y = r.yaw; w2.z = r.yaw_rate; w2.w = Real(0);
  w[0] = w0; w[1] = w1; w[2] = w2;
}
template <typename Real> MDS_DEV Ref<Real> load_ref(const typename Vec4T<Real>::type* w) {
  const typename Vec4T<Real>::type w0 = w[0], w1 = w[1], w2 = w[2];
  Ref<Real> r;
  r.p = {w0.x, w0.y, w0.z}; r.v = {w0.w, w1.x, w1.y}; r.a = {w1.z, w1.w, w2.x};
  r.yaw = w2.y; r.yaw_rate = w2.z;
  return r;
}

}  // namespace mds
