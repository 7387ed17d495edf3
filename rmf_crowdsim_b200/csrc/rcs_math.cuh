// rcs_math.cuh -- per-pair arithmetic of the hot path, written so that every +,-,*,/,sqrt is the
// same IEEE-754 double operation, in the same order, as the reference's Rust (rustc never
// contracts a*b+c into an FMA).  This translation unit MUST be compiled with --fmad=false.
//
// Reference file:line citations are relative to /root/reference/rmf_crowdsim/src.
#pragma once

#include <cstdint>
#include <cuda_runtime.h>

namespace rcs {

#define RCS_INF (__longlong_as_double(0x7ff0000000000000LL))

enum : uint32_t { LP_NONE = 0, LP_ZANLUNGO = 1 };
// HL_ROUTE_TABLE is a host-side kind only: its groups run as HL_ROUTE (a route planner is a table of one leg).
enum : uint32_t { HL_NONE = 0, HL_CONSTANT = 1, HL_PARITY = 2, HL_HOST = 3, HL_ROUTE = 4, HL_ROUTE_TABLE = 5 };

// LocationHash2D geometry (location_hash_2d.rs:14-23, 33-51) in device form.
struct GridDev {
  double offx, offy, res;
  uint64_t nx;    // (width / resolution) as usize -- the stride used by BOTH index formulas (:59, :79)
  uint64_t len;   // data.len() = nx * ny
  int64_t x_max;  // largest x_idx that can still give idx < len for some y >= 0; -1 if len == 0
  double inv_res; // 1 / res, only ever used to PREDICT a quotient (see div_floor)
};

// floor(fl(num / res)) -- the floor of the correctly rounded IEEE quotient the reference computes
// (location_hash_2d.rs:56-57, 69-70) -- without a division in the common case.  q1 = fl(num * fl(1/res)) is within
// 2 ulp of the true quotient and the IEEE quotient within 0.5 ulp, so when q1 is further than 8 ulp from every
// integer all three have the same floor.  Otherwise (q1 next to an integer, huge, NaN) the true division decides.
__device__ __forceinline__ double div_floor(double num, const GridDev& g) {
  const double q1 = num * g.inv_res;
  const double f = floor(q1);
  const double d = q1 - f;                              // [0, 1): exact (Sterbenz) or q1 is huge and d == 0
  const double tol = fabs(q1) * 1.8e-15 + 1e-300;       // 8 ulp
  if (d > tol && (1.0 - d) > tol) return f;
  return floor(num / g.res);
}

// One add_agents group = (high-level planner, local planner, eyesight) (lib.rs:119-125).
struct GroupDev {
  double eyesight;  // Agent::eyesight_range (lib.rs:64,143)
  double thr2;      // smallest double T with sqrt(T) >= eyesight: sqrt(d2) < R  <=>  d2 < T
  double hl_vx, hl_vy;
  // Zanlungo::new arguments that are ever read (zanlungo.rs:31-48) and host-precomputed terms
  double agent_scale;
  double force_distance;
  double inv_mass;  // 1f64 / agent_mass            (zanlungo.rs:216)
  double rr;        // agent_radius * agent_radius  (zanlungo.rs:52)
  double two_r;     // agent_radius * 2f64          (zanlungo.rs:161)
  double inv_fd;    // 1 / force_distance: yield fast path only (the literal routine divides)
  uint32_t lp_kind;
  uint32_t hl_kind;
  uint32_t w0_fast;      // 1: a weight-0 pair can only contribute +-0 or NaN (see pair_force_w0_is_zero)
  int32_t source_sink;   // index into the source-sink table, -1 if none
  uint32_t route_off, route_n;  // HL_ROUTE: the planner's table in the route array (points, not doubles)
};

// Rust `f64 as usize` (saturating, NaN -> 0), location_hash_2d.rs:56-57.
__device__ __forceinline__ uint64_t f64_as_usize(double v) {
  if (!(v > 0.0)) return 0ull;
  if (v >= 18446744073709551616.0) return ~0ull;
  return __double2ull_rz(v);
}
// Rust `f64.floor() as i64` (saturating, NaN -> 0), location_hash_2d.rs:69-70.
__device__ __forceinline__ int64_t f64_floor_as_i64(double v) {
  v = floor(v);
  if (v != v) return 0ll;
  if (v >= 9223372036854775808.0) return 0x7fffffffffffffffLL;
  if (v <= -9223372036854775808.0) return (int64_t)0x8000000000000000ULL;
  return __double2ll_rz(v);
}

// LocationHash2D::location_to_index (location_hash_2d.rs:54-66): insert cell.  Returns false when
// the reference returns Err("Index out of bounds").
__device__ __forceinline__ bool location_to_index(const GridDev& g, double px, double py, uint64_t& idx) {
  // trunc toward zero == floor for the positive quotients; everything <= 0 (and NaN) saturates to 0 either way
  uint64_t x_idx = f64_as_usize(div_floor(px - g.offx, g));
  uint64_t y_idx = f64_as_usize(div_floor(py - g.offy, g));
  idx = x_idx * g.nx + y_idx;  // wrapping, as release-mode Rust
  return idx < g.len;
}

// LocationHash2D::get_bounds (location_hash_2d.rs:103-122): query cell bounds (floor, not trunc).
__device__ __forceinline__ void get_bounds(const GridDev& g, double radius, double px, double py, int64_t& left,
                                           int64_t& right, int64_t& bottom, int64_t& top) {
  right = f64_floor_as_i64(div_floor((px + radius) - g.offx, g));
  left = f64_floor_as_i64(div_floor((px - radius) - g.offx, g));
  top = f64_floor_as_i64(div_floor((py + radius) - g.offy, g));
  bottom = f64_floor_as_i64(div_floor((py - radius) - g.offy, g));
}

// For column x of the scan `for x in left..=right { for y in bottom..=top }` (location_hash_2d.rs:245-246)
// the valid data cells (signed_idx_to_data_idx, :74-85) are one contiguous index range because the index
// is x-major.  Returns false if the column contributes nothing.
__device__ __forceinline__ bool column_cell_range(const GridDev& g, int64_t x, int64_t bottom, int64_t top,
                                                  uint64_t& c_lo, uint64_t& c_hi) {
  if (x < 0 || top < 0 || g.len == 0) return false;
  int64_t ylo = bottom < 0 ? 0 : bottom;
  if (ylo > top) return false;
  uint64_t base = (uint64_t)x * g.nx;
  if (base >= g.len) return false;
  c_lo = base + (uint64_t)ylo;
  if (c_lo >= g.len) return false;
  // base + top can only exceed len-1, never wrap, for x <= x_max
  uint64_t room = g.len - 1 - base;
  c_hi = ((uint64_t)top > room) ? g.len - 1 : base + (uint64_t)top;
  return true;
}

// Zanlungo::time_to_collision (zanlungo.rs:49-74) with rel_vel = (rvx, rvy), rel_pos = (rpx, rpy),
// rp2 = rel_pos.norm_squared() (already computed by the radius filter from the same dx, dy).
// Early exits are exact (DESIGN.md section 4.4); everything else is literal, including the division by 2a == +0.
//  * a == 0 and fl(b*b) == 0 => INF (a NaN a or b*b goes on: the discriminant or both roots are NaN, INF).
//    With a == 0 and fl(b*b) == 0,
//    disc = 0 - (0*c) is +-0 (or NaN for a non-finite c), so both numerators are -b and both roots are
//    -b/+0 of one sign (or NaN): -inf fails every test, +inf is returned as the last root, i.e. INF.
//    a == 0 ALONE is not an exit: a relative speed below ~1.5e-162 underflows a to 0 while fl(b*b) can be a
//    non-zero subnormal whose square root exceeds |b|; the reference then divides by +0, gets t0 = -inf,
//    t1 = +inf and returns 0.
//  * numerator of the larger root <= 0 => INF.  For a > 0 both roots are <= 0 (n0 <= n1).  For a == 0,
//    t1 = n1 / +0 is -inf or NaN and t0 = n0 / +0 with n0 <= n1 <= 0 as well: no root is > 0.
__device__ __forceinline__ double time_to_collision(double rvx, double rvy, double rpx, double rpy, double rp2,
                                                    double rr) {
  double a = rvx * rvx + rvy * rvy;
  double b = 2.0 * (rvx * rpx + rvy * rpy);
  double bb = b * b;
  if ((__double_as_longlong(a) | __double_as_longlong(bb)) == 0ll) return RCS_INF;  // both +0 (squares: never -0)
  double c = rp2 - rr;
  double discriminant = bb - (4.0 * a) * c;
  if (discriminant < 0.0) return RCS_INF;
  double sq = sqrt(discriminant);
  double n1 = -b + sq;
  if (n1 <= 0.0) return RCS_INF;
  double den = 2.0 * a;
  double t0 = (-b - sq) / den;
  double t1 = n1 / den;
  if ((t0 < 0.0 && t1 > 0.0) || (t1 < 0.0 && t0 > 0.0)) return 0.0;
  if (t0 < t1 && t0 > 0.0) return t0;
  if (t1 > 0.0) return t1;
  return RCS_INF;
}

// right_of_way = (self_priority - other_priority).clamp(-1, 1) with priority = id as f64
// (zanlungo.rs:94, 183-185).  Returns -1, 0 or +1 as a double (NaN impossible for integer ids).
__device__ __forceinline__ double right_of_way(uint64_t self_id, uint64_t other_id) {
  double d = (double)self_id - (double)other_id;  // u64 -> f64 round-to-nearest, as Rust `as f64`
  if (d < -1.0) d = -1.0;
  if (d > 1.0) d = 1.0;
  return d;
}

struct PairIn {
  double px, py, vx, vy, pfx, pfy;  // current agent: position, velocity, preferred_vel (lib.rs:271)
  double ox, oy, ovx, ovy;          // other agent; its preferred_vel is always (0,0) (lib.rs:57,285)
  uint64_t id, oid;
};

// Zanlungo::compute_agent_force (zanlungo.rs:93-170) including right_of_way_vel (:173-198) and
// slerp (:23-28), literal.  other.preferred_vel = (0,0) is substituted as the constant it is.
__device__ __noinline__ void pair_force_literal(const PairIn& p, double t_i, const GroupDev& z, double& fx,
                                                double& fy) {
  const double opfx = 0.0, opfy = 0.0;
  double row = right_of_way(p.id, p.oid);
  double w, mvx, mvy, ovx, ovy;
  if (row < 0.0) {
    double r_2 = sqrt(-row);
    mvx = p.vx;
    mvy = p.vy;
    ovx = p.ovx + r_2 * (opfx - p.ovx);
    ovy = p.ovy + r_2 * (opfy - p.ovy);
    w = -r_2;
  } else if (row > 0.0) {
    double r_2 = sqrt(row);
    mvx = p.vx + r_2 * (p.pfx - p.vx);
    mvy = p.vy + r_2 * (p.pfy - p.vy);
    ovx = p.ovx;
    ovy = p.ovy;
    w = r_2;
  } else {
    mvx = p.vx;
    mvy = p.vy;
    ovx = p.ovx;
    ovy = p.ovy;
    w = 0.0;
  }
  double weight = 1.0 - w;
  double futx = p.px + mvx * t_i, futy = p.py + mvy * t_i;
  double ofx = p.ox + ovx * t_i, ofy = p.oy + ovy * t_i;
  double dx = futx - ofx, dy = futy - ofy;
  double dist = sqrt(dx * dx + dy * dy);
  if (weight > 1.0) {
    double pref_speed = sqrt(opfx * opfx + opfy * opfy);
    bool interpolate = true;
    double perpx = 0.0, perpy = 0.0;
    if (pref_speed < 0.0001) {
      double crx = p.px - p.ox, cry = p.py - p.oy;
      perpx = -cry;
      perpy = crx;
      if (perpx * p.vx + perpy * p.vy < 0.0) {
        perpx = -perpx;
        perpy = -perpy;
      }
    } else {  // dead code while neighbours' preferred_vel is (0,0); kept for fidelity (:126-139)
      if (opfx * dx + opfy * dy > 0.0) {
        perpx = -opfy;
        perpy = opfx;
        if (perpx * dx + perpy * dy < 0.0) {
          perpx = -perpx;
          perpy = -perpy;
        }
      } else {
        interpolate = false;
      }
    }
    if (interpolate) {
      double sin_theta = perpx * dy - perpy * dx;
      if (sin_theta < 0.0) sin_theta = -sin_theta;
      if (sin_theta > 1.0) sin_theta = 1.0;
      double t = weight - 1.0;
      double theta = asin(sin_theta);
      double s0 = sin((1.0 - t) * theta) / sin_theta;
      double s1 = sin(t * theta) / sin_theta;
      double ndx = dx * s0 + perpx * s1;
      double ndy = dy * s0 + perpy * s1;
      dx = ndx;
      dy = ndy;
    }
  }
  // zanlungo.rs:155-157: `dist > (fut_pos - other_future_pos).norm()` compares a value with itself.
  double nrm = sqrt(dx * dx + dy * dy);
  double nx = dx / nrm, ny = dy / nrm;
  double surface_dist = dist - z.two_r;
  double rvx = mvx - ovx, rvy = mvy - ovy;
  double magnitude = ((weight * z.agent_scale) * sqrt(rvx * rvx + rvy * rvy)) / t_i;
  if (magnitude >= 1e15) magnitude = 1e15;
  double s = magnitude * exp(-surface_dist / z.force_distance);
  fx = nx * s;
  fy = ny * s;
}

// Per-owner terms of compute_agent_force that do not depend on the neighbour, hoisted out of the pair
// loop.  Each is computed by the same operations the literal code applies per pair, so the hoisting
// is bit-neutral:
//   yield case (row < 0): my_vel = v (zanlungo.rs:188);  fut = p + v*t_i (:109);  with a finite
//     neighbour velocity other_vel = ov + 1*((0,0) - ov) is exactly (+0,+0), hence my_vel - other_vel = v
//     and magnitude = (2*agent_scale)*|v| / t_i, capped at 1e15 (:163-167), is the same for every pair;
//   weight-0 case (row > 0): my_vel = v + 1*(pref - v) (:193);  fut0 = p + my_vel*t_i.
struct OwnerPre {
  double futx, futy;  // p + v * t_i
  double mag;         // capped magnitude of the yield case when the neighbour velocity is finite
  double mvx, mvy;    // my_vel of the weight-0 case
  double f0x, f0y;    // p + my_vel(w0) * t_i
};

__device__ __forceinline__ OwnerPre owner_precompute(double px, double py, double vx, double vy, double pfx,
                                                     double pfy, double t_i, const GroupDev& z) {
  OwnerPre o;
  o.futx = px + vx * t_i;
  o.futy = py + vy * t_i;
  double magnitude = ((2.0 * z.agent_scale) * sqrt(vx * vx + vy * vy)) / t_i;
  if (magnitude >= 1e15) magnitude = 1e15;
  o.mag = magnitude;
  o.mvx = vx + 1.0 * (pfx - vx);
  o.mvy = vy + 1.0 * (pfy - vy);
  o.f0x = px + o.mvx * t_i;
  o.f0y = py + o.mvy * t_i;
  return o;
}

// A pair in which the current agent has the higher id gets weight = 1 - 1 = 0 (zanlungo.rs:108,
// 191-194).  Its contribution is d_hat * ((0*scale*|dv|/t_i) * exp(..)).  With z.w0_fast (host
// checked: agent_scale finite, exp argument bounded) this is exactly (+-0, +-0) -- a no-op for
// the accumulator, which starts at +0 -- unless t_i == 0, |dv|^2 is not finite, or d_ij has zero /
// non-finite length; in those cases it is NaN or +-0 per component.  Returns true when the pair is
// provably such a no-op.
__device__ __forceinline__ bool pair_force_w0_is_zero(const OwnerPre& o, double ox, double oy, double ovx,
                                                      double ovy, double t_i) {
  double dx = o.f0x - (ox + ovx * t_i);
  double dy = o.f0y - (oy + ovy * t_i);
  double dd = dx * dx + dy * dy;
  double rvx = o.mvx - ovx, rvy = o.mvy - ovy;
  double rv2 = rvx * rvx + rvy * rvy;
  return (t_i > 0.0) && (dd > 0.0) && (dd < RCS_INF) && (rv2 < RCS_INF);
}

// Hot-path specialisation of pair_force_literal for row < 0 (current agent has the LOWER id and
// yields: weight = 2, slerp parameter t = 1).  Same operations in the same order as the literal code
// except for the two documented substitutions:
//  (1) per-owner terms come from OwnerPre (bit-neutral, see above);
//  (2) the slerp weights sin((1-t)*theta)/sin_theta and sin(t*theta)/sin_theta with t = 1,
//      theta = asin(sin_theta), sin_theta in [0,1] are replaced by their exact values 0 and 1 for
//      sin_theta > 0 and NaN otherwise (0/0, NaN).  The literal evaluation through libm returns
//      1 +- 2 ulp for the second weight, so this differs from the reference by <= 4e-16 relative --
//      inside the 1e-9 force tolerance, and CUDA's sin/asin would not have matched glibc's last bit
//      anyway.  It removes asin, sin and two divisions from every evaluated pair.
__device__ __forceinline__ void pair_force_yield(const OwnerPre& o, double px, double py, double vx, double vy,
                                                 double ox, double oy, double n_vx, double n_vy, double t_i,
                                                 const GroupDev& z, double& fx, double& fy) {
  double ovx = n_vx + 1.0 * (0.0 - n_vx);
  double ovy = n_vy + 1.0 * (0.0 - n_vy);
  double ofx = ox + ovx * t_i, ofy = oy + ovy * t_i;
  double dx = o.futx - ofx, dy = o.futy - ofy;
  double dist = sqrt(dx * dx + dy * dy);
  double crx = px - ox, cry = py - oy;
  double perpx = -cry, perpy = crx;
  if (perpx * vx + perpy * vy < 0.0) {
    perpx = -perpx;
    perpy = -perpy;
  }
  double sin_theta = perpx * dy - perpy * dx;
  if (sin_theta < 0.0) sin_theta = -sin_theta;
  if (sin_theta > 1.0) sin_theta = 1.0;
  const double qnan = __longlong_as_double(0x7ff8000000000000LL);
  double s0 = sin_theta > 0.0 ? 0.0 : qnan;
  double s1 = sin_theta > 0.0 ? 1.0 : qnan;
  double ndx = dx * s0 + perpx * s1;
  double ndy = dy * s0 + perpy * s1;
  double nrm = sqrt(ndx * ndx + ndy * ndy);
  // (3) normalisation by one reciprocal and the exponent by a host-computed 1 / force_distance instead of three
  //     divisions: <= 2 ulp each on a force compared at 1e-9 relative; feeds no branch
  double inv_nrm = 1.0 / nrm;
  double nx = ndx * inv_nrm, ny = ndy * inv_nrm;
  double surface_dist = dist - z.two_r;
  double magnitude;
  if (ovx == 0.0 && ovy == 0.0) {
    magnitude = o.mag;
  } else {  // non-finite neighbour velocity: literal
    double rvx = vx - ovx, rvy = vy - ovy;
    magnitude = ((2.0 * z.agent_scale) * sqrt(rvx * rvx + rvy * rvy)) / t_i;
    if (magnitude >= 1e15) magnitude = 1e15;
  }
  double s = magnitude * exp(-surface_dist * z.inv_fd);
  fx = nx * s;
  fy = ny * s;
}

// One neighbour's contribution in the force pass, shared by every kernel form so that all of them
// produce the same bits.  Returns false when the pair contributes exactly (+-0, +-0).
__device__ __forceinline__ bool pair_force_dispatch(const OwnerPre& o, double px, double py, double vx, double vy,
                                                    double pfx, double pfy, uint64_t id, double ox, double oy,
                                                    double ovx, double ovy, uint64_t oid, double t_i,
                                                    const GroupDev& z, double& fx, double& fy) {
  double row;
  if (((id | oid) >> 53) == 0ull) row = id < oid ? -1.0 : 1.0;
  else row = right_of_way(id, oid);
  if (row < 0.0) {
    pair_force_yield(o, px, py, vx, vy, ox, oy, ovx, ovy, t_i, z, fx, fy);
    return true;
  }
  if (row > 0.0 && z.w0_fast && pair_force_w0_is_zero(o, ox, oy, ovx, ovy, t_i)) return false;
  PairIn p;
  p.px = px; p.py = py; p.vx = vx; p.vy = vy; p.pfx = pfx; p.pfy = pfy; p.id = id;
  p.ox = ox; p.oy = oy; p.ovx = ovx; p.ovy = ovy; p.oid = oid;
  pair_force_literal(p, t_i, z, fx, fy);
  return true;
}

}  // namespace rcs
