// rcs_step_warp.cuh -- the hot kernel, warp-cooperative form (sm_100a).
//
// step_kernel (rcs_kernels.cuh) gives each agent one thread that walks its own candidates and runs
// time_to_collision / the pair force inline; ncu shows those bodies executing with 3-5 of 32 lanes
// (profiles/r01a_step_kernel_v1.md).  Here a warp owns 32 agents, one per lane.
// The work is split by cost so that cheap, frequent tests stay per lane with no bookkeeping and only the rare,
// expensive bodies are compacted across the warp (profiles/r01b_step_warp_kernel_v3.md explains why):
//
//   1 filter   every lane walks its own candidates -- up to three contiguous slices of the sorted arrays at a
//              time -- and records the strict radius test (location_hash_2d.rs:251) + self filter
//              (lib.rs:284) as one 32-bit mask per slice.  2 loads, 5 DP ops, 2 compares per candidate.
//   2 t_i      every lane walks its own neighbour bits and evaluates the division-free half of
//              time_to_collision (zanlungo.rs:49-60: a, b, c, discriminant).  Only pairs that can return a
//              finite time (a > 0, discriminant >= 0, larger root possibly positive: ~15 % of the neighbours)
//              are appended to a shared pair list; the list is processed one pair per lane with
//              the literal routine (sqrt, two divisions, root selection) and reduced per owner with a 64-bit
//              shared atomicMin on the bit pattern (collision times are >= +0, so integer order == float order,
//              and min is order-independent).  The same walk records which neighbours have the higher id.
//   3 force    owners with a finite t_i split their neighbour bits into yield pairs (own id lower: weight 2,
//              real force, zanlungo.rs:93-170) and weight-0 pairs (provably (+-0, +-0) in the common case,
//              rcs_math.cuh).  Both kinds are compacted into their own lists and evaluated one pair per lane.
//              Every owner's pairs take one contiguous list segment (offsets from a warp scan of the per-lane
//              counts) in canonical neighbour order; pair forces go to per-pair slots and every owner adds its own
//              segment front to back, so the sum is bit-identical to the sequential one.
//
// Two kernels are built from these stages:
//   step_warp_kernel  32 consecutive agents of the canonical (cell, id) order per warp; the radius query of an
//                     agent is three slices (one per stencil column, prepared by gather_sorted_kernel) of at most
//                     32 candidates each: eyesight <= cell size, cells that are not crowded.  One round of 1-2-3.
//   step_aside_kernel the agents step_warp_kernel left aside because their stencil has more than three columns
//                     (eyesight > cell size) or a column holds more than 32 candidates (crowded or coarse cells):
//                     the columns are cut into chunks of 32 and taken three at a time, stage 1-2 over all rounds,
//                     then, with t_i known, stage 3 over all rounds with the masks kept from the first pass (chunks
//                     are visited in canonical order, so the force sum keeps its order).
// Agents whose ids are >= 2^53 or whose planner parameters defeat the weight-0 proof are finished by the tail of
// step_aside_kernel with the sequential routine.  Same arithmetic, same order, same results as step_kernel --
// tests compare the forms bit for bit.
#pragma once

#include "rcs_kernels.cuh"

namespace rcs {

constexpr int SW_WARPS = 4;            // warps per block
constexpr uint32_t SW_CAP = 128;       // stage-3 pair lists (A: evaluate, B: prove zero); >= 3 * SW_SLICE_MAX
constexpr uint32_t SW_SLICE_MAX = 32;  // candidates per slice (mask width)

struct WarpShared {
  double px[32], py[32], vx[32], vy[32], rr[32];                              // owners (stages 2 and 3)
  double pfx[32], pfy[32], ti[32];
  double futx[32], futy[32], mag[32], mvx[32], mvy[32], f0x[32], f0y[32];     // OwnerPre (stage 3)
  unsigned long long id[32];
  unsigned long long tbits[32];
  double sfx[SW_CAP], sfy[SW_CAP];     // pair forces of list A
  uint32_t lj[2 * SW_CAP];             // neighbour slot: list A (and the stage-2 hit list) | list B
  uint32_t grp[32];
  unsigned int poison[32];
  uint32_t hcnt;                       // entries in the stage-2 hit list
  uint8_t lo[2 * SW_CAP];              // owner lane: list A | list B
};

// ---------------- stage 1: radius filter, one mask per candidate slice
// Branch-free body: a lane that has run out of candidates re-reads `iself` (its own slot, or slot 0 for a lane
// without an agent, whose thr2 is 0), which the filter rejects; the loads of the unrolled iterations are
// independent and go out together.
__device__ __forceinline__ void sw_radius_masks(const double2* __restrict__ pos, double mpx, double mpy, double thr2,
                                                uint32_t i, uint32_t iself, uint32_t s0, uint32_t l0, uint32_t s1,
                                                uint32_t l1, uint32_t s2, uint32_t l2, uint32_t& m0, uint32_t& m1,
                                                uint32_t& m2) {
  const unsigned FULL = 0xffffffffu;
  const uint32_t x0 = __reduce_max_sync(FULL, l0), x1 = __reduce_max_sync(FULL, l1), x2 = __reduce_max_sync(FULL, l2);
#define RCS_FILTER_SLICE(MX, S, L, M)                                  \
  _Pragma("unroll 4")                                                  \
  for (uint32_t t = 0; t < (MX); ++t) {                                \
    const uint32_t j = (t < (L)) ? (S) + t : iself;                    \
    const double2 c = pos[j];                                          \
    const double dx = c.x - mpx;                                       \
    const double dy = c.y - mpy;                                       \
    const double d2 = dx * dx + dy * dy;                               \
    (M) |= ((d2 < thr2) && (j != i)) ? (1u << t) : 0u;                 \
  }
  RCS_FILTER_SLICE(x0, s0, l0, m0)
  RCS_FILTER_SLICE(x1, s1, l1, m1)
  RCS_FILTER_SLICE(x2, s2, l2, m2)
#undef RCS_FILTER_SLICE
}

// ---------------- stage 2: min over the masked neighbours of time_to_collision (zanlungo.rs:76-91) -> w.tbits
// Expects w.px/py/vx/vy/rr/tbits of every lane and w.hcnt = 0 to be visible (__syncwarp() after the stores) and
// leaves w.hcnt = 0.  y0..y2 receive the neighbours with the higher id: this agent yields to them
// (right_of_way = -1; exact for own ids < 2^53).
__device__ __forceinline__ void sw_collision_times(WarpShared& w, unsigned lane, const Self& me, double rr,
                                                   uint32_t iself, const double2* __restrict__ pos,
                                                   const double2* __restrict__ vel, const uint64_t* __restrict__ ids,
                                                   uint32_t m0, uint32_t m1, uint32_t m2, uint32_t s0, uint32_t s1,
                                                   uint32_t s2, uint32_t& y0, uint32_t& y1, uint32_t& y2) {
  const unsigned FULL = 0xffffffffu;
  uint32_t it = 0;
  auto flush_hits = [&]() {  // entered after a __syncwarp()
    const uint32_t cnt = *(volatile uint32_t*)&w.hcnt;
    for (uint32_t e = lane; e < cnt; e += 32) {
      const uint32_t o = w.lo[e];
      const uint32_t j = w.lj[e];
      const double2 c = pos[j], cv = vel[j];
      const double dx = c.x - w.px[o];
      const double dy = c.y - w.py[o];
      const double d2 = dx * dx + dy * dy;
      const double ct = time_to_collision(cv.x - w.vx[o], cv.y - w.vy[o], dx, dy, d2, w.rr[o]);
      if (ct < RCS_INF) atomicMin(&w.tbits[o], (unsigned long long)__double_as_longlong(ct));
    }
    __syncwarp();
    if (lane == 0) w.hcnt = 0u;
    __syncwarp();
  };
  // (word, slice start) queue of this lane; empty words are popped with predicated moves, so the walk over
  // the three slices stays free of divergent branches.  Two neighbours are taken per iteration: their loads
  // and arithmetic are independent, which hides half of the load and FP64 latency at this occupancy.
  uint32_t bits = m0, base = s0, nb1 = m1, ns1 = s1, nb2 = m2, ns2 = s2, k = 0;
  auto take = [&](uint32_t& j, uint32_t& t, uint32_t& kk) -> bool {
    const bool empty = bits == 0u;  // one pop per take: a lane with two empty words in a row idles once
    bits = empty ? nb1 : bits;
    base = empty ? ns1 : base;
    nb1 = empty ? nb2 : nb1;
    ns1 = empty ? ns2 : ns1;
    nb2 = empty ? 0u : nb2;
    k += empty ? 1u : 0u;
    const bool v = bits != 0u;
    t = v ? (uint32_t)(__ffs(bits) - 1) : 0u;
    bits &= bits - 1u;          // 0 stays 0
    j = v ? base + t : iself;   // always a valid slot: no branch around the loads
    kk = k;
    return v;
  };
  // the division-free half of time_to_collision for neighbour j; same operations as rcs_math.cuh
  auto probe = [&](bool v, uint32_t j, uint32_t t, uint32_t kk) -> bool {
    const uint32_t bit = (v && me.id < ids[j]) ? (1u << t) : 0u;
    y0 |= (kk == 0u) ? bit : 0u;
    y1 |= (kk == 1u) ? bit : 0u;
    y2 |= (kk == 2u) ? bit : 0u;
    const double2 c = pos[j], cv = vel[j];
    const double dx = c.x - me.px;
    const double dy = c.y - me.py;
    const double rvx = cv.x - me.vx;
    const double rvy = cv.y - me.vy;
    const double qa = rvx * rvx + rvy * rvy;
    const double d2 = dx * dx + dy * dy;
    const double qb = 2.0 * (rvx * dx + rvy * dy);
    const double qc = d2 - rr;
    const double bb = qb * qb;
    const double disc = bb - (4.0 * qa) * qc;
    // A finite time needs a or fl(b*b) != 0 (time_to_collision's first exit: a == 0 alone can still give
    // t_i = 0), disc >= 0 and -b + sqrt(disc) > 0.  For b >= 0, disc < fl(b*b) means disc <= fl(b*b) - 1 unit,
    // which is below the exact b^2 (fl(b*b) is within half a unit of it, normal or subnormal), so
    // sqrt(disc) <= b (correctly rounded sqrt is monotone, b is a double) and the numerator is <= 0: INF.
    // disc == b*b is passed on: sqrt(fl(b*b)) can exceed b when b*b is subnormal, and the same compare covers
    // b*b = inf.  Everything else is decided by the literal routine on the list.  a and b*b are +0, positive or
    // NaN (a NaN fails disc >= 0), so the first test is an integer OR of their bits: no FP64 instruction.
    return v && ((__double_as_longlong(qa) | __double_as_longlong(bb)) != 0ll) && (disc >= 0.0) &&
           ((qb < 0.0) || !(disc < bb));
  };
  while (__any_sync(FULL, (bits | nb1 | nb2) != 0u)) {
    uint32_t jA, tA, kA, jB, tB, kB;
    const bool vA = take(jA, tA, kA);
    const bool vB = take(jB, tB, kB);
    const bool hitA = probe(vA, jA, tA, kA);
    const bool hitB = probe(vB, jB, tB, kB);
    if (hitA) {  // order inside the list is irrelevant (min): a shared counter hands out the slots
      const uint32_t pos = atomicAdd(&w.hcnt, 1u);
      w.lj[pos] = jA;
      w.lo[pos] = (uint8_t)lane;
    }
    if (hitB) {
      const uint32_t pos = atomicAdd(&w.hcnt, 1u);
      w.lj[pos] = jB;
      w.lo[pos] = (uint8_t)lane;
    }
    if ((++it & 1u) == 0u) {  // at most 2 x 64 new entries since the last look at the counter
      __syncwarp();
      if (*(volatile uint32_t*)&w.hcnt > 2 * SW_CAP - 128) flush_hits();
    }
  }
  __syncwarp();
  if (*(volatile uint32_t*)&w.hcnt) flush_hits();
  __syncwarp();
}

// Stage-3 owner terms of one lane (zanlungo.rs:93-120 hoisted out of the pair loop) into shared memory.
__device__ __forceinline__ void sw_store_owner(WarpShared& w, unsigned lane, const Self& me, uint32_t grp) {
  w.pfx[lane] = me.pfx;
  w.pfy[lane] = me.pfy;
  w.id[lane] = me.id;
  w.grp[lane] = grp;
  w.poison[lane] = 0u;
}

__device__ __forceinline__ void sw_store_owner_pre(WarpShared& w, unsigned lane, const Self& me, double t_i,
                                                   const GroupDev& g) {
  const OwnerPre pre = owner_precompute(me.px, me.py, me.vx, me.vy, me.pfx, me.pfy, t_i, g);
  w.ti[lane] = t_i;
  w.futx[lane] = pre.futx;
  w.futy[lane] = pre.futy;
  w.mag[lane] = pre.mag;
  w.mvx[lane] = pre.mvx;
  w.mvy[lane] = pre.mvy;
  w.f0x[lane] = pre.f0x;
  w.f0y[lane] = pre.f0y;
}

// ---------------- stage 3: fx, fy += sum over the masked neighbours of compute_agent_force (zanlungo.rs:210-215)
// a0..a2: yield pairs (evaluate), z0..z2: weight-0 pairs (prove zero), per slice; all zero for lanes without a
// finite t_i.  Expects the owner terms (sw_store_owner, sw_store_owner_pre) to be visible.  NaN contributions of
// weight-0 pairs are collected in w.poison.
__device__ __forceinline__ void sw_pair_forces(const StepArgs& a, WarpShared& w, unsigned lane,
                                               const double2* __restrict__ pos, const double2* __restrict__ vel,
                                               const uint64_t* __restrict__ ids, uint32_t a0, uint32_t a1,
                                               uint32_t a2, uint32_t z0, uint32_t z1, uint32_t z2, uint32_t s0,
                                               uint32_t s1, uint32_t s2, double& fx, double& fy) {
  const unsigned FULL = 0xffffffffu;
  auto load_pre = [&](uint32_t o) {
    OwnerPre p;
    p.futx = w.futx[o]; p.futy = w.futy[o]; p.mag = w.mag[o];
    p.mvx = w.mvx[o]; p.mvy = w.mvy[o]; p.f0x = w.f0x[o]; p.f0y = w.f0y[o];
    return p;
  };
  auto literal = [&](uint32_t o, uint32_t j, double& qx, double& qy) {
    PairIn p;
    p.px = w.px[o]; p.py = w.py[o]; p.vx = w.vx[o]; p.vy = w.vy[o];
    p.pfx = w.pfx[o]; p.pfy = w.pfy[o]; p.id = w.id[o];
    const double2 c = pos[j], cv = vel[j];
    p.ox = c.x; p.oy = c.y; p.ovx = cv.x; p.ovy = cv.y; p.oid = ids[j];
    pair_force_literal(p, w.ti[o], a.groups[w.grp[o]], qx, qy);
  };
  // Every owner's pairs take one contiguous segment of a list, in canonical neighbour order (slice 0, 1, 2;
  // ascending slot), so the owner later adds its own slots front to back.  Segment offsets come from one warp
  // scan of the per-lane counts (list A in the low half-word, list B in the high one).
  const uint32_t cA = __popc(a0) + __popc(a1) + __popc(a2);
  const uint32_t cB = __popc(z0) + __popc(z1) + __popc(z2);
  const uint32_t own_cnt = cA | (cB << 16);
  uint32_t inc = own_cnt;
#pragma unroll
  for (int d = 1; d < 32; d <<= 1) {
    const uint32_t t = __shfl_up_sync(FULL, inc, d);
    if (lane >= (unsigned)d) inc += t;
  }
  const uint32_t exc = inc - own_cnt;
  uint32_t lane_begin = 0;
  while (lane_begin < 32) {  // one round unless the warp holds more pairs than a list does
    const uint32_t base = __shfl_sync(FULL, exc, lane_begin);
    const uint32_t rel = exc - base;  // field-wise: prefix sums are monotone, no borrow between the halves
    const uint32_t offA = rel & 0xffffu, offB = rel >> 16;
    const bool fits = lane >= lane_begin && offA + cA <= SW_CAP && offB + cB <= SW_CAP;
    const unsigned okm = __ballot_sync(FULL, fits || lane < lane_begin);
    const uint32_t lane_end = (okm == FULL) ? 32u : (uint32_t)(__ffs(~okm) - 1);  // > lane_begin: cA, cB <= 96
    const bool part = lane >= lane_begin && lane < lane_end;
    if (part) {
      // one walk per slice feeds both lists: yield pairs to A, weight-0 pairs to B
      uint32_t pA = offA, pB = SW_CAP + offB;
#define RCS_EMIT_SLICE(A, Z, S)                                          \
      for (uint32_t bits = (A) | (Z); bits; bits &= bits - 1u) {         \
        const uint32_t t = __ffs(bits) - 1;                              \
        const bool yv = (((A) >> t) & 1u) != 0u;                         \
        const uint32_t pos = yv ? pA : pB;                               \
        w.lj[pos] = (S) + t;                                             \
        w.lo[pos] = (uint8_t)lane;                                       \
        pA += yv ? 1u : 0u;                                              \
        pB += yv ? 0u : 1u;                                              \
      }
      RCS_EMIT_SLICE(a0, z0, s0)
      RCS_EMIT_SLICE(a1, z1, s1)
      RCS_EMIT_SLICE(a2, z2, s2)
#undef RCS_EMIT_SLICE
    }
    const uint32_t tot = __shfl_sync(FULL, inc, lane_end - 1) - base;
    const uint32_t nA = tot & 0xffffu, nB = tot >> 16;
    __syncwarp();
    for (uint32_t e = lane; e < nA; e += 32) {  // yield pairs: one per lane
      const uint32_t o = w.lo[e];
      const uint32_t j = w.lj[e];
      double qx, qy;
      const double2 c = pos[j], cv = vel[j];
      pair_force_yield(load_pre(o), w.px[o], w.py[o], w.vx[o], w.vy[o], c.x, c.y, cv.x, cv.y, w.ti[o],
                       a.groups[w.grp[o]], qx, qy);
      w.sfx[e] = qx;
      w.sfy[e] = qy;
    }
    for (uint32_t e = lane; e < nB; e += 32) {  // weight-0 pairs: prove the contribution is (+-0, +-0)
      const uint32_t o = w.lo[SW_CAP + e];
      const uint32_t j = w.lj[SW_CAP + e];
      const double2 c = pos[j], cv = vel[j];
      if (!pair_force_w0_is_zero(load_pre(o), c.x, c.y, cv.x, cv.y, w.ti[o])) {
        // contributes NaN or +-0 per component (rcs_math.cuh): NaN is order-independent
        double qx, qy;
        literal(o, j, qx, qy);
        const unsigned bits = (qx != qx ? 1u : 0u) | (qy != qy ? 2u : 0u);
        if (bits) atomicOr(&w.poison[o], bits);
      }
    }
    __syncwarp();
    if (part) {
      for (uint32_t r = 0; r < cA; ++r) {
        fx = fx + w.sfx[offA + r];
        fy = fy + w.sfy[offA + r];
      }
    }
    __syncwarp();
    lane_begin = lane_end;
  }
  __syncwarp();
}

__device__ __forceinline__ void sw_apply_poison(const WarpShared& w, unsigned lane, double& fx, double& fy) {
  const unsigned pz = w.poison[lane];
  if (pz & 1u) fx = fx + __longlong_as_double(0x7ff8000000000000LL);
  if (pz & 2u) fy = fy + __longlong_as_double(0x7ff8000000000000LL);
}

__global__ void __launch_bounds__(32 * SW_WARPS, 6) step_warp_kernel(StepArgs a) {
  __shared__ WarpShared sh[SW_WARPS];
  WarpShared& w = sh[threadIdx.x >> 5];
  const unsigned lane = threadIdx.x & 31u;
  const unsigned FULL = 0xffffffffu;
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;

  const double2* __restrict__ pos = a.in.pos;
  const double2* __restrict__ vel = a.in.vel;
  const uint64_t* __restrict__ ids = a.in.id;

  // This warp's own rows go out first, before the status words are even looked at: every array holds at least
  // a.n entries, so the loads are safe for i < a.n and their (DRAM) latency overlaps the dependent checks below.
  Self me;
  me.px = me.py = me.vx = me.vy = me.pfx = me.pfy = 0.0;
  me.id = 0;
  me.rwp = 0u;
  uint32_t grp = 0, wp_in = 0;
  uint4 sl = make_uint4(0u, 0u, 0u, 0u);
  const bool inb = i < a.n;
  if (inb) {
    const double2 p0 = pos[i], v0 = vel[i];
    me.px = p0.x;
    me.py = p0.y;
    me.vx = v0.x;
    me.vy = v0.y;
    me.id = ids[i];
    grp = a.in.grp[i];
    wp_in = a.in.wp[i];
    sl = a.slices[i];
  }
  if (a.status->failed) return;
  const uint32_t n_live = *a.n_sorted;
  bool active = inb && (i < n_live);

  double velx = 0.0, vely = 0.0, thr2 = 0.0, rr = 0.0;
  uint32_t role = ROLE_PASSIVE;
  bool zan = false;
  uint32_t s0 = 0, s1 = 0, s2 = 0, l0 = 0, l1 = 0, l2 = 0;  // candidate slices of this lane (cooperative path)
  bool fast = false;
  uint32_t cand = 0, nbc = 0;
  uint32_t aside = 0;  // finished by step_aside_kernel: 1 cooperatively (wide list), 2 sequentially (slow list)
  double t_i = RCS_INF, fx = 0.0, fy = 0.0;

  if (active) {
    role = agent_role(a, i);
    if (role == ROLE_PASSIVE) {
      active = false;
      drop_entry(a, i);
    }
  } else if (i < a.n) {
    drop_entry(a, i);
  }
  if (active) {
    const GroupDev& g = a.groups[grp];
    high_level_velocity(a, i, g, me, velx, vely);
    zan = g.lp_kind == LP_ZANLUNGO;
    thr2 = g.thr2;
    rr = g.rr;
    if (zan) {
      // candidate slices of the radius query, prepared by gather_sorted_kernel.  ids >= 2^53 round when they
      // become priorities (zanlungo.rs:94) and groups whose weight-0 pairs cannot be proven zero need the literal
      // routine for every pair: both are left to the sequential routine, wide or crowded stencils to the chunked
      // cooperative one (step_aside_kernel)
      s0 = sl.x; s1 = sl.y; s2 = sl.z;
      l0 = sl.w & 0xffu; l1 = (sl.w >> 8) & 0xffu; l2 = (sl.w >> 16) & 0xffu;
      const bool coop = g.w0_fast && (me.id >> 53) == 0ull;
      fast = coop && (sl.w >> 24) != 0u && l0 <= SW_SLICE_MAX && l1 <= SW_SLICE_MAX && l2 <= SW_SLICE_MAX;
      if (!fast) {
        l0 = l1 = l2 = 0;
        thr2 = 0.0;  // the filter's padding reads of this lane must reject everything (it takes no part)
        active = false;
        zan = false;
        aside = coop ? 1u : 2u;
      } else {
        cand = l0 + l1 + l2;
      }
    }
  }
  // agents for step_aside_kernel keep their neighbours in this warp as neighbours on the list (one slot range per warp)
  {
    const unsigned wm = __ballot_sync(FULL, aside == 1u);
    if (wm) {
      uint32_t at = 0;
      if (lane == (unsigned)(__ffs(wm) - 1)) at = atomicAdd(&a.status->wide_count, (unsigned)__popc(wm));
      at = __shfl_sync(FULL, at, __ffs(wm) - 1);
      if (aside == 1u) a.wide_list[at + __popc(wm & ((1u << lane) - 1u))] = i;
    }
    if (aside == 2u) a.slow_list[atomicAdd(&a.status->slow_count, 1u)] = i;
  }

  uint32_t m0 = 0, m1 = 0, m2 = 0;
  const uint32_t iself = active ? i : 0u;  // lanes without an agent have l = 0 and thr2 = 0
  sw_radius_masks(pos, me.px, me.py, thr2, i, iself, s0, l0, s1, l1, s2, l2, m0, m1, m2);
  nbc = __popc(m0) + __popc(m1) + __popc(m2);

  if (__any_sync(FULL, (m0 | m1 | m2) != 0u)) {
    w.px[lane] = me.px;
    w.py[lane] = me.py;
    w.vx[lane] = me.vx;
    w.vy[lane] = me.vy;
    w.rr[lane] = rr;
    w.tbits[lane] = 0x7ff0000000000000ull;
    if (lane == 0) w.hcnt = 0u;
    __syncwarp();
    uint32_t y0 = 0, y1 = 0, y2 = 0;
    sw_collision_times(w, lane, me, rr, iself, pos, vel, ids, m0, m1, m2, s0, s1, s2, y0, y1, y2);
    if (fast) t_i = __longlong_as_double((long long)w.tbits[lane]);

    const bool fin = fast && (t_i != RCS_INF);
    if (__any_sync(FULL, fin)) {
      uint32_t a0 = 0, a1 = 0, a2 = 0, z0 = 0, z1 = 0, z2 = 0;  // list A bits (evaluate) / list B bits (prove zero)
      sw_store_owner(w, lane, me, grp);
      if (fin) {
        sw_store_owner_pre(w, lane, me, t_i, a.groups[grp]);
        a0 = m0 & y0; a1 = m1 & y1; a2 = m2 & y2;
        z0 = m0 & ~y0; z1 = m1 & ~y1; z2 = m2 & ~y2;
      }
      __syncwarp();
      sw_pair_forces(a, w, lane, pos, vel, ids, a0, a1, a2, z0, z1, z2, s0, s1, s2, fx, fy);
      sw_apply_poison(w, lane, fx, fy);
    }
  }

  if (active) {
    const GroupDev& g = a.groups[grp];
    if (zan) {
      // zanlungo.rs:216
      velx = velx + fx * g.inv_mass;
      vely = vely + fy * g.inv_mass;
    }
    integrate_and_store(a, i, me, g, grp, wp_in, role, velx, vely, t_i, fx, fy, nbc);
  }
  const bool own = active && role == ROLE_OWN;
  warp_stats(a, own ? cand : 0u, own ? nbc : 0u, (own && zan && t_i != RCS_INF) ? 1u : 0u);
}

// The columns of one agent's radius query (location_hash_2d.rs:245-246), each one contiguous slice of the sorted
// arrays, handed out in canonical order in chunks of at most SW_SLICE_MAX candidates.
struct ColumnWalk {
  int64_t col, right, bottom, top;
  uint32_t s, rem;  // what is left of the current column's slice
};

__device__ __forceinline__ void cw_begin(ColumnWalk& c, const GridDev& g, double radius, double px, double py) {
  int64_t left;
  get_bounds(g, radius, px, py, left, c.right, c.bottom, c.top);
  if (left < 0) left = 0;
  if (c.right > g.x_max) c.right = g.x_max;
  c.col = left;
  c.s = 0u;
  c.rem = 0u;
}

__device__ __forceinline__ void cw_none(ColumnWalk& c) {
  c.col = 1;
  c.right = 0;
  c.bottom = c.top = 0;
  c.s = c.rem = 0u;
}

__device__ __forceinline__ bool cw_more(const ColumnWalk& c) { return c.rem != 0u || c.col <= c.right; }

__device__ __forceinline__ void cw_next(ColumnWalk& c, const GridDev& g, const uint32_t* __restrict__ cell_start,
                                        uint32_t& s, uint32_t& l) {
  if (c.rem == 0u && c.col <= c.right) {
    uint64_t c_lo, c_hi;
    if (column_cell_range(g, c.col, c.bottom, c.top, c_lo, c_hi)) {
      c.s = cell_start[c_lo];
      c.rem = cell_start[c_hi + 1] - c.s;
    }
    ++c.col;
  }
  l = c.rem < SW_SLICE_MAX ? c.rem : SW_SLICE_MAX;
  s = c.s;
  c.s += l;
  c.rem -= l;
}

// Consumes what is left of the walk without looking at the candidates; returns how many there were.
__device__ __forceinline__ uint32_t cw_skip_all(ColumnWalk& c, const GridDev& g,
                                                const uint32_t* __restrict__ cell_start) {
  uint32_t total = c.rem;
  c.rem = 0u;
  for (; c.col <= c.right; ++c.col) {
    uint64_t c_lo, c_hi;
    if (column_cell_range(g, c.col, c.bottom, c.top, c_lo, c_hi)) total += cell_start[c_hi + 1] - cell_start[c_lo];
  }
  return total;
}

// The first rounds' masks of the first pass are kept for the second one (one column of words per lane).
constexpr uint32_t SW_WIDE_ROUNDS = 4;
struct WideMasks {
  uint32_t m[3 * SW_WIDE_ROUNDS][32];  // in radius
  uint32_t y[3 * SW_WIDE_ROUNDS][32];  // ... and with the higher id
};

// Finishes the agents step_warp_kernel left aside.  a.wide_list (live, advanced by this rank, Zanlungo, eligible for
// the weight-0 proof): 32 per warp, cooperatively, chunked stencil columns.  a.slow_list: one per thread with the
// sequential routine.  Grid-stride over the device-side counts.
__global__ void __launch_bounds__(32 * SW_WARPS, 4) step_aside_kernel(StepArgs a) {
  __shared__ WarpShared sh[SW_WARPS];
  __shared__ WideMasks shm[SW_WARPS];
  WarpShared& w = sh[threadIdx.x >> 5];
  WideMasks& wm = shm[threadIdx.x >> 5];
  const unsigned lane = threadIdx.x & 31u;
  const unsigned FULL = 0xffffffffu;
  if (a.status->failed) return;
  const uint32_t n_wide = a.status->wide_count;

  const double2* __restrict__ pos = a.in.pos;
  const double2* __restrict__ vel = a.in.vel;
  const uint64_t* __restrict__ ids = a.in.id;
  uint32_t st_cand = 0, st_nbc = 0, st_fin = 0;

  for (uint32_t k0 = blockIdx.x * blockDim.x + (threadIdx.x & ~31u); k0 < n_wide; k0 += gridDim.x * blockDim.x) {
    const bool have = k0 + lane < n_wide;
    const uint32_t i = have ? a.wide_list[k0 + lane] : 0u;
    Self me;
    me.px = me.py = me.vx = me.vy = me.pfx = me.pfy = 0.0;
    me.id = 0;
    me.rwp = 0u;
    uint32_t grp = 0, wp_in = 0, role = ROLE_PASSIVE;
    double velx = 0.0, vely = 0.0, thr2 = 0.0, rr = 0.0, eyesight = 0.0;
    if (have) {
      const double2 p0 = pos[i], v0 = vel[i];
      me.px = p0.x;
      me.py = p0.y;
      me.vx = v0.x;
      me.vy = v0.y;
      me.id = ids[i];
      grp = a.in.grp[i];
      wp_in = a.in.wp[i];
      role = agent_role(a, i);
      const GroupDev& g = a.groups[grp];
      high_level_velocity(a, i, g, me, velx, vely);
      thr2 = g.thr2;
      rr = g.rr;
      eyesight = g.eyesight;
    }
    const uint32_t iself = i;  // slot 0 for lanes without an agent (thr2 = 0 rejects everything)

    w.px[lane] = me.px;
    w.py[lane] = me.py;
    w.vx[lane] = me.vx;
    w.vy[lane] = me.vy;
    w.rr[lane] = rr;
    w.tbits[lane] = 0x7ff0000000000000ull;
    if (lane == 0) w.hcnt = 0u;
    __syncwarp();

    // ---- first pass over the stencil: neighbour count and t_i
    uint32_t cand = 0, nbc = 0;
    ColumnWalk cw;
    if (have) cw_begin(cw, a.grid, eyesight, me.px, me.py);
    else cw_none(cw);
    // An agent whose own position is not finite has no neighbours: every d2 is inf or NaN and fails the strict
    // `<` of location_hash_2d.rs:251.  The reference files such agents in cell 0 (NaN as usize = 0) and their
    // query is the whole of cell 0, so a crowd that has gone non-finite would otherwise cost the square of their
    // number.  Only the candidate statistic still needs the slice lengths.
    if (have && !(isfinite(me.px) && isfinite(me.py))) cand += cw_skip_all(cw, a.grid, a.cell_start);
    for (uint32_t r = 0; __any_sync(FULL, cw_more(cw)); ++r) {
      uint32_t s0, s1, s2, l0, l1, l2;
      cw_next(cw, a.grid, a.cell_start, s0, l0);
      cw_next(cw, a.grid, a.cell_start, s1, l1);
      cw_next(cw, a.grid, a.cell_start, s2, l2);
      cand += l0 + l1 + l2;
      uint32_t m0 = 0, m1 = 0, m2 = 0, y0 = 0, y1 = 0, y2 = 0;
      sw_radius_masks(pos, me.px, me.py, thr2, i, iself, s0, l0, s1, l1, s2, l2, m0, m1, m2);
      nbc += __popc(m0) + __popc(m1) + __popc(m2);
      if (__any_sync(FULL, (m0 | m1 | m2) != 0u))
        sw_collision_times(w, lane, me, rr, iself, pos, vel, ids, m0, m1, m2, s0, s1, s2, y0, y1, y2);
      if (r < SW_WIDE_ROUNDS) {
        wm.m[3 * r + 0][lane] = m0; wm.m[3 * r + 1][lane] = m1; wm.m[3 * r + 2][lane] = m2;
        wm.y[3 * r + 0][lane] = y0; wm.y[3 * r + 1][lane] = y1; wm.y[3 * r + 2][lane] = y2;
      }
    }
    __syncwarp();
    const double t_i = have ? __longlong_as_double((long long)w.tbits[lane]) : RCS_INF;
    const bool fin = t_i != RCS_INF;
    double fx = 0.0, fy = 0.0;

    // ---- second pass, owners with a finite t_i: the force sum in canonical neighbour order
    if (__any_sync(FULL, fin)) {
      sw_store_owner(w, lane, me, grp);
      if (fin) {
        sw_store_owner_pre(w, lane, me, t_i, a.groups[grp]);
        cw_begin(cw, a.grid, eyesight, me.px, me.py);
      } else {
        cw_none(cw);
      }
      __syncwarp();
      for (uint32_t r = 0; __any_sync(FULL, cw_more(cw)); ++r) {  // the same rounds as above for these lanes
        uint32_t s0, s1, s2, l0, l1, l2;
        cw_next(cw, a.grid, a.cell_start, s0, l0);
        cw_next(cw, a.grid, a.cell_start, s1, l1);
        cw_next(cw, a.grid, a.cell_start, s2, l2);
        uint32_t m0 = 0, m1 = 0, m2 = 0, y0 = 0, y1 = 0, y2 = 0;
        if (r < SW_WIDE_ROUNDS) {
          if (fin) {
            m0 = wm.m[3 * r + 0][lane]; m1 = wm.m[3 * r + 1][lane]; m2 = wm.m[3 * r + 2][lane];
            y0 = wm.y[3 * r + 0][lane]; y1 = wm.y[3 * r + 1][lane]; y2 = wm.y[3 * r + 2][lane];
          }
        } else {
          sw_radius_masks(pos, me.px, me.py, thr2, i, iself, s0, l0, s1, l1, s2, l2, m0, m1, m2);
          for (uint32_t b = m0; b; b &= b - 1u) y0 |= (me.id < ids[s0 + __ffs(b) - 1]) ? (b & (0u - b)) : 0u;
          for (uint32_t b = m1; b; b &= b - 1u) y1 |= (me.id < ids[s1 + __ffs(b) - 1]) ? (b & (0u - b)) : 0u;
          for (uint32_t b = m2; b; b &= b - 1u) y2 |= (me.id < ids[s2 + __ffs(b) - 1]) ? (b & (0u - b)) : 0u;
        }
        if (__any_sync(FULL, (m0 | m1 | m2) != 0u))
          sw_pair_forces(a, w, lane, pos, vel, ids, m0 & y0, m1 & y1, m2 & y2, m0 & ~y0, m1 & ~y1, m2 & ~y2, s0, s1,
                         s2, fx, fy);
      }
      __syncwarp();
      sw_apply_poison(w, lane, fx, fy);
    }

    if (have) {
      const GroupDev& g = a.groups[grp];
      // zanlungo.rs:216
      velx = velx + fx * g.inv_mass;
      vely = vely + fy * g.inv_mass;
      integrate_and_store(a, i, me, g, grp, wp_in, role, velx, vely, t_i, fx, fy, nbc);
    }
    if (have && role == ROLE_OWN) {
      st_cand += cand;
      st_nbc += nbc;
      st_fin += fin ? 1u : 0u;
    }
    __syncwarp();  // the next round of this warp reuses the shared arrays
  }

  // ids >= 2^53, planners without the weight-0 proof: the sequential routine, one agent per thread
  const uint32_t n_slow = a.status->slow_count;
  for (uint32_t k = blockIdx.x * blockDim.x + threadIdx.x; k < n_slow; k += gridDim.x * blockDim.x)
    step_one_agent(a, a.slow_list[k], st_cand, st_nbc, st_fin);
  warp_stats(a, st_cand, st_nbc, st_fin);
}

}  // namespace rcs
