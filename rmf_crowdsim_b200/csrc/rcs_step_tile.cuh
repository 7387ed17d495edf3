// rcs_step_tile.cuh -- the hot kernel with the query stencil staged in shared memory (sm_100a).
//
// The reference scans, for every agent, the cells `for x in left..=right { for y in bottom..=top }`
// (location_hash_2d.rs:245-256) and hands the survivors of the strict radius test to the planner twice
// (zanlungo.rs:76-91 and :210-215).  With the agents in canonical (cell, id) order each stencil column is one
// contiguous slice of the sorted arrays, and the slices of CONSECUTIVE agents overlap almost completely: a block of
// 128 consecutive agents (a run of ~32 cells of one cell column at 4 agents per cell) touches three runs of ~34 cells.
// step_warp_kernel (rcs_step_warp.cuh) reads those rows through L1 / L2, agent by agent; ncu attributes 36 % of its
// stall cycles to long-scoreboard waits on them (profiles/r01d_final_build.md).  Here a block copies the union of
// its agents' slices -- three contiguous row ranges of (position, velocity, id), one per stencil column, found by
// gather_sorted_kernel -- into shared memory ONCE, with one-dimensional bulk copies (cp.async.bulk, completion on an
// mbarrier) issued by one thread, and everything after that runs out of shared memory and registers:
//
//   1 filter   every lane walks its own three slices of the staged positions (branch-free, unrolled) and appends the
//              rows that pass the strict radius test (location_hash_2d.rs:251) and the self filter (lib.rs:284) to
//              its neighbour list in shared memory -- 16-bit staged row numbers, canonical order.
//   2 t_i      every lane walks its list two entries at a time and evaluates the division-free half of
//              time_to_collision (zanlungo.rs:49-60); the few pairs that can return a finite time are queued per
//              warp and finished one per lane (sqrt, two divisions); owners' terms travel by warp shuffle, the
//              minimum by a 64-bit shared atomicMin on the bit pattern.  The walk also marks the entries with the
//              higher id (this agent yields to them: weight 2, zanlungo.rs:93-170).
//   3 force    owners with a finite t_i: weight-0 entries are proven to contribute (+-0, +-0) by the lane itself
//              (rcs_math.cuh); yield entries are compacted across the warp (one contiguous list segment per owner
//              from a warp scan), evaluated one pair per lane, and added by their owner front to back in canonical
//              order -- bit-identical to the sequential sum.
//
// Agents the block cannot take -- stencil wider than three columns, more than 32 candidates in a column, more
// neighbours than a list holds, ids >= 2^53, a union larger than the staging buffer -- go to step_aside_kernel's
// lists exactly as in step_warp_kernel.  Same arithmetic, same order, same bits as every other form of the kernel.
#pragma once

#include "rcs_step_warp.cuh"

namespace rcs {

#ifndef RCS_TILE_ROWS
#define RCS_TILE_ROWS (3 * 32 * RCS_TILE_WARPS + 96)  // three ranges of ~(owners + 2 cells) rows each, and slack
#endif
#ifndef RCS_TILE_BLOCKS
#define RCS_TILE_BLOCKS 5
#endif
#ifndef RCS_TILE_PHASED
#define RCS_TILE_PHASED 0
#endif
#ifndef RCS_TILE_TMA
#define RCS_TILE_TMA 1
#endif
#ifndef RCS_TILE_NB
#define RCS_TILE_NB 32
#endif

constexpr uint32_t ST_ROWS = RCS_TILE_ROWS;  // staged rows per block (40 B each)
constexpr uint32_t ST_PAD = 32;              // rows a lane may read beyond its own slice (masked afterwards)
constexpr uint32_t ST_NB = RCS_TILE_NB;      // neighbour-list entries per agent (<= 32: one mask word)
constexpr uint32_t ST_CAP = 128;             // pair list of a warp (stage-2 hit list, stage-3 yield list)

struct TileWarp {
  uint16_t nl[ST_NB][32];        // neighbour lists, one column per lane
  unsigned long long tbits[32];  // min collision time of every owner (bit pattern)
  double2 sf[ST_CAP];            // pair forces of the yield list
  uint16_t lj[2 * ST_CAP];       // staged row of the neighbour: yield list (and stage-2 hit list) | weight-0 list
  uint8_t lo[2 * ST_CAP];        // owner lane
  unsigned int poison[32];
  uint32_t hcnt;
  uint32_t pad_[3];
};

struct TileShared {
  double2 pos[ST_ROWS + ST_PAD];
  double2 vel[ST_ROWS + 2];
  unsigned long long id[ST_ROWS + 4];
  TileWarp w[ST_WARPS];
  unsigned long long mbar;
  unsigned int stat[4];  // candidates, neighbours, agents with a finite t_i of the block (one global atomic each)
};

__device__ __forceinline__ uint32_t st_smem_addr(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

// one-dimensional bulk copy global -> shared; completion is counted in bytes on an mbarrier
__device__ __forceinline__ void st_bulk_copy(void* dst, const void* src, uint32_t bytes, unsigned long long* mbar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                   st_smem_addr(dst)),
               "l"(src), "r"(bytes), "r"(st_smem_addr(mbar))
               : "memory");
}

__device__ __forceinline__ double st_shfl(double v, uint32_t src) { return __shfl_sync(0xffffffffu, v, (int)src); }

// Does step_tile_kernel take this agent on its three-slice path?  (Evaluated identically by gather_sorted_kernel,
// which prepares the block's staging ranges, and by the kernel itself.)
__device__ __forceinline__ bool st_takes(const GroupDev& g, uint64_t id, uint4 sl) {
  return g.lp_kind == LP_ZANLUNGO && g.w0_fast && (id >> 53) == 0ull && (sl.w >> 24) != 0u &&
         (sl.w & 0xffu) <= SW_SLICE_MAX && ((sl.w >> 8) & 0xffu) <= SW_SLICE_MAX &&
         ((sl.w >> 16) & 0xffu) <= SW_SLICE_MAX;
}

// Union of a block's slices per stencil column (TileRange, rcs_kernels.cuh), computed by the block that gathers the
// same 128 agents (gather_sorted_kernel) and read back by step_tile_kernel before it issues the bulk copies.
__device__ __forceinline__ void st_block_ranges(bool takes, uint4 sl, uint32_t (*red)[6], TileRange* out) {
  const unsigned FULL = 0xffffffffu, NONE = 0xffffffffu;
  const unsigned lane = threadIdx.x & 31u, warp = threadIdx.x >> 5;
  const uint32_t l0 = sl.w & 0xffu, l1 = (sl.w >> 8) & 0xffu, l2 = (sl.w >> 16) & 0xffu;
  const uint32_t a0 = __reduce_min_sync(FULL, (takes && l0) ? sl.x : NONE);
  const uint32_t a1 = __reduce_min_sync(FULL, (takes && l1) ? sl.y : NONE);
  const uint32_t a2 = __reduce_min_sync(FULL, (takes && l2) ? sl.z : NONE);
  const uint32_t b0 = __reduce_max_sync(FULL, (takes && l0) ? sl.x + l0 : 0u);
  const uint32_t b1 = __reduce_max_sync(FULL, (takes && l1) ? sl.y + l1 : 0u);
  const uint32_t b2 = __reduce_max_sync(FULL, (takes && l2) ? sl.z + l2 : 0u);
  if (lane == 0) {
    red[warp][0] = a0; red[warp][1] = a1; red[warp][2] = a2;
    red[warp][3] = b0; red[warp][4] = b1; red[warp][5] = b2;
  }
  __syncthreads();
  if (threadIdx.x < 3) {
    const int d = threadIdx.x;
    uint32_t mn = NONE, mx = 0u;
    for (uint32_t ww = 0; ww < (blockDim.x >> 5); ++ww) {
      mn = min(mn, red[ww][d]);
      mx = max(mx, red[ww][3 + d]);
    }
    const uint32_t lo = mx > mn ? (mn & ~1u) : 0u;
    out->lo[d] = lo;
    out->len[d] = mx > mn ? ((mx + 1u) & ~1u) - lo : 0u;
  }
}

// Stage 3, a weight-0 pair that is not provably (+-0, +-0): the literal routine decides between +-0 and NaN per
// component (rcs_math.cuh); NaN is order-independent, so it travels as a poison bit.  Entered by the whole warp
// (the owner's terms come by shuffle); `lit` marks the lanes that hold such a pair.
__device__ __noinline__ void st_w0_literal(TileWarp& w, const GroupDev* groups, bool lit, uint32_t o, double2 c,
                                           double2 cv, unsigned long long oid, double px, double py, double vx,
                                           double vy, double pfx, double pfy, unsigned long long id, uint32_t grp,
                                           double oti) {
  const unsigned FULL = 0xffffffffu;
  PairIn p;
  p.px = st_shfl(px, o); p.py = st_shfl(py, o); p.vx = st_shfl(vx, o); p.vy = st_shfl(vy, o);
  p.pfx = st_shfl(pfx, o); p.pfy = st_shfl(pfy, o);
  p.id = __shfl_sync(FULL, id, (int)o);
  const uint32_t ogrp = __shfl_sync(FULL, grp, (int)o);
  if (lit) {
    p.ox = c.x; p.oy = c.y; p.ovx = cv.x; p.ovy = cv.y; p.oid = oid;
    double qx, qy;
    pair_force_literal(p, oti, groups[ogrp], qx, qy);
    const unsigned pb = (qx != qx ? 1u : 0u) | (qy != qy ? 2u : 0u);
    if (pb) atomicOr(&w.poison[o], pb);
  }
}

// Stage 2, the queued pairs of a warp: the literal time_to_collision (sqrt, two divisions, root selection), one pair
// per lane; the owner's terms come by shuffle, the minimum goes to the owner's slot by a shared atomicMin on the bit
// pattern (collision times are >= +0, so integer order == float order, and min is order-independent).  Entered by
// the whole warp after a __syncwarp(); n_hit = entries in the list.
__device__ __noinline__ void st_flush_hits(TileWarp& w, uint32_t n_hit, const double2* spos, const double2* svel,
                                           unsigned lane, double px, double py, double vx, double vy, double rr) {
  for (uint32_t b = 0; b < n_hit; b += 32) {
    const uint32_t e = b + lane;
    const bool v = e < n_hit;
    const uint32_t o = v ? w.lo[e] : lane;
    const uint32_t j = v ? w.lj[e] : 0u;
    const double opx = st_shfl(px, o), opy = st_shfl(py, o), ovx = st_shfl(vx, o), ovy = st_shfl(vy, o),
                 orr = st_shfl(rr, o);
    if (v) {
      const double2 c = spos[j], cv = svel[j];
      const double dx = c.x - opx;
      const double dy = c.y - opy;
      const double d2 = dx * dx + dy * dy;
      const double ct = time_to_collision(cv.x - ovx, cv.y - ovy, dx, dy, d2, orr);
      if (ct < RCS_INF) atomicMin(&w.tbits[o], (unsigned long long)__double_as_longlong(ct));
    }
  }
  __syncwarp();
}

// STRIPS: the handle is a strip (ownership roles, keep flags by the new column); the plain form has none of that code.
template <bool STRIPS>
__global__ void __launch_bounds__(32 * ST_WARPS, RCS_TILE_BLOCKS) step_tile_kernel(StepArgs a) {
  extern __shared__ __align__(16) unsigned char st_smem_raw[];
  TileShared& sh = *reinterpret_cast<TileShared*>(st_smem_raw);
  const unsigned warp = threadIdx.x >> 5;
  TileWarp& w = sh.w[warp];
  const unsigned lane = threadIdx.x & 31u;
  const unsigned FULL = 0xffffffffu;
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;

  // own row first: its loads are in flight while thread 0 sets up the staging
  Self me;
  me.px = me.py = me.vx = me.vy = me.pfx = me.pfy = 0.0;
  me.id = 0;
  me.rwp = 0u;
  uint32_t grp = 0, wp_in = 0, cell_i = 0;
  uint4 sl = make_uint4(0u, 0u, 0u, 0u);
  const bool inb = i < a.n;
  if (inb) {
    // (strips: the agent's cell decides its role; loaded here, with the own row, it is not one more global-memory
    // latency in front of everything behind the barrier -- that was 4 % of the kernel on a strip handle)
    if (STRIPS) cell_i = a.cell[i];
    const double2 p0 = a.in.pos[i], v0 = a.in.vel[i];
    me.px = p0.x;
    me.py = p0.y;
    me.vx = v0.x;
    me.vy = v0.y;
    me.id = a.in.id[i];
    grp = a.in.grp[i];
    wp_in = a.in.wp[i];
    sl = a.slices[i];
  }

  // ---- staging: one thread reads the block's ranges and issues the bulk copies
  const TileRange tr = a.tile_ranges[blockIdx.x];
  uint32_t off1 = tr.len[0], off2 = tr.len[0] + tr.len[1];
  const uint32_t total = off2 + tr.len[2];
  const bool staged = total <= ST_ROWS;  // block-uniform
  const bool failed = a.status->failed != 0u;
  if (threadIdx.x == 0) {
    sh.stat[0] = sh.stat[1] = sh.stat[2] = 0u;
    asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(st_smem_addr(&sh.mbar)));
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    if (staged && total && !failed) {
      asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(st_smem_addr(&sh.mbar)),
                   "r"(total * 40u)
                   : "memory");
#pragma unroll 1
      for (int d = 0; d < 3; ++d) {  // one copy of the code (instruction cache)
        const uint32_t len = d == 0 ? tr.len[0] : (d == 1 ? tr.len[1] : tr.len[2]);
        const uint32_t lo = d == 0 ? tr.lo[0] : (d == 1 ? tr.lo[1] : tr.lo[2]);
        const uint32_t off = d == 0 ? 0u : (d == 1 ? off1 : off2);
        if (!len) continue;
        st_bulk_copy(&sh.pos[off], a.in.pos + lo, len * 16u, &sh.mbar);
        st_bulk_copy(&sh.vel[off], a.in.vel + lo, len * 16u, &sh.mbar);
        st_bulk_copy(&sh.id[off], a.in.id + lo, len * 8u, &sh.mbar);
      }
    }
  }
  const uint32_t role_i = STRIPS ? agent_role_and_bits(a, cell_i) : (uint32_t)ROLE_OWN;
  const uint32_t n_live = *a.n_sorted;
  __syncthreads();  // the barrier is initialised (and nobody leaves before the copies were issued)
  if (failed) return;
  bool active = inb && (i < n_live);

  double velx = 0.0, vely = 0.0, thr2 = 0.0, rr = 0.0;
  uint32_t role = ROLE_PASSIVE;
  bool zan = false, fast = false, coop = false;
  uint32_t cand = 0, nbc = 0, aside = 0;
  double t_i = RCS_INF, fx = 0.0, fy = 0.0;

  if (active) {
    role = role_i;
    if ((role & ROLE_MASK) == ROLE_PASSIVE) {
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
      coop = g.w0_fast && (me.id >> 53) == 0ull;
      fast = staged && st_takes(g, me.id, sl);
    }
  }
  // slices of this lane as staged rows
  uint32_t l0 = 0, l1 = 0, l2 = 0, q0 = 0, q1 = 0, q2 = 0, self0 = 32u, self1 = 32u, self2 = 32u;
  if (fast) {
    l0 = sl.w & 0xffu; l1 = (sl.w >> 8) & 0xffu; l2 = (sl.w >> 16) & 0xffu;
    q0 = sl.x - tr.lo[0];
    q1 = sl.y - tr.lo[1] + off1;
    q2 = sl.z - tr.lo[2] + off2;
    if (!l0) q0 = 0u;
    if (!l1) q1 = 0u;
    if (!l2) q2 = 0u;
    // the self filter (lib.rs:284): the agent's own row is candidate i - s of the slice that holds its cell
    self0 = i - sl.x; self1 = i - sl.y; self2 = i - sl.z;
    cand = l0 + l1 + l2;
  }

  // ---- wait for the staged rows (phase 0 of the barrier)
  if (staged && total) {
    uint32_t done = 0;
    while (!done) {
      asm volatile(
          "{\n\t.reg .pred p;\n\t"
          "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
          "selp.u32 %0, 1, 0, p;\n\t}"
          : "=r"(done)
          : "r"(st_smem_addr(&sh.mbar)), "r"(0u)
          : "memory");
    }
  }
  const double2* spos = sh.pos;
  const double2* svel = sh.vel;
  const unsigned long long* sid = sh.id;

  // ---- stage 1: radius filter (location_hash_2d.rs:251), one mask per slice.  Branch-free: a lane whose slice is
  // shorter than the warp's longest reads on into the next staged rows (or the padding); those bits, and the agent's
  // own (lib.rs:284), are cleared afterwards.
  uint32_t m0 = 0, m1 = 0, m2 = 0;
  {
#pragma unroll 1
    for (int k = 0; k < 3; ++k) {  // one copy of the loop body for the three slices (instruction cache)
      const uint32_t l = k == 0 ? l0 : (k == 1 ? l1 : l2);
      const uint32_t mx = __reduce_max_sync(FULL, l);
      const double2* rowp = spos + (k == 0 ? q0 : (k == 1 ? q1 : q2));
      uint32_t m = 0u, bit = 1u;
#pragma unroll 4
      for (uint32_t t = 0; t < mx; ++t) {
        const double2 c = rowp[t];
        const double dx = c.x - me.px;
        const double dy = c.y - me.py;
        const double d2 = dx * dx + dy * dy;
        if (d2 < thr2) m |= bit;
        bit <<= 1;
      }
      if (k == 0) m0 = m;
      else if (k == 1) m1 = m;
      else m2 = m;
    }
    m0 &= (l0 >= 32u ? 0xffffffffu : (1u << l0) - 1u) & ~(self0 < 32u ? 1u << self0 : 0u);
    m1 &= (l1 >= 32u ? 0xffffffffu : (1u << l1) - 1u) & ~(self1 < 32u ? 1u << self1 : 0u);
    m2 &= (l2 >= 32u ? 0xffffffffu : (1u << l2) - 1u) & ~(self2 < 32u ? 1u << self2 : 0u);
  }
  nbc = __popc(m0) + __popc(m1) + __popc(m2);
  if (fast && nbc > ST_NB) {  // more neighbours than a list holds: the chunked kernel recounts them
    fast = false;
    nbc = 0u;
    cand = 0u;
  }
  if (zan && !fast) {
    active = false;
    zan = false;
    aside = coop ? 1u : 2u;
  }
  {  // agents for step_aside_kernel keep their neighbours in this warp as neighbours on the list
    const unsigned wm = __ballot_sync(FULL, aside == 1u);
    if (wm) {
      uint32_t at = 0;
      if (lane == (unsigned)(__ffs(wm) - 1)) at = atomicAdd(&a.status->wide_count, (unsigned)__popc(wm));
      at = __shfl_sync(FULL, at, __ffs(wm) - 1);
      if (aside == 1u) a.wide_list[at + __popc(wm & ((1u << lane) - 1u))] = i;
    }
    if (aside == 2u) a.slow_list[atomicAdd(&a.status->slow_count, 1u)] = i;
  }
  const uint32_t cnt = fast ? nbc : 0u;
  uint16_t* const col = &w.nl[0][lane];  // entry k of this lane's neighbour list: col[32 * k]
  if (__any_sync(FULL, cnt != 0u)) {
    // the neighbour list of this lane: staged rows in canonical order (slice 0, 1, 2; ascending row)
    uint32_t n = 0;
#define RCS_TILE_COMPACT(M, Q)                                                  \
    for (uint32_t bits = fast ? (M) : 0u; bits; bits &= bits - 1u) {            \
      col[32u * n] = (uint16_t)((Q) + (uint32_t)(__ffs(bits) - 1));             \
      n += 1u;                                                                  \
    }
    RCS_TILE_COMPACT(m0, q0)
    RCS_TILE_COMPACT(m1, q1)
    RCS_TILE_COMPACT(m2, q2)
#undef RCS_TILE_COMPACT
    __syncwarp();
  }
  const uint32_t maxc = __reduce_max_sync(FULL, cnt);
  // RCS_TILE_PHASED (experiment, off): the warps of a block go through the stages together, so that fewer stages'
  // code is live in the SM's instruction cache at a time -- the hot path is ~2000 instructions, 9 % of the fetches
  // miss.  Measured: slower (the barriers cost more than the misses), profiles/r02_step_tile_kernel.md.
#if RCS_TILE_PHASED
  __syncthreads();
#endif
  uint32_t y = 0;
  if (maxc) {
    // ---- stage 2: t_i = min over the list of time_to_collision (zanlungo.rs:76-91); y = entries with the higher id
    w.tbits[lane] = 0x7ff0000000000000ull;
    __syncwarp();
    // the division-free half of time_to_collision for staged row j; same operations as rcs_math.cuh
    auto probe = [&](bool v, double2 c, double2 cv, unsigned long long oid, uint32_t k, uint32_t& y) -> bool {
      y |= (v && me.id < oid) ? (1u << k) : 0u;
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
    // Pairs that may return a finite time are queued per warp; slots come from ballots (no atomics, and the count is a
    // register the whole warp agrees on, so nothing is read back from shared memory inside the loop).
    uint32_t n_hit = 0;
    const uint32_t lt = (1u << lane) - 1u;
    // list entries are fetched one iteration ahead (their shared-memory latency is off the dependent chain)
    uint32_t jA_n = cnt > 0u ? col[0] : 0u, jB_n = cnt > 1u ? col[32u] : 0u;
    for (uint32_t k = 0; k < maxc; k += 2) {
      const bool vA = k < cnt, vB = k + 1u < cnt;
      const uint32_t jA = jA_n, jB = jB_n;
      jA_n = k + 2u < cnt ? col[32u * k + 64u] : 0u;
      jB_n = k + 3u < cnt ? col[32u * k + 96u] : 0u;
      const bool hitA = probe(vA, spos[jA], svel[jA], sid[jA], k, y);
      const bool hitB = probe(vB, spos[jB], svel[jB], sid[jB], k + 1u, y);
      const unsigned bA = __ballot_sync(FULL, hitA), bB = __ballot_sync(FULL, hitB);
      if (hitA) {  // order inside the list is irrelevant (min)
        const uint32_t p = n_hit + __popc(bA & lt);
        w.lj[p] = (uint16_t)jA;
        w.lo[p] = (uint8_t)lane;
      }
      if (hitB) {
        const uint32_t p = n_hit + __popc(bA) + __popc(bB & lt);
        w.lj[p] = (uint16_t)jB;
        w.lo[p] = (uint8_t)lane;
      }
      n_hit += __popc(bA) + __popc(bB);
      if (n_hit > 2u * ST_CAP - 64u) {  // at most 64 new entries per round
        __syncwarp();
        st_flush_hits(w, n_hit, spos, svel, lane, me.px, me.py, me.vx, me.vy, rr);
        n_hit = 0u;
      }
    }
    __syncwarp();
    if (n_hit) st_flush_hits(w, n_hit, spos, svel, lane, me.px, me.py, me.vx, me.vy, rr);
    __syncwarp();
    if (fast) t_i = __longlong_as_double((long long)w.tbits[lane]);
  }
#if RCS_TILE_PHASED
  __syncthreads();
#endif
  if (maxc) {
    // ---- stage 3: force sum over the list of owners with a finite t_i (zanlungo.rs:210-215)
    const bool fin = fast && (t_i != RCS_INF);
    if (__any_sync(FULL, fin)) {
      OwnerPre pre;
      pre.futx = pre.futy = pre.mag = pre.mvx = pre.mvy = pre.f0x = pre.f0y = 0.0;
      uint32_t ya = 0u, za = 0u;  // yield entries (evaluate) / weight-0 entries (prove zero) of the list
      w.poison[lane] = 0u;
      if (fin) {
        pre = owner_precompute(me.px, me.py, me.vx, me.vy, me.pfx, me.pfy, t_i, a.groups[grp]);
        ya = y;
        za = ~y & (cnt >= 32u ? 0xffffffffu : ((1u << cnt) - 1u));
      }
      // Every owner's pairs take one contiguous segment of a list, in list order, so the owner later adds its own
      // slots front to back.  Segment offsets come from one warp scan of the per-lane counts (yield list in the low
      // half-word, weight-0 list in the high one).
      const uint32_t cA = __popc(ya), cB = __popc(za);
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
        const bool fits = lane >= lane_begin && offA + cA <= ST_CAP && offB + cB <= ST_CAP;
        const unsigned okm = __ballot_sync(FULL, fits || lane < lane_begin);
        const uint32_t lane_end = (okm == FULL) ? 32u : (uint32_t)(__ffs(~okm) - 1);  // > lane_begin: cA, cB <= 32
        const bool part = lane >= lane_begin && lane < lane_end;
        if (part) {  // one walk over the list entries feeds both pair lists
          uint32_t pA = offA, pB = ST_CAP + offB;
          for (uint32_t bits = ya | za; bits;) {  // two entries per turn: their list reads are independent
            const uint32_t k0 = (uint32_t)(__ffs(bits) - 1);
            bits &= bits - 1u;
            const bool two = bits != 0u;
            const uint32_t k1 = two ? (uint32_t)(__ffs(bits) - 1) : k0;
            bits &= bits - 1u;  // 0 stays 0
            const uint16_t e0 = col[32u * k0], e1 = col[32u * k1];
            const bool y0 = ((ya >> k0) & 1u) != 0u, y1 = ((ya >> k1) & 1u) != 0u;
            const uint32_t p0 = y0 ? pA : pB;
            w.lj[p0] = e0;
            w.lo[p0] = (uint8_t)lane;
            pA += y0 ? 1u : 0u;
            pB += y0 ? 0u : 1u;
            if (two) {
              const uint32_t p1 = y1 ? pA : pB;
              w.lj[p1] = e1;
              w.lo[p1] = (uint8_t)lane;
              pA += y1 ? 1u : 0u;
              pB += y1 ? 0u : 1u;
            }
          }
        }
        const uint32_t tot = __shfl_sync(FULL, inc, lane_end - 1) - base;
        const uint32_t nA = tot & 0xffffu, nB = tot >> 16;
        __syncwarp();
        for (uint32_t b = 0; b < nA; b += 32) {  // yield pairs: one per lane
          const uint32_t e = b + lane;
          const bool v = e < nA;
          const uint32_t o = v ? w.lo[e] : lane;
          const uint32_t j = v ? w.lj[e] : 0u;
          OwnerPre op;
          op.futx = st_shfl(pre.futx, o);
          op.futy = st_shfl(pre.futy, o);
          op.mag = st_shfl(pre.mag, o);
          const double opx = st_shfl(me.px, o), opy = st_shfl(me.py, o), ovx = st_shfl(me.vx, o),
                       ovy = st_shfl(me.vy, o), oti = st_shfl(t_i, o);
          const uint32_t ogrp = __shfl_sync(FULL, grp, (int)o);
          if (v) {
            double qx, qy;
            const double2 c = spos[j], cv = svel[j];
            pair_force_yield(op, opx, opy, ovx, ovy, c.x, c.y, cv.x, cv.y, oti, a.groups[ogrp], qx, qy);
            w.sf[e] = make_double2(qx, qy);
          }
        }
        for (uint32_t b = 0; b < nB; b += 32) {  // weight-0 pairs: prove the contribution is (+-0, +-0)
          const uint32_t e = b + lane;
          const bool v = e < nB;
          const uint32_t o = v ? w.lo[ST_CAP + e] : lane;
          const uint32_t j = v ? w.lj[ST_CAP + e] : 0u;
          OwnerPre op;
          op.mvx = st_shfl(pre.mvx, o);
          op.mvy = st_shfl(pre.mvy, o);
          op.f0x = st_shfl(pre.f0x, o);
          op.f0y = st_shfl(pre.f0y, o);
          const double oti = st_shfl(t_i, o);
          bool lit = false;
          double2 c = make_double2(0.0, 0.0), cv = c;
          if (v) {
            c = spos[j];
            cv = svel[j];
            lit = !pair_force_w0_is_zero(op, c.x, c.y, cv.x, cv.y, oti);
          }
          if (__any_sync(FULL, lit))
            st_w0_literal(w, a.groups, lit, o, c, cv, v ? sid[j] : 0ull, me.px, me.py, me.vx, me.vy, me.pfx, me.pfy, me.id,
                          grp, oti);
        }
        __syncwarp();
        if (part) {
          uint32_t r = 0;
          for (; r + 1u < cA; r += 2u) {  // same order of additions, two loads in flight
            const double2 q0 = w.sf[offA + r], q1 = w.sf[offA + r + 1u];
            fx = fx + q0.x;
            fy = fy + q0.y;
            fx = fx + q1.x;
            fy = fy + q1.y;
          }
          if (r < cA) {
            const double2 q = w.sf[offA + r];
            fx = fx + q.x;
            fy = fy + q.y;
          }
        }
        __syncwarp();
        lane_begin = lane_end;
      }
      const unsigned pz = w.poison[lane];
      if (pz & 1u) fx = fx + __longlong_as_double(0x7ff8000000000000LL);
      if (pz & 2u) fy = fy + __longlong_as_double(0x7ff8000000000000LL);
    }
  }

#if RCS_TILE_PHASED
  __syncthreads();
#endif
  if (active) {
    const GroupDev& g = a.groups[grp];
    if (zan) {
      // zanlungo.rs:216
      velx = velx + fx * g.inv_mass;
      vely = vely + fy * g.inv_mass;
    }
    integrate_and_store<STRIPS>(a, i, me, g, grp, wp_in, role, velx, vely, t_i, fx, fy, nbc);
  }
  if (a.collect_stats) {  // per owned agent, so that the totals add up over ranks; one set of atomics per block
    const bool own = active && (role & ROLE_MASK) == ROLE_OWN;
    const uint32_t c = __reduce_add_sync(FULL, own ? cand : 0u);
    const uint32_t nb = __reduce_add_sync(FULL, own ? nbc : 0u);
    const uint32_t ft = __reduce_add_sync(FULL, (own && zan && t_i != RCS_INF) ? 1u : 0u);
    if (lane == 0) {
      if (c) atomicAdd(&sh.stat[0], c);
      if (nb) atomicAdd(&sh.stat[1], nb);
      if (ft) atomicAdd(&sh.stat[2], ft);
    }
    __syncthreads();
    if (threadIdx.x == 0) {
      if (sh.stat[0]) atomicAdd(&a.status->candidate_total, (unsigned long long)sh.stat[0]);
      if (sh.stat[1]) atomicAdd(&a.status->neighbour_total, (unsigned long long)sh.stat[1]);
      if (sh.stat[2]) atomicAdd(&a.status->finite_tti, (unsigned long long)sh.stat[2]);
    }
  }
}

}  // namespace rcs
