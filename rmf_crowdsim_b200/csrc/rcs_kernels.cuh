// rcs_kernels.cuh -- CUDA kernels of the per-step pipeline (sm_100a).
//
//   bin_count -> scan (3 small kernels, warp-shuffle scans) -> scatter_perm -> sort_cells_by_id
//   -> gather_sorted -> step_kernel (radius query + Zanlungo + explicit Euler, fused)
//
// Data layout: structure of arrays -- double2 positions, double2 velocities, u64 ids, u32 group / waypoint --
// physically re-sorted every step into canonical (cell index, agent id) order, so the reference's
// scan `for x in left..=right { for y in bottom..=top }` (location_hash_2d.rs:245-246) is, for each
// x, one contiguous slice of the sorted arrays (the cell index is x-major, :59).
#pragma once

#include "rcs_math.cuh"

namespace rcs {

struct DevStatus {
  unsigned int oob_count;
  unsigned int nonfinite_count;
  unsigned int big_cells;       // cells with more agents than SORT_LOCAL_MAX (handled by the slow sorter)
  unsigned int failed;          // sticky: a previous async step failed (on ANY rank) -> later steps are skipped
  unsigned int local_failed;    // this rank's own verdict for the current step (input of the consensus)
  unsigned int halo_err;        // strips: an owned agent moved further than the halo in one step
  unsigned int capacity_err;    // spawn / ghost append / event buffers ran out of room
  unsigned int spawned;         // agents spawned by source sinks in this step
  unsigned int destroyed;       // agents removed at sinks in this step
  unsigned int slow_count;      // agents left to the sequential routine (tail of step_aside_kernel)
  unsigned int wide_count;      // agents handed to step_aside_kernel's cooperative part (wide or crowded stencils)
  unsigned int sort_ticket;     // sort_big_cells_kernel: blocks done with a grid-ranked cell (returns to 0)
  unsigned long long first_oob_id;
  unsigned long long finite_tti;
  unsigned long long neighbour_total;
  unsigned long long candidate_total;
};

// device-side agent counts (the host only knows upper bounds while steps with churn are in flight)
enum : int { CNT_CUR = 0, CNT_TOT = 1, CNT_SAVE = 2, CNT_EV_SPAWN = 3, CNT_EV_DESTROY = 4, CNT_EV_SPAWN_SAVE = 5,
             CNT_EV_DESTROY_SAVE = 6, CNT_N = 8 };

// one source sink on the device (source_sink.rs:36-60 + the per-step logic of lib.rs:199-254, 305-336)
struct SourceSinkDev {
  double sx, sy;            // source
  double rate;              // MonotonicCrowd::rate (source_sink.rs:85-100)
  double thr2_sink;         // smallest double T with sqrt(T) >= radius_sink
  long long pl, pr, pb, pt; // get_bounds(0.4, source): stencil of the spawn probe (lib.rs:212-214)
  uint32_t wp_off, n_wp;    // waypoints in the shared waypoint table
  uint32_t grp;             // group of the agents it spawns
  uint32_t loop_forever;
  uint32_t alive;           // 0 after remove_source_sink
  uint32_t owned;           // strips: this rank owns the source's cell column and spawns for it (1 on a single handle)
};

// spatial strips (SURVEY.md section 8e): this rank owns cell columns [c0, c1); h = halo ring width
struct StripDev {
  uint32_t enabled;
  uint32_t c0, c1, h;   // own columns [c0, c1); ring width h (columns advanced redundantly on both sides)
  uint32_t lc0, rc1;    // the left neighbour owns [lc0, c0), the right one [c1, rc1)
  uint32_t reach;       // rows / columns a radius query can touch beyond the agent's own cell
  uint32_t pad_;
};

// Structure of arrays with the two f64 components of a vector interleaved, so that every position / velocity
// moves with one 16-byte access.
// Strips: a halo buffer is [count u32, failed u32, pad to 64 B][pos][vel][id][meta][pv], each `cap` entries.
// Packed order is arbitrary (atomic append); the receiver re-sorts.
struct HaloBuf {
  uint32_t* count;
  double2 *pos, *vel;
  unsigned long long* id;
  unsigned long long* meta;  // grp | wp << 32
  double2* pv;
  uint32_t cap;
};

struct AgentArrays {
  double2 *pos, *vel;
  uint64_t* id;
  uint32_t *grp, *wp;
  double2* pv;  // host-planner preferred velocities; NaN in .x = None.  nullptr if no host planner exists
};

// Programmatic dependent launch (RCS_OPT_PDL): the kernels of a step are launched with
// cudaLaunchAttributeProgrammaticStreamSerialization, so the blocks of kernel k + 1 are dispatched while kernel k is
// still running and sit in griddepcontrol.wait until k has completed and its stores are visible -- the launch latency
// between the dozen small kernels of a step overlaps instead of adding up.  pdl_enter() is the FIRST statement of every
// kernel launched that way, executed by every thread (a block that left without it would let its grid complete, and the
// next grid start, before the previous one is done).  Without the launch attribute both instructions do nothing.
__device__ __forceinline__ void pdl_enter() {
  asm volatile("griddepcontrol.launch_dependents;");
  asm volatile("griddepcontrol.wait;" ::: "memory");
}

// Halo packing fused into the binning pass over the owned agents of a strip: an agent whose insert cell lies in
// the outermost `width` columns is appended to the send buffer of that side (both, on a very narrow strip).
struct PackArgs {
  uint32_t enabled;
  uint32_t nx, width;
  int has_left, has_right;
  StripDev st;
  HaloBuf left, right;
  AgentArrays cur;
  const uint32_t* xseq;  // peer-store transport: exchange round (its parity picks the half of the neighbour's buffer)
};

// Strips: agent i of the owned agents sits in cell `idx`; if that is one of the outermost `width` columns of the
// strip it is appended to the send buffer of that side (both, on a very narrow strip).
__device__ __forceinline__ void halo_pack_one(const PackArgs& pk, uint32_t i, uint32_t idx, DevStatus* status) {
  const uint32_t cx = idx / pk.nx;
  const unsigned act = __activemask();  // the lanes that reached this call together
  const unsigned lane = threadIdx.x & 31u;
  const uint32_t par = pk.xseq ? (*pk.xseq & 1u) : 0u;
#pragma unroll
  for (int side = 0; side < 2; ++side) {
    const bool send = side == 0 ? (pk.has_left && cx < pk.st.c0 + pk.width) : (pk.has_right && cx + pk.width >= pk.st.c1);
    // One append per warp, not per agent: the boundary columns are contiguous in storage, so whole warps pack, and
    // 50 000 atomics on one counter were a third of the binning pass (27 us per rank on 8 strips).
    const unsigned m = __ballot_sync(act, send);
    if (!m) continue;
    const HaloBuf& b = side == 0 ? pk.left : pk.right;
    const int leader = __ffs(m) - 1;
    uint32_t base = 0;
    if ((int)lane == leader) base = atomicAdd(b.count, (unsigned)__popc(m));
    base = __shfl_sync(act, base, leader);
    if (!send) continue;
    uint32_t k = base + __popc(m & ((1u << lane) - 1u));
    if (k >= b.cap) {
      atomicAdd(&status->capacity_err, 1u);
      continue;
    }
    k += par * b.cap;  // peer-store transport: the rows go straight into the neighbour's receive buffer
    b.pos[k] = pk.cur.pos[i];
    b.vel[k] = pk.cur.vel[i];
    b.id[k] = pk.cur.id[i];
    b.meta[k] = (unsigned long long)pk.cur.grp[i] | ((unsigned long long)pk.cur.wp[i] << 32);
    if (pk.cur.pv) b.pv[k] = pk.cur.pv[i];
  }
}

// The same for a whole block of the binning pass (every thread of the block calls it, `mine` = this thread has an agent
// to test): ONE append per block and side.  The boundary columns are contiguous in storage, so ~100 blocks per side
// pack; with one atomic per warp the 770 same-address atomics per side were most of the pass's extra time on 8 strips.
template <int THREADS>
__device__ __forceinline__ void halo_pack_block(const PackArgs& pk, bool mine, uint32_t i, uint32_t idx,
                                                DevStatus* status) {
  constexpr int NW = THREADS / 32;
  __shared__ uint32_t s_cnt[2][NW];
  __shared__ uint32_t s_base[2];
  const unsigned lane = threadIdx.x & 31u, warp = threadIdx.x >> 5;
  const uint32_t par = pk.xseq ? (*pk.xseq & 1u) : 0u;
  const uint32_t cx = idx / pk.nx;
  const bool send0 = mine && pk.has_left && cx < pk.st.c0 + pk.width;
  const bool send1 = mine && pk.has_right && cx + pk.width >= pk.st.c1;
  const unsigned m0 = __ballot_sync(0xffffffffu, send0), m1 = __ballot_sync(0xffffffffu, send1);
  if (lane == 0) {
    s_cnt[0][warp] = __popc(m0);
    s_cnt[1][warp] = __popc(m1);
  }
  __syncthreads();
  if (threadIdx.x < 2) {
    uint32_t tot = 0;
#pragma unroll
    for (int w = 0; w < NW; ++w) tot += s_cnt[threadIdx.x][w];
    s_base[threadIdx.x] = tot ? atomicAdd(threadIdx.x == 0 ? pk.left.count : pk.right.count, tot) : 0u;
  }
  __syncthreads();
#pragma unroll
  for (int side = 0; side < 2; ++side) {
    if (!(side == 0 ? send0 : send1)) continue;
    const HaloBuf& b = side == 0 ? pk.left : pk.right;
    uint32_t k = s_base[side] + __popc((side == 0 ? m0 : m1) & ((1u << lane) - 1u));
    for (unsigned w = 0; w < warp; ++w) k += s_cnt[side][w];
    if (k >= b.cap) {
      atomicAdd(&status->capacity_err, 1u);
      continue;
    }
    k += par * b.cap;  // peer-store transport: the rows go straight into the neighbour's receive buffer
    b.pos[k] = pk.cur.pos[i];
    b.vel[k] = pk.cur.vel[i];
    b.id[k] = pk.cur.id[i];
    b.meta[k] = (unsigned long long)pk.cur.grp[i] | ((unsigned long long)pk.cur.wp[i] << 32);
    if (pk.cur.pv) b.pv[k] = pk.cur.pv[i];
  }
}

// Strips, when the previous step's epilogue has already binned the owned agents (cellid, histogram): only the halo
// pack of the binning pass is left to do.
__global__ void halo_pack_kernel(uint32_t n_ub, const uint32_t* __restrict__ last, const uint32_t* __restrict__ cellid,
                                 PackArgs pk, DevStatus* status) {
  if (status->failed) return;
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n_ub || i >= *last) return;
  const uint32_t c = cellid[i];
  if (c != 0xffffffffu) halo_pack_one(pk, i, c, status);
}

constexpr int SCAN_THREADS = 256;
constexpr int SCAN_ITEMS = 16;
constexpr int SCAN_TILE = SCAN_THREADS * SCAN_ITEMS;
constexpr int SORT_LOCAL_MAX = 32;
constexpr uint32_t CELL_DEAD = 0xffffffffu;
constexpr int BIN_THREADS = 256;  // block size of bin_count_kernel

// ---------------------------------------------------------------------------------------------
// A1/A2: cell of every agent (LocationHash2D::location_to_index) + histogram.
// ---------------------------------------------------------------------------------------------
// Files agent i (position p) under its insert cell: cellid[i] and the histogram.  False: not indexed (cellid = dead).
__device__ __forceinline__ bool bin_one(const GridDev& g, uint32_t i, double2 p, uint32_t* __restrict__ cellid,
                                        uint32_t* __restrict__ cell_count, uint64_t cell_lo, uint64_t cell_hi,
                                        DevStatus* status, uint64_t& idx) {
  if (!location_to_index(g, p.x, p.y, idx)) {
    // only reachable through snapshot injection; steps never commit an out-of-bounds position
    cellid[i] = CELL_DEAD;
    atomicAdd(&status->oob_count, 1u);
    return false;
  }
  if (idx < cell_lo || idx >= cell_hi) {
    // strips index only the cells of their own columns and halo; an agent elsewhere (possible only through the
    // row aliasing of location_hash_2d.rs:59 far above the grid) cannot be handled by this rank
    cellid[i] = CELL_DEAD;
    atomicAdd(&status->halo_err, 1u);
    return false;
  }
  cellid[i] = (uint32_t)idx;
  // The agents arrive in last step's canonical order, so the lanes of a warp fall into a handful of cells: one
  // atomic per distinct cell of the warp instead of one per agent.
  const unsigned peers = __match_any_sync(__activemask(), (uint32_t)idx);
  if ((threadIdx.x & 31u) == (unsigned)(__ffs(peers) - 1)) atomicAdd(&cell_count[idx], (unsigned)__popc(peers));
  return true;
}

// Agents [*first (0 if null), min(n_ub, *last)) of the unsorted arrays.  Entries whose keep flag is 0 (despawned
// at a sink, migrated to another strip, ghosts of the previous step) are dropped here: the counting sort of the
// next step is the stream compaction.
// PACK: the strip form (every thread of a block reaches the block-wide halo append); the plain form leaves early and
// keeps the registers for 2048 resident threads (the pass is latency-bound on its loads and atomics).
template <bool PACK>
__global__ void __launch_bounds__(BIN_THREADS, 8) bin_count_kernel(
    GridDev g, uint32_t n_ub, const uint32_t* __restrict__ first, const uint32_t* __restrict__ last,
    const double2* __restrict__ pos, const uint32_t* __restrict__ keep, uint32_t* __restrict__ cellid,
    uint32_t* __restrict__ cell_count, uint64_t cell_lo, uint64_t cell_hi, PackArgs pk, DevStatus* status) {
  pdl_enter();
  if (status->failed) return;
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x + (first ? *first : 0u);
  bool live = i < n_ub && i < *last;
  if (!PACK && !live) return;
  if (live && keep && !keep[i]) {
    cellid[i] = CELL_DEAD;
    live = false;
    if (!PACK) return;
  }
  uint64_t idx = 0;
  if (live) live = bin_one(g, i, pos[i], cellid, cell_count, cell_lo, cell_hi, status, idx);
  if (PACK) halo_pack_block<BIN_THREADS>(pk, live, i, (uint32_t)idx, status);  // (the whole block gets here)
}

// ---------------------------------------------------------------------------------------------
// Exclusive prefix sum over the cell histogram: reduce tiles -> scan tile sums -> scan tiles.
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t warp_inclusive_scan(uint32_t v) {
  const unsigned lane = threadIdx.x & 31u;
#pragma unroll
  for (int d = 1; d < 32; d <<= 1) {
    uint32_t t = __shfl_up_sync(0xffffffffu, v, d);
    if (lane >= (unsigned)d) v += t;
  }
  return v;
}

// exclusive scan of one value per thread across a SCAN_THREADS block; block total in `total`
__device__ __forceinline__ uint32_t block_exclusive_scan(uint32_t v, uint32_t& total) {
  constexpr int NW = SCAN_THREADS / 32;
  __shared__ uint32_t warp_off[NW];
  __shared__ uint32_t s_total;
  const unsigned lane = threadIdx.x & 31u, warp = threadIdx.x >> 5;
  uint32_t inc = warp_inclusive_scan(v);
  if (lane == 31) warp_off[warp] = inc;
  __syncthreads();
  if (warp == 0) {
    uint32_t w = lane < NW ? warp_off[lane] : 0u;
    uint32_t winc = warp_inclusive_scan(w);
    if (lane < NW) warp_off[lane] = winc - w;
    if (lane == NW - 1) s_total = winc;
  }
  __syncthreads();
  total = s_total;
  uint32_t r = warp_off[warp] + inc - v;
  __syncthreads();  // the shared scratch may be reused by the caller's next scan
  return r;
}

__global__ void scan_reduce_kernel(const uint32_t* __restrict__ in, uint64_t len, uint32_t* __restrict__ tile_sums) {
  pdl_enter();
  uint64_t base = (uint64_t)blockIdx.x * SCAN_TILE + (uint64_t)threadIdx.x * SCAN_ITEMS;
  uint32_t s = 0;
  if (base + SCAN_ITEMS <= len) {
    const uint4* p = reinterpret_cast<const uint4*>(in + base);
#pragma unroll
    for (int k = 0; k < SCAN_ITEMS / 4; ++k) {
      uint4 v = p[k];
      s += v.x + v.y + v.z + v.w;
    }
  } else {
    for (int k = 0; k < SCAN_ITEMS; ++k)
      if (base + k < len) s += in[base + k];
  }
  uint32_t total;
  (void)block_exclusive_scan(s, total);
  if (threadIdx.x == 0) tile_sums[blockIdx.x] = total;
}

// single block: in-place exclusive scan of the tile sums; writes the grand total to *total_out
__global__ void scan_tile_sums_kernel(uint32_t* __restrict__ tile_sums, uint32_t n_tiles, uint32_t* total_out) {
  uint32_t carry = 0;
  for (uint32_t base = 0; base < n_tiles; base += SCAN_THREADS) {
    uint32_t i = base + threadIdx.x;
    uint32_t v = i < n_tiles ? tile_sums[i] : 0u;
    uint32_t total;
    uint32_t ex = block_exclusive_scan(v, total);
    if (i < n_tiles) tile_sums[i] = carry + ex;
    carry += total;
    __syncthreads();
  }
  if (threadIdx.x == 0) *total_out = carry;
}

// writes cell_start[c] (exclusive) and cursor[c] (= cell_start[c], bumped by the scatter); the
// thread that owns the last element also writes cell_start[len] = total.
// RAW_SUMS: tile_sums holds the tiles' totals as scan_reduce_kernel left them and every block adds up the ones before
// its own (a few thousand tiles at most: one launch less than scanning them first).
template <bool RAW_SUMS>
__global__ void scan_apply_kernel(const uint32_t* __restrict__ in, uint64_t len,
                                  const uint32_t* __restrict__ tile_sums, uint32_t* __restrict__ cell_start,
                                  uint32_t* __restrict__ cursor) {
  pdl_enter();
  uint64_t base = (uint64_t)blockIdx.x * SCAN_TILE + (uint64_t)threadIdx.x * SCAN_ITEMS;
  uint32_t v[SCAN_ITEMS];
  uint32_t s = 0;
  if (base + SCAN_ITEMS <= len) {
    const uint4* p = reinterpret_cast<const uint4*>(in + base);
#pragma unroll
    for (int k = 0; k < SCAN_ITEMS / 4; ++k) {
      uint4 q = p[k];
      v[4 * k + 0] = q.x;
      v[4 * k + 1] = q.y;
      v[4 * k + 2] = q.z;
      v[4 * k + 3] = q.w;
    }
  } else {
#pragma unroll
    for (int k = 0; k < SCAN_ITEMS; ++k) v[k] = (base + k < len) ? in[base + k] : 0u;
  }
#pragma unroll
  for (int k = 0; k < SCAN_ITEMS; ++k) s += v[k];
  uint32_t total, before;
  if (RAW_SUMS) {
    uint32_t part = 0;
    for (uint32_t t = threadIdx.x; t < blockIdx.x; t += SCAN_THREADS) part += tile_sums[t];
    (void)block_exclusive_scan(part, before);
  } else {
    before = tile_sums[blockIdx.x];
  }
  uint32_t run = before + block_exclusive_scan(s, total);
  if (base + SCAN_ITEMS <= len) {
    uint32_t o[SCAN_ITEMS];
#pragma unroll
    for (int k = 0; k < SCAN_ITEMS; ++k) {
      o[k] = run;
      run += v[k];
    }
    uint4* ps = reinterpret_cast<uint4*>(cell_start + base);
    uint4* pc = reinterpret_cast<uint4*>(cursor + base);
#pragma unroll
    for (int k = 0; k < SCAN_ITEMS / 4; ++k) {
      uint4 q = make_uint4(o[4 * k], o[4 * k + 1], o[4 * k + 2], o[4 * k + 3]);
      ps[k] = q;
      if (cursor) pc[k] = q;
    }
    if (base + SCAN_ITEMS == len) cell_start[len] = run;
  } else {
    for (int k = 0; k < SCAN_ITEMS; ++k) {
      if (base + k < len) {
        cell_start[base + k] = run;
        if (cursor) cursor[base + k] = run;
        run += v[k];
        if (base + k + 1 == len) cell_start[len] = run;
      }
    }
  }
}

// ---------------------------------------------------------------------------------------------
// A2: counting-sort scatter of a permutation (slot order inside a cell is fixed by the next kernel)
// ---------------------------------------------------------------------------------------------
__global__ void scatter_perm_kernel(uint32_t n_ub, const uint32_t* __restrict__ n_ptr,
                                    const uint32_t* __restrict__ cellid, uint32_t* __restrict__ cursor,
                                    uint32_t* __restrict__ perm, const DevStatus* status) {
  pdl_enter();
  if (status->failed) return;
  uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n_ub || i >= *n_ptr) return;
  uint32_t c = cellid[i];
  if (c == CELL_DEAD) return;
  uint32_t pos = atomicAdd(&cursor[c], 1u);  // (one atomic per distinct cell of the warp was measured: 1.5 x slower)
  perm[pos] = i;
}

// Canonical order inside a cell = ascending agent id (the reference's HashSet order is random per
// process; SURVEY.md section 7).  One thread per cell; insertion sort of the cell's permutation
// slice keyed by id.  Cells larger than SORT_LOCAL_MAX go to the block-wide rank sorter.
__global__ void sort_cells_by_id_kernel(uint64_t cell_lo, uint64_t cell_hi, const uint32_t* __restrict__ cell_start,
                                        const uint64_t* __restrict__ id, uint32_t* __restrict__ perm,
                                        uint32_t* __restrict__ big_list, uint32_t big_cap, DevStatus* status) {
  pdl_enter();
  if (status->failed) return;
  uint64_t c = cell_lo + (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= cell_hi) return;
  uint32_t s = cell_start[c], e = cell_start[c + 1];
  uint32_t m = e - s;
  if (m < 2) return;
  if (m > SORT_LOCAL_MAX) {
    uint32_t k = atomicAdd(&status->big_cells, 1u);
    if (k < big_cap) big_list[k] = (uint32_t)c;
    return;
  }
  uint32_t p[SORT_LOCAL_MAX];
  uint64_t key[SORT_LOCAL_MAX];
  bool sorted = true;
  for (uint32_t k = 0; k < m; ++k) {
    p[k] = perm[s + k];
    key[k] = id[p[k]];
    if (k && key[k] < key[k - 1]) sorted = false;
  }
  if (sorted) return;
  for (uint32_t k = 1; k < m; ++k) {
    uint32_t pk = p[k];
    uint64_t kk = key[k];
    int j = (int)k - 1;
    while (j >= 0 && key[j] > kk) {
      key[j + 1] = key[j];
      p[j + 1] = p[j];
      --j;
    }
    key[j + 1] = kk;
    p[j + 1] = pk;
  }
  for (uint32_t k = 0; k < m; ++k) perm[s + k] = p[k];
}

// One block per oversized cell: rank = number of smaller ids (ids are unique), O(m^2 / threads) compares against
// keys staged in shared memory, BIG_SMEM_KEYS at a time.  Cells beyond that size -- in practice cell 0, where the
// reference files every agent whose position went non-finite -- are ranked by the whole grid (rank_huge_cell).
// The cells come from big_list; if more cells were oversized than the list holds (big_cells > big_cap) every
// block sweeps a share of ALL cells instead, whatever their size (ranks accumulate tile by tile in `ranks`).
constexpr uint32_t BIG_SMEM_KEYS = 4096;

__device__ __forceinline__ void sort_one_big_cell(uint32_t s, uint32_t e, const uint64_t* __restrict__ id,
                                                  uint32_t* __restrict__ perm, uint32_t* __restrict__ scratch,
                                                  uint32_t* __restrict__ ranks, unsigned long long* skeys) {
  const uint32_t m = e - s;
  for (uint32_t t0 = 0; t0 < m; t0 += BIG_SMEM_KEYS) {
    const uint32_t tl = min(BIG_SMEM_KEYS, m - t0);
    __syncthreads();
    for (uint32_t j = threadIdx.x; j < tl; j += blockDim.x) skeys[j] = id[perm[s + t0 + j]];
    __syncthreads();
    for (uint32_t k = threadIdx.x; k < m; k += blockDim.x) {  // a thread only ever touches its own entries of ranks
      const uint64_t kk = id[perm[s + k]];
      uint32_t rank = t0 ? ranks[s + k] : 0u;
      for (uint32_t j = 0; j < tl; ++j) rank += (skeys[j] < kk) ? 1u : 0u;
      ranks[s + k] = rank;
    }
  }
  for (uint32_t k = threadIdx.x; k < m; k += blockDim.x) scratch[s + ranks[s + k]] = perm[s + k];
  __syncthreads();
  for (uint32_t k = s + threadIdx.x; k < e; k += blockDim.x) perm[k] = scratch[k];
  __syncthreads();
}

// A cell beyond the shared-memory tile, ranked by the whole grid: a block takes HUGE_ELEMS elements at a time, its
// 32 warps split the keys of every tile between them (all lanes of a warp read the same key: a broadcast), partial
// ranks are added up in shared memory.  Results go to scratch; the block that finishes last copies them back.
constexpr uint32_t HUGE_ELEMS = 64;

__device__ __forceinline__ void rank_huge_cell(uint32_t s, uint32_t e, const uint64_t* __restrict__ id,
                                               const uint32_t* __restrict__ perm, uint32_t* __restrict__ scratch,
                                               unsigned long long* skeys, uint32_t (*partial)[HUGE_ELEMS]) {
  const uint32_t m = e - s;
  const uint32_t warp = threadIdx.x >> 5, lane = threadIdx.x & 31u, nwarps = blockDim.x >> 5;
  for (uint32_t k0 = blockIdx.x * HUGE_ELEMS; k0 < m; k0 += gridDim.x * HUGE_ELEMS) {  // block-uniform
    const uint32_t kA = k0 + lane, kB = k0 + lane + 32u;
    const uint64_t keyA = kA < m ? id[perm[s + kA]] : 0ull, keyB = kB < m ? id[perm[s + kB]] : 0ull;
    uint32_t rA = 0, rB = 0;
    for (uint32_t t0 = 0; t0 < m; t0 += BIG_SMEM_KEYS) {
      const uint32_t tl = min(BIG_SMEM_KEYS, m - t0);
      __syncthreads();
      for (uint32_t j = threadIdx.x; j < tl; j += blockDim.x) skeys[j] = id[perm[s + t0 + j]];
      __syncthreads();
      for (uint32_t j = warp; j < tl; j += nwarps) {
        const uint64_t key = skeys[j];
        rA += (key < keyA) ? 1u : 0u;
        rB += (key < keyB) ? 1u : 0u;
      }
    }
    partial[warp][lane] = rA;
    partial[warp][lane + 32u] = rB;
    __syncthreads();
    if (threadIdx.x < HUGE_ELEMS && k0 + threadIdx.x < m) {
      uint32_t rank = 0;
      for (uint32_t w = 0; w < nwarps; ++w) rank += partial[w][threadIdx.x];
      scratch[s + rank] = perm[s + k0 + threadIdx.x];
    }
    __syncthreads();
  }
}

__global__ void __launch_bounds__(1024) sort_big_cells_kernel(uint64_t cell_lo, uint64_t cell_hi,
                                                              const uint32_t* __restrict__ cell_start,
                                                              const uint64_t* __restrict__ id,
                                                              uint32_t* __restrict__ perm,
                                                              uint32_t* __restrict__ scratch,
                                                              uint32_t* __restrict__ ranks,
                                                              const uint32_t* __restrict__ big_list, uint32_t big_cap,
                                                              DevStatus* status) {
  pdl_enter();
  __shared__ unsigned long long skeys[BIG_SMEM_KEYS];
  __shared__ uint32_t partial[32][HUGE_ELEMS];
  __shared__ bool last_block;
  if (status->failed) return;
  const uint32_t nbig = status->big_cells;
  if (nbig <= big_cap) {
    for (uint32_t b = blockIdx.x; b < nbig; b += gridDim.x) {  // one block per cell that fits a tile
      const uint32_t c = big_list[b];
      const uint32_t cs = cell_start[c], ce = cell_start[c + 1];
      if (ce - cs <= BIG_SMEM_KEYS) sort_one_big_cell(cs, ce, id, perm, scratch, ranks, skeys);
    }
    uint32_t n_huge = 0;
    for (uint32_t b = 0; b < nbig; ++b) {  // every block: the same cells in the same order
      const uint32_t c = big_list[b];
      const uint32_t cs = cell_start[c], ce = cell_start[c + 1];
      if (ce - cs > BIG_SMEM_KEYS) {
        rank_huge_cell(cs, ce, id, perm, scratch, skeys, partial);
        n_huge += 1;
      }
    }
    if (n_huge) {
      __threadfence();
      __syncthreads();
      if (threadIdx.x == 0) last_block = atomicAdd(&status->sort_ticket, 1u) == gridDim.x - 1;
      __syncthreads();
      if (last_block) {  // every block's ranks are in scratch
        __threadfence();
        for (uint32_t b = 0; b < nbig; ++b) {
          const uint32_t c = big_list[b];
          const uint32_t cs = cell_start[c], ce = cell_start[c + 1];
          if (ce - cs > BIG_SMEM_KEYS)
            for (uint32_t k = cs + threadIdx.x; k < ce; k += blockDim.x) perm[k] = __ldcg(scratch + k);
        }
        if (threadIdx.x == 0) status->sort_ticket = 0u;
      }
    }
  } else {
    for (uint64_t c = cell_lo + blockIdx.x; c < cell_hi; c += gridDim.x) {  // block-uniform bounds
      const uint32_t cs = cell_start[c], ce = cell_start[c + 1];
      if (ce - cs > SORT_LOCAL_MAX) sort_one_big_cell(cs, ce, id, perm, scratch, ranks, skeys);
    }
  }
}

// Physical reorder into canonical order: sorted[k] = cur[perm[k]].  This kernel is HBM-bound with idle issue
// slots, so it also prepares the radius query of every Zanlungo agent for the hot kernel: the (at most three)
// candidate slices of the sorted arrays, one per stencil column (get_bounds + signed_idx_to_data_idx,
// location_hash_2d.rs:74-122), as {start0, start1, start2, len0 | len1 << 8 | len2 << 16 | ok << 24}.
// ok = 0: the stencil is wider than three columns (the agent takes the sequential routine); lengths saturate
// at 255.
__device__ __forceinline__ uint4 query_slices(const GridDev& g, const uint32_t* __restrict__ cell_start,
                                              const GroupDev& gr, double px, double py) {
  uint4 sl = make_uint4(0u, 0u, 0u, 0u);
  if (gr.lp_kind == LP_ZANLUNGO) {
    int64_t left, right, bottom, top;
    get_bounds(g, gr.eyesight, px, py, left, right, bottom, top);
    if (left < 0) left = 0;
    if (right > g.x_max) right = g.x_max;
    if (right - left <= 2) {
      uint32_t st[3] = {0, 0, 0}, ln[3] = {0, 0, 0};
#pragma unroll
      for (int c = 0; c < 3; ++c) {
        uint64_t c_lo, c_hi;
        if (left + c <= right && column_cell_range(g, left + c, bottom, top, c_lo, c_hi)) {
          st[c] = cell_start[c_lo];
          const uint32_t l = cell_start[c_hi + 1] - st[c];
          ln[c] = l > 255u ? 255u : l;
        }
      }
      sl = make_uint4(st[0], st[1], st[2], ln[0] | (ln[1] << 8) | (ln[2] << 16) | (1u << 24));
    }
  }
  return sl;
}

// Staging ranges of one block of step_tile_kernel (rcs_step_tile.cuh): the union of its agents' slices per stencil
// column.  Written here, by the block that gathers the same GATHER_THREADS agents.
// Ranges start and end at even rows (the id rows are 8 bytes; bulk copies move multiples of 16 bytes from 16-byte
// aligned addresses).  A block whose ranges hold more rows than its staging buffer does not stage.
struct TileRange {
  uint32_t lo[3];   // first sorted row of the range of stencil column d (even)
  uint32_t len[3];  // rows (even); 0 = no agent of the block has such a slice
};
__device__ __forceinline__ bool st_takes(const GroupDev& g, uint64_t id, uint4 sl);
__device__ __forceinline__ void st_block_ranges(bool takes, uint4 sl, uint32_t (*red)[6], TileRange* out);
#ifndef RCS_TILE_WARPS
#define RCS_TILE_WARPS 4
#endif
constexpr int ST_WARPS = RCS_TILE_WARPS;       // warps per block of step_tile_kernel
constexpr int GATHER_THREADS = 32 * ST_WARPS;  // == block size of step_tile_kernel

// One sorted slot per thread; positions and velocities move as 16-byte elements.  The arrays being gathered are
// last step's sorted output and agents rarely change cell, so perm is close to the identity and the reads coalesce.
__global__ void __launch_bounds__(GATHER_THREADS) gather_sorted_kernel(
    uint32_t n, const uint32_t* __restrict__ perm, AgentArrays cur, AgentArrays srt, const uint32_t* __restrict__ cellid,
    uint32_t* __restrict__ srt_cell, const uint32_t* __restrict__ n_sorted, GridDev g,
    const uint32_t* __restrict__ cell_start, const GroupDev* __restrict__ groups, uint4* __restrict__ slices,
    TileRange* __restrict__ tile_ranges, const DevStatus* status) {
  pdl_enter();
  __shared__ uint32_t red[GATHER_THREADS / 32][6];
  if (status->failed) return;  // block-uniform
  const uint32_t k = blockIdx.x * blockDim.x + threadIdx.x;
  bool takes = false;
  uint4 sl = make_uint4(0u, 0u, 0u, 0u);
  if (k < n && k < *n_sorted) {
    const uint32_t i = perm[k];
    const double2 p = cur.pos[i];
    const uint32_t grp = cur.grp[i];
    const uint64_t id = cur.id[i];
    if (srt_cell) srt_cell[k] = cellid[i];
    srt.pos[k] = p;
    srt.vel[k] = cur.vel[i];
    srt.id[k] = id;
    srt.grp[k] = grp;
    srt.wp[k] = cur.wp[i];
    if (cur.pv) srt.pv[k] = cur.pv[i];
    if (slices) {
      sl = query_slices(g, cell_start, groups[grp], p.x, p.y);
      slices[k] = sl;
      takes = st_takes(groups[grp], id, sl);
    }
  }
  if (tile_ranges) st_block_ranges(takes, sl, red, tile_ranges + blockIdx.x);
}

// ---------------------------------------------------------------------------------------------
// The hot kernel: lib.rs:259-347 for every agent at once (deferred index semantic).
// ---------------------------------------------------------------------------------------------
struct StepArgs {
  GridDev grid;
  uint32_t n;                 // upper bound on live (sorted) agents
  const uint32_t* n_sorted;   // device-side exact count (= cell_start[len])
  AgentArrays in;             // canonical (cell, id) order
  const uint32_t* cell_start; // len + 1
  const GroupDev* groups;
  double dt;                  // Duration::as_secs_f64 (lib.rs:295)
  double2 *opos, *ovel;        // new state, same order
  uint64_t* oid;              // id / group / waypoint / host preferred velocity of the new state
  uint32_t *ogrp, *owp;       //   (all nullptr on the streaming path, which updates x,y,vx,vy in place)
  double2* opv;
  double *t_i, *fx, *fy;      // optional trace outputs (nullptr when tracing is off)
  uint32_t* nb_count;         // optional: neighbour count per agent (trace)
  uint64_t* tr_id;            // optional: id of the agent in each trace slot
  uint32_t* tr_own;           // optional: 1 if the slot holds an agent this rank owns and advanced
  DevStatus* status;
  uint32_t collect_stats;
  uint32_t no_commit;         // RCS_STEP_NO_COMMIT: keep flags select the owned pre-step agents
  const unsigned long long* steps_done;  // device step counter (stamps destroy events)
  // churn: agents that leave (sink reached, lib.rs:318-323; strip ownership) get keep = 0
  uint32_t* keep;                  // nullptr when nothing can leave
  const uint32_t* cell;            // insert cell of every sorted agent (strips)
  StripDev strip;
  const SourceSinkDev* ss;         // nullptr when there are no source sinks
  const double* ss_wp;             // waypoint table, interleaved x,y
  uint32_t* cnt;                   // device counters (CNT_*)
  unsigned long long* ev_destroyed;  // (id, step) pairs of agents removed at sinks
  uint32_t ev_cap;
  uint32_t* slow_list;             // warp kernel: agents left to the sequential routine
  uint32_t* wide_list;             // warp kernel: agents left to the chunked cooperative routine
  const uint4* slices;             // candidate slices prepared by gather_sorted_kernel (sorted path only)
  const TileRange* tile_ranges;    // per block of step_tile_kernel: rows to stage (gather_sorted_kernel)
  // Binning ahead: the epilogue files every agent that stays under the cell of the position the NEXT step starts
  // from (A1 / A2 of that step: cell id + histogram), so that step's rebuild starts at the prefix sum.
  uint32_t* next_cellid;           // nullptr: off
  uint32_t* next_count;
  uint64_t cell_lo, cell_hi;       // cells this handle indexes
  const double* routes;            // HL_ROUTE polylines, interleaved x,y
  double route_thr2;               // smallest double T with sqrt(T) >= 1e-1 (rmf/mod.rs:202)
};

// next_waypoint (lib.rs:61) lives in the low half of the per-agent `wp` word; the high half is the agent's entry
// in the route follower's agent_cache (rmf/mod.rs:86): 0 = absent, k + 1 = heading for route point k.
constexpr uint32_t WP_MASK = 0xffffu;
constexpr int WP_ROUTE_SHIFT = 16;

enum : uint32_t { ROLE_PASSIVE = 0, ROLE_OWN = 1, ROLE_RING = 2, ROLE_MASK = 3,
                  // optional, for integrate_and_store: the old column lies within h of the left / right boundary
                  ROLE_NEAR_L = 1u << 8, ROLE_NEAR_R = 1u << 9, ROLE_HAS_NEAR = 1u << 10 };

// Strips: an agent is advanced by the rank that owns its column AND, redundantly and bit-identically,
// by the neighbour rank that holds it in the inner halo ring (so migration needs no message).
__device__ __forceinline__ uint32_t agent_role_of_cell(const StepArgs& a, uint32_t cell) {
  if (!a.strip.enabled) return ROLE_OWN;
  const uint32_t cx = cell / (uint32_t)a.grid.nx;
  if (cx >= a.strip.c0 && cx < a.strip.c1) return ROLE_OWN;
  if (cx + a.strip.h >= a.strip.c0 && cx < a.strip.c1 + a.strip.h) return ROLE_RING;
  return ROLE_PASSIVE;
}
// ... with the boundary bits, so that the epilogue needs neither the cell nor a second division
__device__ __forceinline__ uint32_t agent_role_and_bits(const StepArgs& a, uint32_t cell) {
  const uint32_t cx = cell / (uint32_t)a.grid.nx;
  uint32_t r = ROLE_PASSIVE;
  if (cx >= a.strip.c0 && cx < a.strip.c1) r = ROLE_OWN;
  else if (cx + a.strip.h >= a.strip.c0 && cx < a.strip.c1 + a.strip.h) r = ROLE_RING;
  if (cx < a.strip.c0 + a.strip.h) r |= ROLE_NEAR_L;
  if (cx + a.strip.h >= a.strip.c1) r |= ROLE_NEAR_R;
  return r | ROLE_HAS_NEAR;
}
__device__ __forceinline__ uint32_t agent_role(const StepArgs& a, uint32_t i) {
  return a.strip.enabled ? agent_role_of_cell(a, a.cell[i]) : (uint32_t)ROLE_OWN;
}

// An entry of the sorted arrays that this rank does not advance (ghost beyond the ring, slot beyond the live count):
// it is not part of the next state.
__device__ __forceinline__ void drop_entry(const StepArgs& a, uint32_t i) {
  if (a.keep) a.keep[i] = 0u;
  if (a.next_cellid) a.next_cellid[i] = CELL_DEAD;
}

struct Self {
  double px, py, vx, vy, pfx, pfy;
  uint64_t id;
  uint32_t rwp;  // route follower entry after this step's get_desired_velocity (HL_ROUTE only)
};

// Walks the reference's radius query for one agent and calls f(j) for every neighbour j that
// passes the strict distance filter (location_hash_2d.rs:251) and the self filter (lib.rs:284),
// in canonical order.  Returns the number of candidates distance-tested.
template <class F>
__device__ __forceinline__ uint32_t for_each_neighbour(const GridDev& g, const uint32_t* __restrict__ cell_start,
                                                       const double2* __restrict__ pos,
                                                       const uint64_t* __restrict__ ids, double px, double py,
                                                       uint64_t self_id, double radius, double thr2, F&& f) {
  int64_t left, right, bottom, top;
  get_bounds(g, radius, px, py, left, right, bottom, top);
  if (left < 0) left = 0;
  if (right > g.x_max) right = g.x_max;
  uint32_t cand = 0;
  for (int64_t cx = left; cx <= right; ++cx) {
    uint64_t c_lo, c_hi;
    if (!column_cell_range(g, cx, bottom, top, c_lo, c_hi)) continue;
    uint32_t s = cell_start[c_lo], e = cell_start[c_hi + 1];
    cand += e - s;
    for (uint32_t j = s; j < e; ++j) {
      const double2 q = pos[j];
      double dx = q.x - px;
      double dy = q.y - py;
      double d2 = dx * dx + dy * dy;
      if (d2 < thr2) {
        if (ids[j] != self_id) f(j, dx, dy, d2);
      }
    }
  }
  return cand;
}

// Zanlungo::get_desired_velocity (zanlungo.rs:201-218) for ONE agent, sequentially, in canonical
// neighbour order: t_i (compute_tti) then the force sum.  The reference form of the hot path; the
// warp-cooperative kernel must reproduce its results bit for bit and uses it for agents whose
// stencil does not fit its fast path.
__device__ __noinline__ void zanlungo_sequential(const StepArgs& a, uint32_t i, const Self& me, const GroupDev& g,
                                                 double& t_i, double& fx, double& fy, uint32_t& nbc,
                                                 uint32_t& cand) {
  const double2* __restrict__ pos = a.in.pos;
  const double2* __restrict__ vel = a.in.vel;
  const uint64_t* __restrict__ ids = a.in.id;
  const double rr = g.rr;
  t_i = RCS_INF;
  fx = 0.0;
  fy = 0.0;
  // Zanlungo::compute_tti, zanlungo.rs:76-91
  cand = for_each_neighbour(a.grid, a.cell_start, pos, ids, me.px, me.py, me.id, g.eyesight, g.thr2,
                            [&](uint32_t j, double dx, double dy, double d2) {
                              nbc++;
                              const double2 nv = vel[j];
                              double col_time = time_to_collision(nv.x - me.vx, nv.y - me.vy, dx, dy, d2, rr);
                              if (col_time < t_i) t_i = col_time;
                            });
  // zanlungo.rs:210-215
  if (t_i != RCS_INF) {
    const OwnerPre pre = owner_precompute(me.px, me.py, me.vx, me.vy, me.pfx, me.pfy, t_i, g);
    const double ti = t_i;
    for_each_neighbour(a.grid, a.cell_start, pos, ids, me.px, me.py, me.id, g.eyesight, g.thr2,
                       [&](uint32_t j, double, double, double) {
                         double qx, qy;
                         const double2 np = pos[j], nv = vel[j];
                         if (pair_force_dispatch(pre, me.px, me.py, me.vx, me.vy, me.pfx, me.pfy, me.id, np.x, np.y,
                                                 nv.x, nv.y, ids[j], ti, g, qx, qy)) {
                           fx = fx + qx;
                           fy = fy + qy;
                         }
                       });
  }
}

// HighLevelPlanner::get_desired_velocity on the device (lib.rs:263-273): returns the recommended
// velocity and sets me.pfx/pfy (the clone's preferred_vel, lib.rs:271).
__device__ __forceinline__ void high_level_velocity(const StepArgs& a, uint32_t i, const GroupDev& g, Self& me,
                                                    double& velx, double& vely) {
  velx = 0.0;
  vely = 0.0;
  me.pfx = 0.0;
  me.pfy = 0.0;
  switch (g.hl_kind) {
    case HL_CONSTANT:
      velx = g.hl_vx;
      vely = g.hl_vy;
      me.pfx = velx;
      me.pfy = vely;
      break;
    case HL_PARITY:
      if ((me.id & 1ull) == 0ull) {
        velx = -g.hl_vx;
        vely = -g.hl_vy;
      } else {
        velx = g.hl_vx;
        vely = g.hl_vy;
      }
      me.pfx = velx;
      me.pfy = vely;
      break;
    case HL_ROUTE: {
      // the per-step half of RMFPlanner::get_desired_velocity (rmf/mod.rs:197-215) on a caller-supplied route
      uint32_t rw = a.in.wp[i] >> WP_ROUTE_SHIFT;
      if (rw != 0u) {  // in agent_cache
        uint32_t wid = rw - 1u;
        const double* r = a.routes + 2 * (size_t)g.route_off;
        double dx = me.px - r[2 * wid], dy = me.py - r[2 * wid + 1];
        if (dx * dx + dy * dy < a.route_thr2 && g.route_n > wid + 1u) {  // (pos - route[wp]).norm() < 1e-1
          wid += 1u;
          rw += 1u;
        }
        dx = r[2 * wid] - me.px;
        dy = r[2 * wid + 1] - me.py;
        const double nrm = sqrt(dx * dx + dy * dy);
        velx = dx / nrm;  // normalize(): component-wise division by the norm
        vely = dy / nrm;
        me.pfx = velx;
        me.pfy = vely;
      }
      me.rwp = rw;
    } break;
    case HL_HOST: {
      const double2 hv = a.in.pv[i];
      double hx = hv.x, hy = hv.y;
      if (hx == hx) {  // NaN in x encodes None
        velx = hx;
        vely = hy;
        me.pfx = hx;
        me.pfy = hy;
      }
    } break;
    default:
      break;
  }
}

// Explicit Euler + commit outputs + error accounting (lib.rs:295-302), then the waypoint / sink test on
// the OLD position (lib.rs:305-336) and, for strips, the ownership decision by the NEW position.
// MAY_STRIP = false: the caller knows the handle is no strip (the strip bookkeeping is compiled out).
template <bool MAY_STRIP = true>
__device__ __forceinline__ void integrate_and_store(const StepArgs& a, uint32_t i, const Self& me, const GroupDev& g,
                                                    uint32_t grp, uint32_t wp_in, uint32_t role, double velx,
                                                    double vely, double t_i, double fx, double fy, uint32_t nbc) {
  const double nx = me.px + velx * a.dt;
  const double ny = me.py + vely * a.dt;
  a.opos[i] = make_double2(nx, ny);
  a.ovel[i] = make_double2(velx, vely);
  const bool own = (role & ROLE_MASK) == ROLE_OWN;
  if (a.t_i) {
    a.t_i[i] = t_i;
    a.fx[i] = fx;
    a.fy[i] = fy;
    a.nb_count[i] = nbc;
    a.tr_id[i] = me.id;
    a.tr_own[i] = own ? 1u : 0u;
  }
  // add_or_update(new_pos) error path, lib.rs:299-302
  const uint64_t x_idx = f64_as_usize(div_floor(nx - a.grid.offx, a.grid));
  const uint64_t y_idx = f64_as_usize(div_floor(ny - a.grid.offy, a.grid));
  const uint64_t idx = x_idx * a.grid.nx + y_idx;
  const bool inb = idx < a.grid.len;
  if (!inb && own) {
    atomicAdd(&a.status->oob_count, 1u);
    atomicMin(&a.status->first_oob_id, (unsigned long long)me.id);
  }
  if (own && !(isfinite(nx) && isfinite(ny) && isfinite(velx) && isfinite(vely)))
    atomicAdd(&a.status->nonfinite_count, 1u);
  if (!a.oid) return;  // streaming path: x,y,vx,vy only
  uint32_t wp = wp_in & WP_MASK;
  uint32_t rwp = g.hl_kind == HL_ROUTE ? me.rwp : (wp_in >> WP_ROUTE_SHIFT);
  bool keep = true;
  if (a.ss && g.source_sink >= 0) {
    const SourceSinkDev& ss = a.ss[g.source_sink];
    if (ss.alive && wp < ss.n_wp) {
      const double ddx = me.px - a.ss_wp[2 * (ss.wp_off + wp)];
      const double ddy = me.py - a.ss_wp[2 * (ss.wp_off + wp) + 1];
      if (ddx * ddx + ddy * ddy < ss.thr2_sink) {  // (position - waypoint).norm() < radius_sink, lib.rs:314
        if (wp == ss.n_wp - 1) {
          if (ss.loop_forever) {
            wp = 0;
          } else {
            keep = false;  // to_be_removed: still moved and committed this step, removed after (lib.rs:378)
            if (own && !a.no_commit) {
              const uint32_t k = atomicAdd(&a.cnt[CNT_EV_DESTROY], 1u);
              if (k < a.ev_cap) {
                a.ev_destroyed[2 * k] = me.id;
                a.ev_destroyed[2 * k + 1] = *a.steps_done;
              } else {
                atomicAdd(&a.status->capacity_err, 1u);
              }
              atomicAdd(&a.status->destroyed, 1u);
            }
          }
        } else {
          wp += 1;
          // HighLevelPlanner::set_target(.., waypoints[next_waypoint], ..) (lib.rs:326-333): the route follower
          // starts over at the head of its route (rmf/mod.rs:217-237 inserts (route, 0))
          if (g.hl_kind == HL_ROUTE) rwp = 1u;
        }
      }
    }
  }
  a.oid[i] = me.id;
  a.ogrp[i] = grp;
  a.owp[i] = wp | (rwp << WP_ROUTE_SHIFT);
  if (a.opv) a.opv[i] = a.in.pv[i];
  if (MAY_STRIP && a.strip.enabled) {
    // The agent stays with the rank that owns its NEW column.  Every agent that leaves a strip must have
    // been in the neighbour's ring (old column within h of the boundary) and must land inside the
    // neighbour's strip; otherwise no rank would keep it.
    const bool mine = inb && x_idx >= a.strip.c0 && x_idx < a.strip.c1;
    if (own && inb && !mine) {
      bool near_l = (role & ROLE_NEAR_L) != 0u, near_r = (role & ROLE_NEAR_R) != 0u;
      if (!(role & ROLE_HAS_NEAR)) {
        const uint32_t ocx = a.cell[i] / (uint32_t)a.grid.nx;
        near_l = ocx < a.strip.c0 + a.strip.h;
        near_r = ocx + a.strip.h >= a.strip.c1;
      }
      const bool ok = x_idx < a.strip.c0 ? (near_l && x_idx >= a.strip.lc0) : (near_r && x_idx < a.strip.rc1);
      if (!ok) atomicAdd(&a.status->halo_err, 1u);
    }
    // a query from the top `reach` rows of the grid runs over into the NEXT column's bottom cells (y_idx >= n_x
    // aliases, location_hash_2d.rs:74-85), which may lie beyond this rank's halo: refuse rather than be inexact
    if (own && inb && y_idx + a.strip.reach >= a.grid.nx) atomicAdd(&a.status->halo_err, 1u);
    keep = keep && mine;
  }
  if (a.no_commit) keep = own;  // the pre-step snapshot stays: this rank keeps exactly what it owned
  if (a.keep) a.keep[i] = keep ? 1u : 0u;
  if (a.next_cellid) {
    // location_to_index (A1) of the position the next step starts from: the new one, or -- without commit -- the old
    uint64_t c = idx;
    bool cin = inb;
    if (a.no_commit) cin = location_to_index(a.grid, me.px, me.py, c);
    if (keep && cin && c >= a.cell_lo && c < a.cell_hi) {
      a.next_cellid[i] = (uint32_t)c;
      atomicAdd(&a.next_count[c], 1u);
    } else {
      a.next_cellid[i] = CELL_DEAD;
      if (keep && cin) atomicAdd(&a.status->halo_err, 1u);  // outside the cells this rank indexes (bin_count_kernel)
    }
  }
}

__device__ __forceinline__ void warp_stats(const StepArgs& a, uint32_t cand, uint32_t nbc, uint32_t finite) {
  if (!a.collect_stats) return;
  // hardware warp reductions; a per-agent count above 2^27 would be needed to overflow 32 bits
  const uint32_t c = __reduce_add_sync(0xffffffffu, cand);
  const uint32_t nb = __reduce_add_sync(0xffffffffu, nbc);
  const uint32_t ft = __reduce_add_sync(0xffffffffu, finite);
  if ((threadIdx.x & 31) == 0) {
    if (c) atomicAdd(&a.status->candidate_total, (unsigned long long)c);
    if (nb) atomicAdd(&a.status->neighbour_total, (unsigned long long)nb);
    if (ft) atomicAdd(&a.status->finite_tti, (unsigned long long)ft);
  }
}

// One agent, sequentially: high-level velocity, Zanlungo, Euler.  Body of the thread-per-agent kernel
// and of the kernel that finishes the agents the warp-cooperative kernel left aside.
__device__ __forceinline__ void step_one_agent(const StepArgs& a, uint32_t i, uint32_t& cand, uint32_t& nbc,
                                               uint32_t& finite) {
  const uint32_t role = agent_role(a, i);
  if (role == ROLE_PASSIVE) {
    drop_entry(a, i);
    return;
  }
  const GroupDev& g = a.groups[a.in.grp[i]];
  Self me;
  const double2 p0 = a.in.pos[i], v0 = a.in.vel[i];
  me.px = p0.x;
  me.py = p0.y;
  me.vx = v0.x;
  me.vy = v0.y;
  me.id = a.in.id[i];
  me.rwp = 0u;
  double velx, vely;
  high_level_velocity(a, i, g, me, velx, vely);
  double t_i = RCS_INF, fx = 0.0, fy = 0.0;
  uint32_t c = 0, nb = 0;
  if (g.lp_kind == LP_ZANLUNGO) {
    zanlungo_sequential(a, i, me, g, t_i, fx, fy, nb, c);
    // zanlungo.rs:216
    velx = velx + fx * g.inv_mass;
    vely = vely + fy * g.inv_mass;
  }
  integrate_and_store(a, i, me, g, a.in.grp[i], a.oid ? a.in.wp[i] : 0u, role, velx, vely, t_i, fx, fy, nb);
  if (role == ROLE_OWN) {  // statistics are per owned agent so that they add up over ranks
    cand += c;
    nbc += nb;
    finite += (g.lp_kind == LP_ZANLUNGO && t_i != RCS_INF) ? 1u : 0u;
  }
}

// Thread-per-agent form of the hot kernel (also the streaming kernel of NoLocalPlan-only crowds).
__global__ void __launch_bounds__(128) step_kernel(StepArgs a) {
  if (a.status->failed) return;
  uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  uint32_t n_live = *a.n_sorted;
  uint32_t cand = 0, nbc = 0, finite = 0;
  if (i < a.n && i < n_live) step_one_agent(a, i, cand, nbc, finite);
  else if (i < a.n) drop_entry(a, i);
  warp_stats(a, cand, nbc, finite);
}

// NoLocalPlan-only crowds without churn (no_local_plan.rs:10-17: the local planner returns the recommended
// velocity, no query can influence the result): lib.rs:259-347 degenerates to a stream over the agents in storage
// order -- high-level velocity, explicit Euler, add_or_update's bounds check.  Two agents per thread with 16-byte
// accesses; 64 algorithmic bytes per agent (SURVEY.md section 8d), HBM-bound.  Same operations as step_one_agent.
__device__ __forceinline__ void stream_one(const StepArgs& a, const GroupDev& g, double px, double py, uint64_t id,
                                           double hx, double hy, double& nx, double& ny, double& velx, double& vely) {
  velx = 0.0;
  vely = 0.0;
  switch (g.hl_kind) {
    case HL_CONSTANT:
      velx = g.hl_vx;
      vely = g.hl_vy;
      break;
    case HL_PARITY:
      velx = (id & 1ull) == 0ull ? -g.hl_vx : g.hl_vx;
      vely = (id & 1ull) == 0ull ? -g.hl_vy : g.hl_vy;
      break;
    case HL_HOST:
      if (hx == hx) {  // NaN in x encodes None
        velx = hx;
        vely = hy;
      }
      break;
    default:
      break;
  }
  nx = px + velx * a.dt;
  ny = py + vely * a.dt;
  const uint64_t x_idx = f64_as_usize(div_floor(nx - a.grid.offx, a.grid));
  const uint64_t y_idx = f64_as_usize(div_floor(ny - a.grid.offy, a.grid));
  if (!(x_idx * a.grid.nx + y_idx < a.grid.len)) {
    atomicAdd(&a.status->oob_count, 1u);
    atomicMin(&a.status->first_oob_id, (unsigned long long)id);
  }
  if (!(isfinite(nx) && isfinite(ny) && isfinite(velx) && isfinite(vely))) atomicAdd(&a.status->nonfinite_count, 1u);
}

__global__ void __launch_bounds__(256) step_stream_kernel(StepArgs a) {
  const uint32_t i = (blockIdx.x * blockDim.x + threadIdx.x) * 2u;
  if (i >= a.n) return;
  const bool pair = i + 1u < a.n;  // every array holds at least a.n entries
  // two agents per thread: 32 bytes of positions, 16 of ids, 8 of groups per access
  double4 pp;
  ulonglong2 p_id;
  uint2 p_g;
  double4 hh = make_double4(0.0, 0.0, 0.0, 0.0);
  if (pair) {
    pp = *reinterpret_cast<const double4*>(a.in.pos + i);
    p_id = *reinterpret_cast<const ulonglong2*>(a.in.id + i);
    p_g = *reinterpret_cast<const uint2*>(a.in.grp + i);
    if (a.in.pv) hh = *reinterpret_cast<const double4*>(a.in.pv + i);
  } else {
    const double2 p = a.in.pos[i];
    pp = make_double4(p.x, p.y, 0.0, 0.0);
    p_id = make_ulonglong2(a.in.id[i], 0ull);
    p_g = make_uint2(a.in.grp[i], 0u);
    if (a.in.pv) {
      const double2 h = a.in.pv[i];
      hh = make_double4(h.x, h.y, 0.0, 0.0);
    }
  }
  if (a.status->failed) return;
  const uint32_t n_live = *a.n_sorted;
  if (i >= n_live) return;
  double4 op = pp, ov = make_double4(0.0, 0.0, 0.0, 0.0);
  stream_one(a, a.groups[p_g.x], pp.x, pp.y, p_id.x, hh.x, hh.y, op.x, op.y, ov.x, ov.y);
  if (pair && i + 1u < n_live) {
    stream_one(a, a.groups[p_g.y], pp.z, pp.w, p_id.y, hh.z, hh.w, op.z, op.w, ov.z, ov.w);
    *reinterpret_cast<double4*>(a.opos + i) = op;
    *reinterpret_cast<double4*>(a.ovel + i) = ov;
  } else {
    a.opos[i] = make_double2(op.x, op.y);
    a.ovel[i] = make_double2(ov.x, ov.y);
  }
}

// Trace: neighbour ids in list order (lib.rs:281-286) as CSR, offsets from an exclusive scan of nb_count.
__global__ void trace_neighbours_kernel(StepArgs a, const uint32_t* __restrict__ nb_offsets,
                                        uint64_t* __restrict__ nb_ids) {
  uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= a.n || i >= *a.n_sorted) return;
  if (agent_role(a, i) == ROLE_PASSIVE) return;  // never advanced: no list (its nb_count stays 0)
  const GroupDev& g = a.groups[a.in.grp[i]];
  if (g.lp_kind != LP_ZANLUNGO) return;
  uint32_t o = nb_offsets[i];
  const double2 p0 = a.in.pos[i];
  for_each_neighbour(a.grid, a.cell_start, a.in.pos, a.in.id, p0.x, p0.y, a.in.id[i], g.eyesight,
                     g.thr2, [&](uint32_t j, double, double, double) { nb_ids[o++] = a.in.id[j]; });
}

// SpatialIndex::get_neighbours_in_radius for arbitrary query points (location_hash_2d.rs:240-258).
// mode 0: count into counts[q]; mode 1: write ids at offsets[q].  No self filter.
__global__ void query_radius_kernel(GridDev g, const uint32_t* __restrict__ cell_start,
                                    const double2* __restrict__ pos, const uint64_t* __restrict__ ids, uint32_t nq,
                                    const double* __restrict__ qxy, const double* __restrict__ radius,
                                    const double* __restrict__ thr2, uint32_t* __restrict__ counts,
                                    const uint64_t* __restrict__ offsets, uint64_t* __restrict__ out_ids, int mode) {
  uint32_t q = blockIdx.x * blockDim.x + threadIdx.x;
  if (q >= nq) return;
  double px = qxy[2 * q], py = qxy[2 * q + 1];
  uint32_t cnt = 0;
  uint64_t o = mode ? offsets[q] : 0;
  // ids are < 2^63 in practice; ~0 never matches an agent so the self filter is a no-op here
  for_each_neighbour(g, cell_start, pos, ids, px, py, ~0ull, radius[q], thr2[q],
                     [&](uint32_t j, double, double, double) {
                       if (mode) out_ids[o++] = ids[j];
                       cnt++;
                     });
  if (!mode) counts[q] = cnt;
}

// ---------------------------------------------------------------------------------------------
// SpatialIndex::get_nearest_neighbours (location_hash_2d.rs:151-238), batched.  The ring walk is the
// reference's, quirks included: the four side loops are half-open, so cell (x-s, y-s) is visited twice
// and cell (x+s, y+s) never; the walk stops after the first ring that brings the candidate count to n
// (not a true kNN); candidates are then STABLY sorted by distance (sort_by + partial_cmp, :226-230).
// f(c) is called for every valid data cell in visiting order and returns the number of agents in it.
//
// The side bounds x_idx +- step and y_idx +- step wrap in two's complement, as release-mode Rust computes them: a
// saturated query cell (x = +inf, or >= 2^63 cells away) leaves the sides whose upper bound wrapped EMPTY.  So the
// visits are counted, not assumed to be 8*step, and a ring whose visits were all out of bounds ends the walk, an empty
// ring included.  Termination: counting the visits makes this walk the reference's, ring for ring.  Away from
// saturation a ring at Chebyshev distance step eventually has every cell at a negative coordinate or past the data;
// for a saturated x the only side that can reach the grid is the column x_idx - step, whose wrapped data index drops
// by nx per step while its row window grows by one, so it leaves [0, len).  A side loop runs at most 2*step times
// (i < hi, so i + 1 never overflows).
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ int64_t wrapping_add_i64(int64_t a, int64_t b) {
  return (int64_t)((uint64_t)a + (uint64_t)b);
}
__device__ __forceinline__ int64_t wrapping_sub_i64(int64_t a, int64_t b) {
  return (int64_t)((uint64_t)a - (uint64_t)b);
}

template <class F>
__device__ __forceinline__ uint64_t knn_walk(const GridDev& g, double px, double py, uint64_t n, F&& f) {
  const int64_t x_idx = f64_floor_as_i64(div_floor(px - g.offx, g));  // location_to_xy_signed_idx, :68-72
  const int64_t y_idx = f64_floor_as_i64(div_floor(py - g.offy, g));
  uint64_t have = 0;
  bool all_oob = false;
  auto visit = [&](int64_t cx, int64_t cy, uint64_t& oob, uint64_t& scanned) {
    // signed_idx_to_data_idx, :74-85
    bool ok = cx >= 0 && cy >= 0;
    uint64_t idx = 0;
    if (ok) {
      idx = (uint64_t)cx * g.nx + (uint64_t)cy;
      ok = idx < g.len;
    }
    if (ok) have += f(idx);
    else oob += 1;
    scanned += 1;
  };
  for (int64_t step = 0; have < n && !all_oob; ++step) {
    uint64_t oob = 0, scanned = 0;
    if (step == 0) {
      visit(x_idx, y_idx, oob, scanned);
    } else {
      const int64_t xl = wrapping_sub_i64(x_idx, step), xh = wrapping_add_i64(x_idx, step);
      const int64_t yl = wrapping_sub_i64(y_idx, step), yh = wrapping_add_i64(y_idx, step);
      for (int64_t i = xl; i < xh; ++i) visit(i, yh, oob, scanned);  // top line
      for (int64_t i = xl; i < xh; ++i) visit(i, yl, oob, scanned);  // bottom line
      for (int64_t i = yl; i < yh; ++i) visit(xl, i, oob, scanned);  // left line
      for (int64_t i = yl; i < yh; ++i) visit(xh, i, oob, scanned);  // right line
    }
    if (oob == scanned) all_oob = true;
  }
  return have;
}

// pass 0: counts[q] = number of candidates the walk collects (duplicates included)
__global__ void knn_count_kernel(GridDev g, const uint32_t* __restrict__ cell_start, uint32_t nq,
                                 const double* __restrict__ qxy, uint64_t k, uint32_t* __restrict__ counts) {
  uint32_t q = blockIdx.x * blockDim.x + threadIdx.x;
  if (q >= nq) return;
  uint64_t m = knn_walk(g, qxy[2 * q], qxy[2 * q + 1], k,
                        [&](uint64_t c) { return (uint64_t)(cell_start[c + 1] - cell_start[c]); });
  counts[q] = (uint32_t)m;
}

// pass 1: candidate slots and distances in visiting order (ascending id inside a cell)
__global__ void knn_fill_kernel(GridDev g, const uint32_t* __restrict__ cell_start,
                                const double2* __restrict__ pos, uint32_t nq, const double* __restrict__ qxy, uint64_t k,
                                const uint32_t* __restrict__ offsets, uint32_t* __restrict__ cand_slot,
                                double* __restrict__ cand_dist) {
  uint32_t q = blockIdx.x * blockDim.x + threadIdx.x;
  if (q >= nq) return;
  const double px = qxy[2 * q], py = qxy[2 * q + 1];
  uint32_t o = offsets[q];
  knn_walk(g, px, py, k, [&](uint64_t c) {
    const uint32_t s = cell_start[c], e = cell_start[c + 1];
    for (uint32_t j = s; j < e; ++j) {
      const double2 c = pos[j];
      const double dx = c.x - px, dy = c.y - py;
      cand_slot[o] = j;
      cand_dist[o] = sqrt(dx * dx + dy * dy);  // (a_pos - position).norm(), :227
      ++o;
    }
    return (uint64_t)(e - s);
  });
}

// pass 2: one warp per query; stable rank by distance, the first min(k, m) go out.  The rank is a permutation only
// under a total order: a NaN distance among >= 2 candidates is where the reference's partial_cmp(..).unwrap() panics
// (:226-230), so it sets *nan_flag instead and the host refuses the whole call.
__global__ void knn_select_kernel(uint32_t nq, uint64_t k, const uint32_t* __restrict__ offsets,
                                  const uint32_t* __restrict__ cand_slot, const double* __restrict__ cand_dist,
                                  const uint64_t* __restrict__ ids, uint64_t* __restrict__ out_ids,
                                  uint64_t* __restrict__ out_counts, uint32_t* __restrict__ nan_flag) {
  const uint32_t q = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const uint32_t lane = threadIdx.x & 31u;
  if (q >= nq) return;
  const uint32_t s = offsets[q], m = offsets[q + 1] - s;
  for (uint32_t t = lane; t < m; t += 32) {
    const double d = cand_dist[s + t];
    if (d != d && m >= 2) *nan_flag = 1u;
    uint32_t rank = 0;
    for (uint32_t u = 0; u < m; ++u) {
      const double du = cand_dist[s + u];
      rank += (du < d || (u < t && !(d < du))) ? 1u : 0u;  // stable: earlier equal elements stay first
    }
    if (rank < k) out_ids[(uint64_t)q * k + rank] = ids[cand_slot[s + t]];
  }
  if (lane == 0) out_counts[q] = m < k ? m : k;
}

// keep[i] = 1 for the sorted agents this rank owns (rollback of a failed step on a strip)
__global__ void role_keep_kernel(uint32_t n_ub, const uint32_t* __restrict__ n_ptr, const uint32_t* __restrict__ cell,
                                 uint32_t nx, StripDev st, uint32_t* __restrict__ keep) {
  uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n_ub) return;
  uint32_t k = 0;
  if (i < *n_ptr) {
    const uint32_t cx = cell[i] / nx;
    k = (cx >= st.c0 && cx < st.c1) ? 1u : 0u;
  }
  keep[i] = k;
}

__global__ void cell_of_kernel(GridDev g, uint32_t n, const double* __restrict__ xy, long long* __restrict__ out) {
  uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  uint64_t idx;
  out[i] = location_to_index(g, xy[2 * i], xy[2 * i + 1], idx) ? (long long)idx : -1ll;
}

// ---------------------------------------------------------------------------------------------
// id-addressed access (the reference's `agents: HashMap<AgentId, Agent>` view, lib.rs:71)
// ---------------------------------------------------------------------------------------------
__global__ void build_slot_of_id_kernel(uint32_t n, const uint64_t* __restrict__ id, uint32_t* __restrict__ slot_of_id,
                                        uint64_t table_len) {
  uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  uint64_t v = id[i];
  if (v < table_len) slot_of_id[v] = i;
}

// out[k] = slot of id ids[k], 0xffffffff if it is not live (the id -> slot table stays on the device)
__global__ void lookup_slots_kernel(uint32_t n, const uint64_t* __restrict__ ids, const uint32_t* __restrict__ slot_of_id,
                                    uint64_t table_len, uint32_t* __restrict__ out) {
  uint32_t k = blockIdx.x * blockDim.x + threadIdx.x;
  if (k >= n) return;
  const uint64_t v = ids[k];
  out[k] = v < table_len ? slot_of_id[v] : 0xffffffffu;
}

// largest live id (strips: agents migrate in with ids this handle never allocated)
__global__ void max_id_kernel(uint32_t n, const uint64_t* __restrict__ id, unsigned long long* out) {
  uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  unsigned long long v = i < n ? (unsigned long long)id[i] : 0ull;
#pragma unroll
  for (int d = 16; d > 0; d >>= 1) {
    unsigned long long o = __shfl_down_sync(0xffffffffu, v, d);
    v = o > v ? o : v;
  }
  if ((threadIdx.x & 31) == 0 && v) atomicMax(out, v);
}

// presence[v] = 1 if id v is live (input of the rank scan that yields ascending-id order)
__global__ void presence_kernel(uint64_t table_len, const uint32_t* __restrict__ slot_of_id,
                                uint32_t* __restrict__ presence) {
  uint64_t v = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (v >= table_len) return;
  presence[v] = slot_of_id[v] != 0xffffffffu ? 1u : 0u;
}

// order_by_id[rank] = slot, for rank = number of live ids smaller than v
__global__ void order_by_id_kernel(uint64_t table_len, const uint32_t* __restrict__ slot_of_id,
                                   const uint32_t* __restrict__ rank, uint32_t* __restrict__ order_by_id) {
  uint64_t v = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (v >= table_len) return;
  uint32_t s = slot_of_id[v];
  if (s != 0xffffffffu) order_by_id[rank[v]] = s;
}

// out[k] = src[order[k] * stride] (order == nullptr: identity); stride 2 picks one component of a double2 array
template <class T>
__global__ void gather_kernel(uint32_t n, const uint32_t* __restrict__ order, const T* __restrict__ src, int stride,
                              T* __restrict__ out) {
  uint32_t k = blockIdx.x * blockDim.x + threadIdx.x;
  if (k >= n) return;
  out[k] = src[(size_t)(order ? order[k] : k) * stride];
}

// x, y, vx, vy of agent order[k] (order == nullptr: identity) into up to four arrays: one 16-byte read per vector
// instead of one strided 8-byte read per component
__global__ void gather_state_kernel(uint32_t n, const uint32_t* __restrict__ order, const double2* __restrict__ pos,
                                    const double2* __restrict__ vel, double* __restrict__ x, double* __restrict__ y,
                                    double* __restrict__ vx, double* __restrict__ vy) {
  uint32_t k = blockIdx.x * blockDim.x + threadIdx.x;
  if (k >= n) return;
  const uint32_t i = order ? order[k] : k;
  if (x || y) {
    const double2 p = pos[i];
    if (x) x[k] = p.x;
    if (y) y[k] = p.y;
  }
  if (vx || vy) {
    const double2 v = vel[i];
    if (vx) vx[k] = v.x;
    if (vy) vy[k] = v.y;
  }
}

// dst[slot(k)] = src[k] where slot(k) = order[k] (ascending-id addressing) or slot_of_id[ids[k]]
template <class T>
__global__ void scatter_by_id_kernel(uint32_t n, const uint32_t* __restrict__ order, const uint64_t* __restrict__ ids,
                                     const uint32_t* __restrict__ slot_of_id, uint64_t table_len,
                                     const T* __restrict__ src, int src_stride, T* __restrict__ dst, int dst_stride,
                                     unsigned int* __restrict__ bad) {
  uint32_t k = blockIdx.x * blockDim.x + threadIdx.x;
  if (k >= n) return;
  uint32_t s;
  if (ids) {
    uint64_t v = ids[k];
    s = v < table_len ? slot_of_id[v] : 0xffffffffu;
    if (s == 0xffffffffu) {
      atomicAdd(bad, 1u);
      return;
    }
  } else {
    s = order[k];
  }
  dst[(size_t)s * dst_stride] = src[(size_t)k * src_stride];
}

// RMFPlanner::set_target for agents addressed by id: (route, 0) into the agent_cache (rmf/mod.rs:217-237)
__global__ void route_set_target_kernel(uint32_t m, const uint64_t* __restrict__ ids,
                                        const uint32_t* __restrict__ slot_of_id, uint64_t table_len,
                                        uint32_t* __restrict__ wp, unsigned int* bad) {
  uint32_t k = blockIdx.x * blockDim.x + threadIdx.x;
  if (k >= m) return;
  uint64_t v = ids[k];
  uint32_t sl = v < table_len ? slot_of_id[v] : 0xffffffffu;
  if (sl == 0xffffffffu) {
    atomicAdd(bad, 1u);
    return;
  }
  wp[sl] = (wp[sl] & WP_MASK) | (1u << WP_ROUTE_SHIFT);
}

__global__ void fill_u32_kernel(uint64_t n, uint32_t* p, uint32_t v) {
  uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) p[i] = v;
}
__global__ void fill_f64_kernel(uint64_t n, double* p, double v) {
  uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) p[i] = v;
}

// ---------------------------------------------------------------------------------------------
// Step bookkeeping on the device.  Steps are enqueued asynchronously; a step that fails makes every
// later kernel of the handle a no-op (status->failed is sticky until rcs_sync reports it).
// ---------------------------------------------------------------------------------------------
// strips: also resets the headers of the two send buffers: [0] = number of packed agents, [1] = "this rank has
// failed" (so that a failure reaches the neighbours with the next exchange and the whole job stops within `world` steps)
__global__ void begin_step_kernel(DevStatus* st, uint32_t* cnt, uint32_t* send_l_hdr, uint32_t* send_r_hdr,
                                  uint32_t* xseq) {
  pdl_enter();
  if (xseq) *xseq += 1u;  // peer-store transport: one exchange round per step, failed steps included
  if (send_l_hdr) {
    send_l_hdr[0] = 0u;
    send_r_hdr[0] = 0u;
    send_l_hdr[1] = st->failed;
    send_r_hdr[1] = st->failed;
  }
  if (st->failed) return;
  st->oob_count = 0;
  st->nonfinite_count = 0;
  st->big_cells = 0;
  st->local_failed = 0;
  st->halo_err = 0;
  st->capacity_err = 0;
  st->spawned = 0;
  st->destroyed = 0;
  st->slow_count = 0;
  st->wide_count = 0;
  st->first_oob_id = ~0ull;
  st->finite_tti = 0;
  st->neighbour_total = 0;
  st->candidate_total = 0;
  cnt[CNT_SAVE] = cnt[CNT_CUR];
  cnt[CNT_TOT] = cnt[CNT_CUR];
  cnt[CNT_EV_SPAWN_SAVE] = cnt[CNT_EV_SPAWN];
  cnt[CNT_EV_DESTROY_SAVE] = cnt[CNT_EV_DESTROY];
}

// Last kernel of a step: does the step stand?  (Out of bounds only fails committed steps.)  A failing step sets
// the sticky flag; nothing has been moved yet -- the pre-step snapshot is still intact for rcs_sync to restore.
// cnt_cur != nullptr on steps with churn: the state now holds *n_sorted entries (some flagged keep = 0).
__global__ void end_step_kernel(DevStatus* st, int oob_fails, unsigned long long* steps_done, uint32_t* cnt_cur,
                                const uint32_t* n_sorted) {
  pdl_enter();
  if (st->failed) return;
  if ((oob_fails && st->oob_count) || st->halo_err || st->capacity_err) {
    st->local_failed = 1;
    st->failed = 1;
    return;
  }
  if (cnt_cur) *cnt_cur = *n_sorted;
  *steps_done += 1;
}

__global__ void set_counts_kernel(uint32_t* cnt, uint32_t n) {
  cnt[CNT_CUR] = n;
  cnt[CNT_TOT] = n;
}

// ---------------------------------------------------------------------------------------------
// Churn: stream compaction of the agents whose keep flag is set (despawn at sinks, lib.rs:378-380;
// strip ownership).  pos = exclusive scan of keep; the new live count is pos[n].
// ---------------------------------------------------------------------------------------------
__global__ void compact_keep_kernel(uint32_t n_ub, const uint32_t* __restrict__ n_ptr,
                                    const uint32_t* __restrict__ keep, const uint32_t* __restrict__ pos,
                                    AgentArrays in, AgentArrays out, const DevStatus* status) {
  if (status && status->failed) return;
  uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n_ub || i >= *n_ptr || !keep[i]) return;
  uint32_t k = pos[i];
  out.pos[k] = in.pos[i];
  out.vel[k] = in.vel[i];
  out.id[k] = in.id[i];
  out.grp[k] = in.grp[i];
  out.wp[k] = in.wp[i];
  if (in.pv) out.pv[k] = in.pv[i];
}

// ---------------------------------------------------------------------------------------------
// Source sinks (lib.rs:199-254).  Spawn probe: `get_neighbours_in_radius(0.4, source)` must be empty.
// The probe runs over the agents (not over the index): an agent blocks source s iff the reference's
// query would have returned it, i.e. its INSERT cell is one of the cells of s's query stencil and its
// distance to the source passes the strict test.  Sources are looked up through a small static grid.
// ---------------------------------------------------------------------------------------------
struct SourceGridDev {
  double x0, y0, cell;        // lower corner and cell size (>= 1 m) of the source lookup grid
  uint32_t nx, ny;
  const uint32_t* start;      // nx*ny+1
  const uint32_t* items;      // source-sink indices
};

__global__ void ss_probe_kernel(GridDev g, SourceGridDev sg, const SourceSinkDev* __restrict__ ss, double thr2_probe,
                                uint32_t n_ub, const uint32_t* __restrict__ n_ptr,
                                const double2* __restrict__ pos, const uint32_t* __restrict__ keep,
                                uint32_t* __restrict__ blocked, const DevStatus* status) {
  if (status->failed) return;
  uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n_ub || i >= *n_ptr) return;
  if (keep && !keep[i]) return;  // removed at the end of the previous step (lib.rs:378-380)
  const double px = pos[i].x, py = pos[i].y;
  // conservative range of lookup cells around the agent (0.4 m radius + slack)
  const double fx0 = floor((px - 0.45 - sg.x0) / sg.cell), fx1 = floor((px + 0.45 - sg.x0) / sg.cell);
  const double fy0 = floor((py - 0.45 - sg.y0) / sg.cell), fy1 = floor((py + 0.45 - sg.y0) / sg.cell);
  if (!(fx1 >= 0.0 && fy1 >= 0.0 && fx0 < (double)sg.nx && fy0 < (double)sg.ny)) return;  // also rejects NaN
  const uint32_t cx0 = fx0 < 0.0 ? 0u : (uint32_t)fx0, cx1 = fx1 >= (double)sg.nx ? sg.nx - 1 : (uint32_t)fx1;
  const uint32_t cy0 = fy0 < 0.0 ? 0u : (uint32_t)fy0, cy1 = fy1 >= (double)sg.ny ? sg.ny - 1 : (uint32_t)fy1;
  uint64_t my_cell;
  if (!location_to_index(g, px, py, my_cell)) return;  // not in the index at all
  for (uint32_t cx = cx0; cx <= cx1; ++cx) {
    for (uint32_t cy = cy0; cy <= cy1; ++cy) {
      const uint32_t c = cx * sg.ny + cy;
      for (uint32_t k = sg.start[c]; k < sg.start[c + 1]; ++k) {
        const uint32_t sidx = sg.items[k];
        const SourceSinkDev& s = ss[sidx];
        const double dx = px - s.sx, dy = py - s.sy;
        if (!(dx * dx + dy * dy < thr2_probe)) continue;  // (agent_pos - source).norm() < 0.4
        // is my insert cell visited by `for x in left..=right { for y in bottom..=top }`?
        long long xl = s.pl < 0 ? 0 : s.pl, xr = s.pr > g.x_max ? g.x_max : s.pr;
        bool hit = false;
        for (long long qx = xl; qx <= xr && !hit; ++qx) {
          uint64_t c_lo, c_hi;
          if (column_cell_range(g, qx, s.pb, s.pt, c_lo, c_hi)) hit = my_cell >= c_lo && my_cell <= c_hi;
        }
        if (hit) blocked[sidx] = 1u;
      }
    }
  }
}

// Strips: which of this rank's sources spawn in this step, as a bitmap over the source ids.  The ranks' bitmaps are
// disjoint (a source is owned by one rank); their sum over the ranks is the global spawn set, from which every rank
// derives the same sequential ids (lib.rs:128-129: ids follow the order of the source sinks).
__global__ void ss_flags_kernel(const SourceSinkDev* __restrict__ ss, uint32_t n_ss, double dt,
                                const uint32_t* __restrict__ blocked, uint32_t* __restrict__ bits,
                                const DevStatus* status) {
  if (status->failed) return;
  const uint32_t k = blockIdx.x * blockDim.x + threadIdx.x;
  if (k >= n_ss) return;
  const SourceSinkDev& s = ss[k];
  const uint64_t want = f64_as_usize(round(dt * s.rate));  // MonotonicCrowd, source_sink.rs:97-100
  if (s.alive && s.owned && want > 0 && !blocked[k]) atomicOr(&bits[k >> 5], 1u << (k & 31u));
}

// bits[w] = sum over the ranks' bitmaps (single-process transport; disjoint bits, so the sum is the union)
__global__ void ss_bits_sum_kernel(uint32_t n_words, uint32_t world, const uint32_t* __restrict__ parts,
                                   uint32_t* __restrict__ bits) {
  const uint32_t w = blockIdx.x * blockDim.x + threadIdx.x;
  if (w >= n_words) return;
  uint32_t v = 0;
  for (uint32_t r = 0; r < world; ++r) v += parts[(size_t)r * n_words + w];
  bits[w] = v;
}

// One block.  Sources in ascending id order; at most ONE agent per source per step and only when the
// generator asks for >= 1 (the reference's loop over spawn_number is commented out, lib.rs:207-219).
// Ids are allocated sequentially (lib.rs:128-129) in that order.  gbits != nullptr (strips): the global spawn set
// (ss_flags_kernel, summed over the ranks) decides and numbers the spawns; this rank materialises its own sources'.
__global__ void ss_spawn_kernel(GridDev g, const SourceSinkDev* __restrict__ ss, const GroupDev* __restrict__ groups,
                                uint32_t n_ss, double dt, const uint32_t* __restrict__ gbits,
                                uint32_t* __restrict__ blocked, AgentArrays cur, uint32_t* __restrict__ keep,
                                uint32_t cap, uint32_t* cnt, unsigned long long* next_id, unsigned long long* ev_id, double* ev_xy, uint32_t ev_cap,
                                DevStatus* status) {
  if (status->failed) return;
  __shared__ uint32_t base_all, base_own;
  if (threadIdx.x == 0) base_all = base_own = 0;
  __syncthreads();
  const uint32_t n0 = cnt[CNT_CUR];
  const unsigned long long id0 = *next_id;
  const uint32_t ev0 = cnt[CNT_EV_SPAWN];
  for (uint32_t b = 0; b < n_ss; b += SCAN_THREADS) {
    const uint32_t k = b + threadIdx.x;
    uint32_t spawn = 0, mine = 0;
    if (k < n_ss) {
      const SourceSinkDev& s = ss[k];
      if (gbits) {
        spawn = (gbits[k >> 5] >> (k & 31u)) & 1u;
      } else {
        const uint64_t want = f64_as_usize(round(dt * s.rate));  // MonotonicCrowd, source_sink.rs:97-100
        spawn = (s.alive && want > 0 && !blocked[k]) ? 1u : 0u;
      }
      mine = (spawn && s.owned) ? 1u : 0u;
      blocked[k] = 0u;
    }
    uint32_t total_all, total_own;
    const uint32_t rank_all = block_exclusive_scan(spawn, total_all);
    const uint32_t rank_own = block_exclusive_scan(mine, total_own);
    const uint32_t off_all = base_all, off_own = base_own;
    __syncthreads();
    if (mine) {
      const uint32_t slot = n0 + off_own + rank_own;
      if (slot < cap) {
        const SourceSinkDev& s = ss[k];
        const unsigned long long id = id0 + off_all + rank_all;
        cur.pos[slot] = make_double2(s.sx, s.sy);
        cur.vel[slot] = make_double2(0.0, 0.0);
        cur.id[slot] = id;
        cur.grp[slot] = s.grp;
        // set_target(agent, waypoints[0], ..) right after the spawn (lib.rs:242-249): a route follower starts at
        // the head of its route
        cur.wp[slot] = groups[s.grp].hl_kind == HL_ROUTE ? (1u << WP_ROUTE_SHIFT) : 0u;
        keep[slot] = 1u;
        if (cur.pv)
          cur.pv[slot] = make_double2(__longlong_as_double(0x7ff8000000000000LL),
                                      __longlong_as_double(0x7ff8000000000000LL));
        const uint32_t e = ev0 + off_own + rank_own;
        if (e < ev_cap) {
          ev_id[e] = id;
          ev_xy[2 * e] = s.sx;
          ev_xy[2 * e + 1] = s.sy;
        } else {
          atomicAdd(&status->capacity_err, 1u);
        }
      } else {
        atomicAdd(&status->capacity_err, 1u);
      }
    }
    if (threadIdx.x == 0) {
      base_all = off_all + total_all;
      base_own = off_own + total_own;
    }
    __syncthreads();
  }
  if (threadIdx.x == 0) {
    uint32_t total = base_own;
    if (n0 + total > cap) total = cap - n0;
    cnt[CNT_CUR] = n0 + total;
    cnt[CNT_TOT] = n0 + total;
    cnt[CNT_EV_SPAWN] = (ev0 + total > ev_cap) ? ev_cap : ev0 + total;
    *next_id = id0 + base_all;
    status->spawned = base_own;
  }
}

// ---------------------------------------------------------------------------------------------
// Strips: halo pack / unpack.  A halo buffer is [count u32, pad][pos][vel][id][meta][pv],
// each array `cap` entries.  Packed order is arbitrary (atomic append); the receiver re-sorts.
// ---------------------------------------------------------------------------------------------
// appends the ghosts of both received buffers after the owned agents; cnt[CNT_TOT] = owned + ghosts
// ---- peer-store transport (one process per GPU, every GPU its own) ----------------------------------------------
// The pack pass stores the boundary rows straight into the neighbour's receive buffer over NVLink (rcs_dist_peer_*:
// the buffers are CUDA IPC mappings); the next kernel on the stream, halo_unpack_kernel, first writes count + failed
// flag behind them and releases the round number (halo_publish), then acquires the neighbours' rounds.  Receive
// buffers have two halves used in turn: a rank packs round k + 2 only after it has unpacked round k + 1, which its
// neighbour published only after it had unpacked round k -- so the half being written is never one still being read.
__device__ __forceinline__ uint32_t ld_acquire_sys(const uint32_t* p) {
  uint32_t v;
  asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ void st_release_sys(uint32_t* p, uint32_t v) {
  asm volatile("st.release.sys.global.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
__device__ __forceinline__ unsigned long long global_timer_ns() {
  unsigned long long t;
  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
  return t;
}

// header of one half of a receive buffer: [count, failed, round, pad].  Run by threads 0 and 1 of the first block of
// halo_unpack_kernel, i.e. after the pack pass has completed (stream order) and before anybody waits.
__device__ __forceinline__ void halo_publish(uint32_t seq, const uint32_t* __restrict__ send_hdr, uint32_t* remote_hdr) {
  if (!remote_hdr) return;
  uint32_t* dst = remote_hdr + 4u * (seq & 1u);
  dst[0] = send_hdr[0];
  dst[1] = send_hdr[1];
  // the rows were stored by the kernel before this one; the fence orders them (and the two words above) before the
  // round number for an observer on the other GPU
  __threadfence_system();
  st_release_sys(dst + 2, seq);
}

constexpr unsigned long long HALO_WAIT_NS = 120ull * 1000000000ull;

__global__ void halo_unpack_kernel(AgentArrays cur, uint32_t* __restrict__ keep, uint32_t cap, HaloBuf left,
                                   HaloBuf right, int has_left, int has_right, uint32_t* cnt, DevStatus* status,
                                   const uint32_t* __restrict__ xseq, GridDev g, uint32_t* __restrict__ cellid,
                                   uint32_t* __restrict__ cell_count, uint64_t cell_lo, uint64_t cell_hi,
                                   const uint32_t* __restrict__ send_l_hdr, const uint32_t* __restrict__ send_r_hdr,
                                   uint32_t* remote_l_hdr, uint32_t* remote_r_hdr) {
  pdl_enter();
  uint32_t par = 0u;
  if (xseq) {
    if (blockIdx.x == 0 && threadIdx.x < 2)  // this rank's own round first: nobody waits for a rank that waits
      halo_publish(*xseq, threadIdx.x == 0 ? send_l_hdr : send_r_hdr, threadIdx.x == 0 ? remote_l_hdr : remote_r_hdr);
    // wait for both neighbours' rounds (another GPU's kernel releases them; bounded, so a dead peer fails the step
    // instead of hanging the device)
    __shared__ uint32_t s_ok;
    const uint32_t seq = *xseq;
    par = seq & 1u;
    if (threadIdx.x == 0) {
      const unsigned long long t0 = global_timer_ns();
      uint32_t ok = 1u;
      for (int side = 0; side < 2 && ok; ++side) {
        if (!(side == 0 ? has_left : has_right)) continue;
        const uint32_t* flag = (side == 0 ? left.count : right.count) + 4u * par + 2u;
        while ((int32_t)(ld_acquire_sys(flag) - seq) < 0) {
          __nanosleep(64);
          if (global_timer_ns() - t0 > HALO_WAIT_NS) {
            ok = 0u;
            break;
          }
        }
      }
      s_ok = ok;
    }
    __syncthreads();
    if (!s_ok) {
      if (blockIdx.x == 0 && threadIdx.x == 0) status->failed = 1;  // reported as "a neighbouring rank failed"
      return;
    }
  }
  if (status->failed) return;
  const uint32_t* lh = left.count + 4u * par;
  const uint32_t* rh = right.count + 4u * par;
  if ((has_left && __ldcg(lh + 1)) || (has_right && __ldcg(rh + 1))) {
    if (blockIdx.x == 0 && threadIdx.x == 0) status->failed = 1;  // a neighbour failed: stop here too
    return;
  }
  const uint32_t n0 = cnt[CNT_CUR];
  uint32_t nl = has_left ? __ldcg(lh) : 0u, nr = has_right ? __ldcg(rh) : 0u;
  if (nl > left.cap) nl = left.cap;
  if (nr > right.cap) nr = right.cap;
  const uint32_t k = blockIdx.x * blockDim.x + threadIdx.x;
  if (k == 0) {
    uint32_t tot = n0 + nl + nr;
    if (tot > cap) {
      atomicAdd(&status->capacity_err, 1u);
      tot = cap;
    }
    cnt[CNT_TOT] = tot;
  }
  if (k >= nl + nr) return;
  const HaloBuf& b = k < nl ? left : right;
  const uint32_t e = (k < nl ? k : k - nl) + par * b.cap;
  const uint32_t slot = n0 + k;
  if (slot >= cap) return;
  // (L1 is not coherent with another GPU's stores: the rows are read at L2)
  const double2 p = __ldcg(b.pos + e);
  cur.pos[slot] = p;
  cur.vel[slot] = __ldcg(b.vel + e);
  cur.id[slot] = __ldcg(b.id + e);
  const unsigned long long meta = __ldcg(b.meta + e);
  cur.grp[slot] = (uint32_t)(meta & 0xffffffffull);
  cur.wp[slot] = (uint32_t)(meta >> 32);
  keep[slot] = 1u;
  if (cur.pv) cur.pv[slot] = __ldcg(b.pv + e);
  uint64_t idx;
  (void)bin_one(g, slot, p, cellid, cell_count, cell_lo, cell_hi, status, idx);  // ghosts join the owned histogram
}

// FP64 pipe peak: independent DFMA / DADD chains.
__global__ void fp64_peak_kernel(double* out, int iters, int use_fma) {
  double a0 = threadIdx.x * 1e-9, a1 = a0 + 1, a2 = a0 + 2, a3 = a0 + 3, a4 = a0 + 4, a5 = a0 + 5, a6 = a0 + 6,
         a7 = a0 + 7;
  const double m = 1.0000001, c = 1e-7;
  if (use_fma) {
    for (int i = 0; i < iters; ++i) {
      a0 = __fma_rn(a0, m, c); a1 = __fma_rn(a1, m, c); a2 = __fma_rn(a2, m, c); a3 = __fma_rn(a3, m, c);
      a4 = __fma_rn(a4, m, c); a5 = __fma_rn(a5, m, c); a6 = __fma_rn(a6, m, c); a7 = __fma_rn(a7, m, c);
    }
  } else {
    for (int i = 0; i < iters; ++i) {
      a0 = __dadd_rn(a0, c); a1 = __dadd_rn(a1, c); a2 = __dadd_rn(a2, c); a3 = __dadd_rn(a3, c);
      a4 = __dadd_rn(a4, c); a5 = __dadd_rn(a5, c); a6 = __dadd_rn(a6, c); a7 = __dadd_rn(a7, c);
    }
  }
  out[blockIdx.x * blockDim.x + threadIdx.x] = a0 + a1 + a2 + a3 + a4 + a5 + a6 + a7;
}

__global__ void flush_l2_kernel(uint4* p, uint64_t n16) {
  uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  uint64_t stride = (uint64_t)gridDim.x * blockDim.x;
  for (; i < n16; i += stride) p[i] = make_uint4((uint32_t)i, 1u, 2u, 3u);
}

}  // namespace rcs
