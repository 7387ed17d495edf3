// rcs_host.h -- the simulation handle and small host helpers shared by the .inl parts of rcs.cu.
//
// One translation unit (rcs.cu) includes the kernels and every host part, so that each __global__
// function is defined exactly once and the whole library is compiled with --fmad=false.
#pragma once

#include "../../include/rcs.h"

#include <algorithm>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <limits>
#include <map>
#include <numeric>
#include <string>
#include <unordered_set>
#include <vector>

#include "rcs_kernels.cuh"
#include "rcs_step_warp.cuh"
#include "rcs_step_tile.cuh"
#include "rcs_inloop.cuh"

namespace rcs_host {

using namespace rcs;

struct LPDesc {
  uint32_t kind;
  double agent_scale, obstacle_scale, reaction_time, force_distance, agent_mass, agent_radius;
};
struct HLDesc {
  uint32_t kind;
  double vx, vy;
  uint32_t route_off, route_n;  // HL_ROUTE / HL_ROUTE_TABLE: the planner's table in the route array
  // HL_ROUTE_TABLE: leg target -> index of the leg's first point within the planner's table.  std::less on doubles
  // is IEEE equality for non-NaN keys (+0 == -0); NaN targets are never inserted, so they never match.
  std::map<std::pair<double, double>, uint32_t> legs;
};
// RouteTablePlan's leg lookup: the leg whose target == (x, y) on both coordinates -> its first point, or -1
inline int64_t leg_of(const HLDesc& h, double x, double y) {
  if (x != x || y != y) return -1;
  const auto it = h.legs.find({x, y});
  return it == h.legs.end() ? -1 : (int64_t)it->second;
}
struct GroupKey {
  uint32_t hl, lp;
  double eyesight;
  int32_t source_sink;
};

// What rcs_sync needs to undo a failed asynchronous step: the pre-step snapshot of every step on the
// sorted path is the `srt` buffer set of the moment the step was enqueued.
struct PendingStep {
  AgentArrays cur, srt;
  bool snapshot_in_srt;  // false on the streaming path (snapshot = cur)
  uint32_t n;
};

struct HaloMem {
  void* base = nullptr;  // one allocation: [header 64 B][x][y][vx][vy][id][meta][pvx][pvy], each `cap` entries
  uint64_t bytes = 0;
  HaloBuf buf{};
};

// Peer-store halo transport (rcs_dist_peer_export / rcs_dist_peer_connect): this rank's receive arena, which the
// neighbours map through CUDA IPC and store into, and the mappings of theirs.
// Arena: [64 B: magic, cap][64 B header left side][64 B header right side][rows left side][rows right side]; a header
// is two halves of [count, failed, round, pad]; the rows of a side are pos, vel, id, meta, pv with 2 x cap entries
// each (two halves, used in turn).
struct PeerHalo {
  bool enabled = false;
  void* arena = nullptr;
  uint64_t arena_bytes = 0;
  uint32_t cap = 0;
  void* nb_arena[2] = {nullptr, nullptr};   // [0] left neighbour's arena, [1] right neighbour's
  HaloBuf remote[2]{};                       // where this rank's left / right boundary columns go
  uint32_t* remote_hdr[2] = {nullptr, nullptr};
  HaloBuf local[2]{};                        // what the left / right neighbour stores into
  uint32_t* xseq = nullptr;                  // device: exchange round, bumped by begin_step_kernel
};

// NCCL entry points, resolved with dlopen at rcs_dist_init (the library itself does not link NCCL, so it
// loads on boxes without it and single-GPU use never touches it).
struct Id128 {
  char internal[128];
};
struct NcclApi {
  void* lib = nullptr;
  int (*GetUniqueId)(void*) = nullptr;
  int (*CommInitRank)(void**, int, Id128 /* ncclUniqueId, by value */, int) = nullptr;
  int (*CommDestroy)(void*) = nullptr;
  int (*Send)(const void*, size_t, int, int, void*, cudaStream_t) = nullptr;
  int (*Recv)(void*, size_t, int, int, void*, cudaStream_t) = nullptr;
  int (*AllReduce)(const void*, void*, size_t, int, int, void*, cudaStream_t) = nullptr;
  int (*GroupStart)() = nullptr;
  int (*GroupEnd)() = nullptr;
  const char* (*GetErrorString)(int) = nullptr;
};

// A steady-state step as an instantiated CUDA graph (rcs_host_step.inl): everything the launch sequence and the
// kernel arguments depend on is in the key; the host-side bookkeeping of a step is replayed next to the launch.
struct StepKey {
  uint64_t epoch = 0, dt_bits = 0;
  const void* cur_pos = nullptr;
  uint32_t flags = 0, n_ub = 0, n = 0;
  uint32_t n_ub_spawn = 0;  // the launch bound after this step's spawns: phase B's grids (spawn_launch_bound)
  bool cur_has_dead = false;
  bool operator==(const StepKey& o) const {
    return epoch == o.epoch && dt_bits == o.dt_bits && cur_pos == o.cur_pos && flags == o.flags && n_ub == o.n_ub &&
           n == o.n && n_ub_spawn == o.n_ub_spawn && cur_has_dead == o.cur_has_dead;
  }
};
struct StepGraph {
  StepKey key;
  cudaGraphExec_t exec = nullptr;
  uint64_t launches = 0;  // kernels in the graph
};

// buffers of rcs_step_in_loop (allocated on first use)
struct InLoopMem {
  double2 *np_a = nullptr, *np_b = nullptr, *nv = nullptr;
  unsigned long long* rank = nullptr;
  uint32_t *cellid = nullptr, *perm = nullptr, *cell_count = nullptr, *cell_start = nullptr, *cursor = nullptr;
  uint32_t* changed = nullptr;
  uint64_t cap = 0, cells = 0;
};

// Small host-to-device uploads on the step stream through two pinned staging buffers used in turn: a buffer is
// rewritten only after its previous copy has run, so an upload per step waits at most for the step before last.
struct UploadRing {
  void* buf[2] = {nullptr, nullptr};
  cudaEvent_t ev[2] = {nullptr, nullptr};
  bool used[2] = {false, false};
  uint64_t cap = 0;  // bytes per buffer
  uint32_t turn = 0;
};

inline void ring_free(UploadRing& r) {
  for (int i = 0; i < 2; ++i) {
    if (r.used[i]) cudaEventSynchronize(r.ev[i]);
    if (r.buf[i]) cudaFreeHost(r.buf[i]);
    if (r.ev[i]) cudaEventDestroy(r.ev[i]);
  }
  r = UploadRing{};
}

inline void inloop_free(InLoopMem*& m) {
  if (!m) return;
  cudaFree(m->np_a); cudaFree(m->np_b); cudaFree(m->nv); cudaFree(m->rank); cudaFree(m->cellid); cudaFree(m->perm);
  cudaFree(m->cell_count); cudaFree(m->cell_start); cudaFree(m->cursor); cudaFree(m->changed);
  delete m;
  m = nullptr;
}

}  // namespace rcs_host

struct rcs_sim {
  rcs_sim_desc desc{};
  rcs::GridDev grid{};
  int device = 0;
  cudaStream_t stream = nullptr;
  uint64_t cap = 0;
  uint32_t n = 0;     // live agents owned by this handle, exact as of the last sync
  uint32_t n_ub = 0;  // upper bound used to size launches while steps with churn are in flight
  uint32_t n_tight = 0, n_coarse = 0xffffffffu;  // source sinks: exact bound / the coarse launch bound made from it
  rcs::AgentArrays cur{}, srt{};
  uint32_t *cellid = nullptr, *perm = nullptr, *cell_count = nullptr, *cell_start = nullptr, *cursor = nullptr;
  uint32_t *tile_sums = nullptr, *scan_total = nullptr, *big_list = nullptr, *slow_list = nullptr, *wide_list = nullptr;
  uint32_t* srt_cell = nullptr;  // strips: insert cell of every sorted agent
  rcs::TileRange* tile_ranges = nullptr;  // per block of step_tile_kernel: staging ranges (gather_sorted_kernel)
  uint4* slices = nullptr;       // per sorted agent: candidate slices of its radius query (gather_sorted_kernel)
  uint32_t* keep = nullptr;      // churn: 0 = the entry leaves (sink reached, migrated, ghost); dropped by the next sort
  bool cur_has_dead = false;     // `cur` holds entries with keep = 0 (compacted lazily, at rcs_sync)
  uint64_t tile_sums_cap = 0;
  // cells this handle indexes: the whole grid, or on a strip the columns it owns plus the halo (a multiple of 4
  // at the lower end: the scan kernels use 16-byte accesses).  cell_start[cell_hi] = number of sorted agents.
  uint64_t cell_lo = 0, cell_hi = 0;
  uint32_t* cnt = nullptr;       // device counters CNT_*
  uint32_t* h_cnt = nullptr;     // pinned copy
  bool cnt_dirty = true;         // host changed n: cnt[CNT_CUR] must be rewritten before the next step
  rcs::GroupDev* d_groups = nullptr;
  uint32_t d_groups_cap = 0;
  std::vector<rcs::GroupDev> groups;
  std::vector<rcs_host::GroupKey> group_keys;
  bool groups_dirty = false;
  std::vector<rcs_host::LPDesc> lps;
  std::vector<rcs_host::HLDesc> hls;
  bool any_zanlungo = false;
  bool any_route = false;            // an HL_ROUTE group exists: steps take the sorted path (it carries `wp`)
  std::vector<double> routes;        // route table, interleaved x,y
  std::vector<uint32_t> route_end;   // per route point: one past the last point of its leg, within its planner's table
  double* d_routes = nullptr;
  uint32_t* d_route_end = nullptr;
  bool routes_dirty = false;
  bool have_host_hl = false;
  rcs::DevStatus* d_status = nullptr;
  rcs::DevStatus* h_status = nullptr;  // pinned
  uint64_t last_alloc_agent_id = 0;
  unsigned long long* d_next_id = nullptr;  // device copy of last_alloc_agent_id (source sinks allocate ids)
  uint64_t max_id_plus1 = 0;
  bool index_valid = false;  // srt + cell_start describe the current positions
  // id-addressed access
  uint32_t *slot_of_id = nullptr, *id_rank = nullptr, *order_by_id = nullptr, *presence = nullptr;
  uint64_t slot_table_cap = 0;
  bool slot_valid = false;
  // trace
  bool trace = false;
  double *tr_ti = nullptr, *tr_fx = nullptr, *tr_fy = nullptr;
  uint32_t *tr_nbc = nullptr, *tr_nbo = nullptr, *tr_own = nullptr;
  uint64_t *tr_nbids = nullptr, *tr_id = nullptr;
  uint64_t tr_nbids_cap = 0, tr_nb_total = 0;
  uint32_t tr_n = 0;
  bool tr_valid = false;
  // source sinks
  std::vector<rcs::SourceSinkDev> sources;  // index = source sink id (removed ones stay with alive = 0)
  std::vector<double> ss_wp;                // shared waypoint table, interleaved
  std::vector<uint32_t> ss_rwp;             // per waypoint (offsets of ss_wp): route-follower entry of set_target
  rcs::SourceSinkDev* d_sources = nullptr;
  double* d_ss_wp = nullptr;
  uint32_t* d_ss_rwp = nullptr;
  uint32_t* d_blocked = nullptr;
  // strips: spawn set of the step as a bitmap over the source ids: this rank's, every rank's (single-process
  // transport: staging for the other ranks' bitmaps), and the sum over the ranks
  uint32_t *d_ss_bits_local = nullptr, *d_ss_bits_parts = nullptr, *d_ss_bits = nullptr;
  uint32_t ss_words = 0;
  cudaEvent_t ev_flags = nullptr;
  uint32_t *d_sg_start = nullptr, *d_sg_items = nullptr;
  rcs::SourceGridDev sgrid{};
  bool sources_dirty = false;
  uint32_t n_sources_alive = 0;
  bool ever_had_sources = false;
  // CrowdGenerators other than MonotonicCrowd (ss_wants_spawn).  PoissonCrowd: per-source thresholds of the dt they
  // were last computed for, uploaded through thr_ring when dt's bits change.  Host generators: the counts of the next
  // step (1 = at least one), mirrored on the host until a step consumes them.
  uint32_t n_poisson_alive = 0, n_host_gen_alive = 0;
  unsigned long long* d_ss_thr = nullptr;
  std::vector<unsigned long long> ss_thr;
  uint64_t ss_thr_dt_bits = 0;
  bool ss_thr_valid = false;
  rcs_host::UploadRing thr_ring;
  uint32_t* d_ss_count = nullptr;
  std::vector<uint32_t> ss_count;
  bool ss_count_consumed = false;  // a step ran since the last rcs_set_spawn_counts (the device copy is all zero)
  rcs_host::UploadRing count_ring;
  // events (EventListener::agent_spawned / agent_destroyed)
  unsigned long long *ev_spawn_id = nullptr, *ev_destroyed = nullptr;
  double* ev_spawn_xy = nullptr;
  uint32_t ev_cap = 0;
  // strips
  rcs::StripDev strip{};
  int rank = 0, world = 1;
  uint32_t halo_width = 0;  // columns sent to each neighbour = ring h + stencil reach q
  std::vector<uint64_t> strip_bounds;  // optional: world + 1 column boundaries (rcs_dist_set_boundaries); empty = equal split
  rcs_host::HaloMem send_l, send_r, recv_l, recv_r;
  rcs_host::PeerHalo peer;
  void* nccl_comm = nullptr;
  std::vector<rcs_sim*> local_group;  // single-process transport: the handles of all ranks, by rank
  cudaEvent_t ev_packed = nullptr, ev_copied = nullptr;
  // staging
  void* stage = nullptr;
  uint64_t stage_bytes = 0;
  // asynchronous read-back (rcs_read_agents_async): gathers on the main stream, copies on a second one
  cudaStream_t copy_stream = nullptr;
  cudaEvent_t ev_gathered = nullptr, ev_read_done = nullptr;
  void* stage2 = nullptr;
  uint64_t stage2_bytes = 0;  // one half
  bool read_inflight = false;
  cudaEvent_t ev_half_done[2] = {nullptr, nullptr};
  bool half_used[2] = {false, false};
  uint64_t read_seq = 0;
  // rcs_set_preferred_velocity: upload stream + staging buffer of its own
  cudaStream_t up_stream = nullptr;
  cudaEvent_t ev_uploaded = nullptr, ev_pv_scattered = nullptr;
  void* pv_stage = nullptr;
  uint64_t pv_stage_bytes = 0;
  bool pv_inflight = false;
  rcs_host::InLoopMem* inloop = nullptr;
  void* flush_buf = nullptr;
  uint64_t flush_bytes = 0;
  unsigned int* d_bad = nullptr;
  unsigned long long* d_bad2 = nullptr;  // 8-byte device scratch
  std::vector<rcs_host::PendingStep> pending;
  uint64_t steps_enqueued = 0;
  unsigned long long* d_steps_done = nullptr;
  uint64_t steps_done_at_sync = 0;
  std::string err;
  uint64_t launches = 0;
  rcs_stats stats{};
  cudaEvent_t events[RCS_NUM_EVENTS]{};
  uint32_t opt_step_kernel = 0;
  bool tile_attr_set = false;
  // CUDA graphs of steady-state steps
  uint32_t opt_graphs = 1;     // RCS_OPT_GRAPHS
  uint64_t graph_epoch = 0;    // bumped by everything that can change a step's launch sequence or kernel arguments
  std::vector<rcs_host::StepGraph> step_graphs;
  rcs_host::StepKey recent_keys[2];  // keys of the last steps that ran eagerly (a key seen again is captured)
  uint64_t graph_launches = 0, graph_captures = 0;
  // dominant-kernel timing
  bool ktiming = false;
  std::vector<std::pair<cudaEvent_t, cudaEvent_t>> kevents;  // pending pairs
  std::vector<cudaEvent_t> kevent_pool;
  double ktime_ms = 0.0;
  uint64_t ktime_n = 0;
};

namespace rcs_host {

extern thread_local std::string g_create_error;

#define CU_TRY(sim, call)                                                                         \
  do {                                                                                            \
    cudaError_t e__ = (call);                                                                     \
    if (e__ != cudaSuccess) {                                                                     \
      (sim)->err = std::string("CUDA error: ") + cudaGetErrorString(e__) + " at " #call;          \
      return RCS_ERR_CUDA;                                                                        \
    }                                                                                             \
  } while (0)

inline uint32_t blocks_for(uint64_t n, uint32_t threads) {
  return (uint32_t)std::max<uint64_t>((n + threads - 1) / threads, 1);
}

template <class T>
inline cudaError_t dalloc(T** p, uint64_t count) {
  return cudaMalloc(reinterpret_cast<void**>(p), std::max<uint64_t>(count, 1) * sizeof(T));
}

inline bool churn(const rcs_sim* s) { return s->ever_had_sources || s->strip.enabled; }

}  // namespace rcs_host
