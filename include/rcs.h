/* rcs.h -- C ABI of the B200-native per-timestep agent update of rmf_crowdsim.
 *
 * This is the drop-in boundary: the entry points below are what a Rust `-sys` crate for the
 * reference (open-rmf/rmf_crowdsim) would bind in place of the reference's CPU hot path.  Plain
 * pointers and sizes only; opaque handle; `int` status (0 = OK).  One handle is used by one
 * thread at a time (the reference is single-threaded, lib.rs:69-91).  The caller owns every host
 * buffer for the duration of the call only; the library owns all device memory.  The library never
 * calls back into the host language: events are polled (rcs_poll_events).
 *
 * There is NO CPU fallback: every entry point that computes needs a CUDA device and fails with
 * RCS_ERR_NO_DEVICE / RCS_ERR_CUDA otherwise.
 *
 * Reference file:line citations are relative to /root/reference/rmf_crowdsim/src.
 *
 * Index semantic (SURVEY.md section 0.1): DEFERRED -- within one step every radius query sees the
 * start-of-step positions of all agents (the reference mutates its index inside a HashMap-ordered
 * loop, lib.rs:299, which makes its own results order-dependent and irreproducible).
 */
#ifndef RCS_H_
#define RCS_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define RCS_ABI_VERSION 1

typedef struct rcs_sim rcs_sim;

/* Status codes.  rcs_last_error() returns the reference's literal message where one exists:
 *   RCS_ERR_OUT_OF_BOUNDS -> "Index out of bounds"               (location_hash_2d.rs:62)
 *   RCS_ERR_SPAWN         -> "Failed to add agents from source"  (lib.rs:252)               */
enum {
  RCS_OK = 0,
  RCS_ERR_OUT_OF_BOUNDS = 1,
  RCS_ERR_SPAWN = 2,
  RCS_ERR_CUDA = 3,
  RCS_ERR_NCCL = 4,
  RCS_ERR_CAPACITY = 5,
  RCS_ERR_ARG = 6,
  RCS_ERR_NO_DEVICE = 7,
  RCS_ERR_HALO = 8 /* multi-GPU: an agent moved further than the halo width in one step */
};

/* LocationHash2D::new(width, height, cell_size, offset)  (location_hash_2d.rs:33-51) plus the
 * device placement.  n_x = (width/cell_size) as usize, n_y = (height/cell_size) as usize. */
typedef struct rcs_sim_desc {
  double width;
  double height;
  double cell_size;
  double offset_x;
  double offset_y;
  uint64_t capacity; /* maximum number of live agents held by this handle (per rank) */
  int32_t device;    /* CUDA device ordinal */
  uint32_t flags;    /* reserved, 0 */
} rcs_sim_desc;

/* Per-step counters (SURVEY.md section 5): non-finite values are NOT errors in the reference
 * (a NaN position lands in cell 0 through the saturating cast), so they are only counted. */
typedef struct rcs_stats {
  uint64_t n_agents;          /* live agents after the step */
  uint64_t oob_count;         /* agents whose new position failed location_to_index */
  uint64_t first_oob_id;      /* smallest such id (UINT64_MAX if none) */
  uint64_t nonfinite_count;   /* agents whose new position or velocity is not finite */
  uint64_t finite_tti_count;  /* agents whose t_i was finite (ran the force pass) */
  uint64_t neighbour_total;   /* sum over agents of neighbour-list lengths (after self filter) */
  uint64_t candidate_total;   /* sum over agents of candidates distance-tested */
  uint64_t spawned;           /* agents spawned by source sinks in this step */
  uint64_t destroyed;         /* agents removed at sinks in this step */
  uint64_t steps;             /* steps executed on this handle */
} rcs_stats;

uint32_t rcs_abi_version(void);

/* Simulation::new(LocationHash2D::new(..))  (lib.rs:103-116) */
int rcs_sim_create(const rcs_sim_desc* desc, rcs_sim** out);
void rcs_sim_destroy(rcs_sim* sim);
/* Message of the last failing call on this handle ("" if none); sim may be NULL for create errors. */
const char* rcs_last_error(const rcs_sim* sim);

/* ---- planner descriptors --------------------------------------------------------------------
 * The reference passes planners as Arc<Mutex<dyn Trait>> per add_agents group (lib.rs:119-125).
 * Here a group names device-side planner descriptors instead. */

/* local_planners::no_local_plan::NoLocalPlan  (no_local_plan.rs:7-18) */
int rcs_lp_none(rcs_sim* sim, uint32_t* out_lp);
/* local_planners::zanlungo::Zanlungo::new, same argument order (zanlungo.rs:31-38) */
int rcs_lp_zanlungo(rcs_sim* sim, double agent_scale, double obstacle_scale, double reaction_time,
                    double force_distance, double agent_mass, double agent_radius, uint32_t* out_lp);

/* HighLevelPlanner::get_desired_velocity (highlevel_planners.rs:9) evaluated on the device:
 *  constant: Some(v) for every agent            (fixture of lib.rs:391-420)
 *  parity  : even id -> Some(-v), odd -> Some(v) (fixture of rmf_crowdsim_viz/src/main.rs:20-30)
 *  route   : rmf::RMFPlanner's waypoint follower on a caller-supplied route (see rcs_hl_route)
 *  route table: the same follower on caller-supplied legs, one per set_target point (see rcs_hl_route_table)
 *  host    : Some(table[id]) as uploaded by rcs_set_preferred_velocity, None for ids never set
 *            (slow path that keeps user-implemented HighLevelPlanner trait objects usable)
 *  none    : always None  => velocity (0,0)     (lib.rs:263-273) */
int rcs_hl_constant(rcs_sim* sim, double vx, double vy, uint32_t* out_hl);
int rcs_hl_parity(rcs_sim* sim, double vx, double vy, uint32_t* out_hl);
int rcs_hl_host(rcs_sim* sim, uint32_t* out_hl);
/* The per-step half of rmf::RMFPlanner (rmf/mod.rs:197-215) on the device: an agent in the planner's
 * agent_cache heads for point k of the route, advances to k+1 once (position - route[k]).norm() < 1e-1, and
 * gets Some(normalize(route[k] - position)); agents not in the cache get None.  The route itself is supplied by
 * the caller (xy = n_points interleaved x,y): the reference plans it with the third-party `mapf` crate
 * (rmf/mod.rs:160-192), which is host-side graph search and out of scope.  Agents enter the cache at route
 * point 0 through HighLevelPlanner::set_target: automatically when a SourceSink spawns them (lib.rs:242-249)
 * and whenever they reach one of its waypoints (lib.rs:326-333), or explicitly with rcs_hl_route_set_target.
 * A SourceSink with a route planner takes exactly ONE waypoint, the sink (the reference plans a new route per waypoint;
 * here a planner is one polyline): rcs_add_source_sink refuses more with RCS_ERR_ARG.  A source sink with
 * intermediate waypoints takes a route-table planner (rcs_hl_route_table).  n_points: 1..65534. */
int rcs_hl_route(rcs_sim* sim, uint64_t n_points, const double* xy, uint32_t* out_hl);
int rcs_hl_route_set_target(rcs_sim* sim, uint64_t n, const uint64_t* ids);
/* RMFPlanner with a route cache the caller has filled: the routes that set_target would plan, as LEGS.
 * Leg k: target (targets_xy[2k], targets_xy[2k+1]), polyline of leg_points[k] points; the legs' points are
 * concatenated in xy.  set_target(agent, point, tolerance) makes the leg whose target == point (IEEE equality on both
 * coordinates; NaN never matches; the tolerance is ignored) the agent's cache entry, at its route point 0.
 * get_desired_velocity is rcs_hl_route's follower on the current leg: it advances from point k to k+1 within 0.1 m
 * unless k is the leg's last point.  In a SourceSink the spawn calls set_target(waypoints[0]) and every advance to
 * waypoint k+1 calls set_target(waypoints[k+1]); a loop_forever wrap calls nothing (lib.rs:305-336), so the agent
 * keeps its last leg.  A one-leg table whose target is the sink runs exactly as rcs_hl_route on the same polyline.
 * RCS_ERR_ARG, nothing registered: no legs, a leg without points, two legs with equal targets, more than 65534
 * points in all.  rcs_add_source_sink refuses (RCS_ERR_ARG, nothing added) a route-table planner with a waypoint
 * that has no leg. */
int rcs_hl_route_table(rcs_sim* sim, uint64_t n_legs, const double* targets_xy, const uint64_t* leg_points,
                       const double* xy, uint32_t* out_hl);
/* set_target(agent, targets_xy[i], ..) of planner hl for the agents ids[i] (agents added with rcs_add_agents; an id
 * listed twice takes its last target).  An unknown id, an agent not driven by hl, a point without a leg, or an hl that
 * is not a route-table planner -> RCS_ERR_ARG and nothing is written. */
int rcs_hl_route_table_set_target(rcs_sim* sim, uint32_t hl, uint64_t n, const uint64_t* ids,
                                  const double* targets_xy);
int rcs_hl_none(rcs_sim* sim, uint32_t* out_hl);

/* ---- agents ---------------------------------------------------------------------------------- */

/* Simulation::add_agents (lib.rs:119-156).  xy = n interleaved (x,y).  Ids are allocated
 * sequentially from last_alloc_agent_id (lib.rs:128-129) and written to out_ids (may be NULL).
 * Velocity starts at (0,0), next_waypoint at 0.  Returns RCS_ERR_OUT_OF_BOUNDS if any position
 * fails location_to_index; in that case NO agent of the call is added (the reference leaves the
 * failing agent half-inserted, lib.rs:133-149 -- documented deviation). */
int rcs_add_agents(rcs_sim* sim, uint64_t n, const double* xy, uint32_t hl, uint32_t lp, double eyesight,
                   uint64_t* out_ids);
/* Simulation::remove_agents (lib.rs:176-192), batched. Unknown ids -> RCS_ERR_ARG. */
int rcs_remove_agents(rcs_sim* sim, uint64_t n, const uint64_t* ids);
/* `agents` is a pub field (lib.rs:71): position and velocity are user-writable.  Takes effect
 * immediately for the index too (snapshot injection).  ids == NULL means "all live agents in
 * ascending-id order". */
int rcs_set_state(rcs_sim* sim, uint64_t n, const uint64_t* ids, const double* x, const double* y,
                  const double* vx, const double* vy);
/* Upload Some(v) results of host-side HighLevelPlanner objects for agents of rcs_hl_host groups.
 * vxy = n interleaved (vx,vy).  ids == NULL: all live agents in ascending-id order.
 * The copy runs on an upload stream of its own, so it overlaps a step that is still in flight; the values take
 * effect for the next rcs_step*.  A pinned `vxy` (rcs_host_alloc) is read asynchronously: leave it untouched until
 * the next call that waits for the step stream (rcs_sync, rcs_step, rcs_read_agents). */
int rcs_set_preferred_velocity(rcs_sim* sim, uint64_t n, const uint64_t* ids, const double* vxy);

#define RCS_ORDER_STORAGE 0u /* device storage order (cell-sorted after a step) */
#define RCS_ORDER_ID 1u      /* ascending agent id */
/* Read back the pub `agents` view (lib.rs:71).  Any output pointer may be NULL.  cap = capacity of
 * the output arrays in agents; *out_n = number of live agents. */
int rcs_read_agents(rcs_sim* sim, uint32_t order, uint64_t cap, uint64_t* ids, double* x, double* y, double* vx,
                    double* vy, uint32_t* next_waypoint, uint64_t* out_n);
int rcs_agent_count(rcs_sim* sim, uint64_t* out_n);
/* The same view without stalling the step stream: the arrays are gathered on the device, copied to the (pinned)
 * host buffers on a second stream, and the call returns at once, so that the next rcs_set_preferred_velocity /
 * rcs_step_async overlap with the copies.  The buffers are valid after rcs_read_wait; a second async read waits
 * (on the device) for the first one's copies.  Use two sets of host buffers to double-buffer. */
int rcs_read_agents_async(rcs_sim* sim, uint32_t order, uint64_t cap, uint64_t* ids, double* x, double* y, double* vx,
                          double* vy, uint64_t* out_n);
int rcs_read_wait(rcs_sim* sim);

/* ---- the hot path ---------------------------------------------------------------------------- */

#define RCS_STEP_DEFAULT 0u
/* Run the whole pipeline but do not commit (state stays the pre-step snapshot).  Used to time the
 * force kernel on crowds that the reference model itself drives non-finite within a few steps
 * (SURVEY.md section 0.4 / 8d "frozen-snapshot mode"). */
#define RCS_STEP_NO_COMMIT 1u

/* Simulation::step(Duration::new(secs, nanos))  (lib.rs:195-383): spawn phase, per-agent update
 * (high-level velocity -> radius query -> local planner -> explicit Euler), commit, removals.
 * dt = secs as f64 + nanos as f64 / 1e9, bit-identical to Duration::as_secs_f64.
 * Synchronous.  On RCS_ERR_OUT_OF_BOUNDS the step is NOT committed (the reference aborts mid-loop
 * with a half-updated index, lib.rs:299-302 -- documented deviation). */
int rcs_step(rcs_sim* sim, uint64_t secs, uint32_t nanos);
/* Enqueue one step without waiting; errors become sticky and are returned by rcs_sync.  A step
 * enqueued after a failed one is skipped on the device. */
int rcs_step_async(rcs_sim* sim, uint64_t secs, uint32_t nanos, uint32_t flags);
int rcs_sync(rcs_sim* sim);
int rcs_step_stats(rcs_sim* sim, rcs_stats* out);

/* Study mode (SURVEY.md 8f-4): one step under the reference's IN-LOOP index semantic -- the index is updated inside
 * the per-agent loop (lib.rs:299), so agent i finds every agent that came earlier in the iteration order at its NEW
 * position and every later one at its old position, while the planner is handed their old states (lib.rs:281-286).
 * `order` = the iteration order as agent ids (the reference's is HashMap-random); n_order == 0: ascending id.  Ids
 * that are not live are ignored, live ids missing from the order come after it in ascending id, and an order that
 * repeats an id is refused with RCS_ERR_ARG before anything runs.  Computed as a fixed-point iteration of whole-crowd
 * sweeps (rcs_inloop.cuh) that ends with exactly the sequential loop's result; *out_sweeps = sweeps used,
 * max_sweeps == 0: no limit.  Sweep 0 has no previous sweep to agree with, so max_sweeps == 1 always fails; a step
 * that finds no fixed point within max_sweeps returns RCS_ERR_ARG, commits nothing and drops the trace.
 * Synchronous; one handle without strips, source sinks or route followers.  Same error behaviour as rcs_step. */
int rcs_step_in_loop(rcs_sim* sim, uint64_t secs, uint32_t nanos, const uint64_t* order, uint64_t n_order,
                     uint32_t max_sweeps, uint32_t* out_sweeps);

/* Events for EventListener::{agent_spawned, agent_destroyed} (lib.rs:22-33), accumulated since the
 * last poll, each list in ascending id order per step.  Any pointer may be NULL; counts are always
 * written. */
int rcs_poll_events(rcs_sim* sim, uint64_t spawned_cap, uint64_t* spawned_ids, double* spawned_xy,
                    uint64_t* n_spawned, uint64_t destroyed_cap, uint64_t* destroyed_ids, uint64_t* n_destroyed);

/* ---- source sinks (lib.rs:159-168, 199-254, 305-336; source_sink.rs:36-100) -------------------- */
typedef struct rcs_source_sink_desc {
  double source_x, source_y;
  double radius_sink;
  double monotonic_rate; /* MonotonicCrowd::new(rate): round(dt*rate) per step (source_sink.rs:96-100) */
  uint32_t hl, lp;
  uint64_t n_waypoints;
  const double* waypoints_xy; /* interleaved; the last waypoint is the sink */
  int32_t loop_forever;
  double agent_eyesight_range;
} rcs_source_sink_desc;
int rcs_add_source_sink(rcs_sim* sim, const rcs_source_sink_desc* desc, uint64_t* out_id);
int rcs_remove_source_sink(rcs_sim* sim, uint64_t id);

/* ---- SpatialIndex trait, batched (spatial_index.rs:4-14) ------------------------------------- */

/* LocationHash2D::location_to_index for n points (location_hash_2d.rs:54-66): data index or -1. */
int rcs_cell_of(rcs_sim* sim, uint64_t n, const double* xy, int64_t* out_idx);
/* SpatialIndex::add_or_update / remove_agent with caller-chosen ids (location_hash_2d.rs:126-149,
 * 260-267), for using the handle as a bare GpuLocationHash2D.  Ids must be < 2^31. */
int rcs_index_add_or_update(rcs_sim* sim, uint64_t n, const uint64_t* ids, const double* xy);
int rcs_index_remove(rcs_sim* sim, uint64_t n, const uint64_t* ids);
/* SpatialIndex::get_neighbours_in_radius for nq queries (location_hash_2d.rs:240-258), CSR output:
 * ids of query q are out_ids[offsets[q] .. offsets[q+1]) in canonical order (cells x-major then y,
 * ascending id inside a cell; the reference's order inside a cell is HashSet-random).  If the total
 * exceeds ids_cap, returns RCS_ERR_CAPACITY with offsets filled (offsets[nq] = required size). */
int rcs_query_radius(rcs_sim* sim, uint64_t nq, const double* qxy, const double* radius, uint64_t* offsets,
                     uint64_t* out_ids, uint64_t ids_cap);
/* SpatialIndex::get_nearest_neighbours for nq queries (location_hash_2d.rs:151-238), including its
 * ring-search quirks; out_ids has nq*k slots, out_counts[q] <= k valid entries per query.  Where the
 * reference's sort panics -- a query collects >= 2 candidates and one distance is NaN (a NaN query point,
 * or an agent at a NaN position in cell 0) -- the whole call returns RCS_ERR_ARG ("get_nearest_neighbours:
 * NaN distance") and writes neither out_ids nor out_counts. */
int rcs_query_knn(rcs_sim* sim, uint64_t nq, const double* qxy, uint64_t k, uint64_t* out_ids,
                  uint64_t* out_counts);

/* ---- parity trace -----------------------------------------------------------------------------
 * With tracing on, each step also records per agent: t_i (zanlungo.rs:76-91), the summed force
 * (zanlungo.rs:210-215), and the neighbour list handed to the local planner (lib.rs:281-286). */
int rcs_set_trace(rcs_sim* sim, int32_t on);
int rcs_trace_sizes(rcs_sim* sim, uint64_t* n_agents, uint64_t* n_neighbours);
/* Ascending-id order; nb_offsets has n_agents+1 entries. */
int rcs_read_trace(rcs_sim* sim, uint64_t* ids, double* t_i, double* fx, double* fy, uint64_t* nb_offsets,
                   uint64_t* nb_ids);

/* ---- options ------------------------------------------------------------------------------------ */
#define RCS_OPT_STEP_KERNEL 1u /* 0 = default (3), 1 = thread-per-agent, 2 = warp-cooperative through L1, 3 = stencil staged in shared memory */
/* Option numbers 2 and 4 are retired and are not reused: rcs_set_option refuses them as unknown options. */
/* 1 (default) = a step whose launch sequence repeats (nothing to upload, no trace, no kernel timing) is captured into a
 * CUDA graph the second time it comes up and is one graph launch from then on; 0 = always launch kernel by kernel. */
#define RCS_OPT_GRAPHS 3u
int rcs_set_option(rcs_sim* sim, uint32_t option, uint64_t value);

/* ---- measurement helpers ---------------------------------------------------------------------- */
#define RCS_NUM_EVENTS 64u
int rcs_event_record(rcs_sim* sim, uint32_t slot);
int rcs_event_elapsed_ms(rcs_sim* sim, uint32_t start_slot, uint32_t stop_slot, float* out_ms);
/* Pinned host memory so that host<->device copies of caller buffers run at full PCIe rate. */
int rcs_host_alloc(uint64_t bytes, void** out);
int rcs_host_free(void* p);
/* Write a device buffer of `bytes` (> L2) on the handle's stream to evict L2 between timed steps. */
int rcs_flush_l2(rcs_sim* sim, uint64_t bytes);
/* Bracket the dominant kernel (step_kernel) of every step with CUDA events on the launching stream;
 * rcs_kernel_time_ms returns the accumulated device time and the number of launches since timing
 * was switched on (it waits for the stream). */
int rcs_kernel_timing(rcs_sim* sim, int32_t on);
int rcs_kernel_time_ms(rcs_sim* sim, double* out_ms, uint64_t* out_launches);
/* Number of kernels launched by this handle so far (kernels inside graph launches included). */
int rcs_launch_count(rcs_sim* sim, uint64_t* out);
/* Steps that ran as one CUDA graph launch, and graphs captured so far (RCS_OPT_GRAPHS). */
int rcs_graph_stats(rcs_sim* sim, uint64_t* out_graph_launches, uint64_t* out_captures);
/* FP64 pipe peak microbenchmark (dependent DFMA chains on all SMs); out_tflops counts FMA = 2. */
int rcs_fp64_peak(int32_t device, double* out_tflops, double* out_dadd_tops);

/* ---- multi-GPU spatial strips (SURVEY.md section 8e) ------------------------------------------
 * One process per GPU.  Strips are whole cell columns in x (the cell index is x-major,
 * location_hash_2d.rs:59), so a strip is a contiguous range of cell indices.  Every step a rank sends
 * the agents of its boundary columns to its two neighbours (NCCL point-to-point over NVLink) and
 * advances the ghosts of the first column beyond its boundary redundantly, which makes migration
 * implicit (see rcs_host_dist.inl).  Results are bit-identical for every number of ranks.
 *
 * rcs_nccl_unique_id is called on rank 0 and the 128 bytes are distributed by the host program (e.g.
 * torch.distributed); rcs_dist_init then builds the NCCL communicator inside the library.  It must be
 * called before agents are added; each rank then adds the agents whose column it owns
 * (rcs_dist_strip) with rcs_dist_add_agents.  halo_capacity = agents per halo buffer (0: capacity/8).
 * A failing step (out of bounds, halo overflow, an agent that jumps over the ring) stops the rank and,
 * through a flag in the halo header, its neighbours within the next steps; the job is then over. */
int rcs_nccl_unique_id(uint8_t out_id[128]);
int rcs_dist_init(rcs_sim* sim, int32_t rank, int32_t world, const uint8_t nccl_id[128], uint64_t halo_capacity);
/* Optional, before rcs_dist_init, the same call on every rank: the strips' cell-column boundaries (world + 1 values
 * rising strictly from 0 to the number of cell columns) instead of the equal split -- e.g. balanced by agent count
 * when the crowd does not fill the grid.  bounds == NULL: back to the equal split. */
int rcs_dist_set_boundaries(rcs_sim* sim, int32_t world, const uint64_t* bounds);
/* Optional, after rcs_dist_init on a multi-process job in which every rank has its own GPU: the peer-store halo
 * transport.  rcs_dist_peer_export returns the CUDA IPC handle (64 bytes) of this rank's receive arena; the host
 * program distributes the handles (e.g. torch.distributed.all_gather) and gives every rank its two neighbours'
 * (NULL where there is none) with rcs_dist_peer_connect.  From then on the binning pass stores the boundary columns
 * straight into the neighbour's memory over NVLink and a one-block kernel releases the round number the neighbour's
 * unpack kernel waits for (at most 120 s, then the step fails): no ncclSend / ncclRecv in the step, and a steady-state
 * step replays as one CUDA graph.  Every rank of the job must connect before the next step.  NCCL stays in use for
 * the spawn-set all-reduce of source sinks. */
int rcs_dist_peer_export(rcs_sim* sim, uint8_t out_handle[64]);
int rcs_dist_peer_connect(rcs_sim* sim, const uint8_t* left_handle, const uint8_t* right_handle);
/* Back to the NCCL transport (e.g. because rcs_dist_peer_connect failed on SOME rank -- no peer access between two of
 * the GPUs -- and the host program has agreed on that over its own channel): every rank of the job calls it before
 * the next step. */
int rcs_dist_peer_disable(rcs_sim* sim);
/* Column range [c0, c1) owned by `rank` of `world` for this handle's grid. */
int rcs_dist_strip(rcs_sim* sim, int32_t rank, int32_t world, uint64_t* c0, uint64_t* c1);
/* add_agents with caller-supplied global ids (the global sequential allocation of lib.rs:128-129
 * is done by the host program across ranks) and initial velocities (vxy may be NULL).  Ghosts carry the number of
 * their (high-level planner, local planner, eyesight) group: EVERY rank makes the same calls in the same order, with
 * n = 0 where none of the batch lies in its strip, so that the group tables agree.  Ids must be < 2^32 (the id -> slot
 * tables are dense over the id range). */
int rcs_dist_add_agents(rcs_sim* sim, uint64_t n, const uint64_t* ids, const double* xy, const double* vxy,
                        uint32_t hl, uint32_t lp, double eyesight);
/* The ids source sinks allocate on this handle (lib.rs:128-129) start at next_id or later.  After rcs_dist_add_agents,
 * every rank calls it with the same value -- one past the largest id the host program has handed out -- so that the
 * ranks number their spawns alike and after the caller's agents.  next_id < 2^32. */
int rcs_dist_reserve_ids(rcs_sim* sim, uint64_t next_id);
/* Single-process transport: sims[r] is rank r of `world` handles that live in this process (on one
 * or several devices); halos move with peer copies ordered by events.  The group is stepped as a
 * whole; rcs_sync / rcs_read_agents / rcs_step_stats work per handle.  Used to test strips on one
 * GPU with the very kernels the NCCL transport runs. */
int rcs_dist_init_local(rcs_sim** sims, int32_t world, uint64_t halo_capacity);
int rcs_dist_step_local(rcs_sim** sims, int32_t world, uint64_t secs, uint32_t nanos, uint32_t flags);

#ifdef __cplusplus
}
#endif
#endif /* RCS_H_ */
