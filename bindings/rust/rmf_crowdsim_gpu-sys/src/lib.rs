//! Raw declarations of `include/rcs.h` (ABI version 1).  Every function returns 0 on success; on failure
//! `rcs_last_error` holds the message (the reference's literal strings where it has one).
#![allow(non_camel_case_types)]
use std::os::raw::{c_char, c_int};

#[repr(C)]
pub struct rcs_sim {
    _private: [u8; 0],
}

pub const RCS_OK: c_int = 0;
pub const RCS_ERR_OUT_OF_BOUNDS: c_int = 1;
pub const RCS_ERR_SPAWN: c_int = 2;
pub const RCS_ERR_CUDA: c_int = 3;
pub const RCS_ERR_NCCL: c_int = 4;
pub const RCS_ERR_CAPACITY: c_int = 5;
pub const RCS_ERR_ARG: c_int = 6;
pub const RCS_ERR_NO_DEVICE: c_int = 7;
pub const RCS_ERR_HALO: c_int = 8;
pub const RCS_ORDER_STORAGE: u32 = 0;
pub const RCS_ORDER_ID: u32 = 1;
pub const RCS_STEP_DEFAULT: u32 = 0;
pub const RCS_STEP_NO_COMMIT: u32 = 1;

/// `LocationHash2D::new(width, height, cell_size, offset)` (spatial_index/location_hash_2d.rs:33) + placement.
#[repr(C)]
pub struct rcs_sim_desc {
    pub width: f64,
    pub height: f64,
    pub cell_size: f64,
    pub offset_x: f64,
    pub offset_y: f64,
    pub capacity: u64,
    pub device: i32,
    pub flags: u32,
}

#[repr(C)]
#[derive(Default, Debug, Clone, Copy)]
pub struct rcs_stats {
    pub n_agents: u64,
    pub oob_count: u64,
    pub first_oob_id: u64,
    pub nonfinite_count: u64,
    pub finite_tti_count: u64,
    pub neighbour_total: u64,
    pub candidate_total: u64,
    pub spawned: u64,
    pub destroyed: u64,
    pub steps: u64,
}

/// `SourceSink` (source_sink/source_sink.rs:36-60) with a `MonotonicCrowd` generator (:85-100).
#[repr(C)]
pub struct rcs_source_sink_desc {
    pub source_x: f64,
    pub source_y: f64,
    pub radius_sink: f64,
    pub monotonic_rate: f64,
    pub hl: u32,
    pub lp: u32,
    pub n_waypoints: u64,
    pub waypoints_xy: *const f64,
    pub loop_forever: i32,
    pub agent_eyesight_range: f64,
}

pub const RCS_CROWD_MONOTONIC: u32 = 0;
pub const RCS_CROWD_POISSON: u32 = 1;
pub const RCS_CROWD_HOST: u32 = 2;

/// `CrowdGenerator` of a source sink (source_sink.rs:63-100): `MonotonicCrowd::new(rate)`, `PoissonCrowd::new(rate)` with
/// a keyed draw (`seed`; reproducible), or a user generator evaluated by the caller (`rcs_set_spawn_counts`).
#[repr(C)]
#[derive(Default, Debug, Clone, Copy)]
pub struct rcs_crowd_generator {
    pub kind: u32,
    pub reserved: u32,
    pub rate: f64,
    pub seed: u64,
}

extern "C" {
    pub fn rcs_abi_version() -> u32;
    pub fn rcs_sim_create(desc: *const rcs_sim_desc, out: *mut *mut rcs_sim) -> c_int;
    pub fn rcs_sim_destroy(sim: *mut rcs_sim);
    pub fn rcs_last_error(sim: *const rcs_sim) -> *const c_char;

    pub fn rcs_lp_none(sim: *mut rcs_sim, out_lp: *mut u32) -> c_int;
    pub fn rcs_lp_zanlungo(sim: *mut rcs_sim, agent_scale: f64, obstacle_scale: f64, reaction_time: f64,
                           force_distance: f64, agent_mass: f64, agent_radius: f64, out_lp: *mut u32) -> c_int;
    pub fn rcs_hl_constant(sim: *mut rcs_sim, vx: f64, vy: f64, out_hl: *mut u32) -> c_int;
    pub fn rcs_hl_parity(sim: *mut rcs_sim, vx: f64, vy: f64, out_hl: *mut u32) -> c_int;
    pub fn rcs_hl_host(sim: *mut rcs_sim, out_hl: *mut u32) -> c_int;
    pub fn rcs_hl_none(sim: *mut rcs_sim, out_hl: *mut u32) -> c_int;
    pub fn rcs_hl_route(sim: *mut rcs_sim, n_points: u64, xy: *const f64, out_hl: *mut u32) -> c_int;
    pub fn rcs_hl_route_set_target(sim: *mut rcs_sim, n: u64, ids: *const u64) -> c_int;
    pub fn rcs_hl_route_table(sim: *mut rcs_sim, n_legs: u64, targets_xy: *const f64, leg_points: *const u64,
                              xy: *const f64, out_hl: *mut u32) -> c_int;
    pub fn rcs_hl_route_table_set_target(sim: *mut rcs_sim, hl: u32, n: u64, ids: *const u64,
                                         targets_xy: *const f64) -> c_int;

    pub fn rcs_add_agents(sim: *mut rcs_sim, n: u64, xy: *const f64, hl: u32, lp: u32, eyesight: f64,
                          out_ids: *mut u64) -> c_int;
    pub fn rcs_remove_agents(sim: *mut rcs_sim, n: u64, ids: *const u64) -> c_int;
    pub fn rcs_set_state(sim: *mut rcs_sim, n: u64, ids: *const u64, x: *const f64, y: *const f64,
                         vx: *const f64, vy: *const f64) -> c_int;
    pub fn rcs_set_preferred_velocity(sim: *mut rcs_sim, n: u64, ids: *const u64, vxy: *const f64) -> c_int;
    pub fn rcs_read_agents(sim: *mut rcs_sim, order: u32, cap: u64, ids: *mut u64, x: *mut f64, y: *mut f64,
                           vx: *mut f64, vy: *mut f64, next_waypoint: *mut u32, out_n: *mut u64) -> c_int;
    pub fn rcs_read_agents_async(sim: *mut rcs_sim, order: u32, cap: u64, ids: *mut u64, x: *mut f64,
                                 y: *mut f64, vx: *mut f64, vy: *mut f64, out_n: *mut u64) -> c_int;
    pub fn rcs_read_wait(sim: *mut rcs_sim) -> c_int;
    pub fn rcs_agent_count(sim: *mut rcs_sim, out_n: *mut u64) -> c_int;

    pub fn rcs_step(sim: *mut rcs_sim, secs: u64, nanos: u32) -> c_int;
    pub fn rcs_step_async(sim: *mut rcs_sim, secs: u64, nanos: u32, flags: u32) -> c_int;
    pub fn rcs_sync(sim: *mut rcs_sim) -> c_int;
    pub fn rcs_step_stats(sim: *mut rcs_sim, out: *mut rcs_stats) -> c_int;
    pub fn rcs_step_in_loop(sim: *mut rcs_sim, secs: u64, nanos: u32, order: *const u64, n_order: u64,
                            max_sweeps: u32, out_sweeps: *mut u32) -> c_int;
    pub fn rcs_poll_events(sim: *mut rcs_sim, spawned_cap: u64, spawned_ids: *mut u64, spawned_xy: *mut f64,
                           n_spawned: *mut u64, destroyed_cap: u64, destroyed_ids: *mut u64,
                           n_destroyed: *mut u64) -> c_int;
    pub fn rcs_add_source_sink(sim: *mut rcs_sim, desc: *const rcs_source_sink_desc, out_id: *mut u64) -> c_int;
    pub fn rcs_remove_source_sink(sim: *mut rcs_sim, id: u64) -> c_int;
    pub fn rcs_add_source_sink_gen(sim: *mut rcs_sim, desc: *const rcs_source_sink_desc, gen: *const rcs_crowd_generator,
                                   out_id: *mut u64) -> c_int;
    pub fn rcs_set_spawn_counts(sim: *mut rcs_sim, n: u64, ids: *const u64, counts: *const u64) -> c_int;

    pub fn rcs_cell_of(sim: *mut rcs_sim, n: u64, xy: *const f64, out_idx: *mut i64) -> c_int;
    pub fn rcs_index_add_or_update(sim: *mut rcs_sim, n: u64, ids: *const u64, xy: *const f64) -> c_int;
    pub fn rcs_index_remove(sim: *mut rcs_sim, n: u64, ids: *const u64) -> c_int;
    pub fn rcs_query_radius(sim: *mut rcs_sim, nq: u64, qxy: *const f64, radius: *const f64, offsets: *mut u64,
                            out_ids: *mut u64, ids_cap: u64) -> c_int;
    pub fn rcs_query_knn(sim: *mut rcs_sim, nq: u64, qxy: *const f64, k: u64, out_ids: *mut u64,
                         out_counts: *mut u64) -> c_int;

    /// options: 1 = step kernel form, 3 = CUDA graphs for steady-state steps (include/rcs.h)
    pub fn rcs_set_option(sim: *mut rcs_sim, option: u32, value: u64) -> c_int;
    pub fn rcs_graph_stats(sim: *mut rcs_sim, out_graph_launches: *mut u64, out_captures: *mut u64) -> c_int;

    pub fn rcs_nccl_unique_id(out_id: *mut u8) -> c_int;
    pub fn rcs_dist_init(sim: *mut rcs_sim, rank: i32, world: i32, nccl_id: *const u8, halo_capacity: u64) -> c_int;
    pub fn rcs_dist_set_boundaries(sim: *mut rcs_sim, world: i32, bounds: *const u64) -> c_int;
    pub fn rcs_dist_reserve_ids(sim: *mut rcs_sim, next_id: u64) -> c_int;
    pub fn rcs_dist_peer_export(sim: *mut rcs_sim, out_handle: *mut u8) -> c_int;
    pub fn rcs_dist_peer_connect(sim: *mut rcs_sim, left_handle: *const u8, right_handle: *const u8) -> c_int;
    pub fn rcs_dist_peer_disable(sim: *mut rcs_sim) -> c_int;
    pub fn rcs_dist_strip(sim: *mut rcs_sim, rank: i32, world: i32, c0: *mut u64, c1: *mut u64) -> c_int;
    pub fn rcs_dist_add_agents(sim: *mut rcs_sim, n: u64, ids: *const u64, xy: *const f64, vxy: *const f64,
                               hl: u32, lp: u32, eyesight: f64) -> c_int;
}
