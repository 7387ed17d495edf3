//! Safe wrapper over `rmf_crowdsim_gpu-sys` that mirrors `rmf_crowdsim::Simulation` (rmf_crowdsim/src/lib.rs:69-384).
//!
//! The reference calls planners per agent per step behind `Arc<Mutex<dyn Trait>>` (lib.rs:264-291); a GPU backend
//! replaces the whole per-step update instead, so planners are DESCRIBED (`LocalPlan`, `HighLevelPlan`) and
//! evaluated on the device.  User-implemented `HighLevelPlanner` trait objects stay usable through
//! `HighLevelPlan::Host` (positions down, preferred velocities up, every step).
use nalgebra::Vector2;
use rmf_crowdsim_gpu_sys as sys;
use std::collections::HashMap;
use std::ffi::CStr;
use std::ptr;
use std::sync::{Arc, Mutex};
use std::time::Duration;

pub type AgentId = usize;
pub type Vec2f = Vector2<f64>;
pub type Point = Vector2<f64>;

/// lib.rs:46-65 (orientation / angular_vel are never written by the reference and stay 0)
#[derive(Clone, Debug)]
pub struct Agent {
    pub agent_id: AgentId,
    pub position: Point,
    pub orientation: f64,
    pub velocity: Vec2f,
    pub angular_vel: f64,
    pub next_waypoint: usize,
    pub eyesight_range: f64,
}

/// highlevel_planners/highlevel_planners.rs:8-16
pub trait HighLevelPlanner {
    fn get_desired_velocity(&mut self, agent: &Agent, time: Duration) -> Option<Vec2f>;
    fn set_target(&mut self, agent: &Agent, point: Point, tolerance: Vec2f);
    fn remove_agent_id(&mut self, agent: AgentId);
}

/// lib.rs:22-33
pub trait EventListener {
    fn agent_spawned(&mut self, position: Vec2f, agent: AgentId);
    fn agent_destroyed(&mut self, agent: AgentId);
    fn waypoint_reached(&mut self, _position: Vec2f, _agent: AgentId) {}
}

/// local_planners/{no_local_plan.rs, zanlungo.rs}; `Zanlungo` has the argument order of `Zanlungo::new` (:31-38)
#[derive(Clone, Copy, Debug)]
pub enum LocalPlan {
    NoLocalPlan,
    Zanlungo { agent_scale: f64, obstacle_scale: f64, reaction_time: f64, force_distance: f64, agent_mass: f64, agent_radius: f64 },
}

#[derive(Clone)]
pub enum HighLevelPlan {
    /// always `Some(v)`
    Constant(Vec2f),
    /// even id -> `Some(-v)`, odd -> `Some(v)` (rmf_crowdsim_viz/src/main.rs:20-30)
    Parity(Vec2f),
    /// always `None`
    None,
    /// the per-step half of `rmf::RMFPlanner` (rmf/mod.rs:197-215) on a route the host planned
    Route(Vec<Point>),
    /// `rmf::RMFPlanner` (rmf/mod.rs:86-241) with a route cache the host filled: (target, route) legs;
    /// `set_target(point)` selects the leg whose target equals the point.  A source sink with this planner may have
    /// any number of waypoints, each with a leg.
    RouteTable(Vec<(Point, Vec<Point>)>),
    /// any user planner, evaluated on the host every step
    Host(Arc<Mutex<dyn HighLevelPlanner>>),
}

/// source_sink/source_sink.rs:36-60 with `MonotonicCrowd::new(rate)`
pub struct SourceSink {
    pub source: Vec2f,
    pub radius_sink: f64,
    pub monotonic_rate: f64,
    pub high_level_planner: HighLevelPlan,
    pub local_planner: LocalPlan,
    pub waypoints: Vec<Vec2f>,
    pub loop_forever: bool,
    pub agent_eyesight_range: f64,
}

pub struct Simulation {
    h: *mut sys::rcs_sim,
    host_hl: HashMap<AgentId, Arc<Mutex<dyn HighLevelPlanner>>>,
    hl_host_handle: Option<u32>,
    eyesight: HashMap<AgentId, f64>,
    listeners: Vec<Arc<Mutex<dyn EventListener>>>,
}

fn check(h: *mut sys::rcs_sim, rc: i32) -> Result<(), String> {
    if rc == sys::RCS_OK {
        return Ok(());
    }
    let msg = unsafe { CStr::from_ptr(sys::rcs_last_error(h)) }.to_string_lossy().into_owned();
    Err(if msg.is_empty() { format!("rcs error {}", rc) } else { msg })
}

impl Simulation {
    /// `Simulation::new(LocationHash2D::new(width, height, cell_size, offset))` (lib.rs:103, location_hash_2d.rs:33)
    pub fn new(width: f64, height: f64, cell_size: f64, offset: Point, capacity: usize, device: i32) -> Result<Self, String> {
        let desc = sys::rcs_sim_desc { width, height, cell_size, offset_x: offset.x, offset_y: offset.y,
                                       capacity: capacity as u64, device, flags: 0 };
        let mut h: *mut sys::rcs_sim = ptr::null_mut();
        check(ptr::null_mut(), unsafe { sys::rcs_sim_create(&desc, &mut h) })?;
        Ok(Simulation { h, host_hl: HashMap::new(), hl_host_handle: None, eyesight: HashMap::new(), listeners: vec![] })
    }

    fn lp(&mut self, lp: LocalPlan) -> Result<u32, String> {
        let mut out = 0u32;
        let rc = match lp {
            LocalPlan::NoLocalPlan => unsafe { sys::rcs_lp_none(self.h, &mut out) },
            LocalPlan::Zanlungo { agent_scale, obstacle_scale, reaction_time, force_distance, agent_mass, agent_radius } => unsafe {
                sys::rcs_lp_zanlungo(self.h, agent_scale, obstacle_scale, reaction_time, force_distance, agent_mass, agent_radius, &mut out)
            },
        };
        check(self.h, rc).map(|_| out)
    }

    fn hl(&mut self, hl: &HighLevelPlan) -> Result<u32, String> {
        let mut out = 0u32;
        let rc = match hl {
            HighLevelPlan::Constant(v) => unsafe { sys::rcs_hl_constant(self.h, v.x, v.y, &mut out) },
            HighLevelPlan::Parity(v) => unsafe { sys::rcs_hl_parity(self.h, v.x, v.y, &mut out) },
            HighLevelPlan::None => unsafe { sys::rcs_hl_none(self.h, &mut out) },
            HighLevelPlan::Route(r) => {
                let xy: Vec<f64> = r.iter().flat_map(|p| [p.x, p.y]).collect();
                unsafe { sys::rcs_hl_route(self.h, r.len() as u64, xy.as_ptr(), &mut out) }
            }
            HighLevelPlan::RouteTable(legs) => {
                let targets: Vec<f64> = legs.iter().flat_map(|(t, _)| [t.x, t.y]).collect();
                let counts: Vec<u64> = legs.iter().map(|(_, r)| r.len() as u64).collect();
                let xy: Vec<f64> = legs.iter().flat_map(|(_, r)| r.iter().flat_map(|p| [p.x, p.y])).collect();
                unsafe {
                    sys::rcs_hl_route_table(self.h, legs.len() as u64, targets.as_ptr(), counts.as_ptr(), xy.as_ptr(),
                                            &mut out)
                }
            }
            HighLevelPlan::Host(_) => {
                if let Some(hh) = self.hl_host_handle {
                    out = hh;
                    sys::RCS_OK
                } else {
                    let rc = unsafe { sys::rcs_hl_host(self.h, &mut out) };
                    self.hl_host_handle = Some(out);
                    rc
                }
            }
        };
        check(self.h, rc).map(|_| out)
    }

    /// lib.rs:119-156 — ids are allocated sequentially; `Err("Index out of bounds")` as the reference
    pub fn add_agents(&mut self, spawn_positions: &Vec<Point>, high_level_planner: HighLevelPlan, local_planner: LocalPlan,
                      agent_eyesight_range: f64) -> Result<Vec<AgentId>, String> {
        let (hl, lp) = (self.hl(&high_level_planner)?, self.lp(local_planner)?);
        let xy: Vec<f64> = spawn_positions.iter().flat_map(|p| [p.x, p.y]).collect();
        let mut ids = vec![0u64; spawn_positions.len()];
        check(self.h, unsafe { sys::rcs_add_agents(self.h, ids.len() as u64, xy.as_ptr(), hl, lp, agent_eyesight_range, ids.as_mut_ptr()) })?;
        let ids: Vec<AgentId> = ids.into_iter().map(|v| v as AgentId).collect();
        for (k, id) in ids.iter().enumerate() {
            self.eyesight.insert(*id, agent_eyesight_range);
            if let HighLevelPlan::Host(p) = &high_level_planner {
                self.host_hl.insert(*id, p.clone());
            }
            for l in &self.listeners {
                l.lock().unwrap().agent_spawned(spawn_positions[k], *id);
            }
        }
        Ok(ids)
    }

    /// lib.rs:159-162 (MonotonicCrowd generators run on the device; PoissonCrowd uses thread_rng and has no device form)
    pub fn add_source_sink(&mut self, ss: &SourceSink) -> Result<usize, String> {
        let (hl, lp) = (self.hl(&ss.high_level_planner)?, self.lp(ss.local_planner)?);
        let wp: Vec<f64> = ss.waypoints.iter().flat_map(|p| [p.x, p.y]).collect();
        let desc = sys::rcs_source_sink_desc { source_x: ss.source.x, source_y: ss.source.y, radius_sink: ss.radius_sink,
            monotonic_rate: ss.monotonic_rate, hl, lp, n_waypoints: ss.waypoints.len() as u64, waypoints_xy: wp.as_ptr(),
            loop_forever: ss.loop_forever as i32, agent_eyesight_range: ss.agent_eyesight_range };
        let mut id = 0u64;
        check(self.h, unsafe { sys::rcs_add_source_sink(self.h, &desc, &mut id) })?;
        Ok(id as usize)
    }

    /// lib.rs:164-168
    pub fn remove_source_sink(&mut self, id: &usize) -> Result<(), String> {
        check(self.h, unsafe { sys::rcs_remove_source_sink(self.h, *id as u64) })
    }

    /// lib.rs:170-173
    pub fn add_event_listener(&mut self, l: Arc<Mutex<dyn EventListener>>) -> usize {
        self.listeners.push(l);
        self.listeners.len() - 1
    }

    /// lib.rs:176-192
    pub fn remove_agents(&mut self, agent: AgentId) -> Result<(), String> {
        let id = agent as u64;
        check(self.h, unsafe { sys::rcs_remove_agents(self.h, 1, &id) })?;
        if let Some(p) = self.host_hl.remove(&agent) {
            p.lock().unwrap().remove_agent_id(agent);
        }
        for l in &self.listeners {
            l.lock().unwrap().agent_destroyed(agent);
        }
        Ok(())
    }

    /// The pub `agents` field of the reference (lib.rs:71), materialised on demand in ascending id.
    pub fn agents(&mut self) -> Result<Vec<Agent>, String> {
        let mut n = 0u64;
        check(self.h, unsafe { sys::rcs_agent_count(self.h, &mut n) })?;
        let n = n as usize;
        let (mut ids, mut wp) = (vec![0u64; n], vec![0u32; n]);
        let (mut x, mut y, mut vx, mut vy) = (vec![0f64; n], vec![0f64; n], vec![0f64; n], vec![0f64; n]);
        let mut out_n = 0u64;
        check(self.h, unsafe {
            sys::rcs_read_agents(self.h, sys::RCS_ORDER_ID, n as u64, ids.as_mut_ptr(), x.as_mut_ptr(), y.as_mut_ptr(),
                                 vx.as_mut_ptr(), vy.as_mut_ptr(), wp.as_mut_ptr(), &mut out_n)
        })?;
        Ok((0..n).map(|k| Agent {
            agent_id: ids[k] as AgentId, position: Point::new(x[k], y[k]), orientation: 0.0,
            velocity: Vec2f::new(vx[k], vy[k]), angular_vel: 0.0, next_waypoint: wp[k] as usize,
            eyesight_range: *self.eyesight.get(&(ids[k] as AgentId)).unwrap_or(&0.0),
        }).collect())
    }

    /// lib.rs:195-383 — one call replaces the spawn phase, the per-agent loop, the commit and the removals.
    pub fn step(&mut self, dur: Duration) -> Result<(), String> {
        if !self.host_hl.is_empty() {
            // slow path for user trait objects (lib.rs:264-273); sim_time is never advanced by the reference (:81, :110)
            let agents = self.agents()?;
            let (mut ids, mut vxy) = (Vec::new(), Vec::new());
            for a in &agents {
                if let Some(p) = self.host_hl.get(&a.agent_id) {
                    let v = p.lock().unwrap().get_desired_velocity(a, Duration::new(0, 0));
                    ids.push(a.agent_id as u64);
                    match v {
                        Some(v) => vxy.extend_from_slice(&[v.x, v.y]),
                        None => vxy.extend_from_slice(&[f64::NAN, f64::NAN]),
                    }
                }
            }
            check(self.h, unsafe { sys::rcs_set_preferred_velocity(self.h, ids.len() as u64, ids.as_ptr(), vxy.as_ptr()) })?;
        }
        check(self.h, unsafe { sys::rcs_step(self.h, dur.as_secs(), dur.subsec_nanos()) })?;
        self.dispatch_events()
    }

    fn dispatch_events(&mut self) -> Result<(), String> {
        let (mut ns, mut nd) = (0u64, 0u64);
        check(self.h, unsafe { sys::rcs_poll_events(self.h, 0, ptr::null_mut(), ptr::null_mut(), &mut ns, 0, ptr::null_mut(), &mut nd) })?;
        if ns == 0 && nd == 0 {
            return Ok(());
        }
        let (mut sid, mut sxy, mut did) = (vec![0u64; ns as usize], vec![0f64; 2 * ns as usize], vec![0u64; nd as usize]);
        check(self.h, unsafe {
            sys::rcs_poll_events(self.h, ns, sid.as_mut_ptr(), sxy.as_mut_ptr(), &mut ns, nd, did.as_mut_ptr(), &mut nd)
        })?;
        for k in 0..ns as usize {
            for l in &self.listeners {
                l.lock().unwrap().agent_spawned(Vec2f::new(sxy[2 * k], sxy[2 * k + 1]), sid[k] as AgentId);
            }
        }
        for k in 0..nd as usize {
            let id = did[k] as AgentId;
            if let Some(p) = self.host_hl.remove(&id) {
                p.lock().unwrap().remove_agent_id(id);
            }
            self.eyesight.remove(&id);
            for l in &self.listeners {
                l.lock().unwrap().agent_destroyed(id);
            }
        }
        Ok(())
    }

    // ---- SpatialIndex trait methods (spatial_index/spatial_index.rs:4-14), served by the same handle --------------
    pub fn get_neighbours_in_radius(&mut self, radius: f64, position: Point) -> Result<Vec<AgentId>, String> {
        let q = [position.x, position.y];
        let mut offsets = [0u64; 2];
        let mut cap = 64u64;
        loop {
            let mut ids = vec![0u64; cap as usize];
            let rc = unsafe { sys::rcs_query_radius(self.h, 1, q.as_ptr(), &radius, offsets.as_mut_ptr(), ids.as_mut_ptr(), cap) };
            if rc == sys::RCS_ERR_CAPACITY {
                cap = offsets[1] + 1;
                continue;
            }
            check(self.h, rc)?;
            ids.truncate(offsets[1] as usize);
            return Ok(ids.into_iter().map(|v| v as AgentId).collect());
        }
    }

    pub fn get_nearest_neighbours(&mut self, n: usize, position: Point) -> Result<Vec<AgentId>, String> {
        let q = [position.x, position.y];
        let mut ids = vec![0u64; n.max(1)];
        let mut count = 0u64;
        check(self.h, unsafe { sys::rcs_query_knn(self.h, 1, q.as_ptr(), n as u64, ids.as_mut_ptr(), &mut count) })?;
        ids.truncate(count as usize);
        Ok(ids.into_iter().map(|v| v as AgentId).collect())
    }
}

/// spatial_index/spatial_index.rs:4-14, verbatim: the trait the reference's `Simulation<T: SpatialIndex>` is generic
/// over.  `GpuLocationHash2D` implements it, so code written against the trait (or against `LocationHash2D`'s own
/// methods, location_hash_2d.rs:126-267) compiles unchanged with the device-backed index.  The trait's read methods
/// take `&self`; the handle needs `&mut`, hence the `RefCell`, as single-threaded as the reference itself.
pub trait SpatialIndex {
    fn add_or_update(&mut self, id: AgentId, position: Point) -> Result<(), String>;
    fn get_nearest_neighbours(&self, n: usize, position: Point) -> Vec<AgentId>;
    fn get_neighbours_in_radius(&self, radius: f64, position: Point) -> Vec<AgentId>;
    fn remove_agent(&mut self, _id: AgentId) {}
}

/// `LocationHash2D::new(width, height, cell_size, offset)` (location_hash_2d.rs:33-51) on the device, usable on its
/// own (rcs_index_add_or_update / rcs_index_remove / rcs_query_radius / rcs_query_knn).
pub struct GpuLocationHash2D {
    sim: std::cell::RefCell<Simulation>,
}

impl GpuLocationHash2D {
    pub fn new(width: f64, height: f64, cell_size: f64, offset: Point, capacity: usize, device: i32) -> Result<Self, String> {
        Ok(GpuLocationHash2D { sim: std::cell::RefCell::new(Simulation::new(width, height, cell_size, offset, capacity, device)?) })
    }
}

impl SpatialIndex for GpuLocationHash2D {
    /// location_hash_2d.rs:126-149; `Err("Index out of bounds")` as the reference
    fn add_or_update(&mut self, id: AgentId, position: Point) -> Result<(), String> {
        let sim = self.sim.get_mut();
        let (ids, xy) = ([id as u64], [position.x, position.y]);
        check(sim.h, unsafe { sys::rcs_index_add_or_update(sim.h, 1, ids.as_ptr(), xy.as_ptr()) })
    }
    /// location_hash_2d.rs:151-238 (ring walk, quirks included)
    fn get_nearest_neighbours(&self, n: usize, position: Point) -> Vec<AgentId> {
        self.sim.borrow_mut().get_nearest_neighbours(n, position).unwrap_or_default()
    }
    /// location_hash_2d.rs:240-258 (strict `<`; cells x-major then y, ascending id inside a cell)
    fn get_neighbours_in_radius(&self, radius: f64, position: Point) -> Vec<AgentId> {
        self.sim.borrow_mut().get_neighbours_in_radius(radius, position).unwrap_or_default()
    }
    /// location_hash_2d.rs:260-267
    fn remove_agent(&mut self, id: AgentId) {
        let sim = self.sim.get_mut();
        let ids = [id as u64];
        let _ = unsafe { sys::rcs_index_remove(sim.h, 1, ids.as_ptr()) };
    }
}

/// local_planners/local_planner.rs:7-18, verbatim.  The per-agent call cannot carry a device backend (one virtual call
/// per agent per step, `Agent::preferred_vel` private: SURVEY.md 8b), so the descriptors implement it only as the
/// planner's host-side definition for ONE agent -- what `Simulation::step` evaluates for all agents on the device.
pub trait LocalPlanner {
    fn get_desired_velocity(&self, agent: &Agent, nearby_agents: &Vec<Agent>, recommended_velocity: Vec2f) -> Vec2f;
    fn add_agent(&mut self, _agent: AgentId) {}
    fn remove_agent(&mut self, _agent: AgentId) {}
}

impl LocalPlanner for LocalPlan {
    fn get_desired_velocity(&self, _agent: &Agent, _nearby_agents: &Vec<Agent>, recommended_velocity: Vec2f) -> Vec2f {
        match self {
            // no_local_plan.rs:10-17
            LocalPlan::NoLocalPlan => recommended_velocity,
            // zanlungo.rs:201-218 runs on the device inside Simulation::step; a one-agent host evaluation would need
            // the private preferred_vel the reference hides from planners outside its crate
            LocalPlan::Zanlungo { .. } => unimplemented!("Zanlungo is evaluated for the whole crowd by Simulation::step"),
        }
    }
}

impl Drop for Simulation {
    fn drop(&mut self) {
        unsafe { sys::rcs_sim_destroy(self.h) }
    }
}
