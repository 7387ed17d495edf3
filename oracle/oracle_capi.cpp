// oracle_capi.cpp -- ctypes-facing C API of the CPU ORACLE (TEST INFRASTRUCTURE ONLY; see
// crowdsim_oracle.hpp).  The functions deliberately mirror include/rcs.h so that the parity
// tests drive oracle and CUDA path with the same calls.  Not part of the product.
#include <cstring>

#include "crowdsim_oracle.hpp"

using namespace orc;

namespace {

struct RecordingListener : EventListener {
  std::vector<AgentId> spawned_ids;
  std::vector<Vec2> spawned_pos;
  std::vector<AgentId> destroyed_ids;
  void agent_spawned(Vec2 p, AgentId a) override {
    spawned_ids.push_back(a);
    spawned_pos.push_back(p);
  }
  void agent_destroyed(AgentId a) override { destroyed_ids.push_back(a); }
};

struct OrcSim {
  std::unique_ptr<Simulation> sim;
  LocationHash2D* index = nullptr;  // owned by sim
  std::vector<Locked<LocalPlanner>> lps;
  std::vector<Locked<HighLevelPlanner>> hls;
  std::vector<std::shared_ptr<TableVelocityPlan>> tables;  // parallel to hls (null if not a table)
  std::shared_ptr<RecordingListener> listener;
  std::string last_error;
};

}  // namespace

extern "C" {

void* orc_sim_create(double width, double height, double cell, double offx, double offy, int index_mode,
                     int iter_order, int canonical_cells) {
  auto* s = new OrcSim();
  auto idx = std::make_unique<LocationHash2D>(width, height, cell, Vec2{offx, offy}, canonical_cells != 0);
  s->index = idx.get();
  s->sim = std::make_unique<Simulation>(std::move(idx), static_cast<IndexMode>(index_mode),
                                        static_cast<IterOrder>(iter_order));
  s->listener = std::make_shared<RecordingListener>();
  s->sim->add_event_listener(s->listener);
  return s;
}

void orc_sim_destroy(void* h) { delete static_cast<OrcSim*>(h); }

const char* orc_last_error(void* h) { return static_cast<OrcSim*>(h)->last_error.c_str(); }

int orc_lp_none(void* h) {
  auto* s = static_cast<OrcSim*>(h);
  s->lps.emplace_back(std::make_shared<NoLocalPlan>());
  return static_cast<int>(s->lps.size() - 1);
}

int orc_lp_zanlungo(void* h, double agent_scale, double obstacle_scale, double reaction_time,
                    double force_distance, double agent_mass, double agent_radius) {
  auto* s = static_cast<OrcSim*>(h);
  s->lps.emplace_back(std::make_shared<Zanlungo>(agent_scale, obstacle_scale, reaction_time, force_distance,
                                                 agent_mass, agent_radius));
  return static_cast<int>(s->lps.size() - 1);
}

static int push_hl(OrcSim* s, std::shared_ptr<HighLevelPlanner> p, std::shared_ptr<TableVelocityPlan> t) {
  s->hls.emplace_back(std::move(p));
  s->tables.push_back(std::move(t));
  return static_cast<int>(s->hls.size() - 1);
}

int orc_hl_constant(void* h, double vx, double vy) {
  return push_hl(static_cast<OrcSim*>(h), std::make_shared<ConstantVelocityPlan>(Vec2{vx, vy}), nullptr);
}
int orc_hl_parity(void* h, double vx, double vy) {
  return push_hl(static_cast<OrcSim*>(h), std::make_shared<ParityVelocityPlan>(Vec2{vx, vy}), nullptr);
}
int orc_hl_host(void* h) {
  auto t = std::make_shared<TableVelocityPlan>();
  return push_hl(static_cast<OrcSim*>(h), t, t);
}
int orc_hl_route(void* h, uint64_t n, const double* xy) {
  std::vector<Vec2> route;
  for (uint64_t i = 0; i < n; ++i) route.push_back({xy[2 * i], xy[2 * i + 1]});
  return push_hl(static_cast<OrcSim*>(h), std::make_shared<RouteFollowPlan>(std::move(route)), nullptr);
}

int orc_add_agents(void* h, uint64_t n, const double* xy, int hl, int lp, double eyesight, uint64_t* out_ids) {
  auto* s = static_cast<OrcSim*>(h);
  std::vector<Vec2> pts;
  for (uint64_t i = 0; i < n; ++i) pts.push_back({xy[2 * i], xy[2 * i + 1]});
  std::vector<AgentId> ids;
  Status st = s->sim->add_agents(pts, s->hls.at(hl), s->lps.at(lp), eyesight, &ids);
  if (out_ids)
    for (size_t i = 0; i < ids.size(); ++i) out_ids[i] = ids[i];
  if (!st.ok) {
    s->last_error = st.msg;
    return 1;
  }
  return 0;
}

int orc_remove_agent(void* h, uint64_t id) {
  auto* s = static_cast<OrcSim*>(h);
  if (!s->sim->agents.count(id)) return 1;
  s->sim->remove_agents(id);
  return 0;
}

// `agents` is a pub field in the reference: position/velocity are user-writable.  The index's
// private copy is refreshed too (snapshot-injection semantic, SURVEY.md section 9).
int orc_set_state(void* h, uint64_t n, const uint64_t* ids, const double* x, const double* y, const double* vx,
                  const double* vy) {
  auto* s = static_cast<OrcSim*>(h);
  for (uint64_t i = 0; i < n; ++i) {
    auto it = s->sim->agents.find(ids[i]);
    if (it == s->sim->agents.end()) {
      s->last_error = "unknown agent id";
      return 1;
    }
    it->second.position = {x[i], y[i]};
    it->second.velocity = {vx[i], vy[i]};
    Status st = s->sim->spatial_index().add_or_update(ids[i], it->second.position);
    if (!st.ok) {
      s->last_error = st.msg;
      return 2;
    }
  }
  return 0;
}

int orc_set_preferred_velocity(void* h, int hl, uint64_t n, const uint64_t* ids, const double* vxy) {
  auto* s = static_cast<OrcSim*>(h);
  auto& t = s->tables.at(hl);
  if (!t) return 1;
  for (uint64_t i = 0; i < n; ++i) t->table[ids[i]] = Vec2{vxy[2 * i], vxy[2 * i + 1]};
  return 0;
}

// HighLevelPlanner::set_target(agent, (0, 0), (0, 0)) for agents addressed by id (the route follower ignores the
// point: rcs_hl_route_set_target).
int orc_hl_set_target(void* h, int hl, uint64_t n, const uint64_t* ids) {
  auto* s = static_cast<OrcSim*>(h);
  auto& p = s->hls.at(hl);
  for (uint64_t i = 0; i < n; ++i) {
    auto it = s->sim->agents.find(ids[i]);
    if (it == s->sim->agents.end()) return 1;
    std::lock_guard<std::mutex> g(*p.mtx);
    p.ptr->set_target(it->second, Vec2{0.0, 0.0}, Vec2{0.0, 0.0});
  }
  return 0;
}

int orc_add_source_sink(void* h, double sx, double sy, double radius_sink, double monotonic_rate, int hl, int lp,
                        uint64_t n_wp, const double* wp_xy, int loop_forever, double eyesight, uint64_t* out_id) {
  auto* s = static_cast<OrcSim*>(h);
  auto ss = std::make_shared<SourceSink>();
  ss->source = {sx, sy};
  ss->radius_sink = radius_sink;
  ss->crowd_generator = std::make_shared<MonotonicCrowd>(monotonic_rate);
  ss->high_level_planner = s->hls.at(hl);
  ss->local_planner = s->lps.at(lp);
  for (uint64_t i = 0; i < n_wp; ++i) ss->waypoints.push_back({wp_xy[2 * i], wp_xy[2 * i + 1]});
  ss->loop_forever = loop_forever != 0;
  ss->agent_eyesight_range = eyesight;
  uint64_t id = s->sim->add_source_sink(ss);
  if (out_id) *out_id = id;
  return 0;
}

void orc_enable_trace(void* h, int on) { static_cast<OrcSim*>(h)->sim->enable_trace(on != 0); }

void orc_set_custom_order(void* h, uint64_t n, const uint64_t* ids) {
  static_cast<OrcSim*>(h)->sim->set_custom_order(std::vector<AgentId>(ids, ids + n));
}

int orc_step(void* h, uint64_t secs, uint32_t nanos) {
  auto* s = static_cast<OrcSim*>(h);
  Status st = s->sim->step(Duration{secs, nanos});
  if (!st.ok) {
    s->last_error = st.msg;
    return st.msg == "Index out of bounds" ? 1 : 2;
  }
  return 0;
}

uint64_t orc_agent_count(void* h) { return static_cast<OrcSim*>(h)->sim->agents.size(); }

// ascending id
void orc_read_agents(void* h, uint64_t* ids, double* x, double* y, double* vx, double* vy, uint64_t* next_wp) {
  auto* s = static_cast<OrcSim*>(h);
  std::vector<AgentId> keys;
  for (auto& kv : s->sim->agents) keys.push_back(kv.first);
  std::sort(keys.begin(), keys.end());
  for (size_t i = 0; i < keys.size(); ++i) {
    const Agent& a = s->sim->agents.at(keys[i]);
    if (ids) ids[i] = keys[i];
    if (x) x[i] = a.position.x;
    if (y) y[i] = a.position.y;
    if (vx) vx[i] = a.velocity.x;
    if (vy) vy[i] = a.velocity.y;
    if (next_wp) next_wp[i] = a.next_waypoint;
  }
}

// trace of the last step: per agent (iteration order) t_i, force, CSR neighbour ids
uint64_t orc_trace_agent_count(void* h) { return static_cast<OrcSim*>(h)->sim->trace().size(); }
uint64_t orc_trace_neighbour_total(void* h) {
  uint64_t t = 0;
  for (auto& a : static_cast<OrcSim*>(h)->sim->trace()) t += a.neighbours.size();
  return t;
}
void orc_read_trace(void* h, uint64_t* ids, double* t_i, double* fx, double* fy, uint64_t* nb_offsets,
                    uint64_t* nb_ids) {
  auto& tr = static_cast<OrcSim*>(h)->sim->trace();
  uint64_t off = 0;
  for (size_t i = 0; i < tr.size(); ++i) {
    ids[i] = tr[i].id;
    t_i[i] = tr[i].t_i;
    fx[i] = tr[i].force.x;
    fy[i] = tr[i].force.y;
    nb_offsets[i] = off;
    for (AgentId n : tr[i].neighbours) nb_ids[off++] = n;
  }
  nb_offsets[tr.size()] = off;
}

uint64_t orc_poll_events(void* h, uint64_t* spawned_ids, double* spawned_xy, uint64_t spawned_cap,
                         uint64_t* n_spawned, uint64_t* destroyed_ids, uint64_t destroyed_cap,
                         uint64_t* n_destroyed) {
  auto* s = static_cast<OrcSim*>(h);
  auto& l = *s->listener;
  *n_spawned = l.spawned_ids.size();
  *n_destroyed = l.destroyed_ids.size();
  for (uint64_t i = 0; i < std::min<uint64_t>(spawned_cap, l.spawned_ids.size()); ++i) {
    spawned_ids[i] = l.spawned_ids[i];
    spawned_xy[2 * i] = l.spawned_pos[i].x;
    spawned_xy[2 * i + 1] = l.spawned_pos[i].y;
  }
  for (uint64_t i = 0; i < std::min<uint64_t>(destroyed_cap, l.destroyed_ids.size()); ++i)
    destroyed_ids[i] = l.destroyed_ids[i];
  l.spawned_ids.clear();
  l.spawned_pos.clear();
  l.destroyed_ids.clear();
  return 0;
}

// --- SpatialIndex trait surface on the simulation's index -------------------------------
int orc_index_add_or_update(void* h, uint64_t id, double x, double y) {
  return static_cast<OrcSim*>(h)->index->add_or_update(id, {x, y}).ok ? 0 : 1;
}
void orc_index_remove(void* h, uint64_t id) { static_cast<OrcSim*>(h)->index->remove_agent(id); }
int64_t orc_cell_of(void* h, double x, double y) {
  auto idx = static_cast<OrcSim*>(h)->index->location_to_index({x, y});
  return idx ? static_cast<int64_t>(*idx) : -1;
}
uint64_t orc_query_radius(void* h, double radius, double x, double y, uint64_t* out, uint64_t cap) {
  auto v = static_cast<OrcSim*>(h)->index->get_neighbours_in_radius(radius, {x, y});
  for (uint64_t i = 0; i < std::min<uint64_t>(cap, v.size()); ++i) out[i] = v[i];
  return v.size();
}
// UINT64_MAX (and orc_last_error) where the reference panics: a NaN distance among >= 2 candidates
uint64_t orc_query_knn(void* h, uint64_t n, double x, double y, uint64_t* out, uint64_t cap) {
  auto* s = static_cast<OrcSim*>(h);
  std::vector<AgentId> v;
  try {
    v = s->index->get_nearest_neighbours(n, {x, y});
  } catch (const LocationHash2D::NanDistance& e) {
    s->last_error = e.what();
    return ~0ull;
  }
  for (uint64_t i = 0; i < std::min<uint64_t>(cap, v.size()); ++i) out[i] = v[i];
  return v.size();
}
void orc_query_bounds(void* h, double radius, double x, double y, int64_t* lrbt) {
  static_cast<OrcSim*>(h)->index->get_bounds(radius, {x, y}, lrbt[0], lrbt[1], lrbt[2], lrbt[3]);
}

// --- pure functions ----------------------------------------------------------------------
double orc_ttc(double agent_radius, double rvx, double rvy, double rpx, double rpy) {
  Zanlungo z(1, 1, 0, 1, 1, agent_radius);
  return z.time_to_collision({rvx, rvy}, {rpx, rpy});
}

// force of `other` on `agent` (zanlungo.rs:93-170); p[] = agent_scale, obstacle_scale, reaction_time,
// force_distance, agent_mass, agent_radius; a[]/o[] = id(as double is NOT used: ids passed separately),
// x, y, vx, vy, pvx, pvy
void orc_agent_force(const double* p, uint64_t aid, const double* a, uint64_t oid, const double* o, double t_i,
                     double* out) {
  Zanlungo z(p[0], p[1], p[2], p[3], p[4], p[5]);
  Agent A, O;
  A.agent_id = aid;
  A.position = {a[0], a[1]};
  A.velocity = {a[2], a[3]};
  A.preferred_vel = {a[4], a[5]};
  O.agent_id = oid;
  O.position = {o[0], o[1]};
  O.velocity = {o[2], o[3]};
  O.preferred_vel = {o[4], o[5]};
  Vec2 f = z.compute_agent_force(A, O, t_i);
  out[0] = f.x;
  out[1] = f.y;
}

double orc_duration_as_secs_f64(uint64_t secs, uint32_t nanos) { return Duration{secs, nanos}.as_secs_f64(); }

}  // extern "C"
