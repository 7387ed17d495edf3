// crowdsim_oracle.hpp -- CPU ORACLE, TEST INFRASTRUCTURE ONLY.
//
// A C++17 restatement of the per-timestep agent update of open-rmf/rmf_crowdsim
// (Rust).  It exists to CHECK the CUDA path; nothing under rmf_crowdsim_b200/
// may include, link or call it.  Only tests/, __graft_entry__.smoke() and
// bench.py's cpu_baseline / --impl reference legs use it.
//
// PARITY PINNING: the Rust reference cannot be compiled in this environment (no
// rustc/cargo, crates not vendored), so this restatement is pinned against the
// reference's own eight tests (restated in oracle/selftest.cpp and
// tests/test_oracle_*.py) and nothing else.  `Zanlungo::compute_agent_force`,
// `right_of_way_vel`, `slerp` and multi-agent Zanlungo stepping are NOT covered
// by any reference test: for those rows parity is UNPINNED beyond this literal
// restatement of the source.
//
// Third-party arithmetic: nalgebra 0.31.4 (Cargo.lock:1495-1497) is not under
// /root/reference.  For Vector2<f64> the assumed semantics are: dot = x*x' + y*y'
// (two products, one add), norm_squared = dot(a,a), norm = sqrt(norm_squared),
// normalize = component-wise DIVISION by norm, all other ops component-wise, no
// FMA contraction (rustc never contracts).  Build with -ffp-contract=off.
//
// Every function cites the reference file:line it follows (paths relative to
// /root/reference/rmf_crowdsim/src).
#pragma once

#include <algorithm>
#include <cmath>
#include <cstdint>
#include <limits>
#include <memory>
#include <mutex>
#include <optional>
#include <stdexcept>
#include <string>
#include <unordered_map>
#include <unordered_set>
#include <utility>
#include <vector>

namespace orc {

using AgentId = uint64_t;  // lib.rs:36 (usize on 64-bit targets)

// ---------------------------------------------------------------------------
// nalgebra Vector2<f64> subset (see header comment for the assumed semantics)
// ---------------------------------------------------------------------------
struct Vec2 {
  double x = 0.0, y = 0.0;
};
inline Vec2 operator+(Vec2 a, Vec2 b) { return {a.x + b.x, a.y + b.y}; }
inline Vec2 operator-(Vec2 a, Vec2 b) { return {a.x - b.x, a.y - b.y}; }
inline Vec2 operator-(Vec2 a) { return {-a.x, -a.y}; }
inline Vec2 operator*(Vec2 a, double s) { return {a.x * s, a.y * s}; }
inline Vec2 operator*(double s, Vec2 a) { return {s * a.x, s * a.y}; }
inline double dot(Vec2 a, Vec2 b) {
  double p = a.x * b.x;
  double q = a.y * b.y;
  return p + q;
}
inline double norm_squared(Vec2 a) { return dot(a, a); }
inline double norm(Vec2 a) { return std::sqrt(norm_squared(a)); }
inline Vec2 normalize(Vec2 a) {
  double n = norm(a);
  return {a.x / n, a.y / n};
}

// Rust `f64 as usize`: truncate toward zero, saturate, NaN -> 0.
inline uint64_t f64_as_usize(double v) {
  if (!(v > 0.0)) return 0;  // NaN, negatives, +-0
  if (v >= 18446744073709551616.0) return std::numeric_limits<uint64_t>::max();
  return static_cast<uint64_t>(v);
}
// Rust `f64 as i64`: truncate toward zero, saturate, NaN -> 0.
inline int64_t f64_as_i64(double v) {
  if (v != v) return 0;
  if (v >= 9223372036854775808.0) return std::numeric_limits<int64_t>::max();
  if (v <= -9223372036854775808.0) return std::numeric_limits<int64_t>::min();
  return static_cast<int64_t>(v);
}

// std::time::Duration::as_secs_f64: secs as f64 + nanos as f64 / 1e9.
struct Duration {
  uint64_t secs = 0;
  uint32_t nanos = 0;
  double as_secs_f64() const {
    return static_cast<double>(secs) + static_cast<double>(nanos) / 1000000000.0;
  }
};

struct Status {
  bool ok = true;
  std::string msg;
  static Status Ok() { return {}; }
  static Status Err(std::string m) { return {false, std::move(m)}; }
};

// lib.rs:46-65
struct Agent {
  AgentId agent_id = 0;
  Vec2 position;
  double orientation = 0.0;
  Vec2 velocity;
  Vec2 preferred_vel;  // private in the reference; only ever set on a local clone (lib.rs:271)
  double angular_vel = 0.0;
  uint64_t next_waypoint = 0;
  double eyesight_range = 0.0;
};

// ---------------------------------------------------------------------------
// spatial_index/spatial_index.rs:4-14
// ---------------------------------------------------------------------------
class SpatialIndex {
 public:
  virtual ~SpatialIndex() = default;
  virtual Status add_or_update(AgentId id, Vec2 position) = 0;
  virtual std::vector<AgentId> get_nearest_neighbours(uint64_t n, Vec2 position) const = 0;
  virtual std::vector<AgentId> get_neighbours_in_radius(double radius, Vec2 position) const = 0;
  virtual void remove_agent(AgentId) {}
  // Oracle-only hook for the deferred index mode: would add_or_update accept p?
  virtual Status check_insertable(Vec2) const { return Status::Ok(); }
};

// ---------------------------------------------------------------------------
// spatial_index/location_hash_2d.rs
// `canonical` makes iteration inside one cell ascending-id (the reference's
// HashSet order is random per process); with canonical=false the cell's
// unordered_set order is used, which is what the CPU-baseline timing runs.
// ---------------------------------------------------------------------------
class LocationHash2D : public SpatialIndex {
 public:
  // location_hash_2d.rs:33-51
  LocationHash2D(double width, double height, double cell_size, Vec2 offset, bool canonical = true)
      : width_(width), height_(height), resolution_(cell_size), offset_(offset), canonical_(canonical) {
    uint64_t nx = f64_as_usize(width / cell_size);
    uint64_t ny = f64_as_usize(height / cell_size);
    data_.resize(nx * ny);
  }

  uint64_t num_cells() const { return data_.size(); }

  // location_hash_2d.rs:54-66 (insert cell; truncating cast, width stride)
  std::optional<uint64_t> location_to_index(Vec2 point) const {
    uint64_t x_idx = f64_as_usize((point - offset_).x / resolution_);
    uint64_t y_idx = f64_as_usize((point - offset_).y / resolution_);
    uint64_t idx = x_idx * f64_as_usize(width_ / resolution_) + y_idx;  // wrapping, as release Rust
    if (idx >= data_.size()) return std::nullopt;
    return idx;
  }

  // location_hash_2d.rs:68-72 (query cell; floor)
  std::pair<int64_t, int64_t> location_to_xy_signed_idx(Vec2 point) const {
    int64_t x_idx = f64_as_i64(std::floor((point - offset_).x / resolution_));
    int64_t y_idx = f64_as_i64(std::floor((point - offset_).y / resolution_));
    return {x_idx, y_idx};
  }

  // location_hash_2d.rs:74-85
  std::optional<uint64_t> signed_idx_to_data_idx(int64_t x_idx, int64_t y_idx) const {
    if (x_idx < 0 || y_idx < 0) return std::nullopt;
    uint64_t idx = static_cast<uint64_t>(x_idx) * f64_as_usize(width_ / resolution_) +
                   static_cast<uint64_t>(y_idx);
    if (idx >= data_.size()) return std::nullopt;
    return idx;
  }

  // location_hash_2d.rs:87-101 (one vector allocation per visited cell, as the reference)
  std::optional<std::vector<std::pair<Vec2, AgentId>>> get_neighbours_in_cell(int64_t x_idx,
                                                                               int64_t y_idx) const {
    std::vector<std::pair<Vec2, AgentId>> agents_in_ring;
    auto idx = signed_idx_to_data_idx(x_idx, y_idx);
    if (!idx) return std::nullopt;
    for (AgentId agent_id : data_[*idx]) {
      agents_in_ring.push_back({id_to_exact_location_.at(agent_id), agent_id});
    }
    if (canonical_) {
      std::sort(agents_in_ring.begin(), agents_in_ring.end(),
                [](const auto& a, const auto& b) { return a.second < b.second; });
    }
    return agents_in_ring;
  }

  // location_hash_2d.rs:103-122 -> (left, right, bottom, top)
  void get_bounds(double radius, Vec2 position, int64_t& left, int64_t& right, int64_t& bottom,
                  int64_t& top) const {
    right = location_to_xy_signed_idx({position.x + radius, position.y}).first;
    left = location_to_xy_signed_idx({position.x - radius, position.y}).first;
    top = location_to_xy_signed_idx({position.x, position.y + radius}).second;
    bottom = location_to_xy_signed_idx({position.x, position.y - radius}).second;
  }

  Status check_insertable(Vec2 p) const override {
    if (!location_to_index(p)) return Status::Err("Index out of bounds");
    return Status::Ok();
  }

  // location_hash_2d.rs:126-149
  Status add_or_update(AgentId id, Vec2 position) override {
    auto new_index = location_to_index(position);
    if (!new_index) return Status::Err("Index out of bounds");
    auto old = id_to_index_.find(id);
    if (old != id_to_index_.end()) {
      if (*new_index != old->second) {
        data_[old->second].erase(id);
        data_[*new_index].insert(id);
        id_to_index_[id] = *new_index;
      }
    } else {
      data_[*new_index].insert(id);
      id_to_index_[id] = *new_index;
    }
    id_to_exact_location_[id] = position;
    return Status::Ok();
  }

  // location_hash_2d.rs:151-238.  Ring search with half-open side ranges (the
  // (x-s,y-s) corner is visited twice, the (x+s,y+s) corner never), stops at the
  // first ring that reaches n candidates, stable sort by distance.  The side bounds
  // wrap as in release-mode Rust (a saturated query cell empties the sides whose
  // upper bound wrapped) and the visits made are counted, so a ring whose visits
  // were all out of bounds -- or that made none -- ends the walk.  The reference
  // sorts with partial_cmp(..).unwrap(), which panics on a NaN distance as soon as
  // two candidates are compared: that is NanDistance here.
  struct NanDistance : std::domain_error {
    NanDistance() : std::domain_error("get_nearest_neighbours: NaN distance") {}
  };
  std::vector<AgentId> get_nearest_neighbours(uint64_t n, Vec2 position) const override {
    auto [x_idx, y_idx] = location_to_xy_signed_idx(position);
    auto wadd = [](int64_t a, int64_t b) { return static_cast<int64_t>(static_cast<uint64_t>(a) + static_cast<uint64_t>(b)); };
    auto wsub = [](int64_t a, int64_t b) { return static_cast<int64_t>(static_cast<uint64_t>(a) - static_cast<uint64_t>(b)); };
    std::vector<AgentId> agents;
    bool all_out_of_bounds = false;
    int64_t step = 0;
    std::vector<std::pair<Vec2, AgentId>> agents_in_ring;
    auto visit = [&](int64_t cx, int64_t cy, uint64_t& num_oob, uint64_t& num_scanned) {
      auto nb = get_neighbours_in_cell(cx, cy);
      if (nb) {
        agents_in_ring.insert(agents_in_ring.end(), nb->begin(), nb->end());
      } else {
        num_oob += 1;
      }
      num_scanned += 1;
    };
    while (agents_in_ring.size() < n && !all_out_of_bounds) {
      uint64_t num_out_of_bounds = 0, num_scanned_cells = 0;
      if (step == 0) {
        visit(x_idx, y_idx, num_out_of_bounds, num_scanned_cells);
      } else {
        const int64_t xl = wsub(x_idx, step), xh = wadd(x_idx, step);
        const int64_t yl = wsub(y_idx, step), yh = wadd(y_idx, step);
        for (int64_t i = xl; i < xh; ++i) visit(i, yh, num_out_of_bounds, num_scanned_cells);  // top line
        for (int64_t i = xl; i < xh; ++i) visit(i, yl, num_out_of_bounds, num_scanned_cells);  // bottom line
        for (int64_t i = yl; i < yh; ++i) visit(xl, i, num_out_of_bounds, num_scanned_cells);  // left line
        for (int64_t i = yl; i < yh; ++i) visit(xh, i, num_out_of_bounds, num_scanned_cells);  // right line
      }
      if (num_out_of_bounds == num_scanned_cells) all_out_of_bounds = true;
      step += 1;
    }
    std::vector<double> dist(agents_in_ring.size());
    std::vector<size_t> perm(agents_in_ring.size());
    for (size_t i = 0; i < agents_in_ring.size(); ++i) {
      dist[i] = norm(agents_in_ring[i].first - position);
      perm[i] = i;
      if (std::isnan(dist[i]) && agents_in_ring.size() >= 2) throw NanDistance();
    }
    std::stable_sort(perm.begin(), perm.end(), [&](size_t a, size_t b) { return dist[a] < dist[b]; });
    for (uint64_t i = 0; i < std::min<uint64_t>(n, perm.size()); ++i)
      agents.push_back(agents_in_ring[perm[i]].second);
    return agents;
  }

  // location_hash_2d.rs:240-258 (strict <, x-major then y scan order)
  std::vector<AgentId> get_neighbours_in_radius(double radius, Vec2 position) const override {
    std::vector<AgentId> agents;
    int64_t left, right, bottom, top;
    get_bounds(radius, position, left, right, bottom, top);
    for (int64_t x_idx = left; x_idx <= right; ++x_idx) {
      for (int64_t y_idx = bottom; y_idx <= top; ++y_idx) {
        auto result = get_neighbours_in_cell(x_idx, y_idx);
        if (result) {
          for (const auto& [agent_pos, agent_id] : *result) {
            if (norm(agent_pos - position) < radius) agents.push_back(agent_id);
          }
        }
      }
    }
    return agents;
  }

  // location_hash_2d.rs:260-267
  void remove_agent(AgentId id) override {
    auto it = id_to_index_.find(id);
    if (it != id_to_index_.end()) {
      data_[it->second].erase(id);
      id_to_exact_location_.erase(id);
      id_to_index_.erase(id);
    }
  }

 private:
  std::vector<std::unordered_set<AgentId>> data_;
  std::unordered_map<AgentId, uint64_t> id_to_index_;
  std::unordered_map<AgentId, Vec2> id_to_exact_location_;
  double width_, height_, resolution_;
  Vec2 offset_;
  bool canonical_;
};

// ---------------------------------------------------------------------------
// local_planners/local_planner.rs:7-18
// ---------------------------------------------------------------------------
class LocalPlanner {
 public:
  virtual ~LocalPlanner() = default;
  virtual Vec2 get_desired_velocity(const Agent& agent, const std::vector<Agent>& nearby_agents,
                                    Vec2 recommended_velocity) const = 0;
  virtual void add_agent(AgentId) {}
  virtual void remove_agent(AgentId) {}
  // oracle-only trace hooks (no effect on arithmetic)
  mutable double last_t_i = std::numeric_limits<double>::infinity();
  mutable Vec2 last_force;
};

// local_planners/no_local_plan.rs:7-18
class NoLocalPlan : public LocalPlanner {
 public:
  Vec2 get_desired_velocity(const Agent&, const std::vector<Agent>&, Vec2 recommended) const override {
    last_t_i = std::numeric_limits<double>::infinity();
    last_force = {0.0, 0.0};
    return recommended;
  }
};

// local_planners/zanlungo.rs
class Zanlungo : public LocalPlanner {
 public:
  // zanlungo.rs:31-48 (obstacle_scale and reaction_time are stored, never read)
  Zanlungo(double agent_scale, double obstacle_scale, double reaction_time, double force_distance,
           double agent_mass, double agent_radius)
      : agent_scale_(agent_scale),
        obstacle_scale_(obstacle_scale),
        reaction_time_(reaction_time),
        force_distance_(force_distance),
        agent_mass_(agent_mass),
        agent_radius_(agent_radius) {}

  // zanlungo.rs:23-28
  static Vec2 slerp(double t, Vec2 p0, Vec2 p1, double sin_theta) {
    double theta = std::asin(sin_theta);
    double t0 = std::sin((1.0 - t) * theta) / sin_theta;
    double t1 = std::sin(t * theta) / sin_theta;
    return p0 * t0 + p1 * t1;
  }

  // zanlungo.rs:49-74
  double time_to_collision(Vec2 rel_vel, Vec2 rel_pos) const {
    double a = norm_squared(rel_vel);
    double b = 2.0 * dot(rel_vel, rel_pos);
    double c = norm_squared(rel_pos) - agent_radius_ * agent_radius_;
    double discriminant = b * b - 4.0 * a * c;
    if (discriminant < 0.0) return std::numeric_limits<double>::infinity();
    double t0 = (-b - std::sqrt(discriminant)) / (2.0 * a);
    double t1 = (-b + std::sqrt(discriminant)) / (2.0 * a);
    if ((t0 < 0.0 && t1 > 0.0) || (t1 < 0.0 && t0 > 0.0)) return 0.0;
    if (t0 < t1 && t0 > 0.0) {
      return t0;
    } else if (t1 > 0.0) {
      return t1;
    } else {
      return std::numeric_limits<double>::infinity();
    }
  }

  // zanlungo.rs:76-91
  double compute_tti(const Agent& current_agent, const std::vector<Agent>& nearby_agents) const {
    double t_i = std::numeric_limits<double>::infinity();
    for (const Agent& n : nearby_agents) {
      Vec2 rel_vel = n.velocity - current_agent.velocity;
      Vec2 rel_pos = n.position - current_agent.position;
      double col_time = time_to_collision(rel_vel, rel_pos);
      if (col_time < t_i) t_i = col_time;
    }
    return t_i;
  }

  struct RightOfWay {
    double weight;
    Vec2 my_vel, other_vel;
  };

  // zanlungo.rs:173-198 (agent_priorities is never populated => priority = id as f64)
  RightOfWay right_of_way_vel(AgentId agent_id, Vec2 agent_vel, Vec2 self_pref_vel, Vec2 other_vel,
                              Vec2 other_pref_vel, double other_priority) const {
    double self_priority = priority_of(agent_id);
    double right_of_way = self_priority - other_priority;
    // f64::clamp(-1, 1): NaN stays NaN
    if (right_of_way < -1.0) right_of_way = -1.0;
    if (right_of_way > 1.0) right_of_way = 1.0;
    if (right_of_way < 0.0) {
      double r_2 = std::sqrt(-right_of_way);
      Vec2 other_adjusted_vel = other_vel + r_2 * (other_pref_vel - other_vel);
      return {-r_2, agent_vel, other_adjusted_vel};
    } else if (right_of_way > 0.0) {
      double r_2 = std::sqrt(right_of_way);
      Vec2 vel = agent_vel + r_2 * (self_pref_vel - agent_vel);
      return {r_2, vel, other_vel};
    } else {
      return {0.0, agent_vel, other_vel};
    }
  }

  // zanlungo.rs:93-170
  Vec2 compute_agent_force(const Agent& agent, const Agent& other_agent, double t_i) const {
    double other_priority = priority_of(other_agent.agent_id);
    RightOfWay row = right_of_way_vel(agent.agent_id, agent.velocity, agent.preferred_vel,
                                      other_agent.velocity, other_agent.preferred_vel, other_priority);
    Vec2 my_vel = row.my_vel, other_vel = row.other_vel;
    double weight = 1.0 - row.weight;
    Vec2 fut_pos = agent.position + my_vel * t_i;
    Vec2 other_future_pos = other_agent.position + other_vel * t_i;
    Vec2 d_ij = fut_pos - other_future_pos;
    double dist = norm(d_ij);
    if (weight > 1.0) {
      double pref_speed = norm(other_agent.preferred_vel);
      bool interpolate = true;
      Vec2 perp_dir{0.0, 0.0};
      if (pref_speed < 0.0001) {
        Vec2 curr_rel_pos = agent.position - other_agent.position;
        perp_dir = Vec2{-curr_rel_pos.y, curr_rel_pos.x};
        if (dot(perp_dir, agent.velocity) < 0.0) perp_dir = -perp_dir;
      } else {
        Vec2 pref_dir = other_agent.preferred_vel;
        if (dot(pref_dir, d_ij) > 0.0) {
          perp_dir = Vec2{-pref_dir.y, pref_dir.x};
          if (dot(perp_dir, d_ij) < 0.0) perp_dir = -perp_dir;
        } else {
          interpolate = false;
        }
      }
      if (interpolate) {
        double sin_theta = perp_dir.x * d_ij.y - perp_dir.y * d_ij.x;
        if (sin_theta < 0.0) sin_theta = -sin_theta;
        if (sin_theta > 1.0) sin_theta = 1.0;
        d_ij = slerp(weight - 1.0, d_ij, perp_dir, sin_theta);
      }
    }
    if (dist > norm(fut_pos - other_future_pos)) return Vec2{0.0, 0.0};
    Vec2 d_ij_normalized = normalize(d_ij);
    double surface_dist = dist - agent_radius_ * 2.0;
    double magnitude = weight * agent_scale_ * norm(my_vel - other_vel) / t_i;
    if (magnitude >= 1e15) magnitude = 1e15;
    return d_ij_normalized * (magnitude * std::exp(-surface_dist / force_distance_));
  }

  // zanlungo.rs:201-218
  Vec2 get_desired_velocity(const Agent& agent, const std::vector<Agent>& nearby_agents,
                            Vec2 recommended_velocity) const override {
    double t_i = compute_tti(agent, nearby_agents);
    Vec2 force{0.0, 0.0};
    if (t_i != std::numeric_limits<double>::infinity()) {
      for (const Agent& nearby_agent : nearby_agents) {
        Vec2 f = compute_agent_force(agent, nearby_agent, t_i);
        force = force + f;
      }
    }
    last_t_i = t_i;
    last_force = force;
    return recommended_velocity + (force * (1.0 / agent_mass_));
  }

 private:
  double priority_of(AgentId id) const {
    auto it = agent_priorities_.find(id);  // always misses (zanlungo.rs:17,46,182)
    if (it != agent_priorities_.end()) return it->second;
    return static_cast<double>(id);
  }
  double agent_scale_, obstacle_scale_, reaction_time_, force_distance_, agent_mass_, agent_radius_;
  std::unordered_map<AgentId, double> agent_priorities_;
};

// ---------------------------------------------------------------------------
// highlevel_planners/highlevel_planners.rs:8-16
// ---------------------------------------------------------------------------
class HighLevelPlanner {
 public:
  virtual ~HighLevelPlanner() = default;
  virtual std::optional<Vec2> get_desired_velocity(const Agent& agent, Duration time) = 0;
  virtual void set_target(const Agent& agent, Vec2 point, Vec2 tolerance) = 0;
  virtual void remove_agent_id(AgentId) {}
};

// The fixture planner of lib.rs:391-420 and tests/event_listeners_test.rs:6-35.
class ConstantVelocityPlan : public HighLevelPlanner {
 public:
  explicit ConstantVelocityPlan(Vec2 v) : default_vel_(v) {}
  std::optional<Vec2> get_desired_velocity(const Agent&, Duration) override { return default_vel_; }
  void set_target(const Agent&, Vec2, Vec2) override {}

 private:
  Vec2 default_vel_;
};

// The fixture planner of rmf_crowdsim_viz/src/main.rs:20-30 (even id -> -v, odd -> +v).
class ParityVelocityPlan : public HighLevelPlanner {
 public:
  explicit ParityVelocityPlan(Vec2 v) : default_vel_(v) {}
  std::optional<Vec2> get_desired_velocity(const Agent& agent, Duration) override {
    if (agent.agent_id % 2 == 0) return -default_vel_;
    return default_vel_;
  }
  void set_target(const Agent&, Vec2, Vec2) override {}

 private:
  Vec2 default_vel_;
};

// Host-table planner: what a user-implemented trait object looks like from the
// step's point of view -- a per-agent preferred velocity, None when unset.
class TableVelocityPlan : public HighLevelPlanner {
 public:
  std::optional<Vec2> get_desired_velocity(const Agent& agent, Duration) override {
    auto it = table.find(agent.agent_id);
    if (it == table.end()) return std::nullopt;
    return it->second;
  }
  void set_target(const Agent&, Vec2, Vec2) override {}
  void remove_agent_id(AgentId id) override { table.erase(id); }
  std::unordered_map<AgentId, Vec2> table;
};

// The per-step half of rmf/mod.rs:197-215 (RMFPlanner::get_desired_velocity) with the
// routes supplied by the caller instead of planned by `mapf` (absent third-party crate).
// set_target (rmf/mod.rs:217-237) is reduced to "pick the route registered for this
// (source sink) group and start at waypoint 0"; remove_agent_id as rmf/mod.rs:239-241.
class RouteFollowPlan : public HighLevelPlanner {
 public:
  explicit RouteFollowPlan(std::vector<Vec2> route) : route_(std::move(route)) {}
  std::optional<Vec2> get_desired_velocity(const Agent& agent, Duration) override {
    auto it = agent_cache_.find(agent.agent_id);
    if (it == agent_cache_.end()) return std::nullopt;
    uint64_t waypoint_id = it->second;
    if (norm(agent.position - route_[waypoint_id]) < 1e-1 && route_.size() > waypoint_id + 1) {
      waypoint_id += 1;
      it->second = waypoint_id;
    }
    return normalize(route_[waypoint_id] - agent.position);
  }
  void set_target(const Agent& agent, Vec2, Vec2) override { agent_cache_[agent.agent_id] = 0; }
  void remove_agent_id(AgentId id) override { agent_cache_.erase(id); }
  uint64_t waypoint_of(AgentId id) const {
    auto it = agent_cache_.find(id);
    return it == agent_cache_.end() ? ~0ull : it->second;
  }

 private:
  std::vector<Vec2> route_;
  std::unordered_map<AgentId, uint64_t> agent_cache_;
};

// ---------------------------------------------------------------------------
// source_sink/source_sink.rs
// ---------------------------------------------------------------------------
class CrowdGenerator {
 public:
  virtual ~CrowdGenerator() = default;
  virtual uint64_t get_number_to_spawn(Duration time_elapsed) const = 0;
};

// source_sink.rs:85-100 (round half away from zero, no fractional carry)
class MonotonicCrowd : public CrowdGenerator {
 public:
  explicit MonotonicCrowd(double rate) : rate(rate) {}
  uint64_t get_number_to_spawn(Duration time_elapsed) const override {
    double num_spawned = time_elapsed.as_secs_f64() * rate;
    return f64_as_usize(std::round(num_spawned));
  }
  double rate;
};
// PoissonCrowd (source_sink.rs:63-82) draws from rand::thread_rng(): not reproducible,
// parity impossible by construction; not restated.

template <class T>
struct Locked {  // Arc<Mutex<dyn T>>: the lock/unlock is kept so the baseline pays for it
  std::shared_ptr<T> ptr;
  std::shared_ptr<std::mutex> mtx = std::make_shared<std::mutex>();
  Locked() = default;
  explicit Locked(std::shared_ptr<T> p) : ptr(std::move(p)) {}
};

// source_sink.rs:36-60
struct SourceSink {
  Vec2 source;
  double radius_sink = 0.0;
  std::shared_ptr<CrowdGenerator> crowd_generator;
  Locked<HighLevelPlanner> high_level_planner;
  Locked<LocalPlanner> local_planner;
  std::vector<Vec2> waypoints;
  bool loop_forever = false;
  double agent_eyesight_range = 0.0;
};

// lib.rs:22-33
class EventListener {
 public:
  virtual ~EventListener() = default;
  virtual void agent_spawned(Vec2 position, AgentId agent) = 0;
  virtual void agent_destroyed(AgentId agent) = 0;
  virtual void waypoint_reached(Vec2, AgentId) {}  // never invoked by the reference
};

// util/registry.rs:3-21
template <class T>
struct Registry {
  std::unordered_map<uint64_t, T> registry;
  uint64_t counter = 0;
  uint64_t add_new_item(T item) {
    uint64_t id = counter;
    registry[id] = std::move(item);
    counter += 1;
    return id;
  }
  std::vector<uint64_t> sorted_keys() const {  // reference order is HashMap-random; canonical = ascending
    std::vector<uint64_t> k;
    for (const auto& kv : registry) k.push_back(kv.first);
    std::sort(k.begin(), k.end());
    return k;
  }
};

// How the spatial index is updated inside step (SURVEY.md section 0.1):
//  InLoop   -- exactly lib.rs:299: add_or_update(new_pos) inside the per-agent loop, so
//              later agents see earlier agents' NEW positions in the radius filter.
//  Deferred -- the contract semantic: all queries see start-of-step positions; the index
//              is refreshed after the loop.  (= the state of the reference's index at the
//              start of every step.)
enum class IndexMode { Deferred = 0, InLoop = 1 };
// Iteration order of `for agent_id in self.agents.keys()` (lib.rs:259): the reference's
// is SipHash-random.  AscendingId is canonical; MapOrder uses this process's
// unordered_map order (baseline timing); Custom takes an explicit permutation.
enum class IterOrder { AscendingId = 0, MapOrder = 1, Custom = 2 };

struct AgentTrace {  // what parity tests compare per agent per step
  AgentId id;
  std::vector<AgentId> neighbours;  // after the self filter, in list order
  double t_i;
  Vec2 force;
  Vec2 preferred;
  bool has_preferred;
};

// ---------------------------------------------------------------------------
// lib.rs:69-384
// ---------------------------------------------------------------------------
class Simulation {
 public:
  std::unordered_map<AgentId, Agent> agents;  // pub field, lib.rs:71

  explicit Simulation(std::unique_ptr<SpatialIndex> index, IndexMode mode = IndexMode::Deferred,
                      IterOrder order = IterOrder::AscendingId)
      : spatial_index_(std::move(index)), index_mode_(mode), iter_order_(order) {}

  SpatialIndex& spatial_index() { return *spatial_index_; }
  void set_custom_order(std::vector<AgentId> order) { custom_order_ = std::move(order); }
  void enable_trace(bool on) { trace_on_ = on; }
  const std::vector<AgentTrace>& trace() const { return trace_; }
  uint64_t last_alloc_agent_id() const { return last_alloc_agent_id_; }

  // lib.rs:119-156
  Status add_agents(const std::vector<Vec2>& spawn_positions, Locked<HighLevelPlanner> hl,
                    Locked<LocalPlanner> lp, double agent_eyesight_range,
                    std::vector<AgentId>* out_ids) {
    for (const Vec2& x : spawn_positions) {
      AgentId agent_id = last_alloc_agent_id_;
      last_alloc_agent_id_ += 1;
      high_level_planner_[agent_id] = hl;
      local_planner_[agent_id] = lp;
      Agent a;
      a.agent_id = agent_id;
      a.position = x;
      a.eyesight_range = agent_eyesight_range;
      agents[agent_id] = a;
      Status s = spatial_index_->add_or_update(agent_id, x);
      if (!s.ok) return s;
      if (out_ids) out_ids->push_back(agent_id);
      for (uint64_t k : event_listeners_.sorted_keys())
        event_listeners_.registry[k]->agent_spawned(x, agent_id);
    }
    return Status::Ok();
  }

  // lib.rs:159-173
  uint64_t add_source_sink(std::shared_ptr<SourceSink> ss) { return source_sinks_.add_new_item(std::move(ss)); }
  void remove_source_sink(uint64_t id) { source_sinks_.registry.erase(id); }
  uint64_t add_event_listener(std::shared_ptr<EventListener> l) {
    return event_listeners_.add_new_item(std::move(l));
  }

  // lib.rs:176-192
  void remove_agents(AgentId agent) {
    {
      auto& hl = high_level_planner_.at(agent);
      std::lock_guard<std::mutex> g(*hl.mtx);
      hl.ptr->remove_agent_id(agent);
    }
    {
      auto& lp = local_planner_.at(agent);
      std::lock_guard<std::mutex> g(*lp.mtx);
      lp.ptr->remove_agent(agent);
    }
    agents.erase(agent);
    update_buffer_.erase(agent);
    source_sink_agent_correspondence_.erase(agent);
    spatial_index_->remove_agent(agent);
    for (uint64_t k : event_listeners_.sorted_keys()) event_listeners_.registry[k]->agent_destroyed(agent);
  }

  // lib.rs:195-383
  Status step(Duration dur) {
    if (iter_order_ == IterOrder::Custom) {  // the reference visits every agent once: a repeated id is refused
      std::unordered_set<AgentId> seen;
      for (AgentId id : custom_order_)
        if (!seen.insert(id).second) return Status::Err("an id occurs twice in the order");
    }
    // --- A. spawn phase, lib.rs:199-254.  All probes run before any insertion.
    struct ToAdd {
      uint64_t id;
      std::shared_ptr<SourceSink> ss;
      std::vector<Vec2> pts;
    };
    std::vector<ToAdd> to_add;
    for (uint64_t sid : source_sinks_.sorted_keys()) {
      auto ss = source_sinks_.registry[sid];
      uint64_t spawn_number = ss->crowd_generator->get_number_to_spawn(dur);
      std::vector<Vec2> pts;
      if (spawn_number > 0) {
        auto neighbours = spatial_index_->get_neighbours_in_radius(0.4, ss->source);  // hard-coded 0.4, lib.rs:214
        if (neighbours.empty()) pts.push_back(ss->source);
      }
      to_add.push_back({sid, ss, std::move(pts)});
    }
    std::vector<std::pair<uint64_t, std::pair<Status, std::vector<AgentId>>>> added;
    for (auto& t : to_add) {
      std::vector<AgentId> ids;
      Status s = add_agents(t.pts, t.ss->high_level_planner, t.ss->local_planner,
                            t.ss->agent_eyesight_range, &ids);
      added.push_back({t.id, {s, ids}});
    }
    for (auto& [source_id, res] : added) {
      if (res.first.ok) {
        for (AgentId agent : res.second) {
          source_sink_agent_correspondence_[agent] = source_id;
          auto& ss = source_sinks_.registry[source_id];
          auto& hl = high_level_planner_.at(agent);
          std::lock_guard<std::mutex> g(*hl.mtx);
          hl.ptr->set_target(agents.at(agent), ss->waypoints.at(0), Vec2{ss->radius_sink, ss->radius_sink});
        }
      } else {
        return Status::Err("Failed to add agents from source");
      }
    }

    std::vector<AgentId> to_be_removed;
    std::vector<AgentId> order = iteration_order();
    if (trace_on_) trace_.clear();
    std::vector<std::pair<AgentId, Vec2>> deferred_updates;

    // --- B. per-agent loop, lib.rs:259-347
    for (AgentId agent_id : order) {
      Agent agent = agents.at(agent_id);  // clone
      Vec2 vel{0.0, 0.0};
      bool has_pref = false;
      auto hl_it = high_level_planner_.find(agent_id);
      if (hl_it != high_level_planner_.end()) {
        std::optional<Vec2> result;
        {
          std::lock_guard<std::mutex> g(*hl_it->second.mtx);
          result = hl_it->second.ptr->get_desired_velocity(agent, sim_time_);
        }
        if (result) {
          vel = *result;
          agent.preferred_vel = vel;
          has_pref = true;
        }
      }
      Vec2 pref = vel;
      auto lp_it = local_planner_.find(agent_id);
      if (lp_it != local_planner_.end()) {
        std::vector<AgentId> neighbour_ids =
            spatial_index_->get_neighbours_in_radius(agent.eyesight_range, agent.position);
        std::vector<Agent> neighbours;
        for (AgentId nid : neighbour_ids) {
          if (nid != agent_id) neighbours.push_back(agents.at(nid));  // OLD state, pref = 0
        }
        {
          std::lock_guard<std::mutex> g(*lp_it->second.mtx);
          vel = lp_it->second.ptr->get_desired_velocity(agent, neighbours, vel);
          if (trace_on_) {
            AgentTrace tr;
            tr.id = agent_id;
            for (const Agent& n : neighbours) tr.neighbours.push_back(n.agent_id);
            tr.t_i = lp_it->second.ptr->last_t_i;
            tr.force = lp_it->second.ptr->last_force;
            tr.preferred = pref;
            tr.has_preferred = has_pref;
            trace_.push_back(std::move(tr));
          }
        }
      }

      // lib.rs:295-297
      Vec2 dx = vel * dur.as_secs_f64();
      Vec2 pos = agent.position;
      Vec2 new_pos = pos + dx;

      // lib.rs:299-302
      if (index_mode_ == IndexMode::InLoop) {
        Status s = spatial_index_->add_or_update(agent_id, new_pos);
        if (!s.ok) return s;
      } else {
        Status s = spatial_index_->check_insertable(new_pos);
        if (!s.ok) return s;
        deferred_updates.push_back({agent_id, new_pos});
      }

      // lib.rs:305-336 (test on the OLD position)
      uint64_t next_waypoint = agent.next_waypoint;
      auto ss_it = source_sink_agent_correspondence_.find(agent_id);
      if (ss_it != source_sink_agent_correspondence_.end()) {
        // .at(): a removed source sink panics in the reference (lib.rs:309)
        const auto& source_sink = source_sinks_.registry.at(ss_it->second);
        if (agent.next_waypoint >= source_sink->waypoints.size()) {
          to_be_removed.push_back(agent_id);  // "rogue agent"; the reference then indexes out of range
        }
        if (norm(agent.position - source_sink->waypoints.at(agent.next_waypoint)) < source_sink->radius_sink) {
          if (agent.next_waypoint == source_sink->waypoints.size() - 1) {
            if (source_sink->loop_forever) {
              next_waypoint = 0;
            } else {
              to_be_removed.push_back(agent_id);
            }
          } else {
            next_waypoint += 1;
            auto& hl = high_level_planner_.at(agent_id);
            std::lock_guard<std::mutex> g(*hl.mtx);
            hl.ptr->set_target(agents.at(agent_id), source_sink->waypoints.at(next_waypoint),
                               Vec2{source_sink->radius_sink, source_sink->radius_sink});
          }
        }
      }
      update_buffer_[agent_id] = StateUpdateBuffer{vel, new_pos, true, next_waypoint};
    }

    // --- C. commit, lib.rs:350-359
    for (auto& [id, state_update] : update_buffer_) {
      if (!state_update.updated) continue;
      Agent& agent = agents.at(id);
      agent.velocity = state_update.new_vel;
      agent.position = state_update.new_pos;
      agent.next_waypoint = state_update.next_waypoint;
      state_update.updated = false;
    }
    if (index_mode_ == IndexMode::Deferred) {
      for (auto& [id, p] : deferred_updates) spatial_index_->add_or_update(id, p);
    }

    // --- D. removals, lib.rs:378-380
    for (AgentId i : to_be_removed) remove_agents(i);
    return Status::Ok();
  }

 private:
  struct StateUpdateBuffer {  // lib.rs:94-99
    Vec2 new_vel, new_pos;
    bool updated;
    uint64_t next_waypoint;
  };

  std::vector<AgentId> iteration_order() const {
    std::vector<AgentId> order;
    if (iter_order_ == IterOrder::Custom) {
      // ids that are not live are ignored; live ids missing from the order come last, in ascending id
      std::unordered_set<AgentId> listed(custom_order_.begin(), custom_order_.end());
      for (AgentId id : custom_order_)
        if (agents.count(id)) order.push_back(id);
      std::vector<AgentId> rest;
      for (const auto& kv : agents)
        if (!listed.count(kv.first)) rest.push_back(kv.first);
      std::sort(rest.begin(), rest.end());
      order.insert(order.end(), rest.begin(), rest.end());
      return order;
    }
    order.reserve(agents.size());
    for (const auto& kv : agents) order.push_back(kv.first);
    if (iter_order_ == IterOrder::AscendingId) std::sort(order.begin(), order.end());
    return order;
  }

  Registry<std::shared_ptr<SourceSink>> source_sinks_;
  std::unique_ptr<SpatialIndex> spatial_index_;
  std::unordered_map<AgentId, Locked<HighLevelPlanner>> high_level_planner_;
  std::unordered_map<AgentId, Locked<LocalPlanner>> local_planner_;
  Duration sim_time_;  // never advanced by the reference (lib.rs:81,110)
  uint64_t last_alloc_agent_id_ = 0;
  std::unordered_map<AgentId, StateUpdateBuffer> update_buffer_;
  Registry<std::shared_ptr<EventListener>> event_listeners_;
  std::unordered_map<AgentId, uint64_t> source_sink_agent_correspondence_;
  IndexMode index_mode_;
  IterOrder iter_order_;
  std::vector<AgentId> custom_order_;
  bool trace_on_ = false;
  std::vector<AgentTrace> trace_;
};

}  // namespace orc
