// oracle_route_table.cpp -- RouteTablePlan for the CPU oracle (TEST INFRASTRUCTURE ONLY).
// oracle/ stays the fixed restatement of the reference; this file builds on it: it compiles oracle_capi.cpp into a
// library of its own (every orc_* call of liboracle.so) and adds a HighLevelPlanner with a caller-filled route cache
// plus the two calls that register and target it.
#include <stdexcept>

#include "../oracle/oracle_capi.cpp"

namespace orc {

// rmf::RMFPlanner (rmf/mod.rs:86-241) whose route cache the caller filled: set_target (rmf/mod.rs:217-237) selects the
// leg whose target == point (both coordinates; NaN never matches) and starts at its route point 0, and throws where no
// leg exists; get_desired_velocity is rmf/mod.rs:197-215 on that leg, exactly as RouteFollowPlan.
class RouteTablePlan : public HighLevelPlanner {
 public:
  struct Leg {
    Vec2 target;
    std::vector<Vec2> route;
  };
  explicit RouteTablePlan(std::vector<Leg> legs) : legs_(std::move(legs)) {}
  std::optional<Vec2> get_desired_velocity(const Agent& agent, Duration) override {
    auto it = agent_cache_.find(agent.agent_id);
    if (it == agent_cache_.end()) return std::nullopt;
    const std::vector<Vec2>& route = legs_[it->second.first].route;
    uint64_t waypoint_id = it->second.second;
    if (norm(agent.position - route[waypoint_id]) < 1e-1 && route.size() > waypoint_id + 1) {
      waypoint_id += 1;
      it->second.second = waypoint_id;
    }
    return normalize(route[waypoint_id] - agent.position);
  }
  void set_target(const Agent& agent, Vec2 point, Vec2) override {
    agent_cache_[agent.agent_id] = {leg_of(point), 0};
  }
  void remove_agent_id(AgentId id) override { agent_cache_.erase(id); }
  size_t leg_of(Vec2 point) const {
    for (size_t k = 0; k < legs_.size(); ++k)
      if (legs_[k].target.x == point.x && legs_[k].target.y == point.y) return k;
    throw std::invalid_argument("RouteTablePlan::set_target: no route to this point");
  }

 private:
  std::vector<Leg> legs_;
  std::unordered_map<AgentId, std::pair<size_t, uint64_t>> agent_cache_;  // agent -> (leg, route point)
};

}  // namespace orc

extern "C" {

// leg k: target targets_xy[2k..2k+1], leg_points[k] points; the legs' points concatenated in xy
int orc_hl_route_table(void* h, uint64_t n_legs, const double* targets_xy, const uint64_t* leg_points,
                       const double* xy) {
  std::vector<RouteTablePlan::Leg> legs(n_legs);
  uint64_t p = 0;
  for (uint64_t k = 0; k < n_legs; ++k) {
    legs[k].target = {targets_xy[2 * k], targets_xy[2 * k + 1]};
    for (uint64_t i = 0; i < leg_points[k]; ++i, ++p) legs[k].route.push_back({xy[2 * p], xy[2 * p + 1]});
  }
  return push_hl(static_cast<OrcSim*>(h), std::make_shared<RouteTablePlan>(std::move(legs)), nullptr);
}

// set_target(agent, targets_xy[i], (0, 0)) on planner hl for the agents ids[i], in order.  1: unknown id, 2: a point
// without a leg (the calls before the failing one stand, as in a sequence of set_target calls).
int orc_hl_route_table_set_target(void* h, int hl, uint64_t n, const uint64_t* ids, const double* targets_xy) {
  auto* s = static_cast<OrcSim*>(h);
  auto& p = s->hls.at(hl);
  for (uint64_t i = 0; i < n; ++i) {
    auto it = s->sim->agents.find(ids[i]);
    if (it == s->sim->agents.end()) return 1;
    std::lock_guard<std::mutex> g(*p.mtx);
    try {
      p.ptr->set_target(it->second, Vec2{targets_xy[2 * i], targets_xy[2 * i + 1]}, Vec2{0.0, 0.0});
    } catch (const std::invalid_argument& e) {
      s->last_error = e.what();
      return 2;
    }
  }
  return 0;
}

}  // extern "C"
