// oracle_crowd_generators.cpp -- keyed PoissonCrowd and host-count generators for the CPU oracle (TEST INFRASTRUCTURE
// ONLY).  oracle/ stays the fixed restatement of the reference; this file builds on it: it compiles oracle_capi.cpp
// into a library of its own (every orc_* call of liboracle.so) and adds
//   - PoissonCrowd with the keyed draw of include/rcs.h (Philox4x64-10, threshold from glibc exp) in plain C++,
//   - a generator whose counts the caller sets for the next step (what a user-implemented CrowdGenerator looks like
//     from the step's point of view),
//   - a step that refuses dt * rate <= 0 for an alive Poisson source (Poisson::new fails, source_sink.rs:79), hands
//     the generators the number of steps executed, and consumes the host counts.
#include <cmath>
#include <map>

#include "../oracle/oracle_capi.cpp"

namespace {

struct GenState {
  uint64_t steps = 0;  // steps executed (a failed step does not count)
  std::map<uint64_t, std::shared_ptr<CrowdGenerator>> gens;  // alive source sinks added here, by id
};
std::map<void*, GenState> g_state;

uint64_t philox4x64_10_w0(uint64_t c0, uint64_t c1, uint64_t k0) {
  uint64_t c2 = 0, c3 = 0, k1 = 0;
  for (int r = 0; r < 10; ++r) {
    const unsigned __int128 p0 = (unsigned __int128)0xD2E7470EE14C6C93ull * c0;
    const unsigned __int128 p1 = (unsigned __int128)0xCA5A826395121157ull * c2;
    const uint64_t hi0 = (uint64_t)(p0 >> 64), lo0 = (uint64_t)p0, hi1 = (uint64_t)(p1 >> 64), lo1 = (uint64_t)p1;
    c0 = hi1 ^ c1 ^ k0;
    c1 = lo1;
    c2 = hi0 ^ c3 ^ k1;
    c3 = lo0;
    k0 += 0x9E3779B97F4A7C15ull;
    k1 += 0xBB67AE8584CAA73Bull;
  }
  return c0;
}

bool poisson_wants(double rate, uint64_t seed, Duration dur, uint64_t step, uint64_t sid) {
  const uint64_t thr = (uint64_t)std::ceil(std::ldexp(std::exp(-(dur.as_secs_f64() * rate)), 53));
  return (philox4x64_10_w0(step + 1, sid, seed) >> 11) >= thr;
}

class KeyedPoissonCrowd : public CrowdGenerator {
 public:
  KeyedPoissonCrowd(double rate, uint64_t seed, const uint64_t* steps) : rate(rate), seed(seed), steps_(steps) {}
  uint64_t get_number_to_spawn(Duration dur) const override { return poisson_wants(rate, seed, dur, *steps_, sid) ? 1 : 0; }
  double rate;
  uint64_t seed;
  uint64_t sid = 0;

 private:
  const uint64_t* steps_;
};

class HostCountCrowd : public CrowdGenerator {
 public:
  uint64_t get_number_to_spawn(Duration) const override { return count; }
  uint64_t count = 0;
};

}  // namespace

extern "C" {

// kind 0 Monotonic, 1 Poisson, 2 host counts.  1: a Poisson rate that is not finite and > 0 (nothing added).
int orc_add_source_sink_gen(void* h, double sx, double sy, double radius_sink, int kind, double rate, uint64_t seed,
                            int hl, int lp, uint64_t n_wp, const double* wp_xy, int loop_forever, double eyesight,
                            uint64_t* out_id) {
  auto* s = static_cast<OrcSim*>(h);
  GenState& st = g_state[h];
  std::shared_ptr<CrowdGenerator> gen;
  if (kind == 1) {
    if (!(std::isfinite(rate) && rate > 0.0)) {
      s->last_error = "PoissonCrowd: the rate must be finite and > 0";
      return 1;
    }
    gen = std::make_shared<KeyedPoissonCrowd>(rate, seed, &st.steps);
  } else if (kind == 2) {
    gen = std::make_shared<HostCountCrowd>();
  } else {
    gen = std::make_shared<MonotonicCrowd>(rate);
  }
  auto ss = std::make_shared<SourceSink>();
  ss->source = {sx, sy};
  ss->radius_sink = radius_sink;
  ss->crowd_generator = gen;
  ss->high_level_planner = s->hls.at(hl);
  ss->local_planner = s->lps.at(lp);
  for (uint64_t i = 0; i < n_wp; ++i) ss->waypoints.push_back({wp_xy[2 * i], wp_xy[2 * i + 1]});
  ss->loop_forever = loop_forever != 0;
  ss->agent_eyesight_range = eyesight;
  const uint64_t id = s->sim->add_source_sink(ss);
  if (kind == 1) static_cast<KeyedPoissonCrowd*>(gen.get())->sid = id;
  st.gens[id] = gen;
  if (out_id) *out_id = id;
  return 0;
}

void orc_remove_source_sink_gen(void* h, uint64_t id) {
  static_cast<OrcSim*>(h)->sim->remove_source_sink(id);
  g_state[h].gens.erase(id);
}

// 1: an id that is not an alive host-count source (nothing written)
int orc_set_spawn_counts(void* h, uint64_t n, const uint64_t* ids, const uint64_t* counts) {
  GenState& st = g_state[h];
  for (uint64_t i = 0; i < n; ++i) {
    auto it = st.gens.find(ids[i]);
    if (it == st.gens.end() || !dynamic_cast<HostCountCrowd*>(it->second.get())) return 1;
  }
  for (uint64_t i = 0; i < n; ++i) static_cast<HostCountCrowd*>(st.gens[ids[i]].get())->count = counts[i];
  return 0;
}

// orc_step with the generators of this file: 3 = dt * rate <= 0 for an alive Poisson source (nothing runs)
int orc_step_gen(void* h, uint64_t secs, uint32_t nanos) {
  auto* s = static_cast<OrcSim*>(h);
  GenState& st = g_state[h];
  const double dt = Duration{secs, nanos}.as_secs_f64();
  for (auto& kv : st.gens) {
    auto* p = dynamic_cast<KeyedPoissonCrowd*>(kv.second.get());
    if (p && !(dt * p->rate > 0.0)) {
      s->last_error = "PoissonCrowd: dt * rate must be > 0";
      return 3;
    }
  }
  const int rc = orc_step(h, secs, nanos);
  if (rc == 0) st.steps += 1;
  for (auto& kv : st.gens)  // the counts were for this step only
    if (auto* c = dynamic_cast<HostCountCrowd*>(kv.second.get())) c->count = 0;
  return rc;
}

uint64_t orc_gen_steps(void* h) { return g_state[h].steps; }

void orc_gen_release(void* h) { g_state.erase(h); }

// the keyed PoissonCrowd decision on its own
int orc_poisson_wants(double rate, uint64_t seed, uint64_t secs, uint32_t nanos, uint64_t step, uint64_t sid) {
  return poisson_wants(rate, seed, Duration{secs, nanos}, step, sid) ? 1 : 0;
}

uint64_t orc_philox4x64_10_w0(uint64_t c0, uint64_t c1, uint64_t k0) { return philox4x64_10_w0(c0, c1, k0); }

}  // extern "C"
