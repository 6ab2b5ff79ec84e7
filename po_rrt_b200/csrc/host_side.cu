// host_side.cu -- the rows of the hot path that are sequential by nature and therefore run on the HOST inside the library
// (SURVEY.md 8(a) rows B4, B5, C5, D2, E1, E2).  They are here so that a caller finds the whole path behind one ABI and so
// that the parity tests cover them; none of them touches a pixel or walks a graph on the CPU on behalf of a device path.
//   B4 heuristic_radius      common.rs:357-369        (libm ln / pow, host only: the device never evaluates them)
//   B5 steer                 common.rs:215-225
//   C5 QMDP walk             qmdp_policy_extractor.rs:38-123  (react_qmdp / get_common_path / get_best_expected_child / get_best_child)
//   D2 Reachability          pto_reachability.rs:6-102
//   E1 samplers              sample_space.rs:6-60     (Pcg64 streams, pcg64.h)
//   E2 SquareGoal            common.rs:304-350
#include <cmath>
#include <unordered_set>

#include "common.cuh"
#include "pcg64.h"

// ------------------------------------------------------------------------------------------------ B4 / B5
PORRT_API int32_t porrt_heuristic_radius(int64_t n_nodes, double max_step, double search_radius, int32_t dim, double* out_radius) {
  if (!out_radius || dim <= 0 || n_nodes < 0) return PORRT_ERR_INVALID_ARG;
  *out_radius = heuristic_radius(n_nodes, max_step, search_radius, dim);
  return PORRT_OK;
}

PORRT_API int32_t porrt_steer(const double* from_xy, double* to_xy, int64_t n, double max_step) {
  return porrt_steer_nd(from_xy, to_xy, n, 2, max_step);
}
// steer<N> for states of `dim` doubles (the reference instantiates N = 2, 3, 7, 9)
PORRT_API int32_t porrt_steer_nd(const double* from, double* to, int64_t n, int32_t dim, double max_step) {
  if (n < 0 || dim <= 0 || dim > PORRT_MAX_STATE_DIM || (n > 0 && (!from || !to))) return PORRT_ERR_INVALID_ARG;
  for (int64_t k = 0; k < n; ++k) {
    const double* f = from + (size_t)dim * k;
    double* t = to + (size_t)dim * k;
    double step = 0.0;                                        // norm1(from, to): sum of |to - from| in dimension order
    for (int d = 0; d < dim; ++d) step += std::fabs(t[d] - f[d]);
    if (step > max_step) {
      const double lambda = max_step / step;
      for (int d = 0; d < dim; ++d) t[d] = f[d] + (t[d] - f[d]) * lambda;
    }
  }
  return PORRT_OK;
}

// ------------------------------------------------------------------------------------------------ E1 samplers
struct porrt_sampler { Pcg64 rng; };

PORRT_API int32_t porrt_sampler_create(uint64_t seed, porrt_sampler** out) {
  if (!out) return PORRT_ERR_INVALID_ARG;
  *out = new porrt_sampler{Pcg64::seed_from_u64(seed)};
  return PORRT_OK;
}
PORRT_API int32_t porrt_sampler_destroy(porrt_sampler* s) {
  delete s;
  return PORRT_OK;
}
// ContinuousSampler::sample, n times: per sample one gen_range(low[d]..up[d]) per dimension, in dimension order
PORRT_API int32_t porrt_sampler_continuous(porrt_sampler* s, const double* low, const double* up, int32_t dim, int64_t n, double* out) {
  if (!s || !low || !up || dim <= 0 || n < 0 || (n > 0 && !out)) return PORRT_ERR_INVALID_ARG;
  for (int d = 0; d < dim; ++d)
    if (!(low[d] < up[d]) || !std::isfinite(low[d]) || !std::isfinite(up[d])) return PORRT_ERR_PANIC;   // rand asserts low < high, finite
  for (int64_t k = 0; k < n; ++k)
    for (int d = 0; d < dim; ++d) out[k * dim + d] = s->rng.range_f64(low[d], up[d]);
  return PORRT_OK;
}
// DiscreteSampler::sample(n_choices), n times
PORRT_API int32_t porrt_sampler_discrete(porrt_sampler* s, uint64_t n_choices, int64_t n, uint64_t* out) {
  if (!s || n < 0 || (n > 0 && !out)) return PORRT_ERR_INVALID_ARG;
  if (n_choices == 0) return PORRT_ERR_PANIC;                 // gen_range(0..0): "cannot sample empty range"
  for (int64_t k = 0; k < n; ++k) out[k] = s->rng.below(n_choices);
  return PORRT_OK;
}

// ------------------------------------------------------------------------------------------------ E2 SquareGoal
static inline bool mask_bit(const uint64_t* m, int64_t w) { return (m[w >> 6] >> (w & 63)) & 1ull; }

// GoalFuncs::goal for a batch of states: index of the FIRST goal with norm1(state, goal) < max_dist (an L1 diamond), -1 = None
PORRT_API int32_t porrt_square_goal(const double* goals_xy, int32_t n_goals, double max_dist, const double* xy, int64_t n, int32_t* out_goal) {
  if (n_goals <= 0 || !goals_xy || n < 0 || (n > 0 && (!xy || !out_goal))) return PORRT_ERR_INVALID_ARG;
  for (int64_t k = 0; k < n; ++k) {
    int32_t hit = -1;
    for (int32_t g = 0; g < n_goals && hit < 0; ++g) {
      double d = 0.0;
      for (int c = 0; c < 2; ++c) d += std::fabs(goals_xy[2 * g + c] - xy[2 * k + c]);   // norm1(state, goal) = sum |goal - state|
      if (d < max_dist) hit = g;
    }
    out_goal[k] = hit;
  }
  return PORRT_OK;
}
// SquareGoal::new's world_to_goal table (goal_example): out_xy[2 * w] = the goal whose mask holds world w, (0, 0) if none;
// PORRT_ERR_PANIC when two masks overlap (assert, common.rs:320)
PORRT_API int32_t porrt_square_goal_examples(const double* goals_xy, const uint64_t* goal_masks, int32_t n_goals, int32_t n_worlds,
                                             double* out_xy) {
  if (n_goals <= 0 || n_worlds <= 0 || !goals_xy || !goal_masks || !out_xy) return PORRT_ERR_INVALID_ARG;
  const int words = (n_worlds + 63) / 64;
  for (int w = 0; w < n_worlds; ++w) {
    bool has = false;
    out_xy[2 * w] = out_xy[2 * w + 1] = 0.0;
    for (int g = 0; g < n_goals; ++g)
      if (mask_bit(goal_masks + (size_t)g * words, w)) {
        if (has) return PORRT_ERR_PANIC;
        out_xy[2 * w] = goals_xy[2 * g]; out_xy[2 * w + 1] = goals_xy[2 * g + 1];
        has = true;
      }
  }
  return PORRT_OK;
}

// ------------------------------------------------------------------------------------------------ D2 Reachability
struct porrt_reach {
  int n_worlds = 0, words = 1;
  std::vector<uint64_t> validity, reach;          // [n_nodes * words]
  std::vector<int64_t> final_ids;
  std::unordered_set<int64_t> final_set;
  std::vector<uint64_t> finalities;               // [n_finals * words]
  std::vector<uint64_t> finality;                 // [words]
  bool dirty = false;
  int64_t n_nodes() const { return (int64_t)(reach.size() / (size_t)words); }
  uint64_t tail_mask() const { return (n_worlds & 63) ? ((1ull << (n_worlds & 63)) - 1ull) : ~0ull; }
};

// Reachability::new + set_root(validity)
PORRT_API int32_t porrt_reach_create(int32_t n_worlds, const uint64_t* root_validity, porrt_reach** out) {
  if (!out || n_worlds <= 0 || !root_validity) return PORRT_ERR_INVALID_ARG;
  porrt_reach* r = new porrt_reach();
  r->n_worlds = n_worlds; r->words = (n_worlds + 63) / 64;
  r->validity.assign(root_validity, root_validity + r->words);
  r->reach.assign(root_validity, root_validity + r->words);      // the root reaches itself where it is valid
  r->finality.assign((size_t)r->words, 0);
  *out = r;
  return PORRT_OK;
}
PORRT_API int32_t porrt_reach_destroy(porrt_reach* r) {
  delete r;
  return PORRT_OK;
}
PORRT_API int32_t porrt_reach_add_node(porrt_reach* r, const uint64_t* validity) {
  if (!r || !validity) return PORRT_ERR_INVALID_ARG;
  r->validity.insert(r->validity.end(), validity, validity + r->words);
  r->reach.insert(r->reach.end(), (size_t)r->words, 0ull);
  return PORRT_OK;
}
PORRT_API int32_t porrt_reach_add_final_node(porrt_reach* r, int64_t id, const uint64_t* finality) {
  if (!r || !finality || id < 0) return PORRT_ERR_INVALID_ARG;
  r->final_ids.push_back(id);
  r->final_set.insert(id);
  r->finalities.insert(r->finalities.end(), finality, finality + r->words);
  r->dirty = true;
  return PORRT_OK;
}
// reach[to] |= reach[from] & edge_validity (the reference's per-bit loop, word-wise); not transitive after the fact ("conservative")
PORRT_API int32_t porrt_reach_add_edge(porrt_reach* r, int64_t from, int64_t to, const uint64_t* edge_validity) {
  if (!r || !edge_validity) return PORRT_ERR_INVALID_ARG;
  const int64_t n = r->n_nodes();
  if (from < 0 || to < 0 || from >= n || to >= n) return PORRT_ERR_PANIC;      // Vec index out of bounds
  for (int w = 0; w < r->words; ++w) r->reach[(size_t)to * r->words + w] |= r->reach[(size_t)from * r->words + w] & edge_validity[w];
  if (r->final_set.count(to)) r->dirty = true;
  return PORRT_OK;
}
PORRT_API int32_t porrt_reach_count(porrt_reach* r, int64_t* out_nodes, int32_t* out_words) {
  if (!r) return PORRT_ERR_INVALID_ARG;
  if (out_nodes) *out_nodes = r->n_nodes();
  if (out_words) *out_words = r->words;
  return PORRT_OK;
}
// reachability(id) for ids first .. first + n - 1, as the filtered nearest-neighbour search takes them (reach_mask, reach_words)
PORRT_API int32_t porrt_reach_masks(porrt_reach* r, int64_t first, int64_t n, uint64_t* out) {
  if (!r || first < 0 || n < 0 || first + n > r->n_nodes() || (n > 0 && !out)) return PORRT_ERR_INVALID_ARG;
  memcpy(out, r->reach.data() + (size_t)first * r->words, (size_t)n * r->words * 8);
  return PORRT_OK;
}
// get_final_nodes_for_world: final nodes (in add_final_node order) reached in `world` and final in it
PORRT_API int32_t porrt_reach_final_nodes_for_world(porrt_reach* r, int32_t world, int64_t* out_ids, int64_t cap, int64_t* out_n) {
  if (!r || world < 0 || world >= r->n_worlds || !out_n) return PORRT_ERR_INVALID_ARG;
  int64_t cnt = 0;
  for (size_t i = 0; i < r->final_ids.size(); ++i) {
    const int64_t id = r->final_ids[i];
    if (id >= r->n_nodes()) return PORRT_ERR_PANIC;
    if (mask_bit(r->reach.data() + (size_t)id * r->words, world) && mask_bit(r->finalities.data() + i * r->words, world)) {
      if (cnt < cap && out_ids) out_ids[cnt] = id;
      ++cnt;
    }
  }
  *out_n = cnt;
  return cnt > cap ? PORRT_ERR_CAPACITY : PORRT_OK;
}
// final_nodes_with_validities: all final nodes with their finality masks, in insertion order
PORRT_API int32_t porrt_reach_finals(porrt_reach* r, int64_t* out_ids, uint64_t* out_masks, int64_t cap, int64_t* out_n) {
  if (!r || !out_n) return PORRT_ERR_INVALID_ARG;
  *out_n = (int64_t)r->final_ids.size();
  if (*out_n > cap) return PORRT_ERR_CAPACITY;
  if (out_ids) for (size_t i = 0; i < r->final_ids.size(); ++i) out_ids[i] = r->final_ids[i];
  if (out_masks && !r->finalities.empty()) memcpy(out_masks, r->finalities.data(), r->finalities.size() * 8);
  return PORRT_OK;
}
PORRT_API int32_t porrt_reach_is_final_set_complete(porrt_reach* r, int32_t* out_complete) {
  if (!r || !out_complete) return PORRT_ERR_INVALID_ARG;
  *out_complete = 0;
  if (r->final_ids.empty()) return PORRT_OK;
  if (r->dirty) {                                             // update_finality: accumulates, never clears
    for (size_t i = 0; i < r->final_ids.size(); ++i) {
      const int64_t id = r->final_ids[i];
      if (id >= r->n_nodes()) return PORRT_ERR_PANIC;
      for (int w = 0; w < r->words; ++w) r->finality[w] |= r->reach[(size_t)id * r->words + w] & r->finalities[i * r->words + w];
    }
    r->dirty = false;
  }
  bool all = true;
  for (int w = 0; w < r->words; ++w) {
    const uint64_t want = w == r->words - 1 ? r->tail_mask() : ~0ull;
    if ((r->finality[w] & want) != want) all = false;
  }
  *out_complete = all ? 1 : 0;
  return PORRT_OK;
}

// ------------------------------------------------------------------------------------------------ C5 QMDP walk
// react_qmdp on the cost table of porrt_sssp_worlds (cost_to_goals[w * V + v]).  start_node = kdtree.nearest_neighbor(start).id
// (porrt_nearest).  Children are visited in stored order and only a STRICTLY smaller value replaces the incumbent, which starts
// as (child 0, +inf) -- so a node without a finite child sends the walk to node 0, exactly like the reference.  Where the
// reference would never return (a cycle of infinite / non-decreasing costs) the call fails with PORRT_ERR_PANIC after
// 10 V + 10 steps.  Output: the paths as node ids; paths[w] = common path + world path w (path_ptr[n_worlds + 1]).
PORRT_API int32_t porrt_qmdp_react(porrt_ctx* ctx, int64_t V, const int64_t* row_ptr, const int32_t* col, const double* xy, int32_t n_worlds,
                                   const double* cost_to_goals, int64_t start_node, const double* belief, int32_t belief_len,
                                   double common_horizon, int64_t* out_path_ptr, int32_t* out_path_nodes, int64_t cap,
                                   int64_t* out_total, int64_t* out_n_common) {
  // (host-only: ctx may be NULL, it is used for porrt_last_error alone)
  if (V <= 0 || !row_ptr || !col || !xy || n_worlds <= 0 || !cost_to_goals || !belief || !out_path_ptr || !out_total || start_node < 0 || start_node >= V)
    return porrt_fail(ctx, PORRT_ERR_INVALID_ARG, "porrt_qmdp_react: bad arguments");
  if (belief_len != n_worlds) return porrt_fail(ctx, PORRT_ERR_PANIC, "belief state size should match the number of worlds (qmdp_policy_extractor.rs:67)");
  if (row_ptr[0] != 0) return porrt_fail(ctx, PORRT_ERR_INVALID_ARG, "porrt_qmdp_react: malformed CSR");
  for (int64_t u = 0; u < V; ++u)
    if (row_ptr[u + 1] < row_ptr[u]) return porrt_fail(ctx, PORRT_ERR_INVALID_ARG, "porrt_qmdp_react: malformed CSR");
  for (int64_t e = 0; e < row_ptr[V]; ++e)
    if (col[e] < 0 || col[e] >= V) return porrt_fail(ctx, PORRT_ERR_INVALID_ARG, "porrt_qmdp_react: malformed CSR");
  const int64_t guard_max = 10 * V + 10;
  // get_common_path (:65-87)
  std::vector<int32_t> common;
  int64_t id = start_node;
  double smallest = INFINITY, acc = 0.0;
  int64_t guard = 0;
  while (acc < common_horizon && smallest > 0.0) {
    common.push_back((int32_t)id);
    int64_t best = 0;                                         // get_best_expected_child (:90-108)
    double best_c = INFINITY;
    for (int64_t e = row_ptr[id]; e < row_ptr[id + 1]; ++e) {
      const int64_t c = col[e];
      double exp_cost = 0.0;
      for (int w = 0; w < n_worlds; ++w) exp_cost += cost_to_goals[(size_t)w * V + c] * belief[w];
      if (exp_cost < best_c) { best = c; best_c = exp_cost; }
    }
    acc += norm2(xy + 2 * id, xy + 2 * best, 2);
    id = best;
    smallest = best_c;
    if (++guard > guard_max) return porrt_fail(ctx, PORRT_ERR_PANIC, "porrt_qmdp_react: the common path never ends (the reference would loop forever)");
  }
  // get_path per world (:51-62) with get_best_child (:110-123)
  std::vector<std::vector<int32_t>> tails((size_t)n_worlds);
  for (int w = 0; w < n_worlds; ++w) {
    const double* cost = cost_to_goals + (size_t)w * V;
    int64_t cur = id;
    guard = 0;
    while (cost[cur] > 0.0) {
      tails[w].push_back((int32_t)cur);
      int64_t best = 0;
      double smaller = INFINITY;
      for (int64_t e = row_ptr[cur]; e < row_ptr[cur + 1]; ++e)
        if (cost[col[e]] < smaller) { smaller = cost[col[e]]; best = col[e]; }
      cur = best;
      if (++guard > guard_max) return porrt_fail(ctx, PORRT_ERR_PANIC, "porrt_qmdp_react: a world path never ends (the reference would loop forever)");
    }
  }
  int64_t total = 0;
  for (int w = 0; w < n_worlds; ++w) total += (int64_t)common.size() + (int64_t)tails[w].size();
  *out_total = total;
  if (out_n_common) *out_n_common = (int64_t)common.size();
  if (total > cap || (total > 0 && !out_path_nodes)) return porrt_fail(ctx, PORRT_ERR_CAPACITY, "porrt_qmdp_react: out_path_nodes too small");
  int64_t o = 0;
  for (int w = 0; w < n_worlds; ++w) {
    out_path_ptr[w] = o;
    for (int32_t v : common) out_path_nodes[o++] = v;
    for (int32_t v : tails[w]) out_path_nodes[o++] = v;
  }
  out_path_ptr[n_worlds] = o;
  return PORRT_OK;
}
