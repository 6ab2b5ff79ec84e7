// rrt_oracle.cpp -- RRT::grow_tree (rrt.rs:102-174) with sample() (:176-181), restated over the oracle's KdTree, ContinuousSampler,
// SquareGoal and map checks (oracle/porrt_oracle.hpp) -- TEST INFRASTRUCTURE, the reference the device RRT growth is compared with.
// tests/rrt_oracle.py compiles it together with oracle/porrt_oracle.cpp (the same flags as oracle/Makefile) and drives it; the map
// and the goal are the handles pyoracle's GridMap and SquareGoal hold.
#include <cstdint>
#include <vector>

#include "../oracle/porrt_oracle.hpp"

#define API extern "C" __attribute__((visibility("default")))

using namespace orc;

namespace {

struct RRT {
  const GridMap* fns;
  ContinuousSampler sampler;
  KdTree kdtree;
  std::vector<State> states;
  std::vector<int64_t> parent;          // -1 at the root
  std::vector<double> dist_from_root;
  std::vector<size_t> finals;           // in the order they were found
  size_t n_it = 0;                      // iterations run; on a panic, the iteration whose check panicked
  RRT(const GridMap* m, State low, State up, uint64_t seed) : fns(m), sampler(low, up, seed), kdtree(State{0.0, 0.0}) {}
  // 0 ok, 1 = no final node ("No path found!"), < -1 = the panic code of the state check or of the first edge check in kd order
  int grow_tree(State start, const SquareGoal& goal, double max_step, double search_radius, size_t n_iter_min, size_t n_iter_max);
};

int RRT::grow_tree(State start, const SquareGoal& goal, double max_step, double search_radius, size_t n_iter_min, size_t n_iter_max) {
  states = {start};       // the start is not checked
  parent = {-1};
  dist_from_root = {0.0};
  finals.clear();
  kdtree.reset(start);
  size_t i = 0;
  while (i < n_iter_min || (finals.empty() && i < n_iter_max)) {
    i += 1;
    State new_state = (i % 100 == 0) ? goal.goal_example(0) : sampler.sample();
    const KdTree::Node& kd_from = kdtree.nearest_neighbor(new_state);
    const size_t from_id = kd_from.id;
    steer(kd_from.state, new_state, max_step);
    const int64_t svid = fns->state_validity(new_state);
    if (svid < NONE) { n_it = i; return (int)svid; }
    if (svid < 0) continue;
    const double radius = heuristic_radius(states.size(), max_step, search_radius, 2);
    std::vector<size_t> neighbours;
    for (const KdTree::Node* n : kdtree.nearest_neighbors(new_state, radius)) {   // kd pre-order
      const int64_t v = fns->transition_validator(n->state, new_state);
      if (v < NONE) { n_it = i; return (int)v; }
      if (v >= 0) neighbours.push_back(n->id);
    }
    if (neighbours.empty()) neighbours.push_back(from_id);   // unchecked
    // choose-parent: the first of equal minima (Iterator::min_by)
    size_t best = 0;
    double best_d = dist_from_root[neighbours[0]] + norm2(states[neighbours[0]], new_state);
    for (size_t k = 1; k < neighbours.size(); ++k) {
      const double d = dist_from_root[neighbours[k]] + norm2(states[neighbours[k]], new_state);
      if (d < best_d) { best = k; best_d = d; }
    }
    const size_t new_id = states.size();
    states.push_back(new_state);
    parent.push_back((int64_t)neighbours[best]);
    dist_from_root.push_back(best_d);
    // rewire: no propagation to descendants, no re-check of new -> c
    for (size_t k = 0; k < neighbours.size(); ++k) {
      if (k == best) continue;
      const size_t c = neighbours[k];
      const double d = dist_from_root[new_id] + norm2(new_state, states[c]);
      if (d < dist_from_root[c]) { parent[c] = (int64_t)new_id; dist_from_root[c] = d; }
    }
    kdtree.add(new_state, new_id);
    WorldMask f;
    if (goal.goal(new_state, &f)) finals.push_back(new_id);
  }
  n_it = i;
  return finals.empty() ? 1 : 0;
}

}  // namespace

// RRT::grow_tree on a fresh tree; returns grow_tree's code, *out = (nodes, finals, iterations); orc_rrt_export copies the tree out
API void* orc_rrt_new(const void* map, const double* low, const double* up, uint64_t seed) {
  return new RRT((const GridMap*)map, {low[0], low[1]}, {up[0], up[1]}, seed);
}
API void orc_rrt_free(void* p) { delete (RRT*)p; }
API int orc_rrt_grow_tree(void* p, const double* start, const void* goal, double max_step, double search_radius, uint64_t n_min,
                          uint64_t n_max, int64_t* out) {
  RRT* t = (RRT*)p;
  const int rc = t->grow_tree({start[0], start[1]}, *(const SquareGoal*)goal, max_step, search_radius, n_min, n_max);
  out[0] = (int64_t)t->states.size(); out[1] = (int64_t)t->finals.size(); out[2] = (int64_t)t->n_it;
  return rc;
}
API void orc_rrt_export(void* p, double* xy, int64_t* parent, double* dist, int64_t* finals) {
  const RRT* t = (RRT*)p;
  for (size_t i = 0; i < t->states.size(); ++i) {
    xy[2 * i] = t->states[i][0]; xy[2 * i + 1] = t->states[i][1];
    parent[i] = t->parent[i]; dist[i] = t->dist_from_root[i];
  }
  for (size_t k = 0; k < t->finals.size(); ++k) finals[k] = (int64_t)t->finals[k];
}
