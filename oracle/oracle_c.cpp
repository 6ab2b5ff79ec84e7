// oracle/oracle_c.cpp -- TEST INFRASTRUCTURE, NOT PRODUCT CODE.
// Flat C interface over the C++ restatement (porrt_oracle.hpp) so that tests/ and bench.py can drive the
// oracle through ctypes.  Handles are opaque pointers; arrays are caller-allocated numpy buffers.
#include <algorithm>
#include <chrono>
#include <cmath>
#include <cstring>

#include "porrt_oracle.hpp"

#ifdef _OPENMP
#include <omp.h>
#endif

using namespace orc;

#define API extern "C" __attribute__((visibility("default")))

static WorldMask mask_from_bytes(const uint8_t* b, size_t n) { return WorldMask(b, b + n); }

// ---------------------------------------------------------------- scalars
API double orc_norm1(const double* a, const double* b) { return norm1({a[0], a[1]}, {b[0], b[1]}); }
API double orc_norm2(const double* a, const double* b) { return norm2({a[0], a[1]}, {b[0], b[1]}); }
API void orc_steer(const double* from, double* to, double max_step) {
  State t = {to[0], to[1]};
  steer({from[0], from[1]}, t, max_step);
  to[0] = t[0]; to[1] = t[1];
}
API double orc_heuristic_radius(uint64_t n, double max_step, double search_radius, uint64_t dim) {
  return heuristic_radius(n, max_step, search_radius, dim);
}
API double orc_transition_probability(const double* parent, const double* child, uint64_t n) {
  return transition_probability(BeliefState(parent, parent + n), BeliefState(child, child + n));
}
API uint64_t orc_belief_hash(const double* b, uint64_t n) { return belief_hash(BeliefState(b, b + n)); }
API int orc_is_compatible(const double* b, const uint8_t* mask, uint64_t n) {
  return is_compatible(BeliefState(b, b + n), mask_from_bytes(mask, n));
}
API int orc_num_threads() {
#ifdef _OPENMP
  return omp_get_max_threads();
#else
  return 1;
#endif
}

// ---------------------------------------------------------------- RNG
API void* orc_pcg_seed_from_u64(uint64_t seed) { return new Pcg64(Pcg64::seed_from_u64(seed)); }
API void* orc_pcg_new(uint64_t state_hi, uint64_t state_lo, uint64_t stream_hi, uint64_t stream_lo) {
  // Lcg128Xsl64::new(state, stream): increment = (stream << 1) | 1
  unsigned __int128 st = ((unsigned __int128)state_hi << 64) | state_lo;
  unsigned __int128 sm = ((unsigned __int128)stream_hi << 64) | stream_lo;
  return new Pcg64(Pcg64::from_state_incr(st, (sm << 1) | 1));
}
API void orc_pcg_free(void* p) { delete (Pcg64*)p; }
API uint64_t orc_pcg_next_u64(void* p) { return ((Pcg64*)p)->next_u64(); }
API double orc_pcg_gen_range_f64(void* p, double l, double u) { return ((Pcg64*)p)->gen_range_f64(l, u); }
API uint64_t orc_pcg_gen_range_usize(void* p, uint64_t n) { return ((Pcg64*)p)->gen_range_usize(n); }
API void orc_pcg_fill_f64(void* p, double l, double u, double* out, uint64_t n) {
  for (uint64_t i = 0; i < n; ++i) out[i] = ((Pcg64*)p)->gen_range_f64(l, u);
}
API void orc_pcg_fill_u64(void* p, uint64_t* out, uint64_t n) {
  for (uint64_t i = 0; i < n; ++i) out[i] = ((Pcg64*)p)->next_u64();
}
// ContinuousSampler::sample() n times -> xy[2n]
API void orc_sampler_fill(void* p, const double* low, const double* up, double* xy, uint64_t n) {
  Pcg64* r = (Pcg64*)p;
  for (uint64_t i = 0; i < n; ++i)
    for (int d = 0; d < 2; ++d) xy[2 * i + d] = r->gen_range_f64(low[d], up[d]);
}

// ---------------------------------------------------------------- Bresenham
API int64_t orc_bresenham(int32_t ax, int32_t ay, int32_t bx, int32_t by, int32_t* out_xy, int64_t cap) {
  Bresenham b(ax, ay, bx, by);
  int64_t n = 0;
  int32_t x, y;
  while (b.next(x, y)) {
    if (n < cap) { out_xy[2 * n] = x; out_xy[2 * n + 1] = y; }
    ++n;
  }
  return n;
}

// ---------------------------------------------------------------- maps
API void* orc_map_create(const uint8_t* occ, const uint8_t* zone, uint32_t H, uint32_t W, const double* low,
                         const double* up, int kind, double visibility) {
  GridMap* m = new GridMap();
  if (!m->build(occ, zone, H, W, {low[0], low[1]}, {up[0], up[1]}, kind, visibility)) { delete m; return nullptr; }
  return m;
}
API void orc_map_free(void* m) { delete (GridMap*)m; }
API void orc_map_info(void* mp, int64_t* n_zones, int64_t* n_worlds, int64_t* n_validities, double* ppm) {
  GridMap* m = (GridMap*)mp;
  *n_zones = (int64_t)m->n_zones; *n_worlds = (int64_t)m->n_worlds;
  *n_validities = (int64_t)m->world_validities.size(); *ppm = m->ppm;
}
API void orc_map_zone_positions(void* mp, double* out) {
  GridMap* m = (GridMap*)mp;
  for (size_t z = 0; z < m->zone_positions.size(); ++z) { out[2 * z] = m->zone_positions[z][0]; out[2 * z + 1] = m->zone_positions[z][1]; }
}
API void orc_map_world_validities(void* mp, uint8_t* out) {  // [n_validities][n_worlds] bytes
  GridMap* m = (GridMap*)mp;
  size_t k = 0;
  for (const WorldMask& wm : m->world_validities)
    for (uint8_t b : wm) out[k++] = b;
}
API void orc_map_to_pixel(void* mp, const double* xy, uint32_t* ij) { ((GridMap*)mp)->to_pixel({xy[0], xy[1]}, ij[0], ij[1]); }
API void orc_map_to_coordinates(void* mp, const uint32_t* ij, double* xy) {
  State s = ((GridMap*)mp)->to_coordinates(ij[0], ij[1]);
  xy[0] = s[0]; xy[1] = s[1];
}
// out[i] = validity id (>=0), -1 = None, <-1 = the panic the reference would hit
API void orc_state_validity_batch(void* mp, const double* xy, int64_t n, int64_t* out) {
  GridMap* m = (GridMap*)mp;
#pragma omp parallel for schedule(static)
  for (int64_t i = 0; i < n; ++i) out[i] = m->state_validity({xy[2 * i], xy[2 * i + 1]});
}
API void orc_edge_validity_batch(void* mp, const double* from, const double* to, int64_t n, int64_t* out) {
  GridMap* m = (GridMap*)mp;
#pragma omp parallel for schedule(static)
  for (int64_t i = 0; i < n; ++i) out[i] = m->transition_validator({from[2 * i], from[2 * i + 1]}, {to[2 * i], to[2 * i + 1]});
}
// single-thread variant storing the grid like the reference (RGB, 3 B/px) is approximated by the same code:
// timing helper -- returns seconds for one pass (threads = 1 forces the reference's single-threaded behaviour)
API double orc_edge_validity_timed(void* mp, const double* from, const double* to, int64_t n, int64_t* out, int threads) {
  GridMap* m = (GridMap*)mp;
  auto t0 = std::chrono::steady_clock::now();
#ifdef _OPENMP
  if (threads < 1) threads = omp_get_max_threads();
#pragma omp parallel for schedule(static) num_threads(threads)
#endif
  for (int64_t i = 0; i < n; ++i) out[i] = m->transition_validator({from[2 * i], from[2 * i + 1]}, {to[2 * i], to[2 * i + 1]});
  auto t1 = std::chrono::steady_clock::now();
  return std::chrono::duration<double>(t1 - t0).count();
}
// exact pixel count of an edge (SURVEY 8(d): n_px = max(|di|,|dj|)+1) and #gray pixels, for the roofline bytes
API void orc_edge_pixel_counts(void* mp, const double* from, const double* to, int64_t n, int64_t* n_px_total) {
  GridMap* m = (GridMap*)mp;
  int64_t tot = 0;
#pragma omp parallel for schedule(static) reduction(+ : tot)
  for (int64_t i = 0; i < n; ++i) {
    uint32_t ai, aj, bi, bj;
    m->to_pixel({from[2 * i], from[2 * i + 1]}, ai, aj);
    m->to_pixel({to[2 * i], to[2 * i + 1]}, bi, bj);
    int64_t di = std::llabs((int64_t)ai - (int64_t)bi), dj = std::llabs((int64_t)aj - (int64_t)bj);
    tot += std::max(di, dj) + 1;
  }
  *n_px_total = tot;
}
API int orc_visible_zones_batch(void* mp, const double* xy, int64_t n, uint64_t* out_mask, int64_t* out_panic) {
  GridMap* m = (GridMap*)mp;
  int bad = 0;
#pragma omp parallel for schedule(static) reduction(| : bad)
  for (int64_t i = 0; i < n; ++i) {
    int64_t panic = 0;
    uint64_t mask = 0;
    if (!m->visible_zones({xy[2 * i], xy[2 * i + 1]}, &mask, &panic)) bad |= 1;
    out_mask[i] = mask;
    out_panic[i] = panic;
  }
  return bad;
}
// observe(): out = [count][n_worlds] f64, returns count or the panic code (<0)
API int64_t orc_observe(void* mp, const double* xy, const double* belief, double* out, int64_t cap) {
  GridMap* m = (GridMap*)mp;
  std::vector<BeliefState> res;
  int64_t panic = 0;
  BeliefState b(belief, belief + m->n_worlds);
  if (!m->observe({xy[0], xy[1]}, b, res, &panic)) return panic;
  for (size_t k = 0; k < res.size() && (int64_t)k < cap; ++k) std::memcpy(out + k * m->n_worlds, res[k].data(), 8 * m->n_worlds);
  return (int64_t)res.size();
}
API int64_t orc_reachable_belief_states(void* mp, const double* b0, double* out, int64_t cap) {
  GridMap* m = (GridMap*)mp;
  std::vector<BeliefState> res = m->reachable_belief_states(BeliefState(b0, b0 + m->n_worlds));
  for (size_t k = 0; k < res.size() && (int64_t)k < cap; ++k) std::memcpy(out + k * m->n_worlds, res[k].data(), 8 * m->n_worlds);
  return (int64_t)res.size();
}
API int64_t orc_successor_beliefs(void* mp, const double* b, uint64_t zone, double* out) {
  GridMap* m = (GridMap*)mp;
  std::vector<BeliefState> res = m->successor_beliefs(BeliefState(b, b + m->n_worlds), zone);
  for (size_t k = 0; k < res.size(); ++k) std::memcpy(out + k * m->n_worlds, res[k].data(), 8 * m->n_worlds);
  return (int64_t)res.size();
}

// ---------------------------------------------------------------- kd-tree
API void* orc_kd_new(const double* s, uint64_t id) { return new KdTree({s[0], s[1]}, id); }
API void orc_kd_free(void* t) { delete (KdTree*)t; }
API void orc_kd_add(void* t, const double* s, uint64_t id) { ((KdTree*)t)->add({s[0], s[1]}, id); }
API void orc_kd_add_batch(void* t, const double* xy, uint64_t first_id, uint64_t n) {
  for (uint64_t i = 0; i < n; ++i) ((KdTree*)t)->add({xy[2 * i], xy[2 * i + 1]}, first_id + i);
}
API uint64_t orc_kd_size(void* t) { return ((KdTree*)t)->nodes.size(); }
// structure export: per node (insertion slot order) id, left slot, right slot
API void orc_kd_export(void* t, int64_t* ids, int32_t* left, int32_t* right, double* xy) {
  KdTree* k = (KdTree*)t;
  for (size_t i = 0; i < k->nodes.size(); ++i) {
    ids[i] = (int64_t)k->nodes[i].id; left[i] = k->nodes[i].left; right[i] = k->nodes[i].right;
    xy[2 * i] = k->nodes[i].state[0]; xy[2 * i + 1] = k->nodes[i].state[1];
  }
}
// excluded: sorted-or-not list of ids rejected by the validator (the tests' closures)
API uint64_t orc_kd_nearest(void* t, const double* q, const uint64_t* excluded, uint64_t n_excl) {
  KdTree* k = (KdTree*)t;
  if (n_excl == 0) return k->nearest_neighbor({q[0], q[1]}).id;
  return k->nearest_neighbor_filtered({q[0], q[1]}, [&](size_t id) {
    return std::find(excluded, excluded + n_excl, (uint64_t)id) == excluded + n_excl;
  }).id;
}
// reach_masks: one u64 per node id; validator(id) = bit `world` of reach_masks[id]  (pto.rs:74-77)
API void orc_kd_nearest_batch(void* t, const double* q, int64_t n, const uint64_t* reach_masks, const uint32_t* world,
                              int64_t* out_id, int threads) {
  KdTree* k = (KdTree*)t;
#ifdef _OPENMP
  if (threads < 1) threads = omp_get_max_threads();
#pragma omp parallel for schedule(static) num_threads(threads)
#endif
  for (int64_t i = 0; i < n; ++i) {
    State s = {q[2 * i], q[2 * i + 1]};
    if (reach_masks) {
      uint32_t w = world[i];
      out_id[i] = (int64_t)k->nearest_neighbor_filtered(s, [&](size_t id) { return ((reach_masks[id] >> w) & 1) != 0; }).id;
    } else {
      out_id[i] = (int64_t)k->nearest_neighbor(s).id;
    }
  }
}
API int64_t orc_kd_radius(void* t, const double* q, double r, int64_t* out_ids, int64_t cap) {
  KdTree* k = (KdTree*)t;
  std::vector<const KdTree::Node*> res = k->nearest_neighbors({q[0], q[1]}, r);
  for (size_t i = 0; i < res.size() && (int64_t)i < cap; ++i) out_ids[i] = (int64_t)res[i]->id;
  return (int64_t)res.size();
}
// batched radius search: offsets[n+1] + ids (kd pre-order per query). Returns total hits; ids written up to cap.
API int64_t orc_kd_radius_batch(void* t, const double* q, const double* radius, int64_t n, int64_t* offsets,
                                int64_t* out_ids, int64_t cap, int threads) {
  KdTree* k = (KdTree*)t;
  std::vector<std::vector<int64_t>> per(n);
#ifdef _OPENMP
  if (threads < 1) threads = omp_get_max_threads();
#pragma omp parallel for schedule(dynamic, 256) num_threads(threads)
#endif
  for (int64_t i = 0; i < n; ++i) {
    std::vector<const KdTree::Node*> res = k->nearest_neighbors({q[2 * i], q[2 * i + 1]}, radius[i]);
    per[i].reserve(res.size());
    for (const KdTree::Node* nd : res) per[i].push_back((int64_t)nd->id);
  }
  int64_t tot = 0;
  for (int64_t i = 0; i < n; ++i) {
    offsets[i] = tot;
    for (int64_t id : per[i]) { if (tot < cap) out_ids[tot] = id; ++tot; }
  }
  offsets[n] = tot;
  return tot;
}

// ---------------------------------------------------------------- PTOGraph
API void* orc_graph_new(const uint8_t* validities, uint64_t n_validities, uint64_t n_worlds) {
  PTOGraph* g = new PTOGraph();
  for (uint64_t v = 0; v < n_validities; ++v) g->validities.push_back(mask_from_bytes(validities + v * n_worlds, n_worlds));
  return g;
}
API void orc_graph_free(void* g) { delete (PTOGraph*)g; }
API uint64_t orc_graph_add_node(void* g, const double* s, uint64_t vid) { return ((PTOGraph*)g)->add_node({s[0], s[1]}, vid); }
API void orc_graph_add_edge(void* g, uint64_t from, uint64_t to, uint64_t vid) { ((PTOGraph*)g)->add_edge(from, to, vid); }
API void orc_graph_add_bi_edge(void* g, uint64_t a, uint64_t b, uint64_t vid) { ((PTOGraph*)g)->add_bi_edge(a, b, vid); }
API uint64_t orc_graph_n_nodes(void* g) { return ((PTOGraph*)g)->nodes.size(); }
API uint64_t orc_graph_n_edges(void* g) {
  uint64_t e = 0;
  for (const PTONode& n : ((PTOGraph*)g)->nodes) e += n.children.size();
  return e;
}
// CSR export in stored (insertion) order. which = 0: children, 1: parents
API void orc_graph_export(void* gp, int which, double* xy, int32_t* node_vid, int64_t* row_ptr, int32_t* col, int32_t* edge_vid) {
  PTOGraph* g = (PTOGraph*)gp;
  int64_t e = 0;
  for (size_t i = 0; i < g->nodes.size(); ++i) {
    const PTONode& n = g->nodes[i];
    if (xy) { xy[2 * i] = n.state[0]; xy[2 * i + 1] = n.state[1]; }
    if (node_vid) node_vid[i] = (int32_t)n.validity_id;
    row_ptr[i] = e;
    for (const PTOEdge& ed : (which ? n.parents : n.children)) { col[e] = (int32_t)ed.id; edge_vid[e] = (int32_t)ed.validity_id; ++e; }
  }
  row_ptr[g->nodes.size()] = e;
}
API void orc_dijkstra(void* g, int world, const uint64_t* finals, uint64_t n_finals, double* out) {
  std::vector<size_t> f(finals, finals + n_finals);
  std::vector<double> d = dijkstra(*(PTOGraph*)g, world, f);
  std::memcpy(out, d.data(), 8 * d.size());
}
API int64_t orc_extract_path(void* g, int world, uint64_t start, const double* costs, double* out_xy, int64_t cap) {
  PTOGraph* gr = (PTOGraph*)g;
  std::vector<double> c(costs, costs + gr->nodes.size());
  std::vector<State> p = extract_path(*gr, world, start, c);
  for (size_t i = 0; i < p.size() && (int64_t)i < cap; ++i) { out_xy[2 * i] = p[i][0]; out_xy[2 * i + 1] = p[i][1]; }
  return (int64_t)p.size();
}
// PTOFuncs::transition_validator default impl (pto_graph.rs:130-148) on a validity table
API int64_t orc_default_transition_validator(const uint8_t* validities, uint64_t n_validities, uint64_t n_worlds, uint64_t from_vid, uint64_t to_vid) {
  std::vector<WorldMask> wv;
  for (uint64_t v = 0; v < n_validities; ++v) wv.push_back(mask_from_bytes(validities + v * n_worlds, n_worlds));
  WorldMask both(n_worlds);
  for (uint64_t w = 0; w < n_worlds; ++w) both[w] = wv[from_vid][w] && wv[to_vid][w];
  for (uint64_t v = 0; v < n_validities; ++v)
    if (wv[v] == both) return (int64_t)v;
  return NONE;
}

// ---------------------------------------------------------------- Reachability
API void* orc_reach_new() { return new Reachability(); }
API void orc_reach_free(void* r) { delete (Reachability*)r; }
API void orc_reach_set_root(void* r, const uint8_t* m, uint64_t n) { ((Reachability*)r)->set_root(mask_from_bytes(m, n)); }
API void orc_reach_add_node(void* r, const uint8_t* m, uint64_t n) { ((Reachability*)r)->add_node(mask_from_bytes(m, n)); }
API void orc_reach_add_final_node(void* r, uint64_t id, const uint8_t* m, uint64_t n) { ((Reachability*)r)->add_final_node(id, mask_from_bytes(m, n)); }
API void orc_reach_add_edge(void* r, uint64_t from, uint64_t to, const uint8_t* m, uint64_t n) { ((Reachability*)r)->add_edge(from, to, mask_from_bytes(m, n)); }
API void orc_reach_get(void* r, uint64_t id, uint8_t* out) {
  const WorldMask& m = ((Reachability*)r)->reachabilities[id];
  std::memcpy(out, m.data(), m.size());
}
API int orc_reach_is_final_set_complete(void* r) { return ((Reachability*)r)->is_final_set_complete(); }
API int64_t orc_reach_final_nodes_for_world(void* r, uint64_t world, uint64_t* out, int64_t cap) {
  std::vector<size_t> f = ((Reachability*)r)->get_final_nodes_for_world(world);
  for (size_t i = 0; i < f.size() && (int64_t)i < cap; ++i) out[i] = f[i];
  return (int64_t)f.size();
}
API int64_t orc_reach_n_finals(void* r) { return (int64_t)((Reachability*)r)->final_node_ids.size(); }
API void orc_reach_finals(void* rp, uint64_t* ids, uint8_t* finalities) {
  Reachability* r = (Reachability*)rp;
  for (size_t k = 0; k < r->final_node_ids.size(); ++k) {
    ids[k] = r->final_node_ids[k];
    std::memcpy(finalities + k * r->n_worlds, r->finalities[k].data(), r->n_worlds);
  }
}
API void orc_reach_all(void* rp, uint8_t* out) {  // [n_nodes][n_worlds]
  Reachability* r = (Reachability*)rp;
  for (size_t i = 0; i < r->reachabilities.size(); ++i) std::memcpy(out + i * r->n_worlds, r->reachabilities[i].data(), r->n_worlds);
}

// ---------------------------------------------------------------- SquareGoal
API void* orc_goal_new(const double* goals_xy, const uint8_t* masks, uint64_t n_goals, uint64_t n_worlds, double max_dist) {
  std::vector<std::pair<State, WorldMask>> g;
  for (uint64_t k = 0; k < n_goals; ++k) g.push_back({State{goals_xy[2 * k], goals_xy[2 * k + 1]}, mask_from_bytes(masks + k * n_worlds, n_worlds)});
  SquareGoal* sg = new SquareGoal();
  if (!sg->init(g, max_dist)) { delete sg; return nullptr; }
  return sg;
}
API void orc_goal_free(void* g) { delete (SquareGoal*)g; }
API int orc_goal_goal(void* g, const double* s, uint8_t* out_mask) {
  WorldMask m;
  if (!((SquareGoal*)g)->goal({s[0], s[1]}, &m)) return 0;
  std::memcpy(out_mask, m.data(), m.size());
  return 1;
}
API void orc_goal_example(void* g, uint64_t world, double* out) {
  State s = ((SquareGoal*)g)->goal_example(world);
  out[0] = s[0]; out[1] = s[1];
}

// ---------------------------------------------------------------- BeliefGraph (hand-built, belief_graph.rs tests)
API void* orc_bg_new(const double* beliefs, uint64_t n_beliefs, uint64_t n_worlds) {
  BeliefGraph* g = new BeliefGraph();
  for (uint64_t b = 0; b < n_beliefs; ++b) g->reachable_belief_states.push_back(BeliefState(beliefs + b * n_worlds, beliefs + (b + 1) * n_worlds));
  return g;
}
API void orc_bg_free(void* g) { delete (BeliefGraph*)g; }
API uint64_t orc_bg_add_node(void* g, const double* s, uint64_t belief_id, int type) { return ((BeliefGraph*)g)->add_node({s[0], s[1]}, belief_id, type); }
API void orc_bg_add_edge(void* g, uint64_t f, uint64_t t) { ((BeliefGraph*)g)->add_edge(f, t); }
API uint64_t orc_bg_n_nodes(void* g) { return ((BeliefGraph*)g)->nodes.size(); }
API uint64_t orc_bg_n_edges(void* g) {
  uint64_t e = 0;
  for (const BeliefNode& n : ((BeliefGraph*)g)->nodes) e += n.children.size();
  return e;
}
API void orc_bg_export(void* gp, int32_t* type, int32_t* belief_id, int64_t* row_ptr, int64_t* col) {
  BeliefGraph* g = (BeliefGraph*)gp;
  int64_t e = 0;
  for (size_t i = 0; i < g->nodes.size(); ++i) {
    type[i] = g->nodes[i].node_type; belief_id[i] = (int32_t)g->nodes[i].belief_id;
    row_ptr[i] = e;
    for (size_t c : g->nodes[i].children) col[e++] = (int64_t)c;
  }
  row_ptr[g->nodes.size()] = e;
}
API int orc_conditional_dijkstra(void* g, const uint64_t* finals, uint64_t n_finals, double* out) {
  std::vector<size_t> f(finals, finals + n_finals);
  std::vector<double> d;
  if (!conditional_dijkstra(*(BeliefGraph*)g, f, d)) return 0;
  std::memcpy(out, d.data(), 8 * d.size());
  return 1;
}
// policy export: per policy node: state xy, belief_id, parent (-1 root), original (belief graph) node id; leafs list
struct PolicyHandle { Policy p; };
API void* orc_extract_policy(void* g, const double* costs) {
  BeliefGraph* bg = (BeliefGraph*)g;
  std::vector<double> c(costs, costs + bg->nodes.size());
  PolicyHandle* h = new PolicyHandle();
  if (!extract_policy(*bg, c, h->p)) { delete h; return nullptr; }
  return h;
}
API void orc_policy_free(void* p) { delete (PolicyHandle*)p; }
API void orc_policy_sizes(void* p, int64_t* n_nodes, int64_t* n_leafs, double* expected) {
  Policy& pol = ((PolicyHandle*)p)->p;
  *n_nodes = (int64_t)pol.nodes.size(); *n_leafs = (int64_t)pol.leafs.size(); *expected = pol.expected_costs;
}
API void orc_policy_export(void* p, double* xy, int64_t* belief_id, int64_t* parent, int64_t* original, int64_t* leafs) {
  Policy& pol = ((PolicyHandle*)p)->p;
  for (size_t i = 0; i < pol.nodes.size(); ++i) {
    xy[2 * i] = pol.nodes[i].state[0]; xy[2 * i + 1] = pol.nodes[i].state[1];
    belief_id[i] = (int64_t)pol.nodes[i].belief_id; parent[i] = pol.nodes[i].parent; original[i] = (int64_t)pol.nodes[i].original_node_id;
  }
  for (size_t i = 0; i < pol.leafs.size(); ++i) leafs[i] = (int64_t)pol.leafs[i];
}

// ---------------------------------------------------------------- PRM
API void* orc_prm_new(void* map, const double* low, const double* up, uint64_t seed) {
  return new PRM((GridMap*)map, {low[0], low[1]}, {up[0], up[1]}, seed);
}
API void orc_prm_free(void* p) { delete (PRM*)p; }
API void orc_prm_init(void* p, const double* start) { ((PRM*)p)->init({start[0], start[1]}); }
API double orc_prm_grow_graph(void* p, double max_step, double search_radius, uint64_t n_iter) {
  auto t0 = std::chrono::steady_clock::now();
  ((PRM*)p)->grow_graph(max_step, search_radius, n_iter);
  return std::chrono::duration<double>(std::chrono::steady_clock::now() - t0).count();
}
API uint64_t orc_prm_add_sample(void* p, const double* s, double max_step, double search_radius) {
  return ((PRM*)p)->add_sample({s[0], s[1]}, max_step, search_radius);
}
// PRM::add_sample over a given sample stream (same samples as the GPU build); returns wall seconds
API double orc_prm_add_samples(void* p, const double* xy, uint64_t n, double max_step, double search_radius) {
  auto t0 = std::chrono::steady_clock::now();
  for (uint64_t k = 0; k < n; ++k) ((PRM*)p)->add_sample({xy[2 * k], xy[2 * k + 1]}, max_step, search_radius);
  return std::chrono::duration<double>(std::chrono::steady_clock::now() - t0).count();
}
API void* orc_prm_graph(void* p) { return &((PRM*)p)->graph; }
API void* orc_prm_kdtree(void* p) { return &((PRM*)p)->kdtree; }
API int64_t orc_prm_plan_path(void* p, const double* start, const double* goal, double* out_xy, int64_t cap) {
  std::vector<State> path = ((PRM*)p)->plan_path({start[0], start[1]}, {goal[0], goal[1]});
  for (size_t i = 0; i < path.size() && (int64_t)i < cap; ++i) { out_xy[2 * i] = path[i][0]; out_xy[2 * i + 1] = path[i][1]; }
  return (int64_t)path.size();
}

// ---------------------------------------------------------------- PTO
API void* orc_pto_new(void* map, const double* low, const double* up, uint64_t seed) {
  return new PTO((GridMap*)map, {low[0], low[1]}, {up[0], up[1]}, seed);
}
API void orc_pto_free(void* p) { delete (PTO*)p; }
API int orc_pto_grow_graph(void* p, const double* start, void* goal, double max_step, double search_radius, uint64_t n_min, uint64_t n_max) {
  return ((PTO*)p)->grow_graph({start[0], start[1]}, *(SquareGoal*)goal, max_step, search_radius, n_min, n_max);
}
// per-query hooks (PTOHooks): the growth then runs as the caller of whoever implements them; null pointers keep the oracle's own
API void orc_pto_set_hooks(void* p, void* nearest_filtered, void* radius, void* state_validity, void* edges, void* add_vertex) {
  PTOHooks& h = ((PTO*)p)->hooks;
  h.nearest_filtered = (decltype(h.nearest_filtered))nearest_filtered;
  h.radius = (decltype(h.radius))radius;
  h.state_validity = (decltype(h.state_validity))state_validity;
  h.edges = (decltype(h.edges))edges;
  h.add_vertex = (decltype(h.add_vertex))add_vertex;
}
API void* orc_pto_graph(void* p) { return &((PTO*)p)->graph; }
API void* orc_pto_kdtree(void* p) { return &((PTO*)p)->kdtree; }
API void* orc_pto_reach(void* p) { return &((PTO*)p)->reach; }
API void* orc_pto_belief_graph(void* p) { return &((PTO*)p)->belief_graph; }
API uint64_t orc_pto_n_it(void* p) { return ((PTO*)p)->n_it; }
API void orc_pto_set_n_worlds(void* p, uint64_t n) { ((PTO*)p)->n_worlds = n; }
API void orc_pto_set_validities(void* p, const uint8_t* validities, uint64_t n_validities, uint64_t n_worlds) {
  PTO* pto = (PTO*)p;
  pto->graph.validities.clear();
  for (uint64_t v = 0; v < n_validities; ++v) pto->graph.validities.push_back(mask_from_bytes(validities + v * n_worlds, n_worlds));
}
API int orc_pto_build_belief_graph(void* p, const double* b0, uint64_t n) {
  return ((PTO*)p)->build_belief_graph(BeliefState(b0, b0 + n)) ? 1 : 0;
}
API int64_t orc_pto_n_beliefs(void* p) { return (int64_t)((PTO*)p)->belief_graph.reachable_belief_states.size(); }
API void orc_pto_beliefs(void* p, double* out) {
  PTO* pto = (PTO*)p;
  size_t k = 0;
  for (const BeliefState& b : pto->belief_graph.reachable_belief_states)
    for (double v : b) out[k++] = v;
}
API int orc_pto_compute_expected_costs(void* p, double* out) {
  PTO* pto = (PTO*)p;
  if (!pto->compute_expected_costs_to_goals()) return 0;
  std::memcpy(out, pto->expected_costs.data(), 8 * pto->expected_costs.size());
  return 1;
}
API int64_t orc_pto_final_belief_nodes(void* p, uint64_t* out, int64_t cap) {
  PTO* pto = (PTO*)p;
  for (size_t i = 0; i < pto->final_belief_nodes.size() && (int64_t)i < cap; ++i) out[i] = pto->final_belief_nodes[i];
  return (int64_t)pto->final_belief_nodes.size();
}
API void* orc_pto_extract_policy(void* p) {
  PTO* pto = (PTO*)p;
  PolicyHandle* h = new PolicyHandle();
  if (!extract_policy(pto->belief_graph, pto->expected_costs, h->p)) { delete h; return nullptr; }
  return h;
}
// refine_solution(PartialShortCut(n)) on the PTO's last extracted policy (main.rs:442: PartialShortCut(1500)); every piece's sampler
// starts from `seed` (the reference's is seed 0)
API void* orc_pto_refine_shortcut(void* p, uint64_t n_iterations, uint64_t seed) {
  PTO* pto = (PTO*)p;
  Policy pol;
  if (!extract_policy(pto->belief_graph, pto->expected_costs, pol)) return nullptr;
  PolicyHandle* h = new PolicyHandle();
  if (!refiner_refine_shortcut(*pto->fns, pol, pto->belief_graph, (size_t)n_iterations, h->p, seed)) { delete h; return nullptr; }
  return h;
}
// Policy::decompose + compute_expected_costs_to_goals on a policy given as arrays (common.rs:85-153; the reference's tests :425-489)
API int64_t orc_policy_decompose_count(const int64_t* parent, uint64_t n) {
  Policy p;
  for (uint64_t k = 0; k < n; ++k) p.nodes.push_back({State{0.0, 0.0}, 0, parent[k], {}, 0});
  for (uint64_t k = 1; k < n; ++k) p.nodes[(size_t)parent[k]].children.push_back(k);
  std::vector<std::pair<size_t, std::vector<size_t>>> pieces;
  std::vector<std::vector<size_t>> skeleton;
  policy_decompose(p, pieces, skeleton);
  return (int64_t)pieces.size();
}
API double orc_policy_expected_cost(const double* xy, const int64_t* belief_id, const int64_t* parent, uint64_t n, const double* beliefs, uint64_t B, uint64_t nw) {
  BeliefGraph g;
  for (uint64_t b = 0; b < B; ++b) g.reachable_belief_states.push_back(BeliefState(beliefs + b * nw, beliefs + (b + 1) * nw));
  Policy p;
  for (uint64_t k = 0; k < n; ++k) p.nodes.push_back({State{xy[2 * k], xy[2 * k + 1]}, (size_t)belief_id[k], parent[k], {}, 0});
  for (uint64_t k = 1; k < n; ++k) if (parent[k] >= 0) p.nodes[(size_t)parent[k]].children.push_back(k);
  return policy_expected_costs(p, g);
}
// refine_solution(Reparent(radius)) on the PTO's last extracted policy (main.rs:221,270: Reparent(0.3))
API void* orc_pto_refine_reparent(void* p, double radius) {
  PTO* pto = (PTO*)p;
  Policy pol;
  if (!extract_policy(pto->belief_graph, pto->expected_costs, pol)) return nullptr;
  PolicyHandle* h = new PolicyHandle();
  if (!refiner_refine_reparent(*pto->fns, pol, pto->belief_graph, radius, h->p)) { delete h; return nullptr; }
  return h;
}
API int orc_pto_plan_qmdp(void* p, double* out /* [n_worlds][n_nodes] */) {
  PTO* pto = (PTO*)p;
  int rc = pto->plan_qmdp();
  if (rc) return rc;
  size_t V = pto->graph.nodes.size();
  for (size_t w = 0; w < pto->n_worlds; ++w) std::memcpy(out + w * V, pto->cost_to_goals[w].data(), 8 * V);
  return 0;
}
// paths flattened: lengths[n_worlds], xy concatenated
API int64_t orc_pto_react_qmdp(void* p, const double* start, const double* belief, double horizon, int64_t* lengths, double* xy, int64_t cap) {
  PTO* pto = (PTO*)p;
  std::vector<std::vector<State>> paths;
  if (!pto->react_qmdp({start[0], start[1]}, BeliefState(belief, belief + pto->n_worlds), horizon, paths)) return -1;
  int64_t tot = 0;
  for (size_t w = 0; w < paths.size(); ++w) {
    lengths[w] = (int64_t)paths[w].size();
    for (const State& s : paths[w]) { if (tot < cap) { xy[2 * tot] = s[0]; xy[2 * tot + 1] = s[1]; } ++tot; }
  }
  return tot;
}


// ---------------------------------------------------------------- pto_policy_refiner.rs
API void orc_refiner_transition_valid_batch(void* mp, const double* from, const double* to, int64_t n, const uint8_t* compat_row, uint64_t n_validities, int64_t* out) {
  GridMap* m = (GridMap*)mp;
  std::vector<bool> row(n_validities);
  for (uint64_t v = 0; v < n_validities; ++v) row[v] = compat_row[v] != 0;
  for (int64_t i = 0; i < n; ++i) out[i] = refiner_is_transition_valid(*m, {from[2 * i], from[2 * i + 1]}, {to[2 * i], to[2 * i + 1]}, row);
}
API int64_t orc_refiner_partial_shortcut(void* mp, double* states, uint64_t L, const uint8_t* compat_row, uint64_t n_validities, uint64_t n_iterations,
                                          uint64_t seed) {
  GridMap* m = (GridMap*)mp;
  std::vector<bool> row(n_validities);
  for (uint64_t v = 0; v < n_validities; ++v) row[v] = compat_row[v] != 0;
  std::vector<State> st(L);
  for (uint64_t k = 0; k < L; ++k) st[k] = {states[2 * k], states[2 * k + 1]};
  const int64_t rc = refiner_partial_shortcut(*m, st, row, (size_t)n_iterations, seed);
  for (uint64_t k = 0; k < L; ++k) { states[2 * k] = st[k][0]; states[2 * k + 1] = st[k][1]; }
  return rc;
}

// ---------------------------------------------------------------- multi-modal PRM (map_shelves_tamp_prm.rs)
struct TampHandle { TampPRM t; Policy policy; bool ok = false; TampHandle(GridMap* m, State lo, State up, uint64_t seed) : t(m, lo, up, seed) {} };
API void* orc_tamp_new(void* map, const double* low, const double* up, uint64_t seed) {
  return new TampHandle((GridMap*)map, {low[0], low[1]}, {up[0], up[1]}, seed);
}
API void orc_tamp_free(void* p) { delete (TampHandle*)p; }
// MapShelfDomainTampPRM::plan; returns 1 ok / 0 reference panic; *seconds = [grow_mm_prm, build_belief_graph, conditional_dijkstra, extract_policy]
API int orc_tamp_plan(void* p, const double* start, const double* b0, uint64_t n_worlds, double max_step, double search_radius,
                      uint64_t n_iter_per_belief, double* seconds) {
  TampHandle* h = (TampHandle*)p;
  BeliefState b(b0, b0 + n_worlds);
  auto now = []() { return std::chrono::steady_clock::now(); };
  auto secs = [](std::chrono::steady_clock::time_point a, std::chrono::steady_clock::time_point c) { return std::chrono::duration<double>(c - a).count(); };
  auto t0 = now();
  h->t.grow_mm_prm({start[0], start[1]}, b, max_step, search_radius, n_iter_per_belief);
  auto t1 = now();
  if (!h->t.build_belief_graph()) return 0;
  auto t2 = now();
  if (!conditional_dijkstra(h->t.belief_graph, h->t.final_belief_node_ids, h->t.expected_costs)) return 0;
  auto t3 = now();
  // no finite cost at the root: the reference's extract_policy would walk an infinite-cost cycle forever; report failure instead
  if (h->t.expected_costs.empty() || !std::isfinite(h->t.expected_costs[0])) return 0;
  h->ok = extract_policy(h->t.belief_graph, h->t.expected_costs, h->policy);
  auto t4 = now();
  if (seconds) { seconds[0] = secs(t0, t1); seconds[1] = secs(t1, t2); seconds[2] = secs(t2, t3); seconds[3] = secs(t3, t4); }
  return h->ok ? 1 : 0;
}
API void* orc_tamp_belief_graph(void* p) { return &((TampHandle*)p)->t.belief_graph; }
API void* orc_tamp_policy(void* p) {   // a copy the caller frees with orc_policy_free
  PolicyHandle* ph = new PolicyHandle();
  ph->p = ((TampHandle*)p)->policy;
  return ph;
}
// sizes: [n_modes, total_nodes, n_transitions, total_pairs, n_finals, B, n_worlds]
API void orc_tamp_sizes(void* p, int64_t* out7) {
  TampPRM& t = ((TampHandle*)p)->t;
  int64_t nodes = 0, pairs = 0, finals = 0;
  for (auto& m : t.modes) { nodes += (int64_t)m->samples.size(); finals += (int64_t)m->final_node_ids.size(); }
  for (auto& tr : t.transitions) pairs += (int64_t)tr.observation_transitions.size();
  out7[0] = (int64_t)t.modes.size(); out7[1] = nodes; out7[2] = (int64_t)t.transitions.size(); out7[3] = pairs; out7[4] = finals;
  out7[5] = (int64_t)t.belief_states.size(); out7[6] = (int64_t)t.domain->n_worlds;
}
// the recorded schedule (inputs of the product's porrt_mmprm_plan) and the expected costs (its expected output)
API void orc_tamp_export(void* p, int64_t* mode_node_ptr, double* samples_xy, double* max_steps, double* search_radii,
                         int32_t* mode_belief_id, double* beliefs /* [B * n_worlds], mode vectors substituted */,
                         int32_t* tr_from_mode, int32_t* tr_to_mode, int64_t* tr_pair_ptr, int32_t* tr_pairs,
                         int64_t* mode_final_ptr, int32_t* mode_final_nodes, double* expected_costs) {
  TampPRM& t = ((TampHandle*)p)->t;
  const size_t nw = t.domain->n_worlds;
  int64_t k = 0, f = 0;
  for (size_t m = 0; m < t.modes.size(); ++m) {
    auto& mode = *t.modes[m];
    mode_node_ptr[m] = k; mode_final_ptr[m] = f;
    for (size_t i = 0; i < mode.samples.size(); ++i, ++k) {
      samples_xy[2 * k] = mode.samples[i][0]; samples_xy[2 * k + 1] = mode.samples[i][1];
      max_steps[k] = mode.max_steps[i]; search_radii[k] = mode.search_radii[i];
    }
    for (size_t id : mode.final_node_ids) mode_final_nodes[f++] = (int32_t)id;
    mode_belief_id[m] = (int32_t)t.belief_graph.belief_states_to_id.at(belief_hash(mode.belief_state));
  }
  mode_node_ptr[t.modes.size()] = k; mode_final_ptr[t.modes.size()] = f;
  for (size_t b = 0; b < t.belief_states.size(); ++b)
    for (size_t w = 0; w < nw; ++w) beliefs[b * nw + w] = t.belief_graph.reachable_belief_states[b][w];
  int64_t q = 0;
  for (size_t i = 0; i < t.transitions.size(); ++i) {
    tr_from_mode[i] = (int32_t)t.transitions[i].from_mode_id; tr_to_mode[i] = (int32_t)t.transitions[i].to_mode_id;
    tr_pair_ptr[i] = q;
    for (auto& e : t.transitions[i].observation_transitions) { tr_pairs[2 * q] = (int32_t)e[0]; tr_pairs[2 * q + 1] = (int32_t)e[1]; ++q; }
  }
  tr_pair_ptr[t.transitions.size()] = q;
  if (expected_costs) std::memcpy(expected_costs, t.expected_costs.data(), 8 * t.expected_costs.size());
}
