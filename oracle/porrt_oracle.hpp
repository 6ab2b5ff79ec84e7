// oracle/porrt_oracle.hpp -- TEST INFRASTRUCTURE, NOT PRODUCT CODE.
//
// CPU restatement (C++17, single-threaded unless a *_batch entry point says otherwise) of the
// hot path of cambyse/po-rrt. Every function cites the reference file:line it follows
// (paths relative to /root/reference/).  Nothing under po_rrt_b200/ may include, link or call
// this; only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference
// legs use it, as the checker / the timed CPU arm.
//
// PARITY STATUS (see DESIGN.md "Oracle"):
//  * The Rust reference cannot be built here (no cargo/rustc, nightly crate, un-vendored deps)
//    and its maps are Git-LFS pointers, so this oracle is pinned by the reference's MAP-FREE
//    golden tests only (kd-tree, dijkstra, conditional_dijkstra/extract_policy, reachability,
//    common.rs) -- tests/test_oracle_golden.py transcribes them.
//  * Third-party arithmetic restated from the published algorithms, PARITY UNPINNED:
//      line_drawing 0.8 (Bresenham + Octant), rand 0.8 / rand_pcg 0.3 (Pcg64, seed_from_u64,
//      gen_range), image 0.23 (PNM decode), priority-queue 1.0.5 (pop order among equal priorities in the
//      refiner's reparent).  The Pcg64 core is checked against the official
//      PCG known-answer vector; the Bresenham restatement against the crate's doc example.
#pragma once
#include <array>
#include <cstdint>
#include <functional>
#include <map>
#include <string>
#include <unordered_map>
#include <unordered_set>
#include <memory>
#include <array>
#include <vector>

namespace orc {

typedef std::array<double, 2> State;            // N = 2 in every BASELINE config
typedef std::vector<uint8_t> WorldMask;          // bitvec::BitVec (common.rs:9), one byte per bit
typedef std::vector<double> BeliefState;         // common.rs:10

// "panic" codes: the reference aborts; the oracle reports which panic it would have hit.
enum : int64_t {
  NONE = -1,              // Option::None  (invalid state / edge)
  PANIC_OOB = -2,         // image::get_pixel out of bounds
  PANIC_ZONE_UNWRAP = -3, // map_io.rs:172/231 unwrap() on a gray pixel without zone id (or "Zones missing")
  PANIC_MULTI_ZONE = -4   // map_io.rs:233 assert "multiple zone traversal not supported"
};

// ---------------------------------------------------------------- RNG (sample_space.rs)
struct Pcg64 {  // rand_pcg::Lcg128Xsl64
  unsigned __int128 state, inc;
  static Pcg64 from_state_incr(unsigned __int128 state, unsigned __int128 incr);
  static Pcg64 seed_from_u64(uint64_t seed);     // rand_core::SeedableRng::seed_from_u64
  uint64_t next_u64();
  double gen_range_f64(double low, double high); // rand 0.8 UniformFloat::sample_single
  uint64_t gen_range_usize(uint64_t n);          // rand 0.8 UniformInt::sample_single (0..n)
};

struct ContinuousSampler {  // sample_space.rs:6-37
  State low, up;
  Pcg64 rng;
  ContinuousSampler(State l, State u, uint64_t seed = 0) : low(l), up(u), rng(Pcg64::seed_from_u64(seed)) {}
  State sample();
};
struct DiscreteSampler {    // sample_space.rs:39-60
  Pcg64 rng;
  explicit DiscreteSampler(uint64_t seed = 0) : rng(Pcg64::seed_from_u64(seed)) {}
  uint64_t sample(uint64_t n) { return rng.gen_range_usize(n); }
};

// ---------------------------------------------------------------- common.rs
double norm1(const State& a, const State& b);                     // common.rs:192-201
double norm2(const State& a, const State& b);                     // common.rs:203-213
void steer(const State& from, State& to, double max_step);        // common.rs:215-225
double heuristic_radius(size_t n_nodes, double max_step, double search_radius, size_t dim);  // :357-369
double transition_probability(const BeliefState& parent, const BeliefState& child);          // :188-190
bool is_compatible(const BeliefState& b, const WorldMask& validity);                          // :256-264
uint64_t belief_hash(const BeliefState& b);                                                   // :352-355

// ---------------------------------------------------------------- Bresenham (line_drawing 0.8)
struct Bresenham {
  int32_t px, py, end_x, dx, dy, err;
  int octant;
  Bresenham(int32_t ax, int32_t ay, int32_t bx, int32_t by);
  bool next(int32_t& ox, int32_t& oy);
};

// ---------------------------------------------------------------- maps (map_io.rs, map_shelves_io.rs)
enum DomainKind { DOOR = 0, SHELF = 1 };
enum Space { FREE = 0, OBSTACLE = 1, ZONE = 2, LOW_OBSTACLE = 3, HIGH_OBSTACLE = 4, SPACE_PANIC = 5 };
struct Traversed { Space space; int64_t zone_or_panic; };

struct GridMap {
  int kind = DOOR;
  uint32_t H = 0, W = 0;
  std::vector<uint8_t> img;    // the reference keeps RGB (map_io.rs:93); channel 0 == the gray value
  std::vector<uint8_t> zones;  // empty when no zone image
  State low{};
  double ppm = 0;
  size_t n_zones = 0, n_worlds = 0;
  std::vector<WorldMask> zones_to_worlds, world_validities;
  std::vector<State> zone_positions;
  double visibility_distance = 0;
  std::string error;

  bool build(const uint8_t* occ, const uint8_t* zone, uint32_t H, uint32_t W, State low, State up,
             int kind, double visibility);
  void to_pixel(const State& xy, uint32_t& i, uint32_t& j) const;   // map_io.rs:176-181
  State to_coordinates(uint32_t i, uint32_t j) const;               // map_io.rs:183-188
  Traversed is_state_valid(const State& xy) const;                  // map_io.rs:165-174 / map_shelves_io.rs:158-163
  Traversed get_traversed_space(const State& a, const State& b) const;  // map_io.rs:216-241 / map_shelves_io.rs:187-203
  int64_t state_validity(const State& xy) const;                    // map_io.rs:487-493 / map_shelves_io.rs:464-469
  int64_t transition_validator(const State& from, const State& to) const;  // map_io.rs:495-513 / :471-488
  std::vector<BeliefState> successor_beliefs(const BeliefState& b, size_t zone) const;  // map_io.rs:244-278 / :206-239
  // returns false on panic (panic code in *panic)
  bool observe(const State& s, const BeliefState& b, std::vector<BeliefState>& out, int64_t* panic) const;  // map_io.rs:281-300 / :242-265
  bool visible_zones(const State& s, uint64_t* mask, int64_t* panic) const;  // geometric part of observe
  std::vector<BeliefState> reachable_belief_states(const BeliefState& b0) const;  // map_io.rs:515-546 / :490-520
};

// ---------------------------------------------------------------- kd-tree (nearest_neighbor.rs)
struct KdTree {
  struct Node { size_t id; State state; int32_t left, right; };
  std::vector<Node> nodes;  // nodes[0] is the root; Box<KdNode> links become indices
  explicit KdTree(State s, size_t id = 0) { reset(s, id); }
  void reset(State s, size_t id = 0) { nodes.clear(); nodes.push_back({id, s, -1, -1}); }
  void add(State s, size_t id);                                                   // :29-46
  const Node& nearest_neighbor_filtered(State q, const std::function<bool(size_t)>& validator) const;  // :52-92
  const Node& nearest_neighbor(State q) const;
  std::vector<const Node*> nearest_neighbors_filtered(State q, double r, const std::function<bool(size_t)>& validator) const;  // :94-122
  std::vector<const Node*> nearest_neighbors(State q, double r) const;
};

// ---------------------------------------------------------------- graph (pto_graph.rs)
struct PTOEdge { size_t id, validity_id; };
struct PTONode { State state; size_t validity_id; std::vector<PTOEdge> parents, children; };
struct PTOGraph {
  std::vector<PTONode> nodes;
  std::vector<WorldMask> validities;
  size_t add_node(State s, size_t vid) { nodes.push_back({s, vid, {}, {}}); return nodes.size() - 1; }  // :197-202
  void add_edge(size_t from, size_t to, size_t vid) {                                                       // :204-207
    nodes[from].children.push_back({to, vid});
    nodes[to].parents.push_back({from, vid});
  }
  void add_bi_edge(size_t a, size_t b, size_t vid) { add_edge(a, b, vid); add_edge(b, a, vid); }
};
// world < 0: plain graph (pto_graph.rs:230-243); world >= 0: PTOGraphWorldView (:245-271)
std::vector<double> dijkstra(const PTOGraph& g, int world, const std::vector<size_t>& finals);  // :275-303
std::vector<State> extract_path(const PTOGraph& g, int world, size_t start, const std::vector<double>& costs);  // :305-359

// ---------------------------------------------------------------- reachability (pto_reachability.rs)
struct Reachability {
  std::vector<WorldMask> validities, reachabilities, finalities;
  std::vector<size_t> final_node_ids;
  std::unordered_set<size_t> final_set;
  WorldMask finality;
  size_t n_worlds = 0;
  bool dirty = false;
  void set_root(const WorldMask& v);
  void add_node(const WorldMask& v);
  void add_final_node(size_t id, const WorldMask& f);
  void add_edge(size_t from, size_t to, const WorldMask& ev);
  std::vector<size_t> get_final_nodes_for_world(size_t world) const;
  bool is_final_set_complete();
};

// ---------------------------------------------------------------- goals (common.rs:304-350)
struct SquareGoal {
  std::vector<std::pair<State, WorldMask>> goal_to_validity;
  std::vector<State> world_to_goal;
  double max_dist = 0;
  bool init(const std::vector<std::pair<State, WorldMask>>& g, double max_dist);
  bool goal(const State& s, WorldMask* out) const;
  State goal_example(size_t world) const { return world_to_goal[world]; }
};

// ---------------------------------------------------------------- belief graph (belief_graph.rs)
enum BeliefNodeType { UNKNOWN = 0, ACTION = 1, OBSERVATION = 2 };
struct BeliefNode {
  State state; size_t belief_id; std::vector<size_t> parents, children; int node_type;
};
struct BeliefGraph {
  std::vector<BeliefNode> nodes;
  std::vector<BeliefState> reachable_belief_states;
  std::unordered_map<uint64_t, size_t> belief_states_to_id;
  size_t add_node(State s, size_t belief_id, int type) { nodes.push_back({s, belief_id, {}, {}, type}); return nodes.size() - 1; }
  void add_edge(size_t f, size_t t) { nodes[f].children.push_back(t); nodes[t].parents.push_back(f); }
  const BeliefState& belief_state(size_t node) const { return reachable_belief_states[nodes[node].belief_id]; }
};
// returns false on a reference panic (assert p > 0 / unknown node type)
bool conditional_dijkstra(const BeliefGraph& g, const std::vector<size_t>& finals, std::vector<double>& dist);  // :89-182
struct PolicyNode { State state; size_t belief_id; int64_t parent; std::vector<size_t> children; size_t original_node_id; };
struct Policy { std::vector<PolicyNode> nodes; std::vector<size_t> leafs; double expected_costs = 0; };
bool extract_policy(const BeliefGraph& g, const std::vector<double>& costs, Policy& out);  // :184-267

// ---------------------------------------------------------------- planners
// ---------------------------------------------------------------- pto_policy_refiner.rs (partial shortcut)
// is_transition_valid (pto_policy_refiner.rs:395-423): both end states valid, transition valid, and the belief compatible
// with the transition's validity.  Returns 1 / 0, or the (negative) panic code the reference would hit first.
int64_t refiner_is_transition_valid(const GridMap& m, const State& from, const State& to, const std::vector<bool>& compat_row);
// partial_shortcut (pto_policy_refiner.rs:158-206) on one path piece: `states` is modified in place; returns the number of
// committed shortcuts, or a negative panic code.  The sampler is a fresh DiscreteSampler(seed); the reference's DiscreteSampler::new()
// is seed 0.
int64_t refiner_partial_shortcut(const GridMap& m, std::vector<State>& states, const std::vector<bool>& compat_row, size_t n_iterations,
                                 uint64_t seed = 0);
// Policy::decompose (common.rs:85-129): path pieces (belief id of the piece's first node, policy node ids) + skeleton (successor pieces)
void policy_decompose(const Policy& p, std::vector<std::pair<size_t, std::vector<size_t>>>& pieces, std::vector<std::vector<size_t>>& skeleton);
// Policy::compute_expected_costs_to_goals (common.rs:131-153)
double policy_expected_costs(const Policy& p, const BeliefGraph& g);
// PTOPolicyRefiner::refine_solution(RefinmentStrategy::PartialShortCut(n)) (pto_policy_refiner.rs:85-133,135-206,324-393): decompose,
// build_path_piece + partial_shortcut per piece, recompose.  Returns false on a reference panic.
bool refiner_refine_shortcut(const GridMap& m, const Policy& policy, const BeliefGraph& g, size_t n_iterations, Policy& out, uint64_t seed = 0);
// refine_solution(RefinmentStrategy::Reparent(radius)) (pto_policy_refiner.rs:85-133,208-322): build_tree + reparent(radius / 2) per
// piece, recompose.  The pop order among equal priorities follows priority-queue 1.0.5's heap (restated; parity unpinned).
bool refiner_refine_reparent(const GridMap& m, const Policy& policy, const BeliefGraph& g, double radius, Policy& out);

struct PRM {  // prm.rs
  const GridMap* fns;
  ContinuousSampler sampler;
  KdTree kdtree;
  PTOGraph graph;
  size_t n_it = 0;
  PRM(const GridMap* m, State low, State up, uint64_t seed = 0);
  void init(State start);
  void grow_graph(double max_step, double search_radius, size_t n_iter);
  size_t add_sample(State s, double max_step, double search_radius);
  std::vector<State> plan_path(State start, State goal);
};

// Per-query answers supplied from outside (tests: the product's per-query wrappers, so that the sequential PTO growth of
// pto.rs:55-139 runs as the CALLER of the drop-in boundary).  Any null entry falls back to the oracle's own function.
struct PTOHooks {
  // 1-NN among the vertices whose reachability bit `world` is set (pto.rs:74-77); the root if none passes (nearest_neighbor.rs:89)
  int64_t (*nearest_filtered)(void* user, const double* q, uint64_t world, const uint64_t* reach_words, uint64_t n_nodes, uint64_t words) = nullptr;
  int64_t (*radius)(void* user, const double* q, double r, int64_t* out_ids, int64_t cap) = nullptr;   // kd pre-order
  int64_t (*state_validity)(void* user, const double* q) = nullptr;
  void (*edges)(void* user, const double* from_xy, const double* to_xy, int64_t n, int64_t* out_vid) = nullptr;
  void (*add_vertex)(void* user, const double* q, uint64_t id) = nullptr;
  void* user = nullptr;
};

struct PTO {  // pto.rs
  PTOHooks hooks;
  const GridMap* fns;
  ContinuousSampler continuous;
  DiscreteSampler discrete;
  KdTree kdtree;
  size_t n_worlds;
  PTOGraph graph;
  Reachability reach;
  std::vector<std::vector<int64_t>> node_to_belief_nodes;
  BeliefGraph belief_graph;
  std::vector<size_t> final_belief_nodes;
  std::vector<double> expected_costs;
  size_t n_it = 0;
  int64_t panic = 0;
  PTO(const GridMap* m, State low, State up, uint64_t seed = 0);
  // 0 ok, 1 = Err("final nodes are not reached for each world"), <0 = panic code
  int grow_graph(State start, const SquareGoal& goal, double max_step, double search_radius,
                 size_t n_iter_min, size_t n_iter_max);
  bool build_belief_graph(const BeliefState& b0);
  bool compute_expected_costs_to_goals();
  // qmdp_policy_extractor.rs
  std::vector<std::vector<double>> cost_to_goals;
  int plan_qmdp();
  bool react_qmdp(State start, const BeliefState& b, double horizon, std::vector<std::vector<State>>& paths);
};

// ---------------------------------------------------------------- map_shelves_tamp_prm.rs (multi-modal PRM baseline)
// MapShelfDomainTampPRM: one PRM per belief "mode", observation transitions between modes, conditional_dijkstra on the
// resulting explicit belief graph.  Every add_sample call is recorded per mode (state, max_step, search_radius): the whole
// growth is driven by the RNG streams only (no validity feedback), so the recorded schedule is a complete description of it.
struct TampPRM {
  struct Mode {   // :61-99
    size_t id; std::vector<size_t> remaining_zones; double reaching_probability; BeliefState belief_state;
    PRM prm; std::vector<size_t> final_node_ids;
    std::unordered_map<size_t, size_t> there, not_there;   // zone -> transition index
    std::vector<State> samples; std::vector<double> max_steps, search_radii;   // the recorded add_sample calls
    Mode(const GridMap* m, const ContinuousSampler& s) : prm(m, s.low, s.up, 0) { prm.sampler = s; }
    size_t add_sample(State s, double max_step, double search_radius);
  };
  struct Transition { size_t observed_zone_id, from_mode_id, to_mode_id; std::vector<std::array<size_t, 2>> observation_transitions; };
  const GridMap* domain;
  ContinuousSampler continuous, zone_sampler;
  DiscreteSampler discrete;
  std::vector<std::unique_ptr<Mode>> modes;
  std::vector<Transition> transitions;
  std::vector<BeliefState> belief_states;
  std::unordered_map<uint64_t, size_t> mode_hash_map;
  BeliefGraph belief_graph;
  std::vector<size_t> final_belief_node_ids;
  std::vector<double> expected_costs;
  TampPRM(const GridMap* m, State low, State up, uint64_t seed = 0);
  size_t add_mode(const std::vector<size_t>& remaining, double reaching_p, const BeliefState& b);      // :122-147
  std::vector<size_t> get_transitions(size_t mode_id, size_t target_zone_id);                           // :166-270
  State sample_observation_of_zone(size_t target_zone_id);                                               // :487-498
  void grow_mm_prm(State start, const BeliefState& b0, double max_step, double search_radius, size_t n_iter_per_belief);  // :328-397
  bool build_belief_graph();                                                                             // :399-473
  bool plan(State start, const BeliefState& b0, double max_step, double search_radius, size_t n_iter_per_belief, Policy& out);  // :308-326
};

}  // namespace orc
