// oracle/porrt_oracle.cpp -- TEST INFRASTRUCTURE, NOT PRODUCT CODE (see porrt_oracle.hpp).
// CPU restatement of po-rrt's hot path; each block cites the reference file:line it follows.
#include "porrt_oracle.hpp"

#include <algorithm>
#include <deque>
#include <cmath>
#include <cstring>
#include <limits>
#include <queue>
#include <unordered_set>

namespace orc {

static const double INF = std::numeric_limits<double>::infinity();

// ============================================================== RNG
// rand_pcg 0.3 Lcg128Xsl64 (pcg128.rs): MULTIPLIER, step, output_xsl_rr, from_state_incr.
static const unsigned __int128 PCG_MUL =
    ((unsigned __int128)0x2360ED051FC65DA4ULL << 64) | (unsigned __int128)0x4385DF649FCCF645ULL;

Pcg64 Pcg64::from_state_incr(unsigned __int128 state, unsigned __int128 incr) {
  Pcg64 p;
  p.state = state;
  p.inc = incr;
  p.state = p.state + p.inc;       // "move away from inital value"
  p.state = p.state * PCG_MUL + p.inc;
  return p;
}

// rand_core 0.6 SeedableRng::seed_from_u64: PCG32 stream fills the 32-byte seed, 4 bytes at a time;
// Lcg128Xsl64::from_seed reads four LE u64: state = s0|s1<<64, incr = (s2|s3<<64) | 1.
Pcg64 Pcg64::seed_from_u64(uint64_t st) {
  const uint64_t MUL = 6364136223846793005ULL, INC = 11634580027462260723ULL;
  uint32_t w[8];
  for (int c = 0; c < 8; ++c) {
    st = st * MUL + INC;
    uint32_t xorshifted = (uint32_t)(((st >> 18) ^ st) >> 27);
    uint32_t rot = (uint32_t)(st >> 59);
    w[c] = (xorshifted >> rot) | (xorshifted << ((32 - rot) & 31));
  }
  uint64_t s[4];
  for (int k = 0; k < 4; ++k) s[k] = (uint64_t)w[2 * k] | ((uint64_t)w[2 * k + 1] << 32);
  unsigned __int128 state = (unsigned __int128)s[0] | ((unsigned __int128)s[1] << 64);
  unsigned __int128 incr = (unsigned __int128)s[2] | ((unsigned __int128)s[3] << 64);
  return from_state_incr(state, incr | 1);
}

uint64_t Pcg64::next_u64() {
  state = state * PCG_MUL + inc;
  uint32_t rot = (uint32_t)(state >> 122);
  uint64_t xsl = (uint64_t)(state >> 64) ^ (uint64_t)state;
  return (xsl >> rot) | (xsl << ((64 - rot) & 63));
}

// rand 0.8 distributions/uniform.rs UniformFloat<f64>::sample_single (sample_space.rs:33).
double Pcg64::gen_range_f64(double low, double high) {
  double scale = high - low;
  for (;;) {
    uint64_t bits = (next_u64() >> 12) | 0x3FF0000000000000ULL;  // into_float_with_exponent(0): [1,2)
    double value1_2;
    std::memcpy(&value1_2, &bits, 8);
    double value0_1 = value1_2 - 1.0;
    double res = value0_1 * scale + low;
    if (res < high) return res;
    // rand's edge-case branch shrinks `scale` by one ulp and retries
    uint64_t sb;
    std::memcpy(&sb, &scale, 8);
    sb -= 1;
    std::memcpy(&scale, &sb, 8);
  }
}

// rand 0.8 UniformInt<usize>::sample_single_inclusive(0, n-1) (sample_space.rs:58).
uint64_t Pcg64::gen_range_usize(uint64_t range) {
  if (range == 0) return next_u64();
  uint64_t zone = (range << __builtin_clzll(range)) - 1;
  for (;;) {
    uint64_t v = next_u64();
    unsigned __int128 m = (unsigned __int128)v * range;
    uint64_t hi = (uint64_t)(m >> 64), lo = (uint64_t)m;
    if (lo <= zone) return hi;
  }
}

State ContinuousSampler::sample() {  // sample_space.rs:30-37
  State s;
  for (int d = 0; d < 2; ++d) s[d] = rng.gen_range_f64(low[d], up[d]);
  return s;
}

// ============================================================== common.rs
double norm1(const State& a, const State& b) {
  double d = 0.0;
  for (int k = 0; k < 2; ++k) d += std::fabs(b[k] - a[k]);
  return d;
}
double norm2(const State& a, const State& b) {
  double d2 = 0.0;
  for (int k = 0; k < 2; ++k) {
    double dx = b[k] - a[k];
    d2 += dx * dx;
  }
  return std::sqrt(d2);
}
void steer(const State& from, State& to, double max_step) {
  double step = norm1(from, to);
  if (step > max_step) {
    double lambda = max_step / step;
    for (int i = 0; i < 2; ++i) to[i] = from[i] + (to[i] - from[i]) * lambda;
  }
}
double heuristic_radius(size_t n_nodes, double max_step, double search_radius, size_t dim) {
  double n = (double)n_nodes;
  double s = search_radius * std::pow(std::log(n) / n, 1.0 / (double)dim);
  return s < max_step ? s : max_step;
}
double transition_probability(const BeliefState& parent, const BeliefState& child) {
  double s = 0.0;
  size_t n = std::min(parent.size(), child.size());
  for (size_t i = 0; i < n; ++i) s = s + (child[i] > 0.0 ? parent[i] : 0.0);
  return s;
}
bool is_compatible(const BeliefState& b, const WorldMask& validity) {
  size_t n = std::min(b.size(), validity.size());
  for (size_t i = 0; i < n; ++i)
    if (b[i] > 0.0 && !validity[i]) return false;
  return true;
}
// common.rs:352-355; usize arithmetic wraps in release builds (overflow from 18 worlds up).
uint64_t belief_hash(const BeliefState& bs) {
  uint64_t h = 0, p10 = 1;
  for (size_t i = 0; i < bs.size(); ++i) {
    double r = std::round(bs[i] * 1000.0);  // f64::round = half away from zero = C round()
    uint64_t v = r <= 0.0 || std::isnan(r) ? 0 : (r >= 18446744073709551615.0 ? UINT64_MAX : (uint64_t)r);
    h += (p10 + 1) * v;
    p10 *= 10;
  }
  return h;
}

// ============================================================== Bresenham (line_drawing 0.8)
static inline void octant_to(int o, int32_t x, int32_t y, int32_t& ox, int32_t& oy) {
  switch (o) {
    case 0: ox = x; oy = y; break;
    case 1: ox = y; oy = x; break;
    case 2: ox = y; oy = -x; break;
    case 3: ox = -x; oy = y; break;
    case 4: ox = -x; oy = -y; break;
    case 5: ox = -y; oy = -x; break;
    case 6: ox = -y; oy = x; break;
    default: ox = x; oy = -y; break;
  }
}
static inline void octant_from(int o, int32_t x, int32_t y, int32_t& ox, int32_t& oy) {
  switch (o) {
    case 0: ox = x; oy = y; break;
    case 1: ox = y; oy = x; break;
    case 2: ox = -y; oy = x; break;
    case 3: ox = -x; oy = y; break;
    case 4: ox = -x; oy = -y; break;
    case 5: ox = -y; oy = -x; break;
    case 6: ox = y; oy = -x; break;
    default: ox = x; oy = -y; break;
  }
}
Bresenham::Bresenham(int32_t ax, int32_t ay, int32_t bx, int32_t by) {
  int value = 0;
  int32_t ddx = bx - ax, ddy = by - ay;
  if (ddy < 0) { ddx = -ddx; ddy = -ddy; value += 4; }
  if (ddx < 0) { int32_t t = ddx; ddx = ddy; ddy = -t; value += 2; }
  if (ddx < ddy) value += 1;
  octant = value;
  int32_t sx, sy, ex, ey;
  octant_to(octant, ax, ay, sx, sy);
  octant_to(octant, bx, by, ex, ey);
  dx = ex - sx;
  dy = ey - sy;
  px = sx; py = sy; end_x = ex;
  err = dy - dx;
}
bool Bresenham::next(int32_t& ox, int32_t& oy) {
  if (px <= end_x) {
    octant_from(octant, px, py, ox, oy);
    if (err >= 0) { py += 1; err -= dx; }
    px += 1;
    err += dy;
    return true;
  }
  return false;
}

// ============================================================== maps
static inline uint32_t f64_as_u32(double v) {  // Rust `as u32`: saturating, NaN -> 0
  if (!(v > 0.0)) return 0;
  if (v >= 4294967295.0) return 4294967295u;
  return (uint32_t)v;
}

bool GridMap::build(const uint8_t* occ, const uint8_t* zone, uint32_t h, uint32_t w, State lo, State up,
                    int k, double visibility) {
  kind = k; H = h; W = w; low = lo;
  ppm = (double)w / (up[0] - lo[0]);  // map_io.rs:91
  img.assign(occ, occ + (size_t)h * w);
  zones.clear(); zones_to_worlds.clear(); world_validities.clear(); zone_positions.clear();
  n_zones = 0; n_worlds = 0; visibility_distance = 0.0;
  if (!zone) {
    if (kind == DOOR) {  // Map::init_without_zones, map_io.rs:108-111
      n_worlds = 1;
      world_validities.push_back(WorldMask(1, 1));
    }
    return true;
  }
  zones.assign(zone, zone + (size_t)h * w);
  // init_zone_ids (map_io.rs:130-145): n_zones = max id + 1 (1 even when no zone pixel exists)
  size_t max_id = 0;
  for (size_t p = 0; p < zones.size(); ++p)
    if (zones[p] != 255 && zones[p] > max_id) max_id = zones[p];
  n_zones = max_id + 1;
  if (kind == DOOR) {
    if (n_zones >= 32) { error = "2_u32.pow(n_zones) overflows"; return false; }
    n_worlds = (size_t)1 << n_zones;
  } else {
    n_worlds = n_zones;  // map_shelves_io.rs:460-462
  }
  // init_zone_positions (map_io.rs:147-163): u32 sums (wrapping as in a release build), integer mean
  std::vector<uint32_t> si(n_zones, 0), sj(n_zones, 0), cnt(n_zones, 0);
  for (uint32_t i = 0; i < h; ++i)
    for (uint32_t j = 0; j < w; ++j) {
      uint8_t z = zones[(size_t)i * w + j];
      if (z != 255) { si[z] += i; sj[z] += j; cnt[z] += 1; }
    }
  for (size_t z = 0; z < n_zones; ++z) {
    if (cnt[z] == 0) { error = "zone without pixels: division by zero panic (map_io.rs:160)"; return false; }
    zone_positions.push_back(to_coordinates(si[z] / cnt[z], sj[z] / cnt[z]));
  }
  visibility_distance = visibility;
  if (kind == DOOR) {
    for (size_t z = 0; z < n_zones; ++z) {  // zone_index_to_world_mask, map_io.rs:198-214
      WorldMask m(n_worlds, 1);
      for (size_t wd = 0; wd < n_worlds; ++wd)
        if ((wd & ((size_t)1 << z)) == 0) m[wd] = 0;
      zones_to_worlds.push_back(m);
    }
    world_validities = zones_to_worlds;
    world_validities.push_back(WorldMask(n_worlds, 1));  // all-ones mask is LAST (map_io.rs:125-126)
  } else {
    world_validities.push_back(WorldMask(n_zones, 1));   // map_shelves_io.rs:113
  }
  return true;
}

void GridMap::to_pixel(const State& xy, uint32_t& i, uint32_t& j) const {
  i = f64_as_u32((double)(H - 1) - (xy[1] - low[1]) * ppm);
  j = f64_as_u32((xy[0] - low[0]) * ppm);
}
State GridMap::to_coordinates(uint32_t i, uint32_t j) const {  // note the swapped low[] indices, as in the reference
  State s;
  s[0] = (double)j / ppm + low[1];
  s[1] = (double)(H - 1 - i) / ppm + low[0];
  return s;
}

static inline Space shelf_class(uint8_t p) {  // pixel_to_occupation, map_shelves_io.rs:150-156
  return p == 255 ? FREE : (p >= 127 ? LOW_OBSTACLE : HIGH_OBSTACLE);
}

Traversed GridMap::is_state_valid(const State& xy) const {
  uint32_t i, j;
  to_pixel(xy, i, j);
  if (i >= H || j >= W) return {SPACE_PANIC, PANIC_OOB};
  uint8_t p = img[(size_t)i * W + j];
  if (kind == SHELF) return {shelf_class(p), 0};
  if (p == 255) return {FREE, 0};
  if (p == 0) return {OBSTACLE, 0};
  if (zones.empty() || zones[(size_t)i * W + j] == 255) return {SPACE_PANIC, PANIC_ZONE_UNWRAP};
  return {ZONE, (int64_t)zones[(size_t)i * W + j]};
}

Traversed GridMap::get_traversed_space(const State& a, const State& b) const {
  uint32_t ai, aj, bi, bj;
  to_pixel(a, ai, aj);
  to_pixel(b, bi, bj);
  Bresenham line((int32_t)ai, (int32_t)aj, (int32_t)bi, (int32_t)bj);
  int32_t i, j;
  if (kind == SHELF) {
    uint8_t lowest = 255;
    while (line.next(i, j)) {
      if ((uint32_t)i >= H || (uint32_t)j >= W) return {SPACE_PANIC, PANIC_OOB};
      uint8_t p = img[(size_t)(uint32_t)i * W + (uint32_t)j];
      lowest = std::min(lowest, p);
      if (lowest == 0) return {HIGH_OBSTACLE, 0};
    }
    return {shelf_class(lowest), 0};
  }
  Traversed t = {FREE, 0};
  while (line.next(i, j)) {
    if ((uint32_t)i >= H || (uint32_t)j >= W) return {SPACE_PANIC, PANIC_OOB};
    size_t at = (size_t)(uint32_t)i * W + (uint32_t)j;
    uint8_t p = img[at];
    if (p == 255) continue;
    if (p == 0) return {OBSTACLE, 0};
    if (zones.empty() || zones[at] == 255) return {SPACE_PANIC, PANIC_ZONE_UNWRAP};
    int64_t z = zones[at];
    if (t.space == ZONE && t.zone_or_panic != z) return {SPACE_PANIC, PANIC_MULTI_ZONE};
    t = {ZONE, z};
  }
  return t;
}

static int64_t space_to_validity(const GridMap& m, const Traversed& t) {
  switch (t.space) {
    case SPACE_PANIC: return t.zone_or_panic;
    case FREE: return (int64_t)m.world_validities.size() - 1;
    case ZONE: return t.zone_or_panic;
    default: return NONE;
  }
}
int64_t GridMap::state_validity(const State& xy) const { return space_to_validity(*this, is_state_valid(xy)); }
int64_t GridMap::transition_validator(const State& from, const State& to) const {
  return space_to_validity(*this, get_traversed_space(from, to));
}

static void normalize(BeliefState& b) {
  double sum = 0.0;
  for (double p : b) sum = sum + p;
  for (double& p : b) p /= sum;
}
static bool any_nan(const BeliefState& b) {
  for (double p : b)
    if (std::isnan(p)) return true;
  return false;
}
std::vector<BeliefState> GridMap::successor_beliefs(const BeliefState& b, size_t zone) const {
  std::vector<BeliefState> out;
  if (kind == DOOR) {
    const WorldMask& mask = zones_to_worlds[zone];
    BeliefState closed = b, open = b;
    for (size_t w = 0; w < mask.size(); ++w) closed[w] = mask[w] ? 0.0 : b[w];
    normalize(closed);
    if (!any_nan(closed)) out.push_back(closed);
    for (size_t w = 0; w < mask.size(); ++w) open[w] = mask[w] ? b[w] : 0.0;
    normalize(open);
    if (!any_nan(open)) out.push_back(open);
  } else {
    BeliefState there = b, not_there = b;
    for (size_t w = 0; w < there.size(); ++w) there[w] = (w == zone) ? there[w] : 0.0;
    normalize(there);
    if (!any_nan(there)) out.push_back(there);
    for (size_t w = 0; w < not_there.size(); ++w) not_there[w] = (w == zone) ? 0.0 : b[w];
    normalize(not_there);
    if (!any_nan(not_there)) out.push_back(not_there);
  }
  return out;
}

bool GridMap::visible_zones(const State& s, uint64_t* mask, int64_t* panic) const {
  uint64_t m = 0;
  for (size_t z = 0; z < n_zones; ++z) {
    if (norm2(s, zone_positions[z]) < visibility_distance) {
      Traversed t = get_traversed_space(s, zone_positions[z]);
      if (t.space == SPACE_PANIC) { if (panic) *panic = t.zone_or_panic; return false; }
      bool fov = kind == DOOR ? (t.space != OBSTACLE) : (t.space != HIGH_OBSTACLE);
      if (fov) m |= (uint64_t)1 << z;
    }
  }
  *mask = m;
  return true;
}

bool GridMap::observe(const State& s, const BeliefState& b, std::vector<BeliefState>& out, int64_t* panic) const {
  out.clear();
  out.push_back(b);
  for (size_t z = 0; z < n_zones; ++z) {
    if (norm2(s, zone_positions[z]) < visibility_distance) {
      Traversed t = get_traversed_space(s, zone_positions[z]);
      if (t.space == SPACE_PANIC) { if (panic) *panic = t.zone_or_panic; return false; }
      bool fov = kind == DOOR ? (t.space != OBSTACLE) : (t.space != HIGH_OBSTACLE);
      if (fov) {
        std::vector<BeliefState> beliefs = out;
        out.clear();
        for (const BeliefState& bel : beliefs) {
          std::vector<BeliefState> succ = successor_beliefs(bel, z);
          out.insert(out.end(), succ.begin(), succ.end());
        }
      }
    }
  }
  return true;
}

std::vector<BeliefState> GridMap::reachable_belief_states(const BeliefState& b0) const {
  std::vector<BeliefState> reachable;
  std::unordered_set<uint64_t> hashes;
  std::vector<std::pair<BeliefState, std::vector<size_t>>> lifo;
  reachable.push_back(b0);
  std::vector<size_t> all(n_zones);
  for (size_t z = 0; z < n_zones; ++z) all[z] = z;
  lifo.push_back({b0, all});
  while (!lifo.empty()) {
    std::pair<BeliefState, std::vector<size_t>> top = lifo.back();
    lifo.pop_back();
    for (size_t zone_id : top.second) {
      std::vector<size_t> remaining;
      for (size_t id : top.second)
        if (id != zone_id) remaining.push_back(id);
      std::vector<BeliefState> succ = successor_beliefs(top.first, zone_id);
      for (const BeliefState& s : succ) {
        if (std::find(reachable.begin(), reachable.end(), s) == reachable.end()) {
          uint64_t h = belief_hash(s);
          if (!hashes.count(h)) {
            reachable.push_back(s);
            hashes.insert(h);
          }
          lifo.push_back({s, remaining});
        }
      }
    }
  }
  return reachable;
}

// ============================================================== kd-tree
void KdTree::add(State s, size_t id) {
  int32_t cur = 0;
  for (size_t axis = 0;; axis = (axis + 1) % 2) {
    int32_t* next = s[axis] < nodes[cur].state[axis] ? &nodes[cur].left : &nodes[cur].right;
    if (*next >= 0) {
      cur = *next;
    } else {
      *next = (int32_t)nodes.size();
      nodes.push_back({id, s, -1, -1});
      return;
    }
  }
}

template <class F>
static void nn_inner(const KdTree& t, const State& q, double& dmin, int32_t& nearest, int32_t from, size_t axis, F& validator) {
  const KdTree::Node& n = t.nodes[from];
  double d = norm2(n.state, q);
  if (d < dmin && validator(n.id)) { dmin = d; nearest = from; }
  size_t next_axis = (axis + 1) % 2;
  if (q[axis] < n.state[axis]) {
    if (q[axis] - dmin < n.state[axis] && n.left >= 0) nn_inner(t, q, dmin, nearest, n.left, next_axis, validator);
    if (q[axis] + dmin >= n.state[axis] && n.right >= 0) nn_inner(t, q, dmin, nearest, n.right, next_axis, validator);
  } else {
    if (q[axis] + dmin >= n.state[axis] && n.right >= 0) nn_inner(t, q, dmin, nearest, n.right, next_axis, validator);
    if (q[axis] - dmin < n.state[axis] && n.left >= 0) nn_inner(t, q, dmin, nearest, n.left, next_axis, validator);
  }
}
template <class F>
static const KdTree::Node& nn_filtered(const KdTree& t, State q, F validator) {
  double dmin = INF;
  int32_t nearest = 0;  // root when nothing passes the filter (nearest_neighbor.rs:89)
  nn_inner(t, q, dmin, nearest, 0, 0, validator);
  return t.nodes[nearest];
}
const KdTree::Node& KdTree::nearest_neighbor_filtered(State q, const std::function<bool(size_t)>& validator) const {
  return nn_filtered(*this, q, validator);
}
const KdTree::Node& KdTree::nearest_neighbor(State q) const {
  return nn_filtered(*this, q, [](size_t) { return true; });
}

template <class F>
static void radius_inner(const KdTree& t, const State& q, double radius, std::vector<const KdTree::Node*>& out,
                         int32_t from, size_t axis, F& validator) {
  const KdTree::Node& n = t.nodes[from];
  double d = norm2(n.state, q);
  if (d <= radius && validator(n.id)) out.push_back(&n);
  size_t next_axis = (axis + 1) % 2;
  if (q[axis] - radius <= n.state[axis] && n.left >= 0) radius_inner(t, q, radius, out, n.left, next_axis, validator);
  if (q[axis] + radius >= n.state[axis] && n.right >= 0) radius_inner(t, q, radius, out, n.right, next_axis, validator);
}
std::vector<const KdTree::Node*> KdTree::nearest_neighbors_filtered(State q, double r, const std::function<bool(size_t)>& validator) const {
  std::vector<const Node*> out;
  radius_inner(*this, q, r, out, 0, 0, validator);
  return out;
}
std::vector<const KdTree::Node*> KdTree::nearest_neighbors(State q, double r) const {
  std::vector<const Node*> out;
  auto all = [](size_t) { return true; };
  radius_inner(*this, q, r, out, 0, 0, all);
  return out;
}

// ============================================================== dijkstra
struct HeapItem {
  double prio; size_t id;
  bool operator<(const HeapItem& o) const { return prio > o.prio; }  // min-heap (Priority reverses the order, common.rs:235-239)
};

static inline bool node_valid_in_world(const PTOGraph& g, size_t id, int world) {
  return world < 0 || g.validities[g.nodes[id].validity_id][(size_t)world];
}

std::vector<double> dijkstra(const PTOGraph& g, int world, const std::vector<size_t>& finals) {
  std::vector<double> dist(g.nodes.size(), INF);
  std::priority_queue<HeapItem> q;
  for (size_t id : finals) { dist[id] = 0.0; q.push({0.0, id}); }
  while (!q.empty()) {
    HeapItem it = q.top();
    q.pop();
    size_t v = it.id;
    for (const PTOEdge& e : g.nodes[v].parents) {
      size_t u = e.id;
      if (!node_valid_in_world(g, u, world)) continue;  // PTOGraphWorldView::parents, pto_graph.rs:264-270
      double alt = dist[v] + norm2(g.nodes[u].state, g.nodes[v].state);
      if (alt < dist[u]) { dist[u] = alt; q.push({alt, u}); }
    }
  }
  return dist;
}

std::vector<State> extract_path(const PTOGraph& g, int world, size_t start, const std::vector<double>& costs) {
  std::vector<State> path;
  size_t node_id = start;
  path.push_back(g.nodes[node_id].state);
  while (costs[node_id] != 0.0) {
    bool found = false;
    size_t best = 0;
    double best_c = 0.0;
    for (const PTOEdge& e : g.nodes[node_id].parents) {   // sic: the reference walks `parents`
      if (!node_valid_in_world(g, e.id, world)) continue;
      double c = costs[e.id] + norm2(g.nodes[e.id].state, g.nodes[node_id].state);
      if (!found || c < best_c) { found = true; best = e.id; best_c = c; }  // Iterator::min_by keeps the first minimum
    }
    if (!found) break;  // reference: unwrap() panic on an empty parent list
    node_id = best;
    path.push_back(g.nodes[node_id].state);
  }
  return path;
}

// ============================================================== reachability
void Reachability::set_root(const WorldMask& v) {
  n_worlds = v.size();
  validities.push_back(v);
  reachabilities.push_back(v);
  finality.assign(n_worlds, 0);
}
void Reachability::add_node(const WorldMask& v) {
  validities.push_back(v);
  reachabilities.push_back(WorldMask(v.size(), 0));
}
void Reachability::add_final_node(size_t id, const WorldMask& f) {
  final_node_ids.push_back(id);
  final_set.insert(id);
  finalities.push_back(f);
  dirty = true;
}
void Reachability::add_edge(size_t from, size_t to, const WorldMask& ev) {
  for (size_t i = 0; i < reachabilities[to].size(); ++i) {
    bool r_to = reachabilities[to][i], r_from = reachabilities[from][i], v = ev[i];
    reachabilities[to][i] = r_to || (r_from && v);
    if (final_set.count(to)) dirty = true;
  }
}
std::vector<size_t> Reachability::get_final_nodes_for_world(size_t world) const {
  std::vector<size_t> out;
  for (size_t i = 0; i < final_node_ids.size(); ++i) {
    size_t id = final_node_ids[i];
    if (reachabilities[id][world] && finalities[i][world]) out.push_back(id);
  }
  return out;
}
bool Reachability::is_final_set_complete() {
  if (final_node_ids.empty()) return false;
  if (dirty) {
    for (size_t k = 0; k < final_node_ids.size(); ++k) {
      const WorldMask& r = reachabilities[final_node_ids[k]];
      for (size_t i = 0; i < r.size(); ++i) finality[i] = finality[i] || (r[i] && finalities[k][i]);
    }
    dirty = false;
  }
  for (uint8_t b : finality)
    if (!b) return false;
  return true;
}

// ============================================================== goals
bool SquareGoal::init(const std::vector<std::pair<State, WorldMask>>& g, double md) {
  if (g.empty()) return false;
  goal_to_validity = g;
  max_dist = md;
  size_t nw = g[0].second.size();
  world_to_goal.assign(nw, State{0.0, 0.0});
  std::vector<bool> has(nw, false);
  for (size_t w = 0; w < nw; ++w)
    for (const auto& gv : g)
      if (gv.second[w]) {
        if (has[w]) return false;  // assert: validities shouldn't overlap (common.rs:320)
        world_to_goal[w] = gv.first;
        has[w] = true;
      }
  return true;
}
bool SquareGoal::goal(const State& s, WorldMask* out) const {
  for (const auto& gv : goal_to_validity)
    if (norm1(s, gv.first) < max_dist) { *out = gv.second; return true; }
  return false;
}

// ============================================================== belief graph DP
bool conditional_dijkstra(const BeliefGraph& g, const std::vector<size_t>& finals, std::vector<double>& dist) {
  dist.assign(g.nodes.size(), INF);
  std::priority_queue<HeapItem> q;
  for (size_t id : finals) { dist[id] = 0.0; q.push({0.0, id}); }
  while (!q.empty()) {
    HeapItem it = q.top();
    q.pop();
    size_t v_id = it.id;
    for (size_t u_id : g.nodes[v_id].parents) {
      const BeliefNode& u = g.nodes[u_id];
      double alt = 0.0;
      if (u.node_type == ACTION) {
        alt += norm2(u.state, g.nodes[v_id].state) + dist[v_id];
      } else if (u.node_type == OBSERVATION) {
        for (size_t vv_id : u.children) {
          const BeliefNode& vv = g.nodes[vv_id];
          double p = transition_probability(g.belief_state(u_id), g.belief_state(vv_id));
          if (!(p > 0.0)) return false;  // assert!(p > 0.0), belief_graph.rs:130
          alt += p * (norm2(u.state, vv.state) + dist[vv_id]);
        }
      } else {
        return false;  // panic "node type should be know at this stage!"
      }
      if (alt < dist[u_id]) { dist[u_id] = alt; q.push({alt, u_id}); }
    }
  }
  return true;
}

static bool best_expected_children(const BeliefGraph& g, size_t node_id, const std::vector<double>& costs,
                                   std::vector<size_t>& best_children) {
  struct C { size_t child_id; double cost_to_child, expected_from_child; };
  std::map<size_t, std::vector<C>> by_belief;  // BTreeMap: ascending belief_id
  const BeliefNode& n = g.nodes[node_id];
  for (size_t child_id : n.children) {
    const BeliefNode& c = g.nodes[child_id];
    by_belief[c.belief_id].push_back({child_id, norm2(n.state, c.state), costs[child_id]});
  }
  best_children.clear();
  for (auto& kv : by_belief) {
    size_t best_id = kv.second[0].child_id;
    double p = transition_probability(g.belief_state(node_id), g.belief_state(best_id));
    if (!(p > 0.0)) return false;
    double best_cost = INF;
    for (const C& c : kv.second) {
      double cost = p * (c.cost_to_child + c.expected_from_child);
      if (cost < best_cost) { best_cost = cost; best_id = c.child_id; }
    }
    if (!(p * costs[best_id] <= costs[node_id])) return false;  // assert, belief_graph.rs:261
    best_children.push_back(best_id);
  }
  return true;
}

bool extract_policy(const BeliefGraph& g, const std::vector<double>& costs, Policy& policy) {
  if (g.nodes.empty()) return false;
  policy = Policy();
  std::vector<std::pair<size_t, size_t>> lifo;
  policy.nodes.push_back({g.nodes[0].state, g.nodes[0].belief_id, -1, {}, 0});
  lifo.push_back({0, 0});
  std::vector<size_t> children;
  while (!lifo.empty()) {
    std::pair<size_t, size_t> top = lifo.back();
    lifo.pop_back();
    if (!best_expected_children(g, top.second, costs, children)) return false;
    for (size_t child_id : children) {
      bool is_leaf = costs[child_id] == 0.0;
      size_t pid = policy.nodes.size();
      policy.nodes.push_back({g.nodes[child_id].state, g.nodes[child_id].belief_id, (int64_t)top.first, {}, child_id});
      if (is_leaf) policy.leafs.push_back(pid);
      policy.nodes[top.first].children.push_back(pid);
      if (!is_leaf) lifo.push_back({pid, child_id});
    }
    // (test infrastructure only: where the costs are infinite -- a start from which some world's goal cannot be reached -- the
    // reference's walk never ends and allocates until it dies; the checker reports that as "would not return" instead)
    if (policy.nodes.size() > 64 * g.nodes.size() + 1024) return false;
  }
  policy.expected_costs = costs[0];
  return true;
}

// ============================================================== PRM
PRM::PRM(const GridMap* m, State low, State up, uint64_t seed)
    : fns(m), sampler(low, up, seed), kdtree(State{0.0, 0.0}) {
  graph.validities = m->world_validities;
}
void PRM::init(State start) {
  graph.add_node(start, 0);
  kdtree.reset(start);
}
void PRM::grow_graph(double max_step, double search_radius, size_t n_iter) {
  for (size_t i = 0; i < n_iter; ++i) {
    State s = sampler.sample();
    add_sample(s, max_step, search_radius);
    n_it += 1;
  }
}
size_t PRM::add_sample(State s, double max_step, double search_radius) {
  if (graph.nodes.empty()) {
    graph.add_node(s, 0);
    kdtree.reset(s);
    return 0;
  }
  size_t new_id = graph.add_node(s, 0);
  double radius = heuristic_radius(graph.nodes.size(), max_step, search_radius, 2);
  std::vector<size_t> neighbours;
  for (const KdTree::Node* n : kdtree.nearest_neighbors(s, radius)) neighbours.push_back(n->id);
  kdtree.add(s, new_id);
  if (neighbours.empty()) return new_id;
  std::vector<size_t> edges;
  for (size_t id : neighbours)
    if (fns->transition_validator(graph.nodes[id].state, graph.nodes[new_id].state) >= 0) edges.push_back(id);
  for (size_t id : edges) graph.add_edge(id, new_id, 0);
  for (size_t id : edges) graph.add_edge(new_id, id, 0);
  return new_id;
}
std::vector<State> PRM::plan_path(State start, State goal) {
  size_t s = kdtree.nearest_neighbor(start).id, gl = kdtree.nearest_neighbor(goal).id;
  std::vector<double> cost = dijkstra(graph, -1, {gl});
  if (std::isinf(cost[s])) return {};
  return extract_path(graph, -1, s, cost);
}

// ============================================================== PTO
PTO::PTO(const GridMap* m, State low, State up, uint64_t seed)
    : fns(m), continuous(low, up, seed), discrete(seed), kdtree(State{0.0, 0.0}), n_worlds(m->n_worlds) {
  graph.validities = m->world_validities;
}

int PTO::grow_graph(State start, const SquareGoal& goal, double max_step, double search_radius,
                    size_t n_iter_min, size_t n_iter_max) {
  int64_t root_vid = fns->state_validity(start);
  if (root_vid < 0) return root_vid == NONE ? -100 : (int)root_vid;  // expect("Start from a valid state!")
  graph.add_node(start, (size_t)root_vid);
  reach.set_root(graph.validities[(size_t)root_vid]);
  kdtree.reset(start);
  if (hooks.add_vertex) hooks.add_vertex(hooks.user, start.data(), 0);
  size_t i = 0;
  std::vector<uint64_t> reach_words;
  std::vector<int64_t> hook_ids;
  while (i < n_iter_min || (!reach.is_final_set_complete() && i < n_iter_max)) {
    i += 1;
    // sample(), pto.rs:141-149
    size_t world = discrete.sample(n_worlds);
    State new_state = (i % 100 == 0) ? goal.goal_example(world) : continuous.sample();
    State from_state;
    size_t from_id;
    if (hooks.nearest_filtered) {
      const size_t V = graph.nodes.size(), words = (n_worlds + 63) / 64;
      reach_words.assign(V * words, 0);
      for (size_t id = 0; id < V; ++id)
        for (size_t w = 0; w < n_worlds; ++w)
          if (reach.reachabilities[id][w]) reach_words[id * words + w / 64] |= 1ull << (w % 64);
      int64_t id = hooks.nearest_filtered(hooks.user, new_state.data(), world, reach_words.data(), V, words);
      if (id < 0 || (size_t)id >= V) return -101;
      from_id = (size_t)id; from_state = graph.nodes[from_id].state;
    } else {
      const KdTree::Node& kd_from = nn_filtered(kdtree, new_state, [&](size_t id) { return reach.reachabilities[id][world] != 0; });
      from_state = kd_from.state; from_id = kd_from.id;
    }
    steer(from_state, new_state, max_step);
    int64_t svid = hooks.state_validity ? hooks.state_validity(hooks.user, new_state.data()) : fns->state_validity(new_state);
    if (svid < NONE) return (int)svid;
    if (svid >= 0) {
      size_t new_id = graph.add_node(new_state, (size_t)svid);
      reach.add_node(graph.validities[(size_t)svid]);
      double radius = heuristic_radius(graph.nodes.size(), max_step, search_radius, 2);
      std::vector<size_t> neighbours;
      if (hooks.radius) {
        hook_ids.resize(graph.nodes.size());
        int64_t cnt = hooks.radius(hooks.user, new_state.data(), radius, hook_ids.data(), (int64_t)hook_ids.size());
        if (cnt < 0 || cnt > (int64_t)hook_ids.size()) return -102;
        for (int64_t k = 0; k < cnt; ++k) neighbours.push_back((size_t)hook_ids[k]);
      } else {
        for (const KdTree::Node* n : kdtree.nearest_neighbors(new_state, radius)) neighbours.push_back(n->id);
      }
      if (neighbours.empty()) neighbours.push_back(from_id);
      std::vector<std::pair<size_t, size_t>> edges;
      std::vector<int64_t> vids(neighbours.size());
      if (hooks.edges) {
        std::vector<double> fr(2 * neighbours.size()), to(2 * neighbours.size());
        for (size_t k = 0; k < neighbours.size(); ++k) {
          fr[2 * k] = graph.nodes[neighbours[k]].state[0]; fr[2 * k + 1] = graph.nodes[neighbours[k]].state[1];
          to[2 * k] = new_state[0]; to[2 * k + 1] = new_state[1];
        }
        hooks.edges(hooks.user, fr.data(), to.data(), (int64_t)neighbours.size(), vids.data());
      } else {
        for (size_t k = 0; k < neighbours.size(); ++k) vids[k] = fns->transition_validator(graph.nodes[neighbours[k]].state, graph.nodes[new_id].state);
      }
      for (size_t k = 0; k < neighbours.size(); ++k) {
        int64_t v = vids[k];
        if (v < NONE) return (int)v;     // (the reference panics at the first offending edge; any of them fails the call here)
        if (v >= 0) edges.push_back({neighbours[k], (size_t)v});
      }
      for (auto& e : edges) {
        reach.add_edge(e.first, new_id, graph.validities[e.second]);
        graph.add_edge(e.first, new_id, e.second);
      }
      for (auto& e : edges) {
        reach.add_edge(new_id, e.first, graph.validities[e.second]);
        graph.add_edge(new_id, e.first, e.second);
      }
      WorldMask finality;
      if (goal.goal(new_state, &finality)) reach.add_final_node(new_id, finality);
      kdtree.add(new_state, new_id);
      if (hooks.add_vertex) hooks.add_vertex(hooks.user, new_state.data(), new_id);
    }
  }
  n_it = i;
  return reach.is_final_set_complete() ? 0 : 1;
}

bool PTO::build_belief_graph(const BeliefState& b0) {  // pto.rs:185-259
  std::vector<BeliefState> beliefs = fns->reachable_belief_states(b0);
  const std::vector<WorldMask>& wv = graph.validities;
  size_t B = beliefs.size(), V = graph.nodes.size();
  std::vector<std::vector<bool>> compat(B, std::vector<bool>(wv.size(), false));  // compute_compatibility, common.rs:266-276
  for (size_t b = 0; b < B; ++b)
    for (size_t v = 0; v < wv.size(); ++v) compat[b][v] = is_compatible(beliefs[b], wv[v]);
  belief_graph = BeliefGraph();
  belief_graph.reachable_belief_states = beliefs;
  for (size_t b = 0; b < B; ++b) belief_graph.belief_states_to_id[belief_hash(beliefs[b])] = b;
  if (belief_graph.belief_states_to_id.size() != B) return false;  // "collision when hashing the belief states!"
  node_to_belief_nodes.assign(V, std::vector<int64_t>(B, -1));
  for (size_t id = 0; id < V; ++id)
    for (size_t b = 0; b < B; ++b) {
      size_t bn = belief_graph.add_node(graph.nodes[id].state, b, UNKNOWN);
      if (compat[b][graph.nodes[id].validity_id]) node_to_belief_nodes[id][b] = (int64_t)bn;
    }
  std::vector<BeliefState> children;
  for (size_t id = 0; id < V; ++id)
    for (size_t b = 0; b < B; ++b) {
      if (!fns->observe(graph.nodes[id].state, beliefs[b], children, &panic)) return false;
      int64_t parent = node_to_belief_nodes[id][b];
      for (const BeliefState& cb : children) {
        if (belief_hash(beliefs[b]) != belief_hash(cb)) {
          auto it = belief_graph.belief_states_to_id.find(belief_hash(cb));
          if (it == belief_graph.belief_states_to_id.end()) return false;  // panic "no if corresponding to this belief state!"
          int64_t child = node_to_belief_nodes[id][it->second];
          if (parent >= 0 && child >= 0) {
            belief_graph.nodes[(size_t)parent].node_type = OBSERVATION;
            belief_graph.add_edge((size_t)parent, (size_t)child);
          }
        }
      }
    }
  for (size_t id = 0; id < V; ++id)
    for (size_t b = 0; b < B; ++b) {
      int64_t parent = node_to_belief_nodes[id][b];
      if (parent < 0) continue;
      if (belief_graph.nodes[(size_t)parent].node_type == OBSERVATION) continue;
      for (const PTOEdge& ce : graph.nodes[id].children) {
        int64_t child = node_to_belief_nodes[ce.id][b];
        if (child < 0) continue;
        if (compat[belief_graph.nodes[(size_t)parent].belief_id][ce.validity_id]) {
          belief_graph.nodes[(size_t)parent].node_type = ACTION;
          belief_graph.add_edge((size_t)parent, (size_t)child);
        }
      }
    }
  return true;
}

bool PTO::compute_expected_costs_to_goals() {  // pto.rs:261-275
  final_belief_nodes.clear();
  for (size_t k = 0; k < reach.final_node_ids.size(); ++k) {
    size_t final_id = reach.final_node_ids[k];
    for (int64_t bn : node_to_belief_nodes[final_id]) {
      if (bn < 0) continue;
      if (is_compatible(belief_graph.belief_state((size_t)bn), reach.finalities[k])) final_belief_nodes.push_back((size_t)bn);
    }
  }
  return conditional_dijkstra(belief_graph, final_belief_nodes, expected_costs);
}

int PTO::plan_qmdp() {  // qmdp_policy_extractor.rs:23-35
  cost_to_goals.assign(n_worlds, {});
  for (size_t w = 0; w < n_worlds; ++w) {
    std::vector<size_t> finals = reach.get_final_nodes_for_world(w);
    if (finals.empty()) return 1;
    cost_to_goals[w] = dijkstra(graph, (int)w, finals);
  }
  return 0;
}

bool PTO::react_qmdp(State start, const BeliefState& belief, double horizon, std::vector<std::vector<State>>& paths) {
  // qmdp_policy_extractor.rs:38-123
  if (belief.size() != n_worlds) return false;
  size_t id = kdtree.nearest_neighbor(start).id;
  std::vector<State> common;
  double smallest = INF, acc = 0.0;
  size_t guard = 0;
  while (acc < horizon && smallest > 0.0) {
    common.push_back(graph.nodes[id].state);
    size_t best = 0;
    double best_c = INF;
    for (const PTOEdge& ce : graph.nodes[id].children) {
      double c = 0.0;
      for (size_t w = 0; w < n_worlds; ++w) c += cost_to_goals[w][ce.id] * belief[w];
      if (c < best_c) { best = ce.id; best_c = c; }
    }
    acc += norm2(graph.nodes[id].state, graph.nodes[best].state);
    id = best;
    smallest = best_c;
    if (++guard > 10 * graph.nodes.size() + 10) return false;  // the reference would loop forever
  }
  paths.assign(n_worlds, {});
  for (size_t w = 0; w < n_worlds; ++w) {
    paths[w] = common;
    size_t cur = id;
    guard = 0;
    while (cost_to_goals[w][cur] > 0.0) {
      paths[w].push_back(graph.nodes[cur].state);
      size_t best = 0;
      double smaller = INF;
      for (const PTOEdge& ce : graph.nodes[cur].children)
        if (cost_to_goals[w][ce.id] < smaller) { smaller = cost_to_goals[w][ce.id]; best = ce.id; }
      cur = best;
      if (++guard > 10 * graph.nodes.size() + 10) return false;
    }
  }
  return true;
}

// ============================================================== pto_policy_refiner.rs (partial shortcut)
int64_t refiner_is_transition_valid(const GridMap& m, const State& from, const State& to, const std::vector<bool>& compat_row) {
  const int64_t fv = m.state_validity(from);       // :396
  if (fv < -1) return fv;
  const int64_t tv = m.state_validity(to);         // :397
  if (tv < -1) return tv;
  if (fv < 0 || tv < 0) return 0;                  // :399 `if let (Some, Some)` ... else false
  const int64_t v = m.transition_validator(from, to);   // :414
  if (v < -1) return v;
  if (v < 0) return 0;                             // None => false (:418)
  return compat_row[(size_t)v] ? 1 : 0;            // :417
}

int64_t refiner_partial_shortcut(const GridMap& m, std::vector<State>& states, const std::vector<bool>& compat_row, size_t n_iterations, uint64_t seed) {
  auto interpolate = [](double a, double b, double lambda) { return a * (1.0 - lambda) + b * lambda; };   // :159-161
  if (states.size() <= 2) return 0;                // :163-165
  const size_t joint_dim = 2;                      // tree.nodes.first().state.len()
  DiscreteSampler sampler(seed);                   // :169 DiscreteSampler::new() (seed 0)
  int64_t commits = 0;
  for (size_t it = 0; it < n_iterations; ++it) {
    const size_t joint = (size_t)sampler.sample(joint_dim);                                   // :172
    const size_t a = (size_t)sampler.sample(states.size() - 2);                               // :173
    const size_t b = a + 2 + (size_t)sampler.sample(states.size() - a - 2);                   // :174
    const State sa = states[a], sb = states[b];
    std::vector<State> sc;                                                                    // :182-190
    for (size_t j = a; j < b; ++j) {
      const double lambda = (double)(j - a) / (double)(b - a);
      State s = states[j];
      s[joint] = interpolate(sa[joint], sb[joint], lambda);
      sc.push_back(s);
    }
    bool should_commit = true;                                                                // :193-197 (short-circuit `&&`)
    for (size_t k = 0; k + 1 < sc.size(); ++k) {
      if (!should_commit) break;
      const int64_t r = refiner_is_transition_valid(m, sc[k], sc[k + 1], compat_row);
      if (r < 0) return r;
      should_commit = r == 1;
    }
    if (should_commit) {
      const int64_t r = refiner_is_transition_valid(m, sc.back(), sb, compat_row);
      if (r < 0) return r;
      should_commit = r == 1;
    }
    if (should_commit) {                                                                      // :200-204
      for (size_t j = a; j < b; ++j) states[j] = sc[j - a];
      ++commits;
    }
  }
  return commits;
}

// Policy::decompose (common.rs:85-129)
void policy_decompose(const Policy& p, std::vector<std::pair<size_t, std::vector<size_t>>>& pieces, std::vector<std::vector<size_t>>& skeleton) {
  pieces.clear(); skeleton.clear();
  size_t n_pieces = 0;
  std::deque<size_t> fifo;
  fifo.push_back(0);                                                 // :91
  while (!fifo.empty()) {
    const size_t id = fifo.front(); fifo.pop_front();                // :94
    std::vector<size_t> ids, successors;
    size_t current_id = id;
    for (;;) {
      ids.push_back(current_id);                                     // :103 (the assert_eq on the belief states, :101, is a debug check)
      const auto& ch = p.nodes[current_id].children;
      if (ch.empty()) break;                                         // :106 final node
      if (ch.size() == 1) { current_id = ch[0]; continue; }          // :107 simple forward
      for (size_t child_id : ch) {                                   // :108-114 branching
        fifo.push_back(child_id);
        n_pieces += 1;
        successors.push_back(n_pieces);
      }
      break;
    }
    pieces.push_back({p.nodes[id].belief_id, ids});                  // :119-124
    skeleton.push_back(successors);
  }
}

// Policy::compute_expected_costs_to_goals_from (common.rs:135-153)
static double policy_expected_from(const Policy& p, const BeliefGraph& g, double prob, size_t id) {
  double expected_future_costs = 0.0;
  const PolicyNode& node = p.nodes[id];
  for (size_t child_id : node.children) {
    const PolicyNode& child = p.nodes[child_id];
    const double q = transition_probability(g.reachable_belief_states[node.belief_id], g.reachable_belief_states[child.belief_id]);
    const double cost = norm2(node.state, child.state);
    expected_future_costs += prob * q * cost + policy_expected_from(p, g, prob * q, child_id);   // :149
  }
  return expected_future_costs;
}
double policy_expected_costs(const Policy& p, const BeliefGraph& g) { return policy_expected_from(p, g, 1.0, 0); }

namespace {
struct TreeNode { State state; int64_t parent; size_t belief_graph_id; double parent_cost = 0.0; };   // RefinmentNode :33-38 (parent: Option<Edge{id, cost}>)
struct Tree {                                                                                          // RefinmentTree :40-63
  std::vector<TreeNode> nodes; size_t belief_state_id = 0, leaf = 0;
  double dist_from_root(size_t id) const {                                                             // :53-62: summed from the node upwards
    double cost = 0.0;
    for (size_t k = id; nodes[k].parent >= 0; k = (size_t)nodes[k].parent) cost += nodes[k].parent_cost;
    return cost;
  }
};
std::vector<std::vector<bool>> refiner_compat(const GridMap& m, const BeliefGraph& g) {                // refiner :79, common.rs:266-276
  std::vector<std::vector<bool>> compat(g.reachable_belief_states.size(), std::vector<bool>(m.world_validities.size(), false));
  for (size_t b = 0; b < compat.size(); ++b)
    for (size_t v = 0; v < m.world_validities.size(); ++v) compat[b][v] = is_compatible(g.reachable_belief_states[b], m.world_validities[v]);
  return compat;
}
void refiner_recompose(const std::vector<Tree>& trees, const std::vector<std::vector<size_t>>& skeleton, const BeliefGraph& g, Policy& out);
}  // namespace

bool refiner_refine_shortcut(const GridMap& m, const Policy& policy, const BeliefGraph& g, size_t n_iterations, Policy& out, uint64_t seed) {
  const std::vector<std::vector<bool>> compat = refiner_compat(m, g);
  std::vector<std::pair<size_t, std::vector<size_t>>> path_pieces;
  std::vector<std::vector<size_t>> skeleton;
  policy_decompose(policy, path_pieces, skeleton);                                                                     // :94
  std::vector<Tree> trees;
  for (const auto& piece : path_pieces) {                                                                               // :97
    const std::vector<size_t>& path = piece.second;
    Tree tree;                                                                                                         // build_path_piece :136-156
    const size_t root_bg = policy.nodes[path.front()].original_node_id;
    tree.nodes.push_back({g.nodes[root_bg].state, -1, root_bg, 0.0});
    for (size_t k = 0; k + 1 < path.size(); ++k) {
      const size_t next_bg = policy.nodes[path[k + 1]].original_node_id;
      tree.nodes.push_back({g.nodes[next_bg].state, (int64_t)tree.nodes.size() - 1, next_bg, 0.0});
    }
    tree.belief_state_id = g.nodes[root_bg].belief_id;
    tree.leaf = tree.nodes.size() - 1;
    std::vector<State> states;                                                                                         // partial_shortcut :158-206
    for (const TreeNode& n : tree.nodes) states.push_back(n.state);
    if (refiner_partial_shortcut(m, states, compat[tree.belief_state_id], n_iterations, seed) < 0) return false;
    for (size_t k = 0; k < states.size(); ++k) tree.nodes[k].state = states[k];
    trees.push_back(tree);
  }
  refiner_recompose(trees, skeleton, g, out);
  return true;
}

namespace {
// recompose :324-393
void refiner_recompose(const std::vector<Tree>& trees, const std::vector<std::vector<size_t>>& skeleton, const BeliefGraph& g, Policy& out) {
  out = Policy();
  const int64_t NONE = -1;
  std::vector<std::pair<int64_t, int64_t>> pieces_start_end(skeleton.size(), {NONE, NONE});
  auto add_node = [&](const State& s, size_t belief_graph_id) {
    out.nodes.push_back({s, g.nodes[belief_graph_id].belief_id, -1, {}, belief_graph_id});
    return (int64_t)out.nodes.size() - 1;
  };
  auto add_edge = [&](int64_t parent, int64_t child) { out.nodes[(size_t)parent].children.push_back((size_t)child); out.nodes[(size_t)child].parent = parent; };
  for (size_t i = 0; i < trees.size(); ++i) {
    const Tree& tree = trees[i];
    std::vector<const TreeNode*> node_path;                                                                            // :337-345
    const TreeNode* node = &tree.nodes[tree.leaf];
    node_path.push_back(node);
    while (node->parent >= 0) { node = &tree.nodes[(size_t)node->parent]; node_path.push_back(node); }
    std::reverse(node_path.begin(), node_path.end());
    int64_t previous_id = NONE;
    for (size_t j = 0; j < node_path.size(); ++j) {                                                                    // :348-367
      const bool is_start = j == 0, is_end = j == node_path.size() - 1;
      const int64_t id = add_node(node_path[j]->state, node_path[j]->belief_graph_id);
      if (is_start) pieces_start_end[i].first = id;                // (a one-node piece is a start only: its end stays None)
      else if (is_end) { add_edge(previous_id, id); pieces_start_end[i].second = id; }
      else add_edge(previous_id, id);
      previous_id = id;
    }
  }
  for (size_t i = 0; i < skeleton.size(); ++i) {                                                                       // :371-381
    const int64_t from_end = pieces_start_end[i].second;
    for (size_t next_piece : skeleton[i]) {
      const int64_t to_start = pieces_start_end[next_piece].first;
      if (from_end != NONE && to_start != NONE) add_edge(from_end, to_start);
    }
  }
  for (size_t i = 0; i < out.nodes.size(); ++i)                                                                        // :384-389
    if (out.nodes[i].children.empty()) out.leafs.push_back(i);
  out.expected_costs = policy_expected_costs(out, g);                                                                  // :391
}

// priority-queue 1.0.5 `PriorityQueue<usize, Priority>` as the refiner uses it (push / pop / is_empty), restated from the crate's
// published algorithm (the crate is a crates.io dependency, Cargo.toml:18, not vendored): an indexed binary heap -- `heap` holds
// item slots, a NEW item is appended and bubbles up while `parent < new`, an item pushed AGAIN gets its priority replaced, bubbles up
// by the same rule and is then sifted down (`heapify`), pop moves the LAST heap entry to the root and sifts it down, looking at the
// left child first and preferring a child only when it is strictly `>`.  Priority's Ord (common.rs:231-251) never says Equal:
// a.cmp(b) = Greater iff a.prio < b.prio, else Less -- so `a < b` means !(a.prio < b.prio) and `a > b` means a.prio < b.prio, which is
// what decides the order among equal priorities.  PARITY UNPINNED: no test of the reference fixes this order.
struct RefPriorityQueue {
  std::vector<size_t> heap;            // item ids
  std::vector<int64_t> pos;            // item id -> heap position, -1 = not queued
  std::vector<double> prio;
  explicit RefPriorityQueue(size_t n_items) : pos(n_items, -1), prio(n_items, 0.0) {}
  static bool lt(double a, double b) { return !(a < b); }   // Priority{a} < Priority{b}
  static bool gt(double a, double b) { return a < b; }      // Priority{a} > Priority{b}
  bool empty() const { return heap.empty(); }
  void bubble_up(size_t i, size_t item) {
    while (i > 0 && lt(prio[heap[(i - 1) / 2]], prio[item])) {
      heap[i] = heap[(i - 1) / 2]; pos[heap[i]] = (int64_t)i;
      i = (i - 1) / 2;
    }
    heap[i] = item; pos[item] = (int64_t)i;
  }
  void heapify(size_t i) {
    for (;;) {
      const size_t l = 2 * i + 1, r = 2 * i + 2;
      size_t largest = (l < heap.size() && gt(prio[heap[l]], prio[heap[i]])) ? l : i;
      if (r < heap.size() && gt(prio[heap[r]], prio[heap[largest]])) largest = r;
      if (largest == i) return;
      std::swap(heap[i], heap[largest]);
      pos[heap[i]] = (int64_t)i; pos[heap[largest]] = (int64_t)largest;
      i = largest;
    }
  }
  void push(size_t item, double p) {
    prio[item] = p;
    if (pos[item] >= 0) {                      // already queued: change_priority
      const size_t at = (size_t)pos[item];
      bubble_up(at, item);
      heapify((size_t)pos[item]);
      return;
    }
    heap.push_back(item);
    bubble_up(heap.size() - 1, item);
  }
  size_t pop() {
    const size_t head = heap[0];
    pos[head] = -1;
    heap[0] = heap.back();
    heap.pop_back();
    if (!heap.empty()) { pos[heap[0]] = 0; heapify(0); }
    return head;
  }
};
}  // namespace

// PTOPolicyRefiner::refine_solution(RefinmentStrategy::Reparent(radius)) (pto_policy_refiner.rs:85-133): per path piece build_tree
// (:208-280) and reparent with half the radius (:282-322), then recompose.
bool refiner_refine_reparent(const GridMap& m, const Policy& policy, const BeliefGraph& g, double radius, Policy& out) {
  const std::vector<std::vector<bool>> compat = refiner_compat(m, g);
  std::vector<std::pair<size_t, std::vector<size_t>>> path_pieces;
  std::vector<std::vector<size_t>> skeleton;
  policy_decompose(policy, path_pieces, skeleton);
  std::vector<Tree> trees;
  for (const auto& piece : path_pieces) {
    const std::vector<size_t>& path = piece.second;
    // ---- build_tree :209-280
    std::unordered_set<size_t> visited;
    Tree tree;
    const size_t root_bg = policy.nodes[path.front()].original_node_id;
    tree.nodes.push_back({g.nodes[root_bg].state, -1, root_bg, 0.0});
    KdTree kdtree(g.nodes[root_bg].state);
    visited.insert(root_bg);
    for (size_t k = 0; k + 1 < path.size(); ++k) {                                           // :227-242
      const size_t prev_bg = policy.nodes[path[k]].original_node_id, next_bg = policy.nodes[path[k + 1]].original_node_id;
      tree.nodes.push_back({g.nodes[next_bg].state, (int64_t)tree.nodes.size() - 1, next_bg, norm2(g.nodes[prev_bg].state, g.nodes[next_bg].state)});
      kdtree.add(g.nodes[next_bg].state, tree.nodes.size() - 1);
      visited.insert(next_bg);
    }
    tree.belief_state_id = g.nodes[root_bg].belief_id;
    tree.leaf = tree.nodes.size() - 1;
    const std::vector<TreeNode> nodes = tree.nodes;                                          // :247 clone: only the path nodes seed the search
    for (size_t node_id = 0; node_id < nodes.size(); ++node_id) {                            // :248-277
      const TreeNode& node = nodes[node_id];
      std::deque<std::pair<size_t, size_t>> q;
      q.push_back({node_id, node.belief_graph_id});
      while (!q.empty()) {
        const std::pair<size_t, size_t> top = q.front(); q.pop_front();
        const size_t tree_id = top.first;
        for (size_t child_id : g.nodes[top.second].children) {
          const BeliefNode& child = g.nodes[child_id];
          if (!visited.count(child_id) && norm2(node.state, child.state) <= radius) {        // distance to the SEED node of the search
            tree.nodes.push_back({child.state, (int64_t)tree_id, child_id, norm2(node.state, child.state)});   // (cost from the seed too, :259-262)
            const size_t new_tree_id = tree.nodes.size() - 1;
            kdtree.add(child.state, new_tree_id);
            visited.insert(child_id);
            for (size_t cc : child.children)
              if (!visited.count(cc)) q.push_back({new_tree_id, cc});                        // :268-272: the CHILDREN of cc are looked at next
          }
        }
      }
    }
    // ---- reparent :282-322 with radius / 2
    {
      const double r2 = 0.5 * radius;
      RefPriorityQueue q(tree.nodes.size());
      for (size_t id = 0; id < tree.nodes.size(); ++id) q.push(id, tree.dist_from_root(id));
      while (!q.empty()) {
        const size_t node_id = q.pop();
        const State node_state = tree.nodes[node_id].state;
        std::vector<size_t> neighbor_ids;
        for (const KdTree::Node* kn : kdtree.nearest_neighbors(node_state, r2)) {
          const int64_t ok = refiner_is_transition_valid(m, node_state, kn->state, compat[tree.belief_state_id]);
          if (ok < 0) return false;
          if (ok) neighbor_ids.push_back(kn->id);
        }
        const double distance_from_root = tree.dist_from_root(node_id);
        std::vector<std::pair<size_t, double>> nd;
        for (size_t id : neighbor_ids) nd.push_back({id, tree.dist_from_root(id)});          // all read BEFORE any reparenting of this pop
        for (const auto& kv : nd) {
          const double cost = norm2(node_state, tree.nodes[kv.first].state);
          if (distance_from_root + cost < kv.second) {
            tree.nodes[kv.first].parent = (int64_t)node_id;
            tree.nodes[kv.first].parent_cost = cost;
            q.push(kv.first, distance_from_root + cost);
          }
        }
      }
    }
    trees.push_back(tree);
  }
  refiner_recompose(trees, skeleton, g, out);
  return true;
}

// ============================================================== map_shelves_tamp_prm.rs
static bool tamp_is_final(const BeliefState& b) {  // :19-21
  double m = b[0];
  for (double p : b) if (p > m) m = p;
  return m >= 0.999;
}
static BeliefState tamp_normalize(const BeliefState& b) {  // :23-26 (map_shelves_tamp_rrt.rs:15-18)
  double sum = 0.0;
  for (double p : b) sum = sum + p;
  BeliefState out;
  for (double p : b) out.push_back(p / sum);
  return out;
}
size_t TampPRM::Mode::add_sample(State s, double max_step, double search_radius) {
  samples.push_back(s); max_steps.push_back(max_step); search_radii.push_back(search_radius);
  return prm.add_sample(s, max_step, search_radius);
}
TampPRM::TampPRM(const GridMap* m, State low, State up, uint64_t seed)
    : domain(m), continuous(low, up, seed), zone_sampler({0.0, 0.0}, {m->visibility_distance, 2.0 * M_PI}, seed), discrete(seed) {}
size_t TampPRM::add_mode(const std::vector<size_t>& remaining, double reaching_p, const BeliefState& b) {
  size_t id = modes.size();
  modes.emplace_back(new Mode(domain, continuous));   // PRM::new(continuous_sampler.clone(), ..): every mode starts the same stream
  Mode& v = *modes.back();
  v.id = id; v.remaining_zones = remaining; v.reaching_probability = reaching_p; v.belief_state = b;
  mode_hash_map[belief_hash(b)] = id;
  return id;
}
std::vector<size_t> TampPRM::get_transitions(size_t mode_id, size_t target_zone_id) {
  std::vector<size_t> successor;
  if (tamp_is_final(modes[mode_id]->belief_state)) return successor;
  auto remaining_without = [&](const Mode& m) {
    std::vector<size_t> r;
    for (size_t z : m.remaining_zones) if (z != target_zone_id) r.push_back(z);
    return r;
  };
  {  // object there (:187-226)
    Mode& mode = *modes[mode_id];
    auto it = mode.there.find(target_zone_id);
    if (it != mode.there.end()) successor.push_back(it->second);
    else {
      BeliefState succ(mode.belief_state.size(), 0.0);
      succ[target_zone_id] = 1.0;
      succ = tamp_normalize(succ);
      double p = mode.reaching_probability * transition_probability(mode.belief_state, succ);
      size_t succ_mode;
      auto hm = mode_hash_map.find(belief_hash(succ));
      if (hm != mode_hash_map.end()) succ_mode = hm->second;
      else {
        succ_mode = add_mode(remaining_without(mode), p, succ);
        Mode& nm = *modes[succ_mode];
        size_t goal_id = nm.add_sample(domain->zone_positions[target_zone_id], 0.0, 0.0);
        nm.final_node_ids.push_back(goal_id);
      }
      size_t t = transitions.size();
      transitions.push_back({target_zone_id, mode_id, succ_mode, {}});
      modes[mode_id]->there[target_zone_id] = t;
      successor.push_back(t);
    }
  }
  {  // object not there (:230-267)
    Mode& mode = *modes[mode_id];
    auto it = mode.not_there.find(target_zone_id);
    if (it != mode.not_there.end()) successor.push_back(it->second);
    else {
      BeliefState succ = mode.belief_state;
      succ[target_zone_id] = 0.0;
      double p = mode.reaching_probability * transition_probability(mode.belief_state, succ);
      succ = tamp_normalize(succ);
      size_t succ_mode;
      auto hm = mode_hash_map.find(belief_hash(succ));
      if (hm != mode_hash_map.end()) succ_mode = hm->second;
      else {
        succ_mode = add_mode(remaining_without(mode), p, succ);
        for (size_t z = 0; z < succ.size(); ++z)
          if (succ[z] == 1.0) {
            Mode& nm = *modes[succ_mode];
            size_t goal_id = nm.add_sample(domain->zone_positions[z], 0.0, 0.0);
            nm.final_node_ids.push_back(goal_id);
            break;
          }
      }
      size_t t = transitions.size();
      transitions.push_back({target_zone_id, mode_id, succ_mode, {}});
      modes[mode_id]->not_there[target_zone_id] = t;
      successor.push_back(t);
    }
  }
  return successor;
}
State TampPRM::sample_observation_of_zone(size_t target_zone_id) {
  State zp = domain->zone_positions[target_zone_id];
  State ra = zone_sampler.sample();
  double radius = domain->visibility_distance, angle = ra[1];
  auto clamp = [](double v, double lo, double hi) { return v < lo ? lo : (v > hi ? hi : v); };
  return {clamp(zp[0] + radius * std::cos(angle), continuous.low[0], continuous.up[0] - 0.0001),
          clamp(zp[1] + radius * std::sin(angle), continuous.low[1], continuous.up[1] - 0.0001)};
}
void TampPRM::grow_mm_prm(State start, const BeliefState& b0, double max_step, double search_radius, size_t n_iter_per_belief) {
  belief_states = domain->reachable_belief_states(b0);
  std::vector<size_t> all(domain->n_zones);
  for (size_t z = 0; z < all.size(); ++z) all[z] = z;
  add_mode(all, 1.0, b0);
  modes[0]->add_sample(start, 0.0, 0.0);
  size_t total = n_iter_per_belief * belief_states.size();
  const size_t batch = 200, per_batch_transitions = 10;
  size_t n_outer = (size_t)((double)total / (double)batch);
  size_t n_within = batch - per_batch_transitions;
  for (size_t i = 0; i < n_outer; ++i) {
    size_t mode_id = discrete.sample(modes.size());
    {
      Mode& mode = *modes[mode_id];
      for (size_t k = 0; k < n_within; ++k) {   // PRM::grow_graph (prm.rs:38-50)
        State s = mode.prm.sampler.sample();
        mode.add_sample(s, max_step, search_radius);
        mode.prm.n_it += 1;
      }
    }
    for (size_t j = 0; j < per_batch_transitions; ++j) {
      if (modes[mode_id]->remaining_zones.empty()) continue;
      size_t zi = discrete.sample(modes[mode_id]->remaining_zones.size());
      size_t target = modes[mode_id]->remaining_zones[zi];
      std::vector<size_t> tids = get_transitions(mode_id, target);
      State ts = sample_observation_of_zone(target);
      size_t obs_node = modes[mode_id]->add_sample(ts, max_step, search_radius);
      for (size_t tid : tids) {
        size_t to_mode = transitions[tid].to_mode_id;
        size_t dst = modes[to_mode]->add_sample(ts, max_step, search_radius);
        transitions[tid].observation_transitions.push_back({obs_node, dst});
      }
    }
  }
}
bool TampPRM::build_belief_graph() {
  belief_graph = BeliefGraph();
  belief_graph.reachable_belief_states = belief_states;
  for (size_t b = 0; b < belief_states.size(); ++b) belief_graph.belief_states_to_id[belief_hash(belief_states[b])] = b;
  final_belief_node_ids.clear();
  std::vector<size_t> base(modes.size());
  for (auto& mp : modes) {
    Mode& mode = *mp;
    auto it = belief_graph.belief_states_to_id.find(belief_hash(mode.belief_state));
    if (it == belief_graph.belief_states_to_id.end()) return false;   // HashMap index panic (:413)
    size_t belief_id = it->second;
    // the reference stores the MODE's belief vector in every belief node (:419); our BeliefGraph resolves beliefs through
    // belief_id, so the table entry of this belief is replaced by the mode's vector (one mode per belief hash)
    belief_graph.reachable_belief_states[belief_id] = mode.belief_state;
    base[mode.id] = belief_graph.nodes.size();
    for (const PTONode& n : mode.prm.graph.nodes) belief_graph.add_node(n.state, belief_id, ACTION);
    for (size_t f : mode.final_node_ids) final_belief_node_ids.push_back(base[mode.id] + f);
  }
  for (const Transition& t : transitions)
    for (const auto& e : t.observation_transitions) {
      size_t from = base[t.from_mode_id] + e[0], to = base[t.to_mode_id] + e[1];
      belief_graph.add_edge(from, to);
      belief_graph.nodes[from].node_type = OBSERVATION;
    }
  for (auto& mp : modes) {
    Mode& mode = *mp;
    for (size_t id = 0; id < mode.prm.graph.nodes.size(); ++id) {
      size_t bn = base[mode.id] + id;
      if (belief_graph.nodes[bn].node_type == OBSERVATION) continue;
      for (const PTOEdge& c : mode.prm.graph.nodes[id].children) belief_graph.add_edge(bn, base[mode.id] + c.id);
    }
  }
  return true;
}
bool TampPRM::plan(State start, const BeliefState& b0, double max_step, double search_radius, size_t n_iter_per_belief, Policy& out) {
  grow_mm_prm(start, b0, max_step, search_radius, n_iter_per_belief);
  if (!build_belief_graph()) return false;
  if (!conditional_dijkstra(belief_graph, final_belief_node_ids, expected_costs)) return false;
  if (expected_costs.empty() || !std::isfinite(expected_costs[0])) return false;   // (the reference would not terminate)
  return extract_policy(belief_graph, expected_costs, out);
}

}  // namespace orc
