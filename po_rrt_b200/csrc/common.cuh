// common.cuh -- context, error handling, device-buffer plumbing and the reference's host formulas shared by the libporrt_b200
// translation units.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include <cmath>
#include <cstdio>
#include <cstring>
#include <limits>
#include <map>
#include <string>
#include <vector>

#include "../../include/porrt_b200.h"

#define PORRT_API extern "C" __attribute__((visibility("default")))

struct DevBuf {  // grow-only device scratch
  void* p = nullptr;
  size_t cap = 0;
  cudaError_t ensure(size_t bytes) {
    if (bytes <= cap) return cudaSuccess;
    if (p) cudaFree(p);
    p = nullptr; cap = 0;
    size_t want = bytes + bytes / 4 + 256;
    cudaError_t e = cudaMalloc(&p, want);
    if (e == cudaSuccess) cap = want;
    return e;
  }
  // grows like ensure() but carries the first keep_bytes over (device-to-device on `st`); the old block is freed after the copy
  cudaError_t grow_keep(size_t bytes, size_t keep_bytes, cudaStream_t st) {
    if (bytes <= cap) return cudaSuccess;
    void* q = nullptr;
    const size_t want = bytes + bytes / 2 + 256;
    cudaError_t e = cudaMalloc(&q, want);
    if (e != cudaSuccess) return e;
    if (p && keep_bytes) {
      e = cudaMemcpyAsync(q, p, keep_bytes, cudaMemcpyDeviceToDevice, st);
      if (e == cudaSuccess) e = cudaStreamSynchronize(st);
      if (e != cudaSuccess) { cudaFree(q); return e; }
    }
    if (p) cudaFree(p);
    p = q; cap = want;
    return cudaSuccess;
  }
  void release() { if (p) cudaFree(p); p = nullptr; cap = 0; }
  template <class T> T* as() const { return (T*)p; }
};

struct PinBuf {  // grow-only pinned host staging
  void* p = nullptr;
  size_t cap = 0;
  cudaError_t ensure(size_t bytes) {
    if (bytes <= cap) return cudaSuccess;
    if (p) cudaFreeHost(p);
    p = nullptr; cap = 0;
    size_t want = bytes + bytes / 4 + 256;
    cudaError_t e = cudaHostAlloc(&p, want, cudaHostAllocDefault);
    if (e == cudaSuccess) cap = want;
    return e;
  }
  void release() { if (p) cudaFreeHost(p); p = nullptr; cap = 0; }
  template <class T> T* as() const { return (T*)p; }
};

// The layout of one block of work space, written once as a function layout(Carve&) that takes its pieces in order.  carve() runs it
// twice: a size pass without a base (offsets as integers), then, after ensure(size), the pass that assigns the real pointers.
// Bases from cudaMalloc / cudaHostAlloc are 256-byte aligned, so a piece's alignment holds for its address too.
struct Carve {
  uintptr_t base = 0, off = 0;   // base 0: the size pass (every take returns nullptr)
  template <class T> T* take(size_t count, size_t align = 16) {
    off = (off + align - 1) & ~(uintptr_t)(align - 1);
    T* p = base ? (T*)(base + off) : nullptr;
    off += count * sizeof(T);
    return p;
  }
};
template <class Layout> size_t carve_size(Layout&& layout) { Carve c; layout(c); return c.off; }
template <class Buf, class Layout> cudaError_t carve(Buf& buf, Layout&& layout) {
  const cudaError_t e = buf.ensure(carve_size(layout));
  if (e != cudaSuccess) return e;
  Carve c{(uintptr_t)buf.p};
  layout(c);
  return cudaSuccess;
}

// Device-side description of an uploaded map (passed by value to kernels).
struct MapDev {
  const uint8_t* grid;  // fused code grid, tiled (see map.cu: tile_addr)
  const uint8_t* coarse;    // large-map path (map.cu): one class byte per 16 x 16 block, row-major (C_* flags)
  int32_t coarse_cw;        // its row pitch
  // edge3.cu: 2-bit class per 16 x 16 block (16 per word, row-major; staged in shared memory by the kernel) and the
  // blocking-pixel bitmaps of the blocks, four orientations x 32 bytes per block
  const uint32_t* plane;
  const uint32_t* bits;
  int32_t plane_cw, plane_ch;  // blocks per block row / block rows
  int32_t plane_bytes;      // padded to a multiple of 16
  int32_t plane_guard;      // free blocks in front of (and behind) block 0 in the plane
  int32_t bits_var_words;   // 32-bit words per orientation (= blocks * 8)
  int32_t H, W;         // logical size
  int32_t tiles_x;      // 128-byte tiles (16 x 8 px) per tile row
  int32_t kind;         // PORRT_DOMAIN_*
  int32_t free_vid;     // validity id of free space (n_validities - 1)
  int32_t mask_words;
  double low0, low1, ppm, hm1;  // hm1 = (double)(H - 1)
};

static const int MAX_SLOTS = 3;

struct porrt_ctx {
  int device = 0;
  int sm_count = 148;
  cudaStream_t stream = nullptr;      // compute stream (own or borrowed)
  cudaStream_t own_stream = nullptr;
  cudaStream_t copy_in = nullptr, copy_out = nullptr;
  cudaEvent_t ev_in[MAX_SLOTS] = {}, ev_k[MAX_SLOTS] = {}, ev_out[MAX_SLOTS] = {};
  std::string err;
  int64_t launches = 0;
  // device-side phase timing of the last host-buffer call (CUDA events on the compute stream)
  cudaEvent_t ev_t[16] = {};
  int n_marks = 0, n_last = 0;
  double last_ms[16] = {};

  // ---- map
  bool has_map = false;
  MapDev map = {};
  int n_zones = 0, n_worlds = 0, n_validities = 0, mask_words = 1;
  double visibility = 0.0;
  std::vector<uint64_t> validities;     // [n_validities * mask_words]
  std::vector<double> zone_pos;         // [2 * n_zones]
  std::vector<uint64_t> zone_world_masks;  // DOOR: zones_to_worlds [n_zones * mask_words]
  DevBuf d_grid, d_coarse, d_validities, d_zone_pos, d_plane, d_bits;
  bool force_large_map_path = false;   // PORRT_OPT_FORCE_LARGE_MAP_PATH (tests): run map.cu's kernel although edge3.cu's would fit
  bool force_global_sweeps = false;    // PORRT_OPT_FORCE_GLOBAL_SWEEPS (tests): value backups by the frontier relaxation (sssp_frontier.cu) although colsolve.cu would fit
  bool force_thread_per_query_nn = false;  // PORRT_OPT_FORCE_THREAD_PER_QUERY_NN (tests): nn.cu's kernels although nn_tile.cu's would serve
  // host copies of the raw images are NOT kept: the product never walks pixels on the CPU.

  // ---- vertices / cell grid (nn.cu)
  int64_t n_vertices = 0;          // vertices in d_vxy (upload order), including appended ones
  int64_t vertex_gen = 0;          // bumped by every porrt_vertices_set / _set_dev / _append: a PRM query knows its roadmap's set
  bool grid_stale = false;         // porrt_vertices_append: the cell grid below is rebuilt on the device before the next query
  double cell_request = 0.0;       // cell size asked for by the last porrt_vertices_set (<= 0: from the density)
  double cell = 0, inv_cell = 0, org_x = 0, org_y = 0;
  int32_t cells_x = 0, cells_y = 0;
  DevBuf d_vxy_sorted, d_vid_sorted, d_cell_start, d_vxy, d_vcell;
  DevBuf nn_bins;        // nn_tile.cu: query bins (nt_layout), or the merge scripts' sizes while they are built
  DevBuf d_nbr_start, d_nbr_script;   // nn_tile.cu: per-cell merge scripts of the 3 x 3 neighbourhood (built lazily per vertex set)
  bool nbr_ready = false;
  DevBuf nn_stage;       // nn_tile.cu: tile-ordered staging of the radius lists + per-query staging offsets
  DevBuf comm_tmp;       // comm.cu: staging of the padded all-gather behind ragged exchanges
  DevBuf nn_stage2;      // nn.cu: fixed-size slots of the thread- / warp-per-query radius kernels (one pass: count + stage)
  int32_t nn_fb_n = 0;   // queries of the last tile pass left to the thread-per-query kernels
  int32_t reach_words = 1;  // u64 words per vertex of the reachability filter of the running NN call

  // ---- last belief VI result (graph.cu), kept for porrt_extract_policy, porrt_belief_result and the refiners (refine.cu)
  struct BeliefState_ {
    int64_t V = 0; int32_t B = 0, n_worlds = 0;
    std::vector<int64_t> row_ptr; std::vector<int32_t> col, edge_vid; std::vector<double> xy;
    std::vector<int32_t> node_vid;                // [V] validity id of each roadmap node
    std::vector<double> beliefs;
    const double* dist = nullptr; const uint8_t* type = nullptr;   // live in ctx->pin_bel (pinned: the V*B table comes back by DMA)
    std::vector<int32_t> node_obs_set;            // [V] index into obs tables
    std::vector<int64_t> succ_ptr;                // [(n_sets*B)+1]
    std::vector<int32_t> succ_belief;             // successor belief ids
    std::vector<uint8_t> compat;                  // [B * n_validities]
    int32_t n_validities = 0;
    // column-solver results stay on the device ([column][node], dedicated buffer); the host copy of the whole table is made only
    // when somebody asks for it (out_dist / porrt_belief_result), the policy walk fetches the few columns it visits
    bool on_host = false;
    DevBuf dev;
    const double* d_dist_cm = nullptr; const uint8_t* d_type_cm = nullptr; const uint8_t* d_type = nullptr; const int32_t* d_colpos = nullptr;
    std::vector<int32_t> colpos;
    std::vector<std::vector<double>> col_dist;    // [B] lazily fetched columns (empty = not fetched)
    std::vector<std::vector<uint8_t>> col_type;
    bool fetch_failed = false;                    // a column fetch failed since the caller last cleared this

    // Value and node type of belief node id = node * B + belief: from the host table, or from the belief's column, fetched from
    // the device on first use (a policy touches a few dozen of the B columns, 8 * V bytes each).  A failed fetch reads as 0.
    double value(porrt_ctx* ctx, int64_t id) {
      if (on_host) return dist[(size_t)id];
      const int b = (int)(id % B);
      return column(ctx, b) ? col_dist[(size_t)b][(size_t)(id / B)] : 0.0;
    }
    uint8_t node_type(porrt_ctx* ctx, int64_t id) {
      if (on_host) return type[(size_t)id];
      const int b = (int)(id % B);
      return column(ctx, b) ? col_type[(size_t)b][(size_t)(id / B)] : (uint8_t)0;
    }
    // fn(child id) for the children of belief node id in the reference's stored order (pto.rs:206-255): an Observation node's
    // successor beliefs compatible with its node's validity, or an Action node's edges whose end and edge validity its belief allows
    template <class F> void for_children(porrt_ctx* ctx, int64_t id, F&& fn) {
      const int64_t n = id / B;
      const int b = (int)(id % B);
      const uint8_t ty = node_type(ctx, id);
      if (ty == PORRT_NODE_OBSERVATION) {
        const int64_t sp = (int64_t)node_obs_set[(size_t)n] * B + b;
        for (int64_t k = succ_ptr[(size_t)sp]; k < succ_ptr[(size_t)sp + 1]; ++k) {
          const int32_t cb = succ_belief[(size_t)k];
          if (compat[(size_t)cb * n_validities + node_vid[(size_t)n]]) fn(n * B + cb);
        }
      } else if (ty == PORRT_NODE_ACTION) {
        for (int64_t e = row_ptr[(size_t)n]; e < row_ptr[(size_t)n + 1]; ++e) {
          const int32_t c = col[(size_t)e];
          if (compat[(size_t)b * n_validities + node_vid[(size_t)c]] && compat[(size_t)b * n_validities + edge_vid[(size_t)e]]) fn((int64_t)c * B + b);
        }
      }
    }
    // whether column b is on the host, fetching it if need be (graph.cu); a failed fetch leaves it unfetched and sets fetch_failed
    bool column(porrt_ctx* ctx, int b) { return !col_dist[(size_t)b].empty() || fetch_column(ctx, b); }
    bool fetch_column(porrt_ctx* ctx, int b);
  } bel;
  DevBuf d_bel_succ;                   // observation successor tables of the running / last porrt_belief_vi (belief_tables.cu)
  // last PRM result, kept on the device (valid until the next call on this ctx)
  int64_t prm_n = 0, prm_edges = 0;
  const int64_t* prm_row_ptr = nullptr;
  const int32_t* prm_col = nullptr;
  const void* radii_ptr = nullptr; int64_t radii_lo = 0, radii_n = 0; double radii_ms = 0, radii_sr = 0;   // what pin_radii holds: heuristic_radius(k + 1) for k in [radii_lo, radii_n)
  DevBuf d_prm_row, d_prm_col;         // dedicated: the retained CSR must survive later calls that reuse the shared scratch
  bool prm_grouped = false;            // the last PRM result is porrt_mmprm_plan's grouped build (its vertex set mixes modes)
  int64_t prm_vertex_gen = -1;         // vertex_gen when the last PRM build bound its vertex set
  int64_t prm_paths_chunk = 0;         // PORRT_OPT_PRM_PATHS_CHUNK_COLUMNS (tests): > 0 caps porrt_prm_plan_paths' columns per chunk
  int64_t reparent_brute_max = 4096;   // PORRT_OPT_REPARENT_BRUTE_MAX_NODES (tests): reparent trees up to this size take the all-pairs sweep

  // ---- last multi-modal PRM result (mmprm.cu): the explicit belief graph, kept for porrt_mmprm_fetch_graph
  struct MmPrm_ {
    std::vector<int64_t> row_ptr; std::vector<int32_t> col, belief_id; std::vector<uint8_t> type;
  } mm;

  // ---- last PTO growth (pto_grow.cu): the roadmap stays on the device until porrt_pto_fetch
  struct PtoGrow* pto = nullptr;
  // ---- last RRT growth (pto_grow.cu, the same machinery): the trees stay on the device until porrt_rrt_fetch_tree
  struct PtoGrow* rrt = nullptr;

  // ---- multi-GPU (comm.cu): NCCL communicator bound at run time; world 1 = no communicator
  void* comm = nullptr;
  int comm_rank = 0, comm_world = 1;

  // ---- work space.  The rule: a function carves only from buffers that no function above it on the call stack holds pointers
  // into.  Call trees that never nest share the large buffers: a DevBuf never shrinks, so a buffer per user would keep the sum of
  // their peaks.  Users of each buffer:
  DevBuf kd_buf;      // kd_preorder_rank_dev (its own: the PRM build runs the rank on a helper thread next to the binning sort)
  cudaStream_t aux_stream = nullptr;   // second compute stream (created on first use): kd rank next to radius / edge batches
  DevBuf ws_main;     // the entry points' inputs and work blocks: porrt_radius_query, knn_host, porrt_state_validity, porrt_visibility,
                      // porrt_transition_valid, the shortcut and Reparent refiners, porrt_sssp_worlds(_prm) and porrt_belief_vi (held
                      // while graph.cu's value-column driver runs, which carves from ws_state),
                      // porrt_conditional_dijkstra_graph, the PRM build's per-node arrays; edge_pipeline's chunk slots;
                      // porrt_prm_plan_paths' queries and per-query results (held while the 1-NN, the kd rank and sssp_core run)
  DevBuf ws_owner;    // map upload: the occupancy image; PRM build: the owner of each candidate, then the packed neighbour lists;
                      // porrt_prm_plan_paths: the paths in query order
  DevBuf ws_vid;      // map upload: the zone image; PRM build: the candidates' validity ids, then the late lists and cursors;
                      // porrt_prm_plan_paths: the paths in chunk order, as the walks write them
  DevBuf ws_table;    // map upload: zone statistics; the radius id lists of porrt_radius_query and the PRM build
                      // (nn_radius_count_fill_dev's ids_buf); sssp_core's world table, world masks and column map;
                      // belief_download_full's [node][belief] table
  DevBuf ws_query;    // nn_radius_count_fill_dev: staging offsets, counts and the wide-query list; nn_vertices_set_dev's bounding
                      // box; edge_pipeline's id check flag; belief_succ_tables' inputs and work space; porrt_measure_l2_gather's sink
  DevBuf ws_seg;      // segments_sort_by_key_dev: its counters, mid-length segment list and inverse key permutation
  DevBuf sort_keys, sort_vals;   // nn_vertices_set_dev's and segments_sort_by_key_dev's (radix path) pairs to sort; sf_build_graph's
                                 // Morton order (keys) and transposed graph (vals); porrt_edge_validity_csr_i8's row_ptr (keys)
  DevBuf ws_state;    // nn_vertices_set_dev: cell counts; sf_relax: the frontier state (sf_state_layout); the value-column driver
                      // (graph.cu): its block behind that state (sf_state_reserve): the Morton-numbered table, the finals, the
                      // column solver's counters and transposed graph
  DevBuf radix_keys, radix_vals, radix_hist;   // radix_sort_pairs: the second key / value array, the histograms and tile bases;
                      // porrt_kd_preorder_rank's coordinates and ranks (radix_vals); the PRM build's shard summaries (radix_hist)
  DevBuf scan_sums;   // scan_exclusive_i64: block sums
  PinBuf pin_edge;    // edge_pipeline: pinned twins of the chunk slots for pageable callers
  PinBuf pin_radii;   // the PRM build's heuristic_radius table (kept across calls: radii_ptr)
  PinBuf pin_bel;     // belief_download_full: the host V x B table of the last porrt_belief_vi (bel.dist / bel.type)
  PinBuf pin_row, pin_col;   // porrt_mmprm_plan: the grouped PRM's CSR
  PinBuf pin_flags;   // a few counters the kernels write straight into host memory (no DMA engine: see read_flags_dev, nn.cu)
};

#define CTX_CHECK(ctx) do { if (!(ctx)) return PORRT_ERR_INVALID_ARG; } while (0)

static inline int32_t porrt_fail(porrt_ctx* ctx, int32_t code, const std::string& msg) {
  if (ctx) ctx->err = msg;
  return code;
}

// (the expression's text is cut at 200 characters: a carve() call spells out its whole layout)
#define CUDA_TRY(ctx, expr)                                                                        \
  do {                                                                                             \
    cudaError_t _e = (expr);                                                                       \
    if (_e != cudaSuccess) {                                                                       \
      char _b[512];                                                                                \
      snprintf(_b, sizeof(_b), "%s:%d %.200s -> %s", __FILE__, __LINE__, #expr, cudaGetErrorString(_e)); \
      return porrt_fail(ctx, PORRT_ERR_CUDA, _b);                                                  \
    }                                                                                              \
  } while (0)

#define LAUNCH_CHECK(ctx)                                                                          \
  do {                                                                                             \
    (ctx)->launches += 1;                                                                          \
    CUDA_TRY(ctx, cudaGetLastError());                                                             \
  } while (0)

static inline bool is_pinned_host(const void* p) {
  cudaPointerAttributes a;
  if (cudaPointerGetAttributes(&a, p) != cudaSuccess) { cudaGetLastError(); return false; }
  return a.type == cudaMemoryTypeHost;
}

static inline void tstart(porrt_ctx* ctx) { ctx->n_marks = 0; if (ctx->ev_t[0]) cudaEventRecord(ctx->ev_t[ctx->n_marks++], ctx->stream); }
static inline void tmark(porrt_ctx* ctx) { if (ctx->ev_t[0] && ctx->n_marks < 16) cudaEventRecord(ctx->ev_t[ctx->n_marks++], ctx->stream); }
static inline void tfinish(porrt_ctx* ctx) {  // call after the stream has been synchronised
  ctx->n_last = 0;
  for (int k = 0; k + 1 < ctx->n_marks; ++k) {
    float ms = 0.f;
    if (cudaEventElapsedTime(&ms, ctx->ev_t[k], ctx->ev_t[k + 1]) != cudaSuccess) { cudaGetLastError(); ms = -1.f; }
    ctx->last_ms[ctx->n_last++] = ms;
  }
}

static inline int div_up(int64_t a, int64_t b) { return (int)((a + b - 1) / b); }

// ---- host formulas of the reference (the kernels have their own __d*_rn forms).  The host objects are built with
// -ffp-contract=off, so these round like the reference's f64 code.
// norm2 (common.rs:203-213): the squares of b - a summed from 0.0 in dimension order
static inline double norm2(const double* a, const double* b, int dim) {
  double d2 = 0.0;
  for (int k = 0; k < dim; ++k) { const double dx = b[k] - a[k]; d2 += dx * dx; }
  return std::sqrt(d2);
}
// transition_probability (common.rs:188-190): the parent's mass on the worlds the child belief holds possible
static inline double transition_probability(const double* parent, const double* child, int n_worlds) {
  double s = 0.0;
  for (int i = 0; i < n_worlds; ++i) s = s + (child[i] > 0.0 ? parent[i] : 0.0);
  return s;
}
// heuristic_radius (common.rs:357-369): libm ln / pow like Rust's f64::ln / powf
static inline double heuristic_radius(int64_t n_nodes, double max_step, double search_radius, int dim) {
  const double n = (double)n_nodes;
  const double s = search_radius * std::pow(std::log(n) / n, 1.0 / (double)dim);
  return s < max_step ? s : max_step;
}

// extract_policy / get_best_expected_children (belief_graph.rs:184-267) on the host, over any belief graph of n_nodes belief
// nodes rooted at id 0: for_children(id, fn) calls fn(child id) in stored order, belief_of(id) is the id's row of
// beliefs[. * n_worlds], cost(parent id, child id) the edge cost, dist(id) the expected cost to the goals.  pol: (belief node
// id, parent, leaf) per policy node in creation order.  The reference's asserts are PORRT_ERR_PANIC; `name` names the caller in
// the message of a walk that does not terminate.
struct PolicyNode { int64_t id; int32_t parent; uint8_t leaf; };
template <class ForChildren, class BeliefOf, class Cost, class Dist>
int32_t get_best_expected_children(porrt_ctx* ctx, const char* name, int64_t n_nodes, const double* beliefs, int n_worlds,
                                   ForChildren&& for_children, BeliefOf&& belief_of, Cost&& cost, Dist&& dist, std::vector<PolicyNode>& pol) {
  struct Child { int64_t id; double cost_to_child, expected_from_child; };
  std::vector<std::pair<int64_t, int64_t>> lifo;   // (policy node, belief node)
  pol.assign(1, PolicyNode{0, -1, 0});
  lifo.push_back({0, 0});
  while (!lifo.empty()) {
    const auto top = lifo.back();
    lifo.pop_back();
    const int64_t bn = top.second;
    std::map<int32_t, std::vector<Child>> by_belief;   // BTreeMap keyed by child.belief_id (:228-241)
    for_children(bn, [&](int64_t c) { by_belief[belief_of(c)].push_back({c, cost(bn, c), dist(c)}); });
    for (auto& kv : by_belief) {
      int64_t best_id = kv.second[0].id;
      const double p = transition_probability(beliefs + (size_t)belief_of(bn) * n_worlds, beliefs + (size_t)belief_of(best_id) * n_worlds, n_worlds);
      if (!(p > 0.0)) return porrt_fail(ctx, PORRT_ERR_PANIC, "assert!(p > 0.0) (belief_graph.rs:250)");
      double best_cost = std::numeric_limits<double>::infinity();
      for (const Child& c : kv.second) {
        const double cst = p * (c.cost_to_child + c.expected_from_child);
        if (cst < best_cost) { best_cost = cst; best_id = c.id; }
      }
      if (!(p * dist(best_id) <= dist(bn))) return porrt_fail(ctx, PORRT_ERR_PANIC, "assert!(p * cost[best] <= cost[node]) (belief_graph.rs:261)");
      const bool leaf = dist(best_id) == 0.0;
      const int64_t pid = (int64_t)pol.size();
      pol.push_back({best_id, (int32_t)top.first, (uint8_t)leaf});
      if (!leaf) lifo.push_back({pid, best_id});
      if ((int64_t)pol.size() > 64 * n_nodes + 1024) return porrt_fail(ctx, PORRT_ERR_PANIC, std::string(name) + ": policy does not terminate");
    }
  }
  return PORRT_OK;
}

// comm.cu
void comm_shard_range(int64_t n, int rank, int world, int64_t* lo, int64_t* hi);
int32_t comm_all_gatherv_dev(porrt_ctx* ctx, const void* send_dev, void* recv_dev, const int64_t* offsets /* host [world+1] */, cudaStream_t st);
// map.cu
struct EdgeOut {   // where an edge batch's results go (device pointers): vid XOR vid8, mask optional
  int32_t* vid = nullptr;
  int8_t* vid8 = nullptr;
  uint64_t* mask = nullptr;
};
int32_t map_edge_validity_dev(porrt_ctx* ctx, const double* from_dev, const double* to_dev, int64_t n,
                              int32_t* out_vid_dev, uint64_t* out_mask_dev, cudaStream_t st);
int32_t map_edge_launch(porrt_ctx* ctx, const double* from_dev, const double* to_dev, const int32_t* from_idx_dev,
                        const int32_t* to_idx_dev, int64_t n, const EdgeOut& out, cudaStream_t st);
int32_t map_edge_validity_indexed_dev(porrt_ctx* ctx, const double* xy_dev, const int32_t* from_idx_dev, const int32_t* to_idx_dev,
                                      int64_t n, int32_t* out_vid_dev, cudaStream_t st);
// edge3.cu
int32_t edge3_build(porrt_ctx* ctx, cudaStream_t st);
bool edge3_usable(const porrt_ctx* ctx);
int32_t edge3_launch(porrt_ctx* ctx, const double* from_dev, const double* to_dev, int64_t n, const EdgeOut& out,
                     const int32_t* from_idx_dev, const int32_t* to_idx_dev, cudaStream_t st);
// nn_tile.cu (TMA-staged vertex tiles); GridDev is defined in nn_dev.cuh
struct GridDev;
bool nn_tile_usable(const porrt_ctx* ctx, int64_t m);
int32_t nn_tile_radius_collect(porrt_ctx* ctx, const GridDev& g, const double* q_dev, const double* radius_dev, int64_t m,
                               const uint32_t* prefix_dev, const uint64_t* reach_dev, const uint32_t* world_dev, int32_t* counts_dev,
                               int64_t* stg_off_dev, const int32_t** staging_out, const int32_t** fb_list_out, int32_t* fb_n_out,
                               int64_t* staged_total_out = nullptr);
int32_t nn_tile_radius_place(porrt_ctx* ctx, const int32_t* staging, const int64_t* stg_off_dev, const int64_t* offsets_dev, int64_t m,
                             int32_t* ids_dev);
int32_t nn_tile_knn(porrt_ctx* ctx, const GridDev& g, const double* q_dev, int64_t m, int k, const uint64_t* reach_dev,
                    const uint32_t* world_dev, int32_t* ids_dev, double* dist_dev, int32_t* ties_dev, const int32_t** fb_list_out,
                    int32_t* fb_n_out);
// nn.cu helpers used by graph.cu
int32_t nn_vertices_set_dev(porrt_ctx* ctx, const double* xy_dev, int64_t n, double cell_size, const double* lo, const double* hi);
int32_t nn_flush_appended(porrt_ctx* ctx);   // re-bins the vertex set if porrt_vertices_append left it stale
int32_t nn_knn_dev(porrt_ctx* ctx, const double* q_dev, int64_t m, int k, const uint64_t* reach_dev, const uint32_t* world_dev,
                   int32_t* ids_dev, double* dist_dev, int32_t* ties_dev);   // knn_host's kernels on device inputs / outputs
int32_t nn_radius_count_fill_dev(porrt_ctx* ctx, const double* q_dev, const double* radius_dev, int64_t m,
                                 const uint32_t* prefix_dev, const uint64_t* reach_dev, const uint32_t* world_dev,
                                 int64_t* offsets_dev /* [m+1] */, DevBuf* ids_buf, int64_t* total_out,
                                 const uint32_t* prefix_lo_dev = nullptr, bool sort_ids = false, bool allow_tiles = true);
int32_t scan_exclusive_i64(porrt_ctx* ctx, const int32_t* counts_dev, int64_t n, int64_t* out_dev /* [n+1] */);
int32_t read_flags_dev(porrt_ctx* ctx, const int32_t* flags_dev, int n, int32_t* out, cudaStream_t st);   // n <= 16; synchronises st
int32_t segments_sort_by_key_dev(porrt_ctx* ctx, const int64_t* offsets_dev, int64_t m, int32_t* ids_dev,
                                 const int32_t* key_of_id_dev, int64_t key_limit, const int32_t* seg_list_dev = nullptr, int64_t n_listed = 0);
int32_t radix_sort_pairs(porrt_ctx* ctx, uint64_t* keys, uint32_t* vals, int64_t n, int key_bits);
int bits_for(uint64_t max_value);
// graph.cu: children CSR from per-node early lists (PRM build tail; PTO growth with edge validity ids)
int32_t late_list_csr_dev(porrt_ctx* ctx, const int64_t* seg_off, int64_t n, const int32_t* compact, const int32_t* early_cnt,
                          const int32_t* early_vid, int32_t* late_cnt, int32_t* cursor, int64_t* late_off, int32_t* late_vals,
                          int64_t* row_ptr, int32_t* col, int32_t* vid);
// pto_grow.cu
void pto_grow_release(porrt_ctx* ctx);
int32_t prm_build_impl(porrt_ctx* ctx, const double* samples_xy, int64_t n, double max_step, double search_radius,
                       const double* ms_arr, const double* sr_arr, int64_t* out_row_ptr, int32_t* out_col, int64_t cap,
                       int64_t* out_n_edges, double* out_phase_ms, const int64_t* group_ptr = nullptr, int32_t n_groups = 0);
// st / err / n_launch: when the rank is computed by a helper thread on its own stream, errors and launch counts come back through
// these instead of touching ctx (st == nullptr: ctx->stream, ctx->err, ctx->launches as usual)
int32_t kd_preorder_rank_dev(porrt_ctx* ctx, const double* xy_dev, int64_t n, int32_t* out_rank_dev, const uint32_t* root_of_dev = nullptr,
                             cudaStream_t st = nullptr, std::string* err = nullptr, int64_t* n_launch = nullptr);
