// belief_explicit.cu -- conditional_dijkstra / extract_policy on an EXPLICIT belief graph (reference src/belief_graph.rs).
//
// porrt_belief_vi (graph.cu) covers PTO::build_belief_graph's dense node x belief product without materialising it.  The
// reference's free functions `conditional_dijkstra(&BeliefGraph, finals, cost)` (belief_graph.rs:89-182) and
// `extract_policy(&BeliefGraph, costs, cost)` (:184-267) are also called on hand-built graphs (its own tests, :276-567) and on
// the multi-modal PRM's graph (map_shelves_tamp_prm.rs:476-484), where belief nodes are arbitrary (state, belief_id, type)
// triples.  This file is that entry point: children adjacency as CSR in add_edge order, one warp per belief node.
//
// Value backup (same fixed-point argument as graph.cu, SURVEY 8(g) note 5): dist is the greatest fixed point reachable from
// +inf by monotone updates; each backup uses the reference's operand order --
//   Action u      : min over children v of  cost(u, v) + dist[v]                      (:121-124; min is order-free)
//   Observation u : ((0.0 + p1 * (cost(u, v1) + dist[v1])) + p2 * (...)) + ...        (:125-135; stored child order, lane 0)
// with p = transition_probability(belief(u), belief(v)) (common.rs:188-190) and cost = norm2 (common.rs:203-213).
// Panics of the reference become PORRT_ERR_PANIC: a parent of a reached node with Unknown type (:139-141) or an Observation
// node with a child of p <= 0 (:130) -- such nodes are never updated (the reference stops at their first evaluation), and the
// call fails iff one of them has a child with a finite distance, which is exactly when the reference would have evaluated it.
#include <math_constants.h>

#include "common.cuh"

namespace {

// per CSR edge u -> v: cost = norm2(state u, state v); p = transition_probability(belief u, belief v) for Observation rows
// (states of `dim` doubles; norm2 accumulates dx * dx in dimension order from 0.0, common.rs:203-213 -- 0.0 + x is exact, so the
// two-dimensional case is the dx*dx + dy*dy it always was)
__global__ void bx_edge_kernel(const int64_t* __restrict__ row_ptr, const int32_t* __restrict__ col, const double* __restrict__ xy, int dim,
                               const uint8_t* __restrict__ type, const int32_t* __restrict__ belief_id, const double* __restrict__ beliefs,
                               int nw, int64_t V, double* __restrict__ cost, double* __restrict__ prob, uint8_t* __restrict__ frozen) {
  const int lane = threadIdx.x & 31;
  const int64_t u = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  if (u >= V) return;
  const double* a = xy + u * dim;
  const uint8_t ty = type[u];
  const double* bu = beliefs + (int64_t)belief_id[u] * nw;
  bool bad = false;
  for (int64_t e = row_ptr[u] + lane; e < row_ptr[u + 1]; e += 32) {
    const int32_t v = col[e];
    const double* c = xy + (int64_t)v * dim;
    double d2 = 0.0;
    for (int k = 0; k < dim; ++k) { const double dx = __dsub_rn(c[k], a[k]); d2 = __dadd_rn(d2, __dmul_rn(dx, dx)); }
    cost[e] = __dsqrt_rn(d2);
    double p = 0.0;
    if (ty == PORRT_NODE_OBSERVATION) {
      const double* bv = beliefs + (int64_t)belief_id[v] * nw;
      for (int i = 0; i < nw; ++i) p = __dadd_rn(p, bv[i] > 0.0 ? bu[i] : 0.0);
      if (!(p > 0.0)) bad = true;
    }
    prob[e] = p;
  }
  bad = __any_sync(0xffffffffu, bad);
  if (lane == 0) frozen[u] = (ty == PORRT_NODE_OBSERVATION ? bad : ty != PORRT_NODE_ACTION) ? 1 : 0;
}

__global__ void __launch_bounds__(256) bx_sweep_kernel(const int64_t* __restrict__ row_ptr, const int32_t* __restrict__ col,
                                                       const double* __restrict__ cost, const double* __restrict__ prob,
                                                       const uint8_t* __restrict__ type, const uint8_t* __restrict__ frozen, int64_t V,
                                                       double* __restrict__ dist, int32_t* __restrict__ changed) {
  const int lane = threadIdx.x & 31;
  const int64_t u = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  if (u >= V || frozen[u]) return;
  const int64_t s = row_ptr[u], e1 = row_ptr[u + 1];
  if (s == e1) return;
  const double old = dist[u];
  double alt;
  if (type[u] == PORRT_NODE_ACTION) {
    alt = old;
    for (int64_t e = s + lane; e < e1; e += 32) {
      const double a = __dadd_rn(cost[e], dist[col[e]]);
      if (a < alt) alt = a;
    }
    for (int o = 16; o; o >>= 1) {
      const double other = __shfl_xor_sync(0xffffffffu, alt, o);
      if (other < alt) alt = other;
    }
  } else {
    alt = 0.0;
    if (lane == 0)
      for (int64_t e = s; e < e1; ++e) alt = __dadd_rn(alt, __dmul_rn(prob[e], __dadd_rn(cost[e], dist[col[e]])));
  }
  if (lane == 0 && alt < old) { dist[u] = alt; *changed = 1; }
}

// the reference evaluates a frozen node (and panics) as soon as one of its children is popped, i.e. has a finite distance
__global__ void bx_panic_kernel(const int64_t* __restrict__ row_ptr, const int32_t* __restrict__ col, const uint8_t* __restrict__ frozen,
                                int64_t V, const double* __restrict__ dist, int32_t* __restrict__ panic_node) {
  const int64_t u = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (u >= V || !frozen[u]) return;
  for (int64_t e = row_ptr[u]; e < row_ptr[u + 1]; ++e)
    if (dist[col[e]] < CUDART_INF) { atomicMin(panic_node, (int32_t)u); return; }
}

__global__ void bx_init_kernel(double* __restrict__ dist, int64_t V, const int32_t* __restrict__ finals, int32_t n_finals) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < V) dist[i] = CUDART_INF;
  (void)finals; (void)n_finals;
}
__global__ void bx_finals_kernel(double* __restrict__ dist, const int32_t* __restrict__ finals, int32_t n_finals) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n_finals) dist[finals[i]] = 0.0;
}

bool graph_args_ok(int64_t V, const int64_t* row_ptr, const int32_t* col, const double* xy, const uint8_t* type,
                   const int32_t* belief_id, const double* beliefs, int32_t B, int32_t nw, int32_t dim = 2) {
  if (dim <= 0 || dim > PORRT_MAX_STATE_DIM) return false;
  if (V <= 0 || !row_ptr || !xy || !type || !belief_id || !beliefs || B <= 0 || nw <= 0) return false;
  if (row_ptr[0] != 0 || (row_ptr[V] > 0 && !col)) return false;
  for (int64_t u = 0; u < V; ++u) {
    if (row_ptr[u + 1] < row_ptr[u] || belief_id[u] < 0 || belief_id[u] >= B) return false;
  }
  for (int64_t e = 0; e < row_ptr[V]; ++e)
    if (col[e] < 0 || col[e] >= V) return false;
  return true;
}
}  // namespace

PORRT_API int32_t porrt_conditional_dijkstra(porrt_ctx* ctx, int64_t V, const int64_t* row_ptr, const int32_t* col, const double* xy,
                                             const uint8_t* node_type, const int32_t* belief_id, const double* beliefs, int32_t B,
                                             int32_t n_worlds, const int32_t* finals, int32_t n_finals, double* out_dist,
                                             int32_t* out_sweeps) {
  return porrt_conditional_dijkstra_nd(ctx, 2, V, row_ptr, col, xy, node_type, belief_id, beliefs, B, n_worlds, finals, n_finals, out_dist, out_sweeps);
}

PORRT_API int32_t porrt_conditional_dijkstra_nd(porrt_ctx* ctx, int32_t dim, int64_t V, const int64_t* row_ptr, const int32_t* col,
                                                const double* xy, const uint8_t* node_type, const int32_t* belief_id, const double* beliefs,
                                                int32_t B, int32_t n_worlds, const int32_t* finals, int32_t n_finals, double* out_dist,
                                                int32_t* out_sweeps) {
  CTX_CHECK(ctx);
  if (!out_dist || n_finals < 0 || (n_finals > 0 && !finals) || !graph_args_ok(V, row_ptr, col, xy, node_type, belief_id, beliefs, B, n_worlds, dim))
    return porrt_fail(ctx, PORRT_ERR_INVALID_ARG, "conditional_dijkstra: bad arguments");
  if (V > 0x7fffffff) return porrt_fail(ctx, PORRT_ERR_UNSUPPORTED, "conditional_dijkstra: more than 2^31 belief nodes");
  for (int32_t k = 0; k < n_finals; ++k)
    if (finals[k] < 0 || finals[k] >= V) return porrt_fail(ctx, PORRT_ERR_INVALID_ARG, "conditional_dijkstra: final id out of range");
  CUDA_TRY(ctx, cudaSetDevice(ctx->device));
  cudaStream_t st = ctx->stream;
  const int64_t E = row_ptr[V];
  int64_t* d_row;
  double *d_xy, *d_cost, *d_prob, *d_dist, *d_beliefs;
  int32_t *d_col, *d_bid, *d_finals, *d_flags;   // d_flags: [0] changed, [1] panic node
  uint8_t *d_type, *d_frozen;
  CUDA_TRY(ctx, carve(ctx->ws_main, [&](Carve& c) {
    d_row = c.take<int64_t>(V + 1);
    d_xy = c.take<double>((size_t)V * dim); d_cost = c.take<double>(E); d_prob = c.take<double>(E); d_dist = c.take<double>(V);
    d_beliefs = c.take<double>((size_t)B * n_worlds);
    d_col = c.take<int32_t>(E); d_bid = c.take<int32_t>(V); d_finals = c.take<int32_t>(n_finals + 1); d_flags = c.take<int32_t>(4);
    d_type = c.take<uint8_t>(V); d_frozen = c.take<uint8_t>(V);
  }));
  CUDA_TRY(ctx, cudaMemcpyAsync(d_row, row_ptr, (size_t)(V + 1) * 8, cudaMemcpyHostToDevice, st));
  if (E) CUDA_TRY(ctx, cudaMemcpyAsync(d_col, col, (size_t)E * 4, cudaMemcpyHostToDevice, st));
  CUDA_TRY(ctx, cudaMemcpyAsync(d_xy, xy, (size_t)V * dim * 8, cudaMemcpyHostToDevice, st));
  CUDA_TRY(ctx, cudaMemcpyAsync(d_bid, belief_id, (size_t)V * 4, cudaMemcpyHostToDevice, st));
  CUDA_TRY(ctx, cudaMemcpyAsync(d_type, node_type, (size_t)V, cudaMemcpyHostToDevice, st));
  CUDA_TRY(ctx, cudaMemcpyAsync(d_beliefs, beliefs, (size_t)B * n_worlds * 8, cudaMemcpyHostToDevice, st));
  if (n_finals) CUDA_TRY(ctx, cudaMemcpyAsync(d_finals, finals, (size_t)n_finals * 4, cudaMemcpyHostToDevice, st));
  const int32_t flags0[2] = {0, 0x7fffffff};
  CUDA_TRY(ctx, cudaMemcpyAsync(d_flags, flags0, 8, cudaMemcpyHostToDevice, st));
  bx_edge_kernel<<<div_up(V * 32, 256), 256, 0, st>>>(d_row, d_col, d_xy, dim, d_type, d_bid, d_beliefs, n_worlds, V, d_cost, d_prob, d_frozen);
  LAUNCH_CHECK(ctx);
  bx_init_kernel<<<div_up(V, 256), 256, 0, st>>>(d_dist, V, d_finals, n_finals);
  LAUNCH_CHECK(ctx);
  if (n_finals) {
    bx_finals_kernel<<<div_up(n_finals, 256), 256, 0, st>>>(d_dist, d_finals, n_finals);
    LAUNCH_CHECK(ctx);
  }
  int sweeps = 0;
  const int BATCH = 8;
  for (;;) {
    CUDA_TRY(ctx, cudaMemsetAsync(d_flags, 0, 4, st));
    for (int k = 0; k < BATCH; ++k) {
      bx_sweep_kernel<<<div_up(V * 32, 256), 256, 0, st>>>(d_row, d_col, d_cost, d_prob, d_type, d_frozen, V, d_dist, d_flags);
      LAUNCH_CHECK(ctx);
    }
    sweeps += BATCH;
    int32_t changed = 0;
    CUDA_TRY(ctx, cudaMemcpyAsync(&changed, d_flags, 4, cudaMemcpyDeviceToHost, st));
    CUDA_TRY(ctx, cudaStreamSynchronize(st));
    if (!changed) break;
    if (sweeps > 4 * V + 64) return porrt_fail(ctx, PORRT_ERR_CUDA, "conditional_dijkstra: no convergence");
  }
  bx_panic_kernel<<<div_up(V, 256), 256, 0, st>>>(d_row, d_col, d_frozen, V, d_dist, d_flags + 1);
  LAUNCH_CHECK(ctx);
  int32_t panic_node = 0x7fffffff;
  CUDA_TRY(ctx, cudaMemcpyAsync(&panic_node, d_flags + 1, 4, cudaMemcpyDeviceToHost, st));
  CUDA_TRY(ctx, cudaMemcpyAsync(out_dist, d_dist, (size_t)V * 8, cudaMemcpyDeviceToHost, st));
  CUDA_TRY(ctx, cudaStreamSynchronize(st));
  if (out_sweeps) *out_sweeps = sweeps;
  if (panic_node != 0x7fffffff)
    return porrt_fail(ctx, PORRT_ERR_PANIC, node_type[panic_node] == PORRT_NODE_OBSERVATION
                                                ? "assert!(p > 0.0) at belief node " + std::to_string(panic_node) + " (belief_graph.rs:130)"
                                                : "node type should be know at this stage! belief node " + std::to_string(panic_node) + " (belief_graph.rs:140)");
  return PORRT_OK;
}

// extract_policy + get_best_expected_children (belief_graph.rs:184-267): host walk over the device result, touching only the
// policy's own nodes.  Policy nodes in creation order: out_belief_node[k] (id in the belief graph), out_parent[k] (-1 root).
PORRT_API int32_t porrt_extract_policy_graph(porrt_ctx* ctx, int64_t V, const int64_t* row_ptr, const int32_t* col, const double* xy,
                                             const uint8_t* node_type, const int32_t* belief_id, const double* beliefs, int32_t B,
                                             int32_t n_worlds, const double* dist, int32_t* out_belief_node, int32_t* out_parent,
                                             uint8_t* out_is_leaf, int64_t cap, int64_t* out_n, double* out_expected_cost) {
  return porrt_extract_policy_graph_nd(ctx, 2, V, row_ptr, col, xy, node_type, belief_id, beliefs, B, n_worlds, dist, out_belief_node, out_parent,
                                       out_is_leaf, cap, out_n, out_expected_cost);
}

PORRT_API int32_t porrt_extract_policy_graph_nd(porrt_ctx* ctx, int32_t dim, int64_t V, const int64_t* row_ptr, const int32_t* col,
                                                const double* xy, const uint8_t* node_type, const int32_t* belief_id, const double* beliefs,
                                                int32_t B, int32_t n_worlds, const double* dist, int32_t* out_belief_node, int32_t* out_parent,
                                                uint8_t* out_is_leaf, int64_t cap, int64_t* out_n, double* out_expected_cost) {
  CTX_CHECK(ctx);
  if (V <= 0) return porrt_fail(ctx, PORRT_ERR_PANIC, "no belief state graph! (belief_graph.rs:186)");
  if (!dist || !graph_args_ok(V, row_ptr, col, xy, node_type, belief_id, beliefs, B, n_worlds, dim))
    return porrt_fail(ctx, PORRT_ERR_INVALID_ARG, "extract_policy_graph: bad arguments");
  std::vector<PolicyNode> pol;
  const int32_t rc = get_best_expected_children(
      ctx, "extract_policy_graph", V, beliefs, n_worlds,
      [&](int64_t id, auto&& fn) { for (int64_t e = row_ptr[id]; e < row_ptr[id + 1]; ++e) fn((int64_t)col[e]); },
      [&](int64_t id) { return belief_id[id]; },
      [&](int64_t a, int64_t c) { return norm2(xy + dim * a, xy + dim * c, dim); },
      [&](int64_t id) { return dist[id]; }, pol);
  if (rc) return rc;
  if (out_n) *out_n = (int64_t)pol.size();
  if (out_expected_cost) *out_expected_cost = dist[0];
  if ((int64_t)pol.size() > cap || !out_belief_node || !out_parent || !out_is_leaf)
    return porrt_fail(ctx, PORRT_ERR_CAPACITY, "extract_policy_graph: cap too small");
  for (size_t k = 0; k < pol.size(); ++k) { out_belief_node[k] = (int32_t)pol[k].id; out_parent[k] = pol[k].parent; out_is_leaf[k] = pol[k].leaf; }
  return PORRT_OK;
}
