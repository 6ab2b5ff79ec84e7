// mmprm.cu -- the multi-modal PRM of the reference's TAMP baseline (src/map_shelves_tamp_prm.rs), SURVEY.md 8(f) rank 3.
//
// MapShelfDomainTampPRM::plan (:308-326) = grow_mm_prm (:328-397: one PRM per belief "mode", grown in batches of 190 samples, plus
// observation samples that are added to a mode and to its successor modes) -> build_belief_graph (:399-473) ->
// conditional_dijkstra -> extract_policy.  Nothing in the growth depends on validity results: which mode grows, which zone is
// observed and every sample are decided by the RNG streams alone.  The caller (the Rust side, which owns the samplers and the
// mode tree) therefore hands over the SCHEDULE -- per mode the add_sample calls in order (state, max_step, search_radius), the
// mode transitions with their (observation node, destination node) pairs, the final nodes -- and this file does the work:
//   1. the PRMs of ALL modes as one grouped, batched build (prm_build_impl: one prefix- and group-restricted radius batch, one edge
//      batch, one CSR; graph.cu);
//   2. the explicit belief graph in the reference's node / edge order (mode after mode; observation edges in transition order;
//      action edges = PRM children, skipped for Observation nodes);
//   3. porrt_conditional_dijkstra on it (belief_explicit.cu).
// porrt_mmprm_fetch_graph returns the assembled graph for porrt_extract_policy_graph.
#include <chrono>

#include "common.cuh"

static double mm_now_ms() {
  return std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now().time_since_epoch()).count();
}

PORRT_API int32_t porrt_mmprm_plan(porrt_ctx* ctx, int32_t n_modes, const int64_t* mode_node_ptr, const double* samples_xy,
                                   const double* max_step, const double* search_radius, const int32_t* mode_belief_id,
                                   const double* beliefs, int32_t B, int32_t n_worlds, int32_t n_transitions,
                                   const int32_t* tr_from_mode, const int32_t* tr_to_mode, const int64_t* tr_pair_ptr,
                                   const int32_t* tr_pairs, const int64_t* mode_final_ptr, const int32_t* mode_final_nodes,
                                   double* out_dist, int64_t* out_n_edges, int32_t* out_sweeps, double* out_phase_ms) {
  CTX_CHECK(ctx);
  if (!ctx->has_map) return porrt_fail(ctx, PORRT_ERR_NO_MAP, "no map uploaded");
  if (n_modes <= 0 || !mode_node_ptr || !samples_xy || !max_step || !search_radius || !mode_belief_id || !beliefs || B <= 0 ||
      n_worlds <= 0 || n_transitions < 0 || (n_transitions > 0 && (!tr_from_mode || !tr_to_mode || !tr_pair_ptr)) || !mode_final_ptr || !out_dist)
    return porrt_fail(ctx, PORRT_ERR_INVALID_ARG, "mmprm_plan: bad arguments");
  const int64_t T = mode_node_ptr[n_modes];
  if (T <= 0 || T > 0x7fffffff) return porrt_fail(ctx, PORRT_ERR_INVALID_ARG, "mmprm_plan: node count out of range");
  for (int m = 0; m < n_modes; ++m)
    if (mode_node_ptr[m + 1] < mode_node_ptr[m] || mode_belief_id[m] < 0 || mode_belief_id[m] >= B || mode_final_ptr[m + 1] < mode_final_ptr[m])
      return porrt_fail(ctx, PORRT_ERR_INVALID_ARG, "mmprm_plan: bad mode table");
  double t0 = mm_now_ms(), t1, ph[4] = {0};

  // 1. the PRMs of all modes in ONE grouped build (prm_build_impl, graph.cu): one binning, one radius batch, one edge batch, one
  //    CSR over global node ids; a node only sees earlier nodes of its own mode.  (Per-mode calls cost ~1 ms of launch latency
  //    each: 66 ms for 63 modes against ~4 ms for the grouped build.)
  CUDA_TRY(ctx, ctx->pin_row.ensure((size_t)(T + 1) * 8));   // pinned staging: the CSR comes back by DMA, not through pageable copies
  int64_t* rp = ctx->pin_row.as<int64_t>();
  const int32_t* cl = nullptr;
  int64_t ne = 0;
  {
    double prm_ph[8] = {0};
    int32_t rc = prm_build_impl(ctx, samples_xy, T, 0.0, 0.0, max_step, search_radius, rp, nullptr, 0, &ne, prm_ph, mode_node_ptr, n_modes);
    if (rc != PORRT_OK && rc != PORRT_ERR_CAPACITY) return rc;
    for (int k = 0; k < 7; ++k) ctx->last_ms[k] = prm_ph[k];   // porrt_ctx_last_phase_ms: [radii, bin, radius, kd_rank, order, edges, csr]
    ctx->n_last = 7;
    CUDA_TRY(ctx, ctx->pin_col.ensure((size_t)std::max<int64_t>(ne, 1) * 4));
    if (ne > 0) {
      rc = porrt_prm_fetch(ctx, nullptr, ctx->pin_col.as<int32_t>(), ne);
      if (rc) return rc;
    }
    cl = ctx->pin_col.as<int32_t>();
  }
  t1 = mm_now_ms(); ph[0] = t1 - t0; t0 = t1;

  // 2. belief graph (build_belief_graph, :399-473): belief node id = mode_node_ptr[mode] + PRM node id
  // observation edges per belief node as a CSR in transition order (a vector per node cost 3 ms of allocations at 1.7e5 nodes)
  std::vector<int64_t> obs_ptr((size_t)T + 1, 0);
  for (int t = 0; t < n_transitions; ++t) {
    const int fm = tr_from_mode[t], tm = tr_to_mode[t];
    if (fm < 0 || fm >= n_modes || tm < 0 || tm >= n_modes) return porrt_fail(ctx, PORRT_ERR_INVALID_ARG, "mmprm_plan: transition mode out of range");
    for (int64_t q = tr_pair_ptr[t]; q < tr_pair_ptr[t + 1]; ++q) {
      const int64_t from = mode_node_ptr[fm] + tr_pairs[2 * q], to = mode_node_ptr[tm] + tr_pairs[2 * q + 1];
      if (tr_pairs[2 * q] < 0 || from >= mode_node_ptr[fm + 1] || tr_pairs[2 * q + 1] < 0 || to >= mode_node_ptr[tm + 1])
        return porrt_fail(ctx, PORRT_ERR_INVALID_ARG, "mmprm_plan: observation pair out of range");
      ++obs_ptr[(size_t)from + 1];
    }
  }
  for (int64_t u = 0; u < T; ++u) obs_ptr[(size_t)u + 1] += obs_ptr[(size_t)u];
  std::vector<int32_t> obs_to((size_t)obs_ptr[(size_t)T]);
  {
    std::vector<int64_t> fill(obs_ptr.begin(), obs_ptr.end() - 1);
    for (int t = 0; t < n_transitions; ++t)
      for (int64_t q = tr_pair_ptr[t]; q < tr_pair_ptr[t + 1]; ++q)
        obs_to[(size_t)fill[(size_t)(mode_node_ptr[tr_from_mode[t]] + tr_pairs[2 * q])]++] = (int32_t)(mode_node_ptr[tr_to_mode[t]] + tr_pairs[2 * q + 1]);
  }
  auto& G = ctx->mm;
  G.row_ptr.assign((size_t)T + 1, 0); G.type.assign((size_t)T, PORRT_NODE_ACTION); G.belief_id.resize((size_t)T);
  for (int m = 0; m < n_modes; ++m)
    for (int64_t u = mode_node_ptr[m]; u < mode_node_ptr[m + 1]; ++u) {
      G.belief_id[(size_t)u] = mode_belief_id[m];
      const int64_t n_obs = obs_ptr[(size_t)u + 1] - obs_ptr[(size_t)u];
      if (n_obs > 0) G.type[(size_t)u] = PORRT_NODE_OBSERVATION;
      G.row_ptr[(size_t)u + 1] = G.row_ptr[(size_t)u] + (n_obs > 0 ? n_obs : rp[u + 1] - rp[u]);
    }
  G.col.resize((size_t)G.row_ptr[(size_t)T]);
  for (int64_t u = 0; u < T; ++u) {
    int32_t* dst = G.col.data() + G.row_ptr[(size_t)u];
    if (G.type[(size_t)u] == PORRT_NODE_OBSERVATION) memcpy(dst, obs_to.data() + obs_ptr[(size_t)u], (size_t)(obs_ptr[(size_t)u + 1] - obs_ptr[(size_t)u]) * 4);
    else if (rp[u + 1] > rp[u]) memcpy(dst, cl + rp[u], (size_t)(rp[u + 1] - rp[u]) * 4);   // PRM children, already global ids
  }
  std::vector<int32_t> finals;
  for (int m = 0; m < n_modes; ++m)
    for (int64_t f = mode_final_ptr[m]; f < mode_final_ptr[m + 1]; ++f) {
      const int64_t u = mode_node_ptr[m] + mode_final_nodes[f];
      if (mode_final_nodes[f] < 0 || u >= mode_node_ptr[m + 1]) return porrt_fail(ctx, PORRT_ERR_INVALID_ARG, "mmprm_plan: final node out of range");
      finals.push_back((int32_t)u);
    }
  if (out_n_edges) *out_n_edges = (int64_t)G.col.size();
  t1 = mm_now_ms(); ph[1] = t1 - t0; t0 = t1;

  // 3. expected costs to the goals
  int32_t rc = porrt_conditional_dijkstra(ctx, T, G.row_ptr.data(), G.col.data(), samples_xy, G.type.data(), G.belief_id.data(), beliefs, B,
                                          n_worlds, finals.data(), (int32_t)finals.size(), out_dist, out_sweeps);
  t1 = mm_now_ms(); ph[2] = t1 - t0;
  if (out_phase_ms) memcpy(out_phase_ms, ph, sizeof(ph));
  return rc;
}

PORRT_API int32_t porrt_mmprm_fetch_graph(porrt_ctx* ctx, int64_t* out_row_ptr, int32_t* out_col, int64_t cap, uint8_t* out_node_type,
                                          int32_t* out_belief_id) {
  CTX_CHECK(ctx);
  auto& G = ctx->mm;
  if (G.row_ptr.empty()) return porrt_fail(ctx, PORRT_ERR_INVALID_ARG, "mmprm_fetch_graph: run porrt_mmprm_plan first");
  if (cap < (int64_t)G.col.size()) return porrt_fail(ctx, PORRT_ERR_CAPACITY, "mmprm_fetch_graph: out_col too small");
  if (out_row_ptr) memcpy(out_row_ptr, G.row_ptr.data(), G.row_ptr.size() * 8);
  if (out_col && !G.col.empty()) memcpy(out_col, G.col.data(), G.col.size() * 4);
  if (out_node_type) memcpy(out_node_type, G.type.data(), G.type.size());
  if (out_belief_id) memcpy(out_belief_id, G.belief_id.data(), G.belief_id.size() * 4);
  return PORRT_OK;
}
