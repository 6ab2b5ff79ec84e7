// refine.cu -- the policy refiner's data-parallel part (SURVEY.md 8(f) rank 1).
//
//  * porrt_transition_valid : PTOPolicyRefiner::is_transition_valid (reference src/pto_policy_refiner.rs:395-423), batched:
//                             state validity of both ends + transition validity + belief/validity compatibility.
//  * porrt_partial_shortcut : PTOPolicyRefiner::partial_shortcut (:158-206) on path pieces.  The reference runs n_iterations
//                             SEQUENTIAL trials per piece, each a handful of short edge checks whose outcome decides what the
//                             next trial sees -- a device round trip per trial (or per speculative wave of trials: round 1,
//                             157-250 round trips, slower than one CPU core on small maps) cannot win.  So the whole loop runs
//                             ON the device: one CTA per piece keeps the path in shared memory and works through the trial list
//                             (joint, interval: drawn on the host from a fresh DiscreteSampler, they depend on the piece length
//                             only); per trial its warps check the transitions of the shortcut in parallel (state validity of
//                             both ends, warp-cooperative edge walk, belief/validity compatibility), then the CTA applies the
//                             reference's short-circuit `&&` chain in order and commits or not.  Pieces run side by side on
//                             different SMs; there is no host round trip inside a call.
// The sampler is rand_pcg 0.3 Pcg64 (Lcg128Xsl64) seeded by rand_core 0.6 seed_from_u64 and rand 0.8's
// UniformInt<usize>::sample_single, restated from their published algorithms (the crates are not vendored in the reference).
#include <algorithm>
#include <chrono>
#include <cstring>
#include <unordered_set>

#include "pcg64.h"
#include "common.cuh"
#include "map_dev.cuh"

// ------------------------------------------------------------------------------------------------ device
// valid / status from the three validity codes, in the reference's evaluation order
// compat: rows of n_validities bytes; row[i] (nullable: row 0) selects the belief state of transition i
__global__ void transition_combine_kernel(const int32_t* __restrict__ sv_from, const int32_t* __restrict__ sv_to,
                                          const int32_t* __restrict__ ev, const uint8_t* __restrict__ compat,
                                          const int32_t* __restrict__ row, int32_t n_validities, int64_t n,
                                          uint8_t* __restrict__ out_valid, int32_t* __restrict__ out_status) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const int32_t f = sv_from[i], t = sv_to[i], e = ev[i];
  int32_t status = 0;
  uint8_t valid = 0;
  if (f < -1) status = f;                 // state_validity(from) panics first (:396)
  else if (t < -1) status = t;            // then state_validity(to) (:397)
  else if (f >= 0 && t >= 0) {            // only then is the transition looked at (:399-414)
    if (e < -1) status = e;
    else if (e >= 0) valid = compat[(row ? (int64_t)row[i] * n_validities : 0) + e] ? 1 : 0;
  }
  out_valid[i] = valid;
  if (out_status) out_status[i] = status;
}

// device buffers in, device buffers out; d_tmp: 3 * n int32
static int32_t transition_valid_dev(porrt_ctx* ctx, const double* d_from, const double* d_to, int64_t n, const uint8_t* d_compat,
                                    const int32_t* d_row, int32_t n_validities, int32_t* d_tmp, uint8_t* d_valid, int32_t* d_status) {
  cudaStream_t st = ctx->stream;
  int32_t rc = porrt_state_validity_dev(ctx, d_from, n, d_tmp);
  if (rc) return rc;
  rc = porrt_state_validity_dev(ctx, d_to, n, d_tmp + n);
  if (rc) return rc;
  rc = map_edge_validity_dev(ctx, d_from, d_to, n, d_tmp + 2 * n, nullptr, st);
  if (rc) return rc;
  transition_combine_kernel<<<div_up(n, 256), 256, 0, st>>>(d_tmp, d_tmp + n, d_tmp + 2 * n, d_compat, d_row, n_validities, n, d_valid, d_status);
  LAUNCH_CHECK(ctx);
  return PORRT_OK;
}

PORRT_API int32_t porrt_transition_valid(porrt_ctx* ctx, const double* from_xy, const double* to_xy, int64_t n,
                                         const uint8_t* compat_row, uint8_t* out_valid, int32_t* out_status) {
  CTX_CHECK(ctx);
  if (!ctx->has_map) return porrt_fail(ctx, PORRT_ERR_NO_MAP, "no map uploaded");
  if (n < 0 || (n > 0 && (!from_xy || !to_xy || !compat_row || !out_valid))) return porrt_fail(ctx, PORRT_ERR_INVALID_ARG, "porrt_transition_valid: bad arguments");
  if (n == 0) return PORRT_OK;
  CUDA_TRY(ctx, cudaSetDevice(ctx->device));
  cudaStream_t st = ctx->stream;
  const size_t nv = (size_t)ctx->n_validities;
  double *d_from, *d_to;
  int32_t *d_tmp, *d_status;
  uint8_t *d_valid, *d_compat;
  CUDA_TRY(ctx, carve(ctx->ws_main, [&](Carve& c) {
    d_from = c.take<double>(2 * n); d_to = c.take<double>(2 * n); d_tmp = c.take<int32_t>(3 * n); d_status = c.take<int32_t>(n);
    d_valid = c.take<uint8_t>(n); d_compat = c.take<uint8_t>(nv);
  }));
  CUDA_TRY(ctx, cudaMemcpyAsync(d_from, from_xy, (size_t)n * 16, cudaMemcpyHostToDevice, st));
  CUDA_TRY(ctx, cudaMemcpyAsync(d_to, to_xy, (size_t)n * 16, cudaMemcpyHostToDevice, st));
  CUDA_TRY(ctx, cudaMemcpyAsync(d_compat, compat_row, nv, cudaMemcpyHostToDevice, st));
  int32_t rc = transition_valid_dev(ctx, d_from, d_to, n, d_compat, nullptr, (int32_t)nv, d_tmp, d_valid, d_status);
  if (rc) return rc;
  CUDA_TRY(ctx, cudaMemcpyAsync(out_valid, d_valid, (size_t)n, cudaMemcpyDeviceToHost, st));
  if (out_status) CUDA_TRY(ctx, cudaMemcpyAsync(out_status, d_status, (size_t)n * 4, cudaMemcpyDeviceToHost, st));
  CUDA_TRY(ctx, cudaStreamSynchronize(st));
  return PORRT_OK;
}

// ------------------------------------------------------------------------------------------------ the trial loop on the device
#define SHORTCUT_MAX_STATES 1024      // states of one piece (shared memory: path + shortcut states + per-transition results)
#define SHORTCUT_THREADS 128

// trial = joint | a << 1 | b << 16 (a, b < 1024)
template <int KIND>
__global__ void __launch_bounds__(SHORTCUT_THREADS) shortcut_loop_kernel(MapDev m, double2* __restrict__ states, const int32_t* __restrict__ piece_ptr,
                                                                         const int32_t* __restrict__ piece_list, const uint32_t* __restrict__ trials,
                                                                         int n_iterations, const uint8_t* __restrict__ compat_rows, int n_validities,
                                                                         int32_t* __restrict__ out_commits, int32_t* __restrict__ out_status) {
  __shared__ double2 s_path[SHORTCUT_MAX_STATES];
  __shared__ double2 s_cut[SHORTCUT_MAX_STATES];
  __shared__ int32_t s_res[SHORTCUT_MAX_STATES];   // per transition: 1 valid, 0 invalid, < -1 the panic its check hits
  __shared__ int32_t s_decision;
  const int piece = piece_list[blockIdx.x];
  const int p0 = piece_ptr[piece], L = piece_ptr[piece + 1] - p0;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, n_warps = SHORTCUT_THREADS / 32;
  const uint8_t* compat = compat_rows + (size_t)piece * n_validities;
  const uint32_t* my_trials = trials + (size_t)blockIdx.x * n_iterations;
  for (int j = tid; j < L; j += SHORTCUT_THREADS) s_path[j] = states[p0 + j];
  __syncthreads();
  int commits = 0, panic = 0;
  for (int it = 0; it < n_iterations; ++it) {
    const uint32_t t = my_trials[it];
    const int joint = (int)(t & 1u), a = (int)((t >> 1) & 0x7fffu), b = (int)(t >> 16);
    const int n_tr = b - a;                                  // transitions: cut[0]->cut[1] .. cut[n-2]->cut[n-1], cut[n-1]->path[b]
    // shortcut states: state j with its `joint` coordinate interpolated between the interval's ends (:182-190)
    const double sa = joint ? s_path[a].y : s_path[a].x, sb = joint ? s_path[b].y : s_path[b].x;
    for (int j = a + tid; j < b; j += SHORTCUT_THREADS) {
      const double lambda = __ddiv_rn((double)(j - a), (double)(b - a));
      const double v = __dadd_rn(__dmul_rn(sa, __dsub_rn(1.0, lambda)), __dmul_rn(sb, lambda));   // a * (1 - lambda) + b * lambda (:160)
      double2 s = s_path[j];
      if (joint) s.y = v; else s.x = v;
      s_cut[j - a] = s;
    }
    __syncthreads();
    // is_transition_valid of every transition (:395-423), one warp each
    for (int k = warp; k < n_tr; k += n_warps) {
      const double2 from = s_cut[k], to = k + 1 < n_tr ? s_cut[k + 1] : s_path[b];
      const int32_t f = state_validity_of(m, from.x, from.y), g = state_validity_of(m, to.x, to.y);
      int32_t res = 0;
      if (f < -1) res = f;                 // state_validity(from) panics first (:396)
      else if (g < -1) res = g;            // then state_validity(to) (:397)
      else if (f >= 0 && g >= 0) {         // only then is the transition looked at (:399-414)
        const EdgeSetup es = make_setup(m, from.x, from.y, to.x, to.y);
        const int32_t e = walk_to_validity(m, walk_warp<KIND>(m, es, lane));
        if (e < -1) res = e;
        else if (e >= 0) res = compat[e] ? 1 : 0;
      }
      if (lane == 0) s_res[k] = res;
    }
    __syncthreads();
    // should_commit = t_0 && t_1 && ... (:193-197): the chain stops at the first false, a panic counts only if it is reached
    if (warp == 0) {
      int decision = 1;
      for (int k0 = 0; k0 < n_tr && decision == 1; k0 += 32) {
        const int k = k0 + lane;
        const int32_t r = k < n_tr ? s_res[k] : 1;
        const unsigned stop = __ballot_sync(0xffffffffu, r != 1);
        if (stop) decision = __shfl_sync(0xffffffffu, r, __ffs(stop) - 1);   // 0: no commit, < -1: the reference panics here
      }
      if (lane == 0) s_decision = decision;
    }
    __syncthreads();
    const int decision = s_decision;
    if (decision < -1) { panic = decision; break; }
    if (decision == 1) {                                                     // :200-204
      for (int j = a + tid; j < b; j += SHORTCUT_THREADS) s_path[j] = s_cut[j - a];
      ++commits;
    }
    __syncthreads();
  }
  for (int j = tid; j < L; j += SHORTCUT_THREADS) states[p0 + j] = s_path[j];
  if (tid == 0) { out_commits[piece] = commits; out_status[piece] = panic; }
}

PORRT_API int32_t porrt_partial_shortcut_batch(porrt_ctx* ctx, double* states_xy, const int32_t* piece_ptr, int32_t n_pieces,
                                               const uint8_t* compat_rows, int32_t n_iterations, uint64_t sampler_seed,
                                               int32_t* out_commits, int32_t* out_waves) {
  CTX_CHECK(ctx);
  if (!ctx->has_map) return porrt_fail(ctx, PORRT_ERR_NO_MAP, "no map uploaded");
  if (n_pieces < 0 || n_iterations < 0 || (n_pieces > 0 && (!states_xy || !piece_ptr || !compat_rows)))
    return porrt_fail(ctx, PORRT_ERR_INVALID_ARG, "porrt_partial_shortcut_batch: bad arguments");
  if (out_waves) *out_waves = 0;
  if (out_commits) std::fill(out_commits, out_commits + n_pieces, 0);   // every entry, also when a later piece is refused
  for (int p = 0; p < n_pieces; ++p) {
    if (piece_ptr[p + 1] < piece_ptr[p] || piece_ptr[p] < 0) return porrt_fail(ctx, PORRT_ERR_INVALID_ARG, "porrt_partial_shortcut_batch: piece_ptr must be non-decreasing");
    if (piece_ptr[p + 1] - piece_ptr[p] > SHORTCUT_MAX_STATES) return porrt_fail(ctx, PORRT_ERR_UNSUPPORTED, "porrt_partial_shortcut_batch: a piece has more than 1024 states");
  }
  if (n_pieces == 0 || n_iterations == 0) return PORRT_OK;
  CUDA_TRY(ctx, cudaSetDevice(ctx->device));
  cudaStream_t st = ctx->stream;
  const size_t nv = (size_t)ctx->n_validities;
  // every piece draws the same kind of sequence from a fresh sampler (:169 DiscreteSampler::new()): joint, interval start,
  // interval end (:172-174) depend on the piece length only, so the whole trial list is known before anything is checked
  std::vector<int32_t> list;
  std::vector<uint32_t> trials;
  for (int p = 0; p < n_pieces; ++p) {
    const int L = piece_ptr[p + 1] - piece_ptr[p];
    if (L <= 2) continue;              // :163-165: can't shortcut with only 2 states or less
    list.push_back(p);
    Pcg64 rng = Pcg64::seed_from_u64(sampler_seed);
    for (int i = 0; i < n_iterations; ++i) {
      const uint32_t joint = (uint32_t)rng.below(2);
      const uint32_t a = (uint32_t)rng.below((uint64_t)(L - 2));
      const uint32_t b = a + 2 + (uint32_t)rng.below((uint64_t)(L - a - 2));
      trials.push_back(joint | (a << 1) | (b << 16));
    }
  }
  if (list.empty()) return PORRT_OK;
  const int64_t n_states = piece_ptr[n_pieces];
  const size_t n_active = list.size();
  double2* d_states;
  int32_t *d_ptr, *d_list, *d_commits, *d_status;
  uint32_t* d_trials;
  uint8_t* d_compat;
  CUDA_TRY(ctx, carve(ctx->ws_main, [&](Carve& c) {
    d_states = c.take<double2>(n_states); d_ptr = c.take<int32_t>(n_pieces + 1); d_list = c.take<int32_t>(n_active);
    d_trials = c.take<uint32_t>(trials.size()); d_compat = c.take<uint8_t>((size_t)n_pieces * nv);
    d_commits = c.take<int32_t>(n_pieces);
    d_status = c.take<int32_t>(n_pieces + 4);   // + 16 bytes: the memset below clears commits and status in one call
  }));
  CUDA_TRY(ctx, cudaMemcpyAsync(d_states, states_xy, (size_t)n_states * 16, cudaMemcpyHostToDevice, st));
  CUDA_TRY(ctx, cudaMemcpyAsync(d_ptr, piece_ptr, (size_t)(n_pieces + 1) * 4, cudaMemcpyHostToDevice, st));
  CUDA_TRY(ctx, cudaMemcpyAsync(d_list, list.data(), n_active * 4, cudaMemcpyHostToDevice, st));
  CUDA_TRY(ctx, cudaMemcpyAsync(d_trials, trials.data(), trials.size() * 4, cudaMemcpyHostToDevice, st));
  CUDA_TRY(ctx, cudaMemcpyAsync(d_compat, compat_rows, (size_t)n_pieces * nv, cudaMemcpyHostToDevice, st));
  CUDA_TRY(ctx, cudaMemsetAsync(d_commits, 0, (size_t)n_pieces * 8 + 16, st));   // commits and status (adjacent, 16-byte aligned)
  if (ctx->map.kind == PORRT_DOMAIN_SHELF)
    shortcut_loop_kernel<PORRT_DOMAIN_SHELF><<<(int)n_active, SHORTCUT_THREADS, 0, st>>>(ctx->map, d_states, d_ptr, d_list, d_trials, n_iterations, d_compat, (int)nv, d_commits, d_status);
  else
    shortcut_loop_kernel<PORRT_DOMAIN_DOOR><<<(int)n_active, SHORTCUT_THREADS, 0, st>>>(ctx->map, d_states, d_ptr, d_list, d_trials, n_iterations, d_compat, (int)nv, d_commits, d_status);
  LAUNCH_CHECK(ctx);
  std::vector<int32_t> commits((size_t)n_pieces), status((size_t)n_pieces);
  std::vector<double> refined((size_t)n_states * 2);
  CUDA_TRY(ctx, cudaMemcpyAsync(refined.data(), d_states, (size_t)n_states * 16, cudaMemcpyDeviceToHost, st));
  CUDA_TRY(ctx, cudaMemcpyAsync(commits.data(), d_commits, (size_t)n_pieces * 4, cudaMemcpyDeviceToHost, st));
  CUDA_TRY(ctx, cudaMemcpyAsync(status.data(), d_status, (size_t)n_pieces * 4, cudaMemcpyDeviceToHost, st));
  CUDA_TRY(ctx, cudaStreamSynchronize(st));
  if (out_waves) *out_waves = 1;       // device round trips of the call
  for (int p = 0; p < n_pieces; ++p)
    if (status[(size_t)p] < -1)        // the caller's states stay untouched, like a panic leaves nothing behind
      return porrt_fail(ctx, PORRT_ERR_PANIC, "partial_shortcut: a transition check hit a reference panic (code " + std::to_string(status[(size_t)p]) + ")");
  memcpy(states_xy, refined.data(), (size_t)n_states * 16);
  if (out_commits) memcpy(out_commits, commits.data(), (size_t)n_pieces * 4);
  return PORRT_OK;
}

PORRT_API int32_t porrt_partial_shortcut(porrt_ctx* ctx, double* states_xy, int32_t n_states, const uint8_t* compat_row,
                                         int32_t n_iterations, uint64_t sampler_seed, int32_t* out_commits, int32_t* out_waves) {
  if (n_states < 0) return porrt_fail(ctx, PORRT_ERR_INVALID_ARG, "porrt_partial_shortcut: bad arguments");
  const int32_t ptr[2] = {0, n_states};
  return porrt_partial_shortcut_batch(ctx, states_xy, ptr, 1, compat_row, n_iterations, sampler_seed, out_commits, out_waves);
}

// Policy::decompose (common.rs:85-129) over flat arrays: a policy as parent[] per node in creation order (parent[0] = -1, parent[k] < k;
// the children of a node in add_edge order = its later nodes in increasing index).  FIFO over piece starts; a piece runs until a leaf
// or a branching node.  piece_ptr / piece_nodes: the pieces back to back; successors[p]: the pieces that start at p's branching.
static void policy_decompose_flat(const int32_t* parent, int64_t n_pol, std::vector<int32_t>& piece_ptr, std::vector<int64_t>& piece_nodes,
                                  std::vector<std::vector<int32_t>>& successors) {
  std::vector<int64_t> ch_ptr((size_t)n_pol + 1, 0);
  for (int64_t k = 1; k < n_pol; ++k) ++ch_ptr[(size_t)parent[k] + 1];
  for (int64_t k = 0; k < n_pol; ++k) ch_ptr[(size_t)k + 1] += ch_ptr[(size_t)k];
  std::vector<int64_t> ch((size_t)std::max<int64_t>(n_pol - 1, 0)), fill(ch_ptr.begin(), ch_ptr.end() - 1);
  for (int64_t k = 1; k < n_pol; ++k) ch[(size_t)fill[(size_t)parent[k]]++] = k;
  piece_ptr.assign(1, 0); piece_nodes.clear(); successors.clear();
  std::vector<int64_t> fifo(1, 0);
  int32_t n_pieces = 0;
  for (size_t head = 0; head < fifo.size(); ++head) {
    int64_t cur = fifo[head];
    std::vector<int32_t> succ;
    for (;;) {
      piece_nodes.push_back(cur);
      const int64_t nc = ch_ptr[(size_t)cur + 1] - ch_ptr[(size_t)cur];
      if (nc == 0) break;
      if (nc == 1) { cur = ch[(size_t)ch_ptr[(size_t)cur]]; continue; }
      for (int64_t e = ch_ptr[(size_t)cur]; e < ch_ptr[(size_t)cur + 1]; ++e) { fifo.push_back(ch[(size_t)e]); succ.push_back(++n_pieces); }
      break;
    }
    piece_ptr.push_back((int32_t)piece_nodes.size());
    successors.push_back(succ);
  }
}
static bool policy_parents_ok(const int32_t* parent, int64_t n) {
  if (n <= 0 || !parent || parent[0] != -1) return false;
  for (int64_t k = 1; k < n; ++k) if (parent[k] < 0 || parent[k] >= k) return false;
  return true;
}

// Policy::compute_expected_costs_to_goals (common.rs:131-153) over flat arrays: a policy as (state, belief, parent) per node in
// creation order; children are folded in increasing index, a child's own sum is complete before its parent adds it.
static double policy_expected_cost_flat(const double* beliefs, int nw, const double* out_xy, const int32_t* out_belief, const int32_t* out_parent, int64_t n_out) {
  std::vector<double> prob((size_t)n_out, 0.0), pq((size_t)n_out, 0.0), edge_term((size_t)n_out, 0.0), below((size_t)n_out, 0.0);
  prob[0] = 1.0;
  for (int64_t k = 1; k < n_out; ++k) {
    const int32_t par = out_parent[k];
    if (par < 0) continue;   // a piece that recompose left unconnected: not under the root
    const double q = transition_probability(beliefs + (size_t)out_belief[par] * nw, beliefs + (size_t)out_belief[k] * nw, nw);
    const double cost = norm2(&out_xy[2 * (size_t)par], &out_xy[2 * k], 2);
    pq[(size_t)k] = prob[(size_t)par] * q;             // p * q
    prob[(size_t)k] = pq[(size_t)k];
    edge_term[(size_t)k] = pq[(size_t)k] * cost;        // (p * q) * cost
  }
  // expected_future_costs(parent) += p * q * cost + expected_future_costs(child), children in order (common.rs:149)
  std::vector<int64_t> oc_ptr((size_t)n_out + 1, 0);
  for (int64_t k = 0; k < n_out; ++k) if (out_parent[k] >= 0) ++oc_ptr[(size_t)out_parent[k] + 1];
  for (int64_t k = 0; k < n_out; ++k) oc_ptr[(size_t)k + 1] += oc_ptr[(size_t)k];
  std::vector<int64_t> oc((size_t)oc_ptr[(size_t)n_out]), ofill(oc_ptr.begin(), oc_ptr.end() - 1);
  for (int64_t k = 0; k < n_out; ++k) if (out_parent[k] >= 0) oc[(size_t)ofill[(size_t)out_parent[k]]++] = k;
  for (int64_t k = n_out - 1; k >= 0; --k) {
    double acc = 0.0;
    for (int64_t e = oc_ptr[(size_t)k]; e < oc_ptr[(size_t)k + 1]; ++e) { const int64_t c = oc[(size_t)e]; acc += edge_term[(size_t)c] + below[(size_t)c]; }
    below[(size_t)k] = acc;
  }
  return below[0];
}

// ================================================================================================ refine_solution(PartialShortCut(n))
// PTOPolicyRefiner::refine_solution with RefinmentStrategy::PartialShortCut (pto_policy_refiner.rs:85-133; what every PTO run of
// the reference's main.rs ends with, e.g. :442 PartialShortCut(1500)) on the policy porrt_extract_policy produced from the last
// porrt_belief_vi of this ctx:
//   Policy::decompose (common.rs:85-129)  ->  build_path_piece (:135-156) + partial_shortcut (:158-206) per piece, all pieces in one
//   batch on the device (porrt_partial_shortcut_batch)  ->  recompose (:324-393) incl. compute_expected_costs_to_goals (common.rs:131-153).
// Everything around the batch is sequential host logic, written here over flat arrays: a policy is (node, belief, parent) per policy
// node in creation order, children of a node = its later nodes in creation order (Policy::add_edge is called right after add_node).
// A piece of ONE node is a start but not an end in recompose (:356-361): its successors are never connected -- kept as is.
PORRT_API int32_t porrt_refine_policy_shortcut(porrt_ctx* ctx, const int32_t* pol_node, const int32_t* pol_belief, const int32_t* pol_parent,
                                               int64_t n_pol, int32_t n_iterations, uint64_t sampler_seed, double* out_xy, int32_t* out_node,
                                               int32_t* out_belief, int32_t* out_parent, uint8_t* out_is_leaf, int64_t cap, int64_t* out_n,
                                               double* out_expected_cost, int64_t* out_commits) {
  CTX_CHECK(ctx);
  auto& R = ctx->bel;
  if (R.V <= 0) return porrt_fail(ctx, PORRT_ERR_INVALID_ARG, "refine_policy_shortcut: run porrt_belief_vi / porrt_extract_policy first");
  if (n_pol <= 0 || !pol_node || !pol_belief || !pol_parent || n_iterations < 0 || !out_n)
    return porrt_fail(ctx, PORRT_ERR_INVALID_ARG, "refine_policy_shortcut: bad arguments");
  const int B = R.B, nw = R.n_worlds, nv = R.n_validities;
  for (int64_t k = 0; k < n_pol; ++k)
    if (pol_node[k] < 0 || pol_node[k] >= R.V || pol_belief[k] < 0 || pol_belief[k] >= B || pol_parent[k] >= k || (k > 0 && pol_parent[k] < 0) || (k == 0 && pol_parent[k] != -1))
      return porrt_fail(ctx, PORRT_ERR_INVALID_ARG, "refine_policy_shortcut: not a policy in creation order");
  // ---- decompose
  std::vector<int32_t> piece_ptr;
  std::vector<int64_t> piece_nodes;                   // policy node ids, piece after piece
  std::vector<std::vector<int32_t>> successors;       // skeleton
  policy_decompose_flat(pol_parent, n_pol, piece_ptr, piece_nodes, successors);
  const int32_t n_pieces = (int32_t)successors.size();
  const int64_t n_out = (int64_t)piece_nodes.size();   // every policy node ends up in exactly one piece
  *out_n = n_out;
  if (n_out > cap || !out_xy || !out_node || !out_belief || !out_parent || !out_is_leaf)
    return porrt_fail(ctx, PORRT_ERR_CAPACITY, "refine_policy_shortcut: cap too small");
  // ---- build_path_piece: the pieces' states back to back; the piece's belief is the one of its first node
  std::vector<uint8_t> rows((size_t)n_pieces * nv);
  for (int64_t k = 0; k < n_out; ++k) {
    const int64_t pn = piece_nodes[(size_t)k];
    out_xy[2 * k] = R.xy[2 * (size_t)pol_node[pn]]; out_xy[2 * k + 1] = R.xy[2 * (size_t)pol_node[pn] + 1];
    out_node[k] = pol_node[pn]; out_belief[k] = pol_belief[pn];
  }
  for (int32_t p = 0; p < n_pieces; ++p)
    memcpy(&rows[(size_t)p * nv], &R.compat[(size_t)pol_belief[piece_nodes[(size_t)piece_ptr[p]]] * nv], (size_t)nv);
  // ---- partial_shortcut on all pieces (device batch, sequential semantics)
  std::vector<int32_t> commits((size_t)n_pieces, 0);
  int32_t rc = porrt_partial_shortcut_batch(ctx, out_xy, piece_ptr.data(), n_pieces, rows.data(), n_iterations, sampler_seed, commits.data(), nullptr);
  if (rc) return rc;
  if (out_commits) { *out_commits = 0; for (int32_t c : commits) *out_commits += c; }
  // ---- recompose: chains inside the pieces, then end of piece i -> start of its successors (an end exists only for >= 2 nodes)
  for (int32_t p = 0; p < n_pieces; ++p)
    for (int32_t k = piece_ptr[p]; k < piece_ptr[p + 1]; ++k) out_parent[k] = k == piece_ptr[p] ? -1 : k - 1;
  for (int32_t p = 0; p < n_pieces; ++p) {
    if (piece_ptr[p + 1] - piece_ptr[p] < 2) continue;
    for (int32_t q : successors[(size_t)p]) out_parent[piece_ptr[q]] = piece_ptr[p + 1] - 1;
  }
  // children of the recomposed policy in add_edge order: the chain edge, or -- at a piece's end -- the successors in skeleton order
  // (successor pieces come later in the arrays, so increasing index = add_edge order); leaves = nodes without children
  std::vector<int32_t> n_children((size_t)n_out, 0);
  for (int64_t k = 0; k < n_out; ++k) if (out_parent[k] >= 0) ++n_children[(size_t)out_parent[k]];
  for (int64_t k = 0; k < n_out; ++k) out_is_leaf[k] = n_children[(size_t)k] == 0;
  if (out_expected_cost) *out_expected_cost = policy_expected_cost_flat(R.beliefs.data(), nw, out_xy, out_belief, out_parent, n_out);
  return PORRT_OK;
}

// ================================================================================================ refine_solution(Reparent(radius))
// PTOPolicyRefiner::refine_solution with RefinmentStrategy::Reparent (pto_policy_refiner.rs:85-133; main.rs:221,270 run Reparent(0.3))
// on the policy of the last porrt_belief_vi / porrt_extract_policy of this ctx.  Per path piece the reference
//   build_tree (:208-280)  grows a tree out of the piece: the path nodes, then every belief-graph descendant within `radius` of a path
//                          node (breadth first from each path node; quirks kept: distances and edge costs are measured from the SEED
//                          path node, and a grandchild enters the queue as a node whose CHILDREN are looked at next),
//   reparent (:282-322)    pops tree nodes by distance from the root and offers itself as parent to every tree node within
//                          radius / 2 it has a valid transition to (is_transition_valid, :395-423) -- label correcting, re-queueing,
// and recompose (:324-393) reads the new path leaf -> root.
// Here: the trees are built on the host from the retained belief-graph description (the implicit graph's children in the reference's
// order); the states of a tree never change, so EVERY (node, neighbour) pair reparent can ever test is known up front: all pairs of
// all pieces go through state validity + the edge kernel + the compatibility row in ONE device batch (the hot path; the reference
// re-evaluates them at every pop).  The label-correcting loop itself is sequential and cheap: host, over the precomputed answers,
// with the pop order of the reference's priority queue (priority-queue 1.0.5's indexed binary heap and Priority's never-Equal Ord,
// common.rs:231-251 -- restated from the published algorithm, parity unpinned: no test of the reference fixes the order among equal
// priorities, which do occur: Observation children share their parent's state).
// one warp per tree node u: the endpoints of its candidate transitions u -> v and the belief row of its piece
__global__ void reparent_pairs_kernel(const int64_t* __restrict__ nb_ptr, const int32_t* __restrict__ nb, const double2* __restrict__ xy,
                                      const int32_t* __restrict__ node_base, const int32_t* __restrict__ node_row, int64_t n_nodes,
                                      double2* __restrict__ from, double2* __restrict__ to, int32_t* __restrict__ row) {
  const int lane = threadIdx.x & 31;
  const int64_t u = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  if (u >= n_nodes) return;
  const double2 a = xy[u];
  const int32_t base = node_base[u], r = node_row[u];
  for (int64_t k = nb_ptr[u] + lane; k < nb_ptr[u + 1]; k += 32) { from[k] = a; to[k] = xy[base + nb[k]]; row[k] = r; }
}

namespace {
struct ReparentHeap {                   // see the comment above; lt / gt are Priority's `<` / `>`
  std::vector<int32_t> heap, pos;
  std::vector<double> prio;
  explicit ReparentHeap(size_t n) : pos(n, -1), prio(n, 0.0) {}
  static bool lt(double a, double b) { return !(a < b); }
  static bool gt(double a, double b) { return a < b; }
  void up(size_t i, int32_t item) {
    while (i > 0 && lt(prio[(size_t)heap[(i - 1) / 2]], prio[(size_t)item])) { heap[i] = heap[(i - 1) / 2]; pos[(size_t)heap[i]] = (int32_t)i; i = (i - 1) / 2; }
    heap[i] = item; pos[(size_t)item] = (int32_t)i;
  }
  void down(size_t i) {
    for (;;) {
      const size_t l = 2 * i + 1, r = l + 1;
      size_t big = (l < heap.size() && gt(prio[(size_t)heap[l]], prio[(size_t)heap[i]])) ? l : i;
      if (r < heap.size() && gt(prio[(size_t)heap[r]], prio[(size_t)heap[big]])) big = r;
      if (big == i) return;
      std::swap(heap[i], heap[big]);
      pos[(size_t)heap[i]] = (int32_t)i; pos[(size_t)heap[big]] = (int32_t)big;
      i = big;
    }
  }
  void push(int32_t item, double p) {
    prio[(size_t)item] = p;
    if (pos[(size_t)item] >= 0) { up((size_t)pos[(size_t)item], item); down((size_t)pos[(size_t)item]); return; }
    heap.push_back(item);
    up(heap.size() - 1, item);
  }
  int32_t pop() {
    const int32_t head = heap[0];
    pos[(size_t)head] = -1;
    heap[0] = heap.back();
    heap.pop_back();
    if (!heap.empty()) { pos[(size_t)heap[0]] = 0; down(0); }
    return head;
  }
};

struct PieceTree {
  std::vector<double> xy;               // 2 per tree node
  std::vector<int32_t> parent;          // -1 = root
  std::vector<double> parent_cost;
  std::vector<int64_t> bgid;            // belief-graph id = node * B + belief
  std::vector<int32_t> kd_left, kd_right;
  int32_t belief = 0, leaf = 0;
  size_t size() const { return parent.size(); }
  int32_t add(const double* s, int32_t par, double cost, int64_t id) {
    xy.push_back(s[0]); xy.push_back(s[1]); parent.push_back(par); parent_cost.push_back(cost); bgid.push_back(id);
    kd_left.push_back(-1); kd_right.push_back(-1);
    const int32_t me = (int32_t)size() - 1;
    if (me > 0) {                        // KdTree::add (nearest_neighbor.rs:29-46), kd node = tree node
      int32_t cur = 0;
      for (int axis = 0;; axis ^= 1) {
        int32_t& next = s[axis] < xy[2 * (size_t)cur + axis] ? kd_left[(size_t)cur] : kd_right[(size_t)cur];
        if (next >= 0) cur = next; else { next = me; break; }
      }
    }
    return me;
  }
  double dist_from_root(int32_t id) const {   // :53-62, summed from the node upwards
    double c = 0.0;
    for (int32_t k = id; parent[(size_t)k] >= 0; k = parent[(size_t)k]) c += parent_cost[(size_t)k];
    return c;
  }
  // nearest_neighbors (:94-126): ids in the reference's visit order
  struct F { int32_t node; int axis; int stage; };
  mutable std::vector<F> st;
  void radius(const double* s, double r, std::vector<int32_t>& out) const {
    st.assign(1, F{0, 0, 0});
    while (!st.empty()) {
      F& f = st.back();
      const double* fs = &xy[2 * (size_t)f.node];
      if (f.stage == 0 && norm2(s, fs, 2) <= r) out.push_back(f.node);   // norm2(from.state, a.state)
      if (f.stage >= 2) { st.pop_back(); continue; }
      const int stage = f.stage++, axis = f.axis;
      int32_t child = -1;
      if (stage == 0) { if (s[axis] - r <= fs[axis]) child = kd_left[(size_t)f.node]; }
      else { if (s[axis] + r >= fs[axis]) child = kd_right[(size_t)f.node]; }
      if (child >= 0) st.push_back(F{child, axis ^ 1, 0});
    }
  }
};
}  // namespace

PORRT_API int32_t porrt_refine_policy_reparent(porrt_ctx* ctx, const int32_t* pol_node, const int32_t* pol_belief, const int32_t* pol_parent,
                                               int64_t n_pol, double radius, double* out_xy, int32_t* out_node, int32_t* out_belief,
                                               int32_t* out_parent, uint8_t* out_is_leaf, int64_t cap, int64_t* out_n,
                                               double* out_expected_cost, int64_t* out_tree_nodes, int64_t* out_transitions) {
  CTX_CHECK(ctx);
  auto& R = ctx->bel;
  if (R.V <= 0) return porrt_fail(ctx, PORRT_ERR_INVALID_ARG, "refine_policy_reparent: run porrt_belief_vi / porrt_extract_policy first");
  if (!ctx->has_map) return porrt_fail(ctx, PORRT_ERR_NO_MAP, "no map uploaded");
  if (n_pol <= 0 || !pol_node || !pol_belief || !pol_parent || !(radius >= 0.0) || !out_n)
    return porrt_fail(ctx, PORRT_ERR_INVALID_ARG, "refine_policy_reparent: bad arguments");
  const int B = R.B, nw = R.n_worlds, nv = R.n_validities;
  for (int64_t k = 0; k < n_pol; ++k)
    if (pol_node[k] < 0 || pol_node[k] >= R.V || pol_belief[k] < 0 || pol_belief[k] >= B || pol_parent[k] >= k || (k > 0 && pol_parent[k] < 0) || (k == 0 && pol_parent[k] != -1))
      return porrt_fail(ctx, PORRT_ERR_INVALID_ARG, "refine_policy_reparent: not a policy in creation order");
  CUDA_TRY(ctx, cudaSetDevice(ctx->device));
  cudaStream_t st = ctx->stream;
  R.fetch_failed = false;
  // ---- Policy::decompose (common.rs:85-129)
  std::vector<std::vector<int64_t>> pieces;
  std::vector<std::vector<int32_t>> successors;
  {
    std::vector<int32_t> piece_ptr;
    std::vector<int64_t> piece_nodes;
    policy_decompose_flat(pol_parent, n_pol, piece_ptr, piece_nodes, successors);
    for (size_t p = 0; p + 1 < piece_ptr.size(); ++p) pieces.emplace_back(piece_nodes.begin() + piece_ptr[p], piece_nodes.begin() + piece_ptr[p + 1]);
  }
  // ---- build_tree per piece
  const bool dbg = getenv("PORRT_DEBUG") != nullptr;
  auto now_ms = [] { return std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now().time_since_epoch()).count(); };
  double tph[6] = {now_ms(), 0, 0, 0, 0, 0};
  std::vector<PieceTree> trees(pieces.size());
  int64_t tree_nodes = 0;
  std::vector<uint32_t> stamp((size_t)R.V * B, 0);   // visited set of build_tree: stamp == piece + 1
  std::vector<uint32_t> expanded((size_t)R.V * B, 0);  // belief nodes already expanded in the running search (tag per seed)
  uint32_t expand_tag = 0;
  struct Visited {
    std::vector<uint32_t>& s; uint32_t tag;
    bool count(int64_t id) const { return s[(size_t)id] == tag; }
    void insert(int64_t id) { s[(size_t)id] = tag; }
  };
  for (size_t p = 0; p < pieces.size(); ++p) {
    PieceTree& T = trees[p];
    Visited visited{stamp, (uint32_t)p + 1};
    for (size_t k = 0; k < pieces[p].size(); ++k) {
      const int64_t pn = pieces[p][k];
      const int64_t bg = (int64_t)pol_node[pn] * B + pol_belief[pn];
      const double* s = &R.xy[2 * (size_t)pol_node[pn]];
      T.add(s, (int32_t)k - 1, k ? norm2(&R.xy[2 * (size_t)pol_node[pieces[p][k - 1]]], s, 2) : 0.0, bg);
      visited.insert(bg);
    }
    T.belief = pol_belief[pieces[p][0]];
    T.leaf = (int32_t)T.size() - 1;
    const size_t n_seed = T.size();
    std::vector<std::pair<int32_t, int64_t>> q;
    for (size_t seed = 0; seed < n_seed; ++seed) {
      const double sx[2] = {T.xy[2 * seed], T.xy[2 * seed + 1]};
      q.assign(1, {(int32_t)seed, T.bgid[seed]});
      ++expand_tag;
      for (size_t head = 0; head < q.size(); ++head) {
        const int32_t tree_id = q[head].first;
        const int64_t from_bg = q[head].second;
        // the reference's queue holds a belief node once per parent that pushed it; only the FIRST entry can add anything (what it
        // leaves behind is visited or beyond the seed's radius for every later one too), so the others are skipped unexpanded
        if (expanded[(size_t)from_bg] == expand_tag) continue;
        expanded[(size_t)from_bg] = expand_tag;
        R.for_children(ctx, from_bg, [&](int64_t child) {
          const double* cs = &R.xy[2 * (size_t)(child / B)];
          if (visited.count(child)) return;
          const double d = norm2(sx, cs, 2);
          if (!(d <= radius)) return;
          const int32_t me = T.add(cs, tree_id, d, child);
          visited.insert(child);
          R.for_children(ctx, child, [&](int64_t cc) { if (!visited.count(cc)) q.push_back({me, cc}); });
        });
        if (R.fetch_failed) return porrt_fail(ctx, PORRT_ERR_CUDA, "refine_policy_reparent: fetching a value column failed");
        if ((int64_t)T.size() > (int64_t)R.V * B) return porrt_fail(ctx, PORRT_ERR_PANIC, "refine_policy_reparent: tree larger than the belief graph");
      }
    }
    tree_nodes += (int64_t)T.size();
  }
  if (out_tree_nodes) *out_tree_nodes = tree_nodes;
  tph[1] = now_ms();
  // ---- every (node, neighbour within radius / 2) pair of every tree: ONE device batch of is_transition_valid
  const double r2 = 0.5 * radius;
  std::vector<int64_t> nb_ptr(1, 0);     // per tree node (trees back to back)
  std::vector<int32_t> nb_ids;           // neighbour = tree node index inside its own tree
  std::vector<int32_t> node_base, node_row;   // per tree node: first node of its tree, belief of its piece
  std::vector<double> node_xy;
  {
    std::vector<int32_t> nb, order, kd_stack;
    std::vector<double> oxy;
    int32_t base = 0;
    for (size_t p = 0; p < trees.size(); ++p) {
      const PieceTree& T = trees[p];
      node_xy.insert(node_xy.end(), T.xy.begin(), T.xy.end());
      // small trees: all pairs against the nodes laid out in kd pre-order (the search visits node, left subtree, right subtree and
      // prunes only what cannot hit, so its hits come in that order) -- a contiguous sweep instead of ~n/2 pointer hops per query
      const bool brute = (int64_t)T.size() <= ctx->reparent_brute_max;   // 4096 unless PORRT_OPT_REPARENT_BRUTE_MAX_NODES says otherwise
      if (brute) {
        order.clear(); oxy.clear();
        kd_stack.assign(1, 0);
        while (!kd_stack.empty()) {
          const int32_t k = kd_stack.back();
          kd_stack.pop_back();
          order.push_back(k); oxy.push_back(T.xy[2 * (size_t)k]); oxy.push_back(T.xy[2 * (size_t)k + 1]);
          if (T.kd_right[(size_t)k] >= 0) kd_stack.push_back(T.kd_right[(size_t)k]);
          if (T.kd_left[(size_t)k] >= 0) kd_stack.push_back(T.kd_left[(size_t)k]);
        }
      }
      for (size_t u = 0; u < T.size(); ++u) {
        node_base.push_back(base); node_row.push_back(T.belief);
        nb.clear();
        if (brute) {                      // hits in kd visit order = the nodes within r2 in pre-order of the kd tree
          const double qx = T.xy[2 * u], qy = T.xy[2 * u + 1];
          // the square root only where it can matter: d2 beyond r2^2 by more than a few ulps is a miss whatever sqrt rounds to
          const double pre = r2 * r2 * (1.0 + 1e-12) + 1e-300;
          for (size_t k = 0; k < T.size(); ++k) {
            const double dx = qx - oxy[2 * k], dy = qy - oxy[2 * k + 1];
            const double d2 = dx * dx + dy * dy;
            if (d2 <= pre && std::sqrt(d2) <= r2) nb.push_back(order[k]);
          }
        } else {
          T.radius(&T.xy[2 * u], r2, nb);
        }
        nb_ids.insert(nb_ids.end(), nb.begin(), nb.end());
        nb_ptr.push_back((int64_t)nb_ids.size());
        if (nb_ids.size() > ((size_t)1 << 26))   // 64 M candidate transitions: a radius far beyond what the reference is run with
          return porrt_fail(ctx, PORRT_ERR_UNSUPPORTED, "refine_policy_reparent: more than 2^26 candidate transitions (radius too large for this roadmap)");
      }
      base += (int32_t)T.size();
    }
  }
  const int64_t n_pairs = (int64_t)nb_ids.size();
  const int64_t n_nodes_all = (int64_t)node_base.size();
  tph[2] = now_ms();
  if (out_transitions) *out_transitions = n_pairs;
  std::vector<uint8_t> valid((size_t)std::max<int64_t>(n_pairs, 1));
  std::vector<int32_t> status((size_t)std::max<int64_t>(n_pairs, 1), 0);
  if (n_pairs > 0) {
    // the device expands (node, neighbour) index pairs into endpoint coordinates itself: 4 bytes per pair cross the bus, not 36
    const size_t n = (size_t)n_pairs, nn = (size_t)n_nodes_all, nrows = (size_t)B * nv;
    double *d_from, *d_to, *d_nxy;
    int32_t *d_tmp, *d_status, *d_row, *d_nb, *d_nbase, *d_nrow;
    uint8_t *d_valid, *d_compat;
    int64_t* d_nptr;
    CUDA_TRY(ctx, carve(ctx->ws_main, [&](Carve& c) {
      d_from = c.take<double>(2 * n, 256); d_to = c.take<double>(2 * n, 256); d_tmp = c.take<int32_t>(3 * n, 256);
      d_status = c.take<int32_t>(n, 256); d_row = c.take<int32_t>(n, 256); d_nb = c.take<int32_t>(n, 256); d_valid = c.take<uint8_t>(n, 256);
      d_nxy = c.take<double>(2 * nn, 256); d_nptr = c.take<int64_t>(nn + 1, 256); d_nbase = c.take<int32_t>(nn, 256);
      d_nrow = c.take<int32_t>(nn, 256); d_compat = c.take<uint8_t>(nrows, 256);
    }));
    CUDA_TRY(ctx, cudaMemcpyAsync(d_nb, nb_ids.data(), n * 4, cudaMemcpyHostToDevice, st));
    CUDA_TRY(ctx, cudaMemcpyAsync(d_nxy, node_xy.data(), nn * 16, cudaMemcpyHostToDevice, st));
    CUDA_TRY(ctx, cudaMemcpyAsync(d_nptr, nb_ptr.data(), (nn + 1) * 8, cudaMemcpyHostToDevice, st));
    CUDA_TRY(ctx, cudaMemcpyAsync(d_nbase, node_base.data(), nn * 4, cudaMemcpyHostToDevice, st));
    CUDA_TRY(ctx, cudaMemcpyAsync(d_nrow, node_row.data(), nn * 4, cudaMemcpyHostToDevice, st));
    CUDA_TRY(ctx, cudaMemcpyAsync(d_compat, R.compat.data(), nrows, cudaMemcpyHostToDevice, st));
    reparent_pairs_kernel<<<div_up(n_nodes_all * 32, 256), 256, 0, st>>>(d_nptr, d_nb, (const double2*)d_nxy, d_nbase, d_nrow, n_nodes_all,
                                                                          (double2*)d_from, (double2*)d_to, d_row);
    LAUNCH_CHECK(ctx);
    const int32_t rc = transition_valid_dev(ctx, d_from, d_to, n_pairs, d_compat, d_row, nv, d_tmp, d_valid, d_status);
    if (rc) return rc;
    CUDA_TRY(ctx, cudaMemcpyAsync(valid.data(), d_valid, n, cudaMemcpyDeviceToHost, st));
    CUDA_TRY(ctx, cudaMemcpyAsync(status.data(), d_status, n * 4, cudaMemcpyDeviceToHost, st));
    CUDA_TRY(ctx, cudaStreamSynchronize(st));
    for (int64_t k = 0; k < n_pairs; ++k)   // every node is popped at least once and tests all its pairs: a panic anywhere is reached
      if (status[(size_t)k] < 0) return porrt_fail(ctx, PORRT_ERR_PANIC, "refine_policy_reparent: is_transition_valid panics (code " + std::to_string(status[(size_t)k]) + ")");
  }
  tph[3] = now_ms();
  // ---- reparent (:282-322)
  {
    int64_t base = 0;                    // first tree node of the piece in nb_ptr
    std::vector<std::pair<int32_t, double>> nd;
    for (PieceTree& T : trees) {
      ReparentHeap q(T.size());
      for (size_t id = 0; id < T.size(); ++id) q.push((int32_t)id, T.dist_from_root((int32_t)id));
      while (!q.heap.empty()) {
        const int32_t u = q.pop();
        const double du = T.dist_from_root(u);
        nd.clear();
        for (int64_t k = nb_ptr[(size_t)(base + u)]; k < nb_ptr[(size_t)(base + u) + 1]; ++k)
          if (valid[(size_t)k]) nd.push_back({nb_ids[(size_t)k], T.dist_from_root(nb_ids[(size_t)k])});   // all read before this pop reparents anybody
        for (const auto& kv : nd) {
          const double cost = norm2(&T.xy[2 * (size_t)u], &T.xy[2 * (size_t)kv.first], 2);
          if (du + cost < kv.second) {
            T.parent[(size_t)kv.first] = u; T.parent_cost[(size_t)kv.first] = cost;
            q.push(kv.first, du + cost);
          }
        }
      }
      base += (int64_t)T.size();
    }
  }
  tph[4] = now_ms();
  if (dbg) fprintf(stderr, "[porrt] reparent: trees %.2f ms, candidate pairs %.2f ms (%lld), device batch %.2f ms, label-correcting loop %.2f ms\n",
                   tph[1] - tph[0], tph[2] - tph[1], (long long)n_pairs, tph[3] - tph[2], tph[4] - tph[3]);
  // ---- recompose (:324-393): leaf -> root of every tree, reversed; then piece ends -> successor piece starts
  std::vector<std::vector<int32_t>> paths(trees.size());
  int64_t n_out = 0;
  for (size_t p = 0; p < trees.size(); ++p) {
    for (int32_t k = trees[p].leaf; k >= 0; k = trees[p].parent[(size_t)k]) paths[p].push_back(k);
    std::reverse(paths[p].begin(), paths[p].end());
    n_out += (int64_t)paths[p].size();
  }
  *out_n = n_out;
  if (n_out > cap || !out_xy || !out_node || !out_belief || !out_parent || !out_is_leaf)
    return porrt_fail(ctx, PORRT_ERR_CAPACITY, "refine_policy_reparent: cap too small");
  std::vector<int32_t> p_start(trees.size()), p_end(trees.size(), -1);
  {
    int32_t o = 0;
    for (size_t p = 0; p < trees.size(); ++p) {
      p_start[p] = o;
      for (size_t j = 0; j < paths[p].size(); ++j, ++o) {
        const int32_t k = paths[p][j];
        out_xy[2 * (size_t)o] = trees[p].xy[2 * (size_t)k]; out_xy[2 * (size_t)o + 1] = trees[p].xy[2 * (size_t)k + 1];
        out_node[o] = (int32_t)(trees[p].bgid[(size_t)k] / B); out_belief[o] = (int32_t)(trees[p].bgid[(size_t)k] % B);
        out_parent[o] = j == 0 ? -1 : o - 1;
      }
      if (paths[p].size() >= 2) p_end[p] = o - 1;
    }
    for (size_t p = 0; p < trees.size(); ++p)
      if (p_end[p] >= 0) for (int32_t q : successors[p]) out_parent[p_start[(size_t)q]] = p_end[p];
  }
  std::vector<int32_t> n_children((size_t)n_out, 0);
  for (int64_t k = 0; k < n_out; ++k) if (out_parent[k] >= 0) ++n_children[(size_t)out_parent[k]];
  for (int64_t k = 0; k < n_out; ++k) out_is_leaf[k] = n_children[(size_t)k] == 0;
  if (out_expected_cost) *out_expected_cost = policy_expected_cost_flat(R.beliefs.data(), nw, out_xy, out_belief, out_parent, n_out);
  return PORRT_OK;
}

// ================================================================================================ Policy::decompose / expected cost (host)
// The two pieces of common.rs the refiners are built around, as host-side rows of the ABI (no device, no ctx): they are what the
// reference's own map-free tests pin (common.rs:425-489: three pieces; 1 + 0.4 sqrt 2 + 0.6 * 2 sqrt 2).
PORRT_API int32_t porrt_policy_decompose(const int32_t* parent, int64_t n, int32_t* out_piece_ptr, int32_t* out_piece_nodes, int32_t* out_succ_ptr,
                                         int32_t* out_succ, int32_t cap_pieces, int32_t* out_n_pieces) {
  if (!policy_parents_ok(parent, n) || !out_n_pieces || n > 0x7fffffff) return PORRT_ERR_INVALID_ARG;
  std::vector<int32_t> piece_ptr;
  std::vector<int64_t> piece_nodes;
  std::vector<std::vector<int32_t>> successors;
  policy_decompose_flat(parent, n, piece_ptr, piece_nodes, successors);
  const int32_t np = (int32_t)successors.size();
  *out_n_pieces = np;
  if (np > cap_pieces || !out_piece_ptr || !out_piece_nodes) return PORRT_ERR_CAPACITY;
  for (int32_t p = 0; p <= np; ++p) out_piece_ptr[p] = piece_ptr[(size_t)p];
  for (size_t k = 0; k < piece_nodes.size(); ++k) out_piece_nodes[k] = (int32_t)piece_nodes[k];
  if (out_succ_ptr && out_succ) {           // skeleton as a CSR: successor pieces of piece p (at most np - 1 entries in all)
    int32_t o = 0;
    for (int32_t p = 0; p < np; ++p) { out_succ_ptr[p] = o; for (int32_t q : successors[(size_t)p]) out_succ[o++] = q; }
    out_succ_ptr[np] = o;
  }
  return PORRT_OK;
}

PORRT_API int32_t porrt_policy_expected_cost(const double* xy, const int32_t* belief_id, const int32_t* parent, int64_t n, const double* beliefs,
                                             int32_t B, int32_t n_worlds, double* out_expected_cost) {
  if (!xy || !belief_id || !beliefs || B <= 0 || n_worlds <= 0 || !out_expected_cost || n <= 0 || !parent || parent[0] != -1) return PORRT_ERR_INVALID_ARG;
  for (int64_t k = 0; k < n; ++k)
    if (belief_id[k] < 0 || belief_id[k] >= B || parent[k] >= k || (k > 0 && parent[k] < -1)) return PORRT_ERR_INVALID_ARG;   // (-1 beyond node 0: an unconnected piece)
  *out_expected_cost = policy_expected_cost_flat(beliefs, n_worlds, xy, belief_id, parent, n);
  return PORRT_OK;
}
