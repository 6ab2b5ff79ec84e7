// belief_tables.cu -- the observation successor tables of the implicit belief graph, built on the device.
//
// Reference: PTO::build_belief_graph's observation edges (pto.rs:209-231): for every node and reachable belief,
// `observe(node.state, belief)` (map_io.rs:281-300, map_shelves_io.rs:242-265) splits the belief by every zone visible from
// the node -- zones ascending, every current belief into [closed, open] resp. [there, not there], zero-mass branches dropped
// (NaN after normalisation, map_io.rs:257-275) -- and each child whose `hash` (common.rs:352-355) differs from the parent's
// becomes an observation edge to `belief_id(child)` (belief_graph.rs:65-72), later weighted by `transition_probability` of the
// STORED belief states (belief_graph.rs:128).
//
// observe() depends on the node only through its SET of visible zones, so one table per distinct set serves all nodes
// (graph.cu).  With k zones in the set an entry (set, belief) has at most 2^k children, the leaves of a binary tree whose
// emission order is the leaf index read as "first = 0 / second = 1 per zone, first zone most significant".  Every leaf is
// independent: one thread follows one root-to-leaf path (mask, sum left to right, divide -- the reference's operations in the
// reference's order; IEEE division, -fmad=false), hashes the result, finds the belief id by binary search over the sorted hashes and
// computes the edge probability.  A flag scan compacts the surviving leaves in emission order.  At the config-4 shape (43 sets x
// 4095 beliefs, 328 k edges) this took 8.3 ms on 16 host threads.
#include <algorithm>

#include "common.cuh"
#include "belief_tables.cuh"

namespace {

struct SuccArgs {
  const double* beliefs;          // [B][nw]
  int32_t B, nw, n_sets, n_zones, kind, mask_words;
  const uint64_t* sets;           // [n_sets] visible-zone masks
  const int64_t* set_off;         // [n_sets + 1] first leaf slot of a set (B << k slots each)
  const uint64_t* zone_worlds;    // DOOR: zones_to_worlds [n_zones][mask_words] (map_io.rs:198-214); unused for SHELF
  const uint64_t* sorted_hash;    // [B] ascending
  const int32_t* sorted_id;       // [B]
  const uint64_t* bhash;          // [B]
  const int32_t* level;           // [B] support size
  const int32_t* colpos;          // [B]
};

// common.rs:352-355: sum of (10^i + 1) * round(1000 p_i), wrapping like usize in a release build
__device__ uint64_t belief_hash_dev(const double* b, int64_t stride, int n) {
  uint64_t h = 0, p10 = 1;
  for (int i = 0; i < n; ++i) {
    const double r = round(__dmul_rn(b[(int64_t)i * stride], 1000.0));
    const uint64_t v = (r <= 0.0 || isnan(r)) ? 0 : (r >= 18446744073709551615.0 ? ~(uint64_t)0 : (uint64_t)r);
    h += (p10 + 1) * v;
    p10 *= 10;
  }
  return h;
}

// one thread per leaf slot; work[w * n_slots + slot] holds the thread's current belief (coalesced over the slots)
__global__ void __launch_bounds__(256) succ_leaf_kernel(SuccArgs g, int64_t n_slots, double* __restrict__ work,
                                                        int32_t* __restrict__ slot_id, double* __restrict__ slot_p, int32_t* __restrict__ err) {
  const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= n_slots) return;
  int s = 0;
  {  // the set this slot belongs to (n_sets is small)
    int lo = 0, hi = g.n_sets;
    while (hi - lo > 1) { const int mid = (lo + hi) >> 1; if (g.set_off[mid] <= t) lo = mid; else hi = mid; }
    s = lo;
  }
  const uint64_t set = g.sets[s];
  const int k = __popcll(set);
  const int64_t local = t - g.set_off[s];
  const int b = (int)(local >> k);
  const unsigned leaf = (unsigned)(local & (((int64_t)1 << k) - 1));
  double* cur = work + t;
  for (int w = 0; w < g.nw; ++w) cur[(int64_t)w * n_slots] = g.beliefs[(int64_t)b * g.nw + w];
  int zi = 0;
  slot_id[t] = -1;
  for (int z = 0; z < g.n_zones; ++z) {
    if (!((set >> z) & 1)) continue;
    const bool second = (leaf >> (k - 1 - zi)) & 1;
    ++zi;
    double sum = 0.0;
    for (int w = 0; w < g.nw; ++w) {
      const bool in_zone_world = g.kind == PORRT_DOMAIN_DOOR ? ((g.zone_worlds[(int64_t)z * g.mask_words + (w >> 6)] >> (w & 63)) & 1) != 0 : (w == z);
      const bool to_first = g.kind == PORRT_DOMAIN_DOOR ? !in_zone_world : in_zone_world;   // DOOR [closed, open]; SHELF [there, not there]
      const double v = (to_first != second) ? cur[(int64_t)w * n_slots] : 0.0;
      cur[(int64_t)w * n_slots] = v;
      sum = __dadd_rn(sum, v);
    }
    bool nan = false;
    for (int w = 0; w < g.nw; ++w) {
      const double p = __ddiv_rn(cur[(int64_t)w * n_slots], sum);
      nan |= isnan(p);
      cur[(int64_t)w * n_slots] = p;
    }
    if (nan) return;   // zero-mass branch: dropped together with everything below it
  }
  const uint64_t h = belief_hash_dev(cur, n_slots, g.nw);
  if (h == g.bhash[b]) return;   // pto.rs:216
  int lo = 0, hi = g.B;
  while (lo < hi) { const int mid = (lo + hi) >> 1; if (g.sorted_hash[mid] < h) lo = mid + 1; else hi = mid; }
  if (lo >= g.B || g.sorted_hash[lo] != h) { atomicOr(err, 1); return; }   // "no id corresponding to this belief state" (belief_graph.rs:69)
  const int cid = g.sorted_id[lo];
  // transition_probability on the STORED belief states (common.rs:188-190, belief_graph.rs:128)
  double p = 0.0;
  for (int w = 0; w < g.nw; ++w) p = __dadd_rn(p, g.beliefs[(int64_t)cid * g.nw + w] > 0.0 ? g.beliefs[(int64_t)b * g.nw + w] : 0.0);
  if (!(p > 0.0)) atomicOr(err, 2);                       // assert!(p > 0.0) (belief_graph.rs:130)
  if (g.level[cid] >= g.level[b]) atomicOr(err, 4);       // not a split of the support: the level order of colsolve.cu does not apply
  slot_id[t] = cid;
  slot_p[t] = p;
}

__global__ void succ_flag_kernel(const int32_t* __restrict__ slot_id, int64_t n, int32_t* __restrict__ flag) {
  const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t < n) flag[t] = slot_id[t] >= 0;
}
__global__ void succ_scatter_kernel(SuccArgs g, int64_t n_slots, const int32_t* __restrict__ slot_id, const double* __restrict__ slot_p,
                                    const int64_t* __restrict__ pos, int64_t* __restrict__ succ_ptr, int32_t* __restrict__ succ_b,
                                    int32_t* __restrict__ succ_col, double* __restrict__ succ_p) {
  const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const int64_t n_sb = (int64_t)g.n_sets * g.B;
  if (t <= n_sb) {   // succ_ptr[s * B + b] = compacted position of the entry's first leaf slot
    if (t == n_sb) succ_ptr[t] = pos[n_slots];
    else {
      const int s = (int)(t / g.B);
      const int b = (int)(t - (int64_t)s * g.B);
      const int k = __popcll(g.sets[s]);
      succ_ptr[t] = pos[g.set_off[s] + (k == 0 ? 0 : ((int64_t)b << k))];   // a set without zones has no slots
    }
  }
  if (t < n_slots && slot_id[t] >= 0) {
    const int64_t q = pos[t];
    succ_b[q] = slot_id[t];
    succ_col[q] = g.colpos[slot_id[t]];
    succ_p[q] = slot_p[t];
  }
}
}  // namespace

int32_t belief_succ_tables(porrt_ctx* ctx, const double* beliefs_host, int32_t B, int32_t nw, const std::vector<uint64_t>& sets,
                           const std::vector<uint64_t>& bhash, const std::vector<int32_t>& level, const std::vector<int32_t>& colpos,
                           BeliefSuccDev* out, cudaStream_t st) {
  const int n_sets = (int)sets.size();
  std::vector<int64_t> set_off((size_t)n_sets + 1, 0);
  for (int s = 0; s < n_sets; ++s) {
    const int k = __builtin_popcountll(sets[(size_t)s]);
    if (k > 20) return porrt_fail(ctx, PORRT_ERR_UNSUPPORTED, "belief_vi: more than 20 zones visible from one node");
    set_off[(size_t)s + 1] = set_off[(size_t)s] + (k == 0 ? 0 : ((int64_t)B << k));   // nothing visible: observe() returns the belief itself
  }
  const int64_t n_slots = set_off[(size_t)n_sets];
  if ((double)n_slots * (nw * 8.0 + 24.0) > 8e9) return porrt_fail(ctx, PORRT_ERR_UNSUPPORTED, "belief_vi: observation tables exceed 8 GB of work space");
  std::vector<std::pair<uint64_t, int32_t>> sorted((size_t)B);
  for (int b = 0; b < B; ++b) sorted[(size_t)b] = {bhash[(size_t)b], b};
  std::sort(sorted.begin(), sorted.end());
  std::vector<uint64_t> sh((size_t)B);
  std::vector<int32_t> sid((size_t)B);
  for (int b = 0; b < B; ++b) { sh[(size_t)b] = sorted[(size_t)b].first; sid[(size_t)b] = sorted[(size_t)b].second; }

  // ---- inputs + work space (ws_query); outputs (ctx->d_bel_succ) are sized after the scan
  const size_t zw = ctx->zone_world_masks.size();
  double *d_beliefs, *d_work, *d_slot_p;
  uint64_t *d_sets, *d_zw, *d_sh, *d_bhash;
  int64_t *d_set_off, *d_pos;
  int32_t *d_sid, *d_level, *d_colpos, *d_err, *d_slot_id, *d_flag;
  CUDA_TRY(ctx, carve(ctx->ws_query, [&](Carve& c) {
    d_beliefs = c.take<double>((size_t)B * nw); d_sets = c.take<uint64_t>(n_sets); d_set_off = c.take<int64_t>(n_sets + 1);
    d_zw = c.take<uint64_t>(zw + 1); d_sh = c.take<uint64_t>(B); d_bhash = c.take<uint64_t>(B);
    d_sid = c.take<int32_t>(B); d_level = c.take<int32_t>(B); d_colpos = c.take<int32_t>(B); d_err = c.take<int32_t>(4);
    d_work = c.take<double>((size_t)n_slots * nw); d_slot_p = c.take<double>(n_slots); d_pos = c.take<int64_t>(n_slots + 1);
    d_slot_id = c.take<int32_t>(n_slots); d_flag = c.take<int32_t>(n_slots);
  }));
  CUDA_TRY(ctx, cudaMemcpyAsync(d_beliefs, beliefs_host, (size_t)B * nw * 8, cudaMemcpyHostToDevice, st));
  CUDA_TRY(ctx, cudaMemcpyAsync(d_sets, sets.data(), (size_t)n_sets * 8, cudaMemcpyHostToDevice, st));
  CUDA_TRY(ctx, cudaMemcpyAsync(d_set_off, set_off.data(), (size_t)(n_sets + 1) * 8, cudaMemcpyHostToDevice, st));
  if (zw) CUDA_TRY(ctx, cudaMemcpyAsync(d_zw, ctx->zone_world_masks.data(), zw * 8, cudaMemcpyHostToDevice, st));
  CUDA_TRY(ctx, cudaMemcpyAsync(d_sh, sh.data(), (size_t)B * 8, cudaMemcpyHostToDevice, st));
  CUDA_TRY(ctx, cudaMemcpyAsync(d_bhash, bhash.data(), (size_t)B * 8, cudaMemcpyHostToDevice, st));
  CUDA_TRY(ctx, cudaMemcpyAsync(d_sid, sid.data(), (size_t)B * 4, cudaMemcpyHostToDevice, st));
  CUDA_TRY(ctx, cudaMemcpyAsync(d_level, level.data(), (size_t)B * 4, cudaMemcpyHostToDevice, st));
  CUDA_TRY(ctx, cudaMemcpyAsync(d_colpos, colpos.data(), (size_t)B * 4, cudaMemcpyHostToDevice, st));
  CUDA_TRY(ctx, cudaMemsetAsync(d_err, 0, 4, st));
  SuccArgs g = {d_beliefs, B, nw, n_sets, ctx->n_zones, ctx->map.kind, ctx->mask_words, d_sets, d_set_off, d_zw, d_sh, d_sid, d_bhash, d_level, d_colpos};
  int64_t n_succ = 0;
  if (n_slots > 0) {
    succ_leaf_kernel<<<div_up(n_slots, 256), 256, 0, st>>>(g, n_slots, d_work, d_slot_id, d_slot_p, d_err);
    LAUNCH_CHECK(ctx);
    succ_flag_kernel<<<div_up(n_slots, 256), 256, 0, st>>>(d_slot_id, n_slots, d_flag);
    LAUNCH_CHECK(ctx);
    int32_t rc = scan_exclusive_i64(ctx, d_flag, n_slots, d_pos);
    if (rc) return rc;
    CUDA_TRY(ctx, cudaMemcpyAsync(&n_succ, d_pos + n_slots, 8, cudaMemcpyDeviceToHost, st));
  } else {
    CUDA_TRY(ctx, cudaMemsetAsync(d_pos, 0, 8, st));
  }
  int32_t err = 0;
  CUDA_TRY(ctx, cudaMemcpyAsync(&err, d_err, 4, cudaMemcpyDeviceToHost, st));
  CUDA_TRY(ctx, cudaStreamSynchronize(st));
  if (err & 1) return porrt_fail(ctx, PORRT_ERR_PANIC, "no id corresponding to this belief state! (belief_graph.rs:69)");
  if (err & 2) return porrt_fail(ctx, PORRT_ERR_PANIC, "assert!(p > 0.0) (belief_graph.rs:130)");
  const int64_t n_sb = (int64_t)n_sets * B;
  // dedicated: the tables are read until the last level is done, while the frontier path works in sort_keys .. ws_state
  CUDA_TRY(ctx, carve(ctx->d_bel_succ, [&](Carve& c) {
    out->succ_ptr = c.take<int64_t>(n_sb + 1); out->succ_p = c.take<double>(n_succ + 1);
    out->succ_b = c.take<int32_t>(n_succ + 1); out->succ_col = c.take<int32_t>(n_succ + 1);
  }));
  out->n_succ = n_succ;
  out->levels_ok = !(err & 4);
  out->beliefs = d_beliefs;
  succ_scatter_kernel<<<div_up(std::max<int64_t>(n_slots, n_sb + 1), 256), 256, 0, st>>>(g, n_slots, d_slot_id, d_slot_p, d_pos, out->succ_ptr,
                                                                                          out->succ_b, out->succ_col, out->succ_p);
  LAUNCH_CHECK(ctx);
  return PORRT_OK;
}
