// pto_grow.cu -- PTO::grow_graph (pto.rs:55-139) as ONE call, the roadmap resident on the device from the root to the end.
//
// The loop is sequential in the reference, but (1) its sample stream never looks at the tree -- iteration i draws a world and a
// state (pto.rs:141-149) -- so every (world_i, sample_i) is drawn on the host up front, and (2) the state only grows: nodes are
// appended, kd nodes become leaves, reachability bits are only ever set, final nodes are appended.  So a WINDOW of consecutive
// iterations is speculated in parallel against the roadmap S0 as it stood when the window started (one CTA per iteration:
// filtered 1-NN, steer, state validity, the radius set for the largest radius the window can use in kd pre-order, its edge
// checks, the kd slot), and one CTA then commits the iterations IN ORDER for as long as nothing committed earlier in the window
// can have changed an iteration's answers (DESIGN.md 3.8):
//   (a) no node added in the window, and no node that gained bit world_i in the window, lies within the speculated nearest
//       distance (+ a few ulps) of sample_i;
//   (b) no node added in the window lies within heuristic_radius(n_i) of the steered state;
//   (c) the kd slot the steered state descends to in S0 is still free.
// The first iteration of a window always commits.  At the first conflict the window ends and the next one starts there.  The
// result is the reference's roadmap bit for bit, whatever the window size.
//
// kd pre-order (the order KdTree::nearest_neighbors returns hits in) is decided by each node's root-to-node branch bits: the first
// 64 are kept as a key (MSB first), deeper ties -- chains of exact duplicates, e.g. repeated goal samples -- are resolved by
// walking parent links, so the key length is not capped.
//
// porrt_pto_grow_batch grows R roadmaps that differ only in their sampler seed through the same kernels: each keeps its own state
// (PtoRoad, control block r), the kernels find roadmap r's pointers in device arrays of descriptors, a speculate launch covers
// every window slot of every roadmap and a commit launch is one CTA per roadmap.  porrt_pto_grow is the batch of one.
#include <algorithm>
#include <cmath>
#include <climits>
#include <cstring>
#include <memory>
#include <string>
#include <vector>

#include "common.cuh"
#include "map_dev.cuh"
#include "pcg64.h"

#define PG_SPEC_THREADS 256
#define PG_COMMIT_THREADS 256
#define PG_WMAX 128               // iterations speculated per window at most (CTAs of a speculate launch)
#define PG_WMIN 4
#define PG_TOUCH_CAP 2048         // pre-window nodes that may gain bits in one window before the window is cut
#define PG_BATCH 8                // windows enqueued between two looks at the progress flags

// control block (int32, device): what the kernels share across launches
enum { C_V = 0, C_IT, C_W, C_DONE, C_PANIC, C_DRAWN, C_STALL, C_NFIN, C_E, C_WINDOWS, C_RESPEC, C_CONF_NN, C_CONF_RAD, C_NODE_CAP,
       C_EDGE_CAP, C_N };

struct PtoRoad {   // one roadmap of a batch: its state, its samples, its speculation scratch and its result
  // roadmap [node_cap]
  DevBuf xy, node_vid, reach, child, parent, depth, key, final_idx, gain, epoch, edge_off, ecnt;
  DevBuf fin_ids, fin_goal, fin_acc;          // finals in add order, the goal each one hit, accumulated finality [words]
  DevBuf log_nbr, log_vid;                    // edge log (neighbour, validity id) grouped by new node, commit order
  DevBuf samples, worlds;                     // iteration i (1-based) at [i - 1]
  DevBuf spec;                                // per-slot speculation results + hit lists [PG_WMAX * node_cap]
  DevBuf csr_row, csr_col, csr_vid;           // the assembled roadmap
  int64_t node_cap = 0, edge_cap = 0;
  // the last result (porrt_pto_fetch_roadmap)
  bool have = false;
  int64_t V = 0, E = 0, n_finals = 0;
  DevBuf* bufs[23] = {&xy, &node_vid, &reach, &child, &parent, &depth, &key, &final_idx, &gain, &epoch, &edge_off, &ecnt, &fin_ids,
                      &fin_goal, &fin_acc, &log_nbr, &log_vid, &samples, &worlds, &spec, &csr_row, &csr_col, &csr_vid};
  PtoRoad() = default;
  PtoRoad(const PtoRoad&) = delete;           // bufs points into this object
  size_t bytes() const { size_t s = 0; for (DevBuf* b : bufs) s += b->cap; return s; }
  void release() { for (DevBuf* b : bufs) b->release(); }
};

struct PtoGrow {
  std::vector<std::unique_ptr<PtoRoad>> roads;   // the roadmaps of the last batch; a single growth is the batch of one
  DevBuf radius;                                 // heuristic_radius(n) at [n]
  DevBuf goals, goal_masks;
  DevBuf ctl;                                    // control blocks, roadmap r at [r * C_N]
  DevBuf pg_desc, spec_desc, caps;               // PgDev / SpecDev of every roadmap; node cap, edge cap, samples drawn of each
  DevBuf work;                                   // CSR assembly work space, one roadmap at a time
  PinBuf ctl_host;                               // every control block, as the last look saw it
  std::vector<char> desc_host;                   // what pg_desc + spec_desc hold
  int64_t radius_n = 0;
  int words = 1;
  int32_t n_have = 0;                            // roadmaps of the last batch; 0: nothing grown
  std::vector<uint64_t> goal_masks_host;
};

void pto_grow_release(porrt_ctx* ctx) {
  PtoGrow* g = ctx->pto;
  if (!g) return;
  for (auto& r : g->roads) r->release();
  DevBuf* all[] = {&g->radius, &g->goals, &g->goal_masks, &g->ctl, &g->pg_desc, &g->spec_desc, &g->caps, &g->work};
  for (DevBuf* b : all) b->release();
  g->ctl_host.release();
  delete g;
  ctx->pto = nullptr;
}

// ------------------------------------------------------------------------------------------------ device
struct PgDev {     // one roadmap's pointers; the kernels read roadmap r's from a device array of them
  double2* xy; int32_t* node_vid; uint64_t* reach; int32_t* child; int32_t* parent; int32_t* depth; uint64_t* key;
  int32_t* final_idx; uint64_t* gain; int32_t* epoch; int64_t* edge_off; int32_t* ecnt;
  int32_t* fin_ids; int32_t* fin_goal; uint64_t* fin_acc; int32_t* log_nbr; int32_t* log_vid;
  const double2* samples; const int32_t* worlds; const double* radius; const double2* goals; const uint64_t* goal_masks;
  const uint64_t* validities; int32_t* ctl;
  int32_t words, n_worlds, n_goals; double goal_max_dist, max_step;
  int64_t n_iter_min, n_iter_max;
};
struct SpecDev {   // speculation results, slot b of the window
  int32_t* nn; double* nn_d; double2* q; int32_t* svid; int32_t* nn_vid; int32_t* n_hits; int32_t* slot;   // slot = 2 * parent + side
  int32_t* hit_id; double* hit_d; int32_t* hit_vid; int32_t* tmp_id; double* tmp_d; int32_t* rank;         // [PG_WMAX * hcap]
  int64_t hcap;
};

// norm2 (common.rs:203-213): sqrt of dx*dx + dy*dy in dimension order, no FMA; a = the node, b = the query
__device__ __forceinline__ double pg_norm2(double2 a, double2 b) {
  const double dx = __dsub_rn(b.x, a.x), dy = __dsub_rn(b.y, a.y);
  return __dsqrt_rn(__dadd_rn(__dmul_rn(dx, dx), __dmul_rn(dy, dy)));
}
__device__ __forceinline__ bool pg_bit(const uint64_t* m, int w) { return (m[w >> 6] >> (w & 63)) & 1ull; }

// a precedes b (a != b) in the kd pre-order: a is an ancestor of b, or a is on the left at the first branch where they part
__device__ bool pg_precedes(const PgDev& g, int32_t a, int32_t b) {
  const int32_t da = g.depth[a], db = g.depth[b];
  const int32_t m = min(da, db), L = min(m, 64);
  const uint64_t mask = L == 0 ? 0ull : (~0ull << (64 - L));
  const uint64_t ka = g.key[a] & mask, kb = g.key[b] & mask;
  if (ka != kb) return ka < kb;
  if (m <= 64) return da < db;
  int32_t x = a, y = b;                                     // same first 64 branches: walk up (duplicate chains only)
  while (g.depth[x] > g.depth[y]) x = g.parent[x];
  while (g.depth[y] > g.depth[x]) y = g.parent[y];
  if (x == y) return da < db;
  while (g.parent[x] != g.parent[y]) { x = g.parent[x]; y = g.parent[y]; }
  return g.child[2 * g.parent[x]] == x;                     // x is the left child
}

// nn_inner (nearest_neighbor.rs:58-88) replayed on the device tree without a stack: strict <,
// near side first, the far side's test evaluated with dmin as it stands after the near side.  Used when several nodes tie.
__device__ int32_t pg_nn_replay(const PgDev& g, double2 q, int world) {
  double dmin = INFINITY;
  int32_t nearest = 0, cur = 0, from = -1;   // from: the child we just came back from (-1: entering cur)
  for (;;) {
    const double2 n = g.xy[cur];
    const int axis = g.depth[cur] & 1;
    const double qa = axis ? q.y : q.x, na = axis ? n.y : n.x;
    const int32_t l = g.child[2 * cur], r = g.child[2 * cur + 1];
    const bool near_left = qa < na;
    const int32_t first = near_left ? l : r, second = near_left ? r : l;
    int32_t next = -1;
    if (from < 0) {
      const double d = pg_norm2(n, q);
      if (d < dmin && pg_bit(g.reach + (size_t)cur * g.words, world)) { dmin = d; nearest = cur; }
      const bool c1 = near_left ? __dsub_rn(qa, dmin) < na : __dadd_rn(qa, dmin) >= na;
      if (c1 && first >= 0) next = first;
    }
    if (next < 0 && (from < 0 || from == first)) {
      const bool c2 = near_left ? __dadd_rn(qa, dmin) >= na : __dsub_rn(qa, dmin) < na;
      if (c2 && second >= 0) next = second;
    }
    if (next >= 0) { cur = next; from = -1; continue; }
    if (cur == 0) return nearest;
    from = cur; cur = g.parent[cur];
  }
}

__device__ __forceinline__ double pg_block_min(double v, double* sh) {
  for (int o = 16; o; o >>= 1) v = fmin(v, __shfl_xor_sync(0xffffffffu, v, o));
  __syncthreads();
  if ((threadIdx.x & 31) == 0) sh[threadIdx.x >> 5] = v;
  __syncthreads();
  double r = sh[0];
  for (int k = 1; k < (int)(blockDim.x >> 5); ++k) r = fmin(r, sh[k]);
  return r;
}

// ---- speculate: one CTA per iteration of the window (blockIdx.x) and roadmap (blockIdx.y), reading only the committed state S0
template <int KIND>
__global__ void __launch_bounds__(PG_SPEC_THREADS) pto_speculate_kernel(MapDev m, const PgDev* __restrict__ gs, const SpecDev* __restrict__ ss) {
  const PgDev& g = gs[blockIdx.y];
  const SpecDev& s = ss[blockIdx.y];
  __shared__ double sh_d[PG_SPEC_THREADS / 32];
  __shared__ int32_t sh_i[4];
  const int32_t* ctl = g.ctl;
  if (ctl[C_DONE]) return;
  const int b = blockIdx.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, n_warps = PG_SPEC_THREADS / 32;
  const int32_t it0 = ctl[C_IT], V0 = ctl[C_V];
  if (b >= ctl[C_W] || it0 + 1 + b > ctl[C_DRAWN]) return;
  const int i = it0 + 1 + b;
  const int world = g.worlds[i - 1];
  const double2 smp = g.samples[i - 1];
  // filtered 1-NN by brute force: the minimum over the passing nodes and how many attain it
  double best = INFINITY;
  int32_t arg = -1, cnt = 0;
  for (int32_t j = tid; j < V0; j += PG_SPEC_THREADS) {
    if (!pg_bit(g.reach + (size_t)j * g.words, world)) continue;
    const double d = pg_norm2(g.xy[j], smp);
    if (d < best) { best = d; arg = j; cnt = 1; }
    else if (d == best) ++cnt;
  }
  const double dmin = pg_block_min(best, sh_d);
  if (tid == 0) { sh_i[0] = 0; sh_i[1] = -1; }
  __syncthreads();
  if (best == dmin && arg >= 0) { atomicAdd(&sh_i[0], cnt); sh_i[1] = arg; }
  __syncthreads();
  if (tid == 0) {
    int32_t nn = 0;                                          // nothing passes: the root (nearest_neighbor.rs:89)
    if (sh_i[0] == 1) nn = sh_i[1];
    else if (sh_i[0] > 1) nn = pg_nn_replay(g, smp, world);  // a tie: the reference's traversal order decides
    // steer (common.rs:215-225)
    const double2 f = g.xy[nn];
    double2 q = smp;
    const double step = __dadd_rn(fabs(__dsub_rn(q.x, f.x)), fabs(__dsub_rn(q.y, f.y)));
    if (step > g.max_step) {
      const double lambda = __ddiv_rn(g.max_step, step);
      q.x = __dadd_rn(f.x, __dmul_rn(__dsub_rn(q.x, f.x), lambda));
      q.y = __dadd_rn(f.y, __dmul_rn(__dsub_rn(q.y, f.y), lambda));
    }
    const int32_t sv = state_validity_of(m, q.x, q.y);
    s.nn[b] = nn; s.nn_d[b] = dmin; s.q[b] = q; s.svid[b] = sv; s.n_hits[b] = 0;
    sh_i[2] = sv;
    if (sv >= 0) {                                           // the kd slot q descends to in S0 (KdTree::add)
      int32_t cur = 0;
      for (;;) {
        const double2 n = g.xy[cur];
        const int side = ((g.depth[cur] & 1) ? q.y < n.y : q.x < n.x) ? 0 : 1;
        const int32_t nx = g.child[2 * cur + side];
        if (nx < 0) { s.slot[b] = 2 * cur + side; break; }
        cur = nx;
      }
    }
  }
  __syncthreads();
  if (sh_i[2] < 0) return;
  const int32_t nn = s.nn[b];
  const double2 q = s.q[b];
  // the radius set for the largest radius this slot can meet: heuristic_radius(n) for n in V0 + 1 .. V0 + 1 + b
  double rs = -INFINITY;
  for (int k = tid; k <= b; k += PG_SPEC_THREADS) rs = fmax(rs, g.radius[V0 + 1 + k]);
  rs = -pg_block_min(-rs, sh_d);
  if (tid == 0) sh_i[3] = 0;
  __syncthreads();
  int32_t* tid_ = s.tmp_id + (size_t)b * s.hcap;
  double* td_ = s.tmp_d + (size_t)b * s.hcap;
  int32_t* rank = s.rank + (size_t)b * s.hcap;
  for (int32_t j = tid; j < V0; j += PG_SPEC_THREADS) {
    const double d = pg_norm2(g.xy[j], q);
    if (d <= rs) { const int k = atomicAdd(&sh_i[3], 1); tid_[k] = j; td_[k] = d; rank[k] = 0; }
  }
  __syncthreads();
  const int32_t k_hits = sh_i[3];
  // kd pre-order: rank = number of hits that precede
  for (int64_t p = tid; p < (int64_t)k_hits * k_hits; p += PG_SPEC_THREADS) {
    const int32_t x = (int32_t)(p / k_hits), y = (int32_t)(p % k_hits);
    if (x != y && pg_precedes(g, tid_[y], tid_[x])) atomicAdd(&rank[x], 1);
  }
  __syncthreads();
  int32_t* hid = s.hit_id + (size_t)b * s.hcap;
  double* hd = s.hit_d + (size_t)b * s.hcap;
  int32_t* hv = s.hit_vid + (size_t)b * s.hcap;
  for (int32_t k = tid; k < k_hits; k += PG_SPEC_THREADS) { hid[rank[k]] = tid_[k]; hd[rank[k]] = td_[k]; }
  __syncthreads();
  // edge checks hit -> new state (pto.rs:103-108), one warp per edge; item k_hits is the nearest neighbour's edge
  for (int32_t k = warp; k <= k_hits; k += n_warps) {
    const int32_t from = k < k_hits ? hid[k] : nn;
    const double2 f = g.xy[from];
    const int32_t v = walk_to_validity(m, walk_warp<KIND>(m, make_setup(m, f.x, f.y, q.x, q.y), lane));
    if (lane == 0) { if (k < k_hits) hv[k] = v; else s.nn_vid[b] = v; }
  }
  if (tid == 0) s.n_hits[b] = k_hits;
}

// block-wide exclusive prefix of a 0/1 flag (blockDim.x = PG_COMMIT_THREADS); returns the total
__device__ __forceinline__ int pg_block_scan(bool f, int* pos, int* sh) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const unsigned bal = __ballot_sync(0xffffffffu, f);
  __syncthreads();
  if (lane == 0) sh[warp] = __popc(bal);
  __syncthreads();
  int before = 0, total = 0;
  for (int k = 0; k < PG_COMMIT_THREADS / 32; ++k) { if (k < warp) before += sh[k]; total += sh[k]; }
  *pos = before + __popc(bal & ((1u << lane) - 1u));
  return total;
}

// ---- commit: one CTA per roadmap walks its window in order, each iteration in the order of pto.rs:79-135
__global__ void __launch_bounds__(PG_COMMIT_THREADS) pto_commit_kernel(const PgDev* __restrict__ gs, const SpecDev* __restrict__ ss) {
  const PgDev& g = gs[blockIdx.x];
  const SpecDev& s = ss[blockIdx.x];
  __shared__ int32_t touched[PG_TOUCH_CAP];
  __shared__ int sh_scan[PG_COMMIT_THREADS / 32];
  __shared__ int32_t n_touched, overflow, conflict_nn, conflict_rad, panic_idx, sh_goal;
  int32_t* ctl = g.ctl;
  if (ctl[C_DONE]) return;
  const int tid = threadIdx.x;
  const int32_t it0 = ctl[C_IT], V0 = ctl[C_V], W = ctl[C_W];
  const int32_t Weff = min(W, ctl[C_DRAWN] - it0);
  if (Weff <= 0) return;                                     // waiting for samples
  const int32_t wid = ctl[C_WINDOWS];
  int32_t V = V0, E = ctl[C_E], nfin = ctl[C_NFIN], committed = 0, done = 0, stall = 0;
  bool cut = false;
  if (tid == 0) { n_touched = 0; overflow = 0; }
  __syncthreads();
  for (int b = 0; b < Weff; ++b) {
    const int i = it0 + 1 + b;
    const int32_t sv = s.svid[b];
    const double2 q = s.q[b];
    if (b > 0) {                                             // could anything committed in this window change i's answers?
      if (tid == 0) { conflict_nn = overflow; conflict_rad = 0; }
      __syncthreads();
      const int world = g.worlds[i - 1];
      const double2 smp = g.samples[i - 1];
      const double dlim = s.nn_d[b] * (1.0 + 1e-14);           // (a) + a few ulps for the rounding corner of the kd pruning test
      for (int32_t j = V0 + tid; j < V; j += PG_COMMIT_THREADS)
        if (pg_bit(g.reach + (size_t)j * g.words, world) && pg_norm2(g.xy[j], smp) <= dlim) conflict_nn = 1;
      for (int k = tid; k < n_touched; k += PG_COMMIT_THREADS) {
        const int32_t t = touched[k];
        if (pg_bit(g.gain + (size_t)t * g.words, world) && pg_norm2(g.xy[t], smp) <= dlim) conflict_nn = 1;
      }
      if (sv >= 0) {
        const double r = g.radius[V + 1];
        for (int32_t j = V0 + tid; j < V; j += PG_COMMIT_THREADS)   // (b)
          if (pg_norm2(g.xy[j], q) <= r) conflict_rad = 1;
        if (tid == 0 && g.child[s.slot[b]] >= 0) conflict_rad = 1;   // (c)
      }
      __syncthreads();
      if (conflict_nn || conflict_rad) {
        if (tid == 0) {
          ctl[C_RESPEC] += Weff - b;
          if (conflict_nn) ctl[C_CONF_NN] += 1; else ctl[C_CONF_RAD] += 1;
        }
        cut = true;
        break;
      }
    }
    if (sv < -1) { if (tid == 0) ctl[C_PANIC] = sv; done = 2; committed = b; break; }   // state_validity panics (map_io.rs:487-493)
    if (sv >= 0) {
      const int32_t k_hits = s.n_hits[b];
      if (V + 1 > ctl[C_NODE_CAP] || (int64_t)E + k_hits + 1 > (int64_t)ctl[C_EDGE_CAP]) { stall = 1; break; }   // the host grows the buffers
      const int32_t nw = V;
      const double r = g.radius[V + 1];                        // heuristic_radius(nodes after add_node)
      const int32_t* hid = s.hit_id + (size_t)b * s.hcap;
      const double* hd = s.hit_d + (size_t)b * s.hcap;
      const int32_t* hv = s.hit_vid + (size_t)b * s.hcap;
      if (tid == 0) panic_idx = INT_MAX;
      __syncthreads();
      // 1. neighbours = the hits within the exact radius, kd order kept; their valid edges go to the log in that order
      int base = 0, kept_any = 0;
      for (int32_t c0 = 0; c0 < k_hits; c0 += PG_COMMIT_THREADS) {
        const int32_t k = c0 + tid;
        const bool kept = k < k_hits && hd[k] <= r;
        const int32_t v = kept ? hv[k] : -1;
        if (kept && v < -1) atomicMin(&panic_idx, k);
        int pos;
        const int tot = pg_block_scan(kept && v >= 0, &pos, sh_scan);
        if (kept && v >= 0) { g.log_nbr[E + base + pos] = hid[k]; g.log_vid[E + base + pos] = v; }
        base += tot;
        kept_any |= __syncthreads_or(kept);
      }
      __syncthreads();
      int32_t pcode = panic_idx < INT_MAX ? hv[panic_idx] : 0;
      if (!kept_any) {                                         // no neighbour within the radius: [nearest] (pto.rs:100-102)
        const int32_t v = s.nn_vid[b];
        if (v < -1) pcode = v;
        else if (v >= 0) { if (tid == 0) { g.log_nbr[E] = s.nn[b]; g.log_vid[E] = v; } base = 1; }
      }
      if (pcode < -1) { if (tid == 0) ctl[C_PANIC] = pcode; done = 2; committed = b; break; }   // 2. an edge check panics
      const int32_t ne = base;
      __syncthreads();
      // 3. reach.add_edge(e, new) for every kept e, then reach.add_edge(new, e); record the bits gained
      const int words = g.words;
      uint64_t* rn = g.reach + (size_t)nw * words;
      for (int w = tid; w < words; w += PG_COMMIT_THREADS) { rn[w] = 0ull; g.gain[(size_t)nw * words + w] = 0ull; }
      __syncthreads();
      for (int64_t p = tid; p < (int64_t)ne * words; p += PG_COMMIT_THREADS) {   // one (edge, word) per thread: OR is order-free
        const int32_t k = (int32_t)(p / words), w = (int32_t)(p % words);
        const uint64_t c = g.reach[(size_t)g.log_nbr[E + k] * words + w] & g.validities[(size_t)g.log_vid[E + k] * words + w];
        if (c) atomicOr((unsigned long long*)(rn + w), (unsigned long long)c);
      }
      __syncthreads();
      for (int64_t p = tid; p < (int64_t)ne * words; p += PG_COMMIT_THREADS) {
        const int32_t k = (int32_t)(p / words), w = (int32_t)(p % words);
        const int32_t e = g.log_nbr[E + k];
        uint64_t* re = g.reach + (size_t)e * words + w;
        const uint64_t gained = rn[w] & g.validities[(size_t)g.log_vid[E + k] * words + w] & ~*re;
        if (gained) {
          *re |= gained;
          if (e < V0) {
            if (atomicExch(&g.epoch[e], wid) != wid) {
              const int slot = atomicAdd(&n_touched, 1);
              if (slot < PG_TOUCH_CAP) touched[slot] = e; else overflow = 1;
            }
            atomicOr((unsigned long long*)(g.gain + (size_t)e * words + w), (unsigned long long)gained);
          }
        }
      }
      __syncthreads();
      // 4. the node, its edges, the goal test (first goal with norm1 < max_dist), the kd slot, finality
      if (tid == 0) {
        g.xy[nw] = q; g.node_vid[nw] = sv; g.edge_off[nw] = E; g.ecnt[nw] = ne; g.final_idx[nw] = -1;
        g.epoch[nw] = -1;
        const int32_t slot = s.slot[b], p = slot >> 1;
        g.child[2 * nw] = g.child[2 * nw + 1] = -1;
        g.child[slot] = nw; g.parent[nw] = p;
        const int32_t dp = g.depth[p];
        g.depth[nw] = dp + 1;
        g.key[nw] = dp < 64 ? (g.key[p] | ((uint64_t)(slot & 1) << (63 - dp))) : g.key[p];
        int32_t hit = -1;
        for (int32_t k = 0; k < g.n_goals && hit < 0; ++k) {
          const double2 gl = g.goals[k];
          if (__dadd_rn(fabs(__dsub_rn(gl.x, q.x)), fabs(__dsub_rn(gl.y, q.y))) < g.goal_max_dist) hit = k;
        }
        if (hit >= 0) { g.final_idx[nw] = nfin; g.fin_ids[nfin] = nw; g.fin_goal[nfin] = hit; }
        sh_goal = hit;
      }
      __syncthreads();
      if (sh_goal >= 0) ++nfin;
      for (int64_t p = tid; p < (int64_t)(ne + 1) * words; p += PG_COMMIT_THREADS) {   // update_finality: accumulates, never clears
        const int32_t k = (int32_t)(p / words), w = (int32_t)(p % words);
        const int32_t e = k < ne ? g.log_nbr[E + k] : nw, fi = g.final_idx[e];
        if (fi >= 0) {
          const uint64_t f = g.reach[(size_t)e * words + w] & g.goal_masks[(size_t)g.fin_goal[fi] * words + w];
          if (f) atomicOr((unsigned long long*)(g.fin_acc + w), (unsigned long long)f);
        }
      }
      E += ne;
      ++V;
    }
    committed = b + 1;
    // 5. the loop condition: i < n_iter_min || (!is_final_set_complete && i < n_iter_max)
    __syncthreads();
    bool all = nfin > 0;
    for (int w = tid; w < g.words; w += PG_COMMIT_THREADS) {
      const int rem = g.n_worlds - 64 * w;
      const uint64_t want = rem >= 64 ? ~0ull : ((1ull << rem) - 1ull);
      if ((g.fin_acc[w] & want) != want) all = false;
    }
    const bool complete = __syncthreads_and(all);
    if (!((int64_t)i < g.n_iter_min || (!complete && (int64_t)i < g.n_iter_max))) { done = 1; break; }
    if (overflow) { cut = true; break; }                      // gained bits no longer tracked: end the window here
  }
  __syncthreads();
  if (overflow)                                               // (rare) some gains went unlisted: clear them all
    for (int64_t p = tid; p < (int64_t)V0 * g.words; p += PG_COMMIT_THREADS) g.gain[p] = 0ull;
  else
    for (int k = tid; k < n_touched; k += PG_COMMIT_THREADS)
      for (int w = 0; w < g.words; ++w) g.gain[(size_t)touched[k] * g.words + w] = 0ull;
  if (tid == 0) {
    ctl[C_V] = V; ctl[C_E] = E; ctl[C_NFIN] = nfin; ctl[C_IT] = it0 + committed;
    ctl[C_WINDOWS] = wid + 1;
    if (done) ctl[C_DONE] = done;
    ctl[C_STALL] = stall;
    ctl[C_W] = cut ? max(PG_WMIN, 2 * committed) : (stall ? W : min(PG_WMAX, 2 * W));
  }
}

// start: node 0 (KdTree root, Reachability::set_root) or the panic of expect("Start from a valid state!"); one CTA per roadmap
__global__ void pto_init_kernel(MapDev m, const PgDev* __restrict__ gs, double2 start) {
  const PgDev& g = gs[blockIdx.x];
  const int tid = threadIdx.x;
  int32_t* ctl = g.ctl;
  const int32_t sv = state_validity_of(m, start.x, start.y);
  if (tid == 0) {
    ctl[C_V] = 1; ctl[C_IT] = 0; ctl[C_W] = PG_WMIN * 2; ctl[C_DONE] = 0; ctl[C_PANIC] = sv < 0 ? sv : 0;
    ctl[C_STALL] = 0; ctl[C_NFIN] = 0; ctl[C_E] = 0; ctl[C_WINDOWS] = 0; ctl[C_RESPEC] = 0; ctl[C_CONF_NN] = 0; ctl[C_CONF_RAD] = 0;
    if (sv < 0) ctl[C_DONE] = 2;
    g.xy[0] = start; g.node_vid[0] = sv; g.child[0] = g.child[1] = -1; g.parent[0] = -1; g.depth[0] = 0; g.key[0] = 0ull;
    g.final_idx[0] = -1; g.epoch[0] = -1; g.edge_off[0] = 0; g.ecnt[0] = 0;
  }
  for (int w = tid; w < g.words; w += blockDim.x) {
    g.reach[w] = sv >= 0 ? g.validities[(size_t)sv * g.words + w] : 0ull;
    g.gain[w] = 0ull;
    g.fin_acc[w] = 0ull;
  }
}

// what the host grew or drew since the last look: caps[3 r ..] = node cap, edge cap, samples drawn of roadmap r
__global__ void pto_caps_kernel(int32_t* ctl, const int32_t* __restrict__ caps, int n) {
  const int r = blockIdx.x * blockDim.x + threadIdx.x;
  if (r >= n) return;
  ctl[(size_t)r * C_N + C_NODE_CAP] = caps[3 * r];
  ctl[(size_t)r * C_N + C_EDGE_CAP] = caps[3 * r + 1];
  ctl[(size_t)r * C_N + C_DRAWN] = caps[3 * r + 2];
}
// every control block into pinned host memory in one look (no DMA engine, like read_flags_dev)
__global__ void pto_ctl_to_host_kernel(const int32_t* __restrict__ d, int n, volatile int32_t* h) {
  for (int k = blockIdx.x * blockDim.x + threadIdx.x; k < n; k += gridDim.x * blockDim.x) h[k] = d[k];
}
__global__ void pto_set_i64_kernel(int64_t* p, const int32_t* ctl, int idx) { *p = ctl[idx]; }

// ------------------------------------------------------------------------------------------------ host
static PgDev pg_dev(porrt_ctx* ctx, PtoGrow* g, PtoRoad* r, int32_t* ctl, double max_step, double goal_max_dist, int n_goals,
                    int64_t nmin, int64_t nmax) {
  PgDev d = {};
  d.xy = r->xy.as<double2>(); d.node_vid = r->node_vid.as<int32_t>(); d.reach = r->reach.as<uint64_t>(); d.child = r->child.as<int32_t>();
  d.parent = r->parent.as<int32_t>(); d.depth = r->depth.as<int32_t>(); d.key = r->key.as<uint64_t>(); d.final_idx = r->final_idx.as<int32_t>();
  d.gain = r->gain.as<uint64_t>(); d.epoch = r->epoch.as<int32_t>(); d.edge_off = r->edge_off.as<int64_t>(); d.ecnt = r->ecnt.as<int32_t>();
  d.fin_ids = r->fin_ids.as<int32_t>(); d.fin_goal = r->fin_goal.as<int32_t>(); d.fin_acc = r->fin_acc.as<uint64_t>();
  d.log_nbr = r->log_nbr.as<int32_t>(); d.log_vid = r->log_vid.as<int32_t>();
  d.samples = r->samples.as<double2>(); d.worlds = r->worlds.as<int32_t>(); d.radius = g->radius.as<double>();
  d.goals = g->goals.as<double2>(); d.goal_masks = g->goal_masks.as<uint64_t>(); d.validities = ctx->d_validities.as<uint64_t>();
  d.ctl = ctl;
  d.words = g->words; d.n_worlds = ctx->n_worlds; d.n_goals = n_goals; d.goal_max_dist = goal_max_dist; d.max_step = max_step;
  d.n_iter_min = nmin; d.n_iter_max = nmax;
  return d;
}

// the speculation block of a roadmap with h hits per slot: 44 bytes per slot, 32 per hit.  The kernels index slot b < C_W <= PG_WMAX
// and hit k < V0 <= node_cap = hcap.
static void spec_layout(Carve& c, SpecDev& s, int64_t h) {
  const size_t W = PG_WMAX, Wh = W * (size_t)h;
  s.nn = c.take<int32_t>(W); s.nn_d = c.take<double>(W); s.q = c.take<double2>(W); s.svid = c.take<int32_t>(W);
  s.nn_vid = c.take<int32_t>(W); s.n_hits = c.take<int32_t>(W); s.slot = c.take<int32_t>(W);
  s.hit_id = c.take<int32_t>(Wh); s.hit_d = c.take<double>(Wh); s.hit_vid = c.take<int32_t>(Wh);
  s.tmp_id = c.take<int32_t>(Wh); s.tmp_d = c.take<double>(Wh); s.rank = c.take<int32_t>(Wh);
  s.hcap = h;
}
static size_t spec_bytes(int64_t h) { SpecDev s; return carve_size([&](Carve& c) { spec_layout(c, s, h); }); }
static SpecDev spec_dev(PtoRoad* r) { SpecDev s = {}; Carve c{(uintptr_t)r->spec.p}; spec_layout(c, s, r->node_cap); return s; }
static size_t node_bytes(int words) { return 72 + 16 * (size_t)words; }   // every per-node array below, per node

// every per-node array holds node_cap entries, kept across growth (DevBuf::grow_keep)
static int32_t pg_grow_nodes(porrt_ctx* ctx, PtoRoad* g, int words, int64_t want, int64_t V_now) {
  if (want <= g->node_cap) return PORRT_OK;
  const int64_t cap = std::max<int64_t>(want, 2 * g->node_cap);
  cudaStream_t st = ctx->stream;
  const size_t w8 = (size_t)words * 8;
  struct { DevBuf* b; size_t per; } arr[] = {{&g->xy, 16}, {&g->node_vid, 4}, {&g->reach, w8}, {&g->child, 8}, {&g->parent, 4},
      {&g->depth, 4}, {&g->key, 8}, {&g->final_idx, 4}, {&g->gain, w8}, {&g->epoch, 4}, {&g->edge_off, 8}, {&g->ecnt, 4},
      {&g->fin_ids, 4}, {&g->fin_goal, 4}};
  for (auto& a : arr) CUDA_TRY(ctx, a.b->grow_keep((size_t)(cap + 1) * a.per, (size_t)(V_now + 1) * a.per, st));
  CUDA_TRY(ctx, g->spec.ensure(spec_bytes(cap)));
  g->node_cap = cap;
  return PORRT_OK;
}

// heuristic_radius(n) for every n a window can reach (host libm, DESIGN.md 4)
static int32_t pg_radius_table(porrt_ctx* ctx, PtoGrow* g, int64_t node_cap, double max_step, double search_radius) {
  const int64_t rn = node_cap + PG_WMAX + 2;
  if (rn <= g->radius_n) return PORRT_OK;
  std::vector<double> r((size_t)rn);
  for (int64_t n = 0; n < rn; ++n) r[(size_t)n] = n == 0 ? 0.0 : heuristic_radius(n, max_step, search_radius, 2);
  CUDA_TRY(ctx, g->radius.ensure((size_t)rn * 8));
  CUDA_TRY(ctx, cudaMemcpyAsync(g->radius.p, r.data(), (size_t)rn * 8, cudaMemcpyHostToDevice, ctx->stream));
  CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
  g->radius_n = rn;
  return PORRT_OK;
}

// one host sample stream per roadmap: pto.rs:141-149, the continuous and the discrete sampler seeded alike
struct PgStream {
  Pcg64 cont, disc;
  int64_t drawn;
  std::vector<double> smp;      // the last draw, until its copy has run (the next look synchronises first)
  std::vector<int32_t> wld;
};

// PTO::grow_graph for n roadmaps that differ only in their sampler seed.  Every roadmap runs the host decisions and the windows the
// single growth would run: each look grows its buffers and draws its samples by the same rules, then PG_BATCH windows of every
// roadmap that is still running go out in one speculate and one commit launch per window.
static int32_t pto_grow_impl(porrt_ctx* ctx, const char* who, int32_t n, const uint64_t* seeds, const double start[2], const double low[2],
                             const double up[2], const double* goals_xy, const uint64_t* goal_masks, int32_t n_goals, double goal_max_dist,
                             double max_step, double search_radius, int64_t n_iter_min, int64_t n_iter_max, int64_t* out_sizes,
                             int32_t* out_status, int32_t* out_panic_code, int64_t* out_counters) {
  CTX_CHECK(ctx);
  if (!ctx->has_map) return porrt_fail(ctx, PORRT_ERR_NO_MAP, "no map uploaded");
  if (!start || !low || !up || (n_goals > 0 && (!goals_xy || !goal_masks)) || n_goals < 0 || n_iter_min < 0 || n_iter_max < 0 ||
      !out_sizes || !out_status || !seeds)
    return porrt_fail(ctx, PORRT_ERR_INVALID_ARG, std::string(who) + ": bad arguments");
  if (n < 1 || n > PORRT_PTO_MAX_ROADMAPS)
    return porrt_fail(ctx, PORRT_ERR_INVALID_ARG, std::string(who) + ": n_roadmaps must be in 1 .. " + std::to_string(PORRT_PTO_MAX_ROADMAPS));
  if (!ctx->pto) ctx->pto = new PtoGrow();
  PtoGrow* g = ctx->pto;
  g->n_have = 0;
  for (auto& r : g->roads) r->have = false;
  for (int64_t k = 0; k < 4 * (int64_t)n; ++k) out_sizes[k] = 0;
  for (int32_t r = 0; r < n; ++r) out_status[r] = 0;
  if (out_panic_code) for (int32_t r = 0; r < n; ++r) out_panic_code[r] = 0;
  if (out_counters) for (int64_t k = 0; k < 4 * (int64_t)n; ++k) out_counters[k] = 0;
  const int words = ctx->mask_words, n_worlds = ctx->n_worlds;
  // SquareGoal::new (common.rs:304-350): world_to_goal, asserting that no world has two goals (:320)
  std::vector<double> world_goal((size_t)n_worlds * 2, 0.0);
  if (n_goals > 0 && porrt_square_goal_examples(goals_xy, goal_masks, n_goals, n_worlds, world_goal.data()) == PORRT_ERR_PANIC)
    return porrt_fail(ctx, PORRT_ERR_PANIC, "SquareGoal: validities shouldn't overlap (common.rs:320)");
  for (int d = 0; d < 2; ++d)
    if (!(low[d] < up[d]) || !std::isfinite(low[d]) || !std::isfinite(up[d]))
      return porrt_fail(ctx, PORRT_ERR_PANIC, "ContinuousSampler: low < up required (rand asserts it)");
  CUDA_TRY(ctx, cudaSetDevice(ctx->device));
  cudaStream_t st = ctx->stream;
  // the loop runs at least n_iter_min and at most max(n_iter_min, n_iter_max) iterations
  const int64_t bound = std::min<int64_t>(std::max(n_iter_min, n_iter_max), INT32_MAX - 2 * PG_WMAX);
  const bool runs = 0 < n_iter_min || 0 < n_iter_max;   // the loop condition before the first iteration (no finals yet)
  const int64_t cap0 = std::min<int64_t>(bound, 4096) + PG_BATCH * PG_WMAX + 1;
  const int64_t draw0 = runs ? std::min(n_iter_min + 4096, bound) : 0;
  {  // every roadmap must fit at its starting size: what the buffers below take, growth factors included
    const double per = 1.5 * (double)(cap0 + 1) * node_bytes(words) + 1.25 * spec_bytes(cap0) + 2 * 1.25 * 64.0 * cap0 +
                       1.5 * 20.0 * draw0 + 1e5;
    size_t free_b = 0, total_b = 0;
    CUDA_TRY(ctx, cudaMemGetInfo(&free_b, &total_b));
    double held = 0;
    for (auto& r : g->roads) held += (double)r->bytes();
    if ((double)n * per > (double)free_b + held)
      return porrt_fail(ctx, PORRT_ERR_INVALID_ARG, std::string(who) + ": " + std::to_string(n) + " roadmaps need about " +
                        std::to_string((int64_t)(n * per / 1e6)) + " MB to start, the device has " +
                        std::to_string((int64_t)((free_b + held) / 1e6)) + " MB");
  }
  for (size_t r = (size_t)n; r < g->roads.size(); ++r) g->roads[r]->release();
  g->roads.resize((size_t)n);
  for (auto& r : g->roads) if (!r) r.reset(new PtoRoad());
  g->words = words;
  g->goal_masks_host.assign(goal_masks ? goal_masks : nullptr, goal_masks ? goal_masks + (size_t)n_goals * words : nullptr);
  // buffers: nodes grow with the roadmap, samples are drawn ahead of the windows
  g->radius_n = 0;
  int32_t rc;
  for (auto& rp : g->roads) {
    PtoRoad* r = rp.get();
    r->node_cap = 0;
    if ((rc = pg_grow_nodes(ctx, r, words, cap0, 0))) return rc;
    r->edge_cap = std::max<int64_t>(r->edge_cap, 16 * r->node_cap);
    CUDA_TRY(ctx, r->log_nbr.ensure((size_t)r->edge_cap * 4));
    CUDA_TRY(ctx, r->log_vid.ensure((size_t)r->edge_cap * 4));
    CUDA_TRY(ctx, r->fin_acc.ensure((size_t)words * 8));
  }
  if ((rc = pg_radius_table(ctx, g, cap0, max_step, search_radius))) return rc;
  CUDA_TRY(ctx, g->goals.ensure((size_t)std::max(n_goals, 1) * 16));
  CUDA_TRY(ctx, g->goal_masks.ensure((size_t)std::max(n_goals, 1) * words * 8));
  CUDA_TRY(ctx, g->ctl.ensure((size_t)n * C_N * 4 + 64));
  CUDA_TRY(ctx, g->ctl_host.ensure((size_t)n * C_N * 4));
  CUDA_TRY(ctx, g->caps.ensure((size_t)n * 3 * 4));
  CUDA_TRY(ctx, g->pg_desc.ensure((size_t)n * sizeof(PgDev)));
  CUDA_TRY(ctx, g->spec_desc.ensure((size_t)n * sizeof(SpecDev)));
  if (n_goals > 0) {
    CUDA_TRY(ctx, cudaMemcpyAsync(g->goals.p, goals_xy, (size_t)n_goals * 16, cudaMemcpyHostToDevice, st));
    CUDA_TRY(ctx, cudaMemcpyAsync(g->goal_masks.p, goal_masks, (size_t)n_goals * words * 8, cudaMemcpyHostToDevice, st));
  }
  int32_t* ctl = g->ctl.as<int32_t>();
  // the descriptors, re-uploaded whenever a buffer moved
  std::vector<char> desc((size_t)n * (sizeof(PgDev) + sizeof(SpecDev)));
  g->desc_host.clear();
  auto upload_desc = [&]() -> int32_t {
    PgDev* pd = (PgDev*)desc.data();
    SpecDev* sd = (SpecDev*)(desc.data() + (size_t)n * sizeof(PgDev));
    for (int32_t r = 0; r < n; ++r) {
      pd[r] = pg_dev(ctx, g, g->roads[r].get(), ctl + (size_t)r * C_N, max_step, goal_max_dist, n_goals, n_iter_min, n_iter_max);
      sd[r] = spec_dev(g->roads[r].get());
    }
    if (desc == g->desc_host) return PORRT_OK;
    CUDA_TRY(ctx, cudaMemcpyAsync(g->pg_desc.p, pd, (size_t)n * sizeof(PgDev), cudaMemcpyHostToDevice, st));
    CUDA_TRY(ctx, cudaMemcpyAsync(g->spec_desc.p, sd, (size_t)n * sizeof(SpecDev), cudaMemcpyHostToDevice, st));
    CUDA_TRY(ctx, cudaStreamSynchronize(st));   // desc is rewritten at the next look
    g->desc_host = desc;
    return PORRT_OK;
  };
  // node cap, edge cap and samples drawn of every roadmap into its control block, when one of them changed
  std::vector<int32_t> caps((size_t)n * 3, 0), caps_dev((size_t)n * 3, -1);
  auto upload_caps = [&]() -> int32_t {
    for (int32_t r = 0; r < n; ++r) {
      caps[3 * (size_t)r] = (int32_t)std::min<int64_t>(g->roads[r]->node_cap, INT32_MAX);
      caps[3 * (size_t)r + 1] = (int32_t)std::min<int64_t>(g->roads[r]->edge_cap, INT32_MAX);
    }
    if (caps == caps_dev) return PORRT_OK;
    CUDA_TRY(ctx, cudaMemcpyAsync(g->caps.p, caps.data(), caps.size() * 4, cudaMemcpyHostToDevice, st));
    pto_caps_kernel<<<div_up(n, 128), 128, 0, st>>>(ctl, g->caps.as<int32_t>(), n);
    LAUNCH_CHECK(ctx);
    CUDA_TRY(ctx, cudaStreamSynchronize(st));   // caps is rewritten at the next look
    caps_dev = caps;
    return PORRT_OK;
  };
  std::vector<PgStream> hs;
  hs.reserve((size_t)n);
  for (int32_t r = 0; r < n; ++r) hs.push_back(PgStream{Pcg64::seed_from_u64(seeds[r]), Pcg64::seed_from_u64(seeds[r]), 0, {}, {}});
  // pto.rs:141-149: one discrete draw per iteration, a continuous draw only when i % 100 != 0 (then goal_example(world))
  auto draw = [&](int32_t r, int64_t upto) -> int32_t {
    PgStream& h = hs[(size_t)r];
    PtoRoad* d = g->roads[r].get();
    upto = std::min(upto, bound);
    if (upto <= h.drawn) return PORRT_OK;
    const int64_t m = upto - h.drawn;
    h.smp.resize((size_t)m * 2); h.wld.resize((size_t)m);
    for (int64_t k = 0; k < m; ++k) {
      const int64_t i = h.drawn + k + 1;
      const int32_t w = (int32_t)h.disc.below((uint64_t)n_worlds);
      h.wld[(size_t)k] = w;
      if (i % 100 == 0) { h.smp[2 * k] = world_goal[2 * (size_t)w]; h.smp[2 * k + 1] = world_goal[2 * (size_t)w + 1]; }
      else { h.smp[2 * k] = h.cont.range_f64(low[0], up[0]); h.smp[2 * k + 1] = h.cont.range_f64(low[1], up[1]); }
    }
    CUDA_TRY(ctx, d->samples.grow_keep((size_t)upto * 16, (size_t)h.drawn * 16, st));
    CUDA_TRY(ctx, d->worlds.grow_keep((size_t)upto * 4, (size_t)h.drawn * 4, st));
    CUDA_TRY(ctx, cudaMemcpyAsync(d->samples.as<double>() + 2 * h.drawn, h.smp.data(), (size_t)m * 16, cudaMemcpyHostToDevice, st));
    CUDA_TRY(ctx, cudaMemcpyAsync(d->worlds.as<int32_t>() + h.drawn, h.wld.data(), (size_t)m * 4, cudaMemcpyHostToDevice, st));
    h.drawn = upto;
    caps[3 * (size_t)r + 2] = (int32_t)upto;
    return PORRT_OK;
  };
  auto look = [&](int32_t* f) -> int32_t {   // every control block
    volatile int32_t* h = g->ctl_host.as<int32_t>();
    const int m = n * C_N;
    pto_ctl_to_host_kernel<<<std::min(div_up(m, 256), 64), 256, 0, st>>>(ctl, m, h);
    LAUNCH_CHECK(ctx);
    CUDA_TRY(ctx, cudaStreamSynchronize(st));
    for (int k = 0; k < m; ++k) f[k] = h[k];
    return PORRT_OK;
  };
  if ((rc = upload_desc())) return rc;
  pto_init_kernel<<<n, 64, 0, st>>>(ctx->map, g->pg_desc.as<PgDev>(), make_double2(start[0], start[1]));
  LAUNCH_CHECK(ctx);
  if (runs) for (int32_t r = 0; r < n; ++r) if ((rc = draw(r, n_iter_min + 4096))) return rc;
  if ((rc = upload_caps())) return rc;
  std::vector<int32_t> fv((size_t)n * C_N);
  int32_t* f = fv.data();
  for (;;) {
    if ((rc = look(f))) return rc;
    if (!runs) break;
    bool running = false;
    int64_t node_cap = 0;
    for (int32_t r = 0; r < n; ++r) {
      const int32_t* fr = f + (size_t)r * C_N;
      PtoRoad* d = g->roads[r].get();
      if (!fr[C_DONE] && fr[C_IT] < bound) {
        running = true;
        const int64_t V = fr[C_V], it = fr[C_IT];
        // room for the next batch of windows: nodes (every commit adds at most one), edges (the commit stalls when they run out)
        if (V + PG_BATCH * PG_WMAX + 1 > d->node_cap && (rc = pg_grow_nodes(ctx, d, words, V + PG_BATCH * PG_WMAX + 1, V))) return rc;
        if (fr[C_STALL] || (int64_t)fr[C_E] + 64 * PG_BATCH * PG_WMAX > d->edge_cap) {
          const int64_t want = std::max<int64_t>(2 * d->edge_cap, (int64_t)fr[C_E] + V + 1 + 64 * PG_BATCH * PG_WMAX);
          CUDA_TRY(ctx, d->log_nbr.grow_keep((size_t)want * 4, (size_t)fr[C_E] * 4, st));
          CUDA_TRY(ctx, d->log_vid.grow_keep((size_t)want * 4, (size_t)fr[C_E] * 4, st));
          d->edge_cap = want;
        }
        const int64_t drawn = hs[(size_t)r].drawn;
        if (drawn < bound && drawn - it < 2 * PG_BATCH * PG_WMAX && (rc = draw(r, drawn + std::max<int64_t>(4096, drawn / 2)))) return rc;
      }
      node_cap = std::max(node_cap, d->node_cap);
    }
    if (!running) break;
    if ((rc = pg_radius_table(ctx, g, node_cap, max_step, search_radius))) return rc;
    if ((rc = upload_caps())) return rc;
    if ((rc = upload_desc())) return rc;
    const PgDev* pd = g->pg_desc.as<PgDev>();
    const SpecDev* sd = g->spec_desc.as<SpecDev>();
    for (int k = 0; k < PG_BATCH; ++k) {
      if (ctx->map.kind == PORRT_DOMAIN_SHELF) pto_speculate_kernel<PORRT_DOMAIN_SHELF><<<dim3(PG_WMAX, n), PG_SPEC_THREADS, 0, st>>>(ctx->map, pd, sd);
      else pto_speculate_kernel<PORRT_DOMAIN_DOOR><<<dim3(PG_WMAX, n), PG_SPEC_THREADS, 0, st>>>(ctx->map, pd, sd);
      LAUNCH_CHECK(ctx);
      pto_commit_kernel<<<n, PG_COMMIT_THREADS, 0, st>>>(pd, sd);
      LAUNCH_CHECK(ctx);
    }
  }
  // per roadmap: outputs, then the children CSR from the edge log (graph.cu's late-list kernels, carrying the validity ids)
  // CSR assembly work space of a roadmap of V nodes and E edges (late_list_csr_dev), one roadmap at a time
  int32_t *late_cnt, *cursor, *late_vals;
  int64_t* late_off;
  auto csr_work = [&](Carve& c, int64_t V, int64_t E) {
    late_cnt = c.take<int32_t>(V); cursor = c.take<int32_t>(V); late_off = c.take<int64_t>(V + 1);
    late_vals = c.take<int32_t>(std::max<int64_t>(E, 1));
  };
  size_t work = 64;
  for (int32_t r = 0; r < n; ++r) {
    const int32_t* fr = f + (size_t)r * C_N;
    int64_t* sz = out_sizes + 4 * (size_t)r;
    sz[0] = fr[C_IT];
    if (out_counters) {
      int64_t* c = out_counters + 4 * (size_t)r;
      c[0] = fr[C_WINDOWS]; c[1] = fr[C_RESPEC]; c[2] = fr[C_CONF_NN]; c[3] = fr[C_CONF_RAD];
    }
    if (fr[C_DONE] == 2) {
      out_status[r] = PORRT_ERR_PANIC;
      if (out_panic_code) out_panic_code[r] = fr[C_PANIC];
      sz[0] = fr[C_WINDOWS] == 0 ? 0 : fr[C_IT] + 1;   // the iteration whose check panicked; 0: the init kernel found the start invalid
      continue;
    }
    const int64_t V = fr[C_V], E = fr[C_E];
    work = std::max(work, carve_size([&](Carve& c) { csr_work(c, V, E); }));
  }
  CUDA_TRY(ctx, g->work.ensure(work));
  std::vector<uint64_t> fin((size_t)n * words);
  for (int32_t r = 0; r < n; ++r) {
    const int32_t* fr = f + (size_t)r * C_N;
    if (out_status[r] == PORRT_ERR_PANIC) continue;
    PtoRoad* d = g->roads[r].get();
    const int64_t V = fr[C_V], E = fr[C_E];
    CUDA_TRY(ctx, d->csr_row.ensure((size_t)(V + 1) * 8));
    CUDA_TRY(ctx, d->csr_col.ensure((size_t)std::max<int64_t>(2 * E, 1) * 4));
    CUDA_TRY(ctx, d->csr_vid.ensure((size_t)std::max<int64_t>(2 * E, 1) * 4));
    Carve c{(uintptr_t)g->work.p};
    csr_work(c, V, E);
    pto_set_i64_kernel<<<1, 1, 0, st>>>(d->edge_off.as<int64_t>() + V, ctl + (size_t)r * C_N, C_E);
    LAUNCH_CHECK(ctx);
    rc = late_list_csr_dev(ctx, d->edge_off.as<int64_t>(), V, d->log_nbr.as<int32_t>(), d->ecnt.as<int32_t>(), d->log_vid.as<int32_t>(),
                           late_cnt, cursor, late_off, late_vals, d->csr_row.as<int64_t>(), d->csr_col.as<int32_t>(), d->csr_vid.as<int32_t>());
    if (rc) return rc;
    CUDA_TRY(ctx, cudaMemcpyAsync(fin.data() + (size_t)r * words, d->fin_acc.p, (size_t)words * 8, cudaMemcpyDeviceToHost, st));
  }
  CUDA_TRY(ctx, cudaStreamSynchronize(st));
  for (int32_t r = 0; r < n; ++r) {
    if (out_status[r] == PORRT_ERR_PANIC) continue;
    const int32_t* fr = f + (size_t)r * C_N;
    PtoRoad* d = g->roads[r].get();
    bool complete = fr[C_NFIN] > 0;
    for (int w = 0; w < words; ++w) {
      const int rem = n_worlds - 64 * w;
      const uint64_t want = rem >= 64 ? ~0ull : ((1ull << rem) - 1ull);
      if ((fin[(size_t)r * words + w] & want) != want) complete = false;
    }
    d->have = true; d->V = fr[C_V]; d->E = 2 * (int64_t)fr[C_E]; d->n_finals = fr[C_NFIN];
    int64_t* sz = out_sizes + 4 * (size_t)r;
    sz[1] = d->V; sz[2] = d->E; sz[3] = d->n_finals;
    out_status[r] = complete ? 0 : 1;
  }
  g->n_have = n;
  return PORRT_OK;
}

PORRT_API int32_t porrt_pto_grow(porrt_ctx* ctx, const double start[2], const double low[2], const double up[2], uint64_t sampler_seed,
                                 const double* goals_xy, const uint64_t* goal_masks, int32_t n_goals, double goal_max_dist,
                                 double max_step, double search_radius, int64_t n_iter_min, int64_t n_iter_max,
                                 int64_t* out_sizes, int32_t* out_complete, int32_t* out_panic_code, int64_t* out_counters) {
  CTX_CHECK(ctx);
  if (!ctx->has_map) return porrt_fail(ctx, PORRT_ERR_NO_MAP, "no map uploaded");
  if (!out_complete) return porrt_fail(ctx, PORRT_ERR_INVALID_ARG, "porrt_pto_grow: bad arguments");
  int32_t status = 0, panic = 0;
  const int32_t rc = pto_grow_impl(ctx, "porrt_pto_grow", 1, &sampler_seed, start, low, up, goals_xy, goal_masks, n_goals, goal_max_dist,
                                   max_step, search_radius, n_iter_min, n_iter_max, out_sizes, &status, &panic, out_counters);
  *out_complete = rc == PORRT_OK && status == 0 ? 1 : 0;
  if (rc) return rc;
  if (out_panic_code) *out_panic_code = panic;
  if (status != PORRT_ERR_PANIC) return PORRT_OK;
  return porrt_fail(ctx, PORRT_ERR_PANIC, out_sizes[0] == 0 ? "Start from a valid state! (pto.rs:57, state validity code " + std::to_string(panic) + ")"
                                                            : "porrt_pto_grow: a state / edge check hit a reference panic (code " + std::to_string(panic) + ")");
}

PORRT_API int32_t porrt_pto_grow_batch(porrt_ctx* ctx, int32_t n_roadmaps, const uint64_t* sampler_seeds, const double start[2],
                                       const double low[2], const double up[2], const double* goals_xy, const uint64_t* goal_masks,
                                       int32_t n_goals, double goal_max_dist, double max_step, double search_radius, int64_t n_iter_min,
                                       int64_t n_iter_max, int64_t* out_sizes, int32_t* out_status, int32_t* out_panic_code,
                                       int64_t* out_counters) {
  return pto_grow_impl(ctx, "porrt_pto_grow_batch", n_roadmaps, sampler_seeds, start, low, up, goals_xy, goal_masks, n_goals, goal_max_dist,
                       max_step, search_radius, n_iter_min, n_iter_max, out_sizes, out_status, out_panic_code, out_counters);
}

PORRT_API int32_t porrt_pto_fetch_roadmap(porrt_ctx* ctx, int32_t r, double* out_xy, int32_t* out_node_vid, int64_t* out_row_ptr,
                                          int32_t* out_col, int32_t* out_edge_vid, uint64_t* out_reach, int64_t* out_final_ids,
                                          uint64_t* out_final_masks) {
  CTX_CHECK(ctx);
  PtoGrow* pg = ctx->pto;
  if (!pg || pg->n_have == 0) return porrt_fail(ctx, PORRT_ERR_INVALID_ARG, "porrt_pto_fetch: no roadmap grown on this ctx");
  if (r < 0 || r >= pg->n_have)
    return porrt_fail(ctx, PORRT_ERR_INVALID_ARG, "porrt_pto_fetch_roadmap: roadmap " + std::to_string(r) + " of " + std::to_string(pg->n_have));
  const PtoRoad* g = pg->roads[r].get();
  if (!g->have) return porrt_fail(ctx, PORRT_ERR_INVALID_ARG, "porrt_pto_fetch: roadmap " + std::to_string(r) + " panicked");
  CUDA_TRY(ctx, cudaSetDevice(ctx->device));
  cudaStream_t st = ctx->stream;
  const int64_t V = g->V, E = g->E, F = g->n_finals;
  const size_t words = (size_t)pg->words;
  if (out_xy) CUDA_TRY(ctx, cudaMemcpyAsync(out_xy, g->xy.p, (size_t)V * 16, cudaMemcpyDeviceToHost, st));
  if (out_node_vid) CUDA_TRY(ctx, cudaMemcpyAsync(out_node_vid, g->node_vid.p, (size_t)V * 4, cudaMemcpyDeviceToHost, st));
  if (out_row_ptr) CUDA_TRY(ctx, cudaMemcpyAsync(out_row_ptr, g->csr_row.p, (size_t)(V + 1) * 8, cudaMemcpyDeviceToHost, st));
  if (out_col && E) CUDA_TRY(ctx, cudaMemcpyAsync(out_col, g->csr_col.p, (size_t)E * 4, cudaMemcpyDeviceToHost, st));
  if (out_edge_vid && E) CUDA_TRY(ctx, cudaMemcpyAsync(out_edge_vid, g->csr_vid.p, (size_t)E * 4, cudaMemcpyDeviceToHost, st));
  if (out_reach) CUDA_TRY(ctx, cudaMemcpyAsync(out_reach, g->reach.p, (size_t)V * words * 8, cudaMemcpyDeviceToHost, st));
  std::vector<int32_t> ids((size_t)F), goal((size_t)F);
  if (F) {
    CUDA_TRY(ctx, cudaMemcpyAsync(ids.data(), g->fin_ids.p, (size_t)F * 4, cudaMemcpyDeviceToHost, st));
    CUDA_TRY(ctx, cudaMemcpyAsync(goal.data(), g->fin_goal.p, (size_t)F * 4, cudaMemcpyDeviceToHost, st));
  }
  CUDA_TRY(ctx, cudaStreamSynchronize(st));
  for (int64_t k = 0; k < F; ++k) {
    if (out_final_ids) out_final_ids[k] = ids[(size_t)k];
    if (out_final_masks) memcpy(out_final_masks + (size_t)k * words, pg->goal_masks_host.data() + (size_t)goal[(size_t)k] * words, words * 8);
  }
  return PORRT_OK;
}

PORRT_API int32_t porrt_pto_fetch(porrt_ctx* ctx, double* out_xy, int32_t* out_node_vid, int64_t* out_row_ptr, int32_t* out_col,
                                  int32_t* out_edge_vid, uint64_t* out_reach, int64_t* out_final_ids, uint64_t* out_final_masks) {
  return porrt_pto_fetch_roadmap(ctx, 0, out_xy, out_node_vid, out_row_ptr, out_col, out_edge_vid, out_reach, out_final_ids, out_final_masks);
}
