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
#include <algorithm>
#include <cmath>
#include <climits>

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

struct PtoGrow {
  // roadmap [node_cap]
  DevBuf xy, node_vid, reach, child, parent, depth, key, final_idx, gain, epoch, edge_off, ecnt;
  DevBuf fin_ids, fin_goal, fin_acc;          // finals in add order, the goal each one hit, accumulated finality [words]
  DevBuf log_nbr, log_vid;                    // edge log (neighbour, validity id) grouped by new node, commit order
  DevBuf samples, worlds, radius;             // iteration i (1-based) at [i - 1]; heuristic_radius(n) at [n]
  DevBuf goals, goal_masks, ctl;
  DevBuf spec;                                // per-slot speculation results + hit lists [PG_WMAX * node_cap]
  DevBuf csr_row, csr_col, csr_vid, work;     // the assembled roadmap + assembly work space
  int64_t node_cap = 0, edge_cap = 0, drawn_cap = 0, radius_n = 0;
  int words = 1;
  // the last result (porrt_pto_fetch)
  bool have = false;
  int64_t V = 0, E = 0, n_finals = 0;
  std::vector<uint64_t> goal_masks_host;
};

void pto_grow_release(porrt_ctx* ctx) {
  PtoGrow* g = ctx->pto;
  if (!g) return;
  DevBuf* all[] = {&g->xy, &g->node_vid, &g->reach, &g->child, &g->parent, &g->depth, &g->key, &g->final_idx, &g->gain, &g->epoch,
                   &g->edge_off, &g->ecnt, &g->fin_ids, &g->fin_goal, &g->fin_acc, &g->log_nbr, &g->log_vid, &g->samples, &g->worlds,
                   &g->radius, &g->goals, &g->goal_masks, &g->ctl, &g->spec, &g->csr_row, &g->csr_col, &g->csr_vid, &g->work};
  for (DevBuf* b : all) b->release();
  delete g;
  ctx->pto = nullptr;
}

// ------------------------------------------------------------------------------------------------ device
struct PgDev {     // roadmap pointers (by value into every kernel)
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

// ---- speculate: one CTA per iteration of the window, reading only the committed state S0
template <int KIND>
__global__ void __launch_bounds__(PG_SPEC_THREADS) pto_speculate_kernel(MapDev m, PgDev g, SpecDev s) {
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

// ---- commit: one CTA walks the window in order, each iteration in the order of pto.rs:79-135
__global__ void __launch_bounds__(PG_COMMIT_THREADS) pto_commit_kernel(PgDev g, SpecDev s) {
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

// start: node 0 (KdTree root, Reachability::set_root) or the panic of expect("Start from a valid state!")
__global__ void pto_init_kernel(MapDev m, PgDev g, double2 start) {
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

__global__ void pto_set_kernel(int32_t* ctl, int idx, int32_t v) { ctl[idx] = v; }
__global__ void pto_fill_i32_kernel(int32_t* p, int64_t n, int32_t v) {
  const int64_t k = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (k < n) p[k] = v;
}
__global__ void pto_set_i64_kernel(int64_t* p, const int32_t* ctl, int idx) { *p = ctl[idx]; }

// ------------------------------------------------------------------------------------------------ host
static double host_heuristic_radius(int64_t n_nodes, double max_step, double search_radius) {   // common.rs:357-369, host libm
  const double n = (double)n_nodes;
  const double s = search_radius * std::pow(std::log(n) / n, 1.0 / 2.0);
  return s < max_step ? s : max_step;
}

static PgDev pg_dev(porrt_ctx* ctx, PtoGrow* g, double max_step, double goal_max_dist, int n_goals, int64_t nmin, int64_t nmax) {
  PgDev d;
  d.xy = g->xy.as<double2>(); d.node_vid = g->node_vid.as<int32_t>(); d.reach = g->reach.as<uint64_t>(); d.child = g->child.as<int32_t>();
  d.parent = g->parent.as<int32_t>(); d.depth = g->depth.as<int32_t>(); d.key = g->key.as<uint64_t>(); d.final_idx = g->final_idx.as<int32_t>();
  d.gain = g->gain.as<uint64_t>(); d.epoch = g->epoch.as<int32_t>(); d.edge_off = g->edge_off.as<int64_t>(); d.ecnt = g->ecnt.as<int32_t>();
  d.fin_ids = g->fin_ids.as<int32_t>(); d.fin_goal = g->fin_goal.as<int32_t>(); d.fin_acc = g->fin_acc.as<uint64_t>();
  d.log_nbr = g->log_nbr.as<int32_t>(); d.log_vid = g->log_vid.as<int32_t>();
  d.samples = g->samples.as<double2>(); d.worlds = g->worlds.as<int32_t>(); d.radius = g->radius.as<double>();
  d.goals = g->goals.as<double2>(); d.goal_masks = g->goal_masks.as<uint64_t>(); d.validities = ctx->d_validities.as<uint64_t>();
  d.ctl = g->ctl.as<int32_t>();
  d.words = g->words; d.n_worlds = ctx->n_worlds; d.n_goals = n_goals; d.goal_max_dist = goal_max_dist; d.max_step = max_step;
  d.n_iter_min = nmin; d.n_iter_max = nmax;
  return d;
}

static SpecDev spec_dev(PtoGrow* g) {
  SpecDev s;
  const int64_t W = PG_WMAX, h = g->node_cap;
  char* p = g->spec.as<char>();
  auto take = [&](size_t bytes) { char* q = p; p += (bytes + 15) & ~(size_t)15; return q; };
  s.nn = (int32_t*)take(W * 4); s.nn_d = (double*)take(W * 8); s.q = (double2*)take(W * 16); s.svid = (int32_t*)take(W * 4);
  s.nn_vid = (int32_t*)take(W * 4); s.n_hits = (int32_t*)take(W * 4); s.slot = (int32_t*)take(W * 4);
  s.hit_id = (int32_t*)take(W * h * 4); s.hit_d = (double*)take(W * h * 8); s.hit_vid = (int32_t*)take(W * h * 4);
  s.tmp_id = (int32_t*)take(W * h * 4); s.tmp_d = (double*)take(W * h * 8); s.rank = (int32_t*)take(W * h * 4);
  s.hcap = h;
  return s;
}
static size_t spec_bytes(int64_t h) { return (size_t)PG_WMAX * (4 + 8 + 16 + 4 * 4 + (size_t)h * 36) + 16 * 16; }

// every per-node array holds node_cap entries, kept across growth (DevBuf::grow_keep)
static int32_t pg_grow_nodes(porrt_ctx* ctx, PtoGrow* g, int64_t want, int64_t V_now) {
  if (want <= g->node_cap) return PORRT_OK;
  const int64_t cap = std::max<int64_t>(want, 2 * g->node_cap);
  cudaStream_t st = ctx->stream;
  const size_t w8 = (size_t)g->words * 8;
  struct { DevBuf* b; size_t per; } arr[] = {{&g->xy, 16}, {&g->node_vid, 4}, {&g->reach, w8}, {&g->child, 8}, {&g->parent, 4},
      {&g->depth, 4}, {&g->key, 8}, {&g->final_idx, 4}, {&g->gain, w8}, {&g->epoch, 4}, {&g->edge_off, 8}, {&g->ecnt, 4},
      {&g->fin_ids, 4}, {&g->fin_goal, 4}};
  for (auto& a : arr) CUDA_TRY(ctx, a.b->grow_keep((size_t)(cap + 1) * a.per, (size_t)(V_now + 1) * a.per, st));
  CUDA_TRY(ctx, g->spec.ensure(spec_bytes(cap)));
  g->node_cap = cap;
  return PORRT_OK;
}

// heuristic_radius(n) for every n a window can reach (host libm, DESIGN.md 4)
static int32_t pg_radius_table(porrt_ctx* ctx, PtoGrow* g, double max_step, double search_radius) {
  const int64_t rn = g->node_cap + PG_WMAX + 2;
  if (rn <= g->radius_n) return PORRT_OK;
  std::vector<double> r((size_t)rn);
  for (int64_t n = 0; n < rn; ++n) r[(size_t)n] = n == 0 ? 0.0 : host_heuristic_radius(n, max_step, search_radius);
  CUDA_TRY(ctx, g->radius.ensure((size_t)rn * 8));
  CUDA_TRY(ctx, cudaMemcpyAsync(g->radius.p, r.data(), (size_t)rn * 8, cudaMemcpyHostToDevice, ctx->stream));
  CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
  g->radius_n = rn;
  return PORRT_OK;
}

PORRT_API int32_t porrt_pto_grow(porrt_ctx* ctx, const double start[2], const double low[2], const double up[2], uint64_t sampler_seed,
                                 const double* goals_xy, const uint64_t* goal_masks, int32_t n_goals, double goal_max_dist,
                                 double max_step, double search_radius, int64_t n_iter_min, int64_t n_iter_max,
                                 int64_t* out_sizes, int32_t* out_complete, int32_t* out_panic_code, int64_t* out_counters) {
  CTX_CHECK(ctx);
  if (!ctx->has_map) return porrt_fail(ctx, PORRT_ERR_NO_MAP, "no map uploaded");
  if (!start || !low || !up || (n_goals > 0 && (!goals_xy || !goal_masks)) || n_goals < 0 || n_iter_min < 0 || n_iter_max < 0 ||
      !out_sizes || !out_complete)
    return porrt_fail(ctx, PORRT_ERR_INVALID_ARG, "porrt_pto_grow: bad arguments");
  if (!ctx->pto) ctx->pto = new PtoGrow();
  PtoGrow* g = ctx->pto;
  g->have = false;
  for (int k = 0; k < 4; ++k) out_sizes[k] = 0;
  *out_complete = 0;
  if (out_panic_code) *out_panic_code = 0;
  if (out_counters) for (int k = 0; k < 4; ++k) out_counters[k] = 0;
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
  g->words = words;
  g->goal_masks_host.assign(goal_masks ? goal_masks : nullptr, goal_masks ? goal_masks + (size_t)n_goals * words : nullptr);
  // the loop runs at least n_iter_min and at most max(n_iter_min, n_iter_max) iterations
  const int64_t bound = std::min<int64_t>(std::max(n_iter_min, n_iter_max), INT32_MAX - 2 * PG_WMAX);
  // buffers: nodes grow with the roadmap, samples are drawn ahead of the windows
  g->node_cap = 0; g->radius_n = 0;
  int32_t rc = pg_grow_nodes(ctx, g, std::min<int64_t>(bound, 4096) + PG_BATCH * PG_WMAX + 1, 0);
  if (rc) return rc;
  rc = pg_radius_table(ctx, g, max_step, search_radius);
  if (rc) return rc;
  g->edge_cap = std::max<int64_t>(g->edge_cap, 16 * g->node_cap);
  CUDA_TRY(ctx, g->log_nbr.ensure((size_t)g->edge_cap * 4));
  CUDA_TRY(ctx, g->log_vid.ensure((size_t)g->edge_cap * 4));
  CUDA_TRY(ctx, g->fin_acc.ensure((size_t)words * 8));
  CUDA_TRY(ctx, g->goals.ensure((size_t)std::max(n_goals, 1) * 16));
  CUDA_TRY(ctx, g->goal_masks.ensure((size_t)std::max(n_goals, 1) * words * 8));
  CUDA_TRY(ctx, g->ctl.ensure(C_N * 4 + 64));
  if (n_goals > 0) {
    CUDA_TRY(ctx, cudaMemcpyAsync(g->goals.p, goals_xy, (size_t)n_goals * 16, cudaMemcpyHostToDevice, st));
    CUDA_TRY(ctx, cudaMemcpyAsync(g->goal_masks.p, goal_masks, (size_t)n_goals * words * 8, cudaMemcpyHostToDevice, st));
  }
  // pto.rs:141-149: one discrete draw per iteration, a continuous draw only when i % 100 != 0 (then goal_example(world))
  Pcg64 cont = Pcg64::seed_from_u64(sampler_seed), disc = Pcg64::seed_from_u64(sampler_seed);
  std::vector<double> smp;
  std::vector<int32_t> wld;
  int64_t drawn = 0;
  auto draw = [&](int64_t upto) -> int32_t {
    upto = std::min(upto, bound);
    if (upto <= drawn) return PORRT_OK;
    const int64_t n = upto - drawn;
    smp.resize((size_t)n * 2); wld.resize((size_t)n);
    for (int64_t k = 0; k < n; ++k) {
      const int64_t i = drawn + k + 1;
      const int32_t w = (int32_t)disc.below((uint64_t)n_worlds);
      wld[(size_t)k] = w;
      if (i % 100 == 0) { smp[2 * k] = world_goal[2 * (size_t)w]; smp[2 * k + 1] = world_goal[2 * (size_t)w + 1]; }
      else { smp[2 * k] = cont.range_f64(low[0], up[0]); smp[2 * k + 1] = cont.range_f64(low[1], up[1]); }
    }
    CUDA_TRY(ctx, g->samples.grow_keep((size_t)upto * 16, (size_t)drawn * 16, st));
    CUDA_TRY(ctx, g->worlds.grow_keep((size_t)upto * 4, (size_t)drawn * 4, st));
    CUDA_TRY(ctx, cudaMemcpyAsync(g->samples.as<double>() + 2 * drawn, smp.data(), (size_t)n * 16, cudaMemcpyHostToDevice, st));
    CUDA_TRY(ctx, cudaMemcpyAsync(g->worlds.as<int32_t>() + drawn, wld.data(), (size_t)n * 4, cudaMemcpyHostToDevice, st));
    CUDA_TRY(ctx, cudaStreamSynchronize(st));   // the host vectors are reused by the next draw
    drawn = upto;
    pto_set_kernel<<<1, 1, 0, st>>>(g->ctl.as<int32_t>(), C_DRAWN, (int32_t)drawn);
    LAUNCH_CHECK(ctx);
    return PORRT_OK;
  };
  auto set_caps = [&]() -> int32_t {
    pto_set_kernel<<<1, 1, 0, st>>>(g->ctl.as<int32_t>(), C_NODE_CAP, (int32_t)std::min<int64_t>(g->node_cap, INT32_MAX));
    LAUNCH_CHECK(ctx);
    pto_set_kernel<<<1, 1, 0, st>>>(g->ctl.as<int32_t>(), C_EDGE_CAP, (int32_t)std::min<int64_t>(g->edge_cap, INT32_MAX));
    LAUNCH_CHECK(ctx);
    return PORRT_OK;
  };
  PgDev d = pg_dev(ctx, g, max_step, goal_max_dist, n_goals, n_iter_min, n_iter_max);
  pto_init_kernel<<<1, 64, 0, st>>>(ctx->map, d, make_double2(start[0], start[1]));
  LAUNCH_CHECK(ctx);
  if ((rc = set_caps())) return rc;
  const bool runs = 0 < n_iter_min || 0 < n_iter_max;   // the loop condition before the first iteration (no finals yet)
  if (runs && (rc = draw(n_iter_min + 4096))) return rc;
  int32_t f[C_N];
  for (;;) {
    if ((rc = read_flags_dev(ctx, g->ctl.as<int32_t>(), C_N, f, st))) return rc;
    if (f[C_DONE] || !runs) break;
    const int64_t V = f[C_V], it = f[C_IT];
    if (it >= bound) break;
    // room for the next batch of windows: nodes (every commit adds at most one), edges (the commit stalls when they run out)
    if (V + PG_BATCH * PG_WMAX + 1 > g->node_cap) {
      if ((rc = pg_grow_nodes(ctx, g, V + PG_BATCH * PG_WMAX + 1, V))) return rc;
      if ((rc = pg_radius_table(ctx, g, max_step, search_radius))) return rc;
      if ((rc = set_caps())) return rc;
    }
    if (f[C_STALL] || (int64_t)f[C_E] + 64 * PG_BATCH * PG_WMAX > g->edge_cap) {
      const int64_t want = std::max<int64_t>(2 * g->edge_cap, (int64_t)f[C_E] + V + 1 + 64 * PG_BATCH * PG_WMAX);
      CUDA_TRY(ctx, g->log_nbr.grow_keep((size_t)want * 4, (size_t)f[C_E] * 4, st));
      CUDA_TRY(ctx, g->log_vid.grow_keep((size_t)want * 4, (size_t)f[C_E] * 4, st));
      g->edge_cap = want;
      if ((rc = set_caps())) return rc;
    }
    if (drawn < bound && drawn - it < 2 * PG_BATCH * PG_WMAX && (rc = draw(drawn + std::max<int64_t>(4096, drawn / 2)))) return rc;
    d = pg_dev(ctx, g, max_step, goal_max_dist, n_goals, n_iter_min, n_iter_max);
    const SpecDev s = spec_dev(g);
    for (int k = 0; k < PG_BATCH; ++k) {
      if (ctx->map.kind == PORRT_DOMAIN_SHELF) pto_speculate_kernel<PORRT_DOMAIN_SHELF><<<PG_WMAX, PG_SPEC_THREADS, 0, st>>>(ctx->map, d, s);
      else pto_speculate_kernel<PORRT_DOMAIN_DOOR><<<PG_WMAX, PG_SPEC_THREADS, 0, st>>>(ctx->map, d, s);
      LAUNCH_CHECK(ctx);
      pto_commit_kernel<<<1, PG_COMMIT_THREADS, 0, st>>>(d, s);
      LAUNCH_CHECK(ctx);
    }
  }
  const int64_t V = f[C_V], E = f[C_E];
  out_sizes[0] = f[C_IT];
  if (out_counters) { out_counters[0] = f[C_WINDOWS]; out_counters[1] = f[C_RESPEC]; out_counters[2] = f[C_CONF_NN]; out_counters[3] = f[C_CONF_RAD]; }
  if (f[C_DONE] == 2) {
    if (out_panic_code) *out_panic_code = f[C_PANIC];
    const bool at_start = f[C_WINDOWS] == 0;   // the init kernel found the start invalid: no window ever ran
    out_sizes[0] = at_start ? 0 : f[C_IT] + 1;  // the iteration whose check panicked
    return porrt_fail(ctx, PORRT_ERR_PANIC, at_start ? "Start from a valid state! (pto.rs:57, state validity code " + std::to_string(f[C_PANIC]) + ")"
                                                     : "porrt_pto_grow: a state / edge check hit a reference panic (code " + std::to_string(f[C_PANIC]) + ")");
  }
  // the children CSR from the edge log (graph.cu's late-list kernels, carrying the validity ids)
  CUDA_TRY(ctx, g->csr_row.ensure((size_t)(V + 1) * 8));
  CUDA_TRY(ctx, g->csr_col.ensure((size_t)std::max<int64_t>(2 * E, 1) * 4));
  CUDA_TRY(ctx, g->csr_vid.ensure((size_t)std::max<int64_t>(2 * E, 1) * 4));
  CUDA_TRY(ctx, g->work.ensure((size_t)V * 8 + (size_t)(V + 1) * 8 + (size_t)std::max<int64_t>(E, 1) * 4 + 64));
  int32_t* late_cnt = g->work.as<int32_t>();
  int32_t* cursor = late_cnt + V;
  int64_t* late_off = (int64_t*)(cursor + V);
  int32_t* late_vals = (int32_t*)(late_off + V + 1);
  pto_set_i64_kernel<<<1, 1, 0, st>>>(g->edge_off.as<int64_t>() + V, g->ctl.as<int32_t>(), C_E);
  LAUNCH_CHECK(ctx);
  rc = late_list_csr_dev(ctx, g->edge_off.as<int64_t>(), V, g->log_nbr.as<int32_t>(), g->ecnt.as<int32_t>(), g->log_vid.as<int32_t>(),
                         late_cnt, cursor, late_off, late_vals, g->csr_row.as<int64_t>(), g->csr_col.as<int32_t>(), g->csr_vid.as<int32_t>());
  if (rc) return rc;
  std::vector<uint64_t> fin((size_t)words);
  CUDA_TRY(ctx, cudaMemcpyAsync(fin.data(), g->fin_acc.p, (size_t)words * 8, cudaMemcpyDeviceToHost, st));
  CUDA_TRY(ctx, cudaStreamSynchronize(st));
  bool complete = f[C_NFIN] > 0;
  for (int w = 0; w < words; ++w) {
    const int rem = n_worlds - 64 * w;
    const uint64_t want = rem >= 64 ? ~0ull : ((1ull << rem) - 1ull);
    if ((fin[(size_t)w] & want) != want) complete = false;
  }
  g->have = true; g->V = V; g->E = 2 * E; g->n_finals = f[C_NFIN];
  out_sizes[1] = V; out_sizes[2] = 2 * E; out_sizes[3] = f[C_NFIN];
  *out_complete = complete ? 1 : 0;
  return PORRT_OK;
}

PORRT_API int32_t porrt_pto_fetch(porrt_ctx* ctx, double* out_xy, int32_t* out_node_vid, int64_t* out_row_ptr, int32_t* out_col,
                                  int32_t* out_edge_vid, uint64_t* out_reach, int64_t* out_final_ids, uint64_t* out_final_masks) {
  CTX_CHECK(ctx);
  PtoGrow* g = ctx->pto;
  if (!g || !g->have) return porrt_fail(ctx, PORRT_ERR_INVALID_ARG, "porrt_pto_fetch: no roadmap grown on this ctx");
  CUDA_TRY(ctx, cudaSetDevice(ctx->device));
  cudaStream_t st = ctx->stream;
  const int64_t V = g->V, E = g->E, F = g->n_finals;
  const size_t words = (size_t)g->words;
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
    if (out_final_masks) memcpy(out_final_masks + (size_t)k * words, g->goal_masks_host.data() + (size_t)goal[(size_t)k] * words, words * 8);
  }
  return PORRT_OK;
}
