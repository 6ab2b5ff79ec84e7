// sssp_frontier.cu -- value columns on roadmaps that do not fit the on-chip column solver (colsolve.cu): a label-correcting
// FRONTIER relaxation over the value table in global memory.  graph.cu's value-column driver runs it for world and belief columns.
//
// Reference: dijkstra over PTOGraphWorldView, one problem per world (pto_graph.rs:245-303, qmdp_policy_extractor.rs:23-35), and
// conditional_dijkstra's Action nodes, one problem per belief of a level (belief_graph.rs:89-182).
//
// At PRM scale (1e6 nodes, 5.3e7 directed edges, 64 worlds) a Bellman-Ford sweep touches E * W = 3.4e9 (edge, world) pairs and the
// roadmap's diameter is several hundred hops: the order-free Jacobi sweeps of round 1 were never run at that size.  Here only
// values that moved do work:
//   * nodes are renumbered along a Morton curve and dist[w][v] is world-major, so the parents of a node (its spatial neighbours)
//     sit in a few short runs of one world's row: the push step is bound by random 32-byte reads of this table;
//   * entries of nodes that are invalid in world w carry the sign bit (fixed, read through |.|, compare below every offer) -- the
//     same encoding as colsolve.cu;
//   * dirty[v] = worlds whose value at v improved since v last pushed; a round's worklist holds the nodes with a non-empty mask;
//   * one warp takes a worklist node v, clears its mask and, for every dirty world w, offers  norm2(u, v) + dist[v][w]  to every
//     parent u (transposed adjacency; norm2 is symmetric bit for bit) with a 64-bit atomicMin (non-negative doubles order like
//     their bit patterns); an improvement marks (u, w) dirty for the next round and appends u to the next worklist once.
// Rounds are launched back to back without host round trips (three rotating counters: read / append / reset); the host looks at
// the worklist length every few rounds only.  The fixed point is the reference's: every stored value is the left-to-right sum
// along an admissible path and the last improvement of every value is always pushed (SURVEY 8(g) note 5).
#include <algorithm>
#include <cmath>

#include "common.cuh"
#include "sssp_frontier.cuh"

namespace {

// ---- Morton numbering: pos = rank of the node's interleaved 16 + 16 bit cell coordinates
__device__ __forceinline__ unsigned long long sf_ord(double x) {   // order-preserving bits
  const unsigned long long b = (unsigned long long)__double_as_longlong(x);
  return (b & 0x8000000000000000ull) ? ~b : (b | 0x8000000000000000ull);
}
__device__ __forceinline__ double sf_unord(unsigned long long e) {
  return __longlong_as_double((long long)((e & 0x8000000000000000ull) ? (e & 0x7fffffffffffffffull) : ~e));
}
__global__ void sf_bbox_kernel(const double2* __restrict__ xy, int64_t V, unsigned long long* __restrict__ box /* min x, min y, max x, max y */) {
  unsigned long long lo_x = ~0ull, lo_y = ~0ull, hi_x = 0, hi_y = 0;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < V; i += (int64_t)gridDim.x * blockDim.x) {
    const double2 p = xy[i];
    const unsigned long long ex = sf_ord(p.x), ey = sf_ord(p.y);
    lo_x = min(lo_x, ex); hi_x = max(hi_x, ex); lo_y = min(lo_y, ey); hi_y = max(hi_y, ey);
  }
  for (int o = 16; o > 0; o >>= 1) {
    lo_x = min(lo_x, __shfl_xor_sync(0xffffffffu, lo_x, o)); lo_y = min(lo_y, __shfl_xor_sync(0xffffffffu, lo_y, o));
    hi_x = max(hi_x, __shfl_xor_sync(0xffffffffu, hi_x, o)); hi_y = max(hi_y, __shfl_xor_sync(0xffffffffu, hi_y, o));
  }
  if ((threadIdx.x & 31) == 0) { atomicMin(&box[0], lo_x); atomicMin(&box[1], lo_y); atomicMax(&box[2], hi_x); atomicMax(&box[3], hi_y); }
}
__device__ __forceinline__ unsigned sf_spread16(unsigned v) {
  v &= 0xffffu; v = (v | (v << 8)) & 0x00ff00ffu; v = (v | (v << 4)) & 0x0f0f0f0fu; v = (v | (v << 2)) & 0x33333333u; v = (v | (v << 1)) & 0x55555555u;
  return v;
}
__global__ void sf_morton_kernel(const double2* __restrict__ xy, int64_t V, const unsigned long long* __restrict__ box,
                                 uint64_t* __restrict__ keys, uint32_t* __restrict__ vals) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= V) return;
  const double x0 = sf_unord(box[0]), y0 = sf_unord(box[1]), x1 = sf_unord(box[2]), y1 = sf_unord(box[3]);
  const double2 p = xy[i];
  const double fx = x1 > x0 ? (p.x - x0) / (x1 - x0) : 0.0, fy = y1 > y0 ? (p.y - y0) / (y1 - y0) : 0.0;   // (a schedule parameter only)
  const unsigned cx = (unsigned)fmin(fmax(fx * 65535.0, 0.0), 65535.0), cy = (unsigned)fmin(fmax(fy * 65535.0, 0.0), 65535.0);
  keys[i] = (uint64_t)(sf_spread16(cx) | (sf_spread16(cy) << 1));
  vals[i] = (uint32_t)i;
}
__global__ void sf_perm_kernel(const uint32_t* __restrict__ order, int64_t V, int32_t* __restrict__ perm) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < V) perm[order[i]] = (int32_t)i;
}

__global__ void sf_count_kernel(const int32_t* __restrict__ col, const int32_t* __restrict__ perm, int64_t E, int32_t* __restrict__ cnt) {
  const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (e < E) atomicAdd(&cnt[perm[col[e]]], 1);
}
// transposed records in the new numbering: row perm[v] lists (perm[u], norm2(u, v)); one warp per row u of the forward CSR
__global__ void sf_fill_kernel(const int64_t* __restrict__ row_ptr, const int32_t* __restrict__ col, const int32_t* __restrict__ evid,
                               const double2* __restrict__ xy, const int32_t* __restrict__ perm, int64_t V, const int64_t* __restrict__ row_t,
                               int32_t* __restrict__ cursor, int32_t* __restrict__ col_t, double* __restrict__ cost_t,
                               uint16_t* __restrict__ evid_t) {
  const int lane = threadIdx.x & 31;
  const int64_t u = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  if (u >= V) return;
  const double2 a = xy[u];
  const int32_t pu = perm[u];
  for (int64_t e = row_ptr[u] + lane; e < row_ptr[u + 1]; e += 32) {
    const int32_t v = col[e];
    const double2 c = xy[v];
    const double dx = __dsub_rn(c.x, a.x), dy = __dsub_rn(c.y, a.y);
    const int32_t pv = perm[v];
    const int64_t pos = row_t[pv] + atomicAdd(&cursor[pv], 1);
    col_t[pos] = pu;
    if (evid) evid_t[pos] = (uint16_t)evid[e];
    cost_t[pos] = __dsqrt_rn(__dadd_rn(__dmul_rn(dx, dx), __dmul_rn(dy, dy)));   // norm2(u, v), common.rs:203-213
  }
}

struct SfArgs {
  const int64_t* row_t; const int32_t* col_t; const double* cost_t;
  const uint16_t* evid_t;         // validity id of the transposed record's edge (nullable)
  const uint64_t* cmask;          // [W][4] admissible validity ids per column (nullable: every edge admissible)
  double* dist; int64_t V; int32_t W, words;   // dist[w * V + v], v in Morton numbering
  unsigned long long* dirty[2];   // [V * words] each
  int32_t* inq[2];                // [V] each: node already on that round's worklist
  int32_t* list[2];               // [V] each
  int32_t* counter;               // [3] rotating: read / append / reset
  unsigned long long* offers;     // (parent, world) pairs looked at
  // near / far ordering: a dirty value pushes only once it is <= the round's threshold, which advances by `delta` per round (or
  // jumps to the smallest deferred value); without it a value is corrected ~19 times at PRM scale (long early edges let the
  // fronts run far ahead with values that are much too large), with it a handful of times
  double* thr;                    // [3] rotating thresholds
  unsigned long long* min_far;    // [3] rotating: smallest deferred value of a round (bits)
  double delta;
  int2* pairs;                    // the round's push list: (node, world) pairs within the threshold
  int32_t* pair_count;            // [2]
  int32_t pair_cap;
};

// Round r, step 1 (one THREAD per worklist node): take the node's dirty mask; a dirty value within the round's threshold becomes a
// (node, world) pair of the push list, the others stay dirty and come back next round.  Deferred values are looked at once per round
// until their turn comes -- by one thread, not by a warp (at PRM scale the long edges of the early samples keep ~10x more values
// waiting than moving).
__global__ void __launch_bounds__(256) sf_classify_kernel(SfArgs a, int round) {
  const int cur = round & 1, nxt = cur ^ 1;
  const int n_cur = a.counter[round % 3];
  const double far_prev = __longlong_as_double((long long)a.min_far[round % 3]);
  const double thr = fmax(__dadd_rn(a.thr[round % 3], a.delta), far_prev < INFINITY ? far_prev : 0.0);
  if (blockIdx.x == 0 && threadIdx.x == 0) {
    a.counter[(round + 2) % 3] = 0;
    a.min_far[(round + 2) % 3] = 0x7ff0000000000000ull;   // +inf
    a.thr[(round + 1) % 3] = thr;
  }
  unsigned long long my_far = 0x7ff0000000000000ull;
  const int lane = threadIdx.x & 31;
  const int stride = gridDim.x * blockDim.x;
  // (the loop runs the same number of times for every lane of a warp: the appends below are aggregated per warp -- one atomicAdd on
  // the list counters per warp instead of one per entry; 8e7 same-address atomics were a third of the run time at PRM scale)
  for (int q0 = (blockIdx.x * blockDim.x + threadIdx.x) - lane; q0 < n_cur; q0 += stride) {
    const int qi = q0 + lane;
    const bool live = qi < n_cur;
    const int32_t v = live ? a.list[cur][qi] : 0;
    if (live) a.inq[cur][v] = 0;
    bool again = false;
    for (int k = 0; k < a.words; ++k) {
      unsigned long long m = live ? atomicExch(&a.dirty[cur][(int64_t)v * a.words + k], 0ull) : 0ull;
      __threadfence();   // the values are read after the mask was taken: a later improvement marks v again
      unsigned long long near = 0, keep = 0;
      for (unsigned long long mm = m; mm; mm &= mm - 1) {
        const int b = __ffsll((long long)mm) - 1;
        const double dv = fabs(*(volatile double*)(a.dist + (int64_t)(k * 64 + b) * a.V + v));
        if (dv <= thr) near |= 1ull << b;
        else {
          keep |= 1ull << b;
          const unsigned long long bits = (unsigned long long)__double_as_longlong(dv);
          if (bits < my_far) my_far = bits;
        }
      }
      // this warp's near pairs go to one reserved stretch of the push list
      const int cnt = __popcll(near);
      int incl = cnt;
      for (int o = 1; o < 32; o <<= 1) { const int t = __shfl_up_sync(0xffffffffu, incl, o); if (lane >= o) incl += t; }
      const int total = __shfl_sync(0xffffffffu, incl, 31);
      if (total) {
        int base = 0;
        if (lane == 31) base = atomicAdd(&a.pair_count[round & 1], total);
        base = __shfl_sync(0xffffffffu, base, 31) + incl - cnt;
        for (unsigned long long mm = near; mm; mm &= mm - 1) {
          const int b = __ffsll((long long)mm) - 1;
          if (base < a.pair_cap) a.pairs[base] = make_int2(v, k * 64 + b);
          else keep |= 1ull << b;   // push list full: wait a round
          ++base;
        }
      }
      if (keep) { atomicOr(&a.dirty[nxt][(int64_t)v * a.words + k], keep); again = true; }
    }
    const bool first = again && atomicExch(&a.inq[nxt][v], 1) == 0;
    const unsigned fm = __ballot_sync(0xffffffffu, first);
    if (fm) {
      int base = 0;
      if (lane == 0) base = atomicAdd(&a.counter[(round + 1) % 3], __popc(fm));
      base = __shfl_sync(0xffffffffu, base, 0);
      if (first) a.list[nxt][base + __popc(fm & ((1u << lane) - 1u))] = v;
    }
  }
  for (int s2 = 16; s2 > 0; s2 >>= 1) { const unsigned long long o = __shfl_xor_sync(0xffffffffu, my_far, s2); if (o < my_far) my_far = o; }
  if ((threadIdx.x & 31) == 0 && my_far < *(volatile unsigned long long*)&a.min_far[(round + 1) % 3]) atomicMin(&a.min_far[(round + 1) % 3], my_far);
}

// Round r, step 2 (one WARP per (node, world) pair of the push list): offer  norm2(u, v) + dist[v][w]  to every parent u.
// (8 lanes per pair, four pairs per warp in flight, was slower: 172 against 150 ms at PRM scale -- the record loads lose their coalescing.)
__global__ void __launch_bounds__(256) sf_push_kernel(SfArgs a, int round) {
  const int nxt = (round & 1) ^ 1;
  const int n_pairs = min(a.pair_count[round & 1], a.pair_cap);
  if (blockIdx.x == 0 && threadIdx.x == 0) a.pair_count[nxt] = 0;   // the next round's classify step appends there
  const int lane = threadIdx.x & 31;
  const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, n_warps = (gridDim.x * blockDim.x) >> 5;
  unsigned long long n_off = 0;
  for (int qi = warp; qi < n_pairs; qi += n_warps) {
    const int2 vw = a.pairs[qi];
    const int32_t v = vw.x;
    const int w = vw.y, k = w >> 6;
    const double dv = fabs(*(volatile double*)(a.dist + (int64_t)w * a.V + v));
    const int64_t e1 = a.row_t[v + 1];
    for (int64_t e0 = a.row_t[v]; e0 < e1; e0 += 32) {
      const int64_t e = e0 + lane;
      bool first = false;
      int32_t u = 0;
      if (e < e1) {
        u = __ldg(a.col_t + e);
        const double alt = __dadd_rn(__ldg(a.cost_t + e), dv);   // norm2(u, v) + dist[v], pto_graph.rs:293 / belief_graph.rs:121-124
        double* du = a.dist + (int64_t)w * a.V + u;
        ++n_off;
        bool admissible = true;
        if (a.cmask) { const unsigned ev = a.evid_t[e]; admissible = (a.cmask[(int64_t)w * 4 + (ev >> 6)] >> (ev & 63)) & 1; }
        if (admissible && alt < *du) {
          const unsigned long long bits = (unsigned long long)__double_as_longlong(alt);
          const unsigned long long old = atomicMin(reinterpret_cast<unsigned long long*>(du), bits);
          if (bits < old) {
            const unsigned long long was = atomicOr(&a.dirty[nxt][(int64_t)u * a.words + k], 1ull << (w & 63));
            // only the one who turned a clean word dirty can be the first to queue the node
            first = was == 0 && atomicExch(&a.inq[nxt][u], 1) == 0;
          }
        }
      }
      const unsigned fm = __ballot_sync(0xffffffffu, first);
      if (fm) {   // one atomicAdd on the list counter per warp
        int base = 0;
        if (lane == 0) base = atomicAdd(&a.counter[(round + 1) % 3], __popc(fm));
        base = __shfl_sync(0xffffffffu, base, 0);
        if (first) a.list[nxt][base + __popc(fm & ((1u << lane) - 1u))] = u;
      }
    }
  }
  if (a.offers) {
    for (int s = 16; s > 0; s >>= 1) n_off += __shfl_xor_sync(0xffffffffu, n_off, s);
    if (lane == 0 && n_off) atomicAdd(a.offers, n_off);
  }
}

__global__ void sf_sum_kernel(const double* __restrict__ x, int64_t n, double* __restrict__ out) {
  double s = 0.0;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) s += x[i];
  for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
  if ((threadIdx.x & 31) == 0) atomicAdd(out, s);   // only the order of magnitude matters (a schedule parameter, not a result)
}

// ---- seeding: every entry that holds a finite value (finals, Observation values) is a source
__global__ void sf_seed_all_kernel(SfArgs a) {
  const int64_t v = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const int lane = threadIdx.x & 31;
  bool any = false;
  if (v < a.V) {
    for (int k = 0; k < a.words; ++k) {
      unsigned long long m = 0;
      for (int b = 0; b < 64 && k * 64 + b < a.W; ++b)
        if (fabs(a.dist[(int64_t)(k * 64 + b) * a.V + v]) < INFINITY) m |= 1ull << b;
      if (m) { a.dirty[0][v * a.words + k] = m; any = true; }
    }
    if (any) a.inq[0][v] = 1;
  }
  const unsigned fm = __ballot_sync(0xffffffffu, any);
  if (fm) {
    int base = 0;
    if (lane == 0) base = atomicAdd(&a.counter[0], __popc(fm));
    base = __shfl_sync(0xffffffffu, base, 0);
    if (any) a.list[0][base + __popc(fm & ((1u << lane) - 1u))] = (int32_t)v;
  }
}
}  // namespace

// Morton numbering (work space: sort_keys) + transposed adjacency (sort_vals) of a roadmap on the device.
int32_t sf_build_graph(porrt_ctx* ctx, const int64_t* d_row, const int32_t* d_col, const int32_t* d_evid, const double* d_xy, int64_t V,
                       int64_t E, SfGraph* out, cudaStream_t st) {
  if (V > 0x7fffffff) return porrt_fail(ctx, PORRT_ERR_UNSUPPORTED, "value backups: more than 2^31 nodes");
  uint64_t* d_keys;
  uint32_t* d_order;
  int32_t* d_perm;
  unsigned long long* d_box;
  CUDA_TRY(ctx, carve(ctx->sort_keys, [&](Carve& c) {
    d_keys = c.take<uint64_t>(V); d_order = c.take<uint32_t>(V); d_perm = c.take<int32_t>(V); d_box = c.take<unsigned long long>(4);
  }));
  const unsigned long long init[4] = {~0ull, ~0ull, 0ull, 0ull};
  CUDA_TRY(ctx, cudaMemcpyAsync(d_box, init, 32, cudaMemcpyHostToDevice, st));
  sf_bbox_kernel<<<ctx->sm_count * 4, 256, 0, st>>>((const double2*)d_xy, V, d_box);
  LAUNCH_CHECK(ctx);
  sf_morton_kernel<<<div_up(V, 256), 256, 0, st>>>((const double2*)d_xy, V, d_box, d_keys, d_order);
  LAUNCH_CHECK(ctx);
  int32_t rc = radix_sort_pairs(ctx, d_keys, d_order, V, 32);   // (runs on ctx->stream == st)
  if (rc) return rc;
  sf_perm_kernel<<<div_up(V, 256), 256, 0, st>>>(d_order, V, d_perm);
  LAUNCH_CHECK(ctx);
  int64_t* d_row_t;
  double *d_cost_t, *d_sum;
  int32_t *d_col_t, *d_cnt;
  uint16_t* d_evid_t;
  CUDA_TRY(ctx, carve(ctx->sort_vals, [&](Carve& c) {
    d_row_t = c.take<int64_t>(V + 1); d_cost_t = c.take<double>(E); d_col_t = c.take<int32_t>(E + 1); d_evid_t = c.take<uint16_t>(E + 2);
    d_cnt = c.take<int32_t>(V); d_sum = c.take<double>(2);
  }));
  CUDA_TRY(ctx, cudaMemsetAsync(d_cnt, 0, (size_t)V * 4, st));
  if (E > 0) {
    sf_count_kernel<<<div_up(E, 256), 256, 0, st>>>(d_col, d_perm, E, d_cnt);
    LAUNCH_CHECK(ctx);
  }
  rc = scan_exclusive_i64(ctx, d_cnt, V, d_row_t);
  if (rc) return rc;
  CUDA_TRY(ctx, cudaMemsetAsync(d_cnt, 0, (size_t)V * 4, st));
  CUDA_TRY(ctx, cudaMemsetAsync(d_sum, 0, 8, st));
  if (E > 0) {
    sf_fill_kernel<<<div_up(V * 32, 256), 256, 0, st>>>(d_row, d_col, d_evid, (const double2*)d_xy, d_perm, V, d_row_t, d_cnt, d_col_t, d_cost_t, d_evid_t);
    LAUNCH_CHECK(ctx);
    sf_sum_kernel<<<ctx->sm_count * 4, 256, 0, st>>>(d_cost_t, E, d_sum);
    LAUNCH_CHECK(ctx);
  }
  double sum = 0.0;
  CUDA_TRY(ctx, cudaMemcpyAsync(&sum, d_sum, 8, cudaMemcpyDeviceToHost, st));
  CUDA_TRY(ctx, cudaStreamSynchronize(st));
  out->V = V; out->E = E; out->row_t = d_row_t; out->col_t = d_col_t; out->cost_t = d_cost_t; out->evid_t = d_evid ? d_evid_t : nullptr;
  out->order = d_order; out->perm = d_perm;
  // delta of the near / far ordering = the mean edge length of the roadmap (one hop of a front).  Measured at PRM scale (1e6 nodes, 64
  // worlds): delta = 0.5 / 0.75 / 1 / 1.5 / 2 / 4 mean edge lengths -> 1.05 / 1.12 / 1.27 / 2.6 / 5.5 / 13.9 full sweeps' worth of pairs in
  // 592 / 400 / 304 / 240 / 224 / 240 rounds; no ordering at all: 19.1
  out->delta = E > 0 && sum > 0.0 && std::isfinite(sum) ? sum / (double)E : 1.0;
  return PORRT_OK;
}

// The frontier state of sf_relax over V nodes and W columns, at the front of ws_state.  Its size grows with W, so state for fewer
// columns fits in the space reserved for more.
static void sf_state_layout(Carve& c, SfArgs& a, int64_t V, int32_t W) {
  const int words = (W + 63) / 64;
  a.pair_cap = (int32_t)std::min<int64_t>(V * (int64_t)W, std::max<int64_t>(4 << 20, 4 * V));
  a.dirty[0] = c.take<unsigned long long>((size_t)V * words); a.dirty[1] = c.take<unsigned long long>((size_t)V * words);
  a.inq[0] = c.take<int32_t>(V); a.inq[1] = c.take<int32_t>(V);
  a.list[0] = c.take<int32_t>(V); a.list[1] = c.take<int32_t>(V);
  a.counter = c.take<int32_t>(4);
  a.offers = c.take<unsigned long long>(2);
  a.thr = c.take<double>(4);
  a.min_far = c.take<unsigned long long>(4);
  a.pair_count = c.take<int32_t>(4);
  a.pairs = c.take<int2>(a.pair_cap);
}
void sf_state_reserve(Carve& c, int64_t V, int32_t W) {
  SfArgs unused = {};
  sf_state_layout(c, unused, V, W);
}

// Relaxes W value columns to their fixed point.  dist[w * V + pos] (Morton numbering) holds the initial values on entry -- +inf, the
// sources' values, the sign bit on every entry that must not be relaxed -- and the result on exit (signs kept).  cmask (nullable):
// [W][4] validity ids an edge must carry to be admissible in column w (needs g.evid_t).  Work space: ws_state, within
// sf_state_reserve(V, W).
int32_t sf_relax(porrt_ctx* ctx, const SfGraph& g, double* dist, int32_t W, const uint64_t* cmask, int32_t* out_rounds, double* out_offers,
                 cudaStream_t st) {
  const int64_t V = g.V;
  const int words = (W + 63) / 64;
  if (W <= 0) { if (out_rounds) *out_rounds = 0; if (out_offers) *out_offers = 0.0; return PORRT_OK; }
  SfArgs a = {};
  CUDA_TRY(ctx, carve(ctx->ws_state, [&](Carve& c) { sf_state_layout(c, a, V, W); }));
  a.row_t = g.row_t; a.col_t = g.col_t; a.cost_t = g.cost_t; a.evid_t = g.evid_t; a.cmask = cmask; a.V = V; a.W = W; a.words = words;
  a.dist = dist; a.delta = g.delta;
  CUDA_TRY(ctx, cudaMemsetAsync(a.dirty[0], 0, 2 * (((size_t)V * words * 8 + 15) & ~(size_t)15), st));
  CUDA_TRY(ctx, cudaMemsetAsync(a.inq[0], 0, 2 * (((size_t)V * 4 + 15) & ~(size_t)15), st));
  CUDA_TRY(ctx, cudaMemsetAsync(a.counter, 0, 32 + 32, st));   // counters, offers, thresholds (0.0)
  CUDA_TRY(ctx, cudaMemsetAsync(a.pair_count, 0, 16, st));
  const unsigned long long inf3[4] = {0x7ff0000000000000ull, 0x7ff0000000000000ull, 0x7ff0000000000000ull, 0};
  CUDA_TRY(ctx, cudaMemcpyAsync(a.min_far, inf3, 32, cudaMemcpyHostToDevice, st));
  sf_seed_all_kernel<<<div_up(V, 256), 256, 0, st>>>(a);
  LAUNCH_CHECK(ctx);
  // ---- rounds: a fixed grid strides over the worklist, whose length lives on the device; the host checks every CHECK rounds
  const int grid = ctx->sm_count * 8;
  const int CHECK = 16;
  int round = 0;
  int32_t counters[4] = {0, 0, 0, 0};
  for (;;) {
    for (int k = 0; k < CHECK; ++k, ++round) {
      sf_classify_kernel<<<grid, 256, 0, st>>>(a, round);
      LAUNCH_CHECK(ctx);
      sf_push_kernel<<<grid, 256, 0, st>>>(a, round);
      LAUNCH_CHECK(ctx);
    }
    CUDA_TRY(ctx, cudaMemcpyAsync(counters, a.counter, 12, cudaMemcpyDeviceToHost, st));
    CUDA_TRY(ctx, cudaStreamSynchronize(st));
    if (counters[round % 3] == 0) break;   // the worklist of the next round is empty: nothing is dirty any more
    if (round > 64 * V + 1024) return porrt_fail(ctx, PORRT_ERR_CUDA, "value backups: no convergence");
  }
  if (out_rounds) *out_rounds = round;
  if (out_offers) {
    unsigned long long off = 0;
    CUDA_TRY(ctx, cudaMemcpyAsync(&off, a.offers, 8, cudaMemcpyDeviceToHost, st));
    CUDA_TRY(ctx, cudaStreamSynchronize(st));
    *out_offers = (double)off;
  }
  return PORRT_OK;
}
