// graph.cu -- roadmap construction and value backups (SURVEY.md 8(a) rows B4, C1-C4, D1).
//
//  * porrt_prm_build      : PRM::grow_graph / add_sample (reference src/prm.rs:38-109) as two device batches
//                           (prefix-restricted radius queries, then edge checks) + CSR assembly in insertion order.
//  * porrt_sssp_worlds    : dijkstra over PTOGraphWorldView per world (src/pto_graph.rs:245-303,
//                           src/qmdp_policy_extractor.rs:23-35) as monotone pull relaxations to the fixed point.
//  * porrt_belief_vi      : PTO::build_belief_graph + conditional_dijkstra (src/pto.rs:185-275,
//                           src/belief_graph.rs:89-182) on the IMPLICIT belief graph (node*B + belief), never materialised.
//  * porrt_extract_policy : extract_policy / get_best_expected_children (src/belief_graph.rs:184-267), host walk.
//
// Bit-exactness: dist values are the greatest fixed point of a monotone min-plus operator evaluated with the reference's
// operand order (SURVEY 8(g) note 5), so any relaxation schedule that runs to quiescence yields identical f64 bit patterns.
#include <algorithm>
#include <chrono>
#include <cmath>
#include <map>
#include <thread>
#include <unordered_map>

#include "common.cuh"
#include "colsolve.cuh"
#include "belief_tables.cuh"
#include "sssp_frontier.cuh"

static double now_ms() {
  return std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now().time_since_epoch()).count();
}

// ================================================================================================ kd pre-order rank
// The reference returns radius-search hits in node-left-right order of its incremental, unbalanced kd-tree
// (nearest_neighbor.rs:29-46 add, :101-117 visit order).  Inserting a leaf never reorders existing nodes, so the
// pre-order rank in the FINAL tree orders every prefix correctly (SURVEY 8(g) note 4).
// Device construction, level-synchronous: every not-yet-placed point sits at the node it would currently be compared
// with; all of them descend one level per round (so the split axis is the round parity), and the child slot (node, side)
// goes to the smallest id that wants it (atomicMin) -- exactly the point that sequential insertion would have put there.
// Subtree sizes are counted on the way down; ranks follow top-down, one depth per launch.
// axis < 0: the split axis is the parity of the depth of the node the point is compared with (points sit at different depths after
// the two-phase start below); axis >= 0: all points are at the same depth, the round's parity
template <bool AGGREGATE>
__global__ void kd_descend_kernel(const double2* __restrict__ xy, int64_t n, int axis, const int32_t* __restrict__ cur,
                                  int32_t* __restrict__ child, int32_t* __restrict__ size, uint8_t* __restrict__ side,
                                  const int32_t* __restrict__ node_depth = nullptr) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const int32_t c = i < n ? cur[i] : -1;
  int s = 0;
  if (c >= 0) {
    const double2 p = xy[i], q = xy[c];
    const int ax = axis >= 0 ? axis : (node_depth[c] & 1);
    s = (ax ? p.y < q.y : p.x < q.x) ? 0 : 1;   // strictly-less goes left (nearest_neighbor.rs:32)
    side[i] = (uint8_t)s;
  }
  if (AGGREGATE) {
    // near the root a million points compete for a handful of child slots: one atomic per (slot, warp) instead of per point
    const int64_t slot = c >= 0 ? 2 * (int64_t)c + s : -1 - (int64_t)(threadIdx.x & 31);
    const unsigned peers = __match_any_sync(0xffffffffu, slot);
    if (c >= 0) {
      const int leader = __ffs(peers) - 1;          // lanes are in id order: the lowest lane holds the smallest id
      if ((int)(threadIdx.x & 31) == leader) {
        atomicMin(&child[slot], (int32_t)i);
        atomicAdd(&size[c], __popc(peers));
      }
    }
  } else if (c >= 0) {
    atomicMin(&child[2 * (int64_t)c + s], (int32_t)i);
    atomicAdd(&size[c], 1);
  }
}
__global__ void kd_place_kernel(int64_t n, int32_t* __restrict__ cur, const int32_t* __restrict__ child,
                                const uint8_t* __restrict__ side, int32_t* __restrict__ parent, int32_t* __restrict__ node_depth,
                                int32_t* __restrict__ remaining, int32_t* __restrict__ max_depth) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  int32_t placed_at = 0;
  if (i < n) {
    const int32_t c = cur[i];
    if (c >= 0) {
      const int32_t w = child[2 * (int64_t)c + side[i]];
      if (w == (int32_t)i) { parent[i] = c; placed_at = node_depth[c] + 1; node_depth[i] = placed_at; cur[i] = -1; }
      else { cur[i] = w; if (remaining) atomicAdd(remaining, 1); }
    }
  }
  placed_at = __reduce_max_sync(0xffffffffu, placed_at);
  if (placed_at > 0 && (threadIdx.x & 31) == 0) atomicMax(max_depth, placed_at);
}
// Two-phase start (single trees of many points): the tree of the first M points does not depend on the later ones, so it is built
// first (the same rounds, on M points); then every later point walks down that finished top tree on its own -- read-only, no
// atomics, no barrier per level -- to the node where it would next compete for an empty child slot.  The rounds that follow work
// on ~n / M points per slot instead of n points on a handful of slots (those first 14 rounds were 1.6 of the rank's 3 ms at 1e6).
__global__ void kd_walk_kernel(const double2* __restrict__ xy, int64_t first, int64_t n, const int32_t* __restrict__ child,
                               const int32_t* __restrict__ node_depth, int32_t* __restrict__ cur, int32_t* __restrict__ exits) {
  const int64_t i = first + (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const double2 p = xy[i];
  int32_t c = 0;
  for (;;) {
    const double2 q = xy[c];
    const int s = ((node_depth[c] & 1) ? p.y < q.y : p.x < q.x) ? 0 : 1;
    const int32_t w = child[2 * (int64_t)c + s];
    if (w == 0x7fffffff) break;
    c = w;
  }
  cur[i] = c;
  atomicAdd(&exits[c], 1);
}
// subtree sizes of the top tree: the later points that pass THROUGH a top node (they leave the top tree below one of its
// children) were never counted by a round at that node; one pass per depth, deepest first.  up[c] = later points below c.
__global__ void kd_top_sizes_kernel(int64_t m, int depth, const int32_t* __restrict__ node_depth, const int32_t* __restrict__ child,
                                    const int32_t* __restrict__ exits, int32_t* __restrict__ up, int32_t* __restrict__ size) {
  const int64_t c = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= m || node_depth[c] != depth) return;
  int32_t through = 0;
  for (int s = 0; s < 2; ++s) {
    const int32_t ch = child[2 * c + s];
    if (ch != 0x7fffffff) through += up[ch];
  }
  up[c] = exits[c] + through;
  size[c] += through;
}
__global__ void kd_rank_kernel(int64_t n, int depth, const int32_t* __restrict__ node_depth, const int32_t* __restrict__ parent,
                               const uint8_t* __restrict__ side, const int32_t* __restrict__ child, const int32_t* __restrict__ size,
                               int32_t* __restrict__ rank) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n || node_depth[i] != depth) return;
  const int32_t p = parent[i];
  int32_t r = rank[p] + 1;
  if (side[i]) {                                    // right child: the whole left subtree of the parent comes first
    const int32_t l = child[2 * (int64_t)p];
    if (l != 0x7fffffff) r += size[l] + 1;
  }
  rank[i] = r;
}
// Pre-order ranks by pointer jumping: rank[i] = rank[root] + sum over the path i -> root of off[a], off[a] = 1 (+ the size of the left
// sibling's subtree + 1 for a right child).  ceil(log2(depth + 1)) rounds over all nodes instead of one launch per tree depth
// (47 launches of 8.7 us at 1e6 points).  Ping-pong buffers: a round reads the previous round's (jump, acc) only.
__global__ void kd_rank_init_kernel(int64_t n, const int32_t* __restrict__ parent, const uint8_t* __restrict__ side,
                                    const int32_t* __restrict__ child, const int32_t* __restrict__ size, const int32_t* __restrict__ node_depth,
                                    const int32_t* __restrict__ rank0, int32_t* __restrict__ jump, int32_t* __restrict__ acc) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  if (node_depth[i] == 0) { jump[i] = -1; acc[i] = rank0[i]; return; }   // a root: its rank is where its tree's ranks start
  const int32_t p = parent[i];
  int32_t off = 1;
  if (side[i]) {                                    // right child: the whole left subtree of the parent comes first
    const int32_t l = child[2 * (int64_t)p];
    if (l != 0x7fffffff) off += size[l] + 1;
  }
  jump[i] = p; acc[i] = off;
}
__global__ void kd_rank_jump_kernel(int64_t n, const int32_t* __restrict__ jump_in, const int32_t* __restrict__ acc_in,
                                    int32_t* __restrict__ jump_out, int32_t* __restrict__ acc_out) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const int32_t j = jump_in[i];
  int32_t a = acc_in[i], nj = -1;
  if (j >= 0) { a += acc_in[j]; nj = jump_in[j]; }
  jump_out[i] = nj; acc_out[i] = a;
}
// root_of (nullable): several independent trees in one id space (the modes of a multi-modal PRM): point i belongs to the tree
// rooted at root_of[i] (= the first id of its group); ranks then start at the root's id, so that the ranks of all trees
// together are still a permutation of 0..n-1 (tree g occupies the id range of group g)
__global__ void kd_init_kernel(int64_t n, int32_t* __restrict__ cur, int32_t* __restrict__ child, int32_t* __restrict__ size,
                               int32_t* __restrict__ node_depth, int32_t* __restrict__ rank, const uint32_t* __restrict__ root_of) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const int64_t root = root_of ? (int64_t)root_of[i] : 0;
  cur[i] = i == root ? -1 : (int32_t)root;
  child[2 * i] = 0x7fffffff; child[2 * i + 1] = 0x7fffffff;
  size[i] = 0; node_depth[i] = i == root ? 0 : -1; rank[i] = i == root ? (int32_t)root : 0;
}

// xy_dev: n vertices (device); out_rank_dev[n]; work space ctx->kd_buf
int32_t kd_preorder_rank_dev(porrt_ctx* ctx, const double* xy_dev, int64_t n, int32_t* out_rank_dev, const uint32_t* root_of_dev,
                             cudaStream_t st_in, std::string* err, int64_t* n_launch) {
  cudaStream_t st = st_in ? st_in : ctx->stream;
  int64_t launches = 0;
  auto fail = [&](const char* what, cudaError_t e) {
    const std::string msg = std::string("kd_preorder_rank: ") + what + " -> " + cudaGetErrorString(e);
    if (err) *err = msg; else ctx->err = msg;
    return PORRT_ERR_CUDA;
  };
#define KD_TRY(expr) do { cudaError_t _e = (expr); if (_e != cudaSuccess) return fail(#expr, _e); } while (0)
#define KD_LAUNCHED() do { ++launches; KD_TRY(cudaGetLastError()); } while (0)
  if (n <= 0) return PORRT_OK;
  int32_t *cur, *child, *size, *parent, *node_depth, *exits, *up, *remaining;
  uint8_t* side;
  KD_TRY(carve(ctx->kd_buf, [&](Carve& c) {
    cur = c.take<int32_t>(n); child = c.take<int32_t>(2 * n); size = c.take<int32_t>(n); parent = c.take<int32_t>(n);
    node_depth = c.take<int32_t>(n);
    exits = c.take<int32_t>(n);     // two-phase start only
    up = c.take<int32_t>(n);
    remaining = c.take<int32_t>(2);
    side = c.take<uint8_t>(n);
  }));
  int32_t* max_depth = remaining + 1;
  const int blocks = div_up(n, 256);
  kd_init_kernel<<<blocks, 256, 0, st>>>(n, cur, child, size, node_depth, out_rank_dev, root_of_dev);
  KD_LAUNCHED();
  KD_TRY(cudaMemsetAsync(remaining, 0, 8, st));
  // level-synchronous rounds over the first m points until all of them are placed; lockstep = every unplaced point is at depth `d`
  // first_check: the host does not look before that round (a random tree of m points is ~3 ln m deep at least)
  auto rounds = [&](int64_t m, bool lockstep, int first_check) -> int32_t {
    const int mb = div_up(m, 256);
    for (int d = 0;; ++d) {
      if ((d & 3) == 0) KD_TRY(cudaMemsetAsync(remaining, 0, 4, st));
      if (lockstep && d < 14 && m > 8192) kd_descend_kernel<true><<<mb, 256, 0, st>>>((const double2*)xy_dev, m, d & 1, cur, child, size, side);
      else kd_descend_kernel<false><<<mb, 256, 0, st>>>((const double2*)xy_dev, m, lockstep ? (d & 1) : -1, cur, child, size, side, node_depth);
      KD_LAUNCHED();
      kd_place_kernel<<<mb, 256, 0, st>>>(m, cur, child, side, parent, node_depth, (d & 3) == 3 ? remaining : nullptr, max_depth);
      KD_LAUNCHED();
      if ((d & 3) != 3 || d < first_check) continue;      // the host looks at the number of unplaced points every fourth level only
      int32_t rem = 0;
      KD_TRY(cudaMemcpyAsync(&rem, remaining, 4, cudaMemcpyDeviceToHost, st));
      KD_TRY(cudaStreamSynchronize(st));
      if (rem == 0) return PORRT_OK;
      if (d > m + 4) return fail("no convergence", cudaErrorUnknown);
    }
  };
  const int64_t KD_TOP = 65536;
  const bool two_phase = !root_of_dev && n >= 8 * KD_TOP;
  if (two_phase) {
    int32_t rc = rounds(KD_TOP, true, 27);              // the top tree: points 0 .. KD_TOP-1 (later points have cur == root but are not looked at)
    if (rc) return rc;
    int32_t top_depth = 0;
    KD_TRY(cudaMemcpyAsync(&top_depth, max_depth, 4, cudaMemcpyDeviceToHost, st));
    KD_TRY(cudaMemsetAsync(exits, 0, (size_t)KD_TOP * 4, st));
    kd_walk_kernel<<<div_up(n - KD_TOP, 256), 256, 0, st>>>((const double2*)xy_dev, KD_TOP, n, child, node_depth, cur, exits);
    KD_LAUNCHED();
    KD_TRY(cudaStreamSynchronize(st));
    for (int d = top_depth; d >= 0; --d) {
      kd_top_sizes_kernel<<<div_up(KD_TOP, 256), 256, 0, st>>>(KD_TOP, d, node_depth, child, exits, up, size);
      KD_LAUNCHED();
    }
    rc = rounds(n, false, 7);                           // everybody else, from where the walk left them
    if (rc) return rc;
  } else {
    int32_t rc = rounds(n, true, n >= 4096 ? 11 : 0);
    if (rc) return rc;
  }
  int32_t depth = 0;
  KD_TRY(cudaMemcpyAsync(&depth, max_depth, 4, cudaMemcpyDeviceToHost, st));
  KD_TRY(cudaStreamSynchronize(st));
  if (depth <= 8) {
    for (int d = 1; d <= depth; ++d) {
      kd_rank_kernel<<<blocks, 256, 0, st>>>(n, d, node_depth, parent, side, child, size, out_rank_dev);
      KD_LAUNCHED();
    }
  } else {
    // cur / exits / up are free now; node_depth is read by the init only, so it serves as the fourth buffer afterwards
    int32_t* jump_a = cur; int32_t* acc_a = exits; int32_t* jump_b = up; int32_t* acc_b = node_depth;
    kd_rank_init_kernel<<<blocks, 256, 0, st>>>(n, parent, side, child, size, node_depth, out_rank_dev, jump_a, acc_a);
    KD_LAUNCHED();
    int covered = 1;                                  // path length a node's acc spans after the rounds so far
    while (covered <= depth) {
      kd_rank_jump_kernel<<<blocks, 256, 0, st>>>(n, jump_a, acc_a, jump_b, acc_b);
      KD_LAUNCHED();
      std::swap(jump_a, jump_b); std::swap(acc_a, acc_b);
      covered *= 2;
    }
    KD_TRY(cudaMemcpyAsync(out_rank_dev, acc_a, (size_t)n * 4, cudaMemcpyDeviceToDevice, st));
  }
#undef KD_TRY
#undef KD_LAUNCHED
  if (n_launch) *n_launch = launches; else ctx->launches += launches;
  return PORRT_OK;
}

PORRT_API int32_t porrt_kd_preorder_rank(porrt_ctx* ctx, const double* xy, int64_t n, int32_t* out_rank) {
  CTX_CHECK(ctx);
  if (!xy) n = ctx->n_vertices;   // xy == NULL: the rank of the ctx's own vertex set (porrt_vertices_set / _append), nothing is uploaded
  if (n < 0 || (n > 0 && !out_rank)) return porrt_fail(ctx, PORRT_ERR_INVALID_ARG, "kd_preorder_rank: bad arguments");
  if (n == 0) return PORRT_OK;
  CUDA_TRY(ctx, cudaSetDevice(ctx->device));
  double* d_xy;
  int32_t* d_rank;
  CUDA_TRY(ctx, carve(ctx->radix_vals, [&](Carve& c) { d_xy = c.take<double>(2 * n); d_rank = c.take<int32_t>(n); }));
  if (xy) CUDA_TRY(ctx, cudaMemcpyAsync(d_xy, xy, (size_t)n * 16, cudaMemcpyHostToDevice, ctx->stream));
  else d_xy = ctx->d_vxy.as<double>();
  int32_t rc = kd_preorder_rank_dev(ctx, d_xy, n, d_rank, nullptr);
  if (rc) return rc;
  CUDA_TRY(ctx, cudaMemcpyAsync(out_rank, d_rank, (size_t)n * 4, cudaMemcpyDeviceToHost, ctx->stream));
  CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
  return PORRT_OK;
}

// ================================================================================================ PRM build
__global__ void iota_u32_kernel(uint32_t* __restrict__ out, int64_t n) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) out[i] = (uint32_t)i;
}

__global__ void seg_owner_kernel(const int64_t* __restrict__ offsets, int64_t m, int32_t base, int32_t* __restrict__ owner) {
  const int lane = threadIdx.x & 31;
  const int64_t seg = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  if (seg >= m) return;
  const int64_t s = offsets[seg], e = offsets[seg + 1];
  for (int64_t k = s + lane; k < e; k += 32) owner[k] = base + (int32_t)seg;
}

// sharded build: the compacted neighbour lists of this rank's segments, packed densely for the exchange
__global__ void prm_pack_kernel(const int64_t* __restrict__ offsets, const int64_t* __restrict__ dense_off, int64_t m,
                                const int32_t* __restrict__ compact, const int32_t* __restrict__ early_cnt, int32_t* __restrict__ dense) {
  const int lane = threadIdx.x & 31;
  const int64_t seg = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  if (seg >= m) return;
  const int64_t s = offsets[seg], o = dense_off[seg];
  const int32_t c = early_cnt[seg];
  for (int32_t k = lane; k < c; k += 32) dense[o + k] = compact[s + k];
}
__global__ void prm_shard_summary_kernel(const int64_t* __restrict__ local_total, const int32_t* __restrict__ flag, int64_t* __restrict__ out2) {
  out2[0] = *local_total; out2[1] = (int64_t)*flag;
}

// ordered compaction of the valid hits of every segment + counts; one warp per segment
__global__ void prm_compact_kernel(const int64_t* __restrict__ offsets, int64_t m, const int32_t* ids,
                                   const int32_t* __restrict__ vid, int32_t* __restrict__ early_cnt,
                                   int32_t* compact /* may alias ids: compaction in place */, int32_t* __restrict__ panic_flag) {
  const int lane = threadIdx.x & 31;
  const int64_t seg = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  if (seg >= m) return;
  const int64_t s = offsets[seg], e = offsets[seg + 1];
  int32_t cnt = 0;
  for (int64_t k0 = s; k0 < e; k0 += 32) {
    const int64_t k = k0 + lane;
    int32_t v = k < e ? vid[k] : -1;
    int32_t id = k < e ? ids[k] : 0;
    if (v < -1) atomicExch(panic_flag, v);
    unsigned ok = __ballot_sync(0xffffffffu, v >= 0);
    __syncwarp();
    if (v >= 0) compact[s + cnt + __popc(ok & ((1u << lane) - 1u))] = id;  // writes land at or before the reads of this round
    cnt += __popc(ok);
    __syncwarp();
  }
  if (lane == 0) early_cnt[seg] = cnt;
}

// Transpose of the (new node k -> valid earlier neighbours j) lists: node j receives every such k as a child, in ascending k
// (insertion order, prm.rs:99-106).  Pass 1 counts per j, pass 2 scatters k behind a per-j cursor in arbitrary order; each row
// is then sorted ascending by the register segment sort (rows are ~26 entries) -- the result is the unique ascending order,
// and it replaces a 3-pass stable radix sort of all (j, k) pairs (3.4 ms at 2.6e7 pairs) by ~1 ms.
__global__ void prm_late_count_kernel(const int64_t* __restrict__ offsets, int64_t m, const int32_t* __restrict__ compact,
                                      const int32_t* __restrict__ early_cnt, int32_t* __restrict__ late_cnt) {
  const int lane = threadIdx.x & 31;
  const int64_t seg = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  if (seg >= m) return;
  const int64_t s = offsets[seg];
  const int32_t c = early_cnt[seg];
  for (int32_t k = lane; k < c; k += 32) atomicAdd(&late_cnt[compact[s + k]], 1);
}
__global__ void prm_late_scatter_kernel(const int64_t* __restrict__ offsets, int64_t m, const int32_t* __restrict__ compact,
                                        const int32_t* __restrict__ early_cnt, const int64_t* __restrict__ late_off,
                                        int32_t* __restrict__ cursor, int32_t* __restrict__ late_vals) {
  const int lane = threadIdx.x & 31;
  const int64_t seg = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  if (seg >= m) return;
  const int64_t s = offsets[seg];
  const int32_t c = early_cnt[seg];
  for (int32_t k = lane; k < c; k += 32) {
    const int32_t j = compact[s + k];
    late_vals[late_off[j] + atomicAdd(&cursor[j], 1)] = (int32_t)seg;
  }
}

__global__ void prm_rowptr_kernel(const int64_t* __restrict__ early_off, const int64_t* __restrict__ late_off, int64_t m,
                                  int64_t* __restrict__ row_ptr) {
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i <= m) row_ptr[i] = early_off[i] + late_off[i];
}

// early_vid / vid (nullable together): the validity id of every edge rides along (PTO growth, pto_grow.cu).  A late entry k of row
// seg is the edge seg <-> k that node k logged in its own early list; its id is looked up there (early lists are short).
__global__ void prm_fill_kernel(const int64_t* __restrict__ offsets, int64_t m, const int32_t* __restrict__ compact,
                                const int32_t* __restrict__ early_cnt, const int64_t* __restrict__ late_off,
                                const int32_t* __restrict__ late_vals, const int64_t* __restrict__ row_ptr, int32_t* __restrict__ col,
                                const int32_t* __restrict__ early_vid, int32_t* __restrict__ vid) {
  const int lane = threadIdx.x & 31;
  const int64_t seg = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  if (seg >= m) return;
  const int64_t s = offsets[seg], r = row_ptr[seg];
  const int32_t c = early_cnt[seg];
  for (int32_t k = lane; k < c; k += 32) {
    col[r + k] = compact[s + k];
    if (vid) vid[r + k] = early_vid[s + k];
  }
  const int64_t ls = late_off[seg], le = late_off[seg + 1];
  for (int64_t k = ls + lane; k < le; k += 32) {
    const int32_t later = late_vals[k];
    col[r + c + (k - ls)] = later;
    if (vid) {
      const int64_t ks = offsets[later];
      int32_t v = -1;
      for (int32_t q = 0; q < early_cnt[later]; ++q)
        if (compact[ks + q] == (int32_t)seg) { v = early_vid[ks + q]; break; }
      vid[r + c + (k - ls)] = v;
    }
  }
}

// The children CSR of a roadmap whose edges were logged per new node (row k = its early list, then the later nodes that listed k,
// ascending): the tail of the PRM build below as one call.  seg_off[n + 1] (seg_off[n] = early entries), early_cnt[n]; work
// buffers: late_cnt / cursor [n] int32, late_off [n + 1] int64, late_vals [seg_off[n]] int32.  Enqueued on ctx->stream.
int32_t late_list_csr_dev(porrt_ctx* ctx, const int64_t* seg_off, int64_t n, const int32_t* compact, const int32_t* early_cnt,
                          const int32_t* early_vid, int32_t* late_cnt, int32_t* cursor, int64_t* late_off, int32_t* late_vals,
                          int64_t* row_ptr, int32_t* col, int32_t* vid) {
  cudaStream_t st = ctx->stream;
  CUDA_TRY(ctx, cudaMemsetAsync(late_cnt, 0, (size_t)n * 4, st));
  CUDA_TRY(ctx, cudaMemsetAsync(cursor, 0, (size_t)n * 4, st));
  prm_late_count_kernel<<<div_up(n * 32, 256), 256, 0, st>>>(seg_off, n, compact, early_cnt, late_cnt);
  LAUNCH_CHECK(ctx);
  int32_t rc = scan_exclusive_i64(ctx, late_cnt, n, late_off);
  if (rc) return rc;
  prm_rowptr_kernel<<<div_up(n + 1, 256), 256, 0, st>>>(seg_off, late_off, n, row_ptr);
  LAUNCH_CHECK(ctx);
  prm_late_scatter_kernel<<<div_up(n * 32, 256), 256, 0, st>>>(seg_off, n, compact, early_cnt, late_off, cursor, late_vals);
  LAUNCH_CHECK(ctx);
  rc = segments_sort_by_key_dev(ctx, late_off, n, late_vals, nullptr, n);   // later nodes ascending
  if (rc) return rc;
  prm_fill_kernel<<<div_up(n * 32, 256), 256, 0, st>>>(seg_off, n, compact, early_cnt, late_off, late_vals, row_ptr, col, early_vid, vid);
  LAUNCH_CHECK(ctx);
  return PORRT_OK;
}

// ms_arr / sr_arr (nullable): per-sample (max_step, search_radius) of the add_sample call that created node k -- the multi-modal
// PRM seeds goal nodes with add_sample(goal, 0.0, 0.0) (map_shelves_tamp_prm.rs:211,256), i.e. radius 0 = exact duplicates only
int32_t prm_build_impl(porrt_ctx* ctx, const double* samples_xy, int64_t n, double max_step, double search_radius,
                       const double* ms_arr, const double* sr_arr,
                       int64_t* out_row_ptr, int32_t* out_col, int64_t cap, int64_t* out_n_edges, double* out_phase_ms,
                       const int64_t* group_ptr, int32_t n_groups) {
  // group_ptr (nullable, [n_groups + 1]): several independent roadmaps in one call -- the samples group_ptr[g] .. group_ptr[g+1]-1
  // form roadmap g (the PRM of mode g of a multi-modal PRM).  Node ids stay global; a node only ever sees earlier nodes of its
  // own group (id range test in the radius kernels), its radius uses its index inside the group, and every group has its own kd
  // order.  One binning, one radius batch, one edge batch and one CSR serve all roadmaps.
  CTX_CHECK(ctx);
  ctx->prm_n = 0;
  if (!ctx->has_map) return porrt_fail(ctx, PORRT_ERR_NO_MAP, "no map uploaded");
  if (n <= 0 || !samples_xy || !out_row_ptr || !out_n_edges) return porrt_fail(ctx, PORRT_ERR_INVALID_ARG, "prm_build: bad arguments");
  std::vector<uint32_t> group_base;   // [n]: first id of the node's group
  if (group_ptr) {
    if (ctx->comm_world > 1) return porrt_fail(ctx, PORRT_ERR_UNSUPPORTED, "prm_build: grouped builds are not sharded");
    if (n_groups <= 0 || group_ptr[0] != 0 || group_ptr[n_groups] != n) return porrt_fail(ctx, PORRT_ERR_INVALID_ARG, "prm_build: bad group table");
    group_base.resize((size_t)n);
    for (int g = 0; g < n_groups; ++g) {
      if (group_ptr[g + 1] < group_ptr[g]) return porrt_fail(ctx, PORRT_ERR_INVALID_ARG, "prm_build: bad group table");
      for (int64_t k = group_ptr[g]; k < group_ptr[g + 1]; ++k) group_base[(size_t)k] = (uint32_t)group_ptr[g];
    }
  }
  const uint32_t* gb = group_ptr ? group_base.data() : nullptr;
  CUDA_TRY(ctx, cudaSetDevice(ctx->device));
  cudaStream_t st = ctx->stream;
  double t0 = now_ms(), t1;
  double ph[8] = {0};

  // radii: node k (k >= 1) queries with heuristic_radius(k + 1) -- n_nodes AFTER adding the new node (prm.rs:61-65).
  // libm on host threads, started now and joined after the device has binned the vertices and ranked the kd-tree
  // (neither needs the radii): ~3.6 ms at n = 1e6 that used to sit in front of the device work.
  CUDA_TRY(ctx, ctx->pin_radii.ensure((size_t)n * 8));   // pinned: the upload after the join is one async DMA
  double* radius = ctx->pin_radii.as<double>();
  // multi-GPU (comm.cu): this rank answers the queries of new nodes [lo, hi) only -- and needs only their radii
  const int world = ctx->comm_world;
  int64_t lo = 0, hi = n;
  // Shard boundaries by estimated WORK, not by count: node k's query covers ~(2 r(k) / cell + 1)^2 cells of a grid whose cell is the
  // last node's radius, so the first nodes cost hundreds of times more than the last ones (equal counts left rank 0 with 2.2 ms of
  // radius queries at 8 GPUs while the others were done in 0.3).  Every rank computes the same boundaries from the same closed form.
  std::vector<int64_t> bnd((size_t)world + 1, 0);
  bnd[(size_t)world] = n;
  if (world > 1) {
    const double r_n = n > 2 ? search_radius * std::sqrt(std::log((double)n) / (double)n) : max_step;
    const double cell_est = std::max(1e-12, std::min(r_n, max_step > 0 ? max_step : r_n));
    auto cost = [&](double k) {   // cells covered + a constant for the candidates that are always looked at
      const double r = k < 2 ? 0.0 : std::min(search_radius * std::sqrt(std::log(k + 1.0) / (k + 1.0)), max_step > 0 ? max_step : 1e300);
      const double side = 2.0 * r / cell_est + 1.0;
      return 40.0 + side * side;
    };
    std::vector<double> ks, cum;   // cumulative cost on a geometric grid of node indices
    for (double k = 1.0; k < (double)n; k = std::max(k + 1.0, k * 1.01)) ks.push_back(k);
    ks.push_back((double)n);
    cum.assign(ks.size(), 0.0);
    for (size_t i = 1; i < ks.size(); ++i) cum[i] = cum[i - 1] + 0.5 * (cost(ks[i - 1]) + cost(ks[i])) * (ks[i] - ks[i - 1]);
    for (int r = 1; r < world; ++r) {
      const double want = cum.back() * (double)r / (double)world;
      const size_t i = (size_t)(std::upper_bound(cum.begin(), cum.end(), want) - cum.begin());
      double k = (double)n;
      if (i > 0 && i < ks.size()) k = ks[i - 1] + (ks[i] - ks[i - 1]) * (want - cum[i - 1]) / std::max(1e-300, cum[i] - cum[i - 1]);
      bnd[(size_t)r] = std::max<int64_t>(bnd[(size_t)r - 1], std::min<int64_t>(n, (int64_t)k));
    }
    lo = bnd[(size_t)ctx->comm_rank]; hi = bnd[(size_t)ctx->comm_rank + 1];
  }
  const int64_t m = hi - lo;
  std::vector<std::thread> th;
  // heuristic_radius is a pure function of (k, max_step, search_radius): a ctx that builds roadmaps of the same parameters again
  // (replanning, seeds, benchmark repetitions) finds its radii in the pinned table from last time
  const bool radii_cached = !gb && !ms_arr && !sr_arr && ctx->radii_ptr == (const void*)radius && ctx->radii_n >= hi && ctx->radii_lo <= lo && ctx->radii_ms == max_step && ctx->radii_sr == search_radius;
  if (!radii_cached) {
    ctx->radii_n = 0;
    int nt = (int)std::min<int64_t>(std::max(2u, std::thread::hardware_concurrency()) / 2, 8);   // leave cores to the driver's copies
    if (world > 1) nt = std::max(1, nt / world + 1);                                                // the box's cores are shared by all ranks
    if (m < 20000) nt = 1;
    for (int t = 0; t < nt; ++t)
      th.emplace_back([=]() {
        const int64_t per = (m + nt - 1) / nt, k0 = lo + t * per, k1 = std::min<int64_t>(hi, k0 + per);   // contiguous: no shared cache lines
        for (int64_t k = k0; k < k1; ++k) {
          const int64_t kl = gb ? k - (int64_t)gb[k] : k;   // index inside the node's own roadmap
          radius[k] = kl == 0 ? -1.0 : heuristic_radius(kl + 1, ms_arr ? ms_arr[k] : max_step, sr_arr ? sr_arr[k] : search_radius, 2);
        }
      });
  }
  struct Joiner { std::vector<std::thread>& t; ~Joiner() { for (auto& x : t) if (x.joinable()) x.join(); } } joiner{th};

  // device inputs
  CUDA_TRY(ctx, ctx->d_vxy.ensure((size_t)n * 16));
  double* d_radius;
  int64_t *d_off, *d_early_off, *d_late_off;
  uint32_t* d_prefix;
  int32_t *d_rank, *d_early_cnt, *d_late_cnt, *d_flag;
  uint32_t* d_group_base = nullptr;
  CUDA_TRY(ctx, carve(ctx->ws_main, [&](Carve& c) {
    d_radius = c.take<double>(n);
    d_off = c.take<int64_t>(n + 1); d_early_off = c.take<int64_t>(n + 1); d_late_off = c.take<int64_t>(n + 1);
    d_prefix = c.take<uint32_t>(n);
    d_rank = c.take<int32_t>(n); d_early_cnt = c.take<int32_t>(n); d_late_cnt = c.take<int32_t>(n);
    d_flag = c.take<int32_t>(4);
    if (gb) d_group_base = c.take<uint32_t>(n);
  }));
  // the result lives in its own buffers: it is retained (porrt_prm_fetch, porrt_graph_from_prm) while later calls reuse the work space
  CUDA_TRY(ctx, ctx->d_prm_row.ensure((size_t)(n + 1) * 8));
  int64_t* d_row_ptr = ctx->d_prm_row.as<int64_t>();
  if (gb) CUDA_TRY(ctx, cudaMemcpyAsync(d_group_base, gb, (size_t)n * 4, cudaMemcpyHostToDevice, st));
  CUDA_TRY(ctx, cudaMemcpyAsync(ctx->d_vxy.p, samples_xy, (size_t)n * 16, cudaMemcpyHostToDevice, st));
  CUDA_TRY(ctx, cudaMemsetAsync(d_late_cnt, 0, (size_t)n * 4, st));
  CUDA_TRY(ctx, cudaMemsetAsync(d_flag, 0, 4, st));

  // the kd pre-order rank of every vertex (restores the reference's neighbour order in step 5) needs only the coordinates: ~150
  // small launches with a host check every fourth tree level, latency-bound.  A helper thread runs it on a second stream while
  // this thread bins, searches and checks edges (throughput-bound kernels); the two meet before the neighbour lists are sorted.
  if (!ctx->aux_stream) CUDA_TRY(ctx, cudaStreamCreateWithFlags(&ctx->aux_stream, cudaStreamNonBlocking));
  CUDA_TRY(ctx, cudaEventRecord(ctx->ev_k[1], st));
  CUDA_TRY(ctx, cudaStreamWaitEvent(ctx->aux_stream, ctx->ev_k[1], 0));
  struct KdJob { int32_t rc = PORRT_OK; std::string err; int64_t launches = 0; std::thread th; bool joined = true; } kd;
  auto start_kd = [&]() {
    porrt_ctx* c = ctx; int32_t* rank_out = d_rank; const uint32_t* roots = d_group_base; KdJob* job = &kd;
    kd.joined = false;
    kd.th = std::thread([c, n, rank_out, roots, job]() {
      if (cudaSetDevice(c->device) != cudaSuccess) { job->rc = PORRT_ERR_CUDA; job->err = "kd thread: cudaSetDevice failed"; return; }
      job->rc = kd_preorder_rank_dev(c, c->d_vxy.as<double>(), n, rank_out, roots, c->aux_stream, &job->err, &job->launches);
      if (job->rc == PORRT_OK && cudaStreamSynchronize(c->aux_stream) != cudaSuccess) { job->rc = PORRT_ERR_CUDA; job->err = "kd thread: stream sync failed"; }
    });
  };
  struct KdJoiner { KdJob& j; ~KdJoiner() { if (!j.joined && j.th.joinable()) j.th.join(); } } kd_joiner{kd};   // early returns
  // (starting the rank after the binning sort instead of next to it was measured: no difference beyond run-to-run noise)
  start_kd();

  // 1. bin vertices; cell = the smallest radius in use (the last one) so late queries touch 3x3 cells
  double r_last = n > 1 ? heuristic_radius(n, max_step, search_radius, 2) : -1.0;
  if (ms_arr || sr_arr) {   // per-sample parameters: the smallest positive radius in use (needs the radii: no overlap here)
    for (auto& x : th) if (x.joinable()) x.join();
    r_last = -1.0;
    for (int64_t k = lo; k < hi; ++k)
      if (radius[k] > 0.0 && (r_last < 0.0 || radius[k] < r_last)) r_last = radius[k];
    if (world > 1) r_last = -1.0;   // (shards would disagree on the cell size; per-sample parameters are a small-n path)
  }
  double cell = r_last > 0 ? r_last : (max_step > 0 ? max_step : 0.05);
  int32_t rc = nn_vertices_set_dev(ctx, ctx->d_vxy.as<double>(), n, cell, nullptr, nullptr);
  if (rc) return rc;
  CUDA_TRY(ctx, cudaStreamSynchronize(st));
  t1 = now_ms(); ph[1] = t1 - t0; t0 = t1;

  for (auto& x : th) if (x.joinable()) x.join();
  if (!radii_cached && !gb && !ms_arr && !sr_arr) { ctx->radii_lo = lo; ctx->radii_n = hi; ctx->radii_ms = max_step; ctx->radii_sr = search_radius; ctx->radii_ptr = radius; }
  if (m > 0) CUDA_TRY(ctx, cudaMemcpyAsync(d_radius + lo, radius + lo, (size_t)m * 8, cudaMemcpyHostToDevice, st));
  iota_u32_kernel<<<div_up(n, 256), 256, 0, st>>>(d_prefix, n);   // prefix limit of query k = k: the tree before node k arrived
  LAUNCH_CHECK(ctx);
  t1 = now_ms(); ph[0] = t1 - t0; t0 = t1;   // what is left of the radii after the overlap

  // (bins and kd ranks above are replicated on every rank; from here on the rank works on its shard [lo, hi))
  // 3. prefix-restricted radius queries: neighbours(k) = { j < k : norm2(x_j, x_k) <= r_k }
  int64_t total = 0;
  rc = nn_radius_count_fill_dev(ctx, ctx->d_vxy.as<double>() + 2 * lo, d_radius + lo, m, d_prefix + lo, nullptr, nullptr, d_off, &ctx->ws_table, &total,
                                d_group_base ? d_group_base + lo : nullptr, false, false);
  if (rc) return rc;
  CUDA_TRY(ctx, cudaStreamSynchronize(st));
  t1 = now_ms(); ph[2] = t1 - t0; t0 = t1;

  int32_t* d_ids = ctx->ws_table.as<int32_t>();

  // 4. edge checks neighbour -> new node (prm.rs:91-96); the order inside a list does not matter to them
  const int64_t tot1 = std::max<int64_t>(total, 1);
  CUDA_TRY(ctx, ctx->ws_owner.ensure((size_t)tot1 * 4));  // owner (= new node id)
  CUDA_TRY(ctx, ctx->ws_vid.ensure((size_t)tot1 * 4));    // validity ids
  int32_t* d_owner = ctx->ws_owner.as<int32_t>();
  int32_t* d_vid = ctx->ws_vid.as<int32_t>();
  if (total > 0) {
    seg_owner_kernel<<<div_up(m * 32, 256), 256, 0, st>>>(d_off, m, (int32_t)lo, d_owner);
    LAUNCH_CHECK(ctx);
    rc = map_edge_validity_indexed_dev(ctx, ctx->d_vxy.as<double>(), d_ids, d_owner, total, d_vid, st);
    if (rc) return rc;
  }
  CUDA_TRY(ctx, cudaStreamSynchronize(st));
  t1 = now_ms(); ph[5] = t1 - t0; t0 = t1;

  // 5. + 6. valid neighbours in kd pre-order, then the CSR in insertion order: row k = valid earlier neighbours (kd order), then later nodes ascending (prm.rs:99-106)
  if (m > 0) {
    prm_compact_kernel<<<div_up(m * 32, 256), 256, 0, st>>>(d_off, m, d_ids, d_vid, d_early_cnt + lo, d_ids, d_flag);
    LAUNCH_CHECK(ctx);
  }
  int64_t n_half = 0;
  int32_t flag = 0;
  const int64_t* d_seg_off = d_off;      // where the compacted list of segment k starts ...
  const int32_t* d_compact = d_ids;      // ... in this array
  if (world == 1) {
    rc = scan_exclusive_i64(ctx, d_early_cnt, n, d_early_off);
    if (rc) return rc;
    CUDA_TRY(ctx, cudaMemcpyAsync(&n_half, d_early_off + n, 8, cudaMemcpyDeviceToHost, st));
    CUDA_TRY(ctx, cudaMemcpyAsync(&flag, d_flag, 4, cudaMemcpyDeviceToHost, st));
    CUDA_TRY(ctx, cudaStreamSynchronize(st));
    if (flag >= -1) {
      // valid neighbours packed densely, then every list put into kd pre-order (2/3 of the candidates are left to sort)
      CUDA_TRY(ctx, ctx->ws_owner.ensure((size_t)std::max<int64_t>(n_half, 1) * 4));   // the owner list is dead by now
      int32_t* d_dense = ctx->ws_owner.as<int32_t>();
      prm_pack_kernel<<<div_up(n * 32, 256), 256, 0, st>>>(d_off, d_early_off, n, d_ids, d_early_cnt, d_dense);
      LAUNCH_CHECK(ctx);
      const double tw = now_ms();
      rc = [&]() -> int32_t {   // meet the kd-rank thread
    if (!kd.joined) { kd.th.join(); kd.joined = true; ctx->launches += kd.launches; }
    if (kd.rc) return porrt_fail(ctx, kd.rc, kd.err);
    return PORRT_OK;
  }();
      if (rc) return rc;
      ph[3] = now_ms() - tw;   // what is left of the kd rank after the overlap
      const double ts = now_ms();
      rc = segments_sort_by_key_dev(ctx, d_early_off, n, d_dense, d_rank, n);
      if (rc) return rc;
      CUDA_TRY(ctx, cudaStreamSynchronize(st));
      ph[4] = now_ms() - ts;
      t0 += ph[3] + ph[4];     // keep them out of the csr phase below
      d_seg_off = d_early_off; d_compact = d_dense;
    }
  } else {
    // the exchange step (SURVEY 8(e)): every rank gets all counts and all valid (neighbour, new node) lists, then
    // assembles the whole CSR itself -- the graph stays device-resident on every GPU for the value backups that follow.
    const double tx0 = now_ms();
    int64_t* d_local_off = d_late_off;   // free until the transpose below
    rc = scan_exclusive_i64(ctx, d_early_cnt + lo, m, d_local_off);
    if (rc) return rc;
    CUDA_TRY(ctx, ctx->radix_hist.ensure((size_t)world * 16 + 64));
    int64_t* d_summary = ctx->radix_hist.as<int64_t>();
    prm_shard_summary_kernel<<<1, 1, 0, st>>>(d_local_off + m, d_flag, d_summary + 2 * ctx->comm_rank);
    LAUNCH_CHECK(ctx);
    std::vector<int64_t> off16(world + 1);
    for (int r = 0; r <= world; ++r) off16[r] = 16 * (int64_t)r;
    rc = comm_all_gatherv_dev(ctx, nullptr, d_summary, off16.data(), st);
    if (rc) return rc;
    std::vector<int64_t> cnt_off(world + 1);
    for (int r = 0; r <= world; ++r) cnt_off[r] = bnd[(size_t)r] * 4;
    rc = comm_all_gatherv_dev(ctx, nullptr, d_early_cnt, cnt_off.data(), st);
    if (rc) return rc;
    std::vector<int64_t> summary(2 * world);
    CUDA_TRY(ctx, cudaMemcpyAsync(summary.data(), d_summary, (size_t)world * 16, cudaMemcpyDeviceToHost, st));
    CUDA_TRY(ctx, cudaStreamSynchronize(st));
    std::vector<int64_t> ids_off(world + 1, 0);
    for (int r = 0; r < world; ++r) {
      ids_off[r + 1] = ids_off[r] + summary[2 * r] * 4;
      if (summary[2 * r + 1] < -1) flag = (int32_t)summary[2 * r + 1];   // a panic on any rank fails the build on every rank
    }
    n_half = ids_off[world] / 4;
    if (flag >= -1) {
      CUDA_TRY(ctx, ctx->ws_owner.ensure((size_t)std::max<int64_t>(n_half, 1) * 4));   // the owner list is dead by now
      int32_t* d_dense = ctx->ws_owner.as<int32_t>();
      if (m > 0) {
        prm_pack_kernel<<<div_up(m * 32, 256), 256, 0, st>>>(d_off, d_local_off, m, d_ids, d_early_cnt + lo, d_dense + ids_off[ctx->comm_rank] / 4);
        LAUNCH_CHECK(ctx);
      }
      rc = [&]() -> int32_t {   // meet the kd-rank thread
    if (!kd.joined) { kd.th.join(); kd.joined = true; ctx->launches += kd.launches; }
    if (kd.rc) return porrt_fail(ctx, kd.rc, kd.err);
    return PORRT_OK;
  }();
      if (rc) return rc;
      if (m > 0) rc = segments_sort_by_key_dev(ctx, d_local_off, m, d_dense + ids_off[ctx->comm_rank] / 4, d_rank, n);   // kd pre-order, this rank's lists
      if (rc) return rc;
      rc = comm_all_gatherv_dev(ctx, nullptr, d_dense, ids_off.data(), st);
      if (rc) return rc;
      rc = scan_exclusive_i64(ctx, d_early_cnt, n, d_early_off);
      if (rc) return rc;
      d_seg_off = d_early_off; d_compact = d_dense;
      CUDA_TRY(ctx, cudaStreamSynchronize(st));
    }
    ctx->last_ms[0] = now_ms() - tx0; ctx->n_last = 1;   // porrt_ctx_last_phase_ms: wall time of the exchange
  }
  if (flag < -1) return porrt_fail(ctx, PORRT_ERR_PANIC, "prm_build: an edge check hit a reference panic (code " + std::to_string(flag) + ")");
  const int64_t n_edges = 2 * n_half;
  *out_n_edges = n_edges;
  const int64_t half1 = std::max<int64_t>(n_half, 1);
  // the validity ids are dead after the compaction: late lists + cursors go there
  int32_t *d_vals, *d_cursor;
  CUDA_TRY(ctx, carve(ctx->ws_vid, [&](Carve& c) { d_vals = c.take<int32_t>(half1); d_cursor = c.take<int32_t>(n); }));
  CUDA_TRY(ctx, ctx->d_prm_col.ensure((size_t)std::max<int64_t>(n_edges, 1) * 4));
  int32_t* d_col = ctx->d_prm_col.as<int32_t>();
  CUDA_TRY(ctx, cudaMemsetAsync(d_cursor, 0, (size_t)n * 4, st));
  prm_late_count_kernel<<<div_up(n * 32, 256), 256, 0, st>>>(d_seg_off, n, d_compact, d_early_cnt, d_late_cnt);
  LAUNCH_CHECK(ctx);
  rc = scan_exclusive_i64(ctx, d_late_cnt, n, d_late_off);
  if (rc) return rc;
  prm_rowptr_kernel<<<div_up(n + 1, 256), 256, 0, st>>>(d_early_off, d_late_off, n, d_row_ptr);   // row lengths are known: early + late counts
  LAUNCH_CHECK(ctx);
  int32_t status = PORRT_OK;
  if (out_col && cap >= n_edges && n >= (1 << 18) && n_edges > 0) {
    // large roadmaps: the column array (211 MB at 1e6 nodes, ~4 ms over PCIe) leaves in row blocks while the later blocks are
    // still being sorted and written.  row_ptr goes first on the copy stream, next to the scatter of the late lists (the block
    // boundaries are read from its host copy); block b = sort of its rows' late lists, fill, copy -- the copy waits for block b only
    // (small blocks first: the copy engine is the critical path from the moment the first block is ready)
    const int NB = 5;
    const int64_t cut[NB + 1] = {0, n / 16, n / 8, n / 4, n / 2, n};
    cudaEvent_t evs[NB] = {ctx->ev_in[0], ctx->ev_in[1], ctx->ev_in[2], ctx->ev_k[1], ctx->ev_k[2]};
    CUDA_TRY(ctx, cudaEventRecord(ctx->ev_k[0], st));
    CUDA_TRY(ctx, cudaStreamWaitEvent(ctx->copy_out, ctx->ev_k[0], 0));
    CUDA_TRY(ctx, cudaMemcpyAsync(out_row_ptr, d_row_ptr, (size_t)(n + 1) * 8, cudaMemcpyDeviceToHost, ctx->copy_out));
    CUDA_TRY(ctx, cudaEventRecord(ctx->ev_out[0], ctx->copy_out));
    prm_late_scatter_kernel<<<div_up(n * 32, 256), 256, 0, st>>>(d_seg_off, n, d_compact, d_early_cnt, d_late_off, d_cursor, d_vals);
    LAUNCH_CHECK(ctx);
    const bool dbg = getenv("PORRT_DEBUG") != nullptr;
    const double td0 = now_ms();
    CUDA_TRY(ctx, cudaEventSynchronize(ctx->ev_out[0]));          // row_ptr is on the host now
    if (dbg) fprintf(stderr, "[porrt] prm tail: since phase start %.3f ms, row_ptr wait %.3f ms\n", td0 - t0, now_ms() - td0);
    for (int b = 0; b < NB; ++b) {
      const int64_t r0 = cut[b], r1 = cut[b + 1];
      if (r1 > r0) {
        rc = segments_sort_by_key_dev(ctx, d_late_off + r0, r1 - r0, d_vals, nullptr, n);   // later nodes ascending
        if (rc) return rc;
        prm_fill_kernel<<<div_up((r1 - r0) * 32, 256), 256, 0, st>>>(d_seg_off + r0, r1 - r0, d_compact, d_early_cnt + r0, d_late_off + r0, d_vals, d_row_ptr + r0, d_col, nullptr, nullptr);
        LAUNCH_CHECK(ctx);
      }
      cudaEvent_t ev = evs[b];
      CUDA_TRY(ctx, cudaEventRecord(ev, st));
      CUDA_TRY(ctx, cudaStreamWaitEvent(ctx->copy_out, ev, 0));
      const int64_t e0 = out_row_ptr[r0], e1 = out_row_ptr[r1];
      if (e1 > e0) CUDA_TRY(ctx, cudaMemcpyAsync(out_col + e0, d_col + e0, (size_t)(e1 - e0) * 4, cudaMemcpyDeviceToHost, ctx->copy_out));
      if (dbg) fprintf(stderr, "[porrt] prm tail: block %d enqueued at %.3f ms (%lld edges)\n", b, now_ms() - t0, (long long)(e1 - e0));
    }
    CUDA_TRY(ctx, cudaStreamSynchronize(st));
    if (dbg) fprintf(stderr, "[porrt] prm tail: kernels done at %.3f ms\n", now_ms() - t0);
    CUDA_TRY(ctx, cudaStreamSynchronize(ctx->copy_out));
    if (dbg) fprintf(stderr, "[porrt] prm tail: copies done at %.3f ms\n", now_ms() - t0);
  } else {
    prm_late_scatter_kernel<<<div_up(n * 32, 256), 256, 0, st>>>(d_seg_off, n, d_compact, d_early_cnt, d_late_off, d_cursor, d_vals);
    LAUNCH_CHECK(ctx);
    rc = segments_sort_by_key_dev(ctx, d_late_off, n, d_vals, nullptr, n);   // later nodes ascending
    if (rc) return rc;
    prm_fill_kernel<<<div_up(n * 32, 256), 256, 0, st>>>(d_seg_off, n, d_compact, d_early_cnt, d_late_off, d_vals, d_row_ptr, d_col, nullptr, nullptr);
    LAUNCH_CHECK(ctx);
    CUDA_TRY(ctx, cudaMemcpyAsync(out_row_ptr, d_row_ptr, (size_t)(n + 1) * 8, cudaMemcpyDeviceToHost, st));
    if (out_col && cap >= n_edges) {
      if (n_edges > 0) CUDA_TRY(ctx, cudaMemcpyAsync(out_col, d_col, (size_t)n_edges * 4, cudaMemcpyDeviceToHost, st));
    } else {
      status = porrt_fail(ctx, PORRT_ERR_CAPACITY, "prm_build: out_col too small");
    }
    CUDA_TRY(ctx, cudaStreamSynchronize(st));
  }
  t1 = now_ms(); ph[6] = t1 - t0;
  ph[7] = (double)total;
  if (out_phase_ms) memcpy(out_phase_ms, ph, sizeof(ph));
  ctx->prm_n = n; ctx->prm_edges = n_edges; ctx->prm_row_ptr = d_row_ptr; ctx->prm_col = d_col;  // retained for porrt_prm_fetch
  return status;
}

PORRT_API int32_t porrt_prm_build(porrt_ctx* ctx, const double* samples_xy, int64_t n, double max_step, double search_radius,
                                  int64_t* out_row_ptr, int32_t* out_col, int64_t cap, int64_t* out_n_edges, double* out_phase_ms) {
  return prm_build_impl(ctx, samples_xy, n, max_step, search_radius, nullptr, nullptr, out_row_ptr, out_col, cap, out_n_edges, out_phase_ms, nullptr, 0);
}

PORRT_API int32_t porrt_prm_fetch(porrt_ctx* ctx, int64_t* out_row_ptr, int32_t* out_col, int64_t cap) {
  CTX_CHECK(ctx);
  if (ctx->prm_n <= 0) return porrt_fail(ctx, PORRT_ERR_INVALID_ARG, "prm_fetch: no retained PRM result");
  if (cap < ctx->prm_edges || !out_col) return porrt_fail(ctx, PORRT_ERR_CAPACITY, "prm_fetch: out_col too small");
  CUDA_TRY(ctx, cudaSetDevice(ctx->device));
  if (out_row_ptr) CUDA_TRY(ctx, cudaMemcpyAsync(out_row_ptr, ctx->prm_row_ptr, (size_t)(ctx->prm_n + 1) * 8, cudaMemcpyDeviceToHost, ctx->stream));
  if (ctx->prm_edges) CUDA_TRY(ctx, cudaMemcpyAsync(out_col, ctx->prm_col, (size_t)ctx->prm_edges * 4, cudaMemcpyDeviceToHost, ctx->stream));
  CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
  return PORRT_OK;
}

// the device kernels index by col[e] without checks: a malformed graph must be refused on the host
static bool csr_ok(int64_t V, const int64_t* row_ptr, const int32_t* col) {
  if (row_ptr[0] != 0) return false;
  for (int64_t u = 0; u < V; ++u)
    if (row_ptr[u + 1] < row_ptr[u]) return false;
  for (int64_t e = 0; e < row_ptr[V]; ++e)
    if (col[e] < 0 || col[e] >= V) return false;
  return true;
}

// ================================================================================================ SSSP per world
// validity ids < 0 (obstacle / panic codes) -> the appended all-zero row `none`
__global__ void clamp_vid_kernel(int32_t* __restrict__ vid, int64_t n, int32_t none) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n && vid[i] < 0) vid[i] = none;
}
__global__ void edge_cost_kernel(const int64_t* __restrict__ row_ptr, const int32_t* __restrict__ col, const double2* __restrict__ xy,
                                 int64_t V, double* __restrict__ cost) {
  // norm2(u, v) (common.rs:203-213) for every CSR edge u -> v; one warp per row
  const int lane = threadIdx.x & 31;
  const int64_t u = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  if (u >= V) return;
  const double2 a = xy[u];
  for (int64_t e = row_ptr[u] + lane; e < row_ptr[u + 1]; e += 32) {
    const double2 c = xy[col[e]];
    const double dx = __dsub_rn(c.x, a.x), dy = __dsub_rn(c.y, a.y);
    cost[e] = __dsqrt_rn(__dadd_rn(__dmul_rn(dx, dx), __dmul_rn(dy, dy)));
  }
}

__global__ void fill_inf_kernel(double* __restrict__ d, int64_t n) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) d[i] = INFINITY;
}
__global__ void scatter_zero_kernel(double* __restrict__ d, const int64_t* __restrict__ idx, int64_t n) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) d[idx[i]] = 0.0;
}

// plan_qmdp on a graph that already lives on the device (all d_* are device pointers; h_val = host copy of the validity table).
// Roadmaps whose value column fits in shared memory go to the on-chip column solver (colsolve.cu, one column per world), larger
// ones to the frontier relaxation over global memory (sssp_frontier.cu).  out_dist (host, [Wall][V]) may be null: the table then
// stays on the device only (timing, device-resident pipelines).  Work space: ws_table; porrt_ctx_last_phase_ms afterwards:
// [0] device ms of the backups, [1] edge records / (parent, world) pairs worked through.
static int32_t sssp_core(porrt_ctx* ctx, const int64_t* d_row, const int32_t* d_col, const double* d_xy, int64_t V, int64_t E,
                         const int32_t* d_nvid, const uint64_t* d_val, const uint64_t* h_val, int32_t n_validities, int32_t mask_words,
                         bool world_view, int Wall, const int64_t* finals_ptr, const int32_t* finals_ids, double* out_dist,
                         int32_t* out_sweeps) {
  cudaStream_t st = ctx->stream;
  // multi-GPU (comm.cu): the worlds are independent problems on one graph -- rank r relaxes worlds [wlo, whi) and the dist
  // rows are all-gathered (SURVEY 8(e)); the plain-graph call (n_worlds == 0) is not sharded
  int64_t wlo = 0, whi = Wall;
  const bool sharded = world_view && ctx->comm_world > 1;
  if (sharded) comm_shard_range(Wall, ctx->comm_rank, ctx->comm_world, &wlo, &whi);
  const int W = (int)(whi - wlo);
  const bool cols = colsolve_fits(V, E, world_view ? n_validities : 1) && !ctx->force_global_sweeps;
  // the finals of this rank's worlds: indices into the [world][node] table (column solver) or (node, local world) pairs (frontier)
  std::vector<int64_t> zero_idx;
  std::vector<int32_t> fin_nw;
  for (int w = 0; w < Wall; ++w)
    for (int64_t k = finals_ptr[w]; k < finals_ptr[w + 1]; ++k) {
      const int32_t f = finals_ids[k];
      if (f < 0 || f >= V) return porrt_fail(ctx, PORRT_ERR_INVALID_ARG, "sssp_worlds: final id out of range");
      if (w >= wlo && w < whi) {
        if (cols) zero_idx.push_back((int64_t)w * V + f);
        else { fin_nw.push_back(f); fin_nw.push_back((int32_t)(w - wlo)); }
      }
    }
  const int64_t n_fin = cols ? (int64_t)zero_idx.size() : (int64_t)fin_nw.size() / 2;
  double* d_out;   // [Wall][V]: this rank fills rows wlo..whi, the gather the rest
  int32_t* d_flag;
  int64_t* d_zero = nullptr;                           // column solver
  double *d_cost = nullptr, *d_cost_t = nullptr;
  uint32_t *d_ce = nullptr, *d_rs = nullptr, *d_cursor = nullptr;
  uint64_t* d_cmask = nullptr;
  int32_t* d_fin = nullptr;                            // frontier
  CUDA_TRY(ctx, carve(ctx->ws_table, [&](Carve& c) {
    d_out = c.take<double>((size_t)V * Wall);
    d_flag = c.take<int32_t>(4);
    if (W > 0 && cols) {
      d_zero = c.take<int64_t>(n_fin + 1);
      d_cost = c.take<double>(E); d_cost_t = c.take<double>(E);
      d_ce = c.take<uint32_t>(E); d_rs = c.take<uint32_t>(V + 1); d_cursor = c.take<uint32_t>(V + 1);
      d_cmask = c.take<uint64_t>((size_t)Wall * 4);
    } else if (W > 0) {
      d_fin = c.take<int32_t>(2 * n_fin + 2);
    }
  }));
  int sweeps = 0;
  double offers = 0.0;
  tstart(ctx);
  if (W > 0 && cols) {
    // one column per world, solved on chip; d_out is the column-major table itself
    std::vector<uint64_t> cmask((size_t)Wall * 4, world_view ? 0 : ~(uint64_t)0);
    if (world_view)
      for (int w = 0; w < Wall; ++w)
        for (int v = 0; v < n_validities; ++v)
          if ((h_val[(size_t)v * mask_words + w / 64] >> (w % 64)) & 1) cmask[(size_t)w * 4 + v / 64] |= (uint64_t)1 << (v % 64);
    CUDA_TRY(ctx, cudaMemcpyAsync(d_cmask, cmask.data(), cmask.size() * 8, cudaMemcpyHostToDevice, st));
    if (n_fin) CUDA_TRY(ctx, cudaMemcpyAsync(d_zero, zero_idx.data(), (size_t)n_fin * 8, cudaMemcpyHostToDevice, st));
    edge_cost_kernel<<<div_up(V * 32, 256), 256, 0, st>>>(d_row, d_col, (const double2*)d_xy, V, d_cost);
    LAUNCH_CHECK(ctx);
    int32_t rc = colsolve_pack(ctx, d_row, d_col, nullptr, d_cost, V, E, d_rs, d_ce, d_cost_t, d_cursor, st);
    if (rc) return rc;
    fill_inf_kernel<<<ctx->sm_count * 8, 256, 0, st>>>(d_out + wlo * V, V * (int64_t)W);
    LAUNCH_CHECK(ctx);
    if (n_fin) {
      scatter_zero_kernel<<<div_up(n_fin, 256), 256, 0, st>>>(d_out, d_zero, n_fin);
      LAUNCH_CHECK(ctx);
    }
    CUDA_TRY(ctx, cudaMemsetAsync(d_flag, 0, 16, st));
    ColSolveArgs ca = {};
    ca.row_start = d_rs; ca.cost = d_cost_t; ca.ce = d_ce; ca.V = (int32_t)V; ca.ld = V; ca.dist_cm = d_out; ca.cmask = d_cmask;
    ca.nvid = world_view ? d_nvid : nullptr; ca.sweeps_out = d_flag; ca.offers_out = (unsigned long long*)(d_flag + 2);
    rc = colsolve_level(ctx, ca, COLSOLVE_WORLD, (int)wlo, (int)whi, st);
    if (rc) return rc;
    tmark(ctx);
    unsigned long long off = 0;
    CUDA_TRY(ctx, cudaMemcpyAsync(&sweeps, d_flag, 4, cudaMemcpyDeviceToHost, st));
    CUDA_TRY(ctx, cudaMemcpyAsync(&off, d_flag + 2, 8, cudaMemcpyDeviceToHost, st));
    CUDA_TRY(ctx, cudaStreamSynchronize(st));
    offers = (double)off;
  } else if (W > 0) {
    // (node, world) pairs interleaved on the host -> two arrays on the device
    std::vector<int32_t> split((size_t)n_fin * 2);
    for (int64_t k = 0; k < n_fin; ++k) { split[(size_t)k] = fin_nw[(size_t)2 * k]; split[(size_t)(n_fin + k)] = fin_nw[(size_t)2 * k + 1]; }
    if (n_fin) CUDA_TRY(ctx, cudaMemcpyAsync(d_fin, split.data(), (size_t)n_fin * 8, cudaMemcpyHostToDevice, st));
    int32_t rc = sssp_frontier_run(ctx, d_row, d_col, d_xy, V, E, world_view ? d_nvid : nullptr, d_val, mask_words, (int32_t)wlo, W, d_fin,
                                   d_fin + n_fin, n_fin, d_out + wlo * V, &sweeps, &offers, st);
    if (rc) return rc;
    tmark(ctx);
  } else {
    tmark(ctx);
  }
  if (sharded) {
    std::vector<int64_t> off(ctx->comm_world + 1);
    for (int r = 0; r < ctx->comm_world; ++r) { int64_t a2, b2; comm_shard_range(Wall, r, ctx->comm_world, &a2, &b2); off[r] = a2 * V * 8; off[r + 1] = b2 * V * 8; }
    int32_t rc = comm_all_gatherv_dev(ctx, nullptr, d_out, off.data(), st);
    if (rc) return rc;
  }
  if (out_dist) CUDA_TRY(ctx, cudaMemcpyAsync(out_dist, d_out, (size_t)V * Wall * 8, cudaMemcpyDeviceToHost, st));
  CUDA_TRY(ctx, cudaStreamSynchronize(st));
  tfinish(ctx);
  ctx->last_ms[1] = offers; ctx->n_last = 2;
  if (out_sweeps) *out_sweeps = sweeps;
  return PORRT_OK;
}

PORRT_API int32_t porrt_sssp_worlds(porrt_ctx* ctx, int64_t V, const int64_t* row_ptr, const int32_t* col, const double* xy,
                                    const int32_t* node_vid, const uint64_t* validities, int32_t n_validities, int32_t mask_words,
                                    int32_t n_worlds, const int64_t* finals_ptr, const int32_t* finals_ids,
                                    double* out_dist, int32_t* out_sweeps) {
  CTX_CHECK(ctx);
  if (V <= 0 || !row_ptr || !xy || !finals_ptr || !out_dist || n_worlds < 0) return porrt_fail(ctx, PORRT_ERR_INVALID_ARG, "sssp_worlds: bad arguments");
  const bool world_view = n_worlds > 0;
  if (world_view && (!node_vid || !validities || n_validities <= 0 || mask_words <= 0)) return porrt_fail(ctx, PORRT_ERR_INVALID_ARG, "sssp_worlds: world view needs validities");
  CUDA_TRY(ctx, cudaSetDevice(ctx->device));
  cudaStream_t st = ctx->stream;
  const int64_t E = row_ptr[V];
  if (E > 0 && !col) return porrt_fail(ctx, PORRT_ERR_INVALID_ARG, "sssp_worlds: null col");
  if (!csr_ok(V, row_ptr, col)) return porrt_fail(ctx, PORRT_ERR_INVALID_ARG, "sssp_worlds: malformed CSR (row_ptr not monotone or edge target out of range)");
  if (world_view)
    for (int64_t u = 0; u < V; ++u)
      if (node_vid[u] < 0 || node_vid[u] >= n_validities) return porrt_fail(ctx, PORRT_ERR_INVALID_ARG, "sssp_worlds: node validity id out of range");
  const size_t nvw = world_view ? (size_t)n_validities * mask_words : 0;
  int64_t* d_row;
  double* d_xy;
  int32_t *d_col, *d_nvid;
  uint64_t* d_val;
  CUDA_TRY(ctx, carve(ctx->ws_main, [&](Carve& c) {
    d_row = c.take<int64_t>(V + 1); d_xy = c.take<double>(2 * V); d_col = c.take<int32_t>(E); d_nvid = c.take<int32_t>(V);
    d_val = c.take<uint64_t>(nvw);
  }));
  CUDA_TRY(ctx, cudaMemcpyAsync(d_row, row_ptr, (size_t)(V + 1) * 8, cudaMemcpyHostToDevice, st));
  if (E) CUDA_TRY(ctx, cudaMemcpyAsync(d_col, col, (size_t)E * 4, cudaMemcpyHostToDevice, st));
  CUDA_TRY(ctx, cudaMemcpyAsync(d_xy, xy, (size_t)V * 16, cudaMemcpyHostToDevice, st));
  if (world_view) {
    CUDA_TRY(ctx, cudaMemcpyAsync(d_nvid, node_vid, (size_t)V * 4, cudaMemcpyHostToDevice, st));
    CUDA_TRY(ctx, cudaMemcpyAsync(d_val, validities, nvw * 8, cudaMemcpyHostToDevice, st));
  }
  return sssp_core(ctx, d_row, d_col, d_xy, V, E, d_nvid, d_val, validities, n_validities, mask_words, world_view, world_view ? n_worlds : 1,
                   finals_ptr, finals_ids, out_dist, out_sweeps);
}

// plan_qmdp straight on the roadmap porrt_prm_build left on the device (graph, vertex coordinates) under the uploaded map's worlds:
// nothing but the final-node lists crosses the bus on the way in.  Node validity ids are the map's state validity of the vertices
// (evaluated on the device); a vertex inside an obstacle is invalid in every world.  out_dist (host, [n_worlds][V]) may be null.
PORRT_API int32_t porrt_sssp_worlds_prm(porrt_ctx* ctx, const int64_t* finals_ptr, const int32_t* finals_ids, double* out_dist,
                                        int32_t* out_sweeps) {
  CTX_CHECK(ctx);
  if (!ctx->has_map) return porrt_fail(ctx, PORRT_ERR_NO_MAP, "no map uploaded");
  if (ctx->prm_n <= 0) return porrt_fail(ctx, PORRT_ERR_INVALID_ARG, "sssp_worlds_prm: no retained PRM result (porrt_prm_build first)");
  if (!finals_ptr) return porrt_fail(ctx, PORRT_ERR_INVALID_ARG, "sssp_worlds_prm: bad arguments");
  CUDA_TRY(ctx, cudaSetDevice(ctx->device));
  const int64_t V = ctx->prm_n, E = ctx->prm_edges;
  const int nv = ctx->n_validities;
  // node validity ids on the device; obstacles (-1) get an extra all-zero validity row appended to the table
  const size_t nvw = (size_t)(nv + 1) * ctx->mask_words;
  int32_t* d_nvid;
  uint64_t* d_val;
  CUDA_TRY(ctx, carve(ctx->ws_main, [&](Carve& c) { d_nvid = c.take<int32_t>(V); d_val = c.take<uint64_t>(nvw); }));
  std::vector<uint64_t> val(ctx->validities);
  val.resize(nvw, 0);
  CUDA_TRY(ctx, cudaMemcpyAsync(d_val, val.data(), nvw * 8, cudaMemcpyHostToDevice, ctx->stream));
  int32_t rc = porrt_state_validity_dev(ctx, ctx->d_vxy.as<double>(), V, d_nvid);
  if (rc) return rc;
  clamp_vid_kernel<<<div_up(V, 256), 256, 0, ctx->stream>>>(d_nvid, V, nv);
  LAUNCH_CHECK(ctx);
  return sssp_core(ctx, ctx->prm_row_ptr, ctx->prm_col, ctx->d_vxy.as<double>(), V, E, d_nvid, d_val, val.data(), nv + 1, ctx->mask_words, true,
                   ctx->n_worlds, finals_ptr, finals_ids, out_dist, out_sweeps);
}

// ================================================================================================ belief-space VI
// host-side belief algebra (common.rs:256-264,352-355; map_io.rs:244-278; map_shelves_io.rs:206-239)
typedef std::vector<double> Belief;
static uint64_t belief_hash(const double* bs, int n) {
  uint64_t h = 0, p10 = 1;
  for (int i = 0; i < n; ++i) {
    double r = std::round(bs[i] * 1000.0);
    uint64_t v = (r <= 0.0 || std::isnan(r)) ? 0 : (r >= 18446744073709551615.0 ? UINT64_MAX : (uint64_t)r);
    h += (p10 + 1) * v;  // wraps like a release build of the reference
    p10 *= 10;
  }
  return h;
}
// observe_impl's split of one belief by one zone (map_io.rs:257-275, map_shelves_io.rs:217-236): [closed, open] resp.
// [there, not there], each normalised; a zero-mass branch (NaN after the division) is dropped.  Appends to `out` (n doubles per
// belief) and returns how many were kept.
static int successor_beliefs(const porrt_ctx* ctx, const double* b, int n, int zone, std::vector<double>& out) {
  const size_t base = out.size();
  out.resize(base + 2 * (size_t)n);
  double* first = out.data() + base;
  double* second = first + n;
  const bool door = ctx->map.kind == PORRT_DOMAIN_DOOR;
  for (int w = 0; w < n; ++w) {
    const bool in_zone_world = door ? ((ctx->zone_world_masks[(size_t)zone * ctx->mask_words + w / 64] >> (w % 64)) & 1) != 0 : (w == zone);
    const bool to_first = door ? !in_zone_world : in_zone_world;
    first[w] = to_first ? b[w] : 0.0;
    second[w] = to_first ? 0.0 : b[w];
  }
  int kept = 0;
  for (int c = 0; c < 2; ++c) {
    const double* src = out.data() + base + (size_t)c * n;
    double sum = 0.0;
    for (int w = 0; w < n; ++w) sum = sum + src[w];
    bool nan = false;
    double* dst = out.data() + base + (size_t)kept * n;
    for (int w = 0; w < n; ++w) { const double p = src[w] / sum; nan |= std::isnan(p); dst[w] = p; }
    if (!nan) ++kept;
  }
  out.resize(base + (size_t)kept * n);
  return kept;
}

// MapShelfDomain / Map::reachable_belief_states (map_shelves_io.rs:490-520, map_io.rs:515-546): LIFO over (belief, zones not yet
// observed); a successor that is not yet in the list (exact f64 equality) is explored, and appended unless its hash is taken.
PORRT_API int32_t porrt_reachable_belief_states(porrt_ctx* ctx, const double* start_belief, double* out, int32_t cap, int32_t* out_B) {
  CTX_CHECK(ctx);
  if (!ctx->has_map) return porrt_fail(ctx, PORRT_ERR_NO_MAP, "no map uploaded");
  if (!start_belief || !out_B) return porrt_fail(ctx, PORRT_ERR_INVALID_ARG, "reachable_belief_states: bad arguments");
  const int nw = ctx->n_worlds, nz = ctx->n_zones;
  if (nz > 64) return porrt_fail(ctx, PORRT_ERR_UNSUPPORTED, "reachable_belief_states: more than 64 zones");
  // `reachable_beliefs.contains(successor)` is a linear scan with exact f64 equality in the reference (71 ms at 12 zones / 4095
  // beliefs); an open-addressing table over the raw bits answers the same question (no NaNs reach this point: zero-mass branches
  // are dropped; the zeros written by the split and 0.0 / sum are +0.0, so equal values have equal bits) and leaves the
  // enumeration order untouched.  Beliefs live back to back in one arena; a LIFO entry is (arena offset, zones left as bits).
  std::vector<double> reachable(start_belief, start_belief + nw);    // the result list, nw doubles per belief
  std::vector<double> arena(start_belief, start_belief + nw);        // every belief ever pushed on the LIFO
  std::vector<int64_t> table(1024, -1);                               // offsets into `reachable`, open addressing
  size_t n_known = 1;
  auto bits_hash = [&](const double* b) {
    uint64_t h = 1469598103934665603ull;
    for (int w = 0; w < nw; ++w) { uint64_t u; memcpy(&u, b + w, 8); h = (h ^ u) * 1099511628211ull; h ^= h >> 29; }
    return h;
  };
  auto same = [&](const double* x, const double* y) {
    for (int w = 0; w < nw; ++w) if (!(x[w] == y[w])) return false;
    return true;
  };
  auto find_slot = [&](const double* b) {   // slot holding b, or the empty slot where it belongs
    size_t k = (size_t)bits_hash(b) & (table.size() - 1);
    while (table[k] >= 0 && !same(reachable.data() + table[k], b)) k = (k + 1) & (table.size() - 1);
    return k;
  };
  table[find_slot(start_belief)] = 0;
  std::unordered_map<uint64_t, int> hashes;
  std::vector<std::pair<int64_t, uint64_t>> lifo;
  lifo.push_back({0, nz >= 64 ? ~(uint64_t)0 : (((uint64_t)1 << nz) - 1)});
  std::vector<double> succ;
  while (!lifo.empty()) {
    const std::pair<int64_t, uint64_t> top = lifo.back();
    lifo.pop_back();
    for (int zone = 0; zone < nz; ++zone) {
      if (!((top.second >> zone) & 1)) continue;
      const uint64_t remaining = top.second & ~((uint64_t)1 << zone);
      succ.clear();
      const int kept = successor_beliefs(ctx, arena.data() + top.first, nw, zone, succ);
      for (int c = 0; c < kept; ++c) {
        const double* sb = succ.data() + (size_t)c * nw;
        size_t slot = find_slot(sb);
        if (table[slot] >= 0) continue;   // known
        const uint64_t h = belief_hash(sb, nw);
        if (!hashes.count(h)) {
          hashes[h] = 1;
          table[slot] = (int64_t)reachable.size();
          reachable.insert(reachable.end(), sb, sb + nw);
          if (++n_known * 2 > table.size()) {   // grow + rehash
            std::vector<int64_t> old;
            old.swap(table);
            table.assign(old.size() * 4, -1);
            for (int64_t off : old) if (off >= 0) table[find_slot(reachable.data() + off)] = off;
          }
        }
        const int64_t at = (int64_t)arena.size();
        arena.insert(arena.end(), sb, sb + nw);
        lifo.push_back({at, remaining});
      }
    }
  }
  const size_t n_b = reachable.size() / (size_t)nw;
  *out_B = (int32_t)n_b;
  if ((int64_t)n_b > cap || !out) return porrt_fail(ctx, PORRT_ERR_CAPACITY, "reachable_belief_states: cap too small");
  memcpy(out, reachable.data(), reachable.size() * 8);
  return PORRT_OK;
}

struct BeliefDev {
  const int64_t* row_ptr; const int32_t* col; const int32_t* edge_vid; const double* cost;
  const int32_t* node_vid; const int32_t* node_set;
  const uint8_t* compat;      // [B][n_validities]
  const int64_t* succ_ptr;    // [n_sets * B + 1]
  const int32_t* succ_belief; const double* succ_p;
  int64_t V; int32_t B, n_validities;
};

// node typing (pto.rs:209-255): Observation iff an observation edge to an EXISTING successor belief node exists,
// else Action iff some admissible geometric child exists, else Unknown.
__global__ void belief_type_kernel(BeliefDev g, uint8_t* __restrict__ type, const int32_t* __restrict__ colpos, uint8_t* __restrict__ type_cm) {
  const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= g.V * g.B) return;
  const int64_t n = t / g.B;
  const int b = (int)(t - n * g.B);
  const int32_t nv = g.node_vid[n];
  uint8_t ty = PORRT_NODE_UNKNOWN;
  if (g.compat[(int64_t)b * g.n_validities + nv]) {
    const int64_t sp = (int64_t)g.node_set[n] * g.B + b;
    for (int64_t k = g.succ_ptr[sp]; k < g.succ_ptr[sp + 1]; ++k)
      if (g.compat[(int64_t)g.succ_belief[k] * g.n_validities + nv]) { ty = PORRT_NODE_OBSERVATION; break; }
    if (ty == PORRT_NODE_UNKNOWN)
      for (int64_t e = g.row_ptr[n]; e < g.row_ptr[n + 1]; ++e)
        if (g.compat[(int64_t)b * g.n_validities + g.node_vid[g.col[e]]] && g.compat[(int64_t)b * g.n_validities + g.edge_vid[e]]) { ty = PORRT_NODE_ACTION; break; }
  } else {
    ty = 255;  // belief node does not exist (node_to_belief_nodes[id][belief] == None)
  }
  type[t] = ty;
  if (type_cm) type_cm[(int64_t)colpos[b] * g.V + n] = ty;   // colsolve.cu reads a belief's column along the nodes
}

// belief nodes that do not exist were typed 255 for the sweeps; the reference adds them anyway, typed Unknown (pto.rs:199)
__global__ void type_finish_kernel(uint8_t* __restrict__ type, int64_t n) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x)
    if (type[i] == 255) type[i] = PORRT_NODE_UNKNOWN;
}

// ---- belief columns through the frontier relaxation (sssp_frontier.cu): roadmaps whose column does not fit in shared memory.
// Initial values of the columns [c_lo, c_hi) of one level in the Morton-numbered table: +inf, 0 at the finals (already scattered),
// the Observation value  sum_k p_k * (0.0 + dist[n][succ_k])  (belief_graph.rs:125-135) from the finished columns; the sign bit on
// everything that is not an Action node (never relaxed).
__global__ void belief_level_init_kernel(int64_t V, int B, int c_lo, int c_hi, const uint32_t* __restrict__ order, const uint8_t* __restrict__ type_cm,
                                         const int32_t* __restrict__ nvid, const int32_t* __restrict__ node_set, const int32_t* __restrict__ col_belief,
                                         const int64_t* __restrict__ succ_ptr, const int32_t* __restrict__ succ_col, const double* __restrict__ succ_p,
                                         const uint64_t* __restrict__ cmask, double* __restrict__ table) {
  const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= (int64_t)(c_hi - c_lo) * V) return;
  const int c = c_lo + (int)(t / V);
  const int64_t pos = t - (int64_t)(c - c_lo) * V;
  if (col_belief[c] < 0) return;                       // padding column
  const int64_t n = order[pos];
  const uint8_t ty = type_cm[(int64_t)c * V + n];
  double v = table[(int64_t)c * V + pos];
  if (ty == PORRT_NODE_OBSERVATION) {
    const int32_t nv = nvid[n];
    const int64_t sp = (int64_t)node_set[n] * B + col_belief[c];
    double alt = 0.0;
    for (int64_t k = succ_ptr[sp]; k < succ_ptr[sp + 1]; ++k) {
      const int32_t cc = succ_col[k];
      if (!((cmask[(int64_t)cc * 4 + (nv >> 6)] >> (nv & 63)) & 1)) continue;   // successor belief node does not exist here
      alt = __dadd_rn(alt, __dmul_rn(succ_p[k], __dadd_rn(0.0, fabs(table[(int64_t)cc * V + pos]))));
    }
    if (alt < v) v = alt;
  }
  table[(int64_t)c * V + pos] = ty != PORRT_NODE_ACTION ? -v : v;
}
// finals: 0 in the Morton-numbered table; idx = column * V + node (caller's numbering)
__global__ void scatter_zero_perm_kernel(double* __restrict__ table, const int64_t* __restrict__ idx, int64_t n, const int32_t* __restrict__ perm, int64_t V) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const int64_t c = idx[i] / V, node = idx[i] - c * V;
  table[c * V + perm[node]] = 0.0;
}
// table (Morton numbering, signs) -> dist_cm[column][node]
__global__ void belief_unpermute_kernel(const double* __restrict__ table, const int32_t* __restrict__ perm, int64_t V, int64_t n_cols, double* __restrict__ dist_cm) {
  const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= n_cols * V) return;
  const int64_t c = t / V, n = t - c * V;
  dist_cm[t] = fabs(table[c * V + perm[n]]);
}

// dist_cm[colpos[b]][n] -> dist[n][b] through a 32 x 32 tile (both sides coalesced)
__global__ void __launch_bounds__(256) belief_untranspose_kernel(const double* __restrict__ dist_cm, int64_t ld, const int32_t* __restrict__ colpos,
                                                                 int64_t V, int B, double* __restrict__ dist) {
  __shared__ double tile[32][33];
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
  const int64_t n0 = (int64_t)blockIdx.x * 32;
  const int b0 = blockIdx.y * 32;
  for (int k = ty; k < 32; k += 8) {
    const int b = b0 + k;
    if (b < B && n0 + tx < V) tile[k][tx] = dist_cm[(int64_t)colpos[b] * ld + n0 + tx];
  }
  __syncthreads();
  for (int k = ty; k < 32; k += 8) {
    const int64_t n = n0 + k;
    if (n < V && b0 + tx < B) dist[n * B + b0 + tx] = tile[tx][k];
  }
}

// The whole V x B table of the last porrt_belief_vi on the host: into the ctx's pinned copy (R.dist / R.type) and, if given, the
// caller's buffers.  d_dist_nb: the [node][belief] table on the device (global sweeps), or null = bring the column solver's
// [column][node] table into that layout first.  The DMA runs in 8 pieces whose hand-over to the caller's buffer overlaps it.
static int32_t belief_download_full(porrt_ctx* ctx, const double* d_dist_nb, double* out_dist, uint8_t* out_type) {
  auto& R = ctx->bel;
  cudaStream_t st = ctx->stream;
  const int64_t V = R.V;
  const int B = R.B;
  const size_t nb = (size_t)V * B;
  if (!d_dist_nb) {
    CUDA_TRY(ctx, ctx->ws_table.ensure(nb * 8));
    double* d = ctx->ws_table.as<double>();
    belief_untranspose_kernel<<<dim3(div_up(V, 32), div_up(B, 32)), 256, 0, st>>>(R.d_dist_cm, V, R.d_colpos, V, B, d);
    LAUNCH_CHECK(ctx);
    d_dist_nb = d;
  }
  double* h_dist;
  uint8_t* h_type;
  CUDA_TRY(ctx, carve(ctx->pin_bel, [&](Carve& c) { h_dist = c.take<double>(nb); h_type = c.take<uint8_t>(nb); }));
  const int n_pieces = nb > (1u << 20) ? 8 : 1;
  for (int k = 0; k < n_pieces; ++k) {
    const size_t lo = nb * (size_t)k / (size_t)n_pieces, hi = nb * (size_t)(k + 1) / (size_t)n_pieces;
    CUDA_TRY(ctx, cudaMemcpyAsync(h_dist + lo, d_dist_nb + lo, (hi - lo) * 8, cudaMemcpyDeviceToHost, st));
    CUDA_TRY(ctx, cudaMemcpyAsync(h_type + lo, R.d_type + lo, hi - lo, cudaMemcpyDeviceToHost, st));
    CUDA_TRY(ctx, cudaEventRecord(ctx->ev_t[k], st));
  }
  const int nt = n_pieces > 1 && (out_dist || out_type) ? 4 : 1;
  std::vector<int> bad((size_t)nt, 0);
  auto hand_on = [&](int t) {
    for (int k = t; k < n_pieces; k += nt) {
      if (cudaEventSynchronize(ctx->ev_t[k]) != cudaSuccess) { bad[(size_t)t] = 1; return; }
      const size_t lo = nb * (size_t)k / (size_t)n_pieces, hi = nb * (size_t)(k + 1) / (size_t)n_pieces;
      if (out_dist) memcpy(out_dist + lo, h_dist + lo, (hi - lo) * 8);
      if (out_type) memcpy(out_type + lo, h_type + lo, hi - lo);
    }
  };
  if (nt == 1) hand_on(0);
  else {
    std::vector<std::thread> th;
    for (int t = 0; t < nt; ++t) th.emplace_back(hand_on, t);
    for (auto& t : th) t.join();
  }
  CUDA_TRY(ctx, cudaStreamSynchronize(st));
  for (int x : bad) if (x) return porrt_fail(ctx, PORRT_ERR_CUDA, "belief_vi: result copy failed");
  R.dist = h_dist; R.type = h_type; R.on_host = true;
  return PORRT_OK;
}

PORRT_API int32_t porrt_belief_vi(porrt_ctx* ctx, int64_t V, const int64_t* row_ptr, const int32_t* col, const int32_t* edge_vid,
                                  const double* xy, const int32_t* node_vid, const uint64_t* validities, int32_t n_validities,
                                  int32_t mask_words, int32_t n_worlds, const double* beliefs, int32_t B,
                                  const uint64_t* visible_zone_mask, const int32_t* finals_ids, const uint64_t* finals_masks,
                                  int32_t n_finals, double* out_dist, uint8_t* out_type, int32_t* out_sweeps, double* out_phase_ms) {
  CTX_CHECK(ctx);
  if (!ctx->has_map) return porrt_fail(ctx, PORRT_ERR_NO_MAP, "no map uploaded");
  if (V <= 0 || B <= 0 || !row_ptr || !xy || !node_vid || !validities || !beliefs || !visible_zone_mask || n_worlds != ctx->n_worlds ||
      mask_words != ctx->mask_words || n_validities <= 0 || (n_finals > 0 && (!finals_ids || !finals_masks)))
    return porrt_fail(ctx, PORRT_ERR_INVALID_ARG, "belief_vi: bad arguments");
  CUDA_TRY(ctx, cudaSetDevice(ctx->device));
  cudaStream_t st = ctx->stream;
  double t0 = now_ms(), t1, ph[4] = {0};
  const int64_t E = row_ptr[V];
  if (E > 0 && (!col || !edge_vid)) return porrt_fail(ctx, PORRT_ERR_INVALID_ARG, "belief_vi: null col/edge_vid");
  if (!csr_ok(V, row_ptr, col)) return porrt_fail(ctx, PORRT_ERR_INVALID_ARG, "belief_vi: malformed CSR (row_ptr not monotone or edge target out of range)");
  for (int64_t e = 0; e < E; ++e)
    if (edge_vid[e] < 0 || edge_vid[e] >= n_validities) return porrt_fail(ctx, PORRT_ERR_INVALID_ARG, "belief_vi: edge validity id out of range");
  for (int64_t u = 0; u < V; ++u)
    if (node_vid[u] < 0 || node_vid[u] >= n_validities) return porrt_fail(ctx, PORRT_ERR_INVALID_ARG, "belief_vi: node validity id out of range");
  const int nw = n_worlds;
  // compute_compatibility (common.rs:266-276)
  // is_compatible(belief, mask) (common.rs:256-264) = "no world with positive probability outside the mask": one AND-NOT per
  // word on the belief's support bits
  std::vector<uint64_t> support((size_t)B * mask_words, 0);
  for (int b = 0; b < B; ++b)
    for (int w = 0; w < nw; ++w)
      if (beliefs[(size_t)b * nw + w] > 0.0) support[(size_t)b * mask_words + w / 64] |= (uint64_t)1 << (w % 64);
  auto compatible = [&](int b, const uint64_t* mask) {
    for (int k = 0; k < mask_words; ++k)
      if (support[(size_t)b * mask_words + k] & ~mask[k]) return false;
    return true;
  };
  std::vector<uint8_t> compat((size_t)B * n_validities);
  for (int b = 0; b < B; ++b)
    for (int v = 0; v < n_validities; ++v) compat[(size_t)b * n_validities + v] = compatible(b, validities + (size_t)v * mask_words);
  // belief ids by hash (belief_graph.rs:75-87); collisions are a reference panic
  std::unordered_map<uint64_t, int> hash_to_id;
  std::vector<uint64_t> bhash(B);
  for (int b = 0; b < B; ++b) { bhash[b] = belief_hash(beliefs + (size_t)b * nw, nw); hash_to_id[bhash[b]] = b; }
  if ((int)hash_to_id.size() != B) return porrt_fail(ctx, PORRT_ERR_PANIC, "collision when hashing the belief states! (belief_graph.rs:84)");
  // observation successor tables, one per distinct set of visible zones (observe_impl is a function of that set only)
  std::map<uint64_t, int> set_index;
  std::vector<int32_t> node_set((size_t)V);
  std::vector<uint64_t> sets;
  const uint64_t zone_bits = ctx->n_zones >= 64 ? ~(uint64_t)0 : (((uint64_t)1 << ctx->n_zones) - 1);
  for (int64_t n = 0; n < V; ++n) {
    const uint64_t vis = visible_zone_mask[n] & zone_bits;
    auto it = set_index.find(vis);
    if (it == set_index.end()) { it = set_index.emplace(vis, (int)sets.size()).first; sets.push_back(vis); }
    node_set[n] = it->second;
  }
  // column order for colsolve.cu: beliefs sorted by the size of their support (observations only ever split it, so a column
  // reads Observation values from columns that come earlier), level by level
  std::vector<int32_t> level((size_t)B, 0), colpos((size_t)B), by_level((size_t)B);
  for (int b2 = 0; b2 < B; ++b2)
    for (int k = 0; k < mask_words; ++k) level[(size_t)b2] += __builtin_popcountll(support[(size_t)b2 * mask_words + k]);
  for (int b2 = 0; b2 < B; ++b2) by_level[(size_t)b2] = b2;
  std::stable_sort(by_level.begin(), by_level.end(), [&](int32_t x, int32_t y) { return level[(size_t)x] < level[(size_t)y]; });
  // Column positions.  On one GPU the columns of a level are simply consecutive.  With a communicator every level is cut into
  // `world` shards of EQUAL width (the last columns of a shard may be unused padding) so that the exchange after a level is one
  // plain ncclAllGather instead of a group of ragged broadcasts; rank r owns the columns [lo + r * per, lo + r * per + count_r).
  const int shards = ctx->comm_world > 1 ? ctx->comm_world : 1;
  struct Level { int lo, per, n_real; };
  std::vector<Level> levels;
  std::vector<int32_t> col_belief;   // belief of a column position, -1 = padding
  for (int c = 0; c < B;) {
    int e = c;
    while (e < B && level[(size_t)by_level[(size_t)e]] == level[(size_t)by_level[(size_t)c]]) ++e;
    const int n_real = e - c, per = (n_real + shards - 1) / shards, lo = (int)col_belief.size();
    col_belief.resize((size_t)lo + (size_t)per * shards, -1);
    for (int r = 0; r < shards; ++r) {
      int64_t a2, b2;
      comm_shard_range(n_real, r, shards, &a2, &b2);
      for (int64_t j = a2; j < b2; ++j) {
        const int pos = lo + r * per + (int)(j - a2);
        col_belief[(size_t)pos] = by_level[(size_t)(c + j)];
        colpos[(size_t)by_level[(size_t)(c + j)]] = pos;
      }
    }
    levels.push_back({lo, per, n_real});
    c = e;
  }
  const int Bp = (int)col_belief.size();   // columns incl. padding (== B on one GPU)
  // observation successor tables, one entry per (set, belief), built on the device (belief_tables.cu)
  BeliefSuccDev succ = {};
  {
    int32_t rc = belief_succ_tables(ctx, beliefs, B, nw, sets, bhash, level, colpos, &succ, st);
    if (rc) return rc;
  }
  // initial distances: 0 at final belief nodes (pto.rs:261-271), +inf elsewhere -- written on the device; only the list of final
  // belief nodes is built here (a host-side V*B table cost 30 ms + a 150 MB upload at B = 4095)
  std::vector<int64_t> zero_idx;
  for (int k = 0; k < n_finals; ++k) {
    const int32_t f = finals_ids[k];
    if (f < 0 || f >= V) return porrt_fail(ctx, PORRT_ERR_INVALID_ARG, "belief_vi: final id out of range");
    for (int b = 0; b < B; ++b)
      if (compat[(size_t)b * n_validities + node_vid[f]] && compatible(b, finals_masks + (size_t)k * mask_words))
        zero_idx.push_back((int64_t)f * B + b);
  }
  t1 = now_ms(); ph[0] = t1 - t0; t0 = t1;

  const bool cols = colsolve_fits(V, E, n_validities) && !ctx->force_global_sweeps && succ.levels_ok;
  const bool sharded = ctx->comm_world > 1;
  if (n_validities > 256) return porrt_fail(ctx, PORRT_ERR_UNSUPPORTED, "belief_vi: more than 256 validity ids");
  if (!succ.levels_ok) return porrt_fail(ctx, PORRT_ERR_UNSUPPORTED, "belief_vi: an observation does not split the belief's support (the level order of the backups does not apply)");
  std::vector<uint64_t> cmask((size_t)Bp * 4, 0);
  {
    for (int c = 0; c < Bp; ++c)
      for (int v = 0; col_belief[(size_t)c] >= 0 && v < n_validities; ++v)
        if (compat[(size_t)col_belief[(size_t)c] * n_validities + v]) cmask[(size_t)c * 4 + v / 64] |= (uint64_t)1 << (v % 64);
  }
  // final belief nodes as indices into the [column][node] table the backups run on
  for (int64_t& z : zero_idx) { const int64_t f = z / B; const int b2 = (int)(z % B); z = (int64_t)colpos[(size_t)b2] * V + f; }

  int64_t* d_row;
  double *d_cost, *d_xy, *d_cost_t;
  double* d_table_m = nullptr;   // frontier path: the table in Morton numbering, [column][pos]
  uint64_t* d_cmask;
  int32_t *d_col, *d_evid, *d_nvid, *d_nset, *d_col_belief, *d_changed;
  uint32_t *d_ce, *d_rs, *d_cursor;
  uint8_t* d_compat;
  int64_t* d_zero;
  CUDA_TRY(ctx, carve(ctx->ws_main, [&](Carve& c) {
    d_row = c.take<int64_t>(V + 1);
    d_cost = c.take<double>(E);
    d_xy = c.take<double>(2 * V);
    if (!cols) d_table_m = c.take<double>((size_t)V * Bp);
    d_cmask = c.take<uint64_t>((size_t)Bp * 4);
    d_col = c.take<int32_t>(E); d_evid = c.take<int32_t>(E);
    d_ce = c.take<uint32_t>(E); d_rs = c.take<uint32_t>(V + 1); d_cursor = c.take<uint32_t>(V + 1);
    d_cost_t = c.take<double>(E);
    d_nvid = c.take<int32_t>(V); d_nset = c.take<int32_t>(V); d_col_belief = c.take<int32_t>(Bp);
    d_changed = c.take<int32_t>(4);
    d_compat = c.take<uint8_t>(compat.size());
    d_zero = c.take<int64_t>(zero_idx.size() + 1);
  }));
  // the column solver's table ([column][node]), the node types and the column map outlive the call (lazy result, policy walk)
  auto& R = ctx->bel;
  R.V = 0; R.on_host = false;
  double* d_dist_cm;
  uint8_t *d_type, *d_type_cm;
  int32_t* d_colpos;
  CUDA_TRY(ctx, carve(R.dev, [&](Carve& c) {
    d_dist_cm = c.take<double>((size_t)V * Bp); d_type = c.take<uint8_t>((size_t)V * B); d_type_cm = c.take<uint8_t>((size_t)V * Bp);
    d_colpos = c.take<int32_t>(B);
  }));
  CUDA_TRY(ctx, cudaMemcpyAsync(d_row, row_ptr, (size_t)(V + 1) * 8, cudaMemcpyHostToDevice, st));
  if (E) {
    CUDA_TRY(ctx, cudaMemcpyAsync(d_col, col, (size_t)E * 4, cudaMemcpyHostToDevice, st));
    CUDA_TRY(ctx, cudaMemcpyAsync(d_evid, edge_vid, (size_t)E * 4, cudaMemcpyHostToDevice, st));
  }
  CUDA_TRY(ctx, cudaMemcpyAsync(d_xy, xy, (size_t)V * 16, cudaMemcpyHostToDevice, st));
  CUDA_TRY(ctx, cudaMemcpyAsync(d_nvid, node_vid, (size_t)V * 4, cudaMemcpyHostToDevice, st));
  CUDA_TRY(ctx, cudaMemcpyAsync(d_nset, node_set.data(), (size_t)V * 4, cudaMemcpyHostToDevice, st));
  CUDA_TRY(ctx, cudaMemcpyAsync(d_compat, compat.data(), compat.size(), cudaMemcpyHostToDevice, st));
  CUDA_TRY(ctx, cudaMemcpyAsync(d_colpos, colpos.data(), (size_t)B * 4, cudaMemcpyHostToDevice, st));
  CUDA_TRY(ctx, cudaMemcpyAsync(d_col_belief, col_belief.data(), (size_t)Bp * 4, cudaMemcpyHostToDevice, st));
  CUDA_TRY(ctx, cudaMemcpyAsync(d_cmask, cmask.data(), cmask.size() * 8, cudaMemcpyHostToDevice, st));
  SfGraph sfg = {};
  if (!cols) {   // Morton numbering + transposed adjacency with edge validity ids (sssp_frontier.cu)
    int32_t rc = sf_build_graph(ctx, d_row, d_col, d_evid, d_xy, V, E, &sfg, st);
    if (rc) return rc;
  }
  double* d_table = cols ? d_dist_cm : d_table_m;
  fill_inf_kernel<<<ctx->sm_count * 8, 256, 0, st>>>(d_table, V * (int64_t)Bp);
  LAUNCH_CHECK(ctx);
  if (!zero_idx.empty()) {
    CUDA_TRY(ctx, cudaMemcpyAsync(d_zero, zero_idx.data(), zero_idx.size() * 8, cudaMemcpyHostToDevice, st));
    if (cols) scatter_zero_kernel<<<div_up((int64_t)zero_idx.size(), 256), 256, 0, st>>>(d_table, d_zero, (int64_t)zero_idx.size());
    else scatter_zero_perm_kernel<<<div_up((int64_t)zero_idx.size(), 256), 256, 0, st>>>(d_table, d_zero, (int64_t)zero_idx.size(), sfg.perm, V);
    LAUNCH_CHECK(ctx);
  }
  edge_cost_kernel<<<div_up(V * 32, 256), 256, 0, st>>>(d_row, d_col, (const double2*)d_xy, V, d_cost);
  LAUNCH_CHECK(ctx);
  BeliefDev gd = {d_row, d_col, d_evid, d_cost, d_nvid, d_nset, d_compat, succ.succ_ptr, succ.succ_b, succ.succ_p, V, B, n_validities};
  const int blocks = div_up(V * (int64_t)B, 256);
  belief_type_kernel<<<blocks, 256, 0, st>>>(gd, d_type, d_colpos, d_type_cm);
  LAUNCH_CHECK(ctx);
  if (cols) {
    int32_t rc = colsolve_pack(ctx, d_row, d_col, d_evid, d_cost, V, E, d_rs, d_ce, d_cost_t, d_cursor, st);
    if (rc) return rc;
    CUDA_TRY(ctx, cudaMemsetAsync(d_changed, 0, 16, st));
  }
  CUDA_TRY(ctx, cudaStreamSynchronize(st));
  t1 = now_ms(); ph[1] = t1 - t0; t0 = t1;
  int sweeps = 0;
  if (cols) {
    // One launch per level; the CTAs of a level solve their columns on chip to the fixed point (colsolve.cu).  With a communicator
    // (SURVEY 8(f) rank 2) the columns of a level are sharded over the ranks and all-gathered before the next level reads them.
    ColSolveArgs ca = {};
    ca.row_start = d_rs; ca.cost = d_cost_t; ca.ce = d_ce; ca.V = (int32_t)V; ca.ld = V; ca.dist_cm = d_dist_cm; ca.cmask = d_cmask;
    ca.nvid = d_nvid; ca.type_cm = d_type_cm; ca.node_set = d_nset; ca.col_belief = d_col_belief; ca.succ_ptr = succ.succ_ptr;
    ca.succ_col = succ.succ_col; ca.succ_p = succ.succ_p; ca.B = B; ca.sweeps_out = d_changed;
    ca.offers_out = (unsigned long long*)(d_changed + 2);
    tstart(ctx);
    for (const Level& L : levels) {
      int64_t a2 = 0, b2 = L.n_real;
      if (sharded) comm_shard_range(L.n_real, ctx->comm_rank, ctx->comm_world, &a2, &b2);
      const int mine = L.lo + (sharded ? ctx->comm_rank * L.per : 0);
      int32_t rc = colsolve_level(ctx, ca, COLSOLVE_BELIEF, mine, mine + (int)(b2 - a2), st);
      if (rc) return rc;
      if (sharded) {
        std::vector<int64_t> off(ctx->comm_world + 1);
        for (int r = 0; r <= ctx->comm_world; ++r) off[r] = (int64_t)(L.lo + r * L.per) * V * 8;   // equal shards: one ncclAllGather
        rc = comm_all_gatherv_dev(ctx, nullptr, d_dist_cm, off.data(), st);
        if (rc) return rc;
      }
    }
    tmark(ctx);
    unsigned long long offers = 0;
    CUDA_TRY(ctx, cudaMemcpyAsync(&sweeps, d_changed, 4, cudaMemcpyDeviceToHost, st));
    CUDA_TRY(ctx, cudaMemcpyAsync(&offers, d_changed + 2, 8, cudaMemcpyDeviceToHost, st));
    CUDA_TRY(ctx, cudaStreamSynchronize(st));
    tfinish(ctx);   // porrt_ctx_last_phase_ms: [0] device ms of the column solver (all levels), [1] edge records it worked through
    ctx->last_ms[1] = (double)offers; ctx->n_last = 2;
  } else {
    // The same levels through the frontier relaxation over global memory (sssp_frontier.cu): a level's columns get their initial
    // values (finals, Observation values from the finished levels, sign bit on everything that is not an Action node) and are
    // relaxed together; shards and exchange as above.  The table is kept in Morton numbering until the end.
    double offers_total = 0.0;
    tstart(ctx);
    for (const Level& L : levels) {
      int64_t a2 = 0, b2 = L.n_real;
      if (sharded) comm_shard_range(L.n_real, ctx->comm_rank, ctx->comm_world, &a2, &b2);
      const int mine = L.lo + (sharded ? ctx->comm_rank * L.per : 0), n_mine = (int)(b2 - a2);
      if (n_mine > 0) {
        belief_level_init_kernel<<<div_up((int64_t)n_mine * V, 256), 256, 0, st>>>(V, B, mine, mine + n_mine, sfg.order, d_type_cm, d_nvid, d_nset,
                                                                                    d_col_belief, succ.succ_ptr, succ.succ_col, succ.succ_p, d_cmask, d_table_m);
        LAUNCH_CHECK(ctx);
        int32_t rounds = 0;
        double offers = 0.0;
        int32_t rc = sf_relax(ctx, sfg, d_table_m + (int64_t)mine * V, n_mine, d_cmask + (int64_t)mine * 4, &rounds, &offers, st);
        if (rc) return rc;
        sweeps = std::max(sweeps, (int)rounds);
        offers_total += offers;
      }
      if (sharded) {
        std::vector<int64_t> off(ctx->comm_world + 1);
        for (int r = 0; r <= ctx->comm_world; ++r) off[r] = (int64_t)(L.lo + r * L.per) * V * 8;
        int32_t rc = comm_all_gatherv_dev(ctx, nullptr, d_table_m, off.data(), st);
        if (rc) return rc;
      }
    }
    tmark(ctx);
    belief_unpermute_kernel<<<div_up((int64_t)Bp * V, 256), 256, 0, st>>>(d_table_m, sfg.perm, V, Bp, d_dist_cm);
    LAUNCH_CHECK(ctx);
    CUDA_TRY(ctx, cudaStreamSynchronize(st));
    tfinish(ctx);
    ctx->last_ms[1] = offers_total; ctx->n_last = 2;
  }
  t1 = now_ms(); ph[2] = t1 - t0; t0 = t1;
  // results: retained for porrt_extract_policy / porrt_belief_result; to the caller if asked for
  R.V = V; R.B = B; R.n_worlds = nw; R.n_validities = n_validities;
  R.row_ptr.assign(row_ptr, row_ptr + V + 1);
  R.col.assign(col, col + E); R.edge_vid.assign(edge_vid, edge_vid + E);
  R.xy.assign(xy, xy + 2 * V);
  R.beliefs.assign(beliefs, beliefs + (size_t)B * nw);
  R.node_obs_set = node_set; R.compat = compat;
  R.succ_ptr.resize(sets.size() * (size_t)B + 1); R.succ_belief.resize((size_t)succ.n_succ);   // the policy walk reads them on the host
  CUDA_TRY(ctx, cudaMemcpyAsync(R.succ_ptr.data(), succ.succ_ptr, R.succ_ptr.size() * 8, cudaMemcpyDeviceToHost, st));
  if (succ.n_succ) CUDA_TRY(ctx, cudaMemcpyAsync(R.succ_belief.data(), succ.succ_b, (size_t)succ.n_succ * 4, cudaMemcpyDeviceToHost, st));
  type_finish_kernel<<<ctx->sm_count * 8, 256, 0, st>>>(d_type, V * (int64_t)B);
  LAUNCH_CHECK(ctx);
  R.d_dist_cm = d_dist_cm; R.d_type_cm = d_type_cm; R.d_type = d_type; R.d_colpos = d_colpos;
  R.colpos = colpos;
  R.col_dist.assign((size_t)B, std::vector<double>()); R.col_type.assign((size_t)B, std::vector<uint8_t>());
  R.dist = nullptr; R.type = nullptr;
  R.node_vid.assign(node_vid, node_vid + V);
  if (out_dist || out_type) {
    int32_t rc = belief_download_full(ctx, nullptr, out_dist, out_type);
    if (rc) return rc;
  } else {
    CUDA_TRY(ctx, cudaStreamSynchronize(st));
  }
  if (out_sweeps) *out_sweeps = sweeps;
  t1 = now_ms(); ph[3] = t1 - t0;
  if (out_phase_ms) memcpy(out_phase_ms, ph, sizeof(ph));
  return PORRT_OK;
}

// The retained table of the last porrt_belief_vi (pinned host memory owned by the ctx, valid until the next call): the
// reference's own FFI hands results out the same way (pointer getters over handle-owned vectors, pto_c.rs:255-270).
PORRT_API int32_t porrt_belief_result(porrt_ctx* ctx, const double** out_dist, const uint8_t** out_type, int64_t* out_V, int32_t* out_B) {
  CTX_CHECK(ctx);
  if (ctx->bel.V <= 0) return porrt_fail(ctx, PORRT_ERR_INVALID_ARG, "belief_result: run porrt_belief_vi first");
  if (!ctx->bel.on_host) {   // the table is still on the device only: bring it over now
    CUDA_TRY(ctx, cudaSetDevice(ctx->device));
    const int32_t rc = belief_download_full(ctx, nullptr, nullptr, nullptr);
    if (rc) return rc;
  }
  if (out_dist) *out_dist = ctx->bel.dist;
  if (out_type) *out_type = ctx->bel.type;
  if (out_V) *out_V = ctx->bel.V;
  if (out_B) *out_B = ctx->bel.B;
  return PORRT_OK;
}

bool porrt_ctx::BeliefState_::fetch_column(porrt_ctx* ctx, int b) {
  std::vector<double>& d = col_dist[(size_t)b];
  std::vector<uint8_t>& t = col_type[(size_t)b];
  d.resize((size_t)V); t.resize((size_t)V);
  const size_t at = (size_t)colpos[(size_t)b] * V;
  if (cudaSetDevice(ctx->device) == cudaSuccess &&
      cudaMemcpyAsync(d.data(), d_dist_cm + at, (size_t)V * 8, cudaMemcpyDeviceToHost, ctx->stream) == cudaSuccess &&
      cudaMemcpyAsync(t.data(), d_type_cm + at, (size_t)V, cudaMemcpyDeviceToHost, ctx->stream) == cudaSuccess &&
      cudaStreamSynchronize(ctx->stream) == cudaSuccess)
    return true;
  d.clear(); t.clear();
  fetch_failed = true;
  return false;
}

// ================================================================================================ policy extraction
PORRT_API int32_t porrt_extract_policy(porrt_ctx* ctx, int32_t* out_node, int32_t* out_belief, int32_t* out_parent,
                                       uint8_t* out_is_leaf, int64_t cap, int64_t* out_n, double* out_expected_cost) {
  CTX_CHECK(ctx);
  auto& R = ctx->bel;
  if (R.V <= 0) return porrt_fail(ctx, PORRT_ERR_INVALID_ARG, "extract_policy: run porrt_belief_vi first");
  const int B = R.B;
  // the walk over the implicit V x B belief graph; an Observation child keeps its parent's state, so its cost is norm2(state n, state n)
  R.fetch_failed = false;
  std::vector<PolicyNode> pol;
  const int32_t rc = get_best_expected_children(
      ctx, "extract_policy", R.V * (int64_t)B, R.beliefs.data(), R.n_worlds,
      [&](int64_t id, auto&& fn) { R.for_children(ctx, id, fn); },
      [&](int64_t id) { return (int32_t)(id % B); },
      [&](int64_t a, int64_t c) { return norm2(&R.xy[2 * (size_t)(a / B)], &R.xy[2 * (size_t)(c / B)], 2); },
      [&](int64_t id) { return R.value(ctx, id); }, pol);
  const double expected_cost = R.value(ctx, 0);
  // a failed fetch read as 0: it outranks any assert the walk tested on such a value
  if (R.fetch_failed) return porrt_fail(ctx, PORRT_ERR_CUDA, "extract_policy: fetching a value column failed");
  if (rc) return rc;
  if (out_n) *out_n = (int64_t)pol.size();
  if (out_expected_cost) *out_expected_cost = expected_cost;
  if ((int64_t)pol.size() > cap || !out_node || !out_belief || !out_parent || !out_is_leaf) return porrt_fail(ctx, PORRT_ERR_CAPACITY, "extract_policy: cap too small");
  for (size_t k = 0; k < pol.size(); ++k) {
    out_node[k] = (int32_t)(pol[k].id / B); out_belief[k] = (int32_t)(pol[k].id % B); out_parent[k] = pol[k].parent; out_is_leaf[k] = pol[k].leaf;
  }
  return PORRT_OK;
}
