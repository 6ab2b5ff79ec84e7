// colsolve.cu -- value backups as shared-memory resident COLUMN problems.
//
// Reference: dijkstra over a PTOGraphWorldView (pto_graph.rs:245-303; one problem per world in plan_qmdp,
// qmdp_policy_extractor.rs:23-35) and conditional_dijkstra over the belief graph (belief_graph.rs:89-182).
//
// Both value tables are made of columns -- dist[.][world] resp. dist[.][belief] -- that are single-source-set shortest path
// problems on the SAME roadmap (V nodes, E edges, a few thousand nodes in BASELINE configs 2-4):
//   * a world's column relaxes node u only if u is valid in that world (PTOGraphWorldView::parents filters by the parent node);
//   * a belief's column relaxes its Action nodes over the edges admissible under the belief (pto.rs:235-255); its Observation
//     nodes hold  sum_k p_k * (0.0 + dist[n][succ_k])  (belief_graph.rs:125-135), which only reads columns of strictly more
//     informed beliefs (observe() splits the support), i.e. a value that is FINAL before the column starts when the columns are
//     processed level by level (level = size of the belief's support).
// A column of V doubles fits in shared memory (227 KB: up to 6 columns of a 4.7 k-node roadmap), so one CTA solves C columns
// completely on chip with a label-correcting worklist: a node whose value improved pushes it to its parents (12-byte records of
// the transposed adjacency, read from L2) with shared-memory atomicMin, rounds until no node is dirty.  No kernel launch, no
// global barrier and no HBM/L2 gather of dist per sweep, and work only where values move -- round 1's thread-per-(node, column)
// Jacobi sweeps re-evaluated the whole table 40-80 times.  graph.cu's value-column driver runs it one level at a time.
// Measured on the config-4 shape (4685 nodes x 4095 beliefs, 12 levels): Jacobi sweeps 43 ms -> pull sweeps on chip 20 ms
// (54 sweeps, issue/latency bound; sweeping the nodes sorted along x / y did not cut the sweeps: a CTA has 256 nodes in flight,
// wider than a hop) -> push worklist 10.6 ms -> dirty nodes collected into a CTA-wide queue per round 5.3 ms.
// dist is the greatest fixed point of a monotone operator (fp +, *, min are monotone; every backup keeps the reference's operand
// order), so the schedule does not change a single bit of the result (SURVEY 8(g) note 5).
//
// Encoding inside shared memory: a value with the SIGN BIT set is fixed (Observation / Unknown / non-existent belief nodes, nodes
// that are invalid in the world): it is read through |.| (free operand modifier of DADD) and never relaxed.
#include <algorithm>

#include "common.cuh"
#include "colsolve.cuh"

namespace {

template <int C>
__device__ __forceinline__ void lds_cols(const double* p, double (&out)[C]) {
  if constexpr (C == 1) {
    out[0] = p[0];
  } else {
#pragma unroll
    for (int j = 0; j < C; j += 2) {
      const double2 t = *reinterpret_cast<const double2*>(p + j);
      out[j] = t.x; out[j + 1] = t.y;
    }
  }
}

// One CTA = columns [col_lo + blockIdx.x * C, +C) of the level [col_lo, col_hi).
// COLSOLVE_BELIEF: relaxable iff type == ACTION, edge admissible iff the column's validity mask holds the edge's validity id.
// COLSOLVE_WORLD : relaxable iff the column's validity mask holds the NODE's validity id, every edge admissible.
// Worklist (push) relaxation: only nodes whose value changed do work.  dirty[v] = columns of v that improved since v last pushed.
// A 4-lane group takes a dirty node v, clears its mask, and offers  norm2(u, v) + dist[v]  to every parent u (transposed
// adjacency; norm2 is symmetric bit for bit) with a 64-bit atomicMin in shared memory (non-negative doubles order like their bit
// patterns); an improvement marks u dirty.  Fixed entries carry the sign bit, i.e. compare below every offer, and are never written.
// The fixed point is the one of the pull sweeps: every value ever stored is the reference's left-to-right sum along some
// admissible path, and the final value of v is always pushed after v's last improvement.
// The kernel's whole body, shared with the batched kernel below (one CTA works on the roadmap whose arguments `a` are).
template <int C, int MODE>
__device__ __forceinline__ void colsolve_push_body(const ColSolveArgs& a, int col_lo, int col_hi) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  double* sd = reinterpret_cast<double*>(smem_raw);                 // [V][C]
  uint8_t* s_adm = smem_raw + (size_t)a.V * C * 8;                  // [256]
  uint32_t* s_dirty = reinterpret_cast<uint32_t*>(s_adm + 256);     // [ceil(V / 4)] one byte per node
  uint16_t* s_queue = reinterpret_cast<uint16_t*>(s_dirty + (a.V + 3) / 4);   // [COLSOLVE_QCAP] dirty nodes of this round
  unsigned* s_qn = reinterpret_cast<unsigned*>(s_queue + COLSOLVE_QCAP);
  const int tid = threadIdx.x;
  const int V = a.V;
  const int c0 = col_lo + blockIdx.x * C;
  const int nc = min(C, col_hi - c0);
  const int nthr = (int)blockDim.x;

  if (tid < 256) {
    unsigned bits = 0;
    if (MODE == COLSOLVE_WORLD) bits = 0xff;
    else
      for (int j = 0; j < nc; ++j) bits |= (unsigned)((a.cmask[(size_t)(c0 + j) * 4 + (tid >> 6)] >> (tid & 63)) & 1) << j;
    s_adm[tid] = (uint8_t)bits;
  }
  for (int i = tid; i < (V + 3) / 4; i += nthr) s_dirty[i] = 0;
  if (tid < 2) s_qn[tid] = 0;
  __syncthreads();
  for (int j = 0; j < C; ++j) {
    if (j >= nc) {
      for (int n = tid; n < V; n += nthr) sd[(size_t)n * C + j] = -INFINITY;
      continue;
    }
    const int cpos = c0 + j;
    const double* gcol = a.dist_cm + (size_t)cpos * a.ld;
    for (int n = tid; n < V; n += nthr) {
      double v = gcol[n];
      bool fixed;
      if (MODE == COLSOLVE_BELIEF) {
        const uint8_t ty = a.type_cm[(size_t)cpos * V + n];
        fixed = ty != PORRT_NODE_ACTION;
        if (ty == PORRT_NODE_OBSERVATION) {
          const int32_t nv = a.nvid[n];
          const int64_t sp = (int64_t)a.node_set[n] * a.B + a.col_belief[cpos];
          double alt = 0.0;
          for (int64_t k = a.succ_ptr[sp]; k < a.succ_ptr[sp + 1]; ++k) {
            const int32_t cc = a.succ_col[k];
            if (!((a.cmask[(size_t)cc * 4 + (nv >> 6)] >> (nv & 63)) & 1)) continue;
            alt = __dadd_rn(alt, __dmul_rn(a.succ_p[k], __dadd_rn(0.0, a.dist_cm[(size_t)cc * a.ld + n])));
          }
          if (alt < v) v = alt;
        }
      } else {
        const int32_t nv = a.nvid ? a.nvid[n] : 0;
        fixed = !((a.cmask[(size_t)cpos * 4 + (nv >> 6)] >> (nv & 63)) & 1);
      }
      sd[(size_t)n * C + j] = fixed ? -v : v;
      if (v < INFINITY) atomicOr(&s_dirty[n >> 2], (1u << j) << ((n & 3) * 8));   // sources: finals and finite Observation values
    }
  }
  __syncthreads();

  const int lane = tid & 31, warp = tid >> 5, nwarp = nthr >> 5;
  const int l = tid % COLSOLVE_LANES, grp = tid / COLSOLVE_LANES, ngrp = nthr / COLSOLVE_LANES;
  const unsigned gmask = ((1u << COLSOLVE_LANES) - 1u) << (lane & ~(COLSOLVE_LANES - 1));
  const uint8_t* dirty8 = reinterpret_cast<const uint8_t*>(s_dirty);
  const int nblk = (V + 31) / 32;
  int rounds = 0;
  unsigned n_offers = 0;   // edge records this thread worked through (measurement: bytes actually read from L2)
  for (;;) {
    // ---- collect: the dirty nodes go to a queue so that the groups of the whole CTA share them evenly (a warp that worked off
    // its own 32-node blocks one after the other paid the L2 latency chain of every block in turn).  Nodes that do not fit stay
    // dirty for the next round; the scan start rotates so that no node waits forever.
    unsigned* qn_ptr = s_qn + (rounds & 1);   // two counters: the other one is reset while this one is in use
    bool found = false;
    const int rot = (rounds * 7) % nblk;
    for (int bi = warp; bi < nblk; bi += nwarp) {
      int blk = bi + rot;
      if (blk >= nblk) blk -= nblk;
      const int n = blk * 32 + lane;
      const bool d = n < V && dirty8[n] != 0;
      const unsigned todo = __ballot_sync(0xffffffffu, d);
      if (!todo) continue;
      found = true;
      int slot = 0;
      if (lane == 0) slot = (int)atomicAdd(qn_ptr, (unsigned)__popc(todo));
      slot = __shfl_sync(0xffffffffu, slot, 0) + __popc(todo & ((1u << lane) - 1u));
      if (d && slot < COLSOLVE_QCAP) s_queue[slot] = (uint16_t)n;
    }
    ++rounds;
    if (!__syncthreads_or(found)) break;
    const int qn = min((int)*qn_ptr, COLSOLVE_QCAP);
    if (tid == 0) s_qn[rounds & 1] = 0;
    // ---- push
    for (int qi = grp; qi < qn; qi += ngrp) {
      {
        const int v = s_queue[qi];
        unsigned m = 0;
        if (l == 0) m = (atomicAnd(&s_dirty[v >> 2], ~(0xffu << ((v & 3) * 8))) >> ((v & 3) * 8)) & 0xffu;
        m = __shfl_sync(gmask, m, lane & ~(COLSOLVE_LANES - 1));
        __threadfence_block();   // the values are read after the mask was taken: a later improvement marks v again
        double dv[C];
        lds_cols<C>(sd + (size_t)v * C, dv);
        const uint32_t e1 = a.row_start[v + 1];
        // the chain  mask -> row -> records -> parents' values  is latency bound (small frontiers, records in L2): every lane
        // first issues the loads of its next COLSOLVE_UNROLL records, then works through them
        for (uint32_t e0 = a.row_start[v] + l; e0 < e1; e0 += COLSOLVE_LANES * COLSOLVE_UNROLL) {
          uint32_t ce_r[COLSOLVE_UNROLL];
          double cost_r[COLSOLVE_UNROLL];
#pragma unroll
          for (int q = 0; q < COLSOLVE_UNROLL; ++q) {
            const uint32_t e = e0 + q * COLSOLVE_LANES;
            ce_r[q] = e < e1 ? __ldg(a.ce + e) : 0xffffffffu;
            cost_r[q] = e < e1 ? __ldg(a.cost + e) : 0.0;
          }
#pragma unroll
          for (int q = 0; q < COLSOLVE_UNROLL; ++q) {
            const uint32_t ce = ce_r[q];
            if (ce == 0xffffffffu) break;
            ++n_offers;
            const double cost = cost_r[q];
            const unsigned adm = (MODE == COLSOLVE_WORLD ? 0xffu : s_adm[ce >> 16]) & m;
            if (!adm) continue;
            const int u = (int)(ce & 0xffffu);
            double du[C];
            lds_cols<C>(sd + (size_t)u * C, du);
            unsigned mark = 0;
#pragma unroll
            for (int j = 0; j < C; ++j) {
              const double alt = __dadd_rn(cost, fabs(dv[j]));   // norm2(u, v) + dist[v]
              if (((adm >> j) & 1) && alt < du[j]) {
                const unsigned long long old = atomicMin(reinterpret_cast<unsigned long long*>(sd + (size_t)u * C + j),
                                                         (unsigned long long)__double_as_longlong(alt));
                if ((unsigned long long)__double_as_longlong(alt) < old) mark |= 1u << j;
              }
            }
            if (mark) atomicOr(&s_dirty[u >> 2], mark << ((u & 3) * 8));
          }
        }
      }
    }
    __syncthreads();   // marks and the reset counter are visible to the next round's scan
  }
  for (int j = 0; j < nc; ++j) {
    double* gcol = a.dist_cm + (size_t)(c0 + j) * a.ld;
    for (int n = tid; n < V; n += nthr) gcol[n] = fabs(sd[(size_t)n * C + j]);
  }
  if (tid == 0 && a.sweeps_out) atomicMax(a.sweeps_out, rounds);
  if (a.offers_out) {
    for (int sft = 16; sft > 0; sft >>= 1) n_offers += __shfl_xor_sync(0xffffffffu, n_offers, sft);
    if (lane == 0) atomicAdd(a.offers_out, (unsigned long long)n_offers);
  }
}

template <int C, int MODE>
__global__ void __launch_bounds__(COLSOLVE_THREADS, 1) colsolve_push_kernel(ColSolveArgs a, int col_lo, int col_hi) {
  colsolve_push_body<C, MODE>(a, col_lo, col_hi);
}

// Belief columns of several roadmaps in one launch: blockIdx.y picks the roadmap, whose arguments the kernel reads from a device
// array of descriptors (the level's columns and the belief tables are the same for all of them; graph.cu, porrt_pto_plan_batch).
template <int C>
__global__ void __launch_bounds__(COLSOLVE_THREADS, 1) colsolve_push_batch_kernel(const ColSolveArgs* __restrict__ descs, int col_lo, int col_hi) {
  colsolve_push_body<C, COLSOLVE_BELIEF>(descs[blockIdx.y], col_lo, col_hi);
}

__global__ void colsolve_count_kernel(const int32_t* __restrict__ col, int64_t E, uint32_t* __restrict__ cnt) {
  const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (e < E) atomicAdd(&cnt[col[e]], 1u);
}
// exclusive scan of cnt[0..V) into start[0..V], one CTA (V <= 65535); cnt becomes the fill cursor (= start)
__global__ void __launch_bounds__(1024) colsolve_scan_kernel(uint32_t* __restrict__ cnt, int V, uint32_t* __restrict__ start) {
  __shared__ uint32_t part[1024];
  const int per = (V + 1023) / 1024;
  const int lo = min(V, (int)threadIdx.x * per), hi = min(V, lo + per);
  uint32_t s = 0;
  for (int i = lo; i < hi; ++i) s += cnt[i];
  part[threadIdx.x] = s;
  __syncthreads();
  for (int d = 1; d < 1024; d <<= 1) {
    const uint32_t add = threadIdx.x >= d ? part[threadIdx.x - d] : 0;
    __syncthreads();
    part[threadIdx.x] += add;
    __syncthreads();
  }
  uint32_t run = part[threadIdx.x] - s;
  for (int i = lo; i < hi; ++i) { const uint32_t c = cnt[i]; start[i] = run; cnt[i] = run; run += c; }
  if (threadIdx.x == 1023) start[V] = part[1023];
}
// transposed records: row v lists (parent u | validity id of u -> v << 16, norm2(u, v)); one warp per row u of the forward CSR
__global__ void colsolve_fill_kernel(const int64_t* __restrict__ row_ptr, const int32_t* __restrict__ col, const int32_t* __restrict__ evid,
                                     const double* __restrict__ cost, int64_t V, uint32_t* __restrict__ cursor,
                                     uint32_t* __restrict__ ce_t, double* __restrict__ cost_t) {
  const int lane = threadIdx.x & 31;
  const int64_t u = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  if (u >= V) return;
  for (int64_t e = row_ptr[u] + lane; e < row_ptr[u + 1]; e += 32) {
    const uint32_t pos = atomicAdd(&cursor[col[e]], 1u);
    ce_t[pos] = (uint32_t)u | ((evid ? (uint32_t)evid[e] : 0u) << 16);
    cost_t[pos] = cost[e];
  }
}

template <int C, int MODE>
cudaError_t launch_one(const porrt_ctx* ctx, const ColSolveArgs& a, int col_lo, int col_hi, size_t smem, cudaStream_t st) {
  static bool configured[16] = {};   // per instantiation and device: the attribute holds for the current device only
  if (!configured[ctx->device & 15]) {
    cudaError_t e = cudaFuncSetAttribute(colsolve_push_kernel<C, MODE>, cudaFuncAttributeMaxDynamicSharedMemorySize, COLSOLVE_SMEM_MAX);
    if (e != cudaSuccess) return e;
    configured[ctx->device & 15] = true;
  }
  const int n_cta = (col_hi - col_lo + C - 1) / C;
  colsolve_push_kernel<C, MODE><<<n_cta, COLSOLVE_THREADS, smem, st>>>(a, col_lo, col_hi);
  return cudaGetLastError();
}
}  // namespace

bool colsolve_fits(int64_t V, int64_t E, int32_t n_validities) {
  return V > 0 && V <= 65535 && E < ((int64_t)1 << 32) && n_validities <= 256 && (size_t)V * 9 + 280 + COLSOLVE_QCAP * 2 <= COLSOLVE_SMEM_MAX;
}

// Transposed adjacency for the push kernel: row_start_t[V + 1], ce_t[E], cost_t[E]; cursor_tmp[V + 1] is work space.
int32_t colsolve_pack(porrt_ctx* ctx, const int64_t* row_ptr_dev, const int32_t* col_dev, const int32_t* evid_dev, const double* cost_dev,
                      int64_t V, int64_t E, uint32_t* row_start_t, uint32_t* ce_t, double* cost_t, uint32_t* cursor_tmp, cudaStream_t st) {
  CUDA_TRY(ctx, cudaMemsetAsync(cursor_tmp, 0, (size_t)(V + 1) * 4, st));
  if (E > 0) {
    colsolve_count_kernel<<<div_up(E, 256), 256, 0, st>>>(col_dev, E, cursor_tmp);
    LAUNCH_CHECK(ctx);
  }
  colsolve_scan_kernel<<<1, 1024, 0, st>>>(cursor_tmp, (int)V, row_start_t);
  LAUNCH_CHECK(ctx);
  if (E > 0) {
    colsolve_fill_kernel<<<div_up(V * 32, 256), 256, 0, st>>>(row_ptr_dev, col_dev, evid_dev, cost_dev, V, cursor_tmp, ce_t, cost_t);
    LAUNCH_CHECK(ctx);
  }
  return PORRT_OK;
}

// Solves the columns [col_lo, col_hi) (one level: they do not depend on each other).  Columns per CTA: as many as fit, but no more
// than needed to give every SM a CTA.
int32_t colsolve_level(porrt_ctx* ctx, const ColSolveArgs& a, int mode, int col_lo, int col_hi, cudaStream_t st) {
  const int n = col_hi - col_lo;
  if (n <= 0) return PORRT_OK;
  const int cap = (int)((COLSOLVE_SMEM_MAX - 280 - COLSOLVE_QCAP * 2 - (size_t)a.V) / ((size_t)a.V * 8));
  const int cmax = cap >= 6 ? 6 : cap >= 4 ? 4 : cap >= 2 ? 2 : 1;
  const int waves = (n + cmax * ctx->sm_count - 1) / (cmax * ctx->sm_count);
  const int want = (n + waves * ctx->sm_count - 1) / (waves * ctx->sm_count);   // columns per CTA that fill `waves` waves
  const int C = want <= 1 ? 1 : want <= 2 ? 2 : want <= 4 ? 4 : 6;
  const int Cc = std::min(C, cmax);
  const size_t smem = (size_t)a.V * Cc * 8 + 256 + (size_t)((a.V + 3) / 4) * 4 + COLSOLVE_QCAP * 2 + 16;
  cudaError_t e;
  if (mode == COLSOLVE_BELIEF) {
    switch (Cc) {
      case 1: e = launch_one<1, COLSOLVE_BELIEF>(ctx, a, col_lo, col_hi, smem, st); break;
      case 2: e = launch_one<2, COLSOLVE_BELIEF>(ctx, a, col_lo, col_hi, smem, st); break;
      case 4: e = launch_one<4, COLSOLVE_BELIEF>(ctx, a, col_lo, col_hi, smem, st); break;
      default: e = launch_one<6, COLSOLVE_BELIEF>(ctx, a, col_lo, col_hi, smem, st); break;
    }
  } else {
    switch (Cc) {
      case 1: e = launch_one<1, COLSOLVE_WORLD>(ctx, a, col_lo, col_hi, smem, st); break;
      case 2: e = launch_one<2, COLSOLVE_WORLD>(ctx, a, col_lo, col_hi, smem, st); break;
      case 4: e = launch_one<4, COLSOLVE_WORLD>(ctx, a, col_lo, col_hi, smem, st); break;
      default: e = launch_one<6, COLSOLVE_WORLD>(ctx, a, col_lo, col_hi, smem, st); break;
    }
  }
  ctx->launches += 1;
  CUDA_TRY(ctx, e);
  return PORRT_OK;
}

// colsolve_level for the belief columns [col_lo, col_hi) of n_roads roadmaps at once (descs_dev: their arguments, device): a grid of
// (CTAs per roadmap, roadmaps).  Columns per CTA and shared memory are what colsolve_level chooses for one roadmap of the largest
// V of the launch, V_max nodes; the roadmaps side by side fill the SMs where one roadmap's level cannot.
int32_t colsolve_level_batch(porrt_ctx* ctx, const ColSolveArgs* descs_dev, int n_roads, int32_t V_max, int col_lo, int col_hi,
                             cudaStream_t st) {
  const int n = col_hi - col_lo;
  if (n <= 0 || n_roads <= 0) return PORRT_OK;
  const int cap = (int)((COLSOLVE_SMEM_MAX - 280 - COLSOLVE_QCAP * 2 - (size_t)V_max) / ((size_t)V_max * 8));
  const int cmax = cap >= 6 ? 6 : cap >= 4 ? 4 : cap >= 2 ? 2 : 1;
  const int waves = (n + cmax * ctx->sm_count - 1) / (cmax * ctx->sm_count);
  const int want = (n + waves * ctx->sm_count - 1) / (waves * ctx->sm_count);
  const int C = std::min(want <= 1 ? 1 : want <= 2 ? 2 : want <= 4 ? 4 : 6, cmax);
  const size_t smem = (size_t)V_max * C * 8 + 256 + (size_t)((V_max + 3) / 4) * 4 + COLSOLVE_QCAP * 2 + 16;
  static bool configured[4][16] = {};   // per instantiation and device
  const int ci = C == 1 ? 0 : C == 2 ? 1 : C == 4 ? 2 : 3;
  const dim3 grid((unsigned)((n + C - 1) / C), (unsigned)n_roads);
  auto launch = [&](auto kernel) -> cudaError_t {
    if (!configured[ci][ctx->device & 15]) {
      const cudaError_t e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, COLSOLVE_SMEM_MAX);
      if (e != cudaSuccess) return e;
      configured[ci][ctx->device & 15] = true;
    }
    kernel<<<grid, COLSOLVE_THREADS, smem, st>>>(descs_dev, col_lo, col_hi);
    return cudaGetLastError();
  };
  cudaError_t e;
  switch (C) {
    case 1: e = launch(colsolve_push_batch_kernel<1>); break;
    case 2: e = launch(colsolve_push_batch_kernel<2>); break;
    case 4: e = launch(colsolve_push_batch_kernel<4>); break;
    default: e = launch(colsolve_push_batch_kernel<6>); break;
  }
  ctx->launches += 1;
  CUDA_TRY(ctx, e);
  return PORRT_OK;
}
