// nn_tile.cu -- nearest-neighbour search over TMA-staged vertex tiles (SURVEY.md 8(a) rows B2/B3 + the k-NN metric).
//
// Replaces, batched, KdTree::nearest_neighbors[_filtered] / nearest_neighbor[_filtered] (reference
// src/nearest_neighbor.rs:48-126).  nn.cu's first version ran one thread per query straight on the cell-sorted
// vertex array in global memory: every query re-read the ~9 cells around it through L1/L2 (124 candidates x 16 B at the
// c5 shape) and k-NN kept its candidate list in local memory.  Here
//   * the QUERIES are binned by grid cell as well (count / scan / scatter), so the queries of a run of NT_W cells of
//     one cell row form a contiguous slice;
//   * a CTA takes such a tile, and the vertices any of its queries can reach -- three cell rows x (NT_W + 2) cells,
//     i.e. three CONTIGUOUS ranges of the cell-sorted arrays -- are staged in shared memory by bulk-async copies
//     (cp.async.bulk, mbarrier byte-count completion): each vertex is fetched once per tile instead of once per query;
//   * every query is owned by one THREAD of the tile's CTA, which walks its (<= 3) candidate runs in shared memory; k-NN
//     keeps its k best in shared memory too (column layout, conflict-free).  Warp-per-query variants (ballot-compacted
//     hit lists; a warp-wide sorted list) cost 2-10x the instructions per candidate -- see the notes at the kernels.
// Distances are the reference's f64 arithmetic (common.rs:203-213) and `sqrt(d2) <= r` is evaluated as d2 <= T(r).
// Queries whose radius reaches beyond the neighbouring cells, tiles whose candidates exceed the staging buffer and k-NN
// queries that need a wider ring go to nn.cu's thread-per-query kernels (exact ring search) through an index list.
#include <algorithm>

#include "nn_dev.cuh"

#define NT_W 8               // cells per tile along x
#define NT_THREADS 128
#define NT_CAP 2048          // staged vertices per tile (radius): 32 KiB + 8 KiB ids
#define NT_CAP_KNN 768       // k-NN: leaves room for the per-thread lists

__device__ __forceinline__ uint32_t nt_smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void nt_mbar_init(uint64_t* bar) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(nt_smem_u32(bar)));
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void nt_mbar_expect(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(nt_smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void nt_bulk_g2s(void* dst, const void* src, uint32_t bytes, uint64_t* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(nt_smem_u32(dst)), "l"(src),
               "r"(bytes), "r"(nt_smem_u32(bar))
               : "memory");
}
__device__ __forceinline__ void nt_mbar_wait0(uint64_t* bar) {
  uint32_t done = 0;
  while (!done)
    asm volatile("{ .reg .pred p; mbarrier.try_wait.parity.shared::cta.b64 p, [%1], 0; selp.u32 %0, 1, 0, p; }"
                 : "=r"(done) : "r"(nt_smem_u32(bar)) : "memory");
}

// ------------------------------------------------------------------------------------------------ query binning
// qcell[t] = cell of query t if the tile path can serve it, -1 -> fallback list, -2 -> no result at all (NaN, r < 0)
template <bool KNN>
__global__ void nt_bin_kernel(GridDev g, const double2* __restrict__ q, const double* __restrict__ radius, int64_t m,
                              int32_t* __restrict__ qcell, int32_t* __restrict__ qcount, int32_t* __restrict__ fb_list, int32_t* __restrict__ fb_n) {
  const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= m) return;
  const double2 p = q[t];
  int32_t c = -2;
  if (p.x == p.x && p.y == p.y) {
    const int cx = cell_coord(p.x, g.org_x, g.inv_cell, g.cells_x), cy = cell_coord(p.y, g.org_y, g.inv_cell, g.cells_y);
    bool ok = true, any = true;
    if (!KNN) {
      const double r = radius[t];
      any = radius_threshold(r) >= 0.0;
      const double rr = isinf(r) ? r : __dadd_rn(__dmul_rn(r, 1.000000001), 1e-300);  // the same conservative cell cover as nn.cu
      const int cx0 = cell_coord(p.x - rr, g.org_x, g.inv_cell, g.cells_x), cx1 = cell_coord(p.x + rr, g.org_x, g.inv_cell, g.cells_x);
      const int cy0 = cell_coord(p.y - rr, g.org_y, g.inv_cell, g.cells_y), cy1 = cell_coord(p.y + rr, g.org_y, g.inv_cell, g.cells_y);
      ok = cx0 >= cx - 1 && cx1 <= cx + 1 && cy0 >= cy - 1 && cy1 <= cy + 1;
    }
    if (any) {
      if (ok) { c = cy * g.cells_x + cx; atomicAdd(&qcount[c], 1); }
      else { c = -1; fb_list[atomicAdd(fb_n, 1)] = (int32_t)t; }
    }
  } else if (KNN) { c = -1; fb_list[atomicAdd(fb_n, 1)] = (int32_t)t; }   // nn.cu writes the "nothing found" record
  qcell[t] = c;
}

__global__ void nt_scatter_kernel(const int32_t* __restrict__ qcell, int64_t m, const int64_t* __restrict__ qstart,
                                  int32_t* __restrict__ cursor, int32_t* __restrict__ qorder) {
  const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= m) return;
  const int32_t c = qcell[t];
  if (c >= 0) qorder[qstart[c] + atomicAdd(&cursor[c], 1)] = (int32_t)t;
}

// ------------------------------------------------------------------------------------------------ tile staging
struct Tile {
  int cy, cxa, cxb;          // query cells: row cy, columns cxa..cxb
  int ca;                    // first staged column
  int64_t qa; int nq;        // slice of qorder
  int64_t k0[3]; int len[3]; // staged vertex ranges of rows cy-1, cy, cy+1 (len 0: row outside the grid)
  int xoff[3], ioff[3];      // their offsets in s_xy / s_id (ids keep their 16-byte phase: element j at ioff + j)
  bool staged;
};

__device__ __forceinline__ Tile tile_setup(const GridDev& g, const int64_t* __restrict__ qstart, int tiles_per_row, int cap) {
  Tile T;
  const int tile = blockIdx.x;
  T.cy = tile / tiles_per_row;
  T.cxa = (tile % tiles_per_row) * NT_W;
  T.cxb = min(T.cxa + NT_W - 1, g.cells_x - 1);
  T.qa = qstart[(int64_t)T.cy * g.cells_x + T.cxa];
  T.nq = (int)(qstart[(int64_t)T.cy * g.cells_x + T.cxb + 1] - T.qa);
  T.ca = max(T.cxa - 1, 0);
  const int cb = min(T.cxb + 1, g.cells_x - 1);
  int tot = 0, itot = 0;
  for (int r = 0; r < 3; ++r) {
    const int row = T.cy - 1 + r;
    T.k0[r] = 0; T.len[r] = 0;
    if (T.nq > 0 && row >= 0 && row < g.cells_y) {
      T.k0[r] = g.cell_start[(int64_t)row * g.cells_x + T.ca];
      T.len[r] = (int)min((int64_t)0x3fffffff, g.cell_start[(int64_t)row * g.cells_x + cb + 1] - T.k0[r]);
    }
    T.xoff[r] = tot; tot += T.len[r];
    T.ioff[r] = itot + (int)(T.k0[r] & 3);                       // copy starts at the 16-byte boundary below k0
    itot += (((int)(T.k0[r] & 3) + T.len[r] + 3) & ~3);
  }
  T.staged = tot <= cap;
  return T;
}

// thread 0 issues the bulk copies; everybody waits for the bytes to land
__device__ __forceinline__ void tile_stage(const GridDev& g, const Tile& T, double2* s_xy, int32_t* s_id, uint64_t* bar) {
  if (threadIdx.x == 0) nt_mbar_init(bar);
  __syncthreads();
  if (T.staged) {
    if (threadIdx.x == 0) {
      uint32_t bytes = 0;
      for (int r = 0; r < 3; ++r)
        if (T.len[r] > 0) bytes += (uint32_t)T.len[r] * 16u + (uint32_t)((((int)(T.k0[r] & 3) + T.len[r] + 3) & ~3) * 4);
      nt_mbar_expect(bar, bytes);
      for (int r = 0; r < 3; ++r)
        if (T.len[r] > 0) {
          nt_bulk_g2s(s_xy + T.xoff[r], g.vxy + T.k0[r], (uint32_t)T.len[r] * 16u, bar);
          const int ph = (int)(T.k0[r] & 3);
          nt_bulk_g2s(s_id + T.ioff[r] - ph, g.vid + (T.k0[r] - ph), (uint32_t)(((ph + T.len[r] + 3) & ~3) * 4), bar);
        }
    }
    nt_mbar_wait0(bar);
  }
}

// ------------------------------------------------------------------------------------------------ radius: one pass
// Round 1 ran the candidates twice (count pass, fill pass), let every thread store its hits one 4-byte word at a time (32 partial
// sectors per store instruction: 400 of the 660 us) and restored the id order afterwards with a register sorting network
// (another 660 us).  Now ONE kernel looks at every candidate once and the order costs almost nothing:
//   S  all queries of one grid cell share their candidates -- the 3 x 3 cells around it, nine id-ascending runs of the staged
//      arrays.  Per query CELL (not per query) the CTA merges those runs into one id-ascending candidate list: a thread per
//      candidate, rank = position in its own run + lower_bound in the other eight (binary searches in shared memory);
//   A  thread per query: walk the cell's merged list, keep the hits' list positions in a per-thread row of shared memory --
//      they come out id-ascending by construction (a prefix limit even ends the walk early);
//   C  warp per 32 queries: one atomicAdd reserves the warp's slots of a staging buffer, then the lanes write each query's ids
//      side by side (128-byte lines instead of 32 partial sectors per store).
// A second, pure copy kernel moves the lists to their CSR places once the global scan of the counts is known.
// The kernel is persistent (as many CTAs as fit an SM, each striding over the tiles) and stages each tile into ONE buffer: 37 KiB,
// 6 CTAs per SM whose other warps cover the copy, 0.545 ms for the whole query at V = Q = 1e6.  Double-buffered (the next tile's
// bulk copies in flight on a second mbarrier) it needs 55 KiB, fits 4 CTAs per SM and takes 0.58 ms; one buffer with 5 CTAs per
// SM 0.57-0.60 ms (interleaved A/B on one box).  More resident warps beat the explicit prefetch here.
// Queries whose list would not fit (> NR_LCAP hits), cells with more than NR_CCAP candidates, tiles too dense to stage and warps
// that find the staging buffer full are appended to the fallback list and answered by nn.cu's thread-per-query kernels -- same
// bits, only slower.
#define NR_THREADS 128
#define NR_CAP 704           // staged vertices per tile: 11 KiB + 3 KiB ids (c5 shape: ~440 per tile)
#define NR_CCAP 176          // merged candidates per query cell (3 x 3 cells; c5 shape: 131 +- 11)
#define NR_LCAP 80           // hits per query kept in the thread's row
#define NR_LSTRIDE 84        // bytes per row (list positions fit a byte): 21 words, odd -> the lanes' rows fall into different banks
#define NR_CTAS_PER_SM 6
#define NR_RUNS 9
#define NR_SMEM (NR_CAP * 16 + (NR_CAP + 24) * 4 + NT_W * NR_CCAP * 2 + NT_W * NR_CCAP * 6 + NR_THREADS * NR_LSTRIDE)

__device__ __forceinline__ void nt_mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(nt_smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void nt_mbar_wait(uint64_t* bar, uint32_t parity) {
  uint32_t done = 0;
  while (!done)
    asm volatile("{ .reg .pred p; mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2; selp.u32 %0, 1, 0, p; }"
                 : "=r"(done) : "r"(nt_smem_u32(bar)), "r"(parity) : "memory");
}

__device__ __forceinline__ Tile tile_setup_at(const GridDev& g, const int64_t* __restrict__ qstart, int tiles_per_row, int cap, int tile) {
  Tile T;
  T.cy = tile / tiles_per_row;
  T.cxa = (tile % tiles_per_row) * NT_W;
  T.cxb = min(T.cxa + NT_W - 1, g.cells_x - 1);
  T.qa = qstart[(int64_t)T.cy * g.cells_x + T.cxa];
  T.nq = (int)(qstart[(int64_t)T.cy * g.cells_x + T.cxb + 1] - T.qa);
  T.ca = max(T.cxa - 1, 0);
  const int cb = min(T.cxb + 1, g.cells_x - 1);
  int tot = 0, itot = 0;
  for (int r = 0; r < 3; ++r) {
    const int row = T.cy - 1 + r;
    T.k0[r] = 0; T.len[r] = 0;
    if (T.nq > 0 && row >= 0 && row < g.cells_y) {
      T.k0[r] = g.cell_start[(int64_t)row * g.cells_x + T.ca];
      T.len[r] = (int)min((int64_t)0x3fffffff, g.cell_start[(int64_t)row * g.cells_x + cb + 1] - T.k0[r]);
    }
    T.xoff[r] = tot; tot += T.len[r];
    T.ioff[r] = itot + (int)(T.k0[r] & 3);
    itot += (((int)(T.k0[r] & 3) + T.len[r] + 3) & ~3);
  }
  T.staged = tot <= cap;
  return T;
}

struct NrRun { uint16_t xy0, id0, len, pad; };   // one cell's slice of the staged arrays: coordinates from xy0, ids from id0

// ---- the merge scripts (built once per vertex set, lazily, by nn_tile_build_scripts)
// All queries of a grid cell share their candidates: the 3 x 3 cells around it, nine id-ascending runs of the cell-sorted
// arrays.  Their merge into ONE id-ascending list depends on the vertex set alone, so it is computed once per cell and kept as a
// script: entry j = (run << 12) | position-in-run of the j-th smallest id.  2 bytes per candidate (~18 B per vertex) instead of
// nine binary searches per candidate and query batch (measured: 44 % of the kernel's instructions when done on the fly).
// Cells with more than NR_CCAP candidates get no script (their queries go to the thread-per-query kernel).
__global__ void nbr_size_kernel(GridDev g, int32_t* __restrict__ sizes) {
  const int64_t c = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= (int64_t)g.cells_x * g.cells_y) return;
  const int cx = (int)(c % g.cells_x), cy = (int)(c / g.cells_x);
  int n = 0;
  for (int r = -1; r <= 1; ++r) {
    const int row = cy + r;
    if (row < 0 || row >= g.cells_y) continue;
    const int c0 = max(cx - 1, 0), c1 = min(cx + 1, g.cells_x - 1);
    n += (int)(g.cell_start[(int64_t)row * g.cells_x + c1 + 1] - g.cell_start[(int64_t)row * g.cells_x + c0]);
  }
  sizes[c] = n <= NR_CCAP ? ((n + 7) & ~7) : 0;          // padded to 16 bytes: the scripts are staged by bulk copies
}

__global__ void __launch_bounds__(256) nbr_script_kernel(GridDev g, const int64_t* __restrict__ nbr_start, uint16_t* __restrict__ script) {
  const int lane = threadIdx.x & 31;
  const int64_t c = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;    // one warp per cell
  if (c >= (int64_t)g.cells_x * g.cells_y) return;
  if (nbr_start[c + 1] == nbr_start[c]) return;
  const int cx = (int)(c % g.cells_x), cy = (int)(c / g.cells_x);
  int64_t rs[NR_RUNS]; int rl[NR_RUNS]; int P[NR_RUNS + 1];
  P[0] = 0;
#pragma unroll
  for (int k = 0; k < NR_RUNS; ++k) {
    const int row = cy - 1 + k / 3, col = cx - 1 + k % 3;
    rs[k] = 0; rl[k] = 0;
    if (row >= 0 && row < g.cells_y && col >= 0 && col < g.cells_x) {
      rs[k] = g.cell_start[(int64_t)row * g.cells_x + col];
      rl[k] = (int)(g.cell_start[(int64_t)row * g.cells_x + col + 1] - rs[k]);
    }
    P[k + 1] = P[k] + rl[k];
  }
  uint16_t* out = script + nbr_start[c];
  for (int e = lane; e < P[NR_RUNS]; e += 32) {
    int k = 0;
#pragma unroll
    for (int j = 1; j < NR_RUNS; ++j) k += (e >= P[j]) ? 1 : 0;
    int pos = e;
    int64_t own = rs[0];
#pragma unroll
    for (int j = 1; j < NR_RUNS; ++j) if (j == k) { pos = e - P[j]; own = rs[j]; }
    const int32_t id = g.vid[own + pos];
    int rank = pos;
#pragma unroll
    for (int j = 0; j < NR_RUNS; ++j) {
      if (j == k) continue;
      int lo = 0, hi = rl[j];
      while (lo < hi) {
        const int mid = (lo + hi) >> 1;
        if (g.vid[rs[j] + mid] < id) lo = mid + 1; else hi = mid;
      }
      rank += lo;
    }
    out[rank] = (uint16_t)((k << 12) | pos);
  }
}

__global__ void __launch_bounds__(NR_THREADS) nt_radius_collect_kernel(
    GridDev g, const double2* __restrict__ q, const double* __restrict__ radius, const uint32_t* __restrict__ prefix,
    const uint64_t* __restrict__ reach, const uint32_t* __restrict__ world, const int32_t* __restrict__ qorder,
    const int64_t* __restrict__ qstart, const int64_t* __restrict__ nbr_start, const uint16_t* __restrict__ script, int tiles_per_row,
    int n_tiles, int32_t* __restrict__ counts, int64_t* __restrict__ stg_off, int32_t* __restrict__ staging,
    unsigned long long* __restrict__ stg_cursor, int64_t stg_cap, int32_t* __restrict__ fb_list, int32_t* __restrict__ fb_n) {
  extern __shared__ __align__(128) unsigned char nr_smem[];
  double2* const s_xy = (double2*)nr_smem;                     // the staging buffer: coordinates | ids | merge scripts
  int32_t* const s_id = (int32_t*)(s_xy + NR_CAP);
  uint16_t* const s_sc = (uint16_t*)(s_id + NR_CAP + 24);
  int32_t* s_cid = (int32_t*)(s_sc + NT_W * NR_CCAP);          // [NT_W][NR_CCAP] merged candidate ids ...
  uint16_t* s_cxy = (uint16_t*)(s_cid + NT_W * NR_CCAP);       // [NT_W][NR_CCAP] ... and where their coordinates are staged
  uint8_t* s_lst = (uint8_t*)(s_cxy + NT_W * NR_CCAP);         // [NR_THREADS][NR_LSTRIDE] list positions of a query's hits
  __shared__ uint64_t s_bar;
  __shared__ NrRun s_run[NT_W][NR_RUNS];
  __shared__ int32_t s_ccnt[NT_W];                             // merged candidates of a query cell; -1: no script (fallback)
  __shared__ int32_t s_coff[NT_W + 1];                         // where the cells' scripts start in the staged script range
  const int tid = threadIdx.x, lane = tid & 31;
  if (tid == 0) nt_mbar_init(&s_bar);
  __syncthreads();
  uint8_t* lst = s_lst + tid * NR_LSTRIDE;
  // thread 0: one phase of s_bar per tile -- the bulk copies of the tile's three vertex ranges and of its cells' scripts
  auto stage = [&](const Tile& T) {
    uint32_t bytes = 0, sc_bytes = 0;
    const int64_t ca = (int64_t)T.cy * g.cells_x + T.cxa, cb = (int64_t)T.cy * g.cells_x + T.cxb;
    if (T.staged && T.nq > 0) {
      for (int r = 0; r < 3; ++r)
        if (T.len[r] > 0) bytes += (uint32_t)T.len[r] * 16u + (uint32_t)((((int)(T.k0[r] & 3) + T.len[r] + 3) & ~3) * 4);
      sc_bytes = (uint32_t)(nbr_start[cb + 1] - nbr_start[ca]) * 2u;
    }
    if (bytes == 0) { nt_mbar_arrive(&s_bar); return; }
    nt_mbar_expect(&s_bar, bytes + sc_bytes);
    for (int r = 0; r < 3; ++r)
      if (T.len[r] > 0) {
        nt_bulk_g2s(s_xy + T.xoff[r], g.vxy + T.k0[r], (uint32_t)T.len[r] * 16u, &s_bar);
        const int ph = (int)(T.k0[r] & 3);
        nt_bulk_g2s(s_id + T.ioff[r] - ph, g.vid + (T.k0[r] - ph), (uint32_t)(((ph + T.len[r] + 3) & ~3) * 4), &s_bar);
      }
    if (sc_bytes) nt_bulk_g2s(s_sc, script + nbr_start[ca], sc_bytes, &s_bar);
  };
  int it = 0;
  for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x, ++it) {
    const Tile T = tile_setup_at(g, qstart, tiles_per_row, NR_CAP, tile);
    if (tid == 0) stage(T);
    nt_mbar_wait(&s_bar, (uint32_t)(it & 1));
    const int n_qc = (T.nq > 0 && T.staged) ? T.cxb - T.cxa + 1 : 0;
    // ---- S: the nine runs of every query cell, then its merged candidate list by the cell's script
    if (tid < n_qc * NR_RUNS) {
      const int qc = tid / NR_RUNS, k = tid % NR_RUNS, r = k / 3, cx = T.cxa + qc - 1 + (k % 3), row = T.cy - 1 + r;
      NrRun R = {0, 0, 0, 0};
      if (cx >= 0 && cx < g.cells_x && row >= 0 && row < g.cells_y) {
        const int64_t cs = g.cell_start[(int64_t)row * g.cells_x + cx], ce = g.cell_start[(int64_t)row * g.cells_x + cx + 1];
        const int64_t k0 = r == 0 ? T.k0[0] : (r == 1 ? T.k0[1] : T.k0[2]);      // (selects: a runtime index would put T in local memory)
        const int xoff = r == 0 ? T.xoff[0] : (r == 1 ? T.xoff[1] : T.xoff[2]);
        const int ioff = r == 0 ? T.ioff[0] : (r == 1 ? T.ioff[1] : T.ioff[2]);
        R.xy0 = (uint16_t)(xoff + (int)(cs - k0));
        R.id0 = (uint16_t)(ioff + (int)(cs - k0));
        R.len = (uint16_t)min((int64_t)0xffff, ce - cs);
      }
      s_run[qc][k] = R;
    } else if (tid >= 96 && tid - 96 <= n_qc && n_qc > 0) {
      const int64_t ca = (int64_t)T.cy * g.cells_x + T.cxa;
      s_coff[tid - 96] = (int)(nbr_start[ca + (tid - 96)] - nbr_start[ca]);
    }
    __syncthreads();
    if (tid < n_qc) {
      int n_c = 0;
#pragma unroll
      for (int k = 0; k < NR_RUNS; ++k) n_c += s_run[tid][k].len;
      s_ccnt[tid] = (s_coff[tid + 1] - s_coff[tid] >= n_c && n_c <= NR_CCAP) ? n_c : -1;   // no script: too many candidates
    }
    __syncthreads();
    for (int qc = 0; qc < n_qc; ++qc) {
      const int n_c = s_ccnt[qc];
      const uint16_t* sc = s_sc + s_coff[qc];
      for (int e = tid; e < n_c; e += NR_THREADS) {
        const uint32_t code = sc[e];
        const NrRun R = s_run[qc][code >> 12];
        const int pos = (int)(code & 0xfffu);
        s_cid[qc * NR_CCAP + e] = s_id[R.id0 + pos];
        s_cxy[qc * NR_CCAP + e] = (uint16_t)(R.xy0 + pos);
      }
    }
    __syncthreads();
    for (int q0 = 0; q0 < T.nq; q0 += NR_THREADS) {
      // ---- A: collect
      const int qi = q0 + tid;
      int32_t t = -1;
      int cnt = 0, qc = 0;
      bool fallback = false;
      if (qi < T.nq) {
        t = qorder[T.qa + qi];
        const double2 p = q[t];
        qc = cell_coord(p.x, g.org_x, g.inv_cell, g.cells_x) - T.cxa;      // the cell it was binned by
        if (!T.staged || s_ccnt[qc] < 0) fallback = true;
        else {
          const double Tr = radius_threshold(radius[t]);
          const uint32_t limit = prefix ? prefix[t] : 0xffffffffu;
          const uint32_t wq = (reach && world) ? world[t] : 0u;
          const uint16_t* cxy = s_cxy + qc * NR_CCAP;
          const int32_t* cid = s_cid + qc * NR_CCAP;
          const int n_c = s_ccnt[qc];
          // ids ascend along the list, so do the hits.  Branch-free body, four candidates in flight: the loop is bound by the
          // latency of its dependent shared-memory loads (index -> coordinates), not by issue
          auto keep = [&](int j, bool hit) {
            if (hit) { lst[min(cnt, NR_LCAP - 1)] = (uint8_t)j; ++cnt; }      // (overflow is caught by cnt > NR_LCAP below)
          };
          int j = 0;
          if (!reach) {
            for (; j + 4 <= n_c; j += 4) {
              const double d0 = dist2(s_xy[cxy[j]], p.x, p.y), d1 = dist2(s_xy[cxy[j + 1]], p.x, p.y);
              const double d2 = dist2(s_xy[cxy[j + 2]], p.x, p.y), d3 = dist2(s_xy[cxy[j + 3]], p.x, p.y);
              const uint32_t i0 = (uint32_t)cid[j], i1 = (uint32_t)cid[j + 1], i2 = (uint32_t)cid[j + 2], i3 = (uint32_t)cid[j + 3];
              keep(j, d0 <= Tr && i0 < limit); keep(j + 1, d1 <= Tr && i1 < limit);
              keep(j + 2, d2 <= Tr && i2 < limit); keep(j + 3, d3 <= Tr && i3 < limit);
            }
            for (; j < n_c; ++j) keep(j, dist2(s_xy[cxy[j]], p.x, p.y) <= Tr && (uint32_t)cid[j] < limit);
          } else {
            for (; j < n_c; ++j)
              keep(j, dist2(s_xy[cxy[j]], p.x, p.y) <= Tr && (uint32_t)cid[j] < limit && reach_bit(reach, g.reach_words, cid[j], wq));
          }
          if (cnt > NR_LCAP) fallback = true;
        }
        if (fallback) cnt = 0;
      }
      // ---- C: the warp reserves its slots and writes its 32 lists side by side
      int incl = cnt;
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) {
        const int v = __shfl_up_sync(0xffffffffu, incl, o);
        if (lane >= o) incl += v;
      }
      const int warp_total = __shfl_sync(0xffffffffu, incl, 31);
      long long base = 0;
      if (lane == 0 && warp_total > 0) base = (long long)atomicAdd(stg_cursor, (unsigned long long)warp_total);
      base = __shfl_sync(0xffffffffu, base, 0);
      const bool room = base + warp_total <= stg_cap;   // (warp-uniform) a full staging buffer sends the warp's queries to the fallback
      const long long mine = base + incl - cnt;
      if (t >= 0) {
        if (fallback || (!room && cnt > 0)) fb_list[atomicAdd(fb_n, 1)] = t;
        else { counts[t] = cnt; stg_off[t] = cnt > 0 ? mine : 0; }
      }
      if (room && warp_total > 0) {
        const unsigned have = __ballot_sync(0xffffffffu, cnt > 0);
        for (unsigned left = have; left; left &= left - 1) {
          const int j = __ffs(left) - 1;
          const int n_j = __shfl_sync(0xffffffffu, cnt, j);
          const long long o_j = __shfl_sync(0xffffffffu, mine, j);
          const int qc_j = __shfl_sync(0xffffffffu, qc, j);
          const uint8_t* l_j = s_lst + ((tid & ~31) + j) * NR_LSTRIDE;
          const int32_t* cid = s_cid + qc_j * NR_CCAP;
          int32_t* dst = staging + o_j;
          if (lane < n_j) dst[lane] = cid[l_j[lane]];
          if (lane + 32 < n_j) dst[lane + 32] = cid[l_j[lane + 32]];
          if (lane + 64 < n_j) dst[lane + 64] = cid[l_j[lane + 64]];
        }
      }
      __syncwarp();                                    // the rows are rewritten by the next chunk of queries
    }
    __syncthreads();                                   // everybody is done with this buffer and the merged lists
  }
}

// the lists leave the staging buffer for their CSR places: a warp takes four queries at a time (their loads are all in flight
// before the first store), lists side by side in 128-byte lines
__global__ void __launch_bounds__(256) nt_radius_place_kernel(const int32_t* __restrict__ staging, const int64_t* __restrict__ stg_off,
                                                              const int64_t* __restrict__ offsets, int64_t m, int32_t* __restrict__ out_ids) {
  const int lane = threadIdx.x & 31;
  const int64_t warp = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int64_t n_warps = ((int64_t)gridDim.x * blockDim.x) >> 5;
  for (int64_t t0 = warp * 4; t0 < m; t0 += n_warps * 4) {
    int64_t so = -1, o = 0, oe = 0;
    if (lane < 4 && t0 + lane < m) { so = stg_off[t0 + lane]; o = offsets[t0 + lane]; oe = offsets[t0 + lane + 1]; }
    int32_t v[4][3];
    int64_t oo[4]; int nn[4];
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      const int64_t s_u = __shfl_sync(0xffffffffu, so, u);
      oo[u] = __shfl_sync(0xffffffffu, o, u);
      nn[u] = s_u < 0 ? 0 : (int)(__shfl_sync(0xffffffffu, oe, u) - oo[u]);   // so < 0: answered by the thread-per-query kernels
#pragma unroll
      for (int c = 0; c < 3; ++c) v[u][c] = (lane + 32 * c < nn[u]) ? staging[s_u + lane + 32 * c] : 0;
    }
#pragma unroll
    for (int u = 0; u < 4; ++u) {
#pragma unroll
      for (int c = 0; c < 3; ++c) if (lane + 32 * c < nn[u]) out_ids[oo[u] + lane + 32 * c] = v[u][c];
      if (nn[u] > 96) {                                   // (NR_LCAP <= 96 today; kept general)
        const int64_t s_u = __shfl_sync(0xffffffffu, so, u);
        for (int k = 96 + lane; k < nn[u]; k += 32) out_ids[oo[u] + k] = staging[s_u + k];
      }
    }
  }
}

// ------------------------------------------------------------------------------------------------ 1-NN / k-NN: thread per query
// k = 1: running minimum (+ the number of vertices at exactly the winning d2, nn.cu: knn_kernel<1>).
// k > 1: a sorted list kept by insertion was measured first (1.75 ms for 1e6 queries, k = 16): lanes insert at different
// candidates, so the warp pays the insertion loop at almost every candidate.  Now two uniform passes over the candidates:
//   pass 1 bins d2 into NT_BINS equal-width bins (equal area: candidates are ~uniform in d2) in a per-thread byte
//          histogram and finds the first bin where the cumulative count reaches k;
//   pass 2 collects the candidates of the bins up to that one (k + a few) into the thread's list, which is then
//          insertion-sorted by (d2, id) and cut at k.
// Exact: both passes evaluate the same expression per candidate; a query is finished here only if its k-th best is
// provably closer than anything outside the 3 x 3 cells (ring_lower_bound2, R = 1), otherwise -- or if its list overflows
// (> k + NT_SLACK candidates in the bins, e.g. many exact duplicates) -- it goes to nn.cu's exact ring search.
// dynamic shared memory: [ s_xy NT_CAP_KNN | s_id NT_CAP_KNN + 24 | list cap x NT_THREADS (u16 codes)
//                          | histogram NT_BINS x NT_THREADS (u8) ],  cap = k + NT_SLACK
#define NT_BINS 32
#define NT_SLACK 16
__global__ void __launch_bounds__(NT_THREADS) nt_knn_kernel(GridDev g, const double2* __restrict__ q, int k,
                                                            const uint64_t* __restrict__ reach, const uint32_t* __restrict__ world,
                                                            const int32_t* __restrict__ qorder, const int64_t* __restrict__ qstart,
                                                            int tiles_per_row, int32_t* __restrict__ out_ids, double* __restrict__ out_dist,
                                                            int32_t* __restrict__ out_ties, int32_t* __restrict__ fb_list, int32_t* __restrict__ fb_n) {
  extern __shared__ __align__(128) unsigned char nt_smem[];
  const int cap = k + NT_SLACK;
  double2* s_xy = (double2*)nt_smem;
  int32_t* s_id = (int32_t*)(nt_smem + (size_t)NT_CAP_KNN * 16);
  uint16_t* s_lst = (uint16_t*)(s_id + NT_CAP_KNN + 24);
  uint8_t* s_hist = (uint8_t*)(s_lst + (size_t)cap * NT_THREADS);
  __shared__ uint64_t s_bar;
  const Tile T = tile_setup(g, qstart, tiles_per_row, NT_CAP_KNN);
  if (T.nq == 0) return;
  tile_stage(g, T, s_xy, s_id, &s_bar);
  uint16_t* lst = s_lst + threadIdx.x; // column layout: entry j of this thread at [j * NT_THREADS]
  uint8_t* hist = s_hist + threadIdx.x;
  // bins cover d2 in [0, (1.5 cell)^2): whatever lies beyond cannot be certified by the R = 1 bound anyway (<= 2 cells)
  const double bin_scale = (double)NT_BINS / (2.25 * g.cell * g.cell);
  for (int qi = threadIdx.x; qi < T.nq; qi += NT_THREADS) {
    const int32_t t = qorder[T.qa + qi];
    const double2 p = q[t];
    const uint32_t wq = (reach && world) ? world[t] : 0u;
    const int cx = cell_coord(p.x, g.org_x, g.inv_cell, g.cells_x);
    const int cx0 = max(cx - 1, 0), cx1 = min(cx + 1, g.cells_x - 1);
    // the query's candidate runs (rows cy-1, cy, cy+1)
    const double2* rx[3]; const int32_t* ri[3]; int rn[3];
#pragma unroll
    for (int rr3 = 0; rr3 < 3; ++rr3) {
      const int row = T.cy - 1 + rr3;
      rn[rr3] = 0; rx[rr3] = s_xy; ri[rr3] = s_id;
      if (row >= 0 && row < g.cells_y) {
        const int64_t s = g.cell_start[(int64_t)row * g.cells_x + cx0], e = g.cell_start[(int64_t)row * g.cells_x + cx1 + 1];
        const int s_run = (int)(s - T.k0[rr3]);
        rn[rr3] = (int)(e - s);
        rx[rr3] = T.staged ? s_xy + T.xoff[rr3] + s_run : g.vxy + s;
        ri[rr3] = T.staged ? s_id + T.ioff[rr3] + s_run : g.vid + s;
      }
    }
    bool done = false;
    if (k == 1) {
      int cnt = 0, ties = 0;
      double best = INFINITY;
      int32_t best_id = 0x7fffffff;
#pragma unroll
      for (int rr3 = 0; rr3 < 3; ++rr3)
        for (int j = 0; j < rn[rr3]; ++j) {
          const double d = dist2(rx[rr3][j], p.x, p.y);
          if (d != d || (cnt != 0 && d > best)) continue;
          const int32_t id = ri[rr3][j];
          if (reach && !reach_bit(reach, g.reach_words, id, wq)) continue;
          if (cnt == 0 || d < best) ties = 1; else ++ties;       // here d == best
          if (cnt == 0 || d < best || id < best_id) { best = d; best_id = id; }
          cnt = 1;
        }
      if (cnt == 1 && best < ring_lower_bound2(g, p.x, p.y, cx, T.cy, 1)) {
        out_ids[t] = best_id;
        if (out_dist) out_dist[t] = __dsqrt_rn(best);
        if (out_ties) out_ties[t] = ties;
        done = true;
      }
    } else {
      // pass 1: histogram of d2
#pragma unroll
      for (int bsel = 0; bsel < NT_BINS; ++bsel) hist[bsel * NT_THREADS] = 0;
      int n_far = 0;   // candidates beyond the last bin are only counted
#pragma unroll
      for (int rr3 = 0; rr3 < 3; ++rr3)
        for (int j = 0; j < rn[rr3]; ++j) {
          const double d = dist2(rx[rr3][j], p.x, p.y);
          if (d != d) continue;
          if (reach && !reach_bit(reach, g.reach_words, ri[rr3][j], wq)) continue;
          const double fb = d * bin_scale;
          if (fb < (double)NT_BINS) { uint8_t* h = hist + (int)fb * NT_THREADS; if (*h < 255) ++*h; }
          else ++n_far;
        }
      int cum = 0, B = -1;
      for (int bsel = 0; bsel < NT_BINS; ++bsel) {
        const int h = hist[bsel * NT_THREADS];
        if (h == 255) break;           // saturated counter: let the exact ring search handle it
        cum += h;
        if (cum >= k) { B = bsel; break; }
      }
      if (B >= 0 && cum <= cap && T.staged) {
        // pass 2: collect the candidates of bins 0..B as 16-bit codes (index into the staged tile), unsorted,
        // then insertion sort by (d2, id) with d2 recomputed from the staged tile.  2 bytes per entry instead of 12: the
        // shared-memory footprint of a CTA drops from 56 to 25 KiB and twice as many warps hide the latencies.
        const double lim = (double)(B + 1);
        int cnt = 0;
#pragma unroll
        for (int rr3 = 0; rr3 < 3; ++rr3)
          for (int j = 0; j < rn[rr3]; ++j) {
            const double d = dist2(rx[rr3][j], p.x, p.y);
            if (d != d || !(d * bin_scale < lim)) continue;
            if (reach && !reach_bit(reach, g.reach_words, ri[rr3][j], wq)) continue;
            lst[cnt * NT_THREADS] = (uint16_t)(rx[rr3] - s_xy + j);    // unsorted append: the warp stays together
            ++cnt;
          }
        // code = index into the staged coordinates; the staged ids sit at a per-row offset from it (16-byte phase of the copy)
        const int x1 = T.xoff[1], x2 = T.xoff[2], d0 = T.ioff[0] - T.xoff[0], d1 = T.ioff[1] - T.xoff[1], d2o = T.ioff[2] - T.xoff[2];
        auto cand_xy = [&](uint32_t code) -> double2 { return s_xy[code]; };
        auto cand_id = [&](uint32_t code) -> int32_t { return s_id[(int)code + ((int)code >= x2 ? d2o : ((int)code >= x1 ? d1 : d0))]; };
        for (int i = 1; i < cnt; ++i) {                              // every lane sorts its k + few entries at the same time
          const uint32_t code = lst[i * NT_THREADS];
          const double d = dist2(cand_xy(code), p.x, p.y);
          int pos = i;
          while (pos > 0) {
            const uint32_t pc = lst[(pos - 1) * NT_THREADS];
            const double pd = dist2(cand_xy(pc), p.x, p.y);
            if (!(d < pd || (d == pd && cand_id(code) < cand_id(pc)))) break;
            lst[pos * NT_THREADS] = (uint16_t)pc;
            --pos;
          }
          lst[pos * NT_THREADS] = (uint16_t)code;
        }
        if (cnt >= k) {
          const double dk = dist2(cand_xy(lst[(k - 1) * NT_THREADS]), p.x, p.y);
          if (dk < ring_lower_bound2(g, p.x, p.y, cx, T.cy, 1)) {
            for (int j = 0; j < k; ++j) {
              const uint32_t code = lst[j * NT_THREADS];
              out_ids[(int64_t)t * k + j] = cand_id(code);
              if (out_dist) out_dist[(int64_t)t * k + j] = __dsqrt_rn(dist2(cand_xy(code), p.x, p.y));
            }
            done = true;
          }
        }
      }
      (void)n_far;
    }
    if (!done) fb_list[atomicAdd(fb_n, 1)] = t;
  }
}

// ------------------------------------------------------------------------------------------------ host side
struct NtBins {
  int32_t *qcell, *qorder, *qcount, *cursor, *fb_list, *fb_n;
  int64_t* qstart;
  int tiles_per_row, n_tiles;
};

static int32_t nt_layout(porrt_ctx* ctx, const GridDev& g, int64_t m, NtBins* B) {
  const int64_t n_cells = (int64_t)g.cells_x * g.cells_y;
  CUDA_TRY(ctx, carve(ctx->nn_bins, [&](Carve& c) {
    B->qcell = c.take<int32_t>(m); B->qorder = c.take<int32_t>(m); B->fb_list = c.take<int32_t>(m);
    B->qcount = c.take<int32_t>(n_cells); B->cursor = c.take<int32_t>(n_cells); B->fb_n = c.take<int32_t>(1);
    B->qstart = c.take<int64_t>(n_cells + 1);
  }));
  B->tiles_per_row = (g.cells_x + NT_W - 1) / NT_W;
  B->n_tiles = B->tiles_per_row * g.cells_y;
  return PORRT_OK;
}

template <bool KNN>
static int32_t nt_bin(porrt_ctx* ctx, const GridDev& g, const double* q_dev, const double* radius_dev, int64_t m, NtBins* B) {
  cudaStream_t st = ctx->stream;
  const int64_t n_cells = (int64_t)g.cells_x * g.cells_y;
  int32_t rc0 = nt_layout(ctx, g, m, B);
  if (rc0) return rc0;
  CUDA_TRY(ctx, cudaMemsetAsync(B->qcount, 0, (char*)(B->fb_n + 1) - (char*)B->qcount, st));   // qcount, cursor and fb_n
  nt_bin_kernel<KNN><<<div_up(m, 256), 256, 0, st>>>(g, (const double2*)q_dev, radius_dev, m, B->qcell, B->qcount, B->fb_list, B->fb_n);
  LAUNCH_CHECK(ctx);
  int32_t rc = scan_exclusive_i64(ctx, B->qcount, n_cells, B->qstart);
  if (rc) return rc;
  nt_scatter_kernel<<<div_up(m, 256), 256, 0, st>>>(B->qcell, m, B->qstart, B->cursor, B->qorder);
  LAUNCH_CHECK(ctx);
  return PORRT_OK;
}

bool nn_tile_usable(const porrt_ctx* ctx, int64_t m) {
  // worth the binning passes only for real batches; the grid must be addressable with 32-bit cell ids and tile counts
  return m >= 2048 && (int64_t)ctx->cells_x * ctx->cells_y < (1ll << 30) && !ctx->force_thread_per_query_nn;
}

// the merge scripts of the current vertex set (see nbr_script_kernel); built on the first large radius batch after
// porrt_vertices_set and reused by every later one
static int32_t nn_tile_build_scripts(porrt_ctx* ctx, const GridDev& g) {
  if (ctx->nbr_ready) return PORRT_OK;
  cudaStream_t st = ctx->stream;
  const int64_t n_cells = (int64_t)g.cells_x * g.cells_y;
  CUDA_TRY(ctx, ctx->d_nbr_start.ensure((size_t)(n_cells + 1) * 8));
  CUDA_TRY(ctx, ctx->nn_bins.ensure((size_t)n_cells * 4));
  int32_t* sizes = ctx->nn_bins.as<int32_t>();
  nbr_size_kernel<<<div_up(n_cells, 256), 256, 0, st>>>(g, sizes);
  LAUNCH_CHECK(ctx);
  int32_t rc = scan_exclusive_i64(ctx, sizes, n_cells, ctx->d_nbr_start.as<int64_t>());
  if (rc) return rc;
  int64_t total = 0;
  CUDA_TRY(ctx, cudaMemcpyAsync(&total, ctx->d_nbr_start.as<int64_t>() + n_cells, 8, cudaMemcpyDeviceToHost, st));
  CUDA_TRY(ctx, cudaStreamSynchronize(st));
  CUDA_TRY(ctx, ctx->d_nbr_script.ensure((size_t)std::max<int64_t>(total, 8) * 2));
  nbr_script_kernel<<<div_up(n_cells * 32, 256), 256, 0, st>>>(g, ctx->d_nbr_start.as<int64_t>(), ctx->d_nbr_script.as<uint16_t>());
  LAUNCH_CHECK(ctx);
  ctx->nbr_ready = true;
  return PORRT_OK;
}

// One pass over the queries the tiles can serve: counts_dev[t] (zero-initialised by the caller) and stg_off_dev[t] (>= 0: the
// query's id-ascending list sits at that offset of *staging_out; -1 = not served here) -- nn_tile_radius_place moves the lists once
// the offsets are known.  *fb_list_out / *fb_n_out: the queries left to the thread-per-query kernels.
int32_t nn_tile_radius_collect(porrt_ctx* ctx, const GridDev& g, const double* q_dev, const double* radius_dev, int64_t m,
                               const uint32_t* prefix_dev, const uint64_t* reach_dev, const uint32_t* world_dev, int32_t* counts_dev,
                               int64_t* stg_off_dev, const int32_t** staging_out, const int32_t** fb_list_out, int32_t* fb_n_out,
                               int64_t* staged_total_out) {
  cudaStream_t st = ctx->stream;
  NtBins B;
  int32_t rc = nn_tile_build_scripts(ctx, g);
  if (rc) return rc;
  rc = nt_bin<false>(ctx, g, q_dev, radius_dev, m, &B);
  if (rc) return rc;
  // staging: room for 64 hits per query on average; warps that find it full fall back
  const int64_t stg_cap = m * 64 + 4096;
  int32_t* staging;
  unsigned long long* cursor;
  CUDA_TRY(ctx, carve(ctx->nn_stage, [&](Carve& c) { staging = c.take<int32_t>(stg_cap); cursor = c.take<unsigned long long>(1); }));
  CUDA_TRY(ctx, cudaMemsetAsync(cursor, 0, 8, st));
  CUDA_TRY(ctx, cudaMemsetAsync(stg_off_dev, 0xff, (size_t)m * 8, st));
  static bool attr_set[16] = {};
  if (!attr_set[ctx->device & 15]) {
    CUDA_TRY(ctx, cudaFuncSetAttribute(nt_radius_collect_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, NR_SMEM));
    attr_set[ctx->device & 15] = true;
  }
  const int ctas = (int)std::min<int64_t>(B.n_tiles, (int64_t)ctx->sm_count * NR_CTAS_PER_SM);   // persistent: as many CTAs as fit an SM
  nt_radius_collect_kernel<<<ctas, NR_THREADS, NR_SMEM, st>>>(g, (const double2*)q_dev, radius_dev, prefix_dev, reach_dev, world_dev, B.qorder,
                                                               B.qstart, ctx->d_nbr_start.as<int64_t>(), ctx->d_nbr_script.as<uint16_t>(),
                                                               B.tiles_per_row, B.n_tiles, counts_dev, stg_off_dev, staging, cursor, stg_cap,
                                                               B.fb_list, B.fb_n);
  LAUNCH_CHECK(ctx);
  unsigned long long staged = 0;
  CUDA_TRY(ctx, cudaMemcpyAsync(&ctx->nn_fb_n, B.fb_n, 4, cudaMemcpyDeviceToHost, st));
  CUDA_TRY(ctx, cudaMemcpyAsync(&staged, cursor, 8, cudaMemcpyDeviceToHost, st));
  CUDA_TRY(ctx, cudaStreamSynchronize(st));
  *staging_out = staging;
  *fb_list_out = B.fb_list;
  *fb_n_out = ctx->nn_fb_n;
  // with nothing left over every reserved slot holds a hit: the cursor IS the total, the caller need not wait for its scan
  if (staged_total_out) *staged_total_out = ctx->nn_fb_n == 0 ? (int64_t)staged : -1;
  if (getenv("PORRT_DEBUG")) fprintf(stderr, "[porrt] nn tiles: %lld queries, %d left to the thread-per-query kernels\n", (long long)m, ctx->nn_fb_n);
  return PORRT_OK;
}

int32_t nn_tile_radius_place(porrt_ctx* ctx, const int32_t* staging, const int64_t* stg_off_dev, const int64_t* offsets_dev, int64_t m,
                             int32_t* ids_dev) {
  nt_radius_place_kernel<<<ctx->sm_count * 8, 256, 0, ctx->stream>>>(staging, stg_off_dev, offsets_dev, m, ids_dev);
  LAUNCH_CHECK(ctx);
  return PORRT_OK;
}

int32_t nn_tile_knn(porrt_ctx* ctx, const GridDev& g, const double* q_dev, int64_t m, int k, const uint64_t* reach_dev,
                    const uint32_t* world_dev, int32_t* ids_dev, double* dist_dev, int32_t* ties_dev, const int32_t** fb_list_out,
                    int32_t* fb_n_out) {
  cudaStream_t st = ctx->stream;
  NtBins B;
  int32_t rc = nt_bin<true>(ctx, g, q_dev, nullptr, m, &B);
  if (rc) return rc;
  const size_t smem = (size_t)NT_CAP_KNN * 16 + (size_t)(NT_CAP_KNN + 24) * 4 + (size_t)(k + NT_SLACK) * NT_THREADS * 2 + (size_t)NT_BINS * NT_THREADS;
  static bool attr_set[16] = {};
  if (!attr_set[ctx->device & 15]) {
    CUDA_TRY(ctx, cudaFuncSetAttribute(nt_knn_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 100 * 1024));
    attr_set[ctx->device & 15] = true;
  }
  nt_knn_kernel<<<B.n_tiles, NT_THREADS, smem, st>>>(g, (const double2*)q_dev, k, reach_dev, world_dev, B.qorder, B.qstart, B.tiles_per_row,
                                                     ids_dev, dist_dev, ties_dev, B.fb_list, B.fb_n);
  LAUNCH_CHECK(ctx);
  CUDA_TRY(ctx, cudaMemcpyAsync(&ctx->nn_fb_n, B.fb_n, 4, cudaMemcpyDeviceToHost, st));
  CUDA_TRY(ctx, cudaStreamSynchronize(st));
  *fb_list_out = B.fb_list;
  *fb_n_out = ctx->nn_fb_n;
  if (getenv("PORRT_DEBUG")) fprintf(stderr, "[porrt] nn tiles: %lld queries, %d left to the thread-per-query kernels\n", (long long)m, ctx->nn_fb_n);
  return PORRT_OK;
}
