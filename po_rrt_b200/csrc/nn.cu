// nn.cu -- batched nearest-neighbour search (SURVEY.md 8(a) rows B2, B3, + k-NN), replacing the per-query walks of
// KdTree<N> (reference src/nearest_neighbor.rs:48-126) and norm2 (src/common.rs:203-213).
//
// B200 design: the unbalanced boxed kd-tree is pointer chasing; here the vertex set is binned once into a uniform
// cell grid (cell >= typical radius) stored as a cell-sorted AoS buffer {x,y} (16 B, one LDG.128 per candidate) plus a
// parallel id array, both ordered (cell row-major, id ascending).  The three cell rows a radius query overlaps are
// three CONTIGUOUS ranges of that buffer.  All distance arithmetic is the reference's f64 sequence (no FMA);
// the inclusive test sqrt(d2) <= r is evaluated as d2 <= T(r) with T(r) = max{t : sqrt(t) <= r} (exact, SURVEY 8(g)3).
//
// Also here: the library's scan and stable LSD radix sort (used for binning and for restoring per-query orders).
#include <algorithm>
#include <cmath>

#include "common.cuh"
#include "nn_dev.cuh"

// ================================================================================================ scan
// exclusive scan of u32 counts into i64 offsets; three-phase (block scan, scan of block sums, add).
#define SCAN_BLOCK 256
#define SCAN_ITEMS 8
#define SCAN_TILE (SCAN_BLOCK * SCAN_ITEMS)

__global__ void __launch_bounds__(SCAN_BLOCK) scan_block_kernel(const int32_t* __restrict__ in, int64_t n, int64_t* __restrict__ out,
                                                                int64_t* __restrict__ block_sums) {
  __shared__ int64_t s_warp[SCAN_BLOCK / 32];
  const int64_t base = (int64_t)blockIdx.x * SCAN_TILE + (int64_t)threadIdx.x * SCAN_ITEMS;
  int64_t v[SCAN_ITEMS], sum = 0;
#pragma unroll
  for (int k = 0; k < SCAN_ITEMS; ++k) {
    v[k] = (base + k < n) ? (int64_t)(uint32_t)in[base + k] : 0;
    sum += v[k];
  }
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  int64_t incl = sum;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    int64_t t = __shfl_up_sync(0xffffffffu, incl, o);
    if (lane >= o) incl += t;
  }
  if (lane == 31) s_warp[wid] = incl;
  __syncthreads();
  if (wid == 0) {
    int64_t w = lane < SCAN_BLOCK / 32 ? s_warp[lane] : 0;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      int64_t t = __shfl_up_sync(0xffffffffu, w, o);
      if (lane >= o) w += t;
    }
    if (lane < SCAN_BLOCK / 32) s_warp[lane] = w;  // inclusive over warps
  }
  __syncthreads();
  int64_t excl = incl - sum + (wid ? s_warp[wid - 1] : 0);
#pragma unroll
  for (int k = 0; k < SCAN_ITEMS; ++k) {
    if (base + k < n) out[base + k] = excl;
    excl += v[k];
  }
  if (threadIdx.x == SCAN_BLOCK - 1) block_sums[blockIdx.x] = s_warp[SCAN_BLOCK / 32 - 1];
}

__global__ void scan_sums_kernel(int64_t* __restrict__ sums, int64_t nb, int64_t* __restrict__ total_out) {
  // single block, sequential over tiles of blockDim: nb is small (n / 2048)
  __shared__ int64_t s_warp[32];
  __shared__ int64_t s_carry;
  if (threadIdx.x == 0) s_carry = 0;
  __syncthreads();
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  for (int64_t base = 0; base < nb; base += blockDim.x) {
    int64_t i = base + threadIdx.x;
    int64_t v = i < nb ? sums[i] : 0, incl = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      int64_t t = __shfl_up_sync(0xffffffffu, incl, o);
      if (lane >= o) incl += t;
    }
    if (lane == 31) s_warp[wid] = incl;
    __syncthreads();
    if (wid == 0) {
      int64_t w = lane < (int)(blockDim.x >> 5) ? s_warp[lane] : 0;
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) {
        int64_t t = __shfl_up_sync(0xffffffffu, w, o);
        if (lane >= o) w += t;
      }
      s_warp[lane] = w;
    }
    __syncthreads();
    int64_t carry = s_carry;
    int64_t excl = carry + incl - v + (wid ? s_warp[wid - 1] : 0);
    if (i < nb) sums[i] = excl;
    __syncthreads();
    if (threadIdx.x == blockDim.x - 1) s_carry = excl + v;
    __syncthreads();
  }
  if (threadIdx.x == 0 && total_out) *total_out = s_carry;
}

__global__ void scan_add_kernel(int64_t* __restrict__ out, int64_t n, const int64_t* __restrict__ sums, int64_t* __restrict__ tail) {
  const int64_t base = (int64_t)blockIdx.x * SCAN_TILE;
  const int64_t add = sums[blockIdx.x];
  for (int k = threadIdx.x; k < SCAN_TILE; k += SCAN_BLOCK)
    if (base + k < n) out[base + k] += add;
  (void)tail;
}

// out[0..n) = exclusive offsets, out[n] = total
int32_t scan_exclusive_i64(porrt_ctx* ctx, const int32_t* counts_dev, int64_t n, int64_t* out_dev) {
  cudaStream_t st = ctx->stream;
  if (n == 0) { CUDA_TRY(ctx, cudaMemsetAsync(out_dev, 0, 8, st)); return PORRT_OK; }
  const int64_t nb = (n + SCAN_TILE - 1) / SCAN_TILE;
  CUDA_TRY(ctx, ctx->scan_sums.ensure((size_t)nb * 8 + 8));
  int64_t* sums = ctx->scan_sums.as<int64_t>();
  scan_block_kernel<<<(int)nb, SCAN_BLOCK, 0, st>>>(counts_dev, n, out_dev, sums);
  LAUNCH_CHECK(ctx);
  scan_sums_kernel<<<1, 1024, 0, st>>>(sums, nb, out_dev + n);
  LAUNCH_CHECK(ctx);
  scan_add_kernel<<<(int)nb, SCAN_BLOCK, 0, st>>>(out_dev, n, sums, nullptr);
  LAUNCH_CHECK(ctx);
  return PORRT_OK;
}

// ================================================================================================ radix sort
// Stable LSD radix sort of (u64 key, u32 value) pairs, 8 bits per pass.  One warp owns a tile of RS_TILE consecutive
// elements and walks it 32 at a time in order, so ranks inside a digit follow the input order (stability) by
// __match_any_sync + popc; no cross-warp ordering problem arises because tile bases come from the scan.
#define RS_TILE 2048
#define RS_WARPS 4

__global__ void __launch_bounds__(RS_WARPS * 32) rs_hist_kernel(const uint64_t* __restrict__ keys, int64_t n, int shift,
                                                                int64_t n_tiles, int32_t* __restrict__ hist /* [256][n_tiles] */) {
  __shared__ int32_t s_h[RS_WARPS][256];
  const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
  const int64_t tile = (int64_t)blockIdx.x * RS_WARPS + wib;
  for (int b = lane; b < 256; b += 32) s_h[wib][b] = 0;
  __syncwarp();
  if (tile < n_tiles) {
    const int64_t lo = tile * RS_TILE, hi = min(n, lo + RS_TILE);
    for (int64_t i = lo + lane; i < hi; i += 32) atomicAdd(&s_h[wib][(int)((keys[i] >> shift) & 255)], 1);
    __syncwarp();
    for (int b = lane; b < 256; b += 32) hist[(int64_t)b * n_tiles + tile] = s_h[wib][b];
  }
}

__global__ void __launch_bounds__(RS_WARPS * 32) rs_scatter_kernel(const uint64_t* __restrict__ keys, const uint32_t* __restrict__ vals,
                                                                   int64_t n, int shift, int64_t n_tiles,
                                                                   const int64_t* __restrict__ bases /* [256][n_tiles] */,
                                                                   uint64_t* __restrict__ out_keys, uint32_t* __restrict__ out_vals) {
  __shared__ int64_t s_b[RS_WARPS][256];
  const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
  const int64_t tile = (int64_t)blockIdx.x * RS_WARPS + wib;
  if (tile >= n_tiles) return;
  for (int b = lane; b < 256; b += 32) s_b[wib][b] = bases[(int64_t)b * n_tiles + tile];
  __syncwarp();
  const int64_t lo = tile * RS_TILE, hi = min(n, lo + RS_TILE);
  for (int64_t i0 = lo; i0 < hi; i0 += 32) {
    const int64_t i = i0 + lane;
    const bool valid = i < hi;
    const unsigned active = __ballot_sync(0xffffffffu, valid);
    if (valid) {
      const uint64_t k = keys[i];
      const uint32_t v = vals[i];
      const int d = (int)((k >> shift) & 255);
      const unsigned peers = __match_any_sync(active, d);
      const int rank = __popc(peers & ((1u << lane) - 1u));
      const int64_t b = s_b[wib][d];
      __syncwarp(active);
      if (rank == 0) s_b[wib][d] = b + __popc(peers);
      __syncwarp(active);
      out_keys[b + rank] = k;
      out_vals[b + rank] = v;
    }
  }
}

// sorts in place (result ends in keys/vals); work space radix_keys, radix_vals, radix_hist
int32_t radix_sort_pairs(porrt_ctx* ctx, uint64_t* keys, uint32_t* vals, int64_t n, int key_bits) {
  if (n <= 1) return PORRT_OK;
  cudaStream_t st = ctx->stream;
  const int64_t n_tiles = (n + RS_TILE - 1) / RS_TILE;
  CUDA_TRY(ctx, ctx->radix_keys.ensure((size_t)n * 8));
  CUDA_TRY(ctx, ctx->radix_vals.ensure((size_t)n * 4));
  int64_t* bases;
  int32_t* hist;
  CUDA_TRY(ctx, carve(ctx->radix_hist, [&](Carve& c) { bases = c.take<int64_t>((size_t)n_tiles * 256 + 1); hist = c.take<int32_t>((size_t)n_tiles * 256); }));
  uint64_t* k2 = ctx->radix_keys.as<uint64_t>();
  uint32_t* v2 = ctx->radix_vals.as<uint32_t>();
  uint64_t *ki = keys, *ko = k2;
  uint32_t *vi = vals, *vo = v2;
  const int blocks = (int)((n_tiles + RS_WARPS - 1) / RS_WARPS);
  int passes = (key_bits + 7) / 8;
  if (passes < 1) passes = 1;
  for (int p = 0; p < passes; ++p) {
    rs_hist_kernel<<<blocks, RS_WARPS * 32, 0, st>>>(ki, n, p * 8, n_tiles, hist);
    LAUNCH_CHECK(ctx);
    int32_t rc = scan_exclusive_i64(ctx, hist, n_tiles * 256, bases);
    if (rc) return rc;
    rs_scatter_kernel<<<blocks, RS_WARPS * 32, 0, st>>>(ki, vi, n, p * 8, n_tiles, bases, ko, vo);
    LAUNCH_CHECK(ctx);
    std::swap(ki, ko);
    std::swap(vi, vo);
  }
  if (ki != keys) {
    CUDA_TRY(ctx, cudaMemcpyAsync(keys, ki, (size_t)n * 8, cudaMemcpyDeviceToDevice, st));
    CUDA_TRY(ctx, cudaMemcpyAsync(vals, vi, (size_t)n * 4, cudaMemcpyDeviceToDevice, st));
  }
  return PORRT_OK;
}

int bits_for(uint64_t max_value) {
  int b = 1;
  while (b < 64 && (max_value >> b)) ++b;
  return b;
}

// ================================================================================================ cell grid
__global__ void bbox_kernel(const double2* __restrict__ xy, int64_t n, double* __restrict__ out /* minx,miny,maxx,maxy as ordered u64 */) {
  double mnx = INFINITY, mny = INFINITY, mxx = -INFINITY, mxy = -INFINITY;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    double2 p = xy[i];
    mnx = fmin(mnx, p.x); mny = fmin(mny, p.y); mxx = fmax(mxx, p.x); mxy = fmax(mxy, p.y);
  }
  for (int o = 16; o; o >>= 1) {
    mnx = fmin(mnx, __shfl_xor_sync(0xffffffffu, mnx, o)); mny = fmin(mny, __shfl_xor_sync(0xffffffffu, mny, o));
    mxx = fmax(mxx, __shfl_xor_sync(0xffffffffu, mxx, o)); mxy = fmax(mxy, __shfl_xor_sync(0xffffffffu, mxy, o));
  }
  if ((threadIdx.x & 31) == 0) {
    // order-preserving map double -> u64 so that atomicMin/Max on integers work for negative values too
    auto enc = [](double d) { unsigned long long b = (unsigned long long)__double_as_longlong(d); return (b & 0x8000000000000000ull) ? ~b : (b | 0x8000000000000000ull); };
    unsigned long long* o = (unsigned long long*)out;
    atomicMin(&o[0], enc(mnx)); atomicMin(&o[1], enc(mny)); atomicMax(&o[2], enc(mxx)); atomicMax(&o[3], enc(mxy));
  }
}

__global__ void cell_key_kernel(const double2* __restrict__ xy, int64_t n, double org_x, double org_y, double inv_cell,
                                int cells_x, int cells_y, uint64_t* __restrict__ keys, uint32_t* __restrict__ vals,
                                int32_t* __restrict__ counts) {
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  double2 p = xy[i];
  int cx = cell_coord(p.x, org_x, inv_cell, cells_x), cy = cell_coord(p.y, org_y, inv_cell, cells_y);
  uint32_t c = (uint32_t)cy * (uint32_t)cells_x + (uint32_t)cx;
  keys[i] = c;
  vals[i] = (uint32_t)i;
  atomicAdd(&counts[c], 1);
}

__global__ void gather_vertices_kernel(const double2* __restrict__ xy, const uint32_t* __restrict__ order, int64_t n,
                                       double2* __restrict__ out_xy, int32_t* __restrict__ out_id) {
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  uint32_t id = order[i];
  out_xy[i] = xy[id];
  out_id[i] = (int32_t)id;
}

static GridDev grid_dev(porrt_ctx* ctx) {
  GridDev g;
  g.vxy = ctx->d_vxy_sorted.as<double2>(); g.vid = ctx->d_vid_sorted.as<int32_t>(); g.cell_start = ctx->d_cell_start.as<int64_t>();
  g.org_x = ctx->org_x; g.org_y = ctx->org_y; g.inv_cell = ctx->inv_cell; g.cell = ctx->cell;
  g.cells_x = ctx->cells_x; g.cells_y = ctx->cells_y; g.n = ctx->n_vertices;
  g.reach_words = ctx->reach_words;
  return g;
}

int32_t nn_vertices_set_dev(porrt_ctx* ctx, const double* xy_dev, int64_t n, double cell_size, const double* lo, const double* hi) {
  cudaStream_t st = ctx->stream;
  ctx->n_vertices = 0;
  ctx->nbr_ready = false;     // the merge scripts of nn_tile.cu belong to the previous vertex set
  if (n <= 0 || n > 0x7fffffff) return porrt_fail(ctx, PORRT_ERR_INVALID_ARG, "vertices_set: n out of range");
  double blo[2], bhi[2];
  if (lo && hi) { blo[0] = lo[0]; blo[1] = lo[1]; bhi[0] = hi[0]; bhi[1] = hi[1]; }
  else {
    CUDA_TRY(ctx, ctx->ws_query.ensure(32));
    unsigned long long init[4] = {~0ull, ~0ull, 0ull, 0ull};
    CUDA_TRY(ctx, cudaMemcpyAsync(ctx->ws_query.p, init, 32, cudaMemcpyHostToDevice, st));
    bbox_kernel<<<ctx->sm_count * 4, 256, 0, st>>>((const double2*)xy_dev, n, ctx->ws_query.as<double>());
    LAUNCH_CHECK(ctx);
    unsigned long long enc[4];
    CUDA_TRY(ctx, cudaMemcpyAsync(enc, ctx->ws_query.p, 32, cudaMemcpyDeviceToHost, st));
    CUDA_TRY(ctx, cudaStreamSynchronize(st));
    double dec[4];
    for (int k = 0; k < 4; ++k) {
      unsigned long long b = (enc[k] & 0x8000000000000000ull) ? (enc[k] & 0x7fffffffffffffffull) : ~enc[k];
      memcpy(&dec[k], &b, 8);
    }
    blo[0] = dec[0]; blo[1] = dec[1]; bhi[0] = dec[2]; bhi[1] = dec[3];
  }
  if (!(blo[0] <= bhi[0]) || !(blo[1] <= bhi[1]) || !std::isfinite(blo[0]) || !std::isfinite(bhi[0]) || !std::isfinite(blo[1]) || !std::isfinite(bhi[1]))
    return porrt_fail(ctx, PORRT_ERR_INVALID_ARG, "vertices_set: non-finite coordinates");
  double ex = bhi[0] - blo[0], ey = bhi[1] - blo[1];
  double cell = cell_size;
  if (!(cell > 0.0)) cell = std::sqrt(std::max(ex * ey, 1e-300) * 2.0 / (double)n);  // ~2 vertices per cell
  if (!(cell > 0.0) || !std::isfinite(cell)) cell = 1.0;
  const double MAX_CELLS = 16777216.0;  // 2^24 -> 3 radix passes, 128 MiB of cell_start at most
  for (;;) {
    double cxs = std::floor(ex / cell) + 1.0, cys = std::floor(ey / cell) + 1.0;
    if (cxs * cys <= MAX_CELLS) { ctx->cells_x = (int)cxs; ctx->cells_y = (int)cys; break; }
    cell *= 1.5;
  }
  ctx->cell = cell; ctx->inv_cell = 1.0 / cell; ctx->org_x = blo[0]; ctx->org_y = blo[1];
  const int64_t n_cells = (int64_t)ctx->cells_x * ctx->cells_y;
  CUDA_TRY(ctx, ctx->sort_keys.ensure((size_t)n * 8));
  CUDA_TRY(ctx, ctx->sort_vals.ensure((size_t)n * 4));
  CUDA_TRY(ctx, ctx->ws_state.ensure((size_t)n_cells * 4));   // cell counts
  CUDA_TRY(ctx, ctx->d_cell_start.ensure((size_t)(n_cells + 1) * 8));
  CUDA_TRY(ctx, ctx->d_vxy_sorted.ensure((size_t)n * 16));
  CUDA_TRY(ctx, ctx->d_vid_sorted.ensure((size_t)n * 4));
  CUDA_TRY(ctx, cudaMemsetAsync(ctx->ws_state.p, 0, (size_t)n_cells * 4, st));
  cell_key_kernel<<<div_up(n, 256), 256, 0, st>>>((const double2*)xy_dev, n, ctx->org_x, ctx->org_y, ctx->inv_cell, ctx->cells_x, ctx->cells_y,
                                                  ctx->sort_keys.as<uint64_t>(), ctx->sort_vals.as<uint32_t>(), ctx->ws_state.as<int32_t>());
  LAUNCH_CHECK(ctx);
  int32_t rc = scan_exclusive_i64(ctx, ctx->ws_state.as<int32_t>(), n_cells, ctx->d_cell_start.as<int64_t>());
  if (rc) return rc;
  rc = radix_sort_pairs(ctx, ctx->sort_keys.as<uint64_t>(), ctx->sort_vals.as<uint32_t>(), n, bits_for((uint64_t)n_cells - 1));
  if (rc) return rc;
  gather_vertices_kernel<<<div_up(n, 256), 256, 0, st>>>((const double2*)xy_dev, ctx->sort_vals.as<uint32_t>(), n,
                                                         ctx->d_vxy_sorted.as<double2>(), ctx->d_vid_sorted.as<int32_t>());
  LAUNCH_CHECK(ctx);
  ctx->n_vertices = n;
  ctx->grid_stale = false;
  return PORRT_OK;
}

PORRT_API int32_t porrt_vertices_set_dev(porrt_ctx* ctx, const double* xy_dev, int64_t n, double cell_size, const double lo[2], const double hi[2]) {
  CTX_CHECK(ctx);
  CUDA_TRY(ctx, cudaSetDevice(ctx->device));
  if (!xy_dev) return porrt_fail(ctx, PORRT_ERR_INVALID_ARG, "vertices_set_dev: null");
  if (n > 0 && xy_dev != ctx->d_vxy.as<double>()) {   // the library keeps its own copy in upload order (porrt_edge_validity_indexed reads it)
    CUDA_TRY(ctx, ctx->d_vxy.ensure((size_t)n * 16));
    CUDA_TRY(ctx, cudaMemcpyAsync(ctx->d_vxy.p, xy_dev, (size_t)n * 16, cudaMemcpyDeviceToDevice, ctx->stream));
  }
  return nn_vertices_set_dev(ctx, xy_dev, n, cell_size, lo, hi);
}

PORRT_API int32_t porrt_vertices_set(porrt_ctx* ctx, const double* xy, int64_t n, double cell_size) {
  CTX_CHECK(ctx);
  CUDA_TRY(ctx, cudaSetDevice(ctx->device));
  if (!xy || n <= 0) return porrt_fail(ctx, PORRT_ERR_INVALID_ARG, "vertices_set: bad arguments");
  CUDA_TRY(ctx, ctx->d_vxy.ensure((size_t)n * 16));
  CUDA_TRY(ctx, cudaMemcpyAsync(ctx->d_vxy.p, xy, (size_t)n * 16, cudaMemcpyHostToDevice, ctx->stream));
  ctx->cell_request = cell_size;
  return nn_vertices_set_dev(ctx, ctx->d_vxy.as<double>(), n, cell_size, nullptr, nullptr);
}

// KdTree::add (nearest_neighbor.rs:29-46), batched: the m new vertices get the ids n .. n+m-1.  Only the new coordinates cross the
// bus (a sequential caller that re-sent the whole set before every query moved O(V^2) bytes); the cell grid is rebuilt from the
// device-resident set -- bounding box, cell size rule of the last porrt_vertices_set, sort by cell -- before the next query.
PORRT_API int32_t porrt_vertices_append(porrt_ctx* ctx, const double* xy, int64_t m) {
  CTX_CHECK(ctx);
  if (m < 0 || (m > 0 && !xy)) return porrt_fail(ctx, PORRT_ERR_INVALID_ARG, "vertices_append: bad arguments");
  if (m == 0) return PORRT_OK;
  CUDA_TRY(ctx, cudaSetDevice(ctx->device));
  const int64_t n = ctx->n_vertices;
  if (n + m > 0x7fffffff) return porrt_fail(ctx, PORRT_ERR_INVALID_ARG, "vertices_append: too many vertices");
  CUDA_TRY(ctx, ctx->d_vxy.grow_keep((size_t)(n + m) * 16, (size_t)n * 16, ctx->stream));
  CUDA_TRY(ctx, cudaMemcpyAsync(ctx->d_vxy.as<char>() + (size_t)n * 16, xy, (size_t)m * 16, cudaMemcpyHostToDevice, ctx->stream));
  CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));   // xy is the caller's (possibly pageable) memory
  ctx->n_vertices = n + m;
  ctx->grid_stale = true;
  return PORRT_OK;
}

int32_t nn_flush_appended(porrt_ctx* ctx) {
  if (!ctx->grid_stale) return PORRT_OK;
  return nn_vertices_set_dev(ctx, ctx->d_vxy.as<double>(), ctx->n_vertices, ctx->cell_request, nullptr, nullptr);
}

PORRT_API int32_t porrt_vertices_count(porrt_ctx* ctx, int64_t* out_n) {
  CTX_CHECK(ctx);
  if (out_n) *out_n = ctx->n_vertices;
  return PORRT_OK;
}

// ================================================================================================ radius query
// Prefix-restricted queries that cover many cells (the early nodes of a PRM: radius up to max_step over a grid whose cell is the
// LAST node's radius, 100-800 cells, almost all of them answered by one id comparison because the list is id-ascending and the
// limit small) are a chain of dependent loads per cell: a thread per query walks them one after the other (the tail of the PRM's
// radius phase), a WARP per query takes 32 cells at a time.  Same hits in the same order (cell rows outer, cells inner).
#define RADIUS_WIDE_CELLS 64   // (24: the wide kernels then cost more than they save -- 1.78 against 1.29 ms for both passes at 1e6 nodes)
__global__ void radius_wide_list_kernel(GridDev g, const double2* __restrict__ q, const double* __restrict__ radius, int64_t m,
                                        const int32_t* __restrict__ list, int32_t* __restrict__ wide, int32_t* __restrict__ n_wide) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= m) return;
  const int64_t t = list ? list[i] : i;
  const double2 p = q[t];
  const double r = radius[t];
  if (!(radius_threshold(r) >= 0.0) || !(p.x == p.x && p.y == p.y)) return;
  const double rr = isinf(r) ? r : __dadd_rn(__dmul_rn(r, 1.000000001), 1e-300);
  const int cx0 = cell_coord(p.x - rr, g.org_x, g.inv_cell, g.cells_x), cx1 = cell_coord(p.x + rr, g.org_x, g.inv_cell, g.cells_x);
  const int cy0 = cell_coord(p.y - rr, g.org_y, g.inv_cell, g.cells_y), cy1 = cell_coord(p.y + rr, g.org_y, g.inv_cell, g.cells_y);
  if ((int64_t)(cx1 - cx0 + 1) * (cy1 - cy0 + 1) > RADIUS_WIDE_CELLS) wide[atomicAdd(n_wide, 1)] = (int32_t)i;   // the position in `list`: it names the query's staging slot
}
// MODE 0: count (counts[t]); 1: fill (out_ids + offsets[t]); 2: ONE pass -- count and keep the first RADIUS_STAGE_CAP hits in the
// query's staging slot (slot = the query's position in `list`); a query with more hits is appended to over_list and filled by a
// second pass of the thread-per-query kernel, everybody else is moved to its CSR place by nn_tile's placement copy
#define RADIUS_STAGE_CAP 96
template <int MODE>
__global__ void __launch_bounds__(128) radius_wide_kernel(GridDev g, const double2* __restrict__ q, const double* __restrict__ radius,
                                                          const int32_t* __restrict__ wide, const int32_t* __restrict__ n_wide,
                                                          const int32_t* __restrict__ list,
                                                          const uint32_t* __restrict__ prefix, const uint64_t* __restrict__ reach,
                                                          const uint32_t* __restrict__ world, int32_t* __restrict__ counts,
                                                          const int64_t* __restrict__ offsets, int32_t* __restrict__ out_ids,
                                                          const uint32_t* __restrict__ prefix_lo, int64_t* __restrict__ stg_off = nullptr,
                                                          int32_t* __restrict__ over_list = nullptr, int32_t* __restrict__ over_n = nullptr) {
  constexpr bool FILL = MODE != 0;
  const int lane = threadIdx.x & 31;
  const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, n_warps = (gridDim.x * blockDim.x) >> 5;
  for (int qi = warp; qi < *n_wide; qi += n_warps) {
    const int32_t slot = wide[qi];
    const int32_t t = list ? list[slot] : slot;
    const double2 p = q[t];
    const double r = radius[t];
    const double T = radius_threshold(r);
    const uint32_t limit = prefix[t];
    const uint32_t lo_limit = prefix_lo ? prefix_lo[t] : 0u;
    const uint32_t wq = (reach && world) ? world[t] : 0u;
    const double rr = isinf(r) ? r : __dadd_rn(__dmul_rn(r, 1.000000001), 1e-300);
    const int cx0 = cell_coord(p.x - rr, g.org_x, g.inv_cell, g.cells_x), cx1 = cell_coord(p.x + rr, g.org_x, g.inv_cell, g.cells_x);
    const int cy0 = cell_coord(p.y - rr, g.org_y, g.inv_cell, g.cells_y), cy1 = cell_coord(p.y + rr, g.org_y, g.inv_cell, g.cells_y);
    const int nx = cx1 - cx0 + 1;
    const int64_t n_cells = (int64_t)nx * (cy1 - cy0 + 1);
    int32_t* out = MODE == 1 ? out_ids + offsets[t] : (MODE == 2 ? out_ids + (int64_t)slot * RADIUS_STAGE_CAP : nullptr);
    int32_t run = 0;
    for (int64_t c0 = 0; c0 < n_cells; c0 += 32) {
      const int64_t ci = c0 + lane;
      int64_t k0 = 0, e = 0;
      if (ci < n_cells) {
        const int64_t c = (int64_t)(cy0 + (int)(ci / nx)) * g.cells_x + (cx0 + (int)(ci % nx));
        k0 = g.cell_start[c]; e = g.cell_start[c + 1];
        if (lo_limit) {   // grouped vertex sets: jump to the first id of the query's own group
          int64_t hi = e;
          while (k0 < hi) { const int64_t mid = (k0 + hi) >> 1; if ((uint32_t)g.vid[mid] < lo_limit) k0 = mid + 1; else hi = mid; }
        }
      }
      int32_t mine = 0;
      for (int64_t k = k0; k < e; ++k) {
        const uint32_t id = (uint32_t)g.vid[k];
        if (id >= limit) break;
        if (dist2(g.vxy[k], p.x, p.y) <= T && (!reach || reach_bit(reach, g.reach_words, id, wq))) ++mine;
      }
      int32_t incl = mine;
      for (int o = 1; o < 32; o <<= 1) { const int32_t v = __shfl_up_sync(0xffffffffu, incl, o); if (lane >= o) incl += v; }
      if (FILL && mine) {
        int32_t at = run + incl - mine;
        for (int64_t k = k0; k < e; ++k) {
          const uint32_t id = (uint32_t)g.vid[k];
          if (id >= limit) break;
          if (dist2(g.vxy[k], p.x, p.y) <= T && (!reach || reach_bit(reach, g.reach_words, id, wq))) {
            if (MODE == 1 || at < RADIUS_STAGE_CAP) out[at] = (int32_t)id;
            ++at;
          }
        }
      }
      run += __shfl_sync(0xffffffffu, incl, 31);
    }
    if (MODE != 1 && lane == 0) {
      counts[t] = run;
      if (MODE == 2) {
        if (run <= RADIUS_STAGE_CAP) stg_off[t] = (int64_t)slot * RADIUS_STAGE_CAP;
        else over_list[atomicAdd(over_n, 1)] = t;
      }
    }
  }
}

template <int MODE>   // as radius_wide_kernel
__global__ void __launch_bounds__(128) radius_kernel(GridDev g, const double2* __restrict__ q, const double* __restrict__ radius, int64_t m,
                                                     const uint32_t* __restrict__ prefix, const uint64_t* __restrict__ reach,
                                                     const uint32_t* __restrict__ world, int32_t* __restrict__ counts,
                                                     const int64_t* __restrict__ offsets, int32_t* __restrict__ out_ids,
                                                     const int32_t* __restrict__ list, const uint32_t* __restrict__ prefix_lo,
                                                     bool skip_wide = false, int64_t* __restrict__ stg_off = nullptr,
                                                     int32_t* __restrict__ over_list = nullptr, int32_t* __restrict__ over_n = nullptr) {
  constexpr bool FILL = MODE != 0;
  const int64_t slot = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (slot >= m) return;
  const int64_t t = list ? list[slot] : slot;   // m = length of the list: the queries nn_tile.cu left to this kernel
  const double2 p = q[t];
  const double r = radius[t];
  const double T = radius_threshold(r);
  int32_t cnt = 0;
  if (T >= 0.0 && p.x == p.x && p.y == p.y) {
    const uint32_t limit = prefix ? prefix[t] : 0xffffffffu;
    const uint32_t lo_limit = prefix_lo ? prefix_lo[t] : 0u;   // ids below belong to other roadmaps sharing the vertex set
    const uint32_t wq = (reach && world) ? world[t] : 0u;
    const double rr = isinf(r) ? r : __dadd_rn(__dmul_rn(r, 1.000000001), 1e-300);  // conservative cell cover
    const int cx0 = cell_coord(p.x - rr, g.org_x, g.inv_cell, g.cells_x), cx1 = cell_coord(p.x + rr, g.org_x, g.inv_cell, g.cells_x);
    const int cy0 = cell_coord(p.y - rr, g.org_y, g.inv_cell, g.cells_y), cy1 = cell_coord(p.y + rr, g.org_y, g.inv_cell, g.cells_y);
    if (skip_wide && prefix && (int64_t)(cx1 - cx0 + 1) * (cy1 - cy0 + 1) > RADIUS_WIDE_CELLS) return;   // radius_wide_kernel's
    int32_t* out = MODE == 1 ? out_ids + offsets[t] : (MODE == 2 ? out_ids + slot * RADIUS_STAGE_CAP : nullptr);
    for (int cy = cy0; cy <= cy1; ++cy) {
      if (prefix) {
        // cell lists are id-ascending: stop at the first id >= limit (the tree as it was when vertex `limit` arrived)
        for (int cx = cx0; cx <= cx1; ++cx) {
          const int64_t c = (int64_t)cy * g.cells_x + cx;
          const int64_t e = g.cell_start[c + 1];
          int64_t k = g.cell_start[c];
          if (lo_limit) {   // grouped vertex sets: jump to the first id of the query's own group (the list is id-ascending)
            int64_t hi = e;
            while (k < hi) { const int64_t mid = (k + hi) >> 1; if ((uint32_t)g.vid[mid] < lo_limit) k = mid + 1; else hi = mid; }
          }
          for (; k < e; ++k) {
            const uint32_t id = (uint32_t)g.vid[k];
            if (id >= limit) break;
            if (dist2(g.vxy[k], p.x, p.y) <= T && (!reach || reach_bit(reach, g.reach_words, id, wq))) {
              if (MODE == 1 || (MODE == 2 && cnt < RADIUS_STAGE_CAP)) out[cnt] = (int32_t)id;
              ++cnt;
            }
          }
        }
      } else {
        const int64_t s = g.cell_start[(int64_t)cy * g.cells_x + cx0], e = g.cell_start[(int64_t)cy * g.cells_x + cx1 + 1];
        for (int64_t k = s; k < e; ++k) {
          if (dist2(g.vxy[k], p.x, p.y) <= T) {
            const uint32_t id = (uint32_t)g.vid[k];
            if (!reach || reach_bit(reach, g.reach_words, id, wq)) {
              if (MODE == 1 || (MODE == 2 && cnt < RADIUS_STAGE_CAP)) out[cnt] = (int32_t)id;
              ++cnt;
            }
          }
        }
      }
    }
  }
  if (MODE != 1) counts[t] = cnt;
  if (MODE == 2) {
    if (cnt <= RADIUS_STAGE_CAP) stg_off[t] = slot * RADIUS_STAGE_CAP;
    else over_list[atomicAdd(over_n, 1)] = (int32_t)t;
  }
}

// offsets_dev[m+1] filled; ids_buf grown to the total; *total_out = total hits (host value).  Large batches go through the
// one-pass tile kernel (nn_tile.cu), which delivers its lists id-ascending; the queries it leaves over, small batches and grouped
// vertex sets (prefix_lo) are answered by the thread-per-query kernel above in cell order -- sort_ids puts those in id order too.
int32_t nn_radius_count_fill_dev(porrt_ctx* ctx, const double* q_dev, const double* radius_dev, int64_t m,
                                 const uint32_t* prefix_dev, const uint64_t* reach_dev, const uint32_t* world_dev,
                                 int64_t* offsets_dev, DevBuf* ids_buf, int64_t* total_out, const uint32_t* prefix_lo_dev, bool sort_ids, bool allow_tiles) {
  cudaStream_t st = ctx->stream;
  if (m <= 0) {   // an empty shard of a sharded batch
    CUDA_TRY(ctx, cudaMemsetAsync(offsets_dev, 0, 8, st));
    CUDA_TRY(ctx, ids_buf->ensure(4));
    *total_out = 0;
    return PORRT_OK;
  }
  GridDev g = grid_dev(ctx);
  // prefix-restricted queries over many cells get a warp each (radius_wide_kernel); the list is built once for both passes
  const bool wide = prefix_dev != nullptr && m >= 1024;
  int64_t* stg_off;
  int32_t* counts;
  int32_t* n_wide = nullptr;   // [0] the length of the wide-query list that follows 16 ints on
  CUDA_TRY(ctx, carve(ctx->ws_query, [&](Carve& c) {
    stg_off = c.take<int64_t>(m);
    counts = c.take<int32_t>(m);
    if (wide) n_wide = c.take<int32_t>(16 + m);
  }));
  int32_t* wide_list = wide ? n_wide + 16 : nullptr;
  // grouped vertex sets (prefix_lo): the other groups' vertices share the cells, staging them all would only cost; the
  // thread-per-query kernel skips to its own group inside each cell list
  // allow_tiles = false (the PRM build): the radii there are LARGER than the cell (cell = the last, smallest radius), so the tiles could
  // serve a quarter of the queries only -- not worth their merge scripts (0.28 ms per vertex set) and binning
  const bool tiles = allow_tiles && nn_tile_usable(ctx, m) && !prefix_lo_dev;
  const int32_t* fb_list = nullptr;
  const int32_t* staging = nullptr;
  int32_t fb_n = 0;
  if (wide) CUDA_TRY(ctx, cudaMemsetAsync(n_wide, 0, 4, st));
  const int wide_grid = ctx->sm_count * 8;
  int64_t staged_total = -1;   // >= 0: the tiles served every query and this is the number of hits
  if (tiles) {
    CUDA_TRY(ctx, cudaMemsetAsync(counts, 0, (size_t)m * 4, st));
    int32_t rc = nn_tile_radius_collect(ctx, g, q_dev, radius_dev, m, prefix_dev, reach_dev, world_dev, counts, stg_off, &staging, &fb_list, &fb_n, &staged_total);
    if (rc) return rc;
  }
  // what the tiles left over (or everything, without tiles): thread per query, a warp per query for prefix-restricted queries over
  // many cells.  ONE pass where the slots fit: every query counts its hits and keeps them in a slot of RADIUS_STAGE_CAP ids
  // (PRM: pi * ln k ~ 43 hits), the placement copy moves them once the scan of the counts is known; only queries with more hits are
  // walked a second time.  (The PRM's radius phase spent 0.53 + 0.70 ms in the count and fill passes of these queries.)
  const int64_t n_rest = tiles ? fb_n : m;
  const int32_t* rest_list = tiles ? fb_list : nullptr;
  const bool one_pass = n_rest > 0 && n_rest <= ((int64_t)8 << 20);
  int32_t* stage2 = nullptr; int64_t* stg_off2 = nullptr; int32_t* over_list = nullptr; int32_t* over_n = nullptr;
  if (one_pass) {
    CUDA_TRY(ctx, carve(ctx->nn_stage2, [&](Carve& c) {
      stg_off2 = c.take<int64_t>(m, 256);
      over_n = c.take<int32_t>(16 + n_rest, 256);   // the count, then the list 16 ints on
      stage2 = c.take<int32_t>((size_t)n_rest * RADIUS_STAGE_CAP, 256);
    }));
    over_list = over_n + 16;
    CUDA_TRY(ctx, cudaMemsetAsync(stg_off2, 0xff, (size_t)m * 8, st));   // -1: not in a slot
    CUDA_TRY(ctx, cudaMemsetAsync(over_n, 0, 4, st));
  }
  if (n_rest > 0) {
    if (wide) {
      radius_wide_list_kernel<<<div_up(n_rest, 256), 256, 0, st>>>(g, (const double2*)q_dev, radius_dev, n_rest, rest_list, wide_list, n_wide);
      LAUNCH_CHECK(ctx);
      if (one_pass) radius_wide_kernel<2><<<wide_grid, 128, 0, st>>>(g, (const double2*)q_dev, radius_dev, wide_list, n_wide, rest_list, prefix_dev, reach_dev, world_dev, counts, nullptr, stage2, prefix_lo_dev, stg_off2, over_list, over_n);
      else radius_wide_kernel<0><<<wide_grid, 128, 0, st>>>(g, (const double2*)q_dev, radius_dev, wide_list, n_wide, rest_list, prefix_dev, reach_dev, world_dev, counts, nullptr, nullptr, prefix_lo_dev);
      LAUNCH_CHECK(ctx);
    }
    if (one_pass) radius_kernel<2><<<div_up(n_rest, 128), 128, 0, st>>>(g, (const double2*)q_dev, radius_dev, n_rest, prefix_dev, reach_dev, world_dev, counts, nullptr, stage2, rest_list, prefix_lo_dev, wide, stg_off2, over_list, over_n);
    else radius_kernel<0><<<div_up(n_rest, 128), 128, 0, st>>>(g, (const double2*)q_dev, radius_dev, n_rest, prefix_dev, reach_dev, world_dev, counts, nullptr, nullptr, rest_list, prefix_lo_dev, wide);
    LAUNCH_CHECK(ctx);
  }
  int32_t rc = scan_exclusive_i64(ctx, counts, m, offsets_dev);
  if (rc) return rc;
  int64_t total = staged_total;
  int32_t n_over = 0;
  if (staged_total < 0) {   // (otherwise the scan and the placement copy follow the search without a host round trip)
    CUDA_TRY(ctx, cudaMemcpyAsync(&total, offsets_dev + m, 8, cudaMemcpyDeviceToHost, st));
    if (one_pass) CUDA_TRY(ctx, cudaMemcpyAsync(&n_over, over_n, 4, cudaMemcpyDeviceToHost, st));
    CUDA_TRY(ctx, cudaStreamSynchronize(st));
  }
  *total_out = total;
  CUDA_TRY(ctx, ids_buf->ensure((size_t)std::max<int64_t>(total, 1) * 4));
  if (total > 0) {
    if (tiles) {
      rc = nn_tile_radius_place(ctx, staging, stg_off, offsets_dev, m, ids_buf->as<int32_t>());
      if (rc) return rc;
    }
    if (n_rest > 0) {
      if (one_pass) {
        rc = nn_tile_radius_place(ctx, stage2, stg_off2, offsets_dev, m, ids_buf->as<int32_t>());
        if (rc) return rc;
        if (n_over > 0) {   // the few lists longer than a slot: second walk, straight to their CSR places
          radius_kernel<1><<<div_up(n_over, 128), 128, 0, st>>>(g, (const double2*)q_dev, radius_dev, n_over, prefix_dev, reach_dev, world_dev, nullptr, offsets_dev, ids_buf->as<int32_t>(), over_list, prefix_lo_dev, false);
          LAUNCH_CHECK(ctx);
        }
      } else {
        if (wide) {
          radius_wide_kernel<1><<<wide_grid, 128, 0, st>>>(g, (const double2*)q_dev, radius_dev, wide_list, n_wide, rest_list, prefix_dev, reach_dev, world_dev, nullptr, offsets_dev, ids_buf->as<int32_t>(), prefix_lo_dev);
          LAUNCH_CHECK(ctx);
        }
        radius_kernel<1><<<div_up(n_rest, 128), 128, 0, st>>>(g, (const double2*)q_dev, radius_dev, n_rest, prefix_dev, reach_dev, world_dev, nullptr, offsets_dev, ids_buf->as<int32_t>(), rest_list, prefix_lo_dev, wide);
        LAUNCH_CHECK(ctx);
      }
      if (sort_ids) {
        rc = segments_sort_by_key_dev(ctx, offsets_dev, m, ids_buf->as<int32_t>(), nullptr, g.n, rest_list, tiles ? fb_n : 0);
        if (rc) return rc;
      }
    }
  }
  return PORRT_OK;
}

// ---- per-segment ordering: sort ids inside each CSR segment by key_of_id (NULL: by id) with one global stable radix sort
__global__ void seg_key_kernel(const int64_t* __restrict__ offsets, int64_t m, const int32_t* __restrict__ ids,
                               const int32_t* __restrict__ key_of_id, int key_bits, uint64_t* __restrict__ keys, uint32_t* __restrict__ vals) {
  // one warp per segment
  const int lane = threadIdx.x & 31;
  const int64_t seg = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  if (seg >= m) return;
  const int64_t s = offsets[seg], e = offsets[seg + 1];
  for (int64_t k = s + lane; k < e; k += 32) {
    const int32_t id = ids[k];
    const uint64_t key = key_of_id ? (uint64_t)(uint32_t)key_of_id[id] : (uint64_t)(uint32_t)id;
    keys[k] = ((uint64_t)seg << key_bits) | key;
    vals[k] = (uint32_t)id;
  }
}
__global__ void copy_u32_i32_kernel(const uint32_t* __restrict__ in, int64_t n, int32_t* __restrict__ out) {
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) out[i] = (int32_t)in[i];
}

// Register path for the common case (<= 256 entries; a radius query at the c5 shape returns ~43): one warp per segment, R
// 32-bit values per lane (element i = r * 32 + lane), bitonic network by __shfl_xor (partner in another lane) or a register
// swap (partner in the same lane); no shared memory, no barriers.  Sorting values are the ids themselves, or -- BY_KEY --
// the keys key_of_id[id], which must then be a permutation of 0..key_limit-1 (kd pre-order ranks are): the sorted keys are
// mapped back through id_of_key.  Longer segments go to seg_sort_mid_kernel or are counted for the global radix sort.
template <int R>
__device__ __forceinline__ void warp_bitonic_u32(uint32_t (&v)[R], int lane, int np2) {
#pragma unroll
  for (int k = 2; k <= 32 * R; k <<= 1) {
    if (k > np2) break;
#pragma unroll
    for (int j = k >> 1; j > 0; j >>= 1) {
      if (j >= 32) {
        const int jr = j >> 5;
#pragma unroll
        for (int r = 0; r < R; ++r)
          if ((r & jr) == 0) {
            const bool up = (((r << 5) & k) == 0);
            const uint32_t a = v[r], b = v[r | jr];
            const uint32_t lo = min(a, b), hi = max(a, b);
            v[r] = up ? lo : hi; v[r | jr] = up ? hi : lo;
          }
      } else {
        const bool lower = (lane & j) == 0;
#pragma unroll
        for (int r = 0; r < R; ++r) {
          const bool up = ((((r << 5) | lane) & k) == 0);
          const uint32_t other = __shfl_xor_sync(0xffffffffu, v[r], j);
          v[r] = (lower == up) ? min(v[r], other) : max(v[r], other);
        }
      }
    }
  }
}
template <int R, bool BY_KEY>
__device__ __forceinline__ void seg_sort_regs(int32_t* __restrict__ seg_ids, int len, int lane, const int32_t* __restrict__ key_of_id,
                                              const int32_t* __restrict__ id_of_key) {
  uint32_t v[R];
#pragma unroll
  for (int r = 0; r < R; ++r) {
    const int i = r * 32 + lane;
    v[r] = 0xffffffffu;
    if (i < len) { const int32_t id = seg_ids[i]; v[r] = BY_KEY ? (uint32_t)key_of_id[id] : (uint32_t)id; }
  }
  int np2 = 2;
  while (np2 < len) np2 <<= 1;
  warp_bitonic_u32<R>(v, lane, np2);
#pragma unroll
  for (int r = 0; r < R; ++r) {
    const int i = r * 32 + lane;
    if (i < len) seg_ids[i] = BY_KEY ? id_of_key[v[r]] : (int32_t)v[r];
  }
}
#define SEG_REG_WARPS 8
#define SEG_REG_CAP 256
#define SEG_MID_CAP 4096
template <bool BY_KEY>
__global__ void __launch_bounds__(SEG_REG_WARPS * 32) seg_sort_reg_kernel(const int64_t* __restrict__ offsets, int64_t m, int32_t* __restrict__ ids,
                                                                          const int32_t* __restrict__ key_of_id, const int32_t* __restrict__ id_of_key,
                                                                          int32_t* __restrict__ n_mid_big, int32_t* __restrict__ mid_list,
                                                                          const int32_t* __restrict__ seg_list /* nullable: m listed segments */) {
  const int lane = threadIdx.x & 31;
  const int64_t slot = (int64_t)blockIdx.x * SEG_REG_WARPS + (threadIdx.x >> 5);
  if (slot >= m) return;
  const int64_t seg = seg_list ? seg_list[slot] : slot;
  const int64_t s = offsets[seg];
  const int64_t len64 = offsets[seg + 1] - s;
  if (len64 <= 1) return;
  if (len64 > SEG_REG_CAP) {   // 257..SEG_MID_CAP: listed for the block kernel below; longer: counted for the global radix sort
    if (lane == 0) {
      if (len64 > SEG_MID_CAP) atomicAdd(&n_mid_big[1], 1);
      else mid_list[atomicAdd(&n_mid_big[0], 1)] = (int32_t)seg;
    }
    return;
  }
  const int len = (int)len64;
  if (len <= 32) seg_sort_regs<1, BY_KEY>(ids + s, len, lane, key_of_id, id_of_key);
  else if (len <= 64) seg_sort_regs<2, BY_KEY>(ids + s, len, lane, key_of_id, id_of_key);
  else if (len <= 128) seg_sort_regs<4, BY_KEY>(ids + s, len, lane, key_of_id, id_of_key);
  else seg_sort_regs<8, BY_KEY>(ids + s, len, lane, key_of_id, id_of_key);
}
// 257..4096 entries (the early rows of a PRM's late lists, wide radius queries): one block per listed segment, bitonic network
// on 32-bit values in shared memory
template <bool BY_KEY>
__global__ void __launch_bounds__(256) seg_sort_mid_kernel(const int64_t* __restrict__ offsets, const int32_t* __restrict__ mid_list,
                                                           int32_t* __restrict__ ids, const int32_t* __restrict__ key_of_id,
                                                           const int32_t* __restrict__ id_of_key) {
  __shared__ uint32_t s_v[SEG_MID_CAP];
  const int64_t seg = mid_list[blockIdx.x];
  const int64_t s = offsets[seg];
  const int len = (int)(offsets[seg + 1] - s);
  int np2 = 512;
  while (np2 < len) np2 <<= 1;
  for (int i = threadIdx.x; i < np2; i += 256) {
    uint32_t v = 0xffffffffu;
    if (i < len) { const int32_t id = ids[s + i]; v = BY_KEY ? (uint32_t)key_of_id[id] : (uint32_t)id; }
    s_v[i] = v;
  }
  __syncthreads();
  for (int k = 2; k <= np2; k <<= 1)
    for (int j = k >> 1; j > 0; j >>= 1) {
      for (int t = threadIdx.x; t < (np2 >> 1); t += 256) {
        const int i = ((t & ~(j - 1)) << 1) | (t & (j - 1));
        const int p = i | j;
        const uint32_t a = s_v[i], b = s_v[p];
        if ((a > b) == ((i & k) == 0)) { s_v[i] = b; s_v[p] = a; }
      }
      __syncthreads();
    }
  for (int i = threadIdx.x; i < len; i += 256) ids[s + i] = BY_KEY ? id_of_key[s_v[i]] : (int32_t)s_v[i];
}
__global__ void invert_perm_kernel(const int32_t* __restrict__ key_of_id, int64_t n, int32_t* __restrict__ id_of_key) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) id_of_key[key_of_id[i]] = (int32_t)i;
}

// key_limit: all keys (ids or key_of_id values) are < key_limit; key_of_id (if given) is a permutation of 0..key_limit-1
// A handful of device counters for the host WITHOUT the copy engine: a one-warp kernel stores them into pinned host memory (mapped
// under unified addressing), the stream is synchronised, the host reads them.  A cudaMemcpyAsync of 8 bytes would queue behind
// whatever the D2H engine is busy with -- the PRM build's 50 MB result blocks held every per-block segment sort up for a millisecond.
__global__ void flags_to_host_kernel(const int32_t* __restrict__ d, int n, volatile int32_t* h) {
  if ((int)threadIdx.x < n) h[threadIdx.x] = d[threadIdx.x];
}
int32_t read_flags_dev(porrt_ctx* ctx, const int32_t* flags_dev, int n, int32_t* out, cudaStream_t st) {
  CUDA_TRY(ctx, ctx->pin_flags.ensure(64));
  volatile int32_t* h = ctx->pin_flags.as<int32_t>();
  flags_to_host_kernel<<<1, 32, 0, st>>>(flags_dev, n, h);
  LAUNCH_CHECK(ctx);
  CUDA_TRY(ctx, cudaStreamSynchronize(st));
  for (int k = 0; k < n; ++k) out[k] = h[k];
  return PORRT_OK;
}

int32_t segments_sort_by_key_dev(porrt_ctx* ctx, const int64_t* offsets_dev, int64_t m, int32_t* ids_dev, const int32_t* key_of_id_dev, int64_t key_limit,
                                 const int32_t* seg_list_dev, int64_t n_listed) {
  // seg_list_dev (nullable): only the n_listed segments named there need sorting (of m segments in all); the rare global radix
  // path ignores the list and sorts everything, which is harmless
  cudaStream_t st = ctx->stream;
  if (m <= 0 || (seg_list_dev && n_listed <= 0)) return PORRT_OK;
  const int64_t m_run = seg_list_dev ? n_listed : m;
  int32_t* d_big;   // [0] n_mid (257..4096, listed), [1] n_big (longer)
  int32_t* d_mid_list;
  int32_t* d_inv = nullptr;
  CUDA_TRY(ctx, carve(ctx->ws_seg, [&](Carve& c) {
    d_big = c.take<int32_t>(4);
    d_mid_list = c.take<int32_t>(m);
    if (key_of_id_dev) d_inv = c.take<int32_t>(key_limit);
  }));
  CUDA_TRY(ctx, cudaMemsetAsync(d_big, 0, 8, st));
  if (key_of_id_dev) {
    invert_perm_kernel<<<div_up(key_limit, 256), 256, 0, st>>>(key_of_id_dev, key_limit, d_inv);
    LAUNCH_CHECK(ctx);
    seg_sort_reg_kernel<true><<<div_up(m_run, SEG_REG_WARPS), SEG_REG_WARPS * 32, 0, st>>>(offsets_dev, m_run, ids_dev, key_of_id_dev, d_inv, d_big, d_mid_list, seg_list_dev);
  } else {
    seg_sort_reg_kernel<false><<<div_up(m_run, SEG_REG_WARPS), SEG_REG_WARPS * 32, 0, st>>>(offsets_dev, m_run, ids_dev, nullptr, nullptr, d_big, d_mid_list, seg_list_dev);
  }
  LAUNCH_CHECK(ctx);
  int32_t cnt[2] = {0, 0};
  { const int32_t rcf = read_flags_dev(ctx, d_big, 2, cnt, st); if (rcf) return rcf; }
  const int32_t n_mid = cnt[0], n_big = cnt[1];
  if (n_mid > 0 && n_big == 0) {
    if (key_of_id_dev) seg_sort_mid_kernel<true><<<n_mid, 256, 0, st>>>(offsets_dev, d_mid_list, ids_dev, key_of_id_dev, d_inv);
    else seg_sort_mid_kernel<false><<<n_mid, 256, 0, st>>>(offsets_dev, d_mid_list, ids_dev, nullptr, nullptr);
    LAUNCH_CHECK(ctx);
  }
  if (n_big == 0) return PORRT_OK;
  int64_t total = 0;
  CUDA_TRY(ctx, cudaMemcpyAsync(&total, offsets_dev + m, 8, cudaMemcpyDeviceToHost, st));
  CUDA_TRY(ctx, cudaStreamSynchronize(st));
  if (total <= 1) return PORRT_OK;
  // some segment is longer than SEG_MID_CAP: one global stable LSD radix sort on (segment, key) orders them all
  const int key_bits = bits_for((uint64_t)(key_limit > 1 ? key_limit - 1 : 1));
  const int seg_bits = bits_for((uint64_t)(m > 1 ? m - 1 : 1));
  CUDA_TRY(ctx, ctx->sort_keys.ensure((size_t)total * 8));
  CUDA_TRY(ctx, ctx->sort_vals.ensure((size_t)total * 4));
  uint64_t* keys = ctx->sort_keys.as<uint64_t>();
  uint32_t* vals = ctx->sort_vals.as<uint32_t>();
  seg_key_kernel<<<div_up(m * 32, 256), 256, 0, st>>>(offsets_dev, m, ids_dev, key_of_id_dev, key_bits, keys, vals);
  LAUNCH_CHECK(ctx);
  int32_t rc = radix_sort_pairs(ctx, keys, vals, total, key_bits + seg_bits);
  if (rc) return rc;
  copy_u32_i32_kernel<<<div_up(total, 256), 256, 0, st>>>(vals, total, ids_dev);
  LAUNCH_CHECK(ctx);
  return PORRT_OK;
}

PORRT_API int32_t porrt_radius_query(porrt_ctx* ctx, const double* q_xy, const double* radius, int64_t m,
                                     const uint32_t* prefix_limit, const uint64_t* reach_mask, int32_t reach_words, const uint32_t* world,
                                     int64_t* out_offsets, int32_t* out_ids, int64_t cap, int64_t* out_total) {
  CTX_CHECK(ctx);
  if (ctx->n_vertices <= 0) return porrt_fail(ctx, PORRT_ERR_NO_VERTICES, "no vertex set");
  if (m < 0 || (m > 0 && (!q_xy || !radius || !out_offsets)) || (reach_mask && (!world || reach_words < 1)))
    return porrt_fail(ctx, PORRT_ERR_INVALID_ARG, "radius_query: bad arguments");
  CUDA_TRY(ctx, cudaSetDevice(ctx->device));
  { const int32_t rcf = nn_flush_appended(ctx); if (rcf) return rcf; }
  ctx->reach_words = reach_mask ? reach_words : 1;
  const size_t reach_bytes = reach_mask ? (size_t)ctx->n_vertices * 8 * (size_t)reach_words : 0;
  CUDA_TRY(ctx, cudaSetDevice(ctx->device));
  cudaStream_t st = ctx->stream;
  if (m == 0) { if (out_offsets) out_offsets[0] = 0; if (out_total) *out_total = 0; return PORRT_OK; }
  const int64_t V = ctx->n_vertices;
  double *d_q, *d_r;
  int64_t* d_off;
  uint64_t* d_reach = nullptr;
  uint32_t* d_prefix = nullptr; uint32_t* d_world = nullptr;
  CUDA_TRY(ctx, carve(ctx->ws_main, [&](Carve& c) {
    d_q = c.take<double>((size_t)m * 2);
    d_r = c.take<double>(m);
    d_off = c.take<int64_t>(m + 1);
    if (reach_mask) d_reach = c.take<uint64_t>(reach_bytes / 8);
    if (prefix_limit) d_prefix = c.take<uint32_t>(m);
    if (world) d_world = c.take<uint32_t>(m);
  }));
  CUDA_TRY(ctx, cudaMemcpyAsync(d_q, q_xy, (size_t)m * 16, cudaMemcpyHostToDevice, st));
  CUDA_TRY(ctx, cudaMemcpyAsync(d_r, radius, (size_t)m * 8, cudaMemcpyHostToDevice, st));
  if (d_prefix) CUDA_TRY(ctx, cudaMemcpyAsync(d_prefix, prefix_limit, (size_t)m * 4, cudaMemcpyHostToDevice, st));
  if (d_world) CUDA_TRY(ctx, cudaMemcpyAsync(d_world, world, (size_t)m * 4, cudaMemcpyHostToDevice, st));
  if (d_reach) CUDA_TRY(ctx, cudaMemcpyAsync(d_reach, reach_mask, reach_bytes, cudaMemcpyHostToDevice, st));
  int64_t total = 0;
  tstart(ctx);  // phases: [count+scan+fill, order restore, D2H]
  int32_t rc = nn_radius_count_fill_dev(ctx, d_q, d_r, m, d_prefix, d_reach, d_world, d_off, &ctx->ws_table, &total, nullptr, true);
  if (rc) return rc;
  tmark(ctx);
  if (out_total) *out_total = total;
  if (total > cap || (total > 0 && !out_ids)) {
    CUDA_TRY(ctx, cudaMemcpyAsync(out_offsets, d_off, (size_t)(m + 1) * 8, cudaMemcpyDeviceToHost, st));
    CUDA_TRY(ctx, cudaStreamSynchronize(st));
    return porrt_fail(ctx, PORRT_ERR_CAPACITY, "radius_query: out_ids too small");
  }
  tmark(ctx);   // (the id order comes out of the search itself now; the phase is kept so that the list keeps its three entries)
  CUDA_TRY(ctx, cudaMemcpyAsync(out_offsets, d_off, (size_t)(m + 1) * 8, cudaMemcpyDeviceToHost, st));
  if (total > 0) CUDA_TRY(ctx, cudaMemcpyAsync(out_ids, ctx->ws_table.p, (size_t)total * 4, cudaMemcpyDeviceToHost, st));
  tmark(ctx);
  CUDA_TRY(ctx, cudaStreamSynchronize(st));
  tfinish(ctx);
  return PORRT_OK;
}

// ================================================================================================ nearest / k-NN
// ring search around the query's cell; exact: stops only when every unvisited cell is provably farther.
#define KNN_THREADS 64
// the k best of one thread's query, ascending by (d2, id); entry j lives at [j][thread] of two shared arrays (a register
// array indexed by a runtime position would be spilled to local memory: measured 0.3 ms for 574 fallback queries)
template <int KMAX>
struct TopK {
  double (*d2)[KNN_THREADS];
  int32_t (*id)[KNN_THREADS];
  int k, cnt, t;
  __device__ __forceinline__ void init(int kk, double (*sd)[KNN_THREADS], int32_t (*si)[KNN_THREADS]) { k = kk; cnt = 0; d2 = sd; id = si; t = threadIdx.x; }
  __device__ __forceinline__ double worst() const { return cnt < k ? INFINITY : d2[k - 1][t]; }
  __device__ __forceinline__ double dist_at(int j) const { return d2[j][t]; }
  __device__ __forceinline__ int32_t id_at(int j) const { return id[j][t]; }
  __device__ __forceinline__ void push(double d, int32_t i) {
    if (cnt == k && !(d < d2[k - 1][t] || (d == d2[k - 1][t] && i < id[k - 1][t]))) return;
    int pos = cnt < k ? cnt : k - 1;
    while (pos > 0 && (d < d2[pos - 1][t] || (d == d2[pos - 1][t] && i < id[pos - 1][t]))) {
      d2[pos][t] = d2[pos - 1][t]; id[pos][t] = id[pos - 1][t]; --pos;
    }
    d2[pos][t] = d; id[pos][t] = i;
    if (cnt < k) ++cnt;
  }
};

template <int KMAX>
__global__ void __launch_bounds__(KNN_THREADS) knn_kernel(GridDev g, const double2* __restrict__ q, int64_t m, int k,
                                                  const uint64_t* __restrict__ reach, const uint32_t* __restrict__ world,
                                                  int32_t* __restrict__ out_ids, double* __restrict__ out_dist, int32_t* __restrict__ out_ties,
                                                  const int32_t* __restrict__ list) {
  int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= m) return;
  if (list) t = list[t];   // m = length of the list: the queries nn_tile.cu left to the exact ring search
  const double2 p = q[t];
  __shared__ double s_d2[KMAX][KNN_THREADS];
  __shared__ int32_t s_id[KMAX][KNN_THREADS];
  TopK<KMAX> top;
  top.init(k, s_d2, s_id);
  int32_t ties = 0;  // KMAX == 1 only: vertices at exactly the winning d2
  const uint32_t wq = (reach && world) ? world[t] : 0u;
  if (p.x == p.x && p.y == p.y) {
    const int cx = cell_coord(p.x, g.org_x, g.inv_cell, g.cells_x), cy = cell_coord(p.y, g.org_y, g.inv_cell, g.cells_y);
    const int maxR = max(max(cx, g.cells_x - 1 - cx), max(cy, g.cells_y - 1 - cy));
    for (int R = 0; R <= maxR; ++R) {
      for (int dy = -R; dy <= R; ++dy) {
        const int yy = cy + dy;
        if (yy < 0 || yy >= g.cells_y) continue;
        const bool full_row = (dy == -R || dy == R);
        for (int side = 0; side < (full_row || R == 0 ? 1 : 2); ++side) {
          int x0, x1;
          if (full_row || R == 0) { x0 = max(cx - R, 0); x1 = min(cx + R, g.cells_x - 1); }
          else { x0 = x1 = side ? cx + R : cx - R; if (x0 < 0 || x0 >= g.cells_x) continue; }
          const int64_t s = g.cell_start[(int64_t)yy * g.cells_x + x0], e = g.cell_start[(int64_t)yy * g.cells_x + x1 + 1];
          for (int64_t kk = s; kk < e; ++kk) {
            const double d = dist2(g.vxy[kk], p.x, p.y);
            if (d <= top.worst() || top.cnt < k) {
              const int32_t id = g.vid[kk];
              if (!reach || reach_bit(reach, g.reach_words, id, wq)) {
                if (KMAX == 1) {
                  if (top.cnt == 0 || d < top.dist_at(0)) ties = 1;
                  else if (d == top.dist_at(0)) ++ties;
                }
                if (d == d) top.push(d, id);
              }
            }
          }
        }
      }
      if (top.cnt == k && top.worst() < ring_lower_bound2(g, p.x, p.y, cx, cy, R)) break;
    }
  }
  for (int j = 0; j < k; ++j) {
    const bool ok = j < top.cnt;
    out_ids[t * k + j] = ok ? top.id_at(j) : -1;
    if (out_dist) out_dist[t * k + j] = ok ? __dsqrt_rn(top.dist_at(j)) : INFINITY;
  }
  if (KMAX == 1 && out_ties) out_ties[t] = ties;
}

// One WARP per query, for the few queries nn_tile.cu could not certify (sparse neighbourhoods: a wider ring is needed).  The
// thread-per-query kernel above is latency bound there (one thread walks ~350 candidates through global memory: 0.3 ms for
// 574 queries).  Lanes stride the candidates of every run of the ring, each lane keeps its own sorted list; after a ring the k
// globally best are drawn from the 32 list heads (k warp-wide arg-min rounds) to test the stopping rule, and once more to write.
template <int KMAX>
__global__ void __launch_bounds__(KNN_THREADS) knn_warp_kernel(GridDev g, const double2* __restrict__ q, int64_t m, int k,
                                                               const uint64_t* __restrict__ reach, const uint32_t* __restrict__ world,
                                                               int32_t* __restrict__ out_ids, double* __restrict__ out_dist,
                                                               int32_t* __restrict__ out_ties, const int32_t* __restrict__ list) {
  __shared__ double s_d2[KMAX][KNN_THREADS];
  __shared__ int32_t s_id[KMAX][KNN_THREADS];
  const int lane = threadIdx.x & 31;
  const int64_t wslot = ((int64_t)blockIdx.x * KNN_THREADS + threadIdx.x) >> 5;
  if (wslot >= m) return;                    // whole warps leave together
  const int64_t t = list ? list[wslot] : wslot;
  const double2 p = q[t];
  TopK<KMAX> top;
  top.init(k, s_d2, s_id);
  int32_t ties = 0;                          // k == 1: vertices at exactly this lane's best d2
  const uint32_t wq = (reach && world) ? world[t] : 0u;
  // k rounds of "smallest (d2, id) among the lane heads"; returns the k-th best d2 (inf if fewer than k exist) and, when
  // `write`, stores the sorted result
  auto draw = [&](bool write) -> double {
    int head = 0, found = 0;
    double kth = INFINITY;
    for (int j = 0; j < k; ++j) {
      double d = head < top.cnt ? top.dist_at(head) : INFINITY;
      int32_t id = head < top.cnt ? top.id_at(head) : 0x7fffffff;
      int src = lane;
#pragma unroll
      for (int o = 16; o; o >>= 1) {
        const double od = __shfl_xor_sync(0xffffffffu, d, o);
        const int32_t oi = __shfl_xor_sync(0xffffffffu, id, o);
        const int os = __shfl_xor_sync(0xffffffffu, src, o);
        if (od < d || (od == d && oi < id)) { d = od; id = oi; src = os; }
      }
      const bool any = d < INFINITY || id != 0x7fffffff;
      if (any) { ++found; kth = d; if (src == lane) ++head; }
      if (write && lane == 0) {
        out_ids[t * k + j] = any ? id : -1;
        if (out_dist) out_dist[t * k + j] = any ? __dsqrt_rn(d) : INFINITY;
      }
    }
    return found == k ? kth : INFINITY;
  };
  if (p.x == p.x && p.y == p.y) {
    const int cx = cell_coord(p.x, g.org_x, g.inv_cell, g.cells_x), cy = cell_coord(p.y, g.org_y, g.inv_cell, g.cells_y);
    const int maxR = max(max(cx, g.cells_x - 1 - cx), max(cy, g.cells_y - 1 - cy));
    for (int R = 0; R <= maxR; ++R) {
      for (int dy = -R; dy <= R; ++dy) {
        const int yy = cy + dy;
        if (yy < 0 || yy >= g.cells_y) continue;
        const bool full_row = (dy == -R || dy == R);
        for (int side = 0; side < (full_row || R == 0 ? 1 : 2); ++side) {
          int x0, x1;
          if (full_row || R == 0) { x0 = max(cx - R, 0); x1 = min(cx + R, g.cells_x - 1); }
          else { x0 = x1 = side ? cx + R : cx - R; if (x0 < 0 || x0 >= g.cells_x) continue; }
          const int64_t s = g.cell_start[(int64_t)yy * g.cells_x + x0], e = g.cell_start[(int64_t)yy * g.cells_x + x1 + 1];
          for (int64_t kk = s + lane; kk < e; kk += 32) {
            const double d = dist2(g.vxy[kk], p.x, p.y);
            if (d <= top.worst() || top.cnt < k) {
              const int32_t id = g.vid[kk];
              if (!reach || reach_bit(reach, g.reach_words, id, wq)) {
                if (KMAX == 1) {
                  if (top.cnt == 0 || d < top.dist_at(0)) ties = 1;
                  else if (d == top.dist_at(0)) ++ties;
                }
                if (d == d) top.push(d, id);
              }
            }
          }
        }
      }
      if (draw(false) < ring_lower_bound2(g, p.x, p.y, cx, cy, R)) break;   // warp-uniform
    }
  }
  const double best = draw(true);
  if (KMAX == 1 && out_ties) {               // ties of the lanes whose own best is the global best
    int32_t tt = (top.cnt > 0 && top.dist_at(0) == best) ? ties : 0;
#pragma unroll
    for (int o = 16; o; o >>= 1) tt += __shfl_xor_sync(0xffffffffu, tt, o);
    if (lane == 0) out_ties[t] = best < INFINITY ? tt : 0;
  }
}

static int32_t knn_host(porrt_ctx* ctx, const double* q_xy, int64_t m, int k, const uint64_t* reach_mask, int32_t reach_words,
                        const uint32_t* world, int32_t* out_ids, double* out_dist, int32_t* out_ties) {
  if (ctx->n_vertices <= 0) return porrt_fail(ctx, PORRT_ERR_NO_VERTICES, "no vertex set");
  if (m < 0 || (m > 0 && (!q_xy || !out_ids)) || k < 1 || k > 32 || (reach_mask && (!world || reach_words < 1)))
    return porrt_fail(ctx, PORRT_ERR_INVALID_ARG, "nearest/knn: bad arguments (1 <= k <= 32)");
  if (m == 0) return PORRT_OK;
  CUDA_TRY(ctx, cudaSetDevice(ctx->device));
  { const int32_t rcf = nn_flush_appended(ctx); if (rcf) return rcf; }
  ctx->reach_words = reach_mask ? reach_words : 1;
  const size_t reach_bytes = reach_mask ? (size_t)ctx->n_vertices * 8 * (size_t)reach_words : 0;
  CUDA_TRY(ctx, cudaSetDevice(ctx->device));
  cudaStream_t st = ctx->stream;
  const int64_t V = ctx->n_vertices;
  double *d_q, *d_dist;
  uint64_t* d_reach = nullptr;
  int32_t *d_ids, *d_ties;
  uint32_t* d_world = nullptr;
  CUDA_TRY(ctx, carve(ctx->ws_main, [&](Carve& c) {
    d_q = c.take<double>((size_t)m * 2);
    d_dist = c.take<double>((size_t)m * k);
    if (reach_mask) d_reach = c.take<uint64_t>(reach_bytes / 8);
    d_ids = c.take<int32_t>((size_t)m * k);
    d_ties = c.take<int32_t>(m);
    if (world) d_world = c.take<uint32_t>(m);
  }));
  CUDA_TRY(ctx, cudaMemcpyAsync(d_q, q_xy, (size_t)m * 16, cudaMemcpyHostToDevice, st));
  if (d_world) CUDA_TRY(ctx, cudaMemcpyAsync(d_world, world, (size_t)m * 4, cudaMemcpyHostToDevice, st));
  if (d_reach) CUDA_TRY(ctx, cudaMemcpyAsync(d_reach, reach_mask, reach_bytes, cudaMemcpyHostToDevice, st));
  GridDev g = grid_dev(ctx);
  tstart(ctx);  // phases: [kernel, D2H]
  int64_t m_run = m;
  const int32_t* list = nullptr;
  if (nn_tile_usable(ctx, m)) {   // TMA-staged tiles, thread per query; whoever needs a wider ring comes back in the list
    int32_t fb_n = 0;
    int32_t rc = nn_tile_knn(ctx, g, d_q, m, k, d_reach, d_world, d_ids, d_dist, k == 1 ? d_ties : nullptr, &list, &fb_n);
    if (rc) return rc;
    m_run = fb_n;
  }
  if (m_run > 0 && list && m_run <= 65536) {   // few hard queries left by the tiles: a warp each
    const int blocks = div_up(m_run * 32, KNN_THREADS);
    if (k == 1) knn_warp_kernel<1><<<blocks, KNN_THREADS, 0, st>>>(g, (const double2*)d_q, m_run, 1, d_reach, d_world, d_ids, d_dist, d_ties, list);
    else if (k <= 8) knn_warp_kernel<8><<<blocks, KNN_THREADS, 0, st>>>(g, (const double2*)d_q, m_run, k, d_reach, d_world, d_ids, d_dist, nullptr, list);
    else knn_warp_kernel<32><<<blocks, KNN_THREADS, 0, st>>>(g, (const double2*)d_q, m_run, k, d_reach, d_world, d_ids, d_dist, nullptr, list);
    LAUNCH_CHECK(ctx);
  } else if (m_run > 0) {
    if (k == 1) knn_kernel<1><<<div_up(m_run, KNN_THREADS), KNN_THREADS, 0, st>>>(g, (const double2*)d_q, m_run, 1, d_reach, d_world, d_ids, d_dist, d_ties, list);
    else if (k <= 8) knn_kernel<8><<<div_up(m_run, KNN_THREADS), KNN_THREADS, 0, st>>>(g, (const double2*)d_q, m_run, k, d_reach, d_world, d_ids, d_dist, nullptr, list);
    else knn_kernel<32><<<div_up(m_run, KNN_THREADS), KNN_THREADS, 0, st>>>(g, (const double2*)d_q, m_run, k, d_reach, d_world, d_ids, d_dist, nullptr, list);
    LAUNCH_CHECK(ctx);
  }
  tmark(ctx);
  CUDA_TRY(ctx, cudaMemcpyAsync(out_ids, d_ids, (size_t)m * k * 4, cudaMemcpyDeviceToHost, st));
  if (out_dist) CUDA_TRY(ctx, cudaMemcpyAsync(out_dist, d_dist, (size_t)m * k * 8, cudaMemcpyDeviceToHost, st));
  if (out_ties && k == 1) CUDA_TRY(ctx, cudaMemcpyAsync(out_ties, d_ties, (size_t)m * 4, cudaMemcpyDeviceToHost, st));
  tmark(ctx);
  CUDA_TRY(ctx, cudaStreamSynchronize(st));
  tfinish(ctx);
  return PORRT_OK;
}

PORRT_API int32_t porrt_nearest(porrt_ctx* ctx, const double* q_xy, int64_t m, const uint64_t* reach_mask, int32_t reach_words,
                                const uint32_t* world, int32_t* out_id, double* out_dist, int32_t* out_ties) {
  CTX_CHECK(ctx);
  return knn_host(ctx, q_xy, m, 1, reach_mask, reach_words, world, out_id, out_dist, out_ties);
}
PORRT_API int32_t porrt_knn(porrt_ctx* ctx, const double* q_xy, int64_t m, int32_t k, int32_t* out_ids, double* out_dist) {
  CTX_CHECK(ctx);
  return knn_host(ctx, q_xy, m, k, nullptr, 1, nullptr, out_ids, out_dist, nullptr);
}
