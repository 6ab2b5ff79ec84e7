// nn_dev.cuh -- device-side pieces shared by the nearest-neighbour kernels (nn.cu: thread per query; nn_tile.cu: TMA-staged
// vertex tiles, warp per query): the cell grid, the reference's distance arithmetic and the exact radius threshold.
#pragma once
#include <cfloat>

#include "common.cuh"

struct GridDev {
  const double2* vxy;       // cell-sorted vertex coordinates
  const int32_t* vid;       // their ids
  const int64_t* cell_start;  // [cells_x*cells_y + 1]
  double org_x, org_y, inv_cell, cell;
  int32_t cells_x, cells_y;
  int64_t n;
  int32_t reach_words;      // u64 words per vertex of the reachability filter of the running call (pto_reachability.rs: one bit per world)
};

// the validator closure of pto.rs:74-77: bit `w` of vertex id's reachability mask (BitVec Lsb0: bit w of word w / 64).
// A world beyond the mask passes nothing (the reference's BitVec index would panic).
__device__ __forceinline__ bool reach_bit(const uint64_t* __restrict__ reach, int words, int32_t id, uint32_t w) {
  if ((w >> 6) >= (uint32_t)words) return false;
  return (reach[(int64_t)id * words + (w >> 6)] >> (w & 63u)) & 1ull;
}

__device__ __forceinline__ int cell_coord(double v, double org, double inv_cell, int n_cells) {
  double c = floor(__dmul_rn(__dsub_rn(v, org), inv_cell));
  if (!(c > 0.0)) return 0;
  if (c >= (double)(n_cells - 1)) return n_cells - 1;
  return (int)c;
}

// T(r) = max{ t : sqrt_rn(t) <= r }  (SURVEY 8(g) note 3): the reference tests `norm2(..) <= radius` on the sqrt-ed value.
// A finite r whose square overflows gets DBL_MAX, not +inf: an overflowed d2 (+inf) has sqrt +inf > r, so it must not pass.
__device__ __forceinline__ double radius_threshold(double r) {
  if (!(r >= 0.0)) return -1.0;  // negative or NaN radius: nothing passes `d <= radius`
  double t = __dmul_rn(r, r);
  if (isinf(t)) return isinf(r) ? t : DBL_MAX;
  while (t > 0.0 && __dsqrt_rn(t) > r) t = __longlong_as_double(__double_as_longlong(t) - 1);
  for (;;) {
    double u = __longlong_as_double(__double_as_longlong(t) + 1);
    if (isfinite(u) && __dsqrt_rn(u) <= r) t = u; else break;
  }
  return t;
}

__device__ __forceinline__ double dist2(double2 v, double qx, double qy) {
  double dx = __dsub_rn(qx, v.x), dy = __dsub_rn(qy, v.y);
  return __dadd_rn(__dmul_rn(dx, dx), __dmul_rn(dy, dy));  // 0.0 + dx*dx is exact, so this is the reference's sum
}

__device__ __forceinline__ double ring_lower_bound2(const GridDev& g, double qx, double qy, int cx, int cy, int R) {
  // squared distance from q to the nearest point outside the square of cells [cx-R,cx+R] x [cy-R,cy+R];
  // sides beyond the grid have nothing behind them.  Cell membership comes from cell_coord's floor((v - org) * inv_cell), the side
  // from org + c * cell: the two disagree by a few ulps of the coordinates' magnitude (at cell 0.1, x = 0.3 lies in cell 3 while
  // 3 * 0.1 = 0.30000000000000004), which can exceed the whole bound of a query next to a side.  The bound is therefore lowered by
  // an absolute margin, 1e-14 of the largest magnitude in play (coordinates, origin, grid extent) -- also covering the rounding of
  // the subtractions below.
  double lb = INFINITY;
  if (cx - R > 0) lb = fmin(lb, qx - (g.org_x + (double)(cx - R) * g.cell));
  if (cx + R < g.cells_x - 1) lb = fmin(lb, (g.org_x + (double)(cx + R + 1) * g.cell) - qx);
  if (cy - R > 0) lb = fmin(lb, qy - (g.org_y + (double)(cy - R) * g.cell));
  if (cy + R < g.cells_y - 1) lb = fmin(lb, (g.org_y + (double)(cy + R + 1) * g.cell) - qy);
  if (isinf(lb)) return INFINITY;
  lb -= 1e-14 * (fabs(qx) + fabs(qy) + fabs(g.org_x) + fabs(g.org_y) + (double)(g.cells_x + g.cells_y) * g.cell);
  if (!(lb > 0.0)) return 0.0;
  return lb * lb;
}

