// map.cu -- occupancy-grid validity kernels (SURVEY.md 8(a) rows A1-A5).
//
// Replaces, batched:  Map::to_pixel_coordinates / is_state_valid / get_traversed_space / observe_impl's
// line-of-sight test (reference src/map_io.rs:165-241,281-300) and the MapShelfDomain equivalents
// (src/map_shelves_io.rs:150-203,259-265), plus line_drawing::Bresenham (crate line_drawing 0.8).
//
// HBM layout: ONE fused code byte per pixel (occupancy + zone id), stored in 128-byte tiles of 16 x 8 px made of
// four 32-byte sectors of 8 x 4 px, so that a 32-pixel stretch of a line touches ~3 cache lines whatever its
// direction (a row-major grid costs up to 32 lines for a vertical stretch).
//   DOOR : 255 free | 0 obstacle | 1..253 zone id + 1 | 254 gray pixel without zone id (reference panics)
//   SHELF: the raw gray value (class = 255 free, 127..254 low obstacle, 0..126 high obstacle)
//
// This file holds the map upload (fused grid, zone positions, world validities, and the class data of both edge kernels),
// the state-validity and visibility kernels, the large-map edge kernel (class bytes in global memory, for maps whose class
// plane does not fit in shared memory; the product's edge kernel is edge3.cu), the dispatch between the two edge kernels,
// and the chunked host-buffer pipeline behind every host-array edge entry point.
#include "common.cuh"
#include "map_dev.cuh"

// ------------------------------------------------------------------------------------------------ kernels
#define EDGE_BLOCK 256

// ================================================================================================ edge validity, large maps
// The product's edge kernel is edge3.cu (class plane staged in shared memory).  Maps whose class plane does not fit in shared
// memory (> ~14000^2 px) take this kernel instead: the same strip decomposition with the class bytes read from global memory
// and per-pixel resolution of mixed strips on the fused byte grid.  INDEXED: endpoints are gathered from a vertex buffer,
// from[e] = xy[from_idx[e]], to[e] = xy[to_idx[e]].
// One CLASS byte per BS x BS block (all free / all obstacle / all low / needs-per-pixel [+ contains gray]) and cuts the line into strips of <= BS
// pixels aligned to the block grid along the major axis; a strip touches at most two blocks (slope <= 1 in octant
// space), so two class bytes settle it unless a block is mixed.  Only mixed strips are queued (shared memory) and
// resolved per pixel afterwards, 32/BS strips per warp round, and strips of edges already known to be blocked are
// dropped.  Work is flattened: the strips of the warp's 32 edges form one sequence that is cut into 32 equal
// contiguous shares, one per lane, so lanes stay busy whatever the mix of edge lengths.
// Exactness: any_obstacle / any_low / zone min-max are order-free reductions; whenever order could matter (two
// different zones, a gray pixel without zone id, an end point outside the map) the edge is re-walked sequentially.
#define C_OBST 1   // every pixel of the block is obstacle (DOOR: 0, SHELF: < 127)          == F_OBST
#define C_LOW 2    // SHELF: every pixel is a low obstacle (127..254)                       == F_LOW
#define C_FINE 4   // block is not uniform: look at the pixels
#define C_GRAY 8   // DOOR: block contains gray pixels (zone ids needed) -- implies C_FINE

#define F_OBST 1
#define F_LOW 2


template <int KIND>
__global__ void coarse_build_kernel(const uint8_t* __restrict__ grid, int H, int W, int tiles_x, int log_bs, int cw, int ch,
                                    uint8_t* __restrict__ coarse) {
  // one warp per block
  const int lane = threadIdx.x & 31;
  const int64_t blk = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  if (blk >= (int64_t)cw * ch) return;
  const int bi = (int)(blk / cw), bj = (int)(blk % cw), bs = 1 << log_bs;
  int n = 0, n_obst = 0, n_free = 0, n_low = 0, n_gray = 0;
  for (int p = lane; p < bs * bs; p += 32) {
    const int i = (bi << log_bs) + (p >> log_bs), j = (bj << log_bs) + (p & (bs - 1));
    if (i < H && j < W) {
      const uint32_t c = grid[tile_addr(i, j, tiles_x)];
      ++n;
      if (c == 255) ++n_free;
      else if (KIND == PORRT_DOMAIN_SHELF) { if (c < 127) ++n_obst; else ++n_low; }
      else { if (c == 0) ++n_obst; else ++n_gray; }
    }
  }
  for (int o = 16; o; o >>= 1) {
    n += __shfl_xor_sync(0xffffffffu, n, o); n_obst += __shfl_xor_sync(0xffffffffu, n_obst, o);
    n_free += __shfl_xor_sync(0xffffffffu, n_free, o); n_low += __shfl_xor_sync(0xffffffffu, n_low, o);
    n_gray += __shfl_xor_sync(0xffffffffu, n_gray, o);
  }
  if (lane == 0) {
    uint8_t cls;
    if (n_free == n) cls = 0;
    else if (n_obst == n) cls = C_OBST;
    else if (KIND == PORRT_DOMAIN_SHELF && n_low == n) cls = C_LOW;
    else cls = C_FINE | (n_gray ? C_GRAY : 0);
    coarse[blk] = cls;
  }
}

struct EdgeRec {        // 48 bytes per edge in shared memory, unpacked for the strip arithmetic of pass 1
  int32_t c0, n0;       // start pixel: major-axis coordinate, minor-axis coordinate
  int32_t dxo, dyo;     // octant-space deltas (major, minor)
  uint32_t m_lo, m_hi;  // M' = floor(2^63/dxo) + 1: floor(k*dyo/dxo) == umul64hi(2*k*dyo, M') exactly, for every dxo >= 1
  int32_t dirs;         // bit0: major axis is i (rows), bit1: major step is -1, bit2: minor step is -1, bit3: no-op edge
  int32_t n_strips;     // strips of <= BS pixels (0 for a no-op edge)
  int32_t lo_raw0;      // k of the first pixel of strip 0's block column (<= 0); strip ts starts at lo_raw0 + ts*BS
  int32_t idx0;         // class-byte index of (major block of strip 0, minor block 0)
  int32_t stride_major; // class-byte index step per strip (signed)
  int32_t stride_minor; // class-byte index step per minor block
};

__device__ __forceinline__ int32_t rec_minor(const EdgeRec& r, int32_t k) {
  return (int32_t)__umul64hi((uint64_t)(2u * (uint32_t)k * (uint32_t)r.dyo), ((uint64_t)r.m_hi << 32) | r.m_lo);
}

#define V2_QCAP 512  // queue entries per warp
#define V2_MINB 4

template <int KIND, bool INDEXED>
__global__ void __launch_bounds__(EDGE_BLOCK, V2_MINB) edge_validity_v2_kernel(MapDev m, const double2* __restrict__ from,
                                                                      const double2* __restrict__ to, int64_t n,
                                                                      int32_t* __restrict__ out_vid,
                                                                      int8_t* __restrict__ out_vid8,
                                                                      uint64_t* __restrict__ out_mask,
                                                                      const uint64_t* __restrict__ validities,
                                                                      const int32_t* __restrict__ from_idx,
                                                                      const int32_t* __restrict__ to_idx) {
  constexpr int LOG_BS = 4;   // the class bytes are built for 16 x 16 blocks
  constexpr int BS = 1 << LOG_BS;
  constexpr int V2_G = 4;     // consecutive strips of one edge handled by a lane per round (amortises the owner search)
  constexpr int WARPS = EDGE_BLOCK / 32;
  __shared__ EdgeRec s_rec[WARPS][32];
  __shared__ uint32_t s_flags[WARPS][32];     // F_* per edge
  __shared__ uint32_t s_zmin[WARPS][32], s_zmax[WARPS][32];
  __shared__ uint32_t s_queue[WARPS][V2_QCAP];
  __shared__ int32_t s_qcount[WARPS];
  const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
  const uint8_t* __restrict__ coarse = m.coarse;
  const int cw = m.coarse_cw;
  const int64_t warp = ((int64_t)blockIdx.x * EDGE_BLOCK + threadIdx.x) >> 5;
  const int64_t n_warps = ((int64_t)gridDim.x * EDGE_BLOCK) >> 5;
  const uint32_t lt_mask = (1u << lane) - 1u;

  // pass 2: per-pixel resolution of the queued strips; one lane per strip, pixels in order, pixel coordinates and the
  // Bresenham remainder stepped incrementally; strips of edges that are already blocked are dropped first
  auto drain = [&]() {
    __syncwarp();
    const int qn = s_qcount[wib];
    int live_n = 0;
    for (int q0 = 0; q0 < qn; q0 += 32) {          // in-place compaction of the live entries
      const int q = q0 + lane;
      uint32_t ent = 0;
      bool live = false;
      if (q < qn) {
        ent = s_queue[wib][q];
        live = !(s_flags[wib][ent & 31] & F_OBST) || (ent & (1u << 25));
      }
      const unsigned lv = __ballot_sync(0xffffffffu, live);
      __syncwarp();
      if (live) s_queue[wib][live_n + __popc(lv & lt_mask)] = ent;
      live_n += __popc(lv);
      __syncwarp();
    }
    for (int q0 = 0; q0 < live_n; q0 += 32) {
      const int q = q0 + lane;
      if (q < live_n) {
        const uint32_t ent = s_queue[wib][q];
        const int e = ent & 31;
        const EdgeRec& r = s_rec[wib][e];
        const int dxo = r.dxo, dyo = r.dyo, dirs = r.dirs;
        const int k0 = (int)((ent >> 5) & 0x7fff);
        int left = (int)((ent >> 20) & 31) + 1;
        const int32_t mnr = rec_minor(r, k0);
        int32_t rem = k0 * dyo - mnr * dxo;   // k*dyo = mnr*dxo + rem, 0 <= rem < dxo
        const int sm = (dirs & 2) ? -1 : 1, sn = (dirs & 4) ? -1 : 1;
        const int major = r.c0 + sm * k0, minor = r.n0 + sn * mnr;
        int i = (dirs & 1) ? major : minor, j = (dirs & 1) ? minor : major;
        const int di_u = (dirs & 1) ? sm : 0, dj_u = (dirs & 1) ? 0 : sm;   // major step
        const int di_v = (dirs & 1) ? 0 : sn, dj_v = (dirs & 1) ? sn : 0;   // minor step
        uint32_t f = 0, zmin = 255, zmax = 0;
        for (; left > 0; --left) {
          const uint32_t code = __ldg(m.grid + tile_addr(i, j, m.tiles_x));
          if (code != 255) {
            if (KIND == PORRT_DOMAIN_SHELF) { f |= code < 127 ? F_OBST : F_LOW; }
            else if (code == 0) f |= F_OBST;
            else { zmin = min(zmin, code); zmax = max(zmax, code); }
          }
          i += di_u; j += dj_u;
          rem += dyo;
          if (rem >= dxo) { rem -= dxo; i += di_v; j += dj_v; }   // dxo == 0 only for single-pixel edges (left == 1)
        }
        if (f) atomicOr(&s_flags[wib][e], f);
        if (zmax) { atomicMin(&s_zmin[wib][e], zmin); atomicMax(&s_zmax[wib][e], zmax); }
      }
    }
    __syncwarp();
    if (lane == 0) s_qcount[wib] = 0;
    __syncwarp();
  };

  for (int64_t base = warp * 32; base < n; base += n_warps * 32) {
    const int64_t eidx = base + lane;
    // ---- per-lane setup of one edge
    EdgeRec mine;
    int my_flags = 0;  // bit0 start OOB, bit1 end OOB
    mine.n_strips = 0; mine.dirs = 8; mine.c0 = mine.n0 = mine.dxo = mine.dyo = 0; mine.m_lo = mine.m_hi = 0;
    mine.lo_raw0 = mine.idx0 = mine.stride_major = mine.stride_minor = 0;
    if (eidx < n) {
      const double2 a = INDEXED ? from[from_idx[eidx]] : from[eidx];
      const double2 b = INDEXED ? to[to_idx[eidx]] : to[eidx];
      const EdgeSetup s = make_setup(m, a.x, a.y, b.x, b.y);
      const int ui = (s.steps & 3) - 1, uj = ((s.steps >> 2) & 3) - 1, vi = ((s.steps >> 4) & 3) - 1, vj = ((s.steps >> 6) & 3) - 1;
      mine.c0 = ui ? s.ai : s.aj; mine.n0 = ui ? s.aj : s.ai;
      mine.dxo = s.dxo; mine.dyo = s.dyo;
      const uint64_t M = s.dxo > 0 ? (0x8000000000000000ull / (uint64_t)s.dxo) + 1ull : 0ull;
      mine.m_lo = (uint32_t)M; mine.m_hi = (uint32_t)(M >> 32);
      mine.dirs = (ui ? 1 : 0) | ((ui + uj) < 0 ? 2 : 0) | ((vi + vj) < 0 ? 4 : 0);
      my_flags = s.flags;
      if (my_flags) mine.dirs |= 8;
      else {
        const int sgn = (mine.dirs & 2) ? -1 : 1;
        const int b0 = mine.c0 >> LOG_BS, b1 = (mine.c0 + sgn * mine.dxo) >> LOG_BS;
        mine.n_strips = (b1 > b0 ? b1 - b0 : b0 - b1) + 1;
        mine.lo_raw0 = sgn * ((b0 << LOG_BS) - mine.c0) - ((mine.dirs & 2) ? BS - 1 : 0);
        mine.stride_major = sgn * ((mine.dirs & 1) ? cw : 1);
        mine.stride_minor = (mine.dirs & 1) ? 1 : cw;
        mine.idx0 = b0 * ((mine.dirs & 1) ? cw : 1);
      }
    }
    s_rec[wib][lane] = mine;
    s_flags[wib][lane] = 0; s_zmin[wib][lane] = 255; s_zmax[wib][lane] = 0;
    // items = groups of V2_G strips; every lane owns at least one (possibly empty) item so that the inclusive prefix
    // sums are strictly increasing and the owner of a flattened position can be ranked with a bitmask
    int incl = max(1, (mine.n_strips + V2_G - 1) / V2_G);
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const int t = __shfl_up_sync(0xffffffffu, incl, o);
      if (lane >= o) incl += t;
    }
    if (lane == 0) s_qcount[wib] = 0;
    const int total = __shfl_sync(0xffffffffu, incl, 31);
    const bool may_overflow = total * V2_G > V2_QCAP;     // warp-uniform
    __syncwarp();

    // ---- pass 1: item w = w0 + lane of the flattened sequence; neighbouring lanes work on neighbouring strips
    for (int w0 = 0; w0 < total; w0 += 32) {
      if (may_overflow && s_qcount[wib] > V2_QCAP - 32 * V2_G) drain();
      const int d = incl - w0;                                    // edge `lane` ends before window position d
      const int e_base = __popc(__ballot_sync(0xffffffffu, d <= 0));
      const unsigned marks = __reduce_or_sync(0xffffffffu, (d >= 1 && d <= 32) ? (1u << (d - 1)) : 0u);
      const int e = min(31, e_base + __popc(marks & lt_mask));
      const int p_prev = __shfl_sync(0xffffffffu, incl, (e + 31) & 31);
      const int w = w0 + lane;
      if (w < total) {
        const EdgeRec& r = s_rec[wib][e];
        const int n_strips = r.n_strips, dxo = r.dxo, n0 = r.n0, stride_minor = r.stride_minor;
        const uint32_t dy2 = 2u * (uint32_t)r.dyo;
        const uint64_t M = ((uint64_t)r.m_hi << 32) | r.m_lo;
        const bool neg_minor = (r.dirs & 4) != 0;
        const int ts0 = (w - (e ? p_prev : 0)) * V2_G;
        int lo_raw = r.lo_raw0 + ts0 * BS;
        int idx_m = r.idx0 + ts0 * r.stride_major;
        const int stride_major = r.stride_major;
        uint32_t cls[V2_G];
        int klo[V2_G], klen[V2_G];
#pragma unroll
        for (int g = 0; g < V2_G; ++g) {
          cls[g] = 0;
          const int k_lo = max(0, lo_raw), k_hi = min(dxo, lo_raw + BS - 1);
          klo[g] = k_lo; klen[g] = k_hi - k_lo;
          if (ts0 + g < n_strips) {
            const int m_a = (int)__umul64hi((uint64_t)((uint32_t)k_lo * dy2), M), m_b = (int)__umul64hi((uint64_t)((uint32_t)k_hi * dy2), M);
            const int bn_a = (neg_minor ? n0 - m_a : n0 + m_a) >> LOG_BS, bn_b = (neg_minor ? n0 - m_b : n0 + m_b) >> LOG_BS;
            const int ia = idx_m + bn_a * stride_minor;
            uint32_t c = coarse[ia];
            if (bn_b != bn_a) c |= coarse[idx_m + bn_b * stride_minor];
            cls[g] = c;
          }
          lo_raw += BS; idx_m += stride_major;
        }
        uint32_t f = 0;
#pragma unroll
        for (int g = 0; g < V2_G; ++g) f |= cls[g];
        if (f & 3) atomicOr(&s_flags[wib][e], f & 3);
        if (f & C_FINE) {
          int n_want = 0;
#pragma unroll
          for (int g = 0; g < V2_G; ++g) n_want += ((cls[g] & C_FINE) && (!(f & C_OBST) || (cls[g] & C_GRAY))) ? 1 : 0;
          if (n_want) {
            int pos = atomicAdd(&s_qcount[wib], n_want);
#pragma unroll
            for (int g = 0; g < V2_G; ++g)
              if ((cls[g] & C_FINE) && (!(f & C_OBST) || (cls[g] & C_GRAY)))
                s_queue[wib][pos++] = (uint32_t)e | ((uint32_t)klo[g] << 5) | ((uint32_t)klen[g] << 20) | ((cls[g] & C_GRAY) ? (1u << 25) : 0u);
          }
        }
      }
      __syncwarp();
    }
    // ---- pass 2: pixels of the strips that are still undecided
    drain();

    // ---- results
    if (eidx < n) {
      int32_t r;
      bool slow = false;
      if (my_flags & 1) r = PORRT_PANIC_OOB;
      else if (my_flags & 2) slow = true;
      else {
        const uint32_t f = s_flags[wib][lane];
        if (KIND == PORRT_DOMAIN_SHELF) r = (f & F_OBST) ? R_BLOCKED : ((f & F_LOW) ? R_LOW : R_FREE);
        else {
          const uint32_t zmin = s_zmin[wib][lane], zmax = s_zmax[wib][lane];
          if (zmax != 0 && (zmin != zmax || zmax == 254)) slow = true;   // order of events decides: re-walk
          else r = (f & F_OBST) ? R_BLOCKED : (zmax ? (int32_t)zmin - 1 : R_FREE);
        }
      }
      if (slow) {
        Walker wk;
        const int sm = (mine.dirs & 2) ? -1 : 1, sn = (mine.dirs & 4) ? -1 : 1;
        wk.dxo = mine.dxo; wk.dyo = mine.dyo;
        wk.M = mine.dxo > 1 ? (0xFFFFFFFFFFFFFFFFull / (uint64_t)mine.dxo) + 1ull : 0ull;
        if (mine.dirs & 1) { wk.ai = mine.c0; wk.aj = mine.n0; wk.ui = sm; wk.uj = 0; wk.vi = 0; wk.vj = sn; }
        else { wk.ai = mine.n0; wk.aj = mine.c0; wk.ui = 0; wk.uj = sm; wk.vi = sn; wk.vj = 0; }
        r = walk_sequential<KIND>(m, wk);
      }
      store_edge_result(m, eidx, walk_to_validity(m, r), out_vid, out_vid8, out_mask, validities);
    }
    __syncwarp();
  }
}

// is_state_valid + state_validity (map_io.rs:165-174,487-493 / map_shelves_io.rs:158-163,464-469); thread per state
__global__ void state_validity_kernel(MapDev m, const double2* __restrict__ xy, int64_t n, int32_t* __restrict__ out_vid) {
  int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= n) return;
  const double2 p = xy[t];
  out_vid[t] = state_validity_of(m, p.x, p.y);
}

// observe_impl's geometric test (map_io.rs:285-288 / map_shelves_io.rs:259-265); one warp per state, zones in turn
template <int KIND>
__global__ void __launch_bounds__(256) visibility_kernel(MapDev m, const double2* __restrict__ xy, int64_t n,
                                                         const double2* __restrict__ zone_pos, int n_zones, double visibility,
                                                         uint64_t* __restrict__ out_mask, int32_t* __restrict__ out_status) {
  const int lane = threadIdx.x & 31;
  const int64_t warp = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  if (warp >= n) return;
  double2 p = xy[warp];
  uint64_t mask = 0;
  int32_t status = 0;
  for (int z = 0; z < n_zones && status == 0; ++z) {
    double2 zp = zone_pos[z];
    // norm2(state, zone_pos) (common.rs:203-213): (b - a), squares summed in dimension order, IEEE sqrt
    double dx = __dsub_rn(zp.x, p.x), dy = __dsub_rn(zp.y, p.y);
    double d = __dsqrt_rn(__dadd_rn(__dadd_rn(0.0, __dmul_rn(dx, dx)), __dmul_rn(dy, dy)));
    if (d < visibility) {
      EdgeSetup s = make_setup(m, p.x, p.y, zp.x, zp.y);
      int32_t r = walk_warp<KIND>(m, s, lane);
      if (r < -1 && r != R_FREE && r != R_LOW) status = r;  // the reference panics here
      else if (r != R_BLOCKED) mask |= 1ull << z;
    }
  }
  if (lane == 0) { out_mask[warp] = status ? 0ull : mask; out_status[warp] = status; }
}

// ------------------------------------------------------------------------------------------------ map build kernels
__global__ void zone_stats_kernel(const uint8_t* __restrict__ zone, int H, int W, uint32_t* __restrict__ stats /* [256*3] */) {
  __shared__ uint32_t s[256 * 3];
  for (int t = threadIdx.x; t < 768; t += blockDim.x) s[t] = 0;
  __syncthreads();
  int64_t total = (int64_t)H * W;
  for (int64_t p = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; p < total; p += (int64_t)gridDim.x * blockDim.x) {
    uint32_t z = zone[p];
    if (z != 255) {
      atomicAdd(&s[z * 3], 1u);
      atomicAdd(&s[z * 3 + 1], (uint32_t)(p / W));  // u32 sums wrap exactly like the reference's release build
      atomicAdd(&s[z * 3 + 2], (uint32_t)(p % W));
    }
  }
  __syncthreads();
  for (int t = threadIdx.x; t < 768; t += blockDim.x)
    if (s[t]) atomicAdd(&stats[t], s[t]);
}

__global__ void fuse_tile_kernel(const uint8_t* __restrict__ occ, const uint8_t* __restrict__ zone, int H, int W,
                                 int tiles_x, int tiles_y, int kind, uint8_t* __restrict__ grid) {
  // one thread per output byte, output-coalesced
  int64_t total = (int64_t)tiles_x * tiles_y * 128;
  for (int64_t a = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; a < total; a += (int64_t)gridDim.x * blockDim.x) {
    int64_t tile = a >> 7;
    int in = (int)(a & 127);
    int ti = (int)(tile / tiles_x), tj = (int)(tile % tiles_x);
    int i = ti * 8 + ((in >> 6) & 1) * 4 + ((in >> 3) & 3);
    int j = tj * 16 + ((in >> 5) & 1) * 8 + (in & 7);
    uint8_t code = 0;
    if (i < H && j < W) {
      uint8_t o = occ[(int64_t)i * W + j];
      if (kind == PORRT_DOMAIN_SHELF) code = o;
      else if (o == 255 || o == 0) code = o;
      else {
        uint8_t z = zone ? zone[(int64_t)i * W + j] : 255;
        code = z == 255 ? 254 : (uint8_t)(z + 1);
      }
    }
    grid[a] = code;
  }
}

// ------------------------------------------------------------------------------------------------ host API
PORRT_API int32_t porrt_map_upload(porrt_ctx* ctx, const uint8_t* occ, const uint8_t* zone, int32_t H, int32_t W,
                                   const double low[2], const double up[2], int32_t kind, double visibility) {
  CTX_CHECK(ctx);
  if (!occ || !low || !up || H <= 0 || W <= 0 || H > 32768 || W > 32768 || (kind != PORRT_DOMAIN_DOOR && kind != PORRT_DOMAIN_SHELF))
    return porrt_fail(ctx, PORRT_ERR_INVALID_ARG, "porrt_map_upload: bad arguments");
  CUDA_TRY(ctx, cudaSetDevice(ctx->device));
  ctx->has_map = false;
  cudaStream_t st = ctx->stream;
  const size_t px = (size_t)H * W;
  CUDA_TRY(ctx, ctx->ws_owner.ensure(px));
  CUDA_TRY(ctx, cudaMemcpyAsync(ctx->ws_owner.p, occ, px, cudaMemcpyHostToDevice, st));
  const uint8_t* d_zone = nullptr;
  int n_zones = 0, n_worlds = 0;
  std::vector<double> zone_pos;
  const double ppm = (double)W / (up[0] - low[0]);  // map_io.rs:91
  if (zone) {
    CUDA_TRY(ctx, ctx->ws_vid.ensure(px));
    CUDA_TRY(ctx, cudaMemcpyAsync(ctx->ws_vid.p, zone, px, cudaMemcpyHostToDevice, st));
    d_zone = ctx->ws_vid.as<uint8_t>();
    CUDA_TRY(ctx, ctx->ws_table.ensure(768 * 4));
    CUDA_TRY(ctx, cudaMemsetAsync(ctx->ws_table.p, 0, 768 * 4, st));
    zone_stats_kernel<<<ctx->sm_count * 4, 256, 0, st>>>(d_zone, H, W, ctx->ws_table.as<uint32_t>());
    LAUNCH_CHECK(ctx);
    uint32_t stats[768];
    CUDA_TRY(ctx, cudaMemcpyAsync(stats, ctx->ws_table.p, sizeof(stats), cudaMemcpyDeviceToHost, st));
    CUDA_TRY(ctx, cudaStreamSynchronize(st));
    int max_id = 0;  // init_zone_ids (map_io.rs:130-145): n_zones = max id + 1, 1 even without any zone pixel
    for (int z = 0; z < 255; ++z)
      if (stats[z * 3]) max_id = z;
    n_zones = max_id + 1;
    for (int z = 0; z < n_zones; ++z) {
      if (!stats[z * 3]) return porrt_fail(ctx, PORRT_ERR_PANIC, "zone without pixels: the reference divides by zero (map_io.rs:160)");
      uint32_t ci = stats[z * 3 + 1] / stats[z * 3], cj = stats[z * 3 + 2] / stats[z * 3];
      // to_coordinates (map_io.rs:183-188), including its swapped low[] indices
      zone_pos.push_back((double)cj / ppm + low[1]);
      zone_pos.push_back((double)(uint32_t)(H - 1 - (int)ci) / ppm + low[0]);
    }
  }
  std::vector<uint64_t> validities, zone_masks;
  int n_validities = 0, words = 1;
  if (kind == PORRT_DOMAIN_DOOR) {
    if (zone) {
      if (n_zones > 16) return porrt_fail(ctx, PORRT_ERR_UNSUPPORTED, "door domain: more than 16 zones (65536 worlds) is not supported");
      n_worlds = 1 << n_zones;                       // map_io.rs:144
      words = (n_worlds + 63) / 64;
      zone_masks.assign((size_t)n_zones * words, 0);
      for (int z = 0; z < n_zones; ++z)              // zone_index_to_world_mask (map_io.rs:198-214)
        for (int w = 0; w < n_worlds; ++w)
          if (w & (1 << z)) zone_masks[(size_t)z * words + w / 64] |= 1ull << (w % 64);
      validities = zone_masks;                       // world_validities = zones_to_worlds + [all ones] (map_io.rs:125-126)
      n_validities = n_zones + 1;
    } else {
      n_worlds = 1; n_validities = 1;                // init_without_zones (map_io.rs:108-111)
    }
    validities.resize((size_t)n_validities * words, 0);
    for (int w = 0; w < n_worlds; ++w) validities[(size_t)(n_validities - 1) * words + w / 64] |= 1ull << (w % 64);
  } else {
    if (!zone) return porrt_fail(ctx, PORRT_ERR_PANIC, "MapShelfDomain without zones: world_validities.len()-1 underflows (map_shelves_io.rs:466)");
    n_worlds = n_zones;                              // map_shelves_io.rs:460-462
    words = (n_worlds + 63) / 64;
    n_validities = 1;                                // single all-ones mask (map_shelves_io.rs:113)
    validities.assign(words, 0);
    for (int w = 0; w < n_worlds; ++w) validities[w / 64] |= 1ull << (w % 64);
  }
  if (n_zones > 64) return porrt_fail(ctx, PORRT_ERR_UNSUPPORTED, "more than 64 zones is not supported");

  const int tiles_x = (W + 15) / 16, tiles_y = (H + 7) / 8;
  const size_t grid_bytes = (size_t)tiles_x * tiles_y * 128;
  CUDA_TRY(ctx, ctx->d_grid.ensure(grid_bytes));
  fuse_tile_kernel<<<ctx->sm_count * 8, 256, 0, st>>>(ctx->ws_owner.as<uint8_t>(), d_zone, H, W, tiles_x, tiles_y, kind,
                                                      ctx->d_grid.as<uint8_t>());
  LAUNCH_CHECK(ctx);
  {  // class bytes of the 16 x 16 blocks (large-map path)
    const int lg = 4, bs = 1 << lg, cwl = (W + bs - 1) / bs, chl = (H + bs - 1) / bs;
    CUDA_TRY(ctx, ctx->d_coarse.ensure((size_t)cwl * chl));
    if (kind == PORRT_DOMAIN_SHELF)
      coarse_build_kernel<PORRT_DOMAIN_SHELF><<<div_up((int64_t)cwl * chl * 32, 256), 256, 0, st>>>(ctx->d_grid.as<uint8_t>(), H, W, tiles_x, lg, cwl, chl, ctx->d_coarse.as<uint8_t>());
    else
      coarse_build_kernel<PORRT_DOMAIN_DOOR><<<div_up((int64_t)cwl * chl * 32, 256), 256, 0, st>>>(ctx->d_grid.as<uint8_t>(), H, W, tiles_x, lg, cwl, chl, ctx->d_coarse.as<uint8_t>());
    LAUNCH_CHECK(ctx);
    ctx->map.coarse = ctx->d_coarse.as<uint8_t>();
    ctx->map.coarse_cw = cwl;
  }
  CUDA_TRY(ctx, ctx->d_validities.ensure(validities.size() * 8));
  CUDA_TRY(ctx, cudaMemcpyAsync(ctx->d_validities.p, validities.data(), validities.size() * 8, cudaMemcpyHostToDevice, st));
  CUDA_TRY(ctx, ctx->d_zone_pos.ensure(zone_pos.size() * 8 + 16));
  if (!zone_pos.empty())
    CUDA_TRY(ctx, cudaMemcpyAsync(ctx->d_zone_pos.p, zone_pos.data(), zone_pos.size() * 8, cudaMemcpyHostToDevice, st));
  MapDev& m = ctx->map;
  m.grid = ctx->d_grid.as<uint8_t>();
  m.H = H; m.W = W; m.tiles_x = tiles_x; m.kind = kind; m.free_vid = n_validities - 1; m.mask_words = words;
  m.low0 = low[0]; m.low1 = low[1]; m.ppm = ppm; m.hm1 = (double)(H - 1);
  { int32_t rc = edge3_build(ctx, st); if (rc) return rc; }   // class plane + block bitmaps (edge3.cu)
  CUDA_TRY(ctx, cudaStreamSynchronize(st));
  ctx->n_zones = n_zones; ctx->n_worlds = n_worlds; ctx->n_validities = n_validities; ctx->mask_words = words;
  ctx->visibility = zone ? visibility : 0.0;
  ctx->validities = validities; ctx->zone_pos = zone_pos; ctx->zone_world_masks = zone_masks;
  ctx->has_map = true;
  return PORRT_OK;
}

PORRT_API int32_t porrt_map_info(porrt_ctx* ctx, int32_t* n_zones, int32_t* n_worlds, int32_t* n_validities, int32_t* mask_words) {
  CTX_CHECK(ctx);
  if (!ctx->has_map) return porrt_fail(ctx, PORRT_ERR_NO_MAP, "no map uploaded");
  if (n_zones) *n_zones = ctx->n_zones;
  if (n_worlds) *n_worlds = ctx->n_worlds;
  if (n_validities) *n_validities = ctx->n_validities;
  if (mask_words) *mask_words = ctx->mask_words;
  return PORRT_OK;
}
PORRT_API int32_t porrt_map_zone_positions(porrt_ctx* ctx, double* out_xy) {
  CTX_CHECK(ctx);
  if (!ctx->has_map) return porrt_fail(ctx, PORRT_ERR_NO_MAP, "no map uploaded");
  if (!ctx->zone_pos.empty()) memcpy(out_xy, ctx->zone_pos.data(), ctx->zone_pos.size() * 8);
  return PORRT_OK;
}
PORRT_API int32_t porrt_map_world_validities(porrt_ctx* ctx, uint64_t* out) {
  CTX_CHECK(ctx);
  if (!ctx->has_map) return porrt_fail(ctx, PORRT_ERR_NO_MAP, "no map uploaded");
  memcpy(out, ctx->validities.data(), ctx->validities.size() * 8);
  return PORRT_OK;
}

static int edge_grid(porrt_ctx* ctx, int64_t n) {
  int64_t warps = (n + 31) / 32;
  int64_t blocks = (warps + (EDGE_BLOCK / 32) - 1) / (EDGE_BLOCK / 32);
  int64_t cap = (int64_t)ctx->sm_count * 8;  // persistent: 8 CTAs of 256 threads per SM = full occupancy
  return (int)(blocks < cap ? (blocks < 1 ? 1 : blocks) : cap);
}

// One edge batch on the device: edge3.cu's kernel, or the large-map kernel above when the class plane does not fit in shared
// memory.  from_idx / to_idx != NULL: endpoints are gathered from the vertex buffer from_dev == to_dev.
int32_t map_edge_launch(porrt_ctx* ctx, const double* from_dev, const double* to_dev, const int32_t* from_idx, const int32_t* to_idx,
                        int64_t n, const EdgeOut& out, cudaStream_t st) {
  if (n == 0) return PORRT_OK;
  if (!ctx->force_large_map_path && edge3_usable(ctx)) return edge3_launch(ctx, from_dev, to_dev, n, out, from_idx, to_idx, st);
  const double2 *from = (const double2*)from_dev, *to = (const double2*)to_dev;
  const uint64_t* val = ctx->d_validities.as<uint64_t>();
  const int grid = edge_grid(ctx, n);
  const bool shelf = ctx->map.kind == PORRT_DOMAIN_SHELF;
#define LAUNCH_LARGE(K, I) edge_validity_v2_kernel<K, I><<<grid, EDGE_BLOCK, 0, st>>>(ctx->map, from, to, n, out.vid, out.vid8, out.mask, val, from_idx, to_idx)
  if (from_idx) { if (shelf) LAUNCH_LARGE(PORRT_DOMAIN_SHELF, true); else LAUNCH_LARGE(PORRT_DOMAIN_DOOR, true); }
  else { if (shelf) LAUNCH_LARGE(PORRT_DOMAIN_SHELF, false); else LAUNCH_LARGE(PORRT_DOMAIN_DOOR, false); }
#undef LAUNCH_LARGE
  LAUNCH_CHECK(ctx);
  return PORRT_OK;
}

int32_t map_edge_validity_dev(porrt_ctx* ctx, const double* from_dev, const double* to_dev, int64_t n,
                              int32_t* out_vid_dev, uint64_t* out_mask_dev, cudaStream_t st) {
  EdgeOut o; o.vid = out_vid_dev; o.mask = out_mask_dev;
  return map_edge_launch(ctx, from_dev, to_dev, nullptr, nullptr, n, o, st);
}

int32_t map_edge_validity_indexed_dev(porrt_ctx* ctx, const double* xy_dev, const int32_t* from_idx_dev, const int32_t* to_idx_dev,
                                      int64_t n, int32_t* out_vid_dev, cudaStream_t st) {
  EdgeOut o; o.vid = out_vid_dev;
  return map_edge_launch(ctx, xy_dev, xy_dev, from_idx_dev, to_idx_dev, n, o, st);
}

PORRT_API int32_t porrt_ctx_set_option(porrt_ctx* ctx, int32_t option, int64_t value) {
  CTX_CHECK(ctx);
  switch (option) {
    case PORRT_OPT_FORCE_LARGE_MAP_PATH: ctx->force_large_map_path = value != 0; return PORRT_OK;
    case PORRT_OPT_FORCE_GLOBAL_SWEEPS: ctx->force_global_sweeps = value != 0; return PORRT_OK;
    case PORRT_OPT_FORCE_THREAD_PER_QUERY_NN: ctx->force_thread_per_query_nn = value != 0; return PORRT_OK;
    default: return porrt_fail(ctx, PORRT_ERR_INVALID_ARG, "porrt_ctx_set_option: unknown option");
  }
}

PORRT_API int32_t porrt_edge_validity_dev(porrt_ctx* ctx, const double* from_dev, const double* to_dev, int64_t n,
                                          int32_t* out_vid_dev, uint64_t* out_mask_dev) {
  CTX_CHECK(ctx);
  if (!ctx->has_map) return porrt_fail(ctx, PORRT_ERR_NO_MAP, "no map uploaded");
  if (n < 0 || (n > 0 && (!from_dev || !to_dev || !out_vid_dev))) return porrt_fail(ctx, PORRT_ERR_INVALID_ARG, "porrt_edge_validity_dev: bad arguments");
  CUDA_TRY(ctx, cudaSetDevice(ctx->device));
  return map_edge_validity_dev(ctx, from_dev, to_dev, n, out_vid_dev, out_mask_dev, ctx->stream);
}

// ids outside [0, V) must never reach the edge kernels (they index the vertex array): clamp them and remember that it happened
__global__ void idx_check_kernel(int32_t* __restrict__ a, int32_t* __restrict__ b, int64_t n, int32_t V, int32_t* __restrict__ bad) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const int32_t x = a[i], y = b ? b[i] : 0;
  if ((uint32_t)x >= (uint32_t)V || (uint32_t)y >= (uint32_t)V) {
    *bad = 1;
    if ((uint32_t)x >= (uint32_t)V) a[i] = 0;
    if (b && (uint32_t)y >= (uint32_t)V) b[i] = 0;
  }
}

// adjacency form: edge e of the CSR lies in row r = the last row with row_ptr[r] <= e; rows[e - e0] = r for e in [e0, e0 + n)
__global__ void csr_rows_kernel(const int64_t* __restrict__ row_ptr, int64_t V, int64_t e0, int64_t n, int32_t* __restrict__ rows) {
  const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= n) return;
  const int64_t e = e0 + t;
  int64_t lo = 0, hi = V;          // row_ptr[lo] <= e < row_ptr[hi]
  while (hi - lo > 1) {
    const int64_t mid = (lo + hi) >> 1;
    if (__ldg(row_ptr + mid) <= e) lo = mid; else hi = mid;
  }
  rows[t] = (int32_t)lo;
}

// ------------------------------------------------------------------------------------------------ host-buffer pipeline
// Every host-buffer edge entry point is one chunked pipeline: H2D(c+1) | kernel(c) | D2H(c-1) on three streams over MAX_SLOTS
// device slots.  Caller buffers that are pinned (cudaHostAlloc / torch pin_memory) are DMA'd directly, pageable ones are
// staged through the ctx's pinned buffer.  Slot pieces are 256-byte aligned (the kernels read endpoints as 16-byte vectors and write
// 8-byte masks; chunk sizes are arbitrary).
struct EdgeJob {
  enum Mode { COORDS, INDEXED, CSR } mode = COORDS;
  const void* in[2] = {nullptr, nullptr};   // per-edge host input arrays: COORDS from/to xy (16 B), INDEXED from/to ids (4 B), CSR col (4 B)
  int in_elem[2] = {0, 0};
  int n_in = 0;
  int32_t* out_vid = nullptr;               // exactly one of out_vid / out_vid8
  int8_t* out_vid8 = nullptr;
  uint64_t* out_mask = nullptr;             // nullable, [n * mask_words]
  const int64_t* row_ptr_dev = nullptr;     // CSR: device copy of row_ptr[V + 1]
  int64_t csr_rows = 0;
  int csr_row_is_to = 1;                    // CSR: 1 = edge col[e] -> row (prm.rs:93, neighbour -> new node), 0 = row -> col[e]
  const char* name = "porrt_edge_validity";
};

static int32_t edge_pipeline(porrt_ctx* ctx, const EdgeJob& job, int64_t n) {
  const int words = ctx->mask_words;
  const int vid_elem = job.out_vid8 ? 1 : 4;
  const size_t in_bytes = (size_t)job.in_elem[0] + (job.n_in > 1 ? (size_t)job.in_elem[1] : 0);
  const size_t out_bytes = (size_t)vid_elem + (job.out_mask ? 8 * (size_t)words : 0);
  // edges per chunk: ~1/8 of the call, between 2^18 and 2^21 edges for 48 B/edge (measured on B200/PCIe 5: 2 Mi-edge chunks of
  // coordinates reach 50 GB/s host->device, 64 Ki-edge chunks 39 GB/s); lighter edges get proportionally longer chunks
  const int64_t scale = (int64_t)(48 / (in_bytes + out_bytes)) < 1 ? 1 : (int64_t)(48 / (in_bytes + out_bytes));
  int64_t CH = n / 8;
  const int64_t ch_lo = ((int64_t)1 << 18) * scale, ch_hi = ((int64_t)1 << 21) * scale;
  CH = CH < ch_lo ? ch_lo : (CH > ch_hi ? ch_hi : CH);
  const int64_t ch = n < CH ? n : CH;
  bool pinned = is_pinned_host(job.in[0]) && (job.n_in < 2 || is_pinned_host(job.in[1])) &&
                is_pinned_host(job.out_vid8 ? (const void*)job.out_vid8 : (const void*)job.out_vid) &&
                (!job.out_mask || is_pinned_host(job.out_mask));
  const int slots = MAX_SLOTS;
  // the slots, laid out alike in the device buffer and, for pageable callers, its pinned twin
  struct Slot { char* in[2]; int32_t* rows; char* vid; char* mask; } dev[MAX_SLOTS] = {}, host[MAX_SLOTS] = {};
  auto slot_layout = [&](Carve& c, Slot* sl) {
    for (int s = 0; s < slots; ++s) {
      for (int k = 0; k < job.n_in; ++k) sl[s].in[k] = c.take<char>((size_t)ch * job.in_elem[k], 256);
      if (job.mode == EdgeJob::CSR) sl[s].rows = c.take<int32_t>(ch, 256);
      sl[s].vid = c.take<char>((size_t)ch * vid_elem, 256);
      if (job.out_mask) sl[s].mask = c.take<char>((size_t)ch * 8 * words, 256);
    }
  };
  CUDA_TRY(ctx, carve(ctx->ws_main, [&](Carve& c) { slot_layout(c, dev); }));
  if (!pinned) CUDA_TRY(ctx, carve(ctx->pin_edge, [&](Carve& c) { slot_layout(c, host); }));
  cudaStream_t st = ctx->stream;
  const int64_t n_chunks = (n + ch - 1) / ch;
  const double* d_xy = ctx->d_vxy.as<double>();
  const int64_t V = ctx->n_vertices;
  int32_t* d_bad = nullptr;
  if (job.mode != EdgeJob::COORDS) {
    CUDA_TRY(ctx, ctx->ws_query.ensure(16));
    d_bad = ctx->ws_query.as<int32_t>();
    CUDA_TRY(ctx, cudaMemsetAsync(d_bad, 0, 4, st));
  }
  // the copy streams must not run ahead of work already queued on the compute stream
  CUDA_TRY(ctx, cudaEventRecord(ctx->ev_k[0], st));
  CUDA_TRY(ctx, cudaStreamWaitEvent(ctx->copy_in, ctx->ev_k[0], 0));
  char* const h_vid_base = job.out_vid8 ? (char*)job.out_vid8 : (char*)job.out_vid;
  auto unstage = [&](int64_t c) {   // pageable outputs: copy chunk c out of its pinned slot
    const int s = (int)(c % slots);
    const int64_t off = c * ch, cnt = (n - off) < ch ? (n - off) : ch;
    memcpy(h_vid_base + (size_t)off * vid_elem, host[s].vid, (size_t)cnt * vid_elem);
    if (job.out_mask) memcpy(job.out_mask + off * words, host[s].mask, (size_t)cnt * 8 * words);
  };
  for (int64_t c = 0; c < n_chunks; ++c) {
    const int s = (int)(c % slots);
    const int64_t off = c * ch, cnt = (n - off) < ch ? (n - off) : ch;
    const Slot& d = dev[s];
    const Slot& h = host[s];
    if (c >= slots) {
      // slot reuse: its previous D2H must be complete (also frees the pinned staging of that slot)
      CUDA_TRY(ctx, cudaEventSynchronize(ctx->ev_out[s]));
      if (!pinned) unstage(c - slots);
    }
    for (int k = 0; k < job.n_in; ++k) {
      const char* src = (const char*)job.in[k] + (size_t)off * job.in_elem[k];
      if (!pinned) { memcpy(h.in[k], src, (size_t)cnt * job.in_elem[k]); src = h.in[k]; }
      CUDA_TRY(ctx, cudaMemcpyAsync(d.in[k], src, (size_t)cnt * job.in_elem[k], cudaMemcpyHostToDevice, ctx->copy_in));
    }
    CUDA_TRY(ctx, cudaEventRecord(ctx->ev_in[s], ctx->copy_in));
    CUDA_TRY(ctx, cudaStreamWaitEvent(st, ctx->ev_in[s], 0));
    EdgeOut o;
    if (job.out_vid8) o.vid8 = (int8_t*)d.vid; else o.vid = (int32_t*)d.vid;
    if (job.out_mask) o.mask = (uint64_t*)d.mask;
    int32_t rc;
    if (job.mode == EdgeJob::COORDS) {
      rc = map_edge_launch(ctx, (const double*)d.in[0], (const double*)d.in[1], nullptr, nullptr, cnt, o, st);
    } else {
      int32_t* d_a = (int32_t*)d.in[0];
      int32_t* d_b = job.mode == EdgeJob::INDEXED ? (int32_t*)d.in[1] : nullptr;
      idx_check_kernel<<<div_up(cnt, 256), 256, 0, st>>>(d_a, d_b, cnt, (int32_t)V, d_bad);
      LAUNCH_CHECK(ctx);
      if (job.mode == EdgeJob::CSR) {
        csr_rows_kernel<<<div_up(cnt, 256), 256, 0, st>>>(job.row_ptr_dev, job.csr_rows, off, cnt, d.rows);
        LAUNCH_CHECK(ctx);
        rc = job.csr_row_is_to ? map_edge_launch(ctx, d_xy, d_xy, d_a, d.rows, cnt, o, st)
                               : map_edge_launch(ctx, d_xy, d_xy, d.rows, d_a, cnt, o, st);
      } else {
        rc = map_edge_launch(ctx, d_xy, d_xy, d_a, d_b, cnt, o, st);
      }
    }
    if (rc) return rc;
    CUDA_TRY(ctx, cudaEventRecord(ctx->ev_k[s], st));
    CUDA_TRY(ctx, cudaStreamWaitEvent(ctx->copy_out, ctx->ev_k[s], 0));
    char* h_vid = pinned ? h_vid_base + (size_t)off * vid_elem : h.vid;
    CUDA_TRY(ctx, cudaMemcpyAsync(h_vid, d.vid, (size_t)cnt * vid_elem, cudaMemcpyDeviceToHost, ctx->copy_out));
    if (job.out_mask) {
      char* h_mask = pinned ? (char*)(job.out_mask + off * words) : h.mask;
      CUDA_TRY(ctx, cudaMemcpyAsync(h_mask, d.mask, (size_t)cnt * 8 * words, cudaMemcpyDeviceToHost, ctx->copy_out));
    }
    CUDA_TRY(ctx, cudaEventRecord(ctx->ev_out[s], ctx->copy_out));
  }
  int32_t bad = 0;
  if (d_bad) CUDA_TRY(ctx, cudaMemcpyAsync(&bad, d_bad, 4, cudaMemcpyDeviceToHost, st));
  CUDA_TRY(ctx, cudaStreamSynchronize(ctx->copy_out));
  CUDA_TRY(ctx, cudaStreamSynchronize(st));
  if (!pinned)
    for (int64_t c = n_chunks > slots ? n_chunks - slots : 0; c < n_chunks; ++c) unstage(c);
  if (bad) return porrt_fail(ctx, PORRT_ERR_INVALID_ARG, std::string(job.name) + ": vertex id out of range");
  return PORRT_OK;
}

static int32_t edge_entry_checks(porrt_ctx* ctx, const char* name, int64_t n, bool ok_args, bool need_vertices) {
  if (!ctx->has_map) return porrt_fail(ctx, PORRT_ERR_NO_MAP, "no map uploaded");
  if (need_vertices && ctx->n_vertices <= 0) return porrt_fail(ctx, PORRT_ERR_NO_VERTICES, "no vertex set");
  if (n < 0 || (n > 0 && !ok_args)) return porrt_fail(ctx, PORRT_ERR_INVALID_ARG, std::string(name) + ": bad arguments");
  return PORRT_OK;
}

PORRT_API int32_t porrt_edge_validity(porrt_ctx* ctx, const double* from_xy, const double* to_xy, int64_t n,
                                      int32_t* out_vid, uint64_t* out_mask) {
  CTX_CHECK(ctx);
  if (int32_t rc = edge_entry_checks(ctx, "porrt_edge_validity", n, from_xy && to_xy && out_vid, false)) return rc;
  if (n == 0) return PORRT_OK;
  CUDA_TRY(ctx, cudaSetDevice(ctx->device));
  EdgeJob j; j.mode = EdgeJob::COORDS; j.in[0] = from_xy; j.in[1] = to_xy; j.in_elem[0] = j.in_elem[1] = 16; j.n_in = 2;
  j.out_vid = out_vid; j.out_mask = out_mask; j.name = "porrt_edge_validity";
  return edge_pipeline(ctx, j, n);
}

PORRT_API int32_t porrt_edge_validity_i8(porrt_ctx* ctx, const double* from_xy, const double* to_xy, int64_t n, int8_t* out_vid8) {
  CTX_CHECK(ctx);
  if (int32_t rc = edge_entry_checks(ctx, "porrt_edge_validity_i8", n, from_xy && to_xy && out_vid8, false)) return rc;
  if (n == 0) return PORRT_OK;
  CUDA_TRY(ctx, cudaSetDevice(ctx->device));
  EdgeJob j; j.mode = EdgeJob::COORDS; j.in[0] = from_xy; j.in[1] = to_xy; j.in_elem[0] = j.in_elem[1] = 16; j.n_in = 2;
  j.out_vid8 = out_vid8; j.name = "porrt_edge_validity_i8";
  return edge_pipeline(ctx, j, n);
}

// transition_validator(&PTONode, &PTONode) as the planners call it (pto.rs:105, prm.rs:93): both ends are NODES.  With the node
// states resident on the device (porrt_vertices_set / porrt_prm_build), an edge is two 4-byte ids instead of four doubles: the
// host->device stream shrinks from 32 to 8 bytes per edge, which is what bounds the end-to-end rate of porrt_edge_validity
// (PCIe).  Same pipeline; results identical to porrt_edge_validity on the same coordinates.
PORRT_API int32_t porrt_edge_validity_indexed(porrt_ctx* ctx, const int32_t* from_idx, const int32_t* to_idx, int64_t n,
                                              int32_t* out_vid, uint64_t* out_mask) {
  CTX_CHECK(ctx);
  if (int32_t rc = edge_entry_checks(ctx, "porrt_edge_validity_indexed", n, from_idx && to_idx && out_vid, true)) return rc;
  if (n == 0) return PORRT_OK;
  CUDA_TRY(ctx, cudaSetDevice(ctx->device));
  EdgeJob j; j.mode = EdgeJob::INDEXED; j.in[0] = from_idx; j.in[1] = to_idx; j.in_elem[0] = j.in_elem[1] = 4; j.n_in = 2;
  j.out_vid = out_vid; j.out_mask = out_mask; j.name = "porrt_edge_validity_indexed";
  return edge_pipeline(ctx, j, n);
}

PORRT_API int32_t porrt_edge_validity_indexed_i8(porrt_ctx* ctx, const int32_t* from_idx, const int32_t* to_idx, int64_t n,
                                                 int8_t* out_vid8) {
  CTX_CHECK(ctx);
  if (int32_t rc = edge_entry_checks(ctx, "porrt_edge_validity_indexed_i8", n, from_idx && to_idx && out_vid8, true)) return rc;
  if (n == 0) return PORRT_OK;
  CUDA_TRY(ctx, cudaSetDevice(ctx->device));
  EdgeJob j; j.mode = EdgeJob::INDEXED; j.in[0] = from_idx; j.in[1] = to_idx; j.in_elem[0] = j.in_elem[1] = 4; j.n_in = 2;
  j.out_vid8 = out_vid8; j.name = "porrt_edge_validity_indexed_i8";
  return edge_pipeline(ctx, j, n);
}

// The candidate edges of a roadmap as the planners hold them: an adjacency (CSR) over the resident vertex set -- row r lists the
// neighbours transition_validator is asked about for node r (prm.rs:91-96, pto.rs:103-108).  4 bytes in, 1 byte out per edge.
PORRT_API int32_t porrt_edge_validity_csr_i8(porrt_ctx* ctx, const int64_t* row_ptr, const int32_t* col, int64_t n_rows,
                                             int32_t row_is_to, int8_t* out_vid8) {
  CTX_CHECK(ctx);
  if (n_rows < 0 || (n_rows > 0 && !row_ptr)) return porrt_fail(ctx, PORRT_ERR_INVALID_ARG, "porrt_edge_validity_csr_i8: bad arguments");
  if (n_rows == 0) return PORRT_OK;
  const int64_t n = row_ptr[n_rows];
  if (int32_t rc = edge_entry_checks(ctx, "porrt_edge_validity_csr_i8", n, col && out_vid8, true)) return rc;
  // (row_ptr need not be scanned: the row of an edge comes from a binary search that always lands inside [0, n_rows), and the
  //  column ids are range-checked on the device; a non-monotone row_ptr gives meaningless rows, never an out-of-range access)
  if (n_rows > ctx->n_vertices || row_ptr[0] != 0 || n < 0) return porrt_fail(ctx, PORRT_ERR_INVALID_ARG, "porrt_edge_validity_csr_i8: rows exceed the vertex set / row_ptr[0] != 0");
  if (n == 0) return PORRT_OK;
  CUDA_TRY(ctx, cudaSetDevice(ctx->device));
  CUDA_TRY(ctx, ctx->sort_keys.ensure((size_t)(n_rows + 1) * 8));
  CUDA_TRY(ctx, cudaMemcpyAsync(ctx->sort_keys.p, row_ptr, (size_t)(n_rows + 1) * 8, cudaMemcpyHostToDevice, ctx->stream));
  EdgeJob j; j.mode = EdgeJob::CSR; j.in[0] = col; j.in_elem[0] = 4; j.n_in = 1; j.out_vid8 = out_vid8;
  j.row_ptr_dev = ctx->sort_keys.as<int64_t>(); j.csr_rows = n_rows; j.csr_row_is_to = row_is_to ? 1 : 0;
  j.name = "porrt_edge_validity_csr_i8";
  return edge_pipeline(ctx, j, n);
}

PORRT_API int32_t porrt_state_validity_dev(porrt_ctx* ctx, const double* xy_dev, int64_t n, int32_t* out_dev) {
  CTX_CHECK(ctx);
  if (!ctx->has_map) return porrt_fail(ctx, PORRT_ERR_NO_MAP, "no map uploaded");
  if (n < 0 || (n > 0 && (!xy_dev || !out_dev))) return porrt_fail(ctx, PORRT_ERR_INVALID_ARG, "porrt_state_validity_dev: bad arguments");
  if (n == 0) return PORRT_OK;
  CUDA_TRY(ctx, cudaSetDevice(ctx->device));
  state_validity_kernel<<<div_up(n, 256), 256, 0, ctx->stream>>>(ctx->map, (const double2*)xy_dev, n, out_dev);
  LAUNCH_CHECK(ctx);
  return PORRT_OK;
}

PORRT_API int32_t porrt_state_validity(porrt_ctx* ctx, const double* xy, int64_t n, int32_t* out_vid) {
  CTX_CHECK(ctx);
  if (!ctx->has_map) return porrt_fail(ctx, PORRT_ERR_NO_MAP, "no map uploaded");
  if (n < 0 || (n > 0 && (!xy || !out_vid))) return porrt_fail(ctx, PORRT_ERR_INVALID_ARG, "porrt_state_validity: bad arguments");
  if (n == 0) return PORRT_OK;
  CUDA_TRY(ctx, cudaSetDevice(ctx->device));
  double* d_xy;
  int32_t* d_out;
  CUDA_TRY(ctx, carve(ctx->ws_main, [&](Carve& c) { d_xy = c.take<double>(2 * n); d_out = c.take<int32_t>(n); }));
  CUDA_TRY(ctx, cudaMemcpyAsync(d_xy, xy, (size_t)n * 16, cudaMemcpyHostToDevice, ctx->stream));
  int32_t rc = porrt_state_validity_dev(ctx, d_xy, n, d_out);
  if (rc) return rc;
  CUDA_TRY(ctx, cudaMemcpyAsync(out_vid, d_out, (size_t)n * 4, cudaMemcpyDeviceToHost, ctx->stream));
  CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
  return PORRT_OK;
}

PORRT_API int32_t porrt_visibility_dev(porrt_ctx* ctx, const double* xy_dev, int64_t n, uint64_t* out_mask_dev, int32_t* out_status_dev) {
  CTX_CHECK(ctx);
  if (!ctx->has_map) return porrt_fail(ctx, PORRT_ERR_NO_MAP, "no map uploaded");
  if (n < 0 || (n > 0 && (!xy_dev || !out_mask_dev || !out_status_dev))) return porrt_fail(ctx, PORRT_ERR_INVALID_ARG, "porrt_visibility_dev: bad arguments");
  if (n == 0) return PORRT_OK;
  CUDA_TRY(ctx, cudaSetDevice(ctx->device));
  int blocks = div_up(n * 32, 256);
  if (ctx->map.kind == PORRT_DOMAIN_SHELF)
    visibility_kernel<PORRT_DOMAIN_SHELF><<<blocks, 256, 0, ctx->stream>>>(ctx->map, (const double2*)xy_dev, n, ctx->d_zone_pos.as<double2>(), ctx->n_zones, ctx->visibility, out_mask_dev, out_status_dev);
  else
    visibility_kernel<PORRT_DOMAIN_DOOR><<<blocks, 256, 0, ctx->stream>>>(ctx->map, (const double2*)xy_dev, n, ctx->d_zone_pos.as<double2>(), ctx->n_zones, ctx->visibility, out_mask_dev, out_status_dev);
  LAUNCH_CHECK(ctx);
  return PORRT_OK;
}

PORRT_API int32_t porrt_visibility(porrt_ctx* ctx, const double* xy, int64_t n, uint64_t* out_mask, int32_t* out_status) {
  CTX_CHECK(ctx);
  if (!ctx->has_map) return porrt_fail(ctx, PORRT_ERR_NO_MAP, "no map uploaded");
  if (n < 0 || (n > 0 && (!xy || !out_mask || !out_status))) return porrt_fail(ctx, PORRT_ERR_INVALID_ARG, "porrt_visibility: bad arguments");
  if (n == 0) return PORRT_OK;
  CUDA_TRY(ctx, cudaSetDevice(ctx->device));
  double* d_xy;
  uint64_t* d_mask;
  int32_t* d_status;
  CUDA_TRY(ctx, carve(ctx->ws_main, [&](Carve& c) { d_xy = c.take<double>(2 * n); d_mask = c.take<uint64_t>(n); d_status = c.take<int32_t>(n); }));
  CUDA_TRY(ctx, cudaMemcpyAsync(d_xy, xy, (size_t)n * 16, cudaMemcpyHostToDevice, ctx->stream));
  int32_t rc = porrt_visibility_dev(ctx, d_xy, n, d_mask, d_status);
  if (rc) return rc;
  CUDA_TRY(ctx, cudaMemcpyAsync(out_mask, d_mask, (size_t)n * 8, cudaMemcpyDeviceToHost, ctx->stream));
  CUDA_TRY(ctx, cudaMemcpyAsync(out_status, d_status, (size_t)n * 4, cudaMemcpyDeviceToHost, ctx->stream));
  CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
  return PORRT_OK;
}
