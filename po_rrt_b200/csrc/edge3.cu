// edge3.cu -- batched edge validity, third design (SURVEY.md 8(a) rows A3/A3'/A5): the headline kernel.
//
// Replaces Map::get_traversed_space + transition_validator (reference src/map_io.rs:216-241,495-513) and the
// MapShelfDomain pair (src/map_shelves_io.rs:187-203,471-488) over line_drawing::Bresenham (crate 0.8).
//
// Why a third design: ncu on v2 (map.cu) showed the L1 data pipe at 57 % of its wavefront peak and 75 warp
// instructions per edge: every class byte and every pixel was a scattered global load (32 distinct lines = 32 L1
// wavefronts per warp instruction) and a resolved pixel cost ~15 instructions.  Here
//   * the coarse level -- a 2-bit class per 16 x 16 block: free / mixed / all blocking / special -- is 64 KiB for an
//     8192^2 map and is staged ONCE per CTA in shared memory (one bulk-async copy, mbarrier completion), so the
//     two class lookups a 16-pixel strip needs are shared-memory reads (bank conflicts ~3 wavefronts instead of 32);
//   * the fine level is a bitmap: 256 bits per block, stored as sixteen 16-bit vectors, one per position along the
//     line's major axis, in the four orientations a line can cross a block (major axis i/j, minor step +/-).  One
//     256-bit load (LDG.E.256) per block brings every pixel a strip can touch in that block; the strip is then
//     tested in registers, 5 instructions per pixel, no further memory traffic;
//   * pixel k of the line is a + k*U + floor(k*dy/dx)*V (closed form, A5) and floor(k*dy/dx) = hi32(k*S + 2^16) with
//     S = min(floor(dy*2^32/dx), 2^32-1): ONE integer multiply-add, exact for dx < 2^15 (proof in DESIGN.md 3.1,
//     exhaustive check in tests/test_oracle_golden.py).
// Work is flattened as in v2: the strips of a warp's 32 edges are cut into items of E3_G consecutive strips of one edge.
// Pass 1 runs in two phases: every lane first takes its own edge's first item, then the remaining items of the edges not
// yet blocked form one sequence that the lanes take in turn.  Items with undecided strips are queued in shared memory and
// resolved strip by strip by full warps afterwards; strips of edges already known to be blocked are dropped.  Blocks
// containing gray pixels (door zones: zone ids and the reference's panics matter) go to a per-pixel pass over the fused
// byte grid; whenever the ORDER of events along the line could matter the edge is re-walked sequentially
// (walk_sequential), which is what makes the panic codes bit-exact.
#include "edge_common.cuh"

// Per-edge record in shared memory, three 16-byte chunks.  The minor axis is MIRRORED for edges whose minor step is
// -1 (n' = 16 * blocks_along_minor - 1 - n), so that in (k, n') space every line has a non-negative slope: block row
// bn' = n' >> 4 only ever grows with k, and the real block index is idx_m + bn' * stride_minor with the sign folded
// into stride_minor / idx0.
struct Rec3 {
  // chunk 0
  int32_t lo_raw0;          // k of the first position (in k order) of strip 0's block column (<= 0)
  int32_t idx0;             // block index of (major block of strip 0, mirrored minor block 0)
  int32_t stride_major;     // block-index step per strip (signed)
  int32_t stride_minor;     // block-index step per mirrored minor block (signed)
  // chunk 1
  int32_t n0m;              // (mirrored) minor coordinate of the start pixel
  int32_t dxo;              // octant-space major delta = pixels on the line - 1
  uint32_t S;               // fixed-point slope: minor offset of pixel k = hi32(k * S + 2^16)
  int32_t n_strips;         // 0: nothing to walk here (start or end outside the map)
  // chunk 2
  int32_t c0, n0;           // start pixel: major-axis / real minor-axis coordinate
  int32_t dirs;             // bit0 major axis is i (rows), bit1 major step is -1, bit2 minor step is -1
  int32_t pad;
};

struct WarpMem {
  uint4 rec[3][32];         // Rec3 chunks, chunk-major (conflict-free 16-byte accesses)
  uint32_t obst[32];        // != 0: a blocking pixel is on the line
  uint32_t zmin[32], zmax[32];
  uint32_t qb[E3_QB];       // items (e | first strip << 5, want mask: bit 4g = strip g) in [0, 2 * E3_QI), strip scratch after
  uint32_t qg[E3_QG];       // e | strip << 5
};

// ------------------------------------------------------------------------------------------------ the kernel
// One persistent CTA per SM; blockDim.x / 32 warps, each with its own WarpMem.  dynamic shared memory:
//   [ class plane (m.plane_bytes) | mbarrier (16) | WarpMem x warps ]
template <int KIND, bool INDEXED>
__global__ void __launch_bounds__(E3_MAX_WARPS * 32, 1)
edge_validity_v3_kernel(MapDev m, const double2* __restrict__ from, const double2* __restrict__ to, int64_t n,
                        int32_t* __restrict__ out_vid, int8_t* __restrict__ out_vid8, uint64_t* __restrict__ out_mask,
                        const uint64_t* __restrict__ validities, const int32_t* __restrict__ from_idx,
                        const int32_t* __restrict__ to_idx) {
  extern __shared__ __align__(128) unsigned char smem[];
  uint64_t* s_mbar = (uint64_t*)(smem + m.plane_bytes);
  const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
  WarpMem& wm = *(WarpMem*)(smem + m.plane_bytes + 16 + (size_t)wib * sizeof(WarpMem));
  const uint32_t lt_mask = (1u << lane) - 1u;

  // ---- stage the class plane: bulk-async copies global -> shared, completion counted in bytes on an mbarrier
  if (threadIdx.x == 0) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(smem_u32(s_mbar)));
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(s_mbar)), "r"((uint32_t)m.plane_bytes) : "memory");
    for (int off = 0; off < m.plane_bytes; off += 32768) {
      const int sz = min(32768, m.plane_bytes - off);
      asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_u32(smem + off)),
                   "l"((const unsigned char*)m.plane + off), "r"((uint32_t)sz), "r"(smem_u32(s_mbar))
                   : "memory");
    }
  }
  bool plane_ready = false;

  const int64_t n_warps = (int64_t)gridDim.x * (blockDim.x >> 5);
  const int64_t warp = (int64_t)blockIdx.x * (blockDim.x >> 5) + wib;
  const int cw = m.plane_cw, ch = m.plane_ch;
  int qb_n = 0, qg_n = 0;   // queue fill, warp-uniform

  // ---- resolution of the queued strips
  auto drain = [&]() {
    __syncwarp();
    // (1) bitmap strips.  The queue holds ITEMS (edge, first strip, mask of the strips that need their bitmaps) in
    // qb[0 .. 2 * E3_QI); per group of 32 items the strips are written out to qb[2 * E3_QI ..) -- prefix sums of the mask
    // popcounts, every lane expands its own item -- so that every lane of a round tests one strip.  Items of edges already
    // blocked contribute nothing.
    for (int i0 = 0; i0 < qb_n; i0 += 32) {
      uint32_t i_ent = 0, i_want = 0;
      if (i0 + lane < qb_n) {
        i_ent = wm.qb[2 * (i0 + lane)]; i_want = wm.qb[2 * (i0 + lane) + 1];
        if (wm.obst[i_ent & 31] != 0) i_want = 0;
      }
      const int i_cnt = __popc(i_want);
      int i_incl = i_cnt;
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) {
        const int t = __shfl_up_sync(0xffffffffu, i_incl, o);
        if (lane >= o) i_incl += t;
      }
      const int live_n = __shfl_sync(0xffffffffu, i_incl, 31);
      uint32_t* qs = wm.qb + 2 * E3_QI;
      for (int pos = i_incl - i_cnt; i_want; i_want &= i_want - 1)
        qs[pos++] = i_ent + ((uint32_t)((__ffs(i_want) - 1) >> 2) << 5);
      __syncwarp();
      for (int q0 = 0; q0 < live_n; q0 += 32) {
        const int q = q0 + lane;
        if (q < live_n) {
          const uint32_t ent = qs[q];
          const int e = ent & 31, ts = (int)(ent >> 5);
          if (wm.obst[e] == 0) {
            const uint4 r0 = wm.rec[0][e], r1 = wm.rec[1][e];
            const int dirs = (int)wm.rec[2][e].z;
            const int dxo = (int)r1.y, n0m = (int)r1.x;
            const uint32_t S = r1.z;
            const int lo_raw = (int)r0.x + ts * E3_BS;
            const int k_lo = max(0, lo_raw), k_hi = min(dxo, lo_raw + E3_BS - 1);
            const bool neg_major = (dirs & 2) != 0;
            const int bn_a = minor_m((uint32_t)k_lo, S, n0m) >> E3_LOG_BS;
            const int bn_b = minor_m((uint32_t)k_hi, S, n0m) >> E3_LOG_BS;
            const int blk_a = (int)r0.y - m.plane_guard + ts * (int)r0.z + bn_a * (int)r0.w;
            const uint32_t* tiles = m.bits + (size_t)(((dirs & 1) << 1) | ((dirs >> 2) & 1)) * (size_t)m.bits_var_words;
            uint32_t A[8], B[8];
#pragma unroll
            for (int w = 0; w < 8; ++w) B[w] = 0;
            ld256(A, tiles + (size_t)blk_a * 8);
            if (bn_b != bn_a) ld256(B, tiles + (size_t)(blk_a + (int)r0.w) * 8);
            // u_t = minor offset (walking direction) of the pixel at major position t, counted from block a's first
            // row: 0..15 in block a, 16..31 in block b.  hi32(Y_t) = u_t - t, Y linear in t.
            const int k0 = neg_major ? lo_raw + E3_BS - 1 : lo_raw;          // k at t = 0
            const int c_hi = n0m - (bn_a << E3_LOG_BS);
            const int t_lo = neg_major ? lo_raw + E3_BS - 1 - k_hi : k_lo - lo_raw;
            const int t_hi = neg_major ? lo_raw + E3_BS - 1 - k_lo : k_hi - lo_raw;
            const uint32_t Vm = ((2u << t_hi) - 1u) & ~((1u << t_lo) - 1u);  // positions that are pixels of this edge
            uint32_t acc = 0;
            uint64_t Y = ((uint64_t)(uint32_t)c_hi << 32) + (uint64_t)((int64_t)k0 * (int64_t)(uint64_t)S) + E3_BIAS;
            const uint64_t D = (neg_major ? (uint64_t)0 - (uint64_t)S : (uint64_t)S) - (1ull << 32);
#pragma unroll
            for (int t = 0; t < E3_BS; ++t) {
              const uint32_t V = (t & 1) ? __byte_perm(A[t >> 1], B[t >> 1], 0x7632) : __byte_perm(A[t >> 1], B[t >> 1], 0x5410);
              const uint32_t x = Vm & (1u << t);
              acc |= __funnelshift_l(x, x, (uint32_t)(Y >> 32)) & V;     // bit t rotated to bit u_t; hi32(Y_t) = u_t - t
              Y += D;
            }
            if (acc) wm.obst[e] = 1;
          }
        }
        __syncwarp();
      }
    }
    // (2) strips through blocks with gray pixels: per pixel on the fused byte grid, 16 lanes per strip
    for (int q0 = 0; q0 < qg_n; q0 += 2) {
      const int q = q0 + (lane >> 4);
      uint32_t code = 255;
      int e = 0;
      if (q < qg_n) {
        const uint32_t ent = wm.qg[q];
        e = ent & 31;
        const int ts = (int)(ent >> 5);
        const uint4 r0 = wm.rec[0][e], r1 = wm.rec[1][e], r2 = wm.rec[2][e];
        const int dirs = (int)r2.z, dxo = (int)r1.y;
        const int lo_raw = (int)r0.x + ts * E3_BS;
        const int k = max(0, lo_raw) + (lane & 15);
        if (k <= min(dxo, lo_raw + E3_BS - 1)) {
          const int mk = minor_m((uint32_t)k, r1.z, 0);
          const int major = (int)r2.x + ((dirs & 2) ? -k : k), minor = (int)r2.y + ((dirs & 4) ? -mk : mk);
          const int i = (dirs & 1) ? major : minor, j = (dirs & 1) ? minor : major;
          code = __ldg(m.grid + tile_addr(i, j, m.tiles_x));
        }
      }
      const bool blocking = KIND == PORRT_DOMAIN_SHELF ? code != 255 : code == 0;
      const bool gray = KIND != PORRT_DOMAIN_SHELF && code != 0 && code != 255;
      const unsigned half_mask = 0xffffu << (lane & 16);
      const unsigned bl = __ballot_sync(0xffffffffu, blocking) & half_mask;
      const unsigned gr_all = __ballot_sync(0xffffffffu, gray);
      if (gr_all) {   // warp-uniform
        uint32_t zmin = gray ? code : 255u, zmax = gray ? code : 0u;
#pragma unroll
        for (int o = 8; o; o >>= 1) {   // within each half warp
          zmin = min(zmin, __shfl_xor_sync(0xffffffffu, zmin, o));
          zmax = max(zmax, __shfl_xor_sync(0xffffffffu, zmax, o));
        }
        if ((gr_all & half_mask) && (lane & 15) == 0) { atomicMin(&wm.zmin[e], zmin); atomicMax(&wm.zmax[e], zmax); }
      }
      if (bl && (lane & 15) == 0) wm.obst[e] = 1;
    }
    __syncwarp();
    qb_n = 0; qg_n = 0;
  };

  for (int64_t base = warp * 32; base < n; base += n_warps * 32) {
    const int64_t eidx = base + lane;
    if (!plane_ready) { mbar_wait0(s_mbar); plane_ready = true; }
    // ---- per-lane setup of one edge
    int my_flags = 0;  // bit0 start outside the map, bit1 end outside
    uint32_t pre_blocked = 0;
    int c0 = 0, n0 = 0, dxo = 0, dyo = 0, dirs = 0, n_strips = 0;
    uint4 r0 = make_uint4(0, 0, 0, 0);
    uint32_t S = 0;
    int n0m = 0;
    if (eidx < n) {
      const double2 a = INDEXED ? from[from_idx[eidx]] : from[eidx];
      const double2 b = INDEXED ? to[to_idx[eidx]] : to[eidx];
      uint32_t ai, aj, bi, bj;
      to_pixel(m, a.x, a.y, ai, aj);
      to_pixel(m, b.x, b.y, bi, bj);
      my_flags = ((ai >= (uint32_t)m.H || aj >= (uint32_t)m.W) ? 1 : 0) | ((bi >= (uint32_t)m.H || bj >= (uint32_t)m.W) ? 2 : 0);
      // line_drawing's octant (Octant::new) reduces to: major axis = the longer delta (ties give the same pixels),
      // unit steps = the signs of the two deltas
      const int di = (int)bi - (int)ai, dj = (int)bj - (int)aj;
      const int adi = abs(di), adj = abs(dj);
      const bool major_i = adi >= adj;
      dxo = major_i ? adi : adj; dyo = major_i ? adj : adi;
      const int d_major = major_i ? di : dj, d_minor = major_i ? dj : di;
      c0 = major_i ? (int)ai : (int)aj; n0 = major_i ? (int)aj : (int)ai;
      dirs = (major_i ? 1 : 0) | (d_major < 0 ? 2 : 0) | (d_minor < 0 ? 4 : 0);
      if (!my_flags) {  // the start pixel blocks: Obstacle at k = 0, nothing to walk (the reference returns at the first pixel)
        const int sb = m.plane_guard + ((int)ai >> E3_LOG_BS) * cw + ((int)aj >> E3_LOG_BS);
        const uint32_t sc = plane_class(smem, (uint32_t)sb);
        pre_blocked = sc == K_BLOCKED ? 1u : 0u;
      }
      if (!my_flags && !pre_blocked) {
        if (dxo > 0) S = slope_fixed_point(dyo, dxo);
        const int sgn = (dirs & 2) ? -1 : 1;
        const int b0 = c0 >> E3_LOG_BS, b1 = (c0 + sgn * dxo) >> E3_LOG_BS;
        n_strips = (b1 > b0 ? b1 - b0 : b0 - b1) + 1;
        const int blocks_minor = major_i ? cw : ch;            // blocks along the minor axis
        int stride_minor = major_i ? 1 : cw;
        int idx0 = m.plane_guard + b0 * (major_i ? cw : 1);
        n0m = n0;
        if (dirs & 4) { n0m = blocks_minor * E3_BS - 1 - n0; idx0 += (blocks_minor - 1) * stride_minor; stride_minor = -stride_minor; }
        r0.x = (uint32_t)(sgn * ((b0 << E3_LOG_BS) - c0) - ((dirs & 2) ? E3_BS - 1 : 0));
        r0.y = (uint32_t)idx0;
        r0.z = (uint32_t)(sgn * (major_i ? cw : 1));
        r0.w = (uint32_t)stride_minor;
      }
    }
    wm.rec[0][lane] = r0;
    wm.rec[1][lane] = make_uint4((uint32_t)n0m, (uint32_t)dxo, S, (uint32_t)n_strips);
    wm.rec[2][lane] = make_uint4((uint32_t)c0, (uint32_t)n0, (uint32_t)dirs, 0u);
    wm.obst[lane] = pre_blocked; wm.zmin[lane] = 255; wm.zmax[lane] = 0;
    // items = groups of E3_G consecutive strips of one edge.  One lane looks at one item per round: classes of the <= 2
    // blocks of each strip from the plane in shared memory.
    const int my_items = (n_strips + E3_G - 1) / E3_G;
    auto process_item = [&](const int e, const int item, const bool has_item) {
      // per strip g the one-hot classes of its blocks OR-ed: bit 4g+1 mixed, 4g+2 blocked, 4g+3 special (4g: free).
      // Branch-free: strips past the end of the edge read the guard zone / neighbouring blocks and are masked out.
      uint32_t cls = 0;
      const int ts0 = has_item ? item * E3_G : 0;
      {
        const uint4 q0 = wm.rec[0][e], q1 = wm.rec[1][e];
        const int sm_ = (int)q0.z, sn_ = (int)q0.w, e_dxo = (int)q1.y, e_n0m = (int)q1.x;
        const uint32_t e_S = q1.z;
        const int left = has_item ? (int)q1.w - ts0 : 0;        // strips of this edge from ts0 on
        int lo_raw = (int)q0.x + ts0 * E3_BS;
        int idx_m = (int)q0.y + ts0 * sm_;
#pragma unroll
        for (int g = 0; g < E3_G; ++g) {
          // only an edge's first strip starts before k = 0; k_lo past the end (masked strips) stays inside the guards
          const int k_lo = g == 0 ? max(0, lo_raw) : lo_raw, k_hi = min(e_dxo, lo_raw + E3_BS - 1);
          const uint32_t na = (uint32_t)minor_m((uint32_t)k_lo, e_S, e_n0m), nb = (uint32_t)minor_m((uint32_t)k_hi, e_S, e_n0m);
          const uint32_t ia = (uint32_t)idx_m + (na >> E3_LOG_BS) * (uint32_t)sn_;
          const uint32_t ib = (uint32_t)idx_m + (nb >> E3_LOG_BS) * (uint32_t)sn_;
          const uint32_t ca = plane_class(smem, ia), cb = plane_class(smem, ib);
          cls += ((1u << ca) | (1u << cb)) * (1u << (4 * g));
          lo_raw += E3_BS; idx_m += sm_;
        }
        cls &= left >= E3_G ? 0xffffffffu : ((1u << (4 * max(left, 0))) - 1u);
      }
      const uint32_t blocked = cls & 0x44444444u, special = (cls >> 3) & 0x11111111u;
      if (blocked) wm.obst[e] = 1;                                 // the bitmaps cannot change the outcome any more
      const uint32_t want = blocked ? 0u : ((cls >> 1) & 0x11111111u & ~special);
      // enqueue the ITEM if any of its strips needs the bitmaps (one ballot; the strips are flattened when the queue is drained)
      {
        const unsigned bal = __ballot_sync(0xffffffffu, want != 0);
        if (bal) {
          if (want) {
            const int pos = 2 * (qb_n + __popc(bal & lt_mask));
            wm.qb[pos] = (uint32_t)e | ((uint32_t)ts0 << 5);
            wm.qb[pos + 1] = want;
          }
          qb_n += __popc(bal);
        }
      }
      if (__any_sync(0xffffffffu, special != 0)) {                 // rare: strips through gray pixels
#pragma unroll
        for (int g = 0; g < E3_G; ++g) {
          const unsigned bal = __ballot_sync(0xffffffffu, (special >> (4 * g)) & 1u);
          if ((special >> (4 * g)) & 1u) wm.qg[qg_n + __popc(bal & lt_mask)] = (uint32_t)e | ((uint32_t)(ts0 + g) << 5);
          qg_n += __popc(bal);
        }
      }
    };
    // Round 0: every lane takes the FIRST item of its own edge (no owner search).  Edges found blocked there -- an
    // all-blocking block within their first 112 pixels -- are finished: what lies behind the first obstacle cannot
    // change the result (the reference returns at it), so their remaining items are never looked at.  The queues are not
    // drained between the two phases: that lets more edges finish early but costs more than it saves (0.905 against 0.760 ms).
    __syncwarp();
    process_item(lane, 0, my_items > 0);
    __syncwarp();
    int rem = (my_items <= 1 || wm.obst[lane] != 0) ? 0 : my_items - 1;
    int incl = rem;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const int t = __shfl_up_sync(0xffffffffu, incl, o);
      if (lane >= o) incl += t;
    }
    const int total = __shfl_sync(0xffffffffu, incl, 31);
    for (int w0 = 0; w0 < total; w0 += 32) {
      if (qb_n > E3_QB_LIMIT || qg_n > E3_QG - 32 * E3_G) drain();
      const int w = w0 + lane;
      int e = 0;                                                    // owner: the first lane whose inclusive sum exceeds w
#pragma unroll
      for (int sft = 16; sft >= 1; sft >>= 1) {
        const int v = __shfl_sync(0xffffffffu, incl, e + sft - 1);
        if (v <= w) e += sft;
      }
      const int excl = __shfl_sync(0xffffffffu, incl - rem, e);
      process_item(e, 1 + w - excl, w < total);
      __syncwarp();
    }
    // ---- pass 2: bitmaps / pixels of the strips that are still undecided
    if (qb_n | qg_n) drain();
    __syncwarp();

    // ---- results
    if (eidx < n) {
      int32_t r;
      bool slow = false;
      if (my_flags & 1) r = PORRT_PANIC_OOB;             // the first pixel read already panics
      else if (my_flags & 2) slow = true;                // end pixel outside: order of events matters
      else {
        const bool is_blocked = wm.obst[lane] != 0;
        if (KIND == PORRT_DOMAIN_SHELF) r = is_blocked ? R_BLOCKED : R_FREE;   // Low and High obstacle both invalidate the edge
        else {
          const uint32_t zmin = wm.zmin[lane], zmax = wm.zmax[lane];
          if (zmax != 0 && (zmin != zmax || zmax == 254)) slow = true;         // order of events decides: re-walk
          else r = is_blocked ? R_BLOCKED : (zmax ? (int32_t)zmin - 1 : R_FREE);
        }
      }
      if (slow) {
        Walker wk;
        const int sm = (dirs & 2) ? -1 : 1, sn = (dirs & 4) ? -1 : 1;
        wk.dxo = dxo; wk.dyo = dyo;
        wk.M = dxo > 1 ? (0xFFFFFFFFFFFFFFFFull / (uint64_t)dxo) + 1ull : 0ull;
        if (dirs & 1) { wk.ai = c0; wk.aj = n0; wk.ui = sm; wk.uj = 0; wk.vi = 0; wk.vj = sn; }
        else { wk.ai = n0; wk.aj = c0; wk.ui = 0; wk.uj = sm; wk.vi = sn; wk.vj = 0; }
        r = walk_sequential<KIND>(m, wk);
        if (KIND == PORRT_DOMAIN_SHELF && r == R_LOW) r = R_BLOCKED;
      }
      store_edge_result(m, eidx, walk_to_validity(m, r), out_vid, out_vid8, out_mask, validities);
    }
    __syncwarp();
  }
  if (!plane_ready) mbar_wait0(s_mbar);  // a warp without work must not leave while the copy is in flight
}

// ------------------------------------------------------------------------------------------------ map build
// One thread per (block, row): 16 fused codes -> 16-bit blocking mask of the row; the column vectors come from
// ballots (a warp holds the 16 rows of two blocks).  Writes the four bitmap orientations and the class plane.
//   orientation 0: major j, minor i ascending  : vec[t = column] bit r        1: the same with bit 15 - r
//   orientation 2: major i, minor j ascending  : vec[t = row]    bit c        3: the same with bit 15 - c
template <int KIND>
__global__ void __launch_bounds__(256) edge3_build_kernel(const uint8_t* __restrict__ grid, int H, int W, int tiles_x, int cw, int ch,
                                                          uint32_t* __restrict__ plane, int guard, uint16_t* __restrict__ bits, size_t var_halfwords) {
  const int lane = threadIdx.x & 31, half = lane >> 4, r = lane & 15;
  const int64_t pair = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int64_t n_blocks = (int64_t)cw * ch;
  const int64_t blk = pair * 2 + half;
  const bool have = blk < n_blocks;
  const int bi = have ? (int)(blk / cw) : 0, bj = have ? (int)(blk % cw) : 0;
  const int i = bi * E3_BS + r;
  uint32_t rowmask = 0, n_in = 0, n_block = 0, n_special = 0;
  if (have && i < H) {
#pragma unroll
    for (int c = 0; c < E3_BS; ++c) {
      const int j = bj * E3_BS + c;
      if (j < W) {
        const uint32_t code = grid[tile_addr(i, j, tiles_x)];
        ++n_in;
        const bool blocking = KIND == PORRT_DOMAIN_SHELF ? code != 255 : code == 0;
        if (blocking) { rowmask |= 1u << c; ++n_block; }
        else if (code != 255) ++n_special;
      }
    }
  }
  uint32_t colvec = 0;
#pragma unroll
  for (int c = 0; c < E3_BS; ++c) {
    const uint32_t bal = __ballot_sync(0xffffffffu, (rowmask >> c) & 1u);
    if (r == c) colvec = (bal >> (16 * half)) & 0xffffu;
  }
  uint32_t cnt = n_in | (n_block << 10) | (n_special << 20);   // <= 256 each: three 10-bit counters
#pragma unroll
  for (int o = 8; o; o >>= 1) cnt += __shfl_xor_sync(0xffffffffu, cnt, o);
  if (have) {
    uint16_t* t0 = bits + (size_t)blk * 16 + r;
    t0[0] = (uint16_t)colvec;
    t0[var_halfwords] = (uint16_t)(__brev(colvec) >> 16);
    t0[2 * var_halfwords] = (uint16_t)rowmask;
    t0[3 * var_halfwords] = (uint16_t)(__brev(rowmask) >> 16);
    if (r == 0) {
      const uint32_t t_in = cnt & 1023u, t_block = (cnt >> 10) & 1023u, t_special = cnt >> 20;
      const uint32_t cls = t_special ? K_SPECIAL : (t_block == 0 ? K_FREE : (t_block == t_in ? K_BLOCKED : K_MIXED));
      const int64_t pb = blk + guard;
      if (cls) atomicOr(&plane[pb >> 4], cls << ((pb & 15) << 1));
    }
  }
}

int32_t edge3_build(porrt_ctx* ctx, cudaStream_t st) {
  MapDev& m = ctx->map;
  const int cw = (m.W + E3_BS - 1) / E3_BS, ch = (m.H + E3_BS - 1) / E3_BS;
  const size_t n_blocks = (size_t)cw * ch;
  // guard zones of >= 4 block rows (class 0 = free) on both sides: the branch-free pass 1 reads up to E3_G - 1 strips
  // past the end of an edge, i.e. at most E3_G block rows / columns outside the map
  const int guard = (int)(((size_t)(E3_G + 1) * cw + 63) / 64 * 64);
  const size_t plane_bytes = ((((n_blocks + 2 * (size_t)guard + 15) / 16) * 4 + 15) / 16) * 16;
  CUDA_TRY(ctx, ctx->d_plane.ensure(plane_bytes));
  CUDA_TRY(ctx, ctx->d_bits.ensure(n_blocks * 32 * 4));
  CUDA_TRY(ctx, cudaMemsetAsync(ctx->d_plane.p, 0, plane_bytes, st));
  const int grid = div_up((int64_t)((n_blocks + 1) / 2) * 32, 256);
  if (m.kind == PORRT_DOMAIN_SHELF)
    edge3_build_kernel<PORRT_DOMAIN_SHELF><<<grid, 256, 0, st>>>(m.grid, m.H, m.W, m.tiles_x, cw, ch, ctx->d_plane.as<uint32_t>(), guard, ctx->d_bits.as<uint16_t>(), n_blocks * 16);
  else
    edge3_build_kernel<PORRT_DOMAIN_DOOR><<<grid, 256, 0, st>>>(m.grid, m.H, m.W, m.tiles_x, cw, ch, ctx->d_plane.as<uint32_t>(), guard, ctx->d_bits.as<uint16_t>(), n_blocks * 16);
  LAUNCH_CHECK(ctx);
  m.plane = ctx->d_plane.as<uint32_t>();
  m.bits = ctx->d_bits.as<uint32_t>();
  m.plane_cw = cw;
  m.plane_ch = ch;
  m.plane_guard = guard;
  m.plane_bytes = (int32_t)plane_bytes;
  m.bits_var_words = (int32_t)(n_blocks * 8);
  return PORRT_OK;
}

static const int E3_SMEM_LIMIT = 227 * 1024;

static int edge3_max_warps(const porrt_ctx* ctx) {
  const int64_t room = (int64_t)E3_SMEM_LIMIT - ctx->map.plane_bytes - 16;
  const int64_t w = room / (int64_t)sizeof(WarpMem);
  return (int)(w > E3_MAX_WARPS ? E3_MAX_WARPS : w);
}

// the class plane has to fit in shared memory next to at least 8 warps' queues, and dx < 2^15 (exact slope)
bool edge3_usable(const porrt_ctx* ctx) {
  return ctx->map.plane != nullptr && edge3_max_warps(ctx) >= 8 && ctx->map.H <= 32768 && ctx->map.W <= 32768;
}

template <int KIND, bool INDEXED>
static int32_t edge3_launch_t(porrt_ctx* ctx, const double2* from, const double2* to, int64_t n, const EdgeOut& out,
                              const int32_t* from_idx, const int32_t* to_idx, cudaStream_t st) {
  auto kern = edge_validity_v3_kernel<KIND, INDEXED>;
  static bool attr_set[16] = {};
  if (!attr_set[ctx->device & 15]) {
    CUDA_TRY(ctx, cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, E3_SMEM_LIMIT));
    attr_set[ctx->device & 15] = true;
  }
  const int max_warps = edge3_max_warps(ctx);
  const int64_t warps_needed = (n + 31) / 32;
  // one CTA per SM; small batches are spread over the SMs with fewer warps each
  int warps = (int)((warps_needed + ctx->sm_count - 1) / ctx->sm_count);
  warps = warps < 4 ? 4 : (warps > max_warps ? max_warps : warps);
  int64_t ctas = (warps_needed + warps - 1) / warps;
  if (ctas > ctx->sm_count) ctas = ctx->sm_count;
  const size_t smem = (size_t)ctx->map.plane_bytes + 16 + (size_t)warps * sizeof(WarpMem);
  kern<<<(int)ctas, warps * 32, smem, st>>>(ctx->map, from, to, n, out.vid, out.vid8, out.mask, ctx->d_validities.as<uint64_t>(), from_idx, to_idx);
  LAUNCH_CHECK(ctx);
  return PORRT_OK;
}

int32_t edge3_launch(porrt_ctx* ctx, const double* from_dev, const double* to_dev, int64_t n, const EdgeOut& out,
                     const int32_t* from_idx_dev, const int32_t* to_idx_dev, cudaStream_t st) {
  const double2* f = (const double2*)from_dev;
  const double2* t = (const double2*)to_dev;
  const bool shelf = ctx->map.kind == PORRT_DOMAIN_SHELF;
  if (from_idx_dev)
    return shelf ? edge3_launch_t<PORRT_DOMAIN_SHELF, true>(ctx, f, t, n, out, from_idx_dev, to_idx_dev, st)
                 : edge3_launch_t<PORRT_DOMAIN_DOOR, true>(ctx, f, t, n, out, from_idx_dev, to_idx_dev, st);
  return shelf ? edge3_launch_t<PORRT_DOMAIN_SHELF, false>(ctx, f, t, n, out, nullptr, nullptr, st)
               : edge3_launch_t<PORRT_DOMAIN_DOOR, false>(ctx, f, t, n, out, nullptr, nullptr, st);
}
