// edge_common.cuh -- constants and device helpers of the edge-validity kernel (edge3.cu)
#pragma once
#include "map_dev.cuh"

#define E3_LOG_BS 4
#define E3_BS 16
#define E3_G 7              // consecutive strips of one edge per item (<= 8: one class nibble each); measured with the
                            // two-phase pass 1 on c5: G = 4 / 5 / 6 / 7 / 8 -> 0.768 / 0.754 / 0.721 / 0.710 / 0.760 ms
#define E3_QB 512           // bitmap-queue words per warp: items, then the strip scratch they are flattened into
#define E3_QG 256           // byte-queue entries per warp
#define E3_QI ((E3_QB - 32 * 8) / 2)          // item entries (2 words each) in front of the strip scratch (32 items x 8 strips)
#define E3_QB_LIMIT (E3_QI - 32)              // items; a round adds at most 32
#define E3_BIAS 65536ull
#define E3_MAX_WARPS 32

#define K_FREE 0u
#define K_MIXED 1u          // blocking and free pixels, nothing else: the bitmap decides
#define K_BLOCKED 2u        // every pixel blocks
#define K_SPECIAL 3u        // contains gray pixels (DOOR zones / gray without zone id): per-pixel pass on the byte grid

// Fixed-point slope S ~ dy * 2^32 / dx for 0 <= dy <= dx < 2^15.  hi32(k * S + 2^16) == floor(k * dy / dx) for every
// 0 <= k <= dx as long as |dy * 2^32 / dx - S| < 1.9 (DESIGN.md 3.1), so S need not be the exact floor: one correctly
// rounded reciprocal, one multiply and a saturating conversion (dy == dx -> 2^32 - 1) on the FP64 pipe replace two 32-bit
// integer divisions (~40 ALU/FMA instructions, the pipes that bound the kernel).
// tests/test_oracle_golden.py::test_fixed_point_minor_offset_is_exact replays this and the exact division in IEEE arithmetic.
__device__ __forceinline__ uint32_t slope_fixed_point(int dy, int dx) {
  return __double2uint_rz(__dmul_rn(__dmul_rn((double)dy, 4294967296.0), __drcp_rn((double)dx)));
}

// n' of pixel k = hi32(k * S + (n0m << 32 | 2^16))
__device__ __forceinline__ int32_t minor_m(uint32_t k, uint32_t S, int32_t n0m) {
  return (int32_t)(((uint64_t)k * (uint64_t)S + (((uint64_t)(uint32_t)n0m << 32) | E3_BIAS)) >> 32);
}


// 2-bit class of block idx from the plane in shared memory (16 per 32-bit word) by a byte load; word loads with a rotate
// were measured slower (DESIGN.md 3.1)
__device__ __forceinline__ uint32_t plane_class(const unsigned char* plane, uint32_t idx) {
  return ((uint32_t)plane[idx >> 2] >> ((idx * 2u) & 6u)) & 3u;
}

__device__ __forceinline__ void ld256(uint32_t (&v)[8], const uint32_t* p) {
  asm volatile("ld.global.nc.v8.u32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
               : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7])
               : "l"(p));
}

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_wait0(uint64_t* bar) {
  uint32_t done = 0;
  while (!done)
    asm volatile("{ .reg .pred p; mbarrier.try_wait.parity.shared::cta.b64 p, [%1], 0; selp.u32 %0, 1, 0, p; }"
                 : "=r"(done) : "r"(smem_u32(bar)) : "memory");
}

