// diag.cu -- measurement aids exported next to the product (bench.py's roofline denominators); no planner functionality.
//
// porrt_measure_l2_gather: the L2-resident gather rate SURVEY.md 8(d) asks the builder to measure -- random, independent
// 32-byte sector reads (one LDG.E.256 per lane, the edge kernel's bitmap access) over a buffer that fits the 126 MB L2.
#include "common.cuh"

__global__ void __launch_bounds__(256) l2_gather_kernel(const uint32_t* __restrict__ buf, uint32_t n_sectors_mask, int rounds,
                                                        uint32_t seed, uint32_t* __restrict__ sink) {
  uint32_t x = (blockIdx.x * blockDim.x + threadIdx.x) * 2654435761u + seed;
  uint32_t acc = 0;
#pragma unroll 4
  for (int r = 0; r < rounds; ++r) {
    x ^= x << 13; x ^= x >> 17; x ^= x << 5;                       // xorshift32: independent addresses, no dependent loads
    const uint32_t* p = buf + (size_t)(x & n_sectors_mask) * 8;
    uint32_t v[8];
    asm volatile("ld.global.nc.v8.u32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
                 : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7])
                 : "l"(p));
    acc += v[0] ^ v[1] ^ v[2] ^ v[3] ^ v[4] ^ v[5] ^ v[6] ^ v[7];
  }
  if (acc == 0x9e3779b9u) *sink = acc;                              // keeps the loads alive
}

// buffer_bytes: rounded down to a power of two (default 64 MiB when <= 0).  *out_gbs = bytes gathered / time of the best of
// five timed launches after a warm-up launch that pulls the buffer into L2.
PORRT_API int32_t porrt_measure_l2_gather(porrt_ctx* ctx, int64_t buffer_bytes, double* out_gbs) {
  CTX_CHECK(ctx);
  if (!out_gbs) return porrt_fail(ctx, PORRT_ERR_INVALID_ARG, "porrt_measure_l2_gather: null output");
  CUDA_TRY(ctx, cudaSetDevice(ctx->device));
  if (buffer_bytes <= 0) buffer_bytes = 64ll << 20;
  int64_t bytes = 1 << 20;
  while (bytes * 2 <= buffer_bytes && bytes < (1ll << 32)) bytes *= 2;
  DevBuf buf;
  CUDA_TRY(ctx, buf.ensure((size_t)bytes + 64));
  cudaStream_t st = ctx->stream;
  CUDA_TRY(ctx, cudaMemsetAsync(buf.p, 1, (size_t)bytes, st));
  CUDA_TRY(ctx, ctx->ws_query.ensure(16));
  const uint32_t mask = (uint32_t)(bytes / 32 - 1);
  const int rounds = 256, blocks = ctx->sm_count * 32;
  cudaEvent_t e0, e1;
  CUDA_TRY(ctx, cudaEventCreate(&e0));
  CUDA_TRY(ctx, cudaEventCreate(&e1));
  double best = 0.0;
  for (int it = 0; it < 6; ++it) {
    cudaEventRecord(e0, st);
    l2_gather_kernel<<<blocks, 256, 0, st>>>(buf.as<uint32_t>(), mask, rounds, 12345u + it, ctx->ws_query.as<uint32_t>());
    ctx->launches += 1;
    cudaEventRecord(e1, st);
    if (cudaEventSynchronize(e1) != cudaSuccess) break;
    float ms = 0.f;
    cudaEventElapsedTime(&ms, e0, e1);
    const double gbs = (double)blocks * 256.0 * rounds * 32.0 / (ms * 1e-3) / 1e9;
    if (it > 0 && gbs > best) best = gbs;
  }
  cudaEventDestroy(e0); cudaEventDestroy(e1);
  buf.release();
  CUDA_TRY(ctx, cudaGetLastError());
  *out_gbs = best;
  return PORRT_OK;
}
