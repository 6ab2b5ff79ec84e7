// ctx.cu -- context lifetime, stream plumbing (no compute kernels here).
#include <ctype.h>
#include <sched.h>

#include <cstdlib>

#include "common.cuh"

PORRT_API const char* porrt_version(void) { return "porrt_b200 0.1 (sm_100a)"; }

PORRT_API int32_t porrt_ctx_create(int32_t device, porrt_ctx** out_ctx) {
  if (!out_ctx) return PORRT_ERR_INVALID_ARG;
  *out_ctx = nullptr;
  int count = 0;
  if (cudaGetDeviceCount(&count) != cudaSuccess || count == 0 || device < 0 || device >= count) {
    cudaGetLastError();
    return PORRT_ERR_CUDA;  // no CPU fallback: the library is unusable without a device
  }
  cudaDeviceProp prop;
  if (cudaGetDeviceProperties(&prop, device) != cudaSuccess) return PORRT_ERR_CUDA;
  if (prop.major != 10) return PORRT_ERR_UNSUPPORTED;  // built for sm_100a only
  if (cudaSetDevice(device) != cudaSuccess) return PORRT_ERR_CUDA;
  porrt_ctx* ctx = new porrt_ctx();
  ctx->device = device;
  ctx->sm_count = prop.multiProcessorCount;
  int prio_least = 0, prio_greatest = 0;
  cudaDeviceGetStreamPriorityRange(&prio_least, &prio_greatest);
  // the helper stream (graph.cu: kd rank next to the radius / edge batches) outranks the main compute stream: its ~170 tiny,
  // latency-bound kernels are what the PRM build ends up waiting for, and they cost the long kernels next to them almost nothing
  // (measured at 1e6 nodes, interleaved: 9.97-10.04 ms against 10.11-10.20 ms with the priorities the other way round)
  bool ok = cudaStreamCreateWithPriority(&ctx->own_stream, cudaStreamNonBlocking, prio_least) == cudaSuccess &&
            cudaStreamCreateWithPriority(&ctx->aux_stream, cudaStreamNonBlocking, prio_greatest) == cudaSuccess &&
            cudaStreamCreateWithFlags(&ctx->copy_in, cudaStreamNonBlocking) == cudaSuccess &&
            cudaStreamCreateWithFlags(&ctx->copy_out, cudaStreamNonBlocking) == cudaSuccess;
  for (int s = 0; ok && s < MAX_SLOTS; ++s)
    ok = cudaEventCreateWithFlags(&ctx->ev_in[s], cudaEventDisableTiming) == cudaSuccess &&
         cudaEventCreateWithFlags(&ctx->ev_k[s], cudaEventDisableTiming) == cudaSuccess &&
         cudaEventCreateWithFlags(&ctx->ev_out[s], cudaEventDisableTiming) == cudaSuccess;
  for (int s = 0; ok && s < 16; ++s) ok = cudaEventCreate(&ctx->ev_t[s]) == cudaSuccess;
  if (!ok) { cudaGetLastError(); porrt_ctx_destroy(ctx); return PORRT_ERR_CUDA; }  // releases whatever was created so far
  ctx->stream = ctx->own_stream;
  *out_ctx = ctx;
  return PORRT_OK;
}

PORRT_API int32_t porrt_ctx_destroy(porrt_ctx* ctx) {
  CTX_CHECK(ctx);
  cudaSetDevice(ctx->device);
  cudaDeviceSynchronize();
  porrt_comm_destroy(ctx);
  ctx->d_grid.release(); ctx->d_coarse.release(); ctx->d_validities.release(); ctx->d_zone_pos.release();
  ctx->d_plane.release(); ctx->d_bits.release();
  ctx->d_vxy_sorted.release(); ctx->d_vid_sorted.release(); ctx->d_cell_start.release();
  ctx->d_vxy.release(); ctx->d_vcell.release();
  ctx->nn_bins.release();
  ctx->nn_stage.release(); ctx->nn_stage2.release(); ctx->comm_tmp.release(); ctx->d_nbr_start.release(); ctx->d_nbr_script.release();
  for (DevBuf* b : {&ctx->ws_main, &ctx->ws_owner, &ctx->ws_vid, &ctx->ws_table, &ctx->ws_query, &ctx->ws_seg, &ctx->sort_keys,
                    &ctx->sort_vals, &ctx->ws_state, &ctx->radix_keys, &ctx->radix_vals, &ctx->radix_hist, &ctx->scan_sums})
    b->release();
  pto_grow_release(ctx);
  ctx->kd_buf.release(); ctx->d_prm_row.release(); ctx->d_prm_col.release(); ctx->d_bel_succ.release(); ctx->bel.dev.release();
  if (ctx->aux_stream) cudaStreamDestroy(ctx->aux_stream);
  for (PinBuf* b : {&ctx->pin_edge, &ctx->pin_radii, &ctx->pin_bel, &ctx->pin_row, &ctx->pin_col, &ctx->pin_flags}) b->release();
  for (int s = 0; s < MAX_SLOTS; ++s) {
    if (ctx->ev_in[s]) cudaEventDestroy(ctx->ev_in[s]);
    if (ctx->ev_k[s]) cudaEventDestroy(ctx->ev_k[s]);
    if (ctx->ev_out[s]) cudaEventDestroy(ctx->ev_out[s]);
  }
  for (int s = 0; s < 16; ++s) if (ctx->ev_t[s]) cudaEventDestroy(ctx->ev_t[s]);
  if (ctx->own_stream) cudaStreamDestroy(ctx->own_stream);
  if (ctx->copy_in) cudaStreamDestroy(ctx->copy_in);
  if (ctx->copy_out) cudaStreamDestroy(ctx->copy_out);
  delete ctx;
  return PORRT_OK;
}

PORRT_API int32_t porrt_ctx_set_stream(porrt_ctx* ctx, void* cuda_stream) {
  CTX_CHECK(ctx);
  ctx->stream = cuda_stream ? (cudaStream_t)cuda_stream : ctx->own_stream;
  return PORRT_OK;
}

PORRT_API int32_t porrt_ctx_synchronize(porrt_ctx* ctx) {
  CTX_CHECK(ctx);
  CUDA_TRY(ctx, cudaSetDevice(ctx->device));
  CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
  return PORRT_OK;
}

// Host-side locality for the H2D / D2H pipelines: bind the CALLING thread to the CPUs of the NUMA node the ctx's GPU hangs off
// (sysfs: /sys/bus/pci/devices/<bus id>/numa_node -> /sys/devices/system/node/node<N>/cpulist).  Pinned buffers touched after
// this call land on that node (first touch), so N processes on a two-socket box do not push their copies through the socket
// interconnect.  *out_node = the node (-1: unknown, nothing changed).  The reference is single-threaded; this is deployment glue.
PORRT_API int32_t porrt_ctx_bind_host_thread(porrt_ctx* ctx, int32_t* out_node) {
  CTX_CHECK(ctx);
  if (out_node) *out_node = -1;
  char bus[32] = {0};
  CUDA_TRY(ctx, cudaDeviceGetPCIBusId(bus, sizeof(bus), ctx->device));
  for (char* c = bus; *c; ++c) *c = (char)tolower(*c);
  char path[160];
  snprintf(path, sizeof(path), "/sys/bus/pci/devices/%s/numa_node", bus);
  FILE* f = fopen(path, "r");
  if (!f) return PORRT_OK;
  int node = -1;
  if (fscanf(f, "%d", &node) != 1) node = -1;
  fclose(f);
  if (node < 0) return PORRT_OK;
  snprintf(path, sizeof(path), "/sys/devices/system/node/node%d/cpulist", node);
  f = fopen(path, "r");
  if (!f) return PORRT_OK;
  char list[4096] = {0};
  const bool got = fgets(list, sizeof(list), f) != nullptr;
  fclose(f);
  if (!got) return PORRT_OK;
  cpu_set_t set;
  CPU_ZERO(&set);
  int n_cpus = 0;
  for (char* tok = strtok(list, ",\n"); tok; tok = strtok(nullptr, ",\n")) {
    int a = 0, b = 0;
    const int k = sscanf(tok, "%d-%d", &a, &b);
    if (k == 1) b = a;
    if (k < 1) continue;
    for (int c = a; c <= b && c < CPU_SETSIZE; ++c) { CPU_SET(c, &set); ++n_cpus; }
  }
  if (n_cpus == 0) return PORRT_OK;
  // keep only CPUs this process is allowed to use (containers): an empty intersection leaves the affinity alone
  cpu_set_t cur, both;
  if (sched_getaffinity(0, sizeof(cur), &cur) == 0) {
    CPU_AND(&both, &set, &cur);
    if (CPU_COUNT(&both) == 0) return PORRT_OK;
    set = both;
  }
  if (sched_setaffinity(0, sizeof(set), &set) != 0) return PORRT_OK;
  if (out_node) *out_node = node;
  return PORRT_OK;
}

PORRT_API const char* porrt_last_error(porrt_ctx* ctx) { return ctx ? ctx->err.c_str() : "null ctx"; }
PORRT_API int64_t porrt_ctx_launch_count(porrt_ctx* ctx) { return ctx ? ctx->launches : 0; }

PORRT_API int32_t porrt_ctx_last_phase_ms(porrt_ctx* ctx, double* out_ms, int32_t cap, int32_t* out_n) {
  CTX_CHECK(ctx);
  int n = ctx->n_last < cap ? ctx->n_last : cap;
  for (int k = 0; k < n; ++k) out_ms[k] = ctx->last_ms[k];
  if (out_n) *out_n = n;
  return PORRT_OK;
}
