// belief_tables.cuh -- device-built observation successor tables (belief_tables.cu) for graph.cu's porrt_belief_vi.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include <vector>

struct porrt_ctx;

struct BeliefSuccDev {        // device pointers (ctx->d_bel_succ / ws_query), valid until the next belief_vi call
  int64_t* succ_ptr;          // [n_sets * B + 1]
  int32_t* succ_b;            // successor belief ids, emission order of observe()
  int32_t* succ_col;          // the same as columns of colsolve.cu (colpos[succ_b])
  double* succ_p;             // transition_probability(belief, successor)
  int64_t n_succ;
  bool levels_ok;             // every successor has a strictly smaller support than its parent
  const double* beliefs;      // [B][nw] device copy of the reachable belief states
};

// sets: distinct visible-zone masks; bhash: common.rs:352-355 of every belief; level: support sizes; colpos: column of a belief.
// Synchronises `st` once (the number of edges sizes the output).  PORRT_ERR_PANIC where the reference panics.
int32_t belief_succ_tables(porrt_ctx* ctx, const double* beliefs_host, int32_t B, int32_t nw, const std::vector<uint64_t>& sets,
                           const std::vector<uint64_t>& bhash, const std::vector<int32_t>& level, const std::vector<int32_t>& colpos,
                           BeliefSuccDev* out, cudaStream_t st);
