// sssp_frontier.cuh -- frontier relaxation over value tables in global memory (sssp_frontier.cu), the schedule of graph.cu's
// value-column driver for roadmaps too large for the on-chip column solver: plan_qmdp's world columns and porrt_belief_vi's belief
// columns.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

struct porrt_ctx;
struct Carve;

struct SfGraph {             // a roadmap in Morton numbering with its TRANSPOSED adjacency (device pointers, ctx scratch)
  int64_t V, E;
  const int64_t* row_t;      // [V + 1]
  const int32_t* col_t;      // parents (Morton numbering)
  const double* cost_t;      // norm2 of the edge
  const uint16_t* evid_t;    // validity id of the edge (null when built without edge validity ids)
  const uint32_t* order;     // order[pos] = node
  const int32_t* perm;       // perm[node] = pos
  double delta;              // threshold step of the near / far ordering (mean edge length)
};

int32_t sf_build_graph(porrt_ctx* ctx, const int64_t* d_row, const int32_t* d_col, const int32_t* d_evid, const double* d_xy, int64_t V,
                       int64_t E, SfGraph* out, cudaStream_t st);
int32_t sf_relax(porrt_ctx* ctx, const SfGraph& g, double* dist, int32_t W, const uint64_t* cmask, int32_t* out_rounds, double* out_offers,
                 cudaStream_t st);
// Takes sf_relax's state over up to W columns from the front of a ws_state layout: what the caller takes behind it stays in place
// while sf_relax runs on at most W columns.
void sf_state_reserve(Carve& c, int64_t V, int32_t W);
