// colsolve.cuh -- interface of the shared-memory column solver (colsolve.cu) used by graph.cu.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

struct porrt_ctx;

#define COLSOLVE_THREADS 1024
#define COLSOLVE_LANES 4                 // lanes that share one node's edge list
#define COLSOLVE_UNROLL 8                // edge records a lane loads ahead
#define COLSOLVE_QCAP 1024              // dirty nodes a CTA works off per round
#define COLSOLVE_SMEM_MAX (227 * 1024)   // opt-in dynamic shared memory per CTA on sm_100
enum { COLSOLVE_BELIEF = 0, COLSOLVE_WORLD = 1 };

struct ColSolveArgs {
  // TRANSPOSED adjacency (colsolve_pack): row v lists the parents u of v
  const uint32_t* row_start;   // [V + 1]
  const double* cost;          // [E] norm2 of the edge's end points
  const uint32_t* ce;          // [E] parent node | validity id of the edge parent -> v << 16
  int32_t V;
  int64_t ld;                  // column pitch of dist_cm in doubles (>= V)
  double* dist_cm;             // [n_columns][ld]: +inf / 0 at the finals on entry, the column's values on exit
  const uint64_t* cmask;       // [n_columns][4]: validity ids the column admits (belief: compat[b][.]; world: validities[.] bit w)
  const int32_t* nvid;         // [V] node validity ids (may be null in world mode: every node valid)
  // belief mode only
  const uint8_t* type_cm;      // [n_columns][V] PORRT_NODE_* (255 = the belief node does not exist)
  const int32_t* node_set;     // [V] index of the node's visible-zone set
  const int32_t* col_belief;   // [positions] the column at a position (belief id), -1 = padding
  const int64_t* succ_ptr;     // [n_sets * B + 1]
  const int32_t* succ_col;     // successor COLUMNS (positions, not belief ids)
  const double* succ_p;
  int32_t B;
  int32_t* sweeps_out;         // max over CTAs (atomicMax), may be null
  unsigned long long* offers_out;   // += edge records worked through (12 bytes each from L2), may be null
};

bool colsolve_fits(int64_t V, int64_t E, int32_t n_validities);
int32_t colsolve_pack(porrt_ctx* ctx, const int64_t* row_ptr_dev, const int32_t* col_dev, const int32_t* evid_dev, const double* cost_dev,
                      int64_t V, int64_t E, uint32_t* row_start_t, uint32_t* ce_t, double* cost_t, uint32_t* cursor_tmp, cudaStream_t st);
int32_t colsolve_level(porrt_ctx* ctx, const ColSolveArgs& a, int mode, int col_lo, int col_hi, cudaStream_t st);
int32_t colsolve_level_batch(porrt_ctx* ctx, const ColSolveArgs* descs_dev, int n_roads, int32_t V_max, int col_lo, int col_hi,
                             cudaStream_t st);
