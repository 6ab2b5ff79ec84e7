/* porrt_b200.h -- C ABI of libporrt_b200.so: the B200 (sm_100a) implementation of po-rrt's data-parallel
 * planning inner loop (SURVEY.md section 8).  This is the drop-in boundary: a Rust `extern "C"` block
 * (INTEGRATION.md) binds exactly these symbols behind a cargo feature; nothing here uses torch or C++ types.
 *
 * Conventions (modelled on the reference's only FFI, src/pto_c.rs):
 *  - opaque handle created by porrt_ctx_create / freed by porrt_ctx_destroy     (pto_c.rs:63-103 new_xxx, delete_xxx)
 *  - arrays are (pointer, length) pairs BORROWED from the caller, never freed    (pto_c.rs:33-41)
 *  - validity results are signed: >= 0 validity id, < 0 invalid                  (pto_c.rs:17-18, :401-409)
 *  - every call returns an int32 status (PORRT_OK == 0) and never aborts/unwinds; where the reference would
 *    panic per element, the element's result carries the panic code instead.
 *  - one ctx per host thread; calls on a ctx serialise on its CUDA stream.
 *  - states are N = 2 (x, y) doubles, interleaved (AoS) exactly like the reference's [f64; 2].
 *  - `*_dev` entry points take DEVICE pointers, enqueue on the ctx stream and do not synchronise.
 *  - there is NO CPU fallback: every entry point fails with PORRT_ERR_CUDA when no sm_100 device is usable.
 */
#ifndef PORRT_B200_H
#define PORRT_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

/* status codes */
#define PORRT_OK 0
#define PORRT_ERR_INVALID_ARG 1
#define PORRT_ERR_CUDA 2
#define PORRT_ERR_NO_MAP 3      /* validity call before porrt_map_upload */
#define PORRT_ERR_CAPACITY 4    /* output buffer too small; *out_total holds the required size */
#define PORRT_ERR_PANIC 5       /* the reference would panic on this input as a whole (see porrt_last_error) */
#define PORRT_ERR_UNSUPPORTED 6
#define PORRT_ERR_NO_VERTICES 7 /* NN call before porrt_vertices_set */
#define PORRT_ERR_COMM 8        /* NCCL not loadable / communicator error (multi-GPU paths only) */

/* per-element validity codes (int32): >= 0 is a validity id into the world-validity table */
#define PORRT_INVALID (-1)            /* Option::None: obstacle                          map_io.rs:491,511 */
#define PORRT_PANIC_OOB (-2)          /* image::get_pixel out of bounds                  map_io.rs:167,226 */
#define PORRT_PANIC_ZONE_UNWRAP (-3)  /* gray pixel without zone id: unwrap() on None    map_io.rs:172,231 */
#define PORRT_PANIC_MULTI_ZONE (-4)   /* "multiple zone traversal not supported"         map_io.rs:233     */

/* domain kinds */
#define PORRT_DOMAIN_DOOR 0   /* map_io.rs `Map`: Z door zones, 2^Z worlds            */
#define PORRT_DOMAIN_SHELF 1  /* map_shelves_io.rs `MapShelfDomain`: Z shelves, Z worlds */

/* belief-graph node types (belief_graph.rs:12-17) */
#define PORRT_NODE_UNKNOWN 0
#define PORRT_NODE_ACTION 1
#define PORRT_NODE_OBSERVATION 2
#define PORRT_MAX_STATE_DIM 16 /* porrt_*_nd entry points */

typedef struct porrt_ctx porrt_ctx;

/* ------------------------------------------------------------------ context */
int32_t porrt_ctx_create(int32_t device, porrt_ctx** out_ctx);
int32_t porrt_ctx_destroy(porrt_ctx* ctx);
/* run all subsequent work of this ctx on an existing CUDA stream (e.g. a torch.cuda.Stream); NULL = the ctx's own
 * stream.  Pass cudaStreamLegacy ((void*)1) to address the legacy default stream explicitly. */
int32_t porrt_ctx_set_stream(porrt_ctx* ctx, void* cuda_stream);
int32_t porrt_ctx_synchronize(porrt_ctx* ctx);
/* bind the calling host thread to the CPUs of the NUMA node next to the ctx's GPU (pinned buffers touched afterwards land there);
 * *out_node (nullable) = that node, -1 if unknown / nothing changed.  Call it once per process before allocating host buffers. */
int32_t porrt_ctx_bind_host_thread(porrt_ctx* ctx, int32_t* out_node);
const char* porrt_last_error(porrt_ctx* ctx);
/* options (tests / tuning); unknown options are refused */
#define PORRT_OPT_FORCE_LARGE_MAP_PATH 1  /* value != 0: edge batches take the large-map kernel (class bytes in global memory, used
                                             by itself for maps > ~14000^2 px) although the map would fit the shared-memory path */
#define PORRT_OPT_FORCE_GLOBAL_SWEEPS 2   /* value != 0: porrt_sssp_worlds / porrt_belief_vi run the thread-per-(node, column) sweeps over
                                             the table in global memory (used by itself for roadmaps whose column of V doubles does not
                                             fit in shared memory, V > ~29000) although the on-chip column solver would fit */
#define PORRT_OPT_FORCE_THREAD_PER_QUERY_NN 3  /* value != 0: radius / 1-NN / k-NN queries skip the tile kernels and run the
                                             thread-per-query ring search (used by itself for batches < 2048 queries and for
                                             the queries the tiles cannot serve) */
int32_t porrt_ctx_set_option(porrt_ctx* ctx, int32_t option, int64_t value);
/* number of kernels this ctx has launched so far (bench.py's gpu_launches) */
int64_t porrt_ctx_launch_count(porrt_ctx* ctx);
const char* porrt_version(void);
/* device time (ms, CUDA events) of the phases of the last host-buffer NN call on this ctx; see the call's docs */
int32_t porrt_ctx_last_phase_ms(porrt_ctx* ctx, double* out_ms, int32_t cap, int32_t* out_n);

/* measurement aid (bench.py's L2 roofline denominator, SURVEY.md 8(d)): GB/s of random independent 32-byte sector reads over a
 * buffer of buffer_bytes (<= 0: 64 MiB) that stays in the 126 MB L2 */
int32_t porrt_measure_l2_gather(porrt_ctx* ctx, int64_t buffer_bytes, double* out_gbs);

/* ------------------------------------------------------------------ maps
 * Replaces Map::open + add_zones / init_without_zones (map_io.rs:82-145) and MapShelfDomain::open + add_zones
 * (map_shelves_io.rs:80-148) for already-decoded 8-bit gray images (row-major, row 0 = top).
 * zone == NULL: DOOR -> init_without_zones (1 world); SHELF -> no zones.  ppm = W / (up[0]-low[0]).
 * Computes n_zones, n_worlds, zone centroids (integer mean, map_io.rs:147-163), the world-validity table
 * (map_io.rs:120-126,198-214 / map_shelves_io.rs:113) and uploads a fused occupancy+zone grid to HBM. */
int32_t porrt_map_upload(porrt_ctx* ctx, const uint8_t* occ, const uint8_t* zone, int32_t H, int32_t W,
                         const double low[2], const double up[2], int32_t domain_kind, double visibility_distance);
int32_t porrt_map_info(porrt_ctx* ctx, int32_t* n_zones, int32_t* n_worlds, int32_t* n_validities, int32_t* mask_words);
int32_t porrt_map_zone_positions(porrt_ctx* ctx, double* out_xy /* [2*n_zones] */);
/* world_validities(): out[n_validities * mask_words], bit w of word w/64 = world w (bitvec Lsb0)  map_io.rs:548-550 */
int32_t porrt_map_world_validities(porrt_ctx* ctx, uint64_t* out_masks);

/* PTOFuncs::state_validity, batched (map_io.rs:487-493, map_shelves_io.rs:464-469) */
int32_t porrt_state_validity(porrt_ctx* ctx, const double* xy, int64_t n, int32_t* out_validity_id);
/* PTOFuncs::transition_validator, batched (map_io.rs:495-513, map_shelves_io.rs:471-488): edge i runs
 * from from_xy[2i..] to to_xy[2i..] IN THAT DIRECTION (Bresenham is direction dependent).
 * out_world_mask (nullable): [n * mask_words] per-world validity bitvec = world_validities[id], 0 if invalid. */
int32_t porrt_edge_validity(porrt_ctx* ctx, const double* from_xy, const double* to_xy, int64_t n,
                            int32_t* out_validity_id, uint64_t* out_world_mask);
/* geometric part of PTOFuncs::observe (map_io.rs:281-300, map_shelves_io.rs:242-265): bit z of out_zone_mask[i]
 * = norm2(state_i, zone_pos[z]) < visibility && line of sight.  out_status[i] = 0 or the panic code (< -1). */
int32_t porrt_visibility(porrt_ctx* ctx, const double* xy, int64_t n, uint64_t* out_zone_mask, int32_t* out_status);
/* transition_validator(&PTONode from, &PTONode to) as the planners call it (pto.rs:105, prm.rs:93): both ends are nodes of the
 * vertex set uploaded with porrt_vertices_set (ids in upload order).  Same results as porrt_edge_validity on the nodes' states;
 * 8 instead of 32 bytes per edge cross the bus.  out_world_mask nullable. */
int32_t porrt_edge_validity_indexed(porrt_ctx* ctx, const int32_t* from_idx, const int32_t* to_idx, int64_t n,
                                    int32_t* out_validity_id, uint64_t* out_world_mask);

/* Compact results: the validity id as ONE signed byte per edge (ids are < 128 -- n_validities <= 17 for the door domain, 1 for
 * shelves -- and the negative codes are the same as in the int32 form); the per-world bitvec of an edge is
 * world_validities[id] (porrt_map_world_validities), exactly what the reference's callers look up (pto.rs:111-118).
 * Per edge 32 B in / 1 B out (coordinates), 8 B in / 1 B out (node ids), 4 B in / 1 B out (adjacency rows). */
int32_t porrt_edge_validity_i8(porrt_ctx* ctx, const double* from_xy, const double* to_xy, int64_t n, int8_t* out_validity_id);
int32_t porrt_edge_validity_indexed_i8(porrt_ctx* ctx, const int32_t* from_idx, const int32_t* to_idx, int64_t n,
                                       int8_t* out_validity_id);
/* The candidate edges of a roadmap as the planners hold them: an adjacency over the resident vertex set.  Row r of the CSR
 * (row_ptr[n_rows + 1], col[row_ptr[n_rows]]) lists the nodes transition_validator is asked about for node r:
 * row_is_to != 0: edge e of row r runs col[e] -> r  (prm.rs:91-96 / pto.rs:103-108: neighbour -> new node);
 * row_is_to == 0: r -> col[e].  out_validity_id[e] in the order of col. */
int32_t porrt_edge_validity_csr_i8(porrt_ctx* ctx, const int64_t* row_ptr, const int32_t* col, int64_t n_rows, int32_t row_is_to,
                                   int8_t* out_validity_id);

int32_t porrt_state_validity_dev(porrt_ctx* ctx, const double* xy_dev, int64_t n, int32_t* out_validity_id_dev);
int32_t porrt_edge_validity_dev(porrt_ctx* ctx, const double* from_xy_dev, const double* to_xy_dev, int64_t n,
                                int32_t* out_validity_id_dev, uint64_t* out_world_mask_dev);
int32_t porrt_visibility_dev(porrt_ctx* ctx, const double* xy_dev, int64_t n, uint64_t* out_zone_mask_dev,
                             int32_t* out_status_dev);

/* ------------------------------------------------------------------ nearest neighbours (nearest_neighbor.rs)
 * The vertex set replaces the KdTree's contents: vertex i has id i (KdTree::add(state, id) with ids 0..n-1).
 * cell_size <= 0 picks one from the vertex density. */
int32_t porrt_vertices_set(porrt_ctx* ctx, const double* xy, int64_t n, double cell_size);
int32_t porrt_vertices_set_dev(porrt_ctx* ctx, const double* xy_dev, int64_t n, double cell_size,
                               const double bbox_lo[2], const double bbox_hi[2]);
/* KdTree::add (nearest_neighbor.rs:29-46), batched: the m new vertices get the ids n .. n+m-1.  Only the new coordinates cross
 * the bus; the cell grid is rebuilt on the device (from the resident set, with the cell-size rule of the last porrt_vertices_set)
 * before the next query.  This is what the sequential planners (RRT, PTO growth) call once per accepted sample. */
int32_t porrt_vertices_append(porrt_ctx* ctx, const double* xy, int64_t m);
int32_t porrt_vertices_count(porrt_ctx* ctx, int64_t* out_n);

/* KdTree::nearest_neighbors[_filtered] (nearest_neighbor.rs:94-126), batched: all ids j with
 *   norm2(vertex_j, q_i) <= radius[i]   (inclusive, on the sqrt-ed f64 value)
 *   and j < prefix_limit[i]             (if prefix_limit != NULL: the tree as it was before vertex prefix_limit[i] was added)
 *   and bit world[i] of vertex j's reachability mask reach_mask[j * reach_words ..]   (if reach_mask != NULL: the validator
 *       closure of pto.rs:74-77; BitVec Lsb0 layout, reach_words = ceil(n_worlds / 64); a world >= 64 * reach_words passes nothing)
 * Result: CSR -- out_offsets[m+1], out_ids ascending per query (the SET contract; the caller restores the reference's kd pre-order by
 * sorting each list by porrt_kd_preorder_rank, as porrt_prm_build does internally).  If the hits exceed cap: PORRT_ERR_CAPACITY, *out_total = needed. */
int32_t porrt_radius_query(porrt_ctx* ctx, const double* q_xy, const double* radius, int64_t m,
                           const uint32_t* prefix_limit, const uint64_t* reach_mask, int32_t reach_words, const uint32_t* world,
                           int64_t* out_offsets, int32_t* out_ids, int64_t cap, int64_t* out_total);
/* KdTree::nearest_neighbor[_filtered] (nearest_neighbor.rs:48-92), batched: argmin over (d2, id); out_id = -1 when
 * nothing passes the filter (the reference then returns the root).  out_dist = norm2 of the winner.
 * out_ties (nullable): number of vertices at exactly the winning squared distance (>1 = tie the kd order decides). */
int32_t porrt_nearest(porrt_ctx* ctx, const double* q_xy, int64_t m, const uint64_t* reach_mask, int32_t reach_words,
                      const uint32_t* world, int32_t* out_id, double* out_dist, int32_t* out_ties);
/* k nearest (no reference counterpart; BASELINE metric "kNN queries/sec"): ids/dists ascending by (d2, id), -1/inf padded */
int32_t porrt_knn(porrt_ctx* ctx, const double* q_xy, int64_t m, int32_t k, int32_t* out_ids, double* out_dist);

/* The kd-tree's pre-order rank of every vertex (the order KdTree::nearest_neighbors returns hits in):
 * rank[i] = position of vertex i in a node-left-right walk of the tree obtained by inserting 0,1,..,n-1 in order.
 * xy == NULL ranks the ctx's own vertex set (porrt_vertices_set / porrt_vertices_append) in place, nothing is uploaded. */
int32_t porrt_kd_preorder_rank(porrt_ctx* ctx, const double* xy, int64_t n, int32_t* out_rank);

/* ------------------------------------------------------------------ PRM (prm.rs)
 * PRM::grow_graph for a given sample stream: node k = samples[k]; node 0 is the start (PRM::init or first sample).
 * Reproduces add_sample (prm.rs:52-109): radius = heuristic_radius(k+1, ...) (computed on the host with libm),
 * neighbours = vertices j < k within radius in kd pre-order, edges validated from neighbour -> new node.
 * Output: children adjacency as CSR in the reference's insertion order (row k = valid earlier neighbours in kd
 * pre-order, then later nodes ascending).  parents(k) == children(k) as sequences (prm.rs:99-106).
 * out_col may be NULL / cap too small: the call then returns PORRT_ERR_CAPACITY with *out_n_edges set and KEEPS the result
 * on the device; porrt_prm_fetch copies it out without recomputing (valid until the next call on this ctx). */
int32_t porrt_prm_build(porrt_ctx* ctx, const double* samples_xy, int64_t n, double max_step, double search_radius,
                        int64_t* out_row_ptr /* [n+1] */, int32_t* out_col, int64_t cap, int64_t* out_n_edges,
                        double* out_phase_ms /* nullable [8] */);

int32_t porrt_prm_fetch(porrt_ctx* ctx, int64_t* out_row_ptr /* nullable */, int32_t* out_col, int64_t cap);

/* ------------------------------------------------------------------ value backups
 * CSR graph = children adjacency of a PTOGraph (pto_graph.rs:171-228): row_ptr[V+1], col[E], edge_vid[E], xy[2V],
 * node_vid[V]; validities[n_validities * mask_words] as returned by porrt_map_world_validities. */

/* QMdpPolicyExtractor::plan_qmdp (qmdp_policy_extractor.rs:23-35): for each world w a multi-source `dijkstra`
 * (pto_graph.rs:275-303) over PTOGraphWorldView{world w} (:245-271) towards finals_ids[finals_ptr[w]..finals_ptr[w+1]].
 * n_worlds == 0 with world_filter == 0 runs the plain-graph dijkstra once (finals_ptr[0..1]).
 * out_dist[w * V + v], bit-identical to the reference's f64 results. out_sweeps (nullable) = relaxation sweeps used. */
int32_t porrt_sssp_worlds(porrt_ctx* ctx, int64_t V, const int64_t* row_ptr, const int32_t* col, const double* xy,
                          const int32_t* node_vid, const uint64_t* validities, int32_t n_validities, int32_t mask_words,
                          int32_t n_worlds, const int64_t* finals_ptr, const int32_t* finals_ids,
                          double* out_dist, int32_t* out_sweeps);
/* plan_qmdp straight on the roadmap porrt_prm_build left on the device (CSR + vertex coordinates) under the uploaded map's worlds:
 * only the final-node lists cross the bus on the way in.  Node validity ids = the map's state validity of the vertices, evaluated
 * on the device (a vertex inside an obstacle is invalid in every world).  finals_ptr[n_worlds + 1]; out_dist[n_worlds * V] may be
 * NULL (the table then stays on the device: timing, device-resident pipelines).
 * Both calls: porrt_ctx_last_phase_ms = [device ms of the backups, edge records / (parent, world) pairs worked through]. */
int32_t porrt_sssp_worlds_prm(porrt_ctx* ctx, const int64_t* finals_ptr, const int32_t* finals_ids, double* out_dist,
                              int32_t* out_sweeps);

/* PTO::build_belief_graph + compute_expected_costs_to_goals (pto.rs:185-275, belief_graph.rs:89-182) on the IMPLICIT
 * belief graph (belief node id = node * B + belief):
 *   beliefs[B * n_worlds]                reachable_belief_states, belief 0 = start belief (pto.rs:187)
 *   visible_zone_mask[V]                 from porrt_visibility
 *   finals: node ids + their finality masks [n_finals * mask_words]   (pto_reachability.rs:77-79)
 * out_dist[V * B] = expected_costs_to_goals (inf where unreachable / non-existent), out_type[V * B] node types. */
/* porrt_ctx_last_phase_ms after the call: [0] device ms of the value backups (all levels of the on-chip column solver, CUDA
 * events), [1] edge records the solver worked through (12 bytes each, read from L2) -- the bytes actually moved. */
int32_t porrt_belief_vi(porrt_ctx* ctx, int64_t V, const int64_t* row_ptr, const int32_t* col, const int32_t* edge_vid,
                        const double* xy, const int32_t* node_vid, const uint64_t* validities, int32_t n_validities,
                        int32_t mask_words, int32_t n_worlds, const double* beliefs, int32_t B,
                        const uint64_t* visible_zone_mask, const int32_t* finals_ids, const uint64_t* finals_masks,
                        int32_t n_finals, double* out_dist, uint8_t* out_type, int32_t* out_sweeps,
                        double* out_phase_ms /* nullable [4] */);
/* The table of the last porrt_belief_vi without a second copy: *out_dist ([V*B], node-major) and *out_type point into pinned
 * host memory owned by the ctx, valid until the next porrt_belief_vi on it (the convention of the reference's own FFI: results stay
 * owned by the handle and are read through pointer getters, pto_c.rs:255-270).  porrt_belief_vi accepts out_dist = out_type = NULL
 * for callers that read the result this way (at B = 4095 the copy into a fresh 172 MB caller buffer costs as much as the backups). */
int32_t porrt_belief_result(porrt_ctx* ctx, const double** out_dist, const uint8_t** out_type, int64_t* out_V, int32_t* out_B);

/* belief_graph.rs:184-267 extract_policy on the implicit graph, walking out_dist/out_type of porrt_belief_vi.
 * Policy nodes in creation order: out_node[k] = graph node, out_belief[k], out_parent[k] (-1 root), out_is_leaf[k].
 * Returns PORRT_ERR_PANIC where the reference's asserts would fire; PORRT_ERR_CAPACITY when cap is too small. */
int32_t porrt_extract_policy(porrt_ctx* ctx, int32_t* out_node, int32_t* out_belief, int32_t* out_parent,
                             uint8_t* out_is_leaf, int64_t cap, int64_t* out_n, double* out_expected_cost);

/* conditional_dijkstra (belief_graph.rs:89-182) on an EXPLICIT BeliefGraph (belief_graph.rs:12-73): the reference's free function
 * as called by its own tests (:276-567) and by the multi-modal PRM (map_shelves_tamp_prm.rs:476).  Belief node k has state
 * xy[2k..], node_type[k] (PORRT_NODE_*), belief_id[k] into beliefs[B * n_worlds]; children adjacency as CSR in add_edge order
 * (parents are implied: add_edge keeps both lists).  cost_evaluator = norm2.  out_dist[V] bit-identical to the reference;
 * PORRT_ERR_PANIC where it would panic (:130 p <= 0 at an evaluated Observation node, :140 Unknown parent of a reached node). */
int32_t porrt_conditional_dijkstra(porrt_ctx* ctx, int64_t V, const int64_t* row_ptr, const int32_t* col, const double* xy,
                                   const uint8_t* node_type, const int32_t* belief_id, const double* beliefs, int32_t B,
                                   int32_t n_worlds, const int32_t* finals, int32_t n_finals, double* out_dist,
                                   int32_t* out_sweeps /* nullable */);
/* The same for states of `dim` doubles (1 <= dim <= PORRT_MAX_STATE_DIM; xy[dim * k ..]): the reference's planner is generic over
 * the state dimension (pto_c.rs:226-241 instantiates N = 2, 3, 7, 9); norm2 sums dx * dx in dimension order (common.rs:203-213). */
int32_t porrt_conditional_dijkstra_nd(porrt_ctx* ctx, int32_t dim, int64_t V, const int64_t* row_ptr, const int32_t* col,
                                      const double* xy, const uint8_t* node_type, const int32_t* belief_id, const double* beliefs,
                                      int32_t B, int32_t n_worlds, const int32_t* finals, int32_t n_finals, double* out_dist,
                                      int32_t* out_sweeps /* nullable */);
int32_t porrt_extract_policy_graph_nd(porrt_ctx* ctx, int32_t dim, int64_t V, const int64_t* row_ptr, const int32_t* col,
                                      const double* xy, const uint8_t* node_type, const int32_t* belief_id, const double* beliefs,
                                      int32_t B, int32_t n_worlds, const double* dist, int32_t* out_belief_node, int32_t* out_parent,
                                      uint8_t* out_is_leaf, int64_t cap, int64_t* out_n, double* out_expected_cost);
/* extract_policy (belief_graph.rs:184-267) on the same explicit graph and the dist of porrt_conditional_dijkstra: host walk from
 * belief node 0.  Policy nodes in creation order: out_belief_node[k], out_parent[k] (-1 = root), out_is_leaf[k].
 * PORRT_ERR_PANIC where the reference's asserts (:250, :261) fire; PORRT_ERR_CAPACITY (with *out_n) when cap is too small. */
int32_t porrt_extract_policy_graph(porrt_ctx* ctx, int64_t V, const int64_t* row_ptr, const int32_t* col, const double* xy,
                                   const uint8_t* node_type, const int32_t* belief_id, const double* beliefs, int32_t B,
                                   int32_t n_worlds, const double* dist, int32_t* out_belief_node, int32_t* out_parent,
                                   uint8_t* out_is_leaf, int64_t cap, int64_t* out_n, double* out_expected_cost);

/* ------------------------------------------------------------------ multi-modal PRM (map_shelves_tamp_prm.rs)
 * MapShelfDomainTampPRM::plan (:308-326) for a given SCHEDULE.  The growth (grow_mm_prm, :328-397) never looks at validity
 * results -- modes, observed zones and samples are decided by the RNG streams -- so the caller, who owns the samplers and the
 * mode tree, passes what they decided and this call does the computing:
 *   mode m owns the add_sample calls mode_node_ptr[m] .. mode_node_ptr[m+1]-1 of samples_xy / max_step / search_radius (in call
 *   order: PRM node k of the mode is its k-th call; goal seeds are calls with (0.0, 0.0)), belief mode_belief_id[m] of
 *   beliefs[B * n_worlds] (the mode's own belief vector, :419) and final nodes mode_final_nodes[mode_final_ptr[m] ..];
 *   transition t goes from mode tr_from_mode[t] to tr_to_mode[t] with the (observation node, destination node) pairs
 *   tr_pairs[2 * tr_pair_ptr[t] ..] (PRM node ids inside the two modes, :386-390).
 * Builds every mode's PRM (prm.rs add_sample semantics), the belief graph of build_belief_graph (:399-473; belief node id =
 * mode_node_ptr[mode] + PRM node id) and runs conditional_dijkstra: out_dist[total nodes], bit-identical to the reference's
 * expected_costs_to_goals.  out_phase_ms (nullable [4]): PRM builds, graph assembly, value backups. */
int32_t porrt_mmprm_plan(porrt_ctx* ctx, int32_t n_modes, const int64_t* mode_node_ptr, const double* samples_xy,
                         const double* max_step, const double* search_radius, const int32_t* mode_belief_id,
                         const double* beliefs, int32_t B, int32_t n_worlds, int32_t n_transitions,
                         const int32_t* tr_from_mode, const int32_t* tr_to_mode, const int64_t* tr_pair_ptr,
                         const int32_t* tr_pairs, const int64_t* mode_final_ptr, const int32_t* mode_final_nodes,
                         double* out_dist, int64_t* out_n_edges, int32_t* out_sweeps, double* out_phase_ms);
/* the belief graph assembled by the last porrt_mmprm_plan (children CSR, node types, belief ids), e.g. for
 * porrt_extract_policy_graph; all outputs nullable except that cap must hold *out_n_edges columns */
int32_t porrt_mmprm_fetch_graph(porrt_ctx* ctx, int64_t* out_row_ptr, int32_t* out_col, int64_t cap, uint8_t* out_node_type,
                                int32_t* out_belief_id);

/* ------------------------------------------------------------------ policy refinement (pto_policy_refiner.rs)
 * PTOPolicyRefiner::is_transition_valid (pto_policy_refiner.rs:395-423), batched: out_valid[i] = 1 iff both end states are
 * valid, the transition from -> to is valid with validity id v, and compat_row[v] != 0, where compat_row[n_validities] is
 * compatibilities[belief_state_id] (compute_compatibility, common.rs:266-276).  Where the reference would panic on element i,
 * out_valid[i] = 0 and out_status[i] (nullable) carries the panic code; otherwise out_status[i] = 0. */
int32_t porrt_transition_valid(porrt_ctx* ctx, const double* from_xy, const double* to_xy, int64_t n,
                               const uint8_t* compat_row, uint8_t* out_valid, int32_t* out_status);
/* PTOPolicyRefiner::partial_shortcut (pto_policy_refiner.rs:158-206) on one path piece: states_xy[2 * n_states] is updated in
 * place.  The trial sequence is the one a DiscreteSampler seeded with sampler_seed draws (the reference uses
 * DiscreteSampler::new(), seed 0).  The whole trial loop runs on the device (one CTA per piece, the path in shared memory, the
 * transitions of a trial checked by its warps, commit decided in the reference's `&&` order), so states and *out_commits equal the
 * sequential result and there is ONE device round trip per call (*out_waves, nullable).  At most 1024 states per piece.
 * PORRT_ERR_PANIC if a transition check hits a reference panic (the states are then left untouched). */
int32_t porrt_partial_shortcut(porrt_ctx* ctx, double* states_xy, int32_t n_states, const uint8_t* compat_row,
                               int32_t n_iterations, uint64_t sampler_seed, int32_t* out_commits, int32_t* out_waves);
/* The same for all path pieces of a policy at once (refine_solution's loop, pto_policy_refiner.rs:102-115): piece p owns the
 * states piece_ptr[p] .. piece_ptr[p+1]-1 of states_xy and the compatibility row compat_rows[p * n_validities ..] of its belief
 * state; every piece draws from its own fresh sampler (same seed), exactly like the reference.  The pieces run side by side on
 * different SMs.  out_commits[n_pieces] (nullable). */
int32_t porrt_partial_shortcut_batch(porrt_ctx* ctx, double* states_xy, const int32_t* piece_ptr, int32_t n_pieces,
                                     const uint8_t* compat_rows, int32_t n_iterations, uint64_t sampler_seed,
                                     int32_t* out_commits, int32_t* out_waves);

/* PTOPolicyRefiner::refine_solution(RefinmentStrategy::PartialShortCut(n_iterations)) (pto_policy_refiner.rs:85-133), the last step
 * of every PTO run in the reference's main.rs (:442 PartialShortCut(1500)), on a policy of the last porrt_belief_vi of this ctx
 * given as porrt_extract_policy returned it (pol_node / pol_belief / pol_parent in creation order): Policy::decompose
 * (common.rs:85-129), build_path_piece + partial_shortcut per piece (all pieces in one device batch), recompose (:324-393) and
 * compute_expected_costs_to_goals (common.rs:131-153).  Output = the refined policy, nodes in recompose's creation order:
 * out_xy[2k..] refined state, out_node / out_belief (original_node_id = node * B + belief), out_parent (-1 = root or a piece
 * recompose leaves unconnected, see the source), out_is_leaf.  cap < *out_n: PORRT_ERR_CAPACITY.  out_commits: accepted shortcuts. */
int32_t porrt_refine_policy_shortcut(porrt_ctx* ctx, const int32_t* pol_node, const int32_t* pol_belief, const int32_t* pol_parent,
                                     int64_t n_pol, int32_t n_iterations, uint64_t sampler_seed, double* out_xy, int32_t* out_node,
                                     int32_t* out_belief, int32_t* out_parent, uint8_t* out_is_leaf, int64_t cap, int64_t* out_n,
                                     double* out_expected_cost, int64_t* out_commits);

/* PTOPolicyRefiner::refine_solution(RefinmentStrategy::Reparent(radius)) (pto_policy_refiner.rs:85-133; main.rs:221,270 run
 * Reparent(0.3)) on the same kind of policy: Policy::decompose, per piece build_tree (:208-280: the piece plus every belief-graph
 * descendant within `radius` of one of its nodes) and reparent with radius / 2 (:282-322), recompose.  The trees' states never change,
 * so every (tree node, neighbour) transition the label-correcting loop can test goes through is_transition_valid in ONE device batch
 * (*out_transitions of them); the loop itself runs on the host over those answers, popping in the order of the reference's priority
 * queue (priority-queue 1.0.5, restated: the order among equal priorities is not pinned by any reference test).  Outputs as for
 * porrt_refine_policy_shortcut (the recomposed policy may have fewer or more nodes than the input: size query by PORRT_ERR_CAPACITY
 * and *out_n); *out_tree_nodes = nodes of all trees. */
int32_t porrt_refine_policy_reparent(porrt_ctx* ctx, const int32_t* pol_node, const int32_t* pol_belief, const int32_t* pol_parent,
                                     int64_t n_pol, double radius, double* out_xy, int32_t* out_node, int32_t* out_belief,
                                     int32_t* out_parent, uint8_t* out_is_leaf, int64_t cap, int64_t* out_n, double* out_expected_cost,
                                     int64_t* out_tree_nodes /* nullable */, int64_t* out_transitions /* nullable */);

/* Policy::decompose (common.rs:85-129) and Policy::compute_expected_costs_to_goals (common.rs:131-153), the two pieces of common.rs the
 * refiners are built around, as host-side rows (no device, no ctx).  A policy = parent[k] per node in creation order (parent[0] = -1,
 * parent[k] < k; children in add_edge order = increasing index).  decompose: pieces back to back (out_piece_ptr[n_pieces + 1],
 * out_piece_nodes[n]) and the skeleton as a CSR (nullable); PORRT_ERR_CAPACITY + *out_n_pieces when cap_pieces is too small.
 * expected_cost: xy[2k..] states, belief_id[k] into beliefs[B * n_worlds], cost = norm2; the reference's summation order. */
int32_t porrt_policy_decompose(const int32_t* parent, int64_t n, int32_t* out_piece_ptr, int32_t* out_piece_nodes, int32_t* out_succ_ptr,
                               int32_t* out_succ, int32_t cap_pieces, int32_t* out_n_pieces);
int32_t porrt_policy_expected_cost(const double* xy, const int32_t* belief_id, const int32_t* parent, int64_t n, const double* beliefs,
                                   int32_t B, int32_t n_worlds, double* out_expected_cost);

/* reachable_belief_states (map_io.rs:515-546 / map_shelves_io.rs:490-520): host-side closure over the uploaded map's
 * zones; out[cap * n_worlds]; *out_B = count (PORRT_ERR_CAPACITY if > cap). */
int32_t porrt_reachable_belief_states(porrt_ctx* ctx, const double* start_belief, double* out, int32_t cap, int32_t* out_B);

/* ------------------------------------------------------------------ QMDP policy (qmdp_policy_extractor.rs)
 * QMdpPolicyExtractor::react_qmdp (:38-49) with get_common_path (:65-87), get_best_expected_child (:90-108), get_path (:51-62) and
 * get_best_child (:110-123), walking the cost table of porrt_sssp_worlds (cost_to_goals[w * V + v], plan_qmdp's result) over the
 * children CSR.  start_node = kdtree.nearest_neighbor(start).id (porrt_nearest).  Host walk; ctx may be NULL.
 * out_path_ptr[n_worlds + 1], out_path_nodes: paths[w] as node ids = the common path (its length in *out_n_common) followed by
 * world w's own path.  PORRT_ERR_PANIC: belief_len != n_worlds (the reference's Err(..).unwrap(), :42), or a walk that would
 * never end in the reference (no finite child); PORRT_ERR_CAPACITY with *out_total when cap is too small. */
int32_t porrt_qmdp_react(porrt_ctx* ctx, int64_t V, const int64_t* row_ptr, const int32_t* col, const double* xy, int32_t n_worlds,
                         const double* cost_to_goals, int64_t start_node, const double* belief, int32_t belief_len,
                         double common_horizon, int64_t* out_path_ptr, int32_t* out_path_nodes, int64_t cap, int64_t* out_total,
                         int64_t* out_n_common);

/* ------------------------------------------------------------------ host-side rows (sequential by nature; no device work)
 * What the reference's sequential callers (PTO::grow_graph pto.rs:55-149, RRT::grow_tree rrt.rs:102-181) need around the batched
 * calls above, bit-faithful to the crate, so that the whole path sits behind one ABI. */
/* heuristic_radius (common.rs:357-369): min(search_radius * (ln n / n)^(1/dim), max_step), libm on the host */
int32_t porrt_heuristic_radius(int64_t n_nodes, double max_step, double search_radius, int32_t dim, double* out_radius);
/* steer (common.rs:215-225), batched: to_xy[k] is pulled towards from_xy[k] when norm1(from, to) > max_step (in place) */
int32_t porrt_steer(const double* from_xy, double* to_xy, int64_t n, double max_step);
/* the same for states of `dim` doubles (1 <= dim <= PORRT_MAX_STATE_DIM; the reference instantiates steer<N> for N = 2, 3, 7, 9) */
int32_t porrt_steer_nd(const double* from, double* to, int64_t n, int32_t dim, double max_step);

/* ContinuousSampler / DiscreteSampler (sample_space.rs:6-60): one Pcg64::seed_from_u64(seed) stream per handle (the reference
 * seeds with 0; PTO keeps one continuous and one discrete sampler, two independent streams with the same seed, pto.rs:141-149) */
typedef struct porrt_sampler porrt_sampler;
int32_t porrt_sampler_create(uint64_t seed, porrt_sampler** out_sampler);
int32_t porrt_sampler_destroy(porrt_sampler* s);
/* n x ContinuousSampler::sample(): out[n * dim], one gen_range(low[d]..up[d]) per dimension in dimension order */
int32_t porrt_sampler_continuous(porrt_sampler* s, const double* low, const double* up, int32_t dim, int64_t n, double* out);
/* n x DiscreteSampler::sample(n_choices) */
int32_t porrt_sampler_discrete(porrt_sampler* s, uint64_t n_choices, int64_t n, uint64_t* out);

/* SquareGoal (common.rs:304-350).  goal(): out_goal[k] = index of the first goal with norm1(state_k, goal) < max_dist, -1 = None
 * (the caller owns the goals' world masks).  goal_example(): out_xy[2 * w] = the goal valid in world w ((0, 0) if none);
 * goal_masks[n_goals * ceil(n_worlds / 64)]; PORRT_ERR_PANIC when masks overlap (assert, :320). */
int32_t porrt_square_goal(const double* goals_xy, int32_t n_goals, double max_dist, const double* xy, int64_t n, int32_t* out_goal);
int32_t porrt_square_goal_examples(const double* goals_xy, const uint64_t* goal_masks, int32_t n_goals, int32_t n_worlds, double* out_xy);

/* Reachability (pto_reachability.rs:6-102): per-node world masks propagated at edge insertion; masks are ceil(n_worlds / 64) u64
 * words (BitVec Lsb0).  porrt_reach_create = new() + set_root(root_validity): node 0. */
typedef struct porrt_reach porrt_reach;
int32_t porrt_reach_create(int32_t n_worlds, const uint64_t* root_validity, porrt_reach** out_reach);
int32_t porrt_reach_destroy(porrt_reach* r);
int32_t porrt_reach_add_node(porrt_reach* r, const uint64_t* validity);                              /* :35-38 */
int32_t porrt_reach_add_final_node(porrt_reach* r, int64_t id, const uint64_t* finality);            /* :40-45 */
int32_t porrt_reach_add_edge(porrt_reach* r, int64_t from, int64_t to, const uint64_t* edge_validity); /* :47-57 */
int32_t porrt_reach_count(porrt_reach* r, int64_t* out_nodes, int32_t* out_words);
/* reachability(id) (:59-61) of nodes first .. first + n - 1: out[n * words], the reach_mask of porrt_nearest / porrt_radius_query */
int32_t porrt_reach_masks(porrt_reach* r, int64_t first, int64_t n, uint64_t* out);
int32_t porrt_reach_final_nodes_for_world(porrt_reach* r, int32_t world, int64_t* out_ids, int64_t cap, int64_t* out_n); /* :63-68 */
int32_t porrt_reach_finals(porrt_reach* r, int64_t* out_ids, uint64_t* out_masks, int64_t cap, int64_t* out_n);          /* :82-84 */
int32_t porrt_reach_is_final_set_complete(porrt_reach* r, int32_t* out_complete);                                       /* :86-95 */

/* ------------------------------------------------------------------ PTO roadmap growth on the device (pto_grow.cu, DESIGN.md 3.8)
 * PTO::grow_graph (pto.rs:55-139) on the uploaded map (Map or MapShelfDomain, N = 2), as ONE call.  The two sampler streams are
 * Pcg64::seed_from_u64(sampler_seed), like PTO::new (seed 0 in the reference); continuous samples in [low, up).  Goals are a
 * SquareGoal (common.rs:304-350): goals_xy[2 * n_goals], goal_masks[n_goals * mask_words], max_dist.  Loop condition as the
 * reference: i < n_iter_min || (!is_final_set_complete && i < n_iter_max).
 * The roadmap stays on the device; porrt_pto_fetch copies it out.  out_sizes[4] = iterations, nodes, directed edges, final nodes.
 * *out_complete = is_final_set_complete() at the end (the reference's plan() fails when 0, pto_c.rs:214).
 * PORRT_ERR_PANIC where the reference panics, with *out_panic_code (nullable) = PORRT_INVALID for expect("Start from a valid
 * state!") or the PORRT_PANIC_* code of the first state / edge check that panics, and out_sizes[0] = that iteration.
 * out_counters (nullable [4]): windows, iterations re-speculated, conflicts by nearest neighbour, conflicts by radius / kd slot. */
int32_t porrt_pto_grow(porrt_ctx* ctx, const double start[2], const double low[2], const double up[2], uint64_t sampler_seed,
                       const double* goals_xy, const uint64_t* goal_masks, int32_t n_goals, double goal_max_dist,
                       double max_step, double search_radius, int64_t n_iter_min, int64_t n_iter_max,
                       int64_t* out_sizes, int32_t* out_complete, int32_t* out_panic_code, int64_t* out_counters);
/* the roadmap of the last porrt_pto_grow on this ctx, every pointer nullable: xy[2V], node_vid[V], children CSR in the reference's
 * insertion order (row_ptr[V+1], col[E], edge_vid[E]; parents(k) == children(k) as sequences, pto.rs:111-120), reach[V * mask_words]
 * (Reachability::reachability), final ids + finality masks in add_final_node order (pto.rs:122-124).
 * After a porrt_pto_grow_batch this is roadmap 0 of that batch (porrt_pto_fetch_roadmap(ctx, 0, ...)). */
int32_t porrt_pto_fetch(porrt_ctx* ctx, double* out_xy, int32_t* out_node_vid, int64_t* out_row_ptr, int32_t* out_col,
                        int32_t* out_edge_vid, uint64_t* out_reach, int64_t* out_final_ids, uint64_t* out_final_masks);
/* porrt_pto_grow for n_roadmaps independent roadmaps in ONE call: roadmap r samples with Pcg64::seed_from_u64(sampler_seeds[r]);
 * map, start, bounds, goals and parameters are shared.  Each roadmap equals porrt_pto_grow with its seed, counters included.
 * out_sizes[4 * n] and out_counters (nullable, [4 * n]) hold porrt_pto_grow's four values per roadmap.  out_status[r] = 0 when
 * roadmap r's final set is complete, 1 when it is not, PORRT_ERR_PANIC when its growth panics: then out_panic_code[r] (nullable
 * [n]) and out_sizes[4 r] are the code and the iteration porrt_pto_grow reports.  A panic stops only its own roadmap; the call
 * still returns PORRT_OK.  The whole call fails like porrt_pto_grow on bad arguments, no map, overlapping goal masks and
 * low >= up.  n_roadmaps must lie in 1 .. PORRT_PTO_MAX_ROADMAPS (a launch grid's y dimension) and the device's free memory must
 * hold them at their starting size (about 28 MB each at 4096 + iterations, DESIGN.md 3.8), else PORRT_ERR_INVALID_ARG; running
 * out of memory while the roadmaps grow is PORRT_ERR_CUDA.  The batch replaces the ctx's last growth: porrt_pto_fetch_roadmap
 * reads roadmap r, porrt_pto_fetch reads roadmap 0. */
#define PORRT_PTO_MAX_ROADMAPS 65535
int32_t porrt_pto_grow_batch(porrt_ctx* ctx, int32_t n_roadmaps, const uint64_t* sampler_seeds, const double start[2], const double low[2],
                             const double up[2], const double* goals_xy, const uint64_t* goal_masks, int32_t n_goals, double goal_max_dist,
                             double max_step, double search_radius, int64_t n_iter_min, int64_t n_iter_max, int64_t* out_sizes,
                             int32_t* out_status, int32_t* out_panic_code, int64_t* out_counters);
/* porrt_pto_fetch for roadmap r of the last porrt_pto_grow_batch (a porrt_pto_grow is a batch of one).  PORRT_ERR_INVALID_ARG
 * when nothing has been grown, r is out of range, or roadmap r panicked. */
int32_t porrt_pto_fetch_roadmap(porrt_ctx* ctx, int32_t r, double* out_xy, int32_t* out_node_vid, int64_t* out_row_ptr, int32_t* out_col,
                                int32_t* out_edge_vid, uint64_t* out_reach, int64_t* out_final_ids, uint64_t* out_final_masks);

/* ------------------------------------------------------------------ multi-GPU (SURVEY.md 8(e))
 * The reference is single-threaded and has no distributed code; what shards are its independent units (edge checks,
 * radius / NN queries, the worlds of plan_qmdp).  One process and one ctx per GPU; map and vertex set replicated.
 * A ctx that was given a communicator runs porrt_prm_build and porrt_sssp_worlds SHARDED (same signatures, same
 * results on every rank, bit-identical to the single-GPU result):
 *   porrt_prm_build   : rank r runs the radius queries and edge checks of new nodes shard_range(n, r, world); the valid
 *                       (neighbour, new node) pairs are all-gathered (NCCL over NVLink) and every rank assembles the CSR.
 *   porrt_sssp_worlds : rank r relaxes worlds shard_range(n_worlds, r, world); the dist rows are all-gathered.
 * Edge / state / NN batches have no exchange step: each rank calls the ordinary entry points on its slice; when a later
 * device-resident stage needs all slices, porrt_comm_all_gather_dev assembles them.
 * NCCL is bound at run time (dlopen "libnccl.so.2", override with PORRT_NCCL_LIB); there is no link-time dependency. */
/* rank 0: create the 128-byte ncclUniqueId; the host carries it to the other ranks (any 128-byte broadcast) */
int32_t porrt_comm_unique_id(uint8_t* out_id128);
int32_t porrt_comm_init(porrt_ctx* ctx, const uint8_t* id128, int32_t rank, int32_t world);   /* collective */
int32_t porrt_comm_destroy(porrt_ctx* ctx);
int32_t porrt_comm_info(porrt_ctx* ctx, int32_t* out_rank, int32_t* out_world, int32_t* out_nccl_version);
/* contiguous shard [lo, hi) of n units: sizes differ by at most one, lower ranks take the extra unit */
int32_t porrt_shard_range(int64_t n, int32_t rank, int32_t world, int64_t* out_lo, int64_t* out_hi);
/* rank r owns rows shard_range(n_total, r, world), bytes_per_unit bytes each; recv_dev gets all n_total rows in rank order on
 * every rank.  send_dev == NULL: the rank's rows already sit at their place in recv_dev (in-place).  Enqueued on the ctx stream. */
int32_t porrt_comm_all_gather_dev(porrt_ctx* ctx, const void* send_dev, void* recv_dev, int64_t n_total, int64_t bytes_per_unit);
/* ragged: rank r contributes byte_counts[r] bytes (host array [world], identical on every rank) */
int32_t porrt_comm_all_gatherv_dev(porrt_ctx* ctx, const void* send_dev, void* recv_dev, const int64_t* byte_counts);

/* ------------------------------------------------------------------ on-disk formats (host code, no GPU work)
 * PNM gray maps, the decode step of Map::open_image (map_io.rs:98-105): P2 (ASCII) and P5 (binary), 8 bit; anything else is the
 * reference's panic "Wrong image format!" (PORRT_ERR_PANIC).  Size query: out == NULL / cap too small -> PORRT_ERR_CAPACITY with
 * *out_h, *out_w set.  ctx is used for error text only and may be NULL. */
int32_t porrt_pgm_read(porrt_ctx* ctx, const char* path, uint8_t* out, int64_t cap, int32_t* out_h, int32_t* out_w);
int32_t porrt_pgm_write(porrt_ctx* ctx, const char* path, const uint8_t* img, int32_t h, int32_t w, int32_t binary);
/* PTOGraph JSON (pto_graph.rs:22-118, serde_json of SerializablePTOGraph) <-> the CSR arrays of the value-backup entry points.
 * Stored (insertion) order of `children` / `parents` is kept.  load -> handle; porrt_graph_info gives the sizes, porrt_graph_arrays
 * copies out whichever arrays are asked for (every pointer nullable): xy[2V], node_vid[V], children as row_ptr[V+1] / col / edge_vid,
 * parents as p_row_ptr / p_col / p_edge_vid, validities[n_validities * n_worlds] (1 = holds in that world). */
typedef struct porrt_graph porrt_graph;
int32_t porrt_graph_load_json(porrt_ctx* ctx, const char* path, porrt_graph** out_graph);
int32_t porrt_graph_info(const porrt_graph* g, int64_t* out_n_nodes, int64_t* out_n_children, int64_t* out_n_parents,
                         int32_t* out_n_validities, int32_t* out_n_worlds);
int32_t porrt_graph_arrays(const porrt_graph* g, double* out_xy, int32_t* out_node_vid, int64_t* out_row_ptr, int32_t* out_col,
                           int32_t* out_edge_vid, int64_t* out_p_row_ptr, int32_t* out_p_col, int32_t* out_p_edge_vid,
                           uint8_t* out_validities);
int32_t porrt_graph_destroy(porrt_graph* g);
/* pto_graph::save: serde_json::to_writer_pretty layout.  p_* == NULL: parents are derived from the children (exact for graphs whose
 * edges were added row by row, e.g. a PRM). */
int32_t porrt_graph_save_json(porrt_ctx* ctx, const char* path, int64_t V, const double* xy, const int32_t* node_vid,
                              const int64_t* row_ptr, const int32_t* col, const int32_t* edge_vid, const int64_t* p_row_ptr,
                              const int32_t* p_col, const int32_t* p_edge_vid, const uint8_t* validities, int32_t n_validities,
                              int32_t n_worlds);

#ifdef __cplusplus
}
#endif
#endif /* PORRT_B200_H */
