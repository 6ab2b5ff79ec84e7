"""Host-side mirror of the reference's interface for the hot path, over the C ABI (include/porrt_b200.h).

Names follow the reference crate so that parity tests read like its own tests:
  Map / MapShelfDomain      src/map_io.rs, src/map_shelves_io.rs  (PTOFuncs<2>: state_validity, transition_validator,
                            world_validities, observe's visibility test, reachable_belief_states)
  KdTree                    src/nearest_neighbor.rs               (nearest_neighbor[_filtered], nearest_neighbors)
  PRM                       src/prm.rs                            (grow_graph)
  plan_qmdp                 src/qmdp_policy_extractor.rs:23-35
  plan_belief_space         src/pto.rs:152-182
Everything is batched (numpy arrays in, numpy arrays out); a batch of one is the per-query trait method.
Python here is only the driver: all computation happens in libporrt_b200.so on the GPU.
"""
import ctypes as C

import numpy as np

from . import _lib

INVALID, PANIC_OOB, PANIC_ZONE_UNWRAP, PANIC_MULTI_ZONE = -1, -2, -3, -4
DOOR, SHELF = 0, 1
NODE_UNKNOWN, NODE_ACTION, NODE_OBSERVATION = 0, 1, 2
ERR_CAPACITY = 4
OPT_FORCE_LARGE_MAP_PATH = 1
OPT_FORCE_GLOBAL_SWEEPS = 2
OPT_FORCE_THREAD_PER_QUERY_NN = 3
OPT_PRM_PATHS_CHUNK_COLUMNS = 4
OPT_REPARENT_BRUTE_MAX_NODES = 5
PATH_FOUND, PATH_NONE, PATH_CYCLE = 0, 1, 2   # PORRT_PATH_* (porrt_prm_plan_paths)
PTO_MAX_ROADMAPS = 65535   # PORRT_PTO_MAX_ROADMAPS


class PorrtError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__("porrt_b200 error %d: %s" % (code, msg))
        self.code = code


def _p(a):
    if a is None:
        return None
    assert a.flags["C_CONTIGUOUS"], "array must be C-contiguous"
    return a.ctypes.data_as(C.c_void_p)


def _f64(x, cols=None):
    a = np.ascontiguousarray(np.asarray(x, dtype=np.float64))
    if cols is not None:
        a = a.reshape(-1, cols)
    return a


class Context:
    """One GPU context (porrt_ctx).  Fails loudly when the library or a B200-class device is missing."""

    def __init__(self, device=0):
        self.lib = _lib.load()
        h = C.c_void_p()
        rc = self.lib.porrt_ctx_create(device, C.byref(h))
        if rc:
            raise PorrtError(rc, "porrt_ctx_create failed (no sm_100 CUDA device? there is no CPU fallback)")
        self.h = h

    def close(self):
        if getattr(self, "h", None):
            self.lib.porrt_ctx_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def check(self, rc):
        if rc:
            raise PorrtError(rc, (self.lib.porrt_last_error(self.h) or b"").decode())

    def set_stream(self, cuda_stream_ptr):
        self.check(self.lib.porrt_ctx_set_stream(self.h, cuda_stream_ptr))

    def synchronize(self):
        self.check(self.lib.porrt_ctx_synchronize(self.h))

    def bind_host_thread(self):
        """bind this thread to the NUMA node next to the GPU; returns the node (-1: unknown)"""
        node = C.c_int32()
        self.check(self.lib.porrt_ctx_bind_host_thread(self.h, C.byref(node)))
        return node.value

    def launch_count(self):
        return self.lib.porrt_ctx_launch_count(self.h)

    def set_option(self, option, value):
        self.check(self.lib.porrt_ctx_set_option(self.h, int(option), int(value)))

    # -- multi-GPU (SURVEY 8(e)): one process and one Context per GPU; see po_rrt_b200/shard.py:init_comm for the plumbing
    def comm_unique_id(self):
        """rank 0: the 128-byte ncclUniqueId every rank must pass to comm_init"""
        out = np.zeros(128, dtype=np.uint8)
        rc = self.lib.porrt_comm_unique_id(_p(out))
        if rc:
            raise PorrtError(rc, "porrt_comm_unique_id failed (libnccl.so.2 not loadable?)")
        return out

    def comm_init(self, unique_id, rank, world):
        uid = np.ascontiguousarray(unique_id, dtype=np.uint8)
        assert uid.size == 128
        self.check(self.lib.porrt_comm_init(self.h, _p(uid), int(rank), int(world)))

    def comm_destroy(self):
        self.check(self.lib.porrt_comm_destroy(self.h))

    def comm_info(self):
        r, w, v = C.c_int32(), C.c_int32(), C.c_int32()
        self.check(self.lib.porrt_comm_info(self.h, C.byref(r), C.byref(w), C.byref(v)))
        return r.value, w.value, v.value

    def all_gather_dev(self, send_ptr, recv_ptr, n_total, bytes_per_unit):
        """device pointers (ints); rank r owns rows shard_range(n_total, r, world); send_ptr None/0 = in place"""
        self.check(self.lib.porrt_comm_all_gather_dev(self.h, send_ptr or None, recv_ptr, int(n_total), int(bytes_per_unit)))

    def last_phase_ms(self):
        out = np.zeros(16)
        n = C.c_int32()
        self.check(self.lib.porrt_ctx_last_phase_ms(self.h, _p(out), 16, C.byref(n)))
        return [float(x) for x in out[:n.value]]


class _GridDomain:
    KIND = DOOR

    def __init__(self, ctx, occ, low, up):
        self.ctx = ctx
        self.occ = np.ascontiguousarray(occ, dtype=np.uint8)
        self.low, self.up = _f64(low), _f64(up)
        self.zones = None
        self.visibility_distance = 0.0
        self._uploaded = False

    # -- construction (Map::open / add_zones / init_without_zones)
    @classmethod
    def open(cls, ctx, filepath, low, up):
        from .pgm import read_pgm
        return cls(ctx, read_pgm(filepath), low, up)

    def add_zones(self, zones, visibility_distance):
        if isinstance(zones, str):
            from .pgm import read_pgm
            zones = read_pgm(zones)
        self.zones = np.ascontiguousarray(zones, dtype=np.uint8)
        assert self.zones.shape == self.occ.shape
        self.visibility_distance = float(visibility_distance)
        self._upload()

    def init_without_zones(self):
        self.zones = None
        self._upload()

    def _upload(self):
        H, W = self.occ.shape
        c = self.ctx
        c.check(c.lib.porrt_map_upload(c.h, _p(self.occ), _p(self.zones), H, W, _p(self.low), _p(self.up), self.KIND,
                                       self.visibility_distance))
        nz, nw, nv, mw = (C.c_int32() for _ in range(4))
        c.check(c.lib.porrt_map_info(c.h, C.byref(nz), C.byref(nw), C.byref(nv), C.byref(mw)))
        self.n_zones, self._n_worlds, self.n_validities, self.mask_words = nz.value, nw.value, nv.value, mw.value
        self._uploaded = True

    def _need(self):
        if not self._uploaded:
            self._upload()

    # -- PTOFuncs<2>
    def n_worlds(self):
        self._need()
        return self._n_worlds

    def world_validities_words(self):
        self._need()
        out = np.zeros((self.n_validities, self.mask_words), np.uint64)
        self.ctx.check(self.ctx.lib.porrt_map_world_validities(self.ctx.h, _p(out)))
        return out

    def world_validities(self):
        """Vec<WorldMask> as a [n_validities, n_worlds] 0/1 array"""
        w = self.world_validities_words()
        bits = np.zeros((self.n_validities, self._n_worlds), np.uint8)
        for k in range(self._n_worlds):
            bits[:, k] = (w[:, k // 64] >> np.uint64(k % 64)) & np.uint64(1)
        return bits

    def zone_positions(self):
        self._need()
        out = np.zeros((self.n_zones, 2))
        self.ctx.check(self.ctx.lib.porrt_map_zone_positions(self.ctx.h, _p(out)))
        return out

    def state_validity(self, xy):
        """Option<usize> per state: >= 0 validity id, -1 None, < -1 the reference's panic"""
        self._need()
        xy = _f64(xy, 2)
        out = np.empty(len(xy), np.int32)
        self.ctx.check(self.ctx.lib.porrt_state_validity(self.ctx.h, _p(xy), len(xy), _p(out)))
        return out

    def transition_validator(self, from_xy, to_xy, want_masks=False, compact=False, vid_out=None):
        """compact=True: one signed byte per edge (porrt_edge_validity_i8), no masks"""
        self._need()
        f, t = _f64(from_xy, 2), _f64(to_xy, 2)
        assert len(f) == len(t)
        if compact:
            out = np.empty(len(f), np.int8) if vid_out is None else vid_out
            self.ctx.check(self.ctx.lib.porrt_edge_validity_i8(self.ctx.h, _p(f), _p(t), len(f), _p(out)))
            return out
        out = np.empty(len(f), np.int32) if vid_out is None else vid_out
        masks = np.empty((len(f), self.mask_words), np.uint64) if want_masks else None
        self.ctx.check(self.ctx.lib.porrt_edge_validity(self.ctx.h, _p(f), _p(t), len(f), _p(out), _p(masks)))
        return (out, masks) if want_masks else out

    def transition_validator_nodes(self, from_idx, to_idx, want_masks=False, vid_out=None, mask_out=None, compact=False):
        """transition_validator between nodes of the uploaded vertex set (KdTree.set / porrt_vertices_set), by id"""
        self._need()
        fi, ti = np.ascontiguousarray(from_idx, np.int32), np.ascontiguousarray(to_idx, np.int32)
        n = len(fi)
        if compact:
            vid = np.empty(n, np.int8) if vid_out is None else vid_out
            self.ctx.check(self.ctx.lib.porrt_edge_validity_indexed_i8(self.ctx.h, _p(fi), _p(ti), n, _p(vid)))
            return vid
        vid = np.empty(n, np.int32) if vid_out is None else vid_out
        masks = (np.empty((n, self.mask_words), np.uint64) if mask_out is None else mask_out) if want_masks else None
        c = self.ctx
        c.check(c.lib.porrt_edge_validity_indexed(c.h, _p(fi), _p(ti), n, _p(vid), _p(masks)))
        return (vid, masks) if want_masks else vid

    def transition_validator_adjacency(self, row_ptr, col, row_is_to=True, vid_out=None):
        """transition_validator for every entry of an adjacency over the uploaded vertex set: entry e of row r is the edge
        col[e] -> r (row_is_to, the planners' neighbour -> new node) or r -> col[e]; one signed byte per entry"""
        self._need()
        rp, cl = np.ascontiguousarray(row_ptr, np.int64), np.ascontiguousarray(col, np.int32)
        vid = np.empty(len(cl), np.int8) if vid_out is None else vid_out
        self.ctx.check(self.ctx.lib.porrt_edge_validity_csr_i8(self.ctx.h, _p(rp), _p(cl), len(rp) - 1, 1 if row_is_to else 0, _p(vid)))
        return vid

    def is_transition_valid(self, from_xy, to_xy, compat_row):
        """PTOPolicyRefiner::is_transition_valid (pto_policy_refiner.rs:395-423), batched -> (valid u8, status i32)"""
        self._need()
        f, t = _f64(from_xy, 2), _f64(to_xy, 2)
        row = np.ascontiguousarray(np.asarray(compat_row, dtype=np.uint8))
        assert len(f) == len(t) and len(row) == self.n_validities
        valid = np.empty(len(f), np.uint8)
        status = np.empty(len(f), np.int32)
        self.ctx.check(self.ctx.lib.porrt_transition_valid(self.ctx.h, _p(f), _p(t), len(f), _p(row), _p(valid), _p(status)))
        return valid, status

    def partial_shortcut(self, states, compat_row, n_iterations, sampler_seed=0):
        """PTOPolicyRefiner::partial_shortcut (pto_policy_refiner.rs:158-206) on one path piece
        -> (refined states, committed shortcuts, device round trips)"""
        self._need()
        st = _f64(states, 2).copy()
        row = np.ascontiguousarray(np.asarray(compat_row, dtype=np.uint8))
        assert len(row) == self.n_validities
        commits, waves = C.c_int32(), C.c_int32()
        self.ctx.check(self.ctx.lib.porrt_partial_shortcut(self.ctx.h, _p(st), len(st), _p(row), int(n_iterations), int(sampler_seed),
                                                           C.byref(commits), C.byref(waves)))
        return st, commits.value, waves.value

    def partial_shortcut_batch(self, pieces, compat_rows, n_iterations, sampler_seed=0):
        """partial_shortcut for all path pieces of a policy in shared device waves -> (list of refined pieces, commits[], waves)"""
        self._need()
        ptr = np.zeros(len(pieces) + 1, np.int32)
        ptr[1:] = np.cumsum([len(p) for p in pieces])
        st = np.ascontiguousarray(np.concatenate([_f64(p, 2) for p in pieces])) if len(pieces) else np.zeros((0, 2))
        rows = np.ascontiguousarray(np.asarray(compat_rows, dtype=np.uint8).reshape(len(pieces), self.n_validities))
        commits = np.zeros(len(pieces), np.int32)
        waves = C.c_int32()
        self.ctx.check(self.ctx.lib.porrt_partial_shortcut_batch(self.ctx.h, _p(st), _p(ptr), len(pieces), _p(rows), int(n_iterations),
                                                                 int(sampler_seed), _p(commits), C.byref(waves)))
        return [st[ptr[k]:ptr[k + 1]].copy() for k in range(len(pieces))], commits, waves.value

    def visible_zones(self, xy):
        """geometric part of observe(): (zone bitmask, status) per state"""
        self._need()
        xy = _f64(xy, 2)
        mask = np.empty(len(xy), np.uint64)
        status = np.empty(len(xy), np.int32)
        self.ctx.check(self.ctx.lib.porrt_visibility(self.ctx.h, _p(xy), len(xy), _p(mask), _p(status)))
        return mask, status

    def reachable_belief_states(self, start_belief, cap=1 << 16):
        self._need()
        b0 = _f64(start_belief)
        out = np.empty((cap, self._n_worlds))
        n = C.c_int32()
        self.ctx.check(self.ctx.lib.porrt_reachable_belief_states(self.ctx.h, _p(b0), _p(out), cap, C.byref(n)))
        return out[:n.value].copy()


class Map(_GridDomain):
    """door/zone domain, 2^Z worlds (src/map_io.rs)"""
    KIND = DOOR


class MapShelfDomain(_GridDomain):
    """object-in-one-of-Z-shelves domain, Z worlds (src/map_shelves_io.rs)"""
    KIND = SHELF


class KdTree:
    """Batched stand-in for KdTree<2> (src/nearest_neighbor.rs): vertex i carries id i."""

    def __init__(self, ctx, xy=None, cell_size=0.0):
        self.ctx = ctx
        self.n = 0
        if xy is not None:
            self.set(xy, cell_size)

    def set(self, xy, cell_size=0.0):
        xy = _f64(xy, 2)
        self.xy = xy
        self.n = len(xy)
        self.ctx.check(self.ctx.lib.porrt_vertices_set(self.ctx.h, _p(xy), len(xy), float(cell_size)))

    def add(self, xy):
        """KdTree::add (nearest_neighbor.rs:29-46) for one or more states: ids continue after the current set; only the new
        coordinates are uploaded (porrt_vertices_append)"""
        xy = _f64(xy, 2)
        if self.n == 0:
            return self.set(xy)
        self.ctx.check(self.ctx.lib.porrt_vertices_append(self.ctx.h, _p(xy), len(xy)))
        self.xy = None          # the device copy is the set now; preorder_rank() ranks it in place
        self.n += len(xy)

    def nearest_neighbors(self, q, radius, prefix_limit=None, reach_mask=None, world=None, cap=None, ids_out=None):
        """radius search -> (offsets[m+1], ids) with ids ascending per query.  ids_out: optional preallocated int32 buffer
        (e.g. pinned host memory) of at least `cap` entries"""
        q = _f64(q, 2)
        m = len(q)
        r = np.ascontiguousarray(np.broadcast_to(np.asarray(radius, np.float64), (m,)))
        pl = None if prefix_limit is None else np.ascontiguousarray(prefix_limit, np.uint32)
        rm = None if reach_mask is None else np.ascontiguousarray(reach_mask, np.uint64).reshape(self.n, -1)
        rw = 1 if rm is None else rm.shape[1]
        w = None if world is None else np.ascontiguousarray(world, np.uint32)
        offs = np.empty(m + 1, np.int64)
        cap = cap if cap is not None else max(1024, 64 * m)
        total = C.c_int64()
        while True:
            ids = ids_out if (ids_out is not None and len(ids_out) >= cap) else np.empty(cap, np.int32)
            rc = self.ctx.lib.porrt_radius_query(self.ctx.h, _p(q), _p(r), m, _p(pl), _p(rm), rw, _p(w), _p(offs), _p(ids), cap,
                                                 C.byref(total))
            if rc == ERR_CAPACITY:
                cap = total.value
                continue
            self.ctx.check(rc)
            return offs, ids[:total.value]

    def nearest_neighbor(self, q, reach_mask=None, world=None):
        """-> (id, dist, ties); id = -1 when the filter rejects everything (the reference returns the root)"""
        q = _f64(q, 2)
        m = len(q)
        rm = None if reach_mask is None else np.ascontiguousarray(reach_mask, np.uint64).reshape(self.n, -1)
        rw = 1 if rm is None else rm.shape[1]
        w = None if world is None else np.ascontiguousarray(world, np.uint32)
        ids, dist, ties = np.empty(m, np.int32), np.empty(m), np.empty(m, np.int32)
        self.ctx.check(self.ctx.lib.porrt_nearest(self.ctx.h, _p(q), m, _p(rm), rw, _p(w), _p(ids), _p(dist), _p(ties)))
        return ids, dist, ties

    def knn(self, q, k, ids_out=None, dist_out=None):
        q = _f64(q, 2)
        m = len(q)
        ids = ids_out if ids_out is not None else np.empty((m, k), np.int32)
        dist = dist_out if dist_out is not None else np.empty((m, k))
        self.ctx.check(self.ctx.lib.porrt_knn(self.ctx.h, _p(q), m, k, _p(ids), _p(dist)))
        return ids, dist

    def preorder_rank(self):
        out = np.empty(self.n, np.int32)
        self.ctx.check(self.ctx.lib.porrt_kd_preorder_rank(self.ctx.h, _p(self.xy) if self.xy is not None else None, self.n, _p(out)))
        return out


class PRM:
    """src/prm.rs: the fully batchable planner.  `fns` is an uploaded Map / MapShelfDomain."""

    def __init__(self, fns):
        self.fns = fns
        self.ctx = fns.ctx
        self.states = np.zeros((0, 2))
        self.row_ptr = np.zeros(1, np.int64)
        self.col = np.zeros(0, np.int32)
        self.phase_ms = np.zeros(8)

    def init(self, start):
        self.states = _f64(start, 2)

    def grow_graph(self, samples, max_step, search_radius, col_out=None, fetch_col=True, row_ptr_out=None):
        """samples: the ContinuousSampler stream (n_iter states); nodes = [init state] + samples.
        fetch_col=False leaves the column array on the device (row_ptr still comes back); col_out / row_ptr_out: caller-owned
        (e.g. pinned) result buffers; samples are used in place (no host copy) when no init state precedes them"""
        self.fns._need()
        samples = _f64(samples, 2)
        xy = samples if len(self.states) == 0 else np.ascontiguousarray(np.vstack([self.states, samples]))
        n = len(xy)
        row_ptr = np.empty(n + 1, np.int64) if row_ptr_out is None else row_ptr_out[:n + 1]
        n_edges = C.c_int64()
        # a caller-owned column buffer goes straight into the build: its copy leaves in row blocks while the CSR is still being
        # assembled (graph.cu); otherwise the size is asked for first (PORRT_ERR_CAPACITY) and the columns are fetched afterwards
        direct = fetch_col and col_out is not None
        rc = self.ctx.lib.porrt_prm_build(self.ctx.h, _p(xy), n, max_step, search_radius, _p(row_ptr), _p(col_out) if direct else None,
                                          len(col_out) if direct else 0, C.byref(n_edges), _p(self.phase_ms))
        if rc != ERR_CAPACITY:
            self.ctx.check(rc)
        if not fetch_col:
            self.states, self.row_ptr, self.col = xy, row_ptr, None
            return self
        col = np.empty(n_edges.value, np.int32) if col_out is None else col_out
        if not direct or rc == ERR_CAPACITY:
            self.ctx.check(self.ctx.lib.porrt_prm_fetch(self.ctx.h, None, _p(col), len(col)))
        self.states, self.row_ptr, self.col = xy, row_ptr, col[:n_edges.value]
        return self

    def plan_paths(self, starts, goals):
        """PRM::plan_path (prm.rs:111-122) for every (start, goal) row, on the roadmap the last PRM build of this context left on the
        device (porrt_prm_plan_paths; only the paths come back).  -> (paths: a list of [L, 2] arrays, cost[n], status[n] (PATH_*),
        start_node[n], goal_node[n]); a query whose status is not PATH_FOUND has an empty path"""
        s, g = _f64(starts, 2), _f64(goals, 2)
        if len(s) != len(g):
            raise ValueError("plan_paths: %d starts, %d goals" % (len(s), len(g)))
        n = len(s)
        sn, gn, st = np.empty(max(n, 1), np.int32), np.empty(max(n, 1), np.int32), np.empty(max(n, 1), np.int32)
        cost, ptr, total = np.empty(max(n, 1)), np.empty(n + 1, np.int64), C.c_int64()
        cap = 64 * n
        while True:
            xy = np.empty((max(cap, 1), 2))
            rc = self.ctx.lib.porrt_prm_plan_paths(self.ctx.h, _p(s), _p(g), n, _p(sn), _p(gn), _p(cost), _p(st), _p(ptr), _p(xy), cap,
                                                   C.byref(total))
            if rc == ERR_CAPACITY and total.value > cap:
                cap = total.value
                continue
            self.ctx.check(rc)
            paths = [xy[ptr[q]:ptr[q + 1]].copy() for q in range(n)]
            return paths, cost[:n].copy(), st[:n].copy(), sn[:n].copy(), gn[:n].copy()

    def plan_path(self, start, goal):
        """PRM::plan_path for one query, as the oracle's PRM.plan_path returns it: the path [L, 2], or an empty (0, 2) array when
        there is none (status PATH_NONE or PATH_CYCLE)"""
        paths, _, status, _, _ = self.plan_paths([start], [goal])
        return paths[0] if status[0] == PATH_FOUND else np.zeros((0, 2))


def dijkstra_worlds(ctx, row_ptr, col, xy, node_vid, validities_words, finals_per_world):
    """plan_qmdp's loop: one dijkstra per world over PTOGraphWorldView -> cost_to_goals[W][V] (+ sweeps).
    finals_per_world=None with validities_words=None runs the plain-graph dijkstra (pass finals as a flat list)."""
    row_ptr = np.ascontiguousarray(row_ptr, np.int64)
    col = np.ascontiguousarray(col, np.int32)
    xy = _f64(xy, 2)
    V = len(xy)
    sweeps = C.c_int32()
    if validities_words is None:
        fin = np.ascontiguousarray(finals_per_world, np.int32)
        fptr = np.array([0, len(fin)], np.int64)
        out = np.empty((1, V))
        ctx.check(ctx.lib.porrt_sssp_worlds(ctx.h, V, _p(row_ptr), _p(col), _p(xy), None, None, 0, 0, 0, _p(fptr), _p(fin), _p(out),
                                            C.byref(sweeps)))
        return out[0], sweeps.value
    vw = np.ascontiguousarray(validities_words, np.uint64)
    nvid = np.ascontiguousarray(node_vid, np.int32)
    W = len(finals_per_world)
    fptr = np.zeros(W + 1, np.int64)
    for w, f in enumerate(finals_per_world):
        fptr[w + 1] = fptr[w] + len(f)
    fin = np.ascontiguousarray(np.concatenate([np.asarray(f, np.int32) for f in finals_per_world]) if fptr[-1] else np.zeros(0, np.int32))
    out = np.empty((W, V))
    ctx.check(ctx.lib.porrt_sssp_worlds(ctx.h, V, _p(row_ptr), _p(col), _p(xy), _p(nvid), _p(vw), vw.shape[0], vw.shape[1], W,
                                        _p(fptr), _p(fin), _p(out), C.byref(sweeps)))
    return out, sweeps.value


def dijkstra_worlds_resident_prm(fns, V, finals_per_world, want_dist=True):
    """plan_qmdp on the roadmap the last PRM build left on the device (porrt_sssp_worlds_prm): node validity ids are the map's state
    validity of the vertices, evaluated on the device.  -> (cost_to_goals[W][V] or None, rounds)"""
    ctx = fns.ctx
    W = len(finals_per_world)
    fptr = np.zeros(W + 1, np.int64)
    for w, f in enumerate(finals_per_world):
        fptr[w + 1] = fptr[w] + len(f)
    fin = np.ascontiguousarray(np.concatenate([np.asarray(f, np.int32) for f in finals_per_world]) if fptr[-1] else np.zeros(0, np.int32))
    out = np.empty((W, V)) if want_dist else None
    sweeps = C.c_int32()
    ctx.check(ctx.lib.porrt_sssp_worlds_prm(ctx.h, _p(fptr), _p(fin), _p(out) if want_dist else None, C.byref(sweeps)))
    return out, sweeps.value


class BeliefPlan:
    """result of plan_belief_space; `dist` / `type` are None when the call was made with copy=None -- fetch_table() then brings
    the ctx-owned table over on demand (porrt_belief_result; valid until the next belief call on the ctx)"""
    dist = None
    type = None

    def fetch_table(self):
        pd, pt = C.POINTER(C.c_double)(), C.POINTER(C.c_uint8)()
        self._ctx.check(self._ctx.lib.porrt_belief_result(self._ctx.h, C.byref(pd), C.byref(pt), None, None))
        self.dist = np.ctypeslib.as_array(pd, shape=self._shape)
        self.type = np.ctypeslib.as_array(pt, shape=self._shape)
        return self.dist, self.type


def plan_belief_space(fns, row_ptr, col, edge_vid, xy, node_vid, start_belief, final_ids, final_masks_words, beliefs=None, copy=True):
    """PTO::plan_belief_space (src/pto.rs:152-182) for a grown roadmap given as CSR (children adjacency).
    Returns a BeliefPlan with beliefs, visible (zone masks), dist[V,B], type[V,B], policy arrays, expected_cost.
    copy=False: dist / type are views of the ctx-owned pinned result (porrt_belief_result), valid until the next call on the ctx.
    copy=None: policy only -- the V x B table stays on the device (the policy walk fetches the few value columns it visits);
    plan.fetch_table() brings it over later if wanted."""
    ctx = fns.ctx
    fns._need()
    row_ptr = np.ascontiguousarray(row_ptr, np.int64)
    col = np.ascontiguousarray(col, np.int32)
    edge_vid = np.ascontiguousarray(edge_vid, np.int32)
    xy = _f64(xy, 2)
    node_vid = np.ascontiguousarray(node_vid, np.int32)
    V = len(xy)
    plan = BeliefPlan()
    plan.beliefs = fns.reachable_belief_states(start_belief) if beliefs is None else _f64(beliefs, fns.n_worlds())
    B = len(plan.beliefs)
    plan.visible, status = fns.visible_zones(xy)
    if (status != 0).any():
        raise PorrtError(5, "observe() would panic at node %d (code %d)" % (int(np.nonzero(status)[0][0]), int(status[status != 0][0])))
    vw = fns.world_validities_words()
    fin = np.ascontiguousarray(final_ids, np.int32)
    fmask = np.ascontiguousarray(final_masks_words, np.uint64).reshape(len(fin), fns.mask_words)
    if copy:
        plan.dist = np.empty((V, B))
        plan.type = np.empty((V, B), np.uint8)
    sweeps = C.c_int32()
    plan.phase_ms = np.zeros(4)
    ctx.check(ctx.lib.porrt_belief_vi(ctx.h, V, _p(row_ptr), _p(col), _p(edge_vid), _p(xy), _p(node_vid), _p(vw), vw.shape[0],
                                      vw.shape[1], fns.n_worlds(), _p(plan.beliefs), B, _p(plan.visible), _p(fin), _p(fmask),
                                      len(fin), _p(plan.dist) if copy else None, _p(plan.type) if copy else None, C.byref(sweeps),
                                      _p(plan.phase_ms)))
    plan.sweeps = sweeps.value
    plan._ctx, plan._shape = ctx, (V, B)
    if copy is False:
        plan.fetch_table()
    cap = 4096
    n, cost = C.c_int64(), C.c_double()
    while True:
        node, belief, parent = (np.empty(cap, np.int32) for _ in range(3))
        leaf = np.empty(cap, np.uint8)
        rc = ctx.lib.porrt_extract_policy(ctx.h, _p(node), _p(belief), _p(parent), _p(leaf), cap, C.byref(n), C.byref(cost))
        if rc == ERR_CAPACITY:
            cap = n.value
            continue
        ctx.check(rc)
        break
    k = n.value
    plan.policy_node, plan.policy_belief, plan.policy_parent = node[:k].copy(), belief[:k].copy(), parent[:k].copy()
    plan.policy_leaf = leaf[:k].copy()
    plan.expected_cost = cost.value
    return plan


def refine_policy_shortcut(ctx, plan, n_iterations, sampler_seed=0):
    """PTOPolicyRefiner::refine_solution(PartialShortCut(n)) on a BeliefPlan of the ctx's last plan_belief_space
    -> dict(xy, node, belief, parent, is_leaf, expected_cost, commits)"""
    n_pol = len(plan.policy_node)
    cap = n_pol
    xy = np.empty((cap, 2))
    node, belief, parent = (np.empty(cap, np.int32) for _ in range(3))
    leaf = np.empty(cap, np.uint8)
    n, cost, commits = C.c_int64(), C.c_double(), C.c_int64()
    pn, pb, pp = (np.ascontiguousarray(a, np.int32) for a in (plan.policy_node, plan.policy_belief, plan.policy_parent))
    ctx.check(ctx.lib.porrt_refine_policy_shortcut(ctx.h, _p(pn), _p(pb), _p(pp), n_pol, int(n_iterations), int(sampler_seed), _p(xy), _p(node),
                                                   _p(belief), _p(parent), _p(leaf), cap, C.byref(n), C.byref(cost), C.byref(commits)))
    k = n.value
    return {"xy": xy[:k], "node": node[:k], "belief": belief[:k], "parent": parent[:k], "is_leaf": leaf[:k], "expected_cost": cost.value,
            "commits": commits.value}


def policy_decompose(parent):
    """Policy::decompose (common.rs:85-129) -> (pieces: list of node-id arrays, skeleton: list of successor-piece lists)"""
    par = np.ascontiguousarray(parent, np.int32)
    n = len(par)
    lib = _lib.load()
    piece_ptr, nodes = np.empty(n + 2, np.int32), np.empty(max(n, 1), np.int32)
    succ_ptr, succ = np.empty(n + 2, np.int32), np.empty(max(n, 1), np.int32)
    npc = C.c_int32()
    rc = lib.porrt_policy_decompose(_p(par), n, _p(piece_ptr), _p(nodes), _p(succ_ptr), _p(succ), n + 1, C.byref(npc))
    if rc:
        raise PorrtError(rc, "porrt_policy_decompose")
    k = npc.value
    return ([nodes[piece_ptr[p]:piece_ptr[p + 1]].copy() for p in range(k)], [succ[succ_ptr[p]:succ_ptr[p + 1]].tolist() for p in range(k)])


def policy_expected_cost(xy, belief_id, parent, beliefs):
    """Policy::compute_expected_costs_to_goals (common.rs:131-153) with cost = norm2"""
    x, bid, par = _f64(xy, 2), np.ascontiguousarray(belief_id, np.int32), np.ascontiguousarray(parent, np.int32)
    bel = np.ascontiguousarray(np.atleast_2d(np.asarray(beliefs, np.float64)))
    out = C.c_double()
    rc = _lib.load().porrt_policy_expected_cost(_p(x), _p(bid), _p(par), len(par), _p(bel), bel.shape[0], bel.shape[1], C.byref(out))
    if rc:
        raise PorrtError(rc, "porrt_policy_expected_cost")
    return out.value


def refine_policy_reparent(ctx, plan, radius):
    """PTOPolicyRefiner::refine_solution(Reparent(radius)) on a BeliefPlan of the ctx's last plan_belief_space
    -> dict(xy, node, belief, parent, is_leaf, expected_cost, tree_nodes, transitions)"""
    n_pol = len(plan.policy_node)
    pn, pb, pp = (np.ascontiguousarray(a, np.int32) for a in (plan.policy_node, plan.policy_belief, plan.policy_parent))
    cap = max(n_pol, 64)
    while True:
        xy = np.empty((cap, 2))
        node, belief, parent = (np.empty(cap, np.int32) for _ in range(3))
        leaf = np.empty(cap, np.uint8)
        n, cost, tn, tr = C.c_int64(), C.c_double(), C.c_int64(), C.c_int64()
        rc = ctx.lib.porrt_refine_policy_reparent(ctx.h, _p(pn), _p(pb), _p(pp), n_pol, float(radius), _p(xy), _p(node), _p(belief), _p(parent),
                                                  _p(leaf), cap, C.byref(n), C.byref(cost), C.byref(tn), C.byref(tr))
        if rc == 4 and n.value > cap:   # PORRT_ERR_CAPACITY
            cap = n.value
            continue
        ctx.check(rc)
        break
    k = n.value
    return {"xy": xy[:k], "node": node[:k], "belief": belief[:k], "parent": parent[:k], "is_leaf": leaf[:k], "expected_cost": cost.value,
            "tree_nodes": tn.value, "transitions": tr.value}


class BeliefGraph:
    """src/belief_graph.rs BeliefGraph as arrays: belief node k = (state xy[k], belief_id[k], node_type[k]); children adjacency
    as CSR in add_edge order.  conditional_dijkstra / extract_policy are the reference's free functions (:89-267)."""

    def __init__(self, ctx, row_ptr, col, xy, node_type, belief_id, beliefs, dim=2):
        """dim: state dimension (BeliefGraph<N>; 2 -> the two-dimensional entry points, else porrt_*_nd)"""
        self.ctx = ctx
        self.dim = int(dim)
        self.row_ptr = np.ascontiguousarray(row_ptr, np.int64)
        self.col = np.ascontiguousarray(col, np.int32)
        self.xy = _f64(xy, self.dim)
        self.node_type = np.ascontiguousarray(node_type, np.uint8)
        self.belief_id = np.ascontiguousarray(belief_id, np.int32)
        self.beliefs = np.ascontiguousarray(np.atleast_2d(np.asarray(beliefs, np.float64)))
        self.V = len(self.xy)
        assert len(self.row_ptr) == self.V + 1 and len(self.node_type) == self.V and len(self.belief_id) == self.V

    def _graph_args(self):
        B, nw = self.beliefs.shape
        return (self.V, _p(self.row_ptr), _p(self.col), _p(self.xy), _p(self.node_type), _p(self.belief_id), _p(self.beliefs), B, nw)

    def conditional_dijkstra(self, final_node_ids):
        fin = np.ascontiguousarray(final_node_ids, np.int32)
        out = np.empty(self.V)
        sweeps = C.c_int32()
        c = self.ctx
        if self.dim == 2:
            c.check(c.lib.porrt_conditional_dijkstra(c.h, *self._graph_args(), _p(fin), len(fin), _p(out), C.byref(sweeps)))
        else:
            c.check(c.lib.porrt_conditional_dijkstra_nd(c.h, self.dim, *self._graph_args(), _p(fin), len(fin), _p(out), C.byref(sweeps)))
        self.sweeps = sweeps.value
        return out

    def extract_policy(self, expected_costs_to_goals):
        """-> (belief_node[k], parent[k], is_leaf[k], expected_cost) in the reference's creation order"""
        dist = _f64(expected_costs_to_goals)
        c = self.ctx
        cap = 1024
        n, cost = C.c_int64(), C.c_double()
        while True:
            node, parent = np.empty(cap, np.int32), np.empty(cap, np.int32)
            leaf = np.empty(cap, np.uint8)
            if self.dim == 2:
                rc = c.lib.porrt_extract_policy_graph(c.h, *self._graph_args(), _p(dist), _p(node), _p(parent), _p(leaf), cap,
                                                      C.byref(n), C.byref(cost))
            else:
                rc = c.lib.porrt_extract_policy_graph_nd(c.h, self.dim, *self._graph_args(), _p(dist), _p(node), _p(parent), _p(leaf), cap,
                                                         C.byref(n), C.byref(cost))
            if rc == ERR_CAPACITY:
                cap = max(n.value, 2 * cap)
                continue
            c.check(rc)
            break
        k = n.value
        return node[:k].copy(), parent[:k].copy(), leaf[:k].copy(), cost.value


def mmprm_plan(fns, schedule):
    """MapShelfDomainTampPRM::plan (src/map_shelves_tamp_prm.rs:308-326) for a recorded schedule (dict with the arrays of
    porrt_mmprm_plan: mode_node_ptr, samples, max_step, search_radius, mode_belief_id, beliefs, tr_from_mode, tr_to_mode,
    tr_pair_ptr, tr_pairs, mode_final_ptr, mode_final_nodes).  Returns (expected costs, BeliefGraph, policy tuple, phase ms)."""
    ctx = fns.ctx
    fns._need()
    s = schedule
    ptr = np.ascontiguousarray(s["mode_node_ptr"], np.int64)
    xy = _f64(s["samples"], 2)
    ms, sr = _f64(s["max_step"]), _f64(s["search_radius"])
    mb = np.ascontiguousarray(s["mode_belief_id"], np.int32)
    beliefs = np.ascontiguousarray(np.atleast_2d(np.asarray(s["beliefs"], np.float64)))
    trf, trt = np.ascontiguousarray(s["tr_from_mode"], np.int32), np.ascontiguousarray(s["tr_to_mode"], np.int32)
    trp = np.ascontiguousarray(s["tr_pair_ptr"], np.int64)
    pairs = np.ascontiguousarray(s["tr_pairs"], np.int32)
    fptr = np.ascontiguousarray(s["mode_final_ptr"], np.int64)
    fin = np.ascontiguousarray(s["mode_final_nodes"], np.int32)
    T = int(ptr[-1])
    dist = np.empty(T)
    n_edges, sweeps = C.c_int64(), C.c_int32()
    phase = np.zeros(4)
    ctx.check(ctx.lib.porrt_mmprm_plan(ctx.h, len(mb), _p(ptr), _p(xy), _p(ms), _p(sr), _p(mb), _p(beliefs), beliefs.shape[0],
                                       beliefs.shape[1], len(trf), _p(trf), _p(trt), _p(trp), _p(pairs), _p(fptr), _p(fin),
                                       _p(dist), C.byref(n_edges), C.byref(sweeps), _p(phase)))
    rp, col = np.empty(T + 1, np.int64), np.empty(n_edges.value, np.int32)
    typ, bid = np.empty(T, np.uint8), np.empty(T, np.int32)
    ctx.check(ctx.lib.porrt_mmprm_fetch_graph(ctx.h, _p(rp), _p(col), len(col), _p(typ), _p(bid)))
    graph = BeliefGraph(ctx, rp, col, xy, typ, bid, beliefs)
    graph.sweeps = sweeps.value
    policy = graph.extract_policy(dist)
    return dist, graph, policy, phase


def words_from_bits(bits):
    """[n, n_worlds] 0/1 -> [n, ceil(n_worlds/64)] u64 (bit w of word w/64 = world w)"""
    bits = np.atleast_2d(np.asarray(bits, np.uint8))
    n, nw = bits.shape
    out = np.zeros((n, (nw + 63) // 64), np.uint64)
    for w in range(nw):
        out[:, w // 64] |= bits[:, w].astype(np.uint64) << np.uint64(w % 64)
    return out


# ---------------------------------------------------------------------------------------------- host-side rows (no device work)
def heuristic_radius(n_nodes, max_step, search_radius, dim=2):
    """common.rs:357-369"""
    out = C.c_double()
    rc = _lib.load().porrt_heuristic_radius(int(n_nodes), float(max_step), float(search_radius), int(dim), C.byref(out))
    if rc:
        raise PorrtError(rc, "porrt_heuristic_radius")
    return out.value


def steer(from_xy, to_xy, max_step, dim=2):
    """common.rs:215-225, batched; returns the steered copies of to_xy (dim: state dimension, steer<N>)"""
    f, t = _f64(from_xy, dim), _f64(to_xy, dim).copy()
    if dim == 2:
        rc = _lib.load().porrt_steer(_p(f), _p(t), len(f), float(max_step))
    else:
        rc = _lib.load().porrt_steer_nd(_p(f), _p(t), len(f), int(dim), float(max_step))
    if rc:
        raise PorrtError(rc, "porrt_steer")
    return t


class Sampler:
    """one Pcg64::seed_from_u64(seed) stream: ContinuousSampler::sample / DiscreteSampler::sample (sample_space.rs)"""

    def __init__(self, seed=0):
        self.lib = _lib.load()
        self.h = C.c_void_p()
        rc = self.lib.porrt_sampler_create(int(seed), C.byref(self.h))
        if rc:
            raise PorrtError(rc, "porrt_sampler_create")

    def __del__(self):
        if getattr(self, "h", None):
            self.lib.porrt_sampler_destroy(self.h)
            self.h = None

    def sample_states(self, low, up, n):
        low, up = _f64(low), _f64(up)
        out = np.empty((n, len(low)))
        rc = self.lib.porrt_sampler_continuous(self.h, _p(low), _p(up), len(low), n, _p(out))
        if rc:
            raise PorrtError(rc, "porrt_sampler_continuous")
        return out

    def sample_discrete(self, n_choices, n):
        out = np.empty(n, np.uint64)
        rc = self.lib.porrt_sampler_discrete(self.h, int(n_choices), n, _p(out))
        if rc:
            raise PorrtError(rc, "porrt_sampler_discrete")
        return out


class SquareGoal:
    """common.rs:304-350: goals [(state, world mask bits)], max_dist"""

    def __init__(self, goal_to_validity, max_dist):
        self.lib = _lib.load()
        self.goals = _f64([g for g, _ in goal_to_validity], 2)
        self.bits = np.asarray([m for _, m in goal_to_validity], np.uint8)
        self.masks = words_from_bits(self.bits)
        self.max_dist = float(max_dist)
        self.n_worlds = self.bits.shape[1]
        self.world_to_goal = np.empty((self.n_worlds, 2))
        rc = self.lib.porrt_square_goal_examples(_p(self.goals), _p(self.masks), len(self.goals), self.n_worlds, _p(self.world_to_goal))
        if rc:
            raise PorrtError(rc, "validities shouldn't overlap (common.rs:320)")

    def goal_index(self, xy):
        xy = _f64(xy, 2)
        out = np.empty(len(xy), np.int32)
        rc = self.lib.porrt_square_goal(_p(self.goals), len(self.goals), self.max_dist, _p(xy), len(xy), _p(out))
        if rc:
            raise PorrtError(rc, "porrt_square_goal")
        return out

    def goal(self, state):
        """Option<WorldMask> as a bit list / None"""
        g = int(self.goal_index([state])[0])
        return None if g < 0 else [int(b) for b in self.bits[g]]

    def goal_example(self, world):
        return self.world_to_goal[world].copy()


class Reachability:
    """pto_reachability.rs; masks as 0/1 lists of length n_worlds"""

    def __init__(self):
        self.lib = _lib.load()
        self.h = None
        self.n_worlds = 0

    def __del__(self):
        if getattr(self, "h", None):
            self.lib.porrt_reach_destroy(self.h)
            self.h = None

    def _w(self, bits):
        assert len(bits) == self.n_worlds
        return words_from_bits([bits])[0].copy()

    def _ck(self, rc, what):
        if rc:
            raise PorrtError(rc, what)

    def set_root(self, validity):
        self.n_worlds = len(validity)
        self.h = C.c_void_p()
        self._ck(self.lib.porrt_reach_create(self.n_worlds, _p(self._w(validity)), C.byref(self.h)), "porrt_reach_create")

    def add_node(self, validity):
        self._ck(self.lib.porrt_reach_add_node(self.h, _p(self._w(validity))), "porrt_reach_add_node")

    def add_final_node(self, id, finality):
        self._ck(self.lib.porrt_reach_add_final_node(self.h, int(id), _p(self._w(finality))), "porrt_reach_add_final_node")

    def add_edge(self, a, b, edge_validity):
        self._ck(self.lib.porrt_reach_add_edge(self.h, int(a), int(b), _p(self._w(edge_validity))), "porrt_reach_add_edge")

    def n_nodes(self):
        n = C.c_int64()
        self._ck(self.lib.porrt_reach_count(self.h, C.byref(n), None), "porrt_reach_count")
        return n.value

    def masks_words(self, first=0, n=None):
        n = self.n_nodes() - first if n is None else n
        out = np.empty((n, (self.n_worlds + 63) // 64), np.uint64)
        self._ck(self.lib.porrt_reach_masks(self.h, first, n, _p(out)), "porrt_reach_masks")
        return out

    def reachability(self, id):
        w = self.masks_words(id, 1)[0]
        return [int((w[k // 64] >> np.uint64(k % 64)) & np.uint64(1)) for k in range(self.n_worlds)]

    def get_final_nodes_for_world(self, world):
        cap = 16
        while True:
            out, n = np.empty(cap, np.int64), C.c_int64()
            rc = self.lib.porrt_reach_final_nodes_for_world(self.h, int(world), _p(out), cap, C.byref(n))
            if rc == ERR_CAPACITY:
                cap = n.value
                continue
            self._ck(rc, "porrt_reach_final_nodes_for_world")
            return [int(x) for x in out[:n.value]]

    def finals(self):
        n = C.c_int64()
        self.lib.porrt_reach_finals(self.h, None, None, 0, C.byref(n))
        ids = np.empty(n.value, np.int64)
        masks = np.empty((n.value, (self.n_worlds + 63) // 64), np.uint64)
        self._ck(self.lib.porrt_reach_finals(self.h, _p(ids), _p(masks), n.value, C.byref(n)), "porrt_reach_finals")
        return ids, masks

    def is_final_set_complete(self):
        if self.h is None:
            return False
        out = C.c_int32()
        self._ck(self.lib.porrt_reach_is_final_set_complete(self.h, C.byref(out)), "porrt_reach_is_final_set_complete")
        return bool(out.value)


class PTO:
    """src/pto.rs PTO::grow_graph on the device (porrt_pto_grow): `fns` is an uploaded Map / MapShelfDomain, the two sampler streams
    are seeded with `seed` like PTO::new.  The roadmap stays on the device until graph_arrays() / reach_masks() / finals() ask."""

    def __init__(self, fns, low, up, seed=0):
        self.fns, self.ctx = fns, fns.ctx
        self.low, self.up, self.seed = _f64(low), _f64(up), int(seed)
        self.n_it, self.sizes, self.counters = 0, (0, 0, 0, 0), (0, 0, 0, 0)

    def grow_graph(self, start, goal, max_step, search_radius, n_iter_min, n_iter_max):
        """-> 0 when every world reaches a final node, 1 otherwise (pto.rs:131-138); PorrtError where the reference panics
        (e.code == 5, e.panic_code = the state / edge check's code, PORRT_INVALID for an invalid start)"""
        self.fns._need()
        c = self.ctx
        start = _f64(start)
        sizes, counters = np.zeros(4, np.int64), np.zeros(4, np.int64)
        complete, panic = C.c_int32(), C.c_int32()
        rc = c.lib.porrt_pto_grow(c.h, _p(start), _p(self.low), _p(self.up), self.seed, _p(goal.goals), _p(goal.masks), len(goal.goals),
                                  goal.max_dist, float(max_step), float(search_radius), int(n_iter_min), int(n_iter_max), _p(sizes),
                                  C.byref(complete), C.byref(panic), _p(counters))
        self.n_it, self.sizes, self.counters = int(sizes[0]), tuple(int(x) for x in sizes), tuple(int(x) for x in counters)
        if rc:
            err = PorrtError(rc, (c.lib.porrt_last_error(c.h) or b"").decode())
            err.panic_code = panic.value
            raise err
        return 0 if complete.value else 1

    def _fetch(self, *outs):
        self.ctx.check(self.ctx.lib.porrt_pto_fetch(self.ctx.h, *outs))

    def graph_arrays(self):
        """-> xy[V,2], node_vid[V], row_ptr[V+1], col[E], edge_vid[E]: the children adjacency in insertion order"""
        return _roadmap_graph_arrays(self._fetch, self.sizes)

    def reach_masks(self):
        """Reachability::reachability of every node as [V, n_worlds] 0/1"""
        return _roadmap_reach_masks(self._fetch, self.sizes, self.fns)

    def finals(self):
        """final node ids and their finality masks ([n, mask_words] u64), in add_final_node order"""
        return _roadmap_finals(self._fetch, self.sizes, self.fns)


class PTOBatch:
    """PTO::grow_graph for one roadmap per seed in `seeds`, all in one device call (porrt_pto_grow_batch); map, start, goal and
    parameters are shared.  Roadmap r is what PTO(fns, low, up, seeds[r]) grows, counters included.  After grow_graph the
    attributes n_it[R], sizes[R, 4], counters[R, 4] and panic_code[R] hold one row per roadmap; graph_arrays(r), reach_masks(r)
    and finals(r) read roadmap r.  The batch replaces the context's last growth (PTO objects on the same context then read
    roadmap 0)."""

    def __init__(self, fns, low, up, seeds):
        self.fns, self.ctx = fns, fns.ctx
        self.low, self.up = _f64(low), _f64(up)
        self.seeds = np.ascontiguousarray(np.asarray(seeds, dtype=np.uint64).reshape(-1))
        R = len(self.seeds)
        self.n_it, self.panic_code = np.zeros(R, np.int64), np.zeros(R, np.int32)
        self.sizes, self.counters = np.zeros((R, 4), np.int64), np.zeros((R, 4), np.int64)

    def __len__(self):
        return len(self.seeds)

    def grow_graph(self, start, goal, max_step, search_radius, n_iter_min, n_iter_max):
        """-> status[R]: 0 when every world of roadmap r reaches a final node, 1 otherwise, PorrtError.code 5 (PORRT_ERR_PANIC)
        where roadmap r's growth panics (its code in panic_code[r], its iteration in n_it[r]).  Raises PorrtError when the call as
        a whole fails (bad arguments, no map, overlapping goal masks, low >= up, too many roadmaps)."""
        self.fns._need()
        c = self.ctx
        R = len(self.seeds)
        status = np.zeros(R, np.int32)
        rc = c.lib.porrt_pto_grow_batch(c.h, R, _p(self.seeds), _p(_f64(start)), _p(self.low), _p(self.up), _p(goal.goals), _p(goal.masks),
                                        len(goal.goals), goal.max_dist, float(max_step), float(search_radius), int(n_iter_min),
                                        int(n_iter_max), _p(self.sizes), _p(status), _p(self.panic_code), _p(self.counters))
        self.n_it = self.sizes[:, 0].copy()
        c.check(rc)
        return status

    def _fetcher(self, r):
        def fetch(*outs):
            self.ctx.check(self.ctx.lib.porrt_pto_fetch_roadmap(self.ctx.h, int(r), *outs))
        return fetch

    def graph_arrays(self, r):
        """PTO.graph_arrays of roadmap r"""
        return _roadmap_graph_arrays(self._fetcher(r), self.sizes[r])

    def reach_masks(self, r):
        """PTO.reach_masks of roadmap r"""
        return _roadmap_reach_masks(self._fetcher(r), self.sizes[r], self.fns)

    def finals(self, r):
        """PTO.finals of roadmap r"""
        return _roadmap_finals(self._fetcher(r), self.sizes[r], self.fns)


class RRT:
    """src/rrt.rs RRT::grow_tree on the device (porrt_rrt_grow): `fns` is an uploaded Map / MapShelfDomain, the sampler is seeded
    with `seed`.  The tree stays on the device until tree() asks.  After grow_tree: n_it, sizes = (iterations, nodes, finals),
    counters = (windows, iterations re-speculated, conflicts by nearest neighbour, conflicts by radius / kd slot)."""

    def __init__(self, fns, low, up, seed=0):
        self.fns, self.ctx = fns, fns.ctx
        self.low, self.up, self.seed = _f64(low), _f64(up), int(seed)
        self.n_it, self.sizes, self.counters = 0, (0, 0, 0), (0, 0, 0, 0)

    def grow_tree(self, start, goal, max_step, search_radius, n_iter_min, n_iter_max):
        """-> 0 when the tree has a final node, 1 when it has none (rrt.rs: "No path found!"); PorrtError where a state or edge check
        panics (e.code == 5, e.panic_code = its code, n_it = its iteration)"""
        self.fns._need()
        c = self.ctx
        sizes, counters = np.zeros(3, np.int64), np.zeros(4, np.int64)
        status, panic = C.c_int32(), C.c_int32()
        rc = c.lib.porrt_rrt_grow(c.h, self.seed, _p(_f64(start)), _p(self.low), _p(self.up), _p(goal.goals), _p(goal.masks), len(goal.goals),
                                  goal.max_dist, float(max_step), float(search_radius), int(n_iter_min), int(n_iter_max), _p(sizes),
                                  C.byref(status), C.byref(panic), _p(counters))
        self.n_it, self.sizes, self.counters = int(sizes[0]), tuple(int(x) for x in sizes), tuple(int(x) for x in counters)
        if rc in (0, 5):
            c._rrt_trees = 1
        if rc:
            err = PorrtError(rc, (c.lib.porrt_last_error(c.h) or b"").decode())
            err.panic_code = panic.value
            raise err
        return int(status.value)

    def tree(self):
        """-> states[V, 2], parent[V] (-1 at the root), dist_from_root[V], final node ids in the order they were found"""
        return _fetch_tree(self.ctx, 0, self.sizes)

    def best_path(self):
        """get_best_solution + get_path_to (rrt.rs:183-193, :48-60) on the device: -> (path[L, 2] root first, cost) of the final
        with the smallest (cost, path length), or None when the tree has no final (porrt_rrt_best_paths)"""
        return _best_paths(self.ctx)[0]

    def plan(self, start, goal, max_step, search_radius, n_iter_min, n_iter_max):
        """rrt.rs:183-193 plan: grow_tree, then the best path -> (path[L, 2], cost), or None ("No path found!"); PorrtError where
        the growth panics"""
        self.grow_tree(start, goal, max_step, search_radius, n_iter_min, n_iter_max)
        return self.best_path()


class RRTBatch:
    """RRT::grow_tree for one tree per seed in `seeds`, all in one device call (porrt_rrt_grow_batch); map, start, goal and parameters
    are shared.  Tree t is what RRT(fns, low, up, seeds[t]) grows, counters included.  After grow_tree the attributes n_it[R],
    sizes[R, 3], counters[R, 4] and panic_code[R] hold one row per tree; tree(t) reads tree t.  The batch replaces the context's
    last RRT growth; PTO growth on the same context is kept apart."""

    def __init__(self, fns, low, up, seeds):
        self.fns, self.ctx = fns, fns.ctx
        self.low, self.up = _f64(low), _f64(up)
        self.seeds = np.ascontiguousarray(np.asarray(seeds, dtype=np.uint64).reshape(-1))
        R = len(self.seeds)
        self.n_it, self.panic_code = np.zeros(R, np.int64), np.zeros(R, np.int32)
        self.sizes, self.counters = np.zeros((R, 3), np.int64), np.zeros((R, 4), np.int64)

    def __len__(self):
        return len(self.seeds)

    def grow_tree(self, start, goal, max_step, search_radius, n_iter_min, n_iter_max):
        """-> status[R]: 0 when tree t has a final node, 1 when it has none, 5 (PORRT_ERR_PANIC) where its growth panics (its code in
        panic_code[t], its iteration in n_it[t]).  Raises PorrtError when the call as a whole fails (bad arguments, no map,
        overlapping goal masks, low >= up, too many trees)."""
        self.fns._need()
        c = self.ctx
        R = len(self.seeds)
        status = np.zeros(R, np.int32)
        rc = c.lib.porrt_rrt_grow_batch(c.h, R, _p(self.seeds), _p(_f64(start)), _p(self.low), _p(self.up), _p(goal.goals), _p(goal.masks),
                                        len(goal.goals), goal.max_dist, float(max_step), float(search_radius), int(n_iter_min),
                                        int(n_iter_max), _p(self.sizes), _p(status), _p(self.panic_code), _p(self.counters))
        self.n_it = self.sizes[:, 0].copy()
        c.check(rc)
        c._rrt_trees = R
        return status

    def grow_queries(self, starts, goals, max_step, search_radius, n_iter_min, n_iter_max):
        """grow_tree with one query per tree (porrt_rrt_grow_queries): tree t starts at starts[t] and heads for goals[t] (a
        SquareGoal) with sampler seed seeds[t]; tree t is what RRT(fns, low, up, seeds[t]).grow_tree(starts[t], goals[t], ...) grows,
        counters included.  -> status[R] as grow_tree; raises PorrtError when the call as a whole fails (grow_tree's errors, a start
        that is not finite, a negative or NaN max_dist, goal masks that overlap within one query)."""
        self.fns._need()
        c = self.ctx
        R = len(self.seeds)
        starts, goals = _f64(starts, 2), list(goals)
        if len(starts) != R or len(goals) != R:
            raise ValueError("one start and one goal per seed")
        ptr = np.zeros(R + 1, np.int64)
        ptr[1:] = np.cumsum([len(g.goals) for g in goals])
        gxy = np.ascontiguousarray(np.concatenate([g.goals for g in goals]))
        gmask = np.ascontiguousarray(np.concatenate([g.masks for g in goals]))
        gmd = np.array([g.max_dist for g in goals], np.float64)
        status = np.zeros(R, np.int32)
        rc = c.lib.porrt_rrt_grow_queries(c.h, R, _p(self.seeds), _p(starts), _p(self.low), _p(self.up), _p(ptr), _p(gxy), _p(gmask),
                                          _p(gmd), float(max_step), float(search_radius), int(n_iter_min), int(n_iter_max),
                                          _p(self.sizes), _p(status), _p(self.panic_code), _p(self.counters))
        self.n_it = self.sizes[:, 0].copy()
        c.check(rc)
        c._rrt_trees = R
        return status

    def tree(self, t):
        """RRT.tree of tree t"""
        return _fetch_tree(self.ctx, t, self.sizes[t])

    def best_paths(self):
        """RRT.best_path of every tree, in one device call: a list of (path[L, 2], cost) or None"""
        return _best_paths(self.ctx)


def _best_paths(ctx):
    """porrt_rrt_best_paths on the last RRT growth of ctx -> [(path[L, 2], cost) or None per tree]"""
    n = getattr(ctx, "_rrt_trees", 0)          # the trees of the context's last RRT growth (set by the growth calls)
    fin, cost, ptr, total = np.empty(max(n, 1), np.int32), np.empty(max(n, 1)), np.empty(n + 1, np.int64), C.c_int64()
    cap = 64 * n
    while True:
        xy = np.empty((max(cap, 1), 2))
        rc = ctx.lib.porrt_rrt_best_paths(ctx.h, _p(fin), _p(cost), _p(ptr), _p(xy), cap, C.byref(total))
        if rc == ERR_CAPACITY and total.value > cap:
            cap = total.value
            continue
        ctx.check(rc)
        return [None if fin[t] < 0 else (xy[ptr[t]:ptr[t + 1]].copy(), float(cost[t])) for t in range(n)]


def _fetch_tree(ctx, t, sizes):
    _, V, F = (int(x) for x in sizes)
    xy, parent, dist, finals = np.empty((V, 2)), np.empty(V, np.int32), np.empty(V), np.empty(F, np.int64)
    ctx.check(ctx.lib.porrt_rrt_fetch_tree(ctx.h, int(t), _p(xy), _p(parent), _p(dist), _p(finals)))
    return xy, parent, dist, finals


# the arrays of a device-grown roadmap; fetch(xy, node_vid, row_ptr, col, edge_vid, reach, final_ids, final_masks) is
# porrt_pto_fetch or porrt_pto_fetch_roadmap, sizes = (iterations, V, E, finals)
def _roadmap_graph_arrays(fetch, sizes):
    _, V, E, _ = (int(x) for x in sizes)
    xy, nv = np.empty((V, 2)), np.empty(V, np.int32)
    rp, col, ev = np.empty(V + 1, np.int64), np.empty(E, np.int32), np.empty(E, np.int32)
    fetch(_p(xy), _p(nv), _p(rp), _p(col), _p(ev), None, None, None)
    return xy, nv, rp, col, ev


def _roadmap_reach_masks(fetch, sizes, fns):
    V = int(sizes[1])
    nw = fns.n_worlds()
    words = np.empty((V, fns.mask_words), np.uint64)
    fetch(None, None, None, None, None, _p(words), None, None)
    bits = np.zeros((V, nw), np.uint8)
    for w in range(nw):
        bits[:, w] = (words[:, w // 64] >> np.uint64(w % 64)) & np.uint64(1)
    return bits


def _roadmap_finals(fetch, sizes, fns):
    F = int(sizes[3])
    ids, masks = np.empty(F, np.int64), np.empty((F, fns.mask_words), np.uint64)
    fetch(None, None, None, None, None, None, _p(ids), _p(masks))
    return ids, masks


def react_qmdp(ctx, row_ptr, col, xy, cost_to_goals, start_node, belief, common_horizon):
    """QMdpPolicyExtractor::react_qmdp (qmdp_policy_extractor.rs:38-123) over plan_qmdp's cost table -> (paths as lists of
    node ids, one per world; length of the common prefix).  ctx may be None (host walk)."""
    lib = _lib.load()
    row_ptr = np.ascontiguousarray(row_ptr, np.int64)
    col = np.ascontiguousarray(col, np.int32)
    xy = _f64(xy, 2)
    cost = np.ascontiguousarray(cost_to_goals, np.float64)
    W, V = cost.shape
    b = _f64(belief)
    ptr = np.empty(W + 1, np.int64)
    total, n_common = C.c_int64(), C.c_int64()
    cap = 1024
    h = ctx.h if ctx is not None else None
    while True:
        nodes = np.empty(cap, np.int32)
        rc = lib.porrt_qmdp_react(h, V, _p(row_ptr), _p(col), _p(xy), W, _p(cost), int(start_node), _p(b), len(b), float(common_horizon),
                                  _p(ptr), _p(nodes), cap, C.byref(total), C.byref(n_common))
        if rc == ERR_CAPACITY:
            cap = total.value
            continue
        if rc:
            raise PorrtError(rc, (lib.porrt_last_error(h) or b"").decode() if h else "porrt_qmdp_react")
        return [nodes[ptr[w]:ptr[w + 1]].copy() for w in range(W)], n_common.value
