"""ctypes driver for oracle/liboracle.so -- TEST INFRASTRUCTURE, NOT PRODUCT CODE.

Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference legs import this.
The oracle is a CPU restatement of the po-rrt hot path (see porrt_oracle.hpp for the parity status).
"""
import ctypes as C
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB = None

vp, i32, i64, u32, u64, f64 = C.c_void_p, C.c_int32, C.c_int64, C.c_uint32, C.c_uint64, C.c_double

_SIGS = {
    # name: (restype, argtypes)
    "orc_norm1": (f64, [vp, vp]), "orc_norm2": (f64, [vp, vp]), "orc_steer": (None, [vp, vp, f64]),
    "orc_heuristic_radius": (f64, [u64, f64, f64, u64]),
    "orc_transition_probability": (f64, [vp, vp, u64]), "orc_belief_hash": (u64, [vp, u64]),
    "orc_is_compatible": (C.c_int, [vp, vp, u64]), "orc_num_threads": (C.c_int, []),
    "orc_pcg_seed_from_u64": (vp, [u64]), "orc_pcg_new": (vp, [u64, u64, u64, u64]), "orc_pcg_free": (None, [vp]),
    "orc_pcg_next_u64": (u64, [vp]), "orc_pcg_gen_range_f64": (f64, [vp, f64, f64]),
    "orc_pcg_gen_range_usize": (u64, [vp, u64]), "orc_pcg_fill_f64": (None, [vp, f64, f64, vp, u64]),
    "orc_pcg_fill_u64": (None, [vp, vp, u64]), "orc_sampler_fill": (None, [vp, vp, vp, vp, u64]),
    "orc_bresenham": (i64, [i32, i32, i32, i32, vp, i64]),
    "orc_map_create": (vp, [vp, vp, u32, u32, vp, vp, C.c_int, f64]), "orc_map_free": (None, [vp]),
    "orc_map_info": (None, [vp, vp, vp, vp, vp]), "orc_map_zone_positions": (None, [vp, vp]),
    "orc_map_world_validities": (None, [vp, vp]), "orc_map_to_pixel": (None, [vp, vp, vp]),
    "orc_map_to_coordinates": (None, [vp, vp, vp]),
    "orc_state_validity_batch": (None, [vp, vp, i64, vp]), "orc_edge_validity_batch": (None, [vp, vp, vp, i64, vp]),
    "orc_edge_validity_timed": (f64, [vp, vp, vp, i64, vp, C.c_int]),
    "orc_edge_pixel_counts": (None, [vp, vp, vp, i64, vp]),
    "orc_visible_zones_batch": (C.c_int, [vp, vp, i64, vp, vp]),
    "orc_observe": (i64, [vp, vp, vp, vp, i64]), "orc_reachable_belief_states": (i64, [vp, vp, vp, i64]),
    "orc_successor_beliefs": (i64, [vp, vp, u64, vp]),
    "orc_kd_new": (vp, [vp, u64]), "orc_kd_free": (None, [vp]), "orc_kd_add": (None, [vp, vp, u64]),
    "orc_kd_add_batch": (None, [vp, vp, u64, u64]), "orc_kd_size": (u64, [vp]),
    "orc_kd_export": (None, [vp, vp, vp, vp, vp]), "orc_kd_nearest": (u64, [vp, vp, vp, u64]),
    "orc_kd_nearest_batch": (None, [vp, vp, i64, vp, vp, vp, C.c_int]),
    "orc_kd_radius": (i64, [vp, vp, f64, vp, i64]),
    "orc_kd_radius_batch": (i64, [vp, vp, vp, i64, vp, vp, i64, C.c_int]),
    "orc_graph_new": (vp, [vp, u64, u64]), "orc_graph_free": (None, [vp]),
    "orc_graph_add_node": (u64, [vp, vp, u64]), "orc_graph_add_edge": (None, [vp, u64, u64, u64]),
    "orc_graph_add_bi_edge": (None, [vp, u64, u64, u64]), "orc_graph_n_nodes": (u64, [vp]),
    "orc_graph_n_edges": (u64, [vp]), "orc_graph_export": (None, [vp, C.c_int, vp, vp, vp, vp, vp]),
    "orc_dijkstra": (None, [vp, C.c_int, vp, u64, vp]), "orc_extract_path": (i64, [vp, C.c_int, u64, vp, vp, i64]),
    "orc_default_transition_validator": (i64, [vp, u64, u64, u64, u64]),
    "orc_reach_new": (vp, []), "orc_reach_free": (None, [vp]), "orc_reach_set_root": (None, [vp, vp, u64]),
    "orc_reach_add_node": (None, [vp, vp, u64]), "orc_reach_add_final_node": (None, [vp, u64, vp, u64]),
    "orc_reach_add_edge": (None, [vp, u64, u64, vp, u64]), "orc_reach_get": (None, [vp, u64, vp]),
    "orc_reach_is_final_set_complete": (C.c_int, [vp]), "orc_reach_final_nodes_for_world": (i64, [vp, u64, vp, i64]),
    "orc_reach_n_finals": (i64, [vp]), "orc_reach_finals": (None, [vp, vp, vp]), "orc_reach_all": (None, [vp, vp]),
    "orc_goal_new": (vp, [vp, vp, u64, u64, f64]), "orc_goal_free": (None, [vp]),
    "orc_goal_goal": (C.c_int, [vp, vp, vp]), "orc_goal_example": (None, [vp, u64, vp]),
    "orc_bg_new": (vp, [vp, u64, u64]), "orc_bg_free": (None, [vp]), "orc_bg_add_node": (u64, [vp, vp, u64, C.c_int]),
    "orc_bg_add_edge": (None, [vp, u64, u64]), "orc_bg_n_nodes": (u64, [vp]), "orc_bg_n_edges": (u64, [vp]),
    "orc_bg_export": (None, [vp, vp, vp, vp, vp]), "orc_conditional_dijkstra": (C.c_int, [vp, vp, u64, vp]),
    "orc_extract_policy": (vp, [vp, vp]), "orc_policy_free": (None, [vp]),
    "orc_policy_sizes": (None, [vp, vp, vp, vp]), "orc_policy_export": (None, [vp, vp, vp, vp, vp, vp]),
    "orc_prm_new": (vp, [vp, vp, vp, u64]), "orc_prm_free": (None, [vp]), "orc_prm_init": (None, [vp, vp]),
    "orc_prm_grow_graph": (f64, [vp, f64, f64, u64]), "orc_prm_add_sample": (u64, [vp, vp, f64, f64]),
    "orc_prm_add_samples": (f64, [vp, vp, u64, f64, f64]), "orc_prm_graph": (vp, [vp]), "orc_prm_kdtree": (vp, [vp]), "orc_prm_plan_path": (i64, [vp, vp, vp, vp, i64]),
    "orc_pto_new": (vp, [vp, vp, vp, u64]), "orc_pto_free": (None, [vp]),
    "orc_pto_grow_graph": (C.c_int, [vp, vp, vp, f64, f64, u64, u64]),
    "orc_pto_set_hooks": (None, [vp, vp, vp, vp, vp, vp]),
    "orc_pto_graph": (vp, [vp]), "orc_pto_kdtree": (vp, [vp]), "orc_pto_reach": (vp, [vp]),
    "orc_pto_belief_graph": (vp, [vp]), "orc_pto_n_it": (u64, [vp]), "orc_pto_set_n_worlds": (None, [vp, u64]),
    "orc_pto_set_validities": (None, [vp, vp, u64, u64]), "orc_pto_build_belief_graph": (C.c_int, [vp, vp, u64]),
    "orc_pto_n_beliefs": (i64, [vp]), "orc_pto_beliefs": (None, [vp, vp]),
    "orc_pto_compute_expected_costs": (C.c_int, [vp, vp]), "orc_pto_final_belief_nodes": (i64, [vp, vp, i64]),
    "orc_pto_extract_policy": (vp, [vp]), "orc_pto_plan_qmdp": (C.c_int, [vp, vp]), "orc_pto_refine_shortcut": (vp, [vp, C.c_uint64, C.c_uint64]), "orc_pto_refine_reparent": (vp, [vp, f64]), "orc_policy_decompose_count": (i64, [vp, u64]),
    "orc_policy_expected_cost": (f64, [vp, vp, vp, u64, vp, u64, u64]),
    "orc_pto_react_qmdp": (i64, [vp, vp, vp, f64, vp, vp, i64]),
    "orc_refiner_transition_valid_batch": (None, [vp, vp, vp, i64, vp, u64, vp]),
    "orc_refiner_partial_shortcut": (i64, [vp, vp, u64, vp, u64, u64, u64]),
    "orc_tamp_new": (vp, [vp, vp, vp, u64]), "orc_tamp_free": (None, [vp]),
    "orc_tamp_plan": (C.c_int, [vp, vp, vp, u64, f64, f64, u64, vp]), "orc_tamp_belief_graph": (vp, [vp]),
    "orc_tamp_policy": (vp, [vp]), "orc_tamp_sizes": (None, [vp, vp]),
    "orc_tamp_export": (None, [vp] * 14),
}


def build(force=False):
    """Compile oracle/liboracle.so with the committed Makefile (g++ only; seconds)."""
    so = os.path.join(_HERE, "liboracle.so")
    if force or not os.path.exists(so) or any(
            os.path.getmtime(os.path.join(_HERE, f)) > os.path.getmtime(so)
            for f in ("porrt_oracle.cpp", "oracle_c.cpp", "porrt_oracle.hpp", "Makefile")):
        subprocess.run(["make", "-C", _HERE], check=True, capture_output=True)
    return so


def lib():
    global _LIB
    if _LIB is None:
        so = build()
        _LIB = C.CDLL(so)
        for name, (res, args) in _SIGS.items():
            fn = getattr(_LIB, name)
            fn.restype = res
            fn.argtypes = args
    return _LIB


def P(a):
    """pointer to a C-contiguous numpy array (or None)"""
    if a is None:
        return None
    assert a.flags["C_CONTIGUOUS"]
    return a.ctypes.data_as(C.c_void_p)


def f64a(x):
    return np.ascontiguousarray(np.asarray(x, dtype=np.float64))


def masks_to_bytes(masks):
    return np.ascontiguousarray(np.asarray(masks, dtype=np.uint8))


NONE, PANIC_OOB, PANIC_ZONE_UNWRAP, PANIC_MULTI_ZONE = -1, -2, -3, -4
DOOR, SHELF = 0, 1
UNKNOWN, ACTION, OBSERVATION = 0, 1, 2


class Pcg64:
    def __init__(self, seed=0, handle=None):
        self.h = handle if handle is not None else lib().orc_pcg_seed_from_u64(seed)

    @classmethod
    def new(cls, state, stream):
        m = (1 << 64) - 1
        return cls(handle=lib().orc_pcg_new(state >> 64, state & m, stream >> 64, stream & m))

    def __del__(self):
        if getattr(self, "h", None):
            lib().orc_pcg_free(self.h)
            self.h = None

    def next_u64(self):
        return lib().orc_pcg_next_u64(self.h)

    def gen_range_f64(self, lo, hi):
        return lib().orc_pcg_gen_range_f64(self.h, lo, hi)

    def gen_range_usize(self, n):
        return lib().orc_pcg_gen_range_usize(self.h, n)

    def fill_f64(self, lo, hi, n):
        out = np.empty(n, np.float64)
        lib().orc_pcg_fill_f64(self.h, lo, hi, P(out), n)
        return out

    def fill_u64(self, n):
        out = np.empty(n, np.uint64)
        lib().orc_pcg_fill_u64(self.h, P(out), n)
        return out

    def sample_states(self, low, up, n):
        """ContinuousSampler::sample() n times (sample_space.rs:30-37) -> [n,2]"""
        out = np.empty((n, 2), np.float64)
        lib().orc_sampler_fill(self.h, P(f64a(low)), P(f64a(up)), P(out), n)
        return out


def bresenham(a, b):
    cap = max(abs(a[0] - b[0]), abs(a[1] - b[1])) + 2
    out = np.empty((cap, 2), np.int32)
    n = lib().orc_bresenham(a[0], a[1], b[0], b[1], P(out), cap)
    return out[:n]


class GridMap:
    """Map (kind=DOOR, map_io.rs) / MapShelfDomain (kind=SHELF, map_shelves_io.rs)."""

    def __init__(self, occ, zones, low, up, kind, visibility=0.0):
        occ = np.ascontiguousarray(occ, dtype=np.uint8)
        self.H, self.W = occ.shape
        z = None if zones is None else np.ascontiguousarray(zones, dtype=np.uint8)
        self.h = lib().orc_map_create(P(occ), P(z), self.H, self.W, P(f64a(low)), P(f64a(up)), kind, visibility)
        if not self.h:
            raise ValueError("reference would panic while building this map")
        nz, nw, nv, ppm = i64(), i64(), i64(), f64()
        lib().orc_map_info(self.h, C.byref(nz), C.byref(nw), C.byref(nv), C.byref(ppm))
        self.n_zones, self.n_worlds, self.n_validities, self.ppm = nz.value, nw.value, nv.value, ppm.value
        self.kind = kind

    def __del__(self):
        if getattr(self, "h", None):
            lib().orc_map_free(self.h)
            self.h = None

    def zone_positions(self):
        out = np.empty((self.n_zones, 2), np.float64)
        lib().orc_map_zone_positions(self.h, P(out))
        return out

    def world_validities(self):
        out = np.empty((self.n_validities, self.n_worlds), np.uint8)
        lib().orc_map_world_validities(self.h, P(out))
        return out

    def to_pixel(self, xy):
        ij = np.empty(2, np.uint32)
        lib().orc_map_to_pixel(self.h, P(f64a(xy)), P(ij))
        return ij

    def to_coordinates(self, ij):
        xy = np.empty(2, np.float64)
        lib().orc_map_to_coordinates(self.h, P(np.asarray(ij, np.uint32)), P(xy))
        return xy

    def state_validity(self, xy):
        xy = f64a(xy).reshape(-1, 2)
        out = np.empty(len(xy), np.int64)
        lib().orc_state_validity_batch(self.h, P(xy), len(xy), P(out))
        return out

    def edge_validity(self, frm, to):
        frm, to = f64a(frm).reshape(-1, 2), f64a(to).reshape(-1, 2)
        out = np.empty(len(frm), np.int64)
        lib().orc_edge_validity_batch(self.h, P(frm), P(to), len(frm), P(out))
        return out

    def edge_validity_timed(self, frm, to, threads):
        out = np.empty(len(frm), np.int64)
        t = lib().orc_edge_validity_timed(self.h, P(frm), P(to), len(frm), P(out), threads)
        return out, t

    def edge_pixel_count(self, frm, to):
        tot = i64()
        lib().orc_edge_pixel_counts(self.h, P(f64a(frm)), P(f64a(to)), len(frm), C.byref(tot))
        return tot.value

    def refiner_transition_valid(self, frm, to, compat_row):
        """pto_policy_refiner.rs:395-423 is_transition_valid, batched: 1 / 0 / negative panic code"""
        frm, to = f64a(frm), f64a(to)
        row = np.ascontiguousarray(np.asarray(compat_row, dtype=np.uint8))
        out = np.empty(len(frm), np.int64)
        lib().orc_refiner_transition_valid_batch(self.h, P(frm), P(to), len(frm), P(row), len(row), P(out))
        return out

    def refiner_partial_shortcut(self, states, compat_row, n_iterations, seed=0):
        """pto_policy_refiner.rs:158-206 partial_shortcut on one path piece -> (new states, commits or panic code); the trials are
        drawn from DiscreteSampler(seed) (the reference's DiscreteSampler::new() is seed 0)"""
        st = f64a(states).copy()
        row = np.ascontiguousarray(np.asarray(compat_row, dtype=np.uint8))
        rc = lib().orc_refiner_partial_shortcut(self.h, P(st), len(st), P(row), len(row), int(n_iterations), int(seed))
        return st, int(rc)

    def visible_zones(self, xy):
        xy = f64a(xy).reshape(-1, 2)
        mask = np.empty(len(xy), np.uint64)
        panic = np.empty(len(xy), np.int64)
        lib().orc_visible_zones_batch(self.h, P(xy), len(xy), P(mask), P(panic))
        return mask, panic

    def observe(self, xy, belief):
        cap = 1 << min(self.n_zones, 12)
        out = np.empty((cap, self.n_worlds), np.float64)
        n = lib().orc_observe(self.h, P(f64a(xy)), P(f64a(belief)), P(out), cap)
        if n < 0:
            raise RuntimeError("panic %d" % n)
        return out[:n].copy()

    def reachable_belief_states(self, b0, cap=1 << 16):
        out = np.empty((cap, self.n_worlds), np.float64)
        n = lib().orc_reachable_belief_states(self.h, P(f64a(b0)), P(out), cap)
        assert n <= cap
        return out[:n].copy()

    def successor_beliefs(self, b, zone):
        out = np.empty((2, self.n_worlds), np.float64)
        n = lib().orc_successor_beliefs(self.h, P(f64a(b)), zone, P(out))
        return out[:n].copy()


class KdTree:
    def __init__(self, state, id=0, handle=None, owner=None):
        self._owner = owner
        self.h = handle if handle is not None else lib().orc_kd_new(P(f64a(state)), id)

    def __del__(self):
        if getattr(self, "h", None) and self._owner is None:
            lib().orc_kd_free(self.h)
        self.h = None

    def add(self, state, id):
        lib().orc_kd_add(self.h, P(f64a(state)), id)

    def add_batch(self, xy, first_id):
        xy = f64a(xy).reshape(-1, 2)
        lib().orc_kd_add_batch(self.h, P(xy), first_id, len(xy))

    def size(self):
        return lib().orc_kd_size(self.h)

    def export(self):
        n = self.size()
        ids, left, right, xy = np.empty(n, np.int64), np.empty(n, np.int32), np.empty(n, np.int32), np.empty((n, 2))
        lib().orc_kd_export(self.h, P(ids), P(left), P(right), P(xy))
        return ids, left, right, xy

    def nearest_neighbor(self, q, excluded=()):
        ex = np.asarray(list(excluded), np.uint64)
        return lib().orc_kd_nearest(self.h, P(f64a(q)), P(ex) if len(ex) else None, len(ex))

    def nearest_batch(self, q, reach_masks=None, world=None, threads=1):
        q = f64a(q).reshape(-1, 2)
        out = np.empty(len(q), np.int64)
        rm = None if reach_masks is None else np.ascontiguousarray(reach_masks, np.uint64)
        w = None if world is None else np.ascontiguousarray(world, np.uint32)
        lib().orc_kd_nearest_batch(self.h, P(q), len(q), P(rm), P(w), P(out), threads)
        return out

    def nearest_neighbors(self, q, radius):
        cap = self.size()
        out = np.empty(cap, np.int64)
        n = lib().orc_kd_radius(self.h, P(f64a(q)), radius, P(out), cap)
        return out[:n].copy()

    def radius_batch(self, q, radius, cap, threads=1):
        q = f64a(q).reshape(-1, 2)
        r = f64a(np.broadcast_to(radius, (len(q),)))
        offs = np.empty(len(q) + 1, np.int64)
        ids = np.empty(cap, np.int64)
        tot = lib().orc_kd_radius_batch(self.h, P(q), P(r), len(q), P(offs), P(ids), cap, threads)
        return offs, ids[:min(tot, cap)], tot


class PTOGraph:
    def __init__(self, validities=None, handle=None, owner=None):
        self._owner = owner
        if handle is not None:
            self.h = handle
        else:
            v = masks_to_bytes(validities)
            self.h = lib().orc_graph_new(P(v), v.shape[0], v.shape[1])

    def __del__(self):
        if getattr(self, "h", None) and self._owner is None:
            lib().orc_graph_free(self.h)
        self.h = None

    def add_node(self, s, vid):
        return lib().orc_graph_add_node(self.h, P(f64a(s)), vid)

    def add_edge(self, a, b, vid):
        lib().orc_graph_add_edge(self.h, a, b, vid)

    def add_bi_edge(self, a, b, vid):
        lib().orc_graph_add_bi_edge(self.h, a, b, vid)

    def n_nodes(self):
        return lib().orc_graph_n_nodes(self.h)

    def n_edges(self):
        return lib().orc_graph_n_edges(self.h)

    def export(self, which=0):
        """-> xy[V,2], node_vid[V], row_ptr[V+1], col[E], edge_vid[E] (children if which==0 else parents)"""
        V, E = self.n_nodes(), self.n_edges()
        xy, nv = np.empty((V, 2)), np.empty(V, np.int32)
        rp, col, ev = np.empty(V + 1, np.int64), np.empty(E, np.int32), np.empty(E, np.int32)
        lib().orc_graph_export(self.h, which, P(xy), P(nv), P(rp), P(col), P(ev))
        return xy, nv, rp, col, ev

    def dijkstra(self, finals, world=-1):
        f = np.asarray(list(finals), np.uint64)
        out = np.empty(self.n_nodes(), np.float64)
        lib().orc_dijkstra(self.h, world, P(f) if len(f) else None, len(f), P(out))
        return out

    def extract_path(self, start, costs, world=-1):
        cap = self.n_nodes() + 1
        out = np.empty((cap, 2))
        n = lib().orc_extract_path(self.h, world, start, P(f64a(costs)), P(out), cap)
        return out[:n].copy()


def default_transition_validator(validities, from_vid, to_vid):
    v = masks_to_bytes(validities)
    return lib().orc_default_transition_validator(P(v), v.shape[0], v.shape[1], from_vid, to_vid)


class Reachability:
    def __init__(self, handle=None, owner=None, n_worlds=None):
        self._owner = owner
        self.h = handle if handle is not None else lib().orc_reach_new()
        self.n_worlds = n_worlds

    def __del__(self):
        if getattr(self, "h", None) and self._owner is None:
            lib().orc_reach_free(self.h)
        self.h = None

    def set_root(self, m):
        m = masks_to_bytes(m)
        self.n_worlds = len(m)
        lib().orc_reach_set_root(self.h, P(m), len(m))

    def add_node(self, m):
        m = masks_to_bytes(m)
        lib().orc_reach_add_node(self.h, P(m), len(m))

    def add_final_node(self, id, m):
        m = masks_to_bytes(m)
        lib().orc_reach_add_final_node(self.h, id, P(m), len(m))

    def add_edge(self, a, b, m):
        m = masks_to_bytes(m)
        lib().orc_reach_add_edge(self.h, a, b, P(m), len(m))

    def reachability(self, id):
        out = np.empty(self.n_worlds, np.uint8)
        lib().orc_reach_get(self.h, id, P(out))
        return out

    def all(self, n_nodes):
        out = np.empty((n_nodes, self.n_worlds), np.uint8)
        lib().orc_reach_all(self.h, P(out))
        return out

    def is_final_set_complete(self):
        return bool(lib().orc_reach_is_final_set_complete(self.h))

    def get_final_nodes_for_world(self, w):
        cap = max(1, lib().orc_reach_n_finals(self.h))
        out = np.empty(cap, np.uint64)
        n = lib().orc_reach_final_nodes_for_world(self.h, w, P(out), cap)
        return [int(x) for x in out[:n]]

    def finals(self):
        n = lib().orc_reach_n_finals(self.h)
        ids = np.empty(n, np.uint64)
        fin = np.empty((n, self.n_worlds), np.uint8)
        lib().orc_reach_finals(self.h, P(ids), P(fin))
        return ids.astype(np.int64), fin


class SquareGoal:
    def __init__(self, goal_to_validity, max_dist):
        xy = f64a([g for g, _ in goal_to_validity])
        masks = masks_to_bytes([m for _, m in goal_to_validity])
        self.n_worlds = masks.shape[1]
        self.goals, self.masks, self.max_dist = xy, masks, max_dist
        self.h = lib().orc_goal_new(P(xy), P(masks), len(xy), self.n_worlds, max_dist)
        if not self.h:
            raise ValueError("SquareGoal::new would panic")

    def __del__(self):
        if getattr(self, "h", None):
            lib().orc_goal_free(self.h)
            self.h = None

    def goal(self, s):
        out = np.empty(self.n_worlds, np.uint8)
        return out if lib().orc_goal_goal(self.h, P(f64a(s)), P(out)) else None

    def goal_example(self, w):
        out = np.empty(2)
        lib().orc_goal_example(self.h, w, P(out))
        return out


class Policy:
    def __init__(self, handle):
        n, nl, e = i64(), i64(), f64()
        lib().orc_policy_sizes(handle, C.byref(n), C.byref(nl), C.byref(e))
        self.expected_costs = e.value
        self.xy = np.empty((n.value, 2))
        self.belief_id, self.parent, self.original = (np.empty(n.value, np.int64) for _ in range(3))
        self.leafs = np.empty(nl.value, np.int64)
        lib().orc_policy_export(handle, P(self.xy), P(self.belief_id), P(self.parent), P(self.original), P(self.leafs))
        lib().orc_policy_free(handle)

    def path_to_leaf(self, k):
        """Policy::path_to_leaf (common.rs:70-83)"""
        node, path = int(self.leafs[k]), []
        while node >= 0:
            path.append(tuple(self.xy[node]))
            node = int(self.parent[node])
        return path[::-1]


class BeliefGraph:
    def __init__(self, beliefs=None, handle=None, owner=None):
        self._owner = owner
        if handle is not None:
            self.h = handle
        else:
            b = f64a(beliefs)
            self.h = lib().orc_bg_new(P(b), b.shape[0], b.shape[1])

    def __del__(self):
        if getattr(self, "h", None) and self._owner is None:
            lib().orc_bg_free(self.h)
        self.h = None

    def add_node(self, s, belief_id, node_type):
        return lib().orc_bg_add_node(self.h, P(f64a(s)), belief_id, node_type)

    def add_edge(self, a, b):
        lib().orc_bg_add_edge(self.h, a, b)

    def n_nodes(self):
        return lib().orc_bg_n_nodes(self.h)

    def export(self):
        n, e = self.n_nodes(), lib().orc_bg_n_edges(self.h)
        typ, bid, rp, col = np.empty(n, np.int32), np.empty(n, np.int32), np.empty(n + 1, np.int64), np.empty(e, np.int64)
        lib().orc_bg_export(self.h, P(typ), P(bid), P(rp), P(col))
        return typ, bid, rp, col

    def conditional_dijkstra(self, finals):
        f = np.asarray(list(finals), np.uint64)
        out = np.empty(self.n_nodes())
        if not lib().orc_conditional_dijkstra(self.h, P(f) if len(f) else None, len(f), P(out)):
            raise RuntimeError("reference panic in conditional_dijkstra")
        return out

    def extract_policy(self, costs):
        h = lib().orc_extract_policy(self.h, P(f64a(costs)))
        if not h:
            raise RuntimeError("reference panic in extract_policy")
        return Policy(h)


class PRM:
    def __init__(self, gridmap, low, up, seed=0):
        self.map = gridmap
        self.h = lib().orc_prm_new(gridmap.h, P(f64a(low)), P(f64a(up)), seed)
        self.graph = PTOGraph(handle=lib().orc_prm_graph(self.h), owner=self)
        self.kdtree = KdTree(None, handle=lib().orc_prm_kdtree(self.h), owner=self)

    def __del__(self):
        if getattr(self, "h", None):
            lib().orc_prm_free(self.h)
            self.h = None

    def init(self, start):
        lib().orc_prm_init(self.h, P(f64a(start)))

    def grow_graph(self, max_step, search_radius, n_iter):
        """returns wall seconds"""
        return lib().orc_prm_grow_graph(self.h, max_step, search_radius, n_iter)

    def add_sample(self, s, max_step, search_radius):
        return lib().orc_prm_add_sample(self.h, P(f64a(s)), max_step, search_radius)

    def add_samples(self, xy, max_step, search_radius):
        """PRM::add_sample for each row of xy; returns wall seconds"""
        xy = f64a(xy).reshape(-1, 2)
        return lib().orc_prm_add_samples(self.h, P(xy), len(xy), max_step, search_radius)

    def plan_path(self, start, goal):
        cap = self.graph.n_nodes() + 1
        out = np.empty((cap, 2))
        n = lib().orc_prm_plan_path(self.h, P(f64a(start)), P(f64a(goal)), P(out), cap)
        return out[:n].copy()


class PTO:
    def __init__(self, gridmap, low, up, seed=0):
        self.map = gridmap
        self.h = lib().orc_pto_new(gridmap.h, P(f64a(low)), P(f64a(up)), seed)
        self.graph = PTOGraph(handle=lib().orc_pto_graph(self.h), owner=self)
        self.kdtree = KdTree(None, handle=lib().orc_pto_kdtree(self.h), owner=self)
        self.reach = Reachability(handle=lib().orc_pto_reach(self.h), owner=self, n_worlds=gridmap.n_worlds)
        self.belief_graph = BeliefGraph(handle=lib().orc_pto_belief_graph(self.h), owner=self)
        self.n_worlds = gridmap.n_worlds

    def __del__(self):
        if getattr(self, "h", None):
            lib().orc_pto_free(self.h)
            self.h = None

    def grow_graph(self, start, goal, max_step, search_radius, n_iter_min, n_iter_max):
        return lib().orc_pto_grow_graph(self.h, P(f64a(start)), goal.h, max_step, search_radius, n_iter_min, n_iter_max)

    # per-query hooks (PTOHooks in porrt_oracle.hpp): the growth runs as the caller of `backend`, an object with
    # nearest_filtered(q, world, reach_words[V, words]) -> id, radius(q, r) -> ids in kd pre-order, state_validity(q) -> id,
    # edges(from[n,2], to[n,2]) -> ids[n], add_vertex(q, id)
    HOOK_TYPES = (C.CFUNCTYPE(i64, vp, C.POINTER(f64), u64, C.POINTER(u64), u64, u64),
                  C.CFUNCTYPE(i64, vp, C.POINTER(f64), f64, C.POINTER(i64), i64),
                  C.CFUNCTYPE(i64, vp, C.POINTER(f64)),
                  C.CFUNCTYPE(None, vp, C.POINTER(f64), C.POINTER(f64), i64, C.POINTER(i64)),
                  C.CFUNCTYPE(None, vp, C.POINTER(f64), u64))

    def set_hooks(self, backend):
        def nearest(_u, q, world, reach, n_nodes, words):
            rw = np.ctypeslib.as_array(reach, shape=(n_nodes, words)).copy()
            return int(backend.nearest_filtered([q[0], q[1]], int(world), rw))

        def radius(_u, q, r, out, cap):
            ids = backend.radius([q[0], q[1]], float(r))
            assert len(ids) <= cap
            for k, v in enumerate(ids):
                out[k] = int(v)
            return len(ids)

        def state(_u, q):
            return int(backend.state_validity([q[0], q[1]]))

        def edges(_u, fr, to, n, out):
            f = np.ctypeslib.as_array(fr, shape=(n, 2)).copy()
            t = np.ctypeslib.as_array(to, shape=(n, 2)).copy()
            for k, v in enumerate(backend.edges(f, t)):
                out[k] = int(v)

        def add_vertex(_u, q, node_id):
            backend.add_vertex([q[0], q[1]], int(node_id))
        self._hooks = [T(f) for T, f in zip(self.HOOK_TYPES, (nearest, radius, state, edges, add_vertex))]   # keep them alive
        lib().orc_pto_set_hooks(self.h, *(C.cast(h, vp) for h in self._hooks))

    def n_it(self):
        return lib().orc_pto_n_it(self.h)

    def set_mock(self, n_worlds, validities):
        v = masks_to_bytes(validities)
        lib().orc_pto_set_n_worlds(self.h, n_worlds)
        lib().orc_pto_set_validities(self.h, P(v), v.shape[0], v.shape[1])
        self.n_worlds = n_worlds
        self.reach.n_worlds = n_worlds

    def build_belief_graph(self, b0):
        b0 = f64a(b0)
        if not lib().orc_pto_build_belief_graph(self.h, P(b0), len(b0)):
            raise RuntimeError("reference panic in build_belief_graph")
        self.belief_graph = BeliefGraph(handle=lib().orc_pto_belief_graph(self.h), owner=self)

    def beliefs(self):
        out = np.empty((lib().orc_pto_n_beliefs(self.h), self.n_worlds))
        lib().orc_pto_beliefs(self.h, P(out))
        return out

    def compute_expected_costs_to_goals(self):
        out = np.empty(self.belief_graph.n_nodes())
        if not lib().orc_pto_compute_expected_costs(self.h, P(out)):
            raise RuntimeError("reference panic in conditional_dijkstra")
        return out

    def final_belief_nodes(self):
        cap = max(1, self.belief_graph.n_nodes())
        out = np.empty(cap, np.uint64)
        n = lib().orc_pto_final_belief_nodes(self.h, P(out), cap)
        return out[:n].astype(np.int64)

    def extract_policy(self):
        h = lib().orc_pto_extract_policy(self.h)
        if not h:
            raise RuntimeError("reference panic in extract_policy")
        return Policy(h)

    def refine_policy_shortcut(self, n_iterations, seed=0):
        """PTOPolicyRefiner::refine_solution(RefinmentStrategy::PartialShortCut(n)) on extract_policy()'s result; every piece's
        trials come from DiscreteSampler(seed) (the reference's is seed 0)"""
        h = lib().orc_pto_refine_shortcut(self.h, n_iterations, int(seed))
        if not h:
            raise RuntimeError("reference panic in refine_solution")
        return Policy(h)

    def refine_policy_reparent(self, radius):
        """PTOPolicyRefiner::refine_solution(RefinmentStrategy::Reparent(radius)) on extract_policy()'s result"""
        h = lib().orc_pto_refine_reparent(self.h, radius)
        if not h:
            raise RuntimeError("reference panic in refine_solution")
        return Policy(h)

    def plan_qmdp(self):
        out = np.empty((self.n_worlds, self.graph.n_nodes()))
        rc = lib().orc_pto_plan_qmdp(self.h, P(out))
        if rc:
            raise RuntimeError("We should have final node ids for each world")
        return out

    def react_qmdp(self, start, belief, horizon):
        cap = (self.graph.n_nodes() + 2) * self.n_worlds * 2
        lengths = np.empty(self.n_worlds, np.int64)
        xy = np.empty((cap, 2))
        tot = lib().orc_pto_react_qmdp(self.h, P(f64a(start)), P(f64a(belief)), horizon, P(lengths), P(xy), cap)
        if tot < 0:
            raise RuntimeError("react_qmdp failed")
        out, o = [], 0
        for n in lengths:
            out.append(xy[o:o + n].copy())
            o += n
        return out


class TampPRM:
    """MapShelfDomainTampPRM (map_shelves_tamp_prm.rs): plan() runs the reference algorithm; schedule() returns the recorded
    add_sample calls per mode + mode transitions (everything the RNG streams decided) and the expected costs."""

    def __init__(self, gridmap, low, up, seed=0):
        self.map = gridmap
        self.h = lib().orc_tamp_new(gridmap.h, P(f64a(low)), P(f64a(up)), seed)

    def __del__(self):
        if getattr(self, "h", None):
            lib().orc_tamp_free(self.h)
            self.h = None

    def plan(self, start, b0, max_step, search_radius, n_iter_per_belief):
        b0 = f64a(b0)
        self.seconds = np.zeros(4)
        if not lib().orc_tamp_plan(self.h, P(f64a(start)), P(b0), len(b0), max_step, search_radius, n_iter_per_belief, P(self.seconds)):
            raise RuntimeError("reference panic in MapShelfDomainTampPRM::plan")
        self.belief_graph = BeliefGraph(handle=lib().orc_tamp_belief_graph(self.h), owner=self)
        return Policy(lib().orc_tamp_policy(self.h))

    def schedule(self):
        sz = np.zeros(7, np.int64)
        lib().orc_tamp_sizes(self.h, P(sz))
        n_modes, nodes, n_tr, pairs, finals, B, nw = (int(x) for x in sz)
        d = dict(mode_node_ptr=np.zeros(n_modes + 1, np.int64), samples=np.zeros((nodes, 2)), max_step=np.zeros(nodes),
                 search_radius=np.zeros(nodes), mode_belief_id=np.zeros(n_modes, np.int32), beliefs=np.zeros((B, nw)),
                 tr_from_mode=np.zeros(n_tr, np.int32), tr_to_mode=np.zeros(n_tr, np.int32), tr_pair_ptr=np.zeros(n_tr + 1, np.int64),
                 tr_pairs=np.zeros((pairs, 2), np.int32), mode_final_ptr=np.zeros(n_modes + 1, np.int64),
                 mode_final_nodes=np.zeros(finals, np.int32), expected_costs=np.zeros(nodes))
        lib().orc_tamp_export(self.h, *(P(d[k]) for k in ("mode_node_ptr", "samples", "max_step", "search_radius", "mode_belief_id",
                                                          "beliefs", "tr_from_mode", "tr_to_mode", "tr_pair_ptr", "tr_pairs",
                                                          "mode_final_ptr", "mode_final_nodes", "expected_costs")))
        return d
