"""The reference's exported C planner API (src/pto_c.rs:63-270) as implemented by po_rrt_b200/libpo_rrt_c.so (include/po_rrt_c.h).

CPU: the library loads, exports every name the header declares, and plan() fails loudly -- through get_planning_error -- when there
is no device for the value backups.  GPU: a C-style client (ctypes callbacks standing in for the C++ caller's world model, backed by
the oracle's map functions) plans on shelf and door problems with seeded samplers and gets the oracle's PTO pipeline
(grow_graph -> plan_belief_space -> refine_solution(PartialShortCut(n))) bit for bit: same iteration count, same paths, same
expected cost."""
import ctypes as C
import os
import re
import subprocess

import numpy as np
import pytest

from oracle import pyoracle as O
from po_rrt_b200 import synth
import porrt_testutil as util

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SO = os.path.join(ROOT, "po_rrt_b200", "libpo_rrt_c.so")
sz, f64p, vp = C.c_size_t, C.POINTER(C.c_double), C.c_void_p

STATE_CB = C.CFUNCTYPE(C.c_int64, f64p, sz)
TRANS_CB = C.CFUNCTYPE(C.c_int64, f64p, sz, f64p, sz)
OBS_CB = C.CFUNCTYPE(None, f64p, sz, f64p, sz, C.POINTER(C.POINTER(C.POINTER(sz))), C.POINTER(sz))
GOAL_CB = C.CFUNCTYPE(C.c_bool, f64p, sz, C.POINTER(C.c_bool), sz)
GOAL_EX_CB = C.CFUNCTYPE(None, sz, f64p, sz)


def _declared():
    src = open(os.path.join(ROOT, "include", "po_rrt_c.h")).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    src = re.sub(r"typedef[^;]*;", "", src)
    return sorted(set(re.findall(r"\b([a-z_]+)\s*\(CPlanningProblem\*|\b(new_planning_problem)\s*\(", src)) - {("", "")})


def _lib():
    if not os.path.exists(SO):
        subprocess.run(["make", "-C", os.path.join(ROOT, "po_rrt_b200", "csrc"), "-j4", "all"], check=True, capture_output=True)
    lib = C.CDLL(SO)
    lib.new_planning_problem.restype = vp
    lib.get_planning_error.restype = C.c_char_p
    lib.get_planning_error.argtypes = [vp]
    lib.delete_planning_problem.argtypes = [vp]
    lib.set_problem_dimensions.argtypes = [vp, sz, sz]
    lib.set_lower_sampling_bound.argtypes = [vp, f64p, sz]
    lib.set_upper_sampling_bound.argtypes = [vp, f64p, sz]
    lib.set_world_validities.argtypes = [vp, C.POINTER(C.POINTER(sz)), sz]
    lib.set_state_validity_callback.argtypes = [vp, STATE_CB]
    lib.set_transition_validity_callback.argtypes = [vp, TRANS_CB]
    lib.set_observer_callback.argtypes = [vp, OBS_CB]
    lib.set_start_belief_state.argtypes = [vp, f64p, sz, C.POINTER(f64p), sz]
    lib.set_goal_callback.argtypes = [vp, GOAL_CB]
    lib.set_goal_example_callback.argtypes = [vp, GOAL_EX_CB]
    lib.set_search_parameters.argtypes = [vp, sz, sz, C.c_double, C.c_double]
    lib.set_refine_parameters.argtypes = [vp, sz]
    lib.set_sampler_seed.argtypes = [vp, C.c_uint64]
    lib.set_observer_array_ownership.argtypes = [vp, C.c_int32]
    lib.plan.argtypes = [vp, f64p, sz]
    lib.get_planning_metrics.argtypes = [vp, C.POINTER(sz)] + [f64p] * 5
    lib.get_paths_info.argtypes = [vp, C.POINTER(sz), C.POINTER(C.POINTER(sz)), f64p]
    lib.get_paths_variable.argtypes = [vp, sz, sz, C.POINTER(f64p), C.POINTER(sz)]
    lib.get_planning_sizes.argtypes = [vp] + [C.POINTER(sz)] * 5
    return lib


class Client:
    """what the reference's C++ caller does: owns the world model (here: the oracle's map), hands callbacks to the planner"""

    def __init__(self, lib, omap, goals, goal_dist, b0, dim=2):
        self.lib, self.omap, self.dim = lib, omap, dim
        self.libc = C.CDLL(None)
        self.libc.malloc.restype = vp
        self.libc.malloc.argtypes = [sz]
        self.nw = omap.n_worlds
        self.goals, self.goal_dist = goals, goal_dist
        self.beliefs = omap.reachable_belief_states(b0)
        self.belief_index = {b.tobytes(): k for k, b in enumerate(self.beliefs)}
        self.validities = np.asarray(omap.world_validities())          # [n_validities, n_worlds] of 0/1
        self.calls = dict(state=0, transition=0, observe=0, goal=0)
        self.h = lib.new_planning_problem()
        lib.set_problem_dimensions(self.h, dim, self.nw)
        self.low = (C.c_double * dim)(*([-1.0] * dim))
        self.up = (C.c_double * dim)(*([1.0] * dim))
        lib.set_lower_sampling_bound(self.h, self.low, dim)
        lib.set_upper_sampling_bound(self.h, self.up, dim)
        self.v_rows = [(sz * self.nw)(*[int(x) for x in row]) for row in self.validities]
        self.v_ptrs = (C.POINTER(sz) * len(self.v_rows))(*[C.cast(r, C.POINTER(sz)) for r in self.v_rows])
        lib.set_world_validities(self.h, self.v_ptrs, len(self.v_rows))
        self.b_rows = [(C.c_double * self.nw)(*b) for b in self.beliefs]
        self.b_ptrs = (f64p * len(self.b_rows))(*[C.cast(r, f64p) for r in self.b_rows])
        self.b0 = (C.c_double * self.nw)(*b0)
        lib.set_start_belief_state(self.h, self.b0, self.nw, self.b_ptrs, len(self.b_rows))
        self.obs_slot = C.POINTER(sz)()                               # the `*mut usize` the observer's out-pointer points at

        def state(s, n):
            self.calls["state"] += 1
            return int(self.omap.state_validity([[s[0], s[1]]])[0])

        def transition(a, na, b, nb):
            self.calls["transition"] += 1
            return int(self.omap.edge_validity([[a[0], a[1]]], [[b[0], b[1]]])[0])

        def observe(s, n, b, nb, out_ids, out_n):
            self.calls["observe"] += 1
            succ = self.omap.observe([s[0], s[1]], [b[k] for k in range(nb)])
            ids = [self.belief_index[x.tobytes()] for x in succ]
            arr = C.cast(self.libc.malloc(8 * max(1, len(ids))), C.POINTER(sz))   # the planner frees it (pto_c.rs:411)
            for k, v in enumerate(ids):
                arr[k] = v
            self.obs_slot = arr
            out_ids[0] = C.pointer(self.obs_slot)
            out_n[0] = len(ids)

        def goal(s, n, validity, nw):
            self.calls["goal"] += 1
            for (gx, gy), mask in self.goals:                          # SquareGoal::goal, common.rs:326-341
                if abs(gx - s[0]) + abs(gy - s[1]) < self.goal_dist:
                    for w in range(nw):
                        validity[w] = bool(mask[w])
                    return True
            return False

        def goal_example(world, s, n):
            for (gx, gy), mask in self.goals:
                if mask[world]:
                    s[0], s[1] = gx, gy
                    return

        self.cbs = [STATE_CB(state), TRANS_CB(transition), OBS_CB(observe), GOAL_CB(goal), GOAL_EX_CB(goal_example)]
        lib.set_state_validity_callback(self.h, self.cbs[0])
        lib.set_transition_validity_callback(self.h, self.cbs[1])
        lib.set_observer_callback(self.h, self.cbs[2])
        lib.set_goal_callback(self.h, self.cbs[3])
        lib.set_goal_example_callback(self.h, self.cbs[4])

    def plan(self, start, n_min, n_max, max_step, search_radius, refine, seed=0):
        self.lib.set_search_parameters(self.h, n_min, n_max, max_step, search_radius)
        self.lib.set_refine_parameters(self.h, refine)
        if seed is not None:
            self.lib.set_sampler_seed(self.h, seed)
        s = (C.c_double * self.dim)(*start)
        self.lib.plan(self.h, s, self.dim)
        err = self.lib.get_planning_error(self.h)
        return err.decode() if err else None

    def paths(self):
        n, lens, cost = sz(), C.POINTER(sz)(), C.c_double()
        self.lib.get_paths_info(self.h, C.byref(n), C.byref(lens), C.byref(cost))
        out = []
        for p in range(n.value):
            path = []
            for k in range(lens[p]):
                st, ns = f64p(), sz()
                self.lib.get_paths_variable(self.h, p, k, C.byref(st), C.byref(ns))
                path.append(tuple(st[d] for d in range(ns.value)))
            out.append(path)
        return out, cost.value

    def metrics(self):
        n = sz()
        t = [C.c_double() for _ in range(5)]
        self.lib.get_planning_metrics(self.h, C.byref(n), *[C.byref(x) for x in t])
        return n.value, [x.value for x in t]

    def sizes(self):
        v = [sz() for _ in range(5)]
        self.lib.get_planning_sizes(self.h, *[C.byref(x) for x in v])
        return [x.value for x in v]

    def close(self):
        self.lib.delete_planning_problem(self.h)
        self.h = None


def _shelf_problem(Z=2, size=200):
    occ, zones = synth.shelf_map(size, n_zones=Z)
    omap = O.GridMap(occ, zones, util.LOW, util.UP, O.SHELF, 0.5)
    zp = omap.zone_positions()
    goals = [((float(zp[z][0]) - 0.06, float(zp[z][1])), [1 if k == z else 0 for k in range(Z)]) for z in range(Z)]
    return omap, goals, [1.0 / Z] * Z, (-0.8, -0.8)


def test_library_exports_the_reference_api():
    _lib()
    out = subprocess.run(["nm", "-D", "--defined-only", SO], check=True, capture_output=True, text=True).stdout
    exported = set(re.findall(r" T ([a-z_]+)", out))
    names = sorted({a or b for a, b in _declared()})
    # pto_c.rs's #[no_mangle] functions, by name
    for ref in ("new_planning_problem", "delete_planning_problem", "set_problem_dimensions", "set_lower_sampling_bound",
                "set_upper_sampling_bound", "set_world_validities", "set_state_validity_callback", "set_transition_validity_callback",
                "set_cost_evaluator_callback", "set_observer_callback", "set_start_belief_state", "set_goal_callback",
                "set_goal_example_callback", "set_search_parameters", "set_refine_parameters", "plan", "get_planning_metrics",
                "get_paths_info", "get_paths_variable"):
        assert ref in names, ref
    missing = [n for n in names if n not in exported]
    assert not missing, missing
    subprocess.run(["gcc", "-std=c99", "-fsyntax-only", "-x", "c", os.path.join(ROOT, "include", "po_rrt_c.h")], check=True)


def test_plan_without_device_fails_loudly():
    """growth runs (host, callbacks), then the value backups need the device: no CPU fallback"""
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    lib = _lib()
    omap, goals, b0, start = _shelf_problem()
    c = Client(lib, omap, goals, 0.05, b0)
    err = c.plan(start, 300, 20000, 0.05, 5.0, 10)
    assert err and "no CPU fallback" in err, err
    paths, cost = c.paths()
    assert paths == [] and cost == 0.0
    assert c.metrics()[0] >= 300 and c.calls["state"] > 300
    # reference panics become messages
    assert "Start from a valid state" in c.plan((5.0, 5.0), 10, 10, 0.05, 5.0, 0)
    c.close()


def _oracle_plan(omap, goals, goal_dist, b0, start, n_min, n_max, max_step, search_radius, refine):
    goal = O.SquareGoal(goals, goal_dist)
    pto = O.PTO(omap, util.LOW, util.UP, seed=0)
    assert pto.grow_graph(start, goal, max_step, search_radius, n_min, n_max) == 0
    pto.build_belief_graph(b0)
    pto.compute_expected_costs_to_goals()
    pto.extract_policy()
    return pto, pto.refine_policy_shortcut(refine)


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["shelf", "door"])
def test_plan_matches_the_oracle_pipeline(kind):
    lib = _lib()
    if kind == "shelf":
        omap, goals, b0, start = _shelf_problem()
        args = (500, 20000, 0.05, 5.0, 200)
    else:
        occ, zones = util.planning_door_map(200)
        omap = O.GridMap(occ, zones, util.LOW, util.UP, O.DOOR, 0.3)
        goals, b0, start = [((0.8, 0.8), [1, 1, 1, 1])], [0.1, 0.1, 0.1, 0.7], (-0.8, -0.8)
        args = (700, 20000, 0.05, 5.0, 200)
    c = Client(lib, omap, goals, 0.05, b0)
    err = c.plan(start, *args)
    assert err is None, err
    pto, want = _oracle_plan(omap, goals, 0.05, b0, start, *args)
    n_it, times = c.metrics()
    assert n_it == pto.n_it()
    n_nodes, n_bn, n_be, sweeps, n_pol = c.sizes()
    assert n_nodes == pto.graph.n_nodes() and n_bn == pto.belief_graph.n_nodes() and sweeps > 0 and n_pol == len(want.xy)
    paths, cost = c.paths()
    assert cost == want.expected_costs                                  # bit for bit
    assert len(paths) == len(want.leafs) > 0
    for k, path in enumerate(paths):
        assert path == want.path_to_leaf(k), k                          # refined states, bit for bit
    assert all(t >= 0.0 for t in times) and times[4] >= times[0]
    assert c.calls["observe"] == n_nodes * len(c.beliefs)
    c.close()


@pytest.mark.gpu
def test_plan_true_random_streams_reach_the_goals():
    """without set_sampler_seed the streams come from the OS like the reference's new_true_random: two runs differ, both solve"""
    lib = _lib()
    occ, zones = util.planning_door_map(200)
    omap = O.GridMap(occ, zones, util.LOW, util.UP, O.DOOR, 0.3)
    goals, b0, start = [((0.8, 0.8), [1, 1, 1, 1])], [0.1, 0.1, 0.1, 0.7], (-0.8, -0.8)
    costs = []
    for _ in range(2):
        c = Client(lib, omap, goals, 0.05, b0)
        errs = []
        for _attempt in range(3):          # (OS-seeded streams: a rare unlucky roadmap may not connect every world within the budget)
            errs.append(c.plan(start, 700, 200000, 0.05, 5.0, 50, seed=None))
            if errs[-1] is None:
                break
        assert errs[-1] is None, errs
        paths, cost = c.paths()
        assert len(paths) >= 1 and np.isfinite(cost) and cost > 0
        for path in paths:
            assert path[0] == start
        costs.append(cost)
        c.close()
    assert costs[0] != costs[1]


@pytest.mark.gpu
@pytest.mark.parametrize("dim", [3, 7])
def test_plan_in_more_dimensions(dim):
    """state_dim 3 and 7 (two of the reference's instantiations, pto_c.rs:236-240): the world model looks at the first two coordinates,
    the others are free.  No oracle exists for N != 2: the plan must solve the problem and every step of every returned path must
    be a transition the caller's own callbacks accept, in a belief the policy can be in"""
    lib = _lib()
    occ, zones = util.planning_door_map(200)
    omap = O.GridMap(occ, zones, util.LOW, util.UP, O.DOOR, 0.3)
    goals, b0, start = [((0.8, 0.8), [1, 1, 1, 1])], [0.1, 0.1, 0.1, 0.7], (-0.8, -0.8) + (0.0,) * (dim - 2)
    c = Client(lib, omap, goals, 0.05, b0, dim=dim)
    err = c.plan(start, 1500, 300000, 0.1 * dim, 5.0, 100, seed=3)
    assert err is None, err
    paths, cost = c.paths()
    n_nodes, n_bn, n_be, sweeps, n_pol = c.sizes()
    assert len(paths) >= 1 and np.isfinite(cost) and cost > 0 and sweeps > 0 and n_bn == n_nodes * len(c.beliefs)
    for path in paths:
        assert len(path[0]) == dim and path[0] == start
        assert abs(path[-1][0] - 0.8) + abs(path[-1][1] - 0.8) < 0.05          # a goal state
        for a, b in zip(path[:-1], path[1:]):
            assert omap.state_validity([[a[0], a[1]]])[0] >= 0 and omap.state_validity([[b[0], b[1]]])[0] >= 0
            assert omap.edge_validity([[a[0], a[1]]], [[b[0], b[1]]])[0] >= 0
    # the expected cost is a probability-weighted mean of the paths' lengths
    lengths = [sum(float(np.linalg.norm(np.subtract(a, b))) for a, b in zip(p[:-1], p[1:])) for p in paths]
    assert min(lengths) - 1e-9 <= cost <= max(lengths) + 1e-9
    c.close()


@pytest.mark.gpu
def test_c_client(tmp_path):
    """tests/pto_c_client.c: the planner API driven from plain C (gcc -std=c99) with the world model in C callbacks, three-dimensional
    states, malloc()ed observer arrays the planner frees -- the policy branches on the observed door as it must"""
    _lib()
    exe = str(tmp_path / "pto_c_client")
    libdir = os.path.join(ROOT, "po_rrt_b200")
    subprocess.run(["gcc", "-std=c99", "-O1", "-Wall", "-Wextra", "-pedantic", "-I", os.path.join(ROOT, "include"),
                    os.path.join(ROOT, "tests", "pto_c_client.c"), "-o", exe, "-L", libdir, "-lpo_rrt_c", "-lm", "-Wl,-rpath," + libdir], check=True)
    r = subprocess.run([exe], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0 and "pto_c_client: ok" in r.stdout, r.stdout + r.stderr


def test_planner_reports_the_references_panics():
    """where pto_c.rs would panic -- and with it abort the calling process -- plan() records the message instead (host-side checks:
    none of these reaches the device)"""
    lib = _lib()
    omap, goals, b0, start = _shelf_problem()
    c = Client(lib, omap, goals, 0.05, b0)
    s3 = (C.c_double * 3)(0.0, 0.0, 0.0)
    lib.set_search_parameters(c.h, 10, 10, 0.05, 5.0)
    lib.plan(c.h, s3, 3)                                                     # assert_eq!(start_size, state_dim), pto_c.rs:229
    assert b"start_size" in lib.get_planning_error(c.h)
    assert "Start from a valid state" in c.plan((5.0, 5.0), 10, 10, 0.05, 5.0, 0)           # pto.rs:61
    assert "final nodes are not reached" in c.plan(start, 5, 5, 0.05, 5.0, 0)               # pto_c.rs:214 .expect(..)
    paths, cost = c.paths()
    assert paths == [] and cost == 0.0                                       # outputs stay empty after a failed plan
    lib.set_problem_dimensions(c.h, 2, 0)
    assert "n_worlds" in c.plan(start, 5, 5, 0.05, 5.0, 0)
    lib.set_problem_dimensions(c.h, 17, c.nw)
    big = (C.c_double * 17)(*([0.0] * 17))
    lib.plan(c.h, big, 17)
    assert b"case not yet handled" in lib.get_planning_error(c.h)            # pto_c.rs:238
    c.close()
    # a problem without callbacks: Option::unwrap() on None in the reference
    h = lib.new_planning_problem()
    lib.set_problem_dimensions(h, 2, 2)
    lo, up = (C.c_double * 2)(-1, -1), (C.c_double * 2)(1, 1)
    lib.set_lower_sampling_bound(h, lo, 2); lib.set_upper_sampling_bound(h, up, 2)
    s2 = (C.c_double * 2)(0.0, 0.0)
    lib.plan(h, s2, 2)
    assert b"callback is missing" in lib.get_planning_error(h)
    lib.delete_planning_problem(h)
    lib.delete_planning_problem(None)                                        # delete_planning_problem(None) is a no-op there too (:103)


def test_growth_matches_the_oracle_without_a_device():
    """PTO::grow_graph inside the planner is host code (N-dimensional kd-tree, steer, reachability, the two sampler streams, the
    caller's callbacks): on a box without a GPU plan() stops at the value backups, but the roadmap it grew must already be the
    oracle's -- same number of iterations, same number of nodes -- on a shelf and a door problem"""
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU present: test_plan_matches_the_oracle_pipeline covers the whole pipeline")
    lib = _lib()
    omap, goals, b0, start = _shelf_problem()
    problems = [(omap, goals, b0, start, (500, 20000, 0.05, 5.0))]
    occ, zones = util.planning_door_map(200)
    problems.append((O.GridMap(occ, zones, util.LOW, util.UP, O.DOOR, 0.3), [((0.8, 0.8), [1, 1, 1, 1])], [0.1, 0.1, 0.1, 0.7], (-0.8, -0.8),
                     (700, 20000, 0.05, 5.0)))
    for omap, goals, b0, start, (n_min, n_max, max_step, search_radius) in problems:
        c = Client(lib, omap, goals, 0.05, b0)
        err = c.plan(start, n_min, n_max, max_step, search_radius, 0)
        assert err and "no CPU fallback" in err
        pto = O.PTO(omap, util.LOW, util.UP, seed=0)
        assert pto.grow_graph(start, O.SquareGoal(goals, 0.05), max_step, search_radius, n_min, n_max) == 0
        assert c.metrics()[0] == pto.n_it() and c.sizes()[0] == pto.graph.n_nodes()
        assert c.sizes()[1] == pto.graph.n_nodes() * len(c.beliefs)          # the belief graph was built (observer callbacks) before the device step
        c.close()
