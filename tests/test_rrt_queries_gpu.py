"""RRT* queries on the device: porrt_rrt_grow_queries (RRTBatch.grow_queries), one start, goal set and seed per tree, against the
oracle's sequential RRT::grow_tree for each query; porrt_rrt_best_paths (RRTBatch.best_paths, RRT.best_path, RRT.plan) against a
restatement of get_best_solution + get_path_to (rrt.rs:183-193, :48-60) over the oracle's tree."""
import ctypes
import math

import numpy as np
import pytest

from oracle import pyoracle as O
import po_rrt_b200 as P
from po_rrt_b200 import synth
import porrt_testutil as util
import rrt_best_oracle as RB
import rrt_mirror as R
import rrt_oracle as RO

pytestmark = pytest.mark.gpu

PARAMS = dict(max_step=0.1, search_radius=1.0, n_min=2500, n_max=10000)


@pytest.fixture(scope="module")
def ctx():
    c = P.Context(0)
    yield c
    c.close()


def best_solution(xy, parent, finals):
    """the restatement: a final's path is its chain of tree parents, root first; its cost is summed root first from 0.0 with norm2;
    the smallest (cost, path length) wins, the final found first among equal pairs.  -> (final id, cost, path states) or None"""
    best = None
    for f in finals:
        chain, v = [], int(f)
        while v >= 0:
            chain.append(v)
            v = int(parent[v])
            assert len(chain) <= len(xy), "parent cycle"
        chain.reverse()
        c = 0.0
        for a, b in zip(chain[:-1], chain[1:]):
            c = c + R.norm2([float(x) for x in xy[a]], [float(x) for x in xy[b]])
        if best is None or (c, len(chain)) < (best[1], len(best[2])):
            best = (int(f), c, chain)
    return None if best is None else (best[0], best[1], np.asarray([xy[v] for v in best[2]]))


def free_points(omap, n, rng, margin=0.9):
    """n states of free space in [-margin, margin]^2 drawn with rng"""
    out = []
    while len(out) < n:
        p = rng.uniform(-margin, margin, 2)
        if omap.state_validity([list(p)])[0] >= 0:
            out.append((float(p[0]), float(p[1])))
    return out


def queries_48(omap):
    """48 queries: distinct seeds, starts, goals and radii from a fixed seed; rows 1-3 share row 0's start, rows 4-5 row 0's goal,
    row 7 repeats row 6, one query has a second goal (holding in no world, so the goal masks do not overlap)"""
    rng = np.random.default_rng(11)
    starts, centres = free_points(omap, 48, rng), free_points(omap, 48, rng)
    radii = [(0.02, 0.05, 0.2)[k % 3] for k in range(48)]
    seeds = [1000 + 7 * k for k in range(48)]
    goals = [[(c, [1])] for c in centres]
    for k in (1, 2, 3):
        starts[k] = starts[0]
    for k in (4, 5):
        goals[k], radii[k] = goals[0], radii[0]
    starts[7], goals[7], radii[7], seeds[7] = starts[6], goals[6], radii[6], seeds[6]
    goals[9] = goals[9] + [(centres[10], [0])]
    return seeds, starts, goals, radii


def grow_both(omap, pmap, seeds, starts, goals, radii, p=PARAMS, low=util.LOW, up=util.UP):
    """-> the device batch, its status, the oracle trees and their codes, query by query"""
    dev = P.RRTBatch(pmap, low, up, seeds)
    status = dev.grow_queries(starts, [P.SquareGoal(g, r) for g, r in zip(goals, radii)], p["max_step"], p["search_radius"], p["n_min"],
                              p["n_max"])
    refs = []
    for s, st, g, r in zip(seeds, starts, goals, radii):
        ref = RO.RRT(omap, low, up, seed=int(s))
        refs.append((ref, ref.grow_tree(st, O.SquareGoal(g, r), p["max_step"], p["search_radius"], p["n_min"], p["n_max"])))
    return dev, status, refs


def assert_trees(dev, status, refs):
    for t, (ref, rc) in enumerate(refs):
        if rc < -1:
            assert status[t] == 5 and dev.panic_code[t] == rc and dev.n_it[t] == ref.n_it(), (t, status[t], rc)
            continue
        assert status[t] == rc and dev.n_it[t] == ref.n_it(), (t, status[t], rc, dev.n_it[t], ref.n_it())
        for a, b in zip(dev.tree(t), ref.tree()):
            np.testing.assert_array_equal(a, b)


def assert_best_paths(dev, refs):
    """every tree's best path against the restatement over the oracle's tree; -> the number of trees where two or more finals
    share the winning (cost, length) pair"""
    got = dev.best_paths()
    assert len(got) == len(refs)
    n_fin, cost, ptr, _ = _raw_best(dev.ctx, len(refs))
    tied = 0
    for t, (ref, rc) in enumerate(refs):
        want = best_solution(*(ref.tree()[k] for k in (0, 1, 3))) if rc >= 0 else None
        if want is None:
            assert got[t] is None and n_fin[t] == -1 and cost[t] == math.inf and ptr[t + 1] == ptr[t], t
            continue
        assert got[t] is not None, t
        path, c = got[t]
        assert n_fin[t] == want[0] and c == want[1], (t, n_fin[t], want[0], c, want[1])
        np.testing.assert_array_equal(path, want[2])
        xy, parent, _, finals = ref.tree()
        keys = [k for k in (_key(xy, parent, f) for f in finals) if k == (want[1], len(want[2]))]
        tied += len(keys) >= 2
        o = RB.best_path(ref.tree())                          # the C++ restatement the benchmark times agrees
        assert o is not None and o[1] == want[1] and np.array_equal(o[0], want[2])
    return tied


def _key(xy, parent, f):
    _, c, path = best_solution(xy, parent, [f])
    return (c, len(path))


def _raw_best(c, n, cap=None):
    """porrt_rrt_best_paths with arrays for n trees and room for cap path states (None: plenty, and the call must succeed)"""
    fin, cost, ptr, total = np.empty(n, np.int32), np.empty(n), np.empty(n + 1, np.int64), ctypes.c_int64()
    xy = np.empty((max(cap or 1 << 20, 1), 2))
    p = P.api._p
    rc = c.lib.porrt_rrt_best_paths(c.h, p(fin), p(cost), p(ptr), p(xy), len(xy) if cap is None else cap, ctypes.byref(total))
    assert cap is not None or rc == 0, rc
    return fin, cost, ptr, (rc, total.value, xy)


# ---- 1, 4: 48 distinct queries; every tree against the oracle, its best path against the restatement

def test_48_queries(ctx):
    omap, pmap = util.make_pair(ctx, synth.rrt_map(), None, P.DOOR, 0.3)
    seeds, starts, goals, radii = queries_48(omap)
    dev, status, refs = grow_both(omap, pmap, seeds, starts, goals, radii)
    assert_trees(dev, status, refs)
    assert (status == 0).sum() >= 24, status
    for a, b in zip(dev.tree(6), dev.tree(7)):
        np.testing.assert_array_equal(a, b)
    assert len(refs[9][0].tree()[3]) > 0
    assert_best_paths(dev, refs)
    got = [tuple(int(x) for x in dev.counters[t]) for t in range(48)]
    for t in (0, 1, 4, 6, 7, 9, 20, 47):                      # the counters equal a single porrt_rrt_grow call's
        one = P.RRT(pmap, util.LOW, util.UP, seed=seeds[t])
        rc = one.grow_tree(starts[t], P.SquareGoal(goals[t], radii[t]), PARAMS["max_step"], PARAMS["search_radius"], PARAMS["n_min"],
                           PARAMS["n_max"])
        assert rc == status[t] and one.sizes == tuple(int(x) for x in dev.sizes[t]) and one.counters == got[t], (t, one.counters, got[t])


# ---- 2: identical rows through the query form equal the seed batch

def test_identical_rows_equal_grow_batch(ctx):
    omap, pmap = util.make_pair(ctx, synth.rrt_map(), None, P.DOOR, 0.3)
    seeds, start, goal = list(range(16)), (-0.8, -0.8), [((0.8, 0.8), [1])]
    a = P.RRTBatch(pmap, util.LOW, util.UP, seeds)
    sa = a.grow_tree(start, P.SquareGoal(goal, 0.05), 0.1, 1.0, 2500, 10000)
    trees = [a.tree(t) for t in range(16)]
    b = P.RRTBatch(pmap, util.LOW, util.UP, seeds)
    sb = b.grow_queries([start] * 16, [P.SquareGoal(goal, 0.05)] * 16, 0.1, 1.0, 2500, 10000)
    np.testing.assert_array_equal(sa, sb)
    np.testing.assert_array_equal(a.sizes, b.sizes)
    np.testing.assert_array_equal(a.counters, b.counters)
    for t in range(16):
        for x, y in zip(trees[t], b.tree(t)):
            np.testing.assert_array_equal(x, y)


# ---- 3, 4: the shelf domain, three goal poses

def test_shelf_domain_three_goals(ctx):
    occ, zones = synth.shelf_map(200, n_zones=2)
    omap, pmap = util.make_pair(ctx, occ, zones, P.SHELF, 0.5)
    zp = omap.zone_positions()

    def beside(z):
        x, y = float(zp[z][0]), float(zp[z][1])
        return next((x - dx, y) for dx in (0.06, 0.1, 0.15, 0.2, 0.3) if omap.state_validity([[x - dx, y]])[0] >= 0)
    goals = [[(beside(0), [1])], [(beside(1), [1])], [((0.5, -0.6), [1])]]
    assert omap.state_validity([[0.5, -0.6]])[0] >= 0
    p = dict(max_step=0.1, search_radius=2.0, n_min=900, n_max=2500)
    dev, status, refs = grow_both(omap, pmap, [0, 1, 2], [(0.0, -0.8), (-0.5, -0.8), (0.0, -0.8)], goals, [0.05] * 3, p=p)
    assert_trees(dev, status, refs)
    assert (status == 0).all(), status
    assert_best_paths(dev, refs)


# ---- 4: repeated goal samples (kd depth > 64): finals tie on cost and on (cost, length)

def test_deep_duplicates_best_paths(ctx):
    omap, pmap = util.make_pair(ctx, synth.rrt_map(), None, P.DOOR, 0.3)
    p = dict(PARAMS, n_min=8000, n_max=10000)
    goal = [((0.8, 0.8), [1])]
    dev, status, refs = grow_both(omap, pmap, [0, 1, 2, 3], [(0.76, 0.76), (0.76, 0.76), (0.7, 0.8), (0.8, 0.72)], [goal] * 4,
                                  [0.05] * 4, p=p)
    assert_trees(dev, status, refs)
    _, counts = np.unique(refs[0][0].tree()[0], axis=0, return_counts=True)
    assert counts.max() > 64
    tied = assert_best_paths(dev, refs)
    assert tied >= 1, "no tree has two finals at the winning (cost, length): the first-found rule is not exercised"


# ---- 5: rrt.rs:254-268 on the device

def test_plan_empty_space(ctx):
    occ = np.full((256, 256), 255, np.uint8)
    omap, pmap = util.make_pair(ctx, occ, None, P.DOOR, 0.3)
    goal = [((0.9, 0.9), [1])]
    rrt = P.RRT(pmap, util.LOW, util.UP, seed=0)
    got = rrt.plan([0.0, 0.0], P.SquareGoal(goal, 0.05), 0.1, 1.0, 1000, 10000)
    assert got is not None
    path, cost = got
    assert len(path) > 2
    assert cost >= R.norm2([0.0, 0.0], [0.9, 0.9]) - 0.05 * 2 ** 0.5 - 1e-9
    ref = RO.RRT(omap, util.LOW, util.UP, seed=0)
    assert ref.grow_tree([0.0, 0.0], O.SquareGoal(goal, 0.05), 0.1, 1.0, 1000, 10000) == 0
    xy, parent, _, finals = ref.tree()
    want = best_solution(xy, parent, finals)
    assert cost == want[1]
    np.testing.assert_array_equal(path, want[2])
    assert rrt.best_path()[1] == cost


# ---- 6: trees without a path, capacity, order of calls, argument errors

def _edge_map():
    occ = synth.rrt_map()
    x, y = synth.pixel_centres(occ.shape[0])
    occ[(np.abs(x - 0.8) <= 0.08) & (np.abs(y - 0.8) <= 0.08)] = 0          # the goal diamond at (0.8, 0.8) is an obstacle
    occ[(np.abs(x - 0.5) <= 0.3) & (np.abs(y + 0.5) <= 0.3)] = 0            # a block no step from its centre (0.5, -0.5) leaves
    return occ


def test_trees_without_a_path_among_healthy_ones(ctx):
    omap, pmap = util.make_pair(ctx, _edge_map(), None, P.DOOR, 0.3)
    rng = np.random.default_rng(5)
    starts, centres = free_points(omap, 6, rng), free_points(omap, 6, rng)
    goals = [[(c, [1])] for c in centres]
    starts[1], goals[1] = (-0.8, -0.8), [((0.8, 0.8), [1])]                # unreachable goal
    starts[3] = (0.5, -0.5)                                                   # root only
    starts[4] = (1.5, 1.5)                                                    # outside the map: the first state check panics
    p = dict(PARAMS, n_min=100, n_max=3000)
    dev, status, refs = grow_both(omap, pmap, list(range(6)), starts, goals, [0.05] * 6, p=p)
    assert_trees(dev, status, refs)
    assert status[1] == 1 and dev.n_it[1] == 3000
    assert status[3] == 1 and dev.sizes[3][1] == 1
    assert status[4] == 5 and dev.panic_code[4] == P.PANIC_OOB
    assert (status[[0, 2, 5]] == 0).all(), status
    assert_best_paths(dev, refs)
    got = dev.best_paths()
    assert got[1] is None and got[3] is None and got[4] is None
    # the trees are intact after best_paths, and a PTO growth in between changes nothing
    assert_trees(dev, status, refs)
    P.PTO(pmap, util.LOW, util.UP, seed=2).grow_graph((-0.8, -0.8), P.SquareGoal([((0.8, 0.8), [1])], 0.05), 0.05, 5.0, 300, 1000)
    again = dev.best_paths()
    for a, b in zip(got, again):
        assert (a is None and b is None) or (a[1] == b[1] and np.array_equal(a[0], b[0]))


def test_capacity_and_no_growth(ctx):
    c2 = P.Context(0)
    try:
        omap, pmap = util.make_pair(c2, synth.rrt_map(), None, P.DOOR, 0.3)
        rc, total, _ = _raw_best(c2, 4, cap=0)[3]
        assert rc == 1                                                          # nothing grown
        dev = P.RRTBatch(pmap, util.LOW, util.UP, [0, 1, 2, 3])
        dev.grow_queries([(-0.8, -0.8)] * 4, [P.SquareGoal([((0.8, 0.8), [1])], 0.05)] * 4, 0.1, 1.0, 2500, 10000)
        want = dev.best_paths()
        n = sum(len(w[0]) for w in want if w is not None)
        assert n > 4
        fin, cost, ptr, (rc, total, _) = _raw_best(c2, 4, cap=n - 1)
        assert rc == 4 and total == n and ptr[4] == n
        fin, cost, ptr, (rc, total, xy) = _raw_best(c2, 4, cap=n)
        assert rc == 0 and total == n
        for t, w in enumerate(want):
            assert cost[t] == w[1] and np.array_equal(xy[ptr[t]:ptr[t + 1]], w[0])
    finally:
        c2.close()


def test_argument_errors(ctx):
    omap, pmap = util.make_pair(ctx, synth.rrt_map(size=256, n_rects=64), None, P.DOOR, 0.3)
    p = P.api._p
    low, up = np.array(util.LOW), np.array(util.UP)

    def call(starts=((-0.8, -0.8), (-0.7, -0.8)), ptr=(0, 1, 2), gmd=(0.05, 0.05), masks=((1,), (1,)), goals=((0.8, 0.8), (0.7, 0.8))):
        st, pt, gm = np.array(starts, np.float64), np.array(ptr, np.int64), np.array(gmd, np.float64)
        gx, mk = np.array(goals, np.float64), np.array(masks, np.uint64)
        seeds, sizes, status = np.arange(2, dtype=np.uint64), np.zeros(6, np.int64), np.zeros(2, np.int32)
        return ctx.lib.porrt_rrt_grow_queries(ctx.h, 2, p(seeds), p(st), p(low), p(up), p(pt), p(gx), p(mk), p(gm), 0.1, 1.0, 10, 100,
                                              p(sizes), p(status), None, None)
    assert call() == 0
    assert call(ptr=(0, 2, 1)) == 1                                             # goal_ptr decreases
    assert call(ptr=(1, 1, 2)) == 1                                             # goal_ptr[0] != 0
    assert call(starts=((-0.8, math.nan), (-0.7, -0.8))) == 1                   # a start that is not finite
    assert call(starts=((-0.8, -0.8), (math.inf, -0.8))) == 1
    assert call(gmd=(0.05, -0.01)) == 1                                         # goal_max_dist negative or NaN
    assert call(gmd=(math.nan, 0.05)) == 1
    assert call(ptr=(0, 0, 2)) == 5                                             # query 1's two goals hold in the same world
    assert b"query 1" in ctx.lib.porrt_last_error(ctx.h)
    assert call(ptr=(0, 0, 2), masks=((1,), (0,))) == 0                         # two goals in one query, disjoint masks
    assert call(ptr=(0, 2, 2), masks=((1,), (0,))) == 0                         # a query without goals
