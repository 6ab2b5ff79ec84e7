"""PRM path queries on the device: porrt_prm_plan_paths (PRM.plan_paths, PRM.plan_path) against the oracle's PRM::plan_path
(prm.rs:111-122: nearest_neighbor for start and goal, dijkstra(graph, [goal]), extract_path, pto_graph.rs:305-359) on a PRM the
oracle grew from the same samples."""
import ctypes as C

import numpy as np
import pytest

from oracle import pyoracle as O
import po_rrt_b200 as P
from po_rrt_b200 import synth
import porrt_testutil as util

pytestmark = pytest.mark.gpu

MS, SR = 0.1, 2.0


@pytest.fixture(scope="module")
def ctx():
    c = P.Context(0)
    yield c
    c.close()


def build(ctx, occ, zones, kind, samples, max_step=MS, search_radius=SR, visibility=0.5):
    """the same samples through PRM::add_sample on the oracle and through porrt_prm_build -> (product PRM, oracle PRM)"""
    omap, pmap = util.make_pair(ctx, occ, zones, kind, visibility)
    oprm = O.PRM(omap, util.LOW, util.UP, seed=0)
    oprm.add_samples(samples, max_step, search_radius)
    prm = P.PRM(pmap).grow_graph(samples, max_step, search_radius)
    _, _, rp, col, _ = oprm.graph.export(0)
    np.testing.assert_array_equal(prm.row_ptr, rp)
    np.testing.assert_array_equal(prm.col.astype(np.int64), col)
    return prm, oprm


def check_oracle(oprm, starts, goals, res, queries=None):
    """every listed query against the oracle: node ids = kd-tree nearest_neighbor, cost = dijkstra([g])[s], path = plan_path"""
    paths, cost, status, sn, gn = res
    columns = {}
    for q in (range(len(starts)) if queries is None else queries):
        s, g = oprm.kdtree.nearest_neighbor(starts[q]), oprm.kdtree.nearest_neighbor(goals[q])
        assert (sn[q], gn[q]) == (s, g), q
        if g not in columns:
            columns[g] = oprm.graph.dijkstra([g])
        assert cost[q] == columns[g][s] or (np.isinf(cost[q]) and np.isinf(columns[g][s])), q
        assert status[q] == (P.PATH_NONE if np.isinf(columns[g][s]) else P.PATH_FOUND), q
        np.testing.assert_array_equal(paths[q], oprm.plan_path(starts[q], goals[q]), err_msg="query %d" % q)


def same(a, b):
    """two plan_paths results are identical"""
    assert len(a[0]) == len(b[0])
    for x, y in zip(a[0], b[0]):
        np.testing.assert_array_equal(x, y)
    for x, y in zip(a[1:], b[1:]):
        np.testing.assert_array_equal(x, y)


def permuted(res, perm):
    return [res[0][k] for k in perm], res[1][perm], res[2][perm], res[3][perm], res[4][perm]


def with_option(ctx, option, value, call):
    ctx.set_option(option, value)
    try:
        return call()
    finally:
        ctx.set_option(option, 0)


def queries_512(samples, rng, n_goals=32):
    """512 queries: 32 distinct goal points, starts drawn at random, every 7th start exactly on a vertex, rows 1-3 repeat row 0 and
    row 9 has start == goal"""
    goal_pts = rng.uniform(-0.95, 0.95, (n_goals, 2))
    goals = goal_pts[np.arange(512) % n_goals].copy()
    starts = rng.uniform(-0.95, 0.95, (512, 2))
    on = np.arange(0, 512, 7)
    starts[on] = samples[rng.integers(0, len(samples), len(on))]
    starts[1:4], goals[1:4] = starts[0], goals[0]
    starts[9] = goals[9]
    return np.ascontiguousarray(starts), np.ascontiguousarray(goals)


def restated_walk(rp, col, xy, cost, s):
    """extract_path restated over the oracle's CSR with a step guard -> (path node ids, whether a step met an equal minimum) or
    (None, _) for a walk that makes V steps without reaching cost 0.0"""
    node, path, tie = s, [s], False
    while cost[node] != 0.0:
        if len(path) > len(xy):
            return None, tie
        ps = col[rp[node]:rp[node + 1]]
        d = xy[ps] - xy[node]
        c = cost[ps] + np.sqrt(d[:, 0] * d[:, 0] + d[:, 1] * d[:, 1])
        k = int(np.argmin(c))                        # numpy keeps the first minimum too
        tie |= int(np.sum(c == c[k])) > 1
        node = int(ps[k])
        path.append(node)
    return path, tie


# ---------------------------------------------------------------------------------------------------------------- planning maps
@pytest.mark.parametrize("kind", [P.DOOR, P.SHELF])
def test_plan_paths_vs_oracle_on_chip_and_frontier(ctx, kind):
    """V = 2500 (on-chip column solver), 512 queries sharing 32 goal columns; the same under FORCE_GLOBAL_SWEEPS"""
    occ, zones = util.small_door_map(seed=11) if kind == P.DOOR else synth.shelf_map(200, n_zones=2)
    rng = np.random.default_rng(1 + kind)
    samples = rng.uniform(-1.0, 1.0, (2500, 2))
    prm, oprm = build(ctx, occ, zones, kind, samples)
    starts, goals = queries_512(samples, rng)
    res = prm.plan_paths(starts, goals)
    assert res[3][9] == res[4][9] and res[1][9] == 0.0 and len(res[0][9]) == 1
    assert (res[2] == P.PATH_FOUND).sum() > 128 and (res[2] == P.PATH_NONE).sum() > 16
    check_oracle(oprm, starts, goals, res)
    same(res, with_option(ctx, P.OPT_FORCE_GLOBAL_SWEEPS, 1, lambda: prm.plan_paths(starts, goals)))
    np.testing.assert_array_equal(prm.plan_path(starts[0], goals[0]), oprm.plan_path(starts[0], goals[0]))


def test_plan_paths_frontier_by_itself(ctx):
    """a roadmap of 40000 nodes: the column solver does not fit on chip, the frontier schedule is taken by itself"""
    occ, zones = synth.door_map(size=1024, n_rects=4096, n_zones=3, seed=12)
    rng = np.random.default_rng(7)
    samples = rng.uniform(-1.0, 1.0, (40000, 2))
    prm, oprm = build(ctx, occ, zones, P.DOOR, samples)
    starts, goals = queries_512(samples, rng, n_goals=16)
    res = prm.plan_paths(starts, goals)
    assert (res[2] == P.PATH_FOUND).sum() > 256
    check_oracle(oprm, starts, goals, res, queries=range(0, 512, 11))
    same(res, with_option(ctx, P.OPT_FORCE_GLOBAL_SWEEPS, 1, lambda: prm.plan_paths(starts, goals)))


def test_tile_and_thread_per_query_nn_agree(ctx):
    """2400 queries = 4800 points: the tile kernels serve the 1-NN; FORCE_THREAD_PER_QUERY_NN gives identical outputs"""
    occ, zones = util.small_door_map(seed=13)
    rng = np.random.default_rng(3)
    samples = rng.uniform(-1.0, 1.0, (3000, 2))
    prm, oprm = build(ctx, occ, zones, P.DOOR, samples)
    starts = np.ascontiguousarray(rng.uniform(-1.0, 1.0, (2400, 2)))
    goals = np.ascontiguousarray(samples[rng.integers(0, 3000, 2400)] + rng.uniform(-0.01, 0.01, (2400, 2)))
    res = prm.plan_paths(starts, goals)
    same(res, with_option(ctx, P.OPT_FORCE_THREAD_PER_QUERY_NN, 1, lambda: prm.plan_paths(starts, goals)))
    check_oracle(oprm, starts, goals, res, queries=range(0, 2400, 37))


# ---------------------------------------------------------------------------------------------------------------- lattices
def lattice(n=16, h=0.125, seed=5):
    """n x n dyadic lattice points (exact coordinates, exact distances) in a shuffled insertion order"""
    c = -0.9375 + h * np.arange(n)
    pts = np.array([(x, y) for y in c for x in c])
    return np.ascontiguousarray(pts[np.random.default_rng(seed).permutation(len(pts))]), c


def free_map():
    return np.full((256, 256), 255, np.uint8), None


def test_nearest_ties_follow_kd_order(ctx):
    """queries at cell centres (4 vertices at one distance) and edge midpoints (2): the start and goal nodes are the oracle kd-tree's,
    and some of them are not the lowest tied id; on the tiles and on the thread-per-query kernels"""
    pts, c = lattice()
    occ, zones = free_map()
    prm, oprm = build(ctx, occ, zones, P.DOOR, pts, max_step=0.2)
    h = c[1] - c[0]
    centres = [(x + h / 2, y + h / 2) for x in c[:-1] for y in c[:-1]]
    mids = [(x + h / 2, y) for x in c[:-1] for y in c] + [(x, y + h / 2) for x in c for y in c[:-1]]
    q = np.array(centres + mids)
    rng = np.random.default_rng(9)
    starts = np.ascontiguousarray(np.concatenate([q, q]))
    goals = np.ascontiguousarray(starts[rng.permutation(len(starts))])
    assert 2 * len(starts) >= 2048
    d2 = ((starts[:, None, :] - pts[None, :, :]) ** 2).sum(-1)
    ties = (d2 == d2.min(1, keepdims=True)).sum(1)
    assert ties.min() >= 2
    res = prm.plan_paths(starts, goals)
    want = np.array([oprm.kdtree.nearest_neighbor(s) for s in starts])
    np.testing.assert_array_equal(res[3], want)
    lowest = np.array([np.flatnonzero(row == row.min())[0] for row in d2])
    assert (res[3] != lowest).any()
    same(res, with_option(ctx, P.OPT_FORCE_THREAD_PER_QUERY_NN, 1, lambda: prm.plan_paths(starts, goals)))
    check_oracle(oprm, starts, goals, res, queries=range(0, len(starts), 13))


def test_walk_takes_the_first_of_equal_minima(ctx):
    """a 4-connected dyadic lattice: between opposite corners every monotone route has the same cost, so the walk meets exact equal
    minima and must keep the first in stored order"""
    pts, c = lattice(n=12)
    occ, zones = free_map()
    prm, oprm = build(ctx, occ, zones, P.DOOR, pts, max_step=0.15, search_radius=50.0)
    xy, _, rp, col, _ = oprm.graph.export(1)
    corners = np.array([(c[0], c[0]), (c[-1], c[-1]), (c[0], c[-1]), (c[-1], c[0]), (c[2], c[3]), (c[9], c[7])])
    starts = np.ascontiguousarray(np.repeat(corners, len(corners), axis=0))
    goals = np.ascontiguousarray(np.tile(corners, (len(corners), 1)))
    res = prm.plan_paths(starts, goals)
    met = False
    for q in range(len(starts)):
        cost = oprm.graph.dijkstra([res[4][q]])
        path, tie = restated_walk(rp, col, xy, cost, res[3][q])
        met |= tie
        np.testing.assert_array_equal(res[0][q], xy[path])
    assert met
    check_oracle(oprm, starts, goals, res)


def test_no_path(ctx):
    """a full wall between start and goal: status NONE, empty path, cost +inf (the oracle returns no path either); a sample inside
    the wall is an isolated node"""
    occ = np.full((256, 256), 255, np.uint8)
    occ[:, 120:136] = 0
    zones = None
    rng = np.random.default_rng(4)
    samples = rng.uniform(-1.0, 1.0, (1500, 2))
    samples[700] = (0.0, 0.3)                       # inside the wall
    prm, oprm = build(ctx, occ, zones, P.DOOR, samples)
    starts = np.array([(-0.6, 0.1), (-0.5, -0.5), (0.0, 0.3), (0.6, 0.6), (-0.7, 0.7)])
    goals = np.array([(0.6, 0.1), (-0.2, 0.5), (-0.5, -0.5), (0.5, -0.6), (0.0, 0.3)])
    res = prm.plan_paths(starts, goals)
    np.testing.assert_array_equal(res[2], [P.PATH_NONE, P.PATH_FOUND, P.PATH_NONE, P.PATH_FOUND, P.PATH_NONE])
    assert res[3][2] == 700 and res[4][4] == 700
    for q in (0, 2, 4):
        assert np.isinf(res[1][q]) and res[0][q].shape == (0, 2) and len(oprm.plan_path(starts[q], goals[q])) == 0
    check_oracle(oprm, starts, goals, res)
    assert prm.plan_path(starts[0], goals[0]).shape == (0, 2)


def test_cycle_through_duplicate_samples(ctx):
    """samples A, A', P, ... with A' a duplicate of A: the first minimum at A is A' and at A' it is A, the reference's walk never ends.
    Status CYCLE (checked against the restated walk with a step guard); the other queries of the call equal the oracle"""
    occ, zones = free_map()
    rng = np.random.default_rng(6)
    A = (-0.7, -0.7)
    rest = rng.uniform(-1.0, 1.0, (1200, 2))
    rest[0] = (-0.68, -0.69)
    samples = np.ascontiguousarray(np.vstack([[A, A], rest]))
    prm, oprm = build(ctx, occ, zones, P.DOOR, samples)
    xy, _, rp, col, _ = oprm.graph.export(1)
    assert col[rp[0]] == 1 and col[rp[1]] == 0
    starts = np.ascontiguousarray(np.vstack([[A, (-0.69, -0.71)], rng.uniform(-1.0, 1.0, (30, 2))]))
    goals = np.ascontiguousarray(np.vstack([[(0.7, 0.6), (0.5, -0.2)], rng.uniform(-1.0, 1.0, (30, 2))]))
    res = prm.plan_paths(starts, goals)
    fine = []
    for q in range(len(starts)):
        cost = oprm.graph.dijkstra([res[4][q]])
        path, _ = restated_walk(rp, col, xy, cost, res[3][q])
        if path is None:
            assert res[2][q] == P.PATH_CYCLE and res[0][q].shape == (0, 2) and res[1][q] == cost[res[3][q]], q
        else:
            fine.append(q)
    assert res[2][0] == P.PATH_CYCLE and res[3][0] == 0
    assert len(fine) >= 20
    check_oracle(oprm, starts, goals, res, queries=fine)
    assert prm.plan_path(starts[0], goals[0]).shape == (0, 2)


# ---------------------------------------------------------------------------------------------------------------- call shape
@pytest.fixture(scope="module")
def door_prm(ctx):
    occ, zones = util.small_door_map(seed=11)
    rng = np.random.default_rng(21)
    samples = rng.uniform(-1.0, 1.0, (2500, 2))
    omap, pmap = util.make_pair(ctx, occ, zones, P.DOOR, 0.5)
    starts, goals = queries_512(samples, rng)
    return pmap, samples, starts, goals


def test_chunking_and_query_order(ctx, door_prm):
    """5 goal columns per chunk (32 distinct goals: 7 chunks) == calls that each fit one chunk; a permutation of the queries gives
    the permuted results"""
    pmap, samples, starts, goals = door_prm
    prm = P.PRM(pmap).grow_graph(samples, MS, SR)
    whole = prm.plan_paths(starts, goals)
    chunked = with_option(ctx, P.OPT_PRM_PATHS_CHUNK_COLUMNS, 5, lambda: prm.plan_paths(starts, goals))
    same(whole, chunked)
    gcol = np.unique(whole[4], return_inverse=True)[1]
    parts = [np.flatnonzero(gcol // 5 == k) for k in range(gcol.max() // 5 + 1)]
    split = [prm.plan_paths(starts[ix], goals[ix]) for ix in parts]
    for ix, r in zip(parts, split):
        same(r, permuted(whole, ix))
    perm = np.random.default_rng(2).permutation(len(starts))
    same(with_option(ctx, P.OPT_PRM_PATHS_CHUNK_COLUMNS, 3, lambda: prm.plan_paths(starts[perm], goals[perm])), permuted(whole, perm))


def raw_call(ctx, starts, goals, n, cap, total):
    m = max(n, 1)
    sn, gn, st, cost = np.empty(m, np.int32), np.empty(m, np.int32), np.empty(m, np.int32), np.empty(m)
    ptr, xy = np.empty(max(n, 0) + 1, np.int64), np.empty((max(cap, 1), 2))
    rc = ctx.lib.porrt_prm_plan_paths(ctx.h, P.api._p(starts), P.api._p(goals), n, P.api._p(sn), P.api._p(gn), P.api._p(cost),
                                      P.api._p(st), P.api._p(ptr), P.api._p(xy), cap, C.byref(total))
    return rc, (sn, gn, st, cost, ptr, xy)


def test_capacity_then_fetch(ctx, door_prm):
    pmap, samples, starts, goals = door_prm
    prm = P.PRM(pmap).grow_graph(samples, MS, SR)
    want = prm.plan_paths(starts, goals)
    need = sum(len(p) for p in want[0])
    total = C.c_int64()
    rc, (sn, gn, st, cost, ptr, _) = raw_call(ctx, starts, goals, len(starts), need - 1, total)
    assert rc == P.api.ERR_CAPACITY and total.value == need and ptr[-1] == need
    np.testing.assert_array_equal(cost, want[1])
    np.testing.assert_array_equal(st, want[2])
    np.testing.assert_array_equal(sn, want[3])
    rc, (sn, gn, st, cost, ptr, xy) = raw_call(ctx, starts, goals, len(starts), need, total)
    assert rc == 0 and total.value == need
    for q in range(len(starts)):
        np.testing.assert_array_equal(xy[ptr[q]:ptr[q + 1]], want[0][q])
    rc, (_, _, _, _, ptr, _) = raw_call(ctx, starts[:0], goals[:0], 0, 0, total)
    assert rc == 0 and total.value == 0 and ptr[0] == 0


def test_argument_errors(ctx, door_prm):
    pmap, samples, starts, goals = door_prm
    total = C.c_int64()
    fresh = P.Context(0)
    try:
        assert raw_call(fresh, starts, goals, 4, 1000, total)[0] == 1           # nothing built
    finally:
        fresh.close()
    prm = P.PRM(pmap).grow_graph(samples, MS, SR)
    assert raw_call(ctx, starts, goals, 4, 1000, total)[0] == 0
    assert raw_call(ctx, starts, goals, -1, 1000, total)[0] == 1
    for bad in (np.nan, np.inf, -np.inf):
        s = starts.copy()
        s[2, 1] = bad
        assert raw_call(ctx, s, goals, 4, 1000, total)[0] == 1
        g = goals.copy()
        g[3, 0] = bad
        assert raw_call(ctx, starts, g, 4, 1000, total)[0] == 1
    P.KdTree(ctx, samples)                                                        # porrt_vertices_set
    assert raw_call(ctx, starts, goals, 4, 1000, total)[0] == 1
    prm = P.PRM(pmap).grow_graph(samples, MS, SR)
    assert raw_call(ctx, starts, goals, 4, 1000, total)[0] == 0
    xy = np.ascontiguousarray(np.array([[0.5, 0.5]]))
    ctx.check(ctx.lib.porrt_vertices_append(ctx.h, P.api._p(xy), 1))
    assert raw_call(ctx, starts, goals, 4, 1000, total)[0] == 1
    socc, szones = synth.shelf_map(200, n_zones=2)
    omap, smap = util.make_pair(ctx, socc, szones, P.SHELF, 0.5)
    tamp = O.TampPRM(omap, util.LOW, util.UP)
    tamp.plan((-0.9, 0.0), [0.5, 0.5], 0.1, 2.0, 2500)
    P.mmprm_plan(smap, tamp.schedule())
    assert raw_call(ctx, starts, goals, 4, 1000, total)[0] == 1                  # the grouped build of porrt_mmprm_plan
    P.PRM(smap).grow_graph(samples, MS, SR)
    assert raw_call(ctx, starts, goals, 4, 1000, total)[0] == 0
