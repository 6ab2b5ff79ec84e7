"""PTO::grow_graph on the device (porrt_pto_grow, speculative windows with an in-order commit) against the oracle's sequential
growth on the same map and seeds: iterations, return code, the whole roadmap, reachability and final nodes must be identical."""
import numpy as np
import pytest

from oracle import pyoracle as O
import po_rrt_b200 as P
from po_rrt_b200 import synth
import porrt_testutil as util

pytestmark = pytest.mark.gpu
COUNTERS = []          # (windows, respeculated, conflicts nn, conflicts radius / kd) of every grown case, for the counter test


@pytest.fixture(scope="module")
def ctx():
    c = P.Context(0)
    yield c
    c.close()


def _grow_both(omap, pmap, start, goals, max_step, search_radius, n_min, n_max=100000, seed=0, max_dist=0.05):
    ref = O.PTO(omap, util.LOW, util.UP, seed=seed)
    want_rc = ref.grow_graph(start, O.SquareGoal(goals, max_dist), max_step, search_radius, n_min, n_max)
    dev = P.PTO(pmap, util.LOW, util.UP, seed=seed)
    return ref, want_rc, dev, P.SquareGoal(goals, max_dist)


def _compare(omap, pmap, start, goals, max_step, search_radius, n_min, n_max=100000, seed=0):
    ref, want_rc, dev, goal = _grow_both(omap, pmap, start, goals, max_step, search_radius, n_min, n_max, seed)
    assert want_rc in (0, 1), want_rc
    got_rc = dev.grow_graph(start, goal, max_step, search_radius, n_min, n_max)
    assert got_rc == want_rc and dev.n_it == ref.n_it()
    want = ref.graph.export(0)
    for a, b in zip(dev.graph_arrays(), want):
        np.testing.assert_array_equal(a, b)
    V = len(want[0])
    np.testing.assert_array_equal(dev.reach_masks(), ref.reach.all(V))
    ids, masks = dev.finals()
    oids, obits = ref.reach.finals()
    np.testing.assert_array_equal(ids, oids)
    np.testing.assert_array_equal(masks, P.words_from_bits(obits) if len(obits) else masks)
    COUNTERS.append(dev.counters)
    return ref, dev


def _door(ctx):
    occ, zones = util.planning_door_map(200)
    return util.make_pair(ctx, occ, zones, P.DOOR, 0.3)


def _shelf(ctx, Z, visibility):
    occ, zones = synth.shelf_map(200, n_rects=10, n_zones=Z, seed=5)
    omap, pmap = util.make_pair(ctx, occ, zones, P.SHELF, visibility)
    zp = omap.zone_positions()
    goals = [((float(zp[z][0]) - 0.08, float(zp[z][1])), [1 if k == z else 0 for k in range(Z)]) for z in range(Z)]
    return omap, pmap, goals


DOOR_GOAL = [((0.8, 0.8), [1, 1, 1, 1])]


def test_door_map(ctx):
    omap, pmap = _door(ctx)
    _compare(omap, pmap, (-0.8, -0.8), DOOR_GOAL, 0.05, 5.0, 700)


@pytest.mark.parametrize("seed", [1, 7, 123])
def test_door_map_other_seeds(ctx, seed):
    omap, pmap = _door(ctx)
    _compare(omap, pmap, (-0.8, -0.8), DOOR_GOAL, 0.05, 5.0, 700, seed=seed)


def test_shelf_config2(ctx):
    occ, zones = synth.shelf_map(200, n_zones=2)
    omap, pmap = util.make_pair(ctx, occ, zones, P.SHELF, 0.5)
    zp = omap.zone_positions()
    goals = [((float(zp[0][0]) - 0.06, float(zp[0][1])), [1, 0]), ((float(zp[1][0]) - 0.06, float(zp[1][1])), [0, 1])]
    _compare(omap, pmap, (-0.8, -0.8), goals, 0.05, 5.0, 2000)


def test_shelf_config3_shape(ctx):
    omap, pmap, goals = _shelf(ctx, 8, 0.5)
    _compare(omap, pmap, (0.0, -0.9), goals, 0.1, 2.0, 5000)


def test_shelf_config4_shape(ctx):
    omap, pmap, goals = _shelf(ctx, 12, 0.2)
    _compare(omap, pmap, (0.0, -0.9), goals, 0.05, 5.0, 5000)


def test_seven_door_zones_two_mask_words(ctx):
    occ, zones = synth.door_map(size=1024, n_rects=1500, n_zones=7, seed=23)
    omap, pmap = util.make_pair(ctx, occ, zones, P.DOOR, 0.3)
    assert pmap.mask_words == 2
    _compare(omap, pmap, (-0.8, -0.8), [((0.8, 0.8), [1] * 128)], 0.05, 5.0, 2500)


def test_truncated_growth_is_incomplete(ctx):
    """n_iter_max too small to reach the goal: return code 1 and the same truncated roadmap"""
    omap, pmap = _door(ctx)
    ref, dev = _compare(omap, pmap, (-0.8, -0.8), DOOR_GOAL, 0.05, 5.0, 50, n_max=120)
    assert dev.n_it == 120 and not ref.reach.is_final_set_complete()


def test_exact_duplicate_states(ctx):
    """every 100th sample is the goal itself (goal_example); once a node sits on the goal, later goal samples steer onto it
    exactly: chains of exact duplicates in the kd-tree exercise the tie replay and the unbounded pre-order keys"""
    omap, pmap = _door(ctx)
    ref, dev = _compare(omap, pmap, (0.7, 0.7), DOOR_GOAL, 0.2, 5.0, 3000)
    xy = ref.graph.export(0)[0]
    _, counts = np.unique(xy, axis=0, return_counts=True)
    assert counts.max() >= 3


def test_counters(ctx):
    """the window / commit scheme really runs: conflicts of both kinds occur and windows cover many iterations each"""
    if len(COUNTERS) < 5:
        pytest.skip("runs after the growth cases of this module")
    tot = np.sum(np.array(COUNTERS), axis=0)
    assert tot[1] > 0 and tot[2] > 0 and tot[3] > 0
    omap, pmap, goals = _shelf(ctx, 8, 0.5)
    _, dev = _compare(omap, pmap, (0.0, -0.9), goals, 0.1, 2.0, 5000)
    assert dev.counters[0] * 4 < dev.n_it


def test_panics_like_the_reference(ctx):
    omap, pmap = _door(ctx)
    # a start inside an obstacle: expect("Start from a valid state!")
    ref, want_rc, dev, goal = _grow_both(omap, pmap, (-1.0, 0.0), DOOR_GOAL, 0.05, 5.0, 100)
    assert want_rc == -100
    with pytest.raises(P.PorrtError) as e:
        dev.grow_graph((-1.0, 0.0), goal, 0.05, 5.0, 100, 1000)
    assert e.value.code == 5 and e.value.panic_code == P.INVALID and dev.n_it == 0
    # door pixels whose zone id alternates row by row: an edge through a door crosses two zones and panics
    # ("multiple zone traversal not supported", map_io.rs:233)
    occ, zones = util.planning_door_map(200)
    door = zones != 255
    zones[door] = (np.nonzero(door)[0] % 2).astype(np.uint8)
    omap2, pmap2 = util.make_pair(ctx, occ, zones, P.DOOR, 0.3)
    ref, want_rc, dev, goal = _grow_both(omap2, pmap2, (-0.8, -0.8), DOOR_GOAL, 0.05, 5.0, 3000)
    assert want_rc < -1
    with pytest.raises(P.PorrtError) as e:
        dev.grow_graph((-0.8, -0.8), goal, 0.05, 5.0, 3000, 100000)
    assert e.value.code == 5 and e.value.panic_code == want_rc


def test_argument_errors(ctx):
    occ, zones = util.planning_door_map(200)
    c2 = P.Context(0)
    try:
        pmap = P.Map(c2, occ, util.LOW, util.UP)       # not uploaded yet
        lib = c2.lib
        sizes = np.zeros(4, np.int64)
        goal = P.SquareGoal(DOOR_GOAL, 0.05)
        start, low, up = (np.array(v, np.float64) for v in ((-0.8, -0.8), util.LOW, util.UP))
        import ctypes as C
        cpl, fl = C.c_int32(), C.c_int32()
        args = lambda s: (c2.h, P.api._p(s), P.api._p(low), P.api._p(up), 0, P.api._p(goal.goals), P.api._p(goal.masks), 1, 0.05,
                          0.05, 5.0, 10, 100, P.api._p(sizes), C.byref(cpl), C.byref(fl), None)
        assert lib.porrt_pto_grow(*args(start)) == 3                                       # no map
        assert lib.porrt_pto_fetch(c2.h, None, None, None, None, None, None, None, None) == 1   # fetch before any grow
        pmap.add_zones(zones, 0.3)
        assert lib.porrt_pto_grow(*args(None)) == 1                                        # null start
        a = list(args(start)); a[11] = -1
        assert lib.porrt_pto_grow(*a) == 1                                                 # negative n_iter_min
        a = list(args(start)); a[7] = -1
        assert lib.porrt_pto_grow(*a) == 1                                                 # n_goals < 0
        bad = np.array([[0xF], [0x3]], np.uint64)                                          # overlapping goal masks
        two = np.array([[0.8, 0.8], [0.5, 0.5]])
        a = list(args(start)); a[5] = P.api._p(two); a[6] = P.api._p(bad); a[7] = 2
        assert lib.porrt_pto_grow(*a) == 5
    finally:
        c2.close()


def test_device_roadmap_feeds_belief_planning(ctx):
    """config-3 shape end to end: the device-grown roadmap into plan_belief_space equals the oracle's whole belief pipeline"""
    import test_gpu_parity as T
    omap, pmap, goals = _shelf(ctx, 8, 0.5)
    ref, dev = _compare(omap, pmap, (0.0, -0.9), goals, 0.1, 2.0, 5000)
    xy, nvid, rp, col, ev = dev.graph_arrays()
    ids, masks = dev.finals()
    b0 = [1.0 / 8] * 8
    plan = P.plan_belief_space(pmap, rp, col, ev, xy, nvid, b0, ids, masks)
    oplan, want, typ = T._belief_compare(ctx, omap, pmap, ref, b0)
    np.testing.assert_array_equal(plan.dist, oplan.dist)
    np.testing.assert_array_equal(plan.policy_node, oplan.policy_node)
    np.testing.assert_array_equal(plan.policy_parent, oplan.policy_parent)
    assert plan.expected_cost == oplan.expected_cost and np.isfinite(want[0])
