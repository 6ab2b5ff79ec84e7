"""PTO::plan_belief_space on every roadmap of a PTO seed batch in one device call (porrt_pto_plan_batch / PTOBatch.plan_belief_space)
against the single-roadmap path on the same grown batch: porrt_pto_fetch_roadmap -> plan_belief_space (porrt_visibility,
porrt_belief_vi, porrt_extract_policy).  Policy nodes, beliefs, parents, leaves and the expected cost must be identical, and each
roadmap's status must be the code the single path fails with.  On the door map the oracle's own grow -> plan_belief_space ->
extract_policy is the reference as well."""
import ctypes as C

import numpy as np
import pytest

from oracle import pyoracle as O
import po_rrt_b200 as P
from po_rrt_b200 import synth
import porrt_testutil as util

pytestmark = pytest.mark.gpu

_p = P.api._p
DOOR_GOAL = [((0.8, 0.8), [1, 1, 1, 1])]
DOOR = dict(start=(-0.8, -0.8), goals=DOOR_GOAL, max_step=0.05, search_radius=5.0, n_min=700, n_max=100000)
DOOR_B0 = [0.1, 0.1, 0.1, 0.7]
CONFIG3 = dict(start=(0.0, -0.9), max_step=0.1, search_radius=2.0, n_min=5000, n_max=100000)
CONFIG4 = dict(start=(0.0, -0.9), max_step=0.05, search_radius=5.0, n_min=5000, n_max=100000)
# colsolve_fits: V * 9 + 280 + 2 * COLSOLVE_QCAP bytes of shared memory at most COLSOLVE_SMEM_MAX (227 KB)
ON_CHIP_MAX_V = (227 * 1024 - 280 - 2 * 1024) // 9


@pytest.fixture(scope="module")
def ctx():
    c = P.Context(0)
    yield c
    c.close()


@pytest.fixture
def door(ctx):
    occ, zones = util.planning_door_map(200)
    return util.make_pair(ctx, occ, zones, P.DOOR, 0.3)


def _shelf(ctx, Z, visibility):
    occ, zones = synth.shelf_map(200, n_rects=10, n_zones=Z, seed=5)
    omap, pmap = util.make_pair(ctx, occ, zones, P.SHELF, visibility)
    zp = omap.zone_positions()
    goals = [((float(zp[z][0]) - 0.08, float(zp[z][1])), [1 if k == z else 0 for k in range(Z)]) for z in range(Z)]
    return omap, pmap, goals


def _grow(pmap, seeds, start, goals, max_step, search_radius, n_min, n_max):
    dev = P.PTOBatch(pmap, util.LOW, util.UP, seeds)
    status = dev.grow_graph(start, P.SquareGoal(goals, 0.05), max_step, search_radius, n_min, n_max)
    return dev, status


def _single(pmap, dev, grow_status, r, b0, beliefs):
    """the single path on roadmap r -> a BeliefPlan, or the PorrtError code it fails with"""
    if grow_status[r] == 5:
        return 5                                   # its growth panicked: nothing to fetch
    xy, nvid, rp, col, ev = dev.graph_arrays(r)
    ids, masks = dev.finals(r)
    try:
        return P.plan_belief_space(pmap, rp, col, ev, xy, nvid, b0, ids, masks, beliefs=beliefs, copy=None)
    except P.PorrtError as e:
        return e.code


def _assert_plan_equal(got, want, r):
    np.testing.assert_array_equal(got.policy_node, want.policy_node, err_msg="roadmap %d" % r)
    np.testing.assert_array_equal(got.policy_belief, want.policy_belief, err_msg="roadmap %d" % r)
    np.testing.assert_array_equal(got.policy_parent, want.policy_parent, err_msg="roadmap %d" % r)
    np.testing.assert_array_equal(got.policy_leaf, want.policy_leaf, err_msg="roadmap %d" % r)
    assert got.expected_cost == want.expected_cost, (r, got.expected_cost, want.expected_cost)


def _assert_equals_single(pmap, dev, grow_status, plans, b0):
    """every roadmap's batch result is the single path's; -> the single path's results"""
    beliefs = plans[0].beliefs
    assert len(plans) == len(dev)
    singles = []
    for r in range(len(dev)):
        want = _single(pmap, dev, grow_status, r, b0, beliefs)
        singles.append(want)
        got = plans[r]
        if isinstance(want, int):
            assert got.status == want, (r, got.status, want)
            assert len(got.policy_node) == 0 and np.isnan(got.expected_cost)
        else:
            assert got.status == 0, (r, got.status)
            _assert_plan_equal(got, want, r)
    return singles


def _plan_all(pmap, dev, grow_status, b0):
    plans = dev.plan_belief_space(b0)
    singles = _assert_equals_single(pmap, dev, grow_status, plans, b0)
    return plans, singles


# ---- against the oracle and the single path

def test_door_map_four_seeds_equal_the_oracle(ctx, door):
    omap, pmap = door
    seeds = [0, 1, 7, 123]
    dev, gs = _grow(pmap, seeds, **DOOR)
    plans, _ = _plan_all(pmap, dev, gs, DOOR_B0)
    for r, s in enumerate(seeds):
        ref = O.PTO(omap, util.LOW, util.UP, seed=s)
        assert ref.grow_graph(DOOR["start"], O.SquareGoal(DOOR_GOAL, 0.05), DOOR["max_step"], DOOR["search_radius"], DOOR["n_min"],
                              DOOR["n_max"]) == 0
        ref.build_belief_graph(DOOR_B0)
        ref.compute_expected_costs_to_goals()
        opol = ref.extract_policy()
        B = len(plans[r].beliefs)
        np.testing.assert_array_equal(plans[r].beliefs, ref.beliefs())
        np.testing.assert_array_equal(plans[r].policy_node.astype(np.int64) * B + plans[r].policy_belief, opol.original)
        np.testing.assert_array_equal(plans[r].policy_parent.astype(np.int64), opol.parent)
        np.testing.assert_array_equal(np.nonzero(plans[r].policy_leaf)[0], opol.leafs)
        assert plans[r].expected_cost == opol.expected_costs
        assert plans[r].policy_leaf.sum() >= 2


def test_config3_shape_eight_seeds(ctx):
    """8 shelves, b0 uniform: B = 255, levels of up to C(8, 4) = 70 columns"""
    _, pmap, goals = _shelf(ctx, 8, 0.5)
    dev, gs = _grow(pmap, list(range(8)), goals=goals, **CONFIG3)
    plans, _ = _plan_all(pmap, dev, gs, [1.0 / 8] * 8)
    assert len(plans[0].beliefs) == 255
    assert all(p.status == 0 and np.isfinite(p.expected_cost) for p in plans)
    assert len({len(p.policy_node) for p in plans}) > 1          # different roadmaps, different policies


def test_config4_shape_three_seeds(ctx):
    """12 shelves: B = 4095, wide levels that put several columns on one CTA.  (Seed 3's policy walk does not end within a minute,
    on the single path as in the batch: the reference's walk would not end at all, and the guard stops it only after 64 V B policy
    nodes, so it is left out.)"""
    _, pmap, goals = _shelf(ctx, 12, 0.2)
    dev, gs = _grow(pmap, [0, 1, 2], goals=goals, **CONFIG4)
    plans, _ = _plan_all(pmap, dev, gs, [1.0 / 12] * 12)
    assert len(plans[0].beliefs) == 4095


def test_roadmaps_of_different_sizes_one_beyond_the_column_solver(ctx, door):
    """a long growth puts the roadmaps' V on both sides of the column solver's limit: the large ones take the frontier schedule on
    their own, the others share the batched launches"""
    _, pmap = door
    seeds = list(range(8))
    kw = dict(DOOR, n_min=27000)
    for _ in range(4):
        dev, gs = _grow(pmap, seeds, **kw)
        V = dev.sizes[:, 1]
        if (V > ON_CHIP_MAX_V).any() and (V <= ON_CHIP_MAX_V).any():
            break
        kw["n_min"] += int(ON_CHIP_MAX_V - np.median(V))
    assert (V > ON_CHIP_MAX_V).any() and (V <= ON_CHIP_MAX_V).any(), V
    assert len(set(V.tolist())) > 1
    _plan_all(pmap, dev, gs, DOOR_B0)


def test_forced_frontier_schedule_equals_the_column_solver(ctx):
    _, pmap, goals = _shelf(ctx, 8, 0.5)
    dev, gs = _grow(pmap, [3, 4, 5], goals=goals, **CONFIG3)
    b0 = [1.0 / 8] * 8
    plans = dev.plan_belief_space(b0)
    ctx.set_option(P.OPT_FORCE_GLOBAL_SWEEPS, 1)
    try:
        forced = dev.plan_belief_space(b0)
        _assert_equals_single(pmap, dev, gs, forced, b0)
    finally:
        ctx.set_option(P.OPT_FORCE_GLOBAL_SWEEPS, 0)
    for r in range(len(dev)):
        _assert_plan_equal(forced[r], plans[r], r)
    _assert_equals_single(pmap, dev, gs, plans, b0)


def test_failures_mixed_with_other_roadmaps(ctx):
    """door pixels whose zone id alternates row by row: some growths panic, the others stop early.  Every roadmap's status is the
    single path's code, and the roadmaps whose growth did not panic get the same results in a batch of their own."""
    occ, zones = util.planning_door_map(200)
    door = zones != 255
    zones[door] = (np.nonzero(door)[0] % 2).astype(np.uint8)
    _, pmap = util.make_pair(ctx, occ, zones, P.DOOR, 0.3)
    seeds = list(range(12))
    for n in (25, 50, 100, 200, 400, 800):
        dev, gs = _grow(pmap, seeds, start=(-0.8, -0.8), goals=DOOR_GOAL, max_step=0.05, search_radius=5.0, n_min=n, n_max=n)
        if (gs == 5).any() and (gs != 5).any():
            break
    assert (gs == 5).any() and (gs != 5).any(), gs
    plans, _ = _plan_all(pmap, dev, gs, DOOR_B0)
    assert all(plans[r].status == 5 for r in range(len(dev)) if gs[r] == 5)
    others = [r for r in range(len(dev)) if gs[r] != 5]
    dev2, _ = _grow(pmap, [seeds[r] for r in others], start=(-0.8, -0.8), goals=DOOR_GOAL, max_step=0.05, search_radius=5.0, n_min=n,
                    n_max=n)
    alone = dev2.plan_belief_space(DOOR_B0)
    for k, r in enumerate(others):
        assert alone[k].status == plans[r].status, (r, alone[k].status, plans[r].status)
        if plans[r].status == 0:
            _assert_plan_equal(alone[k], plans[r], r)


def test_incomplete_final_set_is_planned(ctx, door):
    """roadmaps stopped before every world reaches a final are planned as porrt_belief_vi plans them"""
    _, pmap = door
    seeds = list(range(6))
    dev, gs = _grow(pmap, seeds, start=(-0.8, -0.8), goals=DOOR_GOAL, max_step=0.05, search_radius=5.0, n_min=50, n_max=150)
    assert (gs == 1).any(), gs
    _plan_all(pmap, dev, gs, DOOR_B0)


# ---- call behaviour

def test_batch_of_one(ctx, door):
    _, pmap = door
    dev, gs = _grow(pmap, [5], **DOOR)
    plans, _ = _plan_all(pmap, dev, gs, DOOR_B0)
    assert len(plans) == 1 and plans[0].status == 0


def test_same_seed_twice_gives_identical_policies(ctx, door):
    _, pmap = door
    dev, gs = _grow(pmap, [3, 9, 3], **DOOR)
    plans, _ = _plan_all(pmap, dev, gs, DOOR_B0)
    _assert_plan_equal(plans[0], plans[2], 2)


def _raw(c, beliefs, B, n_worlds, R, cap, status=True, total=True, ptr=True):
    st, cost, pp = np.full(R, -7, np.int32), np.zeros(R), np.zeros(R + 1, np.int64)
    out = np.zeros(max(cap, 1), np.int32), np.zeros(max(cap, 1), np.int32), np.zeros(max(cap, 1), np.int32), np.zeros(max(cap, 1), np.uint8)
    tot = C.c_int64(-1)
    rc = c.lib.porrt_pto_plan_batch(c.h, _p(beliefs) if beliefs is not None else None, B, n_worlds, _p(st) if status else None, _p(cost),
                                    _p(pp) if ptr else None, *(_p(a) for a in out), cap, C.byref(tot) if total else None, None, None)
    return rc, st, cost, pp, tot.value


def test_capacity_too_small(ctx, door):
    _, pmap = door
    dev, gs = _grow(pmap, [0, 1, 2], **DOOR)
    plans = dev.plan_belief_space(DOOR_B0)
    bel = plans[0].beliefs
    rc, st, cost, pp, tot = _raw(ctx, bel, len(bel), pmap.n_worlds(), 3, 0)
    assert rc == 4
    assert tot == sum(len(p.policy_node) for p in plans) and pp[-1] == tot
    np.testing.assert_array_equal(np.diff(pp), [len(p.policy_node) for p in plans])
    assert (st == 0).all() and list(cost) == [p.expected_cost for p in plans]
    rc, st, cost, pp, tot = _raw(ctx, bel, len(bel), pmap.n_worlds(), 3, tot - 1)
    assert rc == 4
    rc, *_ = _raw(ctx, bel, len(bel), pmap.n_worlds(), 3, tot)
    assert rc == 0


def test_argument_errors(ctx):
    occ, zones = util.planning_door_map(200)
    c2 = P.Context(0)
    try:
        m2 = P.Map(c2, occ, util.LOW, util.UP)
        bel = np.array([DOOR_B0])
        assert _raw(c2, bel, 1, 4, 1, 16)[0] == 3                        # no map
        m2.add_zones(zones, 0.3)
        bel = m2.reachable_belief_states(DOOR_B0)
        B = len(bel)
        assert _raw(c2, bel, B, 4, 1, 16)[0] == 1                        # nothing grown yet
        dev, gs = _grow(m2, [0, 1], **DOOR)
        assert _raw(c2, bel, B, 4, 2, 4096)[0] == 0
        assert _raw(c2, bel, B, 3, 2, 4096)[0] == 1                      # n_worlds differs from the map's
        assert _raw(c2, bel, 0, 4, 2, 4096)[0] == 1                      # B <= 0
        assert _raw(c2, bel, -1, 4, 2, 4096)[0] == 1
        assert _raw(c2, None, B, 4, 2, 4096)[0] == 1                     # null beliefs
        assert _raw(c2, bel, B, 4, 2, 4096, status=False)[0] == 1
        assert _raw(c2, bel, B, 4, 2, 4096, total=False)[0] == 1
        assert _raw(c2, bel, B, 4, 2, 4096, ptr=False)[0] == 1
        dup = np.concatenate([bel, bel[1:2]])                             # two beliefs with one hash
        assert _raw(c2, dup, B + 1, 4, 2, 4096)[0] == 5
    finally:
        c2.close()


def test_previous_belief_vi_result_is_kept(ctx, door):
    _, pmap = door
    dev, gs = _grow(pmap, [0, 1], **DOOR)
    xy, nvid, rp, col, ev = dev.graph_arrays(1)
    ids, masks = dev.finals(1)
    plan = P.plan_belief_space(pmap, rp, col, ev, xy, nvid, [0.25] * 4, ids, masks)
    batch = dev.plan_belief_space(DOOR_B0)
    assert batch[0].status == 0 and not np.array_equal(batch[0].beliefs, plan.beliefs)   # the batch planned other beliefs in between
    pd, pt, V, B = C.POINTER(C.c_double)(), C.POINTER(C.c_uint8)(), C.c_int64(), C.c_int32()
    ctx.check(ctx.lib.porrt_belief_result(ctx.h, C.byref(pd), C.byref(pt), C.byref(V), C.byref(B)))
    assert (V.value, B.value) == plan.dist.shape
    np.testing.assert_array_equal(np.ctypeslib.as_array(pd, shape=plan.dist.shape), plan.dist)
    np.testing.assert_array_equal(np.ctypeslib.as_array(pt, shape=plan.type.shape), plan.type)
    cap = len(plan.policy_node)
    node, belief, parent = (np.empty(cap, np.int32) for _ in range(3))
    leaf = np.empty(cap, np.uint8)
    n, cost = C.c_int64(), C.c_double()
    ctx.check(ctx.lib.porrt_extract_policy(ctx.h, _p(node), _p(belief), _p(parent), _p(leaf), cap, C.byref(n), C.byref(cost)))
    assert n.value == cap and cost.value == plan.expected_cost
    np.testing.assert_array_equal(node, plan.policy_node)
    np.testing.assert_array_equal(parent, plan.policy_parent)
