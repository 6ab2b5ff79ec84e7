"""PTO::grow_graph for a batch of sampler seeds in one device call (porrt_pto_grow_batch / PTOBatch) against the oracle's sequential
growth with each seed on the same map: iterations, return code, the whole roadmap, reachability and final nodes of every roadmap
must be identical; against porrt_pto_grow with the same seed, the window counters too."""
import numpy as np
import pytest

from oracle import pyoracle as O
import po_rrt_b200 as P
from po_rrt_b200 import synth
import porrt_testutil as util

pytestmark = pytest.mark.gpu

DOOR_GOAL = [((0.8, 0.8), [1, 1, 1, 1])]
DOOR = dict(start=(-0.8, -0.8), goals=DOOR_GOAL, max_step=0.05, search_radius=5.0, n_min=700, n_max=100000)


@pytest.fixture(scope="module")
def ctx():
    c = P.Context(0)
    yield c
    c.close()


@pytest.fixture
def door(ctx):
    """the door map, uploaded again for every test: the context holds one map at a time"""
    occ, zones = util.planning_door_map(200)
    return util.make_pair(ctx, occ, zones, P.DOOR, 0.3)


def _shelf(ctx, Z, visibility):
    occ, zones = synth.shelf_map(200, n_rects=10, n_zones=Z, seed=5)
    omap, pmap = util.make_pair(ctx, occ, zones, P.SHELF, visibility)
    zp = omap.zone_positions()
    goals = [((float(zp[z][0]) - 0.08, float(zp[z][1])), [1 if k == z else 0 for k in range(Z)]) for z in range(Z)]
    return omap, pmap, goals


CONFIG3 = dict(start=(0.0, -0.9), max_step=0.1, search_radius=2.0, n_min=5000, n_max=100000)
CONFIG4 = dict(start=(0.0, -0.9), max_step=0.05, search_radius=5.0, n_min=5000, n_max=100000)


def _oracle(omap, seed, start, goals, max_step, search_radius, n_min, n_max):
    ref = O.PTO(omap, util.LOW, util.UP, seed=seed)
    rc = ref.grow_graph(start, O.SquareGoal(goals, 0.05), max_step, search_radius, n_min, n_max)
    return ref, rc


def _batch(pmap, seeds, start, goals, max_step, search_radius, n_min, n_max):
    dev = P.PTOBatch(pmap, util.LOW, util.UP, seeds)
    status = dev.grow_graph(start, P.SquareGoal(goals, 0.05), max_step, search_radius, n_min, n_max)
    assert status.shape == (len(seeds),)
    return dev, status


def _assert_roadmap_equals_oracle(dev, status, r, ref, want_rc):
    assert want_rc in (0, 1), want_rc
    assert status[r] == want_rc and dev.n_it[r] == ref.n_it(), (r, status[r], want_rc, dev.n_it[r], ref.n_it())
    want = ref.graph.export(0)
    for a, b in zip(dev.graph_arrays(r), want):
        np.testing.assert_array_equal(a, b)
    np.testing.assert_array_equal(dev.reach_masks(r), ref.reach.all(len(want[0])))
    ids, masks = dev.finals(r)
    oids, obits = ref.reach.finals()
    np.testing.assert_array_equal(ids, oids)
    np.testing.assert_array_equal(masks, P.words_from_bits(obits) if len(obits) else masks)


def _compare(omap, pmap, seeds, **kw):
    dev, status = _batch(pmap, seeds, **kw)
    refs = []
    for r, s in enumerate(seeds):
        ref, rc = _oracle(omap, int(s), **kw)
        _assert_roadmap_equals_oracle(dev, status, r, ref, rc)
        refs.append(ref)
    return dev, status, refs


def _snapshot(dev):
    """every roadmap's arrays, read before a later growth on the same context replaces them"""
    return [(dev.graph_arrays(r), dev.reach_masks(r), dev.finals(r)) for r in range(len(dev))]


# ---- parity with the oracle

def test_door_map_four_seeds(ctx, door):
    omap, pmap = door
    _compare(omap, pmap, [0, 1, 7, 123], **DOOR)


def test_door_map_64_seeds(ctx, door):
    omap, pmap = door
    dev, status, _ = _compare(omap, pmap, list(range(64)), **DOOR)
    assert len(dev) == 64


def test_batch_of_one(ctx, door):
    omap, pmap = door
    _compare(omap, pmap, [5], **DOOR)


def test_same_seed_twice_gives_identical_roadmaps(ctx, door):
    omap, pmap = door
    dev, status, _ = _compare(omap, pmap, [3, 9, 3], **DOOR)
    assert status[0] == status[2] and tuple(dev.counters[0]) == tuple(dev.counters[2])
    for a, b in zip(dev.graph_arrays(0), dev.graph_arrays(2)):
        np.testing.assert_array_equal(a, b)
    np.testing.assert_array_equal(dev.reach_masks(0), dev.reach_masks(2))


def test_exact_duplicate_states(ctx, door):
    """start on the goal with long steps: every 100th sample (the goal) steers onto existing nodes exactly"""
    omap, pmap = door
    _, _, refs = _compare(omap, pmap, [0, 1, 2, 3], start=(0.7, 0.7), goals=DOOR_GOAL, max_step=0.2, search_radius=5.0,
                          n_min=3000, n_max=100000)
    _, counts = np.unique(refs[0].graph.export(0)[0], axis=0, return_counts=True)
    assert counts.max() >= 3


def test_some_complete_some_not(ctx, door):
    """n_iter_max between the seeds' completion iterations: the early ones finish complete, the others stop incomplete there"""
    omap, pmap = door
    seeds = list(range(8))
    kw = dict(start=(-0.8, -0.8), goals=DOOR_GOAL, max_step=0.05, search_radius=5.0, n_min=50)
    n_done = sorted(_oracle(omap, s, n_max=100000, **kw)[0].n_it() for s in seeds)
    n_max = n_done[len(seeds) // 2 - 1]
    dev, status, _ = _compare(omap, pmap, seeds, n_max=n_max, **kw)
    assert 0 < int((status == 0).sum()) < len(seeds), (n_done, status)
    assert (dev.n_it[status == 1] == n_max).all()


def test_seven_door_zones_two_mask_words(ctx):
    occ, zones = synth.door_map(size=1024, n_rects=1500, n_zones=7, seed=23)
    omap, pmap = util.make_pair(ctx, occ, zones, P.DOOR, 0.3)
    assert pmap.mask_words == 2
    _compare(omap, pmap, [0, 1, 2, 3], start=(-0.8, -0.8), goals=[((0.8, 0.8), [1] * 128)], max_step=0.05, search_radius=5.0,
             n_min=2500, n_max=100000)


@pytest.fixture
def config3(ctx):
    omap, pmap, goals = _shelf(ctx, 8, 0.5)
    seeds = list(range(8))
    dev, status, refs = _compare(omap, pmap, seeds, goals=goals, **CONFIG3)
    return omap, pmap, goals, seeds, dev, status, refs, _snapshot(dev)


def test_shelf_config3_shape_8_seeds(config3):
    _, _, _, seeds, dev, status, _, _ = config3
    assert len(dev) == len(seeds) and set(status) <= {0, 1}


def test_shelf_config4_shape_8_seeds(ctx):
    omap, pmap, goals = _shelf(ctx, 12, 0.2)
    seeds = list(range(8))
    dev, status, _ = _compare(omap, pmap, seeds, goals=goals, **CONFIG4)
    _assert_batch_equals_single(pmap, dev, status, _snapshot(dev), seeds, goals, CONFIG4)


# ---- against the single growth

def _assert_batch_equals_single(pmap, dev, status, got, seeds, goals, kw):
    for r, s in enumerate(seeds):
        one = P.PTO(pmap, util.LOW, util.UP, seed=int(s))
        rc = one.grow_graph(kw["start"], P.SquareGoal(goals, 0.05), kw["max_step"], kw["search_radius"], kw["n_min"], kw["n_max"])
        assert rc == status[r] and one.n_it == dev.n_it[r]
        assert tuple(int(x) for x in dev.sizes[r]) == one.sizes
        assert tuple(int(x) for x in dev.counters[r]) == one.counters, (r, dev.counters[r], one.counters)
        arrays, reach, (ids, masks) = got[r]
        for a, b in zip(arrays, one.graph_arrays()):
            np.testing.assert_array_equal(a, b)
        np.testing.assert_array_equal(reach, one.reach_masks())
        oids, omasks = one.finals()
        np.testing.assert_array_equal(ids, oids)
        np.testing.assert_array_equal(masks, omasks)


def test_config3_batch_equals_single_growth(config3):
    _, pmap, goals, seeds, dev, status, _, got = config3
    _assert_batch_equals_single(pmap, dev, status, got, seeds, goals, CONFIG3)


def test_door_batch_equals_single_growth(ctx, door):
    omap, pmap = door
    seeds = [0, 1, 7, 123, 4, 4]
    dev, status = _batch(pmap, seeds, **DOOR)
    _assert_batch_equals_single(pmap, dev, status, _snapshot(dev), seeds, DOOR["goals"], DOOR)


def test_fetch_reads_roadmap_zero_of_the_batch(ctx, door):
    omap, pmap = door
    dev, status = _batch(pmap, [11, 12], **DOOR)

    def fetch(*outs):
        ctx.check(ctx.lib.porrt_pto_fetch(ctx.h, *outs))
    for a, b in zip(P.api._roadmap_graph_arrays(fetch, dev.sizes[0]), dev.graph_arrays(0)):
        np.testing.assert_array_equal(a, b)


# ---- panics, one roadmap at a time

def _panic_iteration(omap, seed, kw, hi):
    """the oracle's panic iteration: the smallest k whose k-iteration growth panics (the reference stops at its first panic)"""
    def panics(k):
        return _oracle(omap, seed, n_min=k, n_max=k, **kw)[1] < -1
    if not panics(hi):
        return None
    lo = 0
    while hi - lo > 1:
        mid = (lo + hi) // 2
        if panics(mid):
            hi = mid
        else:
            lo = mid
    return hi


def test_panics_per_roadmap(ctx):
    """door pixels whose zone id alternates row by row: an edge through a door crosses two zones and panics (map_io.rs:233).
    Every seed's panic code and iteration are the oracle's; the roadmaps that stop before their panic stay fetchable and exact."""
    occ, zones = util.planning_door_map(200)
    door = zones != 255
    zones[door] = (np.nonzero(door)[0] % 2).astype(np.uint8)
    omap, pmap = util.make_pair(ctx, occ, zones, P.DOOR, 0.3)
    kw = dict(start=(-0.8, -0.8), goals=DOOR_GOAL, max_step=0.05, search_radius=5.0)
    seeds = list(range(8))
    at = [_panic_iteration(omap, s, kw, 3000) for s in seeds]
    known = sorted(k for k in at if k is not None)
    assert len(known) >= 2, at
    n = known[len(known) // 2] - 1 if known[0] < known[-1] else known[0]   # some seeds panic within n iterations, others do not
    dev, status = _batch(pmap, seeds, n_min=n, n_max=n, **kw)
    panicked = 0
    for r, s in enumerate(seeds):
        ref, rc = _oracle(omap, s, n_min=n, n_max=n, **kw)
        if rc < -1:
            panicked += 1
            assert status[r] == 5
            assert dev.panic_code[r] == rc and dev.n_it[r] == at[r], (r, dev.panic_code[r], rc, dev.n_it[r], at[r])
            with pytest.raises(P.PorrtError) as e:
                dev.graph_arrays(r)
            assert e.value.code == 1
        else:
            _assert_roadmap_equals_oracle(dev, status, r, ref, rc)
    assert 0 < panicked < len(seeds)


def test_invalid_start_panics_every_roadmap(ctx, door):
    omap, pmap = door
    dev, status = _batch(pmap, [0, 1, 2], start=(-1.0, 0.0), goals=DOOR_GOAL, max_step=0.05, search_radius=5.0, n_min=100, n_max=1000)
    assert _oracle(omap, 0, start=(-1.0, 0.0), goals=DOOR_GOAL, max_step=0.05, search_radius=5.0, n_min=100, n_max=1000)[1] == -100
    assert (status == 5).all() and (dev.panic_code == P.INVALID).all() and (dev.n_it == 0).all()


# ---- argument errors

def test_argument_errors(ctx):
    lib = ctx.lib
    occ, zones = util.planning_door_map(200)
    goal = P.SquareGoal(DOOR_GOAL, 0.05)
    start, low, up = (np.array(v, np.float64) for v in ((-0.8, -0.8), util.LOW, util.UP))

    def call(c, n, seeds, n_alloc=None):
        m = n_alloc if n_alloc is not None else max(n, 1)
        sizes, status = np.zeros(4 * m, np.int64), np.zeros(m, np.int32)
        return c.lib.porrt_pto_grow_batch(c.h, n, P.api._p(seeds), P.api._p(start), P.api._p(low), P.api._p(up), P.api._p(goal.goals),
                                          P.api._p(goal.masks), 1, 0.05, 0.05, 5.0, 10, 100, P.api._p(sizes), P.api._p(status), None, None)

    c2 = P.Context(0)
    try:
        m2 = P.Map(c2, occ, util.LOW, util.UP)           # not uploaded yet
        seeds = np.arange(4, dtype=np.uint64)
        assert call(c2, 4, seeds) == 3                                                     # no map
        assert lib.porrt_pto_fetch_roadmap(c2.h, 0, None, None, None, None, None, None, None, None) == 1   # before any growth
        m2.add_zones(zones, 0.3)
        assert call(c2, 0, seeds) == 1                                                     # no roadmaps
        assert call(c2, -1, seeds) == 1
        assert call(c2, P.api.PTO_MAX_ROADMAPS + 1, seeds, n_alloc=1) == 1                 # above the grid limit
        big = np.arange(60000, dtype=np.uint64)
        assert call(c2, 60000, big) == 1                                                   # more than the device memory holds
        assert b"MB" in c2.lib.porrt_last_error(c2.h)
        assert call(c2, 4, None) == 1                                                      # null seeds
        assert call(c2, 4, seeds) == 0
        assert lib.porrt_pto_fetch_roadmap(c2.h, 4, None, None, None, None, None, None, None, None) == 1   # r out of range
        assert lib.porrt_pto_fetch_roadmap(c2.h, -1, None, None, None, None, None, None, None, None) == 1
        assert lib.porrt_pto_fetch_roadmap(c2.h, 3, None, None, None, None, None, None, None, None) == 0
        bad = np.array([[0xF], [0x3]], np.uint64)                                          # overlapping goal masks
        two = np.array([[0.8, 0.8], [0.5, 0.5]])
        sizes, status = np.zeros(16, np.int64), np.zeros(4, np.int32)
        assert lib.porrt_pto_grow_batch(c2.h, 4, P.api._p(seeds), P.api._p(start), P.api._p(low), P.api._p(up), P.api._p(two),
                                        P.api._p(bad), 2, 0.05, 0.05, 5.0, 10, 100, P.api._p(sizes), P.api._p(status), None, None) == 5
        assert lib.porrt_pto_grow_batch(c2.h, 4, P.api._p(seeds), P.api._p(start), P.api._p(up), P.api._p(low), P.api._p(goal.goals),
                                        P.api._p(goal.masks), 1, 0.05, 0.05, 5.0, 10, 100, P.api._p(sizes), P.api._p(status), None, None) == 5
    finally:
        c2.close()


def test_fetch_roadmap_on_a_panicked_roadmap(ctx, door):
    omap, pmap = door
    dev, status = _batch(pmap, [0], start=(-1.0, 0.0), goals=DOOR_GOAL, max_step=0.05, search_radius=5.0, n_min=10, n_max=10)
    assert status[0] == 5
    assert ctx.lib.porrt_pto_fetch_roadmap(ctx.h, 0, None, None, None, None, None, None, None, None) == 1


# ---- into the belief planner

def test_batch_roadmaps_feed_belief_planning(ctx, config3):
    """two roadmaps of the config-3 batch, each through plan_belief_space, equal the oracle's whole belief pipeline on its seed"""
    import test_gpu_parity as T
    omap, pmap, goals, seeds, dev, status, refs, got = config3
    b0 = [1.0 / 8] * 8
    for r in (1, 5):
        (xy, nvid, rp, col, ev), _, (ids, masks) = got[r]
        plan = P.plan_belief_space(pmap, rp, col, ev, xy, nvid, b0, ids, masks)
        oplan, want, typ = T._belief_compare(ctx, omap, pmap, refs[r], b0)
        np.testing.assert_array_equal(plan.dist, oplan.dist)
        np.testing.assert_array_equal(plan.policy_node, oplan.policy_node)
        np.testing.assert_array_equal(plan.policy_parent, oplan.policy_parent)
        assert plan.expected_cost == oplan.expected_cost and np.isfinite(want[0])
