"""RRT::grow_tree on the device (porrt_rrt_grow / porrt_rrt_grow_batch, RRT / RRTBatch) against the oracle's sequential restatement
with the same seed on the same map: iterations, status, states, parents, dist_from_root and finals of every tree must be identical;
against porrt_rrt_grow with the same seed, the window counters too."""
import numpy as np
import pytest

from oracle import pyoracle as O
import po_rrt_b200 as P
from po_rrt_b200 import synth
import porrt_testutil as util
import rrt_mirror as R
import rrt_oracle as RO

pytestmark = pytest.mark.gpu

GOAL = [((0.8, 0.8), [1])]
CONFIG1 = dict(start=(-0.8, -0.8), goals=GOAL, max_step=0.1, search_radius=1.0, n_min=2500, n_max=10000)


@pytest.fixture(scope="module")
def ctx():
    c = P.Context(0)
    yield c
    c.close()


@pytest.fixture
def map0(ctx):
    """single-world stand-in for the config-1 map, uploaded again for every test: the context holds one map at a time"""
    return util.make_pair(ctx, synth.rrt_map(), None, P.DOOR, 0.3)


def _oracle(omap, seed, start, goals, max_step, search_radius, n_min, n_max, low=util.LOW, up=util.UP):
    ref = RO.RRT(omap, low, up, seed=seed)
    rc = ref.grow_tree(start, O.SquareGoal(goals, 0.05), max_step, search_radius, n_min, n_max)
    return ref, rc


def _batch(pmap, seeds, start, goals, max_step, search_radius, n_min, n_max, low=util.LOW, up=util.UP):
    dev = P.RRTBatch(pmap, low, up, seeds)
    status = dev.grow_tree(start, P.SquareGoal(goals, 0.05), max_step, search_radius, n_min, n_max)
    assert status.shape == (len(seeds),)
    return dev, status


def _assert_tree_equals_oracle(dev, status, t, ref, want_rc):
    assert want_rc in (0, 1), want_rc
    assert status[t] == want_rc and dev.n_it[t] == ref.n_it(), (t, status[t], want_rc, dev.n_it[t], ref.n_it())
    for a, b in zip(dev.tree(t), ref.tree()):
        np.testing.assert_array_equal(a, b)


def _compare(omap, pmap, seeds, **kw):
    dev, status = _batch(pmap, seeds, **kw)
    refs = []
    for t, s in enumerate(seeds):
        ref, rc = _oracle(omap, int(s), **kw)
        _assert_tree_equals_oracle(dev, status, t, ref, rc)
        refs.append(ref)
    return dev, status, refs


# ---- parity with the oracle

def test_shelf_map_shape_and_mirror(ctx):
    """rrt.rs:269-304 shape, the case of test_rrt_star_through_per_query_wrappers; seed 0 also against the Python mirror"""
    occ, zones = synth.shelf_map(200, n_zones=2)
    omap, pmap = util.make_pair(ctx, occ, zones, P.SHELF, 0.5)
    start = (0.0, -0.8)
    zp = omap.zone_positions()
    gx = next(float(zp[0][0]) - dx for dx in (0.06, 0.1, 0.15, 0.2, 0.3) if omap.state_validity([[float(zp[0][0]) - dx, float(zp[0][1])]])[0] >= 0)
    goals = [((gx, float(zp[0][1])), [1])]
    kw = dict(start=start, goals=goals, max_step=0.1, search_radius=2.0, n_min=900, n_max=2500)
    dev, status, refs = _compare(omap, pmap, [0, 1, 2], **kw)
    samples = O.Pcg64(0).sample_states(util.LOW, util.UP, 2500)
    want = R.grow_tree(R.OracleBackend(omap, list(start)), samples, list(start), O.SquareGoal(goals, 0.05), 0.1, 2.0, 900, 2500)
    xy, parent, dist, finals = dev.tree(0)
    np.testing.assert_array_equal(xy, want[0])
    np.testing.assert_array_equal(parent, want[1])
    np.testing.assert_array_equal(dist, want[2])
    assert list(finals) == list(want[3]) and len(want[3]) > 0 and len(xy) > 600


@pytest.mark.parametrize("search_radius", [1.0, 2.0])
def test_config1_shape(ctx, map0, search_radius):
    omap, pmap = map0
    kw = dict(CONFIG1, search_radius=search_radius)
    dev, status, refs = _compare(omap, pmap, [0, 1, 7, 123], **kw)
    assert (status == 0).all(), status
    assert all(dev.sizes[t][1] > 1000 for t in range(4))


def test_64_seeds_equal_single_growth(ctx, map0):
    omap, pmap = map0
    seeds = list(range(64))
    dev, status, _ = _compare(omap, pmap, seeds, **CONFIG1)
    got = [dev.tree(t) for t in range(len(seeds))]
    for t, s in enumerate(seeds):
        one = P.RRT(pmap, util.LOW, util.UP, seed=s)
        rc = one.grow_tree(CONFIG1["start"], P.SquareGoal(GOAL, 0.05), CONFIG1["max_step"], CONFIG1["search_radius"], CONFIG1["n_min"],
                           CONFIG1["n_max"])
        assert rc == status[t] and one.n_it == dev.n_it[t]
        assert tuple(int(x) for x in dev.sizes[t]) == one.sizes
        assert tuple(int(x) for x in dev.counters[t]) == one.counters, (t, dev.counters[t], one.counters)
        for a, b in zip(got[t], one.tree()):
            np.testing.assert_array_equal(a, b)


def test_batch_of_one(ctx, map0):
    omap, pmap = map0
    _compare(omap, pmap, [5], **CONFIG1)


def test_same_seed_twice_gives_identical_trees(ctx, map0):
    omap, pmap = map0
    dev, status, _ = _compare(omap, pmap, [3, 9, 3], **CONFIG1)
    assert status[0] == status[2] and tuple(dev.counters[0]) == tuple(dev.counters[2])
    for a, b in zip(dev.tree(0), dev.tree(2)):
        np.testing.assert_array_equal(a, b)


def test_goal_reached_early_duplicates(ctx, map0):
    """the start next to the goal: every goal sample (each 100th) lands exactly on the goal state, more than 64 times, so the 1-NN
    ties among exact duplicates and the kd keys go deeper than 64 levels"""
    omap, pmap = map0
    kw = dict(CONFIG1, start=(0.76, 0.76), n_min=8000, n_max=10000)
    dev, status, refs = _compare(omap, pmap, [0, 1], **kw)
    assert (status == 0).all() and (dev.n_it == 8000).all()
    _, counts = np.unique(refs[0].tree()[0], axis=0, return_counts=True)
    assert counts.max() > 64


def test_unreachable_goal_and_root_only(ctx):
    occ = synth.rrt_map()
    x, y = synth.pixel_centres(occ.shape[0])
    occ[(np.abs(x - 0.8) <= 0.08) & (np.abs(y - 0.8) <= 0.08)] = 0          # the whole goal diamond is an obstacle
    omap, pmap = util.make_pair(ctx, occ, None, P.DOOR, 0.3)
    dev, status, _ = _compare(omap, pmap, [0, 1], **dict(CONFIG1, n_min=100, n_max=3000))
    assert (status == 1).all() and (dev.n_it == 3000).all()
    dev, status, _ = _compare(omap, pmap, [0, 1], **dict(CONFIG1, n_min=0, n_max=0))
    assert (status == 1).all() and (dev.n_it == 0).all() and (dev.sizes[:, 1] == 1).all()
    xy, parent, dist, finals = dev.tree(1)
    assert xy.tolist() == [list(CONFIG1["start"])] and parent.tolist() == [-1] and dist.tolist() == [0.0] and len(finals) == 0


def test_panics_per_tree(ctx, map0):
    """bounds reaching past the map: a steered state outside it panics (PORRT_PANIC_OOB).  Every panicking tree reports the oracle's
    code and iteration; the trees that do not panic within n iterations stay fetchable and exact."""
    omap, pmap = map0
    low, up = [-1.04, -1.04], [1.04, 1.04]
    seeds = list(range(8))
    kw = dict(CONFIG1, low=low, up=up, n_min=20000, n_max=20000)
    at = []
    for s in seeds:
        ref, rc = _oracle(omap, s, **kw)
        at.append(ref.n_it() if rc < -1 else None)
    known = sorted(k for k in at if k is not None)
    assert len(known) >= 2, at
    n = known[len(known) // 2] - 1 if known[0] < known[-1] else known[0]
    kw = dict(kw, n_min=n, n_max=n)
    dev, status = _batch(pmap, seeds, **kw)
    panicked = 0
    for t, s in enumerate(seeds):
        ref, rc = _oracle(omap, s, **kw)
        if rc < -1:
            panicked += 1
            assert rc == P.PANIC_OOB and status[t] == 5
            assert dev.panic_code[t] == rc and dev.n_it[t] == ref.n_it(), (t, dev.panic_code[t], rc, dev.n_it[t], ref.n_it())
            with pytest.raises(P.PorrtError) as e:
                dev.tree(t)
            assert e.value.code == 1
        else:
            _assert_tree_equals_oracle(dev, status, t, ref, rc)
    assert 0 < panicked < len(seeds)
    one = P.RRT(pmap, low, up, seed=seeds[at.index(known[0])])
    with pytest.raises(P.PorrtError) as e:
        one.grow_tree(kw["start"], P.SquareGoal(GOAL, 0.05), 0.1, 1.0, n, n)
    assert e.value.code == 5 and e.value.panic_code == P.PANIC_OOB and one.n_it == known[0]


# ---- argument and fetch errors

def test_argument_and_fetch_errors(ctx):
    occ = synth.rrt_map(size=256, n_rects=64)
    goal = P.SquareGoal(GOAL, 0.05)
    start, low, up = (np.array(v, np.float64) for v in ((-0.8, -0.8), util.LOW, util.UP))
    p = P.api._p

    def call(c, n, seeds, n_alloc=None, goals=goal.goals, masks=goal.masks, n_goals=1, lo=low, hi=up):
        m = n_alloc if n_alloc is not None else max(n, 1)
        sizes, status = np.zeros(3 * m, np.int64), np.zeros(m, np.int32)
        return c.lib.porrt_rrt_grow_batch(c.h, n, p(seeds), p(start), p(lo), p(hi), p(goals), p(masks), n_goals, 0.05, 0.1, 1.0, 10, 100,
                                          p(sizes), p(status), None, None)

    def fetch(c, t):
        return c.lib.porrt_rrt_fetch_tree(c.h, t, None, None, None, None)

    c2 = P.Context(0)
    try:
        m2 = P.Map(c2, occ, util.LOW, util.UP)           # not uploaded yet
        seeds = np.arange(4, dtype=np.uint64)
        assert call(c2, 4, seeds) == 3                                                     # no map
        assert fetch(c2, 0) == 1                                                           # before any growth
        m2.init_without_zones()
        assert call(c2, 0, seeds) == 1                                                     # no trees
        assert call(c2, -1, seeds) == 1
        assert call(c2, P.api.PTO_MAX_ROADMAPS + 1, seeds, n_alloc=1) == 1                 # above the grid limit
        big = np.arange(60000, dtype=np.uint64)
        assert call(c2, 60000, big) == 1                                                   # more than the device memory holds
        assert b"MB" in c2.lib.porrt_last_error(c2.h)
        assert call(c2, 4, None) == 1                                                      # null seeds
        assert fetch(c2, 0) == 1                                                           # still nothing grown
        bad = np.array([[0x1], [0x1]], np.uint64)                                          # overlapping goal masks
        two = np.array([[0.8, 0.8], [0.5, 0.5]])
        assert call(c2, 4, seeds, goals=two, masks=bad, n_goals=2) == 5
        assert call(c2, 4, seeds, lo=up, hi=low) == 5                                      # low >= up
        assert call(c2, 4, seeds) == 0
        assert fetch(c2, 4) == 1 and fetch(c2, -1) == 1                                    # t out of range
        assert fetch(c2, 3) == 0
        # a panicked tree: bounds far past the map, every tree steps out of it
        assert call(c2, 2, seeds, lo=np.array([-3.0, -3.0]), hi=np.array([3.0, 3.0])) == 0
        assert fetch(c2, 0) == 1 and b"panicked" in c2.lib.porrt_last_error(c2.h)
    finally:
        c2.close()


# ---- RRT and PTO growth keep separate state

def test_rrt_and_pto_growth_are_independent(ctx):
    occ, zones = util.planning_door_map(200)
    omap, pmap = util.make_pair(ctx, occ, zones, P.DOOR, 0.3)
    pto = P.PTOBatch(pmap, util.LOW, util.UP, [0, 1])
    pto.grow_graph((-0.8, -0.8), P.SquareGoal([((0.8, 0.8), [1, 1, 1, 1])], 0.05), 0.05, 5.0, 700, 100000)
    road = [pto.graph_arrays(r) for r in range(2)]
    pto_finals = pto.finals(1)
    rrt = P.RRTBatch(pmap, util.LOW, util.UP, [4, 5, 6])
    rrt.grow_tree((-0.8, -0.8), P.SquareGoal([((0.8, 0.8), [1, 1, 1, 1])], 0.05), 0.1, 1.0, 1500, 5000)
    trees = [rrt.tree(t) for t in range(3)]

    def fetch(*outs):
        ctx.check(ctx.lib.porrt_pto_fetch(ctx.h, *outs))
    for a, b in zip(P.api._roadmap_graph_arrays(fetch, pto.sizes[0]), road[0]):   # porrt_pto_fetch after the RRT growth
        np.testing.assert_array_equal(a, b)
    for a, b in zip(pto.graph_arrays(1), road[1]):
        np.testing.assert_array_equal(a, b)
    for a, b in zip(pto.finals(1), pto_finals):
        np.testing.assert_array_equal(a, b)
    pto2 = P.PTO(pmap, util.LOW, util.UP, seed=9)                                   # and the RRT trees after a PTO growth
    pto2.grow_graph((-0.8, -0.8), P.SquareGoal([((0.8, 0.8), [1, 1, 1, 1])], 0.05), 0.05, 5.0, 300, 100000)
    for t in range(3):
        for a, b in zip(rrt.tree(t), trees[t]):
            np.testing.assert_array_equal(a, b)
