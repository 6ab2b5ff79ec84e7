"""porrt_extract_policy and porrt_refine_policy_reparent on a belief table left on the device (plan_belief_space(copy=None)):
the policy walk and Reparent's tree search then fetch the value / type columns they visit, one belief at a time.  They must give
what they give on the table copied to the host, bit for bit."""
import numpy as np
import pytest

from oracle import pyoracle as O
import po_rrt_b200 as P
from po_rrt_b200 import synth
import porrt_testutil as util

pytestmark = pytest.mark.gpu

RADII = (0.15, 0.3)


@pytest.fixture(scope="module")
def ctx():
    c = P.Context(0)
    yield c
    c.close()


def _door(ctx):
    occ, zones = util.planning_door_map(200)
    omap, pmap = util.make_pair(ctx, occ, zones, P.DOOR, 0.3)
    return omap, pmap, dict(start=(-0.8, -0.8), goals=[((0.8, 0.8), [1, 1, 1, 1])], max_step=0.05, search_radius=5.0, n_min=3000), [0.1, 0.1, 0.1, 0.7]


def _config3(ctx):
    """BASELINE config 3 shape: 8 shelf zones, B = 255 reachable beliefs"""
    Z = 8
    occ, zones = synth.shelf_map(200, n_rects=10, n_zones=Z, seed=5)
    omap, pmap = util.make_pair(ctx, occ, zones, P.SHELF, 0.5)
    zp = omap.zone_positions()
    goals = [((float(zp[z][0]) - 0.08, float(zp[z][1])), [1 if k == z else 0 for k in range(Z)]) for z in range(Z)]
    return omap, pmap, dict(start=(0.0, -0.9), goals=goals, max_step=0.1, search_radius=2.0, n_min=5000), [1.0 / Z] * Z


@pytest.mark.parametrize("shape", [_door, _config3], ids=["door", "config3"])
def test_policy_and_reparent_on_device_table(ctx, shape):
    omap, pmap, grow, b0 = shape(ctx)
    pto = O.PTO(omap, util.LOW, util.UP, seed=0)
    assert pto.grow_graph(grow["start"], O.SquareGoal(grow["goals"], 0.05), grow["max_step"], grow["search_radius"], grow["n_min"], 100000) == 0
    xy, nvid, rp, col, ev = pto.graph.export(0)
    fin_ids, fin_bits = pto.reach.finals()
    runs = {}
    for copy in (True, None):
        plan = P.plan_belief_space(pmap, rp, col, ev, xy, nvid, b0, fin_ids, P.words_from_bits(fin_bits), copy=copy)
        # Reparent reads the ctx's last porrt_belief_vi, so each plan's refinements run before the next plan
        runs[copy] = plan, [P.refine_policy_reparent(ctx, plan, r) for r in RADII]
    (host, host_rep), (dev, dev_rep) = runs[True], runs[None]
    assert host.dist is not None and dev.dist is None   # the second plan left its table on the device
    assert host.policy_leaf.sum() >= 2
    for name in ("policy_node", "policy_belief", "policy_parent", "policy_leaf"):
        np.testing.assert_array_equal(getattr(dev, name), getattr(host, name), err_msg=name)
    assert np.float64(dev.expected_cost).tobytes() == np.float64(host.expected_cost).tobytes()
    for r, want, got in zip(RADII, host_rep, dev_rep):
        assert got["xy"].tobytes() == want["xy"].tobytes(), r
        for name in ("node", "belief", "parent", "is_leaf"):
            np.testing.assert_array_equal(got[name], want[name], err_msg="%s at radius %g" % (name, r))
        assert np.float64(got["expected_cost"]).tobytes() == np.float64(want["expected_cost"]).tobytes(), r
        assert (got["tree_nodes"], got["transitions"]) == (want["tree_nodes"], want["transitions"]), r
