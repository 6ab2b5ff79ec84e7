"""The C++ restatement of RRT::grow_tree (tests/rrt_oracle.cpp, rrt.rs:102-181) against the Python mirror of the same loop (tests/rrt_mirror.py)
over the oracle's per-query answers: states, parents, dist_from_root and finals bit for bit.  The GPU tests take the C++ restatement
as their reference, so it is pinned to the mirror here."""
import numpy as np
import pytest

from oracle import pyoracle as O
from po_rrt_b200 import synth
import rrt_mirror as R
import rrt_oracle as RO

LOW, UP = [-1.0, -1.0], [1.0, 1.0]


def _shelf():
    """the case of test_rrt_star_tree_invariants"""
    occ, zones = synth.shelf_map(200, n_zones=2)
    omap = O.GridMap(occ, zones, LOW, UP, O.SHELF, 0.5)
    return omap, [0.0, -0.8], O.SquareGoal([((0.6, 0.36), [1])], 0.05), (0.1, 2.0, 500, 1500)


def _door():
    """a single-world door map (no zones)"""
    omap = O.GridMap(synth.rrt_map(size=512, n_rects=256), None, LOW, UP, O.DOOR, 0.3)
    return omap, [-0.8, -0.8], O.SquareGoal([((0.8, 0.8), [1])], 0.05), (0.1, 1.0, 500, 3000)


@pytest.mark.parametrize("seed", [0, 1])
@pytest.mark.parametrize("case", [_shelf, _door], ids=["shelf", "door"])
def test_oracle_grow_tree_equals_mirror(case, seed):
    omap, start, goal, (max_step, search_radius, n_min, n_max) = case()
    samples = O.Pcg64(seed).sample_states(LOW, UP, n_max)
    want = R.grow_tree(R.OracleBackend(omap, start), samples, start, goal, max_step, search_radius, n_min, n_max)
    ref = RO.RRT(omap, LOW, UP, seed=seed)
    rc = ref.grow_tree(start, goal, max_step, search_radius, n_min, n_max)
    xy, parent, dist, finals = ref.tree()
    assert rc == (0 if want[3] else 1)
    np.testing.assert_array_equal(xy, want[0])
    np.testing.assert_array_equal(parent, want[1])
    np.testing.assert_array_equal(dist, want[2])
    assert list(finals) == list(want[3])
    assert len(xy) > 300
    assert n_min <= ref.n_it() <= n_max and (ref.n_it() == n_min or ref.n_it() == n_max or len(finals) == 1)


def test_oracle_grow_tree_root_only():
    omap, start, goal, (max_step, search_radius, _, _) = _door()
    ref = RO.RRT(omap, LOW, UP, seed=0)
    assert ref.grow_tree(start, goal, max_step, search_radius, 0, 0) == 1
    xy, parent, dist, finals = ref.tree()
    assert xy.tolist() == [start] and parent.tolist() == [-1] and dist.tolist() == [0.0] and len(finals) == 0 and ref.n_it() == 0
