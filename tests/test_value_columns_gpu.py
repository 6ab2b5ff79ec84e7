"""plan_qmdp's world columns (porrt_sssp_worlds) in the cases the value-column driver must keep right on both schedules: more than
256 validity ids with more than 64 worlds (the frontier relaxation's node rule reads the validity table itself: the column solver's
4-word masks cannot hold such ids), and final nodes that are invalid in their world.  Against the oracle's dijkstra over
PTOGraphWorldView (pto_graph.rs:245-303)."""
import numpy as np
import pytest

from oracle import pyoracle as O
import po_rrt_b200 as P
from po_rrt_b200 import synth

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def ctx():
    c = P.Context(0)
    yield c
    c.close()


def _roadmap(V, radius, seed):
    """every pair of points closer than `radius`, both directions, as CSR"""
    xy = synth.points(V, seed=seed)
    d2 = ((xy[:, None, :] - xy[None, :, :]) ** 2).sum(-1)
    adj = (d2 < radius * radius) & ~np.eye(V, dtype=bool)
    row_ptr = np.concatenate([[0], np.cumsum(adj.sum(1))]).astype(np.int64)
    col = np.nonzero(adj)[1].astype(np.int32)
    return xy, row_ptr, col


def _oracle(xy, row_ptr, col, nvid, bits, finals):
    og = O.PTOGraph(validities=[list(map(int, m)) for m in bits])
    for k in range(len(xy)):
        og.add_node(xy[k], int(nvid[k]))
    for u in range(len(xy)):
        for e in range(row_ptr[u], row_ptr[u + 1]):
            og.add_edge(u, int(col[e]), 0)
    return np.stack([og.dijkstra(f, world=w) if f else np.full(len(xy), np.inf) for w, f in enumerate(finals)])


def _plan(ctx, xy, row_ptr, col, nvid, bits, finals, force):
    ctx.set_option(P.OPT_FORCE_GLOBAL_SWEEPS, force)
    try:
        return P.dijkstra_worlds(ctx, row_ptr, col, xy, nvid, P.words_from_bits(bits), finals)[0]
    finally:
        ctx.set_option(P.OPT_FORCE_GLOBAL_SWEEPS, 0)


def _finals_with_invalid_ones(rng, nvid, bits, V, W):
    """three random finals per world, one of them a node invalid in that world"""
    finals = []
    for w in range(W):
        bad = np.nonzero(bits[nvid, w] == 0)[0]
        finals.append(sorted(set(rng.choice(V, 2, replace=False).tolist()) | {int(rng.choice(bad))}))
    return finals


def test_worlds_with_more_than_256_validity_ids(ctx):
    """300 validity ids, 70 worlds (two mask words): only the frontier relaxation takes this, with or without the option"""
    V, W, NV = 500, 70, 300
    xy, row_ptr, col = _roadmap(V, 0.16, seed=21)
    rng = np.random.default_rng(7)
    bits = (rng.random((NV, W)) < 0.8).astype(np.uint8)
    nvid = rng.integers(0, NV, V).astype(np.int32)
    finals = _finals_with_invalid_ones(rng, nvid, bits, V, W)
    finals[9] = []                                        # no final: the row stays +inf
    want = _oracle(xy, row_ptr, col, nvid, bits, finals)
    for force in (0, 1):
        got = _plan(ctx, xy, row_ptr, col, nvid, bits, finals, force)
        np.testing.assert_array_equal(got, want)
    assert np.isfinite(want).any() and np.isinf(want[9]).all()


def test_worlds_whose_final_is_invalid_in_the_world(ctx):
    """a final node invalid in its world, on chip and on the frontier relaxation"""
    V, W, NV = 700, 8, 12
    xy, row_ptr, col = _roadmap(V, 0.14, seed=3)
    rng = np.random.default_rng(11)
    bits = (rng.random((NV, W)) < 0.7).astype(np.uint8)
    bits[NV - 1] = 0                                      # a validity id that holds in no world (an obstacle)
    nvid = rng.integers(0, NV, V).astype(np.int32)
    finals = _finals_with_invalid_ones(rng, nvid, bits, V, W)
    want = _oracle(xy, row_ptr, col, nvid, bits, finals)
    for force in (0, 1):
        got = _plan(ctx, xy, row_ptr, col, nvid, bits, finals, force)
        np.testing.assert_array_equal(got, want)
    assert all(want[w][f] == 0.0 for w in range(W) for f in finals[w])
